"""Times grad and div (csrc/diffop.cu) against the generic gsp_spmm on the same layouts (GPU box).

    python tools/diffop_probe.py [--n 1000000] [--nsig 64] [--launches 50] [--rounds 5] [--out F]

Graph: Sensor(n, k=10, seed=0, order="morton"), float32, nsig signals.  grad runs over the
edge-major layout of D (the CSR of D^T, Ne x N), div over the vertex-major one (D as CSR, N x Ne);
gsp_spmm_f32 runs on the same CSR arrays (it also streams x_cur[row] for its beta term, so its x
is padded to max(N, Ne) rows).  A device copy of the (Ne, nsig) block is the bandwidth reference.
Each round times every kernel over `launches` back-to-back launches with CUDA events, the kernels
alternating within the round; the median round is reported.  Algorithmic bytes come from the
shapes: CSR records read once, every signal row read or written once.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=30)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        out["power_limit_and_max_sm_clock"] = "not read: %s" % exc
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--nsig", type=int, default=64)
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    import pygsp_b200 as gsp
    from pygsp_b200 import _native as nat

    torch.cuda.set_device(0)
    G = gsp.graphs.Sensor(a.n, k=10, seed=0, order="morton")
    G.compute_differential_operator()
    D, N, Ne, nsig, item = G.D, G.N, G.Ne, a.nsig, 4
    dev = G.device
    st = nat.stream_ptr(dev)
    gen = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn((max(N, Ne), nsig), device=dev, generator=gen)
    y = torch.randn((Ne, nsig), device=dev, generator=gen)
    g_out = torch.empty((Ne, nsig), device=dev)
    d_out = torch.empty((N, nsig), device=dev)
    g_ref = torch.empty_like(g_out)
    d_ref = torch.empty_like(d_out)
    copy_dst = torch.empty_like(y)

    kernels = {
        "grad": lambda: nat.call("gsp_grad_f32", nat.i64(Ne), D.d_indptr, D.d_indices, D.d_data,
                                 x, nat.i64(nsig), g_out, st),
        "spmm_edge_major": lambda: nat.call("gsp_spmm_f32", nat.i64(Ne), D.d_indptr, D.d_indices,
                                            D.d_data, x, nat.i64(nsig), g_ref, st),
        "div": lambda: nat.call("gsp_div_f32", nat.i64(N), D.v_indptr, D.v_indices, D.v_data, y,
                                nat.i64(nsig), d_out, st),
        "spmm_vertex_major": lambda: nat.call("gsp_spmm_f32", nat.i64(N), D.v_indptr,
                                              D.v_indices, D.v_data, y, nat.i64(nsig), d_ref, st),
        "copy": lambda: copy_dst.copy_(y),
    }
    csr_bytes = {"edge_major": (Ne + 1) * 4 + D.nnz * (4 + item),
                 "vertex_major": (N + 1) * 4 + D.nnz * (4 + item)}
    sig_n, sig_e = N * nsig * item, Ne * nsig * item
    algo = {"grad": csr_bytes["edge_major"] + sig_n + sig_e,
            "spmm_edge_major": csr_bytes["edge_major"] + sig_n + sig_e,
            "div": csr_bytes["vertex_major"] + sig_e + sig_n,
            "spmm_vertex_major": csr_bytes["vertex_major"] + sig_e + sig_n,
            "copy": 2 * sig_e}

    for fn in kernels.values():                       # warm every shape
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in kernels}
    for _ in range(a.rounds):
        for name, fn in kernels.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.launches):
                fn()
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1) / a.launches)

    g_rel = float(((g_out - g_ref).abs().max() / g_ref.abs().max()).item())
    d_rel = float(((d_out - d_ref).abs().max() / d_ref.abs().max()).item())
    copy_gbs = algo["copy"] / (float(np.median(times["copy"])) * 1e-3) / 1e9
    res = {"card": card(), "graph": "Sensor(%d, k=10, seed=0, order='morton') float32" % N,
           "N": N, "Ne": Ne, "nnz_D": D.nnz, "nsig": nsig, "launches_per_round": a.launches,
           "rounds": a.rounds, "bytes_note": "algorithmic: CSR records once, each signal row once",
           "max_rel_diff_vs_spmm": {"grad": g_rel, "div": d_rel}, "kernels": {}}
    for name in kernels:
        ms = float(np.median(times[name]))
        gbs = algo[name] / (ms * 1e-3) / 1e9
        res["kernels"][name] = {"ms_median": ms, "ms_all_rounds": times[name],
                                "algorithmic_bytes": algo[name], "GBps": gbs,
                                "of_measured_copy": gbs / copy_gbs}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
