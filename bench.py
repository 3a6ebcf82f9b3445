#!/usr/bin/env python
"""Benchmark of the Chebyshev filtering hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

metric  = cheby_op filtered-vertices/sec = N * Nsig * order / t
workload, 1 GPU : BASELINE configs[1] -- Sensor-type 2-D k-NN graph, N = 1e6, k = 10,
          seed 0 (Morton-numbered), 64 float32 signals, Heat(scale=50), order 30; the same
          line carries `targets`: short runs of the north-star target (10M-vertex k-NN) and of
          configs[2] (10M-vertex grid, 6-filter MexicanHat, order 50) with their parity.
workload, N > 1 : STRONG scaling of the north-star target -- ONE 10M-vertex k-NN graph
          (the 1-GPU `targets.knn10m` graph) 1-D partitioned over the N ranks, halo exchange
          per recurrence step over NVLink peer memory; every line carries `parity_rel_err`
          (partitioned result vs the single-GPU engine on the whole graph, every rank) and the
          one-GPU time of the same graph measured in the same run.  --scaling weak = 1e6
          vertices per GPU (strips of one k-NN graph); --workload config5 = BASELINE configs[4]
          (5e7-vertex 3-D k-NN, 128 signals, order 40; every rank generates its slab on its
          GPU), --workload config4 = configs[3] (SBM); their lines carry the constant-signal
          property and a cross-check of the two exchange transports instead.
A "step" is one complete cheby_op call (order fused recurrence kernels).

value   : CUDA-event time of K calls with graph + signals resident in HBM.
e2e     : the same metric through Filter.filter() with HOST (pinned) signals --
          H2D and D2H copies inside the timed region.
roofline: algorithmic bytes of the recurrence / measured kernel time vs the
          measured HBM copy bandwidth (MEASURED_PEAKS.json).
cpu_baseline: the unmodified reference (baseline/_ref; the oracle port if absent) on one core,
          a bounded sample of the same workload.
--impl reference: the unmodified reference's CPU path on up to 64 host processes
          (one signal column each; the reference is single-threaded by construction).
--dump-outputs DIR: after the timed steps, what the last one returned, (Nscales, vertices,
          signals) float32, as DIR/y.npy (DIR/y_rank<r>.npy on N > 1 GPUs); above DUMP_BYTES
          in all, the rows of a fixed, seeded sample of vertices.  Graph and signals are
          seeded, so two builds given the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "cheby_op_filtered_vertices_per_sec"
UNIT = "vertex*signal*order/s"
WORKLOAD = dict(name="sensor_knn2d_N1e6_k10_seed0_morton_heat50_order30_nsig64",
                N=1_000_000, k=10, seed=0, nsig=64, order=30, scale=50.0, graph="sensor",
                bank="heat", nscales=1)
# the other BASELINE configurations, single GPU, for the record (profiles/): --workload NAME
WORKLOADS = {
    "config2": WORKLOAD,
    "knn10m": dict(WORKLOAD, name="sensor_knn2d_N1e7_k10_seed0_morton_heat50_order30_nsig64",
                   N=10_000_000),
    "config3": dict(name="grid2d_3162x3162_mexicanhat6_order50_nsig64", N=3162 * 3162, k=4,
                    seed=0, nsig=64, order=50, scale=50.0, graph="grid2d", bank="mexicanhat",
                    nscales=6),
    "config4": dict(name="sbm_N1e7_k8_p5e-6_q5e-7_heat50_order30_nsig32", N=10_000_000, k=8,
                    seed=0, nsig=32, order=30, scale=50.0, graph="sbm", bank="heat", nscales=1),
    "config5": dict(name="knn3d_N5e7_k16_seed0_morton_heat50_order40_nsig128", N=50_000_000, k=16,
                    seed=0, nsig=128, order=40, scale=50.0, graph="knn3d", bank="heat", nscales=1),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", "--vertices", dest="n", type=int, default=None,
                    help="override the per-GPU vertex count")
    ap.add_argument("--k", type=int, default=None, help="override the k of the k-NN workloads (probes)")
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS),
                    help="default: config2 on one GPU, knn10m (strong scaling) on N > 1")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="N > 1: one fixed graph split over the ranks (default) or 1e6 vertices per GPU")
    ap.add_argument("--no-targets", action="store_true",
                    help="skip the short runs of the 10M k-NN target and config 3 in the 1-GPU line")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-columns", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed under DIR (see above)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of --impl ours")
    return args


# ------------------------------------------------------------------ workload
def host_graph(n, k, seed):
    """Adjacency of Sensor(N, k, seed) with Morton vertex numbering, built on the
    host with scipy's cKDTree (input fabrication, outside every timed region)."""
    from scipy import sparse, spatial
    from pygsp_b200.graphs import morton_order
    coords = np.random.default_rng(seed).uniform(0, 1, (n, 2))
    coords = coords[morton_order(coords)]
    D, NN = spatial.cKDTree(coords).query(coords, k=k + 1, workers=-1)
    sigma = np.mean(D[:, 1:])
    W = sparse.csr_matrix((np.exp(-D[:, 1:].ravel() ** 2 / sigma),
                           (np.repeat(np.arange(n), k), NN[:, 1:].ravel())), shape=(n, n))
    W = ((W + W.T) / 2).tocsr()
    W.sort_indices()
    return W


def algorithmic_bytes(n, nnz, nsig, nscales, order, itemsize=4, clenshaw=False):
    """Compulsory HBM traffic of one call: (first step, dominant step, whole call).

    Forward recurrence = the reference's algorithm, SURVEY.md 8(d): CSR once, T_{k-1} once,
    T_{k-2} read, T_k written, every r block read + written: 3 + 2 Nscales passes over the
    signal block per step (2 + Nscales for the first).  Clenshaw form (single filter, the
    engine's default): no accumulator block -- b_{k+1} read, b_{k+2} read, source read, b_k
    written = 4 passes (first step 2, second 3: b_K = c_K x is folded into the source)."""
    csr = (4 + itemsize) * nnz + 4 * (n + 1)
    vec = itemsize * n * nsig
    if clenshaw and nscales == 1 and order >= 2:
        first, step = csr + 2 * vec, csr + 4 * vec
        return first, step, order * csr + vec * (2 + 3 + 4 * (order - 2))
    first = csr + vec * (2 + nscales)
    step = csr + vec * (3 + 2 * nscales)
    return first, step, first + (order - 1) * step


def config_dict(wl, world, scaling):
    """The `config` object of a bench line: the same keys and values on both arms."""
    n_global = wl["N"] * (world if scaling == "weak" else 1)
    return {"workload": wl["name"], "N_global": n_global, "N_per_gpu": n_global // world,
            "k": wl["k"], "nsig": wl["nsig"], "order": wl["order"], "nscales": wl["nscales"],
            "scaling": scaling if world > 1 else "single GPU",
            "partition": "single GPU" if world == 1 else
                         "1-D vertex partition, %d contiguous row blocks, halo exchange per "
                         "recurrence step" % world,
            "l2_policy": "inputs_exceed_l2 (the state blocks of a call are >= 0.5 GB per GPU, "
                         "L2 is 126 MB)"}


def pick_workload(args, world):
    """(workload dict, scaling).  One GPU: configs[1].  N > 1: strong scaling of the 10M-vertex
    k-NN target (weak: 1e6-vertex strips); config4 / config5 are strong by definition."""
    name = args.workload or ("config2" if (world == 1 or args.scaling == "weak") else "knn10m")
    wl = dict(WORKLOADS[name])
    if args.n:
        wl["N"] = args.n
    if args.k:
        wl["k"] = args.k
    scaling = "weak" if (world > 1 and name == "config2") else "strong"
    return name, wl, scaling


class ClockSampler:
    """nvidia-smi clocks / throttle reasons, sampled every 20 ms by one long-running
    process (started early: nvidia-smi needs ~1 s to come up); ``summary(t0, t1)`` keeps
    the samples whose timestamp falls inside the timed region."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        import datetime
        for line in self.proc.stdout:
            cells = [c.strip() for c in line.split(",")]
            stamp = time.time()                          # arrival time (pipes may batch lines) ...
            try:                                         # ... so prefer nvidia-smi's own timestamp
                stamp = datetime.datetime.strptime(cells[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except (ValueError, IndexError):
                pass
            self.rows.append((stamp, cells))

    def __exit__(self, *exc):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0=None, t1=None):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def collect(rows):
            sm, mx, power, reasons = [], [], [], set()
            for _, r in rows:
                try:
                    sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
                except (ValueError, IndexError):
                    continue
                for name, val in zip(names, r[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            return sm, mx, power, reasons
        window = "timed region"
        rows = [x for x in self.rows if t0 is None or (t0 - 0.02 <= x[0] <= t1 + 0.03)]
        sm, mx, power, reasons = collect(rows)
        if not sm:                                   # region shorter than a sampling period
            window = "warm-up + timed region"
            rows = [x for x in self.rows if t0 is None or x[0] >= t0 - 1.0]
            sm, mx, power, reasons = collect(rows)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)),
                "power_w_max": float(max(power)), "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full`
    capture of THIS workload on one GPU (profiles/roofline_traffic.json, keyed by workload);
    None when no capture exists (multi-GPU runs, other workloads)."""
    path = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if workload is None or not os.path.exists(path):
        return None
    try:
        entry = json.load(open(path)).get(workload)
        return float(entry["dram_bytes_per_launch"]) if entry else None
    except Exception:
        return None


# -------------------------------------------------------------- CPU reference
_REF = {}          # inherited by the forked workers: nothing big is pickled per task
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def _import_reference():
    """The unmodified PyGSP 0.6.1, pip-installed offline into baseline/_ref (git-ignored,
    travels with the snapshot): `pip install --no-index --no-deps --target baseline/_ref
    /root/reference`.  None when absent -- the oracle port then stands in."""
    if not os.path.isdir(os.path.join(REF_DIR, "pygsp")):
        return None
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    try:
        import logging
        import pygsp
        logging.getLogger("pygsp").setLevel(logging.ERROR)
        return pygsp
    except Exception:
        return None


def _cpu_worker(cols):
    lo, hi = cols
    x = _REF["x"][:, lo:hi]
    if _REF["kind"] == "reference":
        _REF["filter"].filter(x, method="chebyshev", order=_REF["order"])   # stock PyGSP path
    else:
        from oracle import pygsp_oracle as orc
        orc.cheby_op(_REF["L"], _REF["lmax"], _REF["c"], x)
    return hi - lo


class CpuReference:
    """The reference's CPU path on `procs` host processes.

    kind 'reference': the real `pygsp.filters.Heat(G, scale).filter(x, order=...)` (scipy
    csr_matvecs + numpy, float64, single-threaded by construction) with the signal columns
    sharded over forked processes; kind 'port': the oracle restatement of the same
    arithmetic when baseline/_ref is not there."""

    def __init__(self, W, lmax, scale, order, x, procs):
        import multiprocessing as mp
        pygsp = _import_reference()
        _REF.clear()
        _REF.update(lmax=lmax, order=order, x=np.ascontiguousarray(x))
        if pygsp is not None:
            G = pygsp.graphs.Graph(W)
            G._lmax, G._lmax_method = float(lmax), "lanczos"      # same lmax on both sides
            _REF.update(kind="reference", filter=pygsp.filters.Heat(G, scale=scale))
        else:
            from oracle import pygsp_oracle as orc
            _REF.update(kind="port", L=orc.laplacian(W),
                        c=orc.cheby_coeff(orc.heat_kernels(lmax, scale), lmax, order))
        self.kind = _REF["kind"]
        self.procs = max(1, min(procs, x.shape[1]))
        edges = np.linspace(0, x.shape[1], self.procs + 1).astype(int)
        self.chunks = [(int(a), int(b)) for a, b in zip(edges[:-1], edges[1:]) if b > a]
        self.pool = mp.get_context("fork").Pool(self.procs) if self.procs > 1 else None

    def time_once(self):
        t0 = time.perf_counter()
        if self.pool is None:
            _cpu_worker(self.chunks[0])
        else:
            self.pool.map(_cpu_worker, self.chunks, chunksize=1)
        return time.perf_counter() - t0

    def close(self):
        if self.pool is not None:
            self.pool.close()
            self.pool.join()


def run_reference(args):
    """--impl reference: the reference's CPU path on this box's host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import pygsp_oracle as orc
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    name, wl, scaling = pick_workload(args, world)
    cores = os.cpu_count() or 1
    procs = min(cores, 64)
    # The CPU path is timed on the 1e6-vertex instance of the workload's generator (same k,
    # seed, weights, order, filter): that IS configs[1]; for the 10M-vertex target it is the
    # 1/10-scale instance SURVEY.md 8(d) prescribes for CPU timing -- the metric is a rate
    # (vertex*signal*order per second), so no extrapolation enters the value.
    n_cpu = min(wl["N"], 1_000_000)
    W = host_graph(n_cpu, wl["k"], wl["seed"])
    lmax = orc.upper_bound(W)                  # estimate_lmax(method="bounds"): deterministic
    ncols = min(wl["nsig"], procs)              # bounded sample: one signal column per process
    x = np.random.default_rng(0).standard_normal((n_cpu, ncols))
    ref = CpuReference(W, lmax, wl["scale"], wl["order"], x, procs)
    for _ in range(min(args.warmup, 1)):
        ref.time_once()
    times = [ref.time_once() for _ in range(args.steps)]
    ref.close()
    t = float(np.sum(times))
    value = n_cpu * ncols * wl["order"] * args.steps / t
    what = ("unmodified PyGSP 0.6.1 from baseline/_ref, Heat(G, 50).filter(x, order=30)"
            if ref.kind == "reference" else "oracle port of approximations.cheby_op")
    sample = "%d of %d signal columns per step (one per process), %s, full order; %s" % (
        ncols, wl["nsig"], "full graph" if n_cpu == wl["N"] else
        "the N=%d instance of the same generator (1/%d scale)" % (n_cpu, wl["N"] // n_cpu), what)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": config_dict(wl, world, scaling),
        "graph": {"N_timed": n_cpu, "nnz_W": int(W.nnz), "lmax": lmax},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": ref.procs, "kind": ref.kind,
                         "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ------------------------------------------------------------------- our arm
DUMP_BYTES = 48 << 20


def dump_output(torch, path, name, y, max_bytes):
    """y (..., vertices, signals) -> path/name.npy as computed; over max_bytes, the rows of
    a fixed sample of vertices (seed 0: the same rows for the same vertex count)."""
    n = y.shape[-2]
    row_bytes = y.numel() // n * y.element_size()
    if n * row_bytes > max_bytes:
        rows = np.sort(np.random.default_rng(0).choice(n, max_bytes // row_bytes, replace=False))
        y = y.index_select(y.dim() - 2, torch.from_numpy(rows).to(y.device))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, name + ".npy"), y.cpu().numpy())


def build_graph(gsp, wl):
    """The workload's graph through the Graph API: adjacency, Laplacian and lmax on the device."""
    if wl["graph"] == "grid2d":
        side = int(round(wl["N"] ** 0.5))
        G = gsp.graphs.Grid2d(side, side)             # stencil written on the device
    elif wl["graph"] == "sbm":
        G = gsp.graphs.StochasticBlockModel(wl["N"], k=wl["k"], p=5e-6, q=5e-7, seed=wl["seed"])
    else:                                             # grid-hash k-NN + symmetrisation on the device
        G = gsp.graphs.Sensor(wl["N"], k=wl["k"], seed=wl["seed"], order="morton")
    G.estimate_lmax()
    return G


def make_bank(gsp, G, wl):
    bank = (gsp.filters.MexicanHat(G, Nf=wl["nscales"]) if wl["bank"] == "mexicanhat"
            else gsp.filters.Heat(G, scale=wl["scale"]))
    c = np.atleast_2d(gsp.filters.compute_cheby_coeff(bank, m=wl["order"]))
    return bank, c


def device_op(apx, L, lmax, c):
    """The device-to-device operator the public API runs: Clenshaw form for one filter."""
    if c.shape[0] == 1:
        return lambda xx: apx.cheby_clenshaw_device(L, lmax, c, xx)[None]
    return lambda xx: apx.cheby_op_device(L, lmax, c, xx)


def csr_row_block(L, lo, hi):
    """Rows [lo, hi) of a DeviceCSR as a host scipy matrix with global column ids."""
    from scipy import sparse
    ptr = L.indptr[lo:hi + 1].cpu().numpy().astype(np.int64)
    a, b = int(ptr[0]), int(ptr[-1])
    return sparse.csr_matrix((L.data[a:b].cpu().numpy(), L.indices[a:b].cpu().numpy(), ptr - a),
                             shape=(hi - lo, L.shape[1]))


def time_calls(torch, fn, x, steps, warm):
    """ms per call: CUDA events on the current stream around `steps` calls, after `warm` calls."""
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(warm):
        fn(x)
    torch.cuda.synchronize()
    start.record()
    for _ in range(steps):
        fn(x)
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / steps


def oracle_parity(L, lmax, c, x_col, got):
    """max|got - ref| / max|ref| of one signal column against the float64 oracle (CPU)."""
    from oracle import pygsp_oracle as orc
    ref = orc.cheby_op(L.to_scipy().astype(np.float64), lmax, c, x_col.double().cpu().numpy())
    ref = ref.reshape(c.shape[0], -1)
    got = got.double().cpu().numpy().reshape(c.shape[0], -1)
    return float(np.abs(got - ref).max() / np.abs(ref).max())


def run_target(gsp, apx, torch, name, peak):
    """Short run of another BASELINE workload on this GPU: 3 timed calls after 1 warm-up,
    roofline fraction, one signal column checked against the float64 oracle."""
    wl = dict(WORKLOADS[name])
    t0 = time.perf_counter()
    G = build_graph(gsp, wl)
    bank, c = make_bank(gsp, G, wl)
    t_build = time.perf_counter() - t0
    n, nsig, order = G.N, wl["nsig"], wl["order"]
    x = torch.randn(n, nsig, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    op = device_op(apx, G.L, G.lmax, c)
    ms = time_calls(torch, op, x, 3, 1)
    clen = c.shape[0] == 1
    _, b_step, b_call = algorithmic_bytes(n, G.L.nnz, nsig, wl["nscales"], order, clenshaw=clen)
    col = x[:, :1].contiguous()
    parity = oracle_parity(G.L, G.lmax, c, col, device_op(apx, G.L, G.lmax, c)(col))
    out = {"workload": wl["name"], "N": n, "nnz_L": G.L.nnz, "nsig": nsig, "nscales": wl["nscales"],
           "order": order, "steps": 3, "warmup": 1, "ms_per_step": ms,
           "value": n * nsig * order / (ms / 1e3), "value_bank": n * nsig * order * wl["nscales"] / (ms / 1e3),
           "unit": UNIT, "form": "clenshaw" if clen else "forward",
           "roofline_frac": b_call / (ms / 1e3) / 1e9 / peak, "achieved_GBps": b_call / (ms / 1e3) / 1e9,
           "algorithmic_bytes_per_call": b_call, "parity_rel_err_one_column_vs_oracle": parity,
           "lmax": G.lmax, "build_s": t_build}
    del G, x, op, col
    torch.cuda.empty_cache()
    return out


def build_partitioned_sbm(gsp, wl, rank, world, torch, dist):
    """BASELINE config 4 on N > 1 GPUs (strong scaling): every rank samples the SAME 10M-vertex
    SBM (seeded), keeps rows [N p/P, N (p+1)/P) of its Laplacian; the halo is most of the
    graph (no locality), so this is the NVLink-bound case."""
    from pygsp_b200 import distributed as gd
    from pygsp_b200.graphs.generators import laplacian_rows, sbm_adjacency
    W, _ = sbm_adjacency(wl["N"], wl["k"], None, 5e-6, 5e-7, seed=wl["seed"])
    bounds = gd.even_bounds(wl["N"], world)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    L_rows, dw = laplacian_rows(W[lo:hi], lo)
    del W
    plan = gd.HaloPlan(L_rows, bounds, rank)
    op = gd.PartitionedCheby(plan, dtype=torch.float32, exchange=os.environ.get("GSPB200_EXCHANGE"))
    op.fuse_halo = os.environ.get("GSPB200_FUSE_HALO", "1") != "0"
    return op, op.estimate_lmax(), int(L_rows.nnz)


def build_partitioned_strips(gsp, wl, rank, world, torch, dist):
    """Weak scaling: strip q = rank q's 1e6-vertex row block of ONE k-NN graph on
    [0, P) x [0, 1); halo exchange per recurrence step."""
    from pygsp_b200 import distributed as gd
    from pygsp_b200.graphs.generators import SensorStrips, laplacian_rows
    gen = SensorStrips(rank, world, wl["N"], k=wl["k"], seed=wl["seed"])
    tot = torch.tensor(gen.distance_sum(), dtype=torch.float64, device="cuda")
    dist.all_reduce(tot)
    sigma = float(tot[0] / tot[1])
    L_rows, dw = laplacian_rows(gen.adjacency_rows(sigma), rank * wl["N"])
    plan = gd.HaloPlan(L_rows, gd.even_bounds(world * wl["N"], world), rank)
    ov = os.environ.get("GSPB200_OVERLAP")          # default: decided from the halo size
    op = gd.PartitionedCheby(plan, dtype=torch.float32, overlap=None if ov is None else ov != "0",
                             exchange=os.environ.get("GSPB200_EXCHANGE"))   # default: p2p
    op.fuse_halo = os.environ.get("GSPB200_FUSE_HALO", "1") != "0"
    return op, op.estimate_lmax(), int(L_rows.nnz)       # distributed Lanczos, as on one GPU


def build_partitioned_knn_slabs(gsp, wl, rank, world, torch, dist):
    """BASELINE configs[4] (and its smaller instances): rank q generates slab q of ONE k-NN
    graph of N uniform points in the unit cube on its GPU (graphs.KnnSlabs: grid-hash k-NN,
    NNGraph's Gaussian weights and 'average' symmetrisation, Morton numbering inside the slab),
    assembles its rows of L in HBM and plans its halo on the device."""
    from pygsp_b200 import distributed as gd
    from pygsp_b200.graphs.generators import KnnSlabs
    n_per = wl["N"] // world
    gen = KnnSlabs(rank, world, n_per, dim=3 if wl["graph"] == "knn3d" else 2, k=wl["k"],
                   seed=wl["seed"])
    tot = torch.tensor(gen.distance_sum(), dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tot)
    sigma = float(tot[0] / tot[1])
    ptr, idx, val, _ = gen.laplacian_rows_device(sigma)
    del gen
    torch.cuda.empty_cache()
    plan = gd.HaloPlan.from_device(ptr, idx, val, gd.even_bounds(n_per * world, world), rank)
    del ptr, idx, val
    torch.cuda.empty_cache()
    op = gd.PartitionedCheby(plan, dtype=torch.float32, exchange=os.environ.get("GSPB200_EXCHANGE"))
    op.fuse_halo = os.environ.get("GSPB200_FUSE_HALO", "1") != "0"
    return op, op.estimate_lmax(), int(plan.nnz)


def build_partitioned_from_graph(G, rank, world, torch):
    """Strong scaling: every rank holds the SAME graph (built through the Graph API with the
    same seed, exactly the one-GPU graph) and keeps the row block [N p/P, N (p+1)/P) of its
    Laplacian for the partitioned operator; the full copy stays for the in-run parity leg."""
    from pygsp_b200 import distributed as gd
    bounds = gd.even_bounds(G.N, world)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    ptr = G.L.indptr[lo:hi + 1]
    a, b = int(ptr[0].item()), int(ptr[-1].item())
    plan = gd.HaloPlan.from_device(ptr - a, G.L.indices[a:b], G.L.data[a:b], bounds, rank)
    op = gd.PartitionedCheby(plan, dtype=torch.float32, exchange=os.environ.get("GSPB200_EXCHANGE"))
    op.fuse_halo = os.environ.get("GSPB200_FUSE_HALO", "1") != "0"
    return op, (lo, hi)


def run_ours(args):
    import ctypes
    import torch
    import torch.distributed as dist
    import pygsp_b200 as gsp
    from pygsp_b200.filters import approximations as apx

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    numa_cpus = gsp.utils.bind_to_gpu_numa(local)      # pinned staging memory on the GPU's socket
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    name, wl, scaling = pick_workload(args, world)
    nsig, order = wl["nsig"], wl["order"]
    if world > 1 and name == "config3":
        raise SystemExit("--workload config3 is a single-GPU option")
    lib = gsp._native.lib()
    lib.gsp_launch_count.restype = ctypes.c_uint64
    peak, peak_src = measured_peak()

    clocks = ClockSampler(local)
    clocks.__enter__()                       # running long before the timed region

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(v):
        t = torch.tensor([v], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- build the workload (untimed)
    G = op = None
    lo = 0
    t_build0 = time.perf_counter()
    if wl["graph"] != "knn3d" and (world == 1 or (scaling == "strong"
                                                  and wl["graph"] in ("sensor", "grid2d"))):
        G = build_graph(gsp, wl)                     # the one-GPU graph, on every rank
        n_global = wl["N"] = G.N
        lmax, nnz_global = G.lmax, G.L.nnz
        bank, c = make_bank(gsp, G, wl)
        if world > 1:
            op, (lo, hi) = build_partitioned_from_graph(G, rank, world, torch)
            n, nnz = hi - lo, int(op.plan.nnz)
        else:
            n, nnz = G.N, G.L.nnz
    else:
        if wl["graph"] == "sbm":
            op, lmax, nnz = build_partitioned_sbm(gsp, wl, rank, world, torch, dist)
        elif wl["graph"] == "knn3d":
            op, lmax, nnz = build_partitioned_knn_slabs(gsp, wl, rank, world, torch, dist)
        else:
            op, lmax, nnz = build_partitioned_strips(gsp, wl, rank, world, torch, dist)
        n = op.plan.n_local
        n_global = op.plan.n_global
        lo = int(op.plan.bounds[rank])

        class _G:           # coefficients need only lmax (approximations.py:40)
            pass
        g = _G(); g.lmax = lmax; g.N = n
        bank = gsp.filters.Heat(g, scale=wl["scale"])
        c = np.atleast_2d(gsp.filters.compute_cheby_coeff(bank, m=order))
        t = torch.tensor([nnz], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t)
        nnz_global = int(t.item())
    t_build = time.perf_counter() - t_build0
    clen = c.shape[0] == 1                           # the engine's default form for one filter
    if op is not None and world > 1:                 # (the packed-NCCL exchange keeps the forward form)
        clen = clen and op._exchange_mode(nsig) == "p2p" and \
            os.environ.get("GSPB200_BENCH_CLENSHAW") != "0"
    # signals: one seeded global block, every rank takes its rows (strong scaling keeps the
    # whole block for the parity leg against the one-GPU engine)
    gen = torch.Generator(device="cuda").manual_seed(0 if G is not None else rank)
    x_full = torch.randn(n_global if G is not None else n, nsig, device="cuda", generator=gen)
    x = x_full[lo:lo + n].contiguous() if (G is not None and world > 1) else x_full
    if world == 1 and G is not None:
        run_dev = device_op(apx, G.L, lmax, c)
        run_host = lambda xh: bank.filter(xh, order=order)
    else:
        local_order = os.environ.get("GSPB200_BENCH_LOCAL_ORDER") == "1"    # diagnosis only
        form = {"0": False, "1": True}.get(os.environ.get("GSPB200_BENCH_CLENSHAW"))   # diagnosis
        run_dev = lambda xx: op.cheby_op(lmax, c, xx, local_order=local_order, clenshaw=form)
        run_host = lambda xh: op.filter_pinned(lmax, c, xh)[0]

    # ---- device-resident throughput ("value")
    warm = max(args.warmup, 3)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(warm):
        run_dev(x)
    barrier()
    launches0 = lib.gsp_launch_count()
    t_region0 = time.time()
    start.record()
    for _ in range(args.steps):
        y_dev = run_dev(x)
    stop.record()
    barrier()
    t_region1 = time.time()
    launches = int(lib.gsp_launch_count() - launches0)
    time.sleep(0.1)                                      # let the sampler emit its last lines
    clocks.__exit__()
    t_dev = allmax(start.elapsed_time(stop) / 1e3)
    value = n_global * nsig * order * args.steps / t_dev
    if args.dump_outputs:
        dump_output(torch, args.dump_outputs, "y" if world == 1 else "y_rank%d" % rank, y_dev,
                    DUMP_BYTES // world)

    # ---- end to end through the public API with host buffers
    e2e = None
    if not args.no_e2e and wl["nscales"] == 1 and n * nsig * 4 <= (4 << 30):
        xh = torch.empty((n, nsig), dtype=torch.float32).pin_memory()
        xh.copy_(x)
        for _ in range(2):
            yh = run_host(xh)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            yh = run_host(xh)                 # returns a complete host tensor (synchronises)
        torch.cuda.synchronize()
        t_e2e = allmax(time.perf_counter() - t0)
        assert tuple(yh.shape)[:2] == (n, nsig) and not yh.is_cuda
        e2e_err = float((yh.to("cuda") - y_dev[0]).abs().max() / y_dev[0].abs().max())
        from pygsp_b200.filters import pipeline
        chunks = pipeline.chunk_plan(n_global // world, nsig, 4)
        e2e = {"value": n_global * nsig * order * args.steps / t_e2e, "unit": UNIT,
               "h2d_bytes_per_step": 4 * n_global * nsig,
               "d2h_bytes_per_step": 4 * n_global * nsig * wl["nscales"],
               "ms_per_step": 1e3 * t_e2e / args.steps,
               "api": ("%s.filter(pinned_host_tensor, order=%d)" % (
                   "Heat(G, 50)", order)) if world == 1 else
                      "PartitionedCheby.filter_pinned(pinned host block of the rank's rows)",
               "pipeline": "column chunks of %s signals: upload j+1 / recurrence j / download j-1 "
                           "on three streams (strided 2-D copies by %s)" % (
                               " | ".join(str(w) for _, w in chunks),
                               "a zero-copy kernel" if os.environ.get("GSPB200_STAGE") == "kernel"
                               else "the copy engines"),
               "max_abs_diff_vs_device_path_rel": e2e_err, "numa_cpus_bound": numa_cpus}
        del xh, yh

    # ---- parity legs
    parity = {}
    if world > 1 and G is not None:
        # every rank owns the whole graph: the partitioned result must equal the one-GPU
        # engine's on the rank's rows (same kernels, same summation order: expected 0.0)
        single = device_op(apx, G.L, lmax, c)
        full = single(x_full)
        mine = op.cheby_op(lmax, c, x, local_order=False)
        err = float((mine - full[:, lo:lo + n]).abs().max() / full.abs().max())
        parity["parity_rel_err"] = allmax(err)
        parity["parity_bit_identical_on_every_rank"] = allmax(0.0 if torch.equal(
            mine, full[:, lo:lo + n]) else 1.0) == 0.0
        t_single = allmax(time_calls(torch, single, x_full, 3, 1))
        parity["one_gpu_same_graph_ms_per_step"] = t_single
        parity["speedup_vs_one_gpu_same_run"] = t_single / (1e3 * t_dev / args.steps)
        del full, mine
        if rank == 0:        # and the engine itself against the float64 oracle on one column
            col = x_full[:, :1].contiguous()
            parity["parity_rel_err_one_column_vs_oracle"] = oracle_parity(G.L, lmax, c, col, single(col))
    elif op is not None:
        # No rank holds the whole graph.  Two size-independent checks on every rank:
        # (1) L 1 = 0, so filtering the constant signal must return p(0) = c_0/2 + sum_k (-1)^k c_k
        #     on every vertex -- a stale or missing halo row breaks it at the boundary rows;
        # (2) the packed NCCL exchange and the fused peer-store exchange are different transports
        #     around the same kernels: their results on 8 signals must agree bit for bit.
        k_idx = np.arange(c.shape[1])
        p0 = float(0.5 * c[0, 0] + (c[0, 1:] * (-1.0) ** k_idx[1:]).sum())
        ones = torch.ones(n, 8, device="cuda")
        got = op.cheby_op(lmax, c, ones)
        parity["parity_constant_signal_rel_err"] = allmax(float((got - p0).abs().max() / abs(p0)))
        if world > 1:
            from pygsp_b200 import distributed as gd
            other = "nccl" if op._exchange_mode(8) == "p2p" else "p2p"
            op_b = gd.PartitionedCheby(op.plan, dtype=torch.float32, exchange=other)
            xs = x[:, :8].contiguous()
            a8 = op.cheby_op(lmax, c, xs, clenshaw=False)
            b8 = op_b.cheby_op(lmax, c, xs, clenshaw=False)
            parity["parity_exchange_transports_bit_identical"] = allmax(
                0.0 if torch.equal(a8, b8) else 1.0) == 0.0
            parity["parity_rel_err"] = allmax(float((a8 - b8).abs().max() / a8.abs().max()))
            del op_b, a8, b8
        else:
            parity["parity_rel_err"] = parity["parity_constant_signal_rel_err"]
        parity["parity_note"] = ("no rank holds the whole graph for this workload: constant-signal "
                                 "property + transport cross-check here; oracle parity of the same "
                                 "generator and operator at test size in tests/test_distributed_gpu.py")
        del got, ones

    if rank != 0:
        dist.barrier()
        dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (one fused step), per GPU
    b_first, b_step, b_call = algorithmic_bytes(n, nnz, nsig, wl["nscales"], order, clenshaw=clen)
    _, _, b_call_ref = algorithmic_bytes(n, nnz, nsig, wl["nscales"], order, clenshaw=False)
    achieved = b_call * args.steps / t_dev / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": ncu_traffic(name if world == 1 else None),
                "per_gpu": True,
                "kernel": "cheby_step_tiled (TMA-tiled fused step, csrc/cheby_tiled.cu)",
                "form": ("clenshaw: 4 passes over the signal block per step" if clen else
                         "forward: 3 + 2 Nscales passes per step"),
                "peak_source": peak_src, "algorithmic_bytes_per_launch": b_step,
                "algorithmic_bytes_per_call": b_call,
                "avg_launch_ms": 1e3 * t_dev / args.steps * (b_step / b_call),
                "frac_if_counted_with_the_reference_algorithm_bytes":
                    b_call_ref * args.steps / t_dev / 1e9 / peak,
                "timing": "CUDA events on the launching stream over the timed region, max over ranks"}
    # SURVEY.md 8(d): for a graph without locality the x_cur term of the algorithmic bytes
    # (each row once) is unattainable; the gather-aware figure charges every stored entry
    # one neighbour-row read of max(32, 4*nsig) bytes instead (no reuse at all).
    gather = nnz * max(32, 4 * nsig) - 4 * n * nsig
    roofline["gather_aware"] = {"bytes_per_launch": b_step + gather,
                                "frac_if_no_gather_reuse": (b_call + order * gather) * args.steps
                                / t_dev / 1e9 / peak}
    halo = None
    if world > 1:
        halo_bytes = op.plan.n_halo * nsig * 4
        halo = {"rows_received_per_rank": op.plan.n_halo, "boundary_rows": op.plan.n_true_boundary,
                "bytes_received_per_rank_per_step": halo_bytes,
                "nvlink_GBps_per_rank_if_serialised": halo_bytes * order * args.steps / t_dev / 1e9,
                "exchange": op._exchange_mode(nsig) + (
                    ": peer stores over NVLink into the neighbours' halo rows from the step "
                    "kernel's epilogue + flags (csrc/dist.cu, csrc/cheby_tiled.cu)"
                    if op._exchange_mode(nsig) == "p2p" else
                    ": pack + NCCL all_to_all_single, overlapped with the interior rows")}

    # ---- CPU baseline (the reference's scipy path) on a bounded sample, rank 0, one GPU
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        from oracle import pygsp_oracle as orc
        cols = args.cpu_columns
        xs = x[:, :cols].double().cpu().numpy()
        if wl["bank"] == "heat":
            cref = CpuReference(G.W.to_scipy().astype(np.float64), lmax, wl["scale"], order, xs, 1)
            t_cpu, cpu_kind = cref.time_once(), cref.kind
        else:                                   # banks: time the oracle port of cheby_op
            t0 = time.perf_counter()
            orc.cheby_op(G.L.to_scipy().astype(np.float64), lmax, c, xs)
            t_cpu, cpu_kind = time.perf_counter() - t0, "port"
        col = x[:, :1].contiguous()
        cpu = {"value": n * cols * order / t_cpu, "unit": UNIT, "cores": 1, "kind": cpu_kind,
               "host_cores_available": os.cpu_count(),
               "sample": "%d of %d signal columns, full graph, full order, float64; %s" % (
                   cols, nsig, "unmodified PyGSP 0.6.1 (baseline/_ref) g.filter()"
                   if cpu_kind == "reference" else "oracle port (scipy csr_matvecs + numpy)"),
               "parity_rel_err_vs_gpu": oracle_parity(G.L, lmax, c, col, run_dev(col))}

    # ---- the other BASELINE workloads that fit one GPU, short runs in the same line
    targets = None
    if world == 1 and name == "config2" and not args.no_targets:
        del x_full, x, y_dev
        torch.cuda.empty_cache()
        targets = {}
        for tname in ("knn10m", "config3"):
            try:
                targets[tname] = run_target(gsp, apx, torch, tname, peak)
            except Exception as exc:                    # a failed side run must not lose the line
                targets[tname] = {"error": repr(exc)[:300]}

    # Lanczos timing on the workload's graph (estimate_lmax is part of the path)
    lanczos = None
    if G is not None and world == 1:
        G._lmax_method = None
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        G.estimate_lmax()
        torch.cuda.synchronize()
        lanczos = {"estimate_lmax_ms": 1e3 * (time.perf_counter() - t0),
                   "spmv_products": G._lanczos_steps, "lmax": G.lmax}

    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
           "warmup": warm, "ms_per_step": 1e3 * t_dev / args.steps,
           "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
           "dtype": "f32", "data": "synthetic", "config": config_dict(wl, world, scaling),
           "graph": {"nnz_L_global": int(nnz_global), "lmax": lmax, "build_s": t_build},
           "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
           "halo": halo, "targets": targets, "estimate_lmax": lanczos,
           "clocks": clocks.summary(t_region0, t_region1)}
    out.update(parity)
    print(json.dumps(out))
    sys.stdout.flush()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if out.get("parity_rel_err") is not None and out["parity_rel_err"] > 1e-5:
        raise SystemExit("parity check failed: %r" % out["parity_rel_err"])


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
