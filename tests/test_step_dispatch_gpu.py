"""The entry points that share the host step dispatcher, on one GPU, bit for bit.

A. gsp_cheby_step_halo_f32 with a halo that has no neighbours (nothing to wait for, nothing to
   push): its front ("boundary") launch, interior launch and row-group remainder give the bits
   of gsp_cheby_step_f32 and of the exact host oracle for every split of the rows, and the call
   needs a tile plan.
B. gsp_cheby_op_dist_* on a one-rank process group (peer-memory exchange with no peers): the
   forward and Clenshaw recurrences of the partitioned operator give the single-GPU engine's
   bits, with and without the row permutation, fused or separate exchange, tiled or row-group
   widths, float32 and float64.
"""
import ctypes

import numpy as np
import pytest
from scipy import sparse

from oracle import build_oracle
from oracle import pygsp_oracle as orc

pytestmark = pytest.mark.gpu

NSIG = 64
NSCALES = 2


@pytest.fixture(scope="module")
def gsp():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import pygsp_b200
    return pygsp_b200


@pytest.fixture(autouse=True)
def _clean_env(monkeypatch):
    for k in ("GSPB200_KERNEL", "GSPB200_FORCE_HALO", "GSPB200_TILE_R", "GSPB200_TILE_S",
              "GSPB200_TILE_VDIR", "GSPB200_TILE_P2", "GSPB200_TILE_REV"):
        monkeypatch.delenv(k, raising=False)


def _bits(t):
    a = t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)
    return a.view(np.int32 if a.dtype == np.float32 else np.int64)


def _assert_same_bits(got, want, what):
    g, w = _bits(got), _bits(want)
    assert g.shape == w.shape, (what, g.shape, w.shape)
    bad = np.flatnonzero(g.reshape(-1) != w.reshape(-1))
    assert bad.size == 0, "%s: %d elements differ, first at flat index %d" % (what, bad.size, bad[0])


# ------------------------------------------------------------ A: gsp_cheby_step_halo_f32
@pytest.fixture(scope="module")
def mat(gsp):
    """n = 1000: full tiles and a row-group remainder for the 64-signal, 2-filter plan."""
    import torch
    W = sparse.random(1000, 1000, 0.01, random_state=7, format="csr")
    W = W + W.T
    W.setdiag(0)
    W.eliminate_zeros()
    L = sparse.csr_matrix(orc.laplacian(W))
    L.sort_indices()
    D = gsp.graphs.DeviceCSR.from_scipy(L, torch.float32, torch.device("cuda"))
    plan = D.tile_plan(NSIG, NSCALES)
    assert plan is not None and L.shape[0] % plan.rows_per_tile != 0
    return L, D, plan


def _halo_step(nat, D, first, x_cur, x_old, x_new, r, ck, c0, coef, reverse, plan, halo):
    fn = nat.lib().gsp_cheby_step_halo_f32
    fn.restype = ctypes.c_int
    args = [nat.i32(int(first)), nat.i64(D.shape[0]), nat.i64(D.nnz), D.indptr, D.indices, D.data,
            x_cur, x_old, x_new, r, nat.i64(D.shape[0]), nat.i64(NSIG), nat.i32(NSCALES), ck, c0,
            nat.f64(coef[0]), nat.f64(coef[1]), nat.f64(coef[2]), nat.i32(int(reverse)), plan,
            halo, nat.stream_ptr()]
    return fn(*[nat._arg(a) for a in args])


@pytest.mark.parametrize("first", [True, False])
@pytest.mark.parametrize("publish", [0, 1])
@pytest.mark.parametrize("boundary", ["none", "part_tile", "one_tile", "ragged"])
def test_halo_step_without_neighbours_matches_plain_step(gsp, mat, first, publish, boundary):
    import torch
    nat = gsp._native
    L, D, plan = mat
    n, R = L.shape[0], plan.rows_per_tile
    n_boundary = {"none": 0, "part_tile": R // 2 + 1, "one_tile": R, "ragged": 2 * R + 7}[boundary]
    assert n_boundary <= (n // R) * R
    rng = np.random.default_rng(100 * first + 10 * publish + len(boundary))
    x_cur = rng.standard_normal((n, NSIG)).astype(np.float32)
    x_old = None if first else rng.standard_normal((n, NSIG)).astype(np.float32)
    r0 = rng.standard_normal((NSCALES, n, NSIG)).astype(np.float32)
    ck, c0 = rng.standard_normal(NSCALES), rng.standard_normal(NSCALES)
    coef = (float(rng.uniform(0.2, 1.0)), float(rng.standard_normal()), float(rng.standard_normal()))

    h_new, h_r = np.zeros((n, NSIG), np.float32), r0.copy()
    build_oracle.cheby_step_exact(first, 0, n, L.indptr, L.indices, L.data.astype(np.float32),
                                  x_cur, x_old, h_new, h_r, n, NSCALES, ck, c0, *coef)

    dev = lambda a: None if a is None else torch.from_numpy(a).cuda()
    d_cur, d_old = dev(x_cur), dev(x_old)
    p_new, p_r = torch.zeros(n, NSIG, device="cuda"), dev(r0)
    nat.call("gsp_cheby_step_f32", nat.i32(int(first)), nat.i64(0), nat.i64(n), nat.i64(D.nnz),
             D.indptr, D.indices, D.data, d_cur, d_old, p_new, p_r, nat.i64(n), nat.i64(NSIG),
             nat.i32(NSCALES), ck, c0, nat.f64(coef[0]), nat.f64(coef[1]), nat.f64(coef[2]), plan,
             nat.stream_ptr())

    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    halo = nat.HaloFusion()
    halo.push_counter = counter.data_ptr()
    halo.n_boundary_rows = n_boundary
    halo.n_owned = n
    halo.publish = publish
    halo.publish_value = 5
    f_new, f_r = torch.zeros(n, NSIG, device="cuda"), dev(r0)
    rc = _halo_step(nat, D, first, d_cur, d_old, f_new, f_r, ck, c0, coef, not first, plan, halo)
    assert rc == 0, nat.lib().gsp_last_error()
    torch.cuda.synchronize()

    what = "first=%d publish=%d boundary=%d" % (first, publish, n_boundary)
    _assert_same_bits(p_new, h_new, what + " plain x_new")
    _assert_same_bits(p_r, h_r, what + " plain r")
    _assert_same_bits(f_new, h_new, what + " halo x_new")
    _assert_same_bits(f_r, h_r, what + " halo r")
    assert int(counter.item()) == 0          # the last front warp re-arms the counter


def test_halo_step_needs_a_tile_plan(gsp, mat):
    import torch
    nat = gsp._native
    L, D, plan = mat
    n = L.shape[0]
    x = torch.zeros(n, NSIG, device="cuda")
    r = torch.zeros(NSCALES, n, NSIG, device="cuda")
    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    halo = nat.HaloFusion()
    halo.push_counter = counter.data_ptr()
    halo.n_owned = n
    ck = np.ones(NSCALES)
    rc = _halo_step(nat, D, True, x, None, x.clone(), r, ck, ck, (1.0, 0.0, 0.0), False, None, halo)
    assert rc == -3


# ------------------------------------------------------ B: gsp_cheby_op_dist_* on one rank
@pytest.fixture(scope="module")
def one_rank(gsp, tmp_path_factory):
    import torch
    import torch.distributed as dist
    from pygsp_b200 import distributed as gd
    init = tmp_path_factory.mktemp("pg") / "init"
    dist.init_process_group("gloo", init_method="file://%s" % init, world_size=1, rank=0)
    G = gsp.graphs.Sensor(6000, k=8, seed=5, order="morton")
    G.estimate_lmax()
    L = G.L.to_scipy()
    plan = gd.HaloPlan(L, gd.even_bounds(G.N, 1), 0)
    dev = torch.device("cuda")
    ops = {dt: gd.PartitionedCheby(plan, dtype=dt, exchange="p2p")
           for dt in (torch.float32, torch.float64)}
    mats = {dt: gsp.graphs.DeviceCSR.from_scipy(L, dt, dev) for dt in ops}
    yield G.lmax, plan, ops, mats
    for op in ops.values():
        for win in op._windows.values():
            win.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("nsig", [64, 3])
@pytest.mark.parametrize("fuse_halo", [True, False])
@pytest.mark.parametrize("local_order", [False, True])
@pytest.mark.parametrize("clenshaw", [False, True])
def test_partitioned_one_rank_matches_single_gpu(gsp, one_rank, clenshaw, local_order, fuse_halo,
                                                 nsig, dtype):
    import torch
    from pygsp_b200.filters import approximations as apx
    lmax, plan, ops, mats = one_rank
    dt = getattr(torch, dtype)
    op, D = ops[dt], mats[dt]
    op.fuse_halo = fuse_halo
    rng = np.random.default_rng(nsig + 2 * clenshaw)
    c = rng.standard_normal((1 if clenshaw else 2, 13)) / np.arange(1, 14)
    x = torch.from_numpy(rng.standard_normal((plan.n_local, nsig))).to(device="cuda", dtype=dt)
    if clenshaw:
        want = apx.cheby_clenshaw_device(D, lmax, c, x)[None]
    else:
        want = apx.cheby_op_device(D, lmax, c, x)
    if dtype == "float32" and nsig == 64:
        assert D.tile_plan(nsig, c.shape[0]) is not None
    if local_order:
        perm = torch.from_numpy(plan.perm).cuda()
        got = op.cheby_op(lmax, c, x[perm].contiguous(), local_order=True, clenshaw=clenshaw)
        want = want[:, perm]
    else:
        got = op.cheby_op(lmax, c, x, clenshaw=clenshaw)
    torch.cuda.synchronize()
    assert got.dtype == dt and torch.equal(got, want)
