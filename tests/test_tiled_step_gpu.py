"""Bit-exact tests of the Chebyshev step kernels (csrc/cheby.cu row-group kernel, csrc/cheby_tiled.cu
TMA-tiled kernel), at the sizes and edges where the tiled kernel's machinery runs:

  * a ring-wrap graph, sized from the SM count and the actual tile plans so that every persistent
    CTA walks at least 2 * stages + 1 tiles: every ring stage is reused, both barrier parities are
    seen, the one-tile-ahead CSR offset prefetch runs;
  * edge matrices E1..E5 (trailing CSR entries loaded by hand, zero-byte CSR slabs, every row
    start / row length residue mod 4, a hub row that forces a 2-stage ring with one CTA per SM,
    matrices with no / one / a partial tile).

A. gsp_cheby_step_* against the exact host restatement of the ABI (oracle/cheby_oracle.c,
   cheby_step_exact_*) at zero tolerance: the kernels round every fma once, in stored CSR order.
B. Whole calls (forward recurrence, Clenshaw form, fused synthesis): the tiled kernel gives the
   row-group kernel's bits under every tiling setting.
C. The row-group result against the float64 oracle (tolerance), the float64 engine at 1e-10.

Every test asserts the coverage condition it exists for, so that a change of the plan
(rows per tile, stages, grid) fails loudly instead of quietly shrinking what is tested.
"""
import ctypes
import zlib

import numpy as np
import pytest
from scipy import sparse

from conftest import relerr_cols
from oracle import build_oracle
from oracle import pygsp_oracle as orc

pytestmark = pytest.mark.gpu

F32_TOL = 1e-5
F64_TOL = 1e-10
TILED_WIDTHS = (8, 16, 32, 64, 128)
STEP_WIDTHS = (1, 3, 8, 16, 32, 64, 128, 132)
STEP_SCALES = (0, 1, 2, 3, 16, 17, 33)          # 17 / 33: the cheby_axpy_scales path
ORDERS = (1, 2, 3, 12)
MAX_CTAS_PER_SM = 3                              # launch bounds of the two-packet mapping
SMEM_PER_SM = 228 * 1024
ENV_KEYS = ("GSPB200_KERNEL", "GSPB200_FORCE_HALO") + tuple(
    "GSPB200_TILE_" + k for k in ("R", "S", "NW", "SMEM", "VDIR", "P2", "REV", "HINT", "BPS", "U"))

# whole-call cases: (form, nsig, filters / sources)
WHOLE_CASES = [("forward", w, 1) for w in TILED_WIDTHS] + \
              [("forward", 64, 2), ("forward", 32, 3), ("forward", 128, 3)] + \
              [("clenshaw", w, 1) for w in TILED_WIDTHS] + \
              [("synthesis", 64, 2), ("synthesis", 32, 5), ("synthesis", 32, 16)]
# tiling settings on top of the defaults (read when the plan is made / at launch)
SETTINGS = {
    "p2=0,vdir=0": {"GSPB200_TILE_P2": "0", "GSPB200_TILE_VDIR": "0"},
    "p2=0,vdir=1": {"GSPB200_TILE_P2": "0", "GSPB200_TILE_VDIR": "1"},
    "p2=1,vdir=0": {"GSPB200_TILE_P2": "1", "GSPB200_TILE_VDIR": "0"},
    "p2=1,vdir=1": {"GSPB200_TILE_P2": "1", "GSPB200_TILE_VDIR": "1"},
    "rev=0": {"GSPB200_TILE_REV": "0"},
    "hint=0": {"GSPB200_TILE_HINT": "0"},
    "s=2": {"GSPB200_TILE_S": "2"},
    "s=3": {"GSPB200_TILE_S": "3"},
    "s=4": {"GSPB200_TILE_S": "4"},
    "nw=1": {"GSPB200_TILE_NW": "1"},
    "nw=5": {"GSPB200_TILE_NW": "5"},
    "bps=1,r=8": {"GSPB200_TILE_BPS": "1", "GSPB200_TILE_R": "8"},
    "force_halo": {"GSPB200_FORCE_HALO": "1"},
}


def _ring_env(nsig, env):
    """Widths 8 / 16 have 128 / 256-row tiles: one CTA per SM makes each CTA wrap the ring on a
    graph that the other widths need anyway (the host oracle stays affordable)."""
    env = dict(env)
    if nsig <= 16:
        env.setdefault("GSPB200_TILE_BPS", "1")
    return env


# ---------------------------------------------------------------------------- helpers
@pytest.fixture(scope="module")
def gsp():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import pygsp_b200
    return pygsp_b200


@pytest.fixture(autouse=True)
def _clean_env(monkeypatch):
    for k in ENV_KEYS:
        monkeypatch.delenv(k, raising=False)


def _set_env(mp, env):
    for k in ENV_KEYS:
        mp.delenv(k, raising=False)
    for k, v in env.items():
        mp.setenv(k, v)


def _sm_count(nat):
    sm, ma, mi, l2 = ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_int64()
    nat.call("gsp_device_info", ctypes.byref(sm), ctypes.byref(ma), ctypes.byref(mi), ctypes.byref(l2))
    return sm.value


def _plan(nat, D, nsig, nscales):
    """A fresh tile plan under the current environment (None: row-group kernel)."""
    plan = nat.TilePlan()
    nat.call("gsp_cheby_tile_plan", nat.i64(D.shape[0]), D.indptr, nat.i64(nsig), nat.i32(nscales),
             plan, nat.stream_ptr())
    return plan if plan.rows_per_tile > 0 else None


def _default_R(nsig, nscales):
    """Rows per tile of the default plan (cheby_tiled.cu tile_plan); checked against real plans."""
    R = 64 if nscales <= 1 else (32 if nscales <= 2 else 16)
    if nsig == 128:
        R = max(8, R // 2)
    if nsig <= 16:
        R = max(R, 16 * (128 // nsig))
    return R


def _smem_total(plan, nsig, nscales, vec_staged):
    """Dynamic shared memory of one CTA (TileLayout in cheby_tiled.cu)."""
    R, cap, S = plan.rows_per_tile, plan.slab_capacity, plan.stages
    vec = (1 + nscales) * R * nsig * 4 if vec_staged else 0
    stage = vec + 2 * (cap + 16) * 4 + (R + 4) * 4 + 16
    return ((2 * S * 8 + 15) // 16) * 16 + S * stage


def _assert_ring_wraps(plan, n, sm):
    """Every CTA of the persistent grid walks >= 2 * stages + 1 tiles (grid <= sm x CTAs/SM)."""
    assert plan is not None, "tiled plan expected"
    per_sm = plan.blocks_per_sm if plan.blocks_per_sm > 0 else MAX_CTAS_PER_SM
    n_tiles = n // plan.rows_per_tile
    need = (2 * plan.stages + 1) * sm * per_sm
    assert n_tiles >= need, (n_tiles, need, plan.as_dict())


def _bits(a):
    a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
    return a.view(np.int32 if a.dtype == np.float32 else np.int64)


def _assert_same_bits(got, want, what):
    g, w = _bits(got), _bits(want)
    assert g.shape == w.shape, (what, g.shape, w.shape)
    bad = np.flatnonzero(g.reshape(-1) != w.reshape(-1))
    assert bad.size == 0, "%s: %d elements differ, first at flat index %d" % (what, bad.size, bad[0])


class Mat:
    """One test matrix: scipy CSR (float64 values), device copies in float32 and float64, and
    the float32 values the float32 engine actually uses."""

    def __init__(self, gsp, name, L, lmax=None):
        import torch
        L = sparse.csr_matrix(L)
        L.sort_indices()
        self.name, self.L, self.n = name, L, L.shape[0]
        self.indptr = np.ascontiguousarray(L.indptr, dtype=np.int32)
        self.indices = np.ascontiguousarray(L.indices, dtype=np.int32)
        self.data64 = np.ascontiguousarray(L.data, dtype=np.float64)
        self.data32 = self.data64.astype(np.float32)
        dev = torch.device("cuda")
        self.D32 = gsp.graphs.DeviceCSR.from_scipy(L, torch.float32, dev)
        self.D64 = gsp.graphs.DeviceCSR.from_scipy(L, torch.float64, dev)
        self.lmax = lmax if lmax is not None else 1.01 * orc.lambda_max_exact(L)

    def D(self, dtype):
        return self.D32 if dtype == np.float32 else self.D64

    def data(self, dtype):
        return self.data32 if dtype == np.float32 else self.data64


def _laplacian(n, density, seed, isolated=()):
    W = sparse.random(n, n, density, random_state=seed, format="coo")
    iso = np.zeros(n, dtype=bool)
    iso[list(isolated)] = True
    keep = ~(iso[W.row] | iso[W.col])
    W = sparse.csr_matrix((W.data[keep], (W.row[keep], W.col[keep])), shape=(n, n))
    W = W + W.T
    W.setdiag(0)
    W.eliminate_zeros()
    return orc.laplacian(W)


def _e1(nnz_mod4, seed):
    """n % 256 == 0 (so n % R == 0 for every R), last row non-empty, nnz % 4 == nnz_mod4: the
    last full tile ends at nnz and its last <= 3 CSR entries are loaded by hand."""
    n = 512
    iso = []
    L = _laplacian(n, 0.01, seed)
    v = 1
    while L.nnz % 4 != nnz_mod4:             # isolating a vertex removes 2 deg + 1 entries
        iso.append(v)
        v += 1
        L = _laplacian(n, 0.01, seed, iso)
        assert v < 64
    return L


def _e2(seed):
    """>= 2 x 256 consecutive empty rows starting at a row whose indptr is a multiple of 4:
    tiles of empty rows with an aligned start have a zero-byte CSR slab."""
    n, run = 2048, 640
    for s in range(600, 700):
        L = _laplacian(n, 0.004, seed, range(s, s + run))
        if L.indptr[s] % 4 == 0:
            return L
    raise AssertionError("no aligned start found")


def _e3(seed):
    """Row lengths cycling through 0..9: every (row start mod 4, row length mod 4) pair.  Not a
    Laplacian (a step does not care); lmax = 2 x the largest absolute row sum, which bounds the
    spectral radius, so that whole calls stay finite."""
    rng = np.random.default_rng(seed)
    n = 1280
    rows, cols, vals = [], [], []
    for i in range(n):
        k = i % 10
        c = np.sort(rng.choice(n, size=k, replace=False))
        v = -rng.uniform(0.1, 1.0, k)
        if i in c:
            v[np.searchsorted(c, i)] = 0.0
            v[np.searchsorted(c, i)] = -v.sum() + 0.5
        rows += [i] * k
        cols += list(c)
        vals += list(v)
    M = sparse.csr_matrix((vals, (rows, cols)), shape=(n, n))
    M.sort_indices()
    lens = np.diff(M.indptr)
    assert (lens == np.arange(n) % 10).all()
    starts = M.indptr[:-1] % 4
    assert len({(int(s), int(ln) % 4) for s, ln in zip(starts, lens)}) == 16
    return M, 2.0 * float(abs(M).sum(axis=1).max())


def _e4(seed):
    """A hub row of 7000 entries: the slab capacity makes the 3-stage ring of a 3-filter bank
    exceed its budget, the plan drops to 2 stages, and one CTA fits per SM (< 200 KB)."""
    rng = np.random.default_rng(seed)
    n, hub = 8192, 4101
    W = sparse.random(n, n, 6.0 / n, random_state=seed, format="lil")
    nb = rng.choice(np.setdiff1d(np.arange(n), [hub]), size=7000, replace=False)
    W[hub, nb] = rng.uniform(0.5, 1.5, nb.size)
    W = sparse.csr_matrix(W)
    W = W + W.T
    W.setdiag(0)
    W.eliminate_zeros()
    return orc.laplacian(W)


def _e5(n, seed):
    return _laplacian(n, min(0.5, 6.0 / n), seed)


@pytest.fixture(scope="module")
def emats(gsp):
    mats = {"E1_%d" % m: Mat(gsp, "E1_%d" % m, _e1(m, 20 + m)) for m in (1, 2, 3)}
    mats["E2"] = Mat(gsp, "E2", _e2(31))
    M3, lmax3 = _e3(32)
    mats["E3"] = Mat(gsp, "E3", M3, lmax3)
    mats["E4"] = Mat(gsp, "E4", _e4(33))
    return mats


def _assert_edge_condition(mat, plan, nsig, nscales):
    """The condition each edge matrix exists for, under the plan the kernel runs with."""
    ip = mat.indptr
    n, nnz = mat.n, int(ip[-1])
    if plan is None:
        return
    R = plan.rows_per_tile
    if mat.name.startswith("E1"):
        assert n % R == 0 and ip[-1] > ip[-2] and nnz % 4 in (1, 2, 3)
        end = int(ip[(n // R) * R])
        assert end == nnz and ((end + 3) & ~3) > nnz        # last tile: hand-loaded tail
    elif mat.name == "E2":
        t = np.arange(n // R)
        zero = (ip[t * R] == ip[(t + 1) * R]) & (ip[t * R] % 4 == 0)
        assert zero.any()                                    # a tile with a zero-byte slab
    elif mat.name == "E4":
        assert plan.slab_capacity >= 7000                    # the hub row is inside a tile


def _rand_coefs(rng, nscales):
    ck = rng.standard_normal(max(nscales, 1))
    c0 = rng.standard_normal(max(nscales, 1))
    alpha = float(rng.uniform(0.2, 1.0))
    beta = float(rng.standard_normal())
    gamma = float(rng.standard_normal())
    return ck, c0, alpha, beta, gamma


def _step_gpu(gsp, D, first, rb, re, x_cur, x_old, x_new, r, r_rows, nsig, nscales, ck, c0,
              alpha, beta, gamma, plan):
    nat = gsp._native
    nat.call("gsp_cheby_step_" + nat.suffix(D.dtype), nat.i32(int(first)), nat.i64(rb), nat.i64(re),
             nat.i64(D.nnz), D.indptr, D.indices, D.data, x_cur, x_old, x_new, r, nat.i64(r_rows),
             nat.i64(nsig), nat.i32(nscales), np.ascontiguousarray(ck, dtype=np.float64),
             np.ascontiguousarray(c0, dtype=np.float64), nat.f64(alpha), nat.f64(beta),
             nat.f64(gamma), plan, nat.stream_ptr())


def _check_step(gsp, mat, dtype, nsig, nscales, first, plan, seed, r_pad=0, alias=False,
                split=None):
    """One step on the device (one call, or two calls split at row `split`) against the exact
    host restatement, bit for bit; rows of r past n (r_pad) must be left alone."""
    import torch
    rng = np.random.default_rng(seed)
    n = mat.n
    r_rows = n + r_pad
    x_cur = rng.standard_normal((n, nsig)).astype(dtype)
    x_old = None if first else rng.standard_normal((n, nsig)).astype(dtype)
    r0 = rng.standard_normal((max(nscales, 1), r_rows, nsig)).astype(dtype)
    ck, c0, alpha, beta, gamma = _rand_coefs(rng, nscales)
    x_new0 = np.full((n, nsig), 3.0, dtype)

    # host
    h_new = x_old.copy() if alias else x_new0.copy()
    h_r = r0.copy()
    build_oracle.cheby_step_exact(first, 0, n, mat.indptr, mat.indices, mat.data(dtype), x_cur, x_old,
                                  h_new, h_r, r_rows, nscales, ck, c0, alpha, beta, gamma)
    # device
    dev = lambda a: None if a is None else torch.from_numpy(a).cuda()
    d_cur, d_old, d_r = dev(x_cur), dev(x_old), dev(r0)
    d_new = d_old if alias else dev(x_new0)
    D = mat.D(dtype)
    ranges = [(0, n)] if split is None else [(0, split), (split, n)]
    for rb, re in ranges:
        _step_gpu(gsp, D, first, rb, re, d_cur, d_old, d_new, d_r, r_rows, nsig, nscales, ck, c0,
                  alpha, beta, gamma, plan)
    torch.cuda.synchronize()
    what = "%s %s nsig=%d nscales=%d first=%d plan=%s pad=%d alias=%d split=%s" % (
        mat.name, np.dtype(dtype).name, nsig, nscales, first, plan is not None, r_pad, alias, split)
    _assert_same_bits(d_new, h_new, what + " x_new")
    _assert_same_bits(d_r, h_r, what + " r")
    if r_pad:
        _assert_same_bits(d_r[:, n:], r0[:, n:], what + " r padding")


# ---------------------------------------------------------------- A: step ABI, exact
def test_fmaf_canary_on_the_gpu(gsp):
    """fmaf(a, a, -(1 + 2^-11)) = 2^-24 for a = 1 + 2^-12 (0 if a*a were rounded first)."""
    import torch
    a = 1.0 + 2.0 ** -12
    D = gsp.graphs.DeviceCSR(torch.zeros(2, dtype=torch.int32, device="cuda"),
                             torch.zeros(4, dtype=torch.int32, device="cuda"),
                             torch.zeros(4, dtype=torch.float32, device="cuda"), (1, 1))
    x = torch.ones(1, 1, device="cuda")
    x_new = torch.zeros(1, 1, device="cuda")
    r = torch.zeros(1, 1, 1, device="cuda")
    nat = gsp._native
    nat.call("gsp_cheby_step_f32", nat.i32(1), nat.i64(0), nat.i64(1), nat.i64(0), D.indptr,
             D.indices, D.data, x, None, x_new, r, nat.i64(1), nat.i64(1), nat.i32(1),
             np.array([a]), np.array([-(2.0 + 2.0 ** -10)]), nat.f64(0.75), nat.f64(a), nat.f64(0.0),
             None, nat.stream_ptr())
    torch.cuda.synchronize()
    assert float(x_new) == np.float32(a)
    assert float(r) == 2.0 ** -24


@pytest.mark.parametrize("name", ["E1_1", "E1_2", "E1_3", "E2", "E3", "E4"])
def test_step_matches_exact_oracle_on_edge_matrices(gsp, emats, name):
    mat = emats[name]
    nat = gsp._native
    tiled_runs = 0
    seed = 0
    for nsig in STEP_WIDTHS:
        for nscales in STEP_SCALES:
            plan = _plan(nat, mat.D32, nsig, nscales)
            _assert_edge_condition(mat, plan, nsig, nscales)
            tiled_runs += plan is not None
            for first in (True, False):
                seed += 1
                _check_step(gsp, mat, np.float32, nsig, nscales, first, plan, seed)
                if plan is not None and nscales in (1, 3):
                    _check_step(gsp, mat, np.float32, nsig, nscales, first, None, seed)
                if nsig in (3, 64, 132):
                    _check_step(gsp, mat, np.float64, nsig, nscales, first, None, seed)
    # every tiled width x the bank sizes a launch carries by value takes the tiled kernel
    assert tiled_runs >= (20 if name != "E4" else 12), tiled_runs


def test_hub_forces_two_stage_ring_with_one_cta_per_sm(gsp, emats):
    """E4 with a 3-filter bank: the plan's 3-stage default exceeds the budget, drops to 2 stages,
    and a non-first step's CTA needs more than half an SM's shared memory.  All orders run."""
    import torch
    mat = emats["E4"]
    nat = gsp._native
    plan = _plan(nat, mat.D32, 64, 3)
    assert plan is not None and plan.stages == 2 and plan.slab_capacity >= 7000
    smem = _smem_total(plan, 64, 3, vec_staged=True)
    assert SMEM_PER_SM // 2 < smem + 1024 and smem <= 200 * 1024, smem
    for first in (True, False):
        _check_step(gsp, mat, np.float32, 64, 3, first, plan, 500 + first)
    rng = np.random.default_rng(3)
    x = torch.from_numpy(rng.standard_normal((mat.n, 64)).astype(np.float32)).cuda()
    for order in ORDERS:
        c = rng.standard_normal((3, order + 1))
        got = _whole(gsp, mat.D32, "forward", mat.lmax, c, x, plan)
        want = _whole(gsp, mat.D32, "forward", mat.lmax, c, x, None)
        _assert_same_bits(got, want, "E4 order %d" % order)


@pytest.mark.parametrize("name", ["E1_3", "E3", "E2"])
def test_step_variants_compose(gsp, emats, name):
    """r with padding rows (r_rows = n + 4), x_new aliasing x_old, and a row range split in two
    calls at 4k, 4k + 1, 4k + 2 (the second part unaligned: row-group kernel) give the one-call
    bits of the exact oracle."""
    mat = emats[name]
    nat = gsp._native
    seed = 1000
    for nsig in (8, 32, 64, 132):
        for nscales in (0, 1, 3, 17):
            plan = _plan(nat, mat.D32, nsig, nscales)
            _assert_edge_condition(mat, plan, nsig, nscales)
            if nsig in TILED_WIDTHS and nscales <= 3:
                assert plan is not None
            for first in (True, False):
                seed += 1
                _check_step(gsp, mat, np.float32, nsig, nscales, first, plan, seed, r_pad=4)
                if not first:
                    _check_step(gsp, mat, np.float32, nsig, nscales, first, plan, seed, alias=True)
                k = mat.n // 8
                for d in (0, 1, 2):
                    _check_step(gsp, mat, np.float32, nsig, nscales, first, plan, seed,
                                split=4 * k + d)
            _check_step(gsp, mat, np.float64, nsig, nscales, False, None, seed, r_pad=4, alias=True,
                        split=4 * (mat.n // 8) + 1)


@pytest.mark.parametrize("nsig", TILED_WIDTHS)
def test_step_tile_counts_near_one_tile(gsp, nsig):
    """E5: n in {R - 4, R, R + 3, R + 4, 2R + 1}: no tile (plan declines), exactly one tile,
    remainder rows that are not a multiple of 4 (row-group kernel after the tiles)."""
    nat = gsp._native
    seed = 2000 + nsig
    for nscales in (0, 1, 3):
        R = _default_R(nsig, nscales)
        for n in (R - 4, R, R + 3, R + 4, 2 * R + 1):
            mat = Mat(gsp, "E5", _e5(n, seed), lmax=1.0)
            plan = _plan(nat, mat.D32, nsig, nscales)
            if n < R:
                assert plan is None
            else:
                assert plan is not None and plan.rows_per_tile == R and n // R in (1, 2)
            for first in (True, False):
                seed += 1
                _check_step(gsp, mat, np.float32, nsig, nscales, first, plan, seed, r_pad=4)


# ------------------------------------------------------------------ ring-wrap graph
RING_STEP_CASES = [(8, {}), (64, {}), (64, {"GSPB200_TILE_P2": "1"}), (128, {})]


def _ring_configs():
    """Every (environment, nsig, nscales) the ring-wrap graph is used with."""
    out = [(_ring_env(w, env), w, ns) for w, env in RING_STEP_CASES for ns in (0, 1, 3)]
    for env in [{}] + list(SETTINGS.values()):
        for form, w, ns in WHOLE_CASES:
            out.append((_ring_env(w, env), w, ns))
    return out


@pytest.fixture(scope="module")
def ring(gsp):
    """Morton-ordered Sensor (k = 8) large enough that every plan the file uses wraps the ring;
    sized from the SM count and the plans made for a smaller graph of the same family."""
    nat = gsp._native
    sm = _sm_count(nat)
    probe = gsp.graphs.Sensor(20000, k=8, seed=7, order="morton").L
    need = 0
    with pytest.MonkeyPatch.context() as mp:
        for env, nsig, nscales in _ring_configs():
            _set_env(mp, env)
            p = _plan(nat, probe, nsig, nscales)
            assert p is not None, (env, nsig, nscales)
            per_sm = p.blocks_per_sm if p.blocks_per_sm > 0 else MAX_CTAS_PER_SM
            need = max(need, (2 * p.stages + 1) * sm * per_sm * p.rows_per_tile)
    n = int(need * 1.03) + 256
    G = gsp.graphs.Sensor(n, k=8, seed=7, order="morton")
    G.estimate_lmax()
    mat = Mat(gsp, "ring", G.L.to_scipy().astype(np.float64), lmax=G.lmax)
    assert np.array_equal(mat.data32, G.L.data.cpu().numpy())
    return mat, sm


@pytest.mark.parametrize("case", range(len(RING_STEP_CASES)))
def test_step_matches_exact_oracle_on_ring_graph(gsp, ring, monkeypatch, case):
    mat, sm = ring
    nat = gsp._native
    nsig, env = RING_STEP_CASES[case]
    _set_env(monkeypatch, _ring_env(nsig, env))
    for nscales in (0, 1, 3):
        plan = _plan(nat, mat.D32, nsig, nscales)
        _assert_ring_wraps(plan, mat.n, sm)
        for first in (True, False):
            _check_step(gsp, mat, np.float32, nsig, nscales, first, plan, 3000 + 7 * case + nscales + first)
    _check_step(gsp, mat, np.float64, nsig, 1, False, None, 3100 + case)


# -------------------------------------------------------- B: whole calls, tiled == row-group
def _whole(gsp, D, form, lmax, c, x, plan, out=None):
    """forward: gsp_cheby_op (r, (nscales, n, nsig)); clenshaw / synthesis: gsp_cheby_clenshaw
    (x holds the (nsrc, n, nsig) sources)."""
    import torch
    nat = gsp._native
    c = np.ascontiguousarray(np.atleast_2d(c), dtype=np.float64)
    nf, m = c.shape
    n, nsig = x.shape[-2], x.shape[-1]
    work = torch.empty((2, n, nsig), dtype=D.dtype, device="cuda")
    suf = nat.suffix(D.dtype)
    if form == "forward":
        out = torch.empty((nf, n, nsig), dtype=D.dtype, device="cuda")
        nat.call("gsp_cheby_op_" + suf, nat.i64(n), nat.i64(D.nnz), D.indptr, D.indices, D.data,
                 nat.f64(lmax), c, nat.i32(nf), nat.i32(m), x, nat.i64(nsig), out, work, plan,
                 nat.stream_ptr())
    else:
        out = torch.empty((n, nsig), dtype=D.dtype, device="cuda")
        nat.call("gsp_cheby_clenshaw_" + suf, nat.i64(n), nat.i64(D.nnz), D.indptr, D.indices,
                 D.data, nat.f64(lmax), c, nat.i32(nf), nat.i32(m), x, nat.i64(nsig), out, work,
                 plan, nat.stream_ptr())
    return out


def _inputs(form, n, nsig, nf, order, seed, dtype=np.float32):
    import torch
    rng = np.random.default_rng(seed)
    c = rng.standard_normal((nf, order + 1)) / (1.0 + np.arange(order + 1)) ** 2
    shape = (nf, n, nsig) if form == "synthesis" else (n, nsig)
    tdt = torch.float32 if dtype == np.float32 else torch.float64
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(shape, generator=g, device="cuda", dtype=tdt)
    return c, x


@pytest.fixture(scope="module")
def rowgroup_results():
    return {}


def _whole_calls_agree(gsp, mat, env, mp, cache, sm=None):
    """Every whole case x order on `mat` with the tile plan made under `env` == the row-group
    kernel's bits (plan NULL).  Returns the number of tiled runs."""
    import torch
    nat = gsp._native
    runs = 0
    for form, nsig, nf in WHOLE_CASES:
        e = _ring_env(nsig, env) if sm else dict(env)
        _set_env(mp, e)
        plan = _plan(nat, mat.D32, nsig, nf)
        if sm:
            _assert_ring_wraps(plan, mat.n, sm)
        elif plan is None:
            continue
        _assert_edge_condition(mat, plan, nsig, nf)
        for order in ORDERS:
            seed = zlib.crc32(repr((form, nsig, nf, order)).encode())
            c, x = _inputs(form, mat.n, nsig, nf, order, seed)
            key = (mat.name, form, nsig, nf, order)
            if key not in cache:
                cache[key] = _whole(gsp, mat.D32, form, mat.lmax, c, x, None)
            got = _whole(gsp, mat.D32, form, mat.lmax, c, x, plan)
            torch.cuda.synchronize()
            if not torch.equal(got, cache[key]):
                _assert_same_bits(got, cache[key], "%s %s %s nsig=%d nf=%d order=%d" % (
                    mat.name, e, form, nsig, nf, order))
            runs += 1
    return runs


@pytest.mark.parametrize("setting", ["default", "default-again"] + list(SETTINGS))
def test_whole_calls_tiled_equals_rowgroup_on_ring_graph(gsp, ring, rowgroup_results, monkeypatch,
                                                        setting):
    mat, sm = ring
    env = SETTINGS.get(setting, {})
    runs = _whole_calls_agree(gsp, mat, env, monkeypatch, rowgroup_results, sm=sm)
    assert runs == len(WHOLE_CASES) * len(ORDERS)


@pytest.mark.parametrize("setting", ["default"] + list(SETTINGS))
def test_whole_calls_tiled_equals_rowgroup_on_edge_matrices(gsp, emats, rowgroup_results, monkeypatch,
                                                           setting):
    env = SETTINGS.get(setting, {})
    for name in ("E1_1", "E1_2", "E1_3", "E2", "E3", "E4"):
        runs = _whole_calls_agree(gsp, emats[name], env, monkeypatch, rowgroup_results)
        assert runs >= 8 * len(ORDERS), (name, runs)      # most cases do take the tiled kernel


def test_default_whole_call_is_deterministic(gsp, ring):
    """The same call twice gives the same bits (no race in the ring / barrier protocol)."""
    import torch
    mat, sm = ring
    plan = _plan(gsp._native, mat.D32, 64, 1)
    _assert_ring_wraps(plan, mat.n, sm)
    for form in ("forward", "clenshaw"):
        c, x = _inputs(form, mat.n, 64, 1, 12, 77)
        a = _whole(gsp, mat.D32, form, mat.lmax, c, x, plan)
        b = _whole(gsp, mat.D32, form, mat.lmax, c, x, plan)
        torch.cuda.synchronize()
        assert torch.equal(a, b), form


# --------------------------------------------------------------------- C: anchor to the math
@pytest.mark.parametrize("form,nsig,nf", [("forward", 64, 1), ("forward", 128, 3), ("forward", 8, 1),
                                          ("clenshaw", 64, 1), ("clenshaw", 16, 1),
                                          ("synthesis", 32, 5), ("synthesis", 64, 2)])
def test_rowgroup_result_matches_float64_oracle_on_ring_graph(gsp, ring, form, nsig, nf):
    """Every 5th column (every lane packet of every width) against the float64 oracle."""
    mat, _ = ring
    order = 12
    _, x = _inputs(form, mat.n, nsig, nf, order, 4000 + nsig + nf)
    c = orc.cheby_coeff(orc.heat_kernels(mat.lmax, [10.0 * (i + 1) for i in range(nf)]), mat.lmax, order)
    got = _whole(gsp, mat.D32, form, mat.lmax, c, x, None).cpu().numpy()
    cols = np.arange(0, nsig, 5)
    xs = x.double().cpu().numpy()[..., cols]
    if form == "forward":
        ref = orc.cheby_op(mat.L, mat.lmax, c, xs).reshape(nf, mat.n, cols.size)
        got = got[..., cols]
        assert relerr_cols(got.reshape(-1, cols.size), ref.reshape(-1, cols.size)) <= F32_TOL
    else:
        ref = sum(orc.cheby_op(mat.L, mat.lmax, c[i], xs[i] if form == "synthesis" else xs)
                  for i in range(nf))
        assert relerr_cols(got[:, cols], ref) <= F32_TOL


@pytest.mark.parametrize("name", ["E1_1", "E1_3", "E2", "E4"])
def test_float64_engine_matches_oracle_on_edge_matrices(gsp, emats, name):
    mat = emats[name]
    for form, nsig, nf in (("forward", 7, 3), ("forward", 64, 17), ("clenshaw", 33, 1),
                           ("synthesis", 4, 5)):
        for order in ORDERS:
            c, x = _inputs(form, mat.n, nsig, nf, order, 5000 + order + nsig, np.float64)
            got = _whole(gsp, mat.D64, form, mat.lmax, c, x, None).cpu().numpy()
            xs = x.cpu().numpy()
            if form == "forward":
                ref = orc.cheby_op(mat.L, mat.lmax, c, xs)
                assert relerr_cols(got.reshape(-1, nsig), ref) <= F64_TOL, (form, order)
            else:
                ref = sum(orc.cheby_op(mat.L, mat.lmax, c[i], xs[i] if form == "synthesis" else xs)
                          for i in range(nf))
                assert relerr_cols(got, ref) <= F64_TOL, (form, order)
