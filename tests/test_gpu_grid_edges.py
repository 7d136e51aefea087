"""Grid scans at the edges where their kernels change path: grid length (up to the 255-point ceiling), covariate count
(c = 1..8, where the table kernels leave lanes of the warp unused), grid order and repeated points, heritabilities at
the ends of [0, 1) with a rank-deficient kinship, and LODs of (near-)collinear marker / trait pairs through the scan
epilogue's table logarithm and its fix_lod fallback.

The first test runs without a GPU: it mirrors the host-side dispatch formulas and proves that the cases below reach
every trait-statistics / marker-operand / scan-kernel combination the boundaries allow.  Every other test compares
the engine with the float64 oracle (oracle/blmm_oracle.py) and, where digits are at stake, with the longdouble
arbiter (oracle/blmm_arbiter.py)."""
import os

import numpy as np
import pytest

from parity_helpers import TIE_RTOL, assert_h2_panel_explained

import blmm_oracle as orc
from blmm_b200 import BlmmError, bulkscan_alt_grid, bulkscan_null, bulkscan_null_grid, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-8
EPS = np.finfo(np.float64).eps
LOG10E = float(np.log10(np.e))
TT = 128  # traits per scan tile (SCAN_TT)


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b)))) if a.size else 0.0


# ---------------------------------------------------------------------------------------------------------------
# 1. Which kernels a grid scan runs
# ---------------------------------------------------------------------------------------------------------------
WARPS_PER_BLOCK = 8


def paths(n, c, nk):
    """(trait statistics, marker operand, scan kernel) of a grid scan with n subjects, c covariate columns (intercept
    included) and nk grid points.  Mirrors bulklmm.jl_b200/csrc/blmm_prep.cu launch_trait_stats (the
    `table_smem <= 96 * 1024` test; 'a' = table kernel with one batch, which also writes the alt-grid scalars and the
    packed trait operand, 'b' = table kernel with several batches, 'c' = generic trait_stats_kernel),
    launch_marker_operand (`tsmem <= 56 * 1024`) and, in blmm_api.cu run_scan, `P.nq <= scan_max_nq(P.nk)` with
    scan_max_nq = 5 in blmm_scan.cu ('resident' scan_kernel, else the K-streamed scan_stream_kernel)."""
    n_pad = -(-n // 20) * 20  # KC = 20
    kb = 32 // (1 + c)
    nbatch = -(-nk // kb)
    table = (nbatch * n_pad * 32 + WARPS_PER_BLOCK * 2 * n_pad) * 8
    trait = ("a" if nbatch == 1 else "b") if table <= 96 * 1024 else "c"
    tsmem = (2 * nbatch * n_pad * 32 + WARPS_PER_BLOCK * 2 * n_pad + n_pad) * 8
    marker = "table" if tsmem <= 56 * 1024 else "generic"
    scan = "resident" if n_pad // 20 <= 5 else "streamed"
    return trait, marker, scan


def _largest_fitting_nbatch(limit, nbytes):
    nb = 0
    while nbytes(nb + 1) <= limit:
        nb += 1
    return nb


def boundary_nks(n_pad, c):
    """Grid lengths on both sides of every boundary of paths(): KB, KB + 1, the largest nbatch * KB whose table still
    fits (trait and marker tables), one more, and the 255-point ceiling."""
    kb = 32 // (1 + c)
    nbt = _largest_fitting_nbatch(96 * 1024, lambda nb: (nb * n_pad * 32 + WARPS_PER_BLOCK * 2 * n_pad) * 8)
    nbm = _largest_fitting_nbatch(56 * 1024, lambda nb: (2 * nb * n_pad * 32 + WARPS_PER_BLOCK * 2 * n_pad + n_pad) * 8)
    nks = {kb, kb + 1, nbt * kb, nbt * kb + 1, nbm * kb, nbm * kb + 1, 255}
    return sorted(k for k in nks if 1 <= k <= 255)


# (n, p, m, c, nk): p and m ragged around the 64-marker / 128-trait tiles.  Comments give paths().
CASES = [
    dict(n=37, p=70, m=150, c=6, nk=4),      # a, table, resident; KB = 4: 28 of 32 lanes
    dict(n=80, p=130, m=150, c=1, nk=16),    # a, table, resident; n_pad = 80 takes the marker table only at nbatch 1
    dict(n=20, p=130, m=150, c=5, nk=25),    # b, table, resident; KB = 5 (30 lanes), largest fitting marker table
    dict(n=20, p=70, m=300, c=5, nk=26),     # b, generic, resident; one batch more
    dict(n=40, p=70, m=150, c=7, nk=8),      # b, table, resident; KB = 4, all 32 lanes
    dict(n=79, p=130, m=150, c=8, nk=12),    # b, generic, resident; KB = 3: 27 lanes, largest fitting trait table
    dict(n=79, p=70, m=150, c=8, nk=13),     # c, generic, resident
    dict(n=93, p=70, m=300, c=3, nk=8),      # a, generic, resident (n_pad = 100: never the marker table)
    dict(n=113, p=130, m=150, c=2, nk=10),   # a, generic, streamed
    dict(n=113, p=70, m=150, c=7, nk=5),     # b, generic, streamed
    dict(n=113, p=70, m=300, c=4, nk=19),    # c, generic, streamed
    dict(n=20, p=130, m=300, c=1, nk=255),   # b, generic, resident: 16 batches of 16 grid points
    dict(n=79, p=70, m=150, c=2, nk=255),    # c, generic, resident
]
# the 255-point shapes of section 3 (n = 137: K-streamed)
CEILING_SHAPES = [dict(n=79, c=1, nk=255), dict(n=137, c=1, nk=255)]


def _case_id(c):
    return f"n{c['n']}-p{c['p']}-m{c['m']}-c{c['c']}-k{c['nk']}"


def test_case_table_covers_every_dispatch_path():
    # the mirrored thresholds are still the ones in the source: a moved threshold fails here, naming paths()
    with open(os.path.join(ROOT, "bulklmm.jl_b200", "csrc", "blmm_prep.cu")) as f:
        prep = f.read()
    with open(os.path.join(ROOT, "bulklmm.jl_b200", "csrc", "blmm_scan.cu")) as f:
        scan_src = f.read()
    for needle in ("constexpr int WARPS_PER_BLOCK = 8;", "const int KB = 32 / (1 + c);",
                   "if (table_smem <= 96 * 1024)", "if (tsmem <= 56 * 1024)",
                   "(size_t)WARPS_PER_BLOCK * 2 * n_pad + (size_t)n_pad"):
        assert needle in prep, f"blmm_prep.cu no longer has `{needle}`: update paths() and the cases"
    assert "(void)nk;\n  return 5;" in scan_src, "scan_max_nq changed: update paths()"

    required = {}
    for c in range(1, 9):
        for n_pad in (20, 40, 80, 100, 120):
            for nk in boundary_nks(n_pad, c):
                required.setdefault(paths(n_pad, c, nk), []).append((n_pad, c, nk))
    covered = {}
    for case in CASES + CEILING_SHAPES:
        covered.setdefault(paths(case["n"], case["c"], case["nk"]), []).append((case["n"], case["c"], case["nk"]))
    for combo in sorted(covered):
        print(f"[grid-edges] path {combo}: cases (n, c, nk) {covered[combo]}")
    missing = {k: v for k, v in required.items() if k not in covered}
    assert not missing, "dispatch paths no case reaches (with the boundary (n_pad, c, nk) that reach them): " + \
        "; ".join(f"{k}: {v[:4]}" for k, v in sorted(missing.items()))
    # the facts the case comments rely on
    assert paths(80, 1, 16)[1] == "table" and paths(80, 1, 17)[1] == "generic"
    assert all(paths(n_pad, c, 1)[1] == "generic" for n_pad in (100, 120) for c in range(1, 9))
    # every c = 5..8 (lanes left unused by the table kernels) meets a table kernel
    assert {case["c"] for case in CASES if paths(case["n"], case["c"], case["nk"])[0] in "ab"} >= {5, 6, 7, 8}


# ---------------------------------------------------------------------------------------------------------------
# helpers of the GPU tests
# ---------------------------------------------------------------------------------------------------------------
def covariates(n, c, seed):
    """c - 1 random columns (the intercept is added by the API and by the oracle)."""
    if c == 1:
        return None
    rng = np.random.default_rng(seed)
    return rng.standard_normal((n, c - 1))


def full_covar(n, Cv):
    return np.ones((n, 1)) if Cv is None else np.hstack([np.ones((n, 1)), Cv])


def decomposition(K):
    Ut, lam = orc.decompose(K)
    return Ut, lam, (np.asfortranarray(Ut.T), lam)


def heritable_traits(K, m, h, seed, mean=11.0):
    """y = mean + sqrt(h) L_K z + sqrt(1 - h) e with per-trait h (scalar or array)."""
    rng = np.random.default_rng(seed)
    n = K.shape[0]
    w, V = np.linalg.eigh(K)
    LK = V * np.sqrt(np.clip(w, 0.0, None))[None, :]
    h = np.broadcast_to(np.asarray(h, dtype=np.float64), (m,))
    return mean + (LK @ rng.standard_normal((n, m))) * np.sqrt(h)[None, :] + \
        rng.standard_normal((n, m)) * np.sqrt(1.0 - h)[None, :]


def replay_counters(prof):
    """tmax!'s counter (number of strict improvements) of every entry, from the oracle's logL1 profile."""
    mx = prof[0].copy()
    cnt = np.zeros(mx.shape, dtype=np.int64)
    for k in range(1, len(prof)):
        better = mx < prof[k]
        cnt += better
        mx = np.where(better, prof[k], mx)
    return cnt


def tie_free(prof):
    """Entries none of whose tmax! comparisons is a rounding-level tie: their h2 panel value is determined."""
    mx = prof[0].copy()
    ok = np.ones(mx.shape, dtype=bool)
    scale = np.maximum(1.0, np.max(np.abs(np.stack(prof)), axis=0))
    for k in range(1, len(prof)):
        ok &= np.abs(prof[k] - mx) > TIE_RTOL * scale
        mx = np.maximum(mx, prof[k])
    return ok


def check_alt_grid(engine, Y, G, K, grid, Ut, lam, dec, cols, **kw):
    """alt-grid, both panel modes, against the oracle on the trait columns `cols`; returns (engine result, profile)."""
    a = bulkscan_alt_grid(Y, G, K, grid, decomposition=dec, engine=engine, **kw)
    prof = []
    ref = orc.bulkscan_alt_grid(Y[:, cols], G, K, grid, Ut=Ut, lam=lam, profile=prof, **kw)
    assert rel(a.L[:, cols], ref.L) < TOL
    assert_h2_panel_explained(a.h2_panel[:, cols], ref.h2_panel, prof, grid)
    assert np.all(np.isin(a.h2_panel, grid))
    am = bulkscan_alt_grid(Y, G, K, grid, decomposition=dec, engine=engine, h2_panel_mode="argmax", **kw)
    assert np.array_equal(am.L, a.L)  # the panel mode changes the bookkeeping, never the LOD
    ref_am = np.asarray(grid)[np.argmax(np.stack(prof), axis=0)]
    assert_h2_panel_explained(am.h2_panel[:, cols], ref_am, prof, grid, mode="argmax")
    return a, am, ref, prof


def check_null_grid(engine, Y, G, K, grid, Ut, lam, dec, cols, **kw):
    r = bulkscan_null_grid(Y, G, K, grid, decomposition=dec, engine=engine, **kw)
    ref = orc.bulkscan_null_grid(Y[:, cols], G, K, grid, Ut=Ut, lam=lam, **kw)
    assert np.array_equal(r.h2_null_list[cols], ref.h2_null_list)
    assert rel(r.L[:, cols], ref.L) < TOL
    return r, ref


# ---------------------------------------------------------------------------------------------------------------
# 2. grid length x covariate count vs the oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_grid_paths_vs_oracle(engine, case):
    n, p, m, c, nk = case["n"], case["p"], case["m"], case["c"], case["nk"]
    seed = 1000 * c + nk
    Y, G, K = synth.make_problem(n, p, m, seed_g=seed, seed_y=seed + 1)
    Cv = covariates(n, c, seed + 2)
    Ut, lam, dec = decomposition(K)
    grid = np.sort(np.random.default_rng(seed + 3).uniform(0.0, 0.95, size=nk))
    # columns are independent: at 255 points the oracle runs on a seeded sample of the full engine call's columns
    cols = np.sort(np.random.default_rng(seed + 4).choice(m, size=40, replace=False)) if nk == 255 else np.arange(m)
    C1 = full_covar(n, Cv)
    for reml in (False, True):
        kw = dict(Covar=Cv, reml=reml)
        check_null_grid(engine, Y, G, K, grid, Ut, lam, dec, cols, **kw)
        check_alt_grid(engine, Y, G, K, grid, Ut, lam, dec, cols, **kw)
        ell = engine.grid_loglik(Y, C1, dec[0], lam, grid, reml=reml, prior_variance=1.0, prior_sample_size=0.0)
        ell_ref = orc.grid_loglik(Ut @ Y, Ut @ C1, lam, grid, [1.0, 0.0], reml=reml)
        assert rel(ell, ell_ref) < 1e-10


# ---------------------------------------------------------------------------------------------------------------
# 3. the 255-point ceiling
# ---------------------------------------------------------------------------------------------------------------
GRID255_DOWN = np.linspace(0.95, 0.0, 255)
GRID255_UP = np.linspace(0.0, 0.95, 255)


def ceiling_problem(n, p, m, direction, seed):
    """Traits for which logL1 improves at (nearly) every grid point: no genetic signal on a descending grid,
    strongly heritable traits on an ascending one."""
    G = synth.make_geno(n, p, seed=seed)
    K = synth.calc_kinship_host(G)
    if direction == "down":
        Y = 11.0 + np.random.default_rng(seed + 1).standard_normal((n, m))
        grid = GRID255_DOWN
    else:
        Y = heritable_traits(K, m, 0.999, seed + 1)
        grid = GRID255_UP
    return Y, G, K, grid


def word_mates(m):
    """Trait columns whose tmax! counters share one 32-bit register with column j in scan_kernel: columns
    wt*16 + b*8 + 2t + cc of one trait tile for b, cc in {0, 1} (blmm_scan.cu: o = (a*BT + b)*2 + cc, register o >> 2)."""
    j = np.arange(m)
    base = (j // TT) * TT + ((j % TT) // 16) * 16 + ((j % 8) // 2) * 2
    mates = [base + off for off in (0, 1, 8, 9)]
    return [np.where(mt < m, mt, j) for mt in mates]


@pytest.mark.gpu
@pytest.mark.parametrize("direction", ["down", "up"])
def test_counter_reaches_254(engine, direction):
    n, p, m = 79, 70, 150
    Y, G, K, grid = ceiling_problem(n, p, m, direction, seed=61 if direction == "down" else 62)
    Ut, lam, dec = decomposition(K)
    a, am, ref, prof = check_alt_grid(engine, Y, G, K, grid, Ut, lam, dec, np.arange(m))
    cnt = replay_counters(prof)
    top = cnt == 254
    print(f"[grid-edges] {direction}: {int(top.sum())} of {cnt.size} entries reach counter 254")
    assert top.sum() >= 300, int(top.sum())
    # every entry whose comparisons are all clear of rounding: the exact panel value, no tie resolution
    free = tie_free(prof)
    assert np.array_equal(a.h2_panel[free], ref.h2_panel[free])
    assert np.all(a.h2_panel[top & free] == grid[254])
    # the three other counters of a register that reached 254: exact as well where determined
    mates = np.zeros_like(top)
    rows, colsv = np.nonzero(top)
    for mt in word_mates(m):
        mates[rows, mt[colsv]] = True
    assert np.array_equal(a.h2_panel[mates & free], ref.h2_panel[mates & free])


@pytest.mark.gpu
def test_counter_254_host_index_transfer(engine, monkeypatch):
    """The chunked host-buffer alt-grid path sends the h2 panel as one-byte grid indices (0..254) and expands them on
    the host: identical to the device-resident call, bit for bit, at the top index."""
    import torch
    from blmm_b200 import _lib as L
    monkeypatch.setenv("BLMM_B200_H2_TRANSFER", "index")
    monkeypatch.setenv("BLMM_B200_HOST_THREADS", "3")
    n, p, m = 79, 70, 2100  # 17 trait tiles: the chunked path
    Y, G, K, grid = ceiling_problem(n, p, m, "down", seed=63)
    Ut, lam, dec = decomposition(K)
    host = bulkscan_alt_grid(Y, G, K, grid, decomposition=dec, engine=engine)
    dev = torch.device("cuda:0")
    t = lambda x: torch.from_numpy(np.ascontiguousarray(np.asarray(x, dtype=np.float64).T)).to(dev)
    d = [t(Y), t(G), t(np.ones((n, 1))), t(dec[0]), torch.from_numpy(lam.copy()).to(dev)]
    dL = torch.empty((m, p), dtype=torch.float64, device=dev)
    dH = torch.empty((m, p), dtype=torch.float64, device=dev)
    pr = engine.make_problem(n, p, m, 1, *[x.data_ptr() for x in d])
    o, keep = engine.make_opts(method=L.METHOD_ALT_GRID, h2_grid=grid, mem_space=L.MEM_DEVICE)
    engine.bulkscan_raw(pr, o, dL.data_ptr(), dH.data_ptr())
    engine.sync()
    assert np.array_equal(host.L, dL.cpu().numpy().T)
    assert np.array_equal(host.h2_panel, dH.cpu().numpy().T)
    assert np.sum(host.h2_panel == grid[254]) >= 1000
    cols = np.sort(np.random.default_rng(7).choice(m, size=40, replace=False))
    prof = []
    ref = orc.bulkscan_alt_grid(Y[:, cols], G, K, grid, Ut=Ut, lam=lam, profile=prof)
    assert rel(host.L[:, cols], ref.L) < TOL
    assert_h2_panel_explained(host.h2_panel[:, cols], ref.h2_panel, prof, grid)


@pytest.mark.gpu
def test_255_points_streamed(engine):
    """n = 137 > 100: the K-streamed GRID kernel with 255 grid points (its own counter registers and grid copy)."""
    n, p, m = 137, 70, 150
    Y, G, K, grid = ceiling_problem(n, p, m, "up", seed=64)
    Ut, lam, dec = decomposition(K)
    cols = np.sort(np.random.default_rng(8).choice(m, size=40, replace=False))
    check_null_grid(engine, Y, G, K, grid, Ut, lam, dec, cols)
    a, am, ref, prof = check_alt_grid(engine, Y, G, K, grid, Ut, lam, dec, cols)
    cnt = replay_counters(prof)
    free = tie_free(prof)
    assert (cnt == 254).sum() >= 100, int((cnt == 254).sum())
    assert np.array_equal(a.h2_panel[:, cols][free], ref.h2_panel[free])


@pytest.mark.gpu
def test_null_grid_many_bins(engine):
    """A fine 255-point grid and traits of spread heritability: one bin per populated grid point, most of them
    nearly empty (padding columns, col_map = -1, per-warp atomic slots)."""
    n, p, m = 79, 70, 600
    G = synth.make_geno(n, p, seed=65)
    K = synth.calc_kinship_host(G)
    Y = heritable_traits(K, m, np.random.default_rng(66).uniform(0.0, 0.999, size=m), seed=67)
    grid = np.linspace(0.0, 0.99, 255)
    Ut, lam, dec = decomposition(K)
    r, ref = check_null_grid(engine, Y, G, K, grid, Ut, lam, dec, np.arange(m))
    nbins = len(np.unique(ref.h2_null_list))
    print(f"[grid-edges] null-grid: {nbins} populated bins of 255")
    assert nbins >= 100, nbins
    # the per-warp atomics order the columns inside a bin; results do not depend on that order
    r2 = bulkscan_null_grid(Y, G, K, grid, decomposition=dec, engine=engine)
    assert np.array_equal(r2.L, r.L) and np.array_equal(r2.h2_null_list, r.h2_null_list)


@pytest.mark.gpu
def test_256_points_refused(engine):
    Y, G, K = synth.make_problem(79, 40, 20, seed_g=68, seed_y=69)
    Ut, lam, dec = decomposition(K)
    for method in (bulkscan_null_grid, bulkscan_alt_grid):
        with pytest.raises(BlmmError) as e:
            method(Y, G, K, np.linspace(0.0, 0.95, 256), decomposition=dec, engine=engine)
        assert e.value.msg == "h2 grids longer than 255 points are not supported"
    # the context stays usable
    check_null_grid(engine, Y, G, K, GRID255_UP, Ut, lam, dec, np.arange(20))
    check_alt_grid(engine, Y, G, K, GRID255_UP, Ut, lam, dec, np.arange(20))


# ---------------------------------------------------------------------------------------------------------------
# 4. grid order and repeated points: exact engine-vs-engine properties
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n,c", [(79, 2), (113, 1)])
def test_grid_order_and_repeated_points(engine, n, c):
    p, m = 70, 150
    Y, G, K = synth.make_problem(n, p, m, seed_g=70 + n, seed_y=71 + n)
    Cv = covariates(n, c, 72)
    Ut, lam, dec = decomposition(K)
    grid = np.sort(np.random.default_rng(73).uniform(0.0, 0.95, size=12))
    kw = dict(Covar=Cv, decomposition=dec, engine=engine)
    a = bulkscan_alt_grid(Y, G, K, grid, **kw)
    am = bulkscan_alt_grid(Y, G, K, grid, h2_panel_mode="argmax", **kw)
    r = bulkscan_null_grid(Y, G, K, grid, **kw)

    # unsorted: the minimum over k and max ell0 do not depend on the order
    perm = np.random.default_rng(74).permutation(len(grid))
    pgrid = grid[perm]
    ap = bulkscan_alt_grid(Y, G, K, pgrid, **kw)
    assert np.array_equal(ap.L, a.L)
    prof = []
    pref = orc.bulkscan_alt_grid(Y, G, K, pgrid, Covar=Cv, Ut=Ut, lam=lam, profile=prof)
    assert rel(ap.L, pref.L) < TOL
    assert_h2_panel_explained(ap.h2_panel, pref.h2_panel, prof, pgrid)
    rp = bulkscan_null_grid(Y, G, K, pgrid, **kw)
    rp_ref = orc.bulkscan_null_grid(Y, G, K, pgrid, Covar=Cv, Ut=Ut, lam=lam)
    assert np.array_equal(rp.h2_null_list, rp_ref.h2_null_list)
    same = rp.h2_null_list == r.h2_null_list
    assert np.array_equal(rp.L[:, same], r.L[:, same])

    # every point twice: the copy has bit-identical operands, so it never improves strictly
    dgrid = np.repeat(grid, 2)
    ad = bulkscan_alt_grid(Y, G, K, dgrid, **kw)
    assert np.array_equal(ad.L, a.L)
    cnt = np.searchsorted(grid, a.h2_panel)  # the deduplicated call's counter: h2_panel = grid[cnt]
    assert np.array_equal(grid[cnt], a.h2_panel)
    assert np.array_equal(ad.h2_panel, dgrid[cnt])  # tmax!'s counter, not the arg-max: dgrid[cnt] != grid[cnt]
    adm = bulkscan_alt_grid(Y, G, K, dgrid, h2_panel_mode="argmax", **kw)
    assert np.array_equal(adm.L, a.L) and np.array_equal(adm.h2_panel, am.h2_panel)  # first maximum
    rd = bulkscan_null_grid(Y, G, K, dgrid, **kw)
    rd_ref = orc.bulkscan_null_grid(Y, G, K, dgrid, Covar=Cv, Ut=Ut, lam=lam)
    assert np.array_equal(rd.h2_null_list, rd_ref.h2_null_list)
    assert np.array_equal(rd.h2_null_list, r.h2_null_list)
    assert np.array_equal(rd.L, r.L)


# ---------------------------------------------------------------------------------------------------------------
# 5. heritabilities at the ends of [0, 1) against the longdouble arbiter
# ---------------------------------------------------------------------------------------------------------------
GRID_ENDS = np.array([0.0, 1e-12, 0.5, 0.999, 0.999999, 1.0 - 1e-9])


def near_truth(L_eng, L_orc, truth, what):
    """Engine within TOL of the longdouble value; where it is not, its worst error is within 10x the oracle's worst
    + 1e-12 (as test_arbiter_on_worst_entries).  Returns (worst engine error, worst oracle error)."""
    truth = np.asarray(truth, dtype=np.float64)
    scale = np.maximum(1.0, np.abs(truth))
    e_eng = np.abs(L_eng - truth) / scale
    e_orc = np.abs(L_orc - truth) / scale
    assert np.all(np.isfinite(e_eng)), what
    if np.any(e_eng > TOL):
        assert e_eng.max() <= 10 * e_orc.max() + 1e-12, (what, e_eng.max(), e_orc.max())
    return float(e_eng.max()), float(e_orc.max())


@pytest.mark.gpu
@pytest.mark.parametrize("c", [1, 3])
@pytest.mark.parametrize("kinship", ["synthetic", "rank-deficient"])
def test_extreme_heritabilities_vs_longdouble(engine, kinship, c):
    import blmm_arbiter as arb
    n, p, m = 79, 70, 48
    G = synth.make_geno(n, p, seed=75)
    if kinship == "synthetic":
        K = synth.calc_kinship_host(G)
    else:
        # 20 markers without imputed values: rank <= 21, the other eigenvalues are zero up to rounding
        K = synth.calc_kinship_host(synth.make_geno(n, 20, seed=76, fuzz=0.0))
    Y = heritable_traits(K, m, np.linspace(0.0, 0.99, m), seed=77)
    Cv = covariates(n, c, 78)
    C1 = full_covar(n, Cv)
    Ut, lam, dec = decomposition(K)
    nneg = int(np.sum(lam < 0))
    nzero = int(np.sum(np.abs(lam) < 1e-9))
    Y0, G0, C0 = arb.rotate_ld(Ut, Y, G, C1)
    kw = dict(Covar=Cv, decomposition=dec, engine=engine)

    # log-likelihoods on the grid
    ell = engine.grid_loglik(Y, C1, dec[0], lam, GRID_ENDS, prior_variance=1.0, prior_sample_size=0.0)
    ell_orc = orc.grid_loglik(Ut @ Y, Ut @ C1, lam, GRID_ENDS, [1.0, 0.0])
    ell_ld = arb.grid_loglik_ld(Y0, C0, lam, GRID_ENDS, (1.0, 0.0), False)
    near_truth(ell, ell_orc, ell_ld, "grid_loglik")

    # LODs at every single grid point (a one-point alt-grid scan is the LOD at that h2)
    worst = {}
    for h in GRID_ENDS:
        a1 = bulkscan_alt_grid(Y, G, K, [h], **kw)
        o1 = orc.bulkscan_alt_grid(Y, G, K, [h], Covar=Cv, Ut=Ut, lam=lam)
        truth = arb.weighted_liteqtl_ld(Y0, G0, C0, lam, h)
        worst[h] = near_truth(a1.L, o1.L, truth, f"LOD at h2 = {h!r}")

    # alt-grid over the whole grid
    a = bulkscan_alt_grid(Y, G, K, GRID_ENDS, **kw)
    prof = []
    aref = orc.bulkscan_alt_grid(Y, G, K, GRID_ENDS, Covar=Cv, Ut=Ut, lam=lam, profile=prof)
    L_ld, _, _ = arb.bulkscan_alt_grid_ld(Y, G, C1, Ut, lam, GRID_ENDS)
    e_alt = near_truth(a.L, aref.L, L_ld, "alt-grid")
    assert_h2_panel_explained(a.h2_panel, aref.h2_panel, prof, GRID_ENDS)

    # null-grid: the oracle's h2 exactly, LODs against the longdouble LOD at that h2
    r = bulkscan_null_grid(Y, G, K, GRID_ENDS, **kw)
    ref = orc.bulkscan_null_grid(Y, G, K, GRID_ENDS, Covar=Cv, Ut=Ut, lam=lam)
    assert np.array_equal(r.h2_null_list, ref.h2_null_list)
    truth = np.empty((p, m))
    for h in np.unique(r.h2_null_list):
        mk = r.h2_null_list == h
        truth[:, mk] = np.asarray(arb.weighted_liteqtl_ld(Y0[:, mk], G0, C0, lam, h), dtype=np.float64)
    e_null = near_truth(r.L, ref.L, truth, "null-grid")
    print(f"[grid-edges] {kinship} K (c = {c}): lambda in [{lam.min():.3g}, {lam.max():.3g}], {nzero} |lambda| < 1e-9, "
          f"{nneg} negative; worst engine / oracle error vs longdouble: at h2 = 1 - 1e-9 "
          f"{worst[GRID_ENDS[-1]][0]:.2e} / {worst[GRID_ENDS[-1]][1]:.2e}, alt-grid {e_alt[0]:.2e} / {e_alt[1]:.2e}, "
          f"null-grid {e_null[0]:.2e} / {e_null[1]:.2e} (h2 chosen: {sorted(set(r.h2_null_list.tolist()))})")
    if kinship == "rank-deficient":
        assert nzero >= 40  # the case this test is about: weights of ~1 next to weights of ~1e-10 at h2 = 1 - 1e-9


# ---------------------------------------------------------------------------------------------------------------
# 6. LOD extremes through the scan epilogue
# ---------------------------------------------------------------------------------------------------------------
V_TARGETS = np.logspace(-1, -15, 29)
COLLINEAR = [(1.0, 0.0), (-1.0, 0.0), (2.5, 11.0), (0.7, 11.0), (-1.3, 5.0), (1.0, 11.0), (3.0, -2.0), (0.25, 0.0)]


def collinear_problem(n, p, seed):
    """Traits y_j = a g_i + b + eps_j z_j, z_j orthogonal to (1, g_i), with eps_j chosen so that 1 - r^2 (without
    weights) is V_TARGETS[j]; then exactly collinear traits (eps = 0); then ordinary traits.  The markers i_j spread
    over all three 64-marker tiles and the constructed traits share the first 128-trait tile with ordinary ones."""
    G = synth.make_geno(n, p, seed=seed)
    K = synth.calc_kinship_host(G)
    rng = np.random.default_rng(seed + 1)
    cols, idx = [], []
    nc = len(V_TARGETS) + len(COLLINEAR)
    markers = rng.choice(p, size=nc, replace=False)
    for j in range(nc):
        i = int(markers[j])
        g = G[:, i]
        X = np.column_stack([np.ones(n), g])
        if j < len(V_TARGETS):
            a, b = 1.3, 11.0
            v = V_TARGETS[j]
            z = orc.resid(rng.standard_normal(n), X)
            gp = orc.resid(g, np.ones((n, 1)))
            eps = a * np.linalg.norm(gp) * np.sqrt(v / (1.0 - v)) / np.linalg.norm(z)
            y = a * g + b + eps * z
        else:
            a, b = COLLINEAR[j - len(V_TARGETS)]
            y = a * g + b
        cols.append(y)
        idx.append(i)
    Y = np.column_stack(cols[:20] + [synth.make_pheno(G, K, 60, seed=seed + 2)] + cols[20:])
    Y = np.column_stack([Y, synth.make_pheno(G, K, 60, seed=seed + 3)])
    order = list(range(20)) + list(range(80, 80 + nc - 20))  # trait columns of the constructed traits
    n_exact = len(COLLINEAR)
    j_exact = order[-n_exact:]
    exact = np.zeros((p, Y.shape[1]), dtype=bool)
    for jj, i in zip(j_exact, idx[-n_exact:]):
        exact[:, jj] = np.all(G == G[:, [i]], axis=0)  # the marker itself and any identical marker
    return Y, G, K, exact, np.array(order[:len(V_TARGETS)])


def check_extremes(L_eng, L_orc, truth, exact, n, what, per_entry=True):
    """exact: +inf, NaN or a finite LOD of at least (n/2)*13; a non-zero v is one FMA of operands near 1, >= ~2^-106,
    so a finite LOD above (n/2)*40 is the table logarithm applied to an operand fix_lod should have taken.
    v_true < 1e-6: the problem is ill-conditioned.  per_entry: every entry within 4x the oracle's error on that entry +
    the conditioning of 8 eps in v ((n/2) log10(e) 8 eps / v_true).  Otherwise the engine's worst error in v is within
    4x the oracle's worst + 8 eps: for LODs that combine several quantities (the maximum over the grid of alt-grid, the
    per-trait h2 of null-exact) both float64 implementations carry a few tens of eps in v on these entries, shared with
    the reference formula, so one entry's oracle error is no bound for that entry.
    Everything else (the neighbours in the same tiles included): 1e-8 of the longdouble value and of the oracle."""
    half = n / 2.0
    le = L_eng[exact]
    fin = np.isfinite(le)
    assert np.all(np.isnan(le) | (le == np.inf) | (fin & (le >= half * 13) & (le <= half * 40))), (what, le)
    with np.errstate(over="ignore"):
        v_true = np.power(10.0, -np.asarray(truth, dtype=np.float64) / half)
    small = (v_true < 1e-6) & ~exact
    normal = ~small & ~exact
    d_eng = np.abs(L_eng[small] - truth[small])
    d_orc = np.abs(L_orc[small] - truth[small])
    if per_entry:
        bound = 4 * d_orc + half * LOG10E * 8 * EPS / v_true[small]
        assert np.all(d_eng <= bound), (what, np.max(d_eng / bound))
    elif small.any():
        to_v_eps = v_true[small] / (half * LOG10E * EPS)  # LOD error -> error of v in units of eps
        dv_eng, dv_orc = d_eng * to_v_eps, d_orc * to_v_eps
        assert dv_eng.max() <= 4 * dv_orc.max() + 8, (what, dv_eng.max(), dv_orc.max())
    assert rel(L_eng[normal], truth[normal]) < TOL, what
    assert rel(L_eng[normal], L_orc[normal]) < TOL, what
    return int(exact.sum()), int(small.sum()), int(np.sum(le == np.inf)), int(np.sum(np.isnan(le)))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [79, 137])
def test_lod_extremes(engine, n):
    import blmm_arbiter as arb
    p = 130
    Y, G, K, exact, jv = collinear_problem(n, p, seed=80 + n)
    m = Y.shape[1]
    Ut, lam, dec = decomposition(K)
    C1 = np.ones((n, 1))
    Y0, G0, C0 = arb.rotate_ld(Ut, Y, G, C1)
    kw = dict(decomposition=dec, engine=engine)
    grid = np.arange(10) / 10.0
    with np.errstate(divide="ignore", invalid="ignore"):
        # null-grid: LODs at the (shared) null h2 of each trait
        r = bulkscan_null_grid(Y, G, K, grid, **kw)
        ref = orc.bulkscan_null_grid(Y, G, K, grid, Ut=Ut, lam=lam)
        assert np.array_equal(r.h2_null_list, ref.h2_null_list)
        truth = np.empty((p, m))
        for h in np.unique(r.h2_null_list):
            mk = r.h2_null_list == h
            truth[:, mk] = np.asarray(arb.weighted_liteqtl_ld(Y0[:, mk], G0, C0, lam, h), dtype=np.float64)
        stats = check_extremes(r.L, ref.L, truth, exact, n, "null-grid")

        # one-point alt-grid scans: the e - d^2 et epilogue (e = 1) at every grid point, where v is one 1 - r^2
        for h in grid:
            a1 = bulkscan_alt_grid(Y, G, K, [h], **kw)
            o1 = orc.bulkscan_alt_grid(Y, G, K, [h], Ut=Ut, lam=lam)
            t1 = np.asarray(arb.weighted_liteqtl_ld(Y0, G0, C0, lam, h), dtype=np.float64)
            check_extremes(a1.L, o1.L, t1, exact, n, f"alt-grid at h2 = {h}")

        # alt-grid over the grid, both panel modes
        a = bulkscan_alt_grid(Y, G, K, grid, **kw)
        am = bulkscan_alt_grid(Y, G, K, grid, h2_panel_mode="argmax", **kw)
        assert np.array_equal(am.L, a.L, equal_nan=True)
        prof = []
        aref = orc.bulkscan_alt_grid(Y, G, K, grid, Ut=Ut, lam=lam, profile=prof)
        L_ld, _, prof_ld = arb.bulkscan_alt_grid_ld(Y, G, C1, Ut, lam, grid)
        L_ld = np.asarray(L_ld, dtype=np.float64)
        check_extremes(a.L, aref.L, L_ld, exact, n, "alt-grid", per_entry=False)
        assert np.all(np.isin(a.h2_panel, grid)) and np.all(np.isin(am.h2_panel, grid))
        with np.errstate(over="ignore"):
            settled = np.power(10.0, -L_ld / (n / 2.0)) >= 1e-6  # the profile is accurate to well within a tie there
        masked = np.where(settled, a.h2_panel, aref.h2_panel)
        assert_h2_panel_explained(masked, aref.h2_panel, prof, grid)

        # null-exact: the streamed kernel's exact mode (Newton reciprocal), compared at the engine's own h2
        e = bulkscan_null(Y, G, K, **kw)
        eref = orc.bulkscan_null(Y, G, K, Ut=Ut, lam=lam, h2_override=e.h2_null_list)
        truth = np.empty((p, m))
        for j in range(m):
            truth[:, j] = np.asarray(arb.weighted_liteqtl_ld(Y0[:, j:j + 1], G0, C0, lam, e.h2_null_list[j]),
                                     dtype=np.float64)[:, 0]
        check_extremes(e.L, eref.L, truth, exact, n, "null-exact", per_entry=False)
    v_rows = np.array([np.min(np.power(10.0, -np.asarray(truth[:, j]) / (n / 2.0))) for j in jv])
    print(f"[grid-edges] n = {n}: {stats[0]} exactly collinear entries (null-grid: {stats[2]} +inf, {stats[3]} NaN), "
          f"{stats[1]} entries with v < 1e-6; constructed v from {v_rows.max():.1e} to {v_rows.min():.1e}")
