"""The Brent-fitted paths at the edges where their kernels change path, and with ill-conditioned covariates:
null-exact (bulkscan_null), scan_null, the null fit of scan_perms, scan_alt and fit_h2.

The first test runs without a GPU: it mirrors the host-side dispatch rules and proves that the shapes below reach
every fit / exact-scan / rotation / permutation-prologue / scan_alt kernel the boundaries allow.  The GPU tests judge
the scans against the longdouble arbiter (oracle/blmm_arbiter.py) at the engine's own h2 (the scan is a deterministic
function of h2), Brent against the exact optimum (mpmath), the exact scan against the grid scan (the other
arithmetic) at the same h2, and paths that share their arithmetic against each other bit for bit."""
import functools
import os

import numpy as np
import pytest

from parity_helpers import H2_TOL
from test_gpu_grid_edges import decomposition, full_covar, heritable_traits, rel

import blmm_oracle as orc
from blmm_b200 import bulkscan_null, bulkscan_null_grid, scan, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "bulklmm.jl_b200", "csrc")
TOL = 1e-8
ELL_TOL = 1e-9  # log-likelihood at the engine's Brent h2 vs the exact optimum: ell is flat there (H2_TOL^2 ~ 4e-14)


# ---------------------------------------------------------------------------------------------------------------
# 1. Which kernels the Brent-fitted paths run
# ---------------------------------------------------------------------------------------------------------------
KC = 20
FIT_WARPS = 4
FIT_LTAB = 512


def n_pad_of(n):
    return -(-n // KC) * KC


def rotation(n, cols):
    """launch_rotate (blmm_prep.cu): rotate_dmma_kernel when `n >= 128 && cols >= 64`, else rotate_kernel<RI>."""
    if n >= 128 and cols >= 64:
        return "rotate_dmma"
    n_pad = n_pad_of(n)
    tiles128 = -(-n_pad // 128)
    ri = min(8, max(4, (-(-n_pad // tiles128) + 15) // 16))
    return f"rotate_kernel<{ri}>"


def paths(n, c, m, p):
    """The kernels of the Brent-fitted calls with n subjects, c covariate columns (intercept included), m traits and
    p markers.  Mirrors, in blmm_fit.cu, launch_fit_h2 (`blocks > 148 * 4` picks fit_h2_kernel<C, BULK>, staging in
    shared memory while `smem <= 96 * 1024`), null_fit_chain_applies (the fused permutation prologue for n <= 128)
    and launch_scan_alt (scan_alt_kernel<c + 1>); in blmm_kernels.cuh exact_marker_atoms (the EXACT scan's marker
    tile) and SCAN_MAX_NQ (resident scan of the permutations, else K-streamed); in blmm_api.cu the EXACT scan's
    scheduler (`operand_bytes > 100e6`: dynamic unit hand-out); launch_rotate as rotation()."""
    n_pad = n_pad_of(n)
    blocks = -(-m // FIT_WARPS)
    smem = FIT_LTAB * 16 + (1 + c + FIT_WARPS) * n_pad * 8
    tile = 2 * 8 * (4 if c + 2 <= 5 else 2)
    p_pad = -(-p // tile) * tile
    slots = -(-m // 64) * 64
    staged = "staged" if smem <= 96 * 1024 else "unstaged"
    return dict(
        # one label per fit_h2_kernel instantiation and staging: the three choices are combined
        fit=f"fit_h2_kernel<{c},{'BULK' if blocks > 148 * 4 else 'single'}> {staged}",
        staged=staged,
        exact=f"exact<{c}> tile {tile}",
        sched="dynamic" if 8.0 * n_pad * (p_pad + slots * (c + 2)) > 100e6 else "static",
        perms=("chain" if n <= 128 else "separate") + "+" + ("resident" if n_pad // KC <= 5 else "streamed"),
        rotation=frozenset({rotation(n, c), rotation(n, m), rotation(n, p), rotation(n, 1)}),
        alt=f"scan_alt_kernel<{c + 1}>" if c <= 7 else None,
    )


def labels(n, c, m, p, kinds):
    ps = paths(n, c, m, p)
    out = set()
    for k in kinds:
        v = ps[k]
        if isinstance(v, frozenset):
            out |= v
        elif v is not None:
            out.add(v)
    return out


# (n, p, m, c): n around the K-chunk boundary (100 / 101: nq 5 / 6) and the n <= 128 / n >= 128 rules (127, 128, 129);
# p ragged at the 32- and 64-marker EXACT tiles, m ragged at the 8-trait column groups and 64-trait tiles.
CASES = [
    dict(n=20, p=31, m=9, c=5),     # tile 32, p one short; rotate_kernel<4>; chain + resident
    dict(n=79, p=65, m=64, c=3),    # tile 64 (c + 2 = 5: the last 64-marker c), p one past; rotate_kernel<5>
    dict(n=100, p=129, m=65, c=4),  # tile 32 (c + 2 = 6: the first 32-marker c); nq = 5; rotate_kernel<7>
    dict(n=101, p=64, m=17, c=2),   # nq = 6: chain + streamed; rotate_kernel<8>
    dict(n=127, p=33, m=63, c=6),   # chain + streamed, n_pad = 140
    dict(n=128, p=97, m=70, c=8),   # DMMA rotation of traits and markers, chain and streamed scan at once
    dict(n=129, p=130, m=66, c=7),  # separate prologue + streamed
    dict(n=250, p=70, m=7, c=1),    # covariates through rotate_kernel<6>, markers through DMMA
]
# fit_h2_kernel<C, BULK> (m > 2368) and, in the halves test_fit_bulk_equals_small_calls compares it with, <C, single>;
# n = 1900 (n_pad > 1877) takes both unstaged for every c
BULK_SHAPES = [dict(n=n, p=1, m=2400, c=c) for n in (79, 1900) for c in range(1, 9)]
UNSTAGED_SHAPES = [dict(n=900, p=1, m=40, c=8)]  # n_pad = 900 > 866: fit_h2_kernel without shared-memory staging
ALT_SHAPES = [dict(n=(79, 101, 128)[c % 3], p=48, m=1, c=c) for c in range(1, 8)]
PERM_SHAPES = [dict(n=128, p=97, m=1, c=8), dict(n=100, p=129, m=1, c=4), dict(n=129, p=130, m=1, c=2)]

NEEDLES = {
    "blmm_fit.cu": ("const bool bulk = blocks > 148 * 4;", "const int staged = smem <= 96 * 1024 ? 1 : 0;",
                    "bool null_fit_chain_applies(int n) { return n <= 128; }", "constexpr int FIT_WARPS = 4;",
                    "constexpr int FIT_LTAB = 512;",
                    "size_t smem = tab_bytes + (size_t)(1 + c + FIT_WARPS) * n_pad * sizeof(double);",
                    "dispatch_c<1, MAXC - 1>(c, [&](auto C) {", "scan_alt_kernel<C + 1>"),
    "blmm_kernels.cuh": ("constexpr int exact_marker_atoms(int c) { return c + 2 <= 5 ? 4 : 2; }",
                         "constexpr int stream_exact_marker_tile(int c) { return 2 * 8 * exact_marker_atoms(c); }",
                         "constexpr int SCAN_MAX_NQ = 5;"),
    "blmm_prep.cu": ("if (n >= 128 && cols >= 64)",
                     "std::min<int64_t>(8, std::max<int64_t>(4, ((ldo_zero + tiles128 - 1) / tiles128 + 15) / 16))"),
    "blmm_api.cu": ("bool dynamic = operand_bytes > 100e6;",
                    "const double operand_bytes = 8.0 * R.n_pad * ((double)p_pad + (double)xcol_pad);"),
    "blmm_common.cuh": ("constexpr int MAXC = 8;",),
}


def _case_id(s):
    return f"n{s['n']}-p{s['p']}-m{s['m']}-c{s['c']}"


def test_case_table_covers_every_dispatch_path():
    # the mirrored thresholds are still the ones in the source: a moved threshold fails here, naming paths()
    for fname, needles in NEEDLES.items():
        with open(os.path.join(CSRC, fname)) as f:
            src = f.read()
        for needle in needles:
            assert needle in src, f"{fname} no longer has `{needle}`: update paths() and the shapes"

    # Labels are combined where one launch makes several choices (the fit: C x BULK x staged).  The others are separate
    # launches with their own rules (the exact scan's tile depends on c alone, the prologue and the permutation scan on
    # n alone, each rotation on its own column count), so each label is required on its own.
    kinds_exact = ("exact", "perms", "rotation")
    required = set()
    for n in range(1, 2001):
        for c in range(1, 9):
            for m in (1, 63, 64, 65, 2368, 2369):
                required |= labels(n, c, m, 64, ("fit", "rotation", "perms", "alt", "exact"))
                required |= labels(n, c, m, 63, ("rotation",))
    covered = set()
    for s in CASES:
        covered |= labels(s["n"], s["c"], s["m"], s["p"], kinds_exact + ("fit",))
    for s in BULK_SHAPES:
        covered |= labels(s["n"], s["c"], s["m"], s["p"], ("fit",)) | labels(s["n"], s["c"], s["m"] // 2, 1, ("fit",))
    for s in UNSTAGED_SHAPES:
        covered |= labels(s["n"], s["c"], s["m"], s["p"], ("fit",))
    for s in ALT_SHAPES:
        covered |= labels(s["n"], s["c"], s["m"], s["p"], ("alt",))
    for s in PERM_SHAPES:
        covered |= labels(s["n"], s["c"], s["m"], s["p"], ("perms", "rotation"))
    for lab in sorted(covered):
        print(f"[exact-edges] path {lab}")
    missing = required - covered
    assert not missing, f"dispatch paths no shape reaches: {sorted(missing)}"

    # the facts the case comments and the bit-identity tests rely on
    assert paths(128, 8, 70, 97)["rotation"] == {"rotate_dmma", "rotate_kernel<5>"}
    assert paths(128, 8, 1, 97)["perms"] == "chain+streamed"
    assert paths(100, 4, 1, 129)["perms"] == "chain+resident" and paths(101, 2, 1, 64)["perms"] == "chain+streamed"
    assert "single>" in paths(79, 1, 2368, 1)["fit"] and "BULK>" in paths(79, 1, 2369, 1)["fit"]
    assert all("single>" in paths(n, c, 1200, 1)["fit"] for n in (79, 1900) for c in range(1, 9))
    assert all(paths(1900, c, 1, 1)["staged"] == "unstaged" for c in range(1, 9))
    assert paths(79, 8, 1, 1)["staged"] == "staged" and paths(900, 8, 1, 1)["staged"] == "unstaged"
    assert paths(860, 8, 1, 1)["staged"] == "staged" and paths(1860, 1, 1, 1)["staged"] == "staged"
    assert paths(1880, 1, 1, 1)["staged"] == "unstaged"
    # the multi-GPU shard of test_multi_gpu_null_exact_bitwise: m = 3000 is BULK, a 1500-trait shard is not
    assert "BULK>" in paths(79, 1, 3000, 1)["fit"] and "single>" in paths(79, 1, 1536, 1)["fit"]
    # every EXACT instantiation c = 1..8 meets a case, both tiles included
    assert {s["c"] for s in CASES} == set(range(1, 9))
    # the conditioning problem's operands stay far under L2: the static scheduler unless forced
    assert paths(79, 3, 24, 70)["sched"] == "static"


# ---------------------------------------------------------------------------------------------------------------
# helpers of the GPU tests
# ---------------------------------------------------------------------------------------------------------------
def make_case(n, p, m, c, seed, h=None, Cv=None):
    G = synth.make_geno(n, p, seed=seed)
    K = synth.calc_kinship_host(G)
    Y = heritable_traits(K, m, np.linspace(0.02, 0.98, m) if h is None else h, seed + 1)
    if Cv is None and c > 1:
        Cv = np.random.default_rng(seed + 2).standard_normal((n, c - 1))
    Ut, lam, dec = decomposition(K)
    return Y, G, K, Cv, Ut, lam, dec


def lod_truth(Y0, G0, C0, lam, h2s):
    """Longdouble LODs, column j at h2s[j] (columns sharing an h2 share one evaluation)."""
    h2s = np.asarray(h2s)
    out = np.empty((G0.shape[1], Y0.shape[1]))
    for h in np.unique(h2s):
        mk = h2s == h
        out[:, mk] = np.asarray(__import__("blmm_arbiter").weighted_liteqtl_ld(Y0[:, mk], G0, C0, lam, h),
                                dtype=np.float64)
    return out


def first_argmax_agrees(L, truth):
    """The engine's arg-max marker of every trait is the longdouble one, wherever the longdouble runner-up is more than
    TOL below the maximum (closer than that, both are the maximum within the north-star bound)."""
    top = np.argmax(truth, axis=0)
    srt = np.sort(truth, axis=0)
    clear = srt[-1] - srt[-2] > TOL * np.maximum(1.0, np.abs(srt[-1])) if truth.shape[0] > 1 else np.ones(truth.shape[1], bool)
    assert np.array_equal(np.argmax(L, axis=0)[clear], top[clear])


def perm_truth(y0, G0, C0, lam, h2, perm):
    """Longdouble scan_perms_lite (src/scan.jl:485-557) at the given null h2: unpermuted LOD and L_perms."""
    import blmm_arbiter as arb
    n = len(y0)
    sw = np.sqrt(arb.make_weights_ld(h2, lam))
    z = arb._resid_ld((y0 * sw)[:, None], C0 * sw[:, None])[:, 0]
    Z = np.column_stack([z, z[perm]])
    X = arb._resid_ld(G0 * sw[:, None], C0 * sw[:, None])
    Z = Z / np.sqrt(np.sum(Z * Z, axis=0))[None, :]
    X = X / np.sqrt(np.sum(X * X, axis=0))[None, :]
    R = X.T @ Z
    L = np.asarray(-(arb.LD(n) / arb.LD(2)) * np.log10(arb.LD(1) - R * R), dtype=np.float64)
    return L[:, 0], L[:, 1:]


# ---------------------------------------------------------------------------------------------------------------
# 2. exact scans per case against longdouble, both schedulers, and the single-point grid scan
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_exact_scan_vs_longdouble(engine, monkeypatch, case):
    import blmm_arbiter as arb
    n, p, m, c = case["n"], case["p"], case["m"], case["c"]
    seed = 500 + 10 * c + n
    Y, G, K, Cv, Ut, lam, dec = make_case(n, p, m, c, seed)
    C1 = full_covar(n, Cv)
    Y0, G0, C0 = arb.rotate_ld(Ut, Y, G, C1)
    kw = dict(Covar=Cv, decomposition=dec, engine=engine, reml=True)
    runs = []
    for dynamic in ("0", "1"):
        monkeypatch.setenv("BLMM_STREAM_DYNAMIC", dynamic)
        runs.append(bulkscan_null(Y, G, K, **kw))
    monkeypatch.delenv("BLMM_STREAM_DYNAMIC")
    r = runs[0]
    # the schedulers hand the same units to different CTAs; each unit's arithmetic is the same
    assert np.array_equal(runs[1].L, r.L) and np.array_equal(runs[1].h2_null_list, r.h2_null_list)
    truth = lod_truth(Y0, G0, C0, lam, r.h2_null_list)
    assert rel(r.L, truth) < TOL
    first_argmax_agrees(r.L, truth)

    # scan_null (ML, prior (0, 0)): the same exact scan after its own fit
    lod, s2, h2 = engine.scan_null_host(Y, G, C1, dec[0], lam)
    t2 = lod_truth(Y0, G0, C0, lam, h2)
    assert rel(lod, t2) < TOL
    first_argmax_agrees(lod, t2)

    # the other arithmetic: a one-point null-grid scan at the trait's h2 returns that h2 exactly
    for j in np.unique(np.linspace(0, m - 1, 3).astype(int)):
        h = float(r.h2_null_list[j])
        g = bulkscan_null_grid(Y[:, j:j + 1], G, K, [h], **kw)
        assert g.h2_null_list[0] == h
        assert rel(g.L[:, 0], truth[:, j]) < TOL
        assert rel(r.L[:, j], g.L[:, 0]) < TOL


# ---------------------------------------------------------------------------------------------------------------
# 3. bit identity where the arithmetic is the same
# ---------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=1)
def bulk_problem(n):
    Y, G, K, Cv, Ut, lam, dec = make_case(n, 200, 2400, 1, seed=600 + n, h=np.linspace(0.0, 0.99, 2400))
    return Y, dec, lam


@pytest.mark.gpu
@pytest.mark.parametrize("shape", BULK_SHAPES, ids=_case_id)
def test_fit_bulk_equals_small_calls(engine, shape):
    """fit_h2_kernel<C, BULK> (2400 traits) against <C, single> (two calls of 1200): the same objective evaluations in
    the same order, only the unrolling and the occupancy differ; staged at n = 79, unstaged at n = 1900."""
    n, c = shape["n"], shape["c"]
    Y, dec, lam = bulk_problem(n)
    Cv = np.random.default_rng(610 + c).standard_normal((n, c - 1)) if c > 1 else None
    C1 = full_covar(n, Cv)
    for reml in (False, True):
        whole = engine.fit_h2(Y, C1, dec[0], lam, reml=reml)
        a = engine.fit_h2(Y[:, :1200], C1, dec[0], lam, reml=reml)
        b = engine.fit_h2(Y[:, 1200:], C1, dec[0], lam, reml=reml)
        for k in range(3):  # h2, sigma2, ell
            assert np.array_equal(whole[k], np.concatenate([a[k], b[k]])), (reml, k)


@pytest.mark.gpu
@pytest.mark.parametrize("n,c", [(79, 1), (128, 8), (900, 8)])
def test_fit_staged_equals_unstaged(engine, monkeypatch, n, c):
    """fit_h2_kernel reading its operands from shared memory against the same kernel reading them from global memory
    (BLMM_B200_FIT_UNSTAGED forces the latter); n = 900, c = 8 is unstaged on its own, and its fit is judged against
    the longdouble log-likelihood and the oracle's Brent."""
    import blmm_arbiter as arb
    m = UNSTAGED_SHAPES[0]["m"] if n == 900 else 40
    Y, G, K, Cv, Ut, lam, dec = make_case(n, 200, m, c, seed=700 + n + c)
    C1 = full_covar(n, Cv)
    base = engine.fit_h2(Y, C1, dec[0], lam, reml=True)
    monkeypatch.setenv("BLMM_B200_FIT_UNSTAGED", "1")
    forced = engine.fit_h2(Y, C1, dec[0], lam, reml=True)
    monkeypatch.delenv("BLMM_B200_FIT_UNSTAGED")
    for k in range(3):
        assert np.array_equal(base[k], forced[k]), k
    if n == 900:
        Y0, C0 = arb.rotate_ld(Ut, Y, C1)
        ml = engine.fit_h2(Y, C1, dec[0], lam, reml=False)
        ell_ld = np.array([float(arb.grid_loglik_ld(Y0[:, j:j + 1], C0, lam, [ml[0][j]], (0.0, 0.0), False)[0, 0])
                           for j in range(m)])
        assert rel(ml[2], ell_ld) < ELL_TOL
        for j in (0, m // 2, m - 1):
            ref = orc.fitlmm(Ut @ Y[:, j:j + 1], Ut @ C1, lam, [0.0, 0.0], reml=False)
            assert abs(ml[0][j] - ref.h2) < H2_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("shape", PERM_SHAPES, ids=_case_id)
def test_chain_equals_separate(engine, monkeypatch, shape):
    """The fused permutation prologue (null_fit_chain_kernel, n <= 128) against the separate kernels: same rotation,
    same Brent, same weight constants, bit for bit; n = 129 has no chain (both runs take the separate kernels)."""
    n, p, c = shape["n"], shape["p"], shape["c"]
    Y, G, K, Cv, Ut, lam, dec = make_case(n, p, 3, c, seed=800 + n + c, h=[0.3, 0.7, 0.95])
    C1 = full_covar(n, Cv)
    perm = synth.make_perm_indices(n, 130, rndseed=n)
    for j in range(3):
        for reml, oi in ((False, 1), (True, 3)):
            a = engine.scan_perms_host(Y[:, j:j + 1], G, C1, dec[0], lam, perm, reml=reml, optim_interval=oi)
            monkeypatch.setenv("BLMM_B200_NO_CHAIN", "1")
            b = engine.scan_perms_host(Y[:, j:j + 1], G, C1, dec[0], lam, perm, reml=reml, optim_interval=oi)
            monkeypatch.delenv("BLMM_B200_NO_CHAIN")
            for k in ("h2_null", "sigma2_e", "lod", "L_perms", "max_lod"):
                assert np.array_equal(getattr(a, k), getattr(b, k)), (j, reml, k)


@pytest.mark.gpu
def test_multi_gpu_null_exact_bitwise(engine):
    """3000 traits: BULK on one GPU, a non-BULK shard per GPU on two or more; the fits and LODs must not change."""
    import torch
    from blmm_b200 import Engine
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    n, p, m = 79, 130, 3000
    Y, G, K, Cv, Ut, lam, dec = make_case(n, p, m, 2, seed=900, h=np.linspace(0.0, 0.99, m))
    one = bulkscan_null(Y, G, K, Covar=Cv, decomposition=dec, engine=engine)
    multi = Engine(devices=list(range(min(torch.cuda.device_count(), 8))))
    try:
        many = bulkscan_null(Y, G, K, Covar=Cv, decomposition=dec, engine=multi)
    finally:
        multi.close()
    assert np.array_equal(one.h2_null_list, many.h2_null_list)
    assert np.array_equal(one.L, many.L)


# ---------------------------------------------------------------------------------------------------------------
# 4. Brent against the exact optimum; scan_alt at every covariate count
# ---------------------------------------------------------------------------------------------------------------
def check_fit_vs_exact(T, h_eng, ell_eng, reml, what):
    """ell reported at the engine's h2 within ELL_TOL of the exact ell at that h2 (the objective's arithmetic) and of
    ell at the exact optimum (50 digits); h2 within H2_TOL of it where the optimum is interior.  Returns |h2 error|
    (0 at a boundary optimum)."""
    ell_at = float(T.ell(h_eng, reml=reml)[0])
    assert abs(ell_eng - ell_at) <= ELL_TOL * max(1.0, abs(ell_at)), (what, ell_eng, ell_at, h_eng)
    h_mp = T.fit_h2(reml=reml, x0=h_eng)
    ell_mp = float(T.ell(h_mp, reml=reml)[0])
    assert abs(ell_eng - ell_mp) <= ELL_TOL * max(1.0, abs(ell_mp)), (what, ell_eng, ell_mp, h_eng, float(h_mp))
    # the refined optimum is the global one: no point of a 41-point scan of [0, 1) lies above it
    cache = T.__dict__.setdefault("_scan_ell", {})
    if reml not in cache:
        cache[reml] = max(float(T.ell(h, reml=reml)[0]) for h in np.linspace(0.0, 1.0 - 1e-6, 41))
    assert cache[reml] <= ell_mp + ELL_TOL * max(1.0, abs(ell_mp)), (what, cache[reml], ell_mp)
    interior = 1e-6 < float(h_mp) < 1.0 - 1e-6
    if interior:
        assert abs(h_eng - float(h_mp)) < H2_TOL, (what, h_eng, float(h_mp))
    return abs(h_eng - float(h_mp)) if interior else 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("c", range(1, 9))
def test_brent_vs_exact_optimum(engine, c):
    import blmm_arbiter as arb
    n = (79, 101, 128)[c % 3]
    Y, G, K, Cv, Ut, lam, dec = make_case(n, 200, 6, c, seed=1000 + c, h=[0.15, 0.35, 0.5, 0.65, 0.8, 0.95])
    C1 = full_covar(n, Cv)
    cols = (c % 6, (c + 3) % 6)
    traits = {j: arb.TraitMP(Y[:, j], C1, Ut, lam) for j in cols}
    worst = 0.0
    for reml in (False, True):
        for oi in (1, 3):
            h, s2, ell = engine.fit_h2(Y, C1, dec[0], lam, reml=reml, optim_interval=oi)
            for j in cols:
                worst = max(worst, check_fit_vs_exact(traits[j], h[j], ell[j], reml, (c, reml, oi, j)))
    print(f"[exact-edges] Brent c = {c}, n = {n}: worst |h2 - exact optimum| {worst:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("c", [1, 3, 8])
def test_brent_boundary_optima(engine, c):
    """Traits with no genetic variance and traits with nearly all of it on the rank-deficient kinship of the grid-edges
    test: optima at h2 = 0, and interior optima next to 1 where most weights are ~1e-4 of the others.  (Closer to 1,
    at 1 - h2 ~ 2e-6, Brent's stopping tolerance sqrt(eps) h2 = 1.5e-8 is ~1 % of 1 - h2 and ell is curved as
    n / (1 - h2)^2 there: the reference's own Brent leaves ell ~1e-8 relative below its optimum.)"""
    import blmm_arbiter as arb
    n = 79
    K = synth.calc_kinship_host(synth.make_geno(n, 20, seed=76, fuzz=0.0))
    Ut, lam, dec = decomposition(K)
    Y = heritable_traits(K, 4, [0.0, 0.0, 0.99, 0.9999], seed=1100 + c)
    Cv = np.random.default_rng(1101 + c).standard_normal((n, c - 1)) if c > 1 else None
    C1 = full_covar(n, Cv)
    traits = [arb.TraitMP(Y[:, j], C1, Ut, lam) for j in range(4)]
    fits = []
    for reml in (False, True):
        for oi in (1, 3):
            h, s2, ell = engine.fit_h2(Y, C1, dec[0], lam, reml=reml, optim_interval=oi)
            fits.append(h)
            for j in range(4):
                check_fit_vs_exact(traits[j], h[j], ell[j], reml, (c, reml, oi, j))
    print(f"[exact-edges] boundary fits c = {c}: h2 {np.array(fits).round(9).tolist()}")


@pytest.mark.gpu
@pytest.mark.parametrize("c", range(1, 8))
def test_scan_alt_every_c(engine, c):
    """scan_alt_kernel<c + 1> for every c it takes, ML and REML, optim_interval 1 and 3, at the tolerances of
    test_gpu_exact.py's test_scan_alt_per_marker_variance_components (the objective is flat at its optimum)."""
    s = ALT_SHAPES[c - 1]
    n, p = s["n"], s["p"]
    Y, G, K, Cv, Ut, lam, dec = make_case(n, p, 2, c, seed=1200 + c, h=[0.4, 0.8])
    y = Y[:, c % 2]
    for reml, oi in ((False, 1), (True, 3)):
        kw = dict(prior_variance=float(np.var(y, ddof=1)), prior_sample_size=0.1, reml=reml, optim_interval=oi)
        r = scan(y, G, K, covar=Cv, assumption="alt", decomposition=dec, engine=engine, **kw)
        ref = orc.scan(y, G, K, covar=Cv, assumption="alt", Ut=Ut, lam=lam, **kw)
        assert abs(r.h2_null - ref["h2_null"]) < 1e-6
        assert abs(r.sigma2_e - ref["sigma2_e"]) < 1e-6 * max(1.0, ref["sigma2_e"])
        assert np.max(np.abs(r.h2_each_marker - ref["h2_each_marker"])) < 2e-6
        assert rel(r.lod, ref["lod"]) < 1e-6


# ---------------------------------------------------------------------------------------------------------------
# 5. ill-conditioned covariates: intercept, x and x + eps * noise
# ---------------------------------------------------------------------------------------------------------------
NEAR_DUP_EPS = [2e-2, 2e-3, 2e-4, 2e-5]  # kappa(C) ~ 2 / eps: 1e2 .. 1e5


def near_duplicate_covariates(n, eps, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal(n)
    return np.column_stack([x, x + eps * rng.standard_normal(n)])


def conditioning_problem(eps):
    import blmm_arbiter as arb
    n, p, m = 79, 70, 24
    G = synth.make_geno(n, p, seed=1300)
    K = synth.calc_kinship_host(G)
    Cv = near_duplicate_covariates(n, eps, 1301)
    C1 = full_covar(n, Cv)
    Y = heritable_traits(K, m, np.linspace(0.0, 0.99, m), seed=1302) + 2.0 * Cv[:, :1]
    Ut, lam, dec = decomposition(K)
    Y0, G0, C0 = arb.rotate_ld(Ut, Y, G, C1)
    return Y, G, K, Cv, C1, Ut, lam, dec, Y0, G0, C0


@pytest.mark.gpu
@pytest.mark.parametrize("eps", NEAR_DUP_EPS)
def test_conditioning_vs_longdouble(engine, eps):
    """Up to kappa(C) = 1e5 every Brent-fitted scan holds the north-star 1e-8 against longdouble at its own h2 (the
    float64 QR oracle holds ~1e-11 there): null-exact and scan_null, scan_perms (L_perms and the fused maxima), and the
    one-point grid scan at forced h2 and at the exact scan's h2."""
    Y, G, K, Cv, C1, Ut, lam, dec, Y0, G0, C0 = conditioning_problem(eps)
    n, m = Y.shape
    kappa = np.linalg.cond(C1)
    kw = dict(Covar=Cv, decomposition=dec, engine=engine)
    err = {}

    def record(name, L, truth, L_orc=None):
        err[name] = (rel(L, truth), rel(L_orc, truth) if L_orc is not None else float("nan"))

    r = bulkscan_null(Y, G, K, **kw)
    truth = lod_truth(Y0, G0, C0, lam, r.h2_null_list)
    o = orc.bulkscan_null(Y, G, K, Covar=Cv, Ut=Ut, lam=lam, h2_override=r.h2_null_list)
    record("null-exact", r.L, truth, o.L)

    lod, s2, h2 = engine.scan_null_host(Y, G, C1, dec[0], lam, reml=True)
    record("scan_null", lod, lod_truth(Y0, G0, C0, lam, h2))

    for h in (0.5, 0.99):
        g = bulkscan_null_grid(Y, G, K, [h], **kw)
        og = orc.bulkscan_null_grid(Y, G, K, [h], Covar=Cv, Ut=Ut, lam=lam)
        record(f"grid h2={h}", g.L, lod_truth(Y0, G0, C0, lam, np.full(m, h)), og.L)
    j = m // 2
    g = bulkscan_null_grid(Y[:, j:j + 1], G, K, [r.h2_null_list[j]], **kw)
    assert g.h2_null_list[0] == r.h2_null_list[j]
    record("grid at exact's h2", g.L[:, 0], truth[:, j])

    perm = synth.make_perm_indices(n, 100, rndseed=7)
    ep, em = [], []
    for jj in (2, m - 3):
        s = engine.scan_perms_host(Y[:, jj:jj + 1], G, C1, dec[0], lam, perm)
        t0, tp = perm_truth(Y0[:, jj], G0, C0, lam, s.h2_null, perm)
        ep.append(max(rel(s.lod, t0), rel(s.L_perms, tp)))
        em.append(rel(s.max_lod, tp.max(axis=0)))
        assert np.array_equal(s.max_lod, s.L_perms.max(axis=0))
    err["scan_perms L"] = (max(ep), float("nan"))
    err["scan_perms max"] = (max(em), float("nan"))

    print(f"[exact-edges] kappa(C) = {kappa:.1e} (eps = {eps:g}), h2 in [{r.h2_null_list.min():.3g}, "
          f"{r.h2_null_list.max():.3g}]; engine / oracle max rel error vs longdouble: " +
          ", ".join(f"{k} {v[0]:.1e} / {v[1]:.1e}" for k, v in err.items()))
    bad = {k: v[0] for k, v in err.items() if not v[0] < TOL}
    assert not bad, (kappa, bad)


@pytest.mark.gpu
@pytest.mark.parametrize("eps", NEAR_DUP_EPS)
def test_conditioning_fit_loglik(engine, eps):
    """The log-likelihood fit_h2 reports at its own h2 against longdouble (ML, every trait) and 50 digits (REML), and
    Brent's h2 against the exact optimum on a sample of traits, ML and REML."""
    import blmm_arbiter as arb
    Y, G, K, Cv, C1, Ut, lam, dec, Y0, G0, C0 = conditioning_problem(eps)
    m = Y.shape[1]
    hh, ss, ell = engine.fit_h2(Y, C1, dec[0], lam, reml=False)
    ell_ld = np.asarray([arb.grid_loglik_ld(Y0[:, i:i + 1], C0, lam, [hh[i]], (0.0, 0.0), False)[0, 0]
                         for i in range(m)], dtype=np.float64)
    e_ml = rel(ell, ell_ld)
    hr, sr, ellr = engine.fit_h2(Y, C1, dec[0], lam, reml=True)
    er, eh = [], 0.0
    for i in (1, m // 2, m - 2):
        T = arb.TraitMP(Y[:, i], C1, Ut, lam)
        er.append(abs(ellr[i] - float(T.ell(hr[i], reml=True)[0])) / max(1.0, abs(ellr[i])))
        eh = max(eh, check_fit_vs_exact(T, hh[i], ell[i], False, (eps, i, "ML")),
                 check_fit_vs_exact(T, hr[i], ellr[i], True, (eps, i, "REML")))
    print(f"[exact-edges] kappa(C) = {np.linalg.cond(C1):.1e}: fit_h2 ell max rel error ML {e_ml:.1e}, "
          f"REML {max(er):.1e}; worst |h2 - exact optimum| {eh:.1e}")
    assert e_ml < TOL and max(er) < TOL
