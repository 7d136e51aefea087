"""Per-trait LOD peaks (blmm_bulkscan_peaks): for every trait, the first maximum of its LOD column in Julia's findmax
order, the marker where it occurs and the h2 there, reduced in the scan epilogue instead of forming the p x m matrices.

The peaks must be the dense call's values bit for bit (blmm_bulkscan on the same arguments, reduced on the host), agree
with the float64 oracle, resolve ties to the first marker wherever the tied markers sit (one warp block, two marker
tiles, two CTAs, two null-grid bins), handle +inf / NaN LODs as findmax does, and run where the dense L would not fit
in device memory."""
import ctypes as C

import numpy as np
import pytest

from parity_helpers import TIE_RTOL

import blmm_oracle as orc
from blmm_b200 import BlmmError, Engine, bulkscan_peaks, synth, _lib as L

pytestmark = pytest.mark.gpu
GRID = np.arange(10) / 10.0
METHODS = (L.METHOD_NULL_GRID, L.METHOD_ALT_GRID, L.METHOD_NULL_EXACT)
NAMES = {L.METHOD_NULL_GRID: "null-grid", L.METHOD_ALT_GRID: "alt-grid", L.METHOD_NULL_EXACT: "null-exact"}
I64MAX = np.iinfo(np.int64).max


def findmax_rows(Lm):
    """Julia's findmax of every column: NaN above everything (first NaN wins), -0.0 below +0.0, first index on ties."""
    Lm = np.ascontiguousarray(Lm, dtype=np.float64)
    b = Lm.view(np.int64)
    k = np.where(b >= 0, b, b ^ I64MAX)
    k = np.where(np.isnan(Lm), I64MAX, k)
    return np.argmax(k, axis=0)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def problem(n, p, m, c, weighted, seed, engine):
    G = synth.make_geno(n, p, seed=seed)
    K = synth.calc_kinship_host(G)
    Y = synth.make_pheno(G, K, m, seed=seed + 1)
    rng = np.random.default_rng(seed + 2)
    C0 = np.column_stack([np.ones(n)] + [rng.standard_normal(n) for _ in range(c - 1)])
    w = rng.uniform(0.5, 2.0, n) if weighted else None
    Kd = engine.weight_kinship(K, w) if weighted else K
    Ut, lam = orc.decompose(Kd)
    return Y, G, C0, np.asfortranarray(Ut.T), lam, w


def kw(method, reml, mode=L.H2PANEL_REFERENCE, grid=GRID):
    return dict(method=method, h2_grid=grid, reml=reml, prior_variance=0.0 if method == L.METHOD_NULL_EXACT else 1.0,
                prior_sample_size=0.0, h2_panel_mode=mode)


def dense(engine, Y, G, C0, U, lam, w, method, reml, mode=L.H2PANEL_REFERENCE, grid=GRID):
    k = kw(method, reml, mode, grid)
    return engine.bulkscan_host(Y, G, C0, U, lam, k["method"], k["h2_grid"], reml, k["prior_variance"], 0.0,
                                h2_panel_mode=mode, weights=w)


def peaks(engine, Y, G, C0, U, lam, w, method, reml, mode=L.H2PANEL_REFERENCE, grid=GRID, chisq_df=0):
    k = kw(method, reml, mode, grid)
    return engine.bulkscan_peaks_host(Y, G, C0, U, lam, k["method"], k["h2_grid"], reml, k["prior_variance"], 0.0,
                                      h2_panel_mode=mode, weights=w, chisq_df=chisq_df)


def assert_peaks_of(Ld, Hd, pk, method):
    """pk = (lod, marker, h2[, log10p]) is the findmax of the dense (L, h2) bit for bit"""
    lod, mk, h2 = pk[:3]
    m = Ld.shape[1]
    idx = findmax_rows(Ld)
    assert mk.dtype == np.int64 and np.array_equal(mk, idx), np.nonzero(mk != idx)
    assert np.array_equal(bits(lod), bits(Ld[idx, np.arange(m)]))
    ref_h2 = Hd[idx, np.arange(m)] if method == L.METHOD_ALT_GRID else Hd
    assert np.array_equal(bits(h2), bits(ref_h2))


# ---------------------------------------------------------------------------------------------------------------
# 1. Bit for bit the dense call, every method / likelihood / panel mode, c = 1..3, weights, ragged shapes, both kernels
# ---------------------------------------------------------------------------------------------------------------
CASES = [  # n, p, m, c, weighted: p ragged around the 32 / 64-marker blocks, m around the 128-trait tile
    (79, 300, 200, 1, False),
    (79, 63, 129, 2, True),
    (79, 97, 127, 3, False),
    (79, 1, 5, 1, False),
    (137, 130, 257, 1, True),
    (137, 33, 64, 3, False),
    (137, 65, 130, 2, False),
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "n{}_p{}_m{}_c{}{}".format(*c[:4], "_w" if c[4] else ""))
@pytest.mark.parametrize("method", METHODS, ids=lambda m: NAMES[m])
@pytest.mark.parametrize("reml", [False, True], ids=["ml", "reml"])
def test_peaks_equal_dense(engine, case, method, reml):
    n, p, m, c, weighted = case
    Y, G, C0, U, lam, w = problem(n, p, m, c, weighted, seed=1000 + n + p + m + c, engine=engine)
    modes = (L.H2PANEL_REFERENCE, L.H2PANEL_ARGMAX) if method == L.METHOD_ALT_GRID else (L.H2PANEL_REFERENCE,)
    for mode in modes:
        Ld, Hd = dense(engine, Y, G, C0, U, lam, w, method, reml, mode)
        pk = peaks(engine, Y, G, C0, U, lam, w, method, reml, mode, chisq_df=2)
        assert_peaks_of(Ld, Hd, pk, method)
        assert np.array_equal(bits(pk[3]), bits(engine.lod2log10p(pk[0], 2)))


# ---------------------------------------------------------------------------------------------------------------
# 2. Against the float64 oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [79, 137])
@pytest.mark.parametrize("method", METHODS, ids=lambda m: NAMES[m])
def test_peaks_vs_oracle(engine, n, method):
    p, m = 150, 140
    Y, G, C0, U, lam, _ = problem(n, p, m, 1, False, seed=2000 + n, engine=engine)
    Ut = U.T
    lod, mk, h2 = peaks(engine, Y, G, C0, U, lam, None, method, reml=True)
    if method == L.METHOD_NULL_EXACT:  # at the engine's own Brent h2 (two FP64 Brent fits agree to ~1e-8 only)
        Lo = orc.bulkscan_null(Y, G, np.eye(n), reml=True, prior_variance=0.0, Ut=Ut, lam=lam, h2_override=h2).L
    else:
        Lo = orc.bulkscan(Y, G, np.eye(n), method=NAMES[method], h2_grid=GRID, reml=True, Ut=Ut, lam=lam)["L"]
    omax = Lo.max(axis=0)
    assert np.all(np.abs(lod - omax) <= 1e-8 * np.maximum(1.0, np.abs(omax)))
    oidx = np.argmax(Lo, axis=0)
    at_eng = Lo[mk, np.arange(m)]
    tie = np.abs(at_eng - omax) <= TIE_RTOL * np.maximum(1.0, np.abs(omax))
    assert np.all((mk == oidx) | tie)


# ---------------------------------------------------------------------------------------------------------------
# 3. Ties and special values
# ---------------------------------------------------------------------------------------------------------------
def tied_problem(n, p, pairs, m, seed):
    """Marker b is a copy of marker a for every (a, b) in pairs, and a is an independent random genotype (no other
    marker equals it, as neighbours along a chromosome may); trait j carries a strong effect of the a of pair
    j % len(pairs).  The kinship-structured background grows from 0 to 1.5 standard deviations over the traits, so
    their null heritabilities fall into several grid bins, while the peak (by more than 4 LOD units over every other
    marker, in the float64 oracle) stays the tie between a and b."""
    G = synth.make_geno(n, p, seed=seed)
    rng = np.random.default_rng(seed + 1)
    for a, b in pairs:
        G[:, a] = rng.integers(0, 2, n)
        G[:, b] = G[:, a]
    K = synth.calc_kinship_host(G)
    w, V = np.linalg.eigh(K)
    LK = V * np.sqrt(np.clip(w, 0.0, None))[None, :]
    s = np.linspace(0.0, 1.5, m)
    Y = 11.0 + (LK @ rng.standard_normal((n, m))) * s[None, :] + 0.3 * rng.standard_normal((n, m))
    first = np.empty(m, dtype=np.int64)
    for j in range(m):
        a, _ = pairs[j % len(pairs)]
        Y[:, j] += (2.0 + rng.random()) * G[:, a]
        first[j] = a
    Ut, lam = orc.decompose(K)
    return Y, G, np.ones((n, 1)), np.asfortranarray(Ut.T), lam, first


@pytest.mark.parametrize("n", [79, 137])
@pytest.mark.parametrize("method", METHODS, ids=lambda m: NAMES[m])
def test_ties_go_to_the_first_marker(engine, n, method):
    # (3, 17): one warp block; (5, 70): two marker tiles; (100, 19_000): with one trait tile and 300 marker tiles the
    # units are spread over all CTAs, so the two copies are scanned by different CTAs
    p, m = 300 * 64, 100
    pairs = [(3, 17), (5, 70), (100, 19_000)]
    Y, G, C0, U, lam, first = tied_problem(n, p, pairs, m, seed=3000 + n)
    Ld, Hd = dense(engine, Y, G, C0, U, lam, None, method, reml=False)
    for a, b in pairs:
        assert np.array_equal(bits(Ld[a]), bits(Ld[b]))  # the copies tie bit for bit
    pk = peaks(engine, Y, G, C0, U, lam, None, method, reml=False)
    assert np.array_equal(pk[1], first)
    assert_peaks_of(Ld, Hd, pk, method)
    if method == L.METHOD_NULL_GRID:  # the traits sit in several h2 bins (several k-lists of the binned scan)
        assert len(np.unique(Hd)) >= 2


@pytest.mark.parametrize("n", [79, 137])
@pytest.mark.parametrize("method", METHODS, ids=lambda m: NAMES[m])
def test_collinear_traits(engine, n, method):
    """Traits that are exact linear functions of a marker (and of its copy) give LODs of +inf or NaN at those markers:
    the peak and its marker are findmax over the dense L, NaN included."""
    p = 130
    G = synth.make_geno(n, p, seed=4000 + n)
    G[:, 90] = G[:, 20]
    K = synth.calc_kinship_host(G)
    Y = synth.make_pheno(G, K, 40, seed=4001 + n)
    for j, (i, a, b) in enumerate([(20, 1.0, 0.0), (20, -1.3, 5.0), (7, 2.5, 11.0), (64, 0.25, 0.0), (129, 3.0, -2.0)]):
        Y[:, 3 * j] = a * G[:, i] + b
    Ut, lam = orc.decompose(K)
    U = np.asfortranarray(Ut.T)
    C0 = np.ones((n, 1))
    Ld, Hd = dense(engine, Y, G, C0, U, lam, None, method, reml=False)
    assert_peaks_of(Ld, Hd, peaks(engine, Y, G, C0, U, lam, None, method, reml=False), method)


# ---------------------------------------------------------------------------------------------------------------
# 4. A scan whose L does not fit in device memory (p = 2^20, m = 32768: 256 GB of L)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("method", [L.METHOD_NULL_GRID, L.METHOD_ALT_GRID], ids=lambda m: NAMES[m])
def test_beyond_device_memory(engine, method):
    # Every kernel-variant choice of a grid scan depends on n, c, the grid and p, not on m; each column's arithmetic is
    # independent of the others, so the peaks of 64 columns scanned on their own are those of the full scan.
    n, p, m = 20, 1 << 20, 32768
    G = synth.make_geno(n, p, seed=5000)
    K = synth.calc_kinship_host(G)
    Y = synth.make_pheno(G, K, m, seed=5001)
    Ut, lam = orc.decompose(K)
    U = np.asfortranarray(Ut.T)
    C0 = np.ones((n, 1))
    pk = peaks(engine, Y, G, C0, U, lam, None, method, reml=False)
    assert np.all(np.isfinite(pk[0])) and np.all((pk[1] >= 0) & (pk[1] < p))
    cols = np.sort(np.random.default_rng(5002).choice(m, 64, replace=False))
    Ld, Hd = dense(engine, Y[:, cols], G, C0, U, lam, None, method, reml=False)
    assert_peaks_of(Ld, Hd, tuple(a[cols] for a in pk), method)


# ---------------------------------------------------------------------------------------------------------------
# 5. Memory spaces, optional outputs, sizes at the edges, refusals
# ---------------------------------------------------------------------------------------------------------------
def raw_call(engine, space, Y, G, U, lam, method, with_marker=True, with_h2=True, chisq_df=2, grid=GRID, m=None):
    """blmm_bulkscan_peaks with raw pointers in `space`; returns (status, {name: result})"""
    import torch
    n, p = G.shape
    m = Y.shape[1] if m is None else m
    keep = []

    def inp(a):
        a = np.ascontiguousarray(np.asarray(a, dtype=np.float64).ravel(order="F"))
        if space == L.MEM_DEVICE:
            a = torch.from_numpy(a).to("cuda:0")
            keep.append(a)
            return a.data_ptr()
        keep.append(a)
        return a.ctypes.data

    outs = {}

    def out(name, dtype, want):
        if not want:
            return None
        t = torch.full((max(m, 1),), -7, dtype=dtype, device="cuda:0" if space == L.MEM_DEVICE else "cpu")
        outs[name] = t
        return t.data_ptr()

    pr = L.Problem(n, p, m, 1, inp(Y), inp(G), inp(np.ones((n, 1))), inp(U), inp(lam), None)
    lod = out("lod", torch.float64, True)
    mk = out("marker", torch.int64, with_marker)
    h2 = out("h2", torch.float64, with_h2)
    pv = out("log10p", torch.float64, chisq_df > 0)
    o, _ = engine.make_opts(**kw(method, False, grid=grid), mem_space=space, chisq_df=chisq_df, log10p_out=pv)
    vp = lambda a: C.c_void_p(a) if a else None
    st = engine.lib.blmm_bulkscan_peaks(engine.h, C.byref(pr), C.byref(o), vp(lod), vp(mk), vp(h2))
    if st == L.OK:
        engine.sync()
    torch.cuda.synchronize()
    return st, {k: v.cpu().numpy()[:m] for k, v in outs.items()}


@pytest.fixture(scope="module")
def small():
    n, p, m = 79, 200, 150
    G = synth.make_geno(n, p, seed=6000)
    K = synth.calc_kinship_host(G)
    Y = synth.make_pheno(G, K, m, seed=6001)
    Ut, lam = orc.decompose(K)
    return Y, G, np.asfortranarray(Ut.T), lam


@pytest.mark.parametrize("method", METHODS, ids=lambda m: NAMES[m])
def test_device_equals_host_and_optional_outputs(engine, small, method):
    Y, G, U, lam = small
    st, h = raw_call(engine, L.MEM_HOST, Y, G, U, lam, method)
    assert st == L.OK
    st, d = raw_call(engine, L.MEM_DEVICE, Y, G, U, lam, method)
    assert st == L.OK
    for k in h:
        assert np.array_equal(h[k].view(np.int64), d[k].view(np.int64)), k
    for space in (L.MEM_HOST, L.MEM_DEVICE):
        st, r = raw_call(engine, space, Y, G, U, lam, method, with_marker=False, with_h2=False, chisq_df=0)
        assert st == L.OK and set(r) == {"lod"} and np.array_equal(bits(r["lod"]), bits(h["lod"]))
    # m = 0: nothing to do; p = 1: the only marker is every trait's peak
    st, _ = raw_call(engine, L.MEM_HOST, Y[:, :0], G, U, lam, method, m=0)
    assert st == L.OK
    st, r = raw_call(engine, L.MEM_HOST, Y, G[:, :1], U, lam, method)
    assert st == L.OK and np.all(r["marker"] == 0)


def test_refusals_leave_the_context_usable(engine, small):
    Y, G, U, lam = small
    _, before = raw_call(engine, L.MEM_HOST, Y, G, U, lam, L.METHOD_ALT_GRID)
    n, p = G.shape
    Yf, Gf, Cf = np.asfortranarray(Y), np.asfortranarray(G), np.ones((n, 1))
    pr = L.Problem(n, p, Y.shape[1], 1, Yf.ctypes.data, Gf.ctypes.data, Cf.ctypes.data, U.ctypes.data,
                   lam.ctypes.data, None)
    o, _ = engine.make_opts(**kw(L.METHOD_ALT_GRID, False))
    st = engine.lib.blmm_bulkscan_peaks(engine.h, C.byref(pr), C.byref(o), None, None, None)
    assert st == L.E_INVALID and engine.lib.blmm_last_error(engine.h).decode() == "peak_lod_out is NULL"
    st, _ = raw_call(engine, L.MEM_HOST, Y, G, U, lam, L.METHOD_ALT_GRID, grid=np.linspace(0.0, 0.9, 256))
    assert st == L.E_INVALID
    assert "255" in engine.lib.blmm_last_error(engine.h).decode()
    _, after = raw_call(engine, L.MEM_HOST, Y, G, U, lam, L.METHOD_ALT_GRID)
    for k in before:
        assert np.array_equal(before[k].view(np.int64), after[k].view(np.int64)), k


def test_python_function(engine, small):
    Y, G, U, lam = small
    K = synth.calc_kinship_host(G)
    res = bulkscan_peaks(Y, G, K, method="alt-grid", decomposition=(U, lam), output_pvals=True, chisq_df=1,
                         engine=engine)
    Ld, Hd = dense(engine, Y, G, np.ones((Y.shape[0], 1)), U, lam, None, L.METHOD_ALT_GRID, reml=False)
    assert_peaks_of(Ld, Hd, (res.lod, res.marker, res.h2), L.METHOD_ALT_GRID)
    assert np.array_equal(bits(res.log10Pvals), bits(engine.lod2log10p(res.lod, 1)))
    with pytest.raises(BlmmError):
        bulkscan_peaks(Y, G, K, method="nope", decomposition=(U, lam), engine=engine)


# ---------------------------------------------------------------------------------------------------------------
# 6. Multi-GPU context: host buffers, traits sharded
# ---------------------------------------------------------------------------------------------------------------
def test_multi_gpu(small):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    Y, G, U, lam = small
    Y = np.hstack([Y, Y[:, ::-1], Y[:, :40]])  # 340 traits: three 128-trait tiles, sharded over two GPUs
    multi = Engine(devices=[0, 1])
    try:
        C0 = np.ones((Y.shape[0], 1))
        for method in METHODS:
            Ld, Hd = dense(multi, Y, G, C0, U, lam, None, method, reml=False)
            assert_peaks_of(Ld, Hd, peaks(multi, Y, G, C0, U, lam, None, method, reml=False), method)
        st, _ = raw_call(multi, L.MEM_DEVICE, Y, G, U, lam, L.METHOD_NULL_GRID)
        assert st == L.E_INVALID
    finally:
        multi.close()
