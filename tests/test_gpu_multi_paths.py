"""Multi-GPU context (blmm_create_multi) paths that tests/test_gpu_multi.py does not reach: the optional outputs and
inputs of the device-resident (NCCL) calls, caller leading dimensions of host-buffer results, the p-values of the
sharded peaks, and the refusals that come before any GPU work.  Every result is compared bit for bit with the same
call on the one-GPU context; the tests skip below two GPUs."""
import ctypes as C

import numpy as np
import pytest

import blmm_oracle as orc
from blmm_b200 import synth, _lib as L

pytestmark = pytest.mark.gpu

GRID = np.arange(10) / 10.0
SENTINEL = -7.0  # no LOD, -log10 p or h2 takes this value: outputs are filled with it to show what was not written
METHODS = {"null-grid": L.METHOD_NULL_GRID, "alt-grid": L.METHOD_ALT_GRID, "null-exact": L.METHOD_NULL_EXACT}


@pytest.fixture(scope="module")
def multi():
    import torch
    from blmm_b200 import Engine
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    eng = Engine(devices=list(range(min(n, 8))))
    yield eng
    eng.close()


@pytest.fixture(scope="module")
def data():
    """1100 traits: nine 128-trait tiles, ragged over 2..8 GPUs"""
    n, p, m = 79, 300, 1100
    G = synth.make_geno(n, p, seed=7000)
    K = synth.calc_kinship_host(G)
    Y = synth.make_pheno(G, K, m, seed=7001)
    Ut, lam = orc.decompose(K)
    w = np.random.default_rng(7002).uniform(0.5, 2.0, n)
    return Y, G, np.asfortranarray(Ut.T), lam, w


class Buffers:
    """Column-major inputs and sentinel-filled outputs in one memory space, kept alive for the call."""

    def __init__(self, space):
        self.space, self.keep, self.outs = space, [], {}

    def _place(self, t):
        if self.space == L.MEM_DEVICE:
            t = t.to("cuda:0")
        self.keep.append(t)
        return t

    def inp(self, a, dtype=np.float64):
        import torch
        if a is None:
            return None
        a = np.ascontiguousarray(np.asarray(a, dtype=dtype).ravel(order="F"))
        return self._place(torch.from_numpy(a)).data_ptr()

    def out(self, name, size, want=True, dtype=None):
        import torch
        if not want:
            return None
        dtype = dtype or torch.float64
        t = self._place(torch.full((max(size, 1),), SENTINEL, dtype=dtype))
        self.outs[name] = t
        return t.data_ptr()

    def problem(self, Y, G, U, lam, w=None, c=1):
        n = G.shape[0]
        return L.Problem(n, G.shape[1], Y.shape[1], c, self.inp(Y), self.inp(G), self.inp(np.ones((n, max(c, 1)))),
                         self.inp(U), self.inp(lam), self.inp(w))

    def finish(self, eng, st):
        import torch
        if st == L.OK:
            eng.sync()
        torch.cuda.synchronize()
        err = eng.lib.blmm_last_error(eng.h).decode()
        return st, err, {k: v.cpu().numpy() for k, v in self.outs.items()}


def vp(a):
    return C.c_void_p(a) if a else None


def bulkscan(eng, space, Y, G, U, lam, method, w=None, c=1, ld=0, chisq_df=0, want_h2=True, want_pv=None):
    B = Buffers(space)
    p, m = G.shape[1], Y.shape[1]
    rows = ld or p
    alt = method == L.METHOD_ALT_GRID
    pr = B.problem(Y, G, U, lam, w, c)
    Lp = B.out("L", rows * m)
    Hp = B.out("h2", rows * m if alt else m, want_h2)
    Pp = B.out("log10p", rows * m, chisq_df > 0 if want_pv is None else want_pv)
    o, _ = eng.make_opts(method=method, h2_grid=GRID, mem_space=space, ld_out=ld, chisq_df=chisq_df, log10p_out=Pp)
    return B.finish(eng, eng.lib.blmm_bulkscan(eng.h, C.byref(pr), C.byref(o), vp(Lp), vp(Hp)))


def scan_perms(eng, space, y, G, U, lam, idx, ld=0, c=1, want_L=True, want_max=True):
    B = Buffers(space)
    p, nperms = G.shape[1], idx.shape[1]
    pr = B.problem(y, G, U, lam, c=c)
    perm = B.inp(idx, dtype=np.int32) if nperms else None
    lod = B.out("lod", p)
    Lp = B.out("L_perms", (ld or p) * nperms, want_L)
    mx = B.out("max_lod", nperms, want_max)
    s2, h2 = B.out("sigma2", 1), B.out("h2", 1)
    o, _ = eng.make_opts(prior_variance=0.0, mem_space=space, ld_out=ld)
    return B.finish(eng, eng.lib.blmm_scan_perms(eng.h, C.byref(pr), C.byref(o), vp(perm), nperms, vp(lod), vp(Lp),
                                                 vp(mx), vp(s2), vp(h2)))


def assert_same(one, many):
    st1, err1, r1 = one
    st2, err2, r2 = many
    assert st1 == L.OK, err1
    assert st2 == L.OK, err2
    assert r1.keys() == r2.keys()
    for k in r1:
        assert np.array_equal(r1[k].view(np.int64), r2[k].view(np.int64)), k


def assert_padding_untouched(r, name, p, ld):
    a = r[name].reshape(ld, -1, order="F")
    assert np.all(a[p:] == SENTINEL), name
    assert np.all(np.isfinite(a[:p])) and not np.any(a[:p] == SENTINEL), name


# ---- device-resident calls (NCCL) ----------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["pvals", "weights", "no_h2"])
@pytest.mark.parametrize("method", ["null-grid", "alt-grid"])
def test_device_bulkscan_optional_outputs(engine, multi, data, method, variant):
    """chisq_df > 0 gathers log10p_out; observation weights are broadcast; h2_out = NULL gathers nothing for it"""
    Y, G, U, lam, w = data
    kw = dict(method=METHODS[method], w=w if variant == "weights" else None,
              chisq_df=2 if variant == "pvals" else 0, want_h2=variant != "no_h2")
    one = bulkscan(engine, L.MEM_DEVICE, Y, G, U, lam, **kw)
    many = bulkscan(multi, L.MEM_DEVICE, Y, G, U, lam, **kw)
    assert_same(one, many)
    assert multi.last_gather_ms() > 0
    assert ("log10p" in many[2]) == (variant == "pvals") and ("h2" in many[2]) == (variant != "no_h2")


@pytest.mark.parametrize("drop", ["L_perms", "max_lod"])
@pytest.mark.parametrize("nperms", [5, 300])
def test_device_perms_optional_outputs(engine, multi, data, nperms, drop):
    """either gathered output may be NULL; with 5 permutations only the primary has a tile"""
    Y, G, U, lam, _ = data
    idx = synth.make_perm_indices(G.shape[0], nperms, 17)
    kw = dict(want_L=drop != "L_perms", want_max=drop != "max_lod")
    one = scan_perms(engine, L.MEM_DEVICE, Y[:, :1], G, U, lam, idx, **kw)
    many = scan_perms(multi, L.MEM_DEVICE, Y[:, :1], G, U, lam, idx, **kw)
    assert_same(one, many)
    assert drop not in many[2]


# ---- host buffers with a leading dimension of the caller's --------------------------------------------------
@pytest.mark.parametrize("method", ["alt-grid", "null-grid"])
def test_host_bulkscan_ld_out(engine, multi, data, method):
    Y, G, U, lam, _ = data
    p = G.shape[1]
    ld = p + 7
    kw = dict(method=METHODS[method], ld=ld, chisq_df=2 if method == "alt-grid" else 0)
    one = bulkscan(engine, L.MEM_HOST, Y, G, U, lam, **kw)
    many = bulkscan(multi, L.MEM_HOST, Y, G, U, lam, **kw)
    assert_same(one, many)
    for name in ("L", "h2", "log10p") if method == "alt-grid" else ("L",):
        assert_padding_untouched(many[2], name, p, ld)


def test_host_scan_null_ld_out(engine, multi, data):
    Y, G, U, lam, _ = data
    p, m = G.shape[1], Y.shape[1]
    ld = p + 7
    res = []
    for eng in (engine, multi):
        B = Buffers(L.MEM_HOST)
        pr = B.problem(Y, G, U, lam)
        lod, s2, h2 = B.out("lod", ld * m), B.out("sigma2", m), B.out("h2", m)
        pv = B.out("log10p", ld * m)
        o, _ = eng.make_opts(method=L.METHOD_NULL_EXACT, prior_variance=0.0, ld_out=ld, chisq_df=1, log10p_out=pv)
        res.append(B.finish(eng, eng.lib.blmm_scan_null(eng.h, C.byref(pr), C.byref(o), vp(lod), vp(s2), vp(h2))))
    assert_same(*res)
    for name in ("lod", "log10p"):
        assert_padding_untouched(res[1][2], name, p, ld)


def test_host_perms_ld_out(engine, multi, data):
    Y, G, U, lam, _ = data
    p = G.shape[1]
    ld = p + 7
    idx = synth.make_perm_indices(G.shape[0], 700, 18)
    one = scan_perms(engine, L.MEM_HOST, Y[:, 1:2], G, U, lam, idx, ld=ld)
    many = scan_perms(multi, L.MEM_HOST, Y[:, 1:2], G, U, lam, idx, ld=ld)
    assert_same(one, many)
    assert_padding_untouched(many[2], "L_perms", p, ld)


@pytest.mark.parametrize("method", list(METHODS))
def test_host_peaks_pvals(engine, multi, data, method):
    """the per-trait -log10 p of the sharded peaks land at each block's own traits"""
    import torch
    Y, G, U, lam, _ = data
    m = Y.shape[1]
    res = []
    for eng in (engine, multi):
        B = Buffers(L.MEM_HOST)
        pr = B.problem(Y, G, U, lam)
        lod, mk, h2 = B.out("lod", m), B.out("marker", m, dtype=torch.int64), B.out("h2", m)
        pv = B.out("log10p", m)
        o, _ = eng.make_opts(method=METHODS[method], h2_grid=GRID, chisq_df=2, log10p_out=pv,
                             prior_variance=0.0 if method == "null-exact" else 1.0)
        res.append(B.finish(eng, eng.lib.blmm_bulkscan_peaks(eng.h, C.byref(pr), C.byref(o), vp(lod), vp(mk),
                                                             vp(h2))))
    assert_same(*res)
    assert not np.any(res[1][2]["log10p"] == SENTINEL)


# ---- refusals before any GPU work ---------------------------------------------------------------------------
LD_MSG = "multi-GPU device-resident calls need ld_out == p (contiguous slabs)"
BAD_MSG = "bad problem (NULL input or covariate count)"
HOST_ONLY_MSG = "multi-GPU contexts take device pointers in blmm_bulkscan and blmm_scan_perms only"


def test_device_refusals(multi, data):
    Y, G, U, lam, _ = data
    p = G.shape[1]
    idx = synth.make_perm_indices(G.shape[0], 10, 19)
    cases = [
        (bulkscan(multi, L.MEM_DEVICE, Y, G, U, lam, L.METHOD_NULL_GRID, ld=p + 7), LD_MSG),
        (scan_perms(multi, L.MEM_DEVICE, Y[:, :1], G, U, lam, idx, ld=p + 7), LD_MSG),
        (bulkscan(multi, L.MEM_DEVICE, Y, G, U, lam, L.METHOD_NULL_GRID, c=0), BAD_MSG),
        (scan_perms(multi, L.MEM_DEVICE, Y[:, :1], G, U, lam, idx, c=0), BAD_MSG),
        (bulkscan(multi, L.MEM_DEVICE, Y, G, U, lam, L.METHOD_NULL_GRID, chisq_df=2, want_pv=False),
         "chisq_df > 0 but log10p_out is NULL"),
    ]
    for (st, err, _), msg in cases:
        assert st == L.E_INVALID and err == msg


def test_host_only_entry_points_refuse_device_pointers(multi, data):
    Y, G, U, lam, _ = data
    p, m = G.shape[1], Y.shape[1]
    B = Buffers(L.MEM_HOST)
    pr = B.problem(Y, G, U, lam)
    o, _ = multi.make_opts(h2_grid=GRID, mem_space=L.MEM_DEVICE)
    a, b, c = B.out("a", p * m), B.out("b", m), B.out("c", len(GRID) * m)
    lib, h = multi.lib, multi.h
    for st in (lib.blmm_fit_h2(h, C.byref(pr), C.byref(o), vp(b), vp(b), vp(b)),
               lib.blmm_scan_null(h, C.byref(pr), C.byref(o), vp(a), vp(b), vp(b)),
               lib.blmm_grid_loglik(h, C.byref(pr), C.byref(o), vp(c))):
        assert st == L.E_INVALID and lib.blmm_last_error(h).decode() == HOST_ONLY_MSG
