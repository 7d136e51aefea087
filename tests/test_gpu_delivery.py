"""How the scan entry points of the C-ABI deliver their results, called with raw pointers: device-resident calls
(BLMM_MEM_DEVICE, torch tensors) and host-buffer calls (BLMM_MEM_HOST, numpy arrays) give the same bits for every
output; results land in caller matrices with a padded leading dimension without touching the padding; every argument
check reports its code and message and leaves the context usable; profiling times the scan of a call."""
import ctypes as C

import numpy as np
import pytest

import blmm_oracle as orc
from blmm_b200 import synth, _lib as L

pytestmark = pytest.mark.gpu
GRID = np.arange(10) / 10.0
N, P, M, NPERM = 79, 300, 200, 150
SENTINEL = -7.25
ZERO_NORM_MSG = "Dividing by zeros: the input vector can not contain any zeros!"
GRID_METHODS = (L.METHOD_NULL_GRID, L.METHOD_ALT_GRID)
METHODS = GRID_METHODS + (L.METHOD_NULL_EXACT,)


@pytest.fixture(scope="module")
def data():
    Y, G, K = synth.make_problem(N, P, M, seed_g=401, seed_y=402)
    Ut, lam = orc.decompose(K)
    perm = synth.make_perm_indices(N, NPERM, 7)
    return Y, G, np.asfortranarray(Ut.T), lam, perm


class Space:
    """Inputs and outputs of one call in host (numpy) or device (torch, cuda:0) memory, handed out as addresses."""

    def __init__(self, space):
        self.space = space
        self.keep = []
        self.outs = {}

    def inp(self, a, dtype=np.float64):
        a = np.ascontiguousarray(np.asarray(a, dtype=dtype).ravel(order="F"))
        if self.space == L.MEM_DEVICE:
            import torch
            a = torch.from_numpy(a).to("cuda:0")
            self.keep.append(a)
            return a.data_ptr()
        self.keep.append(a)
        return a.ctypes.data

    def out(self, name, count):
        """`count` doubles preset to SENTINEL, or NULL when count is None"""
        if count is None:
            return None
        if self.space == L.MEM_DEVICE:
            import torch
            t = torch.full((count,), SENTINEL, dtype=torch.float64, device="cuda:0")
            self.outs[name] = t
            return t.data_ptr()
        a = np.full(count, SENTINEL)
        self.outs[name] = a
        return a.ctypes.data

    def results(self):
        if self.space == L.MEM_DEVICE:
            import torch
            torch.cuda.synchronize()  # the library's stream included; its device flags are left for blmm_sync
            return {k: v.cpu().numpy() for k, v in self.outs.items()}
        return {k: v.copy() for k, v in self.outs.items()}

    def problem(self, Y, G, U, lam):
        return L.Problem(N, 0 if G is None else G.shape[1], Y.shape[1], 1, self.inp(Y),
                         None if G is None else self.inp(G), self.inp(np.ones((N, 1))), self.inp(U), self.inp(lam),
                         None)


def check(engine, st):
    engine._check(st)
    engine.sync()


def vp(a):
    return C.c_void_p(a) if a else None


def bulkscan(engine, data, space, method, ld=0, with_h2=True, chisq_df=2, Y=None):
    Yd, G, U, lam, _ = data
    Y = Yd if Y is None else Y
    S = Space(space)
    pr = S.problem(Y, G, U, lam)
    rows = ld or P
    alt = method == L.METHOD_ALT_GRID
    Lp = S.out("L", rows * M)
    H = S.out("h2", (rows * M if alt else M) if with_h2 else None)
    Pv = S.out("log10p", rows * M if chisq_df else None)
    o, keep = engine.make_opts(method=method, h2_grid=GRID, mem_space=space, ld_out=ld, chisq_df=chisq_df,
                               log10p_out=Pv)
    check(engine, engine.lib.blmm_bulkscan(engine.h, C.byref(pr), C.byref(o), vp(Lp), vp(H)))
    return S.results()


def scan_perms(engine, data, space, ld=0, with_L=True, with_max=True):
    Y, G, U, lam, perm = data
    S = Space(space)
    pr = S.problem(Y[:, :1], G, U, lam)
    rows = ld or P
    d_perm = S.inp(perm, dtype=np.int32)
    lod, Lp = S.out("lod", P), S.out("L_perms", rows * NPERM if with_L else None)
    mx = S.out("max_lod", NPERM if with_max else None)
    s2, h2 = S.out("sigma2", 1), S.out("h2", 1)
    o, _ = engine.make_opts(prior_variance=0.0, mem_space=space, ld_out=ld)
    check(engine, engine.lib.blmm_scan_perms(engine.h, C.byref(pr), C.byref(o), vp(d_perm), NPERM, vp(lod), vp(Lp),
                                             vp(mx), vp(s2), vp(h2)))
    return S.results()


def scan_null(engine, data, space, optional=True):
    Y, G, U, lam, _ = data
    S = Space(space)
    pr = S.problem(Y, G, U, lam)
    lod = S.out("lod", P * M)
    s2, h2 = S.out("sigma2", M if optional else None), S.out("h2", M if optional else None)
    o, _ = engine.make_opts(method=L.METHOD_NULL_EXACT, reml=True, prior_variance=0.0, mem_space=space)
    check(engine, engine.lib.blmm_scan_null(engine.h, C.byref(pr), C.byref(o), vp(lod), vp(s2), vp(h2)))
    return S.results()


def scan_alt(engine, data, space, optional=True):
    Y, G, U, lam, _ = data
    S = Space(space)
    pr = S.problem(Y[:, 1:2], G, U, lam)
    lod, h2e = S.out("lod", P), S.out("h2_each", P if optional else None)
    s2, h2 = S.out("sigma2", 1 if optional else None), S.out("h2", 1 if optional else None)
    o, _ = engine.make_opts(method=L.METHOD_NULL_EXACT, prior_variance=0.0, mem_space=space)
    check(engine, engine.lib.blmm_scan_alt(engine.h, C.byref(pr), C.byref(o), vp(lod), vp(h2e), vp(s2), vp(h2)))
    return S.results()


def fit_h2(engine, data, space, optional=True):
    Y, _, U, lam, _ = data
    S = Space(space)
    pr = S.problem(Y, None, U, lam)
    h2 = S.out("h2", M)
    s2, ell = S.out("sigma2", M if optional else None), S.out("ell", M if optional else None)
    o, _ = engine.make_opts(reml=True, prior_variance=0.0, mem_space=space)
    check(engine, engine.lib.blmm_fit_h2(engine.h, C.byref(pr), C.byref(o), vp(h2), vp(s2), vp(ell)))
    return S.results()


def grid_loglik(engine, data, space, Y=None):
    Yd, _, U, lam, _ = data
    Y = Yd if Y is None else Y
    S = Space(space)
    pr = S.problem(Y, None, U, lam)
    ell = S.out("ell", len(GRID) * M)
    o, keep = engine.make_opts(h2_grid=GRID, mem_space=space)
    st = engine.lib.blmm_grid_loglik(engine.h, C.byref(pr), C.byref(o), vp(ell))
    assert st == L.OK, engine.lib.blmm_last_error(engine.h).decode()
    return S.results()


def assert_same(host, dev):
    assert host.keys() == dev.keys()
    for k in host:
        assert np.array_equal(host[k], dev[k]), k
        assert not np.any(host[k] == SENTINEL), k  # every entry was written


@pytest.mark.parametrize("method", METHODS)
def test_bulkscan_device_equals_host(engine, data, method):
    assert_same(bulkscan(engine, data, L.MEM_HOST, method), bulkscan(engine, data, L.MEM_DEVICE, method))
    if method in GRID_METHODS:  # no h2 output requested
        h = bulkscan(engine, data, L.MEM_HOST, method, with_h2=False)
        assert_same(h, bulkscan(engine, data, L.MEM_DEVICE, method, with_h2=False))


@pytest.mark.parametrize("with_L,with_max", [(True, True), (False, True), (True, False), (False, False)])
def test_scan_perms_device_equals_host(engine, data, with_L, with_max):
    h = scan_perms(engine, data, L.MEM_HOST, with_L=with_L, with_max=with_max)
    assert_same(h, scan_perms(engine, data, L.MEM_DEVICE, with_L=with_L, with_max=with_max))
    full = scan_perms(engine, data, L.MEM_HOST)
    for k in h:
        assert np.array_equal(h[k], full[k]), k


@pytest.mark.parametrize("optional", [True, False])
def test_exact_scans_device_equal_host(engine, data, optional):
    assert_same(scan_null(engine, data, L.MEM_HOST, optional), scan_null(engine, data, L.MEM_DEVICE, optional))
    assert_same(scan_alt(engine, data, L.MEM_HOST, optional), scan_alt(engine, data, L.MEM_DEVICE, optional))


@pytest.mark.parametrize("optional", [True, False])
def test_fit_h2_device_equals_host(engine, data, optional):
    h = fit_h2(engine, data, L.MEM_HOST, optional)
    assert_same(h, fit_h2(engine, data, L.MEM_DEVICE, optional))
    assert np.array_equal(h["h2"], fit_h2(engine, data, L.MEM_HOST)["h2"])


def test_grid_loglik_device_equals_host(engine, data):
    assert_same(grid_loglik(engine, data, L.MEM_HOST), grid_loglik(engine, data, L.MEM_DEVICE))
    engine.sync()


def padded(a, ld, cols):
    return a.reshape(cols, ld).T


@pytest.mark.parametrize("space", [L.MEM_HOST, L.MEM_DEVICE])
@pytest.mark.parametrize("method", METHODS)
def test_bulkscan_padded_leading_dimension(engine, data, space, method):
    ld = P + 7
    ref = bulkscan(engine, data, space, method)
    r = bulkscan(engine, data, space, method, ld=ld)
    for k in ("L", "log10p") + (("h2",) if method == L.METHOD_ALT_GRID else ()):
        a = padded(r[k], ld, M)
        assert np.array_equal(a[:P], padded(ref[k], P, M)), k
        assert np.all(a[P:] == SENTINEL), k
    if method != L.METHOD_ALT_GRID:
        assert np.array_equal(r["h2"], ref["h2"])


@pytest.mark.parametrize("space", [L.MEM_HOST, L.MEM_DEVICE])
def test_scan_perms_padded_leading_dimension(engine, data, space):
    ld = P + 7
    ref = scan_perms(engine, data, space)
    r = scan_perms(engine, data, space, ld=ld)
    a = padded(r["L_perms"], ld, NPERM)
    assert np.array_equal(a[:P], padded(ref["L_perms"], P, NPERM))
    assert np.all(a[P:] == SENTINEL)
    for k in ("lod", "max_lod", "sigma2", "h2"):
        assert np.array_equal(r[k], ref[k]), k


def test_argument_checks(engine, data):
    """Code and message of each check, in the order the entry points apply them; the context stays usable."""
    Y, G, U, lam, perm = data
    S = Space(L.MEM_HOST)
    pr = S.problem(Y, G, U, lam)
    pr1 = S.problem(Y[:, :1], G, U, lam)
    pr2 = S.problem(Y[:, :2], None, U, lam)  # two traits and no markers: the one-trait check comes first
    d_perm = S.inp(perm, dtype=np.int32)
    out = [S.out(f"o{i}", P * M) for i in range(4)]
    lib, h = engine.lib, engine.h
    ref = bulkscan(engine, data, L.MEM_HOST, L.METHOD_NULL_GRID)

    def opts(**kw):
        o, keep = engine.make_opts(h2_grid=GRID, **kw)
        opts.keep.append(keep)
        return C.byref(o)
    opts.keep = []
    o0, o1 = opts(), opts(method=L.METHOD_NULL_EXACT)
    calls = {
        "bulkscan": lambda o, pr=pr, L_=out[0]: lib.blmm_bulkscan(h, C.byref(pr), o, vp(L_), vp(out[1])),
        "grid_loglik": lambda o, pr=pr, L_=out[0]: lib.blmm_grid_loglik(h, C.byref(pr), o, vp(L_)),
        "fit_h2": lambda o, pr=pr, L_=out[0]: lib.blmm_fit_h2(h, C.byref(pr), o, vp(L_), vp(out[1]), vp(out[2])),
        "scan_perms": lambda o, pr=pr1, L_=out[0]: lib.blmm_scan_perms(h, C.byref(pr), o, vp(d_perm), NPERM, vp(L_),
                                                                      vp(out[1]), vp(out[2]), vp(out[3]), None),
        "scan_null": lambda o, pr=pr, L_=out[0]: lib.blmm_scan_null(h, C.byref(pr), o, vp(L_), vp(out[1]), vp(out[2])),
        "scan_alt": lambda o, pr=pr1, L_=out[0]: lib.blmm_scan_alt(h, C.byref(pr), o, vp(L_), vp(out[1]), vp(out[2]),
                                                                  vp(out[3])),
    }
    cases = [(name, dict(o=None), L.E_INVALID, "opts is NULL") for name in calls]
    cases += [("bulkscan", dict(o=o0, L_=None), L.E_INVALID, "L_out is NULL"),
              ("bulkscan", dict(o=o1, L_=None), L.E_INVALID, "L_out is NULL"),
              ("grid_loglik", dict(o=o0, L_=None), L.E_INVALID, "ell_out is NULL"),
              ("scan_perms", dict(o=o0, L_=None), L.E_INVALID, "lod_out is NULL"),
              ("scan_null", dict(o=o1, L_=None), L.E_INVALID, "L_out is NULL"),
              ("scan_alt", dict(o=o1, L_=None), L.E_INVALID, "lod_out is NULL")]
    o_int = opts(method=L.METHOD_NULL_EXACT, optim_interval=0)
    cases += [(name, dict(o=o_int), L.E_INVALID, "optim_interval must be >= 1")
              for name in ("bulkscan", "fit_h2", "scan_perms", "scan_null", "scan_alt")]
    for method in METHODS:
        cases.append(("bulkscan", dict(o=opts(method=method, ld_out=P - 1)), L.E_INVALID, "ld_out < p"))
    cases += [("scan_perms", dict(o=opts(ld_out=P - 1)), L.E_INVALID, "ld_out < p"),
              ("scan_null", dict(o=opts(method=L.METHOD_NULL_EXACT, ld_out=P - 1)), L.E_INVALID, "ld_out < p"),
              ("scan_perms", dict(o=o0, pr=pr2), L.E_ONE_TRAIT, "Can only handle one trait."),
              ("scan_alt", dict(o=o1, pr=pr2), L.E_ONE_TRAIT, "Can only handle one trait.")]
    for name, kw, code, msg in cases:
        st = calls[name](**kw)
        assert (st, lib.blmm_last_error(h).decode()) == (code, msg), (name, kw)
        engine.sync()
    assert_same(ref, bulkscan(engine, data, L.MEM_HOST, L.METHOD_NULL_GRID))


def test_grid_loglik_zero_trait(engine, data):
    """An all-zero trait is an error for the scans (colDivide!) but not for the grid log-likelihoods; a host-buffer
    grid_loglik clears the device flag it raises, a device-resident one leaves it for the next blmm_sync."""
    from blmm_b200 import BlmmError
    Y = data[0].copy()
    Y[:, 3] = 0.0
    host = grid_loglik(engine, data, L.MEM_HOST, Y=Y)
    engine.sync()
    dev = grid_loglik(engine, data, L.MEM_DEVICE, Y=Y)
    with pytest.raises(BlmmError) as e:
        engine.sync()
    assert (e.value.code, e.value.msg) == (L.E_ZERO_NORM, ZERO_NORM_MSG)
    assert np.array_equal(host["ell"], dev["ell"], equal_nan=True)
    ok = np.delete(host["ell"].reshape(M, len(GRID)), 3, axis=0)
    assert np.array_equal(ok, np.delete(grid_loglik(engine, data, L.MEM_HOST)["ell"].reshape(M, len(GRID)), 3, 0))
    with pytest.raises(BlmmError) as e:
        bulkscan(engine, data, L.MEM_HOST, L.METHOD_NULL_GRID, Y=Y)
    assert (e.value.code, e.value.msg) == (L.E_ZERO_NORM, ZERO_NORM_MSG)
    engine.sync()


def test_profiling_times_the_scan(engine, data):
    engine.set_profiling(True)
    try:
        for method in (L.METHOD_ALT_GRID, L.METHOD_NULL_EXACT):
            bulkscan(engine, data, L.MEM_DEVICE, method)
            assert engine.last_scan_ms() > 0, method
    finally:
        engine.set_profiling(False)
    assert engine.last_scan_ms() == -1.0
