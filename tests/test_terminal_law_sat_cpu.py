"""The saturated, affine and per-instance terminal law (wshmpc_fallback.law_sets / d_law_k / d_law_lo / d_law_hi,
ClosedLoop(..., law_gain, law_offset, law_bounds)) on the host: a long-double statement of the law that the GPU tests replay,
the input box of the model's stage rows, the gain on another model, the plant's discrete model, and the argument checks of
ClosedLoop, Handle.new_fallback and the C struct that need no GPU."""
import ctypes as C
import numpy as np
import pytest

from tests.test_terminal_law_cpu import fallback_reference


def law_input_reference(K, x, k=None, lo=None, hi=None):
    """u = sat_[lo, hi](K_i x + k_i) of n instances in np.longdouble (include/wshmpc.h, wshmpc_fallback).  K [nu, nx] or
    [n, nu, nx], x [n, nx], k None, [nu] or [n, nu], lo and hi None or [nu].  Returns (u [n, nu] long double, terms [n, nu]
    the sums of the magnitudes of the products and the offset each unclamped entry is summed from, clamped [n, nu] bool:
    the entries whose unclamped value lies beyond a bound by more than the rounding of that sum, so that the device's value
    is the bound itself)."""
    ld = np.longdouble
    x = np.asarray(x, dtype=float)
    n = x.shape[0]
    K = np.broadcast_to(np.asarray(K, dtype=float), (n,) + np.shape(K)[-2:])
    u = np.einsum('irc,ic->ir', K.astype(ld), x.astype(ld))
    terms = np.einsum('irc,ic->ir', np.abs(K), np.abs(x))
    if k is not None:
        kk = np.broadcast_to(np.asarray(k, dtype=float), u.shape)
        u = u + kk.astype(ld)
        terms = terms + np.abs(kk)
    clamped = np.zeros(u.shape, bool)
    if lo is not None:
        lo_, hi_ = (np.broadcast_to(np.asarray(b, dtype=float), u.shape) for b in (lo, hi))
        err = 1e-14 * terms
        clamped = (u < lo_.astype(ld) - err) | (u > hi_.astype(ld) + err)
        u = np.where(u < lo_, lo_.astype(ld), np.where(u > hi_, hi_.astype(ld), u))      # NaN passes through
        terms = np.where(clamped, 0., terms)
    return u, terms, clamped


def fallback_reference_sat(A, B, K, T, H, L, live, status, cost, age, law_n, x, plan, inc, k=None, lo=None, hi=None):
    """fallback_reference (tests/test_terminal_law_cpu.py) with the law of law_input_reference on its law steps: the same
    dict, with u, x1, u_terms and x1_terms of the law steps from the saturated law, and 'clamped' [n, nu] (False off the
    law steps)."""
    nu, nx = np.shape(B)[1], np.shape(A)[0]
    ref = fallback_reference(A, B, np.zeros((nu, nx)), T, H, L, live, status, cost, age, law_n, x, plan, inc)
    ref['clamped'] = np.zeros((len(ref['source']), nu), bool)
    idx = np.nonzero(ref['source'] == 2)[0]
    if idx.size == 0:
        return ref
    ld = np.longdouble
    Ks = np.asarray(K, dtype=float)
    Ks = Ks[idx] if Ks.ndim == 3 else Ks
    ks = None if k is None else (np.asarray(k, dtype=float)[idx] if np.ndim(k) == 2 else k)
    xi = np.asarray(x, dtype=float)[idx]
    u, u_terms, clamped = law_input_reference(Ks, xi, ks, lo, hi)
    ref['u'][idx] = u
    ref['u_terms'][idx] = u_terms
    ref['clamped'][idx] = clamped
    ref['x1'][idx] = xi.astype(ld).dot(np.asarray(A, dtype=ld).T) + u.dot(np.asarray(B, dtype=ld).T)
    # the device forms u in double first: its rounding reaches x_1 through B
    ref['x1_terms'][idx] = np.abs(xi).dot(np.abs(A).T) + (np.abs(u.astype(float)) + u_terms).dot(np.abs(B).T)
    return ref


# ---- the numpy statement of the law ----------------------------------------------------------------------------------------
def test_law_reference_hand_built():
    inf = np.inf
    K = np.array([[2., 0.], [0., -1.], [1., 1.]])                 # nu = 3, nx = 2
    x = np.array([[1., 0.5], [-3., 4.], [0.25, -0.25], [np.nan, 1.]])
    lo, hi = np.array([-1., -inf, 0.]), np.array([1., 0., inf])
    u, terms, cl = law_input_reference(K, x, None, lo, hi)
    # K x = [2, -0.5, 1.5], [-6, -4, 1], [0.5, 0.25, 0], [nan, nan, nan] (0 * nan is nan)
    assert u[0].astype(float).tolist() == [1., -0.5, 1.5] and cl[0].tolist() == [True, False, False]
    assert u[1].astype(float).tolist() == [-1., -4., 1.] and cl[1].tolist() == [True, False, False]
    assert u[2].astype(float).tolist() == [0.5, 0., 0.] and cl[2].tolist() == [False, True, False]   # 0.25 > hi = 0
    assert np.isnan(u[3].astype(float)).all() and not cl[3].any()                  # NaN passes the clamp
    assert terms[0].tolist() == [0., 0.5, 1.5] and terms[2].tolist() == [0.5, 0., 0.5]
    # -inf / +inf bounds leave the law linear
    u2, t2, c2 = law_input_reference(K, x[:3], None, np.full(3, -inf), np.full(3, inf))
    u3, t3, _ = law_input_reference(K, x[:3])
    assert np.array_equal(u2, u3) and np.array_equal(t2, t3) and not c2.any()
    # an offset, shared and per instance
    k = np.array([-1., 0.5, -2.])
    u4, t4, c4 = law_input_reference(K, x[:3], k, lo, hi)
    # K x + k = [1, 0, -0.5]: on the upper bounds (not clamped), below the lower one
    assert u4[0].astype(float).tolist() == [1., 0., 0.] and c4[0].tolist() == [False, False, True]
    assert t4[0].tolist() == [3., 1., 0.]
    kk = np.array([[0., 0., 0.], [8., 0., 0.], [0., 0., 10.]])
    u5, _, c5 = law_input_reference(K, x[:3], kk, lo, hi)
    assert u5[:, 0].astype(float).tolist() == [1., 1., 0.5] and u5[2, 2] == 10. and c5[1, 0] and not c5[1, 1:].any()
    assert c5[2].tolist() == [False, True, False]
    # per-instance gains: set i for instance i
    Ki = np.stack([K, -K, 2. * K])
    u6, _, _ = law_input_reference(Ki, x[:3])
    assert u6[0].astype(float).tolist() == [2., -0.5, 1.5] and u6[1].astype(float).tolist() == [6., 4., -1.]
    assert u6[2].astype(float).tolist() == [1., 0.5, 0.]


def test_law_reference_clamps_at_the_bound_itself():
    """a value just inside a bound is not clamped; one beyond it by more than its rounding is, and becomes the bound"""
    K = np.array([[1., 1.]])
    lo, hi = np.array([-1.]), np.array([1.])
    x = np.array([[0.5, 0.5], [0.5, 0.5 + 1e-12], [-0.5, -0.5 - 1e-12], [0.5, 0.5 - 1e-12]])
    u, _, cl = law_input_reference(K, x, None, lo, hi)
    assert cl[:, 0].tolist() == [False, True, True, False]
    assert float(u[1, 0]) == 1. and float(u[2, 0]) == -1. and float(u[3, 0]) < 1.


def test_fallback_reference_sat_on_the_policy_grid():
    """the saturated reference on CP20: the policy and the plan steps are fallback_reference's, the law steps apply the
    saturated law; without offset and bounds and with one set it is fallback_reference"""
    from oracle.models import load_model
    model = load_model('cp20')
    A, B = model['A'], model['B']
    T, nx, nu, H, L = int(model['T']), A.shape[0], B.shape[1], 3, 2
    P, U = (T + 1) * nx + T * nu, (T + 1) * nx
    grid = [(lv, hi, st, a, n) for lv in (0, 1) for hi in (0, 1) for st in (0, 1, 2, 3) for a in (-1, 0, 2, 3)
            for n in (0, 1, 2) if not (hi and st == 1)]
    N = len(grid)
    lv, hi, st, age, law_n = (np.array(c) for c in zip(*grid))
    rng = np.random.default_rng(0)
    x = rng.standard_normal((N, nx))
    plan = rng.standard_normal((N, P)); inc = rng.standard_normal((N, P))
    cost = np.where(hi == 1, rng.uniform(1., 2., N), np.inf)
    K = rng.standard_normal((nu, nx))
    base = fallback_reference(A, B, K, T, H, L, lv, st, cost, age, law_n, x, plan, inc)
    same = fallback_reference_sat(A, B, K, T, H, L, lv, st, cost, age, law_n, x, plan, inc)
    for key in ('source', 'hold', 'active', 'age', 'law_n', 'app_cost', 'plan', 'u_terms', 'x1_terms'):
        assert np.array_equal(base[key], same[key]), key
    for key in ('u', 'x1'):
        assert np.array_equal(np.isnan(base[key]), np.isnan(same[key])) and np.allclose(
            base[key][~np.isnan(base[key])].astype(float), same[key][~np.isnan(same[key])].astype(float), rtol=1e-15, atol=0)
    Ki = K[None] * rng.uniform(.5, 1.5, (N, 1, 1))
    k = rng.standard_normal((N, nu)) * .1
    lo, hi = -np.full(nu, .8), np.full(nu, .8)
    lo[2], hi[3] = -np.inf, np.inf
    r = fallback_reference_sat(A, B, Ki, T, H, L, lv, st, cost, age, law_n, x, plan, inc, k, lo, hi)
    assert np.array_equal(r['hold'], base['hold']) and np.array_equal(r['law_n'], base['law_n'])
    law = r['source'] == 2
    assert law.any() and r['clamped'][law].any() and (~r['clamped'][law]).any() and not r['clamped'][~law].any()
    for i in np.nonzero(law)[0]:
        v = Ki[i].dot(x[i]) + k[i]
        want = np.clip(v, lo, hi)
        assert np.allclose(r['u'][i].astype(float), want, rtol=1e-14, atol=1e-15)
        assert np.array_equal(r['u'][i][r['clamped'][i]].astype(float), want[r['clamped'][i]])
        assert np.allclose(r['x1'][i].astype(float), A.dot(x[i]) + B.dot(want), rtol=1e-13, atol=1e-14)
    for i in np.nonzero(r['source'] == 1)[0]:
        assert np.array_equal(r['u'][i], base['u'][i])


# ---- the controller and the plant ------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def ctl():
    from oracle.models import load_model
    from tests.util import make_controller
    return make_controller(load_model('cp20'))


def test_input_box_of_cp20(ctl):
    lo, hi = ctl.input_box()
    nu = ctl.mld.nu
    assert lo.shape == hi.shape == (nu,)
    assert lo[0] == -1. and hi[0] == 1.                              # |fc| <= 1
    assert lo[1] == 0. and lo[2] == 0. and hi[1] == np.inf and hi[2] == np.inf      # fl, fr >= 0
    assert np.all(lo[3:] == -np.inf) and np.all(hi[3:] == np.inf)
    F, G = ctl.mld.F, ctl.mld.G
    rows = np.nonzero(np.all(F == 0., axis=1) & (np.count_nonzero(G, axis=1) == 1))[0]
    assert rows.tolist() == [8, 9, 14, 23]


def test_input_box_keeps_the_tightest_bound():
    from warm_start_hmpc_b200.controller import HybridModelPredictiveController
    c = HybridModelPredictiveController.__new__(HybridModelPredictiveController)

    class M(object):
        nu, nx = 3, 2
        F = np.array([[0., 0.], [0., 0.], [0., 0.], [1., 0.], [0., 0.]])
        G = np.array([[2., 0., 0.], [4., 0., 0.], [0., -1., 0.], [0., 0., 1.], [0., 1., 1.]])
        h = np.array([4., 4., 3., 1., 1.])
    c.mld = M
    lo, hi = c.input_box()
    assert hi.tolist() == [1., np.inf, np.inf] and lo.tolist() == [-np.inf, -3., -np.inf]


@pytest.mark.parametrize('name', ['cp20', 'cp40'])
def test_terminal_law_on_the_own_model_is_bit_identical(name):
    from oracle.models import load_model
    from tests.util import make_controller
    c = make_controller(load_model(name))
    K = c.terminal_law()
    assert np.array_equal(c.terminal_law(A=c.mld.A, B=c.mld.B), K)
    assert np.array_equal(c.terminal_law(inputs=[0], A=c.mld.A.copy(), B=c.mld.B.copy()), K)
    with pytest.raises(ValueError, match='terminal_law'):
        c.terminal_law(A=np.eye(3))
    with pytest.raises(ValueError, match='terminal_law'):
        c.terminal_law(B=c.mld.B[:, :3])


def test_discrete_model_is_the_mld_model(ctl):
    from warm_start_hmpc_b200.plants import CartPoleWithWalls
    A, B = CartPoleWithWalls().discrete_model(0.05, nu=ctl.mld.nu)
    assert A.shape == ctl.mld.A.shape and B.shape == ctl.mld.B.shape
    assert np.max(np.abs(A - ctl.mld.A)) <= 1e-12
    K = ctl.terminal_law()
    law_cols = np.nonzero(np.any(K != 0., axis=1))[0]
    assert law_cols.tolist() == [0]
    assert np.max(np.abs(B[:, law_cols] - ctl.mld.B[:, law_cols])) <= 1e-12
    assert np.max(np.abs(B[:, :3] - ctl.mld.B[:, :3])) <= 1e-12 and np.all(B[:, 3:] == 0.)
    Kp = ctl.terminal_law(A=A, B=B)
    assert np.max(np.abs(Kp - K)) <= 1e-9 * np.abs(K).max()
    # another plant, another gain: heavier pole, other law
    A2, B2 = CartPoleWithWalls(mp=1.3).discrete_model(0.05, nu=ctl.mld.nu)
    K2 = ctl.terminal_law(A=A2, B=B2)
    assert np.all(K2[1:] == 0.) and np.max(np.abs(K2 - K)) > 1e-3 * np.abs(K).max()
    assert np.max(np.abs(np.linalg.eigvals(A2 + B2.dot(K2)))) < 1.
    with pytest.raises(ValueError, match='discrete_model'):
        CartPoleWithWalls().discrete_model(0.05, nu=2)
    with pytest.raises(ValueError, match='discrete_model'):
        CartPoleWithWalls().discrete_model(0., nu=7)


# ---- argument checks -------------------------------------------------------------------------------------------------------
def test_closed_loop_argument_checks(ctl):
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    nu, nx, N = ctl.mld.nu, ctl.mld.nx, 4
    # what the linear law refused is still refused
    for K in (np.zeros((nx, nu)), np.zeros((1, nx)), np.zeros(nx), np.zeros((nu, nx, 1)), np.zeros((N + 1, nu, nx))):
        with pytest.raises(ValueError, match='law_gain'):
            ClosedLoop(ctl, N, terminal_law=5, law_gain=K)
    for k in (np.zeros(nx), np.zeros((N, nx)), np.zeros((N + 1, nu)), np.zeros((1, N, nu))):
        with pytest.raises(ValueError, match='law_offset'):
            ClosedLoop(ctl, N, terminal_law=5, law_offset=k)
    lo, hi = ctl.input_box()
    bad = [(lo[:3], hi[:3]), (np.zeros((1, nu)), np.ones((1, nu))), (hi, lo), (np.where(np.arange(nu) == 1, np.nan, lo), hi),
           (lo, np.where(np.arange(nu) == 0, np.nan, hi)), (lo, hi, hi), (lo,), 'box', 3.]
    for b in bad:
        with pytest.raises(ValueError, match='law_bounds'):
            ClosedLoop(ctl, N, terminal_law=5, law_bounds=b)
    for kw in (dict(law_offset=np.zeros(nu)), dict(law_bounds='model'), dict(law_bounds=(lo, hi))):
        with pytest.raises(ValueError, match='terminal_law > 0'):
            ClosedLoop(ctl, N, fallback=3, **kw)
    with pytest.raises(ValueError, match='comparator'):
        ClosedLoop(ctl, N, warm=False, comparator=True, terminal_law=5, law_bounds='model')


def test_check_terminal_law_accepts_the_documented_shapes():
    from warm_start_hmpc_b200.capi import check_terminal_law
    nu, nx, N = 3, 2, 5
    K, k, lo, hi = check_terminal_law(N, nu, nx, np.ones((nu, nx)))
    assert K.shape == (nu, nx) and k is None and lo is None and hi is None
    K, k, lo, hi = check_terminal_law(N, nu, nx, np.ones((N, nu, nx)), np.ones((N, nu)), [-1, -np.inf, 0], [1, np.inf, 0])
    assert K.shape == (N, nu, nx) and k.shape == (N, nu) and lo.dtype == float and hi.tolist() == [1., np.inf, 0.]
    with pytest.raises(ValueError, match='terminal law bounds: both'):
        check_terminal_law(N, nu, nx, np.ones((nu, nx)), None, np.zeros(nu), None)
    with pytest.raises(ValueError, match='terminal law gain'):
        check_terminal_law(N, nu, nx, np.ones((nx, nu)))


class _FakeHandle(object):
    """what Handle.new_fallback reads of a handle, on the CPU"""

    def __init__(self, nx, nu, primal):
        class _L(object):
            pass
        self.layout, self.pd = _L(), _L()
        self.layout.primal, self.pd.nx, self.pd.nu = primal, nx, nu
        self.torch_device = 'cpu'


def test_new_fallback_buffers_of_the_law():
    from warm_start_hmpc_b200.capi import Handle
    nx, nu, N = 2, 3, 5
    h = _FakeHandle(nx, nu, 20)
    K = np.arange(nu * nx, dtype=float).reshape(nu, nx)
    fb = Handle.new_fallback(h, N, 1, 4, K)
    assert not {'law_sets', 'law_k', 'law_lo', 'law_hi'} & set(fb) and fb['law_K'].shape == (nu, nx)
    fb = Handle.new_fallback(h, N, 1, 4, K, k=np.ones(nu), lo=-np.ones(nu), hi=np.ones(nu))
    assert 'law_sets' not in fb and fb['law_k'].tolist() == [1.] * nu and fb['law_lo'].tolist() == [-1.] * nu
    # a per-instance offset makes the gain per instance too, and the other way round
    fb = Handle.new_fallback(h, N, 1, 4, K, k=np.arange(N * nu, dtype=float).reshape(N, nu))
    assert fb['law_sets'] == N and fb['law_K'].shape == (N, nu, nx) and all(np.array_equal(fb['law_K'][i].numpy(), K) for i in range(N))
    assert fb['law_k'].is_contiguous() and fb['law_k'][2].tolist() == [6., 7., 8.]
    Ki = np.stack([K * i for i in range(N)])
    fb = Handle.new_fallback(h, N, 1, 4, Ki, k=np.ones(nu))
    assert fb['law_sets'] == N and np.array_equal(fb['law_K'].numpy(), Ki) and fb['law_k'].shape == (N, nu)
    assert fb['law_K'].is_contiguous() and fb['law_k'].is_contiguous()
    for kw, msg in ((dict(K=np.zeros((nx, nu))), 'terminal law gain'), (dict(K=K, k=np.zeros(nx)), 'terminal law offset'),
                    (dict(K=K, lo=np.zeros(nu)), 'terminal law bounds'), (dict(K=K, lo=np.ones(nu), hi=np.zeros(nu)), 'lo <= hi'),
                    (dict(K=K, lo=np.full(nu, np.nan), hi=np.ones(nu)), 'NaN')):
        with pytest.raises(ValueError, match=msg):
            Handle.new_fallback(h, N, 1, 4, **kw)
    fb = Handle.new_fallback(h, N, 1)                                # without the law: no law buffers at all
    assert fb['max_law'] == 0 and 'law_K' not in fb


class _FallbackParent(C.Structure):
    """wshmpc_fallback before the law's sets, offset and bounds"""
    _fields_ = [('max_hold', C.c_int), ('d_plan', C.c_void_p), ('d_age', C.c_void_p), ('d_app_cost', C.c_void_p),
                ('d_app_primal', C.c_void_p), ('d_hold', C.c_void_p), ('max_law', C.c_int), ('d_law_K', C.c_void_p),
                ('d_law_n', C.c_void_p)]


def test_fallback_struct_without_the_new_keys_is_the_previous_one():
    import torch
    from warm_start_hmpc_b200 import capi
    N, P = 5, 224
    f64, i32 = dict(dtype=torch.float64), dict(dtype=torch.int32)
    fb = dict(max_hold=3, plan=torch.zeros((N, P), **f64), age=torch.full((N,), -1, **i32),
              app_cost=torch.zeros(N, **f64), app_primal=torch.zeros((N, P), **f64))
    K, n, hold = torch.zeros((3, 4), **f64), torch.zeros(N, **i32), torch.zeros(N, **i32)
    for d in (fb, dict(fb, max_law=7, law_K=K, law_n=n)):
        c = capi._fallback_struct(d, hold)
        old = _FallbackParent()
        for name, _ in _FallbackParent._fields_:
            setattr(old, name, getattr(c, name))
        raw = C.string_at(C.addressof(c), C.sizeof(c))
        assert raw[:C.sizeof(old)] == C.string_at(C.addressof(old), C.sizeof(old))
        assert raw[C.sizeof(old):] == bytes(C.sizeof(c) - C.sizeof(old))          # a zero tail: the law of one shared gain
    # the tail follows the parent's layout: every earlier field keeps its offset
    for name, _ in _FallbackParent._fields_:
        assert getattr(capi._Fallback, name).offset == getattr(_FallbackParent, name).offset
    # with the new keys
    k, lo, hi = torch.zeros(3, **f64), torch.zeros(3, **f64), torch.ones(3, **f64)
    c = capi._fallback_struct(dict(fb, max_law=7, law_K=K, law_n=n, law_sets=N, law_k=k, law_lo=lo, law_hi=hi), hold)
    assert c.law_sets == N and c.d_law_k == k.data_ptr() and c.d_law_lo == lo.data_ptr() and c.d_law_hi == hi.data_ptr()
    assert c.max_law == 7 and c.d_law_K == K.data_ptr() and c.d_hold == hold.data_ptr()
