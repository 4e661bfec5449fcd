"""-m gpu: the saturated, affine and per-instance terminal law (wshmpc_fallback.law_sets / d_law_k / d_law_lo / d_law_hi,
ClosedLoop(..., terminal_law=L, law_gain, law_offset, law_bounds)).

* with one set, no offset and no bounds spelled out (law_sets = 1), and with per-instance gains that all equal K, the FB
  loop's logs, final states and trees are those of the shared linear law, bit for bit;
* with all three on, the fused loop equals lock step bit for bit (step(), and step_with_plant with the device plant as
  callback): linear and device plant, warm and cold, one and two lanes; the pinned batches take law steps whose K x is
  clamped, and every law step applies u0 = sat(K_i x + k_i) and x_1|t = A x + B u0;
* wshmpc_fallback_step matches the long-double reference: clamped entries exactly, the others within the rounding of their
  sums, NaN passing through;
* the tree of an infeasible step shifted with a clamped law input equals the host construct_warm_start;
* the error paths of the new fields fail with a message.
"""
import ctypes as C
import os
import numpy as np
import pytest
import torch

from oracle.models import load_model, MODELS
from tests.util import make_controller
from tests.test_gpu_fallback import DT, KEYS, _loop, _heavy_plants, _noise, _lock, _equal
from tests.test_terminal_law_cpu import LAW, replay_law
from tests.test_terminal_law_sat_cpu import law_input_reference, fallback_reference_sat

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def cp20():
    model = load_model('cp20')
    return model, make_controller(model)


def _batch(model, case, N, S, seed):
    if case.startswith('plant'):
        plant, x0 = _heavy_plants(model, N)
        return plant, x0, None
    return None, np.load(os.path.join(MODELS, 'cp20_instances.npy'))[:N], _noise(model, S, N, .02, seed)


def _sat_law(ctl, N, plant_case):
    """all three features: a gain per instance (for the heavy plants the DARE gain of each plant's own model, as
    _heavy_plants builds them; otherwise K scaled per instance), an offset on the cart force, and the model's input box"""
    from warm_start_hmpc_b200.plants import CartPoleWithWalls
    nu = ctl.mld.nu
    if plant_case:
        Ks = np.stack([ctl.terminal_law(A=A, B=B) for A, B in
                       (CartPoleWithWalls(mp=m).discrete_model(DT, nu) for m in np.linspace(1.15, 1.3, N))])
    else:
        Ks = ctl.terminal_law()[None] * np.linspace(.8, 1.2, N)[:, None, None]
    k = np.zeros(nu); k[0] = 0.05
    return dict(law_gain=Ks, law_offset=k, law_bounds='model')


def _trees_equal(a, b):
    """the nodes and records in use of two trees, bit for bit"""
    assert torch.equal(a.n_nodes, b.n_nodes) and torch.equal(a.n_recs, b.n_recs)
    nodes = torch.arange(a.cap_nodes, device=a.n_nodes.device)[None] < a.n_nodes[:, None].long()
    recs = torch.arange(a.cap_recs, device=a.n_recs.device)[None] < a.n_recs[:, None].long()
    for k in ('depth', 'alive', 'rec', 'bits', 'mask', 'lb'):
        assert torch.equal(getattr(a, k)[nodes], getattr(b, k)[nodes]), k
    for k in ('rec_dobj', 'rec_dual'):
        assert torch.equal(getattr(a, k)[recs], getattr(b, k)[recs]), k


def _check_sat_law_steps(model, law, xs, hold, u0, x1=None):
    """every law step (hold == -2) applied u0 = sat(K_i x + k_i): the entries the reference clamps exactly, the others to
    the rounding of their sums (and x_1|t = A x + B u0 where x1 is given).  law: dict(K [n, nu, nx], k, lo, hi).  Returns
    (law steps checked, law steps with a clamped entry)."""
    A, B = model['A'], model['B']
    t_i = np.argwhere(hold == LAW)
    n_clamped = 0
    for t, i in t_i:
        x = xs[t, i][None]
        u, terms, cl = law_input_reference(law['K'][i], x, law['k'], law['lo'], law['hi'])
        u, terms, cl, got = u[0], terms[0], cl[0], u0[t, i]
        assert np.array_equal(got[cl], u[cl].astype(float)), (t, i)
        assert np.all(np.abs(got[~cl] - u[~cl].astype(float)) <= 1e-14 * terms[~cl]), (t, i)
        n_clamped += int(cl.any())
        if x1 is not None:
            want = A.dot(x[0]) + B.dot(got)
            assert np.all(np.abs(x1[t, i] - want) <= 1e-14 * (np.abs(A).dot(np.abs(x[0])) + np.abs(B).dot(np.abs(got)))), (t, i)
    return len(t_i), n_clamped


def _law_of(ctl, N, kw):
    lo, hi = ctl.input_box()
    K = np.broadcast_to(np.asarray(kw['law_gain'], dtype=float), (N, ctl.mld.nu, ctl.mld.nx))
    return dict(K=K, k=kw['law_offset'], lo=lo, hi=hi)


# ---- the defaults are the linear law of one shared gain --------------------------------------------------------------------
@pytest.mark.parametrize('case, HL', [('linear_warm', (3, 5)), ('plant_warm', (0, 5)), ('plant_cold', (19, 50))])
def test_one_set_and_equal_per_instance_gains_are_the_shared_law(cp20, case, HL):
    model, ctl = cp20
    H, L = HL
    N = 64
    S = 40 if case.startswith('plant') and H == 19 else 30
    warm = case.endswith('warm')
    plant, x0, e = _batch(model, case, N, S, 7)
    K = ctl.terminal_law()
    runs = []
    for how in ('shared', 'law_sets_1', 'per_instance'):
        F = _loop(ctl, N, warm, H, plant=plant, n_slots=N, terminal_law=L,
                  law_gain=np.repeat(K[None], N, 0) if how == 'per_instance' else None)
        if how == 'law_sets_1':
            F.fb['law_sets'] = 1
        for tr in F.trees:
            tr.rec_dual.zero_()                  # allocated uninitialised: no stale bits in the padding of a record
        assert F.fb.get('law_sets', 0) == {'shared': 0, 'law_sets_1': 1, 'per_instance': N}[how]
        F.reset(x0)
        logs = F.run(S, e=e)
        torch.cuda.synchronize()
        runs.append(({k: v.clone() for k, v in logs.items()}, F))
    (a, Fa) = runs[0]
    assert (a['hold'].cpu().numpy() == LAW).any()
    for b, Fb in runs[1:]:
        _equal(a, b)
        assert torch.equal(Fa.x, Fb.x) and torch.equal(Fa.active, Fb.active) and Fa.cur == Fb.cur
        assert torch.equal(Fa.fb['law_n'], Fb.fb['law_n']) and torch.equal(Fa.fb['app_primal'], Fb.fb['app_primal'])
        for ta, tb in zip(Fa.trees, Fb.trees):
            _trees_equal(ta, tb)


# ---- fused equals lock step with all three features on --------------------------------------------------------------------
@pytest.mark.parametrize('HL', [(0, 5), (3, 5), (19, 50)])
@pytest.mark.parametrize('case', ['linear_warm', 'linear_cold', 'plant_warm', 'plant_cold'])
def test_fused_equals_lock_step_one_lane(cp20, HL, case):
    model, ctl = cp20
    H, L = HL
    N = 64
    S = 40 if case.startswith('plant') and H == 19 else 30
    warm = case.endswith('warm')
    plant, x0, e = _batch(model, case, N, S, 7)
    kw = _sat_law(ctl, N, plant is not None)
    F = _loop(ctl, N, warm, H, plant=plant, n_slots=N, terminal_law=L, **kw)
    assert F.fb['law_sets'] == N and 'law_k' in F.fb and 'law_lo' in F.fb
    F.reset(x0)
    fused = F.run(S, e=e)
    D = _loop(ctl, N, warm, H, plant=plant, n_slots=N, terminal_law=L, **kw)
    D.reset(x0)
    x_before = []
    logs = {k: [] for k in KEYS + ('u0', 'x', 'primal', 'x1')}
    for t in range(S):
        x_before.append(D.x.clone())
        out = D.step(e=e[t] if e is not None else None)
        for k in ('cost', 'n_solves', 'status', 'primal', 'hold'):
            logs[k].append(out[k].clone())
        logs['u0'].append(D.u0.clone()); logs['x'].append(D.x.clone())
        logs['x1'].append(D.fb['app_primal'][:, ctl.mld.nx:2 * ctl.mld.nx].clone())
    lock = {k: torch.stack(v) for k, v in logs.items()}
    torch.cuda.synchronize()
    _equal(fused, lock)
    assert torch.equal(F.x, D.x) and torch.equal(F.active, D.active)
    assert torch.equal(F.fb['law_n'], D.fb['law_n']) and torch.equal(F.fb['age'], D.fb['age'])
    hold = lock['hold'].cpu().numpy()
    assert np.array_equal(hold, replay_law(lock['status'].cpu().numpy(), lock['cost'].cpu().numpy(), H, L))
    law = _law_of(ctl, N, kw)
    n_law, n_clamped = _check_sat_law_steps(model, law, torch.stack(x_before).cpu().numpy(), hold, lock['u0'].cpu().numpy(),
                                            lock['x1'].cpu().numpy())
    print(case, H, L, 'law steps', n_law, 'with a clamped input', n_clamped)
    assert n_law == int((hold == LAW).sum()) and n_clamped > 0
    if plant is not None and HL == (3, 5):
        # step_with_plant with the device plant as its callback
        W = _loop(ctl, N, warm, H, n_slots=N, terminal_law=L, **kw)
        W.reset(x0)
        logs = {k: [] for k in KEYS + ('u0', 'x')}
        U = (ctl.T + 1) * ctl.mld.nx

        def callback(x, u):
            live = ((W.active != 0) & torch.isfinite(W.fb['app_cost'])).cpu().numpy()
            xm = plant.step(W.h, W.x, W.fb['app_primal'][:, U:U + ctl.mld.nu].contiguous()).cpu().numpy()
            assert np.array_equal(xm[live].shape, x.shape)
            return xm[live]
        for t in range(S):
            out, _, _ = W.step_with_plant(callback)
            for k in ('cost', 'n_solves', 'status', 'hold'):
                logs[k].append(out[k].clone())
            logs['u0'].append(W.u0.clone()); logs['x'].append(W.x.clone())
        torch.cuda.synchronize()
        _equal(fused, {k: torch.stack(v) for k, v in logs.items()})


@pytest.mark.parametrize('HL', [(0, 5), (3, 5), (19, 50)])
@pytest.mark.parametrize('case', ['linear_warm', 'linear_cold', 'plant_warm', 'plant_cold'])
def test_fused_equals_lock_step_two_lanes(cp20, HL, case):
    """more solver slots than SMs: the two-lane FB kernels against the one-lane ones and device lock step"""
    model, ctl = cp20
    H, L = HL
    N = 300
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert ctl.default_slots() > sms
    warm = case.endswith('warm')
    # a plan of H = 19 steps outlasts 8 linear steps: 30 reach the law
    S = (40 if H == 19 else 30) if case.startswith('plant') else (30 if H == 19 else 8)
    plant, x0, e = _batch(model, case, N, S, 9)
    kw = _sat_law(ctl, N, plant is not None)
    runs = []
    for slots in (sms, ctl.default_slots()):
        F = _loop(ctl, N, warm, H, plant=plant, n_slots=slots, terminal_law=L, **kw)
        F.reset(x0)
        logs = F.run(S, e=e)
        torch.cuda.synchronize()
        runs.append(({k: v.clone() for k, v in logs.items()}, F.x.clone()))
        del F
    D = _loop(ctl, N, warm, H, plant=plant, terminal_law=L, **kw)
    D.reset(x0)
    lock = _lock(D, S, e)
    torch.cuda.synchronize()
    _equal(runs[0][0], runs[1][0])
    _equal(runs[1][0], lock, KEYS + (('x',) if plant is not None else ()))
    assert torch.equal(runs[0][1], runs[1][1]) and torch.equal(runs[1][1], D.x)
    hold = lock['hold'].cpu().numpy()
    assert np.array_equal(hold, replay_law(lock['status'].cpu().numpy(), lock['cost'].cpu().numpy(), H, L))
    xs = np.concatenate((np.asarray(x0, dtype=float)[None], lock['x'][:-1].cpu().numpy()))     # the state of every step
    n_law, n_clamped = _check_sat_law_steps(model, _law_of(ctl, N, kw), xs, hold, lock['u0'].cpu().numpy())
    print(case, H, L, 'law steps', n_law, 'with a clamped input', n_clamped)
    assert n_law > 0 and n_clamped > 0


# ---- the policy kernel against the long-double reference -------------------------------------------------------------------
def test_fallback_step_matches_the_reference(cp20):
    model, ctl = cp20
    H, L = 3, 2
    h = ctl.handle(1)
    P, nx, nu = h.layout.primal, ctl.mld.nx, ctl.mld.nu
    grid = [(lv, hi, st, a, n) for lv in (0, 1) for hi in (0, 1) for st in (0, 1, 2, 3) for a in (-1, 0, 2, 3)
            for n in (0, 1, 2) if not (hi and st == 1)]
    N = len(grid)
    lv, hi, st, age, law_n = (np.array(c) for c in zip(*grid))
    rng = np.random.default_rng(0)
    dev = lambda a, dt=torch.float64: torch.as_tensor(a, dtype=dt, device='cuda').contiguous()
    x = rng.standard_normal((N, nx))
    plan = rng.standard_normal((N, P)); inc = rng.standard_normal((N, P))
    cost = np.where(hi == 1, rng.uniform(1., 2., N), np.inf)
    Ks = rng.standard_normal((N, nu, nx))
    k = .3 * rng.standard_normal((N, nu))
    lo, hi_b = np.full(nu, -.9), np.full(nu, .9)
    lo[1], hi_b[2], lo[3], hi_b[3] = -np.inf, np.inf, -np.inf, np.inf       # free components
    hi_b[4] = lo[4] = .25                                                     # a pinned one
    ref0 = fallback_reference_sat(model['A'], model['B'], Ks, ctl.T, H, L, lv, st, cost, age, law_n, x, plan, inc, k, lo, hi_b)
    law = np.nonzero(ref0['source'] == 2)[0]
    x[law[0], 1] = np.nan                                                     # NaN passes through the clamp
    ref = fallback_reference_sat(model['A'], model['B'], Ks, ctl.T, H, L, lv, st, cost, age, law_n, x, plan, inc, k, lo, hi_b)
    fb = h.new_fallback(N, H, L, Ks, k, lo, hi_b)
    assert fb['law_sets'] == N
    fb['plan'].copy_(dev(plan)); fb['age'].copy_(dev(age, torch.int32)); fb['law_n'].copy_(dev(law_n, torch.int32))
    fb['app_primal'].fill_(np.nan)
    out = dict(status=dev(st, torch.int32), cost=dev(cost), primal=dev(inc))
    h.fallback_step(fb, dev(x), dev(lv, torch.int32), out)
    torch.cuda.synchronize()
    for key, got in (('hold', fb['hold']), ('age', fb['age']), ('law_n', fb['law_n']), ('plan', fb['plan'])):
        assert np.array_equal(got.cpu().numpy(), ref[key]), key
    ac, ap = fb['app_cost'].cpu().numpy(), fb['app_primal'].cpu().numpy()
    assert np.array_equal(ac, ref['app_cost'])
    U = (ctl.T + 1) * nx
    u, x1 = ap[:, U:U + nu], ap[:, nx:2 * nx]
    assert ref['clamped'][law].any() and (~ref['clamped'][law]).any()
    n_exact = 0
    for i in np.nonzero(ref['source'] > 0)[0]:
        assert np.array_equal(ap[i, :nx], x[i], equal_nan=True)
        ru, rx = ref['u'][i].astype(float), ref['x1'][i].astype(float)
        assert np.array_equal(np.isnan(u[i]), np.isnan(ru)) and np.array_equal(np.isnan(x1[i]), np.isnan(rx)), i
        cl = ref['clamped'][i]
        assert np.array_equal(u[i][cl], ru[cl]), i
        n_exact += int(cl.sum())
        f = ~cl & ~np.isnan(ru)
        assert np.all(np.abs(u[i][f] - ru[f]) <= 1e-14 * ref['u_terms'][i][f]), i
        f = ~np.isnan(rx)
        assert np.all(np.abs(x1[i][f] - rx[f]) <= 1e-14 * ref['x1_terms'][i][f]), i
    assert n_exact > 0 and np.isnan(u[law[0]]).all() and np.isnan(x1[law[0]]).all()
    assert np.all(u[law[1:], 4] == .25)                                       # the pinned input


# ---- the warm start across a clamped law step -----------------------------------------------------------------------------
def test_shift_after_a_clamped_law_step_equals_construct_warm_start(cp20):
    model, ctl = cp20
    N, S = 64, 30
    plant, x0 = _heavy_plants(model, N)
    L = _loop(ctl, N, True, 0, plant=plant, n_slots=N, terminal_law=50, law_bounds='model')
    L.reset(x0)
    A, B = model['A'], model['B']
    K = ctl.terminal_law()
    lo, hi = ctl.input_box()
    nuc = ctl.mld.nu - ctl.mld.nub
    checked = 0
    for t in range(S):
        x = L.x.cpu().numpy().copy()
        out = L.step()
        hold = out['hold'].cpu().numpy()
        u_all = L.u0.cpu().numpy()
        clamped = [i for i in np.nonzero(hold == LAW)[0] if u_all[i, 0] in (lo[0], hi[0])]
        for i in clamped[:2]:
            old, new = L.trees[1 - L.cur], L.trees[L.cur]
            u = u_all[i]
            assert abs(K[0].dot(x[i])) > 1.                       # K x was clamped to the cart-force bound
            x_meas = L.x[i].cpu().numpy()
            e0 = x_meas - (A.dot(x[i]) + B.dot(u))
            leaves = ctl.tree_to_leaves(old, int(i))
            ctl.device_search = False
            try:
                ws_h, _, _ = ctl.construct_warm_start(leaves, x[i], u[:nuc], u[nuc:], e0)
            finally:
                ctl.device_search = True
            ws_d = ctl.tree_to_leaves(new, int(i))
            key = lambda ls: [sorted(l.identifier.items()) for l in ls]
            assert key(ws_d) == key(ws_h)
            a, b = np.array([l.lb for l in ws_d]), np.array([l.lb for l in ws_h])
            assert np.array_equal(np.isinf(a), np.isinf(b)) and np.all(np.abs(a[np.isfinite(a)] - b[np.isfinite(b)]) <= 1e-11)
            none = lambda ls: [l.extra is None or l.extra.dual is None for l in ls]
            assert none(ws_d) == none(ws_h)
            checked += 1
        if checked >= 6:
            break
    assert checked > 0


# ---- error paths -----------------------------------------------------------------------------------------------------------
def test_error_paths_of_the_new_fields(cp20):
    model, ctl = cp20
    from warm_start_hmpc_b200 import capi
    N = 4
    L = _loop(ctl, N, True, 3, n_slots=N, terminal_law=5, law_bounds='model', law_offset=np.zeros(ctl.mld.nu))
    L.reset(np.load(os.path.join(MODELS, 'cp20_instances.npy'))[:N])
    h = L.h
    err = lambda: capi.load_library().wshmpc_last_error().decode()
    call = lambda fb: h.closed_loop(1, True, True, L.cur, L.xbuf, None, L.active, L.trees, L.out, fallback=fb)
    call(L.fb)
    torch.cuda.synchronize()
    cases = [(dict(L.fb, law_sets=2), 'law_sets = 2'), (dict(L.fb, law_sets=-1), 'law_sets = -1'),
             (dict(L.fb, law_sets=N + 1), 'law_sets = 5'), (dict(L.fb, law_lo=None), 'both or neither'),
             (dict(L.fb, law_hi=None), 'both or neither')]
    bare = {kk: v for kk, v in L.fb.items() if kk not in ('law_K', 'law_n', 'law_k', 'law_lo', 'law_hi')}
    for key in ('law_k', 'law_lo', 'law_hi'):
        cases.append((dict(bare, max_law=0, **{key: L.fb[key]}), 'max_law = 0'))
    cases.append((dict(L.fb, max_law=0, law_K=None, law_n=None, law_k=None, law_lo=None, law_hi=None, law_sets=1), 'max_law = 0'))
    for fb, msg in cases:
        with pytest.raises(RuntimeError, match=msg):
            call(fb)
        with pytest.raises(RuntimeError, match=msg):
            h.fallback_step(fb, L.x, L.active, L.out)
    # one set (law_sets 1) and one per instance pass; without the law every new field zero passes
    call(dict(L.fb, law_sets=1))
    call(dict(L.fb, law_sets=N, law_K=L.fb['law_K'][None].expand(N, -1, -1).contiguous(),
              law_k=L.fb['law_k'][None].expand(N, -1).contiguous()))
    call(dict(L.fb, max_law=0, law_K=None, law_n=None, law_k=None, law_lo=None, law_hi=None))
    c = capi._fallback_struct(dict(L.fb, law_sets=7), L.fb['hold'])
    assert h.lib.wshmpc_fallback_step(h._h, N, C.byref(c), C.c_void_p(L.x.data_ptr()), None, C.c_void_p(L.out['status'].data_ptr()),
                                      C.c_void_p(L.out['cost'].data_ptr()), C.c_void_p(L.out['primal'].data_ptr())) != 0
    assert 'law_sets' in err()
    # the refusals of the fallback hold with the new law
    with pytest.raises(ValueError, match='fallback'):
        L.run_mailbox(1, lambda *a: None)
    with pytest.raises(ValueError, match='fallback plans'):
        L.rebalance()
    torch.cuda.synchronize()
