"""-m gpu: the fallback policy through infeasible MIQPs (wshmpc_fallback, ClosedLoop(..., fallback=H)).

* H = 0 through wshmpc_closed_loop_fallback is the loop without a fallback, bit for bit (linear plant warm, cold and with
  errors, device plant; one- and two-lane kernels);
* the fused loop equals lock step bit for bit for H in {1, 3, T - 1}, also step_with_plant with the device plant as callback;
  the pinned batches do fall back, hold plans for H steps in a row and lose instances whose plan ran out;
* a fallback step applies u_a of the last solved step's incumbent and the hold sequence follows the numpy policy;
* the tree of an infeasible step shifted with the plan's input equals the host construct_warm_start;
* wshmpc_fallback_step on hand-built inputs follows the policy table, statuses 2 and 3 included;
* the error paths fail with a message.
"""
import ctypes as C
import os
import numpy as np
import pytest
import torch

from oracle.models import load_model, MODELS
from tests.util import make_controller
from tests.test_fallback_cpu import policy, replay

pytestmark = pytest.mark.gpu

DT = 0.05
KEYS = ('cost', 'n_solves', 'status', 'hold')


@pytest.fixture(scope='module')
def cp20():
    model = load_model('cp20')
    return model, make_controller(model)


def _loop(ctl, N, warm, H, plant=None, n_slots=None, **kw):
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    return ClosedLoop(ctl, N, warm=warm, max_solves=2048, max_roots=1024, n_slots=n_slots, plant=plant, fallback=H, **kw)


def _heavy_plants(model, N):
    """plants heavier than the model (mp 1.15 .. 1.3 x nominal) from x0_nominal: their MIQPs turn infeasible on the way"""
    from warm_start_hmpc_b200.plants import CartPoleWithWalls, DevicePlant
    mp = np.linspace(1.15, 1.3, N)
    return DevicePlant([CartPoleWithWalls(mp=m) for m in mp], DT), np.repeat(model['x0_nominal'][None], N, 0)


def _noise(model, S, N, sigma, seed):
    return torch.as_tensor(sigma * np.random.default_rng(seed).standard_normal((S, N, 4)) * model['x_max'], device='cuda')


def _lock(L, S, e=None):
    """step() S times: the logs of run(), with the state after every step"""
    logs = {k: [] for k in KEYS + ('u0', 'x', 'primal')}
    for t in range(S):
        out = L.step(e=e[t] if e is not None else None)
        for k in ('cost', 'n_solves', 'status', 'primal'):
            logs[k].append(out[k].clone())
        logs['hold'].append(out['hold'].clone()); logs['u0'].append(L.u0.clone()); logs['x'].append(L.x.clone())
    return {k: torch.stack(v) for k, v in logs.items()}


def _equal(a, b, keys=KEYS + ('x',)):
    for k in keys:
        if k in a and k in b:
            assert torch.equal(a[k], b[k]), k
    assert torch.equal(torch.nan_to_num(a['u0'], nan=-7.), torch.nan_to_num(b['u0'], nan=-7.))


# ---- H = 0 is the loop without a fallback -----------------------------------------------------------------------------------
@pytest.mark.parametrize('case', ['warm', 'cold', 'warm_errors', 'plant_warm', 'plant_cold'])
@pytest.mark.parametrize('lanes', [1, 2])
def test_h0_equals_the_loop_without_fallback(cp20, case, lanes):
    model, ctl = cp20
    if lanes == 1:
        N, S, slots = 24, 12, 24
    else:
        N, S, slots = 300, 4, None
        assert ctl.default_slots() > torch.cuda.get_device_properties(0).multi_processor_count
    warm = 'cold' not in case
    plant, x0 = (None, np.load(os.path.join(MODELS, 'cp20_instances.npy'))[:N])
    if 'plant' in case:
        plant, x0 = _heavy_plants(model, N)
    e = _noise(model, S, N, .02, 3) if case in ('warm_errors', 'cold') else None
    runs = []
    for fb in (False, True):
        L = _loop(ctl, N, warm, 0, plant=plant, n_slots=slots)
        if fb:                                   # the FB kernels at H = 0 (ClosedLoop uses them only for H > 0)
            L.fb = L.h.new_fallback(N, 0)
        L.reset(x0)
        logs = L.run(S, e=e)
        torch.cuda.synchronize()
        runs.append(({k: v.clone() for k, v in logs.items()}, L.x.clone(), L.active.clone()))
        del L
    (a, xa, aa), (b, xb, ab) = runs
    _equal(a, b, ('cost', 'n_solves', 'status', 'x'))
    assert torch.equal(xa, xb) and torch.equal(aa, ab)
    hold = b['hold'].cpu().numpy()
    assert set(np.unique(hold)) <= {0, -1}
    assert np.array_equal(hold, replay(b['status'].cpu().numpy(), b['cost'].cpu().numpy(), 0))


# ---- fused equals lock step, and the batches exercise the feature -----------------------------------------------------------
@pytest.mark.parametrize('H', [1, 3, 19])
@pytest.mark.parametrize('case', ['linear_warm', 'linear_cold', 'plant_warm', 'plant_cold'])
def test_fused_equals_lock_step_one_lane(cp20, H, case):
    model, ctl = cp20
    N, S = 64, 30
    warm = case.endswith('warm')
    if case.startswith('plant'):
        plant, x0 = _heavy_plants(model, N)
        e = None
    else:
        plant, x0 = None, np.load(os.path.join(MODELS, 'cp20_instances.npy'))[:N]
        e = _noise(model, S, N, .02, 7)
    F = _loop(ctl, N, warm, H, plant=plant, n_slots=N)
    F.reset(x0)
    fused = F.run(S, e=e)
    D = _loop(ctl, N, warm, H, plant=plant, n_slots=N)
    D.reset(x0)
    lock = _lock(D, S, e)
    torch.cuda.synchronize()
    _equal(fused, lock)
    assert torch.equal(F.x, D.x) and torch.equal(F.active, D.active)
    hold = lock['hold'].cpu().numpy()
    assert np.array_equal(hold, replay(lock['status'].cpu().numpy(), lock['cost'].cpu().numpy(), H))
    print(case, H, 'fallback steps', int((hold > 0).sum()), 'longest hold', int(hold.max()), 'off', int((hold[-1] == -1).sum()))
    assert (hold > 0).any()
    if H < 19 and warm:
        # a run of H fallback steps in a row, and an instance switched off when its plan ran out
        assert (hold == H).any() and ((hold[:-1] == H) & (hold[1:] == -1)).any()
    # the logs of a fallback step: cost +inf, status 1, a finite applied input
    fbk = hold > 0
    assert np.all(np.isinf(lock['cost'].cpu().numpy()[fbk])) and np.all(lock['status'].cpu().numpy()[fbk] == 1)
    assert np.all(np.isfinite(lock['u0'].cpu().numpy()[fbk]))
    # applied input: u_a of the incumbent of the last solved step
    T, nx, nu = ctl.T, ctl.mld.nx, ctl.mld.nu
    prim, u0 = lock['primal'].cpu().numpy(), lock['u0'].cpu().numpy()
    for i in range(N):
        last = None
        for t in range(S):
            if hold[t, i] == 0:
                last = prim[t, i]
                assert np.array_equal(u0[t, i], last[(T + 1) * nx:(T + 1) * nx + nu])
            elif hold[t, i] > 0:
                a = hold[t, i]
                assert hold[t - 1, i] == a - 1
                assert np.array_equal(u0[t, i], last[(T + 1) * nx + a * nu:(T + 1) * nx + (a + 1) * nu]), (i, t, a)
    if plant is not None and H == 3:
        # step_with_plant with the device plant as its callback
        W = _loop(ctl, N, warm, H, n_slots=N)
        W.reset(x0)
        logs = {k: [] for k in KEYS + ('u0', 'x')}

        def callback(x, u):
            # the live rows of a batch with one parameter set per instance: the plant of every instance, then those rows
            live = ((W.active != 0) & torch.isfinite(W.fb['app_cost'])).cpu().numpy()
            U = (ctl.T + 1) * ctl.mld.nx
            xm = plant.step(W.h, W.x, W.fb['app_primal'][:, U:U + ctl.mld.nu].contiguous()).cpu().numpy()
            assert np.array_equal(xm[live].shape, x.shape)
            return xm[live]
        for t in range(S):
            out, _, _ = W.step_with_plant(callback)
            for k in ('cost', 'n_solves', 'status'):
                logs[k].append(out[k].clone())
            logs['hold'].append(out['hold'].clone()); logs['u0'].append(W.u0.clone()); logs['x'].append(W.x.clone())
        torch.cuda.synchronize()
        _equal(fused, {k: torch.stack(v) for k, v in logs.items()})


@pytest.mark.parametrize('case', ['linear_warm', 'plant_warm', 'plant_cold'])
def test_fused_equals_lock_step_two_lanes(cp20, case):
    """more solver slots than SMs: the two-lane FB kernels against the one-lane ones and device lock step"""
    model, ctl = cp20
    N, H = 300, 3
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert ctl.default_slots() > sms
    warm = case.endswith('warm')
    if case.startswith('plant'):
        S = 30
        plant, x0 = _heavy_plants(model, N)
        e = None
    else:
        S = 8
        plant, x0 = None, np.load(os.path.join(MODELS, 'cp20_instances.npy'))[:N]
        e = _noise(model, S, N, .02, 9)
    runs = []
    for slots in (sms, ctl.default_slots()):
        L = _loop(ctl, N, warm, H, plant=plant, n_slots=slots)
        L.reset(x0)
        logs = L.run(S, e=e)
        torch.cuda.synchronize()
        runs.append(({k: v.clone() for k, v in logs.items()}, L.x.clone()))
        del L
    D = _loop(ctl, N, warm, H, plant=plant)
    D.reset(x0)
    lock = _lock(D, S, e)
    torch.cuda.synchronize()
    _equal(runs[0][0], runs[1][0])
    _equal(runs[1][0], lock, KEYS + (('x',) if plant is not None else ()))
    assert torch.equal(runs[0][1], runs[1][1]) and torch.equal(runs[1][1], D.x)
    assert (lock['hold'].cpu().numpy() > 0).any()


# ---- the warm start across the gap ----------------------------------------------------------------------------------------
def test_shift_after_an_infeasible_step_equals_construct_warm_start(cp20):
    model, ctl = cp20
    N, S, H = 64, 30, 19
    plant, x0 = _heavy_plants(model, N)
    L = _loop(ctl, N, True, H, plant=plant, n_slots=N)
    L.reset(x0)
    A, B = model['A'], model['B']
    nuc = ctl.mld.nu - ctl.mld.nub
    checked = 0
    for t in range(S):
        x = L.x.cpu().numpy().copy()
        out = L.step()
        hold = out['hold'].cpu().numpy()
        for i in np.nonzero(hold > 0)[0][:2]:
            old, new = L.trees[1 - L.cur], L.trees[L.cur]
            u = L.u0[i].cpu().numpy()
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


# ---- the policy kernel on hand-built inputs (statuses 2 and 3 included) ----------------------------------------------------
def test_fallback_step_policy_table(cp20):
    model, ctl = cp20
    H = 3
    h = ctl.handle(1)
    P, T, nx, nu = h.layout.primal, ctl.T, ctl.mld.nx, ctl.mld.nu
    grid = [(lv, hi, st, a) for lv in (0, 1) for hi in (0, 1) for st in (0, 1, 2, 3) for a in (-1, 0, 1, 2, 3)
            if not (hi and st == 1)]
    N = len(grid)
    lv, hi, st, age = (np.array(c) for c in zip(*grid))
    rng = np.random.default_rng(0)
    dev = lambda a, dt=torch.float64: torch.as_tensor(a, dtype=dt, device='cuda').contiguous()
    x = rng.standard_normal((N, nx))
    plan = rng.standard_normal((N, P)); inc = rng.standard_normal((N, P))
    cost = np.where(hi == 1, rng.uniform(1., 2., N), np.inf)
    fb = h.new_fallback(N, H)
    fb['plan'].copy_(dev(plan)); fb['age'].copy_(dev(age, torch.int32)); fb['app_primal'].fill_(np.nan)
    out = dict(status=dev(st, torch.int32), cost=dev(cost), primal=dev(inc))
    h.fallback_step(fb, dev(x), dev(lv, torch.int32), out)
    torch.cuda.synchronize()
    src, hold, act, new_age = policy(lv, hi, st, age, H)
    assert np.array_equal(fb['hold'].cpu().numpy(), hold)
    assert np.array_equal(fb['age'].cpu().numpy(), new_age)
    ac, ap, pl = fb['app_cost'].cpu().numpy(), fb['app_primal'].cpu().numpy(), fb['plan'].cpu().numpy()
    assert np.array_equal(np.isfinite(ac), act == 1)
    U = (T + 1) * nx
    for i in range(N):
        if src[i] == 0:
            assert ac[i] == cost[i] and np.array_equal(ap[i], inc[i]) and np.array_equal(pl[i], inc[i])
        else:
            assert np.array_equal(pl[i], plan[i])
        if src[i] == 1:
            a = hold[i]
            u = plan[i, U + a * nu:U + (a + 1) * nu]
            assert np.array_equal(ap[i, :nx], x[i]) and np.array_equal(ap[i, U:U + nu], u)
            x1 = model['A'].dot(x[i]) + model['B'].dot(u)
            assert np.allclose(ap[i, nx:2 * nx], x1, rtol=1e-13, atol=1e-14)


def test_statuses_2_and_3_leave_the_loop(cp20):
    model, ctl = cp20
    N = 8
    x0 = np.load(os.path.join(MODELS, 'cp20_instances.npy'))[:N]
    # capacity: plans exist (two solved steps), then a cold search that may solve one QP only (the root: no incumbent)
    for fused in (False, True):
        L = _loop(ctl, N, False, 19, n_slots=N)
        L.reset(x0)
        L.run(2)
        assert torch.all(L.fb['age'] == 0)
        L.max_solves = 1
        if fused:
            lg = L.run(1)
            st, hold = lg['status'][0], lg['hold'][0]
        else:
            out = L.step()
            st, hold = out['status'], out['hold']
        torch.cuda.synchronize()
        assert torch.all(st == 2) and torch.all(hold == -1) and torch.all(L.active == 0)
    # QP iteration limit: every node QP stops after two iterations
    c3 = make_controller(model, qp_options=dict(max_iter=2))
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    L = ClosedLoop(c3, N, warm=True, max_solves=64, n_slots=N, fallback=19)
    L.reset(x0)
    lg = L.run(2)
    torch.cuda.synchronize()
    assert torch.all(lg['status'][0] == 3) and torch.all(lg['hold'] == -1) and torch.all(L.active == 0)


# ---- error paths ----------------------------------------------------------------------------------------------------------
def test_fallback_error_paths(cp20):
    model, ctl = cp20
    from warm_start_hmpc_b200 import capi
    N = 4
    L = _loop(ctl, N, True, 3, n_slots=N)
    L.reset(np.load(os.path.join(MODELS, 'cp20_instances.npy'))[:N])
    h = L.h
    err = lambda: capi.load_library().wshmpc_last_error().decode()
    call = lambda fb, **kw: h.closed_loop(1, kw.get('warm', True), True, L.cur, L.xbuf, None, L.active, L.trees, L.out,
                                          fallback=fb, mailbox=kw.get('mailbox'))
    call(L.fb)
    torch.cuda.synchronize()
    for fb, msg in ((dict(L.fb, max_hold=-1), 'max_hold'), (dict(L.fb, max_hold=ctl.T), 'max_hold'),
                    (dict(L.fb, plan=None), 'null fallback buffer'), (dict(L.fb, age=None), 'null fallback buffer'),
                    (dict(L.fb, app_cost=None), 'null fallback buffer'), (dict(L.fb, app_primal=L.fb['plan']), 'overlap'),
                    (dict(L.fb, app_primal=L.fb['plan'][1:]), 'overlap')):
        with pytest.raises(RuntimeError, match=msg):
            call(fb)
        with pytest.raises(RuntimeError, match=msg):
            h.fallback_step(fb, L.x, L.active, L.out)
    c = capi._fallback_struct(L.fb, None)           # null hold log
    assert h.lib.wshmpc_fallback_step(h._h, N, C.byref(c), C.c_void_p(L.x.data_ptr()), None, C.c_void_p(L.out['status'].data_ptr()),
                                      C.c_void_p(L.out['cost'].data_ptr()), C.c_void_p(L.out['primal'].data_ptr())) != 0
    assert 'null fallback buffer' in err()
    assert h.lib.wshmpc_fallback_step(h._h, N, None, C.c_void_p(L.x.data_ptr()), None, C.c_void_p(L.out['status'].data_ptr()),
                                      C.c_void_p(L.out['cost'].data_ptr()), C.c_void_p(L.out['primal'].data_ptr())) != 0
    assert 'null fallback' in err()
    # the comparator's node rules (cold trees)
    for rule in (1, 2):
        h.set_node_rule(rule)
        try:
            with pytest.raises(RuntimeError, match='node rule'):
                call(L.fb, warm=False)
            with pytest.raises(RuntimeError, match='node rule'):
                h.fallback_step(L.fb, L.x, L.active, L.out)
        finally:
            h.set_node_rule(0)
    # a mailbox
    mb = capi.Mailbox(h, N)
    try:
        mb.clear()
        with pytest.raises(RuntimeError, match='mailbox'):
            call(L.fb, mailbox=mb)
    finally:
        mb.close()
    with pytest.raises(ValueError, match='fallback'):
        L.run_mailbox(1, lambda *a: None)
    with pytest.raises(ValueError, match='fallback plans'):
        L.rebalance()
    torch.cuda.synchronize()
