"""-m gpu: the terminal law as the last fallback through infeasible MIQPs (wshmpc_fallback.max_law,
ClosedLoop(..., fallback=H, terminal_law=L)).

* the fused loop equals lock step bit for bit (step(), and step_with_plant with the device plant as callback): linear and
  device plant, warm and cold, one and two lanes, (H, L) in {(0, 5), (3, 5), (19, 50)}; the pinned batches take law steps,
  run a law out and leave, and return to an incumbent after law steps; the hold sequence follows the numpy policy;
* a law step applies u0 = K x and x_1|t = A x + B u0;
* the tree of an infeasible step shifted with the law's input equals the host construct_warm_start;
* wshmpc_fallback_step on hand-built inputs follows the extended policy table, statuses 2 and 3 included;
* the error paths fail with a message.
"""
import ctypes as C
import os
import numpy as np
import pytest
import torch

from oracle.models import load_model, MODELS
from tests.util import make_controller
from tests.test_gpu_fallback import KEYS, _loop, _heavy_plants, _noise, _lock, _equal
from tests.test_terminal_law_cpu import LAW, policy_law, replay_law

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


def _counts(hold, L):
    """law steps, laws run out (the L-th law step since the last incumbent, then the instance leaves), returns to an
    incumbent right after a law step"""
    n = np.zeros(hold.shape[1], dtype=int)
    out = 0
    for t in range(hold.shape[0]):
        n = np.where(hold[t] == 0, 0, np.where(hold[t] == LAW, n + 1, n))
        if t + 1 < hold.shape[0]:
            out += int(((hold[t] == LAW) & (n == L) & (hold[t + 1] == -1)).sum())
    return int((hold == LAW).sum()), out, int(((hold[:-1] == LAW) & (hold[1:] == 0)).sum())


def _rel_close(a, b, terms, rtol=1e-14):
    """|a - b| <= rtol * (sum of the magnitudes of the terms b was summed from), elementwise"""
    return np.all(np.abs(a - b) <= rtol * terms)


def _check_law_steps(model, K, xs, hold, u0, x1=None):
    """every law step (hold == -2) applied u0 = K x (and x_1|t = A x + B u0 where x1 is given); returns the steps checked"""
    A, B = model['A'], model['B']
    t_i = np.argwhere(hold == LAW)
    for t, i in t_i:
        x = xs[t, i]
        assert _rel_close(u0[t, i], K.dot(x), np.abs(K).dot(np.abs(x))), (t, i)
        if x1 is not None:
            assert _rel_close(x1[t, i], A.dot(x) + B.dot(u0[t, i]), np.abs(A).dot(np.abs(x)) + np.abs(B).dot(np.abs(u0[t, i]))), (t, i)
    return len(t_i)


@pytest.mark.parametrize('HL', [(0, 5), (3, 5), (19, 50)])
@pytest.mark.parametrize('case', ['linear_warm', 'linear_cold', 'plant_warm', 'plant_cold'])
def test_fused_equals_lock_step_one_lane(cp20, HL, case):
    model, ctl = cp20
    H, L = HL
    N = 64
    # the heavy plants hold their plan for H = 19 steps first: 40 steps reach the law
    S = 40 if case.startswith('plant') and H == 19 else 30
    warm = case.endswith('warm')
    plant, x0, e = _batch(model, case, N, S, 7)
    F = _loop(ctl, N, warm, H, plant=plant, n_slots=N, terminal_law=L)
    F.reset(x0)
    fused = F.run(S, e=e)
    D = _loop(ctl, N, warm, H, plant=plant, n_slots=N, terminal_law=L)
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
    n_law, n_out, n_back = _counts(hold, L)
    print(case, H, L, 'law steps', n_law, 'laws run out', n_out, 'back to an incumbent', n_back,
          'plan steps', int((hold > 0).sum()), 'off', int((hold[-1] == -1).sum()))
    assert n_law > 0
    # the logs of a law step: cost +inf, status 1, the law's input
    law = hold == LAW
    assert np.all(np.isinf(lock['cost'].cpu().numpy()[law])) and np.all(lock['status'].cpu().numpy()[law] == 1)
    K = D.fb['law_K'].cpu().numpy()
    assert np.array_equal(K, ctl.terminal_law())
    assert _check_law_steps(model, K, torch.stack(x_before).cpu().numpy(), hold, lock['u0'].cpu().numpy(),
                            lock['x1'].cpu().numpy()) == n_law
    if plant is not None and HL == (3, 5):
        # step_with_plant with the device plant as its callback
        W = _loop(ctl, N, warm, H, n_slots=N, terminal_law=L)
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


def test_law_runs_end_in_an_incumbent_or_run_out(cp20):
    """law runs of the pinned batches both ways: an instance on the law finds a feasible MIQP again (law_n restarts at the
    next infeasible step), and an instance whose MIQP stays infeasible runs its L law steps out and leaves"""
    model, ctl = cp20
    N, S = 64, 30
    for case, L, back, out in (('linear_warm', 50, True, False), ('plant_warm', 5, False, True)):
        plant, x0, e = _batch(model, case, N, S, 7)
        F = _loop(ctl, N, True, 0, plant=plant, n_slots=N, terminal_law=L)
        F.reset(x0)
        hold = F.run(S, e=e)['hold'].cpu().numpy()
        n_law, n_out, n_back = _counts(hold, L)
        print(case, L, 'law steps', n_law, 'laws run out', n_out, 'back to an incumbent', n_back)
        if back:
            assert n_back > 0
        if out:
            assert n_out > 0 and (hold == LAW).sum(axis=0).max() >= L
        del F


@pytest.mark.parametrize('HL', [(0, 5), (3, 5)])
@pytest.mark.parametrize('case', ['linear_warm', 'linear_cold', 'plant_warm', 'plant_cold'])
def test_fused_equals_lock_step_two_lanes(cp20, HL, case):
    """more solver slots than SMs: the two-lane FB kernels against the one-lane ones and device lock step"""
    model, ctl = cp20
    H, L = HL
    N = 300
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert ctl.default_slots() > sms
    warm = case.endswith('warm')
    S = 30 if case.startswith('plant') else 8
    plant, x0, e = _batch(model, case, N, S, 9)
    runs = []
    for slots in (sms, ctl.default_slots()):
        F = _loop(ctl, N, warm, H, plant=plant, n_slots=slots, terminal_law=L)
        F.reset(x0)
        logs = F.run(S, e=e)
        torch.cuda.synchronize()
        runs.append(({k: v.clone() for k, v in logs.items()}, F.x.clone()))
        del F
    D = _loop(ctl, N, warm, H, plant=plant, terminal_law=L)
    D.reset(x0)
    lock = _lock(D, S, e)
    torch.cuda.synchronize()
    _equal(runs[0][0], runs[1][0])
    _equal(runs[1][0], lock, KEYS + (('x',) if plant is not None else ()))
    assert torch.equal(runs[0][1], runs[1][1]) and torch.equal(runs[1][1], D.x)
    hold = lock['hold'].cpu().numpy()
    assert np.array_equal(hold, replay_law(lock['status'].cpu().numpy(), lock['cost'].cpu().numpy(), H, L))
    assert (hold == LAW).any()


def test_shift_after_a_law_step_equals_construct_warm_start(cp20):
    model, ctl = cp20
    N, S = 64, 30
    plant, x0 = _heavy_plants(model, N)
    L = _loop(ctl, N, True, 0, plant=plant, n_slots=N, terminal_law=50)
    L.reset(x0)
    A, B = model['A'], model['B']
    K = ctl.terminal_law()
    nuc = ctl.mld.nu - ctl.mld.nub
    checked = 0
    for t in range(S):
        x = L.x.cpu().numpy().copy()
        out = L.step()
        hold = out['hold'].cpu().numpy()
        for i in np.nonzero(hold == LAW)[0][:2]:
            old, new = L.trees[1 - L.cur], L.trees[L.cur]
            u = L.u0[i].cpu().numpy()
            assert _rel_close(u, K.dot(x[i]), np.abs(K).dot(np.abs(x[i])))
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


def test_fallback_step_policy_table(cp20):
    model, ctl = cp20
    H, L = 3, 2
    h = ctl.handle(1)
    P, T, nx, nu = h.layout.primal, ctl.T, ctl.mld.nx, ctl.mld.nu
    grid = [(lv, hi, st, a, n) for lv in (0, 1) for hi in (0, 1) for st in (0, 1, 2, 3) for a in (-1, 0, 2, 3)
            for n in (0, 1, 2) if not (hi and st == 1)]
    N = len(grid)
    lv, hi, st, age, law_n = (np.array(c) for c in zip(*grid))
    rng = np.random.default_rng(0)
    dev = lambda a, dt=torch.float64: torch.as_tensor(a, dtype=dt, device='cuda').contiguous()
    x = rng.standard_normal((N, nx))
    plan = rng.standard_normal((N, P)); inc = rng.standard_normal((N, P))
    cost = np.where(hi == 1, rng.uniform(1., 2., N), np.inf)
    K = rng.standard_normal((nu, nx))
    fb = h.new_fallback(N, H, L, K)
    fb['plan'].copy_(dev(plan)); fb['age'].copy_(dev(age, torch.int32)); fb['law_n'].copy_(dev(law_n, torch.int32))
    fb['app_primal'].fill_(np.nan)
    out = dict(status=dev(st, torch.int32), cost=dev(cost), primal=dev(inc))
    h.fallback_step(fb, dev(x), dev(lv, torch.int32), out)
    torch.cuda.synchronize()
    src, hold, act, new_age, new_n = policy_law(lv, hi, st, age, law_n, H, L)
    assert {0, 1, 2, -1} <= set(src.tolist())
    assert np.array_equal(fb['hold'].cpu().numpy(), hold)
    assert np.array_equal(fb['age'].cpu().numpy(), new_age)
    assert np.array_equal(fb['law_n'].cpu().numpy(), new_n)
    ac, ap, pl = fb['app_cost'].cpu().numpy(), fb['app_primal'].cpu().numpy(), fb['plan'].cpu().numpy()
    assert np.array_equal(np.isfinite(ac), act == 1)
    U = (T + 1) * nx
    A, B = model['A'], model['B']
    for i in range(N):
        if src[i] == 0:
            assert ac[i] == cost[i] and np.array_equal(ap[i], inc[i]) and np.array_equal(pl[i], inc[i])
        else:
            assert np.array_equal(pl[i], plan[i])
        if src[i] == 1:
            u = plan[i, U + hold[i] * nu:U + (hold[i] + 1) * nu]
            assert np.array_equal(ap[i, U:U + nu], u)
        if src[i] == 2:
            assert ac[i] == 0.
            u = ap[i, U:U + nu]
            assert _rel_close(u, K.dot(x[i]), np.abs(K).dot(np.abs(x[i])))
        if src[i] in (1, 2):
            assert np.array_equal(ap[i, :nx], x[i])
            assert _rel_close(ap[i, nx:2 * nx], A.dot(x[i]) + B.dot(u), np.abs(A).dot(np.abs(x[i])) + np.abs(B).dot(np.abs(u)))


def test_statuses_2_and_3_leave_the_loop_with_a_law(cp20):
    model, ctl = cp20
    N = 8
    x0 = np.load(os.path.join(MODELS, 'cp20_instances.npy'))[:N]
    for fused in (False, True):
        L = _loop(ctl, N, False, 0, n_slots=N, terminal_law=50)
        L.reset(x0)
        L.run(2)
        L.max_solves = 1                       # a cold search that may solve the root only: status 2 without an incumbent
        if fused:
            lg = L.run(1)
            st, hold = lg['status'][0], lg['hold'][0]
        else:
            out = L.step()
            st, hold = out['status'], out['hold']
        torch.cuda.synchronize()
        assert torch.all(st == 2) and torch.all(hold == -1) and torch.all(L.active == 0)
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    c3 = make_controller(model, qp_options=dict(max_iter=2))
    L = ClosedLoop(c3, N, warm=True, max_solves=64, n_slots=N, terminal_law=50)
    L.reset(x0)
    lg = L.run(2)
    torch.cuda.synchronize()
    assert torch.all(lg['status'][0] == 3) and torch.all(lg['hold'] == -1) and torch.all(L.active == 0)


def test_law_error_paths(cp20):
    model, ctl = cp20
    from warm_start_hmpc_b200 import capi
    N = 4
    L = _loop(ctl, N, True, 3, n_slots=N, terminal_law=5)
    L.reset(np.load(os.path.join(MODELS, 'cp20_instances.npy'))[:N])
    h = L.h
    err = lambda: capi.load_library().wshmpc_last_error().decode()
    call = lambda fb: h.closed_loop(1, True, True, L.cur, L.xbuf, None, L.active, L.trees, L.out, fallback=fb)
    call(L.fb)
    torch.cuda.synchronize()
    for fb, msg in ((dict(L.fb, max_law=-1), 'max_law = -1'), (dict(L.fb, law_K=None), 'null d_law_K or d_law_n'),
                    (dict(L.fb, law_n=None), 'null d_law_K or d_law_n')):
        with pytest.raises(RuntimeError, match=msg):
            call(fb)
        with pytest.raises(RuntimeError, match=msg):
            h.fallback_step(fb, L.x, L.active, L.out)
    # without the law, null law buffers are fine
    call(dict(L.fb, max_law=0, law_K=None, law_n=None))
    c = capi._fallback_struct(dict(L.fb, max_law=-3), L.fb['hold'])
    assert h.lib.wshmpc_fallback_step(h._h, N, C.byref(c), C.c_void_p(L.x.data_ptr()), None, C.c_void_p(L.out['status'].data_ptr()),
                                      C.c_void_p(L.out['cost'].data_ptr()), C.c_void_p(L.out['primal'].data_ptr())) != 0
    assert 'max_law' in err()
    with pytest.raises(ValueError, match='terminal law gain'):
        h.new_fallback(N, 0, 5, np.zeros((ctl.mld.nx, ctl.mld.nu)))
    # the refusals of the fallback hold with the law
    with pytest.raises(ValueError, match='fallback'):
        L.run_mailbox(1, lambda *a: None)
    with pytest.raises(ValueError, match='fallback plans'):
        L.rebalance()
    torch.cuda.synchronize()
