"""-m gpu: the nonlinear cart-pole plant on the device (plants.DevicePlant, wshmpc_plant_step, wshmpc_closed_loop_plant).

* the standalone plant kernel matches CartPoleWithWalls.simulate to 1e-12 (only fp64 sin / cos differ);
* the fused loop with the device plant equals lock step (step_with_plant with the device plant as its callback, and
  ClosedLoop(plant=...).step()) bit for bit: warm, cold and the comparator, one- and two-lane builds, with and without a
  disturbance;
* against the numpy plant the modes of every step are the same and the costs agree to 1e-8;
* per-instance parameter sets are independent of each other;
* the error paths fail with a message.
"""
import ctypes as C
import os
import numpy as np
import pytest
import torch

from oracle.models import load_model, MODELS
from tests.util import make_controller

pytestmark = pytest.mark.gpu

DT = 0.05          # sample time of the cart-pole models


@pytest.fixture(scope='module')
def cp20():
    model = load_model('cp20')
    return model, make_controller(model)


def _modes(ctl, primal):
    T, nx, nu, nub = ctl.T, ctl.mld.nx, ctl.mld.nu, ctl.mld.nub
    p = primal.cpu().numpy() if torch.is_tensor(primal) else primal
    return np.round(p[:, (T + 1) * nx:].reshape(-1, T, nu)[:, :, nu - nub:])


def _loop(ctl, N, mode, plant=None, n_slots=None):
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    if mode == 'comparator':
        return ClosedLoop(ctl, N, warm=False, comparator=True, mip_start=True, max_solves=4096, n_slots=n_slots, plant=plant)
    return ClosedLoop(ctl, N, warm=mode == 'warm', max_solves=2048, max_roots=1024, n_slots=n_slots, plant=plant)


def _live(L):
    return ((L.active != 0) & torch.isfinite(L.out['cost'])).cpu().numpy()


def _assert_logs_equal(a, b):
    for k in ('cost', 'n_solves', 'status', 'x'):
        assert torch.equal(a[k], b[k]), k
    assert torch.equal(torch.nan_to_num(a['u0'], nan=-7.), torch.nan_to_num(b['u0'], nan=-7.))


def _states(model, N):
    return np.repeat(model['x0_nominal'][None], N, 0) * np.linspace(1., 0.8, N)[:, None]


def test_plant_step_matches_numpy(cp20):
    """Free flight, deep penetration of either wall, one parameter set per state; states away from the contact switches."""
    model, ctl = cp20
    from warm_start_hmpc_b200.plants import CartPoleWithWalls, DevicePlant
    rng = np.random.default_rng(5)
    n = 300
    plants = [CartPoleWithWalls(mc=rng.uniform(.7, 1.3), mp=rng.uniform(.7, 1.3), l=rng.uniform(.8, 1.2), d=rng.uniform(.4, .6),
                                stiffness=rng.uniform(70., 130.), damping=rng.uniform(7., 13.), g=rng.uniform(9.5, 10.5))
              for _ in range(n)]
    x = np.zeros((n, 4))
    x[:, 1] = rng.uniform(-.15, .15, n); x[:, 2:] = rng.uniform(-1., 1., (n, 2))
    third = n // 3
    for i in range(n):
        p = plants[i]
        # free flight (tip between the walls), deep in the left wall, deep in the right wall
        tip = rng.uniform(-.6, .6) * p.d if i < third else (-p.d - rng.uniform(.05, .15)) if i < 2 * third else p.d + rng.uniform(.05, .15)
        x[i, 0] = tip + p.l * np.sin(x[i, 1])
    u = np.zeros((n, ctl.mld.nu)); u[:, 0] = rng.uniform(-1., 1., n)
    ref = np.stack([plants[i].simulate(x[i], DT, u[i, 0]) for i in range(n)])
    # away from the switching surfaces along the way: every sub-step's gaps and one-sided forces keep their sign
    keep = np.ones(n, dtype=bool)
    for i in range(n):
        p, xi = plants[i], x[i].copy()
        for _ in range(50):
            gl, gr = p.gaps(xi)
            vtip = xi[2] - p.l * np.cos(xi[1]) * xi[3]
            fl, fr = -p.k * gl - p.c * vtip, -p.k * gr + p.c * vtip
            if min(abs(gl), abs(gr)) < 1e-6 or (gl <= 0 and abs(fl) < 1e-6) or (gr <= 0 and abs(fr) < 1e-6):
                keep[i] = False
            xi = xi + DT / 50 * p.x_dot(xi, u[i, 0])
    assert keep.sum() > 250
    dp = DevicePlant([plants[i] for i in np.nonzero(keep)[0]], DT)
    assert dp.n_sub == 50 and dp.n_sets == keep.sum()
    h = ctl.handle(1)
    out = dp.step(h, torch.as_tensor(x[keep], device='cuda'), torch.as_tensor(u[keep], device='cuda')).cpu().numpy()
    r = ref[keep]
    err = np.abs(out - r).max(axis=1) / np.abs(r).max(axis=1)
    assert err.max() <= 1e-12, err.max()
    # the walls acted: the deep states were pushed back
    assert np.all(np.abs(r[third:] - x[third:]).max(axis=1)[keep[third:]] > 1e-3)
    # one parameter set for every state
    one = DevicePlant(plants[0], DT).step(h, torch.as_tensor(x, device='cuda'), torch.as_tensor(u, device='cuda')).cpu().numpy()
    r0 = plants[0].simulate(x, DT, u[:, 0])
    assert np.all(np.abs(one - r0).max(axis=1) <= 1e-12 * np.abs(r0).max(axis=1))


def _lock_step_with_device_callback(L, dp, S, d):
    """step_with_plant with the device plant as its host callback (+ the disturbance of the live instances)"""
    logs = {k: [] for k in ('cost', 'u0', 'n_solves', 'status', 'x')}
    for t in range(S):
        def plant(x, u):
            xm = dp.step(L.h, torch.as_tensor(x, device='cuda'), torch.as_tensor(u, device='cuda')).cpu().numpy()
            return xm + d[t][_live(L)] if d is not None else xm
        out, _, _ = L.step_with_plant(plant)
        for k in ('cost', 'n_solves', 'status'):
            logs[k].append(out[k].clone())
        logs['u0'].append(L.u0.clone()); logs['x'].append(L.x.clone())
    return {k: torch.stack(v) for k, v in logs.items()}


@pytest.mark.parametrize('mode', ['warm', 'cold', 'comparator'])
@pytest.mark.parametrize('dist', [False, True])
def test_fused_plant_loop_equals_lock_step(cp20, mode, dist):
    model, ctl = cp20
    from warm_start_hmpc_b200.plants import CartPoleWithWalls, DevicePlant
    N, S = 6, 12
    x0 = _states(model, N)
    dp = DevicePlant(CartPoleWithWalls(), DT)
    d = torch.as_tensor(1e-3 * np.random.default_rng(11).standard_normal((S, N, 4)) * model['x_max'], device='cuda') if dist else None
    lock = _loop(ctl, N, mode, n_slots=N)
    lock.reset(x0)
    ref = _lock_step_with_device_callback(lock, dp, S, d.cpu().numpy() if dist else None)
    fused = _loop(ctl, N, mode, plant=dp, n_slots=N)
    fused.reset(x0)
    logs = fused.run(S, e=d)
    dev = _loop(ctl, N, mode, plant=dp, n_slots=N)            # lock step on the device: K3, plant, K2 + K4 per step
    dev.reset(x0)
    dl = {k: [] for k in ('cost', 'u0', 'n_solves', 'status', 'x')}
    for t in range(S):
        out = dev.step(e=d[t] if dist else None)
        for k in ('cost', 'n_solves', 'status'):
            dl[k].append(out[k].clone())
        dl['u0'].append(dev.u0.clone()); dl['x'].append(dev.x.clone())
    torch.cuda.synchronize()
    assert np.isfinite(ref['cost'].cpu().numpy()).mean() > .5
    _assert_logs_equal(ref, logs)
    _assert_logs_equal(ref, {k: torch.stack(v) for k, v in dl.items()})
    assert torch.equal(fused.x, lock.x) and torch.equal(dev.x, lock.x) and torch.equal(fused.active, lock.active)


@pytest.mark.parametrize('mode', ['warm', 'comparator'])
def test_two_lane_plant_loop_equals_one_lane_and_lock_step(cp20, mode):
    """More solver slots than SMs: the two-lane kernels (128 registers) against the one-lane kernels and device lock step."""
    model, ctl = cp20
    from warm_start_hmpc_b200.plants import CartPoleWithWalls, DevicePlant
    N, S = 300, 3
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert ctl.default_slots() > sms
    x0 = np.load(os.path.join(MODELS, 'cp20_instances.npy'))[:N]
    d = torch.as_tensor(1e-3 * np.random.default_rng(12).standard_normal((S, N, 4)) * model['x_max'], device='cuda')
    dp = DevicePlant(CartPoleWithWalls(), DT)
    runs = []
    for slots in (8, ctl.default_slots()):
        L = _loop(ctl, N, mode, plant=dp, n_slots=slots)
        L.reset(x0)
        logs = L.run(S, e=d)
        torch.cuda.synchronize()
        runs.append(({k: v.clone() for k, v in logs.items()}, L.x.clone()))
        del L
    L = _loop(ctl, N, mode, plant=dp)
    L.reset(x0)
    xs = []
    for t in range(S):
        L.step(e=d[t]); xs.append(L.x.clone())
    torch.cuda.synchronize()
    _assert_logs_equal(runs[0][0], runs[1][0])
    assert torch.equal(runs[0][1], runs[1][1]) and torch.equal(runs[1][1], L.x)
    assert torch.equal(torch.stack(xs), runs[1][0]['x'])


def test_device_plant_against_the_numpy_plant(cp20):
    """The states of test_closed_loop_against_the_nonlinear_plant: the fused loop with the device plant against lock step
    with the numpy plant -- the same modes at every step, costs within 1e-8."""
    model, ctl = cp20
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    from warm_start_hmpc_b200.plants import CartPoleWithWalls, DevicePlant
    plant = CartPoleWithWalls()
    N, S = 3, 40
    x0 = np.repeat(model['x0_nominal'][None], N, 0) * np.array([1., 0.9, 0.8])[:, None]
    L = ClosedLoop(ctl, N, warm=True, max_solves=2048, max_roots=1024, n_slots=N)
    L.reset(x0)
    costs, modes = [], []
    for t in range(S):
        out, _, _ = L.step_with_plant(lambda x, u0: plant.simulate(x, DT, u0[:, 0]))
        costs.append(out['cost'].cpu().numpy().copy()); modes.append(_modes(ctl, out['primal']))
    F = ClosedLoop(ctl, N, warm=True, max_solves=2048, max_roots=1024, n_slots=N, plant=DevicePlant(plant, DT))
    F.reset(x0)
    logs = F.run(S)
    torch.cuda.synchronize()
    assert logs['status'].cpu().numpy().tolist() == [[0] * N] * S
    # the fused loop logs u0, not the incumbent's binaries: compare the applied binaries of every step
    nu, nub = ctl.mld.nu, ctl.mld.nub
    ub = logs['u0'].cpu().numpy()[:, :, nu - nub:]
    assert np.array_equal(np.round(ub), np.array(modes)[:, :, 0, :])
    c, cr = logs['cost'].cpu().numpy(), np.array(costs)
    assert np.all(np.abs(c - cr) <= 1e-8 * np.abs(cr)), np.abs(c - cr).max()
    assert np.allclose(F.x.cpu().numpy(), L.x.cpu().numpy(), rtol=1e-8, atol=1e-10)


def test_per_instance_parameter_sets_are_independent(cp20):
    model, ctl = cp20
    from warm_start_hmpc_b200.plants import CartPoleWithWalls, DevicePlant
    N, S = 4, 8
    x0 = _states(model, N)
    sets = [CartPoleWithWalls(mp=1. + .2 * (k - 1.5), stiffness=100. * (1. + .2 * (1.5 - k))) for k in range(N)]
    L = _loop(ctl, N, 'warm', plant=DevicePlant(sets, DT), n_slots=N)
    L.reset(x0)
    mixed = {k: v.clone() for k, v in L.run(S).items()}
    with pytest.raises(ValueError, match='parameter sets'):
        L.rebalance()
    for k in range(N):
        Lk = _loop(ctl, N, 'warm', plant=DevicePlant(sets[k], DT), n_slots=N)
        Lk.reset(x0)
        lk = Lk.run(S)
        torch.cuda.synchronize()
        for key in ('cost', 'n_solves', 'status', 'x'):
            assert torch.equal(mixed[key][:, k], lk[key][:, k]), (k, key)
        assert torch.equal(torch.nan_to_num(mixed['u0'][:, k], nan=-7.), torch.nan_to_num(lk['u0'][:, k], nan=-7.))
    # the sets do differ
    assert not torch.equal(mixed['x'][:, 0], mixed['x'][:, 3])


def test_plant_error_paths(cp20):
    model, ctl = cp20
    from warm_start_hmpc_b200 import capi
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    from warm_start_hmpc_b200.plants import CartPoleWithWalls, DevicePlant
    N = 4
    dp = DevicePlant(CartPoleWithWalls(), DT)
    L = _loop(ctl, N, 'warm', plant=dp, n_slots=N)
    L.reset(_states(model, N))
    with pytest.raises(ValueError, match='host is the plant'):
        L.run_mailbox(1, lambda *a: None)
    with pytest.raises(ValueError, match='parameter sets'):
        ClosedLoop(ctl, N, plant=DevicePlant([CartPoleWithWalls()] * 3, DT))
    h = L.h
    x = torch.zeros((N, 4), dtype=torch.float64, device='cuda')
    u = torch.zeros((N, ctl.mld.nu), dtype=torch.float64, device='cuda')
    out = torch.empty_like(x)

    def raw_step(**kw):
        c = capi._plant_struct(dp)
        for k, v in kw.items():
            setattr(c, k, v)
        return h.lib.wshmpc_plant_step(h._h, C.byref(c), N, C.c_void_p(x.data_ptr()), C.c_void_p(u.data_ptr()),
                                       C.c_void_p(out.data_ptr()))
    assert raw_step() == 0
    for kw, msg in ((dict(kind=2), 'kind'), (dict(n_sets=3), 'n_sets'), (dict(dt=0.), 'dt'), (dict(n_sub=0), 'n_sub'),
                    (dict(fc_index=ctl.mld.nu), 'fc_index'), (dict(fc_index=-1), 'fc_index'), (dict(d_params=None), 'parameters')):
        assert raw_step(**kw) != 0, kw
        assert msg in capi.load_library().wshmpc_last_error().decode(), kw
    with pytest.raises(RuntimeError, match='fc_index'):
        DevicePlant(CartPoleWithWalls(), DT, fc_index=ctl.mld.nu).step(h, x, u)
    # a mailbox together with a plant, through the C ABI
    mb = capi.Mailbox(h, N)
    try:
        mb.clear()
        with pytest.raises(RuntimeError, match='mailbox'):
            h.closed_loop(1, True, True, L.cur, L.xbuf, None, L.active, L.trees, L.out, mailbox=mb, plant=dp)
    finally:
        mb.close()
    # nx != 4: the synthetic 20-state model
    syn = load_model('syn30')
    hs = make_controller(syn).handle(1)
    xs = torch.zeros((N, 20), dtype=torch.float64, device='cuda')
    us = torch.zeros((N, hs.pd.nu), dtype=torch.float64, device='cuda')
    with pytest.raises(RuntimeError, match='4 states'):
        hs.plant_step(dp, xs, us)
    torch.cuda.synchronize()
