"""The controller against the TRUE plant (the cart-pole between soft walls, 50 explicit-Euler sub-steps of 1 ms per 50 ms
sample) on one GPU, four ways and three questions.

    python tools/plant_loop.py OUT_DIR            -> OUT_DIR/plant_loop.json

* throughput, 512 CP20 instances from fresh states, a warm-up window and two timed 20-step windows (steps 20-59):
  (a) run(), linear model + model error sigma = .003 (the reference line); (b) run() with the device plant;
  (c) run_mailbox with the numpy plant on the host; (d) step_with_plant in lock step with the numpy plant.
  QP/s, ms per MPC step of the batch, QPs per instance-step; for (c) plant calls per window and host time inside them;
* the published protocol against the true plant: x0_nominal, 50 steps, 100 trajectories per sigma (trajectory i seeded
  with np.random.seed(i)), sigma an additive disturbance on the plant output; cold vs warm;
* a mismatch sweep: 512 instances at x0_nominal, plant i with its own mp and stiffness on a 16 x 32 grid of +-30 %;
* the plant's cost inside the fused loop: (b) against (a') = run() on the linear model fed the model errors the device
  plant produced (recorded in device lock step), i.e. the same trajectories, alternated; and the plant kernel alone.
The GPU's name, power limit and SM clock are read in the same run and written beside the numbers."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from warm_start_hmpc_b200.instances import load_model, controller_from_model, load_initial_states
from warm_start_hmpc_b200.closed_loop import ClosedLoop
from warm_start_hmpc_b200.plants import CartPoleWithWalls, DevicePlant

DT = 0.05
N, S, WINDOWS = 512, 20, 2


def gpu_info():
    q = 'name,power.limit,clocks.sm,clocks.max.sm'
    try:
        line = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=' + q, '--format=csv,noheader'], capture_output=True,
                              text=True, timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(','), [s.strip() for s in line.split(',')]))
    except Exception as ex:
        return {'name': torch.cuda.get_device_name(0), 'error': str(ex)}


def _rate(L, dt, n_steps):
    d = (L.totals - L._t0).cpu().numpy()
    return {'qp_per_s': float(d[0] / dt), 'ms_per_mpc_step': 1e3 * dt / n_steps, 'qp_per_instance_step': float(d[0] / (n_steps * N)),
            'qps': int(d[0]), 'active_at_end': int(L.active.sum())}


def _mark(L):
    torch.cuda.synchronize()
    L._t0 = L.totals.clone()
    return time.perf_counter()


def throughput(ctl, model):
    x0 = load_initial_states(0, N)
    nx = model['A'].shape[0]
    rng = np.random.default_rng(1)
    e = torch.as_tensor(0.003 * rng.standard_normal((WINDOWS + 1, S, N, nx)) * model['x_max'], device='cuda')
    plant = CartPoleWithWalls()
    dp = DevicePlant(plant, DT)
    out = {'instances': N, 'steps_per_window': S, 'timed_windows': WINDOWS}
    mk = lambda **kw: ClosedLoop(ctl, N, warm=True, max_solves=1024, max_roots=512, **kw)
    # (a) linear model + error, (b) device plant
    for leg, kw, ee in (('a_linear_sigma_003', {}, e), ('b_device_plant', dict(plant=dp), None)):
        L = mk(**kw); L.reset(x0)
        L.run(S, e=ee[0] if ee is not None else None)
        t0 = _mark(L)
        for w in range(WINDOWS):
            L.run(S, e=ee[w + 1] if ee is not None else None)
        torch.cuda.synchronize()
        out[leg] = _rate(L, time.perf_counter() - t0, WINDOWS * S)
        print(leg, json.dumps(out[leg]), flush=True)
        del L
    # (c) mailbox, numpy plant on the host
    L = mk(); L.reset(x0)
    x_meas = np.array(x0, dtype=float)
    stats = {'calls': 0, 'seconds': 0., 'instances': 0}

    def host_plant(idx, step, u0, x_pred):
        t = time.perf_counter()
        x_meas[idx] = plant.simulate(x_meas[idx], DT, u0[:, 0])
        stats['calls'] += 1; stats['instances'] += idx.size; stats['seconds'] += time.perf_counter() - t
        return x_meas[idx]
    L.run_mailbox(S, host_plant)
    t0 = _mark(L)
    stats.update(calls=0, seconds=0., instances=0)
    for w in range(WINDOWS):
        L.run_mailbox(S, host_plant)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    r = _rate(L, dt, WINDOWS * S)
    r.update(plant_calls_per_window=stats['calls'] / WINDOWS, instances_per_call=stats['instances'] / max(stats['calls'], 1),
             ms_per_plant_call=1e3 * stats['seconds'] / max(stats['calls'], 1), host_share_in_plant=stats['seconds'] / dt)
    out['c_mailbox_numpy_plant'] = r
    print('c_mailbox_numpy_plant', json.dumps(r), flush=True)
    del L
    # (d) lock step, numpy plant
    L = mk(); L.reset(x0)
    sim = lambda x, u: plant.simulate(x, DT, u[:, 0])
    for _ in range(S):
        L.step_with_plant(sim)
    t0 = _mark(L)
    for _ in range(WINDOWS * S):
        L.step_with_plant(sim)
    torch.cuda.synchronize()
    out['d_lock_step_numpy_plant'] = _rate(L, time.perf_counter() - t0, WINDOWS * S)
    print('d_lock_step_numpy_plant', json.dumps(out['d_lock_step_numpy_plant']), flush=True)
    out['gpu_idle'] = 'not measured (no trace of the persistent mailbox launch); host time inside the plant is reported for (c)'
    return out


def plant_cost(ctl, model):
    """(b) against (a') on the same trajectories, alternated; and the plant kernel alone"""
    x0 = load_initial_states(0, N)
    dp = DevicePlant(CartPoleWithWalls(), DT)
    nx = model['A'].shape[0]
    # the model errors the device plant produces, recorded in device lock step (identical to the fused loop)
    R = ClosedLoop(ctl, N, warm=True, max_solves=1024, max_roots=512, plant=dp)
    R.reset(x0)
    errs = []
    for t in range((WINDOWS + 1) * S):
        out = R.step()
        live = ((R.active != 0) & torch.isfinite(out['cost']))[:, None]
        errs.append(torch.where(live, R.x - out['primal'][:, nx:2 * nx], torch.zeros_like(R.x)))
    e = torch.stack(errs).reshape(WINDOWS + 1, S, N, nx).contiguous()
    del R
    res = {'plant': [], 'linear_same_trajectories': []}
    for rep in range(2):
        for leg in ('plant', 'linear_same_trajectories'):
            L = ClosedLoop(ctl, N, warm=True, max_solves=1024, max_roots=512, plant=dp if leg == 'plant' else None)
            L.reset(x0)
            L.run(S, e=None if leg == 'plant' else e[0])
            t0 = _mark(L)
            for w in range(WINDOWS):
                L.run(S, e=None if leg == 'plant' else e[w + 1])
            torch.cuda.synchronize()
            res[leg].append(_rate(L, time.perf_counter() - t0, WINDOWS * S))
            if leg == 'plant':
                xp = L.x.clone()
            else:
                res[leg][-1]['final_state_max_abs_diff_vs_plant'] = float((L.x - xp).abs().max())
            del L
    print('plant_cost', json.dumps(res), flush=True)
    # the plant kernel alone: one thread per state, 50 sub-steps -- its time is the latency of one integration
    h = ctl.handle(1)
    x = torch.as_tensor(x0, device='cuda'); u = torch.zeros((N, ctl.mld.nu), dtype=torch.float64, device='cuda')
    o = torch.empty_like(x)
    for _ in range(10):
        dp.step(h, x, u)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 200
    a.record()
    for _ in range(reps):
        h.plant_step(dp, x, u, out=o)
    b.record(); torch.cuda.synchronize()
    res['plant_step_kernel_us_per_launch_512_states'] = 1e3 * a.elapsed_time(b) / reps
    res['lanes'] = int(ctl.default_slots())
    print('plant kernel', res['plant_step_kernel_us_per_launch_512_states'], 'us', flush=True)
    return res


def published_protocol(ctl, model, n_traj=100, n_steps=50, max_solves=4096):
    nx = model['A'].shape[0]
    dp = DevicePlant(CartPoleWithWalls(), DT)
    out = {}
    for sigma in (0., 0.001, 0.003, 0.01):
        n = 1 if sigma == 0. else n_traj
        e = np.zeros((n_steps, n, nx))
        for i in range(n):
            np.random.seed(i)                                       # statistical_analysis.py:73
            for t in range(n_steps):
                e[t, i] = sigma * np.multiply(np.random.randn(nx), model['x_max'])
        ed = torch.as_tensor(e, device='cuda') if sigma > 0. else None
        res = {}
        for leg in ('cold', 'warm'):
            L = ClosedLoop(ctl, n, warm=leg == 'warm', max_solves=max_solves, max_roots=1024, plant=dp)
            L.reset(np.repeat(model['x0_nominal'][None], n, 0))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            logs = L.run(n_steps, e=ed)
            torch.cuda.synchronize()
            res[leg] = dict(n=logs['n_solves'].cpu().numpy(), st=logs['status'].cpu().numpy(), c=logs['cost'].cpu().numpy(),
                            s=time.perf_counter() - t0)
            del L
        row = {'trajectories': int(n)}
        ok_all = np.ones(n, bool)
        for leg, r in res.items():
            ok = np.all(r['st'] == 0, axis=0)
            ok_all &= ok
            row[leg] = {'feasible_for_%d_steps' % n_steps: int(ok.sum()),
                        'qp_per_step': float(r['n'][1:, ok].mean()) if ok.any() else None,
                        'max_qp_per_step': int(r['n'][:, ok].max()) if ok.any() else None,
                        'ms_per_mpc_step': 1e3 * r['s'] / n_steps,
                        'infeasible_steps': int(np.sum(r['st'] == 1)),
                        'capacity_or_iteration_limit_steps': int(np.sum(r['st'] >= 2))}
        if row['cold']['qp_per_step'] and row['warm']['qp_per_step']:
            row['node_reduction'] = row['cold']['qp_per_step'] / row['warm']['qp_per_step']
        cc, cw = res['cold']['c'][:, ok_all], res['warm']['c'][:, ok_all]
        row['max_rel_cost_gap_warm_vs_cold'] = float(np.max(np.abs(cw - cc) / np.abs(cc))) if ok_all.any() else None
        out['sigma_%g' % sigma] = row
        print('sigma %g' % sigma, json.dumps(row), flush=True)
    return out


def mismatch_sweep(ctl, model, n_steps=50):
    f_mp, f_k = np.linspace(.7, 1.3, 16), np.linspace(.7, 1.3, 32)
    grid = [(a, b) for a in f_mp for b in f_k]
    plants = [CartPoleWithWalls(mp=a, stiffness=100. * b) for a, b in grid]
    L = ClosedLoop(ctl, N, warm=True, max_solves=4096, max_roots=1024, plant=DevicePlant(plants, DT))
    L.reset(np.repeat(model['x0_nominal'][None], N, 0))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    logs = L.run(n_steps)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    ns = logs['n_solves'].cpu().numpy().reshape(n_steps, 16, 32)
    st = logs['status'].cpu().numpy()
    ok = np.all(st == 0, axis=0).reshape(16, 32)
    first_bad = [int(st[np.nonzero(st[:, i])[0][0], i]) for i in range(N) if st[:, i].any()]
    qp = ns[1:].mean(axis=0)                                        # warm QPs per step (steps >= 1) of every plant
    qp_ok = np.where(ok, qp, np.nan)
    by_mp = [{'mp_factor': float(f_mp[i]), 'feasible_fraction': float(ok[i].mean()),
              'warm_qp_per_step': float(np.nanmean(qp_ok[i])) if ok[i].any() else None} for i in range(16)]
    by_k = [{'stiffness_factor': float(f_k[j]), 'feasible_fraction': float(ok[:, j].mean()),
             'warm_qp_per_step': float(np.nanmean(qp_ok[:, j])) if ok[:, j].any() else None} for j in range(32)]
    dev = np.maximum(np.abs(f_mp[:, None] - 1.), np.abs(f_k[None, :] - 1.))          # largest relative mismatch of a plant
    bands = []
    for lo, hi in ((0., .05), (.05, .1), (.1, .2), (.2, .31)):
        m = (dev >= lo) & (dev < hi)
        bands.append({'max_mismatch': [lo, hi], 'plants': int(m.sum()), 'feasible_fraction': float(ok[m].mean()),
                      'warm_qp_per_step': float(np.nanmean(qp_ok[m])) if ok[m].any() else None})
    res = {'instances': N, 'steps': n_steps, 'mp_factors': f_mp.tolist(), 'stiffness_factors': f_k.tolist(),
           'feasible_fraction': float(ok.mean()), 'warm_qp_per_step': float(np.nanmean(qp_ok)),
           'plants_left_by_status': {str(k): first_bad.count(k) for k in sorted(set(first_bad))},
           'by_mp': by_mp, 'by_stiffness': by_k, 'by_largest_mismatch': bands,
           'qp_per_step_grid': np.round(qp, 2).tolist(), 'feasible_grid': ok.astype(int).tolist(), 'seconds': dt}
    print('sweep', json.dumps({k: res[k] for k in ('feasible_fraction', 'warm_qp_per_step', 'by_largest_mismatch')}), flush=True)
    return res


def main():
    out_dir = sys.argv[1]
    os.makedirs(out_dir, exist_ok=True)
    model = load_model('cp20')
    ctl = controller_from_model(model)
    res = {'gpu_before': gpu_info()}
    res['throughput'] = throughput(ctl, model)
    res['plant_cost'] = plant_cost(ctl, model)
    res['published_protocol_true_plant'] = published_protocol(ctl, model)
    res['mismatch_sweep'] = mismatch_sweep(ctl, model)
    res['gpu_after'] = gpu_info()
    with open(os.path.join(out_dir, 'plant_loop.json'), 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res['gpu_after']))


if __name__ == '__main__':
    main()
