"""The fallback policy through infeasible MIQPs (ClosedLoop(..., fallback=H)) on one GPU: what it saves and what it costs.

    python tools/fallback_loop.py OUT_DIR            -> OUT_DIR/fallback_loop.json

1. the mismatch sweep of tools/plant_loop.py (512 CP20 instances at x0_nominal, plant i with its own mp and stiffness on a
   16 x 32 grid of +-30 %, 50 warm steps on the device plant) for H in {0, 1, 3, 10, 19}: plants still in the loop after 50
   steps, fallback steps per plant, the longest run of them, QPs per step on solved steps and on the steps right after a
   fallback, ms per MPC step of the batch, and how many plants kept |x| <= x_max (the model's) on every logged state;
2. the published protocol against the true plant (x0_nominal, 50 steps, 100 trajectories per sigma seeded with
   np.random.seed(i), sigma an additive disturbance on the plant output), cold and warm, H = 0 and H = T - 1;
3. no cost when idle: the 512-instance linear loop of tools/loop_timing.py with the existing kernel and with the fallback
   kernel at H = 0, alternated; the logs must be identical.
The GPU's name, power limit and SM clock are read in the same run and written beside the numbers."""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from warm_start_hmpc_b200.instances import load_model, controller_from_model, load_initial_states
from warm_start_hmpc_b200.closed_loop import ClosedLoop
from warm_start_hmpc_b200.plants import CartPoleWithWalls, DevicePlant
from tools.plant_loop import gpu_info

DT = 0.05
N = 512


def _upright(xlog, x_max):
    """[n_inst] bool: |x| <= x_max on every logged state"""
    return np.all(np.abs(xlog) <= x_max[None, None, :] * (1. + 1e-12), axis=(0, 2))


def _qp_split(ns, hold):
    """mean QPs per step over steps t >= 1 with an incumbent, and over the live steps right after a fallback step"""
    live = hold[1:] >= 0
    solved = (hold[1:] == 0)
    after = live & (hold[:-1] > 0)
    m = lambda k: float(ns[1:][k].mean()) if k.any() else None
    return {'qp_per_step_solved': m(solved), 'qp_per_step_after_a_fallback': m(after), 'steps_after_a_fallback': int(after.sum()),
            'qp_per_step_after_a_fallback_solved': m(after & solved), 'qp_per_step_after_a_fallback_infeasible_again': m(after & (hold[1:] > 0))}


def _runs(hold):
    """longest run of consecutive fallback steps of every instance"""
    best = np.zeros(hold.shape[1], dtype=int); cur = np.zeros_like(best)
    for t in range(hold.shape[0]):
        cur = np.where(hold[t] > 0, cur + 1, 0)
        best = np.maximum(best, cur)
    return best


def mismatch_sweep(ctl, model, n_steps=50):
    f_mp, f_k = np.linspace(.7, 1.3, 16), np.linspace(.7, 1.3, 32)
    plants = [CartPoleWithWalls(mp=a, stiffness=100. * b) for a in f_mp for b in f_k]
    dp = DevicePlant(plants, DT)
    out = {'instances': N, 'steps': n_steps, 'mp_factors': f_mp.tolist(), 'stiffness_factors': f_k.tolist(), 'by_H': {}}
    for H in (0, 1, 3, 10, 19):
        L = ClosedLoop(ctl, N, warm=True, max_solves=4096, max_roots=1024, plant=dp, fallback=H)
        if H == 0:
            L.fb = L.h.new_fallback(N, 0)               # the FB kernel at H = 0, for the hold log
        L.reset(np.repeat(model['x0_nominal'][None], N, 0))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        logs = L.run(n_steps)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        hold, ns, st = logs['hold'].cpu().numpy(), logs['n_solves'].cpu().numpy(), logs['status'].cpu().numpy()
        xl = logs['x'].cpu().numpy()
        alive = hold[-1] >= 0
        up = _upright(xl, model['x_max'])
        off = [(int(st[np.nonzero(hold[:, i] < 0)[0][0], i])) for i in range(N) if not alive[i]]
        r = {'in_loop_after_%d_steps' % n_steps: int(alive.sum()),
             'in_loop_and_within_x_max': int((alive & up).sum()),
             'fallback_steps_per_plant': float((hold > 0).sum() / N),
             'plants_with_a_fallback': int((hold > 0).any(axis=0).sum()),
             'longest_fallback_run': int(_runs(hold).max()),
             'left_by_status': {str(k): off.count(k) for k in sorted(set(off))},
             'ms_per_mpc_step': 1e3 * dt / n_steps, 'seconds': dt,
             'in_loop_grid': alive.reshape(16, 32).astype(int).tolist()}
        r.update(_qp_split(ns, hold))
        out['by_H'][str(H)] = r
        print('sweep H=%d' % H, json.dumps({k: v for k, v in r.items() if k != 'in_loop_grid'}), flush=True)
        del L
    return out


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
        row = {'trajectories': int(n)}
        for H in (0, ctl.T - 1):
            res = {}
            for leg in ('cold', 'warm'):
                L = ClosedLoop(ctl, n, warm=leg == 'warm', max_solves=max_solves, max_roots=1024, plant=dp, fallback=H)
                if H == 0:
                    L.fb = L.h.new_fallback(n, 0)
                L.reset(np.repeat(model['x0_nominal'][None], n, 0))
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                logs = L.run(n_steps, e=ed)
                torch.cuda.synchronize()
                res[leg] = dict(n=logs['n_solves'].cpu().numpy(), hold=logs['hold'].cpu().numpy(), x=logs['x'].cpu().numpy(),
                                s=time.perf_counter() - t0)
                del L
            r = {}
            for leg, d in res.items():
                ok = np.all(d['hold'] >= 0, axis=0)
                up = _upright(d['x'], model['x_max'])
                solved = d['hold'][1:] == 0
                r[leg] = {'completed_%d_steps' % n_steps: int(ok.sum()), 'completed_and_within_x_max': int((ok & up).sum()),
                          'fallback_steps': int((d['hold'] > 0).sum()), 'longest_fallback_run': int(_runs(d['hold']).max()),
                          'qp_per_solved_step': float(d['n'][1:][solved & ok[None]].mean()) if (solved & ok[None]).any() else None,
                          'ms_per_mpc_step': 1e3 * d['s'] / n_steps}
            if r['cold']['qp_per_solved_step'] and r['warm']['qp_per_solved_step']:
                r['node_reduction'] = r['cold']['qp_per_solved_step'] / r['warm']['qp_per_solved_step']
            row['H_%d' % H] = r
        out['sigma_%g' % sigma] = row
        print('sigma %g' % sigma, json.dumps(row), flush=True)
    return out


def idle_cost(ctl, model, reps=3, n_windows=2, S=10):
    """the existing kernel against the fallback kernel at H = 0 on the loop_timing.py workload, alternated"""
    x0 = load_initial_states(0, N)
    rng = np.random.default_rng(1)
    e = torch.as_tensor(0.003 * rng.standard_normal((n_windows + 1, S, N, model['A'].shape[0])) * model['x_max'], device='cuda')
    rates = {'existing': [], 'fallback_H0': []}
    logs_of = {}
    for rep in range(reps):
        for leg in ('existing', 'fallback_H0'):
            L = ClosedLoop(ctl, N, warm=True, max_solves=1024, max_roots=512)
            if leg == 'fallback_H0':
                L.fb = L.h.new_fallback(N, 0)
            L.reset(x0)
            L.run(S, e=e[0])
            torch.cuda.synchronize()
            b = L.totals.clone()
            t0 = time.perf_counter()
            got = []
            for w in range(n_windows):
                lg = L.run(S, e=e[w + 1])
                got.append({k: lg[k].clone() for k in ('cost', 'u0', 'n_solves', 'status')})
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            d = (L.totals - b).cpu().numpy()
            rates[leg].append({'qp_per_s': float(d[0] / dt), 'ms_per_mpc_step': 1e3 * dt / (n_windows * S), 'qps': int(d[0])})
            got.append({'x': L.x.clone()})
            if rep == 0:
                logs_of[leg] = got
            del L
    same = True
    for wa, wb in zip(logs_of['existing'], logs_of['fallback_H0']):
        for k in wa:
            same &= bool(torch.equal(torch.nan_to_num(wa[k], nan=-7.), torch.nan_to_num(wb[k], nan=-7.)))
    out = {'instances': N, 'steps_per_window': S, 'timed_windows': n_windows, 'reps': reps, 'rates': rates,
           'outputs_identical': same}
    for leg in rates:
        q = [r['qp_per_s'] for r in rates[leg]]
        out[leg + '_qp_per_s'] = {'mean': float(np.mean(q)), 'min': float(np.min(q)), 'max': float(np.max(q))}
    print('idle', json.dumps(out), flush=True)
    return out


def main():
    out_dir = sys.argv[1]
    os.makedirs(out_dir, exist_ok=True)
    model = load_model('cp20')
    ctl = controller_from_model(model)
    res = {'gpu_before': gpu_info()}
    res['idle_cost'] = idle_cost(ctl, model)
    res['mismatch_sweep'] = mismatch_sweep(ctl, model)
    res['published_protocol_true_plant'] = published_protocol(ctl, model)
    res['gpu_after'] = gpu_info()
    with open(os.path.join(out_dir, 'fallback_loop.json'), 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res['gpu_after']))


if __name__ == '__main__':
    main()
