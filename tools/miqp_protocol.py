"""The paper's three curves on one GPU: cold-started B&B, warm-started B&B and the conventional MIQP comparator
(feedforward_miqp, the "Gurobi fair" leg of statistical_analysis.py:93-196) as a device-side search with a MIP start.

    python tools/miqp_protocol.py OUT_DIR            -> OUT_DIR/miqp_protocol.json

* published protocol, three legs: x0 = x0_nominal, sigma in {0, .001, .003, .01}, trajectory i drawn with np.random.seed(i)
  (bench.published_protocol), 100 trajectories (1 at sigma = 0), 50 steps, max_solves = 4096;
* throughput on the bench workload: the fused comparator loop and the warm loop on the 512 CP20 instances, 20-step windows
  after a warm-up window, QP/s, ms per MPC step, eliminated coordinates per QP;
* one instance: feedforward_miqp_device against the host loop feedforward_miqp (one K1 launch per node) at x0_nominal.
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

PUBLISHED = ('BASELINE.md section 1, Gurobi-fair comparator (presolve, cuts and heuristics off): 19-432 nodes per step at '
             'sigma = 0, up to 2040 at sigma = 0.01.  Context only: this comparator has no presolve and no cuts.')


def gpu_info():
    q = 'name,power.limit,clocks.sm,clocks.max.sm'
    try:
        line = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=' + q, '--format=csv,noheader'], capture_output=True,
                              text=True, timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(','), [s.strip() for s in line.split(',')]))
    except Exception as ex:                                        # the numbers still stand; the card is then named by torch
        return {'name': torch.cuda.get_device_name(0), 'error': str(ex)}


def published_protocol(ctl, model, n_traj=100, n_steps=50, max_solves=4096):
    nx = model['A'].shape[0]
    out = {}
    for sigma in (0., 0.001, 0.003, 0.01):
        N = 1 if sigma == 0. else n_traj
        e = np.zeros((n_steps, N, nx))
        for i in range(N):
            np.random.seed(i)                                       # statistical_analysis.py:73
            for t in range(n_steps):
                e[t, i] = sigma * np.multiply(np.random.randn(nx), model['x_max'])      # :176
        ed = torch.as_tensor(e, device='cuda')
        res = {}
        for leg in ('cold', 'warm', 'comparator'):
            if leg == 'comparator':
                L = ClosedLoop(ctl, N, warm=False, comparator=True, mip_start=True, max_solves=max_solves)
            else:
                L = ClosedLoop(ctl, N, warm=leg == 'warm', max_solves=max_solves, max_roots=1024)
            L.reset(np.repeat(model['x0_nominal'][None], N, 0))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            logs = L.run(n_steps, e=ed)
            torch.cuda.synchronize()
            res[leg] = dict(n=logs['n_solves'].cpu().numpy(), st=logs['status'].cpu().numpy(), c=logs['cost'].cpu().numpy(),
                            s=time.perf_counter() - t0)
            del L
        row = {'trajectories': int(N)}
        ok_all = np.ones(N, bool)
        for leg, r in res.items():
            ok = np.all(r['st'] == 0, axis=0)
            ok_all &= ok
            row[leg] = {'feasible_for_%d_steps' % n_steps: int(ok.sum()),
                        'qp_per_step': float(r['n'][1:, ok].mean()) if ok.any() else None,
                        'max_qp_per_step': int(r['n'][:, ok].max()) if ok.any() else None,
                        'ms_per_mpc_step': 1e3 * r['s'] / n_steps,
                        'capacity_hits': int(np.sum(r['st'] >= 2))}      # status 2 (capacity) or 3 (a node QP at the iteration limit)
        cc, cm = res['cold']['c'][:, ok_all], res['comparator']['c'][:, ok_all]
        row['max_rel_cost_gap_comparator_vs_cold'] = float(np.max(np.abs(cm - cc) / np.abs(cc))) if ok_all.any() else None
        out['sigma_%g' % sigma] = row
        print('sigma %g' % sigma, json.dumps(row), flush=True)
    out['published_gurobi_fair'] = PUBLISHED
    return out


def throughput(ctl, model, N=512, S=20, windows=2):
    x0 = load_initial_states(0, N)
    rng = np.random.default_rng(1)
    e = torch.as_tensor(0.003 * rng.standard_normal((windows + 1, S, N, model['A'].shape[0])) * model['x_max'], device='cuda')
    out = {'instances': N, 'steps_per_window': S, 'timed_windows': windows, 'sigma': 0.003}
    for leg in ('warm', 'comparator'):
        if leg == 'warm':
            L = ClosedLoop(ctl, N, warm=True, max_solves=1024, max_roots=512)
        else:
            L = ClosedLoop(ctl, N, warm=False, comparator=True, mip_start=True, max_solves=4096)
        L.reset(x0)
        L.run(S, e=e[0])                                            # warm-up window (module load, first trees)
        torch.cuda.synchronize()
        b = L.totals.clone()
        t0 = time.perf_counter()
        for w in range(windows):
            L.run(S, e=e[w + 1])
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        d = (L.totals - b).cpu().numpy()
        out[leg] = {'qp_per_s': float(d[0] / dt), 'ms_per_mpc_step': 1e3 * dt / (windows * S), 'qps': int(d[0]),
                    'iterations_per_qp': float(d[1] / d[0]), 'eliminated_coordinates_per_qp': float(d[4] / d[0]),
                    'active_at_end': int(L.active.sum())}
        print('throughput', leg, json.dumps(out[leg]), flush=True)
        del L
    return out


def one_instance(ctl, model, reps=3):
    x0 = model['x0_nominal']
    host, dev = [], []
    for _ in range(reps):
        t0 = time.perf_counter(); vh, oh, nh, _ = ctl.feedforward_miqp(x0); host.append(time.perf_counter() - t0)
        t0 = time.perf_counter(); vd, od, nd, _ = ctl.feedforward_miqp_device(x0); dev.append(time.perf_counter() - t0)
    assert nh == nd and oh == od
    return {'nodes': int(nd), 'objective': od, 'host_loop_ms': 1e3 * float(np.median(host)),
            'device_ms': 1e3 * float(np.median(dev)), 'repetitions': reps}


def main():
    out_dir = sys.argv[1]
    os.makedirs(out_dir, exist_ok=True)
    model = load_model('cp20')
    ctl = controller_from_model(model)
    res = {'gpu_before': gpu_info()}
    res['one_instance'] = one_instance(ctl, model)
    print('one instance', json.dumps(res['one_instance']), flush=True)
    res['throughput'] = throughput(ctl, model)
    res['published_protocol'] = published_protocol(ctl, model)
    res['gpu_after'] = gpu_info()
    with open(os.path.join(out_dir, 'miqp_protocol.json'), 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res['gpu_after']))


if __name__ == '__main__':
    main()
