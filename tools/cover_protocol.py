"""How good each step's warm start is, in the fused loop that runs the published experiment: the cover (warm-start roots
handed to the next step, the reference's len(warm_start)), the share of those roots whose Farkas proof lapsed in the shift
(dual = None) and the active-set iterations per QP, from ClosedLoop(..., stats=True).

    python tools/cover_protocol.py OUT_DIR            -> OUT_DIR/cover_protocol.json

* the published protocol as bench.py runs it: x0 = [0, 0, 1, 0], 50 steps, sigma in {0, .001, .003, .01} (100 trajectories,
  trajectory i seeded with np.random.seed(i); one at sigma = 0), warm and cold; the published len(warm_start) statistics
  (BASELINE.md, data/nodes_len_ws_sd_*.npy) beside the device's;
* the same against the true plant on the device (the cart-pole between soft walls, 50 Euler sub-steps per 50 ms sample, sigma
  = .003 an additive disturbance on its output; the setting of tools/plant_loop.py), where the warm start degrades.
Statistics are over steps t >= 1 of the trajectories that stay feasible in both legs; the cover of row t is the warm start
step t hands to step t + 1.  The GPU's name and power limit are read in the same run and written beside the numbers."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from warm_start_hmpc_b200.instances import load_model, controller_from_model
from warm_start_hmpc_b200.closed_loop import ClosedLoop
from warm_start_hmpc_b200.plants import CartPoleWithWalls, DevicePlant
from tools.plant_loop import gpu_info, DT

N_TRAJ, N_STEPS = 100, 50
# BASELINE.md section 1: len(warm_start) of the reference (Gurobi) per step; 423 is the largest of all four sigmas
PUBLISHED = {0.: {'mean': 77., 'max': 77}, 0.001: {'mean': 77., 'max': 77}, 0.003: {'mean': 78.6}, 0.01: {'mean': 86.7}}
PUBLISHED_MAX_ALL = 423


def _errors(model, sigma, n):
    """statistical_analysis.py:73, 176: e[t, i] = sigma * randn(nx) * x_max with np.random.seed(i)"""
    nx = model['A'].shape[0]
    e = np.zeros((N_STEPS, n, nx))
    for i in range(n):
        np.random.seed(i)
        for t in range(N_STEPS):
            e[t, i] = sigma * np.multiply(np.random.randn(nx), model['x_max'])
    return e


def _leg(logs, ok):
    """statistics of one leg over steps >= 1 of the trajectories `ok`"""
    if not ok.any():
        return None
    g = {k: logs[k].cpu().numpy()[1:, ok] for k in ('cover', 'lapsed', 'iters', 'n_solves')}
    c = g['cover']
    return {'cover_mean': float(c.mean()), 'cover_max': int(c.max()), 'cover_min': int(c.min()),
            'steps_with_cover_77': float(np.mean(c == 77)), 'lapsed_share': float(g['lapsed'].sum() / max(c.sum(), 1)),
            'lapsed_per_step': float(g['lapsed'].mean()), 'qp_per_step': float(g['n_solves'].mean()),
            'iters_per_qp': float(g['iters'].sum() / max(g['n_solves'].sum(), 1))}


def protocol(ctl, model, sigma, plant=None, max_solves=2048):
    n = 1 if sigma == 0. else N_TRAJ
    e = _errors(model, sigma, n)
    ed = torch.as_tensor(e, device='cuda') if (sigma > 0. or plant is None) else None
    logs = {}
    for leg in ('warm', 'cold'):
        L = ClosedLoop(ctl, n, warm=leg == 'warm', max_solves=max_solves, max_roots=1024, plant=plant, stats=True)
        L.reset(np.repeat(model['x0_nominal'][None], n, 0))
        logs[leg] = L.run(N_STEPS, e=ed)
        torch.cuda.synchronize()
        del L
    ok = np.all(logs['warm']['status'].cpu().numpy() == 0, axis=0) & np.all(logs['cold']['status'].cpu().numpy() == 0, axis=0)
    row = {'trajectories': int(n), 'feasible_in_both_legs': int(ok.sum()),
           'warm': _leg(logs['warm'], ok), 'cold': _leg(logs['cold'], ok)}
    if row['warm'] and row['cold']:
        row['node_reduction'] = row['cold']['qp_per_step'] / row['warm']['qp_per_step']
    return row


def main():
    out_dir = sys.argv[1]
    os.makedirs(out_dir, exist_ok=True)
    model = load_model('cp20')
    ctl = controller_from_model(model)
    res = {'gpu_before': gpu_info(), 'steps': N_STEPS,
           'statistics': 'steps t >= 1 of the trajectories feasible in both legs; cover = warm-start roots step t hands to '
                         'step t + 1; lapsed_share = roots with dual = None / roots; iters_per_qp = active-set iterations / QPs',
           'published_len_ws': {'sigma_%g' % s: v for s, v in PUBLISHED.items()} | {'max_all_sigmas': PUBLISHED_MAX_ALL}}
    for sigma in (0., 0.001, 0.003, 0.01):
        res['sigma_%g' % sigma] = row = protocol(ctl, model, sigma)
        print('sigma %g' % sigma, json.dumps(row), flush=True)
    row = protocol(ctl, model, 0.003, plant=DevicePlant(CartPoleWithWalls(), DT), max_solves=4096)
    res['true_plant_sigma_0.003'] = row
    print('true plant, sigma .003', json.dumps(row), flush=True)
    res['gpu_after'] = gpu_info()
    with open(os.path.join(out_dir, 'cover_protocol.json'), 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res['gpu_after']))


if __name__ == '__main__':
    main()
