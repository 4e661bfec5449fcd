"""The terminal law as the last fallback through infeasible MIQPs (ClosedLoop(..., fallback=H, terminal_law=L)) on one GPU:
what it keeps in the loop and what it costs.

    python tools/terminal_law_loop.py OUT_DIR            -> OUT_DIR/terminal_law_loop.json

The protocol of tools/fallback_loop.py, whose helpers it imports:
1. the mismatch sweep (512 CP20 instances at x0_nominal, plant i with its own mp and stiffness on a 16 x 32 grid of +-30 %,
   50 warm steps on the device plant) for (H, L) in {0, 19} x {0, 10, 50};
2. the published protocol against the true plant (x0_nominal, 50 steps, 100 trajectories per sigma seeded with
   np.random.seed(i), sigma an additive disturbance on the plant output), cold and warm, H = T - 1 and L in {0, 50}.
For every run: instances in the loop after 50 steps and those of them with |x| <= x_max on every logged state; law steps per
instance and the longest run of them; law steps whose (x, u) violates the MLD stage rows F x + G u <= h; QPs per step on law
steps and on the steps right after one (solved / infeasible again); ms per MPC step of the batch.
The gain is controller.terminal_law(), the LQR law the model's terminal set and cost were built from.
The GPU's name, power limit and SM clock are read in the same run and written beside the numbers."""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from warm_start_hmpc_b200.instances import load_model, controller_from_model
from warm_start_hmpc_b200.closed_loop import ClosedLoop
from warm_start_hmpc_b200.plants import CartPoleWithWalls, DevicePlant
from tools.plant_loop import gpu_info
from tools.fallback_loop import DT, N, _upright, _runs

LAW = -2            # hold code of a law step


def _stats(model, x0, logs, n_steps, seconds):
    """the per-run numbers of the module docstring from the logs of ClosedLoop.run with a device plant"""
    hold, ns = logs['hold'].cpu().numpy(), logs['n_solves'].cpu().numpy()
    xl, u0 = logs['x'].cpu().numpy(), logs['u0'].cpu().numpy()
    n = hold.shape[1]
    alive = hold[-1] != -1
    up = _upright(xl, model['x_max'])
    law = hold == LAW
    # (x_t, u_t) of every law step: the state the step started from and the law's input
    xs = np.concatenate((np.asarray(x0)[None], xl[:-1]), axis=0)
    viol = np.einsum('ij,tnj->tni', model['F'], xs) + np.einsum('ij,tnj->tni', model['G'], np.nan_to_num(u0)) - model['h']
    worst = viol.max(axis=2)
    tol = 1e-9 * max(1., float(np.abs(model['h']).max()))
    after = law[:-1]                                   # a law step keeps the instance live: the next step is searched
    solved, again = after & (hold[1:] == 0), after & (hold[1:] != 0)
    m = lambda k, a=ns: float(a[k].mean()) if k.any() else None
    return {'in_loop_after_%d_steps' % n_steps: int(alive.sum()),
            'in_loop_and_within_x_max': int((alive & up).sum()),
            'law_steps_per_instance': float(law.sum() / n),
            'instances_with_a_law_step': int(law.any(axis=0).sum()),
            'longest_law_run': int(_runs(law.astype(int)).max()),
            'law_runs_used_up': int(((hold[:-1] == LAW) & (hold[1:] == -1)).sum()),
            'law_steps': int(law.sum()),
            'law_steps_violating_stage_rows': int((law & (worst > tol)).sum()),
            'worst_stage_row_violation_on_law_steps': float(worst[law].max()) if law.any() else None,
            'plan_steps': int((hold > 0).sum()),
            'qp_per_law_step': m(law),
            'steps_after_a_law_step': int(after.sum()),
            'qp_per_step_after_a_law_step_solved': m(solved, ns[1:]),
            'steps_after_a_law_step_solved': int(solved.sum()),
            'qp_per_step_after_a_law_step_infeasible_again': m(again, ns[1:]),
            'ms_per_mpc_step': 1e3 * seconds / n_steps, 'seconds': seconds}


def _run(ctl, model, n, warm, plant, H, L_law, n_steps, e=None):
    L = ClosedLoop(ctl, n, warm=warm, max_solves=4096, max_roots=1024, plant=plant, fallback=H, terminal_law=L_law)
    if L.fb is None:
        L.fb = L.h.new_fallback(n, 0)                   # the FB kernel at H = L = 0, for the hold log
    x0 = np.repeat(model['x0_nominal'][None], n, 0)
    L.reset(x0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    logs = L.run(n_steps, e=e)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    r = _stats(model, x0, logs, n_steps, dt)
    del L
    return r


def mismatch_sweep(ctl, model, n_steps=50):
    f_mp, f_k = np.linspace(.7, 1.3, 16), np.linspace(.7, 1.3, 32)
    dp = DevicePlant([CartPoleWithWalls(mp=a, stiffness=100. * b) for a in f_mp for b in f_k], DT)
    out = {'instances': N, 'steps': n_steps, 'mp_factors': f_mp.tolist(), 'stiffness_factors': f_k.tolist(), 'by_H_L': {}}
    for H in (0, ctl.T - 1):
        for L_law in (0, 10, 50):
            r = _run(ctl, model, N, True, dp, H, L_law, n_steps)
            out['by_H_L']['H%d_L%d' % (H, L_law)] = r
            print('sweep H=%d L=%d' % (H, L_law), json.dumps(r), flush=True)
    return out


def published_protocol(ctl, model, n_traj=100, n_steps=50):
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
        for L_law in (0, 50):
            row['H%d_L%d' % (ctl.T - 1, L_law)] = {leg: _run(ctl, model, n, leg == 'warm', dp, ctl.T - 1, L_law, n_steps, ed)
                                                   for leg in ('cold', 'warm')}
        out['sigma_%g' % sigma] = row
        print('sigma %g' % sigma, json.dumps(row), flush=True)
    return out


def main():
    out_dir = sys.argv[1]
    os.makedirs(out_dir, exist_ok=True)
    model = load_model('cp20')
    ctl = controller_from_model(model)
    res = {'gpu_before': gpu_info(), 'law_gain': ctl.terminal_law().tolist()}
    res['mismatch_sweep'] = mismatch_sweep(ctl, model)
    res['published_protocol_true_plant'] = published_protocol(ctl, model)
    res['gpu_after'] = gpu_info()
    with open(os.path.join(out_dir, 'terminal_law_loop.json'), 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res['gpu_after']))


if __name__ == '__main__':
    main()
