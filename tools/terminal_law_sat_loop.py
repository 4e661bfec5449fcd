"""The saturated and per-plant terminal law on one GPU (ClosedLoop(..., fallback=H, terminal_law=L, law_gain, law_bounds)):
what saturation and per-plant gains change against the linear law of one shared gain.

    python tools/terminal_law_sat_loop.py OUT_DIR            -> OUT_DIR/r07_terminal_law_sat_loop.json

The mismatch sweep of tools/terminal_law_loop.py (512 CP20 instances at x0_nominal, plant i with its own mp and stiffness on a
16 x 32 grid of +-30 %, 50 warm steps on the device plant, one launch per run) at (H, L) in {(0, 50), (19, 50)}, each with
three laws:
  linear        u = K x, K = controller.terminal_law() (the law of r06);
  sat_shared    u = sat(K x), clamped to controller.input_box() (|fc| <= 1, fl, fr >= 0);
  sat_per_plant u = sat(K_i x), K_i = controller.terminal_law(A_i, B_i) on plant i's own model
                (CartPoleWithWalls.discrete_model), the same box.
For every run the columns of tools/terminal_law_loop.py, and the law steps violating a stage row F x + G u <= h split into
those violating an input row (F row zero: what saturation can fix) and those violating a row that involves the state; the
law steps whose unclamped K_i x leaves the box (the steps saturation clamps), and for the per-plant gains the law steps
whose applied input differs from the shared gain's at the same step of the same plant.
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
from tools.fallback_loop import DT, N
from tools.terminal_law_loop import LAW, _stats


def _violations(model, x0, logs, K, lo, hi):
    """law steps violating an input row (F row zero) and a row with the state, and the worst violation of each kind; law
    steps whose unclamped input K_i x leaves the box [lo, hi] (the steps saturation clamps)"""
    hold, xl, u0 = logs['hold'].cpu().numpy(), logs['x'].cpu().numpy(), logs['u0'].cpu().numpy()
    law = hold == LAW
    xs = np.concatenate((np.asarray(x0)[None], xl[:-1]), axis=0)
    v = np.einsum('nrc,tnc->tnr', np.broadcast_to(K, (xs.shape[1],) + K.shape[-2:]), xs)
    out = {'law_steps_with_K_x_outside_the_box': int((law & np.any((v < lo) | (v > hi), axis=2)).sum())}
    viol = np.einsum('ij,tnj->tni', model['F'], xs) + np.einsum('ij,tnj->tni', model['G'], np.nan_to_num(u0)) - model['h']
    tol = 1e-9 * max(1., float(np.abs(model['h']).max()))
    rows = np.all(model['F'] == 0., axis=1)
    for name, sel in (('input_rows', rows), ('state_rows', ~rows)):
        worst = viol[..., sel].max(axis=2)
        out['law_steps_violating_%s' % name] = int((law & (worst > tol)).sum())
        out['worst_%s_violation_on_law_steps' % name] = float(worst[law].max()) if law.any() else None
    return out


def _run(ctl, model, plant, H, L_law, n_steps, **law):
    """one launch of the sweep; returns (the numbers of the run, the logs' hold and u0)"""
    L = ClosedLoop(ctl, N, warm=True, max_solves=4096, max_roots=1024, plant=plant, fallback=H, terminal_law=L_law, **law)
    x0 = np.repeat(model['x0_nominal'][None], N, 0)
    L.reset(x0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    logs = L.run(n_steps)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    r = _stats(model, x0, logs, n_steps, dt)
    lo, hi = ctl.input_box()
    r.update(_violations(model, x0, logs, law.get('law_gain', ctl.terminal_law()), lo, hi))
    r['in_loop_grid'] = (logs['hold'].cpu().numpy()[-1] != -1).reshape(16, 32).astype(int).tolist()
    hold, u0 = logs['hold'].cpu().numpy(), logs['u0'].cpu().numpy()
    del L
    return r, hold, u0


def mismatch_sweep(ctl, model, n_steps=50):
    f_mp, f_k = np.linspace(.7, 1.3, 16), np.linspace(.7, 1.3, 32)
    plants = [CartPoleWithWalls(mp=a, stiffness=100. * b) for a in f_mp for b in f_k]
    dp = DevicePlant(plants, DT)
    nu = ctl.mld.nu
    K_plant = np.stack([ctl.terminal_law(A=A, B=B) for A, B in (p.discrete_model(DT, nu) for p in plants)])
    laws = {'linear': {}, 'sat_shared': dict(law_bounds='model'), 'sat_per_plant': dict(law_gain=K_plant, law_bounds='model')}
    lo, hi = ctl.input_box()
    out = {'instances': N, 'steps': n_steps, 'mp_factors': f_mp.tolist(), 'stiffness_factors': f_k.tolist(),
           'input_box': {'lo': lo.tolist(), 'hi': hi.tolist()}, 'shared_gain': ctl.terminal_law()[0].tolist(),
           'per_plant_gain_fc_row_min': K_plant[:, 0].min(axis=0).tolist(),
           'per_plant_gain_fc_row_max': K_plant[:, 0].max(axis=0).tolist(), 'by_H_L_law': {}}
    for H in (0, ctl.T - 1):
        shared = None
        for name, kw in laws.items():
            r, hold, u0 = _run(ctl, model, dp, H, 50, n_steps, **kw)
            if name == 'sat_shared':
                shared = (hold, u0)
            elif name == 'sat_per_plant':
                # where the per-plant gains applied another input than the shared one, at the same step of the same plant
                law = (hold == LAW) & (shared[0] == LAW)
                r['law_steps_with_another_input_than_sat_shared'] = int((law & np.any(u0 != shared[1], axis=2)).sum())
            out['by_H_L_law']['H%d_L50_%s' % (H, name)] = r
            print('sweep H=%d L=50 %s' % (H, name), json.dumps({k: v for k, v in r.items() if k != 'in_loop_grid'}), flush=True)
    return out


def main():
    out_dir = sys.argv[1]
    os.makedirs(out_dir, exist_ok=True)
    model = load_model('cp20')
    ctl = controller_from_model(model)
    res = {'gpu_before': gpu_info()}
    res['mismatch_sweep'] = mismatch_sweep(ctl, model)
    res['gpu_after'] = gpu_info()
    with open(os.path.join(out_dir, 'r07_terminal_law_sat_loop.json'), 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res['gpu_after']))


if __name__ == '__main__':
    main()
