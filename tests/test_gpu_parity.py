"""-m gpu: parity of the BENCHMARKED regime against the oracle and the reference's golden runs.

The headline numbers come from noisy, multi-instance, warm-started closed loops (lapsing Farkas proofs,
instances that become infeasible, deep shifted trees).  These tests compare exactly that regime with
* tests/golden/cp20_closed_loop.npz `noisy_*`: a noisy trajectory produced by the reference's own
  controller code (oracle/make_golden.py, statistical_analysis.py:93-196 protocol), and
* oracle/bnb_ref.py (restatement pinned bit-exactly against the reference) on oracle/qp_core.c,
on cost (1e-6 relative, north_star), binary mode sequence (exact), applied input, feasibility status per step and
the step at which an instance leaves the loop.  Node COUNTS are compared with a small slack: which of several optimal
multiplier vectors a QP solver returns at a degenerate node decides a child bound here and there (SURVEY.md H3:
Gurobi and HiGHS differ by 1-2 nodes per warm step); the bit-exact explored-set check is tests/test_gpu_facade.py.
"""
import os
import numpy as np
import pytest
import torch

from oracle.models import load_model, GOLDEN, MODELS
from tests.util import make_controller, oracle_loop

pytestmark = pytest.mark.gpu
RTOL = 1e-6


def _ub_of(ctl, primal_row):
    T, nx, nu, nub = ctl.T, ctl.mld.nx, ctl.mld.nu, ctl.mld.nub
    return primal_row[(T + 1) * nx:].reshape(T, nu)[:, nu - nub:]


def test_noisy_golden_trajectory_replay():
    """The noisy (sigma = 0.003) trajectory the REFERENCE's controller code produced (golden `noisy_*`), replayed by
    the device loop with the same model errors: per step cost, mode sequence, applied input, cover of the warm
    start; warm and cold searches agree."""
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    model = load_model('cp20')
    ctl = make_controller(model)
    g = np.load(os.path.join(GOLDEN, 'cp20_closed_loop.npz'))
    e = g['noisy_e']
    S = len(e)
    W = ClosedLoop(ctl, 1, warm=True, max_solves=1024, max_roots=512, n_slots=1)
    Cd = ClosedLoop(ctl, 1, warm=False, max_solves=1024, max_roots=512, n_slots=1)
    W.reset(model['x0_nominal'][None]); Cd.reset(model['x0_nominal'][None])
    for t in range(S):
        assert np.allclose(W.x[0].cpu().numpy(), g['noisy_x'][t], rtol=0, atol=1e-7)
        ed = torch.as_tensor(e[t][None], device='cuda')
        ow = W.step(e=ed); cw = float(ow['cost'][0]); nw = int(ow['n_solves'][0]); ubw = _ub_of(ctl, ow['primal'][0].cpu().numpy()).copy()
        oc = Cd.step(e=ed); cc = float(oc['cost'][0]); nc = int(oc['n_solves'][0])
        assert int(ow['status'][0]) == 0 and int(oc['status'][0]) == 0
        assert abs(cw - g['noisy_cost'][t]) <= RTOL * abs(g['noisy_cost'][t]), (t, cw, g['noisy_cost'][t])
        assert abs(cc - g['noisy_cost'][t]) <= RTOL * abs(g['noisy_cost'][t])
        assert np.array_equal(ubw, g['noisy_ub'][t])                                   # binary mode sequence, exact
        u0 = W.u0[0].cpu().numpy()
        assert np.allclose(u0, g['noisy_u0'][t], rtol=RTOL, atol=1e-7), (t, u0, g['noisy_u0'][t])   # ALL inputs (fc, fl, fr, binaries)
        cover = int(W.trees[W.cur].n_nodes[0])
        assert cover == int(g['noisy_cover'][t]), (t, cover, int(g['noisy_cover'][t]))
        assert abs(nc - int(g['noisy_n_cold'][t])) <= 2, (t, nc, int(g['noisy_n_cold'][t]))
        # warm steps solve ~10 QPs; the device search tends to need FEWER than the golden run (pinned-prefix elimination and
        # the start from the shifted ray give tighter multipliers): never many more
        assert nw <= int(g['noisy_n_warm'][t]) + 3 and nw >= int(g['noisy_n_warm'][t]) - 6, (t, nw, int(g['noisy_n_warm'][t]))


def test_multi_instance_noisy_closed_loop_matches_oracle():
    """32 instances x 12 noisy steps of the bench workload (warm-start-hybrid-mpc_b200/data/cp20_instances.npy,
    sigma = 0.003): the fused device loop against the oracle loop, instance by instance, step by step."""
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    model = load_model('cp20')
    ctl = make_controller(model)
    N, S = 32, 12
    x0 = np.load(os.path.join(MODELS, 'cp20_instances.npy'))[100:100 + N]
    rng = np.random.default_rng(21)
    e = 0.003 * rng.standard_normal((S, N, 4)) * model['x_max']
    L = ClosedLoop(ctl, N, warm=True, max_solves=1024, max_roots=512)
    L.reset(x0)
    # lock-step API: the incumbent's mode sequence is read back every step
    cost = np.zeros((S, N)); status = np.zeros((S, N), int); ns = np.zeros((S, N), int); u0 = np.zeros((S, N, 7)); ubs = []
    for t in range(S):
        out = L.step(e=torch.as_tensor(e[t], device='cuda'))
        cost[t] = out['cost'].cpu().numpy(); status[t] = out['status'].cpu().numpy(); ns[t] = out['n_solves'].cpu().numpy()
        u0[t] = L.u0.cpu().numpy()
        ubs.append(np.stack([_ub_of(ctl, p) for p in out['primal'].cpu().numpy()]))
    # the fused loop gives the same thing (bit for bit)
    F = ClosedLoop(ctl, N, warm=True, max_solves=1024, max_roots=512)
    F.reset(x0)
    logs = F.run(S, e=torch.as_tensor(e, device='cuda'))
    torch.cuda.synchronize()
    assert np.array_equal(logs['cost'].cpu().numpy(), cost) and np.array_equal(logs['n_solves'].cpu().numpy(), ns)
    assert np.all(status <= 1)
    n_dead = 0; worst = 0.; dn = []
    for k in range(N):
        ref = oracle_loop(model, x0[k], e[:, k])
        assert not any('failed' in r for r in ref)
        for t, r in enumerate(ref):
            if np.isinf(r['cost']):
                # the step at which the instance leaves the loop
                assert status[t, k] == 1 and np.isinf(cost[t, k]), (k, t, status[t, k], cost[t, k])
                assert np.all(status[t + 1:, k] == 1)
                n_dead += 1
                break
            assert status[t, k] == 0, (k, t)
            rel = abs(cost[t, k] - r['cost']) / max(abs(r['cost']), 1e-12)
            worst = max(worst, rel)
            assert rel <= RTOL, (k, t, cost[t, k], r['cost'])
            assert np.array_equal(ubs[t][k], np.round(r['ub'])), (k, t)
            assert np.allclose(u0[t, k], r['u0'], rtol=RTOL, atol=1e-6), (k, t, u0[t, k], r['u0'])
            dn.append(ns[t, k] - r['solves'])
    dn = np.array(dn)
    print('multi-instance parity: %d instance-steps, worst relative cost error %.2e, node-count difference mean %.2f max |%d|, '
          '%d instances left the loop' % (len(dn), worst, dn.mean(), np.abs(dn).max(), n_dead))
    # measured on a B200 (round 2): mean -1.3 (the device search solves fewer QPs), mean |difference| 1.8, max 16 on a step of ~100 QPs
    assert dn.mean() <= 1. and np.abs(dn).mean() <= 3.


def test_cp40_warm_start_matches_oracle():
    """BASELINE configs[3] (horizon 40): cold step + 3 warm-started steps with model errors, device vs oracle."""
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    model = load_model('cp40')
    ctl = make_controller(model)
    S = 4
    rng = np.random.default_rng(40)
    e = 0.003 * rng.standard_normal((S, 4)) * model['x_max']
    L = ClosedLoop(ctl, 1, warm=True, max_solves=4096, max_roots=1024, n_slots=1)
    L.reset(model['x0_nominal'][None])
    ref = oracle_loop(model, model['x0_nominal'], e)
    assert len(ref) == S and all(np.isfinite(r['cost']) for r in ref)
    for t in range(S):
        out = L.step(e=torch.as_tensor(e[t][None], device='cuda'))
        assert int(out['status'][0]) == 0
        c = float(out['cost'][0])
        assert abs(c - ref[t]['cost']) <= RTOL * abs(ref[t]['cost']), (t, c, ref[t]['cost'])
        assert np.array_equal(_ub_of(ctl, out['primal'][0].cpu().numpy()), np.round(ref[t]['ub'])), t
        assert np.allclose(L.u0[0].cpu().numpy(), ref[t]['u0'], rtol=RTOL, atol=1e-6), t
        n = int(out['n_solves'][0])
        print('cp40 step %d: %d QPs on the device, %d on the oracle, cover %d / %d'
              % (t, n, ref[t]['solves'], int(L.trees[L.cur].n_nodes[0]), ref[t]['cover']))
        assert abs(n - ref[t]['solves']) <= max(6, ref[t]['solves'] // 20), (t, n, ref[t]['solves'])
    assert ref[1]['solves'] * 3 < ref[0]['solves']          # the warm start pays off on the deep tree too


def test_syn30_bnb_and_shift_match_oracle():
    """BASELINE configs[4] (nx = 20, 8 binaries/step, N = 30: n = 360, 240 binaries): cold B&B, tree shift, one
    warm-started step; reports the largest working set the solver saw (the factor's position capacity is WS_NT)."""
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    model = load_model('syn30')
    ctl = make_controller(model)
    x0 = 0.3 * model['x0_nominal']           # at the full x0_nominal the MIQP needs > 10^4 nodes (best-first stalls at depth 40)
    rng = np.random.default_rng(30)
    e = 0.003 * rng.standard_normal((2, x0.size)) * model['x_max']
    ref = oracle_loop(model, x0, e)
    assert len(ref) == 2 and all(np.isfinite(r['cost']) for r in ref)
    L = ClosedLoop(ctl, 1, warm=True, max_solves=4096, max_roots=2048, n_slots=1)
    L.reset(x0[None])
    for t in range(2):
        out = L.step(e=torch.as_tensor(e[t][None], device='cuda'))
        assert int(out['status'][0]) == 0, int(out['status'][0])
        c = float(out['cost'][0])
        assert abs(c - ref[t]['cost']) <= RTOL * abs(ref[t]['cost']), (t, c, ref[t]['cost'])
        assert np.array_equal(_ub_of(ctl, out['primal'][0].cpu().numpy()), np.round(ref[t]['ub'])), t
        n = int(out['n_solves'][0])
        print('syn30 step %d: %d QPs on the device, %d on the oracle, cover %d / %d' %
              (t, n, ref[t]['solves'], int(L.trees[L.cur].n_nodes[0]), ref[t]['cover']))
        assert abs(n - ref[t]['solves']) <= max(8, ref[t]['solves'] // 10), (t, n, ref[t]['solves'])
    kmax = int(L.totals[3])
    print('syn30: largest working set %d rows (capacity of the removal sweep: %d positions)' % (kmax, 256))
    assert 0 < kmax < 256
