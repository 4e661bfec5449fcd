"""-m gpu: the closed loop's per-step statistics (ClosedLoop(..., stats=True); wshmpc_loop d_log_cover, d_log_lapsed,
d_log_iters).

* on the reference's noisy trajectory the fused loop logs the published cover of 77 every step and the oracle's lapsed counts;
* the fused loop logs what lock step computes from the shifted trees and the search traces, bit for bit: linear model,
  device plant, the fallback policy with the terminal law (on noise and on heavy plants), and the MIQP comparator's cold
  trees; the iterations add up to the launch's totals[1];
* the mailbox loop logs the same three arrays as run(e) when the host answers x_1|t + e_t (the shift of step t runs at
  level t + 1 there);
* asking for the statistics changes nothing else: logs, final states, flags and trees are bit-identical to stats=False,
  whose logs keep exactly their keys.
"""
import os
import numpy as np
import pytest
import torch

from oracle.models import load_model, GOLDEN, MODELS
from tests.util import make_controller
from tests.test_loop_stats_cpu import GOLDEN_NOISY_COVER, GOLDEN_NOISY_LAPSED

pytestmark = pytest.mark.gpu
STATS = ('cover', 'lapsed', 'iters')
N, S = 32, 12                   # the workload of test_gpu_parity.py::test_multi_instance_noisy_closed_loop_matches_oracle


@pytest.fixture(scope='module')
def cp20():
    model = load_model('cp20')
    return model, make_controller(model)


def _case(model, ctl, case, stats):
    """(loop, x0, e [S, N, nx] or None, steps) of one workload"""
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    from warm_start_hmpc_b200.plants import CartPoleWithWalls, DevicePlant
    x0 = np.load(os.path.join(MODELS, 'cp20_instances.npy'))[100:100 + N]
    e = torch.as_tensor(0.003 * np.random.default_rng(21).standard_normal((S, N, 4)) * model['x_max'], device='cuda')
    kw = dict(max_solves=1024, max_roots=512, stats=stats)
    steps = S
    if case == 'linear':
        L = ClosedLoop(ctl, N, warm=True, **kw)
    elif case == 'plant':
        L = ClosedLoop(ctl, N, warm=True, plant=DevicePlant(CartPoleWithWalls(), 0.05), **kw)
    elif case == 'fallback':
        L = ClosedLoop(ctl, N, warm=True, fallback=19, terminal_law=50, **kw)
    elif case == 'plant_fallback':
        # plants heavier than the model from x0_nominal: their MIQPs turn infeasible, hold the plan, then run on the law
        plant = DevicePlant([CartPoleWithWalls(mp=m) for m in np.linspace(1.15, 1.3, N)], 0.05)
        L = ClosedLoop(ctl, N, warm=True, plant=plant, fallback=19, terminal_law=50, max_solves=2048, max_roots=1024, stats=stats)
        x0, e, steps = np.repeat(model['x0_nominal'][None], N, 0), None, 40
    elif case == 'comparator':
        L = ClosedLoop(ctl, N, warm=False, comparator=True, **kw)
    else:
        raise ValueError(case)
    L.reset(x0)
    return L, e, steps


def _lock_step(L, e, steps):
    logs = {k: [] for k in STATS + ('cost', 'n_solves', 'status')}
    for t in range(steps):
        out = L.step(e=e[t] if e is not None else None)
        for k in logs:
            logs[k].append(out[k].clone())
    return {k: torch.stack(v) for k, v in logs.items()}


def _oracle_leaves(pd, layout, tree, nub):
    """the alive leaves of instance 0 of a searched device tree as oracle/bnb_ref.py nodes (identifier, lb, dual record)"""
    from oracle.bnb_ref import Node
    from tests.util import families_from_records
    n = int(tree.n_nodes[0])
    alive, rec, lb = (getattr(tree, k)[0, :n].cpu().numpy() for k in ('alive', 'rec', 'lb'))
    bits, mask = tree.bits[0, :n].cpu().numpy().view(np.uint32), tree.mask[0, :n].cpu().numpy().view(np.uint32)
    duals, dobj = tree.rec_dual[0].cpu().numpy(), tree.rec_dobj[0].cpu().numpy()
    leaves = []
    for j in np.nonzero(alive)[0]:
        assert rec[j] >= 0, j               # every root whose proof lapsed was solved again in the search
        ident = {(q // nub, q % nub): float((bits[j, q >> 5] >> np.uint32(q & 31)) & 1)
                 for q in range(pd.nb) if (mask[j, q >> 5] >> np.uint32(q & 31)) & 1}
        var = families_from_records(pd, layout, 3, None, duals[rec[j], :layout.dual])
        leaves.append(Node(ident, float(lb[j]), dict(variables=var, objective=float(dobj[rec[j]]))))
    return leaves


def test_golden_noisy_trajectory_cover_and_lapsed(cp20):
    """The fused loop along the reference's noisy trajectory (golden noisy_*, sigma = .003): the published cover of 77 every
    step (the cover DESIGN section 5 checks through the lock-step tree), and per step as many lapsed roots as the oracle's
    construct_warm_start finds (dual = None) on the leaves and records of the device's search.  The oracle's own search finds
    the same lapsed counts for steps 0-2 (GOLDEN_NOISY_LAPSED); from step 3 on some of its Farkas proofs differ from the
    device's and lapse where the device's survive the shift (DESIGN section 5)."""
    from oracle.bnb_ref import OracleController
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    model, ctl = cp20
    g = np.load(os.path.join(GOLDEN, 'cp20_closed_loop.npz'))
    e = g['noisy_e']
    W = ClosedLoop(ctl, 1, warm=True, max_solves=1024, max_roots=512, n_slots=1, stats=True)
    W.reset(model['x0_nominal'][None])
    logs = W.run(len(e), e=torch.as_tensor(e[:, None, :], device='cuda'))
    torch.cuda.synchronize()
    assert np.all(logs['status'].cpu().numpy() == 0)
    assert logs['cover'][:, 0].tolist() == GOLDEN_NOISY_COVER == [int(c) for c in g['noisy_cover']]
    assert np.all(logs['iters'].cpu().numpy() > 0)
    # the oracle's warm-start construction on the device's own leaves, step by step in lock step
    octl = OracleController(model, None)
    D = ClosedLoop(ctl, 1, warm=True, max_solves=1024, max_roots=512, n_slots=1, stats=True)
    D.reset(model['x0_nominal'][None])
    lapsed = []
    for t in range(len(e)):
        x = D.x[0].cpu().numpy()
        out = D.step(e=torch.as_tensor(e[t][None], device='cuda'))
        u0 = D.u0[0].cpu().numpy()
        leaves = _oracle_leaves(D.h.pd, D.h.layout, D.trees[1 - D.cur], octl.nub)
        ws = octl.construct_warm_start(leaves, x, u0[:octl.nuc], u0[octl.nuc:], e[t])
        assert len(ws) == int(out['cover'][0]) == int(logs['cover'][t, 0]), t
        lapsed.append(sum(n.dual is None for n in ws))
        assert lapsed[-1] == int(out['lapsed'][0]), t
    assert logs['lapsed'][:, 0].tolist() == lapsed
    assert lapsed[:3] == GOLDEN_NOISY_LAPSED[:3]
    print('lapsed roots per step: device', lapsed, 'oracle search', GOLDEN_NOISY_LAPSED)


@pytest.mark.parametrize('case', ['linear', 'plant', 'fallback', 'plant_fallback', 'comparator'])
def test_fused_equals_lock_step(cp20, case):
    """run() logs what step() reads from the shifted tree (n_nodes, rec <= -2) and sums from the search trace, bit for bit;
    the iterations of a launch are its totals[1]"""
    model, ctl = cp20
    F, e, steps = _case(model, ctl, case, True)
    before = F.totals.clone()
    fused = F.run(steps, e=e)
    torch.cuda.synchronize()
    d_tot = (F.totals - before).cpu().numpy()
    D, e, steps = _case(model, ctl, case, True)
    lock = _lock_step(D, e, steps)
    torch.cuda.synchronize()
    for k in STATS + ('cost', 'n_solves', 'status'):
        assert fused[k].dtype == lock[k].dtype and torch.equal(fused[k], lock[k]), (case, k)
    assert torch.equal(F.x, D.x) and torch.equal(F.active, D.active)
    assert int(fused['iters'].sum()) == int(d_tot[1]) and int(fused['n_solves'].sum()) == int(d_tot[0])
    cover, lapsed = fused['cover'].cpu().numpy(), fused['lapsed'].cpu().numpy()
    off = ~F.active.cpu().numpy().astype(bool)
    assert np.all((lapsed >= 0) & (lapsed <= cover)) and np.all(cover[-1, off] == 0)
    hold = fused['hold'].cpu().numpy() if 'hold' in fused else np.zeros_like(cover)
    print(case, 'cover mean %.1f max %d, lapsed %d of %d roots, %.1f iterations per QP, %d fallback steps, %d instances off'
          % (cover.mean(), cover.max(), lapsed.sum(), cover.sum(), d_tot[1] / d_tot[0], int((hold != 0).sum()), int(off.sum())))
    if case != 'comparator':
        assert lapsed.sum() > 0                     # the warm starts carried proofs that lapsed: the count was exercised
    if case == 'plant_fallback':
        assert np.any(hold > 0) and np.any(hold == -2)


def test_mailbox_logs_equal_run(cp20):
    """run_mailbox answered with x_1|t + e_t and e_t logs the cover, lapsed and iters of run(e): the warm start of step t,
    built at level t + 1 once the host answered, goes to row t -- also across a second launch that resumes the trees"""
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    from warm_start_hmpc_b200.instances import load_initial_states
    model, ctl = cp20
    Sm = 6
    xs = load_initial_states(0, N)
    e = (0.003 * np.random.default_rng(21).standard_normal((2 * Sm, N, 4)) * model['x_max']).reshape(2, Sm, N, 4)
    ref = ClosedLoop(ctl, N, warm=True, max_solves=1024, max_roots=512, stats=True)
    mbx = ClosedLoop(ctl, N, warm=True, max_solves=1024, max_roots=512, stats=True)
    ref.reset(xs); mbx.reset(xs)
    for w in range(2):
        lr = ref.run(Sm, e=torch.as_tensor(e[w], device='cuda'))
        torch.cuda.synchronize()
        lm = mbx.run_mailbox(Sm, lambda idx, step, u0, x1, w=w: (x1 + e[w][step, idx], e[w][step, idx]), timeout_s=60.)
        torch.cuda.synchronize()
        for k in STATS + ('cost', 'n_solves', 'status'):
            assert torch.equal(lr[k], lm[k]), (w, k)
        assert torch.equal(ref.x, mbx.x)
        # the last row: the shift after the host's last answer of the launch
        assert torch.equal(lm['cover'][-1], mbx.trees[mbx.cur].n_nodes)


@pytest.mark.parametrize('case', ['linear', 'plant_fallback', 'comparator'])
def test_stats_change_nothing_else(cp20, case):
    """stats=True against stats=False: every other log, the final states, the active flags, the fallback's state and the
    trees are bit-identical, and the default logs have exactly the keys they have without the statistics"""
    model, ctl = cp20
    runs = {}
    for stats in (False, True):
        L, e, steps = _case(model, ctl, case, stats)
        logs = L.run(steps, e=e)
        torch.cuda.synchronize()
        runs[stats] = (L, logs)
    (A, la), (B, lb) = runs[False], runs[True]
    base = {'cost', 'u0', 'n_solves', 'status'} | ({'x'} if A.plant is not None else set()) | ({'hold'} if A.fb is not None else set())
    assert set(la) == base and set(lb) == base | set(STATS)
    for k in base:
        assert torch.equal(torch.nan_to_num(la[k], nan=-7.), torch.nan_to_num(lb[k], nan=-7.)), (case, k)
    assert torch.equal(A.x, B.x) and torch.equal(A.active, B.active) and torch.equal(A.totals, B.totals)
    for k in ('cost', 'node', 'primal', 'n_solves', 'status'):
        assert torch.equal(torch.nan_to_num(A.out[k], nan=-7.), torch.nan_to_num(B.out[k], nan=-7.)), (case, k)
    if A.fb is not None:
        for k in ('age', 'law_n', 'app_cost', 'app_primal', 'plan'):
            assert torch.equal(A.fb[k], B.fb[k]), (case, k)
    for ta, tb in zip(A.trees, B.trees):
        assert torch.equal(ta.n_nodes, tb.n_nodes) and torch.equal(ta.n_recs, tb.n_recs)
        for i in range(N):
            n, r = int(ta.n_nodes[i]), int(ta.n_recs[i])
            for k in ('depth', 'alive', 'rec', 'bits', 'mask', 'lb'):
                assert torch.equal(getattr(ta, k)[i, :n], getattr(tb, k)[i, :n]), (case, k, i)
            assert torch.equal(ta.rec_dobj[i, :r], tb.rec_dobj[i, :r]) and torch.equal(ta.rec_dual[i, :r], tb.rec_dual[i, :r])
