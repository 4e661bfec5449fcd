"""-m gpu: K1 (batched node QP, through the C ABI) against the CPU oracle and against
solver-independent certificates (oracle/certify.py = the reference fixture's plug-in checkers)."""
import numpy as np
import pytest

from oracle.models import load_model
from oracle.qp_c import CoreC
from oracle.condense import Condensed
from oracle import certify as cert
from tests.util import make_controller, random_nodes, families_from_records, check_node_result, COST_RTOL, PV_SCALED

pytestmark = pytest.mark.gpu


def _check_batch(model, N, seed, n_slots, nodes=None):
    ctl = make_controller(model)
    x0, lb, ub = random_nodes(model, N, seed=seed) if nodes is None else nodes
    h = ctl.handle(n_slots=n_slots)
    out = h.solve_nodes(x0, lb, ub)
    st = out['status'].cpu().numpy(); cost = out['cost'].cpu().numpy(); dobj = out['dobj'].cpu().numpy()
    P = out['primal'].cpu().numpy(); D = out['dual'].cpu().numpy()
    oracle = CoreC(model)
    cond = Condensed(model)
    n_inf = 0
    for i in range(N):
        ref = oracle.solve(x0[i], lb[i], ub[i])
        assert st[i] == ref['status'], (i, st[i], ref['status'])
        check_node_result(model, cond, ctl.problem, h.layout, x0[i], lb[i], ub[i], st[i], cost[i], dobj[i], P[i], D[i],
                          cost_ref=ref.get('cost'), tag=i)
        n_inf += st[i] == 3
    return n_inf


def test_cp20_random_nodes_match_oracle():
    n_inf = _check_batch(load_model('cp20'), 96, seed=0, n_slots=32)
    assert n_inf > 0          # the sample must exercise the Farkas path too


def test_cp20_hot_start_equals_cold_cost():
    """A node solved hot (from another node's working set) must reach the same optimum."""
    model = load_model('cp20')
    ctl = make_controller(model)
    x0, lb, ub = random_nodes(model, 24, seed=3)
    h = ctl.handle(n_slots=24)
    cold = h.solve_nodes(x0, lb, ub)
    hot = h.solve_nodes(x0, lb, ub, slot=np.zeros(24, np.int32), hot=np.ones(24, np.int32))
    sc, sh = cold['status'].cpu().numpy(), hot['status'].cpu().numpy()
    assert np.array_equal(sc, sh)
    cc, ch = cold['cost'].cpu().numpy(), hot['cost'].cpu().numpy()
    ok = sc == 2
    assert np.all(np.abs(cc[ok] - ch[ok]) <= COST_RTOL * np.abs(cc[ok]))


def test_syn30_random_nodes_match_oracle():
    _check_batch(load_model('syn30'), 16, seed=1, n_slots=16)


def test_cp40_random_nodes_match_oracle():
    """BASELINE configs[3]: horizon 40 (n = 280 > threads per CTA, factor columns beyond the shared-memory budget)."""
    n_inf = _check_batch(load_model('cp40'), 12, seed=2, n_slots=12)
    assert n_inf > 0


def test_pins_outside_the_prefix_match_oracle():
    """Only the leading run of pinned binaries is eliminated (problem.py rotation); pins behind a gap stay ordinary
    two-sided rows with lb == ub.  Also the all-pinned leaf (every coordinate of the binaries eliminated)."""
    model = load_model('cp20')
    N = 24
    x0, lb, ub = random_nodes(model, N, seed=5)
    rng = np.random.default_rng(7)
    nb = lb.shape[1]
    for k in range(N - 2):
        d = int(np.argmax(lb[k] != ub[k])) if np.any(lb[k] != ub[k]) else nb
        for j in rng.choice(np.arange(min(d + 2, nb - 1), nb), size=3, replace=False):
            lb[k, j] = ub[k, j] = 0.
    # two fully pinned identifiers: the optimal mode sequence of the golden run, and all zeros
    import os
    from oracle.models import GOLDEN
    g = np.load(os.path.join(GOLDEN, 'cp20_nodes.npz'))
    x0[N - 2] = g['x0']; lb[N - 2] = ub[N - 2] = g['opt_ub'].reshape(-1)
    x0[N - 1] = g['x0']; lb[N - 1] = ub[N - 1] = 0.
    _check_batch(model, N, seed=0, n_slots=12, nodes=(x0, lb, ub))


def test_syn30_dive_nodes_match_golden():
    """BASELINE configs[4] (nx = 20, 8 binaries/step, N = 30: n = 360, m = 2640): the feasible side of K1 on the
    synthetic system -- nodes of a dive frozen by oracle/make_syn30_nodes.py (status, cost), plus certificates."""
    import os
    from oracle.models import GOLDEN
    model = load_model('syn30')
    g = np.load(os.path.join(GOLDEN, 'syn30_nodes.npz'))
    N = len(g['status'])
    assert (g['status'] == 2).sum() >= 8
    ctl = make_controller(model)
    x0 = np.repeat(g['x0'][None], N, 0)
    h = ctl.handle(n_slots=N)
    out = h.solve_nodes(x0, g['lb'], g['ub'])
    st = out['status'].cpu().numpy(); cost = out['cost'].cpu().numpy()
    assert np.array_equal(st, g['status'])
    ok = st == 2
    assert np.all(np.abs(cost[ok] - g['cost'][ok]) <= COST_RTOL * np.abs(g['cost'][ok]))
    cond = Condensed(model)
    P = out['primal'].cpu().numpy(); D = out['dual'].cpu().numpy()
    for i in np.nonzero(ok)[0][:6]:
        fam = families_from_records(ctl.problem, h.layout, 2, P[i], D[i])
        pe, _ = cert.primal_residuals(model, cond, x0[i], g['lb'][i], g['ub'][i], fam)
        pv = cert.primal_violation_scaled(model, cond, x0[i], g['lb'][i], g['ub'][i], fam)
        ds, neg = cert.dual_residuals(model, cond, fam)
        dob = cert.dual_objective(model, cond, x0[i], g['lb'][i], g['ub'][i], fam)
        assert pe <= 1e-9 and pv <= PV_SCALED and ds <= 1e-7 and neg >= 0.
        assert abs(cost[i] - dob) <= 1e-6 * abs(cost[i])
