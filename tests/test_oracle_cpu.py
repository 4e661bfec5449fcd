"""CPU suite (-m "not gpu"), part 1: the oracle pinned against what the reference holds for this path.

* known-answer tests of warm_start_hmpc/test/test_bounded_qp.py:104-189 (feasible QP, Farkas proof)
* KKT / Farkas certificates of warm_start_hmpc/test/cart_pole_with_wall.py:171-268 on the golden nodes
* the reference's OWN controller / branch_and_bound / construct_warm_start code (imported from
  /root/reference when it exists, i.e. in the authoring container) against the oracle restatement
* the golden fixtures under tests/golden (made by oracle/make_golden.py from the reference code) and
  the node counts PUBLISHED in notebooks/cart_pole_with_walls/data (160 cold QPs, cover of 77)
"""
import os
import numpy as np
import pytest

from oracle.models import load_model, GOLDEN
from oracle.qp_c import CoreC
from oracle.qp_numpy import LDP, NodeQP, OPTIMAL, INFEASIBLE
from oracle.condense import Condensed
from oracle import certify as cert
from oracle.bnb_ref import OracleController, closed_loop
from oracle.refload import reference_available


@pytest.fixture(scope='module')
def cp20():
    model = load_model('cp20')
    return model, CoreC(model)


def test_known_answer_feasible():
    """test_bounded_qp.py:104-143: min 1/2|x|^2 s.t. x >= 1  ->  x = 1, multipliers 1, cost n/2."""
    n = 3
    ldp = LDP(np.eye(n))
    st, v, W, lam, it = ldp.solve(np.ones(n), np.full(n, np.inf))
    assert st == OPTIMAL
    assert np.allclose(v, 1.)
    assert sorted(W) == [(i, -1) for i in range(n)]           # lower side active
    assert np.allclose(lam, 1.)                               # |multiplier| 1 (reference: sign -1 for 'ge' rows)
    assert abs(.5 * v.dot(v) - n / 2.) < 1e-12


def test_known_answer_farkas():
    """test_bounded_qp.py:145-189: x <= a < 0 and x >= b > 0 -> Farkas proof p = -q, cost -a.p - b.q > 0."""
    n = 2
    a, b = -1., 2.
    M = np.vstack((np.eye(n), np.eye(n)))
    bl = np.concatenate((np.full(n, -np.inf), np.full(n, b)))
    bu = np.concatenate((np.full(n, a), np.full(n, np.inf)))
    st, p, W, lam, it = LDP(M).solve(bl, bu)
    assert st == INFEASIBLE
    y = np.zeros(2 * n)
    for (r, s), l in zip(W, p):
        y[r] += s * l
    assert np.all(y[:n] >= 0.) and np.all(y[n:] <= 0.)        # p >= 0 on 'le' rows, q <= 0 on 'ge' rows
    assert np.allclose(M.T.dot(y), 0.)                        # p = -q
    cost = -(a * y[:n].sum() + b * y[n:].sum())
    assert cost > 0.


def test_c_core_certificates_on_golden_nodes(cp20):
    """Every 6th of the 160 node QPs the reference B&B solved: status / cost reproduce the fixture and
    the result carries a certificate (cart_pole_with_wall.py:171-268): residuals <= 1e-8, gap <= 1e-8."""
    model, core = cp20
    cond = Condensed(model)
    g = np.load(os.path.join(GOLDEN, 'cp20_nodes.npz'))
    arow = np.linalg.norm(cond.Aall, axis=1)
    for i in range(0, len(g['status']), 6):
        out = core.solve(g['x0'], g['lb'][i], g['ub'][i])
        assert out['status'] == g['status'][i]
        r = cert.certify(model, cond, g['x0'], g['lb'][i], g['ub'][i], out)
        assert r['dual_neg'] >= 0.
        if out['status'] == 2:
            # the fixture holds the bits of one host: the oracle's precompute goes through numpy's BLAS, whose kernels (and
            # last bits) depend on the CPU
            assert abs(out['cost'] - g['cost'][i]) <= 1e-9 * abs(g['cost'][i])
            assert r['prim_eq'] <= 1e-9 and r['prim_viol'] <= 2e-4 and r['dual_stat'] <= 1e-7
            assert abs(r['gap']) <= 1e-6
        else:
            fam = cert.families(model, cond, g['x0'], 3, None, out['y'])
            scale = np.sum(np.concatenate(fam['mu']) * arow[:cond.mc]) + np.sum(np.concatenate(fam['nu_lb'] + fam['nu_ub']))
            assert r['dual_stat'] <= 1e-9 * scale and r['ray_cost'] > 1e-9 * scale
            # the value of a (non-unique) infeasibility proof amplifies the host-BLAS bits above: 4e-9 seen between hosts
            assert abs(out['farkas'] - g['farkas'][i]) <= 1e-6 * abs(g['farkas'][i])


def test_c_core_vs_numpy_referee(cp20):
    """qp_core.c (incremental QR, orthonormal coordinates) vs qp_numpy.py (refactorises every iteration,
    plain condensed coordinates): same status, cost within 1e-6 relative."""
    model, core = cp20
    ref = NodeQP(Condensed(model))
    g = np.load(os.path.join(GOLDEN, 'cp20_nodes.npz'))
    for i in (0, 1, 2, 5, 40, 159):
        a = core.solve(g['x0'], g['lb'][i], g['ub'][i])
        b = ref.solve(g['x0'], g['lb'][i], g['ub'][i])
        assert a['status'] == b['status']
        if a['status'] == 2:
            assert abs(a['cost'] - b['cost']) <= 1e-6 * abs(a['cost'])


def test_published_node_counts():
    """The golden run (reference code + oracle core) reproduces the counts the reference PUBLISHES for
    the nominal loop under Gurobi: 160 cold QPs at step 0 and a warm-start cover of 77 at every step."""
    g = np.load(os.path.join(GOLDEN, 'cp20_closed_loop.npz'))
    assert int(g['published_nodes_cs'][0]) == 160 == int(g['nom_n_cold'][0])
    assert np.all(g['published_nodes_len_ws'][:len(g['nom_cover'])] == 77) and np.all(g['nom_cover'] == 77)
    # later steps are dual-dependent (SURVEY.md H3): within a few nodes of Gurobi's
    k = len(g['nom_n_cold'])
    assert np.all(np.abs(g['nom_n_cold'] - g['published_nodes_cs'][:k]) <= 2)
    assert np.all(np.abs(g['nom_n_warm'][1:] - g['published_nodes_ws'][1:k]) <= 6)
    assert np.allclose(g['nom_cost'], g['nom_cost_warm'], rtol=1e-9)


def test_restatement_reproduces_golden_closed_loop(cp20):
    """oracle/bnb_ref.py (what bench.py times on the GPU box) == the reference code's golden run."""
    model, core = cp20
    g = np.load(os.path.join(GOLDEN, 'cp20_closed_loop.npz'))
    ctl = OracleController(model, core, hot_start=False)
    log = closed_loop(ctl, model['x0_nominal'], 3, warm=True)
    for t, s in enumerate(log):
        assert abs(s['cost'] - g['nom_cost_warm'][t]) <= 1e-9 * g['nom_cost_warm'][t]      # host BLAS: see above
        assert s['solves'] == g['nom_n_warm'][t]
        assert s['cover'] == g['nom_cover'][t]
        assert np.array_equal(s['ub'], g['nom_ub'][t])


def test_restatement_warm_start_equals_golden(cp20):
    """construct_warm_start restated (bnb_ref.py) on the golden leaves vs the reference's output."""
    model, core = cp20
    from tests.util import make_problem, leaves_from_golden
    g = np.load(os.path.join(GOLDEN, 'cp20_warmstart.npz'))
    pd = make_problem(model)
    ctl = OracleController(model, core)
    from oracle.bnb_ref import Node
    leaves = [Node(ident, lb, None if dual is None else dict(variables=dual.variables, objective=dual.objective))
              for ident, lb, dual in leaves_from_golden(pd, g)]
    for tag, e0 in (('zero', np.zeros(4)), ('rand', g['e_rand'])):
        ws = ctl.construct_warm_start(leaves, g['x0'], g['uc0'], g['ub0'], e0)
        assert len(ws) == len(g['ws_%s_lb' % tag]) == 77
        lb = np.array([n.lb for n in ws])
        assert np.array_equal(lb, g['ws_%s_lb' % tag])
        assert [len(n.identifier) for n in ws] == list(g['ws_%s_depth' % tag])


@pytest.mark.skipif(not reference_available(), reason='/root/reference only exists in the authoring container')
def test_bnb_restatement_equals_reference(cp20):
    """The unmodified reference controller (controller.py, branch_and_bound.py, subproblem_solution.py)
    and oracle/bnb_ref.py, both on the oracle QP core: same explored nodes, leaves, cost, warm start."""
    model, core = cp20
    from oracle.ref_facade import make_reference_controller
    x0 = model['x0_nominal'] * 0.9 + np.array([0.02, 0.005, 0., -0.03])
    rc = make_reference_controller(model, lambda x, lb, ub: core.solve(x, lb, ub))
    sol, leaves, n_qp, _ = rc.feedforward(x0, printing_period=None)
    oc = OracleController(model, core, hot_start=False)
    order = []
    inc, oleaves, osolves = oc.feedforward(x0, on_solve=lambda n: order.append(dict(n.identifier)))
    assert osolves == n_qp and inc.primal['objective'] == sol.objective
    # explored order: the facade logged the bounds of every reference solve
    assert len(order) == len(rc.qp.log)
    for ident, (_, lb, ub, _) in zip(order, rc.qp.log):
        l2, u2 = oc.bounds(ident)
        assert np.array_equal(l2.ravel(), lb) and np.array_equal(u2.ravel(), ub)
    assert [l.identifier for l in oleaves] == [l.identifier for l in leaves]
    assert [l.lb for l in oleaves] == [l.lb for l in leaves]
    e0 = 0.002 * np.array([1., -1., .5, 2.])
    uc0, ub0 = sol.variables['uc'][0], sol.variables['ub'][0]
    ws, _, _ = rc.construct_warm_start(leaves, x0, uc0, ub0, e0)
    ows = oc.construct_warm_start(oleaves, x0, uc0, ub0, e0)
    assert [n.identifier for n in ows] == [n.identifier for n in ws]
    assert np.array_equal(np.array([n.lb for n in ows]), np.array([n.lb for n in ws]))
    x1 = sol.variables['x'][1] + e0
    s2, l2, n2, _ = rc.feedforward(x1, warm_start=ws, printing_period=None)
    i2, ol2, on2 = oc.feedforward(x1, warm_start=ows)
    assert on2 == n2 and i2.primal['objective'] == s2.objective


def test_thin_factor_variant_agrees_with_full_factor():
    """oracle/qp_core.c variant 1 (thin Q1 + R^-1, the CUDA kernel's factorisation) against variant 0
    (full Q + R by Householder): same status on every node, same cost to 1e-9, certificates hold."""
    from tests.util import random_nodes
    model = load_model('cp20')
    a, b = CoreC(model, variant=0), CoreC(model, variant=1)
    cond = Condensed(model)
    x0, lb, ub = random_nodes(model, 24, seed=4)
    same_iters = 0
    for i in range(len(x0)):
        ra, rb = a.solve(x0[i], lb[i], ub[i]), b.solve(x0[i], lb[i], ub[i])
        assert ra['status'] == rb['status']
        same_iters += ra['iters'] == rb['iters']
        if ra['status'] == OPTIMAL:
            assert abs(ra['cost'] - rb['cost']) <= 1e-9 * abs(ra['cost'])
            bl, bu = cond.bounds(x0[i], lb[i], ub[i])
            r = cond.Aall.dot(rb['z'])
            assert np.all(r <= bu + 2e-4) and np.all(r >= bl - 2e-4)      # same tolerance as tests/test_gpu_qp.py (tol_p is in scaled rows)
    assert same_iters >= len(x0) - 4          # same pivoting rules: identical paths except at rounding-level ties


def test_persistent_state_and_record_start_reach_the_same_optimum():
    """The three start policies of the oracle (from scratch / persistent factor = a CUDA slot / the dual
    solution the node carries = the reference's active_set hand-over) give the same branch and bound
    optimum and mode sequence on the nominal instance."""
    model = load_model('cp20')
    ref = None
    for kw in (dict(hot_start=False), dict(persistent=True), dict(hot_start='record')):
        ctl = OracleController(model, CoreC(model, variant=1), **kw)
        inc, leaves, solves = ctl.feedforward(model['x0_nominal'])
        assert inc is not None and abs(solves - 160) <= 2
        cur = (inc.primal['objective'], inc.primal['u'][:, ctl.nuc:].copy())
        if ref is None:
            ref = cur
        assert abs(cur[0] - ref[0]) <= 1e-9 * abs(ref[0]) and np.array_equal(cur[1], ref[1])


def test_syn30_golden_nodes_reproduce():
    """tests/golden/syn30_nodes.npz (oracle/make_syn30_nodes.py): the frozen statuses and costs are what the oracle
    computes today (first and last nodes only: the synthetic system is slow on the CPU)."""
    import os
    from oracle.models import GOLDEN
    model = load_model('syn30')
    g = np.load(os.path.join(GOLDEN, 'syn30_nodes.npz'))
    core = CoreC(model)
    for i in (0, len(g['status']) - 2, len(g['status']) - 1):
        r = core.solve(g['x0'], g['lb'][i], g['ub'][i])
        assert r['status'] == g['status'][i]
        if r['status'] == 2:
            assert abs(r['cost'] - g['cost'][i]) <= 1e-9 * abs(g['cost'][i])
