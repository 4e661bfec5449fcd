"""CPU suite (-m "not gpu"), part 2: host logic of the drop-in surface and the C-ABI library.

No compute call is made (there is no GPU here): the library must load, export every symbol
include/wshmpc.h declares, and the product must FAIL LOUDLY (no CPU fallback) when asked to solve.
"""
import ctypes
import os
import re
import numpy as np
import pytest

import warm_start_hmpc_b200 as ws
from warm_start_hmpc_b200 import capi
from warm_start_hmpc_b200.closed_loop import shard
from warm_start_hmpc_b200.subproblem_solution import DualSolution
from oracle.models import load_model, GOLDEN
from oracle.refload import reference_available
from tests.util import make_controller, make_problem, leaves_from_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    import __graft_entry__ as g
    g.build()
    hdr = open(os.path.join(ROOT, 'include', 'wshmpc.h')).read()
    declared = set(re.findall(r'\b(wshmpc_[a-z_]+)\s*\(', hdr))
    assert declared == set(capi.EXPORTS), declared ^ set(capi.EXPORTS)
    lib = ctypes.CDLL(capi.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    ctl = make_controller(load_model('cp1w40'))
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        ctl.feedforward(np.array([0., 0., 1., 0.]), printing_period=None)
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        ctl.feedforward_batch(np.zeros((2, 4)))


def test_mld_and_controller_size_errors():
    """test_mld_system.py:11-30, test_controller.py:12-38: ValueError on inconsistent sizes."""
    m = load_model('cp1w40')
    with pytest.raises(ValueError):
        ws.MLDSystem([m['A'][:3], m['B']], [m['F'], m['G'], m['h']], 2)
    with pytest.raises(ValueError):
        ws.MLDSystem([m['A'], m['B']], [m['F'][:, :3], m['G'], m['h']], 2)
    mld = ws.MLDSystem([m['A'], m['B']], [m['F'], m['G'], m['h']], 2)
    assert mld.V.shape == (2, mld.nu) and np.array_equal(mld.V[:, -2:], np.eye(2))
    with pytest.raises(ValueError):
        ws.HybridModelPredictiveController(mld, 5, [m['Q'][:, :3], m['R'], m['Q_T']], None)
    with pytest.raises(ValueError):
        ws.HybridModelPredictiveController(mld, 5, [m['Q'], m['R'], m['Q_T']], [m['F_T'], m['h_T'][:-1]])


def test_update_matrices():
    """test_controller.py:40-59: rho update exactly 1.1 I on the unit-test fixture; mu update = identity
    on the stage rows, >= 0 and [F G]' M = [F_Tm1 G_Tm1]' with a terminal set."""
    m = load_model('cp1w40')
    ctl = make_controller(m)
    assert np.array_equal(ctl._update['rho'], 1.1 * np.eye(4))
    M = ctl._update['mu']
    nh = m['h'].size
    assert np.array_equal(M[:, :nh], np.eye(nh))
    assert M.min() >= 0.
    assert np.allclose(np.vstack((m['F'].T, m['G'].T)).dot(M), np.vstack((ctl.F_Tm1.T, ctl.G_Tm1.T)), atol=1e-9)
    assert np.allclose(M, m['M_mu'], atol=1e-9)


def test_branch_in_time_and_bounds():
    """controller.py:13-44, 300-327."""
    assert ws.branch_in_time({}, 2) == [{(0, 0): 0.}, {(0, 0): 1.}]
    assert ws.branch_in_time({(0, 0): 1.}, 2) == [{(0, 1): 0.}, {(0, 1): 1.}]
    assert ws.branch_in_time({(0, 0): 1., (0, 1): 0.}, 2) == [{(1, 0): 0.}, {(1, 0): 1.}]
    ctl = make_controller(load_model('cp1w40'))
    lb, ub = ctl._get_bound_binaries({(0, 1): 1., (3, 0): 0.})
    assert lb[0, 1] == ub[0, 1] == 1. and lb[3, 0] == ub[3, 0] == 0. and lb.sum() == 1 and ub.sum() == ub.size - 1


def _knapsack_solver():
    """A toy problem for the generic B&B: minimise c.b over b in {0,1}^4 with a coupling penalty."""
    c = np.array([3., -2., 1.5, -1.])

    def solver(identifier, cutoff, extra):
        fixed = dict((k[1], v) for k, v in identifier.items())
        lb = sum(c[i] * v for i, v in fixed.items()) + sum(min(0., c[i]) for i in range(4) if i not in fixed)
        if fixed.get(1) == 1. and fixed.get(3) == 1.:
            lb = np.inf
        return lb, len(fixed) == 4, 0., None
    return solver


@pytest.mark.parametrize('rule', ['best_first', 'depth_first', 'breadth_first'])
def test_generic_branch_and_bound_equals_reference(rule):
    """branch_and_bound.py:408-563 with arbitrary callables: same incumbent, leaves and solve count as
    the reference implementation (when /root/reference is there), known optimum otherwise."""
    def brancher(node):
        i = len(node.identifier)
        return [ws.Node({**node.identifier, (0, i): v}, node.lb) for v in (0., 1.)]
    inc, leaves, solves, _ = ws.branch_and_bound(_knapsack_solver(), getattr(ws, rule), brancher, printing_period=None)
    assert inc.lb == -2. and inc.identifier == {(0, 0): 0., (0, 1): 1., (0, 2): 0., (0, 3): 0.}
    if reference_available():
        from oracle.refload import import_reference
        _, rb, _, _ = import_reference()
        rinc, rleaves, rsolves, _ = rb.branch_and_bound(
            _knapsack_solver(), getattr(rb, rule),
            lambda node: [rb.Node({**node.identifier, (0, len(node.identifier)): v}, node.lb) for v in (0., 1.)],
            printing_period=None)
        assert rsolves == solves and rinc.identifier == inc.identifier
        assert [l.identifier for l in rleaves] == [l.identifier for l in leaves]
        assert [l.lb for l in rleaves] == [l.lb for l in leaves]


def test_record_round_trip_and_layout():
    model = load_model('cp20')
    pd = make_problem(model)
    L = pd.layout
    assert L.primal == 21 * 4 + 20 * 7 and L.dual == 84 + pd.mc + 160 + 84 + 20
    rec = np.random.default_rng(0).standard_normal(L.dual)
    d = DualSolution.from_record(pd, L, rec, 1.5)
    assert len(d.variables['mu']) == 20 and d.variables['mu'][-1].size == pd.nh1
    assert np.array_equal(DualSolution.to_record(pd, L, d.variables), rec)


def test_host_construct_warm_start_equals_reference_golden():
    """The batched host formulation of construct_warm_start in the product (identifiers a user branch rule may
    produce; prefix identifiers go through kernel K2+K4) on the reference's golden leaves: same cover, same
    dual = None pattern, bounds equal to the reference code's output to rounding (the sums run in another order)."""
    model = load_model('cp20')
    ctl = make_controller(model)
    ctl.device_search = False
    g = np.load(os.path.join(GOLDEN, 'cp20_warmstart.npz'))
    scale = max(1., np.abs(g['dobj']).max())
    for tag, e0 in (('zero', np.zeros(4)), ('rand', g['e_rand'])):
        leaves = [ws.Node(i, lb, ws.SubproblemSolution(None, d)) for i, lb, d in leaves_from_golden(ctl.problem, g)]
        nodes, _, _ = ctl.construct_warm_start(leaves, g['x0'], g['uc0'], g['ub0'], e0)
        assert len(nodes) == 77
        lb, ref = np.array([n.lb for n in nodes]), g['ws_%s_lb' % tag]
        assert np.array_equal(np.isinf(lb), np.isinf(ref))
        fin = np.isfinite(ref)
        assert np.all(np.abs(lb[fin] - ref[fin]) <= 1e-11 * scale)
        none = np.array([n.extra.dual is None for n in nodes])
        assert np.array_equal(none, g['ws_%s_none' % tag])
        dobj = np.array([0. if n.extra.dual is None else n.extra.dual.objective for n in nodes])
        assert np.all(np.abs(dobj[~none] - g['ws_%s_dobj' % tag][~none]) <= 1e-11 * scale)
        wd = np.array([len(n.identifier) for n in nodes])
        assert np.array_equal(wd, g['ws_%s_depth' % tag])
        if tag == 'rand':
            j = int(g['ws_rand_sample'])
            rec = DualSolution.to_record(ctl.problem, ctl.problem.layout, nodes[j].extra.dual.variables)
            assert np.allclose(rec, g['ws_rand_sample_rec'], rtol=1e-13, atol=1e-13)
        # every node carries the start of its solve (multipliers of its shifted dual solution)
        assert all(n.extra.active_set is not None and len(n.extra.active_set['c']) == ctl.qp.NumConstrs for n in nodes)


def test_bounded_qp_surface_without_gpu():
    """The named-family surface of the reference's BoundedQP (bounded_qp.py:127-332) that needs no solve:
    families in the order controller.py:135-166 adds them, rhs edits with the reference's errors, status
    conventions, parameters."""
    model = load_model('cp20')
    ctl = make_controller(model)
    qp = ctl.qp
    T, nx, nu, nub = ctl.T, ctl.mld.nx, ctl.mld.nu, ctl.mld.nub
    assert qp.NumVars == (T + 1) * nx + T * nu and qp.NumConstrs == (T + 1) * nx + 2 * T * nub + ctl.problem.mc
    names = [c.ConstrName for c in qp.getConstrs()]
    assert names[:nx] == ['lam_0[%d]' % i for i in range(nx)] and names[nx] == 'nu_lb_0[0]'
    assert names[nx + 2 * nub] == 'lam_1[0]' and names[2 * nx + 2 * nub] == 'mu_0[0]'
    assert [v.VarName for v in qp.getVars()][:2 * nx + 1] == ['x_0[%d]' % i for i in range(nx)] + ['x_1[%d]' % i for i in range(nx)] + ['uc_0[0]']
    assert np.array_equal(qp.get_constraint_rhs('nu_ub_3'), np.ones(nub)) and np.array_equal(qp.get_constraint_rhs('mu_0'), model['h'])
    assert np.array_equal(qp.get_constraint_rhs('mu_%d' % (T - 1)), ctl.h_Tm1)
    with pytest.raises(ValueError):
        qp.set_constraint_rhs('nu_lb_0', np.zeros(nub + 1))
    with pytest.raises(ValueError):
        qp.set_constraint_rhs('no_such_family', np.zeros(1))
    with pytest.raises(NotImplementedError):
        qp.set_constraint_rhs('mu_0', np.zeros(ctl.problem.nh))
    with pytest.raises(KeyError):
        qp.add_variables(3, lb=[0.] * 3)
    with pytest.raises(ValueError):
        qp.add_constraints([1, 2], None, [1.])
    with pytest.raises(RuntimeError):
        qp.primal_optimizer('x_0')
    with pytest.raises(RuntimeError):
        qp.dual_objective()
    ctl._set_bound_binaries({(0, 0): 1., (2, 3): 0.})
    assert np.array_equal(qp.get_constraint_rhs('nu_lb_0'), [-1., 0., 0., 0.]) and np.array_equal(qp.get_constraint_rhs('nu_ub_2'), [1., 1., 1., 0.])
    qp.setParam('Method', -1); assert qp.Params.Method == -1
    qp.resetParams(); assert qp.Params.Method == 1
    # active-set payload round trip: CBasis of a row = its multiplier, VBasis of the first T*nu variables = proximal centre
    rng = np.random.default_rng(0)
    rec = np.abs(rng.standard_normal(ctl.problem.layout.dual + ctl.problem.n))
    a = qp.active_set_from_record(rec)
    y = qp._signed_multipliers(np.array(a['c']))
    L = ctl.problem.layout
    assert np.array_equal(y[:ctl.problem.mc], rec[L.off_mu:L.off_nu_lb])
    assert np.array_equal(y[ctl.problem.mc:], rec[L.off_nu_ub:L.off_rho] - rec[L.off_nu_lb:L.off_nu_ub])
    assert np.array_equal(np.array(a['v'])[:ctl.problem.n], rec[L.dual:])
    for c, val in zip(qp.getConstrs(), a['c']):
        c.setAttr('CBasis', val)
    assert np.array_equal(qp._cbasis_in, np.array(a['c']))


def test_shard_partition():
    for n, w in ((4096, 8), (10, 4), (3, 8)):
        blocks = [shard(n, r, w) for r in range(w)]
        assert blocks[0][0] == 0 and blocks[-1][1] == n
        assert all(blocks[r][1] == blocks[r + 1][0] for r in range(w - 1))
        assert max(b - a for a, b in blocks) - min(b - a for a, b in blocks) <= 1


@pytest.mark.skipif(not reference_available(), reason='/root/reference only exists in the authoring container')
def test_product_control_flow_equals_reference_on_the_golden_run():
    """The product's host control flow -- branch_and_bound, best_first, _brancher, _solve_subproblem,
    SubproblemSolution.from_controller, construct_warm_start -- against the UNMODIFIED reference classes on the golden
    CP20 run (cold step at x0 = [0, 0, 1, 0], warm start with a model error, warm step), both driving the product's
    BoundedQP front end (its device call replaced by the CPU oracle core: no GPU here).  Bit-identical explored
    sequence, leaves, bounds and costs; warm start bounds to 1e-11 (different summation order)."""
    from oracle.refload import import_reference
    from tests.util import oracle_launch
    model = load_model('cp20')
    ctl = make_controller(model)
    ctl.device_search = False
    asked = {'product': [], 'reference': []}

    def spy(tag, launch):
        def f(x0, lb, ub, y0, yc0):
            asked[tag].append((lb.tobytes(), ub.tobytes(), x0.tobytes(), None if y0 is None else y0.tobytes()))
            return launch(x0, lb, ub, y0, yc0)
        return f
    ctl.qp._launch = spy('product', oracle_launch(model, ctl.problem))
    rc, rb, _, rm = import_reference()
    rqp = ws.BoundedQP(ctl.problem, lambda: None)
    rqp._launch = spy('reference', oracle_launch(model, ctl.problem))

    class Ref(rc.HybridModelPredictiveController):
        def _build_mip(self_):
            return rqp

        def _update_mu(self_):
            return model['M_mu']
    ref = Ref(rm.MLDSystem([model['A'], model['B']], [model['F'], model['G'], model['h']], int(model['nub'])),
              int(model['T']), [model['Q'], model['R'], model['Q_T']], [model['F_T'], model['h_T']])
    g = np.load(os.path.join(GOLDEN, 'cp20_closed_loop.npz'))
    x, e = model['x0_nominal'].copy(), g['noisy_e'][0]
    key = lambda leaves: [sorted(l.identifier.items()) for l in leaves]
    ws_p = ws_r = None
    for step in range(2):
        sp, lp, n_p, _ = ctl.feedforward(x, warm_start=ws_p, printing_period=None)
        sr, lr, n_r, _ = ref.feedforward(x, warm_start=ws_r, printing_period=None)
        assert n_p == n_r and asked['product'] == asked['reference']           # same QPs, same starts, same order
        assert key(lp) == key(lr) and np.array_equal([l.lb for l in lp], [l.lb for l in lr])
        assert sp.objective == sr.objective
        if step == 0:
            assert n_p in (159, 160, 161) and abs(sp.objective - g['noisy_cost'][0]) <= 1e-6 * sp.objective
        uc0, ub0 = sr.variables['uc'][0], sr.variables['ub'][0]
        ws_p, _, _ = ctl.construct_warm_start(lp, x, uc0, ub0, e)
        ws_r, _, _ = ref.construct_warm_start(lr, x, uc0, ub0, e)
        assert key(ws_p) == key(ws_r) and len(ws_p) == int(g['noisy_cover'][0])
        a, b = np.array([l.lb for l in ws_p]), np.array([l.lb for l in ws_r])
        assert np.array_equal(np.isinf(a), np.isinf(b)) and np.all(np.abs(a[np.isfinite(a)] - b[np.isfinite(b)]) <= 1e-11)
        assert [l.extra.dual is None for l in ws_p] == [l.extra.dual is None for l in ws_r]
        # the reference's roots carry no active set (controller.py:487): give both sides the same starts and bounds
        for p, r in zip(ws_p, ws_r):
            r.extra.active_set = p.extra.active_set
            r.lb = p.lb
        x = sr.variables['x'][1] + e
        asked['product'].clear(); asked['reference'].clear()
    assert n_p < 40


def test_product_control_flow_reproduces_the_golden_noisy_loop():
    """The product's host control flow (device_search = False) with the QP answers the golden fixtures were made with
    (oracle core variant 0, every node solved from the empty working set) on the reference's golden noisy CP20 loop
    (cp20_closed_loop.npz): every step the warm-started search reaches the reference's optimum and mode sequence with
    as many QPs, and hands on a warm start of the same size.  The oracle's answers carry the last bits of the host's
    BLAS (tests/test_oracle_cpu.py): costs to 1e-9, and QP counts within 2 where near-ties in best-first order flip."""
    from tests.util import oracle_launch
    model = load_model('cp20')
    ctl = make_controller(model)
    ctl.device_search = False
    ctl.qp.setParam('Method', -1)                    # no active-set hand-over
    launch = oracle_launch(model, ctl.problem, variant=0)
    # the golden run solved every node from the empty working set
    ctl.qp._launch = lambda x0, lb, ub, y0, yc0: launch(x0, lb, ub, None, None)
    g = np.load(os.path.join(GOLDEN, 'cp20_closed_loop.npz'))
    x, ws = model['x0_nominal'].copy(), None
    for t in range(len(g['noisy_cost'])):
        assert np.allclose(x, g['noisy_x'][t], rtol=0, atol=1e-9)
        sol, leaves, n, _ = ctl.feedforward(x, warm_start=ws, printing_period=None)
        assert abs(n - g['noisy_n_warm'][t]) <= 2
        assert abs(sol.objective - g['noisy_cost_warm'][t]) <= 1e-9 * abs(g['noisy_cost_warm'][t])
        assert np.array_equal(np.array(sol.variables['ub']), g['noisy_ub'][t])
        e = g['noisy_e'][t]
        ws, _, _ = ctl.construct_warm_start(leaves, sol.variables['x'][0], sol.variables['uc'][0], sol.variables['ub'][0], e)
        assert len(ws) == g['noisy_cover'][t]
        x = sol.variables['x'][1] + e


def test_miqp_comparator_finds_the_same_optimum():
    """SURVEY.md 8f-1: the Gurobi-free stand-in of `feedforward_gurobi` (controller.py:723-776) -- a conventional MIQP
    branch and bound through the QP seam that ignores the time structure -- must return the optimum the structured
    search returns (the reference asserts exactly this, statistical_analysis.py:171-173), with far more nodes.
    (Device call of the seam replaced by the CPU oracle core: no GPU here.)"""
    from tests.util import oracle_launch
    model = load_model('cp20')
    ctl = make_controller(model)
    ctl.qp._launch = oracle_launch(model, ctl.problem)
    g = np.load(os.path.join(GOLDEN, 'cp20_nodes.npz'))
    variables, objective, nodes, seconds = ctl.feedforward_gurobi(g['x0'], {'OutputFlag': 0, 'MIPGap': 0})
    assert abs(objective - float(g['opt_cost'])) <= 1e-6 * float(g['opt_cost'])
    assert np.array_equal(variables['ub'], g['opt_ub']) and variables['x'].shape == (ctl.T + 1, 4) and variables['uc'].shape == (ctl.T, 3)
    assert nodes > 2 * len(g['status'])          # no dual-bound inheritance, no time structure: many more relaxations
    assert np.allclose(variables['x'][0], g['x0'])


def test_mld_from_symbolic_and_from_pwa():
    """SURVEY.md 8f-4: the modelling builders of the reference's MLDSystem (mld_system.py:68-214).  from_symbolic as in
    the reference's own test (test_mld_system.py:44-68); from_pwa against the reference's output where it is importable
    and against the meaning of the convex-hull formulation everywhere."""
    import sympy as sp
    rng = np.random.default_rng(0)
    nx, nu, nub, nc = 5, 7, 3, 9
    A, B = rng.standard_normal((nx, nx)), rng.standard_normal((nx, nu))
    F, G, h = rng.standard_normal((nc, nx)), rng.standard_normal((nc, nu)), rng.standard_normal(nc)
    x = sp.Matrix(sp.symbols('x:%d' % nx)); u = sp.Matrix(sp.symbols('u:%d' % nu))
    d = sp.Matrix(A) * x + sp.Matrix(B) * u
    c = sp.Matrix(F) * x + sp.Matrix(G) * u - sp.Matrix(h.reshape(nc, 1))
    mld = ws.MLDSystem.from_symbolic(d, c, x, u, nub)
    for got, want in ((mld.A, A), (mld.B, B), (mld.F, F), (mld.G, G), (mld.h, h)):
        np.testing.assert_array_almost_equal(got, want)
    assert sum(sp.Matrix(mld.V) * u - u[-nub:, :]) == 0
    with pytest.raises(ValueError):
        ws.MLDSystem.from_symbolic(d + sp.ones(nx, 1), c, x, u, nub)                # affine dynamics
    # a PWA system with two modes split at x_0 = 0
    nx, nu = 2, 1
    dyn = [[rng.standard_normal((nx, nx)), rng.standard_normal((nx, nu)), rng.standard_normal(nx)] for _ in range(2)]
    box = np.vstack((np.eye(nx + nu), -np.eye(nx + nu)))
    dom = []
    for sgn in (1., -1.):                                  # mode 0: x_0 <= 0, mode 1: x_0 >= 0, both inside |x|, |u| <= 2
        Fi = np.vstack((box[:, :nx], [[sgn, 0.]])); Gi = np.vstack((box[:, nx:], [[0.]])); hi = np.concatenate((2. * np.ones(6), [0.]))
        dom.append([Fi, Gi, hi])
    pwa = ws.MLDSystem.from_pwa([[M.copy() for M in d_] for d_ in dyn], [[M.copy() for M in d_] for d_ in dom])
    assert pwa.nub == 2 and pwa.nu == nu + 2 * (nx + nu) + 2 and np.all(pwa.A == 0.)
    for _ in range(20):
        xk = rng.uniform(-1.5, 1.5, nx); uk = rng.uniform(-1.5, 1.5, nu)
        mode = 0 if xk[0] <= 0 else 1
        for guess in (0, 1):
            v = np.zeros(pwa.nu)
            v[:nu] = uk
            v[nu + guess * nx:nu + (guess + 1) * nx] = xk
            v[nu + 2 * nx + guess * nu:nu + 2 * nx + (guess + 1) * nu] = uk
            v[nu + 2 * (nx + nu) + guess] = 1.
            ok = np.all(pwa.F.dot(xk) + pwa.G.dot(v) <= pwa.h + 1e-12)
            assert ok == (guess == mode)
            if ok:
                assert np.allclose(pwa.A.dot(xk) + pwa.B.dot(v), dyn[mode][0].dot(xk) + dyn[mode][1].dot(uk) + dyn[mode][2])
    if reference_available():
        from oracle.refload import import_reference
        _, _, _, rm = import_reference()
        ref = rm.MLDSystem.from_pwa([[M.copy() for M in d_] for d_ in dyn], [[M.copy() for M in d_] for d_ in dom])
        for name in ('A', 'B', 'F', 'G', 'h'):
            assert np.array_equal(getattr(ref, name), getattr(pwa, name)), name
        xs = sp.Matrix(sp.symbols('x:2')); us = sp.Matrix(sp.symbols('u:1'))
        dsym = [sp.Matrix(d_[0]) * xs + sp.Matrix(d_[1]) * us + sp.Matrix(d_[2].reshape(2, 1)) for d_ in dyn]
        csym = [sp.Matrix(d_[0]) * xs + sp.Matrix(d_[1]) * us - sp.Matrix(d_[2].reshape(-1, 1)) for d_ in dom]
        a, b = ws.MLDSystem.from_symbolic_pwa(dsym, csym, xs, us), rm.MLDSystem.from_symbolic_pwa(dsym, csym, xs, us)
        for name in ('A', 'B', 'F', 'G', 'h'):
            assert np.allclose(getattr(a, name), getattr(b, name)), name


def test_nonlinear_plant():
    """SURVEY.md 8f-4: closed-form cart-pole between soft walls (nonlinear_dynamics.py): its linearisation IS the MLD
    model's (A, B) (explicit Euler, h = 0.05), energy is conserved without forces, the walls push back."""
    from warm_start_hmpc_b200.plants import CartPoleWithWalls
    model = load_model('cp20')
    p = CartPoleWithWalls()
    Ac, Bc = p.linearization()
    assert np.allclose(np.eye(4) + 0.05 * Ac, model['A'], atol=1e-14) and np.allclose(0.05 * Bc, model['B'][:, :3], atol=1e-14)
    J = np.array([(p.x_dot(1e-6 * np.eye(4)[i], 0.) - p.x_dot(-1e-6 * np.eye(4)[i], 0.)) / 2e-6 for i in range(4)]).T
    assert np.abs(J - Ac).max() < 1e-8
    def energy(x):
        c, s = np.cos(x[1]), np.sin(x[1])
        return .5 * (p.mc + p.mp) * x[2] ** 2 - p.mp * p.l * c * x[2] * x[3] + .5 * p.mp * p.l ** 2 * x[3] ** 2 + p.mp * p.g * p.l * c
    x0 = np.array([0., 0.05, 0.1, 0.])
    x1 = p.simulate(x0, 0.2, 0., h_des=1e-5)
    assert abs(energy(x1) - energy(x0)) < 1e-4 * abs(energy(x0))
    # tip inside the right wall, moving in: the wall pushes the tip back (fr > 0, fl = 0); outside: no force
    xin = np.array([0.55, 0., 0.5, 0.])
    fl, fr = p.contact_forces(xin)
    assert fl == 0. and fr > 0. and p.x_dot(xin, 0.)[3] > 0.       # the pole rotates away from the wall (tip x = qc - l sin qp)
    assert p.contact_forces(np.zeros(4)) == (0., 0.)
    # batched
    xb = np.stack((x0, xin)); out = p.simulate(xb, 0.05, np.array([0., 1.]))
    assert out.shape == (2, 4) and np.allclose(out[0], p.simulate(x0, 0.05, 0.))


def test_bench_arguments_follow_the_driver_contract(monkeypatch):
    """`python bench.py --gpus N --steps K --warmup W` is what the driver runs; without flags every workload has its own
    defaults (W >= 3 warm-up steps) and both arms describe the same configuration."""
    import sys
    import bench
    monkeypatch.setattr(sys, 'argv', ['bench.py'])
    a = bench.parse_args()
    assert (a.gpus, a.steps, a.warmup, a.workload, a.impl) == (1, 10, 5, 'cp20', 'b200')
    monkeypatch.setattr(sys, 'argv', ['bench.py', '--gpus', '8', '--steps', '7', '--warmup', '4'])
    a = bench.parse_args()
    assert (a.gpus, a.steps, a.warmup) == (8, 7, 4)
    for w in bench.WORKLOADS:
        monkeypatch.setattr(sys, 'argv', ['bench.py', '--workload', w])
        b = bench.parse_args()
        assert b.warmup >= 3 and b.steps >= 1 and b.instances > 0 and b.window > 0
        monkeypatch.setattr(sys, 'argv', ['bench.py', '--workload', w, '--impl', 'reference'])
        r = bench.parse_args()
        assert bench.workload_config(b, 1) == bench.workload_config(r, 1)


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """--dump-outputs DIR: float64 .npy files of what the last timed step returned; above the size limit the same
    seeded sample of instances in every array, its indices written beside them."""
    import sys
    import bench
    monkeypatch.setattr(sys, 'argv', ['bench.py', '--dump-outputs', str(tmp_path)])
    assert bench.parse_args().dump_outputs == str(tmp_path)
    S, N = 3, 40
    rng = np.random.default_rng(1)
    arrays = {'cost': (rng.standard_normal((S, N)), 1), 'u0': (rng.standard_normal((S, N, 7)), 1),
              'n_solves': (rng.integers(0, 99, (S, N)).astype(np.int32), 1), 'x': (rng.standard_normal((N, 4)), 0)}
    bench.dump_outputs(str(tmp_path / 'all'), arrays)
    for k, (v, _) in arrays.items():
        got = np.load(tmp_path / 'all' / ('%s.npy' % k))
        assert got.dtype == np.float64 and np.array_equal(got, v)
    assert not (tmp_path / 'all' / 'instances.npy').exists()
    monkeypatch.setattr(bench, 'DUMP_LIMIT', 2000)
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), arrays)
    idx = np.load(tmp_path / 'a' / 'instances.npy').astype(int)
    assert 0 < len(idx) < N and np.array_equal(idx, np.load(tmp_path / 'b' / 'instances.npy'))
    assert sum(os.path.getsize(tmp_path / 'a' / ('%s.npy' % k)) for k in arrays) <= 2000 + 4 * 128   # + .npy headers
    for k, (v, axis) in arrays.items():
        assert np.array_equal(np.load(tmp_path / 'a' / ('%s.npy' % k)), np.take(v, idx, axis=axis))
