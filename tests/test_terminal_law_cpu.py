"""The terminal law of the fallback policy (wshmpc_fallback.max_law, ClosedLoop(..., terminal_law=L)) on the host: the gain
of controller.terminal_law() against the model's terminal cost and set, a numpy statement of the extended policy table that
the GPU tests replay, and the argument checks of ClosedLoop that need no GPU."""
import numpy as np
import pytest

from tests.test_fallback_cpu import policy

LAW = -2            # hold code of a law step


def policy_law(live, has_inc, status, age, law_n, H, L):
    """The policy of one instance-step with the terminal law (include/wshmpc.h, wshmpc_fallback), elementwise on numpy
    arrays: returns (source, hold, active after the step, age after the step, law_n after the step); source 0 the incumbent,
    1 the plan, 2 the law, -1 none."""
    live, has_inc = np.asarray(live, bool), np.asarray(has_inc, bool)
    status, age, law_n = np.asarray(status), np.asarray(age), np.asarray(law_n)
    inc = live & has_inc
    plan = live & ~has_inc & (status == 1) & (age >= 0) & (age + 1 <= H)
    law = live & ~has_inc & (status == 1) & ~plan & (law_n + 1 <= L)
    source = np.where(inc, 0, np.where(plan, 1, np.where(law, 2, -1)))
    hold = np.where(inc, 0, np.where(plan, age + 1, np.where(law, LAW, -1)))
    new_age = np.where(inc, 0, np.where(plan, age + 1, age))
    new_n = np.where(inc, 0, np.where(law, law_n + 1, law_n))
    return source, hold, (source >= 0).astype(int), new_age, new_n


def fallback_reference(A, B, K, T, H, L, live, status, cost, age, law_n, x, plan, inc):
    """What wshmpc_fallback_step writes for one step of n instances (include/wshmpc.h, wshmpc_fallback), with the arithmetic in
    np.longdouble: the policy of policy_law, then per instance the applied cost, the new plan and, on plan and law steps,
    u_0 (u_a of the plan, or K x) and x_1 = A x + B u_0.  x [n, nx], plan and inc [n, primal] (records x_0..x_T, u_0..u_T-1).
    Returns a dict: source, hold, active, age, law_n, app_cost, plan, u [n, nu] and x1 [n, nx] (long double; NaN where the
    step applies neither), u_terms and x1_terms (sums of the magnitudes of the products each entry is summed from)."""
    source, hold, active, new_age, new_n = policy_law(live, np.isfinite(cost), status, age, law_n, H, L)
    ld = np.longdouble
    nx, nu = B.shape
    U = (T + 1) * nx
    A_, B_, K_ = (np.asarray(M, dtype=ld) for M in (A, B, K))
    u = np.full((len(source), nu), np.nan, dtype=ld); u_terms = np.zeros((len(source), nu))
    x1 = np.full((len(source), nx), np.nan, dtype=ld); x1_terms = np.zeros((len(source), nx))
    for i in np.nonzero(source > 0)[0]:
        xi = np.asarray(x[i], dtype=ld)
        if source[i] == 1:
            u[i] = plan[i, U + hold[i] * nu:U + (hold[i] + 1) * nu]
            u_err = np.zeros(nu)
        else:
            u[i] = K_.dot(xi)
            u_terms[i] = u_err = np.abs(K).dot(np.abs(x[i]))
        x1[i] = A_.dot(xi) + B_.dot(u[i])
        # the device forms u in double first: its rounding reaches x_1 through B
        x1_terms[i] = np.abs(A).dot(np.abs(x[i])) + np.abs(B).dot(np.abs(u[i].astype(float)) + u_err)
    app_cost = np.where(source == 0, cost, np.where(source > 0, 0., np.inf))
    new_plan = np.where((source == 0)[:, None], inc, plan)
    return dict(source=source, hold=hold, active=active, age=new_age, law_n=new_n, app_cost=app_cost, plan=new_plan, u=u,
                x1=x1, u_terms=u_terms, x1_terms=x1_terms)


def replay_law(status, cost, H, L, active0=None):
    """hold [n_steps, n_inst] the policy gives to the logs of a loop (status, cost [n_steps, n_inst]) started without plans"""
    S, N = status.shape
    live = np.ones(N, bool) if active0 is None else np.asarray(active0, bool)
    age, n = np.full(N, -1), np.zeros(N, dtype=int)
    hold = np.zeros((S, N), dtype=int)
    for t in range(S):
        _, hold[t], act, age, n = policy_law(live, np.isfinite(cost[t]), status[t], age, n, H, L)
        live = act.astype(bool)
    return hold


def test_policy_table_hand_built_cases():
    H, L = 3, 2
    # (live, has incumbent, status, age, law_n) -> (source, hold, active, age after, law_n after)
    cases = [
        ((1, 1, 0, -1, 0), (0, 0, 1, 0, 0)),        # first incumbent
        ((1, 1, 0, -1, 2), (0, 0, 1, 0, 0)),        # an incumbent resets the law counter
        ((1, 1, 2, 3, 1), (0, 0, 1, 0, 0)),         # capacity with an incumbent: applied as today, counter reset
        ((1, 0, 1, -1, 0), (2, -2, 1, -1, 1)),      # infeasible without a plan: the law
        ((1, 0, 1, -1, 1), (2, -2, 1, -1, 2)),      # ... its second step
        ((1, 0, 1, -1, 2), (-1, -1, 0, -1, 2)),     # law used up: off
        ((1, 0, 1, 0, 0), (1, 1, 1, 1, 0)),         # a plan comes before the law
        ((1, 0, 1, 2, 0), (1, 3, 1, 3, 0)),         # ... up to u_H
        ((1, 0, 1, 3, 0), (2, -2, 1, 3, 1)),        # plan used up: the law, age kept
        ((1, 0, 1, 3, 1), (2, -2, 1, 3, 2)),
        ((1, 0, 1, 3, 2), (-1, -1, 0, 3, 2)),       # plan and law used up: off
        ((1, 0, 2, 3, 0), (-1, -1, 0, 3, 0)),       # capacity without an incumbent: no complete cover to shift, off
        ((1, 0, 3, -1, 0), (-1, -1, 0, -1, 0)),     # QP iteration limit: off
        ((1, 0, 2, 0, 0), (-1, -1, 0, 0, 0)),
        ((0, 0, 1, -1, 0), (-1, -1, 0, -1, 0)),     # an instance already off stays off
        ((0, 1, 0, 0, 1), (-1, -1, 0, 0, 1)),
    ]
    for (lv, hi, st, a, n), want in cases:
        got = tuple(int(np.asarray(v)) for v in policy_law(lv, hi, st, a, n, H, L))
        assert got == want, ((lv, hi, st, a, n), got, want)


def test_without_the_law_it_is_the_policy_of_today():
    grid = np.array([(lv, hi, st, a, n) for lv in (0, 1) for hi in (0, 1) for st in (0, 1, 2, 3) for a in (-1, 0, 1, 2, 3, 5)
                     for n in (0, 1, 4)]).T
    for H in (0, 1, 3, 19):
        src, hold, act, age, n = policy_law(*grid, H, 0)
        s0, h0, a0, g0 = policy(*grid[:4], H)
        assert np.array_equal(src, s0) and np.array_equal(hold, h0) and np.array_equal(act, a0) and np.array_equal(age, g0)
        assert np.array_equal(n, np.where(grid[0] & grid[1], 0, grid[4]))


def test_replay_runs_of_law_steps():
    inf = np.inf
    # infeasible from step 0: no plan, the law for L steps, then off
    st = np.ones((6, 1), dtype=int)
    assert replay_law(st, np.full((6, 1), inf), 3, 2)[:, 0].tolist() == [-2, -2, -1, -1, -1, -1]
    # solved, 5 infeasible steps: the plan for H = 2, the law for L = 2, off
    st = np.array([0, 1, 1, 1, 1, 1, 1])[:, None]
    cost = np.where(st == 0, 1., inf)
    assert replay_law(st, cost, 2, 2)[:, 0].tolist() == [0, 1, 2, -2, -2, -1, -1]
    # back to an incumbent after law steps: the counter starts again
    st = np.array([1, 1, 0, 1, 1, 1, 0])[:, None]
    cost = np.where(st == 0, 1., inf)
    assert replay_law(st, cost, 0, 2)[:, 0].tolist() == [-2, -2, 0, -2, -2, -1, -1]
    assert replay_law(st, cost, 1, 2)[:, 0].tolist() == [-2, -2, 0, 1, -2, -2, 0]


def test_fallback_reference_reproduces_the_policy_table():
    """The numpy reference of wshmpc_fallback_step on the hand-built grid of test_gpu_fallback.py's policy-table test (CP20,
    H = 3, without the law), held to what that test asserts of the kernel, then with a law (L = 2) and on values worked out
    by hand."""
    from oracle.models import load_model
    from tests.test_fallback_cpu import policy
    model = load_model('cp20')
    A, B = model['A'], model['B']
    T, nx, nu, H = int(model['T']), A.shape[0], B.shape[1], 3
    P, U = (T + 1) * nx + T * nu, (T + 1) * nx
    grid = [(lv, hi, st, a) for lv in (0, 1) for hi in (0, 1) for st in (0, 1, 2, 3) for a in (-1, 0, 1, 2, 3)
            if not (hi and st == 1)]
    N = len(grid)
    lv, hi, st, age = (np.array(c) for c in zip(*grid))
    rng = np.random.default_rng(0)
    x = rng.standard_normal((N, nx))
    plan = rng.standard_normal((N, P)); inc = rng.standard_normal((N, P))
    cost = np.where(hi == 1, rng.uniform(1., 2., N), np.inf)
    K = rng.standard_normal((nu, nx))
    ref = fallback_reference(A, B, K, T, H, 0, lv, st, cost, age, np.zeros(N, int), x, plan, inc)
    src, hold, act, new_age = policy(lv, hi, st, age, H)
    assert np.array_equal(ref['hold'], hold) and np.array_equal(ref['age'], new_age)
    assert np.array_equal(np.isfinite(ref['app_cost']), act == 1) and np.array_equal(ref['source'], src)
    for i in range(N):
        if src[i] == 0:
            assert ref['app_cost'][i] == cost[i] and np.array_equal(ref['plan'][i], inc[i])
        else:
            assert np.array_equal(ref['plan'][i], plan[i])
        if src[i] == 1:
            u = plan[i, U + hold[i] * nu:U + (hold[i] + 1) * nu]
            assert np.array_equal(ref['u'][i].astype(float), u)
            assert np.allclose(ref['x1'][i].astype(float), A.dot(x[i]) + B.dot(u), rtol=1e-13, atol=1e-14)
        else:
            assert np.isnan(ref['u'][i].astype(float)).all() and np.isnan(ref['x1'][i].astype(float)).all()
    # with the law: the plan first, then K x
    n = np.array([0, 1, 2] * (N // 3 + 1))[:N]
    law = fallback_reference(A, B, K, T, H, 2, lv, st, cost, age, n, x, plan, inc)
    s2, h2, _, a2, n2 = policy_law(lv, hi, st, age, n, H, 2)
    assert np.array_equal(law['hold'], h2) and np.array_equal(law['age'], a2) and np.array_equal(law['law_n'], n2)
    assert (s2 == 2).any()
    for i in np.nonzero(s2 == 2)[0]:
        assert law['app_cost'][i] == 0.
        assert np.allclose(law['u'][i].astype(float), K.dot(x[i]), rtol=1e-13, atol=1e-14)
        assert np.allclose(law['x1'][i].astype(float), A.dot(x[i]) + B.dot(K.dot(x[i])), rtol=1e-13, atol=1e-13)
    # by hand: nx = 2, nu = 1, T = 2; the record is x_0 x_1 x_2 | u_0 u_1
    A2, B2, K2 = np.array([[1., 2.], [0., 1.]]), np.array([[0.], [3.]]), np.array([[-1., 0.5]])
    plan2 = np.array([[0., 0., 0., 0., 0., 0., 10., 20.]] * 3)
    r = fallback_reference(A2, B2, K2, 2, 1, 1, [1, 1, 1], [1, 1, 0], [np.inf, np.inf, 7.], [0, 1, 0], [0, 0, 0],
                           np.array([[1., 1.]] * 3), plan2, np.full((3, 8), 4.))
    assert r['hold'].tolist() == [1, LAW, 0] and r['app_cost'].tolist() == [0., 0., 7.]
    assert r['u'][0, 0] == 20. and r['x1'][0].astype(float).tolist() == [3., 61.]           # u_1 of the plan
    assert r['u'][1, 0] == -0.5 and r['x1'][1].astype(float).tolist() == [3., -0.5]         # K x, then A x + B K x
    assert r['plan'][2].tolist() == [4.] * 8 and r['plan'][0].tolist() == plan2[0].tolist()


@pytest.fixture(scope='module', params=['cp20', 'cp40'])
def model_ctl(request):
    from oracle.models import load_model
    from tests.util import make_controller
    model = load_model(request.param)
    return model, make_controller(model)


def test_terminal_law_is_the_law_of_the_terminal_cost(model_ctl):
    """P of the DARE on the penalised inputs equals Q_T'Q_T, and the gain of terminal_law() is the LQR gain of that P"""
    from scipy.linalg import solve_discrete_are
    model, ctl = model_ctl
    K = ctl.terminal_law()
    A, B, Q, R, Q_T = model['A'], model['B'], model['Q'], model['R'], model['Q_T']
    inputs = np.nonzero(np.any(R != 0., axis=0))[0]
    assert inputs.tolist() == [0]
    assert K.shape == (B.shape[1], A.shape[0]) and np.all(K[1:] == 0.)
    np.testing.assert_array_equal(K, ctl.terminal_law(inputs=[0]))
    Bu, Ru = B[:, inputs], R[:, inputs]
    P_T = Q_T.T.dot(Q_T)
    P = solve_discrete_are(A, Bu, Q.T.dot(Q), Ru.T.dot(Ru))
    assert np.max(np.abs(P - P_T)) <= 1e-9 * np.max(np.abs(P_T))
    K_T = -np.linalg.solve(Bu.T.dot(P_T).dot(Bu) + Ru.T.dot(Ru), Bu.T.dot(P_T).dot(A))
    assert np.max(np.abs(K[inputs] - K_T)) <= 1e-9 * np.max(np.abs(K_T))


def test_terminal_set_is_invariant_and_admissible_under_the_law(model_ctl):
    """on points of the terminal set (random rays from the origin, up to the boundary): F_T (A + B K) x <= h_T and
    F x + G K x <= h"""
    model, ctl = model_ctl
    K = ctl.terminal_law()
    A, B, F, G, h, F_T, h_T = (model[k] for k in ('A', 'B', 'F', 'G', 'h', 'F_T', 'h_T'))
    rng = np.random.default_rng(0)
    d = rng.standard_normal((4000, A.shape[0])) * model['x_max']
    s = F_T.dot(d.T)                                       # [rows, points]
    reach = np.min(np.where(s > 0, h_T[:, None] / np.where(s > 0, s, 1.), np.inf), axis=0)
    assert np.all(np.isfinite(reach))                      # the set is bounded
    frac = np.concatenate((np.ones(1000), rng.uniform(0., 1., d.shape[0] - 1000)))
    x = d * (reach * frac)[:, None]
    assert np.all(F_T.dot(x.T) <= h_T[:, None] + 1e-9 * np.abs(h_T).max())
    x1 = x.dot((A + B.dot(K)).T)
    assert np.all(F_T.dot(x1.T) - h_T[:, None] <= 1e-9 * max(1., np.abs(h_T).max()))
    u = x.dot(K.T)
    assert np.all(F.dot(x.T) + G.dot(u.T) - h[:, None] <= 1e-9 * max(1., np.abs(h).max()))


@pytest.fixture(scope='module')
def ctl():
    from oracle.models import load_model
    from tests.util import make_controller
    return make_controller(load_model('cp20'))


@pytest.mark.parametrize('L', [-1, -5, 1.5])
def test_terminal_law_steps_range(ctl, L):
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    with pytest.raises(ValueError, match='terminal_law'):
        ClosedLoop(ctl, 4, fallback=3, terminal_law=L)


def test_closed_loop_law_value_errors(ctl):
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    nu, nx = ctl.mld.nu, ctl.mld.nx
    for K in (np.zeros((nx, nu)), np.zeros((1, nx)), np.zeros(nx), np.zeros((nu, nx, 1))):
        with pytest.raises(ValueError, match='law_gain'):
            ClosedLoop(ctl, 4, terminal_law=5, law_gain=K)
    with pytest.raises(ValueError, match='comparator'):
        ClosedLoop(ctl, 4, warm=False, comparator=True, terminal_law=5)
    # run_mailbox and rebalance refuse a loop with the law (its buffers are the fallback's) before they touch the device
    L = ClosedLoop.__new__(ClosedLoop)
    L.plant, L.fb = None, dict(max_hold=0, max_law=5)
    with pytest.raises(ValueError, match='fallback'):
        L.run_mailbox(1, lambda *a: None)
    with pytest.raises(ValueError, match='fallback plans'):
        L.rebalance()


def test_fallback_struct_without_and_with_the_law():
    import torch
    from warm_start_hmpc_b200 import capi
    N, P = 5, 224
    fb = dict(max_hold=3, plan=torch.zeros((N, P), dtype=torch.float64), age=torch.full((N,), -1, dtype=torch.int32),
              app_cost=torch.zeros(N, dtype=torch.float64), app_primal=torch.zeros((N, P), dtype=torch.float64))
    c = capi._fallback_struct(fb, None)
    assert c.max_law == 0 and c.d_law_K is None and c.d_law_n is None
    K, n = torch.zeros((3, 4), dtype=torch.float64), torch.zeros(N, dtype=torch.int32)
    c = capi._fallback_struct(dict(fb, max_law=7, law_K=K, law_n=n), None)
    assert c.max_law == 7 and c.d_law_K == K.data_ptr() and c.d_law_n == n.data_ptr()
    assert c.max_hold == 3 and c.d_plan == fb['plan'].data_ptr()
