"""-m gpu: the search variants of the C ABI on the shape grid (tests/shape_grid.py), against the host loop and the oracle.

Every variant below computes addresses and word indices from the sizes the grid varies (nx, nu, nuc, nub, T, nb and the
identifier words): depth-first and breadth-first candidate selection, static branching orders (wshmpc_set_branch_order), the
conventional MIQP comparator (node rules 1 and 2) with its MIP starts (wshmpc_tree_init_guess), the fallback and terminal-law
policy (wshmpc_fallback_step, wshmpc_closed_loop_fallback) and the mailbox.  Per shape:

1. candidate rules 1 and 2: the device search against the host loop node for node, and against the oracle's optimum;
2. static branching orders: the same, and on the loop tier K2 + K4 of non-prefix leaves against the host formulation;
3. the comparator with three MIP starts against the host feedforward_miqp, and wshmpc_tree_init_guess against a numpy packing;
4. the fused loop under rules 1 and 2 and under node rule 2 against lock step (loop tier);
5. wshmpc_fallback_step against a long-double reference, and the fused fallback loop against lock step (loop tier);
6. the mailbox loop against the device-resident loop (loop tier).

Shapes of the search tier (nub > 32, T = 1) are left out of the warm start of section 2, the loops of sections 4 and 5,
and section 6, because the tree shift and the fused loop refuse them (tests/test_gpu_shapes.py checks that refusal).
States: shape.x0(), 0.5 shape.x0() and two seeded states; a host comparison uses only states whose search fits BUDGET
relaxations, and a shape none of whose states fits fails.  Run with -s for one line per shape and variant.
"""
import contextlib
import math
import time

import numpy as np
import pytest
import torch

from oracle.bnb_ref import OracleController
from oracle.qp_c import CoreC
from tests import shape_grid as sg
from tests.util import make_controller, oracle_loop, COST_RTOL
from tests.test_gpu_fallback import _lock, _equal
from tests.test_terminal_law_cpu import LAW, fallback_reference, replay_law

pytestmark = pytest.mark.gpu

SEARCH = [s for s in sg.GRID if s.tier in (sg.K3, sg.ALL)]      # the device search runs
LOOP = [s for s in sg.GRID if s.tier == sg.ALL]                  # ... and the tree shift and the fused loop
BUDGET = 2000           # relaxations a search may take to be compared with the host loop
N_HOST = 2              # states per shape and variant compared with the host loop
MAX_LAW = 5
# (shape, candidate rule) whose cold search from the root never ends within a tree's capacity: breadth-first must finish
# every level above the last before it meets an incumbent, and nub1_T32's 32 binaries (one per step) are rarely pruned as
# infeasible.  The fused loop and lock step must still stop them alike; sections 1 and 2 give them a MIP start instead.
OVER_CAPACITY = {('nub1_T32', 2)}


def _ident_key(identifier):
    return tuple(sorted(identifier.items()))


def _is_prefix(identifier, nub):
    return all((q // nub, q % nub) in identifier for q in range(len(identifier)))


@contextlib.contextmanager
def _rules(h, search=0, order=None, node=0):
    """The handle's search rule, branching order and node rule for the duration of the block (defaults restored after)."""
    h.set_search_rule(search); h.set_branch_order(order); h.set_node_rule(node)
    try:
        yield
    finally:
        h.set_search_rule(0); h.set_branch_order(None); h.set_node_rule(0)


class Built(object):
    """A shape compiled once: model, controller, the states the searches run at and the oracle's optima there."""

    def __init__(self, shape):
        self.shape = shape
        self.model = shape.model()
        self.ctl = make_controller(self.model)
        self.pd = self.ctl.problem
        self.T, self.nx, self.nu, self.nub, self.nuc = self.pd.T, self.pd.nx, self.pd.nu, self.pd.nub, self.pd.nuc
        self.nb = self.pd.nb
        seeded = sg.nodes(shape, 3, seed=11)[0][1:]
        self.states = [shape.x0(), 0.5 * shape.x0(), seeded[0], seeded[1]]
        self._oracle = {}
        self.push = None
        self.fb_runs = {}

    def oracle(self, k):
        """(cost, rounded modes [nb]) of the oracle's best-first optimum at states[k]; (inf, None) if infeasible."""
        if k not in self._oracle:
            inc, _, _ = OracleController(self.model, CoreC(self.model, variant=1), hot_start='record').feedforward(self.states[k])
            self._oracle[k] = (np.inf, None) if inc is None else \
                (inc.primal['objective'], np.round(inc.primal['u'][:, self.nuc:]).ravel())
        return self._oracle[k]

    def check_oracle(self, k, cost, modes, tag):
        c_ref, m_ref = self.oracle(k)
        if m_ref is None:
            assert np.isinf(cost), (tag, cost)
            return
        assert abs(cost - c_ref) <= COST_RTOL * abs(c_ref), (tag, cost, c_ref)
        assert np.array_equal(np.asarray(modes).ravel(), m_ref), tag

    def instances(self, N, seed):
        rng = np.random.default_rng(seed)
        xm = np.asarray(self.model['x_max'], dtype=float)
        return self.shape.x0()[None] + 0.02 * self.shape.x0_scale * rng.uniform(-1, 1, (N, xm.size)) * xm

    def noise(self, S, N, seed, sigma=0.003):
        return sigma * np.random.default_rng(seed).standard_normal((S, N, self.nx)) * self.model['x_max']


@pytest.fixture(scope='module')
def built():
    cache = {}

    def get(shape):
        if shape.name not in cache:
            cache[shape.name] = Built(shape)
        return cache[shape.name]
    return get


# ---- 1 and 2. the device search against the host loop -------------------------------------------------------------------
def _mip_start(b, k):
    """A first cover of the search at states[k]: the oracle's optimal mode sequence, every binary pinned, then the root
    (both without a record, lb = -inf).  Breadth-first solves the pinned node first and prunes with its cost from then on;
    without it, it has to finish every level above the last before it meets an incumbent.  None where the MIQP is
    infeasible."""
    import warm_start_hmpc_b200 as ws
    _, modes = b.oracle(k)
    if modes is None:
        return None
    pinned = {(q // b.nub, q % b.nub): float(modes[q]) for q in range(b.nb)}
    return [ws.Node(pinned, -np.inf, None), ws.Node({}, -np.inf, None)]


def _probe(b, k, search, order, start):
    """(status, relaxations) of the device search at states[k] within BUDGET relaxations (status 2: it does not end
    within them, 3: a node QP stopped at the iteration limit)."""
    h = b.ctl.handle()
    tree = None if start is None else b.ctl.leaves_to_tree(start, max_solves=BUDGET)
    with _rules(h, search, order):
        res, _ = b.ctl.feedforward_batch(np.asarray(b.states[k])[None], warm_start=tree, max_solves=BUDGET, n_slots=1)
        return int(res['status'][0]), int(res['n_solves'][0])


def _against_host(b, k, search_rule, branch_rule, tag, start=None):
    """feedforward at states[k] on the device and in the host loop with the same rules (and the same first cover `start`):
    the same QP count, leaves (identifiers and bounds bit for bit) and objective bit for bit, and the oracle's optimum.
    Returns (device result, host result)."""
    ctl, x = b.ctl, b.states[k]
    copy = lambda: None if start is None else [type(n)(dict(n.identifier), n.lb, None) for n in start]
    ctl.device_search = False
    try:
        sol_h, leaves_h, n_h, _ = ctl.feedforward(x, search_rule=search_rule, branch_rule=branch_rule, warm_start=copy(),
                                                  printing_period=None)
    finally:
        ctl.device_search = True
    sol_d, leaves_d, n_d, _ = ctl.feedforward(x, search_rule=search_rule, branch_rule=branch_rule, warm_start=copy(),
                                              printing_period=None)
    assert n_d == n_h, (tag, n_d, n_h)
    assert [_ident_key(l.identifier) for l in leaves_d] == [_ident_key(l.identifier) for l in leaves_h], tag
    assert np.array_equal(np.array([l.lb for l in leaves_d]), np.array([l.lb for l in leaves_h])), tag
    assert (sol_d is None) == (sol_h is None), tag
    if sol_d is not None:
        assert sol_d.objective == sol_h.objective, (tag, sol_d.objective, sol_h.objective)
        assert np.array_equal(np.array(sol_d.variables['ub']), np.array(sol_h.variables['ub'])), tag
    b.check_oracle(k, np.inf if sol_d is None else sol_d.objective,
                   None if sol_d is None else np.round(np.array(sol_d.variables['ub'])), tag)
    return (sol_d, leaves_d, n_d), (sol_h, leaves_h, n_h)


def _compare_states(b, search_rule, branch_rule, tag):
    """_against_host at the first N_HOST states whose device search ends within BUDGET relaxations, from the root or, where
    that does not, from _mip_start; fails if no state does.  Returns (compared, passed over): compared [(state, form,
    device result, host result)], passed over [(state, form, status)] (status 2: over the budget, 3: a node QP at the
    iteration limit, which the host loop reports as an error)."""
    import warm_start_hmpc_b200 as ws
    search = {ws.best_first: 0, ws.depth_first: 1, ws.breadth_first: 2}[search_rule]
    order = None if branch_rule is ws.branch_in_time else branch_rule.permutation(b.T, b.nub)
    done, passed = [], []
    for k in range(len(b.states)):
        for form in ('root', 'MIP start'):
            start = None if form == 'root' else _mip_start(b, k)
            if form == 'MIP start' and start is None:
                break
            st, _ = _probe(b, k, search, order, start)
            if st <= 1:
                done.append((k, form) + _against_host(b, k, search_rule, branch_rule, tag + (k, form), start))
                break
            passed.append((k, form, st))
        if len(done) == N_HOST:
            break
    if not done:
        pytest.fail('%s: no state of the shape ends its search (%s) within %d relaxations: %s'
                    % (b.shape.name, tag[1:], BUDGET, passed))
    return done, passed


def _summary(done, passed):
    return 'states %s, QPs (device, host) %s, passed over (state, form, status) %s' \
        % ([(d[0], d[1]) for d in done], [(d[2][2], d[3][2]) for d in done], passed)


@pytest.mark.parametrize('rule', ['depth_first', 'breadth_first'])
@pytest.mark.parametrize('shape', SEARCH, ids=str)
def test_candidate_rules_equal_the_host_loop_and_the_oracle(built, shape, rule):
    import warm_start_hmpc_b200 as ws
    b = built(shape)
    t0 = time.time()
    done, passed = _compare_states(b, getattr(ws, rule), ws.branch_in_time, (shape.name, rule))
    print('\n%s %s: %s; %.1f s' % (shape.name, rule, _summary(done, passed), time.time() - t0))


def _orders(b):
    import warm_start_hmpc_b200 as ws
    # a seeded random order of the binaries of every step, the steps in time order: a random permutation of all nb binaries
    # leaves the structured search without the bounds of a time prefix, and on cp21 (84 binaries) no state then ends within
    # BUDGET relaxations
    rng = np.random.default_rng(5)
    shuffled = [(t, int(i)) for t in range(b.T) for i in rng.permutation(b.nub)]
    return [('reverse_time', ws.branch_in_reverse_time(b.T, b.nub)), ('by_index', ws.branch_by_index(b.T, b.nub)),
            ('random', ws.StaticBranchOrder(shuffled))]


@pytest.mark.parametrize('shape', SEARCH, ids=str)
def test_static_branch_orders_equal_the_host_loop_and_the_oracle(built, shape):
    """Three static orders at the shape's states; on the loop tier also the warm start of the non-prefix leaves (K2 + K4
    against the host formulation) and the next step warm-started under the same order against a cold best-first solve."""
    import warm_start_hmpc_b200 as ws
    b = built(shape)
    ctl = b.ctl
    non_prefix = 0
    for name, rule in _orders(b):
        t0 = time.time()
        done, passed = _compare_states(b, ws.best_first, rule, (shape.name, name))
        np_here = sum(not _is_prefix(l.identifier, b.nub) for d in done for l in d[2][1])
        non_prefix += np_here
        warm = '-'
        k, _, (sol_d, leaves_d, _), (sol_h, leaves_h, _) = done[0]
        if shape.tier == sg.ALL and sol_d is not None:
            x = b.states[k]
            e0 = 0.003 * np.random.default_rng(0).standard_normal(b.nx) * b.model['x_max']
            uc, ub = sol_d.variables['uc'][0], sol_d.variables['ub'][0]
            ws_d, _, _ = ctl.construct_warm_start(leaves_d, x, uc, ub, e0)
            ctl.device_search = False
            try:
                ws_h, _, _ = ctl.construct_warm_start(leaves_h, x, sol_h.variables['uc'][0], sol_h.variables['ub'][0], e0)
            finally:
                ctl.device_search = True
            tag = (shape.name, name, k, 'warm start')
            assert [_ident_key(l.identifier) for l in ws_d] == [_ident_key(l.identifier) for l in ws_h], tag
            lb_d, lb_h = np.array([l.lb for l in ws_d]), np.array([l.lb for l in ws_h])
            assert np.array_equal(np.isinf(lb_d), np.isinf(lb_h)), tag
            assert np.all(np.abs(lb_d[np.isfinite(lb_d)] - lb_h[np.isfinite(lb_h)]) <= 1e-11), tag
            assert [l.extra.dual is None for l in ws_d] == [l.extra.dual is None for l in ws_h], tag
            x1 = sol_d.variables['x'][1] + e0
            sol_w, _, n_w, _ = ctl.feedforward(x1, branch_rule=rule, warm_start=ws_d, printing_period=None)
            sol_c, _, n_c, _ = ctl.feedforward(x1, printing_period=None)
            assert (sol_w is None) == (sol_c is None), tag
            if sol_c is not None:
                assert abs(sol_w.objective - sol_c.objective) <= 1e-9 * abs(sol_c.objective), tag
                assert np.array_equal(np.array(sol_w.variables['ub']), np.array(sol_c.variables['ub'])), tag
            warm = '%d leaves, QPs warm %d cold %d' % (len(ws_d), n_w, n_c)
        print('\n%s %s: %s, non-prefix leaves %d; warm start: %s; %.1f s'
              % (shape.name, name, _summary(done, passed), np_here, warm, time.time() - t0))
    assert non_prefix > 0, (shape.name, 'no leaf with a non-prefix identifier')


# ---- 3. the comparator and its MIP starts -------------------------------------------------------------------------------
def _host_miqp(ctl, x0, guess):
    """The host feedforward_miqp with every solved node's identifier and cost recorded; (result or None if a node QP did
    not converge, log of (identifier, cost), identifiers asked)."""
    log, asked = [], []
    orig = ctl._solve_subproblem

    def spy(identifier, x0_, active_set=None):
        asked.append(_ident_key(identifier))
        sol, dt = orig(identifier, x0_, active_set)
        log.append((_ident_key(identifier), sol.primal.objective))
        return sol, dt
    ctl._solve_subproblem = spy
    try:
        out = ctl.feedforward_miqp(x0, ub_guess=guess)
    except RuntimeError as err:
        assert 'did not converge' in str(err)
        out = None
    finally:
        ctl._solve_subproblem = orig
    return out, log, asked


def _modes_of(b, primal_row):
    return np.round(primal_row[(b.T + 1) * b.nx:].reshape(b.T, b.nu)[:, b.nuc:])


@pytest.mark.parametrize('shape', SEARCH, ids=str)
def test_comparator_equals_the_host_loop_node_for_node(built, shape):
    """feedforward_miqp_batch (node rule 1) without a guess, with shift_binary_solution of the host optimum and with all ones,
    against the spied host loop: the solved identifiers in order, their costs bit for bit, the status and the objective;
    where the search is not stopped by the QP iteration limit its optimum is the oracle's."""
    b = built(shape)
    ctl = b.ctl
    t0 = time.time()
    rows = []
    for k, x in enumerate(b.states):
        guesses, gi = [None], 0
        while gi < len(guesses):
            guess = guesses[gi]
            tag = (shape.name, k, gi)
            res, tree = ctl.feedforward_miqp_batch(np.asarray(x)[None], ub_guess=None if guess is None else guess[None],
                                                   trace=True, n_slots=1, max_solves=BUDGET + 1)
            st, n = int(res['status'][0]), int(res['n_solves'][0])
            gi += 1
            if st == 2:                                  # over the budget: not compared with the host loop, but reported
                rows.append((k, gi - 1, n, None, 'over budget'))
                continue
            out, log, asked = _host_miqp(ctl, x, guess)
            solved = res['trace'][0].cpu().numpy().reshape(-1, 2)[:n, 0]
            bits = tree.bits[0].cpu().numpy().view(np.uint32); mask = tree.mask[0].cpu().numpy().view(np.uint32)
            ids = [_ident_key(ctl._identifier(bits[j], mask[j])) for j in solved]
            lb = tree.lb[0].cpu().numpy()[solved]
            if st == 3:
                # the host loop asks for the same nodes, gets the same costs and stops on the node the device stopped on
                assert out is None and len(asked) == n + 1 and ids == asked[:n], tag
                assert np.array_equal(lb, np.array([c for _, c in log])), tag
                rows.append((k, gi - 1, n, len(asked) - 1, 'limit'))
                continue
            var_h, obj_h, nodes_h, _ = out
            assert st == (0 if var_h is not None else 1), (tag, st)
            assert n == nodes_h == len(log), (tag, n, nodes_h)
            assert ids == [i for i, _ in log], tag
            assert np.array_equal(lb, np.array([c for _, c in log])), tag
            assert float(res['cost'][0]) == obj_h, (tag, float(res['cost'][0]), obj_h)
            b.check_oracle(k, float(res['cost'][0]), _modes_of(b, res['primal'][0].cpu().numpy()), tag)
            rows.append((k, gi - 1, n, nodes_h, st))
            if guess is None and var_h is not None:      # the closed loop's MIP start, and a guess that is usually infeasible
                guesses += [ctl.shift_binary_solution(var_h['ub']), np.ones((b.T, b.nub))]
        if len({r[0] for r in rows if r[3] is not None}) == N_HOST:
            break
    if not any(r[3] is not None for r in rows):
        pytest.fail('%s: no state of the shape ends its comparator search within %d relaxations' % (shape.name, BUDGET))
    print('\n%s comparator: (state, guess, QPs device, QPs host, status) %s; %.1f s' % (shape.name, rows, time.time() - t0))


def _pack(v, words):
    out = np.zeros(words, np.uint32)
    for q in np.nonzero(v)[0]:
        out[q >> 5] |= np.uint32(1 << (int(q) & 31))
    return out


@pytest.mark.parametrize('shape', SEARCH, ids=str)
def test_tree_init_guess_packs_every_word(built, shape):
    """wshmpc_tree_init_guess on guesses of 0 / 1 with non-integral and negative entries (rounded with rint, like numpy's
    round half to even) over trees filled with garbage: node 0 pins every binary, the last word only its nb % 32 low bits."""
    b = built(shape)
    h = b.ctl.handle()
    N, nb = 6, b.nb
    rng = np.random.default_rng(9)
    g = rng.integers(0, 2, (N, nb)).astype(float)
    odd = np.array([0.3, 0.5, 0.7, 1.5, 2.5, -0.2, -0.5, -0.7, -1., 0.49999999, 1e-300, -0.])
    for i in range(N):
        pos = rng.choice(nb, size=min(nb, 4), replace=False)
        g[i, pos] = rng.choice(odd, size=pos.size)
    g[1] = 1.                                            # every bit, the partial last word included
    has = np.array([1, 1, 0, 1, 1, 0], np.int32)
    tree = h.new_tree(N, 4, 2)
    for t in (tree.bits, tree.mask, tree.depth, tree.rec, tree.alive, tree.n_nodes, tree.n_recs):
        t.fill_(-1)
    tree.lb.fill_(7.)
    h.tree_init_guess(tree, torch.as_tensor(g, device='cuda').contiguous(), torch.as_tensor(has, device='cuda'))
    torch.cuda.synchronize()
    W = tree.words
    assert W == (nb + 31) // 32
    bits, mask = tree.bits.cpu().numpy().view(np.uint32), tree.mask.cpu().numpy().view(np.uint32)
    full = _pack(np.ones(nb, bool), W)
    for i in range(N):
        tag = (shape.name, i)
        if has[i]:
            assert int(tree.n_nodes[i]) == 2 and int(tree.n_recs[i]) == 0, tag
            assert np.array_equal(bits[i, 0], _pack(np.rint(g[i]) != 0., W)), (tag, bits[i, 0], g[i])
            assert np.array_equal(mask[i, 0], full), tag
            assert tree.depth[i, :2].tolist() == [nb, 0] and tree.rec[i, :2].tolist() == [-1, -1], tag
            assert tree.alive[i, :2].tolist() == [1, 1] and np.all(np.isneginf(tree.lb[i, :2].cpu().numpy())), tag
            root = 1
        else:
            assert int(tree.n_nodes[i]) == 1 and int(tree.n_recs[i]) == 0, tag
            root = 0
        assert not bits[i, root].any() and not mask[i, root].any(), tag
        assert int(tree.depth[i, root]) == 0 and int(tree.rec[i, root]) == -1, tag
    assert bin(int(full[-1])).count('1') == (nb % 32 or 32)


# ---- 4. fused loops of the variants against lock step -------------------------------------------------------------------
def _trees_equal(A, B, N, tag):
    ta, tb = A.trees[A.cur], B.trees[B.cur]
    assert torch.equal(ta.n_nodes, tb.n_nodes), tag
    for i in range(N):
        n = int(ta.n_nodes[i])
        for k in ('lb', 'bits', 'mask', 'depth', 'rec', 'alive'):
            assert torch.equal(getattr(ta, k)[i, :n], getattr(tb, k)[i, :n]), (tag, i, k)


@pytest.mark.parametrize('warm', [True, False], ids=['warm', 'cold'])
@pytest.mark.parametrize('rule', [1, 2], ids=['depth_first', 'breadth_first'])
@pytest.mark.parametrize('shape', LOOP, ids=str)
def test_fused_loop_under_other_candidate_rules_equals_lock_step(built, shape, rule, warm):
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    b = built(shape)
    t0 = time.time()
    N, S = 8, 4
    x0 = b.instances(N, 5)
    e_np = b.noise(S, N, 6)
    e = torch.as_tensor(e_np, device='cuda')
    A = ClosedLoop(b.ctl, N, warm=warm, max_solves=4096, max_roots=2048)
    B = ClosedLoop(b.ctl, N, warm=warm, max_solves=4096, max_roots=2048)
    assert A.h is B.h
    A.reset(x0); B.reset(x0)
    with _rules(A.h, search=rule):
        lock = {k: [] for k in ('cost', 'n_solves', 'status', 'u0')}
        for t in range(S):
            out = A.step(e=e[t])
            for k in ('cost', 'n_solves', 'status'):
                lock[k].append(out[k].clone())
            lock['u0'].append(A.u0.clone())
        logs = B.run(S, e=e)
        torch.cuda.synchronize()
    tag = (shape.name, rule, warm)
    lock = {k: torch.stack(v) for k, v in lock.items()}
    for k in ('cost', 'n_solves', 'status'):
        assert torch.equal(lock[k], logs[k]), (tag, k)
    assert torch.equal(torch.nan_to_num(lock['u0'], nan=-7.), torch.nan_to_num(logs['u0'], nan=-7.)), tag
    assert torch.equal(A.x, B.x) and torch.equal(A.active, B.active), tag
    if warm:
        _trees_equal(A, B, N, tag)
    st, cost = logs['status'].cpu().numpy(), logs['cost'].cpu().numpy()
    if (shape.name, rule) in OVER_CAPACITY:
        assert np.all(st[0] == 2) and not A.active.any(), (tag, st)
        print('\n%s rule %d: every cold search stops at capacity, alike in both loops' % (shape.name, rule))
        return
    assert np.all(st <= 1), (tag, st)
    for i in range(2):
        ref = oracle_loop(b.model, x0[i], e_np[:, i])
        for t, r in enumerate(ref):
            assert not r.get('failed'), (tag, i, t, 'the oracle failed')
            if np.isfinite(r['cost']):
                assert abs(cost[t, i] - r['cost']) <= COST_RTOL * abs(r['cost']), (tag, i, t, cost[t, i], r['cost'])
            else:
                assert np.isinf(cost[t, i]), (tag, i, t)
    print('\n%s rule %d %s: QPs per step %s; %.1f s' % (shape.name, rule, 'warm' if warm else 'cold',
                                                      logs['n_solves'].sum(1).tolist(), time.time() - t0))


@pytest.mark.parametrize('shape', LOOP, ids=str)
def test_fused_comparator_with_mip_starts_equals_lock_step(built, shape):
    """Node rule 2: the fused loop's MIP start (u_1's binaries of the previous incumbent, shifted by one step) against lock
    step driven by the host's shift_binary_solution of that incumbent."""
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    b = built(shape)
    ctl = b.ctl
    t0 = time.time()
    N, S, ms = 8, 4, 4096
    x0 = b.instances(N, 7)
    e = torch.as_tensor(b.noise(S, N, 8), device='cuda')
    F = ClosedLoop(ctl, N, warm=False, comparator=True, mip_start=True, max_solves=ms)
    F.reset(x0)
    logs = F.run(S, e=e)
    h = F.h
    dev = h.torch_device
    trees = [h.new_tree(N, 2 + 2 * ms + 2, 2 + ms + 1) for _ in range(2)]       # the capacities of ClosedLoop's trees
    x = torch.as_tensor(x0, device=dev).contiguous()
    xn = torch.empty_like(x)
    active = torch.ones(N, dtype=torch.int32, device=dev)
    u0 = torch.empty((N, b.nu), dtype=torch.float64, device=dev)
    lock = {k: [] for k in ('cost', 'n_solves', 'status', 'u0')}
    out, n_starts = None, 0
    for t in range(S):
        tree = trees[t & 1]
        if out is None:
            h.tree_init_root(tree)
        else:
            prim, c = out['primal'].cpu().numpy(), out['cost'].cpu().numpy()
            guess = np.stack([ctl.shift_binary_solution(_modes_of(b, prim[i])) for i in range(N)]).reshape(N, b.nb)
            has = ((active.cpu().numpy() != 0) & np.isfinite(c)).astype(np.int32)
            n_starts += int(has.sum())
            h.tree_init_guess(tree, torch.as_tensor(guess, device=dev).contiguous(), torch.as_tensor(has, device=dev))
        with _rules(h, node=1):
            out = h.bnb_solve(x, tree, max_solves=ms, active=active)
        h.shift_tree(x, e[t], tree, out['cost'], out['primal'], trees[1 - (t & 1)], active=active, x_next=xn, u0=u0)
        for k in ('cost', 'n_solves', 'status'):
            lock[k].append(out[k].clone())
        lock['u0'].append(u0.clone())
        x, xn = xn, x
    torch.cuda.synchronize()
    lock = {k: torch.stack(v) for k, v in lock.items()}
    for k in ('cost', 'n_solves', 'status'):
        assert torch.equal(lock[k], logs[k]), (shape.name, k)
    assert torch.equal(torch.nan_to_num(lock['u0'], nan=-7.), torch.nan_to_num(logs['u0'], nan=-7.)), shape.name
    assert torch.equal(F.x, x) and torch.equal(F.active, active), shape.name
    assert n_starts > 0, shape.name
    print('\n%s comparator loop: MIP starts %d, QPs per step %s, statuses %s; %.1f s'
          % (shape.name, n_starts, logs['n_solves'].sum(1).tolist(), np.unique(logs['status'].cpu().numpy()).tolist(),
             time.time() - t0))


# ---- 5. the fallback and terminal-law policy ----------------------------------------------------------------------------
@pytest.mark.parametrize('shape', SEARCH, ids=str)
def test_fallback_step_equals_the_long_double_reference(built, shape):
    """wshmpc_fallback_step with H = T - 1 and L = 2 over statuses 0..3, finite and infinite incumbent costs, every age from
    -1 to T - 1, law counts 0..L and switched-off instances, against tests/test_terminal_law_cpu.fallback_reference."""
    b = built(shape)
    ctl = b.ctl
    T, nx, nu, H, L = b.T, b.nx, b.nu, b.T - 1, 2
    h = ctl.handle()
    P, U = h.layout.primal, (T + 1) * nx
    grid = [(lv, hi, st, a, n) for lv in (0, 1) for hi in (0, 1) for st in (0, 1, 2, 3) for a in range(-1, T)
            for n in (0, L - 1, L) if not (hi and st == 1)]
    N = len(grid)
    lv, hi, st, age, law_n = (np.array(c) for c in zip(*grid))
    rng = np.random.default_rng(1)
    dev = lambda a, dt=torch.float64: torch.as_tensor(a, dtype=dt, device='cuda').contiguous()
    x = rng.standard_normal((N, nx)) * b.model['x_max']
    plan = rng.standard_normal((N, P)); inc = rng.standard_normal((N, P))
    cost = np.where(hi == 1, rng.uniform(1., 2., N), np.inf)
    K = ctl.terminal_law()
    fb = h.new_fallback(N, H, L, K)
    fb['plan'].copy_(dev(plan)); fb['age'].copy_(dev(age, torch.int32)); fb['law_n'].copy_(dev(law_n, torch.int32))
    fb['app_primal'].fill_(np.nan); fb['app_cost'].fill_(-1.)
    h.fallback_step(fb, dev(x), dev(lv, torch.int32), dict(status=dev(st, torch.int32), cost=dev(cost), primal=dev(inc)))
    torch.cuda.synchronize()
    ref = fallback_reference(b.model['A'], b.model['B'], K, T, H, L, lv, st, cost, age, law_n, x, plan, inc)
    src = ref['source']
    assert {0, 2, -1} | ({1} if H > 0 else set()) <= set(src.tolist()), shape.name        # T = 1: H = 0, no plan steps
    for k in ('hold', 'age', 'law_n'):
        assert np.array_equal(fb[k].cpu().numpy(), ref[k]), (shape.name, k)
    assert np.array_equal(fb['app_cost'].cpu().numpy(), ref['app_cost']), shape.name
    assert np.array_equal(fb['plan'].cpu().numpy(), ref['plan']), shape.name
    ap = fb['app_primal'].cpu().numpy()
    eps = np.finfo(float).eps
    tol = 4 * (nx + nu) * eps
    for i in range(N):
        tag = (shape.name, grid[i])
        if src[i] == 0:
            assert np.array_equal(ap[i], inc[i]), tag
        elif src[i] < 0:
            assert np.isnan(ap[i]).all(), tag                               # the record of an instance that leaves is not written
        else:
            assert np.array_equal(ap[i, :nx], x[i]), tag
            u = ap[i, U:U + nu]
            if src[i] == 1:
                assert np.array_equal(u, plan[i, U + ref['hold'][i] * nu:U + (ref['hold'][i] + 1) * nu]), tag
            else:
                assert np.all(np.abs(u - ref['u'][i]) <= tol * ref['u_terms'][i]), (tag, u, ref['u'][i])
            assert np.all(np.abs(ap[i, nx:2 * nx] - ref['x1'][i]) <= tol * ref['x1_terms'][i]), (tag, ap[i, nx:2 * nx], ref['x1'][i])
    print('\n%s fallback step: %d instance-steps, sources %s' % (shape.name, N, np.unique(src, return_counts=True)))


def _push(b):
    """(direction, scale) of a model error at step 0 that makes the MIQP at step 1 infeasible: a seeded direction scaled by
    x_max, grown geometrically from the state x_1|0 of the first step until the device search reports an infeasible MIQP
    there and the oracle loop agrees."""
    if b.push is not None:
        return b.push
    ctl, x0 = b.ctl, b.shape.x0()
    d = np.random.default_rng(13).standard_normal(b.nx) * b.model['x_max']
    res, _ = ctl.feedforward_batch(x0[None], n_slots=1)
    assert int(res['status'][0]) == 0, b.shape.name
    x1 = res['primal'][0, b.nx:2 * b.nx].cpu().numpy()
    scales = 0.02 * 1.5 ** np.arange(20)
    r, _ = ctl.feedforward_batch(x1[None] + scales[:, None] * d[None], n_slots=1)
    st = r['status'].cpu().numpy()
    for s in scales[st == 1]:
        ref = oracle_loop(b.model, x0, np.array([s * d, np.zeros(b.nx)]))
        if len(ref) == 2 and np.isinf(ref[1].get('cost', 0.)):
            b.push = (d, float(s))
            return b.push
    pytest.fail('%s: no model error along the seeded direction makes the next MIQP infeasible (statuses %s)'
                % (b.shape.name, st.tolist()))


def _fallback_runs(b, H, warm):
    """The fused fallback loop and lock step (wshmpc_fallback_step between wshmpc_bnb_solve and wshmpc_shift_tree) over 6
    steps of 8 instances: instance 0 without the push, 1..5 pushed by 1, 1, 1.5, 2 and 3 times the scale of _push at step 0,
    6 and 7 starting pushed (no plan yet: the law first).  Compares them bit for bit; returns the hold log."""
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    key = (H, warm)
    if key in b.fb_runs:
        return b.fb_runs[key]
    N, S = 8, 6
    d, s = _push(b)
    x0 = b.instances(N, 3)
    x0[6:] += np.array([2., 3.])[:, None] * s * d[None]
    e_np = b.noise(S, N, 4)
    e_np[0, 1:6] += np.array([1., 1., 1.5, 2., 3.])[:, None] * s * d[None]
    e = torch.as_tensor(e_np, device='cuda')
    mk = lambda: ClosedLoop(b.ctl, N, warm=warm, max_solves=4096, max_roots=2048, fallback=H, terminal_law=MAX_LAW)
    F, D = mk(), mk()
    F.reset(x0); D.reset(x0)
    fused = F.run(S, e=e)
    lock = _lock(D, S, e)
    torch.cuda.synchronize()
    tag = (b.shape.name, H, warm)
    _equal(fused, lock)
    assert torch.equal(F.x, D.x) and torch.equal(F.active, D.active), tag
    for k in ('age', 'law_n', 'plan'):
        assert torch.equal(F.fb[k], D.fb[k]), (tag, k)
    if warm:
        _trees_equal(F, D, N, tag)
    hold = lock['hold'].cpu().numpy()
    assert np.array_equal(hold, replay_law(lock['status'].cpu().numpy(), lock['cost'].cpu().numpy(), H, MAX_LAW)), tag
    b.fb_runs[key] = hold
    return hold


def _fallback_cases(shape):
    T = sg.dims(shape.model())['T']
    return [(shape, H, warm) for H in sorted({1, T - 1}) for warm in (True, False)]


@pytest.mark.parametrize('shape,H,warm', [c for s in LOOP for c in _fallback_cases(s)],
                         ids=lambda v: v.name if isinstance(v, sg.Shape) else str(v))
def test_fused_fallback_loop_equals_lock_step(built, shape, H, warm):
    b = built(shape)
    t0 = time.time()
    hold = _fallback_runs(b, H, warm)
    print('\n%s fallback H %d %s: hold steps %d, law steps %d, off at the end %d; %.1f s'
          % (shape.name, H, 'warm' if warm else 'cold', int((hold > 0).sum()), int((hold == LAW).sum()),
             int((hold[-1] == -1).sum()), time.time() - t0))


def test_fallback_loops_hold_and_apply_the_law_on_most_shapes(built):
    """The pushed batches of test_fused_fallback_loop_equals_lock_step reach plan steps and law steps on at least two thirds
    of the loop-tier shapes; the shapes where they do not are named."""
    both, neither, one = [], [], []
    for shape in LOOP:
        b = built(shape)
        holds = [_fallback_runs(b, H, warm) for _, H, warm in _fallback_cases(shape)]
        has_hold = any((h > 0).any() for h in holds)
        has_law = any((h == LAW).any() for h in holds)
        (both if has_hold and has_law else one if has_hold or has_law else neither).append(shape.name)
    print('\nfallback: hold and law steps on %s; only one of them on %s; neither on %s' % (both, one, neither))
    assert len(both) >= math.ceil(2 * len(LOOP) / 3), ('hold and law steps on too few shapes', both, one, neither)


# ---- 6. mailbox ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('shape', LOOP, ids=str)
def test_mailbox_loop_equals_the_device_resident_loop(built, shape):
    """The host answers every step with x_1|t + e_t and e_t (the nx-strided copies in and out of the mailbox, the nu-strided
    input): two launches in a row equal wshmpc_closed_loop without a mailbox bit for bit, trees included."""
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    b = built(shape)
    t0 = time.time()
    N, S = 8, 3
    x0 = b.instances(N, 9)
    e = b.noise(2 * S, N, 10).reshape(2, S, N, b.nx)
    ref = ClosedLoop(b.ctl, N, warm=True, max_solves=4096, max_roots=2048)
    mbx = ClosedLoop(b.ctl, N, warm=True, max_solves=4096, max_roots=2048)
    ref.reset(x0); mbx.reset(x0)
    for w in range(2):
        lr = ref.run(S, e=torch.as_tensor(e[w], device='cuda'))
        torch.cuda.synchronize()

        def plant(idx, step, u0, x1, w=w):
            return x1 + e[w][step, idx], e[w][step, idx]
        lm = mbx.run_mailbox(S, plant, timeout_s=60.)
        torch.cuda.synchronize()
        tag = (shape.name, w)
        for k in ('cost', 'n_solves', 'status'):
            assert torch.equal(lr[k], lm[k]), (tag, k)
        assert torch.equal(torch.nan_to_num(lr['u0'], nan=-7.), torch.nan_to_num(lm['u0'], nan=-7.)), tag
        assert torch.equal(ref.x, mbx.x) and torch.equal(ref.active, mbx.active), tag
        live = np.isfinite(lm['host']['cost'])
        assert np.array_equal(lm['host']['u0'][live], lm['u0'].cpu().numpy()[live]), tag
        _trees_equal(ref, mbx, N, tag)
    assert bool(torch.isfinite(lr['cost']).any()), shape.name
    print('\n%s mailbox: %.1f s' % (shape.name, time.time() - t0))
