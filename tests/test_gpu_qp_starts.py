"""-m gpu: K1 (qp_device.cuh qp_solve, through wshmpc_solve_nodes) from every start it accepts.

"Any multipliers >= 0 are dual feasible for every node" (include/wshmpc.h d_hot): whatever a solve starts from -- another
node's multipliers and centre, a Farkas ray, a scaled, sparse, dense or wide start, the working set the slot's previous
node ended with -- it must reach the optimum of the cold solve (hot = 0), or report the iteration limit (status 9).  It
never returns a wrong answer.  The cold solve of every node is checked against the CPU oracle and the certificates first
and is the reference of every other solve of that node.  Primal vectors are not compared across starts: the node QP's
Hessian is only semidefinite, so its optimum need not be unique.
"""
import os

import numpy as np
import pytest
import torch

from oracle.models import load_model, GOLDEN
from oracle.qp_c import CoreC
from oracle.condense import Condensed
from tests.util import (make_controller, random_nodes, check_node_result, prefix_depth, record_to_y0, sparse_start,
                        dense_start, wide_start, out_of_contract)

pytestmark = pytest.mark.gpu

KEYS = ('status', 'cost', 'dobj', 'iters', 'primal', 'dual', 'yc')
# A start from the node's own optimal multipliers and centre rebuilds the optimal working set and needs a few iterations
# at most; from its own Farkas ray an infeasible node rediscovers the ray.  Neither depends on the path of the cold
# solve, but both depend on the multipliers being loaded at the scale the records are written in.  Largest counts over
# the node sets, measured on a B200: (feasible nodes, infeasible nodes).
OWN_ITERS = dict(cp20=(8, 131), cp40=None, syn30=(1, 76))


def _handle(pd, n_slots):
    from warm_start_hmpc_b200.capi import Handle
    return Handle(pd, n_slots=n_slots)


def _cp20_nodes(model):
    """~100 nodes: random prefixes, pins behind a gap, the all-pinned golden leaves, prefixes of every depth 0..nb."""
    nb = int(model['T']) * int(model['nub'])
    x0a, lba, uba = random_nodes(model, 40, seed=21)
    # pins behind a gap: only the leading run of pinned binaries is eliminated, the others are two-sided rows lb == ub
    x0b, lbb, ubb = random_nodes(model, 24, seed=5)
    rng = np.random.default_rng(7)
    for k in range(22):
        d = int(np.argmax(lbb[k] != ubb[k])) if np.any(lbb[k] != ubb[k]) else nb
        for j in rng.choice(np.arange(min(d + 2, nb - 1), nb), size=3, replace=False):
            lbb[k, j] = ubb[k, j] = 0.
    g = np.load(os.path.join(GOLDEN, 'cp20_nodes.npz'))
    x0b[22] = g['x0']; lbb[22] = ubb[22] = g['opt_ub'].reshape(-1)
    x0b[23] = g['x0']; lbb[23] = ubb[23] = 0.
    # every depth: prefixes of the golden optimum at the golden state (mostly feasible) and random prefixes at random states
    rng = np.random.default_rng(8)
    depths = np.linspace(0, nb, 18).astype(int)
    x0c, lbc, ubc = random_nodes(model, 2 * depths.size, seed=9)
    lbc[:] = 0.; ubc[:] = 1.
    opt = g['opt_ub'].reshape(-1)
    for k, d in enumerate(depths):
        x0c[2 * k] = g['x0']
        lbc[2 * k, :d] = ubc[2 * k, :d] = opt[:d]
        lbc[2 * k + 1, :d] = ubc[2 * k + 1, :d] = (rng.random(d) < 0.2).astype(float)
    return np.concatenate((x0a, x0b, x0c)), np.concatenate((lba, lbb, lbc)), np.concatenate((uba, ubb, ubc))


def _cp40_nodes(model):
    nb = int(model['T']) * int(model['nub'])
    x0, lb, ub = random_nodes(model, 12, seed=2)           # the shallowest prefix has depth 8
    for k, d in zip((9, 10, 11), (nb // 2, 3 * nb // 4, nb)):
        lb[k, :d] = ub[k, :d] = 0.
    return x0, lb, ub


def _syn30_nodes(model):
    g = np.load(os.path.join(GOLDEN, 'syn30_nodes.npz'))
    pick = np.arange(0, len(g['status']), 3)[:8]
    x0r, lbr, ubr = random_nodes(model, 4, seed=4)
    lbr[0] = 0.; ubr[0] = 1.
    x0 = np.concatenate((np.repeat(g['x0'][None], pick.size, 0), x0r))
    return x0, np.concatenate((g['lb'][pick], lbr)), np.concatenate((g['ub'][pick], ubr))


NODES = dict(cp20=_cp20_nodes, cp40=_cp40_nodes, syn30=_syn30_nodes)
WIDE_RANK = dict(cp20=100, cp40=100, syn30=257)      # syn30: beyond the removal sweep's 256 rows


class NodeSet(object):
    """A model, its nodes, a handle with one slot per node, and the cold answer of every node (checked here)."""

    def __init__(self, name):
        self.name = name
        self.model = load_model(name)
        self.ctl = make_controller(self.model)
        self.pd = self.ctl.problem
        self.cond = Condensed(self.model)
        self.x0, self.lb, self.ub = NODES[name](self.model)
        self.N = len(self.x0)
        self.d = np.array([prefix_depth(self.lb[i], self.ub[i], self.pd.n_elim) for i in range(self.N)])
        self.h = _handle(self.pd, self.N)
        self.layout = self.h.layout
        self.cold = self.solve()
        oracle = CoreC(self.model)
        for i in range(self.N):
            ref = oracle.solve(self.x0[i], self.lb[i], self.ub[i])
            assert self.cold['status'][i] == ref['status'], (name, i, self.cold['status'][i], ref['status'])
            self.check(self.cold, i, i, cost_ref=ref.get('cost'), tag=(name, 'cold', i))
        self.y_own = record_to_y0(self.cold['dual'], self.layout)
        self.yc_own = self.cold['yc']
        self.feas = np.nonzero(self.cold['status'] == 2)[0]
        self.infeas = np.nonzero(self.cold['status'] == 3)[0]

    def solve(self, idx=None, h=None, **kw):
        idx = np.arange(self.N) if idx is None else np.asarray(idx)
        out = (h or self.h).solve_nodes(self.x0[idx], self.lb[idx], self.ub[idx], **kw)
        return {k: v.cpu().numpy() for k, v in out.items()}

    def check(self, out, j, i, cost_ref=None, tag=None):
        """Certificates of result j of `out`, a solve of node i."""
        check_node_result(self.model, self.cond, self.pd, self.layout, self.x0[i], self.lb[i], self.ub[i], out['status'][j],
                          out['cost'][j], out['dobj'][j], out['primal'][j], out['dual'][j], cost_ref=cost_ref, tag=tag)

    def agree(self, out, idx, what, limit_ok=False):
        """Result j of `out` solved node idx[j]: same status as the cold solve, the cold cost, the certificates.  limit_ok:
        status 9 with cost +inf is accepted too (a budget that bites)."""
        for j, i in enumerate(idx):
            st = out['status'][j]
            if limit_ok and st == 9:
                assert out['cost'][j] == np.inf, (self.name, what, i, out['cost'][j])
                continue
            assert st == self.cold['status'][i], (self.name, what, i, st, self.cold['status'][i], out['iters'][j])
            self.check(out, j, i, cost_ref=self.cold['cost'][i] if st == 2 else None, tag=(self.name, what, i))

    def hot2(self, idx, y0, yc0=None, h=None, slot=None):
        idx = np.asarray(idx)
        return self.solve(idx, h=h, hot=np.full(idx.size, 2, np.int32), y0=y0, yc0=yc0, slot=slot)

    def starts(self, seed=0):
        """name -> (node indices, y0, yc0) of every hot = 2 start family."""
        rng = np.random.default_rng(seed)
        N, idx = self.N, np.arange(self.N)
        pd = self.pd
        S = {'own': (idx, self.y_own, self.yc_own),
             'scaled 1e-6': (idx, self.y_own * 1e-6, self.yc_own),
             'scaled 1e6': (idx, self.y_own * 1e6, self.yc_own)}

        def stranger(pick):
            ii, pp = [], []
            for i in range(N):
                c = np.nonzero(pick(i))[0]
                if c.size:
                    ii.append(i); pp.append(rng.choice(c))
            ii, pp = np.array(ii), np.array(pp)
            return ii, self.y_own[pp], self.yc_own[pp]
        S['stranger x0'] = stranger(lambda i: np.any(self.x0 != self.x0[i], axis=1))
        S['stranger deeper'] = stranger(lambda i: self.d > self.d[i])
        S['stranger shallower'] = stranger(lambda i: self.d < self.d[i])
        S['farkas'] = stranger(lambda i: self.cold['status'] != self.cold['status'][i])
        S['sparse'] = (idx, np.array([sparse_start(rng, pd, int(rng.integers(1, 21))) for _ in idx]), None)
        shallow = np.nonzero(self.d <= max(4, self.d.min()))[0]
        S['wide'] = (shallow, np.array([wide_start(rng, pd, self.d[i], WIDE_RANK[self.name])[0] for i in shallow]), None)
        S['dense'] = (idx, np.array([dense_start(rng, pd) for _ in idx]), None)
        S['centre none'] = (idx, self.y_own, None)
        S['centre other'] = (idx, self.y_own, self.yc_own[(idx + 1) % N])
        scale = np.sqrt(np.mean(self.yc_own[self.feas] ** 2))
        S['centre random'] = (idx, self.y_own, rng.standard_normal((N, pd.n)) * scale)
        return S


_SETS = {}


def node_set(name):
    if name not in _SETS:
        _SETS[name] = NodeSet(name)
    return _SETS[name]


def _bits(out, j=None):
    """Outputs as raw bytes (NaN-safe bitwise comparison)."""
    return tuple(np.ascontiguousarray(out[k] if j is None else out[k][j]).tobytes() for k in KEYS)


@pytest.mark.parametrize('name', ['cp20', 'cp40', 'syn30'])
def test_node_set_covers_the_edges(name):
    S = node_set(name)
    assert S.infeas.size > 0 and S.feas.size > 0
    if name == 'cp20':
        assert S.N >= 96 and S.d.min() == 0 and S.d.max() == S.pd.nb
        assert S.infeas.size >= 10 and S.feas.size >= 10


@pytest.mark.parametrize('name', ['cp20', 'cp40', 'syn30'])
def test_hot2_starts_agree_with_the_cold_answer(name):
    S = node_set(name)
    starts = S.starts()
    for what, (idx, y0, yc0) in starts.items():
        assert idx.size > 0, what
        out = S.hot2(idx, y0, yc0)
        S.agree(out, idx, what)
        if what == 'own':
            own = out
    # the node's own optimum: one iteration per proximal pass (a start loaded with the wrong scaling takes more)
    feas = S.cold['status'] == 2
    it_f, it_i = own['iters'][feas].max(), own['iters'][~feas].max()
    print('%s own start: max iters %d (feasible), %d (infeasible)' % (name, it_f, it_i))
    if OWN_ITERS[name] is not None:
        assert it_f <= OWN_ITERS[name][0] and it_i <= OWN_ITERS[name][1], (name, it_f, it_i)
    # the deeper strangers really carry multipliers on rows this node eliminates, the wide ones overflow the pool
    idx, y0, _ = starts['stranger deeper']
    assert any(np.any(y0[j, S.pd.mc:S.pd.mc + S.d[i]] != 0.) for j, i in enumerate(idx))
    idx, y0, _ = starts['wide']
    assert all(np.linalg.matrix_rank(S.pd.Mh[y0[j] != 0.][:, S.d[i]:]) >= WIDE_RANK[name] for j, i in enumerate(idx))


@pytest.mark.parametrize('name', ['cp20', 'syn30'])
def test_out_of_contract_entries_are_ignored_bit_for_bit(name):
    """Negative multipliers on stage rows (which have no lower side), NaN and +-inf in a start: ignored, i.e. the solve is
    bit-identical to the same start without them."""
    S = node_set(name)
    rng = np.random.default_rng(5)
    starts = S.starts(seed=1)
    for what in ('own', 'sparse', 'dense', 'stranger x0'):
        idx, y0, yc0 = starts[what]
        bad = np.array([out_of_contract(rng, y, S.pd.mc) for y in y0]) if what != 'dense' else y0.copy()
        if what == 'dense':
            # a dense start is non-zero everywhere: flip some stage rows negative and poison others; the start that
            # ignores them is the dense start with those entries zeroed
            for j in range(len(bad)):
                r = rng.choice(S.pd.mc, size=12, replace=False)
                bad[j, r[:3]] *= -1.; bad[j, r[3:6]] = np.nan; bad[j, r[6:9]] = np.inf; bad[j, r[9:]] = -np.inf
            y0 = np.where(~np.isfinite(bad) | ((np.arange(S.pd.m) < S.pd.mc) & ~(bad > 0.)), 0., bad)
        good = S.hot2(idx, y0, yc0)
        out = S.hot2(idx, bad, yc0)
        S.agree(good, idx, what)
        for j, i in enumerate(idx):
            assert _bits(out, j) == _bits(good, j), (name, what, i, out['status'][j], good['status'][j], out['iters'][j],
                                                     good['iters'][j], out['cost'][j], good['cost'][j])


@pytest.mark.parametrize('name', ['cp20', 'cp40', 'syn30'])
def test_hot1_chains_agree_with_the_cold_answer(name):
    """Every node of the set on ONE slot, in a shuffled order, each starting from the working set and centre the previous
    node ended with: as one launch, and as two launches (the first node of the second inherits the first's final state)."""
    S = node_set(name)
    perm = np.random.default_rng(3).permutation(S.N)
    h = _handle(S.pd, 1)
    zero = np.zeros(S.N, np.int32)
    one = S.solve(perm, h=h, slot=zero, hot=np.ones(S.N, np.int32))
    S.agree(one, perm, 'hot1 chain')
    half = S.N // 2
    a = S.solve(perm[:half], h=h, slot=zero[:half], hot=np.r_[0, np.ones(half - 1, np.int32)])
    b = S.solve(perm[half:], h=h, slot=zero[half:], hot=np.ones(S.N - half, np.int32))
    S.agree(a, perm[:half], 'hot1 launch A'); S.agree(b, perm[half:], 'hot1 launch B')
    # the chain restarted from the empty slot state equals the one-launch chain started the same way, bit for bit
    full = S.solve(perm, h=h, slot=zero, hot=np.r_[0, np.ones(S.N - 1, np.int32)])
    for j in range(S.N):
        ab = a if j < half else b
        assert _bits(full, j) == _bits(ab, j if j < half else j - half), (name, j, perm[j])
    h.close()


def test_hot1_after_the_device_search_on_the_same_handle():
    """After bnb_solve the slots hold the sibling memo's rows (and whatever centre the search left): a hot = 1 solve on
    each slot starts from them and must reach the cold answer."""
    S = node_set('cp20')
    n_slots = 8
    h = _handle(S.pd, n_slots)
    tree = h.new_tree(n_slots, 4096, 4096)
    h.tree_init_root(tree)
    xs = torch.as_tensor(S.x0[S.feas[:n_slots]], device='cuda').contiguous()
    res = h.bnb_solve(xs, tree, max_solves=512)
    torch.cuda.synchronize()
    assert int(res['n_solves'].max()) > 2
    idx = np.arange(S.N)
    out = S.solve(idx, h=h, slot=idx % n_slots, hot=np.ones(S.N, np.int32))
    S.agree(out, idx, 'hot1 after bnb')
    h.close()


def test_fresh_slots_start_empty():
    """A slot that never stored a state starts from the empty working set and centre 0, whatever its memory held
    before: hot = 1 as the first launch of a handle is bit-identical to hot = 0.  The new handle takes the memory an
    earlier handle of the same size freed after its slots had stored solver states (centres), or NaN from a freed tensor."""
    S = node_set('cp20')
    idx = S.feas[:2]
    for dirty in ('states', 'nan'):
        if dirty == 'states':
            old = _handle(S.pd, 2)
            S.hot2(idx, S.y_own[idx[::-1]], S.yc_own[idx[::-1]], h=old)
            torch.cuda.synchronize()
            old.close()
        else:
            junk = torch.full((256 << 20,), float('nan'), dtype=torch.float64, device='cuda')        # 2 GB of NaN
            torch.cuda.synchronize()
            del junk
            torch.cuda.empty_cache()
        h = _handle(S.pd, 2)
        first = S.solve(idx, h=h, hot=np.ones(idx.size, np.int32))
        cold = S.solve(idx, h=h, hot=np.zeros(idx.size, np.int32))
        h.close()
        for j in range(idx.size):
            assert _bits(first, j) == _bits(cold, j), (dirty, j, first['iters'][j], cold['iters'][j], first['cost'][j], cold['cost'][j])
        S.agree(first, idx, ('fresh hot1', dirty))


def test_budgets_give_the_cold_answer_or_the_iteration_limit():
    """qp_options max_iter = M / max_prox small: every solve returns status 9 with cost +inf or agrees with the cold answer
    at the default budgets; a cold start stays within M iterations, a hot start within min(hot_cap, M) + M (hot_cap =
    max(2n, 200) iterations, then one restart from the empty working set with M more)."""
    S = node_set('cp20')
    n = S.pd.n
    hot_cap = max(2 * n, 200)
    it_cold = S.cold['iters']
    print('cp20 cold iterations: median %d, 90th percentile %d, max %d' % (np.median(it_cold), np.percentile(it_cold, 90), it_cold.max()))
    starts = S.starts(seed=2)
    # M below and around the cold iteration counts (each below the largest, so that some cold solve runs out)
    Ms = sorted(set(min(int(np.percentile(it_cold, q)), int(it_cold.max()) - 1) for q in (25, 50, 90)))
    restarted = 0
    for opts in [dict(max_iter=M) for M in Ms] + [dict(max_prox=1), dict(max_prox=2)]:
        b = tuple(opts.items())
        M = opts.get('max_iter', S.pd.max_iter)
        ctl = make_controller(S.model, qp_options=opts)
        h = _handle(ctl.problem, S.N)
        n9 = 0
        cold = S.solve(h=h)
        S.agree(cold, np.arange(S.N), ('cold', b), limit_ok=True)
        assert cold['iters'].max() <= M
        n9 += np.sum(cold['status'] == 9)
        for what in ('own', 'scaled 1e6', 'stranger x0', 'stranger deeper', 'stranger shallower', 'farkas', 'sparse',
                     'wide', 'dense', 'centre random'):
            idx, y0, yc0 = starts[what]
            out = S.hot2(idx, y0, yc0, h=h)
            S.agree(out, idx, (what, b), limit_ok=True)
            cap = min(hot_cap, M)
            assert out['iters'].max() <= cap + M, (what, b, out['iters'].max())
            n9 += np.sum(out['status'] == 9)
            restarted += np.sum((out['status'] != 9) & (out['iters'] > cap))
        h.close()
        assert n9 > 0, b                        # the budget bites
    assert restarted > 0                        # some hot start ran into its cap and finished from the cold restart


def test_one_lane_and_two_lane_kernels_agree_bit_for_bit():
    """The same nodes, cold and from the wide and dense starts, with 8 slots and with one slot per SM (the one-lane kernel
    and its large pool) and with more slots than 2 x SMs (the two-lane kernel: factor columns beyond its pool go to L2):
    bit-identical outputs."""
    S = node_set('cp20')
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = 2 * sms + 1
    starts = S.starts(seed=3)
    runs = {}
    for n_slots in (8, sms, B):
        h = _handle(S.pd, n_slots)
        r = [S.solve(np.arange(B) % S.N, h=h)]
        for what in ('wide', 'dense'):
            idx, y0, yc0 = starts[what]
            rep = np.arange(B) % idx.size
            r.append(S.hot2(idx[rep], y0[rep], yc0, h=h))
        runs[n_slots] = [_bits(o) for o in r]
        h.close()
    assert runs[8] == runs[sms] == runs[B]
