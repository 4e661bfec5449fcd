"""-m gpu: the kernels on the shape grid (tests/shape_grid.py), the problem shapes they branch on: odd n, ns, m and dual,
records whose unpadded stride would be odd, identifier words that are exactly full, nub = 32 and nub > 32, nx = 32 and
nx > 32, T = 1 and T = 2, n at the size limit and beyond it, partial and switched-off elimination.

Per shape: the refusals the C ABI documents, K1 against the oracle with its certificates and from its own records, the
elimination settings against each other, lane counts against each other, the search and the tree shift against the
oracle controller, K2 + K4 on the oracle's own leaves (also on trees whose records start off a 16-byte boundary), and
the fused loop against lock step.  Run with -s for one line per shape: the branches it reaches, the staging of the tree
shift, the largest working set, the lanes per CTA and the time.
"""
import time

import numpy as np
import pytest
import torch

from oracle.condense import Condensed
from oracle.qp_c import CoreC
from oracle.bnb_ref import OracleController
from tests import shape_grid as sg
from tests.util import make_controller, make_problem, check_node_result, record_to_y0, oracle_loop, COST_RTOL

pytestmark = pytest.mark.gpu

LIVE = [s for s in sg.GRID if s.tier != sg.REFUSED]
LOOP = [s for s in sg.GRID if s.tier == sg.ALL]
ELIM = [s for s in sg.GRID if s.elim]
N_NODES = dict(n512=16)
# lanes per CTA the handle of n512 chooses from the shared-memory budget, seen on a B200 (227 KB of shared memory a block)
N512_LANES = 1


class Built(object):
    """A shape compiled once: its model, ProblemData, controller (search and loop tiers), nodes and the oracle's answers."""

    def __init__(self, shape):
        t = time.time()
        self.shape = shape
        self.model = shape.model()
        self.ctl = make_controller(self.model) if shape.tier in (sg.K3, sg.ALL) else None
        self.pd = self.ctl.problem if self.ctl is not None else make_problem(self.model)
        self.cond = Condensed(self.model)
        self.opt = sg.oracle_optimum(shape) if self.ctl is not None else None
        self.N = N_NODES.get(shape.name, 100)
        self.x0, self.lb, self.ub = sg.nodes(shape, self.N, seed=3, opt=self.opt)
        core = CoreC(self.model, variant=1)
        self.ref = [core.solve(self.x0[i], self.lb[i], self.ub[i]) for i in range(self.N)]
        self.lanes = None
        self.seconds = time.time() - t

    def handle(self, n_slots, n_elim=None):
        from warm_start_hmpc_b200.capi import Handle, load_library
        pd = self.pd
        if n_elim is not None:
            pd = sg.problem(self.shape, n_elim)
        h = Handle(pd, n_slots=n_slots)
        if n_elim is None and self.lanes is None:
            self.lanes = int(load_library().wshmpc_ctas_per_sm())
        return h

    def solve(self, h, **kw):
        out = h.solve_nodes(self.x0, self.lb, self.ub, **kw)
        return {k: v.cpu().numpy() for k, v in out.items()}

    def check(self, out, layout, i, cost_ref=None, tag=None):
        check_node_result(self.model, self.cond, self.pd, layout, self.x0[i], self.lb[i], self.ub[i], out['status'][i],
                          out['cost'][i], out['dobj'][i], out['primal'][i], out['dual'][i], cost_ref=cost_ref, tag=tag)


@pytest.fixture(scope='module')
def built():
    cache = {}

    def get(shape):
        if shape.name not in cache:
            cache[shape.name] = Built(shape)
        return cache[shape.name]
    return get


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- 1. create, and refuse as documented ---------------------------------------------------------------------------------
def test_n513_is_refused_with_minus_4():
    from warm_start_hmpc_b200.capi import Handle
    pd = make_problem(sg.BY_NAME['n513'].model())
    assert pd.n == 513
    with pytest.raises(RuntimeError, match=r'wshmpc error -4: problem too large: n = 513'):
        Handle(pd, n_slots=1)


@pytest.mark.parametrize('shape', LIVE, ids=str)
def test_library_layout_equals_record_layout(built, shape):
    b = built(shape)
    h = b.handle(1)
    L = b.pd.layout
    for k in ('primal', 'dual', 'off_lam', 'off_mu', 'off_nu_lb', 'off_nu_ub', 'off_rho', 'off_sigma', 'rec_stride'):
        assert getattr(h.layout, k) == getattr(L, k), (shape.name, k, getattr(h.layout, k), getattr(L, k))
    assert h.layout.rec_stride % 2 == 0


@pytest.mark.parametrize('shape', [s for s in sg.GRID if s.tier == sg.K3], ids=str)
def test_search_works_and_shift_refuses(built, shape):
    """nub > 32 and T = 1: the device search solves the MIQP (against the oracle), the tree shift and the fused loop refuse
    with -1 and say why."""
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    b = built(shape)
    ctl = b.ctl
    res, tree = ctl.feedforward_batch(b.shape.x0()[None], n_slots=1)
    ref, _, n_ref = OracleController(b.model, CoreC(b.model, variant=1), hot_start='record').feedforward(b.shape.x0())
    assert int(res['status'][0]) == 0 and ref is not None
    c = float(res['cost'][0])
    assert abs(c - ref.primal['objective']) <= COST_RTOL * abs(ref.primal['objective']), (c, ref.primal['objective'])
    msg = 'tree shifting needs T >= 2' if b.pd.T < 2 else 'tree shifting supports nub <= 32'
    with pytest.raises(RuntimeError, match='wshmpc error -1: ' + msg):
        ctl.construct_warm_start_batch(res, tree)
    L = ClosedLoop(ctl, 1, warm=True, max_solves=1024, max_roots=64, n_slots=1)
    L.reset(b.shape.x0()[None])
    with pytest.raises(RuntimeError, match='wshmpc error -1: ' + msg):
        L.run(1)
    with pytest.raises(RuntimeError, match='wshmpc error -1: ' + msg):
        L.step()


def test_a_handle_keeps_launching_after_a_smaller_problem_gets_one(built):
    """The shared-memory limit of a kernel is set per kernel, not per handle: a handle made later for a smaller problem must
    not stop an earlier handle's node solves, searches and tree shifts from launching."""
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    big, small = built(sg.BY_NAME['cp21']), built(sg.BY_NAME['T1'])
    h = big.handle(8)
    before = big.solve(h, slot=np.arange(big.N) % 8)
    L = ClosedLoop(big.ctl, 2, warm=True, max_solves=1024, max_roots=512, n_slots=2)
    L.reset(np.repeat(big.shape.x0()[None], 2, 0))
    small.handle(8)
    after = big.solve(h, slot=np.arange(big.N) % 8)
    assert all(np.array_equal(after[k], before[k], equal_nan=True) for k in before)
    for _ in range(2):
        out = L.step()
        assert out['status'].tolist() == [0, 0]


# ---- 2. K1 against the oracle, and from its own records --------------------------------------------------------------------
@pytest.mark.parametrize('shape', LIVE, ids=str)
def test_k1_matches_oracle_and_restarts_from_its_records(built, shape):
    b = built(shape)
    t = time.time()
    h = b.handle(b.N)
    out = b.solve(h)
    st = out['status']
    for i in range(b.N):
        assert st[i] == b.ref[i]['status'], (shape.name, i, st[i], b.ref[i]['status'])
        b.check(out, h.layout, i, cost_ref=b.ref[i]['cost'] if st[i] == 2 else None, tag=(shape.name, 'cold', i))
    assert set(st) == {2, 3} or b.N < 50, (shape.name, np.bincount(st))        # optimal and infeasible nodes both
    # hot = 2 from each node's own multipliers and centre
    own = b.solve(h, hot=np.full(b.N, 2, np.int32), y0=record_to_y0(out['dual'], h.layout), yc0=out['yc'])
    assert np.array_equal(own['status'], st), shape.name
    ok = st == 2
    assert np.all(np.abs(own['cost'][ok] - out['cost'][ok]) <= COST_RTOL * np.abs(out['cost'][ok])), shape.name
    for i in range(b.N):
        b.check(own, h.layout, i, cost_ref=out['cost'][i] if ok[i] else None, tag=(shape.name, 'own', i))
    d = sg.dims(b.model)
    print('\n%s: n %d ns %d m %d nb %d dual %d rec_stride %d; shift staging %s; %d nodes (%d feasible); lanes per CTA %d; '
          'K1 %.1f s, set-up %.1f s; reaches: %s' % (shape.name, d['n'], d['ns'], d['m'], d['nb'], d['layout'].dual,
                                                     d['layout'].rec_stride, sg.staging(d), b.N, ok.sum(), b.lanes,
                                                     time.time() - t, b.seconds, '; '.join(sorted(sg.conditions(shape)))))
    if shape.name == 'n512' and N512_LANES is not None:
        assert b.lanes == N512_LANES


# ---- 3. elimination settings agree --------------------------------------------------------------------------------------
@pytest.mark.parametrize('shape', ELIM, ids=str)
def test_elimination_settings_agree(built, shape):
    b = built(shape)
    full = b.solve(b.handle(b.N))
    for k in shape.elim:
        h = b.handle(b.N, n_elim=k)
        out = b.solve(h)
        assert np.array_equal(out['status'], full['status']), (shape.name, k)
        ok = full['status'] == 2
        assert np.all(np.abs(out['cost'][ok] - full['cost'][ok]) <= 1e-9 * np.abs(full['cost'][ok])), (shape.name, k)
        for i in range(b.N):
            b.check(out, h.layout, i, cost_ref=full['cost'][i] if ok[i] else None, tag=(shape.name, 'n_elim', k, i))


# ---- 4. lanes ---------------------------------------------------------------------------------------------------------
def _instances(b, N, seed):
    rng = np.random.default_rng(seed)
    xm = np.asarray(b.model['x_max'], dtype=float)
    return b.shape.x0()[None] + 0.02 * b.shape.x0_scale * rng.uniform(-1, 1, (N, xm.size)) * xm


@pytest.mark.parametrize('shape', LIVE, ids=str)
def test_lane_counts_agree_bit_for_bit(built, shape):
    """K1 with 8 slots, one per SM and more than two per SM (one-lane and two-lane kernels where the budget allows two),
    and on the loop tier a short fused loop as well: bit-identical."""
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    b = built(shape)
    sms = _sms()
    runs = [b.solve(b.handle(s), slot=np.arange(b.N) % s) for s in (8, sms, 2 * sms + 8)]
    for r in runs[1:]:
        for k in ('status', 'cost', 'dobj', 'iters', 'primal', 'dual', 'yc'):
            assert np.array_equal(r[k], runs[0][k], equal_nan=True), (shape.name, k)
    if shape.tier != sg.ALL:
        return
    N, S = 2 * sms + 8, 2
    x0 = _instances(b, N, 1)
    e = torch.as_tensor(0.003 * np.random.default_rng(2).standard_normal((S, N, x0.shape[1])) * b.model['x_max'], device='cuda')
    ctl = make_controller(b.model)                        # its handle grows with the slot count, as in test_gpu_lanes.py
    loops = []
    for slots in (8, sms, 2 * sms + 8):
        L = ClosedLoop(ctl, N, warm=True, max_solves=1024, max_roots=1024, n_slots=slots)
        L.reset(x0)
        logs = L.run(S, e=e)
        torch.cuda.synchronize()
        loops.append((logs['cost'].clone(), logs['n_solves'].clone(), L.x.clone(), L.active.clone(), int(L.totals[1])))
        del L
    for r in loops[1:]:
        assert all(torch.equal(r[q], loops[0][q]) for q in range(4)) and r[4] == loops[0][4], shape.name


# ---- 5. search and shift against the oracle controller -----------------------------------------------------------------
def _ub_of(pd, primal_row):
    return primal_row[(pd.T + 1) * pd.nx:].reshape(pd.T, pd.nu)[:, pd.nu - pd.nub:]


@pytest.mark.parametrize('shape', LOOP, ids=str)
def test_search_and_shift_match_oracle_controller(built, shape):
    """A cold step and three warm-started steps with model errors (0.003 x_max): cost, mode sequence, first input, cover
    of the warm start and node count against the oracle loop."""
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    b = built(shape)
    t0 = time.time()
    S = 4
    x0 = b.shape.x0()
    e = 0.003 * np.random.default_rng(3).standard_normal((S, x0.size)) * b.model['x_max']
    ref = oracle_loop(b.model, x0, e)
    assert len(ref) == S and all(np.isfinite(r['cost']) for r in ref), shape.name
    L = ClosedLoop(b.ctl, 1, warm=True, max_solves=4096, max_roots=2048, n_slots=1)
    L.reset(x0[None])
    counts = []
    for t in range(S):
        out = L.step(e=torch.as_tensor(e[t][None], device='cuda'))
        assert int(out['status'][0]) == 0, (shape.name, t, int(out['status'][0]))
        c = float(out['cost'][0])
        assert abs(c - ref[t]['cost']) <= 1e-6 * abs(ref[t]['cost']), (shape.name, t, c, ref[t]['cost'])
        assert np.array_equal(_ub_of(b.pd, out['primal'][0].cpu().numpy()), np.round(ref[t]['ub'])), (shape.name, t)
        assert np.allclose(L.u0[0].cpu().numpy(), ref[t]['u0'], rtol=1e-6, atol=1e-6), (shape.name, t)
        cover = int(L.trees[L.cur].n_nodes[0])
        assert cover == ref[t]['cover'], (shape.name, t, cover, ref[t]['cover'])
        n = int(out['n_solves'][0])
        counts.append((n, ref[t]['solves']))
        assert abs(n - ref[t]['solves']) <= max(8, ref[t]['solves'] // 10), (shape.name, t, n, ref[t]['solves'])
    print('\n%s: QPs per step (device, oracle) %s; largest working set %d rows; %.1f s'
          % (shape.name, counts, int(L.totals[3]), time.time() - t0))


# ---- 6. K2 + K4 on the oracle's own leaves ------------------------------------------------------------------------------
def _record(var, yc, layout, n):
    """A dual record of a device tree from the oracle's dual variables; the centre (not read by the shift) and the padding
    double carry non-zero values that the shifted records must not inherit."""
    rec = np.full(layout.rec_stride, 5.)
    rec[:layout.dual] = np.concatenate([np.concatenate([np.asarray(v, dtype=float).ravel() for v in var[k]])
                                        for k in ('lam', 'mu', 'nu_lb', 'nu_ub', 'rho', 'sigma')])
    rec[layout.dual:layout.dual + n] = yc if yc is not None else 7.
    return rec


def _offset_records(tree, offset):
    """Moves the tree's records into a view that starts `offset` doubles into a larger allocation."""
    big = torch.zeros(tree.rec_dual.numel() + offset, dtype=torch.float64, device=tree.rec_dual.device)
    view = big[offset:].view(tree.rec_dual.shape)
    view.copy_(tree.rec_dual)
    tree._big, tree.rec_dual = big, view
    tree.c.rec_dual = view.data_ptr()


def _upload_leaves(h, pd, leaves, offset=0):
    nb, nub, L = pd.nb, pd.nub, h.layout
    n0 = len(leaves)
    tree = h.new_tree(1, n0 + 2, n0 + 1)
    if offset:
        _offset_records(tree, offset)
    dev = tree.lb.device
    bits = np.zeros((n0, tree.words), np.uint32); mask = np.zeros((n0, tree.words), np.uint32)
    rec = np.zeros(n0, np.int32); recs, dobj, seen = [], [], {}
    for j, l in enumerate(leaves):
        for (t, i), v in l.identifier.items():
            q = t * nub + i
            mask[j, q >> 5] |= np.uint32(1 << (q & 31))
            if v:
                bits[j, q >> 5] |= np.uint32(1 << (q & 31))
        if id(l.dual) not in seen:
            seen[id(l.dual)] = len(recs)
            recs.append(_record(l.dual['variables'], l.dual.get('yc'), L, pd.n)); dobj.append(l.dual['objective'])
        rec[j] = seen[id(l.dual)]
    tree.n_nodes[0] = n0; tree.n_recs[0] = len(recs)
    tree.depth[0, :n0] = torch.as_tensor([len(l.identifier) for l in leaves], dtype=torch.int32, device=dev)
    tree.alive[0, :n0] = 1
    tree.rec[0, :n0] = torch.as_tensor(rec, device=dev)
    tree.lb[0, :n0] = torch.as_tensor([l.lb for l in leaves], dtype=torch.float64, device=dev)
    tree.bits[0, :n0] = torch.as_tensor(bits.view(np.int32), device=dev)
    tree.mask[0, :n0] = torch.as_tensor(mask.view(np.int32), device=dev)
    tree.rec_dual[0, :len(recs)] = torch.as_tensor(np.vstack(recs), device=dev)
    tree.rec_dobj[0, :len(recs)] = torch.as_tensor(np.array(dobj), device=dev)
    return tree


def _shift(h, pd, leaves, inc, x0, e0, offset=0):
    dev = h.torch_device
    tree = _upload_leaves(h, pd, leaves, offset)
    new = h.new_tree(1, len(leaves) + 2, len(leaves) + 1)
    if offset:
        _offset_records(new, offset)
    primal = torch.as_tensor(np.concatenate((inc.primal['x'].ravel(), inc.primal['u'].ravel()))[None], device=dev).contiguous()
    cost = torch.full((1,), inc.primal['objective'], dtype=torch.float64, device=dev)
    x_next = torch.empty((1, pd.nx), dtype=torch.float64, device=dev)
    u0 = torch.empty((1, pd.nu), dtype=torch.float64, device=dev)
    h.shift_tree(torch.as_tensor(x0[None], device=dev).contiguous(), torch.as_tensor(e0[None], device=dev).contiguous(),
                 tree, cost, primal, new, x_next=x_next, u0=u0)
    torch.cuda.synchronize()
    nn = int(new.n_nodes[0])
    return dict(n=nn, n_recs=int(new.n_recs[0]), depth=new.depth[0, :nn].cpu().numpy(), bits=new.bits[0, :nn].cpu().numpy(),
                mask=new.mask[0, :nn].cpu().numpy(), lb=new.lb[0, :nn].cpu().numpy(), rec=new.rec[0, :nn].cpu().numpy(),
                dobj=new.rec_dobj[0, :nn].cpu().numpy(), recs=new.rec_dual[0, :nn].cpu().numpy(),
                x_next=x_next.cpu().numpy(), u0=u0.cpu().numpy())


@pytest.mark.parametrize('shape', LOOP, ids=str)
def test_shift_tree_matches_oracle_construct_warm_start(built, shape):
    b = built(shape)
    pd, h = b.pd, b.ctl.handle()
    L = h.layout
    x0 = b.shape.x0()
    octl = OracleController(b.model, CoreC(b.model, variant=1), hot_start='record')
    inc, leaves, _ = octl.feedforward(x0)
    e0 = 0.003 * np.random.default_rng(4).standard_normal(x0.size) * b.model['x_max']
    u0 = inc.primal['u'][0]
    ws = octl.construct_warm_start(leaves, x0, u0[:octl.nuc], u0[octl.nuc:], e0)
    got = _shift(h, pd, leaves, inc, x0, e0)
    n = got['n']
    assert n == len(ws) > 0 and got['n_recs'] == n, (shape.name, n, len(ws))
    nb, nub = pd.nb, pd.nub
    scale = max(1., max(abs(l.dual['objective']) for l in leaves))
    for j, node in enumerate(ws):
        assert got['depth'][j] == len(node.identifier), (shape.name, j)
        bits = np.zeros(got['bits'].shape[1], np.uint32); mask = np.zeros_like(bits)
        for (t, i), v in node.identifier.items():
            q = t * nub + i
            mask[q >> 5] |= np.uint32(1 << (q & 31))
            bits[q >> 5] |= np.uint32(int(v) << (q & 31))
        assert np.array_equal(got['bits'][j].view(np.uint32), bits) and np.array_equal(got['mask'][j].view(np.uint32), mask), (shape.name, j)
        assert np.isinf(got['lb'][j]) == np.isinf(node.lb), (shape.name, j)
        if np.isfinite(node.lb):
            assert abs(got['lb'][j] - node.lb) <= 1e-11 * scale, (shape.name, j, got['lb'][j], node.lb)
        rec = got['recs'][j]
        assert np.all(rec[L.dual:] == 0.), (shape.name, j)                 # the centre and the padding double
        if node.dual is None:
            assert got['rec'][j] == -2 - j and got['lb'][j] == 0., (shape.name, j)
            continue
        assert got['rec'][j] == j
        assert abs(got['dobj'][j] - node.dual['objective']) <= 1e-11 * scale, (shape.name, j)
        want = _record(node.dual['variables'], None, L, pd.n)[:L.dual]
        assert np.allclose(rec[:L.dual], want, rtol=1e-13, atol=1e-13 * max(1., np.abs(want).max())), \
            (shape.name, j, np.abs(rec[:L.dual] - want).max())
    assert np.array_equal(got['x_next'][0], inc.primal['x'][1] + e0)
    assert np.array_equal(got['u0'][0], u0)
    if shape.name == 'odd_rec':
        # every record one double off a 16-byte boundary: the shift reads them in place, with the same bits
        off = _shift(h, pd, leaves, inc, x0, e0, offset=1)
        for k, v in got.items():
            assert np.array_equal(np.asarray(off[k]), np.asarray(v)), (shape.name, k)


@pytest.mark.parametrize('shape', [sg.BY_NAME['odd_rec'], sg.BY_NAME['T1']], ids=str)
def test_search_writes_zero_padding(built, shape):
    """The records the device search writes end in the zero padding double where dual + n is odd."""
    b = built(shape)
    L = b.ctl.handle().layout
    assert L.rec_stride == L.dual + b.pd.n + 1
    tree = b.ctl.new_tree(1, 1, 256)
    tree.rec_dual.fill_(np.nan)
    b.ctl.handle().tree_init_root(tree)
    res, _ = b.ctl.feedforward_batch(b.shape.x0()[None], warm_start=tree, max_solves=256, n_slots=1)
    nr = int(tree.n_recs[0])
    assert int(res['status'][0]) == 0 and nr > 1
    recs = tree.rec_dual[0, :nr].cpu().numpy()
    assert np.all(recs[:, -1] == 0.) and not np.isnan(recs).any()


# ---- 7. fused loop equals lock step ------------------------------------------------------------------------------------
@pytest.mark.parametrize('warm', [True, False])
@pytest.mark.parametrize('shape', LOOP, ids=str)
def test_fused_loop_equals_lock_step(built, shape, warm):
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    b = built(shape)
    N, S = 24, 3
    x0 = _instances(b, N, 5)
    e = torch.as_tensor(0.003 * np.random.default_rng(6).standard_normal((S, N, x0.shape[1])) * b.model['x_max'], device='cuda')
    A = ClosedLoop(b.ctl, N, warm=warm, max_solves=4096, max_roots=2048)
    B = ClosedLoop(b.ctl, N, warm=warm, max_solves=4096, max_roots=2048)
    A.reset(x0); B.reset(x0)
    cost, ns, u0 = [], [], []
    for t in range(S):
        out = A.step(e=e[t])
        cost.append(out['cost'].clone()); ns.append(out['n_solves'].clone()); u0.append(A.u0.clone())
    logs = B.run(S, e=e)
    torch.cuda.synchronize()
    assert torch.equal(torch.stack(ns), logs['n_solves']) and torch.equal(torch.stack(cost), logs['cost']), shape.name
    a, c = torch.stack(u0), logs['u0']
    assert torch.equal(torch.isnan(a), torch.isnan(c)) and torch.equal(torch.nan_to_num(a), torch.nan_to_num(c))
    assert torch.equal(A.x, B.x) and torch.equal(A.active, B.active)
    assert bool(torch.isfinite(logs['cost']).any()), shape.name
