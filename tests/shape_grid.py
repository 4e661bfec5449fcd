"""Problem shapes at the branch conditions of the kernels, shared by tests/test_shape_grid_cpu.py,
tests/test_gpu_shapes.py and tests/test_gpu_shape_search.py.

The shipped models (CP20, CP40, CP1W40, SYN30) are even in every dimension the kernels branch on.  Each entry below is a
deterministic generator call (oracle.models.build_synthetic, or CP20 at another horizon, the way CP40 is made) and the
conditions it is there for.  `conditions` computes those conditions from the generated model alone, so that the CPU
suite can prove that the grid still covers every one of COVERAGE.
"""
import functools

import numpy as np

# tiers: which parts of the hot path a shape runs through
REFUSED = 'refused'      # wshmpc_create refuses the problem
K1 = 'K1'                # node QPs only
K3 = 'K1+K3'             # node QPs and the device search; the tree shift and the fused loop refuse the problem
ALL = 'all'              # node QPs, search, tree shift (K2 + K4) and the fused loop

WS_NT, WS_RPT = 256, 2   # threads of a solver lane, rows of the removal sweep per thread (qp_device.cuh)


class Shape(object):
    def __init__(self, name, gen, tier, targets, seed=1, x0_scale=1., elim=()):
        """gen: dict(nx, nuc, nub, T) of build_synthetic, or an int T: CP20 at horizon T.  elim: values of pd.n_elim the
        K1 tests also run with, besides the one the problem compiler chooses (nb on every shape here)."""
        self.name, self.gen, self.tier, self.targets = name, gen, tier, targets
        self.seed, self.x0_scale, self.elim = seed, x0_scale, tuple(elim)

    def __repr__(self):
        return self.name

    def model(self):
        return _model(self.name)

    def x0(self):
        return self.x0_scale * np.asarray(self.model()['x0_nominal'], dtype=float)


GRID = [
    Shape('odd_rec', dict(nx=3, nuc=2, nub=3, T=7), ALL, 'odd n, odd m; even dual + odd n: a stride of dual + n would '
          'put every odd record off a 16-byte boundary', elim=(0, 7)),
    Shape('odd_dual', dict(nx=5, nuc=1, nub=2, T=9), ALL, 'odd n, odd dual: the shift reads every record in place'),
    Shape('cp21', 21, ALL, 'odd T and odd ns on a model with a terminal set (nh1 != nh)', elim=(0, 41)),
    Shape('cp8', 8, ALL, 'nb = 32: one full identifier word', x0_scale=0.3),
    Shape('nub1_T32', dict(nx=4, nuc=2, nub=1, T=32), ALL, 'nub = 1, nb = 32'),
    Shape('nub32', dict(nx=2, nuc=1, nub=32, T=2), ALL, 'nub = 32 (the full-word mask of the shift), T = 2, two full words',
          elim=(0, 33)),
    Shape('nub33', dict(nx=3, nuc=2, nub=33, T=2), K3, 'nub > 32: search works, shift and fused loop refuse'),
    Shape('nx32', dict(nx=32, nuc=1, nub=2, T=3), ALL, 'nx = 32 (the last state count of the warp recursion), odd n'),
    Shape('nx33', dict(nx=33, nuc=2, nub=2, T=4), ALL, 'nx > 32: the second recursion of the record epilogue'),
    Shape('T1', dict(nx=3, nuc=2, nub=3, T=1), K3, 'T = 1: search works, shift and fused loop refuse'),
    Shape('n512', dict(nx=4, nuc=4, nub=12, T=32), K1, 'n = 512, the largest accepted; gp = 0'),
    Shape('n513', dict(nx=3, nuc=2, nub=1, T=171), REFUSED, 'n = 513: wshmpc_create refuses with -4'),
]
BY_NAME = {s.name: s for s in GRID}


@functools.lru_cache(maxsize=None)
def _model(name):
    from oracle.models import build_synthetic, load_model
    s = BY_NAME[name]
    if isinstance(s.gen, int):
        return dict(load_model('cp20'), name=name, T=s.gen)
    return build_synthetic(name, seed=s.seed, **s.gen)


def dims(model):
    """Sizes of the condensed problem and its records (problem.ProblemData and wshmpc_create, without the compile)."""
    from warm_start_hmpc_b200.problem import RecordLayout
    T, nub = int(model['T']), int(model['nub'])
    nx, nu = model['B'].shape
    nh, nh1 = model['h'].size, model['h_Tm1'].size
    n, nb = T * nu, T * nub
    mc = (T - 1) * nh + nh1
    L = RecordLayout(T, nx, nu, nub, mc, model['Q'].shape[0], model['Q_T'].shape[0], model['R'].shape[0])
    ns = n + T * nx
    ns2 = (ns + 1) & ~1
    return dict(T=T, nx=nx, nu=nu, nub=nub, nh=nh, nh1=nh1, n=n, nb=nb, ns=ns, m=mc + nb, mc=mc, layout=L,
                gp=WS_NT // (ns2 // 2))


def staging(d):
    """Host view of the tree shift's staging predicate (csrc/bnb.cuh shift_instance): a warp with a buffer pulls a leaf's
    record into shared memory when n_dual is even and the record starts 16-byte aligned.  Returns 'all', 'none' or
    'even records' for a 16-byte aligned tree."""
    L = d['layout']
    if L.dual & 1:
        return 'none'
    return 'all' if L.rec_stride % 2 == 0 else 'even records'


def conditions(shape):
    """The branch conditions `shape` reaches, as names of COVERAGE."""
    d = dims(shape.model())
    L = d['layout']
    c = set()
    for k in ('n', 'ns', 'm'):
        c.add('%s %s' % (k, 'odd' if d[k] & 1 else 'even'))
    c.add('dual %s' % ('odd' if L.dual & 1 else 'even'))
    c.add('dual + n %s' % ('odd' if (L.dual + d['n']) & 1 else 'even'))
    if shape.tier == ALL and L.dual % 2 == 0 and (L.dual + d['n']) % 2 == 1:
        c.add('shift stages records that dual + n would misalign')
    if shape.tier == ALL and L.dual & 1:
        c.add('shift reads every record in place')
    if d['nb'] % 32 == 0:
        c.add('nb % 32 == 0')
    if d['nub'] == 1:
        c.add('nub == 1')
    if d['nub'] == 32 and shape.tier == ALL:
        c.add('nub == 32 through the shift')
    if d['nub'] > 32:
        c.add('nub > 32')
    if d['nx'] == 32:
        c.add('nx == 32')
    if d['nx'] > 32:
        c.add('nx > 32')
    if shape.tier != REFUSED and (d['n'] * (d['n'] + 1) // 2) % 2 == 1:
        c.add('n (n + 1) / 2 odd')                          # the factor's triangle: an odd whole-factor pool of a lane
    if d['T'] in (1, 2):
        c.add('T == %d' % d['T'])
    if d['T'] == 2 and shape.tier == ALL:
        c.add('H = T - 1 == 1')                             # the longest plan hold of the fallback is one step
    if d['nu'] - d['nub'] > 1:
        c.add('nuc > 1')                                    # binaries start nuc entries into an input, not at 1
    if d['nu'] & 1:
        c.add('nu odd')
    words, tail = (d['nb'] + 31) // 32, d['nb'] % 32
    if words > 1 and tail:
        c.add('words > 1 with a partial last word')
    if words == 1 and tail == 0:
        c.add('one full identifier word')
    if d['T'] & 1 and d['nh1'] != d['nh'] and shape.tier == ALL:
        c.add('odd T with a terminal set')
    if shape.tier != REFUSED:
        c.add('gp == 0' if d['gp'] == 0 else 'gp > 0')
        if d['n'] == WS_RPT * WS_NT:
            c.add('n == 512')
    if d['n'] > WS_RPT * WS_NT and shape.tier == REFUSED:
        c.add('n > 512 refused')
    for k in shape.elim:
        c.add('n_elim == 0' if k == 0 else ('0 < n_elim < nb, odd' if 0 < k < d['nb'] and k & 1 else 'n_elim out of range'))
    if shape.tier != REFUSED:
        c.add('n_elim == nb')
    return c


COVERAGE = ['n odd', 'n even', 'ns odd', 'ns even', 'm odd', 'm even', 'dual odd', 'dual even', 'dual + n odd',
            'dual + n even', 'shift stages records that dual + n would misalign', 'shift reads every record in place',
            'nb % 32 == 0', 'nub == 1', 'nub == 32 through the shift', 'nub > 32', 'nx == 32', 'nx > 32', 'T == 1', 'T == 2',
            'odd T with a terminal set', 'n (n + 1) / 2 odd', 'gp == 0', 'gp > 0', 'n == 512', 'n > 512 refused', 'n_elim == 0',
            '0 < n_elim < nb, odd', 'n_elim == nb', 'nuc > 1', 'nu odd', 'words > 1 with a partial last word',
            'one full identifier word', 'H = T - 1 == 1']


def problem(shape, n_elim=None):
    """problem.ProblemData of the shape, with pd.n_elim overridden (before any handle is made from it)."""
    from tests.util import make_problem
    pd = make_problem(shape.model())
    if n_elim is not None:
        pd.n_elim = int(n_elim)
    return pd


def oracle_optimum(shape):
    """Binary sequence [nb] of the optimum at shape.x0() by the oracle's branch and bound (None if infeasible)."""
    from oracle.bnb_ref import OracleController
    from oracle.qp_c import CoreC
    model = shape.model()
    inc, _, _ = OracleController(model, CoreC(model, variant=1), hot_start='record').feedforward(shape.x0())
    return None if inc is None else np.round(inc.primal['u'][:, model['B'].shape[1] - int(model['nub']):]).ravel()


def nodes(shape, N, seed=0, opt=None):
    """N seeded nodes of the shape: the root, chronological prefixes of every depth parity, pins behind a gap, and
    all-pinned identifiers (all zeros, and random values).  With `opt` (oracle_optimum) every second node is a prefix of
    the optimum at shape.x0(), mostly feasible; the others are random values at random states, mostly infeasible."""
    model = shape.model()
    d = dims(model)
    nb, nx = d['nb'], d['nx']
    rng = np.random.default_rng(seed)
    xm = np.asarray(model['x_max'], dtype=float)
    x0 = rng.uniform(-1, 1, (N, nx)) * xm * 0.5
    x0[0] = shape.x0()
    lb = np.zeros((N, nb)); ub = np.ones((N, nb))
    depths = rng.integers(0, nb + 1, N)
    depths[0] = 0
    for k in range(1, N):
        dk = int(depths[k])
        if k % 8 == 1:
            dk = nb                                              # all pinned
        vals = (rng.random(dk) < 0.3).astype(float) if k % 16 != 1 else np.zeros(dk)
        if opt is not None and k % 2 == 0:
            x0[k] = shape.x0()
            vals = opt[:dk]
        lb[k, :dk] = ub[k, :dk] = vals
        if k % 5 == 2 and dk + 2 < nb:                           # pins behind a gap: two-sided rows, not eliminated
            for j in rng.choice(np.arange(dk + 1, nb), size=min(3, nb - dk - 1), replace=False):
                lb[k, j] = ub[k, j] = float(rng.random() < 0.5)
    return x0, lb, ub
