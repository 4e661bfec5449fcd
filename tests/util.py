"""Shared helpers of the test-suite (test infrastructure: may import oracle/)."""
import numpy as np


def make_controller(model, **kw):
    import warm_start_hmpc_b200 as ws
    mld = ws.MLDSystem([model['A'], model['B']], [model['F'], model['G'], model['h']], int(model['nub']))
    return ws.HybridModelPredictiveController(mld, int(model['T']), [model['Q'], model['R'], model['Q_T']],
                                              [model['F_T'], model['h_T']], **kw)


def make_problem(model, **kw):
    """Host-side problem compiler only (no GPU, no library)."""
    from warm_start_hmpc_b200.problem import ProblemData
    return ProblemData(model['A'], model['B'], model['F'], model['G'], model['h'], int(model['nub']), int(model['T']),
                       model['Q'], model['R'], model['Q_T'], model['F_Tm1'], model['G_Tm1'], model['h_Tm1'],
                       model['M_mu'], model['M_rho'], **kw)


def random_nodes(model, N, seed=0, pin_prob=0.15):
    """Seeded random (x0, partial identifier) pairs: prefix-in-time identifiers like the B&B produces."""
    rng = np.random.default_rng(seed)
    nx = model['A'].shape[0]
    T, nub = int(model['T']), int(model['nub'])
    nb = T * nub
    xm = model['x_max'] * (np.array([0.7, 0.64, 1.0, 0.6]) if nx == 4 else 0.5)
    x0 = rng.uniform(-1, 1, (N, nx)) * xm
    lb = np.zeros((N, nb)); ub = np.ones((N, nb))
    for k in range(N):
        d = int(rng.integers(0, nb // 2))
        vals = (rng.random(d) < pin_prob).astype(float)
        lb[k, :d] = vals; ub[k, :d] = vals
    return x0, lb, ub


def families_from_records(pd, layout, status, primal, dual):
    """GPU records -> the dict oracle/certify.py works on."""
    T, nx, nu, nub, nh, nh1, nq, nqT, nr = pd.T, pd.nx, pd.nu, pd.nub, pd.nh, pd.nh1, pd.nq, pd.nqT, pd.nr
    fam = {}
    lam = dual[layout.off_lam:layout.off_mu].reshape(T + 1, nx)
    mu = dual[layout.off_mu:layout.off_nu_lb]
    fam['lam'] = [lam[t] for t in range(T + 1)]
    fam['mu'] = [mu[t * nh:(t + 1) * nh] for t in range(T - 1)] + [mu[(T - 1) * nh:]]
    fam['nu_lb'] = list(dual[layout.off_nu_lb:layout.off_nu_ub].reshape(T, nub))
    fam['nu_ub'] = list(dual[layout.off_nu_ub:layout.off_rho].reshape(T, nub))
    rho = dual[layout.off_rho:layout.off_sigma]
    fam['rho'] = [rho[t * nq:(t + 1) * nq] for t in range(T)] + [rho[T * nq:]]
    fam['sigma'] = list(dual[layout.off_sigma:layout.dual].reshape(T, nr))
    if status == 2:
        fam['x'] = primal[:(T + 1) * nx].reshape(T + 1, nx)
        fam['u'] = primal[(T + 1) * nx:].reshape(T, nu)
    return fam


# relative cost tolerance of north_star ("optimal cost ... within 1e-6 relative")
COST_RTOL = 1e-6
# primal inequality tolerance: the kernel accepts a row violated by at most tol_p = 1e-7 in the scaling
# max(1, |row of [F G]|), escalated to at most 100 tol_p = 1e-5 on rows that entered the working set degenerately
# (qp_device.cuh pricing; Gurobi's FeasibilityTol default is 1e-6 on rows it scales itself)
PV_SCALED = 1.0e-5 * (1. + 1e-6)


def check_node_result(model, cond, pd, layout, x0, lb, ub, status, cost, dobj, primal, dual, cost_ref=None, tag=None):
    """Solver-independent certificates (oracle/certify.py) of one K1 result, in the records the kernel writes.
    Optimal: primal feasibility (pe <= 1e-9, pv <= PV_SCALED), dual feasibility (ds <= 1e-7, no negative multiplier),
    duality gap 1e-6, dobj == cost, and |cost - cost_ref| <= COST_RTOL |cost_ref| when a reference cost is given.
    Infeasible: a Farkas ray (A'y = 0 to 1e-9 of its scale, positive cost, y >= 0) whose cost dobj reports."""
    from oracle import certify as cert
    assert status in (2, 3), (tag, status)
    fam = families_from_records(pd, layout, status, primal, dual)
    ds, neg = cert.dual_residuals(model, cond, fam)
    assert neg >= 0., (tag, neg)
    dob = cert.dual_objective(model, cond, x0, lb, ub, fam)
    if status == 2:
        if cost_ref is not None:
            assert abs(cost - cost_ref) <= COST_RTOL * abs(cost_ref), (tag, cost, cost_ref)
        pe, _ = cert.primal_residuals(model, cond, x0, lb, ub, fam)
        pv = cert.primal_violation_scaled(model, cond, x0, lb, ub, fam)
        assert pe <= 1e-9 and pv <= PV_SCALED, (tag, pe, pv)
        assert ds <= 1e-7, (tag, ds)
        assert abs(cost - dob) <= 1e-6 * abs(cost), (tag, cost, dob)       # duality gap
        assert dobj == cost, (tag, dobj, cost)
    else:
        assert np.isinf(cost), (tag, cost)
        if id(cond) not in _AROW:
            _AROW[id(cond)] = (cond, np.linalg.norm(cond.Aall, axis=1))      # holds cond: its id is not reused
        arow = _AROW[id(cond)][1]
        y = np.concatenate(fam['mu'] + fam['nu_lb'] + fam['nu_ub'])
        scale = np.sum(np.concatenate(fam['mu']) * arow[:cond.mc]) + np.sum(np.concatenate(fam['nu_lb'] + fam['nu_ub']))
        assert ds <= 1e-9 * scale, (tag, ds, scale)            # A'y = 0
        assert dob > 1e-9 * scale, (tag, dob, scale)           # positive cost: a Farkas proof
        assert abs(dobj - dob) <= 1e-9 * max(1., abs(dob)), (tag, dobj, dob)
        assert y.min() >= 0., (tag, y.min())


_AROW = {}          # id(cond) -> (cond, row norms of [F G])


def leaves_from_golden(pd, g):
    """tests/golden/cp20_warmstart.npz -> [(identifier, lb, DualSolution or None)] in leaf order."""
    from warm_start_hmpc_b200.subproblem_solution import DualSolution
    nub = pd.nub
    cache = {}
    out = []
    for j in range(len(g['lb'])):
        ident = {(q // nub, q % nub): float((g['bits'][j, q >> 5] >> np.uint32(q & 31)) & np.uint32(1))
                 for q in range(int(g['depth'][j]))}
        r = int(g['rec'][j])
        if r >= 0 and r not in cache:
            cache[r] = DualSolution.from_record(pd, pd.layout, g['recs'][r], float(g['dobj'][r]))
        out.append((ident, float(g['lb'][j]), cache.get(r)))
    return out


def start_rows(y0, mc):
    """Rows of signed multipliers y0 [..., m] that enter a hot = 2 start (wshmpc_solve_nodes d_y0): finite entries that
    are non-zero on a bound row (r >= mc: either side) or positive on a stage row (r < mc: no lower side).  Every other
    entry is ignored, i.e. projected to zero."""
    y0 = np.asarray(y0)
    stage = np.arange(y0.shape[-1]) < mc
    return np.isfinite(y0) & np.where(stage, y0 > 0., y0 != 0.)


def prefix_depth(lb, ub, n_elim):
    """Coordinates K1 eliminates for a node: the leading run of pinned binaries (lb == ub), at most n_elim
    (qp_device.cuh set_node_prefix)."""
    free = np.nonzero(np.asarray(lb) != np.asarray(ub))[0]
    return min(int(free[0]) if free.size else len(lb), int(n_elim))


def record_to_y0(dual, layout):
    """Dual records [..., layout.dual] -> signed multipliers [..., m] of a hot = 2 start, [mu | nu_ub - nu_lb]
    (the conversion csrc/bnb.cuh applies to a parent's record)."""
    dual = np.asarray(dual)
    mu = dual[..., layout.off_mu:layout.off_nu_lb]
    return np.concatenate((mu, dual[..., layout.off_nu_ub:layout.off_rho] - dual[..., layout.off_nu_lb:layout.off_nu_ub]), -1)


def y0_to_multipliers(y0, mc):
    """Inverse of record_to_y0 on the multipliers of a record: (mu, nu_lb, nu_ub) >= 0."""
    y0 = np.asarray(y0)
    yb = y0[..., mc:]
    return np.maximum(y0[..., :mc], 0.), np.maximum(-yb, 0.), np.maximum(yb, 0.)


def log_uniform(rng, size, lo=1e-8, hi=1e8):
    return np.exp(rng.uniform(np.log(lo), np.log(hi), size))


def sparse_start(rng, pd, n_rows):
    """n_rows random rows with multipliers log-uniform on [1e-8, 1e8]: positive on stage rows, random side on bound rows."""
    y = np.zeros(pd.m)
    rows = rng.choice(pd.m, size=n_rows, replace=False)
    y[rows] = log_uniform(rng, n_rows) * np.where(rows < pd.mc, 1., rng.choice([-1., 1.], n_rows))
    return y


def dense_start(rng, pd):
    """Non-zero on all m rows (K1 keeps the first n entries in row order)."""
    return log_uniform(rng, pd.m) * np.concatenate((np.ones(pd.mc), rng.choice([-1., 1.], pd.nb)))


def wide_start(rng, pd, d, min_rank):
    """A start on n rows (K1 keeps n) that the node does not eliminate: min_rank independent rows of pd.Mh[:, d:] (the
    leading pivots of a column-pivoted QR of a random sample of rows of every time step), topped up with further rows of
    the sample.  Returns (y, numpy rank of its rows in the coordinates d:)."""
    from scipy.linalg import qr
    cand = np.concatenate((np.arange(pd.mc), pd.mc + np.arange(d, pd.nb)))
    step = np.where(cand < pd.mc, np.minimum(cand // pd.nh, pd.T - 1), (cand - pd.mc) // pd.nub)
    pool = np.concatenate([rng.choice(cand[step == t], size=min(2 * pd.n // pd.T, np.sum(step == t)), replace=False)
                           for t in range(pd.T)])
    piv = qr(pd.Mh[pool][:, d:].T, mode='r', pivoting=True)[1]
    rows = np.sort(np.concatenate((pool[piv[:min_rank]], rng.choice(pool[piv[min_rank:]], size=pd.n - min_rank, replace=False))))
    rank = np.linalg.matrix_rank(pd.Mh[rows][:, d:])
    assert rank >= min_rank, ('no start of rank %d at d = %d' % (min_rank, d), rank)
    y = np.zeros(pd.m)
    y[rows] = log_uniform(rng, rows.size, 1e-3, 1e3) * np.where(rows < pd.mc, 1., rng.choice([-1., 1.], rows.size))
    return y, rank


def out_of_contract(rng, y0, mc, n_each=3):
    """y0 plus entries a start ignores, on rows where y0 is zero: negative values on stage rows (no lower side), NaN,
    +inf and -inf."""
    y = np.array(y0, dtype=float)
    free_stage = np.nonzero((y == 0.) & (np.arange(y.size) < mc))[0]
    neg = rng.choice(free_stage, size=n_each, replace=False)
    y[neg] = -log_uniform(rng, n_each, 1e-6, 1e6)
    free = np.nonzero(y == 0.)[0]
    bad = rng.choice(free, size=3 * n_each, replace=False)
    y[bad] = np.repeat([np.nan, np.inf, -np.inf], n_each)
    return y


def oracle_launch(model, pd, variant=1):
    """A stand-in for BoundedQP._launch (the device call) backed by the CPU oracle core: lets the CPU suite drive the
    product's and the reference's control flow through the product's BoundedQP front end without a GPU.  Same
    contract: (x0, lb, ub, y0, yc0) -> dict(status, cost, dobj, iters, primal, dual, yc, runtime).  variant: of
    oracle/qp_core.c (1 = the CUDA kernel's thin factor, 0 = the full factor the golden fixtures were made with)."""
    from oracle.qp_c import CoreC
    from oracle.condense import Condensed
    from oracle import certify as cert
    core = CoreC(model, variant=variant)
    cond = Condensed(model)
    L = pd.layout

    def launch(x0, lb, ub, y0, yc0):
        warm = None
        if y0 is not None:
            rows = np.nonzero(start_rows(y0, pd.mc))[0]
            warm = dict(rows=rows, sides=np.where(y0[rows] > 0, 1, -1), lam=np.abs(y0[rows]), z=yc0)
        out = core.solve(x0, lb, ub, warm=warm)
        if out['status'] not in (2, 3) and warm is not None:
            out = core.solve(x0, lb, ub, warm=None)
        fam = cert.families(model, cond, x0, out['status'], out.get('z'), out['y'])
        dual = np.concatenate([np.concatenate(fam[k]) for k in ('lam', 'mu', 'nu_lb', 'nu_ub', 'rho', 'sigma')])
        assert dual.size == L.dual
        primal = np.zeros(L.primal)
        if out['status'] == 2:
            primal = np.concatenate((np.asarray(fam['x']).ravel(), np.asarray(fam['u']).ravel()))
        dobj = out['cost'] if out['status'] == 2 else out['farkas']
        yc = out['warm']['z'] if out['status'] == 2 else np.zeros(pd.n)
        return dict(status=out['status'], cost=out['cost'], dobj=dobj, iters=out['iters'], primal=primal, dual=dual,
                    yc=np.array(yc), runtime=0.)
    return launch


def oracle_loop(model, x0, e, warm=True):
    """statistical_analysis.py:93-196 for one instance on the oracle: list of per-step dicts (ends when infeasible)."""
    from oracle.qp_c import CoreC
    from oracle.bnb_ref import OracleController
    ctl = OracleController(model, CoreC(model, variant=1), hot_start='record')
    x = np.array(x0, dtype=float); ws = None; log = []
    for t in range(len(e)):
        try:
            inc, leaves, solves = ctl.feedforward(x, warm_start=ws if warm else None)
        except RuntimeError:
            log.append(dict(failed=True)); break
        if inc is None:
            log.append(dict(cost=np.inf, solves=solves)); break
        u0 = inc.primal['u'][0]
        ws = ctl.construct_warm_start(leaves, x, u0[:ctl.nuc], u0[ctl.nuc:], e[t])
        log.append(dict(cost=inc.primal['objective'], solves=solves, u0=u0.copy(), ub=inc.primal['u'][:, ctl.nuc:].copy(),
                        cover=len(ws), x=x.copy()))
        x = inc.primal['x'][1] + e[t]
    return log
