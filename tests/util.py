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
            rows = np.nonzero(y0)[0]
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
