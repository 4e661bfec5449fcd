"""Hybrid MPC controller with the reference's public surface (controller.py:13-843) on top of the
CUDA kernels.

Drop-in seams kept (SURVEY.md section 8b):
  * ``HybridModelPredictiveController(mld, T, objective, terminal_set)``
  * ``feedforward(x0, gurobi_params={}, search_rule=best_first, branch_rule=branch_in_time, tol=0.,
    warm_start=None, printing_period=3., draw_label=None) -> (PrimalSolution|None, leaves, n_qp, solver_time)``
  * ``construct_warm_start(leaves, x0, uc0, ub0, e0) -> (nodes, t_runtime, t_interstep)``
  * the per-node seam ``_solve_subproblem(identifier, x0) -> (SubproblemSolution, solve_time)``
Errors follow the reference: ValueError on inconsistent sizes; an infeasible node is not an error
(``primal.objective = inf``, Farkas multipliers in ``dual``).

Every QP relaxation is solved on the GPU (kernel K1 through the C ABI); host code here is the
reference's Python control flow.  The all-on-device batched search is ``feedforward_batch``.
"""
import numpy as np
from time import time

from .branch_and_bound import Node, branch_and_bound, best_first, depth_first, breadth_first  # noqa: F401
from .subproblem_solution import SubproblemSolution, PrimalSolution, DualSolution
from .problem import ProblemData
from .bounded_qp import BoundedQP


def _is_prefix(identifier, nub):
    """True iff the identifier pins exactly the first len(identifier) binaries in chronological order."""
    return all((q // nub, q % nub) in identifier for q in range(len(identifier)))


def branch_in_time(identifier, nub):
    """controller.py:13-44: fix the binaries in chronological order, children [value 0, value 1]."""
    t = max([k[0] for k in identifier.keys()] + [0])
    index = max([k[1] + 1 for k in identifier.keys() if k[0] == t] + [0])
    if index < nub:
        return [{(t, index): 0.}, {(t, index): 1.}]
    return [{(t + 1, 0): 0.}, {(t + 1, 0): 1.}]


class StaticBranchOrder(object):
    """A `branch_rule` (controller.py:329, 395-429: callable (identifier, nub) -> list of branch dicts) that picks the next
    binary from a FIXED priority order: the first (t, i) of `order` the identifier does not assign, children
    [value 0, value 1].  `branch_in_time` is the chronological order.  Rules of this family run in the device-side
    search (wshmpc_set_branch_order); any other callable runs the host loop."""

    def __init__(self, order):
        self.order = [tuple(k) for k in order]
        if len(set(self.order)) != len(self.order):
            raise ValueError('a branching order lists every binary once')

    def __call__(self, identifier, nub):
        for k in self.order:
            if k not in identifier:
                return [{k: 0.}, {k: 1.}]
        raise ValueError('every binary of the order is assigned')

    def permutation(self, T, nub):
        if sorted(self.order) != [(t, i) for t in range(T) for i in range(nub)]:
            raise ValueError('the branching order must list every binary (t, i), t < T, i < nub, once')
        return np.array([t * nub + i for t, i in self.order], dtype=np.int32)


def branch_in_reverse_time(T, nub):
    """binaries of the LAST time step first"""
    return StaticBranchOrder([(t, i) for t in range(T - 1, -1, -1) for i in range(nub)])


def branch_by_index(T, nub):
    """all time steps of binary 0, then all of binary 1, ..."""
    return StaticBranchOrder([(t, i) for i in range(nub) for t in range(T)])


class HybridModelPredictiveController(object):

    def __init__(self, mld, T, objective, terminal_set, device=0, qp_options=None):
        self.mld = mld
        self.T = T
        self.Q, self.R, self.Q_T = [np.asarray(M, dtype=float) for M in objective]
        # terminal constraint folded into the stage rows of time T-1 (controller.py:81-87)
        if terminal_set is None:
            terminal_set = [np.empty((0, self.mld.nx)), np.empty(0)]
        self.F_Tm1 = np.vstack((mld.F, terminal_set[0].dot(mld.A)))
        self.G_Tm1 = np.vstack((mld.G, terminal_set[0].dot(mld.B)))
        self.h_Tm1 = np.concatenate((mld.h, terminal_set[1]))
        self._check_input_sizes()
        # warm start construction (controller.py:94-97)
        self._update = {'mu': self._update_mu(), 'rho': np.linalg.pinv(self.Q.T).dot(self.Q_T.T)}
        # problem compiler (replaces _build_mip, controller.py:119-184)
        self.problem = ProblemData.from_controller_data(
            mld, T, [self.Q, self.R, self.Q_T], self.F_Tm1, self.G_Tm1, self.h_Tm1,
            self._update['mu'], self._update['rho'], **(qp_options or {}))
        self.device = device
        self._handle = None
        self._retired = []           # smaller handles handed out earlier stay valid for whoever holds them
        self._n_slots = 1
        self.device_search = True
        self.max_solves = 4096
        # the QP seam (controller.py:90, _build_mip :119-184)
        self.qp = self._build_mip()

    def _build_mip(self):
        """controller.py:119-184: the relaxation of the MIQP as a BoundedQP.  The reference builds a Gurobi model row by
        row; here the model is the device-resident shared operator compiled by problem.py and the BoundedQP object is its
        named-family front end (same families, same order)."""
        return BoundedQP(self.problem, self.handle)

    # -- construction ---------------------------------------------------------------------------
    def _check_input_sizes(self):
        """controller.py:99-117."""
        if self.Q.shape[1] != self.mld.nx:
            raise ValueError('Matrix Q has wrong number of columns.')
        if self.R.shape[1] != self.mld.nu:
            raise ValueError('Matrix R has wrong number of columns.')
        if self.Q_T.shape[1] != self.mld.nx:
            raise ValueError('Matrix Q_T has wrong number of columns.')
        if self.F_Tm1.shape[0] != self.h_Tm1.size:
            raise ValueError('Terminal-set matrices have wrong number of rows.')
        if self.G_Tm1.shape[0] != self.h_Tm1.size:
            raise ValueError('Terminal-set matrices have wrong number of rows.')

    def _update_mu_device(self):
        """controller.py:186-227 as ONE batched launch (wshmpc_lp_batch, SURVEY.md 8f-2): all h_Tm1.size LPs share the
        matrix [F G]' and the cost h and differ in the right-hand side.  Returns M (same optimal values h.M[:, i] as
        `_update_mu`; an LP with several optimal vertices may return another one of them)."""
        from .capi import lp_batch
        mld = self.mld
        E = np.vstack((mld.F.T, mld.G.T))
        R = np.hstack((self.F_Tm1, self.G_Tm1))
        out = lp_batch(E, mld.h, R, device=self.device)
        st = out['status'].cpu().numpy()
        if np.any(st != 2):
            raise ValueError('The conic hull of [F G] does not contain the one of [F_Tm1 G_Tm1].')
        return out['y'].cpu().numpy().T.copy()

    def _update_mu(self):
        """controller.py:186-227: column i of M solves  min h.mu  s.t.  F'mu = F_Tm1[i], G'mu = G_Tm1[i],
        mu >= 0  (host precompute, once per controller; the reference routes these LPs through Gurobi,
        here HiGHS via scipy; `_update_mu_device` is the batched device version)."""
        from scipy.optimize import linprog
        mld = self.mld
        n = mld.h.size
        Aeq = np.vstack((mld.F.T, mld.G.T))
        cols = []
        for i in range(self.h_Tm1.size):
            if i < n and np.array_equal(self.F_Tm1[i], mld.F[i]) and np.array_equal(self.G_Tm1[i], mld.G[i]):
                # the first n rows of [F_Tm1 G_Tm1] ARE the rows of [F G]: unit vector unless the LP finds
                # a strictly cheaper certificate
                ei = np.zeros(n); ei[i] = 1.
                res = linprog(mld.h, A_eq=Aeq, b_eq=np.concatenate((self.F_Tm1[i], self.G_Tm1[i])),
                              bounds=[(0, None)] * n, method='highs')
                if res.status == 0 and res.fun < mld.h[i] - 1e-9 * max(1., abs(mld.h[i])):
                    cols.append(res.x)
                else:
                    cols.append(ei)
                continue
            res = linprog(mld.h, A_eq=Aeq, b_eq=np.concatenate((self.F_Tm1[i], self.G_Tm1[i])),
                          bounds=[(0, None)] * n, method='highs')
            if res.status != 0:
                raise ValueError('The conic hull of [F G] does not contain the one of [F_Tm1 G_Tm1].')
            cols.append(res.x)
        return np.vstack(cols).T if cols else np.zeros((n, 0))

    def terminal_law(self, inputs=None):
        """The linear feedback u = K x of the terminal set, K [nu, nx]: the DARE (LQR) gain of the stage cost on the inputs
        `inputs`, zero for every other input.  inputs: column indices of B (default: the columns of R that are not all
        zero, i.e. the inputs the stage cost penalises).  K solves the DARE on (A, B[:, inputs], Q'Q, R_u'R_u) with
        R_u = R[:, inputs]; when the terminal cost and set were built from that LQR law (a terminal cost Q_T'Q_T = P and
        the maximal admissible set of A + B K), u = K x keeps a state of the terminal set in it."""
        from scipy.linalg import solve_discrete_are
        mld = self.mld
        if inputs is None:
            inputs = np.nonzero(np.any(self.R != 0., axis=0))[0]
        inputs = np.asarray(inputs, dtype=int).ravel()
        if inputs.size == 0:
            raise ValueError('terminal_law: no inputs (R has no nonzero column)')
        Bu, Ru = mld.B[:, inputs], self.R[:, inputs]
        Qc, Rc = self.Q.T.dot(self.Q), Ru.T.dot(Ru)
        P = solve_discrete_are(mld.A, Bu, Qc, Rc)
        K = np.zeros((mld.nu, mld.nx))
        K[inputs] = -np.linalg.inv(Bu.T.dot(P).dot(Bu) + Rc).dot(Bu.T).dot(P).dot(mld.A)
        return K

    # -- device handle --------------------------------------------------------------------------
    @staticmethod
    def _require_gpu():
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError('no CUDA device: the B&B hot path has no CPU fallback')

    def handle(self, n_slots=None):
        from .capi import Handle
        self._require_gpu()
        if n_slots is not None and (self._handle is None or n_slots > self._handle.n_slots):
            if self._handle is not None:
                self._retired.append(self._handle)      # never destroy a handle somebody may still hold
            self._handle = None
            self._n_slots = n_slots
        if self._handle is None:
            self._handle = Handle(self.problem, device=self.device, n_slots=self._n_slots)
        return self._handle

    # -- per-node seam --------------------------------------------------------------------------
    def _get_bound_binaries(self, identifier):
        """controller.py:300-327."""
        ub_lb = np.zeros((self.T, self.mld.nub))
        ub_ub = np.ones((self.T, self.mld.nub))
        for k, v in identifier.items():
            ub_lb[k] = v
            ub_ub[k] = v
        return ub_lb, ub_ub

    def _set_bound_binaries(self, identifier):
        """controller.py:273-298: the node's bounds on the binaries as right-hand sides of the rows nu_lb_t, nu_ub_t."""
        lb, ub = self._get_bound_binaries(identifier)
        for t in range(self.T):
            self.qp.set_constraint_rhs('nu_lb_%d' % t, -lb[t])
            self.qp.set_constraint_rhs('nu_ub_%d' % t, ub[t])

    def _solve_subproblem(self, identifier, x0, active_set=None):
        """controller.py:229-271, same signature: set the right-hand sides, hand the parent's `active_set` to the solver,
        optimise (one K1 launch, bounded_qp.BoundedQP.optimize), wrap the solution."""
        self._set_bound_binaries(identifier)
        self.qp.set_constraint_rhs('lam_0', np.asarray(x0, dtype=float))
        if active_set is not None and self.qp.Params.Method == 1:
            self.qp.set_active_set(active_set)
        self.qp.optimize()
        solution = SubproblemSolution.from_controller(self)
        return solution, self.qp.Runtime

    def _set_gurobi_params(self, gurobi_params):
        """controller.py:778-796.  Only `Method` means something to the CUDA solver (1 = children start from the parent's
        active set, the default; anything else = every node from the empty working set); other keys are recorded."""
        self.qp.resetParams()
        self.qp.setParam('OutputFlag', 0)
        for param, value in gurobi_params.items():
            self.qp.setParam(param, value)

    # -- per-solve seam -------------------------------------------------------------------------
    def feedforward(self, x0, gurobi_params={}, search_rule=best_first, branch_rule=branch_in_time, **kwargs):
        """controller.py:329-393.  With the reference's search rules (best_first, depth_first, breadth_first;
        branch_and_bound.py:501-563), branch_in_time and `device_search=True` the whole search runs in the device-side
        B&B kernel (K3); a user-defined rule, or `device_search=False`, runs the reference's host loop with one K1
        launch per node through `self.qp` -- both visit the same nodes in the same order and return bit-identical
        results."""
        self._set_gurobi_params(gurobi_params)
        self.qp.reset()
        rules = {best_first: 0, depth_first: 1, breadth_first: 2}
        static = branch_rule is branch_in_time or isinstance(branch_rule, StaticBranchOrder)
        if self.device_search and self.qp.Params.Method == 1 and search_rule in rules and static:
            order = None if branch_rule is branch_in_time else branch_rule.permutation(self.T, self.mld.nub)
            return self._feedforward_device(x0, kwargs.get('tol', 0.), kwargs.get('warm_start'), rules[search_rule], order)

        def solver(identifier, cutoff, extra):
            start = extra.active_set if extra is not None else None
            solution, solve_time = self._solve_subproblem(identifier, x0, start)
            return solution.primal.objective, solution.primal.binary_feasible, solve_time, solution

        incumbent, leaves, qp_solves, solver_time = branch_and_bound(
            solver, search_rule, lambda parent: self._brancher(parent, branch_rule), **kwargs)
        primal = None if incumbent is None else incumbent.extra.primal
        return primal, leaves, qp_solves, solver_time

    def _brancher(self, parent, branch_rule):
        """controller.py:395-429: a child's bound is its parent's plus the multiplier of the bound that moves
        (nu_lb for a binary fixed to 1, nu_ub for 0); children share the parent's dual solution and active set."""
        nu = parent.extra.dual.variables
        children = []
        for branch in branch_rule(parent.identifier, self.mld.nub):
            moved = sum(nu['nu_lb' if v == 1 else 'nu_ub'][t][i] for (t, i), v in branch.items())
            children.append(Node({**parent.identifier, **branch}, parent.lb + moved,
                                 SubproblemSolution(None, parent.extra.dual, parent.extra.active_set)))
        return children

    # -- warm start ---------------------------------------------------------------------------------
    def construct_warm_start(self, leaves, x0, uc0, ub0, e0):
        """controller.py:503-564 (with :431-501, :615-721 inside): the leaves of this step's search -> the initial cover
        of the next step's.  Returns (nodes, runtime seconds, inter-step seconds) like the reference; the device kernel
        does both parts at once, so all its time is reported as run time.

        The leaves (any identifiers: device trees hold (assigned mask, values) pairs) are shifted by kernel K2+K4
        (wshmpc_shift_tree): uploaded as a one-instance device tree, shifted, read back.  With `device_search = False`
        the batched host formulation `_shift_records_host` runs instead."""
        leaves = list(leaves)
        if self.device_search:
            return self._construct_warm_start_device(leaves, x0, uc0, ub0, e0)
        tic = time()
        nodes = self._shift_records_host(leaves, np.asarray(x0, float), np.concatenate((uc0, ub0)), np.asarray(e0, float))
        return nodes, time() - tic, 0.

    def _construct_warm_start_device(self, leaves, x0, uc0, ub0, e0):
        import torch
        self._require_gpu()
        h = self.handle()
        nx, nu, T = self.mld.nx, self.mld.nu, self.T
        x0 = np.asarray(x0, dtype=float); u0 = np.concatenate((uc0, ub0)).astype(float)
        tree = self.leaves_to_tree(leaves, max_solves=0)
        new = h.new_tree(1, max(len(leaves), 1) + 2, max(len(leaves), 1) + 1)
        dev = tree.lb.device
        primal = torch.zeros((1, h.layout.primal), dtype=torch.float64, device=dev)
        primal[0, nx:2 * nx] = torch.as_tensor(self.mld.A.dot(x0) + self.mld.B.dot(u0), device=dev)
        primal[0, (T + 1) * nx:(T + 1) * nx + nu] = torch.as_tensor(u0, device=dev)
        cost = torch.zeros(1, dtype=torch.float64, device=dev)
        xd = torch.as_tensor(x0[None], device=dev).contiguous()
        ed = torch.as_tensor(np.asarray(e0, dtype=float)[None], device=dev).contiguous()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        h.shift_tree(xd, ed, tree, cost, primal, new)
        end.record(); end.synchronize()
        return self.tree_to_leaves(new, 0), start.elapsed_time(end) * 1e-3, 0.

    def _shift_records_host(self, leaves, x0, u0, e0):
        """Batched host formulation of the warm start for identifiers that are not chronological prefixes: the same
        record algebra kernel K2+K4 runs (csrc/bnb.cuh shift_instance), on a [leaves x record] matrix.
        Follows controller.py:431-564, 615-721."""
        pd, L = self.problem, self.problem.layout
        T, nx, nu, nub, nuc, nh, nh1, nq, nqT, nr = pd.T, pd.nx, pd.nu, pd.nub, pd.nuc, pd.nh, pd.nh1, pd.nq, pd.nqT, pd.nr
        ub0 = u0[nuc:]
        keep = [l for l in leaves if all(v == ub0[i] for (t, i), v in l.identifier.items() if t == 0)]     # :615-633
        if not keep:
            return []
        D = np.vstack([DualSolution.to_record(pd, L, l.extra.dual.variables) for l in keep])
        obj = np.array([l.extra.dual.objective for l in keep])
        lo = np.zeros((len(keep), nub)); hi = np.ones((len(keep), nub))         # old bounds at t = 0
        for r, l in enumerate(keep):
            for (t, i), v in l.identifier.items():
                if t == 0:
                    lo[r, i] = hi[r, i] = v
        blk = lambda off, width, t0, t1: D[:, off + t0 * width:off + t1 * width]
        S = np.zeros_like(D)                                                     # shifted records (:635-666)
        S[:, L.off_lam:L.off_lam + T * nx] = blk(L.off_lam, nx, 1, T + 1)
        S[:, L.off_nu_lb:L.off_nu_lb + (T - 1) * nub] = blk(L.off_nu_lb, nub, 1, T)
        S[:, L.off_nu_ub:L.off_nu_ub + (T - 1) * nub] = blk(L.off_nu_ub, nub, 1, T)
        S[:, L.off_sigma:L.off_sigma + (T - 1) * nr] = blk(L.off_sigma, nr, 1, T)
        S[:, L.off_mu:L.off_mu + (T - 2) * nh] = blk(L.off_mu, nh, 1, T - 1)
        mu_last = D[:, L.off_mu + (T - 1) * nh:L.off_nu_lb]
        mu_new = mu_last.dot(self._update['mu'].T)
        S[:, L.off_mu + (T - 2) * nh:L.off_mu + (T - 1) * nh] = mu_new
        S[:, L.off_rho:L.off_rho + (T - 1) * nq] = blk(L.off_rho, nq, 1, T)
        rho_T = D[:, L.off_rho + T * nq:L.off_sigma]
        rho_new = rho_T.dot(self._update['rho'].T)
        S[:, L.off_rho + (T - 1) * nq:L.off_rho + T * nq] = rho_new
        # change of the dual objective (:668-721) and the run-time correction pi3 (:541-546)
        Qx0, Ru0 = self.Q.dot(x0), self.R.dot(u0)
        rho_0, sig_0 = blk(L.off_rho, nq, 0, 1), blk(L.off_sigma, nr, 0, 1)
        pi = ((.5 * rho_0 - Qx0) ** 2).sum(1) - Qx0.dot(Qx0) + ((.5 * sig_0 - Ru0) ** 2).sum(1) - Ru0.dot(Ru0)
        pi -= blk(L.off_mu, nh, 0, 1).dot(self.mld.F.dot(x0) + self.mld.G.dot(u0) - self.mld.h)
        pi -= ((lo - ub0) * blk(L.off_nu_lb, nub, 0, 1)).sum(1) + ((ub0 - hi) * blk(L.off_nu_ub, nub, 0, 1)).sum(1)
        pi += .25 * (rho_T ** 2).sum(1) - .25 * (rho_new ** 2).sum(1)
        pi += mu_last.dot(self.h_Tm1) - mu_new.dot(self.mld.h)
        pi -= S[:, L.off_lam:L.off_lam + nx].dot(e0)
        obj = np.maximum(obj + pi, 0.)
        nodes = []
        for r, l in enumerate(keep):
            ident = {(t - 1, i): v for (t, i), v in l.identifier.items() if t > 0}
            dual = DualSolution.from_record(pd, L, S[r], obj[r])
            start = self.qp.active_set_from_dual(dual)
            lb = l.lb
            if not np.isinf(l.lb):
                lb = obj[r]                                                      # :550-551
            elif obj[r] <= 0.:
                lb, dual = 0., None                                              # :555-558 (the ray stays as a START)
            nodes.append(Node(ident, lb, SubproblemSolution(None, dual, start)))
        return nodes

    # -- device-resident batch path (K3, K2 + K4) ----------------------------------------------------
    def _as_device(self, a, shape):
        import torch
        t = torch.as_tensor(np.asarray(a, dtype=float) if not torch.is_tensor(a) else a, dtype=torch.float64,
                            device=torch.device('cuda', self.device)).contiguous()
        assert tuple(t.shape) == tuple(shape), (tuple(t.shape), tuple(shape))
        return t

    def new_tree(self, n_inst, n_roots=1, max_solves=None):
        """Device tree with room for `n_roots` initial leaves and `max_solves` QP solves per instance."""
        ms = self.max_solves if max_solves is None else max_solves
        return self.handle().new_tree(n_inst, n_roots + 2 * ms + 2, n_roots + ms + 1)

    def feedforward_batch(self, x0, warm_start=None, tol=0., max_solves=None, n_slots=None, active=None, trace=False,
                          out=None):
        """Batched feedforward (controller.py:329-393 for many independent initial states at once).
        x0 [N, nx] (numpy or CUDA tensor); warm_start: a device `Tree` (from construct_warm_start_batch)
        or None for the cold root.  Returns (result dict of CUDA tensors, tree); nothing is synchronised."""
        self._require_gpu()
        ms = self.max_solves if max_solves is None else max_solves
        N = x0.shape[0]
        h = self.handle(n_slots if n_slots is not None else max(self._n_slots, min(N, self.default_slots())))
        x0 = self._as_device(x0, (N, self.mld.nx))
        tree = warm_start
        if tree is None:
            tree = self.new_tree(N, 1, ms)
            h.tree_init_root(tree)
        res = h.bnb_solve(x0, tree, tol=tol, max_solves=ms, active=active, out=out, trace=trace)
        res['x0'] = x0
        return res, tree

    def construct_warm_start_batch(self, res, tree, e0=None, new_tree=None, active=None, x_next=None, u0=None,
                                   max_solves=None):
        """Batched construct_warm_start (controller.py:503-564) + plant update x <- x_1 + e0.
        Returns (new_tree, x_next [N, nx], u0 [N, nu])."""
        import torch
        h = self.handle()
        N = tree.n_inst
        dev = torch.device('cuda', self.device)
        if new_tree is None:
            ms = self.max_solves if max_solves is None else max_solves
            new_tree = h.new_tree(N, tree.cap_nodes + 2 * ms + 2, tree.cap_nodes + ms + 1)
        if e0 is not None:
            e0 = self._as_device(e0, (N, self.mld.nx))
        if x_next is None:
            x_next = torch.empty((N, self.mld.nx), dtype=torch.float64, device=dev)
        if u0 is None:
            u0 = torch.empty((N, self.mld.nu), dtype=torch.float64, device=dev)
        h.shift_tree(res['x0'], e0, tree, res['cost'], res['primal'], new_tree, active=active, x_next=x_next, u0=u0)
        return new_tree, x_next, u0

    def default_slots(self):
        """Solver states resident at once: SMs (148 on a B200) x solver CTAs per SM of the library build."""
        import torch
        from .capi import load_library
        self.handle()                # the lanes per CTA are fixed when a handle for THIS problem is created
        return torch.cuda.get_device_properties(self.device).multi_processor_count * int(load_library().wshmpc_ctas_per_sm())

    # -- tree <-> reference Node lists ---------------------------------------------------------------
    def tree_to_leaves(self, tree, inst=0):
        """The reference's `leaves` list (branch_and_bound.py:497) of one instance of a device tree."""
        h = self.handle()
        T, nub = self.T, self.mld.nub
        nn = int(tree.n_nodes[inst])
        depth = tree.depth[inst, :nn].cpu().numpy(); alive = tree.alive[inst, :nn].cpu().numpy()
        rec = tree.rec[inst, :nn].cpu().numpy(); lb = tree.lb[inst, :nn].cpu().numpy()
        bits = tree.bits[inst, :nn].cpu().numpy().view(np.uint32)
        mask = tree.mask[inst, :nn].cpu().numpy().view(np.uint32)
        nr = int(tree.n_recs[inst])
        duals = tree.rec_dual[inst, :nr].cpu().numpy(); dobj = tree.rec_dobj[inst, :nr].cpu().numpy()
        cache = {}

        def record(r):                  # children alias the parent's dual object and active set (controller.py:426)
            if r not in cache:
                cache[r] = (DualSolution.from_record(self.problem, h.layout, duals[r], dobj[r]),
                            self.qp.active_set_from_record(duals[r]))
            return cache[r]
        leaves = []
        for j in range(nn):
            if not alive[j]:
                continue
            ident = self._identifier(bits[j], mask[j])
            r = int(rec[j])
            if r >= 0:
                extra = SubproblemSolution(None, record(r)[0], record(r)[1])
            elif r <= -2:               # dual = None (controller.py:555-558); the shifted ray survives as the START of the solve
                extra = SubproblemSolution(None, None, record(-2 - r)[1])
            else:
                extra = SubproblemSolution(None, None) if depth[j] or np.isfinite(lb[j]) else None
            node = Node(ident, float(lb[j]), extra)
            node.index = j
            leaves.append(node)
        return leaves

    def _identifier(self, bits_j, mask_j):
        """(assigned mask, values) words of a device node -> the reference's identifier dict {(t, i): 0. | 1.}"""
        nub = self.mld.nub
        out = {}
        for q in range(self.problem.nb):
            if (int(mask_j[q >> 5]) >> (q & 31)) & 1:
                out[(q // nub, q % nub)] = float((int(bits_j[q >> 5]) >> (q & 31)) & 1)
        return out

    def leaves_to_tree(self, leaves, max_solves=None):
        """Uploads a reference-style warm start (list of Node with prefix identifiers) as a device tree."""
        import torch
        h = self.handle()
        ms = self.max_solves if max_solves is None else max_solves
        n0 = len(leaves)
        tree = self.new_tree(1, n0, ms)
        nub = self.mld.nub
        depth = np.zeros(n0, np.int32); rec = np.full(n0, -1, np.int32); lb = np.zeros(n0)
        bits = np.zeros((n0, tree.words), np.uint32); mask = np.zeros((n0, tree.words), np.uint32)
        recs, dobj, seen = [], [], {}
        L, n = h.layout, self.problem.n
        for j, l in enumerate(leaves):
            depth[j] = len(l.identifier)
            for (t, i), v in l.identifier.items():
                q = t * nub + i
                mask[j, q >> 5] |= np.uint32(1 << (q & 31))
                if v:
                    bits[j, q >> 5] |= np.uint32(1 << (q & 31))
            lb[j] = l.lb
            dual = None if l.extra is None else l.extra.dual
            start = None if l.extra is None else l.extra.active_set
            key = id(dual) if dual is not None else (id(start) if start is not None else None)
            if key is None:
                continue
            if key not in seen:
                seen[key] = len(recs)
                rec_j = np.zeros(L.rec_stride)
                if dual is not None:
                    rec_j[:L.dual] = DualSolution.to_record(self.problem, L, dual.variables)
                    dobj.append(dual.objective)
                else:                   # only the start survives: rebuild the multiplier part of the record from it
                    y = self.qp._signed_multipliers(np.asarray(start['c'], dtype=float))
                    rec_j[L.off_mu:L.off_nu_lb] = y[:self.problem.mc]
                    rec_j[L.off_nu_lb:L.off_nu_ub] = np.maximum(-y[self.problem.mc:], 0.)
                    rec_j[L.off_nu_ub:L.off_rho] = np.maximum(y[self.problem.mc:], 0.)
                    dobj.append(0.)
                if start is not None:
                    rec_j[L.dual:L.dual + n] = np.asarray(start['v'], dtype=float)[:n]
                recs.append(rec_j)
            rec[j] = seen[key] if dual is not None else -2 - seen[key]
        dev = tree.lb.device
        tree.n_nodes[0] = n0; tree.n_recs[0] = len(recs)
        tree.depth[0, :n0] = torch.as_tensor(depth, device=dev); tree.alive[0, :n0] = 1
        tree.rec[0, :n0] = torch.as_tensor(rec, device=dev); tree.lb[0, :n0] = torch.as_tensor(lb, device=dev)
        tree.bits[0, :n0] = torch.as_tensor(bits.view(np.int32), device=dev)
        tree.mask[0, :n0] = torch.as_tensor(mask.view(np.int32), device=dev)
        if recs:
            tree.rec_dual[0, :len(recs)] = torch.as_tensor(np.vstack(recs), device=dev)
            tree.rec_dobj[0, :len(recs)] = torch.as_tensor(np.array(dobj), device=dev)
        return tree

    def _feedforward_device(self, x0, tol, warm_start, rule=0, order=None):
        import torch
        self._require_gpu()
        tree = None if warm_start is None else self.leaves_to_tree(warm_start)
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        self.handle().set_search_rule(rule)
        self.handle().set_branch_order(order)
        try:
            res, tree = self.feedforward_batch(np.asarray(x0, dtype=float)[None], warm_start=tree, tol=tol, n_slots=1)
        finally:
            self.handle().set_search_rule(0)
            self.handle().set_branch_order(None)
        end.record()
        end.synchronize()
        solver_time = start.elapsed_time(end) * 1e-3
        status = int(res['status'][0])
        if status >= 2:
            raise RuntimeError('device branch and bound failed with status %d (2 = capacity, 3 = QP iteration limit)' % status)
        leaves = self.tree_to_leaves(tree, 0)
        if warm_start is not None:          # the reference mutates the list it is given (branch_and_bound.py:432)
            warm_start[:] = leaves
            leaves = warm_start
        self.last_batch = (res, tree)
        n_qp = int(res['n_solves'][0])
        if status == 1:
            return None, leaves, n_qp, solver_time
        primal = PrimalSolution.from_record(self.problem, res['primal'][0].cpu().numpy(), float(res['cost'][0]), True, True)
        return primal, leaves, n_qp, solver_time

    # -- comparator: a conventional MIQP branch and bound (SURVEY.md 8f-1) ----------------------------------
    def feedforward_miqp(self, x0, gurobi_params={}, ub_guess=None, tol=0.):
        """Stand-in for `feedforward_gurobi` (controller.py:723-776; the paper's third curve, "Gurobi fair": no presolve, no
        heuristics, one thread -- statistical_analysis.py:151-154) that needs no Gurobi: a textbook MIQP branch and bound
        through the same QP seam (`self.qp`, one K1 launch per node) that knows NOTHING about the time structure --
        best-bound node selection, branching on the MOST FRACTIONAL binary of the relaxation wherever it sits in the
        horizon, a node is integral when its relaxation is (not when every binary is pinned), children start from their
        parent's active set like a dual-simplex B&B, bounds are the relaxation values only (no dual-bound inheritance, no
        warm start across time steps).  `ub_guess` [T, nub] is a MIP start (controller.py:798-818).
        Returns (variables {'x', 'uc', 'ub'} stacked over time, objective, nodes, solver seconds) like the reference."""
        self._set_gurobi_params(gurobi_params)
        self.qp.reset()
        T, nub = self.T, self.mld.nub
        solver_time = 0.
        nodes = 0
        best, best_sol = np.inf, None

        def relax(identifier, start):
            nonlocal solver_time, nodes
            sol, dt = self._solve_subproblem(identifier, x0, start)
            solver_time += dt; nodes += 1
            return sol

        if ub_guess is not None:                 # MIP start: the guess, fully pinned
            guess = {(t, i): float(round(ub_guess[t][i])) for t in range(T) for i in range(nub)}
            sol = relax(guess, None)
            if np.isfinite(sol.primal.objective):
                best, best_sol = sol.primal.objective, sol
        frontier = [({}, -np.inf, None)]         # (identifier, bound of the parent, parent's active set)
        while frontier:
            k = int(np.argmin([f[1] for f in frontier]))
            identifier, bound, start = frontier.pop(k)
            if bound >= best - tol:
                continue
            sol = relax(identifier, start)
            cost = sol.primal.objective
            if cost >= best - tol:
                continue
            ub = np.array(sol.primal.variables['ub'])
            frac = np.abs(ub - np.round(ub))
            for key in identifier:               # pinned binaries are integral by construction
                frac[key] = 0.
            if frac.max() <= 1e-9:
                best, best_sol = cost, sol
                continue
            t, i = np.unravel_index(int(np.argmax(frac)), frac.shape)
            for v in (0., 1.):
                frontier.append(({**identifier, (int(t), int(i)): v}, cost, sol.active_set))
        self.qp.reset()
        if best_sol is None:
            return None, np.inf, nodes, solver_time
        variables = {k: np.vstack(best_sol.primal.variables[k]) for k in ('x', 'uc', 'ub')}
        variables['ub'] = np.round(variables['ub'])
        return variables, best, nodes, solver_time

    feedforward_gurobi = feedforward_miqp       # the reference's name for the comparator leg (there is no Gurobi underneath)

    def feedforward_miqp_batch(self, x0, ub_guess=None, tol=0., max_solves=None, n_slots=None, active=None, trace=False):
        """`feedforward_miqp` for many independent initial states in ONE launch of the device-side branch and bound under the
        conventional node rule (wshmpc_set_node_rule 1): most fractional binary, integral relaxations are incumbents, bounds
        are relaxation values only; candidate selection is the handle's search rule (best_first by default).
        x0 [N, nx]; ub_guess: MIP start [N, T, nub], or [T, nub] for every instance, or None.
        Returns (result dict of CUDA tensors, tree) like feedforward_batch; nothing is synchronised.  With trace=True,
        res['trace'][k, 2 s] is the node solved s-th; the tree keeps each solved node's identifier and relaxation cost (lb)."""
        self._require_gpu()
        ms = self.max_solves if max_solves is None else max_solves
        N = x0.shape[0]
        T, nub = self.T, self.mld.nub
        h = self.handle(n_slots if n_slots is not None else max(self._n_slots, min(N, self.default_slots())))
        x0 = self._as_device(x0, (N, self.mld.nx))
        tree = self.new_tree(N, 2, ms)
        if ub_guess is None:
            h.tree_init_root(tree)
        else:
            g = np.asarray(ub_guess, dtype=float) if not hasattr(ub_guess, 'is_cuda') else ub_guess
            g = self._as_device(g, tuple(g.shape))
            if g.dim() == 2:
                g = g[None].expand(N, T, nub)
            if tuple(g.shape) != (N, T, nub):
                raise ValueError('ub_guess must be [N, T, nub] or [T, nub]')
            h.tree_init_guess(tree, g.reshape(N, T * nub).contiguous())
        h.set_node_rule(1)
        try:
            res = h.bnb_solve(x0, tree, tol=tol, max_solves=ms, active=active, trace=trace)
        finally:
            h.set_node_rule(0)              # launch parameters are copied at the launch: the rule can go back at once
        res['x0'] = x0
        return res, tree

    def feedforward_miqp_device(self, x0, gurobi_params={}, ub_guess=None, tol=0.):
        """`feedforward_miqp` (same arguments, same result: variables {'x', 'uc', 'ub'} stacked over time with 'ub' rounded,
        objective, nodes, solver seconds) as one instance of `feedforward_miqp_batch`: the whole search in one launch, no host
        round trip per node.  It visits the same nodes in the same order as the host loop.  Children start from their
        parent's record, which is what `Method` = 1 (the default) means; any other `Method` solves every node from the empty
        working set, and that runs the host loop."""
        import torch
        self._set_gurobi_params(gurobi_params)
        if self.qp.Params.Method != 1:
            return self.feedforward_miqp(x0, gurobi_params, ub_guess=ub_guess, tol=tol)
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        guess = None if ub_guess is None else np.asarray(ub_guess, dtype=float)[None]
        res, _ = self.feedforward_miqp_batch(np.asarray(x0, dtype=float)[None], ub_guess=guess, tol=tol, n_slots=1)
        end.record()
        end.synchronize()
        status, nodes = int(res['status'][0]), int(res['n_solves'][0])
        if status >= 2:
            raise RuntimeError('device branch and bound failed with status %d (2 = capacity, 3 = QP iteration limit)' % status)
        seconds = start.elapsed_time(end) * 1e-3
        if status == 1:
            return None, np.inf, nodes, seconds
        T, nx, nu, nuc = self.T, self.mld.nx, self.mld.nu, self.problem.nuc
        rec = res['primal'][0].cpu().numpy()
        U = rec[(T + 1) * nx:].reshape(T, nu)
        variables = {'x': rec[:(T + 1) * nx].reshape(T + 1, nx).copy(), 'uc': U[:, :nuc].copy(), 'ub': np.round(U[:, nuc:])}
        return variables, float(res['cost'][0]), nodes, seconds

    def shift_binary_solution(self, ub):
        """controller.py:811-812."""
        return np.vstack((ub[1:], np.zeros(self.mld.nub)))
