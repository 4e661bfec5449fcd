"""ctypes binding of the C ABI declared in include/wshmpc.h (libwshmpc.so, built in-tree by
``__graft_entry__.build()``).  PyTorch is used only to own device memory and streams.

There is NO CPU fallback: a missing library or a missing GPU raises.
"""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('WSHMPC_LIB') or os.path.join(_HERE, 'libwshmpc.so')   # WSHMPC_LIB: experiment builds (tools/)
_lib = None


class _Problem(C.Structure):
    _fields_ = ([(k, C.c_int) for k in ('nx', 'nu', 'nub', 'T', 'nh', 'nh1', 'nq', 'nqT', 'nr', 'n', 'm', 'mc', 'nb', 'ns')]
                + [(k, C.c_void_p) for k in ('A', 'B', 'F', 'G', 'h', 'F_Tm1', 'G_Tm1', 'h_Tm1', 'Q', 'R', 'Q_T',
                                             'M_mu', 'M_rho', 'Mh', 'Wf', 'nrm', 'vscale', 'Eh', 'hh', 'Rinv', 'Kx',
                                             'Zmap', 'bin_idx', 'Linv')]
                + [('n_elim', C.c_int)]
                + [(k, C.c_double) for k in ('eps', 'tol_p', 'tol_d', 'tol_sing', 'tol_ray', 'prox_tol')]
                + [(k, C.c_int) for k in ('max_iter', 'max_prox')])


class Layout(C.Structure):
    _fields_ = [(k, C.c_int) for k in ('primal', 'dual', 'off_lam', 'off_mu', 'off_nu_lb', 'off_nu_ub',
                                       'off_rho', 'off_sigma', 'rec_stride')]


def load_library():
    """Loads libwshmpc.so; raises (never falls back) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError('CUDA library %s not built: run `python -c "import __graft_entry__ as g; g.build()"` '
                               '(there is no CPU fallback for the hot path)' % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        lib.wshmpc_last_error.restype = C.c_char_p
        for name in EXPORTS:
            getattr(lib, name)           # AttributeError if the ABI is incomplete
        _lib = lib
    return _lib


EXPORTS = ('wshmpc_last_error', 'wshmpc_ctas_per_sm', 'wshmpc_set_search_rule', 'wshmpc_set_branch_order', 'wshmpc_set_node_rule', 'wshmpc_create', 'wshmpc_destroy', 'wshmpc_get_layout', 'wshmpc_solve_nodes',
           'wshmpc_tree_init_root', 'wshmpc_tree_init_guess', 'wshmpc_bnb_solve', 'wshmpc_shift_tree', 'wshmpc_closed_loop', 'wshmpc_mailbox_create', 'wshmpc_mailbox_destroy', 'wshmpc_lp_batch',
           'wshmpc_plant_step', 'wshmpc_closed_loop_plant', 'wshmpc_closed_loop_fallback', 'wshmpc_fallback_step')


class _Mailbox(C.Structure):
    _fields_ = ([(k, C.c_int) for k in ('n_inst', 'nx', 'nu')]
                + [(k, C.c_void_p) for k in ('out_step', 'out_u0', 'out_x1', 'out_cost', 'out_status', 'in_step', 'in_x', 'in_e', 'stop')]
                + [('timeout_ms', C.c_int), ('priv', C.c_void_p)])


class Mailbox(object):
    """Host mailbox of the fused closed loop (wshmpc_mailbox in include/wshmpc.h): numpy views of the pinned, mapped host
    arrays the running kernel publishes steps to and reads the host's answers from."""

    def __init__(self, handle, n_inst):
        self._handle, self.c = handle, _Mailbox()
        _check(handle.lib.wshmpc_mailbox_create(handle._h, int(n_inst), C.byref(self.c)))
        nx, nu = self.c.nx, self.c.nu

        def view(ptr, ctype, shape):
            n = int(np.prod(shape))
            return np.ctypeslib.as_array((ctype * n).from_address(ptr)).reshape(shape)
        self.out_step = view(self.c.out_step, C.c_int, (n_inst,))
        self.out_u0 = view(self.c.out_u0, C.c_double, (n_inst, nu))
        self.out_x1 = view(self.c.out_x1, C.c_double, (n_inst, nx))
        self.out_cost = view(self.c.out_cost, C.c_double, (n_inst,))
        self.out_status = view(self.c.out_status, C.c_int, (n_inst,))
        self.in_step = view(self.c.in_step, C.c_int, (n_inst,))
        self.in_x = view(self.c.in_x, C.c_double, (n_inst, nx))
        self.in_e = view(self.c.in_e, C.c_double, (n_inst, nx))
        self.stop = view(self.c.stop, C.c_int, (1,))

    def clear(self):
        self.out_step[:] = 0; self.in_step[:] = 0; self.stop[0] = 0

    def close(self):
        if self.c.priv:
            for k in ('out_step', 'out_u0', 'out_x1', 'out_cost', 'out_status', 'in_step', 'in_x', 'in_e', 'stop'):
                setattr(self, k, None)
            self._handle.lib.wshmpc_mailbox_destroy(self._handle._h, C.byref(self.c))


class _Loop(C.Structure):
    _fields_ = ([(k, C.c_int) for k in ('n_steps', 'warm', 'fresh', 'par')]
                + [(k, C.c_void_p) for k in ('d_queue', 'd_step_of', 'd_x', 'd_e', 'd_active', 'd_log_cost', 'd_log_u0',
                                             'd_log_solves', 'd_log_status', 'mailbox')])


class _Plant(C.Structure):
    _fields_ = [('kind', C.c_int), ('n_sets', C.c_int), ('d_params', C.c_void_p), ('dt', C.c_double), ('n_sub', C.c_int),
                ('fc_index', C.c_int), ('d_log_x', C.c_void_p)]


def _plant_struct(plant, log_x=None):
    """wshmpc_plant of a plants.DevicePlant (the cart-pole between soft walls, kind 1)"""
    c = _Plant()
    c.kind, c.n_sets, c.d_params = 1, plant.n_sets, plant.params.data_ptr()
    c.dt, c.n_sub, c.fc_index = plant.dt, plant.n_sub, plant.fc_index
    c.d_log_x = log_x.data_ptr() if log_x is not None else None
    return c


class _Fallback(C.Structure):
    _fields_ = [('max_hold', C.c_int), ('d_plan', C.c_void_p), ('d_age', C.c_void_p), ('d_app_cost', C.c_void_p),
                ('d_app_primal', C.c_void_p), ('d_hold', C.c_void_p), ('max_law', C.c_int), ('d_law_K', C.c_void_p),
                ('d_law_n', C.c_void_p)]


def _fallback_struct(fb, hold):
    """wshmpc_fallback of a dict(max_hold, plan, age, app_cost, app_primal) of CUDA tensors, with the hold log `hold`; the
    terminal law comes from the optional keys max_law, law_K and law_n (without them: max_law = 0 and null pointers)"""
    c = _Fallback()
    c.max_hold = int(fb['max_hold'])
    for k in ('plan', 'age', 'app_cost', 'app_primal'):
        setattr(c, 'd_' + k, fb[k].data_ptr() if fb[k] is not None else None)
    c.d_hold = hold.data_ptr() if hold is not None else None
    c.max_law = int(fb.get('max_law', 0))
    for k in ('law_K', 'law_n'):
        setattr(c, 'd_' + k, fb[k].data_ptr() if fb.get(k) is not None else None)
    return c


class _Tree(C.Structure):
    _fields_ = ([(k, C.c_int) for k in ('cap_nodes', 'cap_recs', 'words')]
                + [(k, C.c_void_p) for k in ('n_nodes', 'n_recs', 'depth', 'alive', 'rec', 'bits', 'mask', 'lb', 'rec_dobj',
                                             'rec_dual')])


class Tree(object):
    """Device-resident B&B trees of `n_inst` independent MPC instances (wshmpc_tree in include/wshmpc.h).
    torch owns the memory; the kernels read and write it in place."""

    def __init__(self, n_inst, nb, n_dual, cap_nodes, cap_recs, device):
        """n_dual = layout.rec_stride: doubles per dual record (reference duals followed by the proximal centre)."""
        import torch
        self.n_inst, self.nb, self.n_dual = n_inst, nb, n_dual
        self.cap_nodes, self.cap_recs, self.words = cap_nodes, cap_recs, (nb + 31) // 32
        i32 = dict(dtype=torch.int32, device=device)
        f64 = dict(dtype=torch.float64, device=device)
        self.n_nodes = torch.zeros(n_inst, **i32)
        self.n_recs = torch.zeros(n_inst, **i32)
        self.depth = torch.zeros((n_inst, cap_nodes), **i32)
        self.alive = torch.zeros((n_inst, cap_nodes), **i32)
        self.rec = torch.zeros((n_inst, cap_nodes), **i32)
        self.bits = torch.zeros((n_inst, cap_nodes, self.words), **i32)     # uint32 payload: values of the assigned binaries
        self.mask = torch.zeros((n_inst, cap_nodes, self.words), **i32)     # uint32 payload: which binaries are assigned
        self.lb = torch.zeros((n_inst, cap_nodes), **f64)
        self.rec_dobj = torch.zeros((n_inst, cap_recs), **f64)
        self.rec_dual = torch.empty((n_inst, cap_recs, n_dual), **f64)
        c = _Tree()
        c.cap_nodes, c.cap_recs, c.words = cap_nodes, cap_recs, self.words
        for k in ('n_nodes', 'n_recs', 'depth', 'alive', 'rec', 'bits', 'mask', 'lb', 'rec_dobj', 'rec_dual'):
            setattr(c, k, getattr(self, k).data_ptr())
        self.c = c

    def nbytes(self):
        return sum(getattr(self, k).numel() * getattr(self, k).element_size()
                   for k in ('n_nodes', 'n_recs', 'depth', 'alive', 'rec', 'bits', 'mask', 'lb', 'rec_dobj', 'rec_dual'))


def _check(rc):
    if rc != 0:
        raise RuntimeError('wshmpc error %d: %s' % (rc, load_library().wshmpc_last_error().decode()))


class Handle(object):
    """Owns one wshmpc_handle (one GPU, one stream, `n_slots` solver states)."""

    def __init__(self, pd, device=0, n_slots=1, stream=None):
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError('no CUDA device: the B&B hot path has no CPU fallback')
        self.lib = load_library()
        self.pd = pd
        self.device = device
        self.torch_device = torch.device('cuda', device)
        self.n_slots = n_slots
        p = _Problem()
        for k in ('nx', 'nu', 'nub', 'T', 'nh', 'nh1', 'nq', 'nqT', 'nr', 'n', 'm', 'mc', 'nb', 'ns', 'n_elim', 'max_iter', 'max_prox',
                  'eps', 'tol_p', 'tol_d', 'tol_sing', 'tol_ray', 'prox_tol'):
            setattr(p, k, getattr(pd, k))
        for k in ('A', 'B', 'F', 'G', 'h', 'F_Tm1', 'G_Tm1', 'h_Tm1', 'Q', 'R', 'Q_T', 'M_mu', 'M_rho', 'Mh', 'Wf', 'nrm',
                  'vscale', 'Eh', 'hh', 'Rinv', 'Kx', 'Zmap', 'bin_idx', 'Linv'):
            a = getattr(pd, k)
            assert a.flags['C_CONTIGUOUS']
            setattr(p, k, a.ctypes.data)
        self._h = C.c_void_p()
        self.stream = stream
        sptr = C.c_void_p(stream.cuda_stream if stream is not None else 0)
        _check(self.lib.wshmpc_create(C.byref(p), device, n_slots, sptr, C.byref(self._h)))
        self.layout = Layout()
        _check(self.lib.wshmpc_get_layout(self._h, C.byref(self.layout)))

    def set_search_rule(self, rule):
        """0 best_first, 1 depth_first, 2 breadth_first (branch_and_bound.py:501-563) for the device-side B&B."""
        _check(self.lib.wshmpc_set_search_rule(self._h, int(rule)))

    def set_node_rule(self, rule):
        """0 the structured search (default), 1 the conventional MIQP branch and bound of feedforward_miqp (most fractional
        binary, controller.py:530-582), 2 rule 1 with a MIP start at every step of the fused closed loop (wshmpc_set_node_rule)."""
        _check(self.lib.wshmpc_set_node_rule(self._h, int(rule)))

    def set_branch_order(self, order):
        """Static branching order of the device-side B&B: permutation of the binaries j = t * nub + i, or None for the
        chronological order of branch_in_time (wshmpc_set_branch_order)."""
        if order is None:
            _check(self.lib.wshmpc_set_branch_order(self._h, None))
        else:
            a = np.ascontiguousarray(order, dtype=np.int32)
            _check(self.lib.wshmpc_set_branch_order(self._h, a.ctypes.data_as(C.c_void_p)))

    def close(self):
        if self._h:
            self.lib.wshmpc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- K1 -------------------------------------------------------------------------------------
    def solve_nodes(self, x0, lb, ub, slot=None, hot=None, y0=None, yc0=None):
        """x0 [N, nx], lb/ub [N, nb] (torch CUDA fp64 or numpy).  hot: 0 empty working set, 1 the slot's previous
        node, 2 start from the signed multipliers y0 [N, m] (and proximal centre yc0 [N, n]).
        Returns dict of torch CUDA tensors."""
        import torch
        dev = self.torch_device
        t = lambda a, dt: torch.as_tensor(np.asarray(a) if not torch.is_tensor(a) else a, dtype=dt, device=dev).contiguous()
        x0, lb, ub = t(x0, torch.float64), t(lb, torch.float64), t(ub, torch.float64)
        N = x0.shape[0]
        assert x0.shape == (N, self.pd.nx) and lb.shape == (N, self.pd.nb) and ub.shape == (N, self.pd.nb)
        slot = torch.arange(N, dtype=torch.int32, device=dev) % self.n_slots if slot is None else t(slot, torch.int32)
        hot = torch.zeros(N, dtype=torch.int32, device=dev) if hot is None else t(hot, torch.int32)
        if int(slot.max()) >= self.n_slots:
            raise ValueError('slot index out of range')
        out = dict(status=torch.zeros(N, dtype=torch.int32, device=dev),
                   cost=torch.zeros(N, dtype=torch.float64, device=dev),
                   dobj=torch.zeros(N, dtype=torch.float64, device=dev),
                   iters=torch.zeros(N, dtype=torch.int32, device=dev),
                   primal=torch.zeros((N, self.layout.primal), dtype=torch.float64, device=dev),
                   dual=torch.zeros((N, self.layout.dual), dtype=torch.float64, device=dev),
                   yc=torch.zeros((N, self.pd.n), dtype=torch.float64, device=dev))
        if y0 is not None:
            y0 = t(y0, torch.float64); assert y0.shape == (N, self.pd.m)
        if yc0 is not None:
            yc0 = t(yc0, torch.float64); assert yc0.shape == (N, self.pd.n)
        P = lambda a: C.c_void_p(a.data_ptr()) if a is not None else None
        _check(self.lib.wshmpc_solve_nodes(self._h, N, P(x0), P(lb), P(ub), P(slot), P(hot), P(y0), P(yc0), P(out['status']),
                                           P(out['cost']), P(out['dobj']), P(out['iters']), P(out['primal']),
                                           P(out['dual']), P(out['yc'])))
        return out

    # -- trees / K3 / K2+K4 ---------------------------------------------------------------------
    def new_tree(self, n_inst, cap_nodes, cap_recs):
        return Tree(n_inst, self.pd.nb, self.layout.rec_stride, cap_nodes, cap_recs, self.torch_device)

    def tree_init_root(self, tree):
        _check(self.lib.wshmpc_tree_init_root(self._h, tree.n_inst, C.byref(tree.c)))

    def tree_init_guess(self, tree, guess, has=None):
        """MIP start (wshmpc_tree_init_guess): instance k gets [guess, root], or the root alone where has[k] == 0.
        guess [n_inst, nb] CUDA fp64 tensor of binary values (rounded on the device); has [n_inst] CUDA int32 tensor or None."""
        import torch
        N = tree.n_inst
        assert guess.is_cuda and guess.dtype == torch.float64 and guess.is_contiguous() and tuple(guess.shape) == (N, self.pd.nb)
        if has is not None:
            assert has.is_cuda and has.dtype == torch.int32 and has.is_contiguous() and tuple(has.shape) == (N,)
        P = lambda a: C.c_void_p(a.data_ptr()) if a is not None else None
        _check(self.lib.wshmpc_tree_init_guess(self._h, N, C.byref(tree.c), P(guess), P(has)))

    def bnb_solve(self, x0, tree, tol=0., max_solves=1024, active=None, out=None, trace=False, totals=None):
        """K3: branch and bound of every instance of `tree` at states x0 [n_inst, nx] (CUDA fp64 tensor).
        Asynchronous on the handle's stream; returns a dict of CUDA tensors."""
        import torch
        dev = self.torch_device
        N = tree.n_inst
        assert x0.is_cuda and x0.dtype == torch.float64 and x0.is_contiguous() and x0.shape == (N, self.pd.nx)
        if out is None:
            out = dict(cost=torch.empty(N, dtype=torch.float64, device=dev),
                       node=torch.empty(N, dtype=torch.int32, device=dev),
                       primal=torch.zeros((N, self.layout.primal), dtype=torch.float64, device=dev),
                       n_solves=torch.empty(N, dtype=torch.int32, device=dev),
                       status=torch.empty(N, dtype=torch.int32, device=dev))
        if trace:
            out['trace'] = torch.full((N, 2 * max_solves), -1, dtype=torch.int32, device=dev)
        P = lambda a: C.c_void_p(a.data_ptr()) if a is not None else None
        _check(self.lib.wshmpc_bnb_solve(self._h, N, P(x0), P(active), C.byref(tree.c), C.c_double(tol), int(max_solves),
                                         P(out['cost']), P(out['node']), P(out['primal']), P(out['n_solves']),
                                         P(out['status']), P(out.get('trace')), P(totals)))
        return out

    def shift_tree(self, x0, e0, old_tree, inc_cost, inc_primal, new_tree, active=None, x_next=None, u0=None):
        """K2 + K4: warm start for the next step + plant update.  Asynchronous."""
        P = lambda a: C.c_void_p(a.data_ptr()) if a is not None else None
        _check(self.lib.wshmpc_shift_tree(self._h, old_tree.n_inst, P(x0), P(e0), C.byref(old_tree.c), P(inc_cost),
                                          P(inc_primal), P(active), C.byref(new_tree.c), P(x_next), P(u0)))

    def plant_step(self, plant, x, u, out=None):
        """wshmpc_plant_step: the states after one sample of the device plant `plant` (plants.DevicePlant) from x [n, nx]
        under inputs u [n, nu] (CUDA fp64 tensors).  Returns out [n, nx].  Asynchronous."""
        import torch
        n = x.shape[0]
        for a, w in ((x, self.pd.nx), (u, self.pd.nu)):
            assert a.is_cuda and a.dtype == torch.float64 and tuple(a.shape) == (n, w)
        x, u = x.contiguous(), u.contiguous()
        if out is None:
            out = torch.empty_like(x)
        c = _plant_struct(plant)
        _check(self.lib.wshmpc_plant_step(self._h, C.byref(c), n, C.c_void_p(x.data_ptr()), C.c_void_p(u.data_ptr()),
                                          C.c_void_p(out.data_ptr())))
        return out

    def new_fallback(self, n_inst, max_hold, max_law=0, K=None):
        """Caller-owned buffers of the fallback policy (wshmpc_fallback) for n_inst instances, without plans (age -1):
        dict(max_hold, plan, age, app_cost, app_primal, hold [n_inst]) of CUDA tensors.  With max_law > 0 also the terminal
        law: dict(max_law, law_K = a device copy of the gain K [nu, nx], law_n [n_inst] = 0)."""
        import torch
        f64 = dict(dtype=torch.float64, device=self.torch_device)
        i32 = dict(dtype=torch.int32, device=self.torch_device)
        P, nx, nu = self.layout.primal, self.pd.nx, self.pd.nu
        fb = dict(max_hold=int(max_hold), plan=torch.zeros((n_inst, P), **f64), age=torch.full((n_inst,), -1, **i32),
                  app_cost=torch.zeros(n_inst, **f64), app_primal=torch.zeros((n_inst, P), **f64),
                  hold=torch.zeros(n_inst, **i32), max_law=int(max_law))
        if max_law:
            K = np.asarray(K, dtype=float)
            if K.shape != (nu, nx):
                raise ValueError('terminal law gain of shape %s: [nu, nx] = [%d, %d]' % (K.shape, nu, nx))
            fb.update(law_K=torch.as_tensor(np.ascontiguousarray(K), **f64), law_n=torch.zeros(n_inst, **i32))
        return fb

    def fallback_step(self, fb, x, active, out):
        """wshmpc_fallback_step: the fallback policy after a lock-step branch and bound (`out` of bnb_solve) at states
        x [n_inst, nx]; writes fb['app_cost'], fb['app_primal'], fb['age'], fb['plan'] and fb['hold'].  Asynchronous."""
        N = x.shape[0]
        c = _fallback_struct(fb, fb['hold'])
        V = lambda a: C.c_void_p(a.data_ptr()) if a is not None else None
        _check(self.lib.wshmpc_fallback_step(self._h, N, C.byref(c), V(x), V(active), V(out['status']), V(out['cost']),
                                             V(out['primal'])))

    def closed_loop(self, n_steps, warm, fresh, par, xbuf, e, active, trees, out, tol=0., max_solves=1024, totals=None, logs=None,
                    mailbox=None, plant=None, fallback=None):
        """Fused closed loop (wshmpc_closed_loop): `n_steps` receding-horizon steps of every instance in one
        launch.  xbuf [2, n_inst, nx]; e [n_steps, n_inst, nx] or None; trees = (tree0, tree1).  Asynchronous.
        mailbox: a Mailbox -- the host is in the loop every step (the caller must answer it while the kernel runs).
        plant: a plants.DevicePlant -- the nonlinear plant advances the state on the device (wshmpc_closed_loop_plant), e is
        an additive disturbance on its output, and the logs gain 'x' [n_steps, n_inst, nx], the state after every step.
        fallback: buffers of new_fallback -- the loop runs under the fallback policy (wshmpc_closed_loop_fallback, also with
        max_hold = 0, and with the terminal law when the buffers have one) and the logs gain 'hold' [n_steps, n_inst].
        Returns the dict of per-step logs (CUDA tensors)."""
        import torch
        dev = self.torch_device
        N = trees[0].n_inst
        nx, nu = self.pd.nx, self.pd.nu
        assert xbuf.is_cuda and xbuf.dtype == torch.float64 and xbuf.is_contiguous() and tuple(xbuf.shape) == (2, N, nx)
        if e is not None:
            assert e.is_cuda and e.dtype == torch.float64 and e.is_contiguous() and tuple(e.shape) == (n_steps, N, nx)
        if logs is None:
            logs = dict(cost=torch.empty((n_steps, N), dtype=torch.float64, device=dev),
                        u0=torch.empty((n_steps, N, nu), dtype=torch.float64, device=dev),
                        n_solves=torch.empty((n_steps, N), dtype=torch.int32, device=dev),
                        status=torch.empty((n_steps, N), dtype=torch.int32, device=dev))
        need = 4 + (N + 2) * (n_steps + 1)
        if getattr(self, '_queue', None) is None or self._queue.numel() < need:
            self._queue = torch.empty(need, dtype=torch.int32, device=dev)
        if getattr(self, '_step_of', None) is None or self._step_of.numel() < N:
            self._step_of = torch.empty(N, dtype=torch.int32, device=dev)
        P = lambda a: a.data_ptr() if a is not None else None
        L = _Loop()
        L.n_steps, L.warm, L.fresh, L.par = int(n_steps), int(bool(warm)), int(bool(fresh)), int(par) & 1
        L.d_queue, L.d_step_of, L.d_x, L.d_e, L.d_active = P(self._queue), P(self._step_of), P(xbuf), P(e), P(active)
        L.d_log_cost, L.d_log_u0, L.d_log_solves, L.d_log_status = P(logs['cost']), P(logs['u0']), P(logs['n_solves']), P(logs['status'])
        L.mailbox = C.addressof(mailbox.c) if mailbox is not None else None
        V = lambda a: C.c_void_p(a.data_ptr()) if a is not None else None
        tail = (C.byref(trees[0].c), C.byref(trees[1].c), C.c_double(tol), int(max_solves), V(out['cost']), V(out['node']),
                V(out['primal']), V(out['n_solves']), V(out['status']), V(totals))
        c = None
        if plant is not None:
            if 'x' not in logs:
                logs['x'] = torch.empty((n_steps, N, nx), dtype=torch.float64, device=dev)
            assert logs['x'].is_contiguous() and tuple(logs['x'].shape) == (n_steps, N, nx)
            c = _plant_struct(plant, logs['x'])
        if fallback is not None:
            if 'hold' not in logs:
                logs['hold'] = torch.empty((n_steps, N), dtype=torch.int32, device=dev)
            assert logs['hold'].is_contiguous() and tuple(logs['hold'].shape) == (n_steps, N)
            f = _fallback_struct(fallback, logs['hold'])
            _check(self.lib.wshmpc_closed_loop_fallback(self._h, N, C.byref(L), C.byref(c) if c is not None else None,
                                                        C.byref(f), *tail))
        elif plant is None:
            _check(self.lib.wshmpc_closed_loop(self._h, N, C.byref(L), *tail))
        else:
            _check(self.lib.wshmpc_closed_loop_plant(self._h, N, C.byref(L), C.byref(c), *tail))
        return logs


def lp_batch(E, c, r, device=0, tol=1e-9, max_iter=None):
    """Batched standard-form LPs on the device (wshmpc_lp_batch):  min c'y s.t. E y = r_k, y >= 0.
    E [m, n] (shared) or [K, m, n]; c [n] (shared) or [K, n]; r [K, m] (numpy or CUDA tensors).
    Returns dict(status [K], obj [K], y [K, n], dual [K, m], iters [K]) of CUDA tensors."""
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError('no CUDA device: wshmpc_lp_batch runs on the GPU')
    lib = load_library()
    dev = torch.device('cuda', device)
    t = lambda a: torch.as_tensor(np.asarray(a, dtype=float) if not torch.is_tensor(a) else a, dtype=torch.float64, device=dev).contiguous()
    E, c, r = t(E), t(c), t(r)
    K, m = r.shape
    n = E.shape[-1]
    assert E.shape[-2] == m and c.shape[-1] == n
    sE = m * n if E.dim() == 3 else 0
    sc = n if c.dim() == 2 else 0
    out = dict(status=torch.zeros(K, dtype=torch.int32, device=dev), obj=torch.zeros(K, dtype=torch.float64, device=dev),
               y=torch.zeros((K, n), dtype=torch.float64, device=dev), dual=torch.zeros((K, m), dtype=torch.float64, device=dev),
               iters=torch.zeros(K, dtype=torch.int32, device=dev))
    P = lambda a: C.c_void_p(a.data_ptr())
    _check(lib.wshmpc_lp_batch(device, C.c_void_p(0), K, m, n, P(E), C.c_longlong(sE), P(c), C.c_longlong(sc), P(r), C.c_double(tol),
                               int(max_iter if max_iter is not None else 50 * (m + n)), P(out['status']), P(out['obj']), P(out['y']),
                               P(out['dual']), P(out['iters'])))
    return out
