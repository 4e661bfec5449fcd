"""Batched closed loop of independent MPC instances, entirely on the device.

Restates the experiment loop of notebooks/cart_pole_with_walls/statistical_analysis.py:93-196
(without its Gurobi legs) for `n_inst` instances at once: per step  branch and bound (K3, warm- or
cold-started)  ->  construct_warm_start + plant update x <- x_1|t + e_t (K2 + K4).  Two device trees
are used alternately (the shift reads one and writes the other); nothing synchronises with the host
unless the caller reads a result.  Instances are independent: under torch.distributed each rank owns
a contiguous block of instances (`shard`) and no collective is on the data path.
"""
import numpy as np


def shard(n_total, rank, world):
    """Contiguous block [lo, hi) of the instances owned by `rank` (SURVEY.md section 8e)."""
    base, rem = divmod(n_total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class ClosedLoop(object):

    def __init__(self, controller, n_inst, warm=True, tol=0., max_solves=1024, max_roots=None, n_slots=None, comparator=False,
                 mip_start=True, plant=None, fallback=0, terminal_law=0, law_gain=None):
        """comparator=True runs the conventional MIQP branch and bound of `feedforward_miqp` (controller.py:530-582, the
        paper's third curve) instead of the structured search, cold-started every step; with mip_start the previous step's
        incumbent binaries, shifted by one step, are the MIP start (shift_binary_solution).  max_roots: initial leaves a
        tree holds (default 512; 2 for the comparator, whose trees hold a guess and a root).
        plant: a plants.DevicePlant -- step() and run() advance the state through the nonlinear plant on the device instead
        of x <- x_1|t + e: x_{t+1} = Phi(x_t, u0) + e_t (e an optional disturbance), and the warm start is corrected with
        the measured model error x_{t+1} - x_1|t.  It has one parameter set, or one per instance.
        fallback: H, 0 <= H <= T - 1.  With H > 0 an instance whose MIQP is infeasible applies the next input of its last plan
        for up to H steps in a row instead of leaving the loop, and the shifted tree of the infeasible step warm-starts the
        next one (wshmpc_fallback in include/wshmpc.h); out['hold'] and the logs' 'hold' say where each applied input came
        from (0 the incumbent, a > 0 input u_a of the plan, -2 the terminal law, -1 none).  Not with the comparator.
        terminal_law: L >= 0.  With L > 0 an instance whose MIQP is infeasible and that has no plan step left applies the
        terminal law u = K x for up to L steps in a row (counted since its last incumbent) instead of leaving the loop; also
        with fallback = 0.  law_gain: K [nu, nx], default controller.terminal_law()."""
        import torch
        if comparator and warm:
            raise ValueError('the MIQP comparator runs cold trees only: use ClosedLoop(..., warm=False, comparator=True)')
        if plant is not None and plant.n_sets not in (1, n_inst):
            raise ValueError('the plant has %d parameter sets: 1, or one per instance (%d)' % (plant.n_sets, n_inst))
        if int(fallback) != fallback or not 0 <= fallback <= controller.T - 1:
            raise ValueError('fallback = %r: the steps an instance may hold its plan, 0 .. T - 1 = %d' % (fallback, controller.T - 1))
        if int(terminal_law) != terminal_law or terminal_law < 0:
            raise ValueError('terminal_law = %r: the steps an instance may run on the terminal law, >= 0' % (terminal_law,))
        if (fallback or terminal_law) and comparator:
            raise ValueError('the fallback policy runs under the structured search only, not with the MIQP comparator')
        if terminal_law:
            law_gain = controller.terminal_law() if law_gain is None else np.asarray(law_gain, dtype=float)
            if law_gain.shape != (controller.mld.nu, controller.mld.nx):
                raise ValueError('law_gain of shape %s: the terminal law gain is [nu, nx] = [%d, %d]'
                                 % (law_gain.shape, controller.mld.nu, controller.mld.nx))
        self.plant = plant
        if max_roots is None:
            max_roots = 2 if comparator else 512
        self.comparator, self.mip_start = comparator, mip_start
        self.node_rule = (2 if mip_start else 1) if comparator else 0
        self.ctl, self.n_inst, self.warm, self.tol = controller, n_inst, warm, tol
        self.max_solves, self.max_roots = max_solves, max_roots
        slots = n_slots if n_slots is not None else min(n_inst, controller.default_slots())
        self.h = h = controller.handle(slots)
        dev = h.torch_device
        cap_nodes, cap_recs = max_roots + 2 * max_solves + 2, max_roots + max_solves + 1
        self.trees = [h.new_tree(n_inst, cap_nodes, cap_recs) for _ in range(2)]
        self.cur = 0
        nx, nu = controller.mld.nx, controller.mld.nu
        f64 = dict(dtype=torch.float64, device=dev)
        self.xbuf = torch.zeros((2, n_inst, nx), **f64)     # states, ping-pong (the shift writes the other half)
        self.xpar = 0
        self.u0 = torch.zeros((n_inst, nu), **f64)
        self.active = torch.ones(n_inst, dtype=torch.int32, device=dev)
        self.out = dict(cost=torch.zeros(n_inst, **f64), node=torch.zeros(n_inst, dtype=torch.int32, device=dev),
                        primal=torch.zeros((n_inst, h.layout.primal), **f64),
                        n_solves=torch.zeros(n_inst, dtype=torch.int32, device=dev),
                        status=torch.zeros(n_inst, dtype=torch.int32, device=dev))
        self.totals = torch.zeros(8, dtype=torch.int64, device=dev)     # wshmpc.h d_totals: QP solves, iterations, working-set statistics
        self.gid = torch.arange(n_inst, dtype=torch.int64, device=dev)     # global identity of the instance in every slot (rebalance moves instances)
        self.fresh = True
        self.launches = 0
        self.events = None          # list -> (start, after K3, after K2+K4) CUDA events of every step
        # plans, ages, applied pairs and the terminal law (wshmpc_fallback)
        self.fb = h.new_fallback(n_inst, fallback, int(terminal_law), law_gain) if (fallback or terminal_law) else None
        if self.fb is not None:
            self.out['hold'] = self.fb['hold']

    @property
    def x(self):
        """Current states [n_inst, nx] (CUDA tensor view)."""
        return self.xbuf[self.xpar]

    def nbytes(self):
        return sum(t.nbytes() for t in self.trees)

    def reset(self, x0):
        """New initial states [n_inst, nx]; the next step starts from the root node."""
        import torch
        self.x.copy_(torch.as_tensor(np.asarray(x0, dtype=float) if not torch.is_tensor(x0) else x0))
        self.active.fill_(1)
        if self.fb is not None:
            self.fb['age'].fill_(-1)
            if self.fb.get('law_n') is not None:
                self.fb['law_n'].zero_()
        self.totals.zero_()
        self.fresh = True

    def rebalance(self, group=None, min_gap=2):
        """Periodic load balancing between the ranks of a torch.distributed job (rebalance.py): live instances move from
        the busiest ranks into the slots of dead instances of the idlest ones, with their warm-start trees.  Call it
        between steps / windows.  Returns (sent, received, plan)."""
        if self.plant is not None and self.plant.n_sets > 1:
            raise ValueError('rebalance does not move per-instance plant parameter sets with their instances')
        if self.fb is not None:
            raise ValueError('rebalance does not move the fallback plans with their instances')
        from .rebalance import rebalance
        return rebalance(self.trees[self.cur], self.x, self.active, self.gid, group, min_gap)

    def _init_tree(self, tree):
        """Root node of a cold step; in comparator mode with mip_start, [MIP start, root] for every instance whose previous
        step left an incumbent (what the fused loop builds on the device, wshmpc_set_node_rule 2)."""
        import torch
        h = self.h
        if self.node_rule == 2 and not self.fresh:
            T, nx, nu, nub = self.ctl.T, self.ctl.mld.nx, self.ctl.mld.nu, self.ctl.mld.nub
            ub = self.out['primal'][:, (T + 1) * nx:].reshape(self.n_inst, T, nu)[:, :, nu - nub:]
            guess = torch.zeros((self.n_inst, T, nub), dtype=torch.float64, device=ub.device)
            guess[:, :T - 1] = torch.round(ub[:, 1:])                    # shift_binary_solution (controller.py:586-588)
            has = ((self.active != 0) & torch.isfinite(self.out['cost'])).to(torch.int32)
            h.tree_init_guess(tree, guess.reshape(self.n_inst, T * nub), has)
        else:
            h.tree_init_root(tree)
        self.launches += 1
        self.fresh = False

    def _bnb(self, tree):
        h = self.h
        if self.node_rule:
            h.set_node_rule(self.node_rule)
        try:
            h.bnb_solve(self.x, tree, tol=self.tol, max_solves=self.max_solves, active=self.active, out=self.out,
                        totals=self.totals)
        finally:
            if self.node_rule:
                h.set_node_rule(0)
        self.launches += 1

    def _closed_loop(self, n_steps, par, e, logs, mailbox=None):
        h = self.h
        fresh = self.fresh if (self.warm or self.comparator) else True
        if self.node_rule:
            h.set_node_rule(self.node_rule)
        try:
            return h.closed_loop(n_steps, self.warm, fresh, par, self.xbuf, e, self.active, self.trees, self.out,
                                 tol=self.tol, max_solves=self.max_solves, totals=self.totals, logs=logs, mailbox=mailbox,
                                 plant=self.plant, fallback=self.fb)
        finally:
            if self.node_rule:
                h.set_node_rule(0)

    def _applied(self):
        """(cost, primal) of the pair the plant and K2 + K4 apply: the incumbent, or with a fallback the policy's choice
        (wshmpc_fallback_step, run right after the branch and bound)"""
        if self.fb is None:
            return self.out['cost'], self.out['primal']
        self.h.fallback_step(self.fb, self.x, self.active, self.out)
        return self.fb['app_cost'], self.fb['app_primal']

    def step(self, e=None, x=None):
        """One receding-horizon step of every instance.  `x` (optional, [n_inst, nx] CUDA tensor)
        overrides the state (measured state fed back from the host); `e` is the model error e_t.
        With a device plant: branch and bound (K3), the plant from the live instances' states and inputs (plus e, a
        disturbance), the model error x_meas - x_1|t, K2 + K4, and the next state x_meas -- all on the device.
        With a fallback, the plant and K2 + K4 apply the policy's input (out['hold'])."""
        h = self.h
        if x is not None:
            self.x.copy_(x)
        tree = self.trees[self.cur]
        if self.fresh or not self.warm:
            self._init_tree(tree)
        if self.events is not None:
            import torch
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            ev[0].record()
        self._bnb(tree)
        if self.events is not None:
            ev[1].record()
        cost, prim = self._applied()
        # K2 + K4 (in cold mode only its plant update matters: the next step re-initialises the root)
        new = self.trees[1 - self.cur]
        x_meas = None
        if self.plant is not None:
            x_meas, e = self._device_plant(e, cost, prim)
        h.shift_tree(self.x, e, tree, cost, prim, new, active=self.active,
                     x_next=self.xbuf[1 - self.xpar], u0=self.u0)
        if x_meas is not None:
            self.xbuf[1 - self.xpar].copy_(x_meas)
        self.cur = 1 - self.cur
        self.launches += 1
        if self.events is not None:
            ev[2].record()
            self.events.append(tuple(ev))
        self.xpar = 1 - self.xpar
        return self.out

    def _device_plant(self, d, cost, prim):
        """(x_meas, e) of step(): x_meas = Phi(x, u0) + d where the step has an applied pair (cost, prim), else x;
        e = x_meas - x_1|t there, else 0 (what the fused loop computes in the lane)"""
        import torch
        nx, nu, T = self.ctl.mld.nx, self.ctl.mld.nu, self.ctl.T
        live = ((self.active != 0) & torch.isfinite(cost))[:, None]
        x_meas = self.plant.step(self.h, self.x, prim[:, (T + 1) * nx:(T + 1) * nx + nu])
        if d is not None:
            x_meas = x_meas + d
        x_meas = torch.where(live, x_meas, self.x)
        return x_meas, torch.where(live, x_meas - prim[:, nx:2 * nx], torch.zeros_like(x_meas))

    def step_with_plant(self, plant):
        """One receding-horizon step against a TRUE plant instead of the linear model + noise: branch and bound (K3), the
        applied input goes to `plant(x [n, nx], u0 [n, nu]) -> next measured state [n, nx]` (host numpy, e.g.
        plants.CartPoleWithWalls.simulate), the model error e_t = x_measured - x_1|t is what the warm start of the next
        step is corrected with (construct_warm_start's e0, controller.py:503-564), then K2 + K4.  With a fallback the plant
        gets the policy's input and x_1|t is that of the applied pair (out['hold']).
        Returns (out, u0 [n, nu] numpy, e [n, nx] numpy)."""
        import torch
        h = self.h
        tree = self.trees[self.cur]
        if self.fresh or not self.warm:
            self._init_tree(tree)
        self._bnb(tree)
        cost_d, prim_d = self._applied()
        nx, nu, T = self.ctl.mld.nx, self.ctl.mld.nu, self.ctl.T
        prim = prim_d.cpu().numpy()
        x_now = self.x.cpu().numpy()
        u0 = prim[:, (T + 1) * nx:(T + 1) * nx + nu]
        x_pred = prim[:, nx:2 * nx]
        live = (self.active.cpu().numpy() != 0) & np.isfinite(cost_d.cpu().numpy())
        x_meas = np.array(x_now)
        if live.any():
            x_meas[live] = plant(x_now[live], u0[live])
        e = np.where(live[:, None], x_meas - x_pred, 0.)
        ed = torch.as_tensor(e, device=self.x.device)
        new = self.trees[1 - self.cur]
        h.shift_tree(self.x, ed, tree, cost_d, prim_d, new, active=self.active,
                     x_next=self.xbuf[1 - self.xpar], u0=self.u0)
        if live.any():
            # the next step starts from the MEASURED state itself (x_1|t + (x_measured - x_1|t) is one rounding away from it)
            lv = torch.as_tensor(live, device=self.x.device)
            self.xbuf[1 - self.xpar][lv] = torch.as_tensor(x_meas[live], device=self.x.device)
        self.cur = 1 - self.cur
        self.xpar = 1 - self.xpar
        self.launches += 1
        return self.out, u0, e

    def run(self, n_steps, e=None, logs=None):
        """`n_steps` receding-horizon steps of every instance in ONE launch (wshmpc_closed_loop): the fused
        form of calling step() n_steps times, without a barrier between the steps of different instances.
        e: [n_steps, n_inst, nx] CUDA tensor of model errors or None (with a device plant: of disturbances on the plant's
        output).  Returns per-step logs (cost, u0, n_solves, status), each [n_steps, n_inst, ...], with a device plant
        also x, the state after every step, and with a fallback also hold; self.x holds the final states."""
        par = self.cur
        # states and trees flip together: make the state parity equal to the tree parity
        if self.xpar != par:
            self.xbuf[par].copy_(self.xbuf[self.xpar]); self.xpar = par
        logs = self._closed_loop(n_steps, par, e, logs)
        self.launches += 2
        self.fresh = False
        self.cur = (self.cur + n_steps) & 1
        self.xpar = (self.xpar + n_steps) & 1
        return logs


    def run_mailbox(self, n_steps, plant, timeout_s=120., logs=None):
        """`n_steps` receding-horizon steps of every instance with the HOST in the loop every step and no barrier between
        instances (wshmpc_closed_loop with a wshmpc_mailbox): one persistent launch solves; this thread polls the pinned
        mailbox, and whenever instances have published a step it calls
            plant(idx [k] instance indices, step [k], u0 [k, nu], x_pred [k, nx]) -> x_measured [k, nx]  or  (x_measured, e)
        (host numpy; u0 is NaN where a step has no incumbent) and hands the measured states and the model errors
        e = x_measured - x_pred back -- the per-step use of `feedforward` + `construct_warm_start`
        (statistical_analysis.py:120-196) for a batch of independent plants.  Returns the device logs of run() plus
        'host' = dict(u0, x1, cost, status) numpy arrays [n_steps, n_inst, ...] as the host saw them."""
        import time
        import torch
        from .capi import Mailbox
        if self.plant is not None:
            raise ValueError('run_mailbox: the host is the plant there; this loop has a device plant (use run or step)')
        if self.fb is not None:
            raise ValueError('run_mailbox has no fallback policy: use run, step or step_with_plant')
        h, N = self.h, self.n_inst
        if getattr(self, '_mailbox', None) is None:
            self._mailbox = Mailbox(h, N)
        mb = self._mailbox
        mb.clear()
        par = self.cur
        if self.xpar != par:
            self.xbuf[par].copy_(self.xbuf[self.xpar]); self.xpar = par
        nx, nu = self.ctl.mld.nx, self.ctl.mld.nu
        host = dict(u0=np.full((n_steps, N, nu), np.nan), x1=np.zeros((n_steps, N, nx)), cost=np.full((n_steps, N), np.inf),
                    status=np.zeros((n_steps, N), dtype=np.int32))
        logs = self._closed_loop(n_steps, par, None, logs, mailbox=mb)
        self.launches += 2
        seen = np.zeros(N, dtype=np.int32)
        t_end = time.time() + timeout_s
        n_left = N * n_steps
        try:
            while n_left > 0:
                idx = np.nonzero(mb.out_step > seen)[0]
                if idx.size == 0:
                    if time.time() > t_end:
                        raise RuntimeError('run_mailbox: the kernel published nothing for %.0f s' % timeout_s)
                    continue
                s = seen[idx]
                u0 = mb.out_u0[idx].copy(); x1 = mb.out_x1[idx].copy()
                host['u0'][s, idx] = u0; host['x1'][s, idx] = x1
                host['cost'][s, idx] = mb.out_cost[idx]; host['status'][s, idx] = mb.out_status[idx]
                ans = plant(idx, s, u0, x1)
                if isinstance(ans, tuple):
                    xm, e = ans
                else:
                    xm = np.asarray(ans, dtype=float); e = xm - x1
                live = np.isfinite(u0).all(axis=1)
                mb.in_x[idx] = np.where(live[:, None], xm, x1)
                mb.in_e[idx] = np.where(live[:, None], e, 0.)
                mb.in_step[idx] = s + 1            # after the data (x86 stores are not reordered)
                seen[idx] = s + 1
                n_left -= idx.size
                t_end = time.time() + timeout_s
        except BaseException:
            mb.stop[0] = 1                          # never leave the kernel waiting for an answer
            torch.cuda.synchronize(h.torch_device)
            raise
        self.fresh = False
        self.cur = (self.cur + n_steps) & 1
        self.xpar = (self.xpar + n_steps) & 1
        logs['host'] = host
        return logs


def reduce_stats(n_units, elapsed_ms, device=None):
    """Whole-job aggregate under torch.distributed (one process per GPU, no data-path collective):
    units are summed over ranks, time is the MAX over ranks.  Works with NCCL (CUDA tensors) and gloo
    (CPU tensors); without an initialised process group it returns the inputs."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return int(n_units), float(elapsed_ms)
    dev = device if device is not None else ('cuda' if dist.get_backend() == 'nccl' else 'cpu')
    u = torch.tensor([int(n_units)], dtype=torch.int64, device=dev)
    t = torch.tensor([float(elapsed_ms)], dtype=torch.float64, device=dev)
    dist.all_reduce(u, op=dist.ReduceOp.SUM)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return int(u.item()), float(t.item())
