#!/usr/bin/env python
"""bench.py -- B&B QP relaxations/s (and ms per MPC step, warm vs cold) of the hybrid-MPC hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cp20|cp40|syn30]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Workloads (BASELINE.json configs):
  cp20  (default; configs[1] per instance, batched as configs[2]): closed loop of the notebook two-wall cart-pole
        (T = 20), `--instances` independent initial states per GPU (data/cp20_instances.npy), model error
        e_t = sigma * randn * x_max, warm-started branch and bound with tree shifting;
  cp40  (configs[3]): the same system with horizon 40, states around the nominal x0;
  syn30 (configs[4]): synthetic MLD system nx = 20, 8 binaries / step, N = 30.
One bench "step" = ONE fused launch (wshmpc_closed_loop) that advances every instance of the batch by `--window`
receding-horizon steps = K3 (device B&B, K1 inside) + K2/K4 (tree shift + plant update) per MPC step, with no
barrier between instances.  Instances are independent: ranks own contiguous blocks of instances, there is no
collective on the data path (weak scaling; `--scaling strong` fixes the total instead).

Prints ONE JSON line (rank 0).  `value` = QP relaxations solved by all ranks / max-over-ranks device time,
states resident in HBM; `e2e` = the same loop with the HOST in it every MPC step of every instance through the public
Python API (ClosedLoop.run_mailbox: the kernel publishes each step's input to pinned mapped memory, a host plant answers
with the measured state and model error; `e2e.per_window_io` = host I/O once per window instead).
`--impl reference` times the CPU path (oracle/bnb_ref.py + oracle/qp_core.c, the restatement of the
reference's Python B&B pinned bit-exactly against it -- Gurobi is not available offline) on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'bnb_qp_relaxations_per_s'
UNIT = 'QP/s'

WORKLOADS = {
    'cp20': dict(model='cp20', instances=512, window=20, max_solves=1024, max_roots=512, steps=10, warmup=5,
                 text='cp20_closed_loop_warm_start (two-wall cart-pole, T=20, nx=4, nu=7, 4 binaries/step; '
                      'BASELINE configs[1] per instance, batched as configs[2])'),
    'cp40': dict(model='cp40', instances=592, window=4, max_solves=2048, max_roots=1024, steps=4, warmup=3,
                 text='cp40_closed_loop_warm_start (two-wall cart-pole, T=40: n=280 condensed inputs, 160 binaries, deep trees; '
                      'BASELINE configs[3])'),
    'syn30': dict(model='syn30', instances=148, window=2, max_solves=4096, max_roots=2048, steps=2, warmup=3,
                  text='syn30_closed_loop_warm_start (synthetic MLD, nx=20, nu=12 of which 8 binary, T=30: n=360, 240 binaries; '
                       'BASELINE configs[4]; states 0.3 x0_nominal (1 + 0.1 randn): at x0_nominal the MIQP needs > 10^4 nodes)'),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None, help='timed bench steps (default: 10; cp40 4; syn30 2)')
    ap.add_argument('--warmup', type=int, default=None, help='untimed warm-up bench steps (default: 5; cp40 / syn30 3)')
    ap.add_argument('--workload', default='cp20', choices=sorted(WORKLOADS))
    ap.add_argument('--window', type=int, default=None, help='receding-horizon steps per bench step (one fused launch)')
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--instances', type=int, default=None, help='independent MPC instances per GPU')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help='weak: --instances per GPU; strong: --instances-total split over the GPUs')
    ap.add_argument('--instances-total', type=int, default=4096, help='(strong scaling) instances of the whole job')
    ap.add_argument('--sigma', type=float, default=0.003, help='model error std (fraction of x_max)')
    ap.add_argument('--max-solves', type=int, default=None)
    ap.add_argument('--max-roots', type=int, default=None)
    ap.add_argument('--no-mailbox', action='store_true', help='e2e with host I/O once per window instead of the per-step mailbox (for runs '
                    'under ncu: it serialises launches, and a mailbox launch would wait for a host that cannot answer)')
    ap.add_argument('--no-extras', action='store_true', help='skip the legs outside the headline (cold / fresh start / per-step API / '
                                                             'published protocol / K2+K4 roofline / cpu baseline)')
    ap.add_argument('--cpu-seconds', type=float, default=15., help='budget of the cpu_baseline sample')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed bench step returned (ClosedLoop.run logs cost / u0 / n_solves / status and '
                         'the final states x) to DIR/<name>.npy as float64, to compare two builds output for output; '
                         'steps without a solution (status != 0, cost inf) are written as cost 0 and u0 0')
    a = ap.parse_args()
    w = WORKLOADS[a.workload]
    for k in ('instances', 'window', 'max_solves', 'max_roots', 'steps', 'warmup'):
        if getattr(a, k) is None:
            setattr(a, k, w[k])
    return a


def workload_config(args, world):
    n_total = args.instances_total if args.scaling == 'strong' else args.instances * world
    return {'workload': WORKLOADS[args.workload]['text'],
            'instances_per_gpu': n_total // world if args.scaling == 'strong' else args.instances, 'instances_total': n_total,
            'horizon': {'cp20': 20, 'cp40': 40, 'syn30': 30}[args.workload], 'sigma': args.sigma, 'tol': 0.,
            'window': args.window,
            'step': 'one fused launch = %d receding-horizon steps of every instance: device B&B (K3+K1) + tree shift/plant '
                    'update (K2+K4) per MPC step, task queue over (instance, step), no barrier between instances' % args.window,
            'timed_region': 'bench steps after `warmup` windows of the same loop (step 0 of every instance = cold solve, inside the '
                            'warm-up); inputs larger than L2 (two device trees of several GB per rank, leaf records touched per step >> 126 MB)',
            'search': 'best_first / branch_in_time, reference order, no speculative solves',
            'parallelism': 'instances sharded over %d GPU(s), no data-path collective' % world}


def initial_states(workload, model, lo, hi):
    """Frozen / seeded initial states lo..hi-1 of a workload (identical bits for the CPU and the GPU arm)."""
    if workload == 'cp20':
        x = np.load(os.path.join(ROOT, 'warm-start-hybrid-mpc_b200', 'data', 'cp20_instances.npy'))
        return np.ascontiguousarray(x[np.arange(lo, hi) % len(x)])
    nx = model['A'].shape[0]
    out = np.zeros((hi - lo, nx))
    for k in range(lo, hi):
        rng = np.random.default_rng(10_000 + k)
        if workload == 'cp40':
            # x0_nominal = [0, 0, 1, 0] sits at the edge of the set the horizon-40 MIQP is feasible on (a faster cart cannot be
            # stopped before the wall): scale it DOWN by up to 15 % and add a small offset in the other coordinates
            out[k - lo] = model['x0_nominal'] * rng.uniform(0.85, 1.0) + rng.uniform(-1, 1, nx) * np.array([0.005, 0.0025, 0., 0.0125])
        else:
            out[k - lo] = 0.3 * model['x0_nominal'] * (1. + 0.1 * rng.standard_normal(nx))
    return out


def noise(model, n_steps, n_inst, sigma, seed):
    rng = np.random.default_rng(seed)
    return sigma * rng.standard_normal((n_steps, n_inst, model['A'].shape[0])) * model['x_max']


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays, suffix=''):
    """Writes {name: array [..., n_inst, ...] with the instance axis given per array} as out_dir/<name><suffix>.npy in
    float64.  Above DUMP_LIMIT bytes in all, a fixed seeded sample of the instances is written instead, and its indices
    as instances<suffix>.npy."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: (np.asarray(v, dtype=np.float64), axis) for k, (v, axis) in arrays.items()}
    v0, axis0 = next(iter(arrays.values()))
    n_inst = v0.shape[axis0]
    total = sum(v.nbytes for v, _ in arrays.values())
    if total > DUMP_LIMIT:
        keep = max(1, n_inst * DUMP_LIMIT // total)
        idx = np.sort(np.random.default_rng(0).choice(n_inst, keep, replace=False))
        arrays = {k: (np.take(v, idx, axis=axis), axis) for k, (v, axis) in arrays.items()}
        np.save(os.path.join(out_dir, 'instances%s.npy' % suffix), idx.astype(np.float64))
    for k, (v, _) in arrays.items():
        np.save(os.path.join(out_dir, '%s%s.npy' % (k, suffix)), v)


# ---------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.samples.append(line.strip())
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2.)
        sm, mx, reasons = [], [], set()
        for s in self.samples:
            f = [v.strip() for v in s.split(',')]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except Exception:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons), 'samples': len(sm)}


# ---------------------------------------------------------------------------------------------------
# CPU path (oracle restatement of the reference; the only place bench.py touches oracle/)
# ---------------------------------------------------------------------------------------------------
def _cpu_worker(job):
    """Closed loop of one instance on one host core.  Returns per-step (t_start, t_end, solves)."""
    name, x0, e, n_steps, budget = job
    from oracle.models import load_model
    from oracle.qp_c import CoreC
    from oracle.bnb_ref import OracleController
    model = load_model(name)
    ctl = OracleController(model, CoreC(model, variant=1), hot_start='record')
    x = x0.copy(); ws = None; rows = []
    t_begin = time.perf_counter()
    for t in range(n_steps):
        t0 = time.perf_counter()
        try:
            inc, leaves, solves = ctl.feedforward(x, warm_start=ws)
        except RuntimeError:                     # the CPU QP core gave up on a node: this trajectory ends here
            break
        if inc is None:
            rows.append((t0, time.perf_counter(), solves)); break
        u0 = inc.primal['u'][0]
        ws = ctl.construct_warm_start(leaves, x, u0[:ctl.nuc], u0[ctl.nuc:], e[t])
        x = inc.primal['x'][1] + e[t]
        rows.append((t0, time.perf_counter(), solves))
        if budget is not None and time.perf_counter() - t_begin > budget:
            break
    return rows, ctl.qp_time


def cpu_baseline_sample(args, x0, e, seconds):
    """rank 0, N = 1: instance 0 of the workload on ONE host core (the reference loop is single-threaded)."""
    from oracle import qp_c
    qp_c.build()
    t0 = time.perf_counter()
    rows, qp_time = _cpu_worker((WORKLOADS[args.workload]['model'], x0[0], e[:, 0], e.shape[0], seconds))
    wall = time.perf_counter() - t0
    solves = sum(r[2] for r in rows)
    return {'value': solves / wall, 'unit': UNIT, 'cores': 1, 'kind': 'port',
            'sample': 'instance 0 of the workload, %d closed-loop steps (1 cold + %d warm), %d QPs in %.1f s; '
                      'oracle/bnb_ref.py + oracle/qp_core.c variant 1 (dual active-set, thin QR, each node started from the dual '
                      'solution it carries; no pinned-prefix elimination), Python overhead included'
                      % (len(rows), len(rows) - 1, solves, wall),
            'qp_only_value': solves / max(qp_time, 1e-9), 'ms_per_qp': 1e3 * wall / max(solves, 1),
            'host_cores_available': os.cpu_count()}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    world = args.gpus
    import multiprocessing as mp
    from oracle import qp_c
    from oracle.models import load_model
    qp_c.build()
    name = WORKLOADS[args.workload]['model']
    model = load_model(name)
    cores = max(1, os.cpu_count() or 1)
    S = args.window
    n_steps = (args.warmup + args.steps) * S
    if args.workload != 'cp20':
        # the big systems cost ~35 ms per QP on a core: a bounded sample = a cold step + the timed warm steps
        n_steps = min(n_steps, (1 + args.steps) * S)
    warm_steps = n_steps - args.steps * S
    x0 = initial_states(args.workload, model, 0, cores)
    e = noise(model, n_steps, cores, args.sigma, 1000)
    jobs = [(name, x0[k], e[:, k], n_steps, None) for k in range(cores)]
    with mp.get_context('fork').Pool(cores) as pool:
        res = pool.map(_cpu_worker, jobs)
    solves, t_lo, t_hi = 0, [], []
    for rows, _ in res:
        timed = rows[warm_steps:]
        if not timed:
            continue
        solves += sum(r[2] for r in timed)
        t_lo.append(timed[0][0]); t_hi.append(timed[-1][1])
    # each worker has its own clock origin (perf_counter is monotonic system-wide on Linux): whole-job time
    elapsed = max(hi - lo for lo, hi in zip(t_lo, t_hi)) if t_lo else float('nan')
    value = solves / elapsed
    cfg = workload_config(args, world)
    sample = ('%d instances (one per host core, fork pool) x %d timed closed-loop MPC steps (= %d bench steps of %d) after %d '
              'warm-up MPC steps (step 0 = cold solve); %d QPs' % (cores, args.steps * S, args.steps, S, warm_steps, solves))
    line = {'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': 1e3 * elapsed / args.steps, 'higher_is_better': True, 'scaling': args.scaling,
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic', 'config': cfg,
            'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample,
                             'note': 'Gurobi (the reference QP back end) is not installable offline; the reference B&B / '
                                     'warm-start logic is restated in oracle/bnb_ref.py (pinned bit-exactly against the '
                                     'reference code) on the oracle C QP core'},
            'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# B200 path
# ---------------------------------------------------------------------------------------------------
def fp64_peak_probe(torch, dev):
    """cuBLAS DGEMM 4096^3, best of 5 (MEASURED_PEAKS.json has no fp64 entry)."""
    n = 4096
    a = torch.randn((n, n), dtype=torch.float64, device=dev); b = torch.randn((n, n), dtype=torch.float64, device=dev)
    torch.matmul(a, b); torch.cuda.synchronize()
    best = float('inf')
    for _ in range(5):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); torch.matmul(a, b); e.record(); e.synchronize()
        best = min(best, s.elapsed_time(e))
    del a, b
    return 2. * n ** 3 / (best * 1e-3) / 1e12


def timed_loop(torch, dist, loop, steps, world, body):
    """Times `steps` bench steps bracketed by barrier + synchronize; body(t) launches step t.
    Returns (elapsed ms max over ranks, QPs of all ranks, iterations of all ranks, QPs of this rank); the counter deltas
    of this rank (wshmpc.h d_totals) are left in timed_loop.last."""
    from warm_start_hmpc_b200.closed_loop import reduce_stats
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    before = loop.totals.clone()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for t in range(steps):
        body(t)
    e.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = s.elapsed_time(e)
    d = (loop.totals - before).cpu().numpy()
    timed_loop.last = d
    qps, ms_max = reduce_stats(int(d[0]), ms)
    iters, _ = reduce_stats(int(d[1]), ms)
    return ms_max, qps, iters, int(d[0])


def published_protocol(torch, ctl, model, n_traj=100, n_steps=50):
    """The reference's experiment (notebooks/cart_pole_with_walls/statistical_analysis.py:58-196): x0 = [0, 0, 1, 0],
    sigma in {0, .001, .003, .01}, trajectory i drawn with np.random.seed(i), 50 closed-loop steps, cold-started and
    warm-started B&B side by side; QPs per step of both and their ratio (steps >= 1, trajectories that stay feasible)
    next to the published Gurobi-backed numbers (BASELINE.md: 12.6 / 12.6 / 11.7 / 8.9)."""
    from warm_start_hmpc_b200.closed_loop import ClosedLoop
    published = {0.: 12.6, 0.001: 12.6, 0.003: 11.7, 0.01: 8.9}
    out = {}
    nx = model['A'].shape[0]
    for sigma in (0., 0.001, 0.003, 0.01):
        N = 1 if sigma == 0. else n_traj
        e = np.zeros((n_steps, N, nx))
        for i in range(N):
            np.random.seed(i)                                       # statistical_analysis.py:73
            for t in range(n_steps):
                e[t, i] = sigma * np.multiply(np.random.randn(nx), model['x_max'])      # :176
        ed = torch.as_tensor(e, device='cuda')
        res = {}
        for warm in (True, False):
            L = ClosedLoop(ctl, N, warm=warm, max_solves=2048, max_roots=1024)
            L.reset(np.repeat(model['x0_nominal'][None], N, 0))
            t0 = time.perf_counter()
            logs = L.run(n_steps, e=ed)
            torch.cuda.synchronize()
            res[warm] = (logs['n_solves'].cpu().numpy(), logs['status'].cpu().numpy(), logs['cost'].cpu().numpy(), time.perf_counter() - t0)
            del L
        ok = np.all(res[True][1] == 0, axis=0) & np.all(res[False][1] == 0, axis=0)
        nw, nc = res[True][0][1:, ok], res[False][0][1:, ok]
        cw, cc = res[True][2][:, ok], res[False][2][:, ok]
        out['sigma_%g' % sigma] = {
            'trajectories': int(N), 'feasible_for_50_steps': int(ok.sum()),
            'cold_qp_per_step': float(nc.mean()) if ok.any() else None, 'warm_qp_per_step': float(nw.mean()) if ok.any() else None,
            'cold_over_warm': float(nc.mean() / nw.mean()) if ok.any() else None, 'published_cold_over_warm': published[sigma],
            'max_rel_cost_gap_warm_vs_cold': float(np.max(np.abs(cw - cc) / np.abs(cc))) if ok.any() else None,
            'ms_per_mpc_step_warm': 1e3 * res[True][3] / n_steps, 'ms_per_mpc_step_cold': 1e3 * res[False][3] / n_steps}
    out['published'] = 'BASELINE.md section 1 (Gurobi default method): cold 159.0 QPs/step, warm 12.6 QPs/step at sigma = 0'
    return out


def k2k4_roofline(torch, loop, pd, hbm_peak):
    """shift_tree_kernel (K2+K4) alone on the trees the timed loop left behind: algorithmic bytes = one dual record read
    and one written per retained leaf (+ the node arrays) / CUDA-event time, against the measured HBM copy bandwidth."""
    h = loop.h
    cur, nxt = loop.trees[loop.cur], loop.trees[1 - loop.cur]
    n_inst = loop.n_inst
    # one more search (K3) on the current trees gives the leaves a real step hands to the shift; K2+K4 is then timed on
    # (cur -> nxt), which it does not modify
    h.bnb_solve(loop.x, cur, tol=loop.tol, max_solves=loop.max_solves, active=loop.active, out=loop.out)
    args = (loop.x, None, cur, loop.out['cost'], loop.out['primal'], nxt)
    act = loop.active.clone()
    h.shift_tree(*args, active=act)
    torch.cuda.synchronize()
    leaves = int(nxt.n_nodes.sum()); nodes_in = int(cur.n_nodes.sum())
    reps = 5
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        act.copy_(loop.active)
        h.shift_tree(*args, active=act)
    e.record(); torch.cuda.synchronize()
    ms = s.elapsed_time(e) / reps
    rec_bytes = 8 * h.layout.rec_stride
    node_bytes = 4 * 3 + 8 + 4 * cur.words
    algo = leaves * 2 * rec_bytes + nodes_in * node_bytes + leaves * node_bytes
    gbs = algo / (ms * 1e-3) / 1e9
    return {'bound': 'hbm', 'kernel': 'shift_tree_kernel', 'achieved': gbs, 'peak': hbm_peak, 'unit': 'GB/s',
            'frac': gbs / hbm_peak if hbm_peak else None, 'ms': ms, 'instances': n_inst, 'retained_leaves': leaves,
            'algorithmic_bytes': algo,
            'note': 'K2+K4 alone, one CTA per instance, one warp per retained leaf: reads + writes one dual record (%d B) per leaf; '
                    'inside the fused loop the same code runs on the solver lanes' % rec_bytes}


def run_b200(args):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as g
    rank = int(os.environ.get('RANK', '0')); world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise RuntimeError('bench.py --impl b200 needs a GPU (there is no CPU fallback)')
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    if not os.path.exists(g.LIB):
        if rank == 0:
            g.build()
        if world > 1:
            dist.barrier()
    from warm_start_hmpc_b200.instances import load_model, controller_from_model
    from warm_start_hmpc_b200.closed_loop import ClosedLoop, shard
    model = load_model(WORKLOADS[args.workload]['model'])
    ctl = controller_from_model(model, device=local)
    dev = torch.device('cuda', local)
    S = args.window
    n_total = args.instances_total if args.scaling == 'strong' else args.instances * world
    lo, hi = shard(n_total, rank, world)
    n_inst = hi - lo
    x0 = initial_states(args.workload, model, lo, hi)
    n_win = args.warmup + args.steps
    nx, nu = ctl.mld.nx, ctl.mld.nu
    e_host = noise(model, (3 * n_win + 4) * S, n_inst, args.sigma, 1000 + rank).reshape(3 * n_win + 4, S, n_inst, -1)
    e_dev = torch.as_tensor(e_host, device=dev)

    tiny = ClosedLoop(ctl, 1, warm=True, max_solves=64, max_roots=64, n_slots=1)      # loads the module, creates the context
    tiny.reset(x0[:1]); tiny.run(1); torch.cuda.synchronize()
    del tiny
    loop = ClosedLoop(ctl, n_inst, warm=True, max_solves=args.max_solves, max_roots=args.max_roots)
    tree_bytes = loop.nbytes()
    f64 = dict(dtype=torch.float64, device=dev)
    logs = dict(cost=torch.empty((S, n_inst), **f64), u0=torch.empty((S, n_inst, nu), **f64),
                n_solves=torch.empty((S, n_inst), dtype=torch.int32, device=dev),
                status=torch.empty((S, n_inst), dtype=torch.int32, device=dev))
    loop.reset(x0)
    # warm-up windows; their wall time (from fresh states, cold step 0 included) is reported as `from_fresh_states`
    torch.cuda.synchronize(); t_fresh = time.perf_counter(); b_fresh = loop.totals.clone()
    for w in range(args.warmup):
        loop.run(S, e=e_dev[w], logs=logs)
    torch.cuda.synchronize(); t_fresh = time.perf_counter() - t_fresh
    q_fresh = int((loop.totals - b_fresh)[0])

    # ---- device-resident timed region: args.steps fused launches
    sampler = ClockSampler(local); sampler.start(); time.sleep(0.3)
    ev = []

    def dev_step(t):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); loop.run(S, e=e_dev[args.warmup + t], logs=logs); b.record()
        ev.append((a, b))
    l0 = loop.launches
    ms, qps, iters, my_qps = timed_loop(torch, dist, loop, args.steps, world, dev_step)
    if args.dump_outputs:            # the legs below reuse `logs` and the loop: copy the last timed step's results now
        out = {k: logs[k].cpu().numpy() for k in ('cost', 'u0', 'n_solves', 'status')}
        # a step without a solution (status != 0 and no incumbent: the instance has left the loop) comes back as cost inf and
        # u0 NaN; it is written as 0 and `status` tells which entries those are
        none = (out['status'] != 0) & ~np.isfinite(out['cost'])
        out['cost'] = np.where(none, 0., out['cost'])
        out['u0'] = np.where(none[..., None], 0., out['u0'])
        dump_outputs(args.dump_outputs, {k: (v, 1) for k, v in out.items()} | {'x': (loop.x.cpu().numpy(), 0)},
                     '_rank%d' % rank if world > 1 else '')
    cnt = timed_loop.last.astype(float)
    launches = loop.launches - l0
    clocks = sampler.stop()
    ker_ms = [a.elapsed_time(b) for a, b in ev]
    n_active = int(loop.active.sum())
    leaves_mean = float(loop.trees[loop.cur].n_nodes.double().mean())      # warm-start roots per instance after the last shift
    status = loop.out['status'].cpu().numpy()
    value = qps / (ms * 1e-3)

    def revive():
        """The synthetic system's closed loops end after a few steps (the MIQP becomes infeasible): a leg that would start
        with most instances off re-starts the batch from its initial states and replays the warm-up windows (untimed)."""
        if int(loop.active.sum()) * 2 >= n_inst:
            return False
        loop.reset(x0)
        for w in range(args.warmup):
            loop.run(S, e=e_dev[w], logs=logs)
        torch.cuda.synchronize()
        return True

    # ---- end-to-end through the public API with HOST buffers: per bench step H2D of the measured states and of the
    # window's model errors (pinned), one fused launch, D2H of the applied inputs, costs and final states
    pin = lambda *shape: torch.empty(shape, dtype=torch.float64).pin_memory()
    xh, eh, uh, ch, xnh = pin(n_inst, nx), pin(S, n_inst, nx), pin(S, n_inst, nu), pin(S, n_inst), pin(n_inst, nx)
    ed = torch.empty((S, n_inst, nx), **f64)
    revived = revive()
    xh.copy_(loop.x); torch.cuda.synchronize()
    e_host_t = torch.as_tensor(e_host)

    def e2e_step(t):
        eh.copy_(e_host_t[n_win + t])
        loop.x.copy_(xh, non_blocking=True); ed.copy_(eh, non_blocking=True)      # measured states, model errors
        loop.run(S, e=ed, logs=logs)
        uh.copy_(logs['u0'], non_blocking=True); ch.copy_(logs['cost'], non_blocking=True); xnh.copy_(loop.x, non_blocking=True)
        torch.cuda.synchronize()                                                    # the host needs the inputs now
        xh.copy_(xnh)
    ms_e, qps_e, _, _ = timed_loop(torch, dist, loop, args.steps, world, e2e_step)
    e2e_window = {'value': qps_e / (ms_e * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': (S + 1) * n_inst * nx * 8,
                  'd2h_bytes_per_step': n_inst * (S * (nu + 1) + nx) * 8, 'ms_per_step': ms_e / args.steps,
                  'ms_per_mpc_step_of_the_batch': ms_e / args.steps / S,
                  'api': 'ClosedLoop.run(n_steps, e): host I/O once per window of %d MPC steps, the plant (linear model + error) '
                         'is advanced on the device' % S}

    # ---- end to end with the HOST IN THE LOOP EVERY MPC STEP of every instance (the headline e2e): one persistent launch
    # per bench step; after each B&B the kernel publishes the applied input / predicted state of that instance to a pinned
    # mailbox, the host plant (numpy) answers with the measured state and the model error, and the instance's next step
    # starts as soon as a lane picks it up -- no barrier between instances (wshmpc_mailbox, ClosedLoop.run_mailbox)
    plant_calls = [0]

    def mailbox_step(t):
        ew = e_host[n_win + args.steps + t]

        def plant(idx, step, u0, x1):
            plant_calls[0] += 1
            return x1 + ew[step, idx], ew[step, idx]
        loop.run_mailbox(S, plant, logs=logs)
    if args.no_mailbox:
        e2e = e2e_window
    else:
        revived = revive() or revived
        mailbox_step(-1)                                                        # allocates the mailbox (untimed)
        plant_calls[0] = 0
        ms_m, qps_m, _, _ = timed_loop(torch, dist, loop, args.steps, world, mailbox_step)
        e2e = {'value': qps_m / (ms_m * 1e-3), 'unit': UNIT,
               'h2d_bytes_per_step': S * n_inst * (2 * nx * 8 + 4), 'd2h_bytes_per_step': S * n_inst * ((nu + nx + 1) * 8 + 8),
               'ms_per_step': ms_m / args.steps, 'ms_per_mpc_step_of_the_batch': ms_m / args.steps / S,
               'host_plant_calls_per_step': plant_calls[0] / max(args.steps, 1),
               'api': 'ClosedLoop.run_mailbox(n_steps, plant) of warm_start_hmpc_b200 (ctypes -> C ABI wshmpc_closed_loop with a '
                      'wshmpc_mailbox): host I/O EVERY MPC step of EVERY instance through pinned mapped memory -- D2H applied input, '
                      'predicted state, cost, status; H2D measured state and model error (host numpy plant x_1|t + e_t) -- with no '
                      'barrier between instances; results bit-identical to the device-resident loop (tests/test_gpu_bnb.py)',
               'per_window_io': e2e_window}
    if revived:
        e2e['note'] = 'most instances of this workload had left the loop (infeasible MIQP) by the end of the device-resident leg: the ' \
                      'batch was re-started from its initial states and the warm-up windows replayed (untimed) before this leg'

    # ---- roofline of the dominant kernel (closed_loop_kernel = K3 with K1 inside + K2/K4)
    pd = ctl.problem
    F_dense = 2. * pd.n ** 2 + 4. * pd.mc * pd.n                     # SURVEY.md 8(d): dense shared-operator form
    # executed form, with the MEASURED mean sizes of this rank's timed solves: a node with d pinned binaries is solved in
    # n_eff = n - d coordinates with a working set of k rows (wshmpc.h d_totals[2], [4], [5])
    my_q = max(cnt[0], 1.)
    kbar, n_eff, k0bar = cnt[2] / my_q, pd.n - cnt[4] / my_q, cnt[5] / my_q
    F_iter = 2. * pd.ns * n_eff + 2. * pd.mc * (pd.nx + pd.nu) + 2. * pd.nb + 4. * n_eff * kbar + kbar ** 2   # pricing + one append
    F_rebuild = k0bar * (4. * n_eff * k0bar / 2. + (k0bar / 2.) ** 2)                                       # k0 appends at growing k
    it_per_qp = iters / max(qps, 1)
    F_qp = it_per_qp * F_iter + F_rebuild
    qp_per_launch = qps / world / max(len(ker_ms), 1)
    it_per_launch = iters / world / max(len(ker_ms), 1)
    ker_avg_ms = float(np.mean(ker_ms))
    achieved = F_qp * qp_per_launch / (ker_avg_ms * 1e-3) / 1e12
    peak = fp64_peak_probe(torch, dev)
    peaks_file = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    hbm_peak = json.load(open(peaks_file)).get('hbm_gbs') if os.path.exists(peaks_file) else 6650.
    hbm_src = 'MEASURED_PEAKS.json (measured copy bandwidth)' if os.path.exists(peaks_file) else 'fallback of B200_PROFILING.md'
    B_node = 8 * (2 * pd.nb + pd.nx + pd.n + 2 * pd.m) + 12
    rec_bytes = 8 * loop.h.layout.rec_stride
    algo_hbm = qp_per_launch * B_node + S * n_inst * leaves_mean * 2 * rec_bytes
    roofline = {'bound': 'fp64-pipe (the kernel is LATENCY bound: neither the fp64 pipe nor HBM is near its roof)',
                'kernel': 'closed_loop_kernel', 'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s',
                'frac': achieved / peak, 'traffic': None,
                'peak_source': 'measured in this run: cuBLAS DGEMM 4096^3 best of 5 (fp64 pipe; MEASURED_PEAKS.json has no fp64 entry)',
                'algorithmic': 'flops per QP in the form the kernel executes: iterations x [2 ns n_eff (pricing operator) + 2 mc (nx+nu) '
                               '(stage rows) + 4 n_eff k + k^2 (Gram-Schmidt append, R^-1 column)] + re-factorisation of the k0 inherited '
                               'rows, with the measured means n_eff = n - d = %.1f, k = %.1f, k0 = %.1f, %.1f iterations/QP: %.0f flop/iteration, '
                               '%.0f flop/QP (the dense shared-operator form of SURVEY 8d would be %.0f flop/iteration); %.0f QPs/launch'
                               % (n_eff, kbar, k0bar, it_per_qp, F_iter, F_qp, F_dense, qp_per_launch),
                'achieved_dense_form_tflops': F_dense * it_per_launch / (ker_avg_ms * 1e-3) / 1e12,
                'kernel_ms_avg': ker_avg_ms, 'kernel_share_of_step': float(np.sum(ker_ms) / ms),
                'hbm': {'achieved_gbs': algo_hbm / (ker_avg_ms * 1e-3) / 1e9, 'peak_gbs': hbm_peak, 'peak_source': hbm_src,
                        'frac': algo_hbm / (ker_avg_ms * 1e-3) / 1e9 / hbm_peak,
                        'algorithmic_bytes_per_launch': algo_hbm,
                        'note': '%.0f QPs x %d B (K1) + %d steps x %d instances x %.1f leaves x 2 x %d B (K2+K4 tree shift)'
                                % (qp_per_launch, B_node, S, n_inst, leaves_mean, rec_bytes)},
                'solver_lanes_per_sm': int(ctl.default_slots() // torch.cuda.get_device_properties(local).multi_processor_count)}
    traffic_file = os.path.join(ROOT, 'profiles', 'closed_loop_kernel_traffic.json')
    if os.path.exists(traffic_file) and args.workload == 'cp20':
        roofline['traffic'] = json.load(open(traffic_file)).get('dram_bytes_per_launch')

    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None,
            'dtype': 'f64', 'data': 'synthetic', 'config': workload_config(args, world),
            'roofline': roofline, 'e2e': e2e, 'gpu_launches': launches, 'clocks': clocks,
            'ms_per_mpc_step_of_the_batch': ms / args.steps / S,
            'qp_per_mpc_step_per_instance': qps / args.steps / S / max(n_total, 1),
            'tree_bytes_per_rank': tree_bytes, 'active_instances_rank0': n_active, 'bnb_status_counts_rank0': {int(k): int((status == k).sum()) for k in np.unique(status)},
            'from_fresh_states': {'mpc_steps': args.warmup * S, 'qp': q_fresh, 'value': q_fresh / max(t_fresh, 1e-9), 'unit': UNIT,
                                  'ms_per_mpc_step_of_the_batch': 1e3 * t_fresh / max(args.warmup * S, 1),
                                  'note': 'rank 0, wall clock of the warm-up windows: MPC steps 0..%d of every instance from its fresh '
                                          'initial state, the cold solve of step 0 and the contact-mode transient included '
                                          '(BASELINE configs[1] asks for 100 steps)' % (args.warmup * S - 1)}}

    # ---- extras (outside the timed region)
    if not args.no_extras:
        line['roofline_k2k4'] = k2k4_roofline(torch, loop, pd, hbm_peak)
        del loop
        torch.cuda.empty_cache()
        # the same MPC steps 0 .. warmup x window - 1 from fresh states as ONE launch (BASELINE configs[1]: 100 receding-horizon
        # steps on CP20): no launch boundary every `window` steps, so no instance waits for the slowest one of a window
        n_fr = args.warmup * S
        if n_fr > 0:
            fr = ClosedLoop(ctl, n_inst, warm=True, max_solves=args.max_solves, max_roots=args.max_roots)
            fr.reset(x0)
            ms_f, qps_f, _, _ = timed_loop(torch, dist, fr, 1, world, lambda t: fr.run(n_fr, e=e_dev[:args.warmup].reshape(n_fr, n_inst, nx)))
            line['from_fresh_states']['one_launch'] = {
                'value': qps_f / max(ms_f * 1e-3, 1e-9), 'unit': UNIT, 'mpc_steps': n_fr, 'qp': qps_f, 'ms_per_mpc_step_of_the_batch': ms_f / n_fr,
                'note': 'all ranks, CUDA events: the same steps and model errors in ONE fused launch'}
            del fr
            torch.cuda.empty_cache()
        cold = ClosedLoop(ctl, n_inst, warm=False, max_solves=args.max_solves, max_roots=args.max_roots)
        cold.reset(x0)
        cold.run(1, e=e_dev[0, :1])
        ms_c, qps_c, _, _ = timed_loop(torch, dist, cold, 1, world, lambda t: cold.run(2, e=e_dev[1, :2]))
        line['cold_start'] = {'value': qps_c / (ms_c * 1e-3), 'unit': UNIT, 'ms_per_mpc_step_of_the_batch': ms_c / 2,
                              'qp_per_mpc_step_per_instance': qps_c / 2 / max(n_total, 1)}
        line['warm_start'] = {'value': value, 'unit': UNIT, 'ms_per_mpc_step_of_the_batch': ms / args.steps / S,
                              'qp_per_mpc_step_per_instance': line['qp_per_mpc_step_per_instance']}
        del cold
        torch.cuda.empty_cache()
        # per-MPC-step API with HOST I/O every step: H2D of the measured state and model error, K3, K2+K4, D2H of the applied
        # input and cost; every instance waits for the slowest one of the step (lock step)
        lock = ClosedLoop(ctl, n_inst, warm=True, max_solves=args.max_solves, max_roots=args.max_roots)
        lock.reset(x0)
        for t in range(3):
            lock.step(e=e_dev[0, t % S])
        xs_h, es_h, us_h, cs_h = pin(n_inst, nx), pin(n_inst, nx), pin(n_inst, nu), pin(n_inst)
        es_d = torch.empty((n_inst, nx), **f64)
        xs_h.copy_(lock.x); torch.cuda.synchronize()
        n_lock = 5

        def lock_step(t):
            es_h.copy_(e_host_t[1, t % S])
            es_d.copy_(es_h, non_blocking=True); lock.x.copy_(xs_h, non_blocking=True)
            out = lock.step(e=es_d)
            us_h.copy_(lock.u0, non_blocking=True); cs_h.copy_(out['cost'], non_blocking=True); xs_h.copy_(lock.x, non_blocking=True)
            torch.cuda.synchronize()
        ms_l, qps_l, _, _ = timed_loop(torch, dist, lock, n_lock, world, lock_step)
        line['per_mpc_step_api'] = {'value': qps_l / (ms_l * 1e-3), 'unit': UNIT, 'ms_per_mpc_step_of_the_batch': ms_l / n_lock,
                                    'h2d_bytes_per_mpc_step': 2 * n_inst * nx * 8, 'd2h_bytes_per_mpc_step': n_inst * (nu + 1 + nx) * 8,
                                    'note': 'ClosedLoop.step(): host I/O every MPC step IN LOCK STEP, one launch pair per step, every '
                                            'instance waits for the slowest one of the step (10-30x the median number of QPs); the '
                                            'mailbox loop timed in `e2e` has the same host I/O without that barrier'}
        del lock
        torch.cuda.empty_cache()
        if rank == 0:
            single = {}
            for warm in (True, False):
                L = ClosedLoop(ctl, 1, warm=warm, max_solves=4096, max_roots=args.max_roots, n_slots=1)
                L.reset(x0[:1] if args.workload != 'cp20' else model['x0_nominal'][None])
                L.step(); torch.cuda.synchronize()
                before = L.totals.clone()
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                k = 5
                s.record()
                for _ in range(k):
                    L.step()
                e.record(); torch.cuda.synchronize()
                d = (L.totals - before).cpu().numpy()
                single['warm' if warm else 'cold'] = {'ms_per_mpc_step': s.elapsed_time(e) / k, 'qp_per_step': float(d[0]) / k,
                                                      'qp_per_s': float(d[0]) / (s.elapsed_time(e) * 1e-3)}
                del L
            if args.workload == 'cp20':
                single['reference_published'] = {'cold_ms_per_mpc_step': 530., 'warm_ms_per_mpc_step': 37.4, 'qp_per_s': 300.,
                                                 'source': 'BASELINE.md (Gurobi, unknown CPU)'}
            line['single_instance_nominal'] = single
            if args.workload == 'cp20':
                try:
                    line['published_protocol'] = published_protocol(torch, ctl, model)
                except Exception as ex:                     # information only
                    line['published_protocol'] = {'error': repr(ex)}
    if rank == 0 and world == 1 and not args.no_extras:
        line['cpu_baseline'] = cpu_baseline_sample(args, x0, e_host.reshape(-1, n_inst, nx), args.cpu_seconds)
    elif rank == 0:
        line['cpu_baseline'] = None
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    a = parse_args()
    if a.impl == 'reference':
        if a.dump_outputs:
            sys.exit('bench.py: --dump-outputs is implemented for --impl b200')
        run_reference(a)
    else:
        run_b200(a)
