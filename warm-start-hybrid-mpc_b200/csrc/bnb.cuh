// bnb.cuh -- device-side branch and bound (K3) and warm-start construction (K2 + K4).
//
// K3 replaces branch_and_bound.py:408-499 driven by the closures of controller.py:365-380 and the
// child-bound rule of controller.py:395-429.  K2/K4 replace controller.py:431-564, 615-721.
// One CTA owns one MPC instance at a time; instances are handed out by an atomic work counter, so
// thousands of independent closed-loop instances keep every SM busy with no host round trip per node.
#pragma once
#include "qp_device.cuh"
#include "records.cuh"
#include "plant.cuh"

struct TreeView {
    int cap_nodes, cap_recs, words;
    int *n_nodes, *n_recs, *depth, *alive, *rec;
    unsigned int *bits;      // values of the assigned binaries
    unsigned int *mask;      // which binaries are assigned (a chronological prefix for branch_in_time trees; any set otherwise)
    double *lb, *rec_dobj, *rec_dual;
};

#define BNB_OK 0
#define BNB_INFEASIBLE 1
#define BNB_CAPACITY 2
#define BNB_QP_LIMIT 3

// node rules of K3 (wshmpc_set_node_rule): 0 the structured search (branch on the first unassigned binary of the branching
// order, a node is an incumbent iff every binary is pinned, children inherit dual bounds); 1 the conventional MIQP branch and
// bound of feedforward_miqp (controller.py:530-582); 2 = 1 with a MIP start at every step of the fused closed loop
#define BNB_RULE_MIQP 1
#define BNB_RULE_MIQP_START 2
#define BNB_INTEGRAL_TOL 1e-9     // largest |u - rint(u)| of an integral relaxation (feedforward_miqp)

// per-slot scratch of the B&B kernel (doubles): lb | ub | primal record | cost | dobj
__host__ __device__ __forceinline__ size_t bnb_scratch_doubles(int nb, int n_primal) { return 2 * (size_t)nb + n_primal + 4; }

#if WS_TU_HAS(0)
__global__ void init_root_kernel(int n_inst, TreeView tr)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_inst) return;
    const size_t o = (size_t)k * tr.cap_nodes;
    tr.n_nodes[k] = 1; tr.n_recs[k] = 0;
    tr.depth[o] = 0; tr.alive[o] = 1; tr.rec[o] = -1; tr.lb[o] = -INFINITY;
    for (int w = 0; w < tr.words; ++w) { tr.bits[o * tr.words + w] = 0u; tr.mask[o * tr.words + w] = 0u; }
}
#endif

// ---------------------------------------------------------------------------------------------
// K3
// ---------------------------------------------------------------------------------------------
// branch and bound of ONE instance by the calling CTA (all threads).  Returns the status.
// RULE: 0 the structured search, 1 the conventional MIQP rule (BNB_RULE_MIQP; the branching binary is chosen AFTER the
// node's solve, from its relaxation) -- a template parameter, so that the default kernels carry none of the rule-1 code.
// n_iters (null: not wanted): every thread gets the active-set iterations of the search, the sum it adds to totals[1].
template <int RULE>
__device__ __forceinline__ int bnb_instance(const DevProblem &P, const Ctx &cx, const SlotPtrs &sp, double *y, double *sc, int *iters_s,
                                   int inst, const double *xi, const TreeView &tr, double tol, int max_solves,
                                   double *inc_cost, int *inc_node, double *inc_primal, int *n_solves, int *trace,
                                   unsigned long long *totals, int *n_iters = nullptr)
{
    const int nb = P.nb;
    double *lbv = sc, *ubv = sc + nb, *prim = sc + 2 * nb, *cost_s = prim + P.n_primal, *dobj_s = cost_s + 1;
    const size_t no = (size_t)inst * tr.cap_nodes;
    int *depth = tr.depth + no, *alive = tr.alive + no, *rec = tr.rec + no;
    unsigned int *bits = tr.bits + no * tr.words, *mask = tr.mask + no * tr.words;
    double *lb = tr.lb + no;
    double *rdobj = tr.rec_dobj + (size_t)inst * tr.cap_recs;
    double *rdual = tr.rec_dual + (size_t)inst * tr.cap_recs * P.n_rec;
    int *tr_i = trace ? trace + (size_t)inst * 2 * max_solves : nullptr;

    int nn = tr.n_nodes[inst], nr = tr.n_recs[inst];
    const int nn0 = nn;                      // nodes >= nn0 are children created by this search
    int memo_rec = -1, memo_d = -1;          // sibling memo of the slot: (parent record, eliminated prefix) of the parked factor
    double ub = INFINITY;
    int inc = -1, solves = 0, st = -1, k = 0;
    long long iters = 0, ksum = 0, dsum = 0, k0sum = 0;
    int kmx = 0;

    while (st < 0) {
        // ---- select: candidates = alive leaves with lb < ub - tol, in list (= creation) order ;
        //      best_first = first minimum of lb (branch_and_bound.py:541-563), depth_first = last candidate (:521-538),
        //      breadth_first = first candidate (:501-518)
        const double cutoff = ub - tol;
        double best = INFINITY; int bi = -1;
        const int rule = P.search_rule;
        for (int j = WS_TID; j < nn; j += WS_NT)
            if (alive[j]) {
                const double l = lb[j];
                const double key = rule == 0 ? l : (rule == 1 ? -(double)j : (double)j);
                if (l < cutoff && (bi < 0 || key < best)) { best = key; bi = j; }
            }
        block_argmin(best, bi, SMV(red), SMI(ired));
        if (bi < 0) { st = inc >= 0 ? BNB_OK : BNB_INFEASIBLE; break; }
        if (solves >= max_solves || nn + 2 > tr.cap_nodes || nr + 1 > tr.cap_recs) { st = BNB_CAPACITY; break; }
        // ---- bounds of the node (controller.py:273-298); the binary it would be branched on: the first unassigned one in the
        //      branching order (chronological = branch_in_time, controller.py:13-44, or the handle's static order); the
        //      eliminated prefix = the leading run of assigned binaries
        const int d = depth[bi];
        const unsigned int *bw = bits + (size_t)bi * tr.words, *mw = mask + (size_t)bi * tr.words;
        double first_free = (double)nb, first_in_order = (double)nb; int ff = -1, fo = -1;
        for (int j = WS_TID; j < nb; j += WS_NT) {
            const bool as = (mw[j >> 5] >> (j & 31)) & 1u;
            const double v = (double)((bw[j >> 5] >> (j & 31)) & 1u);
            lbv[j] = as ? v : 0.;
            ubv[j] = as ? v : 1.;
            if (!as && ff < 0) { ff = j; first_free = (double)j; }
        }
        block_argmin(first_free, ff, SMV(red), SMI(ired));
        const int d_elim = ff < 0 ? nb : ff;
        int jb = d_elim;
        if (RULE == 0 && P.border) {
            for (int p = WS_TID; p < nb; p += WS_NT) {
                const int j = P.border[p];
                if (!((mw[j >> 5] >> (j & 31)) & 1u) && fo < 0) { fo = p; first_in_order = (double)p; }
            }
            block_argmin(first_in_order, fo, SMV(red), SMI(ired));
            jb = fo < 0 ? nb : P.border[fo];
        }
        set_node_prefix_known(P, cx, d_elim);
        WS_SYNC();
        prof_mark(0);
        // ---- solve (K1), started from the node's OWN dual record: the multipliers (and proximal centre) of its
        //      parent, or its shifted dual solution for a warm-start root (controller.py:262-264, 426, 487);
        //      no record (root node, dual = None) = empty working set
        int memo = 0, memo_r0 = -1;
        {
            // rec <= -2: dual = None for the reference's bookkeeping (the shifted Farkas proof of an infeasible leaf no longer
            // holds, controller.py:555-558), but record -2 - rec still holds that shifted ray: its rows are where the new
            // proof (or the optimum) is most likely found, and any multipliers >= 0 are a valid start of the dual method
            const int r00 = rec[bi];
            const int r0 = r00 <= -2 ? -2 - r00 : r00;
            // children of this search share their parent's record: the second sibling takes the factor the first one built
            memo = (r0 >= 0 && bi >= nn0) ? ((r0 == memo_rec && min(d_elim, P.n_elim) == memo_d) ? 2 : 1) : 0;
            memo_r0 = r0;
            if (memo == 2) {
                const double *D = rdual + (size_t)r0 * P.n_rec;
                for (int i = WS_TID; i < P.n; i += WS_NT) SMV(yc)[i] = D[P.n_dual + i];      // the proximal centre load_ws would set
                WS_SYNC();
            } else if (r0 >= 0) {
                const double *D = rdual + (size_t)r0 * P.n_rec;
                const double *mu = D + P.off_mu, *nl = D + P.off_nulb, *nu_ = D + P.off_nuub;
                const int mc = P.mc;
                load_ws_from_multipliers(P, cx, [&](int r) { return r < mc ? mu[r] : nu_[r - mc] - nl[r - mc]; }, D + P.n_dual, k);
            } else {
                load_slot(P, cx, sp, k, true);
            }
        }
        prof_mark(1);
        int memo_saved = 0;
        const int qs = qp_solve(P, cx, k, xi, lbv, ubv, y, iters_s, iters_s + 1, memo, sp, memo_saved);
        if (memo == 1) { memo_rec = memo_saved ? memo_r0 : -1; memo_d = min(d_elim, P.n_elim); }
        if (qs == WS_ITER_LIMIT) { st = BNB_QP_LIMIT; break; }
        double *dual = rdual + (size_t)nr * P.n_rec;
        build_records(P, qs, SMV(yc), y, xi, lbv, ubv, prim, dual, cost_s, dobj_s, SMV(part), SMV(red));
        for (int j = WS_TID; j < P.n_rec - P.n_dual; j += WS_NT) dual[P.n_dual + j] = qs == WS_OPTIMAL && j < P.n ? SMV(yc)[j] : 0.;
        prof_mark(17);
        const double cost = *cost_s;
        if (WS_TID == 0) {
            lb[bi] = cost; rec[bi] = nr; rdobj[nr] = *dobj_s;
#ifdef WS_PROF
            // experiment builds: iterations | k after the rebuild << 12 | final k << 20 | infeasible << 28 | proximal passes << 29
            if (tr_i) { tr_i[2 * solves] = bi | (d << 16); tr_i[2 * solves + 1] = (*iters_s & 0xfff) | ((iters_s[2] & 0xff) << 12) | ((k & 0xff) << 20) | ((qs == WS_INFEASIBLE) << 28) | (((iters_s[2] >> 16) & 3) << 29); }
#else
            if (tr_i) { tr_i[2 * solves] = bi; tr_i[2 * solves + 1] = *iters_s; }
#endif
        }
        const int myrec = nr;
        iters += *iters_s; ksum += k; kmx = max(kmx, iters_s[1]); dsum += min(d_elim, P.n_elim); k0sum += iters_s[2] & 0xffff;
        ++nr; ++solves;
        bool integral = d == nb;
        if (RULE != 0 && cost < cutoff) {
            // conventional MIQP rule (controller.py:567-576): the unassigned binary j = t nub + i whose relaxed value u is the
            // most fractional, |u - rint(u)| largest, ties to the smaller j (np.argmax); pinned binaries count as 0.  The
            // node is integral (an incumbent) when that largest fractionality is <= BNB_INTEGRAL_TOL.
            const double *ubp = prim + (size_t)(P.T + 1) * P.nx + P.nuc;
            double fr = 0.; int fj = -1;
            for (int j = WS_TID; j < nb; j += WS_NT) {
                if ((mw[j >> 5] >> (j & 31)) & 1u) continue;
                const double u = ubp[(j / P.nub) * P.nu + j % P.nub], f = fabs(u - rint(u));
                if (fj < 0 || f > fr) { fr = f; fj = j; }
            }
            block_argmax(fr, fj, SMV(red), SMI(ired));
            integral = fj < 0 || fr <= BNB_INTEGRAL_TOL;
            jb = fj;
        }
        // ---- prune / incumbent / branch (branch_and_bound.py:476-489)
        if (cost >= cutoff) {
            // pruned: the node stays a leaf with its new bound
        } else if (integral) {
            inc = bi; ub = cost;
            double *ip = inc_primal + (size_t)inst * P.n_primal;
            for (int j = WS_TID; j < P.n_primal; j += WS_NT) ip[j] = prim[j];
        } else {
            // children [value 0, value 1] of binary jb = (t, i); bound += multiplier of the bound that moves (rule 0) or
            // = the parent's relaxation cost (conventional rule: no dual-bound inheritance)
            const double l0 = RULE == 0 ? cost + dual[P.off_nuub + jb] : cost, l1 = RULE == 0 ? cost + dual[P.off_nulb + jb] : cost;
            unsigned int *c0 = bits + (size_t)nn * tr.words, *c1 = c0 + tr.words;
            unsigned int *m0 = mask + (size_t)nn * tr.words, *m1 = m0 + tr.words;
            for (int w = WS_TID; w < tr.words; w += WS_NT) {
                const unsigned int b = bw[w], bit = (w == (jb >> 5)) ? (1u << (jb & 31)) : 0u;
                c0[w] = b & ~bit;
                c1[w] = b | bit;
                m0[w] = m1[w] = mw[w] | bit;
            }
            if (WS_TID == 0) {
                alive[bi] = 0;
                depth[nn] = d + 1; alive[nn] = 1; rec[nn] = myrec; lb[nn] = l0;
                depth[nn + 1] = d + 1; alive[nn + 1] = 1; rec[nn + 1] = myrec; lb[nn + 1] = l1;
            }
            nn += 2;
        }
        WS_SYNC();
        prof_mark(18);
    }
    if (WS_TID == 0) {
        tr.n_nodes[inst] = nn; tr.n_recs[inst] = nr;
        inc_cost[inst] = ub; inc_node[inst] = inc; n_solves[inst] = solves;
        if (totals) {
            atomicAdd(totals, (unsigned long long)solves); atomicAdd(totals + 1, (unsigned long long)iters);
            atomicAdd(totals + 2, (unsigned long long)ksum); atomicMax(totals + 3, (unsigned long long)kmx);
            atomicAdd(totals + 4, (unsigned long long)dsum); atomicAdd(totals + 5, (unsigned long long)k0sum);
        }
    }
    if (n_iters) *n_iters = (int)iters;
    WS_SYNC();
    return st;
}

template <int LANES, int RULE>
__device__ __forceinline__ void
bnb_body(const DevProblem &P, double *slot_d, int *slot_i, double *ybuf, double *scratch, int *work_counter, int n_slots,
           int n_inst, const double *__restrict__ x0, const int *__restrict__ active, const TreeView &tr,
           double tol, int max_solves,
           double *inc_cost, int *inc_node, double *inc_primal, int *n_solves, int *status_out, int *trace,
           unsigned long long *totals)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_inst[WS_MAXL];
    const int slot = blockIdx.x * LANES + WS_LANE;
    SlotPtrs sp = slot_ptrs(slot_d, slot_i, slot < n_slots ? slot : 0, P.n, P.ld);
    const Ctx cx = make_ctx(P, smem_raw, sp);
    init_shared_tables(P, cx);
    if (slot >= n_slots) return;                       // a lane without a solver state (after the CTA-wide barrier)
    double *y = ybuf + (size_t)slot * P.m;
    double *sc = scratch + (size_t)slot * bnb_scratch_doubles(P.nb, P.n_primal);
    int *iters_s = slot_i + (size_t)slot * slot_ints(P.n) + 2 * (P.n + 1) + 1;

    for (;;) {
        WS_SYNC();
        if (WS_TID == 0) s_inst[WS_LANE] = atomicAdd(work_counter, 1);
        WS_SYNC();
        const int inst = s_inst[WS_LANE];
        if (inst >= n_inst) break;
        if (active && !active[inst]) {
            if (WS_TID == 0) { inc_cost[inst] = INFINITY; inc_node[inst] = -1; n_solves[inst] = 0; status_out[inst] = BNB_INFEASIBLE; }
            continue;
        }
        const int st = bnb_instance<RULE>(P, cx, sp, y, sc, iters_s, inst, x0 + (size_t)inst * P.nx, tr, tol, max_solves,
                                    inc_cost, inc_node, inc_primal, n_solves, trace, totals);
        if (WS_TID == 0) status_out[inst] = st;
    }
}


#define WS_BNB_ARGS DevProblem P, double *slot_d, int *slot_i, double *ybuf, double *scratch, int *work_counter, int n_slots, \
    int n_inst, const double *__restrict__ x0, const int *__restrict__ active, TreeView tr, double tol, int max_solves, \
    double *inc_cost, int *inc_node, double *inc_primal, int *n_solves, int *status_out, int *trace, unsigned long long *totals
#define WS_BNB_PASS P, slot_d, slot_i, ybuf, scratch, work_counter, n_slots, n_inst, x0, active, tr, tol, max_solves, \
    inc_cost, inc_node, inc_primal, n_solves, status_out, trace, totals
#define WS_BNB_BODY(LANES, RULE, PLANT, FB) bnb_body<LANES, RULE>(WS_BNB_PASS)

// ---------------------------------------------------------------------------------------------
// K2 + K4: retain / shift identifiers / shift duals / re-evaluate the bounds / plant update
// ---------------------------------------------------------------------------------------------
#define SH_NT 256
#define SH_NW (SH_NT / 32)

// a warp asks L2 for the `n` doubles at p (one request per 128-byte line): the dual records of the tree shift are
// streamed from HBM once, and a leaf's loops would otherwise expose one DRAM latency each
__device__ __forceinline__ void warp_prefetch_l2(const double *p, int n, int lane) {
    for (int e = lane * 16; e < n; e += 32 * 16) asm volatile("prefetch.global.L2 [%0];" :: "l"(p + e));
}

// dst[e] = src[e], e < n, by one warp: eight independent loads in flight per lane (src and dst never overlap)
__device__ __forceinline__ void warp_copy(double *__restrict__ dst, const double *__restrict__ src, int n, int lane) {
    int e = lane;
    for (; e + 224 < n; e += 256) {
        double v[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) v[q] = src[e + 32 * q];
#pragma unroll
        for (int q = 0; q < 8; ++q) dst[e + 32 * q] = v[q];
    }
    for (; e + 96 < n; e += 128) {
        const double v0 = src[e], v1 = src[e + 32], v2 = src[e + 64], v3 = src[e + 96];
        dst[e] = v0; dst[e + 32] = v1; dst[e + 64] = v2; dst[e + 96] = v3;
    }
    for (; e < n; e += 32) dst[e] = src[e];
}

// doubles of shared scratch the shift needs with NT threads
__host__ __device__ __forceinline__ size_t shift_smem_doubles(const DevProblem &P, int nt) {
    // ... + one mbarrier per warp (TMA staging of the dual records), kept even so that what follows is 16-byte aligned
    return ((size_t)2 * P.nx + P.nu + P.nq + P.nr + P.nh + (size_t)(nt / 32) * (P.nh1 + P.nqT + P.nh + P.nq) + 8 + nt / 32 + 1) & ~(size_t)1;
}
// doubles of one staging buffer: the dual part of a record (the proximal centre behind it is not read by the shift)
__host__ __device__ __forceinline__ size_t shift_stage_doubles(const DevProblem &P) { return ((size_t)P.n_dual + 1) & ~(size_t)1; }

// warm start of ONE instance by the calling CTA (NT threads): shm = shared scratch (shift_smem_doubles),
// s_wsum (NT / 32 ints) and s_base (1 int) shared as well.
// Returns 0, or 1 if the retained leaves do not fit min(nt.cap_nodes, nt.cap_recs) (every retained leaf takes a node AND a
// dual record of the new tree): the instance is then switched off (active = 0, empty new tree) instead of continuing
// with an incomplete cover -- a truncated cover could report a suboptimal or "infeasible" MIQP as solved.
// LANE: the caller is a solver lane of WS_NT threads (fused loop): lane-local thread index and the lane's named barrier;
// otherwise a whole CTA of NT threads.
// stage_avail: doubles of shared memory behind the scratch (shm + shift_smem_doubles) that may hold staging buffers.  A warp
// with a buffer pulls the WHOLE dual record of its leaf into shared memory with one TMA bulk copy (cp.async.bulk,
// completion on the warp's mbarrier) and runs every loop of the shift on that copy: one DRAM / L2 latency per leaf instead
// of one per field of the record (HBM-bound stream, SURVEY 8d).  Warps without a buffer read the record in place; the
// arithmetic is the same either way.
template <int NT, bool LANE>
__device__ __forceinline__ int shift_instance(const DevProblem &P, double *shm, int stage_avail, int *s_wsum, int *s_base_p, int inst,
                                      const double *__restrict__ x0, const double *__restrict__ e0,
                                      const TreeView &ot, const double *__restrict__ inc_cost, const double *__restrict__ inc_primal,
                                      int *active, const TreeView &nt, double *x_next, double *u0_out)
{
    const int nx = P.nx, nu = P.nu, nub = P.nub, nuc = P.nuc, T = P.T, nh = P.nh, nh1 = P.nh1;
    const int nq = P.nq, nqT = P.nqT, nr_ = P.nr;
    const int tid_ = LANE ? WS_TID : (int)threadIdx.x;
    auto sync = [] { if (LANE) WS_SYNC(); else __syncthreads(); };
    const int lane = tid_ & 31, w = tid_ >> 5;
    // shared: x0 | u0 | e0 | Qx0 | Ru0 | res_mu | per-warp scratch (nh1 + nqT each)
    double *xs = shm, *us = xs + nx, *es = us + nu, *Qx = es + nx, *Ru = Qx + nq, *rmu = Ru + nr_;
    double *wscr = rmu + nh + (size_t)w * (nh1 + nqT + nh + nq);
#define s_base (*s_base_p)
    sync();
    const double *ip = inc_primal + (size_t)inst * P.n_primal;
    const bool on = (!active || active[inst]) && inc_cost[inst] < INFINITY;
    if (!on) {
        if (tid_ == 0) {
            if (active) active[inst] = 0;
            nt.n_nodes[inst] = 0; nt.n_recs[inst] = 0;
        }
        for (int j = tid_; j < nx; j += NT) if (x_next) x_next[(size_t)inst * nx + j] = x0[(size_t)inst * nx + j];
        for (int j = tid_; j < nu; j += NT) if (u0_out) u0_out[(size_t)inst * nu + j] = nan("");
        return 0;
    }
    for (int j = tid_; j < nx; j += NT) { xs[j] = x0[(size_t)inst * nx + j]; es[j] = e0 ? e0[(size_t)inst * nx + j] : 0.; }
    for (int j = tid_; j < nu; j += NT) us[j] = ip[(size_t)(T + 1) * nx + j];
    if (tid_ == 0) s_base = 0;
    sync();
    for (int i = tid_; i < nq; i += NT) { double s = 0.; for (int c = 0; c < nx; ++c) s += P.Q[i * nx + c] * xs[c]; Qx[i] = s; }
    for (int i = tid_; i < nr_; i += NT) { double s = 0.; for (int c = 0; c < nu; ++c) s += P.R[i * nu + c] * us[c]; Ru[i] = s; }
    for (int i = tid_; i < nh; i += NT) {
        double s = -P.h[i];
        for (int c = 0; c < nx; ++c) s += P.F[i * nx + c] * xs[c];
        for (int c = 0; c < nu; ++c) s += P.G[i * nu + c] * us[c];
        rmu[i] = s;
    }
    // plant update and applied input
    for (int j = tid_; j < nx; j += NT) if (x_next) x_next[(size_t)inst * nx + j] = ip[nx + j] + es[j];
    for (int j = tid_; j < nu; j += NT) if (u0_out) u0_out[(size_t)inst * nu + j] = us[j];
    sync();

    const size_t oo = (size_t)inst * ot.cap_nodes, on_ = (size_t)inst * nt.cap_nodes;
    const int nn = ot.n_nodes[inst];
    const int cap_new = nt.cap_nodes < nt.cap_recs ? nt.cap_nodes : nt.cap_recs;
    // ---- pass 1: _retain_leaf (controller.py:615-633) + ordered compaction + identifier shift (:476)
    for (int base = 0; base < nn; base += NT) {
        const int j = base + tid_;
        int keep = 0;
        if (j < nn && ot.alive[oo + j]) {
            keep = 1;
            const unsigned int b0 = ot.bits[(oo + j) * ot.words], m0 = ot.mask[(oo + j) * ot.words];
            for (int i = 0; i < nub; ++i)
                if (((m0 >> i) & 1u) && (double)((b0 >> i) & 1u) != us[nuc + i]) keep = 0;
        }
        const unsigned int bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_wsum[w] = __popc(bal);
        sync();
        int pre = s_base;
        for (int q = 0; q < w; ++q) pre += s_wsum[q];
        const int idx = pre + __popc(bal & ((1u << lane) - 1u));
        if (keep && idx < cap_new) {
            const unsigned int first = ot.mask[(oo + j) * ot.words] & (nub >= 32 ? 0xffffffffu : ((1u << nub) - 1u));
            const int dn = ot.depth[oo + j] - __popc(first);                       // assigned binaries that survive the shift
            nt.depth[on_ + idx] = dn; nt.alive[on_ + idx] = 1; nt.rec[on_ + idx] = j;   // rec = source node (pass 2 rewrites it)
            const unsigned int *srcb = ot.bits + (oo + j) * ot.words, *srcm = ot.mask + (oo + j) * ot.words;
            unsigned int *dstb = nt.bits + (on_ + idx) * nt.words, *dstm = nt.mask + (on_ + idx) * nt.words;
            for (int q = 0; q < nt.words; ++q) {
                // shift both bit strings right by nub bits (identifier shift, controller.py:476)
                const int sb = q * 32 + nub;
                const int wq = sb >> 5, sh = sb & 31;
                const unsigned int lob = wq < ot.words ? srcb[wq] : 0u, hib = wq + 1 < ot.words ? srcb[wq + 1] : 0u;
                const unsigned int lom = wq < ot.words ? srcm[wq] : 0u, him = wq + 1 < ot.words ? srcm[wq + 1] : 0u;
                const unsigned int vm = sh ? ((lom >> sh) | (him << (32 - sh))) : lom;
                const unsigned int vb = sh ? ((lob >> sh) | (hib << (32 - sh))) : lob;
                dstm[q] = vm;
                dstb[q] = vb & vm;
            }
        }
        sync();
        if (tid_ == 0) { int s = s_base; for (int q = 0; q < (NT / 32); ++q) s += s_wsum[q]; s_base = s; }
        sync();
    }
    if (s_base > cap_new) {
        // capacity of the new tree exceeded: never truncate the cover
        sync();
        if (tid_ == 0) { if (active) active[inst] = 0; nt.n_nodes[inst] = 0; nt.n_recs[inst] = 0; }
        return 1;
    }
    const int nnew = s_base;
    // ---- pass 2: one warp per retained leaf
    const size_t scr = shift_smem_doubles(P, NT), sbuf = shift_stage_doubles(P);
#if defined(WS_NO_STAGE)
    stage_avail = 0;
#endif
    // has_buf: the warp owns a staging buffer.  A leaf is staged only if its record starts 16-byte aligned, as cp.async.bulk
    // requires: the even record stride keeps every record of an aligned tree aligned, and the check per leaf covers trees on
    // any caller pointer.  Other leaves are read in place.
    const bool has_buf = (P.n_dual & 1) == 0 && stage_avail > 0 && (size_t)stage_avail >= (size_t)(w + 1) * sbuf;
    double *stage = shm + scr + (size_t)w * sbuf;
    uint64_t *bar = reinterpret_cast<uint64_t *>(shm + scr - (NT / 32 + 1)) + w;
    uint32_t par = 0;
    if (has_buf) {
        if (lane == 0) { mbar_init(bar, 1); fence_async_smem(); }
        __syncwarp();
    }
    // the bookkeeping of a leaf (source node -> record, bound, running objective, first-stage bits) is a chain of dependent
    // loads: it is fetched one leaf AHEAD, while the current leaf's record is in flight / being processed
    int j_n = 0, ro_n = -1; double lb_n = 0., dobj_n = 0.; unsigned int b0_n = 0u, m0_n = 0u;
    auto fetch_leaf = [&](int ix) {
        j_n = nt.rec[on_ + ix];
        ro_n = ot.rec[oo + j_n];
        lb_n = ot.lb[oo + j_n];
        b0_n = ot.bits[(oo + j_n) * ot.words]; m0_n = ot.mask[(oo + j_n) * ot.words];
        dobj_n = ro_n >= 0 ? ot.rec_dobj[(size_t)inst * ot.cap_recs + ro_n] : 0.;
    };
    if (w < nnew) fetch_leaf(w);
    for (int idx = w; idx < nnew; idx += (NT / 32)) {
        const int j = j_n, ro = ro_n;
        const double lbo = lb_n, dobj_o = dobj_n;
        const unsigned int b0 = b0_n, m0 = m0_n;
        const int nx_idx = idx + (NT / 32);
        (void)j;
        double *E = nt.rec_dual + ((size_t)inst * nt.cap_recs + idx) * P.n_rec;
        if (ro < 0) {
            // dual = None (controller.py:556-558 on the previous step, never solved since): trivial bound
            if (nx_idx < nnew) fetch_leaf(nx_idx);
            for (int e = lane; e < P.n_rec; e += 32) E[e] = 0.;
            if (lane == 0) { nt.lb[on_ + idx] = 0.; nt.rec[on_ + idx] = -1; nt.rec_dobj[(size_t)inst * nt.cap_recs + idx] = 0.; }
            continue;
        }
        const double *Dg = ot.rec_dual + ((size_t)inst * ot.cap_recs + ro) * P.n_rec;
        const bool staged = has_buf && ((uintptr_t)Dg & 15) == 0;
        if (staged) {
            __syncwarp();                                  // every lane is done with the previous leaf's copy
            if (lane == 0) {
                fence_async_smem();
                mbar_expect_tx(bar, (uint32_t)(P.n_dual * 8));
                bulk_g2s(stage, Dg, (uint32_t)(P.n_dual * 8), bar);
            }
        } else {
            warp_prefetch_l2(Dg, P.n_dual, lane);
        }
        if (nx_idx < nnew) {   // ... the bookkeeping of the leaf this warp takes next, and its record on the way to L2
            fetch_leaf(nx_idx);
            if (ro_n >= 0) warp_prefetch_l2(ot.rec_dual + ((size_t)inst * ot.cap_recs + ro_n) * P.n_rec, P.n_dual, lane);
        }
        for (int e = P.n_dual + lane; e < P.n_rec; e += 32) E[e] = 0.;          // a shifted root starts from the centre 0
        const double *D = Dg;
        if (staged) { mbar_wait(bar, par); par ^= 1u; D = stage; }
        double acc = 0.;                     // pi_sum + pi3, lane-partial
        // lam: drop t = 0, append zero ; pi3 = -lam'_0 . e0 (controller.py:544)
        {
            const double *s = D + P.off_lam + nx; double *t = E + P.off_lam;
            for (int e = lane; e < T * nx; e += 32) { const double v = s[e]; t[e] = v; if (e < nx) acc -= v * es[e]; }
            for (int e = lane; e < nx; e += 32) t[T * nx + e] = 0.;
        }
        // nu_lb, nu_ub: complementarity terms with the OLD identifier's bounds at t = 0 (controller.py:703-709)
        {
            const double *sl = D + P.off_nulb, *su = D + P.off_nuub;
            double *tl = E + P.off_nulb, *tu = E + P.off_nuub;
            warp_copy(tl, sl + nub, (T - 1) * nub, lane); warp_copy(tu, su + nub, (T - 1) * nub, lane);
            for (int e = lane; e < nub; e += 32) {
                tl[(T - 1) * nub + e] = 0.; tu[(T - 1) * nub + e] = 0.;
                const double bit = (double)((b0 >> e) & 1u);
                const bool as = (m0 >> e) & 1u;
                const double l0 = as ? bit : 0., u0b = as ? bit : 1.;
                const double vu = us[nuc + e];
                acc -= (l0 - vu) * sl[e] + (vu - u0b) * su[e];
            }
        }
        // sigma: suboptimality term |sigma_0 / 2 - R u0|^2 - |R u0|^2
        {
            const double *s = D + P.off_sigma; double *t = E + P.off_sigma;
            for (int e = lane; e < (T - 1) * nr_; e += 32) t[e] = s[nr_ + e];
            for (int e = lane; e < nr_; e += 32) { t[(T - 1) * nr_ + e] = 0.; const double a = .5 * s[e] - Ru[e]; acc += a * a - Ru[e] * Ru[e]; }
        }
        // rho: rho'_{T-1} = M_rho rho_T (controller.py:96, 662-664)
        {
            const double *s = D + P.off_rho; double *t = E + P.off_rho;
            warp_copy(t, s + nq, (T - 1) * nq, lane);
            for (int e = lane; e < nq; e += 32) { const double a = .5 * s[e] - Qx[e]; acc += a * a - Qx[e] * Qx[e]; }
            double *rT = wscr;                              // rho_T staged for the small mat-vec
            for (int e = lane; e < nqT; e += 32) { const double v = s[T * nq + e]; rT[e] = v; acc += .25 * v * v; t[T * nq + e] = 0.; }
            __syncwarp();
            for (int i = lane; i < nq; i += 32) {
                double v = 0.;
                for (int c = 0; c < nqT; ++c) v += P.Mrho[i * nqT + c] * rT[c];
                t[(T - 1) * nq + i] = v; acc -= .25 * v * v;
            }
        }
        // mu: mu'_{T-2} = M_mu mu_{T-1} (controller.py:186-227, 662-664)
        {
            const double *s = D + P.off_mu; double *t = E + P.off_mu;
            warp_copy(t, s + nh, (T - 2) * nh, lane);
            for (int e = lane; e < nh; e += 32) acc -= rmu[e] * s[e];
            double *mT = wscr + nqT;
            int nz = 0;
            for (int e = lane; e < nh1; e += 32) { const double v = s[(T - 1) * nh + e]; mT[e] = v; nz |= (v != 0.) ? 1 : 0; acc += P.h1[e] * v; t[(T - 1) * nh + e] = 0.; }
            __syncwarp();
            // A leaf that has been shifted before has mu_{T-1} = 0 (written just above, one step ago): M_mu mu_{T-1} is then
            // +0 in every entry whatever the order of the sums, and the nh1 x nh operator -- 29 KB streamed from L2 by every
            // leaf, 43 % of the stall samples of this kernel (profiles/r02b_shift_tree_kernel_ncu_summary.txt) -- is not read.
            const bool any_mu = __any_sync(0xffffffffu, nz) != 0;
            // M_mu stored transposed: the lanes of a warp read consecutive words, four independent chains per lane
            for (int i = lane; i < nh; i += 32) {
                double v0 = 0., v1 = 0., v2 = 0., v3 = 0.;
                const double *mc_ = P.MmuT + i;
                int c = 0;
                if (any_mu) {
                    for (; c + 3 < nh1; c += 4) {
                        v0 += __ldg(mc_ + (size_t)c * nh) * mT[c]; v1 += __ldg(mc_ + (size_t)(c + 1) * nh) * mT[c + 1];
                        v2 += __ldg(mc_ + (size_t)(c + 2) * nh) * mT[c + 2]; v3 += __ldg(mc_ + (size_t)(c + 3) * nh) * mT[c + 3];
                    }
                    for (; c < nh1; ++c) v0 += __ldg(mc_ + (size_t)c * nh) * mT[c];
                }
                const double v = (v0 + v1) + (v2 + v3);
                t[(T - 2) * nh + i] = v; acc -= P.h[i] * v;
            }
            __syncwarp();
        }
        acc = warp_sum(acc);
        if (lane == 0) {
            double obj = dobj_o + acc;
            obj = obj > 0. ? obj : 0.;                     // controller.py:546
            double lbn; int rn = idx;
            if (!isinf(lbo)) lbn = obj;                    // :550-551
            else if (obj <= 0.) { lbn = 0.; rn = -2 - idx; }   // :555-558: dual = None; the shifted ray stays in record idx as a START for the node's QP
            else lbn = INFINITY;
            nt.lb[on_ + idx] = lbn; nt.rec[on_ + idx] = rn; nt.rec_dobj[(size_t)inst * nt.cap_recs + idx] = obj;
        }
    }
    if (has_buf) {
        // the barrier's memory goes back to the solver (LANE) / is initialised again for the next instance: invalidate it
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" :: "r"(smem_u32(bar)) : "memory");
    }
    sync();
    if (tid_ == 0) { nt.n_nodes[inst] = nnew; nt.n_recs[inst] = nnew; }
    return 0;
#undef s_base
}

#if WS_TU_HAS(0)
__global__ void __launch_bounds__(SH_NT)
shift_tree_kernel(DevProblem P, int n_inst, const double *__restrict__ x0, const double *__restrict__ e0,
                  TreeView ot, const double *__restrict__ inc_cost, const double *__restrict__ inc_primal,
                  int *active, TreeView nt, double *x_next, double *u0_out, int stage_avail)
{
    extern __shared__ __align__(16) double shm[];
    __shared__ int s_wsum[SH_NW];
    __shared__ int s_base_v;
    for (int inst = blockIdx.x; inst < n_inst; inst += gridDim.x) {
        __syncthreads();
        shift_instance<SH_NT, false>(P, shm, stage_avail, s_wsum, &s_base_v, inst, x0, e0, ot, inc_cost, inc_primal, active, nt, x_next, u0_out);
    }
}
#endif

// scratch + as many staging buffers as warps, if the device's shared memory holds them (else fewer; 0 = none)
__host__ inline size_t shift_smem_bytes(const DevProblem &P, size_t optin, int *stage_avail) {
    const size_t scr = shift_smem_doubles(P, SH_NT), sbuf = shift_stage_doubles(P);
    size_t nb = SH_NT / 32;
#if defined(WS_NO_STAGE)
    nb = 0;
#endif
    while (nb > 0 && (scr + nb * sbuf) * sizeof(double) > optin) --nb;
    *stage_avail = (int)(nb * sbuf);
    return sizeof(double) * (scr + nb * sbuf);
}


// ---------------------------------------------------------------------------------------------
// Fused closed loop (K3 + K2/K4 of many receding-horizon steps in ONE launch).
// Restates the experiment driver notebooks/cart_pole_with_walls/statistical_analysis.py:93-196 (linear
// plant + model error, no Gurobi legs) for a batch of independent instances WITHOUT a barrier between
// the steps of different instances: a task is (instance, its next step); CTAs pop tasks from a queue in
// global memory, run branch and bound + warm-start construction + plant update for that step, and push
// the instance back.  An instance is owned by one CTA at a time; its trees and state live in global
// memory, so any CTA can continue it.  Results are identical to stepping the batch in lock step.
// ---------------------------------------------------------------------------------------------
struct LoopView {
    int n_steps, warm, fresh, par;
    int *q;                 // [0] head, [1] tail, [2 ...] items
    int *step_of;           // [n_inst]
    double *x;              // [2][n_inst][nx]
    const double *e;        // [n_steps][n_inst][nx] or null
    int *active;            // [n_inst]
    double *log_cost;       // [n_steps][n_inst]
    double *log_u0;         // [n_steps][n_inst][nu]
    int *log_solves;        // [n_steps][n_inst]
    int *log_status;        // [n_steps][n_inst]
    int *log_cover;         // [n_steps][n_inst] or null: roots of the tree the shift of the step built
    int *log_lapsed;        // [n_steps][n_inst] or null: of those, roots whose Farkas proof lapsed in the shift (rec <= -2)
    int *log_iters;         // [n_steps][n_inst] or null: active-set iterations of the step's branch and bound
    // host mailbox (wshmpc_mailbox; all null = the plant is advanced on the device).  mb_* point into pinned, mapped HOST
    // memory and are read / written with system-scope ordering; mb_stage is device scratch [n_inst][nx].
    volatile int *mb_in_step, *mb_out_step, *mb_stop;
    const volatile double *mb_in_x, *mb_in_e;
    double *mb_out_u0, *mb_out_x1, *mb_out_cost;
    int *mb_out_status;
    double *mb_stage;
    unsigned long long mb_timeout_ns;   // a lane gives up on a silent host after this long (the launch then drains)
};
#define BNB_HOST_ABORT 4          // mailbox mode: the host stopped answering (stop flag or time-out)

#if WS_TU_HAS(0)
__global__ void loop_init_kernel(int n_inst, int n_items, LoopView L)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    // q: [0] tasks completed, [1] lowest step with unclaimed tasks (hint), [4 + s] head of step s, [4 + S + s] tail of
    // step s, [4 + 2 S + s n_inst + pos] instances ready for step s in the order they became ready
    const int S = L.n_steps + (L.mb_in_step ? 1 : 0);       // mailbox mode: one more level (the warm start after the last answer)
    if (i == 0) { L.q[0] = 0; L.q[1] = 0; L.q[2] = 0; L.q[3] = 0; }
    if (i < S) { L.q[4 + i] = 0; L.q[4 + S + i] = i == 0 ? n_inst : 0; }
    if (i < n_items) L.q[4 + 2 * S + i] = i < n_inst ? i : -1;
    if (i < n_inst) L.step_of[i] = 0;
}
#endif

__device__ __forceinline__ void init_root(const TreeView &tr, int k)
{
    const size_t o = (size_t)k * tr.cap_nodes;
    tr.n_nodes[k] = 1; tr.n_recs[k] = 0;
    tr.depth[o] = 0; tr.alive[o] = 1; tr.rec[o] = -1; tr.lb[o] = -INFINITY;
    for (int w = 0; w < tr.words; ++w) { tr.bits[o * tr.words + w] = 0u; tr.mask[o * tr.words + w] = 0u; }
}

// MIP start (feedforward_miqp's ub_guess, controller.py:552-556): node 0 = the guess, every binary j pinned to rint(g(j))
// (a value of 0 or 1), lb = -inf and no record (solved from the empty working set, first under best-first); node 1 = the
// root.  Threads tid = 0 .. nt - 1 of the caller share the work; the caller provides the barrier.
template <class Guess>
__device__ __forceinline__ void init_guess(const TreeView &tr, int k, int nb, Guess g, int tid, int nt)
{
    const size_t o = (size_t)k * tr.cap_nodes;
    for (int w = tid; w < tr.words; w += nt) {
        unsigned int b = 0u, m = 0u;
        for (int q = 0; q < 32 && 32 * w + q < nb; ++q) {
            m |= 1u << q;
            if (rint(g(32 * w + q)) != 0.) b |= 1u << q;
        }
        tr.bits[o * tr.words + w] = b; tr.mask[o * tr.words + w] = m;
        tr.bits[(o + 1) * tr.words + w] = 0u; tr.mask[(o + 1) * tr.words + w] = 0u;
    }
    if (tid == 0) {
        tr.n_nodes[k] = 2; tr.n_recs[k] = 0;
        tr.depth[o] = nb; tr.alive[o] = 1; tr.rec[o] = -1; tr.lb[o] = -INFINITY;
        tr.depth[o + 1] = 0; tr.alive[o + 1] = 1; tr.rec[o + 1] = -1; tr.lb[o + 1] = -INFINITY;
    }
}

#if WS_TU_HAS(0)
// wshmpc_tree_init_guess: [guess, root] for every instance with has[k] != 0 (has = null: all), the root alone otherwise
__global__ void init_guess_kernel(int n_inst, int nb, TreeView tr, const double *__restrict__ guess, const int *__restrict__ has)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_inst) return;
    if (has && !has[k]) { init_root(tr, k); return; }
    const double *gk = guess + (size_t)k * nb;
    init_guess(tr, k, nb, [&](int j) { return gk[j]; }, 0, 1);
}
#endif

// Fallback through infeasible MIQPs (wshmpc_fallback): caller-owned buffers, so that plans survive launches and windows.
struct FallbackView {
    int max_hold;            // H: steps an instance may run on its last plan, 0 <= H <= T - 1
    double *plan;            // [n_inst][n_primal] primal record of the last step with an incumbent
    int *age;                // [n_inst] steps since that step, -1 = no plan
    double *app_cost;        // [n_inst] applied pair: +inf = the instance leaves the loop, finite otherwise
    double *app_primal;      // [n_inst][n_primal] (a fallback step defines x_0, x_1 and u_0 only)
    int *hold;               // [n_inst] of the step: 0 the incumbent, a > 0 input u_a of the plan, -2 the law, -1 none
    int max_law;             // L: consecutive steps an instance may run on the terminal law, 0 = no law
    const double *law_K;     // [law_sets][nu][nx] the law's gain (null when L = 0)
    int *law_n;              // [n_inst] law steps since the last incumbent (null when L = 0)
    int law_sets;            // 0 or 1: one gain (and offset) for all instances; n_inst: set i for instance i
    const double *law_k;     // [law_sets][nu] the law's offset, or null (no offset)
    const double *law_lo;    // [nu] lower and upper bounds of the law's input, or both null (no saturation)
    const double *law_hi;
};

// u_r = sat_[lo_r, hi_r]((K_i x)_r + k_ir), K_i and k_i set i = inst of the law (set 0 when there is one): fused
// multiply-adds over the columns in order, then the offset, then the clamp (every caller and every thread gets the same
// bits).  The offset is added only when there is one (adding +0. would turn a -0. into +0.); the clamp leaves NaN and a
// component with infinite bounds as they are.
__device__ __forceinline__ double law_input(const FallbackView &fb, int inst, const double *__restrict__ x, int r, int nx, int nu)
{
    const size_t set = fb.law_sets > 1 ? (size_t)inst : 0;
    const double *__restrict__ K = fb.law_K + set * nu * nx;
    double s = 0.;
    for (int c = 0; c < nx; ++c) s = __fma_rn(K[r * nx + c], x[c], s);
    if (fb.law_k) s = __dadd_rn(s, fb.law_k[set * nu + r]);
    if (fb.law_lo) {
        const double lo = fb.law_lo[r], hi = fb.law_hi[r];
        s = s < lo ? lo : (s > hi ? hi : s);
    }
    return s;
}

// The fallback policy for instance `inst` after its branch and bound (status st; the fused loop and wshmpc_fallback_step):
//   incumbent                            plan <- incumbent, age 0, law_n 0, applied pair = incumbent, hold 0;
//   status 1, a plan with age + 1 <= H   age += 1, applied u_0 = u_age of the plan, x_1 = A x + B u_0 (fused multiply-adds
//                                        in a fixed order, so that every caller gets the same bits), hold = age;
//   status 1, otherwise, law_n + 1 <= L  law_n += 1, applied u_0 = the law's input (law_input), x_1 = A x + B u_0 (the same
//                                        order), age kept, hold -2;
//   otherwise                            applied cost +inf (K2 + K4 switch the instance off), hold -1.
// Threads tid = 0 .. nt - 1 share the copies; `sync` is the callers' barrier (age and law_n are read by all before thread 0
// writes them).  With L = 0, law_n and the law's gain, offset and bounds are never touched.
template <class Sync>
__device__ __forceinline__ void fallback_apply(const DevProblem &P, const FallbackView &fb, int inst, bool live, int st,
                                               const double *__restrict__ x, const double *__restrict__ inc_cost,
                                               const double *__restrict__ inc_primal, int *hold, int tid, int nt, Sync sync)
{
    const int nx = P.nx, nu = P.nu, np_ = P.n_primal;
    const size_t o = (size_t)inst * np_;
    const int a = fb.age[inst];
    int mode = !live ? 2 : inc_cost[inst] < INFINITY ? 0 : (st == BNB_INFEASIBLE && a >= 0 && a + 1 <= fb.max_hold) ? 1 : 2;
    const int n = fb.max_law > 0 ? fb.law_n[inst] : 0;
    if (mode == 2 && live && st == BNB_INFEASIBLE && n + 1 <= fb.max_law) mode = 3;
    if (mode == 0) {
        for (int j = tid; j < np_; j += nt) { const double v = inc_primal[o + j]; fb.plan[o + j] = v; fb.app_primal[o + j] = v; }
    } else if (mode == 1) {
        const double *u = fb.plan + o + (size_t)(P.T + 1) * nx + (size_t)(a + 1) * nu;
        double *ap = fb.app_primal + o;
        for (int j = tid; j < nx; j += nt) {
            double s = 0.;
            for (int c = 0; c < nx; ++c) s = __fma_rn(P.A[j * nx + c], x[c], s);
            for (int c = 0; c < nu; ++c) s = __fma_rn(P.B[j * nu + c], u[c], s);
            ap[j] = x[j]; ap[nx + j] = s;
        }
        for (int j = tid; j < nu; j += nt) ap[(size_t)(P.T + 1) * nx + j] = u[j];
    } else if (mode == 3) {
        // every thread forms the inputs it needs from K x itself: no barrier between u and x_1
        double *ap = fb.app_primal + o;
        for (int j = tid; j < nx; j += nt) {
            double s = 0.;
            for (int c = 0; c < nx; ++c) s = __fma_rn(P.A[j * nx + c], x[c], s);
            for (int c = 0; c < nu; ++c) s = __fma_rn(P.B[j * nu + c], law_input(fb, inst, x, c, nx, nu), s);
            ap[j] = x[j]; ap[nx + j] = s;
        }
        for (int j = tid; j < nu; j += nt) ap[(size_t)(P.T + 1) * nx + j] = law_input(fb, inst, x, j, nx, nu);
    }
    sync();
    if (tid == 0) {
        if (mode == 0) { fb.age[inst] = 0; fb.app_cost[inst] = inc_cost[inst]; hold[inst] = 0; if (fb.max_law > 0) fb.law_n[inst] = 0; }
        else if (mode == 1) { fb.age[inst] = a + 1; fb.app_cost[inst] = 0.; hold[inst] = a + 1; }
        else if (mode == 3) { fb.law_n[inst] = n + 1; fb.app_cost[inst] = 0.; hold[inst] = -2; }
        else { fb.app_cost[inst] = INFINITY; hold[inst] = -1; }
    }
}

#if WS_TU_HAS(0)
// wshmpc_fallback_step: one thread per instance
__global__ void fallback_step_kernel(DevProblem P, int n_inst, FallbackView fb, const double *__restrict__ x, const int *__restrict__ active,
                                     const int *__restrict__ status, const double *__restrict__ inc_cost, const double *__restrict__ inc_primal)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_inst) return;
    fallback_apply(P, fb, i, !active || active[i] != 0, status[i], x + (size_t)i * P.nx, inc_cost, inc_primal, fb.hold, 0, 1, [] {});
}
#endif

// The cover and lapsed logs of row `lo` (wshmpc_loop d_log_cover, d_log_lapsed), right after a shift_instance of the lane
// built `nt`: its roots, and how many of them carry a Farkas proof the shift let lapse.  Writes nothing when neither log
// is wanted.
__device__ __forceinline__ void log_shifted_tree(const DevProblem &P, const Ctx &cx, const LoopView &L, const TreeView &nt,
                                                 int inst, size_t lo)
{
    if (!L.log_cover && !L.log_lapsed) return;
    WS_SYNC();                                         // n_nodes (thread 0) and rec (every warp) of the new tree
    const int nn = nt.n_nodes[inst];
    if (WS_TID == 0 && L.log_cover) L.log_cover[lo] = nn;
    if (L.log_lapsed) {
        const int *rec = nt.rec + (size_t)inst * nt.cap_nodes;
        double c = 0.;
        for (int j = WS_TID; j < nn; j += WS_NT) c += rec[j] <= -2 ? 1. : 0.;
        c = block_sum(c, SMV(red));
        if (WS_TID == 0) L.log_lapsed[lo] = (int)c;
    }
}

// PLANT: the state advances through the nonlinear plant on the device (wshmpc_closed_loop_plant, `pv`) instead of the linear
// model plus an additive error; the kernels without it carry no code of the plant and never read `pv`.
// FB: the fallback policy (wshmpc_closed_loop_fallback, `fv`): after K3 the plant and K2 + K4 read the applied pair
// fv.app_cost / fv.app_primal instead of the incumbent; the kernels without it never read `fv`.
template <int LANES, int RULE, bool PLANT, bool FB>
__device__ __forceinline__ void
closed_loop_body(const DevProblem &P, double *slot_d, int *slot_i, double *ybuf, double *scratch, const LoopView &L, int n_slots, int n_inst,
                   const TreeView &t0, const TreeView &t1, double tol, int max_solves,
                   double *inc_cost, int *inc_node, double *inc_primal, int *n_solves, int *status_out,
                   unsigned long long *totals, const PlantView &pv, const FallbackView &fv)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_inst_[WS_MAXL];
    const int slot = blockIdx.x * LANES + WS_LANE;
    SlotPtrs sp = slot_ptrs(slot_d, slot_i, slot < n_slots ? slot : 0, P.n, P.ld);
    const Ctx cx = make_ctx(P, smem_raw, sp);
    init_shared_tables(P, cx);
    if (slot >= n_slots) return;                       // a lane without a solver state (after the CTA-wide barrier)
#define s_inst s_inst_[WS_LANE]
    double *y = ybuf + (size_t)slot * P.m;
    double *sc = scratch + (size_t)slot * bnb_scratch_doubles(P.nb, P.n_primal);
    int *iters_s = slot_i + (size_t)slot * slot_ints(P.n) + 2 * (P.n + 1) + 1;
    // Mailbox mode (L.mb_in_step != null): the host is in the loop EVERY step of every instance, still without a barrier
    // between instances.  Level t of an instance = [wait for the host's answer to step t - 1, then its warm start
    // (K2 + K4) with the measured state and model error the host sent] + [B&B of step t, published to the host]; there is
    // one level more than steps (the warm start after the last answer), so a launch ends in the same state as the
    // device-resident loop.
    const bool mbx = L.mb_in_step != nullptr;
    const int S = L.n_steps + (mbx ? 1 : 0);
    const int total = n_inst * S;
    const size_t xs = (size_t)n_inst * P.nx;
    prof_mark(127);

    for (;;) {
        WS_SYNC();
        if (WS_TID == 0) {
            // pop a ready task of the LOWEST step: the instance that lags behind never waits in a queue, so the launch
            // ends with the longest chain of solves of one instance, not with that chain plus its queueing delays
            volatile int *q = L.q;
            int *head = L.q + 4, *items = L.q + 4 + 2 * S;
            volatile int *tail = L.q + 4 + S;
            int inst = -1;
            for (;;) {
                int s = q[1];
                bool claimed = false;
                while (s < S) {
                    const int hd = ((volatile int *)head)[s];
                    if (hd >= n_inst) { if (s == q[1]) atomicMax(L.q + 1, s + 1); ++s; continue; }
                    if (hd < tail[s]) {
                        if (atomicCAS(head + s, hd, hd + 1) == hd) {
                            volatile int *item = items + (size_t)s * n_inst + hd;
                            while ((inst = *item) < 0) __nanosleep(64);
                            claimed = true;
                            break;
                        }
                        continue;                          // lost the race: look at the same step again
                    }
                    ++s;
                }
                if (claimed || q[0] >= total) break;
                __nanosleep(256);
            }
            s_inst = inst;
        }
        WS_SYNC();
        const int inst = s_inst;
        prof_mark(20);
        if (inst < 0) break;
        __threadfence();                                   // acquire: drop stale L1 lines of the instance's data
        const int t = L.step_of[inst];
        if (mbx && t > 0) {
            // the warm start of step t - 1, once the host has answered it
            const int ts = t - 1, ps = (L.par + ts) & 1;
            const TreeView &cur = ps ? t1 : t0;
            const TreeView &nxt = ps ? t0 : t1;
            const double *xc = L.x + (size_t)ps * xs;
            double *xn = L.x + (size_t)(ps ^ 1) * xs;
            const bool live = L.active[inst] != 0;
            if (live) {
                if (WS_TID == 0) {
                    unsigned long long t_begin = 0, now = 0;
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_begin));
                    int ok = 1;
                    while (L.mb_in_step[inst] < t) {
                        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                        if (*L.mb_stop != 0 || now - t_begin > L.mb_timeout_ns) { ok = 0; break; }
                        __nanosleep(1000);
                    }
                    __threadfence_system();
                    s_inst = ok;
                }
                WS_SYNC();
                const int ok = s_inst;
                WS_SYNC();
                if (ok) {
                    for (int j = WS_TID; j < P.nx; j += WS_NT) {
                        xn[(size_t)inst * P.nx + j] = L.mb_in_x[(size_t)inst * P.nx + j];
                        L.mb_stage[(size_t)inst * P.nx + j] = L.mb_in_e[(size_t)inst * P.nx + j];
                    }
                } else {
                    for (int j = WS_TID; j < P.nx; j += WS_NT) { xn[(size_t)inst * P.nx + j] = xc[(size_t)inst * P.nx + j]; L.mb_stage[(size_t)inst * P.nx + j] = 0.; }
                    if (WS_TID == 0) { inc_cost[inst] = INFINITY; status_out[inst] = BNB_HOST_ABORT; L.log_status[(size_t)ts * n_inst + inst] = BNB_HOST_ABORT; }
                }
            } else {
                for (int j = WS_TID; j < P.nx; j += WS_NT) xn[(size_t)inst * P.nx + j] = xc[(size_t)inst * P.nx + j];
            }
            WS_SYNC();
            const int ovf = shift_instance<WS_NT, true>(P, SMV(pool), P.so.pool_sz - (int)shift_smem_doubles(P, WS_NT), SMI(ired), SMI(ired) + 16, inst, xc, L.mb_stage, cur, inc_cost, inc_primal,
                                                  L.active, nxt, nullptr, L.log_u0 + (size_t)ts * n_inst * P.nu);
            if (ovf && WS_TID == 0) { status_out[inst] = BNB_CAPACITY; L.log_status[(size_t)ts * n_inst + inst] = BNB_CAPACITY; }
            log_shifted_tree(P, cx, L, nxt, inst, (size_t)ts * n_inst + inst);
            prof_mark(19);
            WS_SYNC();
        }
        if (t < L.n_steps) {
            const int par = (L.par + t) & 1;
            const TreeView &cur = par ? t1 : t0;
            const TreeView &nxt = par ? t0 : t1;
            const double *xc = L.x + (size_t)par * xs;
            double *xn = L.x + (size_t)(par ^ 1) * xs;
            if (!L.warm || (t == 0 && L.fresh)) {
                if (RULE != 0 && P.node_rule == BNB_RULE_MIQP_START && !(t == 0 && L.fresh) && L.active[inst] && inc_cost[inst] < INFINITY) {
                    // MIP start: the previous step's incumbent binaries shifted by one step, zero at the end
                    // (shift_binary_solution, controller.py:586-588)
                    const double *ub1 = inc_primal + (size_t)inst * P.n_primal + (size_t)(P.T + 1) * P.nx + P.nu + P.nuc;
                    const int T = P.T, nub = P.nub, nu = P.nu;
                    init_guess(cur, inst, P.nb, [&](int j) { const int tt = j / nub; return tt < T - 1 ? ub1[tt * nu + j % nub] : 0.; },
                               WS_TID, WS_NT);
                } else if (WS_TID == 0) {
                    init_root(cur, inst);
                }
                WS_SYNC();
            }
            int st, it = 0;
            if (!L.active[inst]) {
                if (WS_TID == 0) { inc_cost[inst] = INFINITY; inc_node[inst] = -1; n_solves[inst] = 0; }
                st = BNB_INFEASIBLE;
                WS_SYNC();
            } else {
                st = bnb_instance<RULE>(P, cx, sp, y, sc, iters_s, inst, xc + (size_t)inst * P.nx, cur, tol, max_solves,
                                  inc_cost, inc_node, inc_primal, n_solves, nullptr, totals, &it);
            }
            if (WS_TID == 0) {
                status_out[inst] = st;
                const size_t lo = (size_t)t * n_inst + inst;
                L.log_cost[lo] = inc_cost[inst]; L.log_solves[lo] = n_solves[inst]; L.log_status[lo] = st;
                if (L.log_iters) L.log_iters[lo] = it;
            }
            WS_SYNC();
            // the pair the plant and K2 + K4 apply: the incumbent, or under FB the policy's choice
            const double *a_cost = inc_cost, *a_primal = inc_primal;
            if (FB) {
                fallback_apply(P, fv, inst, L.active[inst] != 0, st, xc + (size_t)inst * P.nx, inc_cost, inc_primal,
                               fv.hold + (size_t)t * n_inst, WS_TID, WS_NT, [] { WS_SYNC(); });
                WS_SYNC();
                a_cost = fv.app_cost; a_primal = fv.app_primal;
            }
            if (PLANT && !mbx) {
                // x_meas = Phi(x_t, u0[fc_index]) (+ d_e[t]) is the next state; e = x_meas - x_1|t corrects the warm start,
                // handed over through pv.stage like the mailbox's answer.  Without an incumbent the state is kept.
                if (WS_TID == 0) {
                    const double *xi = xc + (size_t)inst * 4;
                    double *xo = xn + (size_t)inst * 4, *ei = pv.stage + (size_t)inst * 4;
                    if (L.active[inst] != 0 && a_cost[inst] < INFINITY) {
                        const double *ip = a_primal + (size_t)inst * P.n_primal;
                        double x[4] = {xi[0], xi[1], xi[2], xi[3]};
                        cartpole_walls_step(pv.prm + (pv.n_sets == 1 ? 0 : (size_t)inst * WS_PLANT_NPARAM), x,
                                            ip[(size_t)(P.T + 1) * P.nx + pv.fc_index], pv.h, pv.n_sub);
                        const double *de = L.e ? L.e + (size_t)t * xs + (size_t)inst * 4 : nullptr;
                        for (int j = 0; j < 4; ++j) {
                            const double xm = de ? __dadd_rn(x[j], de[j]) : x[j];
                            xo[j] = xm; ei[j] = __dsub_rn(xm, ip[4 + j]);
                        }
                    } else {
                        for (int j = 0; j < 4; ++j) { xo[j] = xi[j]; ei[j] = 0.; }
                    }
                    if (pv.log_x) for (int j = 0; j < 4; ++j) pv.log_x[(size_t)t * xs + (size_t)inst * 4 + j] = xo[j];
                }
                const int ovf = shift_instance<WS_NT, true>(P, SMV(pool), P.so.pool_sz - (int)shift_smem_doubles(P, WS_NT), SMI(ired), SMI(ired) + 16, inst, xc, pv.stage,
                                                      cur, a_cost, a_primal, L.active, nxt, nullptr, L.log_u0 + (size_t)t * n_inst * P.nu);
                if (ovf && WS_TID == 0) { status_out[inst] = BNB_CAPACITY; L.log_status[(size_t)t * n_inst + inst] = BNB_CAPACITY; }
                log_shifted_tree(P, cx, L, nxt, inst, (size_t)t * n_inst + inst);
                prof_mark(19);
            } else if (!mbx) {
                const int ovf = shift_instance<WS_NT, true>(P, SMV(pool), P.so.pool_sz - (int)shift_smem_doubles(P, WS_NT), SMI(ired), SMI(ired) + 16, inst, xc, L.e ? L.e + (size_t)t * xs : nullptr,
                                                      cur, a_cost, a_primal, L.active, nxt, xn, L.log_u0 + (size_t)t * n_inst * P.nu);
                if (ovf && WS_TID == 0) { status_out[inst] = BNB_CAPACITY; L.log_status[(size_t)t * n_inst + inst] = BNB_CAPACITY; }
                log_shifted_tree(P, cx, L, nxt, inst, (size_t)t * n_inst + inst);
                prof_mark(19);
            } else {
                // publish step t: applied input, predicted next state, cost, status -- then the step counter
                const bool has = L.active[inst] != 0 && inc_cost[inst] < INFINITY;
                const double *ip = inc_primal + (size_t)inst * P.n_primal;
                for (int j = WS_TID; j < P.nu; j += WS_NT) L.mb_out_u0[(size_t)inst * P.nu + j] = has ? ip[(size_t)(P.T + 1) * P.nx + j] : nan("");
                for (int j = WS_TID; j < P.nx; j += WS_NT) L.mb_out_x1[(size_t)inst * P.nx + j] = has ? ip[P.nx + j] : xc[(size_t)inst * P.nx + j];
                if (WS_TID == 0) { L.mb_out_cost[inst] = has ? inc_cost[inst] : INFINITY; L.mb_out_status[inst] = st; }
                __threadfence_system();
                WS_SYNC();
                if (WS_TID == 0) L.mb_out_step[inst] = t + 1;
            }
        }
        if (WS_TID == 0) L.step_of[inst] = t + 1;
        __threadfence();                                   // release: the instance's data before the token
        WS_SYNC();
        if (WS_TID == 0 && t + 1 < S) {
            const int p = atomicAdd(L.q + 4 + S + (t + 1), 1);
            atomicExch(L.q + 4 + 2 * S + (size_t)(t + 1) * n_inst + p, inst);
        }
        if (WS_TID == 0) atomicAdd(L.q, 1);
    }
}
#undef s_inst

#define WS_LOOP_ARGS DevProblem P, double *slot_d, int *slot_i, double *ybuf, double *scratch, LoopView L, int n_slots, int n_inst, \
    TreeView t0, TreeView t1, double tol, int max_solves, double *inc_cost, int *inc_node, double *inc_primal, int *n_solves, \
    int *status_out, unsigned long long *totals, PlantView pv, FallbackView fv
#define WS_LOOP_PASS P, slot_d, slot_i, ybuf, scratch, L, n_slots, n_inst, t0, t1, tol, max_solves, inc_cost, inc_node, inc_primal, \
    n_solves, status_out, totals, pv, fv
#define WS_LOOP_BODY(LANES, RULE, PLANT, FB) closed_loop_body<LANES, RULE, PLANT, FB>(WS_LOOP_PASS)

#if WS_TU_HAS(0)
// wshmpc_plant_step: one thread per state, x_out[i] = Phi(x[i], u[i][fc_index]; parameter set i or 0)
__global__ void plant_step_kernel(PlantView pv, int n, int nu, const double *__restrict__ x, const double *__restrict__ u,
                                  double *__restrict__ x_out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double xi[4] = {x[(size_t)i * 4], x[(size_t)i * 4 + 1], x[(size_t)i * 4 + 2], x[(size_t)i * 4 + 3]};
    cartpole_walls_step(pv.prm + (pv.n_sets == 1 ? 0 : (size_t)i * WS_PLANT_NPARAM), xi, u[(size_t)i * nu + pv.fc_index], pv.h, pv.n_sub);
    for (int j = 0; j < 4; ++j) x_out[(size_t)i * 4 + j] = xi[j];
}
#endif
