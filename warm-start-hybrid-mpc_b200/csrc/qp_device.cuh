// qp_device.cuh -- lane-cooperative dual active-set solver for one branch-and-bound node QP (K1).
//
// Replaces the Gurobi call of bounded_qp.py:200-228 (reached from controller.py:229-271) for the
// relaxation of one node.  All nodes of all instances share the least-distance operator
//     min_v 1/2 |v|^2   s.t.   bl_r <= mh_r . v <= bu_r        (unit rows mh_r, r < m)
// and differ only in the bounds (x0 and the bounds on the relaxed binaries), see DESIGN.md.
//
// Execution model.  A CTA holds up to WS_MAXL independent solver LANES of WS_NT threads each (one CTA per SM); a
// lane owns one solver state ("slot") and synchronises with a NAMED barrier of its own (bar.sync lane + 1, WS_NT), so
// the lanes of a CTA run different QPs of different MPC instances at their own pace and hide each other's latencies
// (every phase of an iteration is a short chain of dependent shared-memory loads and fp64 operations).  The lanes of
// a CTA SHARE one copy of the read-only tables (stage rows, row scalings, row map) in shared memory; everything else
// is per lane.  Lane state:
//     working set W (rows, sides, multipliers lam >= 0 of the sign-normalised rows),
//     THIN factorisation  Mw' = Q1 R  kept as
//         Q1  (n - d) x k  orthonormal columns over the coordinates the node does NOT eliminate (d = pinned prefix),
//             column major with a per-node leading dimension ldc,
//         Ri  = R^-1 upper triangular, packed by columns (column j at j (j + 1) / 2),
//     (no R, no null-space basis); the first `ks` columns of both live in the lane's shared-memory POOL, later
//     columns in the slot's global home / L2.  ks is fixed per node from d (a deep node has short columns, so more of
//     them fit); every sum runs in an order that does not depend on where a column lives, so results do not depend
//     on ks, on the number of lanes or on the shared-memory budget;
//     u = R^-T (-d_W), ls = R^-1 u (the multipliers of the equality-constrained sub-problem) and
//     v = -Q1 u (its primal point) are kept up to date INCREMENTALLY: O(n + k) per append / removal;
//     yc = proximal centre.
// Appending a row is classical Gram-Schmidt against Q1 with one re-orthogonalisation pass when more than
// a digit was lost (Daniel, Gragg, Kaufman & Stewart 1976); removing position kp rotates the columns of
// Q1 and Ri with the Givens sequence that carries row kp of Ri into its last entry: every rotation is
// known up front from prefix sums of squares of that row, so the removal has no chain of dependent
// square roots and all matrix work is parallel over rows.  Every solve with R is a mat-vec with Ri.
// Rows are priced in FACTORED form: mh_r . x = a_r . (Wf x) / nrm_r with Wf = N Rinv (ns x n, shared by
// every CTA, L2 resident, stored transposed so that a thread owns two output rows and streams 16-byte
// words) and a_r the sparse stage row [F_t G_t] of the MLD system (shared memory), instead of streaming
// the dense m x n operator (6x less L2 traffic on the cart-pole).
// Every node rebuilds the factor of the working set it starts from, so rounding never accumulates across nodes;
// a hot-started solve that degenerates (iteration cap, exploding multipliers) is restarted once from the
// empty working set.
// The sequential twin of this file (same pivoting rules, same factorisation) is oracle/qp_core.c variant 1.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

// Translation units.  The large kernels (the kernel table in wshmpc.cu: one row per kernel) take about a minute of ptxas
// each; wshmpc.cu can be compiled as ONE unit (WS_TU undefined: everything) or as one unit per large kernel plus unit 0 in
// parallel (-DWS_TU=0: C ABI + the small kernels, -DWS_TU=u: the kernel of row u; __graft_entry__.build()).  A unit that
// does not define a kernel only declares it.
#ifndef WS_TU
#define WS_TU_HAS(id) 1
#else
#define WS_TU_HAS(id) (WS_TU == (id))
#endif

// Measured on the 512-instance warm-started cart-pole loop (B200, round 2, tools/loop_timing.py; QP/s):
//   1 lane  x 256 threads, 255 registers  257 k   (the round-1 configuration: 250 k with the round-1 code)
//   1 lane  x 256 threads, 128 registers  195 k   (what the register cap of two lanes costs one lane)
//   2 lanes x 256 threads, 128 registers  342 k   (350 k with 2048 instances)       <- shipped
//   3 lanes x 128 threads, 168 registers  194 k   (250 k with 2048 instances; a 128-thread lane alone: 126 k)
#ifndef WS_NT
#define WS_NT 256            // threads per solver lane
#endif
#ifndef WS_MAXL
#define WS_MAXL 2               // solver lanes per CTA at most (WS_MAXL * WS_NT threads, one CTA per SM)
#endif
#define WS_NW (WS_NT / 32)
#ifndef WS_RPT
#define WS_RPT ((384 + WS_NT - 1) / WS_NT)    // rows of Q1 a thread sweeps in a removal: n <= WS_RPT * WS_NT (>= 384)
#endif
#ifndef WS_RRT
#define WS_RRT (256 / WS_NT)    // rows of Ri a thread sweeps in a removal: working sets of up to WS_RRT * WS_NT = 256 rows
#endif
#ifndef WS_NOINLINE
#define WS_NOINLINE __forceinline__      // measured: out-of-line phases (__noinline__) shrink the code by a third and cost 25 % (call ABI spills)
#endif
// Register-budget knobs of a translation unit: the one-lane kernels (the odd units of the kernel table, which checks this)
// have 255 registers per thread, the two-lane kernels (even units; also single-unit builds) 128.  None of them changes a result.
#if defined(WS_TU) && WS_TU % 2 == 1
#define WS_WIDE_REGS 1
#else
#define WS_WIDE_REGS 0
#endif
#ifndef WS_CH
// columns per chunk of the removal sweep (results do not depend on it).  Measured on the 512-instance loop, two-lane build
// (128 registers): 1: 407 k, 2: 417 k, 3: 412 k, 4: 403 k, 8: 370 k QP/s; one-lane build (255 registers, CP40): 4 and 2 within 1 %
#if WS_WIDE_REGS
#define WS_CH 4                 // the one-lane kernels
#else
#define WS_CH 2                 // the two-lane kernels (and single-unit builds)
#endif
#endif
// loads of the pricing operator a thread keeps in flight: 8 with 255 registers; 4 under the 128-register cap (the same
// accumulators take the same columns in the same order either way; measured +0.7 % on the 512-instance loop)
#if !WS_WIDE_REGS && !defined(WS_PRICE8)
#define WS_PRICE4 1
#endif
#define WS_OPTIMAL 2
#define WS_INFEASIBLE 3
#define WS_ITER_LIMIT 9
#define WS_REORTH 1e-2          // re-orthogonalise when |z|^2 < WS_REORTH |m_j[d:]|^2
#define WS_LAM_MAX 1e13         // sum of multipliers beyond which a hot-started solve is declared degenerate

// lane-local thread index, lane index inside the CTA, lane barrier
#define WS_TID ((int)(threadIdx.x & (WS_NT - 1)))
#define WS_LANE ((int)(threadIdx.x / WS_NT))
#define WS_SYNC() asm volatile("bar.sync %0, %1;" :: "r"(WS_LANE + 1), "n"(WS_NT) : "memory")

// offsets (in doubles unless noted) of the shared-memory arrays, resolved on the host (wshmpc_create).
// Per-lane arrays are relative to the lane's base, tables (t_*) to the start of the CTA's shared memory.
struct SmemOff {
    int z, c1, c2, t, u, ls, lam, cw, yc, wv, v, bu, blb, xi, part, red;
    int vf0, vf;                          // eliminated coordinates of v: node-constant part / value in the current proximal pass
    int pool, pool_sz;                    // factor pool of the lane (Ri columns, then Q1 columns) and its size in doubles
    int irow, iside, ired, iscr;          // int offsets (from the start of the lane's int area)
    int idep;                             // node geometry: [0] d, [1] ignore-list flag, [2] d0, [3] he, [4] ldc, [5] ks, [6] triR, [7] G, [8] W
    int ints;                             // start of the lane's int area, in doubles
    int binW, bign, bnadd;                // byte offsets from the start of the lane's byte area
    int bytes;                            // start of the lane's byte area, in doubles
    int lane_doubles;                     // size of a lane's area
    int t_inr, t_vsc, t_sF, t_sG, t_sF1, t_sG1, t_rinfo;   // shared tables (t_rinfo: doubles offset of an int array)
    int tab_doubles;                      // size of the table area
    int total_bytes;
};

struct DevProblem {
    int nx, nu, nub, nuc, T, nh, nh1, nq, nqT, nr, n, m, mc, nb, ns;
    const double *A, *B, *F, *G, *h, *F1, *G1, *h1, *Q, *R, *QT, *Mmu, *MmuT, *Mrho;
    const double *Mh, *WfT, *nrm, *inr, *vscale, *Eh, *hh, *Rinv, *RinvT, *Kx, *ZmapT, *Linv, *LinvT, *Msq;
    const int *bin_idx;
    int n_elim;              // leading binaries that may be eliminated when pinned (0 = never)
    int search_rule;         // candidate selection of the device B&B: 0 best_first, 1 depth_first, 2 breadth_first
    const int *border;       // branching order of the device B&B: permutation of the nb binaries, or null = chronological (branch_in_time)
    double eps, tol_p, tol_d, tol_sing, tol_ray, prox_tol;
    int max_iter, max_prox;
    int lanes;               // solver lanes per CTA of this handle (<= WS_MAXL)
    int ld;                  // leading dimension of the global home of Q1 (>= every per-node ldc)
    int np;                  // n rounded up to even
    int ns2;                 // ns rounded up to even
    int gp;                  // groups of the ns-pair-indexed phases
    int hot_cap;             // iteration cap of a hot-started solve before it is restarted cold
    SmemOff so;
    // record layout
    int n_primal, n_dual, off_lam, off_mu, off_nulb, off_nuub, off_rho, off_sigma;
    int n_rec;               // stride of a dual record in a tree: n_dual + n (the proximal centre of the solve follows the duals)
    int node_rule;           // node rule of the device B&B (wshmpc_set_node_rule): 0 structured, 1 conventional MIQP, 2 = 1 + MIP start
};

// Phase timing of the critical path (experiment builds only, -DWS_PROF; read back by tools/ through
// wshmpc_prof_read): mark(id) charges the cycles since the previous mark of lane 0's thread 0 to phase `id`.
#ifdef WS_PROF
__device__ unsigned long long g_prof[256];
__device__ __forceinline__ void prof_mark(int id) {
    __shared__ long long s_prof_last;
    if (threadIdx.x == 0) {
        const long long t = clock64();
        atomicAdd(&g_prof[2 * id], (unsigned long long)(t - s_prof_last)); atomicAdd(&g_prof[2 * id + 1], 1ull);
        s_prof_last = clock64();
    }
}
__device__ __forceinline__ void prof_add(int id, int value) {
    if (threadIdx.x == 0) { atomicAdd(&g_prof[2 * id], (unsigned long long)value); atomicAdd(&g_prof[2 * id + 1], 1ull); }
}
#else
#define prof_mark(id) ((void)0)
#define prof_add(id, value) ((void)0)
#endif

__host__ __device__ __forceinline__ int tri_off(int j) { return j * (j + 1) / 2; }

// per-slot persistent state in global memory
struct SlotPtrs {
    double *Q;      // n*ld  (home of the columns >= ks of Q1; its first doubles park the sibling memo)
    double *Ri;     // n(n+1)/2
    double *lam;    // n+1
    double *yc;     // n
    int *row;       // n+1
    int *side;      // n+1
    int *nW;        // 1
};

__host__ __device__ __forceinline__ size_t slot_doubles(int n, int ld) { return (((size_t)n * ld + (size_t)tri_off(n) + (n + 1) + n + 4) + 1) & ~(size_t)1; }   // even: 16-byte aligned slots
__host__ __device__ __forceinline__ size_t slot_ints(int n) { return 2 * (size_t)(n + 1) + 4; }

__device__ __forceinline__ SlotPtrs slot_ptrs(double *dbase, int *ibase, int slot, int n, int ld) {
    SlotPtrs s;
    double *d = dbase + (size_t)slot * slot_doubles(n, ld);
    int *i = ibase + (size_t)slot * slot_ints(n);
    s.Q = d; d += (size_t)n * ld;
    s.Ri = d; d += tri_off(n);
    s.lam = d; d += n + 1;
    s.yc = d;
    s.row = i; i += n + 1;
    s.side = i; i += n + 1;
    s.nW = i;
    return s;
}

// what a thread keeps in registers
struct Ctx {
    double *smd;             // base of the lane's shared memory
    double *tab;             // base of the CTA's shared tables
    double *gQ, *gRi;        // global homes of the columns >= ks
    int pg, prp;             // (group, pair) of the ns-pair-indexed phases
};

#define SMV(name) (cx.smd + P.so.name)
#define SMI(name) (reinterpret_cast<int *>(cx.smd + P.so.ints) + P.so.name)
#define SMB(name) (reinterpret_cast<unsigned char *>(cx.smd + P.so.bytes) + P.so.name)
#define TBV(name) (cx.tab + P.so.t_##name)
#define TBI(name) (reinterpret_cast<const int *>(cx.tab + P.so.t_##name))

__device__ __forceinline__ Ctx make_ctx(const DevProblem &P, unsigned char *smem_raw, const SlotPtrs &sp) {
    Ctx cx;
    cx.tab = reinterpret_cast<double *>(smem_raw);
    cx.smd = cx.tab + P.so.tab_doubles + (size_t)WS_LANE * P.so.lane_doubles;
    cx.gQ = sp.Q; cx.gRi = sp.Ri;
    const int hs = P.ns2 >> 1;
    cx.pg = WS_TID / hs; cx.prp = WS_TID - cx.pg * hs;
    return cx;
}

// geometry of the node being solved (set_node_prefix*): which coordinates the factor spans and where its columns live
struct Geom {
    int d;       // eliminated coordinates (pinned prefix)
    int d0;      // d rounded down to even: the factor stores coordinates d0 .. np-1 (pairs stay 16-byte aligned)
    int he;      // pairs of stored coordinates: (np - d0) / 2
    int ldc;     // leading dimension of the shared-memory columns: 2 (he | 1)  (ldc / 2 odd: conflict-free 16-byte column reads)
    int ks;      // columns of Q1 and Ri in the lane's pool
    int triR;    // doubles the Ri part of the pool takes
    int G, W;    // the pair-indexed phases run as G groups of W threads (W >= he unless he > WS_NT)
};

__device__ __forceinline__ Geom load_geom(const DevProblem &P, const Ctx &cx) {
    const int *g = SMI(idep);
    Geom q;
    q.d = g[0]; q.d0 = g[2]; q.he = g[3]; q.ldc = g[4]; q.ks = g[5]; q.triR = g[6]; q.G = g[7]; q.W = g[8];
    return q;
}

// thread 0 of the lane: geometry for d eliminated coordinates.  The caller provides the barrier.
__device__ __forceinline__ void store_geom(const DevProblem &P, const Ctx &cx, int d) {
    int *g = SMI(idep);
    d = d < P.n_elim ? d : P.n_elim;
    const int d0 = d & ~1, he = (P.np - d0) >> 1, ldc = 2 * (he | 1);
    int ks = P.n - d;                                       // a working set never holds more independent rows
    while (ks > 0 && (size_t)ks * ldc + ((tri_off(ks) + 1) & ~1) > (size_t)P.so.pool_sz) --ks;
    const int G = he <= WS_NT ? (WS_NT / he < 8 ? WS_NT / he : 8) : 1;
    g[0] = d; g[2] = d0; g[3] = he; g[4] = ldc; g[5] = ks; g[6] = (tri_off(ks) + 1) & ~1; g[7] = G; g[8] = WS_NT / G;
}

__device__ __forceinline__ double warp_sum(double x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
}

// The lane-wide ("block") reductions below reduce inside each warp by shuffles, park one value per warp in shared
// memory, and finish with a second shuffle tree over the WS_NW per-warp values (every warp does it
// redundantly, so the result reaches all threads with two barriers and ~25 instructions).
#define WS_FULL 0xffffffffu
static_assert(WS_NW == 16 || WS_NW == 8 || WS_NW == 4 || WS_NW == 2, "the two-level reductions assume 2, 4, 8 or 16 warps per CTA");

// block-wide sum, result to all threads
__device__ __forceinline__ double block_sum(double x, double *red) {
    const int lane = WS_TID & 31, w = WS_TID >> 5;
    x = warp_sum(x);
    WS_SYNC();
    if (lane == 0) red[w] = x;
    WS_SYNC();
    double s = lane < WS_NW ? red[lane] : 0.;
#pragma unroll
    for (int o = WS_NW / 2; o > 0; o >>= 1) s += __shfl_xor_sync(WS_FULL, s, o);
    return __shfl_sync(WS_FULL, s, 0);
}

// two block-wide sums at once
__device__ __forceinline__ void block_sum2(double &x, double &y, double *red) {
    const int lane = WS_TID & 31, w = WS_TID >> 5;
    x = warp_sum(x); y = warp_sum(y);
    WS_SYNC();
    if (lane == 0) { red[w] = x; red[16 + w] = y; }
    WS_SYNC();
    // lanes 0..15 take the x partials, lanes 16..31 the y partials
    double s = (lane & 15) < WS_NW ? red[lane] : 0.;
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(WS_FULL, s, o);
    x = __shfl_sync(WS_FULL, s, 0); y = __shfl_sync(WS_FULL, s, 16);
}

__device__ __forceinline__ bool better_max(double ov, int oi, double val, int idx) {
    return oi >= 0 && (idx < 0 || ov > val || (ov == val && oi < idx));
}

// block-wide arg-max of (val, idx): larger val wins, ties -> smaller idx.  idx < 0 = no candidate.
__device__ __forceinline__ void block_argmax(double &val, int &idx, double *red, int *ired) {
    const int lane = WS_TID & 31, w = WS_TID >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(WS_FULL, val, o);
        const int oi = __shfl_xor_sync(WS_FULL, idx, o);
        if (better_max(ov, oi, val, idx)) { val = ov; idx = oi; }
    }
    WS_SYNC();
    if (lane == 0) { red[w] = val; ired[w] = idx; }
    WS_SYNC();
    val = lane < WS_NW ? red[lane] : 0.; idx = lane < WS_NW ? ired[lane] : -1;
#pragma unroll
    for (int o = WS_NW / 2; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(WS_FULL, val, o);
        const int oi = __shfl_xor_sync(WS_FULL, idx, o);
        if (better_max(ov, oi, val, idx)) { val = ov; idx = oi; }
    }
    val = __shfl_sync(WS_FULL, val, 0); idx = __shfl_sync(WS_FULL, idx, 0);
}

// block-wide max of a non-negative value
__device__ __forceinline__ double block_max(double x, double *red) {
    const int lane = WS_TID & 31, w = WS_TID >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x = fmax(x, __shfl_xor_sync(WS_FULL, x, o));
    WS_SYNC();
    if (lane == 0) red[w] = x;
    WS_SYNC();
    double s = lane < WS_NW ? red[lane] : 0.;
#pragma unroll
    for (int o = WS_NW / 2; o > 0; o >>= 1) s = fmax(s, __shfl_xor_sync(WS_FULL, s, o));
    return __shfl_sync(WS_FULL, s, 0);
}

// block-wide arg-min (ratio tests): smaller val wins, ties -> smaller idx
__device__ __forceinline__ void block_argmin(double &val, int &idx, double *red, int *ired) {
    double nv = -val;
    block_argmax(nv, idx, red, ired);
    val = -nv;
}

// warp-wide arg-min (ties -> smaller idx) and sum, result in every lane
__device__ __forceinline__ void warp_argmin_sum(double &val, int &idx, double &sum) {
    double nv = -val;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(WS_FULL, nv, o);
        const int oi = __shfl_xor_sync(WS_FULL, idx, o);
        sum += __shfl_xor_sync(WS_FULL, sum, o);
        if (better_max(ov, oi, nv, idx)) { nv = ov; idx = oi; }
    }
    val = -nv;
}

// arg-min and a sum in one pass (ratio test + sum of the positive multipliers)
__device__ __forceinline__ void block_argmin_sum(double &val, int &idx, double &sum, double *red, int *ired) {
    const int lane = WS_TID & 31, w = WS_TID >> 5;
    double nv = -val;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(WS_FULL, nv, o);
        const int oi = __shfl_xor_sync(WS_FULL, idx, o);
        sum += __shfl_xor_sync(WS_FULL, sum, o);
        if (better_max(ov, oi, nv, idx)) { nv = ov; idx = oi; }
    }
    WS_SYNC();
    if (lane == 0) { red[w] = nv; ired[w] = idx; red[16 + w] = sum; }
    WS_SYNC();
    nv = lane < WS_NW ? red[lane] : 0.; idx = lane < WS_NW ? ired[lane] : -1;
    sum = lane < WS_NW ? red[16 + lane] : 0.;
#pragma unroll
    for (int o = WS_NW / 2; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(WS_FULL, nv, o);
        const int oi = __shfl_xor_sync(WS_FULL, idx, o);
        sum += __shfl_xor_sync(WS_FULL, sum, o);
        if (better_max(ov, oi, nv, idx)) { nv = ov; idx = oi; }
    }
    val = -__shfl_sync(WS_FULL, nv, 0); idx = __shfl_sync(WS_FULL, idx, 0); sum = __shfl_sync(WS_FULL, sum, 0);
}

// ---------------------------------------------------------------------------------------------
// grouped mat-vec with a shared operator:  out(i, sum_{j0 <= j < j1} M[j * ld + i] * x[j])  for i < rows.
// Adjacent threads take adjacent i (coalesced); when rows <= WS_NT the threads form G = WS_NT / rows
// groups that split the j range and combine through `part` (>= max(WS_NT, rows) doubles).
// Ends with a barrier-protected combine; `out` is called once per row.  Contains lane barriers.
// (refresh / record paths only: once per proximal pass, not per iteration)
// ---------------------------------------------------------------------------------------------
template <class Out>
__device__ __forceinline__ void grouped_matvec(const double *__restrict__ M, int ld, int rows, int j0, int j1,
                                      const double *x, double *part, Out out) {
    if (rows <= WS_NT) {
        const int G = WS_NT / rows;
        const int g = WS_TID / rows, i = WS_TID - g * rows;
        if (g < G) {
            double s0 = 0., s1 = 0., s2 = 0., s3 = 0.;
            int j = j0 + g;
            // the operators come from L2: 8 independent loads in flight per thread
            for (; j + 7 * G < j1; j += 8 * G) {
                double w[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) w[q] = __ldg(M + (size_t)(j + q * G) * ld + i);
                s0 += w[0] * x[j] + w[4] * x[j + 4 * G];
                s1 += w[1] * x[j + G] + w[5] * x[j + 5 * G];
                s2 += w[2] * x[j + 2 * G] + w[6] * x[j + 6 * G];
                s3 += w[3] * x[j + 3 * G] + w[7] * x[j + 7 * G];
            }
            for (; j + 3 * G < j1; j += 4 * G) {
                s0 += M[(size_t)j * ld + i] * x[j];
                s1 += M[(size_t)(j + G) * ld + i] * x[j + G];
                s2 += M[(size_t)(j + 2 * G) * ld + i] * x[j + 2 * G];
                s3 += M[(size_t)(j + 3 * G) * ld + i] * x[j + 3 * G];
            }
            for (; j < j1; j += G) s0 += M[(size_t)j * ld + i] * x[j];
            part[g * rows + i] = (s0 + s1) + (s2 + s3);
        }
        WS_SYNC();
        if (WS_TID < rows) {
            double s = part[WS_TID];
            for (int q = 1; q < G; ++q) s += part[q * rows + WS_TID];
            out(WS_TID, s);
        }
        WS_SYNC();
    } else {
        // more rows than threads: a thread owns the rows tid, tid + WS_NT, ... and all columns, 8 loads in flight
        for (int i = WS_TID; i < rows; i += WS_NT) {
            double s0 = 0., s1 = 0., s2 = 0., s3 = 0.;
            int j = j0;
            for (; j + 7 < j1; j += 8) {
                double w[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) w[q] = __ldg(M + (size_t)(j + q) * ld + i);
                s0 += w[0] * x[j] + w[4] * x[j + 4];
                s1 += w[1] * x[j + 1] + w[5] * x[j + 5];
                s2 += w[2] * x[j + 2] + w[6] * x[j + 6];
                s3 += w[3] * x[j + 3] + w[7] * x[j + 7];
            }
            for (; j < j1; ++j) s0 += M[(size_t)j * ld + i] * x[j];
            out(i, (s0 + s1) + (s2 + s3));
        }
        WS_SYNC();
    }
}

// ---------------------------------------------------------------------------------------------
// thin factor: products with Q1 and Ri.  Columns < ks in the lane's pool, the rest in the global home.
// A column of Q1 is addressed by the COORDINATE index i >= d0 (its storage starts at coordinate d0).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double *pool_Ri(const DevProblem &P, const Ctx &cx) { return SMV(pool); }
// SM: every column the caller touches is in the pool (the common case): plain shared-memory addressing instead of the
// per-column shared / global choice.  The arithmetic is the same either way.
template <bool SM>
__device__ __forceinline__ double *qcol_w(const DevProblem &P, const Ctx &cx, const Geom &g, int j) {
    if (SM) return SMV(pool) + g.triR + j * g.ldc - g.d0;
    return (j < g.ks ? SMV(pool) + g.triR + j * g.ldc : cx.gQ + (size_t)j * P.ld) - g.d0;
}
template <bool SM>
__device__ __forceinline__ double *ricol_w(const DevProblem &P, const Ctx &cx, const Geom &g, int j) {
    if (SM) return SMV(pool) + tri_off(j);
    return (j < g.ks ? SMV(pool) : cx.gRi) + tri_off(j);
}

// The k-indexed phases (one output per working-set position) give every output to a team of ng = 2^lg lanes of one warp
// that split the other dimension and combine by shuffles: WS_NT / ng outputs per pass, no partial sums through shared
// memory, one barrier.  ng is the largest power of two <= 32 with k ng <= WS_NT (so all warps have work).  The members
// of a team are the lanes l, l + C, l + 2C, ... (C = 32 / ng outputs per warp): ADJACENT lanes work on adjacent outputs
// at the same position of the other dimension, i.e. on different columns with an odd 16-byte stride -- no bank conflicts.
__device__ __forceinline__ int team_log2(int k) { return k >= WS_NT ? 0 : min(5, 31 - __clz(WS_NT / max(k, 1))); }

__device__ __forceinline__ double team_sum(double s, int lg) {
    for (int o = 32 >> lg; o < 32; o <<= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    return s;
}

// out[j] = q_j . x  for j < k  (x indexed by coordinate, entries below d0 ignored).  Ends with a barrier.
template <bool SM>
__device__ __forceinline__ void qt_dots_t(const DevProblem &P, const Ctx &cx, int k, const double *x, double *out) {
    const Geom gm = load_geom(P, cx);
    const int lg = team_log2(k), ng = 1 << lg, C = 32 >> lg, jw = WS_NT >> lg;
    const int lane = WS_TID & 31, g = lane >> (5 - lg), jl = (WS_TID >> 5) * C + (lane & (C - 1));
    const int p0 = (gm.d0 >> 1) + g, p1 = P.np >> 1;
    const double2 *x2 = reinterpret_cast<const double2 *>(x);
    const int kr = (k + jw - 1) / jw * jw;                          // whole warps take part in the shuffles
    for (int j = jl; j < kr; j += jw) {
        double s0 = 0., s1 = 0.;
        if (j < k) {
            const double2 *q2 = reinterpret_cast<const double2 *>(qcol_w<SM>(P, cx, gm, j));
            for (int p = p0; p < p1; p += ng) { const double2 a = q2[p], b = x2[p]; s0 += a.x * b.x; s1 += a.y * b.y; }
        }
        const double s = team_sum(s0 + s1, lg);
        if (g == 0 && j < k) out[j] = s;
    }
    WS_SYNC();
}

// zout = zin - sum_{j < k} q_j c[j] on the coordinates >= d0 (zin == nullptr: zero; zout may alias zin).  Returns
// |zout|^2 and the lane-wide sum of `extra` (a second quantity the caller wants reduced: it rides on the barrier this
// phase needs anyway) in every thread.  Ends with a barrier.
template <bool SM>
__device__ __forceinline__ double q_apply_t(const DevProblem &P, const Ctx &cx, int k, const double *c, const double *zin, double *zout,
                                 double extra = 0., double *extra_sum = nullptr) {
    const Geom gm = load_geom(P, cx);
    double2 *part2 = reinterpret_cast<double2 *>(SMV(part));
    const int G = gm.G, W = gm.W, he = gm.he, dh = gm.d0 >> 1;
    const int grp = WS_TID / W, t = WS_TID - grp * W;
    if (grp < G) {
        for (int pp = t; pp < he; pp += W) {
            double ax = 0., ay = 0., bx = 0., by = 0.;
            int j = grp;
            for (; j + G < k; j += 2 * G) {
                const double2 a = reinterpret_cast<const double2 *>(qcol_w<SM>(P, cx, gm, j))[dh + pp];
                const double2 b = reinterpret_cast<const double2 *>(qcol_w<SM>(P, cx, gm, j + G))[dh + pp];
                const double ca = c[j], cb = c[j + G];
                ax += a.x * ca; ay += a.y * ca; bx += b.x * cb; by += b.y * cb;
            }
            if (j < k) { const double2 a = reinterpret_cast<const double2 *>(qcol_w<SM>(P, cx, gm, j))[dh + pp]; const double ca = c[j]; ax += a.x * ca; ay += a.y * ca; }
            part2[grp * he + pp] = make_double2(ax + bx, ay + by);
        }
    }
    WS_SYNC();
    const double *part = SMV(part);
    double zz = 0.;
    for (int i = WS_TID; i < 2 * he; i += WS_NT) {
        double s = part[i];
        for (int q = 1; q < G; ++q) s += part[q * 2 * he + i];
        const double zi = (zin ? zin[gm.d0 + i] : 0.) - s;
        zout[gm.d0 + i] = zi; zz += zi * zi;
    }
    {
        const int lane = WS_TID & 31, w = WS_TID >> 5;
        double *red = SMV(red) + 72;                     // [w]: |z|^2 partials, [16 + w]: partials of `extra`
        zz = warp_sum(zz); extra = warp_sum(extra);
        if (lane == 0) { red[w] = zz; red[16 + w] = extra; }
        WS_SYNC();
        double sv = (lane & 15) < WS_NW ? red[lane] : 0.;
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) sv += __shfl_xor_sync(WS_FULL, sv, o);
        zz = __shfl_sync(WS_FULL, sv, 0);
        if (extra_sum) *extra_sum = __shfl_sync(WS_FULL, sv, 16);
    }
    return zz;
}

// t_i = (Ri c[:k])_i = sum_{j >= i} Ri[tri_off(j) + i] c_j handed to out(i, t_i) by the leader of the team of row i
// (columns j = i + g, i + g + ng, ...).  No barrier.
template <bool SM, class Out>
__device__ __forceinline__ void ri_matvec_ep(const DevProblem &P, const Ctx &cx, int k, const double *c, Out out) {
    const Geom gm = load_geom(P, cx);
    const int lg = team_log2(k), ng = 1 << lg, C = 32 >> lg, jw = WS_NT >> lg;
    const int lane = WS_TID & 31, g = lane >> (5 - lg), il = (WS_TID >> 5) * C + (lane & (C - 1));
    const int kr = (k + jw - 1) / jw * jw;
    for (int i = il; i < kr; i += jw) {
        double s0 = 0., s1 = 0.;
        if (i < k) {
            int j = i + g;
            for (; j + ng < k; j += 2 * ng) { s0 += ricol_w<SM>(P, cx, gm, j)[i] * c[j]; s1 += ricol_w<SM>(P, cx, gm, j + ng)[i] * c[j + ng]; }
            if (j < k) s0 += ricol_w<SM>(P, cx, gm, j)[i] * c[j];
        }
        const double sv = team_sum(s0 + s1, lg);
        if (g == 0 && i < k) out(i, sv);
    }
}

// t = Ri * c[:k].  Ends with a barrier.
template <bool SM>
__device__ __forceinline__ void ri_matvec(const DevProblem &P, const Ctx &cx, int k, const double *c, double *t) {
    ri_matvec_ep<SM>(P, cx, k, c, [&](int i, double s) { t[i] = s; });
    WS_SYNC();
}

// u = Ri' * d[:k]  (u_j = sum_{i <= j} Ri[tri_off(j) + i] d_i).  Refresh path only.  Ends with a barrier.
template <bool SM>
__device__ __forceinline__ void rit_matvec_t(const DevProblem &P, const Ctx &cx, int k, const double *d, double *u) {
    const Geom gm = load_geom(P, cx);
    const int lg = team_log2(k), ng = 1 << lg, C = 32 >> lg, jw = WS_NT >> lg;
    const int lane = WS_TID & 31, g = lane >> (5 - lg), jl = (WS_TID >> 5) * C + (lane & (C - 1));
    const int kr = (k + jw - 1) / jw * jw;
    for (int j = jl; j < kr; j += jw) {
        double s = 0.;
        if (j < k) { const double *col = ricol_w<SM>(P, cx, gm, j); for (int i = g; i <= j; i += ng) s += col[i] * d[i]; }
        s = team_sum(s, lg);
        if (g == 0 && j < k) u[j] = s;
    }
    WS_SYNC();
}

// -(signed bound of row r on side s): the entry of c = -d_W
__device__ __forceinline__ double neg_bound(const DevProblem &P, const Ctx &cx, int r, int s) {
    return -(s > 0 ? SMV(bu)[r] : -SMV(blb)[r - P.mc]);
}

// u = R^-T (-d_W), ls = R^-1 u, v = -Q1 u from scratch (new bounds: node start, proximal pass)
__device__ __forceinline__ void refresh_uv(const DevProblem &P, const Ctx &cx, int k) {
    const Geom gm = load_geom(P, cx);
    const int *row = SMI(irow), *side = SMI(iside);
    for (int i = WS_TID; i < k; i += WS_NT) SMV(cw)[i] = neg_bound(P, cx, row[i], side[i]);
    for (int i = WS_TID; i < P.np; i += WS_NT) SMV(v)[i] = 0.;
    WS_SYNC();
    if (k <= gm.ks) { rit_matvec_t<true>(P, cx, k, SMV(cw), SMV(u)); ri_matvec<true>(P, cx, k, SMV(u), SMV(ls)); q_apply_t<true>(P, cx, k, SMV(u), nullptr, SMV(v)); }
    else { rit_matvec_t<false>(P, cx, k, SMV(cw), SMV(u)); ri_matvec<false>(P, cx, k, SMV(u), SMV(ls)); q_apply_t<false>(P, cx, k, SMV(u), nullptr, SMV(v)); }
}

// entries d0 + tid, d0 + tid + WS_NT, ... of row r (zero below d and beyond n): what a thread stages for an append
struct RowEnt { double e[WS_RPT]; };

__device__ __forceinline__ RowEnt load_row_entries(const DevProblem &P, int r, int d, int d0) {
    RowEnt x;
#pragma unroll
    for (int q = 0; q < WS_RPT; ++q) {
        const int i = d0 + WS_TID + q * WS_NT;
        x.e[q] = (i < P.n && i >= d) ? __ldg(P.Mh + (size_t)r * P.n + i) : 0.;
    }
    return x;
}

// Try to append the sign-normalised row (r, sgn).  Returns 1 if appended (lam = 0), 0 if the row is
// numerically in the span of the working rows; either way t = R^-1 Q1' mj  (mj = Mw' t if dependent).
// Returns -1 (nothing done) if the working set is at the capacity of the removal sweep (WS_RRT WS_NT positions).
// `track`: also bring u, ls, v up to date (false while the factor of an inherited working set is rebuilt).
// `pre`: the row's entries, already loaded by the caller (rebuild: the load of the next row overlaps the append of the
// current one).
template <bool SM>
__device__ __forceinline__ int thin_append_t(const DevProblem &P, const Ctx &cx, int &k, int r, int sgn, bool track, const RowEnt *pre = nullptr) {
    const Geom gm = load_geom(P, cx);
    const int n = P.n, d = gm.d;
    if (k >= WS_RRT * WS_NT) return -1;
    double *z = SMV(z), *c1 = SMV(c1), *t = SMV(t);
    const int pb = track ? 30 : 40;                  // phase ids of the WS_PROF timeline
    (void)pb;
    {
        const RowEnt e = pre ? *pre : load_row_entries(P, r, d, gm.d0);
#pragma unroll
        for (int q = 0; q < WS_RPT; ++q) { const int i = gm.d0 + WS_TID + q * WS_NT; if (i < P.np) z[i] = (double)sgn * e.e[q]; }
    }
    WS_SYNC();
    prof_mark(pb);
    qt_dots_t<SM>(P, cx, k, z, c1);
    prof_mark(pb + 1);
    double cu = 0.;
    if (track) for (int j = WS_TID; j < k; j += WS_NT) cu += c1[j] * SMV(u)[j];
    double rho2 = q_apply_t<SM>(P, cx, k, c1, z, z, cu, &cu);
    prof_mark(pb + 2);
    if (k > 0 && rho2 < WS_REORTH * __ldg(P.Msq + (size_t)r * (P.nb + 1) + d)) {
        double *c2 = SMV(c2);
        qt_dots_t<SM>(P, cx, k, z, c2);
        double cu2 = 0.;
        for (int j = WS_TID; j < k; j += WS_NT) { const double dc = c2[j]; c1[j] += dc; if (track) cu2 += dc * SMV(u)[j]; }
        rho2 = q_apply_t<SM>(P, cx, k, c2, z, z, cu2, &cu2);
        cu += cu2;
        prof_mark(pb + 4);
    }
    // t = Ri c1 and, if the row is independent, the new column of Ri / the update of ls straight from the team leaders:
    // the triangular product and the write-out are ONE phase
    const bool dep = k >= n - d || rho2 <= P.tol_sing * P.tol_sing;
    const double ir = dep ? 0. : 1. / sqrt(rho2);
    double *qk = qcol_w<SM>(P, cx, gm, k), *rk = ricol_w<SM>(P, cx, gm, k);
    double uk = 0., lk = 0.;
    if (track && !dep) { uk = (neg_bound(P, cx, r, sgn) - cu) * ir; lk = uk * ir; }
    ri_matvec_ep<SM>(P, cx, k, c1, [&](int i, double ti) {
        t[i] = ti;
        if (!dep) { rk[i] = -ti * ir; if (track) SMV(ls)[i] -= ti * lk; }
    });
    if (dep) { WS_SYNC(); prof_mark(pb + 5); return 0; }
    for (int i = gm.d0 + WS_TID; i < P.np; i += WS_NT) {
        const double q = z[i] * ir;
        qk[i] = q;
        if (track) SMV(v)[i] -= q * uk;
    }
    if (WS_TID == 0) {
        rk[k] = ir;
        SMI(irow)[k] = r; SMI(iside)[k] = sgn; SMV(lam)[k] = 0.;
        if (track) { SMV(u)[k] = uk; SMV(ls)[k] = lk; }
    }
    k += 1;
    // while the factor is rebuilt the next append starts with a barrier of its own (after the row is staged) and nothing
    // in between reads what was written here; rebuild_factor ends with a barrier
    if (track) WS_SYNC();
    prof_mark(pb + 6);
    return 1;
}

// Remove position kp from the working set (u, ls, v follow).  Returns the smallest position >= kp whose
// diagonal of R collapsed (|Ri_ii| >= 1 / tol_sing) after the removal, or -1.
template <bool SM>
__device__ __forceinline__ int thin_remove_t(const DevProblem &P, const Ctx &cx, int &k, int kp) {
    const Geom gm = load_geom(P, cx);
    auto QC = [&](int j) -> double * { return qcol_w<SM>(P, cx, gm, j); };
    auto RC = [&](int j) -> double * { return ricol_w<SM>(P, cx, gm, j); };
    const int lane = WS_TID & 31, w = WS_TID >> 5, tid = WS_TID;
    double *gc = SMV(c2), *gs = SMV(cw), *u = SMV(u);           // rotation cosines / sines (c2, cw are free during a removal)
    int *row = SMI(irow), *side = SMI(iside), *flag = SMI(ired) + 32;
    if (tid == 0) *flag = 0x7fffffff;
    prof_add(100, k - 1 - kp);
    prof_add(101, k);
    if (kp == k - 1) {
        // last position: Q1, Ri lose their last column; v += q_last u_last
        const double ul = u[kp];
        const double *qk = QC(kp);
        for (int i = gm.d0 + tid; i < P.np; i += WS_NT) SMV(v)[i] += qk[i] * ul;
        // ls = Ri u loses the term of the last column
        const double *rl = RC(kp);
        for (int i = tid; i < kp; i += WS_NT) SMV(ls)[i] -= rl[i] * ul;
        k -= 1;
        WS_SYNC();
        prof_mark(50);
        return -1;
    }
    // ---- 1. warp 0: rotations i = kp .. k-2 of the column pairs (i, i+1) from prefix sums of squares of row kp of Ri
    if (w == 0) {
        const double wkp = RC(kp)[kp];
        double run = 0.;
        for (int b = kp; b < k; b += 32) {
            const int j = b + lane;
            const double wj = j < k ? RC(j)[kp] : 0.;
            double s = wj * wj;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const double y = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += y; }
            s += run;                                             // sigma_j^2 (inclusive)
            double excl = __shfl_up_sync(0xffffffffu, s, 1);      // sigma_{j-1}^2
            if (lane == 0) excl = run;
            if (j > kp && j < k) {
                const double isj = 1. / sqrt(s);
                const double tau = (j - 1 == kp) ? wkp : sqrt(excl);
                gc[j - 1] = wj * isj; gs[j - 1] = -tau * isj;
            }
            run = __shfl_sync(0xffffffffu, s, 31);
        }
    }
    // bookkeeping shift: read now, write after the barrier that publishes the rotations
    int rw[WS_RRT], sd[WS_RRT]; double lm[WS_RRT];
#pragma unroll
    for (int q = 0; q < WS_RRT; ++q) {
        const int ts = kp + 1 + tid + q * WS_NT;
        rw[q] = 0; sd[q] = 0; lm[q] = 0.;
        if (ts < k) { rw[q] = row[ts]; sd[q] = side[ts]; lm[q] = SMV(lam)[ts]; }
    }
    // ---- 2. sweep over the columns in chunks: rows d0 + tid + q WS_NT of Q1, rows WS_NT - 1 - tid + q WS_NT of Ri,
    //         the u chain in the first thread of the first warp without a row of Q1 (thread 0 if every warp has one)
    int qr[WS_RPT]; double qcarry[WS_RPT];
#pragma unroll
    for (int q = 0; q < WS_RPT; ++q) { const int i = gm.d0 + tid + q * WS_NT; qr[q] = i < P.np ? i : -1; }
    int rr[WS_RRT], ro[WS_RRT]; double rcarry[WS_RRT], ls_old[WS_RRT];
#pragma unroll
    for (int q = 0; q < WS_RRT; ++q) {
        const int r = WS_NT - 1 - tid + q * WS_NT;
        rr[q] = r < k - 1 ? r : -1;
        ro[q] = r < kp ? r : r + 1;
    }
    const int nq1 = (2 * gm.he + 31) & ~31;
    const bool uth = tid == (nq1 < WS_NT ? nq1 : 0);
    const double big = 1. / P.tol_sing;
    WS_SYNC();                                                              // gc, gs visible; row / side / lam have been read
    prof_mark(51);
#pragma unroll
    for (int q = 0; q < WS_RRT; ++q) {
        const int ts = kp + 1 + tid + q * WS_NT;
        if (ts < k) { row[ts - 1] = rw[q]; side[ts - 1] = sd[q]; SMV(lam)[ts - 1] = lm[q]; }
    }
#pragma unroll
    for (int q = 0; q < WS_RPT; ++q) qcarry[q] = qr[q] >= 0 ? QC(kp)[qr[q]] : 0.;
#pragma unroll
    for (int q = 0; q < WS_RRT; ++q) {
        rcarry[q] = (rr[q] >= 0 && ro[q] <= kp) ? RC(kp)[ro[q]] : 0.;
    }
    double ucarry = uth ? u[kp] : 0.;
    for (int i0 = kp; i0 < k - 1; i0 += WS_CH) {
        double b[WS_RRT][WS_CH];
#pragma unroll
        for (int q = 0; q < WS_RRT; ++q) if (rr[q] >= 0) {
#pragma unroll
            for (int c = 0; c < WS_CH; ++c) { const int i = i0 + c; b[q][c] = (i < k - 1 && ro[q] <= i + 1) ? RC(i + 1)[ro[q]] : 0.; }
        }
        WS_SYNC();                                                          // every old entry of the chunk has been read
        prof_mark(54);
#pragma unroll
        for (int q = 0; q < WS_RRT; ++q) if (rr[q] >= 0 && ro[q] <= i0 + WS_CH) {
#pragma unroll
            for (int c = 0; c < WS_CH; ++c) {
                const int i = i0 + c;
                if (i < k - 1) {
                    const double cs = gc[i], sn = gs[i];
                    const double o = cs * rcarry[q] + sn * b[q][c];
                    rcarry[q] = -sn * rcarry[q] + cs * b[q][c];
                    if (rr[q] <= i) {
                        RC(i)[rr[q]] = o;
                        if (rr[q] == i && fabs(o) >= big) atomicMin(flag, rr[q]);
                    }
                }
            }
        }
        const int iend = (i0 + WS_CH < k - 1) ? i0 + WS_CH : k - 1;
        prof_mark(55);
#pragma unroll
        for (int q = 0; q < WS_RPT; ++q) if (qr[q] >= 0) {
            for (int i = i0; i < iend; ++i) {
                const double bq = QC(i + 1)[qr[q]];
                const double cs = gc[i], sn = gs[i];
                QC(i)[qr[q]] = cs * qcarry[q] + sn * bq;
                qcarry[q] = -sn * qcarry[q] + cs * bq;
            }
        }
        if (uth) {
            for (int i = i0; i < iend; ++i) {
                const double bu_ = u[i + 1];
                const double cs = gc[i], sn = gs[i];
                u[i] = cs * ucarry + sn * bu_;
                ucarry = -sn * ucarry + cs * bu_;
            }
        }
        prof_mark(56);
    }
    if (uth) SMV(red)[40] = ucarry;                                  // (G u)_last
#pragma unroll
    for (int q = 0; q < WS_RRT; ++q) ls_old[q] = rr[q] >= 0 ? SMV(ls)[ro[q]] : 0.;   // read before any thread writes its new entry (after the barrier)
    k -= 1;
    WS_SYNC();
    prof_mark(52);
    // v = -Q1_new u_new = v_old + q_last (G u)_last
#pragma unroll
    for (int q = 0; q < WS_RPT; ++q) if (qr[q] >= 0) SMV(v)[qr[q]] += qcarry[q] * SMV(red)[40];
    // ls = Ri u = (Ri G')(G u): dropping the rotated-out last column leaves  ls_new[rr] = ls_old[ro] - (Ri G')[ro, last] (G u)_last,
    // and the carry of row rr IS that last-column entry
#pragma unroll
    for (int q = 0; q < WS_RRT; ++q) if (rr[q] >= 0) SMV(ls)[rr[q]] = ls_old[q] - rcarry[q] * SMV(red)[40];
    const int bad = *flag;
    WS_SYNC();
    prof_mark(53);
    return bad == 0x7fffffff ? -1 : bad;
}

__device__ __forceinline__ int thin_append(const DevProblem &P, const Ctx &cx, int &k, int r, int sgn, bool track, const RowEnt *pre = nullptr) {
    const Geom gm = load_geom(P, cx);
    return k < gm.ks ? thin_append_t<true>(P, cx, k, r, sgn, track, pre) : thin_append_t<false>(P, cx, k, r, sgn, track, pre);
}
__device__ __forceinline__ int thin_remove(const DevProblem &P, const Ctx &cx, int &k, int kp) {
    const Geom gm = load_geom(P, cx);
    return k <= gm.ks ? thin_remove_t<true>(P, cx, k, kp) : thin_remove_t<false>(P, cx, k, kp);
}

// remove position kp, then every row whose diagonal of R collapsed (see oracle/qp_core.c thin_ws_remove)
__device__ __forceinline__ void ws_remove(const DevProblem &P, const Ctx &cx, int &k, int kp) {
    signed char *inW = reinterpret_cast<signed char *>(SMB(binW));
    int pos = kp;
    do {                                   // ONE inlined copy of the removal (code size: the kernel's hot loop must stay in the instruction cache)
        if (WS_TID == 0) inW[SMI(irow)[pos]] = 0;
        WS_SYNC();
        pos = thin_remove(P, cx, k, pos);
    } while (pos >= 0);
}

// sv_r = mh_r . x for all rows in factored form; calls f(r, sv) once per row.
//   xi = Wf x  (ns = n + T nx entries: inputs zeta_t, then states xi_1 .. xi_T of the homogeneous dynamics)
//   row (t, i):  sv = (F_t[i] . xi_t + G_t[i] . zeta_t) / nrm_r   (xi_0 = 0: the x0 part is in the bounds)
//   binary (t, i): sv = zeta_t[nuc + i] / nrm_r
// WfT is the operator transposed (n x ns2): a thread owns two adjacent outputs and streams 16-byte words,
// gp groups split the columns.
// x[c] = 0 for c < c0 (the eliminated coordinates): those columns of the operator are skipped.
// skip(r): rows whose value is not wanted (in the working set, eliminated) are dropped BEFORE their products.
template <class Skip, class Fn>
__device__ __forceinline__ void price_rows(const DevProblem &P, const Ctx &cx, const double *x, int c0, int pid, Skip skip, Fn f) {
    const int n = P.n, m = P.m, mc = P.mc, nx = P.nx, nu = P.nu;
    const int hs = P.ns2 >> 1;
    double *xi = SMV(xi);
    {
        double2 *part2 = reinterpret_cast<double2 *>(SMV(part));
        if (cx.pg < P.gp) {
            const double2 *w2 = reinterpret_cast<const double2 *>(P.WfT) + cx.prp;
            double ax = 0., ay = 0., bx = 0., by = 0., ex = 0., ey = 0., dx = 0., dy = 0.;
            int c = c0 + cx.pg;
            const int G = P.gp;
            // 8 independent 16-byte loads in flight per thread: the operator comes from L2 (~700 cycles a round trip)
#ifndef WS_PRICE4
            for (; c + 7 * G < n; c += 8 * G) {
                double2 w[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) w[q] = __ldg(w2 + (size_t)(c + q * G) * hs);
#pragma unroll
                for (int q = 0; q < 8; q += 4) {
                    const double xa = x[c + q * G], xb = x[c + (q + 1) * G], xe = x[c + (q + 2) * G], xd = x[c + (q + 3) * G];
                    ax += w[q].x * xa; ay += w[q].y * xa; bx += w[q + 1].x * xb; by += w[q + 1].y * xb;
                    ex += w[q + 2].x * xe; ey += w[q + 2].y * xe; dx += w[q + 3].x * xd; dy += w[q + 3].y * xd;
                }
            }
#endif
            for (; c + 3 * G < n; c += 4 * G) {
                const double2 a = __ldg(w2 + (size_t)c * hs), b = __ldg(w2 + (size_t)(c + G) * hs),
                              e = __ldg(w2 + (size_t)(c + 2 * G) * hs), d = __ldg(w2 + (size_t)(c + 3 * G) * hs);
                const double xa = x[c], xb = x[c + G], xe = x[c + 2 * G], xd = x[c + 3 * G];
                ax += a.x * xa; ay += a.y * xa; bx += b.x * xb; by += b.y * xb;
                ex += e.x * xe; ey += e.y * xe; dx += d.x * xd; dy += d.y * xd;
            }
            for (; c < n; c += G) { const double2 a = __ldg(w2 + (size_t)c * hs); const double xa = x[c]; ax += a.x * xa; ay += a.y * xa; }
            part2[cx.pg * hs + cx.prp] = make_double2((ax + bx) + (ex + dx), (ay + by) + (ey + dy));
        }
        if (P.gp == 0) {
            // more output pairs than threads: a thread owns the pairs tid, tid + WS_NT, ... and all columns
            double2 *xi2 = reinterpret_cast<double2 *>(xi);
            for (int pp = WS_TID; pp < hs; pp += WS_NT) {
                const double2 *w2 = reinterpret_cast<const double2 *>(P.WfT) + pp;
                double ax = 0., ay = 0., bx = 0., by = 0.;
                int c = c0;
                for (; c + 1 < n; c += 2) {
                    const double2 a = __ldg(w2 + (size_t)c * hs), b = __ldg(w2 + (size_t)(c + 1) * hs);
                    const double xa = x[c], xb = x[c + 1];
                    ax += a.x * xa; ay += a.y * xa; bx += b.x * xb; by += b.y * xb;
                }
                if (c < n) { const double2 a = __ldg(w2 + (size_t)c * hs); const double xa = x[c]; ax += a.x * xa; ay += a.y * xa; }
                xi2[pp] = make_double2(ax + bx, ay + by);
            }
        }
        WS_SYNC();
        if (P.gp > 0) {
            const double *part = SMV(part);
            for (int r = WS_TID; r < P.ns2; r += WS_NT) {
                double s = part[r];
                for (int q = 1; q < P.gp; ++q) s += part[q * P.ns2 + r];
                xi[r] = s;
            }
        }
        WS_SYNC();
        prof_mark(pid);
    }
    const int *rinfo = TBI(rinfo);
    const double *inr = TBV(inr);
    for (int r = WS_TID; r < m; r += WS_NT) {
        if (skip(r)) continue;
        double s;
        const int info = rinfo[r];
        if (r < mc) {
            const int t = info >> 16, i = info & 0xffff;
            const bool last = t == P.T - 1;
            const int rs = last ? P.nh1 : P.nh;                   // rows of the stage = stride of the transposed tables
            const double *Fr = (last ? TBV(sF1) : TBV(sF)) + i;
            const double *Gr = (last ? TBV(sG1) : TBV(sG)) + i;
            const double *zt = xi + t * nu;
            double s0 = 0., s1 = 0.;
            int c = 0;
            for (; c + 1 < nu; c += 2) { s0 += Gr[c * rs] * zt[c]; s1 += Gr[(c + 1) * rs] * zt[c + 1]; }
            if (c < nu) s0 += Gr[c * rs] * zt[c];
            if (t > 0) {
                const double *xt = xi + n + (t - 1) * nx;
                c = 0;
                for (; c + 1 < nx; c += 2) { s0 += Fr[c * rs] * xt[c]; s1 += Fr[(c + 1) * rs] * xt[c + 1]; }
                if (c < nx) s0 += Fr[c * rs] * xt[c];
            }
            s = s0 + s1;
        } else {
            s = xi[info];
        }
        f(r, s * inr[r]);
    }
}

// ---------------------------------------------------------------------------------------------
// slot state
// ---------------------------------------------------------------------------------------------

// ---------------------------------------------------------------------------------------------
// TMA bulk copies (cp.async.bulk, SASS UBLKCP): the copy engine moves a contiguous image between the lane's pool and
// the slot's global home while the threads do something else; completion of a load is signalled on an mbarrier.
// Sizes are multiples of 16 bytes, both addresses 16-byte aligned.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bulk_g2s(void *sdst, const void *gsrc, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(sdst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_s2g(void *gdst, const void *ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" :: "l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit_wait() {
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}
// the lane's mbarrier (one 64-bit word of `red`) and its phase bit (idep[9])
#define WS_MBAR (reinterpret_cast<uint64_t *>(SMV(red) + 100))

// once per kernel launch, by ALL threads of the CTA: the shared copies of the stage rows, row scalings and the
// row -> (stage, index) map (one copy for all lanes), then every lane clears its own vectors.  Contains __syncthreads:
// call it before any lane leaves the kernel.
__device__ __forceinline__ void init_shared_tables(const DevProblem &P, const Ctx &cx) {
    // stage rows TRANSPOSED (entry (row i, column c) at c * rows + i): adjacent threads price adjacent rows, so
    // their reads of one column are consecutive words (no bank conflicts)
    const int nt = blockDim.x, t0 = threadIdx.x;
    double *sF = cx.tab + P.so.t_sF, *sG = cx.tab + P.so.t_sG, *sF1 = cx.tab + P.so.t_sF1, *sG1 = cx.tab + P.so.t_sG1;
    for (int e = t0; e < P.nh * P.nx; e += nt) { const int i = e / P.nx, c = e - i * P.nx; sF[c * P.nh + i] = P.F[e]; }
    for (int e = t0; e < P.nh * P.nu; e += nt) { const int i = e / P.nu, c = e - i * P.nu; sG[c * P.nh + i] = P.G[e]; }
    for (int e = t0; e < P.nh1 * P.nx; e += nt) { const int i = e / P.nx, c = e - i * P.nx; sF1[c * P.nh1 + i] = P.F1[e]; }
    for (int e = t0; e < P.nh1 * P.nu; e += nt) { const int i = e / P.nu, c = e - i * P.nu; sG1[c * P.nh1 + i] = P.G1[e]; }
    int *rinfo = reinterpret_cast<int *>(cx.tab + P.so.t_rinfo);
    for (int r = t0; r < P.m; r += nt) {
        (cx.tab + P.so.t_inr)[r] = P.inr[r]; (cx.tab + P.so.t_vsc)[r] = P.vscale[r];
        int info;
        if (r < P.mc) { int t = r / P.nh; if (t > P.T - 1) t = P.T - 1; info = (t << 16) | (r - t * P.nh); }
        else info = P.bin_idx[r - P.mc];
        rinfo[r] = info;
    }
    for (int i = WS_TID; i < P.np + 2; i += WS_NT) { SMV(z)[i] = 0.; SMV(v)[i] = 0.; SMV(wv)[i] = 0.; SMV(yc)[i] = 0.; }
    for (int i = WS_TID; i < P.ns2; i += WS_NT) SMV(xi)[i] = 0.;
    if (WS_TID == 0) { store_geom(P, cx, 0); SMI(idep)[9] = 0; mbar_init(WS_MBAR, 1); fence_async_smem(); }
    __syncthreads();
}

// working set of the slot: empty (reset) or the one stored by the previous launch.  The factor is NOT
// loaded: every node rebuilds it (rebuild_factor).
__device__ __forceinline__ void load_slot(const DevProblem &P, const Ctx &cx, const SlotPtrs &sp, int &k, bool reset) {
    const int n = P.n;
    if (reset) {
        for (int i = WS_TID; i < n; i += WS_NT) SMV(yc)[i] = 0.;
        k = 0;
    } else {
        k = *sp.nW;
        for (int i = WS_TID; i < n; i += WS_NT) SMV(yc)[i] = sp.yc[i];
        for (int i = WS_TID; i < k; i += WS_NT) { SMI(irow)[i] = sp.row[i]; SMI(iside)[i] = sp.side[i]; SMV(lam)[i] = sp.lam[i]; }
    }
    WS_SYNC();
}

__device__ __forceinline__ void store_slot(const DevProblem &P, const Ctx &cx, const SlotPtrs &sp, int k) {
    const int n = P.n;
    for (int i = WS_TID; i < n; i += WS_NT) sp.yc[i] = SMV(yc)[i];
    for (int i = WS_TID; i < k; i += WS_NT) { sp.row[i] = SMI(irow)[i]; sp.side[i] = SMI(iside)[i]; sp.lam[i] = SMV(lam)[i]; }
    if (WS_TID == 0) *sp.nW = k;
    WS_SYNC();
}

// Working set from signed multipliers of the ORIGINAL rows (ysigned(r) > 0: upper side, < 0: lower side) and a
// proximal centre: the start the reference hands from a parent to its children (`active_set`,
// controller.py:262-264, 426) and what a shifted dual solution gives a warm-start root.  Rows keep their
// natural order.  yc0 may be null (centre 0).  A row enters only if its multiplier is finite and it is a bound row
// (either side) or a stage row with y > 0: a stage row has no lower side, so every other entry is ignored (projected
// to zero), and the start stays dual feasible whatever the caller passes.
template <class Y>
__device__ __forceinline__ void load_ws_from_multipliers(const DevProblem &P, const Ctx &cx, Y ysigned, const double *yc0, int &k) {
    const int lane = WS_TID & 31, w = WS_TID >> 5;
    int *wsum = SMI(ired);                       // WS_NW ints
    int *row = SMI(irow), *side = SMI(iside);
    double *lam = SMV(lam);
    const int d = SMI(idep)[0];
    for (int i = WS_TID; i < P.n; i += WS_NT) SMV(yc)[i] = yc0 ? yc0[i] : 0.;
    int base = 0;
    for (int r0 = 0; r0 < P.m; r0 += WS_NT) {
        const int r = r0 + WS_TID;
        double yv = 0.;
        if (r < P.m) yv = ysigned(r);
        const bool entry = isfinite(yv) && (r < P.mc ? yv > 0. : yv != 0.);
        const int keep = entry && base < P.n && !(r >= P.mc && r - P.mc < d);   // eliminated rows carry no working-set entry
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        WS_SYNC();
        if (lane == 0) wsum[w] = __popc(bal);
        WS_SYNC();
        int pre = base, tot = 0;
        for (int q = 0; q < WS_NW; ++q) { const int c = wsum[q]; if (q < w) pre += c; tot += c; }
        const int idx = pre + __popc(bal & ((1u << lane) - 1u));
        if (keep && idx < P.n) { row[idx] = r; side[idx] = yv > 0. ? 1 : -1; lam[idx] = fabs(yv) * P.nrm[r]; }
        base += tot;
    }
    k = base < P.n ? base : P.n;
    WS_SYNC();
#ifndef WS_NO_SORT
    // Order the start by DECREASING multiplier: the rows the ratio test drops first (small multipliers) sit at the end
    // of the factor, where a removal rotates few columns (position k - 1 costs nothing); rank by counting, ties by row.
    {
        int *scr = SMI(iscr); double *tmp = SMV(cw);
        for (int i = WS_TID; i < k; i += WS_NT) {
            const double li = lam[i];
            int rank = 0;
            for (int j = 0; j < k; ++j) { const double lj = lam[j]; rank += (lj > li || (lj == li && j < i)) ? 1 : 0; }
            scr[i] = rank | (row[i] << 10) | (side[i] > 0 ? (1 << 30) : 0);     // rank < 1024 (k <= n <= 2 WS_NT), row < 2^20
            tmp[i] = li;
        }
        WS_SYNC();
        for (int i = WS_TID; i < k; i += WS_NT) {
            const int e = scr[i], rank = e & 0x3ff;
            row[rank] = (e >> 10) & 0xfffff; side[rank] = (e >> 30) & 1 ? 1 : -1; lam[rank] = tmp[i];
        }
        WS_SYNC();
    }
#endif
}

// Start of a node: rebuild the factor of the inherited working set (rows in their stored order, keeping
// their multipliers, dropping rows that have become dependent) and reset the anti-cycling bookkeeping.
// Mirrors the warm start of oracle/qp_core.c qp_solve.
__device__ __forceinline__ void rebuild_factor(const DevProblem &P, const Ctx &cx, int &k) {
    const Geom gm = load_geom(P, cx);
    signed char *inW = reinterpret_cast<signed char *>(SMB(binW));
    unsigned char *ign = SMB(bign), *nadd = SMB(bnadd);
    const int d = gm.d;
    for (int r = WS_TID; r < P.m; r += WS_NT) { inW[r] = 0; ign[r] = (r >= P.mc && r - P.mc < d) ? 3 : 0; nadd[r] = 0; }
    // the inherited rows are parked in scratch while the factor grows from the front
    const int k0 = k;
    double *lam0 = SMV(cw), *lam = SMV(lam);
    int *row = SMI(irow), *side = SMI(iside);
    int *row0 = SMI(iscr);                           // (row, side) packed, n + 1 ints
    WS_SYNC();
    for (int i = WS_TID; i < k0; i += WS_NT) { row0[i] = row[i] * 2 + (side[i] > 0 ? 1 : 0); lam0[i] = lam[i]; }
    WS_SYNC();
    k = 0;
    RowEnt pre = load_row_entries(P, k0 > 0 ? row0[0] >> 1 : 0, d, gm.d0);
    for (int i = 0; i < k0; ++i) {
        const int r = row0[i] >> 1, s = (row0[i] & 1) ? 1 : -1;
        const RowEnt cur = pre;
        if (i + 1 < k0) pre = load_row_entries(P, row0[i + 1] >> 1, d, gm.d0);      // in flight during this append
        if (r >= P.mc && r - P.mc < d) continue;          // eliminated in this node
        if (thin_append(P, cx, k, r, s, false, &cur) > 0) {
            if (WS_TID == 0) { lam[k - 1] = lam0[i]; inW[r] = (signed char)s; }
        }
    }
    WS_SYNC();
}

// ---------------------------------------------------------------------------------------------
// Sibling memo.  The two children of a node start from the same rows (their parent's, in the same order) with the same
// eliminated prefix, so the factor the first one rebuilds is, bit for bit, the factor the second one would rebuild.
// It is parked in the slot's global home (the columns < ks of the home are otherwise unused) right after the rebuild
// and read back by the sibling: 2 x 50 KB of L2 traffic instead of ~40 Gram-Schmidt appends.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void save_factor(const DevProblem &P, const Ctx &cx, const SlotPtrs &sp, int k) {
    const Geom gm = load_geom(P, cx);
    // the k columns are all in the pool (caller checks k <= ks): the Ri image, then the Q1 columns at their pool stride, go
    // to the slot's home as two bulk copies issued by one thread while the others write the bookkeeping
#ifdef WS_NO_TMA
    for (int e = WS_TID; e < tri_off(k); e += WS_NT) sp.Ri[e] = SMV(pool)[e];
    for (int e = WS_TID; e < k * gm.ldc; e += WS_NT) sp.Q[e] = (SMV(pool) + gm.triR)[e];
    if (WS_TID == 0) *sp.nW = k;
#else
    if (WS_TID == 0) {
        fence_async_smem();                               // the factor was written through the generic proxy
        bulk_s2g(sp.Ri, SMV(pool), (uint32_t)(((tri_off(k) + 1) & ~1) * 8));
        bulk_s2g(sp.Q, SMV(pool) + gm.triR, (uint32_t)(k * gm.ldc * 8));
        bulk_commit_wait();                               // the sibling reads the home much later, from this lane
        *sp.nW = k;
    }
#endif
    for (int i = WS_TID; i < k; i += WS_NT) { sp.row[i] = SMI(irow)[i]; sp.side[i] = SMI(iside)[i]; sp.lam[i] = SMV(lam)[i]; }
    WS_SYNC();
}

// the state rebuild_factor leaves behind, from the memo (same eliminated prefix, hence same geometry).  Ends with a barrier.
__device__ __forceinline__ void restore_factor(const DevProblem &P, const Ctx &cx, const SlotPtrs &sp, int &k) {
    const Geom gm = load_geom(P, cx);
    signed char *inW = reinterpret_cast<signed char *>(SMB(binW));
    unsigned char *ign = SMB(bign), *nadd = SMB(bnadd);
    const int d = gm.d;
    k = *sp.nW;
    int *phase = SMI(idep) + 9;
    const uint32_t par = (uint32_t)*phase;
    WS_SYNC();                                            // nobody still reads the pool; everybody has read the phase bit
#ifdef WS_NO_TMA
    for (int e = WS_TID; e < tri_off(k); e += WS_NT) SMV(pool)[e] = sp.Ri[e];
    for (int e = WS_TID; e < k * gm.ldc; e += WS_NT) (SMV(pool) + gm.triR)[e] = sp.Q[e];
#else
    if (WS_TID == 0) {
        const uint32_t bR = (uint32_t)(((tri_off(k) + 1) & ~1) * 8), bQ = (uint32_t)(k * gm.ldc * 8);
        fence_async_smem();
        mbar_expect_tx(WS_MBAR, bR + bQ);
        bulk_g2s(SMV(pool), sp.Ri, bR, WS_MBAR);
        bulk_g2s(SMV(pool) + gm.triR, sp.Q, bQ, WS_MBAR);
        *phase = (int)(par ^ 1u);
    }
#endif
    // ... while the copy engine streams the factor in, the threads reset the row flags and fetch the bookkeeping
    for (int r = WS_TID; r < P.m; r += WS_NT) { inW[r] = 0; ign[r] = (r >= P.mc && r - P.mc < d) ? 3 : 0; nadd[r] = 0; }
    for (int i = WS_TID; i < k; i += WS_NT) { SMI(irow)[i] = sp.row[i]; SMI(iside)[i] = sp.side[i]; SMV(lam)[i] = sp.lam[i]; }
    WS_SYNC();
    for (int i = WS_TID; i < k; i += WS_NT) inW[SMI(irow)[i]] = (signed char)SMI(iside)[i];
#ifndef WS_NO_TMA
    mbar_wait(WS_MBAR, par);
#endif
    WS_SYNC();
}

// ---------------------------------------------------------------------------------------------
// pinned-prefix elimination.  problem.py rotates v so that the bound row of binary j (chronological order) has
// its non-zeros in columns 0..j.  A node whose first d binaries are pinned (lb == ub: every node branch_in_time
// creates, controller.py:13-44) has v[:d] fixed by those d rows; the solver works in the coordinates d..n-1
// (rows enter the factor with their first d entries dropped, the bounds are shifted by mh_r[:d] . v_f) and
// the multipliers of the d eliminated rows follow from stationarity in the eliminated coordinates.
// ---------------------------------------------------------------------------------------------

// d from the bounds of the node; fixes the geometry of the factor.  Ends with a barrier.
__device__ __forceinline__ void set_node_prefix(const DevProblem &P, const Ctx &cx, const double *lb, const double *ub) {
    double far = 0.;                                        // nb - (first binary that is not pinned)
    for (int j = WS_TID; j < P.nb; j += WS_NT) if (lb[j] != ub[j]) far = fmax(far, (double)(P.nb - j));
    far = block_max(far, SMV(red));
    if (WS_TID == 0) store_geom(P, cx, P.nb - (int)far);
    WS_SYNC();
}

// d known by the caller (depth of a branch_in_time node).  The caller provides the barrier.
__device__ __forceinline__ void set_node_prefix_known(const DevProblem &P, const Ctx &cx, int d) {
    if (WS_TID == 0) store_geom(P, cx, d);
}

// y_out of the eliminated rows:  L' eta = -( [v_f] + sum_i coef_i mh_{row_i}[:d] + pcoef mh_pend[:d] )
__device__ __forceinline__ void pinned_multipliers(const DevProblem &P, const Ctx &cx, int k, int d, const double *coef,
                                          int pend, double pcoef, bool with_v, double *y_out) {
    if (d == 0) return;
    double *g = SMV(c2);
    const int *row = SMI(irow);
    for (int c = WS_TID; c < d; c += WS_NT) {
        double s0 = with_v ? SMV(vf)[c] : 0., s1 = 0.;
        int i = 0;
        for (; i + 1 < k; i += 2) {
            s0 += coef[i] * __ldg(P.Mh + (size_t)row[i] * P.n + c);
            s1 += coef[i + 1] * __ldg(P.Mh + (size_t)row[i + 1] * P.n + c);
        }
        if (i < k) s0 += coef[i] * __ldg(P.Mh + (size_t)row[i] * P.n + c);
        if (pend >= 0) s1 += pcoef * __ldg(P.Mh + (size_t)pend * P.n + c);
        g[c] = s0 + s1;
    }
    WS_SYNC();
    for (int j = WS_TID; j < d; j += WS_NT) {
        double s0 = 0., s1 = 0.;
        int c = j;
        for (; c + 1 < d; c += 2) { s0 += __ldg(P.Linv + (size_t)c * P.nb + j) * g[c]; s1 += __ldg(P.Linv + (size_t)(c + 1) * P.nb + j) * g[c + 1]; }
        if (c < d) s0 += __ldg(P.Linv + (size_t)c * P.nb + j) * g[c];
        y_out[P.mc + j] = -(s0 + s1) * TBV(inr)[P.mc + j];
    }
    WS_SYNC();
}

// ---------------------------------------------------------------------------------------------
// the solver.  Inputs: x0 (global), lb/ub (global, nb).  The working set (rows, sides, lam, k) must be
// loaded (load_slot) -- its factor is rebuilt here.  Outputs: status; yc = solution in orthonormal
// coordinates (if optimal); y_out (global, m): signed multipliers of the ORIGINAL rows (>0 upper side,
// <0 lower side; Farkas ray if infeasible).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int qp_solve(const DevProblem &P, const Ctx &cx, int &k,
                               const double *x0, const double *lb, const double *ub,
                               double *y_out, int *iters_out, int *kmax_out,
                               int memo, const SlotPtrs &sp, int &memo_saved)
{
    // memo: 0 rebuild the factor of the loaded working set; 1 rebuild it and park it in the slot's home (*memo_saved = 1
    // if it fitted); 2 the working set was NOT loaded: take it and its factor from the slot's home (sibling memo)
    const int n = P.n, m = P.m, mc = P.mc, nx = P.nx;
    signed char *inW = reinterpret_cast<signed char *>(SMB(binW));
    unsigned char *ign = SMB(bign), *nadd = SMB(bnadd);
    double *lam = SMV(lam), *ls = SMV(ls), *t = SMV(t), *bu = SMV(bu), *blb = SMV(blb), *vsc = TBV(vsc);
    int *row = SMI(irow), *side = SMI(iside);
    double *red = SMV(red); int *ired = SMI(ired);
    int it = 0, status = WS_ITER_LIMIT, kmax = 0;
    bool hot = k > 0 || memo == 2;
    int cap = hot ? min(P.hot_cap, P.max_iter) : P.max_iter;
    memo_saved = 0;

    // eliminated coordinates: L v_f = b with b_j = ub_j / nrm_j + (Mh wv)_j  =>  v_f = vf0 + wv[:d], vf0 = L^-1 (ub / nrm)
    const int d = SMI(idep)[0];
    for (int c = WS_TID; c < d; c += WS_NT) {
        double s0 = 0., s1 = 0.;
        int j = 0;
        for (; j + 1 <= c; j += 2) {
            s0 += __ldg(P.LinvT + (size_t)j * P.nb + c) * (ub[j] * TBV(inr)[mc + j]);
            s1 += __ldg(P.LinvT + (size_t)(j + 1) * P.nb + c) * (ub[j + 1] * TBV(inr)[mc + j + 1]);
        }
        if (j <= c) s0 += __ldg(P.LinvT + (size_t)j * P.nb + c) * (ub[j] * TBV(inr)[mc + j]);
        SMV(vf0)[c] = s0 + s1;
    }
    WS_SYNC();
    prof_mark(2);

restart:
    if (memo == 2) {
        restore_factor(P, cx, sp, k);
    } else {
        rebuild_factor(P, cx, k);
        if (memo == 1 && k > 0 && k <= SMI(idep)[5]) { save_factor(P, cx, sp, k); memo_saved = 1; }
    }
    memo = 0;                                   // a restart from the empty working set rebuilds
    prof_mark(3);
    kmax = max(kmax, k);
    const int k_start = k; int n_prox = 0;
    int pending = -1, pside = 0, just_added = -1, n_verify = 0;
    bool prox_conv = false;
    if (WS_TID == 0) SMI(idep)[1] = 0;
    double plam = 0.;
    for (int pk = 0; pk < P.max_prox; ++pk) {
        ++n_prox;
        // wv = Kx x0 - eps Rinv' yc     ((Rinv' yc)_c = sum_r Rinv[r][c] yc[r], coalesced over c)
        grouped_matvec(P.Rinv, n, n, 0, n, SMV(yc), SMV(part), [&](int c, double a) {
            double s = 0.;
            for (int j = 0; j < nx; ++j) s += P.Kx[(size_t)c * nx + j] * x0[j];
            const double w = s - P.eps * a;
            if (c < d) { SMV(vf)[c] = SMV(vf0)[c] + w; SMV(wv)[c] = -SMV(vf0)[c]; }      // wv - [v_f; 0]: the bounds below come out shifted
            else SMV(wv)[c] = w;
        });
        prof_mark(4);
        // bounds of this proximal sub-problem: g = Mh wv
        price_rows(P, cx, SMV(wv), 0, 60, [](int) { return false; }, [&](int r, double g) {
            if (r < mc) {
                double e = 0.;
                for (int j = 0; j < nx; ++j) e += P.Eh[(size_t)r * nx + j] * x0[j];
                bu[r] = P.hh[r] - e + g;
            } else {
                const int i = r - mc;
                const double inr = TBV(inr)[r];
                bu[r] = ub[i] * inr + g;
                blb[i] = lb[i] * inr + g;
            }
        });
        WS_SYNC();
        prof_mark(5);
        refresh_uv(P, cx, k);
        prof_mark(6);

        status = WS_ITER_LIMIT;
        while (it < cap) {
            ++it;
            // an iteration decides on at most one removal (position `rem`) and one append (row `app`, side `apps`); both are
            // carried out at the END of the iteration, by the only inlined copies of the removal and of the tracked append
            int rem = -1, app = -1, apps = 0;
            if (pending < 0) {
                // ratio test on the way to lam* = ls ; sum of the positive multipliers
                // every warp runs the whole test (k / 32 entries per lane): no barrier, same bits in every thread
                double amin = INFINITY, lpart = 0.; int kmin = -1;
                for (int i = WS_TID & 31; i < k; i += 32) {
                    const double l = ls[i];
                    if (l < -P.tol_d) {
                        const double a = lam[i] / (lam[i] - l);
                        if (a < amin || (a == amin && i < kmin)) { amin = a; kmin = i; }
                    }
                    lpart += l > 0. ? l : 0.;
                }
                warp_argmin_sum(amin, kmin, lpart);
                WS_SYNC();                                  // every warp has read lam, ls before they change
                prof_mark(7);
                if (hot && !(lpart < WS_LAM_MAX)) break;          // degenerate hot start: restart cold
                if (kmin >= 0) {
                    for (int i = WS_TID; i < k; i += WS_NT) lam[i] += amin * (ls[i] - lam[i]);
                    WS_SYNC();
                    if (WS_TID == 0) {
                        const int rr = row[kmin];
                        if (rr == just_added && lam[kmin] == 0.) { ign[rr] |= (side[kmin] > 0 ? 1 : 2); SMI(idep)[1] = 1; }
                        if (amin <= 1e-9 && nadd[rr] < 255) ++nadd[rr];
                    }
                    just_added = -1;
                    prof_mark(8);
                    rem = kmin;
                } else {
                for (int i = WS_TID; i < k; i += WS_NT) lam[i] = ls[i] > 0. ? ls[i] : 0.;
                const double vnoise = 1e-14 * lpart, vcap = 100. * P.tol_p;
                double vbest = 0.; int ibest = -1;                 // ibest = 2 r + (lower side)
                price_rows(P, cx, SMV(v), d, 62, [&](int r) { return inW[r] != 0 || ign[r] == 3; }, [&](int r, double sv) {
                    const int na = nadd[r];
                    double tolr = P.tol_p * (na == 0 ? 1. : (na == 1 ? 10. : 100.));
                    const double vs = vsc[r];
                    const double fl = vnoise * vs < vcap ? vnoise * vs : vcap;
                    if (fl > tolr) tolr = fl;
                    const int ig = ign[r];
                    if (!(ig & 1)) {
                        const double vu = (sv - bu[r]) * vs;
                        if (vu > tolr && (vu > vbest || (vu == vbest && 2 * r < ibest))) { vbest = vu; ibest = 2 * r; }
                    }
                    if (r >= mc && !(ig & 2)) {
                        const double vl = (blb[r - mc] - sv) * vs;
                        if (vl > tolr && (vl > vbest || (vl == vbest && 2 * r + 1 < ibest))) { vbest = vl; ibest = 2 * r + 1; }
                    }
                });
                prof_mark(10);
                block_argmax(vbest, ibest, red, ired);
                prof_mark(11);
                if (ibest < 0) {
                    // Rows put on the anti-cycling ignore list stay there across the proximal passes although the bounds move:
                    // before the point is declared optimal, price them once more, unfiltered, against the loosest tolerance the
                    // pricing ever uses (100 tol_p); a row violated beyond that is given back to the method (at most twice).
                    if (SMI(idep)[1] != 0 && n_verify < 2) {
                        double wbest = 0.; int wi = -1;
                        price_rows(P, cx, SMV(v), d, 63, [&](int r) { return inW[r] != 0 || ign[r] == 3 || ign[r] == 0; }, [&](int r, double sv) {
                            const double vs = vsc[r];
                            const double vu = (sv - bu[r]) * vs;
                            if (vu > vcap && vu > wbest) { wbest = vu; wi = r; }
                            if (r >= mc) { const double vl = (blb[r - mc] - sv) * vs; if (vl > vcap && vl > wbest) { wbest = vl; wi = r; } }
                        });
                        block_argmax(wbest, wi, red, ired);
                        ++n_verify;
                        if (WS_TID == 0) SMI(idep)[1] = 0;
                        if (wi >= 0) {
                            for (int r = WS_TID; r < m; r += WS_NT) if (ign[r] != 3) ign[r] = 0;
                            WS_SYNC();
                            continue;
                        }
                        WS_SYNC();
                    }
                    status = WS_OPTIMAL; break;
                }
                app = ibest >> 1; apps = (ibest & 1) ? -1 : 1;
                }
            } else {
                // dependent entering row: dual ray (p_W, 1), p_W = -t
                double pm = 1.;
                for (int i = WS_TID; i < k; i += WS_NT) pm = fmax(pm, fabs(t[i]));
                pm = block_max(pm, red);
                double amin = INFINITY; int kmin = -1;
                for (int i = WS_TID; i < k; i += WS_NT) if (t[i] > P.tol_ray * pm) {
                    const double a = lam[i] / t[i];
                    if (a < amin || (a == amin && i < kmin)) { amin = a; kmin = i; }
                }
                block_argmin(amin, kmin, red, ired);
                prof_mark(13);
                if (kmin < 0) {
                    double cpart = 0., wpart = 0.;
                    for (int i = WS_TID; i < k; i += WS_NT) {
                        const double pi = t[i] < 0. ? -t[i] : 0.;
                        const int r = row[i];
                        cpart -= pi * (side[i] > 0 ? bu[r] : -blb[r - mc]);
                        wpart += pi / vsc[r];
                    }
                    double cost = cpart, wsum = wpart;
                    block_sum2(cost, wsum, red);
                    cost -= (pside > 0 ? bu[pending] : -blb[pending - mc]);
                    wsum += 1. / vsc[pending];
                    if (cost > P.tol_p * wsum) {
                        for (int r = WS_TID; r < m; r += WS_NT) y_out[r] = 0.;
                        WS_SYNC();
                        for (int i = WS_TID; i < k; i += WS_NT) {
                            const double pi = t[i] < 0. ? -t[i] : 0.;
                            const int r = row[i];
                            y_out[r] = (double)side[i] * pi * TBV(inr)[r];
                        }
                        if (WS_TID == 0) y_out[pending] = (double)pside * TBV(inr)[pending];
                        for (int i = WS_TID; i < k; i += WS_NT) SMV(cw)[i] = (double)side[i] * (t[i] < 0. ? -t[i] : 0.);
                        WS_SYNC();
                        pinned_multipliers(P, cx, k, d, SMV(cw), pending, (double)pside, false, y_out);
                        status = WS_INFEASIBLE;
                        break;
                    }
                    if (WS_TID == 0) { ign[pending] |= (pside > 0 ? 1 : 2); SMI(idep)[1] = 1; }
                    pending = -1;
                    WS_SYNC();
                    continue;
                }
                for (int i = WS_TID; i < k; i += WS_NT) lam[i] -= amin * t[i];
                plam += amin;
                WS_SYNC();
                if (WS_TID == 0 && amin <= 1e-9 * (1. + plam) && nadd[row[kmin]] < 255) ++nadd[row[kmin]];
                rem = kmin; app = pending; apps = pside;
            }
            if (rem >= 0) ws_remove(P, cx, k, rem);
            if (app >= 0) {
                const int ar = thin_append(P, cx, k, app, apps, true);
                if (pending < 0) {
                    if (ar < 0) break;                                  // capacity: reported as iteration limit
                    if (ar) {
                        kmax = max(kmax, k);
                        if (WS_TID == 0) inW[app] = (signed char)apps;
                        just_added = app;
                        WS_SYNC();
                    } else { pending = app; pside = apps; plam = 0.; }
                } else if (ar > 0) {
                    if (WS_TID == 0) { lam[k - 1] = plam; inW[pending] = (signed char)pside; }
                    pending = -1;
                    WS_SYNC();
                }
            }
        }
        if (status != WS_OPTIMAL) break;
        // yc <- Rinv (v - wv) ; proximal convergence
        WS_SYNC();
        for (int r = WS_TID; r < n; r += WS_NT) SMV(c1)[r] = SMV(v)[r] - SMV(wv)[r];
        WS_SYNC();
        double dz = 0.;
        grouped_matvec(P.RinvT, n, n, 0, n, SMV(c1), SMV(part), [&](int r, double s) {
            dz = fmax(dz, fabs(s - SMV(yc)[r]));
            SMV(c2)[r] = s;
        });
        dz = block_max(dz, red);
        prof_mark(15);
        for (int r = WS_TID; r < n; r += WS_NT) SMV(yc)[r] = SMV(c2)[r];
        WS_SYNC();
        if (P.eps * dz <= P.prox_tol) { prox_conv = true; break; }
    }
    // max_prox passes without meeting the proximal tolerance: the iterate is not the optimum -- report it as an iteration limit
    if (status == WS_OPTIMAL && !prox_conv) status = WS_ITER_LIMIT;
    if (status == WS_ITER_LIMIT && hot) {
        // a hot start from a stale, nearly dependent working set can degenerate: solve once more from scratch
        hot = false; cap = it + P.max_iter; k = 0;
        for (int i = WS_TID; i < n; i += WS_NT) SMV(yc)[i] = 0.;
        WS_SYNC();
        goto restart;
    }
    if (status == WS_OPTIMAL) {
        for (int r = WS_TID; r < m; r += WS_NT) y_out[r] = 0.;
        WS_SYNC();
        for (int i = WS_TID; i < k; i += WS_NT) {
            const int r = row[i];
#ifdef WS_KEEPW
            y_out[r] = (double)side[i] * fmax(lam[i], 1e-200) * TBV(inr)[r];
#else
            y_out[r] = (double)side[i] * lam[i] * TBV(inr)[r];
#endif
            SMV(cw)[i] = (double)side[i] * lam[i];
        }
        WS_SYNC();
        pinned_multipliers(P, cx, k, d, SMV(cw), -1, 0., true, y_out);
    }
    prof_mark(16);
    if (WS_TID == 0) { *iters_out = it; if (kmax_out) { kmax_out[0] = kmax; kmax_out[1] = k_start | (n_prox << 16); } }
    return status;
}
