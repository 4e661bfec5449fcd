// wshmpc.cu -- kernels + C ABI (include/wshmpc.h) of the B200-native hybrid-MPC B&B hot path.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
#include "../../include/wshmpc.h"
#include "qp_device.cuh"
#include "records.cuh"
#include "bnb.cuh"
#if WS_TU_HAS(0)
#include "lp_batch.cuh"
#endif
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

static thread_local std::string g_err;
#define WS_FAIL(code, ...) do { char _b[512]; snprintf(_b, sizeof(_b), __VA_ARGS__); g_err = _b; return code; } while (0)
#define WS_CUDA(x) do { cudaError_t _e = (x); if (_e != cudaSuccess) WS_FAIL(-2, "%s failed: %s (%s:%d)", #x, cudaGetErrorString(_e), __FILE__, __LINE__); } while (0)

#if WS_TU_HAS(0)
struct wshmpc_handle {
    DevProblem P;            // shared-memory layout for P.lanes solver lanes per CTA (throughput launches)
    DevProblem P1;           // the same problem laid out for ONE lane per CTA (launches that cannot fill two lanes per SM)
    int n_sm;
    int *d_border;           // device copy of the branching order (wshmpc_set_branch_order)
    void *hot_ptr; size_t hot_bytes; int l2_window;      // L2 persistence window over WfT | Mh (l2_window = 1 if it was accepted)
    int device, n_slots;
    cudaStream_t stream;
    std::vector<void *> allocs;
    double *slot_d;
    int *slot_i;
    double *ybuf;            // n_slots x m : signed row multipliers of the node being solved
    double *scratch;         // n_slots x bnb_scratch_doubles : node bounds, primal record of the node being solved
    int *work_counter;       // instance hand-out of the B&B kernel
    size_t shift_smem; int shift_stage;      // dynamic shared memory of shift_tree_kernel, of which staging buffers (doubles)
    size_t smem;
    wshmpc_layout layout;
    double *plant_stage; int plant_stage_n;              // wshmpc_closed_loop_plant: [n][nx] model errors (allocated on first use)
};

extern "C" const char *wshmpc_last_error(void) { return g_err.c_str(); }
static int g_lanes_last = WS_MAXL;
// solver states resident per SM: lanes per CTA of the most recently created handle (WS_MAXL before any handle exists)
extern "C" int wshmpc_ctas_per_sm(void) { return g_lanes_last; }
#ifdef WS_PROF
// experiment builds only: [2 id] cycles, [2 id + 1] visits of phase id (see prof_mark)
extern "C" int wshmpc_prof_read(unsigned long long *out, int reset) {
    if (out) cudaMemcpyFromSymbol(out, g_prof, sizeof(g_prof));
    if (reset) { static unsigned long long z[256]; cudaMemcpyToSymbol(g_prof, z, sizeof(z)); }
    return 0;
}
#endif

#endif

// ---------------------------------------------------------------------------------------------
// K1: one CTA per solver slot; the CTA solves, in index order, every node assigned to its slot
// ---------------------------------------------------------------------------------------------
// LANES: solver lanes per CTA the kernel is compiled for (its register budget is 65536 / (LANES WS_NT) per thread): the
// one-lane instantiation keeps 255 registers per thread and serves launches that cannot fill two lanes per SM anyway
// (single-instance latency, the large systems); results do not depend on the choice.
template <int LANES>
__device__ __forceinline__ void
solve_nodes_body(const DevProblem &P, double *slot_d, int *slot_i, double *ybuf, int n_slots, int n_nodes,
                   const double *__restrict__ x0, const double *__restrict__ lb, const double *__restrict__ ub,
                   const int *__restrict__ slot_of, const int *__restrict__ hot,
                   const double *__restrict__ y0, const double *__restrict__ yc0,
                   int *status, double *cost, double *dobj, int *iters, double *primal, double *dual, double *yc_out)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int slot = blockIdx.x * LANES + WS_LANE;
    SlotPtrs sp = slot_ptrs(slot_d, slot_i, slot < n_slots ? slot : 0, P.n, P.ld);
    const Ctx cx = make_ctx(P, smem_raw, sp);
    init_shared_tables(P, cx);
    if (slot >= n_slots) return;                       // a lane without a solver state (after the CTA-wide barrier)
    double *y = ybuf + (size_t)slot * P.m;
    int k = 0;
    bool loaded = false;
    for (int i = 0; i < n_nodes; ++i) {
        if (slot_of[i] != slot) continue;
        const int hm = hot[i];
        const double *xi = x0 + (size_t)i * P.nx, *lbi = lb + (size_t)i * P.nb, *ubi = ub + (size_t)i * P.nb;
        set_node_prefix(P, cx, lbi, ubi);
        if (hm == 2 && y0) {
            const double *yy = y0 + (size_t)i * P.m;
            load_ws_from_multipliers(P, cx, [&](int r) { return yy[r]; }, yc0 ? yc0 + (size_t)i * P.n : nullptr, k);
            loaded = true;
        } else {
            const bool reset = hm == 0;
            if (!loaded || reset) { load_slot(P, cx, sp, k, reset); loaded = true; }
        }
        int memo_saved = 0;
        const int st = qp_solve(P, cx, k, xi, lbi, ubi, y, iters + i, nullptr, 0, sp, memo_saved);
        build_records(P, st, SMV(yc), y, xi, lbi, ubi, primal + (size_t)i * P.n_primal,
                      dual + (size_t)i * P.n_dual, cost + i, dobj + i, SMV(part), SMV(red));
        if (yc_out) for (int j = WS_TID; j < P.n; j += WS_NT) yc_out[(size_t)i * P.n + j] = st == WS_OPTIMAL ? SMV(yc)[j] : 0.;
        if (WS_TID == 0) status[i] = st;
        WS_SYNC();
    }
    if (loaded) store_slot(P, cx, sp, k);
}

#define WS_K1_ARGS DevProblem P, double *slot_d, int *slot_i, double *ybuf, int n_slots, int n_nodes, \
    const double *__restrict__ x0, const double *__restrict__ lb, const double *__restrict__ ub, const int *__restrict__ slot_of, \
    const int *__restrict__ hot, const double *__restrict__ y0, const double *__restrict__ yc0, \
    int *status, double *cost, double *dobj, int *iters, double *primal, double *dual, double *yc_out
#define WS_K1_PASS P, slot_d, slot_i, ybuf, n_slots, n_nodes, x0, lb, ub, slot_of, hot, y0, yc0, status, cost, dobj, iters, primal, dual, yc_out
#define WS_K1_BODY(LANES, RULE, PLANT, FB) solve_nodes_body<LANES>(WS_K1_PASS)

// ---------------------------------------------------------------------------------------------
// The large kernels.  Row u is translation unit u (-DWS_TU=u compiles exactly that kernel; unit 0 holds the C ABI and the
// small kernels).  Columns: unit, name, family (K1: solve_nodes_body, BNB: bnb_body, LOOP: closed_loop_body), solver lanes
// per CTA, node rule (0 the structured search, BNB_RULE_MIQP the conventional MIQP search of wshmpc_set_node_rule 1 and 2),
// nonlinear plant on the device (wshmpc_closed_loop_plant), fallback policy (wshmpc_closed_loop_fallback).  One lane keeps
// 255 registers per thread for launches that cannot fill WS_MAXL lanes per SM (latency mode, large systems); WS_MAXL lanes
// get 65536 / (WS_MAXL WS_NT) (throughput mode).  The one-lane kernels take the odd units, which set WS_WIDE_REGS
// (qp_device.cuh).  The host sets the kernels' attributes and picks the kernel of a launch from this table (kernel_for).
// ---------------------------------------------------------------------------------------------
#define WS_ROW_1(X)  X(1,  solve_nodes_kernel_1,            K1,   1,       0,             0, 0)
#define WS_ROW_2(X)  X(2,  solve_nodes_kernel_m,            K1,   WS_MAXL, 0,             0, 0)
#define WS_ROW_3(X)  X(3,  bnb_kernel_1,                    BNB,  1,       0,             0, 0)
#define WS_ROW_4(X)  X(4,  bnb_kernel_m,                    BNB,  WS_MAXL, 0,             0, 0)
#define WS_ROW_5(X)  X(5,  closed_loop_kernel_1,            LOOP, 1,       0,             0, 0)
#define WS_ROW_6(X)  X(6,  closed_loop_kernel_m,            LOOP, WS_MAXL, 0,             0, 0)
#define WS_ROW_7(X)  X(7,  bnb_miqp_kernel_1,               BNB,  1,       BNB_RULE_MIQP, 0, 0)
#define WS_ROW_8(X)  X(8,  bnb_miqp_kernel_m,               BNB,  WS_MAXL, BNB_RULE_MIQP, 0, 0)
#define WS_ROW_9(X)  X(9,  closed_loop_miqp_kernel_1,       LOOP, 1,       BNB_RULE_MIQP, 0, 0)
#define WS_ROW_10(X) X(10, closed_loop_miqp_kernel_m,       LOOP, WS_MAXL, BNB_RULE_MIQP, 0, 0)
#define WS_ROW_11(X) X(11, closed_loop_plant_kernel_1,      LOOP, 1,       0,             1, 0)
#define WS_ROW_12(X) X(12, closed_loop_plant_kernel_m,      LOOP, WS_MAXL, 0,             1, 0)
#define WS_ROW_13(X) X(13, closed_loop_miqp_plant_kernel_1, LOOP, 1,       BNB_RULE_MIQP, 1, 0)
#define WS_ROW_14(X) X(14, closed_loop_miqp_plant_kernel_m, LOOP, WS_MAXL, BNB_RULE_MIQP, 1, 0)
#define WS_ROW_15(X) X(15, closed_loop_fb_kernel_1,         LOOP, 1,       0,             0, 1)
#define WS_ROW_16(X) X(16, closed_loop_fb_kernel_m,         LOOP, WS_MAXL, 0,             0, 1)
#define WS_ROW_17(X) X(17, closed_loop_plant_fb_kernel_1,   LOOP, 1,       0,             1, 1)
#define WS_ROW_18(X) X(18, closed_loop_plant_fb_kernel_m,   LOOP, WS_MAXL, 0,             1, 1)
#define WS_KERNELS(X) WS_ROW_1(X) WS_ROW_2(X) WS_ROW_3(X) WS_ROW_4(X) WS_ROW_5(X) WS_ROW_6(X) WS_ROW_7(X) WS_ROW_8(X) \
    WS_ROW_9(X) WS_ROW_10(X) WS_ROW_11(X) WS_ROW_12(X) WS_ROW_13(X) WS_ROW_14(X) WS_ROW_15(X) WS_ROW_16(X) WS_ROW_17(X) WS_ROW_18(X)

#define WS_KERNEL_SIG(name, fam, lanes) __global__ void __launch_bounds__((lanes) * WS_NT, 1) name(WS_##fam##_ARGS)
#define WS_DECLARE(u, name, fam, lanes, rule, plant, fb) WS_KERNEL_SIG(name, fam, lanes);
#define WS_DEFINE(u, name, fam, lanes, rule, plant, fb) WS_KERNEL_SIG(name, fam, lanes) { WS_##fam##_BODY(lanes, rule, plant, fb); }
WS_KERNELS(WS_DECLARE)
#ifndef WS_TU
WS_KERNELS(WS_DEFINE)
#elif WS_TU > 0
#define WS_DEFINE_UNIT(u, name, fam, lanes, rule, plant, fb) \
    static_assert(((lanes) == 1) == (WS_WIDE_REGS == 1), #name ": one-lane kernels take the odd units, the others the even ones"); \
    WS_DEFINE(u, name, fam, lanes, rule, plant, fb)
#define WS_CAT_(a, b) a##b
#define WS_CAT(a, b) WS_CAT_(a, b)
WS_CAT(WS_ROW_, WS_TU)(WS_DEFINE_UNIT)
#endif

#if WS_TU_HAS(0)          // the C ABI (host code) lives in unit 0

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
template <class Tv>
static int upload(wshmpc_handle *h, const Tv *src, size_t count, const Tv **dst) {
    void *d = nullptr;
    if (count == 0) count = 1;
    WS_CUDA(cudaMalloc(&d, count * sizeof(Tv)));
    h->allocs.push_back(d);
    if (src) WS_CUDA(cudaMemcpy(d, src, count * sizeof(Tv), cudaMemcpyHostToDevice));
    *dst = (const Tv *)d;
    return 0;
}

static std::vector<double> transpose(const double *a, int rows, int cols) {
    std::vector<double> t((size_t)rows * cols);
    for (int i = 0; i < rows; ++i) for (int j = 0; j < cols; ++j) t[(size_t)j * rows + i] = a[(size_t)i * cols + j];
    return t;
}

enum KernelFamily { FAMILY_K1, FAMILY_BNB, FAMILY_LOOP };
struct KernelRow { void *fn; KernelFamily family; int lanes; bool miqp, plant, fb; };
#define WS_KERNEL_ROW(u, name, fam, lanes, rule, plant, fb) {(void *)name, FAMILY_##fam, lanes, (rule) != 0, (plant) != 0, (fb) != 0},
static const KernelRow g_kernels[] = {WS_KERNELS(WS_KERNEL_ROW)};

// the kernel of `family` compiled for (lanes, node rule != 0, plant, fb); a combination without a row fails with a message
template <class F>
static int kernel_for(KernelFamily family, int lanes, bool miqp, bool plant, bool fb, F *out)
{
    for (const KernelRow &r : g_kernels)
        if (r.family == family && r.lanes == lanes && r.miqp == miqp && r.plant == plant && r.fb == fb) { *out = (F)r.fn; return 0; }
    WS_FAIL(-1, "no kernel of family %d for %d lanes, node rule %s, plant %d, fallback %d", (int)family, lanes, miqp ? "!= 0" : "0",
            (int)plant, (int)fb);
}

// launch shape of a large kernel over `slots` solver states: one lane per CTA (P1) when the states cannot fill P.lanes lanes
// on every SM or the handle has one lane, P.lanes lanes per CTA (P) otherwise.  `lanes` is what the kernel is compiled for.
struct LaunchShape { int lanes; const DevProblem *P; dim3 grid, block; size_t smem; };
static LaunchShape launch_shape(const wshmpc_handle *h, int slots)
{
    const bool one = slots <= h->n_sm || h->P.lanes == 1;
    const DevProblem &P = one ? h->P1 : h->P;
    return {one ? 1 : WS_MAXL, &P, dim3((slots + P.lanes - 1) / P.lanes), dim3(P.lanes * WS_NT), (size_t)P.so.total_bytes};
}

// dynamic shared memory a launch of `fn` may use: the device's opt-in budget less the kernel's static shared memory
static cudaError_t raise_smem_limit(const void *fn, size_t optin)
{
    cudaFuncAttributes fa;
    const cudaError_t e = cudaFuncGetAttributes(&fa, fn);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(optin - fa.sharedSizeBytes));
}

extern "C" int wshmpc_create(const wshmpc_problem *p, int device, int n_slots, void *stream, wshmpc_handle **out)
{
    if (!p || !out) WS_FAIL(-1, "null argument");
    if (n_slots <= 0) WS_FAIL(-1, "n_slots must be positive");
    if (p->n != p->T * p->nu || p->nb != p->T * p->nub || p->m != p->mc + p->nb ||
        p->mc != (p->T - 1) * p->nh + p->nh1 || p->ns != p->n + p->T * p->nx)
        WS_FAIL(-1, "inconsistent sizes: n=%d m=%d mc=%d nb=%d", p->n, p->m, p->mc, p->nb);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) WS_FAIL(-3, "no CUDA device: the hot path has no CPU fallback");
    WS_CUDA(cudaSetDevice(device));
    wshmpc_handle *h = new wshmpc_handle();
    h->device = device; h->n_slots = n_slots; h->stream = (cudaStream_t)stream;
    DevProblem &P = h->P;
    memset(&P, 0, sizeof(P));
    P.nx = p->nx; P.nu = p->nu; P.nub = p->nub; P.nuc = p->nu - p->nub; P.T = p->T; P.nh = p->nh; P.nh1 = p->nh1;
    P.nq = p->nq; P.nqT = p->nqT; P.nr = p->nr; P.n = p->n; P.m = p->m; P.mc = p->mc; P.nb = p->nb; P.ns = p->ns;
    P.eps = p->eps; P.tol_p = p->tol_p; P.tol_d = p->tol_d; P.tol_sing = p->tol_sing; P.tol_ray = p->tol_ray;
    P.prox_tol = p->prox_tol; P.max_iter = p->max_iter; P.max_prox = p->max_prox;
    const int nx = p->nx, nu = p->nu, n = p->n, m = p->m;
    int rc = 0;
#define UP(field, src, cnt) if ((rc = upload(h, src, (size_t)(cnt), &P.field))) { wshmpc_destroy(h); return rc; }
    UP(A, p->A, nx * nx) UP(B, p->B, nx * nu) UP(F, p->F, p->nh * nx) UP(G, p->G, p->nh * nu) UP(h, p->h, p->nh)
    UP(F1, p->F_Tm1, p->nh1 * nx) UP(G1, p->G_Tm1, p->nh1 * nu) UP(h1, p->h_Tm1, p->nh1)
    UP(Q, p->Q, p->nq * nx) UP(R, p->R, p->nr * nu) UP(QT, p->Q_T, p->nqT * nx)
    UP(Mmu, p->M_mu, p->nh * p->nh1) UP(Mrho, p->M_rho, p->nq * p->nqT)
    { std::vector<double> mt = transpose(p->M_mu, p->nh, p->nh1); UP(MmuT, mt.data(), mt.size()) }
    UP(nrm, p->nrm, m) UP(vscale, p->vscale, m) UP(Eh, p->Eh, (size_t)p->mc * nx)
    UP(hh, p->hh, p->mc) UP(Rinv, p->Rinv, (size_t)n * n) UP(Kx, p->Kx, (size_t)n * nx)
    UP(bin_idx, p->bin_idx, p->nb)
    {
        // Msq[r][d] = |mh_r[d:]|^2 for d <= nb: the length of a row once the first d coordinates are eliminated
        const int nb1 = p->nb + 1;
        std::vector<double> sq((size_t)m * nb1);
        for (int r = 0; r < m; ++r) {
            double s = 0.;
            for (int c = n - 1; c >= p->nb; --c) s += p->Mh[(size_t)r * n + c] * p->Mh[(size_t)r * n + c];
            sq[(size_t)r * nb1 + p->nb] = s;
            for (int c = p->nb - 1; c >= 0; --c) { s += p->Mh[(size_t)r * n + c] * p->Mh[(size_t)r * n + c]; sq[(size_t)r * nb1 + c] = s; }
        }
        UP(Msq, sq.data(), sq.size())
    }
    P.n_elim = p->n_elim;
    if (p->n_elim < 0 || p->n_elim > p->nb || (p->n_elim > 0 && !p->Linv)) { wshmpc_destroy(h); WS_FAIL(-1, "n_elim = %d out of range or Linv missing", p->n_elim); }
    {
        std::vector<double> li((size_t)p->nb * p->nb, 0.);
        if (p->Linv) memcpy(li.data(), p->Linv, li.size() * sizeof(double));
        UP(Linv, li.data(), li.size())
        std::vector<double> lt = transpose(li.data(), p->nb, p->nb); UP(LinvT, lt.data(), lt.size())
    }
    {
        std::vector<double> ir(m); for (int r = 0; r < m; ++r) ir[r] = 1. / p->nrm[r]; UP(inr, ir.data(), m)
        std::vector<double> r = transpose(p->Rinv, n, n); UP(RinvT, r.data(), (size_t)n * n)
        std::vector<double> z = transpose(p->Zmap, n, n); UP(ZmapT, z.data(), (size_t)n * n)
        // pricing operator transposed and padded to an even number of outputs: WfT[c * ns2 + r] = Wf[r][c]
        const int ns2 = (p->ns + 1) & ~1;
        std::vector<double> wt((size_t)n * ns2, 0.);
        for (int r2 = 0; r2 < p->ns; ++r2) for (int c = 0; c < n; ++c) wt[(size_t)c * ns2 + r2] = p->Wf[(size_t)r2 * n + c];
        // the two operators every iteration of every lane streams (pricing operator WfT, rows Mh) live in ONE allocation:
        // a single L2 access-policy window keeps them resident while the dual records of the trees stream through L2
        std::vector<double> hot(wt.size() + (size_t)m * n);
        memcpy(hot.data(), wt.data(), wt.size() * sizeof(double));
        memcpy(hot.data() + wt.size(), p->Mh, (size_t)m * n * sizeof(double));
        UP(WfT, hot.data(), hot.size())
        P.Mh = P.WfT + wt.size();
        h->hot_ptr = (void *)P.WfT; h->hot_bytes = hot.size() * sizeof(double);
    }
#undef UP
    // record layout (subproblem_solution.py:86-91, 137-166)
    wshmpc_layout &L = h->layout;
    L.primal = (p->T + 1) * nx + p->T * nu;
    L.off_lam = 0;
    L.off_mu = (p->T + 1) * nx;
    L.off_nu_lb = L.off_mu + p->mc;
    L.off_nu_ub = L.off_nu_lb + p->nb;
    L.off_rho = L.off_nu_ub + p->nb;
    L.off_sigma = L.off_rho + p->T * p->nq + p->nqT;
    L.dual = L.off_sigma + p->T * p->nr;
    L.rec_stride = (L.dual + n + 1) & ~1;          // even: every record of a tree allocation starts 16-byte aligned
    P.n_primal = L.primal; P.n_dual = L.dual; P.n_rec = L.rec_stride; P.off_lam = L.off_lam; P.off_mu = L.off_mu; P.off_nulb = L.off_nu_lb;
    P.off_nuub = L.off_nu_ub; P.off_rho = L.off_rho; P.off_sigma = L.off_sigma;
    // shared memory budget: one CTA per SM holding `lanes` solver lanes; the lanes share the read-only tables, each lane has
    // its vectors and a pool for the leading columns of its factor
    cudaDeviceProp prop;
    WS_CUDA(cudaGetDeviceProperties(&prop, device));
    const size_t optin = prop.sharedMemPerBlockOptin;
    if (n > WS_RPT * WS_NT) { wshmpc_destroy(h); WS_FAIL(-4, "problem too large: n = %d condensed inputs, at most %d supported", n, WS_RPT * WS_NT); }
    if (p->T > 32767 || p->nh > 65535 || p->nh1 > 65535) { wshmpc_destroy(h); WS_FAIL(-4, "problem too large for the packed row map"); }
    P.np = (n + 1) & ~1;
    P.ns2 = (p->ns + 1) & ~1;
    P.ld = 2 * ((P.np >> 1) | 1);                               // >= the ldc of every node
    P.gp = WS_NT / (P.ns2 >> 1);
    P.hot_cap = 2 * n > 200 ? 2 * n : 200;
    {
        SmemOff &so = P.so;
        memset(&so, 0, sizeof(so));
        const int nvl = P.np + 2;
        int part = 2 * WS_NT > P.np + 2 ? 2 * WS_NT : P.np + 2;
        if (part < P.ns2 + 2) part = P.ns2 + 2;                             // partial sums of the pricing operator (one group)
        if (part < 2 * (p->T + 1) * nx) part = 2 * (p->T + 1) * nx;         // scratch of the record epilogue
        int o = 0;
        auto take = [&](int cnt) { const int at = o; o += (cnt + 1) & ~1; return at; };   // keep 16-byte alignment
        // shared tables
        so.t_inr = take(m); so.t_vsc = take(m);
        so.t_sF = take(p->nh * nx); so.t_sG = take(p->nh * nu); so.t_sF1 = take(p->nh1 * nx); so.t_sG1 = take(p->nh1 * nu);
        so.t_rinfo = take((m + 1) / 2);
        so.tab_doubles = o;
        // one lane
        o = 0;
        so.z = take(nvl); so.c1 = take(nvl); so.c2 = take(nvl); so.t = take(nvl); so.u = take(nvl); so.ls = take(nvl);
        so.lam = take(nvl); so.cw = take(nvl); so.yc = take(nvl); so.wv = take(nvl); so.v = take(nvl);
        so.vf0 = take(nvl); so.vf = take(nvl);
        so.bu = take(m); so.blb = take(p->nb); so.xi = take(P.ns2); so.part = take(part);
        so.red = take(112);
        so.ints = o;
        int io = 0;
        so.irow = io; io += n + 1; so.iside = io; io += n + 1; so.ired = io; io += 40; so.iscr = io; io += n + 1;
        so.idep = io; io += 10;
        o += (io + 1) / 2; o = (o + 1) & ~1;
        so.bytes = o;
        so.binW = 0; so.bign = m; so.bnadd = 2 * m;
        o += (3 * m + 7) / 8; o = (o + 1) & ~1;
        const int fixed = o;                                                // doubles of a lane without its pool
        // lanes: as many as leave every lane a pool that holds the factor of a typical deep node (half of the coordinates
        // eliminated, working set of n / 3 rows); at least one
        const size_t avail = optin / 8 - 8;
        const int n_half = P.np / 2, k_typ = n / 3 + 8;
        const size_t pool_want = (size_t)k_typ * (2 * ((n_half >> 1) | 1)) + tri_off(k_typ) + 2;
        const size_t need_shift = shift_smem_doubles(P, WS_NT) + 2;
        int lanes = WS_MAXL;
        const char *env = getenv("WSHMPC_LANES");
        if (env && atoi(env) >= 1 && atoi(env) <= WS_MAXL) lanes = atoi(env);
        else while (lanes > 1 && (size_t)so.tab_doubles + (size_t)lanes * (fixed + (pool_want > need_shift ? pool_want : need_shift)) > avail) --lanes;
        if ((size_t)so.tab_doubles + (size_t)lanes * (fixed + 64) > avail) {
            wshmpc_destroy(h);
            WS_FAIL(-4, "problem too large: %zu bytes of shared memory needed, %zu available", ((size_t)so.tab_doubles + (size_t)lanes * (fixed + 64)) * 8, optin);
        }
        P.lanes = lanes;
        g_lanes_last = lanes;
        h->n_sm = prop.multiProcessorCount;
        // the whole factor of the largest node, and at least the scratch of the fused loop's tree shift (few inputs, many states)
        size_t pool_max = (size_t)n * P.ld + tri_off(n) + 2;
        if (pool_max < need_shift) pool_max = need_shift;
        auto lay = [&](DevProblem &D, int L) {
            size_t pool = (avail - so.tab_doubles) / L - fixed;
            if (pool > pool_max) pool = pool_max;
            pool &= ~(size_t)1;                         // even (pool_max is odd when n = 1, 2 mod 4): lane 1 starts 16-byte aligned
            D.lanes = L;
            D.so.pool = fixed; D.so.pool_sz = (int)pool;
            D.so.lane_doubles = fixed + (int)pool;
            D.so.total_bytes = (D.so.tab_doubles + L * D.so.lane_doubles) * 8;
        };
        lay(P, lanes);
        h->P1 = P;
        lay(h->P1, 1);
        h->smem = (size_t)(P.so.total_bytes > h->P1.so.total_bytes ? P.so.total_bytes : h->P1.so.total_bytes);
    }
    // the limit is an attribute of the kernel, not of the handle: raise it to what the device allows, so that a handle created
    // later for a smaller problem cannot lower it below what this handle launches with
    for (const KernelRow &r : g_kernels) WS_CUDA(raise_smem_limit(r.fn, optin));
    // slot memory
    void *d = nullptr;
    // both cleared: a slot that never stored a state starts from the empty working set AND the centre 0 (hot = 1 on a fresh
    // slot equals hot = 0), whatever an earlier allocation left in the pages
    WS_CUDA(cudaMalloc(&d, (size_t)n_slots * slot_doubles(n, P.ld) * sizeof(double))); h->allocs.push_back(d); h->slot_d = (double *)d;
    WS_CUDA(cudaMemset(h->slot_d, 0, (size_t)n_slots * slot_doubles(n, P.ld) * sizeof(double)));
    WS_CUDA(cudaMalloc(&d, (size_t)n_slots * slot_ints(n) * sizeof(int))); h->allocs.push_back(d); h->slot_i = (int *)d;
    WS_CUDA(cudaMemset(h->slot_i, 0, (size_t)n_slots * slot_ints(n) * sizeof(int)));
    WS_CUDA(cudaMalloc(&d, (size_t)n_slots * m * sizeof(double))); h->allocs.push_back(d); h->ybuf = (double *)d;
    WS_CUDA(cudaMalloc(&d, (size_t)n_slots * bnb_scratch_doubles(p->nb, L.primal) * sizeof(double))); h->allocs.push_back(d); h->scratch = (double *)d;
    WS_CUDA(cudaMalloc(&d, 64)); h->allocs.push_back(d); h->work_counter = (int *)d;
    h->shift_smem = shift_smem_bytes(P, optin, &h->shift_stage);
    WS_CUDA(raise_smem_limit((const void *)shift_tree_kernel, optin));
    {
        // best effort: persisting L2 lines for the shared operators (1.2 MB on the T = 20 cart-pole; the trees are GBs)
        h->l2_window = 0;
        cudaDeviceProp pr;
        if (!getenv("WSHMPC_NO_L2_WINDOW") && cudaGetDeviceProperties(&pr, device) == cudaSuccess && pr.persistingL2CacheMaxSize > 0 && h->hot_bytes > 0) {
            size_t want = h->hot_bytes < (size_t)pr.persistingL2CacheMaxSize ? h->hot_bytes : (size_t)pr.persistingL2CacheMaxSize;
            cudaStreamAttrValue av;
            memset(&av, 0, sizeof(av));
            av.accessPolicyWindow.base_ptr = h->hot_ptr;
            av.accessPolicyWindow.num_bytes = h->hot_bytes < (size_t)pr.accessPolicyMaxWindowSize ? h->hot_bytes : (size_t)pr.accessPolicyMaxWindowSize;
            av.accessPolicyWindow.hitRatio = 1.f;
            av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
            av.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
            if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) == cudaSuccess &&
                cudaStreamSetAttribute(h->stream, cudaStreamAttributeAccessPolicyWindow, &av) == cudaSuccess) h->l2_window = 1;
            cudaGetLastError();                         // a refused window is not an error of the handle
        }
    }
    *out = h;
    return 0;
}

extern "C" int wshmpc_destroy(wshmpc_handle *h)
{
    if (!h) return 0;
    cudaSetDevice(h->device);
    for (void *p : h->allocs) cudaFree(p);
    if (h->plant_stage) cudaFree(h->plant_stage);
    delete h;
    return 0;
}

extern "C" int wshmpc_set_search_rule(wshmpc_handle *h, int rule)
{
    if (!h) WS_FAIL(-1, "null handle");
    if (rule < 0 || rule > 2) WS_FAIL(-1, "search rule %d: 0 best_first, 1 depth_first, 2 breadth_first", rule);
    h->P.search_rule = rule; h->P1.search_rule = rule;
    return 0;
}

extern "C" int wshmpc_set_node_rule(wshmpc_handle *h, int rule)
{
    if (!h) WS_FAIL(-1, "null handle");
    if (rule < 0 || rule > 2) WS_FAIL(-1, "node rule %d: 0 structured, 1 conventional MIQP, 2 conventional MIQP with a MIP start", rule);
    h->P.node_rule = rule; h->P1.node_rule = rule;
    return 0;
}

extern "C" int wshmpc_set_branch_order(wshmpc_handle *h, const int *order)
{
    if (!h) WS_FAIL(-1, "null handle");
    if (!order) { h->P.border = nullptr; h->P1.border = nullptr; return 0; }
    const int nb = h->P.nb;
    std::vector<char> seen(nb, 0);
    for (int p = 0; p < nb; ++p) {
        if (order[p] < 0 || order[p] >= nb || seen[order[p]]) WS_FAIL(-1, "branch order is not a permutation of 0..%d", nb - 1);
        seen[order[p]] = 1;
    }
    WS_CUDA(cudaSetDevice(h->device));
    if (!h->d_border) { void *d = nullptr; WS_CUDA(cudaMalloc(&d, nb * sizeof(int))); h->allocs.push_back(d); h->d_border = (int *)d; }
    WS_CUDA(cudaMemcpy(h->d_border, order, nb * sizeof(int), cudaMemcpyHostToDevice));
    h->P.border = h->d_border; h->P1.border = h->d_border;
    return 0;
}

extern "C" int wshmpc_get_layout(const wshmpc_handle *h, wshmpc_layout *out)
{
    if (!h || !out) WS_FAIL(-1, "null argument");
    *out = h->layout;
    return 0;
}

extern "C" int wshmpc_solve_nodes(wshmpc_handle *h, int n_nodes, const double *d_x0, const double *d_lb,
                                  const double *d_ub, const int *d_slot, const int *d_hot,
                                  const double *d_y0, const double *d_yc0,
                                  int *d_status, double *d_cost, double *d_dobj, int *d_iters,
                                  double *d_primal, double *d_dual, double *d_yc)
{
    if (!h) WS_FAIL(-1, "null handle");
    if (n_nodes <= 0) return 0;
    WS_CUDA(cudaSetDevice(h->device));
    const LaunchShape s = launch_shape(h, h->n_slots);
    void (*k)(WS_K1_ARGS);
    int rc = kernel_for(FAMILY_K1, s.lanes, false, false, false, &k); if (rc) return rc;
    k<<<s.grid, s.block, s.smem, h->stream>>>(*s.P, h->slot_d, h->slot_i, h->ybuf, h->n_slots, n_nodes, d_x0, d_lb, d_ub, d_slot, d_hot,
                                              d_y0, d_yc0, d_status, d_cost, d_dobj, d_iters, d_primal, d_dual, d_yc);
    WS_CUDA(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------
// trees, K3, K2 + K4
// ---------------------------------------------------------------------------------------------
static int tree_view(const wshmpc_handle *h, const wshmpc_tree *t, TreeView *v)
{
    if (!t) WS_FAIL(-1, "null tree");
    if (t->words != (h->P.nb + 31) / 32) WS_FAIL(-1, "tree.words = %d, expected %d", t->words, (h->P.nb + 31) / 32);
    if (t->cap_nodes < 3 || t->cap_recs < 1) WS_FAIL(-1, "tree capacity too small");
    if (!t->n_nodes || !t->n_recs || !t->depth || !t->alive || !t->rec || !t->bits || !t->mask || !t->lb || !t->rec_dobj || !t->rec_dual)
        WS_FAIL(-1, "null pointer in tree");
    v->cap_nodes = t->cap_nodes; v->cap_recs = t->cap_recs; v->words = t->words;
    v->n_nodes = t->n_nodes; v->n_recs = t->n_recs; v->depth = t->depth; v->alive = t->alive; v->rec = t->rec;
    v->bits = t->bits; v->mask = t->mask; v->lb = t->lb; v->rec_dobj = t->rec_dobj; v->rec_dual = t->rec_dual;
    return 0;
}

extern "C" int wshmpc_tree_init_root(wshmpc_handle *h, int n_inst, const wshmpc_tree *tree)
{
    if (!h) WS_FAIL(-1, "null handle");
    if (n_inst <= 0) return 0;
    TreeView tv; int rc = tree_view(h, tree, &tv); if (rc) return rc;
    WS_CUDA(cudaSetDevice(h->device));
    init_root_kernel<<<(n_inst + 127) / 128, 128, 0, h->stream>>>(n_inst, tv);
    WS_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int wshmpc_tree_init_guess(wshmpc_handle *h, int n_inst, const wshmpc_tree *tree, const double *d_guess, const int *d_has)
{
    if (!h) WS_FAIL(-1, "null handle");
    if (n_inst <= 0) return 0;
    if (!d_guess) WS_FAIL(-1, "null guess");
    TreeView tv; int rc = tree_view(h, tree, &tv); if (rc) return rc;
    WS_CUDA(cudaSetDevice(h->device));
    init_guess_kernel<<<(n_inst + 127) / 128, 128, 0, h->stream>>>(n_inst, h->P.nb, tv, d_guess, d_has);
    WS_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int wshmpc_bnb_solve(wshmpc_handle *h, int n_inst, const double *d_x0, const int *d_active,
                                const wshmpc_tree *tree, double tol, int max_solves,
                                double *d_inc_cost, int *d_inc_node, double *d_inc_primal, int *d_n_solves,
                                int *d_status, int *d_trace, unsigned long long *d_totals)
{
    if (!h) WS_FAIL(-1, "null handle");
    if (n_inst <= 0) return 0;
    if (max_solves <= 0) WS_FAIL(-1, "max_solves must be positive");
    if (!d_x0 || !d_inc_cost || !d_inc_node || !d_inc_primal || !d_n_solves || !d_status) WS_FAIL(-1, "null argument");
    TreeView tv; int rc = tree_view(h, tree, &tv); if (rc) return rc;
    WS_CUDA(cudaSetDevice(h->device));
    WS_CUDA(cudaMemsetAsync(h->work_counter, 0, sizeof(int), h->stream));
    const int slots = n_inst < h->n_slots ? n_inst : h->n_slots;
    const LaunchShape s = launch_shape(h, slots);
    // the node rule picks the kernel: the structured search's kernels carry no code of the conventional rule
    void (*k)(WS_BNB_ARGS);
    rc = kernel_for(FAMILY_BNB, s.lanes, h->P.node_rule != 0, false, false, &k); if (rc) return rc;
    k<<<s.grid, s.block, s.smem, h->stream>>>(*s.P, h->slot_d, h->slot_i, h->ybuf, h->scratch, h->work_counter, slots, n_inst, d_x0,
                                              d_active, tv, tol, max_solves, d_inc_cost, d_inc_node, d_inc_primal, d_n_solves,
                                              d_status, d_trace, d_totals);
    WS_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int wshmpc_shift_tree(wshmpc_handle *h, int n_inst, const double *d_x0, const double *d_e0,
                                 const wshmpc_tree *old_tree, const double *d_inc_cost, const double *d_inc_primal,
                                 int *d_active, const wshmpc_tree *new_tree, double *d_x_next, double *d_u0)
{
    if (!h) WS_FAIL(-1, "null handle");
    if (n_inst <= 0) return 0;
    if (!d_x0 || !d_inc_cost || !d_inc_primal) WS_FAIL(-1, "null argument");
    if (h->P.T < 2) WS_FAIL(-1, "tree shifting needs T >= 2");
    if (h->P.nub > 32) WS_FAIL(-1, "tree shifting supports nub <= 32");
    TreeView ov, nv; int rc = tree_view(h, old_tree, &ov); if (rc) return rc;
    rc = tree_view(h, new_tree, &nv); if (rc) return rc;
    if (ov.rec_dual == nv.rec_dual || ov.lb == nv.lb) WS_FAIL(-1, "old and new tree must be distinct buffers");
    if (ov.words != nv.words) WS_FAIL(-1, "old and new tree differ in words");
    WS_CUDA(cudaSetDevice(h->device));
    shift_tree_kernel<<<n_inst, SH_NT, h->shift_smem, h->stream>>>(
        h->P, n_inst, d_x0, d_e0, ov, d_inc_cost, d_inc_primal, d_active, nv, d_x_next, d_u0, h->shift_stage);
    WS_CUDA(cudaGetLastError());
    return 0;
}

// a wshmpc_plant checked against the handle's problem; n = the states it is applied to
static int plant_view(const wshmpc_handle *h, const wshmpc_plant *pl, int n, PlantView *v)
{
    if (!pl) WS_FAIL(-1, "null plant");
    if (pl->kind != 1) WS_FAIL(-1, "plant kind %d: 1 is the cart-pole between two soft walls, the only kind", pl->kind);
    if (h->P.nx != 4) WS_FAIL(-1, "the cart-pole plant has 4 states, the problem has nx = %d", h->P.nx);
    if (pl->fc_index < 0 || pl->fc_index >= h->P.nu) WS_FAIL(-1, "plant fc_index = %d out of range (nu = %d)", pl->fc_index, h->P.nu);
    if (!(pl->dt > 0.) || pl->n_sub <= 0) WS_FAIL(-1, "plant needs dt > 0 and n_sub > 0 (dt = %g, n_sub = %d)", pl->dt, pl->n_sub);
    if (pl->n_sets != 1 && pl->n_sets != n) WS_FAIL(-1, "plant n_sets = %d: 1 or one per instance (%d)", pl->n_sets, n);
    if (!pl->d_params) WS_FAIL(-1, "null plant parameters");
    v->prm = pl->d_params; v->n_sets = pl->n_sets; v->n_sub = pl->n_sub; v->h = pl->dt / pl->n_sub; v->fc_index = pl->fc_index;
    v->log_x = pl->d_log_x; v->stage = nullptr;
    return 0;
}

extern "C" int wshmpc_plant_step(wshmpc_handle *h, const wshmpc_plant *pl, int n, const double *d_x, const double *d_u, double *d_x_out)
{
    if (!h) WS_FAIL(-1, "null handle");
    if (n <= 0) return 0;
    if (!d_x || !d_u || !d_x_out) WS_FAIL(-1, "null argument");
    PlantView v; int rc = plant_view(h, pl, n, &v); if (rc) return rc;
    WS_CUDA(cudaSetDevice(h->device));
    plant_step_kernel<<<(n + 127) / 128, 128, 0, h->stream>>>(v, n, h->P.nu, d_x, d_u, d_x_out);
    WS_CUDA(cudaGetLastError());
    return 0;
}

// a wshmpc_fallback checked against the handle's problem; n = the instances it serves
static int fallback_view(const wshmpc_handle *h, const wshmpc_fallback *fb, int n, FallbackView *v)
{
    if (!fb) WS_FAIL(-1, "null fallback");
    if (h->P.node_rule != 0) WS_FAIL(-1, "node rule %d: the fallback policy runs under the structured search (node rule 0) only", h->P.node_rule);
    if (fb->max_hold < 0 || fb->max_hold > h->P.T - 1) WS_FAIL(-1, "fallback max_hold = %d out of range 0 .. T - 1 = %d", fb->max_hold, h->P.T - 1);
    if (!fb->d_plan || !fb->d_age || !fb->d_app_cost || !fb->d_app_primal || !fb->d_hold) WS_FAIL(-1, "null fallback buffer");
    const size_t bytes = (size_t)n * h->P.n_primal * sizeof(double);
    const char *p = (const char *)fb->d_plan, *a = (const char *)fb->d_app_primal;
    if (p < a + bytes && a < p + bytes) WS_FAIL(-1, "fallback d_plan and d_app_primal overlap");
    if (fb->max_law < 0) WS_FAIL(-1, "fallback max_law = %d: the law steps an instance may take, >= 0", fb->max_law);
    if (fb->max_law > 0 && (!fb->d_law_K || !fb->d_law_n)) WS_FAIL(-1, "fallback max_law = %d with a null d_law_K or d_law_n", fb->max_law);
    if (fb->max_law == 0 && (fb->law_sets != 0 || fb->d_law_k || fb->d_law_lo || fb->d_law_hi))
        WS_FAIL(-1, "fallback law_sets, d_law_k, d_law_lo or d_law_hi set with max_law = 0");
    if (fb->law_sets != 0 && fb->law_sets != 1 && fb->law_sets != n)
        WS_FAIL(-1, "fallback law_sets = %d: 0 or 1 (one set) or one per instance (%d)", fb->law_sets, n);
    if (!fb->d_law_lo != !fb->d_law_hi) WS_FAIL(-1, "fallback d_law_lo and d_law_hi: both or neither");
    v->max_hold = fb->max_hold; v->plan = fb->d_plan; v->age = fb->d_age; v->app_cost = fb->d_app_cost;
    v->app_primal = fb->d_app_primal; v->hold = fb->d_hold;
    v->max_law = fb->max_law; v->law_K = fb->max_law > 0 ? fb->d_law_K : nullptr; v->law_n = fb->max_law > 0 ? fb->d_law_n : nullptr;
    v->law_sets = fb->law_sets; v->law_k = fb->d_law_k; v->law_lo = fb->d_law_lo; v->law_hi = fb->d_law_hi;
    return 0;
}

extern "C" int wshmpc_fallback_step(wshmpc_handle *h, int n_inst, const wshmpc_fallback *fb, const double *d_x, const int *d_active,
                                    const int *d_status, const double *d_inc_cost, const double *d_inc_primal)
{
    if (!h) WS_FAIL(-1, "null handle");
    if (n_inst <= 0) return 0;
    if (!d_x || !d_status || !d_inc_cost || !d_inc_primal) WS_FAIL(-1, "null argument");
    FallbackView v; int rc = fallback_view(h, fb, n_inst, &v); if (rc) return rc;
    WS_CUDA(cudaSetDevice(h->device));
    fallback_step_kernel<<<(n_inst + 127) / 128, 128, 0, h->stream>>>(h->P, n_inst, v, d_x, d_active, d_status, d_inc_cost, d_inc_primal);
    WS_CUDA(cudaGetLastError());
    return 0;
}

// wshmpc_closed_loop (plant = null: x <- x_1|t + e_t), wshmpc_closed_loop_plant and wshmpc_closed_loop_fallback (fb != null)
static int closed_loop_launch(wshmpc_handle *h, int n_inst, const wshmpc_loop *loop, const wshmpc_plant *plant,
                              const wshmpc_fallback *fb,
                              const wshmpc_tree *tree0, const wshmpc_tree *tree1, double tol, int max_solves,
                              double *d_inc_cost, int *d_inc_node, double *d_inc_primal, int *d_n_solves,
                              int *d_status, unsigned long long *d_totals)
{
    if (!h || !loop) WS_FAIL(-1, "null argument");
    if (n_inst <= 0 || loop->n_steps <= 0) return 0;
    if (max_solves <= 0) WS_FAIL(-1, "max_solves must be positive");
    if (!loop->d_queue || !loop->d_step_of || !loop->d_x || !loop->d_active || !loop->d_log_cost || !loop->d_log_u0 ||
        !loop->d_log_solves || !loop->d_log_status || !d_inc_cost || !d_inc_node || !d_inc_primal || !d_n_solves || !d_status)
        WS_FAIL(-1, "null argument");
    if (h->P.T < 2) WS_FAIL(-1, "tree shifting needs T >= 2");
    if (h->P.nub > 32) WS_FAIL(-1, "tree shifting supports nub <= 32");
    if (loop->warm && h->P.node_rule != 0) WS_FAIL(-1, "node rule %d: the conventional MIQP search runs cold trees only (warm = 0)", h->P.node_rule);
    if ((size_t)h->P.so.pool_sz < shift_smem_doubles(h->P, WS_NT)) WS_FAIL(-4, "shared memory too small for the fused warm start");
    if ((long long)n_inst * (loop->n_steps + 1) > 0x7fffffffLL) WS_FAIL(-1, "too many tasks");
    TreeView v0, v1; int rc = tree_view(h, tree0, &v0); if (rc) return rc;
    rc = tree_view(h, tree1, &v1); if (rc) return rc;
    if (v0.rec_dual == v1.rec_dual || v0.lb == v1.lb) WS_FAIL(-1, "the two trees must be distinct buffers");
    PlantView pv;
    memset(&pv, 0, sizeof(pv));
    if (plant) {
        if (loop->mailbox) WS_FAIL(-1, "a plant and a mailbox: with a mailbox the host is the plant");
        rc = plant_view(h, plant, n_inst, &pv); if (rc) return rc;
        WS_CUDA(cudaSetDevice(h->device));
        if (h->plant_stage_n < n_inst) {
            if (h->plant_stage) { WS_CUDA(cudaFree(h->plant_stage)); h->plant_stage = nullptr; h->plant_stage_n = 0; }
            WS_CUDA(cudaMalloc((void **)&h->plant_stage, (size_t)n_inst * 4 * sizeof(double)));
            h->plant_stage_n = n_inst;
        }
        pv.stage = h->plant_stage;
    }
    FallbackView fv;
    memset(&fv, 0, sizeof(fv));
    if (fb) {
        if (loop->mailbox) WS_FAIL(-1, "a fallback and a mailbox: the mailbox loop has no fallback policy");
        rc = fallback_view(h, fb, n_inst, &fv); if (rc) return rc;
    }
    LoopView L;
    L.n_steps = loop->n_steps; L.warm = loop->warm; L.fresh = loop->fresh; L.par = loop->par & 1;
    L.q = loop->d_queue; L.step_of = loop->d_step_of; L.x = loop->d_x; L.e = loop->d_e; L.active = loop->d_active;
    L.log_cost = loop->d_log_cost; L.log_u0 = loop->d_log_u0; L.log_solves = loop->d_log_solves; L.log_status = loop->d_log_status;
    L.log_cover = loop->d_log_cover; L.log_lapsed = loop->d_log_lapsed; L.log_iters = loop->d_log_iters;
    WS_CUDA(cudaSetDevice(h->device));
    L.mb_in_step = L.mb_out_step = L.mb_stop = nullptr; L.mb_in_x = L.mb_in_e = nullptr;
    L.mb_out_u0 = L.mb_out_x1 = L.mb_out_cost = nullptr; L.mb_out_status = nullptr; L.mb_stage = nullptr; L.mb_timeout_ns = 0;
    if (loop->mailbox) {
        const wshmpc_mailbox *mb = loop->mailbox;
        if (mb->n_inst < n_inst || mb->nx != h->P.nx || mb->nu != h->P.nu || !mb->priv) WS_FAIL(-1, "mailbox does not match the problem / batch");
        void *dp;
#define MB_DEV(dst, type, src) WS_CUDA(cudaHostGetDevicePointer(&dp, (void *)(src), 0)); dst = (type)dp
        MB_DEV(L.mb_in_step, volatile int *, mb->in_step); MB_DEV(L.mb_out_step, volatile int *, mb->out_step);
        MB_DEV(L.mb_stop, volatile int *, mb->stop);
        MB_DEV(L.mb_in_x, const volatile double *, mb->in_x); MB_DEV(L.mb_in_e, const volatile double *, mb->in_e);
        MB_DEV(L.mb_out_u0, double *, mb->out_u0); MB_DEV(L.mb_out_x1, double *, mb->out_x1); MB_DEV(L.mb_out_cost, double *, mb->out_cost);
        MB_DEV(L.mb_out_status, int *, mb->out_status);
#undef MB_DEV
        L.mb_stage = (double *)mb->priv;
        L.mb_timeout_ns = (unsigned long long)(mb->timeout_ms > 0 ? mb->timeout_ms : 5000) * 1000000ull;
    }
    const int slots = n_inst < h->n_slots ? n_inst : h->n_slots;
    const LaunchShape s = launch_shape(h, slots);
    void (*k)(WS_LOOP_ARGS);
    rc = kernel_for(FAMILY_LOOP, s.lanes, h->P.node_rule != 0, plant != nullptr, fb != nullptr, &k); if (rc) return rc;
    const int n_items = n_inst * (loop->n_steps + 1);
    loop_init_kernel<<<(n_items + 255) / 256, 256, 0, h->stream>>>(n_inst, n_items, L);
    WS_CUDA(cudaGetLastError());
    k<<<s.grid, s.block, s.smem, h->stream>>>(*s.P, h->slot_d, h->slot_i, h->ybuf, h->scratch, L, slots, n_inst, v0, v1, tol, max_solves,
                                              d_inc_cost, d_inc_node, d_inc_primal, d_n_solves, d_status, d_totals, pv, fv);
    WS_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int wshmpc_closed_loop(wshmpc_handle *h, int n_inst, const wshmpc_loop *loop,
                                  const wshmpc_tree *tree0, const wshmpc_tree *tree1, double tol, int max_solves,
                                  double *d_inc_cost, int *d_inc_node, double *d_inc_primal, int *d_n_solves,
                                  int *d_status, unsigned long long *d_totals)
{
    return closed_loop_launch(h, n_inst, loop, nullptr, nullptr, tree0, tree1, tol, max_solves, d_inc_cost, d_inc_node, d_inc_primal,
                              d_n_solves, d_status, d_totals);
}

extern "C" int wshmpc_closed_loop_plant(wshmpc_handle *h, int n_inst, const wshmpc_loop *loop, const wshmpc_plant *plant,
                                        const wshmpc_tree *tree0, const wshmpc_tree *tree1, double tol, int max_solves,
                                        double *d_inc_cost, int *d_inc_node, double *d_inc_primal, int *d_n_solves,
                                        int *d_status, unsigned long long *d_totals)
{
    if (!plant) WS_FAIL(-1, "null plant");
    return closed_loop_launch(h, n_inst, loop, plant, nullptr, tree0, tree1, tol, max_solves, d_inc_cost, d_inc_node, d_inc_primal,
                              d_n_solves, d_status, d_totals);
}

extern "C" int wshmpc_closed_loop_fallback(wshmpc_handle *h, int n_inst, const wshmpc_loop *loop, const wshmpc_plant *plant,
                                           const wshmpc_fallback *fb, const wshmpc_tree *tree0, const wshmpc_tree *tree1, double tol,
                                           int max_solves, double *d_inc_cost, int *d_inc_node, double *d_inc_primal, int *d_n_solves,
                                           int *d_status, unsigned long long *d_totals)
{
    if (!fb) WS_FAIL(-1, "null fallback");
    return closed_loop_launch(h, n_inst, loop, plant, fb, tree0, tree1, tol, max_solves, d_inc_cost, d_inc_node, d_inc_primal,
                              d_n_solves, d_status, d_totals);
}

// host mailbox: pinned, mapped host memory the running kernel and the host both see
extern "C" int wshmpc_mailbox_create(wshmpc_handle *h, int n_inst, wshmpc_mailbox *mb)
{
    if (!h || !mb || n_inst <= 0) WS_FAIL(-1, "null argument");
    memset(mb, 0, sizeof(*mb));
    WS_CUDA(cudaSetDevice(h->device));
    const int nx = h->P.nx, nu = h->P.nu;
    const size_t n_d = (size_t)n_inst * (nu + nx + 1 + nx + nx), n_i = (size_t)n_inst * 3 + 16;
    double *hd = nullptr; int *hi = nullptr; double *stage = nullptr;
    WS_CUDA(cudaHostAlloc((void **)&hd, n_d * sizeof(double), cudaHostAllocMapped | cudaHostAllocPortable));
    if (cudaHostAlloc((void **)&hi, n_i * sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) { cudaFreeHost(hd); WS_FAIL(-2, "cudaHostAlloc failed"); }
    if (cudaMalloc((void **)&stage, (size_t)n_inst * nx * sizeof(double)) != cudaSuccess) { cudaFreeHost(hd); cudaFreeHost(hi); WS_FAIL(-2, "cudaMalloc failed"); }
    memset(hd, 0, n_d * sizeof(double)); memset(hi, 0, n_i * sizeof(int));
    mb->n_inst = n_inst; mb->nx = nx; mb->nu = nu;
    mb->out_u0 = hd; hd += (size_t)n_inst * nu;
    mb->out_x1 = hd; hd += (size_t)n_inst * nx;
    mb->out_cost = hd; hd += n_inst;
    mb->in_x = hd; hd += (size_t)n_inst * nx;
    mb->in_e = hd;
    mb->out_step = hi; mb->in_step = hi + n_inst; mb->out_status = hi + 2 * (size_t)n_inst; mb->stop = hi + 3 * (size_t)n_inst;
    mb->priv = stage;
    return 0;
}

extern "C" int wshmpc_mailbox_destroy(wshmpc_handle *h, wshmpc_mailbox *mb)
{
    if (!mb) return 0;
    if (h) cudaSetDevice(h->device);
    if (mb->out_u0) cudaFreeHost(mb->out_u0);
    if (mb->out_step) cudaFreeHost((void *)mb->out_step);
    if (mb->priv) cudaFree(mb->priv);
    memset(mb, 0, sizeof(*mb));
    return 0;
}

// ---------------------------------------------------------------------------------------------
// batched small LPs (SURVEY.md 8f-2; controller.py:186-227 _update_mu, mcais.py:44-184)
// ---------------------------------------------------------------------------------------------
extern "C" int wshmpc_lp_batch(int device, void *stream, int n_lp, int m, int n, const double *d_E, long long stride_E,
                               const double *d_c, long long stride_c, const double *d_r, double tol, int max_iter,
                               int *d_status, double *d_obj, double *d_y, double *d_dual, int *d_iters)
{
    if (n_lp <= 0) return 0;
    if (m <= 0 || n <= 0 || m > LP_MAX_M) WS_FAIL(-1, "wshmpc_lp_batch: need 0 < m <= %d equality rows and n > 0 columns (m = %d, n = %d)", LP_MAX_M, m, n);
    if (!d_E || !d_c || !d_r || !d_status || !d_obj || !d_y || !d_dual || !d_iters) WS_FAIL(-1, "null argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) WS_FAIL(-3, "no CUDA device");
    WS_CUDA(cudaSetDevice(device));
    const size_t smem = sizeof(double) * (size_t)(m + 1) * (n + m + 1);
    cudaDeviceProp prop;
    WS_CUDA(cudaGetDeviceProperties(&prop, device));
    if (smem > prop.sharedMemPerBlockOptin) WS_FAIL(-4, "wshmpc_lp_batch: tableau of %zu bytes does not fit shared memory", smem);
    if (smem > 48 * 1024) WS_CUDA(cudaFuncSetAttribute(lp_std_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    lp_std_kernel<<<n_lp, LP_NT, smem, (cudaStream_t)stream>>>(n_lp, m, n, d_E, stride_E, d_c, stride_c, d_r, tol, max_iter,
                                                              d_status, d_obj, d_y, d_dual, d_iters);
    WS_CUDA(cudaGetLastError());
    return 0;
}
#endif  // WS_TU_HAS(0)
