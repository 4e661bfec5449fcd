/* wshmpc.h -- C ABI of the B200-native hybrid-MPC branch-and-bound hot path.
 *
 * Drop-in boundary for the per-node / per-solve seams of TobiaMarcucci/warm-start-hybrid-mpc
 * (SURVEY.md section 8b).  The reference has no FFI layer: its seams are Python callables, so every
 * entry point below cites the reference callable it replaces.  All matrices are fp64, row-major,
 * caller-owned; "d_" arguments are DEVICE pointers (torch CUDA tensors' data_ptr()), everything else
 * is host memory.  Every call returns 0 on success, < 0 on error (message in wshmpc_last_error).
 * One handle per (GPU, stream); not thread-safe; never throws; never falls back to the CPU.
 */
#ifndef WSHMPC_H
#define WSHMPC_H
#ifdef __cplusplus
extern "C" {
#endif

typedef struct wshmpc_handle wshmpc_handle;

/* Problem description: the MLD system + controller data of
 * HybridModelPredictiveController.__init__ (controller.py:58-97) and the shared least-distance
 * operator the QP kernel runs on (host-side precompute, north_star "condensing stays host-side";
 * built by warm-start-hybrid-mpc_b200/problem.py). */
typedef struct {
    /* sizes */
    int nx, nu, nub, T;          /* mld_system.py:37-41, controller.py:78 */
    int nh, nh1;                 /* rows of F (stage) and of F_Tm1 (last stage, controller.py:85-87) */
    int nq, nqT, nr;             /* rows of Q, Q_T, R (controller.py:79) */
    int n, m, mc, nb;            /* n = T*nu condensed inputs, m = mc + nb rows, nb = T*nub */
    int ns;                      /* n + T*nx : inputs and states of the sparse form */
    /* stage data (host pointers, row-major) */
    const double *A, *B, *F, *G, *h, *F_Tm1, *G_Tm1, *h_Tm1, *Q, *R, *Q_T;
    const double *M_mu;          /* nh x nh1, controller.py:186-227 */
    const double *M_rho;         /* nq x nqT, controller.py:96 */
    /* shared least-distance operator (host pointers) */
    const double *Mh;            /* m x n, unit rows */
    const double *Wf;            /* ns x n : N Rinv, maps v to (inputs, states) for factored row pricing */
    const double *nrm;           /* m */
    const double *vscale;        /* m */
    const double *Eh;            /* mc x nx */
    const double *hh;            /* mc */
    const double *Rinv;          /* n x n */
    const double *Kx;            /* n x nx */
    const double *Zmap;          /* n x n */
    const int *bin_idx;          /* nb */
    const double *Linv;          /* nb x nb, lower triangular: inverse of the leading block of the binaries' bound rows
                                    Mh[mc + j][0..j] (problem.py rotates v so that these rows are lower triangular) */
    int n_elim;                  /* leading binaries (chronological order) that may be eliminated when pinned; 0 = off */
    /* solver parameters */
    double eps, tol_p, tol_d, tol_sing, tol_ray, prox_tol;
    int max_iter, max_prox;
} wshmpc_problem;

/* sizes of the per-node records, in doubles */
typedef struct {
    int primal;                  /* (T+1)*nx + T*nu : x_0..x_T, u_0..u_{T-1}  (subproblem_solution.py:86-91) */
    int dual;                    /* lam | mu | nu_lb | nu_ub | rho | sigma     (subproblem_solution.py:137-166) */
    int off_lam, off_mu, off_nu_lb, off_nu_ub, off_rho, off_sigma;
    int rec_stride;              /* doubles per dual record INSIDE a wshmpc_tree: dual + n.  The n extra doubles hold the
                                    proximal centre (orthonormal coordinates) of the solve the record came from, i.e. the
                                    `active_set` payload the reference hands from a parent to its children
                                    (subproblem_solution.py:10, controller.py:426) */
} wshmpc_layout;

const char *wshmpc_last_error(void);

/* solver lanes (independent solver states) resident per SM for the handle created last: n_slots = SMs x this fills the GPU */
int wshmpc_ctas_per_sm(void);

/* create / destroy.  `n_slots` = number of independent solver states (one per concurrently solved
 * MPC instance); `stream` is a cudaStream_t passed as void* (0 = default stream). */
int wshmpc_create(const wshmpc_problem *p, int device, int n_slots, void *stream, wshmpc_handle **out);
int wshmpc_destroy(wshmpc_handle *h);
int wshmpc_get_layout(const wshmpc_handle *h, wshmpc_layout *out);

/* candidate selection of the device-side branch and bound (wshmpc_bnb_solve, wshmpc_closed_loop), the
 * `candidate_selection` argument of branch_and_bound (branch_and_bound.py:408-416):
 * 0 best_first (:541-563, default), 1 depth_first (:521-538), 2 breadth_first (:501-518).  Sticky per handle. */
int wshmpc_set_search_rule(wshmpc_handle *h, int rule);

/* branching order of the device-side branch and bound, the `branch_rule` argument of feedforward (controller.py:329,
 * 395-429) restricted to rules that pick the next binary from a FIXED priority order: `order` (host, nb ints) is a
 * permutation of the binaries j = t*nub+i; a node is branched on the first binary of the order its identifier does not
 * assign, children [value 0, value 1].  NULL = chronological order = branch_in_time (controller.py:13-44, default).
 * Identifiers are (assigned mask, values) pairs, so any order -- and any warm start a host-side rule produced -- is
 * representable; only the leading run of assigned binaries is eliminated from the node's QP.  Sticky per handle. */
int wshmpc_set_branch_order(wshmpc_handle *h, const int *order);

/* node rule of the device-side branch and bound (wshmpc_bnb_solve, wshmpc_closed_loop).  Sticky per handle.
 *   0  the structured search (default): branch on the first unassigned binary of the branching order, a node is an incumbent
 *      iff every binary is pinned, a child's bound = parent cost + the multiplier of the bound that moves (controller.py:395-429).
 *   1  the conventional MIQP branch and bound of feedforward_miqp (controller.py:530-582), the paper's "Gurobi fair" comparator
 *      (feedforward_gurobi, controller.py:723-776) without Gurobi: after a node's solve, branch on the unassigned binary
 *      j = t*nub+i whose relaxed value u is the most fractional (|u - rint(u)| largest, ties to the smaller j; the branching
 *      order is ignored); the node is an incumbent when that fractionality is <= 1e-9; children [value 0, value 1] both get
 *      bound = the parent's relaxation cost and start from the parent's record.  Candidate selection (wshmpc_set_search_rule)
 *      is unchanged.  A MIP start is a tree from wshmpc_tree_init_guess.
 *   2  rule 1, and in wshmpc_closed_loop a MIP start at every step of an instance whose previous step left an incumbent: the
 *      previous incumbent's binaries shifted by one step, zero at the end (shift_binary_solution, controller.py:586-588); no
 *      guess on step 0 of a `fresh` launch.
 * Rules 1 and 2 run cold trees only: wshmpc_closed_loop with warm = 1 fails under them. */
int wshmpc_set_node_rule(wshmpc_handle *h, int rule);

/* K1 -- batched node QP relaxation.
 * Replaces, per node: controller._solve_subproblem (controller.py:229-271) = _set_bound_binaries
 * (:273-298) + BoundedQP.optimize (bounded_qp.py:200-228) + SubproblemSolution.from_controller
 * (subproblem_solution.py:18-45).
 *   d_x0   [n_nodes][nx]     initial state of each node's problem          (rhs of 'lam_0')
 *   d_lb   [n_nodes][nb]     lower bounds on the relaxed binaries, (t,i) -> t*nub+i   (-rhs of 'nu_lb_t')
 *   d_ub   [n_nodes][nb]     upper bounds                                  (rhs of 'nu_ub_t')
 *   d_slot [n_nodes]         solver state used by the node; nodes sharing a slot are solved in index
 *                            order by one CTA
 *   d_hot  [n_nodes]         start of the dual active-set method (any multipliers >= 0 are dual feasible for every node):
 *                            0: empty working set; 1: the working set the slot's previous node ended with;
 *                            2: the multipliers d_y0 / proximal centre d_yc0 of this node -- what the reference hands
 *                               from a parent to its children as `active_set` (controller.py:262-264, 426)
 *   d_y0   [n_nodes][m]      (hot = 2; may be NULL otherwise) signed multipliers of the rows mu_0..mu_{T-1} | binaries:
 *                            m = layout.off_nu_lb - layout.off_mu + nb; > 0 upper side (mu, nu_ub), < 0 lower (nu_lb).
 *                            Only finite entries that are > 0 on a row mu or != 0 on a binary enter the start; every
 *                            other entry (negative on a row mu, which has no lower side, NaN, +-inf) is ignored, i.e.
 *                            projected to zero, so the start stays dual feasible
 *   d_yc0  [n_nodes][n]      (hot = 2; may be NULL = 0) proximal centre, n = T * nu
 * outputs
 *   d_status [n_nodes]       2 optimal, 3 infeasible (Gurobi status codes, bounded_qp.py:212), 9 iteration limit (also: the
 *                            proximal outer loop did not converge in max_prox passes, or the working set hit its capacity)
 *   d_cost   [n_nodes]       primal objective, +inf if infeasible          (bounded_qp.py:292-311)
 *   d_dobj   [n_nodes]       dual objective / cost of the Farkas proof     (bounded_qp.py:313-332)
 *   d_iters  [n_nodes]       active-set iterations
 *   d_primal [n_nodes][layout.primal]   (undefined if infeasible)
 *   d_dual   [n_nodes][layout.dual]
 *   d_yc     [n_nodes][n] or NULL       proximal centre the solve ended at (0 if infeasible): d_yc0 of the children
 */
int wshmpc_solve_nodes(wshmpc_handle *h, int n_nodes, const double *d_x0, const double *d_lb,
                       const double *d_ub, const int *d_slot, const int *d_hot,
                       const double *d_y0, const double *d_yc0,
                       int *d_status, double *d_cost, double *d_dobj, int *d_iters,
                       double *d_primal, double *d_dual, double *d_yc);

/* ---------------------------------------------------------------------------------------------
 * Branch-and-bound trees of a batch of independent MPC instances (device memory, caller-owned:
 * torch tensors).  Replaces the Python `leaves` list of branch_and_bound.py:432 and the Node objects
 * (branch_and_bound.py:7-55): instance k owns nodes [k][0 .. n_nodes[k]) in CREATION order, which is
 * the order of the reference's list (children are appended, branch_and_bound.py:488-489; a branched
 * node is removed = alive 0).  With the reference's default `branch_in_time` rule (controller.py:13-44)
 * every identifier is a prefix of the chronological order (0,0),(0,1),...,(T-1,nub-1), so a node is
 * (depth, value bits); time shifting keeps it a prefix (controller.py:476).
 * Dual records follow the layout struct above (stride rec_stride); children alias the parent's record (controller.py:426)
 * and start their QP from its multipliers.
 */
typedef struct {
    int cap_nodes, cap_recs, words;   /* words = ceil(T*nub / 32) uint32 per identifier */
    int *n_nodes;                     /* [n_inst] */
    int *n_recs;                      /* [n_inst] */
    int *depth;                       /* [n_inst][cap_nodes]  number of pinned binaries (= popcount of the node's mask) */
    int *alive;                       /* [n_inst][cap_nodes]  1 = leaf, 0 = branched (removed from `leaves`) */
    int *rec;                         /* [n_inst][cap_nodes]  dual record of the node, < 0 = None (-2 - r: None, but record r
                                         holds the shifted ray of a leaf whose proof lapsed: used to start its QP) */
    unsigned int *bits;               /* [n_inst][cap_nodes][words]  bit j = value of binary j = t*nub+i if it is assigned */
    unsigned int *mask;               /* [n_inst][cap_nodes][words]  bit j = 1 iff binary j is assigned by the node's identifier (the low `depth` bits
                                         for branch_in_time trees; any set for other branching orders / user-built warm starts) */
    double *lb;                       /* [n_inst][cap_nodes]  Node.lb */
    double *rec_dobj;                 /* [n_inst][cap_recs]   DualSolution.objective */
    double *rec_dual;                 /* [n_inst][cap_recs][layout.rec_stride]  DualSolution.variables | proximal centre */
} wshmpc_tree;

/* K3 -- device-side branch and bound, one solver lane (256 threads; up to two lanes per CTA / SM) per instance at a time, no
 * host round trip per node.
 * Replaces branch_and_bound(solver, best_first, brancher, tol, warm_start) (branch_and_bound.py:408-499)
 * with the controller's closures (controller.py:365-380): select = best_first (first minimum wins,
 * branch_and_bound.py:541-563), solve = K1 (hot-started from the node solved before it), prune /
 * incumbent / branch with child bounds from the parent's multipliers (controller.py:395-429).
 * `tree` holds the initial leaves on entry (root node or warm start) and the final leaves on exit.
 *   d_active    [n_inst] or NULL  instances with 0 are skipped
 *   d_inc_cost  [n_inst]          optimal cost, +inf if the MIQP is infeasible
 *   d_inc_node  [n_inst]          node index of the incumbent, -1 if none
 *   d_inc_primal[n_inst][layout.primal]
 *   d_n_solves  [n_inst]          number of QP relaxations solved
 *   d_status    [n_inst]          0 optimal, 1 infeasible MIQP, 2 capacity reached, 3 QP iteration limit
 *   d_trace     [n_inst][2*max_solves] or NULL : (node index, active-set iterations) of every solve, in order
 *   d_totals    [8] or NULL : running 64-bit counters: [0] += QP relaxations solved, [1] += active-set iterations,
 *                             [2] += working-set size at the end of every solve, [3] max= largest working set seen,
 *                             [4] += eliminated (pinned-prefix) coordinates of every solve, [5] += rows of the inherited
 *                             working set re-factorised at the start of every solve, [6..7] reserved
 */
int wshmpc_bnb_solve(wshmpc_handle *h, int n_inst, const double *d_x0, const int *d_active,
                     const wshmpc_tree *tree, double tol, int max_solves,
                     double *d_inc_cost, int *d_inc_node, double *d_inc_primal, int *d_n_solves,
                     int *d_status, int *d_trace, unsigned long long *d_totals);

/* cold start: every instance gets the single root node Node({}) with lb = -inf (branch_and_bound.py:432) */
int wshmpc_tree_init_root(wshmpc_handle *h, int n_inst, const wshmpc_tree *tree);

/* MIP start (the ub_guess of feedforward_miqp, controller.py:552-556): instance k gets node 0 = the guess (every binary pinned,
 * lb = -inf, no record: solved first under best_first, from the empty working set) and node 1 = the root, or the root alone
 * where d_has[k] == 0.  The guess's solve counts in n_solves; after it the node is never a candidate again (its lb is the
 * incumbent's cost or +inf).
 *   d_guess [n_inst][nb] binary values j = t*nub+i, rounded with rint (to 0 or 1)
 *   d_has   [n_inst] or NULL (every instance has a guess) */
int wshmpc_tree_init_guess(wshmpc_handle *h, int n_inst, const wshmpc_tree *tree, const double *d_guess, const int *d_has);

/* K2 + K4 -- warm start for the next time step, one CTA per instance, one warp per leaf.
 * Replaces construct_warm_start (controller.py:431-564) = _retain_leaf (:615-633) + identifier shift
 * (:476) + _shift_dual_variables (:635-666) + _pi_sum (:668-721) + the runtime pi3 / lb rules
 * (:541-558), and the plant update x <- x_1|t + e_t of the closed loop
 * (notebooks/cart_pole_with_walls/statistical_analysis.py:194).
 *   d_x0 [n_inst][nx] state the old tree was solved at; d_e0 [n_inst][nx] model error (NULL = 0)
 *   d_inc_cost / d_inc_primal : incumbents of the old tree (u_0 = applied input)
 *   d_active [n_inst] in/out or NULL : instances without incumbent are switched off
 *   d_x_next [n_inst][nx] = x_1 + e0 ; d_u0 [n_inst][nu] applied input (either may be NULL)
 * Capacity rule: every retained leaf takes one node AND one dual record of `new_tree`, so
 * min(new_tree.cap_nodes, new_tree.cap_recs) must be >= the number of retained leaves (<= old_tree's n_nodes), and
 * the search that follows needs 2 more nodes and 1 more record per QP it solves.  An instance whose cover does not
 * fit is switched off (d_active = 0, empty new tree; in wshmpc_closed_loop its status becomes 2 = capacity) instead
 * of continuing with a truncated cover, which could report a suboptimal or "infeasible" MIQP as solved.
 */
int wshmpc_shift_tree(wshmpc_handle *h, int n_inst, const double *d_x0, const double *d_e0,
                      const wshmpc_tree *old_tree, const double *d_inc_cost, const double *d_inc_primal,
                      int *d_active, const wshmpc_tree *new_tree, double *d_x_next, double *d_u0);

/* Fused closed loop -- many receding-horizon steps of a batch of independent instances in ONE launch,
 * with no barrier between the steps of different instances (a queue of (instance, next step) tasks in
 * global memory feeds the CTAs).  Replaces the experiment loop of
 * notebooks/cart_pole_with_walls/statistical_analysis.py:93-196 (cold or warm-started feedforward,
 * construct_warm_start, x <- x_1|t + e_t on the linear plant) for the whole batch; results are identical to
 * calling wshmpc_bnb_solve + wshmpc_shift_tree once per step.  An instance without an incumbent leaves the loop, unless a
 * fallback is configured (wshmpc_closed_loop_fallback).
 */
/* Host mailbox of the fused closed loop: the host is in the loop EVERY receding-horizon step of every instance (a true
 * plant, measured states) and there is still no barrier between instances -- what a per-step call of
 * `feedforward` + `construct_warm_start` (statistical_analysis.py:120-196) costs the reference once per instance, without
 * the lock step a batched per-step call would impose.  All arrays are pinned, mapped HOST memory owned by the library; the
 * kernel of wshmpc_closed_loop runs while the host polls them:
 *   kernel, after the B&B of step s of instance i:  writes out_u0 / out_x1 / out_cost / out_status [i], then out_step[i] = s + 1
 *   host, when it sees out_step[i] == s + 1:        applies out_u0[i] to its plant, writes the measured state in_x[i] and the
 *                                                   model error in_e[i] = in_x[i] - out_x1[i] (construct_warm_start's e0,
 *                                                   controller.py:503-564), then in_step[i] = s + 1
 *   kernel, when a lane next picks instance i:      waits for in_step[i] >= s + 1, builds the warm start (K2 + K4), solves step s + 1
 * The host answers EVERY published step, also the last one of the launch and those of instances that report no incumbent.
 * `stop` != 0 (or `timeout_ms` without an answer; 0 = 5000 ms) makes the kernel abandon the instances it waits for
 * (status 4) and drain -- a dead host, or a profiler that serialises launches, can never leave the GPU spinning.
 * Counters are per launch: zero in_step / out_step / stop before each wshmpc_closed_loop. */
typedef struct {
    int n_inst, nx, nu;
    volatile int *out_step;           /* [n_inst] steps of the instance published in this launch */
    double *out_u0;                   /* [n_inst][nu] input to apply (NaN: the step has no incumbent) */
    double *out_x1;                   /* [n_inst][nx] predicted next state x_1|t */
    double *out_cost;                 /* [n_inst] optimal cost (+inf: none) */
    int *out_status;                  /* [n_inst] status of the step's branch and bound (wshmpc_bnb_solve) */
    volatile int *in_step;            /* [n_inst] steps of the instance answered in this launch */
    double *in_x;                     /* [n_inst][nx] measured state the next step starts from */
    double *in_e;                     /* [n_inst][nx] model error */
    volatile int *stop;               /* [1] */
    int timeout_ms;                   /* how long a lane waits for one answer before it gives the instance up (0: 5000 ms) */
    void *priv;                       /* library-owned (device scratch) */
} wshmpc_mailbox;

int wshmpc_mailbox_create(wshmpc_handle *h, int n_inst, wshmpc_mailbox *mb);
int wshmpc_mailbox_destroy(wshmpc_handle *h, wshmpc_mailbox *mb);

typedef struct {
    int n_steps;                      /* receding-horizon steps to run per instance */
    int warm;                         /* 1: warm start by tree shifting, 0: every step from the root node */
    int fresh;                        /* 1: step 0 starts from the root node (no tree yet) */
    int par;                          /* which tree / state buffer (0 or 1) holds the data of step 0 */
    int *d_queue;                     /* [4 + (n_inst + 2) * (n_steps + 1)] scratch (per-step task queues) */
    int *d_step_of;                   /* [n_inst] scratch */
    double *d_x;                      /* [2][n_inst][nx] states, buffer `par` holds the current ones */
    const double *d_e;                /* [n_steps][n_inst][nx] model errors, or NULL */
    int *d_active;                    /* [n_inst] in/out */
    double *d_log_cost;               /* [n_steps][n_inst] optimal cost of every step (+inf: infeasible) */
    double *d_log_u0;                 /* [n_steps][n_inst][nu] applied input (NaN once an instance is off) */
    int *d_log_solves;                /* [n_steps][n_inst] QP relaxations solved */
    int *d_log_status;                /* [n_steps][n_inst] status of wshmpc_bnb_solve */
    const wshmpc_mailbox *mailbox;    /* NULL: the plant x <- x_1|t + e_t is advanced on the device (d_e); else the host is
                                       * in the loop every step (d_e unused) and the call returns while the kernel runs */
} wshmpc_loop;

int wshmpc_closed_loop(wshmpc_handle *h, int n_inst, const wshmpc_loop *loop,
                       const wshmpc_tree *tree0, const wshmpc_tree *tree1, double tol, int max_solves,
                       double *d_inc_cost, int *d_inc_node, double *d_inc_primal, int *d_n_solves,
                       int *d_status, unsigned long long *d_totals);

/* The nonlinear benchmark plant on the device: the cart-pole between two soft walls (plants.CartPoleWithWalls), integrated
 * by explicit Euler with n_sub sub-steps of dt / n_sub and the cart force held constant over dt -- the rule of
 * CartPoleWithWalls.simulate.  The state is x = (qc, qp, qc', qp') (nx = 4); the cart force is input component fc_index. */
#define WSHMPC_PLANT_CARTPOLE_NPARAM 7      /* mc, mp, l, d, stiffness, damping, g */
typedef struct {
    int kind;              /* 1: cart-pole between two soft walls (plants.CartPoleWithWalls); other values are errors */
    int n_sets;            /* 1: every instance uses set 0;  n_inst (or n for wshmpc_plant_step): set k for instance k */
    const double *d_params;/* [n_sets][WSHMPC_PLANT_CARTPOLE_NPARAM], device */
    double dt;             /* sample time of the controller's model */
    int n_sub;             /* Euler sub-steps per sample */
    int fc_index;          /* input component applied as the cart force */
    double *d_log_x;       /* [n_steps][n_inst][nx] state after every step, or NULL (closed loop only) */
} wshmpc_plant;

/* d_x_out[i] = the plant's state after dt from d_x[i] under the input d_u[i] (one thread per state; asynchronous).
 *   d_x, d_x_out [n][nx] (may not overlap), d_u [n][nu] */
int wshmpc_plant_step(wshmpc_handle *h, const wshmpc_plant *pl, int n, const double *d_x, const double *d_u, double *d_x_out);

/* wshmpc_closed_loop against the nonlinear plant, advanced on the device.  For every step t of a live instance i with an
 * incumbent:  u0 = the incumbent's first input,  x_meas = Phi(x_t, u0[fc_index]; set i) + d_e[t][i] (loop->d_e optional:
 * an additive disturbance on the plant output),  the warm start is corrected with e = x_meas - x_1|t (construct_warm_start's
 * e0), and x_{t+1} = x_meas.  An instance without an incumbent keeps its state and is switched off, unless a fallback is
 * configured (wshmpc_closed_loop_fallback).  Results equal calling
 * wshmpc_bnb_solve, wshmpc_plant_step and wshmpc_shift_tree (with e0 = e) once per step.  A mailbox is an error (the host is
 * the plant there). */
int wshmpc_closed_loop_plant(wshmpc_handle *h, int n_inst, const wshmpc_loop *loop, const wshmpc_plant *plant,
                             const wshmpc_tree *tree0, const wshmpc_tree *tree1, double tol, int max_solves,
                             double *d_inc_cost, int *d_inc_node, double *d_inc_primal, int *d_n_solves,
                             int *d_status, unsigned long long *d_totals);

/* Fallback through infeasible MIQPs: an instance whose step has no incumbent applies the next input of its last plan and
 * solves again at the next sample, instead of leaving the loop.  The plan is the primal record of the last step with an
 * incumbent and `age` counts the steps since then (-1: no plan).  At step t of a live instance, after its branch and bound:
 *   incumbent                                 plan <- incumbent, age <- 0; the applied pair is the incumbent;       hold 0
 *   status 1 (infeasible), age + 1 <= max_hold  age <- age + 1; applied u_0 = u_age of the plan,
 *                                             x_1|t = A x_t + B u_0; the instance stays live;                      hold age
 *   status 1, otherwise (no plan or plan used up), law_n + 1 <= max_law
 *                                             law_n <- law_n + 1; applied u_0 = K x_t (the terminal law),
 *                                             x_1|t = A x_t + B u_0; age kept; the instance stays live;              hold -2
 *   otherwise (law used up, status 2 or 3, instance off)   the instance is switched off as without a fallback;      hold -1
 * An incumbent also resets law_n to 0.  The terminal law is the linear feedback of the terminal set (e.g. the LQR gain it was
 * built with), without offset or saturation; K is [nu][nx], row-major, shared by all instances.
 * A status-1 step ran its search to the end: its leaves are a complete cover (Farkas proofs and bounds) and K2 + K4 shift them
 * with the applied input like a solved tree, for any input.  The logs of a fallback step keep cost +inf and status 1; u0 is
 * the applied input.  All buffers are device memory owned by the caller, so plans survive launches.
 *   d_plan       [n_inst][layout.primal]
 *   d_age        [n_inst] in/out (fill with -1 to start without plans)
 *   d_app_cost   [n_inst] applied pair, what K2 + K4 and the plant read in place of the incumbent: the incumbent's cost, 0 on a
 *                fallback step, +inf where the instance leaves the loop
 *   d_app_primal [n_inst][layout.primal] the incumbent's record; on a fallback step only x_0, x_1 and u_0 are defined.
 *                Must not overlap d_plan.
 *   d_hold       [n_steps][n_inst] (wshmpc_closed_loop_fallback) or [n_inst] (wshmpc_fallback_step): 0 the incumbent,
 *                a > 0 input u_a of the plan, -2 the terminal law, -1 the instance left the loop (or was off)
 *   d_law_K      [nu][nx] the terminal law's gain (read when max_law > 0)
 *   d_law_n      [n_inst] in/out, law steps since the last incumbent (fill with 0 to start; read when max_law > 0)
 * max_hold = max_law = 0 is the behaviour without a fallback, bit for bit; max_law = 0 is the policy without the law. */
typedef struct {
    int max_hold;          /* H, 0 <= H <= T - 1 */
    double *d_plan;
    int *d_age;
    double *d_app_cost;
    double *d_app_primal;
    int *d_hold;
    int max_law;           /* L >= 0 */
    const double *d_law_K;
    int *d_law_n;
} wshmpc_fallback;

/* wshmpc_closed_loop (plant = NULL: the linear plant x <- x_1|t + e_t) or wshmpc_closed_loop_plant under the fallback policy:
 * the plant and the warm start of every step use the applied pair.  Fails under node rules 1 and 2 (the comparator), with a
 * mailbox, for max_hold outside 0 .. T - 1, null buffers, d_plan overlapping d_app_primal, max_law < 0, or max_law > 0 with a
 * null d_law_K or d_law_n. */
int wshmpc_closed_loop_fallback(wshmpc_handle *h, int n_inst, const wshmpc_loop *loop, const wshmpc_plant *plant,
                                const wshmpc_fallback *fb, const wshmpc_tree *tree0, const wshmpc_tree *tree1, double tol,
                                int max_solves, double *d_inc_cost, int *d_inc_node, double *d_inc_primal, int *d_n_solves,
                                int *d_status, unsigned long long *d_totals);

/* Lock-step form of the policy, between wshmpc_bnb_solve and wshmpc_shift_tree / wshmpc_plant_step (one thread per instance,
 * asynchronous): writes d_app_cost, d_app_primal, d_age, d_plan and d_hold [n_inst] from the step's d_status / d_inc_cost /
 * d_inc_primal at states d_x; d_active (NULL: every instance) marks the live instances.  The caller then passes d_app_cost and
 * d_app_primal to wshmpc_shift_tree as the incumbent (and u_0 of d_app_primal to the plant).  Same failures as above. */
int wshmpc_fallback_step(wshmpc_handle *h, int n_inst, const wshmpc_fallback *fb, const double *d_x, const int *d_active,
                         const int *d_status, const double *d_inc_cost, const double *d_inc_primal);

/* Batched small LPs in standard form (SURVEY.md 8f-2):   min c'y  s.t.  E y = r,  y >= 0   for n_lp problems at once,
 * one CTA per LP (two-phase tableau simplex in shared memory).  Replaces the host LP loops the reference runs through
 * BoundedQP / Gurobi while a controller is built: `_update_mu` (controller.py:186-227: h_Tm1.size LPs sharing [F G]' and h,
 * one right-hand side each) and, through the dual, the `max c.x s.t. D x <= e` LPs of mcais.py:44-184.
 *   d_E [n_lp or 1][m][n] row-major, stride_E = m*n or 0 (shared); d_c [n_lp or 1][n], stride_c = n or 0; d_r [n_lp][m]
 *   d_status [n_lp]: 2 optimal, 3 infeasible, 5 unbounded, 9 iteration limit;  d_obj [n_lp];  d_y [n_lp][n];
 *   d_dual [n_lp][m]: multipliers pi of the equality rows (c - E'pi >= 0, obj = r.pi);  d_iters [n_lp] pivots.
 * m <= 64.  All pointers are device pointers. */
int wshmpc_lp_batch(int device, void *stream, int n_lp, int m, int n, const double *d_E, long long stride_E,
                    const double *d_c, long long stride_c, const double *d_r, double tol, int max_iter,
                    int *d_status, double *d_obj, double *d_y, double *d_dual, int *d_iters);

#ifdef __cplusplus
}
#endif
#endif
