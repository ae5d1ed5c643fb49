/*
 * tzddpc.h -- C ABI of libtzddpc.so: the B200 (sm_100a) hot path of TZDDPC.
 *
 * The reference (rssalessio/TZDDPC) is pure Python; its hot path calls into the
 * third-party packages pyzonotope / pydatadrivenreachability / cvxpy.  Each entry
 * point below replaces one of those call sites (cited as file:line relative to the
 * reference root) and is what a ctypes / torch-custom-op binding on the reference
 * side would bind (see INTEGRATION.md).
 *
 * Conventions
 *   - return 0 on success, a negative TZ_E* code otherwise; nothing throws across the ABI;
 *     tz_last_error() returns a thread-local message for the last failing call;
 *   - every `double*` / `int32_t*` is CALLER-OWNED DEVICE memory unless the name ends in
 *     `_host`; the library allocates nothing on the device except inside
 *     tz_program_create (freed by tz_program_destroy);
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*), no implicit sync;
 *   - thread-safe: the only process-wide state is a cache of "dynamic shared-memory attribute already set for kernel k
 *     on device d" bits (idempotent, atomic) and the per-thread stream pool of tz_closed_loop_step_host; per-scenario
 *     failures go to `status[S]` (TZ_STATUS_*), never to the return code;
 *   - arithmetic is IEEE fp64 throughout.
 *
 * Layouts
 *   SoA ("scenario-fastest"), used by the fused closed-loop path: a batch of S vectors of
 *       length d is a d x S row-major array, element (i, s) at [i*S + s].
 *   AoS ("one zonotope per block"), used by the stand-alone zonotope ops: a batch of S
 *       zonotopes is S x n x (1+g) row-major, Z[s] = [c, G] with column 0 the centre.
 */
#ifndef TZDDPC_H
#define TZDDPC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TZ_OK 0
#define TZ_EINVAL (-22)    /* bad argument / shape                                  */
#define TZ_ENOMEM (-12)    /* allocation failed                                     */
#define TZ_ERANGE (-34)    /* program larger than every compiled kernel bucket      */
#define TZ_ECUDA (-5)      /* CUDA runtime error (message in tz_last_error)         */

/* per-scenario status written by the solve kernels (SURVEY.md section 5) */
#define TZ_STATUS_OK 0
#define TZ_STATUS_MAXITER 1     /* ADMM hit max_iter before eps                     */
#define TZ_STATUS_INFEASIBLE 2  /* reference: raises 'Problem is unbounded', tzddpc/tzddpc.py:374-375 */
#define TZ_STATUS_NONFINITE 3

const char* tz_version(void);
/* copies the calling thread's last error message, returns its length */
size_t tz_last_error(char* buf, size_t cap);
/* compute capability (major*10+minor) of the current device, or a negative error */
int tz_device_cc(void);

/* ------------------------------------------------------------------------------------
 * Parametric per-step program (the canonicalised form of tzddpc/tzddpc.py:132-241).
 *
 *   minimise   0.5 z'Pz + (q0 + Qp p)'z + sum_i wabs_i |(Az)_i - kink0_i - r_i(p)| + c0(p)
 *   subject to l0 + r(p) <= A z <= u0 + r(p),      r(p) = R [1; p; alpha(p)],
 *              alpha_j(p) = |Bt_j p + gam_j|,       p = [xbar0; e0]  (tzddpc/tzddpc.py:155-157)
 *   feasible (parameter-only rows, e.g. xbar0 + e0 in X) iff  Rchk [1; p; alpha] <= 0
 *   c0(p) = cc [1; p; alpha] + p' CC2 p
 *
 * All arrays are HOST pointers, row-major, unscaled; D, E, c are the Ruiz scalings
 * (z = D zbar, Abar = E A D, Pbar = c D P D).  Rows with wabs > 0 must come first.
 * ------------------------------------------------------------------------------------ */
typedef struct TzProgramDesc {
  int32_t n, m, horizon;      /* dim_x, dim_u, N                                          */
  int32_t nv, nz, nc;         /* N*m decision inputs, nv + epigraph variables, rows       */
  int32_t npar, na, nchk;     /* 2n, #alpha atoms, #parameter-only check rows             */
  int32_t nkink;              /* rows [0, nkink) carry an |.| cost                         */
  int32_t g1;                 /* generators of Ze[1] (tzddpc/tzddpc.py:205-207,377)       */
  int32_t nterms;             /* nnz of the Ze[1] term table                              */
  const double *P, *q0, *Qp;  /* nz*nz, nz, nz*npar                                       */
  const double *A;            /* nc*nz                                                    */
  const double *l0, *u0, *kink0, *wabs;   /* nc each (+-inf allowed in l0/u0)             */
  const double *R;            /* nc*(1+npar+na)                                           */
  const double *Bt, *gam;     /* na*npar, na                                              */
  const double *Rchk;         /* nchk*(1+npar+na)                                         */
  const double *cc, *CC2;     /* 1+npar+na, npar*npar                                     */
  const double *XB;           /* (N+1)n * (1+nv+npar): xbar_0..xbar_N = XB [1; v; p]      */
  const int32_t *ze1_ptr;     /* n(1+g1)+1 : CSR over the entries of Ze[1].Z, row-major   */
  const int32_t *ze1_idx;     /* nterms: index into w = [1; v; p]                         */
  const double *ze1_val;      /* nterms                                                   */
  const double *D, *E;        /* nz, nc                                                   */
  double c;                   /* cost scaling                                             */
  const double *K;            /* m*n feedback gain theta.K (examples/2.pulley_sim.py:91)  */
} TzProgramDesc;

typedef struct TzProgram TzProgram;   /* opaque */

int tz_program_create(const TzProgramDesc* desc, TzProgram** out);
void tz_program_destroy(TzProgram* prog);
/* D programs of one structure (the same problem built from D data sets: the data-set axis) created at once -- packed on the
 * host, one device allocation and one copy for all of them.  tz_program_batch_get(batch, d) is a program handle as
 * tz_program_create returns it, borrowed from the batch: pass it to tz_solve, tz_program_set_create, ...; do not destroy
 * it, destroy the batch (after every set built from it). */
typedef struct TzProgramBatch TzProgramBatch;   /* opaque */
int tz_program_create_batch(const TzProgramDesc* descs, int32_t D, TzProgramBatch** out);
const TzProgram* tz_program_batch_get(const TzProgramBatch* batch, int32_t d);
void tz_program_batch_destroy(TzProgramBatch* batch);
/* which compiled kernel bucket serves this program: writes e.g. "B2(NZ=2,NC=28,G=4)" into buf */
int tz_program_bucket(const TzProgram* prog, char* buf, size_t cap);
/* rows of the `warm` scratch array (rows x S doubles) that tz_solve / tz_closed_loop_step accept */
int tz_program_warm_rows(const TzProgram* prog);

/* Array sizes of a program, for bindings that validate caller buffers:
 * out8 = [n, m, N*m, (N+1)*n, n*(1+g1), n_nz (packed tube rows), tz_program_warm_rows, CUDA device of the program]. */
int tz_program_dims(const TzProgram* prog, int32_t* out8);

/* Sparsity pattern of Ze[1].Z: returns n_nz, the number of entries that are not structurally zero, and (when
 * entries_host != NULL, cap >= n_nz) writes their row-major indices r*(1+g1)+j into entries_host.  Centre column included. */
int tz_program_tube_pattern(const TzProgram* prog, int32_t* entries_host, int32_t cap);

typedef struct TzSolverOpts {
  double rho;        /* base ADMM penalty (scaled problem)         default 0.1  */
  double rho_active; /* multiplier for rows detected active        default 100  */
  double rho_inactive;/* multiplier for rows detected inactive     default 0.1  */
  double sigma;      /* proximal weight                            default 1e-6 */
  double alpha;      /* over-relaxation                            default 1.6  */
  double eps_abs, eps_rel;   /*                                     default 1e-6 */
  int32_t max_iter;  /*                                            default 4000 */
  int32_t check_every;/* residual check period                     default 8    */
  int32_t polish;    /* masked augmented-Lagrangian polish: number of iterations, 0 = off   default 3 */
  int32_t warm_start;/* 0 cold; 1 reuse (x, y) of the previous call from the `warm` buffer; 2 active-set hint:
                        the previous call's optimal active set is tried first and accepted only when the KKT
                        conditions hold there; a code that cannot mean anything for its row (equality on a row
                        whose bounds differ, kink on a row without an |.| cost, a missing bound) rejects the
                        hint.  So a stale or arbitrary hint only costs the test (tested against an exact
                        optimum for every hint with up to two active rows and for random words, two-variable
                        programs; against the oracle for larger ones); the buffer carries one word per lane
                        default 0 */
  int32_t cert_first;/* first iteration at which the active-set KKT certificate is tried (then on a
                        geometric schedule); a certified iterate is an exact solution and ends the
                        solve at once.  0 = off (terminate on residuals only)        default 3    */
  int32_t tube_packed;/* 0: `ze1` is the dense n(1+g1) x S matrix the reference returns (Zek.Z.value).
                        1: `ze1` is n_nz x S -- row i holds entry tz_program_tube_pattern()[i] of Ze[1].Z; the other
                        entries are zero for EVERY (xbar0, e0) (boxed M_K / M_Delta: 88 % of the 5-dim tube) and are
                        neither written to HBM nor copied to the host                  default 0 */
  int32_t hot_path;  /* 1: with warm_start == 2, programs with two decision variables (horizon 2, one input: every shipped
                        example) run fast_step_kernel -- one thread per scenario, closed-form KKT certificate of the hinted
                        active set -- and only the 16-scenario tiles it cannot decide go through the ADMM kernel.
                        0: the ADMM kernel for everything (same results bit for bit)      default 1 */
} TzSolverOpts;

void tz_solver_opts_default(TzSolverOpts* o);

/* ------------------------------------------------------------------------------------
 * tz_solve: batched replacement of TZDDPC.solve(xbar0, e0), tzddpc/tzddpc.py:357-377.
 *   in : xbar0, e0           n x S   (SoA)
 *   out: cost                S
 *        v                   (N*m) x S
 *        xbar_traj           ((N+1)*n) x S
 *        ze1                 (n*(1+g1)) x S   Ze[1].Z, entry (r, j) at row r*(1+g1)+j   (n_nz x S with opts->tube_packed)
 *        status, iters       S   (int32)
 *   warm: tz_program_warm_rows(prog) x S scratch carrying the ADMM iterate between calls, or NULL
 *   any of cost / v / xbar_traj / ze1 / iters may be NULL (not written).
 * ------------------------------------------------------------------------------------ */
int tz_solve(const TzProgram* prog, const TzSolverOpts* opts, int64_t S,
             const double* xbar0, const double* e0,
             double* cost, double* v, double* xbar_traj, double* ze1,
             int32_t* status, int32_t* iters, double* warm, void* stream);

/* ------------------------------------------------------------------------------------
 * tz_closed_loop_step: one fused closed-loop step for S scenarios
 * (examples/2.pulley_sim.py:81-96 ; examples/3.5dimsystem_sim.py:73-89):
 *     (cost, v, xbar_traj, Ze1) = solve(xbar, e)
 *     u = K e + v[0];  x+ = A_true x + B_true u + w;  xbar+ = xbar_traj[1];  e+ = x+ - xbar+
 *   x, xbar, e    n x S, updated IN PLACE
 *   noise         n x S   the realisation w_t (an input: W.sample(), :92)
 *   x_restart     n x S or NULL.  The reference ends a run when a step is infeasible (raises, tzddpc/tzddpc.py:374-375).
 *                 With x_restart such a scenario starts a new run: x = xbar = x_restart, e = 0
 *                 (examples/2.pulley_sim.py:66-72); with NULL it keeps its state (and stays infeasible).
 *   A_true,B_true device n*n, n*m row-major (the simulated plant)
 *   u_out         m x S or NULL
 *   stats         TZ_NSTATS doubles accumulated with atomics, or NULL:
 *                 [sum |x+|_2, sum |x+|_2^2, sum cost, #infeasible, #maxiter, sum iters, #non-finite, S]
 * ------------------------------------------------------------------------------------ */
#define TZ_NSTATS 8
int tz_closed_loop_step(const TzProgram* prog, const TzSolverOpts* opts, int64_t S,
                        double* x, double* xbar, double* e, const double* noise, const double* x_restart,
                        const double* A_true, const double* B_true,
                        double* cost, double* v, double* xbar_traj, double* ze1, double* u_out,
                        int32_t* status, int32_t* iters, double* warm, double* stats, void* stream);

/* K closed-loop steps in ONE launch (the whole loop of examples/2.pulley_sim.py:81-96 for a small batch, where the launch
 * per step is what a step costs): exactly K consecutive tz_closed_loop_step calls, bit for bit.  Scenarios are
 * independent, so a warp keeps its scenarios for all steps.  `noise` and every per-step output hold K consecutive
 * blocks (step-major: noise K x n x S, cost K x S, v K x nv x S, xbar_traj K x (N+1)n x S, ze1 K x rows x S,
 * u_out K x m x S, status / iters K x S, stats K x TZ_NSTATS); x_hist, xbar_hist, e_hist (K x n x S each, or NULL) receive
 * the state after every step; x, xbar, e are updated in place.  Programs of the register buckets (up to 12 variables). */
int tz_closed_loop_run(const TzProgram* prog, const TzSolverOpts* opts, int64_t S, int32_t nsteps, double* x, double* xbar,
                       double* e, const double* noise, const double* x_restart, const double* A_true, const double* B_true,
                       double* cost, double* v, double* xbar_traj, double* ze1, double* u_out, double* x_hist, double* xbar_hist,
                       double* e_hist, int32_t* status, int32_t* iters, double* warm, double* stats, void* stream);

/* ------------------------------------------------------------------------------------
 * A plant per scenario: tz_closed_loop_step / tz_closed_loop_run (and tz_closed_loop_step_set below) with
 *   AB_true       n(n+m) x S   (SoA) in place of A_true, B_true: entry (i, k) of scenario s's [A_true B_true] at
 *                 AB_true[(i (n+m) + k) S + s] -- the layout tz_sample_plants writes.
 * Run a closed loop per plant of a set (e.g. plants drawn from M_Sigma, to check the tube guarantee on every plant the data
 * cannot rule out), or each data set's closed loop on the system that produced its data.  With every column equal to
 * [A_true B_true] the results equal the shared-plant call bit for bit.
 * ------------------------------------------------------------------------------------ */
int tz_closed_loop_step_plants(const TzProgram* prog, const TzSolverOpts* opts, int64_t S,
                               double* x, double* xbar, double* e, const double* noise, const double* x_restart,
                               const double* AB_true,
                               double* cost, double* v, double* xbar_traj, double* ze1, double* u_out,
                               int32_t* status, int32_t* iters, double* warm, double* stats, void* stream);
int tz_closed_loop_run_plants(const TzProgram* prog, const TzSolverOpts* opts, int64_t S, int32_t nsteps, double* x, double* xbar,
                              double* e, const double* noise, const double* x_restart, const double* AB_true,
                              double* cost, double* v, double* xbar_traj, double* ze1, double* u_out, double* x_hist, double* xbar_hist,
                              double* e_hist, int32_t* status, int32_t* iters, double* warm, double* stats, void* stream);

/* ------------------------------------------------------------------------------------
 * Data-set axis (BASELINE.json north_star: scenarios = noise realisations x initial states x data sets).
 * The reference builds one TZDDPC object -- one model M_Sigma, one problem -- per data set (tzddpc/tzddpc.py:20-28,
 * 67-85,132-241) and runs them one after another.  A program set runs D such programs in ONE launch: scenarios
 * [begin[j], begin[j+1]) of the batch use progs[j].  The programs must be the same problem (dimensions, horizon,
 * cost / constraint structure, hence kernel bucket and table sizes) built from different data; begin[0] = 0, begin[j]
 * a multiple of 16, begin[D] = S of every later call.  The set borrows the programs: destroy it before them.
 * tz_solve_set / tz_closed_loop_step_set take the arguments of tz_solve / tz_closed_loop_step.
 * ------------------------------------------------------------------------------------ */
typedef struct TzProgramSet TzProgramSet;   /* opaque */
int tz_program_set_create(const TzProgram* const* progs, int32_t nprog, const int64_t* begin, TzProgramSet** out);
void tz_program_set_destroy(TzProgramSet* set);
int64_t tz_program_set_scenarios(const TzProgramSet* set);
int tz_program_set_dims(const TzProgramSet* set, int32_t* out8);      /* as tz_program_dims (the programs share them) */
int tz_solve_set(const TzProgramSet* set, const TzSolverOpts* opts, int64_t S,
                 const double* xbar0, const double* e0,
                 double* cost, double* v, double* xbar_traj, double* ze1,
                 int32_t* status, int32_t* iters, double* warm, void* stream);
int tz_closed_loop_step_set(const TzProgramSet* set, const TzSolverOpts* opts, int64_t S,
                            double* x, double* xbar, double* e, const double* noise, const double* x_restart,
                            const double* A_true, const double* B_true,
                            double* cost, double* v, double* xbar_traj, double* ze1, double* u_out,
                            int32_t* status, int32_t* iters, double* warm, double* stats, void* stream);
/* tz_closed_loop_step_set with a plant per scenario, AB_true n(n+m) x S as tz_closed_loop_step_plants */
int tz_closed_loop_step_set_plants(const TzProgramSet* set, const TzSolverOpts* opts, int64_t S,
                                   double* x, double* xbar, double* e, const double* noise, const double* x_restart,
                                   const double* AB_true,
                                   double* cost, double* v, double* xbar_traj, double* ze1, double* u_out,
                                   int32_t* status, int32_t* iters, double* warm, double* stats, void* stream);
/* tz_closed_loop_run / tz_closed_loop_run_plants over a program set: K closed-loop steps of every data set's scenarios in
 * ONE launch, exactly K consecutive tz_closed_loop_step_set (_plants) calls, bit for bit (nsteps = 1 is one such call).
 * The layout of tz_closed_loop_run: per-step blocks of S scenarios (K x n x S noise, K x S status, ...), the histories
 * included.  S must be tz_program_set_scenarios(set); nsteps < 1 or another S is TZ_EINVAL. */
int tz_closed_loop_run_set(const TzProgramSet* set, const TzSolverOpts* opts, int64_t S, int32_t nsteps, double* x, double* xbar,
                           double* e, const double* noise, const double* x_restart, const double* A_true, const double* B_true,
                           double* cost, double* v, double* xbar_traj, double* ze1, double* u_out, double* x_hist, double* xbar_hist,
                           double* e_hist, int32_t* status, int32_t* iters, double* warm, double* stats, void* stream);
int tz_closed_loop_run_set_plants(const TzProgramSet* set, const TzSolverOpts* opts, int64_t S, int32_t nsteps, double* x,
                                  double* xbar, double* e, const double* noise, const double* x_restart, const double* AB_true,
                                  double* cost, double* v, double* xbar_traj, double* ze1, double* u_out, double* x_hist,
                                  double* xbar_hist, double* e_hist, int32_t* status, int32_t* iters, double* warm, double* stats,
                                  void* stream);

/* Same step with HOST buffers (pinned or pageable): H2D of (x, xbar, e, noise), the fused
 * kernel, D2H of every non-NULL output, chunked over `nchunks` internal streams so that
 * copies overlap compute; synchronises before returning.  `dev_scratch` is caller-owned
 * device memory of at least tz_closed_loop_step_host_scratch_bytes(prog, S).  With opts->warm_start != 0 its tail
 * carries the solver's warm-start rows (active-set hints) from one call to the next: zero it once before the first
 * call of a run and pass the same buffer every step (a stale or foreign hint is KKT-checked before use, and rejected
 * when a code does not fit its row, so it can cost time but not correctness; see warm_start).  With opts->tube_packed,
 * ze1_host is n_nz x S. */
size_t tz_closed_loop_step_host_scratch_bytes(const TzProgram* prog, int64_t S);
int tz_closed_loop_step_host(const TzProgram* prog, const TzSolverOpts* opts, int64_t S,
                             double* x_host, double* xbar_host, double* e_host, const double* noise_host,
                             const double* A_true_host, const double* B_true_host,
                             double* cost_host, double* v_host, double* xbar_traj_host, double* ze1_host,
                             int32_t* status_host, void* dev_scratch, int32_t nchunks);

/* The closed loop with the state RESIDENT on the device: (x, xbar, e), x_restart, the plant matrices and the active-set
 * hints live in `dev_scratch` (same size query as above) from one call to the next, as the reference keeps them in its
 * Python lists between calls of `solve` (examples/2.pulley_sim.py:81-96).
 *   flags & 1   upload x, xbar, e (and x_restart when non-NULL: an infeasible scenario starts a new run from it), A_true,
 *               B_true before the step -- the first call of a run (zero dev_scratch once before it);
 *   flags & 2   download xbar and e after the step, too (x always comes down).
 * Per call only the step's noise goes up and x+ and the non-NULL outputs (cost, v, xbar_traj, ze1, u = K e + v[0], status)
 * come down.  x_restart_host is only read with flags & 1. */
int tz_closed_loop_run_host(const TzProgram* prog, const TzSolverOpts* opts, int64_t S, int32_t flags,
                            double* x_host, double* xbar_host, double* e_host, const double* x_restart_host,
                            const double* noise_host, const double* A_true_host, const double* B_true_host,
                            double* cost_host, double* v_host, double* xbar_traj_host, double* ze1_host, double* u_host,
                            int32_t* status_host, void* dev_scratch, int32_t nchunks);

/* ------------------------------------------------------------------------------------
 * Stand-alone zonotope ops (AoS batches).
 * ------------------------------------------------------------------------------------ */

/* Interval hull  c -+ sum_j |G[:, j]|   (Zonotope.interval, tzddpc/tzddpc.py:191-197).
 * Z: S x n x (1+g);  lo, hi: S x n. */
int tz_interval_hull(int64_t S, int32_t n, int32_t g, const double* Z, double* lo, double* hi, void* stream);

/* MatrixZonotope x Zonotope (+ Zonotope)  (tzddpc/tzddpc.py:175-176,181,185,205):
 *   Zout[s] = [C Z_s, G_1 Z_s, ..., G_N Z_s]  (+) W      with Z_s = [c, G]  (p x (1+g))
 * C: n x p, Gm: N x n x p (shared by all scenarios when model_stride == 0, else per scenario
 * with C at C + s*n*p and Gm at Gm + s*N*n*p).  W: n x (1+gW) or NULL (gW = 0).
 * Zout: S x n x ((N+1)(1+g) + gW). */
int tz_reach_step(int64_t S, int32_t n, int32_t p, int32_t N, int32_t g, int32_t gW,
                  const double* C, const double* Gm, int32_t per_scenario_model,
                  const double* Z, const double* W, double* Zout, void* stream);

/* Girard order reduction (Zonotope.reduce / MatrixZonotope.reduce, tzddpc/tzddpc.py:126-128,
 * examples/1.double_integrator_sim.py:170; SURVEY.md App. A.5):
 *   drop all-zero generators; if g' <= order*n keep; else box the g' - floor(n(order-1))
 *   generators of smallest metric (ties: lowest index) into diag(sum|.|), kept ones first
 *   in original order.  metric: 0 = l1 - linf, 1 = l1, 2 = l2.
 * Z: S x n x (1+g) -> Zout: S x n x (1+gout_cap), gout[s] = generators written (<= gout_cap,
 * columns beyond are zero).  gout_cap >= max(n*order rounded up, g when no reduction). */
int tz_girard_reduce(int64_t S, int32_t n, int32_t g, double order, int32_t metric,
                     const double* Z, int32_t gout_cap, double* Zout, int32_t* gout, void* stream);

/* Tube rollout with in-loop order reduction (BASELINE.json configs[4]; tzddpc/tzddpc.py:175-186,205 evaluated
 * numerically + Zonotope.reduce of examples/1.double_integrator_sim.py:170 after every step):
 *   Z_{k+1} = reduce( M_K (x) Z_k  (+)  M_Delta (x) <[xbar_k; v_k], 0>  (+)  W ,  order ),   k = 0 .. steps-1
 * one CTA per scenario, the zonotope stays in shared memory for all steps.
 *   CK: n x n centre of M_K, GK: NK x n x n, GD: ND x n x (n+m) generators of M_Delta (zero centre); shared by all
 *   scenarios, or per scenario (S x ...) when per_scenario_model != 0.
 *   Z0: S x n x (1+g0);  XU: S x steps x (n+m) the nominal [xbar_k; v_k];  W: n x (1+gW) or NULL.
 *   Zfinal: S x n x (1+gcap), gfinal[s] generators of the final zonotope (negative: gcap too small, truncated);
 *   hull_lo, hull_hi: S x steps x n interval hull of Z_{k+1} (tzddpc/tzddpc.py:191-197).
 * gcap >= max(g0, floor(n (order-1)) + n).  Column order of the pre-reduction block as pyzonotope's product:
 *   [C_K G | G^K_1 c, G^K_1 G | ... | G^D_1 z .. | G_W]; reduction as tz_girard_reduce.
 * Two kernels, the same results bit for bit.  Where the pre-reduction block (n x g_pre doubles, g_pre =
 * (NK+1) gcap + NK + ND + gW) fits in shared memory with the zonotope, the matrices and 9 bytes per column (220 KiB in
 * all; at n = 5, m = 1 with the 25 + 30 + 1 generators of the stress workload: order <= 31), it is built there once per
 * step.  Otherwise its entries are recomputed wherever the reduction reads them, and only two zonotopes, the matrices and
 * the 9 bytes per column take shared memory (order <= 135 at that size).  Beyond that: TZ_EINVAL naming both sizes.
 * The environment variable TZDDPC_ROLLOUT = resident / recompute (read per call) forces one of the two where it fits. */
int tz_tube_rollout(int64_t S, int32_t n, int32_t m, int32_t NK, int32_t ND, int32_t gW, int32_t g0, int32_t steps,
                    double order, int32_t metric, const double* CK, const double* GK, const double* GD,
                    int32_t per_scenario_model, const double* Z0, const double* XU, const double* W, int32_t gcap,
                    double* Zfinal, int32_t* gfinal, double* hull_lo, double* hull_hi, void* stream);

/* Data-driven model  M_Sigma = (X1 - M_w) pinv([X0; U0])  (tzddpc/tzddpc.py:81-83) followed by
 * tzddpc/tzddpc.py:119-128 (MdataK = Mdata [I;K], Mdelta, order-1 reduction), batched over S datasets:
 *   X: S x T x n, U: S x T x m (as Data.x / Data.u), WZ: n x (1+gW) shared, K: S x m x n or NULL
 *   AB    S x n x (n+m)      centre of Mdata
 *   dAB   S x n x (n+m)      box of Mdata/Mdelta after reduce(1):  sum_i |G_i|
 *   dK    S x n x n          box of MdataK after reduce(1) (needs K)
 *   Pinv  S x (T-1) x (n+m)  pinv([X0;U0]) (optional, NULL to skip)
 * status[s] = NONFINITE when the Gram matrix is not positive definite. */
int tz_identify(int64_t S, int32_t T, int32_t n, int32_t m, int32_t gW,
                const double* X, const double* U, const double* WZ, const double* K,
                double* AB, double* dAB, double* dK, double* Pinv, int32_t* status, void* stream);

/* Batched robust gain synthesis -- the counterpart of compute_theta / is_gain_robust (tzddpc/utils.py:58-129), one CTA per
 * data set.  OPT-IN: the reference's K is "any feasible point" of an LMI found by an SDP solver and its adversary needs
 * DCCP + MOSEK (utils.py:37,43-56), so K is not reproducible; this routine keeps compute_theta's alternation
 *   K <- stabilising gain of (An, Bn)  [LQR gain of the DARE, Q = R = I]
 *   (An, Bn) <- argmax ||A + B K||_F over M_Sigma, independent beta_A / beta_B (utils.py:13-41)
 *               [convex-concave iteration beta <- -sign(gradient) from the centre and num_init-1 Philox starts]
 *   until max(rho(An + Bn K), rho(A0 + B0 K)) < 1, or it changes by less than tol, or max_iter (utils.py:80-94)
 * and the Monte-Carlo check of utils.py:105-129 with N = ceil(ln(1/confidence)/ln(1/(1-accuracy))) samples of M_Sigma.
 *   AB    D x n x (n+m)      centre of M_Sigma (tz_identify)          Pinv  D x (T-1) x (n+m)  (tz_identify)
 *   WZ    n x (1+gW)         the noise zonotope [c_W, G_W]
 *   K     D x m x n          dA D x n x n = An - A0,  dB D x n x m = Bn - B0   (Theta, tzddpc/objects.py)
 *   rho   D x 3              [rho(A0 + B0 K), rho(An + Bn K), largest sampled rho]
 *   robust, iters, status    D (int32): is_gain_robust, outer iterations, TZ_STATUS_OK / TZ_STATUS_NONFINITE (DARE failed)
 * Draws: Philox stream (seed, dataset_offset + data set, start or sample index, purposes 4 / 5). */
int tz_gain_synthesis(int64_t D, int32_t T, int32_t n, int32_t m, int32_t gW, const double* AB, const double* Pinv,
                      const double* WZ, double tol, int32_t max_iter, int32_t num_init, double accuracy, double confidence,
                      uint64_t seed, int64_t dataset_offset, double* K, double* dA, double* dB, double* rho,
                      int32_t* robust, int32_t* iters, int32_t* status, void* stream);
/* compute_A_B and is_gain_robust (tzddpc/utils.py:13-41, 105-129) for a GIVEN gain K (D x m x n): the adversarial pair
 * (A0 + dA, B0 + dB) of M_Sigma for that gain -- one pass of the convex-concave iteration above from the centre and
 * num_init-1 Philox starts -- and the Monte-Carlo check.  rho: D x 3 as tz_gain_synthesis. */
int tz_gain_adversary(int64_t D, int32_t T, int32_t n, int32_t m, int32_t gW, const double* AB, const double* Pinv,
                      const double* WZ, const double* K, int32_t num_init, double accuracy, double confidence,
                      uint64_t seed, int64_t dataset_offset, double* dA, double* dB, double* rho,
                      int32_t* robust, int32_t* status, void* stream);
/* N of the robustness check (utils.py:120), or -1 for arguments outside (0, 1) */
int32_t tz_gain_robust_samples(double accuracy, double confidence);

/* ------------------------------------------------------------------------------------
 * Counter-based random numbers (Philox4x32-10): key = seed, counter = (global scenario index, t, purpose, block).
 * The draws do not depend on how scenarios are sharded over GPUs (pass the shard's first scenario as scenario_offset);
 * oracle/philox.py restates the stream in numpy.
 * ------------------------------------------------------------------------------------ */

/* One block of the generator, on the host (for tests and bindings that want to reproduce the stream). */
void tz_philox4x32_10_host(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t* out4);

/* Closed-loop noise of step t:  w = c_W + G_W beta,  beta ~ U[-1,1)^gW (W.sample(), examples/2.pulley_sim.py:92) or, with
 * vertex != 0, beta in {-1,+1}^gW (a random vertex of W, examples/1.double_integrator_sim.py:85).  out: n x S (SoA, ld >= S). */
int tz_sample_noise(int64_t S, int64_t ld, int32_t n, int32_t gW, const double* WZ, int32_t vertex, uint64_t seed,
                    int64_t scenario_offset, uint32_t t, double* out, void* stream);

/* generate_trajectories of examples/utils.py:6-45, batched over S data sets (one trajectory each), on the device:
 *   x_0 ~ X0, u_t ~ U, x_{t+1} = A x_t + B u_t + (random vertex of W); the first returned state row is the origin (the
 *   reference's quirk, SURVEY.md 3.5-Q9).  X0Z: n x (1+g0), UZ: m x (1+gU), WZ: n x (1+gW) as [centre, generators].
 *   U: S x T x m, X: S x T x n -- the layout tz_identify reads. */
int tz_generate_trajectories(int64_t S, int32_t T, int32_t n, int32_t m, int32_t g0, int32_t gU, int32_t gW,
                             const double* A, const double* B, const double* X0Z, const double* UZ, const double* WZ,
                             uint64_t seed, int64_t scenario_offset, double* U, double* X, void* stream);
/* The same with a plant per data set: A S x n x n, B S x n x m (data set s from A + s n n, B + s n m). */
int tz_generate_trajectories_plants(int64_t S, int32_t T, int32_t n, int32_t m, int32_t g0, int32_t gU, int32_t gW,
                                    const double* A, const double* B, const double* X0Z, const double* UZ, const double* WZ,
                                    uint64_t seed, int64_t scenario_offset, double* U, double* X, void* stream);

/* Plants drawn from the data-consistent model set M_Sigma = (X1 - M_w) pinv([X0; U0]) (tzddpc/tzddpc.py:81-83), one per scenario:
 *   [A B] = AB_d - G_W R,   R[k, :] = sum_j beta_kj Pinv_d[j, :],   beta_kj ~ U[-1, 1)
 * i.e. AB_d + sum_g beta_g G_g over the generators G_g = -G_W[:, k] Pinv_d[j, :], g = k (T-1) + j, of the UN-REDUCED M_Sigma
 * (the order-1 box of tz_identify's dAB is larger than M_Sigma: a plant drawn from it is not covered by the tube).
 *   AB    D x n x (n+m), Pinv  D x (T-1) x (n+m)   as tz_identify writes them;  WZ  n x (1+gW)
 *   dataset  S int32: data set d of each scenario (an index outside [0, D) gives a NaN plant), or NULL: data set 0
 *   AB_out   n(n+m) x S  -- the AB_true layout of tz_closed_loop_step_plants
 * Draws: Philox stream (seed, scenario_offset + s, t = 0, purpose 6, draw g); gW (T-1) <= 131072. */
int tz_sample_plants(int64_t S, int32_t D, int32_t T, int32_t n, int32_t m, int32_t gW, const double* AB, const double* Pinv,
                     const double* WZ, const int32_t* dataset, uint64_t seed, int64_t scenario_offset, double* AB_out,
                     void* stream);

/* Generic batched ADMM QP on an explicit instance batch (the solver stage alone):
 *   minimise 0.5 z'Pz + q_s'z  s.t. l_s <= A z <= u_s   with (P, A) from `prog`
 *   q: nz x S, l,u: nc x S (SoA, unscaled);  z: nz x S, y: nc x S. */
int tz_qp_solve(const TzProgram* prog, const TzSolverOpts* opts, int64_t S,
                const double* q, const double* l, const double* u,
                double* z, double* y, int32_t* status, int32_t* iters, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TZDDPC_H */
