/*
 * mgb200.h -- C ABI of the B200-native geometric-multigrid hot path.
 *
 * Drop-in boundary for ONE path of soniareilly/HPCClassMultigridProject: the
 * geometric-multigrid V/W-cycle that solves the Crank-Nicolson system of the 2-D
 * advection-diffusion step.  Each entry point names the reference interface it
 * replaces (file:line into the reference repository).  Plain pointers and sizes
 * only; no C++ or torch types.  include/mgb200_compat.hpp re-creates the reference's
 * own spellings (gs.h / gscu.h / multigrid.cu signatures) on top of this file.
 *
 * Conventions
 *   - fields are FP64, (n+1) x (n+1) nodes, row-major; element (i,j) of an operator
 *     argument lives at  p[i*ld + j]  (the reference hard-wires ld = n+1).
 *   - "device" pointers are CUDA device pointers of the current device; `stream`
 *     is a cudaStream_t passed as void* (NULL = default stream).
 *   - every function returns MGB200_OK or an error code; mgb200_last_error() holds
 *     the text.  There is NO CPU fallback: without a usable sm_100 device every
 *     compute call fails with MGB200_ERR_CUDA / MGB200_ERR_NO_DEVICE.
 *   - arithmetic: MGB200_ARITH_EXACT reproduces the reference's expression order
 *     with unfused IEEE multiply/add and IEEE division (u is bit-identical to
 *     gs.cpp); MGB200_ARITH_FAST contracts to FMAs and multiplies by the
 *     precomputed reciprocal of the diagonal (<= a few ulp per update).
 */
#ifndef MGB200_H
#define MGB200_H

#ifdef __cplusplus
extern "C" {
#endif

#define MGB200_VERSION 200

enum {
    MGB200_OK = 0,
    MGB200_ERR_INVALID = 1,    /* bad argument */
    MGB200_ERR_CUDA = 2,       /* a CUDA runtime call failed */
    MGB200_ERR_NO_DEVICE = 3,  /* no CUDA device / not sm_100 */
    MGB200_ERR_NCCL = 4,       /* a NCCL call failed */
    MGB200_ERR_STATE = 5       /* call sequence error (e.g. solve before set_fields) */
};

enum { MGB200_ARITH_FAST = 0, MGB200_ARITH_EXACT = 1 };
enum { MGB200_PLAN_FUSED = 0, MGB200_PLAN_UNFUSED = 1 };
/* options.restriction: how the residual moves to the next coarser level */
enum { MGB200_RESTRICT_INJECT = 0, MGB200_RESTRICT_FW_UNFUSED = 1, MGB200_RESTRICT_FW = 2 };

int         mgb200_version(void);
const char *mgb200_last_error(void);

/* ------------------------------------------------------------------------------------------
 * Grid operators on DEVICE pointers.  Replace gs.h:3-17 (CPU) / gscu.h:3-16 (CUDA kernels and
 * the host launchers gauss_seidel, compute_norm).  `arith` is MGB200_ARITH_*.
 * ------------------------------------------------------------------------------------------ */

/* `iters` red-black Gauss-Seidel iterations in place (red = (i+j) even first).
 * gs.h:9 gauss_seidel / gscu.h:16 gauss_seidel + gscu.h:12 gs_ker (gs.cpp:109-189, gs.cu:307-392) */
int mgb200_gauss_seidel(double *u, const double *rhs, long n, long ld, const double *v1,
                        const double *v2, double dt, double nu, double dx, int iters, int arith,
                        void *stream);

/* res = rhs - A u on the interior; boundary of res untouched.
 * gs.h:3 residual / gscu.h:10 residual kernel (gs.cpp:55-83, gs.cu:157-218) */
int mgb200_residual(double *res, const double *u, const double *rhs, long n, long ld,
                    const double *v1, const double *v2, double dt, double nu, double dx, int arith,
                    void *stream);

/* sqrt(sum over the INTERIOR of a^2) -> *out_host (synchronises `stream`).  Does not clobber a.
 * gs.h:5 compute_norm / gscu.h:15 compute_norm + square_ker + reduction_kernel
 * (gs.cpp:86-107; gs.cu:13-60 sums all (N+1)^2 entries destructively -- we follow gs.cpp) */
int mgb200_compute_norm(const double *a, long n, long ld, double *out_host, void *stream);

/* sum over the interior of a^2 -> *out_dev (device double), asynchronous on `stream` */
int mgb200_norm2_async(const double *a, long n, long ld, double *out_dev, void *stream);

/* fused residual + sum of squares of it -> *out_dev; `res` may be NULL (norm only).
 * multigrid.cpp:104-105,112-113 (residual followed by compute_norm) in one pass */
int mgb200_residual_norm2_async(double *res, const double *u, const double *rhs, long n, long ld,
                                const double *v1, const double *v2, double dt, double nu,
                                double dx, int arith, double *out_dev, void *stream);

/* rhs = B u on the interior.  gs.h:13 compute_rhs / gscu.h:9 (gs.cpp:24-53, gs.cu:94-155) */
int mgb200_compute_rhs(double *rhs, const double *u, long n, long ld, const double *v1,
                       const double *v2, double dt, double nu, double dx, int arith, void *stream);

/* injection coarse[I][J] = fine[2I][2J], I,J in [0, nf/2] (boundary included).
 * gs.h:17 restriction / gscu.h:8 (gs.cpp:268-292, gs.cu:83-92); nf = FINE n */
int mgb200_restriction(double *coarse, long ldc, const double *fine, long ldf, long nf,
                       void *stream);

/* OPT-IN, not on the reference's active path: the full-weighting restriction the reference sketches
 * in commented-out lines (gs.cpp:277-280): [1 2 1; 2 4 2; 1 2 1]/16 on the coarse interior, boundary
 * injected. */
int mgb200_restriction_fw(double *coarse, long ldc, const double *fine, long ldf, long nf,
                          void *stream);

/* bilinear interpolation, every one of the (2nc+1)^2 fine nodes written.
 * gs.h:16 prolongation / gscu.h:7 (gs.cpp:228-266, gs.cu:63-81); nc = COARSE n */
int mgb200_prolongation(double *fine, long ldf, const double *coarse, long ldc, long nc,
                        void *stream);

/* u_fine += P(coarse): prolongation fused with the correction add.
 * multigrid.cpp:81-83 (prolongation; u += tmp) / multigrid.cu:85-87 (prolongation; vecadd) */
int mgb200_prolong_correct(double *u_fine, long ldf, const double *coarse, long ldc, long nc,
                           void *stream);

/* c = a + b over the (n+1)^2 nodes.  gscu.h:3 vecadd(x,y,z,len) computes x = y + z (gs.cu:7-11):
 * it maps to mgb200_vecadd(x, y, z, ...) -- output first in both */
int mgb200_vecadd(double *c, const double *a, const double *b, long n, long ld, void *stream);

/* Initial conditions of the reference main (multigrid.cpp:206-233; NOT the buggy gs.cu:221-241):
 * Gaussian u0 with the boundary lines zeroed, vortex velocity scaled by vscale. */
int mgb200_initial_conditions(double *u0, double *v1, double *v2, long n, long ld, double vscale,
                              void *stream);
/* the same for rows row_lo..row_hi only: the arrays hold just those rows (row row_lo at offset 0) */
int mgb200_initial_conditions_rows(double *u0, double *v1, double *v2, long n, long ld, double vscale,
                                   long row_lo, long row_hi, void *stream);

/* ------------------------------------------------------------------------------------------
 * Solver handle: the V/W-cycle driver.  Replaces mg_inner / mg_outer / timestepper
 * (multigrid.cpp:17-186, multigrid.cu:17-200).  The handle owns the level towers, in an
 * internal colour-split padded layout; user fields are copied in and out.
 * ------------------------------------------------------------------------------------------ */
typedef struct mgb200_solver mgb200_solver;

typedef struct mgb200_options {
    int    struct_size;     /* = sizeof(mgb200_options), set by mgb200_default_options */
    int    shape;           /* 1 = V-cycle, 2 = W-cycle (multigrid.cpp:35,52); default 1 */
    int    niter;           /* pre- and post-smoothing RB-GS iterations (NITER, multigrid.cpp:41); 3 */
    int    coarse_maxit;    /* coarsest-level iteration cap (multigrid.cpp:60); 1000 */
    double coarse_tol;      /* coarsest-level ABSOLUTE residual tolerance (multigrid.cpp:60); 1e-5 */
    int    max_cycle;       /* MAX_CYCLE (multigrid.cpp:94); 50 */
    int    arith;           /* MGB200_ARITH_*; default FAST */
    int    plan;            /* MGB200_PLAN_*; default FUSED */
    int    correct_towers;  /* 0 = reproduce the reference's coarse-velocity tower (multigrid.cpp:148-160,
                               SURVEY.md 8/P1); 1 = true injection of the velocities.  default 0 */
    int    use_graph;       /* capture one cycle into a CUDA graph and replay it; default 1 */
    int    device;          /* CUDA device ordinal, -1 = current; default -1 */
    int    restriction;     /* MGB200_RESTRICT_*.  0 = injection of the residual (the reference, gs.cpp:283); 1 = full
                               weighting (gs.cpp:277-280, commented out there), UNFUSED plan only; 2 = the same full
                               weighting on either plan (FUSED: inside the down-leg streaming pass; sharded handles
                               too).  Opt-in: it converges in fewer cycles at large diffusion numbers but leaves
                               the reference's cycle-for-cycle parity; default 0 */
    int    coarse_exact;    /* 0 = coarsest level by iterated RB-GS (the reference, multigrid.cpp:55-65); 1 = direct
                               solve by a banded LU factorisation without pivoting of the (n-1)^2 interior system
                               (what exact_solve.cpp:1-55 set out to do with dgbtrf/dgbtrs; the matrix is strictly
                               diagonally dominant, so partial pivoting would not exchange rows).  Opt-in; default 0 */
    int    reserved[6];
} mgb200_options;

typedef struct mgb200_solve_info {
    int    cycles;          /* V/W-cycles executed by the last solve */
    int    converged;       /* res/res0 <= tol reached */
    double res0;            /* residual norm before the first cycle */
    double res;             /* residual norm after the last cycle */
    double hist[52];        /* hist[0] = res0, hist[k] = norm after cycle k */
} mgb200_solve_info;

void mgb200_default_options(mgb200_options *opt);

/* n: finest grid (power of two >= 32); maxlvl: number of levels (multigrid.cpp:193 uses
 * int(log2 n) - 4, coarsest n = 32); nu, dt, dx, tol: as timestepper's arguments. */
int mgb200_create(mgb200_solver **out, long n, int maxlvl, double nu, double dt, double dx,
                  double tol, const mgb200_options *opt);
int mgb200_destroy(mgb200_solver *s);

/* ------------------------------------------------------------------------------------------
 * Batched handle: `batch` >= 1 independent problems ("members") of one grid size advanced by the same
 * kernel launches (no reference counterpart).  All members share n, maxlvl, nu, dt, dx, tol and the
 * options; each has its own u0, v1, v2, coarse towers and cycle count.  In solve / timestep every
 * member runs mg_outer's loop on its own and is frozen once its condition fails (its fields stay as a
 * handle of that problem alone would leave them); the cycles go on while any member runs.  A member's
 * u on every level, cycle counts and converged flags equal those of a single-problem handle bit for
 * bit; its norms may differ from one in the last bits for batch >= 2 (the per-tile partial sums follow
 * the batch's tiling).  Fused plan with niter >= 1 only (MGB200_ERR_INVALID otherwise), at most 65535
 * members.  The calls of the single-problem handle take or return `batch` consecutive items:
 *   set_fields_host / set_fields_device / get_u_*: member b at + b*(n+1)*ld doubles (ld = n+1 on the host);
 *   get_level_host: batch dense (n_l+1)^2 arrays;  set_fields_reference_ic: the same fields for every member;
 *   form_rhs, cycle, last_norm: batch norms;  cycle / cycle_async: every member cycles;
 *   solve: batch infos;  timestep: nsteps x batch infos, step-major (infos[k*batch + b]).
 * cycle_bytes and profile_level0 count every member.
 * ------------------------------------------------------------------------------------------ */
int mgb200_create_batched(mgb200_solver **out, long n, int maxlvl, int batch, double nu, double dt,
                          double dx, double tol, const mgb200_options *opt);
/* members of the handle: `batch` for a batched handle, 1 for every other */
int mgb200_batch_size(mgb200_solver *s);

/* ------------------------------------------------------------------------------------------
 * Row-slab sharding over the GPUs of one node, one process per GPU (no reference counterpart: the
 * reference is single-GPU; SURVEY.md section 8e).  Rank 0 calls mgb200_comm_unique_id and the host
 * program broadcasts the 128 bytes (bench.py uses torch.distributed); every rank then calls
 * mgb200_create_sharded on its own device.  Fine levels are cut into row slabs at even rows (own
 * rows + 8 halo rows exchanged with the slab neighbours after every streaming pass); levels with
 * fewer than shard_min_rows rows per rank (0 = default 256) run whole on rank 0, fed by a gather of
 * the restricted residual and followed by a scatter of the correction; the residual norm is summed
 * over the ranks.  All of these transfers are stores into the peers' memory (CUDA IPC over NVLink)
 * synchronised by device-side counters; NCCL bootstraps (one all-gather of the IPC handles) and is
 * the fallback transport (environment MGB200_P2P=0).  One rank per GPU: ranks of one communicator
 * must not share a device.  The handle is then used like a single-GPU one: set_fields_* take the
 * FULL-SIZE arrays on every rank (each rank keeps its window), get_u_* fill only the rows the rank
 * owns; form_rhs / cycle / solve / timestep are collective.  Fused plan only.
 * ------------------------------------------------------------------------------------------ */
int mgb200_comm_unique_id(unsigned char id[128]);
int mgb200_create_sharded(mgb200_solver **out, long n, int maxlvl, double nu, double dt, double dx,
                          double tol, const mgb200_options *opt, int rank, int nranks,
                          const unsigned char id[128], long shard_min_rows);
/* the handle's row window at a level: out = {sharded, present, own_lo, own_hi, mem_lo, mem_hi} */
int mgb200_slab(mgb200_solver *s, int lvl, long out[6]);
/* the same rule as pure arithmetic (no GPU needed): window of `rank` of `nranks` at level lvl */
int mgb200_slab_plan(long n, int maxlvl, int nranks, int rank, long shard_min_rows, int lvl, long out[6]);

/* copy u0, v1, v2 in (dense (n+1)^2 DEVICE arrays, row stride ld) and build the level towers
 * (timestepper prologue, multigrid.cpp:138-160) */
int mgb200_set_fields_device(mgb200_solver *s, const double *u0, const double *v1,
                             const double *v2, long ld);
/* same from HOST arrays (dense, ld = n+1); pinned memory makes the copies asynchronous */
int mgb200_set_fields_host(mgb200_solver *s, const double *u0, const double *v1, const double *v2);
/* generate the reference initial conditions directly on the device (multigrid.cpp:206-233) */
int mgb200_set_fields_reference_ic(mgb200_solver *s, double vscale);

/* rhs_0 = B u_0 and the initial residual norm (multigrid.cpp:167 + :104-105) */
int mgb200_form_rhs(mgb200_solver *s, double *res0);
/* one cycle + convergence check: mg_inner(lvl 0) ; residual ; compute_norm (multigrid.cpp:110-113).
 * Synchronous: *res receives the new residual norm. */
int mgb200_cycle(mgb200_solver *s, double *res);
/* asynchronous variant (no host read-back): the norm stays on the device until mgb200_last_norm */
int mgb200_cycle_async(mgb200_solver *s);
int mgb200_last_norm(mgb200_solver *s, double *res);
/* mg_outer (multigrid.cpp:97-120) for the current rhs.  With options.use_graph the loop itself runs
 * on the device (one CUDA graph: k_loop_begin -> WHILE { cycle ; k_loop_check }), the host reads the
 * loop state once afterwards.  Environment MGB200_DEVICE_LOOP=0 keeps the loop on the host (one
 * 8-byte read-back per cycle; needed under Nsight Compute). */
int mgb200_solve(mgb200_solver *s, mgb200_solve_info *info);
/* nsteps x { compute_rhs ; mg_outer } (multigrid.cpp:165-172).  infos may be NULL, else nsteps
 * entries.  All steps are enqueued back to back; the host synchronises once at the end. */
int mgb200_timestep(mgb200_solver *s, int nsteps, mgb200_solve_info *infos);

/* copy u_0 out: dense DEVICE array with row stride ld / dense HOST array (multigrid.cpp:175) */
int mgb200_get_u_device(mgb200_solver *s, double *u, long ld);
int mgb200_get_u_host(mgb200_solver *s, double *u);
/* any level array to a dense HOST array of (n_l+1)^2 doubles, for tests.
 * which: 0 = u, 1 = rhs, 2 = v1, 3 = v2 */
int mgb200_get_level_host(mgb200_solver *s, int lvl, int which, double *out);
int mgb200_synchronize(mgb200_solver *s);
/* the stream all of the handle's work runs on (cudaStream_t as void*) */
void *mgb200_stream(mgb200_solver *s);
/* kernels launched by this handle since creation (graph replays count their kernel nodes) */
long mgb200_kernel_launches(mgb200_solver *s);
/* algorithmic HBM bytes of one cycle + convergence check under the handle's pass plan
 * (DESIGN.md "bytes model"): 8 B per node per level-sized array read or written per pass */
double mgb200_cycle_bytes(mgb200_solver *s);

/* Measurement aid for bench.py (the roofline of the dominant kernel): launches the level-0
 * kernels of the handle's plan `reps` times, each launch bracketed by CUDA events on the handle's
 * stream, and reports the average duration and the algorithmic bytes of ONE launch.
 *   FUSED  : a = down-leg pass {niter RB iterations + residual + injection (full weighting with
 *            options.restriction = 2)},
 *            b = up-leg pass {prolong + correct + niter RB iterations + residual norm}
 *   UNFUSED: a = one colour half-sweep, b = residual
 * The iterate of level 0 keeps being smoothed; call it after the timed region. */
int mgb200_profile_level0(mgb200_solver *s, int reps, double *ms_a, double *bytes_a, double *ms_b,
                          double *bytes_b);

/* ------------------------------------------------------------------------------------------
 * One-call drivers with the reference's own argument list
 * (timestepper: multigrid.cpp:124-126 host pointers; multigrid.cu:130-132 device pointers).
 * T/dt steps are taken exactly as (int)(T/dt) (multigrid.cpp:165).  opt may be NULL.
 * ------------------------------------------------------------------------------------------ */
int mgb200_timestepper_host(double *uT, const double *u0, const double *v1, const double *v2,
                            double nu, int maxlvl, int n, double dt, double T, double dx,
                            double tol, int shape, const mgb200_options *opt,
                            mgb200_solve_info *last);
int mgb200_timestepper_device(double *uT, const double *u0, const double *v1, const double *v2,
                              double nu, int maxlvl, int n, double dt, double T, double dx,
                              double tol, int shape, const mgb200_options *opt,
                              mgb200_solve_info *last);
/* ------------------------------------------------------------------------------------------
 * mg_inner / mg_outer with the reference's own argument lists on CALLER-OWNED towers
 * (multigrid.cpp:17-21, 97-99 = multigrid.cu:17-21, 101-103): u, rhs, v1, v2 are HOST arrays of maxlvl
 * DEVICE pointers; level l is a dense (n_l+1)^2 array with row stride n_l+1 (n_l = n_0 / 2^l, whatever the
 * size of its allocation: the reference gives every coarse level (N/2+1)^2 doubles); tmp is one device array
 * of (n+1)^2 doubles re-used on every level with that level's stride (multigrid.cpp:162).  The cycle runs
 * operator by operator in the reference's order on those arrays; opt (may be NULL) supplies niter,
 * coarse_maxit, coarse_tol, max_cycle and arith -- the literals of multigrid.cpp:41,60,94 by default.
 * mg_outer returns the history in *info (may be NULL) and warns on stderr like multigrid.cpp:117-119 when
 * the tolerance was not met (MGB200_QUIET=1 silences it).  Both synchronise `stream` (the coarsest-level loop
 * and the cycle loop test a norm on the host, as the reference does).
 * ------------------------------------------------------------------------------------------ */
int mgb200_mg_inner(double **u, double **rhs, double **v1, double **v2, double *tmp, double dx, int n,
                    int lvl, int maxlvl, int shape, double dt, double nu, const mgb200_options *opt,
                    void *stream);
int mgb200_mg_outer(double **utow, double **v1tow, double **v2tow, double **rhstow, double *tmp,
                    double nu, int maxlvl, int n, double dt, double dx, double tol, int shape,
                    const mgb200_options *opt, void *stream, mgb200_solve_info *info);

/* ------------------------------------------------------------------------------------------
 * The gs.h operators on HOST pointers with gs.h's argument lists (gs.h:3-17; ld = n+1): each call
 * copies its operands to the device, runs the operator above and copies the result back.  For
 * operator-level drop-in and tests (include/compat/gs.h builds the reference's unmodified
 * multigrid.cpp on them); a time loop should use the handle API, which keeps the fields in HBM.
 * ------------------------------------------------------------------------------------------ */
int mgb200_host_residual(double *res, const double *u, const double *rhs, long n, const double *v1,
                         const double *v2, double k, double nu, double h, int arith);
int mgb200_host_compute_norm(const double *res, long n, double *out);
int mgb200_host_gauss_seidel(double *u, const double *rhs, long n, const double *v1, const double *v2,
                             double k, double nu, double h, int iters, int arith);
int mgb200_host_compute_rhs(double *rhs, const double *u, long n, const double *v1, const double *v2,
                            double k, double nu, double h, int arith);
int mgb200_host_prolongation(double *up, const double *u, int n);   /* n = COARSE n (gs.h:16) */
int mgb200_host_restriction(double *u, const double *up, int n);    /* n = FINE n   (gs.h:17) */

/* The one-call drivers keep their last handle (the level towers in HBM) alive and reuse it when
 * the next call has the same shape and parameters; this frees it.  MGB200_TIMESTEPPER_CACHE=0 in the
 * environment makes the drivers free everything on return, like multigrid.cpp:177-185. */
int mgb200_release_cached(void);

#ifdef __cplusplus
}
#endif
#endif /* MGB200_H */
