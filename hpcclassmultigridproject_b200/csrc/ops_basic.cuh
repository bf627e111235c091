// ops_basic.cuh -- one-operator-per-launch kernels (the reference's operator granularity),
// layout-generic.  They back the C-ABI operator entry points (natural layout) and the solver's
// UNFUSED plan (split layout), and serve as the on-device cross-check of the fused streaming
// kernels.  Declarations only; definitions in ops_basic.cu.
#pragma once
#include "common.cuh"

namespace mgb200 {

// one-time kernel attribute setup (dynamic shared memory opt-in); safe to call repeatedly
int ops_basic_init();

// one colour of RB-GS in place: nodes with (i+j)%2 == colour      (gs.cpp:121-184, gs.cu:307-376)
int launch_gs_colour(double* u, const double* rhs, const double* v1, const double* v2, long n, Layout L,
                     const Stencil& st, int colour, int arith, cudaStream_t s);
// res = rhs - A u (interior).  res may be null.  If partials != null the squares of the residual
// are block-summed into partials[0..nblocks) (use residual_partials_count) -- gs.cpp:55-107
int launch_residual(double* res, const double* u, const double* rhs, const double* v1, const double* v2,
                    long n, Layout L, const Stencil& st, int arith, double* partials, cudaStream_t s);
long residual_partials_count(long n);
// rhs = B u (interior); if partials != null also the squares of (rhs - A u)  -- gs.cpp:24-53
// row_lo/row_hi (optional) restrict the rows produced (row slabs); partials then has
// rows_partials_count(n, rows) entries
int launch_compute_rhs(double* rhs, const double* u, const double* v1, const double* v2, long n, Layout L,
                       const Stencil& st, int arith, double* partials, cudaStream_t s, long row_lo = 1, long row_hi = -1);
long rows_partials_count(long n, long nrows);
// entries launch_compute_rhs writes into `partials` for a band of nrows rows in layout L
long compute_rhs_partials_count(long n, long nrows, Layout L);
// sum of squares over the interior of a -> partials (same count as residual_partials_count)
int launch_square_partials(const double* a, long n, Layout L, double* partials, cudaStream_t s);
// out[0] = sum(partials[0..count)) in a fixed order (single block)
int launch_reduce_partials(const double* partials, long count, double* out, cudaStream_t s);
// coarse[I][J] = fine[2I][2J], I,J in [0,nf/2]                     -- gs.cpp:268-292
int launch_restrict(double* coarse, Layout Lc, const double* fine, Layout Lf, long nf, cudaStream_t s);
// interior-only injection (coarse boundary left untouched)
int launch_restrict_interior(double* coarse, Layout Lc, const double* fine, Layout Lf, long nf, cudaStream_t s);
// fine = P(coarse) (add=false) or fine += P(coarse) (add=true)      -- gs.cpp:228-266, multigrid.cpp:83
// full weighting of gs.cpp:277-280 (commented out in the reference; opt-in): interior stencil, injected boundary
int launch_restrict_fw(double* coarse, Layout Lc, const double* fine, Layout Lf, long nf, bool interior_only, cudaStream_t s);
int launch_prolong(double* fine, Layout Lf, const double* coarse, Layout Lc, long nc, bool add, cudaStream_t s);
int launch_vecadd(double* c, const double* a, const double* b, long n, Layout L, cudaStream_t s);
// dst(layout Ld) = src(layout Ls) over the (n+1)^2 nodes
int launch_convert(double* dst, Layout Ld, const double* src, Layout Ls, long n, cudaStream_t s, long row_lo = 0, long row_hi = -1);
// reference ICs (multigrid.cpp:206-233), velocity times vscale
int launch_initial_conditions(double* u0, double* v1, double* v2, long n, Layout L, double vscale, cudaStream_t s,
                              long row_lo = 0, long row_hi = -1);
// coarse velocity towers, reference-compatible (multigrid.cpp:148-160, SURVEY.md 8/P1):
//   flat_out[i*(q+1)+j] = src_flat[2i*(h+1)+2j], i,j in [0,q], q = N/4, h = N/2,
// where src_flat is either the dense level-0 field read through (layout, N) [from_level0] or a
// previous flat buffer.  flat buffers hold (h+1)^2 doubles and must be zero-filled beforehand.
int launch_tower_flat(double* flat_out, const double* src, bool from_level0, Layout L0, long N, cudaStream_t s);
// level array (split layout, n_l) = flat[i*(n_l+1)+j]
int launch_flat_to_level(double* dst, Layout Ld, const double* flat, long nl, cudaStream_t s, long row_lo = 0, long row_hi = -1);
// coarsest level solved on the device by ONE thread block: u = 0 (if zero_init); repeat
// { RB-GS ; residual ; norm } until norm <= tol or maxit  (multigrid.cpp:55-65).  n <= 64.
// iters_out (device int, may be null) receives the iteration count.
int launch_coarse_solve(double* u, const double* rhs, const double* v1, const double* v2, long n, Layout L,
                        const Stencil& st, int arith, bool zero_init, int maxit, double tol, int* iters_out,
                        cudaStream_t s);

// opt-in direct coarsest-level solve (exact_solve.cpp:1-55): banded LU without pivoting of the (n-1)^2 interior
// system in `ab` (coarse_lu_bytes(n) bytes of device memory), factor once per set of velocities, solve per visit
size_t coarse_lu_bytes(long n);
int launch_coarse_lu_factor(double* ab, const double* v1, const double* v2, long n, Layout L, const Stencil& st, cudaStream_t s);
int launch_coarse_lu_solve(double* u, const double* rhs, const double* v1, const double* v2, const double* ab, long n, Layout L,
                           const Stencil& st, bool zero_init, cudaStream_t s);

// Batched solver handles: `members` problems of one size, member b of every field at + b * mstride.
// rhs = B u and the sum of squares of the initial residual of every member (partials of member b at
// + b * pstride: compute_rhs_partials_count(n, n - 1, L) each)
int launch_compute_rhs_batched(double* rhs, const double* u, const double* v1, const double* v2, long n, Layout L,
                               const Stencil& st, int arith, double* partials, long pstride, int members, long mstride,
                               cudaStream_t s);
// out[b] = sum of member b's `count` partials (in launch_reduce_partials' order) for every member with active[b] != 0
// (active == NULL: every member)
int launch_reduce_partials_batched(const double* partials, long count, long pstride, double* out, const int* active, int members,
                                   cudaStream_t s);
// the coarsest-level solves of the active members, one block each (iters_out[b], factors of member b at + b * abstride)
int launch_coarse_solve_batched(double* u, const double* rhs, const double* v1, const double* v2, long n, Layout L,
                                const Stencil& st, int arith, bool zero_init, int maxit, double tol, int* iters_out,
                                int members, long mstride, const int* active, cudaStream_t s);
int launch_coarse_lu_solve_batched(double* u, const double* rhs, const double* v1, const double* v2, const double* ab, long n,
                                   Layout L, const Stencil& st, bool zero_init, int members, long mstride, long abstride,
                                   const int* active, cudaStream_t s);

}  // namespace mgb200
