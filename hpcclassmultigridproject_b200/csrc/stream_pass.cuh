// stream_pass.cuh -- interface of the fused streaming kernel (definition: syst_pass.cu, per-thread logic:
// syst_pass_body.cuh).
//
// One launch = one "pass" over one level in the solver's split layout:
//     [u += P(coarse u)]  ->  K red-black Gauss-Seidel iterations  ->  [residual epilogue]
// read once from HBM, written once (out-of-place: in != out, so tiles never see each other's
// results), the whole chain staged through shared memory by bulk (TMA) copies.
#pragma once
#include "common.cuh"

namespace mgb200 {

enum StreamPost {
    POST_NONE = 0,
    POST_INJECT = 1,   // coarse_rhs[I][J] = residual(2I,2J) on the coarse interior (residual ; restriction)
    POST_NORM2 = 2,    // sum of squares of the residual over the interior -> partials (residual ; compute_norm)
    POST_FW = 3        // coarse_rhs[I][J] = full weighting of the residual on the coarse interior (residual ;
                       // restriction_fw); down leg only (no prolongation in the same pass)
};

struct StreamPassArgs {
    long n;                 // this level's n (even)
    Layout L;               // split layout of this level
    Stencil st;
    const double* u_in;     // may be null: u is identically zero on entry (fresh coarse level)
    double* u_out;          // != u_in
    const double* rhs;
    const double* v1;
    const double* v2;
    int iters;              // K in [1,3]
    // optional prologue: u += P(coarse)
    const double* coarse_u; // null = none
    Layout Lc;              // layout of the (n/2) level
    // optional epilogue
    int post;               // StreamPost
    double* coarse_rhs;     // POST_INJECT / POST_FW target (layout Lc)
    double* partials;       // POST_NORM2: one double per tile, stream_pass_tiles() entries
    int arith;
    // row window (row-slab sharding).  rows_mem == 0 means "whole level": rows 0..n owned and held.
    long own_lo, own_hi;    // rows to produce
    long row0, rows_mem;    // fine arrays hold global rows row0 .. row0+rows_mem-1
    long crow0, crows_mem;  // same for the coarse arrays
    // Halo push fused into the pass (row slabs over NVLink peer memory; all null / 0 otherwise).  The pass stores
    // the first / last `push_rows` rows it produces (and the matching rows of the coarse rhs of a POST_INJECT / POST_FW
    // pass whose child level is sharded too) straight into the slab neighbours' halo rows, raises their arrival
    // counters when it ends and, at its start, lets only the tiles that stage halo rows wait for the
    // neighbours' previous pass.  peer_*: the neighbours' copies of u_out / coarse_rhs, addressed like ours
    // (pointer to THEIR memory row of global row 0, i.e. base - row0 * pitch); sync: this rank's counter block
    // (comm.cuh); raise_*: the neighbours' arrival counters.
    double* peer_u_up; double* peer_u_dn;
    double* peer_c_up; double* peer_c_dn;
    long push_rows;         // halo depth (rows), fine and coarse
    long c_own_lo, c_own_hi;   // coarse rows this rank owns (for the coarse-rhs push)
    int* sync;
    int* raise_up; int* raise_dn;
    // Batched pass (single GPU, whole levels): members >= 1 problems of this size in one launch (0: one problem, the
    // plain kernel).  Member b of u_in / u_out / rhs / v1 / v2 starts b * mstride doubles after the first, of
    // coarse_u / coarse_rhs b * cmstride after, its partial sums at partials + b * pstride.  active[b] == 0: member b
    // is frozen, the pass leaves everything of it untouched.
    int members;
    long mstride, cmstride, pstride;
    const int* active;
};

// number of tiles (= partial sums written by POST_NORM2) of a pass over level n with `iters`
// fused iterations; iters < 1: the maximum over all iteration counts (buffer sizing).  members: the pass's
// StreamPassArgs::members (the count is per member)
long stream_pass_tiles(long n, long nrows, int iters, int members = 0);
// most members a batched pass takes (gridDim.y)
constexpr int STREAM_PASS_MAX_MEMBERS = 65535;
// one-time attribute setup
int stream_pass_init();
int stream_pass(const StreamPassArgs& a, cudaStream_t s);

}  // namespace mgb200
