// ops_basic.cu -- one-operator-per-launch kernels, layout-generic (see ops_basic.cuh).
//
// Thread mapping: threadIdx.x runs along the contiguous (column) index, a block covers
// ROWS_PER_BLOCK rows x 256 columns; blockIdx.x indexes row groups (no 65535 limit), blockIdx.y
// column chunks.  Every global access of a warp is a unit-stride run (split layout: one run
// per parity).
#include <mutex>

#include "ops_basic.cuh"

namespace mgb200 {

namespace {

constexpr int TPB = 256;
constexpr int ROWS_PER_BLOCK = 8;

inline dim3 tile_grid(long rows, long cols)
{
    return dim3((unsigned)((rows + ROWS_PER_BLOCK - 1) / ROWS_PER_BLOCK), (unsigned)((cols + TPB - 1) / TPB), 1);
}

// ---------------------------------------------------------------------------------------------
template <int ARITH>
__global__ void __launch_bounds__(TPB) k_gs_colour(double* __restrict__ u, const double* __restrict__ rhs,
                                                   const double* __restrict__ v1, const double* __restrict__ v2,
                                                   long n, Layout L, Stencil st, int colour)
{
    const long k = (long)blockIdx.y * TPB + threadIdx.x;
    const long i0 = 1 + (long)blockIdx.x * ROWS_PER_BLOCK;
#pragma unroll 2
    for (int r = 0; r < ROWS_PER_BLOCK; ++r) {
        const long i = i0 + r;
        if (i >= n) break;
        const long p = (i + colour) & 1;      // column parity of this colour in row i
        const long j = 2 * k + 2 - p;         // p=1: 1,3,5,...   p=0: 2,4,6,...
        if (j >= n) continue;
        const long q = L.at(i, j);
        const Coef4 c = Arith<ARITH>::coef(v1[q], v2[q], st);
        u[q] = Arith<ARITH>::gs(rhs[q], u[L.at(i - 1, j)], u[L.at(i, j - 1)], u[L.at(i + 1, j)],
                                u[L.at(i, j + 1)], c, st);
    }
}

// MODE bit0: write res, bit1: accumulate squares into partials
template <int ARITH, int MODE>
__global__ void __launch_bounds__(TPB) k_residual(double* __restrict__ res, const double* __restrict__ u,
                                                  const double* __restrict__ rhs, const double* __restrict__ v1,
                                                  const double* __restrict__ v2, long n, Layout L, Stencil st,
                                                  double* __restrict__ partials)
{
    __shared__ double scratch[32];
    const long j = 1 + (long)blockIdx.y * TPB + threadIdx.x;
    const long i0 = 1 + (long)blockIdx.x * ROWS_PER_BLOCK;
    double acc = 0.0;
    for (int r = 0; r < ROWS_PER_BLOCK; ++r) {
        const long i = i0 + r;
        if (i >= n || j >= n) break;
        const long q = L.at(i, j);
        const Coef4 c = Arith<ARITH>::coef(v1[q], v2[q], st);
        const double rv = Arith<ARITH>::residual(rhs[q], u[q], u[L.at(i - 1, j)], u[L.at(i, j - 1)],
                                                 u[L.at(i + 1, j)], u[L.at(i, j + 1)], c, st);
        if (MODE & 1) res[q] = rv;
        if (MODE & 2) acc += rv * rv;
    }
    if (MODE & 2) {
        const double t = block_sum(acc, scratch);
        if (threadIdx.x == 0) partials[(long)blockIdx.x * gridDim.y + blockIdx.y] = t;
    }
}

template <int ARITH, bool WITH_RES0>
__global__ void __launch_bounds__(TPB) k_compute_rhs(double* __restrict__ rhs, const double* __restrict__ u,
                                                     const double* __restrict__ v1, const double* __restrict__ v2,
                                                     long n, Layout L, Stencil st, double* __restrict__ partials,
                                                     long ilo, long ihi)
{
    __shared__ double scratch[32];
    const long j = 1 + (long)blockIdx.y * TPB + threadIdx.x;
    const long i0 = ilo + (long)blockIdx.x * ROWS_PER_BLOCK;
    double acc = 0.0;
    for (int r = 0; r < ROWS_PER_BLOCK; ++r) {
        const long i = i0 + r;
        if (i > ihi || j >= n) break;
        const long q = L.at(i, j);
        const Coef4 c = Arith<ARITH>::coef(v1[q], v2[q], st);
        const double uc = u[q], up = u[L.at(i - 1, j)], lf = u[L.at(i, j - 1)], dn = u[L.at(i + 1, j)],
                     rt = u[L.at(i, j + 1)];
        const double f = Arith<ARITH>::rhs(uc, up, lf, dn, rt, c, st);
        rhs[q] = f;
        if (WITH_RES0) {
            const double rv = Arith<ARITH>::residual(f, uc, up, lf, dn, rt, c, st);
            acc += rv * rv;
        }
    }
    if (WITH_RES0) {
        const double t = block_sum(acc, scratch);
        if (threadIdx.x == 0) partials[(long)blockIdx.x * gridDim.y + blockIdx.y] = t;
    }
}

// compute_rhs for the colour-split layout (the solver's own arrays): one thread owns two column
// pairs (four nodes: even columns 2k, 2k+2 in the E run, odd columns 2k+1, 2k+3 in the O run) and
// walks down a band of rows with the three rows of u it needs in registers.  Every global access
// is a 16-byte vector, u is read once (plus two halo rows per band), horizontal neighbours across
// lanes come from shuffles.  Same operands in the same order as k_compute_rhs: identical rhs.
constexpr int RHS_TPB = 128, RHS_ROWS = 32;
template <int ARITH, bool WITH_RES0>
__device__ __forceinline__ void compute_rhs_split_body(double* __restrict__ rhs, const double* __restrict__ u,
                                                       const double* __restrict__ v1, const double* __restrict__ v2,
                                                       long n, Layout L, Stencil st, double* __restrict__ partials,
                                                       long ilo, long ihi)
{
    __shared__ double scratch[32];
    const int lane = threadIdx.x & 31;
    const long k = 2 * ((long)blockIdx.x * RHS_TPB + threadIdx.x);      // first of the thread's two pairs
    const long r0 = ilo + (long)blockIdx.y * RHS_ROWS;
    const long r1 = r0 + RHS_ROWS - 1 < ihi ? r0 + RHS_ROWS - 1 : ihi;
    const long nh = n / 2;                                               // E run: k = 0..nh, O run: k = 0..nh-1
    const bool live = k <= nh;                                           // (the layout's slack covers k+1)
    // interior columns 1..n-1
    const bool okE0 = live && k >= 1 && 2 * k <= n - 1, okE1 = live && 2 * (k + 1) <= n - 1;
    const bool okO0 = live && 2 * k + 1 <= n - 1, okO1 = live && 2 * k + 3 <= n - 1;
    auto ldE = [&](const double* a, long i) { return live ? *reinterpret_cast<const double2*>(a + (i - L.row0) * L.pitch + k) : make_double2(0.0, 0.0); };
    auto ldO = [&](const double* a, long i) { return live ? *reinterpret_cast<const double2*>(a + (i - L.row0) * L.pitch + L.odd + k) : make_double2(0.0, 0.0); };
    double acc = 0.0;
    double2 upE = ldE(u, r0 - 1), upO = ldO(u, r0 - 1), cE = ldE(u, r0), cO = ldO(u, r0);
    for (long i = r0; i <= r1; ++i) {
        const double2 dnE = ldE(u, i + 1), dnO = ldO(u, i + 1);
        const double2 aE = ldE(v1, i), aO = ldO(v1, i), bE = ldE(v2, i), bO = ldO(v2, i);
        // E[k]'s left neighbour is O[k-1] (previous lane's cO.y), O[k+1]'s right one is E[k+2] (next lane's cE.x)
        double lfE = __shfl_up_sync(0xffffffffu, cO.y, 1), rtO = __shfl_down_sync(0xffffffffu, cE.x, 1);
        if (lane == 0 && okE0) lfE = u[(i - L.row0) * L.pitch + L.odd + k - 1];
        if (lane == 31 && okO1) rtO = u[(i - L.row0) * L.pitch + k + 2];
        const Coef4 kE0 = Arith<ARITH>::coef(aE.x, bE.x, st), kE1 = Arith<ARITH>::coef(aE.y, bE.y, st);
        const Coef4 kO0 = Arith<ARITH>::coef(aO.x, bO.x, st), kO1 = Arith<ARITH>::coef(aO.y, bO.y, st);
        const double fE0 = Arith<ARITH>::rhs(cE.x, upE.x, lfE, dnE.x, cO.x, kE0, st);
        const double fE1 = Arith<ARITH>::rhs(cE.y, upE.y, cO.x, dnE.y, cO.y, kE1, st);
        const double fO0 = Arith<ARITH>::rhs(cO.x, upO.x, cE.x, dnO.x, cE.y, kO0, st);
        const double fO1 = Arith<ARITH>::rhs(cO.y, upO.y, cE.y, dnO.y, rtO, kO1, st);
        double* rowp = rhs + (i - L.row0) * L.pitch;
        if (okE0 && okE1) *reinterpret_cast<double2*>(rowp + k) = make_double2(fE0, fE1);
        else { if (okE0) rowp[k] = fE0; if (okE1) rowp[k + 1] = fE1; }
        if (okO0 && okO1) *reinterpret_cast<double2*>(rowp + L.odd + k) = make_double2(fO0, fO1);
        else { if (okO0) rowp[L.odd + k] = fO0; if (okO1) rowp[L.odd + k + 1] = fO1; }
        if (WITH_RES0) {
            // row-major order of the four nodes: columns 2k, 2k+1, 2k+2, 2k+3
            if (okE0) { const double rv = Arith<ARITH>::residual(fE0, cE.x, upE.x, lfE, dnE.x, cO.x, kE0, st); acc += rv * rv; }
            if (okO0) { const double rv = Arith<ARITH>::residual(fO0, cO.x, upO.x, cE.x, dnO.x, cE.y, kO0, st); acc += rv * rv; }
            if (okE1) { const double rv = Arith<ARITH>::residual(fE1, cE.y, upE.y, cO.x, dnE.y, cO.y, kE1, st); acc += rv * rv; }
            if (okO1) { const double rv = Arith<ARITH>::residual(fO1, cO.y, upO.y, cE.y, dnO.y, rtO, kO1, st); acc += rv * rv; }
        }
        upE = cE; upO = cO; cE = dnE; cO = dnO;
    }
    if (WITH_RES0) {
        const double t = block_sum(acc, scratch);
        if (threadIdx.x == 0) partials[(long)blockIdx.y * gridDim.x + blockIdx.x] = t;
    }
}

template <int ARITH, bool WITH_RES0>
__global__ void __launch_bounds__(RHS_TPB) k_compute_rhs_split(double* __restrict__ rhs, const double* __restrict__ u,
                                                               const double* __restrict__ v1, const double* __restrict__ v2,
                                                               long n, Layout L, Stencil st, double* __restrict__ partials,
                                                               long ilo, long ihi)
{
    compute_rhs_split_body<ARITH, WITH_RES0>(rhs, u, v1, v2, n, L, st, partials, ilo, ihi);
}

// a batch of problems (batched solver handles): member blockIdx.z at + blockIdx.z * mstride in every field, its
// partial sums at + blockIdx.z * pstride, each member's in the order of k_compute_rhs_split
template <int ARITH>
__global__ void __launch_bounds__(RHS_TPB) k_compute_rhs_split_batched(double* __restrict__ rhs, const double* __restrict__ u,
                                                                       const double* __restrict__ v1, const double* __restrict__ v2,
                                                                       long n, Layout L, Stencil st, double* __restrict__ partials,
                                                                       long ilo, long ihi, long mstride, long pstride)
{
    const long mo = (long)blockIdx.z * mstride;
    compute_rhs_split_body<ARITH, true>(rhs + mo, u + mo, v1 + mo, v2 + mo, n, L, st, partials + (long)blockIdx.z * pstride, ilo, ihi);
}

__global__ void __launch_bounds__(TPB) k_square_partials(const double* __restrict__ a, long n, Layout L,
                                                         double* __restrict__ partials)
{
    __shared__ double scratch[32];
    const long j = 1 + (long)blockIdx.y * TPB + threadIdx.x;
    const long i0 = 1 + (long)blockIdx.x * ROWS_PER_BLOCK;
    double acc = 0.0;
    for (int r = 0; r < ROWS_PER_BLOCK; ++r) {
        const long i = i0 + r;
        if (i >= n || j >= n) break;
        const double x = a[L.at(i, j)];
        acc += x * x;
    }
    const double t = block_sum(acc, scratch);
    if (threadIdx.x == 0) partials[(long)blockIdx.x * gridDim.y + blockIdx.y] = t;
}

__global__ void __launch_bounds__(1024) k_reduce_partials(const double* __restrict__ partials, long count,
                                                          double* __restrict__ out)
{
    __shared__ double scratch[32];
    double acc = 0.0;
    for (long q = threadIdx.x; q < count; q += 1024) acc += partials[q];
    const double t = block_sum(acc, scratch);
    if (threadIdx.x == 0) out[0] = t;
}

// one block per member, each summing in the order of k_reduce_partials; active == null: every member
__global__ void __launch_bounds__(1024) k_reduce_partials_batched(const double* __restrict__ partials, long count, long pstride,
                                                                  double* __restrict__ out, const int* __restrict__ active)
{
    __shared__ double scratch[32];
    if (active && !active[blockIdx.x]) return;
    const double* part = partials + (long)blockIdx.x * pstride;
    double acc = 0.0;
    for (long q = threadIdx.x; q < count; q += 1024) acc += part[q];
    const double t = block_sum(acc, scratch);
    if (threadIdx.x == 0) out[blockIdx.x] = t;
}

template <bool INTERIOR>
__global__ void __launch_bounds__(TPB) k_restrict(double* __restrict__ coarse, Layout Lc,
                                                  const double* __restrict__ fine, Layout Lf, long nc)
{
    const long lo = INTERIOR ? 1 : 0, hi = INTERIOR ? nc - 1 : nc;
    const long J = lo + (long)blockIdx.y * TPB + threadIdx.x;
    const long I0 = lo + (long)blockIdx.x * ROWS_PER_BLOCK;
    for (int r = 0; r < ROWS_PER_BLOCK; ++r) {
        const long I = I0 + r;
        if (I > hi || J > hi) break;
        coarse[Lc.at(I, J)] = fine[Lf.at(2 * I, 2 * J)];
    }
}

// full weighting as sketched in gs.cpp:277-280 (commented out in the reference; opt-in here):
// [1 2 1; 2 4 2; 1 2 1]/16 on the coarse interior, grouped by fine rows as written there
// (x/16 == x*0.0625 exactly); the boundary is injected.
template <bool INTERIOR>
__global__ void __launch_bounds__(TPB) k_restrict_fw(double* __restrict__ coarse, Layout Lc,
                                                     const double* __restrict__ fine, Layout Lf, long nc)
{
    const long lo = INTERIOR ? 1 : 0, hi = INTERIOR ? nc - 1 : nc;
    const long J = lo + (long)blockIdx.y * TPB + threadIdx.x;
    const long I0 = lo + (long)blockIdx.x * ROWS_PER_BLOCK;
    for (int r = 0; r < ROWS_PER_BLOCK; ++r) {
        const long I = I0 + r;
        if (I > hi || J > hi) break;
        if (I == 0 || J == 0 || I == nc || J == nc) { coarse[Lc.at(I, J)] = fine[Lf.at(2 * I, 2 * J)]; continue; }
        auto row = [&](long i, double w) {
            const double s1 = __dadd_rn(__dmul_rn(w, fine[Lf.at(i, 2 * J - 1)]), __dmul_rn(2.0 * w, fine[Lf.at(i, 2 * J)]));
            return __dmul_rn(__dadd_rn(s1, __dmul_rn(w, fine[Lf.at(i, 2 * J + 1)])), 0.0625);
        };
        double t = row(2 * I - 1, 1.0);
        t = __dadd_rn(t, row(2 * I, 2.0));
        t = __dadd_rn(t, row(2 * I + 1, 1.0));
        coarse[Lc.at(I, J)] = t;
    }
}

template <bool ADD>
__global__ void __launch_bounds__(TPB) k_prolong(double* __restrict__ fine, Layout Lf,
                                                 const double* __restrict__ coarse, Layout Lc, long nc)
{
    const long nf = 2 * nc;
    const long j = (long)blockIdx.y * TPB + threadIdx.x;
    const long i0 = (long)blockIdx.x * ROWS_PER_BLOCK;
    for (int r = 0; r < ROWS_PER_BLOCK; ++r) {
        const long i = i0 + r;
        if (i > nf || j > nf) break;
        const long I = i >> 1, J = j >> 1;
        const double c00 = coarse[Lc.at(I, J)];
        double v;
        if ((i & 1) == 0 && (j & 1) == 0) {
            v = c00;                                                                  // gs.cpp:238
        } else if ((i & 1) == 1 && (j & 1) == 0) {
            v = __dmul_rn(__dadd_rn(c00, coarse[Lc.at(I + 1, J)]), 0.5);            // gs.cpp:239
        } else if ((i & 1) == 0) {
            v = __dmul_rn(__dadd_rn(c00, coarse[Lc.at(I, J + 1)]), 0.5);            // gs.cpp:240
        } else {
            double t = __dadd_rn(c00, coarse[Lc.at(I + 1, J)]);                     // gs.cpp:241
            t = __dadd_rn(t, coarse[Lc.at(I, J + 1)]);
            t = __dadd_rn(t, coarse[Lc.at(I + 1, J + 1)]);
            v = __dmul_rn(t, 0.25);
        }
        const long q = Lf.at(i, j);
        fine[q] = ADD ? __dadd_rn(fine[q], v) : v;                                    // multigrid.cpp:83
    }
}

__global__ void __launch_bounds__(TPB) k_vecadd(double* __restrict__ c, const double* __restrict__ a,
                                                const double* __restrict__ b, long n, Layout L)
{
    const long j = (long)blockIdx.y * TPB + threadIdx.x;
    const long i0 = (long)blockIdx.x * ROWS_PER_BLOCK;
    for (int r = 0; r < ROWS_PER_BLOCK; ++r) {
        const long i = i0 + r;
        if (i > n || j > n) break;
        const long q = L.at(i, j);
        c[q] = __dadd_rn(a[q], b[q]);
    }
}

__global__ void __launch_bounds__(TPB) k_convert(double* __restrict__ dst, Layout Ld, const double* __restrict__ src,
                                                 Layout Ls, long n, long ilo, long ihi)
{
    const long j = (long)blockIdx.y * TPB + threadIdx.x;
    const long i0 = ilo + (long)blockIdx.x * ROWS_PER_BLOCK;
    for (int r = 0; r < ROWS_PER_BLOCK; ++r) {
        const long i = i0 + r;
        if (i > ihi || j > n) break;
        dst[Ld.at(i, j)] = src[Ls.at(i, j)];
    }
}

__global__ void __launch_bounds__(TPB) k_initial_conditions(double* __restrict__ u0, double* __restrict__ v1,
                                                            double* __restrict__ v2, long n, Layout L, double vscale,
                                                            long ilo, long ihi)
{
    const double PI = 3.1415926535897932;                    // multigrid.cpp:14
    const double x0 = 0.2, y0 = 0.4, sigma = 100.0;          // multigrid.cpp:206-207
    const double kx = 1.0 * PI, ky = 1.0 * PI;
    const double dx = 1.0 / (double)n;
    const long j = (long)blockIdx.y * TPB + threadIdx.x;
    const long i0 = ilo + (long)blockIdx.x * ROWS_PER_BLOCK;
    for (int r = 0; r < ROWS_PER_BLOCK; ++r) {
        const long i = i0 + r;
        if (i > ihi || j > n) break;
        const double x = i * dx, y = j * dx;
        double g = exp(-sigma * ((x - x0) * (x - x0) + (y - y0) * (y - y0)));        // multigrid.cpp:219
        // boundary lines zeroed with a loop bound of N: node (N,0) keeps its value (multigrid.cpp:227-233)
        const bool zeroed = (i == 0 && j < n) || (j == n && i < n) || (i == n && j >= 1) || (j == 0 && i < n);
        if (zeroed) g = 0.0;
        const long q = L.at(i, j);
        u0[q] = g;
        v1[q] = (-ky * sin(kx * i * dx) * cos(ky * j * dx)) * vscale;                // multigrid.cpp:222
        v2[q] = (kx * cos(kx * i * dx) * sin(ky * j * dx)) * vscale;                 // multigrid.cpp:223
    }
}

__global__ void __launch_bounds__(TPB) k_tower_flat(double* __restrict__ flat_out, const double* __restrict__ src,
                                                    int from_level0, Layout L0, long N)
{
    const long h = N / 2, q = N / 4;
    const long j = (long)blockIdx.y * TPB + threadIdx.x;
    const long i0 = (long)blockIdx.x * ROWS_PER_BLOCK;
    for (int r = 0; r < ROWS_PER_BLOCK; ++r) {
        const long i = i0 + r;
        if (i > q || j > q) break;
        const long f = 2 * i * (h + 1) + 2 * j;              // flat index into the source (gs.cpp:283, n = N/2)
        double v;
        if (from_level0) v = src[L0.at(f / (N + 1), f % (N + 1))];   // level 0 is a dense (N+1)^2 array
        else v = src[f];
        flat_out[i * (q + 1) + j] = v;
    }
}

__global__ void __launch_bounds__(TPB) k_flat_to_level(double* __restrict__ dst, Layout Ld,
                                                       const double* __restrict__ flat, long nl, long ilo, long ihi)
{
    const long j = (long)blockIdx.y * TPB + threadIdx.x;
    const long i0 = ilo + (long)blockIdx.x * ROWS_PER_BLOCK;
    for (int r = 0; r < ROWS_PER_BLOCK; ++r) {
        const long i = i0 + r;
        if (i > ihi || j > nl) break;
        dst[Ld.at(i, j)] = flat[i * (nl + 1) + j];
    }
}

// ---------------------------------------------------------------------------------------------
// Coarsest level on ONE thread block, all fields staged in shared memory (natural order).
template <int ARITH>
__device__ __forceinline__ void coarse_solve_body(double* __restrict__ u, const double* __restrict__ rhs,
                                                  const double* __restrict__ v1, const double* __restrict__ v2,
                                                  int n, Layout L, Stencil st, int zero_init, int maxit,
                                                  double tol, int* __restrict__ iters_out)
{
    extern __shared__ double sm[];
    __shared__ double scratch[32];
    __shared__ double s_norm2;
    const int ld = n + 1, m = ld * ld;
    double* su = sm;
    double* sf = sm + m;
    double* s1 = sm + 2 * m;
    double* s2 = sm + 3 * m;
    for (int q = threadIdx.x; q < m; q += blockDim.x) {
        const int i = q / ld, j = q % ld;
        const long g = L.at(i, j);
        su[q] = zero_init ? 0.0 : u[g];
        sf[q] = rhs[g];
        s1[q] = v1[g];
        s2[q] = v2[g];
    }
    __syncthreads();
    const int ni = n - 1, npts = ni * ni;
    int it = 0;
    double rn = 1.0;                                                     // multigrid.cpp:58
    while (it < maxit && rn > tol) {                                     // multigrid.cpp:60
        for (int colour = 0; colour < 2; ++colour) {
            for (int p = threadIdx.x; p < npts; p += blockDim.x) {
                const int i = 1 + p / ni, j = 1 + p % ni;
                if (((i + j) & 1) != colour) continue;
                const int q = i * ld + j;
                const Coef4 c = Arith<ARITH>::coef(s1[q], s2[q], st);
                su[q] = Arith<ARITH>::gs(sf[q], su[q - ld], su[q - 1], su[q + ld], su[q + 1], c, st);
            }
            __syncthreads();
        }
        double acc = 0.0;
        for (int p = threadIdx.x; p < npts; p += blockDim.x) {
            const int i = 1 + p / ni, j = 1 + p % ni;
            const int q = i * ld + j;
            const Coef4 c = Arith<ARITH>::coef(s1[q], s2[q], st);
            const double rv = Arith<ARITH>::residual(sf[q], su[q], su[q - ld], su[q - 1], su[q + ld], su[q + 1], c, st);
            acc += rv * rv;
        }
        const double t = block_sum(acc, scratch);
        if (threadIdx.x == 0) s_norm2 = t;
        __syncthreads();
        rn = sqrt(s_norm2);
        ++it;
        __syncthreads();
    }
    for (int p = threadIdx.x; p < npts; p += blockDim.x) {
        const int i = 1 + p / ni, j = 1 + p % ni;
        u[L.at(i, j)] = su[i * ld + j];
    }
    if (zero_init) {   // the boundary of a freshly zeroed level is zero as well (multigrid.cpp:77)
        for (int q = threadIdx.x; q <= n; q += blockDim.x) {
            u[L.at(0, q)] = 0.0; u[L.at(n, q)] = 0.0; u[L.at(q, 0)] = 0.0; u[L.at(q, n)] = 0.0;
        }
    }
    if (threadIdx.x == 0 && iters_out) *iters_out = it;
}

template <int ARITH>
__global__ void __launch_bounds__(1024) k_coarse_solve(double* __restrict__ u, const double* __restrict__ rhs,
                                                       const double* __restrict__ v1, const double* __restrict__ v2,
                                                       int n, Layout L, Stencil st, int zero_init, int maxit,
                                                       double tol, int* __restrict__ iters_out)
{
    coarse_solve_body<ARITH>(u, rhs, v1, v2, n, L, st, zero_init, maxit, tol, iters_out);
}

// one block per member (blockIdx.x, fields mstride apart); a frozen member (active == 0) is left as it is
template <int ARITH>
__global__ void __launch_bounds__(1024) k_coarse_solve_batched(double* __restrict__ u, const double* __restrict__ rhs,
                                                               const double* __restrict__ v1, const double* __restrict__ v2,
                                                               int n, Layout L, Stencil st, int zero_init, int maxit,
                                                               double tol, int* __restrict__ iters_out, long mstride,
                                                               const int* __restrict__ active)
{
    const int b = blockIdx.x;
    if (!active[b]) return;
    const long mo = (long)b * mstride;
    coarse_solve_body<ARITH>(u + mo, rhs + mo, v1 + mo, v2 + mo, n, L, st, zero_init, maxit, tol, iters_out + b);
}

// ---- opt-in direct solve of the coarsest level (the unfinished exact_solve.cpp:1-55 of the reference) -------------
// Unknowns: the (n-1)^2 interior nodes, p = (i-1)(n-1) + (j-1); half bandwidth w = n-1; band storage
// AB[p][w + q - p] for |q - p| <= w (row p of A, (2w+1) doubles per row).  LU without pivoting (A is strictly
// diagonally dominant), multipliers stored in place of the eliminated entries.  One thread block; every
// floating-point operation is a single rounded IEEE operation in a fixed order (k-outer elimination, then the
// two substitutions), so that a plain C statement of the same factorisation reproduces it bit for bit.
__global__ void __launch_bounds__(1024) k_coarse_lu_factor(double* __restrict__ ab, const double* __restrict__ v1,
                                                           const double* __restrict__ v2, int n, Layout L, Stencil st)
{
    const int ni = n - 1, m = ni * ni, w = ni, bw = 2 * w + 1;
    for (long q = threadIdx.x; q < (long)m * bw; q += blockDim.x) ab[q] = 0.0;
    __syncthreads();
    for (int p = threadIdx.x; p < m; p += blockDim.x) {
        const int i = 1 + p / ni, j = 1 + p % ni;
        const long g = L.at(i, j);
        const Coef4 c = Arith<MGB200_ARITH_EXACT>::coef(v1[g], v2[g], st);
        double* row = ab + (long)p * bw + w;
        row[0] = st.diag;
        if (i > 1) row[-ni] = c.c;
        if (i < n - 1) row[ni] = c.d;
        if (j > 1) row[-1] = c.a;
        if (j < n - 1) row[1] = c.b;
    }
    __syncthreads();
    for (int k = 0; k < m - 1; ++k) {
        const int rmax = min(w, m - 1 - k), nel = rmax * (rmax + 1);
        const double pivot = ab[(long)k * bw + w];
        // element e = (r, c) of the trailing update, r in 1..rmax, c in 0..rmax; c == 0 is the multiplier itself.
        // At most 4 elements per thread (n <= 64: 63 * 64 <= 4 * 1024): read everything, barrier, write.
        double val[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int e = (int)threadIdx.x + q * (int)blockDim.x;
            val[q] = 0.0;
            if (e < nel) {
                const int r = 1 + e / (rmax + 1), c = e % (rmax + 1);
                const double l = __ddiv_rn(ab[(long)(k + r) * bw + w - r], pivot);
                val[q] = c ? __dsub_rn(ab[(long)(k + r) * bw + w - r + c], __dmul_rn(l, ab[(long)k * bw + w + c])) : l;
            }
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int e = (int)threadIdx.x + q * (int)blockDim.x;
            if (e < nel) {
                const int r = 1 + e / (rmax + 1), c = e % (rmax + 1);
                ab[(long)(k + r) * bw + w - r + c] = val[q];
            }
        }
        __syncthreads();
    }
}

// u(interior) = A^-1 (rhs - boundary terms): forward substitution with the stored multipliers, back substitution
// with U.  y lives in shared memory.
__device__ __forceinline__ void coarse_lu_solve_body(double* __restrict__ u, const double* __restrict__ rhs,
                                                     const double* __restrict__ v1, const double* __restrict__ v2,
                                                     const double* __restrict__ ab, int n, Layout L, Stencil st, int zero_init)
{
    extern __shared__ double y[];
    const int ni = n - 1, m = ni * ni, w = ni, bw = 2 * w + 1;
    if (zero_init) {   // the boundary of a freshly zeroed level is zero (multigrid.cpp:77)
        for (int q = threadIdx.x; q <= n; q += blockDim.x) { u[L.at(0, q)] = 0.0; u[L.at(n, q)] = 0.0; u[L.at(q, 0)] = 0.0; u[L.at(q, n)] = 0.0; }
        __syncthreads();
    }
    for (int p = threadIdx.x; p < m; p += blockDim.x) {
        const int i = 1 + p / ni, j = 1 + p % ni;
        const long g = L.at(i, j);
        const Coef4 c = Arith<MGB200_ARITH_EXACT>::coef(v1[g], v2[g], st);
        double b = rhs[g];
        // Dirichlet neighbours move to the right-hand side, in the order of gs.cpp:130 (north, west, south, east)
        if (i == 1) b = __dsub_rn(b, __dmul_rn(c.c, u[L.at(0, j)]));
        if (j == 1) b = __dsub_rn(b, __dmul_rn(c.a, u[L.at(i, 0)]));
        if (i == n - 1) b = __dsub_rn(b, __dmul_rn(c.d, u[L.at(n, j)]));
        if (j == n - 1) b = __dsub_rn(b, __dmul_rn(c.b, u[L.at(i, n)]));
        y[p] = b;
    }
    __syncthreads();
    for (int k = 0; k < m - 1; ++k) {                                  // L y = b
        const int rmax = min(w, m - 1 - k);
        const double yk = y[k];
        for (int r = 1 + threadIdx.x; r <= rmax; r += blockDim.x) y[k + r] = __dsub_rn(y[k + r], __dmul_rn(ab[(long)(k + r) * bw + w - r], yk));
        __syncthreads();
    }
    for (int k = m - 1; k >= 0; --k) {                                 // U x = y
        const double xk = __ddiv_rn(y[k], ab[(long)k * bw + w]);
        const int rmax = min(w, k);
        __syncthreads();                                               // everybody has read y[k]
        for (int r = 1 + threadIdx.x; r <= rmax; r += blockDim.x) y[k - r] = __dsub_rn(y[k - r], __dmul_rn(ab[(long)(k - r) * bw + w + r], xk));
        if (threadIdx.x == 0) y[k] = xk;
        __syncthreads();
    }
    for (int p = threadIdx.x; p < m; p += blockDim.x) u[L.at(1 + p / ni, 1 + p % ni)] = y[p];
}

__global__ void __launch_bounds__(128) k_coarse_lu_solve(double* __restrict__ u, const double* __restrict__ rhs,
                                                         const double* __restrict__ v1, const double* __restrict__ v2,
                                                         const double* __restrict__ ab, int n, Layout L, Stencil st, int zero_init)
{
    coarse_lu_solve_body(u, rhs, v1, v2, ab, n, L, st, zero_init);
}

// one block per member: fields mstride apart, factors abstride apart; a frozen member is left as it is
__global__ void __launch_bounds__(128) k_coarse_lu_solve_batched(double* __restrict__ u, const double* __restrict__ rhs,
                                                                 const double* __restrict__ v1, const double* __restrict__ v2,
                                                                 const double* __restrict__ ab, int n, Layout L, Stencil st,
                                                                 int zero_init, long mstride, long abstride,
                                                                 const int* __restrict__ active)
{
    const int b = blockIdx.x;
    if (!active[b]) return;
    const long mo = (long)b * mstride;
    coarse_lu_solve_body(u + mo, rhs + mo, v1 + mo, v2 + mo, ab + (long)b * abstride, n, L, st, zero_init);
}

}  // namespace

int ops_basic_init()
{
    // function attributes are per device
    static std::mutex mu;
    static bool done[64] = {};
    int dev = 0;
    MGB_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    if (dev >= 0 && dev < 64 && done[dev]) return MGB200_OK;
    const int smem = 4 * 65 * 65 * (int)sizeof(double);
    MGB_CUDA(cudaFuncSetAttribute(k_coarse_solve<MGB200_ARITH_EXACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    MGB_CUDA(cudaFuncSetAttribute(k_coarse_solve<MGB200_ARITH_FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    MGB_CUDA(cudaFuncSetAttribute(k_coarse_solve_batched<MGB200_ARITH_EXACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    MGB_CUDA(cudaFuncSetAttribute(k_coarse_solve_batched<MGB200_ARITH_FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    if (dev >= 0 && dev < 64) done[dev] = true;
    return MGB200_OK;
}

size_t coarse_lu_bytes(long n) { return (size_t)(n - 1) * (n - 1) * (2 * (n - 1) + 1) * sizeof(double); }

int launch_coarse_lu_factor(double* ab, const double* v1, const double* v2, long n, Layout L, const Stencil& st, cudaStream_t s)
{
    if (n > 64 || n < 4) return fail(MGB200_ERR_INVALID, "coarse_lu: 4 <= n <= 64");
    k_coarse_lu_factor<<<1, 1024, 0, s>>>(ab, v1, v2, (int)n, L, st);
    return check_launch("k_coarse_lu_factor");
}

int launch_coarse_lu_solve(double* u, const double* rhs, const double* v1, const double* v2, const double* ab, long n, Layout L,
                           const Stencil& st, bool zero_init, cudaStream_t s)
{
    if (n > 64 || n < 4) return fail(MGB200_ERR_INVALID, "coarse_lu: 4 <= n <= 64");
    k_coarse_lu_solve<<<1, 128, (size_t)(n - 1) * (n - 1) * sizeof(double), s>>>(u, rhs, v1, v2, ab, (int)n, L, st, zero_init ? 1 : 0);
    return check_launch("k_coarse_lu_solve");
}

// ---------------------------------------------------------------------------------------------
// the colour-split layout of a level (common.cuh: split_layout) as opposed to a natural (row-major) one
static bool is_split(const Layout& L, long n) { const Layout S = split_layout(n); return L.odd == S.odd && L.pitch == S.pitch && L.odd > 0; }
static dim3 rhs_split_grid(long n, long nrows)
{
    const long pairs = n / 2 + 1;
    return dim3((unsigned)((pairs + 2 * RHS_TPB - 1) / (2 * RHS_TPB)), (unsigned)((nrows + RHS_ROWS - 1) / RHS_ROWS), 1);
}
long compute_rhs_partials_count(long n, long nrows, Layout L)
{
    if (is_split(L, n)) { const dim3 g = rhs_split_grid(n, nrows); return (long)g.x * g.y; }
    return rows_partials_count(n, nrows);
}

long residual_partials_count(long n)
{
    dim3 g = tile_grid(n - 1, n - 1);
    return (long)g.x * g.y;
}

long rows_partials_count(long n, long nrows)
{
    dim3 g = tile_grid(nrows, n - 1);
    return (long)g.x * g.y;
}

int launch_gs_colour(double* u, const double* rhs, const double* v1, const double* v2, long n, Layout L,
                     const Stencil& st, int colour, int arith, cudaStream_t s)
{
    if (n < 2) return MGB200_OK;
    dim3 g = tile_grid(n - 1, (n - 1 + 1) / 2);
    if (arith == MGB200_ARITH_EXACT)
        k_gs_colour<MGB200_ARITH_EXACT><<<g, TPB, 0, s>>>(u, rhs, v1, v2, n, L, st, colour);
    else
        k_gs_colour<MGB200_ARITH_FAST><<<g, TPB, 0, s>>>(u, rhs, v1, v2, n, L, st, colour);
    return check_launch("k_gs_colour");
}

int launch_residual(double* res, const double* u, const double* rhs, const double* v1, const double* v2,
                    long n, Layout L, const Stencil& st, int arith, double* partials, cudaStream_t s)
{
    if (n < 2) return MGB200_OK;
    dim3 g = tile_grid(n - 1, n - 1);
    const int mode = (res ? 1 : 0) | (partials ? 2 : 0);
    if (mode == 0) return fail(MGB200_ERR_INVALID, "launch_residual: nothing to produce");
#define MGB_RES(A, M) k_residual<A, M><<<g, TPB, 0, s>>>(res, u, rhs, v1, v2, n, L, st, partials)
    if (arith == MGB200_ARITH_EXACT) {
        if (mode == 1) MGB_RES(MGB200_ARITH_EXACT, 1); else if (mode == 2) MGB_RES(MGB200_ARITH_EXACT, 2); else MGB_RES(MGB200_ARITH_EXACT, 3);
    } else {
        if (mode == 1) MGB_RES(MGB200_ARITH_FAST, 1); else if (mode == 2) MGB_RES(MGB200_ARITH_FAST, 2); else MGB_RES(MGB200_ARITH_FAST, 3);
    }
#undef MGB_RES
    return check_launch("k_residual");
}

int launch_compute_rhs(double* rhs, const double* u, const double* v1, const double* v2, long n, Layout L,
                       const Stencil& st, int arith, double* partials, cudaStream_t s, long row_lo, long row_hi)
{
    if (n < 2) return MGB200_OK;
    const long ilo = row_lo < 1 ? 1 : row_lo, ihi = (row_hi < 0 || row_hi > n - 1) ? n - 1 : row_hi;
    if (ihi < ilo) return MGB200_OK;
    if (is_split(L, n)) {
        const dim3 g = rhs_split_grid(n, ihi - ilo + 1);
        if (arith == MGB200_ARITH_EXACT) {
            if (partials) k_compute_rhs_split<MGB200_ARITH_EXACT, true><<<g, RHS_TPB, 0, s>>>(rhs, u, v1, v2, n, L, st, partials, ilo, ihi);
            else k_compute_rhs_split<MGB200_ARITH_EXACT, false><<<g, RHS_TPB, 0, s>>>(rhs, u, v1, v2, n, L, st, partials, ilo, ihi);
        } else {
            if (partials) k_compute_rhs_split<MGB200_ARITH_FAST, true><<<g, RHS_TPB, 0, s>>>(rhs, u, v1, v2, n, L, st, partials, ilo, ihi);
            else k_compute_rhs_split<MGB200_ARITH_FAST, false><<<g, RHS_TPB, 0, s>>>(rhs, u, v1, v2, n, L, st, partials, ilo, ihi);
        }
        return check_launch("k_compute_rhs_split");
    }
    dim3 g = tile_grid(ihi - ilo + 1, n - 1);
    if (arith == MGB200_ARITH_EXACT) {
        if (partials) k_compute_rhs<MGB200_ARITH_EXACT, true><<<g, TPB, 0, s>>>(rhs, u, v1, v2, n, L, st, partials, ilo, ihi);
        else k_compute_rhs<MGB200_ARITH_EXACT, false><<<g, TPB, 0, s>>>(rhs, u, v1, v2, n, L, st, partials, ilo, ihi);
    } else {
        if (partials) k_compute_rhs<MGB200_ARITH_FAST, true><<<g, TPB, 0, s>>>(rhs, u, v1, v2, n, L, st, partials, ilo, ihi);
        else k_compute_rhs<MGB200_ARITH_FAST, false><<<g, TPB, 0, s>>>(rhs, u, v1, v2, n, L, st, partials, ilo, ihi);
    }
    return check_launch("k_compute_rhs");
}

int launch_square_partials(const double* a, long n, Layout L, double* partials, cudaStream_t s)
{
    dim3 g = tile_grid(n - 1, n - 1);
    k_square_partials<<<g, TPB, 0, s>>>(a, n, L, partials);
    return check_launch("k_square_partials");
}

int launch_reduce_partials(const double* partials, long count, double* out, cudaStream_t s)
{
    k_reduce_partials<<<1, 1024, 0, s>>>(partials, count, out);
    return check_launch("k_reduce_partials");
}

int launch_restrict(double* coarse, Layout Lc, const double* fine, Layout Lf, long nf, cudaStream_t s)
{
    const long nc = nf / 2;
    k_restrict<false><<<tile_grid(nc + 1, nc + 1), TPB, 0, s>>>(coarse, Lc, fine, Lf, nc);
    return check_launch("k_restrict");
}

int launch_restrict_interior(double* coarse, Layout Lc, const double* fine, Layout Lf, long nf, cudaStream_t s)
{
    const long nc = nf / 2;
    if (nc < 2) return MGB200_OK;
    k_restrict<true><<<tile_grid(nc - 1, nc - 1), TPB, 0, s>>>(coarse, Lc, fine, Lf, nc);
    return check_launch("k_restrict");
}

int launch_restrict_fw(double* coarse, Layout Lc, const double* fine, Layout Lf, long nf, bool interior_only, cudaStream_t s)
{
    const long nc = nf / 2;
    if (interior_only) {
        if (nc < 2) return MGB200_OK;
        k_restrict_fw<true><<<tile_grid(nc - 1, nc - 1), TPB, 0, s>>>(coarse, Lc, fine, Lf, nc);
    } else {
        k_restrict_fw<false><<<tile_grid(nc + 1, nc + 1), TPB, 0, s>>>(coarse, Lc, fine, Lf, nc);
    }
    return check_launch("k_restrict_fw");
}

int launch_prolong(double* fine, Layout Lf, const double* coarse, Layout Lc, long nc, bool add, cudaStream_t s)
{
    dim3 g = tile_grid(2 * nc + 1, 2 * nc + 1);
    if (add) k_prolong<true><<<g, TPB, 0, s>>>(fine, Lf, coarse, Lc, nc);
    else k_prolong<false><<<g, TPB, 0, s>>>(fine, Lf, coarse, Lc, nc);
    return check_launch("k_prolong");
}

int launch_vecadd(double* c, const double* a, const double* b, long n, Layout L, cudaStream_t s)
{
    k_vecadd<<<tile_grid(n + 1, n + 1), TPB, 0, s>>>(c, a, b, n, L);
    return check_launch("k_vecadd");
}

int launch_convert(double* dst, Layout Ld, const double* src, Layout Ls, long n, cudaStream_t s, long row_lo, long row_hi)
{
    const long ilo = row_lo < 0 ? 0 : row_lo, ihi = (row_hi < 0 || row_hi > n) ? n : row_hi;
    if (ihi < ilo) return MGB200_OK;
    k_convert<<<tile_grid(ihi - ilo + 1, n + 1), TPB, 0, s>>>(dst, Ld, src, Ls, n, ilo, ihi);
    return check_launch("k_convert");
}

int launch_initial_conditions(double* u0, double* v1, double* v2, long n, Layout L, double vscale, cudaStream_t s,
                              long row_lo, long row_hi)
{
    const long ilo = row_lo < 0 ? 0 : row_lo, ihi = (row_hi < 0 || row_hi > n) ? n : row_hi;
    if (ihi < ilo) return MGB200_OK;
    k_initial_conditions<<<tile_grid(ihi - ilo + 1, n + 1), TPB, 0, s>>>(u0, v1, v2, n, L, vscale, ilo, ihi);
    return check_launch("k_initial_conditions");
}

int launch_tower_flat(double* flat_out, const double* src, bool from_level0, Layout L0, long N, cudaStream_t s)
{
    const long q = N / 4;
    k_tower_flat<<<tile_grid(q + 1, q + 1), TPB, 0, s>>>(flat_out, src, from_level0 ? 1 : 0, L0, N);
    return check_launch("k_tower_flat");
}

int launch_flat_to_level(double* dst, Layout Ld, const double* flat, long nl, cudaStream_t s, long row_lo, long row_hi)
{
    const long ilo = row_lo < 0 ? 0 : row_lo, ihi = (row_hi < 0 || row_hi > nl) ? nl : row_hi;
    if (ihi < ilo) return MGB200_OK;
    k_flat_to_level<<<tile_grid(ihi - ilo + 1, nl + 1), TPB, 0, s>>>(dst, Ld, flat, nl, ilo, ihi);
    return check_launch("k_flat_to_level");
}

int launch_coarse_solve(double* u, const double* rhs, const double* v1, const double* v2, long n, Layout L,
                        const Stencil& st, int arith, bool zero_init, int maxit, double tol, int* iters_out,
                        cudaStream_t s)
{
    if (n > 64) return fail(MGB200_ERR_INVALID, "coarse_solve: n > 64 not supported by the single-block kernel");
    const size_t smem = 4 * (size_t)(n + 1) * (n + 1) * sizeof(double);
    MGB_TRY(ops_basic_init());
    if (arith == MGB200_ARITH_EXACT) {
        k_coarse_solve<MGB200_ARITH_EXACT><<<1, 1024, smem, s>>>(u, rhs, v1, v2, (int)n, L, st, zero_init ? 1 : 0, maxit, tol, iters_out);
    } else {
        k_coarse_solve<MGB200_ARITH_FAST><<<1, 1024, smem, s>>>(u, rhs, v1, v2, (int)n, L, st, zero_init ? 1 : 0, maxit, tol, iters_out);
    }
    return check_launch("k_coarse_solve");
}

// ---------------------------------------------------------------------------------------------
// batched solver handles: `members` problems, member b of every array at + b * mstride
int launch_compute_rhs_batched(double* rhs, const double* u, const double* v1, const double* v2, long n, Layout L,
                               const Stencil& st, int arith, double* partials, long pstride, int members, long mstride,
                               cudaStream_t s)
{
    if (!is_split(L, n) || n < 4 || members < 1 || members > 65535) return fail(MGB200_ERR_INVALID, "compute_rhs_batched: bad argument");
    dim3 g = rhs_split_grid(n, n - 1);
    if ((long)g.x * g.y > pstride) return fail(MGB200_ERR_INVALID, "compute_rhs_batched: partials stride too small");
    g.z = (unsigned)members;
    if (arith == MGB200_ARITH_EXACT)
        k_compute_rhs_split_batched<MGB200_ARITH_EXACT><<<g, RHS_TPB, 0, s>>>(rhs, u, v1, v2, n, L, st, partials, 1, n - 1, mstride, pstride);
    else
        k_compute_rhs_split_batched<MGB200_ARITH_FAST><<<g, RHS_TPB, 0, s>>>(rhs, u, v1, v2, n, L, st, partials, 1, n - 1, mstride, pstride);
    return check_launch("k_compute_rhs_split_batched");
}

int launch_reduce_partials_batched(const double* partials, long count, long pstride, double* out, const int* active, int members,
                                   cudaStream_t s)
{
    k_reduce_partials_batched<<<members, 1024, 0, s>>>(partials, count, pstride, out, active);
    return check_launch("k_reduce_partials_batched");
}

int launch_coarse_solve_batched(double* u, const double* rhs, const double* v1, const double* v2, long n, Layout L,
                                const Stencil& st, int arith, bool zero_init, int maxit, double tol, int* iters_out,
                                int members, long mstride, const int* active, cudaStream_t s)
{
    if (n > 64) return fail(MGB200_ERR_INVALID, "coarse_solve: n > 64 not supported by the single-block kernel");
    const size_t smem = 4 * (size_t)(n + 1) * (n + 1) * sizeof(double);
    MGB_TRY(ops_basic_init());
    if (arith == MGB200_ARITH_EXACT)
        k_coarse_solve_batched<MGB200_ARITH_EXACT><<<members, 1024, smem, s>>>(u, rhs, v1, v2, (int)n, L, st, zero_init ? 1 : 0, maxit, tol,
                                                                              iters_out, mstride, active);
    else
        k_coarse_solve_batched<MGB200_ARITH_FAST><<<members, 1024, smem, s>>>(u, rhs, v1, v2, (int)n, L, st, zero_init ? 1 : 0, maxit, tol,
                                                                             iters_out, mstride, active);
    return check_launch("k_coarse_solve_batched");
}

int launch_coarse_lu_solve_batched(double* u, const double* rhs, const double* v1, const double* v2, const double* ab, long n,
                                   Layout L, const Stencil& st, bool zero_init, int members, long mstride, long abstride,
                                   const int* active, cudaStream_t s)
{
    if (n > 64 || n < 4) return fail(MGB200_ERR_INVALID, "coarse_lu: 4 <= n <= 64");
    k_coarse_lu_solve_batched<<<members, 128, (size_t)(n - 1) * (n - 1) * sizeof(double), s>>>(u, rhs, v1, v2, ab, (int)n, L, st,
                                                                                               zero_init ? 1 : 0, mstride, abstride, active);
    return check_launch("k_coarse_lu_solve_batched");
}

}  // namespace mgb200
