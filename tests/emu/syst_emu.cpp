// syst_emu.cpp -- TEST INFRASTRUCTURE: a host model of the systolic streaming kernel.
//
// There is no GPU in the build container, so the index logic AND the synchronisation protocol of
// the pass (csrc/syst_pass_body.cuh) are exercised here by compiling the very same per-thread code
// for the host and running every lane of a thread block as a real thread:
//   * the progress counters are atomics with release / acquire ordering, the TMA full barriers atomics with
//     the hardware's phase-parity semantics;
//   * the TMA engine and the bulk-store engine are memcpy in the issuing thread;
//   * shared memory starts as NaN, so a read of a cell that was never staged poisons the result;
//   * built with -fsanitize=thread (tests/test_syst_pass_emu.py does both builds), every pair of
//     conflicting shared-memory accesses that the barrier protocol does not order is reported as a
//     data race: the protocol is checked, not just one interleaving of it.
// Never linked into libmgb200.so.
#include <execinfo.h>
#include <pthread.h>
#include <signal.h>
#include <unistd.h>
#include <sched.h>

#include <atomic>
#include <chrono>
#include <cstdio>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <thread>
#include <vector>

static inline double __dmul_rn(double a, double b) { return a * b; }
static inline double __dadd_rn(double a, double b) { return a + b; }
static inline double __dsub_rn(double a, double b) { return a - b; }
static inline double __ddiv_rn(double a, double b) { return a / b; }
static inline double __shfl_down_sync(unsigned, double v, int) { return v; }   // (common.cuh's block_sum: unused here)
static inline void __syncthreads() {}
#define SY_FN static inline
#define SY_HOST_MODEL 1
#include <cuda_runtime.h>
static uint3 threadIdx, blockDim;
#include "../../hpcclassmultigridproject_b200/csrc/syst_pass_body.cuh"

namespace mgb200 {
void set_error(const std::string&) {}
int fail(int code, const std::string&) { return code; }
long& launch_counter() { static long c = 0; return c; }
namespace sy {

static thread_local int t_lane = 0, t_warp = 0;
static pthread_barrier_t g_wbar[WARPS];
// mbarrier model: completed-phase count; arrival count 1 (+ transaction bytes for the full barriers)
struct MBar { std::atomic<unsigned long> phases{0}; std::atomic<long> tx{0}; };
static MBar g_full[NGROUP];
static std::atomic<unsigned> g_prog[NPROG];       // steps completed per stage warp
static std::atomic<long> g_spins{0};
static int g_jitter = 0;

static inline void jitter()
{
    if (!g_jitter) return;
    static thread_local unsigned rng = 0;
    if (!rng) rng = 2654435761u * (unsigned)(t_warp * 32 + t_lane + 1);
    rng = rng * 1664525u + 1013904223u;
    if (((rng >> 16) % 16) < (unsigned)g_jitter) sched_yield();
}

static std::atomic<long> g_done[WARPS];          // steps published per warp (diagnostics of a deadlock)
static inline void mbar_wait(MBar& b, unsigned parity, const char* what = "", int idx = 0)
{
    // true iff the phase with this parity is the immediately preceding one (hardware semantics)
    long spins = 0;
    while (((b.phases.load(std::memory_order_acquire)) & 1ul) == parity) {
        sched_yield();
        if (++spins > 3000000L) {                         // a protocol deadlock: die loudly instead of hanging the suite
            static std::atomic<int> first{0};
            if (first.fetch_add(1) == 0) {
                std::fprintf(stderr, "syst_emu: warp %d stuck waiting for %s %d parity %u; steps published:", t_warp, what, idx, parity);
                for (int w = 0; w < NSTAGE; ++w) std::fprintf(stderr, " %ld", g_done[w].load());
                std::fprintf(stderr, "\n");
            }
            std::this_thread::sleep_for(std::chrono::milliseconds(200));
            std::abort();
        }
    }
    g_spins.fetch_add(spins, std::memory_order_relaxed);
}

SY_FN int sy_lane() { return t_lane; }
SY_FN bool sy_elect() { return t_lane == 0; }
SY_FN void sy_syncwarp() { pthread_barrier_wait(&g_wbar[t_warp]); }
SY_FN void sy_full_expect(const Smem&, int g, unsigned bytes) { g_full[g].tx.store((long)bytes, std::memory_order_relaxed); }
// software model of the 3-D tensor copy: box {inner, 2, rows} at (x, 0, z), zeros outside the tensor
SY_FN void sy_tma_load(const Params& p, const Smem& sm, int which, unsigned soff, int x, int z, int g)
{
    double* sdst = reinterpret_cast<double*>(sm.raw + soff);
    const double* src = which == FIELD_U ? p.u_in : which == FIELD_F ? p.rhs : which == FIELD_V1 ? p.v1 : which == FIELD_V2 ? p.v2 : p.cu;
    const bool coarse = which == FIELD_C;
    const long odd = coarse ? p.codd : p.odd, pitch = coarse ? p.cpitch : p.pitch;
    const long nrows = coarse ? p.crows_mem : p.rows_mem;
    const int inner = coarse ? p.CW : p.SWK, brows = coarse ? CROWS : GROUP;
    for (int zz = 0; zz < brows; ++zz)
        for (int par = 0; par < 2; ++par)
            for (int xx = 0; xx < inner; ++xx) {
                const long gx = (long)x + xx, gz = (long)z + zz;
                const bool in = gx >= 0 && gx < odd && gz >= 0 && gz < nrows;
                sdst[((long)zz * 2 + par) * inner + xx] = in ? src[gz * pitch + par * odd + gx] : 0.0;
            }
    const long left = g_full[g].tx.fetch_sub((long)brows * 2 * inner * 8, std::memory_order_relaxed) - (long)brows * 2 * inner * 8;
    if (left == 0) g_full[g].phases.fetch_add(1, std::memory_order_release);
}
SY_FN void sy_tma_prefetch(const Params&, int, int, int) {}
SY_FN void sy_full_wait(const Smem&, int g, unsigned parity) { jitter(); mbar_wait(g_full[g], parity, "TMA group slot", g); }
SY_FN void sy_prog_publish(const Smem&, int warp, unsigned steps_done)
{
    jitter();
    g_done[warp].store((long)steps_done, std::memory_order_relaxed);
    g_prog[warp].store(steps_done, std::memory_order_release);
}
SY_FN Prog2 sy_prog_peek(const Smem&, int stage)
{
    jitter();
    Prog2 v;
    v.h0 = g_prog[2 * stage].load(std::memory_order_acquire);
    v.h1 = g_prog[2 * stage + 1].load(std::memory_order_acquire);
    return v;
}
SY_FN void sy_backoff(int pair)
{
    static thread_local long spins = 0;
    sched_yield();
    if (++spins % 3000000L == 0) {                        // a protocol deadlock: die loudly instead of hanging the suite
        std::fprintf(stderr, "syst_emu: warp %d lane %d has been spinning on the progress counters of pair %d; steps published:", t_warp, t_lane, pair);
        for (int w = 0; w < NSTAGE; ++w) std::fprintf(stderr, " %ld", g_done[w].load());
        std::fprintf(stderr, "\n");
        std::abort();
    }
}
SY_FN void sy_bulk_store(const Smem& sm, double* gdst, unsigned soff, unsigned bytes) { std::memcpy(gdst, sm.raw + soff, bytes); }
SY_FN void sy_store_commit() {}
SY_FN void sy_store_wait_read0() {}
SY_FN void sy_store_wait_read1() {}
SY_FN void sy_store_wait_all() {}
SY_FN void sy_fence_async() {}
SY_FN D2 sy_lds2(const Smem& sm, unsigned off) { return *reinterpret_cast<const D2*>(sm.raw + off); }
SY_FN double sy_lds1(const Smem& sm, unsigned off) { return *reinterpret_cast<const double*>(sm.raw + off); }
SY_FN void sy_sts2(const Smem& sm, unsigned off, D2 v) { *reinterpret_cast<D2*>(sm.raw + off) = v; }
SY_FN void sy_sts1(const Smem& sm, unsigned off, double v) { *reinterpret_cast<double*>(sm.raw + off) = v; }
// a real shuffle between the lane threads of a warp: write the own value, rendezvous, read the neighbour's,
// rendezvous (every lane of the warp must call it, as on the device)
static double g_shfl[WARPS][2][32];
SY_FN double sy_side(const Smem& sm, const D2& mid, unsigned off, int dir, bool outer)
{
    g_shfl[t_warp][0][t_lane] = mid.x; g_shfl[t_warp][1][t_lane] = mid.y;
    pthread_barrier_wait(&g_wbar[t_warp]);
    double x;
    if (dir < 0) x = t_lane > 0 ? g_shfl[t_warp][1][t_lane - 1] : 0.0;
    else x = t_lane < 31 ? g_shfl[t_warp][0][t_lane + 1] : 0.0;
    pthread_barrier_wait(&g_wbar[t_warp]);
    if (t_lane == (dir < 0 ? 0 : 31)) x = outer ? 0.0 : sy_lds1(sm, off);
    return x;
}

}  // namespace sy
}  // namespace mgb200

using namespace mgb200;
using namespace mgb200::sy;

extern "C" {

// Runs one pass over level n on HOST arrays in the split layout (rows_mem == 0: the whole level;
// otherwise a row slab: the arrays hold global rows row0.. and rows own_lo..own_hi are produced).
// wk/nbands <= 0: use the planner.  jitter: 0..16, how often a thread yields around a barrier
// operation.  partials: >= ntiles doubles.  Returns the number of tiles, or -1 on a bad argument.
static void on_abort(int)
{
    void* bt[48];
    const int nb = backtrace(bt, 48);
    backtrace_symbols_fd(bt, nb, 2);
    _exit(134);
}

long syst_emu_run(long n, long pitch, long odd, long cpitch, long codd, const double* u_in, double* u_out,
                  const double* rhs, const double* v1, const double* v2, const double* cu, double* crhs,
                  double* partials, int K, int post, int arith, double dt, double nu, double dx, int wk, int nbands,
                  int jitter_level, long own_lo, long own_hi, long row0, long rows_mem, long crow0, long crows_mem)
{
    if (K < 1 || K > KMAX || n < 8 || (n & 3)) return -1;
    if (getenv("SYST_EMU_BACKTRACE")) signal(SIGABRT, on_abort);
    if (rows_mem == 0) { own_lo = 0; own_hi = n; row0 = 0; rows_mem = n + 1; crow0 = 0; crows_mem = n / 2 + 1; }
    g_jitter = jitter_level;
    Params p{};
    p.n = n; p.nhalf = n / 2; p.pitch = pitch; p.odd = odd; p.cpitch = cpitch; p.codd = codd;
    p.own_lo = own_lo; p.own_hi = own_hi; p.row0 = row0; p.rows_mem = rows_mem;
    p.mem_lo = row0; p.mem_hi = row0 + rows_mem - 1; p.crow0 = crow0; p.crows_mem = crows_mem;
    Plan pl = make_plan(n, own_hi - own_lo + 1, K, 148);
    if (wk > 0) {
        pl.WK = wk; pl.SWK = wk + 2 * HK; pl.nstrips = (int)((n / 2 + 1 + wk - 1) / wk);
    }
    if (nbands > 0) {
        const long nr = own_hi - own_lo + 1;
        pl.RBAND = (nr + nbands - 1) / nbands; pl.nbands = (int)((nr + pl.RBAND - 1) / pl.RBAND);
    }
    if (pl.SWK > SWK_MAX || (pl.SWK & 15)) return -1;
    p.RBAND = pl.RBAND; p.WK = pl.WK; p.SWK = pl.SWK; p.nstrips = pl.nstrips; p.nbands = pl.nbands;
    p.K = K; p.pre = cu ? 1 : 0; p.post = post; p.u_is_zero = u_in ? 0 : 1;
    // Stencil exactly as make_stencil (solver.cu)
    {
        volatile double r = 0.5 * dt / (dx * dx);
        volatile double four_r = 4.0 * r;
        volatile double four_r_nu = four_r * nu;
        p.st.r = r; p.st.nu = nu; p.st.h = dx; p.st.diag = 1.0 - four_r_nu; p.st.diag_rhs = 1.0 + four_r_nu;
        p.st.inv_diag = 1.0 / p.st.diag; p.st.hr = r * dx * 0.5; p.st.rnu = r * nu;
    }
    p.CW = pl.SWK / 2 + 8;
    p.u_in = u_in; p.rhs = rhs; p.v1 = v1; p.v2 = v2; p.cu = cu;
    p.u_out = u_out; p.crhs = crhs; p.partials = partials;
    const long ntiles = (long)pl.nstrips * pl.nbands;
    std::vector<unsigned char> smem(SMEM_BYTES + 64);
    unsigned char* sbase = smem.data() + ((64 - reinterpret_cast<uintptr_t>(smem.data()) % 64) % 64);
    for (int w = 0; w < WARPS; ++w) pthread_barrier_init(&g_wbar[w], nullptr, 32);
    for (long tile = 0; tile < ntiles; ++tile) {
        double* sd = reinterpret_cast<double*>(sbase);
        for (size_t q = 0; q < SMEM_BYTES / 8; ++q) sd[q] = std::numeric_limits<double>::quiet_NaN();
        for (auto& b : g_full) { b.phases.store(0); b.tx.store(0); }
        for (auto& c : g_prog) c.store(0);
        for (auto& d : g_done) d.store(0);
        Smem sm;
        carve(sm, sbase, p.SWK);
        const Tile tl = make_tile(p, tile);
        const Geo geo = make_geo(p);
        std::vector<double> acc(THREADS, 0.0);
        std::vector<std::thread> thr;
        for (int tid = 0; tid < THREADS; ++tid)
            thr.emplace_back([&, tid] {
                t_warp = tid >> 5; t_lane = tid & 31;
                double a = 0.0;
#define RUN(AR, PRE, PK) a = run_warp<AR, PRE, PK>(p, tl, geo, sm, t_warp, t_lane)
#define RUN_POST(AR, PRE) do { if (post == POST_NORM2) RUN(AR, PRE, POST_NORM2); else if (post == POST_INJECT) RUN(AR, PRE, POST_INJECT); else RUN(AR, PRE, POST_NONE); } while (0)
                if (arith == MGB200_ARITH_EXACT) { if (p.pre) RUN_POST(MGB200_ARITH_EXACT, true); else RUN_POST(MGB200_ARITH_EXACT, false); }
                else { if (p.pre) RUN_POST(MGB200_ARITH_FAST, true); else RUN_POST(MGB200_ARITH_FAST, false); }
#undef RUN_POST
#undef RUN
                acc[tid] = a;
            });
        for (auto& t : thr) t.join();
        if (post == POST_NORM2) {
            double s = 0.0;
            for (double a : acc) s += a;
            partials[tile] = s;
        }
    }
    for (int w = 0; w < WARPS; ++w) pthread_barrier_destroy(&g_wbar[w]);
    return ntiles;
}

}  // extern "C"
