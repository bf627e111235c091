// syst_emu_batched.cpp -- TEST INFRASTRUCTURE: the host model of the streaming kernel (syst_emu_fw.cpp, which
// includes syst_emu.cpp) extended by the batched flavour (k_syst_pass_batched): `members` problems of one size,
// member b of every fine / coarse array b * mstride / b * cmstride doubles after the first, tile t of member b run
// with sy_member() = b.  A member whose active flag is 0 is skipped whole, as the kernel's blocks return before they
// touch anything.  The 4-D tensor copy zero-fills outside the member's rows.  Also exports make_plan.  Never linked
// into libmgb200.so.
#include "syst_emu_fw.cpp"

namespace mgb200 {
namespace sy {
static int t_member = 0;            // set before the tile's threads start
static long g_mstride = 0, g_cmstride = 0, g_members = 0;

SY_FN int sy_member() { return t_member; }
SY_FN void sy_tma_load_m(const Params& p, const Smem& sm, int which, unsigned soff, int x, int z, int m, int g)
{
    // the member coordinate must name an existing member; then it is the 3-D copy on that member's arrays
    if (m < 0 || m >= g_members) std::abort();
    Params q = p;
    const long mo = (long)m * g_mstride, cmo = (long)m * g_cmstride;
    q.u_in = p.u_in ? p.u_in + mo : nullptr; q.rhs = p.rhs + mo; q.v1 = p.v1 + mo; q.v2 = p.v2 + mo;
    q.cu = p.cu ? p.cu + cmo : nullptr;
    sy_tma_load(q, sm, which, soff, x, z, g);
}
SY_FN void sy_tma_prefetch_m(const Params&, int, int, int, int) {}
}  // namespace sy
}  // namespace mgb200

extern "C" {

long syst_emu_plan(long n, long nrows, int K, int sms, int members, long out[5])
{
    const Plan pl = members > 0 ? make_plan(n, nrows, K, sms, 0, members) : make_plan(n, nrows, K, sms);
    out[0] = pl.WK; out[1] = pl.SWK; out[2] = pl.nstrips; out[3] = pl.nbands; out[4] = pl.RBAND;
    return (long)pl.nstrips * pl.nbands;
}

// One batched pass over whole levels (rows 0..n); post: StreamPost (POST_FW without cu).  partials: members x
// pstride doubles.  Returns the number of tiles per member, or -1 on a bad argument.
long syst_emu_batched_run(long n, long pitch, long odd, long cpitch, long codd, int members, long mstride, long cmstride,
                          const int* active, const double* u_in, double* u_out, const double* rhs, const double* v1,
                          const double* v2, const double* cu, double* crhs, double* partials, long pstride, int K, int post,
                          int arith, double dt, double nu, double dx, int wk, int nbands, int jitter_level)
{
    if (K < 1 || K > KMAX || n < 8 || (n & 3) || members < 1 || (post == POST_FW && cu)) return -1;
    g_jitter = jitter_level;
    g_members = members; g_mstride = mstride; g_cmstride = cmstride;
    Params p{};
    p.n = n; p.nhalf = n / 2; p.pitch = pitch; p.odd = odd; p.cpitch = cpitch; p.codd = codd;
    p.own_lo = 0; p.own_hi = n; p.row0 = 0; p.rows_mem = n + 1;
    p.mem_lo = 0; p.mem_hi = n; p.crow0 = 0; p.crows_mem = n / 2 + 1;
    Plan pl = make_plan(n, n + 1, K, 148, 0, members);
    if (wk > 0) {
        pl.WK = wk; pl.SWK = wk + 2 * HK; pl.nstrips = (int)((n / 2 + 1 + wk - 1) / wk);
    }
    if (nbands > 0) {
        pl.RBAND = (n + 1 + nbands - 1) / nbands; pl.nbands = (int)((n + 1 + pl.RBAND - 1) / pl.RBAND);
    }
    if (pl.SWK > SWK_MAX || (pl.SWK & 15)) return -1;
    const long ntiles = (long)pl.nstrips * pl.nbands;
    if (post == POST_NORM2 && pstride < ntiles) return -1;
    p.RBAND = pl.RBAND; p.WK = pl.WK; p.SWK = pl.SWK; p.nstrips = pl.nstrips; p.nbands = pl.nbands;
    p.K = K; p.pre = cu ? 1 : 0; p.post = post; p.u_is_zero = u_in ? 0 : 1;
    {   // Stencil exactly as make_stencil (solver.cu)
        volatile double r = 0.5 * dt / (dx * dx);
        volatile double four_r = 4.0 * r;
        volatile double four_r_nu = four_r * nu;
        p.st.r = r; p.st.nu = nu; p.st.h = dx; p.st.diag = 1.0 - four_r_nu; p.st.diag_rhs = 1.0 + four_r_nu;
        p.st.inv_diag = 1.0 / p.st.diag; p.st.hr = r * dx * 0.5; p.st.rnu = r * nu;
    }
    p.CW = pl.SWK / 2 + 8;
    p.u_in = u_in; p.rhs = rhs; p.v1 = v1; p.v2 = v2; p.cu = cu;
    p.u_out = u_out; p.crhs = crhs; p.partials = partials;
    p.mstride = mstride; p.cmstride = cmstride; p.pstride = pstride; p.active = active;
    std::vector<unsigned char> smem(SMEM_BYTES + 64);
    unsigned char* sbase = smem.data() + ((64 - reinterpret_cast<uintptr_t>(smem.data()) % 64) % 64);
    for (int w = 0; w < WARPS; ++w) pthread_barrier_init(&g_wbar[w], nullptr, 32);
    for (int m = 0; m < members; ++m) {
        if (active[m] == 0) continue;
        t_member = m;
        for (long tile = 0; tile < ntiles; ++tile) {
            double* sd = reinterpret_cast<double*>(sbase);
            for (size_t q = 0; q < SMEM_BYTES / 8; ++q) sd[q] = std::numeric_limits<double>::quiet_NaN();
            for (auto& b : g_full) { b.phases.store(0); b.tx.store(0); }
            for (auto& c : g_prog) c.store(0);
            for (auto& d : g_done) d.store(0);
            Smem sm;
            carve(sm, sbase, p.SWK);
            const Tile tl = make_tile(p, tile, post == POST_FW ? 1 : 0);
            const Geo geo = make_geo(p);
            std::vector<double> acc(THREADS, 0.0);
            std::vector<std::thread> thr;
            for (int tid = 0; tid < THREADS; ++tid)
                thr.emplace_back([&, tid] {
                    t_warp = tid >> 5; t_lane = tid & 31;
                    double a = 0.0;
#define RUN(AR, PRE, PK) a = run_warp<AR, PRE, PK, true>(p, tl, geo, sm, t_warp, t_lane)
#define RUN_POST(AR, PRE) do { if (post == POST_NORM2) RUN(AR, PRE, POST_NORM2); else if (post == POST_INJECT) RUN(AR, PRE, POST_INJECT); \
                               else if (post == POST_FW) RUN(AR, false, POST_FW); else RUN(AR, PRE, POST_NONE); } while (0)
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
                partials[(long)m * pstride + tile] = s;
            }
        }
    }
    for (int w = 0; w < WARPS; ++w) pthread_barrier_destroy(&g_wbar[w]);
    return ntiles;
}

}  // extern "C"
