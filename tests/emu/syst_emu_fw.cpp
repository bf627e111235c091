// syst_emu_fw.cpp -- TEST INFRASTRUCTURE: the host model of the streaming kernel (syst_emu.cpp, included whole: its
// primitives and its syst_emu_run) extended by the full-weighting down-leg flavour, POST_FW.  Same arguments as
// syst_emu_run without the coarse u (the flavour has no prolongation); the tiles carry the extra halo row of the
// flavour (make_tile, extra = 1), as the kernel's do.  Never linked into libmgb200.so.
#include "syst_emu.cpp"

extern "C" long syst_emu_fw_run(long n, long pitch, long odd, long cpitch, long codd, const double* u_in, double* u_out,
                                const double* rhs, const double* v1, const double* v2, double* crhs, int K, int arith,
                                double dt, double nu, double dx, int wk, int nbands, int jitter_level, long own_lo,
                                long own_hi, long row0, long rows_mem, long crow0, long crows_mem)
{
    if (K < 1 || K > KMAX || n < 8 || (n & 3) || !crhs) return -1;
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
    p.K = K; p.pre = 0; p.post = POST_FW; p.u_is_zero = u_in ? 0 : 1;
    {   // Stencil exactly as make_stencil (solver.cu)
        volatile double r = 0.5 * dt / (dx * dx);
        volatile double four_r = 4.0 * r;
        volatile double four_r_nu = four_r * nu;
        p.st.r = r; p.st.nu = nu; p.st.h = dx; p.st.diag = 1.0 - four_r_nu; p.st.diag_rhs = 1.0 + four_r_nu;
        p.st.inv_diag = 1.0 / p.st.diag; p.st.hr = r * dx * 0.5; p.st.rnu = r * nu;
    }
    p.CW = pl.SWK / 2 + 8;
    p.u_in = u_in; p.rhs = rhs; p.v1 = v1; p.v2 = v2; p.cu = nullptr;
    p.u_out = u_out; p.crhs = crhs; p.partials = nullptr;
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
        const Tile tl = make_tile(p, tile, 1);
        const Geo geo = make_geo(p);
        std::vector<std::thread> thr;
        for (int tid = 0; tid < THREADS; ++tid)
            thr.emplace_back([&, tid] {
                t_warp = tid >> 5; t_lane = tid & 31;
                if (arith == MGB200_ARITH_EXACT) run_warp<MGB200_ARITH_EXACT, false, POST_FW>(p, tl, geo, sm, t_warp, t_lane);
                else run_warp<MGB200_ARITH_FAST, false, POST_FW>(p, tl, geo, sm, t_warp, t_lane);
            });
        for (auto& t : thr) t.join();
    }
    for (int w = 0; w < WARPS; ++w) pthread_barrier_destroy(&g_wbar[w]);
    return ntiles;
}
