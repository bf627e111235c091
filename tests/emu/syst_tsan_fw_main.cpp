// syst_tsan_fw_main.cpp -- TEST INFRASTRUCTURE: driver of the ThreadSanitizer build of the host model (syst_emu_fw.cpp)
// for the full-weighting down-leg pass (POST_FW): the residual rows shared by the last stage and the two warps of the
// EPI role add write-after-read hazards that the progress counters must order.  Results are checked by
// tests/test_syst_pass_emu_fw.py with the plain build of the same model.
#include <cstdio>
#include <vector>

extern "C" long syst_emu_fw_run(long n, long pitch, long odd, long cpitch, long codd, const double* u_in, double* u_out,
                                const double* rhs, const double* v1, const double* v2, double* crhs, int K, int arith,
                                double dt, double nu, double dx, int wk, int nbands, int jitter_level, long own_lo,
                                long own_hi, long row0, long rows_mem, long crow0, long crows_mem);

static long lay_odd(long n) { return (n / 2 + 1 + 15) / 16 * 16 + 32; }

static std::vector<double> field(long rows, long pitch, unsigned seed)
{
    std::vector<double> a((size_t)rows * pitch);
    unsigned r = seed * 2654435761u + 12345u;
    for (auto& x : a) { r = r * 1664525u + 1013904223u; x = (double)(r >> 8) / (1 << 24) - 0.5; }
    return a;
}

int main()
{
    struct Case { long n; int K, wk, nbands, jitter; };
    const Case cases[] = {
        {64, 3, 24, 2, 4},       // one warp per stage
        {96, 1, 0, 0, 2},        // K = 1: the last stage is stage 1
        {96, 2, 56, 2, 8},       // K = 2
        {288, 3, 120, 2, 4},     // two warps per stage: the EPI warps read each other's residual rows
        {512, 3, 120, 3, 2},     // interior strips: the mask-free last stage
    };
    for (const Case& c : cases) {
        const long n = c.n, odd = lay_odd(n), pitch = 2 * odd, codd = lay_odd(n / 2), cpitch = 2 * codd;
        auto u = field(n + 1, pitch, 1), rhs = field(n + 1, pitch, 2), v1 = field(n + 1, pitch, 3), v2 = field(n + 1, pitch, 4);
        std::vector<double> out((size_t)(n + 1) * pitch, 0.0), crhs((size_t)(n / 2 + 1) * cpitch, 0.0);
        const double dx = 1.0 / n, dt = dx / 10;
        const long nt = syst_emu_fw_run(n, pitch, odd, cpitch, codd, u.data(), out.data(), rhs.data(), v1.data(), v2.data(),
                                        crhs.data(), c.K, 1, dt, -4e-4, dx, c.wk, c.nbands, c.jitter, 0, 0, 0, 0, 0, 0);
        std::printf("n=%ld K=%d wk=%d bands=%d: %ld tiles\n", n, c.K, c.wk, c.nbands, nt);
        std::fflush(stdout);
        if (nt <= 0) return 2;
    }
    std::printf("all passes done\n");
    return 0;
}
