// multigrid_b200 -- command-line front end equivalent to the reference's `multigrid` / `multigrid_cu`
// executables (multigrid.cpp:188-293, multigrid.cu:210-273), whose parameters are hard-coded
// literals there and flags here.  Same initial conditions, same solver parameters, same output
// format: uT.txt with one "%d\t%d\t%f\n" line per node, row-major (multigrid.cpp:269-275), plus an
// optional raw float64 dump.  Host side only: every compute call goes through the C ABI.
//
//   multigrid_b200 [--N 256] [--steps 100] [--nu -4e-4] [--vscale 1] [--tol 1e-6] [--shape 1]
//                  [--niter 3] [--coarse-tol 1e-5] [--coarse-maxit 1000] [--max-cycle 50]     (multigrid.cpp:41,60,94)
//                  [--correct-towers] [--exact] [--unfused] [--full-weighting] [--gpus 1]
//                  [--out uT.txt] [--bin uT.f64] [--quiet]
// --gpus P > 1: the program forks P processes, one per GPU (row slabs, include/mgb200.h "Row-slab sharding");
// process 0 creates the communicator id and hands it to the others through pipes, every process writes the rows
// it owns into a shared mapping, the parent prints and dumps.
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <sys/mman.h>
#include <sys/wait.h>
#include <unistd.h>

#include "../include/mgb200.h"

static void die(const char* what)
{
    std::fprintf(stderr, "multigrid_b200: %s: %s\n", what, mgb200_last_error());
    std::exit(1);
}

struct Run {
    long N; int steps, shape, gpus; double nu, vscale, tol; mgb200_options opt;
};
struct Report { double sec; long cycles; double last_ratio; int ok; };

// one process = one GPU: rank `rank` of `r.gpus`; fills its own rows of uT (full-size array) and *rep
static int run_rank(const Run& r, int rank, const unsigned char* id, double* uT, Report* rep)
{
    const int maxlvl = int(std::log2((double)r.N)) - 4;    // multigrid.cpp:193
    const double dx = 1.0 / r.N, dt = dx / 10;             // :194, :238
    mgb200_options opt = r.opt;
    if (r.gpus > 1) opt.device = rank;
    mgb200_solver* s = nullptr;
    const int rc = r.gpus == 1 ? mgb200_create(&s, r.N, maxlvl, r.nu, dt, dx, r.tol, &opt)
                               : mgb200_create_sharded(&s, r.N, maxlvl, r.nu, dt, dx, r.tol, &opt, rank, r.gpus, id, 0);
    if (rc != MGB200_OK) die("create");
    if (mgb200_set_fields_reference_ic(s, r.vscale) != MGB200_OK) die("initial conditions");
    std::vector<mgb200_solve_info> infos(r.steps > 0 ? r.steps : 1);
    const auto t0 = std::chrono::steady_clock::now();
    if (mgb200_timestep(s, r.steps, infos.data()) != MGB200_OK) die("timestep");
    if (mgb200_synchronize(s) != MGB200_OK) die("synchronize");
    rep->sec = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    rep->cycles = 0;
    for (int k = 0; k < r.steps; ++k) rep->cycles += infos[k].cycles;
    rep->last_ratio = r.steps > 0 ? infos[r.steps - 1].res / infos[r.steps - 1].res0 : 0.0;
    if (mgb200_get_u_host(s, uT) != MGB200_OK) die("get_u");     // a slab rank fills the rows it owns
    mgb200_destroy(s);
    rep->ok = 1;
    return 0;
}

int main(int argc, char** argv)
{
    long N = 256;                       // multigrid.cpp:192
    int steps = 100, shape = 1, gpus = 1;   // :239, :241
    double nu = -4e-4, vscale = 1.0, tol = 1e-6;   // :235, :240
    std::string out = "uT.txt", bin;
    bool quiet = false;
    mgb200_options opt;
    mgb200_default_options(&opt);
    for (int a = 1; a < argc; ++a) {
        const std::string k = argv[a];
        auto val = [&]() -> const char* { if (a + 1 >= argc) { std::fprintf(stderr, "missing value for %s\n", k.c_str()); std::exit(2); } return argv[++a]; };
        if (k == "--N") N = std::atol(val());
        else if (k == "--steps") steps = std::atoi(val());
        else if (k == "--nu") nu = std::atof(val());
        else if (k == "--vscale") vscale = std::atof(val());
        else if (k == "--tol") tol = std::atof(val());
        else if (k == "--shape") shape = std::atoi(val());
        else if (k == "--niter") opt.niter = std::atoi(val());
        else if (k == "--coarse-tol") opt.coarse_tol = std::atof(val());        // multigrid.cpp:60
        else if (k == "--coarse-maxit") opt.coarse_maxit = std::atoi(val());    // multigrid.cpp:60
        else if (k == "--max-cycle") opt.max_cycle = std::atoi(val());          // multigrid.cpp:94
        else if (k == "--correct-towers") opt.correct_towers = 1;               // instead of multigrid.cpp:148-160
        else if (k == "--gpus") gpus = std::atoi(val());
        else if (k == "--exact") opt.arith = MGB200_ARITH_EXACT;
        else if (k == "--unfused") opt.plan = MGB200_PLAN_UNFUSED;
        else if (k == "--full-weighting") opt.restriction = MGB200_RESTRICT_FW;
        else if (k == "--out") out = val();
        else if (k == "--bin") bin = val();
        else if (k == "--quiet") quiet = true;
        else { std::fprintf(stderr, "unknown flag %s\n", k.c_str()); return 2; }
    }
    opt.shape = shape;
    Run r{N, steps, shape, gpus, nu, vscale, tol, opt};
    const size_t m0 = (size_t)(N + 1) * (N + 1);
    double* uT = nullptr;
    Report rep{};
    if (gpus == 1) {
        uT = (double*)std::malloc(m0 * sizeof(double));
        run_rank(r, 0, nullptr, uT, &rep);
    } else {
        // shared result + one report per rank; pipes carry the 128-byte communicator id from rank 0
        uT = (double*)mmap(nullptr, m0 * sizeof(double), PROT_READ | PROT_WRITE, MAP_SHARED | MAP_ANONYMOUS, -1, 0);
        Report* reps = (Report*)mmap(nullptr, sizeof(Report) * gpus, PROT_READ | PROT_WRITE, MAP_SHARED | MAP_ANONYMOUS, -1, 0);
        if (uT == MAP_FAILED || reps == MAP_FAILED) { std::perror("mmap"); return 1; }
        std::vector<int> fds(2 * gpus);
        for (int g = 1; g < gpus; ++g) if (pipe(&fds[2 * g]) != 0) { std::perror("pipe"); return 1; }
        std::vector<pid_t> kids;
        for (int g = 0; g < gpus; ++g) {
            const pid_t pid = fork();                       // before any CUDA call of this process
            if (pid < 0) { std::perror("fork"); return 1; }
            if (pid == 0) {
                unsigned char id[128];
                if (g == 0) {
                    if (mgb200_comm_unique_id(id) != MGB200_OK) die("comm_unique_id");
                    for (int q = 1; q < gpus; ++q) if (write(fds[2 * q + 1], id, 128) != 128) { std::perror("write"); _exit(1); }
                } else if (read(fds[2 * g], id, 128) != 128) { std::perror("read"); _exit(1); }
                run_rank(r, g, id, uT, &reps[g]);
                _exit(0);
            }
            kids.push_back(pid);
        }
        int bad = 0;
        for (pid_t pid : kids) { int st = 0; waitpid(pid, &st, 0); if (!WIFEXITED(st) || WEXITSTATUS(st) != 0) bad = 1; }
        for (int g = 0; g < gpus; ++g) if (!reps[g].ok) bad = 1;
        if (bad) { std::fprintf(stderr, "multigrid_b200: a rank failed\n"); return 1; }
        rep = reps[0];
    }
    const double sec = rep.sec;
    const long cycles = rep.cycles;
    if (!quiet)
        std::printf("\nB200 time, N = %ld, %d GPU(s): %f s  (%d steps, %ld cycles, last ||r||/||r0|| = %.3e)\n%g\n", N, gpus, sec, steps, cycles,
                    rep.last_ratio, uT[(N / 2) * (N + 1) + N / 2]);
    if (!out.empty() && out != "-") {
        FILE* f = std::fopen(out.c_str(), "w");
        if (!f) { std::perror(out.c_str()); return 1; }
        for (long i = 0; i <= N; ++i)
            for (long j = 0; j <= N; ++j) std::fprintf(f, "%ld\t%ld\t%f\n", i, j, uT[i * (N + 1) + j]);   // multigrid.cpp:272
        std::fclose(f);
    }
    if (!bin.empty()) {
        FILE* f = std::fopen(bin.c_str(), "wb");
        if (!f) { std::perror(bin.c_str()); return 1; }
        std::fwrite(uT, sizeof(double), m0, f);
        std::fclose(f);
    }
    return 0;
}
