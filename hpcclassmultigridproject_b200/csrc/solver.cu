// solver.cu -- the V/W-cycle driver (C++ host side) behind the C ABI of include/mgb200.h.
//
// Re-creates the control flow of the reference driver -- mg_inner / mg_outer / timestepper,
// multigrid.cpp:17-186 (= multigrid.cu:17-200) -- on level towers that live in HBM in the
// split layout (common.cuh).  Two pass plans produce the same field:
//   UNFUSED  one launch per reference operator (ops_basic.cu): 2 launches per RB iteration,
//            residual, injection, zero, prolong+add.   W = 320 B/node/level (SURVEY.md 8d).
//   FUSED    one streaming launch per leg (syst_pass.cu): {3 RB iterations + residual +
//            injection} going down, {prolong + correct + 3 RB iterations (+ residual norm on
//            level 0)} coming up.                      W = 84 B/node/level.
// One whole cycle + convergence check is captured into a CUDA graph and replayed; the only
// host decision per cycle is the comparison of the norm (multigrid.cpp:108), read back through
// pinned memory.  The coarsest level is solved by one thread block on the device
// (multigrid.cpp:55-65), so no host round trip happens inside a cycle.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "comm.cuh"
#include "ops_basic.cuh"
#include "stream_pass.cuh"

namespace mgb200 {

// ---------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;
void set_error(const std::string& msg) { g_last_error = msg; }
int fail(int code, const std::string& msg)
{
    g_last_error = msg;
    return code;
}
long& launch_counter()
{
    static thread_local long c = 0;
    return c;
}

Stencil make_stencil(double dt, double nu, double dx)
{
    // volatile: keep the host compiler from contracting or re-associating; the sequence is the
    // reference's (gs.cpp:10, :44, :75).
    volatile double r = 0.5 * dt / (dx * dx);
    volatile double four_r = 4.0 * r;
    volatile double four_r_nu = four_r * nu;
    Stencil s;
    s.r = r; s.nu = nu; s.h = dx;
    s.diag = 1.0 - four_r_nu;
    s.diag_rhs = 1.0 + four_r_nu;
    s.inv_diag = 1.0 / s.diag;
    s.hr = r * dx * 0.5;
    s.rnu = r * nu;
    return s;
}

struct Level {
    long n = 0;
    Layout L{0, 0};                    // split layout; L.row0 = first row held (row slabs)
    Stencil st{};
    size_t elems = 0;
    double* u[2] = {nullptr, nullptr};
    int cur = 0;                       // which of u[] holds the current iterate
    double *rhs = nullptr, *v1 = nullptr, *v2 = nullptr;
    // row window.  A single GPU owns and holds rows 0..n of every level.  With P ranks the fine
    // levels are cut into row slabs (own rows + HALO rows received from the slab neighbours); the
    // coarse levels live whole on rank 0, and the first of them also as a slab on the other ranks
    // (target of the injection, source of the prolongation).
    long own_lo = 0, own_hi = 0;       // rows this rank produces
    long mem_lo = 0, mem_hi = 0;       // rows held in memory
    bool sharded = false;              // cut across all ranks
    bool present = true;               // arrays exist on this rank
    long rows_mem() const { return mem_hi - mem_lo + 1; }
};

constexpr long SLAB_HALO = 8;          // >= 2K+1 = 7 rows a streaming pass recomputes per side, 2K+2 = 8 with full weighting

// Row slab of `rank` at a level of size n cut over P ranks: even cuts (injection stays local), the
// last rank also owns row n.  Pure arithmetic: every rank can compute every other rank's window.
struct Slab { long own_lo, own_hi, mem_lo, mem_hi; };
static Slab slab_of(long n, int P, int rank)
{
    Slab w;
    const long per = n / P;
    w.own_lo = rank * per;
    w.own_hi = (rank + 1) * per - 1 + (rank == P - 1 ? 1 : 0);
    w.mem_lo = w.own_lo - SLAB_HALO < 0 ? 0 : w.own_lo - SLAB_HALO;
    w.mem_hi = w.own_hi + SLAB_HALO > n ? n : w.own_hi + SLAB_HALO;
    return w;
}
// slab of the first agglomerated level on a non-root rank: the coarse rows under its fine slab
static Slab child_slab_of(long n_fine, int P, int rank)
{
    const Slab f = slab_of(n_fine, P, rank);
    const long nc = n_fine / 2;
    Slab w;
    w.own_lo = (f.own_lo + 1) / 2;
    w.own_hi = f.own_hi / 2;
    w.mem_lo = w.own_lo - SLAB_HALO < 0 ? 0 : w.own_lo - SLAB_HALO;
    w.mem_hi = w.own_hi + SLAB_HALO > nc ? nc : w.own_hi + SLAB_HALO;
    return w;
}

// The sharding rule: the row window of `rank` at level `lvl` of an n-point hierarchy of maxlvl levels over P ranks.
// A level is cut into slabs while it is not the coarsest, its slabs keep shard_min_rows and 2 SLAB_HALO rows each,
// and every finer level is cut too.  The other levels live whole on rank 0; the first of them also as the slab under
// each other rank's fine slab.  Pure arithmetic: mgb200_slab_plan gives it without a GPU.
struct Window { bool sharded, present; Slab rows; };
static Window slab_window(long n, int maxlvl, int P, int rank, long shard_min_rows, int lvl)
{
    Window w{};
    int last = -1;                     // the coarsest level cut so far
    for (int l = 0; l <= lvl; ++l) {
        const long nl = n >> l;
        w = Window{false, true, Slab{0, nl, 0, nl}};
        if (P == 1) continue;
        if (l < maxlvl - 1 && nl / P >= shard_min_rows && nl / P >= 2 * SLAB_HALO && last == l - 1) {
            w.sharded = true;
            w.rows = slab_of(nl, P, rank);
            last = l;
        } else if (rank != 0) {
            if (l == last + 1 && l > 0) w.rows = child_slab_of(n >> (l - 1), P, rank);
            else w.present = false;
        }
    }
    return w;
}

// mg_outer's loop state (multigrid.cpp:100-116) when the loop itself runs on the device
struct LoopState {
    double res0, tol;
    int iter, max_cycle;
    double hist[52];
};

// while (iter < max_cycle && res/res0 > tol) -- the test before the first cycle (res == res0)
__global__ void k_loop_begin(cudaGraphConditionalHandle h, const double* norm2, LoopState* st, double tol, int max_cycle)
{
    const double r0 = sqrt(norm2[0]);                                             // gs.cpp:106
    st->res0 = r0; st->tol = tol; st->iter = 0; st->max_cycle = max_cycle; st->hist[0] = r0;
    cudaGraphSetConditional(h, (0 < max_cycle && r0 / r0 > tol) ? 1u : 0u);
}

// ... and after every cycle
__global__ void k_loop_check(cudaGraphConditionalHandle h, const double* norm2, LoopState* st)
{
    const double r = sqrt(norm2[0]);
    const int it = ++st->iter;
    st->hist[it] = r;
    cudaGraphSetConditional(h, (it < st->max_cycle && r / st->res0 > st->tol) ? 1u : 0u);
}

// Batched handles: the same loop per member (one block, members strided over its threads).  A member runs while its
// own condition holds; active[b] tells the passes of the next cycle whether to touch member b, and the loop goes on
// while any member is active.
__global__ void k_loop_begin_batched(cudaGraphConditionalHandle h, const double* norm2, LoopState* st, int* active, double tol,
                                     int max_cycle, int members)
{
    int any = 0;
    for (int b = threadIdx.x; b < members; b += blockDim.x) {
        const double r0 = sqrt(norm2[b]);
        LoopState& s = st[b];
        s.res0 = r0; s.tol = tol; s.iter = 0; s.max_cycle = max_cycle; s.hist[0] = r0;
        const int go = (0 < max_cycle && r0 / r0 > tol) ? 1 : 0;
        active[b] = go; any |= go;
    }
    any = __syncthreads_or(any);
    if (threadIdx.x == 0) cudaGraphSetConditional(h, any ? 1u : 0u);
}

__global__ void k_loop_check_batched(cudaGraphConditionalHandle h, const double* norm2, LoopState* st, int* active, int members)
{
    int any = 0;
    for (int b = threadIdx.x; b < members; b += blockDim.x) {
        if (!active[b]) continue;
        LoopState& s = st[b];
        const double r = sqrt(norm2[b]);
        const int it = ++s.iter;
        s.hist[it] = r;
        const int go = (it < s.max_cycle && r / s.res0 > s.tol) ? 1 : 0;
        active[b] = go; any |= go;
    }
    any = __syncthreads_or(any);
    if (threadIdx.x == 0) cudaGraphSetConditional(h, any ? 1u : 0u);
}

__global__ void k_fill_int(int* a, int n, int v)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) a[i] = v;
}

}  // namespace mgb200

using namespace mgb200;

struct mgb200_solver {
    long N = 0;
    int maxlvl = 0;
    double nu = 0, dt = 0, dx = 0, tol = 0;
    mgb200_options opt{};
    int device = 0;
    std::vector<Level> lv;
    cudaStream_t stream = nullptr;
    double* d_partials = nullptr;      // block partial sums of squares
    long partials_cap = 0;
    double* d_norm2 = nullptr;         // [0] current ||r||^2
    double* h_norm2 = nullptr;         // pinned mirror
    int* d_coarse_iters = nullptr;
    double* d_coarse_lu = nullptr;     // opt-in direct coarsest solve: the factored band matrix (options.coarse_exact)
    double* d_flat[2] = {nullptr, nullptr};
    // Batched handle (mgb200_create_batched): `batch` independent problems of this size; member b of every level
    // array lives at + b * elems of one allocation, its partial sums at d_partials + b * pstride, its norm in
    // d_norm2[b], its loop state in d_loop[b].  0: a handle of one problem.
    int batch = 0;
    long pstride = 0;
    int* d_active = nullptr;           // per member: 1 while it iterates (a pass leaves a member with 0 untouched)
    int* h_active = nullptr;           // pinned mirror (host loop)
    std::vector<double> res0_b, res_b; // per member: host copies of res0 / the last norm
    int  members() const { return batch > 0 ? batch : 1; }
    int  activate_all();
    int  read_norms(double* out);
    int  solve_batched(mgb200_solve_info* infos);
    int  timestep_batched(int nsteps, mgb200_solve_info* infos);
    void fill_pass_batch(StreamPassArgs& a, const Level& g, const Level& c) const;
    cudaGraphExec_t graph_exec = nullptr;
    long graph_kernels = 0;
    // the whole mg_outer loop as one graph: a WHILE node around the cycle, condition set on the device
    cudaGraphExec_t loop_exec = nullptr;
    bool loop_failed = false;
    long loop_kernels = 0;             // kernels of one trip through the loop body
    LoopState* d_loop = nullptr;
    LoopState* h_loop = nullptr;       // pinned
    int  build_loop_graph();
    LoopState* h_steps = nullptr;      // pinned: loop state of every step of a multi-step run
    int h_steps_cap = 0;
    int  timestep(int nsteps, mgb200_solve_info* infos);
    bool device_loop() const { return opt.use_graph && !loop_failed && (P == 1 || p2p); }
    long launches = 0;
    bool have_fields = false, have_rhs = false;
    bool norm_is_res0 = false;         // d_norm2[0] holds ||r0||^2 of the current right-hand side (no cycle since form_rhs)
    bool res0_on_host = false;         // ... and `res0` has been read back
    double res0 = 0, res = 0;
    // row-slab sharding (one process per GPU)
    Comm* comm = nullptr;
    int rank = 0, P = 1;
    int last_sharded = -1;             // index of the coarsest sharded level (-1: none)
    long shard_min_rows = 256;
    double* d_top[3] = {nullptr, nullptr, nullptr};   // dense rows 0..N/4+1 of u0,v1,v2 (tower input when sharded)
    // peer-memory halo exchange: the slab neighbours' u twins and rhs of every sharded level and
    // their counter blocks, mapped with CUDA IPC.  peer[0] = rank-1, peer[1] = rank+1.
    struct PeerLevel { double* u[2] = {nullptr, nullptr}; double* rhs = nullptr; };
    struct PeerRank { std::vector<PeerLevel> lv; int* sync = nullptr; double* red = nullptr; };
    bool p2p = false;
    std::vector<PeerRank> peers;       // indexed by rank; only neighbours and rank 0 <-> everybody are mapped
    int* d_sync = nullptr;             // this rank's counter block (layout: comm.cuh)
    double* d_red = nullptr;           // landing block of the norm reduction through rank 0
    int  allreduce_norm();             // d_norm2[0] <- sum over ranks
    int  check_peers();                // after a synchronisation: did a device-side wait for a peer give up?
    std::vector<void*> ipc_mapped;
    int  setup_p2p();
    double* d_flat_scratch() { return d_norm2 + 4; }   // a spare double for set-up collectives
    // MGB200_TRACE=1: CUDA events between the phases of a cycle, printed by rank 0 (diagnostics)
    bool tracing = false;
    std::vector<std::pair<std::string, cudaEvent_t>> marks;
    void mark(const std::string& name)
    {
        if (!tracing) return;
        cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, stream);
        marks.emplace_back(name, e);
    }
    void dump_marks()
    {
        if (!tracing || marks.empty()) return;
        cudaStreamSynchronize(stream);
        if (rank == 0) {
            std::string line = "MGB200_TRACE";
            for (size_t k = 1; k < marks.size(); ++k) {
                float ms = 0; cudaEventElapsedTime(&ms, marks[k - 1].second, marks[k].second);
                char buf[96]; snprintf(buf, sizeof buf, " | %s %.3f", marks[k].first.c_str(), ms);
                line += buf;
            }
            float tot = 0; cudaEventElapsedTime(&tot, marks.front().second, marks.back().second);
            fprintf(stderr, "%s | total %.3f ms\n", line.c_str(), tot);
        }
        for (auto& m : marks) cudaEventDestroy(m.second);
        marks.clear();
    }

    ~mgb200_solver() { release(); }
    void release();
    int  init(long n, int maxlvl_, double nu_, double dt_, double dx_, double tol_, const mgb200_options* o);
    int  build_towers();
    int  cycle_body(int l);
    int  smooth(Level& g, int iters);
    int  residual_norm_level0();
    int  record_cycle();               // cycle_body(0) + convergence norm, on `stream`
    int  run_cycle_async();
    int  read_norm(double* out);
    int  form_rhs(double* res0_out, bool sync = true);
    int  solve(mgb200_solve_info* info);
    int  get_u_natural(double* dst_dev, long ld);
    int  alloc_levels();
    int  alloc_top();
    void fill_pass_window(StreamPassArgs& a, const Level& g, const Level& c) const;
    int  exchange_halo(Level& g, double* a, Level* g2 = nullptr, double* a2 = nullptr);
    int  gather_to_root(Level& c, double* arr);
    int  scatter_from_root(Level& c, double* arr);
    bool runs_level(int l) const { return P == 1 || rank == 0 || lv[l].sharded; }
    long count(long before) { long d = launch_counter() - before; launches += d; return d; }
};

void mgb200_solver::release()
{
    if (graph_exec) { cudaGraphExecDestroy(graph_exec); graph_exec = nullptr; }
    if (loop_exec) { cudaGraphExecDestroy(loop_exec); loop_exec = nullptr; }
    cudaFree(d_loop); d_loop = nullptr;
    if (h_loop) { cudaFreeHost(h_loop); h_loop = nullptr; }
    if (h_steps) { cudaFreeHost(h_steps); h_steps = nullptr; h_steps_cap = 0; }
    if (stream) cudaStreamSynchronize(stream);
    for (void* m : ipc_mapped) cudaIpcCloseMemHandle(m);     // the neighbours' memory first, then ours
    ipc_mapped.clear();
    p2p = false;
    for (auto& g : lv) {
        cudaFree(g.u[0]); cudaFree(g.u[1]); cudaFree(g.rhs); cudaFree(g.v1); cudaFree(g.v2);
    }
    lv.clear();
    cudaFree(d_partials); d_partials = nullptr;
    cudaFree(d_norm2); d_norm2 = nullptr;
    cudaFree(d_coarse_iters); d_coarse_iters = nullptr;
    cudaFree(d_coarse_lu); d_coarse_lu = nullptr;
    cudaFree(d_active); d_active = nullptr;
    if (h_active) { cudaFreeHost(h_active); h_active = nullptr; }
    cudaFree(d_flat[0]); cudaFree(d_flat[1]); d_flat[0] = d_flat[1] = nullptr;
    for (auto& t : d_top) { cudaFree(t); t = nullptr; }
    cudaFree(d_sync); d_sync = nullptr;
    cudaFree(d_red); d_red = nullptr;
    if (comm) { comm_destroy(comm); comm = nullptr; }
    if (h_norm2) { cudaFreeHost(h_norm2); h_norm2 = nullptr; }
    if (stream) { cudaStreamDestroy(stream); stream = nullptr; }
}

int mgb200_solver::init(long n, int maxlvl_, double nu_, double dt_, double dx_, double tol_, const mgb200_options* o)
{
    if (o) {
        if (o->struct_size != (int)sizeof(mgb200_options)) return fail(MGB200_ERR_INVALID, "mgb200_options.struct_size mismatch");
        opt = *o;
    } else {
        mgb200_default_options(&opt);
    }
    if (n < 4 || (n & (n - 1)) != 0) return fail(MGB200_ERR_INVALID, "n must be a power of two >= 4");
    if (maxlvl_ < 1 || (n >> (maxlvl_ - 1)) < 4) return fail(MGB200_ERR_INVALID, "maxlvl out of range for n");
    if ((n >> (maxlvl_ - 1)) > 64)
        return fail(MGB200_ERR_INVALID, "coarsest level must have n <= 64 (on-device coarse solve); raise maxlvl");
    if (opt.shape < 1 || opt.niter < 0 || opt.max_cycle < 0 || opt.max_cycle > 50)
        return fail(MGB200_ERR_INVALID, "bad options (shape >= 1, niter >= 0, 0 <= max_cycle <= 50)");
    if (opt.coarse_exact != 0 && opt.coarse_exact != 1) return fail(MGB200_ERR_INVALID, "options.coarse_exact: 0 or 1");
    if (batch > 0) {
        if (batch > STREAM_PASS_MAX_MEMBERS) return fail(MGB200_ERR_INVALID, "batch: at most 65535 members (gridDim.y of the batched pass)");
        if (opt.plan != MGB200_PLAN_FUSED) return fail(MGB200_ERR_INVALID, "a batched handle runs the fused plan only (options.plan = 0)");
        if (opt.niter == 0) return fail(MGB200_ERR_INVALID, "a batched handle needs niter >= 1 (niter = 0 implies the unfused plan)");
    }
    if (opt.restriction != MGB200_RESTRICT_INJECT && opt.restriction != MGB200_RESTRICT_FW &&
        (opt.restriction != MGB200_RESTRICT_FW_UNFUSED || opt.plan != MGB200_PLAN_UNFUSED))
        return fail(MGB200_ERR_INVALID, "options.restriction: 0 (injection), 1 (full weighting, UNFUSED plan only) or 2 (full weighting)");
    if (P > 1 && (opt.plan != MGB200_PLAN_FUSED || opt.correct_towers))
        return fail(MGB200_ERR_INVALID, "the sharded solver supports the fused plan with reference-compatible towers only");
    // niter == 0 (no smoothing at all: multigrid.cpp:69-72 and :85-88 become empty loops) leaves nothing to fuse:
    // the streaming pass is defined for 1..3 iterations, so such a solver runs the one-operator plan
    if (opt.niter == 0) {
        if (P > 1) return fail(MGB200_ERR_INVALID, "niter == 0 is not supported by the sharded solver");
        opt.plan = MGB200_PLAN_UNFUSED;
    }
    // the sharded cycle (kernels + peer-memory transfers, or NCCL groups as the fallback) is captured like the
    // single-GPU one; MGB200_SHARDED_GRAPH=0 issues everything directly on the stream instead
    if (P > 1) { const char* e = getenv("MGB200_SHARDED_GRAPH"); if (e && atoi(e) == 0) opt.use_graph = 0; }
    if (getenv("MGB200_TRACE")) { tracing = true; opt.use_graph = 0; }
    { const char* e = getenv("MGB200_DEVICE_LOOP"); if (e && atoi(e) == 0) loop_failed = true; }   // host-side mg_outer loop
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(MGB200_ERR_NO_DEVICE, "no CUDA device visible; this library has no CPU path");
    if (opt.device >= 0) MGB_CUDA(cudaSetDevice(opt.device));
    MGB_CUDA(cudaGetDevice(&device));
    cudaDeviceProp prop;
    MGB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(MGB200_ERR_NO_DEVICE, std::string("device is sm_") + std::to_string(prop.major) + std::to_string(prop.minor) +
                                              ", this library is built for sm_100a only");
    N = n; maxlvl = maxlvl_; nu = nu_; dt = dt_; dx = dx_; tol = tol_;
    MGB_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    MGB_TRY(ops_basic_init());
    if (opt.plan == MGB200_PLAN_FUSED) MGB_TRY(stream_pass_init());
    MGB_TRY(alloc_levels());
    if (batch == 0) {
        partials_cap = std::max(residual_partials_count(N), stream_pass_tiles(N, lv[0].own_hi - lv[0].own_lo + 1, -1)) + 8;
    } else {
        pstride = std::max(std::max(residual_partials_count(N), compute_rhs_partials_count(N, N - 1, lv[0].L)),
                           stream_pass_tiles(N, N + 1, -1, batch)) + 8;
        partials_cap = pstride * batch;
    }
    const size_t mb = (size_t)members();
    MGB_CUDA(cudaMalloc(&d_partials, partials_cap * sizeof(double)));
    MGB_CUDA(cudaMalloc(&d_norm2, (8 + mb) * sizeof(double)));
    MGB_CUDA(cudaMemsetAsync(d_norm2, 0, (8 + mb) * sizeof(double), stream));
    MGB_CUDA(cudaMalloc(&d_coarse_iters, mb * sizeof(int)));
    MGB_CUDA(cudaMallocHost(&h_norm2, (8 + mb) * sizeof(double)));
    MGB_CUDA(cudaMalloc(&d_loop, mb * sizeof(LoopState)));
    MGB_CUDA(cudaMemsetAsync(d_loop, 0, mb * sizeof(LoopState), stream));
    MGB_CUDA(cudaMallocHost(&h_loop, mb * sizeof(LoopState)));
    if (batch > 0) {
        MGB_CUDA(cudaMalloc(&d_active, mb * sizeof(int)));
        MGB_CUDA(cudaMallocHost(&h_active, mb * sizeof(int)));
        res0_b.assign(mb, 0.0); res_b.assign(mb, 0.0);
        MGB_TRY(activate_all());
    }
    MGB_CUDA(cudaStreamSynchronize(stream));
    if (P > 1) MGB_TRY(setup_p2p());
    return MGB200_OK;
}

int mgb200_solver::alloc_levels()
{
    lv.resize(maxlvl);
    last_sharded = -1;
    for (int l = 0; l < maxlvl; ++l) {
        Level& g = lv[l];
        g.n = N >> l;
        g.L = split_layout(g.n);
        g.st = make_stencil(dt, nu, dx * (double)(1L << l));    // dx2 = 2*dx per level (multigrid.cpp:49)
        const Window w = slab_window(N, maxlvl, P, rank, shard_min_rows, l);
        g.own_lo = w.rows.own_lo; g.own_hi = w.rows.own_hi; g.mem_lo = w.rows.mem_lo; g.mem_hi = w.rows.mem_hi;
        g.sharded = w.sharded; g.present = w.present;
        if (g.sharded) last_sharded = l;
        if (P > 1 && l == 0 && !g.sharded) return fail(MGB200_ERR_INVALID, "level 0 is too small to be cut over the ranks");
        g.L.row0 = g.mem_lo;
        if (!g.present) continue;
        g.elems = (size_t)g.L.pitch * (size_t)g.rows_mem();
        const size_t bytes = g.elems * sizeof(double) * (size_t)members();      // batched: the members back to back
        MGB_CUDA(cudaMalloc(&g.u[0], bytes));
        MGB_CUDA(cudaMalloc(&g.u[1], bytes));
        MGB_CUDA(cudaMalloc(&g.rhs, bytes));
        MGB_CUDA(cudaMalloc(&g.v1, bytes));
        MGB_CUDA(cudaMalloc(&g.v2, bytes));
        MGB_CUDA(cudaMemsetAsync(g.u[0], 0, bytes, stream));
        MGB_CUDA(cudaMemsetAsync(g.u[1], 0, bytes, stream));
        MGB_CUDA(cudaMemsetAsync(g.rhs, 0, bytes, stream));     // coarse rhs starts as zeros (multigrid.cpp:159)
        MGB_CUDA(cudaMemsetAsync(g.v1, 0, bytes, stream));
        MGB_CUDA(cudaMemsetAsync(g.v2, 0, bytes, stream));
    }
    return MGB200_OK;
}

// dense rows 0..N/4+1 of the level-0 fields: all the reference's flat tower mapping ever reads
int mgb200_solver::alloc_top()
{
    const size_t tb = (size_t)(N / 4 + 2) * (N + 1) * sizeof(double);
    for (auto& t : d_top)
        if (!t) MGB_CUDA(cudaMalloc(&t, tb));
    return MGB200_OK;
}

void mgb200_solver::fill_pass_window(StreamPassArgs& a, const Level& g, const Level& c) const
{
    if (P == 1) return;                // rows_mem == 0: whole level
    a.own_lo = g.own_lo; a.own_hi = g.own_hi;
    a.row0 = g.mem_lo; a.rows_mem = g.rows_mem();
    a.crow0 = c.mem_lo; a.crows_mem = c.rows_mem();
}

// Map the other ranks' arrays into this process (CUDA IPC over NVLink peer access): the slab
// neighbours' u twins / rhs of every sharded level, and for the agglomeration step rank 0's coarse
// rhs (on every rank) and every rank's coarse u (on rank 0).  All ranks agree on the outcome: if
// any mapping fails, everybody falls back to NCCL send/receive.
int mgb200_solver::setup_p2p()
{
    p2p = false;
    const char* e = getenv("MGB200_P2P");
    const bool want = !(e && atoi(e) == 0) && P <= 8;
    const int nl = last_sharded + 1;               // sharded levels 0..nl-1, level nl is the first agglomerated one
    const int nh = 3 * (nl + 1) + 2;               // u[0], u[1], rhs per level, then the counter and reduction blocks
    MGB_CUDA(cudaMalloc(&d_sync, SYNC_INTS * sizeof(int)));
    MGB_CUDA(cudaMemsetAsync(d_sync, 0, SYNC_INTS * sizeof(int), stream));
    MGB_CUDA(cudaMalloc(&d_red, RED_DOUBLES * sizeof(double)));
    MGB_CUDA(cudaMemsetAsync(d_red, 0, RED_DOUBLES * sizeof(double), stream));
    std::vector<cudaIpcMemHandle_t> mine(nh), all((size_t)nh * P);
    bool ok = want;
    for (int l = 0; l <= nl && ok; ++l) {
        ok = ok && cudaIpcGetMemHandle(&mine[3 * l + 0], lv[l].u[0]) == cudaSuccess;
        ok = ok && cudaIpcGetMemHandle(&mine[3 * l + 1], lv[l].u[1]) == cudaSuccess;
        ok = ok && cudaIpcGetMemHandle(&mine[3 * l + 2], lv[l].rhs) == cudaSuccess;
    }
    ok = ok && cudaIpcGetMemHandle(&mine[3 * (nl + 1)], d_sync) == cudaSuccess;
    ok = ok && cudaIpcGetMemHandle(&mine[3 * (nl + 1) + 1], d_red) == cudaSuccess;
    cudaGetLastError();
    // handles travel through one byte all-gather (collective: every rank takes part, ok or not)
    void *d_send = nullptr, *d_recv = nullptr;
    const size_t hb = (size_t)nh * sizeof(cudaIpcMemHandle_t);
    MGB_CUDA(cudaMalloc(&d_send, hb));
    MGB_CUDA(cudaMalloc(&d_recv, hb * P));
    MGB_CUDA(cudaMemcpyAsync(d_send, mine.data(), hb, cudaMemcpyHostToDevice, stream));
    MGB_TRY(comm_allgather_bytes(comm, d_send, d_recv, hb, stream));
    MGB_CUDA(cudaMemcpyAsync(all.data(), d_recv, hb * P, cudaMemcpyDeviceToHost, stream));
    MGB_CUDA(cudaStreamSynchronize(stream));
    cudaFree(d_send); cudaFree(d_recv);
    peers.assign(P, PeerRank{});
    auto open = [&](int r, int idx) -> void* {
        void* ptr = nullptr;
        if (!ok) return nullptr;
        if (cudaIpcOpenMemHandle(&ptr, all[(size_t)r * nh + idx], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
            cudaGetLastError(); ok = false; return nullptr;
        }
        ipc_mapped.push_back(ptr);
        return ptr;
    };
    for (int r = 0; r < P; ++r) {
        if (r == rank) continue;
        const bool neighbour = r == rank - 1 || r == rank + 1;
        const bool agglo = rank == 0 || r == 0;          // rank 0 <-> everybody
        if (!neighbour && !agglo) continue;
        PeerRank& pr = peers[r];
        pr.lv.assign(nl + 1, PeerLevel{});
        if (neighbour)
            for (int l = 0; l < nl; ++l) {
                pr.lv[l].u[0] = (double*)open(r, 3 * l + 0);
                pr.lv[l].u[1] = (double*)open(r, 3 * l + 1);
                pr.lv[l].rhs = (double*)open(r, 3 * l + 2);
            }
        if (rank == 0) { pr.lv[nl].u[0] = (double*)open(r, 3 * nl + 0); pr.lv[nl].u[1] = (double*)open(r, 3 * nl + 1); }
        if (r == 0) pr.lv[nl].rhs = (double*)open(r, 3 * nl + 2);
        pr.sync = (int*)open(r, 3 * (nl + 1));
        if (agglo) pr.red = (double*)open(r, 3 * (nl + 1) + 1);
    }
    // unanimous or not at all
    double flag = ok ? 1.0 : 0.0;
    MGB_CUDA(cudaMemcpyAsync(d_flat_scratch(), &flag, sizeof(double), cudaMemcpyHostToDevice, stream));
    MGB_TRY(comm_allreduce_sum(comm, d_flat_scratch(), 1, stream));
    MGB_CUDA(cudaMemcpyAsync(&flag, d_flat_scratch(), sizeof(double), cudaMemcpyDeviceToHost, stream));
    MGB_CUDA(cudaStreamSynchronize(stream));
    p2p = flag > P - 0.5;
    if (!p2p) {
        for (void* m : ipc_mapped) cudaIpcCloseMemHandle(m);
        ipc_mapped.clear();
        peers.clear();
    }
    if (getenv("MGB200_TRACE") && rank == 0) fprintf(stderr, "MGB200_TRACE halo transport: %s\n", p2p ? "peer memory" : "nccl send/recv");
    return MGB200_OK;
}

// The device-side waits for a peer (halo arrivals, gather / scatter, norm) give up after SYNC_SPIN_BUDGET ticks and
// set a flag instead of spinning for ever when a rank has died or left the collective sequence; the host reads the
// flag after it has synchronised and turns it into an error.
int mgb200_solver::check_peers()
{
    if (P == 1 || !p2p || !d_sync) return MGB200_OK;
    int flag = 0;
    MGB_CUDA(cudaMemcpyAsync(&flag, d_sync + SYNC_ABORT, sizeof(int), cudaMemcpyDeviceToHost, stream));
    MGB_CUDA(cudaStreamSynchronize(stream));
    if (flag) return fail(MGB200_ERR_STATE, "a peer rank did not arrive within the spin budget of a device-side wait (it failed or left the collective sequence); results are invalid");
    return MGB200_OK;
}

// d_norm2[0] <- sum over ranks: through rank 0 over peer memory, or NCCL all-reduce
int mgb200_solver::allreduce_norm()
{
    if (P == 1) return MGB200_OK;
    if (!p2p) return comm_allreduce_sum(comm, d_norm2, 1, stream);
    NormReduce a{};
    a.value = d_norm2; a.red = d_red; a.sync = d_sync; a.rank = rank; a.nranks = P;
    if (rank == 0) for (int r = 1; r < P; ++r) { a.peer_red[r] = peers[r].red; a.peer_sync[r] = peers[r].sync; }
    else { a.peer_red[0] = peers[0].red; a.peer_sync[0] = peers[0].sync; }
    return launch_norm_allreduce(a, stream);
}

// Slab neighbours swap SLAB_HALO boundary rows of array `a` of level g (and optionally of a second
// array of another sharded level).  Rows are contiguous: no packing.  Peer-memory transport: one
// kernel stores the rows straight into the neighbours' halo rows and synchronises through
// device-side counters (see comm.cuh); otherwise one NCCL send/receive group.
//
// Why a neighbour may write into our halo rows while we are still computing: consecutive
// exchanges target different arrays (the u twins alternate, rhs belongs to the child level), a
// pass never reads the halo rows of the array it produces, and a rank cannot run more than one
// exchange ahead of its neighbour because it has to wait for that neighbour's counter.
int mgb200_solver::exchange_halo(Level& g, double* a, Level* g2, double* a2)
{
    if (P == 1) return MGB200_OK;
    if (p2p) {
        PeerPush pp{};
        pp.sync = d_sync;
        if (rank > 0) {         // we are rank-1's lower neighbour
            pp.raise[pp.nraise++] = peers[rank - 1].sync + SYNC_FROM_DOWN;
            pp.wait_slot[pp.nwait] = SYNC_FROM_UP; pp.wait_count[pp.nwait++] = 1;
        }
        if (rank < P - 1) {     // and rank+1's upper neighbour
            pp.raise[pp.nraise++] = peers[rank + 1].sync + SYNC_FROM_UP;
            pp.wait_slot[pp.nwait] = SYNC_FROM_DOWN; pp.wait_count[pp.nwait++] = 1;
        }
        Level* lvls[2] = {&g, g2};
        double* arrs[2] = {a, a2};
        for (int k = 0; k < 2; ++k) {
            Level* q = lvls[k];
            if (!q || !q->sharded) continue;
            const int l = (int)(q - lv.data());
            const long cnt = SLAB_HALO * q->L.pitch;
            for (int d = 0; d < 2; ++d) {
                const int nb = d == 0 ? rank - 1 : rank + 1;
                if (nb < 0 || nb >= P) continue;
                const PeerLevel& pl = peers[nb].lv[l];
                double* pbase = arrs[k] == q->u[0] ? pl.u[0] : arrs[k] == q->u[1] ? pl.u[1] : arrs[k] == q->rhs ? pl.rhs : nullptr;
                if (!pbase) return fail(MGB200_ERR_INVALID, "exchange_halo: array is not shared with the neighbours");
                const Slab w = slab_of(q->n, P, nb);
                const long row = d == 0 ? q->own_lo : q->own_hi - SLAB_HALO + 1;   // our first / last owned rows
                pp.seg[pp.nseg++] = PeerSeg{arrs[k] + (row - q->mem_lo) * q->L.pitch, pbase + (row - w.mem_lo) * q->L.pitch, cnt};
            }
        }
        return launch_peer_push(pp, stream);
    }
    P2P ops[8];
    int n = 0;
    Level* lvls[2] = {&g, g2};
    double* arrs[2] = {a, a2};
    for (int k = 0; k < 2; ++k) {
        Level* q = lvls[k];
        if (!q || !q->sharded) continue;
        double* base = arrs[k];
        const size_t cnt = (size_t)SLAB_HALO * q->L.pitch;
        auto rowptr = [&](long row) { return base + (row - q->mem_lo) * q->L.pitch; };
        if (rank > 0) {
            ops[n++] = P2P{rank - 1, rowptr(q->own_lo), cnt, true};                 // my first rows -> upper neighbour
            ops[n++] = P2P{rank - 1, rowptr(q->own_lo - SLAB_HALO), cnt, false};    // its last rows -> my upper halo
        }
        if (rank < P - 1) {
            ops[n++] = P2P{rank + 1, rowptr(q->own_hi - SLAB_HALO + 1), cnt, true};
            ops[n++] = P2P{rank + 1, rowptr(q->own_hi + 1), cnt, false};
        }
    }
    return comm_p2p(comm, ops, n, stream);
}

// first agglomerated level: every rank's owned rows -> rank 0's whole array
int mgb200_solver::gather_to_root(Level& c, double* arr)
{
    if (P == 1) return MGB200_OK;
    const long nf = lv[last_sharded].n;
    if (p2p) {
        // every other rank stores its rows into rank 0's array; rank 0 waits for P-1 arrivals.
        // (Rank 0 last read this array in the previous cycle, which every rank has left behind:
        // nobody starts a cycle before the scatter of the one before.)
        PeerPush pp{};
        pp.sync = d_sync;
        if (rank == 0) {
            pp.wait_slot[0] = SYNC_GATHER; pp.wait_count[0] = P - 1; pp.nwait = 1;
        } else {
            if (arr != c.rhs) return fail(MGB200_ERR_INVALID, "gather_to_root: only the coarse rhs is shared with rank 0");
            const int lc = (int)(&c - lv.data());
            const Slab w0 = Slab{0, c.n, 0, c.n};
            pp.seg[0] = PeerSeg{arr + (c.own_lo - c.mem_lo) * c.L.pitch, peers[0].lv[lc].rhs + (c.own_lo - w0.mem_lo) * c.L.pitch,
                                (c.own_hi - c.own_lo + 1) * c.L.pitch};
            pp.nseg = 1;
            pp.raise[0] = peers[0].sync + SYNC_GATHER; pp.nraise = 1;
        }
        return launch_peer_push(pp, stream);
    }
    std::vector<P2P> ops;
    if (rank == 0) {
        for (int r = 1; r < P; ++r) {
            const Slab w = child_slab_of(nf, P, r);
            ops.push_back(P2P{r, arr + (w.own_lo - c.mem_lo) * c.L.pitch, (size_t)(w.own_hi - w.own_lo + 1) * c.L.pitch, false});
        }
    } else {
        ops.push_back(P2P{0, arr + (c.own_lo - c.mem_lo) * c.L.pitch, (size_t)(c.own_hi - c.own_lo + 1) * c.L.pitch, true});
    }
    return comm_p2p(comm, ops.data(), (int)ops.size(), stream);
}

// rank 0's whole array -> every rank's slab window (own rows + halo) of the first agglomerated level
int mgb200_solver::scatter_from_root(Level& c, double* arr)
{
    if (P == 1) return MGB200_OK;
    const long nf = lv[last_sharded].n;
    if (p2p) {
        // rank 0 stores every rank's window into that rank's array, the others wait for it.  The
        // twin index is the same on every rank: a level's passes come in pairs (down + up), and
        // the ranks that do not run the coarse levels never flip theirs.
        PeerPush pp{};
        pp.sync = d_sync;
        const int lc = (int)(&c - lv.data());
        const int twin = arr == c.u[0] ? 0 : arr == c.u[1] ? 1 : -1;
        if (twin != 0) return fail(MGB200_ERR_STATE, "scatter_from_root: coarse iterate is not in twin 0");
        if (rank == 0) {
            for (int r = 1; r < P; ++r) {
                const Slab w = child_slab_of(nf, P, r);
                pp.seg[pp.nseg++] = PeerSeg{arr + (w.mem_lo - c.mem_lo) * c.L.pitch, peers[r].lv[lc].u[twin],
                                            (w.mem_hi - w.mem_lo + 1) * c.L.pitch};
                pp.raise[pp.nraise++] = peers[r].sync + SYNC_SCATTER;
            }
        } else {
            pp.wait_slot[0] = SYNC_SCATTER; pp.wait_count[0] = 1; pp.nwait = 1;
        }
        return launch_peer_push(pp, stream);
    }
    std::vector<P2P> ops;
    if (rank == 0) {
        for (int r = 1; r < P; ++r) {
            const Slab w = child_slab_of(nf, P, r);
            ops.push_back(P2P{r, arr + (w.mem_lo - c.mem_lo) * c.L.pitch, (size_t)(w.mem_hi - w.mem_lo + 1) * c.L.pitch, true});
        }
    } else {
        ops.push_back(P2P{0, arr, (size_t)c.rows_mem() * c.L.pitch, false});
    }
    return comm_p2p(comm, ops.data(), (int)ops.size(), stream);
}

// Coarse velocity towers (timestepper prologue, multigrid.cpp:148-160).
int mgb200_solver::build_towers()
{
    if (maxlvl == 1) return MGB200_OK;
    // (a batch: the towers of every member, one after another; member b of level l at + b * lv[l].elems)
    auto mo = [&](int l, int b) { return (size_t)b * lv[l].elems; };
    if (opt.correct_towers) {
        for (int b = 0; b < members(); ++b)
            for (int l = 1; l < maxlvl; ++l) {
                MGB_TRY(launch_restrict(lv[l].v1 + mo(l, b), lv[l].L, lv[l - 1].v1 + mo(l - 1, b), lv[l - 1].L, lv[l - 1].n, stream));
                MGB_TRY(launch_restrict(lv[l].v2 + mo(l, b), lv[l].L, lv[l - 1].v2 + mo(l - 1, b), lv[l - 1].L, lv[l - 1].n, stream));
            }
        return MGB200_OK;
    }
    // Reference-compatible: every level is restriction(dst, src, N/2) on flat zero-filled
    // (N/2+1)^2 buffers, read back with the level's true stride (SURVEY.md section 8, P1).
    const long h = N / 2;
    const size_t fb = (size_t)(h + 1) * (h + 1) * sizeof(double);
    for (int k = 0; k < 2; ++k)
        if (!d_flat[k]) MGB_CUDA(cudaMalloc(&d_flat[k], fb));
    // The flat mapping only reads rows 0..N/4+1 of the level-0 velocity.  A single GPU reads them
    // from its own level 0; a slab rank from the dense copy of those rows that set_fields left in
    // d_top (every rank builds every flat buffer redundantly and keeps the rows of its windows).
    for (int b = 0; b < members(); ++b)
    for (int which = 0; which < 2; ++which) {
        const double* src0 = P == 1 ? (which == 0 ? lv[0].v1 : lv[0].v2) + mo(0, b) : d_top[1 + which];
        const Layout L0 = P == 1 ? lv[0].L : natural_layout(N + 1);
        int cur = 0;
        for (int l = 1; l < maxlvl; ++l) {
            MGB_CUDA(cudaMemsetAsync(d_flat[cur], 0, fb, stream));
            if (l == 1) MGB_TRY(launch_tower_flat(d_flat[cur], src0, true, L0, N, stream));
            else MGB_TRY(launch_tower_flat(d_flat[cur], d_flat[1 - cur], false, L0, N, stream));
            if (lv[l].present) {
                double* dst = (which == 0 ? lv[l].v1 : lv[l].v2) + mo(l, b);
                MGB_TRY(launch_flat_to_level(dst, lv[l].L, d_flat[cur], lv[l].n, stream, lv[l].mem_lo, lv[l].mem_hi));
            }
            cur = 1 - cur;
        }
    }
    return MGB200_OK;
}

// `iters` RB-GS iterations on the current iterate (unfused: two colour launches each)
int mgb200_solver::smooth(Level& g, int iters)
{
    for (int it = 0; it < iters; ++it) {
        MGB_TRY(launch_gs_colour(g.u[g.cur], g.rhs, g.v1, g.v2, g.n, g.L, g.st, 0, opt.arith, stream));
        MGB_TRY(launch_gs_colour(g.u[g.cur], g.rhs, g.v1, g.v2, g.n, g.L, g.st, 1, opt.arith, stream));
    }
    return MGB200_OK;
}

// mg_inner (multigrid.cpp:17-92)
int mgb200_solver::cycle_body(int l)
{
    Level& g = lv[l];
    const bool split = P > 1 && g.sharded;                                        // this level is cut over the ranks
    for (int rep = 0; rep < opt.shape; ++rep) {                                   // multigrid.cpp:52
        if (l == maxlvl - 1) {
            // coarsest level: on-device loop {GS; residual; norm} (multigrid.cpp:55-65).  A level
            // entered from above starts from u = 0 (multigrid.cpp:77); the kernel zero-fills itself.
            const bool fresh = (l > 0 && rep == 0);
            if (batch > 0) {
                if (opt.coarse_exact)
                    MGB_TRY(launch_coarse_lu_solve_batched(g.u[g.cur], g.rhs, g.v1, g.v2, d_coarse_lu, g.n, g.L, g.st, fresh, batch, (long)g.elems,
                                                           (long)(coarse_lu_bytes(g.n) / sizeof(double)), d_active, stream));
                else
                    MGB_TRY(launch_coarse_solve_batched(g.u[g.cur], g.rhs, g.v1, g.v2, g.n, g.L, g.st, opt.arith, fresh, opt.coarse_maxit,
                                                        opt.coarse_tol, d_coarse_iters, batch, (long)g.elems, d_active, stream));
                continue;
            }
            if (opt.coarse_exact) MGB_TRY(launch_coarse_lu_solve(g.u[g.cur], g.rhs, g.v1, g.v2, d_coarse_lu, g.n, g.L, g.st, fresh, stream));
            else MGB_TRY(launch_coarse_solve(g.u[g.cur], g.rhs, g.v1, g.v2, g.n, g.L, g.st, opt.arith, fresh,
                                             opt.coarse_maxit, opt.coarse_tol, d_coarse_iters, stream));
            continue;
        }
        Level& c = lv[l + 1];
        if (opt.plan == MGB200_PLAN_UNFUSED) {
            MGB_TRY(smooth(g, opt.niter));                                        // :69-72
            double* tmp = g.u[1 - g.cur];                                         // the idle twin is the scratch
            MGB_TRY(launch_residual(tmp, g.u[g.cur], g.rhs, g.v1, g.v2, g.n, g.L, g.st, opt.arith, nullptr, stream)); // :73
            if (opt.restriction != MGB200_RESTRICT_INJECT) MGB_TRY(launch_restrict_fw(c.rhs, c.L, tmp, g.L, g.n, true, stream));   // gs.cpp:277-280, opt-in
            else MGB_TRY(launch_restrict_interior(c.rhs, c.L, tmp, g.L, g.n, stream)); // :75
            if (l + 1 != maxlvl - 1)                                              // :77 (coarsest zero-fills itself)
                MGB_CUDA(cudaMemsetAsync(c.u[c.cur], 0, c.elems * sizeof(double), stream));
            MGB_TRY(cycle_body(l + 1));                                           // :79
            MGB_TRY(launch_prolong(g.u[g.cur], g.L, c.u[c.cur], c.L, c.n, true, stream)); // :81-83
            MGB_TRY(smooth(g, opt.niter));                                        // :85-88
        } else {
            // ---- down leg: niter RB iterations, residual, injection (or full weighting): one streaming launch ----
            const bool zero_in = (l > 0 && rep == 0);     // fresh coarse level: u == 0, nothing to read
            int left = opt.niter;
            bool first = true;
            do {
                const int k = left > 3 ? 3 : left;
                left -= k;
                StreamPassArgs a{};
                a.n = g.n; a.L = g.L; a.st = g.st; a.arith = opt.arith;
                a.u_in = (first && zero_in) ? nullptr : g.u[g.cur];
                a.u_out = g.u[1 - g.cur];
                a.rhs = g.rhs; a.v1 = g.v1; a.v2 = g.v2;
                a.iters = k;
                a.Lc = c.L;
                if (left == 0) { a.post = opt.restriction == MGB200_RESTRICT_FW ? POST_FW : POST_INJECT; a.coarse_rhs = c.rhs; }
                fill_pass_window(a, g, c);
                fill_pass_batch(a, g, c);
                MGB_TRY(stream_pass(a, stream));
                g.cur = 1 - g.cur;
                first = false;
                if (split && left > 0) MGB_TRY(exchange_halo(g, g.u[g.cur]));
            } while (left > 0);
            mark("L" + std::to_string(l) + "dn");
            if (split) {
                // the new iterate's halo rows (read by the up leg) and the coarse right-hand side: halo rows to the
                // slab neighbours, or everything to rank 0 if the child is agglomerated
                if (c.sharded) MGB_TRY(exchange_halo(g, g.u[g.cur], &c, c.rhs));
                else { MGB_TRY(exchange_halo(g, g.u[g.cur])); MGB_TRY(gather_to_root(c, c.rhs)); }
            }
            mark("L" + std::to_string(l) + "x");
            if (runs_level(l + 1)) MGB_TRY(cycle_body(l + 1));
            if (split && !c.sharded) { mark("sub"); MGB_TRY(scatter_from_root(c, c.u[c.cur])); mark("scat"); }
            // ---- up leg: prolong + correct, niter RB iterations (+ residual norm on level 0) ----
            left = opt.niter;
            first = true;
            do {
                const int k = left > 3 ? 3 : left;
                left -= k;
                StreamPassArgs a{};
                a.n = g.n; a.L = g.L; a.st = g.st; a.arith = opt.arith;
                a.u_in = g.u[g.cur];
                a.u_out = g.u[1 - g.cur];
                a.rhs = g.rhs; a.v1 = g.v1; a.v2 = g.v2;
                a.iters = k;
                a.Lc = c.L;
                if (first) a.coarse_u = c.u[c.cur];
                if (left == 0 && l == 0 && rep == opt.shape - 1) { a.post = POST_NORM2; a.partials = d_partials; }
                fill_pass_window(a, g, c);
                fill_pass_batch(a, g, c);
                MGB_TRY(stream_pass(a, stream));
                g.cur = 1 - g.cur;
                first = false;
                mark("L" + std::to_string(l) + "up");
                if (split) { MGB_TRY(exchange_halo(g, g.u[g.cur])); mark("L" + std::to_string(l) + "x"); }
            } while (left > 0);
        }
    }
    return MGB200_OK;
}

// residual ; compute_norm on level 0 (multigrid.cpp:112-113) -> d_norm2[0]
int mgb200_solver::residual_norm_level0()
{
    Level& g = lv[0];
    if (batch > 0) {
        // a batched handle with one level: every member's norm (a frozen member's comes out as before: its u and rhs
        // are unchanged), then the active members' sums
        for (int b = 0; b < batch; ++b)
            MGB_TRY(launch_residual(nullptr, g.u[g.cur] + (size_t)b * g.elems, g.rhs + (size_t)b * g.elems, g.v1 + (size_t)b * g.elems,
                                    g.v2 + (size_t)b * g.elems, g.n, g.L, g.st, opt.arith, d_partials + (size_t)b * pstride, stream));
        return launch_reduce_partials_batched(d_partials, residual_partials_count(g.n), pstride, d_norm2, d_active, batch, stream);
    }
    MGB_TRY(launch_residual(nullptr, g.u[g.cur], g.rhs, g.v1, g.v2, g.n, g.L, g.st, opt.arith, d_partials, stream));
    MGB_TRY(launch_reduce_partials(d_partials, residual_partials_count(g.n), d_norm2, stream));
    return MGB200_OK;
}

int mgb200_solver::record_cycle()
{
    mark("start");
    MGB_TRY(cycle_body(0));
    if (opt.plan == MGB200_PLAN_FUSED && maxlvl > 1) {
        // the level-0 up leg already produced the per-tile sums of squares (its LAST chunk did)
        const int last_k = opt.niter == 0 ? 0 : ((opt.niter - 1) % 3) + 1;
        if (batch > 0) {
            MGB_TRY(launch_reduce_partials_batched(d_partials, stream_pass_tiles(N, N + 1, last_k, batch), pstride, d_norm2, d_active, batch, stream));
            return MGB200_OK;
        }
        MGB_TRY(launch_reduce_partials(d_partials, stream_pass_tiles(N, lv[0].own_hi - lv[0].own_lo + 1, last_k), d_norm2, stream));
        MGB_TRY(allreduce_norm());
        mark("norm");
    } else {
        MGB_TRY(residual_norm_level0());
    }
    return MGB200_OK;
}

int mgb200_solver::run_cycle_async()
{
    if (!have_rhs) return fail(MGB200_ERR_STATE, "cycle before form_rhs");
    if (!res0_on_host && norm_is_res0) { MGB_TRY(read_norm(&res0)); res0_on_host = true; }
    norm_is_res0 = false;
    if (!opt.use_graph) {
        const long before = launch_counter();
        MGB_TRY(record_cycle());
        count(before);
        dump_marks();
        return MGB200_OK;
    }
    if (!graph_exec) {
        // every level's `cur` returns to its starting value after one cycle (two flips per
        // level per repetition), so one captured graph is valid for every later cycle
        std::vector<int> cur0;
        for (auto& g : lv) cur0.push_back(g.cur);
        cudaGraph_t graph = nullptr;
        const long before = launch_counter();
        MGB_CUDA(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
        int rc = record_cycle();
        cudaError_t e = cudaStreamEndCapture(stream, &graph);
        graph_kernels = launch_counter() - before;
        launch_counter() = before;      // captured, not launched
        if (rc != MGB200_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (e != cudaSuccess) return fail(MGB200_ERR_CUDA, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e));
        for (size_t l = 0; l < lv.size(); ++l)
            if (lv[l].cur != cur0[l]) { cudaGraphDestroy(graph); return fail(MGB200_ERR_STATE, "cycle does not restore buffer parity"); }
        e = cudaGraphInstantiate(&graph_exec, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) return fail(MGB200_ERR_CUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e));
    }
    MGB_CUDA(cudaGraphLaunch(graph_exec, stream));
    launches += graph_kernels;
    return MGB200_OK;
}

// mg_outer as ONE graph: [k_loop_begin] -> WHILE { cycle ; k_loop_check }.  The host launches it
// once per time step and reads the loop state afterwards; no round trip per cycle.
int mgb200_solver::build_loop_graph()
{
    std::vector<int> cur0;
    for (auto& g : lv) cur0.push_back(g.cur);
    cudaGraph_t graph = nullptr;
    auto bail = [&](const char* what, cudaError_t e) {
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        loop_failed = true;
        return fail(MGB200_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
    };
    cudaError_t e = cudaGraphCreate(&graph, 0);
    if (e != cudaSuccess) return bail("cudaGraphCreate", e);
    cudaGraphConditionalHandle h;
    e = cudaGraphConditionalHandleCreate(&h, graph, 0, 0);
    if (e != cudaSuccess) return bail("cudaGraphConditionalHandleCreate", e);
    cudaKernelNodeParams kp{};
    double tol_ = tol; int maxc = opt.max_cycle, nmb = batch;
    void* args[] = {&h, &d_norm2, &d_loop, &tol_, &maxc};
    void* bargs[] = {&h, &d_norm2, &d_loop, &d_active, &tol_, &maxc, &nmb};
    kp.func = (void*)k_loop_begin; kp.gridDim = dim3(1); kp.blockDim = dim3(1); kp.kernelParams = args;
    if (batch > 0) { kp.func = (void*)k_loop_begin_batched; kp.blockDim = dim3(1024); kp.kernelParams = bargs; }
    cudaGraphNode_t n_begin, n_while;
    e = cudaGraphAddKernelNode(&n_begin, graph, nullptr, 0, &kp);
    if (e != cudaSuccess) return bail("cudaGraphAddKernelNode", e);
    cudaGraphNodeParams cp{};
    cp.type = cudaGraphNodeTypeConditional;
    cp.conditional.handle = h; cp.conditional.type = cudaGraphCondTypeWhile; cp.conditional.size = 1;
    e = cudaGraphAddNode(&n_while, graph, &n_begin, 1, &cp);
    if (e != cudaSuccess) return bail("cudaGraphAddNode(conditional)", e);
    cudaGraph_t body = cp.conditional.phGraph_out[0];
    const long before = launch_counter();
    e = cudaStreamBeginCaptureToGraph(stream, body, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal);
    if (e != cudaSuccess) return bail("cudaStreamBeginCaptureToGraph", e);
    int rc = record_cycle();
    if (rc == MGB200_OK && batch > 0) { k_loop_check_batched<<<1, 1024, 0, stream>>>(h, d_norm2, d_loop, d_active, batch); rc = check_launch("k_loop_check_batched"); }
    else if (rc == MGB200_OK) { k_loop_check<<<1, 1, 0, stream>>>(h, d_norm2, d_loop); rc = check_launch("k_loop_check"); }
    cudaGraph_t captured = nullptr;
    e = cudaStreamEndCapture(stream, &captured);
    loop_kernels = launch_counter() - before;
    launch_counter() = before;          // captured, not launched
    if (rc != MGB200_OK) { cudaGraphDestroy(graph); loop_failed = true; return rc; }
    if (e != cudaSuccess) return bail("cudaStreamEndCapture(loop body)", e);
    for (size_t l = 0; l < lv.size(); ++l)
        if (lv[l].cur != cur0[l]) { cudaGraphDestroy(graph); loop_failed = true; return fail(MGB200_ERR_STATE, "cycle does not restore buffer parity"); }
    e = cudaGraphInstantiate(&loop_exec, graph, 0);
    if (e != cudaSuccess) { loop_exec = nullptr; return bail("cudaGraphInstantiate(loop)", e); }
    cudaGraphDestroy(graph);
    return MGB200_OK;
}

int mgb200_solver::read_norm(double* out)
{
    MGB_CUDA(cudaMemcpyAsync(h_norm2, d_norm2, sizeof(double), cudaMemcpyDeviceToHost, stream));
    MGB_CUDA(cudaStreamSynchronize(stream));
    res = std::sqrt(h_norm2[0]);                                                  // gs.cpp:106
    if (out) *out = res;
    return MGB200_OK;
}

// compute_rhs (multigrid.cpp:167) fused with the initial residual norm (multigrid.cpp:104-105)
int mgb200_solver::form_rhs(double* res0_out, bool sync)
{
    if (!have_fields) return fail(MGB200_ERR_STATE, "form_rhs before set_fields");
    Level& g = lv[0];
    const long before = launch_counter();
    if (batch > 0) {
        MGB_TRY(activate_all());
        MGB_TRY(launch_compute_rhs_batched(g.rhs, g.u[g.cur], g.v1, g.v2, g.n, g.L, g.st, opt.arith, d_partials, pstride, batch, (long)g.elems, stream));
        MGB_TRY(launch_reduce_partials_batched(d_partials, compute_rhs_partials_count(g.n, g.n - 1, g.L), pstride, d_norm2, nullptr, batch, stream));
        count(before);
        have_rhs = true;
        norm_is_res0 = true; res0_on_host = false;
        if (!sync) return MGB200_OK;
        MGB_TRY(read_norms(res0_out));
        res0_b = res_b;
        res0_on_host = true;
        return MGB200_OK;
    }
    if (P == 1) {
        MGB_TRY(launch_compute_rhs(g.rhs, g.u[g.cur], g.v1, g.v2, g.n, g.L, g.st, opt.arith, d_partials, stream));
        MGB_TRY(launch_reduce_partials(d_partials, compute_rhs_partials_count(g.n, g.n - 1, g.L), d_norm2, stream));
    } else {
        const long ilo = g.own_lo < 1 ? 1 : g.own_lo, ihi = g.own_hi > g.n - 1 ? g.n - 1 : g.own_hi;
        MGB_TRY(launch_compute_rhs(g.rhs, g.u[g.cur], g.v1, g.v2, g.n, g.L, g.st, opt.arith, d_partials, stream, ilo, ihi));
        MGB_TRY(launch_reduce_partials(d_partials, compute_rhs_partials_count(g.n, ihi - ilo + 1, g.L), d_norm2, stream));
        MGB_TRY(allreduce_norm());
        MGB_TRY(exchange_halo(g, g.rhs));
    }
    count(before);
    have_rhs = true;
    norm_is_res0 = true; res0_on_host = false;
    if (!sync) return MGB200_OK;       // the device-side loop takes res0 from d_norm2 itself
    MGB_TRY(read_norm(&res0));
    res0_on_host = true;
    if (res0_out) *res0_out = res0;
    return MGB200_OK;
}

namespace mgb200 {
bool report_solve(int cycles, int max_cycle, double res0, double res, double tol)
{
    const bool finite = std::isfinite(res) && std::isfinite(res0);
    const bool ok = finite && (res / res0 <= tol || res0 == 0.0);
    if (ok) return true;
    static const bool quiet = [] { const char* e = getenv("MGB200_QUIET"); return e && atoi(e) != 0; }();
    if (!quiet) {
        if (!finite) fprintf(stderr, "mgb200: residual norm is not finite after %d cycle(s) (res0 = %g, res = %g): the iteration diverged\n", cycles, res0, res);
        else fprintf(stderr, "multigrid did not converge in %d cycles (res/res0 = %.3e > tol = %.3e)\n", max_cycle, res / res0, tol);   // multigrid.cpp:118
    }
    return false;
}
}  // namespace mgb200

void mgb200_solver::fill_pass_batch(StreamPassArgs& a, const Level& g, const Level& c) const
{
    if (batch == 0) return;
    a.members = batch; a.mstride = (long)g.elems; a.cmstride = (long)c.elems; a.pstride = pstride; a.active = d_active;
}

int mgb200_solver::activate_all()
{
    k_fill_int<<<(batch + 255) / 256, 256, 0, stream>>>(d_active, batch, 1);
    return check_launch("k_fill_int");
}

// every member's current norm -> res_b (and out[0..batch) if given)
int mgb200_solver::read_norms(double* out)
{
    MGB_CUDA(cudaMemcpyAsync(h_norm2, d_norm2, (size_t)batch * sizeof(double), cudaMemcpyDeviceToHost, stream));
    MGB_CUDA(cudaStreamSynchronize(stream));
    for (int b = 0; b < batch; ++b) {
        res_b[b] = std::sqrt(h_norm2[b]);                                         // gs.cpp:106
        if (out) out[b] = res_b[b];
    }
    return MGB200_OK;
}

static void fill_info(mgb200_solve_info* info, const LoopState& ls, double tol)
{
    const int it = ls.iter;
    std::memset(info, 0, sizeof(*info));
    for (int k = 0; k <= it; ++k) info->hist[k] = ls.hist[k];
    info->cycles = it; info->res0 = ls.res0; info->res = ls.hist[it]; info->converged = (info->res / info->res0 <= tol) ? 1 : 0;
}

// mg_outer for every member of a batch: each member runs its own loop (multigrid.cpp:108) and is frozen once its
// condition fails; the cycles go on while any member runs.  infos: `batch` entries (may be null).
int mgb200_solver::solve_batched(mgb200_solve_info* infos)
{
    if (!have_rhs) return fail(MGB200_ERR_STATE, "solve before form_rhs");
    if (device_loop() && norm_is_res0 && !loop_exec) {
        if (build_loop_graph() != MGB200_OK)
            fprintf(stderr, "mgb200: device-side solve loop unavailable (%s); using the host loop\n", mgb200_last_error());
    }
    if (device_loop() && norm_is_res0 && loop_exec) {
        MGB_CUDA(cudaGraphLaunch(loop_exec, stream));
        MGB_CUDA(cudaMemcpyAsync(h_loop, d_loop, (size_t)batch * sizeof(LoopState), cudaMemcpyDeviceToHost, stream));
        MGB_CUDA(cudaStreamSynchronize(stream));
        norm_is_res0 = false; res0_on_host = true;
        int trips = 0;
        for (int b = 0; b < batch; ++b) {
            const LoopState& ls = h_loop[b];
            trips = std::max(trips, ls.iter);
            res0_b[b] = ls.res0; res_b[b] = ls.hist[ls.iter];
            if (infos) fill_info(&infos[b], ls, tol);
            report_solve(ls.iter, opt.max_cycle, ls.res0, ls.hist[ls.iter], tol);
        }
        launches += 1 + (long)trips * loop_kernels;
        return MGB200_OK;
    }
    if (!res0_on_host) {
        if (!norm_is_res0) return fail(MGB200_ERR_STATE, "solve: initial residual norm unknown; call form_rhs first");
        MGB_TRY(read_norms(nullptr));
        res0_b = res_b;
        res0_on_host = true;
    }
    std::vector<LoopState> ls((size_t)batch);
    for (int b = 0; b < batch; ++b) {
        ls[b].res0 = res0_b[b]; ls[b].iter = 0; ls[b].hist[0] = res0_b[b];
        res_b[b] = res0_b[b];
    }
    std::vector<double> r(res0_b);
    for (;;) {                                                                    // :108, per member
        bool any = false;
        for (int b = 0; b < batch; ++b) {
            h_active[b] = (ls[b].iter < opt.max_cycle && r[b] / res0_b[b] > tol) ? 1 : 0;
            any = any || h_active[b];
        }
        if (!any) break;
        MGB_CUDA(cudaMemcpyAsync(d_active, h_active, (size_t)batch * sizeof(int), cudaMemcpyHostToDevice, stream));
        MGB_TRY(run_cycle_async());                                               // :110-112
        MGB_TRY(read_norms(nullptr));                                             // :113
        for (int b = 0; b < batch; ++b)
            if (h_active[b]) { r[b] = res_b[b]; ls[b].hist[++ls[b].iter] = r[b]; }
    }
    for (int b = 0; b < batch; ++b) {
        if (infos) fill_info(&infos[b], ls[b], tol);
        report_solve(ls[b].iter, opt.max_cycle, res0_b[b], r[b], tol);
    }
    return MGB200_OK;
}

// nsteps x { compute_rhs ; mg_outer } for every member; infos: nsteps x batch entries, step-major
int mgb200_solver::timestep_batched(int nsteps, mgb200_solve_info* infos)
{
    if (nsteps <= 0) return MGB200_OK;
    int k0 = 0;
    if (device_loop() && !loop_exec) {
        MGB_TRY(form_rhs(nullptr, false));
        MGB_TRY(solve_batched(infos));
        k0 = 1;
    }
    if (!(device_loop() && loop_exec)) {
        for (int k = k0; k < nsteps; ++k) {
            MGB_TRY(form_rhs(nullptr, false));
            MGB_TRY(solve_batched(infos ? infos + (size_t)k * batch : nullptr));
        }
        return MGB200_OK;
    }
    const int todo = nsteps - k0;
    if (todo <= 0) return MGB200_OK;
    const long need = (long)todo * batch;
    if (h_steps_cap < need) {
        if (h_steps) cudaFreeHost(h_steps);
        h_steps = nullptr; h_steps_cap = 0;
        MGB_CUDA(cudaMallocHost(&h_steps, (size_t)need * sizeof(LoopState)));
        h_steps_cap = (int)need;
    }
    for (int k = 0; k < todo; ++k) {
        MGB_TRY(form_rhs(nullptr, false));
        MGB_CUDA(cudaGraphLaunch(loop_exec, stream));
        MGB_CUDA(cudaMemcpyAsync(&h_steps[(size_t)k * batch], d_loop, (size_t)batch * sizeof(LoopState), cudaMemcpyDeviceToHost, stream));
    }
    MGB_CUDA(cudaStreamSynchronize(stream));
    norm_is_res0 = false; res0_on_host = true;
    for (int k = 0; k < todo; ++k) {
        int trips = 0;
        for (int b = 0; b < batch; ++b) {
            const LoopState& ls = h_steps[(size_t)k * batch + b];
            trips = std::max(trips, ls.iter);
            res0_b[b] = ls.res0; res_b[b] = ls.hist[ls.iter];
            if (infos) fill_info(&infos[(size_t)(k0 + k) * batch + b], ls, tol);
            report_solve(ls.iter, opt.max_cycle, ls.res0, ls.hist[ls.iter], tol);
        }
        launches += 1 + (long)trips * loop_kernels;
    }
    return MGB200_OK;
}

// mg_outer (multigrid.cpp:97-120)
int mgb200_solver::solve(mgb200_solve_info* info)
{
    if (batch > 0) return solve_batched(info);
    if (!have_rhs) return fail(MGB200_ERR_STATE, "solve before form_rhs");
    if (device_loop() && norm_is_res0 && !loop_exec) {
        // every rank takes the same decision: the capture works everywhere or nowhere
        if (build_loop_graph() != MGB200_OK) {
            fprintf(stderr, "mgb200: device-side solve loop unavailable (%s); using the host loop\n", mgb200_last_error());
            if (P > 1) return MGB200_ERR_CUDA;
        }
    }
    if (device_loop() && norm_is_res0 && loop_exec) {
        // d_norm2[0] still holds ||r0||^2 from form_rhs (multigrid.cpp:104-105)
        MGB_CUDA(cudaGraphLaunch(loop_exec, stream));
        MGB_CUDA(cudaMemcpyAsync(h_loop, d_loop, sizeof(LoopState), cudaMemcpyDeviceToHost, stream));
        MGB_CUDA(cudaStreamSynchronize(stream));
        norm_is_res0 = false; res0_on_host = true;
        const int it = h_loop->iter;
        launches += 1 + (long)it * loop_kernels;
        res0 = h_loop->res0; res = h_loop->hist[it];
        if (info) {
            std::memset(info, 0, sizeof(*info));
            for (int k = 0; k <= it; ++k) info->hist[k] = h_loop->hist[k];
            info->cycles = it; info->res0 = res0; info->res = res; info->converged = (res / res0 <= tol) ? 1 : 0;
        }
        if (rank == 0) report_solve(it, opt.max_cycle, res0, res, tol);
        return check_peers();
    }
    if (!res0_on_host) {
        if (!norm_is_res0) return fail(MGB200_ERR_STATE, "solve: initial residual norm unknown; call form_rhs first");
        MGB_TRY(read_norm(&res0));
        res0_on_host = true;
    }
    double r0 = res0, r = res0;
    int it = 0;
    if (info) { std::memset(info, 0, sizeof(*info)); info->hist[0] = r0; }
    for (; it < opt.max_cycle && r / r0 > tol; ++it) {                            // :108
        MGB_TRY(run_cycle_async());                                               // :110-112
        MGB_TRY(read_norm(&r));                                                   // :113
        if (info) info->hist[it + 1] = r;
    }
    if (info) { info->cycles = it; info->res0 = r0; info->res = r; info->converged = (r / r0 <= tol) ? 1 : 0; }
    if (rank == 0) report_solve(it, opt.max_cycle, r0, r, tol);
    return MGB200_OK;
}

// the time loop (multigrid.cpp:165-172).  With the device-side solve loop nothing in a step needs
// the host: compute_rhs, the solve graph and an asynchronous copy of the loop state are enqueued for
// all steps back to back and the host synchronises once at the end.
int mgb200_solver::timestep(int nsteps, mgb200_solve_info* infos)
{
    if (batch > 0) return timestep_batched(nsteps, infos);
    if (nsteps <= 0) return MGB200_OK;
    int k0 = 0;
    if (device_loop() && !loop_exec) {
        // first use: the graph is captured inside solve(), after the first compute_rhs
        MGB_TRY(form_rhs(nullptr, false));                                        // :167
        MGB_TRY(solve(infos ? &infos[0] : nullptr));                              // :169
        k0 = 1;
    }
    if (!(device_loop() && loop_exec)) {
        for (int k = k0; k < nsteps; ++k) {
            MGB_TRY(form_rhs(nullptr, false));
            MGB_TRY(solve(infos ? &infos[k] : nullptr));
        }
        return MGB200_OK;
    }
    const int todo = nsteps - k0;
    if (todo <= 0) return MGB200_OK;
    if (h_steps_cap < todo) {
        if (h_steps) cudaFreeHost(h_steps);
        h_steps = nullptr; h_steps_cap = 0;
        MGB_CUDA(cudaMallocHost(&h_steps, (size_t)todo * sizeof(LoopState)));
        h_steps_cap = todo;
    }
    for (int k = 0; k < todo; ++k) {
        MGB_TRY(form_rhs(nullptr, false));
        MGB_CUDA(cudaGraphLaunch(loop_exec, stream));
        MGB_CUDA(cudaMemcpyAsync(&h_steps[k], d_loop, sizeof(LoopState), cudaMemcpyDeviceToHost, stream));
    }
    MGB_CUDA(cudaStreamSynchronize(stream));
    norm_is_res0 = false; res0_on_host = true;
    for (int k = 0; k < todo; ++k) {
        const LoopState& ls = h_steps[k];
        const int it = ls.iter;
        launches += 1 + (long)it * loop_kernels;
        res0 = ls.res0; res = ls.hist[it];
        if (infos) {
            mgb200_solve_info& info = infos[k0 + k];
            std::memset(&info, 0, sizeof(info));
            for (int c = 0; c <= it; ++c) info.hist[c] = ls.hist[c];
            info.cycles = it; info.res0 = res0; info.res = res; info.converged = (res / res0 <= tol) ? 1 : 0;
        }
        if (rank == 0) report_solve(it, opt.max_cycle, res0, res, tol);
    }
    return check_peers();
}

int mgb200_solver::get_u_natural(double* dst_dev, long ld)
{
    Level& g = lv[0];
    const long before = launch_counter();
    // a slab rank fills its own rows only (the destination is a full-size array); member b of a batch at + b (n+1) ld
    for (int b = 0; b < members(); ++b)
        MGB_TRY(launch_convert(dst_dev + (size_t)b * (g.n + 1) * ld, natural_layout(ld), g.u[g.cur] + (size_t)b * g.elems, g.L, g.n, stream,
                               g.own_lo, g.own_hi));
    count(before);
    return MGB200_OK;
}

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

int mgb200_version(void) { return MGB200_VERSION; }
const char* mgb200_last_error(void) { return g_last_error.c_str(); }

void mgb200_default_options(mgb200_options* o)
{
    std::memset(o, 0, sizeof(*o));
    o->struct_size = (int)sizeof(mgb200_options);
    o->shape = 1;
    o->niter = 3;
    o->coarse_maxit = 1000;
    o->coarse_tol = 1e-5;
    o->max_cycle = 50;
    o->arith = MGB200_ARITH_FAST;
    o->plan = MGB200_PLAN_FUSED;
    o->correct_towers = 0;
    o->use_graph = 1;
    o->device = -1;
}

int mgb200_create(mgb200_solver** out, long n, int maxlvl, double nu, double dt, double dx, double tol,
                  const mgb200_options* opt)
{
    if (!out) return fail(MGB200_ERR_INVALID, "out == NULL");
    *out = nullptr;
    mgb200_solver* s = new mgb200_solver();
    int rc = s->init(n, maxlvl, nu, dt, dx, tol, opt);
    if (rc != MGB200_OK) { delete s; return rc; }
    *out = s;
    return MGB200_OK;
}

int mgb200_create_batched(mgb200_solver** out, long n, int maxlvl, int batch, double nu, double dt, double dx, double tol,
                          const mgb200_options* opt)
{
    if (!out) return fail(MGB200_ERR_INVALID, "out == NULL");
    *out = nullptr;
    if (batch < 1) return fail(MGB200_ERR_INVALID, "create_batched: batch must be >= 1");
    mgb200_solver* s = new mgb200_solver();
    s->batch = batch;
    int rc = s->init(n, maxlvl, nu, dt, dx, tol, opt);
    if (rc != MGB200_OK) { delete s; return rc; }
    *out = s;
    return MGB200_OK;
}

int mgb200_batch_size(mgb200_solver* s) { return s ? s->members() : 0; }

int mgb200_comm_unique_id(unsigned char id[128]) { return comm_unique_id(id); }

int mgb200_create_sharded(mgb200_solver** out, long n, int maxlvl, double nu, double dt, double dx, double tol,
                          const mgb200_options* opt, int rank, int nranks, const unsigned char id[128], long shard_min_rows)
{
    if (!out) return fail(MGB200_ERR_INVALID, "out == NULL");
    *out = nullptr;
    if (nranks < 1 || (nranks & (nranks - 1)) || rank < 0 || rank >= nranks)
        return fail(MGB200_ERR_INVALID, "create_sharded: nranks must be a power of two, 0 <= rank < nranks");
    mgb200_solver* s = new mgb200_solver();
    s->rank = rank; s->P = nranks;
    if (shard_min_rows > 0) s->shard_min_rows = shard_min_rows;
    int rc = MGB200_OK;
    if (nranks > 1) {
        if (opt && opt->device >= 0) cudaSetDevice(opt->device);   // the communicator binds to the current device
        rc = comm_create(&s->comm, rank, nranks, id);
    }
    if (rc == MGB200_OK) rc = s->init(n, maxlvl, nu, dt, dx, tol, opt);
    if (rc != MGB200_OK) { delete s; return rc; }
    *out = s;
    return MGB200_OK;
}

int mgb200_slab_plan(long n, int maxlvl, int nranks, int rank, long shard_min_rows, int lvl, long out[6])
{
    // the window alloc_levels gives `rank` at level `lvl`.  out = {sharded, present, own_lo, own_hi, mem_lo, mem_hi}
    if (!out || lvl < 0 || lvl >= maxlvl || nranks < 1 || rank < 0 || rank >= nranks) return fail(MGB200_ERR_INVALID, "slab_plan: bad argument");
    if (shard_min_rows <= 0) shard_min_rows = 256;
    const Window w = slab_window(n, maxlvl, nranks, rank, shard_min_rows, lvl);
    out[0] = w.sharded; out[1] = w.present; out[2] = w.rows.own_lo; out[3] = w.rows.own_hi; out[4] = w.rows.mem_lo; out[5] = w.rows.mem_hi;
    return MGB200_OK;
}

int mgb200_slab(mgb200_solver* s, int lvl, long out[6])
{
    if (!s || !out || lvl < 0 || lvl >= s->maxlvl) return fail(MGB200_ERR_INVALID, "slab: bad argument");
    const Level& g = s->lv[lvl];
    out[0] = g.sharded; out[1] = g.present; out[2] = g.own_lo; out[3] = g.own_hi; out[4] = g.mem_lo; out[5] = g.mem_hi;
    return MGB200_OK;
}

int mgb200_destroy(mgb200_solver* s)
{
    if (!s) return MGB200_OK;
    cudaSetDevice(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    delete s;
    return MGB200_OK;
}

static int after_fields(mgb200_solver* s)
{
    MGB_TRY(s->build_towers());
    if (s->opt.coarse_exact && (s->P == 1 || s->rank == 0)) {
        // the coarsest operator depends on the (new) velocities only: factor it once
        Level& c = s->lv[s->maxlvl - 1];
        if (!s->d_coarse_lu) MGB_CUDA(cudaMalloc(&s->d_coarse_lu, coarse_lu_bytes(c.n) * s->members()));
        for (int b = 0; b < s->members(); ++b)                  // (a batch: one factorisation per member)
            MGB_TRY(launch_coarse_lu_factor(s->d_coarse_lu + b * (coarse_lu_bytes(c.n) / sizeof(double)), c.v1 + (size_t)b * c.elems,
                                            c.v2 + (size_t)b * c.elems, c.n, c.L, c.st, s->stream));
    }
    if (s->P > 1) {                    // the tower inputs are no longer needed
        MGB_CUDA(cudaStreamSynchronize(s->stream));
        for (auto& t : s->d_top) { cudaFree(t); t = nullptr; }
        cudaFree(s->d_flat[0]); cudaFree(s->d_flat[1]); s->d_flat[0] = s->d_flat[1] = nullptr;
    }
    s->have_fields = true;
    s->have_rhs = false;
    return MGB200_OK;
}

int mgb200_set_fields_device(mgb200_solver* s, const double* u0, const double* v1, const double* v2, long ld)
{
    if (!s || !u0 || !v1 || !v2 || ld < s->N + 1) return fail(MGB200_ERR_INVALID, "set_fields_device: bad argument");
    Level& g = s->lv[0];
    const long before = launch_counter();
    // (slab ranks take the rows of their window out of the full-size arrays; member b of a batch is at + b (n+1) ld)
    for (int b = 0; b < s->members(); ++b) {
        const size_t mo = (size_t)b * g.elems, io = (size_t)b * (g.n + 1) * ld;
        MGB_TRY(launch_convert(g.u[g.cur] + mo, g.L, u0 + io, natural_layout(ld), g.n, s->stream, g.mem_lo, g.mem_hi));
        MGB_TRY(launch_convert(g.v1 + mo, g.L, v1 + io, natural_layout(ld), g.n, s->stream, g.mem_lo, g.mem_hi));
        MGB_TRY(launch_convert(g.v2 + mo, g.L, v2 + io, natural_layout(ld), g.n, s->stream, g.mem_lo, g.mem_hi));
    }
    if (s->P > 1) {
        MGB_TRY(s->alloc_top());
        const long top = s->N / 4 + 1;
        MGB_TRY(launch_convert(s->d_top[1], natural_layout(s->N + 1), v1, natural_layout(ld), s->N, s->stream, 0, top));
        MGB_TRY(launch_convert(s->d_top[2], natural_layout(s->N + 1), v2, natural_layout(ld), s->N, s->stream, 0, top));
    }
    MGB_TRY(after_fields(s));
    s->count(before);
    MGB_CUDA(cudaStreamSynchronize(s->stream));     // the caller may free its arrays on return
    return MGB200_OK;
}

int mgb200_set_fields_host(mgb200_solver* s, const double* u0, const double* v1, const double* v2)
{
    if (!s || !u0 || !v1 || !v2) return fail(MGB200_ERR_INVALID, "set_fields_host: bad argument");
    Level& g = s->lv[0];
    const long n = g.n;
    // rows of this rank's window (all rows on a single GPU), dense in the host arrays
    const size_t off = (size_t)g.mem_lo * (n + 1);
    const size_t bytes = (size_t)g.rows_mem() * (n + 1) * sizeof(double);
    const Layout dense = natural_layout(n + 1, g.mem_lo);
    // two staging areas (both larger than a dense window): the idle twin of u and the rhs array
    double* stage_a = g.u[1 - g.cur];
    double* stage_b = g.rhs;
    const long before = launch_counter();
    // Coarse-velocity towers of a sharded solver (P1): every rank needs rows 0..N/4+1 of the level-0 velocities.
    // Each of those rows crosses PCIe ONCE, inside the window of the rank that owns it; the owner copies it from
    // its staging area into the dense tower input and broadcasts it to the other ranks over NVLink.
    const long top = s->N / 4 + 1;
    auto towers_from_stage = [&](double* stage, double* dtop) -> int {
        const long a = g.own_lo, b = g.own_hi < top ? g.own_hi : top;
        if (a <= b)
            MGB_CUDA(cudaMemcpyAsync(dtop + (size_t)a * (n + 1), stage + (size_t)(a - g.mem_lo) * (n + 1), (size_t)(b - a + 1) * (n + 1) * sizeof(double),
                                     cudaMemcpyDeviceToDevice, s->stream));
        for (int r = 0; r < s->P; ++r) {
            const Slab w = slab_of(g.n, s->P, r);
            const long ra = w.own_lo, rb = w.own_hi < top ? w.own_hi : top;
            if (ra <= rb) MGB_TRY(comm_broadcast(s->comm, dtop + (size_t)ra * (n + 1), (size_t)(rb - ra + 1) * (n + 1), r, s->stream));
        }
        return MGB200_OK;
    };
    if (s->P > 1) MGB_TRY(s->alloc_top());
    if (s->batch > 0) {
        // member b: host arrays at + b (n+1)^2, staged through its own idle twin and rhs
        for (int b = 0; b < s->batch; ++b) {
            const size_t mo = (size_t)b * g.elems, ho = (size_t)b * (n + 1) * (n + 1);
            MGB_CUDA(cudaMemcpyAsync(stage_a + mo, u0 + ho, bytes, cudaMemcpyHostToDevice, s->stream));
            MGB_TRY(launch_convert(g.u[g.cur] + mo, g.L, stage_a + mo, dense, n, s->stream));
            MGB_CUDA(cudaMemcpyAsync(stage_b + mo, v1 + ho, bytes, cudaMemcpyHostToDevice, s->stream));
            MGB_TRY(launch_convert(g.v1 + mo, g.L, stage_b + mo, dense, n, s->stream));
            MGB_CUDA(cudaMemcpyAsync(stage_a + mo, v2 + ho, bytes, cudaMemcpyHostToDevice, s->stream));
            MGB_TRY(launch_convert(g.v2 + mo, g.L, stage_a + mo, dense, n, s->stream));
        }
        MGB_CUDA(cudaMemsetAsync(stage_a, 0, g.elems * s->batch * sizeof(double), s->stream));
        MGB_CUDA(cudaMemsetAsync(stage_b, 0, g.elems * s->batch * sizeof(double), s->stream));
        MGB_TRY(after_fields(s));
        s->count(before);
        MGB_CUDA(cudaStreamSynchronize(s->stream));
        return MGB200_OK;
    }
    MGB_CUDA(cudaMemcpyAsync(stage_a, u0 + off, bytes, cudaMemcpyHostToDevice, s->stream));
    MGB_TRY(launch_convert(g.u[g.cur], g.L, stage_a, dense, n, s->stream, g.mem_lo, g.mem_hi));
    MGB_CUDA(cudaMemcpyAsync(stage_b, v1 + off, bytes, cudaMemcpyHostToDevice, s->stream));
    MGB_TRY(launch_convert(g.v1, g.L, stage_b, dense, n, s->stream, g.mem_lo, g.mem_hi));
    if (s->P > 1) MGB_TRY(towers_from_stage(stage_b, s->d_top[1]));
    MGB_CUDA(cudaMemcpyAsync(stage_a, v2 + off, bytes, cudaMemcpyHostToDevice, s->stream));
    MGB_TRY(launch_convert(g.v2, g.L, stage_a, dense, n, s->stream, g.mem_lo, g.mem_hi));
    if (s->P > 1) MGB_TRY(towers_from_stage(stage_a, s->d_top[2]));
    MGB_CUDA(cudaMemsetAsync(stage_a, 0, g.elems * sizeof(double), s->stream));
    MGB_CUDA(cudaMemsetAsync(stage_b, 0, g.elems * sizeof(double), s->stream));
    MGB_TRY(after_fields(s));
    s->count(before);
    MGB_CUDA(cudaStreamSynchronize(s->stream));
    return MGB200_OK;
}

int mgb200_set_fields_reference_ic(mgb200_solver* s, double vscale)
{
    if (!s) return fail(MGB200_ERR_INVALID, "solver == NULL");
    Level& g = s->lv[0];
    const long before = launch_counter();
    for (int b = 0; b < s->members(); ++b)      // (a batch: the same fields for every member)
        MGB_TRY(launch_initial_conditions(g.u[g.cur] + (size_t)b * g.elems, g.v1 + (size_t)b * g.elems, g.v2 + (size_t)b * g.elems, g.n, g.L,
                                          vscale, s->stream, g.mem_lo, g.mem_hi));
    if (s->P > 1) {
        MGB_TRY(s->alloc_top());
        MGB_TRY(launch_initial_conditions(s->d_top[0], s->d_top[1], s->d_top[2], g.n, natural_layout(g.n + 1), vscale, s->stream, 0, s->N / 4 + 1));
    }
    MGB_TRY(after_fields(s));
    s->count(before);
    return MGB200_OK;
}

int mgb200_form_rhs(mgb200_solver* s, double* res0)
{
    if (!s) return fail(MGB200_ERR_INVALID, "solver == NULL");
    return s->form_rhs(res0);
}

int mgb200_cycle(mgb200_solver* s, double* res)
{
    if (!s) return fail(MGB200_ERR_INVALID, "solver == NULL");
    if (s->batch > 0) {                 // every member cycles
        MGB_TRY(s->activate_all());
        MGB_TRY(s->run_cycle_async());
        return s->read_norms(res);
    }
    MGB_TRY(s->run_cycle_async());
    return s->read_norm(res);
}

int mgb200_cycle_async(mgb200_solver* s)
{
    if (!s) return fail(MGB200_ERR_INVALID, "solver == NULL");
    if (s->batch > 0) MGB_TRY(s->activate_all());
    return s->run_cycle_async();
}

int mgb200_last_norm(mgb200_solver* s, double* res)
{
    if (!s) return fail(MGB200_ERR_INVALID, "solver == NULL");
    if (s->batch > 0) return s->read_norms(res);
    return s->read_norm(res);
}

int mgb200_solve(mgb200_solver* s, mgb200_solve_info* info)
{
    if (!s) return fail(MGB200_ERR_INVALID, "solver == NULL");
    return s->solve(info);
}

int mgb200_timestep(mgb200_solver* s, int nsteps, mgb200_solve_info* infos)
{
    if (!s) return fail(MGB200_ERR_INVALID, "solver == NULL");
    return s->timestep(nsteps, infos);                                            // multigrid.cpp:165-172
}

int mgb200_get_u_device(mgb200_solver* s, double* u, long ld)
{
    if (!s || !u || ld < s->N + 1) return fail(MGB200_ERR_INVALID, "get_u_device: bad argument");
    MGB_TRY(s->get_u_natural(u, ld));
    MGB_CUDA(cudaStreamSynchronize(s->stream));
    return MGB200_OK;
}

int mgb200_get_u_host(mgb200_solver* s, double* u)
{
    if (!s || !u) return fail(MGB200_ERR_INVALID, "get_u_host: bad argument");
    Level& g = s->lv[0];
    // dense staging of the OWNED rows (a slab rank fills only its rows of the full-size host array); member b of a
    // batch goes to + b (n+1)^2, staged in its own idle twin
    const long before = launch_counter();
    for (int b = 0; b < s->members(); ++b) {
        double* stage = g.u[1 - g.cur] + (size_t)b * g.elems;      // idle between passes
        MGB_TRY(launch_convert(stage, natural_layout(g.n + 1, g.own_lo), g.u[g.cur] + (size_t)b * g.elems, g.L, g.n, s->stream, g.own_lo, g.own_hi));
        MGB_CUDA(cudaMemcpyAsync(u + (size_t)b * (g.n + 1) * (g.n + 1) + (size_t)g.own_lo * (g.n + 1), stage,
                                 (size_t)(g.own_hi - g.own_lo + 1) * (g.n + 1) * sizeof(double), cudaMemcpyDeviceToHost, s->stream));
    }
    s->count(before);
    MGB_CUDA(cudaStreamSynchronize(s->stream));
    // (the staging buffer is the next pass's output: every pass rewrites all owned rows of its output
    // and the exchange refreshes the halo rows, so nothing needs restoring)
    return MGB200_OK;
}

int mgb200_get_level_host(mgb200_solver* s, int lvl, int which, double* out)
{
    if (!s || !out || lvl < 0 || lvl >= s->maxlvl || which < 0 || which > 3) return fail(MGB200_ERR_INVALID, "get_level_host: bad argument");
    Level& g = s->lv[lvl];
    if (!g.present) return MGB200_OK;    // nothing of this level lives on this rank
    const double* src = which == 0 ? g.u[g.cur] : which == 1 ? g.rhs : which == 2 ? g.v1 : g.v2;
    double* tmp = nullptr;
    // the rows held by this rank (all rows on a single GPU) land in their place of the full-size array
    const size_t bytes = (size_t)g.rows_mem() * (g.n + 1) * sizeof(double);
    out += (size_t)g.mem_lo * (g.n + 1);
    MGB_CUDA(cudaMalloc(&tmp, bytes));
    int rc = MGB200_OK;
    for (int b = 0; b < s->members() && rc == MGB200_OK; ++b) {       // member b of a batch: + b (n_l+1)^2
        rc = launch_convert(tmp, natural_layout(g.n + 1, g.mem_lo), src + (size_t)b * g.elems, g.L, g.n, s->stream, g.mem_lo, g.mem_hi);
        if (rc == MGB200_OK) {
            cudaError_t e = cudaMemcpyAsync(out + (size_t)b * (g.n + 1) * (g.n + 1), tmp, bytes, cudaMemcpyDeviceToHost, s->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
            if (e != cudaSuccess) rc = fail(MGB200_ERR_CUDA, cudaGetErrorString(e));
        }
    }
    cudaFree(tmp);
    return rc;
}

int mgb200_synchronize(mgb200_solver* s)
{
    if (!s) return fail(MGB200_ERR_INVALID, "solver == NULL");
    MGB_CUDA(cudaStreamSynchronize(s->stream));
    return s->check_peers();
}

void* mgb200_stream(mgb200_solver* s) { return s ? (void*)s->stream : nullptr; }
long mgb200_kernel_launches(mgb200_solver* s) { return s ? s->launches : 0; }

// DESIGN.md "bytes model": 8 B per node for every level-sized array a pass reads or writes,
// 2 B per fine node for an array of the next coarser level.
double mgb200_cycle_bytes(mgb200_solver* s)
{
    if (!s) return 0.0;
    double total = 0.0;
    for (int l = 0; l < s->maxlvl; ++l) {
        const double m = (double)(s->lv[l].n + 1) * (double)(s->lv[l].n + 1);
        const int reps = 1;   // shape repetitions multiply every coarser level
        double per_node;
        if (l == s->maxlvl - 1) {
            per_node = 40.0;  // one read of u,rhs,v1,v2 + one write of u; iterations stay on chip
        } else if (s->opt.plan == MGB200_PLAN_UNFUSED) {
            per_node = 2.0 * s->opt.niter * 40.0 + 40.0 + 4.0 + 2.0 + 26.0;   // GS pre/post, residual, inject, zero, prolong+add
        } else {
            const int chunks = s->opt.niter <= 3 ? 1 : (s->opt.niter + 2) / 3;
            const double down = (l > 0 ? 32.0 : 40.0) + 2.0 + (chunks - 1) * 40.0;  // u,rhs,v1,v2 in (u skipped when zero) + u out + coarse rhs
            const double up = 40.0 + 2.0 + (chunks - 1) * 40.0;                     // + coarse u in
            per_node = down + up;
        }
        double mult = 1.0;
        for (int k = 0; k < l; ++k) mult *= s->opt.shape;
        total += per_node * m * mult * reps;
    }
    if (s->opt.plan == MGB200_PLAN_UNFUSED || s->maxlvl == 1) total += 32.0 * (double)(s->N + 1) * (double)(s->N + 1);
    return total * s->members();        // a batch: every member's cycle
}

int mgb200_profile_level0(mgb200_solver* s, int reps, double* ms_a, double* bytes_a, double* ms_b, double* bytes_b)
{
    if (!s || reps < 1 || !s->have_rhs) return fail(MGB200_ERR_STATE, "profile_level0: needs a formed rhs");
    if (s->maxlvl < 2) return fail(MGB200_ERR_INVALID, "profile_level0: needs at least two levels");
    Level& g = s->lv[0];
    Level& c = s->lv[1];
    const double m0 = (double)(g.own_hi - g.own_lo + 1) * (double)(g.n + 1) * s->members();   // nodes this rank produces (every member)
    if (s->batch > 0) MGB_TRY(s->activate_all());
    cudaEvent_t e0, e1;
    MGB_CUDA(cudaEventCreate(&e0));
    MGB_CUDA(cudaEventCreate(&e1));
    double acc[2] = {0.0, 0.0};
    const long before = launch_counter();
    int rc = MGB200_OK;
    for (int which = 0; which < 2 && rc == MGB200_OK; ++which) {
        for (int r = 0; r < reps && rc == MGB200_OK; ++r) {
            cudaEventRecord(e0, s->stream);
            if (s->opt.plan == MGB200_PLAN_FUSED) {
                StreamPassArgs a{};
                a.n = g.n; a.L = g.L; a.st = g.st; a.arith = s->opt.arith;
                a.u_in = g.u[g.cur]; a.u_out = g.u[1 - g.cur];
                a.rhs = g.rhs; a.v1 = g.v1; a.v2 = g.v2;
                a.iters = s->opt.niter > 3 ? 3 : s->opt.niter;
                a.Lc = c.L;
                if (which == 0) { a.post = s->opt.restriction == MGB200_RESTRICT_FW ? POST_FW : POST_INJECT; a.coarse_rhs = c.rhs; }
                else { a.coarse_u = c.u[c.cur]; a.post = POST_NORM2; a.partials = s->d_partials; }
                s->fill_pass_window(a, g, c);
                s->fill_pass_batch(a, g, c);
                rc = stream_pass(a, s->stream);
                g.cur = 1 - g.cur;
            } else if (which == 0) {
                rc = launch_gs_colour(g.u[g.cur], g.rhs, g.v1, g.v2, g.n, g.L, g.st, r & 1, s->opt.arith, s->stream);
            } else {
                rc = launch_residual(g.u[1 - g.cur], g.u[g.cur], g.rhs, g.v1, g.v2, g.n, g.L, g.st, s->opt.arith, nullptr, s->stream);
            }
            cudaEventRecord(e1, s->stream);
            cudaEventSynchronize(e1);
            float ms = 0.f;
            cudaEventElapsedTime(&ms, e0, e1);
            acc[which] += ms;
        }
    }
    s->count(before);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    MGB_TRY(rc);
    if (ms_a) *ms_a = acc[0] / reps;
    if (ms_b) *ms_b = acc[1] / reps;
    const bool fused = s->opt.plan == MGB200_PLAN_FUSED;
    if (bytes_a) *bytes_a = (fused ? 42.0 : 24.0) * m0;   // fused: u,rhs,v1,v2 in + u out + coarse rhs out; colour: u in, half of rhs,v1,v2 in, half of u out
    if (bytes_b) *bytes_b = (fused ? 42.0 : 40.0) * m0;   // fused: + coarse u in; residual: u,rhs,v1,v2 in + res out
    return MGB200_OK;
}

// The reference's timestepper allocates and frees its towers on every call (multigrid.cpp:138-162,
// 177-185).  Allocating and zero-filling ~14 GB of HBM per call would dominate an N=16384 call, so
// the one-call drivers keep the last handle alive and reuse it when the next call has the same
// shape and parameters; mgb200_release_cached() frees it, and with MGB200_TIMESTEPPER_CACHE=0 in the
// environment nothing is kept at all.
namespace {
struct CachedHandle {
    std::mutex mu;
    mgb200_solver* s = nullptr;
    long n = 0; int maxlvl = 0; double nu = 0, dt = 0, dx = 0, tol = 0;
    mgb200_options opt{};
};
CachedHandle g_cached;
}  // namespace

static int timestepper_common(double* uT, const double* u0, const double* v1, const double* v2, double nu, int maxlvl,
                              int n, double dt, double T, double dx, double tol, int shape, const mgb200_options* opt,
                              mgb200_solve_info* last, bool host)
{
    mgb200_options o;
    if (opt) o = *opt; else mgb200_default_options(&o);
    o.shape = shape;
    std::lock_guard<std::mutex> lock(g_cached.mu);
    const bool reuse = g_cached.s && g_cached.n == n && g_cached.maxlvl == maxlvl && g_cached.nu == nu && g_cached.dt == dt &&
                       g_cached.dx == dx && g_cached.tol == tol && std::memcmp(&g_cached.opt, &o, sizeof(o)) == 0;
    if (!reuse) {
        if (g_cached.s) { mgb200_destroy(g_cached.s); g_cached.s = nullptr; }
        MGB_TRY(mgb200_create(&g_cached.s, n, maxlvl, nu, dt, dx, tol, &o));
        g_cached.n = n; g_cached.maxlvl = maxlvl; g_cached.nu = nu; g_cached.dt = dt; g_cached.dx = dx; g_cached.tol = tol;
        g_cached.opt = o;
    }
    mgb200_solver* s = g_cached.s;
    MGB_CUDA(cudaSetDevice(s->device));
    int rc = host ? mgb200_set_fields_host(s, u0, v1, v2) : mgb200_set_fields_device(s, u0, v1, v2, n + 1);
    const int nsteps = (int)(T / dt);                                             // multigrid.cpp:165
    mgb200_solve_info info;
    std::memset(&info, 0, sizeof(info));
    if (rc == MGB200_OK && nsteps > 0) {
        std::vector<mgb200_solve_info> infos((size_t)nsteps);
        rc = s->timestep(nsteps, infos.data());
        if (rc == MGB200_OK) info = infos.back();
    }
    if (rc == MGB200_OK) rc = host ? mgb200_get_u_host(s, uT) : mgb200_get_u_device(s, uT, n + 1);   // :175
    if (last) *last = info;
    // MGB200_TIMESTEPPER_CACHE=0: free everything on return, as the reference does (multigrid.cpp:177-185)
    const char* keep = getenv("MGB200_TIMESTEPPER_CACHE");
    if (rc != MGB200_OK || (keep && keep[0] == '0')) { mgb200_destroy(s); g_cached.s = nullptr; }
    return rc;
}

int mgb200_release_cached(void)
{
    std::lock_guard<std::mutex> lock(g_cached.mu);
    if (g_cached.s) { mgb200_destroy(g_cached.s); g_cached.s = nullptr; }
    return MGB200_OK;
}

int mgb200_timestepper_host(double* uT, const double* u0, const double* v1, const double* v2, double nu, int maxlvl,
                            int n, double dt, double T, double dx, double tol, int shape, const mgb200_options* opt,
                            mgb200_solve_info* last)
{
    if (!uT || !u0 || !v1 || !v2) return fail(MGB200_ERR_INVALID, "timestepper: NULL array");
    return timestepper_common(uT, u0, v1, v2, nu, maxlvl, n, dt, T, dx, tol, shape, opt, last, true);
}

int mgb200_timestepper_device(double* uT, const double* u0, const double* v1, const double* v2, double nu, int maxlvl,
                              int n, double dt, double T, double dx, double tol, int shape, const mgb200_options* opt,
                              mgb200_solve_info* last)
{
    if (!uT || !u0 || !v1 || !v2) return fail(MGB200_ERR_INVALID, "timestepper: NULL array");
    return timestepper_common(uT, u0, v1, v2, nu, maxlvl, n, dt, T, dx, tol, shape, opt, last, false);
}

}  // extern "C"
