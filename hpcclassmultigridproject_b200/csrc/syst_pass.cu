// syst_pass.cu -- device primitives (inline PTX: mbarrier, cp.async.bulk.tensor = the TMA engine,
// bulk stores), the kernel and the launcher of the systolic streaming pass.  The per-thread logic
// lives in syst_pass_body.cuh.
#include <cuda.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <tuple>

#include "syst_pass_body.cuh"

namespace mgb200 {
namespace sy {

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

SY_FN int sy_lane() { return threadIdx.x & 31; }

SY_FN bool sy_elect()
{
    unsigned pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

SY_FN void sy_syncwarp() { __syncwarp(); }

SY_FN void sy_full_expect(const Smem& sm, int g, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(sm.base32 + sm.full_off + 8u * g), "r"(bytes) : "memory");
}

SY_FN void sy_tma_load(const Params& p, const Smem& sm, int which, unsigned soff, int x, int z, int g)
{
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
            sm.base32 + soff),
        "l"(&p.maps[which]), "r"(x), "r"(0), "r"(z), "r"(sm.base32 + sm.full_off + 8u * g)
        : "memory");
}

SY_FN void sy_tma_prefetch(const Params& p, int which, int x, int z)
{
    asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(&p.maps[which]), "r"(x), "r"(0), "r"(z)
                 : "memory");
}

SY_FN void sy_tma_load_m(const Params& p, const Smem& sm, int which, unsigned soff, int x, int z, int m, int g)
{
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(
            sm.base32 + soff),
        "l"(&p.maps[which]), "r"(x), "r"(0), "r"(z), "r"(m), "r"(sm.base32 + sm.full_off + 8u * g)
        : "memory");
}

SY_FN void sy_tma_prefetch_m(const Params& p, int which, int x, int z, int m)
{
    asm volatile("cp.async.bulk.prefetch.tensor.4d.L2.global.tile [%0, {%1, %2, %3, %4}];" ::"l"(&p.maps[which]), "r"(x), "r"(0), "r"(z),
                 "r"(m)
                 : "memory");
}

SY_FN int sy_member() { return (int)blockIdx.y; }

__device__ __forceinline__ void mbar_wait(unsigned a, unsigned parity)
{
    unsigned done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(a), "r"(parity)
            : "memory");
    } while (!done);
}

SY_FN void sy_full_wait(const Smem& sm, int g, unsigned parity) { mbar_wait(sm.base32 + sm.full_off + 8u * g, parity); }

SY_FN void sy_prog_publish(const Smem& sm, int warp, unsigned steps_done)
{
    asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(sm.base32 + sm.pb_off + 4u * (unsigned)warp), "r"(steps_done) : "memory");
}

SY_FN Prog2 sy_prog_peek(const Smem& sm, int stage)
{
    Prog2 v;
    asm volatile("ld.acquire.cta.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.h0), "=r"(v.h1) : "r"(sm.base32 + sm.pb_off + 8u * (unsigned)stage) : "memory");
    return v;
}

SY_FN void sy_backoff(int) {}

SY_FN void sy_bulk_store(const Smem& sm, double* gdst, unsigned soff, unsigned bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(sm.base32 + soff), "r"(bytes) : "memory");
}

SY_FN void sy_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
SY_FN void sy_store_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
SY_FN void sy_store_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
SY_FN void sy_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
SY_FN void sy_fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

SY_FN D2 sy_lds2(const Smem& sm, unsigned off)
{
    D2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(sm.base32 + off));
    return v;
}
SY_FN double sy_lds1(const Smem& sm, unsigned off)
{
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(sm.base32 + off));
    return v;
}
SY_FN void sy_sts2(const Smem& sm, unsigned off, D2 v)
{
    asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(sm.base32 + off), "d"(v.x), "d"(v.y) : "memory");
}
SY_FN void sy_sts1(const Smem& sm, unsigned off, double v)
{
    asm volatile("st.shared.f64 [%0], %1;" ::"r"(sm.base32 + off), "d"(v) : "memory");
}

SY_FN double sy_side(const Smem& sm, const D2& mid, unsigned off, int dir, bool outer)
{
    const int lane = threadIdx.x & 31;
    double x = dir < 0 ? __shfl_up_sync(0xffffffffu, mid.y, 1) : __shfl_down_sync(0xffffffffu, mid.x, 1);
    if (lane == (dir < 0 ? 0 : 31)) x = outer ? 0.0 : sy_lds1(sm, off);
    return x;
}

// One kernel image per pass flavour (PRE: prolongation folded into stage 0; POSTK: epilogue kind
// folded into the last stage): each image holds only the loops it runs, and the hot loops of all
// roles together stay well inside the SM's instruction cache.  BATCH: grid (tiles, members), the block
// works on member blockIdx.y; a frozen member's blocks leave before they touch anything, so its arrays and
// partial sums keep what its last active pass left there.
template <int ARITH, bool PRE, int POSTK, bool BATCH>
__global__ void __launch_bounds__(THREADS, 1) k_syst_pass(const __grid_constant__ Params p)
{
    if (BATCH && p.active[blockIdx.y] == 0) return;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ double scratch[32];
    Smem sm;
    carve(sm, smem_raw, p.SWK);
    sm.base32 = smem_u32(smem_raw);
    const Tile tl = make_tile(p, blockIdx.x, POSTK == POST_FW ? 1 : 0);
    const Geo geo = make_geo(p);
    // warp index through a shuffle: provably warp-uniform, so that role branches are uniform and
    // the load and store warps' operands live in uniform registers
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31;
    if (threadIdx.x < NGROUP)
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(sm.base32 + sm.full_off + 8u * threadIdx.x) : "memory");
    if (threadIdx.x < NPROG) *reinterpret_cast<volatile unsigned*>(smem_raw + sm.pb_off + 4u * threadIdx.x) = 0u;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    sy_fence_async();
    __syncthreads();
    const double acc = run_warp<ARITH, PRE, POSTK, BATCH>(p, tl, geo, sm, warp, lane);
    if (POSTK == POST_NORM2) {
        const double tot = block_sum(acc, scratch);
        if (threadIdx.x == 0) p.partials[member_off<BATCH>(p.pstride) + blockIdx.x] = tot;
    }
}

static int g_sms = 0;

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;

// {run, parity, row} view of a split-layout field: dim0 = pairs of one run (stride 8 B, extent = the
// run stride `odd`, slack included), dim1 = parity (stride odd*8), dim2 = rows (stride pitch*8).
// members > 0: a 4-D {run, parity, row, member} view of a batch (dim3 stride mstride*8), box one member deep.
static int encode_field(TensorMapStorage* out, const double* base, long odd, long pitch, long rows, int box_x, int box_rows,
                        int members = 0, long mstride = 0)
{
    static_assert(sizeof(CUtensorMap) == sizeof(TensorMapStorage), "CUtensorMap size");
    CUtensorMap m;
    const cuuint64_t dims[4] = {(cuuint64_t)odd, 2, (cuuint64_t)rows, (cuuint64_t)(members > 0 ? members : 1)};
    const cuuint64_t strides[3] = {(cuuint64_t)odd * 8, (cuuint64_t)pitch * 8, (cuuint64_t)mstride * 8};
    const cuuint32_t box[4] = {(cuuint32_t)box_x, 2, (cuuint32_t)box_rows, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = g_encode(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, members > 0 ? 4 : 3, const_cast<double*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(MGB200_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
    std::memcpy(out, &m, sizeof(m));
    return MGB200_OK;
}

// members: StreamPassArgs::members (0 and 1 give the same plan)
static Plan plan_for(long n, long nrows, int K, int members = 0)
{
    static std::map<std::tuple<long, long, int, int>, Plan> cache;
    static std::mutex mu;
    std::lock_guard<std::mutex> lock(mu);
    const int mb = members > 1 ? members : 1;
    auto key = std::make_tuple(n, nrows, K, mb);
    auto it = cache.find(key);
    if (it == cache.end()) {
        int force = 0;
        if (const char* e = getenv("MGB200_SWK")) force = atoi(e);       // tuning aid: pin the strip width
        it = cache.emplace(key, make_plan(n, nrows, K, g_sms > 0 ? g_sms : 148, force, mb)).first;
    }
    return it->second;
}

using PassKernel = void (*)(const Params);
template <int ARITH, bool BATCH>
static PassKernel pass_kernel_of(bool pre, int post)
{
    // full weighting: down leg only, no prolongation flavour
    if (post == POST_FW) return k_syst_pass<ARITH, false, POST_FW, BATCH>;
    if (pre) return post == POST_NORM2 ? k_syst_pass<ARITH, true, POST_NORM2, BATCH> : post == POST_INJECT ? k_syst_pass<ARITH, true, POST_INJECT, BATCH>
                                                                                                          : k_syst_pass<ARITH, true, POST_NONE, BATCH>;
    return post == POST_NORM2 ? k_syst_pass<ARITH, false, POST_NORM2, BATCH> : post == POST_INJECT ? k_syst_pass<ARITH, false, POST_INJECT, BATCH>
                                                                                                    : k_syst_pass<ARITH, false, POST_NONE, BATCH>;
}
static PassKernel pass_kernel(int arith, bool pre, int post, bool batch)
{
    if (arith == MGB200_ARITH_EXACT) return batch ? pass_kernel_of<MGB200_ARITH_EXACT, true>(pre, post) : pass_kernel_of<MGB200_ARITH_EXACT, false>(pre, post);
    return batch ? pass_kernel_of<MGB200_ARITH_FAST, true>(pre, post) : pass_kernel_of<MGB200_ARITH_FAST, false>(pre, post);
}

}  // namespace sy

using namespace sy;

// per-device set-up (function attributes are per device)
int stream_pass_init()
{
    static std::mutex mu;
    static bool done[64] = {};
    int dev = 0;
    MGB_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    if (dev >= 0 && dev < 64 && done[dev]) return MGB200_OK;
    MGB_CUDA(cudaDeviceGetAttribute(&g_sms, cudaDevAttrMultiProcessorCount, dev));
    for (int batch = 0; batch < 2; ++batch)
        for (int arith = 0; arith < 2; ++arith)
            for (int pre = 0; pre < 2; ++pre)
                for (int post = 0; post <= POST_FW; ++post)
                    MGB_CUDA(cudaFuncSetAttribute(pass_kernel(arith, pre != 0, post, batch != 0), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
    if (!g_encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        MGB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (!fn || qres != cudaDriverEntryPointSuccess) return fail(MGB200_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
        g_encode = (EncodeTiledFn)fn;
    }
    if (dev >= 0 && dev < 64) done[dev] = true;
    return MGB200_OK;
}

long stream_pass_tiles(long n, long nrows, int iters, int members)
{
    if (iters >= 1) {
        const Plan pl = plan_for(n, nrows, iters > KMAX ? KMAX : iters, members);
        return (long)pl.nstrips * pl.nbands;
    }
    long m = 0;
    for (int K = 1; K <= KMAX; ++K) {
        const Plan pl = plan_for(n, nrows, K, members);
        m = std::max(m, (long)pl.nstrips * pl.nbands);
    }
    return m;
}

static int build_params(const StreamPassArgs& a, Params& p, unsigned& grid_out, size_t& smem_out)
{
    if (a.iters < 1 || a.iters > KMAX) return fail(MGB200_ERR_INVALID, "stream_pass: iters must be 1..3");
    if (a.n < 8 || (a.n & 3)) return fail(MGB200_ERR_INVALID, "stream_pass: n must be a multiple of 4, >= 8");
    if (!a.L.split() || a.u_out == a.u_in) return fail(MGB200_ERR_INVALID, "stream_pass: needs the split layout and u_out != u_in");
    MGB_TRY(stream_pass_init());
    const bool whole = a.rows_mem == 0;
    const long own_lo = whole ? 0 : a.own_lo, own_hi = whole ? a.n : a.own_hi;
    if (a.members < 0 || a.members > STREAM_PASS_MAX_MEMBERS) return fail(MGB200_ERR_INVALID, "stream_pass: members must be 0..65535");
    const bool batch = a.members > 0;
    if (batch && (!whole || !a.active || a.mstride <= 0 || (a.coarse_u && a.cmstride <= 0)))
        return fail(MGB200_ERR_INVALID, "stream_pass: a batched pass needs whole levels, member strides and the active flags");
    const Plan pl = plan_for(a.n, own_hi - own_lo + 1, a.iters, a.members);
    p = Params{};
    p.n = a.n; p.nhalf = a.n / 2;
    p.own_lo = own_lo; p.own_hi = own_hi;
    p.row0 = whole ? 0 : a.row0; p.rows_mem = whole ? a.n + 1 : a.rows_mem;
    p.mem_lo = p.row0; p.mem_hi = p.row0 + p.rows_mem - 1;
    p.crow0 = whole ? 0 : a.crow0; p.crows_mem = whole ? a.n / 2 + 1 : a.crows_mem;
    p.pitch = a.L.pitch; p.odd = a.L.odd;
    p.cpitch = a.Lc.pitch; p.codd = a.Lc.odd;
    p.RBAND = pl.RBAND; p.WK = pl.WK; p.SWK = pl.SWK; p.nstrips = pl.nstrips; p.nbands = pl.nbands;
    p.K = a.iters;
    p.pre = a.coarse_u ? 1 : 0;
    p.post = a.post;
    p.u_is_zero = a.u_in ? 0 : 1;
    p.CW = pl.SWK / 2 + 8;
    p.st = a.st;
    p.u_in = a.u_in; p.rhs = a.rhs; p.v1 = a.v1; p.v2 = a.v2; p.cu = a.coarse_u;
    // the u map of a zero-input pass is never dereferenced (its boxes lie out of bounds): any valid field will do
    const int mb = a.members;
    MGB_TRY(encode_field(&p.maps[FIELD_U], a.u_in ? a.u_in : a.rhs, a.L.odd, a.L.pitch, p.rows_mem, pl.SWK, GROUP, mb, a.mstride));
    MGB_TRY(encode_field(&p.maps[FIELD_F], a.rhs, a.L.odd, a.L.pitch, p.rows_mem, pl.SWK, GROUP, mb, a.mstride));
    MGB_TRY(encode_field(&p.maps[FIELD_V1], a.v1, a.L.odd, a.L.pitch, p.rows_mem, pl.SWK, GROUP, mb, a.mstride));
    MGB_TRY(encode_field(&p.maps[FIELD_V2], a.v2, a.L.odd, a.L.pitch, p.rows_mem, pl.SWK, GROUP, mb, a.mstride));
    if (a.coarse_u) MGB_TRY(encode_field(&p.maps[FIELD_C], a.coarse_u, a.Lc.odd, a.Lc.pitch, p.crows_mem, p.CW, CROWS, mb, a.cmstride));
    p.u_out = a.u_out; p.crhs = a.coarse_rhs; p.partials = a.partials;
    if (batch) { p.mstride = a.mstride; p.cmstride = a.cmstride; p.pstride = a.pstride; p.active = a.active; }
    if (p.post == POST_INJECT && !p.crhs) return fail(MGB200_ERR_INVALID, "stream_pass: POST_INJECT without coarse_rhs");
    if (p.post == POST_FW && (!p.crhs || p.pre)) return fail(MGB200_ERR_INVALID, "stream_pass: POST_FW needs coarse_rhs and no prolongation");
    if (p.post == POST_NORM2 && !p.partials) return fail(MGB200_ERR_INVALID, "stream_pass: POST_NORM2 without partials");
    grid_out = (unsigned)(pl.nstrips * pl.nbands);
    smem_out = smem_bytes(pl.SWK);
    if (batch && p.post == POST_NORM2 && a.pstride < (long)grid_out) return fail(MGB200_ERR_INVALID, "stream_pass: partials stride below the tile count");
    return MGB200_OK;
}

int stream_pass(const StreamPassArgs& a, cudaStream_t s)
{
    // The kernel parameter block (five encoded tensor maps, the tile plan, the row window) depends
    // only on the argument record: a solver issues the same few dozen passes every cycle, so blocks
    // are built once and looked up by the raw bytes of the arguments (per device: tensor maps hold
    // device addresses, which are unique across the devices of a process).
    struct Entry { Params p; unsigned grid; size_t smem; int members; };
    static std::map<std::string, Entry> cache;
    static std::mutex mu;
    Entry e;
    {
        std::lock_guard<std::mutex> lock(mu);
        StreamPassArgs key;
        std::memset(&key, 0, sizeof(key));              // padding bytes must compare equal
        key.n = a.n; key.L = a.L; key.st = a.st; key.u_in = a.u_in; key.u_out = a.u_out; key.rhs = a.rhs; key.v1 = a.v1; key.v2 = a.v2;
        key.iters = a.iters; key.coarse_u = a.coarse_u; key.Lc = a.Lc; key.post = a.post; key.coarse_rhs = a.coarse_rhs;
        key.partials = a.partials; key.arith = a.arith; key.own_lo = a.own_lo; key.own_hi = a.own_hi; key.row0 = a.row0;
        key.rows_mem = a.rows_mem; key.crow0 = a.crow0; key.crows_mem = a.crows_mem;
        key.members = a.members; key.mstride = a.mstride; key.cmstride = a.cmstride; key.pstride = a.pstride; key.active = a.active;
        std::string k(reinterpret_cast<const char*>(&key), sizeof(key));
        auto it = cache.find(k);
        if (it == cache.end()) {
            Entry fresh;
            MGB_TRY(build_params(a, fresh.p, fresh.grid, fresh.smem));
            fresh.members = a.members;
            if (cache.size() > 4096) cache.clear();     // many short-lived solvers: do not grow without bound
            it = cache.emplace(std::move(k), fresh).first;
        }
        e = it->second;                                 // copied under the lock: the map may be cleared by another thread
    }
    const bool batch = e.members > 0;
    pass_kernel(a.arith, e.p.pre != 0, e.p.post, batch)<<<dim3(e.grid, batch ? (unsigned)e.members : 1u), THREADS, e.smem, s>>>(e.p);
    return check_launch("k_syst_pass");
}

}  // namespace mgb200
