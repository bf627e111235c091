// syst_pass_body.cuh -- the fused streaming pass as a SYSTOLIC pipeline of warps: geometry and the
// per-thread step logic (no CUDA-specific instruction in this file: everything asynchronous goes
// through the sy_* primitives, inline PTX in syst_pass.cu, a thread-per-lane host model in
// tests/emu/syst_emu.cpp).
//
// One pass = [u += P(coarse u)] -> K red-black Gauss-Seidel iterations -> [residual -> injection |
// residual -> full weighting | residual -> sum of squares] on one level (reference: multigrid.cpp:69-88 around gs.cpp:109-189,
// :55-83, :268-292, :228-266), u / rhs / v1 / v2 read once from HBM and u written once.
//
// One tile = a column strip x a row band, one thread block, streaming DOWN the rows.  TMA boxes
// bring GROUP rows of the four fields (plus the coarse rows their prolongation needs) into a
// shared-memory ring; 2K half-sweep stages follow the load front, stage s (colour s&1) two rows
// behind stage s-1, updating the ring in place; finished rows leave through bulk stores.
//
// What is different from a barrier-per-row pipeline: the warps are coupled ONLY by the data
// dependencies of the half-sweeps.  Every stage warp publishes the number of steps it has completed in
// a shared-memory counter (store-release after its row is written) and a warp waits (load-acquire,
// one 8-byte load for both warps of a stage) for exactly the warps whose results it reads:
//
//     stage s, step k   needs   stage s-1 (both column halves), step k-1          [row below + strip-half edge]
//     stage 0           needs   the TMA group of its lower row                     [full barriers]
//     store warp, step k needs  the last stage, step k                             [row to hand to the bulk-store engine]
//     load warp, step k  needs  the last role, step k, and the store warp's count  [ring slots to refill]
//
// The reverse (write-after-read) hazards are implied by these: stage s+1 cannot touch a row before
// stage s has finished the row below it, and by then stage s has long read everything it needs of
// it.  The first look at a counter is issued before the step's own loads, so in the steady state the
// wait costs no latency at all; there is no block barrier in the row loop, and a slow step of one warp is
// absorbed by the slack of the ring instead of stalling all the others.  (An earlier version kept the
// progress in rings of mbarriers: mbarrier.try_wait costs ~90 cycles even when the phase is complete,
// two or three of them per step made the step longer than the per-row barrier they replaced.)
//
// Every role of the pipeline is a pair of warps doing about the same work per row, so that no role paces the
// others: the prolongation + correction has a role of its own in front of stage 0 (it touches the nodes of the
// second colour only: a Gauss-Seidel update never reads its own old value, so the first colour is overwritten
// unread), and the residual epilogue a role of its own behind the last stage, built like a half-sweep on the
// first colour (the last stage sums the second colour's residual itself: all its operands are in registers).
// (Folding both into stage 0 and the last stage saves shared-memory traffic but makes those two warps do 2-3
// times the work of the others, and the pipeline runs at the pace of its slowest warp: measured slower.)
//
// Warps: 2 per role (64 column pairs each, one 16-byte vector = 2 nodes per lane) + the load warp + the store warp.
#pragma once
#include "common.cuh"
#include "stream_pass.cuh"

#ifndef SY_FN
#define SY_FN __device__ __forceinline__
#endif

namespace mgb200 {
namespace sy {

constexpr int SWK_MAX = 128;   // pairs (= 2 columns) per shared-memory row
constexpr int HK = 4;          // halo pairs per strip side (8 columns >= 2K+1 for K <= 3)
constexpr int GROUP = 4;       // rows per TMA box
constexpr int RING = 24;       // fine-row ring slots
constexpr int NGROUP = RING / GROUP;
constexpr int CROWS = 3;       // coarse rows travelling with a group of fine rows
constexpr int KMAX = 3;
constexpr int NSTW = 2;        // warps per half-sweep stage (64 pairs each)
constexpr int NPAIR = 2 * KMAX + 2;      // half-sweep stages + the prolongation role + the residual role
constexpr int NSTAGE = NPAIR * NSTW;      // warps of those roles (a progress counter each)
constexpr int WARPS = NSTAGE + 2;          // + the load warp + the store warp
constexpr int THREADS = WARPS * 32;
constexpr int PRODUCER_WARP = NSTAGE;      // requests the TMA groups
constexpr int STORE_WARP = NSTAGE + 1;     // hands finished rows to the bulk-store engine
constexpr int NPROG = NSTAGE + 2;          // progress counters: the role warps' + a pair slot for the store warp
// POST_FW: rows of residual (both runs, ring-row layout) between the last stage / EPI and the restriction.  They live
// where a pass with prolongation keeps its coarse rows (POST_FW passes have none): 8 rows of 2 SWK doubles take
// 128 SWK bytes, the coarse rows 144 SWK + 2304.
constexpr int FW_ROWS = 8;
// opaque storage for a CUtensorMap (128 bytes, 64-byte aligned); filled by the host launcher
struct alignas(64) TensorMapStorage { unsigned long long q[16]; };

struct Params {
    TensorMapStorage maps[5];  // Field order: u_in, rhs, v1, v2, coarse u
    long n, nhalf;             // level size, n/2
    long pitch, odd;           // split layout of this level
    long cpitch, codd;         // split layout of the next coarser level
    long RBAND;                // owned rows per band
    // row window (row-slab sharding; a single GPU owns and holds rows 0..n):
    long own_lo, own_hi;       // rows this launch must produce
    long mem_lo, mem_hi;       // rows present in the arrays (own rows + halo rows received from neighbours)
    long row0, crow0;          // global row index of memory row 0 of the fine / coarse arrays
    long rows_mem, crows_mem;  // rows held by the fine / coarse arrays
    int WK, SWK;               // owned pairs per strip, pairs per smem row (WK + 2 HK)
    int nstrips, nbands;
    int K;                     // fused RB iterations, 1..3
    int pre;                   // 1: u += P(coarse u) before smoothing
    int post;                  // StreamPost
    int u_is_zero;             // u_in == 0 everywhere: rows are zero-filled by an out-of-bounds box
    int CW;                    // SWK/2 + 8: coarse pairs per smem run
    Stencil st;
    const double* u_in;
    const double* rhs;
    const double* v1;
    const double* v2;
    const double* cu;          // coarse u (pre)
    double* u_out;
    double* crhs;              // coarse rhs (POST_INJECT, POST_FW)
    double* partials;          // POST_NORM2
    // batched passes (BATCH): member b of every fine / coarse array starts b * mstride / b * cmstride
    // doubles after the first, its partial sums at b * pstride; a member whose active[b] is 0 is not touched
    long mstride, cmstride, pstride;
    const int* active;
};

struct Tile {
    int R0, R1;                // rows staged: [R0, R1]
    int rb0, rb1;              // rows owned:  [rb0, rb1]
    int k0;                    // global pair index of smem column 0 (may be -HK)
    int kb;                    // first owned pair
};

struct Smem {
    unsigned char* raw;        // start of the dynamic shared memory (generic address; host emulation)
    unsigned base32;           // its shared-space address (device only)
    unsigned full_off;         // byte offset of the NGROUP load-completion barriers
    unsigned pb_off;           // byte offset of the progress counters: one unsigned per stage warp, the two warps of a stage adjacent
};
// byte offsets from `raw`: U ring at 0, rhs / v1 / v2 rings at ringb, 2 ringb, 3 ringb, the coarse
// rows [NGROUP][CROWS][2][CW] at 4 ringb, then the barriers

enum Field { FIELD_U = 0, FIELD_F = 1, FIELD_V1 = 2, FIELD_V2 = 3, FIELD_C = 4 };

constexpr size_t smem_bytes(int swk)
{
    return (size_t)4 * RING * 2 * swk * 8 + (size_t)NGROUP * CROWS * 2 * (swk / 2 + 8) * 8 + NGROUP * 8 + NPROG * 4 + 128;
}
constexpr size_t SMEM_BYTES = smem_bytes(SWK_MAX);

struct alignas(16) D2 { double x, y; };    // 16-byte vector; aligned accesses only (even pair index)

SY_FN void carve(Smem& sm, unsigned char* base, int swk)
{
    sm.raw = base; sm.base32 = 0;
    sm.full_off = (unsigned)(4 * RING * 2 * swk * 8 + NGROUP * CROWS * 2 * (swk / 2 + 8) * 8);
    sm.pb_off = sm.full_off + NGROUP * 8;
}

// Halo rows per band side: after the 2K half-sweeps the rows within 2K of the first / last staged row are stale, so
// the residual is exact from rb0 on (injection reads no more).  Full weighting also needs the residual one row outside
// the owned rows: `extra` = 1.  (Columns: 4 halo pairs = 8 columns leave one column of margin for that.)
SY_FN Tile make_tile(const Params& p, long tile, int extra = 0)
{
    Tile tl;
    const long strip = tile % p.nstrips, band = tile / p.nstrips;
    const long HR = 2 * p.K + 1 + extra;
    long rb0 = p.own_lo + band * p.RBAND, rb1 = rb0 + p.RBAND - 1;
    if (rb1 > p.own_hi) rb1 = p.own_hi;
    long R0 = rb0 - HR, R1 = rb1 + HR;
    if (R0 < p.mem_lo) R0 = p.mem_lo;
    if (R1 > p.mem_hi) R1 = p.mem_hi;
    tl.kb = (int)(strip * p.WK);
    tl.k0 = tl.kb - HK;
    tl.rb0 = (int)rb0; tl.rb1 = (int)rb1; tl.R0 = (int)R0; tl.R1 = (int)R1;
    return tl;
}

// ------------------------------------------------------------------------------------------
// primitives (inline PTX in syst_pass.cu, plain C++ / atomics in the host emulation).  Shared
// memory is addressed by byte offsets from the start of the U ring.
SY_FN int  sy_lane();
SY_FN bool sy_elect();                                   // true in exactly one lane of the converged warp
SY_FN void sy_syncwarp();                                // execution + memory barrier among the warp's lanes
SY_FN void sy_full_expect(const Smem& sm, int g, unsigned bytes);
// 3-D tensor load of field `which`: box {SWK (CW for FIELD_C), 2, GROUP (CROWS)} whose first element
// is (pair x, parity 0, memory row z) of the field; out-of-bounds elements arrive as zeros
SY_FN void sy_tma_load(const Params& p, const Smem& sm, int which, unsigned soff, int x, int z, int g);
SY_FN void sy_tma_prefetch(const Params& p, int which, int x, int z);   // same box, into L2 only
// batched passes: the maps are 4-D {pair, parity, row, member}; the same box (one member deep) of member m, zeros
// outside that member's rows
SY_FN void sy_tma_load_m(const Params& p, const Smem& sm, int which, unsigned soff, int x, int z, int m, int g);
SY_FN void sy_tma_prefetch_m(const Params& p, int which, int x, int z, int m);
SY_FN int sy_member();                                   // batched passes: the member of this block
// first element of this block's member in an array whose members lie `stride` doubles apart (0 unless BATCH; the
// batched primitives are only named in batched code, so a host model without them still builds the others)
template <bool BATCH>
SY_FN long member_off(long stride)
{
    if constexpr (BATCH) return (long)sy_member() * stride;
    else return 0L;
}
SY_FN void sy_full_wait(const Smem& sm, int g, unsigned parity);
// progress counters: steps completed by a stage warp.  Publish = store-release by one lane after
// sy_syncwarp (orders the whole warp's earlier shared-memory writes); peek = load-acquire of the
// counters of both warps of a stage.
struct Prog2 { unsigned h0, h1; };
SY_FN void sy_prog_publish(const Smem& sm, int warp, unsigned steps_done);
SY_FN Prog2 sy_prog_peek(const Smem& sm, int stage);
// between two unsuccessful peeks at the counters of pair `pair`: nothing on the device; the host model yields there
// and reports a deadlock
SY_FN void sy_backoff(int pair);
SY_FN void sy_bulk_store(const Smem& sm, double* gdst, unsigned soff, unsigned bytes);
SY_FN void sy_store_commit();
SY_FN void sy_store_wait_read0();                        // every committed store has read its shared memory
SY_FN void sy_store_wait_read1();                        // ... all but the most recent one
SY_FN void sy_store_wait_all();
SY_FN void sy_fence_async();                             // generic -> async proxy (rows handed to the bulk-store engine)
SY_FN D2 sy_lds2(const Smem& sm, unsigned off);
SY_FN double sy_lds1(const Smem& sm, unsigned off);
SY_FN void sy_sts2(const Smem& sm, unsigned off, D2 v);
SY_FN void sy_sts1(const Smem& sm, unsigned off, double v);
// The third horizontal neighbour of a lane's vector `mid` (run R of some row): the node of run R
// just left of it (dir < 0: mid.y of the previous lane) or just right (dir > 0: mid.x of the next
// lane).  Lanes 0 / 31 read it from shared memory at `off` (it belongs to the other warp of the
// stage); `outer`: the lane sits on the strip's outer edge, where the value is never used: 0.
// (The host emulation reads shared memory in every lane: the value is the same.)
SY_FN double sy_side(const Smem& sm, const D2& mid, unsigned off, int dir, bool outer);

// ------------------------------------------------------------------------------------------
struct Geo {
    unsigned swkb;    // bytes of one parity run: SWK * 8
    unsigned rowb;    // bytes of one ring row (both runs)
    unsigned ringb;   // bytes of one field's ring
    unsigned cwb;     // bytes of one coarse parity run
    unsigned cgrpb;   // bytes of the coarse rows of one group
    int nh;           // warps per stage that hold live pairs (1 for strips of <= 64 pairs)
};
SY_FN Geo make_geo(const Params& p)
{
    Geo g;
    g.swkb = (unsigned)p.SWK * 8u; g.rowb = 2u * g.swkb; g.ringb = (unsigned)RING * g.rowb;
    g.cwb = (unsigned)p.CW * 8u; g.cgrpb = (unsigned)CROWS * 2u * g.cwb;
    g.nh = p.SWK > 64 ? 2 : 1;
    return g;
}

SY_FN unsigned ring_adv(unsigned a, const Geo& g, unsigned lim)
{
    a += g.rowb;
    return a >= lim ? a - g.ringb : a;
}

SY_FN int num_groups(const Tile& tl) { return (tl.R1 - tl.R0) / GROUP + 1; }

// Roles.  Every role is a pair of warps (column halves) walking down the rows one row per step; role R at
// step k (t = R0 + k) works on row t - off(R):
//   PRE      (passes with prolongation) row t: adds P(coarse u) to the SECOND-colour nodes (a Gauss-Seidel update
//            never reads its own old value, so the first colour is overwritten unread)            off = 0
//   stage s  half-sweep s (colour s & 1), s = 0 .. 2K-1                                           off = 1 + 2s (+1 with PRE)
//   EPI      (passes with a residual epilogue) residual of the FIRST-colour nodes behind the last stage:
//            injection of the even columns of even rows, or sum of squares (the second colour's
//            residual is summed by the last stage itself: all its operands are in registers)      off = off(last) + 2
// Pair index in the progress counters: stage s -> s, PRE -> 2 KMAX, EPI -> 2 KMAX + 1.
constexpr int PAIR_PRE = 2 * KMAX, PAIR_EPI = 2 * KMAX + 1, PAIR_STORE = NPAIR;

SY_FN int off_stage(const Params& p, int s) { return 1 + 2 * s + (p.pre ? 1 : 0); }
SY_FN int off_epi(const Params& p) { return off_stage(p, 2 * p.K - 1) + 2; }
// the slowest role must still visit row rb1 (POST_FW: xr = 2, the EPI role restricts row rb1 + 1 one step after
// reaching row rb1 + 2; every role runs the same number of steps)
SY_FN int last_step(const Params& p, const Tile& tl, int xr = 0) { return tl.rb1 + xr + (p.post != POST_NONE ? off_epi(p) : off_stage(p, 2 * p.K - 1)); }

// per-thread state of a role, advanced by one row per step
struct Stage {
    int pair;           // own pair index in the progress counters
    int up;             // pair index of the role whose results this one reads (-1: the TMA full barriers)
    int h;              // column half
    int s;              // stage number (colour = s & 1; the EPI role counts as stage 2K: first colour)
    int kk;             // first local pair of the lane's vector (even)
    int off;            // row = t - off
    int row;            // the role's row at the current step
    int lo, hi;         // rows the role updates: [lo, hi]
    unsigned a_prev, a_cur, a_next;   // ring offsets of even-run element kk of rows row-1, row, row+1
    unsigned lim;       // ringb + kk*8: wrap limit of those offsets
    unsigned okp0, okp1;   // update masks of the lane's two targets for column parity 0 / 1 (scalars: a dynamically
                           // indexed array would live in local memory)
    bool outer_l, outer_r;            // the lane's left / right side neighbour lies outside the strip
    bool live;          // the lane's vector lies inside the strip (strips narrower than the role's 64 x NSTW pairs)
    // operands carried in registers from step to step: the other-parity nodes of the current row become
    // the next row's upper neighbours, the nodes loaded from the row below become the next row's
    // horizontal neighbours (no other role writes them in between: the next one is two rows behind)
    D2 c_up, c_mid;
    unsigned rmask0, rmask1;   // owned nodes with an interior column, per column parity
    int elo, ehi;       // owned interior rows
    double acc;         // POST_NORM2 accumulator
    unsigned cmask0, cmask1;   // interior-column bits per column parity (PRE)
};

// POST_FW, EPI role: weighted row sums of the last even row 2I and of the last odd row 2I-1, per coarse column
struct FwSums { D2 e, o; };

SY_FN Stage init_role(const Params& p, const Tile& tl, const Geo& geo, int pair, int up, int s, int off, int h, int lane)
{
    Stage st;
    st.pair = pair; st.up = up; st.s = s; st.h = h; st.off = off;
    int kk = 64 * h + 2 * lane;
    if (kk > p.SWK - 2) kk = p.SWK - 2;               // lanes beyond the strip shadow its last vector (all their masks are 0)
    const bool live = 64 * h + 2 * lane < p.SWK;
    st.kk = kk;
    st.row = tl.R0 - off;
    st.lo = tl.R0 + 1; st.hi = tl.R1 - 1;             // rows row-1 and row+1 must be staged
    st.c_up = D2{0.0, 0.0}; st.c_mid = D2{0.0, 0.0};
    st.acc = 0.0;
    st.elo = tl.rb0 < 1 ? 1 : tl.rb0; st.ehi = tl.rb1 > p.n - 1 ? (int)p.n - 1 : tl.rb1;
    st.okp0 = st.okp1 = st.rmask0 = st.rmask1 = st.cmask0 = st.cmask1 = 0;
    for (int e = 0; e < 2 && live; ++e) {
        const int k = kk + e;
        const long kg = (long)tl.k0 + k;
        const bool owned = k >= HK && k < HK + p.WK;
        // even column 2kg: interior for 1 <= kg <= nhalf-1, neighbours O[k-1], O[k]
        const bool int0 = kg >= 1 && kg <= p.nhalf - 1;
        // odd column 2kg+1: interior for 0 <= kg <= nhalf-1, neighbours E[k], E[k+1]
        const bool int1 = kg >= 0 && kg <= p.nhalf - 1;
        if (int0 && k >= 1) st.okp0 |= 1u << e;
        if (int1 && k <= p.SWK - 2) st.okp1 |= 1u << e;
        if (int0 && owned) st.rmask0 |= 1u << e;
        if (int1 && owned) st.rmask1 |= 1u << e;
        if (int0) st.cmask0 |= 1u << e;
        if (int1) st.cmask1 |= 1u << e;
    }
    st.live = live;
    st.outer_l = kk == 0;
    st.outer_r = kk + 2 >= p.SWK;
    const int slot = ((RING - off) % RING + RING) % RING;            // row R0 sits in slot 0
    st.lim = geo.ringb + (unsigned)kk * 8u;
    st.a_cur = (unsigned)slot * geo.rowb + (unsigned)kk * 8u;
    st.a_next = ring_adv(st.a_cur, geo, st.lim);
    st.a_prev = (slot == 0 ? (unsigned)(RING - 1) : (unsigned)(slot - 1)) * geo.rowb + (unsigned)kk * 8u;
    return st;
}

SY_FN void advance_row(const Geo& geo, Stage& st)
{
    st.row += 1;
    st.a_prev = st.a_cur; st.a_cur = st.a_next; st.a_next = ring_adv(st.a_next, geo, st.lim);
}

// wait until the warps of pair `pair` have completed `need0` / `need1` steps (pv: a peek taken earlier)
SY_FN void prog_wait(const Smem& sm, int pair, unsigned need0, unsigned need1, Prog2 pv)
{
    while (pv.h0 < need0 || pv.h1 < need1) { sy_backoff(pair); pv = sy_prog_peek(sm, pair); }
}

// wait for the data of step k: the TMA group of row t (roles fed by the TMA engine) or step k-1 of the role above
SY_FN void wait_inputs(const Tile& tl, const Geo& geo, const Smem& sm, const Stage& st, int k, Prog2 seen)
{
    if (st.up < 0) {
        const int t = tl.R0 + k;
        if ((k & (GROUP - 1)) == 0 && t <= tl.R1) {
            const int g = k / GROUP;
            sy_full_wait(sm, g % NGROUP, (unsigned)(g / NGROUP) & 1u);
        }
    } else {
        prog_wait(sm, st.up, (unsigned)k, geo.nh == 2 ? (unsigned)k : 0u, seen);
    }
}

SY_FN void publish(const Smem& sm, const Stage& st, int k)
{
    sy_syncwarp();
    if (sy_elect()) sy_prog_publish(sm, st.pair * NSTW + st.h, (unsigned)k + 1u);
}

// ------------------------------------------------------------------------------------------
// PRE role, step k: row t = R0 + k.  Bilinear prolongation (gs.cpp:238-240) of the coarse iterate at the lane's
// two SECOND-colour nodes of the row (even columns of odd rows, odd columns of even rows) added to u
// (multigrid.cpp:83), interior nodes only.  The coarse rows of a group start at coarse row (first fine row of
// the group) >> 1; coarse column (k0 + k) sits at local index k: even k in the E run at k/2, odd k in the O run.
SY_FN void pre_step(const Params& p, const Tile& tl, const Geo& geo, const Smem& sm, Stage& st, const int k)
{
    const int t = st.row;
    wait_inputs(tl, geo, sm, st, k, Prog2{0u, 0u});
    if (t >= tl.R0 && t <= tl.R1 && t >= 1 && t <= (int)p.n - 1) {
        const int PAR = (t + 1) & 1;
        const unsigned a = st.a_cur + (PAR ? geo.swkb : 0u);
        const int g = k / GROUP, G0 = tl.R0 + g * GROUP;
        const int crow = (t >> 1) - (G0 >> 1);                       // 0..2; an odd fine row also uses crow+1
        const unsigned c0 = 4u * geo.ringb + (unsigned)(g % NGROUP) * geo.cgrpb + (unsigned)crow * 2u * geo.cwb + (unsigned)(st.kk >> 1) * 8u;
        D2 u{0.0, 0.0};
#ifdef SY_HOST_MODEL
        if (st.live)
#endif
        u = sy_lds2(sm, a);
        const double a0 = sy_lds1(sm, c0), a1 = sy_lds1(sm, c0 + geo.cwb);
        D2 e;
        if (PAR) {                                                   // even row, odd columns (gs.cpp:240)
            const double a2 = sy_lds1(sm, c0 + 8u);
            e.x = __dmul_rn(__dadd_rn(a0, a1), 0.5); e.y = __dmul_rn(__dadd_rn(a1, a2), 0.5);
        } else {                                                     // odd row, even columns (gs.cpp:239)
            const unsigned c1 = c0 + 2u * geo.cwb;
            const double b0 = sy_lds1(sm, c1), b1 = sy_lds1(sm, c1 + geo.cwb);
            e.x = __dmul_rn(__dadd_rn(a0, b0), 0.5); e.y = __dmul_rn(__dadd_rn(a1, b1), 0.5);
        }
        const unsigned cm = PAR ? st.cmask1 : st.cmask0;
        u.x = __dadd_rn(u.x, e.x); u.y = __dadd_rn(u.y, e.y);
        if (cm == 3u) sy_sts2(sm, a, u);
        else {
            if (cm & 1u) sy_sts1(sm, a, u.x);
            if (cm & 2u) sy_sts1(sm, a + 8u, u.y);
        }
    }
    publish(sm, st, k);
    advance_row(geo, st);
}

SY_FN void pre_loop(const Params& p, const Tile& tl, const Geo& geo, const Smem& sm, Stage& st)
{
    const int klast = last_step(p, tl) - tl.R0;
    for (int k = 0; k <= klast; ++k) pre_step(p, tl, geo, sm, st, k);
}

// ------------------------------------------------------------------------------------------
// Coarse right-hand side node pair (cr, kg), (cr, kg+1) of a lane whose vector starts at global pair kg (even: the
// strips start at even pairs): kg -> E run at kg/2, kg+1 -> O run; only the owned interior columns (rmask0).
template <bool BATCH>
SY_FN void store_coarse(const Params& p, const Stage& st, long kg, long cr, double r0, double r1)
{
    double* crow = p.crhs + member_off<BATCH>(p.cmstride) + (cr - p.crow0) * p.cpitch + (kg >> 1);
    if (st.rmask0 & 1u) crow[0] = r0;
    if (st.rmask0 & 2u) crow[p.codd] = r1;
}

// POST_FW: byte offset of node kk of residual row `row` (E run; the O run follows at + swkb)
SY_FN unsigned fw_off(const Tile& tl, const Geo& geo, const Stage& st, int row)
{
    return 4u * geo.ringb + (unsigned)((row - tl.R0) & (FW_ROWS - 1)) * geo.rowb + (unsigned)st.kk * 8u;
}

// one fine row of the full-weighting stencil, grouped as k_restrict_fw (ops_basic.cu): ((w a + 2w b) + w c) / 16
SY_FN double fw_row(double a, double b, double c, double w)
{
    return __dmul_rn(__dadd_rn(__dadd_rn(__dmul_rn(w, a), __dmul_rn(2.0 * w, b)), __dmul_rn(w, c)), 0.0625);
}

// POST_FW, EPI role at step k (its row q + 1 published): restrict residual row q.  Row q's residual is complete in
// the residual rows -- its second colour from the last stage (published step k-1 covers row q + 2), its first colour
// from this role -- once the other EPI warp has published row q as well (lane 0 reads that warp's last node).  The
// horizontal sums of the lane's two coarse columns J = kg, kg+1 (fine columns 2J-1, 2J, 2J+1 = O[J-1], E[J], O[J])
// are kept in registers: an even row waits in fw.e, an odd row 2I+1 completes coarse row I and becomes fw.o.
template <bool BATCH>
SY_FN void fw_restrict_row(const Params& p, const Tile& tl, const Geo& geo, const Smem& sm, const Stage& st, FwSums& fw,
                           const int k, const int q, const bool live)
{
    prog_wait(sm, PAIR_EPI, (unsigned)k, geo.nh == 2 ? (unsigned)k : 0u, sy_prog_peek(sm, PAIR_EPI));
    const unsigned b = fw_off(tl, geo, st, q);
    D2 e{0.0, 0.0}, o{0.0, 0.0};
    if (live) { e = sy_lds2(sm, b); o = sy_lds2(sm, b + geo.swkb); }
    const double ol = sy_side(sm, o, b + geo.swkb - 8u, -1, st.outer_l);
    const double w = (q & 1) ? 1.0 : 2.0;
    const D2 h{fw_row(ol, e.x, o.x, w), fw_row(o.x, e.y, o.y, w)};
    if ((q & 1) == 0) { fw.e = h; return; }
    if (q - 1 >= st.elo && q - 1 <= st.ehi)
        store_coarse<BATCH>(p, st, (long)tl.k0 + st.kk, (long)(q >> 1), __dadd_rn(__dadd_rn(fw.o.x, fw.e.x), h.x),
                     __dadd_rn(__dadd_rn(fw.o.y, fw.e.y), h.y));
    fw.o = h;
}

// ------------------------------------------------------------------------------------------
// One step of a half-sweep stage (RESID = false) or of the EPI role (RESID = true) on row st.row, one 16-byte
// vector per lane, PAR = the column parity of the role's colour in this row.  With pair index kk even, the
// horizontal neighbours of targets (kk, kk+1) are three consecutive nodes of the OTHER run: from kk-1 (even
// columns: O[kk-1], O[kk], O[kk+1]) or from kk (odd columns: E[kk], E[kk+1], E[kk+2]).
//   LAST    the warp's rows go to the bulk-store engine; NORM1: it also sums the residual of its own targets
//   RESID   nothing is updated: the residual of the nodes is injected (EPI = POST_INJECT: even columns of even
//           rows), squared and summed (POST_NORM2) or stored for the full weighting (POST_FW)
//   EPI = POST_FW on the last stage (RESID = false): it stores the residual of its own nodes (all operands in
//           registers) into the residual rows before it publishes the step
//   CHECKED the step may touch rows outside [R0, R1] (first and last steps of a tile): their loads are skipped
//   FULL    steady state of a strip that touches neither side of the domain: the update is active and every lane
//           stores (the strip's outermost pairs are halo: what is computed there is never used), so the step
//           carries no mask, no range test and no predicated load
template <int ARITH, bool LAST, bool NORM1, bool RESID, int EPI, bool FULL, bool BATCH>
SY_FN void stage_step(const Params& p, const Tile& tl, const Geo& geo, const Smem& sm, Stage& st, const int k, const int PAR,
                      const bool CHECKED, FwSums* fw)
{
    const unsigned po = PAR ? geo.swkb : 0u, oo = PAR ? 0u : geo.swkb;
    const unsigned c = st.a_cur + po;
    const int row = st.row;
    // is the row itself / the row below staged?  (a lane outside the strip shadows the last live vector and
    // must not load what that lane is storing)
    const bool own_ok = !CHECKED || (row >= tl.R0 && row <= tl.R1);
    const bool dn_ok = !CHECKED || (row + 1 >= tl.R0 && row + 1 <= tl.R1);
#ifdef SY_HOST_MODEL
    const bool live = st.live;       // (the race detector of the host model would flag the shadow lanes' loads)
#else
    const bool live = true;          // on the device a duplicate load is harmless and cheaper than a predicate
#endif
    // ---- first look at the counters this step depends on: issued before the step's own loads, so that in the
    // steady state the answer is there when it is needed
    Prog2 seen{0u, 0u};
    if (st.up >= 0) seen = sy_prog_peek(sm, st.up);
    Prog2 seen_epi{0u, 0u};
    if (EPI == POST_FW && !RESID) seen_epi = sy_prog_peek(sm, PAIR_EPI);
    // ---- before the wait: everything that does not depend on the last step of the role above
    const bool work = !RESID || EPI == POST_NORM2 || EPI == POST_FW || PAR == 0;   // injection: even columns (of even rows) only
    D2 f{0.0, 0.0}, w1{0.0, 0.0}, w2{0.0, 0.0}, own{0.0, 0.0};
    double x = 0.0;
    const D2 up = st.c_up, m = st.c_mid;
    if (work && own_ok && live) {
        f = sy_lds2(sm, c + geo.ringb); w1 = sy_lds2(sm, c + 2u * geo.ringb); w2 = sy_lds2(sm, c + 3u * geo.ringb);
        if (RESID) own = sy_lds2(sm, c);
    }
    if (work && own_ok) x = sy_side(sm, m, st.a_cur + oo + (PAR ? 16u : 0u) - (PAR ? 0u : 8u), PAR ? 1 : -1, PAR ? st.outer_r : st.outer_l);
    const double n0 = PAR ? m.x : x, n1 = PAR ? m.y : m.x, n2 = PAR ? x : m.y;
    const Coef4 c0 = Arith<ARITH>::coef(w1.x, w2.x, p.st);
    const Coef4 c1 = Arith<ARITH>::coef(w1.y, w2.y, p.st);
    double h0 = 0.0, h1 = 0.0;
    if (!RESID) { h0 = Arith<ARITH>::gs_head(f.x, up.x, n0, c0); h1 = Arith<ARITH>::gs_head(f.y, up.y, n1, c1); }
    // ---- wait for the data of the row below
    wait_inputs(tl, geo, sm, st, k, seen);
    // ---- after the wait
    D2 dn{0.0, 0.0};
    if (dn_ok && live) dn = sy_lds2(sm, st.a_next + po);
    const unsigned rm = PAR ? st.rmask1 : st.rmask0;
    if (!RESID) {
        const double o0 = Arith<ARITH>::gs_tail(h0, dn.x, n1, c0.d, c0.b, p.st);
        const double o1 = Arith<ARITH>::gs_tail(h1, dn.y, n2, c1.d, c1.b, p.st);
        const bool act = FULL || (row >= st.lo && row <= st.hi);
        const unsigned okb = FULL ? 3u : act ? (PAR ? st.okp1 : st.okp0) : 0u;
        // one 16-byte store in the common case: two 8-byte stores at a 16-byte lane stride cost twice the wavefronts
        if (okb == 3u) sy_sts2(sm, c, D2{o0, o1});
        else {
            if (okb & 1u) sy_sts1(sm, c, o0);
            if (okb & 2u) sy_sts1(sm, c + 8u, o1);
        }
        if (EPI == POST_FW) {
            // the row's slot in the residual rows last held row - FW_ROWS, which the EPI warps have finished with once
            // both have published their step on row - FW_ROWS + 2 (they restrict row q after publishing row q + 1):
            // EPI step k + 5 - FW_ROWS (its rows trail this stage's by 2)
            const int need = k + 5 - FW_ROWS;
            if (need > 0) prog_wait(sm, PAIR_EPI, (unsigned)need, geo.nh == 2 ? (unsigned)need : 0u, seen_epi);
            const double r0 = Arith<ARITH>::residual(f.x, o0, up.x, n0, dn.x, n1, c0, p.st);
            const double r1 = Arith<ARITH>::residual(f.y, o1, up.y, n1, dn.y, n2, c1, p.st);
            if (live) sy_sts2(sm, fw_off(tl, geo, st, row) + po, D2{r0, r1});
        }
        // the row is written: publish.  (The last stage's rows go to the bulk-store engine; the generic -> async proxy
        // fence that must lie between these stores and the engine's reads is executed by the STORE warp, after it has
        // acquired this publication: in the stage it cost the one role that never waits for anybody a fifth of its step.)
        publish(sm, st, k);
        if (NORM1 && row >= st.elo && row <= st.ehi) {
            // gs.cpp:75 on the nodes just updated, every operand in registers (owned nodes are never masked)
            const double r0 = Arith<ARITH>::residual(f.x, o0, up.x, n0, dn.x, n1, c0, p.st);
            const double r1 = Arith<ARITH>::residual(f.y, o1, up.y, n1, dn.y, n2, c1, p.st);
            if (rm & 1u) st.acc += r0 * r0;
            if (rm & 2u) st.acc += r1 * r1;
        }
    } else if (EPI == POST_FW) {
        // the first colour's residual into the residual rows, then the step (ring rows released, residual written)
        if (own_ok && live) {
            const double r0 = Arith<ARITH>::residual(f.x, own.x, up.x, n0, dn.x, n1, c0, p.st);
            const double r1 = Arith<ARITH>::residual(f.y, own.y, up.y, n1, dn.y, n2, c1, p.st);
            sy_sts2(sm, fw_off(tl, geo, st, row) + po, D2{r0, r1});
        }
        publish(sm, st, k);
        fw_restrict_row<BATCH>(p, tl, geo, sm, st, *fw, k, row - 1, live);
    } else {
        publish(sm, st, k);                              // nothing written: only the rows' release is signalled
        if (work && row >= st.elo && row <= st.ehi && (EPI == POST_NORM2 || (row & 1) == 0)) {
            const double r0 = Arith<ARITH>::residual(f.x, own.x, up.x, n0, dn.x, n1, c0, p.st);
            const double r1 = Arith<ARITH>::residual(f.y, own.y, up.y, n1, dn.y, n2, c1, p.st);
            if (EPI == POST_INJECT) {
                // gs.cpp:283: coarse node (row/2, kg) for fine even column 2kg
                store_coarse<BATCH>(p, st, (long)tl.k0 + st.kk, row >> 1, r0, r1);
            } else {
                if (rm & 1u) st.acc += r0 * r0;
                if (rm & 2u) st.acc += r1 * r1;
            }
        }
    }
    st.c_up = m; st.c_mid = dn;
    advance_row(geo, st);
}

template <int ARITH, bool LAST, bool NORM1, bool RESID, int EPI, int XR = 0, bool BATCH = false>
SY_FN void stage_loop(const Params& p, const Tile& tl, const Geo& geo, const Smem& sm, Stage& st)
{
    const int klast = last_step(p, tl, XR) - tl.R0;
    FwSums fw{D2{0.0, 0.0}, D2{0.0, 0.0}};
    // column parity of the role's colour in its row: (s + row) & 1
    int par = (st.s + st.row) & 1;
    int k = 0;
    // first steps: rows above R0 (checked); then align the unrolled loop on parity 0; last steps: rows below R1
    // (checked: the slots of unstaged rows may still be in use by the roles behind).  Unchecked steps: the update
    // is active (row in [R0+1, R1-1]), hence rows row-1 .. row+1 staged.
    const int kchk = st.off + 1;
    int kmain = tl.R1 - tl.R0 + st.off - 1;
    if (kmain > klast) kmain = klast;
    // a strip that touches neither side of the domain runs the mask-free step (every lane must be live)
    const bool full = !RESID && tl.k0 >= 1 && (long)tl.k0 + p.SWK <= p.nhalf && (p.SWK & 63) == 0;
    for (; k <= klast && (k < kchk || par != 0); ++k, par ^= 1)
        stage_step<ARITH, LAST, NORM1, RESID, EPI, false, BATCH>(p, tl, geo, sm, st, k, par, true, &fw);
    if (full) {
        for (; k + 1 <= kmain; k += 2) {
            stage_step<ARITH, LAST, NORM1, RESID, EPI, true, BATCH>(p, tl, geo, sm, st, k, 0, false, &fw);
            stage_step<ARITH, LAST, NORM1, RESID, EPI, true, BATCH>(p, tl, geo, sm, st, k + 1, 1, false, &fw);
        }
    } else {
        for (; k + 1 <= kmain; k += 2) {
            stage_step<ARITH, LAST, NORM1, RESID, EPI, false, BATCH>(p, tl, geo, sm, st, k, 0, false, &fw);
            stage_step<ARITH, LAST, NORM1, RESID, EPI, false, BATCH>(p, tl, geo, sm, st, k + 1, 1, false, &fw);
        }
    }
    for (; k <= klast; ++k, par ^= 1)
        stage_step<ARITH, LAST, NORM1, RESID, EPI, false, BATCH>(p, tl, geo, sm, st, k, par, true, &fw);
}

// ------------------------------------------------------------------------------------------
// load warp: request group g (first memory row z) into its ring slot: the four fields plus the three
// coarse rows its prolongation needs, all completing on the slot's full barrier; then start the HBM
// fetch of the group after next, whose shared-memory request will hit L2.  Whole (converged) warp,
// warp-uniform operands; one elected lane issues.
template <bool BATCH>
SY_FN void issue_group_loads(const Params& p, const Tile& tl, const Geo& geo, const Smem& sm, int g)
{
    if (!sy_elect()) return;
    const int gs = g % NGROUP;
    const int z = tl.R0 + GROUP * g - (int)p.row0;
    const unsigned fine = (unsigned)GROUP * geo.rowb;
    sy_full_expect(sm, gs, 4u * fine + (p.pre ? geo.cgrpb : 0u));
    const unsigned so = (unsigned)gs * fine;
    // a zero iterate is produced by a box that lies entirely below the last memory row
    if constexpr (BATCH) {                                           // the same boxes of member sy_member()
        const int m = sy_member();
        sy_tma_load_m(p, sm, FIELD_U, so, tl.k0, p.u_is_zero ? (int)p.rows_mem + 64 : z, m, gs);
        sy_tma_load_m(p, sm, FIELD_F, so + geo.ringb, tl.k0, z, m, gs);
        sy_tma_load_m(p, sm, FIELD_V1, so + 2u * geo.ringb, tl.k0, z, m, gs);
        sy_tma_load_m(p, sm, FIELD_V2, so + 3u * geo.ringb, tl.k0, z, m, gs);
        if (p.pre)
            sy_tma_load_m(p, sm, FIELD_C, 4u * geo.ringb + (unsigned)gs * geo.cgrpb, tl.k0 / 2, (z >> 1), m, gs);
        const int zp = z + 2 * GROUP;
        if (g + 2 >= NGROUP && zp <= tl.R1) {
            if (!p.u_is_zero) sy_tma_prefetch_m(p, FIELD_U, tl.k0, zp, m);
            sy_tma_prefetch_m(p, FIELD_F, tl.k0, zp, m);
            sy_tma_prefetch_m(p, FIELD_V1, tl.k0, zp, m);
            sy_tma_prefetch_m(p, FIELD_V2, tl.k0, zp, m);
        }
        return;
    }
    sy_tma_load(p, sm, FIELD_U, so, tl.k0, p.u_is_zero ? (int)p.rows_mem + 64 : z, gs);
    sy_tma_load(p, sm, FIELD_F, so + geo.ringb, tl.k0, z, gs);
    sy_tma_load(p, sm, FIELD_V1, so + 2u * geo.ringb, tl.k0, z, gs);
    sy_tma_load(p, sm, FIELD_V2, so + 3u * geo.ringb, tl.k0, z, gs);
    if (p.pre)
        sy_tma_load(p, sm, FIELD_C, 4u * geo.ringb + (unsigned)gs * geo.cgrpb, tl.k0 / 2, ((z + (int)p.row0) >> 1) - (int)p.crow0, gs);
    const int zp = z + 2 * GROUP;
    if (g + 2 >= NGROUP && zp + (int)p.row0 <= tl.R1) {               // (the first NGROUP groups are requested at once)
        if (!p.u_is_zero) sy_tma_prefetch(p, FIELD_U, tl.k0, zp);
        sy_tma_prefetch(p, FIELD_F, tl.k0, zp);
        sy_tma_prefetch(p, FIELD_V1, tl.k0, zp);
        sy_tma_prefetch(p, FIELD_V2, tl.k0, zp);
    }
}

// Two single warps drain and feed the ring (warp-uniform code, one elected lane issues).
//
// The STORE warp follows the last stage.  In step k that stage finishes row rs = t - off(last): the row goes to the
// bulk-store engine as soon as both of its warps have published the step -- after the generic -> async proxy fence,
// executed here, on the acquiring side (see stage_step).  The stores are committed as ONE bulk group
// per ring group (a commit per row flushes the TMA command queue every row); after the commit the warp waits until the
// engine has read the group's rows and publishes the number of groups done in its own counter.
//
// The LOAD warp follows the last ROLE (the EPI role if the pass has one, else the last stage), which releases the ring
// rows: once it has published its step on row rl it needs no row <= rl any more (what it still uses of row rl+1 it
// carries in registers), so group g (first row G), which replaces rows G-RING .. G-RING+GROUP-1 (ring group g - NGROUP),
// is requested once row G-RING+GROUP-1 is published and the store warp has counted that group.
template <int XR = 0, bool BATCH = false>
SY_FN void store_loop(const Params& p, const Tile& tl, const Geo& geo, const Smem& sm)
{
    const int klast = last_step(p, tl, XR) - tl.R0;
    const int pair_s = 2 * p.K - 1, off_s = off_stage(p, pair_s);
    long eE = (long)tl.kb + p.WK, eO = eE;
    if (eE > p.nhalf + 1) eE = p.nhalf + 1;
    if (eO > p.nhalf) eO = p.nhalf;
    const unsigned nE8 = (unsigned)(((eE - tl.kb + 1) & ~1L) * 8);   // whole 16-byte units (the layout has slack)
    const unsigned nO8 = (unsigned)((eO - tl.kb) * 8);
    int rs = tl.R0 - off_s;                                          // the last stage's row in step 0
    const long pitch = p.pitch;
    double* gstE = p.u_out + member_off<BATCH>(p.mstride) + ((long)rs - p.row0) * pitch + tl.kb;    // destinations of the row's two runs
    double* gstO = gstE + p.odd;
    unsigned a = (unsigned)((((rs - tl.R0) % RING) + RING) % RING) * geo.rowb + (unsigned)HK * 8u;
    const unsigned awrap = geo.ringb + (unsigned)HK * 8u;
    const unsigned need_h1 = geo.nh == 2 ? 1u : 0u;
    Prog2 seen_s{0u, 0u};
    unsigned groups = 0;
    for (int k = 0; k <= klast; ++k, ++rs) {
        const bool store = rs >= tl.rb0 && rs <= tl.rb1;
        const bool close = rs >= tl.R0 && ((rs - tl.R0) & (GROUP - 1)) == GROUP - 1;     // the row closes a ring group
        // (the last stage is usually more than one row ahead: the counters are read again only when the values seen
        // last do not cover this row)
        if ((store || close) && (seen_s.h0 < (unsigned)k + 1u || seen_s.h1 < need_h1 * ((unsigned)k + 1u))) {
            seen_s = sy_prog_peek(sm, pair_s);
            while (seen_s.h0 < (unsigned)k + 1u || seen_s.h1 < need_h1 * ((unsigned)k + 1u)) { sy_backoff(pair_s); seen_s = sy_prog_peek(sm, pair_s); }
        }
        if (close) ++groups;
        if ((store || close) && sy_elect()) {
            if (store) {
                sy_fence_async();                                    // the stages' stores (acquired above) -> the engine's reads
                if (nE8) sy_bulk_store(sm, gstE, a, nE8);
                if (nO8) sy_bulk_store(sm, gstO, a + geo.swkb, nO8);
            }
            if (close) {
                sy_store_commit();
                sy_store_wait_read0();
                sy_prog_publish(sm, 2 * PAIR_STORE, groups);
            }
        }
        gstE += pitch; gstO += pitch;
        a += geo.rowb;
        if (a >= awrap) a -= geo.ringb;
    }
    if (sy_elect()) { sy_store_commit(); sy_store_wait_all(); sy_prog_publish(sm, 2 * PAIR_STORE, groups + 64u); }
}

template <int XR = 0, bool BATCH = false>
SY_FN void producer_loop(const Params& p, const Tile& tl, const Geo& geo, const Smem& sm)
{
    const int ng = num_groups(tl);
    int gnext = 0;
    for (; gnext < ng && gnext < NGROUP; ++gnext) issue_group_loads<BATCH>(p, tl, geo, sm, gnext);   // fresh slots
    const int klast = last_step(p, tl, XR) - tl.R0;
    const int pair_s = 2 * p.K - 1, off_s = off_stage(p, pair_s);
    const bool epi = p.post != POST_NONE;
    const int pair_l = epi ? PAIR_EPI : pair_s, off_l = epi ? off_epi(p) : off_s;
    const unsigned need_h1 = geo.nh == 2 ? 1u : 0u;
    int rl = tl.R0 - off_l;                                          // the last role's row in step 0
    for (int k = 0; k <= klast && gnext < ng; ++k, ++rl) {
        if (rl < tl.R0 + GROUP * gnext - RING + GROUP - 1) continue;
        prog_wait(sm, pair_l, (unsigned)k + 1u, need_h1 * ((unsigned)k + 1u), sy_prog_peek(sm, pair_l));
        // ring group gnext - NGROUP must have left shared memory: the store warp has counted gnext - NGROUP + 1 groups
        prog_wait(sm, PAIR_STORE, (unsigned)(gnext - NGROUP + 1), 0u, sy_prog_peek(sm, PAIR_STORE));
        if (sy_elect()) sy_fence_async();                            // the stages' stores into the slots -> the engine's writes
        issue_group_loads<BATCH>(p, tl, geo, sm, gnext);
        ++gnext;
    }
}

// the work of one warp on one tile; returns the thread's share of the POST_NORM2 sum.  BATCH: the tile belongs to
// member sy_member() of a batch, whose fields the 4-D tensor maps address
template <int ARITH, bool PRE, int POSTK, bool BATCH = false>
SY_FN double run_warp(const Params& p, const Tile& tl, const Geo& geo, const Smem& sm, int warp, int lane)
{
    constexpr int XR = POSTK == POST_FW ? 2 : 0;       // extra steps of every role (last_step)
    if (warp == PRODUCER_WARP) {
        // the producer's lanes run in lockstep on the device (warp-uniform code, one elected lane issues); the host
        // model runs lanes as free threads, so it lets only the issuing lane walk the loop
#ifdef SY_HOST_MODEL
        if (lane != 0) return 0.0;
#endif
        producer_loop<XR, BATCH>(p, tl, geo, sm);
        return 0.0;
    }
    if (warp == STORE_WARP) {
#ifdef SY_HOST_MODEL
        if (lane != 0) return 0.0;
#endif
        store_loop<XR, BATCH>(p, tl, geo, sm);
        return 0.0;
    }
    const int pair = warp / NSTW, h = warp % NSTW;
    if (h >= geo.nh) return 0.0;
    const int last = 2 * p.K - 1;
    if (pair == PAIR_PRE) {
        if (!PRE) return 0.0;
        Stage st = init_role(p, tl, geo, PAIR_PRE, -1, 1, 0, h, lane);
        pre_loop(p, tl, geo, sm, st);
        return 0.0;
    }
    if (pair == PAIR_EPI) {
        if (POSTK == POST_NONE) return 0.0;
        Stage st = init_role(p, tl, geo, PAIR_EPI, last, 2 * p.K, off_epi(p), h, lane);
        stage_loop<ARITH, false, false, true, POSTK, XR, BATCH>(p, tl, geo, sm, st);
        return st.acc;
    }
    if (pair > last) return 0.0;
    Stage st = init_role(p, tl, geo, pair, pair == 0 ? (PRE ? PAIR_PRE : -1) : pair - 1, pair, off_stage(p, pair), h, lane);
    // (the last stage differs from the others only where it sums or stores its own residual)
    if (pair == last && POSTK == POST_NORM2) stage_loop<ARITH, true, true, false, POST_NONE, 0, BATCH>(p, tl, geo, sm, st);
    else if (pair == last && POSTK == POST_FW) stage_loop<ARITH, true, false, false, POST_FW, XR, BATCH>(p, tl, geo, sm, st);
    else stage_loop<ARITH, false, false, false, POST_NONE, XR, BATCH>(p, tl, geo, sm, st);
    return st.acc;
}

// ------------------------------------------------------------------------------------------
// Tile planner.  Cost model (relative): a tile takes (rows + fill) steps, a step costs
// c0 + SWK (latency + work proportional to the strip width); tiles run one per SM in waves of
// `sms`.  Search strip width (SWK a multiple of 16: TMA boxes land 128-byte aligned) and band
// count for the cheapest plan.  A batched pass runs the same tiles for each of `members` members,
// so its waves count members x tiles (members = 1: the plan of a single problem).
struct Plan { int WK, SWK, nstrips, nbands; long RBAND; };

// n: level size (columns); nrows: rows this launch produces (n+1 on a single GPU, the slab otherwise)
inline Plan make_plan(long n, long nrows, int K, int sms, int force_swk = 0, int members = 1)
{
    const long npairs = n / 2 + 1;
    Plan best{};
    double best_cost = 1e300;
    for (int SWK = 32; SWK <= SWK_MAX; SWK += 16) {
        if (force_swk && SWK != force_swk) continue;
        const int WK = SWK - 2 * HK;
        const int nstrips = (int)((npairs + WK - 1) / WK);
        for (int nb = 1; nb <= 4096; nb = nb < 16 ? nb + 1 : nb * 2) {
            const long RB = (nrows + nb - 1) / nb;
            if (nb > 1 && RB < 8) break;
            const int nbands = (int)((nrows + RB - 1) / RB);
            const long tiles = (long)nstrips * nbands * members;
            const long waves = (tiles + sms - 1) / sms;
            const double steps = (double)RB + 2.0 * (2 * K + 1) + 4.0 * K + 2.0 * GROUP;
            const double per_step = 96.0 + SWK;
            const double cost = (double)waves * steps * per_step;
            if (cost < best_cost) { best_cost = cost; best = Plan{WK, SWK, nstrips, nbands, RB}; }
        }
    }
    return best;
}

}  // namespace sy
}  // namespace mgb200
