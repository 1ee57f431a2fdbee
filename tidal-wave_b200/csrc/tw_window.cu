// tw_window.cu -- K4 / K5 for the Gaussian window of radius 15 (winSize 30 / 31, the reference's default): ONE persistent,
// warp-specialised CTA per SM that slides down 64-column strips of the M planes.
//
//   Farneback stages A.5 (window blur of the five M planes + 2x2 solve) and A.4 (next update-matrices) of SURVEY App. A --
//   the per-iteration body of cv::calcOpticalFlowFarneback, /root/reference/src/opticalflow.cpp:83-85 -- fused into one
//   pass: per iteration M (20 B/px), R0 (20), R1 (20) are read once and M' (20) is written once.
//
// Roles of the warps of a CTA (one CTA per SM, ~206 KB of shared memory).  The kernel is launched with 20 warps at 96 registers;
// the four warps of the last warpgroup (the TMA producer and three spares that exit) shrink to 24 registers and the sixteen working
// warps grow to 112 (setmaxnreg; USETMAXREG in SASS).  Every scheduler of the SM holds two V warps and two H / U warps, so the
// FFMA2-dense vertical pass and the load / FP64 / address-heavy solve and update passes share each issue port:
//   warps 0-7    V walkers: thread = (column, channel pair) [warps 0-5] or (column pair, h2) [warps 6-7, 48 lanes].  Each keeps a
//                40-row sliding window of its column in REGISTERS for the whole strip, so an M row is read from L2 exactly once
//                per strip and there is no cold start per tile; per 8-row group: 8 new rows from the M ring, 8 outputs x 31
//                taps as packed f32x2 (FFMA2), taps in the oracle's order -> the P ring.
//   warps 8-15   two teams of four warps that take alternate groups, each H + solve + U: horizontal taps from the P ring (lane =
//                row x 4-pixel quad, conflict-free LDS.128), 2x2 solve in double -> the team's flow tile in shared memory; then
//                (not last) the next update matrices (A.4) with R0 / R1 read from shared memory, two vertically adjacent pixels
//                per packed f32x2 instruction on the warp-uniform fast path (all pixels inside, within the staged R1 window,
//                off the damped frame border), a scalar per-pixel path otherwise (pixels whose displaced position leaves the
//                staged window -- large motion -- gather from global memory; same values, same arithmetic) -> M' stores;
//                (last) flow stores + the fused span-grid threshold count.
//   warp 16      TMA producer (one lane): tensor-map bulk copies (cp.async.bulk.tensor, UTMALDG) issued as far ahead as the rings
//                allow -- the M rows (8-row chunks, one 8-row box per plane; at the frame top / bottom one row per copy with the
//                row coordinate clamped = the replicate border of App. A.5; 3 slots), the R0 tile of each group (64 x 8 x 5
//                channels; 3 slots) and the R1 rows its bilinear gather can touch (72 columns x rows y-8 .. y+15, a 6-chunk row
//                ring).  Out-of-frame parts are zero-filled by the TMA unit and never read.  It polls the "empty" barriers
//                (mbarrier.test_wait) and never blocks on one stream while another could be served.
//   All hand-offs are mbarrier pipelines (full / empty per ring slot; an R1 chunk is read by three consecutive groups, i.e. by
//   both teams: each team arrives after its last use of the chunk) plus one 128-thread named barrier per team between H and U.
//   Every wait traps after ~2 s instead of hanging the device.
//
// What was measured on the way (DESIGN.md section 4.1): 96-column strips with 10 V + 6 H / U warps and the producers inside two V
// warps ran 38 % SLOWER than the tile kernel (the H / U warps, 1.5 per scheduler and latency-bound, held the V walkers back, and
// the producers' polling sat on the V warps' critical path); 64-column strips with a dedicated producer warp at 96 registers and
// eight software-pipelined H / U warps (2 pixels per lane: too little ILP) 23 % slower; the same with the producer replaced by
// "the last consumer of a slot refills it" 40 % slower (the refill code and its atomics moved onto the consumers' critical
// path).  This form comes within 1-2 % of the tile kernel at 1920x1080 in the relaxed arithmetic (2.36 vs 2.33 ms per step) and is
// 5-7 % slower in the faithful arithmetic (three packed instructions per tap pair instead of two) and at 3840x2160: it is an
// opt-in ("window_tiles" = 0, TW_WINDOW=strip), the tile kernel stays the default.
//
// Arithmetic per output is exactly that of gauss_iter2_kernel (tw_kernels.cu): FMA = 0 the oracle's add-mul-add order
// (bit-identical to oracle/farneback_ref.c), FMA = 2 the direct-form fmaf taps of the relaxed default (oracle relax bit 7).
#include "tw_device.cuh"

#include <cuda.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>

namespace tw {

namespace {

constexpr int WS_SW = 64;                 // output columns per strip
constexpr int WS_XH = 16;                 // left halo of the V columns (15 needed, 16 keeps the copies 64-byte aligned)
constexpr int WS_VC = WS_SW + 2 * WS_XH;  // 96 V columns
constexpr int WS_G = 8;                   // rows per group
constexpr int WS_MR = 15;
constexpr int WS_WIN = 40;                // register window rows = 5 chunks
constexpr int WS_NR0 = 3;
constexpr int WS_NM = 3, WS_NP = 3, WS_NR1 = 6, WS_NF = 4; // WS_NF: 2 teams x 2 slots
constexpr int WS_MPROW = 2 * WS_VC * 4, WS_MHROW = WS_VC * 4;         // bytes per staged row of a channel-pair plane / of the h2 plane
constexpr int WS_MP1OFF = WS_G * WS_MPROW, WS_MHOFF = 2 * WS_MP1OFF;  // chunk layout: pair01[8 rows] | pair23[8 rows] | h2[8 rows]
constexpr int WS_MCHUNK = WS_MHOFF + WS_G * WS_MHROW;                 // 15360
constexpr int WS_P2 = 98, WS_P4 = 100;                                // float2 / float pitches of the P planes (= 4 words mod 32)
constexpr int WS_P23OFF = WS_G * WS_P2 * 8, WS_P4OFF = 2 * WS_P23OFF; // 6272, 12544
constexpr int WS_PSLOT = WS_P4OFF + WS_G * WS_P4 * 4;                 // 15744
constexpr int WS_R0SLOT = WS_G * 5 * WS_SW * 4;                       // 10240
constexpr int WS_R1C = 72, WS_R1X = 4;                                // staged R1 columns: x0 - 4 .. x0 + 67
constexpr int WS_R1ROW = 5 * WS_R1C;                                  // floats per ring row
constexpr int WS_R1CHUNK = WS_G * WS_R1ROW * 4;                       // 11520
constexpr int WS_R1RING = WS_NR1 * WS_G;                              // ring rows
constexpr int WS_FP = 65;                                             // flow tile pitch
constexpr int WS_FSLOT = 2 * WS_G * WS_FP * 4;                        // 4352

constexpr int WS_OFF_M = 0;
constexpr int WS_OFF_P = WS_OFF_M + WS_NM * WS_MCHUNK;
constexpr int WS_OFF_R0 = WS_OFF_P + WS_NP * WS_PSLOT;
constexpr int WS_OFF_R1 = WS_OFF_R0 + WS_NR0 * WS_R0SLOT;
constexpr int WS_OFF_F = WS_OFF_R1 + WS_NR1 * WS_R1CHUNK;
constexpr int WS_OFF_BAR = WS_OFF_F + WS_NF * WS_FSLOT;
constexpr int WS_NBAR = 2 * (WS_NM + WS_NP + WS_NR0 + WS_NR1); // full / empty per ring slot
constexpr int WS_SMEM = WS_OFF_BAR + WS_NBAR * 8;
static_assert(WS_OFF_P % 128 == 0 && WS_OFF_R0 % 128 == 0 && WS_OFF_R1 % 128 == 0 && WS_R0SLOT % 128 == 0 && WS_R1CHUNK % 128 == 0 &&
                  WS_MPROW % 128 == 0 && WS_MHROW % 128 == 0 && WS_MCHUNK % 128 == 0,
              "TMA destinations are 128-byte aligned");
static_assert(WS_OFF_F % 16 == 0 && WS_OFF_BAR % 8 == 0 && WS_SMEM <= 227 * 1024, "shared memory budget");

constexpr int WS_NVW = 8, WS_NHW = 8;                  // V walker warps, H / U warps (two teams of WS_TEAMW)
constexpr int WS_TEAMW = 4, WS_TEAM_THREADS = WS_TEAMW * 32;
constexpr int WS_VLANES = 2 * WS_VC + WS_VC / 2;       // 240 walkers
constexpr int WS_PRODW = WS_NVW + WS_NHW;              // the producer warp; it and the three spare warps of its warpgroup give their
constexpr int WS_THREADS = (WS_NVW + WS_NHW + 4) * 32; // registers to the other sixteen (setmaxnreg): 640 threads launched at 96
constexpr int WS_REGS_WORK = 112, WS_REGS_PROD = 24;

// barrier indices
constexpr int B_FULLM = 0, B_EMPTYM = B_FULLM + WS_NM, B_FULLP = B_EMPTYM + WS_NM, B_EMPTYP = B_FULLP + WS_NP,
              B_FULLR0 = B_EMPTYP + WS_NP, B_EMPTYR0 = B_FULLR0 + WS_NR0, B_FULLR1 = B_EMPTYR0 + WS_NR0, B_EMPTYR1 = B_FULLR1 + WS_NR1;

__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ unsigned mbar_try(unsigned bar, unsigned parity)
{
    unsigned done;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done)
                 : "r"(bar), "r"(parity)
                 : "memory");
    return done;
}
// Waits for the phase with the given parity: try_wait suspends the warp in hardware for a short, implementation-defined time
// and is simply repeated.  A wait of more than ~2 s means a broken pipeline: trap (the launch fails with an error) instead of
// hanging the device.
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity)
{
    if (mbar_try(bar, parity)) return;
#pragma unroll 1
    for (unsigned it = 0; !mbar_try(bar, parity); ++it)
        if (it > (1u << 26)) __trap();
}
__device__ __forceinline__ void tma_load_3d(unsigned dst, const CUtensorMap *map, int x, int y, int z, unsigned bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
                 "l"(reinterpret_cast<unsigned long long>(map)), "r"(bar), "r"(x), "r"(y), "r"(z)
                 : "memory");
}
__device__ __forceinline__ float lds32(unsigned addr)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ float2 lds64(unsigned addr)
{
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts64(unsigned addr, float2 v)
{
    asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(v.x), "f"(v.y) : "memory");
}
// non-blocking probe (the producer polls with it)
__device__ __forceinline__ unsigned mbar_test(unsigned bar, unsigned parity)
{
    unsigned done;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done)
                 : "r"(bar), "r"(parity)
                 : "memory");
    return done;
}
__device__ __forceinline__ void team_barrier(int team) { asm volatile("bar.sync %0, %1;" ::"r"(1 + team), "n"(WS_TEAM_THREADS) : "memory"); }

struct Unit {
    int b, x0, y0, ng;
};

} // namespace

struct StripArgs {
    const float *R; // [B][2][5] planes (global gathers of pixels that leave the staged R1 window)
    float *Mout;    // [B][5] planes
    float *flow;    // [B][2] planes (LAST)
    LevelDims d;
    int nsx, nsy, segh, nunits;
    int span;
    double thr2;
    int *counts;
    int dbg; // TW_STRIP_DEBUG builds only: bit 0 skip the V taps, bit 1 skip H + solve, bit 3 skip U
    unsigned *prof; // TW_STRIP_DEBUG builds only: [grid][16 warps][8] phase clocks
};

namespace {

#ifdef TW_STRIP_DEBUG
#define WS_DBG(bit) (a.dbg & (bit))
#define WS_PROF_DECL unsigned pacc_[8] = {0, 0, 0, 0, 0, 0, 0, 0}, pt0_ = clock();
#define WS_PROF(i) { const unsigned t1_ = clock(); pacc_[i] += t1_ - pt0_; pt0_ = t1_; }
#define WS_PROF_DUMP if (a.prof && lane == 0) for (int i_ = 0; i_ < 8; i_++) a.prof[(blockIdx.x * 16 + warp) * 8 + i_] = pacc_[i_];
#else
#define WS_DBG(bit) 0
#define WS_PROF_DECL
#define WS_PROF(i)
#define WS_PROF_DUMP
#endif

__device__ __forceinline__ Unit decode_unit(const StripArgs &a, int u)
{
    Unit U;
    const int sy = u % a.nsy, rest = u / a.nsy;
    const int sx = rest % a.nsx;
    U.b = rest / a.nsx;
    U.x0 = sx * WS_SW;
    U.y0 = sy * a.segh;
    U.ng = (min(a.segh, a.d.h - U.y0) + WS_G - 1) / WS_G;
    return U;
}

// ---- TMA producer: three streams that run across the CTA's unit sequence; each pump issues while a ring slot is free ----
// M rows: every unit contributes ng + 4 chunks of 8 rows (rows y0 - 15 + 8c ..); R0 tiles: one per group; R1 row chunks: ng + 2
// per unit (rows y0 - 8 + 8c .. + 7 of the target image's expansion).
struct Stream {
    int u, c;
    Unit U;
    unsigned n; // chunks issued so far
};

__device__ __forceinline__ bool pump_m(Stream &ms, const StripArgs &a, unsigned smem, const CUtensorMap *mp1, const CUtensorMap *mh1,
                                       const CUtensorMap *mp8, const CUtensorMap *mh8)
{
    bool any = false;
    while (ms.u < a.nunits) {
        const unsigned s = ms.n % WS_NM;
        if (!mbar_test(smem + WS_OFF_BAR + 8 * (B_EMPTYM + s), ((ms.n / WS_NM) & 1) ^ 1)) break;
        const unsigned bar = smem + WS_OFF_BAR + 8 * (B_FULLM + s);
        mbar_expect_tx(bar, WS_MCHUNK);
        const unsigned dst = smem + WS_OFF_M + s * WS_MCHUNK;
        const int xs = ms.U.x0 - WS_XH, pitch = a.d.pitch, h = a.d.h;
        const int yf = ms.U.y0 - WS_MR + WS_G * ms.c;
        if (yf >= 0 && yf + WS_G - 1 <= h - 1) {
            tma_load_3d(dst, mp8, 2 * xs, yf, ms.U.b, bar);
            tma_load_3d(dst + WS_MP1OFF, mp8, 2 * pitch + 2 * xs, yf, ms.U.b, bar);
            tma_load_3d(dst + WS_MHOFF, mh8, 4 * pitch + xs, yf, ms.U.b, bar);
        } else { // frame top / bottom: replicate = clamped row coordinate, one row per copy
#pragma unroll 1
            for (int r = 0; r < WS_G; r++) {
                const int y = clampi(yf + r, 0, h - 1);
                tma_load_3d(dst + r * WS_MPROW, mp1, 2 * xs, y, ms.U.b, bar);
                tma_load_3d(dst + WS_MP1OFF + r * WS_MPROW, mp1, 2 * pitch + 2 * xs, y, ms.U.b, bar);
                tma_load_3d(dst + WS_MHOFF + r * WS_MHROW, mh1, 4 * pitch + xs, y, ms.U.b, bar);
            }
        }
        any = true;
        ms.n++;
        if (++ms.c == ms.U.ng + 4) {
            ms.c = 0;
            ms.u += gridDim.x;
            if (ms.u < a.nunits) ms.U = decode_unit(a, ms.u);
        }
    }
    return any;
}

__device__ __forceinline__ bool pump_r0(Stream &rs, const StripArgs &a, unsigned smem, const CUtensorMap *r0map)
{
    bool any = false;
    while (rs.u < a.nunits) {
        const unsigned s = rs.n % WS_NR0;
        if (!mbar_test(smem + WS_OFF_BAR + 8 * (B_EMPTYR0 + s), ((rs.n / WS_NR0) & 1) ^ 1)) break;
        const unsigned bar = smem + WS_OFF_BAR + 8 * (B_FULLR0 + s);
        mbar_expect_tx(bar, WS_R0SLOT);
        tma_load_3d(smem + WS_OFF_R0 + s * WS_R0SLOT, r0map, rs.U.x0, 5 * (rs.U.y0 + WS_G * rs.c), 2 * rs.U.b, bar);
        any = true;
        rs.n++;
        if (++rs.c == rs.U.ng) {
            rs.c = 0;
            rs.u += gridDim.x;
            if (rs.u < a.nunits) rs.U = decode_unit(a, rs.u);
        }
    }
    return any;
}

__device__ __forceinline__ bool pump_r1(Stream &rs, const StripArgs &a, unsigned smem, const CUtensorMap *r1map)
{
    bool any = false;
    while (rs.u < a.nunits) {
        const unsigned s = rs.n % WS_NR1;
        if (!mbar_test(smem + WS_OFF_BAR + 8 * (B_EMPTYR1 + s), ((rs.n / WS_NR1) & 1) ^ 1)) break;
        const unsigned bar = smem + WS_OFF_BAR + 8 * (B_FULLR1 + s);
        mbar_expect_tx(bar, WS_R1CHUNK);
        tma_load_3d(smem + WS_OFF_R1 + s * WS_R1CHUNK, r1map, rs.U.x0 - WS_R1X, 5 * (rs.U.y0 - WS_G + WS_G * rs.c), 2 * rs.U.b + 1, bar);
        any = true;
        rs.n++;
        if (++rs.c == rs.U.ng + 2) {
            rs.c = 0;
            rs.u += gridDim.x;
            if (rs.u < a.nunits) rs.U = decode_unit(a, rs.u);
        }
    }
    return any;
}

// 8 outputs x 31 taps of one walker from its register window (rows 8g .. 8g + 39 of the unit's M rows) -> P slot.
template <int FMA>
__device__ __forceinline__ void v_compute(const float2 (&win)[WS_WIN], unsigned pd, unsigned dstride, const WinTaps &t, bool store)
{
    const float2 one2 = make_float2(t.one, t.one);
    float2 v[WS_G];
#pragma unroll
    for (int o = 0; o < WS_G; o++) v[o] = tw_mul2(win[o + WS_MR], make_float2(t.k[0], t.k[0]));
#pragma unroll
    for (int i = 1; i <= WS_MR; i++) {
        const float2 kk = make_float2(t.k[i], t.k[i]);
        if (FMA == 2) { // direct form (oracle relax bit 7): upper row first
#pragma unroll
            for (int o = 0; o < WS_G; o++) v[o] = tw_fma2(win[o + WS_MR - i], kk, v[o]);
#pragma unroll
            for (int o = 0; o < WS_G; o++) v[o] = tw_fma2(win[o + WS_MR + i], kk, v[o]);
        } else {
#pragma unroll
            for (int o = 0; o < WS_G; o++) {
                const float2 sum = tw_add2(win[o + WS_MR + i], win[o + WS_MR - i]);
                v[o] = tw_fma2(tw_mul2(sum, kk), one2, v[o]); // = v + round(sum * k): see tw_fma2 in tw_device.cuh
            }
        }
    }
    if (store) {
#pragma unroll
        for (int o = 0; o < WS_G; o++) sts64(pd + o * dstride, v[o]);
    }
}

// Horizontal taps + solve for 4 adjacent pixels of one row (P slot pointers already offset to the row and the quad).
template <int FMA>
__device__ __forceinline__ void h_quad(const float2 *__restrict__ p01, const float2 *__restrict__ p23, const float *__restrict__ p4, const WinTaps &t,
                                       float (&fx)[4], float (&fy)[4])
{
    constexpr int MR = WS_MR;
    constexpr int LO = (16 - MR) & ~3;               // first needed V column relative to the quad, 16-byte aligned
    constexpr int NV = ((3 + 16 + MR) | 3) + 1 - LO; // values loaded per plane (multiple of 4)
    const float2 one2 = make_float2(t.one, t.one);
    float2 r01[4], r23[4];
    float r4[4];
#pragma unroll
    for (int pr = 0; pr < 2; pr++) {
        const float4 *src = reinterpret_cast<const float4 *>((pr ? p23 : p01) + LO);
        float2 v[NV];
#pragma unroll
        for (int q = 0; q < NV / 2; q++) {
            const float4 u = src[q];
            v[2 * q] = make_float2(u.x, u.y); v[2 * q + 1] = make_float2(u.z, u.w);
        }
        float2 sacc[4];
#pragma unroll
        for (int p = 0; p < 4; p++) sacc[p] = tw_mul2(v[p + 16 - LO], make_float2(t.k[0], t.k[0]));
#pragma unroll
        for (int i = 1; i <= MR; i++) {
            const float2 kk = make_float2(t.k[i], t.k[i]);
            if (FMA == 2) { // direct form: left tap first
#pragma unroll
                for (int p = 0; p < 4; p++) sacc[p] = tw_fma2(kk, v[p + 16 - LO - i], sacc[p]);
#pragma unroll
                for (int p = 0; p < 4; p++) sacc[p] = tw_fma2(kk, v[p + 16 - LO + i], sacc[p]);
            } else {
#pragma unroll
                for (int p = 0; p < 4; p++) {
                    const int ctr = p + 16 - LO;
                    const float2 sum = tw_add2(v[ctr - i], v[ctr + i]);
                    sacc[p] = tw_fma2(tw_mul2(kk, sum), one2, sacc[p]);
                }
            }
        }
#pragma unroll
        for (int p = 0; p < 4; p++) { if (pr) r23[p] = sacc[p]; else r01[p] = sacc[p]; }
    }
    {
        const float4 *src = reinterpret_cast<const float4 *>(p4 + LO);
        float v[NV];
#pragma unroll
        for (int q = 0; q < NV / 4; q++) {
            const float4 u = src[q];
            v[4 * q] = u.x; v[4 * q + 1] = u.y; v[4 * q + 2] = u.z; v[4 * q + 3] = u.w;
        }
#pragma unroll
        for (int p = 0; p < 4; p += 2) { // pixels (p, p+1) packed
            const int ctr = p + 16 - LO;
            float2 sacc = tw_mul2(make_float2(v[ctr], v[ctr + 1]), make_float2(t.k[0], t.k[0]));
#pragma unroll
            for (int i = 1; i <= MR; i++) {
                const float2 kk = make_float2(t.k[i], t.k[i]);
                if (FMA == 2) {
                    sacc = tw_fma2(kk, make_float2(v[ctr - i], v[ctr + 1 - i]), sacc);
                    sacc = tw_fma2(kk, make_float2(v[ctr + i], v[ctr + 1 + i]), sacc);
                } else {
                    const float2 sum = tw_add2(make_float2(v[ctr - i], v[ctr + 1 - i]), make_float2(v[ctr + i], v[ctr + 1 + i]));
                    sacc = tw_fma2(tw_mul2(kk, sum), one2, sacc);
                }
            }
            r4[p] = sacc.x; r4[p + 1] = sacc.y;
        }
    }
#pragma unroll
    for (int p = 0; p < 4; p++) solve2x2(r01[p].x, r01[p].y, r23[p].x, r23[p].y, r4[p], fx[p], fy[p]);
}

template <int FMA, bool LAST>
__global__ void __launch_bounds__(WS_THREADS, 1)
gauss_strip_kernel(const __grid_constant__ CUtensorMap mapMp, const __grid_constant__ CUtensorMap mapMh, const __grid_constant__ CUtensorMap mapMp8,
                   const __grid_constant__ CUtensorMap mapMh8, const __grid_constant__ CUtensorMap mapR0, const __grid_constant__ CUtensorMap mapR1,
                   const StripArgs a, const WinTaps t)
{
    extern __shared__ __align__(1024) unsigned char ws_smem[];
    const unsigned smem = (unsigned)__cvta_generic_to_shared(ws_smem);
    const unsigned bars = smem + WS_OFF_BAR;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int w = a.d.w, h = a.d.h, pitch = a.d.pitch;
    const size_t plane = a.d.plane;

    if (tid == 0) {
        // R1 chunks are released by both teams (each arrives once per warp after its last use of the chunk, twice where the
        // other team never reads it): 2 x WS_TEAMW arrivals
        for (int i = 0; i < WS_NM; i++) { mbar_init(bars + 8 * (B_FULLM + i), 1); mbar_init(bars + 8 * (B_EMPTYM + i), WS_NVW); }
        for (int i = 0; i < WS_NP; i++) { mbar_init(bars + 8 * (B_FULLP + i), WS_NVW); mbar_init(bars + 8 * (B_EMPTYP + i), WS_TEAMW); }
        for (int i = 0; i < WS_NR0; i++) { mbar_init(bars + 8 * (B_FULLR0 + i), 1); mbar_init(bars + 8 * (B_EMPTYR0 + i), WS_TEAMW); }
        for (int i = 0; i < WS_NR1; i++) { mbar_init(bars + 8 * (B_FULLR1 + i), 1); mbar_init(bars + 8 * (B_EMPTYR1 + i), 2 * WS_TEAMW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp >= WS_PRODW) {
        // ================= TMA producer (one lane); its warpgroup hands its registers to the working warps =================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(WS_REGS_PROD));
        if (warp != WS_PRODW || lane != 0) return;
        Stream ms, r0, r1;
        ms.u = r0.u = r1.u = blockIdx.x; ms.c = r0.c = r1.c = 0; ms.n = r0.n = r1.n = 0;
        if (ms.u < a.nunits) ms.U = r0.U = r1.U = decode_unit(a, ms.u);
        if (LAST) r0.u = r1.u = a.nunits;
        unsigned idle = 0;
        while (ms.u < a.nunits || r0.u < a.nunits || r1.u < a.nunits) {
            bool any = pump_m(ms, a, smem, &mapMp, &mapMh, &mapMp8, &mapMh8);
            if (!LAST) {
                any |= pump_r1(r1, a, smem, &mapR1);
                any |= pump_r0(r0, a, smem, &mapR0);
            }
            if (any) idle = 0;
            else if (++idle > (1u << 24)) __trap();
        }
        return;
    }
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(WS_REGS_WORK));

    if (warp < WS_NVW) {
        // ================= V walkers =================
        const bool pairlane = tid < 2 * WS_VC, active = tid < WS_VLANES;
        unsigned nM = 0, nP = 0; // chunks consumed, groups blurred (global over the CTA's units)
        WS_PROF_DECL
        for (int u = blockIdx.x; u < a.nunits; u += gridDim.x) {
            const Unit U = decode_unit(a, u);
            const int xs = U.x0 - WS_XH;
            unsigned srcA, srcB, dst, dstride;
            if (pairlane) { // (column, channel pair)
                const int pair = tid >= WS_VC, j = tid - pair * WS_VC;
                const int cj = clampi(xs + j, 0, w - 1) - xs;
                srcA = pair * WS_MP1OFF + cj * 8; srcB = srcA + 4;
                dst = (pair ? WS_P23OFF : 0) + j * 8; dstride = WS_P2 * 8;
            } else { // (column pair, h2); the 16 spare lanes of warp 7 shadow the last walker and do not store
                const int jj = min(tid - 2 * WS_VC, WS_VC / 2 - 1);
                const int ca = clampi(xs + 2 * jj, 0, w - 1) - xs, cb = clampi(xs + 2 * jj + 1, 0, w - 1) - xs;
                srcA = WS_MHOFF + ca * 4; srcB = WS_MHOFF + cb * 4;
                dst = WS_P4OFF + jj * 8; dstride = WS_P4 * 4;
            }
            float2 win[WS_WIN];
#define WS_CONSUME_CHUNK(WIN_INDEX)                                                                                              \
    {                                                                                                                            \
        const unsigned s_ = nM % WS_NM;                                                                                          \
        WS_PROF(0)                                                                                                               \
        mbar_wait(bars + 8 * (B_FULLM + s_), (nM / WS_NM) & 1);                                                                  \
        WS_PROF(1)                                                                                                               \
        const unsigned base_ = smem + WS_OFF_M + s_ * WS_MCHUNK;                                                                 \
        if (pairlane) {                                                                                                          \
            _Pragma("unroll") for (int r = 0; r < WS_G; r++) win[WIN_INDEX] = lds64(base_ + r * WS_MPROW + srcA);                \
        } else {                                                                                                                 \
            _Pragma("unroll") for (int r = 0; r < WS_G; r++)                                                                     \
                win[WIN_INDEX] = make_float2(lds32(base_ + r * WS_MHROW + srcA), lds32(base_ + r * WS_MHROW + srcB));            \
        }                                                                                                                        \
        __syncwarp();                                                                                                            \
        if (lane == 0) mbar_arrive(bars + 8 * (B_EMPTYM + s_));                                                                  \
        nM++;                                                                                                                    \
        WS_PROF(2)                                                                                                               \
    }
            // the first four chunks of the unit; every group then pulls one more into the last 8 window rows and, when it is
            // done, moves the window down by 8 rows.  (The moves cost 64 register copies per step on the otherwise idle ALU
            // pipe; rotating the window at compile time instead -- five unrolled copies of the tap loops, 26 KB of code -- made
            // the SM's instruction cache thrash: 28 % of all warp samples were instruction-fetch stalls.)
#pragma unroll
            for (int c = 0; c < 4; c++) WS_CONSUME_CHUNK(8 * c + r)
#pragma unroll 1
            for (int g = 0; g < U.ng; g++) {
                const unsigned ps = nP % WS_NP;
                WS_CONSUME_CHUNK(32 + r)
                mbar_wait(bars + 8 * (B_EMPTYP + ps), ((nP / WS_NP) & 1) ^ 1);
                WS_PROF(3)
                const unsigned pd = smem + WS_OFF_P + ps * WS_PSLOT + dst;
                if (!WS_DBG(1)) v_compute<FMA>(win, pd, dstride, t, active);
                else if (active)
                    for (int o = 0; o < WS_G; o++) sts64(pd + o * dstride, win[o + WS_MR]);
                __syncwarp();
                if (lane == 0) mbar_arrive(bars + 8 * (B_FULLP + ps));
                nP++;
                WS_PROF(4)
#pragma unroll
                for (int r = 0; r < WS_WIN - WS_G; r++) win[r] = win[r + WS_G];
            }
#undef WS_CONSUME_CHUNK
        }
        WS_PROF_DUMP
        return;
    }

    // ================= H + solve + U warps: two teams of four warps, alternate groups =================
    {
        const int hw = warp - WS_NVW, team = hw >> 2, tw_ = hw & 3, tt = tid - (WS_NVW + WS_TEAMW * team) * 32;
        const int hrow = lane & 7, cbase = 16 * tw_ + 4 * (lane >> 3);    // H: lane = (row, 4-pixel quad)
        const int urow0 = 4 * (tw_ >> 1), ucol = 32 * (tw_ & 1) + lane;   // U: warp = 4 rows x 32 columns
        unsigned n = 0, nR1 = 0; // groups / R1 chunks of the CTA's unit sequence so far
        WS_PROF_DECL
        for (int u = blockIdx.x; u < a.nunits; u += gridDim.x) {
            const Unit U = decode_unit(a, u);
            const unsigned r1base = nR1;
            const bool h_active = U.x0 + 16 * tw_ < w;        // warp-uniform: ragged last strip
            const bool u_active = U.x0 + 32 * (tw_ & 1) < w;
            for (int g = 0; g < U.ng; g++, n++) {
                if ((int)(n & 1) != team) continue;
                const int yg = U.y0 + WS_G * g;
                const unsigned ps = n % WS_NP;
                float *Fb = reinterpret_cast<float *>(ws_smem + WS_OFF_F + (2 * team + ((n >> 1) & 1)) * WS_FSLOT);
                WS_PROF(0)
                mbar_wait(bars + 8 * (B_FULLP + ps), (n / WS_NP) & 1);
                WS_PROF(1)
                if (h_active) {
                    float fx[4] = {0.25f, 0.25f, 0.25f, 0.25f}, fy[4] = {-0.25f, -0.25f, -0.25f, -0.25f};
                    if (!WS_DBG(2)) {
                        const unsigned char *P = ws_smem + WS_OFF_P + ps * WS_PSLOT;
                        const float2 *p01 = reinterpret_cast<const float2 *>(P) + hrow * WS_P2 + cbase;
                        const float2 *p23 = reinterpret_cast<const float2 *>(P + WS_P23OFF) + hrow * WS_P2 + cbase;
                        const float *p4 = reinterpret_cast<const float *>(P + WS_P4OFF) + hrow * WS_P4 + cbase;
                        h_quad<FMA>(p01, p23, p4, t, fx, fy);
                    }
#pragma unroll
                    for (int p = 0; p < 4; p++) {
                        Fb[hrow * WS_FP + cbase + p] = fx[p];
                        Fb[(WS_G + hrow) * WS_FP + cbase + p] = fy[p];
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(bars + 8 * (B_EMPTYP + ps));
                WS_PROF(2)
                team_barrier(team);
                WS_PROF(3) // the team's flow tile of this group is complete (the tile is double-buffered: a warp may
                                    // still read the previous one)
                if (LAST) {
                    float *f = a.flow + (size_t)U.b * 2 * plane;
#pragma unroll
                    for (int i = tt; i < WS_G * WS_SW; i += WS_TEAM_THREADS) {
                        const int row = i / WS_SW, col = i - row * WS_SW;
                        const int x = U.x0 + col, y = yg + row;
                        if (x < w && y < h) {
                            const size_t o = (size_t)y * pitch + x;
                            f[o] = Fb[row * WS_FP + col];
                            f[o + plane] = Fb[(WS_G + row) * WS_FP + col];
                        }
                    }
                    if (a.span > 0) { // span-grid threshold test on the tile (reference src/consumer.cpp:60-77), count by warp shuffles
                        const int sx0 = (U.x0 + a.span - 1) / a.span, sy0 = (yg + a.span - 1) / a.span;
                        const int nsx = max(0, (min(U.x0 + WS_SW, w) - 1) / a.span - sx0 + 1), nsy = max(0, (min(yg + WS_G, h) - 1) / a.span - sy0 + 1);
                        int hit = 0;
                        for (int i = tt; i < nsx * nsy; i += WS_TEAM_THREADS) {
                            const int j = i / nsx, col = (sx0 + i - j * nsx) * a.span - U.x0, row = (sy0 + j) * a.span - yg;
                            const float dx = Fb[row * WS_FP + col], dy = Fb[(WS_G + row) * WS_FP + col];
                            const float len = (dx * dx) + (dy * dy);
                            hit += ((double)len > a.thr2) ? 1 : 0;
                        }
                        if (nsx * nsy > 0) {
#pragma unroll
                            for (int off = 16; off > 0; off >>= 1) hit += __shfl_xor_sync(0xffffffffu, hit, off);
                            if (lane == 0 && hit > 0) atomicAdd(a.counts + U.b, hit);
                        }
                    }
                    continue;
                }
                // ---- U: next update matrices (A.4) from the staged R0 / R1 ----
                const unsigned rs = n % WS_NR0;
                mbar_wait(bars + 8 * (B_FULLR0 + rs), (n / WS_NR0) & 1);
#pragma unroll
                for (int k = 0; k < 3; k++) { // the chunks with the rows yg - 8 .. yg + 15
                    const unsigned nc = r1base + g + k;
                    mbar_wait(bars + 8 * (B_FULLR1 + nc % WS_NR1), (nc / WS_NR1) & 1);
                }
                WS_PROF(4)
                if (u_active && !WS_DBG(8)) {
                    const float *R0s = reinterpret_cast<const float *>(ws_smem + WS_OFF_R0 + rs * WS_R0SLOT) + urow0 * 5 * WS_SW + ucol; // [8][5][64]
                    const float *R1s = reinterpret_cast<const float *>(ws_smem + WS_OFF_R1);                                             // [48][5][72]
                    const float *Fu = Fb + urow0 * WS_FP + ucol;
                    float *Mo = a.Mout + (size_t)U.b * 5 * plane;
                    const int x = U.x0 + ucol, y0u = yg + urow0;
                    const int xw = U.x0 - WS_R1X;
                    // ring row of frame row yy (yg - 8 <= yy <= yg + 15) = (yy - (yg - 8) + rr0) mod 48, rr0 = first ring row of chunk g
                    const int rr0 = WS_G * (int)((r1base + g) % WS_NR1) - (yg - WS_G);
                    // positions of the thread's four vertically adjacent pixels
                    float dxs[4], dys[4], fxr[4], fyr[4];
                    int x1s[4], y1s[4];
                    bool fast = (unsigned)(x - 5) < (unsigned)(w - 10) && y0u >= 5 && y0u + 3 < h - 5;
#pragma unroll
                    for (int q4 = 0; q4 < 4; q4++) {
                        dxs[q4] = Fu[q4 * WS_FP]; dys[q4] = Fu[(WS_G + q4) * WS_FP];
                        const float pxf = (float)x + dxs[q4], pyf = (float)(y0u + q4) + dys[q4];
                        x1s[q4] = __float2int_rd(pxf); y1s[q4] = __float2int_rd(pyf);
                        fxr[q4] = pxf - (float)x1s[q4]; fyr[q4] = pyf - (float)y1s[q4];
                        // inside the frame (A.4) and inside the staged R1 window
                        fast = fast && (unsigned)x1s[q4] < (unsigned)(w - 1) && (unsigned)y1s[q4] < (unsigned)(h - 1) &&
                               (unsigned)(x1s[q4] - xw) <= (unsigned)(WS_R1C - 2) && (unsigned)(y1s[q4] - yg + WS_G) <= (unsigned)(3 * WS_G - 2);
                    }
                    if (__all_sync(0xffffffffu, fast)) {
#pragma unroll
                        for (int pr = 0; pr < 4; pr += 2) { // pixels (pr, pr + 1) packed
                            float2 q[5], pt[5][2], pb[5][2], m[5];
                            int ria = y1s[pr] + rr0, rib = y1s[pr + 1] + rr0;
                            ria -= ria >= WS_R1RING ? WS_R1RING : 0; rib -= rib >= WS_R1RING ? WS_R1RING : 0;
                            const int rja = ria + 1 == WS_R1RING ? 0 : ria + 1, rjb = rib + 1 == WS_R1RING ? 0 : rib + 1;
                            const float *a0 = R1s + ria * WS_R1ROW + (x1s[pr] - xw), *a1 = R1s + rja * WS_R1ROW + (x1s[pr] - xw);
                            const float *b0 = R1s + rib * WS_R1ROW + (x1s[pr + 1] - xw), *b1 = R1s + rjb * WS_R1ROW + (x1s[pr + 1] - xw);
#pragma unroll
                            for (int c = 0; c < 5; c++) {
                                q[c] = make_float2(R0s[(pr * 5 + c) * WS_SW], R0s[((pr + 1) * 5 + c) * WS_SW]);
                                pt[c][0] = make_float2(a0[c * WS_R1C], b0[c * WS_R1C]); pt[c][1] = make_float2(a0[c * WS_R1C + 1], b0[c * WS_R1C + 1]);
                                pb[c][0] = make_float2(a1[c * WS_R1C], b1[c * WS_R1C]); pb[c][1] = make_float2(a1[c * WS_R1C + 1], b1[c * WS_R1C + 1]);
                            }
                            upd_core2(q, pt, pb, make_float2(fxr[pr], fxr[pr + 1]), make_float2(fyr[pr], fyr[pr + 1]), make_float2(dxs[pr], dxs[pr + 1]),
                                      make_float2(dys[pr], dys[pr + 1]), t.one, m);
                            const float ma[5] = {m[0].x, m[1].x, m[2].x, m[3].x, m[4].x}, mb[5] = {m[0].y, m[1].y, m[2].y, m[3].y, m[4].y};
                            store_M(Mo, pitch, y0u + pr, x, ma);
                            store_M(Mo, pitch, y0u + pr + 1, x, mb);
                        }
                    } else { // frame borders, ragged tiles, large motion: one pixel at a time
                        const float *R1g = a.R + ((size_t)U.b * 10 + 5) * plane;
#pragma unroll 1
                        for (int q4 = 0; q4 < 4; q4++) {
                            const int y = y0u + q4;
                            if (x >= w || y >= h) continue;
                            const float dx = Fu[q4 * WS_FP], dy = Fu[(WS_G + q4) * WS_FP];
                            const float pxf = (float)x + dx, pyf = (float)y + dy;
                            const int x1 = __float2int_rd(pxf), y1 = __float2int_rd(pyf);
                            const float fx1 = pxf - (float)x1, fy1 = pyf - (float)y1;
                            const bool inside = (unsigned)x1 < (unsigned)(w - 1) && (unsigned)y1 < (unsigned)(h - 1);
                            float q[5], pt[5][2], pb[5][2];
#pragma unroll
                            for (int c = 0; c < 5; c++) q[c] = R0s[(q4 * 5 + c) * WS_SW];
                            if (inside) {
                                if ((unsigned)(x1 - xw) <= (unsigned)(WS_R1C - 2) && (unsigned)(y1 - yg + WS_G) <= (unsigned)(3 * WS_G - 2)) {
                                    int ri = y1 + rr0;
                                    ri -= ri >= WS_R1RING ? WS_R1RING : 0;
                                    const int rj = ri + 1 == WS_R1RING ? 0 : ri + 1;
                                    const float *a0 = R1s + ri * WS_R1ROW + (x1 - xw), *a1 = R1s + rj * WS_R1ROW + (x1 - xw);
#pragma unroll
                                    for (int c = 0; c < 5; c++) {
                                        pt[c][0] = a0[c * WS_R1C]; pt[c][1] = a0[c * WS_R1C + 1];
                                        pb[c][0] = a1[c * WS_R1C]; pb[c][1] = a1[c * WS_R1C + 1];
                                    }
                                } else { // the same values from global memory
                                    const float *p = R1g + (size_t)y1 * 5 * pitch + x1;
#pragma unroll
                                    for (int c = 0; c < 5; c++) {
                                        pt[c][0] = __ldg(p + c * pitch); pt[c][1] = __ldg(p + c * pitch + 1);
                                        pb[c][0] = __ldg(p + (5 + c) * pitch); pb[c][1] = __ldg(p + (5 + c) * pitch + 1);
                                    }
                                }
                            }
                            float m[5];
                            upd_core<true>(q, pt, pb, inside, fx1, fy1, w, h, x, y, dx, dy, m);
                            store_M(Mo, pitch, y, x, m);
                        }
                    }
                }
                __syncwarp();
                WS_PROF(5)
                if (lane == 0) {
                    // release.  Chunk c = g + k is read by the groups c - 2 .. c of the unit, i.e. by both teams; each team arrives
                    // (once per warp) after ITS last use of the chunk, twice where the other team has no group that reads it.
                    mbar_arrive(bars + 8 * (B_EMPTYR0 + rs));
                    const unsigned e0 = bars + 8 * (B_EMPTYR1 + (r1base + g) % WS_NR1), e1 = bars + 8 * (B_EMPTYR1 + (r1base + g + 1) % WS_NR1);
                    mbar_arrive(e0);
                    if (g == 0) mbar_arrive(e0);
                    mbar_arrive(e1);
                    if (g == 0 && g + 1 >= U.ng) mbar_arrive(e1);
                    if (g + 2 >= U.ng) {
                        const unsigned e2 = bars + 8 * (B_EMPTYR1 + (r1base + g + 2) % WS_NR1);
                        mbar_arrive(e2);
                        if (g + 1 >= U.ng) mbar_arrive(e2);
                    }
                }
                WS_PROF(6)
            }
            nR1 = r1base + U.ng + 2;
        }
        WS_PROF_DUMP
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled()
{
    static EncodeTiledFn fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

bool encode3(CUtensorMap *m, const float *base, cuuint64_t d0, cuuint64_t d1, cuuint64_t d2, cuuint64_t s1_bytes, cuuint64_t s2_bytes, cuuint32_t b0,
             cuuint32_t b1)
{
    EncodeTiledFn fn = encode_tiled();
    if (!fn) return false;
    const cuuint64_t dims[3] = {d0, d1, d2}, strides[2] = {s1_bytes, s2_bytes};
    const cuuint32_t box[3] = {b0, b1, 1}, estr[3] = {1, 1, 1};
    return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

int sm_count()
{
    static int n[64] = {};
    int d = 0;
    cudaGetDevice(&d);
    if (d < 0 || d >= 64) d = 0;
    if (!n[d]) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, d) != cudaSuccess || v < 1) v = 148;
        n[d] = v;
    }
    return n[d];
}

template <int FMA, bool LAST>
cudaError_t launch_strip(cudaStream_t s, const StripMaps &m, const StripArgs &sa, const WinTaps &t, int grid)
{
    static std::atomic<bool> configured_dev[64]; // consumer threads sharing a device may get here together; the attribute call is idempotent
    int d = 0;
    cudaGetDevice(&d);
    if (d < 0 || d >= 64) d = 0;
    if (!configured_dev[d]) {
        cudaError_t e = cudaFuncSetAttribute(gauss_strip_kernel<FMA, LAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, WS_SMEM);
        if (e != cudaSuccess) return e;
        configured_dev[d] = true;
    }
    const CUtensorMap *maps = reinterpret_cast<const CUtensorMap *>(m.opaque);
    gauss_strip_kernel<FMA, LAST><<<grid, WS_THREADS, WS_SMEM, s>>>(maps[0], maps[1], maps[2], maps[3], maps[4], maps[5], sa, t);
    return cudaGetLastError();
}

} // namespace

static_assert(sizeof(CUtensorMap) * 6 <= sizeof(StripMaps::opaque), "StripMaps holds six tensor maps");
static_assert(sizeof(CUtensorMap) <= sizeof(TileMap::opaque), "TileMap holds one tensor map");

// Tensor maps of one (M buffer, R buffer) pair at one scale: M as [B][h][5*pitch] floats (boxes 192 x {1, 8} and 96 x {1, 8}: rows
// of a channel-pair plane / of the h2 plane), R as [2B][5h][pitch] floats (boxes 64 x 40 and 72 x 40: 8 rows x 5 channels).
bool make_strip_maps(const float *M, const float *R, const LevelDims &d, int batch, StripMaps *out)
{
    CUtensorMap *maps = reinterpret_cast<CUtensorMap *>(out->opaque);
    const cuuint64_t pitch = (cuuint64_t)d.pitch, h = (cuuint64_t)d.h, plane = (cuuint64_t)d.plane;
    out->valid = 0;
    if (d.pitch % 4 != 0 || 5 * pitch < 2 * WS_VC) return false;
    if (!encode3(&maps[0], M, 5 * pitch, h, (cuuint64_t)batch, 5 * pitch * 4, 5 * plane * 4, 2 * WS_VC, 1)) return false;
    if (!encode3(&maps[1], M, 5 * pitch, h, (cuuint64_t)batch, 5 * pitch * 4, 5 * plane * 4, WS_VC, 1)) return false;
    if (!encode3(&maps[2], M, 5 * pitch, h, (cuuint64_t)batch, 5 * pitch * 4, 5 * plane * 4, 2 * WS_VC, WS_G)) return false;
    if (!encode3(&maps[3], M, 5 * pitch, h, (cuuint64_t)batch, 5 * pitch * 4, 5 * plane * 4, WS_VC, WS_G)) return false;
    if (!encode3(&maps[4], R, pitch, 5 * h, (cuuint64_t)batch * 2, pitch * 4, 5 * plane * 4, WS_SW, 5 * WS_G)) return false;
    if (!encode3(&maps[5], R, pitch, 5 * h, (cuuint64_t)batch * 2, pitch * 4, 5 * plane * 4, WS_R1C, 5 * WS_G)) return false;
    out->valid = 1;
    return true;
}

// Tensor map of the level images I ([nimg][h][pitch] floats) for the poly-exp's staged input tile: box 112 columns x (32 + 2 polyN) rows.
bool make_polyexp_map(const float *I, const LevelDims &d, int nimg, int polyN, TileMap *out)
{
    out->valid = 0;
    if (d.pitch % 4 != 0 || d.pitch < 112 || polyN < 1 || 32 + 2 * polyN > 256) return false;
    if (!encode3(reinterpret_cast<CUtensorMap *>(out->opaque), I, (cuuint64_t)d.pitch, (cuuint64_t)d.h, (cuuint64_t)nimg, (cuuint64_t)d.pitch * 4,
                 (cuuint64_t)d.plane * 4, 112, (cuuint32_t)(32 + 2 * polyN)))
        return false;
    out->valid = 1;
    return true;
}

bool gauss_strip_ok(const IterArgs &a, const WinTaps &t)
{
    return t.m == WS_MR && a.d.w >= 1 && a.d.h >= 1;
}

cudaError_t launch_gauss_strip(cudaStream_t s, const IterArgs &a, const WinTaps &t, const StripMaps &m)
{
    if (!m.valid || !gauss_strip_ok(a, t)) return cudaErrorInvalidValue;
    StripArgs sa{};
    sa.R = a.R; sa.Mout = a.Mout; sa.flow = a.flow; sa.d = a.d;
    sa.span = a.last ? a.span : 0; sa.thr2 = a.thr2; sa.counts = a.counts;
#ifdef TW_STRIP_DEBUG
    if (const char *e = getenv("TW_STRIP_DBG")) sa.dbg = atoi(e);
    static unsigned *prof_dev = nullptr;
    const bool prof = getenv("TW_STRIP_PROF") && !a.last && a.d.w >= 1920;
    if (prof && !prof_dev) cudaMalloc(&prof_dev, 148 * 16 * 8 * 4);
    sa.prof = prof ? prof_dev : nullptr;
#endif
    const int sms = sm_count();
    sa.nsx = (a.d.w + WS_SW - 1) / WS_SW;
    // vertical segments per strip: the split that minimises (rounds of units over the SMs) x (rows per unit + the cost of a unit's
    // window refill, about one group); a segment is at least 64 rows
    const int per = a.batch * sa.nsx;
    int best_nsy = 1;
    long best_cost = -1;
    for (int n = 1; n <= std::max(1, std::min(a.d.h / 64, 32)); n++) {
        const int segh = ((a.d.h + n - 1) / n + WS_G - 1) & ~(WS_G - 1);
        const int nsy = (a.d.h + segh - 1) / segh;
        const long rounds = ((long)per * nsy + sms - 1) / sms;
        const long cost = rounds * (segh + WS_G);
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best_nsy = n; }
    }
    sa.segh = ((a.d.h + best_nsy - 1) / best_nsy + WS_G - 1) & ~(WS_G - 1);
    sa.nsy = (a.d.h + sa.segh - 1) / sa.segh;
    sa.nunits = per * sa.nsy;
    const int grid = std::min(sa.nunits, sms);
    if (a.last) return a.fma == 2 ? launch_strip<2, true>(s, m, sa, t, grid) : launch_strip<0, true>(s, m, sa, t, grid);
#ifdef TW_STRIP_DEBUG
    if (sa.prof) { // per-role phase clocks of one level-0 launch, averaged over the CTAs
        cudaError_t e = a.fma == 2 ? launch_strip<2, false>(s, m, sa, t, grid) : launch_strip<0, false>(s, m, sa, t, grid);
        static int printed = 0;
        if (e == cudaSuccess && printed++ == 6) {
            static unsigned hostp[148 * 16 * 8];
            cudaStreamSynchronize(s);
            cudaMemcpy(hostp, sa.prof, sizeof(hostp), cudaMemcpyDeviceToHost);
            for (int wp = 0; wp < 16; wp++) {
                double acc[8] = {};
                for (int b = 0; b < grid; b++)
                    for (int i = 0; i < 8; i++) acc[i] += hostp[(b * 16 + wp) * 8 + i];
                fprintf(stderr, "strip prof warp %2d:", wp);
                for (int i = 0; i < 8; i++) fprintf(stderr, " %9.0f", acc[i] / grid);
                fprintf(stderr, "\n");
            }
        }
        return e;
    }
#endif
    return a.fma == 2 ? launch_strip<2, false>(s, m, sa, t, grid) : launch_strip<0, false>(s, m, sa, t, grid);
}

} // namespace tw
