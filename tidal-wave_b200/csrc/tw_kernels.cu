// tw_kernels.cu -- hand-written sm_100a kernels of the Farneback hot path.
//
// Compiled with -fmad=false: the oracle's results depend on the rounding of every add / mul
// (SURVEY.md App. A, "hard part 1"), so nothing may be contracted implicitly.  Fused multiply-adds
// appear only where the oracle itself uses them (pre-blur, App. A.2a) and are written as fmaf().
//
// The algorithm restated here is OpenCV's calcOpticalFlowFarneback -- the single library call at
// /root/reference/src/opticalflow.cpp:83-85 -- and the sampling loop of /root/reference/src/consumer.cpp:60-77.
#include "tw_kernels.cuh"
#include "tw_device.cuh"

#include <atomic>

namespace tw {

// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute: remember what was configured per device, not
// per process (an in-process multi-GPU pool launches the same kernel on every device).
constexpr int kMaxDevices = 64;
static int current_device()
{
    int d = 0;
    cudaGetDevice(&d);
    return (d >= 0 && d < kMaxDevices) ? d : 0;
}

// base + stride * row as ONE instruction (IMAD.WIDE.U32).  nvcc otherwise strength-reduces the unrolled row
// addresses into chains of 64-bit adds + LEA pairs: 4 integer instructions per load in kernels whose inner loops
// are bound by instruction issue.
__device__ __forceinline__ const char *row_ptr(const char *base, unsigned stride_bytes, unsigned row)
{
    unsigned long long out;
    asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(out) : "r"(stride_bytes), "r"(row), "l"(reinterpret_cast<unsigned long long>(base)));
    return reinterpret_cast<const char *>(out);
}

__device__ __forceinline__ int reflect101(int p, int len)
{
    if (len == 1) return 0;
    while (p < 0 || p >= len) p = p < 0 ? -p : 2 * (len - 1) - p;
    return p;
}

// single-bounce REFLECT_101, valid for -len < p < 2*len - 1
__device__ __forceinline__ int reflect1(int p, int len)
{
    p = p < 0 ? -p : p;
    return p >= len ? 2 * (len - 1) - p : p;
}

// ------------------------------------------------------------------------------------------------
// K1  level image: u8 -> float, GaussianBlur(ksize) REFLECT_101 (rows first, then columns), bilinear
//     resize to (w, h).  One block = one output tile; the u8 source tile (with halo) is staged in shared
//     memory, the row pass is evaluated only at the source columns the resize reads, the column pass
//     only at the source rows it reads.   SURVEY App. A.2 / A.2a / A.2b.
// ------------------------------------------------------------------------------------------------
// exact u8 -> float without the XU pipe: 0x4B000000 | b is 8388608.0f + b.
__device__ __forceinline__ float u8_to_float(unsigned b) { return __uint_as_float(0x4B000000u | b) - 8388608.0f; }

template <bool IDENT>
__global__ void __launch_bounds__(256) level_image_kernel(LevelImageArgs a)
{
    extern __shared__ __align__(16) float li_smem[];
    const int K = a.ksize, c = K / 2;
    const int d0 = blockIdx.x * a.tile_w, e0 = blockIdx.y * a.tile_h;
    const int d1 = min(d0 + a.tile_w, a.d.w) - 1, e1 = min(e0 + a.tile_h, a.d.h) - 1;
    const int tw_ = d1 - d0 + 1, th_ = e1 - e0 + 1;
    const int W = a.W, H = a.H;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // source tile (unclamped extents; border pixels are staged through REFLECT_101 so the tap loops index directly).
    // The tile origin is aligned down to 4 source columns so that interior words are staged with one 4-byte load,
    // two instructions per pixel for the exact u8 -> float conversion (PRMT + FADD) and one 16-byte shared store.
    const int xs_lo = (a.xi[d0] - c) & ~3, ys_lo = a.yi[e0] - c;
    const int SW = min(a.xi[d1] + 1, W - 1) + c - xs_lo + 1, SH = min(a.yi[e1] + 1, H - 1) + c - ys_lo + 1;
    const int SWp = a.smem_w; // multiple of 4
    const int NC = IDENT ? a.tile_w : a.tile_w * 2;
    float *tile = li_smem;                        // [smem_h][SWp]
    float *rp = tile + (size_t)a.smem_h * SWp;    // [smem_h][NC]
    float *ktab = rp + (size_t)a.smem_h * NC;     // [K]

    const uint8_t *src = a.src + (size_t)blockIdx.z * H * a.spitch;
    for (int i = threadIdx.x; i < K; i += 256) ktab[i] = a.taps[i];
    if (a.small) { // image smaller than the blur radius: REFLECT_101 may bounce more than once
        for (int r = warp; r < SH; r += 8) {
            const uint8_t *srow = src + (size_t)reflect101(ys_lo + r, H) * a.spitch;
            for (int q = lane; q < SW; q += 32) tile[r * SWp + q] = u8_to_float(srow[reflect101(xs_lo + q, W)]);
        }
    } else {
        const int nwords = (SW + 3) >> 2;
        for (int r = warp; r < SH; r += 16) {
            const int r2 = min(r + 8, SH - 1);
            const uint8_t *srow0 = src + (size_t)reflect1(ys_lo + r, H) * a.spitch;
            const uint8_t *srow1 = src + (size_t)reflect1(ys_lo + r2, H) * a.spitch;
#pragma unroll 2
            for (int q4 = lane; q4 < nwords; q4 += 32) {
                const int gx = xs_lo + 4 * q4;
                float4 f0, f1;
                if (gx >= 0 && gx + 3 < W) {
                    const unsigned w0 = __ldg(reinterpret_cast<const unsigned *>(srow0 + gx));
                    const unsigned w1 = __ldg(reinterpret_cast<const unsigned *>(srow1 + gx));
                    f0.x = __uint_as_float(__byte_perm(w0, 0x4B000000u, 0x7650)) - 8388608.0f;
                    f0.y = __uint_as_float(__byte_perm(w0, 0x4B000000u, 0x7651)) - 8388608.0f;
                    f0.z = __uint_as_float(__byte_perm(w0, 0x4B000000u, 0x7652)) - 8388608.0f;
                    f0.w = __uint_as_float(__byte_perm(w0, 0x4B000000u, 0x7653)) - 8388608.0f;
                    f1.x = __uint_as_float(__byte_perm(w1, 0x4B000000u, 0x7650)) - 8388608.0f;
                    f1.y = __uint_as_float(__byte_perm(w1, 0x4B000000u, 0x7651)) - 8388608.0f;
                    f1.z = __uint_as_float(__byte_perm(w1, 0x4B000000u, 0x7652)) - 8388608.0f;
                    f1.w = __uint_as_float(__byte_perm(w1, 0x4B000000u, 0x7653)) - 8388608.0f;
                } else {
                    const int g0 = reflect1(gx, W), g1 = reflect1(gx + 1, W), g2 = reflect1(gx + 2, W), g3 = reflect1(gx + 3, W);
                    f0 = make_float4(u8_to_float(__ldg(srow0 + g0)), u8_to_float(__ldg(srow0 + g1)), u8_to_float(__ldg(srow0 + g2)),
                                     u8_to_float(__ldg(srow0 + g3)));
                    f1 = make_float4(u8_to_float(__ldg(srow1 + g0)), u8_to_float(__ldg(srow1 + g1)), u8_to_float(__ldg(srow1 + g2)),
                                     u8_to_float(__ldg(srow1 + g3)));
                }
                *reinterpret_cast<float4 *>(tile + r * SWp + 4 * q4) = f0;
                *reinterpret_cast<float4 *>(tile + r2 * SWp + 4 * q4) = f1;
            }
        }
    }
    __syncthreads();

    // row pass, only at the source columns the resize reads; (row, slot) items are spread over all 256 threads (tiles
    // behind a long pre-blur kernel are only a few columns wide)
    const int ncol = IDENT ? tw_ : tw_ * 2;
    for (int i = threadIdx.x; i < SH * ncol; i += 256) {
        const int r = i / ncol, slot = i - r * ncol;
        int xl; // local column of tap 0
        if (IDENT) xl = d0 + slot - c - xs_lo;
        else xl = min(a.xi[d0 + (slot >> 1)] + (slot & 1), W - 1) - c - xs_lo;
        const float *p = tile + r * SWp + xl;
        float o;
        if (K == 3) {
            o = fmaf(p[1], ktab[1], (p[0] + p[2]) * ktab[0]);
        } else {
            o = p[0] * ktab[0];
#pragma unroll 4
            for (int j = 1; j < K; j++) o = fmaf(p[j], ktab[j], o);
        }
        rp[r * NC + slot] = o;
    }
    __syncthreads();

    // column pass at the source rows the resize reads, then the bilinear blend (A.2b)
    float *dst = a.dst + (size_t)blockIdx.z * a.d.plane;
    for (int i = threadIdx.x; i < th_ * tw_; i += 256) {
        const int ty = i / tw_, tx = i - ty * tw_;
        const int e = e0 + ty;
        const int y0 = a.yi[e], y1 = min(y0 + 1, H - 1);
        const float fy = IDENT ? 0.f : a.yf[e];
        {
            const int d = d0 + tx;
            float res[2][2];
#pragma unroll
            for (int yy = 0; yy < (IDENT ? 1 : 2); yy++) {
                const float *col = rp + ((yy ? y1 : y0) - ys_lo) * NC + (IDENT ? tx : tx * 2);
#pragma unroll
                for (int xx = 0; xx < (IDENT ? 1 : 2); xx++) {
                    const float *q = col + xx;
                    float o;
                    if (K == 3) {
                        o = fmaf(q[-NC] + q[NC], ktab[0], q[0] * ktab[1]);
                    } else {
                        o = q[0] * ktab[c];
                        for (int j = 1; j <= c; j++) o = fmaf(q[-j * NC] + q[j * NC], ktab[c + j], o);
                    }
                    res[yy][xx] = o;
                }
            }
            float out;
            if (IDENT) {
                out = res[0][0];
            } else {
                const float fx = a.xf[d], gx = 1.f - fx, gy = 1.f - fy;
                const float r0 = res[0][0] * gx + res[0][1] * fx;
                const float r1 = res[1][0] * gx + res[1][1] * fx;
                out = r0 * gy + r1 * fy;
            }
            dst[(size_t)e * a.d.pitch + d] = out;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K1, long pre-blur kernels (deep pyramids: the 1/32-scale level of config 3 blurs with 79 taps before a non-integer
// down-scale).  A tile of the generic kernel would stage (32 * tile + 79)^2 source pixels to produce a handful of outputs; here
// the separable blur runs as two small kernels through an intermediate in global memory (L2-resident):
//   level_rows_kernel: one CTA per (source row, image): the row is staged once as floats (REFLECT_101 halo), the row pass is
//                      evaluated at the 2 source columns each output column reads -> T[image][row][2w]
//   level_cols_kernel: one thread per output pixel: column pass at the 2 rows x 2 columns it reads (rows through REFLECT_101),
//                      then the bilinear blend.
// Same operations in the same order as level_image_kernel (App. A.2a / A.2b): bit-identical.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) level_rows_kernel(LevelImageArgs a, float *__restrict__ T, int tpitch)
{
    extern __shared__ float lr_smem[]; // [W + 2c] padded by one word per 32 (the slots of a warp are 32 source columns apart) | K taps
    const int K = a.ksize, c = K / 2, W = a.W;
    const int n = W + 2 * c;
    float *row = lr_smem, *ktab = lr_smem + n + (n >> 5) + 1;
    const int y = blockIdx.x;
    const uint8_t *srow = a.src + ((size_t)blockIdx.y * a.H + y) * a.spitch;
    for (int i = threadIdx.x; i < K; i += 256) ktab[i] = a.taps[i];
    // interior columns as 4-byte words (all loads of a thread in flight together), the two REFLECT_101 halos and a ragged tail as bytes
    const int W4 = W & ~3;
#pragma unroll 4
    for (int q4 = threadIdx.x; q4 < W4 / 4; q4 += 256) {
        const unsigned wd = __ldg(reinterpret_cast<const unsigned *>(srow) + q4);
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int q = c + 4 * q4 + i;
            row[q + (q >> 5)] = __uint_as_float(__byte_perm(wd, 0x4B000000u, 0x7650 + i)) - 8388608.0f;
        }
    }
    for (int i = threadIdx.x; i < 2 * c + (W - W4); i += 256) {
        const int q = i < c ? i : i < 2 * c ? W + i : W4 + c + (i - 2 * c); // left halo | right halo | tail columns
        row[q + (q >> 5)] = u8_to_float(__ldg(srow + reflect1(q - c, W)));
    }
    __syncthreads();
    float *out = T + ((size_t)blockIdx.y * a.H + y) * tpitch;
    for (int slot = threadIdx.x; slot < 2 * a.d.w; slot += 256) {
        const int xs = min(a.xi[slot >> 1] + (slot & 1), W - 1); // tap j reads source column xs - c + j = staged entry xs + j
        float o = row[xs + (xs >> 5)] * ktab[0];
#pragma unroll 4
        for (int j = 1; j < K; j++) {
            const int q = xs + j;
            o = fmaf(row[q + (q >> 5)], ktab[j], o);
        }
        out[slot] = o;
    }
}

__global__ void __launch_bounds__(256) level_cols_kernel(LevelImageArgs a, const float *__restrict__ T, int tpitch)
{
    const int d = blockIdx.x * 32 + (threadIdx.x & 31), e = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (d >= a.d.w || e >= a.d.h) return;
    const int K = a.ksize, c = K / 2, H = a.H;
    const float *Tb = T + (size_t)blockIdx.z * H * tpitch + 2 * d;
    const int y0 = a.yi[e], y1 = min(y0 + 1, H - 1);
    float res[2][2];
#pragma unroll
    for (int yy = 0; yy < 2; yy++) {
        const int yc = yy ? y1 : y0;
        float o0 = 0.f, o1 = 0.f;
        {
            const float2 q = __ldg(reinterpret_cast<const float2 *>(Tb + (size_t)yc * tpitch));
            o0 = q.x * __ldg(a.taps + c); o1 = q.y * __ldg(a.taps + c);
        }
        for (int j = 1; j <= c; j++) {
            const float2 up = __ldg(reinterpret_cast<const float2 *>(Tb + (size_t)reflect1(yc - j, H) * tpitch));
            const float2 dn = __ldg(reinterpret_cast<const float2 *>(Tb + (size_t)reflect1(yc + j, H) * tpitch));
            const float kk = __ldg(a.taps + c + j);
            o0 = fmaf(up.x + dn.x, kk, o0);
            o1 = fmaf(up.y + dn.y, kk, o1);
        }
        res[yy][0] = o0; res[yy][1] = o1;
    }
    const float fx = a.xf[d], gx = 1.f - fx, fy = a.yf[e], gy = 1.f - fy;
    const float r0 = res[0][0] * gx + res[0][1] * fx;
    const float r1 = res[1][0] * gx + res[1][1] * fx;
    a.dst[(size_t)blockIdx.z * a.d.plane + (size_t)e * a.d.pitch + d] = r0 * gy + r1 * fy;
}

bool level_image_big_ok(const LevelImageArgs &a) { return !a.identity && !a.small && a.ksize >= 31 && a.ksize / 2 < a.W && a.ksize / 2 < a.H; }
size_t level_image_big_floats(int H, int w, int nimg) { return (size_t)nimg * H * ((2 * w + 31) & ~31); }

cudaError_t launch_level_image_big(cudaStream_t s, const LevelImageArgs &a, float *T)
{
    if (!level_image_big_ok(a) || !T) return cudaErrorNotSupported;
    const int tpitch = (2 * a.d.w + 31) & ~31;
    const int n = a.W + 2 * (a.ksize / 2);
    const size_t smem = sizeof(float) * (size_t)(n + (n >> 5) + 1 + a.ksize);
    if (smem > 48 * 1024) return cudaErrorNotSupported;
    level_rows_kernel<<<dim3(a.H, a.nimg), 256, smem, s>>>(a, T, tpitch);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    level_cols_kernel<<<dim3((a.d.w + 31) / 32, (a.d.h + 7) / 8, a.nimg), 256, 0, s>>>(a, T, tpitch);
    return cudaGetLastError();
}

size_t level_image_smem_bytes(int smem_w, int smem_h, int tile_w, int ksize, int identity)
{
    return sizeof(float) * ((size_t)smem_h * smem_w + (size_t)smem_h * (identity ? tile_w : tile_w * 2) + ksize);
}

cudaError_t launch_level_image(cudaStream_t s, const LevelImageArgs &a)
{
    size_t smem = level_image_smem_bytes(a.smem_w, a.smem_h, a.tile_w, a.ksize, a.identity);
    static std::atomic<size_t> configured_dev[kMaxDevices][2];
    std::atomic<size_t> *configured = configured_dev[current_device()];
    if (smem > 48 * 1024 && smem > configured[a.identity ? 1 : 0]) {
        cudaError_t e = a.identity ? cudaFuncSetAttribute(level_image_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                                   : cudaFuncSetAttribute(level_image_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        configured[a.identity ? 1 : 0] = smem;
    }
    dim3 grid((a.d.w + a.tile_w - 1) / a.tile_w, (a.d.h + a.tile_h - 1) / a.tile_h, a.nimg);
    if (a.identity) level_image_kernel<true><<<grid, 256, smem, s>>>(a);
    else level_image_kernel<false><<<grid, 256, smem, s>>>(a);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// K1 fast paths.  The generic kernel above handles any pyrScale; these two cover what the reference's default
// pyrScale = 0.5 produces whenever the frame size is divisible by the scale: (a) the full-resolution level
// (3-tap blur, no resize) and (b) exact integer down-scales S = 2, 4, 8, 16 where the bilinear resize reads
// source columns/rows S*d + S/2 - 1 and S*d + S/2 with weight 0.5 each (checked on the host against the A.2b
// tables).  Compile-time tile geometry: taps from the constant bank, no index arithmetic in the tap loops,
// lane = source row with a 4*odd shared pitch so that the row pass reads its K+1 inputs as conflict-free LDS.128.
// ------------------------------------------------------------------------------------------------
struct LevelFastArgs {
    const uint8_t *src; // [nimg][H][spitch]
    int W, H, spitch;
    float *dst;         // [nimg][h][pitch]
    LevelDims d;
    float k[40];        // ksize taps
};

template <int SH, int SWP>
__device__ __forceinline__ void stage_tile_u8(const uint8_t *__restrict__ src, int spitch, int W, int H, int xs_lo, int ys_lo,
                                              float *__restrict__ tile, int warp, int lane)
{
    constexpr int NW = SWP / 4;
#pragma unroll 4
    for (int r = warp; r < SH; r += 8) {
        const uint8_t *srow = src + (size_t)reflect1(ys_lo + r, H) * spitch;
#pragma unroll
        for (int q4 = lane; q4 < NW; q4 += 32) {
            const int gx = xs_lo + 4 * q4;
            float4 f;
            if (gx >= 0 && gx + 3 < W) {
                const unsigned w0 = __ldg(reinterpret_cast<const unsigned *>(srow + gx));
                f.x = __uint_as_float(__byte_perm(w0, 0x4B000000u, 0x7650)) - 8388608.0f;
                f.y = __uint_as_float(__byte_perm(w0, 0x4B000000u, 0x7651)) - 8388608.0f;
                f.z = __uint_as_float(__byte_perm(w0, 0x4B000000u, 0x7652)) - 8388608.0f;
                f.w = __uint_as_float(__byte_perm(w0, 0x4B000000u, 0x7653)) - 8388608.0f;
            } else {
                f = make_float4(u8_to_float(__ldg(srow + reflect1(gx, W))), u8_to_float(__ldg(srow + reflect1(gx + 1, W))),
                                u8_to_float(__ldg(srow + reflect1(gx + 2, W))), u8_to_float(__ldg(srow + reflect1(gx + 3, W))));
            }
            *reinterpret_cast<float4 *>(tile + r * SWP + 4 * q4) = f;
        }
    }
}

// (a) full resolution: out = colpass3(rowpass3(u8)), tile 128 x 32, thread = column x 16 rows with a rolling window.
constexpr int LI_TW = 128, LI_TH = 32, LI_SH = LI_TH + 2, LI_SWP = LI_TW + 8;

__global__ void __launch_bounds__(256) level_ident_kernel(LevelFastArgs a)
{
    __shared__ __align__(16) float tile[LI_SH * LI_SWP];
    const int x0 = blockIdx.x * LI_TW, y0 = blockIdx.y * LI_TH;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint8_t *src = a.src + (size_t)blockIdx.z * a.H * a.spitch;
    stage_tile_u8<LI_SH, LI_SWP>(src, a.spitch, a.W, a.H, x0 - 4, y0 - 1, tile, warp, lane);
    __syncthreads();
    const int col = threadIdx.x & (LI_TW - 1), g = threadIdx.x >> 7;
    const int x = x0 + col;
    if (x >= a.d.w) return;
    const float k0 = a.k[0], k1 = a.k[1];
    const float *p = tile + (g * 16) * LI_SWP + col + 3; // left neighbour of column x in tile row g*16 (source row y0-1+g*16)
    float *dst = a.dst + (size_t)blockIdx.z * a.d.plane + x;
    float h0 = fmaf(p[1], k1, (p[0] + p[2]) * k0);
    p += LI_SWP;
    float h1 = fmaf(p[1], k1, (p[0] + p[2]) * k0);
#pragma unroll
    for (int i = 0; i < 16; i++) {
        p += LI_SWP;
        const float h2 = fmaf(p[1], k1, (p[0] + p[2]) * k0);
        const int y = y0 + g * 16 + i;
        if (y < a.d.h) dst[(size_t)y * a.d.pitch] = fmaf(h0 + h2, k0, h1 * k1);
        h0 = h1; h1 = h2;
    }
}

// (b) exact integer down-scale S with a K-tap pre-blur.
template <int S, int K, int TWO, int THO>
struct PyrGeom {
    static constexpr int C = K / 2;
    static constexpr int OFF = ((S / 2 - 1 - C) % 4 + 4) % 4;      // tile column of tap 0 of output column 0
    static constexpr int SH = S * THO - S + 2 * C + 2;
    static constexpr int SWRAW = S * TWO - S + 2 * C + 2 + OFF;
    static constexpr int SW4 = (SWRAW + 3) / 4;
    static constexpr int SWP = 4 * (SW4 | 1);                       // 4 * odd: conflict-free LDS.128 with lane = row
    static constexpr int RPP = TWO + 1;                             // float2 pitch of the row-pass buffer
    static constexpr int CPI = S >= 4 ? 1 : 4 / S;                  // output columns per row-pass item (keeps LDS.128 aligned)
    static constexpr int NLD = (OFF + K + 1 + S * (CPI - 1) + 3) / 4; // float4 loads per row-pass item
    static constexpr size_t SMEM = sizeof(float) * ((size_t)SH * SWP + (size_t)SH * RPP * 2);
};

template <int S, int K, int TWO, int THO>
__global__ void __launch_bounds__(256) level_pyr_kernel(LevelFastArgs a)
{
    using G = PyrGeom<S, K, TWO, THO>;
    constexpr int C = G::C;
    extern __shared__ __align__(16) float lp_smem[];
    float *tile = lp_smem;                                             // [SH][SWP]
    float2 *rp = reinterpret_cast<float2 *>(lp_smem + G::SH * G::SWP);  // [SH][RPP] (slot 0, slot 1)
    const int d0 = blockIdx.x * TWO, e0 = blockIdx.y * THO;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint8_t *src = a.src + (size_t)blockIdx.z * a.H * a.spitch;
    const int xs_lo = S * d0 + S / 2 - 1 - C - G::OFF, ys_lo = S * e0 + S / 2 - 1 - C;
    stage_tile_u8<G::SH, G::SWP>(src, a.spitch, a.W, a.H, xs_lo, ys_lo, tile, warp, lane);
    __syncthreads();

    // row pass: lane = tile row, warps stride over output columns; two adjacent source columns per item
    for (int rb = 0; rb < G::SH; rb += 32) {
        const int r = rb + lane;
        if (r < G::SH) {
            for (int dp = warp; dp < TWO / G::CPI; dp += 8) {
                const float4 *p4 = reinterpret_cast<const float4 *>(tile + r * G::SWP + S * G::CPI * dp);
                float v[G::NLD * 4];
#pragma unroll
                for (int q = 0; q < G::NLD; q++) {
                    const float4 u = p4[q];
                    v[4 * q] = u.x; v[4 * q + 1] = u.y; v[4 * q + 2] = u.z; v[4 * q + 3] = u.w;
                }
#pragma unroll
                for (int u = 0; u < G::CPI; u++) {
                    constexpr int O = G::OFF;
                    const int b = O + S * u;
                    float o0, o1;
                    if (K == 3) {
                        o0 = fmaf(v[b + 1], a.k[1], (v[b] + v[b + 2]) * a.k[0]);
                        o1 = fmaf(v[b + 2], a.k[1], (v[b + 1] + v[b + 3]) * a.k[0]);
                    } else {
                        o0 = v[b] * a.k[0];
                        o1 = v[b + 1] * a.k[0];
#pragma unroll
                        for (int j = 1; j < K; j++) {
                            o0 = fmaf(v[b + j], a.k[j], o0);
                            o1 = fmaf(v[b + 1 + j], a.k[j], o1);
                        }
                    }
                    rp[r * G::RPP + G::CPI * dp + u] = make_float2(o0, o1);
                }
            }
        }
    }
    __syncthreads();

    // column pass at the two source rows each output row reads, then the 0.5 / 0.5 bilinear blend
    float *dst = a.dst + (size_t)blockIdx.z * a.d.plane;
    for (int i = threadIdx.x; i < TWO * THO; i += 256) {
        const int el = i / TWO, dl = i - el * TWO;
        const int d = d0 + dl, e = e0 + el;
        if (d >= a.d.w || e >= a.d.h) continue;
        const float2 *q = rp + (S * el + C) * G::RPP + dl; // source row y0 of this output row
        float2 ra, rb2;
        if (K == 3) {
            const float2 u = q[-G::RPP], c0 = q[0], c1 = q[G::RPP], dn = q[2 * G::RPP];
            ra = make_float2(fmaf(u.x + c1.x, a.k[0], c0.x * a.k[1]), fmaf(u.y + c1.y, a.k[0], c0.y * a.k[1]));
            rb2 = make_float2(fmaf(c0.x + dn.x, a.k[0], c1.x * a.k[1]), fmaf(c0.y + dn.y, a.k[0], c1.y * a.k[1]));
        } else {
            const float2 c0 = q[0], c1 = q[G::RPP];
            ra = make_float2(c0.x * a.k[C], c0.y * a.k[C]);
            rb2 = make_float2(c1.x * a.k[C], c1.y * a.k[C]);
#pragma unroll
            for (int j = 1; j <= C; j++) {
                const float2 am = q[-j * G::RPP], ap = q[j * G::RPP], bm = q[(1 - j) * G::RPP], bp = q[(1 + j) * G::RPP];
                ra.x = fmaf(am.x + ap.x, a.k[C + j], ra.x); ra.y = fmaf(am.y + ap.y, a.k[C + j], ra.y);
                rb2.x = fmaf(bm.x + bp.x, a.k[C + j], rb2.x); rb2.y = fmaf(bm.y + bp.y, a.k[C + j], rb2.y);
            }
        }
        const float fx = 0.5f, gx = 1.f - fx, fy = 0.5f, gy = 1.f - fy;
        const float r0 = ra.x * gx + ra.y * fx;
        const float r1 = rb2.x * gx + rb2.y * fx;
        dst[(size_t)e * a.d.pitch + d] = r0 * gy + r1 * fy;
    }
}

template <int S, int K, int TWO, int THO>
static cudaError_t launch_pyr(cudaStream_t s, const LevelFastArgs &fa, int nimg)
{
    using G = PyrGeom<S, K, TWO, THO>;
    static std::atomic<bool> configured_dev[kMaxDevices];
    std::atomic<bool> &configured = configured_dev[current_device()];
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(level_pyr_kernel<S, K, TWO, THO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G::SMEM);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    dim3 grid((fa.d.w + TWO - 1) / TWO, (fa.d.h + THO - 1) / THO, nimg);
    level_pyr_kernel<S, K, TWO, THO><<<grid, 256, G::SMEM, s>>>(fa);
    return cudaGetLastError();
}

// (c) all four level images of the reference's default pyramid (pyrScale 0.5, pyrLevels 3 on a frame whose sides are
// multiples of 8: full resolution + S = 2, 4, 8) from ONE staged source tile: the u8 -> float staging, the dominant
// cost of (a)/(b), is paid once instead of four times and three launches disappear.  One CTA = 16 x 6 outputs of the
// coarsest level = 128 x 48 source pixels (+ halo).  Arithmetic per level is exactly that of (a) / (b).
constexpr int LF_TW3 = 16, LF_TH3 = 6, LF_SH = 60, LF_SWP = 148, LF_RPP = 65;
constexpr int LF_RAWP = 176; // bytes per staged raw row: 148 source columns + up to 8 of 16-byte alignment slack, multiple of 16
constexpr size_t LF_SMEM = sizeof(float) * ((size_t)LF_SH * LF_SWP + (size_t)LF_SH * LF_RPP * 2) + 16; // + mbarrier

struct LevelFusedArgs {
    const uint8_t *src; // [nimg][H][spitch]
    int W, H, spitch;
    float *dst[4];      // [nimg][h][pitch] for S = 8, 4, 2, 1 (coarse -> fine, the plan's scale order)
    LevelDims d[4];
    float k8[19], k4[9], k2[3], k1[3];
};

// row pass of scale S over the whole staged tile (lane = tile row), two adjacent source columns per output column
template <int S, int K, int TWO, int BASE>
__device__ __forceinline__ void lf_row_pass(const float *__restrict__ tile, float2 *__restrict__ rp, const float *__restrict__ k, int lane, int warp)
{
    constexpr int C = K / 2;
    constexpr int OFFL = S / 2 - 1 - C + 8 - BASE;              // tile column of tap 0 of output column 0, minus BASE
    constexpr int CPI = S >= 4 ? 1 : 4 / S;
    constexpr int NLD = (OFFL + K + 1 + S * (CPI - 1) + 3) / 4;
    constexpr int RPP = TWO + 1;
    static_assert(OFFL >= 0 && BASE % 4 == 0, "alignment");
    for (int rb = 0; rb < LF_SH; rb += 32) {
        const int r = rb + lane;
        if (r >= LF_SH) continue;
        for (int dp = warp; dp < TWO / CPI; dp += 8) {
            const float4 *p4 = reinterpret_cast<const float4 *>(tile + r * LF_SWP + BASE + S * CPI * dp);
            float v[NLD * 4];
#pragma unroll
            for (int q = 0; q < NLD; q++) {
                const float4 u = p4[q];
                v[4 * q] = u.x; v[4 * q + 1] = u.y; v[4 * q + 2] = u.z; v[4 * q + 3] = u.w;
            }
#pragma unroll
            for (int u = 0; u < CPI; u++) {
                const int b = OFFL + S * u;
                float o0, o1;
                if (K == 3) {
                    o0 = fmaf(v[b + 1], k[1], (v[b] + v[b + 2]) * k[0]);
                    o1 = fmaf(v[b + 2], k[1], (v[b + 1] + v[b + 3]) * k[0]);
                } else {
                    o0 = v[b] * k[0];
                    o1 = v[b + 1] * k[0];
#pragma unroll
                    for (int j = 1; j < K; j++) {
                        o0 = fmaf(v[b + j], k[j], o0);
                        o1 = fmaf(v[b + 1 + j], k[j], o1);
                    }
                }
                rp[r * RPP + CPI * dp + u] = make_float2(o0, o1);
            }
        }
    }
}

template <int S, int K, int TWO, int THO>
__device__ __forceinline__ void lf_col_pass(const float2 *__restrict__ rp, const float *__restrict__ k, float *__restrict__ dst, const LevelDims &d,
                                            int d0, int e0, int tid)
{
    constexpr int C = K / 2, RPP = TWO + 1;
    constexpr int ROFF = S / 2 - 1 - C + 6; // tile row of tap 0 of output row 0
    for (int i = tid; i < TWO * THO; i += 256) {
        const int el = i / TWO, dl = i - el * TWO;
        const int dd = d0 + dl, e = e0 + el;
        if (dd >= d.w || e >= d.h) continue;
        const float2 *q = rp + (ROFF + S * el + C) * RPP + dl;
        float2 ra, rb2;
        if (K == 3) {
            const float2 u = q[-RPP], c0 = q[0], c1 = q[RPP], dn = q[2 * RPP];
            ra = make_float2(fmaf(u.x + c1.x, k[0], c0.x * k[1]), fmaf(u.y + c1.y, k[0], c0.y * k[1]));
            rb2 = make_float2(fmaf(c0.x + dn.x, k[0], c1.x * k[1]), fmaf(c0.y + dn.y, k[0], c1.y * k[1]));
        } else {
            const float2 c0 = q[0], c1 = q[RPP];
            ra = make_float2(c0.x * k[C], c0.y * k[C]);
            rb2 = make_float2(c1.x * k[C], c1.y * k[C]);
#pragma unroll
            for (int j = 1; j <= C; j++) {
                const float2 am = q[-j * RPP], ap = q[j * RPP], bm = q[(1 - j) * RPP], bp = q[(1 + j) * RPP];
                ra.x = fmaf(am.x + ap.x, k[C + j], ra.x); ra.y = fmaf(am.y + ap.y, k[C + j], ra.y);
                rb2.x = fmaf(bm.x + bp.x, k[C + j], rb2.x); rb2.y = fmaf(bm.y + bp.y, k[C + j], rb2.y);
            }
        }
        const float fx = 0.5f, gx = 1.f - fx, fy = 0.5f, gy = 1.f - fy;
        const float r0 = ra.x * gx + ra.y * fx;
        const float r1 = rb2.x * gx + rb2.y * fx;
        dst[(size_t)e * d.pitch + dd] = r0 * gy + r1 * fy;
    }
}

__global__ void __launch_bounds__(256) level_fused_kernel(LevelFusedArgs a)
{
    extern __shared__ __align__(16) float lf_smem[];
    float *tile = lf_smem;                                              // [60][148]
    float2 *rp = reinterpret_cast<float2 *>(lf_smem + LF_SH * LF_SWP);  // [60][<= 65]
    const int d0 = blockIdx.x * LF_TW3, e0 = blockIdx.y * LF_TH3;       // coarsest-level tile origin
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint8_t *src = a.src + (size_t)blockIdx.z * a.H * a.spitch;
    const int xs_lo = 8 * d0 - 8, ys_lo = 8 * e0 - 6, xs16 = xs_lo & ~15;
    // Interior tiles (no REFLECT_101 needed) are staged by the TMA engine: 60 bulk row copies global -> shared
    // (cp.async.bulk, completion on an mbarrier), then one pass converts the raw bytes to the float tile.  The raw
    // buffer aliases the row-pass buffer, which is not live yet.  Border tiles take the per-thread reflecting loads.
    const bool interior = xs_lo >= 0 && xs_lo + LF_SWP <= a.W && xs16 + LF_RAWP <= a.spitch && ys_lo >= 0 && ys_lo + LF_SH <= a.H;
    if (interior) {
        unsigned char *raw = reinterpret_cast<unsigned char *>(rp);
        unsigned long long *mbar = reinterpret_cast<unsigned long long *>(lf_smem + LF_SH * LF_SWP + LF_SH * LF_RPP * 2);
        const unsigned mbar_s = (unsigned)__cvta_generic_to_shared(mbar);
        if (tid == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar_s));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar_s), "r"(LF_SH * LF_RAWP) : "memory");
            const uint8_t *g = src + (size_t)ys_lo * a.spitch + xs16;
            const unsigned raw_s = (unsigned)__cvta_generic_to_shared(raw);
            for (int r = 0; r < LF_SH; r++)
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(raw_s + r * LF_RAWP),
                             "l"(g + (size_t)r * a.spitch), "r"(LF_RAWP), "r"(mbar_s)
                             : "memory");
        }
        __syncthreads(); // the mbarrier is initialised before anybody polls it
        unsigned done = 0;
        for (int spin = 0; !done; spin++) {
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(mbar_s) : "memory");
            if (spin > (1 << 24)) __trap(); // never hang the GPU on a lost completion
        }
        const int off = xs_lo - xs16; // 0 or 8
        for (int i = tid; i < LF_SH * (LF_SWP / 4); i += 256) {
            const int r = i / (LF_SWP / 4), q4 = i - r * (LF_SWP / 4);
            const unsigned w0 = *reinterpret_cast<const unsigned *>(raw + r * LF_RAWP + off + 4 * q4);
            float4 f;
            f.x = __uint_as_float(__byte_perm(w0, 0x4B000000u, 0x7650)) - 8388608.0f;
            f.y = __uint_as_float(__byte_perm(w0, 0x4B000000u, 0x7651)) - 8388608.0f;
            f.z = __uint_as_float(__byte_perm(w0, 0x4B000000u, 0x7652)) - 8388608.0f;
            f.w = __uint_as_float(__byte_perm(w0, 0x4B000000u, 0x7653)) - 8388608.0f;
            *reinterpret_cast<float4 *>(tile + r * LF_SWP + 4 * q4) = f;
        }
    } else {
        stage_tile_u8<LF_SH, LF_SWP>(src, a.spitch, a.W, a.H, xs_lo, ys_lo, tile, warp, lane);
    }
    __syncthreads();

    // full resolution (3-tap blur, no resize): thread = column x 24 rows, rolling window; tile col = x - 8*d0 + 8, row = y - 8*e0 + 6
    {
        const int col = tid & 127, g = tid >> 7;
        const int x = 8 * d0 + col;
        if (x < a.d[3].w) {
            const float k0 = a.k1[0], k1 = a.k1[1];
            const float *p = tile + (g * 24 + 5) * LF_SWP + col + 7; // left neighbour of x in the row above the first output row
            float *dst = a.dst[3] + (size_t)blockIdx.z * a.d[3].plane + x;
            float h0 = fmaf(p[1], k1, (p[0] + p[2]) * k0);
            p += LF_SWP;
            float h1 = fmaf(p[1], k1, (p[0] + p[2]) * k0);
#pragma unroll
            for (int i = 0; i < 24; i++) {
                p += LF_SWP;
                const float h2 = fmaf(p[1], k1, (p[0] + p[2]) * k0);
                const int y = 8 * e0 + g * 24 + i;
                if (y < a.d[3].h) dst[(size_t)y * a.d[3].pitch] = fmaf(h0 + h2, k0, h1 * k1);
                h0 = h1; h1 = h2;
            }
        }
    }
    // S = 2 (K = 3), 64 x 24 outputs
    lf_row_pass<2, 3, 64, 4>(tile, rp, a.k2, lane, warp);
    __syncthreads();
    lf_col_pass<2, 3, 64, 24>(rp, a.k2, a.dst[2] + (size_t)blockIdx.z * a.d[2].plane, a.d[2], 4 * d0, 4 * e0, tid);
    __syncthreads();
    // S = 4 (K = 9), 32 x 12 outputs
    lf_row_pass<4, 9, 32, 4>(tile, rp, a.k4, lane, warp);
    __syncthreads();
    lf_col_pass<4, 9, 32, 12>(rp, a.k4, a.dst[1] + (size_t)blockIdx.z * a.d[1].plane, a.d[1], 2 * d0, 2 * e0, tid);
    __syncthreads();
    // S = 8 (K = 19), 16 x 6 outputs
    lf_row_pass<8, 19, 16, 0>(tile, rp, a.k8, lane, warp);
    __syncthreads();
    lf_col_pass<8, 19, 16, 6>(rp, a.k8, a.dst[0] + (size_t)blockIdx.z * a.d[0].plane, a.d[0], d0, e0, tid);
}

cudaError_t launch_level_fused(cudaStream_t s, const uint8_t *src, int W, int H, int spitch, float *const dst[4], const LevelDims d[4],
                               const float *k8, const float *k4, const float *k2, const float *k1, int nimg)
{
    static std::atomic<bool> configured_dev[kMaxDevices];
    std::atomic<bool> &configured = configured_dev[current_device()];
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(level_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LF_SMEM);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    LevelFusedArgs a{};
    a.src = src; a.W = W; a.H = H; a.spitch = spitch;
    for (int i = 0; i < 4; i++) { a.dst[i] = dst[i]; a.d[i] = d[i]; }
    for (int i = 0; i < 19; i++) a.k8[i] = k8[i];
    for (int i = 0; i < 9; i++) a.k4[i] = k4[i];
    for (int i = 0; i < 3; i++) { a.k2[i] = k2[i]; a.k1[i] = k1[i]; }
    dim3 grid((d[0].w + LF_TW3 - 1) / LF_TW3, (d[0].h + LF_TH3 - 1) / LF_TH3, nimg);
    level_fused_kernel<<<grid, 256, LF_SMEM, s>>>(a);
    return cudaGetLastError();
}

// Returns cudaErrorNotSupported when no fast path applies (the caller then uses the generic kernel).
cudaError_t launch_level_image_fast(cudaStream_t s, const LevelImageArgs &a, const float *host_taps, int int_scale)
{
    if (a.small || a.ksize > 40) return cudaErrorNotSupported;
    LevelFastArgs fa{};
    fa.src = a.src; fa.W = a.W; fa.H = a.H; fa.spitch = a.spitch; fa.dst = a.dst; fa.d = a.d;
    for (int i = 0; i < a.ksize; i++) fa.k[i] = host_taps[i];
    if (a.identity && a.ksize == 3) {
        dim3 grid((a.d.w + LI_TW - 1) / LI_TW, (a.d.h + LI_TH - 1) / LI_TH, a.nimg);
        level_ident_kernel<<<grid, 256, 0, s>>>(fa);
        return cudaGetLastError();
    }
    if (int_scale == 2 && a.ksize == 3) return launch_pyr<2, 3, 64, 15>(s, fa, a.nimg);
    if (int_scale == 4 && a.ksize == 9) return launch_pyr<4, 9, 32, 6>(s, fa, a.nimg);
    if (int_scale == 8 && a.ksize == 19) return launch_pyr<8, 19, 16, 6>(s, fa, a.nimg);
    if (int_scale == 16 && a.ksize == 39) return launch_pyr<16, 39, 8, 2>(s, fa, a.nimg);
    return cudaErrorNotSupported;
}

// ------------------------------------------------------------------------------------------------
// K2  polynomial expansion, SURVEY App. A.3.  Separable: vertical pass in float (no FMA) into shared
//     memory (r0, r1, r2), horizontal pass with double accumulators.
// ------------------------------------------------------------------------------------------------
constexpr int PE_TW = 64, PE_TH = 16;

__global__ void __launch_bounds__(256) polyexp_kernel(const float *__restrict__ I, float *__restrict__ R, LevelDims d,
                                                      PolyTables t)
{
    extern __shared__ float pe_smem[];
    const int n = t.n;
    const int SWD = PE_TW + 2 * n;
    float *s0 = pe_smem, *s1 = s0 + PE_TH * SWD, *s2 = s1 + PE_TH * SWD;
    const int x0 = blockIdx.x * PE_TW, y0 = blockIdx.y * PE_TH;
    const float *img = I + (size_t)blockIdx.z * d.plane;
    const int w = d.w, h = d.h, pitch = d.pitch;

    for (int i = threadIdx.x; i < SWD * PE_TH; i += blockDim.x) {
        int row = i / SWD, col = i - row * SWD;
        int gy = y0 + row;
        if (gy >= h) continue;
        int gx = clampi(x0 - n + col, 0, w - 1);
        float r0 = img[(size_t)gy * pitch + gx] * t.g[0], r1 = 0.f, r2 = 0.f;
        for (int k = 1; k <= n; k++) {
            float up = img[(size_t)max(gy - k, 0) * pitch + gx], dn = img[(size_t)min(gy + k, h - 1) * pitch + gx];
            float p = up + dn, q = dn - up;
            r0 = r0 + t.g[k] * p;
            r1 = r1 + t.xg[k] * q;
            r2 = r2 + t.xxg[k] * p;
        }
        s0[i] = r0; s1[i] = r1; s2[i] = r2;
    }
    __syncthreads();

    float *out = R + (size_t)blockIdx.z * 5 * d.plane;
    for (int i = threadIdx.x; i < PE_TW * PE_TH; i += blockDim.x) {
        int row = i / PE_TW, col = i - row * PE_TW;
        int gx = x0 + col, gy = y0 + row;
        if (gx >= w || gy >= h) continue;
        const float *p0 = s0 + row * SWD + col + n, *p1 = s1 + row * SWD + col + n, *p2 = s2 + row * SWD + col + n;
        float g0 = t.g[0];
        double b1 = (double)(p0[0] * g0), b2 = 0, b3 = (double)(p1[0] * g0), b4 = 0, b5 = (double)(p2[0] * g0), b6 = 0;
        for (int k = 1; k <= n; k++) {
            float a0 = p0[k], m0 = p0[-k], a1 = p1[k], m1 = p1[-k], a2 = p2[k], m2 = p2[-k];
            double tg = (double)(a0 + m0);
            b1 = b1 + tg * t.gd[k];
            b4 = b4 + tg * t.xxgd[k];
            b2 = b2 + (double)((a0 - m0) * t.xg[k]);
            b3 = b3 + (double)((a1 + m1) * t.g[k]);
            b6 = b6 + (double)((a1 - m1) * t.xg[k]);
            b5 = b5 + (double)((a2 + m2) * t.g[k]);
        }
        size_t o = (size_t)gy * 5 * pitch + gx; // R is row-interleaved: (y, c, x) at (y*5 + c)*pitch + x
        out[o] = (float)(b3 * t.ig11);
        out[o + pitch] = (float)(b2 * t.ig11);
        out[o + 2 * pitch] = (float)(b1 * t.ig03 + b5 * t.ig33);
        out[o + 3 * pitch] = (float)(b1 * t.ig03 + b4 * t.ig33);
        out[o + 4 * pitch] = (float)(b6 * t.ig55);
    }
}

// K2 fast path (polyN = 7 or 5): tile 96 x 16, 256 threads.
//   phase V: thread = (column, 8-row group): 8 + 2N inputs in registers, (r0, r1, r2) for 8 rows -> shared [3][16][112]
//   phase H: lane = x (conflict-free LDS, coalesced stores), taps unrolled, double accumulators exactly as App. A.3.
// The F2F.F64.F32 conversions (3 + 5N per pixel) run on the XU pipe at 16 lanes/clk/SM and bound this kernel.
constexpr int PF_TW = 96, PF_TH = 16, PF_VW = 112, PF_RV = 8;

template <int N, int PITCH>
__global__ void __launch_bounds__(256) polyexp_fast_kernel(const float *__restrict__ I, float *__restrict__ R, LevelDims d, PolyTables t)
{
    __shared__ float sm[3][PF_TH * PF_VW];
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * PF_TW, y0 = blockIdx.y * PF_TH;
    const float *img = I + (size_t)blockIdx.z * d.plane;
    const int w = d.w, h = d.h, pitch = PITCH ? PITCH : d.pitch;
    const bool interior = (y0 - N >= 0) && (y0 + PF_TH + N - 1 <= h - 1); // block-uniform

    if (tid < 2 * PF_VW) {
        const int g = tid / PF_VW, j = tid - g * PF_VW;
        const int gx = clampi(x0 - 8 + j, 0, w - 1);
        const int ybase = y0 + g * PF_RV - N;
        float in[PF_RV + 2 * N];
        if (interior) {
            const unsigned rsb = (unsigned)pitch * 4u;
            const char *p = row_ptr(reinterpret_cast<const char *>(img + gx), rsb, (unsigned)ybase);
#pragma unroll
            for (int r = 0; r < PF_RV + 2 * N; r++) {
                if (PITCH) in[r] = __ldg(reinterpret_cast<const float *>(p) + (size_t)r * PITCH);
                else in[r] = __ldg(reinterpret_cast<const float *>(row_ptr(p, rsb, (unsigned)r)));
            }
        } else {
#pragma unroll
            for (int r = 0; r < PF_RV + 2 * N; r++) in[r] = __ldg(img + (size_t)clampi(ybase + r, 0, h - 1) * pitch + gx);
        }
#pragma unroll
        for (int o = 0; o < PF_RV; o++) {
            float r0 = in[o + N] * t.g[0], r1 = 0.f, r2 = 0.f;
#pragma unroll
            for (int k = 1; k <= N; k++) {
                float up = in[o + N - k], dn = in[o + N + k];
                float p = up + dn, q = dn - up;
                r0 = r0 + t.g[k] * p;
                r1 = r1 + t.xg[k] * q;
                r2 = r2 + t.xxg[k] * p;
            }
            const int si = (g * PF_RV + o) * PF_VW + j;
            sm[0][si] = r0; sm[1][si] = r1; sm[2][si] = r2;
        }
    }
    __syncthreads();

    float *out = R + (size_t)blockIdx.z * 5 * d.plane;
    const float g0 = t.g[0];
    // 2 adjacent pixels per thread: 2N+2 floats per plane as 8-byte shared loads (lane stride 8 B: conflict-free)
#pragma unroll 1
    for (int i = tid; i < (PF_TW / 2) * PF_TH; i += 256) {
        const int row = i / (PF_TW / 2), col = (i - row * (PF_TW / 2)) * 2;
        const int gx = x0 + col, gy = y0 + row;
        if (gx >= w || gy >= h) continue;
        // taps of pixel col are smem columns col+8-N .. col+8+N; col is even, so col+8-NE (NE = N rounded up to even) is 8B-aligned
        constexpr int NE = (N + 1) & ~1, NF = 2 * NE + 2;
        float v[3][NF];
#pragma unroll
        for (int pl = 0; pl < 3; pl++) {
            const float2 *src = reinterpret_cast<const float2 *>(&sm[pl][row * PF_VW + col + 8 - NE]);
#pragma unroll
            for (int q = 0; q < NF / 2; q++) { float2 u = src[q]; v[pl][2 * q] = u.x; v[pl][2 * q + 1] = u.y; }
        }
        float res[2][5];
#pragma unroll
        for (int px = 0; px < 2; px++) {
            const int ctr = NE + px;
            double b1 = (double)(v[0][ctr] * g0), b2 = 0, b3 = (double)(v[1][ctr] * g0), b4 = 0, b5 = (double)(v[2][ctr] * g0), b6 = 0;
#pragma unroll
            for (int k = 1; k <= N; k++) {
                const float a0 = v[0][ctr + k], m0 = v[0][ctr - k], a1 = v[1][ctr + k], m1 = v[1][ctr - k], a2 = v[2][ctr + k], m2 = v[2][ctr - k];
                const double tg = (double)(a0 + m0);
                b1 = b1 + tg * t.gd[k];
                b4 = b4 + tg * t.xxgd[k];
                b2 = b2 + (double)((a0 - m0) * t.xg[k]);
                b3 = b3 + (double)((a1 + m1) * t.g[k]);
                b6 = b6 + (double)((a1 - m1) * t.xg[k]);
                b5 = b5 + (double)((a2 + m2) * t.g[k]);
            }
            res[px][0] = (float)(b3 * t.ig11);
            res[px][1] = (float)(b2 * t.ig11);
            res[px][2] = (float)(b1 * t.ig03 + b5 * t.ig33);
            res[px][3] = (float)(b1 * t.ig03 + b4 * t.ig33);
            res[px][4] = (float)(b6 * t.ig55);
        }
        const size_t o = (size_t)gy * 5 * pitch + gx; // row-interleaved R
        if (gx + 1 < w) {
#pragma unroll
            for (int c = 0; c < 5; c++) *reinterpret_cast<float2 *>(out + o + c * pitch) = make_float2(res[0][c], res[1][c]);
        } else {
#pragma unroll
            for (int c = 0; c < 5; c++) out[o + c * pitch] = res[0][c];
        }
    }
}

// K2, relaxed arithmetic (tw_set_option "arithmetic" = 1; Gaussian window with winSize >= 30 only -- see tw_context.cu).
// The faithful kernel above is bound by its 3 + 5N float -> double conversions per pixel (XU pipe, 16 lanes/clk/SM).
// Here the horizontal pass converts each staged value ONCE per thread (4 adjacent pixels share 2N+4 values per plane)
// and only for the three sums that meet in a cancelling combination (b1, b4, b5 -> the second-derivative
// coefficients); b2, b3, b6 (first derivatives, mixed term) are float fmaf chains.  What is dropped relative to App. A.3
// are float roundings of sums / products that the double accumulation then carried exactly; the vertical pass is
// unchanged.  The same arithmetic is restated in oracle/farneback_ref.c under twref_set_relax(16): the GPU result is
// checked bit for bit against that, and against the faithful oracle within the north-star tolerance
// (measured <= 2.6e-4 px at 1920x1080, 2.1e-3 px on the reference's fixture; tools/relax_study.py).
//   tile 96 x 32, 256 threads; phase V: thread = (column pair, 8-row group), 8 + 2N float2 inputs in registers, packed f32x2;
//   phase H: thread = 4 adjacent pixels, LDS.128 (lane stride 16 B: conflict-free), float4 stores.
constexpr int PM_TW = 96, PM_TH = 32, PM_VW = 112, PM_RV = 8;

template <int N, int PITCH>
__global__ void __launch_bounds__(256, 2) polyexp_mixed_kernel(const float *__restrict__ I, float *__restrict__ R, LevelDims d, PolyTables t,
                                                               const __grid_constant__ TileMap imap)
{
    // dynamic shared memory: input tile staged by TMA [PM_TH + 2N][PM_VW] (interior tiles) | mbarrier | the three V planes
    extern __shared__ __align__(128) unsigned char pm_smem[];
    float *sin_ = reinterpret_cast<float *>(pm_smem);
    constexpr int PM_IN_BYTES = (PM_TH + 2 * N) * PM_VW * 4;
    constexpr int PM_BAR_OFF = (PM_IN_BYTES + 127) & ~127;
    float (*sm)[PM_TH * PM_VW] = reinterpret_cast<float (*)[PM_TH * PM_VW]>(pm_smem + PM_BAR_OFF + 128);
    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * PM_TW, y0 = blockIdx.y * PM_TH;
    const float *img = I + (size_t)blockIdx.z * d.plane;
    const int w = d.w, h = d.h, pitch = PITCH ? PITCH : d.pitch;
    const bool interior = (y0 - N >= 0) && (y0 + PM_TH + N - 1 <= h - 1); // block-uniform

    // Interior tiles (the whole 112 x (32 + 2N) input window inside the frame): ONE tensor-map TMA copy stages the tile
    // (cp.async.bulk.tensor, UTMALDG); tiles that touch the frame border keep the per-thread loads with the replicate clamp.
    const bool tma_tile = imap.valid && interior && x0 - 8 >= 0 && x0 - 8 + PM_VW <= w;
    if (tma_tile) {
        const unsigned bar = (unsigned)__cvta_generic_to_shared(pm_smem + PM_BAR_OFF);
        if (tid == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((unsigned)PM_IN_BYTES) : "memory");
            asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
                             (unsigned)__cvta_generic_to_shared(pm_smem)),
                         "l"(reinterpret_cast<unsigned long long>(&imap)), "r"(bar), "r"(x0 - 8), "r"(y0 - N), "r"((int)blockIdx.z)
                         : "memory");
        }
        __syncthreads(); // the barrier is initialised before anybody probes it
        unsigned done = 0;
        while (!done)
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(bar) : "memory");
    }
    // phase V, packed f32x2: thread = (column PAIR, 8-row group); every operation of App. A.3's vertical pass is issued once for the
    // two columns (each half one IEEE operation, so the values are those of the scalar form; the rounded sum "acc + k * p" is
    // fma(k * p, one, acc) with the runtime 1.0f, see tw_fma2)
    if (tid < (PM_VW / 2) * (PM_TH / PM_RV)) {
        const int g = tid / (PM_VW / 2), jj = tid - g * (PM_VW / 2);
        const int xa = x0 - 8 + 2 * jj;
        const int ybase = y0 + g * PM_RV - N;
        const bool pairok = xa >= 0 && xa + 1 <= w - 1; // both columns inside: one 8-byte load per row
        const int ga = clampi(xa, 0, w - 1), gb = clampi(xa + 1, 0, w - 1);
        float2 in[PM_RV + 2 * N];
        if (tma_tile) {
#pragma unroll
            for (int r = 0; r < PM_RV + 2 * N; r++) in[r] = *reinterpret_cast<const float2 *>(sin_ + (g * PM_RV + r) * PM_VW + 2 * jj);
        } else if (interior && pairok) {
            const unsigned rsb = (unsigned)pitch * 4u;
            const char *p = row_ptr(reinterpret_cast<const char *>(img + xa), rsb, (unsigned)ybase);
#pragma unroll
            for (int r = 0; r < PM_RV + 2 * N; r++) {
                if (PITCH) in[r] = __ldg(reinterpret_cast<const float2 *>(reinterpret_cast<const float *>(p) + (size_t)r * PITCH));
                else in[r] = __ldg(reinterpret_cast<const float2 *>(row_ptr(p, rsb, (unsigned)r)));
            }
        } else {
#pragma unroll
            for (int r = 0; r < PM_RV + 2 * N; r++) {
                const float *row = img + (size_t)clampi(ybase + r, 0, h - 1) * pitch;
                in[r] = make_float2(__ldg(row + ga), __ldg(row + gb));
            }
        }
        const float2 one2 = make_float2(t.one, t.one);
#pragma unroll
        for (int o = 0; o < PM_RV; o++) {
            float2 r0 = tw_mul2(in[o + N], make_float2(t.g[0], t.g[0])), r1 = make_float2(0.f, 0.f), r2 = make_float2(0.f, 0.f);
#pragma unroll
            for (int k = 1; k <= N; k++) {
                const float2 up = in[o + N - k], dn = in[o + N + k];
                const float2 p = tw_add2(up, dn), q = tw_sub2(dn, up);
                r0 = tw_fma2(tw_mul2(make_float2(t.g[k], t.g[k]), p), one2, r0);
                r1 = tw_fma2(tw_mul2(make_float2(t.xg[k], t.xg[k]), q), one2, r1);
                r2 = tw_fma2(tw_mul2(make_float2(t.xxg[k], t.xxg[k]), p), one2, r2);
            }
            const int si = (g * PM_RV + o) * PM_VW + 2 * jj;
            *reinterpret_cast<float2 *>(&sm[0][si]) = r0;
            *reinterpret_cast<float2 *>(&sm[1][si]) = r1;
            *reinterpret_cast<float2 *>(&sm[2][si]) = r2;
        }
    }
    __syncthreads();

    float *out = R + (size_t)blockIdx.z * 5 * d.plane;
    constexpr int LO = (8 - N) & ~3;                 // first staged column read, 16-byte aligned
    constexpr int NV = ((3 + 8 + N) | 3) + 1 - LO;   // floats read per plane (multiple of 4)
#pragma unroll 1
    for (int i = tid; i < (PM_TW / 4) * PM_TH; i += 256) {
        const int row = i / (PM_TW / 4), col = (i - row * (PM_TW / 4)) * 4;
        const int gx = x0 + col, gy = y0 + row;
        if (gx >= w || gy >= h) continue;
        float res[5][4];
        double t1[4]; // b1 * ig03
        float v[NV];
        double dv[NV];
        auto load_plane = [&](int pl) {
            const float4 *src = reinterpret_cast<const float4 *>(&sm[pl][row * PM_VW + col + LO]);
#pragma unroll
            for (int q = 0; q < NV / 4; q++) {
                const float4 u = src[q];
                v[4 * q] = u.x; v[4 * q + 1] = u.y; v[4 * q + 2] = u.z; v[4 * q + 3] = u.w;
            }
        };
        // plane 0 (r0): b1, b4 in double; b2 in float, two pixels per packed fmaf (each half the scalar fmaf of oracle relax bit 4)
        load_plane(0);
#pragma unroll
        for (int q = 0; q < NV; q++) dv[q] = (double)v[q];
#pragma unroll
        for (int px = 0; px < 4; px++) {
            const int ctr = px + 8 - LO;
            double b1 = dv[ctr] * t.gd[0], b4 = 0.0;
#pragma unroll
            for (int k = 1; k <= N; k++) {
                const double tg = dv[ctr + k] + dv[ctr - k];
                b1 = fma(tg, t.gd[k], b1);
                b4 = fma(tg, t.xxgd[k], b4);
            }
            t1[px] = b1 * t.ig03;
            res[3][px] = (float)(t1[px] + b4 * t.ig33);
        }
#pragma unroll
        for (int px = 0; px < 4; px += 2) {
            const int ctr = px + 8 - LO;
            float2 b2 = make_float2(0.f, 0.f);
#pragma unroll
            for (int k = 1; k <= N; k++)
                b2 = tw_fma2(make_float2(v[ctr + k] - v[ctr - k], v[ctr + 1 + k] - v[ctr + 1 - k]), make_float2(t.xg[k], t.xg[k]), b2);
            res[1][px] = b2.x * t.fig11;
            res[1][px + 1] = b2.y * t.fig11;
        }
        // plane 2 (r2): b5 in double
        load_plane(2);
#pragma unroll
        for (int q = 0; q < NV; q++) dv[q] = (double)v[q];
#pragma unroll
        for (int px = 0; px < 4; px++) {
            const int ctr = px + 8 - LO;
            double b5 = dv[ctr] * t.gd[0];
#pragma unroll
            for (int k = 1; k <= N; k++) b5 = fma(dv[ctr + k] + dv[ctr - k], t.gd[k], b5);
            res[2][px] = (float)(t1[px] + b5 * t.ig33);
        }
        // plane 1 (r1): b3, b6 in float, packed as (b3, b6): fmaf(sum, g, b3) and fmaf(diff, xg, b6) in one instruction
        load_plane(1);
#pragma unroll
        for (int px = 0; px < 4; px++) {
            const int ctr = px + 8 - LO;
            float2 b36 = make_float2(v[ctr] * t.g[0], 0.f);
#pragma unroll
            for (int k = 1; k <= N; k++)
                b36 = tw_fma2(make_float2(v[ctr + k] + v[ctr - k], v[ctr + k] - v[ctr - k]), make_float2(t.g[k], t.xg[k]), b36);
            res[0][px] = b36.x * t.fig11;
            res[4][px] = b36.y * t.fig55;
        }
        const size_t o = (size_t)gy * 5 * pitch + gx; // row-interleaved R
        if (gx + 3 < w) {
#pragma unroll
            for (int c = 0; c < 5; c++) *reinterpret_cast<float4 *>(out + o + c * pitch) = make_float4(res[c][0], res[c][1], res[c][2], res[c][3]);
        } else {
#pragma unroll
            for (int px = 0; px < 4; px++) {
                if (gx + px < w) {
#pragma unroll
                    for (int c = 0; c < 5; c++) out[o + c * pitch + px] = res[c][px];
                }
            }
        }
    }
}

template <int N, int PITCH>
static cudaError_t launch_polyexp_mixed_p(cudaStream_t s, const float *I, float *R, const LevelDims &d, int nimg, const PolyTables &t, const TileMap &imap)
{
    static std::atomic<bool> configured_dev[kMaxDevices];
    std::atomic<bool> &configured = configured_dev[current_device()];
    constexpr int smem = (((PM_TH + 2 * N) * PM_VW * 4 + 127) & ~127) + 128 + 3 * PM_TH * PM_VW * 4;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(polyexp_mixed_kernel<N, PITCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    dim3 grid((d.w + PM_TW - 1) / PM_TW, (d.h + PM_TH - 1) / PM_TH, nimg);
    polyexp_mixed_kernel<N, PITCH><<<grid, 256, smem, s>>>(I, R, d, t, imap);
    return cudaGetLastError();
}

template <int N>
static cudaError_t launch_polyexp_mixed(cudaStream_t s, const float *I, float *R, const LevelDims &d, int nimg, const PolyTables &t, const TileMap *imap)
{
    TileMap none{};
    const TileMap &m = (imap && imap->valid) ? *imap : none;
    if (d.pitch == 2048) return launch_polyexp_mixed_p<N, 2048>(s, I, R, d, nimg, t, m);
    if (d.pitch == 4096) return launch_polyexp_mixed_p<N, 4096>(s, I, R, d, nimg, t, m);
    return launch_polyexp_mixed_p<N, 0>(s, I, R, d, nimg, t, m);
}

cudaError_t launch_polyexp(cudaStream_t s, const float *I, float *R, const LevelDims &d, int nimg, const PolyTables &t, int relaxed, const TileMap *imap)
{
    if (relaxed && t.n == 7) return launch_polyexp_mixed<7>(s, I, R, d, nimg, t, imap);
    if (relaxed && t.n == 5) return launch_polyexp_mixed<5>(s, I, R, d, nimg, t, imap);
    if (t.n == 7 || t.n == 5) {
        dim3 grid((d.w + PF_TW - 1) / PF_TW, (d.h + PF_TH - 1) / PF_TH, nimg);
        if (t.n == 7) {
            if (d.pitch == 2048) polyexp_fast_kernel<7, 2048><<<grid, 256, 0, s>>>(I, R, d, t);
            else if (d.pitch == 4096) polyexp_fast_kernel<7, 4096><<<grid, 256, 0, s>>>(I, R, d, t);
            else polyexp_fast_kernel<7, 0><<<grid, 256, 0, s>>>(I, R, d, t);
        } else {
            if (d.pitch == 2048) polyexp_fast_kernel<5, 2048><<<grid, 256, 0, s>>>(I, R, d, t);
            else if (d.pitch == 4096) polyexp_fast_kernel<5, 4096><<<grid, 256, 0, s>>>(I, R, d, t);
            else polyexp_fast_kernel<5, 0><<<grid, 256, 0, s>>>(I, R, d, t);
        }
        return cudaGetLastError();
    }
    dim3 grid((d.w + PE_TW - 1) / PE_TW, (d.h + PE_TH - 1) / PE_TH, nimg);
    size_t smem = sizeof(float) * 3 * PE_TH * (PE_TW + 2 * t.n);
    polyexp_kernel<<<grid, 256, smem, s>>>(I, R, d, t);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// A.4  update matrices for one pixel.  All float, no FMA.  R0/R1 point at channel 0 of the pair's planes.
// ------------------------------------------------------------------------------------------------
// The epilogues are latency-bound, so the 25 loads of a pixel are issued first (upd_load) for several pixels
// and consumed afterwards (upd_compute).
struct UpdLoad {
    float q[5];    // R0 at (x, y)
    float p[5][4]; // R1 at (x1, y1), (x1+1, y1), (x1, y1+1), (x1+1, y1+1)
    float fx, fy;
    bool inside;
};

__device__ __forceinline__ void upd_load(const float *__restrict__ R0, const float *__restrict__ R1, int pitch, int w,
                                         int h, int x, int y, float dx, float dy, UpdLoad &L)
{
    const float *q0 = R0 + (size_t)y * 5 * pitch + x;
    float fx = (float)x + dx, fy = (float)y + dy;
    const int x1 = __float2int_rd(fx), y1 = __float2int_rd(fy);
    L.fx = fx - (float)x1;
    L.fy = fy - (float)y1;
    L.inside = (unsigned)x1 < (unsigned)(w - 1) && (unsigned)y1 < (unsigned)(h - 1);
#pragma unroll
    for (int c = 0; c < 5; c++) L.q[c] = __ldg(q0 + c * pitch);
    if (L.inside) {
        const float *p = R1 + (size_t)y1 * 5 * pitch + x1;
#pragma unroll
        for (int c = 0; c < 5; c++) {
            L.p[c][0] = __ldg(p + c * pitch); L.p[c][1] = __ldg(p + c * pitch + 1);
            L.p[c][2] = __ldg(p + (5 + c) * pitch); L.p[c][3] = __ldg(p + (5 + c) * pitch + 1);
        }
    }
}

__device__ __forceinline__ void upd_compute(const UpdLoad &L, int w, int h, int x, int y, float dx, float dy, float m[5])
{
    float pt[5][2], pb[5][2];
#pragma unroll
    for (int c = 0; c < 5; c++) { pt[c][0] = L.p[c][0]; pt[c][1] = L.p[c][1]; pb[c][0] = L.p[c][2]; pb[c][1] = L.p[c][3]; }
    upd_core(L.q, pt, pb, L.inside, L.fx, L.fy, w, h, x, y, dx, dy, m);
}

__device__ __forceinline__ void update_matrices_px(const float *__restrict__ R0, const float *__restrict__ R1,
                                                   int pitch, int w, int h, int x, int y, float dx, float dy, float m[5])
{
    UpdLoad L;
    upd_load(R0, R1, pitch, w, h, x, y, dx, dy, L);
    upd_compute(L, w, h, x, y, dx, dy, m);
}

// ------------------------------------------------------------------------------------------------
// K3  flow initialisation for a scale (zero, or bilinear upsample of the coarser flow * 1/pyrScale,
//     App. A.1 / A.2b) fused with the first update-matrices (A.4).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void upsample_flow_px(const FirstUpdateArgs &a, int b, int x, int y, float &dx, float &dy)
{
    dx = 0.f; dy = 0.f;
    if (a.flow_in) { // same-size flow (box window: the solve ran in its own kernel)
        const float *f = a.flow_in + (size_t)b * 2 * a.d.plane + (size_t)y * a.d.pitch + x;
        dx = __ldg(f); dy = __ldg(f + a.d.plane);
        return;
    }
    if (!a.coarse) return;
    const float *cf = a.coarse + (size_t)b * 2 * a.cd.plane;
    const int x0 = __ldg(a.xi + x), x1 = min(x0 + 1, a.cd.w - 1);
    const int sy = __ldg(a.yi + y), y0 = clampi(sy, 0, a.cd.h - 1), y1 = clampi(sy + 1, 0, a.cd.h - 1); // rows clipped, fraction kept
    const float fx = __ldg(a.xf + x), gx = 1.f - fx, fy = __ldg(a.yf + y), gy = 1.f - fy;
    const float *r0 = cf + (size_t)y0 * a.cd.pitch, *r1 = cf + (size_t)y1 * a.cd.pitch;
    const float a00 = __ldg(r0 + x0), a01 = __ldg(r0 + x1), a10 = __ldg(r1 + x0), a11 = __ldg(r1 + x1);
    r0 += a.cd.plane; r1 += a.cd.plane;
    const float b00 = __ldg(r0 + x0), b01 = __ldg(r0 + x1), b10 = __ldg(r1 + x0), b11 = __ldg(r1 + x1);
    float t0 = a00 * gx + a01 * fx, t1 = a10 * gx + a11 * fx;
    dx = (t0 * gy + t1 * fy) * a.inv_scale;
    t0 = b00 * gx + b01 * fx; t1 = b10 * gx + b11 * fx;
    dy = (t0 * gy + t1 * fy) * a.inv_scale;
}

template <int PITCH>
__global__ void __launch_bounds__(256, 6) first_update_kernel(FirstUpdateArgs a)
{
    // one pixel per thread and <= 42 registers: 48 warps / SM keep enough loads in flight for this HBM-latency-bound
    // kernel (measured: two pixels per thread at 78 registers was 15 % slower).
    if (PITCH) { a.d.pitch = PITCH; a.cd.pitch = PITCH; } // compile-time row pitch: the 4 bilinear neighbours become load immediates
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    const int b = blockIdx.z;
    // The R1 gather can only be addressed after the table and coarse-flow loads (two dependent latencies): start the
    // DRAM -> L2 transfer of this warp's R0 / R1 row segments now (lanes 0..9 = image x channel).
    if (a.M && threadIdx.x < 10 && y < a.d.h) {
        const float *Rb = a.R + (size_t)b * 10 * a.d.plane + (size_t)(threadIdx.x / 5) * 5 * a.d.plane;
        const int xs = min((int)blockIdx.x * 32, a.d.w - 1);
        asm volatile("prefetch.global.L2 [%0];" ::"l"(Rb + ((size_t)y * 5 + threadIdx.x % 5) * a.d.pitch + xs));
    }
    if (x >= a.d.w || y >= a.d.h) return;
    float dx, dy;
    upsample_flow_px(a, b, x, y, dx, dy);
    if (a.flow_out) {
        float *f = a.flow_out + (size_t)b * 2 * a.d.plane + (size_t)y * a.d.pitch + x;
        f[0] = dx; f[a.d.plane] = dy;
    }
    if (a.M) {
        const float *R0 = a.R + (size_t)b * 10 * a.d.plane, *R1 = R0 + 5 * a.d.plane;
        float m[5];
        update_matrices_px(R0, R1, a.d.pitch, a.d.w, a.d.h, x, y, dx, dy, m);
        store_M(a.M + (size_t)b * 5 * a.d.plane, a.d.pitch, y, x, m);
    }
}

cudaError_t launch_first_update(cudaStream_t s, const FirstUpdateArgs &a)
{
    dim3 grid((a.d.w + 31) / 32, (a.d.h + 7) / 8, a.batch);
    // the compile-time pitch stands for both levels: only when the coarse flow has the same row pitch ("tight_pitch" gives
    // every level its own, e.g. 2048 over 1024)
    const bool one_pitch = !a.coarse || a.cd.pitch == a.d.pitch;
    if (one_pitch && a.d.pitch == 2048) first_update_kernel<2048><<<grid, dim3(32, 8), 0, s>>>(a);
    else if (one_pitch && a.d.pitch == 4096) first_update_kernel<4096><<<grid, dim3(32, 8), 0, s>>>(a);
    else first_update_kernel<0><<<grid, dim3(32, 8), 0, s>>>(a);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// K4/K5 (generic radius)  Gaussian window blur (A.5) of the five M planes, 2x2 solve in double, then either
//     the next update-matrices (A.4) or, on the last iteration, the flow write.  One block = 64x16 tile;
//     per channel: vertical pass (global -> shared), horizontal pass (shared -> registers).
// ------------------------------------------------------------------------------------------------
constexpr int GI_TW = 64, GI_TH = 16;

__global__ void __launch_bounds__(256) gauss_iter_generic_kernel(IterArgs a, WinTaps t)
{
    extern __shared__ float gi_smem[];
    const int m = t.m, SWD = GI_TW + 2 * m;
    const int x0 = blockIdx.x * GI_TW, y0 = blockIdx.y * GI_TH, b = blockIdx.z;
    const int w = a.d.w, h = a.d.h, pitch = a.d.pitch;
    const size_t plane = a.d.plane;
    const float *Min = a.Min + (size_t)b * 5 * plane;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    float acc[5][4];
    for (int c = 0; c < 5; c++) {
        int es;
        const float *Mc = M_channel(Min, pitch, c, es);
        const size_t rs = (size_t)5 * pitch;
        for (int i = threadIdx.x; i < SWD * GI_TH; i += blockDim.x) {
            int row = i / SWD, col = i - row * SWD;
            int gy = y0 + row;
            if (gy >= h) continue;
            int gx = clampi(x0 - m + col, 0, w - 1) * es;
            float v = Mc[gy * rs + gx] * t.k[0];
            if (a.fma == 2) {
                for (int k = 1; k <= m; k++) { v = fmaf(Mc[max(gy - k, 0) * rs + gx], t.k[k], v); v = fmaf(Mc[min(gy + k, h - 1) * rs + gx], t.k[k], v); }
            } else {
                for (int k = 1; k <= m; k++) v = v + (Mc[min(gy + k, h - 1) * rs + gx] + Mc[max(gy - k, 0) * rs + gx]) * t.k[k];
            }
            gi_smem[i] = v;
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 4; j++) {
            int col = tx + 32 * (j & 1), row = ty + 8 * (j >> 1);
            const float *p = gi_smem + row * SWD + col + m;
            float v = p[0] * t.k[0];
            if (a.fma == 2) {
                for (int k = 1; k <= m; k++) { v = fmaf(t.k[k], p[-k], v); v = fmaf(t.k[k], p[k], v); }
            } else {
                for (int k = 1; k <= m; k++) v = v + t.k[k] * (p[-k] + p[k]);
            }
            acc[c][j] = v;
        }
        __syncthreads();
    }
    const float *R0 = a.R + (size_t)b * 10 * plane, *R1 = R0 + 5 * plane;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        int x = x0 + tx + 32 * (j & 1), y = y0 + ty + 8 * (j >> 1);
        if (x >= w || y >= h) continue;
        float fx, fy;
        solve2x2(acc[0][j], acc[1][j], acc[2][j], acc[3][j], acc[4][j], fx, fy);
        size_t o = (size_t)y * pitch + x;
        if (a.last) {
            float *f = a.flow + (size_t)b * 2 * plane;
            f[o] = fx; f[o + plane] = fy;
        } else {
            float mm[5];
            update_matrices_px(R0, R1, pitch, w, h, x, y, fx, fy, mm);
            store_M(a.Mout + (size_t)b * 5 * plane, pitch, y, x, mm);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K4/K5 (window radius MR = 15 or 7)  register-blocked Gaussian window blur + solve + update.
//   tile 96 x 32 outputs, 256 threads, 2 CTAs / SM.
//   phase V: vertical tap sums of the tile's 128 columns (coalesced global loads, row / column replicate = clamped
//            addresses) -> shared
//   phase H: lane = row, warp = 12-column segment, 3 groups of 4 pixels x 5 channels; 2x2 solve in double;
//            flow -> shared Fb[2][32][97]
//   phase U: lane = x (coalesced): next update-matrices (A.4) or, last iteration, the flow write.
// FMA = 0 keeps the oracle's add-mul-add tap order bit for bit; FMA = 2 is the validated relaxation, the direct-form fmaf
// taps (oracle relax bit 7; SURVEY App. B.5).
// ------------------------------------------------------------------------------------------------
constexpr int GK_TW = 96, GK_TH = 32, GK_FP = 97;

#ifdef TW_TIMELINE // development builds only (tools/timeline.py): per-CTA phase timestamps of the level-0 window kernel
__device__ unsigned long long g_timeline[16384 * 24];
__device__ int g_tl_on;
__device__ int g_dev_flags; // experiments: 1 = no R prefetch, 2 = no M prefetch, 4 = R prefetch at the start of phase H, 8 = no U sub-stamps
#define TW_TL_BEGIN(on) if (threadIdx.x == 0) g_tl_on = (on);
#define TW_TL(slot)                                                                                              \
    if (threadIdx.x == 0 && g_tl_on) {                                                                           \
        const unsigned lin_ = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);                    \
        if (lin_ < 16384) {                                                                                      \
            unsigned long long c_;                                                                               \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(c_));                                               \
            g_timeline[lin_ * 24 + (slot)] = c_;                                                                 \
            if ((slot) == 0) { unsigned sm_; asm volatile("mov.u32 %0, %%smid;" : "=r"(sm_)); g_timeline[lin_ * 24 + 23] = sm_; } \
        }                                                                                                        \
    }
#define TW_TL_DEP(slot, dep)                                                                                     \
    { float d_ = (dep); asm volatile("" ::"f"(d_) : "memory"); }                                                 \
    TW_TL(slot)
#define TW_DEV_FLAG(bit) (g_dev_flags & (bit))
#else
#define TW_TL_BEGIN(on)
#define TW_TL(slot)
#define TW_TL_DEP(slot, dep)
#define TW_DEV_FLAG(bit) 0
#endif

// Per-pixel path of phase U for one thread's run of 4 vertically adjacent pixels (motion boundaries, frame borders,
// partial tiles): two pixels' 2 x 25 loads in flight at a time.  Kept out of line so that its registers do not
// weigh on the shared-row path.
__device__ __noinline__ void upd_run_slow(const float *__restrict__ R0, const float *__restrict__ R1, float *__restrict__ M,
                                          const float *__restrict__ Fb, int pitch, int w, int h, int x, int yb, int rowb, int col)
{
#pragma unroll
    for (int hf = 0; hf < 4; hf += 2) {
        UpdLoad L[2];
        bool ok[2];
        float fxs[2], fys[2];
#pragma unroll
        for (int u = 0; u < 2; u++) {
            ok[u] = x < w && yb + hf + u < h;
            fxs[u] = Fb[(rowb + hf + u) * GK_FP + col]; fys[u] = Fb[(GK_TH + rowb + hf + u) * GK_FP + col];
            if (ok[u]) upd_load(R0, R1, pitch, w, h, x, yb + hf + u, fxs[u], fys[u], L[u]);
        }
#pragma unroll
        for (int u = 0; u < 2; u++) {
            if (!ok[u]) continue;
            float mm[5];
            upd_compute(L[u], w, h, x, yb + hf + u, fxs[u], fys[u], mm);
            store_M(M, pitch, yb + hf + u, x, mm);
        }
    }
}

// phase U of K4/K5: lane = x, coalesced.  Last iteration: write the flow tile; otherwise the next update-matrices.
__device__ __forceinline__ void gauss_epilogue(const IterArgs &a, const float *__restrict__ Fb, int tid, int x0, int y0, int b, int pitch)
{
    const int w = a.d.w, h = a.d.h;
    const size_t plane = a.d.plane;
    if (a.last) {
        float *f = a.flow + (size_t)b * 2 * plane;
#pragma unroll 4
        for (int i = tid; i < GK_TW * GK_TH; i += 256) {
            const int row = i / GK_TW, col = i - row * GK_TW;
            const int x = x0 + col, y = y0 + row;
            if (x >= w || y >= h) continue;
            const size_t o = (size_t)y * pitch + x;
            f[o] = Fb[row * GK_FP + col];
            f[o + plane] = Fb[(GK_TH + row) * GK_FP + col];
        }
        if (a.span > 0) {
            // sample points of this tile: multiples of span in [x0, x0+96) x [y0, y0+32); one per thread
            const int sx0 = (x0 + a.span - 1) / a.span, sy0 = (y0 + a.span - 1) / a.span;
            const int nsx = max(0, (min(x0 + GK_TW, w) - 1) / a.span - sx0 + 1), nsy = max(0, (min(y0 + GK_TH, h) - 1) / a.span - sy0 + 1);
            int hit = 0;
            for (int i = tid; i < nsx * nsy; i += 256) { // block-uniform trip count (<= 1 for span >= 4)
                const int j = i / nsx, col = (sx0 + i - j * nsx) * a.span - x0, row = (sy0 + j) * a.span - y0;
                const float dx = Fb[row * GK_FP + col], dy = Fb[(GK_TH + row) * GK_FP + col];
                const float len = (dx * dx) + (dy * dy);
                hit += ((double)len > a.thr2) ? 1 : 0;
            }
            if (nsx * nsy > 0) {
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) hit += __shfl_xor_sync(0xffffffffu, hit, off);
                if ((tid & 31) == 0 && hit > 0) atomicAdd(a.counts + b, hit);
            }
        }
        return;
    }
    const float *R0 = a.R + (size_t)b * 10 * plane, *R1 = R0 + 5 * plane;
    float *M = a.Mout + (size_t)b * 5 * plane;
    // 12 pixels per thread: warp = 4 consecutive rows, lane = column of a 32-column chunk, 3 chunks.  A thread's 4
    // vertically adjacent pixels usually gather from 5 consecutive R1 rows at one x1 (smooth flow): then the bottom
    // row of pixel u IS the top row of pixel u+1 and the warp takes the shared-row path -- 50 + 20 loads for 4 pixels
    // instead of 4 x 25, all in flight together, every address one base register + an immediate.  Any lane that does
    // not fit (motion boundary, frame border, partial tile) sends its warp through the per-pixel path; both paths load
    // the same values and run the same arithmetic.
    const int warp = tid >> 5, lane = tid & 31;
    const int rowb = 4 * warp;
#pragma unroll 1
    for (int k = 0; k < 3; k++) {
        const int col = lane + 32 * k, x = x0 + col;
        int yb = y0 + rowb;
        asm volatile("" : "+r"(yb)); // opaque per chunk: keeps the row-only subexpressions (border scales, float rows) out of registers across the loop
        // pass 1 (registers released before the loads): does every pixel of the run gather at (X1, Y1 + u)?
        bool fast;
        int X1, Y1;
        {
            int x1[4], y1[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const float px = (float)x + Fb[(rowb + u) * GK_FP + col], py = (float)(yb + u) + Fb[(GK_TH + rowb + u) * GK_FP + col];
                x1[u] = __float2int_rd(px); y1[u] = __float2int_rd(py);
            }
            X1 = x1[0]; Y1 = y1[0];
            // (also: no pixel of the run in the 5-pixel damped frame border, which implies x < w and yb + 3 < h)
            fast = (unsigned)(x - 5) < (unsigned)(w - 10) && yb >= 5 && yb + 3 < h - 5 && (unsigned)X1 < (unsigned)(w - 1) && Y1 >= 0 &&
                   Y1 + 4 < h && x1[1] == X1 && x1[2] == X1 && x1[3] == X1 && y1[1] == Y1 + 1 && y1[2] == Y1 + 2 && y1[3] == Y1 + 3;
        }
        if (__all_sync(0xffffffffu, fast)) {
            if (!TW_DEV_FLAG(8)) { TW_TL(8 + 4 * k) } // after the vote
            float q[4][5], rr[5][5][2];
            const float *q0 = R0 + (size_t)yb * 5 * pitch + x;
            const float *p = R1 + (size_t)Y1 * 5 * pitch + X1;
#pragma unroll
            for (int r = 0; r < 5; r++)
#pragma unroll
                for (int c = 0; c < 5; c++) { rr[r][c][0] = __ldg(p + (r * 5 + c) * pitch); rr[r][c][1] = __ldg(p + (r * 5 + c) * pitch + 1); }
#pragma unroll
            for (int u = 0; u < 4; u++)
#pragma unroll
                for (int c = 0; c < 5; c++) q[u][c] = __ldg(q0 + (u * 5 + c) * pitch);
            // the flow is re-read from shared memory (through an opaque index, so that the values of pass 1 are not
            // kept in registers under the 70 loads); x1 = X1 and y1 = Y1 + u here, hence the same fractions as pass 1
            if (!TW_DEV_FLAG(8)) { TW_TL_DEP(9 + 4 * k, q[3][4] + rr[4][4][1] + rr[0][0][0]) } // last-issued and first-issued loads have arrived
            int col2 = col;
            asm volatile("" : "+r"(col2));
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const float fxu = Fb[(rowb + u) * GK_FP + col2], fyu = Fb[(GK_TH + rowb + u) * GK_FP + col2];
                const float px = (float)x + fxu, py = (float)(yb + u) + fyu;
                float mm[5];
                upd_core<false>(q[u], rr[u], rr[u + 1], true, px - (float)X1, py - (float)(Y1 + u), w, h, x, yb + u, fxu, fyu, mm);
                store_M(M, pitch, yb + u, x, mm);
                asm volatile("" ::: "memory"); // one pixel at a time: interleaving the four pixels' arithmetic costs more registers than there are
            }
        } else {
            upd_run_slow(R0, R1, M, Fb, pitch, w, h, x, yb, rowb, col);
        }
        TW_TL(4 + k)
    }
}


// ------------------------------------------------------------------------------------------------
// K4/K5 gauss_iter2_kernel: the tap sums are issued as PACKED f32x2 instructions (FADD2 / FMUL2 / FFMA2, sm_100+).
// Each half of a packed op is an independent IEEE-754 op, so the result stays bit-identical to the oracle's scalar
// add-mul-add order while the FP32 instruction count halves (measured, tools/ubench2.cu: the faithful tap runs 1.41x
// faster packed than scalar).
//   Packing: phase V pairs the CHANNELS (G11,G12) and (G22,h1) of one pixel column, and for h2 two adjacent
//   columns; phase H reads them back as float2 (pitch 130 float2 = conflict-free LDS.128 with lane = row) and
//   pairs h2 over adjacent pixels.  Shared: P01[32][130] float2, P23[32][130] float2, P4[32][132] float, flow tile.
// ------------------------------------------------------------------------------------------------
constexpr int G2_P2 = 130, G2_P4 = 132, G2_RV = 8;
constexpr size_t G2_SMEM = sizeof(float) * (2 * GK_TH * G2_P2 * 2 + GK_TH * G2_P4 + 2 * GK_TH * GK_FP);

template <int MR, int FMA, bool INTERIOR, bool CPITCH>
__device__ __forceinline__ void gauss_v_item2(const float2 *__restrict__ src, int rstride /* float2 per row */, float2 *__restrict__ dst,
                                              int dstride, int ybase, int h, const WinTaps &t)
{
    constexpr int NIN = G2_RV + 2 * MR;
    const float2 one2 = make_float2(t.one, t.one);
    float2 in[NIN];
    // one IMAD.WIDE.U32 per load: byte offset = (32-bit row stride in bytes) * (row), added to a 64-bit base
    const unsigned rsb = (unsigned)rstride * 8u;
    const char *base = reinterpret_cast<const char *>(src);
    if (INTERIOR) {
        base = row_ptr(base, rsb, (unsigned)ybase);
#pragma unroll
        for (int r = 0; r < NIN; r++) {
            if (CPITCH) in[r] = __ldg(reinterpret_cast<const float2 *>(base) + (size_t)r * rstride); // rstride is a constant: immediate offset
            else in[r] = __ldg(reinterpret_cast<const float2 *>(row_ptr(base, rsb, (unsigned)r)));
        }
    } else {
#pragma unroll
        for (int r = 0; r < NIN; r++)
            in[r] = __ldg(reinterpret_cast<const float2 *>(row_ptr(base, rsb, (unsigned)clampi(ybase + r, 0, h - 1))));
    }
    // taps outer, outputs inner: 8 independent accumulator chains are interleaved explicitly
    float2 v[G2_RV];
#pragma unroll
    for (int o = 0; o < G2_RV; o++) v[o] = tw_mul2(in[o + MR], make_float2(t.k[0], t.k[0]));
#pragma unroll
    for (int i = 1; i <= MR; i++) {
        const float2 kk = make_float2(t.k[i], t.k[i]);
        if (FMA == 2) { // direct form (oracle relax bit 7): upper tap first; no add -> fma dependency
#pragma unroll
            for (int o = 0; o < G2_RV; o++) v[o] = tw_fma2(in[o + MR - i], kk, v[o]);
#pragma unroll
            for (int o = 0; o < G2_RV; o++) v[o] = tw_fma2(in[o + MR + i], kk, v[o]);
        } else {
#pragma unroll
            for (int o = 0; o < G2_RV; o++) {
                const float2 sum = tw_add2(in[o + MR + i], in[o + MR - i]);
                v[o] = tw_fma2(tw_mul2(sum, kk), one2, v[o]); // = v + round(sum * k): see tw_fma2 note
            }
        }
    }
#pragma unroll
    for (int o = 0; o < G2_RV; o++) dst[o * dstride] = v[o];
}

// Column walker: one thread owns one column of one channel pair for ALL rows of the tile.  The 8+2*MR-row register
// window slides down by 8 rows per group; the 8 new rows of the next group are requested BEFORE the current group's
// 8 x (1 + 3*MR) packed operations, so only the first window of a tile exposes load latency, and a tile column is
// read 32+2*MR times instead of 4 x (8+2*MR).
template <int MR, int FMA, bool INTERIOR, bool CPITCH, class PF>
__device__ __forceinline__ void gauss_v_walk2(const float2 *__restrict__ src, int rstride /* float2 per row */, float2 *__restrict__ dst,
                                              int dstride, int ybase, int h, const WinTaps &t, PF &&after_first_loads)
{
    constexpr int NIN = G2_RV + 2 * MR, NG = GK_TH / G2_RV;
    const float2 one2 = make_float2(t.one, t.one);
    const unsigned rsb = (unsigned)rstride * 8u;
    const char *base = reinterpret_cast<const char *>(src);
    if (INTERIOR) base = row_ptr(base, rsb, (unsigned)ybase);
    auto ld = [&](int r) -> float2 {
        if (INTERIOR) {
            if (CPITCH) return __ldg(reinterpret_cast<const float2 *>(base) + (size_t)r * rstride);
            return __ldg(reinterpret_cast<const float2 *>(row_ptr(base, rsb, (unsigned)r)));
        }
        return __ldg(reinterpret_cast<const float2 *>(row_ptr(base, rsb, (unsigned)clampi(ybase + r, 0, h - 1))));
    };
    float2 win[NIN];
#pragma unroll
    for (int r = 0; r < NIN; r++) win[r] = ld(r);
    after_first_loads(); // the tile's L2 prefetches are issued under the latency of the first window
#pragma unroll
    for (int g = 0; g < NG; g++) {
        float2 nxt[G2_RV];
        if (g + 1 < NG) {
#pragma unroll
            for (int r = 0; r < G2_RV; r++) nxt[r] = ld(NIN + G2_RV * g + r);
        }
        float2 v[G2_RV];
#pragma unroll
        for (int o = 0; o < G2_RV; o++) v[o] = tw_mul2(win[o + MR], make_float2(t.k[0], t.k[0]));
#pragma unroll
        for (int i = 1; i <= MR; i++) {
            const float2 kk = make_float2(t.k[i], t.k[i]);
            if (FMA == 2) {
#pragma unroll
                for (int o = 0; o < G2_RV; o++) v[o] = tw_fma2(win[o + MR - i], kk, v[o]);
#pragma unroll
                for (int o = 0; o < G2_RV; o++) v[o] = tw_fma2(win[o + MR + i], kk, v[o]);
            } else {
#pragma unroll
                for (int o = 0; o < G2_RV; o++) {
                    const float2 sum = tw_add2(win[o + MR + i], win[o + MR - i]);
                    v[o] = tw_fma2(tw_mul2(sum, kk), one2, v[o]);
                }
            }
        }
#pragma unroll
        for (int o = 0; o < G2_RV; o++) dst[(G2_RV * g + o) * dstride] = v[o];
        if (g + 1 < NG) {
#pragma unroll
            for (int r = 0; r < NIN - G2_RV; r++) win[r] = win[r + G2_RV];
#pragma unroll
            for (int r = 0; r < G2_RV; r++) win[NIN - G2_RV + r] = nxt[r];
        }
    }
}

// 5 items per thread: (G11,G12) and (G22,h1) float2 planes at (column j, row groups g and g+2), then the h2 plane at
// (column pair jj, row group g) -- every item is "38 8-byte loads, 8 packed outputs".  Columns are replicated by
// clamping the address; the h2 column pair is clamped as a pair (x0 and w are even multiples of the tile / pitch
// except at the right edge, where both columns clamp to w-1 via the scalar fallback).
template <int MR, int FMA, bool INTERIOR, bool CPITCH, class PF>
__device__ __forceinline__ void gauss_v_phase2(const float *__restrict__ Min, float *__restrict__ sm, const WinTaps &t, int tid, int x0,
                                               int y0, int w, int h, int pitch, size_t plane, PF &&after_first_loads)
{
    float2 *P01 = reinterpret_cast<float2 *>(sm);
    float2 *P23 = P01 + GK_TH * G2_P2;
    float2 *P4 = P23 + GK_TH * G2_P2; // float2 view of the plain float plane (pitch 132 floats = 66 float2)
    {
        // 256 threads = 128 columns x 2 channel pairs, each walking the 32 rows of the tile
        const int pair = tid >> 7, j = tid & 127;
        const int gx = clampi(x0 - 16 + j, 0, w - 1);
        const float2 *src = reinterpret_cast<const float2 *>(Min + pair * 2 * pitch) + gx;
        float2 *dst = (pair ? P23 : P01) + j;
        gauss_v_walk2<MR, FMA, INTERIOR, CPITCH>(src, 5 * pitch / 2, dst, G2_P2, y0 - MR, h, t, after_first_loads);
    }
    TW_TL(1)
    {
        const int jj = tid & 63, g = tid >> 6;
        const int xa = x0 - 16 + 2 * jj;
        float2 *dst = P4 + g * G2_RV * (G2_P4 / 2) + jj;
        const float *P = Min + 4 * pitch;
        if (xa >= 0 && xa + 1 <= w - 1) {
            gauss_v_item2<MR, FMA, INTERIOR, CPITCH>(reinterpret_cast<const float2 *>(P + xa), 5 * pitch / 2, dst, G2_P4 / 2, y0 + g * G2_RV - MR, h, t);
        } else { // edge column pair: clamp each column separately (scalar loads)
            const int ca = clampi(xa, 0, w - 1), cb = clampi(xa + 1, 0, w - 1), ybase = y0 + g * G2_RV - MR;
            constexpr int NIN = G2_RV + 2 * MR;
            const float2 one2 = make_float2(t.one, t.one);
            float2 in[NIN];
#pragma unroll
            for (int r = 0; r < NIN; r++) {
                const size_t o = (size_t)clampi(ybase + r, 0, h - 1) * 5 * pitch;
                in[r] = make_float2(__ldg(P + o + ca), __ldg(P + o + cb));
            }
#pragma unroll
            for (int o = 0; o < G2_RV; o++) {
                float2 v = tw_mul2(in[o + MR], make_float2(t.k[0], t.k[0]));
#pragma unroll
                for (int i = 1; i <= MR; i++) {
                    const float2 sum = tw_add2(in[o + MR + i], in[o + MR - i]);
                    const float2 kk = make_float2(t.k[i], t.k[i]);
                    if (FMA == 2) v = tw_fma2(in[o + MR + i], kk, tw_fma2(in[o + MR - i], kk, v));
                    else v = tw_fma2(tw_mul2(sum, kk), one2, v);
                }
                dst[o * (G2_P4 / 2)] = v;
            }
        }
    }
}

// PITCH > 0: the row pitch is a compile-time constant (the plan pads every level to 2048 or 4096 floats), so the
// unrolled row addresses become LDG immediates instead of 3-4 integer instructions per load.

template <int MR, int FMA, int PITCH>
__global__ void __launch_bounds__(256, 2) gauss_iter2_kernel(IterArgs a, WinTaps t)
{
    extern __shared__ __align__(16) float gk_smem[];
    float *Fb = gk_smem + 2 * GK_TH * G2_P2 * 2 + GK_TH * G2_P4;
    const int tid = threadIdx.x, lane = tid & 31;
    const int x0 = blockIdx.x * GK_TW, y0 = blockIdx.y * GK_TH, b = blockIdx.z;
    const int w = a.d.w, h = a.d.h, pitch = PITCH ? PITCH : a.d.pitch;
    const size_t plane = a.d.plane;
    const float *Min = a.Min + (size_t)b * 5 * plane;

    // Every V item starts with a burst of loads whose latency is exposed (registers leave no room for double
    // buffering).  The walker's first window goes to DRAM directly; UNDER that latency every thread then issues its share
    // of L2 prefetches for the rest of the tile -- the M rows below the first window and the h2 plane (so that the later
    // window refills and the h2 item see L2 latency) and the epilogue's R0 / R1 lines.
    // (shift-only index arithmetic: this runs while the co-resident CTA saturates the FMA pipe, which also executes IMAD
    // -- the divisions of a flat index cost 7 % of a CTA's lifetime in the first version)
    auto prefetch_R = [&]() {
        const float *Rb = a.R + (size_t)b * 10 * plane;
        const int row = tid >> 3, u = tid & 7; // 32 rows x 8 threads; 30 lines per row (10 planes x 3 segments)
        const int y = min(y0 + row, h - 1);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int idx = u + 8 * j;
            if (idx < 30) {
                const int pl = (idx * 11) >> 5, seg = idx - pl * 3; // idx / 3 for idx < 32
                const int x = min(x0 + seg * 32, w - 1);
                asm volatile("prefetch.global.L2 [%0];" ::"l"(Rb + (size_t)(pl >= 5) * 5 * plane + ((size_t)y * 5 + (pl >= 5 ? pl - 5 : pl)) * pitch + x));
            }
        }
    };
    auto prefetch_tile = [&]() {
        if (!TW_DEV_FLAG(2)) {
            constexpr int NR = GK_TH + 2 * MR; // rows; per row 20 x 128-byte lines: 8 + 8 (float2 planes) + 4 (float plane)
            constexpr int NW = G2_RV + 2 * MR; // rows of the walkers' first window: their float2 planes are loaded, not prefetched
            const int xl = max(x0 - 16, 0);
            const int row = tid >> 2, q = tid & 3; // 64 row slots x 4 threads, 5 lines each
            if (row < NR) {
                const float *rowp = Min + (size_t)clampi(y0 - MR + row, 0, h - 1) * 5 * pitch;
#pragma unroll
                for (int j = 0; j < 5; j++) {
                    const int seg = q * 5 + j;
                    const float *p;
                    if (seg < 16) p = rowp + (seg >> 3) * 2 * pitch + min(xl + (seg & 7) * 16, w - 1) * 2;
                    else p = rowp + 4 * pitch + min(xl + (seg - 16) * 32, w - 1);
                    if (seg >= 16 || row >= NW) asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
                }
            }
        }
        if (!a.last && !TW_DEV_FLAG(1) && !TW_DEV_FLAG(4)) prefetch_R();
    };

    TW_TL_BEGIN(gridDim.x == 20 && !a.last)
    TW_TL(0)
    // ---- phase V (packed) ----
    if ((y0 - MR >= 0) && (y0 + GK_TH + MR - 1 <= h - 1))
        gauss_v_phase2<MR, FMA, true, (PITCH > 0)>(Min, gk_smem, t, tid, x0, y0, w, h, pitch, plane, prefetch_tile);
    else
        gauss_v_phase2<MR, FMA, false, (PITCH > 0)>(Min, gk_smem, t, tid, x0, y0, w, h, pitch, plane, prefetch_tile);
    __syncthreads();
    TW_TL(2)
    if (!a.last && TW_DEV_FLAG(4)) prefetch_R();

    // ---- phase H (packed) + solve ----
    {
        const float2 *P01 = reinterpret_cast<const float2 *>(gk_smem);
        const float2 *P23 = P01 + GK_TH * G2_P2;
        const float *P4 = gk_smem + 2 * GK_TH * G2_P2 * 2;
        const int seg = tid >> 5;
        constexpr int LO = (16 - MR) & ~3;
        constexpr int NV = ((3 + 16 + MR) | 3) + 1 - LO;
        const float2 one2 = make_float2(t.one, t.one);
#pragma unroll 1
        for (int grp = 0; grp < 3; grp++) {
            const int cbase = seg * 12 + grp * 4;
            float2 r01[4], r23[4];
            float r4[4];
#pragma unroll
            for (int pr = 0; pr < 2; pr++) {
                const float4 *src = reinterpret_cast<const float4 *>((pr ? P23 : P01) + lane * G2_P2 + cbase + LO);
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
                const float4 *src = reinterpret_cast<const float4 *>(P4 + lane * G2_P4 + cbase + LO);
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
            for (int p = 0; p < 4; p++) {
                float fx, fy;
                solve2x2(r01[p].x, r01[p].y, r23[p].x, r23[p].y, r4[p], fx, fy);
                Fb[lane * GK_FP + cbase + p] = fx;
                Fb[(GK_TH + lane) * GK_FP + cbase + p] = fy;
            }
        }
    }
    __syncthreads();
    TW_TL(3)
    // (Tried and measured slower, 2.73 vs 2.33 ms per step: staging the tile's R1 gather window -- 5 x 39 x 104 floats centred
    // on the tile's mean flow -- in the 83 KB the dead planes leave, with 16-byte coalesced loads and the corners read by
    // LDS.  The extra barrier and the exposed window load cost more than the gathers save, because phase U is paced by
    // the co-resident CTA's hold on the FMA pipe / issue slots rather than by its own loads; DESIGN.md 4.1.)
    gauss_epilogue(a, Fb, tid, x0, y0, b, pitch);
#ifdef TW_TIMELINE
    __syncthreads();
#endif
    TW_TL(7)
}

template <int MR, int FMA, int PITCH>
static cudaError_t launch_gauss_fast2p(cudaStream_t s, const IterArgs &a, const WinTaps &t)
{
    static std::atomic<bool> configured_dev[kMaxDevices];
    std::atomic<bool> &configured = configured_dev[current_device()];
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(gauss_iter2_kernel<MR, FMA, PITCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G2_SMEM);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    dim3 grid((a.d.w + GK_TW - 1) / GK_TW, (a.d.h + GK_TH - 1) / GK_TH, a.batch);
    gauss_iter2_kernel<MR, FMA, PITCH><<<grid, 256, G2_SMEM, s>>>(a, t);
    return cudaGetLastError();
}

template <int MR, int FMA>
static cudaError_t launch_gauss_fast2(cudaStream_t s, const IterArgs &a, const WinTaps &t)
{
    if (a.d.pitch == 2048) return launch_gauss_fast2p<MR, FMA, 2048>(s, a, t);
    if (a.d.pitch == 4096) return launch_gauss_fast2p<MR, FMA, 4096>(s, a, t);
    return launch_gauss_fast2p<MR, FMA, 0>(s, a, t);
}

// The two arithmetics of the library: faithful (IterArgs::fma = 0) and relaxed = direct form (2).
template <int MR>
static cudaError_t launch_gauss_mr(cudaStream_t s, const IterArgs &a, const WinTaps &t)
{
#ifdef TW_DEV_ONE // development builds: one instantiation only (fast compile while tuning the kernel)
    if (MR == 15 && a.d.pitch == 2048 && a.fma == 2) return launch_gauss_fast2p<15, 2, 2048>(s, a, t);
    return cudaErrorNotSupported;
#else
    if (a.fma == 2) return launch_gauss_fast2<MR, 2>(s, a, t);
    return launch_gauss_fast2<MR, 0>(s, a, t);
#endif
}

cudaError_t launch_gauss_iter(cudaStream_t s, const IterArgs &a, const WinTaps &t)
{
    if (t.m == 15) return launch_gauss_mr<15>(s, a, t);
    if (t.m == 7) return launch_gauss_mr<7>(s, a, t);
    dim3 grid((a.d.w + GI_TW - 1) / GI_TW, (a.d.h + GI_TH - 1) / GI_TH, a.batch);
    size_t smem = sizeof(float) * GI_TH * (GI_TW + 2 * t.m);
    gauss_iter_generic_kernel<<<grid, 256, smem, s>>>(a, t);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// K5s  LAST iteration of the FINEST scale when only the classification is wanted (the dispatcher path: the reference's
//      Response carries the sampled vectors, never the dense field -- src/consumer.cpp:59-88, src/message_queue.h:27-40).
//      The window blur + 2x2 solve are evaluated only where src/consumer.cpp:60-77 samples the flow: rows y = j * span get
//      the vertical pass at every column, the horizontal pass + solve run at the columns x = i * span only.  Same operand
//      order as the dense kernels in each arithmetic (IterArgs::fma), so the sampled (dx, dy) -- written at their positions
//      of the flow planes, where sample_kernel picks them up -- are bit-identical to the dense path; the rest of the planes
//      is NOT produced (tw_batch_flow refuses after such a run).  FP work drops ~16x; what remains is one pass over M.
//      One CTA = one sampled row x (256 - 2m) columns; thread = column (all five channels, 2m + 1 rows in registers' reach);
//      then (sample, channel) threads walk the taps in the oracle's order; then one thread per sample solves and tests.
// ------------------------------------------------------------------------------------------------
constexpr int SP_THREADS = 256, SP_MAXS = 64; // SP_MAXS: most samples one CTA can own (span >= 4 with m = 0 .. )

__global__ void __launch_bounds__(SP_THREADS) gauss_last_sparse_kernel(IterArgs a, WinTaps t)
{
    __shared__ float sv[5][SP_THREADS];
    __shared__ float sb[SP_MAXS][5];
    const int m = t.m, tw_cols = SP_THREADS - 2 * m;
    const int tid = threadIdx.x, b = blockIdx.z;
    const int x0 = blockIdx.x * tw_cols, y = blockIdx.y * a.span;
    const int w = a.d.w, h = a.d.h, pitch = a.d.pitch;
    const float *Min = a.Min + (size_t)b * 5 * a.d.plane;
    // ---- vertical pass at row y, column gx (replicated past the frame like App. A.5) ----
    {
        const int gx = clampi(x0 - m + tid, 0, w - 1);
        const size_t rs = (size_t)5 * pitch;
        const float *c01 = Min + 2 * gx, *c23 = Min + 2 * pitch + 2 * gx, *c4 = Min + 4 * pitch + gx;
        float v[5];
        {
            const float2 p = __ldg(reinterpret_cast<const float2 *>(c01 + y * rs)), q = __ldg(reinterpret_cast<const float2 *>(c23 + y * rs));
            const float r = __ldg(c4 + y * rs), k0 = t.k[0];
            v[0] = __fmul_rn(p.x, k0); v[1] = __fmul_rn(p.y, k0); v[2] = __fmul_rn(q.x, k0); v[3] = __fmul_rn(q.y, k0); v[4] = __fmul_rn(r, k0);
        }
#pragma unroll 5
        for (int i = 1; i <= m; i++) {
            const size_t od = (size_t)min(y + i, h - 1) * rs, ou = (size_t)max(y - i, 0) * rs;
            const float2 pd = __ldg(reinterpret_cast<const float2 *>(c01 + od)), pu = __ldg(reinterpret_cast<const float2 *>(c01 + ou));
            const float2 qd = __ldg(reinterpret_cast<const float2 *>(c23 + od)), qu = __ldg(reinterpret_cast<const float2 *>(c23 + ou));
            const float rd = __ldg(c4 + od), ru = __ldg(c4 + ou), k = t.k[i];
            const float dn[5] = {pd.x, pd.y, qd.x, qd.y, rd}, up[5] = {pu.x, pu.y, qu.x, qu.y, ru};
#pragma unroll
            for (int c = 0; c < 5; c++) {
                if (a.fma == 2) { v[c] = fmaf(up[c], k, v[c]); v[c] = fmaf(dn[c], k, v[c]); }
                else v[c] = __fadd_rn(v[c], __fmul_rn(__fadd_rn(dn[c], up[c]), k));
            }
        }
#pragma unroll
        for (int c = 0; c < 5; c++) sv[c][tid] = v[c];
    }
    __syncthreads();
    // ---- horizontal pass at the sampled columns of this CTA: x = i * span in [x0, min(x0 + tw_cols, w)) ----
    const int s0 = (x0 + a.span - 1) / a.span;
    const int ns = max(0, (min(x0 + tw_cols, w) - 1) / a.span - s0 + 1);
    for (int idx = tid; idx < ns * 5; idx += SP_THREADS) {
        const int s = idx / 5, c = idx - s * 5;
        const float *p = &sv[c][(s0 + s) * a.span - x0 + m];
        float r = __fmul_rn(p[0], t.k[0]);
        for (int i = 1; i <= m; i++) {
            const float k = t.k[i];
            if (a.fma == 2) { r = fmaf(k, p[-i], r); r = fmaf(k, p[i], r); }
            else r = __fadd_rn(r, __fmul_rn(k, __fadd_rn(p[-i], p[i])));
        }
        sb[s][c] = r;
    }
    __syncthreads();
    int hit = 0;
    if (tid < ns) {
        float fx, fy;
        solve2x2(sb[tid][0], sb[tid][1], sb[tid][2], sb[tid][3], sb[tid][4], fx, fy);
        const int x = (s0 + tid) * a.span;
        float *f = a.flow + (size_t)b * 2 * a.d.plane + (size_t)y * pitch + x;
        f[0] = fx; f[a.d.plane] = fy;
        const float len = __fadd_rn(__fmul_rn(fx, fx), __fmul_rn(fy, fy));
        hit = ((double)len > a.thr2) ? 1 : 0;
    }
    if (tid < 64) { // ns <= SP_MAXS = 64: two warps cover every sample
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) hit += __shfl_xor_sync(0xffffffffu, hit, off);
        if ((tid & 31) == 0 && hit > 0) atomicAdd(a.counts + b, hit);
    }
}

// K5s for the default geometry (window radius 15, span 10): one CTA = THREE consecutive sampled rows.  Their 31-row windows
// overlap by 21 rows, so a thread reads the 51 rows y0 - 15 .. y0 + 35 of its column ONCE into registers (one channel pair at
// a time) and forms the three vertical sums from them -- 17 rows per output instead of 31 through L2 / L1, the quantity the
// one-row kernel is bound by.  Tap order per output unchanged, so the results are the same bits.
constexpr int SP3_R = 3, SP3_M = 15, SP3_SPAN = 10, SP3_ROWS = 2 * SP3_M + 1 + SP3_SPAN * (SP3_R - 1);

template <int FMA> __device__ __forceinline__ float sp3_taps(const float (&win)[SP3_ROWS], const int c, const WinTaps &t)
{
    float v = __fmul_rn(win[c], t.k[0]);
#pragma unroll
    for (int i = 1; i <= SP3_M; i++) {
        const float k = t.k[i], dn = win[c + i], up = win[c - i];
        if (FMA == 2) { v = fmaf(up, k, v); v = fmaf(dn, k, v); }
        else v = __fadd_rn(v, __fmul_rn(__fadd_rn(dn, up), k));
    }
    return v;
}

template <int FMA> __global__ void __launch_bounds__(SP_THREADS, 2) gauss_last_sparse3_kernel(IterArgs a, WinTaps t)
{
    __shared__ float sv[SP3_R][5][SP_THREADS];
    __shared__ float sb[SP3_R][SP_MAXS][5];
    constexpr int m = SP3_M, tw_cols = SP_THREADS - 2 * m;
    const int tid = threadIdx.x, b = blockIdx.z;
    const int x0 = blockIdx.x * tw_cols, y0 = blockIdx.y * (SP3_R * SP3_SPAN);
    const int w = a.d.w, h = a.d.h, pitch = a.d.pitch;
    const float *Min = a.Min + (size_t)b * 5 * a.d.plane;
    {
        const int gx = clampi(x0 - m + tid, 0, w - 1);
        const size_t rs = (size_t)5 * pitch;
        const bool interior = y0 - m >= 0 && y0 - m + SP3_ROWS <= h; // CTA-uniform: no row of the window is replicated
        float wx[SP3_ROWS], wy[SP3_ROWS];
#pragma unroll
        for (int pr = 0; pr < 2; pr++) { // channel pairs (0, 1) and (2, 3): 8-byte loads
            const float *col = Min + (size_t)(2 * pr) * pitch + 2 * gx;
            if (interior) {
                const float *p = col + (size_t)(y0 - m) * rs;
#pragma unroll
                for (int r = 0; r < SP3_ROWS; r++) {
                    const float2 v = __ldg(reinterpret_cast<const float2 *>(p + r * rs));
                    wx[r] = v.x; wy[r] = v.y;
                }
            } else {
#pragma unroll
                for (int r = 0; r < SP3_ROWS; r++) {
                    const float2 v = __ldg(reinterpret_cast<const float2 *>(col + (size_t)clampi(y0 - m + r, 0, h - 1) * rs));
                    wx[r] = v.x; wy[r] = v.y;
                }
            }
#pragma unroll
            for (int j = 0; j < SP3_R; j++) {
                sv[j][2 * pr][tid] = sp3_taps<FMA>(wx, m + SP3_SPAN * j, t);
                sv[j][2 * pr + 1][tid] = sp3_taps<FMA>(wy, m + SP3_SPAN * j, t);
            }
        }
        {
            const float *col = Min + (size_t)4 * pitch + gx;
            if (interior) {
                const float *p = col + (size_t)(y0 - m) * rs;
#pragma unroll
                for (int r = 0; r < SP3_ROWS; r++) wx[r] = __ldg(p + r * rs);
            } else {
#pragma unroll
                for (int r = 0; r < SP3_ROWS; r++) wx[r] = __ldg(col + (size_t)clampi(y0 - m + r, 0, h - 1) * rs);
            }
#pragma unroll
            for (int j = 0; j < SP3_R; j++) sv[j][4][tid] = sp3_taps<FMA>(wx, m + SP3_SPAN * j, t);
        }
    }
    __syncthreads();
    // ---- horizontal pass at the sampled columns, for each of the (up to) three rows that exist ----
    const int s0 = (x0 + SP3_SPAN - 1) / SP3_SPAN;
    const int ns = max(0, (min(x0 + tw_cols, w) - 1) / SP3_SPAN - s0 + 1);
    const int nr = min(SP3_R, (h - 1 - y0) / SP3_SPAN + 1); // sampled rows y0 + 10 j < h
    for (int idx = tid; idx < nr * ns * 5; idx += SP_THREADS) {
        const int j = idx / (ns * 5), rem = idx - j * (ns * 5), s = rem / 5, c = rem - s * 5;
        const float *p = &sv[j][c][(s0 + s) * SP3_SPAN - x0 + m];
        float r = __fmul_rn(p[0], t.k[0]);
#pragma unroll
        for (int i = 1; i <= m; i++) {
            const float k = t.k[i];
            if (FMA == 2) { r = fmaf(k, p[-i], r); r = fmaf(k, p[i], r); }
            else r = __fadd_rn(r, __fmul_rn(k, __fadd_rn(p[-i], p[i])));
        }
        sb[j][s][c] = r;
    }
    __syncthreads();
    int hit = 0;
    if (tid < nr * ns) {
        const int j = tid / ns, s = tid - j * ns;
        float fx, fy;
        solve2x2(sb[j][s][0], sb[j][s][1], sb[j][s][2], sb[j][s][3], sb[j][s][4], fx, fy);
        const int x = (s0 + s) * SP3_SPAN, y = y0 + SP3_SPAN * j;
        float *f = a.flow + (size_t)b * 2 * a.d.plane + (size_t)y * pitch + x;
        f[0] = fx; f[a.d.plane] = fy;
        const float len = __fadd_rn(__fmul_rn(fx, fx), __fmul_rn(fy, fy));
        hit = ((double)len > a.thr2) ? 1 : 0;
    }
    if (tid < 96) { // nr * ns <= 3 * 23: three warps cover every sample
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) hit += __shfl_xor_sync(0xffffffffu, hit, off);
        if ((tid & 31) == 0 && hit > 0) atomicAdd(a.counts + b, hit);
    }
}

// Applicable when the samples of a CTA fit its table and the window fits the CTA: else the caller runs the dense kernel.
bool gauss_last_sparse_ok(const IterArgs &a, const WinTaps &t)
{
    if (a.span < 1 || t.m < 0 || 2 * t.m + 32 > SP_THREADS) return false;
    const int cols = SP_THREADS - 2 * t.m;
    return (cols + a.span - 1) / a.span + 1 <= SP_MAXS;
}

cudaError_t launch_gauss_last_sparse(cudaStream_t s, const IterArgs &a, const WinTaps &t)
{
    if (!gauss_last_sparse_ok(a, t)) return cudaErrorInvalidValue;
    const int cols = SP_THREADS - 2 * t.m;
    const int rows = (a.d.h + a.span - 1) / a.span;
    static const bool one_row = getenv("TW_SPARSE_ROWS") && atoi(getenv("TW_SPARSE_ROWS")) == 1; // measurement switch
    if (t.m == SP3_M && a.span == SP3_SPAN && !one_row) {
        dim3 grid((a.d.w + cols - 1) / cols, (rows + SP3_R - 1) / SP3_R, a.batch);
        if (a.fma == 2) gauss_last_sparse3_kernel<2><<<grid, SP_THREADS, 0, s>>>(a, t);
        else gauss_last_sparse3_kernel<0><<<grid, SP_THREADS, 0, s>>>(a, t);
        return cudaGetLastError();
    }
    dim3 grid((a.d.w + cols - 1) / cols, rows, a.batch);
    gauss_last_sparse_kernel<<<grid, SP_THREADS, 0, s>>>(a, t);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Box window (flags == 0), App. A.6.  Both running sums are evaluated in the oracle's order, because the
// regularised 2x2 solve amplifies even 1e-16-relative re-association differences on screenshot content
// (measured: a direct window sum moved config 4 by up to 0.12 px on 3e-5 of the pixels).
//   box_vsum : one thread per (column, plane) walks DOWN the column:  vs += double(float(M[y+m] - M[y-m-1]))
//              (the float difference is part of the answer); V is stored transposed, VT[plane][x][y].
//   box_hscan: one lane per row walks ALONG the row: g += V[x+m] - V[x-m-1] in double (coalesced reads of VT),
//              b = g / winSize^2, 2x2 solve, flow staged through a 32x32 shared tile for coalesced writes.
//   The next update-matrices then runs as first_update_kernel with flow_in.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) box_vsum_kernel(const float *__restrict__ Min, double *__restrict__ VT, LevelDims d, int m,
                                                       int pitchT, size_t planeT)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= d.w) return;
    int es;
    const float *M = M_channel(Min + (size_t)(blockIdx.y / 5) * 5 * d.plane, d.pitch, blockIdx.y % 5, es) + (size_t)x * es;
    double *v = VT + (size_t)blockIdx.y * planeT + (size_t)x * pitchT;
    const int h = d.h, pitch = d.pitch * 5;
    double vs = (double)(M[0] * (float)(m + 2));
    for (int y = 1; y < m; y++) vs = vs + (double)M[(size_t)min(y, h - 1) * pitch];
    // 16 rows per step: the 32 loads and 16 float differences are independent (issued together), only the double
    // accumulation is sequential; each thread writes whole 32-byte sectors of its VT row.
    int y = 0;
    for (; y + 16 <= h; y += 16) {
        float diff[16];
#pragma unroll
        for (int k = 0; k < 16; k++)
            diff[k] = __ldg(M + (size_t)min(y + k + m, h - 1) * pitch) - __ldg(M + (size_t)max(y + k - m - 1, 0) * pitch);
        double o[16];
#pragma unroll
        for (int k = 0; k < 16; k++) { vs = vs + (double)diff[k]; o[k] = vs; }
#pragma unroll
        for (int k = 0; k < 16; k += 2) *reinterpret_cast<double2 *>(v + y + k) = make_double2(o[k], o[k + 1]);
    }
    for (; y < h; y++) {
        float diff = __ldg(M + (size_t)min(y + m, h - 1) * pitch) - __ldg(M + (size_t)max(y - m - 1, 0) * pitch);
        vs = vs + (double)diff;
        v[y] = vs;
    }
}

cudaError_t launch_box_vsum(cudaStream_t s, const float *Min, double *VT, const LevelDims &d, int batch, int m)
{
    const int pitchT = (d.h + 31) & ~31;
    dim3 grid((d.w + 127) / 128, batch * 5);
    box_vsum_kernel<<<grid, 128, 0, s>>>(Min, VT, d, m, pitchT, (size_t)d.w * pitchT);
    return cudaGetLastError();
}

__global__ void __launch_bounds__(128) box_hscan_kernel(const double *__restrict__ VT, float *__restrict__ flow, LevelDims d, int m,
                                                        double scale, int pitchT, size_t planeT)
{
    __shared__ float tile[4][2][32][33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int y0 = (blockIdx.x * 4 + warp) * 32, b = blockIdx.y;
    const int w = d.w, h = d.h;
    if (y0 >= h) return;
    const int y = min(y0 + lane, h - 1);
    const double *V = VT + (size_t)b * 5 * planeT + y;
    double g[5];
#pragma unroll
    for (int c = 0; c < 5; c++) {
        const double *Vc = V + c * planeT;
        double t = Vc[0] * (double)(m + 2);
        for (int x = 1; x < m; x++) t = t + Vc[(size_t)min(x, w - 1) * pitchT];
        g[c] = t;
    }
    float *fxp = flow + (size_t)b * 2 * d.plane, *fyp = fxp + d.plane;
    for (int xc = 0; xc < w; xc += 32) {
        const int n = min(32, w - xc);
        for (int i0 = 0; i0 < n; i0 += 4) {
            // the differences V[x+m] - V[x-m-1] of 4 steps are independent: load and subtract them first
            double dv[4][5];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int x = min(xc + i0 + u, w - 1);
                const size_t oa = (size_t)min(x + m, w - 1) * pitchT, ob = (size_t)max(x - m - 1, 0) * pitchT;
#pragma unroll
                for (int c = 0; c < 5; c++) dv[u][c] = V[c * planeT + oa] - V[c * planeT + ob];
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                if (i0 + u >= n) break;
                double bb[5];
#pragma unroll
                for (int c = 0; c < 5; c++) {
                    g[c] = g[c] + dv[u][c];
                    bb[c] = g[c] * scale;
                }
                float fx, fy;
                solve2x2d(bb[0], bb[1], bb[2], bb[3], bb[4], fx, fy);
                tile[warp][0][lane][i0 + u] = fx;
                tile[warp][1][lane][i0 + u] = fy;
            }
        }
        __syncwarp();
        for (int r = 0; r < 32 && y0 + r < h; r++) {
            if (lane < n) {
                const size_t o = (size_t)(y0 + r) * d.pitch + xc + lane;
                fxp[o] = tile[warp][0][r][lane];
                fyp[o] = tile[warp][1][r][lane];
            }
        }
        __syncwarp();
    }
}

cudaError_t launch_box_hscan(cudaStream_t s, const double *VT, float *flow, const LevelDims &d, int batch, int m, int winSize)
{
    const int pitchT = (d.h + 31) & ~31;
    dim3 grid((d.h + 127) / 128, batch);
    box_hscan_kernel<<<grid, 128, 0, s>>>(VT, flow, d, m, 1. / ((double)winSize * winSize), pitchT, (size_t)d.w * pitchT);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Box window, fused form (window radius m <= 16): no V round trip through HBM.
//   box_ckpt : the vertical running sums again, but only their state at the top of every 32-row band is kept
//              (CK[b][band][5 * pitch] doubles, 1.25 B / px instead of 40).
//   box_band : one CTA = (pair, 32-row band), sweeping the band left to right in 32-column chunks:
//                (i)   threads = (column, channel) of the chunk + its m + 1 / m halo columns: restart the vertical running sum
//                      at the band's checkpoint and run it down the 32 rows -- the same additions in the same order as the
//                      full-column scan, so V is bit-identical -- into shared memory (doubles);
//                (ii)  threads = (row, channel): the horizontal running sum g += V[x+m] - V[x-m-1] continues across the chunks
//                      in a register; b = g / winSize^2 -> shared memory (doubles);
//                (iii) threads = pixels: 2x2 solve (double), then the next update matrices (A.4) from R0 / R1 (coalesced rows,
//                      bilinear gather) -> M', or on the last iteration the flow store.
//              Every running sum is evaluated in the oracle's order (App. A.6); nothing is re-associated.
// ------------------------------------------------------------------------------------------------
constexpr int BX_BH = 32, BX_CW = 32, BX_THREADS = 256, BX_MAXM = 16; // (16-row bands at 4 CTAs / SM measured slower: 1 293 vs 1 485 pairs/s)
__host__ __device__ constexpr int bx_vpitch(int nv) { return ((5 * nv + 10) / 16) * 16 + 5; } // doubles; = 5 mod 16, >= 5 * nv
constexpr int BX_BPITCH = 165;                                                              // doubles per row of the b tile (= 5 mod 16)

// offset of plane group pg (0: channels 0,1 interleaved; 1: channels 2,3; 2: channel 4) element i in a 5 * pitch M row
__device__ __forceinline__ int bx_off(int pitch, int pg, int i) { return pg * 2 * pitch + i; }

__global__ void __launch_bounds__(128) box_ckpt_kernel(const float *__restrict__ Min, double *__restrict__ CK, LevelDims d, int m, int nb)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x, w = d.w, h = d.h;
    if (j >= 5 * w) return;
    const int off = j < 2 * w ? j : j < 4 * w ? 2 * d.pitch + (j - 2 * w) : 4 * d.pitch + (j - 4 * w);
    const size_t rs = (size_t)5 * d.pitch;
    const float *M = Min + (size_t)blockIdx.y * 5 * d.plane + off;
    double *ck = CK + (size_t)blockIdx.y * nb * rs + off;
    double vs = (double)(M[0] * (float)(m + 2));
    for (int y = 1; y < m; y++) vs = vs + (double)M[(size_t)min(y, h - 1) * rs];
    for (int y0 = 0; y0 < h; y0 += BX_BH) {
        ck[(size_t)(y0 / BX_BH) * rs] = vs;
        // the scan is latency-bound: all 2 x 32 loads of a band are in flight before the first dependent addition
        float diff[BX_BH];
#pragma unroll
        for (int k = 0; k < BX_BH; k++) {
            const int y = y0 + k;
            diff[k] = __ldg(M + (size_t)min(y + m, h - 1) * rs) - __ldg(M + (size_t)max(min(y, h - 1) - m - 1, 0) * rs);
        }
#pragma unroll
        for (int k = 0; k < BX_BH; k++)
            if (y0 + k < h) vs = vs + (double)diff[k];
    }
}

struct BoxBandArgs {
    const float *Min;  // [B][5] planes
    const double *CK;  // [B][nb][5 * pitch]
    const float *R;    // [B][2][5] planes
    float *Mout;       // [B][5] planes (not last)
    float *flow;       // [B][2] planes (last)
    LevelDims d;
    int m, nb;
    double scale;
};

template <bool LAST>
__global__ void __launch_bounds__(BX_THREADS, 2) box_band_kernel(BoxBandArgs a)
{
    extern __shared__ __align__(16) double bx_smem[];
    const int m = a.m, nv = BX_CW + 2 * m + 1, vp = bx_vpitch(nv);
    double *Vs = bx_smem, *Bs = bx_smem + BX_BH * vp;
    const int tid = threadIdx.x, b = blockIdx.y, y0 = blockIdx.x * BX_BH;
    const int w = a.d.w, h = a.d.h, pitch = a.d.pitch;
    const size_t plane = a.d.plane, rs = (size_t)5 * pitch;
    const float *Mb = a.Min + (size_t)b * 5 * plane;
    const double *ck = a.CK + ((size_t)b * a.nb + blockIdx.x) * rs;
    const float *R0 = a.R + (size_t)b * 10 * plane, *R1 = R0 + 5 * plane;
    const int hr = tid / 5, hc = tid - hr * 5; // stage (ii): (row, channel) for tid < 160
    const bool hact = tid < BX_BH * 5 && y0 + hr < h;
    double g = 0.;
    for (int x0 = 0; x0 < w; x0 += BX_CW) {
        // ---- (i) vertical running sums of the chunk's V columns x0 - m - 1 .. x0 + 31 + m (clamped = the replicate border) ----
        for (int t = tid; t < 5 * nv; t += BX_THREADS) {
            int pg, i, ci, ch;
            if (t < 4 * nv) { pg = t >= 2 * nv; i = t - pg * 2 * nv; ci = i >> 1; ch = 2 * pg + (i & 1); }
            else { pg = 2; ci = t - 4 * nv; ch = 4; i = 0; }
            const int x = clampi(x0 - m - 1 + ci, 0, w - 1);
            const int off = pg < 2 ? bx_off(pitch, pg, 2 * x + (i & 1)) : bx_off(pitch, 2, x);
            const float *M = Mb + off;
            double vs = ck[off];
            double *vo = Vs + ci * 5 + ch;
#pragma unroll
            for (int q = 0; q < BX_BH; q += 8) { // (all 64 loads up front was measured slower: 0.32 vs 0.30 ms per pair)
                float diff[8];
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const int y = min(y0 + q + k, h - 1);
                    diff[k] = __ldg(M + (size_t)min(y + m, h - 1) * rs) - __ldg(M + (size_t)max(y - m - 1, 0) * rs);
                }
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    vs = vs + (double)diff[k];
                    vo[(q + k) * vp] = vs;
                }
            }
        }
        __syncthreads();
        // ---- (ii) horizontal running sums, one (row, channel) per thread, continued across the chunks ----
        if (hact) {
            const double *V = Vs + hr * vp + hc;
            if (x0 == 0) { // columns 0 .. m - 1 are entries m + 1 .. 2m of the first chunk
                double t = V[(m + 1) * 5] * (double)(m + 2);
                for (int x = 1; x < m; x++) t = t + V[(m + 1 + x) * 5];
                g = t;
            }
            double *Bo = Bs + hr * BX_BPITCH + hc;
            const int n = min(BX_CW, w - x0);
            for (int s = 0; s < n; s++) {
                g = g + (V[(s + 2 * m + 1) * 5] - V[s * 5]);
                Bo[s * 5] = g * a.scale;
            }
        }
        __syncthreads();
        // ---- (iii) solve + update matrices / flow store: 4 pixels per thread, two at a time (this stage is bound by the latency of
        //      its R0 / R1 loads: the 50 loads of two pixels are in flight together) ----
        {
            const int lx = tid & 31, ly = tid >> 5, x = x0 + lx;
#pragma unroll 1
            for (int jp = 0; jp < BX_BH / 8; jp += 2) {
                float fx[2], fy[2];
                bool ok[2];
#pragma unroll
                for (int k = 0; k < 2; k++) {
                    const int r = ly + 8 * (jp + k);
                    ok[k] = x < w && y0 + r < h;
                    const double *bb = Bs + r * BX_BPITCH + lx * 5;
                    fx[k] = fy[k] = 0.f;
                    if (ok[k]) solve2x2d(bb[0], bb[1], bb[2], bb[3], bb[4], fx[k], fy[k]);
                }
                if (LAST) {
#pragma unroll
                    for (int k = 0; k < 2; k++)
                        if (ok[k]) {
                            float *f = a.flow + (size_t)b * 2 * plane + (size_t)(y0 + ly + 8 * (jp + k)) * pitch + x;
                            f[0] = fx[k]; f[plane] = fy[k];
                        }
                } else {
                    UpdLoad L[2];
#pragma unroll
                    for (int k = 0; k < 2; k++)
                        if (ok[k]) upd_load(R0, R1, pitch, w, h, x, y0 + ly + 8 * (jp + k), fx[k], fy[k], L[k]);
#pragma unroll
                    for (int k = 0; k < 2; k++)
                        if (ok[k]) {
                            const int y = y0 + ly + 8 * (jp + k);
                            float mm[5];
                            upd_compute(L[k], w, h, x, y, fx[k], fy[k], mm);
                            store_M(a.Mout + (size_t)b * 5 * plane, pitch, y, x, mm);
                        }
                }
            }
        }
        // the next chunk's stage (i) only writes Vs; its barrier orders this stage's Bs reads before the next stage (ii)
    }
}

int box_band_height() { return BX_BH; }
bool box_fused_ok(const LevelDims &d, int m) { return m >= 1 && m <= BX_MAXM && d.w >= 1 && d.h >= 1; }

cudaError_t launch_box_ckpt(cudaStream_t s, const float *Min, double *CK, const LevelDims &d, int batch, int m)
{
    const int nb = (d.h + BX_BH - 1) / BX_BH;
    dim3 grid((5 * d.w + 127) / 128, batch);
    box_ckpt_kernel<<<grid, 128, 0, s>>>(Min, CK, d, m, nb);
    return cudaGetLastError();
}

cudaError_t launch_box_band(cudaStream_t s, const float *Min, const double *CK, const float *R, float *Mout, float *flow, const LevelDims &d,
                            int batch, int m, int winSize, int last)
{
    static std::atomic<bool> configured_dev[kMaxDevices][2];
    BoxBandArgs a{};
    a.Min = Min; a.CK = CK; a.R = R; a.Mout = Mout; a.flow = flow; a.d = d; a.m = m; a.nb = (d.h + BX_BH - 1) / BX_BH;
    a.scale = 1. / ((double)winSize * winSize);
    const size_t smem = sizeof(double) * (size_t)BX_BH * (bx_vpitch(BX_CW + 2 * m + 1) + BX_BPITCH);
    const size_t smem_max = sizeof(double) * (size_t)BX_BH * (bx_vpitch(BX_CW + 2 * BX_MAXM + 1) + BX_BPITCH);
    const int dev = current_device();
    if (!configured_dev[dev][last ? 1 : 0]) {
        cudaError_t e = last ? cudaFuncSetAttribute(box_band_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max)
                             : cudaFuncSetAttribute(box_band_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max);
        if (e != cudaSuccess) return e;
        configured_dev[dev][last ? 1 : 0] = true;
    }
    dim3 grid(a.nb, batch);
    if (last) box_band_kernel<true><<<grid, BX_THREADS, smem, s>>>(a);
    else box_band_kernel<false><<<grid, BX_THREADS, smem, s>>>(a);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Size-tolerance path of OpticalFlow::calculate (/root/reference/src/opticalflow.cpp:64-68): cv::resize of the
// 8-bit target to the expected size, INTER_LINEAR in effect.  OpenCV's fixed-point bilinear: 11-bit coefficients,
// horizontal pass in int, vertical pass (((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2.
// Tables: xi/xa clamped along x; yi/ya with the fraction kept and the row indices clipped (see resize_coeffs).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) resize_u8_kernel(ResizeU8Args a)
{
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    if (x >= a.w || y >= a.h) return;
    const int sy = a.yi[y], y0 = clampi(sy, 0, a.H - 1), y1 = clampi(sy + 1, 0, a.H - 1);
    const int x0 = a.xi[x], x1 = min(x0 + 1, a.W - 1);
    const int a0 = a.xa[2 * x], a1 = a.xa[2 * x + 1], b0 = a.ya[2 * y], b1 = a.ya[2 * y + 1];
    const uint8_t *s0 = a.src + (size_t)y0 * a.spitch, *s1 = a.src + (size_t)y1 * a.spitch;
    const int r0 = s0[x0] * a0 + s0[x1] * a1, r1 = s1[x0] * a0 + s1[x1] * a1;
    const int v = (((b0 * (r0 >> 4)) >> 16) + ((b1 * (r1 >> 4)) >> 16) + 2) >> 2;
    a.dst[(size_t)y * a.dpitch + x] = (uint8_t)min(max(v, 0), 255);
}

cudaError_t launch_resize_u8(cudaStream_t s, const ResizeU8Args &a)
{
    dim3 grid((a.w + 31) / 32, (a.h + 7) / 8);
    resize_u8_kernel<<<grid, dim3(32, 8), 0, s>>>(a);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Span sampling + threshold test + ordered compaction (reference src/consumer.cpp:60-77):
//   len = f32(f32(dx*dx) + f32(dy*dy));  keep iff double(len) > threshold*threshold (strict), row-major order.
// One block per pair; each thread owns a contiguous run of sample points so a block-wide exclusive scan of
// the per-thread counts yields row-major output positions.  Counts are reduced with warp shuffles.
// `skip(x, y)`: sample points the caller leaves out (ignore regions); the same test in both passes.
// ------------------------------------------------------------------------------------------------
struct DevVector { int x, y; double dx, dy; };

struct SkipNone {
    __device__ __forceinline__ bool operator()(int, int) const { return false; }
};

// The regions of one pair, staged in shared memory by sample_ignore_kernel.
struct SkipRegions {
    const int4 *r;
    int n;
    __device__ __forceinline__ bool operator()(int x, int y) const
    {
        bool in = false;
        for (int k = 0; k < n; k++) {
            const int4 q = r[k];
            in |= (x >= q.x) & (x < q.z) & (y >= q.y) & (y < q.w);
        }
        return in;
    }
};

// Block-wide exclusive scan of one count per thread (blockDim.x a multiple of 32): returns the sum of the counts of the threads
// before this one and leaves the block's sum in *total.  warp_sums[32] and *total are the caller's shared memory.
__device__ __forceinline__ int block_exclusive_scan(const int cnt, int *warp_sums, int *total)
{
    int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int incl = cnt;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        int v = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += v;
    }
    if (lane == 31) warp_sums[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        int v = lane < (int)(blockDim.x >> 5) ? warp_sums[lane] : 0;
        int s = v;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            int u = __shfl_up_sync(0xffffffffu, s, off);
            if (lane >= off) s += u;
        }
        warp_sums[lane] = s - v; // exclusive
        if (lane == 31) *total = s;
    }
    __syncthreads();
    return warp_sums[wid] + incl - cnt;
}

template <class Skip>
__device__ __forceinline__ void sample_body(const SampleArgs &a, const int b, const Skip &skip)
{
    __shared__ int warp_sums[32];
    __shared__ int total;
    const float *fxp = a.flow + (size_t)b * 2 * a.d.plane, *fyp = fxp + a.d.plane;
    const int nsx = (a.d.w + a.span - 1) / a.span, nsy = (a.d.h + a.span - 1) / a.span, ns = nsx * nsy;
    const int per = (ns + blockDim.x - 1) / blockDim.x;
    const int i0 = min(threadIdx.x * per, ns), i1 = min(i0 + per, ns);
    int cnt = 0;
    for (int i = i0; i < i1; i++) {
        int sy = i / nsx, sx = i - sy * nsx;
        if (skip(sx * a.span, sy * a.span)) continue;
        size_t o = (size_t)(sy * a.span) * a.d.pitch + sx * a.span;
        float dx = fxp[o], dy = fyp[o];
        float len = (dx * dx) + (dy * dy);
        cnt += ((double)len > a.thr2) ? 1 : 0;
    }
    int pos = block_exclusive_scan(cnt, warp_sums, &total);
    if (threadIdx.x == 0) a.counts[b] = total;
    if (cnt == 0) return;
    DevVector *out = reinterpret_cast<DevVector *>(a.vectors) + (size_t)b * a.cap;
    for (int i = i0; i < i1; i++) {
        int sy = i / nsx, sx = i - sy * nsx;
        if (skip(sx * a.span, sy * a.span)) continue;
        size_t o = (size_t)(sy * a.span) * a.d.pitch + sx * a.span;
        float dx = fxp[o], dy = fyp[o];
        float len = (dx * dx) + (dy * dy);
        if ((double)len > a.thr2) {
            if (pos < a.cap) {
                DevVector v;
                v.x = sx * a.span; v.y = sy * a.span; v.dx = (double)dx; v.dy = (double)dy;
                out[pos] = v;
            }
            pos++;
        }
    }
}

__global__ void __launch_bounds__(1024) sample_kernel(SampleArgs a)
{
    const int b = blockIdx.x;
    if (a.counted && a.counts[b] == 0) return; // OK pair: nothing to compact (block-uniform)
    sample_body(a, b, SkipNone{});
}

__global__ void __launch_bounds__(1024) sample_ignore_kernel(SampleArgs a, IgnoreRegions g)
{
    __shared__ int4 rects[kMaxIgnore];
    const int b = blockIdx.x;
    // counts[b] written by the fused last iteration (K5, K5s, the strip kernel's LAST form) is the count WITHOUT the regions, an
    // upper bound of the count with them: a pair with 0 there has 0 here too and may exit with counts[b] == 0 as it stands.  Any
    // other pair is counted again below, with the regions, and counts[b] rewritten -- so the hot kernels need no ignore form.
    if (a.counted && a.counts[b] == 0) return; // block-uniform
    const int n = min(g.n[b], kMaxIgnore);
    if ((int)threadIdx.x < n) rects[threadIdx.x] = g.rects[(size_t)b * kMaxIgnore + threadIdx.x];
    __syncthreads();
    sample_body(a, b, SkipRegions{rects, n});
}

// The mask of one pair (NULL: the pair has none), then its regions as SkipRegions tests them.
struct SkipMask {
    const uint8_t *m;
    int spitch;
    SkipRegions r;
    __device__ __forceinline__ bool operator()(int x, int y) const
    {
        if (m && m[(size_t)y * spitch + x]) return true;
        return r(x, y);
    }
};

__global__ void __launch_bounds__(1024) sample_mask_kernel(SampleArgs a, IgnoreRegions g, IgnoreMasks k)
{
    __shared__ int4 rects[kMaxIgnore];
    const int b = blockIdx.x;
    // A mask, like the regions, only removes sample points: the fused count is an upper bound here too, and the early exit of
    // sample_ignore_kernel (see its comment) holds as it stands.
    if (a.counted && a.counts[b] == 0) return; // block-uniform
    const int n = g.n ? min(g.n[b], kMaxIgnore) : 0;
    if ((int)threadIdx.x < n) rects[threadIdx.x] = g.rects[(size_t)b * kMaxIgnore + threadIdx.x];
    __syncthreads();
    const uint8_t *m = k.has[b] ? k.m + (size_t)b * k.H * k.spitch : nullptr;
    sample_body(a, b, SkipMask{m, k.spitch, SkipRegions{rects, n}});
}

cudaError_t launch_sample(cudaStream_t s, const SampleArgs &a)
{
    sample_kernel<<<a.batch, 1024, 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_sample_ignore(cudaStream_t s, const SampleArgs &a, const IgnoreRegions &g)
{
    sample_ignore_kernel<<<a.batch, 1024, 0, s>>>(a, g);
    return cudaGetLastError();
}

cudaError_t launch_sample_mask(cudaStream_t s, const SampleArgs &a, const IgnoreRegions &g, const IgnoreMasks &k)
{
    sample_mask_kernel<<<a.batch, 1024, 0, s>>>(a, g, k);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Change regions: the 8-connected components of a pair's suspicious sample points, labelled from its compact vector list, so every
// last-iteration and sample form feeds it alike.  One CTA per pair; thread t owns the run [t * per, (t + 1) * per) of vector indices,
// as sample_body owns sample points.
//   1. the cell -> vector index map over the pair's sample grid.  It is not cleared: an entry counts only if the vector it names
//      is in range and stands at that cell, which holds exactly for the cells that have a vector in this run.  A vector whose W
//      neighbour is the previous vector of the same thread's run takes that run's parent directly (no global find);
//   2. union-find (Playne and Hawick) over the neighbours W (first vector of a run), N, NW and NE, with the usual 8-connectivity
//      decision: N alone if it is there (NW and NE are its row neighbours), else NW unless W is there (W reaches it through its
//      own N), and NE; roots are joined by atomicMin on the parent of the larger one, so the root of a component is its smallest
//      vector index -- its first point in scan order -- whatever the scheduling;
//   3. flatten; the roots, in index order, take the region slots 0, 1, ... (block scan), and the slot of a root is kept in the map;
//   4. each vector folds its point into its region if that is stored (slot < kMaxChangeRegions): atomicMin / atomicMax of the
//      corners and atomicAdd of the count, summed over a thread's run of one region first; the peak is a 64-bit atomicMax of
//      (len bits << 32 | ~index), held in peak.dx until step 5 (len >= 0 orders as its bits; the tie goes to the smaller index);
//   5. one thread per stored region turns the corners into a rectangle clipped to the frame and the peak key into the vector.
// Parents change under the other threads' atomics, so they are read through L2 (__ldcg); the region fields likewise in step 5.
// ------------------------------------------------------------------------------------------------
struct DevChangeRegion { int x, y, w, h, n, pad; DevVector peak; }; // tw_change_region

__device__ __forceinline__ int uf_find(const int *par, int i)
{
    for (int q = __ldcg(par + i); q != i; q = __ldcg(par + i)) i = q;
    return i;
}

__device__ __forceinline__ void uf_union(int *par, int a, int b)
{
    for (;;) {
        a = uf_find(par, a); b = uf_find(par, b);
        if (a == b) return;
        if (a > b) { const int t = a; a = b; b = t; }
        const int old = atomicMin(par + b, a);
        if (old == b) return; // b was still a root: it now hangs below a
        b = old;              // b was linked meanwhile: join a with where it went
    }
}

__device__ __forceinline__ void fold_region(DevChangeRegion *r, int x0, int y0, int x1, int y1, int n, unsigned long long key)
{
    atomicMin(&r->x, x0); atomicMin(&r->y, y0);
    atomicMax(&r->w, x1); atomicMax(&r->h, y1);
    atomicAdd(&r->n, n);
    atomicMax(reinterpret_cast<unsigned long long *>(&r->peak.dx), key);
}

__global__ void __launch_bounds__(1024) change_regions_kernel(ChangeRegionArgs a)
{
    __shared__ int warp_sums[32];
    __shared__ int total;
    const int b = blockIdx.x;
    const int nv = min(a.counts[b], a.cap);
    if (nv == 0) { // block-uniform: an OK pair has no region
        if (threadIdx.x == 0) a.n_regions[b] = 0;
        return;
    }
    const DevVector *v = reinterpret_cast<const DevVector *>(a.vectors) + (size_t)b * a.cap;
    int *cell = a.scratch + (size_t)b * 2 * a.cap, *par = cell + a.cap;
    DevChangeRegion *reg = reinterpret_cast<DevChangeRegion *>(a.regions) + (size_t)b * kMaxChangeRegions;
    const int span = a.span, nsx = (a.w + span - 1) / span;
    const int per = (nv + blockDim.x - 1) / blockDim.x;
    const int i0 = min((int)threadIdx.x * per, nv), i1 = min(i0 + per, nv);
    // the vector i's W neighbour is vector i - 1 (scan order) if that one stands one span to its left
    auto has_w = [&](int i, int x, int y) { return i > 0 && v[i - 1].y == y && v[i - 1].x == x - span; };
    // the vector at cell c, which is (x, y), or -1
    auto at = [&](int c, int x, int y) {
        const int j = cell[c];
        return (j >= 0 && j < nv && v[j].x == x && v[j].y == y) ? j : -1;
    };
    // 1.
    for (int i = i0, head = i0; i < i1; i++) {
        const int x = v[i].x, y = v[i].y;
        cell[(y / span) * nsx + x / span] = i;
        if (!(i > i0 && has_w(i, x, y))) head = i;
        par[i] = head;
    }
    __syncthreads();
    // 2. the cells W, NW, N, NE come before i in scan order
    for (int i = i0; i < i1; i++) {
        const int x = v[i].x, y = v[i].y;
        const bool w = has_w(i, x, y);
        if (w && i == i0) uf_union(par, i, i - 1);
        if (y == 0) continue;
        const int cx = x / span, c = (y / span) * nsx + cx - nsx;
        const int n = at(c, x, y - span), nw = cx > 0 ? at(c - 1, x - span, y - span) : -1;
        if (n >= 0) {
            if (!(w && nw >= 0)) uf_union(par, i, n);
        } else {
            if (nw >= 0 && !w) uf_union(par, i, nw);
            const int ne = cx + 1 < nsx ? at(c + 1, x + span, y - span) : -1;
            if (ne >= 0) uf_union(par, i, ne);
        }
    }
    __syncthreads();
    // 3.
    int roots = 0;
    for (int i = i0; i < i1; i++) {
        const int r = uf_find(par, i);
        par[i] = r;
        roots += r == i;
    }
    int slot = block_exclusive_scan(roots, warp_sums, &total); // its barrier also ends the flattening
    if (threadIdx.x == 0) a.n_regions[b] = total;
    for (int i = i0; i < i1 && roots > 0; i++) {
        if (par[i] != i) continue;
        cell[i] = slot; // the map is not read any more: from here on it holds the slot of each root
        if (slot < kMaxChangeRegions) {
            DevChangeRegion &r = reg[slot];
            r.x = 0x7fffffff; r.y = 0x7fffffff; r.w = -1; r.h = -1; r.n = 0;
            *reinterpret_cast<unsigned long long *>(&r.peak.dx) = 0ull;
        }
        slot++;
        roots--;
    }
    __syncthreads();
    // 4.
    int cur = -1, x0 = 0, y0 = 0, x1 = 0, y1 = 0, n = 0;
    unsigned long long key = 0;
    for (int i = i0; i < i1; i++) {
        const int s = cell[par[i]];
        if (s >= kMaxChangeRegions) continue;
        if (s != cur) {
            if (cur >= 0) fold_region(reg + cur, x0, y0, x1, y1, n, key);
            cur = s; x0 = 0x7fffffff; y0 = 0x7fffffff; x1 = -1; y1 = -1; n = 0; key = 0;
        }
        const DevVector p = v[i];
        const float dx = (float)p.dx, dy = (float)p.dy;
        const float len = (dx * dx) + (dy * dy); // the sample kernel's len (this unit is built with -fmad=false)
        x0 = min(x0, p.x); y0 = min(y0, p.y); x1 = max(x1, p.x); y1 = max(y1, p.y); n++;
        const unsigned long long k = ((unsigned long long)__float_as_uint(len) << 32) | (unsigned)~i;
        key = k > key ? k : key;
    }
    if (cur >= 0) fold_region(reg + cur, x0, y0, x1, y1, n, key);
    __syncthreads();
    // 5.
    for (int s = threadIdx.x; s < min(total, kMaxChangeRegions); s += blockDim.x) {
        DevChangeRegion &r = reg[s];
        const int rx = __ldcg(&r.x), ry = __ldcg(&r.y), mx = __ldcg(&r.w), my = __ldcg(&r.h);
        const unsigned long long k = __ldcg(reinterpret_cast<const unsigned long long *>(&r.peak.dx));
        r.w = min(mx + span, a.w) - rx;
        r.h = min(my + span, a.h) - ry;
        r.pad = 0;
        r.peak = v[~(unsigned)k];
    }
}

cudaError_t launch_change_regions(cudaStream_t s, const ChangeRegionArgs &a)
{
    change_regions_kernel<<<a.batch, 1024, 0, s>>>(a);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Intensity cells.  Step 1, intensity_sum_kernel: one CTA per 64 x 32 pixel tile of a pair; thread = one column of the tile and 8
// consecutive rows, so its cell column (one division) is fixed and its cell row advances by comparison.  Before the pixels:
//   - each cell the tile meets gets its shift from the flow at its sample point (clamped to the frame, rounded half to even, 0 for a
//     non-finite component), once, into shared memory;
//   - the target around the tile is staged in shared memory, clamped to the frame as the definition clamps it: rows y0 - 9 ..
//     y0 + 40, columns x0 - 12 .. x0 + 75 (whole words where the columns lie in the frame).  A cell whose shift is at most 8 rows
//     and 11 columns reads its 3 x 3 taps there at fixed offsets; a larger shift reads them from global memory with clamps;
//   - the ignore test runs per pixel only when the pair has a mask or a region meets the tile.
// The tile of E is staged too, so that every global load of the tile is issued before the first pixel waits on one.
// A pixel's residual is the least |E - T| over the taps.  Each thread sums its pixels per cell and adds them to 32-bit shared bins
// (a tile holds 2048 pixels of at most 255 each) when its cell changes; the bins go to the pair's per-cell totals with one global
// atomic per (tile, cell) and total.  Integer atomics commute, so the totals do not depend on the scheduling.
// Steps 2 and 3 read the totals in chunks of kIntChunk cells, one CTA per (chunk, pair), thread = 8 consecutive cells: step 2
// counts the intensity cells of each chunk, step 3 adds up the counts of the chunks before its own and writes its cells from there
// in scan order (block scan, as sample_body).  Step 3 also clears the totals it read: they are zero between runs (they are cleared
// once when allocated), so no memset runs per step.
// ------------------------------------------------------------------------------------------------
constexpr int kIntTileW = 64, kIntTileH = 32, kIntRows = 8;            // 64 columns x 4 row groups = 256 threads
constexpr int kIntHaloY = 9, kIntHaloX = 12;                          // staged rows / columns on each side of the tile
constexpr int kIntStageW = kIntTileW + 2 * kIntHaloX, kIntStageH = kIntTileH + 2 * kIntHaloY;

__device__ __forceinline__ int intensity_shift(float f, int lim)
{
    if (!isfinite(f)) return 0;
    return __float2int_rn(fminf(fmaxf(f, (float)-lim), (float)lim));
}

__global__ void __launch_bounds__(256) intensity_sum_kernel(IntensityArgs a)
{
    __shared__ unsigned bin_s[kIntTileW * kIntTileH], bin_n[kIntTileW * kIntTileH];
    __shared__ int2 bin_shift[kIntTileW * kIntTileH];
    __shared__ __align__(16) uint8_t st[kIntStageH * kIntStageW];
    __shared__ __align__(16) uint8_t se[kIntTileH * kIntTileW];
    __shared__ int4 rects[kMaxIgnore];
    const int b = blockIdx.z, w = a.d.w, h = a.d.h, span = a.span;
    const int x0 = blockIdx.x * kIntTileW, y0 = blockIdx.y * kIntTileH;
    const int x1 = min(x0 + kIntTileW, w), y1 = min(y0 + kIntTileH, h);
    const int cx0 = x0 / span, cy0 = y0 / span;
    const int ncx = (x1 - 1) / span - cx0 + 1, ncy = (y1 - 1) / span - cy0 + 1; // the tile's cells: at most 64 x 32
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    const float *fxp = a.flow + (size_t)b * 2 * a.d.plane, *fyp = fxp + a.d.plane;
    for (int i = tid; i < ncx * ncy; i += 256) {
        bin_s[i] = 0; bin_n[i] = 0;
        const size_t o = (size_t)((cy0 + i / ncx) * span) * a.d.pitch + (size_t)(cx0 + i % ncx) * span;
        bin_shift[i] = make_int2(intensity_shift(__ldg(fxp + o), w), intensity_shift(__ldg(fyp + o), h));
    }
    const int nr = a.g.n ? min(a.g.n[b], kMaxIgnore) : 0;
    bool meets = false;
    if (tid < nr) {
        const int4 q = a.g.rects[(size_t)b * kMaxIgnore + tid];
        rects[tid] = q;
        meets = q.x < x1 && q.z > x0 && q.y < y1 && q.w > y0;
    }
    const uint8_t *mask = a.k.m && a.k.has[b] ? a.k.m + (size_t)b * a.k.H * a.k.spitch : nullptr;
    const uint8_t *E = a.src + (size_t)b * 2 * h * a.spitch, *T = E + (size_t)h * a.spitch;
    const int sx0 = x0 - kIntHaloX, sy0 = y0 - kIntHaloY;
    if (sx0 >= 0 && sx0 + kIntStageW <= w) { // whole words: x0 and spitch are multiples of 16
        for (int i = tid; i < kIntStageH * (kIntStageW / 4); i += 256) {
            const int r = i / (kIntStageW / 4), c = i - r * (kIntStageW / 4);
            const int gy = min(max(sy0 + r, 0), h - 1);
            reinterpret_cast<unsigned *>(st)[i] = __ldg(reinterpret_cast<const unsigned *>(T + (size_t)gy * a.spitch + sx0) + c);
        }
    } else {
        for (int i = tid; i < kIntStageH * kIntStageW; i += 256) {
            const int r = i / kIntStageW, c = i - r * kIntStageW;
            st[i] = __ldg(T + (size_t)min(max(sy0 + r, 0), h - 1) * a.spitch + min(max(sx0 + c, 0), w - 1));
        }
    }
    for (int i = tid; i < kIntTileH * (kIntTileW / 4); i += 256) { // E: whole words of the tile's rows, up to the row pitch
        const int r = i / (kIntTileW / 4), c = 4 * (i - r * (kIntTileW / 4));
        if (y0 + r < h && x0 + c < a.spitch)
            reinterpret_cast<unsigned *>(se)[i] = __ldg(reinterpret_cast<const unsigned *>(E + (size_t)(y0 + r) * a.spitch + x0 + c));
    }
    const bool test_ignore = __syncthreads_or(meets || mask != nullptr);
    const SkipRegions in_region{rects, nr};
    const int x = x0 + threadIdx.x, ya = y0 + threadIdx.y * kIntRows;
    if (x < w && ya < h) {
        const int cx = x / span, yb = min(ya + kIntRows, h);
        int cy = ya / span, next = (cy + 1) * span;
        int bin = (cy - cy0) * ncx + (cx - cx0);
        int2 sh = bin_shift[bin];
        bool near = abs(sh.x) < kIntHaloX && abs(sh.y) < kIntHaloY;
        unsigned s = 0, n = 0;
        for (int y = ya; y < yb; y++) {
            if (y >= next) { // the next cell down
                if (n > 0) { atomicAdd(&bin_s[bin], s); atomicAdd(&bin_n[bin], n); }
                s = 0; n = 0;
                cy++; next += span; bin += ncx;
                sh = bin_shift[bin];
                near = abs(sh.x) < kIntHaloX && abs(sh.y) < kIntHaloY;
            }
            if (test_ignore && ((mask && mask[(size_t)y * a.k.spitch + x]) || in_region(x, y))) continue;
            const int e = se[(y - y0) * kIntTileW + threadIdx.x];
            int r = 255;
            if (near) {
                const uint8_t *c = st + (y - sy0 + sh.y) * kIntStageW + (x - sx0 + sh.x);
#pragma unroll
                for (int v = -1; v <= 1; v++)
#pragma unroll
                    for (int u = -1; u <= 1; u++) r = min(r, abs(e - (int)c[v * kIntStageW + u]));
            } else {
#pragma unroll
                for (int v = -1; v <= 1; v++) {
                    const uint8_t *row = T + (size_t)min(max(y + sh.y + v, 0), h - 1) * a.spitch;
#pragma unroll
                    for (int u = -1; u <= 1; u++) r = min(r, abs(e - (int)__ldg(row + min(max(x + sh.x + u, 0), w - 1))));
                }
            }
            s += r; n++;
        }
        if (n > 0) { atomicAdd(&bin_s[bin], s); atomicAdd(&bin_n[bin], n); }
    }
    __syncthreads();
    const int nsx = (w + span - 1) / span;
    for (int i = tid; i < ncx * ncy; i += 256) {
        const unsigned bn = bin_n[i];
        if (bn == 0) continue;
        const size_t c = (size_t)b * a.cell_cap + (size_t)(cy0 + i / ncx) * nsx + cx0 + i % ncx;
        atomicAdd(a.sum + c, (unsigned long long)bin_s[i]);
        atomicAdd(a.cnt + c, bn);
    }
}

struct DevIntensityCell { int x, y, n, residual; }; // tw_intensity_cell

// Flags of the 8 cells [i0, i0 + 8) of a pair (bit j: cell i0 + j; cells past ns are not flagged).
__device__ __forceinline__ unsigned intensity_flags(const IntensityArgs &a, const unsigned long long *sum, const unsigned *cnt, int i0, int ns)
{
    unsigned f = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const int i = i0 + j;
        const unsigned n = i < ns ? cnt[i] : 0u;
        const unsigned long long s = i < ns ? sum[i] : 0ull;
        f |= (n > 0 && s > (unsigned long long)a.t * n) ? 1u << j : 0u;
    }
    return f;
}

__global__ void __launch_bounds__(1024) intensity_count_kernel(IntensityArgs a)
{
    __shared__ int warp_sums[32];
    __shared__ int total;
    const int b = blockIdx.y, k = blockIdx.x;
    const int ns = ((a.d.w + a.span - 1) / a.span) * ((a.d.h + a.span - 1) / a.span);
    const int i0 = k * kIntChunk + threadIdx.x * 8;
    const unsigned f = intensity_flags(a, a.sum + (size_t)b * a.cell_cap, a.cnt + (size_t)b * a.cell_cap, i0, ns);
    block_exclusive_scan(__popc(f), warp_sums, &total);
    if (threadIdx.x == 0) a.chunk_counts[(size_t)b * a.max_chunks + k] = total;
}

__global__ void __launch_bounds__(1024) intensity_compact_kernel(IntensityArgs a)
{
    __shared__ int warp_sums[32];
    __shared__ int total;
    const int b = blockIdx.y, k = blockIdx.x;
    const int nsx = (a.d.w + a.span - 1) / a.span, ns = nsx * ((a.d.h + a.span - 1) / a.span);
    // the cells of the chunks before this one
    int before = 0;
    for (int j = threadIdx.x; j < k; j += blockDim.x) before += a.chunk_counts[(size_t)b * a.max_chunks + j];
    block_exclusive_scan(before, warp_sums, &total);
    const int base = total;
    __syncthreads(); // every thread has read `total` before the next scan writes it
    unsigned long long *sum = a.sum + (size_t)b * a.cell_cap;
    unsigned *cnt = a.cnt + (size_t)b * a.cell_cap;
    const int i0 = k * kIntChunk + threadIdx.x * 8;
    unsigned f = intensity_flags(a, sum, cnt, i0, ns);
    int pos = base + block_exclusive_scan(__popc(f), warp_sums, &total);
    if (k == gridDim.x - 1 && threadIdx.x == 0) a.n_cells[b] = base + total;
    DevIntensityCell *out = reinterpret_cast<DevIntensityCell *>(a.cells) + (size_t)b * kMaxIntensityCells;
    for (; f && pos < kMaxIntensityCells; f &= f - 1, pos++) {
        const int i = i0 + __ffs(f) - 1;
        const int sy = i / nsx, sx = i - sy * nsx;
        out[pos] = DevIntensityCell{sx * a.span, sy * a.span, (int)cnt[i], (int)min(sum[i], 0x7fffffffull)};
    }
    __syncthreads(); // the chunk's totals are read (above, by the thread that owns each cell) before they are cleared, coalesced
    for (int i = k * kIntChunk + threadIdx.x; i < min((k + 1) * kIntChunk, ns); i += blockDim.x) { sum[i] = 0; cnt[i] = 0; }
}

int intensity_chunks(int w, int h, int span)
{
    const int ns = ((w + span - 1) / span) * ((h + span - 1) / span);
    return (ns + kIntChunk - 1) / kIntChunk;
}

cudaError_t launch_intensity_sum(cudaStream_t s, const IntensityArgs &a)
{
    const dim3 grid((a.d.w + kIntTileW - 1) / kIntTileW, (a.d.h + kIntTileH - 1) / kIntTileH, a.batch);
    intensity_sum_kernel<<<grid, dim3(kIntTileW, kIntTileH / kIntRows), 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_intensity_count(cudaStream_t s, const IntensityArgs &a)
{
    intensity_count_kernel<<<dim3(intensity_chunks(a.d.w, a.d.h, a.span), a.batch), kIntChunk / 8, 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_intensity_compact(cudaStream_t s, const IntensityArgs &a)
{
    intensity_compact_kernel<<<dim3(intensity_chunks(a.d.w, a.d.h, a.span), a.batch), kIntChunk / 8, 0, s>>>(a);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Ignore regions, step 1: the expected pixels inside each region replace the target's (after the +-5 px resize, before the level
// images).  One CTA per (region, pair); warp = row, lane = 16-byte column where the row segment is aligned, bytes at its ends.
// The expected and target slots of a pair share their alignment (spitch and H * spitch are multiples of 16).  Overlapping regions
// write the same bytes, so the CTAs need no ordering.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ignore_paint_kernel(uint8_t *src, int H, int spitch, IgnoreRegions g)
{
    const int b = blockIdx.y, r = blockIdx.x;
    if (r >= g.n[b]) return;
    const int4 q = g.rects[(size_t)b * kMaxIgnore + r];
    const uint8_t *e = src + (size_t)b * 2 * H * spitch;
    uint8_t *t = src + ((size_t)b * 2 + 1) * H * spitch;
    const int a0 = (q.x + 15) & ~15, a1 = q.z & ~15; // the 16-byte aligned columns [a0, a1) of [x0, x1)
    const int lane = threadIdx.x & 31;
    for (int y = q.y + (int)(threadIdx.x >> 5); y < q.w; y += 8) {
        const size_t row = (size_t)y * spitch;
        if (a0 < a1) {
            for (int x = a0 + 16 * lane; x < a1; x += 16 * 32)
                *reinterpret_cast<uint4 *>(t + row + x) = *reinterpret_cast<const uint4 *>(e + row + x);
            for (int x = q.x + lane; x < a0; x += 32) t[row + x] = e[row + x];
            for (int x = a1 + lane; x < q.z; x += 32) t[row + x] = e[row + x];
        } else {
            for (int x = q.x + lane; x < q.z; x += 32) t[row + x] = e[row + x];
        }
    }
}

cudaError_t launch_ignore_paint(cudaStream_t s, uint8_t *src, int H, int spitch, const IgnoreRegions &g, int batch)
{
    ignore_paint_kernel<<<dim3(kMaxIgnore, batch), 256, 0, s>>>(src, H, spitch, g);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Ignore masks, step 1: the expected pixels where the pair's mask is nonzero replace the target's (after the +-5 px resize, before
// the level images).  Thread = 16 bytes of a row: expected, target and mask vectors in, t = m ? e : t per byte (__vcmpne4 gives
// 0xff for every nonzero mask byte), the target vector out.  When W is not a multiple of 16 the last vector of a row reaches past
// column W into the row's padding: that one goes byte by byte up to W, so the padding of the mask plane is never read.  The mask
// plane shares the slots' pitch and alignment.  With ignore regions as well, both kernels write expected bytes, so their order
// does not matter.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) mask_paint_kernel(uint8_t *src, IgnoreMasks k)
{
    const int b = blockIdx.y;
    if (!k.has[b]) return; // block-uniform: pairs without a mask
    const int nc = (k.W + 15) >> 4;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= k.H * nc) return;
    const int y = i / nc, x = (i - y * nc) << 4;
    const size_t plane = (size_t)k.H * k.spitch, row = (size_t)y * k.spitch + x;
    const uint8_t *e = src + (size_t)b * 2 * plane + row;
    uint8_t *t = src + ((size_t)b * 2 + 1) * plane + row;
    const uint8_t *m = k.m + (size_t)b * plane + row;
    if (x + 16 <= k.W) {
        const uint4 ev = *reinterpret_cast<const uint4 *>(e), mv = *reinterpret_cast<const uint4 *>(m);
        uint4 tv = *reinterpret_cast<const uint4 *>(t);
        unsigned s;
        s = __vcmpne4(mv.x, 0u); tv.x = (ev.x & s) | (tv.x & ~s);
        s = __vcmpne4(mv.y, 0u); tv.y = (ev.y & s) | (tv.y & ~s);
        s = __vcmpne4(mv.z, 0u); tv.z = (ev.z & s) | (tv.z & ~s);
        s = __vcmpne4(mv.w, 0u); tv.w = (ev.w & s) | (tv.w & ~s);
        *reinterpret_cast<uint4 *>(t) = tv;
    } else {
        for (int j = 0; j < k.W - x; j++)
            if (m[j]) t[j] = e[j];
    }
}

cudaError_t launch_mask_paint(cudaStream_t s, uint8_t *src, const IgnoreMasks &k, int batch)
{
    const long long threads = (long long)k.H * ((k.W + 15) >> 4);
    mask_paint_kernel<<<dim3((unsigned)((threads + 255) / 256), batch), 256, 0, s>>>(src, k);
    return cudaGetLastError();
}

} // namespace tw

#ifdef TW_TIMELINE
extern "C" int tw_debug_set_flags(int flags) { return (int)cudaMemcpyToSymbol(tw::g_dev_flags, &flags, sizeof(int)); }
extern "C" int tw_debug_timeline(unsigned long long *out, int n_words)
{
    return (int)cudaMemcpyFromSymbol(out, tw::g_timeline, sizeof(unsigned long long) * n_words);
}
#endif
