// tw_device.cuh -- device helpers shared by the kernel translation units (tw_kernels.cu, tw_window.cu).  Both are compiled
// with -fmad=false: the oracle's results depend on the rounding of every add / mul (SURVEY.md App. A), so nothing may be
// contracted implicitly; fused multiply-adds appear only where written as fmaf() / fma.rn.
#pragma once
#include "tw_kernels.cuh"

namespace tw {

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }


// border damping {0.14, 0.14, 0.4472, 0.4472, 0.4472} indexed by the distance to the edge (App. A.4)
__device__ __forceinline__ float border_tab(int i) { return i < 2 ? 0.14f : 0.4472f; }


// ------------------------------------------------------------------------------------------------
// R and M are ROW-INTERLEAVED planar (5*plane floats per image / pair): the five channels of image row y are the
// five consecutive pitch-sized rows (y*5 + c).  With the compile-time pitch every channel, every bilinear neighbour
// and every row of a register-blocked column is ONE base register + an immediate offset.
//   R row group: [dy | dx | yy | xx | xy]                     each `pitch` floats
//   M row group: [(G11,G12) float2 x pitch | (G22,h1) float2 x pitch | h2 float x pitch]   = 5*pitch floats
// The packed f32x2 window kernel loads both channels of an M pair with one 8-byte load; writers store float2.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void store_M(float *__restrict__ Mb, int pitch, int y, int x, const float m[5])
{
    float *row = Mb + (size_t)y * 5 * pitch;
    *reinterpret_cast<float2 *>(row + 2 * x) = make_float2(m[0], m[1]);
    *reinterpret_cast<float2 *>(row + 2 * pitch + 2 * x) = make_float2(m[2], m[3]);
    row[4 * pitch + x] = m[4];
}
// channel c of M as a strided scalar view: element (y, x) is base[(size_t)y * 5 * pitch + x * stride]
__device__ __forceinline__ const float *M_channel(const float *Mb, int pitch, int c, int &stride)
{
    if (c < 4) { stride = 2; return Mb + (c >> 1) * 2 * pitch + (c & 1); }
    stride = 1;
    return Mb + 4 * pitch;
}


// The oracle's mul / add sequence of App. A.4 (-fmad=false TU: no contraction).  BORDER = false: the caller knows the pixel
// is outside the damped 5-pixel frame border.
// pt / pb = R1 at rows y1 / y1+1, columns (x1, x1+1); q = R0 at (x, y).
template <bool BORDER = true>
__device__ __forceinline__ void upd_core(const float q[5], const float pt[5][2], const float pb[5][2], bool inside, float fx, float fy,
                                         int w, int h, int x, int y, float dx, float dy, float m[5])
{
    float r[5];
    if (inside) {
        const float a00 = (1.f - fx) * (1.f - fy), a01 = fx * (1.f - fy), a10 = (1.f - fx) * fy, a11 = fx * fy;
#pragma unroll
        for (int c = 0; c < 5; c++) r[c] = a00 * pt[c][0] + a01 * pt[c][1] + a10 * pb[c][0] + a11 * pb[c][1];
        r[2] = (q[2] + r[2]) * 0.5f;
        r[3] = (q[3] + r[3]) * 0.5f;
        r[4] = (q[4] + r[4]) * 0.25f;
    } else {
        r[0] = r[1] = 0.f;
        r[2] = q[2];
        r[3] = q[3];
        r[4] = q[4] * 0.5f;
    }
    float r2 = (q[0] - r[0]) * 0.5f, r3 = (q[1] - r[1]) * 0.5f, r4 = r[2], r5 = r[3], r6 = r[4];
    r2 = r2 + (r4 * dy + r6 * dx);
    r3 = r3 + (r6 * dy + r5 * dx);
    if (BORDER && ((unsigned)(x - 5) >= (unsigned)(w - 10) || (unsigned)(y - 5) >= (unsigned)(h - 10))) {
        float sc = (x < 5 ? border_tab(x) : 1.f) * (x >= w - 5 ? border_tab(w - x - 1) : 1.f) * (y < 5 ? border_tab(y) : 1.f) *
                   (y >= h - 5 ? border_tab(h - y - 1) : 1.f);
        r2 *= sc; r3 *= sc; r4 *= sc; r5 *= sc; r6 *= sc;
    }
    m[0] = r4 * r4 + r6 * r6;
    m[1] = (r4 + r5) * r6;
    m[2] = r5 * r5 + r6 * r6;
    m[3] = r4 * r2 + r6 * r3;
    m[4] = r6 * r2 + r5 * r3;
}


__device__ __forceinline__ void solve2x2(float g11f, float g12f, float g22f, float h1f, float h2f, float &fx, float &fy)
{
    double g11 = g11f, g12 = g12f, g22 = g22f, h1 = h1f, h2 = h2f;
    double idet = 1. / (g11 * g22 - g12 * g12 + 1e-3);
    fx = (float)((g11 * h2 - g12 * h1) * idet);
    fy = (float)((g22 * h1 - g12 * h2) * idet);
}

__device__ __forceinline__ void solve2x2d(double g11, double g12, double g22, double h1, double h2, float &fx, float &fy)
{
    double idet = 1. / (g11 * g22 - g12 * g12 + 1e-3);
    fx = (float)((g11 * h2 - g12 * h1) * idet);
    fy = (float)((g22 * h1 - g12 * h2) * idet);
}


// Packed f32x2 arithmetic (sm_100+), written as PTX with explicit .rn so that neither NVVM nor ptxas may contract a
// multiply and an add into an FFMA2: each half is one IEEE-754 operation, exactly like the scalar oracle code.
// (The CUDA intrinsics __fmul2_rn + __fadd2_rn WERE contracted into FFMA2 by nvcc 12.9 even with -fmad=false.)
__device__ __forceinline__ unsigned long long f2_pack(float2 v)
{
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(v.x), "f"(v.y));
    return r;
}
__device__ __forceinline__ float2 f2_unpack(unsigned long long r)
{
    float2 v;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(v.x), "=f"(v.y) : "l"(r));
    return v;
}
__device__ __forceinline__ float2 tw_add2(float2 a, float2 b)
{
    unsigned long long d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_pack(a)), "l"(f2_pack(b)));
    return f2_unpack(d);
}
__device__ __forceinline__ float2 tw_mul2(float2 a, float2 b)
{
    unsigned long long d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_pack(a)), "l"(f2_pack(b)));
    return f2_unpack(d);
}
// NOTE: ptxas 12.9 contracts mul.rn.f32x2 feeding add.rn.f32x2 into one FFMA2 even with --fmad false (the scalar
// mul.rn/add.rn pair is respected).  The faithful accumulate "v + p" is therefore issued as fma(p, one, v) with
// `one` a RUNTIME 1.0f (WinTaps.one): p * 1.0 is exact, so the result is round(p + v) -- one IEEE add -- and ptxas
// cannot fold it because it does not know the value.
__device__ __forceinline__ float2 tw_fma2(float2 a, float2 b, float2 c)
{
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(f2_pack(a)), "l"(f2_pack(b)), "l"(f2_pack(c)));
    return f2_unpack(d);
}


__device__ __forceinline__ float2 tw_sub2(float2 a, float2 b)
{
    unsigned long long d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_pack(a)), "l"(f2_pack(b)));
    return f2_unpack(d);
}

// A.4 for TWO pixels at once (packed f32x2: .x / .y = the two pixels), both "inside" and both outside the damped 5-pixel frame
// border: the operation sequence of upd_core<false> with inside = true, every half of every packed instruction one
// IEEE-754 operation, so the result is bit-identical to the scalar code.  A rounded sum whose second operand is a product is
// issued as fma(product, one, first) with `one` the RUNTIME 1.0f (see tw_fma2): ptxas would otherwise contract the packed
// multiply into the packed add.
__device__ __forceinline__ void upd_core2(const float2 q[5], const float2 pt[5][2], const float2 pb[5][2], float2 fx, float2 fy, float2 dx,
                                          float2 dy, float one, float2 m[5])
{
    const float2 one2 = make_float2(one, one), c1 = make_float2(1.f, 1.f), half = make_float2(0.5f, 0.5f), quarter = make_float2(0.25f, 0.25f);
    const float2 gx = tw_sub2(c1, fx), gy = tw_sub2(c1, fy);
    const float2 a00 = tw_mul2(gx, gy), a01 = tw_mul2(fx, gy), a10 = tw_mul2(gx, fy), a11 = tw_mul2(fx, fy);
    float2 r[5];
#pragma unroll
    for (int c = 0; c < 5; c++) {
        float2 t = tw_mul2(a00, pt[c][0]);
        t = tw_fma2(tw_mul2(a01, pt[c][1]), one2, t);
        t = tw_fma2(tw_mul2(a10, pb[c][0]), one2, t);
        r[c] = tw_fma2(tw_mul2(a11, pb[c][1]), one2, t);
    }
    const float2 r4 = tw_mul2(tw_add2(q[2], r[2]), half), r5 = tw_mul2(tw_add2(q[3], r[3]), half), r6 = tw_mul2(tw_add2(q[4], r[4]), quarter);
    float2 r2 = tw_mul2(tw_sub2(q[0], r[0]), half), r3 = tw_mul2(tw_sub2(q[1], r[1]), half);
    r2 = tw_add2(r2, tw_fma2(tw_mul2(r6, dx), one2, tw_mul2(r4, dy)));
    r3 = tw_add2(r3, tw_fma2(tw_mul2(r5, dx), one2, tw_mul2(r6, dy)));
    m[0] = tw_fma2(tw_mul2(r6, r6), one2, tw_mul2(r4, r4));
    m[1] = tw_mul2(tw_add2(r4, r5), r6);
    m[2] = tw_fma2(tw_mul2(r6, r6), one2, tw_mul2(r5, r5));
    m[3] = tw_fma2(tw_mul2(r6, r3), one2, tw_mul2(r4, r2));
    m[4] = tw_fma2(tw_mul2(r5, r3), one2, tw_mul2(r6, r2));
}

} // namespace tw
