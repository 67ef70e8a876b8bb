// gf_s8.cuh -- the headline kernel: warp-private fused guided filter, gray float32, 8 ADJACENT
// columns per lane, 256-bit global accesses, packed f32x2 arithmetic (sm_100a).
//
// Design target (DESIGN.md section 3): on B200 this filter is bound by the shuffle/shared-memory
// pipe (MIO) and by FP32 issue long before HBM, so the kernel is built to minimise both per pixel:
//   * a lane owns 8 adjacent columns -> one LDG.256 per plane and row, one STG.256 per output row
//     (the coalescing minimum of 8 L1 wavefronts per kB), and the cross-lane traffic of a
//     (2R+1)-window sum drops to 2R/8 values per pixel and quantity: for R = 8 exactly one value
//     from the left neighbour and one from the right neighbour per pixel (16 SHFL per 8 px);
//   * window sums use additions only (float32 error ~1e-7 relative):
//         w_j(l) = A_j(l-m) + p_j(l+m),  A_j = x_j + .. + x_7 + [totals of the next 2m-1 lanes],
//         p_j = x_0 + .. + x_j,           m = R/8
//     i.e. 23 additions per 8 pixels and quantity at R = 8;
//   * vertical running sums, the a/b algebra and the output are FADD2/FFMA2/FMUL2 on column pairs
//     (half the issue slots of scalar code; the pairs come straight out of the 256-bit loads);
//   * every WARP is an independent worker (32*8-column window, a band of rows): no barriers; the
//     stage-2 row ring (2R+1 rows of sum_x a, sum_x b) is the only shared-memory traffic, laid out
//     so that every LDS.128/STS.128 is conflict-free;
//   * the row that leaves the vertical window is re-read from L2 2R+1 rows later and doubles as
//     the guide row of the next output; rows are loaded one iteration ahead into registers and
//     hinted into L2 a few rows further ahead;
//   * the row loop is cut into phases with compile-time stage flags (straight-line steady state);
//     the vertical border is a row-index map, the horizontal border (REFLECT/REFLECT101) is
//     per-lane mirror loads in the first/last strip only (mirrored columns give mirrored a, b, so
//     no other code changes); TRUNCATE zero-fills and divides by per-pixel counts.
// A/B outputs, unaligned planes and radii without an instantiation use the older kernels
// (gf_wp.cuh, gf_fast.cuh, gf_generic.cuh).
#pragma once
#include "gf_wp.cuh"

#ifndef GF_S8_NEWTON
#define GF_S8_NEWTON 1        // one Newton step after MUFU.RCP
#endif
#ifndef GF_S8_RESEED2
#define GF_S8_RESEED2 1       // re-seed the stage-2 running sums from pure additions every 2R+1 rows
#endif
#ifndef GF_S8_RESEED1
#define GF_S8_RESEED1 1       // same for the four stage-1 column sums
#endif
// Developer ablations (timing experiments only -- results are WRONG with any of them set):
#ifndef GF_S8_ABL
#define GF_S8_ABL 0           // bit 0: no shuffles, bit 1: no ring traffic, bit 2: no steady-state loads, bit 3: no stores
#endif
#if GF_S8_ABL & 1
#define GF_S8_SHFL_UP(v, d) (v)
#define GF_S8_SHFL_DOWN(v, d) (v)
#else
#define GF_S8_SHFL_UP(v, d) __shfl_up_sync(0xffffffffu, v, d)
#define GF_S8_SHFL_DOWN(v, d) __shfl_down_sync(0xffffffffu, v, d)
#endif
#ifndef GF_S8_EDGE_PCT
#define GF_S8_EDGE_PCT 85     // band height of the two edge strips (mirror loads, clipped counts, column map), % of the interior strips'
#endif
#ifndef GF_S8_PF
#define GF_S8_PF 4            // rows ahead for the L2 prefetch hint (0 = off)
#endif

// ---- packed float32x2 and 256-bit access helpers -------------------------------------------------
#ifdef GF_CPU_EMU
static inline float2 gf_add2(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
static inline float2 gf_sub2(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
static inline float2 gf_mul2(float2 a, float2 b) { return make_float2(a.x * b.x, a.y * b.y); }
static inline float2 gf_fma2(float2 a, float2 b, float2 c) { return make_float2(std::fmaf(a.x, b.x, c.x), std::fmaf(a.y, b.y, c.y)); }
static inline void gf_ld8(const float* p, float2 (&v)[4])
{
    for (int i = 0; i < 4; ++i) v[i] = make_float2(p[2 * i], p[2 * i + 1]);
}
static inline void gf_st8(float* p, const float2 (&v)[4])
{
    for (int i = 0; i < 4; ++i) { p[2 * i] = v[i].x; p[2 * i + 1] = v[i].y; }
}
#else
__device__ __forceinline__ float2 gf_add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 gf_sub2(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
__device__ __forceinline__ float2 gf_mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 gf_fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ void gf_ld8(const float* p, float2 (&v)[4])
{
    asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(v[0].x), "=f"(v[0].y), "=f"(v[1].x), "=f"(v[1].y), "=f"(v[2].x), "=f"(v[2].y), "=f"(v[3].x), "=f"(v[3].y)
                 : "l"(p));
}
__device__ __forceinline__ void gf_st8(float* p, const float2 (&v)[4])
{
    asm volatile("st.global.v8.f32 [%8], {%0,%1,%2,%3,%4,%5,%6,%7};"
                 ::"f"(v[0].x), "f"(v[0].y), "f"(v[1].x), "f"(v[1].y), "f"(v[2].x), "f"(v[2].y), "f"(v[3].x), "f"(v[3].y), "l"(p)
                 : "memory");
}
#endif
// ---- uint8 I/O (SURVEY 8(f) rank 2: convertTo(CV_32F, 1/255) on load, convertTo(CV_8U, 255) on store,
// main.cpp:121-122,158 fused into the kernel: 3 B/px instead of 12) ----------------------------------
// The uint8 build works in the INTEGER domain: I' = 255 I, p' = 255 p are loaded as the floats 0..255.
// a is scale-free, b' = 255 b, q' = mean_a I' + mean_b' = 255 q is exactly the value convertTo(CV_8U, 255)
// rounds, and eps becomes 255^2 eps -- so neither conversion costs an operation.  Better than free: the
// vertical running sums of I', p', I'p', I'I' are integers below 2^24, i.e. EXACT in float32 (no drift,
// no re-seed), and so are the lane prefixes of the window sums; only sums above 2^24 (17 x 17 x 255^2
// = 1.9e7) round, by at most one part in 2^24.  The byte conversions themselves (gf_u8_to_f, gf_f_to_u8,
// gf_ld1, gf_st1) are in gf_common.cuh: the fast guided filter's uint8 build uses them too.
__device__ __forceinline__ float gf_bits_f(unsigned u)
{
#ifdef GF_CPU_EMU
    float f; std::memcpy(&f, &u, 4); return f;
#else
    return __uint_as_float(u);
#endif
}
__device__ __forceinline__ unsigned gf_f_bits(float f)
{
#ifdef GF_CPU_EMU
    unsigned u; std::memcpy(&u, &f, 4); return u;
#else
    return __float_as_uint(f);
#endif
}
// 8 pixels = 8 bytes, kept RAW in v[0] (two registers); gf_u8_expand converts them where the row is consumed,
// one iteration later -- a conversion right behind the load would make the warp wait for the load there.
__device__ __forceinline__ void gf_ld8(const unsigned char* p, float2 (&v)[4])
{
    const uint2 t = *reinterpret_cast<const uint2*>(p);
    v[0] = make_float2(gf_bits_f(t.x), gf_bits_f(t.y));
    v[1] = v[2] = v[3] = make_float2(0.f, 0.f);
}
__device__ __forceinline__ void gf_u8_expand(float2 (&v)[4])
{
    const unsigned x = gf_f_bits(v[0].x), y = gf_f_bits(v[0].y);
    v[0] = make_float2(gf_u8_to_f(x, 0), gf_u8_to_f(x, 1));
    v[1] = make_float2(gf_u8_to_f(x, 2), gf_u8_to_f(x, 3));
    v[2] = make_float2(gf_u8_to_f(y, 0), gf_u8_to_f(y, 1));
    v[3] = make_float2(gf_u8_to_f(y, 2), gf_u8_to_f(y, 3));
}
__device__ __forceinline__ void gf_st8(unsigned char* p, const float2 (&v)[4])
{
    uint2 t;
    t.x = gf_f_to_u8(v[0].x) | (gf_f_to_u8(v[0].y) << 8) | (gf_f_to_u8(v[1].x) << 16) | (gf_f_to_u8(v[1].y) << 24);
    t.y = gf_f_to_u8(v[2].x) | (gf_f_to_u8(v[2].y) << 8) | (gf_f_to_u8(v[3].x) << 16) | (gf_f_to_u8(v[3].y) << 24);
    *reinterpret_cast<uint2*>(p) = t;
}
__device__ __forceinline__ float2 gf_neg2(float2 a) { return make_float2(-a.x, -a.y); }
__device__ __forceinline__ float2 gf_dup2(float a) { return make_float2(a, a); }

// ---- (2R+1)-window sums over the 8 columns of every lane ------------------------------------------
// R a multiple of 8 (m = R/8): left term = suffix of lane l-m extended by the totals of lanes
// l-m+1 .. l+m-1 (folded in at the SENDER: one chain of 8 additions), right term = prefix of lane
// l+m.  Complete for lanes [m, 32-m).
template <int R>
__device__ __forceinline__ void gf_s8_window_m8(const float2 (&c)[4], float2 (&w)[4])
{
    constexpr int M = R / 8;
    static_assert(R % 8 == 0 && M >= 1 && M <= 4, "folded window sum needs R = 8, 16, 24, 32");
    const float x[8] = {c[0].x, c[0].y, c[1].x, c[1].y, c[2].x, c[2].y, c[3].x, c[3].y};
    // Prefixes and extended suffixes as shallow trees (dependency depth 4 instead of 8): the serial
    // chains left the warp waiting on FADD latency; the 4 extra additions per quantity are free.
    const float t01 = x[0] + x[1], t23 = x[2] + x[3], t45 = x[4] + x[5], t67 = x[6] + x[7];
    const float q03 = t01 + t23, q47 = t45 + t67;
    float p[8];
    p[0] = x[0]; p[1] = t01; p[2] = t01 + x[2]; p[3] = q03;
    p[4] = q03 + x[4]; p[5] = q03 + t45; p[6] = p[5] + x[6]; p[7] = q03 + q47;
    // totals of the following lanes: tn[d] = T(l+d)
    float tn[2 * M];
#pragma unroll
    for (int d = 1; d <= 2 * M - 1; ++d) tn[d] = GF_S8_SHFL_DOWN(p[7], d);
    float e = tn[1];
#pragma unroll
    for (int d = 2; d <= 2 * M - 1; ++d) e += tn[d];
    float a[8];
    a[7] = x[7] + e; a[6] = t67 + e;
    a[5] = x[5] + a[6]; a[4] = t45 + a[6];
    a[3] = x[3] + a[4]; a[2] = t23 + a[4];
    a[1] = x[1] + a[2]; a[0] = t01 + a[2];
    float l[8], r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) l[j] = GF_S8_SHFL_UP(a[j], M);
#pragma unroll
    for (int j = 0; j < 7; ++j) r[j] = GF_S8_SHFL_DOWN(p[j], M);
    r[7] = tn[M];
#pragma unroll
    for (int i = 0; i < 4; ++i) w[i] = gf_add2(make_float2(l[2 * i], l[2 * i + 1]), make_float2(r[2 * i], r[2 * i + 1]));
}

template <int R>
__device__ __forceinline__ void gf_s8_window(const float2 (&c)[4], float2 (&w)[4], int lane)
{
    if constexpr (R % 8 == 0) {
        gf_s8_window_m8<R>(c, w);
    } else {
        const float x[8] = {c[0].x, c[0].y, c[1].x, c[1].y, c[2].x, c[2].y, c[3].x, c[3].y};
        float o[8];
        gf_window_k<R, 8>(x, o, lane);
#pragma unroll
        for (int i = 0; i < 4; ++i) w[i] = make_float2(o[2 * i], o[2 * i + 1]);
    }
}

// ---- geometry ------------------------------------------------------------------------------------
template <int R>
struct GfS8Geom {
    static constexpr int H1 = (R + 7) / 8;           // halo lanes per side per stage
    static constexpr int VL = 32 - 4 * H1;           // lanes that produce output
    static constexpr int WOUT = 8 * VL;              // output columns per warp
    static constexpr int WIN = 256;                  // columns a warp loads
    static constexpr int KW = 2 * R + 1;
    static constexpr int SLOT_F2 = 2 * 4 * VL;       // float2 per ring row: [q][pair][cell]
    static constexpr size_t ring_bytes = (size_t)KW * SLOT_F2 * 8;
};

template <int R, class T = float>
struct GfS8Ctx {
    const T* gI; const T* gP; T* gQ;     // frame bases at (row buf_y0 / out_y0, this lane's first column)
    int gs, ss, ds;                                  // row strides; (rows * stride) fits 31 bits (host check)
    float2* ring;                                    // this lane's cell of ring row 0
    int lane, x0, width, height, border, buf_y0, buf_ylast, out_y0, yi0;
    bool vec_ok, ring_lane, out_lane;
    bool out_l, out_r;                               // MODE 3 only: lane lies left / right of the image
    int vofs, sofs;                                  // MODE 3 only: vector / scalar source offsets relative to x0
    bool lane_in;                                    // MODE 4 only: this lane's 8 columns lie inside the image
    float2 cx[4];                                    // MODE 4 only: in-image columns in the window [x-R, x+R] of each column
    int sx[8];                                       // XMAP only: source column of each of the 8 columns, relative to x0
    float eps;
    GfNorm nk;                                       // 1 / (2R+1)^2
    float2 cI[4], cP[4], cIP[4], cII[4], sA[4], sB[4], va[4], vb[4];
    float2 fI[4], fP[4], fIP[4], fII[4], fA[4], fB[4];   // re-seed accumulators
    float2 nI[4], nP[4], oI[4], oP[4];               // oI doubles as the guide row of the next output
    float sc[4];                                     // MODE 3 only: the mirror scalar of nI, nP, oI, oP (rows are held raw)
};

// single reflection (callers guarantee |overshoot| < n)
__device__ __forceinline__ int gf_s8_map_y(int y, int n, int border)
{
    const int e = border == GF_REFLECT ? 1 : 0;
    if (y < 0) y = -y - e;
    if (y >= n) y = 2 * n - 2 + e - y;
    return y;
}

__device__ __forceinline__ float gf_s8_rcp(float d)
{
#ifdef GF_CPU_EMU
    return 1.0f / d;
#else
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d));    // MUFU.RCP, no range fix-up: |d| is in [eps N^2, ~2 N^2]
    return r;
#endif
}

// Strip modes: 0 interior; 3 mirror loads -- REFLECT101,
// width % 8 == 0: a lane that lies outside the image reads the aligned 8-column group that holds
// 7 of its 8 mirror columns plus one scalar, and permutes at compile time (no per-column gather);
// 2 generic per-column border map (any border, any width; slow, rarely needed); 4 TRUNCATE border
// (the class API): pixels outside the image contribute nothing and every mean divides by the number of
// in-image pixels of its window (guided_filter_d.cu:251-262) -- zero-filled loads, per-pixel counts.
template <int MODE, int R, class T>
__device__ __forceinline__ void gf_s8_ld(const GfS8Ctx<R, T>& c, const T* rowp, float2 (&v)[4], float& sc)
{
    if (MODE == 3) {
        // RAW mirror data: the permutation is applied where the row is consumed (gf_s8_fix), one iteration later --
        // selects right behind the loads would make the warp wait for them here and expose the memory latency
        gf_ld8(rowp + c.vofs, v);
        sc = 0.f;                                       // only the lanes outside the image need the scalar (a predicated
        if (c.out_l || c.out_r) sc = gf_ld1(rowp + c.sofs);   // load: 1-2 wavefronts instead of 8 for the whole warp)
    } else if (MODE == 4) {
        if (c.lane_in) {
            gf_ld8(rowp, v);
        } else {
#pragma unroll
            for (int i = 0; i < 4; ++i) v[i] = make_float2(0.f, 0.f);
        }
    } else if (MODE != 2 || c.vec_ok) {
        gf_ld8(rowp, v);
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = make_float2(gf_ld1(rowp + c.sx[2 * i]), gf_ld1(rowp + c.sx[2 * i + 1]));
    }
}

// MODE 3: raw mirror data -> the lane's 8 columns
//   left of the image:  column -8k+j <- column 8k-j   = {sc, e7, e6, .., e1}
//   right of the image: column W+8m+j <- W-2-8m-j     = {e6, e5, .., e0, sc}
template <int MODE, int R, class T>
__device__ __forceinline__ void gf_s8_fix(const GfS8Ctx<R, T>& c, float2 (&v)[4], float sc)
{
    if (sizeof(T) == 1) {                               // uint8 build: the vector part of the row is still raw bytes
        if (MODE == 2) {                                // (lanes that gathered column by column already hold floats)
            float2 t[4] = {v[0], v[1], v[2], v[3]};
            gf_u8_expand(t);
#pragma unroll
            for (int i = 0; i < 4; ++i) v[i] = c.vec_ok ? t[i] : v[i];
        } else if (MODE == 4) {
            if (c.lane_in) gf_u8_expand(v);
        } else {
            gf_u8_expand(v);
        }
    }
    if (MODE != 3) return;
    const float e[8] = {v[0].x, v[0].y, v[1].x, v[1].y, v[2].x, v[2].y, v[3].x, v[3].y};
    float d[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float lv = j == 0 ? sc : e[8 - j];
        const float rv = j == 7 ? sc : e[6 - j];
        d[j] = c.out_l ? lv : (c.out_r ? rv : e[j]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = make_float2(d[2 * i], d[2 * i + 1]);
}

// Row y (any integer) of both planes: REFLECT borders map the row index; MODE 4 (TRUNCATE) rows outside
// the image are zeros.
template <int MODE, int R, class T>
__device__ __forceinline__ void gf_s8_ld_row(const GfS8Ctx<R, T>& c, int y, float2 (&vI)[4], float2 (&vP)[4], float& scI, float& scP)
{
    if (MODE == 4) {
        if (y < 0 || y > c.buf_ylast) {
#pragma unroll
            for (int i = 0; i < 4; ++i) { vI[i] = make_float2(0.f, 0.f); vP[i] = make_float2(0.f, 0.f); }
            return;
        }
        const int o = y - c.buf_y0;
        gf_s8_ld<MODE>(c, c.gI + o * c.gs, vI, scI);
        gf_s8_ld<MODE>(c, c.gP + o * c.ss, vP, scP);
    } else {
        int rn = gf_s8_map_y(y, c.height, c.border);
        rn = rn > c.buf_ylast ? c.buf_ylast : rn;
        const int o = rn - c.buf_y0;
        gf_s8_ld<MODE>(c, c.gI + o * c.gs, vI, scI);
        gf_s8_ld<MODE>(c, c.gP + o * c.ss, vP, scP);
    }
}

// TRUNCATE: number of image rows in [y-R, y+R]
template <int R>
__device__ __forceinline__ float gf_s8_cnt_y(int y, int height)
{
    const int lo = y - R < 0 ? 0 : y - R, hi = y + R > height - 1 ? height - 1 : y + R;
    return (float)(hi - lo + 1 > 0 ? hi - lo + 1 : 1);
}

// c = f, f = 0: f holds exactly the rows of the current window, summed without a subtraction
template <int R, class T>
__device__ __forceinline__ void gf_s8_reseed1(GfS8Ctx<R, T>& c)
{
    if (!GF_S8_RESEED1 || sizeof(T) != 4) return;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        c.cI[i] = c.fI[i]; c.cP[i] = c.fP[i]; c.cIP[i] = c.fIP[i]; c.cII[i] = c.fII[i];
        c.fI[i] = c.fP[i] = c.fIP[i] = c.fII[i] = make_float2(0.f, 0.f);
    }
}
template <int R, class T>
__device__ __forceinline__ void gf_s8_reseed2(GfS8Ctx<R, T>& c)
{
    if (!GF_S8_RESEED2) return;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        c.sA[i] = c.fA[i]; c.sB[i] = c.fB[i];
        c.fA[i] = c.fB[i] = make_float2(0.f, 0.f);
    }
}

// Iteration t >= 2R: phase A = stage 2 of the a, b row produced by iteration t-1 (ring row `slot`)
// and, once the stage-2 window is complete (`full`, t >= 4R+1), the output row t-1-2R; phase B =
// stage 1 of input row yi = yi0 + t.  ONE copy of this code per strip mode serves the whole band
// (instruction-cache footprint): ramp-up is data, not code -- the first a, b row (t = 2R) and the
// first "old" row are zeros, and while `full` is false the ring is written but not subtracted.
template <int R, int MODE, class T>
__device__ __forceinline__ void gf_s8_iter(GfS8Ctx<R, T>& c, int t, int slot, bool full)
{
    using G = GfS8Geom<R>;
    constexpr int KW = G::KW, VL = G::VL;
    constexpr bool XMAP = MODE == 2;
    const int yi = c.yi0 + t;
    const int lane = c.lane;

    // ================= phase B, part 1: vertical sums of row yi =================
    // (first, so that the loads of the next iteration can be issued right away and have a whole
    // iteration to land)
    gf_s8_fix<MODE>(c, c.nI, c.sc[0]); gf_s8_fix<MODE>(c, c.nP, c.sc[1]);
    gf_s8_fix<MODE>(c, c.oI, c.sc[2]); gf_s8_fix<MODE>(c, c.oP, c.sc[3]);
    float2 gI[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) gI[i] = c.oI[i];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        c.cI[i] = gf_add2(c.cI[i], gf_sub2(c.nI[i], c.oI[i]));
        c.cP[i] = gf_add2(c.cP[i], gf_sub2(c.nP[i], c.oP[i]));
        c.cIP[i] = gf_fma2(gf_neg2(c.oI[i]), c.oP[i], gf_fma2(c.nI[i], c.nP[i], c.cIP[i]));
        c.cII[i] = gf_fma2(gf_neg2(c.oI[i]), c.oI[i], gf_fma2(c.nI[i], c.nI[i], c.cII[i]));
        if (GF_S8_RESEED1 && sizeof(T) == 4) {       // (uint8 build: integer sums below 2^24 are exact)
            c.fI[i] = gf_add2(c.fI[i], c.nI[i]);
            c.fP[i] = gf_add2(c.fP[i], c.nP[i]);
            c.fIP[i] = gf_fma2(c.nI[i], c.nP[i], c.fIP[i]);
            c.fII[i] = gf_fma2(c.nI[i], c.nI[i], c.fII[i]);
        }
    }
    // rows of the next iteration, consumed at the top of it
    if (!(GF_S8_ABL & 4)) {
        gf_s8_ld_row<MODE>(c, yi + 1, c.nI, c.nP, c.sc[0], c.sc[1]);
        gf_s8_ld_row<MODE>(c, yi + 1 - KW, c.oI, c.oP, c.sc[2], c.sc[3]);
        if (GF_S8_PF > 0 && MODE <= 1 && lane < 8) {
            // L2 prefetch hint a few rows ahead: 8 lanes x one 128-byte line = the warp's 256 columns.
            // (Measured: +3% over no hint; a hint per 32-byte sector from all 32 lanes is 10% SLOWER.)
            const int rp = yi + 1 + GF_S8_PF;
            if (rp <= c.buf_ylast) {
                const int op = rp - c.buf_y0;
                constexpr int LINE = 128 / (int)sizeof(T);      // elements per 128-byte line
                if (lane * LINE < 256) {
                    gf_prefetch_l2(c.gI + op * c.gs + (LINE - 8) * lane);
                    gf_prefetch_l2(c.gP + op * c.ss + (LINE - 8) * lane);
                }
            }
        }
    }
    // ================= phase A: stage 2 of centre row yi-1-R (guide row of its output: gI) =================
    {
        float2 hA[4], hB[4];
        gf_s8_window<R>(c.va, hA, lane);
        gf_s8_window<R>(c.vb, hB, lane);
        if (c.ring_lane && !(GF_S8_ABL & 2)) {
            float2* s = c.ring + slot * G::SLOT_F2;
            if (full) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    c.sA[i] = gf_add2(c.sA[i], gf_sub2(hA[i], s[i * VL]));
                    c.sB[i] = gf_add2(c.sB[i], gf_sub2(hB[i], s[(4 + i) * VL]));
                }
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) { c.sA[i] = gf_add2(c.sA[i], hA[i]); c.sB[i] = gf_add2(c.sB[i], hB[i]); }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) { s[i * VL] = hA[i]; s[(4 + i) * VL] = hB[i]; }
        }
        if (GF_S8_RESEED2) {
#pragma unroll
            for (int i = 0; i < 4; ++i) { c.fA[i] = gf_add2(c.fA[i], hA[i]); c.fB[i] = gf_add2(c.fB[i], hB[i]); }
        }
        if (full) {                                     // q of row yo = yi-1-2R; its guide row is oI
            const int yo = yi - 1 - 2 * R;
            float2 q[4];
            if (MODE == 4) {                           // mean over the in-image part of the window of (x, yo)
                const float2 cy = gf_dup2(gf_s8_cnt_y<R>(yo, c.height));
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float2 n2 = gf_mul2(c.cx[i], cy);
                    float2 rn = make_float2(gf_s8_rcp(n2.x), gf_s8_rcp(n2.y));
                    rn = gf_fma2(gf_fma2(gf_neg2(n2), rn, gf_dup2(1.0f)), rn, rn);
                    q[i] = gf_mul2(gf_fma2(c.sA[i], gI[i], c.sB[i]), rn);
                }
            } else {
                const float2 nh = gf_dup2(c.nk.hi), nl = gf_dup2(c.nk.lo);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float2 v = gf_fma2(c.sA[i], gI[i], c.sB[i]);
                    q[i] = gf_fma2(v, nh, gf_mul2(v, nl));
                }
            }
            T* pq = c.gQ + (yo - c.out_y0) * c.ds;
            if (c.out_lane && !(GF_S8_ABL & 8)) {
                if (!XMAP || c.vec_ok) {
                    gf_st8(pq, q);
                } else {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        if (c.x0 + 2 * i >= 0 && c.x0 + 2 * i < c.width) gf_st1(pq + 2 * i, q[i].x);
                        if (c.x0 + 2 * i + 1 >= 0 && c.x0 + 2 * i + 1 < c.width) gf_st1(pq + 2 * i + 1, q[i].y);
                    }
                }
            }
        }
    }

    // ================= phase B, part 2 =================
    {
        // horizontal -> a, b of row yi - R.  Every window is full (REFLECT borders mirror the data):
        //   a = (N S_Ip - S_I S_p) / (N S_II - S_I^2 + eps N^2),   b = (S_p - a S_I) / N
        float2 hI[4], hP[4], hIP[4], hII[4];
        gf_s8_window<R>(c.cI, hI, lane);
        gf_s8_window<R>(c.cP, hP, lane);
        gf_s8_window<R>(c.cIP, hIP, lane);
        gf_s8_window<R>(c.cII, hII, lane);
        if (MODE == 4) {
            // TRUNCATE: N = (in-image columns) x (in-image rows) of the window of (x, yc); a, b are zero outside the image
            const int yc = yi - R;
            const bool ok = c.lane_in && yc >= 0 && yc < c.height;
            const float2 cy = gf_dup2(gf_s8_cnt_y<R>(yc, c.height));
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float2 n2 = gf_mul2(c.cx[i], cy), mn2 = gf_neg2(n2);
                const float2 nnum = gf_fma2(hI[i], hP[i], gf_mul2(hIP[i], mn2));
                const float2 nden = gf_fma2(hI[i], hI[i], gf_fma2(hII[i], mn2, gf_mul2(gf_mul2(n2, n2), gf_dup2(-c.eps))));
                float2 rc = make_float2(gf_s8_rcp(nden.x), gf_s8_rcp(nden.y));
                rc = gf_fma2(gf_fma2(gf_neg2(nden), rc, gf_dup2(1.0f)), rc, rc);
                float2 rn = make_float2(gf_s8_rcp(n2.x), gf_s8_rcp(n2.y));
                rn = gf_fma2(gf_fma2(mn2, rn, gf_dup2(1.0f)), rn, rn);
                const float2 aa = gf_mul2(nnum, rc);
                const float2 bb = gf_mul2(gf_fma2(gf_neg2(aa), hI[i], hP[i]), rn);
                c.va[i] = ok ? aa : make_float2(0.f, 0.f);
                c.vb[i] = ok ? bb : make_float2(0.f, 0.f);
            }
            return;
        }
        const float N = (float)(KW * KW);
        const float2 mN = gf_dup2(-N), mE = gf_dup2(-c.eps * N * N);
        const float2 nh = gf_dup2(c.nk.hi), nl = gf_dup2(c.nk.lo);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 nnum = gf_fma2(hI[i], hP[i], gf_mul2(hIP[i], mN));           // -(numerator)
            const float2 nden = gf_fma2(hI[i], hI[i], gf_fma2(hII[i], mN, mE));       // -(denominator) < 0
            float2 rc = make_float2(gf_s8_rcp(nden.x), gf_s8_rcp(nden.y));
            if (GF_S8_NEWTON) {
                const float2 e = gf_fma2(gf_neg2(nden), rc, gf_dup2(1.0f));
                rc = gf_fma2(e, rc, rc);
            }
            const float2 aa = gf_mul2(nnum, rc);
            const float2 bn = gf_fma2(gf_neg2(aa), hI[i], hP[i]);                      // N * b
            c.va[i] = aa;
            c.vb[i] = gf_fma2(bn, nh, gf_mul2(bn, nl));
        }
    }
}

// Warm-up rows t in [0, 2R): vertical accumulation only.  Nothing else is going on, so a single
// row in flight would expose the full DRAM latency 2R times; rows are loaded CH at a time instead.
// On entry nI/nP hold row yi0 (t = 0); on exit they hold row yi0 + 2R.
template <int R, int MODE, class T>
__device__ __forceinline__ void gf_s8_warmup(GfS8Ctx<R, T>& c)
{
    constexpr int CH = 4, NROWS = 2 * R;
    float2 bI[CH][4], bP[CH][4];
    float bsI[CH], bsP[CH];
#pragma unroll 1
    for (int t0 = 0; t0 < NROWS; t0 += CH) {
        // rows t0+1 .. t0+CH  (row t0 is already in nI/nP)
#pragma unroll
        for (int k = 0; k < CH; ++k) {
            gf_s8_ld_row<MODE>(c, c.yi0 + t0 + 1 + k, bI[k], bP[k], bsI[k], bsP[k]);
        }
#pragma unroll
        for (int k = 0; k < CH; ++k) {
            if (t0 + k < NROWS) {
                gf_s8_fix<MODE>(c, c.nI, c.sc[0]); gf_s8_fix<MODE>(c, c.nP, c.sc[1]);
                c.sc[0] = bsI[k]; c.sc[1] = bsP[k];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    c.cI[i] = gf_add2(c.cI[i], c.nI[i]);
                    c.cP[i] = gf_add2(c.cP[i], c.nP[i]);
                    c.cIP[i] = gf_fma2(c.nI[i], c.nP[i], c.cIP[i]);
                    c.cII[i] = gf_fma2(c.nI[i], c.nI[i], c.cII[i]);
                    c.nI[i] = bI[k][i]; c.nP[i] = bP[k][i];
                }
            }
        }
    }
}

// The row loop of one band: 2R warm-up rows, then iterations t = 2R .. steps in periods of 2R+1
// (= ring length = re-seed period; the inner loop is straight-line code, `slot` is its counter).
// The last iteration only needs its phase A; its phase B works on clamped rows and is discarded.
template <int R, int MODE, class T>
__device__ __forceinline__ void gf_s8_band(GfS8Ctx<R, T>& c, int steps)
{
    constexpr int KW = 2 * R + 1;
    gf_s8_warmup<R, MODE>(c);
    int t = 2 * R;
    bool full = false;
#pragma unroll 1
    while (t <= steps) {
        const int n = steps + 1 - t < KW ? steps + 1 - t : KW;
#pragma unroll 1
        for (int s = 0; s < n; ++s, ++t) gf_s8_iter<R, MODE>(c, t, s, full);
        if (n == KW) {
            gf_s8_reseed1(c);
            gf_s8_reseed2(c);
        }
        full = true;
    }
}

// Strip geometry: strip s outputs columns [s * WOUT, (s + 1) * WOUT) and reads 2 * H1 lanes of halo
// on either side.  Strips that overhang the image use mirror loads (MODE 3: REFLECT101,
// width % 8 == 0), clipped counts (MODE 4: TRUNCATE) or the generic per-column border map (MODE 2).
template <int R, int MINB, class T>
__global__ void __launch_bounds__(32, MINB) gf_s8_gray_kernel(const GF_GRID_CONSTANT GfWpArgs a)
{
    using G = GfS8Geom<R>;
    constexpr int H1 = G::H1, KW = G::KW, VL = G::VL;
    GF_DYN_SMEM(float, smem);
    auto run = [&](int64_t f, int strip, int yo0, int yo1) {
    GfS8Ctx<R, T> c;
    c.lane = threadIdx.x & 31;
    const int xl = strip * G::WOUT - 2 * H1 * 8, lane_lo = 2 * H1;
    int mode = 0;
    if (a.border == GF_TRUNCATE) {
        // interior warps (every window they touch is full) run the plain code; the others count pixels
        const bool inside = xl >= 0 && xl + G::WIN <= a.width && yo0 - 2 * R >= 0 && yo1 + 2 * R <= a.height;
        mode = inside ? 0 : 4;
    } else if (xl < 0 || xl + G::WIN > a.width) {
        mode = (a.border == GF_REFLECT101 && (a.width & 7) == 0 && a.width >= G::WIN) ? 3 : 2;
    }
    c.x0 = xl + 8 * c.lane;
    // (GfWpArgs carries the planes as float*; T = unsigned char builds reinterpret them, strides are in elements)
    c.gI = reinterpret_cast<const T*>(a.guide) + f * a.gfs + c.x0; c.gP = reinterpret_cast<const T*>(a.src) + f * a.sfs + c.x0;
    c.gQ = reinterpret_cast<T*>(a.dst) + f * a.dfs + c.x0;
    c.gs = (int)a.gs; c.ss = (int)a.ss; c.ds = (int)a.ds;
    c.ring_lane = c.lane >= lane_lo && c.lane < lane_lo + VL;
    c.out_lane = c.ring_lane && c.x0 < a.width;
    c.ring = reinterpret_cast<float2*>(smem) + (c.ring_lane ? c.lane - lane_lo : 0);
    c.width = a.width; c.height = a.height; c.border = a.border; c.buf_y0 = a.buf_y0; c.out_y0 = a.out_y0;
    {
        const int yl = a.buf_y0 + a.buf_rows - 1;
        c.buf_ylast = yl < a.height - 1 ? yl : a.height - 1;
    }
    c.vec_ok = c.x0 >= 0 && c.x0 + 7 < a.width;
    c.lane_in = c.vec_ok;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        c.cx[i] = make_float2(gf_count(c.x0 + 2 * i, a.width, R, GF_TRUNCATE), gf_count(c.x0 + 2 * i + 1, a.width, R, GF_TRUNCATE));
    c.out_l = mode == 3 && c.x0 < 0;
    c.out_r = mode == 3 && c.x0 >= a.width;
    c.vofs = c.out_l ? -2 * c.x0 - 8 : (c.out_r ? 2 * a.width - 8 - 2 * c.x0 : 0);
    c.sofs = c.out_l ? -2 * c.x0 : (c.out_r ? 2 * a.width - 9 - 2 * c.x0 : 0);
    c.yi0 = yo0 - 2 * R;
    c.eps = sizeof(T) == 4 ? a.eps : a.eps * 65025.0f;      // uint8 build: integer domain, eps scales with 255^2
    c.nk = gf_norm_make((float)(KW * KW));
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        c.cI[i] = c.cP[i] = c.cIP[i] = c.cII[i] = c.sA[i] = c.sB[i] = c.va[i] = c.vb[i] = make_float2(0.f, 0.f);
        c.fI[i] = c.fP[i] = c.fIP[i] = c.fII[i] = c.fA[i] = c.fB[i] = make_float2(0.f, 0.f);
        c.oI[i] = c.oP[i] = make_float2(0.f, 0.f);
    }
    c.sc[0] = c.sc[1] = c.sc[2] = c.sc[3] = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) c.sx[j] = mode == 2 ? gf_map(c.x0 + j, a.width, a.border) - c.x0 : j;

    const int steps = (yo1 - yo0) + 4 * R;
    const int o0 = gf_s8_map_y(c.yi0, a.height, a.border) - a.buf_y0;       // row of iteration 0
    if (mode == 2) {
        gf_s8_ld<2>(c, c.gI + o0 * c.gs, c.nI, c.sc[0]); gf_s8_ld<2>(c, c.gP + o0 * c.ss, c.nP, c.sc[1]);
        gf_s8_band<R, 2>(c, steps);
    } else if (mode == 3) {
        gf_s8_ld<3>(c, c.gI + o0 * c.gs, c.nI, c.sc[0]); gf_s8_ld<3>(c, c.gP + o0 * c.ss, c.nP, c.sc[1]);
        gf_s8_band<R, 3>(c, steps);
    } else if (mode == 4) {
        gf_s8_ld_row<4>(c, c.yi0, c.nI, c.nP, c.sc[0], c.sc[1]);
        gf_s8_band<R, 4>(c, steps);
    } else {
        gf_s8_ld<0>(c, c.gI + o0 * c.gs, c.nI, c.sc[0]); gf_s8_ld<0>(c, c.gP + o0 * c.ss, c.nP, c.sc[1]);
        gf_s8_band<R, 0>(c, steps);
    }
    };
    gf_tape_run(a, (long long)blockIdx.x, run);
}

// ---- host side ------------------------------------------------------------------------------------
#ifndef GF_NO_HOST   // (stand-alone SASS builds of one kernel define GF_NO_HOST)
// Band height for a grid of 1-warp CTAs that all take the same time: CTAs run in waves of `slots`
// (resident warps of the whole GPU), an item costs its rows plus the ramp (2R cheap warm-up rows
// and 2R+1 full iterations without output), so   time ~ ceil(items / slots) * (hb + ramp).
// Returns the hb that minimises it (ties: fewer, taller bands).
static inline int gf_pick_band_rows(int rows, int r, long nstrips_x_count, long slots, int hb_min)
{
    const double ramp = 2.3 * r + 1.0;
    int best_hb = rows;
    double best = 1e300;
    const int nb_max = rows / (hb_min > 0 ? hb_min : 1) > 0 ? rows / (hb_min > 0 ? hb_min : 1) : 1;
    for (int nb = 1; nb <= nb_max && nb <= 4096; ++nb) {
        const int hb = (rows + nb - 1) / nb;
        const long items = nstrips_x_count * ((rows + hb - 1) / hb);
        const long waves = (items + slots - 1) / slots;
        const double cost = (double)waves * (hb + ramp);
        if (cost < best * 0.999) { best = cost; best_hb = hb; }
    }
    return best_hb;
}

// Tape plan (gf_tape_run in gf_wp.cuh): fills a.tape_* and returns the grid size (one 1-warp CTA per
// piece, at most `slots` so that the job is one wave; pieces are at least hb_min rows + one ramp long).
// EXPERIMENT, off unless GF_TAPE=1: on B200 it measured 2-25 % SLOWER than the uniform split on
// every gray case and on large colour batches, and only 3-8 % faster on 16-32 frame colour batches
// (profiles/r1_tape_scheduling_ab.jsonl, profiles/r1_c4_band_sweep.jsonl): pieces of neighbouring
// strips no longer walk the same rows at the same time, so the strip halos stop hitting in L2, and
// a piece that crosses into the next strip pays a second ramp that costs more than the model says.
static inline long gf_tape_plan(GfWpArgs& a, int r, long slots, int hb_min, int we_pct, int on_by_default = 0)
{
    a.tape_piece = 0; a.tape_rho = (int)(2.3 * r + 1.0); a.tape_we = we_pct < 100 ? 100 : we_pct;
    if (GF_KNOB("GF_TAPE", on_by_default) == 0) return 0;
    slots = GF_KNOB("GF_TAPE_SLOTS", (int)slots);       // tests / experiments: pieces that span several strips
    const bool edges = a.nstrips >= 3 && a.tape_we != 100;
    const long long zi = (long long)(a.tape_rho + a.out_rows) * 100, ze = (long long)(a.tape_rho + a.out_rows) * a.tape_we;
    const long long total = (edges ? 2 * ze + (a.nstrips - 2) * zi : a.nstrips * zi) * a.count;
    const long long min_piece = (long long)(hb_min + a.tape_rho) * 100;
    long long n = total / min_piece;
    if (n > slots) n = slots;
    if (n < 1) n = 1;
    a.tape_piece = (total + n - 1) / n;
    return (long)((total + a.tape_piece - 1) / a.tape_piece);
}

#ifndef GF_S8_NO_TRY     // (translation units that only need the helpers above: gf_tu_ws.cu, gf_tu_c4.cu, gf_api.cu)
template <int R, class T = float>
static const char* gf_s8_launch(const Job& j)
{
    using G = GfS8Geom<R>;
    static_assert(G::VL >= 8, "too few output lanes");
    int sms = 148, mj = 0, mn = 0;
    gf_rt_device_info(&sms, &mj, &mn);
    GfWpArgs a;
    a.guide = j.guide.ptr; a.src = j.src.ptr; a.dst = const_cast<float*>(j.dst.ptr);
    a.A = nullptr; a.B = nullptr;
    a.gs = j.guide.stride; a.ss = j.src.stride; a.ds = j.dst.stride; a.abs_ = 0;
    a.gfs = j.guide.frame_stride; a.sfs = j.src.frame_stride; a.dfs = j.dst.frame_stride; a.abfs = 0;
    a.width = j.width; a.height = j.height; a.buf_y0 = j.buf_y0; a.buf_rows = j.buf_rows; a.out_y0 = j.out_y0;
    a.out_rows = j.out_rows; a.border = j.border; a.eps = j.eps; a.count = j.count;
    a.tape_piece = 0; a.tape_rho = 0; a.tape_we = 100;
    a.nstrips = (j.width + G::WOUT - 1) / G::WOUT;
    size_t smem = G::ring_bytes;
    smem += (size_t)GF_KNOB("GF_S8_EXTRA_SMEM", 0);      // experiments: lower the residency
    // resident warps per SM: the ring in shared memory (228 kB per SM, 1 kB reserved per CTA).  A ring
    // in global memory (L2) would lift this limit but measured 1.6x slower (DESIGN.md section 3).
    int warps_sm = (int)((size_t)228 * 1024 / (smem + 1024));
    if (warps_sm > 8) warps_sm = 8;
    if (warps_sm < 1) warps_sm = 1;
    warps_sm = GF_KNOB("GF_S8_WARPS_PER_SM", warps_sm);
    if (warps_sm < 1) warps_sm = 1;
    // Bands: waves of resident warps x (band rows + ramp), see gf_pick_band_rows
    int hb_min = 2 * R + 8;
    hb_min = GF_KNOB("GF_S8_HB_MIN", hb_min);
    int hb = gf_pick_band_rows(j.out_rows, R, (long)a.nstrips * j.count, (long)sms * warps_sm, hb_min);
    hb = GF_KNOB("GF_S8_HB", hb);
    if (hb < 1) hb = 1;
    if (hb > j.out_rows) hb = j.out_rows;
    a.hb = hb;
    a.nbands = (j.out_rows + hb - 1) / hb;
    // The two edge strips run slower code (mirror loads / clipped counts, ~15 % more instructions):
    // they get shorter bands, in proportion.  Measured on B200
    // (profiles/r1_s8_edge_band_pct.txt): 4K r=16 90.9 -> 85.7 us, 8K r=32 515 -> 483 us, 4K r=8 66.2 -> 65.1 us.
    int edge_pct = GF_S8_EDGE_PCT;
    edge_pct = GF_KNOB("GF_S8_EDGE_PCT", edge_pct);
    a.hb_e = 0; a.nbands_e = 0;
    if (a.nstrips >= 3 && edge_pct > 0 && edge_pct < 100 && a.nbands > 1) {
        const long slots = (long)sms * warps_sm;
        const bool one_wave = (long)a.nstrips * a.nbands * j.count <= slots;
        for (;;) {
            int hbe = hb * edge_pct / 100;
            if (hbe < hb_min) hbe = hb_min;
            if (hbe >= hb) { a.hb_e = 0; a.nbands_e = 0; break; }
            a.hb_e = hbe; a.nbands_e = (j.out_rows + hbe - 1) / hbe;
            a.nbands = (j.out_rows + hb - 1) / hb;
            const long items = (2L * a.nbands_e + (long)(a.nstrips - 2) * a.nbands) * j.count;
            if (!one_wave || items <= slots || hb >= j.out_rows) break;     // a job that fitted one wave must still fit
            ++hb;
        }
        a.hb = hb;
        a.nbands = (j.out_rows + hb - 1) / hb;
    }
    const long per_frame = a.nbands_e > 0 ? 2L * a.nbands_e + (long)(a.nstrips - 2) * a.nbands : (long)a.nstrips * a.nbands;
    long items = per_frame * j.count;
    if (!GF_KNOB_SET("GF_S8_HB"))
        if (const long n = gf_tape_plan(a, R, (long)sms * warps_sm, hb_min, edge_pct > 0 && edge_pct < 100 ? 10000 / edge_pct : 100)) items = n;
    dim3 grid((unsigned)items), block(32);
    constexpr int FIT = (int)((size_t)228 * 1024 / (G::ring_bytes + 1024));
    constexpr int MINB = FIT > 7 ? 7 : (FIT < 1 ? 1 : FIT);
    auto k = gf_s8_gray_kernel<R, MINB, T>;
    if (const char* e = gf_rt_set_smem(k, smem)) return e;
    GF_LAUNCH(k, grid, block, smem, j.stream, a);
    return gf_rt_launch_error();
}

// u8 = true: the planes hold unsigned char (Plane::ptr reinterpreted, strides in elements): uint8 in,
// uint8 out, conversions fused into the loads and stores (gf_guided_gray_u8).
static const char* gf_s8_try(const Job& j, bool* done, const char** name, bool u8 = false)
{
    *done = false;
    if (j.color || j.A.ptr) return nullptr;
    if (j.border == GF_TRUNCATE && ((j.width & 7) || j.width < 256)) return nullptr;
    if (!u8 && (GF_KNOB("GF_DISABLE_S8", 0) || GF_KNOB("GF_DISABLE_FAST", 0))) return nullptr;
    const Plane* pl[3] = {&j.guide, &j.src, &j.dst};
    const uintptr_t amask = u8 ? 7 : 31;                  // one 8-byte / 32-byte vector per lane and row
    for (int i = 0; i < 3; ++i)
        if (pl[i]->channels != 1 || pl[i]->coff != 0 || (pl[i]->stride & 7) || (pl[i]->frame_stride & 7) ||
            ((uintptr_t)pl[i]->ptr & amask))
            return nullptr;
    // row offsets inside a frame are 32-bit in the kernel
    if ((int64_t)j.buf_rows * j.guide.stride >= (1ll << 31) || (int64_t)j.buf_rows * j.src.stride >= (1ll << 31) ||
        (int64_t)j.out_rows * j.dst.stride >= (1ll << 31))
        return nullptr;
    // single reflections only, and at least one full warp window of columns
    if (j.height < 4 * j.r + 2 || j.width < 4 * j.r + 2 || j.width < 64) return nullptr;
    if (u8) {
        switch (j.r) {
#define GF_S8_CASE(RR) case RR: *done = true; *name = "s8u8_r" #RR; return gf_s8_launch<RR, unsigned char>(j);
#ifdef GF_CPU_EMU
        GF_S8_CASE(4) GF_S8_CASE(7) GF_S8_CASE(8) GF_S8_CASE(16)
#else      // every radius of the reference's sweep (run.py:4-6: r = 1..7) plus the BASELINE radii
        GF_S8_CASE(1) GF_S8_CASE(2) GF_S8_CASE(3) GF_S8_CASE(4) GF_S8_CASE(5) GF_S8_CASE(6) GF_S8_CASE(7) GF_S8_CASE(8) GF_S8_CASE(16)
#endif
#undef GF_S8_CASE
        default: return nullptr;
        }
    }
    switch (j.r) {
#define GF_S8_CASE(RR) case RR: *done = true; *name = "s8_r" #RR; return gf_s8_launch<RR>(j);
#ifdef GF_CPU_EMU   // the test-only emulator build keeps its compile time down: one radius per code shape
    GF_S8_CASE(4) GF_S8_CASE(7) GF_S8_CASE(8) GF_S8_CASE(16) GF_S8_CASE(32)
#else
    GF_S8_CASE(1) GF_S8_CASE(2) GF_S8_CASE(3) GF_S8_CASE(4) GF_S8_CASE(5) GF_S8_CASE(6) GF_S8_CASE(7) GF_S8_CASE(8)
    GF_S8_CASE(10) GF_S8_CASE(12) GF_S8_CASE(16) GF_S8_CASE(20) GF_S8_CASE(24) GF_S8_CASE(32)
#endif
#undef GF_S8_CASE
    default: return nullptr;
    }
}
#endif  // GF_S8_NO_TRY
#endif  // GF_NO_HOST
