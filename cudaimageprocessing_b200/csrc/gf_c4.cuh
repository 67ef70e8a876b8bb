// gf_c4.cuh -- tuned colour-guide kernel (3-channel interleaved guide, 1-channel src/dst, float32):
// the 3x3-covariance guided filter of He et al. (TPAMI 2013, eqs. 19-21), fused in one pass.
// The reference has no colour-guide implementation (guided_filter_d.cu:976-979 refuses it); the
// arithmetic follows oracle/gf_oracle.py::guided_filter_color and GfColorModel (gf_generic.cuh).
//
// Same architecture as gf_s8.cuh, sized for 13 + 4 box-filtered quantities instead of 4 + 2:
//   * every WARP is an independent worker; a lane owns 4 ADJACENT columns (13 x 4 vertical running
//     sums in registers; 8 columns per lane would need 104 and spill);
//   * stage 1: vertical running sums of I_r, I_g, I_b, p, I_c p (3), I_c I_d (6); horizontal
//     (2R+1)-window sums across lanes with the folded scheme of gf_s8 (left term = suffix of lane
//     l-M extended by the totals of the 2M-1 lanes in between, right term = prefix of lane l+M,
//     M = R/4; 13 shuffles and 15 additions per quantity and 4 pixels at R = 16, additions only);
//     per pixel the symmetric 3x3 system (Sigma + eps U) a = cov(I, p) by cofactors;
//   * stage 2: window sums of a_r, a_g, a_b, b, vertical running sums through a (2R+1)-row ring in
//     shared memory (one float4 per lane, quantity and row: conflict-free LDS.128/STS.128);
//   * q = mean_a . I + mean_b; the guide row of the output is the row that leaves the stage-1
//     window in the same iteration (re-read from L2, never parked);
//   * image borders (width % 4 == 0), template BM: 0 REFLECT101 and 1 REFLECT -- lanes outside the image take
//     their rows from the mirror lanes by shuffle (32 extra SHFL per iteration, border strips only); 2 TRUNCATE
//     (the class API's border, guided_filter.cpp:22-60) -- rows and lanes outside the image are zeros and every
//     mean divides by its own in-image pixel count; any other width uses the generic kernel.
// R must be a multiple of 4 and <= 16 (M <= 4 halo lanes per side and stage).
//
// T = unsigned char: the same kernel on 8-bit planes (gf_guided_color_u8), in the integer domain of the gray
// uint8 build (gf_s8.cuh): I' = 255 I and p' = 255 p are the bytes as floats 0..255, the host passes
// eps' = 255^2 eps, and q' = 255 q is rounded and saturated by the store.  The stage-1 column sums are then
// integers below 33 x 255^2 < 2^24, exact in float32.  A row is kept raw (3 guide words, 1 or 3 src words)
// and expanded where it is consumed.  The frames of a launch are the source channels (count = 1 or 3,
// frame strides 0): frame f reads and writes byte f of every interleaved src / dst pixel.
#pragma once
#include "gf_s8.cuh"

template <int R>
struct GfC4Geom {
    static constexpr int M = R / 4;                  // halo lanes per side per stage
    static constexpr int VL = 32 - 4 * M;            // lanes that produce output
    static constexpr int WOUT = 4 * VL;              // output columns per warp
    static constexpr int WIN = 128;                  // columns a warp loads
    static constexpr int KW = 2 * R + 1;
    static constexpr int SLOT_F4 = 4 * VL;           // float4 per ring row: [q][cell]
    static constexpr size_t ring_bytes = (size_t)KW * SLOT_F4 * 16;
};

// (2R+1)-window sums of the 4 columns of every lane; complete for lanes [M, 32-M).
template <int R>
__device__ __forceinline__ void gf_c4_window(const float (&x)[4], float (&w)[4])
{
    constexpr int M = R / 4;
    static_assert(R % 4 == 0 && M >= 1 && M <= 4, "gf_c4 needs R = 4, 8, 12 or 16");
    const unsigned full = 0xffffffffu;
    const float p0 = x[0], p1 = x[0] + x[1], p2 = p1 + x[2], T = (x[0] + x[1]) + (x[2] + x[3]);
    // e = T(l+1) + .. + T(l+2M-1)
    float e;
    if (M == 1) {
        e = __shfl_down_sync(full, T, 1);
    } else {
        const float u2 = T + __shfl_down_sync(full, T, 1);                     // T(l..l+1)
        float s;                                                               // T(l..l+2M-2)
        if (M == 2) s = u2 + __shfl_down_sync(full, T, 2);
        else if (M == 3) s = (u2 + __shfl_down_sync(full, u2, 2)) + __shfl_down_sync(full, T, 4);
        else s = (u2 + __shfl_down_sync(full, u2, 2)) + (__shfl_down_sync(full, u2, 4) + __shfl_down_sync(full, T, 6));
        e = __shfl_down_sync(full, s, 1);
    }
    const float a3 = x[3] + e, a2 = (x[2] + x[3]) + e, a1 = x[1] + a2, a0 = T + e;
    const float l0 = __shfl_up_sync(full, a0, M), l1 = __shfl_up_sync(full, a1, M), l2 = __shfl_up_sync(full, a2, M),
                l3 = __shfl_up_sync(full, a3, M);
    const float r0 = __shfl_down_sync(full, p0, M), r1 = __shfl_down_sync(full, p1, M), r2 = __shfl_down_sync(full, p2, M),
                r3 = __shfl_down_sync(full, T, M);
    w[0] = l0 + r0; w[1] = l1 + r1; w[2] = l2 + r2; w[3] = l3 + r3;
}

template <int R, class T = float>
struct GfC4Ctx {
    const T* gI; const T* gP; T* gQ;                 // frame bases at this lane's first column (gI: 3 elements per column)
    int gs, ss, ds;
    float4* ring;
    int lane, x0, width, height, border, buf_y0, buf_ylast, out_y0, yi0;
    bool ring_lane, out_lane, mirror, out_l, out_r, src_l;   // mirror: this warp overhangs the image
    int s0, s1, s2;                                  // mirror source lanes for column j = 0, j = 1..2, j = 3
    float eps;
    float icx[4];                                    // BM 2: 1 / (in-image columns of the window of column j)
    bool nz, oz;                                     // BM 2: nI/nP (oI/oP) stand for a row outside the image: zeros
    float c[13][4];                                  // stage-1 column sums
    float sa[4][4];                                  // stage-2 running sums (a_r, a_g, a_b, b)
    float va[4][4];                                  // a, b of the row produced by the previous iteration
    float nI[12], nP[4], oI[12], oP[4];              // newest row / row leaving the window (= guide row of the output)
    bool p3;                                         // uint8 only: 3-channel src / dst (gQ then points at channel ch)
    unsigned selA, selB;                             // uint8 only: byte selectors of the src words (gf_c4_expand)
};

// uint8 build: a raw row (vi[0..2]: the 12 guide bytes; vp[0..2]: the src words, as float bit patterns) -> floats 0..255.
// The src pixels are gathered into one word first: 1 channel: bytes 0..3 of vp[0] (= vp[1]); 3 channels: pixel j,
// channel ch is byte 3j + ch of the 12 bytes, i.e. byte ch, 3 + ch of (vp[0], vp[1]) and 2 + ch, 5 + ch of (vp[1], vp[2]).
template <int R, class T>
__device__ __forceinline__ void gf_c4_expand(const GfC4Ctx<R, T>& c, float (&vi)[12], float (&vp)[4])
{
    const unsigned g0 = gf_f_bits(vi[0]), g1 = gf_f_bits(vi[1]), g2 = gf_f_bits(vi[2]);
    const unsigned w0 = gf_f_bits(vp[0]), w1 = gf_f_bits(vp[1]), w2 = gf_f_bits(vp[2]);
    const unsigned pw = gf_prmt(gf_prmt(w0, w1, c.selA), gf_prmt(w1, w2, c.selB), 0x7610u);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        vi[k] = gf_u8_to_f(g0, k); vi[4 + k] = gf_u8_to_f(g1, k); vi[8 + k] = gf_u8_to_f(g2, k);
        vp[k] = gf_u8_to_f(pw, k);
    }
}

// Raw loads of one row: 12 guide floats (3 x LDG.128) and 4 src floats.  A lane outside the image
// loads its mirror lane's address instead (any valid address would do) and is patched by gf_c4_mirror.
// uint8: 12 guide bytes (3 x LDG.32) and 4 (1 x LDG.32) or 12 src bytes, kept raw for gf_c4_expand.
template <int R, class T>
__device__ __forceinline__ void gf_c4_ld(const GfC4Ctx<R, T>& c, int row_ofs_I, int row_ofs_P, float (&vi)[12], float (&vp)[4])
{
    if constexpr (sizeof(T) == 1) {
        const unsigned* pi = reinterpret_cast<const unsigned*>(c.gI + row_ofs_I);
        const unsigned* pp = reinterpret_cast<const unsigned*>(c.gP + row_ofs_P);
        vi[0] = gf_bits_f(pi[0]); vi[1] = gf_bits_f(pi[1]); vi[2] = gf_bits_f(pi[2]);
        vp[0] = gf_bits_f(pp[0]);
        vp[1] = vp[0]; vp[2] = 0.f;
        if (c.p3) { vp[1] = gf_bits_f(pp[1]); vp[2] = gf_bits_f(pp[2]); }
#pragma unroll
        for (int i = 3; i < 12; ++i) vi[i] = 0.f;
        vp[3] = 0.f;
        return;
    }
    const float4* pi = reinterpret_cast<const float4*>(c.gI + row_ofs_I);
    const float4 t0 = pi[0], t1 = pi[1], t2 = pi[2];
    const float4 tp = *reinterpret_cast<const float4*>(c.gP + row_ofs_P);
    vi[0] = t0.x; vi[1] = t0.y; vi[2] = t0.z; vi[3] = t0.w; vi[4] = t1.x; vi[5] = t1.y; vi[6] = t1.z; vi[7] = t1.w;
    vi[8] = t2.x; vi[9] = t2.y; vi[10] = t2.z; vi[11] = t2.w;
    vp[0] = tp.x; vp[1] = tp.y; vp[2] = tp.z; vp[3] = tp.w;
}

// Mirror for lanes outside the image (width % 4 == 0).  REFLECT101:
//   left : column -4k+j <- column 4k-j      = {col0 of lane s0, col3, col2, col1 of lane s1}
//   right: column W+4m+j <- column W-2-4m-j = {col2, col1, col0 of lane s1(=s0), col3 of lane s2}
// REFLECT (edge pixel repeated): column -4k+j <- 4k-1-j and W+4m+j <- W-1-4m-j: the four columns of ONE lane (s0), reversed.
// TRUNCATE: zeros.  A warp overhangs at most one side (width >= 128), so all its lanes publish that side's pattern.
template <int R, int BM, class T>
__device__ __forceinline__ void gf_c4_mirror(const GfC4Ctx<R, T>& c, float (&vi)[12], float (&vp)[4], bool zero_row = false)
{
    const unsigned full = 0xffffffffu;
    const bool out = c.out_l || c.out_r;
    if (BM == 2) {                                  // (also run by interior strips: rows above / below the image)
        const bool z = out || zero_row;
#pragma unroll
        for (int i = 0; i < 12; ++i) vi[i] = z ? 0.f : vi[i];
#pragma unroll
        for (int j = 0; j < 4; ++j) vp[j] = z ? 0.f : vp[j];
        return;
    }
    // per destination column j: source column index in the source lane (left pattern / right pattern)
    //   REFLECT101  j:  0  1  2  3          REFLECT  j:  0  1  2  3
    //   left:           0  3  2  1   s0 s1 s1 s1         3  2  1  0   s0 s0 s0 s0
    //   right:          2  1  0  3   s0 s0 s0 s2         3  2  1  0   s0 s0 s0 s0     (s1 == s0 for right lanes)
    float ni[12], np[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (BM == 1) {
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) ni[3 * j + ch] = __shfl_sync(full, vi[3 * (3 - j) + ch], c.s0);
            np[j] = __shfl_sync(full, vp[3 - j], c.s0);
        } else {
            const int jl = j == 0 ? 0 : 4 - j, jr = j == 3 ? 3 : 2 - j;
            const int sl = j == 0 ? c.s0 : c.s1;
            const int sr = j == 3 ? c.s2 : c.s0;
            const int srcl = c.out_l ? sl : sr;
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                const float pub = c.src_l ? vi[3 * jl + ch] : vi[3 * jr + ch];
                ni[3 * j + ch] = __shfl_sync(full, pub, srcl);
            }
            const float pubp = c.src_l ? vp[jl] : vp[jr];
            np[j] = __shfl_sync(full, pubp, srcl);
        }
    }
#pragma unroll
    for (int i = 0; i < 12; ++i) vi[i] = out ? ni[i] : vi[i];
#pragma unroll
    for (int j = 0; j < 4; ++j) vp[j] = out ? np[j] : vp[j];
}

// Returns true when the row stands for zeros (TRUNCATE, row outside the image or past the resident rows): the loads are
// issued anyway, from a clamped row, so that the load schedule has no branch; gf_c4_mirror<.., 2> clears the values.
template <int R, bool MIRROR, int BM, class T>
__device__ __forceinline__ bool gf_c4_load_row(const GfC4Ctx<R, T>& c, int y, float (&vi)[12], float (&vp)[4])
{
    int rn = BM == 2 ? (y < 0 ? 0 : y) : gf_s8_map_y(y, c.height, c.border);
    const bool zero = BM == 2 && (y < 0 || y > c.buf_ylast);
    rn = rn > c.buf_ylast ? c.buf_ylast : rn;
    const int o = rn - c.buf_y0;
    gf_c4_ld<R>(c, o * c.gs, o * c.ss, vi, vp);     // RAW for lanes outside the image: gf_c4_mirror runs where the row is
                                                    // consumed (shuffles right behind the loads would wait for them here)
    return zero;
}

// the 13 products of one pixel, added to (SUB = false) or removed from (SUB = true) the column sums
template <bool SUB>
__device__ __forceinline__ void gf_c4_accum(float (&c)[13][4], int j, float i0, float i1, float i2, float p)
{
    const float s = SUB ? -1.f : 1.f;
    c[0][j] += s * i0; c[1][j] += s * i1; c[2][j] += s * i2; c[3][j] += s * p;
    const float m0 = s * i0, m1 = s * i1, m2 = s * i2;
    c[4][j] = fmaf(m0, p, c[4][j]); c[5][j] = fmaf(m1, p, c[5][j]); c[6][j] = fmaf(m2, p, c[6][j]);
    c[7][j] = fmaf(m0, i0, c[7][j]); c[8][j] = fmaf(m0, i1, c[8][j]); c[9][j] = fmaf(m0, i2, c[9][j]);
    c[10][j] = fmaf(m1, i1, c[10][j]); c[11][j] = fmaf(m1, i2, c[11][j]); c[12][j] = fmaf(m2, i2, c[12][j]);
}

// Iteration t >= 2R (see gf_s8_iter for the schedule: ramp-up is data, not code).
template <int R, bool MIRROR, int BM, class T>
__device__ __forceinline__ void gf_c4_iter(GfC4Ctx<R, T>& c, int t, int slot, bool full)
{
    using G = GfC4Geom<R>;
    constexpr int KW = G::KW, VL = G::VL;
    const int yi = c.yi0 + t;

    if constexpr (sizeof(T) == 1) { gf_c4_expand(c, c.nI, c.nP); gf_c4_expand(c, c.oI, c.oP); }
    if (MIRROR || BM == 2) { gf_c4_mirror<R, BM>(c, c.nI, c.nP, c.nz); gf_c4_mirror<R, BM>(c, c.oI, c.oP, c.oz); }
    // ---- stage 1, vertical: add row yi, drop row yi - KW (its guide pixels are kept for the output)
    float gI[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) gI[i] = c.oI[i];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        gf_c4_accum<false>(c.c, j, c.nI[3 * j], c.nI[3 * j + 1], c.nI[3 * j + 2], c.nP[j]);
        gf_c4_accum<true>(c.c, j, c.oI[3 * j], c.oI[3 * j + 1], c.oI[3 * j + 2], c.oP[j]);
    }
    // rows of the next iteration
    c.nz = gf_c4_load_row<R, MIRROR, BM>(c, yi + 1, c.nI, c.nP);
    c.oz = gf_c4_load_row<R, MIRROR, BM>(c, yi + 1 - KW, c.oI, c.oP);

    // ---- stage 2 of the a, b row produced by the previous iteration
    {
        float h[4][4];
#pragma unroll
        for (int q = 0; q < 4; ++q) gf_c4_window<R>(c.va[q], h[q]);
        if (c.ring_lane) {
            float4* s = c.ring + slot * G::SLOT_F4;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (full) {
                    const float4 o = s[q * VL];
                    c.sa[q][0] += h[q][0] - o.x; c.sa[q][1] += h[q][1] - o.y; c.sa[q][2] += h[q][2] - o.z; c.sa[q][3] += h[q][3] - o.w;
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) c.sa[q][j] += h[q][j];
                }
                s[q * VL] = make_float4(h[q][0], h[q][1], h[q][2], h[q][3]);
            }
        }
        if (full) {                                   // q of row yo = yi-1-2R; guide row gI
            const int yo = yi - 1 - 2 * R;
            const float inv = 1.0f / (float)(KW * KW);
            const float icy = BM == 2 ? 1.0f / gf_s8_cnt_y<R>(yo, c.height) : 0.f;
            float qv[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float v = fmaf(c.sa[0][j], gI[3 * j], fmaf(c.sa[1][j], gI[3 * j + 1], fmaf(c.sa[2][j], gI[3 * j + 2], c.sa[3][j])));
                qv[j] = v * (BM == 2 ? c.icx[j] * icy : inv);
            }
            if (c.out_lane) {
                T* q = c.gQ + (yo - c.out_y0) * c.ds;
                if constexpr (sizeof(T) == 1) {             // q' = 255 q: round half to even, saturate
                    if (c.p3) {                             // byte stores: the other channels are other warps' frames
#pragma unroll
                        for (int j = 0; j < 4; ++j) q[3 * j] = (unsigned char)gf_f_to_u8(qv[j]);
                    } else {
                        *reinterpret_cast<unsigned*>(q) =
                            gf_f_to_u8(qv[0]) | (gf_f_to_u8(qv[1]) << 8) | (gf_f_to_u8(qv[2]) << 16) | (gf_f_to_u8(qv[3]) << 24);
                    }
                } else {
                    *reinterpret_cast<float4*>(q) = make_float4(qv[0], qv[1], qv[2], qv[3]);
                }
            }
        }
    }

    // ---- stage 1, horizontal -> a, b of row yi - R
    {
        float h[13][4];
#pragma unroll
        for (int q = 0; q < 13; ++q) gf_c4_window<R>(c.c[q], h[q]);
        const float inv1 = 1.0f / (float)(KW * KW);
        const int yc = yi - R;
        const float icy = BM == 2 ? 1.0f / gf_s8_cnt_y<R>(yc, c.height) : 0.f;
        const bool ok = BM != 2 || (!(c.out_l || c.out_r) && yc >= 0 && yc < c.height);     // TRUNCATE: a, b are zero outside the image
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float inv = BM == 2 ? c.icx[j] * icy : inv1;
            const float m0 = h[0][j] * inv, m1 = h[1][j] * inv, m2 = h[2][j] * inv, mp = h[3][j] * inv;
            const float c0 = fmaf(h[4][j], inv, -m0 * mp), c1 = fmaf(h[5][j], inv, -m1 * mp), c2 = fmaf(h[6][j], inv, -m2 * mp);
            const float s00 = fmaf(h[7][j], inv, -m0 * m0) + c.eps, s01 = fmaf(h[8][j], inv, -m0 * m1),
                        s02 = fmaf(h[9][j], inv, -m0 * m2), s11 = fmaf(h[10][j], inv, -m1 * m1) + c.eps,
                        s12 = fmaf(h[11][j], inv, -m1 * m2), s22 = fmaf(h[12][j], inv, -m2 * m2) + c.eps;
            const float i00 = s11 * s22 - s12 * s12, i01 = s02 * s12 - s01 * s22, i02 = s01 * s12 - s02 * s11,
                        i11 = s00 * s22 - s02 * s02, i12 = s01 * s02 - s00 * s12, i22 = s00 * s11 - s01 * s01;
            const float det = s00 * i00 + s01 * i01 + s02 * i02;
            float rd = gf_s8_rcp(det);
            rd = fmaf(fmaf(-det, rd, 1.0f), rd, rd);
            const float a0 = (i00 * c0 + i01 * c1 + i02 * c2) * rd;
            const float a1 = (i01 * c0 + i11 * c1 + i12 * c2) * rd;
            const float a2 = (i02 * c0 + i12 * c1 + i22 * c2) * rd;
            c.va[0][j] = ok ? a0 : 0.f; c.va[1][j] = ok ? a1 : 0.f; c.va[2][j] = ok ? a2 : 0.f;
            c.va[3][j] = ok ? mp - (a0 * m0 + a1 * m1 + a2 * m2) : 0.f;
        }
    }
}

template <int R, bool MIRROR, int BM, class T>
__device__ __forceinline__ void gf_c4_band(GfC4Ctx<R, T>& c, int steps)
{
    constexpr int KW = 2 * R + 1;
    // warm-up rows t in [0, 2R): vertical accumulation only; rows are loaded four at a time so that
    // the band start costs 2R/4 DRAM latencies instead of 2R (2R is a multiple of 4: R % 4 == 0)
    {
        float bI[4][12], bP[4][4];
        bool bz[4];
#pragma unroll 1
        for (int t = 0; t < 2 * R; t += 4) {
#pragma unroll
            for (int k = 0; k < 4; ++k) bz[k] = gf_c4_load_row<R, MIRROR, BM>(c, c.yi0 + t + 1 + k, bI[k], bP[k]);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if constexpr (sizeof(T) == 1) gf_c4_expand(c, c.nI, c.nP);
                if (MIRROR || BM == 2) gf_c4_mirror<R, BM>(c, c.nI, c.nP, c.nz);
                c.nz = bz[k];
#pragma unroll
                for (int j = 0; j < 4; ++j) gf_c4_accum<false>(c.c, j, c.nI[3 * j], c.nI[3 * j + 1], c.nI[3 * j + 2], c.nP[j]);
#pragma unroll
                for (int i = 0; i < 12; ++i) c.nI[i] = bI[k][i];
#pragma unroll
                for (int j = 0; j < 4; ++j) c.nP[j] = bP[k][j];
            }
        }
    }
    int t = 2 * R;
    bool full = false;
#pragma unroll 1
    while (t <= steps) {
        const int n = steps + 1 - t < KW ? steps + 1 - t : KW;
#pragma unroll 1
        for (int s = 0; s < n; ++s, ++t) gf_c4_iter<R, MIRROR, BM>(c, t, s, full);
        full = true;
    }
}

template <int R, int MINB, int BM, class T = float>
__global__ void __launch_bounds__(32, MINB) gf_c4_color_kernel(const GF_GRID_CONSTANT GfWpArgs a)
{
    using G = GfC4Geom<R>;
    constexpr int M = G::M, VL = G::VL;
    GF_DYN_SMEM(float, smem);
    auto run = [&](int64_t f, int strip, int yo0, int yo1) {
    GfC4Ctx<R, T> c;
    c.lane = threadIdx.x & 31;
    const int xl = strip * G::WOUT - 2 * M * 4;
    c.x0 = xl + 4 * c.lane;
    c.mirror = xl < 0 || xl + G::WIN > a.width;
    c.out_l = c.x0 < 0;
    c.out_r = c.x0 >= a.width;
    // mirror source lanes (see gf_c4_mirror)
    {
        const int lw = (a.width - xl) / 4 - 1;       // last lane inside the image (may be >= 32: then no lane is out_r)
        const int X = 4 * M - c.lane;                // left: lane of column -x0 (j = 0)
        const int Y = 2 * lw + 1 - c.lane;           // right: lane of column W-2-(x0-W) (j = 0..2)
        c.s0 = c.out_l ? (BM == 1 ? X - 1 : X) : Y;  // REFLECT: the whole lane comes from lane X-1 (left) or Y (right)
        c.s1 = c.out_l ? X - 1 : Y;
        c.s2 = Y - 1;
        // lanes far outside the image (beyond the 2M halo lanes) mirror nothing anyone uses: clamp
        // their sources to lanes inside the image so that every shuffle and address stays valid
        const int lo_in = xl < 0 ? 2 * M : 0, hi_in = lw < 31 ? lw : 31;
        c.s0 = c.s0 < lo_in ? lo_in : (c.s0 > hi_in ? hi_in : c.s0);
        c.s1 = c.s1 < lo_in ? lo_in : (c.s1 > hi_in ? hi_in : c.s1);
        c.s2 = c.s2 < lo_in ? lo_in : (c.s2 > hi_in ? hi_in : c.s2);
        c.src_l = xl < 0;                            // width >= 128: a warp overhangs at most one side of the image
    }
    // lanes outside the image load from a valid address (their mirror lane's); the data is replaced
    const int xa = (c.out_l || c.out_r) ? 4 * c.s0 + xl : c.x0;
    // (GfWpArgs carries the planes as float*; the uint8 build reinterprets them, strides are in elements)
    const int pch = sizeof(T) == 1 ? a.count : 1;   // interleaved src / dst channels: uint8 frames are the channels
    c.gI = reinterpret_cast<const T*>(a.guide) + f * a.gfs + (int64_t)3 * xa;
    c.gP = reinterpret_cast<const T*>(a.src) + f * a.sfs + (int64_t)pch * xa;
    c.gQ = reinterpret_cast<T*>(a.dst) + f * a.dfs + (int64_t)pch * c.x0;
    if constexpr (sizeof(T) == 1) {
        const unsigned ch = (unsigned)f;
        c.p3 = pch == 3;
        c.gQ += c.p3 ? ch : 0u;
        c.selA = c.p3 ? ch | (3 + ch) << 4 : 0x3210u;
        c.selB = c.p3 ? (2 + ch) << 8 | (5 + ch) << 12 : 0x3210u;
    }
    c.gs = (int)a.gs; c.ss = (int)a.ss; c.ds = (int)a.ds;
    c.ring_lane = c.lane >= 2 * M && c.lane < 32 - 2 * M;
    c.out_lane = c.ring_lane && c.x0 < a.width;
    c.ring = reinterpret_cast<float4*>(smem) + (c.ring_lane ? c.lane - 2 * M : 0);
    c.width = a.width; c.height = a.height; c.border = a.border; c.buf_y0 = a.buf_y0; c.out_y0 = a.out_y0;
    {
        const int yl = a.buf_y0 + a.buf_rows - 1;
        c.buf_ylast = yl < a.height - 1 ? yl : a.height - 1;
    }
    c.yi0 = yo0 - 2 * R;
    c.eps = a.eps;
#pragma unroll
    for (int j = 0; j < 4; ++j) c.icx[j] = BM == 2 ? 1.0f / gf_count(c.x0 + j, a.width, R, GF_TRUNCATE) : 0.f;
    c.oz = true;
#pragma unroll
    for (int q = 0; q < 13; ++q)
#pragma unroll
        for (int j = 0; j < 4; ++j) c.c[q][j] = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int j = 0; j < 4; ++j) { c.sa[q][j] = 0.f; c.va[q][j] = 0.f; }
#pragma unroll
    for (int i = 0; i < 12; ++i) c.oI[i] = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) c.oP[j] = 0.f;
    (void)VL;
    const int steps = (yo1 - yo0) + 4 * R;
    if (c.mirror) {
        c.nz = gf_c4_load_row<R, true, BM>(c, c.yi0, c.nI, c.nP);
        gf_c4_band<R, true, BM>(c, steps);
    } else {
        c.nz = gf_c4_load_row<R, false, BM>(c, c.yi0, c.nI, c.nP);
        gf_c4_band<R, false, BM>(c, steps);
    }
    };
    gf_tape_run(a, (long long)blockIdx.x, run);
}

// ---- host side ------------------------------------------------------------------------------------
#ifndef GF_NO_HOST   // (stand-alone SASS builds of one kernel define GF_NO_HOST)
template <int R, class T>
static const char* gf_c4_launch(const Job& j)
{
    using G = GfC4Geom<R>;
    int sms = 148, mj = 0, mn = 0;
    gf_rt_device_info(&sms, &mj, &mn);
    GfWpArgs a;
    a.guide = j.guide.ptr; a.src = j.src.ptr; a.dst = const_cast<float*>(j.dst.ptr);
    a.A = nullptr; a.B = nullptr;
    a.gs = j.guide.stride; a.ss = j.src.stride; a.ds = j.dst.stride; a.abs_ = 0;
    a.gfs = j.guide.frame_stride; a.sfs = j.src.frame_stride; a.dfs = j.dst.frame_stride; a.abfs = 0;
    a.width = j.width; a.height = j.height; a.buf_y0 = j.buf_y0; a.buf_rows = j.buf_rows; a.out_y0 = j.out_y0;
    a.out_rows = j.out_rows; a.border = j.border; a.count = j.count;
    a.eps = sizeof(T) == 1 ? j.eps * 65025.0f : j.eps;       // uint8 build: integer domain, eps scales with 255^2
    a.tape_piece = 0; a.tape_rho = 0; a.tape_we = 100;
    a.nstrips = (j.width + G::WOUT - 1) / G::WOUT;
    a.hb_e = 0; a.nbands_e = 0;
    const size_t smem = G::ring_bytes;
    constexpr int FIT = (int)((size_t)228 * 1024 / (G::ring_bytes + 1024));
    constexpr int MINB = FIT > 8 ? 8 : (FIT < 1 ? 1 : FIT);
    int warps_sm = MINB;
    warps_sm = GF_KNOB("GF_C4_WARPS_PER_SM", warps_sm);
    if (warps_sm < 1) warps_sm = 1;
    int hb = gf_pick_band_rows(j.out_rows, R, (long)a.nstrips * j.count, (long)sms * warps_sm, 2 * R + 8);
    hb = GF_KNOB("GF_C4_HB", hb);
    if (hb < 1) hb = 1;
    if (hb > j.out_rows) hb = j.out_rows;
    a.hb = hb;
    a.nbands = (j.out_rows + hb - 1) / hb;
    long items = (long)a.nstrips * a.nbands * j.count;
    // One wave of equal-cost pieces ("tape", gf_tape_run) instead of uniform bands: measured 3-8 % FASTER on colour batches
    // that fill the GPU a few times over (16 x 1080p: 0.987 vs 1.073 ms, 32 x: 1.897 vs 1.953 ms, edge weight 120) and
    // slower on single frames and on long batches (64 x: 3.76 vs 3.66 ms) -- profiles/r1_c4_band_sweep.jsonl.  32 frames
    // per GPU is BASELINE configs[2] at 8 GPUs, so that window is where the tape is on by default.
    const double mpx = (double)j.width * j.out_rows * j.count * 1e-6;
    const int tape_dflt = (j.count >= 8 && mpx >= 25.0 && mpx <= 110.0) ? 1 : 0;
    int we = tape_dflt ? 120 : 100;
    we = GF_KNOB("GF_C4_EDGE_WEIGHT", we);
    if (!GF_KNOB_SET("GF_C4_HB"))
        if (const long n = gf_tape_plan(a, R, (long)sms * warps_sm, 2 * R + 8, we, tape_dflt)) items = n;
    dim3 grid((unsigned)items), block(32);
    auto go = [&](auto k) -> const char* {
        if (const char* e = gf_rt_set_smem(k, smem)) return e;
        GF_LAUNCH(k, grid, block, smem, j.stream, a);
        return gf_rt_launch_error();
    };
    if (j.border == GF_REFLECT) return go(gf_c4_color_kernel<R, MINB, 1, T>);
    if (j.border == GF_TRUNCATE) return go(gf_c4_color_kernel<R, MINB, 2, T>);
    return go(gf_c4_color_kernel<R, MINB, 0, T>);
}

// T = unsigned char (gf_guided_color_u8): the planes hold unsigned char (Plane::ptr reinterpreted, strides in
// elements), the frames are the src_channels (1 or 3) interleaved source channels: count = src.channels = dst.channels,
// every frame stride 0.  Each kernel family is instantiated in its own translation unit (gf_tu_c4.cu, gf_tu_c4u8.cu).
template <class T>
static const char* gf_c4_try(const Job& j, bool* done, const char** name)
{
    constexpr bool u8 = sizeof(T) == 1;
    *done = false;
    if (!j.color || j.A.ptr) return nullptr;
    if (j.border != GF_REFLECT101 && j.border != GF_REFLECT && j.border != GF_TRUNCATE) return nullptr;
    const Plane* pl[3] = {&j.guide, &j.src, &j.dst};
    if (u8) {
        if (j.guide.channels != 3 || (j.count != 1 && j.count != 3) || j.src.channels != j.count || j.dst.channels != j.count)
            return nullptr;
        for (int i = 0; i < 3; ++i)
            if (pl[i]->coff != 0 || pl[i]->frame_stride != 0 || (pl[i]->stride & 3) || ((uintptr_t)pl[i]->ptr & 3)) return nullptr;
        if ((int64_t)j.buf_rows * j.src.stride >= (1ll << 31)) return nullptr;
    } else {
        if (GF_KNOB("GF_DISABLE_C4", 0) || GF_KNOB("GF_DISABLE_FAST", 0)) return nullptr;
        if (j.guide.channels != 3 || j.guide.coff != 0 || j.src.channels != 1 || j.src.coff != 0 || j.dst.channels != 1 || j.dst.coff != 0)
            return nullptr;
        for (int i = 0; i < 3; ++i)
            if ((pl[i]->stride & 3) || (pl[i]->frame_stride & 3) || ((uintptr_t)pl[i]->ptr & 15)) return nullptr;
    }
    if ((j.width & 3) || j.width < 128 || j.height < 4 * j.r + 2) return nullptr;
    if ((int64_t)j.buf_rows * j.guide.stride >= (1ll << 31) || (int64_t)j.out_rows * j.dst.stride >= (1ll << 31)) return nullptr;
    switch (j.r) {
    case 4: *done = true; *name = u8 ? "c4u8_r4" : "c4_r4"; return gf_c4_launch<4, T>(j);
    case 8: *done = true; *name = u8 ? "c4u8_r8" : "c4_r8"; return gf_c4_launch<8, T>(j);
    case 12: *done = true; *name = u8 ? "c4u8_r12" : "c4_r12"; return gf_c4_launch<12, T>(j);
    case 16: *done = true; *name = u8 ? "c4u8_r16" : "c4_r16"; return gf_c4_launch<16, T>(j);
    default: return nullptr;
    }
}
#endif  // GF_NO_HOST
