// gf_fgf.cuh -- the kernels of the fast guided filter (He & Sun, "Fast Guided Filter", arXiv:1505.00996;
// fastguidedfilter.m) that the library's exact filters do not already provide: area subsampling of I and p by s, the
// bilinear upsample of the mean planes fused into q, and the low-res a/b solve of the colour guide.  Between them run the
// library's existing kernels (gf_api.cu: gf_fast_guided_gray, gf_fast_guided_color).
//
//   gf_fgf_down_kernel      thread <-> low-res column, grid-stride over low-res rows: reads the s x s block
//                           of I and of p (a warp covers 32*s contiguous pixels of every row), writes the
//                           means.  GC / PC: interleaved channels of I and p; I_s is written as one GC-channel
//                           plane, p_s as one plane per source channel.  (4 GC + 4 PC) B/px of HBM traffic at
//                           full resolution, (4 GC + 4 PC)/s^2 B/px written.
//   gf_fgf_up_apply_kernel  gray guide.  CTA <-> full-res tile of GF_FGF_TY x GF_FGF_TX: stages the (tile/s + 2)^2
//                           low-res samples of mean_a and mean_b it needs in shared memory, then reads I
//                           and writes q once.  8 B/px at full resolution plus the low-res planes.
//                           Needs s >= 2 (the staging buffers hold tile/2 + 2 samples per side).
//   gf_fgf_color_ab_kernel  colour guide, low resolution: a (3-vector) and b of every low-res pixel, per source channel.
//   gf_fgf_up_apply_color_kernel  colour guide: the tile of gf_fgf_up_apply_kernel, C source channels.
//
// T = unsigned char: the gray kernels on 8-bit planes (gf_fast_guided_gray_u8), in the integer domain of the other
// uint8 builds: I' = 255 I and p' = 255 p are the bytes as floats, the low-res planes hold block means in 0..255 and the
// a/b job runs with eps' = 255^2 eps, so a is scale-free, mean_b' = 255 mean_b and q' = mean_a I' + mean_b' = 255 q goes
// straight to the saturating round-half-even store.  The block sums of bytes are int (<= 1024 x 255 < 2^24: exact, in
// any order).  2 B/px at full resolution in each kernel instead of 8.
#pragma once
#include <type_traits>

#include "gf_common.cuh"
#include "gf_generic.cuh"

#define GF_FGF_MAX_S 32
#define GF_FGF_DOWN_THREADS 128
#define GF_FGF_TX 128                                        // tile columns: 32 threads x 4
#define GF_FGF_TY 32                                         // tile rows: 8 threads x 4
#define GF_FGF_SW (GF_FGF_TX / 2 + 2)                        // staged low-res columns at s >= 2
#define GF_FGF_SH (GF_FGF_TY / 2 + 2)                        // staged low-res rows at s >= 2

template <typename T>
struct GfFgfDownArgs {
    const T* I; const T* p;
    float* Is; float* ps;
    int64_t si, sp, sl;              // row strides (elements): guide, source, low-res planes (GC = 1: all of them)
    int width, height, ws, hs, s;
    int64_t sls, spl;                // GC > 1: row stride of I_s; PC > 1: stride between the planes of p_s
};

template <typename T, int GC = 1, int PC = 1>
__global__ void __launch_bounds__(GF_FGF_DOWN_THREADS) gf_fgf_down_kernel(const GfFgfDownArgs<T> a)
{
    typedef typename std::conditional<sizeof(T) == 1, int, float>::type Sum;
    const int X = blockIdx.x * GF_FGF_DOWN_THREADS + threadIdx.x;
    if (X >= a.ws) return;
    const int s = a.s;
    const int x0 = X * s, x1 = min(x0 + s, a.width);
    const float inv_full = 1.0f / (float)(s * s);
    const int64_t sls = GC == 1 ? a.sl : a.sls;
    for (int Y = blockIdx.y; Y < a.hs; Y += gridDim.y) {
        const int y0 = Y * s, y1 = min(y0 + s, a.height);
        Sum si[GC], sp[PC];                                  // at most 32 x 32 = 1024 terms
#pragma unroll
        for (int c = 0; c < GC; ++c) si[c] = 0;
#pragma unroll
        for (int c = 0; c < PC; ++c) sp[c] = 0;
        for (int y = y0; y < y1; ++y) {
            const T* ri = a.I + (int64_t)y * a.si;
            const T* rp = a.p + (int64_t)y * a.sp;
#pragma unroll 4
            for (int x = x0; x < x1; ++x) {
#pragma unroll
                for (int c = 0; c < GC; ++c) si[c] += ri[x * GC + c];
#pragma unroll
                for (int c = 0; c < PC; ++c) sp[c] += rp[x * PC + c];
            }
        }
        const int n = (y1 - y0) * (x1 - x0);
        float mi[GC], mp[PC];
        if (n == s * s) {
#pragma unroll
            for (int c = 0; c < GC; ++c) mi[c] = (float)si[c] * inv_full;
#pragma unroll
            for (int c = 0; c < PC; ++c) mp[c] = (float)sp[c] * inv_full;
        } else {                                             // partial block of the last row / column
#pragma unroll
            for (int c = 0; c < GC; ++c) mi[c] = (float)si[c] / (float)n;
#pragma unroll
            for (int c = 0; c < PC; ++c) mp[c] = (float)sp[c] / (float)n;
        }
#pragma unroll
        for (int c = 0; c < GC; ++c) a.Is[(int64_t)Y * sls + X * GC + c] = mi[c];
#pragma unroll
        for (int c = 0; c < PC; ++c) (a.ps + c * a.spl)[(int64_t)Y * a.sl + X] = mp[c];
    }
}

// Low-res sample coordinate of full-res coordinate x: u = clamp((x + 0.5)/s - 0.5, 0, n - 1) = i0 + f,
// i1 = min(i0 + 1, n - 1).  (x + 0.5)/s - 0.5 = (2x + 1 - s) / 2s, so i0 and f come from integers and are
// periodic in x with period s.
__host__ __device__ __forceinline__ void gf_fgf_coord(int x, int s, int n, int* i0, int* i1, float* f)
{
    const int num = 2 * x + 1 - s, den = 2 * s;
    int i = 0;
    float w = 0.f;
    if (num > 0) {
        i = num / den;
        w = (float)(num - i * den) / (float)den;
    }
    if (i >= n - 1) { i = n - 1; w = 0.f; }
    *i0 = i;
    *i1 = i + 1 < n ? i + 1 : n - 1;
    *f = w;
}

template <typename T>
struct GfFgfApplyArgs {
    const T* I; T* q;
    const float* ma; const float* mb;    // low-res mean_a, mean_b
    int64_t si, sq, sl;
    int width, height, ws, hs, s;
};

// The 4 adjacent pixels of a thread on the vector path: one 16-byte access for float, one 4-byte access for bytes.
__device__ __forceinline__ float4 gf_fgf_ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 gf_fgf_ld4(const unsigned char* p)
{
    const unsigned w = *reinterpret_cast<const unsigned*>(p);
    return make_float4(gf_u8_to_f(w, 0), gf_u8_to_f(w, 1), gf_u8_to_f(w, 2), gf_u8_to_f(w, 3));
}
__device__ __forceinline__ void gf_fgf_st4(float* p, const float4& v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void gf_fgf_st4(unsigned char* p, const float4& v)
{
    *reinterpret_cast<unsigned*>(p) = gf_f_to_u8(v.x) | gf_f_to_u8(v.y) << 8 | gf_f_to_u8(v.z) << 16 | gf_f_to_u8(v.w) << 24;
}

// Per tile: the low-res samples are staged, then every staged row is interpolated horizontally to the tile's 128
// columns (h_a, h_b), so that a pixel costs one vertical blend: 2 shared loads per plane instead of 4.  Both load paths
// evaluate the same expressions in the same order -- top/bottom = fmaf(fx, t[x1] - t[x0], t[x0]), then
// fmaf(fy, bot - top, top), then q = fmaf(mean_a, I, mean_b) -- so they give the same bits.  VEC needs width % 4 == 0
// and I and q aligned to 4 elements, base and row stride.
template <bool VEC, typename T>
__global__ void __launch_bounds__(256) gf_fgf_up_apply_kernel(const GfFgfApplyArgs<T> a)
{
    __shared__ float s_a[GF_FGF_SH * GF_FGF_SW];
    __shared__ float s_b[GF_FGF_SH * GF_FGF_SW];
    __shared__ __align__(16) float h_a[GF_FGF_SH * GF_FGF_TX];
    __shared__ __align__(16) float h_b[GF_FGF_SH * GF_FGF_TX];
    const int s = a.s;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int x0 = blockIdx.x * GF_FGF_TX;
    const int xl = min(x0 + GF_FGF_TX, a.width) - 1;
    int X0, X1, dummy;
    float fd;
    gf_fgf_coord(x0, s, a.ws, &X0, &dummy, &fd);
    gf_fgf_coord(xl, s, a.ws, &dummy, &X1, &fd);
    const int nx = X1 - X0 + 1;                              // <= GF_FGF_TX/s + 2
    // the tile column this thread interpolates horizontally (columns past the image repeat the last one)
    const int hx = threadIdx.x & (GF_FGF_TX - 1);
    int hx0, hx1;
    float hfx;
    gf_fgf_coord(min(x0 + hx, a.width - 1), s, a.ws, &hx0, &hx1, &hfx);
    hx0 -= X0;
    hx1 -= X0;

    const int ntiles_y = (a.height + GF_FGF_TY - 1) / GF_FGF_TY;
    for (int tile = blockIdx.y; tile < ntiles_y; tile += gridDim.y) {
        const int y0 = tile * GF_FGF_TY;
        const int yl = min(y0 + GF_FGF_TY, a.height) - 1;
        int Y0, Y1;
        gf_fgf_coord(y0, s, a.hs, &Y0, &dummy, &fd);
        gf_fgf_coord(yl, s, a.hs, &dummy, &Y1, &fd);
        const int ny = Y1 - Y0 + 1;                          // <= GF_FGF_TY/s + 2
        __syncthreads();                                     // the previous tile's reads of h_a / h_b are done
        for (int i = threadIdx.x; i < nx * ny; i += 256) {
            const int yy = i / nx, xx = i - yy * nx;
            const int64_t o = (int64_t)(Y0 + yy) * a.sl + X0 + xx;
            s_a[yy * GF_FGF_SW + xx] = a.ma[o];
            s_b[yy * GF_FGF_SW + xx] = a.mb[o];
        }
        __syncthreads();
        for (int yy = threadIdx.x / GF_FGF_TX; yy < ny; yy += 256 / GF_FGF_TX) {
            const float* ta = s_a + yy * GF_FGF_SW;
            const float* tb = s_b + yy * GF_FGF_SW;
            h_a[yy * GF_FGF_TX + hx] = fmaf(hfx, ta[hx1] - ta[hx0], ta[hx0]);
            h_b[yy * GF_FGF_TX + hx] = fmaf(hfx, tb[hx1] - tb[hx0], tb[hx0]);
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int y = y0 + ty + 8 * j;
            if (y >= a.height) break;
            int r0, r1;
            float fy;
            gf_fgf_coord(y, s, a.hs, &r0, &r1, &fy);
            const float* ta = h_a + (r0 - Y0) * GF_FGF_TX;
            const float* ba = h_a + (r1 - Y0) * GF_FGF_TX;
            const float* tb = h_b + (r0 - Y0) * GF_FGF_TX;
            const float* bb = h_b + (r1 - Y0) * GF_FGF_TX;
            const T* rowI = a.I + (int64_t)y * a.si;
            T* rowq = a.q + (int64_t)y * a.sq;
            if (VEC) {
                const int x = x0 + 4 * tx;
                if (x >= a.width) continue;                   // width % 4 == 0: the 4 columns are all in or all out
                const float4 iv = gf_fgf_ld4(rowI + x);
                const float4 at = *reinterpret_cast<const float4*>(ta + 4 * tx), ab = *reinterpret_cast<const float4*>(ba + 4 * tx);
                const float4 bt = *reinterpret_cast<const float4*>(tb + 4 * tx), bw = *reinterpret_cast<const float4*>(bb + 4 * tx);
                float4 o;
                o.x = fmaf(fmaf(fy, ab.x - at.x, at.x), iv.x, fmaf(fy, bw.x - bt.x, bt.x));
                o.y = fmaf(fmaf(fy, ab.y - at.y, at.y), iv.y, fmaf(fy, bw.y - bt.y, bt.y));
                o.z = fmaf(fmaf(fy, ab.z - at.z, at.z), iv.z, fmaf(fy, bw.z - bt.z, bt.z));
                o.w = fmaf(fmaf(fy, ab.w - at.w, at.w), iv.w, fmaf(fy, bw.w - bt.w, bt.w));
                gf_fgf_st4(rowq + x, o);
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int c = tx + 32 * k;
                    if (x0 + c >= a.width) break;
                    const float v = fmaf(fmaf(fy, ba[c] - ta[c], ta[c]), gf_ld1(&rowI[x0 + c]), fmaf(fy, bb[c] - tb[c], tb[c]));
                    gf_st1(&rowq[x0 + c], v);
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Colour guide.  Low-res a/b: gf_box_kernel's skeleton (thread <-> extended column x0 - r + t, vertical running sums that
// add the entering row and subtract the leaving one, gf_hsum, the border rule through gf_map / gf_count / GfNorm) over the
// 13 quantities of GfColorModel::load, solved by GfColorModel::solve: the borders and the numerics of generic_color.
// guide: I_s, 3 channels interleaved (frame stride 0); src: p_s, one frame per source channel (blockIdx.z); dst: one
// 4-channel plane (a_r, a_g, a_b, b) per source channel, 16-byte aligned pixels.  r <= GF_FGF_MAX_RL: a CTA of
// GF_FGF_AB_THREADS columns keeps at least 32 of them as outputs.
#define GF_FGF_AB_THREADS 128
#define GF_FGF_MAX_RL ((GF_FGF_AB_THREADS - 32) / 2)

__global__ void __launch_bounds__(GF_FGF_AB_THREADS) gf_fgf_color_ab_kernel(const GfArgs a)
{
    constexpr int NQ = GfColorModel::NQ1;
    __shared__ float s_cs[NQ * GF_FGF_AB_THREADS];
    __shared__ float s_tot[NQ * 32];
    const int tid = threadIdx.x, win = GF_FGF_AB_THREADS;
    const int r = a.r, k = 2 * r + 1;
    const int64_t f = blockIdx.z;
    const int xe = blockIdx.x * a.wc - r + tid;
    const int sx = gf_map(xe, a.width, a.border);
    const float cnt_x = gf_count(xe, a.width, r, a.border);
    const int yo0 = blockIdx.y * a.hb;
    const int yo1 = min(a.height, yo0 + a.hb);
    const bool out_col = tid >= r && tid < r + a.wc && xe < a.width;

    float cs[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) cs[q] = 0.f;
    const int steps = (yo1 - yo0) + 2 * r;
    for (int t = 0; t < steps; ++t) {
        const int yi = yo0 - r + t;
        if (sx >= 0) {
            const int sy = gf_map(yi, a.height, a.border);
            if (sy >= 0) {
                float v[NQ];
                GfColorModel::load(a, f, sy, sx, v);
#pragma unroll
                for (int q = 0; q < NQ; ++q) cs[q] += v[q];
            }
            if (t >= k) {
                const int so = gf_map(yi - k, a.height, a.border);
                if (so >= 0) {
                    float v[NQ];
                    GfColorModel::load(a, f, so, sx, v);
#pragma unroll
                    for (int q = 0; q < NQ; ++q) cs[q] -= v[q];
                }
            }
        }
        if (t < 2 * r) continue;              // uniform across the CTA
        float h[NQ];
        gf_hsum<NQ>(cs, h, s_cs, s_tot, r, tid, win);
        __syncthreads();                      // s_cs is rewritten next step
        if (out_col) {
            const int yo = yi - r;
            float ab[GfColorModel::NQ2];
            GfColorModel::solve(h, gf_norm_make(cnt_x * gf_count(yo, a.height, r, a.border)), a.eps, ab);
            float* d = a.dst.ptr + f * a.dst.frame_stride + (int64_t)yo * a.dst.stride + (int64_t)xe * 4;
            *reinterpret_cast<float4*>(d) = make_float4(ab[0], ab[1], ab[2], ab[3]);
        }
    }
}

struct GfFgfApplyColorArgs {
    const float* I; float* q;           // guide: 3 channels interleaved; q: C channels interleaved
    const float* m;                     // low-res (mean_a_r, mean_a_g, mean_a_b, mean_b), one 4-channel plane per channel
    int64_t si, sq, sl, pl;             // row strides (floats): guide, q, low-res; low-res plane stride
    int width, height, ws, hs, s;
};

// q of one pixel from the rows of the four horizontally interpolated mean planes above (t) and below (b) it: the one
// expression both load paths evaluate, so that they give the same bits
__device__ __forceinline__ float gf_fgf_q3(float fy, const float (&t)[4], const float (&b)[4], const float (&g)[3])
{
    float m[4];
#pragma unroll
    for (int p = 0; p < 4; ++p) m[p] = fmaf(fy, b[p] - t[p], t[p]);
    return fmaf(m[2], g[2], fmaf(m[1], g[1], fmaf(m[0], g[0], m[3])));
}

// The tile and thread layout of gf_fgf_up_apply_kernel (a thread owns 4 columns in each of 4 rows) with a 3-channel guide
// and C source channels.  A thread reads the guide of its 16 pixels once per tile and writes every channel of them, so
// dst may be the guide.  The four mean planes of one source channel at a time are interpolated horizontally to the tile's
// columns in shared memory (36 KB; the low-res samples come from L2: the plane of a channel is 16 B per low-res pixel),
// then a pixel costs one vertical blend per plane.  VEC: 16-byte guide loads (and, for C = 1, stores); needs width % 4 ==
// 0, guide and q 16-byte aligned with strides multiples of 4.
template <bool VEC, int C>
__global__ void __launch_bounds__(256) gf_fgf_up_apply_color_kernel(const GfFgfApplyColorArgs a)
{
    constexpr int PS = GF_FGF_SH * GF_FGF_TX;                // one staged plane
    __shared__ __align__(16) float h_m[4 * PS];
    const int s = a.s;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int x0 = blockIdx.x * GF_FGF_TX;
    // the tile column this thread interpolates horizontally (columns past the image repeat the last one)
    const int hx = threadIdx.x & (GF_FGF_TX - 1);
    int hx0, hx1, dummy;
    float hfx, fd;
    gf_fgf_coord(min(x0 + hx, a.width - 1), s, a.ws, &hx0, &hx1, &hfx);

    const int ntiles_y = (a.height + GF_FGF_TY - 1) / GF_FGF_TY;
    for (int tile = blockIdx.y; tile < ntiles_y; tile += gridDim.y) {
        const int y0 = tile * GF_FGF_TY;
        const int yl = min(y0 + GF_FGF_TY, a.height) - 1;
        int Y0, Y1;
        gf_fgf_coord(y0, s, a.hs, &Y0, &dummy, &fd);
        gf_fgf_coord(yl, s, a.hs, &dummy, &Y1, &fd);
        const int ny = Y1 - Y0 + 1;                          // <= GF_FGF_TY/s + 2
        float g[4][4][3];                                    // [row][pixel][channel]
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int y = y0 + ty + 8 * j;
            if (y >= a.height) break;
            const float* rowI = a.I + (int64_t)y * a.si;
            if (VEC) {
                const int x = x0 + 4 * tx;
                if (x >= a.width) continue;
                const float4 v0 = gf_fgf_ld4(rowI + 3 * x), v1 = gf_fgf_ld4(rowI + 3 * x + 4), v2 = gf_fgf_ld4(rowI + 3 * x + 8);
                g[j][0][0] = v0.x; g[j][0][1] = v0.y; g[j][0][2] = v0.z;
                g[j][1][0] = v0.w; g[j][1][1] = v1.x; g[j][1][2] = v1.y;
                g[j][2][0] = v1.z; g[j][2][1] = v1.w; g[j][2][2] = v2.x;
                g[j][3][0] = v2.y; g[j][3][1] = v2.z; g[j][3][2] = v2.w;
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int x = x0 + tx + 32 * k;
                    if (x >= a.width) break;
#pragma unroll
                    for (int c = 0; c < 3; ++c) g[j][k][c] = rowI[3 * (int64_t)x + c];
                }
            }
        }
#pragma unroll 1
        for (int c = 0; c < C; ++c) {
            const float* m = a.m + c * a.pl;
            __syncthreads();                                 // the previous pass's reads of h_m are done
            for (int yy = threadIdx.x / GF_FGF_TX; yy < ny; yy += 256 / GF_FGF_TX) {
                const float* row = m + (int64_t)(Y0 + yy) * a.sl;
                const float4 t0 = *reinterpret_cast<const float4*>(row + 4 * hx0);
                const float4 t1 = *reinterpret_cast<const float4*>(row + 4 * hx1);
                float* hr = h_m + yy * GF_FGF_TX + hx;
                hr[0] = fmaf(hfx, t1.x - t0.x, t0.x);
                hr[PS] = fmaf(hfx, t1.y - t0.y, t0.y);
                hr[2 * PS] = fmaf(hfx, t1.z - t0.z, t0.z);
                hr[3 * PS] = fmaf(hfx, t1.w - t0.w, t0.w);
            }
            __syncthreads();
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int y = y0 + ty + 8 * j;
                if (y >= a.height) break;
                int r0, r1;
                float fy;
                gf_fgf_coord(y, s, a.hs, &r0, &r1, &fy);
                const float* top = h_m + (r0 - Y0) * GF_FGF_TX;
                const float* bot = h_m + (r1 - Y0) * GF_FGF_TX;
                float* rowq = a.q + (int64_t)y * a.sq;
                if (VEC) {
                    const int x = x0 + 4 * tx;
                    if (x >= a.width) continue;              // width % 4 == 0: the 4 columns are all in or all out
                    float4 t4[4], b4[4];
#pragma unroll
                    for (int p = 0; p < 4; ++p) {
                        t4[p] = *reinterpret_cast<const float4*>(top + p * PS + 4 * tx);
                        b4[p] = *reinterpret_cast<const float4*>(bot + p * PS + 4 * tx);
                    }
                    float o[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        float t[4], b[4];
#pragma unroll
                        for (int p = 0; p < 4; ++p) { t[p] = (&t4[p].x)[k]; b[p] = (&b4[p].x)[k]; }
                        o[k] = gf_fgf_q3(fy, t, b, g[j][k]);
                    }
                    if (C == 1) {
                        gf_fgf_st4(rowq + x, make_float4(o[0], o[1], o[2], o[3]));
                    } else {
#pragma unroll
                        for (int k = 0; k < 4; ++k) rowq[(int64_t)(x + k) * C + c] = o[k];
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int col = tx + 32 * k;
                        if (x0 + col >= a.width) break;
                        float t[4], b[4];
#pragma unroll
                        for (int p = 0; p < 4; ++p) { t[p] = top[p * PS + col]; b[p] = bot[p * PS + col]; }
                        rowq[(int64_t)(x0 + col) * C + c] = gf_fgf_q3(fy, t, b, g[j][k]);
                    }
                }
            }
        }
    }
}
