// gf_fgf.cuh -- the two full-resolution passes of the fast guided filter (He & Sun, "Fast Guided Filter",
// arXiv:1505.00996; fastguidedfilter.m): area subsampling of I and p by s, and the bilinear upsample of
// mean_a / mean_b fused into q = mean_a*I + mean_b.  The low-resolution a/b solve and the box means of a
// and b in between are the library's existing kernels (gf_api.cu: gf_fast_guided_gray).
//
//   gf_fgf_down_kernel      thread <-> low-res column, grid-stride over low-res rows: reads the s x s block
//                           of I and of p (a warp covers 32*s contiguous floats of every row), writes the
//                           two means.  8 B/px of HBM traffic at full resolution, 8/s^2 B/px written.
//   gf_fgf_up_apply_kernel  CTA <-> full-res tile of GF_FGF_TY x GF_FGF_TX: stages the (tile/s + 2)^2
//                           low-res samples of mean_a and mean_b it needs in shared memory, then reads I
//                           and writes q once.  8 B/px at full resolution plus the low-res planes.
//                           Needs s >= 2 (the staging buffers hold tile/2 + 2 samples per side).
//
// T = unsigned char: the same two kernels on 8-bit planes (gf_fast_guided_gray_u8), in the integer domain of the other
// uint8 builds: I' = 255 I and p' = 255 p are the bytes as floats, the low-res planes hold block means in 0..255 and the
// a/b job runs with eps' = 255^2 eps, so a is scale-free, mean_b' = 255 mean_b and q' = mean_a I' + mean_b' = 255 q goes
// straight to the saturating round-half-even store.  The block sums of bytes are int (<= 1024 x 255 < 2^24: exact, in
// any order).  2 B/px at full resolution in each kernel instead of 8.
#pragma once
#include <type_traits>

#include "gf_common.cuh"

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
    int64_t si, sp, sl;              // row strides (elements): guide, source, low-res planes
    int width, height, ws, hs, s;
};

template <typename T>
__global__ void __launch_bounds__(GF_FGF_DOWN_THREADS) gf_fgf_down_kernel(const GfFgfDownArgs<T> a)
{
    typedef typename std::conditional<sizeof(T) == 1, int, float>::type Sum;
    const int X = blockIdx.x * GF_FGF_DOWN_THREADS + threadIdx.x;
    if (X >= a.ws) return;
    const int s = a.s;
    const int x0 = X * s, x1 = min(x0 + s, a.width);
    const float inv_full = 1.0f / (float)(s * s);
    for (int Y = blockIdx.y; Y < a.hs; Y += gridDim.y) {
        const int y0 = Y * s, y1 = min(y0 + s, a.height);
        Sum si = 0, sp = 0;                                  // at most 32 x 32 = 1024 terms
        for (int y = y0; y < y1; ++y) {
            const T* ri = a.I + (int64_t)y * a.si;
            const T* rp = a.p + (int64_t)y * a.sp;
#pragma unroll 4
            for (int x = x0; x < x1; ++x) {
                si += ri[x];
                sp += rp[x];
            }
        }
        const int n = (y1 - y0) * (x1 - x0);
        float mi, mp;
        if (n == s * s) { mi = (float)si * inv_full; mp = (float)sp * inv_full; }
        else { mi = (float)si / (float)n; mp = (float)sp / (float)n; }   // partial block of the last row / column
        a.Is[(int64_t)Y * a.sl + X] = mi;
        a.ps[(int64_t)Y * a.sl + X] = mp;
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
