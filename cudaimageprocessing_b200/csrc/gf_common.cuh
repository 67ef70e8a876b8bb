// gf_common.cuh -- shared device/host definitions of the B200 guided-filter kernels.
#pragma once
#include <stdint.h>

#ifdef GF_CPU_EMU
// Test-only build (tests/emu): kernels compiled by g++ and run by the SIMT emulator.
#include "cuda_emu.h"
#define GF_DYN_SMEM(T, name) T* name = reinterpret_cast<T*>(emu::dyn_smem())
#define GF_GRID_CONSTANT
#else
#include <cuda_runtime.h>
#define GF_DYN_SMEM(T, name)                                       \
    extern __shared__ __align__(16) unsigned char name##_raw_[];   \
    T* name = reinterpret_cast<T*>(name##_raw_)
#define GF_GRID_CONSTANT __grid_constant__      // kernel parameters stay in the constant bank when referenced by address
#endif

// L2 prefetch hint (no registers, no scoreboard): rows a few iterations ahead of the loads.
#ifdef GF_CPU_EMU
static inline void gf_prefetch_l2(const void*) {}
#else
__device__ __forceinline__ void gf_prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
#endif

// ---- uint8 planes in the integer domain (gf_s8.cuh, gf_c4.cuh, gf_fgf.cuh): a byte is loaded as the float 0..255 and
// q' = 255 q is stored as saturate_cast<uchar>(cvRound(q')) ------------------------------------------------------------
__device__ __forceinline__ float gf_u8_to_f(unsigned word, int k)   // byte k of word as a float, no I2F:
{                                                                   // 0x4B0000bb is the float 8388608 + bb
#ifdef GF_CPU_EMU
    return (float)((word >> (8 * k)) & 255u);
#else
    return __uint_as_float(__byte_perm(word, 0x4B000000u, 0x7650 + k)) - 8388608.0f;
#endif
}
__device__ __forceinline__ unsigned gf_f_to_u8(float q255)
{
#ifdef GF_CPU_EMU
    const int r = (int)std::nearbyint(q255);
#else
    const int r = __float2int_rn(q255);                // cvRound: round half to even
#endif
    return (unsigned)(r < 0 ? 0 : (r > 255 ? 255 : r));   // saturate_cast<uchar>
}
__device__ __forceinline__ float gf_ld1(const float* p) { return *p; }
__device__ __forceinline__ float gf_ld1(const unsigned char* p) { return (float)*p; }
__device__ __forceinline__ void gf_st1(float* p, float v) { *p = v; }
__device__ __forceinline__ void gf_st1(unsigned char* p, float v) { *p = (unsigned char)gf_f_to_u8(v); }

#define GF_REFLECT101 0
#define GF_TRUNCATE 1
#define GF_REFLECT 2

// One image plane as the kernels see it: element (y, x, c) of frame f lives at
// ptr[f*frame_stride + y*stride + x*xstep + coff].
struct GfPlane {
    float* ptr;
    int64_t stride;        // row stride, floats
    int64_t frame_stride;  // batch stride, floats
    int xstep;             // floats between horizontally adjacent pixels (= channel count)
    int coff;              // channel offset
};

struct GfArgs {
    GfPlane guide, src, dst, A, B;  // A/B optional (ptr == nullptr)
    int width;
    int height;     // height of the WHOLE image: the border rule refers to it
    int buf_y0;     // global row index of row 0 of guide/src
    int out_y0;     // first output row (global); dst.ptr points at it
    int out_rows;
    int r;
    int border;
    int wc;         // output columns per CTA (strip width)
    int hb;         // output rows per CTA (band height)
    float eps;
    float* ring;    // global scratch for the stage-2 row ring when it does not fit in smem
};

// Source coordinate of extended coordinate i under the border rule; -1 = contributes nothing.
// REFLECT101 for a single overshoot is the reference's reflectBorder (guided_filter_d.cu:
// 415-418); the periodic extension keeps it defined for r >= n (cv::borderInterpolate).
__host__ __device__ __forceinline__ int gf_map(int i, int n, int border)
{
    if (i >= 0 && i < n) return i;
    if (border == GF_TRUNCATE) return -1;
    if (n == 1) return 0;
    if (border == GF_REFLECT101) {
        const int period = 2 * n - 2;
        int m = i % period;
        if (m < 0) m += period;
        return m < n ? m : period - m;
    }
    const int period = 2 * n;
    int m = i % period;
    if (m < 0) m += period;
    return m < n ? m : period - 1 - m;
}

// 1 / (number of pixels the 1-D window [i-r, i+r] covers).  TRUNCATE: the true count
// (gIntegralToMean, guided_filter_d.cu:251-262); otherwise 2r+1.
__host__ __device__ __forceinline__ float gf_inv_count(int i, int n, int r, int border)
{
    if (border != GF_TRUNCATE) return 1.0f / (float)(2 * r + 1);
    int lo = i - r < 0 ? 0 : i - r;
    int hi = i + r > n - 1 ? n - 1 : i + r;
    int c = hi - lo + 1;
    return 1.0f / (float)(c < 1 ? 1 : c);
}

// Division by a pixel count as a two-term reciprocal: x/cnt = x*hi + x*lo to ~2^-45.
// A single rounded reciprocal (x * fl(1/cnt)) biases every mean by up to 6e-8 relative in ONE
// direction; that systematic shift was enough to flip ~150 pixels of the reference's uint8 KAT
// (values sitting on x.5), against ~10 with an exact division (profiles/, DESIGN.md).
struct GfNorm { float hi, lo; };
__host__ __device__ __forceinline__ GfNorm gf_norm_make(float cnt)
{
    GfNorm n;
    n.hi = 1.0f / cnt;
    n.lo = fmaf(-cnt, n.hi, 1.0f) * n.hi;      // first Newton residual of the rounded reciprocal
    return n;
}
// device-speed variant: hi from the fast reciprocal; hi + lo is just as accurate because lo is
// the residual of whatever hi is
__device__ __forceinline__ GfNorm gf_norm_fast(float cnt)
{
    GfNorm n;
    n.hi = __fdividef(1.0f, cnt);
    n.lo = fmaf(-cnt, n.hi, 1.0f) * n.hi;
    return n;
}
__host__ __device__ __forceinline__ float gf_norm_apply(float x, const GfNorm& n) { return fmaf(x, n.hi, x * n.lo); }

// number of pixels the 1-D window [i-r, i+r] covers, as an exact float
__host__ __device__ __forceinline__ float gf_count(int i, int n, int r, int border)
{
    if (border != GF_TRUNCATE) return (float)(2 * r + 1);
    int lo = i - r < 0 ? 0 : i - r;
    int hi = i + r > n - 1 ? n - 1 : i + r;
    int c = hi - lo + 1;
    return (float)(c < 1 ? 1 : c);
}
