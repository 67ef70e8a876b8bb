// gf_api.cu -- implementation of the C ABI declared in include/gf_b200.h.
//
// Host logic only: argument checks, kernel-family choice, launch geometry.  Every compute entry
// launches hand-written sm_100a kernels; there is no CPU path (a missing device surfaces as
// GF_ERR_CUDA from the first launch).
#include <stdarg.h>
#include <stddef.h>
#include <stdio.h>

#include <atomic>
#include <mutex>
#include <string>

#include "../../include/gf_b200.h"
#include "gf_generic.cuh"
#include "gf_job.h"
#include "gf_pointwise.cuh"
#include "gf_integral.cuh"
#include "gf_gauss.cuh"
#include "gf_fgf.cuh"
#include "gf_scan.cuh"
#include "gf_rt.h"
#ifdef GF_HAVE_FAST
#include "gf_fast.cuh"
#include "gf_wp.cuh"
// the big kernel families live in their own translation units (gf_tu_s8.cu, gf_tu_ws.cu, gf_tu_c4.cu, gf_tu_c4u8.cu) so
// that the library builds in parallel
const char* gf_s8_try_x(const Job& j, bool* done, const char** name, bool u8);
const char* gf_ws_try_x(const Job& j, bool* done, const char** name);
const char* gf_c4_try_x(const Job& j, bool* done, const char** name);
const char* gf_c4u8_try_x(const Job& j, bool* done, const char** name);
static inline const char* gf_s8_try(const Job& j, bool* done, const char** name, bool u8 = false) { return gf_s8_try_x(j, done, name, u8); }
static inline const char* gf_ws_try(const Job& j, bool* done, const char** name) { return gf_ws_try_x(j, done, name); }
static inline const char* gf_c4_try(const Job& j, bool* done, const char** name) { return gf_c4_try_x(j, done, name); }
#endif

namespace {

thread_local std::string g_err;
thread_local const char* g_kernel = "none";
thread_local std::string g_kernel_fgf;       // "fgf/<low-res kernel>" ("fgf_u8/..."), the name gf_fast_guided_gray(_u8) reports
std::atomic<int64_t> g_launches{0};

int fail(gf_status s, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return (int)s;
}

inline int div_up(int a, int b) { return (a + b - 1) / b; }
inline int round_up(int a, int b) { return div_up(a, b) * b; }

int check_common(const Job& j)
{
    if (!j.guide.ptr || !j.src.ptr || !j.dst.ptr) return fail(GF_ERR_INVALID, "null image pointer");
    if (j.width <= 0 || j.height <= 0 || j.out_rows <= 0 || j.count <= 0)
        return fail(GF_ERR_INVALID, "non-positive size (w=%d h=%d rows=%d count=%d)", j.width, j.height, j.out_rows, j.count);
    if (j.r < 0) return fail(GF_ERR_INVALID, "negative radius %d", j.r);
    if (j.border < 0 || j.border > 2) return fail(GF_ERR_INVALID, "unknown border mode %d", j.border);
    if (!(j.eps >= 0.f)) return fail(GF_ERR_INVALID, "eps must be >= 0");
    if (j.guide.stride < (int64_t)j.width * j.guide.channels || j.src.stride < (int64_t)j.width * j.src.channels ||
        j.dst.stride < (int64_t)j.width * j.dst.channels)
        return fail(GF_ERR_INVALID, "row stride smaller than a row");
    if ((j.A.ptr == nullptr) != (j.B.ptr == nullptr)) return fail(GF_ERR_INVALID, "A and B must both be given or both be NULL");
    if (j.A.ptr && (j.A.stride < (int64_t)j.width || j.B.stride < (int64_t)j.width)) return fail(GF_ERR_INVALID, "A/B row stride smaller than a row");
    if (j.out_y0 < 0 || j.out_y0 + j.out_rows > j.height) return fail(GF_ERR_INVALID, "output rows outside the image");
    // the rows the filter reads (after the border rule) must be inside the buffer
    int lo = j.height, hi = -1;
    for (int y = j.out_y0 - 2 * j.r; y < j.out_y0 + j.out_rows + 2 * j.r; ++y) {
        const int s = gf_map(y, j.height, j.border);
        if (s < 0) continue;
        lo = s < lo ? s : lo;
        hi = s > hi ? s : hi;
    }
    if (lo < j.buf_y0 || hi >= j.buf_y0 + j.buf_rows)
        return fail(GF_ERR_INVALID, "input buffer holds rows [%d,%d) but rows [%d,%d] are needed (2r halo missing?)",
                    j.buf_y0, j.buf_y0 + j.buf_rows, lo, hi);
    return GF_OK;
}

// ---- generic kernel geometry -------------------------------------------------------------------
struct GenericCfg {
    int win, wc, hb, nstrips, nbands;
    bool ring_smem;
    size_t smem_bytes, ring_floats_per_cta;
};

// nq_pub: values published per thread for the horizontal sums; nq_ring: values in the row ring
int plan_generic(const Job& j, int halo_cols, int halo_rows, int nq_pub, int nq_ring, GenericCfg* c)
{
    auto smem_floats = [&](int win, bool ring) {
        size_t n = (size_t)nq_pub * (win + 32);
        if (ring) n += (size_t)nq_ring * (2 * j.r + 1) * win;
        return n;
    };
    // halo_cols = 4r for the fused filter, 2r for the box filter
    int sms = 148, cc_major = 0, cc_minor = 0;
    gf_rt_device_info(&sms, &cc_major, &cc_minor);
    const int cands[5] = {round_up(j.width + halo_cols, 32), 128, 256, 512, 1024};
    const size_t max_smem = gf_rt_max_smem();
    int best = -1;
    double best_score = -1;
    bool best_ring = false;
    for (int i = 0; i < 5; ++i) {
        const int win = cands[i];
        if (win > 1024 || win - halo_cols < 32) {
            if (!(i == 0 && win <= 1024 && win - halo_cols >= j.width)) continue;
        }
        const int wc = win - halo_cols;
        if (wc < 1) continue;
        const bool ring_fits = smem_floats(win, true) * sizeof(float) <= max_smem;
        const int used = wc < j.width ? wc : j.width;
        double score = (double)used / win + (ring_fits ? 1.0 : 0.0) - 1e-4 * win / 1024.0;
        if (score > best_score) { best_score = score; best = win; best_ring = ring_fits; }
    }
    if (best < 0)
        return fail(GF_ERR_UNSUPPORTED, "radius %d too large for the streaming kernel (needs %d halo columns of at most 1024 threads)",
                    j.r, halo_cols);
    c->win = best;
    c->wc = best - halo_cols;
    c->ring_smem = best_ring;
    c->nstrips = div_up(j.width, c->wc);
    const int target = 4 * sms;
    int nb = target / (c->nstrips * j.count);
    if (nb < 1) nb = 1;
    int hb = div_up(j.out_rows, nb);
    const int hb_min = 2 * halo_rows > 16 ? 2 * halo_rows : 16;   // keep the warm-up rows <= 50% of a band
    if (hb < hb_min) hb = hb_min;
    if (hb > j.out_rows) hb = j.out_rows;
    c->hb = hb;
    c->nbands = div_up(j.out_rows, hb);
    c->smem_bytes = smem_floats(c->win, c->ring_smem) * sizeof(float);
    c->ring_floats_per_cta = c->ring_smem ? 0 : (size_t)nq_ring * (2 * j.r + 1) * c->win;
    return GF_OK;
}

GfArgs mk_args(const Job& j)
{
    GfArgs a;
    a.guide = mk(j.guide); a.src = mk(j.src); a.dst = mk(j.dst); a.A = mk(j.A); a.B = mk(j.B);
    a.width = j.width; a.height = j.height; a.buf_y0 = j.buf_y0; a.out_y0 = j.out_y0; a.out_rows = j.out_rows;
    a.r = j.r; a.border = j.border; a.eps = j.eps; a.wc = 0; a.hb = 0; a.ring = nullptr;
    return a;
}

template <class M>
int launch_generic(const Job& j)
{
    GenericCfg c;
    int rc = plan_generic(j, 4 * j.r, 4 * j.r, M::NQ1 + M::NQ2, M::NQ2, &c);
    if (rc) return rc;
    GfArgs a = mk_args(j);
    a.wc = c.wc; a.hb = c.hb;
    void* ring = nullptr;
    if (!c.ring_smem) {
        const size_t n = c.ring_floats_per_cta * c.nstrips * c.nbands * j.count * sizeof(float);
        if (const char* e = gf_rt_alloc_async(&ring, n, j.stream)) return fail(GF_ERR_NOMEM, "ring scratch (%zu bytes): %s", n, e);
        a.ring = (float*)ring;
    }
    auto kfn = gf_generic_kernel<M>;
    if (const char* e = gf_rt_set_smem(kfn, c.smem_bytes)) return fail(GF_ERR_CUDA, "smem attribute: %s", e);
    dim3 grid(c.nstrips, c.nbands, j.count), block(c.win);
    GF_LAUNCH(kfn, grid, block, c.smem_bytes, j.stream, a);
    const char* e = gf_rt_launch_error();
    if (ring) gf_rt_free_async(ring, j.stream);
    if (e) return fail(GF_ERR_CUDA, "gf_generic_kernel launch: %s", e);
    g_launches++;
    g_kernel = M::NQ1 == 4 ? "generic_gray" : "generic_color";
    return GF_OK;
}

// Do `count` frames of a (a_rows rows each) and of b (b_rows rows each) share memory?  A strip job's destination holds
// its out_rows rows, its guide and source the buf_rows rows of the buffer.
bool overlaps(const Plane& a, int a_rows, const Plane& b, int b_rows, int count)
{
    if (!a.ptr || !b.ptr) return false;
    const float* a1 = a.ptr + (count - 1) * a.frame_stride + (int64_t)a_rows * a.stride;
    const float* b1 = b.ptr + (count - 1) * b.frame_stride + (int64_t)b_rows * b.stride;
    return a.ptr < b1 && b.ptr < a1;
}

// ---- scan path (gf_scan.cuh): any radius, full frames, gray ------------------------------------------------
static bool scan_ok(const Job& j)
{
    if (j.color || j.guide.channels != 1 || j.src.channels != 1 || j.dst.channels != 1 || j.guide.coff || j.src.coff || j.dst.coff) return false;
    if (j.buf_y0 != 0 || j.out_y0 != 0 || j.buf_rows != j.height || j.out_rows != j.height) return false;     // full frames only
    return j.r >= 1 && (j.border == GF_TRUNCATE || (j.r < j.width && j.r < j.height));                       // single reflections (TRUNCATE: any radius)
}

// box mean of plane `a` (or of a*b) into `out`, through the row-prefix scratch P
static const char* scan_box(const float* a, int64_t sa, const float* b, int64_t sb, float* out, int64_t so, double* P, int w, int h, int r,
                            int border, void* stream)
{
    GfScanPrefixArgs pa;
    pa.a = a; pa.b = b; pa.P = P; pa.width = w; pa.height = h; pa.sa = sa; pa.sb = sb; pa.sp = w;
    dim3 g1(h < 8192 ? h : 8192), b1(256);
    if (b) { auto k = gf_rowprefix_kernel<1, float, double>; GF_LAUNCH(k, g1, b1, 0, stream, pa); }
    else { auto k = gf_rowprefix_kernel<0, float, double>; GF_LAUNCH(k, g1, b1, 0, stream, pa); }
    GfScanBoxArgs ba;
    ba.P = P; ba.out = out; ba.width = w; ba.height = h; ba.r = r; ba.border = border; ba.sp = w; ba.so = so;
    // bands: enough CTAs to fill the GPU, but tall enough that the 2r-row warm-up of a band stays below half its rows
    int sms = 148, mj = 0, mn = 0;
    gf_rt_device_info(&sms, &mj, &mn);
    const int cols = div_up(w, 128);
    int nb = div_up(8 * sms, cols);
    int hb = div_up(h, nb < 1 ? 1 : nb);
    if (hb < 2 * r) hb = 2 * r;
    if (hb > h) hb = h;
    ba.hb = hb;
    dim3 g2(cols, div_up(h, hb)), b2(128);
    auto k2 = gf_boxcols_kernel<double, float, true>;
    GF_LAUNCH(k2, g2, b2, 0, stream, ba);
    return gf_rt_launch_error();
}

// exact window sums of uint8 planes (or of their product) as int64
static const char* scan_sums_u8(const unsigned char* a, int64_t sa, const unsigned char* b, int64_t sb, long long* out, int64_t so, long long* P,
                                int w, int h, int r, int border, void* stream)
{
    GfScanPrefixArgsU8 pa;
    pa.a = a; pa.b = b; pa.P = P; pa.width = w; pa.height = h; pa.sa = sa; pa.sb = sb; pa.sp = w;
    dim3 g1(h < 8192 ? h : 8192), b1(256);
    if (b) { auto k = gf_rowprefix_kernel<1, unsigned char, long long>; GF_LAUNCH(k, g1, b1, 0, stream, pa); }
    else { auto k = gf_rowprefix_kernel<0, unsigned char, long long>; GF_LAUNCH(k, g1, b1, 0, stream, pa); }
    GfScanBoxArgsU8 ba;
    ba.P = P; ba.out = out; ba.width = w; ba.height = h; ba.r = r; ba.border = border; ba.sp = w; ba.so = so;
    int sms = 148, mj = 0, mn = 0;
    gf_rt_device_info(&sms, &mj, &mn);
    const int cols = div_up(w, 128);
    int nb = div_up(8 * sms, cols);
    int hb = div_up(h, nb < 1 ? 1 : nb);
    if (hb < 2 * r) hb = 2 * r;
    if (hb > h) hb = h;
    ba.hb = hb;
    dim3 g2(cols, div_up(h, hb)), b2(128);
    auto k2 = gf_boxcols_kernel<long long, long long, false>;
    GF_LAUNCH(k2, g2, b2, 0, stream, ba);
    return gf_rt_launch_error();
}

static int run_scan_gray(const Job& j)
{
    const int w = j.width, h = j.height;
    const size_t n = (size_t)w * h;
    void* scratch = nullptr;
    if (const char* e = gf_rt_alloc_async(&scratch, n * (8 + 4 * 4), j.stream)) return fail(GF_ERR_NOMEM, "scan-path scratch (%zu bytes): %s", n * 24, e);
    double* P = (double*)scratch;
    float* im = (float*)(P + n), *pm = im + n, *ipm = pm + n, *iim = ipm + n;
    const char* e = nullptr;
    for (int f = 0; f < j.count && !e; ++f) {
        const float* I = j.guide.ptr + f * j.guide.frame_stride;
        const float* p = j.src.ptr + f * j.src.frame_stride;
        float* q = const_cast<float*>(j.dst.ptr) + f * j.dst.frame_stride;
        if (!e) e = scan_box(I, j.guide.stride, nullptr, 0, im, w, P, w, h, j.r, j.border, j.stream);
        if (!e) e = scan_box(p, j.src.stride, nullptr, 0, pm, w, P, w, h, j.r, j.border, j.stream);
        if (!e) e = scan_box(I, j.guide.stride, p, j.src.stride, ipm, w, P, w, h, j.r, j.border, j.stream);
        if (!e) e = scan_box(I, j.guide.stride, I, j.guide.stride, iim, w, P, w, h, j.r, j.border, j.stream);
        if (!e) {
            GfScanAbArgs ab;
            ab.im = im; ab.pm = pm; ab.ipm_a = ipm; ab.iim_b = iim; ab.width = w; ab.height = h; ab.s = w; ab.eps = j.eps;
            dim3 g(div_up(w, 256), h < 1024 ? h : 1024), b(256);
            auto k = gf_scan_ab_kernel;
            GF_LAUNCH(k, g, b, 0, j.stream, ab);
            e = gf_rt_launch_error();
        }
        if (!e && j.A.ptr) {
            float* A = const_cast<float*>(j.A.ptr) + f * j.A.frame_stride;
            float* B = const_cast<float*>(j.B.ptr) + f * j.B.frame_stride;
            e = gf_rt_copy2d_async(A, j.A.stride * 4, ipm, (size_t)w * 4, (size_t)w * 4, h, j.stream);
            if (!e) e = gf_rt_copy2d_async(B, j.B.stride * 4, iim, (size_t)w * 4, (size_t)w * 4, h, j.stream);
        }
        if (!e) e = scan_box(ipm, w, nullptr, 0, im, w, P, w, h, j.r, j.border, j.stream);       // mean_a -> im
        if (!e) e = scan_box(iim, w, nullptr, 0, pm, w, P, w, h, j.r, j.border, j.stream);       // mean_b -> pm
        if (!e) {
            GfPwArgs a;
            a.in0 = I; a.in1 = im; a.in2 = pm; a.in3 = nullptr; a.out = q;
            a.width = w; a.height = h; a.cs = 1; a.cg = 1; a.ss = w; a.sg = j.guide.stride; a.eps = 0.f;
            // q = I * mean_a + mean_b: the source-shaped operands (mean_a, mean_b, q) share ONE stride in the kernel, so a
            // pitched destination goes through a packed temporary row layout only when it has to
            if (j.dst.stride == w) {
                dim3 g(div_up(w, 256), h < 1024 ? h : 1024), b(256);
                auto k = gf_pointwise_kernel<GF_PW_LINEAR>;
                GF_LAUNCH(k, g, b, 0, j.stream, a);
                e = gf_rt_launch_error();
            } else {
                a.out = ipm;
                dim3 g(div_up(w, 256), h < 1024 ? h : 1024), b(256);
                auto k = gf_pointwise_kernel<GF_PW_LINEAR>;
                GF_LAUNCH(k, g, b, 0, j.stream, a);
                e = gf_rt_launch_error();
                if (!e) e = gf_rt_copy2d_async(q, j.dst.stride * 4, ipm, (size_t)w * 4, (size_t)w * 4, h, j.stream);
            }
        }
    }
    gf_rt_free_async(scratch, j.stream);
    if (e) return fail(GF_ERR_CUDA, "scan path: %s", e);
    g_launches += 15L * j.count;
    g_kernel = "scan_gray";
    return GF_OK;
}

int run_job(const Job& j)
{
    int rc = GF_OK;
    bool done = false;
    if (GF_KNOB("GF_SCAN", 0) && scan_ok(j)) return run_scan_gray(j);      // measurement / tests: force the scan path
#ifdef GF_HAVE_FAST
    {
        const char* name = nullptr;
        const char* e = gf_c4_try(j, &done, &name);
        if (!done) e = gf_ws_try(j, &done, &name);
        if (!done) e = gf_s8_try(j, &done, &name);
        if (!done) e = gf_wp_try(j, &done, &name);
        if (!done) e = gf_fast_try(j, &done, &name);
        if (done) {
            if (e) rc = fail(GF_ERR_CUDA, "%s launch: %s", name, e);
            else { rc = GF_OK; g_launches++; g_kernel = name; }
        }
    }
#endif
    // radii beyond the tuned kernels: the scan path is O(1) in r and measured faster than the thread-per-column kernel
    // from r ~ 48 on (profiles/r2_scan_vs_sliding.jsonl: 4K r=64 2.26 ms against 2.94 ms)
    if (!done && !j.color && j.r >= 48 && !j.A.ptr && scan_ok(j)) return run_scan_gray(j);
    if (!done) rc = j.color ? launch_generic<GfColorModel>(j) : launch_generic<GfGrayModel>(j);
    // radii the streaming kernels cannot hold (4r halo columns of at most 1024 threads): the scan path takes any radius
    if (!done && rc == GF_ERR_UNSUPPORTED && scan_ok(j)) rc = run_scan_gray(j);
    return rc;
}

// Runs n jobs that write (channels of) one destination buffer.  The streaming kernels read
// halos that other CTAs may already have overwritten, so a destination that aliases an input
// goes through a stream-ordered temporary (the reference can run in place only because every
// stage round-trips its scratch planes).
int run_jobs(Job* js, int n)
{
    const Job& j0 = js[0];
    for (int i = 0; i < n; ++i)
        if (int rc0 = check_common(js[i])) return rc0;     // refuse bad arguments before anything is allocated
    const bool alias = overlaps(j0.dst, j0.out_rows, j0.guide, j0.buf_rows, j0.count) ||
                       overlaps(j0.dst, j0.out_rows, j0.src, j0.buf_rows, j0.count);
    void* tmp = nullptr;
    const size_t row_bytes = (size_t)j0.width * j0.dst.channels * sizeof(float);
    const Plane user_dst = j0.dst;
    int rc = GF_OK;
    if (alias) {
        const size_t bytes = row_bytes * j0.out_rows * j0.count;
        if (const char* e = gf_rt_alloc_async(&tmp, bytes, j0.stream)) return fail(GF_ERR_NOMEM, "in-place temporary: %s", e);
        for (int i = 0; i < n; ++i) {
            js[i].dst.ptr = (const float*)tmp;
            js[i].dst.stride = (int64_t)j0.width * j0.dst.channels;
            js[i].dst.frame_stride = js[i].dst.stride * j0.out_rows;
        }
    }
    for (int i = 0; i < n && rc == GF_OK; ++i) rc = run_job(js[i]);
    if (tmp) {
        if (rc == GF_OK)
            for (int f = 0; f < j0.count; ++f)
                if (const char* e = gf_rt_copy2d_async(const_cast<float*>(user_dst.ptr) + f * user_dst.frame_stride,
                                                       user_dst.stride * sizeof(float),
                                                       (const float*)tmp + f * js[0].dst.frame_stride, row_bytes, row_bytes,
                                                       j0.out_rows, j0.stream))
                    rc = fail(GF_ERR_CUDA, "copy back: %s", e);
        gf_rt_free_async(tmp, j0.stream);
    }
    return rc;
}

int64_t or_packed(int64_t stride, int width, int channels) { return stride > 0 ? stride : (int64_t)width * channels; }

}  // namespace

struct gf_filter {
    int width, height, gch, sch;
};


#ifdef GF_HAVE_FAST
// The class API's multi-channel modes ((1,3): one gray guide for three source channels -- the reference's
// own demo, main.cpp:141-150 -- and (3,3): channel by channel) on the tuned planar kernel: de-interleave the
// source (and a 3-channel guide) into stream-ordered scratch planes, ONE s8 launch over the channels as
// "frames" (a gray guide is shared: frame stride 0), re-interleave.  Returns false when the tuned kernel does
// not take the job (the caller then runs the generic per-channel path); *rc is the status otherwise.
static bool run_planar(const gf_filter& h, const float* guide, const float* src, float* dst, int64_t gs, int64_t ss, int64_t ds,
                       int r, float eps, int border, void* stream, int* rc)
{
    const int w = h.width, hh = h.height, C = h.sch;
    if (!(h.gch == 1 || h.gch == C) || C < 2 || C > 4) return false;
    if (!guide || !src || !dst || r < 0 || !(eps >= 0.f)) return false;       // let the generic path report it
    // nothing is launched on the caller's pointers before the arguments are known to be sane (the generic path reports them)
    if (ss < (int64_t)w * C || ds < (int64_t)w * C || gs < (int64_t)w * h.gch || border < 0 || border > 2) return false;
    const int64_t pitch = ((int64_t)w + 7) / 8 * 8, plane = pitch * hh;
    const int nplanes = 2 * C + (h.gch > 1 ? C : 0);
    void* scratch = nullptr;
    if (const char* ae = gf_rt_alloc_async(&scratch, (size_t)nplanes * plane * sizeof(float), stream)) {
        *rc = fail(GF_ERR_NOMEM, "scratch planes of the class path (%zu bytes): %s", (size_t)nplanes * plane * sizeof(float), ae);
        return true;
    }
    float* sp = (float*)scratch;                 // [src planes | dst planes | guide planes]
    float* dp = sp + (int64_t)C * plane;
    float* gp = dp + (int64_t)C * plane;
    Job j;
    j.count = C;
    j.width = w; j.height = hh; j.buf_rows = hh; j.out_rows = hh;
    j.r = r; j.eps = eps; j.border = border; j.stream = stream;
    j.guide = h.gch == 1 ? Plane{guide, gs, 0, 1, 0} : Plane{gp, pitch, plane, 1, 0};
    j.src = Plane{sp, pitch, plane, 1, 0};
    j.dst = Plane{dp, pitch, plane, 1, 0};
    j.A = j.B = Plane{nullptr, 0, 0, 1, 0};
    auto shuffle = [&](bool to_planar, const float* inter, int64_t stride, float* planar, int ch) {
        GfIlArgs a;
        a.inter = const_cast<float*>(inter); a.planar = planar; a.stride = stride; a.pitch = pitch; a.plane = plane;
        a.width = w; a.height = hh; a.channels = ch;
        dim3 block(256), grid(div_up(w, 256), hh < 2048 ? hh : 2048);
        if (to_planar) { auto k = gf_interleave_kernel<true>; GF_LAUNCH(k, grid, block, 0, stream, a); }
        else { auto k = gf_interleave_kernel<false>; GF_LAUNCH(k, grid, block, 0, stream, a); }
    };
    shuffle(true, src, ss, sp, C);
    if (h.gch > 1) shuffle(true, guide, gs, gp, C);
    bool done = false;
    const char* name = nullptr;
    const char* e = nullptr;
    if (check_common(j) == GF_OK) {
        e = gf_ws_try(j, &done, &name);
        if (!done) e = gf_s8_try(j, &done, &name);
    }
    if (!done) {                                   // not a job for the tuned kernel: nothing was written to dst
        gf_rt_free_async(scratch, stream);
        return false;
    }
    if (!e) shuffle(false, dst, ds, dp, C);
    if (!e) e = gf_rt_launch_error();
    gf_rt_free_async(scratch, stream);
    if (e) { *rc = fail(GF_ERR_CUDA, "%s (planar class path): %s", name, e); return true; }
    g_launches += 3 + (h.gch > 1 ? 1 : 0);
    g_kernel = name;
    *rc = GF_OK;
    return true;
}
#endif

template <class T>
static int integral_entry(const unsigned char* src, T* integral, T* scratch, int sw, int sh, int w, int h, int64_t ss, int64_t ds,
                          void* stream, const char* name)
{
    if (!src || !integral) return fail(GF_ERR_INVALID, "%s: null pointer", name);
    if (sw <= 0 || sh <= 0 || w < sw || h < sh) return fail(GF_ERR_INVALID, "%s: bad size %dx%d -> %dx%d", name, sw, sh, w, h);
    if (ss <= 0) ss = sw;
    if (ds <= 0) ds = w;
    if (ss < sw || ds < w) return fail(GF_ERR_INVALID, "%s: row stride smaller than a row", name);
    int launches = 0;
    if (const char* e = gf_sat_launch<T>(src, integral, scratch, sw, sh, w, h, ss, ds, stream, &launches)) return fail(GF_ERR_CUDA, "%s: %s", name, e);
    g_launches += launches;
    g_kernel = sizeof(T) == 4 ? "integral_i32" : "integral_i64";
    return GF_OK;
}

extern "C" {

const char* gf_last_error(void) { return g_err.c_str(); }
int gf_version(void) { return 100; }
int gf_integral_u8_i32(const unsigned char* src, int32_t* integral, int32_t* scratch, int width, int height, int64_t src_stride,
                       int64_t dst_stride, void* stream)
{
    return integral_entry<int32_t>(src, integral, scratch, width, height, width, height, src_stride, dst_stride, stream, "gf_integral_u8_i32");
}
int gf_integral_u8_i64(const unsigned char* src, int64_t* integral, int64_t* scratch, int width, int height, int64_t src_stride,
                       int64_t dst_stride, void* stream)
{
    return integral_entry<int64_t>(src, integral, scratch, width, height, width, height, src_stride, dst_stride, stream, "gf_integral_u8_i64");
}
int gf_integral_u8_i32_padded(const unsigned char* src, int32_t* integral, int src_width, int src_height, int64_t src_stride,
                              int dst_width, int dst_height, void* stream)
{
    return integral_entry<int32_t>(src, integral, nullptr, src_width, src_height, dst_width, dst_height, src_stride, dst_width, stream,
                                   "gf_integral_u8_i32_padded");
}

int gf_gaussian_gray(const float* src, float* dst, int width, int height, int64_t src_stride, int64_t dst_stride, int radius,
                     double sigma, void* stream)
{
    if (!src || !dst) return fail(GF_ERR_INVALID, "gf_gaussian_gray: null pointer");
    if (src == dst) return fail(GF_ERR_INVALID, "gf_gaussian_gray: in-place filtering is not supported");
    if (width <= 0 || height <= 0) return fail(GF_ERR_INVALID, "gf_gaussian_gray: bad size %dx%d", width, height);
    if (radius < 0 || radius > GF_GAUSS_MAX_R) return fail(GF_ERR_INVALID, "gf_gaussian_gray: radius %d outside [0, %d]", radius, GF_GAUSS_MAX_R);
    if (src_stride <= 0) src_stride = width;
    if (dst_stride <= 0) dst_stride = width;
    if (src_stride < width || dst_stride < width) return fail(GF_ERR_INVALID, "gf_gaussian_gray: row stride smaller than a row");
    bool fast = false;
    if (const char* e = gf_gauss_launch(src, dst, width, height, src_stride, dst_stride, radius, sigma, stream, &fast))
        return fail(GF_ERR_CUDA, "gf_gaussian_gray: %s", e);
    g_launches += 1;
    g_kernel = fast ? "gauss4" : "gauss";
    return GF_OK;
}

const char* gf_last_kernel(void) { return g_kernel; }

int gf_set_option(const char* name, int value)
{
    if (!name || std::strncmp(name, "GF_", 3) != 0) return fail(GF_ERR_INVALID, "gf_set_option: option names start with GF_");
    GfKnobSlot* s = gf_knob_slot(name);
    if (!s) return fail(GF_ERR_NOMEM, "gf_set_option: option table full");
    s->value.store(value < 0 ? -1 : value, std::memory_order_relaxed);
    return GF_OK;
}
int64_t gf_launch_count(void) { return g_launches.load(); }

int gf_device_info(int* sm_count, int* cc_major, int* cc_minor)
{
    int a = 0, b = 0, c = 0;
    if (const char* e = gf_rt_device_info(&a, &b, &c)) return fail(GF_ERR_CUDA, "%s", e);
    if (sm_count) *sm_count = a;
    if (cc_major) *cc_major = b;
    if (cc_minor) *cc_minor = c;
    return GF_OK;
}

int gf_create(gf_handle* out, int width, int height, int guide_channels, int src_channels)
{
    if (!out) return fail(GF_ERR_INVALID, "null handle pointer");
    *out = nullptr;
    if (width <= 0 || height <= 0) return fail(GF_ERR_INVALID, "non-positive size %dx%d", width, height);
    const bool ok = (guide_channels == 1 && (src_channels == 1 || src_channels == 3)) ||
                    (guide_channels == 3 && (src_channels == 3 || src_channels == 1));
    if (!ok) return fail(GF_ERR_UNSUPPORTED, "Do not support channel: %d, %d", guide_channels, src_channels);
    gf_filter* f = new gf_filter{width, height, guide_channels, src_channels};
    *out = f;
    return GF_OK;
}

int gf_destroy(gf_handle h)
{
    delete h;
    return GF_OK;
}

int gf_run(gf_handle h, const float* guide, const float* src, float* dst, int r, float eps, int border,
           int64_t guide_stride, int64_t src_stride, int64_t dst_stride, void* stream)
{
    if (!h) return fail(GF_ERR_INVALID, "null handle");
    Job j;
    j.width = h->width; j.height = h->height; j.buf_rows = h->height; j.out_rows = h->height;
    j.r = r; j.eps = eps; j.border = border; j.stream = stream;
    const int64_t gs = or_packed(guide_stride, h->width, h->gch), ss = or_packed(src_stride, h->width, h->sch),
                  ds = or_packed(dst_stride, h->width, h->sch);
    if (h->gch == 3 && h->sch == 1) {           // colour guide, 3x3 covariance
        j.color = true;
        j.guide = Plane{guide, gs, 0, 3, 0};
        j.src = Plane{src, ss, 0, 1, 0};
        j.dst = Plane{dst, ds, 0, 1, 0};
        j.A = j.B = Plane{nullptr, 0, 0, 1, 0};
        return run_jobs(&j, 1);
    }
    // (1,1); (3,3) channel by channel; (1,3) one guide for three source channels
    // (guided_filter_d.cu:968-975)
#ifdef GF_HAVE_FAST
    if (h->sch > 1) {
        int rc = GF_OK;
        if (run_planar(*h, guide, src, dst, gs, ss, ds, r, eps, border, stream, &rc)) return rc;
    }
#endif
    Job js[3];
    for (int c = 0; c < h->sch; ++c) {
        js[c] = j;
        js[c].guide = Plane{guide, gs, 0, h->gch, h->gch == 1 ? 0 : c};
        js[c].src = Plane{src, ss, 0, h->sch, c};
        js[c].dst = Plane{dst, ds, 0, h->sch, c};
        js[c].A = js[c].B = Plane{nullptr, 0, 0, 1, 0};
    }
    return run_jobs(js, h->sch);
}

int gf_guided_gray(const float* guide, const float* src, float* dst, float* A, float* B, int width, int height,
                   int64_t guide_stride, int64_t src_stride, int64_t dst_stride, int64_t ab_stride, int r, float eps,
                   int border, void* stream)
{
    Job j;
    j.width = width; j.height = height; j.buf_rows = height; j.out_rows = height;
    j.r = r; j.eps = eps; j.border = border; j.stream = stream;
    j.guide = Plane{guide, or_packed(guide_stride, width, 1), 0, 1, 0};
    j.src = Plane{src, or_packed(src_stride, width, 1), 0, 1, 0};
    j.dst = Plane{dst, or_packed(dst_stride, width, 1), 0, 1, 0};
    j.A = Plane{A, or_packed(ab_stride, width, 1), 0, 1, 0};
    j.B = Plane{B, or_packed(ab_stride, width, 1), 0, 1, 0};
    return run_jobs(&j, 1);
}

int gf_guided_gray_u8(const unsigned char* guide, const unsigned char* src, unsigned char* dst, int width, int height,
                      int64_t guide_stride, int64_t src_stride, int64_t dst_stride, int r, float eps, int border, void* stream)
{
#ifdef GF_HAVE_FAST
    Job j;
    j.width = width; j.height = height; j.buf_rows = height; j.out_rows = height;
    j.r = r; j.eps = eps; j.border = border; j.stream = stream;
    // Plane carries float*: the u8 planes are reinterpreted, every stride is in ELEMENTS (= bytes here)
    j.guide = Plane{reinterpret_cast<const float*>(guide), or_packed(guide_stride, width, 1), 0, 1, 0};
    j.src = Plane{reinterpret_cast<const float*>(src), or_packed(src_stride, width, 1), 0, 1, 0};
    j.dst = Plane{reinterpret_cast<const float*>(dst), or_packed(dst_stride, width, 1), 0, 1, 0};
    j.A = j.B = Plane{nullptr, 0, 0, 1, 0};
    if (int rc = check_common(j)) return rc;
    {   // any overlap of the output with an input, not just equal pointers (byte ranges: the planes hold unsigned char)
        auto ov = [&](const unsigned char* a, int64_t sa, const unsigned char* b, int64_t sb) {
            return a < b + (int64_t)height * sb && b < a + (int64_t)height * sa;
        };
        if (ov(dst, j.dst.stride, guide, j.guide.stride) || ov(dst, j.dst.stride, src, j.src.stride))
            return fail(GF_ERR_UNSUPPORTED, "gf_guided_gray_u8: in-place filtering is not supported");
    }
    bool done = false;
    const char* name = nullptr;
    const char* e = gf_s8_try(j, &done, &name, true);
    if (!done)
        return fail(GF_ERR_UNSUPPORTED, "gf_guided_gray_u8 needs r in {1..8,16}, width >= 64, height >= 4r+2, 8-byte aligned rows "
                                        "(stride %% 8 == 0) and, for the TRUNCATE border, width %% 8 == 0 and >= 256");
    if (e) return fail(GF_ERR_CUDA, "%s launch: %s", name, e);
    g_launches++;
    g_kernel = name;
    return GF_OK;
#else
    return fail(GF_ERR_UNSUPPORTED, "gf_guided_gray_u8: built without the tuned kernels");
#endif
}

int gf_guided_color(const float* guide3, const float* src, float* dst, int width, int height, int src_channels,
                    int64_t guide_stride, int64_t src_stride, int64_t dst_stride, int r, float eps, int border, void* stream)
{
    if (src_channels != 1 && src_channels != 3) return fail(GF_ERR_UNSUPPORTED, "Do not support channel: 3, %d", src_channels);
    Job j;
    j.width = width; j.height = height; j.buf_rows = height; j.out_rows = height;
    j.r = r; j.eps = eps; j.border = border; j.stream = stream; j.color = true;
    j.guide = Plane{guide3, or_packed(guide_stride, width, 3), 0, 3, 0};
    j.A = j.B = Plane{nullptr, 0, 0, 1, 0};
    Job js[3];
    for (int c = 0; c < src_channels; ++c) {
        js[c] = j;
        js[c].src = Plane{src, or_packed(src_stride, width, src_channels), 0, src_channels, c};
        js[c].dst = Plane{dst, or_packed(dst_stride, width, src_channels), 0, src_channels, c};
    }
    return run_jobs(js, src_channels);
}

int gf_guided_color_u8(const unsigned char* guide3, const unsigned char* src, unsigned char* dst, int width, int height,
                       int src_channels, int64_t guide_stride, int64_t src_stride, int64_t dst_stride, int r, float eps,
                       int border, void* stream)
{
#ifdef GF_HAVE_FAST
    if (src_channels != 1 && src_channels != 3) return fail(GF_ERR_UNSUPPORTED, "Do not support channel: 3, %d", src_channels);
    Job j;
    j.count = src_channels;                 // one launch: the frames of the c4 kernel are the source channels
    j.width = width; j.height = height; j.buf_rows = height; j.out_rows = height;
    j.r = r; j.eps = eps; j.border = border; j.stream = stream; j.color = true;
    // Plane carries float*: the u8 planes are reinterpreted, every stride is in ELEMENTS (= bytes here)
    j.guide = Plane{reinterpret_cast<const float*>(guide3), or_packed(guide_stride, width, 3), 0, 3, 0};
    j.src = Plane{reinterpret_cast<const float*>(src), or_packed(src_stride, width, src_channels), 0, src_channels, 0};
    j.dst = Plane{reinterpret_cast<const float*>(dst), or_packed(dst_stride, width, src_channels), 0, src_channels, 0};
    j.A = j.B = Plane{nullptr, 0, 0, 1, 0};
    if (int rc = check_common(j)) return rc;
    {   // any overlap of the output with an input, not just equal pointers (byte ranges: the planes hold unsigned char)
        auto ov = [&](const unsigned char* a, int64_t sa, const unsigned char* b, int64_t sb) {
            return a < b + (int64_t)height * sb && b < a + (int64_t)height * sa;
        };
        if (ov(dst, j.dst.stride, guide3, j.guide.stride) || ov(dst, j.dst.stride, src, j.src.stride))
            return fail(GF_ERR_UNSUPPORTED, "gf_guided_color_u8: in-place filtering is not supported");
    }
    bool done = false;
    const char* name = nullptr;
    const char* e = gf_c4u8_try_x(j, &done, &name);
    if (!done)
        return fail(GF_ERR_UNSUPPORTED, "gf_guided_color_u8 needs r in {4,8,12,16}, width %% 4 == 0, width >= 128, height >= 4r+2, "
                                        "rows x stride < 2^31 and 4-byte aligned planes and row strides");
    if (e) return fail(GF_ERR_CUDA, "%s launch: %s", name, e);
    g_launches++;
    g_kernel = name;
    return GF_OK;
#else
    return fail(GF_ERR_UNSUPPORTED, "gf_guided_color_u8: built without the tuned kernels");
#endif
}

int gf_guided_batch(const float* guide, const float* src, float* dst, int count, int width, int height, int guide_channels,
                    int64_t guide_stride, int64_t src_stride, int64_t dst_stride, int64_t guide_frame_stride,
                    int64_t src_frame_stride, int64_t dst_frame_stride, int r, float eps, int border, void* stream)
{
    if (guide_channels != 1 && guide_channels != 3) return fail(GF_ERR_UNSUPPORTED, "Do not support channel: %d, 1", guide_channels);
    Job j;
    j.count = count;
    j.width = width; j.height = height; j.buf_rows = height; j.out_rows = height;
    j.r = r; j.eps = eps; j.border = border; j.stream = stream; j.color = guide_channels == 3;
    const int64_t gs = or_packed(guide_stride, width, guide_channels), ss = or_packed(src_stride, width, 1),
                  ds = or_packed(dst_stride, width, 1);
    j.guide = Plane{guide, gs, guide_frame_stride > 0 ? guide_frame_stride : gs * height, guide_channels, 0};
    j.src = Plane{src, ss, src_frame_stride > 0 ? src_frame_stride : ss * height, 1, 0};
    j.dst = Plane{dst, ds, dst_frame_stride > 0 ? dst_frame_stride : ds * height, 1, 0};
    j.A = j.B = Plane{nullptr, 0, 0, 1, 0};
    return run_jobs(&j, 1);
}

static Job strip_job(const float* guide, const float* src, float* dst, int width, int global_height, int buf_y0, int buf_rows, int out_y0,
                     int out_rows, int64_t guide_stride, int64_t src_stride, int64_t dst_stride, int r, float eps, int border, void* stream)
{
    Job j;
    j.width = width; j.height = global_height; j.buf_y0 = buf_y0; j.buf_rows = buf_rows; j.out_y0 = out_y0; j.out_rows = out_rows;
    j.r = r; j.eps = eps; j.border = border; j.stream = stream;
    j.guide = Plane{guide, or_packed(guide_stride, width, 1), 0, 1, 0};
    j.src = Plane{src, or_packed(src_stride, width, 1), 0, 1, 0};
    j.dst = Plane{dst, or_packed(dst_stride, width, 1), 0, 1, 0};
    j.A = j.B = Plane{nullptr, 0, 0, 1, 0};
    return j;
}

int gf_guided_gray_strip(const float* guide, const float* src, float* dst, int width, int global_height, int buf_y0,
                         int buf_rows, int out_y0, int out_rows, int64_t guide_stride, int64_t src_stride,
                         int64_t dst_stride, int r, float eps, int border, void* stream)
{
    if (buf_rows <= 0 || buf_y0 < 0 || buf_y0 + buf_rows > global_height) return fail(GF_ERR_INVALID, "buffer rows outside the image");
    Job j = strip_job(guide, src, dst, width, global_height, buf_y0, buf_rows, out_y0, out_rows, guide_stride, src_stride, dst_stride, r, eps,
                      border, stream);
    return run_jobs(&j, 1);
}

// Copies up to four row blocks (the 2r halo rows of two planes from two neighbour ranks) from peer-mapped memory into
// the local strip buffers: blockIdx.y = region, grid-stride over its 16-byte (or 4-byte) elements.
struct GfHaloPullArgs {
    float* dst[4]; const float* src[4];
    int64_t dstride[4], sstride[4];
    int rows[4];
    int width, vec4;
};
#ifndef GF_CPU_EMU
__global__ void __launch_bounds__(256) gf_halo_pull_kernel(const GfHaloPullArgs g)
{
    const int rg = blockIdx.y;
    const int rows = g.rows[rg];
    if (rows <= 0) return;
    float* d = g.dst[rg];
    const float* s = g.src[rg];
    const int64_t ds = g.dstride[rg], ss = g.sstride[rg];
    if (g.vec4) {
        const int w4 = g.width >> 2;
        const int64_t n = (int64_t)rows * w4;
        if (n < (1ll << 31)) {
            // NVLink reads have ~3 us of latency: U independent 16-byte loads per thread before the first store keep
            // the whole region in flight (one load per thread and trip measured 409 GB/s on 16 MiB)
            constexpr int U = 8;
            const unsigned nt = gridDim.x * blockDim.x, n32 = (unsigned)n;
            for (unsigned i0 = blockIdx.x * blockDim.x + threadIdx.x; i0 < n32; i0 += U * nt) {
                float4 v[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const unsigned i = i0 + u * nt;
                    if (i < n32) { const unsigned y = i / (unsigned)w4, x = i - y * (unsigned)w4; v[u] = reinterpret_cast<const float4*>(s + y * ss)[x]; }
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const unsigned i = i0 + u * nt;
                    if (i < n32) { const unsigned y = i / (unsigned)w4, x = i - y * (unsigned)w4; reinterpret_cast<float4*>(d + y * ds)[x] = v[u]; }
                }
            }
            return;
        }
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
            const int y = (int)(i / w4), x = (int)(i - (int64_t)y * w4);
            reinterpret_cast<float4*>(d + y * ds)[x] = reinterpret_cast<const float4*>(s + y * ss)[x];
        }
    } else {
        const int64_t n = (int64_t)rows * g.width;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
            const int y = (int)(i / g.width), x = (int)(i - (int64_t)y * g.width);
            d[y * ds + x] = s[y * ss + x];
        }
    }
}
#endif

// ---- row strips with the halo exchange inside the call (SURVEY 8(b): gf_run_strips) ------------------------
#ifndef GF_CPU_EMU
namespace {
// one side stream + fork/join events per device for the interior bands of gf_run_strips; the lock covers the enqueue
struct StripSide {
    std::mutex mu;
    cudaStream_t s = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    bool init = false;
};
StripSide g_strip_side[64];
std::mutex g_strip_side_mu;
StripSide* strip_side()
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    StripSide* sd = &g_strip_side[dev];
    std::lock_guard<std::mutex> lock(g_strip_side_mu);
    if (!sd->init) {
        if (cudaStreamCreateWithFlags(&sd->s, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
        if (cudaEventCreateWithFlags(&sd->e0, cudaEventDisableTiming) != cudaSuccess) return nullptr;
        if (cudaEventCreateWithFlags(&sd->e1, cudaEventDisableTiming) != cudaSuccess) return nullptr;
        sd->init = true;
    }
    return sd;
}
}  // namespace
#endif
static void strip_halo_rows(int global_height, int y0, int rows, int r, int* top, int* bot)
{
    *top = y0 > 0 ? (2 * r < y0 ? 2 * r : y0) : 0;
    const int below = global_height - (y0 + rows);
    *bot = below > 0 ? (2 * r < below ? 2 * r : below) : 0;
}

int gf_strip_layout(int global_height, int y0, int rows, int r, int* top, int* bot)
{
    if (!top || !bot) return fail(GF_ERR_INVALID, "gf_strip_layout: null pointer");
    if (global_height <= 0 || y0 < 0 || rows <= 0 || y0 + rows > global_height || r < 0) return fail(GF_ERR_INVALID, "gf_strip_layout: rows outside the image");
    strip_halo_rows(global_height, y0, rows, r, top, bot);
    return GF_OK;
}

int gf_run_strips(float* guide_buf, float* src_buf, float* dst, int width, int global_height, int y0, int rows, int64_t guide_stride,
                  int64_t src_stride, int64_t dst_stride, int r, float eps, int border, const gf_strip_peer* up, const gf_strip_peer* down,
                  void* stream)
{
    if (!guide_buf || !src_buf || !dst) return fail(GF_ERR_INVALID, "gf_run_strips: null image pointer");
    if (width <= 0 || global_height <= 0 || y0 < 0 || rows <= 0 || y0 + rows > global_height || r < 0)
        return fail(GF_ERR_INVALID, "gf_run_strips: strip [%d,%d) outside the %d-row image", y0, y0 + rows, global_height);
    int top = 0, bot = 0;
    strip_halo_rows(global_height, y0, rows, r, &top, &bot);
    const int64_t gs = or_packed(guide_stride, width, 1), ss = or_packed(src_stride, width, 1);
    // every neighbour must be able to supply the halo from its OWN rows (checked identically on every rank:
    // the numbers come from the geometry, not from what a neighbour says about itself)
    if ((up && top > 0 && up->rows < top) || (down && bot > 0 && down->rows < bot))
        return fail(GF_ERR_INVALID, "gf_run_strips: a neighbour strip is shorter than the %d-row halo it must supply", 2 * r);
    // ONE small kernel pulls all four halo regions (2 planes x 2 neighbours) straight out of the peers' memory with
    // 16-byte loads over NVLink.  Measured at 8 GPUs (32768^2, r=16, 16 MiB of halos per rank): four cudaMemcpy2DAsync
    // cost 0.061 ms back to back on the stream and 0.063 ms on four side streams (copy-engine set-up and cross-stream
    // events, not bandwidth), the pull kernel 0.041 ms.
    GfHaloPullArgs pa;
    int nreg = 0;
    auto add = [&](float* dst_rows, int64_t dstride, const float* peer, int64_t pstride, int first_row, int n) {
        if (n <= 0) return;
        const int64_t ps = pstride > 0 ? pstride : width;
        pa.dst[nreg] = dst_rows; pa.src[nreg] = peer + (int64_t)first_row * ps; pa.dstride[nreg] = dstride; pa.sstride[nreg] = ps; pa.rows[nreg] = n;
        ++nreg;
    };
    if (up && top > 0) {           // the LAST `top` own rows of the strip above -> my first `top` rows
        if (!up->guide || !up->src) return fail(GF_ERR_INVALID, "gf_run_strips: null peer pointer (up)");
        const int first = up->top + up->rows - top;
        add(guide_buf, gs, up->guide, up->guide_stride, first, top);
        add(src_buf, ss, up->src, up->src_stride, first, top);
    }
    if (down && bot > 0) {         // the FIRST `bot` own rows of the strip below -> my last `bot` rows
        if (!down->guide || !down->src) return fail(GF_ERR_INVALID, "gf_run_strips: null peer pointer (down)");
        const int64_t off = (int64_t)(top + rows);
        add(guide_buf + off * gs, gs, down->guide, down->guide_stride, down->top, bot);
        add(src_buf + off * ss, ss, down->src, down->src_stride, down->top, bot);
    }
    auto pull = [&](void* on) -> int {
        if (nreg == 0) return GF_OK;
#ifndef GF_CPU_EMU
        for (int i = nreg; i < 4; ++i) { pa.dst[i] = nullptr; pa.src[i] = nullptr; pa.dstride[i] = pa.sstride[i] = 0; pa.rows[i] = 0; }
        pa.width = width;
        bool v4 = (width & 3) == 0;
        for (int i = 0; i < nreg; ++i)
            v4 = v4 && !((uintptr_t)pa.dst[i] & 15) && !((uintptr_t)pa.src[i] & 15) && !(pa.dstride[i] & 3) && !(pa.sstride[i] & 3);
        pa.vec4 = v4 ? 1 : 0;
        int sms = 148, mj = 0, mn = 0;
        gf_rt_device_info(&sms, &mj, &mn);
        dim3 grid(sms, nreg), block(256);
        auto k = gf_halo_pull_kernel;
        GF_LAUNCH(k, grid, block, 0, on, pa);
        if (const char* le = gf_rt_launch_error()) return fail(GF_ERR_CUDA, "gf_run_strips: halo pull kernel: %s", le);
        g_launches++;
#else
        for (int i = 0; i < nreg; ++i)
            for (int y = 0; y < pa.rows[i]; ++y)
                std::memcpy(pa.dst[i] + y * pa.dstride[i], pa.src[i] + y * pa.sstride[i], (size_t)width * sizeof(float));
#endif
        return GF_OK;
    };
    Job j = strip_job(guide_buf, src_buf, dst, width, global_height, y0 - top, top + rows + bot, y0, rows, gs, ss, dst_stride, r, eps, border, stream);
    // OPTION GF_STRIP_OVERLAP=1 (off by default: measured slower): exchange off the critical path.  Only the first and the
    // last 2r OUTPUT rows of the strip read halo rows, so the strip is filtered in three jobs: rows [2r, rows-2r) on the
    // caller's stream at once; the pull and then the two 2r-row seam jobs on a side stream.
    // Measured (32768-column strips of 4096 rows, r = 16; profiles/r2_strip_overlap_8gpu.jsonl, r2_strip_phases.jsonl):
    //   8 GPUs   pull-then-launch 0.967 ms   this option 0.992 ms
    //   1 GPU, neighbours faked on the same GPU: main job alone 0.913 ms, both seam jobs alone 0.099 ms, main + seams
    //   together 0.947 ms, everything 0.956 ms, against 0.932 ms for pull-then-launch.
    // The seam jobs pay a 4r-row ramp for 2r output rows (4.5 % more row iterations), and the slots the main job leaves
    // idle (s8_r16 keeps 4 warps per SM: 171 column strips x 3 bands = 513 of 592) are not free: a fourth warp on an SM
    // slows the other three (profiles/r2_s8_residency.jsonl), so hiding a 0.02-0.04 ms pull costs 0.034 ms.  The other
    // split that was tried -- first and last BAND of every column strip after the pull, the middle bands before it --
    // lost by more (1.02-1.04 ms): with 3 bands per strip two of them wait for the pull.
    const int cut_top = (up && top > 0) ? 2 * r : 0, cut_bot = (down && bot > 0) ? 2 * r : 0;
    const int min_main = GF_KNOB("GF_STRIP_MIN_MAIN_ROWS", 16 * r + 64);
    if (nreg > 0 && GF_KNOB("GF_STRIP_OVERLAP", 0) && rows - cut_top - cut_bot >= min_main && check_common(j) == GF_OK &&
        !overlaps(j.dst, j.out_rows, j.guide, j.buf_rows, 1) && !overlaps(j.dst, j.out_rows, j.src, j.buf_rows, 1)) {
        const int64_t dstr = or_packed(dst_stride, width, 1);
        void* side = stream;
#ifndef GF_CPU_EMU
        StripSide* sd = strip_side();
        if (!sd) return fail(GF_ERR_CUDA, "gf_run_strips: side stream");
        std::lock_guard<std::mutex> lock(sd->mu);
        side = sd->s;
        if (cudaEventRecord(sd->e0, (cudaStream_t)stream) != cudaSuccess || cudaStreamWaitEvent(sd->s, sd->e0, 0) != cudaSuccess)
            return fail(GF_ERR_CUDA, "gf_run_strips: fork");
#endif
        auto part = [&](int first, int n, void* on) -> int {       // output rows [first, first + n) of the strip
            if (n <= 0) return GF_OK;
            Job p = j;
            p.out_y0 = y0 + first; p.out_rows = n; p.stream = on;
            p.dst.ptr = dst + (int64_t)first * dstr;
            return run_jobs(&p, 1);
        };
#ifdef GF_STRIP_DEBUG   // timing builds only (bench_tools/strip_phases.py): parts can be left out, the pixels are then WRONG
        const int skip = GF_KNOB("GF_STRIP_DEBUG_SKIP", 0);      // 1 no main job, 2 no pull, 4 no seam jobs
#else
        const int skip = 0;
#endif
        int rc = (skip & 1) ? GF_OK : part(cut_top, rows - cut_top - cut_bot, stream);
        if (rc == GF_OK && !(skip & 2)) rc = pull(side);
        if (rc == GF_OK && !(skip & 4)) rc = part(0, cut_top, side);
        if (rc == GF_OK && !(skip & 4)) rc = part(rows - cut_bot, cut_bot, side);
#ifndef GF_CPU_EMU
        // join even after an error: the caller's stream must not run ahead of what was already queued on the side stream
        if (cudaEventRecord(sd->e1, sd->s) != cudaSuccess || cudaStreamWaitEvent((cudaStream_t)stream, sd->e1, 0) != cudaSuccess)
            return rc ? rc : fail(GF_ERR_CUDA, "gf_run_strips: join");
#endif
        return rc;
    }
    if (int rc = pull(stream)) return rc;
    return run_jobs(&j, 1);
}

// device allocations that can be shared with the other ranks of a node (CUDA IPC needs allocation base pointers)
int gf_device_alloc(void** ptr, size_t bytes)
{
    if (!ptr) return fail(GF_ERR_INVALID, "null pointer");
#ifdef GF_CPU_EMU
    *ptr = std::aligned_alloc(256, (bytes + 255) / 256 * 256);
    return *ptr ? GF_OK : fail(GF_ERR_NOMEM, "malloc");
#else
    cudaError_t e = cudaMalloc(ptr, bytes);
    return e == cudaSuccess ? GF_OK : fail(GF_ERR_NOMEM, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
#endif
}

int gf_device_free(void* ptr)
{
#ifdef GF_CPU_EMU
    std::free(ptr);
    return GF_OK;
#else
    cudaError_t e = cudaFree(ptr);
    return e == cudaSuccess ? GF_OK : fail(GF_ERR_CUDA, "cudaFree: %s", cudaGetErrorString(e));
#endif
}

int gf_ipc_export(const void* ptr, void* handle64)
{
    if (!ptr || !handle64) return fail(GF_ERR_INVALID, "null pointer");
#ifdef GF_CPU_EMU
    return fail(GF_ERR_UNSUPPORTED, "no IPC in the emulator build");
#else
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, const_cast<void*>(ptr));
    if (e != cudaSuccess) return fail(GF_ERR_CUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e));
    std::memcpy(handle64, &h, 64);
    return GF_OK;
#endif
}

int gf_ipc_open(const void* handle64, void** ptr)
{
    if (!ptr || !handle64) return fail(GF_ERR_INVALID, "null pointer");
#ifdef GF_CPU_EMU
    return fail(GF_ERR_UNSUPPORTED, "no IPC in the emulator build");
#else
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle64, 64);
    cudaError_t e = cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess);
    return e == cudaSuccess ? GF_OK : fail(GF_ERR_CUDA, "cudaIpcOpenMemHandle: %s", cudaGetErrorString(e));
#endif
}

int gf_ipc_close(void* ptr)
{
#ifdef GF_CPU_EMU
    return GF_OK;
#else
    cudaError_t e = cudaIpcCloseMemHandle(ptr);
    return e == cudaSuccess ? GF_OK : fail(GF_ERR_CUDA, "cudaIpcCloseMemHandle: %s", cudaGetErrorString(e));
#endif
}

int gf_window_sums_u8(const unsigned char* guide, const unsigned char* src, long long* sum_i, long long* sum_p, long long* sum_ip,
                      long long* sum_ii, int width, int height, int64_t guide_stride, int64_t src_stride, int r, int border, void* stream)
{
    if (!guide || !src || !sum_i || !sum_p || !sum_ip || !sum_ii) return fail(GF_ERR_INVALID, "gf_window_sums_u8: null pointer");
    if (width <= 0 || height <= 0 || r < 0) return fail(GF_ERR_INVALID, "gf_window_sums_u8: bad geometry %dx%d r=%d", width, height, r);
    if (border != GF_TRUNCATE && (r >= width || r >= height)) return fail(GF_ERR_UNSUPPORTED, "gf_window_sums_u8: r >= image size with a reflecting border");
    const int64_t gs = guide_stride > 0 ? guide_stride : width, ss = src_stride > 0 ? src_stride : width;
    void* P = nullptr;
    if (const char* e = gf_rt_alloc_async(&P, (size_t)width * height * 8, stream)) return fail(GF_ERR_NOMEM, "prefix scratch: %s", e);
    const char* e = scan_sums_u8(guide, gs, nullptr, 0, sum_i, width, (long long*)P, width, height, r, border, stream);
    if (!e) e = scan_sums_u8(src, ss, nullptr, 0, sum_p, width, (long long*)P, width, height, r, border, stream);
    if (!e) e = scan_sums_u8(guide, gs, src, ss, sum_ip, width, (long long*)P, width, height, r, border, stream);
    if (!e) e = scan_sums_u8(guide, gs, guide, gs, sum_ii, width, (long long*)P, width, height, r, border, stream);
    gf_rt_free_async(P, stream);
    if (e) return fail(GF_ERR_CUDA, "gf_window_sums_u8: %s", e);
    g_launches += 8;
    g_kernel = "scan_sums_u8";
    return GF_OK;
}

int gf_box_filter(const float* src, float* dst, int width, int height, int channels, int64_t src_stride, int64_t dst_stride,
                  int r, int border, void* stream)
{
    if (channels < 1 || channels > 4) return fail(GF_ERR_UNSUPPORTED, "gScanLongRow Do not support channel: %d", channels);
    Job j;
    j.width = width; j.height = height; j.buf_rows = height; j.out_rows = height;
    j.r = r; j.border = border; j.stream = stream;
    j.src = Plane{src, or_packed(src_stride, width, channels), 0, channels, 0};
    j.guide = j.src;
    j.dst = Plane{dst, or_packed(dst_stride, width, channels), 0, channels, 0};
    j.A = j.B = Plane{nullptr, 0, 0, 1, 0};
    // reuse the halo check with r/2 semantics: the box filter needs r rows, not 2r -- the full
    // image is always in the buffer here, so check_common cannot fail on coverage
    int rc = check_common(j);
    if (rc) return rc;
    void* tmp = nullptr;
    Job jj = j;
    const size_t row_bytes = (size_t)width * channels * sizeof(float);
    if (overlaps(j.dst, height, j.src, height, 1)) {   // in place, as guided_filter.cpp:59-60 does
        if (const char* e = gf_rt_alloc_async(&tmp, row_bytes * height, stream)) return fail(GF_ERR_NOMEM, "in-place temporary: %s", e);
        jj.dst.ptr = (const float*)tmp;
        jj.dst.stride = (int64_t)width * channels;
    }
    GenericCfg c;
    rc = plan_generic(jj, 2 * r, 2 * r, channels, 0, &c);
    if ((rc == GF_ERR_UNSUPPORTED || GF_KNOB("GF_SCAN", 0)) && channels == 1 && r >= 1 && (border == GF_TRUNCATE || (r < width && r < height))) {
        // any radius: row prefixes + column pass (gf_scan.cuh); the prefix scratch doubles as the in-place temporary
        void* P = nullptr;
        if (const char* e = gf_rt_alloc_async(&P, (size_t)width * height * 8, stream)) { if (tmp) gf_rt_free_async(tmp, stream); return fail(GF_ERR_NOMEM, "scan-path scratch: %s", e); }
        const char* e = scan_box(src, jj.src.stride, nullptr, 0, dst, or_packed(dst_stride, width, 1), (double*)P, width, height, r, border, stream);
        gf_rt_free_async(P, stream);
        if (tmp) gf_rt_free_async(tmp, stream);
        if (e) return fail(GF_ERR_CUDA, "scan box: %s", e);
        g_launches += 2;
        g_kernel = "scan_box";
        return GF_OK;
    }
    if (rc) { if (tmp) gf_rt_free_async(tmp, stream); return rc; }
    GfArgs a = mk_args(jj);
    a.wc = c.wc; a.hb = c.hb;
    const size_t smem = c.smem_bytes;
    dim3 grid(c.nstrips, c.nbands, 1), block(c.win);
    switch (channels) {
    case 1: { auto k = gf_box_kernel<1>; GF_LAUNCH(k, grid, block, smem, stream, a); break; }
    case 2: { auto k = gf_box_kernel<2>; GF_LAUNCH(k, grid, block, smem, stream, a); break; }
    case 3: { auto k = gf_box_kernel<3>; GF_LAUNCH(k, grid, block, smem, stream, a); break; }
    default: { auto k = gf_box_kernel<4>; GF_LAUNCH(k, grid, block, smem, stream, a); break; }
    }
    const char* e = gf_rt_launch_error();
    if (!e && tmp) e = gf_rt_copy2d_async(dst, j.dst.stride * sizeof(float), tmp, row_bytes, row_bytes, height, stream);
    if (tmp) gf_rt_free_async(tmp, stream);
    if (e) return fail(GF_ERR_CUDA, "gf_box_kernel: %s", e);
    g_launches++;
    g_kernel = "box";
    return GF_OK;
}

}  // extern "C"

// Fast guided filter (He & Sun 2015; gf_fgf.cuh): a and b solved on I and p subsampled s times with radius r/s by the
// library's own gray a/b job, mean_a and mean_b by the box kernel, the bilinear upsample fused into q = mean_a*I + mean_b.
// T = float: gf_fast_guided_gray; T = unsigned char: gf_fast_guided_gray_u8, in the integer domain (eps' = 255^2 eps, the
// low-res planes hold 0..255; gf_fgf.cuh).  Strides are in elements.
template <typename T>
static int fast_guided_gray(const T* guide, const T* src, T* dst, int width, int height, int64_t guide_stride,
                            int64_t src_stride, int64_t dst_stride, int r, float eps, int s, int border, void* stream,
                            const char* fn, const char* tag)
{
    constexpr bool u8 = sizeof(T) == 1;
    if (!guide || !src || !dst) return fail(GF_ERR_INVALID, "%s: null pointer", fn);
    if (width <= 0 || height <= 0) return fail(GF_ERR_INVALID, "%s: non-positive size %dx%d", fn, width, height);
    const int64_t gs = or_packed(guide_stride, width, 1), ss = or_packed(src_stride, width, 1), ds = or_packed(dst_stride, width, 1);
    if (gs < width || ss < width || ds < width) return fail(GF_ERR_INVALID, "%s: row stride smaller than a row", fn);
    if (u8 && s == 1)
        return fail(GF_ERR_INVALID, "%s: s = 1 is the exact filter, whose 8-bit entry is gf_guided_gray_u8", fn);
    if (s < 1 || s > GF_FGF_MAX_S) return fail(GF_ERR_INVALID, "%s: subsampling factor s = %d outside [%d, %d]", fn, s, u8 ? 2 : 1, GF_FGF_MAX_S);
    if (r < 0 || r % s != 0)
        return fail(GF_ERR_INVALID, "%s: r = %d must be a non-negative multiple of s = %d (the low-res radius is r/s)", fn, r, s);
    if (!(eps >= 0.f)) return fail(GF_ERR_INVALID, "%s: eps must be >= 0", fn);
    if (border < 0 || border > 2) return fail(GF_ERR_INVALID, "%s: unknown border mode %d", fn, border);
    // dst may BE an input (same pointer and stride): every full-resolution pass writes only the pixels it has just read.
    // Planes that share a row stride may interleave their rows (columns side by side) without sharing a pixel.
    auto partial = [&](const T* in, int64_t is) {
        if (in == dst && is == ds) return false;
        if (!(dst < in + (int64_t)(height - 1) * is + width && in < dst + (int64_t)(height - 1) * ds + width)) return false;
        if (is != ds) return true;
        const int64_t c = (((intptr_t)dst - (intptr_t)in) / (int64_t)sizeof(T) % is + is) % is;   // column offset
        return !(c >= width && c + width <= is);
    };
    if (partial(guide, gs) || partial(src, ss))
        return fail(GF_ERR_UNSUPPORTED, "%s: dst overlaps an input without being exactly that input (same pointer and stride)", fn);

    // the low-res a/b job, refused here if run_job would refuse it: the streaming kernels plan it, or the scan path takes it
    const int ws = div_up(width, s), hs = div_up(height, s), rl = r / s;
    const int64_t pitch = round_up(ws, 4);                   // 16-byte rows
    Job lo;
    lo.width = ws; lo.height = hs; lo.buf_rows = hs; lo.out_rows = hs;
    lo.r = rl; lo.eps = u8 ? eps * 65025.0f : eps; lo.border = border; lo.stream = stream;
    lo.guide = lo.src = lo.dst = lo.A = lo.B = Plane{nullptr, pitch, 0, 1, 0};
    {
        GenericCfg c;
        if (plan_generic(lo, 4 * rl, 4 * rl, GfGrayModel::NQ1 + GfGrayModel::NQ2, GfGrayModel::NQ2, &c) != GF_OK && !scan_ok(lo))
            return fail(GF_ERR_UNSUPPORTED, "%s: no kernel runs the %dx%d low-res job at radius r/s = %d with border %d "
                                            "(a reflecting border needs r/s below both low-res dimensions at this radius)", fn, ws, hs, rl, border);
    }
    if (s == 1) {                                            // the exact filter (float only: s = 1 is refused above for u8)
        Job j;
        j.width = width; j.height = height; j.buf_rows = height; j.out_rows = height;
        j.r = r; j.eps = eps; j.border = border; j.stream = stream;
        j.guide = Plane{reinterpret_cast<const float*>(guide), gs, 0, 1, 0};
        j.src = Plane{reinterpret_cast<const float*>(src), ss, 0, 1, 0};
        j.dst = Plane{reinterpret_cast<const float*>(dst), ds, 0, 1, 0};
        j.A = j.B = Plane{nullptr, 0, 0, 1, 0};
        const int rc = run_jobs(&j, 1);
        if (rc == GF_OK) { g_kernel_fgf = std::string(tag) + g_kernel; g_kernel = g_kernel_fgf.c_str(); }
        return rc;
    }

    const size_t plane = (size_t)pitch * hs;
    void* scratch = nullptr;
    if (const char* e = gf_rt_alloc_async(&scratch, 5 * plane * sizeof(float), stream))
        return fail(GF_ERR_NOMEM, "%s: low-res scratch (%zu bytes): %s", fn, 5 * plane * sizeof(float), e);
    float* Is = (float*)scratch;                             // I_s, then mean_a
    float* ps = Is + plane;                                  // p_s, then mean_b
    float* A = ps + plane, *B = A + plane, *Q = B + plane;   // a, b and the low-res q the a/b job also writes
    int rc = GF_OK;
    {
        GfFgfDownArgs<T> a;
        a.I = guide; a.p = src; a.Is = Is; a.ps = ps; a.si = gs; a.sp = ss; a.sl = pitch;
        a.width = width; a.height = height; a.ws = ws; a.hs = hs; a.s = s;
        dim3 grid(div_up(ws, GF_FGF_DOWN_THREADS), hs < 65535 ? hs : 65535), block(GF_FGF_DOWN_THREADS);
        auto k = gf_fgf_down_kernel<T>;
        GF_LAUNCH(k, grid, block, 0, stream, a);
        if (const char* e = gf_rt_launch_error()) rc = fail(GF_ERR_CUDA, "gf_fgf_down_kernel launch: %s", e);
        else g_launches++;
    }
    const char* lo_name = "none";
    if (rc == GF_OK) {
        lo.guide.ptr = Is; lo.src.ptr = ps; lo.dst.ptr = Q; lo.A.ptr = A; lo.B.ptr = B;
        rc = run_job(lo);
        lo_name = g_kernel;
    }
    // mean_a, mean_b: gf_box_kernel on CTAs of 128 columns and bands short enough for 16 CTAs per SM.  A CTA waits for
    // one row load per step, so its time is (hb + 2r) load latencies: gf_box_filter's own plan (one strip of up to 1024
    // columns, bands of at least 16 rows) measured 19-22 us a plane at 4K s = 4 and 46-58 us at 8K s = 4.  Radii that
    // leave fewer than 32 columns go through gf_box_filter.
    auto box = [&](const float* in, float* out) -> int {
        const int win = 128, wc = win - 2 * rl;
        if (wc < 32) return gf_box_filter(in, out, ws, hs, 1, pitch, pitch, rl, border, stream);
        Job jb = lo;
        jb.src = jb.guide = Plane{in, pitch, 0, 1, 0};
        jb.dst = Plane{out, pitch, 0, 1, 0};
        jb.A = jb.B = Plane{nullptr, 0, 0, 1, 0};
        GfArgs a = mk_args(jb);
        int sms = 148, mj = 0, mn = 0;
        gf_rt_device_info(&sms, &mj, &mn);
        const int nstrips = div_up(ws, wc);
        const int hb = div_up(hs, div_up(16 * sms, nstrips));
        a.wc = wc; a.hb = hb;
        dim3 grid(nstrips, div_up(hs, hb), 1), block(win);
        auto k = gf_box_kernel<1>;
        GF_LAUNCH(k, grid, block, (win + 32) * sizeof(float), stream, a);
        if (const char* e = gf_rt_launch_error()) return fail(GF_ERR_CUDA, "gf_box_kernel launch: %s", e);
        g_launches++;
        return GF_OK;
    };
    // I_s and p_s have been read by the a/b job (stream order): they take mean_a and mean_b
    if (rc == GF_OK) rc = box(A, Is);
    if (rc == GF_OK) rc = box(B, ps);
    if (rc == GF_OK) {
        GfFgfApplyArgs<T> a;
        a.I = guide; a.q = dst; a.ma = Is; a.mb = ps; a.si = gs; a.sq = ds; a.sl = pitch;
        a.width = width; a.height = height; a.ws = ws; a.hs = hs; a.s = s;
        const uintptr_t al = 4 * sizeof(T) - 1;             // 4 pixels per access: 16 bytes (float), 4 bytes (u8)
        const bool vec = width % 4 == 0 && gs % 4 == 0 && ds % 4 == 0 && !((uintptr_t)guide & al) && !((uintptr_t)dst & al);
        const int ty = div_up(height, GF_FGF_TY);
        dim3 grid(div_up(width, GF_FGF_TX), ty < 65535 ? ty : 65535), block(256);
        if (vec) { auto k = gf_fgf_up_apply_kernel<true, T>; GF_LAUNCH(k, grid, block, 0, stream, a); }
        else { auto k = gf_fgf_up_apply_kernel<false, T>; GF_LAUNCH(k, grid, block, 0, stream, a); }
        if (const char* e = gf_rt_launch_error()) rc = fail(GF_ERR_CUDA, "gf_fgf_up_apply_kernel launch: %s", e);
        else g_launches++;
    }
    gf_rt_free_async(scratch, stream);
    if (rc == GF_OK) { g_kernel_fgf = std::string(tag) + lo_name; g_kernel = g_kernel_fgf.c_str(); }
    return rc;
}

extern "C" {

int gf_fast_guided_gray(const float* guide, const float* src, float* dst, int width, int height, int64_t guide_stride,
                        int64_t src_stride, int64_t dst_stride, int r, float eps, int s, int border, void* stream)
{
    return fast_guided_gray(guide, src, dst, width, height, guide_stride, src_stride, dst_stride, r, eps, s, border, stream,
                            "gf_fast_guided_gray", "fgf/");
}

int gf_fast_guided_gray_u8(const unsigned char* guide, const unsigned char* src, unsigned char* dst, int width, int height,
                           int64_t guide_stride, int64_t src_stride, int64_t dst_stride, int r, float eps, int s, int border,
                           void* stream)
{
    return fast_guided_gray(guide, src, dst, width, height, guide_stride, src_stride, dst_stride, r, eps, s, border, stream,
                            "gf_fast_guided_gray_u8", "fgf_u8/");
}

static int pointwise(int op, const float* i0, const float* i1, const float* i2, const float* i3, float* out, int width,
                     int height, int cs, int cg, int64_t ss, int64_t sg, float eps, void* stream, const char* name)
{
    if (!i0 || !i1 || !out || (op != GF_PW_MUL && !i2) || (op == GF_PW_CALC_A && !i3)) return fail(GF_ERR_INVALID, "%s: null pointer", name);
    if (width <= 0 || height <= 0) return fail(GF_ERR_INVALID, "%s: non-positive size", name);
    if (cs < 1 || !(cg == cs || cg == 1)) return fail(GF_ERR_UNSUPPORTED, "%s Do not support channel: %d, %d", name, cs, cg);
    GfPwArgs a;
    a.in0 = i0; a.in1 = i1; a.in2 = i2; a.in3 = i3; a.out = out;
    a.width = width; a.height = height; a.cs = cs; a.cg = cg;
    a.ss = or_packed(ss, width, cs); a.sg = or_packed(sg, width, cg); a.eps = eps;
    dim3 block(256), grid(div_up(width, 256), height < 1024 ? height : 1024);
    switch (op) {
    case GF_PW_MUL: { auto k = gf_pointwise_kernel<GF_PW_MUL>; GF_LAUNCH(k, grid, block, 0, stream, a); break; }
    case GF_PW_CALC_A: { auto k = gf_pointwise_kernel<GF_PW_CALC_A>; GF_LAUNCH(k, grid, block, 0, stream, a); break; }
    case GF_PW_CALC_B: { auto k = gf_pointwise_kernel<GF_PW_CALC_B>; GF_LAUNCH(k, grid, block, 0, stream, a); break; }
    default: { auto k = gf_pointwise_kernel<GF_PW_LINEAR>; GF_LAUNCH(k, grid, block, 0, stream, a); break; }
    }
    if (const char* e = gf_rt_launch_error()) return fail(GF_ERR_CUDA, "%s: %s", name, e);
    g_launches++;
    g_kernel = "pointwise";
    return GF_OK;
}

int gf_multiply(const float* a, const float* b, float* c, int width, int height, int channels_a, int channels_b,
                int64_t stride_a, int64_t stride_b, void* stream)
{
    return pointwise(GF_PW_MUL, a, b, nullptr, nullptr, c, width, height, channels_a, channels_b, stride_a, stride_b, 0.f, stream, "gMultiply");
}

int gf_calc_a(float* a, const float* pm, const float* im, const float* ipm, const float* iim, int width, int height,
              int channels_s, int channels_g, int64_t stride_s, int64_t stride_g, float eps, void* stream)
{
    return pointwise(GF_PW_CALC_A, pm, im, ipm, iim, a, width, height, channels_s, channels_g, stride_s, stride_g, eps, stream, "gCalcA");
}

int gf_calc_b(float* b, const float* a, const float* pm, const float* im, int width, int height, int channels_s,
              int channels_g, int64_t stride_s, int64_t stride_g, void* stream)
{
    return pointwise(GF_PW_CALC_B, a, im, pm, nullptr, b, width, height, channels_s, channels_g, stride_s, stride_g, 0.f, stream, "gCalcB");
}

int gf_linear_transform(const float* src, float* dst, const float* a, const float* b, int width, int height, int channels_d,
                        int channels_s, int64_t stride_d, int64_t stride_s, void* stream)
{
    return pointwise(GF_PW_LINEAR, src, a, b, nullptr, dst, width, height, channels_d, channels_s, stride_d, stride_s, 0.f, stream, "gLinearTransform");
}

}  // extern "C"

#include "gf_host.inl"
