/*
 * gf_b200.h -- C ABI of libgf_b200.so, the B200 (sm_100a) guided-filter library.
 *
 * This is the drop-in boundary for the GuidedFilter hot path of MrAoTian/CudaImageProcessing.
 * Each entry point names the reference interface it replaces (paths relative to the
 * reference repo).  Plain pointers and sizes only; no C++ or torch types.  The C++ shims
 * include/guided_filter.h and include/guided_filter_d.h keep the reference's own signatures
 * and forward here.
 *
 * Conventions (same as the reference, SURVEY 8(b)):
 *   - every image pointer is a DEVICE pointer owned by the caller unless the function name
 *     ends in _host;
 *   - layout is row-major, channel-interleaved (HWC) float32; strides are ROW strides in
 *     floats (`stride = pitch / sizeof(float)`, GuidedFilter/main.cpp:226);
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls are
 *     asynchronous on that stream, like the reference's hGuidedFilter; gf_run and the
 *     element-wise launchers do not add the reference's cudaDeviceSynchronize().
 *   - every function returns a gf_status; gf_last_error() gives the message (thread-local).
 *     The reference prints and exit(-1)s (cuda_utils.h:12-31) or silently returns
 *     (guided_filter_d.cu:893,1090); this library never does either.
 *   - there is no CPU fallback: without a CUDA device every compute call returns
 *     GF_ERR_CUDA.
 */
#ifndef GF_B200_H
#define GF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum gf_status {
    GF_OK = 0,
    GF_ERR_INVALID = 1,     /* bad argument (null pointer, non-positive size, stride < row) */
    GF_ERR_UNSUPPORTED = 2, /* channel combination or radius this build cannot run */
    GF_ERR_CUDA = 3,        /* CUDA runtime error (message holds cudaGetErrorString) */
    GF_ERR_NOMEM = 4
} gf_status;

typedef enum gf_border {
    /* gfedcb|abcdefgh|gfedcba, divisor (2r+1)^2: hGuidedFilter (guided_filter_d.cu:415-418,
       1051-1052) and the cv::blur composition (main.cpp:236-252). */
    GF_BORDER_REFLECT101 = 0,
    /* window clipped to the image, divided by the true pixel count: GuidedFilter::run /
       hBoxFilter (guided_filter_d.cu:251-262). */
    GF_BORDER_TRUNCATE = 1,
    /* fedcba|abcdefgh|hgfedcb: cv::ximgproc::guidedFilter (main.cpp:234). */
    GF_BORDER_REFLECT = 2
} gf_border;

typedef struct gf_filter* gf_handle;

const char* gf_last_error(void);
int gf_version(void);
/* SM count and compute capability of the current device. */
int gf_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- class GuidedFilter (GuidedFilter/guided_filter.h:5-55) ------------------------------- */

/* GuidedFilter::init (guided_filter.cpp:18-25).  Channel pairs (guide, src): (1,1), (3,3)
   filtered per channel, (1,3) -- as the reference (guided_filter_d.cu:968-979) -- plus
   (3,1): colour guide with the 3x3 covariance inverse (He et al. 2013), which the reference
   names but refuses.  The fused kernels need no scratch planes, so nothing is allocated. */
int gf_create(gf_handle* out, int width, int height, int guide_channels, int src_channels);
/* GuidedFilter::run (guided_filter.cpp:28-66).  border = GF_BORDER_TRUNCATE reproduces the
   class.  Strides in floats; pass 0 for "tightly packed" (width*channels). */
int gf_run(gf_handle h, const float* guide, const float* src, float* dst, int r, float eps,
           int border, int64_t guide_stride, int64_t src_stride, int64_t dst_stride, void* stream);
/* ~GuidedFilter (guided_filter.cpp:12-15). */
int gf_destroy(gf_handle h);

/* ---- hGuidedFilter (GuidedFilter/guided_filter_d.h:21, guided_filter_d.cu:1047-1093) ------- */

/* Gray guide, gray source, ANY radius >= 0 (the reference is a silent no-op outside 1..7).
   A and B may be NULL; when given they receive the per-pixel coefficients a and b like the
   reference's d_A / d_B (main.cpp:278-279).  One fused kernel; a, b never touch HBM unless
   requested. */
int gf_guided_gray(const float* guide, const float* src, float* dst, float* A, float* B,
                   int width, int height, int64_t guide_stride, int64_t src_stride,
                   int64_t dst_stride, int64_t ab_stride, int r, float eps, int border,
                   void* stream);

/* Fast guided filter (He & Sun, "Fast Guided Filter", arXiv:1505.00996): gray guide, gray source, float32, any
   width, height, stride and alignment.  An approximation of gf_guided_gray whose full-resolution cost does not grow
   with the radius: with hs = ceil(height/s), ws = ceil(width/s),
     - I_s, p_s: the mean of the in-image pixels of every s x s block (only the last row and column of blocks can be
       partial);
     - mean_a, mean_b: the gray guided filter of gf_guided_gray on (I_s, p_s) at radius r/s, with eps and border, up to
       its box means of a and b;
     - q = up(mean_a) * I + up(mean_b), up = bilinear with half-pixel centres and replicated edges:
       u = clamp((x + 0.5)/s - 0.5, 0, ws - 1), and the same for y.
   s = 1 is gf_guided_gray.  dst may be exactly the guide or the source (same pointer and stride): in place without a
   temporary.  Strides in floats, 0 = tightly packed.  Low-res scratch comes from the library's stream-ordered pool.
   GF_ERR_INVALID: a null pointer, a non-positive size, a stride smaller than a row, s outside [1, 32], r < 0 or r not a
   multiple of s, eps < 0, an unknown border.  GF_ERR_UNSUPPORTED: dst overlapping an input without being exactly it,
   or a low-res job no kernel of gf_guided_gray runs (a reflecting border with a radius r/s that is not below both
   low-res dimensions and too large for the streaming kernels).  Every refusal comes before anything is launched.
   gf_last_kernel() gives "fgf/<kernel of the low-res job>". */
int gf_fast_guided_gray(const float* guide, const float* src, float* dst, int width, int height,
                        int64_t guide_stride, int64_t src_stride, int64_t dst_stride,
                        int r, float eps, int s, int border, void* stream);

/* The fast guided filter of gf_fast_guided_gray on 8-bit gray planes (CV_8UC1), with the conversions fused into its two
   full-resolution kernels: the input is x/255, the output saturate_cast<uchar>(cvRound(255 q)) (round half to even), eps
   on the [0,1] scale.  2 bytes of HBM traffic per pixel in each full-resolution kernel instead of 8, and no conversion
   passes around the call.  Any width, height, stride and base alignment; strides in ELEMENTS (= bytes), 0 = tightly
   packed.  dst may be exactly the guide or the source (same pointer and stride).  s in [2, 32] (s = 1 is the exact
   filter: gf_guided_gray_u8), r a multiple of s.  Refusals as gf_fast_guided_gray's, before anything is launched.
   gf_last_kernel() gives "fgf_u8/<kernel of the low-res job>". */
int gf_fast_guided_gray_u8(const unsigned char* guide, const unsigned char* src, unsigned char* dst, int width, int height,
                           int64_t guide_stride, int64_t src_stride, int64_t dst_stride, int r, float eps, int s, int border,
                           void* stream);

/* The fast guided filter with a colour guide: a 3-channel interleaved float32 guide (CV_32FC3) and a source and
   destination of src_channels = 1 or 3 interleaved channels, any width, height, stride and alignment.  An approximation
   of gf_guided_color whose full-resolution cost does not grow with the radius: with hs = ceil(height/s), ws =
   ceil(width/s),
     - I_s (3 channels), p_s (src_channels channels): the per-channel mean of the in-image pixels of every s x s block;
     - for every source channel c: a (3-vector) and b of the colour guided filter of gf_guided_color on (I_s, p_s[c]) at
       radius r/s, with eps and border, and mean_a (3 planes), mean_b their box means at radius r/s with that border;
     - q_c = sum_k up(mean_a_k) * I_k + up(mean_b), up the bilinear upsample of gf_fast_guided_gray.
   s = 1 is gf_guided_color, and the call runs it.  Four kernel launches for s >= 2 whatever src_channels is (the source
   channels are frames of each launch).  dst may be exactly the source, and with src_channels = 3 exactly the guide
   (same pointer and stride), so guide == src == dst filters an image in place without a temporary.  Strides in floats,
   0 = tightly packed (3 width for the guide, src_channels width for src and dst).  Low-res scratch comes from the
   library's stream-ordered pool.
   GF_ERR_INVALID: a null pointer, a non-positive size, a stride smaller than a row, s outside [1, 32], r < 0 or r not a
   multiple of s, eps < 0 or NaN, an unknown border.  GF_ERR_UNSUPPORTED: src_channels not 1 or 3; dst overlapping an
   input without being exactly the source or (src_channels = 3) the guide; s >= 2 with r/s > 48 (the low-res kernels run
   CTAs of 128 low-res columns, at least 32 of them outputs beside the 2 r/s halo columns); s = 1 with r > 248 and
   width + 4r > 1024 (the radius gf_guided_color's streaming kernel cannot hold).  Every refusal comes before anything is
   allocated or launched.  gf_last_kernel() gives "fgfc/color_ab" (the low-res a/b kernel), for s = 1 "fgfc/" followed
   by the kernel gf_guided_color ran. */
int gf_fast_guided_color(const float* guide3, const float* src, float* dst, int width, int height, int src_channels,
                         int64_t guide_stride, int64_t src_stride, int64_t dst_stride,
                         int r, float eps, int s, int border, void* stream);

/* Colour guide (3 interleaved channels), `src_channels` (1 or 3) source/destination channels.
   a = (Sigma + eps U)^-1 cov(I, p), b = mean(p) - a.mean(I), q = mean(a).I + mean(b). */
int gf_guided_color(const float* guide3, const float* src, float* dst, int width, int height,
                    int src_channels, int64_t guide_stride, int64_t src_stride,
                    int64_t dst_stride, int r, float eps, int border, void* stream);

/* `count` frames of identical geometry in one launch; frame k starts at base + k*frame_stride
   (in floats).  guide_channels in {1,3}; src_channels 1.  This is the batch-sharded unit of
   work (BASELINE config 3): each GPU gets a contiguous block of frames, no collective. */
int gf_guided_batch(const float* guide, const float* src, float* dst, int count, int width,
                    int height, int guide_channels, int64_t guide_stride, int64_t src_stride,
                    int64_t dst_stride, int64_t guide_frame_stride, int64_t src_frame_stride,
                    int64_t dst_frame_stride, int r, float eps, int border, void* stream);

/* Row strip of a taller image (BASELINE config 5).  The image has `global_height` rows; the
   guide/src buffers hold its rows [buf_y0, buf_y0 + buf_rows) (pointer = first of them); the
   call writes output rows [out_y0, out_y0 + out_rows) to dst (pointer = row out_y0).  Rows
   needed beyond the image are produced by the border rule; rows needed beyond a strip seam
   must be in the buffer, i.e. the caller has exchanged 2r halo rows with its neighbours
   (NCCL send/recv, see cudaimageprocessing_b200/dist.py).  GF_ERR_INVALID if the buffer does
   not cover [out_y0 - 2r, out_y0 + out_rows + 2r) after border mapping. */
int gf_guided_gray_strip(const float* guide, const float* src, float* dst, int width,
                         int global_height, int buf_y0, int buf_rows, int out_y0, int out_rows,
                         int64_t guide_stride, int64_t src_stride, int64_t dst_stride, int r,
                         float eps, int border, void* stream);

/* ---- the five path-A launchers (GuidedFilter/guided_filter_d.h:6-18) ----------------------- */

/* ---- row strips of ONE huge image over the GPUs of a node, halo exchange inside the call -----------------
   (BASELINE configs[4]; SURVEY 8(b) "gf_run_strips"; the reference is single-GPU, main.cpp:17, so there is no
   reference interface to cite -- this is the C-host form of what cudaimageprocessing_b200/dist.py does in Python.)

   Rank g owns image rows [y0, y0 + rows).  Its strip buffers (guide_buf, src_buf) hold
       `top` halo rows | the `rows` own rows | `bot` halo rows          (gf_strip_layout: top/bot = 2r, clipped
   at the image's real top and bottom, where the border rule applies instead), so buffer row 0 is image row y0 - top.
   `up` / `down` describe the strip buffers of the rank above / below AS SEEN FROM THIS DEVICE: device pointers to THEIR
   buffer row 0 (the same process with peer access enabled, or another process's gf_device_alloc'ed buffer opened with
   gf_ipc_open), their strides, their own `top` and `rows`.  The call PULLS the halo rows it needs straight out of the
   neighbours' own rows -- one small kernel on `stream` that reads the peers' memory with 16-byte loads over
   NVLink (no NCCL, no staging, no copy-engine set-up) -- and launches the strip kernel behind it on the same stream.
   up == NULL / down == NULL: that halo (if the layout has one) is already in the buffer, e.g. after an
   ncclSend/ncclRecv exchange done by the caller (dist.exchange_halos_inplace).
   Ordering across ranks is the caller's: the neighbours' own rows must be complete before the call and unchanged
   until `stream` has passed it (one barrier / IPC event on either side; bench.py).  GF_ERR_INVALID if a neighbour
   strip is shorter than the halo it must supply. */
typedef struct gf_strip_peer {
    const float* guide;
    const float* src;
    int64_t guide_stride, src_stride;      /* floats; 0 = width */
    int top;                               /* halo rows above the neighbour's own rows in ITS buffers */
    int rows;                              /* the neighbour's own rows */
} gf_strip_peer;
int gf_strip_layout(int global_height, int y0, int rows, int r, int* top, int* bot);
int gf_run_strips(float* guide_buf, float* src_buf, float* dst, int width, int global_height, int y0, int rows,
                  int64_t guide_stride, int64_t src_stride, int64_t dst_stride, int r, float eps, int border,
                  const gf_strip_peer* up, const gf_strip_peer* down, void* stream);
/* Device buffers that other ranks of the node can map: cudaMalloc'ed (IPC exports allocation bases only), the
   64-byte cudaIpcMemHandle_t of one, and mapping / unmapping a neighbour's. */
int gf_device_alloc(void** ptr, size_t bytes);
int gf_device_free(void* ptr);
int gf_ipc_export(const void* ptr, void* handle64);
int gf_ipc_open(const void* handle64, void** ptr);
int gf_ipc_close(void* ptr);

/* The four stage-1 window sums of UINT8 planes, EXACT (north_star: "bit-exact integral sums for uint8 input (64-bit
   accumulators where the image is large enough to overflow 32-bit)"): sum over the (2r+1)^2 window (border rule applied)
   of I, p, I*p and I*I as int64, width x height each, tightly packed.  Integer row prefixes + integer column sums: no
   rounding anywhere.  The fused uint8 filter (gf_guided_gray_u8) works in float32 and is checked against these. */
int gf_window_sums_u8(const unsigned char* guide, const unsigned char* src, long long* sum_i, long long* sum_p,
                      long long* sum_ip, long long* sum_ii, int width, int height, int64_t guide_stride,
                      int64_t src_stride, int r, int border, void* stream);

/* hBoxFilter (guided_filter_d.cu:868-924): box mean of a `channels`-interleaved image.  One
   streaming kernel with exact window sums; no integral image, so no `integral` scratch.
   In-place (src == dst) is allowed, as in the reference (guided_filter.cpp:59-60). */
int gf_box_filter(const float* src, float* dst, int width, int height, int channels,
                  int64_t src_stride, int64_t dst_stride, int r, int border, void* stream);
/* hMultiply (:927-954): c = a*b; b has channels_a channels or 1. */
int gf_multiply(const float* a, const float* b, float* c, int width, int height, int channels_a,
                int channels_b, int64_t stride_a, int64_t stride_b, void* stream);
/* hCalcA (:957-984): a = (ipm - pm*im) / (iim - im*im + eps); guide planes have channels_s or 1. */
int gf_calc_a(float* a, const float* pm, const float* im, const float* ipm, const float* iim,
              int width, int height, int channels_s, int channels_g, int64_t stride_s,
              int64_t stride_g, float eps, void* stream);
/* hCalcB (:987-1014): b = pm - a*im  (the reference's CN1 variant is wrong, :371-372; this is
   the formula of the equal-channel variant for both). */
int gf_calc_b(float* b, const float* a, const float* pm, const float* im, int width, int height,
              int channels_s, int channels_g, int64_t stride_s, int64_t stride_g, void* stream);
/* hLinearTransform (:1017-1044): dst = src*a + b; src has channels_d channels or 1. */
int gf_linear_transform(const float* src, float* dst, const float* a, const float* b, int width,
                        int height, int channels_d, int channels_s, int64_t stride_d,
                        int64_t stride_s, void* stream);

/* ---- host-buffer entry (what a caller with cv::Mat data uses; the `e2e` number) ------------ */

/* Gray filter on HOST buffers (tightly packed rows): H2D of guide and src, the fused kernel,
   D2H of dst, pipelined in row bands over internal streams; returns when dst is complete.
   Pinned (gf_host_alloc) or registered (gf_host_register) buffers are copied by the DMA engines
   directly; pageable buffers are staged through pinned planes by a few copy threads of the library.  Replaces the cudaMemcpy2D + hGuidedFilter + cudaMemcpy2D sequence of
   main.cpp:229-279. */
int gf_guided_gray_host(const float* guide, const float* src, float* dst, int width, int height,
                        int r, float eps, int border);

/* Pinned host allocation helpers for callers that want the fast path of the call above.
   gf_host_register pins memory the caller already owns (the data of a cv::Mat that is reused frame after frame,
   main.cpp:229-230) in place: registering costs milliseconds once, afterwards the call above runs at the pinned
   speed instead of the pageable one (1.5 against 7 ms per 4K frame).  Unregister before the memory is freed. */
int gf_host_alloc(void** ptr, size_t bytes);
int gf_host_free(void* ptr);
int gf_host_register(void* ptr, size_t bytes);
int gf_host_unregister(void* ptr);

/* ---- uint8 in / uint8 out (SURVEY 8(f) rank 2) ------------------------------------------------
   The conversions the reference's demo does around the filter -- Mat::convertTo(CV_32F, 1/255) before
   (main.cpp:121-122,205-206) and convertTo(CV_8U, 255) with saturating round-half-even after
   (main.cpp:158,295-297) -- fused into the kernel's loads and stores: 3 bytes of HBM traffic per pixel
   instead of 12.  Strides in ELEMENTS (= bytes).  Served by the s8 kernel only: r in {1..8, 16},
   width >= 64, height >= 4r+2, rows 8-byte aligned; other arguments return GF_ERR_UNSUPPORTED. */
int gf_guided_gray_u8(const unsigned char* guide, const unsigned char* src, unsigned char* dst, int width, int height,
                      int64_t guide_stride, int64_t src_stride, int64_t dst_stride, int r, float eps, int border,
                      void* stream);

/* The gray guided filter of gf_guided_gray_u8 on every channel of an 8-bit 3-channel image (CV_8UC3 src and dst):
   guide_channels = 1 filters each source channel with the one gray guide (the class API's (1,3) mode,
   GuidedFilter::init(w, h, 1, 3)); guide_channels = 3 filters source channel c with guide channel c (the (3,3) mode).
   Channel c of dst is byte for byte what gf_guided_gray_u8 gives on the planes of channel c: the input is x/255, eps
   on the [0,1] scale, the output saturate_cast<uchar>(cvRound(255 q)); any border.  Strides in ELEMENTS (= bytes),
   0 = tightly packed (3 width, guide_channels width).  One launch of the s8 kernel, whose frames are the source
   channels; gf_last_kernel() gives "s8u8_g1c3_r<r>" or "s8u8_g3c3_r<r>".  Served by that kernel only: r in {1..8, 16},
   width >= 64, width and height >= 4r+2, every plane's base address and row stride 8-byte aligned, rows x stride
   < 2^31, for TRUNCATE width % 8 == 0 and width >= 256, dst overlapping neither input; other arguments return
   GF_ERR_UNSUPPORTED (guide_channels not 1 or 3 too), before anything is launched. */
int gf_guided_per_channel_u8(const unsigned char* guide, const unsigned char* src, unsigned char* dst, int width, int height,
                             int guide_channels, int64_t guide_stride, int64_t src_stride, int64_t dst_stride,
                             int r, float eps, int border, void* stream);

/* The colour-guide filter of gf_guided_color on 8-bit planes (a CV_8UC3 guide; a CV_8UC1 or CV_8UC3 source and
   destination of `src_channels` interleaved channels), with the same fused conversions: the input is x/255, the output
   saturate_cast<uchar>(cvRound(255 q)), eps on the [0,1] scale.  Strides in ELEMENTS (= bytes), 0 = tightly packed.
   One launch of the c4 kernel for 1 or 3 source channels.  Served by that kernel only: r in {4, 8, 12, 16},
   width % 4 == 0, width >= 128, height >= 4r+2, rows x stride < 2^31, every plane's base address and row stride
   4-byte aligned, dst overlapping neither input; other arguments return GF_ERR_UNSUPPORTED. */
int gf_guided_color_u8(const unsigned char* guide3, const unsigned char* src, unsigned char* dst, int width, int height,
                       int src_channels, int64_t guide_stride, int64_t src_stride, int64_t dst_stride,
                       int r, float eps, int border, void* stream);

/* ---- Integral/ module (SURVEY 8(f) rank 1): summed-area table of a uint8 image ----------------
   Replace hIntegral / hAligned4Integral (Integral/integral_d.h:5-8, integral_d.cu:863-930):
   integral[y*dst_stride + x] = sum of src over rows <= y and columns <= x (inclusive, W x H).
   Strides in ELEMENTS.  The int32 form wraps modulo 2^32 exactly like the reference's int
   accumulators; the int64 form never overflows (use it above 8.4 Mpix).  `scratch` (optional):
   at least ceil(height/16) * width elements -- the reference's w*h `buff` is always enough; used
   when the per-band / per-strip carries fit, else (and when NULL) they live in a stream-ordered
   temporary.  The padded form writes a dst_width x dst_height table
   (>= the source size, e.g. aligned to 4) of the zero-extended image. */
int gf_integral_u8_i32(const unsigned char* src, int32_t* integral, int32_t* scratch, int width, int height,
                       int64_t src_stride, int64_t dst_stride, void* stream);
int gf_integral_u8_i64(const unsigned char* src, int64_t* integral, int64_t* scratch, int width, int height,
                       int64_t src_stride, int64_t dst_stride, void* stream);
int gf_integral_u8_i32_padded(const unsigned char* src, int32_t* integral, int src_width, int src_height,
                              int64_t src_stride, int dst_width, int dst_height, void* stream);

/* Separable Gaussian blur of a float32 gray image (SURVEY 8(f) rank 3; replaces the reference's
   GaussianFilter/gaussian.cu kernels gGaussNaive/Const/Share/Split/Optim, :25-306, as driven by
   gaussianComparasion, :409-660): taps = cv::getGaussianKernel(2*radius+1, sigma, CV_32F)
   (sigma <= 0: OpenCV's rule), border REFLECT101 (reflectBorder, GaussianFilter/gaussian.h),
   i.e. the result of cv::GaussianBlur(src, dst, Size(2r+1, 2r+1), sigma, sigma) to float32
   rounding.  DEVICE pointers, strides in elements (0 = width), radius 0..64, src != dst. */
int gf_gaussian_gray(const float* src, float* dst, int width, int height, int64_t src_stride, int64_t dst_stride,
                     int radius, double sigma, void* stream);

/* Which kernel family the last gf_guided_* call on this thread used ("fast_r8", "generic"...)
   and how many kernels it launched; for tests and bench.py's gpu_launches. */
const char* gf_last_kernel(void);
int64_t gf_launch_count(void);

/* Developer / test options of the launch paths (kernel family, band height, residency: names in
   DESIGN.md section 8, e.g. "GF_DISABLE_WS", "GF_WS_K", "GF_S8_HB").  No option changes results.
   The library never reads the environment on a launch: an option is seeded ONCE, when a launch
   path first looks at it, from the environment variable of the same name, and this call overrides
   it from then on.  value >= 0 sets it, value < 0 restores the built-in default. */
int gf_set_option(const char* name, int value);

#ifdef __cplusplus
}
#endif
#endif /* GF_B200_H */
