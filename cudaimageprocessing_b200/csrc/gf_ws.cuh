// gf_ws.cuh -- round-2 headline kernel: WARP-SPECIALISED fused guided filter (gray, float32).
//
// Why (VERDICT r1, profiles/r1_s8_full_summary.txt): gf_s8 issues 28 M warp-instructions per 4K frame
// (485 per 224 output px), a third of them in band ramps, at 255 registers and 1.7 warps per scheduler.
// This kernel is built around the instruction count instead:
//   * a lane owns K ADJACENT columns (K = 8, 12 or 16): the cross-lane traffic of a (2R+1)-window sum is
//     2R/K shuffles per pixel and quantity (K = 12, R = 8: 1.33 instead of 2), the strip halo shrinks from
//     12.5 % to 8.3 % of the loaded columns, and there are fewer, taller strips;
//   * the window sums run on QUANTITY pairs -- (S_I, S_p), (S_Ip, S_II), (a, b) -- as packed f32x2
//     prefix/suffix chains: 2(K-1) + ~1.3 K FADD2 per pair and K pixels (the 114 scalar FADDs of gf_s8's
//     trees are gone), 4 independent chains per producer warp = exactly the FADD2 pipe's latency;
//   * the two stages are split over WARPS (one CTA per SM, NS streams, 2 NS warps): the producer warp of a
//     stream owns the four stage-1 column sums (vertical running sums, window sums, a/b solve) and writes
//     raw (a, b N) rows into a shared-memory ring; the consumer warp owns stage 2 VERTICAL-FIRST (running
//     column sums of a, b from the ring, ONE window pair per OUTPUT row, q = mean_a I + mean_b, store).
//     Each scheduler hosts one producer and one consumer, so one warp's shuffle/LDS bursts overlap the
//     other's arithmetic, and neither carries the other's registers;
//   * the NS streams of a CTA walk adjacent sub-bands of ONE strip in ALTERNATING directions and share
//     their a/b rows across the sub-band boundaries through the rings (a stream's first R rows pre-populate
//     its partner's window, its last R rows complete its other neighbour's), so a band pays the 4R-row ramp
//     once per CTA (at its two outer ends) instead of once per warp: only the 2R cheap vertical warm-up
//     rows (loads + adds) remain per stream.
// Hand-off: monotonic row counters in shared memory (st.release / ld.acquire at CTA scope, nanosleep
// back-off); the ring has 2R+2 rows, a producer waits only when its consumer is a full row behind.
// Numerics: additions only inside a window (prefix + suffix, no subtraction of prefixes); the vertical
// sums slide (add the entering row, subtract the leaving one) over at most GF_WS_MAX_SUB rows per stream
// before the band is cut (random-walk drift ~1e-7 per 100 rows on [0,1] data; measured in the tests).
// Borders: the vertical rule is a row map (TRUNCATE: zero rows + counts); horizontally, lanes that lie
// (partly) outside the image gather their columns through a per-lane column map (the first and last
// strip only), so mirrored inputs give mirrored a, b and nothing else changes.
#pragma once
#include "gf_s8.cuh"

#ifndef GF_WS_NEWTON
#define GF_WS_NEWTON 1       // one Newton step after MUFU.RCP in the a/b solve
#endif
#ifndef GF_WS_SPLIT
#define GF_WS_SPLIT 0        // prefix / suffix chains of the window sums in two halves: measured 1-2 % SLOWER (r2_ws_variants.jsonl)
#endif
#ifndef GF_WS_PF
#define GF_WS_PF 0           // rows ahead for an L2 prefetch hint of the entering row; measured 4-6 % SLOWER at 4K/8K
                             // (profiles/r2_ws_variants.jsonl), so off
#endif
#ifndef GF_WS_NORM2
#define GF_WS_NORM2 1        // two-term reciprocal of the pixel count (see GfNorm)
#endif

struct GfWsArgs {
    const float* guide; const float* src; float* dst; float* A; float* B;
    int64_t gs, ss, ds, abs_;        // row strides (floats)
    int64_t gfs, sfs, dfs, abfs;     // frame strides
    int width, height, buf_y0, buf_rows, out_y0, out_rows, border;
    int nstrips, nbands, hb, count;
    int nbands_e, hb_e;              // band count / height of the first and last strip (0: same as the others)
    float eps;
    int pen;                         // rows the two outer streams of a CTA get fewer than the inner ones (gf_ws_plan)
    long long* dbg;                  // -DGF_WS_TIMING experiment builds only: per-warp (start, end) clocks; nullptr in the product
};

template <int R, int K, int NS>
struct GfWsGeom {
    static_assert(K % 4 == 0 && K >= 4 && K <= 16, "K columns per lane: 4, 8, 12 or 16");
    static_assert(2 * R + 1 > K, "window must be wider than a lane");
    static constexpr int KW = 2 * R + 1;
    static constexpr int HALO = (2 * R + 3) / 4 * 4;     // columns of halo per side (both stages), 16-byte granular
    static constexpr int WIN = 32 * K;                   // columns a stream loads
    static constexpr int WOUT = WIN - 2 * HALO;          // columns it writes
    static constexpr int RING = 2 * R + 2;               // a/b rows per stream
    static constexpr int ROW_F4 = (K / 2) * 32;          // float4 per ring row: [pair of columns][lane] = (a0, b0, a1, b1)
    static constexpr size_t ring_bytes = (size_t)RING * ROW_F4 * 16;
    static constexpr int NBAR = 2 * RING + 1;            // mbarriers per stream: row ready + products ready per ring slot, "stream finished"
    static constexpr size_t ctrl_bytes = 64 + (size_t)NS * NBAR * 8;      // 2 NS row counters + the mbarriers
    static constexpr size_t smem_bytes = (size_t)NS * ring_bytes + (ctrl_bytes + 127) / 128 * 128;
    static constexpr int MIN_SUB = R + 1;                // shortest sub-band whose neighbours can share rows with it
};

// ---- hand-off primitives --------------------------------------------------------------------------
// GF_WS_SYNC: how a consumer learns that an a/b row is in the ring.
//   2 (default)  one mbarrier per ring slot (phase = use count of the slot): the producer's lane 0 arrives
//                (release at CTA scope, no MEMBAR), consumers sleep in mbarrier.try_wait (hardware wake-up);
//   1            monotonic row counter, st.release / ld.acquire, consumers spin;
//   0            same counter with a nanosleep back-off (first version: the sleep quantum turned out to be
//                longer than a row, profiles/r2_ws_sync_variants.jsonl).
// The consumed-rows counter (consumer -> producer) is a counter in every variant: a producer reads it once
// per row and practically never has to wait (the consumer releases a ring row as soon as it is in registers).
#ifndef GF_WS_SYNC
#define GF_WS_SYNC 2
#endif
#ifdef GF_CPU_EMU
static inline int gf_ws_ld_acq(const volatile int* p) { return *p; }
static inline void gf_ws_st_rel(volatile int* p, int v) { *p = v; }
static inline void gf_ws_pause() { emu::yield_to_scheduler(emu::RUNNABLE); }
// emulated mbarrier: the word counts completed phases
static inline void gf_ws_bar_init(unsigned long long* b) { *b = 0; }
static inline void gf_ws_bar_arrive(unsigned long long* b) { *(volatile unsigned long long*)b = *b + 1; }
static inline void gf_ws_bar_wait(const unsigned long long* b, int phase)
{
    while (*(const volatile unsigned long long*)b <= (unsigned long long)phase) gf_ws_pause();
}
#else
__device__ __forceinline__ int gf_ws_ld_acq(const volatile int* p)
{
    int v;
    asm volatile("ld.acquire.cta.shared.s32 %0, [%1];" : "=r"(v) : "r"((unsigned)__cvta_generic_to_shared(const_cast<const int*>(p))) : "memory");
    return v;
}
__device__ __forceinline__ void gf_ws_st_rel(volatile int* p, int v)
{
    asm volatile("st.release.cta.shared.s32 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(const_cast<int*>(p))), "r"(v) : "memory");
}
__device__ __forceinline__ void gf_ws_pause()
{
#if GF_WS_SYNC == 0
    __nanosleep(32);
#endif
}
__device__ __forceinline__ void gf_ws_bar_init(unsigned long long* b)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"((unsigned)__cvta_generic_to_shared(b)) : "memory");
}
__device__ __forceinline__ void gf_ws_bar_arrive(unsigned long long* b)
{
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"((unsigned)__cvta_generic_to_shared(b)) : "memory");
}
__device__ __forceinline__ void gf_ws_bar_wait(const unsigned long long* b, int phase)
{
    const unsigned addr = (unsigned)__cvta_generic_to_shared(const_cast<unsigned long long*>(b));
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "GF_WS_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@!p bra GF_WS_WAIT_%=;\n\t}"
        ::"r"(addr), "r"((unsigned)(phase & 1)) : "memory");
}
#endif
__device__ __forceinline__ void gf_ws_wait(const volatile int* ctr, int need)
{
    while (gf_ws_ld_acq(ctr) < need) gf_ws_pause();
}
__device__ __forceinline__ void gf_ws_publish(volatile int* ctr, int val, int lane)
{
    __syncwarp();                       // every lane's ring accesses are ordered before lane 0's release
    if (lane == 0) gf_ws_st_rel(ctr, val);
}
// row `idx` (count from the stream's first own row) of a stream is in its ring
template <int RING>
__device__ __forceinline__ void gf_ws_row_ready(volatile int* prod, unsigned long long* bars, int idx, int slot, int lane)
{
#if GF_WS_SYNC == 2
    __syncwarp();
    if (lane == 0) gf_ws_bar_arrive(bars + slot);
#else
    gf_ws_publish(prod, idx + 1, lane);
#endif
}
// `last_rows`: the row is one of the LAST rows of another stream (the neighbour across a shared end).  A slot
// barrier only tells phase p from p-1 (one parity bit): a consumer that arrives while that producer is still more
// than a ring behind would take the completion of phase p-1 for phase p.  Those rows wait for the producer's
// "stream finished" barrier instead (its last row is the first one needed anyway).
template <int RING>
__device__ __forceinline__ void gf_ws_row_wait(const volatile int* prod, const unsigned long long* bars, int idx, bool last_rows)
{
#if GF_WS_SYNC == 2
    if (last_rows) gf_ws_bar_wait(bars + 2 * RING, 0);
    else gf_ws_bar_wait(bars + idx % RING, idx / RING);
#else
    gf_ws_wait(prod, idx + 1);
#endif
}

// ---- (2R+1)-window sums of K adjacent columns per lane, on packed quantity pairs --------------------
// Column j of lane l covers [j-R, j+R] in lane-local coordinates: the part left of column 0 is a SUFFIX of
// lane l-dl (plus the totals of the lanes in between when R > K), the part right of column K-1 a PREFIX of
// lane l+dr, the rest a local prefix / suffix / total.  Additions only.  Complete for every column at least
// R away from the warp's first and last column.
__device__ __forceinline__ float2 gf_ws_shfl_up(float2 v, int d)
{
    return make_float2(__shfl_up_sync(0xffffffffu, v.x, d), __shfl_up_sync(0xffffffffu, v.y, d));
}
__device__ __forceinline__ float2 gf_ws_shfl_down(float2 v, int d)
{
    return make_float2(__shfl_down_sync(0xffffffffu, v.x, d), __shfl_down_sync(0xffffffffu, v.y, d));
}
__host__ __device__ constexpr int gf_ws_fdiv(int a, int k) { return a >= 0 ? a / k : -((-a + k - 1) / k); }

template <int K, int R>
__device__ __forceinline__ void gf_ws_window(const float2 (&v)[K], float2 (&w)[K])
{
    float2 P[K], S[K];
#if GF_WS_SPLIT
    // two half-length chains per direction instead of one (dependency depth K/2 + 1 instead of K - 1; K/2 more
    // additions): a lone producer warp per scheduler otherwise waits on FADD2 latency at every step
    constexpr int HF = K / 2;
    P[0] = v[0];
    P[HF] = v[HF];
#pragma unroll
    for (int j = 1; j < HF; ++j) { P[j] = gf_add2(P[j - 1], v[j]); P[HF + j] = gf_add2(P[HF + j - 1], v[HF + j]); }
#pragma unroll
    for (int j = HF; j < K; ++j) P[j] = gf_add2(P[j], P[HF - 1]);
    S[K - 1] = v[K - 1];
    S[HF - 1] = v[HF - 1];
#pragma unroll
    for (int j = 1; j < HF; ++j) { S[K - 1 - j] = gf_add2(S[K - j], v[K - 1 - j]); S[HF - 1 - j] = gf_add2(S[HF - j], v[HF - 1 - j]); }
#pragma unroll
    for (int j = 0; j < HF; ++j) S[j] = gf_add2(S[j], S[HF]);
#else
    P[0] = v[0];
#pragma unroll
    for (int j = 1; j < K; ++j) P[j] = gf_add2(P[j - 1], v[j]);
    S[K - 1] = v[K - 1];
#pragma unroll
    for (int j = K - 2; j >= 0; --j) S[j] = gf_add2(S[j + 1], v[j]);
#endif
    constexpr int CM = (R + K - 1) / K;      // farthest lane a window reaches
    // cumulative totals of the c nearest lanes on either side (only when R > K)
    float2 TL[CM + 1], TR[CM + 1];
    TL[0] = TR[0] = make_float2(0.f, 0.f);
#pragma unroll
    for (int c = 1; c < CM; ++c) {
        TL[c] = gf_add2(TL[c - 1], gf_ws_shfl_up(P[K - 1], c));
        TR[c] = gf_add2(TR[c - 1], gf_ws_shfl_down(P[K - 1], c));
    }
#pragma unroll
    for (int j = 0; j < K; ++j) {
        const int a = j - R, b = j + R;
        const int dl = gf_ws_fdiv(a, K), al = a - dl * K;
        const int dr = gf_ws_fdiv(b, K), bl = b - dr * K;
        float2 acc = (dl < 0 && dr > 0) ? P[K - 1] : (dl < 0 ? P[b < K ? b : K - 1] : S[a > 0 ? a : 0]);
        if (dl < 0) {
            acc = gf_add2(acc, gf_ws_shfl_up(S[al], -dl));
            if (-dl - 1 > 0) acc = gf_add2(acc, TL[-dl - 1]);
        }
        if (dr > 0) {
            acc = gf_add2(acc, gf_ws_shfl_down(P[bl], dr));
            if (dr - 1 > 0) acc = gf_add2(acc, TR[dr - 1]);
        }
        w[j] = acc;
    }
}

// ---- image edges of the first / last strip: mirror the COLUMN SUMS, not the loads ----------------------
// A column outside the image carries the sums of the in-image column it mirrors (REFLECT101: u' = C - u in strip
// coordinates, REFLECT: the same with C shifted by one), so instead of gathering mirrored pixels for every loaded
// row the producer copies the four vertical sums across lanes once per row: for source register js the target
// register is (C - js) mod K and the source lane is q - lane, both compile-time per js.  K shuffles per
// component, only in the two edge strips.  TRUNCATE: the outside columns are simply zero.
template <int K, int C>
__device__ __forceinline__ void gf_ws_mirror(float2 (&v)[K], int lane, unsigned oob)
{
    float2 t[K];
#pragma unroll
    for (int js = 0; js < K; ++js) {
        const int j = ((C - js) % K + K) % K;            // target register fed by source register js
        const int q = (C - j - js) / K;                  // source lane = q - lane
        t[j] = make_float2(__shfl_sync(0xffffffffu, v[js].x, (q - lane) & 31), __shfl_sync(0xffffffffu, v[js].y, (q - lane) & 31));
    }
#pragma unroll
    for (int j = 0; j < K; ++j)
        if (oob >> j & 1) v[j] = t[j];
}

// ---- sub-band plan of one CTA ----------------------------------------------------------------------
// Stream k of n walks output rows ys, ys+d, .. (L of them).  Streams alternate direction (even: up, odd:
// down), so the boundary between streams 2p and 2p+1 is where both START and the boundary between 2p+1 and
// 2p+2 is where both END.  At a shared start the partner's first R a/b rows stand in for this stream's
// rows -1 .. -R; at a shared end the neighbour's last R rows for rows L .. L+R-1.  An outer boundary (the
// CTA's own band edge) is computed by the stream itself (R extra a/b rows).
struct GfWsStream {
    int ys, d, L;
    int m0, m1;        // own a/b rows [m0, m1) in stream coordinates (row m = image row ys + d m)
    int sp, ep;        // stream sharing the start / end boundary, -1 = outer
};
template <int NS>
struct GfWsPlan {
    int n;
    GfWsStream s[NS];
};

template <int R, int NS>
__host__ __device__ inline void gf_ws_plan(int y0, int y1, int pen, GfWsPlan<NS>& pl)
{
    const int H = y1 - y0;
    // balance: an outer boundary costs its stream R more producer rows, a shared END costs its consumer R more steps after
    // the producers have finished (measured with -DGF_WS_TIMING: ~0.6 producer rows each), so the first and the last stream
    // get `pen` ~ 3R/8 rows fewer than the inner ones; every stream of a shared plan needs at least R+1 rows
    int Ls[NS];
    int n = NS;
    for (; n > 1; --n) {
        const int base = (H + 2 * pen) / n, rem = H + 2 * pen - base * n;     // rem in [0, n): one extra row for the first rem streams
        bool ok = true;
        for (int k = 0; k < n; ++k) {
            Ls[k] = base + (k < rem ? 1 : 0) - ((k == 0) + (k == n - 1)) * pen;
            ok = ok && Ls[k] >= R + 1;
        }
        if (ok) break;
    }
    if (n == 1) Ls[0] = H;
    pl.n = n;
    int b = y0;
    for (int k = 0; k < NS; ++k) {
        GfWsStream& s = pl.s[k];
        if (k >= n) { s.ys = 0; s.d = 1; s.L = 0; s.m0 = s.m1 = 0; s.sp = s.ep = -1; continue; }
        const int lo = b, hi = b + Ls[k];
        b = hi;
        s.L = Ls[k];
        if (n == 1) { s.d = 1; s.ys = lo; s.sp = s.ep = -1; }
        else if ((k & 1) == 0) { s.d = -1; s.ys = hi - 1; s.sp = k + 1 < n ? k + 1 : -1; s.ep = k >= 1 ? k - 1 : -1; }
        else { s.d = 1; s.ys = lo; s.sp = k - 1; s.ep = k + 1 < n ? k + 1 : -1; }
        s.m0 = s.sp >= 0 ? 0 : -R;
        s.m1 = s.ep >= 0 ? s.L : s.L + R;
    }
}

// ---- stage 1: producer warp -------------------------------------------------------------------------
// EM: 0 the strip window lies inside the image, 1 it overhangs the left edge by exactly HALO columns, 2 the right
// edge by exactly HALO (the last strip is placed that way), 3 anything else: per-column map + gathered loads.
// ROLE: 0 one producer warp per stream; 1 / 2 the producer split over TWO warps (3 warps per scheduler instead of 2,
// each with half the dependent chain): warp 2 owns Y = (sum Ip, sum II), its window sums go into the ring slot of the
// row (the slot is free by then); warp 1 owns X = (sum I, sum p), picks the Y sums up from the slot, solves for a, b
// and overwrites the slot with them.
template <int R, int K, int NS, bool TRUNC, int EM, int ROLE>
__device__ __forceinline__ void gf_ws_stage1(const GfWsArgs& a, const GfWsPlan<NS>& pl, int k, int lane, int64_t f, int xl,
                                             int out_lo, int out_hi, float4* rings, volatile int* ctrl)
{
    using G = GfWsGeom<R, K, NS>;
    constexpr int RING = G::RING, KW = G::KW;
    const GfWsStream st = pl.s[k];
    float4* ring = rings + (size_t)k * RING * G::ROW_F4 + lane;
    const int x0 = xl + lane * K;
    constexpr bool EDGE = EM == 3;
    const bool vec = !EDGE || (x0 >= 0 && x0 + K <= a.width);
    int sx[EDGE ? K : 1];
    if (EDGE) {
#pragma unroll
        for (int j = 0; j < K; ++j) sx[j] = gf_map(x0 + j, a.width, a.border);
    }
    unsigned oob = 0, cmask = ~0u;            // EM 1, 2: columns outside the image / 4-column groups that may be loaded
    if (EM == 1 || EM == 2) {
#pragma unroll
        for (int j = 0; j < K; ++j) oob |= (x0 + j < 0 || x0 + j >= a.width) ? 1u << j : 0u;
#pragma unroll
        for (int c = 0; c < K / 4; ++c)
            if (x0 + 4 * c < 0 || x0 + 4 * c + 4 > a.width) cmask &= ~(1u << c);
    }
    const float* gI = a.guide + f * a.gfs;            // column 0 (the column map of EDGE lanes is absolute)
    const float* gP = a.src + f * a.sfs;
    const float* gIx = gI + x0;                        // this lane's first column
    const float* gPx = gP + x0;
    const int rows_hi = (a.buf_y0 + a.buf_rows < a.height ? a.buf_y0 + a.buf_rows : a.height) - 1 - a.buf_y0;

    // buffer row of stream-local input row t, -1 = a row of zeros (TRUNCATE outside the image)
    // (streams whose whole input range [m0-R, m1+R] lies inside the image and the buffer skip the border map)
    const int t_first = st.m0 - R, t_last = st.m1 + R;
    const int ya = st.ys + st.d * t_first, yb = st.ys + st.d * t_last;
    const bool simple = (ya < yb ? ya : yb) >= a.buf_y0 && (ya > yb ? ya : yb) <= a.buf_y0 + rows_hi;
    const int rbase = st.ys - a.buf_y0;
    auto row_of = [&](int t) -> int {
        if (simple) return rbase + st.d * t;
        int y = st.ys + st.d * t;
        if (TRUNC) { if (y < 0 || y >= a.height) return -1; }
        else y = gf_s8_map_y(y, a.height, a.border);
        int rr = y - a.buf_y0;
        rr = rr < 0 ? 0 : (rr > rows_hi ? rows_hi : rr);
        return rr;
    };
    // L2 prefetch hint for the row that enters GF_WS_PF iterations from now: one 128-byte line per lane and plane
    auto prefetch_row = [&](int t) {
        if (GF_WS_PF == 0 || EM == 3) return;
        if (lane * 32 < G::WIN) {
            int rr = row_of(t);
            if (!simple) { if (TRUNC && rr < 0) return; }
            const int64_t c0 = (int64_t)xl + lane * 32;
            if (c0 >= 0 && c0 + 32 <= a.width) {
                gf_prefetch_l2(gI + (int64_t)rr * a.gs + c0);
                gf_prefetch_l2(gP + (int64_t)rr * a.ss + c0);
            }
        }
    };
    // the K columns of this lane from a row pointer that already points at the lane's first column
    auto ld_vec = [&](const float* rp, float (&v)[K]) {
            if (EM == 1 || EM == 2) {      // edge strip: groups outside the image are not read (their sums are mirrored in)
#pragma unroll
                for (int c = 0; c < K / 4; ++c) {
                    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (cmask >> c & 1) t = *reinterpret_cast<const float4*>(rp + 4 * c);
                    v[4 * c] = t.x; v[4 * c + 1] = t.y; v[4 * c + 2] = t.z; v[4 * c + 3] = t.w;
                }
            } else if (K % 8 == 0) {       // one 32-byte access per 8 columns: lane stride = access size, fully coalesced
#pragma unroll
                for (int c = 0; c < K / 8; ++c) {
                    float2 t[4];
                    gf_ld8(rp + 8 * c, t);
#pragma unroll
                    for (int i = 0; i < 4; ++i) { v[8 * c + 2 * i] = t[i].x; v[8 * c + 2 * i + 1] = t[i].y; }
                }
            } else {
#pragma unroll
                for (int c = 0; c < K / 4; ++c) {
                    const float4 t = *reinterpret_cast<const float4*>(rp + 4 * c);
                    v[4 * c] = t.x; v[4 * c + 1] = t.y; v[4 * c + 2] = t.z; v[4 * c + 3] = t.w;
                }
            }
    };
    auto ld_row = [&](const float* plane, const float* planex, int64_t stride, int rr, float (&v)[K]) {
        if (TRUNC && rr < 0) {
#pragma unroll
            for (int j = 0; j < K; ++j) v[j] = 0.f;
            return;
        }
        const int64_t ro = (int64_t)rr * stride;
        if (vec) {
            const float* rp = planex + ro;
            if (EM == 1 || EM == 2) {      // edge strip: groups outside the image are not read (their sums are mirrored in)
#pragma unroll
                for (int c = 0; c < K / 4; ++c) {
                    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (cmask >> c & 1) t = *reinterpret_cast<const float4*>(rp + 4 * c);
                    v[4 * c] = t.x; v[4 * c + 1] = t.y; v[4 * c + 2] = t.z; v[4 * c + 3] = t.w;
                }
            } else if (K % 8 == 0) {       // one 32-byte access per 8 columns: lane stride = access size, fully coalesced
#pragma unroll
                for (int c = 0; c < K / 8; ++c) {
                    float2 t[4];
                    gf_ld8(rp + 8 * c, t);
#pragma unroll
                    for (int i = 0; i < 4; ++i) { v[8 * c + 2 * i] = t[i].x; v[8 * c + 2 * i + 1] = t[i].y; }
                }
            } else {
#pragma unroll
                for (int c = 0; c < K / 4; ++c) {
                    const float4 t = *reinterpret_cast<const float4*>(rp + 4 * c);
                    v[4 * c] = t.x; v[4 * c + 1] = t.y; v[4 * c + 2] = t.z; v[4 * c + 3] = t.w;
                }
            }
        } else if (EDGE) {
            const float* rp = plane + ro;
#pragma unroll
            for (int j = 0; j < K; ++j) v[j] = sx[j] >= 0 ? rp[sx[j]] : 0.f;
        }
    };

    // X = (sum I, sum p), Y = (sum I p, sum I I) over the current 2R+1 rows, per column
    float2 X[K], Y[K];
#pragma unroll
    for (int j = 0; j < K; ++j) X[j] = Y[j] = make_float2(0.f, 0.f);

    // warm-up: input rows [m0-R, m0+R) -- loads and adds only, CH rows in flight
    {
        constexpr int CH = K >= 16 ? 2 : 4;
        const int t_end = st.m0 + R;
#pragma unroll 1
        for (int t0 = st.m0 - R; t0 < t_end; t0 += CH) {
            float bI[CH][K], bP[CH][K];
#pragma unroll
            for (int q = 0; q < CH; ++q) {
                const int rr = row_of(t0 + q < t_end ? t0 + q : t_end - 1);     // (rows past the end: loaded again, not added)
                ld_row(gI, gIx, a.gs, rr, bI[q]);
                ld_row(gP, gPx, a.ss, rr, bP[q]);
            }
#pragma unroll
            for (int q = 0; q < CH; ++q) {
                if (t0 + q >= t_end) break;
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    if (ROLE != 2) { X[j].x += bI[q][j]; X[j].y += bP[q][j]; }
                    if (ROLE != 1) {
                        Y[j].x = fmaf(bI[q][j], bP[q][j], Y[j].x);
                        Y[j].y = fmaf(bI[q][j], bI[q][j], Y[j].y);
                    }
                }
            }
        }
    }

    float nI[K], nP[K], oI[K], oP[K];
    {
        const int rr = row_of(st.m0 + R);
        ld_row(gI, gIx, a.gs, rr, nI);
        ld_row(gP, gPx, a.ss, rr, nP);
#pragma unroll
        for (int j = 0; j < K; ++j) oI[j] = oP[j] = 0.f;
    }
    // running pointers (simple streams): the rows of iteration m0 -- entering row m0+R, leaving row m0-R-1 (not used)
    const int64_t stepI = (int64_t)st.d * a.gs, stepP = (int64_t)st.d * a.ss;
    const float* pnI = gIx + (int64_t)(rbase + st.d * (st.m0 + R)) * a.gs;
    const float* pnP = gPx + (int64_t)(rbase + st.d * (st.m0 + R)) * a.ss;
    const float* poI = gIx + (int64_t)(rbase + st.d * (st.m0 - R - 1)) * a.gs;
    const float* poP = gPx + (int64_t)(rbase + st.d * (st.m0 - R - 1)) * a.ss;
    float cx[K];                     // TRUNCATE: in-image columns of the window of each column
    if (TRUNC) {
#pragma unroll
        for (int j = 0; j < K; ++j) cx[j] = gf_count(x0 + j, a.width, R, GF_TRUNCATE);
    }
    const float Nf = (float)(KW * KW);
    const float epsNN = a.eps * Nf * Nf;
    const GfNorm nk = gf_norm_make(Nf);
    volatile int* prod = ctrl + 2 * k;
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(const_cast<int*>(ctrl) + 16);
    const volatile int* cons_own = ctrl + 2 * k + 1;
    const volatile int* cons_sp = ctrl + 2 * (st.sp >= 0 ? st.sp : k) + 1;
    const int n_last = st.L - 1 + R;
    const int n_last_sp = st.sp >= 0 ? pl.s[st.sp].L - 1 + R : 0;
    int slot = 0;

#pragma unroll 1
    for (int m = st.m0; m < st.m1; ++m) {
        // ---- vertical: row m+R enters, row m-R-1 leaves ----
        if (ROLE != 2) {
#pragma unroll
            for (int c = 0; c < K / 2; ++c) {      // (entering - leaving) on the column pairs the loads deliver: FADD2
                const float2 dI = gf_sub2(make_float2(nI[2 * c], nI[2 * c + 1]), make_float2(oI[2 * c], oI[2 * c + 1]));
                const float2 dP = gf_sub2(make_float2(nP[2 * c], nP[2 * c + 1]), make_float2(oP[2 * c], oP[2 * c + 1]));
                X[2 * c].x += dI.x; X[2 * c + 1].x += dI.y;
                X[2 * c].y += dP.x; X[2 * c + 1].y += dP.y;
            }
        }
        if (ROLE != 1) {
#pragma unroll
            for (int j = 0; j < K; ++j) {
                Y[j].x = fmaf(-oI[j], oP[j], fmaf(nI[j], nP[j], Y[j].x));
                Y[j].y = fmaf(-oI[j], oI[j], fmaf(nI[j], nI[j], Y[j].y));
            }
        }
        if (EM == 1 || EM == 2) {
            if (TRUNC) {
#pragma unroll
                for (int j = 0; j < K; ++j)
                    if (oob >> j & 1) X[j] = Y[j] = make_float2(0.f, 0.f);
            } else {
                constexpr int CL0 = 2 * G::HALO, CR0 = 2 * (G::WIN - G::HALO - 1);
                if (a.border == GF_REFLECT) {
                    if (EM == 1) { if (ROLE != 2) gf_ws_mirror<K, CL0 - 1>(X, lane, oob); if (ROLE != 1) gf_ws_mirror<K, CL0 - 1>(Y, lane, oob); }
                    else { if (ROLE != 2) gf_ws_mirror<K, CR0 + 1>(X, lane, oob); if (ROLE != 1) gf_ws_mirror<K, CR0 + 1>(Y, lane, oob); }
                } else {
                    if (EM == 1) { if (ROLE != 2) gf_ws_mirror<K, CL0>(X, lane, oob); if (ROLE != 1) gf_ws_mirror<K, CL0>(Y, lane, oob); }
                    else { if (ROLE != 2) gf_ws_mirror<K, CR0>(X, lane, oob); if (ROLE != 1) gf_ws_mirror<K, CR0>(Y, lane, oob); }
                }
            }
        }
        // ---- rows of the next iteration (a whole iteration to land) ----
        if (ROLE != 1 && m + GF_WS_PF + 1 < st.m1) prefetch_row(m + 1 + R + GF_WS_PF);
        const int cons_seen = ROLE != 1 ? gf_ws_ld_acq(cons_own) : 0;      // read early, needed just before the ring store
        if (m + 1 < st.m1) {
            if (EM != 3 && simple) {       // rows never leave the image: four running row pointers, no per-row address arithmetic
                pnI += stepI; pnP += stepP; poI += stepI; poP += stepP;
                ld_vec(pnI, nI);
                ld_vec(pnP, nP);
                ld_vec(poI, oI);
                ld_vec(poP, oP);
            } else {
                const int rn = row_of(m + 1 + R), ro = row_of(m - R);
                ld_row(gI, gIx, a.gs, rn, nI);
                ld_row(gP, gPx, a.ss, rn, nP);
                ld_row(gI, gIx, a.gs, ro, oI);
                ld_row(gP, gPx, a.ss, ro, oP);
            }
        }
        // ---- horizontal: window sums of the two quantity pairs ----
        const int idx = m - st.m0;
        float2 hX[K], hY[K];
        if (ROLE != 2) gf_ws_window<K, R>(X, hX);
        if (ROLE != 1) gf_ws_window<K, R>(Y, hY);
        if (ROLE == 2) {
            // products warp: wait until every consumer is done with the row the slot held, park the Y sums in it
            if (idx >= RING) {
                const int mm = m - RING;
                const int use = mm + KW < n_last ? mm + KW : n_last;
                if (cons_seen < use + R + 1) gf_ws_wait(cons_own, use + R + 1);
                if (st.sp >= 0 && mm < R) {
                    const int usep = 2 * R - mm < n_last_sp ? 2 * R - mm : n_last_sp;
                    gf_ws_wait(cons_sp, usep + R + 1);
                }
            }
            float4* rp = ring + slot * G::ROW_F4;
#pragma unroll
            for (int c = 0; c < K / 2; ++c) rp[c * 32] = make_float4(hY[2 * c].x, hY[2 * c].y, hY[2 * c + 1].x, hY[2 * c + 1].y);
            __syncwarp();
            if (lane == 0) gf_ws_bar_arrive(bars + k * G::NBAR + RING + slot);
            slot = slot + 1 == RING ? 0 : slot + 1;
            continue;
        }
        if (ROLE == 1) {
            gf_ws_bar_wait(bars + k * G::NBAR + RING + slot, idx / RING);
            const float4* rp = ring + slot * G::ROW_F4;
#pragma unroll
            for (int c = 0; c < K / 2; ++c) {
                const float4 t = rp[c * 32];
                hY[2 * c] = make_float2(t.x, t.y); hY[2 * c + 1] = make_float2(t.z, t.w);
            }
        }
        // ---- a = (N S_Ip - S_I S_p) / (N S_II - S_I^2 + eps N^2),  bN = S_p - a S_I  (b = bN / N) ----
        float av[K], bv[K];
        if (TRUNC) {
            const int yc = st.ys + st.d * m;
            const bool rowin = yc >= 0 && yc < a.height;
            const float cy = gf_s8_cnt_y<R>(yc, a.height);
#pragma unroll
            for (int j = 0; j < K; ++j) {
                const float n2 = cx[j] * cy;
                const float num = fmaf(n2, hY[j].x, -(hX[j].x * hX[j].y));
                const float den = fmaf(-hX[j].x, hX[j].x, fmaf(n2, hY[j].y, a.eps * n2 * n2));
                float rc = gf_s8_rcp(den);
                rc = fmaf(fmaf(-den, rc, 1.0f), rc, rc);
                float rn = gf_s8_rcp(n2);
                rn = fmaf(fmaf(-n2, rn, 1.0f), rn, rn);
                const float aa = num * rc;
                const float bb = fmaf(-aa, hX[j].x, hX[j].y) * rn;
                const bool ok = rowin && (EDGE ? sx[j] >= 0 : !(oob >> j & 1));
                av[j] = ok ? aa : 0.f;
                bv[j] = ok ? bb : 0.f;
            }
        } else {
            // (num, den) = N (S_Ip, S_II) + (0, eps N^2) - S_I (S_p, S_I): two FFMA2 (the broadcast and the
            // swapped operand are operand modifiers of the packed instructions on sm_100)
            const float2 cN = make_float2(Nf, Nf), cE = make_float2(0.f, epsNN);
#pragma unroll
            for (int j = 0; j < K; ++j) {
                const float2 t = gf_fma2(cN, hY[j], cE);
                const float2 u = gf_fma2(make_float2(-hX[j].x, -hX[j].x), make_float2(hX[j].y, hX[j].x), t);
                float rc = gf_s8_rcp(u.y);
                if (GF_WS_NEWTON) rc = fmaf(fmaf(-u.y, rc, 1.0f), rc, rc);
                av[j] = u.x * rc;
                bv[j] = fmaf(-av[j], hX[j].x, hX[j].y);
            }
        }
        // ---- the ring slot of row m held row m-RING: every consumer of that row must be done with it ----
        if (ROLE == 0 && idx >= RING) {
            const int mm = m - RING;
            const int use = mm + KW < n_last ? mm + KW : n_last;          // last step of the own consumer that reads row mm
            if (cons_seen < use + R + 1) gf_ws_wait(cons_own, use + R + 1);
            if (st.sp >= 0 && mm < R) {                                    // ... and of the start partner (its row -1-mm)
                const int usep = 2 * R - mm < n_last_sp ? 2 * R - mm : n_last_sp;
                gf_ws_wait(cons_sp, usep + R + 1);
            }
        }
        {
            float4* rp = ring + slot * G::ROW_F4;
#pragma unroll
            for (int c = 0; c < K / 2; ++c) rp[c * 32] = make_float4(av[2 * c], bv[2 * c], av[2 * c + 1], bv[2 * c + 1]);
        }
        gf_ws_row_ready<RING>(prod, bars + k * G::NBAR, idx, slot, lane);
        slot = slot + 1 == RING ? 0 : slot + 1;
        // ---- optional A / B planes (hGuidedFilter's d_A, d_B): own territory rows, output columns ----
        if (a.A != nullptr && m >= 0 && m < st.L) {
            const int y = st.ys + st.d * m;
            float* pa = a.A + f * a.abfs + (int64_t)(y - a.out_y0) * a.abs_ + x0;
            float* pb = a.B + f * a.abfs + (int64_t)(y - a.out_y0) * a.abs_ + x0;
#pragma unroll
            for (int c = 0; c < K / 4; ++c) {
                const int xc = x0 + 4 * c;
                if (xc >= out_lo && xc + 4 <= out_hi) {
                    float b4[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) b4[i] = TRUNC ? bv[4 * c + i] : gf_norm_apply(bv[4 * c + i], nk);
                    *reinterpret_cast<float4*>(pa + 4 * c) = make_float4(av[4 * c], av[4 * c + 1], av[4 * c + 2], av[4 * c + 3]);
                    *reinterpret_cast<float4*>(pb + 4 * c) = make_float4(b4[0], b4[1], b4[2], b4[3]);
                }
            }
        }
    }
#if GF_WS_SYNC == 2
    __syncwarp();
    if (ROLE != 2 && lane == 0) gf_ws_bar_arrive(bars + k * G::NBAR + 2 * RING);        // "stream finished": every own row is in the ring
#endif
}

// ---- stage 2: consumer warp -------------------------------------------------------------------------
template <int R, int K, int NS, bool TRUNC>
__device__ __forceinline__ void gf_ws_stage2(const GfWsArgs& a, const GfWsPlan<NS>& pl, int k, int lane, int64_t f, int xl,
                                             int out_lo, int out_hi, const float4* rings, volatile int* ctrl)
{
    using G = GfWsGeom<R, K, NS>;
    constexpr int RING = G::RING, KW = G::KW;
    const GfWsStream st = pl.s[k];
    const int x0 = xl + lane * K;
    const float* gI = a.guide + f * a.gfs + x0;
    float* gQ = a.dst + f * a.dfs + x0;
    unsigned omask = 0;                       // 4-column groups this lane stores
#pragma unroll
    for (int c = 0; c < K / 4; ++c) {
        const int u = lane * K + 4 * c, xc = x0 + 4 * c;
        if (u >= G::HALO && u + 4 <= G::WIN - G::HALO && xc >= out_lo && xc + 4 <= out_hi) omask |= 1u << c;
    }
    float cx[K];
    if (TRUNC) {
#pragma unroll
        for (int j = 0; j < K; ++j) cx[j] = gf_count(x0 + j, a.width, R, GF_TRUNCATE);
    }
    // mean_a = sum_a / N, mean_b = sum_bN / N^2, both as two-term reciprocals, on the (a, b) pair at once
    const GfNorm nk1 = gf_norm_make((float)(KW * KW)), nk2 = gf_norm_make((float)(KW * KW) * (float)(KW * KW));
    const float2 nh = make_float2(nk1.hi, nk2.hi), nl = make_float2(nk1.lo, nk2.lo);
    volatile int* cons = ctrl + 2 * k + 1;
    const int ep_last = st.ep >= 0 ? pl.s[st.ep].L - 1 - pl.s[st.ep].m0 + st.L : 0;    // ring index of row n >= L in the end partner: ep_last - n

    // ring row and producer counter of stream-local a/b row n
    const unsigned long long* bars = reinterpret_cast<const unsigned long long*>(const_cast<const int*>(ctrl) + 16);
    auto resolve = [&](int n, const float4*& base, const volatile int*& prod, const unsigned long long*& bar, int& idx) {
        int t = k;
        idx = n - st.m0;
        if (n < 0 && st.sp >= 0) { t = st.sp; idx = -1 - n; }              // (a shared start: the partner's m0 is 0)
        else if (n >= st.L && st.ep >= 0) { t = st.ep; idx = ep_last - n; }
        base = rings + (t * RING + idx % RING) * G::ROW_F4 + lane;
        prod = ctrl + 2 * t;
        bar = bars + t * G::NBAR;
    };
    const int64_t stepG = (int64_t)st.d * a.gs, stepQ = (int64_t)st.d * a.ds;
    const float* gp = gI + (int64_t)(st.ys - a.buf_y0) * a.gs - stepG;      // advanced by one row per ld_guide call (rows i = 0, 1, ..)
    float* qrow = gQ + (int64_t)(st.ys - a.out_y0) * a.ds - stepQ;
    auto ld_guide = [&](int, float (&g)[K]) {
        gp += stepG;
        const float* rp = gp;
#pragma unroll
        for (int c = 0; c < K / 4; ++c) {
            float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
            if (omask >> c & 1) t = *reinterpret_cast<const float4*>(rp + 4 * c);
            g[4 * c] = t.x; g[4 * c + 1] = t.y; g[4 * c + 2] = t.z; g[4 * c + 3] = t.w;
        }
    };

    float2 V[K];                              // (sum a, sum bN) over the current 2R+1 rows, per column
#pragma unroll
    for (int j = 0; j < K; ++j) V[j] = make_float2(0.f, 0.f);
    float g[K];
    ld_guide(0, g);
    const int n_last = st.L - 1 + R;
#pragma unroll 1
    for (int n = -R; n <= n_last; ++n) {
        const float4* nb; const volatile int* np; const unsigned long long* nbar; int ni;
        resolve(n, nb, np, nbar, ni);
        gf_ws_row_wait<RING>(np, nbar, ni, n >= st.L && st.ep >= 0);
        float4 nw[K / 2];
#pragma unroll
        for (int c = 0; c < K / 2; ++c) nw[c] = nb[c * 32];
        if (n - KW >= -R) {
            const float4* ob; const volatile int* op; const unsigned long long* obar; int oi;
            resolve(n - KW, ob, op, obar, oi);
#pragma unroll
            for (int c = 0; c < K / 2; ++c) {
                const float4 o = ob[c * 32];
                V[2 * c] = gf_add2(V[2 * c], gf_sub2(make_float2(nw[c].x, nw[c].y), make_float2(o.x, o.y)));
                V[2 * c + 1] = gf_add2(V[2 * c + 1], gf_sub2(make_float2(nw[c].z, nw[c].w), make_float2(o.z, o.w)));
            }
        } else {
#pragma unroll
            for (int c = 0; c < K / 2; ++c) {
                V[2 * c] = gf_add2(V[2 * c], make_float2(nw[c].x, nw[c].y));
                V[2 * c + 1] = gf_add2(V[2 * c + 1], make_float2(nw[c].z, nw[c].w));
            }
        }
        gf_ws_publish(cons, n + R + 1, lane);       // the ring rows are in registers: the producer may move on
        if (n < R) continue;
        // ---- output row i = n - R ----
        const int i = n - R;
        float2 W[K];
        gf_ws_window<K, R>(V, W);
        float q[K];
        if (TRUNC) {
            const int y = st.ys + st.d * i;
            const float cy = gf_s8_cnt_y<R>(y, a.height);
#pragma unroll
            for (int j = 0; j < K; ++j) {
                const float n2 = cx[j] * cy;
                float rn = gf_s8_rcp(n2);
                rn = fmaf(fmaf(-n2, rn, 1.0f), rn, rn);
                q[j] = fmaf(W[j].x, g[j], W[j].y) * rn;
            }
        } else {
#pragma unroll
            for (int j = 0; j < K; ++j) {
                const float2 m = GF_WS_NORM2 ? gf_fma2(W[j], nh, gf_mul2(W[j], nl)) : gf_mul2(W[j], nh);
                q[j] = fmaf(m.x, g[j], m.y);
            }
        }
        {
            qrow += stepQ;
            float* qp = qrow;
#pragma unroll
            for (int c = 0; c < K / 4; ++c)
                if (omask >> c & 1) *reinterpret_cast<float4*>(qp + 4 * c) = make_float4(q[4 * c], q[4 * c + 1], q[4 * c + 2], q[4 * c + 3]);
        }
        if (i + 1 < st.L) ld_guide(i + 1, g);
    }
}

// ---- kernel: one CTA = one (frame, strip, band) ---------------------------------------------------------
// SPLIT = false: warps [0, NS) produce, [NS, 2 NS) consume.  SPLIT = true: [0, NS) sums + solve, [NS, 2 NS) products,
// [2 NS, 3 NS) consume (warp w, NS + w, 2 NS + w of a 4-stream CTA share a scheduler).
template <int R, int K, int NS, bool TRUNC, bool SPLIT>
__global__ void __launch_bounds__((SPLIT ? 96 : 64) * NS, 1) gf_ws_gray_kernel(const GF_GRID_CONSTANT GfWsArgs a)
{
    using G = GfWsGeom<R, K, NS>;
    GF_DYN_SMEM(float4, smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    volatile int* ctrl = reinterpret_cast<volatile int*>(smem + (size_t)NS * G::RING * G::ROW_F4);
    const long item = (long)blockIdx.x;
    // items of a frame: (optionally) the two edge strips first, in their own shorter bands -- their producers run the
    // mirror code and take longer per row --, then the other strips band by band (strips of one band run side by side:
    // their halos hit in L2)
    const bool two = a.nbands_e > 0;
    const long per_frame = two ? 2L * a.nbands_e + (long)(a.nstrips - 2) * a.nbands : (long)a.nstrips * a.nbands;
    const int64_t f = item / per_frame;
    const int rem = (int)(item % per_frame);
    int band, strip, hbw;
    if (two && rem < 2 * a.nbands_e) { band = rem >> 1; strip = (rem & 1) ? a.nstrips - 1 : 0; hbw = a.hb_e; }
    else if (two) { const int q = rem - 2 * a.nbands_e; band = q / (a.nstrips - 2); strip = 1 + q % (a.nstrips - 2); hbw = a.hb; }
    else { band = rem / a.nstrips; strip = rem % a.nstrips; hbw = a.hb; }
    const int y0 = a.out_y0 + band * hbw;
    const int y1 = y0 + hbw < a.out_y0 + a.out_rows ? y0 + hbw : a.out_y0 + a.out_rows;
    if (threadIdx.x < 2 * NS) ctrl[threadIdx.x] = 0;
    for (int i = threadIdx.x; i < NS * G::NBAR; i += blockDim.x)          // (2-stream CTAs have fewer threads than barriers)
        gf_ws_bar_init(reinterpret_cast<unsigned long long*>(const_cast<int*>(ctrl) + 16) + i);
    __syncthreads();
    GfWsPlan<NS> pl;
    gf_ws_plan<R, NS>(y0, y1, a.pen, pl);
    // strips tile the width in steps of WOUT; the LAST one is pulled back so that its window ends exactly HALO columns
    // past the image (its mirror is then the compile-time twin of the first strip's) and writes only the columns
    // the strip before it left over
    const int out_lo = strip * G::WOUT;
    const int out_hi = out_lo + G::WOUT < a.width ? out_lo + G::WOUT : a.width;
    int xl = strip * G::WOUT - G::HALO;
    if (strip == a.nstrips - 1 && a.nstrips > 1 && a.width + G::HALO - G::WIN >= 0) xl = a.width + G::HALO - G::WIN;
    const int k = warp % NS, part = warp / NS;
    if (k >= pl.n) return;
#ifdef GF_WS_TIMING
    const long long t_start = clock64();
    struct DbgStamp {
        long long* p; long long t0; int lane; int info0, info1;
        __device__ ~DbgStamp() { if (p && lane == 0) { p[0] = t0; p[1] = clock64(); p[2] = info0; p[3] = info1; } }
    } dbg_stamp{a.dbg ? a.dbg + ((long long)blockIdx.x * (3 * NS) + warp) * 4 : nullptr, t_start, lane,
                (strip << 16) | band, (pl.s[k].L << 16) | ((pl.s[k].m1 - pl.s[k].m0) & 0xffff)};
#endif
    const bool in_l = xl >= 0, in_r = xl + G::WIN <= a.width;
    const int em = (in_l && in_r) ? 0 : ((xl == -G::HALO && in_r) ? 1 : ((in_l && xl + G::WIN == a.width + G::HALO) ? 2 : 3));
#define GF_WS_S1(ROLE)                                                                                                   \
    do {                                                                                                                 \
        if (em == 0) gf_ws_stage1<R, K, NS, TRUNC, 0, ROLE>(a, pl, k, lane, f, xl, out_lo, out_hi, smem, ctrl);            \
        else if (em == 1) gf_ws_stage1<R, K, NS, TRUNC, 1, ROLE>(a, pl, k, lane, f, xl, out_lo, out_hi, smem, ctrl);       \
        else if (em == 2) gf_ws_stage1<R, K, NS, TRUNC, 2, ROLE>(a, pl, k, lane, f, xl, out_lo, out_hi, smem, ctrl);       \
        else gf_ws_stage1<R, K, NS, TRUNC, 3, ROLE>(a, pl, k, lane, f, xl, out_lo, out_hi, smem, ctrl);                    \
    } while (0)
    if (SPLIT) {
        if (part == 0) GF_WS_S1(1);
        else if (part == 1) GF_WS_S1(2);
        else gf_ws_stage2<R, K, NS, TRUNC>(a, pl, k, lane, f, xl, out_lo, out_hi, smem, ctrl);
    } else {
        if (part == 0) GF_WS_S1(0);
        else gf_ws_stage2<R, K, NS, TRUNC>(a, pl, k, lane, f, xl, out_lo, out_hi, smem, ctrl);
    }
#undef GF_WS_S1
}

// ---- host side --------------------------------------------------------------------------------------
#ifndef GF_NO_HOST
// Longest sub-band a stream walks with sliding (add / subtract) vertical sums before the band is cut.
// Whether gf_guided_gray & co. take this kernel when they can (option GF_WS overrides)
#ifndef GF_WS_DEFAULT
#define GF_WS_DEFAULT 0
#endif
// Producer split over two warps (option GF_WS_SPLIT1 overrides)
#ifndef GF_WS_SPLIT1_DEFAULT
#define GF_WS_SPLIT1_DEFAULT 0
#endif
#ifndef GF_WS_WITH_SPLIT1
#ifdef GF_CPU_EMU
#define GF_WS_WITH_SPLIT1 1
#else
#define GF_WS_WITH_SPLIT1 0
#endif
#endif
#ifndef GF_WS_MAX_SUB
#define GF_WS_MAX_SUB 512
#endif

// Band heights: CTAs run in waves of `sms` (one CTA per SM); a CTA's time ~ its slowest stream:
//   (hb + 2 x 0.85 R outer rows) / NS  +  2R warm-up rows at ~0.2  +  ~2 rows of start-up,
// times `edge_pct` % for the first and the last strip (mirror shuffles in the producer, measured ~1.35x per row:
// profiles/r2_ws_edge_rows.txt), which therefore get their own, shorter bands.
struct GfWsBands { int hb, nbands, hb_e, nbands_e; };
template <int R, int NS>
static inline GfWsBands gf_ws_pick_bands(int rows, int nstrips, long count, int sms, int edge_pct)
{
    const int hb_min = NS * (R + 1) + 2 * R;
    auto cost = [](int hb) { return (hb + 1.7 * R) / NS + 0.4 * R + 2.0; };
    GfWsBands best{rows, 1, 0, 0};
    double best_t = 1e300;
    const bool edges = nstrips >= 3 && edge_pct > 100;
    for (int nb = 1; nb <= 4096; ++nb) {
        const int hb = (rows + nb - 1) / nb;
        if (hb < hb_min && nb > 1) break;
        if (hb > NS * GF_WS_MAX_SUB) continue;
        const int nbr = (rows + hb - 1) / hb;
        for (int nbe = nbr; nbe <= (edges ? 2 * nbr : nbr); ++nbe) {
            const int hbe = (rows + nbe - 1) / nbe;
            if (nbe > nbr && hbe < hb_min) break;
            const int nber = (rows + hbe - 1) / hbe;
            const long items = count * (edges ? 2L * nber + (long)(nstrips - 2) * nbr : (long)nstrips * nbr);
            const long waves = (items + sms - 1) / sms;
            const double ti = cost(hb), te = edges ? cost(hbe) * edge_pct / 100.0 : 0.0;
            const double t = (double)waves * (ti > te ? ti : te);
            if (t < best_t * 0.999) { best_t = t; best = GfWsBands{hb, nbr, edges && nber != nbr ? hbe : 0, edges && nber != nbr ? nber : 0}; }
        }
    }
    return best;
}

template <int R, int K, int NS>
static const char* gf_ws_launch(const Job& j)
{
    using G = GfWsGeom<R, K, NS>;
    static_assert(G::smem_bytes <= 227 * 1024, "rings do not fit");
    int sms = 148, mj = 0, mn = 0;
    gf_rt_device_info(&sms, &mj, &mn);
    GfWsArgs a;
    a.guide = j.guide.ptr; a.src = j.src.ptr; a.dst = const_cast<float*>(j.dst.ptr);
    a.A = const_cast<float*>(j.A.ptr); a.B = const_cast<float*>(j.B.ptr);
    a.gs = j.guide.stride; a.ss = j.src.stride; a.ds = j.dst.stride; a.abs_ = j.A.ptr ? j.A.stride : 0;
    a.gfs = j.guide.frame_stride; a.sfs = j.src.frame_stride; a.dfs = j.dst.frame_stride; a.abfs = j.A.ptr ? j.A.frame_stride : 0;
    a.width = j.width; a.height = j.height; a.buf_y0 = j.buf_y0; a.buf_rows = j.buf_rows; a.out_y0 = j.out_y0;
    a.out_rows = j.out_rows; a.border = j.border; a.eps = j.eps; a.count = j.count;
    a.nstrips = (j.width + G::WOUT - 1) / G::WOUT;
    a.pen = GF_KNOB("GF_WS_PEN", (3 * R) / 8);
    if (a.pen > 2 * R) a.pen = 2 * R;
    a.dbg = nullptr;
#ifdef GF_WS_TIMING
    a.dbg = (long long*)(((unsigned long long)(unsigned)GF_KNOB("GF_WS_DBG_HI", 0) << 31) | (unsigned long long)(unsigned)GF_KNOB("GF_WS_DBG_LO", 0));
#endif
    GfWsBands bd = gf_ws_pick_bands<R, NS>(j.out_rows, a.nstrips, j.count, sms, GF_KNOB("GF_WS_EDGE_PCT", 135));
    if (GF_KNOB_SET("GF_WS_HB")) {
        int hb = GF_KNOB("GF_WS_HB", bd.hb);
        hb = hb > j.out_rows ? j.out_rows : (hb < 1 ? 1 : hb);
        bd = GfWsBands{hb, (j.out_rows + hb - 1) / hb, 0, 0};
    }
    a.hb = bd.hb; a.nbands = bd.nbands; a.hb_e = bd.hb_e; a.nbands_e = bd.nbands_e;
    const long items = (a.nbands_e > 0 ? 2L * a.nbands_e + (long)(a.nstrips - 2) * a.nbands : (long)a.nstrips * a.nbands) * j.count;
    // The split-producer kernels (measured 20-90 % slower, DESIGN.md section 3.3) are compiled only into the emulator
    // build (their hand-off logic stays under test) and into -DGF_WS_WITH_SPLIT1=1 experiment builds.
#if GF_WS_WITH_SPLIT1
    const bool split = GF_KNOB("GF_WS_SPLIT1", GF_WS_SPLIT1_DEFAULT) != 0;
#else
    const bool split = false;
#endif
    dim3 grid((unsigned)items), block((split ? 96 : 64) * NS);
    const char* e;
#define GF_WS_GO(TR, SP)                                                        \
    do {                                                                        \
        auto kf = gf_ws_gray_kernel<R, K, NS, TR, SP>;                          \
        if ((e = gf_rt_set_smem(kf, G::smem_bytes))) return e;                  \
        GF_LAUNCH(kf, grid, block, G::smem_bytes, j.stream, a);                 \
    } while (0)
#if GF_WS_WITH_SPLIT1
    if (j.border == GF_TRUNCATE) { if (split) GF_WS_GO(true, true); else GF_WS_GO(true, false); }
    else { if (split) GF_WS_GO(false, true); else GF_WS_GO(false, false); }
#else
    if (j.border == GF_TRUNCATE) GF_WS_GO(true, false); else GF_WS_GO(false, false);
#endif
#undef GF_WS_GO
    return gf_rt_launch_error();
}

static const char* gf_ws_try(const Job& j, bool* done, const char** name)
{
    *done = false;
    // default ON for: jobs that want the a / b planes (hGuidedFilter's d_A, d_B through the drop-in shim) -- the producer warps store
    // them on the side, where the round-1 kernels fall back to their first generation (wp: 103 us at 4K r=8); plain jobs
    // stay on gf_s8, which is as fast at 4K and faster above (DESIGN.md section 3.3)
    // ... and single frames of up to 12 Mpx at r = 8 (the headline shape: 62.4 us against 65.7 us at 4K, 35.5 against 37.1 at
    // 1080p; above that size gf_s8's steady state wins: 8K 192 vs 170 us, profiles/r2_ws_matrix_final.jsonl, r2_ws_pen.jsonl)
    const bool small_r8 = j.r == 8 && j.count == 1 && (int64_t)j.width * j.out_rows <= 12000000;
    if (j.color || !GF_KNOB("GF_WS", (j.A.ptr || small_r8) ? 1 : GF_WS_DEFAULT) || GF_KNOB("GF_DISABLE_FAST", 0) ||
        GF_KNOB("GF_DISABLE_S8", 0))          // (GF_DISABLE_S8 = "first-generation kernels only" in the differential tests)
        return nullptr;
    const int force_k = GF_KNOB("GF_WS_K", 0);
    if ((j.A.ptr == nullptr) != (j.B.ptr == nullptr)) return nullptr;
    const Plane* pl[5] = {&j.guide, &j.src, &j.dst, &j.A, &j.B};
    for (int i = 0; i < 5; ++i) {
        if (!pl[i]->ptr) continue;
        if (pl[i]->channels != 1 || pl[i]->coff != 0 || (pl[i]->stride & 3) || (pl[i]->frame_stride & 3) || ((uintptr_t)pl[i]->ptr & 15))
            return nullptr;
    }
    if (j.A.ptr && (j.A.stride != j.B.stride || j.A.frame_stride != j.B.frame_stride)) return nullptr;
    if (j.width & 3) return nullptr;
    // K = 8 / 16 read the two input planes with 32-byte accesses
    const bool in32 = !((j.guide.stride | j.src.stride | j.guide.frame_stride | j.src.frame_stride) & 7) &&
                      !(((uintptr_t)j.guide.ptr | (uintptr_t)j.src.ptr) & 31);
    // single reflections only (rows), and bands tall enough for at least one stream with its ramp
    if (j.height < 4 * j.r + 2 || j.out_rows < 1) return nullptr;
#define GF_WS_CASE(RR, KK, NN, NAME)                                                  \
    if (j.r == RR && (force_k == 0 || force_k == KK) && j.width >= GfWsGeom<RR, KK, NN>::WOUT && (KK % 8 != 0 || in32)) { \
        *done = true; *name = NAME; return gf_ws_launch<RR, KK, NN>(j);              \
    }
    // (the emulator build compiles the same list: every instantiation that ships is under its tests)
    GF_WS_CASE(8, 12, 4, "ws_r8_k12")
    GF_WS_CASE(8, 8, 6, "ws_r8_k8")
    GF_WS_CASE(7, 12, 4, "ws_r7_k12")
    GF_WS_CASE(4, 8, 6, "ws_r4_k8")
    GF_WS_CASE(16, 12, 2, "ws_r16_k12")
#undef GF_WS_CASE
    return nullptr;
}
#endif  // GF_NO_HOST
