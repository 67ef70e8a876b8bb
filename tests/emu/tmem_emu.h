// tmem_emu.h -- tensor memory (tcgen05) for the test-only SIMT emulator (cuda_emu.h).
//
// TEST INFRASTRUCTURE, like cuda_emu.h: included by the kernels only in the -DGF_CPU_EMU build.  The emulator runs the
// fibers of one block on one host thread and the blocks of that thread one after the other, so a thread-local store is
// one CTA's tensor memory: 128 lanes x 512 32-bit columns.  alloc / dealloc are collective over the calling warp (lane 0
// acts, every lane waits); a 32x32b access of lane i reaches TMEM lane (taddr >> 16) + i, columns [taddr & 0xffff, + n),
// and a warp reaches only the 32 lanes of quarter warp % 4.  Misuse aborts with a message: an access from the wrong
// quarter or to columns that are not allocated, an allocation while columns are still allocated (a block that did not
// free its columns shows up at the next allocation of its host thread).  Freshly allocated columns hold NaN.
#pragma once
#include <vector>

#include "cuda_emu.h"

namespace emu {

struct Tmem {
    static const int kLanes = 128, kCols = 512;
    std::vector<uint32_t> cell = std::vector<uint32_t>((size_t)kLanes * kCols);
    unsigned used = 0;     // allocated 32-column chunks
};
inline Tmem& tmem() { static thread_local Tmem t; return t; }

[[noreturn]] inline void tmem_fail(const char* what, unsigned taddr, int n)
{
    std::fprintf(stderr, "cuda_emu: tensor memory: %s (block (%u,%u,%u), thread %d, address lane %u column %u, %d columns)\n", what,
                 g_blockIdx.x, g_blockIdx.y, g_blockIdx.z, linear_tid(), taddr >> 16, taddr & 0xffff, n);
    std::abort();
}
inline unsigned tmem_chunks(unsigned col, int ncols) { return ((1u << (ncols / 32)) - 1) << (col / 32); }

inline void tmem_alloc(unsigned* dst, int ncols)
{
    Tmem& t = tmem();
    if ((linear_tid() & 31) == 0) {
        if (ncols < 32 || ncols > Tmem::kCols || (ncols & (ncols - 1))) tmem_fail("allocation size not a power of 2 in [32, 512]", 0, ncols);
        if (t.used) tmem_fail("allocation while columns are still allocated (here or by an earlier block)", 0, ncols);
        t.used = tmem_chunks(0, ncols);
        for (int l = 0; l < Tmem::kLanes; ++l)
            for (int c = 0; c < ncols; ++c) t.cell[(size_t)l * Tmem::kCols + c] = 0x7fc00000u;
        *dst = 0u;
    }
    yield_to_scheduler(AT_WARP);
}

inline void tmem_dealloc(unsigned taddr, int ncols)
{
    Tmem& t = tmem();
    if ((linear_tid() & 31) == 0) {
        const unsigned col = taddr & 0xffff, m = tmem_chunks(col, ncols);
        if ((taddr >> 16) != 0 || col % ncols || (t.used & m) != m) tmem_fail("freeing columns that are not allocated", taddr, ncols);
        t.used &= ~m;
    }
    yield_to_scheduler(AT_WARP);
}

inline uint32_t* tmem_at(unsigned taddr, int n)
{
    Tmem& t = tmem();
    const int tid = linear_tid();
    const unsigned lane0 = taddr >> 16, col = taddr & 0xffff;
    if (lane0 != 32u * ((tid >> 5) % 4)) tmem_fail("a warp reaches only the lanes of its own quarter", taddr, n);
    for (unsigned c = col; c < col + n; ++c)
        if (c >= (unsigned)Tmem::kCols || !(t.used >> (c / 32) & 1)) tmem_fail("access to columns that are not allocated", taddr, n);
    return t.cell.data() + (size_t)(lane0 + (tid & 31)) * Tmem::kCols + col;
}

inline void tmem_st(unsigned taddr, int n, const float* v) { std::memcpy(tmem_at(taddr, n), v, 4 * n); }
inline void tmem_ld(unsigned taddr, int n, float* v) { std::memcpy(v, tmem_at(taddr, n), 4 * n); }

}  // namespace emu
