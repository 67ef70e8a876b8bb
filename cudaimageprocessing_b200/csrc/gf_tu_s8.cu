// gf_tu_s8.cu -- translation unit of the gf_s8 kernels (one per kernel family: the families compile in parallel)
#define GF_WP_NO_TRY
#define GF_FAST_NO_TRY
#include "gf_s8.cuh"

const char* gf_s8_try_x(const Job& j, bool* done, const char** name, bool u8) { return gf_s8_try(j, done, name, u8); }
#ifdef GF_CPU_EMU   // the test-only emulator build compiles no gf_tu_s8pc.cu: the per-channel instances come with this unit there
const char* gf_s8pc_try_x(const Job& j, bool* done, const char** name) { return gf_s8_per_channel_try(j, done, name); }
#endif
