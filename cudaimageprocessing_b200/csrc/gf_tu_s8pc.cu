// gf_tu_s8pc.cu -- translation unit of the uint8 per-channel s8 kernels (gf_s8.cuh, T = unsigned char, 3 interleaved
// src / dst channels: gf_guided_per_channel_u8)
#define GF_WP_NO_TRY
#define GF_FAST_NO_TRY
#define GF_S8_PER_CHANNEL_TRY
#include "gf_s8.cuh"

const char* gf_s8pc_try_x(const Job& j, bool* done, const char** name) { return gf_s8_per_channel_try(j, done, name); }
