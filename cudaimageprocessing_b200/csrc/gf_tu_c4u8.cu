// gf_tu_c4u8.cu -- translation unit of the uint8 colour-guide kernels (gf_c4.cuh, T = unsigned char: gf_guided_color_u8)
#define GF_S8_NO_TRY
#define GF_WP_NO_TRY
#define GF_FAST_NO_TRY
#include "gf_c4.cuh"

const char* gf_c4u8_try_x(const Job& j, bool* done, const char** name) { return gf_c4_try<unsigned char>(j, done, name); }
