// gf_tu_c4.cu -- translation unit of the colour-guide kernels (gf_c4.cuh)
#define GF_S8_NO_TRY
#define GF_WP_NO_TRY
#define GF_FAST_NO_TRY
#include "gf_c4.cuh"

const char* gf_c4_try_x(const Job& j, bool* done, const char** name) { return gf_c4_try<float>(j, done, name); }
#ifdef GF_CPU_EMU   // the test-only emulator build compiles one unit per kernel family and no gf_tu_c4u8.cu: the uint8
                    // instances of the same kernel come with this one there
const char* gf_c4u8_try_x(const Job& j, bool* done, const char** name) { return gf_c4_try<unsigned char>(j, done, name); }
#endif
