// Host build of the fp16 weight packing in csrc/pilot_api.cu (upload_weights, the conv1 row weights): __float2half_rn from
// cuda_fp16.h, compiled for the CPU, so tests/test_pilot_bounds_host.py can hold numpy's float16 rounding to it.
#include <cuda_fp16.h>
#include <stdint.h>
#include <string.h>

static uint16_t bits(__half h)
{
    uint16_t u;
    memcpy(&u, &h, sizeof u);
    return u;
}

extern "C" void pack_rn(const float* in, uint16_t* out, long long n)
{
    for (long long i = 0; i < n; ++i) out[i] = bits(__float2half_rn(in[i]));
}

// conv1: the 1 / 255 of the input scaling folded into the weights, fp32 division first (pilot_api.cu:245, 378)
extern "C" void pack_conv1(const float* in, uint16_t* out, long long n)
{
    for (long long i = 0; i < n; ++i) out[i] = bits(__float2half_rn(in[i] / 255.0f));
}
