// sspsd_mix_kernel.cuh -- the heterodyne mixer of ZoomCascade (sspsd_heterodyne_f32 of include/sspsd.h):
//   i[n] = x[n] cos(2 pi phi_n / 2^32),  q[n] = -x[n] sin(2 pi phi_n / 2^32),  phi_n = ((pos0 + n) ftw) mod 2^32
// so that i + i q = x exp(-2 pi i phi_n / 2^32).  The phase is formed in integer arithmetic from the absolute sample
// index (a u64 product taken mod 2^32), so it stays exact and phase-continuous however far the stream runs and
// however it is split over calls.
//
// Accuracy (DESIGN.md 3c): the quadrant is the phase's top two bits; the rest, r < 2^30, is the exact f64 argument
// r 2^-31 of sincospi, whose results are rounded once to f32 (at most 2^-25 off for values up to 1) and rotated by
// the quadrant without rounding.  One f32 product with x adds at most 2^-24 |x|, so every output is within
// 2^-23 |x| of the f64 product, and at a quarter turn (r = 0) the factors are exactly 0 and +-1.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace sspsd {

// (cos, sin) of 2 pi phi / 2^32, each rounded once to f32, exact at multiples of a quarter turn
__device__ __forceinline__ float2 phase_cos_sin(uint32_t phi)
{
    const uint32_t quad = phi >> 30;
    double s, c;
    sincospi((double)(phi & 0x3fffffffu) * 0x1p-31, &s, &c);
    const float cf = (float)c, sf = (float)s;
    switch (quad) {  // exp(i pi/2 quad) exp(i a)
        case 0: return make_float2(cf, sf);
        case 1: return make_float2(-sf, cf);
        case 2: return make_float2(-cf, -sf);
        default: return make_float2(sf, -cf);
    }
}

static __global__ void heterodyne_kernel(const float* __restrict__ x, size_t n, uint64_t pos0, uint32_t ftw,
                                         float* __restrict__ i_out, float* __restrict__ q_out)
{
    for (size_t k = blockIdx.x * (size_t)blockDim.x + threadIdx.x; k < n; k += (size_t)gridDim.x * blockDim.x) {
        const uint32_t phi = (uint32_t)((pos0 + k) * (uint64_t)ftw);
        const float2 cs = phase_cos_sin(phi);
        const float v = x[k];
        i_out[k] = v * cs.x;
        q_out[k] = -(v * cs.y);
    }
}

}  // namespace sspsd
