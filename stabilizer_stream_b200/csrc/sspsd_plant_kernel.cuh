// sspsd_plant_kernel.cuh -- plants: K outputs, each an FIR mix of M independent seekable inputs (include/sspsd.h,
// sspsd_plant_*; DESIGN.md 3d):
//   y_i[n] = round_f32( sum_{m < M} sum_{t < L} h[i][m][t] u_m[n - t] ),  u_m[n] = 0 for n < 0,
// the sum formed in f64 in that order (m ascending, then t ascending).  Every product of two f32 values is exact in
// f64, so an FMA and a multiply followed by an add round alike, and one rounding per term is all there is.
// Inputs are counter-based, so any position can be produced directly:
//   NOISE  the stream of sspsd_source NOISE(e, seed), e = 0 .. 8: white Philox noise (noise_block of
//          sspsd_source_kernel.cuh) differenced e times in f32, in source_diff_kernel's order
//   TONE   a * c(phi_n), phi_n = (n ftw) mod 2^32, c the cosine factor of the heterodyne mixer (phase_cos_sin)
//
// One CTA produces PLANT_TILE consecutive positions of all K outputs.  It generates every input's samples for its
// tile, the L samples before it and the differencing history once into shared memory; every thread then forms
// four consecutive positions of all K outputs from there and writes each output with one 16-byte store.  The
// inputs are generated once per CTA whatever K is.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "sspsd_device.cuh"
#include "sspsd_mix_kernel.cuh"
#include "sspsd_source_kernel.cuh"

namespace sspsd {

constexpr int PLANT_MAX_K = 4;
constexpr int PLANT_MAX_M = 4;
constexpr int PLANT_MAX_L = 32;
constexpr int PLANT_NT = 256;
constexpr int PLANT_TILE = 4 * PLANT_NT;  // positions per CTA
// window per input, in samples from a multiple of 4 at or before tile start - L - e_max: the tile, L + e_max history
// samples (the sliding window's last shift reads one more than the FIR uses) and up to 3 of Philox-block alignment
constexpr int PLANT_WIN = PLANT_TILE + PLANT_MAX_L + SRC_MAX_DIFF + 4;  // 1068: 267 Philox blocks
constexpr int PLANT_WQ = PLANT_WIN / 4;
constexpr int PLANT_WPAD = PLANT_WIN + PLANT_WIN / 32 + 1;  // padded (conflict-free strided reads)
enum { PLANT_IN_NOISE = 0, PLANT_IN_TONE = 1 };

struct PlantParams {
    unsigned long long pos;  // absolute position of out[i][0]
    unsigned long long n;    // positions to produce
    int m, taps_len, emax;   // inputs, taps per (output, input), largest differencing order
    int kind[PLANT_MAX_M];
    int order[PLANT_MAX_M];  // NOISE: e
    uint32_t key0[PLANT_MAX_M], key1[PLANT_MAX_M];
    uint32_t ftw[PLANT_MAX_M];
    float amp[PLANT_MAX_M];
    float scale;             // sqrt(12) in f32, as sspsd_source
    float* out[PLANT_MAX_K];
    float taps[PLANT_MAX_K * PLANT_MAX_M * PLANT_MAX_L];  // [k][m][taps_len], dense
};

__device__ __forceinline__ int plant_pad(int i) { return i + (i >> 5); }

template <int K>
__global__ void __launch_bounds__(PLANT_NT) plant_kernel(PlantParams p)
{
    __shared__ float s[PLANT_MAX_M][PLANT_WPAD];
    __shared__ __align__(16) double tap[PLANT_MAX_M][PLANT_MAX_L][PLANT_MAX_K];  // [m][t][i]: one (m, t) is K consecutive doubles
    const int tid = threadIdx.x;
    const int M = p.m, L = p.taps_len;
    const long long P0 = (long long)(p.pos + (unsigned long long)blockIdx.x * PLANT_TILE);
    const long long q0 = (P0 - L - p.emax) >> 2;  // first Philox block of the window (floor, may be negative)
    const int off0 = (int)(P0 - 4 * q0);          // window index of position P0

    for (int idx = tid; idx < M * L * PLANT_MAX_K; idx += PLANT_NT) {
        const int i = idx % PLANT_MAX_K, t = (idx / PLANT_MAX_K) % L, m = idx / (PLANT_MAX_K * L);
        tap[m][t][i] = i < K ? (double)p.taps[(i * M + m) * L + t] : 0.0;
    }
    for (int idx = tid; idx < M * PLANT_WQ; idx += PLANT_NT) {
        const int m = idx / PLANT_WQ, qq = idx - m * PLANT_WQ;
        const long long q = q0 + qq;
        float x[4];
        if (p.kind[m] == PLANT_IN_NOISE) {
            SourceParams sp{};
            sp.key0 = p.key0[m];
            sp.key1 = p.key1[m];
            sp.scale = p.scale;
            noise_block(q, sp, x);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const long long n = 4 * q + j;
                x[j] = n < 0 ? 0.f : __fmul_rn(p.amp[m], phase_cos_sin((uint32_t)((unsigned long long)n * p.ftw[m])).x);
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) s[m][plant_pad(4 * qq + j)] = x[j];
    }
    // e-fold differencing of the noise inputs, level by level as source_diff_kernel: level k at n is level k - 1 at n
    // minus level k - 1 at n - 1.  Window index w is valid at level k from w = k on; the FIR reads w >= e_max.
    constexpr int R = (PLANT_WIN + PLANT_NT - 1) / PLANT_NT;
    for (int lev = 1; lev <= p.emax; ++lev) {
        float v[PLANT_MAX_M][R];
        __syncthreads();
#pragma unroll
        for (int m = 0; m < PLANT_MAX_M; ++m) {
            if (m >= M || lev > p.order[m] || p.kind[m] != PLANT_IN_NOISE) continue;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int w = tid + r * PLANT_NT;
                if (w < PLANT_WIN) v[m][r] = __fsub_rn(s[m][plant_pad(w)], w ? s[m][plant_pad(w - 1)] : 0.f);
            }
        }
        __syncthreads();
#pragma unroll
        for (int m = 0; m < PLANT_MAX_M; ++m) {
            if (m >= M || lev > p.order[m] || p.kind[m] != PLANT_IN_NOISE) continue;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int w = tid + r * PLANT_NT;
                if (w < PLANT_WIN) s[m][plant_pad(w)] = v[m][r];
            }
        }
    }
    __syncthreads();

    const int base = off0 + 4 * tid;  // window index of this thread's first position
    double acc[K][4];
#pragma unroll
    for (int i = 0; i < K; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
    for (int m = 0; m < M; ++m) {
        const float* u = s[m];
        // w_j = u at position (base + j - t)
        double w0 = u[plant_pad(base)], w1 = u[plant_pad(base + 1)], w2 = u[plant_pad(base + 2)],
               w3 = u[plant_pad(base + 3)];
        for (int t = 0; t < L; ++t) {
            double h[K];
            if (K == 1) {
                h[0] = tap[m][t][0];
            } else {
                const double2 a = *reinterpret_cast<const double2*>(&tap[m][t][0]);
                h[0] = a.x;
                h[1] = a.y;
                if (K > 2) {
                    const double2 b = *reinterpret_cast<const double2*>(&tap[m][t][2]);
                    h[2] = b.x;
                    if (K > 3) h[3] = b.y;
                }
            }
#pragma unroll
            for (int i = 0; i < K; ++i) {
                acc[i][0] = fma(h[i], w0, acc[i][0]);
                acc[i][1] = fma(h[i], w1, acc[i][1]);
                acc[i][2] = fma(h[i], w2, acc[i][2]);
                acc[i][3] = fma(h[i], w3, acc[i][3]);
            }
            w3 = w2;
            w2 = w1;
            w1 = w0;
            w0 = u[plant_pad(base - t - 1)];
        }
    }

    const unsigned long long i0 = (unsigned long long)blockIdx.x * PLANT_TILE + 4ull * tid;  // index into out[i]
#pragma unroll
    for (int i = 0; i < K; ++i) {
        float* o = p.out[i] + i0;
        const float4 y = make_float4((float)acc[i][0], (float)acc[i][1], (float)acc[i][2], (float)acc[i][3]);
        if (i0 + 4 <= p.n && (reinterpret_cast<uintptr_t>(o) & 15) == 0) {
            SSPSD_ASSERT(i0 + 3 < p.n);
            *reinterpret_cast<float4*>(o) = y;
        } else {
            const float v[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (i0 + j < p.n) {
                    SSPSD_ASSERT(i0 + j < p.n);
                    o[j] = v[j];
                }
        }
    }
}

}  // namespace sspsd
