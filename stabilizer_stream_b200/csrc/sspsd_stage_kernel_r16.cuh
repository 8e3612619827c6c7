// sspsd_stage_kernel_r16.cuh -- K2 for N = 4096, second generation.
//
// Same contract as psd_stage_kernel<12> (sspsd_stage_kernel.cuh; reference src/psd.rs:210-233) but
// with 16 points per thread: 128 threads per segment, M = 2048 = 16 * 16 * 8, i.e. two radix-16
// passes and a final radix-8 pass on 8 contiguous points that is fused with the real-input split
// and |X|^2.  Compared with the radix-8 version (profiles/r01_ncu_summary.md: 37 % issue
// utilisation, LSU pipe the busiest at 49 %, 5 barriers per segment over 8 warps) this does one
// shared-memory exchange less per segment, syncs 4 warps instead of 8 and gives every warp twice
// the independent work between barriers.
//
// Shared-memory layout of a segment's workspace: split re/im planes, element i at
//   L(i) = i + 4*(i>>5) + 8*(i>>7)
// which is conflict free for all three access patterns (pass-0 stores j+128t, pass-1 loads/stores
// 128b+o+8t, last-pass 128-bit loads of 8q..8q+7).
#pragma once
#include "sspsd_stage_kernel.cuh"

namespace sspsd {

struct R16 {
    static constexpr int LOG2N = 12;
    static constexpr int N = 4096, M = 2048;
    static constexpr int TPS = 128;  // threads per segment
    static constexpr int NT = 256;   // threads per CTA
    static constexpr int G = NT / TPS;
    static constexpr int K = M / 8;  // butterflies of the last pass
    static constexpr int WS = 2432;  // floats per plane (>= L(2047)+1, multiple of 4)
};

__device__ __forceinline__ int r16_pos(int i) { return i + ((i >> 5) << 2) + ((i >> 7) << 3); }

__device__ __forceinline__ float2 cmulc(float2 a, float cr, float ci) { return cmul(a, make_float2(cr, ci)); }

// in-place 16-point forward DFT: v[k] = sum_n v[n] exp(-2 pi i n k / 16)
__device__ __forceinline__ void dft16(float2 (&v)[16])
{
    constexpr float h = 0.70710678118654752440f;
    constexpr float c1 = 0.92387953251128675613f, s1 = 0.38268343236508977173f;
    // inner DFT4 over m for each a: inputs v[a + 4m] -> Y_a[b] stored at v[a + 4b]
#pragma unroll
    for (int a = 0; a < 4; ++a) dft4(v[a], v[a + 4], v[a + 8], v[a + 12]);
    // twiddle Y_a[b] *= W16^(a b)   (W^4 = -i is folded into the outer DFT4 of b = 2 below)
    v[1 + 4] = cmulc(v[1 + 4], c1, -s1);    // W^1
    v[1 + 8] = cmulc(v[1 + 8], h, -h);      // W^2
    v[1 + 12] = cmulc(v[1 + 12], s1, -c1);  // W^3
    v[2 + 4] = cmulc(v[2 + 4], h, -h);      // W^2
    v[2 + 12] = cmulc(v[2 + 12], -h, -h);   // W^6
    v[3 + 4] = cmulc(v[3 + 4], s1, -c1);    // W^3
    v[3 + 8] = cmulc(v[3 + 8], -h, -h);     // W^6
    v[3 + 12] = cmulc(v[3 + 12], -c1, s1);  // W^9
    // outer DFT4 over a for each b: inputs v[a + 4b] -> X[b + 4c] stored at v[c + 4b]
    dft4(v[0], v[1], v[2], v[3]);
    dft4(v[4], v[5], v[6], v[7]);
    {
        // b = 2: inputs (v8, v9, -i v10, v11)
        float2 e0 = cadd_mi(v[8], v[10]), e1 = cadd_pi(v[8], v[10]), f0 = cadd(v[9], v[11]), d = csub(v[9], v[11]);
        v[8] = cadd(e0, f0);
        v[10] = csub(e0, f0);
        v[9] = cadd_mi(e1, d);
        v[11] = cadd_pi(e1, d);
    }
    dft4(v[12], v[13], v[14], v[15]);
    // v[c + 4b] holds X[b + 4c]: transpose the 4x4 index to natural order
#pragma unroll
    for (int b = 0; b < 4; ++b)
#pragma unroll
        for (int c = b + 1; c < 4; ++c) {
            float2 t = v[c + 4 * b];
            v[c + 4 * b] = v[b + 4 * c];
            v[b + 4 * c] = t;
        }
}

// multiply v[1..15] by w^1 .. w^15 given w1, w2, w4, w8 (11 extra complex products instead of 15 loads)
__device__ __forceinline__ void twiddle16(float2 (&v)[16], float2 w1, float2 w2, float2 w4, float2 w8)
{
    float2 w3 = cmul(w1, w2), w5 = cmul(w1, w4), w6 = cmul(w2, w4), w7 = cmul(w3, w4);
    v[1] = cmul(v[1], w1);
    v[2] = cmul(v[2], w2);
    v[3] = cmul(v[3], w3);
    v[4] = cmul(v[4], w4);
    v[5] = cmul(v[5], w5);
    v[6] = cmul(v[6], w6);
    v[7] = cmul(v[7], w7);
    v[8] = cmul(v[8], w8);
    v[9] = cmul(v[9], cmul(w1, w8));
    v[10] = cmul(v[10], cmul(w2, w8));
    v[11] = cmul(v[11], cmul(w3, w8));
    v[12] = cmul(v[12], cmul(w4, w8));
    v[13] = cmul(v[13], cmul(w5, w8));
    v[14] = cmul(v[14], cmul(w6, w8));
    v[15] = cmul(v[15], cmul(w7, w8));
}

__global__ void __launch_bounds__(R16::NT, 2) psd_stage_kernel_r16(const StageParams p)
{
    constexpr int N = R16::N, M = R16::M, TPS = R16::TPS, NT = R16::NT, G = R16::G, K = R16::K, WS = R16::WS;
    extern __shared__ __align__(16) float smem[];
    float* tile = smem;
    float* wsb = smem + p.tile_cap;
    float* wgt = wsb + G * 2 * WS;
    float* red = wgt + ((p.T + 3) & ~3);

    const int tid = threadIdx.x;
    const int group = tid / TPS;
    const int j = tid % TPS;
    const int hop = p.hop;
    const int seg0 = blockIdx.x * p.T;
    const int ns = min(p.T, p.nseg - seg0);
    const long long g0 = (p.k0 + seg0) * (long long)hop;
    const int tile_len = (ns - 1) * hop + N;

    for (int v = tid; v < tile_len / 4; v += NT)
        reinterpret_cast<float4*>(tile)[v] = ld_stream4(p.src, g0 + 4ll * v);

    if (tid < ns) wgt[tid] = ewma_weight(p, seg0 + tid);

    // ---- segment-invariant per-thread constants ----
    // the window is re-read through L1 for every segment (16 LDG.64): with the arithmetic on aligned
    // register pairs, 32 registers of window values no longer fit without spilling
    const float2* __restrict__ win2 = reinterpret_cast<const float2*>(p.win) + j;
    // pass-0 twiddles W_M^(j t): bases t = 1, 2, 4, 8
    const float2 a1 = __ldg(&p.twM[j]), a2 = __ldg(&p.twM[2 * j]), a4 = __ldg(&p.twM[4 * j]), a8 = __ldg(&p.twM[8 * j]);
    // pass-1 twiddles W_128^(o t) = W_M^(16 o t), o = j % 8
    const int o = j & 7;
    const float2 b1 = __ldg(&p.twM[16 * o]), b2 = __ldg(&p.twM[32 * o]), b4 = __ldg(&p.twM[64 * o]),
                 b8 = __ldg(&p.twM[128 * o]);
    // last pass: butterflies qA, qB (position digits q = 16 k0 + k1, frequency k_low = k0 + 16 k1)
    const int qA = 16 * (j >> 3) + (j & 7);
    const int kA = (j >> 3) + 16 * (j & 7);
    const int kB = K - kA;
    const int qB = (j == 0) ? 8 : (16 * (kB & 15) + (kB >> 4));
    const int posA = r16_pos(8 * qA), posB = r16_pos(8 * qB);
    const float2 w0 = __ldg(&p.twN[kA]);
    const float2 w32 = __ldg(&p.twN[128]);  // W_N^128 = W_32^1 (thread 0 only)
    // pass-1 addressing
    const int base1 = ((j >> 3) << 7) + o;
    const int pos1 = r16_pos(base1);
    const int pos0 = r16_pos(j);

    float* wre = wsb + group * 2 * WS;
    float* wim = wre + WS;
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.f;
    float accx = 0.f;

    __syncthreads();

    const int iters = (ns + G - 1) / G;
    for (int it = 0; it < iters; ++it) {
        const int s = it * G + group;
        const bool valid = s < ns;
        const int sc = valid ? s : ns - 1;
        const float* seg = tile + sc * hop;
        const float wseg = valid ? wgt[sc] : 0.f;

        // ---- pass 0: z[n] = x[2n] + i x[2n+1], n = j + 128 t; detrend; window; radix 16 ----
        float2 v[16];
#pragma unroll
        for (int t = 0; t < 16; ++t) v[t] = *reinterpret_cast<const float2*>(seg + 2 * (j + t * TPS));

        if (p.detrend == 1) {
            float off = seg[N / 2];
#pragma unroll
            for (int t = 0; t < 16; ++t) v[t] = __fadd2_rn(v[t], make_float2(-off, -off));
        } else if (p.detrend == 2) {
            float x0 = seg[0];
            float slope = (seg[N - 1] - x0) / (float)(N - 1);
#pragma unroll
            for (int t = 0; t < 16; ++t) {
                float n0 = (float)(2 * (j + t * TPS));
                v[t].x -= fmaf(slope, n0, x0);
                v[t].y -= fmaf(slope, n0 + 1.f, x0);
            }
        } else if (p.detrend == 3) {
            float sum = 0.f;
#pragma unroll
            for (int t = 0; t < 16; ++t) sum += v[t].x + v[t].y;
#pragma unroll
            for (int m = 16; m > 0; m >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, m);
            constexpr int WPG = TPS / 32;
            if ((tid & 31) == 0) red[group * WPG + (j >> 5)] = sum;
            group_sync<TPS, NT>(group);
            sum = 0.f;
#pragma unroll
            for (int w = 0; w < WPG; ++w) sum += red[group * WPG + w];
            float off = sum * (1.0f / (float)N);
#pragma unroll
            for (int t = 0; t < 16; ++t) v[t] = __fadd2_rn(v[t], make_float2(-off, -off));
        }
#pragma unroll
        for (int t = 0; t < 16; ++t) v[t] = __fmul2_rn(v[t], __ldg(win2 + t * TPS));

        dft16(v);
        twiddle16(v, a1, a2, a4, a8);
#pragma unroll
        for (int t = 0; t < 16; ++t) {
            // L(j + 128 t) = L(j) + t * (128 + 16 + 8)
            wre[pos0 + t * 152] = v[t].x;
            wim[pos0 + t * 152] = v[t].y;
        }
        group_sync<TPS, NT>(group);

        // ---- pass 1: radix 16 on 128 b + o + 8 t ----
#pragma unroll
        for (int t = 0; t < 16; ++t) {
            // L(base + 8 t) = L(base) + 8 t + 4 * ((8 t) >> 5)
            const int a = pos1 + 8 * t + 4 * ((8 * t) >> 5);
            v[t] = make_float2(wre[a], wim[a]);
        }
        dft16(v);
        twiddle16(v, b1, b2, b4, b8);
#pragma unroll
        for (int t = 0; t < 16; ++t) {
            const int a = pos1 + 8 * t + 4 * ((8 * t) >> 5);
            wre[a] = v[t].x;
            wim[a] = v[t].y;
        }
        group_sync<TPS, NT>(group);

        // ---- last pass: radix 8 on contiguous points, real-input split, |X|^2 ----
        float4 ar0 = *reinterpret_cast<const float4*>(wre + posA), ar1 = *reinterpret_cast<const float4*>(wre + posA + 4);
        float4 ai0 = *reinterpret_cast<const float4*>(wim + posA), ai1 = *reinterpret_cast<const float4*>(wim + posA + 4);
        float4 br0 = *reinterpret_cast<const float4*>(wre + posB), br1 = *reinterpret_cast<const float4*>(wre + posB + 4);
        float4 bi0 = *reinterpret_cast<const float4*>(wim + posB), bi1 = *reinterpret_cast<const float4*>(wim + posB + 4);
        group_sync<TPS, NT>(group);  // workspace may be overwritten by the next segment from here on

        float2 za[8], zb[8];
        dft8_planes(ar0, ar1, ai0, ai1, za);
        dft8_planes(br0, br1, bi0, bi1, zb);

        constexpr float h = 0.70710678118654752440f;
        constexpr float c1 = 0.92387953251128675613f, s1 = 0.38268343236508977173f;
        // W_16^t, t = 0..7
        constexpr float wr16[8] = {1.f, c1, h, s1, 0.f, -s1, -h, -c1};
        constexpr float wi16[8] = {0.f, -s1, -h, -c1, -1.f, -c1, -h, -s1};
        float pk, pm;
        if (j != 0) {
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                split_power(za[t], zb[7 - t], cmulc(w0, wr16[t], wi16[t]), pk, pm);
                acc[2 * t] = fmaf(wseg, pk, acc[2 * t]);
                acc[2 * t + 1] = fmaf(wseg, pm, acc[2 * t + 1]);
            }
        } else {
            // butterfly 0 (k = 256 t) and butterfly 8 (k = 128 + 256 t) pair with themselves
            split_power(za[0], za[0], make_float2(1.f, 0.f), pk, pm);  // bins 0 and M
            acc[0] = fmaf(wseg, pk, acc[0]);
            acc[1] = fmaf(wseg, pm, acc[1]);
#pragma unroll
            for (int t = 1; t < 4; ++t) {  // bins 256 t and M - 256 t
                split_power(za[t], za[8 - t], make_float2(wr16[t], wi16[t]), pk, pm);
                acc[2 * t] = fmaf(wseg, pk, acc[2 * t]);
                acc[2 * t + 1] = fmaf(wseg, pm, acc[2 * t + 1]);
            }
            split_power(za[4], za[4], make_float2(0.f, -1.f), pk, pm);  // bin M/2, once
            accx = fmaf(wseg, pk, accx);
#pragma unroll
            for (int u = 0; u < 4; ++u) {  // bins 128 + 256 u and M - 128 - 256 u
                split_power(zb[u], zb[7 - u], cmulc(w32, wr16[u], wi16[u]), pk, pm);
                acc[8 + 2 * u] = fmaf(wseg, pk, acc[8 + 2 * u]);
                acc[9 + 2 * u] = fmaf(wseg, pm, acc[9 + 2 * u]);
            }
        }
    }

    const AccSink sink = acc_sink(nullptr, p.acc, p.part, p.part_stride, blockIdx.x * G + group);
    if (j != 0) {
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            int k = kA + K * t;
            sink.add(k, acc[2 * t]);
            sink.add(M - k, acc[2 * t + 1]);
        }
    } else {
        sink.add(0, acc[0]);
        sink.add(M, acc[1]);
#pragma unroll
        for (int t = 1; t < 4; ++t) {
            sink.add(K * t, acc[2 * t]);
            sink.add(M - K * t, acc[2 * t + 1]);
        }
        sink.add(M / 2, accx);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            sink.add(K / 2 + K * u, acc[8 + 2 * u]);
            sink.add(M - K / 2 - K * u, acc[9 + 2 * u]);
        }
    }
}

inline size_t stage_r16_smem_bytes(int T, int hop)
{
    size_t tile = (size_t)(T - 1) * hop + R16::N;
    size_t fl = tile + (size_t)R16::G * 2 * R16::WS + ((T + 3) & ~3) + (size_t)R16::G * (R16::TPS / 32);
    return fl * sizeof(float);
}

}  // namespace sspsd
