// sspsd_stage_kernel_ring.cuh -- K2 for N = 4096, third generation: persistent CTAs streaming
// through a contiguous range of segments with a shared-memory ring of hop slots filled by TMA bulk
// copies (cp.async.bulk + mbarrier complete_tx), so that the HBM latency of hop h+3.. is hidden behind
// the FFTs of hop h (profiles/r01_ncu_summary.md: after the radix-16 rewrite the top stall of the
// tiled kernel was long_scoreboard = the synchronous tile load at every CTA start).
//
// The transform itself (radix 16/16/8, split re/im planes, in-register real-input split and |X|^2)
// is the one of sspsd_stage_kernel_r16.cuh.  New here:
//   * one CTA owns segments [c0, c1) of the launch; its two 128-thread groups take alternate
//     segments; segment s needs hops s and s+1, a hop (N/2 samples) is loaded exactly once per CTA;
//   * ring of RING hop slots; one elected thread issues the bulk copies (two per hop when the hop
//     straddles the carry/fresh boundary of the stage's StreamSrc) and arms the slot's mbarrier
//     with the byte count; consumers wait on the slot's phase parity;
//   * a slot is refilled only after a CTA-wide barrier that follows the last read of the hop;
//   * |X|^2 accumulators stay in registers for the CTA's whole range: one atomicAdd per bin per
//     thread per launch (296 CTAs) instead of per tile.
#pragma once
#include "sspsd_stage_kernel_r16.cuh"

namespace sspsd {

struct RingCfg {
    static constexpr int RING = 6;        // hop slots (8 KiB each at N = 4096)
    static constexpr int RING1 = 4;       // single-group variant: hops s, s + 1 in use, two in flight
    static constexpr int MAX_W = 2048;    // per-CTA weight table (segments per CTA upper bound)
};

// G = 128-thread groups (segments in flight) per CTA, RING = hop slots, WIN_SMEM = window table in shared memory (else
// re-read through L1 with LDG.64: the table is 16 KiB per CTA, too much for four single-group CTAs per SM)
template <int G, int RING, bool WIN_SMEM>
__device__ __forceinline__ void psd_stage_ring_body(const StageParams& p)
{
    constexpr int N = R16::N, M = R16::M, TPS = R16::TPS, NT = TPS * G, K = R16::K, WS = R16::WS;
    constexpr int HOP = N / 2;  // Hann; the rectangular window uses the tiled kernel
    extern __shared__ __align__(16) float smem[];
    float* ring = smem;                      // RING * HOP
    float2* wtab = reinterpret_cast<float2*>(ring + RING * HOP);  // the window as N/2 pairs (16 KiB), if WIN_SMEM
    float* wsb = ring + RING * HOP + (WIN_SMEM ? N : 0);      // G * 2 * WS
    float* wgt = wsb + G * 2 * WS;           // p.T entries (segments per CTA)
    float* red = wgt + ((p.T + 3) & ~3);     // G * 4
    uint64_t* bars = reinterpret_cast<uint64_t*>(red + 8);  // RING mbarriers (8-byte aligned: all counts above are even)

    const int tid = threadIdx.x;
    const int group = tid / TPS;
    const int j = tid % TPS;
    // this CTA's segments [c0, c1) of the launch; p.T = segments per CTA
    const int c0 = blockIdx.x * p.T;
    const int ns = min(p.T, p.nseg - c0);
    const long long g0 = (p.k0 + c0) * (long long)HOP;  // stream index of hop 0 of this CTA
    const int nhops = ns + 1;

    if (tid == 0) {
#pragma unroll
        for (int r = 0; r < RING; ++r) mbar_init(&bars[r], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        const int pre = nhops < RING ? nhops : RING;
        for (int h = 0; h < pre; ++h) ring_issue(p.src, g0 + (long long)h * HOP, HOP, ring + h * HOP, &bars[h]);
    }

    for (int i = tid; i < ns; i += NT) wgt[i] = ewma_weight(p, c0 + i);

    // ---- segment-invariant per-thread constants (as in the tiled radix-16 kernel) ----
    // the window lives in shared memory (one LDS.64 per point and segment): the packed arithmetic needs
    // aligned register pairs, and 32 registers of window values no longer fit beside it
    if constexpr (WIN_SMEM)
        for (int i = tid; i < N / 2; i += NT) wtab[i] = __ldg(reinterpret_cast<const float2*>(p.win) + i);
    const float2* __restrict__ gwin = reinterpret_cast<const float2*>(p.win);
    const float2 a1 = __ldg(&p.twM[j]), a2 = __ldg(&p.twM[2 * j]), a4 = __ldg(&p.twM[4 * j]), a8 = __ldg(&p.twM[8 * j]);
    const int o = j & 7;
    const float2 b1 = __ldg(&p.twM[16 * o]), b2 = __ldg(&p.twM[32 * o]), b4 = __ldg(&p.twM[64 * o]),
                 b8 = __ldg(&p.twM[128 * o]);
    const int qA = 16 * (j >> 3) + (j & 7);
    const int kA = (j >> 3) + 16 * (j & 7);
    const int kB = K - kA;
    const int qB = (j == 0) ? 8 : (16 * (kB & 15) + (kB >> 4));
    const int posA = r16_pos(8 * qA), posB = r16_pos(8 * qB);
    const float2 w0 = __ldg(&p.twN[kA]);
    const float2 w32 = __ldg(&p.twN[128]);
    const int pos1 = r16_pos(((j >> 3) << 7) + o);
    const int pos0 = r16_pos(j);

    float* wre = wsb + group * 2 * WS;
    float* wim = wre + WS;
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.f;
    float accx = 0.f;

    __syncthreads();  // weight table visible

    const int iters = (ns + G - 1) / G;
    for (int it = 0; it < iters; ++it) {
        const int s = it * G + group;
        const bool valid = s < ns;
        const int sc = valid ? s : ns - 1;
        const float wseg = valid ? wgt[sc] : 0.f;
        // hops sc and sc + 1
        const int hA = sc, hB = sc + 1;
        const int slA = hA % RING, slB = hB % RING;
        mbar_wait(&bars[slA], (uint32_t)(hA / RING) & 1u);
        mbar_wait(&bars[slB], (uint32_t)(hB / RING) & 1u);
        const float* sA = ring + slA * HOP;
        const float* sB = ring + slB * HOP;

        // ---- pass 0: points n = j + 128 t; t < 8 lies in hop A, t >= 8 in hop B ----
        float2 v[16];
#pragma unroll
        for (int t = 0; t < 8; ++t) v[t] = *reinterpret_cast<const float2*>(sA + 2 * (j + t * TPS));
#pragma unroll
        for (int t = 8; t < 16; ++t) v[t] = *reinterpret_cast<const float2*>(sB + 2 * (j + (t - 8) * TPS));

        if (p.detrend == 1) {
            float off = sB[0];  // x[N/2]
#pragma unroll
            for (int t = 0; t < 16; ++t) v[t] = __fadd2_rn(v[t], make_float2(-off, -off));
        } else if (p.detrend == 2) {
            float x0 = sA[0];
            float slope = (sB[HOP - 1] - x0) / (float)(N - 1);
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
        for (int t = 0; t < 16; ++t) v[t] = __fmul2_rn(v[t], WIN_SMEM ? wtab[j + t * TPS] : __ldg(gwin + j + t * TPS));

        dft16(v);
        twiddle16(v, a1, a2, a4, a8);
#pragma unroll
        for (int t = 0; t < 16; ++t) {
            wre[pos0 + t * 152] = v[t].x;
            wim[pos0 + t * 152] = v[t].y;
        }
        group_sync<TPS, NT>(group);

        // ---- pass 1 ----
#pragma unroll
        for (int t = 0; t < 16; ++t) {
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

        // ---- last pass ----
        float4 ar0 = *reinterpret_cast<const float4*>(wre + posA), ar1 = *reinterpret_cast<const float4*>(wre + posA + 4);
        float4 ai0 = *reinterpret_cast<const float4*>(wim + posA), ai1 = *reinterpret_cast<const float4*>(wim + posA + 4);
        float4 br0 = *reinterpret_cast<const float4*>(wre + posB), br1 = *reinterpret_cast<const float4*>(wre + posB + 4);
        float4 bi0 = *reinterpret_cast<const float4*>(wim + posB), bi1 = *reinterpret_cast<const float4*>(wim + posB + 4);

        // CTA-wide: both groups are done with hops 2 it and 2 it + 1 (and with their workspaces)
        __syncthreads();
        if (tid == 0) {
            // refill the two slots just released with hops 2 it + RING, 2 it + RING + 1
#pragma unroll
            for (int d = 0; d < G; ++d) {
                const int h = it * G + d + RING;
                if (h < nhops) ring_issue(p.src, g0 + (long long)h * HOP, HOP, ring + (h % RING) * HOP, &bars[h % RING]);
            }
        }

        float2 za[8], zb[8];
        dft8_planes(ar0, ar1, ai0, ai1, za);
        dft8_planes(br0, br1, bi0, bi1, zb);

        constexpr float h = 0.70710678118654752440f;
        constexpr float c1 = 0.92387953251128675613f, s1 = 0.38268343236508977173f;
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
            split_power(za[0], za[0], make_float2(1.f, 0.f), pk, pm);
            acc[0] = fmaf(wseg, pk, acc[0]);
            acc[1] = fmaf(wseg, pm, acc[1]);
#pragma unroll
            for (int t = 1; t < 4; ++t) {
                split_power(za[t], za[8 - t], make_float2(wr16[t], wi16[t]), pk, pm);
                acc[2 * t] = fmaf(wseg, pk, acc[2 * t]);
                acc[2 * t + 1] = fmaf(wseg, pm, acc[2 * t + 1]);
            }
            split_power(za[4], za[4], make_float2(0.f, -1.f), pk, pm);
            accx = fmaf(wseg, pk, accx);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
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

// default: two groups per CTA, two CTAs per SM, window in shared memory
__global__ void __launch_bounds__(R16::NT, 2) psd_stage_kernel_ring(const StageParams p)
{
    psd_stage_ring_body<R16::G, RingCfg::RING, true>(p);
}

// variant (SSPSD_K2=ring1): four independent single-group CTAs per SM -- no CTA-wide barrier couples two groups, the
// groups of an SM drift apart freely; 3-slot ring, window through L1
__global__ void __launch_bounds__(R16::TPS, 4) psd_stage_kernel_ring1(const StageParams p)
{
    psd_stage_ring_body<1, RingCfg::RING1, false>(p);
}

// variant (SSPSD_K2=ring1x5): five single-group CTAs per SM (20 warps instead of 16) at <= 96 registers, 3-slot ring
__global__ void __launch_bounds__(R16::TPS, 5) psd_stage_kernel_ring1x5(const StageParams p)
{
    psd_stage_ring_body<1, 3, false>(p);
}

inline size_t stage_ring_smem_bytes(int segs_per_cta, int groups = R16::G, int ring = RingCfg::RING, bool win_smem = true)
{
    size_t fl = (size_t)ring * (R16::N / 2) + (win_smem ? R16::N : 0) + (size_t)groups * 2 * R16::WS + ((segs_per_cta + 3) & ~3) + 8;
    return fl * sizeof(float) + ring * sizeof(uint64_t) + 16;
}

}  // namespace sspsd
