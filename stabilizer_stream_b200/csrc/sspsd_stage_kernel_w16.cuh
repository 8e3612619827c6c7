// sspsd_stage_kernel_w16.cuh -- K2 for N = 512 with the Hann window: the FFT size every binary of the reference
// instantiates (PsdCascade::<{1 << 9}>, src/bin/psd.rs:176, src/bin/stream_test.rs:40, src/psd.rs:554, 614).
//
// Same contract as psd_stage_kernel<9> (sspsd_stage_kernel.cuh; reference src/psd.rs:210-233), restructured around
// the warp:
//   * a segment (M = 256 complex points z[n] = x[2n] + i x[2n+1]) belongs to HALF a warp: 16 lanes x 16 points,
//     M = 16 x 16, i.e. two radix-16 passes in registers with ONE transposition between them (the generic kernel
//     uses 32 lanes x 8 points and radix 8 / 8 / 4: two exchanges and a third shared-memory round for the last
//     pass); the transposition goes through a padded per-half-warp tile in shared memory, ordered by __syncwarp
//     only -- there is no block barrier anywhere in the transform;
//   * after the second pass lane l holds Z[l + 16 k1]; the real-input split pairs bin k with M - k, which lives in
//     lane (16 - l) & 15, register 15 - k1: the partner's upper eight values arrive by warp shuffles
//     (shfl.sync), lanes 0 and 8 are their own partners, and every lane ends up owning 16 of the 257 bins;
//   * persistent CTAs over a contiguous range of segments with a ring of 4096-sample chunks (16 hops) filled by
//     TMA bulk copies, as in the N = 4096 ring kernel: one block barrier per 16 segments, for the refill only;
//   * |X|^2 stays in registers for the CTA's whole range; Mean detrend sums with xor-shuffles inside the half warp.
#pragma once
#include "sspsd_stage_kernel_r16.cuh"

namespace sspsd {

struct W16 {
    static constexpr int N = 512, M = 256, HOP = 256;
    static constexpr int NT = 256;               // threads per CTA: 8 warps = 16 segments per iteration
    static constexpr int SPI = 16;               // segments per iteration
    static constexpr int CHUNK = SPI * HOP;      // samples per ring slot (16 KiB)
    static constexpr int RING = 3;               // chunks it and it + 1 are in use, chunk it + 2 is in flight
    static constexpr int XROW = 17;              // padded row length (float2) of the 16 x 16 transposition tile
    static constexpr int XT = 16 * XROW;         // float2 per half-warp tile
    static constexpr int MAX_T = 4096;           // segments per CTA (weight table)
};

__global__ void __launch_bounds__(W16::NT, 2) psd_stage_kernel_w16(const StageParams p)
{
    constexpr int N = W16::N, M = W16::M, HOP = W16::HOP, NT = W16::NT, SPI = W16::SPI, CHUNK = W16::CHUNK,
                  RING = W16::RING, XROW = W16::XROW, XT = W16::XT;
    extern __shared__ __align__(16) float smem[];
    float* ring = smem;                                              // RING * CHUNK
    float2* wtab = reinterpret_cast<float2*>(ring + RING * CHUNK);   // window as M pairs (2 KiB)
    float2* xch = wtab + M;                                          // SPI tiles of XT float2
    float* wgt = reinterpret_cast<float*>(xch + SPI * XT);           // p.T weights
    uint64_t* bars = reinterpret_cast<uint64_t*>(wgt + ((p.T + 3) & ~3));

    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    const int half = lane >> 4, l = lane & 15;
    const int q = 2 * warp + half;  // segment slot of this half warp within an iteration
    const int c0 = blockIdx.x * p.T;
    const int ns = min(p.T, p.nseg - c0);
    const long long g0 = (p.k0 + c0) * (long long)HOP;
    const int nsamp = (ns + 1) * HOP;                    // samples this CTA reads
    const int nchunks = (nsamp + CHUNK - 1) / CHUNK;
    auto issue = [&](int c) {
        const int len = min(CHUNK, nsamp - c * CHUNK);
        ring_issue(p.src, g0 + (long long)c * CHUNK, len, ring + (c % RING) * CHUNK, &bars[c % RING]);
    };
    if (tid == 0) {
#pragma unroll
        for (int r = 0; r < RING; ++r) mbar_init(&bars[r], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0)
        for (int c = 0; c < min(nchunks, RING); ++c) issue(c);

    for (int i = tid; i < ns; i += NT) wgt[i] = ewma_weight(p, c0 + i);
    for (int i = tid; i < M; i += NT) wtab[i] = __ldg(reinterpret_cast<const float2*>(p.win) + i);

    // ---- segment-invariant per-lane constants ----
    // pass-0 twiddles W_256^(l t): bases t = 1, 2, 4, 8 (p.twM[q] = exp(-2 pi i q / M))
    const float2 a1 = __ldg(&p.twM[l]), a2 = __ldg(&p.twM[2 * l]), a4 = __ldg(&p.twM[4 * l]), a8 = __ldg(&p.twM[8 * l]);
    const float2 w0 = __ldg(&p.twN[l]);  // W_512^l; bin k = l + 16 k1 uses W_512^k = w0 * W_32^k1
    const int src_lane = (half << 4) | ((16 - l) & 15);
    float2* xw = xch + q * XT;
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.f;
    float accx = 0.f;

    __syncthreads();  // weight + window tables visible

    const int iters = (ns + SPI - 1) / SPI;
    for (int it = 0; it < iters; ++it) {
        const int s = it * SPI + q;
        const bool valid = s < ns;
        const int qc = valid ? q : (ns - 1 - it * SPI);   // an invalid slot re-reads the CTA's last segment with weight 0
        const float wseg = valid ? wgt[it * SPI + qc] : 0.f;
        mbar_wait(&bars[it % RING], (uint32_t)(it / RING) & 1u);
        if (it + 1 < nchunks) mbar_wait(&bars[(it + 1) % RING], (uint32_t)((it + 1) / RING) & 1u);
        const float* sA = ring + (it % RING) * CHUNK + qc * HOP;
        const float* sB = qc < SPI - 1 ? sA + HOP : ring + ((it + 1) % RING) * CHUNK;

        // ---- pass 0: points n = l + 16 t; t < 8 lies in hop A, t >= 8 in hop B ----
        float2 v[16];
#pragma unroll
        for (int t = 0; t < 8; ++t) v[t] = *reinterpret_cast<const float2*>(sA + 2 * (l + 16 * t));
#pragma unroll
        for (int t = 8; t < 16; ++t) v[t] = *reinterpret_cast<const float2*>(sB + 2 * (l + 16 * (t - 8)));

        if (p.detrend == 1) {  // Midpoint, psd.rs:87-93
            const float off = sB[0];
#pragma unroll
            for (int t = 0; t < 16; ++t) v[t] = __fadd2_rn(v[t], make_float2(-off, -off));
        } else if (p.detrend == 2) {  // Span, psd.rs:94-102
            const float x0 = sA[0];
            const float slope = (sB[HOP - 1] - x0) / (float)(N - 1);
#pragma unroll
            for (int t = 0; t < 16; ++t) {
                const float n0 = (float)(2 * (l + 16 * t));
                v[t].x -= fmaf(slope, n0, x0);
                v[t].y -= fmaf(slope, n0 + 1.f, x0);
            }
        } else if (p.detrend == 3) {  // Mean, psd.rs:103-109
            float sum = 0.f;
#pragma unroll
            for (int t = 0; t < 16; ++t) sum += v[t].x + v[t].y;
#pragma unroll
            for (int m = 8; m > 0; m >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, m);  // stays inside the half warp
            const float off = sum * (1.0f / (float)N);
#pragma unroll
            for (int t = 0; t < 16; ++t) v[t] = __fadd2_rn(v[t], make_float2(-off, -off));
        }
#pragma unroll
        for (int t = 0; t < 16; ++t) v[t] = __fmul2_rn(v[t], wtab[l + 16 * t]);

        dft16(v);
        twiddle16(v, a1, a2, a4, a8);

        // ---- transposition inside the half warp: (k2 in registers, n1 in lanes) -> (n1 in registers, k2 in lanes) ----
#pragma unroll
        for (int t = 0; t < 16; ++t) xw[t * XROW + l] = v[t];
        __syncwarp();
#pragma unroll
        for (int t = 0; t < 16; ++t) v[t] = xw[l * XROW + t];
        __syncwarp();  // the tile may be overwritten by the next iteration from here on

        // ---- pass 1: v[k1] = Z[l + 16 k1] ----
        dft16(v);

        // ---- real-input split: Z[M - k] for k = l + 16 k1 (k1 < 8) is register 15 - k1 of lane (16 - l) & 15; lane 0
        // is its own partner with register (16 - k1) & 15.  The sender picks what its receiver needs. ----
        float2 zm[8];
#pragma unroll
        for (int k1 = 0; k1 < 8; ++k1) {
            const float2 snd = (l == 0) ? v[(16 - k1) & 15] : v[15 - k1];
            zm[k1].x = __shfl_sync(0xffffffffu, snd.x, src_lane);
            zm[k1].y = __shfl_sync(0xffffffffu, snd.y, src_lane);
        }
        // W_32^k1, k1 = 0..7
        constexpr float c1 = 0.98078528040323044913f, s1 = 0.19509032201612826785f;
        constexpr float c2 = 0.92387953251128675613f, s2 = 0.38268343236508977173f;
        constexpr float c3 = 0.83146961230254523708f, s3 = 0.55557023301960222474f;
        constexpr float h = 0.70710678118654752440f;
        constexpr float wr32[8] = {1.f, c1, c2, c3, h, s3, s2, s1};
        constexpr float wi32[8] = {0.f, -s1, -s2, -s3, -h, -c3, -c2, -c1};
        float pk, pm;
#pragma unroll
        for (int k1 = 0; k1 < 8; ++k1) {
            split_power(v[k1], zm[k1], cmulc(w0, wr32[k1], wi32[k1]), pk, pm);
            acc[2 * k1] = fmaf(wseg, pk, acc[2 * k1]);
            acc[2 * k1 + 1] = fmaf(wseg, pm, acc[2 * k1 + 1]);
        }
        // bin M / 2 = 128 pairs with itself: lane 0, register 8 (computed by every lane, kept by lane 0)
        split_power(v[8], v[8], make_float2(0.f, -1.f), pk, pm);
        accx = fmaf(wseg, pk, accx);

        // every warp is done with chunk `it` (chunk it + 1 stays in use): refill its slot
        __syncthreads();
        if (tid == 0 && it + RING < nchunks) issue(it + RING);
    }

    // ---- flush: lane l owns bins l + 16 k1 and M - (l + 16 k1), k1 < 8; lane 0 also bin M / 2 ----
    const AccSink sink = acc_sink(nullptr, p.acc, p.part, p.part_stride, blockIdx.x * SPI + q);
#pragma unroll
    for (int k1 = 0; k1 < 8; ++k1) {
        const int k = l + 16 * k1;
        sink.add(k, acc[2 * k1]);
        sink.add(M - k, acc[2 * k1 + 1]);
    }
    if (l == 0) sink.add(M / 2, accx);
}

inline size_t stage_w16_smem_bytes(int segs_per_cta)
{
    size_t fl = (size_t)W16::RING * W16::CHUNK + 2 * (size_t)W16::M + 2 * (size_t)W16::SPI * W16::XT + ((segs_per_cta + 3) & ~3);
    return fl * sizeof(float) + W16::RING * sizeof(uint64_t) + 16;
}

}  // namespace sspsd
