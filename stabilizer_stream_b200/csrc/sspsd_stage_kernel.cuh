// sspsd_stage_kernel.cuh -- K2: fused detrend + window + real FFT + |X|^2 accumulate for one
// PSD stage (reference src/psd.rs:210-233, one iteration of the `while` loop per segment).
//
// Generic version for N = 64 ... 8192 (N = 4096 has its own kernels).  A persistent CTA walks over a
// contiguous range of tiles; a tile is `T` consecutive hops (+ the overlap) of the stage's stream,
// brought into one of two shared-memory buffers by TMA bulk copies (every sample crosses HBM once; the
// 50 % overlap is served from shared memory; tile t+1 streams in while tile t is transformed).  The
// segments of a tile are transformed by groups of TPS = N/16 threads.  |X|^2 is accumulated in
// registers over ALL tiles of the CTA (each thread owns the same 8 bins for every segment) and
// flushed with one atomicAdd per bin per thread at the end.
#pragma once
#include "sspsd_device.cuh"

namespace sspsd {

struct StageParams {
    StreamSrc src;
    long long k0;      // global index of the first segment of this launch
    int nseg;          // segments in this launch
    int T;             // segments per tile (ring kernel: segments per CTA)
    int tpc;           // tiles per CTA (persistent tiled kernel)
    int hop;           // N - overlap
    int detrend;       // SSPSD_DETREND_*
    int tile_cap;      // floats reserved for the tile in shared memory
    const float* win;  // N window values
    const float2* twM; // M entries: exp(-2 pi i q / M)
    const float2* twN; // M entries: exp(-2 pi i k / N)
    float* acc;        // N/2+1 accumulators of this stage
    float* part;       // deterministic mode: per-(CTA, group) partial rows of part_stride floats (else nullptr)
    int part_stride;
    // EWMA weights (psd.rs:218-233): segment j of this launch is scaled by
    //   g_s^(nseg-1-max(j,jb)) * (j < jb && jb < nseg ? g_first : 1);  boxcar: jb >= nseg
    int jb;
    float g_first;
    float g_s;
};

// Flush of a thread's register accumulators.  Default: one atomicAdd per owned bin (order of the ~300 CTAs is
// arbitrary, so the f32 sum is not bit-reproducible from run to run).  Deterministic mode (SURVEY.md App. D):
// every (CTA, group) writes its own partial row -- each bin of a row has exactly one owner thread -- and
// reduce_partials_kernel adds the rows to the accumulator in row order.
struct AccSink {
    float* acc;
    float* row;  // nullptr: atomics
    __device__ __forceinline__ void add(int k, float v) const
    {
        if (row)
            row[k] = v;
        else
            atomicAdd(&acc[k], v);
    }
};
__device__ __forceinline__ AccSink acc_sink(const float* /*unused*/, float* acc, float* part, int part_stride, int row_index)
{
    return AccSink{acc, part ? part + (size_t)row_index * part_stride : nullptr};
}

// acc[k] += sum over rows (in row order, f64) of part[r][k]  (internal linkage: included by more than one unit)
static __global__ void reduce_partials_kernel(float* __restrict__ acc, const float* __restrict__ part, int nrows, int stride, int nbins)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nbins) return;
    double s = 0.0;
    for (int r = 0; r < nrows; ++r) s += (double)part[(size_t)r * stride + k];
    acc[k] = (float)((double)acc[k] + s);
}

// acc[i] *= s (EWMA rescale of the running average before a batch, psd.rs:218-232; internal linkage as above)
static __global__ void scale_kernel(float* __restrict__ acc, int n, float s)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
        acc[i] *= s;
}

template <int TPS, int NT>
__device__ __forceinline__ void group_sync(int group)
{
    if constexpr (TPS >= NT) {
        __syncthreads();
    } else if constexpr (TPS <= 32) {
        __syncwarp();
    } else {
        asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "n"(TPS) : "memory");
    }
}

// |A2 + W B2|^2 and |A2 - W B2|^2 for the real-input split of the pair (k, M-k):
//   X[k] = (A2 + W B2)/2,  X[M-k] = conj(A2 - W B2)/2,  A2 = Zk + conj(Zm),  B2 = -i (Zk - conj(Zm))
__device__ __forceinline__ void split_power(float2 zk, float2 zm, float2 w, float& pk, float& pm)
{
    float2 a2 = __fadd2_rn(zk, make_float2(zm.x, -zm.y));   // Zk + conj(Zm)
    float2 d = __fadd2_rn(zk, make_float2(-zm.x, zm.y));    // Zk - conj(Zm)
    // W * (-i d) = w.x (d.y, -d.x) + w.y (d.x, d.y)
    float2 wb = __ffma2_rn(d, make_float2(w.y, w.y), __fmul2_rn(make_float2(d.y, -d.x), make_float2(w.x, w.x)));
    float2 s = cadd(a2, wb), t = csub(a2, wb);
    pk = fmaf(s.y, s.y, s.x * s.x);
    pm = fmaf(t.y, t.y, t.x * t.x);
}

template <int LOG2N, int PASS>
__device__ __forceinline__ void load_pass_twiddles(float2 (&tw)[Plan<LOG2N>::P - 1][7], const float2* __restrict__ twM, int j)
{
    using PL = Plan<LOG2N>;
    if constexpr (PASS < PL::P - 1) {
        constexpr int LR = PL::log2radix(PASS), R = 1 << LR;
        constexpr int LS = PL::log2stride(PASS), S = 1 << LS;
        constexpr int BPT = 8 / R;
#pragma unroll
        for (int u = 0; u < BPT; ++u) {
            int bf = j + u * PL::TPS;
            int o = bf & (S - 1);
#pragma unroll
            for (int t = 1; t < R; ++t)
                tw[PASS][u * (R - 1) + t - 1] = __ldg(&twM[(o * t) << (PL::LOG2M - LR - LS)]);
        }
        load_pass_twiddles<LOG2N, PASS + 1>(tw, twM, j);
    }
}

// passes 1 .. P-2: in place on the padded re/im planes, each followed by a group barrier
template <int LOG2N, int PASS>
__device__ __forceinline__ void mid_passes(float* __restrict__ wre, float* __restrict__ wim, int j, int group,
                                           const float2 (&tw)[Plan<LOG2N>::P - 1][7])
{
    using PL = Plan<LOG2N>;
    if constexpr (PASS < PL::P - 1) {
        constexpr int LR = PL::log2radix(PASS), R = 1 << LR;
        constexpr int LS = PL::log2stride(PASS), S = 1 << LS;
        constexpr int BPT = 8 / R;
#pragma unroll
        for (int u = 0; u < BPT; ++u) {
            int bf = j + u * PL::TPS;
            int o = bf & (S - 1);
            int base = ((bf >> LS) << (LR + LS)) + o;
            int a0 = ws_pos(base);
            float2 v[R];
#pragma unroll
            for (int t = 0; t < R; ++t) {
                int a = a0 + t * S + 4 * ((t * S) >> 5);
                v[t] = make_float2(wre[a], wim[a]);
            }
            butterfly<R>(v);
#pragma unroll
            for (int t = 0; t < R; ++t) {
                int a = a0 + t * S + 4 * ((t * S) >> 5);
                float2 y = t ? cmul(v[t], tw[PASS][u * (R - 1) + t - 1]) : v[0];
                wre[a] = y.x;
                wim[a] = y.y;
            }
        }
        group_sync<PL::TPS, PL::NT>(group);
        mid_passes<LOG2N, PASS + 1>(wre, wim, j, group, tw);
    }
}

template <int LOG2N>
__device__ __forceinline__ int klow_of_q(int q)
{
    using PL = Plan<LOG2N>;
    int k = 0;
#pragma unroll
    for (int p = 0; p < PL::P - 1; ++p) {
        int t = (q >> (PL::log2stride(p) - 2)) & ((1 << PL::log2radix(p)) - 1);
        k |= t << PL::log2weight(p);
    }
    return k;
}

template <int LOG2N>
__device__ __forceinline__ int q_of_klow(int k)
{
    using PL = Plan<LOG2N>;
    int q = 0;
#pragma unroll
    for (int p = 0; p < PL::P - 1; ++p) {
        int t = (k >> PL::log2weight(p)) & ((1 << PL::log2radix(p)) - 1);
        q |= t << (PL::log2stride(p) - 2);
    }
    return q;
}

template <int LOG2N>
__global__ void __launch_bounds__(Plan<LOG2N>::NT, Plan<LOG2N>::NT <= 256 ? 2 : 1)
psd_stage_kernel(const StageParams p)
{
    using PL = Plan<LOG2N>;
    constexpr int N = PL::N, M = PL::M, TPS = PL::TPS, NT = PL::NT, G = PL::G, K = PL::K, WS = PL::WS;
    extern __shared__ __align__(16) float smem[];
    float* tiles = smem;                       // 2 * p.tile_cap
    float* wsb = smem + 2 * p.tile_cap;
    float* wgt = wsb + G * 2 * WS;
    float* red = wgt + ((p.T + 3) & ~3);
    uint64_t* bars = reinterpret_cast<uint64_t*>(red + ((G * (TPS > 32 ? TPS / 32 : 1) + 1) & ~1));

    const int tid = threadIdx.x;
    const int group = tid / TPS;
    const int j = tid % TPS;
    const int hop = p.hop;
    const int ntiles = (p.nseg + p.T - 1) / p.T;
    const int tile0 = blockIdx.x * p.tpc;
    const int tile1 = min(tile0 + p.tpc, ntiles);

    auto issue_tile = [&](int tl) {
        const int s0 = tl * p.T;
        const int n_s = min(p.T, p.nseg - s0);
        const int b = (tl - tile0) & 1;
        ring_issue(p.src, (p.k0 + s0) * (long long)hop, (n_s - 1) * hop + N, tiles + b * p.tile_cap, &bars[b]);
    };
    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0 && tile0 < tile1) {
        issue_tile(tile0);
        if (tile0 + 1 < tile1) issue_tile(tile0 + 1);
    }

    // ---- segment-invariant per-thread constants ----
    float2 wv[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) wv[t] = __ldg(reinterpret_cast<const float2*>(p.win) + (j + t * TPS));
    float2 tw[PL::P - 1][7];
    load_pass_twiddles<LOG2N, 0>(tw, p.twM, j);

    // last pass: this thread owns butterflies qA and qB whose outputs pair up as (k, M-k)
    constexpr int RL = 1 << PL::log2radix(PL::P - 2);
    constexpr int HALF = RL / 2;
    const int qA = RL * (j / HALF) + (j % HALF);
    const int kA = klow_of_q<LOG2N>(qA);
    const int qB = (j == 0) ? HALF : q_of_klow<LOG2N>(K - kA);
    const int posA = ws_pos(4 * qA), posB = ws_pos(4 * qB);
    constexpr float h = 0.70710678118654752440f;
    float2 wp[4];
    {
        float2 w0 = __ldg(&p.twN[kA]); // exp(-2 pi i kA / N); times W_8^t for k = kA + K t
        wp[0] = w0;
        wp[1] = make_float2(h * (w0.x + w0.y), h * (w0.y - w0.x));
        wp[2] = make_float2(w0.y, -w0.x);
        wp[3] = make_float2(h * (w0.y - w0.x), -h * (w0.x + w0.y));
    }
    float2 w16a = make_float2(0.f, 0.f), w16b = make_float2(0.f, 0.f);
    if (j == 0) {
        w16a = __ldg(&p.twN[K / 2]);     // W_N^(K/2)
        w16b = __ldg(&p.twN[K / 2 + K]); // W_N^(K/2 + K)
    }

    float* wre = wsb + group * 2 * WS;
    float* wim = wre + WS;
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    float accx = 0.f;

    for (int tl = tile0; tl < tile1; ++tl) {
    const int buf = (tl - tile0) & 1;
    const int seg0 = tl * p.T;
    const int ns = min(p.T, p.nseg - seg0);
    const float* tile = tiles + buf * p.tile_cap;
    // per-segment averaging weights of this tile
    for (int i = tid; i < ns; i += NT) wgt[i] = ewma_weight(p, seg0 + i);
    mbar_wait(&bars[buf], (uint32_t)((tl - tile0) >> 1) & 1u);
    __syncthreads();

    const int iters = (ns + G - 1) / G;
    for (int it = 0; it < iters; ++it) {
        const int s = it * G + group;
        const bool valid = s < ns;
        const int sc = valid ? s : ns - 1;
        const float* seg = tile + sc * hop;
        const float wseg = valid ? wgt[sc] : 0.f;

        // ---- pass 0: read z[n] = x[2n] + i x[2n+1] from the tile, detrend, window ----
        float2 v[8];
#pragma unroll
        for (int t = 0; t < 8; ++t)
            v[t] = *reinterpret_cast<const float2*>(seg + 2 * (j + t * TPS));

        if (p.detrend == 1) { // Midpoint, psd.rs:87-93
            float off = seg[N / 2];
#pragma unroll
            for (int t = 0; t < 8; ++t) v[t] = __fadd2_rn(v[t], make_float2(-off, -off));
        } else if (p.detrend == 2) { // Span, psd.rs:94-102
            float x0 = seg[0];
            float slope = (seg[N - 1] - x0) / (float)(N - 1);
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                float n0 = (float)(2 * (j + t * TPS));
                v[t].x -= fmaf(slope, n0, x0);
                v[t].y -= fmaf(slope, n0 + 1.f, x0);
            }
        } else if (p.detrend == 3) { // Mean, psd.rs:103-109
            float sum = 0.f;
#pragma unroll
            for (int t = 0; t < 8; ++t) sum += v[t].x + v[t].y;
            if constexpr (TPS <= 32) {
#pragma unroll
                for (int m = TPS / 2; m > 0; m >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, m);
            } else {
#pragma unroll
                for (int m = 16; m > 0; m >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, m);
                constexpr int WPG = TPS / 32;
                if ((tid & 31) == 0) red[group * WPG + (j >> 5)] = sum;
                group_sync<TPS, NT>(group);
                sum = 0.f;
#pragma unroll
                for (int w = 0; w < WPG; ++w) sum += red[group * WPG + w];
            }
            float off = sum * (1.0f / (float)N);
#pragma unroll
            for (int t = 0; t < 8; ++t) v[t] = __fadd2_rn(v[t], make_float2(-off, -off));
        }
#pragma unroll
        for (int t = 0; t < 8; ++t) v[t] = __fmul2_rn(v[t], wv[t]);

        butterfly<8>(v);
        {
            const int a0 = ws_pos(j);
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                int a = a0 + t * TPS + 4 * ((t * TPS) >> 5);
                float2 y = t ? cmul(v[t], tw[0][t - 1]) : v[0];
                wre[a] = y.x;
                wim[a] = y.y;
            }
        }
        group_sync<TPS, NT>(group);

        // ---- passes 1 .. P-2 ----
        mid_passes<LOG2N, 1>(wre, wim, j, group, tw);

        // ---- last pass (radix 4 on contiguous points) + real-input split + |X|^2 ----
        float4 ar = *reinterpret_cast<const float4*>(wre + posA);
        float4 ai = *reinterpret_cast<const float4*>(wim + posA);
        float4 br = *reinterpret_cast<const float4*>(wre + posB);
        float4 bi = *reinterpret_cast<const float4*>(wim + posB);
        // all reads of this segment's workspace are done once every thread passes this barrier
        group_sync<TPS, NT>(group);

        float2 za[4], zb[4];
        dft4_planes(ar, ai, za);
        dft4_planes(br, bi, zb);
        float pk, pm;
        if (j != 0) {
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                split_power(za[t], zb[3 - t], wp[t], pk, pm);
                acc[2 * t] = fmaf(wseg, pk, acc[2 * t]);
                acc[2 * t + 1] = fmaf(wseg, pm, acc[2 * t + 1]);
            }
        } else {
            // butterfly 0 (k = K t) pairs with itself, butterfly q(K/2) (k = K/2 + K t) too
            split_power(za[0], za[0], make_float2(1.f, 0.f), pk, pm); // bins 0 and M
            acc[0] = fmaf(wseg, pk, acc[0]);
            acc[1] = fmaf(wseg, pm, acc[1]);
            split_power(za[1], za[3], make_float2(h, -h), pk, pm); // bins K and 3K
            acc[2] = fmaf(wseg, pk, acc[2]);
            acc[3] = fmaf(wseg, pm, acc[3]);
            split_power(za[2], za[2], make_float2(0.f, -1.f), pk, pm); // bin 2K = M/2 (once)
            accx = fmaf(wseg, pk, accx);
            split_power(zb[0], zb[3], w16a, pk, pm); // bins K/2 and M - K/2
            acc[4] = fmaf(wseg, pk, acc[4]);
            acc[5] = fmaf(wseg, pm, acc[5]);
            split_power(zb[1], zb[2], w16b, pk, pm); // bins K/2 + K and M - K/2 - K
            acc[6] = fmaf(wseg, pk, acc[6]);
            acc[7] = fmaf(wseg, pm, acc[7]);
        }
    }

    // every thread is done with this tile buffer and weight table: refill it with tile tl + 2
    __syncthreads();
    if (tid == 0 && tl + 2 < tile1) issue_tile(tl + 2);
    }  // tiles

    // ---- flush: one atomic (or partial-row store) per owned bin ----
    const AccSink sink = acc_sink(nullptr, p.acc, p.part, p.part_stride, blockIdx.x * G + group);
    if (j != 0) {
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            int k = kA + K * t;
            sink.add(k, acc[2 * t]);
            sink.add(M - k, acc[2 * t + 1]);
        }
    } else {
        sink.add(0, acc[0]);
        sink.add(M, acc[1]);
        sink.add(K, acc[2]);
        sink.add(3 * K, acc[3]);
        sink.add(2 * K, accx);
        sink.add(K / 2, acc[4]);
        sink.add(M - K / 2, acc[5]);
        sink.add(K / 2 + K, acc[6]);
        sink.add(M - K / 2 - K, acc[7]);
    }
}

// shared memory (bytes) needed by psd_stage_kernel<LOG2N> for tiles of T segments
template <int LOG2N>
inline size_t stage_smem_bytes(int T, int hop)
{
    using PL = Plan<LOG2N>;
    size_t tile = (size_t)(T - 1) * hop + PL::N;
    size_t redn = ((size_t)PL::G * (PL::TPS > 32 ? PL::TPS / 32 : 1) + 1) & ~(size_t)1;
    size_t fl = 2 * tile + (size_t)PL::G * 2 * PL::WS + ((T + 3) & ~3) + redn;
    return fl * sizeof(float) + 2 * sizeof(uint64_t);
}

}  // namespace sspsd
