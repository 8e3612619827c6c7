// sspsd_csd_kernel.cuh -- fused detrend + window + FFT + cross-spectrum accumulate for one stage of a
// two-channel cascade (XCascade).  For every segment s of the launch it adds, per bin k = 0 .. N/2,
//   Sxx[k] += w_s |X_s[k]|^2,  Syy[k] += w_s |Y_s[k]|^2,  Sxy[k] += w_s conj(X_s[k]) Y_s[k]
// (scipy.signal.csd's convention: H = Sxy / Sxx for y = h * x), with the PSD kernel's weights w_s.
// iq_stage_kernel shares the body (pair_stage) up to the per-bin epilogue and adds instead the two sides of the
// spectrum of z = x + i y itself: P+[k] += w_s |Z_s[k]|^2, P-[k] += w_s |Z_s[N-k]|^2 (DESIGN.md 3c).
//
// Two-for-one transform: z[n] = x~[n] + i y~[n] (both channels detrended on their own, same window) is
// transformed by ONE N-point complex FFT, and
//   X[k] = (Z[k] + conj(Z[N-k])) / 2,   Y[k] = (Z[k] - conj(Z[N-k])) / (2i).
// The FFT passes are psd_stage_kernel's, instantiated at Plan<LOG2N + 1> (M = N points, N/8 threads per
// segment), so N = 64 ... 4096: Plan stops at 2^13 points and N = 8192 is rejected by the host.
//
// Structure as psd_stage_kernel: a persistent CTA walks a contiguous range of tiles; a tile holds T
// consecutive hops (+ overlap) of BOTH channels, each brought in by TMA bulk copies from its own StreamSrc
// (one mbarrier per buffer with two arrivals, one per channel); the epilogue's rows accumulate in registers over
// the CTA's whole range and are flushed with one atomicAdd (or one partial-row store) per value.
#pragma once
#include "sspsd_stage_kernel.cuh"

namespace sspsd {

// rows of one stage's accumulator block (each acc_stride floats): Sxx, Syy, Re Sxy, Im Sxy
enum { CSD_ROWS = 4 };

// Parameters of both block kernels of a stage (csd_stage_kernel reads src[0..1], csm_cross_kernel src[0..nch-1]).
struct XStageParams {
    StreamSrc src[4];  // channels: same bookkeeping, own buffers
    int nch;           // csm_cross_kernel: 3 or 4 (src[3] unused when 3)
    long long k0;
    int nseg, T, tpc, hop, detrend, tile_cap;
    const float* win;   // N window values
    const float2* tw;   // N entries: exp(-2 pi i q / N)
    float* acc;         // the kernel's rows of `stride` floats
    int stride;
    float* part;        // deterministic mode: per-(CTA, group) partial blocks of part_stride floats
    int part_stride;
    int jb;
    float g_first, g_s;
};

// one owned bin: Z[k] and Z[N-k] -> the four row increments (0.25 w folded into wseg)
//   a = Zk + conj(Zm) = 2X,  d = Zk - conj(Zm) = 2iY,  conj(X) Y = conj(a) (-i d) / 4
__device__ __forceinline__ void csd_bin(float2 zk, float2 zm, float wseg, float (&a4)[4])
{
    const float2 a = __fadd2_rn(zk, make_float2(zm.x, -zm.y));
    const float2 d = __fadd2_rn(zk, make_float2(-zm.x, zm.y));
    a4[0] = fmaf(wseg, fmaf(a.y, a.y, a.x * a.x), a4[0]);
    a4[1] = fmaf(wseg, fmaf(d.y, d.y, d.x * d.x), a4[1]);
    a4[2] = fmaf(wseg, fmaf(a.x, d.y, -a.y * d.x), a4[2]);
    a4[3] = fmaf(-wseg, fmaf(a.x, d.x, a.y * d.y), a4[3]);
}

template <int LOG2N>
struct CsdPlan {
    using PL = Plan<LOG2N + 1>;
    static constexpr int RED = PL::TPS > 32 ? PL::TPS / 32 : 1;  // mean-detrend partial sums per group and channel
};

// read-at-each-use operand of pair_pass0: v[t] = p[(first + t) * stride], through the read-only data cache
template <class T>
struct LdgStrided {
    const T* p;
    int first, stride;
    __device__ __forceinline__ T operator[](int t) const { return __ldg(p + (first + t) * stride); }
};

// pass 0 of one pair: z[n] = x[n] + i y[n], each channel detrended on its own, windowed (wv[t]: window value of the
// thread's point t), radix-8 butterfly, twiddled (tw0[t - 1] = W_N^(j t), t = 1 .. 7), stored to the pair's work
// planes.  red: this pair's mean-detrend partial sums.  wv and tw0 are arrays held in registers (csd_stage_kernel) or
// LdgStrided views read at each use (csm_cross_kernel's register budget, DESIGN.md 3b).
template <int LOG2N, class WV, class TW>
__device__ __forceinline__ void pair_pass0(const float* sx, const float* sy, int detrend, const WV& wv, const TW& tw0,
                                           float* red, float* wre, float* wim, int tid, int j, int group)
{
    using PL = Plan<LOG2N + 1>;
    constexpr int N = PL::M, TPS = PL::TPS, NT = PL::NT;
    constexpr int WPG = CsdPlan<LOG2N>::RED;
    float2 v[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) v[t] = make_float2(sx[j + t * TPS], sy[j + t * TPS]);

    if (detrend == 1) {  // Midpoint
        const float2 off = make_float2(-sx[N / 2], -sy[N / 2]);
#pragma unroll
        for (int t = 0; t < 8; ++t) v[t] = __fadd2_rn(v[t], off);
    } else if (detrend == 2) {  // Span
        const float2 x0 = make_float2(sx[0], sy[0]);
        const float2 slope = make_float2((sx[N - 1] - x0.x) / (float)(N - 1), (sy[N - 1] - x0.y) / (float)(N - 1));
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            const float n0 = (float)(j + t * TPS);
            v[t].x -= fmaf(slope.x, n0, x0.x);
            v[t].y -= fmaf(slope.y, n0, x0.y);
        }
    } else if (detrend == 3) {  // Mean
        float2 sum = make_float2(0.f, 0.f);
#pragma unroll
        for (int t = 0; t < 8; ++t) sum = __fadd2_rn(sum, v[t]);
        if constexpr (TPS <= 32) {
#pragma unroll
            for (int m = TPS / 2; m > 0; m >>= 1) {
                sum.x += __shfl_xor_sync(0xffffffffu, sum.x, m);
                sum.y += __shfl_xor_sync(0xffffffffu, sum.y, m);
            }
        } else {
#pragma unroll
            for (int m = 16; m > 0; m >>= 1) {
                sum.x += __shfl_xor_sync(0xffffffffu, sum.x, m);
                sum.y += __shfl_xor_sync(0xffffffffu, sum.y, m);
            }
            if ((tid & 31) == 0) {
                red[2 * (group * WPG + (j >> 5))] = sum.x;
                red[2 * (group * WPG + (j >> 5)) + 1] = sum.y;
            }
            group_sync<TPS, NT>(group);
            sum = make_float2(0.f, 0.f);
#pragma unroll
            for (int w = 0; w < WPG; ++w) {
                sum.x += red[2 * (group * WPG + w)];
                sum.y += red[2 * (group * WPG + w) + 1];
            }
        }
        const float2 off = make_float2(-sum.x * (1.0f / (float)N), -sum.y * (1.0f / (float)N));
#pragma unroll
        for (int t = 0; t < 8; ++t) v[t] = __fadd2_rn(v[t], off);
    }
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        const float w = wv[t];
        v[t] = __fmul2_rn(v[t], make_float2(w, w));
    }

    butterfly<8>(v);
    const int a0 = ws_pos(j);
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        const int a = a0 + t * TPS + 4 * ((t * TPS) >> 5);
        const float2 y = t ? cmul(v[t], tw0[t - 1]) : v[0];
        wre[a] = y.x;
        wim[a] = y.y;
    }
}

// The bins a thread owns under the last-pass map (butterflies qA and qB, whose outputs pair up as (k, N - k)):
// j != 0: kA, kA + K, 2K - kA, K - kA (and -1: none);  j == 0: 0, K, 2K = N/2, K/2, 3K/2.
template <int LOG2N>
__device__ __forceinline__ void owned_bins(int j, int kA, int (&bins)[5])
{
    constexpr int K = Plan<LOG2N + 1>::K;
    if (j != 0) {
        bins[0] = kA; bins[1] = kA + K; bins[2] = 2 * K - kA; bins[3] = K - kA; bins[4] = -1;
    } else {
        bins[0] = 0; bins[1] = K; bins[2] = 2 * K; bins[3] = K / 2; bins[4] = 3 * K / 2;
    }
}

// flush of a thread's accumulators acc[owned bin][row]: one atomic (or partial-row store) per owned value, row r
// at r * stride
template <int LOG2N, int ROWS>
__device__ __forceinline__ void pair_flush(const float (&acc)[5][ROWS], int j, int kA, const AccSink& sink, int stride)
{
    int bins[5];
    owned_bins<LOG2N>(j, kA, bins);
#pragma unroll
    for (int b = 0; b < 5; ++b) {
        if (bins[b] < 0) continue;
        SSPSD_ASSERT(bins[b] <= Plan<LOG2N + 1>::M / 2);
#pragma unroll
        for (int r = 0; r < ROWS; ++r) sink.add(r * stride + bins[b], acc[b][r]);
    }
}

// The per-bin epilogues of pair_stage: what one owned bin's Z[k] and Z[N-k] add to the thread's ROWS accumulators.
// CsdEpi: the two-for-one split into Sxx, Syy, Re Sxy, Im Sxy (csd_stage_kernel).
struct CsdEpi {
    static constexpr int ROWS = CSD_ROWS;
    static __device__ __forceinline__ void bin(float2 zk, float2 zm, float wseg, float (&a)[ROWS])
    {
        csd_bin(zk, zm, wseg, a);
    }
};

// IqEpi: the two sides of the spectrum of z itself, P+ = |Z[k]|^2 and P- = |Z[N-k]|^2 (iq_stage_kernel).  wseg
// carries ewma_weight's 0.25 of the split, which has no place here: 4 wseg is the weight, exactly (a power of two).
enum { IQ_ROWS = 2 };
struct IqEpi {
    static constexpr int ROWS = IQ_ROWS;
    static __device__ __forceinline__ void bin(float2 zk, float2 zm, float wseg, float (&a)[ROWS])
    {
        const float w = 4.0f * wseg;
        a[0] = fmaf(w, fmaf(zk.y, zk.y, zk.x * zk.x), a[0]);
        a[1] = fmaf(w, fmaf(zm.y, zm.y, zm.x * zm.x), a[1]);
    }
};

// The body of both pair kernels: tiles of both channels, two-for-one transform of z = x + i y, EPI per owned bin,
// flush of EPI::ROWS rows.  tid is threadIdx.x read in the kernel, where the compiler knows its range from the launch
// bounds (csd_stage_kernel then compiles exactly as it did before the body was shared).
template <int LOG2N, class EPI>
__device__ __forceinline__ void pair_stage(const XStageParams& p, const int tid)
{
    using PL = Plan<LOG2N + 1>;
    constexpr int N = PL::M, TPS = PL::TPS, NT = PL::NT, G = PL::G, K = PL::K, WS = PL::WS;
    constexpr int WPG = CsdPlan<LOG2N>::RED;
    extern __shared__ __align__(16) float smem[];
    float* tiles = smem;                    // [buffer][channel] tile_cap floats
    float* wsb = smem + 4 * p.tile_cap;
    float* wgt = wsb + G * 2 * WS;
    float* red = wgt + ((p.T + 3) & ~3);
    uint64_t* bars = reinterpret_cast<uint64_t*>(red + ((2 * G * WPG + 1) & ~1));

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
        const long long g = (p.k0 + s0) * (long long)hop;
        ring_issue(p.src[0], g, (n_s - 1) * hop + N, tiles + (2 * b) * p.tile_cap, &bars[b]);
        ring_issue(p.src[1], g, (n_s - 1) * hop + N, tiles + (2 * b + 1) * p.tile_cap, &bars[b]);
    };
    if (tid == 0) {
        mbar_init(&bars[0], 2);  // one arrival per channel
        mbar_init(&bars[1], 2);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0 && tile0 < tile1) {
        issue_tile(tile0);
        if (tile0 + 1 < tile1) issue_tile(tile0 + 1);
    }

    float wv[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) wv[t] = __ldg(p.win + j + t * TPS);
    float2 tw[PL::P - 1][7];
    load_pass_twiddles<LOG2N + 1, 0>(tw, p.tw, j);

    // last pass: butterflies qA and qB, whose outputs pair up as (k, N - k)
    constexpr int RL = 1 << PL::log2radix(PL::P - 2);
    constexpr int HALF = RL / 2;
    const int qA = RL * (j / HALF) + (j % HALF);
    const int kA = klow_of_q<LOG2N + 1>(qA);
    const int qB = (j == 0) ? HALF : q_of_klow<LOG2N + 1>(K - kA);
    const int posA = ws_pos(4 * qA), posB = ws_pos(4 * qB);

    float* wre = wsb + group * 2 * WS;
    float* wim = wre + WS;
    float acc[5][EPI::ROWS];  // [owned_bins][EPI's rows]
#pragma unroll
    for (int b = 0; b < 5; ++b)
#pragma unroll
        for (int r = 0; r < EPI::ROWS; ++r) acc[b][r] = 0.f;

    for (int tl = tile0; tl < tile1; ++tl) {
    const int buf = (tl - tile0) & 1;
    const int seg0 = tl * p.T;
    const int ns = min(p.T, p.nseg - seg0);
    const float* tile_x = tiles + (2 * buf) * p.tile_cap;
    const float* tile_y = tile_x + p.tile_cap;
    for (int i = tid; i < ns; i += NT) wgt[i] = ewma_weight(p, seg0 + i);
    mbar_wait(&bars[buf], (uint32_t)((tl - tile0) >> 1) & 1u);
    __syncthreads();

    const int iters = (ns + G - 1) / G;
    for (int it = 0; it < iters; ++it) {
        const int s = it * G + group;
        const bool valid = s < ns;
        const int sc = valid ? s : ns - 1;
        const float* sx = tile_x + sc * hop;
        const float* sy = tile_y + sc * hop;
        const float wseg = valid ? wgt[sc] : 0.f;

        pair_pass0<LOG2N>(sx, sy, p.detrend, wv, tw[0], red, wre, wim, tid, j, group);
        group_sync<TPS, NT>(group);

        mid_passes<LOG2N + 1, 1>(wre, wim, j, group, tw);

        // ---- last pass (radix 4 on contiguous points) + the epilogue of the owned bins ----
        float4 ar = *reinterpret_cast<const float4*>(wre + posA);
        float4 ai = *reinterpret_cast<const float4*>(wim + posA);
        float4 br = *reinterpret_cast<const float4*>(wre + posB);
        float4 bi = *reinterpret_cast<const float4*>(wim + posB);
        // the red[] partial sums of the next segment's mean detrend are written after this barrier too
        group_sync<TPS, NT>(group);

        float2 za[4], zb[4];
        dft4_planes(ar, ai, za);  // Z[kA + K t]
        dft4_planes(br, bi, zb);  // Z[N - kA - K (3 - t)]  (j == 0: Z[K/2 + K t])
        if (j != 0) {
            EPI::bin(za[0], zb[3], wseg, acc[0]);  // bin kA
            EPI::bin(za[1], zb[2], wseg, acc[1]);  // bin kA + K
            EPI::bin(zb[1], za[2], wseg, acc[2]);  // bin 2K - kA
            EPI::bin(zb[0], za[3], wseg, acc[3]);  // bin K - kA
        } else {
            EPI::bin(za[0], za[0], wseg, acc[0]);  // bin 0
            EPI::bin(za[1], za[3], wseg, acc[1]);  // bin K
            EPI::bin(za[2], za[2], wseg, acc[2]);  // bin 2K = N/2
            EPI::bin(zb[0], zb[3], wseg, acc[3]);  // bin K/2
            EPI::bin(zb[1], zb[2], wseg, acc[4]);  // bin 3K/2
        }
    }

    __syncthreads();
    if (tid == 0 && tl + 2 < tile1) issue_tile(tl + 2);
    }  // tiles

    pair_flush<LOG2N>(acc, j, kA, acc_sink(nullptr, p.acc, p.part, p.part_stride, blockIdx.x * G + group), p.stride);
}

template <int LOG2N>
__global__ void __launch_bounds__(Plan<LOG2N + 1>::NT, Plan<LOG2N + 1>::NT <= 256 ? 2 : 1)
csd_stage_kernel(const XStageParams p)
{
    pair_stage<LOG2N, CsdEpi>(p, threadIdx.x);
}

// The two-sided spectrum of z = x + i y (XCascade's I/Q kind): P+[k] += w |Z[k]|^2, P-[k] += w |Z[N-k]|^2 for
// k = 0 .. N/2, csd_stage_kernel's transform, tiles, launch shape and shared memory (csd_smem_bytes).
template <int LOG2N>
__global__ void __launch_bounds__(Plan<LOG2N + 1>::NT, Plan<LOG2N + 1>::NT <= 256 ? 2 : 1)
iq_stage_kernel(const XStageParams p)
{
    pair_stage<LOG2N, IqEpi>(p, threadIdx.x);
}

// shared memory (bytes) of csd_stage_kernel<LOG2N> for tiles of T segments
template <int LOG2N>
inline size_t csd_smem_bytes(int T, int hop)
{
    using PL = Plan<LOG2N + 1>;
    size_t tile = (size_t)(T - 1) * hop + PL::M;
    size_t redn = ((size_t)2 * PL::G * CsdPlan<LOG2N>::RED + 1) & ~(size_t)1;
    size_t fl = 4 * tile + (size_t)PL::G * 2 * PL::WS + ((T + 3) & ~3) + redn;
    return fl * sizeof(float) + 2 * sizeof(uint64_t);
}

}  // namespace sspsd
