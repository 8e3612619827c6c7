// sspsd_csm_kernel.cuh -- the off-diagonal 2x2 block of a cross-spectral matrix (XCascade with K = 3 or 4
// channels).  Channels pair up as A = (0, 1) and B = (2, 3); the diagonal blocks (A, A) and (B, B) are
// csd_stage_kernel's.  For every segment s of the launch this kernel adds, per bin k = 0 .. N/2,
//   S02 += w_s conj(X0) X2,  S03 += w_s conj(X0) X3,  S12 += w_s conj(X1) X2,  S13 += w_s conj(X1) X3
// as 8 real rows (Re, Im of S02, S03, S12, S13), with the PSD kernel's weights w_s.
//
// Each pair goes through csd_stage_kernel's two-for-one transform: z_A = x0~ + i x1~, z_B = x2~ + i x3~, one
// N-point complex FFT each (Plan<LOG2N + 1> passes, csd_stage_kernel's thread -> bin map), then
//   2 X0 = a_A = Z_A[k] + conj(Z_A[N-k]),  2i X1 = d_A = Z_A[k] - conj(Z_A[N-k])   (and B likewise), so
//   conj(X0) X2 = conj(a_A) a_B / 4,  conj(X0) X3 = -i conj(a_A) d_B / 4,
//   conj(X1) X2 = i conj(d_A) a_B / 4,  conj(X1) X3 = conj(d_A) d_B / 4.
//
// Register budget (DESIGN.md 3b): 40 accumulators (5 bins x 8 rows) must fit beside one transform in 128
// registers.  So, unlike csd_stage_kernel, the two transforms run in two work-plane pairs of shared memory
// (the last pass of A is not held in registers while B runs), and the pass twiddles are read from the
// (L1-resident) global table at each use instead of being pinned in registers.
//
// K = 3: channel 3 does not exist.  Its tile slots are zero-filled once and never copied to (nch == 3); the
// rows that involve it (S03, S13) are computed from zeros and never read out.
#pragma once
#include "sspsd_csd_kernel.cuh"

namespace sspsd {

// rows of the cross block: Re/Im of S02, S03, S12, S13
enum { CSM_XROWS = 8 };

// one owned bin of both pairs: (Z_A[k], Z_A[N-k]) and (Z_B[k], Z_B[N-k]) -> the 8 row increments (0.25 w in wseg)
__device__ __forceinline__ void csm_bin(float2 pk, float2 pm, float2 qk, float2 qm, float wseg, float (&a8)[8])
{
    const float2 aA = __fadd2_rn(pk, make_float2(pm.x, -pm.y));
    const float2 dA = __fadd2_rn(pk, make_float2(-pm.x, pm.y));
    const float2 aB = __fadd2_rn(qk, make_float2(qm.x, -qm.y));
    const float2 dB = __fadd2_rn(qk, make_float2(-qm.x, qm.y));
    // conj(p) q = (p.x q.x + p.y q.y, p.x q.y - p.y q.x)
    a8[0] = fmaf(wseg, fmaf(aA.x, aB.x, aA.y * aB.y), a8[0]);   // Re conj(aA) aB
    a8[1] = fmaf(wseg, fmaf(aA.x, aB.y, -aA.y * aB.x), a8[1]);  // Im conj(aA) aB
    a8[2] = fmaf(wseg, fmaf(aA.x, dB.y, -aA.y * dB.x), a8[2]);  // Re -i conj(aA) dB = Im conj(aA) dB
    a8[3] = fmaf(-wseg, fmaf(aA.x, dB.x, aA.y * dB.y), a8[3]);  // Im -i conj(aA) dB = -Re conj(aA) dB
    a8[4] = fmaf(-wseg, fmaf(dA.x, aB.y, -dA.y * aB.x), a8[4]); // Re i conj(dA) aB = -Im conj(dA) aB
    a8[5] = fmaf(wseg, fmaf(dA.x, aB.x, dA.y * aB.y), a8[5]);   // Im i conj(dA) aB = Re conj(dA) aB
    a8[6] = fmaf(wseg, fmaf(dA.x, dB.x, dA.y * dB.y), a8[6]);   // Re conj(dA) dB
    a8[7] = fmaf(wseg, fmaf(dA.x, dB.y, -dA.y * dB.x), a8[7]);  // Im conj(dA) dB
}

// passes 1 .. P-2 over both pairs' planes (mid_passes with the twiddles read at each use), one barrier per pass
template <int LOG2N, int PASS>
__device__ __forceinline__ void csm_mid_passes(float* __restrict__ ws, int j, int group, const float2* __restrict__ twg)
{
    using PL = Plan<LOG2N + 1>;
    if constexpr (PASS < PL::P - 1) {
        constexpr int LR = PL::log2radix(PASS), R = 1 << LR;
        constexpr int LS = PL::log2stride(PASS), S = 1 << LS;
        constexpr int BPT = 8 / R;
#pragma unroll
        for (int pr = 0; pr < 2; ++pr) {
            float* wre = ws + pr * 2 * PL::WS;
            float* wim = wre + PL::WS;
#pragma unroll
            for (int u = 0; u < BPT; ++u) {
                const int bf = j + u * PL::TPS;
                const int o = bf & (S - 1);
                const int base = ((bf >> LS) << (LR + LS)) + o;
                const int a0 = ws_pos(base);
                float2 v[R];
#pragma unroll
                for (int t = 0; t < R; ++t) {
                    const int a = a0 + t * S + 4 * ((t * S) >> 5);
                    v[t] = make_float2(wre[a], wim[a]);
                }
                butterfly<R>(v);
#pragma unroll
                for (int t = 0; t < R; ++t) {
                    const int a = a0 + t * S + 4 * ((t * S) >> 5);
                    const float2 y = t ? cmul(v[t], __ldg(&twg[(o * t) << (PL::LOG2M - LR - LS)])) : v[0];
                    wre[a] = y.x;
                    wim[a] = y.y;
                }
            }
        }
        group_sync<PL::TPS, PL::NT>(group);
        csm_mid_passes<LOG2N, PASS + 1>(ws, j, group, twg);
    }
}

template <int LOG2N>
__global__ void __launch_bounds__(Plan<LOG2N + 1>::NT, Plan<LOG2N + 1>::NT <= 256 ? 2 : 1)
csm_cross_kernel(const XStageParams p)
{
    using PL = Plan<LOG2N + 1>;
    constexpr int N = PL::M, TPS = PL::TPS, NT = PL::NT, G = PL::G, K = PL::K, WS = PL::WS;
    constexpr int WPG = CsdPlan<LOG2N>::RED;
    extern __shared__ __align__(16) float smem[];
    float* tiles = smem;                    // [buffer][channel] tile_cap floats
    float* wsb = smem + 8 * p.tile_cap;     // [group][pair][re, im] WS floats
    float* wgt = wsb + G * 4 * WS;
    float* red = wgt + ((p.T + 3) & ~3);    // [pair][group][WPG] (x, y) sums
    uint64_t* bars = reinterpret_cast<uint64_t*>(red + ((4 * G * WPG + 1) & ~1));

    const int tid = threadIdx.x;
    const int group = tid / TPS;
    const int j = tid % TPS;
    const int hop = p.hop;
    const int nch = p.nch;
    const int ntiles = (p.nseg + p.T - 1) / p.T;
    const int tile0 = blockIdx.x * p.tpc;
    const int tile1 = min(tile0 + p.tpc, ntiles);

    auto issue_tile = [&](int tl) {
        const int s0 = tl * p.T;
        const int n_s = min(p.T, p.nseg - s0);
        const int b = (tl - tile0) & 1;
        const long long g = (p.k0 + s0) * (long long)hop;
        for (int c = 0; c < nch; ++c)
            ring_issue(p.src[c], g, (n_s - 1) * hop + N, tiles + (4 * b + c) * p.tile_cap, &bars[b]);
    };
    if (nch == 3) {  // the absent channel reads as zeros in both buffers
        for (int i = tid; i < p.tile_cap; i += NT) {
            tiles[3 * p.tile_cap + i] = 0.f;
            tiles[7 * p.tile_cap + i] = 0.f;
        }
    }
    if (tid == 0) {
        mbar_init(&bars[0], nch);  // one arrival per channel
        mbar_init(&bars[1], nch);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0 && tile0 < tile1) {
        issue_tile(tile0);
        if (tile0 + 1 < tile1) issue_tile(tile0 + 1);
    }

    // last pass: butterflies qA and qB, whose outputs pair up as (k, N - k)  (csd_stage_kernel's map)
    constexpr int RL = 1 << PL::log2radix(PL::P - 2);
    constexpr int HALF = RL / 2;
    const int qA = RL * (j / HALF) + (j % HALF);
    const int kA = klow_of_q<LOG2N + 1>(qA);
    const int qB = (j == 0) ? HALF : q_of_klow<LOG2N + 1>(K - kA);
    const int posA = ws_pos(4 * qA), posB = ws_pos(4 * qB);

    float* ws = wsb + group * 4 * WS;
    float acc[5][8];  // [owned_bins][Re/Im of S02, S03, S12, S13]
#pragma unroll
    for (int b = 0; b < 5; ++b)
#pragma unroll
        for (int r = 0; r < 8; ++r) acc[b][r] = 0.f;

    for (int tl = tile0; tl < tile1; ++tl) {
    const int buf = (tl - tile0) & 1;
    const int seg0 = tl * p.T;
    const int ns = min(p.T, p.nseg - seg0);
    const float* tile = tiles + (4 * buf) * p.tile_cap;
    for (int i = tid; i < ns; i += NT) wgt[i] = ewma_weight(p, seg0 + i);
    mbar_wait(&bars[buf], (uint32_t)((tl - tile0) >> 1) & 1u);
    __syncthreads();

    const int iters = (ns + G - 1) / G;
    for (int it = 0; it < iters; ++it) {
        const int s = it * G + group;
        const bool valid = s < ns;
        const int sc = valid ? s : ns - 1;
        const float* s0 = tile + sc * hop;
        const float wseg = valid ? wgt[sc] : 0.f;

        // ---- pass 0 of both pairs, each into its own work planes; window and twiddles read at each use ----
#pragma unroll
        for (int pr = 0; pr < 2; ++pr)
            pair_pass0<LOG2N>(s0 + (2 * pr) * p.tile_cap, s0 + (2 * pr + 1) * p.tile_cap, p.detrend,
                              LdgStrided<float>{p.win + j, 0, TPS}, LdgStrided<float2>{p.tw, 1, j},
                              red + pr * 2 * G * WPG, ws + pr * 2 * WS, ws + pr * 2 * WS + WS, tid, j, group);
        group_sync<TPS, NT>(group);

        csm_mid_passes<LOG2N, 1>(ws, j, group, p.tw);

        // ---- last pass (radix 4 on contiguous points) of both pairs + split + the four cross products ----
        float2 za[4], zb[4], zc[4], zd[4];
        {
            const float* wre = ws;
            const float* wim = ws + WS;
            dft4_planes(*reinterpret_cast<const float4*>(wre + posA), *reinterpret_cast<const float4*>(wim + posA), za);
            dft4_planes(*reinterpret_cast<const float4*>(wre + posB), *reinterpret_cast<const float4*>(wim + posB), zb);
            wre += 2 * WS;
            wim += 2 * WS;
            dft4_planes(*reinterpret_cast<const float4*>(wre + posA), *reinterpret_cast<const float4*>(wim + posA), zc);
            dft4_planes(*reinterpret_cast<const float4*>(wre + posB), *reinterpret_cast<const float4*>(wim + posB), zd);
        }
        // the red[] partial sums of the next segment's mean detrend are written after this barrier too
        group_sync<TPS, NT>(group);

        if (j != 0) {
            csm_bin(za[0], zb[3], zc[0], zd[3], wseg, acc[0]);  // bin kA
            csm_bin(za[1], zb[2], zc[1], zd[2], wseg, acc[1]);  // bin kA + K
            csm_bin(zb[1], za[2], zd[1], zc[2], wseg, acc[2]);  // bin 2K - kA
            csm_bin(zb[0], za[3], zd[0], zc[3], wseg, acc[3]);  // bin K - kA
        } else {
            csm_bin(za[0], za[0], zc[0], zc[0], wseg, acc[0]);  // bin 0
            csm_bin(za[1], za[3], zc[1], zc[3], wseg, acc[1]);  // bin K
            csm_bin(za[2], za[2], zc[2], zc[2], wseg, acc[2]);  // bin 2K = N/2
            csm_bin(zb[0], zb[3], zd[0], zd[3], wseg, acc[3]);  // bin K/2
            csm_bin(zb[1], zb[2], zd[1], zd[2], wseg, acc[4]);  // bin 3K/2
        }
    }

    __syncthreads();
    if (tid == 0 && tl + 2 < tile1) issue_tile(tl + 2);
    }  // tiles

    pair_flush<LOG2N>(acc, j, kA, acc_sink(nullptr, p.acc, p.part, p.part_stride, blockIdx.x * G + group), p.stride);
}

// shared memory (bytes) of csm_cross_kernel<LOG2N> for tiles of T segments
template <int LOG2N>
inline size_t csm_smem_bytes(int T, int hop)
{
    using PL = Plan<LOG2N + 1>;
    size_t tile = (size_t)(T - 1) * hop + PL::M;
    size_t redn = ((size_t)4 * PL::G * CsdPlan<LOG2N>::RED + 1) & ~(size_t)1;
    size_t fl = 8 * tile + (size_t)PL::G * 4 * PL::WS + ((T + 3) & ~3) + redn;
    return fl * sizeof(float) + 2 * sizeof(uint64_t);
}

}  // namespace sspsd
