// sspsd_decim_kernel.cuh -- K3: decimate-by-8 half-band cascade between PSD stages.
//
// Replaces `HBF_DEC_CASCADE.inner.1.inner.1.block(&mut self.hbf, xb, y)` (reference
// src/psd.rs:246-253, idsp::hbf::HbfDec8) and the once-per-stage drain of the first
// hbf_dec_response_length(3) outputs (psd.rs:149, 254-260).  The three half-band FIRs are finite
// impulse responses, so the persistent filter state of the reference is exactly "the last H-1
// input samples": the host keeps them in the stage's carry buffer (StreamSrc) and every CTA
// recomputes its own warm-up from that halo (overlap-save), which makes CTAs independent.
//
// Per CTA: OB final outputs.  The x tile is de-interleaved into even/odd planes in shared memory
// (a half-band FIR only touches the odd phase plus one even centre tap) and each thread computes
// DEC_P = 8 consecutive outputs from a sliding register window (2M+7 loads for 8 outputs; the kernel
// is bound by the shared-memory data pipe, profiles/r01_ncu_summary.md).  Lanes therefore read plane
// elements 8w + c for a common c: planes are stored "polyphase by 8" (element i at (i&7)*S + (i>>3)),
// which makes every such read unit-stride across lanes for every c (the first version padded 1/32
// and measured 38 % conflicting wavefronts); S = 4 mod 32 keeps the phase groups a store instruction
// touches on disjoint banks.
#pragma once
#include "sspsd_device.cuh"
#include "sspsd_hbf_taps.h"

namespace sspsd {

__constant__ __align__(8) float c_hbf_taps[SSPSD_HBF_NPRESET][3][SSPSD_HBF_MAXTAPS + 1];
// the same taps shifted by one position, so that the pairs (t1,t2), (t3,t4), ... are 8-byte aligned too
__constant__ __align__(8) float c_hbf_taps_sh[SSPSD_HBF_NPRESET][3][SSPSD_HBF_MAXTAPS + 1];

constexpr int DEC_OB = 960;   // outputs per CTA (7680 input samples + 488 of halo)
constexpr int DEC_P = 8;      // consecutive outputs per thread
constexpr int DEC_LP = 3;
constexpr int DEC_NT = 256;

constexpr int roundup(int v, int m) { return (v + m - 1) / m * m; }

// Tap counts: MA = highest-rate stage (tap set 2), MB = set 1, MC = lowest-rate stage (set 0); OB = final
// outputs per tile
template <int MA, int MB, int MC, int OB_ = DEC_OB>
struct DecGeom {
    static constexpr int OB = OB_;
    static constexpr int NB = roundup(2 * OB + 4 * MC - 2, DEC_P);  // stage-B outputs computed per CTA
    static constexpr int NA = roundup(2 * NB + 4 * MB - 2, DEC_P);      // stage-A outputs
    static constexpr int NX = roundup(2 * NA + 4 * MA - 2, 8);      // input samples loaded
    static constexpr int HALO = NX - 8 * OB;                        // history needed before the block
    // polyphase-by-8 plane layout: phase stride S = ceil(len/8) rounded up to 4 mod 32
    static constexpr int phase_stride(int len) { return ((len + DEC_P - 1) / DEC_P + 27) / 32 * 32 + 4; }
    static constexpr int SX = phase_stride(NX / 2), SA = phase_stride(NA / 2), SB = phase_stride(NB / 2);
    static constexpr int SMEM_FLOATS = 2 * DEC_P * (SX + SA + SB);
};

// One half-band stage over de-interleaved, padded planes.
//   ine/ino : input planes; plane index r <-> input sample in_base + 2r (+1 for the odd plane)
//   outputs j = out_base + 4w + q (q < 4), for work items w < n_out/4, where
//   y[j] = e[r-M+1] + sum_i t[i]*(o[r-2M+1+i] + o[r-i]),  r = j - in_base/2   (DC gain 2 per stage)
// rel0 = out_base - in_base/2 (relative index of the first output).
// If FINAL, outputs go to the next stage's stream (DecimParams) for m in [m0, m1); otherwise to
// the padded planes oute/outo with plane index (j - out_base)/2.
__device__ __forceinline__ void carry_job(const StreamSrc& src, const CarryJob& c)
{
    SSPSD_ASSERT(c.n >= 0 && c.n <= c.dst_cap && c.head_n >= 0 && c.head_n < 4);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < c.n; i += gridDim.x * blockDim.x) {
        const float v = ld_stream1(src, c.g0 + i);
        c.dst[i] = v;
        if (i >= c.n - c.head_n) c.head_dst[i - (c.n - c.head_n)] = v;
    }
}

struct DecimParams {
    CarryJob cc;
    StreamSrc src;
    long long m0, m1;  // outputs m in [m0, m1) are produced by this launch (m = chunk index of 8 inputs)
    long long drain;   // outputs m < drain are discarded (psd.rs:254-260)
    // output m is sample g = m - drain of the next stage's stream; it is stored at
    // out_fresh[g - out_split] (out_split = floor4 of the next stage's sample count, so g >= out_split)
    float* out_fresh;
    long long out_split;
    long long out_cap;  // floats available at out_fresh (bounds-checking build)
    int preset;
};

// The P consecutive outputs q of one run, starting at an even output: y[q] = centre(q) + a_q, where a_q is the tap
// sum over the run's odd-phase window win[0 .. 2M + P - 2] (output q reads win[q .. q + 2M - 1]), held as aligned
// register pairs wp[m] = (win[2m], win[2m+1]).  Every decimator kernel computes its outputs with this one expression,
// which is what makes them bit-identical.
template <int M, int P, int PRESET, int SET, class Centre>
__device__ __forceinline__ void hbf_outputs(const float2 (&wp)[M + P / 2], Centre centre, float (&y)[P])
{
    static_assert(P % 2 == 0, "runs start and end on an output pair");
    // Taps are paired so that both window operands of a packed add are aligned pairs: for even q the
    // pairs (0,1), (2,3), ..., for odd q the pairs (1,2), (3,4), ...; tap i multiplies
    // win[q+i] + win[q+2M-1-i], and the mirrored operand of a pair is the swapped pair (free swizzle).
    // The two halves of the packed accumulator hold the even- and the odd-tap partial sums.
    const float2* __restrict__ tp0 = reinterpret_cast<const float2*>(&c_hbf_taps[PRESET][SET][0]);
    const float2* __restrict__ tp1 = reinterpret_cast<const float2*>(&c_hbf_taps_sh[PRESET][SET][0]);
#pragma unroll
    for (int q = 0; q < P; ++q) {
        float2 acc = make_float2(0.f, 0.f);
        const int i0 = q & 1;  // first paired tap
#pragma unroll
        for (int i = i0; i + 1 < M; i += 2) {
            const float2 l = wp[(q + i) >> 1];
            const float2 r = wp[(q + 2 * M - 2 - i) >> 1];
            const float2 sum = __fadd2_rn(l, make_float2(r.y, r.x));
            acc = __ffma2_rn(sum, (q & 1) ? tp1[(i - 1) >> 1] : tp0[i >> 1], acc);
        }
        float a = acc.x + acc.y;
        auto winv = [&](int k) { return (k & 1) ? wp[k >> 1].y : wp[k >> 1].x; };
        if (q & 1) a = fmaf(winv(q) + winv(q + 2 * M - 1), c_hbf_taps[PRESET][SET][0], a);  // tap 0
        // the last tap is unpaired when the paired range [i0, M) has odd length
        if (((M - i0) & 1) != 0) a = fmaf(winv(q + M - 1) + winv(q + M), c_hbf_taps[PRESET][SET][M - 1], a);
        y[q] = centre(q) + a;
    }
}

template <int M, int SI, int SO, int REL0, bool FINAL, int PRESET, int SET>
__device__ __forceinline__ void hbf_stage(const float* __restrict__ ine, const float* __restrict__ ino,
                                          int n_out, float* __restrict__ oute,
                                          float* __restrict__ outo, float* __restrict__ gout, int rel_lo, int rel_hi,
                                          long long gidx0 = 0, long long gcap = 0)
{
    (void)gidx0;
    (void)gcap;
    constexpr int P = DEC_P, LP = DEC_LP;
    for (int w = threadIdx.x; w < n_out / P; w += DEC_NT) {
        // plane index of window element i is P w + (REL0 - 2M + 1 + i): its phase and offset are compile
        // time constants, only `w` is per thread (unit stride across lanes)
        // window of odd-plane samples as aligned register pairs (win[2m], win[2m+1])
        constexpr int NW = 2 * M + P - 1;
        float2 wp[(NW + 1) / 2];
#pragma unroll
        for (int i = 0; i < NW; ++i) {
            const int c = REL0 - 2 * M + 1 + i;
            const float x = ino[(c & (P - 1)) * SI + (c >> LP) + w];
            if (i & 1) wp[i >> 1].y = x; else wp[i >> 1].x = x;
        }
        float y[P];
        hbf_outputs<M, P, PRESET, SET>(wp, [&](int q) {
            const int ce = REL0 + q - M + 1;
            return ine[(ce & (P - 1)) * SI + (ce >> LP) + w];
        }, y);
        if constexpr (FINAL) {
            // gout points at the block's first output; only [rel_lo, rel_hi) of the block is stored
#pragma unroll
            for (int q = 0; q < P; ++q) {
                const int r = P * w + q;
                if (r >= rel_lo && r < rel_hi) {
                    SSPSD_ASSERT(gidx0 + r >= 0 && gidx0 + r < gcap);
                    gout[r] = y[q];
                }
            }
        } else {
            // out_base is even: q even -> even plane, q odd -> odd plane, plane index (P/2) w + q/2, whose
            // polyphase position is phase (P/2)(w&1) + q/2, offset w >> 1
            const int pb = (w & 1) * (P / 2) * SO + (w >> 1);
#pragma unroll
            for (int r = 0; r < P / 2; ++r) {
                oute[pb + r * SO] = y[2 * r];
                outo[pb + r * SO] = y[2 * r + 1];
            }
        }
    }
}

template <int MA, int MB, int MC, int PRESET>
__global__ void __launch_bounds__(DEC_NT) decim8_kernel(const DecimParams p)
{
    using GE = DecGeom<MA, MB, MC>;
    extern __shared__ __align__(16) float smem[];
    float* xe = smem;
    float* xo = xe + DEC_P * GE::SX;
    float* ae = xo + DEC_P * GE::SX;
    float* ao = ae + DEC_P * GE::SA;
    float* be = ao + DEC_P * GE::SA;
    float* bo = be + DEC_P * GE::SB;

    // blocks are counted down from the top of the range so that every block is full size and only
    // the lowest one is clipped (by the m >= m0 store guard)
    const long long mhi = p.m1 - (long long)blockIdx.x * DEC_OB;
    const long long x_base = 8 * mhi - GE::NX;          // multiple of 8
    const long long c_base = mhi - DEC_OB;

    // ---- load + de-interleave into the polyphase planes: x[x_base + 4v .. +3] = (e, o, e, o) ----
    // plane index r = 2v (+1): phase (r & 7) = 2 (v & 3) (+1), offset r >> 3 = v >> 2
    if (x_base >= p.src.split) {
        // whole block inside the fresh buffer (all but the first block of a batch): straight 128-bit loads
        const float4* __restrict__ gx = reinterpret_cast<const float4*>(p.src.fresh + (x_base - p.src.split));
        constexpr int NV = GE::NX / 4;
#pragma unroll 2
        for (int v0 = 0; v0 < NV; v0 += 4 * DEC_NT) {
            float4 f[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int v = v0 + u * DEC_NT + threadIdx.x;
                if (v < NV) f[u] = __ldg(gx + v);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int v = v0 + u * DEC_NT + threadIdx.x;
                if (v < NV) {
                    const int pos = 2 * (v & 3) * GE::SX + (v >> 2);
                    xe[pos] = f[u].x;
                    xo[pos] = f[u].y;
                    xe[pos + GE::SX] = f[u].z;
                    xo[pos + GE::SX] = f[u].w;
                }
            }
        }
    } else {
        for (int v = threadIdx.x; v < GE::NX / 4; v += DEC_NT) {
            float4 f = ld_stream4(p.src, x_base + 4ll * v);
            const int pos = 2 * (v & 3) * GE::SX + (v >> 2);
            xe[pos] = f.x;
            xo[pos] = f.y;
            xe[pos + GE::SX] = f.z;
            xo[pos + GE::SX] = f.w;
        }
    }
    __syncthreads();
    // REL0 = relative index of each stage's first output inside its input planes: out_base - in_base/2
    hbf_stage<MA, GE::SX, GE::SA, GE::NX / 2 - GE::NA, false, PRESET, 2>(xe, xo, GE::NA, ae, ao, nullptr, 0, 0);
    __syncthreads();
    hbf_stage<MB, GE::SA, GE::SB, GE::NA / 2 - GE::NB, false, PRESET, 1>(ae, ao, GE::NB, be, bo, nullptr, 0, 0);
    __syncthreads();
    // outputs m in [max(m0, drain), mhi) of this block [c_base, mhi); output m is sample m - drain of the
    // next stage's stream, stored at out_fresh[m - drain - out_split]
    const long long lo = p.m0 > p.drain ? p.m0 : p.drain;
    const int rel_lo = lo > c_base ? (int)(lo - c_base) : 0;
    hbf_stage<MC, GE::SB, GE::SB, GE::NB / 2 - DEC_OB, true, PRESET, 0>(be, bo, DEC_OB, nullptr, nullptr,
                                                            p.out_fresh + (c_base - p.drain - p.out_split), rel_lo,
                                                            DEC_OB, c_base - p.drain - p.out_split, p.out_cap);
}

// ---------------------------------------------------------------------------------------------
// K3, second generation: persistent CTAs with the x tile staged by ONE TMA bulk copy.
//
// ncu on the tiled kernel above (profiles/r02_ncu_summary.md): 38 % of all stall samples sit on the
// de-interleaving STS waiting for its LDG (long_scoreboard) -- the synchronous tile load at the start of
// every CTA, hidden only by the other two CTAs of the SM.  Here a CTA walks over tiles blockIdx.x,
// blockIdx.x + gridDim.x, ...; the raw tile (NX contiguous floats, two copies when it straddles the
// carry/fresh boundary of the StreamSrc) is fetched by cp.async.bulk into a staging buffer and reported
// to an mbarrier; the threads de-interleave it into the polyphase planes (LDS.128 + 4 STS, both short
// latency), and as soon as the staging buffer has been consumed the NEXT tile's copy is issued, so it
// lands while stages A, B and C of the current tile run.  Same arithmetic and tile geometry as above
// (hbf_stage), therefore bit-identical output.
// ---------------------------------------------------------------------------------------------
template <int MA, int MB, int MC, int PRESET, int OB, int CTAS>
__global__ void __launch_bounds__(DEC_NT, CTAS) decim8_tma_kernel(const DecimParams p, const int ntiles)
{
    using GE = DecGeom<MA, MB, MC, OB>;
    extern __shared__ __align__(16) float smem[];
    float* stg = smem;                      // GE::NX floats, 16-byte aligned
    float* xe = stg + GE::NX;
    float* xo = xe + DEC_P * GE::SX;
    float* ae = xo + DEC_P * GE::SX;
    float* ao = ae + DEC_P * GE::SA;
    float* be = ao + DEC_P * GE::SA;
    float* bo = be + DEC_P * GE::SB;
    uint64_t* bar = reinterpret_cast<uint64_t*>(bo + DEC_P * GE::SB);  // (all counts above are even)

    const int tid = threadIdx.x;
    if (tid == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // tile t covers outputs [m1 - (t+1) OB, m1 - t OB): counted down from the top, so that every tile is full
    // size and only the lowest one is clipped by the store guard
    // The lowest tile starts up to OB - 1 outputs below m0, i.e. its x range may begin before the carry buffer
    // does; that part only feeds outputs the store guard discards, so it is simply not copied.
    auto issue = [&](int t) {
        const long long g = 8 * (p.m1 - (long long)t * OB) - GE::NX;
        long long skip = p.src.carry_start - g;
        skip = skip < 0 ? 0 : (skip > GE::NX ? GE::NX : skip);
        ring_issue(p.src, g + skip, GE::NX - (int)skip, stg + skip, bar);
    };
    int tile = blockIdx.x;
    if (tid == 0 && tile < ntiles) issue(tile);
    if (p.cc.n) carry_job(p.src, p.cc);  // while the first tile is in flight
    const long long lo = p.m0 > p.drain ? p.m0 : p.drain;
    for (unsigned it = 0; tile < ntiles; tile += gridDim.x, ++it) {
        const long long mhi = p.m1 - (long long)tile * OB;
        const long long c_base = mhi - OB;
        mbar_wait(bar, it & 1u);
        // ---- de-interleave the staged tile into the polyphase planes (as in the tiled kernel) ----
        {
            const float4* __restrict__ s4 = reinterpret_cast<const float4*>(stg);
            constexpr int NV = GE::NX / 4;
#pragma unroll 4
            for (int v = tid; v < NV; v += DEC_NT) {
                const float4 f = s4[v];
                const int pos = 2 * (v & 3) * GE::SX + (v >> 2);
                xe[pos] = f.x;
                xo[pos] = f.y;
                xe[pos + GE::SX] = f.z;
                xo[pos + GE::SX] = f.w;
            }
        }
        __syncthreads();  // planes complete; staging buffer consumed
        if (tid == 0 && tile + (int)gridDim.x < ntiles) issue(tile + (int)gridDim.x);
        hbf_stage<MA, GE::SX, GE::SA, GE::NX / 2 - GE::NA, false, PRESET, 2>(xe, xo, GE::NA, ae, ao, nullptr, 0, 0);
        __syncthreads();
        hbf_stage<MB, GE::SA, GE::SB, GE::NA / 2 - GE::NB, false, PRESET, 1>(ae, ao, GE::NB, be, bo, nullptr, 0, 0);
        __syncthreads();
        const int rel_lo = lo > c_base ? (int)(lo - c_base) : 0;
        hbf_stage<MC, GE::SB, GE::SB, GE::NB / 2 - OB, true, PRESET, 0>(be, bo, OB, nullptr, nullptr,
                                                                        p.out_fresh + (c_base - p.drain - p.out_split),
                                                                        rel_lo, OB, c_base - p.drain - p.out_split, p.out_cap);
        // no barrier needed here: the next tile's de-interleave only writes xe/xo (last read before the
        // barrier after stage A), its stage A writes ae/ao (last read before the barrier after stage B), and
        // its stage B writes be/bo after two more barriers
    }
}

// ---------------------------------------------------------------------------------------------
// K3, fifth generation (default): persistent CTAs, stage A reads the contiguous TMA-staged tile itself.
//
// The TMA-staged kernel above spends 510 of its 1866 shared-memory wavefronts per 960-output tile (hbf140) on
// reading the staging buffer back and de-interleaving it into polyphase planes, only so that stage A can read
// unit-stride planes.  Here each thread computes DIR_P = 18 consecutive stage-A outputs from a window of the raw tile
// read with LDS.128: run w starts at 16-byte chunk 9w of the staging buffer, so at every step the lanes of a quarter
// warp sit on chunks 9w + k, whose bank groups (w + k) mod 8 are distinct -- an odd lane stride in chunks makes
// lane-contiguous windows conflict-free with no padding and no swizzle.  The runs cover NRUN * 18 >= NA outputs; the
// lowest D of them lie below the tile's stage-A range, are computed from samples that may not even have been copied
// (below the carry buffer) and are not stored, so the tile geometry, its halo and the host's carry are those of
// DecGeom.  Two staging buffers: tile t + gridDim.x is copied into the other one when tile t starts.  Stages B and C
// are hbf_stage as everywhere, and every output is hbf_outputs' expression: bit-identical to the kernels above.
// ---------------------------------------------------------------------------------------------
constexpr int DIR_P = 18;  // stage-A outputs per run; P = 2 mod 4 makes the lane stride P/2 chunks odd

__device__ __forceinline__ float4 lds128(const float4* p)
{
    float4 v;
    asm volatile("ld.volatile.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(smem_u32(p)) : "memory");
    return v;
}

constexpr int floor4(int v) { return v >= 0 ? v / 4 * 4 : -((3 - v) / 4 * 4); }

template <int MA, int MB, int MC, int OB>
struct DirectGeom {
    using GE = DecGeom<MA, MB, MC, OB>;
    static constexpr int P = DIR_P;
    static constexpr int NRUN = (GE::NA + P - 1) / P;  // runs per tile (one per thread at most)
    static constexpr int D = NRUN * P - GE::NA;        // outputs of run 0 below the tile's stage-A range: not stored
    static constexpr int REL0 = GE::NX / 2 - GE::NA;   // as in hbf_stage: odd-plane index of output j is j + REL0
    // Relative to the tile's x_base = 8 mhi - NX: run 0's first odd sample (output -D, window element 0) is at F; the
    // staging buffer starts at the 16-byte chunk holding it and ends with the tile, NXS samples
    static constexpr int F = 2 * (REL0 - 2 * MA + 1 - D) + 1;
    static constexpr int XB = floor4(F);
    static constexpr int NXS = GE::NX - XB;
    static constexpr int NW = 2 * MA + P - 1;                         // odd samples per run window
    static constexpr int W0 = F - XB;                                 // window element i = window sample W0 + 2i
    static constexpr int C0 = 2 * (REL0 - MA + 1 - D) - XB;           // centre of output q = window sample C0 + 2q
    static constexpr int WCH = (W0 + 2 * (NW - 1)) / 4 + 1;           // LDS.128 per run window
    // stage-B input planes: polyphase by 8 like hbf_stage's, phase stride = 3 mod 32 (no stride makes the stage-A
    // stores of lane-consecutive runs conflict-free; with this one about two thirds of them are 2-way)
    static constexpr int SA = (GE::NA / 2 / DEC_P + 1 - 3 + 31) / 32 * 32 + 3;
    static constexpr int SMEM_FLOATS = 2 * NXS + 2 * DEC_P * (SA + GE::SB);
    static_assert(NXS % 4 == 0 && XB <= 0 && W0 >= 0 && C0 >= 0, "staging geometry");
    static_assert((P / 2) * (NRUN - 1) + WCH <= NXS / 4, "the last run's window ends inside the staging buffer");
    static_assert(C0 + 2 * (P - 1) < 4 * WCH, "centre samples inside the window");
    static_assert(NRUN <= DEC_NT && D % 2 == 0 && D < P, "one run per thread; runs start at even outputs");
    static_assert(SA >= (GE::NA / 2 + DEC_P - 1) / DEC_P, "stage-B planes hold NA / 2 samples each");
};

template <int MA, int MB, int MC, int OB>
constexpr size_t decim_direct_smem_bytes()
{
    return (size_t)DirectGeom<MA, MB, MC, OB>::SMEM_FLOATS * sizeof(float) + 16;
}

template <int MA, int MB, int MC, int PRESET, int OB, int CTAS>
__global__ void __launch_bounds__(DEC_NT, CTAS) decim8_direct_kernel(const DecimParams p, const int ntiles)
{
    using GE = DecGeom<MA, MB, MC, OB>;
    using DG = DirectGeom<MA, MB, MC, OB>;
    constexpr int P = DG::P;
    extern __shared__ __align__(16) float smem[];
    float* stg = smem;                      // two staging buffers of DG::NXS floats, 16-byte aligned
    float* ae = stg + 2 * DG::NXS;
    float* ao = ae + DEC_P * DG::SA;
    float* be = ao + DEC_P * DG::SA;
    float* bo = be + DEC_P * GE::SB;
    uint64_t* bar = reinterpret_cast<uint64_t*>(bo + DEC_P * GE::SB);  // one per staging buffer (all counts above are even)

    const int tid = threadIdx.x;
    if (tid == 0) {
        mbar_init(bar, 1);
        mbar_init(bar + 1, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // tiles as in decim8_tma_kernel; samples below the carry buffer are not copied (they only feed discarded outputs)
    auto issue = [&](int t, int b) {
        const long long g = 8 * (p.m1 - (long long)t * OB) - DG::NXS;
        long long skip = p.src.carry_start - g;
        skip = skip < 0 ? 0 : (skip > DG::NXS ? DG::NXS : skip);
        ring_issue(p.src, g + skip, DG::NXS - (int)skip, stg + b * DG::NXS + skip, bar + b);
    };
    int tile = blockIdx.x;
    if (tid == 0 && tile < ntiles) issue(tile, 0);
    if (p.cc.n) carry_job(p.src, p.cc);  // while the first tile is in flight
    const long long lo = p.m0 > p.drain ? p.m0 : p.drain;
    for (unsigned it = 0; tile < ntiles; tile += gridDim.x, ++it) {
        const long long mhi = p.m1 - (long long)tile * OB;
        const long long c_base = mhi - OB;
        const unsigned b = it & 1u;
        // the other buffer was last read by stage A of the previous tile, two barriers ago
        if (tid == 0 && tile + (int)gridDim.x < ntiles) issue(tile + (int)gridDim.x, (int)(b ^ 1u));
        mbar_wait(bar + b, (it >> 1) & 1u);
        // ---- stage A: run w = stage-A outputs j = P w - D + q, q < P, from the staged tile ----
        for (int w = tid; w < DG::NRUN; w += DEC_NT) {
            const float4* __restrict__ s4 = reinterpret_cast<const float4*>(stg + b * DG::NXS) + (P / 2) * w;
            SSPSD_ASSERT((P / 2) * w + DG::WCH <= DG::NXS / 4);
            // whole chunks even where only the odd samples are used: a scalar LDS at a lane stride of 36 floats would
            // be a 4-way bank conflict, so the loads are kept as LDS.128 explicitly
            float4 v[DG::WCH];
#pragma unroll
            for (int k = 0; k < DG::WCH; ++k) v[k] = lds128(s4 + k);
            auto sample = [&](int s) {
                const float4& c = v[s >> 2];
                return (s & 3) == 0 ? c.x : (s & 3) == 1 ? c.y : (s & 3) == 2 ? c.z : c.w;
            };
            float2 wp[MA + P / 2];
#pragma unroll
            for (int i = 0; i < DG::NW; ++i) {
                const float x = sample(DG::W0 + 2 * i);
                if (i & 1) wp[i >> 1].y = x; else wp[i >> 1].x = x;
            }
            float y[P];
            hbf_outputs<MA, P, PRESET, 2>(wp, [&](int q) { return sample(DG::C0 + 2 * q); }, y);
            // output j (even: plane ae, odd: ao) has plane index j >> 1 = (P/2) w + (q - D) >> 1
#pragma unroll
            for (int q = 0; q < P; ++q) {
                if (q >= DG::D || w > 0) {
                    const int r = (P / 2) * w + ((q - DG::D) >> 1);
                    SSPSD_ASSERT(r >= 0 && r < GE::NA / 2);
                    ((q & 1) ? ao : ae)[(r & (DEC_P - 1)) * DG::SA + (r >> DEC_LP)] = y[q];
                }
            }
        }
        __syncthreads();
        hbf_stage<MB, DG::SA, GE::SB, GE::NA / 2 - GE::NB, false, PRESET, 1>(ae, ao, GE::NB, be, bo, nullptr, 0, 0);
        __syncthreads();
        const int rel_lo = lo > c_base ? (int)(lo - c_base) : 0;
        hbf_stage<MC, GE::SB, GE::SB, GE::NB / 2 - OB, true, PRESET, 0>(be, bo, OB, nullptr, nullptr,
                                                                        p.out_fresh + (c_base - p.drain - p.out_split),
                                                                        rel_lo, OB, c_base - p.drain - p.out_split, p.out_cap);
        // no barrier needed here: the next tile's stage A writes ae/ao (last read by stage B, before the barrier
        // after it) and its stage B writes be/bo after the barrier that follows stage A
    }
}

// ---------------------------------------------------------------------------------------------
// K3, third generation: persistent CTAs, the NEXT tile's samples are scattered straight into a second set
// of polyphase x planes by 4-byte cp.async (LDGSTS) while stages A, B, C of the current tile run.
//
// The TMA-staged kernel above removed the exposed LDG latency but paid for it in the resource that bounds
// the decimator, the shared-memory data pipe: one extra LDS.128 per four samples to read the staging buffer
// back (+19 % wavefronts; 0.250 -> 0.234 ms per 200e6 samples only).  A 4-byte cp.async writes its element
// where the de-interleaving STS would have, with no register round trip and no second pass: lane l of an
// instruction takes element 32 k + l of the tile (one 128-byte line of global memory), which lands in plane
// (e|o), phase (l >> 1) & 7, offset +(l >> 4): with the odd planes shifted by two banks the 32 lanes hit 32
// distinct banks, one wavefront per instruction -- the same shared-memory traffic as the tiled kernel's
// stores, issued a whole tile ahead.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async4(float* dst, const float* src, bool valid)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(valid ? 4 : 0) : "memory");
}

template <int MA, int MB, int MC, int PRESET, int OB, int CTAS>
__global__ void __launch_bounds__(DEC_NT, CTAS) decim8_async_kernel(const DecimParams p, const int ntiles)
{
    using GE = DecGeom<MA, MB, MC, OB>;
    constexpr int XP = 2 * DEC_P * GE::SX + 4;  // floats per x plane set: even planes, +2 banks, odd planes, pad
    static_assert(GE::NX % DEC_NT == 0 || true, "");
    extern __shared__ __align__(16) float smem[];
    float* xs = smem;                       // two plane sets
    float* ae = xs + 2 * XP;
    float* ao = ae + DEC_P * GE::SA;
    float* be = ao + DEC_P * GE::SA;
    float* bo = be + DEC_P * GE::SB;

    const int tid = threadIdx.x;
    // element i = DEC_NT k + tid of a tile: plane index r = i >> 1 = (DEC_NT / 2) k + (tid >> 1); DEC_NT / 2 is a
    // multiple of 8, so the phase r & 7 is per thread and the offset r >> 3 advances by DEC_NT / 16 per k
    const int dst0 = ((tid >> 1) & 7) * GE::SX + (tid >> 4) + ((tid & 1) ? DEC_P * GE::SX + 2 : 0);
    auto issue = [&](int t, float* planes) {
        const long long g0 = 8 * (p.m1 - (long long)t * OB) - GE::NX;  // first sample of the tile (multiple of 8)
        float* d = planes + dst0;
        if (g0 >= p.src.split) {
            const float* __restrict__ gx = p.src.fresh + (g0 - p.src.split) + tid;
#pragma unroll 8
            for (int k = 0; k < GE::NX / DEC_NT; ++k) cp_async4(d + (DEC_NT / 16) * k, gx + DEC_NT * k, true);
            if (GE::NX % DEC_NT != 0 && tid < GE::NX % DEC_NT)
                cp_async4(d + (DEC_NT / 16) * (GE::NX / DEC_NT), gx + DEC_NT * (GE::NX / DEC_NT), true);
        } else {
            // first tiles of a batch: carry / fresh per element, zeros before the carry buffer begins
            for (int k = 0; DEC_NT * k + tid < GE::NX; ++k) {
                const long long g = g0 + DEC_NT * k + tid;
                const float* src = g >= p.src.split ? p.src.fresh + (g - p.src.split)
                                                    : p.src.carry + (g >= p.src.carry_start ? g - p.src.carry_start : 0);
                cp_async4(d + (DEC_NT / 16) * k, src, g >= p.src.carry_start);
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    int tile = blockIdx.x;
    if (tile < ntiles) issue(tile, xs);
    const long long lo = p.m0 > p.drain ? p.m0 : p.drain;
    for (unsigned it = 0; tile < ntiles; tile += gridDim.x, ++it) {
        float* xe = xs + (it & 1u) * XP;
        float* xo = xe + DEC_P * GE::SX + 2;
        const int next = tile + (int)gridDim.x;
        // the other plane set was last read by stage A of the previous tile, two barriers ago
        if (next < ntiles) {
            issue(next, xs + ((it + 1u) & 1u) * XP);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();  // every thread's copies of this tile have landed
        const long long mhi = p.m1 - (long long)tile * OB;
        const long long c_base = mhi - OB;
        hbf_stage<MA, GE::SX, GE::SA, GE::NX / 2 - GE::NA, false, PRESET, 2>(xe, xo, GE::NA, ae, ao, nullptr, 0, 0);
        __syncthreads();
        hbf_stage<MB, GE::SA, GE::SB, GE::NA / 2 - GE::NB, false, PRESET, 1>(ae, ao, GE::NB, be, bo, nullptr, 0, 0);
        __syncthreads();
        const int rel_lo = lo > c_base ? (int)(lo - c_base) : 0;
        hbf_stage<MC, GE::SB, GE::SB, GE::NB / 2 - OB, true, PRESET, 0>(be, bo, OB, nullptr, nullptr,
                                                                        p.out_fresh + (c_base - p.drain - p.out_split),
                                                                        rel_lo, OB, c_base - p.drain - p.out_split, p.out_cap);
    }
}

// ---------------------------------------------------------------------------------------------
// K3, fourth generation: persistent CTAs, the NEXT tile prefetched into REGISTERS.
//
// Shared-memory wavefronts per 960-output tile of the TMA-staged kernel (hbf140): TMA write of the staging buffer 255,
// LDS.128 read-back 255, de-interleaving STS 255, stage A 528, stage B 344, stage C 229 -- the staging round trip is
// 27 % of the traffic of the pipe that bounds the kernel (73 % busy).  Here every thread issues its 8 LDG.128 of tile
// t + 1 right after the barrier that completes the planes of tile t, keeps them in 32 registers while stages A and B of
// tile t run (~1.3 us, longer than an HBM round trip), and scatters them into the x planes -- free since stage A --
// before stage C: no staging buffer, no exposed load latency.  Same arithmetic and tile geometry (hbf_stage):
// bit-identical output.
// ---------------------------------------------------------------------------------------------
template <int MA, int MB, int MC, int PRESET, int OB, int CTAS>
__global__ void __launch_bounds__(DEC_NT, CTAS) decim8_pf_kernel(const DecimParams p, const int ntiles)
{
    using GE = DecGeom<MA, MB, MC, OB>;
    extern __shared__ __align__(16) float smem[];
    float* xe = smem;
    float* xo = xe + DEC_P * GE::SX;
    float* ae = xo + DEC_P * GE::SX;
    float* ao = ae + DEC_P * GE::SA;
    float* be = ao + DEC_P * GE::SA;
    float* bo = be + DEC_P * GE::SB;
    constexpr int NV = GE::NX / 4;
    constexpr int NR = (NV + DEC_NT - 1) / DEC_NT;
    const int tid = threadIdx.x;
    float4 pf[NR];
    // tile t covers outputs [m1 - (t+1) OB, m1 - t OB) (counted down from the top; only the lowest one is clipped by
    // the store guard, and what it would read below the carry buffer is zero: ld_stream4)
    auto fetch = [&](int t) {
        const long long g = 8 * (p.m1 - (long long)t * OB) - GE::NX;
        if (g >= p.src.split) {
            const float4* __restrict__ gx = reinterpret_cast<const float4*>(p.src.fresh + (g - p.src.split));
#pragma unroll
            for (int u = 0; u < NR; ++u) {
                const int v = u * DEC_NT + tid;
                if (v < NV) {
                    SSPSD_ASSERT(g + 4ll * v + 4 <= p.src.end);
                    pf[u] = __ldg(gx + v);
                }
            }
        } else {
#pragma unroll
            for (int u = 0; u < NR; ++u) {
                const int v = u * DEC_NT + tid;
                if (v < NV) pf[u] = ld_stream4(p.src, g + 4ll * v);
            }
        }
    };
    auto scatter = [&]() {
#pragma unroll
        for (int u = 0; u < NR; ++u) {
            const int v = u * DEC_NT + tid;
            if (v < NV) {
                const int pos = 2 * (v & 3) * GE::SX + (v >> 2);
                xe[pos] = pf[u].x;
                xo[pos] = pf[u].y;
                xe[pos + GE::SX] = pf[u].z;
                xo[pos + GE::SX] = pf[u].w;
            }
        }
    };
    int tile = blockIdx.x;
    if (tile < ntiles) {
        fetch(tile);
        scatter();
    }
    const long long lo = p.m0 > p.drain ? p.m0 : p.drain;
    for (; tile < ntiles; tile += gridDim.x) {
        const long long mhi = p.m1 - (long long)tile * OB;
        const long long c_base = mhi - OB;
        const int next = tile + (int)gridDim.x;
        __syncthreads();  // x planes of this tile complete; stage C of the previous tile has read be/bo
        if (next < ntiles) fetch(next);
        hbf_stage<MA, GE::SX, GE::SA, GE::NX / 2 - GE::NA, false, PRESET, 2>(xe, xo, GE::NA, ae, ao, nullptr, 0, 0);
        __syncthreads();
        hbf_stage<MB, GE::SA, GE::SB, GE::NA / 2 - GE::NB, false, PRESET, 1>(ae, ao, GE::NB, be, bo, nullptr, 0, 0);
        __syncthreads();
        if (next < ntiles) scatter();  // the x planes were last read by stage A, two barriers ago
        const int rel_lo = lo > c_base ? (int)(lo - c_base) : 0;
        hbf_stage<MC, GE::SB, GE::SB, GE::NB / 2 - OB, true, PRESET, 0>(be, bo, OB, nullptr, nullptr,
                                                                        p.out_fresh + (c_base - p.drain - p.out_split),
                                                                        rel_lo, OB, c_base - p.drain - p.out_split, p.out_cap);
    }
}

template <int MA, int MB, int MC, int OB>
constexpr size_t decim_pf_smem_bytes()
{
    return (size_t)DecGeom<MA, MB, MC, OB>::SMEM_FLOATS * sizeof(float);
}

template <int MA, int MB, int MC, int OB>
constexpr size_t decim_async_smem_bytes()
{
    using GE = DecGeom<MA, MB, MC, OB>;
    return (size_t)(2 * (2 * DEC_P * GE::SX + 4) + 2 * DEC_P * (GE::SA + GE::SB)) * sizeof(float);
}

template <int MA, int MB, int MC, int OB>
constexpr size_t decim_tma_smem_bytes()
{
    using GE = DecGeom<MA, MB, MC, OB>;
    return (size_t)(GE::NX + GE::SMEM_FLOATS) * sizeof(float) + 16;
}

// ---------------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------------
// dst[i] = stream[g0 + i], i < n  (builds the next batch's carry buffer = [g0, L)); additionally the
// last `head_n` (< 4) samples, [L - head_n, L), are written to the head of the buffer the NEXT batch's
// fresh samples go to, so that buffer is valid from floor4(L) on and aligned 128-bit loads never have
// to straddle the carry/fresh boundary.
__global__ void carry_copy_kernel(StreamSrc src, long long g0, int n, float* __restrict__ dst,
                                  float* __restrict__ head_dst, int head_n, int dst_cap)
{
    carry_job(src, CarryJob{g0, n, head_n, dst, head_dst, dst_cap});
}

}  // namespace sspsd
