// sspsd_device.cuh -- device-side building blocks shared by the sm_100a kernels.
//
// Replaces, on the device, the per-stage hot loop of the reference (src/psd.rs:196-269):
//   Detrend::apply (psd.rs:75-113) -> rustfft Fft::process (psd.rs:213) -> |X|^2 accumulate
//   (psd.rs:228-233) -> idsp HBF_DEC_CASCADE decimate-by-8 (psd.rs:246-253).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

// Bounds-checking build (make libsspsd_bounds.so, -DSSPSD_BOUNDS): every global-memory index a kernel forms from
// run-time bookkeeping is asserted on the device against the extents the host passes along.  compute-sanitizer is
// closed on the pool these kernels were developed on (profiles/r02_compute_sanitizer_refused.log), so this build
// -- run over the parity, fuzz and group tests (tests/test_gpu_bounds.py) -- is the memory-safety evidence.
#ifdef SSPSD_BOUNDS
#include <assert.h>
#define SSPSD_ASSERT(c) assert(c)
#else
#define SSPSD_ASSERT(c) ((void)0)
#endif

namespace sspsd {

// ---------------------------------------------------------------------------------------------
// A stage's input stream as seen by a kernel: logical sample index g (0 = first sample the stage
// ever received) lives in `carry` for g < split (history + pending samples kept from earlier
// batches, zeros for g < 0) and in `fresh` for g >= split (this batch).  carry_start and split
// are multiples of 4 and both bases are 16-byte aligned, so aligned float4 groups never straddle.
// ---------------------------------------------------------------------------------------------
struct StreamSrc {
    const float* carry;
    const float* fresh;
    long long carry_start;
    long long split;
    long long end;  // one past the last valid sample (stream length after this batch)
};

// The next batch's carry buffer of the stage being decimated, built by the decimator launch itself when there is one
// (one launch less per stage and batch): dst[i] = stream[g0 + i], i < n; the last head_n (< 4) samples also go to the head
// of the buffer the next batch's fresh samples will be written to (see carry_copy_kernel).  n == 0: nothing to do.
struct CarryJob {
    long long g0;
    int n, head_n;
    float* dst;
    float* head_dst;
    int dst_cap;
};

__device__ __forceinline__ float4 ld_stream4(const StreamSrc& s, long long g)
{
    SSPSD_ASSERT(g + 4 <= s.end && (g & 3) == 0);
    if (g >= s.split)
        return __ldg(reinterpret_cast<const float4*>(s.fresh + (g - s.split)));
    if (g >= s.carry_start)
        return *reinterpret_cast<const float4*>(s.carry + (g - s.carry_start));
    return make_float4(0.f, 0.f, 0.f, 0.f);
}

__device__ __forceinline__ float ld_stream1(const StreamSrc& s, long long g)
{
    SSPSD_ASSERT(g < s.end);
    if (g >= s.split)
        return __ldg(s.fresh + (g - s.split));
    if (g >= s.carry_start)
        return s.carry[g - s.carry_start];
    return 0.f;
}

// EWMA weight of segment j of a launch of p.nseg segments (psd.rs:218-233), the product of the factors applied after
// it: g_s^(nseg-1-max(j,jb)) * (j < jb && jb < nseg ? g_first : 1), in f64; boxcar: jb >= nseg.  The 0.25 folds the
// /2 of the real-input (or two-for-one) split.  p: any stage kernel's parameters; its fields are read where they are
// used (pow is a call: a value read before it would be held across it).
template <class P>
__device__ __forceinline__ float ewma_weight(const P& p, int j)
{
    const int n_s = p.nseg - 1 - max(j, p.jb);
    double w = 1.0;
    if (n_s > 0) w = pow((double)p.g_s, (double)n_s);
    if (j < p.jb && p.jb < p.nseg) w *= (double)p.g_first;
    return (float)(0.25 * w);
}

// ---------------------------------------------------------------------------------------------
// TMA bulk copies (cp.async.bulk, SASS UBLKCP) completing on an mbarrier
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// 1-D TMA bulk copy global -> shared, completion reported to an mbarrier in bytes
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// issue the copies of stream samples [g, g + n) into dst (n multiple of 4, g multiple of 4)
__device__ __forceinline__ void ring_issue(const StreamSrc& s, long long g, int n, float* dst, uint64_t* bar)
{
    SSPSD_ASSERT(n >= 0 && (n & 3) == 0 && (g & 3) == 0 && (n == 0 || (g >= s.carry_start && g + n <= s.end)));
    mbar_expect_tx(bar, (uint32_t)n * 4u);
    long long nc = s.split - g;  // samples that live in the carry
    if (nc > n) nc = n;
    if (nc > 0) {
        bulk_g2s(dst, s.carry + (g - s.carry_start), (uint32_t)nc * 4u, bar);
    } else {
        nc = 0;
    }
    if (nc < n) bulk_g2s(dst + nc, s.fresh + (g + nc - s.split), (uint32_t)(n - nc) * 4u, bar);
}

// ---------------------------------------------------------------------------------------------
// FFT plan: an N-point real segment is transformed as an M = N/2 point complex FFT of
// z[n] = x[2n] + i x[2n+1] followed by the real-input split.  The complex FFT is an in-place
// decimation-in-frequency transform in shared memory; every thread owns 8 points per pass.
// Radices: as many radix-8 passes as fit, one radix-2 or radix-4 pass for the remainder, and a
// final radix-4 pass on 4 contiguous points (which is where the split pairs k with M-k).
// ---------------------------------------------------------------------------------------------
template <int LOG2N>
struct Plan {
    static constexpr int N = 1 << LOG2N;
    static constexpr int LOG2M = LOG2N - 1;
    static constexpr int M = 1 << LOG2M;
    static constexpr int TPS = M / 8;                      // threads per segment
    static constexpr int NT = TPS > 256 ? TPS : 256;       // threads per CTA
    static constexpr int G = NT / TPS;                     // segments in flight per CTA
    static constexpr int REM = LOG2M - 2;
    static constexpr int A = REM / 3;                      // radix-8 passes
    static constexpr int EXTRA = REM % 3;                  // log2 radix of the odd pass (0 = none)
    static constexpr int P = A + (EXTRA ? 1 : 0) + 1;      // total passes
    static constexpr int K = M / 4;                        // butterflies of the last pass
    static constexpr int WS = M + 4 * (M / 32);            // padded floats per re/im plane
    static_assert(LOG2N >= 6 && LOG2N <= 13, "supported FFT sizes: 64..8192");
    static_assert(A >= 1, "first pass must be radix 8");

    __host__ __device__ static constexpr int log2radix(int p) { return p < A ? 3 : (p == P - 1 ? 2 : EXTRA); }
    // log2 of the element stride inside pass p's butterflies (= size of the sub-transforms left)
    __host__ __device__ static constexpr int log2stride(int p)
    {
        int s = LOG2M;
        for (int q = 0; q <= p; ++q) s -= log2radix(q);
        return s;
    }
    // log2 of the weight of pass p's output digit in the frequency index
    __host__ __device__ static constexpr int log2weight(int p)
    {
        int s = 0;
        for (int q = 0; q < p; ++q) s += log2radix(q);
        return s;
    }
};

// padded shared-memory position of complex element i (4 floats of padding per 32 elements)
__device__ __forceinline__ int ws_pos(int i) { return i + ((i >> 5) << 2); }

// ---------------------------------------------------------------------------------------------
// Complex arithmetic on packed FP32 pairs.  sm_100 has FADD2 / FMUL2 / FFMA2: one instruction, one
// issue slot, both halves of a 64-bit register pair, with per-operand swizzle (LO_HI), per-half
// negation and 32-bit broadcast modifiers, so a complex value (re, im) adds in ONE instruction,
// multiplies in TWO, and a multiplication by +-i is free (it folds into the consumer's operand
// modifiers).  The PSD kernels are bound by instruction issue (profiles/r01_ncu_summary.md), and
// three quarters of their instructions were scalar FADD/FMUL/FFMA on exactly such pairs.
// The FP32 pipe does the same number of lane operations either way (tools/microbench/ffma2.cu).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
// a - i b  and  a + i b
__device__ __forceinline__ float2 cadd_mi(float2 a, float2 b) { return __fadd2_rn(a, make_float2(b.y, -b.x)); }
__device__ __forceinline__ float2 cadd_pi(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.y, b.x)); }

__device__ __forceinline__ float2 cmul(float2 a, float2 b)
{
    // (a.x b.x - a.y b.y, a.x b.y + a.y b.x) = b.x (a.x, a.y) + b.y (-a.y, a.x): the pair operand takes the
    // swizzle + half negation (FFMA2 -Ra.LO_HI.NP), b's halves are 32-bit broadcasts (or immediates)
    float2 t = __fmul2_rn(a, make_float2(b.x, b.x));
    return __ffma2_rn(make_float2(-a.y, a.x), make_float2(b.y, b.y), t);
}

// in-place forward DFTs, v[k] = sum_t v[t] exp(-2 pi i t k / R)
__device__ __forceinline__ void dft2(float2& a, float2& b)
{
    float2 t = a;
    a = cadd(t, b);
    b = csub(t, b);
}

__device__ __forceinline__ void dft4(float2& c0, float2& c1, float2& c2, float2& c3)
{
    float2 e0 = cadd(c0, c2), e1 = csub(c0, c2), f0 = cadd(c1, c3), d = csub(c1, c3);
    c0 = cadd(e0, f0);
    c2 = csub(e0, f0);
    c1 = cadd_mi(e1, d);  // e1 - i (c1 - c3)
    c3 = cadd_pi(e1, d);
}

template <int R>
__device__ __forceinline__ void butterfly(float2 (&v)[R])
{
    if constexpr (R == 2) {
        dft2(v[0], v[1]);
    } else if constexpr (R == 4) {
        dft4(v[0], v[1], v[2], v[3]);
    } else {
        static_assert(R == 8, "radix");
        constexpr float h = 0.70710678118654752440f;
        float2 a0 = cadd(v[0], v[4]), a1 = cadd(v[1], v[5]), a2 = cadd(v[2], v[6]), a3 = cadd(v[3], v[7]);
        float2 b0 = csub(v[0], v[4]), d1 = csub(v[1], v[5]), d2 = csub(v[2], v[6]), d3 = csub(v[3], v[7]);
        float2 b1 = cmul(d1, make_float2(h, -h));    // * (1 - i)/sqrt2
        float2 b3 = cmul(d3, make_float2(-h, -h));   // * (-1 - i)/sqrt2
        dft4(a0, a1, a2, a3);
        // dft4 of (b0, b1, -i d2, b3) with the -i folded into the operand modifiers
        float2 e0 = cadd_mi(b0, d2), e1 = cadd_pi(b0, d2), f0 = cadd(b1, b3), d = csub(b1, b3);
        v[0] = a0; v[2] = a1; v[4] = a2; v[6] = a3;
        v[1] = cadd(e0, f0);
        v[5] = csub(e0, f0);
        v[3] = cadd_mi(e1, d);
        v[7] = cadd_pi(e1, d);
    }
}

// Radix-8 forward DFT of 8 contiguous points that arrive as separate re / im planes (two LDS.128 per
// plane).  The planes are consumed as packed pairs of NEIGHBOURING points ((re0,re1), (re2,re3), ...),
// which needs no register shuffling: the distance-4 stage and the even half's distance-2 stage are
// element-wise packed operations; everything that mixes the halves of a pair (the distance-1 stage, the
// odd half with its W8 twiddles) is scalar and reads the halves in place.  The 1/sqrt2 of W8 and W8^3
// is applied by the FFMAs of the last stage.
__device__ __forceinline__ void dft8_planes(float4 r0, float4 r1, float4 i0, float4 i1, float2 (&z)[8])
{
    constexpr float h = 0.70710678118654752440f;
    const float2 zr01 = make_float2(r0.x, r0.y), zr23 = make_float2(r0.z, r0.w), zr45 = make_float2(r1.x, r1.y),
                 zr67 = make_float2(r1.z, r1.w);
    const float2 zi01 = make_float2(i0.x, i0.y), zi23 = make_float2(i0.z, i0.w), zi45 = make_float2(i1.x, i1.y),
                 zi67 = make_float2(i1.z, i1.w);
    // distance 4: a_t = z_t + z_{t+4}, d_t = z_t - z_{t+4}
    const float2 ar01 = cadd(zr01, zr45), ar23 = cadd(zr23, zr67), ai01 = cadd(zi01, zi45), ai23 = cadd(zi23, zi67);
    const float2 dr01 = csub(zr01, zr45), dr23 = csub(zr23, zr67), di01 = csub(zi01, zi45), di23 = csub(zi23, zi67);
    // even outputs: DFT4 of a.  distance 2 packed: c_t = a_t + a_{t+2}, e_t = a_t - a_{t+2}; distance 1 scalar
    const float2 cr = cadd(ar01, ar23), ci = cadd(ai01, ai23), er = csub(ar01, ar23), ei = csub(ai01, ai23);
    z[0] = make_float2(cr.x + cr.y, ci.x + ci.y);
    z[4] = make_float2(cr.x - cr.y, ci.x - ci.y);
    z[2] = make_float2(er.x + ei.y, ei.x - er.y);  // e0 - i e1
    z[6] = make_float2(er.x - ei.y, ei.x + er.y);
    // odd outputs: DFT4 of (d0, d1 W8, -i d2, d3 W8^3) with W8 = h (1 - i), W8^3 = h (-1 - i)
    const float f0r = dr01.x + di23.x, f0i = di01.x - dr23.x;   // d0 + (-i d2)
    const float g0r = dr01.x - di23.x, g0i = di01.x + dr23.x;   // d0 - (-i d2)
    const float p = dr01.y + di01.y, q = di01.y - dr01.y;       // d1 (1 - i)
    const float r = di23.y - dr23.y, s = di23.y + dr23.y;       // d3 (-1 - i) = (r, -s)
    const float f1r = p + r, f1i = q - s, g1r = p - r, g1i = q + s;
    z[1] = make_float2(fmaf(h, f1r, f0r), fmaf(h, f1i, f0i));
    z[5] = make_float2(fmaf(-h, f1r, f0r), fmaf(-h, f1i, f0i));
    z[3] = make_float2(fmaf(h, g1i, g0r), fmaf(-h, g1r, g0i));  // g0 - i h g1
    z[7] = make_float2(fmaf(-h, g1i, g0r), fmaf(h, g1r, g0i));
}

// Radix-4 forward DFT of 4 contiguous points given as one LDS.128 per plane (same idea as dft8_planes)
__device__ __forceinline__ void dft4_planes(float4 r, float4 i, float2 (&z)[4])
{
    const float2 zr01 = make_float2(r.x, r.y), zr23 = make_float2(r.z, r.w);
    const float2 zi01 = make_float2(i.x, i.y), zi23 = make_float2(i.z, i.w);
    const float2 cr = cadd(zr01, zr23), ci = cadd(zi01, zi23), er = csub(zr01, zr23), ei = csub(zi01, zi23);
    z[0] = make_float2(cr.x + cr.y, ci.x + ci.y);
    z[2] = make_float2(cr.x - cr.y, ci.x - ci.y);
    z[1] = make_float2(er.x + ei.y, ei.x - er.y);  // e0 - i e1
    z[3] = make_float2(er.x - ei.y, ei.x + er.y);
}

}  // namespace sspsd
