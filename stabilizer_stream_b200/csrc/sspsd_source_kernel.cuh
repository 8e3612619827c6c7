// sspsd_source_kernel.cuh -- synthetic sources generated on the device (no PCIe on the input side).
//
// Replaces the reference's Data::Noise and Data::Dsm generators (src/source.rs:66-73, 104-134):
//   noise: uniform (0,1) -> (u - 0.5) * sqrt(12), folded through |noise| cascaded first-order
//          integrators (noise < 0) or differentiators (noise > 0) whose state persists between calls;
//   dsm:   sine of a wrapping u32 phase accumulator quantised by a MASH-1-1-1 modulator.
// The reference runs both one sample at a time.  Here the recurrences are evaluated as scans:
// every thread owns SRC_SPT consecutive samples, a run of samples is summarised as the affine map
// it applies to the recurrence state, and maps compose associatively.  For both recurrences the
// matrix part is lower-triangular Toeplitz, i.e. a truncated polynomial in the shift z:
//   integrators   s' = (1 + z) s + e0 x          (real arithmetic, carried in f64)
//   MASH-1-1-1    a' = (1 + z + z^2)(a + e0 x)   (arithmetic mod 2^32, exact)
// so a map is 2K numbers and composing two maps is a K x K truncated polynomial product.
// Three launches per generate(): per-block summaries -> one-CTA scan of the summaries -> apply.
// The uniform stream is Philox4x32-10 (counter = sample index / 4, key = seed), so any thread can
// produce any sample; differentiators need no scan at all (y depends on K+1 neighbouring inputs).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sspsd {

constexpr int SRC_SPT = 16;                  // samples per thread
constexpr int SRC_NT = 256;                  // threads per CTA
constexpr int SRC_SPB = SRC_SPT * SRC_NT;    // samples per CTA
constexpr int SRC_MAX_ORDER = 4;             // integrator orders with a device path (f64 binomials)
constexpr int SRC_MAX_DIFF = 8;              // differentiator orders with a device path

struct SourceParams {
    unsigned long long pos;  // stream index of out[0]
    unsigned long long n;    // samples to produce
    uint32_t key0, key1;     // Philox key (seed)
    uint32_t ftw;            // dsm frequency tuning word
    int order;               // differentiator order of the white/diff kernel
    float scale;             // sqrt(12) in f32
    float* out;
    void* state;             // K values of the recurrence state (in/out, device)
    void* block_elems;       // per-block summaries
    void* block_init;        // per-block initial states
    unsigned int nblocks;
};

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 with counter (c0, c1, 0, 0)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t k0, uint32_t k1, uint32_t (&r)[4])
{
    uint32_t c2 = 0, c3 = 0;
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
        c1 = l1;
        c3 = l0;
        c0 = n0;
        c2 = n2;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    r[0] = c0; r[1] = c1; r[2] = c2; r[3] = c3;
}

// uniform in (0,1) from 23 random bits, then zero mean / unit RMS (source.rs:109)
__device__ __forceinline__ float noise_from_bits(uint32_t r, float scale)
{
    float u = __fsub_rn(__uint_as_float(0x3f800000u | (r >> 9)), 1.0f - 5.9604645e-8f);
    return __fmul_rn(__fsub_rn(u, 0.5f), scale);
}

// white sample of stream index i (0 for i < 0, the reference's zero-initialised state)
__device__ __forceinline__ void noise_block(long long q, const SourceParams& p, float (&x)[4])
{
    if (q < 0) {
        x[0] = x[1] = x[2] = x[3] = 0.f;
        return;
    }
    uint32_t r[4];
    philox4x32_10((uint32_t)q, (uint32_t)((unsigned long long)q >> 32), p.key0, p.key1, r);
#pragma unroll
    for (int j = 0; j < 4; ++j) x[j] = noise_from_bits(r[j], p.scale);
}

// the DSM input word of stream index i (source.rs:119-126); the sine goes through double so that
// the host restatement and the device agree bit for bit
__device__ __forceinline__ uint32_t dsm_input(unsigned long long i, uint32_t ftw)
{
    const float M = 4294967296.0f;
    uint32_t x = 1u + (uint32_t)i * ftw;
    float arg = __fmul_rn((float)x, 6.28318530717958647692f / M);
    float sn = (float)sin((double)arg);
    float v = __fmul_rn(__fadd_rn(__fmul_rn(sn, 0.4999f), 0.5f), M);
    return (uint32_t)v;
}

// ---------------------------------------------------------------------------------------------
// White noise and differentiated noise: one Philox block (4 samples) per thread
// ---------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256) source_diff_kernel(SourceParams p)
{
    const long long q0 = (long long)(p.pos >> 2);
    const long long nq = (long long)((p.pos + p.n + 3) >> 2) - q0;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < nq; t += (long long)gridDim.x * blockDim.x) {
        const long long q = q0 + t;
        // v[8..11] = samples 4q..4q+3, v[0..7] = the eight before them
        float v[12] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        {
            float x[4];
            noise_block(q, p, x);
#pragma unroll
            for (int j = 0; j < 4; ++j) v[8 + j] = x[j];
            if (p.order > 0) {
                noise_block(q - 1, p, x);
#pragma unroll
                for (int j = 0; j < 4; ++j) v[4 + j] = x[j];
            }
            if (p.order > 4) {
                noise_block(q - 2, p, x);
#pragma unroll
                for (int j = 0; j < 4; ++j) v[j] = x[j];
            }
        }
        // level k value at index n is level k-1 at n minus level k-1 at n-1; every level is 0 for n < 0
        for (int k = 0; k < p.order; ++k) {
#pragma unroll
            for (int j = 11; j >= 1; --j)
                if (j > k) v[j] = __fsub_rn(v[j], v[j - 1]);
        }
        const long long i0 = 4 * q - (long long)p.pos;  // position of v[8] in out
        if (i0 >= 0 && i0 + 4 <= (long long)p.n && ((reinterpret_cast<uintptr_t>(p.out + i0) & 15) == 0)) {
            *reinterpret_cast<float4*>(p.out + i0) = make_float4(v[8], v[9], v[10], v[11]);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (i0 + j >= 0 && i0 + j < (long long)p.n) p.out[i0 + j] = v[8 + j];
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Affine maps of a K-state recurrence with Toeplitz matrix part
// ---------------------------------------------------------------------------------------------
template <typename T, int K>
struct Aff {
    T c[K];  // matrix = sum_d c[d] z^d, c[0] == 1
    T v[K];  // offset
};

template <typename T, int K>
__device__ __forceinline__ Aff<T, K> aff_identity()
{
    Aff<T, K> e;
#pragma unroll
    for (int i = 0; i < K; ++i) {
        e.c[i] = (T)(i == 0);
        e.v[i] = (T)0;
    }
    return e;
}

// state after applying map m to state s
template <typename T, int K>
__device__ __forceinline__ void aff_apply(const Aff<T, K>& m, const T (&s)[K], T (&r)[K])
{
#pragma unroll
    for (int i = 0; i < K; ++i) {
        T acc = m.v[i];
#pragma unroll
        for (int d = 0; d <= i; ++d) acc += m.c[d] * s[i - d];
        r[i] = acc;
    }
}

// map "a, then b"
template <typename T, int K>
__device__ __forceinline__ Aff<T, K> aff_then(const Aff<T, K>& a, const Aff<T, K>& b)
{
    Aff<T, K> r;
#pragma unroll
    for (int i = 0; i < K; ++i) {
        T c = (T)0, v = b.v[i];
#pragma unroll
        for (int d = 0; d <= i; ++d) {
            c += b.c[d] * a.c[i - d];
            v += b.c[d] * a.v[i - d];
        }
        r.c[i] = c;
        r.v[i] = v;
    }
    return r;
}

__device__ __forceinline__ double shfl_up_t(double x, int d) { return __shfl_up_sync(0xffffffffu, x, d); }
__device__ __forceinline__ uint32_t shfl_up_t(uint32_t x, int d) { return __shfl_up_sync(0xffffffffu, x, d); }

// inclusive scan over the 256 threads of the CTA (thread order = stream order); returns this
// thread's exclusive prefix, and the CTA total in *total.  smem: 8 maps.
template <typename T, int K>
__device__ __forceinline__ Aff<T, K> block_exclusive(Aff<T, K> e, Aff<T, K>* smem, Aff<T, K>* total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    Aff<T, K> inc = e;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        Aff<T, K> o;
#pragma unroll
        for (int i = 0; i < K; ++i) {
            o.c[i] = shfl_up_t(inc.c[i], d);
            o.v[i] = shfl_up_t(inc.v[i], d);
        }
        if (lane >= d) inc = aff_then(o, inc);
    }
    if (lane == 31) smem[warp] = inc;
    __syncthreads();
    Aff<T, K> pre = aff_identity<T, K>();
    for (int w = 0; w < warp; ++w) pre = aff_then(pre, smem[w]);
    if (total) {
        Aff<T, K> tot = pre;
        for (int w = warp; w < SRC_NT / 32; ++w) tot = aff_then(tot, smem[w]);
        *total = tot;
    }
    // exclusive = warps before, then lanes before
    Aff<T, K> exc;
#pragma unroll
    for (int i = 0; i < K; ++i) {
        exc.c[i] = shfl_up_t(inc.c[i], 1);
        exc.v[i] = shfl_up_t(inc.v[i], 1);
    }
    if (lane == 0) exc = aff_identity<T, K>();
    __syncthreads();
    return aff_then(pre, exc);
}

// ---------------------------------------------------------------------------------------------
// Recurrence models
// ---------------------------------------------------------------------------------------------
// |noise| cascaded integrators, the fold at source.rs:110-114 with diff == false:
//   (x, s) = (s, x + s): each level outputs its old state and adds its input to it
template <int K_>
struct IntegratorModel {
    using T = double;
    using In = float;
    static constexpr int K = K_;
    __device__ static void load(const SourceParams& p, unsigned long long i0, int cnt, In (&x)[SRC_SPT])
    {
        // the run starts at stream index i0, which need not be aligned to a Philox block
        long long q = (long long)(i0 >> 2);
        int lane = (int)(i0 & 3);
        float b[4];
        noise_block(q, p, b);
#pragma unroll
        for (int j = 0; j < SRC_SPT; ++j) {
            const float bl = lane == 0 ? b[0] : (lane == 1 ? b[1] : (lane == 2 ? b[2] : b[3]));
            x[j] = j < cnt ? bl : 0.f;
            if (++lane == 4) {
                lane = 0;
                ++q;
                if (j + 1 < cnt) noise_block(q, p, b);
            }
        }
    }
    __device__ static void step(T (&s)[K], In xin, T& out)
    {
        T in = (T)xin;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            T t = s[k];
            s[k] = t + in;
            in = t;
        }
        out = in;
    }
    __device__ static void poly_step(T (&c)[K])
    {
#pragma unroll
        for (int d = K - 1; d >= 1; --d) c[d] += c[d - 1];  // times (1 + z)
    }
    struct Ctx {};
    __device__ static void ctx_init(Ctx&, const SourceParams&, const T (&)[K], unsigned long long) {}
    __device__ static float emit(Ctx&, const T (&)[K], In, T out) { return (float)out; }
};

// MASH-1-1-1 over three wrapping u32 accumulators; y = c1 + D c2 + D^2 c3 (D = first difference)
struct MashModel {
    using T = uint32_t;
    using In = uint32_t;
    static constexpr int K = 3;
    __device__ static void load(const SourceParams& p, unsigned long long i0, int cnt, In (&x)[SRC_SPT])
    {
#pragma unroll
        for (int j = 0; j < SRC_SPT; ++j) x[j] = j < cnt ? dsm_input(i0 + j, p.ftw) : 0u;
    }
    __device__ static void step(T (&a)[K], In x, T& out)
    {
        a[0] += x;
        a[1] += a[0];
        a[2] += a[1];
        out = 0;
    }
    __device__ static void poly_step(T (&c)[K])
    {
        c[2] += c[1] + c[0];  // times (1 + z + z^2)
        c[1] += c[0];
    }
    struct Ctx {
        int c2z, c3z, c3zz;
    };
    // carries of the two samples before i0, recovered by running the (invertible) recurrence backwards
    __device__ static void ctx_init(Ctx& cx, const SourceParams&, const T (&a)[K], unsigned long long i0)
    {
        cx.c2z = cx.c3z = cx.c3zz = 0;
        if (i0 == 0) return;
        T b0 = a[0], b1 = a[1], b2 = a[2];
        cx.c2z = b1 < b0;
        cx.c3z = b2 < b1;
        if (i0 == 1) return;
        b2 -= b1;
        b1 -= b0;
        cx.c3zz = b2 < b1;
    }
    __device__ static float emit(Ctx& cx, const T (&a)[K], In x, T)
    {
        // a holds the accumulators after this sample: a carry out of t = old + in shows as t < in
        int c1 = a[0] < x, c2 = a[1] < a[0], c3 = a[2] < a[1];
        int y = c1 + (c2 - cx.c2z) + (c3 - 2 * cx.c3z + cx.c3zz);
        cx.c2z = c2;
        cx.c3zz = cx.c3z;
        cx.c3z = c3;
        return (float)y - 0.5f;  // source.rs:127
    }
};

// the map applied by cnt samples starting from a zero state
template <typename Mo>
__device__ __forceinline__ Aff<typename Mo::T, Mo::K> run_summary(const typename Mo::In (&x)[SRC_SPT], int cnt)
{
    using T = typename Mo::T;
    Aff<T, Mo::K> e = aff_identity<T, Mo::K>();
#pragma unroll
    for (int j = 0; j < SRC_SPT; ++j) {
        if (j < cnt) {
            T out;
            Mo::step(e.v, x[j], out);
            Mo::poly_step(e.c);
        }
    }
    return e;
}

// pass 1: summary of every CTA's SRC_SPB samples
template <typename Mo>
__global__ void __launch_bounds__(SRC_NT) source_reduce_kernel(SourceParams p)
{
    using T = typename Mo::T;
    using E = Aff<T, Mo::K>;
    __shared__ E sm[SRC_NT / 32];
    const unsigned long long off = (unsigned long long)blockIdx.x * SRC_SPB + (unsigned long long)threadIdx.x * SRC_SPT;
    long long left = (long long)p.n - (long long)off;
    const int cnt = left <= 0 ? 0 : (left < SRC_SPT ? (int)left : SRC_SPT);
    typename Mo::In x[SRC_SPT];
    Mo::load(p, p.pos + off, cnt, x);
    E e = run_summary<Mo>(x, cnt);
    E total;
    (void)block_exclusive<T, Mo::K>(e, sm, &total);
    if (threadIdx.x == 0) reinterpret_cast<E*>(p.block_elems)[blockIdx.x] = total;
}

// pass 2 (one CTA): initial state of every CTA, and the state after the whole call
template <typename Mo>
__global__ void __launch_bounds__(SRC_NT) source_scan_kernel(SourceParams p)
{
    using T = typename Mo::T;
    using E = Aff<T, Mo::K>;
    __shared__ E sm[SRC_NT / 32];
    T s0[Mo::K];
#pragma unroll
    for (int i = 0; i < Mo::K; ++i) s0[i] = reinterpret_cast<const T*>(p.state)[i];
    E carry = aff_identity<T, Mo::K>();
    for (unsigned int base = 0; base < p.nblocks; base += SRC_NT) {
        const unsigned int b = base + threadIdx.x;
        E e = b < p.nblocks ? reinterpret_cast<const E*>(p.block_elems)[b] : aff_identity<T, Mo::K>();
        E total;
        E exc = block_exclusive<T, Mo::K>(e, sm, &total);
        if (b < p.nblocks) {
            E m = aff_then(carry, exc);
            T s[Mo::K];
            aff_apply(m, s0, s);
#pragma unroll
            for (int i = 0; i < Mo::K; ++i) reinterpret_cast<T*>(p.block_init)[(size_t)b * Mo::K + i] = s[i];
        }
        carry = aff_then(carry, total);
    }
    __syncthreads();  // every thread has read the old state
    if (threadIdx.x == 0) {
        T s[Mo::K];
        aff_apply(carry, s0, s);
#pragma unroll
        for (int i = 0; i < Mo::K; ++i) reinterpret_cast<T*>(p.state)[i] = s[i];
    }
}

// pass 3: every thread replays its samples from its true initial state
template <typename Mo>
__global__ void __launch_bounds__(SRC_NT) source_apply_kernel(SourceParams p)
{
    using T = typename Mo::T;
    using E = Aff<T, Mo::K>;
    __shared__ E sm[SRC_NT / 32];
    __shared__ float tile[SRC_SPB + SRC_SPB / 32];
    const unsigned long long boff = (unsigned long long)blockIdx.x * SRC_SPB;
    const unsigned long long off = boff + (unsigned long long)threadIdx.x * SRC_SPT;
    long long left = (long long)p.n - (long long)off;
    const int cnt = left <= 0 ? 0 : (left < SRC_SPT ? (int)left : SRC_SPT);
    typename Mo::In x[SRC_SPT];
    Mo::load(p, p.pos + off, cnt, x);
    E e = run_summary<Mo>(x, cnt);
    E exc = block_exclusive<T, Mo::K>(e, sm, nullptr);
    T sb[Mo::K], s[Mo::K];
#pragma unroll
    for (int i = 0; i < Mo::K; ++i) sb[i] = reinterpret_cast<const T*>(p.block_init)[(size_t)blockIdx.x * Mo::K + i];
    aff_apply(exc, sb, s);
    typename Mo::Ctx cx;
    Mo::ctx_init(cx, p, s, p.pos + off);
#pragma unroll
    for (int j = 0; j < SRC_SPT; ++j) {
        if (j < cnt) {
            T out;
            Mo::step(s, x[j], out);
            const int i = threadIdx.x * SRC_SPT + j;
            tile[i + (i >> 5)] = Mo::emit(cx, s, x[j], out);
        }
    }
    __syncthreads();
    long long bleft = (long long)p.n - (long long)boff;
    const int bcnt = bleft < SRC_SPB ? (int)bleft : SRC_SPB;
    for (int i = threadIdx.x; i < bcnt; i += SRC_NT) p.out[boff + i] = tile[i + (i >> 5)];
}

}  // namespace sspsd
