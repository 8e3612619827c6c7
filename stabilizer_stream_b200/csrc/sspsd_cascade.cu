// sspsd_cascade.cu -- host-side state machine + kernel launches of the device cascade.
// See sspsd_cascade.cuh for the bookkeeping model and include/sspsd.h for the reference citations.
#if defined(__x86_64__)
#include <emmintrin.h>
#endif

#include "sspsd_cascade.cuh"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "sspsd_decim_kernel.cuh"
#include "sspsd_stage_kernel.cuh"
#include "sspsd_stage_kernel_r16.cuh"
#include "sspsd_stage_kernel_ring.cuh"
#include "sspsd_stage_kernel_w16.cuh"

namespace sspsd {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
const char* last_error() { return g_err.c_str(); }

bool cuda_ok(cudaError_t e, const char* what)
{
    if (e == cudaSuccess)
        return true;
    set_error(std::string(what) + ": " + cudaGetErrorString(e));
    return false;
}

namespace {

inline long long floor4(long long v) { return v & ~3ll; }

// ---- kernel dispatch over the FFT size ----
template <int LOG2N>
int launch_stage_t(const StageParams& p, int grid, cudaStream_t s)
{
    size_t smem = stage_smem_bytes<LOG2N>(p.T, p.hop);
    psd_stage_kernel<LOG2N><<<grid, Plan<LOG2N>::NT, smem, s>>>(p);
    return cuda_ok(cudaGetLastError(), "psd_stage_kernel launch") ? SSPSD_OK : SSPSD_ECUDA;
}

template <int LOG2N>
int prepare_stage_t(int hop, int budget_bytes, int* tmax)
{
    using PL = Plan<LOG2N>;
    int t = 256;
    while (t > 1 && (long long)stage_smem_bytes<LOG2N>(t, hop) > budget_bytes)
        --t;
    if ((long long)stage_smem_bytes<LOG2N>(t, hop) > budget_bytes) {
        set_error("FFT size does not fit in shared memory");
        return SSPSD_EINVAL;
    }
    *tmax = t;
    (void)PL::N;
    if (!cuda_ok(cudaFuncSetAttribute(psd_stage_kernel<LOG2N>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)stage_smem_bytes<LOG2N>(t, hop)),
                 "cudaFuncSetAttribute(psd_stage_kernel)"))
        return SSPSD_ECUDA;
    return SSPSD_OK;
}

#define SSPSD_FOR_SIZES(X) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13)

// K2 variant for N = 4096 (A/B switch for profiling): SSPSD_K2 = r8 | r16 | ring (default ring:
// persistent TMA-ring kernel for the Hann window, tiled radix-16 kernel for the rectangular one)
// (read when a handle is created and stored in it: no process-wide mutable state)
int k2_variant_from_env()
{
    const char* e = getenv("SSPSD_K2");
    std::string m = e ? e : "ring";
    return m == "r8" ? 0 : m == "r16" ? 1 : m == "ring1" ? 3 : m == "ring1x5" ? 4 : 2;
}

int launch_stage(int log2n, bool r16, const StageParams& p, int grid, cudaStream_t s)
{
    if (log2n == 12 && r16) {
        psd_stage_kernel_r16<<<grid, R16::NT, stage_r16_smem_bytes(p.T, p.hop), s>>>(p);
        return cuda_ok(cudaGetLastError(), "psd_stage_kernel_r16 launch") ? SSPSD_OK : SSPSD_ECUDA;
    }
    switch (log2n) {
#define X(L) \
    case L:  \
        return launch_stage_t<L>(p, grid, s);
        SSPSD_FOR_SIZES(X)
#undef X
    default:
        return SSPSD_EINVAL;
    }
}

int prepare_stage(int log2n, bool r16, int hop, int* tmax, int* nt)
{
    if (log2n == 12 && r16) {
        int t = 64;
        while (t > 1 && (long long)stage_r16_smem_bytes(t, hop) > 112 * 1024) --t;
        *tmax = t;
        *nt = R16::NT;
        SSPSD_CUDA(cudaFuncSetAttribute(psd_stage_kernel_r16, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)stage_r16_smem_bytes(t, hop)));
        SSPSD_CUDA(cudaFuncSetAttribute(psd_stage_kernel_ring, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)stage_ring_smem_bytes(RingCfg::MAX_W)));
        SSPSD_CUDA(cudaFuncSetAttribute(psd_stage_kernel_ring1, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)stage_ring_smem_bytes(1024, 1, RingCfg::RING1, false)));
        SSPSD_CUDA(cudaFuncSetAttribute(psd_stage_kernel_ring1x5, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)stage_ring_smem_bytes(384, 1, 3, false)));
        return SSPSD_OK;
    }
    if (log2n == 9)
        SSPSD_CUDA(cudaFuncSetAttribute(psd_stage_kernel_w16, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)stage_w16_smem_bytes(W16::MAX_T)));
    switch (log2n) {
#define X(L)                                                                   \
    case L:                                                                    \
        *nt = Plan<L>::NT;                                                     \
        return prepare_stage_t<L>(hop, Plan<L>::NT <= 256 ? 100 * 1024 : 200 * 1024, tmax);
        SSPSD_FOR_SIZES(X)
#undef X
    default:
        set_error("n_fft must be a power of two in 64..8192");
        return SSPSD_EINVAL;
    }
}

template <int MA, int MB, int MC, int PRESET>
int launch_decim_t(const DecimParams& p, int grid, cudaStream_t s)
{
    using GE = DecGeom<MA, MB, MC>;
    decim8_kernel<MA, MB, MC, PRESET><<<grid, DEC_NT, GE::SMEM_FLOATS * sizeof(float), s>>>(p);
    return cuda_ok(cudaGetLastError(), "decim8_kernel launch") ? SSPSD_OK : SSPSD_ECUDA;
}

// persistent TMA-staged decimator (default; SSPSD_K3=tiled selects the first-generation kernel)
template <int MA, int MB, int MC, int PRESET, int OB, int CTAS>
int launch_decim_tma_t(const DecimParams& p, long long n_out, int num_sms, cudaStream_t s)
{
    const int ntiles = (int)((n_out + OB - 1) / OB);
    const int grid = std::min(ntiles, num_sms * CTAS);
    decim8_tma_kernel<MA, MB, MC, PRESET, OB, CTAS><<<grid, DEC_NT, decim_tma_smem_bytes<MA, MB, MC, OB>(), s>>>(p, ntiles);
    return cuda_ok(cudaGetLastError(), "decim8_tma_kernel launch") ? SSPSD_OK : SSPSD_ECUDA;
}

template <int MA, int MB, int MC, int PRESET, int OB, int CTAS>
int launch_decim_async_t(const DecimParams& p, long long n_out, int num_sms, cudaStream_t s)
{
    const int ntiles = (int)((n_out + OB - 1) / OB);
    const int grid = std::min(ntiles, num_sms * CTAS);
    decim8_async_kernel<MA, MB, MC, PRESET, OB, CTAS><<<grid, DEC_NT, decim_async_smem_bytes<MA, MB, MC, OB>(), s>>>(p, ntiles);
    return cuda_ok(cudaGetLastError(), "decim8_async_kernel launch") ? SSPSD_OK : SSPSD_ECUDA;
}

template <int MA, int MB, int MC, int PRESET, int OB, int CTAS>
int launch_decim_pf_t(const DecimParams& p, long long n_out, int num_sms, cudaStream_t s)
{
    const int ntiles = (int)((n_out + OB - 1) / OB);
    const int grid = std::min(ntiles, num_sms * CTAS);
    decim8_pf_kernel<MA, MB, MC, PRESET, OB, CTAS><<<grid, DEC_NT, decim_pf_smem_bytes<MA, MB, MC, OB>(), s>>>(p, ntiles);
    return cuda_ok(cudaGetLastError(), "decim8_pf_kernel launch") ? SSPSD_OK : SSPSD_ECUDA;
}

int decim_halo(int preset)
{
    return preset == SSPSD_HBF_98 ? DecGeom<3, 6, 15>::HALO : DecGeom<5, 10, 23>::HALO;
}

// Constant-memory tap tables and kernel attributes are per device and set once per device; handles may be
// created concurrently on different threads (one per GPU), so the "once" is a mutex-guarded flag and the
// staging arrays are locals.
int upload_taps_once(int device)
{
    static std::mutex mu;
    static bool done[64] = {false};
    std::lock_guard<std::mutex> lock(mu);
    if (device < 64 && done[device])
        return SSPSD_OK;
    static_assert(sizeof(sspsd_hbf_taps) == sizeof(float) * SSPSD_HBF_NPRESET * 3 * SSPSD_HBF_MAXTAPS, "tap table");
    {
        // rows padded to an even length (8-byte aligned pairs) + a copy shifted by one tap
        float t0[SSPSD_HBF_NPRESET][3][SSPSD_HBF_MAXTAPS + 1], t1[SSPSD_HBF_NPRESET][3][SSPSD_HBF_MAXTAPS + 1];
        for (int p = 0; p < SSPSD_HBF_NPRESET; ++p)
            for (int s = 0; s < 3; ++s)
                for (int i = 0; i <= SSPSD_HBF_MAXTAPS; ++i) {
                    t0[p][s][i] = i < SSPSD_HBF_MAXTAPS ? sspsd_hbf_taps[p][s][i] : 0.f;
                    t1[p][s][i] = i + 1 < SSPSD_HBF_MAXTAPS ? sspsd_hbf_taps[p][s][i + 1] : 0.f;
                }
        SSPSD_CUDA(cudaMemcpyToSymbol(c_hbf_taps, t0, sizeof(t0)));
        SSPSD_CUDA(cudaMemcpyToSymbol(c_hbf_taps_sh, t1, sizeof(t1)));
    }
    SSPSD_CUDA(cudaFuncSetAttribute(decim8_kernel<5, 10, 23, SSPSD_HBF_140>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)(DecGeom<5, 10, 23>::SMEM_FLOATS * sizeof(float))));
    SSPSD_CUDA(cudaFuncSetAttribute(decim8_kernel<3, 6, 15, SSPSD_HBF_98>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)(DecGeom<3, 6, 15>::SMEM_FLOATS * sizeof(float))));
    SSPSD_CUDA(cudaFuncSetAttribute(decim8_async_kernel<5, 10, 23, SSPSD_HBF_140, 960, 2>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)decim_async_smem_bytes<5, 10, 23, 960>()));
    SSPSD_CUDA(cudaFuncSetAttribute(decim8_async_kernel<5, 10, 23, SSPSD_HBF_140, 640, 3>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)decim_async_smem_bytes<5, 10, 23, 640>()));
    SSPSD_CUDA(cudaFuncSetAttribute(decim8_async_kernel<3, 6, 15, SSPSD_HBF_98, 960, 2>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)decim_async_smem_bytes<3, 6, 15, 960>()));
    SSPSD_CUDA(cudaFuncSetAttribute(decim8_async_kernel<3, 6, 15, SSPSD_HBF_98, 640, 3>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)decim_async_smem_bytes<3, 6, 15, 640>()));
    SSPSD_CUDA(cudaFuncSetAttribute(decim8_tma_kernel<5, 10, 23, SSPSD_HBF_140, 960, 2>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)decim_tma_smem_bytes<5, 10, 23, 960>()));
    SSPSD_CUDA(cudaFuncSetAttribute(decim8_tma_kernel<5, 10, 23, SSPSD_HBF_140, 640, 3>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)decim_tma_smem_bytes<5, 10, 23, 640>()));
    SSPSD_CUDA(cudaFuncSetAttribute(decim8_tma_kernel<3, 6, 15, SSPSD_HBF_98, 960, 2>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)decim_tma_smem_bytes<3, 6, 15, 960>()));
    SSPSD_CUDA(cudaFuncSetAttribute(decim8_tma_kernel<3, 6, 15, SSPSD_HBF_98, 640, 3>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)decim_tma_smem_bytes<3, 6, 15, 640>()));
    SSPSD_CUDA(cudaFuncSetAttribute(decim8_tma_kernel<5, 10, 23, SSPSD_HBF_140, 768, 3>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)decim_tma_smem_bytes<5, 10, 23, 768>()));
    SSPSD_CUDA(cudaFuncSetAttribute(decim8_tma_kernel<3, 6, 15, SSPSD_HBF_98, 768, 3>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)decim_tma_smem_bytes<3, 6, 15, 768>()));
    SSPSD_CUDA(cudaFuncSetAttribute(decim8_pf_kernel<5, 10, 23, SSPSD_HBF_140, 960, 2>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)decim_pf_smem_bytes<5, 10, 23, 960>()));
    SSPSD_CUDA(cudaFuncSetAttribute(decim8_pf_kernel<5, 10, 23, SSPSD_HBF_140, 640, 3>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)decim_pf_smem_bytes<5, 10, 23, 640>()));
    SSPSD_CUDA(cudaFuncSetAttribute(decim8_pf_kernel<3, 6, 15, SSPSD_HBF_98, 960, 2>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)decim_pf_smem_bytes<3, 6, 15, 960>()));
    SSPSD_CUDA(cudaFuncSetAttribute(decim8_pf_kernel<3, 6, 15, SSPSD_HBF_98, 640, 3>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)decim_pf_smem_bytes<3, 6, 15, 640>()));
    if (device < 64)
        done[device] = true;
    return SSPSD_OK;
}

EwmaPlan ewma_plan(uint32_t count, uint32_t avg, uint64_t S)
{
    EwmaPlan e{};
    uint32_t steady = avg + 1u;  // count in the steady state (wraps only for avg == u32::MAX, unused then)
    e.g_s = (float)avg / (float)steady;
    uint64_t jb;
    if (count > avg) {
        jb = 0;
        e.g_first = (float)avg / (float)count;
    } else {
        jb = (uint64_t)avg - count + 1;
        e.g_first = e.g_s;
    }
    if (jb >= S) {
        e.jb = (int)S;
        e.total = 1.0f;
        e.count_after = (uint32_t)(count + S);
    } else {
        e.jb = (int)jb;
        double t = (double)e.g_first;
        uint64_t n_s = S - 1 - jb;
        if (n_s > 0)
            t *= std::pow((double)e.g_s, (double)n_s);
        e.total = (float)t;
        e.count_after = steady;
    }
    return e;
}

}  // namespace

int hbf_info(int hbf, uint32_t* drain, uint32_t* halo)
{
    if (hbf != SSPSD_HBF_98 && hbf != SSPSD_HBF_140) return SSPSD_EINVAL;
    if (drain) *drain = (uint32_t)sspsd_hbf_drain[hbf];
    if (halo) *halo = (uint32_t)decim_halo(hbf);
    return SSPSD_OK;
}

// =============================================================================================
Cascade::~Cascade()
{
    if (n_ == 0)
        return;
    DeviceGuard g(cfg_.device);
    if (stream_)
        cudaStreamSynchronize(stream_);
    if (deep_stream_) cudaStreamSynchronize(deep_stream_);
    if (psd_stream_) cudaStreamSynchronize(psd_stream_);
    free_stages(false);
    cudaFree(d_win_);
    cudaFree(d_twM_);
    cudaFree(d_twN_);
    cudaFree(d_acc_);
    cudaFree(d_in_[0]);
    cudaFree(d_in_[1]);
    cudaFree(d_sink_);
    cudaFree(d_tail_);
    cudaFree(d_part_[0]);
    cudaFree(d_part_[1]);
    if (h_stage_[0]) cudaFreeHost(h_stage_[0]);
    if (h_stage_[1]) cudaFreeHost(h_stage_[1]);
    if (h_acc_) cudaFreeHost(h_acc_);
    for (int i = 0; i < 2; ++i) {
        if (ev_copied_[i]) cudaEventDestroy(ev_copied_[i]);
        if (ev_free_[i]) cudaEventDestroy(ev_free_[i]);
        if (ev_stage_[i]) cudaEventDestroy(ev_stage_[i]);
    }
    if (ev_stage0_) cudaEventDestroy(ev_stage0_);
    if (ev_deep_) cudaEventDestroy(ev_deep_);
    if (ev_psd_join_) cudaEventDestroy(ev_psd_join_);
    if (psd_stream_) cudaStreamDestroy(psd_stream_);
    if (deep_stream_) cudaStreamDestroy(deep_stream_);
    if (copy_stream_) cudaStreamDestroy(copy_stream_);
    if (own_stream_ && stream_) cudaStreamDestroy(stream_);
}

int Cascade::init(const sspsd_config& cfg, uint32_t max_stages)
{
    cfg_ = cfg;
    uint32_t n = cfg.n_fft;
    if (n < 64 || n > 8192 || (n & (n - 1))) {
        set_error("n_fft must be a power of two in 64..8192");
        return SSPSD_EINVAL;
    }
    if (cfg.window != SSPSD_WINDOW_RECT && cfg.window != SSPSD_WINDOW_HANN) {
        set_error("unknown window");
        return SSPSD_EINVAL;
    }
    if (cfg.hbf != SSPSD_HBF_98 && cfg.hbf != SSPSD_HBF_140) {
        set_error("unknown half-band preset");
        return SSPSD_EINVAL;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        set_error("no CUDA device: this library has no CPU fallback");
        return SSPSD_ECUDA;
    }
    if (cfg.device < 0 || cfg.device >= ndev) {
        set_error("bad device ordinal");
        return SSPSD_EINVAL;
    }
    DeviceGuard g(cfg.device);
    if (!g.ok)
        return SSPSD_ECUDA;
    uint32_t l2 = 0;
    while ((1u << l2) < n) ++l2;
    log2n_ = l2;
    max_stages_ = std::min<uint32_t>(max_stages, SSPSD_MAX_STAGES);
    if (cfg_.max_batch == 0) cfg_.max_batch = 1ull << 28;
    if (cfg_.host_stage == 0) cfg_.host_stage = 1ull << 22;
    cfg_.max_batch = std::max<uint64_t>(cfg_.max_batch, 16ull * n);
    cfg_.max_batch = std::min<uint64_t>(cfg_.max_batch, 1ull << 30);

    // Window::rectangular / ::hann, psd.rs:24-55 (same f32 expression as the reference)
    std::vector<float> win(n);
    if (cfg.window == SSPSD_WINDOW_RECT) {
        std::fill(win.begin(), win.end(), 1.0f);
        win_ = {1.0f, 1.0f, 0};
    } else {
        const float pi = 3.14159265358979323846f;
        float df = pi / (float)n;
        for (uint32_t i = 0; i < n; ++i) {
            float s = sinf(df * (float)i);
            win[i] = s * s;
        }
        win_ = {0.25f, 1.5f, n / 2};
    }
    hop_ = n - win_.overlap;
    drain_ = sspsd_hbf_drain[cfg.hbf];
    int halo = decim_halo(cfg.hbf);
    hb_ = std::max<int>((int)win_.overlap, halo);
    hb_ = (hb_ + 7) & ~7;

    SSPSD_CUDA(cudaDeviceGetAttribute(&num_sms_, cudaDevAttrMultiProcessorCount, cfg.device));
    if (cfg.stream) {
        stream_ = (cudaStream_t)cfg.stream;
    } else {
        SSPSD_CUDA(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
        own_stream_ = true;
    }
    SSPSD_CUDA(cudaStreamCreateWithFlags(&copy_stream_, cudaStreamNonBlocking));
    // Stages >= deep_from_ (default 1; SSPSD_OVERLAP=k selects k, 0 disables) run on a second, high
    // priority stream: across consecutive process() calls their many small launches hide behind the
    // next batch's stage-0 kernels instead of adding their latency (176 -> 210 GS/s in bench.py; a
    // readout joins the streams, so nothing changes for a caller that reads out after every batch).
    const char* ov = getenv("SSPSD_OVERLAP");
    deep_from_ = ov ? (size_t)atoi(ov) : 1;
    if (max_stages_ > 1 && deep_from_ > 0 && !one_stream_) {
        // high priority: the small deep-stage grids should be scheduled ahead of the remaining stage-0 CTAs
        int lo_prio = 0, hi_prio = 0;
        SSPSD_CUDA(cudaDeviceGetStreamPriorityRange(&lo_prio, &hi_prio));
        SSPSD_CUDA(cudaStreamCreateWithPriority(&deep_stream_, cudaStreamNonBlocking, hi_prio));
        SSPSD_CUDA(cudaEventCreateWithFlags(&ev_stage0_, cudaEventDisableTiming));
        SSPSD_CUDA(cudaEventCreateWithFlags(&ev_deep_, cudaEventDisableTiming));
        // A deep stage's PSD kernel and its decimator only share their input, so the PSD kernels get a
        // stream of their own: the dependent chain a readout has to wait for is then decimator ->
        // decimator -> ... instead of PSD -> decimator -> carry copy per stage.
        const char* ps = getenv("SSPSD_PSD_STREAM");
        if (!ps || atoi(ps) != 0) {
            SSPSD_CUDA(cudaStreamCreateWithPriority(&psd_stream_, cudaStreamNonBlocking, hi_prio));
            SSPSD_CUDA(cudaEventCreateWithFlags(&ev_psd_join_, cudaEventDisableTiming));
        }
    }
    for (int i = 0; i < 2; ++i) {
        SSPSD_CUDA(cudaEventCreateWithFlags(&ev_copied_[i], cudaEventDisableTiming));
        SSPSD_CUDA(cudaEventCreateWithFlags(&ev_free_[i], cudaEventDisableTiming));
        SSPSD_CUDA(cudaEventCreateWithFlags(&ev_stage_[i], cudaEventDisableTiming));
    }
    int rc = upload_taps_once(cfg.device);
    if (rc) return rc;
    // measured (profiles/r02_variants*.jsonl): letting the deep stages' input pile up for a few batches makes their
    // kernels efficient (N = 512: 0.21 -> 0.13 ms of PSD-kernel time per 200e6-sample step, whole step 0.81 ->
    // 0.72 ms; N = 4096: neutral, their launches already hide inside the next batch's stage-0 kernels)
    defer_ = cfg_.deep_defer ? cfg_.deep_defer : (1ull << 26);
    if (const char* e = getenv("SSPSD_DEFER")) defer_ = strtoull(e, nullptr, 0);
    k2_variant_ = k2_variant_from_env();
    {
        // K3 variant (A/B switch): SSPSD_K3 = tiled | tma960 | tma640 | async960 | async640
        const char* e = getenv("SSPSD_K3");
        std::string m = e ? e : "tma960";
        k3_variant_ = m == "tiled" ? 0 : m == "tma960" ? 1 : m == "tma640" ? 2 : m == "async640" ? 4 : m == "pf960" ? 5 :
                      m == "pf640" ? 6 : m == "tma768" ? 7 : 3;
    }
    rc = prepare_stage((int)log2n_, k2_variant_ >= 1, (int)hop_, &tmax_, &nt_);
    if (rc) return rc;

    const uint32_t m = n / 2;
    std::vector<float2> twM(m), twN(m);
    for (uint32_t k = 0; k < m; ++k) {
        double a = -2.0 * M_PI * (double)k / (double)m;
        twM[k] = make_float2((float)std::cos(a), (float)std::sin(a));
        double b = -2.0 * M_PI * (double)k / (double)n;
        twN[k] = make_float2((float)std::cos(b), (float)std::sin(b));
    }
    acc_stride_ = (m + 1 + 63) & ~63u;
    SSPSD_CUDA(cudaMalloc(&d_win_, n * sizeof(float)));
    SSPSD_CUDA(cudaMalloc(&d_twM_, m * sizeof(float2)));
    SSPSD_CUDA(cudaMalloc(&d_twN_, m * sizeof(float2)));
    SSPSD_CUDA(cudaMalloc(&d_acc_, (size_t)SSPSD_MAX_STAGES * acc_stride_ * sizeof(float)));
    SSPSD_CUDA(cudaMemcpyAsync(d_win_, win.data(), n * sizeof(float), cudaMemcpyHostToDevice, stream_));
    SSPSD_CUDA(cudaMemcpyAsync(d_twM_, twM.data(), m * sizeof(float2), cudaMemcpyHostToDevice, stream_));
    SSPSD_CUDA(cudaMemcpyAsync(d_twN_, twN.data(), m * sizeof(float2), cudaMemcpyHostToDevice, stream_));
    SSPSD_CUDA(cudaMemsetAsync(d_acc_, 0, (size_t)SSPSD_MAX_STAGES * acc_stride_ * sizeof(float), stream_));
    SSPSD_CUDA(cudaMallocHost(&h_acc_, (size_t)SSPSD_MAX_STAGES * acc_stride_ * sizeof(float)));
    SSPSD_CUDA(cudaStreamSynchronize(stream_));  // the host vectors above go out of scope
    stages_.reserve(SSPSD_MAX_STAGES);
    n_ = n;
    return SSPSD_OK;
}

uint32_t Cascade::stage_avg(size_t i) const
{
    // (avg.count >> (DEPTH * i)).min(avg.limit), psd.rs:434,449
    unsigned sh = (unsigned)(SSPSD_DEPTH * i);
    uint32_t v = sh >= 32 ? 0u : (avg_.count >> sh);
    return std::min(v, avg_.limit);
}

int Cascade::add_stage()
{
    // get_or_add, psd.rs:445-453 + Psd::new, psd.rs:137-152
    if (stages_.size() >= SSPSD_MAX_STAGES) {
        set_error("too many stages");
        return SSPSD_EINVAL;
    }
    StageState st;
    const size_t cap = (size_t)hb_ + n_ + 16;
    cudaStream_t ss = stage_stream(stages_.size());
    if (!spare_.empty()) {
        // buffers of a stage released by reset(): reuse them (a reset is the GUI's Cmd::Reset; re-creating
        // every device buffer each time cost milliseconds)
        StageState old = spare_.back();
        spare_.pop_back();
        st.carry[0] = old.carry[0];
        st.carry[1] = old.carry[1];
        st.fresh[0] = old.fresh[0];
        st.fresh[1] = old.fresh[1];
        st.fresh_cap = old.fresh_cap;
        st.ev_read[0] = old.ev_read[0];
        st.ev_read[1] = old.ev_read[1];
        st.ev_in = old.ev_in;
        st.ev_psd[0] = old.ev_psd[0];
        st.ev_psd[1] = old.ev_psd[1];
    } else {
        SSPSD_CUDA(cudaMalloc(&st.carry[0], cap * sizeof(float)));
        SSPSD_CUDA(cudaMalloc(&st.carry[1], cap * sizeof(float)));
        for (int b = 0; b < 2; ++b) SSPSD_CUDA(cudaEventCreateWithFlags(&st.ev_read[b], cudaEventDisableTiming));
        for (int b = 0; b < 2; ++b) SSPSD_CUDA(cudaEventCreateWithFlags(&st.ev_psd[b], cudaEventDisableTiming));
        SSPSD_CUDA(cudaEventCreateWithFlags(&st.ev_in, cudaEventDisableTiming));
    }
    st.avg = single_stage_avg_set_ ? single_stage_avg_ : stage_avg(stages_.size());
    // zero history for g < 0: the decimator starts from HbfDec8::default() (psd.rs:141)
    SSPSD_CUDA(cudaMemsetAsync(st.carry[0], 0, cap * sizeof(float), ss));
    SSPSD_CUDA(cudaMemsetAsync(st.carry[1], 0, cap * sizeof(float), ss));
    st.carry_start = -(long long)hb_;
    // time-chunk mode: warm-up contamination propagates down the cascade (see seek())
    st.valid_from = stages_.empty() ? seek_pos_ : next_valid_from(stages_.back().valid_from);
    SSPSD_CUDA(cudaMemsetAsync(d_acc_ + stages_.size() * acc_stride_, 0, acc_stride_ * sizeof(float), ss));
    stages_.push_back(st);
    return SSPSD_OK;
}

int Cascade::ensure_fresh(StageState& st, size_t need, size_t reserve)
{
    if (need <= st.fresh_cap)
        return SSPSD_OK;
    // earlier batches may still be reading the old buffers; the head of fresh[fb] (copies of the carry tail,
    // written by the previous batch's carry_copy_kernel) and the samples accumulated there since the stage last
    // ran (deferred deep stages) have to survive the reallocation
    SSPSD_CUDA(cudaStreamSynchronize(stream_));
    if (deep_stream_) SSPSD_CUDA(cudaStreamSynchronize(deep_stream_));
    if (psd_stream_) SSPSD_CUDA(cudaStreamSynchronize(psd_stream_));
    const size_t keep = std::min<size_t>(st.fresh_cap, 4 + (size_t)st.pending_in);
    size_t cap = std::max(std::max(need + 64, st.fresh_cap * 2), need + reserve);
    for (int b = 0; b < 2; ++b) {
        float* nb = nullptr;
        SSPSD_CUDA(cudaMalloc(&nb, cap * sizeof(float)));
        if (st.fresh[b]) {
            SSPSD_CUDA(cudaMemcpy(nb, st.fresh[b], (b == st.fb ? keep : std::min<size_t>(4, st.fresh_cap)) * sizeof(float),
                                  cudaMemcpyDeviceToDevice));
            SSPSD_CUDA(cudaFree(st.fresh[b]));
        }
        st.fresh[b] = nb;
        st.ev_read_pending[b] = false;
    }
    st.fresh_cap = cap;
    return SSPSD_OK;
}

// stage i's PSD kernel over segments [k0, k0 + nseg), after the EWMA pre-scale of the stage's running sum
int Cascade::launch_psd(size_t i, const StreamSrc& src, uint64_t k0, uint64_t nseg, const EwmaPlan& e)
{
    if (hook_) return hook_->stage_psd(*this, i, src, k0, nseg, e);
    if (e.total != 1.0f) {
        int nb = (int)(n_ / 2 + 1);
        prof_begin(SSPSD_PROF_OTHER, 0, psd_stream(i));
        scale_kernel<<<(nb + 255) / 256, 256, 0, psd_stream(i)>>>(d_acc_ + i * acc_stride_, nb, e.total);
        prof_end(psd_stream(i));
        SSPSD_CUDA(cudaGetLastError());
    }
    StageParams p{};
    p.src = src;
    p.k0 = (long long)k0;
    p.nseg = (int)nseg;
    long long t = ((long long)nseg + 2ll * num_sms_ - 1) / (2ll * num_sms_);
    if (log2n_ == 9 && k2_variant_ >= 2 && hop_ * 2 == n_) {
        // N = 512, Hann: warp-level kernel (half a warp per segment, shuffles for the real-input split), persistent
        p.T = (int)std::max<long long>(W16::SPI, std::min<long long>(t, W16::MAX_T));
        p.hop = (int)hop_;
        p.detrend = detrend_;
        p.tile_cap = 0;
        p.win = d_win_;
        p.twM = d_twM_;
        p.twN = d_twN_;
        p.acc = d_acc_ + i * acc_stride_;
        p.jb = e.jb;
        p.g_first = e.g_first;
        p.g_s = e.g_s;
        int grid = (int)((nseg + p.T - 1) / p.T);
        int rcp = prepare_partials(i, grid * W16::SPI, &p);
        if (rcp) return rcp;
        prof_begin(i == 0 ? SSPSD_PROF_PSD_STAGE0 : SSPSD_PROF_PSD_DEEP, nseg * (uint64_t)hop_, psd_stream(i));
        psd_stage_kernel_w16<<<grid, W16::NT, stage_w16_smem_bytes(p.T), psd_stream(i)>>>(p);
        prof_end(psd_stream(i));
        if (!cuda_ok(cudaGetLastError(), "psd_stage_kernel_w16 launch")) return SSPSD_ECUDA;
        return reduce_partials(i, grid * W16::SPI, p);
    }
    const bool ring = log2n_ == 12 && k2_variant_ >= 2 && hop_ * 2 == n_;
    if (ring && k2_variant_ >= 3) {
        // four (five: ring1x5, 96 registers) independent single-group CTAs per SM (A/B variants, SSPSD_K2=ring1|ring1x5)
        const bool x5 = k2_variant_ == 4;
        const long long per_sm = x5 ? 5 : 4;
        long long t1 = ((long long)nseg + per_sm * num_sms_ - 1) / (per_sm * num_sms_);
        p.T = (int)std::max<long long>(1, std::min<long long>(t1, x5 ? 384 : 1024));
        p.hop = (int)hop_;
        p.detrend = detrend_;
        p.tile_cap = 0;
        p.win = d_win_;
        p.twM = d_twM_;
        p.twN = d_twN_;
        p.acc = d_acc_ + i * acc_stride_;
        p.jb = e.jb;
        p.g_first = e.g_first;
        p.g_s = e.g_s;
        int grid = (int)((nseg + p.T - 1) / p.T);
        int rcp = prepare_partials(i, grid, &p);
        if (rcp) return rcp;
        prof_begin(i == 0 ? SSPSD_PROF_PSD_STAGE0 : SSPSD_PROF_PSD_DEEP, nseg * (uint64_t)hop_, psd_stream(i));
        if (x5)
            psd_stage_kernel_ring1x5<<<grid, R16::TPS, stage_ring_smem_bytes(p.T, 1, 3, false), psd_stream(i)>>>(p);
        else
            psd_stage_kernel_ring1<<<grid, R16::TPS, stage_ring_smem_bytes(p.T, 1, RingCfg::RING1, false), psd_stream(i)>>>(p);
        prof_end(psd_stream(i));
        if (!cuda_ok(cudaGetLastError(), "psd_stage_kernel_ring1 launch")) return SSPSD_ECUDA;
        return reduce_partials(i, grid, p);
    }
    if (ring) {
        // persistent kernel: two CTAs per SM, each streams through a contiguous range of segments
        // with the deep stages overlapping on a second stream, stage 0 is cut into ~4 waves of CTAs so
        // that SM slots free up for them while it runs (a fully persistent grid would hold every slot)
        if (i == 0 && deep_stream_ && getenv("SSPSD_OVERLAP_WAVES")) t = (t + 3) / 4;
        p.T = (int)std::max<long long>(2, std::min<long long>(t, RingCfg::MAX_W));
        p.hop = (int)hop_;
        p.detrend = detrend_;
        p.tile_cap = 0;
        p.win = d_win_;
        p.twM = d_twM_;
        p.twN = d_twN_;
        p.acc = d_acc_ + i * acc_stride_;
        p.jb = e.jb;
        p.g_first = e.g_first;
        p.g_s = e.g_s;
        int grid = (int)((nseg + p.T - 1) / p.T);
        int rcp = prepare_partials(i, grid * R16::G, &p);
        if (rcp) return rcp;
        prof_begin(i == 0 ? SSPSD_PROF_PSD_STAGE0 : SSPSD_PROF_PSD_DEEP, nseg * (uint64_t)hop_, psd_stream(i));
        psd_stage_kernel_ring<<<grid, R16::NT, stage_ring_smem_bytes(p.T), psd_stream(i)>>>(p);
        prof_end(psd_stream(i));
        if (!cuda_ok(cudaGetLastError(), "psd_stage_kernel_ring launch")) return SSPSD_ECUDA;
        return reduce_partials(i, grid * R16::G, p);
    }
    const bool tiled_r16 = log2n_ == 12 && k2_variant_ >= 1;
    if (tiled_r16) {
        p.T = (int)std::max<long long>(1, std::min<long long>(t, tmax_));
    } else {
        // persistent tiled kernel: tiles as large as shared memory allows once there is enough work, CTAs
        // (2 per SM) walk over contiguous ranges of tiles
        int groups = std::max(1, nt_ / (int)(n_ / 16));
        p.T = (int)std::max<long long>(std::min<long long>(groups, (long long)nseg), std::min<long long>(t, tmax_));
        p.T = std::min(p.T, tmax_);
    }
    p.hop = (int)hop_;
    p.detrend = detrend_;
    p.tile_cap = (p.T - 1) * (int)hop_ + (int)n_;
    p.win = d_win_;
    p.twM = d_twM_;
    p.twN = d_twN_;
    p.acc = d_acc_ + i * acc_stride_;
    p.jb = e.jb;
    p.g_first = e.g_first;
    p.g_s = e.g_s;
    long long ntiles = ((long long)nseg + p.T - 1) / p.T;
    p.tpc = tiled_r16 ? 1 : (int)std::max<long long>(1, (ntiles + 2ll * num_sms_ - 1) / (2ll * num_sms_));
    int grid = (int)((ntiles + p.tpc - 1) / p.tpc);
    const int groups = tiled_r16 ? R16::G : std::max(1, nt_ / (int)(n_ / 16));
    int rc = prepare_partials(i, grid * groups, &p);
    if (rc) return rc;
    prof_begin(i == 0 ? SSPSD_PROF_PSD_STAGE0 : SSPSD_PROF_PSD_DEEP, nseg * (uint64_t)hop_, psd_stream(i));
    rc = launch_stage((int)log2n_, k2_variant_ >= 1, p, grid, psd_stream(i));
    prof_end(psd_stream(i));
    if (rc) return rc;
    return reduce_partials(i, grid * groups, p);
}

// Deterministic accumulation (sspsd_config::flags & SSPSD_FLAG_DETERMINISTIC): the PSD kernel writes one
// partial row per (CTA, group) and reduce_partials_kernel adds them to the stage's accumulator in row order, so a
// readout is bit-reproducible from run to run (the default flush is one atomicAdd per bin per thread).
int Cascade::prepare_partials(size_t i, int rows, StageParams* p)
{
    p->part = nullptr;
    p->part_stride = 0;
    if (!(cfg_.flags & SSPSD_FLAG_DETERMINISTIC)) return SSPSD_OK;
    // one buffer per PSD stream (stage 0 on stream_, the deep stages' kernels are ordered on their own stream)
    const int which = psd_stream(i) == stream_ ? 0 : 1;
    const size_t need = (size_t)rows * acc_stride_;
    if (need > part_cap_[which]) {
        SSPSD_CUDA(cudaStreamSynchronize(psd_stream(i)));
        if (d_part_[which]) SSPSD_CUDA(cudaFree(d_part_[which]));
        d_part_[which] = nullptr;
        SSPSD_CUDA(cudaMalloc(&d_part_[which], need * sizeof(float)));
        part_cap_[which] = need;
    }
    p->part = d_part_[which];
    p->part_stride = (int)acc_stride_;
    return SSPSD_OK;
}

int Cascade::reduce_partials(size_t i, int rows, const StageParams& p)
{
    if (!p.part) return SSPSD_OK;
    const int nb = (int)(n_ / 2 + 1);
    prof_begin(SSPSD_PROF_OTHER, 0, psd_stream(i));
    reduce_partials_kernel<<<(nb + 127) / 128, 128, 0, psd_stream(i)>>>(p.acc, p.part, rows, p.part_stride, nb);
    prof_end(psd_stream(i));
    return cuda_ok(cudaGetLastError(), "reduce_partials_kernel launch") ? SSPSD_OK : SSPSD_ECUDA;
}

int Cascade::launch_decim(size_t i, const StreamSrc& src, uint64_t m0, uint64_t m1, float* out_fresh,
                          long long out_split, long long out_cap)
{
    DecimParams p{};
    p.src = src;
    p.m0 = (long long)m0;
    p.m1 = (long long)m1;
    p.drain = drain_;
    p.out_fresh = out_fresh;
    p.out_split = out_split;
    p.out_cap = out_cap;
    p.preset = cfg_.hbf;
    long long lo = std::max<long long>(p.m0, p.drain);
    if (p.m1 <= lo)
        return SSPSD_OK;
    int grid = (int)((p.m1 - lo + DEC_OB - 1) / DEC_OB);
    cudaStream_t ss = stage_stream(i);
    static const bool fuse_carry = !getenv("SSPSD_CARRY_KERNEL");  // A/B switch: keep the separate carry_copy_kernel launch
    if (cc_valid_ && fuse_carry && (k3_variant_ == 1 || k3_variant_ == 2 || k3_variant_ == 7)) {
        p.cc = cc_pending_;  // the TMA-staged kernels build the stage's next carry buffer themselves
        cc_valid_ = false;
    }
    prof_begin(i == 0 ? SSPSD_PROF_DECIM_STAGE0 : SSPSD_PROF_DECIM_DEEP, (uint64_t)(p.m1 - lo) * 8, ss);
    int rc;
    if (k3_variant_ == 0) {
        rc = cfg_.hbf == SSPSD_HBF_98 ? launch_decim_t<3, 6, 15, SSPSD_HBF_98>(p, grid, ss)
                                      : launch_decim_t<5, 10, 23, SSPSD_HBF_140>(p, grid, ss);
    } else if (k3_variant_ == 1) {
        rc = cfg_.hbf == SSPSD_HBF_98 ? launch_decim_tma_t<3, 6, 15, SSPSD_HBF_98, 960, 2>(p, p.m1 - lo, num_sms_, ss)
                                      : launch_decim_tma_t<5, 10, 23, SSPSD_HBF_140, 960, 2>(p, p.m1 - lo, num_sms_, ss);
    } else if (k3_variant_ == 2) {
        rc = cfg_.hbf == SSPSD_HBF_98 ? launch_decim_tma_t<3, 6, 15, SSPSD_HBF_98, 640, 3>(p, p.m1 - lo, num_sms_, ss)
                                      : launch_decim_tma_t<5, 10, 23, SSPSD_HBF_140, 640, 3>(p, p.m1 - lo, num_sms_, ss);
    } else if (k3_variant_ == 3) {
        rc = cfg_.hbf == SSPSD_HBF_98 ? launch_decim_async_t<3, 6, 15, SSPSD_HBF_98, 960, 2>(p, p.m1 - lo, num_sms_, ss)
                                      : launch_decim_async_t<5, 10, 23, SSPSD_HBF_140, 960, 2>(p, p.m1 - lo, num_sms_, ss);
    } else if (k3_variant_ == 7) {
        rc = cfg_.hbf == SSPSD_HBF_98 ? launch_decim_tma_t<3, 6, 15, SSPSD_HBF_98, 768, 3>(p, p.m1 - lo, num_sms_, ss)
                                      : launch_decim_tma_t<5, 10, 23, SSPSD_HBF_140, 768, 3>(p, p.m1 - lo, num_sms_, ss);
    } else if (k3_variant_ == 5) {
        rc = cfg_.hbf == SSPSD_HBF_98 ? launch_decim_pf_t<3, 6, 15, SSPSD_HBF_98, 960, 2>(p, p.m1 - lo, num_sms_, ss)
                                      : launch_decim_pf_t<5, 10, 23, SSPSD_HBF_140, 960, 2>(p, p.m1 - lo, num_sms_, ss);
    } else if (k3_variant_ == 6) {
        rc = cfg_.hbf == SSPSD_HBF_98 ? launch_decim_pf_t<3, 6, 15, SSPSD_HBF_98, 640, 3>(p, p.m1 - lo, num_sms_, ss)
                                      : launch_decim_pf_t<5, 10, 23, SSPSD_HBF_140, 640, 3>(p, p.m1 - lo, num_sms_, ss);
    } else {
        rc = cfg_.hbf == SSPSD_HBF_98 ? launch_decim_async_t<3, 6, 15, SSPSD_HBF_98, 640, 3>(p, p.m1 - lo, num_sms_, ss)
                                      : launch_decim_async_t<5, 10, 23, SSPSD_HBF_140, 640, 3>(p, p.m1 - lo, num_sms_, ss);
    }
    prof_end(ss);
    return rc;
}

// One batch of one stage: n_new samples have been appended to the stage's stream.  They live in
// `fresh` from logical index split = floor4(L) on (fresh[0 .. L - split) are copies of the carry tail).
// Stage 0 runs on stream_, stages >= 1 on deep_stream_ (if enabled) so that they overlap the next
// batch's stage 0; the only cross-stream hazards are the next stage's two fresh buffers.
int Cascade::run_stage(size_t i, const float* fresh, long long split, uint64_t n_new)
{
    StageState& st = stages_[i];
    cudaStream_t ss = stage_stream(i);
    cudaStream_t ps = psd_stream(i);  // == ss unless the stage's PSD kernel runs beside the decimation chain
    const uint64_t L1 = st.L + n_new;
    const uint64_t craw0 = st.craw;
    const uint64_t craw1 = L1 < n_ ? 0 : 1 + (L1 - n_) / hop_;
    const StreamSrc src{st.carry[st.cur], fresh, st.carry_start, split, (long long)L1};
    int rc;
    bool psd_launched = false;
    if (ps != ss && craw1 > craw0) {
        // everything queued on ss so far (previous decimator, carry copy of the last batch) made this
        // stage's input: the PSD stream may read it from here on
        SSPSD_CUDA(cudaEventRecord(st.ev_in, ss));
        SSPSD_CUDA(cudaStreamWaitEvent(ps, st.ev_in, 0));
    }

    if (windowed_ && i < n_local_ && craw1 > craw0) {
        // time-chunk mode: accumulate only the fully valid segments this rank owns; their start position
        // own(i, k*hop) = 8^i k hop + c_i must lie in [own_lo, own_hi)
        const uint64_t step = (uint64_t)hop_ << (SSPSD_DEPTH * i);
        const uint64_t c = own_offset(i);
        auto first_at_or_after = [&](uint64_t pos) { return pos <= c ? 0ull : (pos - c + step - 1) / step; };
        uint64_t klo = std::max<uint64_t>(first_at_or_after(own_lo_), (st.valid_from + hop_ - 1) / hop_);
        uint64_t khi = own_hi_ == ~0ull ? ~0ull : first_at_or_after(own_hi_);
        uint64_t a = std::max(craw0, klo), b = std::min(craw1, khi);
        if (b > a) {
            if (st.avg == 0xffffffffu) {
                rc = launch_psd(i, src, a, b - a, EwmaPlan{(int)(b - a), 1.0f, 1.0f, 1.0f, 0});  // boxcar
            } else {
                // EWMA follows the global segment order: before global segment a the reference's count
                // is min(a, avg + 1) (psd.rs:218-225).  The row ends up normalised "as if the stream ended
                // at b"; the caller multiplies it by g^(segments scaled after b) before the reduction.
                const uint32_t cnt = (uint32_t)std::min<uint64_t>(a, (uint64_t)st.avg + 1);
                rc = launch_psd(i, src, a, b - a, ewma_plan(cnt, st.avg, b - a));
            }
            if (rc) return rc;
            psd_launched = true;
            st.count = (uint32_t)std::min<uint64_t>((uint64_t)st.count + (b - a), 0xffffffffull);
        }
    } else if (craw1 > craw0) {
        const uint64_t S = craw1 - craw0;
        const EwmaPlan e = ewma_plan(st.count, st.avg, S);
        rc = launch_psd(i, src, craw0, S, e);
        if (rc) return rc;
        st.count = e.count_after;
        psd_launched = true;
    }
    if (ps != ss && psd_launched) {
        // the PSD kernel reads carry[cur] and fresh[fb]: whoever overwrites them next waits for this
        SSPSD_CUDA(cudaEventRecord(st.ev_psd[st.fb], ps));
        psd_dirty_ = true;
    }

    const uint64_t D0 = decimated(st);
    st.craw = craw1;
    const uint64_t D1 = decimated(st);
    uint64_t n_next = 0;
    long long nsplit = 0;
    // next batch's carry: history for the decimator + pending samples, [D1 - hb, L1); the last L1 % 4
    // samples are also copied to the head of the buffer the next batch's fresh samples will go to.  The job is
    // handed to this stage's decimator launch when there is one below (launch_decim), else to carry_copy_kernel.
    const long long cs = (long long)D1 - hb_;
    {
        const int n = (int)((long long)L1 - cs);
        const int head_n = (int)(L1 & 3);
        float* head_dst = nullptr;
        if (head_n) {
            if (i == 0) {
                // stage 0: the next batch goes through the staging buffer d_in_[in_buf_] whenever L % 4 != 0
                rc = ensure_in_buffers(1);
                if (rc) return rc;
                head_dst = d_in_[in_buf_];
            } else {
                head_dst = st.fresh[st.fb ^ 1];
            }
        }
        if (n < 0 || n > hb_ + (int)n_ + 16) {
            set_error("internal: carry overflow");
            return SSPSD_EINVAL;
        }
        // the copy overwrites carry[cur ^ 1] and the head of fresh[fb ^ 1], which the previous batch's PSD
        // kernel read (a wait on an event that was never recorded returns at once)
        if (ps != ss) SSPSD_CUDA(cudaStreamWaitEvent(ss, st.ev_psd[st.fb ^ 1], 0));
        cc_pending_ = CarryJob{cs, n, head_n, st.carry[st.cur ^ 1], head_dst, hb_ + (int)n_ + 16};
        cc_valid_ = true;
    }
    if (D1 > D0) {
        const uint64_t m0 = D0 / 8, m1 = D1 / 8;
        const uint64_t em1 = m1 > (uint64_t)drain_ ? m1 - drain_ : 0;
        n_next = em1 - st.emitted;
        if (n_next > 0) {
            if (windowed_ && i + 1 == n_local_) {
                // time-chunk mode: the input stream of the first non-local stage is collected for export
                if (tail_len_ + n_next > tail_cap_) {
                    size_t cap = std::max<size_t>(2 * tail_cap_, tail_len_ + n_next + (1u << 16));
                    float* nb = nullptr;
                    SSPSD_CUDA(cudaMalloc(&nb, cap * sizeof(float)));
                    if (d_tail_) {
                        SSPSD_CUDA(cudaMemcpyAsync(nb, d_tail_, tail_len_ * sizeof(float), cudaMemcpyDeviceToDevice, ss));
                        SSPSD_CUDA(cudaStreamSynchronize(ss));
                        SSPSD_CUDA(cudaFree(d_tail_));
                    }
                    d_tail_ = nb;
                    tail_cap_ = cap;
                }
                if (tail_len_ == 0) tail_first_ = st.emitted;
                rc = launch_decim(i, src, m0, m1, d_tail_ + tail_len_, (long long)st.emitted, (long long)(tail_cap_ - tail_len_));
                if (rc) return rc;
                tail_len_ += n_next;
                st.emitted = em1;
                n_next = 0;
            } else if (i + 1 >= max_stages_) {
                // single-stage API: the decimated items of this call are collected in the sink
                if (sink_len_ + n_next > sink_cap_) {
                    set_error("internal: sink overflow");
                    return SSPSD_EINVAL;
                }
                rc = launch_decim(i, src, m0, m1, d_sink_ + sink_len_, (long long)st.emitted, (long long)(sink_cap_ - sink_len_));
                if (rc) return rc;
                sink_len_ += n_next;
                st.emitted = em1;
                n_next = 0;
            } else {
                if (i + 1 >= stages_.size()) {
                    rc = add_stage();
                    if (rc) return rc;
                }
                StageState& nx = stages_[i + 1];
                nsplit = floor4((long long)nx.L);
                // the deferral window adapts to the caller's batch size (at most 16 batches, at most defer_): small
                // batches keep the buffers small, and the window is reserved in ONE allocation (a reallocation
                // synchronises all streams, moves what has accumulated and frees hundreds of MB: growing by
                // doubling cost 0.5 s over the first 4e8 samples of a small-call stream)
                defer_window_ = std::min<uint64_t>(defer_threshold(i + 1), 16 * n_next);
                rc = ensure_fresh(nx, (size_t)((long long)em1 - nsplit), (size_t)(defer_window_ + n_next));
                if (rc) return rc;
                const int b = nx.fb;
                // the next stage may still be reading this buffer from two batches ago (other stream)
                if (nx.ev_read_pending[b] && stage_stream(i) != stage_stream(i + 1)) {
                    SSPSD_CUDA(cudaStreamWaitEvent(ss, nx.ev_read[b], 0));
                    // ... and so may its PSD kernel (on the deep stream itself this is implied: that stream
                    // waits for ev_psd before every carry copy, which precedes this launch in stream order)
                    if (psd_stream(i + 1) != stage_stream(i + 1)) SSPSD_CUDA(cudaStreamWaitEvent(ss, nx.ev_psd[b], 0));
                    nx.ev_read_pending[b] = false;
                }
                rc = launch_decim(i, src, m0, m1, nx.fresh[b], nsplit, (long long)nx.fresh_cap);
                if (rc) return rc;
                stages_[i].emitted = em1;
                nx.pending_in += n_next;
            }
        }
    }

    {
        StageState& s2 = stages_[i];  // (add_stage() above may have moved the vector)
        if (cc_valid_) {
            // no decimator launch took the job (no new output this batch, or an A/B decimator variant)
            const CarryJob& cj = cc_pending_;
            prof_begin(SSPSD_PROF_OTHER, 0, ss);
            carry_copy_kernel<<<std::max(1, std::min(64, (cj.n + 255) / 256)), 256, 0, ss>>>(src, cj.g0, cj.n, cj.dst, cj.head_dst,
                                                                                            cj.head_n, cj.dst_cap);
            prof_end(ss);
            SSPSD_CUDA(cudaGetLastError());
            cc_valid_ = false;
        }
        s2.cur ^= 1;
        s2.carry_start = cs;
        s2.L = L1;
        if (i > 0) {
            // this stage is done with fresh[fb]: the previous stage's decimator may reuse it
            SSPSD_CUDA(cudaEventRecord(s2.ev_read[s2.fb], ss));
            s2.ev_read_pending[s2.fb] = true;
            s2.fb ^= 1;
        }
    }
    // The next stage runs once enough of its input has accumulated (see run_pending): with a 200e6-sample batch
    // the stages >= 1 are ~20 small dependent launches that cost 0.27 ms when serialised for 1/7 of the work;
    // letting their input pile up for a few batches gives them stage-0-sized grids.  Invisible to the caller:
    // every call that observes state (psd, sync, set_*, clone, ...) runs what is pending first.
    if (n_next > 0 && stages_[i + 1].pending_in >= defer_window_) return run_pending(i + 1);
    return SSPSD_OK;
}

uint64_t Cascade::defer_threshold(size_t j) const
{
    if (windowed_ || max_stages_ == 1 || defer_ <= 1 || j == 0) return 0;
    const unsigned sh = (unsigned)(SSPSD_DEPTH * (j - 1));
    return sh >= 63 ? 0 : (defer_ >> sh);
}

// run stage j over the samples the previous stage's decimator has accumulated in fresh[fb]
int Cascade::run_pending(size_t j)
{
    StageState& st = stages_[j];
    const uint64_t n = st.pending_in;
    if (n == 0) return SSPSD_OK;
    st.pending_in = 0;
    if (j == deep_from_ && deep_stream_) {
        // hand over to the deep stream: it may start once the decimator launches queued so far have run
        SSPSD_CUDA(cudaEventRecord(ev_stage0_, stream_));
        SSPSD_CUDA(cudaStreamWaitEvent(deep_stream_, ev_stage0_, 0));
        deep_dirty_ = true;
    }
    return run_stage(j, st.fresh[st.fb], floor4((long long)st.L), n);
}

int Cascade::flush_deferred()
{
    for (size_t j = 1; j < stages_.size(); ++j) {
        int rc = run_pending(j);  // may append to stage j + 1, which the loop reaches next
        if (rc) return rc;
    }
    return SSPSD_OK;
}

int Cascade::join_streams()
{
    if (psd_stream_ && psd_dirty_) {
        SSPSD_CUDA(cudaEventRecord(ev_psd_join_, psd_stream_));
        SSPSD_CUDA(cudaStreamWaitEvent(stream_, ev_psd_join_, 0));
        psd_dirty_ = false;
    }
    if (deep_stream_ && deep_dirty_) {
        SSPSD_CUDA(cudaEventRecord(ev_deep_, deep_stream_));
        SSPSD_CUDA(cudaStreamWaitEvent(stream_, ev_deep_, 0));
        deep_dirty_ = false;
    }
    return SSPSD_OK;
}

void Cascade::free_stages(bool keep_buffers)
{
    if (keep_buffers) {
        // deepest stage last in, first out: add_stage() hands the buffers back in the same order
        for (size_t i = stages_.size(); i-- > 0;) spare_.push_back(stages_[i]);
        stages_.clear();
        return;
    }
    for (auto* v : {&stages_, &spare_}) {
        for (auto& st : *v) {
            cudaFree(st.carry[0]);
            cudaFree(st.carry[1]);
            cudaFree(st.fresh[0]);
            cudaFree(st.fresh[1]);
            for (int b = 0; b < 2; ++b) {
                if (st.ev_read[b]) cudaEventDestroy(st.ev_read[b]);
                if (st.ev_psd[b]) cudaEventDestroy(st.ev_psd[b]);
            }
            if (st.ev_in) cudaEventDestroy(st.ev_in);
        }
        v->clear();
    }
}

// x: device memory, valid in stream order
int Cascade::feed_device_chunk(const float* x, size_t n)
{
    if (n == 0)
        return SSPSD_OK;
    int rc;
    if (stages_.empty()) {
        rc = add_stage();
        if (rc) return rc;
    }
    StageState& st = stages_[0];
    const long long split = floor4((long long)st.L);
    const size_t head = (size_t)((long long)st.L - split);
    if (head == 0 && (reinterpret_cast<uintptr_t>(x) & 15u) == 0)
        return run_stage(0, x, split, n);  // zero copy: the kernels read the caller's buffer in place
    // unaligned stream position or pointer: realign through the staging buffer (one extra device copy);
    // its head already holds the carry tail (written by the previous batch's carry_copy_kernel)
    rc = ensure_in_buffers(n + 4);
    if (rc) return rc;
    const int b = in_buf_;
    float* buf = d_in_[b];
    SSPSD_CUDA(cudaMemcpyAsync(buf + head, x, n * sizeof(float), cudaMemcpyDeviceToDevice, stream_));
    in_buf_ ^= 1;
    rc = run_stage(0, buf, split, n);
    if (rc) return rc;
    // a later host-pointer call refills this buffer from the copy stream: it must wait for these kernels
    SSPSD_CUDA(cudaEventRecord(ev_free_[b], stream_));
    return SSPSD_OK;
}

int Cascade::process_device(const float* x, size_t n)
{
    // chunks of at most max_batch; inputs above 2^26 samples are cut into >= 2 roughly equal chunks so
    // that the deep stages of chunk c (deep_stream_) overlap stage 0 of chunk c+1 (stream_)
    size_t nchunks = (n + cfg_.max_batch - 1) / cfg_.max_batch;
    if (deep_stream_ && getenv("SSPSD_OVERLAP_CHUNKS") && n > (1ull << 26))
        nchunks = std::max<size_t>(nchunks, (n + (1ull << 26) - 1) >> 26);
    size_t per = (n + nchunks - 1) / nchunks;
    per = (per + 4095) & ~(size_t)4095;  // keep chunk boundaries 16-byte aligned relative to x
    size_t pos = 0;
    while (pos < n) {
        size_t c = std::min<size_t>(n - pos, per);
        int rc = feed_device_chunk(x + pos, c);
        if (rc) return rc;
        pos += c;
    }
    return SSPSD_OK;
}

int Cascade::ensure_in_buffers(size_t need)
{
    if (need <= d_in_cap_)
        return SSPSD_OK;
    SSPSD_CUDA(cudaStreamSynchronize(stream_));
    SSPSD_CUDA(cudaStreamSynchronize(copy_stream_));
    size_t cap = need + 64;
    for (int i = 0; i < 2; ++i) {
        float* nb = nullptr;
        SSPSD_CUDA(cudaMalloc(&nb, cap * sizeof(float)));
        if (d_in_[i]) {
            SSPSD_CUDA(cudaMemcpy(nb, d_in_[i], 4 * sizeof(float), cudaMemcpyDeviceToDevice));  // keep the head
            SSPSD_CUDA(cudaFree(d_in_[i]));
        }
        d_in_[i] = nb;
    }
    d_in_cap_ = cap;
    return SSPSD_OK;
}

// One chunk of host samples: H2D on the copy stream (double buffered against the compute stream)
int Cascade::feed_host_chunk(const float* xh, size_t n)
{
    if (n == 0)
        return SSPSD_OK;
    int rc;
    if (stages_.empty()) {
        rc = add_stage();
        if (rc) return rc;
    }
    // sized for the usual chunk so that a stream of equal chunks allocates once; never smaller than n
    rc = ensure_in_buffers(std::max<uint64_t>(n, std::min<uint64_t>(host_chunk(), cfg_.max_batch)) + 4);
    if (rc) return rc;
    StageState& st = stages_[0];
    const long long split = floor4((long long)st.L);
    const size_t head = (size_t)((long long)st.L - split);
    const int b = in_buf_;
    // d_in_[b][0 .. head) already holds the carry tail (previous batch's carry_copy_kernel on stream_);
    // the copy below touches only [head, head + n)
    SSPSD_CUDA(cudaStreamWaitEvent(copy_stream_, ev_free_[b], 0));
    SSPSD_CUDA(cudaMemcpyAsync(d_in_[b] + head, xh, n * sizeof(float), cudaMemcpyHostToDevice, copy_stream_));
    SSPSD_CUDA(cudaEventRecord(ev_copied_[b], copy_stream_));
    SSPSD_CUDA(cudaStreamWaitEvent(stream_, ev_copied_[b], 0));
    last_copy_ = b;
    in_buf_ ^= 1;
    rc = run_stage(0, d_in_[b], split, n);
    if (rc) return rc;
    SSPSD_CUDA(cudaEventRecord(ev_free_[b], stream_));
    return SSPSD_OK;
}

int Cascade::flush_staged()
{
    if (staged_ == 0)
        return SSPSD_OK;
    const int hb = stage_buf_;
#if defined(__x86_64__) && defined(__SSE2__)
    _mm_sfence();  // stage_copy's non-temporal stores must be globally visible before the DMA reads the buffer
#endif
    // max_batch bounds every launch, also when it is smaller than the staging buffer
    const size_t chunk = (size_t)std::min<uint64_t>(host_chunk(), cfg_.max_batch);
    for (size_t pos = 0; pos < staged_; pos += chunk) {
        int rc = feed_host_chunk(h_stage_[hb] + pos, std::min(chunk, staged_ - pos));
        if (rc) return rc;
    }
    // the pinned buffer may be refilled only after this H2D copy has completed
    SSPSD_CUDA(cudaEventRecord(ev_stage_[hb], copy_stream_));
    stage_pending_[hb] = true;
    staged_ = 0;
    stage_buf_ ^= 1;
    if (stage_pending_[stage_buf_]) {
        SSPSD_CUDA(cudaEventSynchronize(ev_stage_[stage_buf_]));
        stage_pending_[stage_buf_] = false;
    }
    return SSPSD_OK;
}

// Copy of a small host slice into the pinned staging buffer.  The buffer is written once and then read by the DMA engine
// only, so slices of 16 KiB and more (the reference's 4096-sample slices, src/source.rs:116,123) are copied with
// non-temporal stores: no read-for-ownership of the destination lines, no cache pollution; flush_staged() fences them
// before it queues the H2D copy.  Measured with tools/small_calls.c: 3.1-3.4 GS/s against 2.55-3.0 with memcpy for
// 4096-sample slices, but 1.40 against 1.78 GS/s for 1000-sample slices, hence the threshold.
static inline void stage_copy(float* __restrict__ dst, const float* __restrict__ src, size_t n)
{
#if defined(__x86_64__) && defined(__SSE2__)
    static const bool plain = getenv("SSPSD_STAGE_MEMCPY") != nullptr;  // A/B switch: plain memcpy
    if (n >= 4096 && !plain) {
        while ((reinterpret_cast<uintptr_t>(dst) & 15u) && n) {
            *dst++ = *src++;
            --n;
        }
        size_t i = 0;
        for (; i + 16 <= n; i += 16) {
            const __m128 a = _mm_loadu_ps(src + i), b = _mm_loadu_ps(src + i + 4), c = _mm_loadu_ps(src + i + 8),
                         d = _mm_loadu_ps(src + i + 12);
            _mm_stream_ps(dst + i, a);
            _mm_stream_ps(dst + i + 4, b);
            _mm_stream_ps(dst + i + 8, c);
            _mm_stream_ps(dst + i + 12, d);
        }
        for (; i < n; ++i) dst[i] = src[i];
        return;
    }
#endif
    std::memcpy(dst, src, n * sizeof(float));
}

int Cascade::process_host(const float* x, size_t n)
{
    if (n == 0)
        return SSPSD_OK;
    int rc;
    if (n < cfg_.host_stage) {
        // small call (the reference's callers hand over 176..4096 items, src/source.rs:116-157):
        // collect in pinned memory, launch once enough is pending
        if (!h_stage_[0]) {
            SSPSD_CUDA(cudaMallocHost(&h_stage_[0], cfg_.host_stage * sizeof(float)));
            SSPSD_CUDA(cudaMallocHost(&h_stage_[1], cfg_.host_stage * sizeof(float)));
        }
        while (n) {
            size_t take = std::min<size_t>(n, cfg_.host_stage - staged_);
            stage_copy(h_stage_[stage_buf_] + staged_, x, take);
            staged_ += take;
            x += take;
            n -= take;
            if (staged_ == cfg_.host_stage) {
                rc = flush_staged();
                if (rc) return rc;
            }
        }
        return SSPSD_OK;
    }
    rc = flush_staged();
    if (rc) return rc;
    const size_t chunk = (size_t)std::min<uint64_t>(host_chunk(), cfg_.max_batch);
    size_t pos = 0;
    last_copy_ = -1;
    while (pos < n) {
        size_t c = std::min(n - pos, chunk);
        rc = feed_host_chunk(x + pos, c);
        if (rc) return rc;
        pos += c;
    }
    // the caller's buffer is borrowed for the call only: wait for the last H2D copy (not the compute)
    if (last_copy_ >= 0)
        SSPSD_CUDA(cudaEventSynchronize(ev_copied_[last_copy_]));
    return SSPSD_OK;
}

int Cascade::process(const float* x, size_t n, int mem)
{
    if (n == 0)
        return SSPSD_OK;  // psd.rs:459: no chunk, no stage
    if (!x) {
        set_error("null input");
        return SSPSD_EINVAL;
    }
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    sink_len_ = 0;
    if (max_stages_ == 1) {
        // PsdStage::process returns at most n/8 + N/8 decimated items
        size_t need = n / 8 + n_ / 8 + 16 + staged_ / 8;
        if (need > sink_cap_) {
            SSPSD_CUDA(cudaStreamSynchronize(stream_));
            if (d_sink_) SSPSD_CUDA(cudaFree(d_sink_));
            d_sink_ = nullptr;
            SSPSD_CUDA(cudaMalloc(&d_sink_, need * sizeof(float)));
            sink_cap_ = need;
        }
    }
    if (mem == SSPSD_MEM_DEVICE) {
        int rc = flush_staged();
        if (rc) return rc;
        return process_device(x, n);
    }
    if (mem != SSPSD_MEM_HOST) {
        set_error("bad mem kind");
        return SSPSD_EINVAL;
    }
    if (max_stages_ == 1) {
        // the single-stage API returns its decimated output synchronously: no deferred staging
        size_t pos = 0;
        const size_t chunk = (size_t)std::min<uint64_t>(host_chunk(), cfg_.max_batch);
        last_copy_ = -1;
        while (pos < n) {
            size_t c = std::min(n - pos, chunk);
            int rc = feed_host_chunk(x + pos, c);
            if (rc) return rc;
            pos += c;
        }
        if (last_copy_ >= 0)
            SSPSD_CUDA(cudaEventSynchronize(ev_copied_[last_copy_]));
        return SSPSD_OK;
    }
    return process_host(x, n);
}

int Cascade::flush()
{
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    int rc = flush_staged();
    if (rc) return rc;
    return flush_deferred();
}

int Cascade::sync()
{
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    int rc = flush_staged();
    if (rc) return rc;
    rc = flush_deferred();
    if (rc) return rc;
    rc = join_streams();
    if (rc) return rc;
    SSPSD_CUDA(cudaStreamSynchronize(stream_));
    return SSPSD_OK;
}

// launch everything pending, make stream_ wait for the handle's side streams and record `ev` there: work queued on
// another stream behind `ev` sees the handle's complete state without a host synchronisation
int Cascade::fence(cudaEvent_t ev)
{
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    int rc = flush_staged();
    if (rc) return rc;
    rc = flush_deferred();
    if (rc) return rc;
    rc = join_streams();
    if (rc) return rc;
    SSPSD_CUDA(cudaEventRecord(ev, stream_));
    return SSPSD_OK;
}

int Cascade::set_avg(sspsd_avg_opts a)
{
    // options apply to segments completed after the call: launch what is staged first
    int rc = flush();
    if (rc) return rc;
    avg_ = a;  // psd.rs:431-436
    for (size_t i = 0; i < stages_.size(); ++i)
        stages_[i].avg = stage_avg(i);
    return SSPSD_OK;
}

int Cascade::set_stage_avg(uint32_t avg)
{
    int rc = flush();
    if (rc) return rc;
    single_stage_avg_set_ = true;
    single_stage_avg_ = avg;
    if (!stages_.empty())
        stages_[0].avg = avg;
    return SSPSD_OK;
}

int Cascade::set_detrend(int d)
{
    if (d == SSPSD_DETREND_LINEAR) {
        set_error("Detrend::Linear is unimplemented!() in the reference (src/psd.rs:110)");
        return SSPSD_EUNIMPLEMENTED;
    }
    if (d < 0 || d > SSPSD_DETREND_LINEAR) {
        set_error("unknown detrend");
        return SSPSD_EINVAL;
    }
    int rc = flush();
    if (rc) return rc;
    detrend_ = d;  // psd.rs:438-443 (all stages share the option)
    return SSPSD_OK;
}

int Cascade::reset()
{
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    SSPSD_CUDA(cudaStreamSynchronize(stream_));
    SSPSD_CUDA(cudaStreamSynchronize(copy_stream_));
    if (deep_stream_) SSPSD_CUDA(cudaStreamSynchronize(deep_stream_));
    if (psd_stream_) SSPSD_CUDA(cudaStreamSynchronize(psd_stream_));
    free_stages(true);
    deep_dirty_ = false;
    psd_dirty_ = false;
    seek_pos_ = 0;
    windowed_ = false;
    tail_len_ = 0;
    staged_ = 0;
    sink_len_ = 0;
    SSPSD_CUDA(cudaMemsetAsync(d_acc_, 0, (size_t)SSPSD_MAX_STAGES * acc_stride_ * sizeof(float), stream_));
    return SSPSD_OK;
}

int Cascade::clone_from(Cascade& o, const sspsd_config* cfg)
{
    int rc = o.sync();
    if (rc) return rc;
    rc = init(cfg ? *cfg : o.cfg_, o.max_stages_);
    if (rc) return rc;
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    detrend_ = o.detrend_;
    avg_ = o.avg_;
    single_stage_avg_set_ = o.single_stage_avg_set_;
    single_stage_avg_ = o.single_stage_avg_;
    for (size_t i = 0; i < o.stages_.size(); ++i) {
        rc = add_stage();
        if (rc) return rc;
        // add_stage() zeroes the carry buffers and the accumulator row on stage_stream(i); the copies below run
        // on stream_, and nothing else orders the two non-blocking streams
        SSPSD_CUDA(cudaStreamSynchronize(stage_stream(i)));
        StageState& d = stages_[i];
        const StageState& s = o.stages_[i];
        d.L = s.L;
        d.craw = s.craw;
        d.count = s.count;
        d.avg = s.avg;
        d.emitted = s.emitted;
        d.carry_start = s.carry_start;
        d.cur = 0;
        const size_t cap = (size_t)hb_ + n_ + 16;
        SSPSD_CUDA(cudaMemcpyAsync(d.carry[0], s.carry[s.cur], cap * sizeof(float), cudaMemcpyDeviceToDevice, stream_));
        if (i > 0 && s.fresh[s.fb]) {
            // the head of the next incoming fresh buffer (copies of the carry tail) is stream state too
            int rc2 = ensure_fresh(d, 8);
            if (rc2) return rc2;
            d.fb = 0;
            SSPSD_CUDA(cudaMemcpyAsync(d.fresh[0], s.fresh[s.fb], 4 * sizeof(float), cudaMemcpyDeviceToDevice, stream_));
        }
    }
    if (o.d_in_[o.in_buf_]) {
        int rc2 = ensure_in_buffers(8);
        if (rc2) return rc2;
        SSPSD_CUDA(cudaMemcpyAsync(d_in_[in_buf_], o.d_in_[o.in_buf_], 4 * sizeof(float), cudaMemcpyDeviceToDevice, stream_));
    }
    SSPSD_CUDA(cudaMemcpyAsync(d_acc_, o.d_acc_, (size_t)SSPSD_MAX_STAGES * acc_stride_ * sizeof(float),
                               cudaMemcpyDeviceToDevice, stream_));
    SSPSD_CUDA(cudaStreamSynchronize(stream_));
    if (deep_stream_) SSPSD_CUDA(cudaStreamSynchronize(deep_stream_));
    if (psd_stream_) SSPSD_CUDA(cudaStreamSynchronize(psd_stream_));
    return SSPSD_OK;
}

float Cascade::gain_of(uint32_t count) const
{
    // PsdStage::gain, psd.rs:279-283; N/2*count formed in 64 bits (the reference wraps in u32 for
    // count > 2^32/(N/2), SURVEY.md D6)
    uint64_t nc = (uint64_t)(n_ / 2) * (uint64_t)count;
    return (float)nc * win_.nenbw * win_.power;
}

float Cascade::stage_gain() const { return gain_of(stages_.empty() ? 0 : stages_[0].count); }

// Stage bookkeeping in a flat form that can travel (channel gather of a multi-process group):
// book[4 i .. 4 i + 3] = (L, craw, count, avg) of stage i, book[4 * SSPSD_MAX_STAGES] = number of stages
void Cascade::export_book(uint64_t* book) const
{
    std::memset(book, 0, (4 * SSPSD_MAX_STAGES + 2) * sizeof(uint64_t));
    for (size_t i = 0; i < stages_.size(); ++i) {
        book[4 * i] = stages_[i].L;
        book[4 * i + 1] = stages_[i].craw;
        book[4 * i + 2] = stages_[i].count;
        book[4 * i + 3] = stages_[i].avg;
    }
    book[4 * SSPSD_MAX_STAGES] = stages_.size();
}

// PsdCascade::psd, psd.rs:479-543, on host copies of the accumulator rows and the stage bookkeeping
int Cascade::merge_host(const sspsd_config& cfg, const uint64_t* book, const float* rows, size_t stride,
                        const sspsd_merge_opts& o, float* p, size_t* p_len, sspsd_break* b, size_t* b_len)
{
    const size_t ns = (size_t)book[4 * SSPSD_MAX_STAGES];
    const size_t N = cfg.n_fft;
    const bool hann = cfg.window == SSPSD_WINDOW_HANN;
    const float power = hann ? 0.25f : 1.0f, nenbw = hann ? 1.5f : 1.0f;
    const uint64_t overlap = hann ? N / 2 : 0, hop = N - overlap;
    // first pass: sizes
    size_t plen = 0;
    {
        size_t end = 0;
        uint64_t dec = 1ull << (SSPSD_DEPTH * ns);
        for (size_t r = ns; r-- > 0;) {
            dec >>= SSPSD_DEPTH;
            size_t start = !o.keep_overlap ? (end + 7) >> 3 : 0;
            end = (dec > 1 && !o.keep_transition_band) ? 2 * N / 5 : N / 2 + 1;
            if (book[4 * r + 2] >= o.min_count)
                plen += end - start;
            else
                end = start;
        }
    }
    const bool fits = (plen <= *p_len) && (ns <= *b_len) && (plen == 0 || p) && (ns == 0 || b);
    *p_len = plen;
    *b_len = ns;
    if (!fits) {
        set_error("output capacity too small");
        return SSPSD_ESHORT;
    }
    size_t pl = 0, bl = 0, end = 0;
    uint64_t dec = 1ull << (SSPSD_DEPTH * ns);
    for (size_t r = ns; r-- > 0;) {
        const uint64_t L = book[4 * r], craw = book[4 * r + 1];
        const uint32_t count = (uint32_t)book[4 * r + 2], avg = (uint32_t)book[4 * r + 3];
        dec >>= SSPSD_DEPTH;
        size_t start = !o.keep_overlap ? (end + 7) >> 3 : 0;
        end = (dec > 1 && !o.keep_transition_band) ? 2 * N / 5 : N / 2 + 1;
        bool include = count >= o.min_count;
        sspsd_break& bk = b[bl++];
        std::memset(&bk, 0, sizeof(bk));
        bk.start = pl;
        bk.include = include;
        bk.count = count;
        bk.avg = avg;
        bk.bins_start = start;
        bk.bins_end = end;
        bk.fft_size = N;
        bk.decimation = dec;
        uint32_t cm1 = count > 0 ? count - 1 : 0;
        bk.processed = (uint64_t)N * count - overlap * cm1;
        bk.pending = craw ? L - craw * hop : L;
        if (include) {
            // PsdStage::gain, psd.rs:279-283; N/2*count formed in 64 bits (the reference wraps in u32 for
            // count > 2^32/(N/2), SURVEY.md D6)
            const float gain = (float)((uint64_t)(N / 2) * (uint64_t)count) * nenbw * power;
            float gg = 1.0f / (gain * (float)dec);
            const float* sp = rows + r * stride;
            for (size_t k = start; k < end; ++k)
                p[pl++] = sp[k] * gg;
        } else {
            end = start;
        }
    }
    return SSPSD_OK;
}

int Cascade::psd(const sspsd_merge_opts& o, float* p, size_t* p_len, sspsd_break* b, size_t* b_len)
{
    if (!p_len || !b_len) {
        set_error("null length pointer");
        return SSPSD_EINVAL;
    }
    // launch what is pending and join the side streams; the one host synchronisation is behind the read-back below
    // (the bookkeeping is closed-form host state, it does not wait for the device)
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    int rc = flush_staged();
    if (rc) return rc;
    rc = flush_deferred();
    if (rc) return rc;
    rc = join_streams();
    if (rc) return rc;
    const size_t ns = stages_.size();
    uint64_t book[4 * SSPSD_MAX_STAGES + 2];
    export_book(book);
    // sizes first: a too small buffer is reported without touching the device
    {
        size_t pl = 0, bl = 0;
        int rs = merge_host(cfg_, book, nullptr, acc_stride_, o, nullptr, &pl, nullptr, &bl);
        const bool fits = (pl <= *p_len) && (ns <= *b_len) && (pl == 0 || p) && (ns == 0 || b);
        (void)rs;
        if (!fits || ns == 0) {
            *p_len = pl;
            *b_len = ns;
            if (!fits) {
                set_error("output capacity too small");
                return SSPSD_ESHORT;
            }
            return SSPSD_OK;
        }
    }
    SSPSD_CUDA(cudaMemcpyAsync(h_acc_, d_acc_, ns * acc_stride_ * sizeof(float), cudaMemcpyDeviceToHost, stream_));
    SSPSD_CUDA(cudaStreamSynchronize(stream_));
    return merge_host(cfg_, book, h_acc_, acc_stride_, o, p, p_len, b, b_len);
}

void Cascade::prof_begin(int cls, uint64_t units, cudaStream_t s)
{
    launches_[cls]++;
    if (!prof_on_) return;
    ProfRec r{cls, nullptr, nullptr, units};
    if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return;
    cudaEventRecord(r.a, s);
    prof_.push_back(r);
}

void Cascade::prof_end(cudaStream_t s)
{
    if (!prof_on_ || prof_.empty()) return;
    cudaEventRecord(prof_.back().b, s);
}

int Cascade::profile_read(sspsd_profile* out)
{
    if (!out) return SSPSD_EINVAL;
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    int rcj = flush_deferred();
    if (rcj) return rcj;
    rcj = join_streams();
    if (rcj) return rcj;
    SSPSD_CUDA(cudaStreamSynchronize(stream_));
    std::memset(out, 0, sizeof(*out));
    for (auto& r : prof_) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
            out->ms[r.cls] += ms;
            out->launches[r.cls]++;
            out->units[r.cls] += r.units;
        }
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
    }
    prof_.clear();
    for (int c = 0; c < SSPSD_PROF_NCLASS; ++c) {
        out->launches_total += launches_[c];
        launches_[c] = 0;
    }
    return SSPSD_OK;
}

uint64_t Cascade::next_valid_from(uint64_t valid) const
{
    // decimator outputs m are free of warm-up contamination once every input 8m+7-(H-1) .. 8m+7 is:
    // m >= (valid + halo + 1) / 8 (halo >= H-1); output m is sample m - R of the next stage
    if (valid == 0) return 0;
    const uint64_t mv = (valid + (uint64_t)decim_halo(cfg_.hbf) + 1) / 8;
    return mv > (uint64_t)drain_ ? mv - drain_ : 0;
}

uint64_t Cascade::own_offset(size_t i) const
{
    // own(i, j) = 8^i j + c_i with c_0 = 0, c_{i+1} = 8 (c_i + R): sample j of stage i+1 is decimator
    // output j + R of stage i, whose input chunk starts at stage-i sample 8 (j + R)
    uint64_t c = 0;
    for (size_t q = 0; q < i; ++q) c = 8 * (c + (uint64_t)drain_);
    return c;
}

int Cascade::seek(uint64_t pos)
{
    if (!stages_.empty() || staged_) {
        set_error("seek() needs a fresh cascade");
        return SSPSD_EINVAL;
    }
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    // closed-form state of a sequential run after `pos` samples (SURVEY.md A.2), unknown history = zeros
    seek_pos_ = pos;
    uint64_t L = pos;
    for (size_t i = 0; L > 0 && i < max_stages_; ++i) {
        int rc = add_stage();
        if (rc) return rc;
        StageState& st = stages_[i];
        st.L = L;
        st.craw = L < n_ ? 0 : 1 + (L - n_) / hop_;
        const uint64_t D = decimated(st);
        st.emitted = D / 8 > (uint64_t)drain_ ? D / 8 - drain_ : 0;
        st.count = 0;
        st.carry_start = (long long)D - hb_;
        L = st.emitted;
    }
    return SSPSD_OK;
}

int Cascade::set_window(uint64_t own_lo, uint64_t own_hi, uint32_t n_local)
{
    if (n_local == 0 || n_local > SSPSD_MAX_STAGES || own_hi < own_lo) {
        set_error("bad window");
        return SSPSD_EINVAL;
    }
    windowed_ = true;
    own_lo_ = own_lo;
    own_hi_ = own_hi;
    n_local_ = n_local;
    return SSPSD_OK;
}

int Cascade::take_tail(uint64_t j_lo, uint64_t j_hi, float* out, size_t* len, uint64_t* first, int mem)
{
    if (!len) return SSPSD_EINVAL;
    int rc = sync();
    if (rc) return rc;
    const uint64_t have_lo = tail_first_, have_hi = tail_first_ + tail_len_;
    const uint64_t a = std::max(j_lo, have_lo), b = std::min(j_hi, have_hi);
    const size_t n = b > a ? (size_t)(b - a) : 0;
    if (first) *first = a;
    if (*len < n || (n && !out)) {
        *len = n;
        set_error("output capacity too small");
        return SSPSD_ESHORT;
    }
    *len = n;
    if (!n) return SSPSD_OK;
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    SSPSD_CUDA(cudaMemcpyAsync(out, d_tail_ + (a - have_lo), n * sizeof(float),
                               mem == SSPSD_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, stream_));
    SSPSD_CUDA(cudaStreamSynchronize(stream_));
    return SSPSD_OK;
}

int Cascade::process_stage(uint32_t stage, const float* x, size_t n, int mem)
{
    if (stage == 0) return process(x, n, mem);
    if (n == 0) return SSPSD_OK;
    if (!x || stage >= max_stages_) return SSPSD_EINVAL;
    int rc = flush();
    if (rc) return rc;
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    while (stages_.size() <= stage) {
        rc = add_stage();
        if (rc) return rc;
    }
    size_t pos = 0;
    while (pos < n) {
        const size_t c = std::min<size_t>(n - pos, cfg_.max_batch);
        StageState& st = stages_[stage];
        const long long split = floor4((long long)st.L);
        const size_t head = (size_t)((long long)st.L - split);
        rc = ensure_fresh(st, c + 8);
        if (rc) return rc;
        float* buf = st.fresh[st.fb];
        SSPSD_CUDA(cudaMemcpyAsync(buf + head, x + pos, c * sizeof(float),
                                   mem == SSPSD_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice,
                                   stage_stream(stage)));
        if (mem != SSPSD_MEM_DEVICE) SSPSD_CUDA(cudaStreamSynchronize(stage_stream(stage)));
        rc = run_stage(stage, buf, split, c);
        if (rc) return rc;
        pos += c;
    }
    return SSPSD_OK;
}

int Cascade::set_stream_state(uint32_t stage, uint64_t samples, uint64_t segments)
{
    if (stage >= stages_.size()) return SSPSD_EINVAL;
    StageState& st = stages_[stage];
    st.L = samples;
    st.craw = samples < n_ ? 0 : 1 + (samples - n_) / hop_;
    st.count = (uint32_t)std::min<uint64_t>(segments, 0xffffffffull);
    return SSPSD_OK;
}

int Cascade::partials(sspsd_partials* out)
{
    if (!out) return SSPSD_EINVAL;
    int rc = flush();
    if (rc) return rc;
    std::memset(out, 0, sizeof(*out));
    out->acc = d_acc_;
    out->acc_stride = acc_stride_;
    out->n_stages = (uint32_t)stages_.size();
    for (size_t i = 0; i < stages_.size(); ++i)
        out->count_raw[i] = windowed_ ? stages_[i].count : stages_[i].craw;
    return SSPSD_OK;
}

int Cascade::set_counts(const uint64_t* craw, uint32_t n)
{
    if (!craw || n > SSPSD_MAX_STAGES) return SSPSD_EINVAL;
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    while (stages_.size() < n) {
        int rc = add_stage();
        if (rc) return rc;
    }
    for (uint32_t i = 0; i < n; ++i)
        stages_[i].count = (uint32_t)std::min<uint64_t>(craw[i], 0xffffffffull);
    return SSPSD_OK;
}

static int copy_out(float* dst, const float* src_dev, size_t n, int mem, cudaStream_t s)
{
    if (n == 0) return SSPSD_OK;
    SSPSD_CUDA(cudaMemcpyAsync(dst, src_dev, n * sizeof(float),
                               mem == SSPSD_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s));
    if (mem != SSPSD_MEM_DEVICE) SSPSD_CUDA(cudaStreamSynchronize(s));
    return SSPSD_OK;
}

int Cascade::stage_spectrum(float* out, size_t* len, int mem)
{
    if (!len) return SSPSD_EINVAL;
    const size_t need = n_ / 2 + 1;
    if (*len < need || !out) {
        *len = need;
        set_error("output capacity too small");
        return SSPSD_ESHORT;
    }
    *len = need;
    int rc = flush();
    if (rc) return rc;
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    return copy_out(out, d_acc_, need, mem, stream_);
}

int Cascade::stage_buf(float* out, size_t* len, int mem)
{
    if (!len) return SSPSD_EINVAL;
    int rc = flush();
    if (rc) return rc;
    size_t pending = 0;
    if (!stages_.empty()) {
        const StageState& st = stages_[0];
        pending = (size_t)(st.craw ? st.L - st.craw * (uint64_t)hop_ : st.L);
    }
    if (*len < pending || (pending && !out)) {
        *len = pending;
        set_error("output capacity too small");
        return SSPSD_ESHORT;
    }
    *len = pending;
    if (!pending) return SSPSD_OK;
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    const StageState& st = stages_[0];
    return copy_out(out, st.carry[st.cur] + ((long long)(st.L - pending) - st.carry_start), pending, mem, stream_);
}

int Cascade::take_sink(float* y, size_t* y_len, int mem)
{
    if (!y_len) return SSPSD_EINVAL;
    if (*y_len < sink_len_ || (sink_len_ && !y)) {
        *y_len = sink_len_;
        set_error("output capacity too small");
        return SSPSD_ESHORT;
    }
    *y_len = sink_len_;
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    return copy_out(y, d_sink_, sink_len_, mem, stream_);
}

}  // namespace sspsd
