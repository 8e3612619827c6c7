// sspsd_xcascade.cu -- XCascade: the cascaded cross-spectral density of two streams (sspsd_csd_* of
// include/sspsd.h).
//
// Two Cascades, one per channel, are driven in lockstep.  Their bookkeeping (segments, decimation, deferral,
// EWMA counts) does not depend on the data, so both run exactly the same stages over the same segment ranges;
// their own PSD launches are replaced by a hook (Cascade::hook_).  Channel y runs a chunk first and leaves, per
// stage, the StreamSrc its PSD kernel would have read; channel x then runs the same chunk and, where its PSD
// kernel would go, launches csd_stage_kernel over both sources.  Both cascades order all their work on ONE
// stream (no deep / PSD side streams), so stream order alone makes every CSD launch follow both channels'
// decimators and precede any later overwrite of the buffers it reads; between two lockstep steps each stage
// runs at most once, so the source y left for a stage is the one x's launch needs.
#include "sspsd_cascade.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include "sspsd_csd_kernel.cuh"

namespace sspsd {

namespace {

template <int LOG2N>
int prepare_csd_t(int hop, int* tmax, int* groups)
{
    using PL = Plan<LOG2N + 1>;
    const long long budget = PL::NT <= 256 ? 100 * 1024 : 200 * 1024;
    int t = 256;
    while (t > 1 && (long long)csd_smem_bytes<LOG2N>(t, hop) > budget) --t;
    if ((long long)csd_smem_bytes<LOG2N>(t, hop) > budget) {
        set_error("FFT size does not fit in shared memory");
        return SSPSD_EINVAL;
    }
    *tmax = t;
    *groups = PL::G;
    SSPSD_CUDA(cudaFuncSetAttribute(csd_stage_kernel<LOG2N>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)csd_smem_bytes<LOG2N>(t, hop)));
    return SSPSD_OK;
}

template <int LOG2N>
int launch_csd_t(const CsdParams& p, int grid, cudaStream_t s)
{
    csd_stage_kernel<LOG2N><<<grid, Plan<LOG2N + 1>::NT, csd_smem_bytes<LOG2N>(p.T, p.hop), s>>>(p);
    return cuda_ok(cudaGetLastError(), "csd_stage_kernel launch") ? SSPSD_OK : SSPSD_ECUDA;
}

#define SSPSD_CSD_SIZES(X) X(6) X(7) X(8) X(9) X(10) X(11) X(12)

int prepare_csd(int log2n, int hop, int* tmax, int* groups)
{
    switch (log2n) {
#define X(L) \
    case L:  \
        return prepare_csd_t<L>(hop, tmax, groups);
        SSPSD_CSD_SIZES(X)
#undef X
    default:
        set_error("CsdCascade supports n_fft = 64 .. 4096 (the two-for-one transform is an N-point complex FFT)");
        return SSPSD_EINVAL;
    }
}

int launch_csd(int log2n, const CsdParams& p, int grid, cudaStream_t s)
{
    switch (log2n) {
#define X(L) \
    case L:  \
        return launch_csd_t<L>(p, grid, s);
        SSPSD_CSD_SIZES(X)
#undef X
    default:
        return SSPSD_EINVAL;
    }
}

}  // namespace

class XCascade : public StageHook {
public:
    XCascade() = default;
    ~XCascade();
    int init(const sspsd_config& cfg);
    int clone_from(XCascade& o);
    int reset();
    int process(const float* x, const float* y, size_t n, int mem);
    int set_avg(sspsd_avg_opts a);
    int set_detrend(int d);
    int flush();
    int sync();
    int read(const sspsd_merge_opts& o, float* pxx, float* pyy, float* pxy, size_t* p_len, sspsd_break* b,
             size_t* b_len);
    int num_stages(uint32_t* n);
    float rbw() const { return x_.rbw(); }
    cudaStream_t stream() const { return stream_; }
    int stage_psd(Cascade& c, size_t i, const StreamSrc& src, uint64_t k0, uint64_t nseg, int jb, float g_first,
                  float g_s) override;

private:
    int setup(const sspsd_config& cfg);
    sspsd_config channel_cfg() const;
    int feed_chunk(const float* x, const float* y, size_t n, bool device);
    int flush_staged();
    int flush_all();

    // destroyed after the channels, whose destructors still synchronise the stream
    struct OwnedStream {
        cudaStream_t s = nullptr;
        int device = 0;
        ~OwnedStream()
        {
            if (!s) return;
            DeviceGuard g(device);
            cudaStreamDestroy(s);
        }
    } own_;
    Cascade x_, y_;
    sspsd_config cfg_{};
    cudaStream_t stream_ = nullptr;
    uint32_t n_ = 0, log2n_ = 0;
    int num_sms_ = 148, tmax_ = 1, groups_ = 1;
    uint32_t stride_ = 0;  // floats per row; a stage's block is CSD_ROWS rows
    float* d_win_ = nullptr;
    float2* d_tw_ = nullptr;
    float* d_acc_ = nullptr;  // [SSPSD_MAX_STAGES][CSD_ROWS][stride_]
    float* h_acc_ = nullptr;
    float* d_part_ = nullptr;
    size_t part_cap_ = 0;
    struct YSource {
        StreamSrc src;
        uint64_t k0, nseg;
        bool valid;
    } ysrc_[SSPSD_MAX_STAGES] = {};
};

XCascade::~XCascade()
{
    if (n_ == 0) return;
    DeviceGuard g(cfg_.device);
    cudaStreamSynchronize(stream_);
    cudaFree(d_win_);
    cudaFree(d_tw_);
    cudaFree(d_acc_);
    cudaFree(d_part_);
    if (h_acc_) cudaFreeHost(h_acc_);
}

sspsd_config XCascade::channel_cfg() const
{
    sspsd_config c = cfg_;
    c.stream = stream_;
    return c;
}

// everything but the two channels: the stream, the window and twiddle tables, the accumulator blocks
int XCascade::setup(const sspsd_config& cfg)
{
    const uint32_t n = cfg.n_fft;
    if (n < 64 || n > 4096 || (n & (n - 1))) {
        set_error("CsdCascade supports n_fft = 64 .. 4096 (the two-for-one transform is an N-point complex FFT)");
        return SSPSD_EINVAL;
    }
    if (cfg.window != SSPSD_WINDOW_RECT && cfg.window != SSPSD_WINDOW_HANN) {
        set_error("unknown window");
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
    if (!g.ok) return SSPSD_ECUDA;
    cfg_ = cfg;
    if (cfg.stream) {
        stream_ = (cudaStream_t)cfg.stream;
    } else {
        SSPSD_CUDA(cudaStreamCreateWithFlags(&own_.s, cudaStreamNonBlocking));
        own_.device = cfg.device;
        stream_ = own_.s;
    }
    while ((1u << log2n_) < n) ++log2n_;
    SSPSD_CUDA(cudaDeviceGetAttribute(&num_sms_, cudaDevAttrMultiProcessorCount, cfg.device));
    const int hop = cfg.window == SSPSD_WINDOW_HANN ? (int)n / 2 : (int)n;
    int rc = prepare_csd((int)log2n_, hop, &tmax_, &groups_);
    if (rc) return rc;

    // Window::hann / ::rectangular with the PSD path's f32 expression; twiddles exp(-2 pi i q / N)
    std::vector<float> win(n, 1.0f);
    if (cfg.window == SSPSD_WINDOW_HANN) {
        const float pi = 3.14159265358979323846f;
        const float df = pi / (float)n;
        for (uint32_t i = 0; i < n; ++i) {
            const float s = sinf(df * (float)i);
            win[i] = s * s;
        }
    }
    std::vector<float2> tw(n);
    for (uint32_t q = 0; q < n; ++q) {
        const double a = -2.0 * M_PI * (double)q / (double)n;
        tw[q] = make_float2((float)std::cos(a), (float)std::sin(a));
    }
    stride_ = (n / 2 + 1 + 63) & ~63u;
    const size_t acc_bytes = (size_t)SSPSD_MAX_STAGES * CSD_ROWS * stride_ * sizeof(float);
    SSPSD_CUDA(cudaMalloc(&d_win_, n * sizeof(float)));
    SSPSD_CUDA(cudaMalloc(&d_tw_, n * sizeof(float2)));
    SSPSD_CUDA(cudaMalloc(&d_acc_, acc_bytes));
    SSPSD_CUDA(cudaMallocHost(&h_acc_, acc_bytes));
    SSPSD_CUDA(cudaMemcpyAsync(d_win_, win.data(), n * sizeof(float), cudaMemcpyHostToDevice, stream_));
    SSPSD_CUDA(cudaMemcpyAsync(d_tw_, tw.data(), n * sizeof(float2), cudaMemcpyHostToDevice, stream_));
    SSPSD_CUDA(cudaMemsetAsync(d_acc_, 0, acc_bytes, stream_));
    SSPSD_CUDA(cudaStreamSynchronize(stream_));  // the host vectors above go out of scope
    for (Cascade* c : {&x_, &y_}) {
        c->one_stream_ = true;
        c->hook_ = this;
    }
    n_ = n;
    return SSPSD_OK;
}

int XCascade::init(const sspsd_config& cfg)
{
    int rc = setup(cfg);
    if (rc) return rc;
    const sspsd_config c = channel_cfg();
    rc = x_.init(c, SSPSD_MAX_STAGES);
    if (rc) return rc;
    return y_.init(c, SSPSD_MAX_STAGES);
}

int XCascade::clone_from(XCascade& o)
{
    int rc = o.sync();
    if (rc) return rc;
    rc = setup(o.cfg_);  // the caller's stream (cfg.stream) is shared by the copy, a private one is not
    if (rc) return rc;
    const sspsd_config c = channel_cfg();
    rc = x_.clone_from(o.x_, &c);
    if (rc) return rc;
    rc = y_.clone_from(o.y_, &c);
    if (rc) return rc;
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    SSPSD_CUDA(cudaMemcpyAsync(d_acc_, o.d_acc_, (size_t)SSPSD_MAX_STAGES * CSD_ROWS * stride_ * sizeof(float),
                               cudaMemcpyDeviceToDevice, stream_));
    SSPSD_CUDA(cudaStreamSynchronize(stream_));
    return SSPSD_OK;
}

int XCascade::reset()
{
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    int rc = x_.reset();
    if (rc) return rc;
    rc = y_.reset();
    if (rc) return rc;
    for (auto& s : ysrc_) s.valid = false;
    SSPSD_CUDA(cudaMemsetAsync(d_acc_, 0, (size_t)SSPSD_MAX_STAGES * CSD_ROWS * stride_ * sizeof(float), stream_));
    return SSPSD_OK;
}

// Channel y's PSD launch leaves its source; channel x's launches the CSD kernel over both.
int XCascade::stage_psd(Cascade& c, size_t i, const StreamSrc& src, uint64_t k0, uint64_t nseg, int jb, float g_first,
                        float g_s)
{
    YSource& ys = ysrc_[i];
    if (&c == &y_) {
        ys = YSource{src, k0, nseg, true};
        return SSPSD_OK;
    }
    if (!ys.valid || ys.k0 != k0 || ys.nseg != nseg) {
        set_error("internal: channels out of lockstep");
        return SSPSD_EINVAL;
    }
    ys.valid = false;
    float* acc = d_acc_ + i * CSD_ROWS * stride_;
    const int nblock = (int)(CSD_ROWS * stride_);
    if ((uint64_t)jb < nseg) {
        // the EWMA pre-scale of the running sums before this batch (Cascade::run_stage, ewma_plan: same f32 factor)
        double t = (double)g_first;
        const uint64_t n_s = nseg - 1 - (uint64_t)jb;
        if (n_s > 0) t *= std::pow((double)g_s, (double)n_s);
        const float total = (float)t;
        if (total != 1.0f) {
            csd_scale_kernel<<<(nblock + 255) / 256, 256, 0, stream_>>>(acc, nblock, total);
            SSPSD_CUDA(cudaGetLastError());
        }
    }
    CsdParams p{};
    p.src[0] = src;
    p.src[1] = ys.src;
    p.k0 = (long long)k0;
    p.nseg = (int)nseg;
    p.hop = (int)x_.hop_;
    p.detrend = x_.detrend_;
    p.win = d_win_;
    p.tw = d_tw_;
    p.acc = acc;
    p.stride = (int)stride_;
    p.jb = jb;
    p.g_first = g_first;
    p.g_s = g_s;
    // persistent tiled launch as psd_stage_kernel's: tiles as large as shared memory allows once there is enough
    // work, about two CTAs per SM walking contiguous ranges of tiles
    const long long t = ((long long)nseg + 2ll * num_sms_ - 1) / (2ll * num_sms_);
    p.T = (int)std::max<long long>(std::min<long long>(groups_, (long long)nseg), std::min<long long>(t, tmax_));
    p.T = std::min(p.T, tmax_);
    p.tile_cap = (p.T - 1) * p.hop + (int)n_;
    const long long ntiles = ((long long)nseg + p.T - 1) / p.T;
    p.tpc = (int)std::max<long long>(1, (ntiles + 2ll * num_sms_ - 1) / (2ll * num_sms_));
    const int grid = (int)((ntiles + p.tpc - 1) / p.tpc);
    const int rows = grid * groups_;
    if (cfg_.flags & SSPSD_FLAG_DETERMINISTIC) {
        // one partial block per (CTA, group), summed in row order by reduce_partials_kernel
        const size_t need = (size_t)rows * nblock;
        if (need > part_cap_) {
            SSPSD_CUDA(cudaStreamSynchronize(stream_));
            if (d_part_) SSPSD_CUDA(cudaFree(d_part_));
            d_part_ = nullptr;
            SSPSD_CUDA(cudaMalloc(&d_part_, need * sizeof(float)));
            // the row padding is never written: keep it zero so that the reduction adds nothing there
            SSPSD_CUDA(cudaMemsetAsync(d_part_, 0, need * sizeof(float), stream_));
            part_cap_ = need;
        }
        p.part = d_part_;
        p.part_stride = nblock;
    }
    int rc = launch_csd((int)log2n_, p, grid, stream_);
    if (rc) return rc;
    if (p.part) {
        reduce_partials_kernel<<<(nblock + 127) / 128, 128, 0, stream_>>>(acc, p.part, rows, nblock, nblock);
        SSPSD_CUDA(cudaGetLastError());
    }
    return SSPSD_OK;
}

// one lockstep step: the same chunk through y's stages, then through x's (which launch the CSD kernels)
int XCascade::feed_chunk(const float* x, const float* y, size_t n, bool device)
{
    int rc = device ? y_.feed_device_chunk(y, n) : y_.feed_host_chunk(y, n);
    if (rc) return rc;
    rc = device ? x_.feed_device_chunk(x, n) : x_.feed_host_chunk(x, n);
    if (rc) return rc;
    // y's input buffer of this chunk was read by the CSD kernels queued just now: its next refill waits for them
    SSPSD_CUDA(cudaEventRecord(y_.ev_free_[y_.in_buf_ ^ 1], stream_));
    return SSPSD_OK;
}

// Cascade::flush_staged for both channels, chunk by chunk in lockstep
int XCascade::flush_staged()
{
    const size_t staged = x_.staged_;
    if (staged == 0) return SSPSD_OK;
    const int hb = x_.stage_buf_;
    const size_t chunk = (size_t)std::min<uint64_t>(Cascade::host_chunk(), x_.cfg_.max_batch);
    for (size_t pos = 0; pos < staged; pos += chunk) {
        int rc = feed_chunk(x_.h_stage_[hb] + pos, y_.h_stage_[hb] + pos, std::min(chunk, staged - pos), false);
        if (rc) return rc;
    }
    for (Cascade* c : {&x_, &y_}) {
        SSPSD_CUDA(cudaEventRecord(c->ev_stage_[hb], c->copy_stream_));
        c->stage_pending_[hb] = true;
        c->staged_ = 0;
        c->stage_buf_ ^= 1;
        if (c->stage_pending_[c->stage_buf_]) {
            SSPSD_CUDA(cudaEventSynchronize(c->ev_stage_[c->stage_buf_]));
            c->stage_pending_[c->stage_buf_] = false;
        }
    }
    return SSPSD_OK;
}

// staged input and deferred deep stages, in lockstep: afterwards the channels' own flush() finds nothing to do
int XCascade::flush_all()
{
    int rc = flush_staged();
    if (rc) return rc;
    for (size_t j = 1; j < x_.stages_.size(); ++j) {
        rc = y_.run_pending(j);
        if (rc) return rc;
        rc = x_.run_pending(j);
        if (rc) return rc;
    }
    return SSPSD_OK;
}

int XCascade::process(const float* x, const float* y, size_t n, int mem)
{
    if (n == 0) return SSPSD_OK;
    if (!x || !y) {
        set_error("null input");
        return SSPSD_EINVAL;
    }
    if (mem != SSPSD_MEM_HOST && mem != SSPSD_MEM_DEVICE) {
        set_error("bad mem kind");
        return SSPSD_EINVAL;
    }
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    int rc;
    const uint64_t max_batch = x_.cfg_.max_batch;
    if (mem == SSPSD_MEM_DEVICE) {
        rc = flush_staged();
        if (rc) return rc;
        // Cascade::process_device's chunks: at most max_batch, boundaries 16-byte aligned relative to x and y
        const size_t nchunks = (n + max_batch - 1) / max_batch;
        size_t per = (n + nchunks - 1) / nchunks;
        per = (per + 4095) & ~(size_t)4095;
        for (size_t pos = 0; pos < n; pos += per) {
            rc = feed_chunk(x + pos, y + pos, std::min<size_t>(n - pos, per), true);
            if (rc) return rc;
        }
        return SSPSD_OK;
    }
    const uint64_t hs = x_.cfg_.host_stage;
    if (n < hs) {
        // small calls are collected in the channels' pinned staging buffers (Cascade::process_host)
        for (Cascade* c : {&x_, &y_}) {
            if (!c->h_stage_[0]) {
                SSPSD_CUDA(cudaMallocHost(&c->h_stage_[0], hs * sizeof(float)));
                SSPSD_CUDA(cudaMallocHost(&c->h_stage_[1], hs * sizeof(float)));
            }
        }
        while (n) {
            const size_t take = std::min<size_t>(n, hs - x_.staged_);
            std::memcpy(x_.h_stage_[x_.stage_buf_] + x_.staged_, x, take * sizeof(float));
            std::memcpy(y_.h_stage_[y_.stage_buf_] + y_.staged_, y, take * sizeof(float));
            x_.staged_ += take;
            y_.staged_ += take;
            x += take;
            y += take;
            n -= take;
            if (x_.staged_ == hs) {
                rc = flush_staged();
                if (rc) return rc;
            }
        }
        return SSPSD_OK;
    }
    rc = flush_staged();
    if (rc) return rc;
    const size_t chunk = (size_t)std::min<uint64_t>(Cascade::host_chunk(), max_batch);
    x_.last_copy_ = y_.last_copy_ = -1;
    for (size_t pos = 0; pos < n; pos += chunk) {
        rc = feed_chunk(x + pos, y + pos, std::min(chunk, n - pos), false);
        if (rc) return rc;
    }
    // the caller's buffers are borrowed for the call only: wait for the last H2D copies
    for (Cascade* c : {&x_, &y_})
        if (c->last_copy_ >= 0) SSPSD_CUDA(cudaEventSynchronize(c->ev_copied_[c->last_copy_]));
    return SSPSD_OK;
}

int XCascade::set_avg(sspsd_avg_opts a)
{
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    int rc = flush_all();  // options apply to segments completed after the call
    if (rc) return rc;
    rc = x_.set_avg(a);
    if (rc) return rc;
    return y_.set_avg(a);
}

int XCascade::set_detrend(int d)
{
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    int rc = flush_all();
    if (rc) return rc;
    rc = x_.set_detrend(d);  // validates d (Linear: SSPSD_EUNIMPLEMENTED)
    if (rc) return rc;
    return y_.set_detrend(d);
}

int XCascade::flush()
{
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    return flush_all();
}

int XCascade::sync()
{
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    int rc = flush_all();
    if (rc) return rc;
    SSPSD_CUDA(cudaStreamSynchronize(stream_));
    return SSPSD_OK;
}

int XCascade::num_stages(uint32_t* n)
{
    int rc = flush();
    if (rc) return rc;
    *n = x_.n_stages();
    return SSPSD_OK;
}

// PsdCascade::psd's merge (Cascade::merge_host) applied to each row: same breaks, same 1/(gain_i 8^i) per stage
int XCascade::read(const sspsd_merge_opts& o, float* pxx, float* pyy, float* pxy, size_t* p_len, sspsd_break* b,
                   size_t* b_len)
{
    if (!p_len || !b_len) {
        set_error("null length pointer");
        return SSPSD_EINVAL;
    }
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    int rc = flush_all();
    if (rc) return rc;
    const size_t ns = x_.stages_.size();
    uint64_t book[4 * SSPSD_MAX_STAGES + 2];
    x_.export_book(book);
    size_t pl = 0, bl = 0;
    Cascade::merge_host(x_.cfg_, book, nullptr, 0, o, nullptr, &pl, nullptr, &bl);
    const bool fits = (pl <= *p_len) && (ns <= *b_len) && (pl == 0 || (pxx && pyy && pxy)) && (ns == 0 || b);
    if (!fits || ns == 0) {
        *p_len = pl;
        *b_len = ns;
        if (!fits) {
            set_error("output capacity too small");
            return SSPSD_ESHORT;
        }
        return SSPSD_OK;
    }
    const size_t block = (size_t)CSD_ROWS * stride_;
    SSPSD_CUDA(cudaMemcpyAsync(h_acc_, d_acc_, ns * block * sizeof(float), cudaMemcpyDeviceToHost, stream_));
    SSPSD_CUDA(cudaStreamSynchronize(stream_));
    std::vector<float> re(pl), im(pl);
    float* outs[CSD_ROWS] = {pxx, pyy, re.data(), im.data()};
    for (int r = 0; r < CSD_ROWS; ++r) {
        size_t pr = pl, br = ns;
        rc = Cascade::merge_host(x_.cfg_, book, h_acc_ + (size_t)r * stride_, block, o, outs[r], &pr, b, &br);
        if (rc) return rc;
    }
    for (size_t k = 0; k < pl; ++k) {
        pxy[2 * k] = re[k];
        pxy[2 * k + 1] = im[k];
    }
    *p_len = pl;
    *b_len = ns;
    return SSPSD_OK;
}

}  // namespace sspsd

struct sspsd_csd {
    sspsd::XCascade c;
};

using sspsd::set_error;

int32_t sspsd_csd_create(const sspsd_config* cfg, sspsd_csd** out)
{
    if (!cfg || !out) {
        set_error("null argument");
        return SSPSD_EINVAL;
    }
    *out = nullptr;
    sspsd_csd* h = new (std::nothrow) sspsd_csd();
    if (!h) return SSPSD_ENOMEM;
    int rc = h->c.init(*cfg);
    if (rc) {
        delete h;
        return rc;
    }
    *out = h;
    return SSPSD_OK;
}

void sspsd_csd_destroy(sspsd_csd* h) { delete h; }

int32_t sspsd_csd_clone(sspsd_csd* h, sspsd_csd** out)
{
    if (!h || !out) {
        set_error("null argument");
        return SSPSD_EINVAL;
    }
    *out = nullptr;
    sspsd_csd* n = new (std::nothrow) sspsd_csd();
    if (!n) return SSPSD_ENOMEM;
    int rc = n->c.clone_from(h->c);
    if (rc) {
        delete n;
        return rc;
    }
    *out = n;
    return SSPSD_OK;
}

int32_t sspsd_csd_reset(sspsd_csd* h) { return h ? h->c.reset() : SSPSD_EINVAL; }

int32_t sspsd_csd_process_f32(sspsd_csd* h, const float* x, const float* y, size_t n, int32_t mem)
{
    if (!h) return SSPSD_EINVAL;
    return h->c.process(x, y, n, mem);
}

int32_t sspsd_csd_set_avg(sspsd_csd* h, sspsd_avg_opts avg) { return h ? h->c.set_avg(avg) : SSPSD_EINVAL; }

int32_t sspsd_csd_set_detrend(sspsd_csd* h, int32_t d) { return h ? h->c.set_detrend(d) : SSPSD_EINVAL; }

int32_t sspsd_csd_rbw(const sspsd_csd* h, float* rbw)
{
    if (!h || !rbw) return SSPSD_EINVAL;
    *rbw = h->c.rbw();
    return SSPSD_OK;
}

int32_t sspsd_csd_read(sspsd_csd* h, const sspsd_merge_opts* opts, float* pxx, float* pyy, float* pxy, size_t* p_len,
                       sspsd_break* b, size_t* b_len)
{
    if (!h) return SSPSD_EINVAL;
    sspsd_merge_opts o{0, 1, 0};  // MergeOpts::default(), psd.rs:350-358
    if (opts) o = *opts;
    return h->c.read(o, pxx, pyy, pxy, p_len, b, b_len);
}

int32_t sspsd_csd_num_stages(sspsd_csd* h, uint32_t* n)
{
    if (!h || !n) return SSPSD_EINVAL;
    return h->c.num_stages(n);
}

int32_t sspsd_csd_stream(const sspsd_csd* h, void** stream)
{
    if (!h || !stream) return SSPSD_EINVAL;
    *stream = (void*)h->c.stream();
    return SSPSD_OK;
}

int32_t sspsd_csd_flush(sspsd_csd* h) { return h ? h->c.flush() : SSPSD_EINVAL; }
int32_t sspsd_csd_sync(sspsd_csd* h) { return h ? h->c.sync() : SSPSD_EINVAL; }
