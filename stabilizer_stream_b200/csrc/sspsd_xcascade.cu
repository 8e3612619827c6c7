// sspsd_xcascade.cu -- XCascade: the cascaded cross-spectral density of two streams (sspsd_csd_* of
// include/sspsd.h), the cross-spectral matrix of K = 2 .. 4 streams (sspsd_csm_*) and the two-sided spectrum of
// z = i + i q (ZoomCascade, sspsd_zoom_*: I/Q streams, or a real stream mixed down around a carrier).
//
// K Cascades, one per channel, are driven in lockstep.  Their bookkeeping (segments, decimation, deferral,
// EWMA counts) does not depend on the data, so all run exactly the same stages over the same segment ranges;
// their own PSD launches are replaced by a hook (Cascade::hook_).  Channels K-1 .. 1 run a chunk first and
// leave, per stage, the StreamSrc their PSD kernel would have read; channel 0 then runs the same chunk and,
// where its PSD kernel would go, launches the block kernels over all sources.  All cascades order all their
// work on ONE stream (no deep / PSD side streams), so stream order alone makes every launch follow all
// channels' decimators and precede any later overwrite of the buffers it reads; between two lockstep steps each
// stage runs at most once, so the source a channel left for a stage is the one channel 0's launch needs.
//
// Block decomposition (DESIGN.md 3b): channels pair up as (0, 1) and (2, 3).  The diagonal block of each pair
// is csd_stage_kernel's four rows; the off-diagonal block (K >= 3) is csm_cross_kernel's eight.  A stage's
// accumulator block is [pair (0,1): Sxx Syy ReSxy ImSxy][pair (2,3): the same][cross: 8 rows], so K = 2 (the
// CSD) has exactly the first four rows.  K = 3 runs pair (2,3)'s csd_stage_kernel with channel 2 in both slots:
// its rows 1..3 are S22 again and are never read.  The two-sided kind (K = 2, DESIGN.md 3c) runs iq_stage_kernel
// instead: a block of two rows, P+ and P-.
#include "sspsd_xcascade.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include "sspsd_csm_kernel.cuh"
#include "sspsd_mix_kernel.cuh"

namespace sspsd {

namespace {

enum { DIAG = 0, CROSS = 1, IQ = 2 };  // BlockKernels::k

template <int LOG2N>
BlockKernels block_kernels_t()
{
    using PL = Plan<LOG2N + 1>;
    // two CTAs per SM up to 256 threads, one above; the cross kernel's 110 KB: 2 x (110 KB + 1 KB reserved) of the
    // SM's 228 KB
    const bool two = PL::NT <= 256;
    return {{{csd_stage_kernel<LOG2N>, csd_smem_bytes<LOG2N>, two ? 100 * 1024 : 200 * 1024, CSD_ROWS,
              "csd_stage_kernel launch"},
             {csm_cross_kernel<LOG2N>, csm_smem_bytes<LOG2N>, two ? 110 * 1024 : 220 * 1024, CSM_XROWS,
              "csm_cross_kernel launch"},
             {iq_stage_kernel<LOG2N>, csd_smem_bytes<LOG2N>, two ? 100 * 1024 : 200 * 1024, IQ_ROWS,
              "iq_stage_kernel launch"}},
            PL::NT,
            PL::G};
}

int block_kernels(int log2n, BlockKernels* out)
{
    switch (log2n) {
#define X(L)                          \
    case L:                           \
        *out = block_kernels_t<L>();  \
        return SSPSD_OK;
        X(6) X(7) X(8) X(9) X(10) X(11) X(12)
#undef X
    default:
        set_error("CsdCascade supports n_fft = 64 .. 4096 (the two-for-one transform is an N-point complex FFT)");
        return SSPSD_EINVAL;
    }
}

// the largest tile (segments) that fits the kernel's budget; raises its dynamic shared-memory limit to that
int prepare_block(const BlockKernel& k, int hop, int* tmax)
{
    int t = 256;
    while (t > 1 && (long long)k.smem(t, hop) > k.budget) --t;
    if ((long long)k.smem(t, hop) > k.budget) {
        set_error("FFT size does not fit in shared memory");
        return SSPSD_EINVAL;
    }
    *tmax = t;
    SSPSD_CUDA(cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.smem(t, hop)));
    return SSPSD_OK;
}

// persistent tiled launch as psd_stage_kernel's: tiles as large as shared memory allows once there is enough
// work, about two CTAs per SM walking contiguous ranges of tiles
struct TiledLaunch {
    int T, tile_cap, tpc, grid;
};
TiledLaunch tiled_launch(uint64_t nseg, int groups, int tmax, int hop, int n, int num_sms)
{
    TiledLaunch l;
    const long long t = ((long long)nseg + 2ll * num_sms - 1) / (2ll * num_sms);
    l.T = (int)std::max<long long>(std::min<long long>(groups, (long long)nseg), std::min<long long>(t, tmax));
    l.T = std::min(l.T, tmax);
    l.tile_cap = (l.T - 1) * hop + n;
    const long long ntiles = ((long long)nseg + l.T - 1) / l.T;
    l.tpc = (int)std::max<long long>(1, (ntiles + 2ll * num_sms - 1) / (2ll * num_sms));
    l.grid = (int)((ntiles + l.tpc - 1) / l.tpc);
    return l;
}

}  // namespace

size_t XCascade::block_rows() const { return two_sided_ ? IQ_ROWS : k_ == 2 ? CSD_ROWS : 2 * CSD_ROWS + CSM_XROWS; }

XCascade::~XCascade()
{
    if (n_ == 0) return;
    DeviceGuard g(cfg_.device);
    cudaStreamSynchronize(stream_);
    cudaFree(d_win_);
    cudaFree(d_tw_);
    cudaFree(d_acc_);
    cudaFree(d_part_);
    cudaFree(d_xpart_);
    if (h_acc_) cudaFreeHost(h_acc_);
}

sspsd_config XCascade::channel_cfg() const
{
    sspsd_config c = cfg_;
    c.stream = stream_;
    return c;
}

// everything but the channels: the stream, the window and twiddle tables, the accumulator blocks
int XCascade::setup(const sspsd_config& cfg, int k, bool two_sided)
{
    if (k < 2 || k > 4 || (two_sided && k != 2)) {
        set_error("CsmCascade supports 2 .. 4 channels");
        return SSPSD_EINVAL;
    }
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
    k_ = k;
    two_sided_ = two_sided;
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
    int rc = block_kernels((int)log2n_, &kern_);
    if (rc) return rc;
    if (two_sided_) {
        rc = prepare_block(kern_.k[IQ], hop, &tmax_[IQ]);
        if (rc) return rc;
    }
    for (int kind = DIAG; !two_sided_ && kind <= (k_ > 2 ? CROSS : DIAG); ++kind) {
        rc = prepare_block(kern_.k[kind], hop, &tmax_[kind]);
        if (rc) return rc;
    }

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
    const size_t acc_bytes = acc_floats() * sizeof(float);
    SSPSD_CUDA(cudaMalloc(&d_win_, n * sizeof(float)));
    SSPSD_CUDA(cudaMalloc(&d_tw_, n * sizeof(float2)));
    SSPSD_CUDA(cudaMalloc(&d_acc_, acc_bytes));
    SSPSD_CUDA(cudaMallocHost(&h_acc_, acc_bytes));
    SSPSD_CUDA(cudaMemcpyAsync(d_win_, win.data(), n * sizeof(float), cudaMemcpyHostToDevice, stream_));
    SSPSD_CUDA(cudaMemcpyAsync(d_tw_, tw.data(), n * sizeof(float2), cudaMemcpyHostToDevice, stream_));
    SSPSD_CUDA(cudaMemsetAsync(d_acc_, 0, acc_bytes, stream_));
    SSPSD_CUDA(cudaStreamSynchronize(stream_));  // the host vectors above go out of scope
    for (int c = 0; c < k_; ++c) {
        ch_[c].one_stream_ = true;
        ch_[c].hook_ = this;
    }
    n_ = n;
    return SSPSD_OK;
}

int XCascade::init(const sspsd_config& cfg, int k, bool two_sided)
{
    int rc = setup(cfg, k, two_sided);
    if (rc) return rc;
    const sspsd_config c = channel_cfg();
    for (int i = 0; i < k_; ++i) {
        rc = ch_[i].init(c, SSPSD_MAX_STAGES);
        if (rc) return rc;
    }
    return SSPSD_OK;
}

int XCascade::clone_from(XCascade& o)
{
    int rc = o.sync();
    if (rc) return rc;
    rc = setup(o.cfg_, o.k_, o.two_sided_);  // the caller's stream (cfg.stream) is shared by the copy, a private one is not
    if (rc) return rc;
    const sspsd_config c = channel_cfg();
    for (int i = 0; i < k_; ++i) {
        rc = ch_[i].clone_from(o.ch_[i], &c);
        if (rc) return rc;
    }
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    SSPSD_CUDA(cudaMemcpyAsync(d_acc_, o.d_acc_, acc_floats() * sizeof(float), cudaMemcpyDeviceToDevice, stream_));
    SSPSD_CUDA(cudaStreamSynchronize(stream_));
    return SSPSD_OK;
}

int XCascade::reset()
{
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    for (int i = 0; i < k_; ++i) {
        int rc = ch_[i].reset();
        if (rc) return rc;
    }
    for (auto& row : srcs_)
        for (auto& s : row) s.valid = false;
    SSPSD_CUDA(cudaMemsetAsync(d_acc_, 0, acc_floats() * sizeof(float), stream_));
    return SSPSD_OK;
}

int XCascade::ensure_part(float** part, size_t* cap, size_t need)
{
    if (need <= *cap) return SSPSD_OK;
    SSPSD_CUDA(cudaStreamSynchronize(stream_));
    if (*part) SSPSD_CUDA(cudaFree(*part));
    *part = nullptr;
    SSPSD_CUDA(cudaMalloc(part, need * sizeof(float)));
    // the row padding is never written: keep it zero so that the reduction adds nothing there
    SSPSD_CUDA(cudaMemsetAsync(*part, 0, need * sizeof(float), stream_));
    *cap = need;
    return SSPSD_OK;
}

// One block kernel over a stage's segments, its rows at acc: tiles, the partial buffer in deterministic mode (one
// partial block per (CTA, group), summed in row order by reduce_partials_kernel), the launch and the reduction.
int XCascade::launch_block(int kind, XStageParams p, uint64_t nseg, float* acc, float** part, size_t* part_cap)
{
    const BlockKernel& k = kern_.k[kind];
    const int block = (int)(k.rows * stride_);
    const TiledLaunch l = tiled_launch(nseg, kern_.groups, tmax_[kind], p.hop, (int)n_, num_sms_);
    p.T = l.T;
    p.tile_cap = l.tile_cap;
    p.tpc = l.tpc;
    p.acc = acc;
    const int rows = l.grid * kern_.groups;
    if (cfg_.flags & SSPSD_FLAG_DETERMINISTIC) {
        int rc = ensure_part(part, part_cap, (size_t)rows * block);
        if (rc) return rc;
        p.part = *part;
        p.part_stride = block;
    }
    k.fn<<<l.grid, kern_.nt, k.smem(p.T, p.hop), stream_>>>(p);
    if (!cuda_ok(cudaGetLastError(), k.what)) return SSPSD_ECUDA;
    if (p.part) {
        reduce_partials_kernel<<<(block + 127) / 128, 128, 0, stream_>>>(p.acc, p.part, rows, block, block);
        SSPSD_CUDA(cudaGetLastError());
    }
    return SSPSD_OK;
}

// Channels 1 .. k_-1 leave their sources; channel 0's launches the block kernels over all of them.
int XCascade::stage_psd(Cascade& c, size_t i, const StreamSrc& src, uint64_t k0, uint64_t nseg, const EwmaPlan& e)
{
    for (int ci = 1; ci < k_; ++ci) {
        if (&c == &ch_[ci]) {
            srcs_[ci][i] = Source{src, k0, nseg, true};
            return SSPSD_OK;
        }
    }
    for (int ci = 1; ci < k_; ++ci) {
        Source& s = srcs_[ci][i];
        if (!s.valid || s.k0 != k0 || s.nseg != nseg) {
            set_error("internal: channels out of lockstep");
            return SSPSD_EINVAL;
        }
        s.valid = false;
    }
    XStageParams p{};
    p.src[0] = src;
    for (int ci = 1; ci < k_; ++ci) p.src[ci] = srcs_[ci][i].src;
    if (k_ == 3) p.src[3] = p.src[2];  // pair (2, 3)'s diagonal block: channel 2 in both slots, rows 1..3 unused
    p.nch = k_;
    p.k0 = (long long)k0;
    p.nseg = (int)nseg;
    p.hop = (int)ch_[0].hop_;
    p.detrend = ch_[0].detrend_;
    p.win = d_win_;
    p.tw = d_tw_;
    p.stride = (int)stride_;
    p.jb = e.jb;
    p.g_first = e.g_first;
    p.g_s = e.g_s;

    float* acc = d_acc_ + i * block_rows() * stride_;
    if (e.total != 1.0f) {
        // the EWMA pre-scale of the running sums before this batch, over the stage's whole block
        const int nblock = (int)(block_rows() * stride_);
        scale_kernel<<<(nblock + 255) / 256, 256, 0, stream_>>>(acc, nblock, e.total);
        SSPSD_CUDA(cudaGetLastError());
    }
    if (two_sided_) return launch_block(IQ, p, nseg, acc, &d_part_, &part_cap_);
    // diagonal blocks: csd_stage_kernel over pair (0, 1), then (2, 3)
    int rc = launch_block(DIAG, p, nseg, acc, &d_part_, &part_cap_);
    if (rc || k_ == 2) return rc;
    XStageParams q = p;
    q.src[0] = p.src[2];
    q.src[1] = p.src[3];
    rc = launch_block(DIAG, q, nseg, acc + CSD_ROWS * stride_, &d_part_, &part_cap_);
    if (rc) return rc;
    // off-diagonal block: csm_cross_kernel over all channels
    return launch_block(CROSS, p, nseg, acc + 2 * CSD_ROWS * stride_, &d_xpart_, &xpart_cap_);
}

// one lockstep step: the same chunk through channels k_-1 .. 1, then through channel 0 (which launches the kernels)
int XCascade::feed_chunk(const float* const* x, size_t n, bool device)
{
    for (int c = k_ - 1; c >= 0; --c) {
        int rc = device ? ch_[c].feed_device_chunk(x[c], n) : ch_[c].feed_host_chunk(x[c], n);
        if (rc) return rc;
    }
    // the other channels' input buffers of this chunk were read by the kernels queued just now: their next
    // refill waits for them
    for (int c = 1; c < k_; ++c) SSPSD_CUDA(cudaEventRecord(ch_[c].ev_free_[ch_[c].in_buf_ ^ 1], stream_));
    return SSPSD_OK;
}

// Cascade::flush_staged for all channels, chunk by chunk in lockstep
int XCascade::flush_staged()
{
    const size_t staged = ch_[0].staged_;
    if (staged == 0) return SSPSD_OK;
    const int hb = ch_[0].stage_buf_;
    const size_t chunk = (size_t)std::min<uint64_t>(Cascade::host_chunk(), ch_[0].cfg_.max_batch);
    for (size_t pos = 0; pos < staged; pos += chunk) {
        const float* xs[4];
        for (int c = 0; c < k_; ++c) xs[c] = ch_[c].h_stage_[hb] + pos;
        int rc = feed_chunk(xs, std::min(chunk, staged - pos), false);
        if (rc) return rc;
    }
    for (int i = 0; i < k_; ++i) {
        Cascade* c = &ch_[i];
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
    for (size_t j = 1; j < ch_[0].stages_.size(); ++j) {
        for (int c = k_ - 1; c >= 0; --c) {
            rc = ch_[c].run_pending(j);
            if (rc) return rc;
        }
    }
    return SSPSD_OK;
}

int XCascade::process(const float* const* x, size_t n, int mem)
{
    if (n == 0) return SSPSD_OK;
    if (!x) {
        set_error("null input");
        return SSPSD_EINVAL;
    }
    for (int c = 0; c < k_; ++c) {
        if (!x[c]) {
            set_error("null input");
            return SSPSD_EINVAL;
        }
    }
    if (mem != SSPSD_MEM_HOST && mem != SSPSD_MEM_DEVICE) {
        set_error("bad mem kind");
        return SSPSD_EINVAL;
    }
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    int rc;
    const float* xs[4];
    const uint64_t max_batch = ch_[0].cfg_.max_batch;
    if (mem == SSPSD_MEM_DEVICE) {
        rc = flush_staged();
        if (rc) return rc;
        // Cascade::process_device's chunks: at most max_batch, boundaries 16-byte aligned relative to every input
        const size_t nchunks = (n + max_batch - 1) / max_batch;
        size_t per = (n + nchunks - 1) / nchunks;
        per = (per + 4095) & ~(size_t)4095;
        for (size_t pos = 0; pos < n; pos += per) {
            for (int c = 0; c < k_; ++c) xs[c] = x[c] + pos;
            rc = feed_chunk(xs, std::min<size_t>(n - pos, per), true);
            if (rc) return rc;
        }
        return SSPSD_OK;
    }
    const uint64_t hs = ch_[0].cfg_.host_stage;
    if (n < hs) {
        // small calls are collected in the channels' pinned staging buffers (Cascade::process_host)
        for (int i = 0; i < k_; ++i) {
            Cascade* c = &ch_[i];
            if (!c->h_stage_[0]) {
                SSPSD_CUDA(cudaMallocHost(&c->h_stage_[0], hs * sizeof(float)));
                SSPSD_CUDA(cudaMallocHost(&c->h_stage_[1], hs * sizeof(float)));
            }
        }
        size_t pos = 0;
        while (pos < n) {
            const size_t take = std::min<size_t>(n - pos, hs - ch_[0].staged_);
            for (int i = 0; i < k_; ++i) {
                Cascade* c = &ch_[i];
                std::memcpy(c->h_stage_[c->stage_buf_] + c->staged_, x[i] + pos, take * sizeof(float));
                c->staged_ += take;
            }
            pos += take;
            if (ch_[0].staged_ == hs) {
                rc = flush_staged();
                if (rc) return rc;
            }
        }
        return SSPSD_OK;
    }
    rc = flush_staged();
    if (rc) return rc;
    const size_t chunk = (size_t)std::min<uint64_t>(Cascade::host_chunk(), max_batch);
    for (int c = 0; c < k_; ++c) ch_[c].last_copy_ = -1;
    for (size_t pos = 0; pos < n; pos += chunk) {
        for (int c = 0; c < k_; ++c) xs[c] = x[c] + pos;
        rc = feed_chunk(xs, std::min(chunk, n - pos), false);
        if (rc) return rc;
    }
    // the caller's buffers are borrowed for the call only: wait for the last H2D copies
    for (int i = 0; i < k_; ++i) {
        Cascade* c = &ch_[i];
        if (c->last_copy_ >= 0) SSPSD_CUDA(cudaEventSynchronize(c->ev_copied_[c->last_copy_]));
    }
    return SSPSD_OK;
}

int XCascade::set_avg(sspsd_avg_opts a)
{
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    int rc = flush_all();  // options apply to segments completed after the call
    if (rc) return rc;
    for (int c = 0; c < k_; ++c) {
        rc = ch_[c].set_avg(a);
        if (rc) return rc;
    }
    return SSPSD_OK;
}

int XCascade::set_detrend(int d)
{
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    int rc = flush_all();
    if (rc) return rc;
    for (int c = 0; c < k_; ++c) {
        rc = ch_[c].set_detrend(d);  // validates d (Linear: SSPSD_EUNIMPLEMENTED)
        if (rc) return rc;
    }
    return SSPSD_OK;
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
    *n = ch_[0].n_stages();
    return SSPSD_OK;
}

// Time-chunk mode: the channels' bookkeeping stays identical, so windowed channels still run the same stages over the
// same (owned) segment ranges and channel 0's hook launches the block kernels over exactly the segments the rank owns.
int XCascade::seek(uint64_t pos)
{
    for (int c = 0; c < k_; ++c) {
        int rc = ch_[c].seek(pos);
        if (rc) return rc;
    }
    return SSPSD_OK;
}

int XCascade::set_window(uint64_t own_lo, uint64_t own_hi, uint32_t n_local)
{
    for (int c = 0; c < k_; ++c) {
        int rc = ch_[c].set_window(own_lo, own_hi, n_local);
        if (rc) return rc;
    }
    return SSPSD_OK;
}

int XCascade::take_tail(uint64_t j_lo, uint64_t j_hi, float* const* out, size_t* len, uint64_t* first)
{
    int rc = sync();  // staged input in lockstep first: the channels' own sync() then finds nothing to run
    if (rc) return rc;
    const size_t cap = *len;
    for (int c = 0; c < k_; ++c) {
        *len = cap;
        rc = ch_[c].take_tail(j_lo, j_hi, out[c], len, first, SSPSD_MEM_DEVICE);
        if (rc) return rc;
    }
    return SSPSD_OK;
}

// feed_chunk's order for a deep stage: per chunk, channels k_-1 .. 1 leave their sources, then channel 0 launches
int XCascade::process_stage(uint32_t stage, const float* const* x, size_t n)
{
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    int rc = flush_all();
    if (rc) return rc;
    const size_t chunk = (size_t)ch_[0].cfg_.max_batch;
    for (size_t pos = 0; pos < n; pos += chunk) {
        const size_t m = std::min(chunk, n - pos);
        for (int c = k_ - 1; c >= 0; --c) {
            rc = ch_[c].process_stage(stage, x[c] + pos, m, SSPSD_MEM_DEVICE);
            if (rc) return rc;
        }
    }
    return SSPSD_OK;
}

int XCascade::set_stream_state(uint32_t stage, uint64_t samples, uint64_t segments)
{
    for (int c = 0; c < k_; ++c) {
        int rc = ch_[c].set_stream_state(stage, samples, segments);
        if (rc) return rc;
    }
    return SSPSD_OK;
}

int XCascade::partials(sspsd_partials* out)
{
    if (!out) return SSPSD_EINVAL;
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    int rc = flush_all();
    if (rc) return rc;
    rc = ch_[0].partials(out);  // the counts (every channel has the same)
    if (rc) return rc;
    out->acc = d_acc_;
    out->acc_stride = stride_;
    return SSPSD_OK;
}

// The common start of read() and read_matrix(): flush, export the book, size the readout (*pl bins, *ns breaks) and
// check the caller's capacity (outs: the output pointers are non-null), then copy every stage's block to h_acc_.
// With nothing to merge (*ns == 0) or too little room, *p_len and *b_len are set here and the caller returns rc.
int XCascade::read_rows(const sspsd_merge_opts& o, bool outs, size_t* p_len, sspsd_break* b, size_t* b_len,
                        uint64_t (&book)[4 * SSPSD_MAX_STAGES + 2], size_t* pl, size_t* ns)
{
    *ns = 0;
    if (!p_len || !b_len) {
        set_error("null length pointer");
        return SSPSD_EINVAL;
    }
    DeviceGuard g(cfg_.device);
    if (!g.ok) return SSPSD_ECUDA;
    int rc = flush_all();
    if (rc) return rc;
    const size_t n_st = ch_[0].stages_.size();
    ch_[0].export_book(book);
    size_t bl = 0;
    *pl = 0;
    Cascade::merge_host(ch_[0].cfg_, book, nullptr, 0, o, nullptr, pl, nullptr, &bl);
    const bool fits = (*pl <= *p_len) && (n_st <= *b_len) && (*pl == 0 || outs) && (n_st == 0 || b);
    if (!fits || n_st == 0) {
        *p_len = *pl;
        *b_len = n_st;
        if (!fits) {
            set_error("output capacity too small");
            return SSPSD_ESHORT;
        }
        return SSPSD_OK;
    }
    *ns = n_st;
    SSPSD_CUDA(cudaMemcpyAsync(h_acc_, d_acc_, n_st * block_rows() * stride_ * sizeof(float), cudaMemcpyDeviceToHost,
                               stream_));
    SSPSD_CUDA(cudaStreamSynchronize(stream_));
    return SSPSD_OK;
}

// PsdCascade::psd's merge (Cascade::merge_host) applied to each row: same breaks, same 1/(gain_i 8^i) per stage
int XCascade::read(const sspsd_merge_opts& o, float* pxx, float* pyy, float* pxy, size_t* p_len, sspsd_break* b,
                   size_t* b_len)
{
    uint64_t book[4 * SSPSD_MAX_STAGES + 2];
    size_t pl, ns;
    int rc = read_rows(o, pxx && pyy && pxy, p_len, b, b_len, book, &pl, &ns);
    if (rc || ns == 0) return rc;
    const size_t block = block_rows() * stride_;
    std::vector<float> re(pl), im(pl);
    float* outs[CSD_ROWS] = {pxx, pyy, re.data(), im.data()};
    for (int r = 0; r < CSD_ROWS; ++r) {
        size_t pr = pl, br = ns;
        rc = Cascade::merge_host(ch_[0].cfg_, book, h_acc_ + (size_t)r * stride_, block, o, outs[r], &pr, b, &br);
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

// The two-sided kind: P+ and P- merged as read() merges its rows, then halved (exact): the two-sided density, so a
// real x fed as (x, 0) reads back psd(x) / 2 on each side.
int XCascade::read_two_sided(const sspsd_merge_opts& o, float* p_pos, float* p_neg, size_t* p_len, sspsd_break* b,
                             size_t* b_len)
{
    uint64_t book[4 * SSPSD_MAX_STAGES + 2];
    size_t pl, ns;
    int rc = read_rows(o, p_pos && p_neg, p_len, b, b_len, book, &pl, &ns);
    if (rc || ns == 0) return rc;
    const size_t block = block_rows() * stride_;
    float* outs[IQ_ROWS] = {p_pos, p_neg};
    for (int r = 0; r < IQ_ROWS; ++r) {
        size_t pr = pl, br = ns;
        rc = Cascade::merge_host(ch_[0].cfg_, book, h_acc_ + (size_t)r * stride_, block, o, outs[r], &pr, b, &br);
        if (rc) return rc;
        for (size_t k = 0; k < pl; ++k) outs[r][k] *= 0.5f;
    }
    *p_len = pl;
    *b_len = ns;
    return SSPSD_OK;
}

// The whole K x K matrix, s[2 ((i K + j) p_len + k) + {0, 1}]: every stored row merged as read() merges its rows,
// the diagonal real (imaginary part 0), the lower triangle the conjugate of the upper.
int XCascade::read_matrix(const sspsd_merge_opts& o, float* s, size_t* p_len, sspsd_break* b, size_t* b_len)
{
    uint64_t book[4 * SSPSD_MAX_STAGES + 2];
    size_t pl, ns;
    int rc = read_rows(o, s != nullptr, p_len, b, b_len, book, &pl, &ns);
    if (rc || ns == 0) return rc;
    const size_t block = block_rows() * stride_;
    // stored rows of the upper triangle: (i, j) -> (row of Re, row of Im); the diagonal has no Im row
    int re_row[4][4], im_row[4][4];
    for (int a = 0; 2 * a < k_; ++a) {
        const int i = 2 * a, r = a * CSD_ROWS;
        re_row[i][i] = r;
        re_row[i + 1][i + 1] = r + 1;
        re_row[i][i + 1] = r + 2;
        im_row[i][i + 1] = r + 3;
    }
    for (int i = 0; i < 2; ++i)
        for (int j = 2; j < 4; ++j) {
            const int r = 2 * CSD_ROWS + 2 * (2 * i + (j - 2));  // S02, S03, S12, S13
            re_row[i][j] = r;
            im_row[i][j] = r + 1;
        }
    std::vector<float> re(pl), im(pl);
    auto merged = [&](int row, float* out) {
        size_t pr = pl, br = ns;
        return Cascade::merge_host(ch_[0].cfg_, book, h_acc_ + (size_t)row * stride_, block, o, out, &pr, b, &br);
    };
    for (int i = 0; i < k_; ++i) {
        for (int j = i; j < k_; ++j) {
            float* up = s + 2 * ((size_t)(i * k_ + j) * pl);
            float* lo = s + 2 * ((size_t)(j * k_ + i) * pl);
            rc = merged(re_row[i][j], re.data());
            if (rc) return rc;
            if (i == j) {
                for (size_t k = 0; k < pl; ++k) {
                    up[2 * k] = re[k];
                    up[2 * k + 1] = 0.0f;
                }
                continue;
            }
            rc = merged(im_row[i][j], im.data());
            if (rc) return rc;
            for (size_t k = 0; k < pl; ++k) {
                up[2 * k] = re[k];
                up[2 * k + 1] = im[k];
                lo[2 * k] = re[k];
                lo[2 * k + 1] = -im[k];
            }
        }
    }
    *p_len = pl;
    *b_len = ns;
    return SSPSD_OK;
}


ZoomCascade::~ZoomCascade()
{
    if (!d_i_ && !h_stage_[0]) return;
    DeviceGuard g(x_.device());
    cudaStreamSynchronize(x_.stream());
    cudaFree(d_i_);
    cudaFree(d_q_);
    cudaFree(d_x_);
    for (int b = 0; b < 2; ++b) {
        if (h_stage_[b]) cudaFreeHost(h_stage_[b]);
        if (ev_stage_[b]) cudaEventDestroy(ev_stage_[b]);
    }
}

int ZoomCascade::init(const sspsd_config& cfg, int mode, uint32_t ftw)
{
    if (mode != SSPSD_ZOOM_IQ && mode != SSPSD_ZOOM_HETERODYNE) {
        set_error("unknown zoom mode");
        return SSPSD_EINVAL;
    }
    if (mode == SSPSD_ZOOM_IQ && ftw != 0) {
        set_error("I/Q mode has no carrier: ftw must be 0");
        return SSPSD_EINVAL;
    }
    mode_ = mode;
    ftw_ = ftw;
    stage_cap_ = std::max<size_t>(4096, (cfg.host_stage ? (size_t)cfg.host_stage : (size_t)1 << 22) & ~(size_t)3);
    return x_.init(cfg, 2, true);
}

int ZoomCascade::clone_from(ZoomCascade& o)
{
    int rc = o.flush_host();  // XCascade::clone_from then syncs the source's stream
    if (rc) return rc;
    rc = x_.clone_from(o.x_);
    if (rc) return rc;
    mode_ = o.mode_;
    ftw_ = o.ftw_;
    pos_ = o.pos_;
    stage_cap_ = o.stage_cap_;
    return SSPSD_OK;
}

int ZoomCascade::reset()
{
    int rc = x_.reset();
    if (rc) return rc;
    pos_ = 0;
    staged_ = 0;
    return SSPSD_OK;
}

int ZoomCascade::seek(uint64_t pos)
{
    if (staged_) {
        set_error("seek() needs a fresh cascade");
        return SSPSD_EINVAL;
    }
    int rc = x_.seek(pos);
    if (rc) return rc;
    pos_ = pos;
    return SSPSD_OK;
}

int ZoomCascade::ensure_mix()
{
    if (d_i_) return SSPSD_OK;
    mix_cap_ = (size_t)1 << 23;  // as Cascade::host_chunk()
    SSPSD_CUDA(cudaMalloc(&d_i_, mix_cap_ * sizeof(float)));
    SSPSD_CUDA(cudaMalloc(&d_q_, mix_cap_ * sizeof(float)));
    return SSPSD_OK;
}

// Mixer launches of at most mix_cap_ samples (a multiple of 4, so that a stream position that is a multiple of 4
// stays one and stage 0 reads the mix buffers in place), each followed by the XCascade's launches over them.
int ZoomCascade::mix_and_feed(const float* d_x, size_t n)
{
    int rc = ensure_mix();
    if (rc) return rc;
    for (size_t off = 0; off < n; off += mix_cap_) {
        const size_t m = std::min(mix_cap_, n - off);
        const int grid = (int)std::min<size_t>((m + 255) / 256, 148 * 16);
        heterodyne_kernel<<<grid, 256, 0, x_.stream()>>>(d_x + off, m, pos_, ftw_, d_i_, d_q_);
        SSPSD_CUDA(cudaGetLastError());
        const float* xs[2] = {d_i_, d_q_};
        rc = x_.process(xs, m, SSPSD_MEM_DEVICE);
        if (rc) return rc;
        pos_ += m;
    }
    return SSPSD_OK;
}

// the staged host samples: H2D copy, mixer, cascade, all on the stream; the other pinned buffer becomes current
int ZoomCascade::flush_host()
{
    if (staged_ == 0) return SSPSD_OK;
    DeviceGuard g(x_.device());
    if (!g.ok) return SSPSD_ECUDA;
    const int b = stage_buf_;
    SSPSD_CUDA(cudaMemcpyAsync(d_x_, h_stage_[b], staged_ * sizeof(float), cudaMemcpyHostToDevice, x_.stream()));
    SSPSD_CUDA(cudaEventRecord(ev_stage_[b], x_.stream()));
    stage_pending_[b] = true;
    const size_t n = staged_;
    staged_ = 0;
    stage_buf_ ^= 1;
    return mix_and_feed(d_x_, n);
}

int ZoomCascade::process_iq(const float* i, const float* q, size_t n, int mem)
{
    if (mode_ != SSPSD_ZOOM_IQ) {
        set_error("heterodyne mode takes one real stream (sspsd_zoom_process_f32)");
        return SSPSD_EINVAL;
    }
    if (n && (!i || !q)) {
        set_error("null input");
        return SSPSD_EINVAL;
    }
    const float* xs[2] = {i, q};
    return x_.process(xs, n, mem);
}

int ZoomCascade::process_device_mixed(const float* x, size_t n)
{
    int rc = flush_host();
    if (rc) return rc;
    return mix_and_feed(x, n);
}

int ZoomCascade::process(const float* x, size_t n, int mem)
{
    if (mode_ != SSPSD_ZOOM_HETERODYNE) {
        set_error("I/Q mode takes two streams (sspsd_zoom_process_iq_f32)");
        return SSPSD_EINVAL;
    }
    if (n == 0) return SSPSD_OK;
    if (!x) {
        set_error("null input");
        return SSPSD_EINVAL;
    }
    if (mem != SSPSD_MEM_HOST && mem != SSPSD_MEM_DEVICE) {
        set_error("bad mem kind");
        return SSPSD_EINVAL;
    }
    DeviceGuard g(x_.device());
    if (!g.ok) return SSPSD_ECUDA;
    if (mem == SSPSD_MEM_DEVICE) return process_device_mixed(x, n);
    if (!h_stage_[0]) {
        for (int b = 0; b < 2; ++b) {
            SSPSD_CUDA(cudaMallocHost(&h_stage_[b], stage_cap_ * sizeof(float)));
            SSPSD_CUDA(cudaEventCreateWithFlags(&ev_stage_[b], cudaEventDisableTiming));
        }
        SSPSD_CUDA(cudaMalloc(&d_x_, stage_cap_ * sizeof(float)));
    }
    for (size_t pos = 0; pos < n;) {
        const int b = stage_buf_;
        if (stage_pending_[b]) {  // its previous H2D copy still reads it
            SSPSD_CUDA(cudaEventSynchronize(ev_stage_[b]));
            stage_pending_[b] = false;
        }
        const size_t take = std::min(n - pos, stage_cap_ - staged_);
        std::memcpy(h_stage_[b] + staged_, x + pos, take * sizeof(float));
        staged_ += take;
        pos += take;
        if (staged_ == stage_cap_) {
            int rc = flush_host();
            if (rc) return rc;
        }
    }
    return SSPSD_OK;
}

int ZoomCascade::set_avg(sspsd_avg_opts a)
{
    int rc = flush_host();
    return rc ? rc : x_.set_avg(a);
}

int ZoomCascade::set_detrend(int d)
{
    int rc = flush_host();
    return rc ? rc : x_.set_detrend(d);
}

int ZoomCascade::flush()
{
    int rc = flush_host();
    return rc ? rc : x_.flush();
}

int ZoomCascade::sync()
{
    int rc = flush_host();
    return rc ? rc : x_.sync();
}

int ZoomCascade::read(const sspsd_merge_opts& o, float* p_pos, float* p_neg, size_t* p_len, sspsd_break* b,
                      size_t* b_len)
{
    int rc = flush_host();
    return rc ? rc : x_.read_two_sided(o, p_pos, p_neg, p_len, b, b_len);
}

int ZoomCascade::num_stages(uint32_t* n)
{
    int rc = flush_host();
    return rc ? rc : x_.num_stages(n);
}

}  // namespace sspsd

using sspsd::set_error;

namespace {

// create / clone of either handle (sspsd_csd: k = 2)
template <class H>
int32_t x_create(const sspsd_config* cfg, int k, H** out)
{
    if (!cfg || !out) {
        set_error("null argument");
        return SSPSD_EINVAL;
    }
    *out = nullptr;
    H* h = new (std::nothrow) H();
    if (!h) return SSPSD_ENOMEM;
    int rc = h->c.init(*cfg, k);
    if (rc) {
        delete h;
        return rc;
    }
    *out = h;
    return SSPSD_OK;
}

template <class H>
int32_t x_clone(H* h, H** out)
{
    if (!h || !out) {
        set_error("null argument");
        return SSPSD_EINVAL;
    }
    *out = nullptr;
    H* n = new (std::nothrow) H();
    if (!n) return SSPSD_ENOMEM;
    int rc = n->c.clone_from(h->c);
    if (rc) {
        delete n;
        return rc;
    }
    *out = n;
    return SSPSD_OK;
}

// Channel i <- trace map[i] of every decoded sub-chunk: one XCascade::process on the handle's one stream.  All
// channels sit at one stream position and the decoder's trace buffers share one alignment, so either every channel
// reads its sub-chunk in place or every channel takes the realigning copy.
struct XSink : sspsd::FrameSink {
    sspsd::XCascade& x;
    const uint32_t* map;
    XSink(sspsd::XCascade& x_, const uint32_t* map_) : x(x_), map(map_) {}
    int check_device(int device) override
    {
        if (x.device() != device) {
            set_error("cross-spectral handle and decoder live on different devices");
            return SSPSD_EINVAL;
        }
        return SSPSD_OK;
    }
    int accept(unsigned int fmt) override
    {
        const uint32_t ntr = fmt == SSPSD_FORMAT_MPLL ? 3 : 4;
        for (int i = 0; i < x.channels(); ++i)
            if (map[i] >= ntr) {
                set_error("trace index " + std::to_string(map[i]) + " past the " + std::to_string(ntr) +
                          " traces of the frames' format");
                return SSPSD_EINVAL;
            }
        return SSPSD_OK;
    }
    int consume(sspsd_decoder* d, float* const* tr, uint32_t, size_t ns, cudaEvent_t ready) override
    {
        const float* xs[4];
        for (int i = 0; i < x.channels(); ++i) xs[i] = tr[map[i]];
        if (ready) SSPSD_CUDA(cudaStreamWaitEvent(x.stream(), ready, 0));
        int rc = x.process(xs, ns, SSPSD_MEM_DEVICE);
        if (rc) return rc;
        for (int i = 0; i < x.channels(); ++i) {
            rc = sspsd::trace_consumed(d, (int)map[i], x.stream());
            if (rc) return rc;
        }
        return SSPSD_OK;
    }
};

// Heterodyne mode: trace map[0] of every decoded sub-chunk, mixed and fed on the handle's one stream (the mixer reads
// the decoder's trace buffer in stream order, so the consumption event recorded after it covers that read).
struct MixSink : sspsd::FrameSink {
    sspsd::ZoomCascade& z;
    uint32_t trace;
    MixSink(sspsd::ZoomCascade& z_, uint32_t t) : z(z_), trace(t) {}
    int check_device(int device) override
    {
        if (z.x().device() != device) {
            set_error("zoom handle and decoder live on different devices");
            return SSPSD_EINVAL;
        }
        return SSPSD_OK;
    }
    int accept(unsigned int fmt) override
    {
        const uint32_t ntr = fmt == SSPSD_FORMAT_MPLL ? 3 : 4;
        if (trace >= ntr) {
            set_error("trace index " + std::to_string(trace) + " past the " + std::to_string(ntr) +
                      " traces of the frames' format");
            return SSPSD_EINVAL;
        }
        return SSPSD_OK;
    }
    int consume(sspsd_decoder* d, float* const* tr, uint32_t, size_t ns, cudaEvent_t ready) override
    {
        const cudaStream_t s = z.x().stream();
        if (ready) SSPSD_CUDA(cudaStreamWaitEvent(s, ready, 0));
        int rc = z.process_device_mixed(tr[trace], ns);
        return rc ? rc : sspsd::trace_consumed(d, (int)trace, s);
    }
};

// sspsd_csd / sspsd_csm_process_frames; traces: one index per channel, NULL for 0 .. K-1
template <class H>
int32_t x_process_frames(sspsd_decoder* d, H* h, const uint32_t* traces, const uint8_t* frames, size_t n_frames,
                         size_t frame_len, size_t frame_stride, int32_t frames_mem, sspsd_loss* loss,
                         sspsd_decode_info* info)
{
    if (!d || !h || (n_frames && !frames) || frame_stride < frame_len) {
        set_error("bad argument");
        return SSPSD_EINVAL;
    }
    uint32_t map[4] = {0, 1, 2, 3};
    if (traces) {
        for (int i = 0; i < h->c.channels(); ++i) {
            if (traces[i] >= SSPSD_MAX_TRACES) {
                set_error("trace index " + std::to_string(traces[i]) + " out of range (frames carry at most 4 traces)");
                return SSPSD_EINVAL;
            }
            map[i] = traces[i];
        }
    }
    XSink sink(h->c, map);
    return sspsd::process_frames(d, sink, frames, n_frames, frame_len, frame_stride, frames_mem, loss, info);
}

// the trace map of a zoom handle: I/Q mode two indices (i, q), heterodyne mode one; NULL for 0 (.. 1)
int check_traces(const uint32_t* traces, int n, uint32_t* map)
{
    for (int i = 0; i < n; ++i) {
        map[i] = traces ? traces[i] : (uint32_t)i;
        if (map[i] >= SSPSD_MAX_TRACES) {
            set_error("trace index " + std::to_string(map[i]) + " out of range (frames carry at most 4 traces)");
            return SSPSD_EINVAL;
        }
    }
    return SSPSD_OK;
}

}  // namespace

int32_t sspsd_csd_create(const sspsd_config* cfg, sspsd_csd** out) { return x_create(cfg, 2, out); }

void sspsd_csd_destroy(sspsd_csd* h) { delete h; }

int32_t sspsd_csd_clone(sspsd_csd* h, sspsd_csd** out) { return x_clone(h, out); }

int32_t sspsd_csd_reset(sspsd_csd* h) { return h ? h->c.reset() : SSPSD_EINVAL; }

int32_t sspsd_csd_process_f32(sspsd_csd* h, const float* x, const float* y, size_t n, int32_t mem)
{
    if (!h) return SSPSD_EINVAL;
    if (n && (!x || !y)) {
        set_error("null input");
        return SSPSD_EINVAL;
    }
    const float* xs[2] = {x, y};
    return h->c.process(xs, n, mem);
}

int32_t sspsd_csd_process_frames(sspsd_decoder* d, sspsd_csd* c, uint32_t trace_x, uint32_t trace_y,
                                 const uint8_t* frames, size_t n_frames, size_t frame_len, size_t frame_stride,
                                 int32_t frames_mem, sspsd_loss* loss, sspsd_decode_info* info)
{
    const uint32_t traces[2] = {trace_x, trace_y};
    return x_process_frames(d, c, traces, frames, n_frames, frame_len, frame_stride, frames_mem, loss, info);
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

int32_t sspsd_csm_create(const sspsd_config* cfg, int32_t k, sspsd_csm** out) { return x_create(cfg, k, out); }

void sspsd_csm_destroy(sspsd_csm* h) { delete h; }

int32_t sspsd_csm_clone(sspsd_csm* h, sspsd_csm** out) { return x_clone(h, out); }

int32_t sspsd_csm_channels(const sspsd_csm* h, int32_t* k)
{
    if (!h || !k) return SSPSD_EINVAL;
    *k = h->c.channels();
    return SSPSD_OK;
}

int32_t sspsd_csm_reset(sspsd_csm* h) { return h ? h->c.reset() : SSPSD_EINVAL; }

int32_t sspsd_csm_process_f32(sspsd_csm* h, const float* const* x, size_t n, int32_t mem)
{
    if (!h) return SSPSD_EINVAL;
    return h->c.process(x, n, mem);
}

int32_t sspsd_csm_process_frames(sspsd_decoder* d, sspsd_csm* m, const uint32_t* traces, const uint8_t* frames,
                                 size_t n_frames, size_t frame_len, size_t frame_stride, int32_t frames_mem,
                                 sspsd_loss* loss, sspsd_decode_info* info)
{
    return x_process_frames(d, m, traces, frames, n_frames, frame_len, frame_stride, frames_mem, loss, info);
}

int32_t sspsd_csm_set_avg(sspsd_csm* h, sspsd_avg_opts avg) { return h ? h->c.set_avg(avg) : SSPSD_EINVAL; }

int32_t sspsd_csm_set_detrend(sspsd_csm* h, int32_t d) { return h ? h->c.set_detrend(d) : SSPSD_EINVAL; }

int32_t sspsd_csm_rbw(const sspsd_csm* h, float* rbw)
{
    if (!h || !rbw) return SSPSD_EINVAL;
    *rbw = h->c.rbw();
    return SSPSD_OK;
}

int32_t sspsd_csm_read(sspsd_csm* h, const sspsd_merge_opts* opts, float* s, size_t* p_len, sspsd_break* b,
                       size_t* b_len)
{
    if (!h) return SSPSD_EINVAL;
    sspsd_merge_opts o{0, 1, 0};  // MergeOpts::default(), psd.rs:350-358
    if (opts) o = *opts;
    return h->c.read_matrix(o, s, p_len, b, b_len);
}

int32_t sspsd_csm_num_stages(sspsd_csm* h, uint32_t* n)
{
    if (!h || !n) return SSPSD_EINVAL;
    return h->c.num_stages(n);
}

int32_t sspsd_csm_stream(const sspsd_csm* h, void** stream)
{
    if (!h || !stream) return SSPSD_EINVAL;
    *stream = (void*)h->c.stream();
    return SSPSD_OK;
}

int32_t sspsd_csm_flush(sspsd_csm* h) { return h ? h->c.flush() : SSPSD_EINVAL; }
int32_t sspsd_csm_sync(sspsd_csm* h) { return h ? h->c.sync() : SSPSD_EINVAL; }

int32_t sspsd_zoom_create(const sspsd_config* cfg, int32_t mode, uint32_t ftw, sspsd_zoom** out)
{
    if (!cfg || !out) {
        set_error("null argument");
        return SSPSD_EINVAL;
    }
    *out = nullptr;
    sspsd_zoom* h = new (std::nothrow) sspsd_zoom();
    if (!h) return SSPSD_ENOMEM;
    int rc = h->z.init(*cfg, mode, ftw);
    if (rc) {
        delete h;
        return rc;
    }
    *out = h;
    return SSPSD_OK;
}

void sspsd_zoom_destroy(sspsd_zoom* h) { delete h; }

int32_t sspsd_zoom_clone(sspsd_zoom* h, sspsd_zoom** out)
{
    if (!h || !out) {
        set_error("null argument");
        return SSPSD_EINVAL;
    }
    *out = nullptr;
    sspsd_zoom* n = new (std::nothrow) sspsd_zoom();
    if (!n) return SSPSD_ENOMEM;
    int rc = n->z.clone_from(h->z);
    if (rc) {
        delete n;
        return rc;
    }
    *out = n;
    return SSPSD_OK;
}

int32_t sspsd_zoom_reset(sspsd_zoom* h) { return h ? h->z.reset() : SSPSD_EINVAL; }

int32_t sspsd_zoom_process_iq_f32(sspsd_zoom* h, const float* i, const float* q, size_t n, int32_t mem)
{
    return h ? h->z.process_iq(i, q, n, mem) : SSPSD_EINVAL;
}

int32_t sspsd_zoom_process_f32(sspsd_zoom* h, const float* x, size_t n, int32_t mem)
{
    return h ? h->z.process(x, n, mem) : SSPSD_EINVAL;
}

int32_t sspsd_zoom_process_frames(sspsd_decoder* d, sspsd_zoom* z, const uint32_t* traces, const uint8_t* frames,
                                  size_t n_frames, size_t frame_len, size_t frame_stride, int32_t frames_mem,
                                  sspsd_loss* loss, sspsd_decode_info* info)
{
    if (!d || !z || (n_frames && !frames) || frame_stride < frame_len) {
        set_error("bad argument");
        return SSPSD_EINVAL;
    }
    uint32_t map[2];
    const bool iq = z->z.mode() == SSPSD_ZOOM_IQ;
    int rc = check_traces(traces, iq ? 2 : 1, map);
    if (rc) return rc;
    if (iq) {
        XSink sink(z->z.x(), map);
        return sspsd::process_frames(d, sink, frames, n_frames, frame_len, frame_stride, frames_mem, loss, info);
    }
    MixSink sink(z->z, map[0]);
    return sspsd::process_frames(d, sink, frames, n_frames, frame_len, frame_stride, frames_mem, loss, info);
}

int32_t sspsd_zoom_set_avg(sspsd_zoom* h, sspsd_avg_opts avg) { return h ? h->z.set_avg(avg) : SSPSD_EINVAL; }

int32_t sspsd_zoom_set_detrend(sspsd_zoom* h, int32_t d) { return h ? h->z.set_detrend(d) : SSPSD_EINVAL; }

int32_t sspsd_zoom_rbw(const sspsd_zoom* h, float* rbw)
{
    if (!h || !rbw) return SSPSD_EINVAL;
    *rbw = h->z.x().rbw();
    return SSPSD_OK;
}

int32_t sspsd_zoom_read(sspsd_zoom* h, const sspsd_merge_opts* opts, float* p_pos, float* p_neg, size_t* p_len,
                        sspsd_break* b, size_t* b_len)
{
    if (!h) return SSPSD_EINVAL;
    sspsd_merge_opts o{0, 1, 0};  // MergeOpts::default(), psd.rs:350-358
    if (opts) o = *opts;
    return h->z.read(o, p_pos, p_neg, p_len, b, b_len);
}

int32_t sspsd_zoom_carrier(const sspsd_zoom* h, int32_t* mode, uint32_t* ftw)
{
    if (!h || !mode || !ftw) return SSPSD_EINVAL;
    *mode = h->z.mode();
    *ftw = h->z.ftw();
    return SSPSD_OK;
}

int32_t sspsd_zoom_num_stages(sspsd_zoom* h, uint32_t* n)
{
    if (!h || !n) return SSPSD_EINVAL;
    return h->z.num_stages(n);
}

int32_t sspsd_zoom_stream(const sspsd_zoom* h, void** stream)
{
    if (!h || !stream) return SSPSD_EINVAL;
    *stream = (void*)h->z.x().stream();
    return SSPSD_OK;
}

int32_t sspsd_zoom_flush(sspsd_zoom* h) { return h ? h->z.flush() : SSPSD_EINVAL; }
int32_t sspsd_zoom_sync(sspsd_zoom* h) { return h ? h->z.sync() : SSPSD_EINVAL; }

int32_t sspsd_heterodyne_f32(void* stream, const float* x, size_t n, uint64_t pos0, uint32_t ftw, float* i_out,
                             float* q_out)
{
    if (n == 0) return SSPSD_OK;
    if (!x || !i_out || !q_out) {
        set_error("null argument");
        return SSPSD_EINVAL;
    }
    const int grid = (int)std::min<size_t>((n + 255) / 256, 148 * 16);
    sspsd::heterodyne_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, n, pos0, ftw, i_out, q_out);
    return sspsd::cuda_ok(cudaGetLastError(), "heterodyne_kernel launch") ? SSPSD_OK : SSPSD_ECUDA;
}
