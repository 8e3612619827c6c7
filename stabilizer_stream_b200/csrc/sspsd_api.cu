// sspsd_api.cu -- extern "C" boundary (include/sspsd.h) over the internal C++ classes.
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "sspsd_cascade.cuh"
#include "sspsd_decode_kernel.cuh"

using sspsd::Cascade;
using sspsd::set_error;


struct sspsd_decoder {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    uint8_t* d_frames = nullptr;
    size_t frames_cap = 0;
    unsigned int* d_status = nullptr;
    size_t status_cap = 0;
    static constexpr int MAX_SUB = 8;      // sub-chunks of one sspsd_cascade_process_frames call (host frames)
    sspsd::DecodeResult* d_res = nullptr;  // MAX_SUB result slots
    sspsd::DecodeResult* h_res = nullptr;  // pinned, MAX_SUB
    cudaStream_t h2d_stream = nullptr;     // the sub-chunks' copies, so that decode k runs while sub-chunk k + 1 crosses PCIe
    cudaEvent_t ev_copied[MAX_SUB] = {};

    float* d_traces[SSPSD_MAX_TRACES] = {nullptr, nullptr, nullptr, nullptr};
    size_t traces_cap = 0;
    cudaEvent_t ev_decoded = nullptr;
    cudaEvent_t ev_consumed[SSPSD_MAX_TRACES] = {nullptr, nullptr, nullptr, nullptr};
    bool consumed_pending[SSPSD_MAX_TRACES] = {false, false, false, false};
};

namespace {
using DevGuard = sspsd::DeviceGuard;

float powi_f32(float x, int e)
{
    int n = e < 0 ? -e : e;
    float r = 1.0f, b = x;
    while (n) {
        if (n & 1) r *= b;
        b *= b;
        n >>= 1;
    }
    return e < 0 ? 1.0f / r : r;
}
}  // namespace

extern "C" {

const char* sspsd_last_error(void) { return sspsd::last_error(); }

int32_t sspsd_hbf_info(int32_t hbf, uint32_t* drain, uint32_t* halo) { return sspsd::hbf_info(hbf, drain, halo); }

int32_t sspsd_config_default(uint32_t n_fft, sspsd_config* cfg)
{
    if (!cfg) return SSPSD_EINVAL;
    std::memset(cfg, 0, sizeof(*cfg));
    cfg->n_fft = n_fft;
    cfg->window = SSPSD_WINDOW_HANN;  // psd.rs:419
    cfg->hbf = SSPSD_HBF_140;
    cfg->device = 0;
    return SSPSD_OK;
}

// ---------------------------------------------------------------------------------------------
int32_t sspsd_cascade_create(const sspsd_config* cfg, sspsd_cascade** out)
{
    if (!cfg || !out) {
        set_error("null argument");
        return SSPSD_EINVAL;
    }
    *out = nullptr;
    if (cfg->window != SSPSD_WINDOW_HANN && cfg->window != SSPSD_WINDOW_RECT) {
        set_error("unknown window");
        return SSPSD_EINVAL;
    }
    sspsd_cascade* h = new (std::nothrow) sspsd_cascade();
    if (!h) return SSPSD_ENOMEM;
    int rc = h->c.init(*cfg, SSPSD_MAX_STAGES);
    if (rc) {
        delete h;
        return rc;
    }
    *out = h;
    return SSPSD_OK;
}

void sspsd_cascade_destroy(sspsd_cascade* h) { delete h; }

int32_t sspsd_cascade_clone(sspsd_cascade* h, sspsd_cascade** out)
{
    if (!h || !out) return SSPSD_EINVAL;
    *out = nullptr;
    sspsd_cascade* n = new (std::nothrow) sspsd_cascade();
    if (!n) return SSPSD_ENOMEM;
    int rc = n->c.clone_from(h->c);
    if (rc) {
        delete n;
        return rc;
    }
    *out = n;
    return SSPSD_OK;
}

int32_t sspsd_cascade_reset(sspsd_cascade* h) { return h ? h->c.reset() : SSPSD_EINVAL; }

int32_t sspsd_cascade_process_f32(sspsd_cascade* h, const float* x, size_t n, int32_t mem)
{
    if (!h) return SSPSD_EINVAL;
    return h->c.process(x, n, mem);
}

int32_t sspsd_cascade_set_avg(sspsd_cascade* h, sspsd_avg_opts avg) { return h ? h->c.set_avg(avg) : SSPSD_EINVAL; }

int32_t sspsd_cascade_set_detrend(sspsd_cascade* h, int32_t d) { return h ? h->c.set_detrend(d) : SSPSD_EINVAL; }

int32_t sspsd_cascade_rbw(const sspsd_cascade* h, float* rbw)
{
    if (!h || !rbw) return SSPSD_EINVAL;
    *rbw = h->c.rbw();
    return SSPSD_OK;
}

int32_t sspsd_cascade_psd(sspsd_cascade* h, const sspsd_merge_opts* opts, float* p, size_t* p_len, sspsd_break* b,
                          size_t* b_len)
{
    if (!h) return SSPSD_EINVAL;
    sspsd_merge_opts o{0, 1, 0};  // MergeOpts::default(), psd.rs:350-358
    if (opts) o = *opts;
    return h->c.psd(o, p, p_len, b, b_len);
}

int32_t sspsd_cascade_num_stages(sspsd_cascade* h, uint32_t* n)
{
    if (!h || !n) return SSPSD_EINVAL;
    int rc = h->c.flush();
    if (rc) return rc;
    *n = h->c.n_stages();
    return SSPSD_OK;
}

int32_t sspsd_cascade_stream(const sspsd_cascade* h, void** stream)
{
    if (!h || !stream) return SSPSD_EINVAL;
    *stream = (void*)h->c.stream();
    return SSPSD_OK;
}

int32_t sspsd_cascade_flush(sspsd_cascade* h) { return h ? h->c.flush() : SSPSD_EINVAL; }
int32_t sspsd_cascade_sync(sspsd_cascade* h) { return h ? h->c.sync() : SSPSD_EINVAL; }

int32_t sspsd_break_frequencies(const sspsd_break* b, size_t nb, float* f, size_t* f_len)
{
    // Break::frequencies, psd.rs:315-327; Break::rbw, psd.rs:334-336
    if (!f_len || (nb && !b)) return SSPSD_EINVAL;
    size_t need = 0;
    for (size_t i = 0; i < nb; ++i)
        if (b[i].include) need += (size_t)(b[i].bins_end - b[i].bins_start);
    if (need > *f_len || (need && !f)) {
        *f_len = need;
        set_error("output capacity too small");
        return SSPSD_ESHORT;
    }
    *f_len = need;
    size_t n = 0;
    for (size_t i = 0; i < nb; ++i) {
        if (!b[i].include) continue;
        float rbw = 1.0f / (float)(b[i].fft_size * b[i].decimation);
        for (uint64_t k = b[i].bins_start; k < b[i].bins_end; ++k) f[n++] = (float)k * rbw;
    }
    return SSPSD_OK;
}

int32_t sspsd_cascade_partials(sspsd_cascade* h, sspsd_partials* out) { return h ? h->c.partials(out) : SSPSD_EINVAL; }

int32_t sspsd_cascade_set_counts(sspsd_cascade* h, const uint64_t* craw, uint32_t n)
{
    return h ? h->c.set_counts(craw, n) : SSPSD_EINVAL;
}

int32_t sspsd_cascade_seek(sspsd_cascade* h, uint64_t pos) { return h ? h->c.seek(pos) : SSPSD_EINVAL; }
int32_t sspsd_cascade_set_window(sspsd_cascade* h, uint64_t own_lo, uint64_t own_hi, uint32_t n_local)
{
    return h ? h->c.set_window(own_lo, own_hi, n_local) : SSPSD_EINVAL;
}
int32_t sspsd_cascade_take_tail(sspsd_cascade* h, uint64_t j_lo, uint64_t j_hi, float* out, size_t* len,
                                uint64_t* first, int32_t mem)
{
    return h ? h->c.take_tail(j_lo, j_hi, out, len, first, mem) : SSPSD_EINVAL;
}
int32_t sspsd_cascade_process_stage(sspsd_cascade* h, uint32_t stage, const float* x, size_t n, int32_t mem)
{
    return h ? h->c.process_stage(stage, x, n, mem) : SSPSD_EINVAL;
}
int32_t sspsd_cascade_set_stream_state(sspsd_cascade* h, uint32_t stage, uint64_t samples, uint64_t segments)
{
    return h ? h->c.set_stream_state(stage, samples, segments) : SSPSD_EINVAL;
}

int32_t sspsd_cascade_profile_enable(sspsd_cascade* h, int32_t on)
{
    if (!h) return SSPSD_EINVAL;
    h->c.profile_enable(on != 0);
    return SSPSD_OK;
}

int32_t sspsd_cascade_profile_read(sspsd_cascade* h, sspsd_profile* out)
{
    return h ? h->c.profile_read(out) : SSPSD_EINVAL;
}

// ---------------------------------------------------------------------------------------------
int32_t sspsd_stage_create(const sspsd_config* cfg, sspsd_stage** out)
{
    if (!cfg || !out) {
        set_error("null argument");
        return SSPSD_EINVAL;
    }
    *out = nullptr;
    sspsd_stage* h = new (std::nothrow) sspsd_stage();
    if (!h) return SSPSD_ENOMEM;
    int rc = h->c.init(*cfg, 1);
    if (rc) {
        delete h;
        return rc;
    }
    *out = h;
    return SSPSD_OK;
}

void sspsd_stage_destroy(sspsd_stage* h) { delete h; }

int32_t sspsd_stage_stream(const sspsd_stage* h, void** stream)
{
    if (!h || !stream) return SSPSD_EINVAL;
    *stream = (void*)h->c.stream();
    return SSPSD_OK;
}

int32_t sspsd_stage_set_avg(sspsd_stage* h, uint32_t avg) { return h ? h->c.set_stage_avg(avg) : SSPSD_EINVAL; }
int32_t sspsd_stage_set_detrend(sspsd_stage* h, int32_t d) { return h ? h->c.set_detrend(d) : SSPSD_EINVAL; }

int32_t sspsd_stage_process_f32(sspsd_stage* h, const float* x, size_t n, int32_t x_mem, float* y, size_t* y_len,
                                int32_t y_mem)
{
    if (!h || !y_len) return SSPSD_EINVAL;
    if (n == 0) {
        *y_len = 0;
        return SSPSD_OK;
    }
    int rc = h->c.process(x, n, x_mem);
    if (rc) return rc;
    return h->c.take_sink(y, y_len, y_mem);
}

int32_t sspsd_stage_spectrum(sspsd_stage* h, float* out, size_t* len, int32_t mem)
{
    return h ? h->c.stage_spectrum(out, len, mem) : SSPSD_EINVAL;
}

int32_t sspsd_stage_count(sspsd_stage* h, uint32_t* count)
{
    if (!h || !count) return SSPSD_EINVAL;
    *count = h->c.stage_count();
    return SSPSD_OK;
}

int32_t sspsd_stage_gain(sspsd_stage* h, float* gain)
{
    if (!h || !gain) return SSPSD_EINVAL;
    *gain = h->c.stage_gain();
    return SSPSD_OK;
}

int32_t sspsd_stage_buf(sspsd_stage* h, float* out, size_t* len, int32_t mem)
{
    return h ? h->c.stage_buf(out, len, mem) : SSPSD_EINVAL;
}

// ---------------------------------------------------------------------------------------------
int32_t sspsd_decoder_create(int32_t device, void* stream, sspsd_decoder** out)
{
    if (!out) return SSPSD_EINVAL;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        set_error("no CUDA device: this library has no CPU fallback");
        return SSPSD_ECUDA;
    }
    if (device < 0 || device >= ndev) {
        set_error("bad device ordinal");
        return SSPSD_EINVAL;
    }
    DevGuard g(device);
    if (!g.ok) return SSPSD_ECUDA;
    sspsd_decoder* d = new (std::nothrow) sspsd_decoder();
    if (!d) return SSPSD_ENOMEM;
    d->device = device;
    bool ok = true;
    if (stream) {
        d->stream = (cudaStream_t)stream;
    } else {
        ok = ok && sspsd::cuda_ok(cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking), "cudaStreamCreate");
        d->own_stream = ok;
    }
    ok = ok && sspsd::cuda_ok(cudaMalloc(&d->d_res, sspsd_decoder::MAX_SUB * sizeof(sspsd::DecodeResult)), "cudaMalloc");
    ok = ok && sspsd::cuda_ok(cudaMallocHost(&d->h_res, sspsd_decoder::MAX_SUB * sizeof(sspsd::DecodeResult)), "cudaMallocHost");
    ok = ok && sspsd::cuda_ok(cudaStreamCreateWithFlags(&d->h2d_stream, cudaStreamNonBlocking), "cudaStreamCreate");
    for (int k = 0; k < sspsd_decoder::MAX_SUB && ok; ++k)
        ok = sspsd::cuda_ok(cudaEventCreateWithFlags(&d->ev_copied[k], cudaEventDisableTiming), "cudaEventCreate");
    ok = ok && sspsd::cuda_ok(cudaEventCreateWithFlags(&d->ev_decoded, cudaEventDisableTiming), "cudaEventCreate");
    for (int t = 0; t < SSPSD_MAX_TRACES && ok; ++t)
        ok = sspsd::cuda_ok(cudaEventCreateWithFlags(&d->ev_consumed[t], cudaEventDisableTiming), "cudaEventCreate");
    if (!ok) {
        sspsd_decoder_destroy(d);
        return SSPSD_ECUDA;
    }
    *out = d;
    return SSPSD_OK;
}

int32_t sspsd_decoder_stream(const sspsd_decoder* d, void** stream)
{
    if (!d || !stream) return SSPSD_EINVAL;
    *stream = (void*)d->stream;
    return SSPSD_OK;
}

void sspsd_decoder_destroy(sspsd_decoder* d)
{
    if (!d) return;
    DevGuard g(d->device);
    if (d->stream) cudaStreamSynchronize(d->stream);
    if (d->h2d_stream) {
        cudaStreamSynchronize(d->h2d_stream);
        cudaStreamDestroy(d->h2d_stream);
    }
    for (auto& e : d->ev_copied)
        if (e) cudaEventDestroy(e);
    cudaFree(d->d_frames);
    cudaFree(d->d_status);
    cudaFree(d->d_res);
    if (d->h_res) cudaFreeHost(d->h_res);
    for (int t = 0; t < SSPSD_MAX_TRACES; ++t) {
        cudaFree(d->d_traces[t]);
        if (d->ev_consumed[t]) cudaEventDestroy(d->ev_consumed[t]);
    }
    if (d->ev_decoded) cudaEventDestroy(d->ev_decoded);
    if (d->own_stream && d->stream) cudaStreamDestroy(d->stream);
    delete d;
}

}  // extern "C"

namespace {

// make room for `n_bytes` of frames in the decoder's device buffer
int frames_reserve(sspsd_decoder* d, size_t n_bytes)
{
    size_t need = (n_bytes + 15) & ~(size_t)15;
    if (need > d->frames_cap) {
        SSPSD_CUDA(cudaStreamSynchronize(d->stream));
        SSPSD_CUDA(cudaStreamSynchronize(d->h2d_stream));
        if (d->d_frames) SSPSD_CUDA(cudaFree(d->d_frames));
        d->d_frames = nullptr;
        SSPSD_CUDA(cudaMalloc(&d->d_frames, need + 64));
        d->frames_cap = need;
    }
    return SSPSD_OK;
}

// queue the H2D copy of `n_bytes` of frames into the decoder's device buffer (d->stream)
int frames_h2d(sspsd_decoder* d, const uint8_t* frames, size_t n_bytes)
{
    int rc = frames_reserve(d, n_bytes);
    if (rc) return rc;
    SSPSD_CUDA(cudaMemcpyAsync(d->d_frames, frames, n_bytes, cudaMemcpyHostToDevice, d->stream));
    return SSPSD_OK;
}

int status_reserve(sspsd_decoder* d, size_t n_frames)
{
    if (n_frames > d->status_cap) {
        SSPSD_CUDA(cudaStreamSynchronize(d->stream));
        if (d->d_status) SSPSD_CUDA(cudaFree(d->d_status));
        d->d_status = nullptr;
        SSPSD_CUDA(cudaMalloc(&d->d_status, (n_frames + 64) * sizeof(unsigned int)));
        d->status_cap = n_frames + 64;
    }
    return SSPSD_OK;
}

// the trace buffers the decode kernels are about to overwrite may still be read by the cascades of the previous
// sspsd_cascade_process_frames call (other streams)
int wait_traces_consumed(sspsd_decoder* d)
{
    for (int t = 0; t < SSPSD_MAX_TRACES; ++t)
        if (d->consumed_pending[t]) {
            SSPSD_CUDA(cudaStreamWaitEvent(d->stream, d->ev_consumed[t], 0));
            d->consumed_pending[t] = false;
        }
    return SSPSD_OK;
}

// Queues scan + loss + payload decode of `n_frames` DEVICE-resident frames on d->stream and the read-back of the result
// into h_res[slot].  `fmt` = format byte of frame 0 (selects the payload kernel), status words at d_status + status_off,
// dst[t] device pointers (16-byte aligned if `dst_aligned`) with room for dst_cap items each.
int queue_decode(sspsd_decoder* d, const uint8_t* dfr, size_t n_frames, size_t status_off, size_t frame_len, size_t frame_stride,
                 const sspsd_loss* loss, float* const* dst, bool dst_aligned, size_t dst_cap, unsigned int fmt, int slot)
{
    using namespace sspsd;
    const size_t n_bytes = n_frames ? (n_frames - 1) * frame_stride + frame_len : 0;
    DecodeResult init{};
    init.first_bad = n_frames;
    d->h_res[slot] = init;
    SSPSD_CUDA(cudaMemcpyAsync(d->d_res + slot, d->h_res + slot, sizeof(init), cudaMemcpyHostToDevice, d->stream));
    DecodeParams p{};
    p.frames = dfr;
    p.n_frames = n_frames;
    p.frame_len = frame_len;
    p.frame_stride = frame_stride;
    p.status = d->d_status + status_off;
    p.res = d->d_res + slot;
    p.prev_seq = loss ? loss->seq : 0;
    p.has_prev = loss ? (loss->has_seq != 0) : 0;
    const int nt = 256;
    const unsigned int gf = (unsigned int)((n_frames + nt - 1) / nt);
    frame_scan_kernel<<<gf, nt, 0, d->stream>>>(p);
    loss_kernel<<<(unsigned int)((n_frames + 1 + nt - 1) / nt), nt, 0, d->stream>>>(p);
    SSPSD_CUDA(cudaGetLastError());
    if (dst && fmt >= 1 && fmt <= 4 && frame_len >= SSPSD_HEADER_SIZE) {
        TraceOut out{};
        for (int t = 0; t < SSPSD_MAX_TRACES; ++t) out.t[t] = dst[t];
        out.cap = dst_cap;
        const bool flat_ok = dst_aligned && (reinterpret_cast<uintptr_t>(dfr) % 8 == 0) && (frame_stride % 8 == 0) &&
                             ((frame_len - SSPSD_HEADER_SIZE) % 64 == 0);
        if (fmt == SSPSD_FORMAT_ADCDAC && flat_ok) {
            const unsigned long long n_words8 = n_bytes / 8;
            const unsigned long long per_cta = (unsigned long long)ADC_NT * ADC_ITERS;
            adcdac_flat_kernel<<<(unsigned int)((n_words8 + per_cta - 1) / per_cta), ADC_NT, 0, d->stream>>>(
                dfr, n_words8, frame_stride, frame_len, d->d_res + slot, out);
        } else {
            const unsigned int bb = batch_bytes(fmt);
            unsigned long long per = (frame_len - SSPSD_HEADER_SIZE) / bb;
            unsigned long long total = n_frames * per;
            if (total)
                decode_generic_kernel<<<(unsigned int)((total + nt - 1) / nt), nt, 0, d->stream>>>(
                    dfr, frame_stride, d->d_res + slot, out);
        }
        SSPSD_CUDA(cudaGetLastError());
    }
    SSPSD_CUDA(cudaMemcpyAsync(d->h_res + slot, d->d_res + slot, sizeof(DecodeResult), cudaMemcpyDeviceToHost, d->stream));
    return SSPSD_OK;
}

// Runs scan + loss + payload decode on d->stream.  dst[t] are device pointers (aligned if `aligned`).
// On return (stream synchronised) d->h_res[0] holds the batch result.  `sink` (if any) is shown the format byte
// before the decode is queued and may refuse it.
int decode_on_device(sspsd_decoder* d, const uint8_t* frames, size_t n_frames, size_t frame_len, size_t frame_stride,
                     int frames_mem, const sspsd_loss* loss, float* const* dst, bool dst_aligned, size_t dst_cap,
                     sspsd::FrameSink* sink = nullptr)
{
    const size_t n_bytes = n_frames ? (n_frames - 1) * frame_stride + frame_len : 0;
    const uint8_t* dfr = frames;
    int rc;
    if (frames_mem == SSPSD_MEM_HOST) {
        rc = frames_h2d(d, frames, n_bytes);
        if (rc) return rc;
        dfr = d->d_frames;
    }
    rc = wait_traces_consumed(d);
    if (rc) return rc;
    rc = status_reserve(d, n_frames);
    if (rc) return rc;
    // The format byte of frame 0 decides the kernel; peek at it on the host when the frames are host
    // memory, otherwise read it back (4 bytes) -- the call synchronises for the result anyway.
    uint8_t hdr[4] = {0, 0, 0, 0};
    if (dst) {
        if (frames_mem == SSPSD_MEM_HOST) {
            if (n_bytes >= 4) std::memcpy(hdr, frames, 4);
        } else if (n_bytes >= 4) {
            SSPSD_CUDA(cudaMemcpyAsync(hdr, dfr, 4, cudaMemcpyDeviceToHost, d->stream));
            SSPSD_CUDA(cudaStreamSynchronize(d->stream));
        }
    }
    if (sink) {
        rc = sink->accept(hdr[2]);
        if (rc) return rc;
    }
    rc = queue_decode(d, dfr, n_frames, 0, frame_len, frame_stride, loss, dst, dst_aligned, dst_cap, hdr[2], 0);
    if (rc) return rc;
    SSPSD_CUDA(cudaStreamSynchronize(d->stream));
    return SSPSD_OK;
}

int decode_wait(sspsd_decoder* d)
{
    SSPSD_CUDA(cudaStreamSynchronize(d->stream));
    return SSPSD_OK;
}

void apply_result(const sspsd::DecodeResult& r, size_t n_frames, sspsd_loss* loss, sspsd_decode_info* info,
                  unsigned int trace_div)
{
    if (loss && r.first_bad > 0) {
        loss->received += r.received;
        loss->dropped += r.dropped;
        loss->seq = r.last_seq_end;
        loss->has_seq = 1;
    }
    if (info) {
        std::memset(info, 0, sizeof(*info));
        info->frames_ok = r.first_bad;
        if (r.first_bad > 0) {
            info->format = r.format;
            info->n_traces = r.format == SSPSD_FORMAT_MPLL ? 3 : 4;
            info->samples_per_trace = (uint64_t)r.first_bad * r.batches * trace_div;
        }
    }
    (void)n_frames;
}

}  // namespace

extern "C" {

int32_t sspsd_decode_frames(sspsd_decoder* d, const uint8_t* frames, size_t n_frames, size_t frame_len,
                            size_t frame_stride, int32_t frames_mem, sspsd_loss* loss, float* const* traces,
                            size_t trace_cap, int32_t traces_mem, sspsd_decode_info* info)
{
    if (!d || (n_frames && !frames) || frame_stride < frame_len) {
        set_error("bad argument");
        return SSPSD_EINVAL;
    }
    if (info) std::memset(info, 0, sizeof(*info));
    if (n_frames == 0) return SSPSD_OK;
    if (frame_len < SSPSD_HEADER_SIZE) {
        set_error("frame shorter than its header");
        return SSPSD_ESHORT;
    }
    DevGuard g(d->device);
    if (!g.ok) return SSPSD_ECUDA;
    // worst-case items per trace: AdcDac yields 8 per 64 payload bytes, the others 1 per >= 24 bytes
    const size_t payload = frame_len - SSPSD_HEADER_SIZE;
    const size_t worst = n_frames * std::max<size_t>(payload / 64 * 8, payload / 24);
    float* dst[SSPSD_MAX_TRACES] = {nullptr, nullptr, nullptr, nullptr};
    bool aligned = true;
    const bool want = traces != nullptr;
    if (want) {
        if (traces_mem == SSPSD_MEM_DEVICE) {
            for (int t = 0; t < SSPSD_MAX_TRACES; ++t) {
                dst[t] = traces[t];
                if (reinterpret_cast<uintptr_t>(dst[t]) % 16) aligned = false;
            }
            if (trace_cap < worst) {
                set_error("trace capacity too small");
                return SSPSD_ESHORT;
            }
        } else {
            if (worst > d->traces_cap) {
                SSPSD_CUDA(cudaStreamSynchronize(d->stream));
                for (int t = 0; t < SSPSD_MAX_TRACES; ++t) {
                    if (d->d_traces[t]) SSPSD_CUDA(cudaFree(d->d_traces[t]));
                    d->d_traces[t] = nullptr;
                    SSPSD_CUDA(cudaMalloc(&d->d_traces[t], (worst + 64) * sizeof(float)));
                }
                d->traces_cap = worst;
            }
            for (int t = 0; t < SSPSD_MAX_TRACES; ++t) dst[t] = d->d_traces[t];
        }
    }
    int rc = decode_on_device(d, frames, n_frames, frame_len, frame_stride, frames_mem, loss, want ? dst : nullptr, aligned,
                              traces_mem == SSPSD_MEM_DEVICE ? trace_cap : d->traces_cap);
    if (rc) return rc;
    const sspsd::DecodeResult r = *d->h_res;
    const unsigned int div = r.format == SSPSD_FORMAT_ADCDAC ? 8 : 1;
    if (want && traces_mem != SSPSD_MEM_DEVICE && r.first_bad > 0 &&
        (size_t)r.first_bad * r.batches * div > trace_cap) {
        // capacity-in / length-out retry: report the needed length and leave `loss` untouched, so that the
        // retried call accounts for the batch exactly once (Loss stays bit-exact against loss.rs)
        if (info) {
            std::memset(info, 0, sizeof(*info));
            info->format = r.format;
            info->n_traces = r.format == SSPSD_FORMAT_MPLL ? 3 : 4;
            info->samples_per_trace = (uint64_t)r.first_bad * r.batches * div;
        }
        set_error("trace capacity too small");
        return SSPSD_ESHORT;
    }
    apply_result(r, n_frames, loss, info, div);
    if (want && traces_mem != SSPSD_MEM_DEVICE && r.first_bad > 0) {
        const size_t ns = (size_t)r.first_bad * r.batches * div;
        const int ntr = r.format == SSPSD_FORMAT_MPLL ? 3 : 4;
        for (int t = 0; t < ntr; ++t)
            if (traces[t])
                SSPSD_CUDA(cudaMemcpyAsync(traces[t], dst[t], ns * sizeof(float), cudaMemcpyDeviceToHost, d->stream));
        SSPSD_CUDA(cudaStreamSynchronize(d->stream));
    }
    if (r.first_bad < n_frames) {
        set_error("malformed frame");
        return (int32_t)r.status;
    }
    return SSPSD_OK;
}

}  // extern "C"

namespace sspsd {

int trace_consumed(sspsd_decoder* d, int t, cudaStream_t s)
{
    SSPSD_CUDA(cudaEventRecord(d->ev_consumed[t], s));
    d->consumed_pending[t] = true;
    return SSPSD_OK;
}

// The frame pipeline of sspsd_cascade_process_frames and sspsd_csd / sspsd_csm_process_frames: header scan, copies,
// decode, loss cross-check; what the decoded traces feed is the sink's business.
int process_frames(sspsd_decoder* d, FrameSink& sink, const uint8_t* frames, size_t n_frames, size_t frame_len,
                   size_t frame_stride, int frames_mem, sspsd_loss* loss, sspsd_decode_info* info)
{
    if (info) std::memset(info, 0, sizeof(*info));
    if (n_frames == 0) return SSPSD_OK;
    if (frame_len < SSPSD_HEADER_SIZE) {
        set_error("frame shorter than its header");
        return SSPSD_ESHORT;
    }
    int rc = sink.check_device(d->device);
    if (rc) return rc;
    DevGuard g(d->device);
    if (!g.ok) return SSPSD_ECUDA;
    if (frames_mem == SSPSD_MEM_HOST) {
        rc = sink.accept(frames[2]);
        if (rc) return rc;
    }
    const size_t payload = frame_len - SSPSD_HEADER_SIZE;
    const size_t worst = n_frames * std::max<size_t>(payload / 64 * 8, payload / 24);
    // (the previous batch's traces may still be read by the cascades' streams: decode_on_device makes the decode
    // kernels -- not the frames' H2D copy, which only touches the frame buffer -- wait for them, so the copy of
    // batch c + 1 overlaps the cascades of batch c)
    if (worst > d->traces_cap) {
        SSPSD_CUDA(cudaDeviceSynchronize());
        for (int t = 0; t < SSPSD_MAX_TRACES; ++t) {
            if (d->d_traces[t]) SSPSD_CUDA(cudaFree(d->d_traces[t]));
            d->d_traces[t] = nullptr;
            SSPSD_CUDA(cudaMalloc(&d->d_traces[t], (worst + 64) * sizeof(float)));
        }
        d->traces_cap = worst;
    }
    if (frames_mem == SSPSD_MEM_HOST) {
        // Host frames.  The batch is cut into up to MAX_SUB sub-chunks whose H2D copies are all queued up front on the
        // decoder's copy stream.  While sub-chunk k crosses PCIe the host validates its 8-byte headers (the same
        // frame_status() the scan kernel runs, one cache line per frame, prefetched ahead) and applies Loss::update to
        // them, so the number of good frames, the format, the batch count and the sequence state the NEXT sub-chunk starts
        // from are known without a device round trip; scan / loss / payload decode of sub-chunk k are queued behind its
        // copy and the sink's work behind its decode, so they run while sub-chunk k + 1 is still being copied.  The one
        // wait is at the end (the caller's buffer is borrowed for the call only, and the loss counters the device
        // computed are the ones returned: the host's serve as a cross-check).
        static const bool trace = getenv("SSPSD_FRAMES_TRACE") != nullptr;
        using clk = std::chrono::steady_clock;
        const auto t0 = clk::now();
        const size_t n_bytes = (n_frames - 1) * frame_stride + frame_len;
        rc = frames_reserve(d, n_bytes);
        if (rc) return rc;
        rc = status_reserve(d, n_frames);
        if (rc) return rc;
        // sub-chunks of >= 16384 frames: the host needs ~0.2 ms per sub-chunk (headers + launching the cascades)
        const size_t n_sub = std::max<size_t>(1, std::min<size_t>(sspsd_decoder::MAX_SUB, n_frames >> 14));
        const size_t per = (n_frames + n_sub - 1) / n_sub;
        for (size_t k = 0; k < n_sub; ++k) {
            const size_t f0 = k * per, f1 = std::min(n_frames, f0 + per);
            const size_t nb = (f1 - 1 - f0) * frame_stride + frame_len;
            SSPSD_CUDA(cudaMemcpyAsync(d->d_frames + f0 * frame_stride, frames + f0 * frame_stride, nb, cudaMemcpyHostToDevice,
                                       d->h2d_stream));
            SSPSD_CUDA(cudaEventRecord(d->ev_copied[k], d->h2d_stream));
        }
        const auto t1 = clk::now();
        rc = wait_traces_consumed(d);
        if (rc) return rc;
        const unsigned int fmt0 = frames[2];
        const unsigned int want_fmt = (fmt0 >= 1 && fmt0 <= 4) ? fmt0 : 0;
        const unsigned int batches = frames[3];
        const unsigned int div = fmt0 == SSPSD_FORMAT_ADCDAC ? 8 : 1;
        const uint32_t ntr = fmt0 == SSPSD_FORMAT_MPLL ? 3 : 4;
        sspsd_loss hl{};  // the host's own Loss::update over the headers
        if (loss) hl = *loss;
        size_t n_ok = 0, queued = 0;
        unsigned int bad_status = SSPSD_OK;
        size_t sub_n[sspsd_decoder::MAX_SUB] = {};
        double us_scan = 0, us_launch = 0;
        for (size_t k = 0; k < n_sub && bad_status == SSPSD_OK; ++k) {
            const auto ta = clk::now();
            const size_t f0 = k * per, f1 = std::min(n_frames, f0 + per);
            const sspsd_loss at_start = hl;
            size_t f = f0;
            for (; f < f1; ++f) {
                const uint8_t* fr = frames + f * frame_stride;
                if (f + 24 < n_frames) __builtin_prefetch(fr + 24 * frame_stride);
                bad_status = sspsd::frame_status(fr, frame_len, want_fmt);
                if (bad_status != SSPSD_OK) break;
                uint32_t seq;
                std::memcpy(&seq, fr + 4, 4);  // little endian, frame.rs:31
                sspsd_loss_update(&hl, seq, fr[3]);
            }
            n_ok = f;
            const size_t nk = f - f0;
            sub_n[k] = nk;
            const auto tb = clk::now();
            if (nk) {
                const size_t off = f0 * batches * div;  // items per trace before this sub-chunk
                float* dst[SSPSD_MAX_TRACES];
                for (int t = 0; t < SSPSD_MAX_TRACES; ++t) dst[t] = d->d_traces[t] + off;
                SSPSD_CUDA(cudaStreamWaitEvent(d->stream, d->ev_copied[k], 0));
                rc = queue_decode(d, d->d_frames + f0 * frame_stride, nk, f0, frame_len, frame_stride, loss ? &at_start : nullptr,
                                  dst, off % 4 == 0, d->traces_cap - off, fmt0, (int)k);
                if (rc) return rc;
                SSPSD_CUDA(cudaEventRecord(d->ev_decoded, d->stream));
                rc = sink.consume(d, dst, ntr, nk * batches * div, d->ev_decoded);
                if (rc) return rc;
                queued = k + 1;
            }
            if (trace) {
                us_scan += std::chrono::duration<double, std::micro>(tb - ta).count();
                us_launch += std::chrono::duration<double, std::micro>(clk::now() - tb).count();
            }
        }
        const auto t3 = clk::now();
        SSPSD_CUDA(cudaStreamSynchronize(d->h2d_stream));  // the caller's buffer is borrowed for the call only
        rc = decode_wait(d);
        if (rc) return rc;
        if (trace)
            fprintf(stderr, "[sspsd frames] n=%zu in %zu sub-chunks: enqueue h2d %.0f us, header scan %.0f us, launches %.0f us, wait %.0f us\n",
                    n_frames, n_sub, std::chrono::duration<double, std::micro>(t1 - t0).count(), us_scan, us_launch,
                    std::chrono::duration<double, std::micro>(clk::now() - t3).count());
        if (n_ok == 0) {
            if (info) std::memset(info, 0, sizeof(*info));
            set_error("malformed frame");
            return (int32_t)bad_status;
        }
        // the device's results, sub-chunk by sub-chunk, against the host's walk over the headers
        sspsd::DecodeResult sum{};
        for (size_t k = 0; k < queued; ++k) {
            const sspsd::DecodeResult& r = d->h_res[k];
            if (r.first_bad != sub_n[k] || r.format != fmt0 || r.batches != batches) {
                set_error("internal: device scan disagrees with the host pre-scan");
                return SSPSD_EINVAL;
            }
            sum.received += r.received;
            sum.dropped += r.dropped;
            sum.last_seq_end = r.last_seq_end;
        }
        sum.first_bad = n_ok;
        sum.format = fmt0;
        sum.batches = batches;
        if (loss && (loss->received + sum.received != hl.received || loss->dropped + sum.dropped != hl.dropped ||
                     sum.last_seq_end != hl.seq)) {
            set_error("internal: device loss counters disagree with the host's");
            return SSPSD_EINVAL;
        }
        apply_result(sum, n_ok, loss, info, div);
        if (n_ok < n_frames) {
            set_error("malformed frame");
            return (int32_t)bad_status;
        }
        return SSPSD_OK;
    }
    rc = decode_on_device(d, frames, n_frames, frame_len, frame_stride, frames_mem, loss, d->d_traces, true, d->traces_cap,
                          &sink);
    if (rc) return rc;
    const sspsd::DecodeResult r = *d->h_res;
    const unsigned int div = r.format == SSPSD_FORMAT_ADCDAC ? 8 : 1;
    apply_result(r, n_frames, loss, info, div);
    if (r.first_bad > 0) {
        const size_t ns = (size_t)r.first_bad * r.batches * div;
        const uint32_t ntr = r.format == SSPSD_FORMAT_MPLL ? 3 : 4;
        // decode_on_device synchronised d->stream, so the traces are complete for any stream
        rc = sink.consume(d, d->d_traces, ntr, ns, nullptr);
        if (rc) return rc;
    }
    if (r.first_bad < n_frames) {
        set_error("malformed frame");
        return (int32_t)r.status;
    }
    return SSPSD_OK;
}

}  // namespace sspsd

namespace {

// sspsd_cascade_process_frames: trace t -> cascades[t], each on its own stream
struct CascadeSink : sspsd::FrameSink {
    sspsd_cascade* const* c;
    uint32_t n;
    CascadeSink(sspsd_cascade* const* c_, uint32_t n_) : c(c_), n(n_) {}
    int check_device(int device) override
    {
        for (uint32_t t = 0; t < n; ++t)
            if (c[t] && c[t]->c.device() != device) {
                set_error("cascade and decoder live on different devices");
                return SSPSD_EINVAL;
            }
        return SSPSD_OK;
    }
    int accept(unsigned int) override { return SSPSD_OK; }  // cascades past the format's traces get nothing
    int consume(sspsd_decoder* d, float* const* tr, uint32_t n_traces, size_t ns, cudaEvent_t ready) override
    {
        for (uint32_t t = 0; t < n && t < n_traces; ++t) {
            if (!c[t]) continue;
            if (ready) SSPSD_CUDA(cudaStreamWaitEvent(c[t]->c.stream(), ready, 0));
            int rc = c[t]->c.process(tr[t], ns, SSPSD_MEM_DEVICE);
            if (rc) return rc;
            rc = sspsd::trace_consumed(d, (int)t, c[t]->c.stream());
            if (rc) return rc;
        }
        return SSPSD_OK;
    }
};

}  // namespace

extern "C" {

int32_t sspsd_cascade_process_frames(sspsd_decoder* d, sspsd_cascade* const* cascades, uint32_t n_cascades,
                                     const uint8_t* frames, size_t n_frames, size_t frame_len, size_t frame_stride,
                                     int32_t frames_mem, sspsd_loss* loss, sspsd_decode_info* info)
{
    if (!d || (n_frames && !frames) || frame_stride < frame_len || n_cascades > SSPSD_MAX_TRACES ||
        (n_cascades && !cascades)) {
        set_error("bad argument");
        return SSPSD_EINVAL;
    }
    CascadeSink sink(cascades, n_cascades);
    return sspsd::process_frames(d, sink, frames, n_frames, frame_len, frame_stride, frames_mem, loss, info);
}

void sspsd_loss_update(sspsd_loss* l, uint32_t seq, uint8_t batches)
{
    // Loss::update, loss.rs:11-26
    if (!l) return;
    l->received += batches;
    if (l->has_seq) l->dropped += (uint32_t)(seq - l->seq);
    l->seq = seq + batches;
    l->has_seq = 1;
}

float sspsd_loss_ratio(const sspsd_loss* l)
{
    // loss.rs:29-30
    if (!l) return 0.f;
    return (float)l->dropped / (float)(l->received + l->dropped);
}

int32_t sspsd_trace_plot(const sspsd_plot_opts* o, const float* psd, const float* frequencies, size_t n,
                         float* integral, double* xy, size_t* n_points)
{
    // Trace::plot + Trapezoidal, bin/psd.rs:96-157 (f32 running sums in the reference's order)
    sspsd_plot_opts d{1.0f, 1e-6f, 0.5f, 0};  // AcqOpts defaults, bin/psd.rs:37-38, 63-69
    if (o) d = *o;
    if (!n_points || (n && (!psd || !frequencies))) {
        set_error("null argument");
        return SSPSD_EINVAL;
    }
    size_t need = 0;
    for (size_t i = 0; i < n; ++i)
        if (std::fpclassify(frequencies[i]) == FP_NORMAL) ++need;
    if (xy && *n_points < need) {
        *n_points = need;
        set_error("output capacity too small");
        return SSPSD_ESHORT;
    }
    const float logfs = log10f(d.fs);
    float tx = 0.f, ty = 0.f, ti = 0.f;  // Trapezoidal::default()
    float pi = 0.f;
    size_t np = 0;
    for (size_t i = 0; i < n; ++i) {
        const float p = psd[i], f = frequencies[i];
        const float di = (p + ty) * 0.5f * (f - tx);  // Trapezoidal::push, bin/psd.rs:104-110
        tx = f;
        ty = p;
        ti += di;
        const float ff = d.fs * f;
        if (ff >= d.integral_start && ff <= d.integral_end) pi += di;  // bin/psd.rs:136-139
        if (std::fpclassify(f) == FP_NORMAL) {  // f.is_normal(), bin/psd.rs:140
            if (xy) {
                xy[2 * np] = (double)(log10f(f) + logfs);
                xy[2 * np + 1] = (double)(d.integrate ? sqrtf(ti) : 10.0f * (log10f(p) - logfs));
            }
            ++np;
        }
    }
    *n_points = np;
    if (integral) *integral = sqrtf(pi);
    return SSPSD_OK;
}

float sspsd_var_eval(const sspsd_var* v, const float* phase_psd, const float* frequencies, size_t n, float tau)
{
    // Var::eval, var.rs:26-45
    sspsd_var d{-2, 4, 3.40282347e38f, 0, 2};
    if (v) d = *v;
    const float pi = 3.14159265358979323846f;
    float accu = 0.f, a0 = 0.f, f0 = 0.f;
    for (size_t i = (size_t)d.dc_cut; i < n; ++i) {
        float sp = phase_psd[i], f = frequencies[i];
        if (!(f <= d.clip / tau)) break;
        float sy = sp * f * f;
        float pft = pi * (f * tau);
        float hahd = powi_f32(sinf(pft), d.sinx_exp) * powi_f32(pft, d.x_exp);
        float a = sy * hahd;
        accu = accu + (a + a0) * (f - f0);
        a0 = a;
        f0 = f;
    }
    return accu;
}

}  // extern "C"
