// sspsd_cascade.cuh -- host-side state machine of the device cascade (internal C++).
//
// Mirrors the streaming semantics of the reference's Psd<N>::process / PsdCascade<N>::process
// (src/psd.rs:196-269, 445-468) in closed form (SURVEY.md App. A.2): after L samples a stage has
// completed  craw = L < N ? 0 : 1 + (L-N)/hop  segments, has decimated its first
// D = craw ? N + (craw-1)*hop : 0  samples, and has handed  max(D/8 - R, 0)  samples to the next
// stage.  All integer bookkeeping lives on the host; the device only sees batches.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <string>
#include <vector>

#include "../../include/sspsd.h"
#include "sspsd_device.cuh"

namespace sspsd {

struct StageParams;
void set_error(const std::string& msg);
const char* last_error();
int hbf_info(int hbf, uint32_t* drain, uint32_t* halo);
bool cuda_ok(cudaError_t e, const char* what);

// Makes `dev` current for the scope and restores the caller's device afterwards: an entry point never leaves the
// calling thread's current device changed (a host application -- or torch -- keeps its own notion of it).
struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        ok = prev == dev || cuda_ok(cudaSetDevice(dev), "cudaSetDevice");
        if (prev == dev) prev = -1;  // nothing to restore
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};
#define SSPSD_CUDA(call)                     \
    do {                                     \
        if (!::sspsd::cuda_ok((call), #call)) return SSPSD_ECUDA; \
    } while (0)

struct WindowInfo {
    float power, nenbw;
    uint32_t overlap;
};

struct StageState {
    uint64_t L = 0;       // samples received so far
    uint64_t craw = 0;    // segments completed so far
    uint32_t count = 0;   // effective averaging count (Psd::count, psd.rs:128)
    uint32_t avg = 0xffffffffu;
    uint64_t emitted = 0; // samples handed to the next stage
    uint64_t valid_from = 0;  // time-chunk mode: first stream index not contaminated by the warm-up
    // device stream storage: carry[cur] holds [carry_start, L); the batch's new samples live in a
    // "fresh" buffer from split = floor4(L) on (its first L - split entries are copies of the carry tail)
    float* carry[2] = {nullptr, nullptr};
    int cur = 0;
    long long carry_start = 0;
    // stages >= 1: two fresh buffers written alternately by the previous stage's decimator
    float* fresh[2] = {nullptr, nullptr};
    int fb = 0;  // buffer the next incoming batch is written to
    size_t fresh_cap = 0;
    uint64_t pending_in = 0;  // samples the previous stage's decimator has written to fresh[fb] since this stage last ran
    cudaEvent_t ev_read[2] = {nullptr, nullptr};  // recorded when this stage has finished reading fresh[b]
    bool ev_read_pending[2] = {false, false};
    // stages on the deep stream run their PSD kernel on a third stream beside the decimation chain:
    cudaEvent_t ev_in = nullptr;                  // deep stream: this batch's input of the stage is complete
    cudaEvent_t ev_psd[2] = {nullptr, nullptr};   // PSD stream: the PSD kernel has finished reading fresh[b] + carry
};

// EWMA bookkeeping for a batch of S segments, psd.rs:215-225
struct EwmaPlan {
    int jb;         // first segment of the batch whose factor differs from 1 (>= S: pure boxcar)
    float g_first;  // factor applied at segment jb
    float g_s;      // factor applied at every later segment: avg / (avg + 1)
    float total;    // product of all factors (scales the running sum before the batch)
    uint32_t count_after;
};

class Cascade;
// Multi-channel mode (XCascade): a stage's PSD launch, EWMA pre-scale included, is handed to the hook instead, with
// the launch's segment range and EWMA plan; the cascade's own accumulator rows are then never touched.
struct StageHook {
    virtual int stage_psd(Cascade& c, size_t i, const StreamSrc& src, uint64_t k0, uint64_t nseg, const EwmaPlan& e) = 0;
};

class Cascade {
    friend class XCascade;

public:
    Cascade() = default;
    ~Cascade();
    int init(const sspsd_config& cfg, uint32_t max_stages);
    int clone_from(Cascade& o, const sspsd_config* cfg = nullptr);  // cfg: configuration of the copy (default o's)
    int reset();

    int process(const float* x, size_t n, int mem);
    int set_avg(sspsd_avg_opts a);
    int set_stage_avg(uint32_t avg);  // Psd::set_avg on stage 0 (single-stage API)
    int set_detrend(int d);
    int flush();
    int sync();
    int fence(cudaEvent_t ev);
    int psd(const sspsd_merge_opts& o, float* p, size_t* p_len, sspsd_break* b, size_t* b_len);
    int partials(sspsd_partials* out);
    void export_book(uint64_t* book) const;  // 4 * SSPSD_MAX_STAGES + 2 words
    static int merge_host(const sspsd_config& cfg, const uint64_t* book, const float* rows, size_t stride,
                          const sspsd_merge_opts& o, float* p, size_t* p_len, sspsd_break* b, size_t* b_len);
    int seek(uint64_t pos);
    int set_window(uint64_t own_lo, uint64_t own_hi, uint32_t n_local);
    int take_tail(uint64_t j_lo, uint64_t j_hi, float* out, size_t* len, uint64_t* first, int mem);
    int process_stage(uint32_t stage, const float* x, size_t n, int mem);
    int set_stream_state(uint32_t stage, uint64_t samples, uint64_t segments);
    void profile_enable(bool on) { prof_on_ = on; }
    int profile_read(sspsd_profile* out);
    int set_counts(const uint64_t* craw, uint32_t n);

    // single-stage helpers (PsdStage trait)
    int stage_spectrum(float* out, size_t* len, int mem);
    int stage_buf(float* out, size_t* len, int mem);
    int take_sink(float* y, size_t* y_len, int mem);  // decimated output of the last process()
    float stage_gain() const;
    uint32_t stage_count() const { return stages_.empty() ? 0 : stages_[0].count; }

    uint32_t n_stages() const { return (uint32_t)stages_.size(); }
    uint32_t n_fft() const { return n_; }
    float rbw() const { return 8.0f / ((float)n_ * 0.4f); }  // psd.rs:427-429
    cudaStream_t stream() const { return stream_; }
    int device() const { return cfg_.device; }
    // device-side entry used by the fused decode path: x is device memory valid in stream order
    int process_device(const float* x, size_t n);

private:
    int add_stage();
    void free_stages(bool keep_buffers);
    int run_stage(size_t i, const float* fresh, long long split, uint64_t n_new);
    int launch_psd(size_t i, const StreamSrc& src, uint64_t k0, uint64_t nseg, const EwmaPlan& e);
    int launch_decim(size_t i, const StreamSrc& src, uint64_t m0, uint64_t m1, float* out_fresh,
                     long long out_split, long long out_cap);
    int prepare_partials(size_t i, int rows, struct StageParams* p);
    int reduce_partials(size_t i, int rows, const struct StageParams& p);
    cudaStream_t stage_stream(size_t i) const { return (i < deep_from_ || !deep_stream_) ? stream_ : deep_stream_; }
    // stream of stage i's PSD kernel (and its EWMA pre-scale): beside the decimation chain for the deep stages
    cudaStream_t psd_stream(size_t i) const { return (i >= deep_from_ && psd_stream_) ? psd_stream_ : stage_stream(i); }
    int join_streams();  // make stream_ wait for everything queued on deep_stream_
    uint64_t defer_threshold(size_t j) const;  // stage j >= 1 runs once this many samples are pending (0: at once)
    int run_pending(size_t j);
    int flush_deferred();
    int ensure_fresh(StageState& st, size_t need, size_t reserve = 0);
    int ensure_in_buffers(size_t need);
    int process_host(const float* x, size_t n);
    int flush_staged();
    int feed_device_chunk(const float* x, size_t n);
    int feed_host_chunk(const float* xh, size_t n);
    static uint64_t host_chunk() { return 1ull << 23; }  // samples per pipelined H2D copy
    float gain_of(uint32_t count) const;
    uint32_t stage_avg(size_t i) const;
    uint64_t decimated(const StageState& st) const { return st.craw ? n_ + (st.craw - 1) * (uint64_t)hop_ : 0; }

    struct ProfRec {
        int cls;
        cudaEvent_t a, b;
        uint64_t units;
    };
    bool prof_on_ = false;
    std::vector<ProfRec> prof_;
    uint64_t launches_[SSPSD_PROF_NCLASS] = {0, 0, 0, 0, 0};
    void prof_begin(int cls, uint64_t units, cudaStream_t s);
    void prof_end(cudaStream_t s);

    // time-chunk mode
    bool windowed_ = false;
    uint64_t own_lo_ = 0, own_hi_ = ~0ull;
    uint32_t n_local_ = SSPSD_MAX_STAGES;
    float* d_tail_ = nullptr;
    size_t tail_cap_ = 0, tail_len_ = 0;
    uint64_t tail_first_ = 0;
    uint64_t seek_pos_ = 0;
    uint64_t next_valid_from(uint64_t valid) const;
    uint64_t own_offset(size_t i) const;  // stage-0 position of sample 0 of stage i

    StageHook* hook_ = nullptr;
    bool one_stream_ = false;  // set before init(): every stage and PSD launch on stream_ (no side streams)
    sspsd_config cfg_{};
    uint32_t n_ = 0, log2n_ = 0, hop_ = 0, max_stages_ = SSPSD_MAX_STAGES;
    WindowInfo win_{};
    int detrend_ = 0;
    sspsd_avg_opts avg_{0xffffffffu, 0xffffffffu};
    int hb_ = 0;       // history kept in the carry: max(overlap, decimator halo), multiple of 8
    int drain_ = 0;    // hbf_dec_response_length(3)
    int num_sms_ = 148;
    int tmax_ = 1, nt_ = 256;  // largest tile (segments per CTA) and CTA size of the stage kernel
    uint64_t defer_ = 1ull << 26;  // sspsd_config::deep_defer
    uint64_t defer_window_ = 0;    // threshold in force for the stage that has just received samples
    CarryJob cc_pending_{};    // carry copy of the stage being run, until a decimator launch (or the fallback kernel) takes it
    bool cc_valid_ = false;
    int k3_variant_ = 1;       // SSPSD_K3 at creation: 0 = tiled, 1 = persistent TMA (960 outputs/tile), 2 = (640)
    int k2_variant_ = 2;       // SSPSD_K2 at creation: 0 = radix-8 tiled, 1 = radix-16 tiled, 2 = TMA ring (N = 4096)
    bool single_stage_avg_set_ = false;
    uint32_t single_stage_avg_ = 0xffffffffu;
    cudaStream_t stream_ = nullptr;
    bool own_stream_ = false;
    cudaStream_t copy_stream_ = nullptr;
    cudaStream_t deep_stream_ = nullptr;  // stages >= 1 run here, overlapping the next batch's stage 0
    cudaStream_t psd_stream_ = nullptr;   // PSD kernels of stages >= deep_from_ (SSPSD_PSD_STREAM=0 disables)
    cudaEvent_t ev_stage0_ = nullptr, ev_deep_ = nullptr, ev_psd_join_ = nullptr;
    bool deep_dirty_ = false, psd_dirty_ = false;
    size_t deep_from_ = 1;  // first stage that runs on deep_stream_
    cudaEvent_t ev_copied_[2] = {nullptr, nullptr}, ev_free_[2] = {nullptr, nullptr};
    cudaEvent_t ev_stage_[2] = {nullptr, nullptr};
    int last_copy_ = -1;
    std::vector<StageState> stages_;
    std::vector<StageState> spare_;  // device buffers of stages released by reset(), reused by add_stage()
    // device tables + accumulators
    float* d_win_ = nullptr;
    float2* d_twM_ = nullptr;
    float2* d_twN_ = nullptr;
    float* d_acc_ = nullptr;  // [SSPSD_MAX_STAGES][acc_stride_]
    uint32_t acc_stride_ = 0;
    // host-input staging
    float* h_stage_[2] = {nullptr, nullptr};  // pinned, cfg_.host_stage floats each
    int stage_buf_ = 0;
    bool stage_pending_[2] = {false, false};
    size_t staged_ = 0;
    float* d_in_[2] = {nullptr, nullptr};
    size_t d_in_cap_ = 0;
    int in_buf_ = 0;
    float* h_acc_ = nullptr;  // pinned readback buffer
    // sink of the single-stage API
    float* d_part_[2] = {nullptr, nullptr};  // deterministic mode: partial rows (stage-0 stream, deep PSD stream)
    size_t part_cap_[2] = {0, 0};
    float* d_sink_ = nullptr;
    size_t sink_cap_ = 0, sink_len_ = 0;
};

// What a frame batch is decoded into (sspsd_api.cu's frame pipeline): the PsdCascades of
// sspsd_cascade_process_frames, or one CsdCascade / CsmCascade and its trace map.
struct FrameSink {
    // before anything is queued: handles on the decoder's device
    virtual int check_device(int device) = 0;
    // the batch's format byte (frame 0), once known and before anything is queued: can the sink take its traces
    virtual int accept(unsigned int fmt) = 0;
    // one decoded sub-chunk: trace t at tr[t] (t < n_traces), ns samples each, complete once `ready` has fired
    // (nullptr: already complete).  Every trace read is reported with trace_consumed() on the stream that reads it.
    virtual int consume(sspsd_decoder* d, float* const* tr, uint32_t n_traces, size_t ns, cudaEvent_t ready) = 0;
};
int process_frames(sspsd_decoder* d, FrameSink& sink, const uint8_t* frames, size_t n_frames, size_t frame_len,
                   size_t frame_stride, int frames_mem, sspsd_loss* loss, sspsd_decode_info* info);
// the decoder's trace buffer t is read by work queued on s so far: the next decode into it waits for that
int trace_consumed(sspsd_decoder* d, int t, cudaStream_t s);

}  // namespace sspsd

// the opaque handles of include/sspsd.h
struct sspsd_cascade {
    sspsd::Cascade c;
};
struct sspsd_stage {
    sspsd::Cascade c;
};
