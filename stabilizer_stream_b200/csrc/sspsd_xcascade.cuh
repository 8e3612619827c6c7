// sspsd_xcascade.cuh -- XCascade (the cross-spectral handles sspsd_csd / sspsd_csm and the two-sided kind) and
// ZoomCascade (sspsd_zoom), defined in sspsd_xcascade.cu; sspsd_group.cu drives them as the ranks of a time-chunked
// group of a cross kind.
#pragma once
#include "sspsd_cascade.cuh"

namespace sspsd {

struct XStageParams;

// One of the block kernels at one N, its rows and its shared-memory budget per CTA
struct BlockKernel {
    void (*fn)(XStageParams);
    size_t (*smem)(int T, int hop);  // bytes for tiles of T segments
    long long budget;
    int rows;
    const char* what;
};
struct BlockKernels {
    BlockKernel k[3];  // [DIAG]: csd_stage_kernel, [CROSS]: csm_cross_kernel, [IQ]: iq_stage_kernel
    int nt, groups;    // threads per CTA, segments in flight per CTA (all kernels)
};

class XCascade : public StageHook {
public:
    XCascade() = default;
    ~XCascade();
    int init(const sspsd_config& cfg, int k, bool two_sided = false);
    int clone_from(XCascade& o);
    int reset();
    int process(const float* const* x, size_t n, int mem);
    int set_avg(sspsd_avg_opts a);
    int set_detrend(int d);
    int flush();
    int sync();
    int read(const sspsd_merge_opts& o, float* pxx, float* pyy, float* pxy, size_t* p_len, sspsd_break* b,
             size_t* b_len);
    int read_matrix(const sspsd_merge_opts& o, float* s, size_t* p_len, sspsd_break* b, size_t* b_len);
    int read_two_sided(const sspsd_merge_opts& o, float* p_pos, float* p_neg, size_t* p_len, sspsd_break* b,
                       size_t* b_len);
    int num_stages(uint32_t* n);
    int channels() const { return k_; }
    int device() const { return cfg_.device; }
    float rbw() const { return ch_[0].rbw(); }
    cudaStream_t stream() const { return stream_; }
    int stage_psd(Cascade& c, size_t i, const StreamSrc& src, uint64_t k0, uint64_t nseg, const EwmaPlan& e) override;
    // accumulator rows per stage: the block of stage i is rows [i * block_rows(), (i + 1) * block_rows())
    size_t block_rows() const;

    // Time-chunk mode (sspsd_cascade_seek & co. of include/sspsd.h) on all channels in lockstep
    int seek(uint64_t pos);
    int set_window(uint64_t own_lo, uint64_t own_hi, uint32_t n_local);
    // out[c]: channel c's slice of the stage-n_local input stream (device memory); len: capacity in, length out
    int take_tail(uint64_t j_lo, uint64_t j_hi, float* const* out, size_t* len, uint64_t* first);
    // x[c]: the next n samples of channel c's stage-`stage` stream, device memory
    int process_stage(uint32_t stage, const float* const* x, size_t n);
    int set_stream_state(uint32_t stage, uint64_t samples, uint64_t segments);
    // acc: the accumulator blocks, acc_stride: floats per ROW (block_rows() rows per stage); counts of channel 0
    int partials(sspsd_partials* out);

private:
    int setup(const sspsd_config& cfg, int k, bool two_sided);
    sspsd_config channel_cfg() const;
    int feed_chunk(const float* const* x, size_t n, bool device);
    int flush_staged();
    int flush_all();
    size_t acc_floats() const { return (size_t)SSPSD_MAX_STAGES * block_rows() * stride_; }
    int ensure_part(float** part, size_t* cap, size_t need);
    int launch_block(int kind, XStageParams p, uint64_t nseg, float* acc, float** part, size_t* part_cap);
    int read_rows(const sspsd_merge_opts& o, bool outs, size_t* p_len, sspsd_break* b, size_t* b_len,
                  uint64_t (&book)[4 * SSPSD_MAX_STAGES + 2], size_t* pl, size_t* ns);

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
    Cascade ch_[4];  // channel 0 launches the block kernels; 1 .. k_-1 leave their sources
    int k_ = 2;
    bool two_sided_ = false;  // K = 2: iq_stage_kernel's rows P+, P- instead of the CSD's four
    sspsd_config cfg_{};
    cudaStream_t stream_ = nullptr;
    uint32_t n_ = 0, log2n_ = 0;
    int num_sms_ = 148;
    BlockKernels kern_{};
    int tmax_[3] = {1, 1, 1};  // largest tile of each block kernel
    uint32_t stride_ = 0;  // floats per row; a stage's block is block_rows() rows
    float* d_win_ = nullptr;
    float2* d_tw_ = nullptr;
    float* d_acc_ = nullptr;  // [SSPSD_MAX_STAGES][block_rows()][stride_]
    float* h_acc_ = nullptr;
    float* d_part_ = nullptr;   // deterministic mode: csd_stage_kernel's partial blocks
    size_t part_cap_ = 0;
    float* d_xpart_ = nullptr;  // and csm_cross_kernel's (another row layout: its padding must stay zero too)
    size_t xpart_cap_ = 0;
    struct Source {
        StreamSrc src;
        uint64_t k0, nseg;
        bool valid;
    } srcs_[4][SSPSD_MAX_STAGES] = {};
};

// ZoomCascade: the two-sided XCascade over z = i + i q, fed either I/Q streams as they are (SSPSD_ZOOM_IQ) or one real
// stream mixed down by the carrier ftw / 2^32 (SSPSD_ZOOM_HETERODYNE, DESIGN.md 3c).  The mixer runs on the
// XCascade's one stream into buffers owned here, which the XCascade then reads in place (SSPSD_MEM_DEVICE): stream
// order alone makes their reuse by the next mixer launch safe.  Host input is collected in pinned staging buffers,
// as Cascade::process_host collects small calls, and goes to the device by cudaMemcpyAsync on the same stream.
class ZoomCascade {
public:
    ~ZoomCascade();
    int init(const sspsd_config& cfg, int mode, uint32_t ftw);
    int clone_from(ZoomCascade& o);
    int reset();
    // time-chunk mode: the cascade's seek, and the mixer starts at the absolute sample index pos
    int seek(uint64_t pos);
    int process_iq(const float* i, const float* q, size_t n, int mem);
    int process(const float* x, size_t n, int mem);
    int process_device_mixed(const float* x, size_t n);  // x: device memory valid in stream order
    int set_avg(sspsd_avg_opts a);
    int set_detrend(int d);
    int flush();
    int sync();
    int read(const sspsd_merge_opts& o, float* p_pos, float* p_neg, size_t* p_len, sspsd_break* b, size_t* b_len);
    int num_stages(uint32_t* n);
    int mode() const { return mode_; }
    uint32_t ftw() const { return ftw_; }
    XCascade& x() { return x_; }
    const XCascade& x() const { return x_; }

private:
    int ensure_mix();
    int flush_host();
    int mix_and_feed(const float* d_x, size_t n);

    XCascade x_;
    int mode_ = SSPSD_ZOOM_IQ;
    uint32_t ftw_ = 0;
    uint64_t pos_ = 0;  // absolute index of the next sample mixed: phi_n = (n ftw) mod 2^32
    size_t mix_cap_ = 0;  // samples per mixer launch (a multiple of 4) and of d_i_, d_q_
    float* d_i_ = nullptr;
    float* d_q_ = nullptr;
    size_t stage_cap_ = 0;  // host staging, cfg.host_stage rounded to a multiple of 4: pinned h_stage_[2], d_x_
    float* h_stage_[2] = {nullptr, nullptr};
    float* d_x_ = nullptr;
    cudaEvent_t ev_stage_[2] = {nullptr, nullptr};  // the H2D copy of h_stage_[b] has completed
    bool stage_pending_[2] = {false, false};
    int stage_buf_ = 0;
    size_t staged_ = 0;
};

}  // namespace sspsd

struct sspsd_csd {
    sspsd::XCascade c;
};

struct sspsd_csm {
    sspsd::XCascade c;
};

struct sspsd_zoom {
    sspsd::ZoomCascade z;
};
