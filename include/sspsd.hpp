// sspsd.hpp -- header-only C++17 mirror of the reference's Rust API on top of the C ABI (sspsd.h).
//
// Same names, argument meaning and error behaviour as quartiq/stabilizer-stream:
//   PsdCascade<N>  src/psd.rs:399-544      Psd<N> / PsdStage  src/psd.rs:119-288
//   Break          src/psd.rs:290-337      MergeOpts / AvgOpts src/psd.rs:339-376
//   Detrend        src/psd.rs:59-72        Window              src/psd.rs:12-56
//   Loss           src/loss.rs:4-38        FrameDecoder        src/de/frame.rs:49-60 + src/de/data.rs
//   Var            src/var.rs:4-45
// The reference's PSD API is infallible (it panics on programming errors such as Detrend::Linear,
// src/psd.rs:110); here such conditions throw sspsd::Error.  Decode errors map de::Error
// (src/de/mod.rs:19-27) onto DecodeError::status.
#pragma once
#include <cstddef>
#include <cstdint>
#include <limits>
#include <stdexcept>
#include <string>
#include <utility>
#include <array>
#include <vector>

#include "sspsd.h"

namespace sspsd {

struct Error : std::runtime_error {
    int32_t status;
    Error(int32_t st, const char* msg) : std::runtime_error(std::string(msg ? msg : "")), status(st) {}
};

inline void check(int32_t st)
{
    if (st != SSPSD_OK) throw Error(st, sspsd_last_error());
}

/// enum Detrend, src/psd.rs:59-72
enum class Detrend : int32_t { None = 0, Midpoint = 1, Span = 2, Mean = 3, Linear = 4 };
/// Window::rectangular / Window::hann, src/psd.rs:24-55
enum class Window : int32_t { Rectangular = 0, Hann = 1 };
enum class Mem : int32_t { Host = SSPSD_MEM_HOST, Device = SSPSD_MEM_DEVICE };

/// src/psd.rs:360-376
struct AvgOpts {
    uint32_t limit = std::numeric_limits<uint32_t>::max();
    uint32_t count = std::numeric_limits<uint32_t>::max();
};

/// src/psd.rs:339-358
struct MergeOpts {
    bool keep_overlap = false;
    uint32_t min_count = 1;
    bool keep_transition_band = false;
};

/// src/psd.rs:290-337
struct Break {
    size_t start;
    bool include;
    uint32_t count;
    uint32_t avg;
    std::pair<size_t, size_t> bins;  // Range<usize>: [first, second)
    size_t fft_size;
    size_t decimation;
    size_t pending;
    size_t processed;

    size_t effective_fft_size() const { return fft_size * decimation; }
    float rbw() const { return 1.0f / (float)effective_fft_size(); }

    /// Break::frequencies, src/psd.rs:315-327
    static std::vector<float> frequencies(const std::vector<Break>& b)
    {
        std::vector<float> f;
        for (const auto& bi : b) {
            if (!bi.include) continue;
            float r = bi.rbw();
            for (size_t k = bi.bins.first; k < bi.bins.second; ++k) f.push_back((float)k * r);
        }
        return f;
    }
};

/// PsdCascade<N>, src/psd.rs:399-544.  Default construction == PsdCascade::<N>::default().
template <size_t N>
class PsdCascade {
public:
    explicit PsdCascade(int device = 0, void* stream = nullptr, int32_t hbf = SSPSD_HBF_140)
    {
        sspsd_config cfg;
        check(sspsd_config_default((uint32_t)N, &cfg));
        cfg.device = device;
        cfg.stream = stream;
        cfg.hbf = hbf;
        check(sspsd_cascade_create(&cfg, &h_));
    }
    PsdCascade(const PsdCascade& o) { check(sspsd_cascade_clone(o.h_, &h_)); }  // #[derive(Clone)]
    PsdCascade& operator=(const PsdCascade& o)
    {
        if (this != &o) {
            sspsd_cascade* n = nullptr;
            check(sspsd_cascade_clone(o.h_, &n));
            sspsd_cascade_destroy(h_);
            h_ = n;
        }
        return *this;
    }
    PsdCascade(PsdCascade&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    ~PsdCascade() { sspsd_cascade_destroy(h_); }

    float rbw() const
    {
        float r;
        check(sspsd_cascade_rbw(h_, &r));
        return r;
    }
    void set_avg(AvgOpts a) { check(sspsd_cascade_set_avg(h_, sspsd_avg_opts{a.limit, a.count})); }
    void set_detrend(Detrend d) { check(sspsd_cascade_set_detrend(h_, (int32_t)d)); }
    /// process(&mut self, x: &[f32])
    void process(const float* x, size_t n, Mem mem = Mem::Host) { check(sspsd_cascade_process_f32(h_, x, n, (int32_t)mem)); }
    void process(const std::vector<float>& x) { process(x.data(), x.size()); }
    /// psd(&self, &MergeOpts) -> (Vec<f32>, Vec<Break>)
    std::pair<std::vector<float>, std::vector<Break>> psd(const MergeOpts& o = MergeOpts()) const
    {
        sspsd_merge_opts mo{o.keep_overlap, o.min_count, o.keep_transition_band};
        std::vector<float> p(SSPSD_MAX_STAGES * (N / 2 + 1));
        sspsd_break cb[SSPSD_MAX_STAGES];
        size_t pl = p.size(), bl = SSPSD_MAX_STAGES;
        check(sspsd_cascade_psd(h_, &mo, p.data(), &pl, cb, &bl));
        p.resize(pl);
        std::vector<Break> b;
        for (size_t i = 0; i < bl; ++i)
            b.push_back(Break{(size_t)cb[i].start, cb[i].include != 0, cb[i].count, cb[i].avg,
                              {(size_t)cb[i].bins_start, (size_t)cb[i].bins_end}, (size_t)cb[i].fft_size,
                              (size_t)cb[i].decimation, (size_t)cb[i].pending, (size_t)cb[i].processed});
        return {std::move(p), std::move(b)};
    }
    void reset() { check(sspsd_cascade_reset(h_)); }
    void sync() { check(sspsd_cascade_sync(h_)); }
    sspsd_cascade* handle() const { return h_; }

private:
    sspsd_cascade* h_ = nullptr;
};

/// Cascaded cross-spectral density of two streams (sspsd_csd_* in sspsd.h), N = 64 .. 4096.  pxx and pyy are what a
/// PsdCascade<N> fed x or y alone returns; pxy accumulates conj(X) Y, so pxy / pxx is the transfer function x -> y.
template <size_t N>
class CsdCascade {
public:
    struct Spectra {
        std::vector<float> pxx, pyy;
        std::vector<std::pair<float, float>> pxy;  // (re, im)
        std::vector<Break> breaks;
    };
    explicit CsdCascade(int device = 0, void* stream = nullptr, int32_t hbf = SSPSD_HBF_140, Window w = Window::Hann)
    {
        sspsd_config cfg;
        check(sspsd_config_default((uint32_t)N, &cfg));
        cfg.device = device;
        cfg.stream = stream;
        cfg.hbf = hbf;
        cfg.window = (int32_t)w;
        check(sspsd_csd_create(&cfg, &h_));
    }
    CsdCascade(const CsdCascade& o) { check(sspsd_csd_clone(o.h_, &h_)); }
    CsdCascade& operator=(const CsdCascade& o)
    {
        if (this != &o) {
            sspsd_csd* n = nullptr;
            check(sspsd_csd_clone(o.h_, &n));
            sspsd_csd_destroy(h_);
            h_ = n;
        }
        return *this;
    }
    CsdCascade(CsdCascade&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    ~CsdCascade() { sspsd_csd_destroy(h_); }

    float rbw() const
    {
        float r;
        check(sspsd_csd_rbw(h_, &r));
        return r;
    }
    void set_avg(AvgOpts a) { check(sspsd_csd_set_avg(h_, sspsd_avg_opts{a.limit, a.count})); }
    void set_detrend(Detrend d) { check(sspsd_csd_set_detrend(h_, (int32_t)d)); }
    void process(const float* x, const float* y, size_t n, Mem mem = Mem::Host)
    {
        check(sspsd_csd_process_f32(h_, x, y, n, (int32_t)mem));
    }
    void process(const std::vector<float>& x, const std::vector<float>& y)
    {
        if (x.size() != y.size()) throw Error(SSPSD_EINVAL, "x and y must have the same length");
        process(x.data(), y.data(), x.size());
    }
    Spectra csd(const MergeOpts& o = MergeOpts()) const
    {
        sspsd_merge_opts mo{o.keep_overlap, o.min_count, o.keep_transition_band};
        Spectra s;
        const size_t cap = SSPSD_MAX_STAGES * (N / 2 + 1);
        s.pxx.resize(cap);
        s.pyy.resize(cap);
        std::vector<float> xy(2 * cap);
        sspsd_break cb[SSPSD_MAX_STAGES];
        size_t pl = cap, bl = SSPSD_MAX_STAGES;
        check(sspsd_csd_read(h_, &mo, s.pxx.data(), s.pyy.data(), xy.data(), &pl, cb, &bl));
        s.pxx.resize(pl);
        s.pyy.resize(pl);
        for (size_t k = 0; k < pl; ++k) s.pxy.emplace_back(xy[2 * k], xy[2 * k + 1]);
        for (size_t i = 0; i < bl; ++i)
            s.breaks.push_back(Break{(size_t)cb[i].start, cb[i].include != 0, cb[i].count, cb[i].avg,
                                     {(size_t)cb[i].bins_start, (size_t)cb[i].bins_end}, (size_t)cb[i].fft_size,
                                     (size_t)cb[i].decimation, (size_t)cb[i].pending, (size_t)cb[i].processed});
        return s;
    }
    uint32_t num_stages() const
    {
        uint32_t n;
        check(sspsd_csd_num_stages(h_, &n));
        return n;
    }
    void reset() { check(sspsd_csd_reset(h_)); }
    void flush() { check(sspsd_csd_flush(h_)); }
    void sync() { check(sspsd_csd_sync(h_)); }
    sspsd_csd* handle() const { return h_; }

private:
    sspsd_csd* h_ = nullptr;
};

/// Two-sided cascaded spectrum of a complex stream (sspsd_zoom_* in sspsd.h), N = 64 .. 4096: I/Q streams as they are
/// (ZoomCascade::iq()), or one real stream mixed down by the carrier ftw / 2^32 (ZoomCascade::heterodyne(ftw)).
/// p_pos[j] is the density at f0 + f_j and p_neg[j] at f0 - f_j, f_j of Break::frequencies.
template <size_t N>
class ZoomCascade {
public:
    struct Spectra {
        std::vector<float> p_pos, p_neg;
        std::vector<Break> breaks;
    };
    static ZoomCascade iq(int device = 0, void* stream = nullptr, int32_t hbf = SSPSD_HBF_140, Window w = Window::Hann)
    {
        return ZoomCascade(SSPSD_ZOOM_IQ, 0, device, stream, hbf, w);
    }
    static ZoomCascade heterodyne(uint32_t ftw, int device = 0, void* stream = nullptr, int32_t hbf = SSPSD_HBF_140,
                                  Window w = Window::Hann)
    {
        return ZoomCascade(SSPSD_ZOOM_HETERODYNE, ftw, device, stream, hbf, w);
    }
    ZoomCascade(int32_t mode, uint32_t ftw, int device = 0, void* stream = nullptr, int32_t hbf = SSPSD_HBF_140,
                Window w = Window::Hann)
    {
        sspsd_config cfg;
        check(sspsd_config_default((uint32_t)N, &cfg));
        cfg.device = device;
        cfg.stream = stream;
        cfg.hbf = hbf;
        cfg.window = (int32_t)w;
        check(sspsd_zoom_create(&cfg, mode, ftw, &h_));
    }
    ZoomCascade(const ZoomCascade& o) { check(sspsd_zoom_clone(o.h_, &h_)); }
    ZoomCascade& operator=(const ZoomCascade& o)
    {
        if (this != &o) {
            sspsd_zoom* n = nullptr;
            check(sspsd_zoom_clone(o.h_, &n));
            sspsd_zoom_destroy(h_);
            h_ = n;
        }
        return *this;
    }
    ZoomCascade(ZoomCascade&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    ~ZoomCascade() { sspsd_zoom_destroy(h_); }

    float rbw() const
    {
        float r;
        check(sspsd_zoom_rbw(h_, &r));
        return r;
    }
    /// (mode, ftw)
    std::pair<int32_t, uint32_t> carrier() const
    {
        int32_t m;
        uint32_t f;
        check(sspsd_zoom_carrier(h_, &m, &f));
        return {m, f};
    }
    void set_avg(AvgOpts a) { check(sspsd_zoom_set_avg(h_, sspsd_avg_opts{a.limit, a.count})); }
    void set_detrend(Detrend d) { check(sspsd_zoom_set_detrend(h_, (int32_t)d)); }
    /// I/Q mode
    void process(const float* i, const float* q, size_t n, Mem mem = Mem::Host)
    {
        check(sspsd_zoom_process_iq_f32(h_, i, q, n, (int32_t)mem));
    }
    void process(const std::vector<float>& i, const std::vector<float>& q)
    {
        if (i.size() != q.size()) throw Error(SSPSD_EINVAL, "i and q must have the same length");
        process(i.data(), q.data(), i.size());
    }
    /// heterodyne mode
    void process(const float* x, size_t n, Mem mem = Mem::Host) { check(sspsd_zoom_process_f32(h_, x, n, (int32_t)mem)); }
    void process(const std::vector<float>& x) { process(x.data(), x.size()); }
    Spectra spectrum(const MergeOpts& o = MergeOpts()) const
    {
        sspsd_merge_opts mo{o.keep_overlap, o.min_count, o.keep_transition_band};
        Spectra s;
        const size_t cap = SSPSD_MAX_STAGES * (N / 2 + 1);
        s.p_pos.resize(cap);
        s.p_neg.resize(cap);
        sspsd_break cb[SSPSD_MAX_STAGES];
        size_t pl = cap, bl = SSPSD_MAX_STAGES;
        check(sspsd_zoom_read(h_, &mo, s.p_pos.data(), s.p_neg.data(), &pl, cb, &bl));
        s.p_pos.resize(pl);
        s.p_neg.resize(pl);
        for (size_t i = 0; i < bl; ++i)
            s.breaks.push_back(Break{(size_t)cb[i].start, cb[i].include != 0, cb[i].count, cb[i].avg,
                                     {(size_t)cb[i].bins_start, (size_t)cb[i].bins_end}, (size_t)cb[i].fft_size,
                                     (size_t)cb[i].decimation, (size_t)cb[i].pending, (size_t)cb[i].processed});
        return s;
    }
    uint32_t num_stages() const
    {
        uint32_t n;
        check(sspsd_zoom_num_stages(h_, &n));
        return n;
    }
    /// traces the frame entry points read: two in I/Q mode, one in heterodyne mode
    int traces() const { return carrier().first == SSPSD_ZOOM_IQ ? 2 : 1; }
    void reset() { check(sspsd_zoom_reset(h_)); }
    void flush() { check(sspsd_zoom_flush(h_)); }
    void sync() { check(sspsd_zoom_sync(h_)); }
    sspsd_zoom* handle() const { return h_; }

private:
    sspsd_zoom* h_ = nullptr;
};

/// Cascaded cross-spectral matrix of K = 2 .. 4 streams (sspsd_csm_* in sspsd.h), N = 64 .. 4096.  s(i, j) accumulates
/// conj(X_i) X_j: s(0, 1) is CsdCascade's pxy of (x0, x1), and s(i, i) what a PsdCascade<N> fed x_i alone returns.
template <size_t N>
class CsmCascade {
public:
    struct Matrix {
        size_t k = 0, bins = 0;
        std::vector<std::pair<float, float>> s;  // (re, im) of S_ij[b] at (i k + j) bins + b
        std::vector<Break> breaks;
        std::pair<float, float> operator()(size_t i, size_t j, size_t b) const { return s[(i * k + j) * bins + b]; }
    };
    explicit CsmCascade(int k, int device = 0, void* stream = nullptr, int32_t hbf = SSPSD_HBF_140,
                        Window w = Window::Hann)
    {
        sspsd_config cfg;
        check(sspsd_config_default((uint32_t)N, &cfg));
        cfg.device = device;
        cfg.stream = stream;
        cfg.hbf = hbf;
        cfg.window = (int32_t)w;
        check(sspsd_csm_create(&cfg, k, &h_));
        k_ = k;
    }
    CsmCascade(const CsmCascade& o) : k_(o.k_) { check(sspsd_csm_clone(o.h_, &h_)); }
    CsmCascade& operator=(const CsmCascade& o)
    {
        if (this != &o) {
            sspsd_csm* n = nullptr;
            check(sspsd_csm_clone(o.h_, &n));
            sspsd_csm_destroy(h_);
            h_ = n;
            k_ = o.k_;
        }
        return *this;
    }
    CsmCascade(CsmCascade&& o) noexcept : h_(o.h_), k_(o.k_) { o.h_ = nullptr; }
    ~CsmCascade() { sspsd_csm_destroy(h_); }

    int channels() const { return k_; }
    float rbw() const
    {
        float r;
        check(sspsd_csm_rbw(h_, &r));
        return r;
    }
    void set_avg(AvgOpts a) { check(sspsd_csm_set_avg(h_, sspsd_avg_opts{a.limit, a.count})); }
    void set_detrend(Detrend d) { check(sspsd_csm_set_detrend(h_, (int32_t)d)); }
    /// x: channels() pointers to n samples each
    void process(const float* const* x, size_t n, Mem mem = Mem::Host)
    {
        check(sspsd_csm_process_f32(h_, x, n, (int32_t)mem));
    }
    void process(const std::vector<std::vector<float>>& x)
    {
        if ((int)x.size() != k_) throw Error(SSPSD_EINVAL, "one vector per channel");
        const float* p[4];
        for (int c = 0; c < k_; ++c) {
            if (x[c].size() != x[0].size()) throw Error(SSPSD_EINVAL, "channels must have the same length");
            p[c] = x[c].data();
        }
        process(p, x[0].size());
    }
    Matrix csm(const MergeOpts& o = MergeOpts()) const
    {
        sspsd_merge_opts mo{o.keep_overlap, o.min_count, o.keep_transition_band};
        const size_t cap = SSPSD_MAX_STAGES * (N / 2 + 1);
        std::vector<float> s(2 * (size_t)k_ * k_ * cap);
        sspsd_break cb[SSPSD_MAX_STAGES];
        size_t pl = cap, bl = SSPSD_MAX_STAGES;
        check(sspsd_csm_read(h_, &mo, s.data(), &pl, cb, &bl));
        Matrix m;
        m.k = (size_t)k_;
        m.bins = pl;
        for (size_t r = 0; r < m.k * m.k * pl; ++r) m.s.emplace_back(s[2 * r], s[2 * r + 1]);
        for (size_t i = 0; i < bl; ++i)
            m.breaks.push_back(Break{(size_t)cb[i].start, cb[i].include != 0, cb[i].count, cb[i].avg,
                                     {(size_t)cb[i].bins_start, (size_t)cb[i].bins_end}, (size_t)cb[i].fft_size,
                                     (size_t)cb[i].decimation, (size_t)cb[i].pending, (size_t)cb[i].processed});
        return m;
    }
    uint32_t num_stages() const
    {
        uint32_t n;
        check(sspsd_csm_num_stages(h_, &n));
        return n;
    }
    void reset() { check(sspsd_csm_reset(h_)); }
    void flush() { check(sspsd_csm_flush(h_)); }
    void sync() { check(sspsd_csm_sync(h_)); }
    sspsd_csm* handle() const { return h_; }

private:
    sspsd_csm* h_ = nullptr;
    int k_ = 0;
};

/// Psd<N> + trait PsdStage, src/psd.rs:119-288
template <size_t N>
class Psd {
public:
    explicit Psd(Window w = Window::Hann, int device = 0, void* stream = nullptr)
    {
        sspsd_config cfg;
        check(sspsd_config_default((uint32_t)N, &cfg));
        cfg.window = (int32_t)w;
        cfg.device = device;
        cfg.stream = stream;
        check(sspsd_stage_create(&cfg, &h_));
    }
    Psd(const Psd&) = delete;
    Psd& operator=(const Psd&) = delete;
    ~Psd() { sspsd_stage_destroy(h_); }
    void set_avg(uint32_t avg) { check(sspsd_stage_set_avg(h_, avg)); }
    void set_detrend(Detrend d) { check(sspsd_stage_set_detrend(h_, (int32_t)d)); }
    /// process(x, y) -> number of items written to y
    size_t process(const float* x, size_t n, float* y, size_t y_cap, Mem xm = Mem::Host, Mem ym = Mem::Host)
    {
        size_t yl = y_cap;
        check(sspsd_stage_process_f32(h_, x, n, (int32_t)xm, y, &yl, (int32_t)ym));
        return yl;
    }
    std::vector<float> spectrum()
    {
        std::vector<float> s(N / 2 + 1);
        size_t l = s.size();
        check(sspsd_stage_spectrum(h_, s.data(), &l, SSPSD_MEM_HOST));
        return s;
    }
    uint32_t count()
    {
        uint32_t c;
        check(sspsd_stage_count(h_, &c));
        return c;
    }
    float gain()
    {
        float g;
        check(sspsd_stage_gain(h_, &g));
        return g;
    }
    std::vector<float> buf()
    {
        std::vector<float> b(N);
        size_t l = b.size();
        check(sspsd_stage_buf(h_, b.data(), &l, SSPSD_MEM_HOST));
        b.resize(l);
        return b;
    }

private:
    sspsd_stage* h_ = nullptr;
};

/// struct Loss, src/loss.rs:4-38
struct Loss {
    sspsd_loss c{0, 0, 0, 0};
    void update(uint32_t seq, uint8_t batches) { sspsd_loss_update(&c, seq, batches); }
    float ratio() const { return sspsd_loss_ratio(&c); }
};

struct DecodeError : std::runtime_error {
    int32_t status;       // SSPSD_EHEADER / EFORMAT / ESIZE (de::Error) or EBATCHES / ESHORT (reference panics)
    uint64_t frames_ok;   // frames decoded (and accounted in Loss) before the malformed one
    DecodeError(int32_t st, uint64_t ok) : std::runtime_error("malformed frame"), status(st), frames_ok(ok) {}
};

/// Batched Frame::from_bytes + Loss::update + Payload::traces
class FrameDecoder {
public:
    explicit FrameDecoder(int device = 0, void* stream = nullptr) { check(sspsd_decoder_create(device, stream, &d_)); }
    FrameDecoder(const FrameDecoder&) = delete;
    ~FrameDecoder() { sspsd_decoder_destroy(d_); }
    /// n_frames equally sized frames -> traces[t] (host vectors, resized); returns the batch info
    sspsd_decode_info decode(const uint8_t* frames, size_t n_frames, size_t frame_len, Loss* loss,
                             std::vector<float> (&traces)[SSPSD_MAX_TRACES], size_t frame_stride = 0)
    {
        if (!frame_stride) frame_stride = frame_len;
        size_t payload = frame_len > SSPSD_HEADER_SIZE ? frame_len - SSPSD_HEADER_SIZE : 0;
        size_t cap = n_frames * std::max<size_t>(payload / 64 * 8, payload / 24) + 1;
        float* ptr[SSPSD_MAX_TRACES];
        for (int t = 0; t < SSPSD_MAX_TRACES; ++t) {
            traces[t].assign(cap, 0.f);
            ptr[t] = traces[t].data();
        }
        sspsd_decode_info info{};
        int32_t st = sspsd_decode_frames(d_, frames, n_frames, frame_len, frame_stride, SSPSD_MEM_HOST,
                                         loss ? &loss->c : nullptr, ptr, cap, SSPSD_MEM_HOST, &info);
        for (int t = 0; t < SSPSD_MAX_TRACES; ++t) traces[t].resize(t < (int)info.n_traces ? info.samples_per_trace : 0);
        if (st >= SSPSD_EHEADER && st <= SSPSD_ESHORT && info.frames_ok < n_frames) throw DecodeError(st, info.frames_ok);
        check(st);
        return info;
    }
    template <size_t N>
    sspsd_decode_info process_frames(PsdCascade<N>* const* cascades, uint32_t n, const uint8_t* frames, size_t n_frames,
                                     size_t frame_len, Loss* loss, Mem mem = Mem::Host)
    {
        sspsd_cascade* hs[SSPSD_MAX_TRACES] = {nullptr, nullptr, nullptr, nullptr};
        for (uint32_t t = 0; t < n && t < SSPSD_MAX_TRACES; ++t) hs[t] = cascades[t] ? cascades[t]->handle() : nullptr;
        sspsd_decode_info info{};
        int32_t st = sspsd_cascade_process_frames(d_, hs, n, frames, n_frames, frame_len, frame_len, (int32_t)mem,
                                                  loss ? &loss->c : nullptr, &info);
        if (st >= SSPSD_EHEADER && st <= SSPSD_ESHORT && info.frames_ok < n_frames) throw DecodeError(st, info.frames_ok);
        check(st);
        return info;
    }
    /// fused decode -> cross-spectral density: x <- trace trace_x, y <- trace trace_y of every frame
    template <size_t N>
    sspsd_decode_info process_frames(CsdCascade<N>& c, uint32_t trace_x, uint32_t trace_y, const uint8_t* frames,
                                     size_t n_frames, size_t frame_len, Loss* loss, Mem mem = Mem::Host,
                                     size_t frame_stride = 0)
    {
        sspsd_decode_info info{};
        int32_t st = sspsd_csd_process_frames(d_, c.handle(), trace_x, trace_y, frames, n_frames, frame_len,
                                              frame_stride ? frame_stride : frame_len, (int32_t)mem,
                                              loss ? &loss->c : nullptr, &info);
        return finish(st, info);
    }
    /// fused decode -> cross-spectral matrix: channel i <- trace traces[i] (one index per channel; empty: 0 .. K-1)
    template <size_t N>
    sspsd_decode_info process_frames(CsmCascade<N>& m, const std::vector<uint32_t>& traces, const uint8_t* frames,
                                     size_t n_frames, size_t frame_len, Loss* loss, Mem mem = Mem::Host,
                                     size_t frame_stride = 0)
    {
        sspsd_decode_info info{};
        int32_t st = sspsd_csm_process_frames(d_, m.handle(), trace_map(m, traces), frames, n_frames, frame_len,
                                              frame_stride ? frame_stride : frame_len, (int32_t)mem,
                                              loss ? &loss->c : nullptr, &info);
        return finish(st, info);
    }
    /// fused decode -> two-sided spectrum: I/Q mode i, q <- traces[0], traces[1]; heterodyne mode x <- traces[0],
    /// mixed on the device (empty: 0 .. 1 / 0)
    template <size_t N>
    sspsd_decode_info process_frames(ZoomCascade<N>& z, const std::vector<uint32_t>& traces, const uint8_t* frames,
                                     size_t n_frames, size_t frame_len, Loss* loss, Mem mem = Mem::Host,
                                     size_t frame_stride = 0)
    {
        sspsd_decode_info info{};
        int32_t st = sspsd_zoom_process_frames(d_, z.handle(), trace_map(z, traces), frames, n_frames, frame_len,
                                               frame_stride ? frame_stride : frame_len, (int32_t)mem,
                                               loss ? &loss->c : nullptr, &info);
        return finish(st, info);
    }
    sspsd_decoder* handle() const { return d_; }

    /// the C ABI's view of a ZoomCascade trace map (NULL for the identity); throws unless one index per trace read
    template <size_t N>
    static const uint32_t* trace_map(const ZoomCascade<N>& z, const std::vector<uint32_t>& traces)
    {
        if (traces.empty()) return nullptr;
        if (traces.size() != (size_t)z.traces()) throw Error(SSPSD_EINVAL, "one trace index per stream of the mode");
        return traces.data();
    }
    /// the C ABI's view of a CsmCascade trace map (NULL for the identity); throws unless one index per channel
    template <size_t N>
    static const uint32_t* trace_map(const CsmCascade<N>& m, const std::vector<uint32_t>& traces)
    {
        if (traces.empty()) return nullptr;
        if (traces.size() != (size_t)m.channels()) throw Error(SSPSD_EINVAL, "one trace index per channel");
        return traces.data();
    }
    /// the result of a fused call: a malformed frame throws DecodeError, any other failure Error
    static sspsd_decode_info finish(int32_t st, const sspsd_decode_info& info)
    {
        if (st >= SSPSD_EHEADER && st <= SSPSD_ESHORT) throw DecodeError(st, info.frames_ok);
        check(st);
        return info;
    }

private:
    sspsd_decoder* d_ = nullptr;
};

/// Data::Noise / Data::Dsm of src/source.rs:66-79, 104-134, generated on the device.
class Source {
public:
    static constexpr uint64_t SEED = 0x7654321;  // source.rs:69
    /// `--noise e` (source.rs:40-42): PSD ~ f^e
    static Source noise(int32_t exponent, uint64_t seed = SEED, int device = 0, void* stream = nullptr)
    {
        return Source(SSPSD_SOURCE_NOISE, exponent, seed, device, stream);
    }
    /// `--dsm ftw` (source.rs:44-46): MASH-1-1-1 modulated sine marker
    static Source dsm(uint32_t ftw, int device = 0, void* stream = nullptr)
    {
        return Source(SSPSD_SOURCE_DSM, (int64_t)ftw, 0, device, stream);
    }
    Source(int32_t kind, int64_t param, uint64_t seed, int device, void* stream)
    {
        check(sspsd_source_create(kind, param, seed, device, stream, &h_));
    }
    Source(const Source&) = delete;
    Source& operator=(const Source&) = delete;
    Source(Source&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    ~Source() { sspsd_source_destroy(h_); }
    void reset() { check(sspsd_source_reset(h_)); }
    uint64_t position() const
    {
        uint64_t p;
        check(sspsd_source_position(h_, &p));
        return p;
    }
    /// Source::get: the next n samples into device memory
    void get(float* d_out, size_t n) { check(sspsd_source_generate(h_, d_out, n)); }
    /// feed the next n samples to a cascade without touching host memory
    template <size_t N>
    void feed(PsdCascade<N>& c, size_t n)
    {
        check(sspsd_cascade_process_source(c.handle(), h_, n));
    }

private:
    sspsd_source* h_ = nullptr;
};

/// Data::Udp of src/source.rs:81-93, 159-165: recvmmsg into page-locked slots, decoded per batch.
class Receiver {
public:
    explicit Receiver(const char* ip = "0.0.0.0", uint16_t port = 9293, uint32_t slot_bytes = 2048,
                      uint32_t n_slots = 1024, bool pinned = true)
    {
        check(sspsd_receiver_create(ip, port, slot_bytes, n_slots, pinned ? SSPSD_RECV_PINNED : SSPSD_RECV_PAGEABLE, &h_));
    }
    Receiver(const Receiver&) = delete;
    Receiver& operator=(const Receiver&) = delete;
    ~Receiver() { sspsd_receiver_destroy(h_); }
    uint16_t port() const
    {
        uint16_t p;
        check(sspsd_receiver_info(h_, &p, nullptr, nullptr));
        return p;
    }
    /// next run of equally sized datagrams: {first slot, count, datagram length}; slots are slot_bytes apart
    struct Run {
        const uint8_t* frames;
        size_t n_frames, frame_len;
    };
    Run recv(uint32_t max_frames = 1024, int32_t timeout_ms = 1000)
    {
        Run r{};
        check(sspsd_receiver_recv(h_, max_frames, timeout_ms, &r.frames, &r.n_frames, &r.frame_len));
        return r;
    }
    /// recv + FrameDecoder::process_frames into a CsdCascade (info.frames_ok == 0 on timeout)
    template <size_t N>
    sspsd_decode_info pump(FrameDecoder& d, CsdCascade<N>& c, uint32_t trace_x, uint32_t trace_y, Loss* loss,
                           uint32_t max_frames = 1024, int32_t timeout_ms = 1000)
    {
        sspsd_decode_info info{};
        int32_t st = sspsd_receiver_pump_csd(h_, d.handle(), c.handle(), trace_x, trace_y, max_frames, timeout_ms,
                                             loss ? &loss->c : nullptr, &info);
        return FrameDecoder::finish(st, info);
    }
    /// recv + FrameDecoder::process_frames into a CsmCascade (info.frames_ok == 0 on timeout)
    template <size_t N>
    sspsd_decode_info pump(FrameDecoder& d, CsmCascade<N>& m, const std::vector<uint32_t>& traces, Loss* loss,
                           uint32_t max_frames = 1024, int32_t timeout_ms = 1000)
    {
        sspsd_decode_info info{};
        int32_t st = sspsd_receiver_pump_csm(h_, d.handle(), m.handle(), FrameDecoder::trace_map(m, traces), max_frames,
                                             timeout_ms, loss ? &loss->c : nullptr, &info);
        return FrameDecoder::finish(st, info);
    }
    /// recv + FrameDecoder::process_frames into a ZoomCascade (info.frames_ok == 0 on timeout)
    template <size_t N>
    sspsd_decode_info pump(FrameDecoder& d, ZoomCascade<N>& z, const std::vector<uint32_t>& traces, Loss* loss,
                           uint32_t max_frames = 1024, int32_t timeout_ms = 1000)
    {
        sspsd_decode_info info{};
        int32_t st = sspsd_receiver_pump_zoom(h_, d.handle(), z.handle(), FrameDecoder::trace_map(z, traces),
                                              max_frames, timeout_ms, loss ? &loss->c : nullptr, &info);
        return FrameDecoder::finish(st, info);
    }
    sspsd_receiver* handle() const { return h_; }

private:
    sspsd_receiver* h_ = nullptr;
};

/// struct Var + VarBuilder defaults, src/var.rs:4-45
struct Var {
    int32_t x_exp = -2;
    int32_t sinx_exp = 4;
    float clip = std::numeric_limits<float>::max();
    size_t dc_cut = 2;
    float eval(const std::vector<float>& phase_psd, const std::vector<float>& frequencies, float tau) const
    {
        sspsd_var v{x_exp, sinx_exp, clip, 0, dc_cut};
        return sspsd_var_eval(&v, phase_psd.data(), frequencies.data(), std::min(phase_psd.size(), frequencies.size()), tau);
    }
};

/// struct Trace + Trace::plot + struct Trapezoidal, src/bin/psd.rs:96-157
struct Trace {
    std::string name;
    std::vector<Break> breaks;
    std::vector<float> psd;
    std::vector<float> frequencies;
    /// -> (sqrt of the trapezoidal integral over [integral_start, integral_end] in units of fs * f, plot points)
    std::pair<float, std::vector<std::array<double, 2>>> plot(float fs = 1.0f, float integral_start = 1e-6f,
                                                              float integral_end = 0.5f, bool integrate = false) const
    {
        sspsd_plot_opts o{fs, integral_start, integral_end, integrate ? 1u : 0u};
        const size_t n = std::min(psd.size(), frequencies.size());
        std::vector<std::array<double, 2>> xy(n ? n : 1);
        size_t np = xy.size();
        float integral = 0.f;
        check(sspsd_trace_plot(&o, psd.data(), frequencies.data(), n, &integral, &xy[0][0], &np));
        xy.resize(np);
        return {integral, std::move(xy)};
    }
};

/// The receiver loop's `Vec<(&str, PsdCascade<N>)>` (src/bin/psd.rs:170-183) spread over the GPUs of the box:
/// channel (trace) c lives on devices[c % devices.size()], or ONE long capture is cut into time chunks; NCCL / peer
/// loads stay inside the library (sspsd_group_*).
template <size_t N>
class Group {
public:
    enum class Shard : int32_t { Channels = SSPSD_SHARD_CHANNELS, Time = SSPSD_SHARD_TIME };
    explicit Group(const std::vector<int32_t>& devices, Shard mode = Shard::Channels, int32_t hbf = SSPSD_HBF_140)
    {
        sspsd_config cfg;
        check(sspsd_config_default((uint32_t)N, &cfg));
        cfg.hbf = hbf;
        check(sspsd_group_create(&cfg, devices.data(), (uint32_t)devices.size(), (int32_t)mode, &g_));
    }
    Group(const Group&) = delete;
    Group& operator=(const Group&) = delete;
    ~Group() { sspsd_group_destroy(g_); }
    void set_avg(AvgOpts a) { check(sspsd_group_set_avg(g_, sspsd_avg_opts{a.limit, a.count})); }
    void set_detrend(Detrend d) { check(sspsd_group_set_detrend(g_, (int32_t)d)); }
    /// `dec[channel].process(&trace)`
    void process(uint32_t channel, const float* x, size_t n, Mem mem = Mem::Host)
    {
        check(sspsd_group_process_f32(g_, channel, x, n, (int32_t)mem));
    }
    void process(uint32_t channel, const std::vector<float>& x) { process(channel, x.data(), x.size()); }
    std::pair<std::vector<float>, std::vector<Break>> psd(uint32_t channel = 0, const MergeOpts& o = MergeOpts()) const
    {
        sspsd_merge_opts mo{o.keep_overlap, o.min_count, o.keep_transition_band};
        std::vector<float> p(SSPSD_MAX_STAGES * (N / 2 + 1));
        sspsd_break cb[SSPSD_MAX_STAGES];
        size_t pl = p.size(), bl = SSPSD_MAX_STAGES;
        check(sspsd_group_psd(g_, channel, &mo, p.data(), &pl, cb, &bl));
        p.resize(pl);
        std::vector<Break> b;
        for (size_t i = 0; i < bl; ++i)
            b.push_back(Break{(size_t)cb[i].start, cb[i].include != 0, cb[i].count, cb[i].avg,
                              {(size_t)cb[i].bins_start, (size_t)cb[i].bins_end}, (size_t)cb[i].fft_size,
                              (size_t)cb[i].decimation, (size_t)cb[i].pending, (size_t)cb[i].processed});
        return {std::move(p), std::move(b)};
    }
    // time chunks of one stream
    void time_plan(uint64_t total, uint32_t n_local_stages = 0) { check(sspsd_group_time_plan(g_, total, n_local_stages)); }
    sspsd_time_chunk time_chunk(uint32_t rank) const
    {
        sspsd_time_chunk c;
        check(sspsd_group_time_chunk(g_, rank, &c));
        return c;
    }
    void time_process(uint32_t rank, const float* x, size_t n, Mem mem = Mem::Host)
    {
        check(sspsd_group_time_process_f32(g_, rank, x, n, (int32_t)mem));
    }
    void time_process_all(const std::vector<float>& x) { check(sspsd_group_time_process_all_f32(g_, x.data(), x.size())); }
    void time_finish() { check(sspsd_group_time_finish(g_)); }
    void sync() { check(sspsd_group_sync(g_)); }

private:
    sspsd_group* g_ = nullptr;
};

}  // namespace sspsd
