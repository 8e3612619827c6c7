/* sspsd.h -- C ABI of the B200-native cascaded power-spectral-density library.
 *
 * Drop-in boundary for the hot path of quartiq/stabilizer-stream: every entry point replaces one
 * item of the reference's Rust API (file:line cited per function, relative to the reference
 * repository).  The reference has no FFI of its own; this is the interface its `gpu` module would
 * bind (see INTEGRATION.md for the Rust `extern "C"` block, build.rs and safe wrappers).
 *
 * Conventions
 *   - every function returns an int32 status (SSPSD_OK == 0); nothing unwinds or aborts across the
 *     boundary; sspsd_last_error() gives a thread-local human-readable message for the last failure;
 *   - host pointers are borrowed for the duration of the call only; SSPSD_MEM_DEVICE input is read
 *     asynchronously, in place (zero copy), on the handle's stream: it must stay valid and unmodified in
 *     stream order, i.e. until work queued on that stream after the call (an event recorded there, or
 *     sspsd_cascade_sync()) has completed; the caller owns output buffers;
 *     variable-length outputs use "capacity in / length out" size_t* parameters and return
 *     SSPSD_ESHORT (with the needed length written) when the capacity is too small;
 *   - `mem` says where a buffer lives: SSPSD_MEM_HOST (pageable or pinned host memory) or
 *     SSPSD_MEM_DEVICE (memory of the handle's CUDA device);
 *   - a handle is not thread-safe but may be moved between threads (`Send`, like the reference's
 *     PsdCascade, src/bin/psd.rs:170-176); distinct handles are independent;
 *   - all device work of a handle is ordered on one CUDA stream; calls that return data to the
 *     host synchronise that stream, process() on device memory does not;
 *   - there is no CPU fallback: if no CUDA device is usable every create call fails with
 *     SSPSD_ECUDA.
 */
#ifndef SSPSD_H
#define SSPSD_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSPSD_VERSION 1

/* status codes */
enum {
    SSPSD_OK = 0,
    SSPSD_EINVAL = 1,         /* bad argument (NULL handle, unsupported N, ...) */
    SSPSD_EUNIMPLEMENTED = 2, /* Detrend::Linear: `unimplemented!()` in the reference, src/psd.rs:110 */
    SSPSD_ECUDA = 3,          /* CUDA runtime error / no device */
    SSPSD_ENOMEM = 4,
    SSPSD_EHEADER = 5,        /* de::Error::InvalidHeader, src/de/mod.rs:21-22 */
    SSPSD_EFORMAT = 6,        /* de::Error::UnknownFormat, src/de/mod.rs:23-24 */
    SSPSD_ESIZE = 7,          /* de::Error::PayloadSize,   src/de/mod.rs:25-26 */
    SSPSD_EBATCHES = 8,       /* header batch count != payload batches: assert_eq! panic, src/de/data.rs:24,93,150,174 */
    SSPSD_ESHORT = 9,         /* output capacity too small, or frame shorter than its header (src/de/frame.rs:50 panics) */
    SSPSD_ENCCL = 10,         /* reserved for collective failures */
    SSPSD_EIO = 11            /* socket error of the UDP receiver (std::io::Error in src/source.rs:81-93, 161) */
};

enum { SSPSD_MEM_HOST = 0, SSPSD_MEM_DEVICE = 1 };

/* Window<N>::rectangular / ::hann, src/psd.rs:24-55 */
enum { SSPSD_WINDOW_RECT = 0, SSPSD_WINDOW_HANN = 1 };

/* enum Detrend, src/psd.rs:59-72 */
enum {
    SSPSD_DETREND_NONE = 0,
    SSPSD_DETREND_MIDPOINT = 1,
    SSPSD_DETREND_SPAN = 2,
    SSPSD_DETREND_MEAN = 3,
    SSPSD_DETREND_LINEAR = 4 /* rejected with SSPSD_EUNIMPLEMENTED */
};

/* Half-band decimator tap family restating idsp::hbf (src/psd.rs:2,124,246-253).
 * 140 = idsp HBF_TAPS ("140 dB"), 98 = idsp HBF_TAPS_98.  See DESIGN.md "parity unpinned". */
enum { SSPSD_HBF_98 = 0, SSPSD_HBF_140 = 1 };

/* const DEPTH, src/psd.rs:117: every stage decimates by 1 << 3 */
#define SSPSD_DEPTH 3
#define SSPSD_MAX_STAGES 16

typedef struct {
    uint32_t n_fft;      /* const generic N of Psd<N>/PsdCascade<N>; power of two, 64..8192 */
    int32_t window;      /* SSPSD_WINDOW_*; PsdCascade::default() uses Hann, src/psd.rs:419 */
    int32_t hbf;         /* SSPSD_HBF_* */
    int32_t device;      /* CUDA device ordinal */
    void *stream;        /* cudaStream_t to order all work on (cudaStreamLegacy / cudaStreamPerThread are
                            accepted), or NULL for a private non-blocking stream */
    uint64_t max_batch;  /* largest number of samples handed to one kernel batch (0 = default 1<<28) */
    uint64_t host_stage; /* host-pointer process() calls are staged in pinned memory and launched once
                            this many samples are pending (0 = default 1<<22); psd()/set_*()/flush() launch
                            whatever is staged */
    uint64_t deep_defer; /* stages >= 1 run once this many samples are pending at stage 1 (>> 3 per deeper stage), so
                            that their kernels get full-size grids instead of ~20 small dependent launches per batch
                            (fewer launches; +12 % throughput at N = 512, neutral at N = 4096); every call that observes
                            state runs what is pending first, results do not depend on it (0 = default 1 << 26,
                            1 = run them with every batch) */
    uint32_t flags;      /* SSPSD_FLAG_* */
    uint32_t _pad;
} sspsd_config;
/* accumulate |X|^2 through per-CTA partial rows summed in fixed order instead of float atomics: readouts become
 * bit-reproducible from run to run (one extra small kernel per stage and batch) */
#define SSPSD_FLAG_DETERMINISTIC 1u

/* AvgOpts, src/psd.rs:360-376 */
typedef struct {
    uint32_t limit;
    uint32_t count;
} sspsd_avg_opts;

/* MergeOpts, src/psd.rs:339-358 */
typedef struct {
    uint32_t keep_overlap;
    uint32_t min_count;
    uint32_t keep_transition_band;
} sspsd_merge_opts;

/* struct Break, src/psd.rs:290-311 (`bins: Range<usize>` is bins_start..bins_end) */
typedef struct {
    uint64_t start;
    uint32_t include;
    uint32_t count;
    uint32_t avg;
    uint32_t _pad;
    uint64_t bins_start;
    uint64_t bins_end;
    uint64_t fft_size;
    uint64_t decimation;
    uint64_t pending;
    uint64_t processed;
} sspsd_break;

const char *sspsd_last_error(void);
/* constants of a half-band tap family: drain = hbf_dec_response_length(3) (src/psd.rs:149), halo = input
 * history the decimator kernel needs before a block (>= FIR span - 1); pure host query */
int32_t sspsd_hbf_info(int32_t hbf, uint32_t *drain, uint32_t *halo);
/* fills cfg with PsdCascade::default() (src/psd.rs:408-423): Hann, HBF_140, device 0 */
int32_t sspsd_config_default(uint32_t n_fft, sspsd_config *cfg);

/* ---------------------------------------------------------------------------------------------
 * PsdCascade<N>, src/psd.rs:399-544
 * --------------------------------------------------------------------------------------------- */
typedef struct sspsd_cascade sspsd_cascade;

/* PsdCascade::default(), src/psd.rs:408-423 */
int32_t sspsd_cascade_create(const sspsd_config *cfg, sspsd_cascade **out);
/* Drop */
void sspsd_cascade_destroy(sspsd_cascade *h);
/* #[derive(Clone)], src/psd.rs:399: deep copy of all per-stage state on the same device */
int32_t sspsd_cascade_clone(sspsd_cascade *h, sspsd_cascade **out);
/* `dec.clear()` + fresh default (Cmd::Reset, src/bin/psd.rs:190): forget all stages, keep options */
int32_t sspsd_cascade_reset(sspsd_cascade *h);
/* PsdCascade::process(&mut self, x: &[f32]), src/psd.rs:455-468.  Any n including 0.  Results do not
 * depend on how the stream is split over calls. */
int32_t sspsd_cascade_process_f32(sspsd_cascade *h, const float *x, size_t n, int32_t mem);
/* PsdCascade::set_avg(AvgOpts), src/psd.rs:431-436; applies to segments completed after the call */
int32_t sspsd_cascade_set_avg(sspsd_cascade *h, sspsd_avg_opts avg);
/* PsdCascade::set_detrend(Detrend), src/psd.rs:438-443 */
int32_t sspsd_cascade_set_detrend(sspsd_cascade *h, int32_t detrend);
/* PsdCascade::rbw(), src/psd.rs:427-429 */
int32_t sspsd_cascade_rbw(const sspsd_cascade *h, float *rbw);
/* PsdCascade::psd(&MergeOpts) -> (Vec<f32>, Vec<Break>), src/psd.rs:479-543.
 * p_len / b_len: capacity in, length out.  p needs at most stages*(N/2+1) floats. */
int32_t sspsd_cascade_psd(sspsd_cascade *h, const sspsd_merge_opts *opts, float *p, size_t *p_len,
                          sspsd_break *b, size_t *b_len);
/* number of stages currently alive (self.stages.len()) */
int32_t sspsd_cascade_num_stages(sspsd_cascade *h, uint32_t *n);
/* the CUDA stream (cudaStream_t) all work of the handle is ordered on: cfg.stream, or the private stream */
int32_t sspsd_cascade_stream(const sspsd_cascade *h, void **stream);
/* launch everything staged from host-pointer process() calls */
int32_t sspsd_cascade_flush(sspsd_cascade *h);
/* flush + wait for the handle's stream */
int32_t sspsd_cascade_sync(sspsd_cascade *h);

/* ---------------------------------------------------------------------------------------------
 * Cross-spectral density of two streams (no reference analogue: the reference's Psd::process with |c|^2
 * replaced by conj(cx) cy, see DESIGN.md).  Traces that belong together -- ADC0/DAC0 of a dual-IIR
 * channel, BI/BQ of a lock-in, ADC0/ADC1 -- are fed pairwise; x and y go through the same cascade
 * (segments, window, detrend, half-band decimators, EWMA weights), and every stage accumulates
 *   Sxx = sum w |X|^2,  Syy = sum w |Y|^2,  Sxy = sum w conj(X) Y   (scipy.signal.csd's convention)
 * so for y = h * x the transfer function is H = pxy / pxx and the coherence |pxy|^2 / (pxx pyy).  The
 * readout has the breaks of sspsd_cascade_psd and the same 1/(gain_i 8^i) scale on every row: pxx is what
 * a cascade fed x alone returns.  n_fft = 64 .. 4096 (8192 returns SSPSD_EINVAL: the two-for-one transform
 * is an N-point complex FFT).  SSPSD_MEM_DEVICE input follows the rule of sspsd_cascade_process_f32 for
 * BOTH x and y, on the handle's stream (sspsd_csd_stream).  One long capture can be spread over GPUs in time
 * chunks: a group of kind SSPSD_GROUP_CSD (sspsd_group_create_kind).
 * --------------------------------------------------------------------------------------------- */
typedef struct sspsd_csd sspsd_csd;
int32_t sspsd_csd_create(const sspsd_config *cfg, sspsd_csd **out);
void sspsd_csd_destroy(sspsd_csd *h);
/* deep copy of all per-stage state of both channels */
int32_t sspsd_csd_clone(sspsd_csd *h, sspsd_csd **out);
int32_t sspsd_csd_reset(sspsd_csd *h);
/* the next n samples of both streams (x and y in the same memory kind); any n including 0; results do not
 * depend on how the streams are split over calls */
int32_t sspsd_csd_process_f32(sspsd_csd *h, const float *x, const float *y, size_t n, int32_t mem);
int32_t sspsd_csd_set_avg(sspsd_csd *h, sspsd_avg_opts avg);
int32_t sspsd_csd_set_detrend(sspsd_csd *h, int32_t detrend);
int32_t sspsd_csd_rbw(const sspsd_csd *h, float *rbw);
/* pxx, pyy: *p_len floats; pxy: 2 * *p_len floats, (re, im) interleaved; breaks as sspsd_cascade_psd */
int32_t sspsd_csd_read(sspsd_csd *h, const sspsd_merge_opts *opts, float *pxx, float *pyy, float *pxy,
                       size_t *p_len, sspsd_break *b, size_t *b_len);
int32_t sspsd_csd_num_stages(sspsd_csd *h, uint32_t *n);
int32_t sspsd_csd_stream(const sspsd_csd *h, void **stream);
int32_t sspsd_csd_flush(sspsd_csd *h);
int32_t sspsd_csd_sync(sspsd_csd *h);

/* ---------------------------------------------------------------------------------------------
 * Cross-spectral matrix of k = 2, 3 or 4 streams (a Stabilizer stream's traces: ADC0, ADC1, DAC0, DAC1 of
 * AdcDac, ...).  All k go through one cascade, and every stage accumulates the Hermitian matrix
 *   S_ij = sum w conj(X_i) X_j
 * (sspsd_csd_*'s convention: S[0,1] is pxy of a sspsd_csd fed (x0, x1)), with sspsd_csd_*'s limits
 * (n_fft = 64 .. 4096, Hann or rectangular, Linear detrend SSPSD_EUNIMPLEMENTED).  Every transform is
 * shared by all pairs, so the matrix costs k decimations and k FFTs per segment, where k (k - 1) / 2
 * sspsd_csd handles cost k (k - 1) of each.  k = 2 computes exactly what sspsd_csd_* computes.  Time-chunked
 * multi-GPU groups: kind SSPSD_GROUP_CSM (sspsd_group_create_kind).
 * --------------------------------------------------------------------------------------------- */
typedef struct sspsd_csm sspsd_csm;
/* k not in {2, 3, 4}: SSPSD_EINVAL */
int32_t sspsd_csm_create(const sspsd_config *cfg, int32_t k, sspsd_csm **out);
void sspsd_csm_destroy(sspsd_csm *h);
int32_t sspsd_csm_clone(sspsd_csm *h, sspsd_csm **out);
int32_t sspsd_csm_channels(const sspsd_csm *h, int32_t *k);
int32_t sspsd_csm_reset(sspsd_csm *h);
/* x: k pointers to the next n samples of each stream (all in the same memory kind); any n including 0 */
int32_t sspsd_csm_process_f32(sspsd_csm *h, const float *const *x, size_t n, int32_t mem);
int32_t sspsd_csm_set_avg(sspsd_csm *h, sspsd_avg_opts avg);
int32_t sspsd_csm_set_detrend(sspsd_csm *h, int32_t detrend);
int32_t sspsd_csm_rbw(const sspsd_csm *h, float *rbw);
/* s: 2 k k *p_len floats, S_ij[b] at s[2 ((i k + j) *p_len + b) + {0, 1}] (re, im) with *p_len the merged
 * length on return; the diagonal is real (imaginary part exactly 0) and S_ji = conj(S_ij) exactly.  On input
 * *p_len is the capacity per (i, j); too small: SSPSD_ESHORT with the lengths needed, as sspsd_csd_read */
int32_t sspsd_csm_read(sspsd_csm *h, const sspsd_merge_opts *opts, float *s, size_t *p_len, sspsd_break *b,
                       size_t *b_len);
int32_t sspsd_csm_num_stages(sspsd_csm *h, uint32_t *n);
int32_t sspsd_csm_stream(const sspsd_csm *h, void **stream);
int32_t sspsd_csm_flush(sspsd_csm *h);
int32_t sspsd_csm_sync(sspsd_csm *h);

/* ---------------------------------------------------------------------------------------------
 * Two-sided spectrum of a complex stream z (DESIGN.md 3c), in one of two modes fixed at creation:
 *   SSPSD_ZOOM_IQ          z[n] = i[n] + i q[n] of two real streams (a lock-in's BI / BQ); ftw must be 0
 *   SSPSD_ZOOM_HETERODYNE  z[n] = x[n] exp(-2 pi i phi_n / 2^32), phi_n = (n ftw) mod 2^32, of one real stream:
 *                          x mixed down by the carrier f0 = ftw / 2^32 (in units of the sample rate; the DDS /
 *                          lock-in convention of sspsd_source's dsm), n the absolute sample index since create or
 *                          reset (integer arithmetic: exact over any stream length, independent of the call split)
 * z goes through the cascade of sspsd_cascade_* with its real and imaginary parts in lockstep (same segments,
 * window, EWMA weights, detrend of each part, half-band decimators), and every stage accumulates
 *   P+[k] = sum w |Z[k]|^2,  P-[k] = sum w |Z[N-k]|^2,  k = 0 .. N/2   (P-[0] = P+[0], P-[N/2] = P+[N/2]).
 * The readout has the breaks of sspsd_cascade_psd with the same options; each row is scaled by
 * 1 / (2 gain_i 8^i), the two-sided density: a real x fed as (x, 0) reads back about psd(x) / 2 on each side.
 * p_pos[j] is the density at f0 + f_j and p_neg[j] at f0 - f_j, f_j of sspsd_break_frequencies (f0 = 0 in I/Q
 * mode).  Limits as sspsd_csd_*: n_fft = 64 .. 4096 (else SSPSD_EINVAL), Hann or rectangular window, Linear
 * detrend SSPSD_EUNIMPLEMENTED.  SSPSD_MEM_DEVICE input follows the rule of sspsd_cascade_process_f32, on the
 * handle's stream (sspsd_zoom_stream).  Time-chunked multi-GPU groups: kind SSPSD_GROUP_ZOOM
 * (sspsd_group_create_kind); every rank's mixer starts at the absolute index of its first sample.
 * --------------------------------------------------------------------------------------------- */
typedef struct sspsd_zoom sspsd_zoom;
enum { SSPSD_ZOOM_IQ = 0, SSPSD_ZOOM_HETERODYNE = 1 };
/* an unknown mode, or ftw != 0 in I/Q mode: SSPSD_EINVAL */
int32_t sspsd_zoom_create(const sspsd_config *cfg, int32_t mode, uint32_t ftw, sspsd_zoom **out);
void sspsd_zoom_destroy(sspsd_zoom *h);
/* deep copy, the mixer's sample position included */
int32_t sspsd_zoom_clone(sspsd_zoom *h, sspsd_zoom **out);
/* back to no samples: the mixer's position restarts at 0, the carrier is kept */
int32_t sspsd_zoom_reset(sspsd_zoom *h);
/* the next n samples of i and q (I/Q mode; in heterodyne mode SSPSD_EINVAL with nothing consumed) */
int32_t sspsd_zoom_process_iq_f32(sspsd_zoom *h, const float *i, const float *q, size_t n, int32_t mem);
/* the next n samples of x (heterodyne mode; in I/Q mode SSPSD_EINVAL with nothing consumed) */
int32_t sspsd_zoom_process_f32(sspsd_zoom *h, const float *x, size_t n, int32_t mem);
int32_t sspsd_zoom_set_avg(sspsd_zoom *h, sspsd_avg_opts avg);
int32_t sspsd_zoom_set_detrend(sspsd_zoom *h, int32_t detrend);
int32_t sspsd_zoom_rbw(const sspsd_zoom *h, float *rbw);
/* p_pos, p_neg: *p_len floats each; capacity and SSPSD_ESHORT as sspsd_csd_read */
int32_t sspsd_zoom_read(sspsd_zoom *h, const sspsd_merge_opts *opts, float *p_pos, float *p_neg, size_t *p_len,
                        sspsd_break *b, size_t *b_len);
int32_t sspsd_zoom_carrier(const sspsd_zoom *h, int32_t *mode, uint32_t *ftw);
int32_t sspsd_zoom_num_stages(sspsd_zoom *h, uint32_t *n);
int32_t sspsd_zoom_stream(const sspsd_zoom *h, void **stream);
int32_t sspsd_zoom_flush(sspsd_zoom *h);
int32_t sspsd_zoom_sync(sspsd_zoom *h);
/* The mixer of heterodyne mode on its own, asynchronously on `stream`, all pointers device memory:
 *   i_out[k] = x[k] cos(2 pi phi / 2^32),  q_out[k] = -x[k] sin(2 pi phi / 2^32),  phi = ((pos0 + k) ftw) mod 2^32.
 * Every output is within 2^-23 |x[k]| of the float64 product; at multiples of a quarter turn the factors are
 * exactly 0 and +-1. */
int32_t sspsd_heterodyne_f32(void *stream, const float *x, size_t n, uint64_t pos0, uint32_t ftw, float *i_out,
                             float *q_out);

/* Break::frequencies(&[Break]) -> Vec<f32>, src/psd.rs:315-327 (pure host helper) */
int32_t sspsd_break_frequencies(const sspsd_break *b, size_t n_breaks, float *f, size_t *f_len);

/* ---- partial-accumulator access for multi-GPU readout (north_star item 5; no reference analogue:
 * the reference is single threaded, src/bin/psd.rs:170-183) ----
 * The per-stage |X|^2 accumulators of a cascade live in ONE device array
 * acc[SSPSD_MAX_STAGES][acc_stride] so that a single collective (NCCL sum over NVLink) can combine
 * the partial sums of several GPUs that processed disjoint segment ranges of the same stream. */
typedef struct {
    float *acc;          /* device pointer, SSPSD_MAX_STAGES * acc_stride floats */
    uint64_t acc_stride; /* floats per stage (>= N/2+1) */
    uint32_t n_stages;
    uint32_t _pad;
    uint64_t count_raw[SSPSD_MAX_STAGES]; /* segments accumulated per stage */
} sspsd_partials;
int32_t sspsd_cascade_partials(sspsd_cascade *h, sspsd_partials *out);
/* overwrite the per-stage segment counts after an external reduction of `acc` (boxcar averaging only) */
int32_t sspsd_cascade_set_counts(sspsd_cascade *h, const uint64_t *count_raw, uint32_t n_stages);

/* ---- time-chunked processing of ONE long stream by several handles (GPUs) ----
 * BASELINE config 5 / north_star item 5; no reference analogue (the reference is sequential).  The
 * stream is cut into chunks [own_lo, own_hi) of stage-0 samples.  A rank positions a fresh cascade with
 * sspsd_cascade_seek() somewhat before its chunk (FIR warm-up halo), restricts it with
 * sspsd_cascade_set_window() and feeds it the samples [pos, feed_hi) of the stream.  All bookkeeping then
 * runs in GLOBAL stream coordinates (segment k of every stage covers exactly the samples it covers in
 * a sequential run); a segment is accumulated iff it is fully valid (no warm-up contaminated sample)
 * and its start lies in [own_lo, own_hi) (stage-0 position own(i, j) = 8^i j + R 8 (8^i - 1)/7 of sample
 * j of stage i, R = drain), so the ranks' partial accumulators sum to the sequential result.  Only
 * stages < n_local run locally; the input stream of stage n_local is exported with
 * sspsd_cascade_take_tail(), gathered, and fed to rank 0's handle with sspsd_cascade_process_stage(),
 * which then runs the deep stages; sspsd_cascade_set_stream_state() installs the reduced counts.
 * Averaging (psd.rs:215-233) follows the GLOBAL segment order: with a finite `avg`, a rank weights its owned
 * segments as the reference would if the stream ended right after its last owned segment; the caller
 * multiplies each accumulator row by g^(later segments that rescale), g = avg/(avg+1), before the
 * reduction (stabilizer_stream_b200/multi.py: ewma_tail_factors).  Options must be set before the first
 * sample and stay constant for the run. */
int32_t sspsd_cascade_seek(sspsd_cascade *h, uint64_t pos);
int32_t sspsd_cascade_set_window(sspsd_cascade *h, uint64_t own_lo, uint64_t own_hi, uint32_t n_local);
/* samples [j_lo, j_hi) of the stage-n_local input stream produced so far (clipped to what exists);
 * len: capacity in, length out; *first = stream index of out[0] */
int32_t sspsd_cascade_take_tail(sspsd_cascade *h, uint64_t j_lo, uint64_t j_hi, float *out, size_t *len,
                                uint64_t *first, int32_t mem);
/* feed n samples directly into stage `stage`'s stream (the next samples of that stream, in order) */
int32_t sspsd_cascade_process_stage(sspsd_cascade *h, uint32_t stage, const float *x, size_t n, int32_t mem);
/* overwrite stage bookkeeping after an external reduction: samples received, averaging count (Psd::count) */
int32_t sspsd_cascade_set_stream_state(sspsd_cascade *h, uint32_t stage, uint64_t samples, uint64_t segments);

/* ---------------------------------------------------------------------------------------------
 * Multi-GPU partitioning (north_star item 5).  No reference analogue: the reference is ONE process that
 * loops over its traces on one thread (src/bin/psd.rs:170-183).  A group spreads that loop over GPUs:
 *   SSPSD_SHARD_CHANNELS  channel (trace) c lives on rank c % n_ranks; nothing is exchanged while processing;
 *   SSPSD_SHARD_TIME      ONE long stream is cut into n_ranks chunks (see "time-chunked processing" above); the
 *                         readout is ONE sum-reduction of [accumulator rows | counts | tail slices] to rank 0.
 * A group holds either all ranks in ONE process -- sspsd_group_create(devices[]): one handle per device,
 * ncclCommInitAll, or (ranks sharing a GPU, SSPSD_GROUP_REDUCE=p2p) a root kernel that sums the peers' rows
 * through peer pointers in fixed order -- or one rank of a multi-process job (torchrun, MPI):
 * sspsd_group_unique_id() on rank 0, the 128 bytes broadcast by the caller, sspsd_group_create_rank() everywhere.
 * NCCL (libnccl.so.2) is loaded on first use; collective failures return SSPSD_ENCCL.  Like a cascade handle, a group
 * is not thread-safe but may be moved between threads; in a multi-process group the calls marked "collective"
 * (sspsd_group_psd_all, sspsd_group_time_finish) must be made by every process, in the same order.
 * --------------------------------------------------------------------------------------------- */
typedef struct sspsd_group sspsd_group;
enum { SSPSD_SHARD_CHANNELS = 0, SSPSD_SHARD_TIME = 1 };
enum { SSPSD_REDUCE_NCCL = 0, SSPSD_REDUCE_P2P = 1 };
#define SSPSD_GROUP_ID_BYTES 128
#define SSPSD_GROUP_MAX_RANKS 64

int32_t sspsd_group_create(const sspsd_config *cfg, const int32_t *devices, uint32_t n_devices, int32_t shard_mode,
                           sspsd_group **out);
int32_t sspsd_group_unique_id(uint8_t id[SSPSD_GROUP_ID_BYTES]);
/* cfg->device = this rank's device, cfg->stream = the stream the rank's work is ordered on (NULL: private) */
int32_t sspsd_group_create_rank(const sspsd_config *cfg, const uint8_t id[SSPSD_GROUP_ID_BYTES], uint32_t rank,
                                uint32_t n_ranks, int32_t shard_mode, sspsd_group **out);
void sspsd_group_destroy(sspsd_group *g);
/* any pointer may be NULL; first_rank / n_local_ranks: the ranks this process holds; reduce: SSPSD_REDUCE_* in use */
int32_t sspsd_group_info(const sspsd_group *g, uint32_t *n_ranks, uint32_t *first_rank, uint32_t *n_local_ranks,
                         int32_t *shard_mode, int32_t *reduce);
/* PsdCascade::set_avg / set_detrend on every cascade of the group (existing and future ones) */
int32_t sspsd_group_set_avg(sspsd_group *g, sspsd_avg_opts avg);
int32_t sspsd_group_set_detrend(sspsd_group *g, int32_t detrend);
/* wait for all device work of the group's handles in this process */
int32_t sspsd_group_sync(sspsd_group *g);

/* ---- channels: `dec[channel].process(&trace)` of src/bin/psd.rs:174-182 ----
 * The cascade of a channel is created on first use on device (channel % n_ranks).  In a multi-process group a
 * call for a channel another process owns is a no-op returning SSPSD_OK, so every process can run the same loop. */
int32_t sspsd_group_process_f32(sspsd_group *g, uint32_t channel, const float *x, size_t n, int32_t mem);
/* where a channel lives: device = -1 if another process owns it */
int32_t sspsd_group_channel_device(const sspsd_group *g, uint32_t channel, int32_t *device, uint32_t *rank);
/* the cascade of a channel this process owns (borrowed: valid until the group is destroyed; NULL if the channel has not
 * received a sample yet or lives elsewhere) -- for the per-handle calls the group does not wrap (profile hooks, clone) */
int32_t sspsd_group_channel_handle(sspsd_group *g, uint32_t channel, sspsd_cascade **out);
/* psd() of one channel (single-process channel groups), or of THE stream of a time-chunked group after
 * sspsd_group_time_finish (result on the process that holds rank 0; lengths 0 elsewhere) */
int32_t sspsd_group_psd(sspsd_group *g, uint32_t channel, const sspsd_merge_opts *opts, float *p, size_t *p_len,
                        sspsd_break *b, size_t *b_len);
/* psd() of channels 0..n_channels-1 at once: channel c's spectrum at p + c * p_stride (p_lens[c] floats), its breaks
 * at b + c * b_stride.  In a multi-process group this is a collective (every process calls it): ONE
 * ncclAllGather of the accumulator rows + bookkeeping, merged on rank 0 (lengths 0 on the other ranks). */
int32_t sspsd_group_psd_all(sspsd_group *g, uint32_t n_channels, const sspsd_merge_opts *opts, float *p, size_t p_stride,
                            size_t *p_lens, sspsd_break *b, size_t b_stride, size_t *b_lens);

/* ---- time chunks of one stream ---- */
typedef struct {
    uint64_t own_lo, own_hi;   /* ownership interval in stage-0 samples (own_hi = UINT64_MAX for the last rank) */
    uint64_t feed_lo, feed_hi; /* samples the rank must be fed: its chunk + FIR warm-up halo + completion halo */
    uint64_t tail_lo, tail_hi; /* owned index range of the stage-n_local input stream (tail_hi = UINT64_MAX: open) */
    uint32_t n_local;          /* stages that run on every rank; deeper ones run on rank 0 after the exchange */
    uint32_t _pad;
} sspsd_time_chunk;
/* pure host planner: what rank `rank` of `n_ranks` is fed for a stream of `total` samples (n_local_stages 0 = auto) */
int32_t sspsd_time_plan(uint32_t n_fft, int32_t window, int32_t hbf, uint64_t total, uint32_t n_ranks, uint32_t rank,
                        uint32_t n_local_stages, sspsd_time_chunk *out);
/* start a capture of `total` samples: plans every rank, creates + positions this process's handles */
int32_t sspsd_group_time_plan(sspsd_group *g, uint64_t total, uint32_t n_local_stages);
int32_t sspsd_group_time_chunk(const sspsd_group *g, uint32_t rank, sspsd_time_chunk *out);
/* the next n samples of rank `rank`'s range [feed_lo, feed_hi), in order (no-op for ranks of other processes) */
int32_t sspsd_group_time_process_f32(sspsd_group *g, uint32_t rank, const float *x, size_t n, int32_t mem);
/* single-process groups: x = the whole stream in host memory, the library feeds every rank its range */
int32_t sspsd_group_time_process_all_f32(sspsd_group *g, const float *x, size_t n);
/* every local rank generates its own range of the synthetic stream (SSPSD_SOURCE_NOISE, exponent >= 0) on its device */
int32_t sspsd_group_time_process_noise(sspsd_group *g, int64_t exponent, uint64_t seed);
/* the exchange (collective in a multi-process group): ONE reduction to rank 0, which then runs the deep stages */
int32_t sspsd_group_time_finish(sspsd_group *g);

/* ---- group kinds: time chunks of the cross-spectral handles ----
 * A group made by sspsd_group_create / _create_rank is of kind SSPSD_GROUP_PSD.  The other kinds spread one capture of
 * several streams over GPUs as the PSD kind spreads one stream: the same planner (sspsd_time_plan, sspsd_time_chunk),
 * every rank a sspsd_csd / sspsd_csm / sspsd_zoom handle positioned and windowed on all its channels alike, and ONE
 * reduction of [accumulator rows | counts | every channel's tail slices] to rank 0, which runs the deep stages.  Cross
 * kinds are SSPSD_SHARD_TIME only (SSPSD_SHARD_CHANNELS: SSPSD_EINVAL, the channels of a cross-spectrum share every
 * transform) and take the limits of their handles (n_fft = 64 .. 4096, else SSPSD_EINVAL).  In heterodyne mode every
 * rank's mixer starts at its feed_lo, so phi_n = (n ftw) mod 2^32 runs over the absolute index of the whole stream.
 *   kind       SSPSD_GROUP_*
 *   channels   CSM: k = 2 .. 4; CSD and zoom: 2 (0 = that); PSD: 1 (0 = that)
 *   zoom_mode  SSPSD_ZOOM_IQ / SSPSD_ZOOM_HETERODYNE (zoom only, else 0); ftw: the carrier (heterodyne only, else 0)
 * On a group of another kind, sspsd_group_psd, sspsd_group_time_process_f32 / _all_f32 / _noise of a cross kind and the
 * cross readouts return SSPSD_EINVAL with nothing consumed. */
enum { SSPSD_GROUP_PSD = 0, SSPSD_GROUP_CSD = 1, SSPSD_GROUP_CSM = 2, SSPSD_GROUP_ZOOM = 3 };
typedef struct {
    int32_t kind;
    int32_t channels;
    int32_t zoom_mode;
    uint32_t ftw;
} sspsd_group_kind;
int32_t sspsd_group_create_kind(const sspsd_config *cfg, const sspsd_group_kind *kind, const int32_t *devices,
                                uint32_t n_devices, int32_t shard_mode, sspsd_group **out);
int32_t sspsd_group_create_kind_rank(const sspsd_config *cfg, const sspsd_group_kind *kind,
                                     const uint8_t id[SSPSD_GROUP_ID_BYTES], uint32_t rank, uint32_t n_ranks,
                                     int32_t shard_mode, sspsd_group **out);
/* the kind of a group, channels filled in */
int32_t sspsd_group_kind_of(const sspsd_group *g, sspsd_group_kind *out);
/* x: one pointer per input stream of the kind, in the order of the handle's process call (PSD 1, CSD 2 (x, y),
 * CSM k, zoom I/Q 2 (i, q), zoom heterodyne 1), all in the same memory kind; otherwise as sspsd_group_time_process_f32 */
int32_t sspsd_group_time_process_multi_f32(sspsd_group *g, uint32_t rank, const float *const *x, size_t n, int32_t mem);
/* single-process groups: x[i] = the whole of stream i in host memory, the library feeds every rank its range */
int32_t sspsd_group_time_process_all_multi_f32(sspsd_group *g, const float *const *x, size_t n);
/* rank 0's result after sspsd_group_time_finish, with the layouts and SSPSD_ESHORT rules of sspsd_csd_read /
 * sspsd_csm_read / sspsd_zoom_read (lengths 0 on the processes that do not hold rank 0) */
int32_t sspsd_group_csd_read(sspsd_group *g, const sspsd_merge_opts *opts, float *pxx, float *pyy, float *pxy,
                             size_t *p_len, sspsd_break *b, size_t *b_len);
int32_t sspsd_group_csm_read(sspsd_group *g, const sspsd_merge_opts *opts, float *s, size_t *p_len, sspsd_break *b,
                             size_t *b_len);
int32_t sspsd_group_zoom_read(sspsd_group *g, const sspsd_merge_opts *opts, float *p_pos, float *p_neg, size_t *p_len,
                              sspsd_break *b, size_t *b_len);

/* ---- measurement hooks (no reference analogue) ----
 * With profiling enabled every kernel launch of the handle is bracketed by CUDA events on the
 * handle's stream; sspsd_cascade_profile_read() synchronises, sums the event times per kernel class
 * and clears the log.  `launches` counts kernel launches since creation / the last read, whether
 * profiling is enabled or not. */
enum {
    SSPSD_PROF_PSD_STAGE0 = 0, /* psd_stage_kernel on stage 0 (units: input samples) */
    SSPSD_PROF_PSD_DEEP = 1,   /* psd_stage_kernel on stages >= 1 */
    SSPSD_PROF_DECIM_STAGE0 = 2,
    SSPSD_PROF_DECIM_DEEP = 3,
    SSPSD_PROF_OTHER = 4,      /* carry copies, EWMA rescale */
    SSPSD_PROF_NCLASS = 5
};
typedef struct {
    double ms[SSPSD_PROF_NCLASS];       /* summed device time per class */
    uint64_t launches[SSPSD_PROF_NCLASS];
    uint64_t units[SSPSD_PROF_NCLASS];  /* input samples consumed by those launches */
    uint64_t launches_total;
} sspsd_profile;
int32_t sspsd_cascade_profile_enable(sspsd_cascade *h, int32_t on);
int32_t sspsd_cascade_profile_read(sspsd_cascade *h, sspsd_profile *out);

/* ---------------------------------------------------------------------------------------------
 * Psd<N> + trait PsdStage, src/psd.rs:119-288 (a single stage with its decimated output exposed)
 * --------------------------------------------------------------------------------------------- */
typedef struct sspsd_stage sspsd_stage;

/* Psd::new(fft, win), src/psd.rs:137-152 (the FFT plan is internal) */
int32_t sspsd_stage_create(const sspsd_config *cfg, sspsd_stage **out);
void sspsd_stage_destroy(sspsd_stage *h);
/* the CUDA stream the stage's work is ordered on (see sspsd_cascade_stream) */
int32_t sspsd_stage_stream(const sspsd_stage *h, void **stream);
/* Psd::set_avg / set_detrend, src/psd.rs:154-160 */
int32_t sspsd_stage_set_avg(sspsd_stage *h, uint32_t avg);
int32_t sspsd_stage_set_detrend(sspsd_stage *h, int32_t detrend);
/* PsdStage::process(x, y) -> &mut y[..n], src/psd.rs:196-269.  y_len: capacity in, length out */
int32_t sspsd_stage_process_f32(sspsd_stage *h, const float *x, size_t n, int32_t x_mem, float *y,
                                size_t *y_len, int32_t y_mem);
/* PsdStage::spectrum(): N/2+1 accumulated powers, src/psd.rs:271-273 */
int32_t sspsd_stage_spectrum(sspsd_stage *h, float *out, size_t *len, int32_t mem);
/* PsdStage::count(), src/psd.rs:275-277 */
int32_t sspsd_stage_count(sspsd_stage *h, uint32_t *count);
/* PsdStage::gain(), src/psd.rs:279-283 (the N/2*count product is formed in 64 bits, SURVEY.md D6) */
int32_t sspsd_stage_gain(sspsd_stage *h, float *gain);
/* PsdStage::buf(): currently buffered input items incl. overlap, src/psd.rs:285-287 */
int32_t sspsd_stage_buf(sspsd_stage *h, float *out, size_t *len, int32_t mem);

/* ---------------------------------------------------------------------------------------------
 * Frame decode + loss accounting, src/de/{frame,data}.rs, src/loss.rs
 * --------------------------------------------------------------------------------------------- */
/* enum Format, src/de/mod.rs:9-17 */
enum { SSPSD_FORMAT_ADCDAC = 1, SSPSD_FORMAT_FLS = 2, SSPSD_FORMAT_THERMOSTAT_EEM = 3, SSPSD_FORMAT_MPLL = 4 };
#define SSPSD_MAX_TRACES 4
#define SSPSD_HEADER_SIZE 8 /* src/de/frame.rs:8 */

/* struct Loss, src/loss.rs:4-8 (`seq: Option<u32>` is has_seq + seq) */
typedef struct {
    uint64_t received;
    uint64_t dropped;
    uint32_t seq;
    uint32_t has_seq;
} sspsd_loss;

typedef struct sspsd_decoder sspsd_decoder;
int32_t sspsd_decoder_create(int32_t device, void *stream, sspsd_decoder **out);
void sspsd_decoder_destroy(sspsd_decoder *d);
/* the CUDA stream the decoder's kernels run on; SSPSD_MEM_DEVICE frames must be complete in that stream's order */
int32_t sspsd_decoder_stream(const sspsd_decoder *d, void **stream);

typedef struct {
    uint32_t format;            /* Header.format of the batch (all frames of a call share it) */
    uint32_t n_traces;          /* 4 (AdcDac, Fls, ThermostatEem) or 3 (Mpll) */
    uint64_t samples_per_trace; /* f32 items written to each trace */
    uint64_t frames_ok;         /* frames decoded before the first error (== n_frames on success) */
} sspsd_decode_info;

/* Batched Frame::from_bytes (src/de/frame.rs:49-60) + Loss::update (src/loss.rs:11-26) +
 * payload.traces() (src/de/data.rs:28-82, 97-139, 154-163, 178-211) over n_frames equally sized
 * frames (`frame_len` bytes each, `frame_stride` bytes apart -- the file source's fixed
 * --frame-size, src/source.rs:29-31,135-148).  Traces are concatenated in frame order (lost frames
 * are not gap filled, like the reference).  `traces[t]` must hold `trace_cap` floats each, in
 * `traces_mem`.  On a malformed frame the call returns that frame's error code; `loss` and the
 * traces then cover exactly the frames before it (info->frames_ok), like a caller looping over
 * Frame::from_bytes would have seen. */
int32_t sspsd_decode_frames(sspsd_decoder *d, const uint8_t *frames, size_t n_frames, size_t frame_len,
                            size_t frame_stride, int32_t frames_mem, sspsd_loss *loss, float *const *traces,
                            size_t trace_cap, int32_t traces_mem, sspsd_decode_info *info);

/* Fused decode -> cascades: trace t of every frame is fed to cascades[t] (one PsdCascade per trace,
 * src/bin/psd.rs:174-182) without the f32 traces ever leaving the device.  cascades[t] may be NULL
 * to drop a trace.  SSPSD_MEM_HOST frames are fully consumed (copied and decoded) when the call
 * returns; the cascades' kernels may still be running (they are ordered on the cascades' own
 * streams).  Large host batches are copied in sub-chunks on a private copy stream so that decode
 * and cascades of one sub-chunk overlap the copy of the next; pass stream = NULL to
 * sspsd_decoder_create (a private stream) unless the decoder must be ordered on a caller stream. */
int32_t sspsd_cascade_process_frames(sspsd_decoder *d, sspsd_cascade *const *cascades, uint32_t n_cascades,
                                     const uint8_t *frames, size_t n_frames, size_t frame_len,
                                     size_t frame_stride, int32_t frames_mem, sspsd_loss *loss,
                                     sspsd_decode_info *info);

/* Fused decode -> cross-spectral matrix: channel i of `m` is fed trace traces[i] of every frame (traces == NULL:
 * channel i <- trace i), all K channels in lockstep on the handle's stream.  Host / device frames, loss accounting,
 * malformed frames (the good prefix before one is consumed by all K channels) and `info` exactly as
 * sspsd_cascade_process_frames.  An index may repeat (the matrix of repeated channels).  SSPSD_EINVAL, with nothing
 * consumed and `loss` unchanged: a NULL handle, an index >= 4, an index at or above the trace count of the frames'
 * format (Mpll has 3; checked against frame 0 before anything is queued), decoder and handle on different devices.
 * `traces` holds one index per channel (sspsd_csm_channels). */
int32_t sspsd_csm_process_frames(sspsd_decoder *d, sspsd_csm *m, const uint32_t *traces, const uint8_t *frames,
                                 size_t n_frames, size_t frame_len, size_t frame_stride, int32_t frames_mem,
                                 sspsd_loss *loss, sspsd_decode_info *info);
/* the same into a zoom handle: I/Q mode i <- traces[0], q <- traces[1] (Fls: BI, BQ are traces 2, 3); heterodyne
 * mode x <- traces[0], mixed on the device before it is fed.  traces == NULL: 0 (and 1). */
int32_t sspsd_zoom_process_frames(sspsd_decoder *d, sspsd_zoom *z, const uint32_t *traces, const uint8_t *frames,
                                  size_t n_frames, size_t frame_len, size_t frame_stride, int32_t frames_mem,
                                  sspsd_loss *loss, sspsd_decode_info *info);
/* the same into a cross-spectral density: x <- trace trace_x, y <- trace trace_y */
int32_t sspsd_csd_process_frames(sspsd_decoder *d, sspsd_csd *c, uint32_t trace_x, uint32_t trace_y,
                                 const uint8_t *frames, size_t n_frames, size_t frame_len, size_t frame_stride,
                                 int32_t frames_mem, sspsd_loss *loss, sspsd_decode_info *info);

/* Loss::update on one header (host helper, bit-exact u64/u32 wrapping arithmetic), src/loss.rs:11-26 */
void sspsd_loss_update(sspsd_loss *loss, uint32_t seq, uint8_t batches);
/* the ratio logged by Loss::analyze, src/loss.rs:28-30 */
float sspsd_loss_ratio(const sspsd_loss *loss);

/* ---------------------------------------------------------------------------------------------
 * Synthetic sources generated on the device: Data::Noise and Data::Dsm of src/source.rs:66-79,
 * 104-134 (SourceOpts --noise / --dsm, source.rs:40-47).  The generator state persists between
 * calls, so the stream does not depend on how it is cut into calls (the reference cuts it into
 * 4096-sample blocks, source.rs:116, 120).
 *   SSPSD_SOURCE_NOISE  param = the reference's `noise` exponent: PSD ~ f^param; |param| cascaded
 *                       first-order differentiators (param > 0, up to 8) or integrators (param < 0,
 *                       down to -4) over zero-mean unit-RMS uniform noise; seed keys the uniform
 *                       stream (Philox4x32-10; the reference's default seed is 0x7654321)
 *   SSPSD_SOURCE_DSM    param = the reference's `dsm` frequency tuning word (u32): sine marker
 *                       through a MASH-1-1-1 modulator, output in {-3.5 .. 3.5}; seed unused
 * Errors: SSPSD_EUNIMPLEMENTED for exponents outside -4..=8, SSPSD_EINVAL for bad arguments.
 * --------------------------------------------------------------------------------------------- */
typedef struct sspsd_source sspsd_source;
enum { SSPSD_SOURCE_NOISE = 0, SSPSD_SOURCE_DSM = 1 };
/* stream: as in sspsd_config (NULL = private stream, (void*)1 = legacy default stream) */
int32_t sspsd_source_create(int32_t kind, int64_t param, uint64_t seed, int32_t device, void *stream,
                            sspsd_source **out);
void sspsd_source_destroy(sspsd_source *s);
/* back to sample 0 with zeroed state (Source::new) */
int32_t sspsd_source_reset(sspsd_source *s);
/* the next n samples into device memory d_out, asynchronously on the source's stream (Source::get) */
int32_t sspsd_source_generate(sspsd_source *s, float *d_out, size_t n);
int32_t sspsd_source_position(const sspsd_source *s, uint64_t *pos);
/* continue the stream at sample `pos` (counter-based uniform stream: white and differentiated noise only;
 * integrated noise and the modulator carry state and return SSPSD_EUNIMPLEMENTED) */
int32_t sspsd_source_seek(sspsd_source *s, uint64_t pos);
/* generate the next n samples straight into the cascade (stream_test.rs:52-58 with a synthetic
 * source): no host memory is touched; generation and consumption share the cascade's stream */
int32_t sspsd_cascade_process_source(sspsd_cascade *c, sspsd_source *s, size_t n);

/* ---------------------------------------------------------------------------------------------
 * Plants (DESIGN.md 3d): seeded multi-channel test signals generated on the device, with a cross-spectral matrix
 * known in closed form.  A plant has m = 1 .. 4 independent inputs and k = 1 .. 4 outputs, each an FIR mix of all
 * the inputs with taps h[k][m][taps_len], taps_len = 1 .. 32:
 *   y_i[n] = round_f32( sum_{m'} sum_{t} h[i][m'][t] u_m'[n - t] ),   u[n] = 0 for n < 0,
 * the sum formed in f64, m' ascending then t ascending, rounded to f32 once; n is the absolute position since
 * create, reset or seek, so the outputs do not depend on how they are cut into calls.  Inputs:
 *   SSPSD_PLANT_NOISE  param = exponent e (0 .. 8), seed: exactly the stream of sspsd_source_create(SSPSD_SOURCE_NOISE,
 *                      e, seed) from position 0 (negative exponents carry state: SSPSD_EUNIMPLEMENTED, as
 *                      sspsd_source_seek; e > 8 likewise)
 *   SSPSD_PLANT_TONE   param = ftw (u32), amplitude a: u[n] = a c(phi_n), phi_n = (n ftw) mod 2^32, c the cosine
 *                      factor of the heterodyne mixer (sspsd_heterodyne_f32), rounded to f32; seed unused
 * A plant with k = m = taps_len = 1, tap 1.0 and a NOISE(e, seed) input reproduces sspsd_source NOISE(e, seed) bit for
 * bit.  The spec is copied at create.  Bad counts, lengths, kinds or tuning words: SSPSD_EINVAL.
 * --------------------------------------------------------------------------------------------- */
enum { SSPSD_PLANT_NOISE = 0, SSPSD_PLANT_TONE = 1 };
typedef struct {
    int32_t kind;
    int32_t _pad;
    int64_t param;   /* NOISE: exponent; TONE: ftw */
    uint64_t seed;   /* NOISE: Philox key */
    float amplitude; /* TONE */
    uint32_t _pad2;
} sspsd_plant_input;
typedef struct {
    uint32_t k, m, taps_len, _pad;
    const float *taps;                /* [k][m][taps_len] */
    const sspsd_plant_input *inputs;  /* m of them */
} sspsd_plant_spec;
typedef struct sspsd_plant sspsd_plant;
/* stream: as in sspsd_config (NULL = private stream, (void*)1 = legacy default stream) */
int32_t sspsd_plant_create(const sspsd_plant_spec *spec, int32_t device, void *stream, sspsd_plant **out);
void sspsd_plant_destroy(sspsd_plant *p);
/* back to position 0 */
int32_t sspsd_plant_reset(sspsd_plant *p);
/* continue at position pos (every input is counter-based) */
int32_t sspsd_plant_seek(sspsd_plant *p, uint64_t pos);
int32_t sspsd_plant_position(const sspsd_plant *p, uint64_t *pos);
/* the next n positions of all k outputs into the device buffers d_out[0 .. k-1], asynchronously on the plant's stream */
int32_t sspsd_plant_generate(sspsd_plant *p, float *const *d_out, size_t n);
/* Generate the next n positions straight into a handle, in bounded slices into scratch buffers the plant owns, on the
 * handle's stream (no host memory is touched).  k must equal the handle's input streams: PSD 1, CSD 2 (x, y), CSM the
 * handle's k, zoom I/Q 2 (i, q), zoom heterodyne 1 (mixed by the handle's own mixer).  A k mismatch, or a plant and a
 * handle on different devices: SSPSD_EINVAL with nothing consumed. */
int32_t sspsd_cascade_process_plant(sspsd_cascade *c, sspsd_plant *p, size_t n);
int32_t sspsd_csd_process_plant(sspsd_csd *c, sspsd_plant *p, size_t n);
int32_t sspsd_csm_process_plant(sspsd_csm *c, sspsd_plant *p, size_t n);
int32_t sspsd_zoom_process_plant(sspsd_zoom *z, sspsd_plant *p, size_t n);
/* Time-chunked groups (any kind): every local rank builds its own plant from `spec` on its device and stream, seeks
 * it to the rank's next unfed position (feed_lo + samples fed so far) and feeds the rest of its range; spec->k must
 * equal the kind's input streams.  The plants are cached on the group while the spec stays the same.  Nothing is
 * waited for on the host.  A k mismatch: SSPSD_EINVAL; a spec sspsd_plant_create refuses: its code; both with nothing
 * fed. */
int32_t sspsd_group_time_process_plant(sspsd_group *g, const sspsd_plant_spec *spec);

/* ---------------------------------------------------------------------------------------------
 * UDP ingest: the Data::Udp source of src/source.rs:81-93 (socket set-up: 1 MiB receive buffer,
 * reuse-address, multicast join, bind) and 159-165 (one `socket.read` + Frame::from_bytes +
 * loss.update + traces per datagram).  Here datagrams are collected with recvmmsg into a ring of
 * page-locked slots of slot_bytes each (default 2048 like the reference's read buffer,
 * source.rs:160; a longer datagram is cut the same way) and handed over as one strided frame array,
 * so a batch crosses PCIe once and is decoded by one kernel pass.
 * --------------------------------------------------------------------------------------------- */
typedef struct sspsd_receiver sspsd_receiver;
enum { SSPSD_RECV_PINNED = 0, SSPSD_RECV_PAGEABLE = 1 /* plain host memory: hosts without a CUDA device */ };
/* ip: dotted IPv4 (SourceOpts::ip, default "0.0.0.0"); port: SourceOpts::port (default 9293), 0 picks
 * a free port; slot_bytes: 0 = 2048, multiple of 8; n_slots: 0 = 1024 */
int32_t sspsd_receiver_create(const char *ip, uint16_t port, uint32_t slot_bytes, uint32_t n_slots, int32_t flags,
                              sspsd_receiver **out);
void sspsd_receiver_destroy(sspsd_receiver *r);
/* bound port, slot size (= frame_stride of the runs) and datagrams received so far; any pointer may be NULL */
int32_t sspsd_receiver_info(const sspsd_receiver *r, uint16_t *port, size_t *slot_bytes, uint64_t *datagrams);
/* The next run of up to max_frames equally sized datagrams, in arrival order: *frames points at the
 * first slot, consecutive frames are slot_bytes apart, the memory stays valid until the next call.
 * Waits up to timeout_ms for the first datagram (the reference's read timeout is 1000 ms,
 * source.rs:83); *n_frames == 0 on timeout. */
int32_t sspsd_receiver_recv(sspsd_receiver *r, uint32_t max_frames, int32_t timeout_ms, const uint8_t **frames,
                            size_t *n_frames, size_t *frame_len);
/* recv + sspsd_cascade_process_frames in one call (info->frames_ok == 0 on timeout) */
int32_t sspsd_receiver_pump(sspsd_receiver *r, sspsd_decoder *d, sspsd_cascade *const *cascades, uint32_t n_cascades,
                            uint32_t max_frames, int32_t timeout_ms, sspsd_loss *loss, sspsd_decode_info *info);
/* recv + sspsd_csm_process_frames / sspsd_csd_process_frames.  NULL handles and indices >= 4 are refused before a
 * datagram is taken; a trace map the frames' format cannot serve refuses (and drops) that run. */
int32_t sspsd_receiver_pump_csm(sspsd_receiver *r, sspsd_decoder *d, sspsd_csm *m, const uint32_t *traces,
                                uint32_t max_frames, int32_t timeout_ms, sspsd_loss *loss, sspsd_decode_info *info);
int32_t sspsd_receiver_pump_csd(sspsd_receiver *r, sspsd_decoder *d, sspsd_csd *c, uint32_t trace_x, uint32_t trace_y,
                                uint32_t max_frames, int32_t timeout_ms, sspsd_loss *loss, sspsd_decode_info *info);
/* recv + sspsd_zoom_process_frames, with the checks of sspsd_receiver_pump_csm */
int32_t sspsd_receiver_pump_zoom(sspsd_receiver *r, sspsd_decoder *d, sspsd_zoom *z, const uint32_t *traces,
                                 uint32_t max_frames, int32_t timeout_ms, sspsd_loss *loss, sspsd_decode_info *info);

/* ---------------------------------------------------------------------------------------------
 * Var::eval (AVAR/MVAR/FVAR from a phase PSD), src/var.rs:26-45 -- host helper on psd() output
 * --------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t x_exp;    /* default -2 */
    int32_t sinx_exp; /* default 4 */
    float clip;       /* default f32::MAX */
    uint32_t _pad;
    uint64_t dc_cut;  /* default 2 */
} sspsd_var;
float sspsd_var_eval(const sspsd_var *v, const float *phase_psd, const float *frequencies, size_t n, float tau);

/* ---------------------------------------------------------------------------------------------
 * Trace::plot + struct Trapezoidal, src/bin/psd.rs:96-157 -- host helper on psd() output: trapezoidal
 * integration over the irregular frequency grid of the merged spectrum (f32 running sums in the
 * reference's order).  `integral` receives sqrt(sum of the trapezoids whose upper frequency fs*f lies in
 * [integral_start, integral_end]); xy (may be NULL; n_points: capacity in points in, points out) receives
 * the plot points [log10(f) + log10(fs), integrate ? sqrt(running integral) : 10 (log10(p) - log10(fs))]
 * for every f that is a normal f32 (the DC bin is skipped, like `f.is_normal()` does).
 * --------------------------------------------------------------------------------------------- */
typedef struct {
    float fs;             /* AcqOpts::fs, default 1.0 */
    float integral_start; /* AcqOpts::integral_start, default 1e-6 */
    float integral_end;   /* AcqOpts::integral_end, default 0.5 */
    uint32_t integrate;   /* AcqOpts::integrate */
} sspsd_plot_opts;
int32_t sspsd_trace_plot(const sspsd_plot_opts *opts, const float *psd, const float *frequencies, size_t n,
                         float *integral, double *xy, size_t *n_points);

#ifdef __cplusplus
}
#endif
#endif /* SSPSD_H */
