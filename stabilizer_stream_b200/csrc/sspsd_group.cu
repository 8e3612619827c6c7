// sspsd_group.cu -- multi-GPU partitioning behind the C ABI (include/sspsd.h, "sspsd_group_*").
//
// The reference is one process looping over its traces on one thread (src/bin/psd.rs:170-183); north_star item 5
// asks for two partitionings that fall out of the cascade's structure (SURVEY.md 8e):
//   * channels: every trace owns an independent PsdCascade -> channel c lives on rank c % n_ranks, nothing is
//     exchanged while processing, the accumulators are gathered to rank 0 at readout (one ncclAllGather);
//   * time chunks of ONE stream: rank g owns the segments that start in its chunk of the stream, runs the
//     stages < K locally from a FIR warm-up halo (Cascade::seek / set_window), and at readout ONE sum-reduction
//     combines [K accumulator rows | K segment counts | the ranks' slices of the stage-K input stream]; rank 0
//     then runs the deep stages (<= 0.2 % of the work) on the gathered stream.
// The time-chunked mode also serves the cross-spectral kinds (sspsd_group_create_kind): a rank then holds an XCascade
// (CSD, CSM) or a ZoomCascade, whose K channels are windowed alike; the reduction carries R accumulator rows per stage
// and C tail streams (DESIGN.md 5, "Cross kinds").
// A group is either all ranks in ONE process (sspsd_group_create: one handle per device, ncclCommInitAll, or
// direct peer loads over NVLink) or one rank of a multi-process job (sspsd_group_create_rank: torchrun / MPI,
// ncclCommInitRank with an id made by sspsd_group_unique_id on rank 0).  NCCL is loaded with dlopen at the first
// group that needs it, so the library has no link-time dependency on it and shares whatever libnccl.so.2 the
// process already uses (e.g. torch's).
#include <dlfcn.h>
#include <nccl.h>

#include <time.h>

#include <algorithm>
#include <cstdio>
#include <cmath>
#include <cstring>
#include <mutex>
#include <new>
#include <vector>

#include "sspsd_plant.cuh"

using sspsd::Cascade;
using sspsd::XCascade;
using sspsd::ZoomCascade;
using sspsd::set_error;

extern "C" int32_t sspsd_source_seek(sspsd_source* s, uint64_t pos);

namespace {

// ---------------------------------------------------------------------------------------------
// NCCL through dlopen
// ---------------------------------------------------------------------------------------------
struct NcclApi {
    void* h = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Reduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};

NcclApi& nccl()
{
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* nm : names) {
            api.h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
            if (api.h) break;
        }
        if (!api.h) return;
        bool all = true;
        auto sym = [&](const char* s) {
            void* p = dlsym(api.h, s);
            if (!p) all = false;
            return p;
        };
        api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
        api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
        api.CommInitAll = (decltype(api.CommInitAll))sym("ncclCommInitAll");
        api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
        api.Reduce = (decltype(api.Reduce))sym("ncclReduce");
        api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
        api.GroupStart = (decltype(api.GroupStart))sym("ncclGroupStart");
        api.GroupEnd = (decltype(api.GroupEnd))sym("ncclGroupEnd");
        api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
        api.ok = all;
    });
    return api;
}

bool nccl_ok(ncclResult_t r, const char* what)
{
    if (r == ncclSuccess) return true;
    set_error(std::string(what) + ": " + (nccl().GetErrorString ? nccl().GetErrorString(r) : "NCCL error"));
    return false;
}
#define SSPSD_NCCL(call)                                  \
    do {                                                  \
        if (!nccl_ok((call), #call)) return SSPSD_ENCCL;  \
    } while (0)

double now_s()
{
    timespec t;
    clock_gettime(CLOCK_MONOTONIC, &t);
    return (double)t.tv_sec + 1e-9 * (double)t.tv_nsec;
}

using DevGuard = sspsd::DeviceGuard;

// ---------------------------------------------------------------------------------------------
// Planner of the time-chunked mode.  Mirrors the integer bookkeeping of the cascade (Cascade::seek,
// next_valid_from, own_offset; SURVEY.md App. A.2) so that every rank's owned segments are provably valid
// (free of FIR warm-up contamination) and complete.
// ---------------------------------------------------------------------------------------------
constexpr uint64_t NONE = ~0ull;

struct Geo {
    uint64_t n, hop, drain, halo;
};

uint64_t own_offset(unsigned i, uint64_t drain)
{
    // stage-0 position of sample 0 of stage i: c_0 = 0, c_{i+1} = 8 (c_i + R)
    uint64_t c = 0;
    for (unsigned q = 0; q < i; ++q) c = 8 * (c + drain);
    return c;
}

struct StreamSt {
    uint64_t L, craw, emitted;
};

// closed-form state of a sequential cascade after `total` samples
std::vector<StreamSt> stream_state(uint64_t total, const Geo& g, unsigned max_stages = SSPSD_MAX_STAGES)
{
    std::vector<StreamSt> out;
    uint64_t L = total;
    while (L > 0 && out.size() < max_stages) {
        const uint64_t craw = L < g.n ? 0 : 1 + (L - g.n) / g.hop;
        const uint64_t D = craw ? g.n + (craw - 1) * g.hop : 0;
        const uint64_t em = D / 8 > g.drain ? D / 8 - g.drain : 0;
        out.push_back({L, craw, em});
        L = em;
    }
    return out;
}

// stage-0 samples needed so that stage `stage` has received at least j_end samples
uint64_t needed_input(unsigned stage, uint64_t j_end, const Geo& g)
{
    for (unsigned q = 0; q < stage; ++q) {
        const uint64_t d = 8 * (j_end + g.drain);  // the previous stage must have decimated D >= d
        const uint64_t craw = d <= g.n ? 1 : 1 + (d - g.n + g.hop - 1) / g.hop;
        j_end = g.n + (craw - 1) * g.hop;
    }
    return j_end;
}

// smallest k with own(i, k * unit) >= pos (unit = hop for segments, 1 for samples)
uint64_t first_at_or_after(uint64_t pos, unsigned i, uint64_t unit, uint64_t drain)
{
    const uint64_t c = own_offset(i, drain);
    uint64_t step = unit;
    for (unsigned q = 0; q < i; ++q) step *= 8;
    return pos <= c ? 0 : (pos - c + step - 1) / step;
}

void plan_rank(uint64_t total, uint32_t world, uint32_t rank, const Geo& g, uint32_t n_local, sspsd_time_chunk* out)
{
    auto bound = [&](uint32_t r) -> uint64_t {
        if (r >= world) return total;
        // (128-bit product: total up to 2^63 samples, world up to 2^16)
        return (uint64_t)(((unsigned __int128)r * total) / world) / g.hop * g.hop;
    };
    const uint64_t own_lo = bound(rank), own_hi = bound(rank + 1);
    const bool last = rank + 1 == world;
    // ---- how far forward: every owned segment complete, every owned tail sample produced ----
    uint64_t feed_hi = total;
    if (!last) {
        uint64_t need = own_hi;
        for (unsigned i = 0; i < n_local; ++i) {
            const uint64_t k_hi = first_at_or_after(own_hi, i, g.hop, g.drain);
            if (k_hi > 0) need = std::max(need, needed_input(i, (k_hi - 1) * g.hop + g.n, g));
        }
        const uint64_t j_hi = first_at_or_after(own_hi, n_local, 1, g.drain);
        need = std::max(need, needed_input(n_local, j_hi, g));
        feed_hi = std::min(total, need);
    }
    // ---- how far back: the first owned segment / tail sample of every stage must be valid ----
    uint64_t feed_lo = 0;
    if (own_lo != 0) {
        uint64_t back = 64;
        for (unsigned q = 0; q < n_local; ++q) back *= 8;
        for (;;) {
            feed_lo = own_lo > back ? (own_lo - back) / 8 * 8 : 0;
            // per-stage first stream index free of warm-up contamination for a cascade seek()ed to feed_lo
            bool ok = true;
            uint64_t v = feed_lo;
            for (unsigned i = 0; i <= n_local; ++i) {
                const uint64_t first = i < n_local ? first_at_or_after(own_lo, i, g.hop, g.drain) * g.hop
                                                   : first_at_or_after(own_lo, n_local, 1, g.drain);
                if (first < v) ok = false;
                const uint64_t mv = (v + g.halo + 1) / 8;
                v = v == 0 ? 0 : (mv > g.drain ? mv - g.drain : 0);
            }
            if (ok || feed_lo == 0) break;
            back *= 2;
        }
    }
    out->own_lo = own_lo;
    out->own_hi = last ? NONE : own_hi;
    out->feed_lo = feed_lo;
    out->feed_hi = feed_hi;
    out->tail_lo = first_at_or_after(own_lo, n_local, 1, g.drain);
    out->tail_hi = last ? NONE : first_at_or_after(own_hi, n_local, 1, g.drain);
    out->n_local = n_local;
    out->_pad = 0;
}

uint32_t stage_avg_of(sspsd_avg_opts a, unsigned i)
{
    const unsigned sh = SSPSD_DEPTH * i;
    const uint32_t v = sh >= 32 ? 0u : (a.count >> sh);
    return std::min(v, a.limit);
}

uint32_t auto_n_local(uint64_t total, uint32_t world, const Geo& g)
{
    // largest K whose warm-up halo (8^K * 64 stage-0 samples) stays below 1/64 of a rank's chunk, at least 1 and
    // at most the number of stages the stream reaches minus one (the deepest stages see too few segments to cut)
    const uint64_t chunk = total / std::max<uint32_t>(world, 1);
    const size_t reach = stream_state(total, g).size();
    uint32_t k = 1;
    uint64_t halo = 64 * 8;
    while (k + 1 < reach && k < 8 && halo * 8 * 64 <= chunk) {
        halo *= 8;
        ++k;
    }
    return k;
}

// ---------------------------------------------------------------------------------------------
// device helpers of the exchange
// ---------------------------------------------------------------------------------------------
// buf[0 .. n_local*R*stride) = acc rows * factor[stage] (R rows of `stride` per stage); tail stream c (tail + c * pitch)
// at buf[tail_off + c * gap ..][0 .. tail_len); the rest of buf zero
__global__ void pack_exchange_kernel(double* __restrict__ buf, size_t size, const float* __restrict__ acc, uint32_t n_local,
                                     uint32_t R, size_t stride, const double* __restrict__ factor,
                                     const float* __restrict__ tail, uint32_t C, size_t pitch, size_t tail_off, size_t gap,
                                     size_t tail_len)
{
    const size_t per_stage = (size_t)R * stride, nacc = (size_t)n_local * per_stage;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < size; i += (size_t)gridDim.x * blockDim.x) {
        double v = 0.0;
        if (i < nacc) {
            v = (double)acc[i] * factor[i / per_stage];
        } else if (i >= tail_off) {
            const size_t c = (i - tail_off) / gap, j = (i - tail_off) % gap;
            if (c < C && j < tail_len) v = (double)tail[c * pitch + j];
        }
        buf[i] = v;
    }
}

// rows: buf[0 .. nacc) -> acc (float); the gathered tail slices of stream c -> tail_out[c * len ..][0 .. len), one
// contiguous float stream each (len = out_off[n_ranks]); stream c's slot of rank r is at slot_off[r] + c * gap
struct UnpackArgs {
    const double* buf;
    float* acc;
    size_t nacc;
    float* tail_out;
    uint32_t n_ranks, C;
    size_t gap;
    size_t slot_off[SSPSD_GROUP_MAX_RANKS];  // offset of rank r's slot of stream 0 in buf
    size_t out_off[SSPSD_GROUP_MAX_RANKS + 1];  // prefix sums of the slice lengths
};
__global__ void unpack_exchange_kernel(const UnpackArgs a)
{
    const size_t len = a.out_off[a.n_ranks], total = a.nacc + a.C * len;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        if (i < a.nacc) {
            a.acc[i] = (float)a.buf[i];
        } else {
            const size_t c = (i - a.nacc) / len, j = (i - a.nacc) % len;
            uint32_t r = 0;
            while (r + 1 < a.n_ranks && j >= a.out_off[r + 1]) ++r;
            a.tail_out[c * len + j] = (float)a.buf[a.slot_off[r] + c * a.gap + (j - a.out_off[r])];
        }
    }
}

// direct reduction on the root device: sums the ranks' accumulator rows through peer pointers (NVLink loads when
// the ranks are different GPUs, plain loads when several ranks share one), in fixed rank order and in f64, so the
// result is bit-reproducible from run to run
struct PeerRows {
    const float* acc[SSPSD_GROUP_MAX_RANKS];
    double factor[SSPSD_GROUP_MAX_RANKS][SSPSD_MAX_STAGES];
    uint32_t n_ranks, n_local, R;  // R rows of `stride` floats per stage
    size_t stride;
    float* out;
};
__global__ void peer_reduce_rows_kernel(const PeerRows a)
{
    const size_t per_stage = (size_t)a.R * a.stride, n = (size_t)a.n_local * per_stage;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const uint32_t st = (uint32_t)(i / per_stage);
        double s = 0.0;
        for (uint32_t r = 0; r < a.n_ranks; ++r) s += (double)a.acc[r][i] * a.factor[r][st];
        a.out[i] = (float)s;
    }
}

}  // namespace

// =============================================================================================
struct sspsd_group {
    int32_t mode = SSPSD_SHARD_CHANNELS;
    bool multi_process = false;
    uint32_t n_ranks = 1;
    uint32_t first_rank = 0;            // global rank of local index 0
    std::vector<int> devices;           // device of every LOCAL rank
    std::vector<ncclComm_t> comms;      // one per local rank (empty: no NCCL, direct peer path)
    sspsd_config cfg{};
    sspsd_avg_opts avg{0xffffffffu, 0xffffffffu};
    bool avg_set = false;
    int detrend = 0;
    int32_t reduce = SSPSD_REDUCE_NCCL;
    // channels: cascade of channel c (nullptr if another process owns it)
    std::vector<sspsd_cascade*> chan;
    // what the group computes: SSPSD_GROUP_PSD (cascades) or a cross kind (time chunks only)
    sspsd_group_kind kind{SSPSD_GROUP_PSD, 1, 0, 0};
    // time chunks: one cascade per local rank (kind PSD) ...
    std::vector<sspsd_cascade*> tc;
    // ... or one XCascade (CSD, CSM: owned; zoom: the ZoomCascade's) and, for the zoom kind, its ZoomCascade
    std::vector<XCascade*> xc;
    std::vector<ZoomCascade*> zc;
    std::vector<sspsd_time_chunk> plan;  // per GLOBAL rank
    uint64_t total = 0;
    uint32_t n_local_stages = 0;
    std::vector<uint64_t> fed;           // per local rank: samples fed so far
    bool finished = false;
    // exchange scratch per local rank
    std::vector<double*> d_buf;
    std::vector<float*> d_tail;
    std::vector<double*> d_factor;
    std::vector<size_t> buf_cap, tail_cap;
    float* d_tail_all = nullptr;
    size_t tail_all_cap = 0;
    // channel gather scratch
    uint8_t* d_rec = nullptr;
    uint8_t* d_all = nullptr;
    uint8_t* h_all = nullptr;
    size_t rec_cap = 0, all_cap = 0;
    cudaStream_t gather_stream = nullptr;
    // SSPSD_GROUP_TRACE=1: host seconds spent in the phases of sspsd_group_psd_all, printed when the group is destroyed
    cudaEvent_t ev_chan = nullptr;
    uint64_t* h_book = nullptr;  // pinned
    size_t book_cap = 0;
    bool trace = false;
    double t_wait = 0, t_pack = 0, t_gather = 0, t_d2h = 0, t_merge = 0;
    uint64_t n_readouts = 0;
    std::vector<sspsd_source*> noise_src;  // per local rank, for sspsd_group_time_process_noise
    int64_t noise_exp = 0;
    uint64_t noise_seed = 0;
    std::vector<sspsd_plant*> plants;  // per local rank, for sspsd_group_time_process_plant
    std::vector<uint8_t> plant_key;    // the spec they were made from (k, m, taps_len, taps, inputs)

    uint32_t n_local() const { return (uint32_t)devices.size(); }
    bool cross() const { return kind.kind != SSPSD_GROUP_PSD; }
    // streams a rank is fed: PSD 1, CSD 2, CSM k, zoom I/Q 2, zoom heterodyne 1
    uint32_t n_inputs() const
    {
        if (kind.kind == SSPSD_GROUP_ZOOM) return kind.zoom_mode == SSPSD_ZOOM_IQ ? 2 : 1;
        return (uint32_t)kind.channels;
    }
    bool is_root() const { return first_rank == 0; }
    int local_of(uint32_t rank) const
    {
        return rank >= first_rank && rank < first_rank + n_local() ? (int)(rank - first_rank) : -1;
    }
};

namespace {

Geo geo_of(const sspsd_config& cfg)
{
    uint32_t drain = 0, halo = 0;
    sspsd::hbf_info(cfg.hbf, &drain, &halo);
    const uint64_t n = cfg.n_fft;
    const uint64_t overlap = cfg.window == SSPSD_WINDOW_HANN ? n / 2 : 0;
    return {n, n - overlap, drain, halo};
}

int create_common(const sspsd_config* cfg, int32_t mode, sspsd_group** out, sspsd_group** gp)
{
    if (!cfg || !out) {
        set_error("null argument");
        return SSPSD_EINVAL;
    }
    *out = nullptr;
    if (mode != SSPSD_SHARD_CHANNELS && mode != SSPSD_SHARD_TIME) {
        set_error("unknown shard mode");
        return SSPSD_EINVAL;
    }
    sspsd_group* g = new (std::nothrow) sspsd_group();
    if (!g) return SSPSD_ENOMEM;
    g->cfg = *cfg;
    g->cfg.stream = nullptr;  // every handle of a group owns its stream
    g->mode = mode;
    g->trace = getenv("SSPSD_GROUP_TRACE") != nullptr;
    *gp = g;
    return SSPSD_OK;
}

int make_cascade(sspsd_group* g, int device, sspsd_cascade** out)
{
    sspsd_config c = g->cfg;
    c.device = device;
    int rc = sspsd_cascade_create(&c, out);
    if (rc) return rc;
    if (g->avg_set) rc = (*out)->c.set_avg(g->avg);
    if (!rc && g->detrend) rc = (*out)->c.set_detrend(g->detrend);
    if (rc) {
        sspsd_cascade_destroy(*out);
        *out = nullptr;
    }
    return rc;
}

// the handle of a cross kind on `device`: *x its XCascade, *z its ZoomCascade (zoom kind) or nullptr
int make_xrank(sspsd_group* g, int device, XCascade** x, ZoomCascade** z)
{
    sspsd_config c = g->cfg;
    c.device = device;
    *x = nullptr;
    *z = nullptr;
    int rc;
    if (g->kind.kind == SSPSD_GROUP_ZOOM) {
        *z = new (std::nothrow) ZoomCascade();
        if (!*z) return SSPSD_ENOMEM;
        rc = (*z)->init(c, g->kind.zoom_mode, g->kind.ftw);
        *x = &(*z)->x();
    } else {
        *x = new (std::nothrow) XCascade();
        if (!*x) return SSPSD_ENOMEM;
        rc = (*x)->init(c, g->kind.channels);
    }
    if (!rc && g->avg_set) rc = (*x)->set_avg(g->avg);
    if (!rc && g->detrend) rc = (*x)->set_detrend(g->detrend);
    return rc;
}

void destroy_xrank(XCascade* x, ZoomCascade* z)
{
    if (z)
        delete z;
    else
        delete x;
}

int ensure_time_cascades(sspsd_group* g)
{
    if (!g->tc.empty() || !g->xc.empty()) return SSPSD_OK;
    const uint32_t nl = g->n_local();
    if (g->cross()) {
        std::vector<XCascade*> xc(nl, nullptr);
        std::vector<ZoomCascade*> zc(nl, nullptr);
        for (uint32_t l = 0; l < nl; ++l) {
            int rc = make_xrank(g, g->devices[l], &xc[l], &zc[l]);
            if (rc) {
                for (uint32_t m = 0; m <= l; ++m) destroy_xrank(xc[m], zc[m]);  // all or nothing, as below
                return rc;
            }
        }
        g->xc = xc;
        if (g->kind.kind == SSPSD_GROUP_ZOOM) g->zc = zc;
    } else {
        std::vector<sspsd_cascade*> tc(nl, nullptr);
        for (uint32_t l = 0; l < nl; ++l) {
            int rc = make_cascade(g, g->devices[l], &tc[l]);
            if (rc) {
                // all or nothing: a half-built set would pass the "already made" test above on the next call
                for (auto* c : tc) sspsd_cascade_destroy(c);
                return rc;
            }
        }
        g->tc = tc;
    }
    g->fed.assign(nl, 0);
    g->d_buf.assign(nl, nullptr);
    g->d_tail.assign(nl, nullptr);
    g->d_factor.assign(nl, nullptr);
    g->buf_cap.assign(nl, 0);
    g->tail_cap.assign(nl, 0);
    return SSPSD_OK;
}

// a kind is valid for a group of shard mode `mode` and FFT size n: *out is the kind with its channel count filled in
int check_kind(const sspsd_group_kind* k, int32_t mode, uint32_t n, sspsd_group_kind* out)
{
    if (!k) {
        set_error("null argument");
        return SSPSD_EINVAL;
    }
    sspsd_group_kind v = *k;
    switch (v.kind) {
    case SSPSD_GROUP_PSD:
        if (v.channels == 0) v.channels = 1;
        if (v.channels != 1 || v.zoom_mode || v.ftw) {
            set_error("a PSD group has one channel and no carrier");
            return SSPSD_EINVAL;
        }
        break;
    case SSPSD_GROUP_CSD:
    case SSPSD_GROUP_ZOOM:
        if (v.channels == 0) v.channels = 2;
        if (v.channels != 2) {
            set_error("CSD and zoom groups have two channels");
            return SSPSD_EINVAL;
        }
        if (v.kind == SSPSD_GROUP_CSD && (v.zoom_mode || v.ftw)) {
            set_error("a CSD group has no carrier");
            return SSPSD_EINVAL;
        }
        if (v.kind == SSPSD_GROUP_ZOOM && v.zoom_mode != SSPSD_ZOOM_IQ && v.zoom_mode != SSPSD_ZOOM_HETERODYNE) {
            set_error("unknown zoom mode");
            return SSPSD_EINVAL;
        }
        if (v.kind == SSPSD_GROUP_ZOOM && v.zoom_mode == SSPSD_ZOOM_IQ && v.ftw) {
            set_error("I/Q mode has no carrier: ftw must be 0");
            return SSPSD_EINVAL;
        }
        break;
    case SSPSD_GROUP_CSM:
        if (v.channels < 2 || v.channels > 4 || v.zoom_mode || v.ftw) {
            set_error("a CSM group has 2 .. 4 channels and no carrier");
            return SSPSD_EINVAL;
        }
        break;
    default:
        set_error("unknown group kind");
        return SSPSD_EINVAL;
    }
    if (v.kind != SSPSD_GROUP_PSD) {
        if (mode != SSPSD_SHARD_TIME) {
            // every transform of a cross-spectrum is shared by its channels: they cannot live on different GPUs
            set_error("cross-spectral groups are time-chunked only (SSPSD_SHARD_TIME)");
            return SSPSD_EINVAL;
        }
        if (n < 64 || n > 4096 || (n & (n - 1))) {
            set_error("cross-spectral groups support n_fft = 64 .. 4096");
            return SSPSD_EINVAL;
        }
    }
    *out = v;
    return SSPSD_OK;
}

// the zoom handle of a local rank takes the rank's input in its own mode; the others take all streams at once
int process_rank(sspsd_group* g, uint32_t l, const float* const* x, size_t n, int32_t mem)
{
    if (g->kind.kind == SSPSD_GROUP_PSD) return g->tc[l]->c.process(x[0], n, mem);
    if (g->kind.kind != SSPSD_GROUP_ZOOM) return g->xc[l]->process(x, n, mem);
    if (g->kind.zoom_mode == SSPSD_ZOOM_IQ) return g->zc[l]->process_iq(x[0], x[1], n, mem);
    return g->zc[l]->process(x[0], n, mem);
}

int wrong_kind(const char* what)
{
    set_error(what);
    return SSPSD_EINVAL;
}

}  // namespace

extern "C" {

// pure host planner (exported so that callers and tests can see exactly what a rank will be fed)
int32_t sspsd_time_plan(uint32_t n_fft, int32_t window, int32_t hbf, uint64_t total, uint32_t n_ranks, uint32_t rank,
                        uint32_t n_local_stages, sspsd_time_chunk* out)
{
    if (!out || n_ranks == 0 || rank >= n_ranks || n_local_stages > SSPSD_MAX_STAGES - 1 || n_fft < 16 || (n_fft & (n_fft - 1))) {
        set_error("bad argument");
        return SSPSD_EINVAL;
    }
    sspsd_config cfg{};
    cfg.n_fft = n_fft;
    cfg.window = window;
    cfg.hbf = hbf;
    uint32_t d = 0, h = 0;
    if (sspsd::hbf_info(hbf, &d, &h)) {
        set_error("unknown half-band preset");
        return SSPSD_EINVAL;
    }
    const Geo g = geo_of(cfg);
    if (n_local_stages == 0) n_local_stages = auto_n_local(total, n_ranks, g);
    plan_rank(total, n_ranks, rank, g, n_local_stages, out);
    return SSPSD_OK;
}

int32_t sspsd_group_create(const sspsd_config* cfg, const int32_t* devices, uint32_t n_devices, int32_t shard_mode,
                           sspsd_group** out)
{
    sspsd_group* g = nullptr;
    int rc = create_common(cfg, shard_mode, out, &g);
    if (rc) return rc;
    if (!devices || n_devices == 0 || n_devices > SSPSD_GROUP_MAX_RANKS) {
        set_error("bad device list");
        delete g;
        return SSPSD_EINVAL;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        set_error("no CUDA device: this library has no CPU fallback");
        delete g;
        return SSPSD_ECUDA;
    }
    bool distinct = true;
    for (uint32_t i = 0; i < n_devices; ++i) {
        if (devices[i] < 0 || devices[i] >= ndev) {
            set_error("bad device ordinal");
            delete g;
            return SSPSD_EINVAL;
        }
        for (uint32_t j = 0; j < i; ++j)
            if (devices[j] == devices[i]) distinct = false;
        g->devices.push_back(devices[i]);
    }
    g->n_ranks = n_devices;
    g->first_rank = 0;
    // Ranks that share a GPU (a single-GPU box playing several ranks) cannot form an NCCL communicator; they are
    // reduced by direct loads, which also serves distinct GPUs through peer access (SSPSD_REDUCE_P2P).
    g->reduce = distinct && n_devices > 1 ? SSPSD_REDUCE_NCCL : SSPSD_REDUCE_P2P;
    if (const char* e = getenv("SSPSD_GROUP_REDUCE")) {
        if (!strcmp(e, "p2p")) g->reduce = SSPSD_REDUCE_P2P;
    }
    if (shard_mode == SSPSD_SHARD_TIME && n_devices > 1) {
        if (g->reduce == SSPSD_REDUCE_NCCL) {
            if (!nccl().ok) {
                set_error("libnccl.so.2 could not be loaded");
                delete g;
                return SSPSD_ENCCL;
            }
            g->comms.assign(n_devices, nullptr);
            if (!nccl_ok(nccl().CommInitAll(g->comms.data(), (int)n_devices, g->devices.data()), "ncclCommInitAll")) {
                g->comms.clear();
                delete g;
                return SSPSD_ENCCL;
            }
        } else {
            // root reads the peers' accumulators in place
            DevGuard dg(g->devices[0]);
            for (uint32_t i = 1; i < n_devices; ++i) {
                if (g->devices[i] == g->devices[0]) continue;
                int can = 0;
                cudaDeviceCanAccessPeer(&can, g->devices[0], g->devices[i]);
                if (!can) {
                    set_error("no peer access between the group's devices");
                    delete g;
                    return SSPSD_ECUDA;
                }
                cudaError_t e = cudaDeviceEnablePeerAccess(g->devices[i], 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
                    sspsd::cuda_ok(e, "cudaDeviceEnablePeerAccess");
                    delete g;
                    return SSPSD_ECUDA;
                }
                cudaGetLastError();
            }
        }
    }
    *out = g;
    return SSPSD_OK;
}

int32_t sspsd_group_unique_id(uint8_t id[SSPSD_GROUP_ID_BYTES])
{
    static_assert(SSPSD_GROUP_ID_BYTES == NCCL_UNIQUE_ID_BYTES, "id size");
    if (!id) return SSPSD_EINVAL;
    if (!nccl().ok) {
        set_error("libnccl.so.2 could not be loaded");
        return SSPSD_ENCCL;
    }
    ncclUniqueId u;
    SSPSD_NCCL(nccl().GetUniqueId(&u));
    std::memcpy(id, u.internal, SSPSD_GROUP_ID_BYTES);
    return SSPSD_OK;
}

int32_t sspsd_group_create_rank(const sspsd_config* cfg, const uint8_t id[SSPSD_GROUP_ID_BYTES], uint32_t rank,
                                uint32_t n_ranks, int32_t shard_mode, sspsd_group** out)
{
    sspsd_group* g = nullptr;
    int rc = create_common(cfg, shard_mode, out, &g);
    if (rc) return rc;
    if (n_ranks == 0 || n_ranks > SSPSD_GROUP_MAX_RANKS || rank >= n_ranks || (n_ranks > 1 && !id)) {
        set_error("bad rank / world size");
        delete g;
        return SSPSD_EINVAL;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        set_error("no CUDA device: this library has no CPU fallback");
        delete g;
        return SSPSD_ECUDA;
    }
    if (cfg->device < 0 || cfg->device >= ndev) {
        set_error("bad device ordinal");
        delete g;
        return SSPSD_EINVAL;
    }
    g->multi_process = true;
    g->cfg.stream = cfg->stream;  // one rank, one device: the caller may order the rank's work on its own stream
    g->n_ranks = n_ranks;
    g->first_rank = rank;
    g->devices.push_back(cfg->device);
    g->reduce = SSPSD_REDUCE_NCCL;
    if (n_ranks > 1) {
        if (!nccl().ok) {
            set_error("libnccl.so.2 could not be loaded");
            delete g;
            return SSPSD_ENCCL;
        }
        DevGuard dg(cfg->device);
        ncclUniqueId u;
        std::memcpy(u.internal, id, SSPSD_GROUP_ID_BYTES);
        g->comms.assign(1, nullptr);
        if (!nccl_ok(nccl().CommInitRank(&g->comms[0], (int)n_ranks, u, (int)rank), "ncclCommInitRank")) {
            g->comms.clear();
            delete g;
            return SSPSD_ENCCL;
        }
    }
    *out = g;
    return SSPSD_OK;
}

int32_t sspsd_group_create_kind(const sspsd_config* cfg, const sspsd_group_kind* kind, const int32_t* devices,
                                uint32_t n_devices, int32_t shard_mode, sspsd_group** out)
{
    if (out) *out = nullptr;
    sspsd_group_kind k{};
    if (!cfg || !out) {
        set_error("null argument");
        return SSPSD_EINVAL;
    }
    int rc = check_kind(kind, shard_mode, cfg->n_fft, &k);
    if (rc) return rc;
    rc = sspsd_group_create(cfg, devices, n_devices, shard_mode, out);
    if (rc) return rc;
    (*out)->kind = k;
    return SSPSD_OK;
}

int32_t sspsd_group_create_kind_rank(const sspsd_config* cfg, const sspsd_group_kind* kind,
                                     const uint8_t id[SSPSD_GROUP_ID_BYTES], uint32_t rank, uint32_t n_ranks,
                                     int32_t shard_mode, sspsd_group** out)
{
    if (out) *out = nullptr;
    sspsd_group_kind k{};
    if (!cfg || !out) {
        set_error("null argument");
        return SSPSD_EINVAL;
    }
    int rc = check_kind(kind, shard_mode, cfg->n_fft, &k);
    if (rc) return rc;
    rc = sspsd_group_create_rank(cfg, id, rank, n_ranks, shard_mode, out);
    if (rc) return rc;
    (*out)->kind = k;
    return SSPSD_OK;
}

int32_t sspsd_group_kind_of(const sspsd_group* g, sspsd_group_kind* out)
{
    if (!g || !out) return SSPSD_EINVAL;
    *out = g->kind;
    return SSPSD_OK;
}

void sspsd_group_destroy(sspsd_group* g)
{
    if (!g) return;
    if (g->trace && g->n_readouts)
        fprintf(stderr, "[sspsd_group rank %u] psd_all x%llu: wait %.1f us, pack %.1f us, gather %.1f us, d2h %.1f us, merge %.1f us per call\n",
                g->first_rank, (unsigned long long)g->n_readouts, 1e6 * g->t_wait / g->n_readouts, 1e6 * g->t_pack / g->n_readouts,
                1e6 * g->t_gather / g->n_readouts, 1e6 * g->t_d2h / g->n_readouts, 1e6 * g->t_merge / g->n_readouts);
    for (auto* s : g->noise_src) sspsd_source_destroy(s);
    for (auto* p : g->plants) sspsd_plant_destroy(p);
    for (auto* c : g->chan) sspsd_cascade_destroy(c);
    for (auto* c : g->tc) sspsd_cascade_destroy(c);
    for (size_t l = 0; l < g->xc.size(); ++l) destroy_xrank(g->xc[l], g->zc.empty() ? nullptr : g->zc[l]);
    for (uint32_t l = 0; l < g->d_buf.size(); ++l) {
        DevGuard dg(g->devices[l]);
        cudaFree(g->d_buf[l]);
        cudaFree(g->d_tail[l]);
        cudaFree(g->d_factor[l]);
    }
    if (!g->devices.empty()) {
        DevGuard dg(g->devices[0]);
        cudaFree(g->d_tail_all);
        cudaFree(g->d_rec);
        cudaFree(g->d_all);
        if (g->h_all) cudaFreeHost(g->h_all);
        if (g->gather_stream) cudaStreamDestroy(g->gather_stream);
        if (g->ev_chan) cudaEventDestroy(g->ev_chan);
        if (g->h_book) cudaFreeHost(g->h_book);
    }
    for (uint32_t l = 0; l < g->comms.size(); ++l)
        if (g->comms[l]) nccl().CommDestroy(g->comms[l]);
    delete g;
}

int32_t sspsd_group_info(const sspsd_group* g, uint32_t* n_ranks, uint32_t* first_rank, uint32_t* n_local_ranks,
                         int32_t* shard_mode, int32_t* reduce)
{
    if (!g) return SSPSD_EINVAL;
    if (n_ranks) *n_ranks = g->n_ranks;
    if (first_rank) *first_rank = g->first_rank;
    if (n_local_ranks) *n_local_ranks = g->n_local();
    if (shard_mode) *shard_mode = g->mode;
    if (reduce) *reduce = g->comms.empty() ? SSPSD_REDUCE_P2P : SSPSD_REDUCE_NCCL;
    return SSPSD_OK;
}

int32_t sspsd_group_set_avg(sspsd_group* g, sspsd_avg_opts avg)
{
    if (!g) return SSPSD_EINVAL;
    g->avg = avg;
    g->avg_set = true;
    for (auto* c : g->chan)
        if (c) {
            int rc = c->c.set_avg(avg);
            if (rc) return rc;
        }
    for (size_t l = 0; l < g->tc.size(); ++l)
        if (g->tc[l]) {
            if (g->total && g->fed[l]) {
                set_error("time-chunked mode: options must be set before the first sample");
                return SSPSD_EINVAL;
            }
            int rc = g->tc[l]->c.set_avg(avg);
            if (rc) return rc;
        }
    for (size_t l = 0; l < g->xc.size(); ++l) {
        if (g->total && g->fed[l]) {
            set_error("time-chunked mode: options must be set before the first sample");
            return SSPSD_EINVAL;
        }
        int rc = g->xc[l]->set_avg(avg);
        if (rc) return rc;
    }
    return SSPSD_OK;
}

int32_t sspsd_group_set_detrend(sspsd_group* g, int32_t d)
{
    if (!g) return SSPSD_EINVAL;
    if (d == SSPSD_DETREND_LINEAR) {
        set_error("Detrend::Linear is unimplemented!() in the reference (src/psd.rs:110)");
        return SSPSD_EUNIMPLEMENTED;
    }
    if (d < 0 || d > SSPSD_DETREND_LINEAR) {
        set_error("unknown detrend");
        return SSPSD_EINVAL;
    }
    g->detrend = d;
    for (auto* c : g->chan)
        if (c) {
            int rc = c->c.set_detrend(d);
            if (rc) return rc;
        }
    for (auto* c : g->tc)
        if (c) {
            int rc = c->c.set_detrend(d);
            if (rc) return rc;
        }
    for (auto* x : g->xc) {
        int rc = x->set_detrend(d);
        if (rc) return rc;
    }
    return SSPSD_OK;
}

// ---------------------------------------------------------------------------------------------
// channels
// ---------------------------------------------------------------------------------------------
int32_t sspsd_group_process_f32(sspsd_group* g, uint32_t channel, const float* x, size_t n, int32_t mem)
{
    if (!g || g->mode != SSPSD_SHARD_CHANNELS) {
        set_error("not a channel-sharded group");
        return SSPSD_EINVAL;
    }
    if (channel >= 65536) {
        set_error("channel index too large");
        return SSPSD_EINVAL;
    }
    const int l = g->local_of(channel % g->n_ranks);
    if (g->chan.size() <= channel) g->chan.resize(channel + 1, nullptr);
    if (l < 0) return SSPSD_OK;  // another process owns this channel: every process can run the same loop over all traces
    if (!g->chan[channel]) {
        int rc = make_cascade(g, g->devices[l], &g->chan[channel]);
        if (rc) return rc;
    }
    return g->chan[channel]->c.process(x, n, mem);
}

int32_t sspsd_group_channel_device(const sspsd_group* g, uint32_t channel, int32_t* device, uint32_t* rank)
{
    if (!g || g->mode != SSPSD_SHARD_CHANNELS) return SSPSD_EINVAL;
    const uint32_t r = channel % g->n_ranks;
    if (rank) *rank = r;
    const int l = g->local_of(r);
    if (device) *device = l >= 0 ? g->devices[l] : -1;
    return SSPSD_OK;
}

int32_t sspsd_group_channel_handle(sspsd_group* g, uint32_t channel, sspsd_cascade** out)
{
    if (!g || !out || g->mode != SSPSD_SHARD_CHANNELS) return SSPSD_EINVAL;
    *out = channel < g->chan.size() ? g->chan[channel] : nullptr;
    return SSPSD_OK;
}

int32_t sspsd_group_sync(sspsd_group* g)
{
    if (!g) return SSPSD_EINVAL;
    for (auto* c : g->chan)
        if (c) {
            int rc = c->c.flush();
            if (rc) return rc;
        }
    for (auto* c : g->chan)
        if (c) {
            int rc = c->c.sync();
            if (rc) return rc;
        }
    for (auto* c : g->tc)
        if (c) {
            int rc = c->c.sync();
            if (rc) return rc;
        }
    for (size_t l = 0; l < g->xc.size(); ++l) {
        int rc = g->zc.empty() ? g->xc[l]->sync() : g->zc[l]->sync();
        if (rc) return rc;
    }
    return SSPSD_OK;
}

int32_t sspsd_group_psd(sspsd_group* g, uint32_t channel, const sspsd_merge_opts* opts, float* p, size_t* p_len,
                        sspsd_break* b, size_t* b_len)
{
    if (!g || !p_len || !b_len) return SSPSD_EINVAL;
    if (g->cross()) return wrong_kind("a cross-spectral group reads out with sspsd_group_csd_read / _csm_read / _zoom_read");
    sspsd_merge_opts o{0, 1, 0};
    if (opts) o = *opts;
    if (g->mode == SSPSD_SHARD_TIME) {
        if (!g->finished) {
            set_error("time-chunked group: call sspsd_group_time_finish first");
            return SSPSD_EINVAL;
        }
        if (!g->is_root()) {
            *p_len = 0;
            *b_len = 0;
            return SSPSD_OK;
        }
        return g->tc[0]->c.psd(o, p, p_len, b, b_len);
    }
    if (g->multi_process && g->n_ranks > 1) {
        set_error("multi-process channel groups read out with sspsd_group_psd_all (one collective for all channels)");
        return SSPSD_EINVAL;
    }
    if (channel >= g->chan.size() || !g->chan[channel]) {
        *p_len = 0;
        *b_len = 0;
        return SSPSD_OK;  // a channel that never received a sample: PsdCascade::default().psd() is empty
    }
    return g->chan[channel]->c.psd(o, p, p_len, b, b_len);
}

// One record per channel: [SSPSD_MAX_STAGES rows of stride floats][SSPSD_MAX_STAGES x (L, craw, count, avg) u64][n_stages u64]
int32_t sspsd_group_psd_all(sspsd_group* g, uint32_t n_channels, const sspsd_merge_opts* opts, float* p, size_t p_stride,
                            size_t* p_lens, sspsd_break* b, size_t b_stride, size_t* b_lens)
{
    if (!g || g->mode != SSPSD_SHARD_CHANNELS || !p_lens || !b_lens || n_channels == 0) {
        set_error("bad argument");
        return SSPSD_EINVAL;
    }
    sspsd_merge_opts o{0, 1, 0};
    if (opts) o = *opts;
    if (g->chan.size() < n_channels) g->chan.resize(n_channels, nullptr);
    const bool collective = g->multi_process && g->n_ranks > 1;
    if (!collective) {
        // all channels live in this process: launch everything first, then read out one by one
        for (uint32_t c = 0; c < n_channels; ++c)
            if (g->chan[c]) {
                int rc = g->chan[c]->c.flush();
                if (rc) return rc;
            }
        for (uint32_t c = 0; c < n_channels; ++c) {
            size_t pl = p_stride, bl = b_stride;
            if (!g->chan[c]) {
                p_lens[c] = b_lens[c] = 0;
                continue;
            }
            int rc = g->chan[c]->c.psd(o, p + (size_t)c * p_stride, &pl, b + (size_t)c * b_stride, &bl);
            p_lens[c] = pl;
            b_lens[c] = bl;
            if (rc) return rc;
        }
        return SSPSD_OK;
    }
    // ---- one process per rank: ONE ncclAllGather of every rank's channel records, merged on rank 0 ----
    const uint32_t per_rank = (n_channels + g->n_ranks - 1) / g->n_ranks;
    const size_t stride = ((size_t)g->cfg.n_fft / 2 + 1 + 63) & ~(size_t)63;
    const size_t rec = ((size_t)SSPSD_MAX_STAGES * stride * sizeof(float) + (SSPSD_MAX_STAGES * 4 + 2) * sizeof(uint64_t) + 255) &
                       ~(size_t)255;
    const size_t mine = rec * per_rank, all = mine * g->n_ranks;
    DevGuard dg(g->devices[0]);
    if (!dg.ok) return SSPSD_ECUDA;
    if (mine > g->rec_cap || all > g->all_cap) {
        cudaFree(g->d_rec);
        cudaFree(g->d_all);
        if (g->h_all) cudaFreeHost(g->h_all);
        g->d_rec = g->d_all = g->h_all = nullptr;
        SSPSD_CUDA(cudaMalloc(&g->d_rec, mine));
        SSPSD_CUDA(cudaMalloc(&g->d_all, all));
        SSPSD_CUDA(cudaMallocHost(&g->h_all, std::max(all, mine)));
        g->rec_cap = mine;
        g->all_cap = all;
    }
    if (!g->gather_stream) SSPSD_CUDA(cudaStreamCreateWithFlags(&g->gather_stream, cudaStreamNonBlocking));
    cudaStream_t s = g->gather_stream;
    // Nothing below waits on the host until the very end: the pack, the collective and the read-back are queued
    // behind an event on each channel's stream, so they start the moment the GPU finishes the channel's work
    // (a host synchronisation here would put two launch latencies on the critical path of every readout).
    double t0 = g->trace ? now_s() : 0;
    if (!g->ev_chan) SSPSD_CUDA(cudaEventCreateWithFlags(&g->ev_chan, cudaEventDisableTiming));
    const size_t book_words = SSPSD_MAX_STAGES * 4 + 2;
    if (!g->h_book || g->book_cap < per_rank) {
        if (g->h_book) cudaFreeHost(g->h_book);
        g->h_book = nullptr;
        SSPSD_CUDA(cudaMallocHost(&g->h_book, (size_t)per_rank * book_words * sizeof(uint64_t)));
        g->book_cap = per_rank;
    }
    double t1 = t0;
    SSPSD_CUDA(cudaMemsetAsync(g->d_rec, 0, mine, s));
    for (uint32_t k = 0; k < per_rank; ++k) {
        const uint32_t c = g->first_rank + k * g->n_ranks;
        if (c >= n_channels || !g->chan[c]) continue;
        Cascade& cs = g->chan[c]->c;
        int rc = cs.fence(g->ev_chan);  // launches what is staged, joins the handle's side streams, records the event
        if (rc) return rc;
        SSPSD_CUDA(cudaStreamWaitEvent(s, g->ev_chan, 0));
        sspsd_partials pa;
        rc = cs.partials(&pa);
        if (rc) return rc;
        uint8_t* dst = g->d_rec + (size_t)k * rec;
        SSPSD_CUDA(cudaMemcpyAsync(dst, pa.acc, (size_t)SSPSD_MAX_STAGES * stride * sizeof(float), cudaMemcpyDeviceToDevice, s));
        uint64_t* bk = g->h_book + (size_t)k * book_words;  // pinned: the bookkeeping is closed-form on the host
        cs.export_book(bk);
        SSPSD_CUDA(cudaMemcpyAsync(dst + (size_t)SSPSD_MAX_STAGES * stride * sizeof(float), bk, book_words * sizeof(uint64_t),
                                   cudaMemcpyHostToDevice, s));
    }
    double t2 = g->trace ? now_s() : 0;
    SSPSD_NCCL(nccl().AllGather(g->d_rec, g->d_all, mine, ncclUint8, g->comms[0], s));
    if (!g->is_root()) {
        SSPSD_CUDA(cudaStreamSynchronize(s));
        if (g->trace) {
            g->t_wait += t1 - t0;
            g->t_pack += t2 - t1;
            g->t_gather += now_s() - t2;
            g->n_readouts++;
        }
        for (uint32_t c = 0; c < n_channels; ++c) p_lens[c] = b_lens[c] = 0;
        return SSPSD_OK;
    }
    double t3 = 0;
    if (g->trace) {
        SSPSD_CUDA(cudaStreamSynchronize(s));
        t3 = now_s();
    }
    SSPSD_CUDA(cudaMemcpyAsync(g->h_all, g->d_all, all, cudaMemcpyDeviceToHost, s));
    SSPSD_CUDA(cudaStreamSynchronize(s));
    double t4 = g->trace ? now_s() : 0;
    for (uint32_t c = 0; c < n_channels; ++c) {
        const uint32_t r = c % g->n_ranks, k = c / g->n_ranks;
        const uint8_t* src = g->h_all + (size_t)r * mine + (size_t)k * rec;
        const float* rows = reinterpret_cast<const float*>(src);
        const uint64_t* bk = reinterpret_cast<const uint64_t*>(src + (size_t)SSPSD_MAX_STAGES * stride * sizeof(float));
        size_t pl = p_stride, bl = b_stride;
        int rc = Cascade::merge_host(g->cfg, bk, rows, stride, o, p ? p + (size_t)c * p_stride : nullptr, &pl,
                                     b ? b + (size_t)c * b_stride : nullptr, &bl);
        p_lens[c] = pl;
        b_lens[c] = bl;
        if (rc) return rc;
    }
    if (g->trace) {
        g->t_wait += t1 - t0;
        g->t_pack += t2 - t1;
        g->t_gather += t3 - t2;
        g->t_d2h += t4 - t3;
        g->t_merge += now_s() - t4;
        g->n_readouts++;
    }
    return SSPSD_OK;
}

// ---------------------------------------------------------------------------------------------
// time chunks of one stream
// ---------------------------------------------------------------------------------------------
int32_t sspsd_group_time_plan(sspsd_group* g, uint64_t total, uint32_t n_local_stages)
{
    if (!g || g->mode != SSPSD_SHARD_TIME) {
        set_error("not a time-chunked group");
        return SSPSD_EINVAL;
    }
    if (total == 0 || n_local_stages > SSPSD_MAX_STAGES - 1) {
        set_error("bad argument");
        return SSPSD_EINVAL;
    }
    const Geo geo = geo_of(g->cfg);
    if (n_local_stages == 0) n_local_stages = auto_n_local(total, g->n_ranks, geo);
    // a previous capture's handles are reset and reused (their device buffers stay allocated)
    int rc = ensure_time_cascades(g);
    if (rc) return rc;
    for (auto* c : g->tc) {
        rc = c->c.reset();
        if (rc) return rc;
    }
    for (size_t l = 0; l < g->xc.size(); ++l) {
        rc = g->zc.empty() ? g->xc[l]->reset() : g->zc[l]->reset();
        if (rc) return rc;
    }
    g->total = total;
    g->n_local_stages = n_local_stages;
    g->finished = false;
    g->plan.assign(g->n_ranks, sspsd_time_chunk{});
    for (uint32_t r = 0; r < g->n_ranks; ++r) plan_rank(total, g->n_ranks, r, geo, n_local_stages, &g->plan[r]);
    for (uint32_t l = 0; l < g->n_local(); ++l) {
        const sspsd_time_chunk& pl = g->plan[g->first_rank + l];
        if (g->cross()) {
            // the zoom kind's mixer starts at the rank's absolute position: phi_n = (n ftw) mod 2^32 of the whole stream
            rc = g->zc.empty() ? g->xc[l]->seek(pl.feed_lo) : g->zc[l]->seek(pl.feed_lo);
            if (rc) return rc;
            rc = g->xc[l]->set_window(pl.own_lo, pl.own_hi, n_local_stages);
        } else {
            Cascade& c = g->tc[l]->c;
            rc = c.seek(pl.feed_lo);
            if (rc) return rc;
            rc = c.set_window(pl.own_lo, pl.own_hi, n_local_stages);
        }
        if (rc) return rc;
        g->fed[l] = 0;
    }
    return SSPSD_OK;
}

int32_t sspsd_group_time_chunk(const sspsd_group* g, uint32_t rank, sspsd_time_chunk* out)
{
    if (!g || !out || g->mode != SSPSD_SHARD_TIME || rank >= g->plan.size()) {
        set_error("no plan (call sspsd_group_time_plan first)");
        return SSPSD_EINVAL;
    }
    *out = g->plan[rank];
    return SSPSD_OK;
}

int32_t sspsd_group_time_process_multi_f32(sspsd_group* g, uint32_t rank, const float* const* x, size_t n, int32_t mem)
{
    if (!g || g->mode != SSPSD_SHARD_TIME || g->plan.empty()) {
        set_error("no plan (call sspsd_group_time_plan first)");
        return SSPSD_EINVAL;
    }
    const int l = g->local_of(rank);
    if (l < 0) return SSPSD_OK;  // another process feeds that rank
    const sspsd_time_chunk& pl = g->plan[rank];
    if (g->fed[l] + n > pl.feed_hi - pl.feed_lo) {
        set_error("more samples than the rank's range [feed_lo, feed_hi)");
        return SSPSD_EINVAL;
    }
    if (n && !x) {
        set_error("null input");
        return SSPSD_EINVAL;
    }
    for (uint32_t i = 0; n && i < g->n_inputs(); ++i)
        if (!x[i]) {
            set_error("null input");
            return SSPSD_EINVAL;
        }
    int rc = n ? process_rank(g, (uint32_t)l, x, n, mem) : SSPSD_OK;
    if (rc) return rc;
    g->fed[l] += n;
    return SSPSD_OK;
}

int32_t sspsd_group_time_process_f32(sspsd_group* g, uint32_t rank, const float* x, size_t n, int32_t mem)
{
    if (g && g->cross()) return wrong_kind("a cross-spectral group takes sspsd_group_time_process_multi_f32");
    return sspsd_group_time_process_multi_f32(g, rank, &x, n, mem);
}

int32_t sspsd_group_time_process_all_multi_f32(sspsd_group* g, const float* const* x, size_t n)
{
    if (!g || g->mode != SSPSD_SHARD_TIME || g->plan.empty() || g->multi_process) {
        set_error("needs a planned single-process time-chunked group");
        return SSPSD_EINVAL;
    }
    if (n != g->total || !x) {
        set_error("x must hold the whole planned stream");
        return SSPSD_EINVAL;
    }
    for (uint32_t i = 0; i < g->n_inputs(); ++i)
        if (!x[i]) {
            set_error("null input");
            return SSPSD_EINVAL;
        }
    for (uint32_t r = 0; r < g->n_ranks; ++r) {
        const sspsd_time_chunk& pl = g->plan[r];
        const float* xs[4];
        for (uint32_t i = 0; i < g->n_inputs(); ++i) xs[i] = x[i] + pl.feed_lo;
        int rc = sspsd_group_time_process_multi_f32(g, r, xs, (size_t)(pl.feed_hi - pl.feed_lo), SSPSD_MEM_HOST);
        if (rc) return rc;
    }
    return SSPSD_OK;
}

int32_t sspsd_group_time_process_all_f32(sspsd_group* g, const float* x, size_t n)
{
    if (g && g->cross()) return wrong_kind("a cross-spectral group takes sspsd_group_time_process_all_multi_f32");
    if (!g || g->mode != SSPSD_SHARD_TIME || g->plan.empty() || g->multi_process) {
        set_error("needs a planned single-process time-chunked group");
        return SSPSD_EINVAL;
    }
    if (n != g->total || (n && !x)) {
        set_error("x must hold the whole planned stream");
        return SSPSD_EINVAL;
    }
    for (uint32_t r = 0; r < g->n_ranks; ++r) {
        const sspsd_time_chunk& pl = g->plan[r];
        int rc = sspsd_group_time_process_f32(g, r, x + pl.feed_lo, (size_t)(pl.feed_hi - pl.feed_lo), SSPSD_MEM_HOST);
        if (rc) return rc;
    }
    return SSPSD_OK;
}

int32_t sspsd_group_time_process_noise(sspsd_group* g, int64_t exponent, uint64_t seed)
{
    if (g && g->cross()) return wrong_kind("device-generated noise feeds PSD groups only");
    if (!g || g->mode != SSPSD_SHARD_TIME || g->plan.empty()) {
        set_error("no plan (call sspsd_group_time_plan first)");
        return SSPSD_EINVAL;
    }
    // every local rank generates its own range of the counter-based stream on its own device; generation and
    // consumption are ordered on the rank's stream, nothing is waited for here (the sources live with the group)
    if (g->noise_src.size() != g->n_local() || g->noise_exp != exponent || g->noise_seed != seed) {
        for (auto* s : g->noise_src) sspsd_source_destroy(s);
        g->noise_src.assign(g->n_local(), nullptr);
        for (uint32_t l = 0; l < g->n_local(); ++l) {
            int rc = sspsd_source_create(SSPSD_SOURCE_NOISE, exponent, seed, g->devices[l], (void*)g->tc[l]->c.stream(),
                                         &g->noise_src[l]);
            if (rc) return rc;
        }
        g->noise_exp = exponent;
        g->noise_seed = seed;
    }
    for (uint32_t l = 0; l < g->n_local(); ++l) {
        const sspsd_time_chunk& pl = g->plan[g->first_rank + l];
        int rc = sspsd_source_seek(g->noise_src[l], pl.feed_lo + g->fed[l]);
        if (rc) return rc;
        const uint64_t n = pl.feed_hi - pl.feed_lo - g->fed[l];
        rc = sspsd_cascade_process_source(g->tc[l], g->noise_src[l], (size_t)n);
        if (rc) return rc;
        g->fed[l] += n;
    }
    return SSPSD_OK;
}

int32_t sspsd_group_time_process_plant(sspsd_group* g, const sspsd_plant_spec* spec)
{
    if (!g || g->mode != SSPSD_SHARD_TIME || g->plan.empty()) {
        set_error("no plan (call sspsd_group_time_plan first)");
        return SSPSD_EINVAL;
    }
    int rc = sspsd::plant_check(spec);
    if (rc) return rc;
    if (spec->k != g->n_inputs()) {
        set_error("the plant's outputs must match the group's input streams");
        return SSPSD_EINVAL;
    }
    // as sspsd_group_time_process_noise: every local rank generates its own range on its device and stream, and
    // nothing is waited for here; the plants live with the group while the spec stays the same
    std::vector<uint8_t> key(4 * sizeof(uint32_t));
    const uint32_t dims[4] = {spec->k, spec->m, spec->taps_len, 0};
    std::memcpy(key.data(), dims, sizeof(dims));
    const uint8_t* taps = reinterpret_cast<const uint8_t*>(spec->taps);
    key.insert(key.end(), taps, taps + sizeof(float) * spec->k * spec->m * spec->taps_len);
    for (uint32_t m = 0; m < spec->m; ++m) {
        const sspsd_plant_input& in = spec->inputs[m];
        uint32_t amp;
        std::memcpy(&amp, &in.amplitude, sizeof(amp));
        const int64_t f[4] = {in.kind, in.param, (int64_t)in.seed, amp};
        const uint8_t* b = reinterpret_cast<const uint8_t*>(f);
        key.insert(key.end(), b, b + sizeof(f));
    }
    if (g->plants.size() != g->n_local() || g->plant_key != key) {
        for (auto* p : g->plants) sspsd_plant_destroy(p);
        g->plants.assign(g->n_local(), nullptr);
        g->plant_key.clear();
        for (uint32_t l = 0; l < g->n_local(); ++l) {
            void* s = g->cross() ? (void*)g->xc[l]->stream() : (void*)g->tc[l]->c.stream();
            rc = sspsd_plant_create(spec, g->devices[l], s, &g->plants[l]);
            if (rc) return rc;
        }
        g->plant_key = key;
    }
    for (uint32_t l = 0; l < g->n_local(); ++l) {
        const sspsd_time_chunk& pl = g->plan[g->first_rank + l];
        rc = sspsd_plant_seek(g->plants[l], pl.feed_lo + g->fed[l]);
        if (rc) return rc;
        const size_t n = (size_t)(pl.feed_hi - pl.feed_lo - g->fed[l]);
        if (g->kind.kind == SSPSD_GROUP_PSD)
            rc = sspsd::plant_feed(g->plants[l], g->tc[l]->c, n);
        else if (g->kind.kind == SSPSD_GROUP_ZOOM)
            rc = sspsd::plant_feed(g->plants[l], *g->zc[l], n);
        else
            rc = sspsd::plant_feed(g->plants[l], *g->xc[l], n);
        if (rc) return rc;
        g->fed[l] += n;
    }
    return SSPSD_OK;
}

int32_t sspsd_group_time_finish(sspsd_group* g)
{
    if (!g || g->mode != SSPSD_SHARD_TIME || g->plan.empty()) {
        set_error("no plan (call sspsd_group_time_plan first)");
        return SSPSD_EINVAL;
    }
    if (g->finished) return SSPSD_OK;
    const Geo geo = geo_of(g->cfg);
    const uint32_t K = g->n_local_stages, W = g->n_ranks, NL = g->n_local();
    const std::vector<StreamSt> st = stream_state(g->total, geo);
    const size_t stride = ((size_t)g->cfg.n_fft / 2 + 1 + 63) & ~(size_t)63;
    // R accumulator rows per stage, C tail streams (PSD: 1 and 1; CSD 4 and 2, CSM k >= 3 16 and k, zoom 2 and 2)
    const uint32_t R = g->cross() ? (uint32_t)g->xc[0]->block_rows() : 1;
    const uint32_t C = g->cross() ? (uint32_t)g->xc[0]->channels() : 1;
    // layout of the single reduction buffer (float64 words):
    // [K stages x R accumulator rows of `stride`] [C tail streams x W slots of `slot`] [K counts] [W x (first, length)]
    const uint64_t tail_total = st.size() > K ? st[K].L : 0;
    // slot = the longest slice any rank owns (the ownership boundaries are cut in stage-0 samples, so the slices
    // differ by a few samples; every rank derives the same number from the plan)
    size_t slot = 64;
    for (uint32_t r = 0; r < W; ++r) {
        const uint64_t hi = std::min<uint64_t>(g->plan[r].tail_hi, tail_total), lo = std::min<uint64_t>(g->plan[r].tail_lo, hi);
        slot = std::max<size_t>(slot, (size_t)(hi - lo) + 64);
    }
    const size_t nacc = (size_t)K * R * stride, gap = (size_t)W * slot, meta = nacc + C * gap, size = meta + K + 2 * (size_t)W;
    for (uint32_t l = 0; l < NL; ++l)
        if (g->fed[l] != g->plan[g->first_rank + l].feed_hi - g->plan[g->first_rank + l].feed_lo) {
            set_error("a rank has not been fed its whole range yet");
            return SSPSD_EINVAL;
        }
    // ---- per local rank: wait, export the tail slices, weight the rows for what follows the rank's chunk ----
    std::vector<std::vector<double>> factor(NL, std::vector<double>(SSPSD_MAX_STAGES, 1.0));
    std::vector<std::vector<double>> book(NL, std::vector<double>(K + 2 * (size_t)W, 0.0));
    std::vector<sspsd_partials> parts(NL);
    std::vector<uint64_t> tfirst(NL, 0);
    std::vector<size_t> tlen(NL, 0);
    for (uint32_t l = 0; l < NL; ++l) {
        const uint32_t r = g->first_rank + l;
        const sspsd_time_chunk& pl = g->plan[r];
        DevGuard dg(g->devices[l]);
        if (!dg.ok) return SSPSD_ECUDA;
        if (C * slot > g->tail_cap[l]) {
            cudaFree(g->d_tail[l]);
            g->d_tail[l] = nullptr;
            SSPSD_CUDA(cudaMalloc(&g->d_tail[l], C * slot * sizeof(float)));
            g->tail_cap[l] = C * slot;
        }
        if (!g->d_factor[l]) SSPSD_CUDA(cudaMalloc(&g->d_factor[l], SSPSD_MAX_STAGES * sizeof(double)));
        size_t n = slot;
        int rc;
        if (g->cross()) {
            if (!g->zc.empty()) {
                rc = g->zc[l]->flush();  // the zoom handle's staged host input
                if (rc) return rc;
            }
            float* outs[4];
            for (uint32_t c = 0; c < C; ++c) outs[c] = g->d_tail[l] + c * slot;
            rc = g->xc[l]->take_tail(pl.tail_lo, pl.tail_hi, outs, &n, &tfirst[l]);  // (synchronises)
            if (rc) return rc;
            rc = g->xc[l]->partials(&parts[l]);
        } else {
            Cascade& c = g->tc[l]->c;
            rc = c.take_tail(pl.tail_lo, pl.tail_hi, g->d_tail[l], &n, &tfirst[l], SSPSD_MEM_DEVICE);  // (synchronises)
            if (rc) return rc;
            rc = c.partials(&parts[l]);
        }
        if (rc) return rc;
        tlen[l] = n;
        // EWMA (psd.rs:218-225) follows the GLOBAL segment order: a rank's row is normalised as if the stream
        // ended after its last owned segment b; every later segment j rescales by g = avg/(avg+1) iff j >= avg+1
        for (uint32_t i = 0; i < K; ++i) {
            const uint32_t a = stage_avg_of(g->avg, i);
            const uint64_t s_i = i < st.size() ? st[i].craw : 0;
            if (a == 0xffffffffu) continue;
            const uint64_t bseg = pl.own_hi == NONE ? s_i : std::min(s_i, first_at_or_after(pl.own_hi, i, geo.hop, geo.drain));
            const uint64_t from = std::max<uint64_t>(bseg, (uint64_t)a + 1);
            const uint64_t later = s_i > from ? s_i - from : 0;
            const double gf = (double)((float)a / (float)(a + 1u));  // the reference divides in f32 (psd.rs:219)
            factor[l][i] = std::pow(gf, (double)later);
        }
        for (uint32_t i = 0; i < K; ++i) book[l][i] = (double)(i < parts[l].n_stages ? parts[l].count_raw[i] : 0);
        book[l][K + 2 * r] = (double)tfirst[l];
        book[l][K + 2 * r + 1] = (double)tlen[l];
    }
    auto rank_stream = [&](uint32_t l) { return g->cross() ? g->xc[l]->stream() : g->tc[l]->c.stream(); };
    // ---- combine: rows and counts are summed, the slices land in disjoint slots ----
    std::vector<double> red_book(K + 2 * (size_t)W, 0.0);
    const bool have_root = g->is_root();
    if (!g->comms.empty()) {
        for (uint32_t l = 0; l < NL; ++l) {
            DevGuard dg(g->devices[l]);
            if (size > g->buf_cap[l]) {
                cudaFree(g->d_buf[l]);
                g->d_buf[l] = nullptr;
                SSPSD_CUDA(cudaMalloc(&g->d_buf[l], size * sizeof(double)));
                g->buf_cap[l] = size;
            }
            cudaStream_t s = rank_stream(l);
            SSPSD_CUDA(cudaMemcpyAsync(g->d_factor[l], factor[l].data(), SSPSD_MAX_STAGES * sizeof(double), cudaMemcpyHostToDevice, s));
            const uint32_t r = g->first_rank + l;
            pack_exchange_kernel<<<296, 256, 0, s>>>(g->d_buf[l], meta, parts[l].acc, K, R, stride, g->d_factor[l], g->d_tail[l],
                                                     C, slot, nacc + (size_t)r * slot, gap, tlen[l]);
            SSPSD_CUDA(cudaGetLastError());
            SSPSD_CUDA(cudaMemcpyAsync(g->d_buf[l] + meta, book[l].data(), book[l].size() * sizeof(double), cudaMemcpyHostToDevice, s));
        }
        SSPSD_NCCL(nccl().GroupStart());
        for (uint32_t l = 0; l < NL; ++l) {
            DevGuard dg(g->devices[l]);
            SSPSD_NCCL(nccl().Reduce(g->d_buf[l], g->d_buf[l], size, ncclFloat64, ncclSum, 0, g->comms[l], rank_stream(l)));
        }
        SSPSD_NCCL(nccl().GroupEnd());
        if (have_root) {
            DevGuard dg(g->devices[0]);
            SSPSD_CUDA(cudaMemcpyAsync(red_book.data(), g->d_buf[0] + meta, red_book.size() * sizeof(double), cudaMemcpyDeviceToHost,
                                       rank_stream(0)));
        }
        for (uint32_t l = 0; l < NL; ++l) {
            DevGuard dg(g->devices[l]);
            SSPSD_CUDA(cudaStreamSynchronize(rank_stream(l)));
        }
    } else {
        // all ranks in this process: the root kernel reads the peers' rows in place (fixed order, f64)
        for (uint32_t l = 0; l < NL; ++l)
            for (size_t i = 0; i < red_book.size(); ++i) red_book[i] += book[l][i];
    }
    if (!have_root) {
        g->finished = true;
        return SSPSD_OK;
    }
    // ---- root: install rows + bookkeeping, gather the slices into one stream per channel, run the deep stages ----
    DevGuard dg(g->devices[0]);
    if (!dg.ok) return SSPSD_ECUDA;
    std::vector<uint64_t> first(W), len(W);
    uint64_t pos = 0;
    UnpackArgs ua{};
    ua.n_ranks = W;
    ua.C = C;
    ua.gap = gap;
    ua.nacc = nacc;
    for (uint32_t r = 0; r < W; ++r) {
        first[r] = (uint64_t)std::llround(red_book[K + 2 * r]);
        len[r] = (uint64_t)std::llround(red_book[K + 2 * r + 1]);
        if (len[r] && first[r] != pos) {
            set_error("internal: tail slices are not contiguous");
            return SSPSD_EINVAL;
        }
        ua.slot_off[r] = nacc + (size_t)r * slot;
        ua.out_off[r] = (size_t)pos;
        pos += len[r];
    }
    ua.out_off[W] = (size_t)pos;
    if (st.size() > K && pos != st[K].L) {
        set_error("internal: gathered stage-K stream has the wrong length");
        return SSPSD_EINVAL;
    }
    for (uint32_t i = 0; i < K && i < st.size(); ++i)
        if ((uint64_t)std::llround(red_book[i]) != st[i].craw) {
            set_error("internal: reduced segment count differs from the closed form");
            return SSPSD_EINVAL;
        }
    // the gathered stream of channel c at d_tail_all + c * pos
    if (C * pos > g->tail_all_cap) {
        cudaFree(g->d_tail_all);
        g->d_tail_all = nullptr;
        SSPSD_CUDA(cudaMalloc(&g->d_tail_all, (C * pos + 64) * sizeof(float)));
        g->tail_all_cap = C * pos;
    }
    sspsd_partials pr;
    int rc = g->cross() ? g->xc[0]->partials(&pr) : g->tc[0]->c.partials(&pr);
    if (rc) return rc;
    cudaStream_t rs = rank_stream(0);
    if (!g->comms.empty()) {
        ua.buf = g->d_buf[0];
        ua.acc = pr.acc;
        ua.tail_out = g->d_tail_all;
        unpack_exchange_kernel<<<296, 256, 0, rs>>>(ua);
        SSPSD_CUDA(cudaGetLastError());
    } else {
        PeerRows a{};
        a.n_ranks = NL;
        a.n_local = K;
        a.R = R;
        a.stride = stride;
        a.out = pr.acc;
        for (uint32_t l = 0; l < NL; ++l) {
            a.acc[l] = parts[l].acc;
            for (uint32_t i = 0; i < SSPSD_MAX_STAGES; ++i) a.factor[l][i] = factor[l][i];
        }
        peer_reduce_rows_kernel<<<148, 256, 0, rs>>>(a);
        SSPSD_CUDA(cudaGetLastError());
        for (uint32_t l = 0; l < NL; ++l)
            for (uint32_t c = 0; c < C && tlen[l]; ++c) {
                float* dst = g->d_tail_all + c * pos + ua.out_off[l];
                const float* src = g->d_tail[l] + c * slot;
                if (g->devices[l] == g->devices[0])
                    SSPSD_CUDA(cudaMemcpyAsync(dst, src, tlen[l] * sizeof(float), cudaMemcpyDeviceToDevice, rs));
                else
                    SSPSD_CUDA(cudaMemcpyPeerAsync(dst, g->devices[0], src, g->devices[l], tlen[l] * sizeof(float), rs));
            }
    }
    for (uint32_t i = 0; i < K && i < st.size(); ++i) {
        const uint32_t a = stage_avg_of(g->avg, i);
        const uint64_t segs = a == 0xffffffffu ? st[i].craw : std::min<uint64_t>(st[i].craw, (uint64_t)a + 1);
        rc = g->cross() ? g->xc[0]->set_stream_state(i, st[i].L, segs) : g->tc[0]->c.set_stream_state(i, st[i].L, segs);
        if (rc) return rc;
    }
    SSPSD_CUDA(cudaStreamSynchronize(rs));  // process_stage copies on the stage's own stream
    if (pos) {
        if (g->cross()) {
            // the zoom kind's tails are the mixed I and Q: the deep stages take them as they are
            const float* xs[4];
            for (uint32_t c = 0; c < C; ++c) xs[c] = g->d_tail_all + c * pos;
            rc = g->xc[0]->process_stage(K, xs, (size_t)pos);
        } else {
            rc = g->tc[0]->c.process_stage(K, g->d_tail_all, (size_t)pos, SSPSD_MEM_DEVICE);
        }
        if (rc) return rc;
    }
    rc = g->cross() ? g->xc[0]->sync() : g->tc[0]->c.sync();
    if (rc) return rc;
    g->finished = true;
    return SSPSD_OK;
}

// ---------------------------------------------------------------------------------------------
// readouts of the cross kinds: rank 0's handle after sspsd_group_time_finish (lengths 0 on the other processes)
// ---------------------------------------------------------------------------------------------
namespace {
int cross_ready(sspsd_group* g, int32_t kind, size_t* p_len, size_t* b_len, bool* empty)
{
    *empty = false;
    if (!g || !p_len || !b_len) return SSPSD_EINVAL;
    if (g->kind.kind != kind) return wrong_kind("the readout does not match the group's kind");
    if (!g->finished) {
        set_error("time-chunked group: call sspsd_group_time_finish first");
        return SSPSD_EINVAL;
    }
    if (!g->is_root()) {
        *p_len = 0;
        *b_len = 0;
        *empty = true;
    }
    return SSPSD_OK;
}
}  // namespace

int32_t sspsd_group_csd_read(sspsd_group* g, const sspsd_merge_opts* opts, float* pxx, float* pyy, float* pxy,
                             size_t* p_len, sspsd_break* b, size_t* b_len)
{
    bool empty;
    int rc = cross_ready(g, SSPSD_GROUP_CSD, p_len, b_len, &empty);
    if (rc || empty) return rc;
    sspsd_merge_opts o{0, 1, 0};
    if (opts) o = *opts;
    return g->xc[0]->read(o, pxx, pyy, pxy, p_len, b, b_len);
}

int32_t sspsd_group_csm_read(sspsd_group* g, const sspsd_merge_opts* opts, float* s, size_t* p_len, sspsd_break* b,
                             size_t* b_len)
{
    bool empty;
    int rc = cross_ready(g, SSPSD_GROUP_CSM, p_len, b_len, &empty);
    if (rc || empty) return rc;
    sspsd_merge_opts o{0, 1, 0};
    if (opts) o = *opts;
    return g->xc[0]->read_matrix(o, s, p_len, b, b_len);
}

int32_t sspsd_group_zoom_read(sspsd_group* g, const sspsd_merge_opts* opts, float* p_pos, float* p_neg, size_t* p_len,
                              sspsd_break* b, size_t* b_len)
{
    bool empty;
    int rc = cross_ready(g, SSPSD_GROUP_ZOOM, p_len, b_len, &empty);
    if (rc || empty) return rc;
    sspsd_merge_opts o{0, 1, 0};
    if (opts) o = *opts;
    return g->zc[0]->read(o, p_pos, p_neg, p_len, b, b_len);
}

}  // extern "C"
