// sspsd_plant.cu -- plants behind the C ABI (include/sspsd.h, sspsd_plant_*; DESIGN.md 3d): seeded multi-channel
// test signals generated on the device and fed straight into the cascades, like sspsd_cascade_process_source.
// Every input is counter-based, so a plant keeps no device state: its position lives on the host, and any position
// can be generated directly (seek).
#include <cmath>
#include <cstring>
#include <functional>
#include <new>

#include "sspsd_plant.cuh"
#include "sspsd_plant_kernel.cuh"

namespace sspsd {

int plant_check(const sspsd_plant_spec* spec)
{
    if (!spec || spec->k < 1 || spec->k > PLANT_MAX_K || spec->m < 1 || spec->m > PLANT_MAX_M || spec->taps_len < 1 ||
        spec->taps_len > PLANT_MAX_L || !spec->taps || !spec->inputs) {
        set_error("plant: k and m must be 1 .. 4, taps_len 1 .. 32, taps and inputs given");
        return SSPSD_EINVAL;
    }
    for (uint32_t m = 0; m < spec->m; ++m) {
        const sspsd_plant_input& in = spec->inputs[m];
        if (in.kind == SSPSD_PLANT_NOISE) {
            if (in.param < 0 || in.param > SRC_MAX_DIFF) {
                // integrated noise carries state and cannot be entered at any position (sspsd_source_seek's rule)
                set_error("plant: noise exponents 0 .. 8 only (the counter-based, seekable ones)");
                return SSPSD_EUNIMPLEMENTED;
            }
        } else if (in.kind == SSPSD_PLANT_TONE) {
            if (in.param < 0 || in.param > 0xffffffffll || !std::isfinite(in.amplitude)) {
                set_error("plant: a tone's ftw must fit u32 and its amplitude be finite");
                return SSPSD_EINVAL;
            }
        } else {
            set_error("plant: unknown input kind");
            return SSPSD_EINVAL;
        }
    }
    return SSPSD_OK;
}

class Plant {
public:
    ~Plant()
    {
        DeviceGuard g(device_);
        for (float* b : buf_) cudaFree(b);
        if (own_stream_ && stream_) cudaStreamDestroy(stream_);
    }

    int init(const sspsd_plant_spec& spec, int device, void* stream)
    {
        int rc = plant_check(&spec);
        if (rc) return rc;
        device_ = device;
        k_ = spec.k;
        base_ = PlantParams{};
        base_.m = (int)spec.m;
        base_.taps_len = (int)spec.taps_len;
        base_.scale = sqrtf(12.0f);
        for (uint32_t m = 0; m < spec.m; ++m) {
            const sspsd_plant_input& in = spec.inputs[m];
            base_.kind[m] = in.kind == SSPSD_PLANT_NOISE ? PLANT_IN_NOISE : PLANT_IN_TONE;
            if (in.kind == SSPSD_PLANT_NOISE) {
                base_.order[m] = (int)in.param;
                base_.key0[m] = (uint32_t)in.seed;
                base_.key1[m] = (uint32_t)(in.seed >> 32);
                if (base_.order[m] > base_.emax) base_.emax = base_.order[m];
            } else {
                base_.ftw[m] = (uint32_t)in.param;
                base_.amp[m] = in.amplitude;
            }
        }
        std::memcpy(base_.taps, spec.taps, sizeof(float) * spec.k * spec.m * spec.taps_len);
        DeviceGuard g(device_);
        if (!g.ok) return SSPSD_ECUDA;
        if (stream) {
            stream_ = stream == (void*)1 ? cudaStreamLegacy : (cudaStream_t)stream;
        } else {
            SSPSD_CUDA(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
            own_stream_ = true;
        }
        return SSPSD_OK;
    }

    // the next n positions of all k outputs into d_out[0 .. k-1] (device memory), in order on stream s
    int generate(float* const* d_out, size_t n, cudaStream_t s)
    {
        DeviceGuard g(device_);
        if (!g.ok) return SSPSD_ECUDA;
        // the scratch buffers a previous call on another stream filled may still be read there
        if (last_stream_ && last_stream_ != s) SSPSD_CUDA(cudaStreamSynchronize(last_stream_));
        last_stream_ = s;
        const size_t max_call = (size_t)1 << 30;
        PlantParams p = base_;
        for (size_t off = 0; off < n;) {
            const size_t c = n - off < max_call ? n - off : max_call;
            p.pos = pos_;
            p.n = c;
            for (uint32_t i = 0; i < k_; ++i) p.out[i] = d_out[i] + off;
            const unsigned int grid = (unsigned int)((c + PLANT_TILE - 1) / PLANT_TILE);
            switch (k_) {
            case 1: plant_kernel<1><<<grid, PLANT_NT, 0, s>>>(p); break;
            case 2: plant_kernel<2><<<grid, PLANT_NT, 0, s>>>(p); break;
            case 3: plant_kernel<3><<<grid, PLANT_NT, 0, s>>>(p); break;
            default: plant_kernel<4><<<grid, PLANT_NT, 0, s>>>(p); break;
            }
            SSPSD_CUDA(cudaGetLastError());
            pos_ += c;
            off += c;
        }
        return SSPSD_OK;
    }

    // Slices of at most `slice` positions into scratch buffers, each handed to `consume` in order on stream s.  Slices
    // are multiples of 4 positions, so a handle at a multiple of 4 reads every slice in place; stream order makes the
    // reuse of the buffers by the next slice safe.
    int feed(int device, cudaStream_t s, uint32_t k, size_t n, const std::function<int(float* const*, size_t)>& consume)
    {
        if (device != device_) {
            set_error("plant and handle live on different devices");
            return SSPSD_EINVAL;
        }
        if (k != k_) {
            set_error("plant has " + std::to_string(k_) + " outputs, the handle takes " + std::to_string(k) + " streams");
            return SSPSD_EINVAL;
        }
        if (n == 0) return SSPSD_OK;
        DeviceGuard g(device_);
        if (!g.ok) return SSPSD_ECUDA;
        const size_t slice = (size_t)1 << 24;
        const size_t need = n < slice ? n : slice;
        if (need > buf_cap_) {
            // the old buffers may still be read by the handle the last call fed
            if (last_stream_) SSPSD_CUDA(cudaStreamSynchronize(last_stream_));
            for (float*& b : buf_) {
                SSPSD_CUDA(cudaFree(b));
                b = nullptr;
            }
            buf_cap_ = 0;
            for (uint32_t i = 0; i < k_; ++i) SSPSD_CUDA(cudaMalloc(&buf_[i], need * sizeof(float)));
            buf_cap_ = need;
        }
        while (n) {
            const size_t cnt = n < slice ? n : slice;
            int rc = generate(buf_, cnt, s);
            if (rc) return rc;
            rc = consume(buf_, cnt);
            if (rc) return rc;
            n -= cnt;
        }
        return SSPSD_OK;
    }

    uint64_t position() const { return pos_; }
    uint32_t k() const { return k_; }
    void seek(uint64_t pos) { pos_ = pos; }
    cudaStream_t stream() const { return stream_; }

private:
    PlantParams base_{};
    uint32_t k_ = 1;
    int device_ = 0;
    bool own_stream_ = false;
    uint64_t pos_ = 0;
    cudaStream_t stream_ = nullptr, last_stream_ = nullptr;
    float* buf_[PLANT_MAX_K] = {nullptr, nullptr, nullptr, nullptr};
    size_t buf_cap_ = 0;
};

}  // namespace sspsd

struct sspsd_plant {
    sspsd::Plant p;
};

namespace sspsd {

int plant_feed(sspsd_plant* p, Cascade& c, size_t n)
{
    return p->p.feed(c.device(), c.stream(), 1, n,
                     [&](float* const* b, size_t cnt) { return c.process(b[0], cnt, SSPSD_MEM_DEVICE); });
}

int plant_feed(sspsd_plant* p, XCascade& x, size_t n)
{
    return p->p.feed(x.device(), x.stream(), (uint32_t)x.channels(), n,
                     [&](float* const* b, size_t cnt) { return x.process(b, cnt, SSPSD_MEM_DEVICE); });
}

int plant_feed(sspsd_plant* p, ZoomCascade& z, size_t n)
{
    if (z.mode() == SSPSD_ZOOM_IQ)
        return p->p.feed(z.x().device(), z.x().stream(), 2, n,
                         [&](float* const* b, size_t cnt) { return z.process_iq(b[0], b[1], cnt, SSPSD_MEM_DEVICE); });
    // heterodyne: the handle's own mixer path
    return p->p.feed(z.x().device(), z.x().stream(), 1, n,
                     [&](float* const* b, size_t cnt) { return z.process(b[0], cnt, SSPSD_MEM_DEVICE); });
}

}  // namespace sspsd

using namespace sspsd;

extern "C" {

int32_t sspsd_plant_create(const sspsd_plant_spec* spec, int32_t device, void* stream, sspsd_plant** out)
{
    if (!out) return SSPSD_EINVAL;
    *out = nullptr;
    int rc = plant_check(spec);
    if (rc) return rc;
    sspsd_plant* h = new (std::nothrow) sspsd_plant;
    if (!h) return SSPSD_ENOMEM;
    rc = h->p.init(*spec, device, stream);
    if (rc) {
        delete h;
        return rc;
    }
    *out = h;
    return SSPSD_OK;
}

void sspsd_plant_destroy(sspsd_plant* p) { delete p; }

int32_t sspsd_plant_reset(sspsd_plant* p)
{
    if (!p) return SSPSD_EINVAL;
    p->p.seek(0);
    return SSPSD_OK;
}

int32_t sspsd_plant_seek(sspsd_plant* p, uint64_t pos)
{
    if (!p) return SSPSD_EINVAL;
    p->p.seek(pos);
    return SSPSD_OK;
}

int32_t sspsd_plant_position(const sspsd_plant* p, uint64_t* pos)
{
    if (!p || !pos) return SSPSD_EINVAL;
    *pos = p->p.position();
    return SSPSD_OK;
}

int32_t sspsd_plant_generate(sspsd_plant* p, float* const* d_out, size_t n)
{
    if (!p || (n && !d_out)) return SSPSD_EINVAL;
    for (uint32_t i = 0; n && i < p->p.k(); ++i)
        if (!d_out[i]) {
            set_error("null output buffer");
            return SSPSD_EINVAL;
        }
    return p->p.generate(d_out, n, p->p.stream());
}

int32_t sspsd_cascade_process_plant(sspsd_cascade* c, sspsd_plant* p, size_t n)
{
    if (!c || !p) return SSPSD_EINVAL;
    return plant_feed(p, c->c, n);
}

int32_t sspsd_csd_process_plant(sspsd_csd* c, sspsd_plant* p, size_t n)
{
    if (!c || !p) return SSPSD_EINVAL;
    return plant_feed(p, c->c, n);
}

int32_t sspsd_csm_process_plant(sspsd_csm* c, sspsd_plant* p, size_t n)
{
    if (!c || !p) return SSPSD_EINVAL;
    return plant_feed(p, c->c, n);
}

int32_t sspsd_zoom_process_plant(sspsd_zoom* z, sspsd_plant* p, size_t n)
{
    if (!z || !p) return SSPSD_EINVAL;
    return plant_feed(p, z->z, n);
}

}  // extern "C"
