// The C++ ZoomCascade: both modes, the frame and pump overloads.  Heterodyne mode at carrier 0 reads what I/Q mode reads
// for (x, -(x * 0)), the samples the mixer forms there.  Exit code 3 without a GPU.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>

#include "sspsd.hpp"

using namespace sspsd;

static std::vector<uint8_t> fls_frames(size_t n, uint8_t batches, uint32_t seq)
{
    const size_t flen = 8 + 56 * (size_t)batches;
    std::vector<uint8_t> out(n * flen);
    uint32_t x = 777;
    for (size_t f = 0; f < n; ++f) {
        uint8_t* p = &out[f * flen];
        p[0] = 0x7B, p[1] = 0x05, p[2] = SSPSD_FORMAT_FLS, p[3] = batches;
        std::memcpy(p + 4, &seq, 4);
        seq += batches;
        for (size_t i = 8; i < flen; ++i) p[i] = (uint8_t)((x = x * 1664525u + 1013904223u) >> 24);
    }
    return out;
}

int main()
{
    try {
        std::vector<float> x(300000), zero(x.size());
        uint32_t s = 1;
        for (auto& v : x) v = (float)((s = s * 1664525u + 1013904223u) >> 8) * 0x1p-24f - 0.5f;
        for (size_t k = 0; k < x.size(); ++k) zero[k] = -(x[k] * 0.0f);
        auto h = ZoomCascade<512>::heterodyne(0);
        auto z = ZoomCascade<512>::iq();
        h.process(x);
        z.process(x, zero);
        const auto a = h.spectrum(), b = z.spectrum();
        if (a.p_pos.empty() || a.p_pos.size() != b.p_pos.size() || a.breaks.size() != b.breaks.size()) return 1;
        for (size_t k = 0; k < a.p_pos.size(); ++k)
            if (std::fabs(a.p_pos[k] - b.p_pos[k]) > 1e-4f * b.p_pos[k] + 1e-12f ||
                std::fabs(a.p_neg[k] - b.p_neg[k]) > 1e-4f * b.p_neg[k] + 1e-12f)
                return 1;
        if (h.carrier().first != SSPSD_ZOOM_HETERODYNE || z.traces() != 2) return 1;
        bool threw = false;
        try {
            h.process(x, x);  // I/Q samples into a heterodyne handle
        } catch (const Error& e) {
            threw = e.status == SSPSD_EINVAL;
        }
        if (!threw) return 1;

        FrameDecoder dec;
        const uint8_t batches = 60;
        const auto frames = fls_frames(2000, batches, 0xFFFFFF00u);
        const size_t flen = 8 + 56 * batches;
        std::vector<float> tr[SSPSD_MAX_TRACES];
        dec.decode(frames.data(), 2000, flen, nullptr, tr);
        ZoomCascade<512> f = ZoomCascade<512>::iq(), g = ZoomCascade<512>::iq();
        Loss l;
        dec.process_frames(f, {2, 3}, frames.data(), 2000, flen, &l);  // BI, BQ
        g.process(tr[2], tr[3]);
        const auto fa = f.spectrum(), ga = g.spectrum();
        if (fa.p_pos.size() != ga.p_pos.size() || l.c.received == 0) return 1;
        for (size_t k = 0; k < fa.p_pos.size(); ++k)
            if (std::fabs(fa.p_neg[k] - ga.p_neg[k]) > 1e-4f * ga.p_neg[k] + 1e-12f) return 1;
        auto m = ZoomCascade<512>::heterodyne(0x10000000u);
        dec.process_frames(m, {1}, frames.data(), 2000, flen, nullptr);
        if (m.spectrum().p_pos.empty()) return 1;
        threw = false;
        try {
            dec.process_frames(m, {0, 1}, frames.data(), 2000, flen, nullptr);  // one index in heterodyne mode
        } catch (const Error& e) {
            threw = e.status == SSPSD_EINVAL;
        }
        if (!threw) return 1;
        Receiver rx("127.0.0.1", 0, 2048, 16);
        if (rx.pump(dec, f, {2, 3}, nullptr, 16, 10).frames_ok != 0) return 1;  // no traffic: a timeout
        std::puts("zoom ok");
        return 0;
    } catch (const Error& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return e.status == SSPSD_ECUDA ? 3 : 2;
    }
}
