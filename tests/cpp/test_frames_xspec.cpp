// The C++ overloads of FrameDecoder::process_frames and Receiver::pump for CsdCascade / CsmCascade: frames into the
// cross-spectral cascades equal the decoded traces fed to process().  Exit code 3 without a GPU.
#include <cstdio>
#include <cstring>
#include <vector>

#include "sspsd.hpp"

using namespace sspsd;

static std::vector<uint8_t> adcdac_frames(size_t n, uint8_t batches, uint32_t seq)
{
    const size_t flen = 8 + 64 * (size_t)batches;
    std::vector<uint8_t> out(n * flen);
    uint32_t x = 12345;
    for (size_t f = 0; f < n; ++f) {
        uint8_t* p = &out[f * flen];
        p[0] = 0x7B, p[1] = 0x05, p[2] = SSPSD_FORMAT_ADCDAC, p[3] = batches;
        std::memcpy(p + 4, &seq, 4);
        seq += batches;
        for (size_t i = 8; i < flen; ++i) p[i] = (uint8_t)((x = x * 1664525u + 1013904223u) >> 24);
    }
    return out;
}

int main()
{
    try {
        FrameDecoder dec;
        const uint8_t batches = 22;
        const size_t n = 3000, flen = 8 + 64 * batches;
        const auto frames = adcdac_frames(n, batches, 0xFFFFF000u);
        std::vector<float> tr[SSPSD_MAX_TRACES];
        Loss l0;
        dec.decode(frames.data(), n, flen, &l0, tr);

        CsmCascade<512> a(3), b(3);
        Loss la;
        dec.process_frames(a, {2, 0, 1}, frames.data(), n, flen, &la);
        const float* x[3] = {tr[2].data(), tr[0].data(), tr[1].data()};
        b.process(x, tr[0].size());
        const auto ma = a.csm(), mb = b.csm();
        if (la.c.received != l0.c.received || ma.breaks.size() != mb.breaks.size() || ma.s.size() != mb.s.size()) return 1;
        for (size_t i = 0; i < 3; ++i)  // the diagonal: the PSD of trace 2, 0, 1
            for (size_t k = 0; k < ma.bins; ++k) {
                const float d = ma(i, i, k).first - mb(i, i, k).first, s = mb(i, i, k).first;
                if (d > 1e-4f * s || d < -1e-4f * s) return 1;
            }
        CsdCascade<512> c;
        dec.process_frames(c, 0, 2, frames.data(), n, flen, nullptr);
        if (c.csd().pxx.empty()) return 1;
        bool threw = false;
        try {
            dec.process_frames(a, {0, 1}, frames.data(), n, flen, nullptr);  // one index per channel
        } catch (const Error& e) {
            threw = e.status == SSPSD_EINVAL;
        }
        if (!threw) return 1;
        Receiver rx("127.0.0.1", 0, 2048, 16);
        const auto r = rx.pump(dec, a, {}, nullptr, 16, 10);  // no traffic: a timeout, nothing consumed
        if (r.frames_ok != 0) return 1;
        std::puts("frames xspec ok");
        return 0;
    } catch (const Error& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return e.status == SSPSD_ECUDA ? 3 : 2;
    }
}
