// The C++ Plant: spec checks that need no device, the feed overloads, and the identity plant against Source::noise.
// Exit code 3 without a GPU.
#include <cmath>
#include <cstdio>
#include <vector>

#include "sspsd.hpp"

using namespace sspsd;

static bool refuses(int32_t status, uint32_t k, uint32_t m, uint32_t l, const std::vector<float>& taps,
                    const std::vector<Plant::Input>& in)
{
    try {
        Plant p(k, m, l, taps, in);
    } catch (const Error& e) {
        return e.status == status;
    }
    return false;
}

int main()
{
    // refused before any device is touched
    if (!refuses(SSPSD_EINVAL, 0, 1, 1, {}, {Plant::noise()})) return 1;
    if (!refuses(SSPSD_EINVAL, 5, 1, 1, std::vector<float>(5, 1.f), {Plant::noise()})) return 1;
    if (!refuses(SSPSD_EINVAL, 1, 1, 33, std::vector<float>(33, 1.f), {Plant::noise()})) return 1;
    if (!refuses(SSPSD_EUNIMPLEMENTED, 1, 1, 1, {1.f}, {Plant::noise(-1)})) return 1;
    if (!refuses(SSPSD_EUNIMPLEMENTED, 1, 1, 1, {1.f}, {Plant::noise(9)})) return 1;
    if (!refuses(SSPSD_EINVAL, 1, 1, 1, {1.f}, {Plant::Input{7, 0, 0, 0.f}})) return 1;
    if (!refuses(SSPSD_EINVAL, 1, 1, 1, {1.f}, {Plant::tone(1, NAN)})) return 1;
    try {
        Plant id(1, 1, 1, {1.f}, {Plant::noise(1, 42)});
        auto src = Source::noise(1, 42);
        PsdCascade<512> a, b;
        id.feed(a, 3000001);
        src.feed(b, 3000001);
        if (id.position() != 3000001) return 1;
        const auto pa = a.psd(), pb = b.psd();
        if (pa.first.empty() || pa.first.size() != pb.first.size()) return 1;
        for (size_t i = 0; i < pa.first.size(); ++i)
            if (std::fabs(pa.first[i] - pb.first[i]) > 1e-5f * std::fabs(pb.first[i]) + 1e-20f) return 1;
        Plant two(2, 2, 2, {1.f, 0.5f, 0.f, 1.f, 0.25f, 0.f, 1.f, -1.f}, {Plant::noise(0, 1), Plant::tone(1u << 28, 0.5f)});
        CsdCascade<512> c;
        CsmCascade<512> m(2);
        auto z = ZoomCascade<512>::iq();
        two.feed(c, 100000);
        two.seek(0);
        two.feed(m, 100000);
        two.reset();
        two.feed(z, 100000);
        bool threw = false;
        try {
            two.feed(a, 10);  // two outputs into a one-stream handle
        } catch (const Error& e) {
            threw = e.status == SSPSD_EINVAL;
        }
        if (!threw || two.position() != 100000) return 1;
        if (c.csd().pxx.empty() || m.csm().s.empty() || z.spectrum().p_pos.empty()) return 1;
        std::puts("plant ok");
        return 0;
    } catch (const Error& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return e.status == SSPSD_ECUDA ? 3 : 2;
    }
}
