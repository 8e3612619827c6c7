// The C++ Group of a cross kind: kind and argument checks that need no device (run first), then a time-chunked CSM
// group of three ranks on device 0 against one CsmCascade fed the whole capture, and a zoom group's readout shape.
// Exit code 3 without a GPU.
#include <cmath>
#include <cstdio>
#include <vector>

#include "sspsd.hpp"

using namespace sspsd;

template <class F>
static bool einval(F f)
{
    try {
        f();
    } catch (const Error& e) {
        return e.status == SSPSD_EINVAL;
    }
    return false;
}

int main()
{
    try {
        const std::vector<int32_t> devs{0, 0, 0};
        using G = Group<512>;
        // refused before any device is touched
        if (!einval([&] { G g(devs, G::kind_csm(4), G::Shard::Channels); })) return 1;  // channels of a cross kind
        if (!einval([&] { Group<8192> g(devs, Group<8192>::kind_csd()); })) return 1;   // N above 4096
        if (!einval([&] { Group<32> g(devs, Group<32>::kind_zoom_iq()); })) return 1;   // N below 64
        if (!einval([&] { G g(devs, G::kind_csm(5)); })) return 1;
        if (!einval([&] { G g(devs, sspsd_group_kind{SSPSD_GROUP_ZOOM, 2, SSPSD_ZOOM_IQ, 7}); })) return 1;  // I/Q carrier

        const size_t total = 1500000;
        std::vector<std::vector<float>> x(3, std::vector<float>(total));
        uint32_t s = 7;
        for (size_t k = 0; k < total; ++k) {
            const float u = (float)((s = s * 1664525u + 1013904223u) >> 8) * 0x1p-24f - 0.5f;
            const float v = (float)((s = s * 1664525u + 1013904223u) >> 8) * 0x1p-24f - 0.5f;
            x[0][k] = u;
            x[1][k] = 0.5f * u + v;
            x[2][k] = v - 0.25f * u;
        }
        G g(devs, G::kind_csm(3));  // ECUDA without a device: exit 3
        if (g.inputs() != 3 || g.kind().kind != SSPSD_GROUP_CSM) return 1;
        g.time_plan(total, 2);
        if (!einval([&] { g.time_process(0, {x[0].data(), x[1].data()}, 16); })) return 1;  // two streams for three
        if (!einval([&] { g.psd(); })) return 1;                                            // the PSD readout
        g.time_process_all(x);
        g.time_finish();
        const auto m = g.csm();
        CsmCascade<512> seq(3);
        seq.process(x);
        const auto r = seq.csm();
        if (m.k != 3 || m.bins != r.bins || m.breaks.size() != r.breaks.size() || m.bins == 0) return 1;
        for (size_t i = 0; i < m.breaks.size(); ++i)
            if (m.breaks[i].count != r.breaks[i].count || m.breaks[i].start != r.breaks[i].start) return 1;
        for (size_t i = 0; i < 3; ++i)
            for (size_t j = 0; j < 3; ++j)
                for (size_t b = 2; b < m.bins; ++b) {
                    const double sii = r(i, i, b).first, sjj = r(j, j, b).first;
                    const double tol = 1e-4 * std::sqrt(sii * sjj) + 1e-12;
                    if (std::fabs(m(i, j, b).first - r(i, j, b).first) > tol ||
                        std::fabs(m(i, j, b).second - r(i, j, b).second) > tol)
                        return 1;
                }
        Group<512> z({0, 0}, Group<512>::kind_zoom_heterodyne(0x12345679u));
        z.time_plan(total, 1);
        for (uint32_t rk = 0; rk < 2; ++rk) {
            const sspsd_time_chunk c = z.time_chunk(rk);
            z.time_process(rk, std::array<const float*, 1>{x[0].data() + c.feed_lo}, (size_t)(c.feed_hi - c.feed_lo));
        }
        z.time_finish();
        const auto zs = z.spectrum();
        if (zs.p_pos.empty() || zs.p_pos.size() != zs.p_neg.size()) return 1;
        std::puts("xgroup ok");
        return 0;
    } catch (const Error& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return e.status == SSPSD_ECUDA ? 3 : 2;
    }
}
