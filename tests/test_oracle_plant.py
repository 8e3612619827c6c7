"""CPU checks of the plants' restatement (oracle/sspsd_poracle.c) and of Plant.expected_csm: the restatement against a
plain numpy convolution mix of the oracle's own sources, and the closed-form cross-spectral matrix against the float64
model's estimate (oracle/csm.py over oracle/model_f64_csd.py) of a 2^22-sample plant, within bounds derived from the
segment counts and the Hann window's bias."""
import numpy as np
import pytest

from oracle import binding as orc
from oracle import csm as ocsm
from oracle import pbinding


def _ulps(a, b):
    a = np.asarray(a, np.float32).view(np.int32).astype(np.int64)
    b = np.asarray(b, np.float32).view(np.int32).astype(np.int64)
    a = np.where(a < 0, -(a & 0x7FFFFFFF), a)
    b = np.where(b < 0, -(b & 0x7FFFFFFF), b)
    return np.abs(a - b)


def _inputs_np(inputs, n):
    """each input from the oracle's sources / the mixer's cosine restated in numpy (f64 libm, one rounding)"""
    out = []
    for kind, param, seed, amp in inputs:
        if kind == pbinding.NOISE:
            out.append(orc.Source(orc.SOURCE_NOISE, param, seed).get(n))
        else:
            phi = (np.arange(n, dtype=np.uint64) * np.uint64(param)) & np.uint64(0xFFFFFFFF)
            quad = (phi >> np.uint64(30)).astype(np.int64)
            a = (phi & np.uint64(0x3FFFFFFF)).astype(np.float64) * 2.0 ** -31 * np.pi
            cf, sf = np.cos(a).astype(np.float32), np.sin(a).astype(np.float32)
            c = np.choose(quad, [cf, -sf, -cf, sf])
            out.append((np.float32(amp) * c).astype(np.float32))
    return out


CASES = [
    # taps shape, inputs
    ((1, 1, 1), [(0, 0, 11, 0.0)]),
    ((2, 2, 7), [(0, 1, 3, 0.0), (0, 3, 4, 0.0)]),
    ((4, 3, 32), [(0, 0, 5, 0.0), (1, 0x1234567, 0, 0.75), (0, 8, 6, 0.0)]),
    ((3, 4, 5), [(1, 0x40000000, 0, 1.0), (0, 2, 7, 0.0), (1, 0xDEADBEEF, 0, -2.0), (0, 0, 8, 0.0)]),
]


@pytest.mark.parametrize("shape,inputs", CASES)
def test_restatement_matches_a_numpy_convolution_mix(shape, inputs):
    k, m, nt = shape
    rng = np.random.default_rng(sum(shape))
    taps = rng.standard_normal(shape).astype(np.float32)
    n = 20000
    y = pbinding.plant(taps, inputs, n)
    u = _inputs_np(inputs, n)
    for i in range(k):
        ref = np.zeros(n)
        for q in range(m):
            ref += np.convolve(taps[i, q].astype(np.float64), u[q].astype(np.float64))[:n]
        assert np.max(_ulps(y[i], ref.astype(np.float32))) <= 1, i
    # any window of the stream is the same slice of it
    np.testing.assert_array_equal(pbinding.plant(taps, inputs, 777, pos=12345), y[:, 12345:12345 + 777])


def test_identity_plant_is_the_noise_source():
    for e in (0, 1, 3, 8):
        y = pbinding.plant(np.ones((1, 1, 1)), [(0, e, 99, 0.0)], 5000)
        np.testing.assert_array_equal(y[0].view(np.uint32), orc.Source(orc.SOURCE_NOISE, e, 99).get(5000).view(np.uint32))


def test_tone_factor_is_exact_at_quarter_turns():
    assert [pbinding.plant_cos(q << 30) for q in range(4)] == [1.0, 0.0, -1.0, 0.0]


def test_restatement_refuses_what_the_plant_refuses():
    with pytest.raises(ValueError):
        pbinding.plant(np.ones((1, 1, 1)), [(0, -1, 0, 0.0)], 10)
    with pytest.raises(ValueError):
        pbinding.plant(np.ones((1, 1, 1)), [(2, 0, 0, 0.0)], 10)


def bin_axis(breaks, n):
    """frequency (cycles per stage-0 sample) and segment count of every merged bin of model_f64 breaks"""
    f, cnt, dec = [], [], []
    for b in breaks:
        if not b["include"]:
            continue
        lo, hi = b["bins"]
        f.extend(np.arange(lo, hi) / (n * b["decimation"]))
        cnt.extend([b["count"]] * (hi - lo))
        dec.extend([b["decimation"]] * (hi - lo))
    return np.array(f), np.array(cnt, np.float64), np.array(dec, np.float64)


def spread(cnt, p=2.9e-7):
    """relative deviation of an average of `cnt` Hann segments at 50 % overlap that is exceeded with probability p (the
    two-sided 5 sigma tail): the average is chi^2 with nu = 2 count_eff degrees of freedom over nu, count_eff = count / 1.2
    (Welch's variance factor 1 + 2 rho^2, rho = 0.167, rounded up).  For large counts this is 5 / sqrt(count_eff); for the
    few segments of the deepest stages the chi^2 tail is far longer than the Gaussian's."""
    from scipy.stats import chi2
    nu = 2.0 * np.asarray(cnt, np.float64) / 1.2
    return np.maximum(chi2.isf(p, nu) / nu - 1.0, 1.0 - chi2.ppf(p, nu) / nu)


def rounding_floor(S_true, expected, dec, gamma=1e-7):
    """section 4's f32 rounding floor per channel and bin, gamma sqrt(S_ii r) + gamma^2 r with r = 2 P_i dec the density
    channel i's total power P_i would have as white noise at the bin's stage -> (floor [K, bins], r [K, bins])"""
    grid = np.linspace(0.0, 0.5, 8193)
    power = 0.5 * np.mean(np.real(np.einsum("iib->ib", expected(grid))), axis=1)       # P_i = int_0^1/2 S_ii df
    r = 2.0 * power[:, None] * np.asarray(dec, np.float64)[None, :]
    t = np.maximum(np.real(np.einsum("iib->ib", S_true)), 0)
    return gamma * np.sqrt(t * r) + gamma ** 2 * r, r


def csm_bound(S_true, expected, f, cnt, n, dec, gamma=1e-7):
    """per-bin bound on |S_est - S_true|:
      - spread(count) * sqrt(S_ii S_jj): the chi^2 tail of the segment average (5 sigma for large counts);
      - the window's bias, bounded by the second difference of S over one bin (the Hann spectral window's second moment
        is 1/3 bin^2);
      - the f32 rounding floor of section 4's dynamic-range budget, gamma sqrt(S r) + gamma^2 r with r_i = 2 P_i dec the
        density channel i's total power P_i would have as white noise at the bin's stage: where a differenced input
        makes S_ii fall far below its total power (the deep stages near DC), the decimators' rounding, not S, sets the
        estimate;
      - 2e-4 of sqrt(S_ii S_jj): f32 accumulation over long runs."""
    df = 1.0 / (n * dec)
    bias = np.abs(expected(f + df) - 2 * S_true + expected(np.abs(f - df)))
    floor_d, r = rounding_floor(S_true, expected, dec, gamma)
    t = np.real(np.einsum("iib->ib", S_true))
    # the spread follows the powers the estimate sees: the diagonal as the window smooths it, over the rounding floor
    d = t + np.real(np.einsum("iib->ib", bias)) + floor_d
    scale = np.sqrt(np.maximum(d[:, None, :] * d[None, :, :], 0))
    floor = np.sqrt(floor_d[:, None, :] * floor_d[None, :, :]) + gamma * np.sqrt(
        np.maximum(t[:, None, :] * r[None, :, :], 0) + np.maximum(t[None, :, :] * r[:, None, :], 0))
    return spread(cnt) * scale + bias + floor + 2e-4 * scale


def test_expected_csm_matches_the_f64_model():
    from stabilizer_stream_b200.psd import Plant, PlantSpec
    n, total = 512, 1 << 22
    taps = np.array([[[1.0, 0.5, -0.25, 0.0], [0.0, 0.0, 0.0, 0.0]],
                     [[0.0, 0.0, 0.0, 0.0], [0.5, -1.0, 0.3, 0.1]],
                     [[0.7, 0.0, 0.2, 0.0], [0.0, 0.6, 0.0, -0.4]]], np.float32)
    inputs = [Plant.noise(0, 21), Plant.noise(1, 22)]
    p = Plant.__new__(Plant)
    p._spec, p.k, p._h = PlantSpec(taps, inputs), 3, None
    y = pbinding.plant(taps, inputs, total)
    S, breaks = ocsm.f64_matrix([y[i] for i in range(3)], n)
    f, cnt, dec = bin_axis(breaks, n)
    want = p.expected_csm(f)
    bound = csm_bound(want, p.expected_csm, f, cnt, n, dec)
    ratio = np.abs(S - want) / bound
    print("worst ratio to the bound %.3f" % ratio.max())
    assert ratio.max() < 1.0
    # the estimate is not trivially inside: the bound is tight enough to see a wrong factor of 2 or a wrong sign
    many = cnt >= 1000
    assert np.median(np.abs(0.5 * want[0, 0] - S[0, 0])[many] / bound[0, 0][many]) > 1.0
    assert np.median(np.abs(np.conj(want[0, 2]) - S[0, 2])[many] / bound[0, 2][many]) > 1.0
