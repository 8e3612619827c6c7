"""The CPU restatement of the two-sided spectrum (oracle.zbinding.ZCascade) against the float64 model
(oracle.model_f64_zoom) and the PSD oracle, and the mixer's model against the integer-phase definition.  CPU only."""
import numpy as np
import pytest

from conftest import uniform_noise
from oracle import model_f64_zoom as mz
from oracle import zbinding


def tuples64(b64):
    return [(d["start"], d["include"], d["count"], d["avg"], d["bins"][0], d["bins"][1], d["fft_size"],
             d["decimation"], d["pending"], d["processed"]) for d in b64]


def feed_ragged(c, seed, n, *xs):
    rng = np.random.default_rng(seed)
    pos = 0
    while pos < xs[0].size:
        k = int(rng.integers(0, 5 * n))
        c.process(*[x[pos:pos + k] for x in xs])
        pos += k


@pytest.mark.parametrize("preset", [0, 1])
@pytest.mark.parametrize("det", [0, 1, 2, 3])
def test_restatement_matches_f64_model(det, preset):
    n = 256
    i = uniform_noise(300 * n + 77, 3) + np.float32(0.25)
    q = (0.6 * i + uniform_noise(i.size, 8) + np.float32(-0.75)).astype(np.float32)
    c = zbinding.ZCascade(n, hbf=preset)
    c.set_detrend(det)
    feed_ragged(c, det, n, i, q)
    pp, pn, b = c.spectrum()
    p64p, p64n, b64 = mz.merge_zoom(mz.zoom_cascade(i, q, n, det, preset=preset), n)
    assert [bi.as_tuple() for bi in b] == tuples64(b64)
    # tests/test_oracle_psd.py's rule: 1e-4 per bin plus 1e-6
    np.testing.assert_allclose(pp, p64p, rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(pn, p64n, rtol=1e-4, atol=1e-6)


def test_restatement_heterodyne_matches_f64_model():
    n, ftw = 512, 0x12345679
    x = uniform_noise(200 * n + 5, 12)
    c = zbinding.ZCascade(n, ftw=ftw)
    feed_ragged(c, 1, n, x)
    pp, pn, b = c.spectrum()
    i, q = mz.mix(x, ftw)
    p64p, p64n, b64 = mz.merge_zoom(mz.zoom_cascade(i, q, n), n)
    assert [bi.as_tuple() for bi in b] == tuples64(b64)
    np.testing.assert_allclose(pp, p64p, rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(pn, p64n, rtol=1e-4, atol=1e-6)


def test_real_input_is_half_the_psd(oracle):
    """(x, 0): Z = X of the real transform, so both sides are |X|^2 and each is psd(x) / 2"""
    n = 512
    x = uniform_noise(200 * n + 37, 4) + np.float32(0.5)
    c = zbinding.ZCascade(n)
    c.process(x, np.zeros_like(x))
    pp, pn, b = c.spectrum()
    ref = oracle.Cascade(n)
    ref.process(x)
    p, bp = ref.psd()
    assert [bi.as_tuple() for bi in b] == [bi.as_tuple() for bi in bp]
    np.testing.assert_array_equal(pp, p * np.float32(0.5))
    np.testing.assert_allclose(pn, pp, rtol=1e-6, atol=0)


def test_f64_model_sides_of_a_complex_tone():
    """a unit exponential at +f lands in P+ only; its image bin in P- is at the float64 floor"""
    n, k0 = 1024, 37
    t = np.arange(64 * n)
    z = np.exp(2j * np.pi * k0 * t / n)
    st = mz.zoom_stage(z.real, z.imag, n)
    assert np.argmax(st["spectrum"]) == k0
    assert st["spectrum_neg"][k0] < 1e-20 * st["spectrum"][k0]
    np.testing.assert_array_equal(st["spectrum_neg"][[0, n // 2]], st["spectrum"][[0, n // 2]])


def test_mixer_model_against_the_definition():
    rng = np.random.default_rng(5)
    x = rng.standard_normal(4096)
    for ftw in [1, 0x40000000, 0x9E3779B9, 0xFFFFFFFF, 0x12345678]:
        for pos0 in [0, 3, (1 << 32) - 17, (1 << 40) + 12345]:
            i, q = zbinding.heterodyne(x, ftw, pos0)
            nn = np.arange(x.size, dtype=object) + pos0
            phi = np.array([(int(v) * ftw) % (1 << 32) for v in nn], dtype=np.float64)
            want = x * np.exp(-2j * np.pi * phi / 2.0 ** 32)
            assert np.max(np.abs(i - want.real)) <= 1e-15 * np.max(np.abs(x)) * 8
            assert np.max(np.abs(q - want.imag)) <= 1e-15 * np.max(np.abs(x)) * 8


def test_mixer_model_quarter_turns_are_exact():
    x = np.arange(1, 17, dtype=np.float64)
    i, q = zbinding.heterodyne(x, 1 << 30)  # phases 0, 1/4, 1/2, 3/4 turn
    c = np.tile([1.0, 0.0, -1.0, 0.0], 4)
    s = np.tile([0.0, 1.0, 0.0, -1.0], 4)
    np.testing.assert_array_equal(i, x * c)
    np.testing.assert_array_equal(q, -x * s)
    cs = zbinding.phase_cos_sin(np.arange(8, dtype=np.uint64), 1 << 31)
    np.testing.assert_array_equal(cs[0], np.tile([1.0, -1.0], 4))
    np.testing.assert_array_equal(cs[1], np.zeros(8))
