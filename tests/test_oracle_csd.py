"""The CPU oracle of the cross-spectral density (oracle.xbinding.XCascade) against the PSD oracle, the float64
model (model_f64_csd.cross_cascade) and scipy.signal.csd.  CPU only.  The transfer-function fixture and its tolerance
are shared with tests/test_gpu_csd.py."""
import numpy as np
import pytest
from scipy import signal

from conftest import uniform_noise
from oracle import model_f64_csd as mcsd
from oracle import xbinding

TF_N = 512
TF_TAPS = np.array([0.0, 0.0, 0.0, 0.5, 0.25])  # y = h * x: H(f) = 0.5 e^{-6 pi i f} + 0.25 e^{-8 pi i f}


def tuples64(b64):
    return [(d["start"], d["include"], d["count"], d["avg"], d["bins"][0], d["bins"][1], d["fft_size"],
             d["decimation"], d["pending"], d["processed"]) for d in b64]


def transfer_fixture():
    """x: 2^22 samples of white noise; y = h * x (float64 filter, rounded to f32 like any input)"""
    x = uniform_noise(1 << 22, 11)
    y = np.convolve(x.astype(np.float64), TF_TAPS)[:x.size].astype(np.float32)
    return x, y


def transfer_expected(breaks, n=TF_N):
    """H at every merged bin, frequencies in stage-0 units (bin k of a break with decimation d: f = k / (N d)),
    plus each bin's decimation and segment count.  `breaks`: (include, count, bins_start, bins_end, decimation)."""
    f, dec, cnt = [], [], []
    for inc, count, b0, b1, d in breaks:
        if inc:
            k = np.arange(b0, b1)
            f.append(k / (n * d))
            dec.append(np.full(k.size, d))
            cnt.append(np.full(k.size, count))
    f = np.concatenate(f)
    h = 0.5 * np.exp(-6j * np.pi * f) + 0.25 * np.exp(-8j * np.pi * f)
    return h, np.concatenate(dec), np.concatenate(cnt)


def transfer_tolerance(h, dec, cnt, coh, n=TF_N):
    """Allowed |pxy/pxx - H| per bin.
      - Random error of the estimate: sigma = |H| sqrt((1 - g2) / (2 K g2)) (Bendat & Piersol, K = averaged
        segments, g2 = coherence); 5 sigma.  The coherence is below 1 because the 3..4-sample delay of h moves
        samples across the segment edges.
      - Bias of the same origin: a delay of d samples scales the windowed cross-spectrum by about
        1 - (pi d / N)^2 (Hann); d = 4 / 8^i samples at stage i.
      - Floor 2e-4 |H|: f32 input rounding and accumulation; it carries the deepest stages, whose K = 2..30
        segments make the coherence estimate meaningless.
    On the float64 model (seed 11) the largest error is 0.40 of this bound."""
    g2 = np.clip(coh, 1e-12, 1.0)
    sigma = np.abs(h) * np.sqrt((1.0 - g2) / (2.0 * cnt * g2))
    bias = (np.pi * 4.0 / (dec * n)) ** 2 * np.abs(h)
    return 5.0 * sigma + bias + 2e-4 * np.abs(h)


def test_oracle_y_equals_x_is_the_psd(oracle):
    n = 512
    x = uniform_noise(200 * n + 37, 4) + np.float32(0.5)
    c = xbinding.XCascade(n)
    c.process(x, x)
    pxx, pyy, pxy, b = c.csd()
    ref = oracle.Cascade(n)
    ref.process(x)
    p, bp = ref.psd()
    assert np.all(pxy.imag == 0)
    assert np.array_equal(pxy.real, pxx) and np.array_equal(pyy, pxx) and np.array_equal(pxx, p)
    assert [bi.as_tuple() for bi in b] == [bi.as_tuple() for bi in bp]


@pytest.mark.parametrize("preset", [0, 1])
@pytest.mark.parametrize("det", [0, 1, 2, 3])
def test_oracle_matches_f64_model(oracle, det, preset):
    n = 256
    x = uniform_noise(300 * n + 77, 3) + np.float32(0.25)
    y = (0.6 * x + uniform_noise(x.size, 8) + np.float32(-0.75)).astype(np.float32)
    c = xbinding.XCascade(n, hbf=preset)
    c.set_detrend(det)
    rng = np.random.default_rng(det)  # ragged feeding, x and y split identically
    pos = 0
    while pos < x.size:
        k = int(rng.integers(0, 5 * n))
        c.process(x[pos:pos + k], y[pos:pos + k])
        pos += k
    ref = mcsd.cross_cascade(x, y, n, det, preset=preset)
    pxx, pyy, pxy, b = c.csd()
    p64x, p64y, p64xy, b64 = mcsd.merge_cross(ref, n)
    assert [bi.as_tuple() for bi in b] == tuples64(b64)
    # the existing rule (tests/test_oracle_psd.py): 1e-4 per bin plus 1e-6; the cross row on the Cauchy-Schwarz
    # scale sqrt(pxx pyy), since |pxy| itself can be ~0 for uncorrelated bins
    np.testing.assert_allclose(pxx, p64x, rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(pyy, p64y, rtol=1e-4, atol=1e-6)
    scale = np.sqrt(p64x * p64y)
    assert np.all(np.abs(pxy.real - p64xy.real) <= 1e-4 * scale + 1e-6)
    assert np.all(np.abs(pxy.imag - p64xy.imag) <= 1e-4 * scale + 1e-6)


def test_f64_model_single_stage_matches_scipy():
    n = 1024
    x = uniform_noise(64 * n, 21).astype(np.float64)
    y = np.convolve(x, [0.3, -0.2, 0.7])[:x.size] + 0.1 * uniform_noise(x.size, 22)
    st = mcsd.cross_stage(x, y, n)
    kw = dict(window="hann", nperseg=n, noverlap=n // 2, detrend=False)  # scipy's "hann" is periodic by default
    _, sxy = signal.csd(x, y, **kw)
    _, sxx = signal.welch(x, **kw)
    # the scaling conventions differ (one-sided doubling, density): the ratio is what both estimate
    np.testing.assert_allclose(st["spectrum_xy"] / st["spectrum"], sxy / sxx, rtol=1e-9, atol=1e-12)


def test_f64_model_transfer_function():
    x, y = transfer_fixture()
    st = mcsd.cross_cascade(x, y, TF_N)
    pxx, pyy, pxy, b64 = mcsd.merge_cross(st, TF_N)
    assert len(b64) >= 4
    h, dec, cnt = transfer_expected([(d["include"], d["count"], d["bins"][0], d["bins"][1], d["decimation"])
                                     for d in b64])
    coh = np.abs(pxy) ** 2 / (pxx * pyy)
    err = np.abs(pxy / pxx - h)
    tol = transfer_tolerance(h, dec, cnt, coh)
    assert np.all(err <= tol), "worst bin: err %.3g > tol %.3g" % (err[np.argmax(err / tol)], tol[np.argmax(err / tol)])
