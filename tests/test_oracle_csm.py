"""The cross-spectral matrix references (oracle.csm: pairwise f32 restatement and float64 model) and the host-side
helpers CsmCascade.coherence / .transfer.  CPU only.  The MIMO fixture and its tolerance are shared with
tests/test_gpu_csm.py."""
import numpy as np
import pytest

from conftest import uniform_noise
from oracle import csm as ocsm
from test_oracle_csd import TF_N, tuples64
from stabilizer_stream_b200 import CsdCascade, CsmCascade

# y_o = sum_i h[o][i] * u_i: four short FIR paths, delays up to 4 samples like the CSD fixture
MIMO_TAPS = [[np.array([0.0, 0.0, 0.0, 0.5, 0.25]), np.array([0.2, -0.1])],
             [np.array([0.0, 0.3]), np.array([0.0, 0.0, 0.7, 0.0, -0.2])]]
MIMO_DELAY = 4.0


def mimo_fixture(n_samples=1 << 22):
    """channels (u0, u1, y0, y1): two independent noise inputs and two outputs mixing both (float64 filters,
    rounded to f32 like any input)"""
    u = [uniform_noise(n_samples, 51), uniform_noise(n_samples, 52)]
    y = []
    for o in range(2):
        acc = np.zeros(n_samples)
        for i in range(2):
            acc += np.convolve(u[i].astype(np.float64), MIMO_TAPS[o][i])[:n_samples]
        y.append(acc.astype(np.float32))
    return u + y


def mimo_expected(breaks, n=TF_N):
    """H [2, 2, bins] at every merged bin, plus each bin's decimation and segment count.  `breaks`: (include, count,
    bins_start, bins_end, decimation)."""
    f, dec, cnt = [], [], []
    for inc, count, b0, b1, d in breaks:
        if inc:
            k = np.arange(b0, b1)
            f.append(k / (n * d))
            dec.append(np.full(k.size, d))
            cnt.append(np.full(k.size, count))
    f = np.concatenate(f)
    h = np.zeros((2, 2, f.size), np.complex128)
    for o in range(2):
        for i in range(2):
            for t, c in enumerate(MIMO_TAPS[o][i]):
                h[o, i] += c * np.exp(-2j * np.pi * f * t)
    return h, np.concatenate(dec), np.concatenate(cnt)


def mimo_tolerance(S, h, dec, cnt, n=TF_N):
    """Allowed |H_est - H| per element and bin, transfer_tolerance's terms for two inputs:
      - random error (Bendat & Piersol, multiple-input): sigma_oi = sqrt(S_nn,o / (2 K S_ii.rest)), with S_nn,o the
        output power the inputs do not explain, S_nn,o = S_oo - S_uo^H S_uu^-1 S_uo, and S_ii.rest = 1 / [S_uu^-1]_ii
        the power of input i not explained by the other; 5 sigma.  The residual is not 0 because the delays of h
        move samples across the segment edges.
      - bias of the same origin, (pi d / N)^2 |H| with d = 4 / 8^i samples at stage i;
      - floor 2e-4 (|H_o0| + |H_o1|): f32 input rounding and accumulation (the deepest stages)."""
    S = np.asarray(S, np.complex128)
    m = S.shape[-1]
    tol = np.zeros((2, 2, m))
    suu = np.moveaxis(S[:2, :2], -1, 0)
    inv = np.linalg.inv(suu)
    for o in range(2):
        suo = np.moveaxis(S[:2, 2 + o], -1, 0)[..., None]
        expl = np.real(np.conj(np.swapaxes(suo, 1, 2)) @ inv @ suo)[:, 0, 0]
        snn = np.maximum(np.real(S[2 + o, 2 + o]) - expl, 0.0)
        for i in range(2):
            rest = 1.0 / np.real(inv[:, i, i])
            sigma = np.sqrt(snn / (2.0 * cnt * rest))
            bias = (np.pi * MIMO_DELAY / (dec * n)) ** 2 * np.abs(h[o, i])
            tol[o, i] = 5.0 * sigma + bias + 2e-4 * (np.abs(h[o, 0]) + np.abs(h[o, 1]))
    return tol


def assert_mimo(S, breaks):
    h, dec, cnt = mimo_expected(breaks)
    est = CsmCascade.transfer(S, [0, 1], [2, 3])
    assert est.shape == h.shape
    err = np.abs(est - h)
    tol = mimo_tolerance(S, h, dec, cnt)
    r = err / tol
    assert np.all(err <= tol), "worst H[%d,%d] bin %d: %.3g of the bound" % (*np.unravel_index(np.argmax(r), r.shape),
                                                                             np.max(r))
    return float(np.max(r))


@pytest.mark.parametrize("k", [2, 3, 4])
@pytest.mark.parametrize("det,preset", [(0, 1), (3, 0)])
def test_pairwise_restatement_matches_f64(oracle, k, det, preset):
    n = 256
    base = uniform_noise(250 * n + 77, 3)
    xs = [(0.5 * base + uniform_noise(base.size, 10 + c) + np.float32(0.25 * c)).astype(np.float32) for c in range(k)]
    o = ocsm.CsmCascade(n, k, hbf=preset)
    o.set_detrend(det)
    o.process(xs)
    s, b = o.csm()
    t, b64 = ocsm.f64_matrix(xs, n, det, preset=preset)
    assert [bi.as_tuple() for bi in b] == tuples64(b64)
    d = np.real(np.einsum("iib->ib", t))
    for i in range(k):
        assert np.all(s[i, i].imag == 0)
        np.testing.assert_allclose(s[i, i].real, d[i], rtol=1e-4, atol=1e-6)
        for j in range(k):
            assert np.array_equal(s[j, i], np.conj(s[i, j]))
            scale = np.sqrt(d[i] * d[j])
            for part in (np.real, np.imag):
                assert np.all(np.abs(part(s[i, j]) - part(t[i, j])) <= 1e-4 * scale + 1e-6), (i, j)


def test_coherence_and_transfer_on_hand_built_matrices():
    rng = np.random.default_rng(1)
    bins = 7
    # S = A^H A per bin (Hermitian positive definite) for 3 channels
    a = rng.standard_normal((bins, 5, 3)) + 1j * rng.standard_normal((bins, 5, 3))
    S = np.moveaxis(np.conj(np.swapaxes(a, 1, 2)) @ a, 0, -1)
    coh = CsmCascade.coherence(S)
    for i in range(3):
        for j in range(3):
            np.testing.assert_allclose(coh[i, j], np.abs(S[i, j]) ** 2 / (S[i, i].real * S[j, j].real), rtol=1e-12)
    np.testing.assert_allclose(np.einsum("iib->ib", coh), 1.0, rtol=1e-12)
    # one input: CsdCascade.transfer
    h1 = CsmCascade.transfer(S, [0], [1, 2])
    assert h1.shape == (2, 1, bins)
    for o in (1, 2):
        np.testing.assert_allclose(h1[o - 1, 0], CsdCascade.transfer(S[0, 0].real, S[0, o]), rtol=1e-12)
    np.testing.assert_allclose(coh[0, 1], CsdCascade.coherence(S[0, 0].real, S[1, 1].real, S[0, 1]), rtol=1e-12)
    # two inputs, noiseless: y = H u exactly  ->  S_uy = S_uu H^T, S_yy = H S_uu H^H (conj(X_i) X_j convention)
    suu = np.moveaxis(S[:2, :2], -1, 0)
    H = rng.standard_normal((bins, 2, 2)) + 1j * rng.standard_normal((bins, 2, 2))  # [bins, out, in]
    full = np.zeros((bins, 4, 4), complex)
    full[:, :2, :2] = suu
    full[:, :2, 2:] = suu @ np.swapaxes(H, 1, 2)
    full[:, 2:, :2] = np.conj(np.swapaxes(full[:, :2, 2:], 1, 2))
    full[:, 2:, 2:] = np.conj(H) @ suu @ np.swapaxes(H, 1, 2)
    est = CsmCascade.transfer(np.moveaxis(full, 0, -1), [0, 1], [2, 3])
    np.testing.assert_allclose(np.moveaxis(est, -1, 0), H, rtol=1e-9, atol=1e-12)
    # singular input block (u1 = 2 u0) and a zero bin give 0
    sing = np.moveaxis(full, 0, -1).copy()
    sing[:, :, 3] = 0
    sing[1, 1, 2] = 4 * sing[0, 0, 2]
    sing[0, 1, 2] = sing[1, 0, 2] = 2 * sing[0, 0, 2]
    est = CsmCascade.transfer(sing, [0, 1], [2, 3])
    assert np.all(est[:, :, 2] == 0) and np.all(est[:, :, 3] == 0)
    assert np.all(CsmCascade.coherence(sing)[:, :, 3] == 0)


def test_mimo_fixture_on_the_restatement(oracle):
    xs = mimo_fixture()
    o = ocsm.CsmCascade(TF_N, 4)
    o.process(xs)
    s, b = o.csm()
    assert sum(bi.include for bi in b) >= 4
    assert_mimo(s, [(bi.include, bi.count, bi.bins_start, bi.bins_end, bi.decimation) for bi in b])
