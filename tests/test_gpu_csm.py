"""CsmCascade (cross-spectral matrix of 2 .. 4 streams) on the device against the pairwise CPU oracle (oracle.csm),
the float64 model, CsdCascade, PsdCascade and exact relations.  Needs a B200."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import uniform_noise
from oracle import csm as ocsm
from oracle import xbinding
from test_gpu_csd import assert_bins_close, assert_cross_close, btuple, RTOL
from test_oracle_csm import assert_mimo, mimo_fixture
from test_oracle_csd import TF_N

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BOUNDS = os.path.join(ROOT, "stabilizer_stream_b200", "libsspsd_bounds.so")


@pytest.fixture(scope="module")
def sp():
    import torch
    assert torch.cuda.is_available()
    import stabilizer_stream_b200 as m
    return m


def channels(k, n_samples, seed):
    """correlated channels with offsets: x_c = 0.6 common + own noise + 0.25 c"""
    base = uniform_noise(n_samples, seed)
    return [(0.6 * base + uniform_noise(n_samples, seed + 1000 * (c + 1)) + np.float32(0.25 * (c - 1))).astype(np.float32)
            for c in range(k)]


def feed(c, xs, device, seed):
    """ragged calls, every channel split identically; device=True feeds CUDA tensors (alternately as K tensors and
    as one (K, n) tensor)"""
    import torch
    rng = np.random.default_rng(seed)
    pos, i = 0, 0
    while pos < xs[0].size:
        k = int(rng.integers(0, max(8, xs[0].size // 6)))
        part = [x[pos:pos + k] for x in xs]
        if device:
            t = torch.from_numpy(np.stack(part)).cuda()
            part = t if i % 2 else list(t)
        c.process(part)
        pos += k
        i += 1


def check_matrix(c, o, det=0, xs=None, window=1, preset=1):
    """test_gpu_csd.py's rules on every entry: diagonals under the PSD rule, off-diagonals within 1e-4 sqrt(S_ii S_jj),
    breaks bit-equal; plus the matrix's exact structure (real diagonal, Hermitian)"""
    s, b = c.csm()
    so, ob = o.csm()
    k = c.channels
    assert s.shape == so.shape == (k, k, so.shape[-1])
    assert [btuple(bi) for bi in b] == [bi.as_tuple() for bi in ob]
    assert np.all(np.einsum("iib->ib", s).imag == 0)
    for i in range(k):
        for j in range(k):
            assert np.array_equal(s[j, i], np.conj(s[i, j])), (i, j)
    truth = None
    if det in (2, 3) and xs is not None:
        truth, _ = ocsm.f64_matrix(xs, c.n, det, preset=preset, win_kind=window)
    d = np.real(np.einsum("iib->ib", so)).astype(np.float64)

    def loose(i, j):
        if truth is None:
            return None, None
        t, w = truth[i, j], so[i, j].astype(np.complex128)
        m = np.zeros(w.size, bool)
        m[:2] = True
        if det == 2:
            ref = np.sqrt(np.real(truth[i, i]) * np.real(truth[j, j])) if i != j else np.abs(t)
            m |= np.abs(w - t) > 0.5 * RTOL * ref
        return m, t

    for i in range(k):
        m, t = loose(i, i)
        assert_bins_close(s[i, i].real, d[i], "S%d%d" % (i, i), m, None if t is None else t.real)
        for j in range(i + 1, k):
            m, t = loose(i, j)
            assert_cross_close(s[i, j], so[i, j], d[i], d[j], "S%d%d" % (i, j), m, t)
    return s, b


# ---- 1. device against the pairwise oracle ----
CASES = [(k, n, det, (det + ni) % 2) for k in (2, 3, 4) for ni, n in enumerate((64, 512, 2048, 4096))
         for det in (0, 1, 2, 3)]


@pytest.mark.parametrize("k,n,det,preset", CASES)
def test_oracle_parity(sp, oracle, k, n, det, preset):
    xs = channels(k, 150 * n + 77, n + det + k)
    c = sp.CsmCascade(n, k, hbf=sp.Hbf(preset))
    c.set_detrend(sp.Detrend(det))
    o = ocsm.CsmCascade(n, k, hbf=preset)
    o.set_detrend(det)
    feed(c, xs, device=(det % 2 == 1), seed=n + det)
    o.process(xs)
    assert c.num_stages() == o.num_stages() >= 2
    check_matrix(c, o, det, xs, preset=preset)


@pytest.mark.parametrize("k", [3, 4])
def test_oracle_parity_rectangular(sp, oracle, k):
    n = 1024
    xs = channels(k, n * 40 + 5, 3)
    c = sp.CsmCascade(n, k, window=sp.Window.RECTANGULAR)
    o = ocsm.CsmCascade(n, k, window=xbinding.WINDOW_RECT)
    feed(c, xs, device=False, seed=2)
    o.process(xs)
    check_matrix(c, o)


@pytest.mark.parametrize("k", [3, 4])
def test_ragged_host_and_device(sp, oracle, k):
    import torch
    n = 512
    xs = channels(k, 3_000_000 + 3, 17)
    c = sp.CsmCascade(n, k, host_stage=1 << 16)
    o = ocsm.CsmCascade(n, k)
    rng = np.random.default_rng(5)
    pos, i = 0, 0
    while pos < xs[0].size:
        m = int(rng.choice([0, 1, 3, 4096, 100_003, 700_001]))
        part = [x[pos:pos + m] for x in xs]
        if i % 3 == 2:
            part = [torch.from_numpy(p.copy()).cuda() for p in part]
        c.process(part)
        pos += m
        i += 1
    o.process(xs)
    check_matrix(c, o)


# ---- 2. bit-exact relations (deterministic accumulation) ----
@pytest.mark.parametrize("n", [512, 4096])
def test_k2_is_the_csd_and_block00_of_k4_too(sp, n):
    import torch
    xs = channels(4, 3_000_000 + 11, n)
    xd = [torch.from_numpy(x).cuda() for x in xs]
    d = sp.CsdCascade(n, deterministic=True)
    d.process(xd[0], xd[1])
    pxx, pyy, pxy, bd = d.csd()
    for k in (2, 4):
        c = sp.CsmCascade(n, k, deterministic=True)
        c.process(xd[:k])
        s, b = c.csm()
        assert [btuple(bi) for bi in b] == [btuple(bi) for bi in bd]
        assert np.array_equal(s[0, 0].real, pxx), k
        assert np.array_equal(s[1, 1].real, pyy), k
        assert np.array_equal(s[0, 1].view(np.uint32), pxy.view(np.uint32)), k


@pytest.mark.parametrize("k", [3, 4])
def test_diagonal_is_the_psd(sp, k):
    n = 512
    xs = channels(k, 2_000_000 + 9, k)
    c = sp.CsmCascade(n, k)
    c.process(xs)
    s, b = c.csm()
    for i in range(k):
        p = sp.PsdCascade(n)
        p.process(xs[i])
        pp, bp = p.psd()
        assert [btuple(bi) for bi in b] == [btuple(bi) for bi in bp]
        assert_bins_close(s[i, i].real, pp, "S%d%d vs PsdCascade" % (i, i))


def test_power_of_two_scaling_is_exact(sp):
    n = 1024
    xs = channels(4, 1_500_000, 23)
    out = []
    for a in (0, 7, -5):
        c = sp.CsmCascade(n, 4, deterministic=True)
        c.process([(x * np.float32(2.0 ** a)).astype(np.float32) for x in xs])
        out.append((a, c.csm()[0]))
    for a, s in out[1:]:
        assert np.array_equal(s, (out[0][1] * np.float32(2.0 ** (2 * a))).astype(np.complex64)), a


# ---- 3. cross-block relations ----
@pytest.mark.parametrize("n", [64, 512, 4096])
@pytest.mark.parametrize("deterministic", [True, False])
def test_cross_block_relations(sp, n, deterministic):
    """channels (x, u, 2x, -u): S02 = 2 S00, S13 = -S11, S03 = -S01, S12 = 2 conj(S01).  The two sides come from
    different FFTs (pair (0, 1) and pair (2, 3) run through separate transforms) and, for S03 and S12, from different
    kernels, so they differ by f32 transform rounding.  Measured on a B200 at N = 64, 512, 4096: at most 4.2e-7 of
    sqrt(S_ii S_jj) with fixed-order accumulation, bound 1e-6; at most 5.8e-6 with the default atomic flush, which
    adds the two sides' partial sums in different orders, bound 2e-5.  A swapped product, a wrong sign or split
    constant in the cross kernel is off by O(1)."""
    tol = 1e-6 if deterministic else 2e-5
    x, u = uniform_noise(1_000_000, 77), uniform_noise(1_000_000, 78)
    c = sp.CsmCascade(n, 4, deterministic=deterministic)
    c.process([x, u, (2 * x).astype(np.float32), (-u).astype(np.float32)])
    s, _ = c.csm()
    s = s.astype(np.complex128)
    d = np.real(np.einsum("iib->ib", s))
    worst = {}
    for (i, j), want in (((0, 2), 2 * s[0, 0]), ((1, 3), -s[1, 1]), ((0, 3), -s[0, 1]), ((1, 2), 2 * np.conj(s[0, 1]))):
        scale = np.sqrt(d[i] * d[j])
        e = np.maximum(np.abs(s[i, j].real - want.real), np.abs(s[i, j].imag - want.imag)) / scale
        worst[(i, j)] = float(np.max(e))
    print("cross-block relations, worst relative deviation:", worst)
    assert max(worst.values()) <= tol, worst


# ---- 4. tone between channels 0 and 2 ----
@pytest.mark.parametrize("n", [512, 4096])
@pytest.mark.parametrize("f0,dec", [(0.1234567, 1), (0.0031234, 64)])
def test_tone_phase_and_amplitude(sp, n, f0, dec):
    m = 1 << 23
    t = np.arange(m, dtype=np.float64)
    x0 = (np.cos(2 * np.pi * f0 * t + 0.2) + 1e-5 * uniform_noise(m, 1)).astype(np.float32)
    x2 = (0.3 * np.cos(2 * np.pi * f0 * t + 1.2) + 1e-5 * uniform_noise(m, 2)).astype(np.float32)
    c = sp.CsmCascade(n, 4)
    c.process([x0, uniform_noise(m, 3), x2, uniform_noise(m, 4)])
    s, b = c.csm()
    bk = [bi for bi in b if bi.decimation == dec and bi.include][0]
    sl = slice(bk.start, bk.start + bk.bins.stop - bk.bins.start)
    p0 = s[0, 0].real
    k = bk.start + int(np.argmax(p0[sl]))
    assert abs((k - bk.start + bk.bins.start) / (n * dec) - f0) <= 1.0 / (n * dec)
    assert abs(np.angle(s[0, 2, k]) - 1.0) <= 1e-4
    assert abs(abs(s[0, 2, k]) / p0[k] - 0.3) <= 1e-4
    assert abs(np.angle(s[2, 0, k]) + 1.0) <= 1e-4


# ---- 5. the MIMO fixture ----
def test_mimo_transfer_matrix(sp):
    import torch
    xs = mimo_fixture()
    c = sp.CsmCascade(TF_N, 4)
    c.process(torch.from_numpy(np.stack(xs)).cuda())
    s, b = c.csm()
    t, b64 = ocsm.f64_matrix(xs, TF_N)
    d = np.real(np.einsum("iib->ib", t))
    for i in range(4):
        assert_bins_close(s[i, i].real, d[i], "S%d%d vs f64" % (i, i))
        for j in range(i + 1, 4):
            assert_cross_close(s[i, j], t[i, j], d[i], d[j], "S%d%d vs f64" % (i, j))
    r = assert_mimo(s, [(bi.include, bi.count, bi.bins.start, bi.bins.stop, bi.decimation) for bi in b])
    print("MIMO fixture: worst error %.2f of the bound" % r)


# ---- 6. API behaviour ----
@pytest.mark.parametrize("n", [512, 4096])
def test_deterministic_bit_identical(sp, n):
    import torch
    xd = torch.from_numpy(np.stack(channels(4, 3_000_000, 31))).cuda()
    out = []
    for _ in range(2):
        c = sp.CsmCascade(n, 4, deterministic=True)
        c.process(xd)
        out.append(c.csm()[0])
    assert np.array_equal(out[0].view(np.uint32), out[1].view(np.uint32))


@pytest.mark.parametrize("k", [3, 4])
def test_midstream_avg_and_detrend(sp, oracle, k):
    n = 512
    xs = channels(k, 1_500_000, 41)
    c = sp.CsmCascade(n, k)
    o = ocsm.CsmCascade(n, k)
    a, b = 400_003, 900_001
    c.process([x[:a] for x in xs]); o.process([x[:a] for x in xs])
    c.set_avg(sp.AvgOpts(limit=999, count=2 ** 32 - 2)); o.set_avg(999, 2 ** 32 - 2)
    c.process([x[a:b] for x in xs]); o.process([x[a:b] for x in xs])
    c.set_detrend(sp.Detrend.MIDPOINT); o.set_detrend(1)
    c.set_avg(sp.AvgOpts(limit=50, count=400)); o.set_avg(50, 400)
    c.process([x[b:] for x in xs]); o.process([x[b:] for x in xs])
    check_matrix(c, o)


def test_reset_clone_and_empty_calls(sp, oracle):
    n = 1024
    k = 4
    xs = channels(k, 700_000, 43)
    c = sp.CsmCascade(n, k)
    c.process([x[:0] for x in xs])
    assert c.num_stages() == 0
    s, b = c.csm()
    assert s.shape == (k, k, 0) and b == []
    c.process([x[:300_000] for x in xs])
    d = c.clone()
    assert d.channels == k
    c.process([x[300_000:] for x in xs])
    d.process([x[300_000:] for x in xs])
    (s1, b1), (s2, b2) = c.csm(), d.csm()
    assert [btuple(bi) for bi in b1] == [btuple(bi) for bi in b2]
    for i in range(k):
        for j in range(k):
            assert_bins_close(np.abs(s1[i, j]), np.abs(s2[i, j]), "clone S%d%d" % (i, j))
    c.reset()
    assert c.num_stages() == 0
    c.process(xs)
    o = ocsm.CsmCascade(n, k)
    o.process(xs)
    check_matrix(c, o)


def test_device_input_on_another_torch_stream(sp, oracle):
    import torch
    n = 512
    xs = channels(3, 2_000_000, 47)
    c = sp.CsmCascade(n, 3)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        xd = torch.from_numpy(np.stack(xs)).cuda() * 1.0
        c.process(xd)
        del xd
    o = ocsm.CsmCascade(n, 3)
    o.process(xs)
    check_matrix(c, o)


# ---- 7. the bounds-checking build over cases 1 and 6 ----
@pytest.mark.skipif(bool(os.environ.get("SSPSD_LIB")), reason="already running against another build")
def test_bounds_build():
    if not os.path.exists(BOUNDS):
        pytest.skip("libsspsd_bounds.so not built")
    env = dict(os.environ, SSPSD_LIB=BOUNDS)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "tests"), env.get("PYTHONPATH", "")])
    r = subprocess.run([sys.executable, "-m", "pytest", "-m", "gpu", "-x", "-q", os.path.abspath(__file__), "-k",
                        "oracle_parity or ragged or deterministic_bit or midstream or reset_clone or another_torch_stream"],
                       env=env, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]


# ---- 8. error paths ----
def test_error_paths(sp):
    import ctypes as C
    from stabilizer_stream_b200 import _lib as L
    for k in (0, 1, 5):
        with pytest.raises(L.SspsdError) as e:
            sp.CsmCascade(512, k)
        assert e.value.status == L.EINVAL
    with pytest.raises(L.SspsdError) as e:
        sp.CsmCascade(8192, 4)
    assert e.value.status == L.EINVAL and "4096" in str(e.value)
    c = sp.CsmCascade(512, 3)
    with pytest.raises(L.SspsdError) as e:
        c.set_detrend(sp.Detrend.LINEAR)
    assert e.value.status == L.EUNIMPLEMENTED
    with pytest.raises(ValueError):
        c.process([np.zeros(8, np.float32)] * 2)
    with pytest.raises(ValueError):
        c.process([np.zeros(8, np.float32), np.zeros(8, np.float32), np.zeros(9, np.float32)])
    lib = L.lib()
    cfg = L.Config()
    L.check(lib.sspsd_config_default(8192, C.byref(cfg)))
    h = C.c_void_p()
    assert lib.sspsd_csm_create(C.byref(cfg), 4, C.byref(h)) == L.EINVAL and not h.value
    L.check(lib.sspsd_config_default(512, C.byref(cfg)))
    assert lib.sspsd_csm_create(C.byref(cfg), 5, C.byref(h)) == L.EINVAL and not h.value
    assert lib.sspsd_csm_create(None, 4, C.byref(h)) == L.EINVAL
    assert lib.sspsd_csm_process_f32(None, None, 0, L.MEM_HOST) == L.EINVAL
    assert lib.sspsd_csm_process_f32(c._h, None, 16, L.MEM_HOST) == L.EINVAL
    x = np.zeros(16, np.float32)
    ptrs = (C.c_void_p * 3)(x.ctypes.data, None, x.ctypes.data)
    assert lib.sspsd_csm_process_f32(c._h, ptrs, 16, L.MEM_HOST) == L.EINVAL
    assert lib.sspsd_csm_set_detrend(c._h, 4) == L.EUNIMPLEMENTED
    assert lib.sspsd_csm_read(c._h, None, None, None, None, None) == L.EINVAL
    assert lib.sspsd_csm_num_stages(None, None) == L.EINVAL
    assert lib.sspsd_csm_sync(None) == L.EINVAL
    # short capacity: SSPSD_ESHORT with the lengths needed
    xs = channels(3, 20_000, 5)
    c.process(xs)
    pl, bl = C.c_size_t(1), C.c_size_t(8)
    b = (L.BreakC * 8)()
    s = np.zeros(2 * 9, np.float32)
    assert lib.sspsd_csm_read(c._h, None, s.ctypes.data, C.byref(pl), b, C.byref(bl)) == L.ESHORT
    assert pl.value == c.csm()[0].shape[-1] > 1
