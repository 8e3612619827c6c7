"""CsdCascade (cross-spectral density of two streams) on the device against the CPU oracle (oracle.xbinding.XCascade),
the float64 model, PsdCascade and exact relations.  Needs a B200."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import uniform_noise
from oracle import model_f64_csd as mcsd
from oracle import xbinding
from test_oracle_csd import TF_N, transfer_expected, transfer_fixture, transfer_tolerance

pytestmark = pytest.mark.gpu

RTOL = 1e-4    # per-bin rule of tests/test_gpu_psd.py
AFLOOR = 1e-5
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BOUNDS = os.path.join(ROOT, "stabilizer_stream_b200", "libsspsd_bounds.so")


@pytest.fixture(scope="module")
def sp():
    import torch
    assert torch.cuda.is_available()
    import stabilizer_stream_b200 as m
    return m


def assert_bins_close(got, want, what="", loose=None, truth=None):
    """tests/test_gpu_psd.py's rule: 1e-4 per bin above a floor of 1e-5 x median.  Bins in the mask `loose` (DC under
    Span / Mean detrend; under Span also wherever the oracle's own sequentially accumulated f32 trend line is off the
    float64 truth by more than 5e-5) must instead be at least as close to the float64 truth as the oracle is."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert got.shape == want.shape, what
    if want.size == 0:
        return
    err = np.abs(got - want) - AFLOOR * np.median(np.abs(want))
    rel = err / np.maximum(np.abs(want), 1e-300)
    if loose is not None:
        truth = np.asarray(truth, np.float64)
        dg, do = np.abs(got[loose] - truth[loose]), np.abs(want[loose] - truth[loose])
        assert np.all(dg <= do + RTOL * np.median(np.abs(truth))), "%s: loose bins %s > %s" % (what, dg, do)
        rel = rel[~loose]
    assert rel.size == 0 or np.max(rel) <= RTOL, "%s: max rel err %.3g at %d" % (what, np.max(rel), np.argmax(rel))


def assert_cross_close(got, want, pxx, pyy, what="", loose=None, truth=None):
    """|got - want| <= 1e-4 sqrt(pxx pyy) + floor on the real and imaginary parts (Cauchy-Schwarz scale: |pxy| of
    uncorrelated bins is ~0, a relative error on it means nothing); `loose` as in assert_bins_close"""
    got, want = np.asarray(got, np.complex128), np.asarray(want, np.complex128)
    assert got.shape == want.shape, what
    if want.size == 0:
        return
    scale = np.sqrt(np.asarray(pxx, np.float64) * np.asarray(pyy, np.float64))
    tol = RTOL * scale + AFLOOR * np.median(scale)
    for part in (np.real, np.imag):
        e = np.abs(part(got) - part(want))
        if loose is not None:
            t = part(np.asarray(truth, np.complex128))
            dg, do = np.abs(part(got) - t)[loose], np.abs(part(want) - t)[loose]
            assert np.all(dg <= do + RTOL * np.median(scale)), "%s: loose bins %s > %s" % (what, dg, do)
            e, tl = e[~loose], tol[~loose]
        else:
            tl = tol
        assert np.all(e <= tl), "%s: worst excess %.3g" % (what, np.max(e - tl))


def btuple(b):
    return (b.start, b.include, b.count, b.avg, b.bins.start, b.bins.stop, b.fft_size, b.decimation, b.pending,
            b.processed)


def pair(n_samples, seed):
    """correlated inputs with an offset: y = 0.6 x + independent noise"""
    x = uniform_noise(n_samples, seed) + np.float32(0.25)
    y = (0.6 * x + uniform_noise(n_samples, seed + 1000)).astype(np.float32)
    return x, y


def feed(sp, c, x, y, device, seed):
    """ragged calls, x and y split identically; device=True feeds CUDA tensors"""
    import torch
    rng = np.random.default_rng(seed)
    pos = 0
    while pos < x.size:
        k = int(rng.integers(0, max(8, x.size // 6)))
        a, b = x[pos:pos + k], y[pos:pos + k]
        if device:
            a, b = torch.from_numpy(a.copy()).cuda(), torch.from_numpy(b.copy()).cuda()
        c.process(a, b)
        pos += k


def check_against_oracle(sp, oracle, c, o, det=0, x=None, y=None, window=1, preset=1):
    pxx, pyy, pxy, b = c.csd()
    oxx, oyy, oxy, ob = o.csd()
    assert [btuple(bi) for bi in b] == [bi.as_tuple() for bi in ob]
    masks, truths = [None] * 3, [None] * 3
    if det in (2, 3) and x is not None:
        n = c.n
        truths = mcsd.merge_cross(mcsd.cross_cascade(x, y, n, det, preset=preset, win_kind=window), n)[:3]
        for i, (w, t) in enumerate(zip((oxx, oyy, oxy), truths)):
            m = np.zeros(w.size, bool)
            m[:2] = True
            if det == 2:
                ref = np.sqrt(truths[0] * truths[1]) if i == 2 else np.abs(t)
                m |= np.abs(w - t) > 0.5 * RTOL * ref
            masks[i] = m
    assert_bins_close(pxx, oxx, "pxx", masks[0], truths[0])
    assert_bins_close(pyy, oyy, "pyy", masks[1], truths[1])
    assert_cross_close(pxy, oxy, oxx, oyy, "pxy", masks[2], truths[2])
    return pxx, pyy, pxy, b


# ---- 1. device against the oracle ----
@pytest.mark.parametrize("preset", [0, 1])
@pytest.mark.parametrize("det", [0, 1, 2, 3])
@pytest.mark.parametrize("n", [64, 512, 1024, 4096])
def test_oracle_parity(sp, oracle, n, det, preset):
    x, y = pair(150 * n + 77, n + det)
    c = sp.CsdCascade(n, hbf=sp.Hbf(preset))
    c.set_detrend(sp.Detrend(det))
    o = xbinding.XCascade(n, hbf=preset)
    o.set_detrend(det)
    feed(sp, c, x, y, device=(det % 2 == 1), seed=n + det)
    o.process(x, y)
    assert c.num_stages() == o.num_stages() >= 2
    check_against_oracle(sp, oracle, c, o, det, x, y, preset=preset)


def test_oracle_parity_rectangular(sp, oracle):
    n = 1024
    x, y = pair(n * 40 + 5, 3)
    c = sp.CsdCascade(n, window=sp.Window.RECTANGULAR)
    o = xbinding.XCascade(n, window=xbinding.WINDOW_RECT)
    feed(sp, c, x, y, device=False, seed=2)
    o.process(x, y)
    pxx, _, _, b = check_against_oracle(sp, oracle, c, o)
    # and the stage-0 spectrum of x is what the single-stage Psd computes with the same window
    g = sp.Psd(n, sp.Window.RECTANGULAR)
    g.process(x)
    s0 = [bi for bi in b if bi.decimation == 1][0]
    row = g.spectrum()[s0.bins.start:s0.bins.stop] / (g.gain() * 1.0)
    assert_bins_close(pxx[s0.start:s0.start + row.size], row, "rect stage 0 vs Psd")


def test_ragged_host_and_device(sp, oracle):
    n = 512
    x, y = pair(3_000_000 + 3, 17)
    c = sp.CsdCascade(n, host_stage=1 << 16)
    o = xbinding.XCascade(n)
    import torch
    rng = np.random.default_rng(5)
    pos, i = 0, 0
    while pos < x.size:
        k = int(rng.choice([0, 1, 3, 4096, 100_003, 700_001]))
        a, b = x[pos:pos + k], y[pos:pos + k]
        if i % 3 == 2:
            a, b = torch.from_numpy(a.copy()).cuda(), torch.from_numpy(b.copy()).cuda()
        c.process(a, b)
        pos += k
        i += 1
    o.process(x, y)
    check_against_oracle(sp, oracle, c, o)


# ---- 2. against PsdCascade ----
@pytest.mark.parametrize("n", [512, 4096])
def test_pxx_is_the_psd(sp, n):
    x, y = pair(2_000_000 + 9, n)
    c = sp.CsdCascade(n)
    c.process(x, y)
    p = sp.PsdCascade(n)
    p.process(x)
    pxx, _, _, b = c.csd()
    pp, bp = p.psd()
    assert [btuple(bi) for bi in b] == [btuple(bi) for bi in bp]
    assert_bins_close(pxx, pp, "pxx vs PsdCascade")


# ---- 3. exact relations ----
@pytest.mark.parametrize("deterministic", [True, False])
def test_exact_relations(sp, deterministic):
    """y = x, -x, 2x.  With fixed-order accumulation the relations hold to 1e-6 per bin.  The default flush adds each
    row's per-CTA partial sums with float atomics in whatever order the CTAs finish, independently for every row, so
    pxx and Re pxy carry different summation rounding (a few 1e-7, occasionally above 1e-6): 1e-5 there.  Either
    bound catches a wrong split constant or swapped X and Y."""
    n = 512
    tol = 1e-6 if deterministic else 1e-5
    x = uniform_noise(1_000_000, 77)
    for k in (1.0, -1.0, 2.0):
        c = sp.CsdCascade(n, deterministic=deterministic)
        c.process(x, (k * x).astype(np.float32))
        pxx, pyy, pxy, _ = c.csd()
        assert np.all(np.abs(pxy.real - k * pxx) <= tol * abs(k) * pxx), k
        assert np.all(np.abs(pxy.imag) <= tol * abs(k) * pxx), k
        assert np.all(np.abs(pyy - k * k * pxx) <= tol * k * k * pxx), k


# ---- 4. tone ----
@pytest.mark.parametrize("n", [512, 4096])
@pytest.mark.parametrize("f0,dec", [(0.1234567, 1), (0.0031234, 64)])
def test_tone_phase_and_amplitude(sp, n, f0, dec):
    m = 1 << 23
    t = np.arange(m, dtype=np.float64)
    x = (np.cos(2 * np.pi * f0 * t + 0.2) + 1e-5 * uniform_noise(m, 1)).astype(np.float32)
    y = (0.3 * np.cos(2 * np.pi * f0 * t + 1.2) + 1e-5 * uniform_noise(m, 2)).astype(np.float32)
    c = sp.CsdCascade(n)
    c.process(x, y)
    pxx, pyy, pxy, b = c.csd()
    bk = [bi for bi in b if bi.decimation == dec and bi.include][0]
    sl = slice(bk.start, bk.start + bk.bins.stop - bk.bins.start)
    k = bk.start + int(np.argmax(pxx[sl]))
    assert abs((k - bk.start + bk.bins.start) / (n * dec) - f0) <= 1.0 / (n * dec)
    assert abs(np.angle(pxy[k]) - 1.0) <= 1e-4
    assert abs(abs(pxy[k]) / pxx[k] - 0.3) <= 1e-4


# ---- 5. transfer function through the whole cascade ----
def test_transfer_function(sp):
    import torch
    x, y = transfer_fixture()
    c = sp.CsdCascade(TF_N)
    c.process(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda())
    pxx, pyy, pxy, b = c.csd()
    tx, ty, txy, b64 = mcsd.merge_cross(mcsd.cross_cascade(x, y, TF_N), TF_N)
    assert [btuple(bi) for bi in b] == [(d["start"], d["include"], d["count"], d["avg"], d["bins"][0], d["bins"][1],
                                         d["fft_size"], d["decimation"], d["pending"], d["processed"]) for d in b64]
    assert_bins_close(pxx, tx, "pxx vs f64")
    assert_bins_close(pyy, ty, "pyy vs f64")
    assert_cross_close(pxy, txy, tx, ty, "pxy vs f64")
    h, dec, cnt = transfer_expected([(bi.include, bi.count, bi.bins.start, bi.bins.stop, bi.decimation) for bi in b])
    pxx, pyy, pxy = pxx.astype(np.float64), pyy.astype(np.float64), pxy.astype(np.complex128)
    coh = sp.CsdCascade.coherence(pxx, pyy, pxy)
    err = np.abs(sp.CsdCascade.transfer(pxx, pxy) - h)
    tol = transfer_tolerance(h, dec, cnt, coh)
    assert np.all(err <= tol), "worst bin %d: %.3g > %.3g" % (np.argmax(err / tol), np.max(err), tol[np.argmax(err / tol)])


# ---- 6. deterministic mode ----
@pytest.mark.parametrize("n", [512, 4096])
def test_deterministic_bit_identical(sp, n):
    import torch
    x, y = pair(4_000_000, 31)
    xd, yd = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    out = []
    for _ in range(2):
        c = sp.CsdCascade(n, deterministic=True)
        c.process(xd, yd)
        out.append(c.csd())
    for a, b in zip(out[0][:3], out[1][:3]):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))


# ---- 7. mid-stream changes, reset / clone / empty calls, torch streams ----
def test_midstream_avg_and_detrend(sp, oracle):
    n = 512
    x, y = pair(1_500_000, 41)
    c = sp.CsdCascade(n)
    o = xbinding.XCascade(n)
    a, b = 400_003, 900_001
    c.process(x[:a], y[:a]); o.process(x[:a], y[:a])
    c.set_avg(sp.AvgOpts(limit=999, count=2 ** 32 - 2)); o.set_avg(999, 2 ** 32 - 2)  # the psd binary's EWMA preset
    c.process(x[a:b], y[a:b]); o.process(x[a:b], y[a:b])
    c.set_detrend(sp.Detrend.MIDPOINT); o.set_detrend(1)
    c.set_avg(sp.AvgOpts(limit=50, count=400)); o.set_avg(50, 400)
    c.process(x[b:], y[b:]); o.process(x[b:], y[b:])
    check_against_oracle(sp, oracle, c, o)


def test_reset_clone_and_empty_calls(sp, oracle):
    n = 1024
    x, y = pair(700_000, 43)
    c = sp.CsdCascade(n)
    c.process(x[:0], y[:0])
    assert c.num_stages() == 0
    pxx, pyy, pxy, b = c.csd()
    assert pxx.size == pyy.size == pxy.size == 0 and b == []
    c.process(x[:300_000], y[:300_000])
    d = c.clone()
    c.process(x[300_000:], y[300_000:])
    d.process(x[300_000:], y[300_000:])
    r1, r2 = c.csd(), d.csd()
    for u, v in zip(r1[:3], r2[:3]):
        assert_bins_close(np.abs(u), np.abs(v), "clone")
    assert [btuple(bi) for bi in r1[3]] == [btuple(bi) for bi in r2[3]]
    c.reset()
    assert c.num_stages() == 0
    c.process(x, y)
    o = xbinding.XCascade(n)
    o.process(x, y)
    check_against_oracle(sp, oracle, c, o)


def test_device_input_on_another_torch_stream(sp, oracle):
    import torch
    n = 512
    x, y = pair(2_000_000, 47)
    c = sp.CsdCascade(n)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        xd = torch.from_numpy(x).cuda() * 1.0
        yd = torch.from_numpy(y).cuda() * 1.0
        c.process(xd, yd)
        del xd, yd
    o = xbinding.XCascade(n)
    o.process(x, y)
    check_against_oracle(sp, oracle, c, o)


# ---- 8. the bounds-checking build over cases 1 and 7 ----
@pytest.mark.skipif(bool(os.environ.get("SSPSD_LIB")), reason="already running against another build")
def test_bounds_build():
    if not os.path.exists(BOUNDS):
        pytest.skip("libsspsd_bounds.so not built")
    env = dict(os.environ, SSPSD_LIB=BOUNDS)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "tests"), env.get("PYTHONPATH", "")])
    r = subprocess.run([sys.executable, "-m", "pytest", "-m", "gpu", "-x", "-q", os.path.abspath(__file__), "-k",
                        "oracle_parity or ragged or midstream or reset_clone or another_torch_stream"],
                       env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]


# ---- 9. error paths ----
def test_error_paths(sp):
    import ctypes as C
    from stabilizer_stream_b200 import _lib as L
    with pytest.raises(L.SspsdError) as e:
        sp.CsdCascade(8192)
    assert e.value.status == L.EINVAL and "4096" in str(e.value)
    c = sp.CsdCascade(512)
    with pytest.raises(L.SspsdError) as e:
        c.set_detrend(sp.Detrend.LINEAR)
    assert e.value.status == L.EUNIMPLEMENTED
    lib = L.lib()
    cfg = L.Config()
    L.check(lib.sspsd_config_default(8192, C.byref(cfg)))
    h = C.c_void_p()
    assert lib.sspsd_csd_create(C.byref(cfg), C.byref(h)) == L.EINVAL and not h.value
    assert lib.sspsd_csd_create(None, C.byref(h)) == L.EINVAL
    assert lib.sspsd_csd_process_f32(None, None, None, 0, L.MEM_HOST) == L.EINVAL
    assert lib.sspsd_csd_process_f32(c._h, None, None, 16, L.MEM_HOST) == L.EINVAL
    assert lib.sspsd_csd_set_detrend(c._h, 4) == L.EUNIMPLEMENTED
    assert lib.sspsd_csd_read(c._h, None, None, None, None, None, None, None) == L.EINVAL
    assert lib.sspsd_csd_num_stages(None, None) == L.EINVAL
    assert lib.sspsd_csd_sync(None) == L.EINVAL
