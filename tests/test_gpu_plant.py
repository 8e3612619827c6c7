"""Plants on the device (sspsd_plant_*, DESIGN.md 3d): generation against the CPU restatement (oracle/sspsd_poracle.c),
process_plant of every handle kind against process() of the generated arrays, the long-run known answer of the cross
kinds against Plant.expected_csm, and time-chunked groups of every kind fed by time_process_plant."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import pbinding
from test_gpu_group import breaks_tuple, device_lists
from test_oracle_csm import mimo_tolerance
from test_oracle_plant import csm_bound, rounding_floor, spread

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BOUNDS = os.path.join(ROOT, "stabilizer_stream_b200", "libsspsd_bounds.so")
FTW = 0x9E3779B9


@pytest.fixture(scope="module")
def sp():
    import torch
    assert torch.cuda.is_available()
    import stabilizer_stream_b200 as m
    return m


def taps_of(k, m, nt, seed):
    return np.random.default_rng(seed).standard_normal((k, m, nt)).astype(np.float32)


def noise_inputs(sp, m, seed):
    return [sp.Plant.noise((0, 1, 3)[(seed + q) % 3], seed * 7 + q) for q in range(m)]


def ulps(a, b):
    a = np.asarray(a, np.float32).view(np.int32).astype(np.int64)
    b = np.asarray(b, np.float32).view(np.int32).astype(np.int64)
    a = np.where(a < 0, -(a & 0x7FFFFFFF), a)
    b = np.where(b < 0, -(b & 0x7FFFFFFF), b)
    return np.abs(a - b)


# ---- 1. generation ----
@pytest.mark.parametrize("k", [1, 2, 3, 4])
@pytest.mark.parametrize("m", [1, 2, 3, 4])
@pytest.mark.parametrize("nt", [1, 7, 32])
def test_generation_noise_bit_exact(sp, k, m, nt):
    taps = taps_of(k, m, nt, 100 * k + 10 * m + nt)
    ins = noise_inputs(sp, m, k + m + nt)
    p = sp.Plant(taps, ins)
    n, pos = 9000, 70_001
    p.seek(pos)
    got = p.generate(n).cpu().numpy()
    want = pbinding.plant(taps, ins, n, pos=pos)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert p.position() == pos + n


def test_generation_tones_within_one_ulp(sp):
    taps = taps_of(3, 4, 9, 5)
    ins = [sp.Plant.tone(FTW, 0.75), sp.Plant.noise(1, 3), sp.Plant.tone(0x40000000, -2.0), sp.Plant.tone(12345, 1.0)]
    p = sp.Plant(taps, ins)
    got = p.generate(40_000).cpu().numpy()
    want = pbinding.plant(taps, ins, 40_000)
    assert ulps(got, want).max() <= 1


def test_identity_plant_is_the_source(sp):
    for e in (0, 1, 3, 8):
        p = sp.Plant(np.ones((1, 1, 1)), [sp.Plant.noise(e, 77)])
        s = sp.Source.noise(e, 77)
        a, b = p.generate(1_000_003)[0], s.get(1_000_003)
        assert np.array_equal(a.cpu().numpy().view(np.uint32), b.cpu().numpy().view(np.uint32))


def test_ragged_calls_and_seek_equal_one_generation(sp):
    import torch
    taps = taps_of(4, 3, 32, 9)
    ins = [sp.Plant.noise(3, 1), sp.Plant.tone(FTW, 1.0), sp.Plant.noise(0, 2)]
    p = sp.Plant(taps, ins)
    total = 3_000_000
    ref = p.generate(total).clone()
    p.reset()
    parts, done = [], 0
    for n in (1, 3, 30, 1021, 4097, 999_999, total):
        n = min(n, total - done)
        parts.append(p.generate(n).clone())
        done += n
        if done == total:
            break
    assert torch.equal(torch.cat(parts, dim=1), ref)
    for pos in (0, 1, 5, 17, 31, 33, 1023, 1024, 1025, 2_000_001):   # inside the first L - 1 samples too
        p.seek(pos)
        assert torch.equal(p.generate(777), ref[:, pos:pos + 777]), pos
    # an unaligned output buffer takes the scalar stores
    out = torch.zeros((4, 5001), dtype=torch.float32, device="cuda:0")
    p.seek(10)
    p.generate(5000, out=out[:, 1:])
    assert torch.equal(out[:, 1:], ref[:, 10:5010])


# ---- 2. consumers ----
def handle(sp, kind, n):
    kw = dict(deterministic=True)
    if kind == "psd":
        return sp.PsdCascade(n, **kw), 1
    if kind == "csd":
        return sp.CsdCascade(n, **kw), 2
    if kind.startswith("csm"):
        return sp.CsmCascade(n, int(kind[3]), **kw), int(kind[3])
    if kind == "zoom_iq":
        return sp.ZoomCascade.iq(n, **kw), 2
    return sp.ZoomCascade.heterodyne(n, FTW, **kw), 1


def read(h, kind):
    if kind == "psd":
        p, b = h.psd()
        return [p], b
    if kind == "csd":
        pxx, pyy, pxy, b = h.csd()
        return [pxx, pyy, pxy], b
    if kind.startswith("csm"):
        s, b = h.csm()
        return [s], b
    pp, pn, b = h.spectrum()
    return [pp, pn], b


@pytest.mark.parametrize("kind", ["psd", "csd", "csm2", "csm3", "csm4", "zoom_iq", "zoom_het"])
def test_process_plant_equals_process_of_generated(sp, kind):
    n = 512
    a, k = handle(sp, kind, n)
    b, _ = handle(sp, kind, n)
    taps = taps_of(k, 2, 5, 11)
    ins = [sp.Plant.noise(0, 4), sp.Plant.noise(1, 5)]
    pa, pb = sp.Plant(taps, ins), sp.Plant(taps, ins)
    slice_ = 1 << 24   # process_plant's slice: the same calls on both sides
    for n_ in (1, 4093, 3, 2_000_001, 17_000_003, 123):   # ragged, and past one slice
        a.process_plant(pa, n_)
        for lo in range(0, n_, slice_):
            y = pb.generate(min(slice_, n_ - lo)).clone()
            if kind.startswith("csm"):
                b.process(list(y))
            elif k > 1:
                b.process(y[0], y[1])
            else:
                b.process(y[0])
    ra, ba = read(a, kind)
    rb, bb = read(b, kind)
    assert [breaks_tuple(x) for x in ba] == [breaks_tuple(x) for x in bb]
    for x, y in zip(ra, rb):
        assert np.array_equal(x, y)


def test_k_mismatch_and_device_checks(sp):
    from stabilizer_stream_b200._lib import SspsdError, EINVAL
    p = sp.Plant(taps_of(3, 1, 1, 0), [sp.Plant.noise()])
    for h in (sp.PsdCascade(512), sp.CsdCascade(512), sp.CsmCascade(512, 2), sp.ZoomCascade.iq(512),
              sp.ZoomCascade.heterodyne(512, 5)):
        with pytest.raises(SspsdError) as e:
            h.process_plant(p, 1000)
        assert e.value.status == EINVAL
    assert p.position() == 0  # nothing consumed


# ---- 3. known answer at length ----
def bins(breaks):
    f, cnt, dec = [], [], []
    for b in breaks:
        if b.include:
            f.extend(np.arange(b.bins.start, b.bins.stop) / (b.fft_size * b.decimation))
            cnt.extend([b.count] * (b.bins.stop - b.bins.start))
            dec.extend([b.decimation] * (b.bins.stop - b.bins.start))
    return np.array(f), np.array(cnt, np.float64), np.array(dec, np.float64)


KA_TAPS = np.array([[[1.0, 0, 0, 0], [0, 0, 0, 0]],
                    [[0, 0, 0, 0], [1.0, 0, 0, 0]],
                    [[0.6, -0.3, 0.15, 0.0], [0.0, 0.8, 0.0, -0.2]],
                    [[0.0, 0.2, 0.5, 0.0], [-0.4, 0.0, 0.3, 0.1]]], np.float32)


def test_known_answer_csm_4096_at_2_32(sp):
    """the first long-run accuracy check of the cross kinds: 2^32 samples per channel into CsmCascade(4096, 4)"""
    n, total = 4096, 1 << 32
    p = sp.Plant(KA_TAPS, [sp.Plant.noise(0, 31), sp.Plant.noise(1, 32)])
    c = sp.CsmCascade(n, 4)
    c.process_plant(p, total)
    S, b = c.csm()
    f, cnt, dec = bins(b)
    want = p.expected_csm(f)
    bound = csm_bound(want, p.expected_csm, f, cnt, n, dec)
    ratio = np.abs(S.astype(np.complex128) - want) / bound
    print("CSM(4096, 4) at 2^32: worst ratio to the bound %.3f (bins %d)" % (ratio.max(), f.size))
    w = np.unravel_index(np.argmax(ratio), ratio.shape)
    print("  worst at S[%d, %d], f %.4g (decimation %d, count %d): got %s, closed form %s, bound %.3g" %
          (w[0], w[1], f[w[2]], dec[w[2]], cnt[w[2]], S[w], want[w], bound[w]))
    assert ratio.max() < 1.0
    H = sp.CsmCascade.transfer(S, [0, 1], [2, 3])
    e = np.exp(-2j * np.pi * f[None, :] * np.arange(4)[:, None])
    h = np.einsum("omt,tf->omf", KA_TAPS[2:].astype(np.float64), e)
    tol = mimo_tolerance(S, h, dec, cnt, n=n)
    # the transfer function is defined where both inputs stand above the rounding floor: the once-differenced input falls
    # below it near DC of the deep stages, where the outputs' share of it is rounding noise, not a mix of it
    fl, _ = rounding_floor(want, p.expected_csm, dec)
    ok = np.all(fl[:2] <= 1e-4 * np.real(np.einsum("iib->ib", want))[:2], axis=0)
    print("  transfer checked on %.0f %% of the bins (both inputs 1e4 above the rounding floor)" % (100 * ok.mean()))
    assert ok.mean() > 0.3
    err = np.abs(H - h)[:, :, ok]
    assert np.all(err <= tol[:, :, ok]), float(np.max(err / tol[:, :, ok]))
    coh = sp.CsmCascade.coherence(S)[0, 2]
    want_coh = np.abs(want[0, 2]) ** 2 / (np.real(want[0, 0]) * np.real(want[2, 2]))
    ok = ok & (cnt >= 1000)
    assert np.max(np.abs(coh - want_coh)[ok]) < 0.02


def test_known_answer_csd_512(sp):
    n, total = 512, 1 << 30
    taps = KA_TAPS[2:4, :, :]
    p = sp.Plant(taps, [sp.Plant.noise(0, 41), sp.Plant.noise(1, 42)])
    c = sp.CsdCascade(n)
    c.process_plant(p, total)
    pxx, pyy, pxy, b = c.csd()
    f, cnt, dec = bins(b)
    S = np.array([[pxx, pxy], [np.conj(pxy), pyy]])
    want = p.expected_csm(f)
    ratio = np.abs(S - want) / csm_bound(want, p.expected_csm, f, cnt, n, dec)
    print("CSD(512) at 2^30: worst ratio to the bound %.3f" % ratio.max())
    assert ratio.max() < 1.0


def test_known_answer_zoom_heterodyne_tone_side(sp):
    """a tone at the carrier + an offset over white noise lands on the positive side; p_neg shows no image"""
    n, total = 512, 1 << 28
    off = 1 << 20                                   # offset ftw / 2^32 = 2^-12 of the sample rate
    p = sp.Plant(np.array([[[1.0], [1.0]]], np.float32), [sp.Plant.noise(0, 51), sp.Plant.tone(FTW + off, 1.0)])
    z = sp.ZoomCascade.heterodyne(n, FTW)
    z.process_plant(p, total)
    pp, pn, b = z.spectrum()
    f, cnt, dec = bins(b)
    k = np.argmax(pp)
    assert abs(f[k] - off / 2.0 ** 32) <= 2.0 / (n * dec[k])
    floor = 1.0  # a real unit-RMS white stream reads 2 one-sided: 1 per side of the two-sided density
    bound = floor * (1 + spread(cnt)) + 2e-4
    # bins at least 64 of their own widths from the tone in absolute frequency, out of reach of its Hann leakage
    width = 1.0 / (n * dec)
    t = off / 2.0 ** 32
    # the real tone's own negative-frequency line sits at -(f0 + offset), i.e. p_neg at 2 f0 + offset (mod 1): a line, not
    # an image; the image would be p_neg at the offset
    twin = (2 * FTW + off) % 2 ** 32 / 2.0 ** 32
    far_pos = np.abs(f - t) > 64 * width
    far_neg = ((f + t) > 64 * width) & (np.abs(f - twin) > 64 * width)
    near_image = (np.abs(f - t) <= 2 * width) & ((f + t) > 64 * width)
    assert np.any(near_image) and np.all(pn[near_image] <= bound[near_image])
    assert np.all(pn[far_neg] <= bound[far_neg]), float(np.max(pn[far_neg] / bound[far_neg]))  # no image
    dev = np.abs(pp - floor) / (bound - floor)
    w = np.argmax(np.where(far_pos, dev, 0))
    print("zoom heterodyne: worst p_pos deviation %.3f of the bound at f %.4g (decimation %d, count %d): %.6g" %
          (dev[w], f[w], dec[w], cnt[w], pp[w]))
    assert np.all(np.abs(pp[far_pos] - floor) <= bound[far_pos] - floor)
    print("zoom heterodyne: tone at %.3g, worst p_neg / bound %.3f" % (f[k], float(np.max(pn[far_neg] / bound[far_neg]))))


# ---- 4. groups ----
GKINDS = {"psd": dict(kind=0), "csd": dict(kind=1), "csm3": dict(kind=2, channels=3), "csm4": dict(kind=2, channels=4),
          "zoom_iq": dict(kind=3, zoom_mode=0), "zoom_het": dict(kind=3, zoom_mode=1, ftw=FTW)}


def group_read(g, kind):
    if kind == "psd":
        p, b = g.psd(0)
        return [p], [], b
    if kind == "csd":
        pxx, pyy, pxy, b = g.csd()
        return [pxx, pyy], [(pxy, pxx, pyy)], b
    if kind.startswith("csm"):
        s, b = g.csm()
        d = [s[i, i].real for i in range(s.shape[0])]
        return d, [(s[i, j], d[i], d[j]) for i in range(len(d)) for j in range(i + 1, len(d))], b
    pp, pn, b = g.spectrum()
    return [pp, pn], [], b


def seq_read(h, kind):
    if kind == "psd":
        p, b = h.psd()
        return [p], [], b
    return group_read(h, kind)


@pytest.mark.parametrize("kind", list(GKINDS))
@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_group_time_process_plant_equals_sequential(sp, kind, world):
    n, total = 512, 6_000_017
    k = {"psd": 1, "csd": 2, "csm3": 3, "csm4": 4, "zoom_iq": 2, "zoom_het": 1}[kind]
    taps = taps_of(k, 2, 6, world)
    ins = [sp.Plant.noise(0, 61), sp.Plant.noise(1, 62)]
    seq, _ = handle(sp, kind, n)
    seq.process_plant(sp.Plant(taps, ins), total)
    want = seq_read(seq, kind)
    for devs in device_lists(world):
        g = sp.Group(n, devices=devs, mode=sp.ShardMode.TIME, deterministic=True, **GKINDS[kind])
        g.time_plan(total, 2)
        g.time_process_plant(sp.Plant(taps, ins).spec())
        g.time_finish()
        got = group_read(g, kind)
        assert [breaks_tuple(v) for v in got[2]] == [breaks_tuple(v) for v in want[2]]
        for r, w in zip(got[0], want[0]):
            np.testing.assert_allclose(r, w, rtol=1e-5, atol=1e-6 * float(np.median(w)))
        for (c, _, _), (s, sii, sjj) in zip(got[1], want[1]):
            tol = 1e-5 * np.sqrt(np.asarray(sii, np.float64) * np.asarray(sjj, np.float64)) + 1e-7 * float(np.median(sii))
            assert np.all(np.abs(c.astype(np.complex128) - s) <= tol)
        if devs == [0] * world and world > 1:
            # deterministic mode on the peer path: a second run is bit-identical
            g.time_plan(total, 2)
            g.time_process_plant(sp.Plant(taps, ins))
            g.time_finish()
            again = group_read(g, kind)
            for r, w in zip(again[0], got[0]):
                assert np.array_equal(r, w)
            for (c, _, _), (d, _, _) in zip(again[1], got[1]):
                assert np.array_equal(c, d)


def test_group_plant_continues_after_partial_feed(sp):
    """ranks fed the first part of their range as arrays: time_process_plant continues at feed_lo + fed"""
    n, total = 512, 4_000_003
    taps = taps_of(3, 2, 6, 8)
    ins = [sp.Plant.noise(0, 81), sp.Plant.noise(1, 82)]
    seq = sp.CsmCascade(n, 3, deterministic=True)
    seq.process_plant(sp.Plant(taps, ins), total)
    want = seq_read(seq, "csm3")
    g = sp.Group(n, devices=[0, 0], mode=sp.ShardMode.TIME, deterministic=True, **GKINDS["csm3"])
    g.time_plan(total, 2)
    p = sp.Plant(taps, ins)
    for r in range(2):
        c = g.time_chunk(r)
        p.seek(c.feed_lo)
        g.time_process(r, *p.generate(100_003).clone())
    g.time_process_plant(p)
    g.time_finish()
    got = group_read(g, "csm3")
    assert [breaks_tuple(v) for v in got[2]] == [breaks_tuple(v) for v in want[2]]
    for (c, _, _), (s, sii, sjj) in zip(got[1], want[1]):
        tol = 1e-5 * np.sqrt(np.asarray(sii, np.float64) * np.asarray(sjj, np.float64)) + 1e-7 * float(np.median(sii))
        assert np.all(np.abs(c.astype(np.complex128) - s) <= tol)


def test_group_errors_feed_nothing(sp):
    from stabilizer_stream_b200._lib import SspsdError, EINVAL, EUNIMPLEMENTED
    g = sp.Group(512, devices=[0, 0], mode=sp.ShardMode.TIME, kind=2, channels=3)
    g.time_plan(1_000_000, 2)
    with pytest.raises(SspsdError) as e:
        g.time_process_plant(sp.PlantSpec(taps_of(2, 1, 1, 0), [sp.Plant.noise()]))
    assert e.value.status == EINVAL
    with pytest.raises(SspsdError) as e:
        g.time_process_plant(sp.PlantSpec(taps_of(3, 1, 1, 0), [sp.Plant.noise(-1)]))
    assert e.value.status == EUNIMPLEMENTED
    with pytest.raises(SspsdError):
        g.time_finish()                                  # nothing was fed
    g.time_process_plant(sp.PlantSpec(taps_of(3, 1, 2, 0), [sp.Plant.noise()]))
    g.time_finish()
    assert g.csm()[0].shape[0] == 3


def test_group_csm4_at_config5_size(sp):
    """4.8e9 samples per channel over the ranks of the box (shared GPU 0 on a one-GPU box), against the closed form"""
    import torch
    n, total = 4096, 4_800_000_000
    world = max(2, torch.cuda.device_count())
    devs = list(range(world)) if torch.cuda.device_count() >= 2 else [0, 0]
    p = sp.Plant(KA_TAPS, [sp.Plant.noise(0, 71), sp.Plant.noise(1, 72)])
    g = sp.Group(n, devices=devs, mode=sp.ShardMode.TIME, kind=2, channels=4)
    g.time_plan(total)
    g.time_process_plant(p)
    g.time_finish()
    S, b = g.csm()
    f, cnt, dec = bins(b)
    want = p.expected_csm(f)
    ratio = np.abs(S.astype(np.complex128) - want) / csm_bound(want, p.expected_csm, f, cnt, n, dec)
    print("group CSM(4096, 4) at 4.8e9 over %s: worst ratio to the bound %.3f" % (devs, ratio.max()))
    assert ratio.max() < 1.0


# ---- 5. bounds build ----
@pytest.mark.skipif(bool(os.environ.get("SSPSD_LIB")), reason="already running against another build")
def test_bounds_build():
    """generation, consumers and groups on the bounds-checking build: no device-side assert fires"""
    if not os.path.exists(BOUNDS):
        pytest.skip("libsspsd_bounds.so not built")
    env = dict(os.environ, SSPSD_LIB=BOUNDS)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "tests"), env.get("PYTHONPATH", "")])
    r = subprocess.run([sys.executable, "-m", "pytest", "-m", "gpu", "-x", "-q", os.path.abspath(__file__), "-k",
                        "generation_noise_bit_exact and (32-4-4 or 1-1-1 or 7-3-2) or ragged or tones or "
                        "(equals_sequential and 2-)"],
                       env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and " passed" in r.stdout, r.stdout[-1500:] + r.stderr[-1500:]
