"""Stabilizer frames straight into CsdCascade / CsmCascade (sspsd_csd_process_frames, sspsd_csm_process_frames and the
receiver's pump): against the same decoded traces fed to process(), the PsdCascade frame path and the CPU oracle's
loss accounting.  The cascades run in deterministic mode, so "equal" is bit-equal.  Needs a B200."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from frames_util import make_frames, oracle_decode_stream
from test_gpu_csd import assert_bins_close, btuple

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BOUNDS = os.path.join(ROOT, "stabilizer_stream_b200", "libsspsd_bounds.so")
# (format, batches): AdcDac yields 8 samples per batch and keeps sub-chunks 16-byte aligned; the other formats yield
# one sample per batch, so sub-chunk and call boundaries fall at any stream position
FORMATS = [(1, 22), (2, 25), (3, 18), (4, 60)]


@pytest.fixture(scope="module")
def sp():
    import torch
    assert torch.cuda.is_available()
    import stabilizer_stream_b200 as m
    return m


def samples_per_frame(fmt, batches):
    return batches * (8 if fmt == 1 else 1)


def subchunks(n, host):
    """the frame ranges one process_frames call of n frames feeds to the cascades: host frames are cut into up to 8
    sub-chunks of at least 16384 frames, device frames are decoded in one pass"""
    if not host:
        return [(0, n)]
    k = max(1, min(8, n >> 14))
    per = -(-n // k)
    return [(f0, min(n, f0 + per)) for f0 in range(0, n, per)]


def make_target(sp, kind, n):
    """kind: 'csd' or the CsmCascade channel count"""
    return sp.CsdCascade(n, deterministic=True) if kind == "csd" else sp.CsmCascade(n, kind, deterministic=True)


def readout(target):
    """the handle's readout as exact bits"""
    if hasattr(target, "csm"):
        s, b = target.csm()
        return [s.view(np.uint32)], b
    pxx, pyy, pxy, b = target.csd()
    return [pxx.view(np.uint32), pyy.view(np.uint32), pxy.view(np.uint32)], b


def assert_same(a, b):
    ra, ba = readout(a)
    rb, bb = readout(b)
    assert ba == bb
    for x, y in zip(ra, rb):
        assert np.array_equal(x, y)


def decoded(sp, data, flen, stride, n_frames):
    fmt, traces, ok = sp.FrameDecoder().decode(data, flen, frame_stride=stride, n_frames=n_frames)
    assert ok == n_frames
    return [t for _, t in traces]


def feed_reference(target, traces, tmap, calls, spf, host):
    """process() with the decoded traces, cut exactly where process_frames cuts them"""
    import torch
    for lo, hi in calls:
        for a, b in subchunks(hi - lo, host):
            s0, s1 = (lo + a) * spf, (lo + b) * spf
            xs = [torch.from_numpy(np.ascontiguousarray(traces[t][s0:s1])).cuda() for t in tmap]
            if hasattr(target, "csm"):
                target.process(xs)
            else:
                target.process(xs[0], xs[1])


def feed_frames(sp, dec, target, data, flen, stride, calls, loss, tmap, host):
    import torch
    for lo, hi in calls:
        part = data[lo * stride:(hi - 1) * stride + flen]
        src = part if host else torch.frombuffer(bytearray(part), dtype=torch.uint8).cuda()
        info = dec.process_frames(target, src, flen, loss, frame_stride=stride, n_frames=hi - lo, traces=tmap)
        assert info.frames_ok == hi - lo


def ragged_calls(n_frames, seed, big=0):
    """ragged call sizes; `big` frames first in one call"""
    rng = np.random.default_rng(seed)
    calls, pos = [], 0
    if big:
        calls.append((0, big))
        pos = big
    while pos < n_frames:
        k = int(rng.integers(1, 900))
        calls.append((pos, min(n_frames, pos + k)))
        pos = min(n_frames, pos + k)
    return calls


def identity(kind):
    return [0, 1] if kind == "csd" else list(range(kind))


# ---- 1. process_frames == process() of the decoded traces, every format, every K ----
@pytest.mark.parametrize("fmt,batches", FORMATS)
@pytest.mark.parametrize("kind", ["csd", 2, 3, 4])
@pytest.mark.parametrize("host", [True, False])
def test_frames_equal_process(sp, oracle, fmt, batches, kind, host):
    if fmt == 4 and kind == 4:
        pytest.skip("Mpll carries three traces")
    n = 512
    n_frames = 2600
    data, flen, stride, _ = make_frames(fmt, batches, n_frames, seed=fmt * 10 + (2 if kind == "csd" else kind),
                                        drop_every=41, start_seq=2 ** 32 - 30 * batches)
    tmap = identity(kind)
    calls = ragged_calls(n_frames, seed=fmt + 7)
    a, b = make_target(sp, kind, n), make_target(sp, kind, n)
    loss = sp.Loss()
    feed_frames(sp, sp.FrameDecoder(), a, data, flen, stride, calls, loss, tmap if kind != "csd" else None, host)
    feed_reference(b, decoded(sp, data, flen, stride, n_frames), tmap, calls, samples_per_frame(fmt, batches), host)
    assert_same(a, b)
    st, ok, oloss, _ = oracle_decode_stream(oracle, data, flen, stride, n_frames)
    assert st == 0 and (loss.received, loss.dropped, loss.seq) == (oloss.c.received, oloss.c.dropped, oloss.c.seq)


@pytest.mark.parametrize("kind", ["csd", 4])
@pytest.mark.parametrize("host", [True, False])
def test_large_call_and_stride(sp, kind, host):
    """one call of 40000 frames (host frames: the sub-chunk pipeline), then ragged calls; frames 24 bytes apart beyond
    their length"""
    fmt, batches, n_frames = 1, 22, 44000
    flen = 8 + 64 * batches
    data, flen, stride, _ = make_frames(fmt, batches, n_frames, seed=5, drop_every=1009, stride=flen + 24)
    tmap = identity(kind)
    calls = ragged_calls(n_frames, seed=3, big=40000)
    a, b = make_target(sp, kind, 4096), make_target(sp, kind, 4096)
    feed_frames(sp, sp.FrameDecoder(), a, data, flen, stride, calls, sp.Loss(), None, host)
    feed_reference(b, decoded(sp, data, flen, stride, n_frames), tmap, calls, samples_per_frame(fmt, batches), host)
    assert_same(a, b)


@pytest.mark.parametrize("fmt,batches", [(2, 25), (4, 60)])
def test_large_call_unaligned_formats(sp, fmt, batches):
    """the sub-chunk pipeline with one sample per batch: the second sub-chunk starts at an unaligned position"""
    n_frames = 33001
    data, flen, stride, _ = make_frames(fmt, batches, n_frames, seed=fmt, drop_every=77)
    calls = [(0, n_frames)]
    a, b = make_target(sp, 3, 512), make_target(sp, 3, 512)
    feed_frames(sp, sp.FrameDecoder(), a, data, flen, stride, calls, sp.Loss(), [2, 0, 1], True)
    feed_reference(b, decoded(sp, data, flen, stride, n_frames), [2, 0, 1], calls, samples_per_frame(fmt, batches), True)
    assert_same(a, b)


# ---- 2. trace maps ----
def test_csd_trace_map_is_adc0_dac0(sp):
    data, flen, stride, _ = make_frames(1, 22, 3000, seed=21)
    a, b = make_target(sp, "csd", 1024), make_target(sp, "csd", 1024)
    sp.FrameDecoder().process_frames(a, data, flen, sp.Loss(), traces=(0, 2))
    # CsdCascade.process(adc0, dac0)
    feed_reference(b, decoded(sp, data, flen, stride, 3000), [0, 2], [(0, 3000)], 8 * 22, True)
    assert_same(a, b)


def test_csm_permuted_and_duplicate_maps(sp):
    data, flen, stride, _ = make_frames(1, 22, 4000, seed=22)
    ident = make_target(sp, 4, 512)
    perm = make_target(sp, 3, 512)
    dup = make_target(sp, 3, 512)
    dec = sp.FrameDecoder()
    dec.process_frames(ident, data, flen, sp.Loss())
    dec.process_frames(perm, data, flen, sp.Loss(), traces=(3, 1, 0))
    dec.process_frames(dup, data, flen, sp.Loss(), traces=[0, 0, 2])
    s4, b4 = ident.csm()
    s3, b3 = perm.csm()
    assert b3 == b4
    p = [3, 1, 0]
    want = s4[np.ix_(p, p)]
    scale = np.sqrt(np.abs(np.einsum("iib->ib", want))[:, None, :] * np.abs(np.einsum("iib->ib", want))[None, :, :])
    assert np.all(np.abs(s3 - want) <= 1e-4 * scale + 1e-30)
    # a repeated trace gives equal rows (up to the rounding of the pair in which a channel is transformed)
    sd, _ = dup.csm()
    scale = np.sqrt(np.abs(np.einsum("iib->ib", sd))[:, None, :] * np.abs(np.einsum("iib->ib", sd))[None, :, :])
    assert np.all(np.abs(sd[0] - sd[1]) <= 1e-5 * scale[0] + 1e-30)
    coh = sp.CsmCascade.coherence(sd)
    assert np.all(np.abs(coh[0, 1] - 1) < 1e-4)


@pytest.mark.parametrize("host", [True, False])
def test_mpll_trace_3_is_einval_and_consumes_nothing(sp, host):
    import torch
    from stabilizer_stream_b200 import _lib as L
    data, flen, stride, _ = make_frames(4, 60, 800, seed=4)
    m = make_target(sp, 2, 512)
    dec = sp.FrameDecoder()
    loss = sp.Loss()
    dec.process_frames(m, data[:400 * flen], flen, loss, traces=(0, 2))
    before, lb = readout(m), (loss.received, loss.dropped, loss.seq)
    src = data[400 * flen:] if host else torch.frombuffer(bytearray(data[400 * flen:]), dtype=torch.uint8).cuda()
    with pytest.raises(L.SspsdError) as e:
        dec.process_frames(m, src, flen, loss, traces=(0, 3))
    assert e.value.status == L.EINVAL
    c = make_target(sp, "csd", 512)
    with pytest.raises(L.SspsdError):
        dec.process_frames(c, src, flen, loss, traces=(3, 1))
    after = readout(m)
    assert (loss.received, loss.dropped, loss.seq) == lb and before[1] == after[1]
    assert all(np.array_equal(x, y) for x, y in zip(before[0], after[0]))
    with pytest.raises(ValueError):
        dec.process_frames(m, src, flen, loss, traces=(0, 1, 2))


# ---- 3. loss accounting and malformed frames ----
@pytest.mark.parametrize("host", [True, False])
def test_loss_matches_psd_path_and_oracle(sp, oracle, host):
    import torch
    n_frames = 3000
    data, flen, stride, _ = make_frames(1, 22, n_frames, seed=31, drop_every=13, start_seq=2 ** 32 - 22 * 500)
    src = data if host else torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    lx, lp = sp.Loss(), sp.Loss()
    sp.FrameDecoder().process_frames(make_target(sp, 4, 512), src, flen, lx)
    sp.FrameDecoder().process_frames([sp.PsdCascade(512) for _ in range(4)], src, flen, lp)
    st, ok, oloss, _ = oracle_decode_stream(oracle, data, flen, stride, n_frames)
    assert st == 0
    assert (lx.received, lx.dropped, lx.seq) == (lp.received, lp.dropped, lp.seq)
    assert (lx.received, lx.dropped, lx.seq) == (oloss.c.received, oloss.c.dropped, oloss.c.seq)


@pytest.mark.parametrize("host", [True, False])
@pytest.mark.parametrize("kind", ["csd", 3])
def test_malformed_frame_mid_batch(sp, host, kind):
    import torch
    n_frames, bad = 5000, 3001
    data, flen, stride, _ = make_frames(1, 22, n_frames, seed=41, drop_every=97)
    broken = bytearray(data)
    broken[bad * flen + 1] = 0x06  # wrong magic: de::Error::InvalidHeader
    src = bytes(broken) if host else torch.frombuffer(bytearray(broken), dtype=torch.uint8).cuda()
    x, lx = make_target(sp, kind, 512), sp.Loss()
    with pytest.raises(sp.DecodeError) as ex:
        sp.FrameDecoder().process_frames(x, src, flen, lx)
    with pytest.raises(sp.DecodeError) as ep:
        sp.FrameDecoder().process_frames([sp.PsdCascade(512) for _ in range(4)], src, flen, sp.Loss())
    assert ex.value.status == ep.value.status == 5 and ex.value.frames_ok == ep.value.frames_ok == bad
    ref, lr = make_target(sp, kind, 512), sp.Loss()
    good = data[:bad * flen] if host else torch.frombuffer(bytearray(data[:bad * flen]), dtype=torch.uint8).cuda()
    sp.FrameDecoder().process_frames(ref, good, flen, lr)
    assert (lx.received, lx.dropped, lx.seq) == (lr.received, lr.dropped, lr.seq)
    assert_same(x, ref)


# ---- 4. one decoder alternating between a CsmCascade and four PsdCascades ----
@pytest.mark.parametrize("host", [True, False])
def test_decoder_alternates_between_csm_and_psd(sp, host):
    import torch
    n_frames = 24000
    data, flen, stride, _ = make_frames(1, 22, n_frames, seed=51, drop_every=211)
    calls = ragged_calls(n_frames, seed=9, big=20000)

    def run(shared):
        m = make_target(sp, 4, 4096)
        ps = [sp.PsdCascade(4096, deterministic=True) for _ in range(4)]
        dm = sp.FrameDecoder()
        dp = dm if shared else sp.FrameDecoder()
        lm, lp = sp.Loss(), sp.Loss()
        for lo, hi in calls:
            part = data[lo * stride:hi * stride]
            src = part if host else torch.frombuffer(bytearray(part), dtype=torch.uint8).cuda()
            dm.process_frames(m, src, flen, lm)
            dp.process_frames(ps, src, flen, lp)
        return m, ps, (lm.received, lm.dropped, lm.seq), (lp.received, lp.dropped, lp.seq)

    m1, p1, l1m, l1p = run(True)
    m2, p2, l2m, l2p = run(False)
    assert l1m == l2m == l1p == l2p
    assert_same(m1, m2)
    for a, b in zip(p1, p2):
        pa, ba = a.psd()
        pb, bb = b.psd()
        assert ba == bb and np.array_equal(pa.view(np.uint32), pb.view(np.uint32))
    # and the CSM's diagonal is each PsdCascade's spectrum (the same stage launches' rule as test_gpu_csm)
    s, b = m1.csm()
    for t in range(4):
        pp, bp = p1[t].psd()
        assert [btuple(k) for k in b] == [btuple(k) for k in bp]
        assert_bins_close(s[t, t].real, pp, "S%d%d vs PsdCascade" % (t, t))


# ---- 5. UDP ----
@pytest.mark.parametrize("kind", ["csd", 4])
def test_udp_pump_matches_frames_from_memory(sp, oracle, kind):
    n_frames, batches = 700, 22
    data, flen, stride, _ = make_frames(1, batches, n_frames, seed=61, drop_every=97, start_seq=2 ** 32 - 5000)
    rx = sp.Receiver("127.0.0.1", 0, n_slots=256)
    tx = socket.socket(socket.AF_INET, socket.SOCK_DGRAM)
    tx.connect(("127.0.0.1", rx.port))
    dec = sp.FrameDecoder()
    tmap = (1, 3) if kind == "csd" else (0, 1, 2, 3)
    x = make_target(sp, kind, 512)
    loss = sp.Loss()
    runs = []
    done = 0
    for base in range(0, n_frames, 16):
        for f in range(base, min(base + 16, n_frames)):
            tx.send(data[f * stride:f * stride + flen])
        want = min(base + 16, n_frames)
        while done < want:
            info = rx.pump(dec, x, loss, max_frames=256, timeout_ms=2000, traces=tmap)
            assert info.frames_ok > 0 and info.format == 1 and info.n_traces == 4
            runs.append((done, done + info.frames_ok))
            done += info.frames_ok
    assert rx.datagrams == n_frames
    # the same frames from memory, in the same runs
    ref, rloss = make_target(sp, kind, 512), sp.Loss()
    feed_frames(sp, sp.FrameDecoder(), ref, data, flen, stride, runs, rloss, list(tmap), True)
    assert (loss.received, loss.dropped, loss.seq) == (rloss.received, rloss.dropped, rloss.seq)
    st, ok, oloss, _ = oracle_decode_stream(oracle, data, flen, stride, n_frames)
    assert st == 0 and (loss.received, loss.dropped) == (oloss.c.received, oloss.c.dropped)
    assert_same(x, ref)


def test_udp_pump_refuses_bad_map_before_receiving(sp):
    from stabilizer_stream_b200 import _lib as L
    rx = sp.Receiver("127.0.0.1", 0, n_slots=16)
    tx = socket.socket(socket.AF_INET, socket.SOCK_DGRAM)
    tx.connect(("127.0.0.1", rx.port))
    data, flen, _, _ = make_frames(1, 22, 1, seed=1)
    tx.send(data[:flen])
    m = make_target(sp, 2, 512)
    with pytest.raises(L.SspsdError) as e:
        rx.pump(sp.FrameDecoder(), m, sp.Loss(), timeout_ms=2000, traces=(0, 7))
    assert e.value.status == L.EINVAL
    info = rx.pump(sp.FrameDecoder(), m, sp.Loss(), timeout_ms=2000)
    assert info.frames_ok == 1  # the datagram is still there


# ---- 6. the headless driver ----
def test_driver_csm_from_file(sp, tmp_path):
    """tools/stream_psd.py --file --csm 0,2 --save: the diagonal it reports and the matrix it saves are those of a
    CsmCascade fed the same frames through process_frames"""
    import json
    n_frames = 3000
    data, flen, stride, _ = make_frames(1, 22, n_frames, seed=71, drop_every=101)
    f = tmp_path / "frames.bin"
    f.write_bytes(data)
    out = tmp_path / "s.npz"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "stream_psd.py"), "--file", str(f), "--frame-size",
                        str(flen), "--csm", "0,2", "--trace", "2", "--save", str(out), "--json"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["trace"] == "DAC0" and res["traces"] == 2 and res["items_per_trace"] == n_frames * 22 * 8
    assert [c["traces"] for c in res["csm"]["coherence"]] == [[0, 2]]
    m = sp.CsmCascade(512, 2)
    m.set_detrend(sp.Detrend.MIDPOINT)
    sp.FrameDecoder().process_frames(m, data, flen, sp.Loss(), traces=(0, 2))
    s, b = m.csm()
    saved = np.load(out)
    assert saved["S"].shape == s.shape and list(saved["traces"]) == [0, 2]
    assert saved["breaks"].shape == (len(b), 10) and np.array_equal(saved["frequencies"], sp.Break.frequencies(b))
    np.testing.assert_allclose(saved["S"], s, rtol=1e-5, atol=1e-6 * float(np.max(np.abs(s))))
    assert res["psd_median"] == pytest.approx(float(np.median(np.real(s[1, 1]))), rel=1e-5)
    coh = sp.CsmCascade.coherence(s)
    assert res["csm"]["coherence"][0]["median"] == pytest.approx(float(np.median(coh[0, 1])), rel=1e-4, abs=1e-6)


# ---- 7. the bounds-checking build: one host-frame and one device-frame case ----
@pytest.mark.skipif(bool(os.environ.get("SSPSD_LIB")), reason="already running against another build")
def test_bounds_build():
    if not os.path.exists(BOUNDS):
        pytest.skip("libsspsd_bounds.so not built")
    env = dict(os.environ, SSPSD_LIB=BOUNDS)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "tests"), env.get("PYTHONPATH", "")])
    r = subprocess.run([sys.executable, "-m", "pytest", "-m", "gpu", "-x", "-q", os.path.abspath(__file__), "-k",
                        "test_large_call_unaligned_formats or (test_large_call_and_stride and 4)"],
                       env=env, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0 and " passed" in r.stdout, r.stdout[-1500:] + r.stderr[-1500:]
