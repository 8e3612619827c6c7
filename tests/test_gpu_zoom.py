"""ZoomCascade (two-sided spectra of I/Q streams and of a real stream mixed down around a carrier) on the device
against the CPU restatement (oracle.zbinding.ZCascade), the float64 model (oracle.model_f64_zoom), exact relations,
the high-dynamic-range budget of DESIGN.md section 4, the mixer's bound, and Stabilizer frames.  Needs a B200."""
import ctypes as C
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from conftest import uniform_noise
from frames_util import make_frames, oracle_decode_stream
from oracle import model_f64 as m64
from oracle import model_f64_zoom as mz
from oracle import zbinding
from test_gpu_csd import RTOL, assert_bins_close, btuple

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BOUNDS = os.path.join(ROOT, "stabilizer_stream_b200", "libsspsd_bounds.so")
GAMMA = 1e-7  # tests/dynamic_range_cases.py's device budget
FTW = 0x1F9ADD37  # a carrier near 0.1234 of the sample rate


@pytest.fixture(scope="module")
def sp():
    import torch
    assert torch.cuda.is_available()
    import stabilizer_stream_b200 as m
    return m


def tuples64(b64):
    return [(d["start"], d["include"], d["count"], d["avg"], d["bins"][0], d["bins"][1], d["fft_size"],
             d["decimation"], d["pending"], d["processed"]) for d in b64]


def iq_pair(n_samples, seed):
    """correlated I/Q with offsets, so that the two sides differ"""
    i = uniform_noise(n_samples, seed) + np.float32(0.25)
    q = (0.6 * i + uniform_noise(n_samples, seed + 1000) - np.float32(0.5)).astype(np.float32)
    return i, q


def cuts(total, seed, big=None):
    rng = np.random.default_rng(seed)
    out, pos = [], 0
    while pos < total:
        k = min(total - pos, int(rng.integers(0, big or max(8, total // 6))))
        out.append((pos, pos + k))
        pos += k
    return out


def feed(c, xs, device, seed):
    """ragged calls, every stream split identically; device=True feeds CUDA tensors"""
    import torch
    for lo, hi in cuts(xs[0].size, seed):
        parts = [x[lo:hi] for x in xs]
        if device:
            parts = [torch.from_numpy(p.copy()).cuda() for p in parts]
        c.process(*parts)


def bits(r):
    pp, pn, b = r
    return pp.view(np.uint32).copy(), pn.view(np.uint32).copy(), [btuple(k) for k in b]


def assert_same(r1, r2):
    a, b = bits(r1), bits(r2)
    assert a[2] == b[2]
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def check_parity(sp, c, o, det, truth_streams, preset=1, window=1):
    """the device against the restatement under tests/test_gpu_psd.py's per-bin rule; under Span / Mean detrend the DC
    bins (and under Span every bin where the restatement's own f32 trend line is off the f64 truth) must be at least as
    close to the float64 truth as the restatement is.  Breaks bit-equal to psd()'s of the same options."""
    pp, pn, b = c.spectrum()
    op, on, ob = o.spectrum()
    assert [btuple(k) for k in b] == [k.as_tuple() for k in ob]
    masks, truths = [None, None], [None, None]
    if det in (2, 3):
        n = c.n
        t = mz.merge_zoom(mz.zoom_cascade(*truth_streams, n, det, preset=preset, win_kind=window), n)
        for r, (w, tr) in enumerate(zip((op, on), t[:2])):
            m = np.zeros(w.size, bool)
            m[:2] = True
            if det == 2:
                m |= np.abs(w - tr) > 0.5 * RTOL * np.abs(tr)
            masks[r], truths[r] = m, tr
    assert_bins_close(pp, op, "p_pos", masks[0], truths[0])
    assert_bins_close(pn, on, "p_neg", masks[1], truths[1])
    return pp, pn, b


# ---- 1. parity against the restatement ----
@pytest.mark.parametrize("preset", [0, 1])
@pytest.mark.parametrize("det", [0, 1, 2, 3])
@pytest.mark.parametrize("n", [64, 512, 4096])
def test_iq_parity(sp, n, det, preset):
    i, q = iq_pair(120 * n + 77, n + det)
    c = sp.ZoomCascade.iq(n, hbf=sp.Hbf(preset))
    c.set_detrend(sp.Detrend(det))
    o = zbinding.ZCascade(n, hbf=preset)
    o.set_detrend(det)
    feed(c, (i, q), device=(det % 2 == 1), seed=n + det)
    o.process(i, q)
    assert c.num_stages() == o.num_stages() >= 2
    check_parity(sp, c, o, det, (i, q), preset)


@pytest.mark.parametrize("n", [128, 256, 1024, 2048])
def test_iq_parity_other_sizes_and_psd_breaks(sp, n):
    i, q = iq_pair(100 * n + 3, n)
    c = sp.ZoomCascade.iq(n)
    o = zbinding.ZCascade(n)
    feed(c, (i, q), device=(n >= 1024), seed=n)
    o.process(i, q)
    _, _, b = check_parity(sp, c, o, 0, (i, q))
    p = sp.PsdCascade(n)
    p.process(i)
    assert [btuple(k) for k in b] == [btuple(k) for k in p.psd()[1]]


def test_iq_parity_rectangular(sp):
    n = 1024
    i, q = iq_pair(n * 40 + 5, 3)
    c = sp.ZoomCascade.iq(n, window=sp.Window.RECTANGULAR)
    o = zbinding.ZCascade(n, window=zbinding.WINDOW_RECT)
    c.process(i, q)
    o.process(i, q)
    check_parity(sp, c, o, 0, (i, q), window=0)


@pytest.mark.parametrize("n,det,preset,device", [(512, 0, 1, False), (4096, 3, 0, True), (64, 1, 1, True),
                                                 (1024, 2, 1, False)])
def test_heterodyne_parity(sp, n, det, preset, device):
    x = uniform_noise(150 * n + 11, n + 5) + np.float32(0.3)
    c = sp.ZoomCascade.heterodyne(n, FTW, hbf=sp.Hbf(preset))
    c.set_detrend(sp.Detrend(det))
    o = zbinding.ZCascade(n, hbf=preset, ftw=FTW)
    o.set_detrend(det)
    feed(c, (x,), device, seed=n)
    o.process(x)
    check_parity(sp, c, o, det, zbinding.heterodyne(x, FTW), preset)


# ---- 2. exact relations (deterministic mode) ----
def on_device(*xs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in xs]


def test_ftw_zero_is_iq_of_x_and_zero(sp):
    x = uniform_noise(1_000_003, 7)
    h = sp.ZoomCascade.heterodyne(512, 0, deterministic=True)
    h.process(*on_device(x))
    z = sp.ZoomCascade.iq(512, deterministic=True)
    z.process(*on_device(x, -(x * np.float32(0))))  # what the mixer forms at phase 0: x * 1 and -(x * 0)
    assert_same(h.spectrum(), z.spectrum())


def test_quarter_turn_carrier_is_the_exact_rotation(sp):
    x = uniform_noise(1_000_004, 8)
    c = np.tile(np.array([1, 0, -1, 0], np.float32), x.size // 4)
    s = np.tile(np.array([0, 1, 0, -1], np.float32), x.size // 4)
    h = sp.ZoomCascade.heterodyne(1024, 1 << 30, deterministic=True)
    h.process(*on_device(x))
    z = sp.ZoomCascade.iq(1024, deterministic=True)
    z.process(*on_device(x * c, -(x * s)))
    assert_same(h.spectrum(), z.spectrum())


@pytest.mark.parametrize("device", [True, False])
def test_split_clone_and_reset(sp, device):
    """The mixer's phase runs on over call boundaries: ragged heterodyne calls equal I/Q calls, cut alike, of the same
    samples premixed by sspsd_heterodyne_f32 at their absolute positions (host calls are collected and reach the
    device in one piece between flushes here).  The clone flushes the source (staged input, deferred stages), so the
    references flush at the same point.  Another split reads the same to rounding; clone and reset-and-replay bit for
    bit."""
    import torch
    from stabilizer_stream_b200 import _lib as L
    n, total = 512, 3_000_001
    x = uniform_noise(total, 9)
    xd = torch.from_numpy(x).cuda()
    id_, qd = torch.empty_like(xd), torch.empty_like(xd)
    L.check(L.lib().sspsd_heterodyne_f32(None, xd.data_ptr(), total, 0, FTW, id_.data_ptr(), qd.data_ptr()))
    torch.cuda.synchronize()
    calls = cuts(total, 3)
    h = sp.ZoomCascade.heterodyne(n, FTW, deterministic=True)
    z = sp.ZoomCascade.iq(n, deterministic=True)
    half = len(calls) // 2
    mid = calls[half][0]
    for c, (lo, hi) in enumerate(calls):
        if c == half:
            hc = h.clone()
            if not device:
                z.process(id_[:mid], qd[:mid])
            z.flush()
        h.process(xd[lo:hi] if device else x[lo:hi])
        if c >= half:
            hc.process(xd[lo:hi] if device else x[lo:hi])
        if device:
            z.process(id_[lo:hi], qd[lo:hi])
    if not device:
        z.process(id_[mid:], qd[mid:])
    r = h.spectrum()
    assert_same(r, z.spectrum())
    assert_same(r, hc.spectrum())
    h.reset()
    assert h.num_stages() == 0 and h.carrier() == (L.ZOOM_HETERODYNE, FTW)
    for c, (lo, hi) in enumerate(calls):
        if c == half:
            h.flush()
        h.process(xd[lo:hi] if device else x[lo:hi])
    assert_same(r, h.spectrum())
    other = sp.ZoomCascade.heterodyne(n, FTW, deterministic=True)
    for lo, hi in cuts(total, 4):
        other.process(xd[lo:hi] if device else x[lo:hi])
    pp, pn, b = other.spectrum()
    assert [btuple(k) for k in b] == bits(r)[2]
    assert_bins_close(pp, r[0], "other split p_pos")
    assert_bins_close(pn, r[1], "other split p_neg")


@pytest.mark.parametrize("mode", ["iq", "heterodyne"])
def test_power_of_two_scaling(sp, mode):
    i, q = iq_pair(700_001, 13)
    out = []
    for a in (0, 3, -2):
        s = np.float32(2.0 ** a)
        if mode == "iq":
            c = sp.ZoomCascade.iq(256, deterministic=True)
            c.process(i * s, q * s)
        else:
            c = sp.ZoomCascade.heterodyne(256, FTW, deterministic=True)
            c.process(i * s)
        pp, pn, b = c.spectrum()
        out.append((pp / np.float32(4.0 ** a), pn / np.float32(4.0 ** a)))
    for pp, pn in out[1:]:
        assert np.array_equal(pp, out[0][0]) and np.array_equal(pn, out[0][1])


def test_swapped_streams_mirror(sp):
    """q + i i = i conj(z): its P+ is z's P-, equal up to the rounding of the two transforms"""
    i, q = iq_pair(1_000_000, 17)
    a = sp.ZoomCascade.iq(1024, deterministic=True)
    a.process(i, q)
    b = sp.ZoomCascade.iq(1024, deterministic=True)
    b.process(q, i)
    ap, an, ab = a.spectrum()
    bp, bn, bb = b.spectrum()
    assert [btuple(k) for k in ab] == [btuple(k) for k in bb]
    assert_bins_close(bp, an, "swapped p_pos")
    assert_bins_close(bn, ap, "swapped p_neg")


def test_sides_sum_to_the_psd(sp):
    x = uniform_noise(2_000_000, 19)
    z = sp.ZoomCascade.iq(512)
    z.process(x, np.zeros_like(x))
    pp, pn, b = z.spectrum()
    p = sp.PsdCascade(512)
    p.process(x)
    ps, bs = p.psd()
    assert [btuple(k) for k in b] == [btuple(k) for k in bs]
    assert_bins_close(pp + pn, ps, "p_pos + p_neg vs psd")
    f, pt = sp.ZoomCascade.two_sided(pp, pn, b, FTW)
    assert np.all(np.diff(f) > 0) and f.size == 2 * pp.size - 2 and pt.size == f.size


# ---- 3. image rejection at high dynamic range ----
def budget(rows, truth, breaks, n, power):
    """tests/dynamic_range_cases.py's rule on a merged two-sided row: |dev - t| <= 1e-4 t + g sqrt(t S) + g^2 S, S the
    power stage i handled (mean |z|^2 of the input, 64^i of the half-bands, window energy), on the readout's scale"""
    w, pw, nenbw, _ = m64.window(n, 1)
    out = []
    for bk in breaks:
        if not bk.include:
            continue
        i = int(round(np.log(bk.decimation) / np.log(8)))
        s = np.sum(w ** 2) * 8.0 ** i * power / (nenbw * pw)
        k = slice(bk.start, bk.start + bk.bins.stop - bk.bins.start)
        t = truth[k]
        excess = np.abs(rows[k].astype(np.float64) - t) - (RTOL * t + GAMMA * np.sqrt(t * s) + GAMMA ** 2 * s)
        out.append(np.max(excess / s))
    return max(out)


@pytest.mark.parametrize("preset", [0, 1])
@pytest.mark.parametrize("delta", [3.0 / (512 * 64), 3.37 / (512 * 64)])  # on and off a bin of stage 2
def test_iq_tone_image_rejection(sp, preset, delta):
    n, m = 512, 1 << 21
    t = np.arange(m, dtype=np.float64)
    z = np.exp(2j * np.pi * delta * t)
    i = (z.real + 1e-5 * uniform_noise(m, 1)).astype(np.float32)
    q = (z.imag + 1e-5 * uniform_noise(m, 2)).astype(np.float32)
    c = sp.ZoomCascade.iq(n, hbf=sp.Hbf(preset))
    c.process(i, q)
    pp, pn, b = c.spectrum()
    stages = mz.zoom_cascade(i, q, n, preset=preset)
    tp, tn, b64 = mz.merge_zoom(stages, n)
    assert [btuple(k) for k in b] == tuples64(b64) and sum(k.include for k in b) >= 3
    power = np.mean(i.astype(np.float64) ** 2 + q.astype(np.float64) ** 2)
    assert budget(pp, tp, b, n, power) <= 0
    assert budget(pn, tn, b, n, power) <= 0


@pytest.mark.parametrize("preset", [0, 1])
def test_heterodyne_tone_image_rejection(sp, preset):
    n, m = 512, 1 << 21
    f0 = FTW / 2.0 ** 32
    t = np.arange(m, dtype=np.float64)
    x = (np.cos(2 * np.pi * (f0 + 3.37 / (n * 64)) * t) + 1e-5 * uniform_noise(m, 3)).astype(np.float32)
    c = sp.ZoomCascade.heterodyne(n, FTW, hbf=sp.Hbf(preset))
    c.process(x)
    pp, pn, b = c.spectrum()
    i, q = zbinding.heterodyne(x, FTW)
    stages = mz.zoom_cascade(i, q, n, preset=preset)
    tp, tn, b64 = mz.merge_zoom(stages, n)
    assert [btuple(k) for k in b] == tuples64(b64)
    power = np.mean(x.astype(np.float64) ** 2)
    assert budget(pp, tp, b, n, power) <= 0
    assert budget(pn, tn, b, n, power) <= 0


# ---- 4. the mixer ----
def test_mixer_bound_and_quarter_turns(sp):
    import torch
    from stabilizer_stream_b200 import _lib as L
    m = 1 << 20
    x = (uniform_noise(m, 23) * np.float32(3.0)).astype(np.float32)
    xd = torch.from_numpy(x).cuda()
    io, qo = torch.empty_like(xd), torch.empty_like(xd)
    rng = np.random.default_rng(29)
    ftws = [0, 1, 1 << 30, 1 << 31, 3 << 30, 0xFFFFFFFF, FTW] + [int(v) for v in rng.integers(0, 2 ** 32, 9)]
    for k, ftw in enumerate(ftws):
        pos0 = [0, 5, (1 << 32) - 1000, (1 << 43) + 7][k % 4]
        L.check(L.lib().sspsd_heterodyne_f32(None, xd.data_ptr(), m, pos0, ftw, io.data_ptr(), qo.data_ptr()))
        torch.cuda.synchronize()
        i64, q64 = zbinding.heterodyne(x, ftw, pos0)
        bound = 2.0 ** -23 * np.abs(x.astype(np.float64))
        assert np.all(np.abs(io.cpu().numpy() - i64) <= bound), hex(ftw)
        assert np.all(np.abs(qo.cpu().numpy() - q64) <= bound), hex(ftw)
        if ftw % (1 << 30) == 0:  # every phase a quarter turn: exactly 0 and +-x
            assert np.array_equal(io.cpu().numpy(), i64.astype(np.float32))
            assert np.array_equal(qo.cpu().numpy(), q64.astype(np.float32))


# ---- 5. frames and UDP ----
def frame_calls(n_frames, seed):
    rng = np.random.default_rng(seed)
    out, pos = [], 0
    while pos < n_frames:
        k = int(rng.integers(1, 900))
        out.append((pos, min(n_frames, pos + k)))
        pos += k
    return out


@pytest.mark.parametrize("host", [True, False])
@pytest.mark.parametrize("mode", ["iq", "heterodyne"])
def test_frames_equal_process(sp, oracle, host, mode):
    """Fls BI / BQ (traces 2, 3) in I/Q mode, an AdcDac trace heterodyned: bit-equal to process() of the decoded
    traces cut where process_frames cuts them (host frames of these sizes: one sub-chunk per call)"""
    import torch
    fmt, batches = (2, 25) if mode == "iq" else (1, 22)
    spf = batches * (8 if fmt == 1 else 1)
    n_frames = 2600
    data, flen, stride, _ = make_frames(fmt, batches, n_frames, seed=71, drop_every=41, start_seq=2 ** 32 - 700)
    tmap = [2, 3] if mode == "iq" else [1]

    def make():
        if mode == "iq":
            return sp.ZoomCascade.iq(512, deterministic=True)
        return sp.ZoomCascade.heterodyne(512, FTW, deterministic=True)

    a, b = make(), make()
    loss = sp.Loss()
    dec = sp.FrameDecoder()
    calls = frame_calls(n_frames, 5)
    for lo, hi in calls:
        part = data[lo * stride:(hi - 1) * stride + flen]
        src = part if host else torch.frombuffer(bytearray(part), dtype=torch.uint8).cuda()
        assert dec.process_frames(a, src, flen, loss, n_frames=hi - lo, traces=tmap).frames_ok == hi - lo
    _, traces, ok = sp.FrameDecoder().decode(data, flen)
    assert ok == n_frames
    tr = [t for _, t in traces]
    for lo, hi in calls:
        xs = [torch.from_numpy(np.ascontiguousarray(tr[t][lo * spf:hi * spf])).cuda() for t in tmap]
        b.process(*xs)
    assert_same(a.spectrum(), b.spectrum())
    st, _, oloss, _ = oracle_decode_stream(oracle, data, flen, stride, n_frames)
    assert st == 0 and (loss.received, loss.dropped, loss.seq) == (oloss.c.received, oloss.c.dropped, oloss.c.seq)


@pytest.mark.parametrize("mode", ["iq", "heterodyne"])
def test_malformed_frame_and_bad_maps(sp, mode):
    from stabilizer_stream_b200 import _lib as L
    n_frames, bad = 3000, 1801
    data, flen, _, _ = make_frames(1, 22, n_frames, seed=43, drop_every=97)
    broken = bytearray(data)
    broken[bad * flen + 1] = 0x06  # wrong magic
    make = (lambda: sp.ZoomCascade.iq(512, deterministic=True)) if mode == "iq" else \
        (lambda: sp.ZoomCascade.heterodyne(512, FTW, deterministic=True))
    tmap = [0, 2] if mode == "iq" else [3]
    z, lz = make(), sp.Loss()
    with pytest.raises(sp.DecodeError) as e:
        sp.FrameDecoder().process_frames(z, bytes(broken), flen, lz, traces=tmap)
    assert e.value.frames_ok == bad
    ref, lr = make(), sp.Loss()
    sp.FrameDecoder().process_frames(ref, data[:bad * flen], flen, lr, traces=tmap)
    assert (lz.received, lz.dropped, lz.seq) == (lr.received, lr.dropped, lr.seq)
    assert_same(z.spectrum(), ref.spectrum())
    # Mpll has three traces: index 3 refused before anything is consumed; wrong map lengths never reach the library
    mp, flm, _, _ = make_frames(4, 60, 10, seed=1)
    lm = sp.Loss()
    with pytest.raises(L.SspsdError) as e:
        sp.FrameDecoder().process_frames(make(), mp, flm, lm, traces=[3] * len(tmap))
    assert e.value.status == L.EINVAL and lm.received == 0
    with pytest.raises(ValueError):
        sp.FrameDecoder().process_frames(make(), data, flen, traces=[0, 1, 2])


@pytest.mark.parametrize("mode", ["iq", "heterodyne"])
def test_udp_pump(sp, oracle, mode):
    n_frames, batches = 500, 22
    data, flen, stride, _ = make_frames(1, batches, n_frames, seed=61, drop_every=97, start_seq=2 ** 32 - 5000)
    rx = sp.Receiver("127.0.0.1", 0, n_slots=256)
    tx = socket.socket(socket.AF_INET, socket.SOCK_DGRAM)
    tx.connect(("127.0.0.1", rx.port))
    make = (lambda: sp.ZoomCascade.iq(512, deterministic=True)) if mode == "iq" else \
        (lambda: sp.ZoomCascade.heterodyne(512, FTW, deterministic=True))
    tmap = (1, 3) if mode == "iq" else (2,)
    from stabilizer_stream_b200 import _lib as L
    with pytest.raises(L.SspsdError):  # refused before a datagram is taken
        rx.pump(sp.FrameDecoder(), make(), sp.Loss(), timeout_ms=10, traces=(7,) * len(tmap))
    dec, z, loss = sp.FrameDecoder(), make(), sp.Loss()
    runs, done = [], 0
    for base in range(0, n_frames, 16):
        for f in range(base, min(base + 16, n_frames)):
            tx.send(data[f * stride:f * stride + flen])
        want = min(base + 16, n_frames)
        while done < want:
            info = rx.pump(dec, z, loss, max_frames=256, timeout_ms=2000, traces=tmap)
            assert info.frames_ok > 0
            runs.append((done, done + info.frames_ok))
            done += info.frames_ok
    ref, rloss, rdec = make(), sp.Loss(), sp.FrameDecoder()
    for lo, hi in runs:
        rdec.process_frames(ref, data[lo * stride:hi * stride], flen, rloss, frame_stride=stride, n_frames=hi - lo,
                            traces=tmap)
    assert (loss.received, loss.dropped, loss.seq) == (rloss.received, rloss.dropped, rloss.seq)
    st, _, oloss, _ = oracle_decode_stream(oracle, data, flen, stride, n_frames)
    assert st == 0 and (loss.received, loss.dropped) == (oloss.c.received, oloss.c.dropped)
    assert_same(z.spectrum(), ref.spectrum())


# ---- 6. bounds build, errors and devices ----
@pytest.mark.skipif(bool(os.environ.get("SSPSD_LIB")), reason="already running against another build")
def test_bounds_build():
    if not os.path.exists(BOUNDS):
        pytest.skip("libsspsd_bounds.so not built")
    env = dict(os.environ, SSPSD_LIB=BOUNDS)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "tests"), env.get("PYTHONPATH", "")])
    r = subprocess.run([sys.executable, "-m", "pytest", "-m", "gpu", "-x", "-q", os.path.abspath(__file__), "-k",
                        "(iq_parity and 4096) or heterodyne_parity or split_clone or frames_equal or mixer"],
                       env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]


def test_error_paths_and_current_device(sp):
    import torch
    from stabilizer_stream_b200 import _lib as L
    lib = L.lib()
    with pytest.raises(L.SspsdError) as e:
        sp.ZoomCascade.iq(8192)
    assert e.value.status == L.EINVAL
    h = sp.ZoomCascade.heterodyne(512, FTW)
    with pytest.raises(L.SspsdError) as e:
        h.set_detrend(sp.Detrend.LINEAR)
    assert e.value.status == L.EUNIMPLEMENTED
    z = sp.ZoomCascade.iq(512)
    x = uniform_noise(10_000, 1)
    # the call that does not match the mode: EINVAL, nothing consumed
    assert lib.sspsd_zoom_process_f32(z._h, x.ctypes.data, x.size, L.MEM_HOST) == L.EINVAL
    assert lib.sspsd_zoom_process_iq_f32(h._h, x.ctypes.data, x.ctypes.data, x.size, L.MEM_HOST) == L.EINVAL
    assert z.num_stages() == 0 and h.num_stages() == 0
    with pytest.raises(ValueError):
        z.process(x)
    with pytest.raises(ValueError):
        h.process(x, x)
    cfg = L.Config()
    L.check(lib.sspsd_config_default(512, C.byref(cfg)))
    hh = C.c_void_p()
    assert lib.sspsd_zoom_create(C.byref(cfg), 2, 0, C.byref(hh)) == L.EINVAL and not hh.value
    assert lib.sspsd_zoom_create(C.byref(cfg), L.ZOOM_IQ, 5, C.byref(hh)) == L.EINVAL and not hh.value
    assert lib.sspsd_zoom_process_iq_f32(z._h, None, None, 16, L.MEM_HOST) == L.EINVAL
    assert lib.sspsd_zoom_process_f32(h._h, x.ctypes.data, x.size, 7) == L.EINVAL
    # capacity: ESHORT with the lengths needed
    h.process(x)
    pl, bl = C.c_size_t(1), C.c_size_t(0)
    b = (L.BreakC * 1)()
    one = np.zeros(1, np.float32)
    assert lib.sspsd_zoom_read(h._h, None, one.ctypes.data, one.ctypes.data, C.byref(pl), b, C.byref(bl)) == L.ESHORT
    assert pl.value > 1 and bl.value == h.num_stages()
    # the caller's current device is left as it was
    ndev = torch.cuda.device_count()
    torch.cuda.set_device(0)
    d = sp.ZoomCascade.heterodyne(256, FTW, device=ndev - 1)
    d.process(x)
    d.spectrum()
    assert torch.cuda.current_device() == 0
