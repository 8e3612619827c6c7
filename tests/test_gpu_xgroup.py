"""Time-chunked groups of the cross-spectral kinds (sspsd_group_create_kind): CSD, CSM and zoom captures cut over ranks
against one sequential handle of the same kind fed the whole capture, against the float64 models, and the kinds'
error paths.  Ranks share GPU 0 (the direct peer-load reduction) and, where the box has them, take one GPU each
(ncclCommInitAll); tools/group_rank.py --kind covers the one-process-per-GPU path."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import uniform_noise
from oracle import csm as ocsm
from oracle import model_f64_csd as mcsd
from oracle import model_f64_zoom as mz
from oracle import zbinding
from test_gpu_csd import assert_bins_close, assert_cross_close
from test_gpu_group import breaks_tuple, device_lists

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BOUNDS = os.path.join(ROOT, "stabilizer_stream_b200", "libsspsd_bounds.so")
FTW = 0x9E3779B9  # a large odd tuning word: a carrier near 0.618 of the sample rate


@pytest.fixture(scope="module")
def sp():
    import torch
    assert torch.cuda.is_available()
    import stabilizer_stream_b200 as m
    return m


def streams(kind, total, seed):
    """y = h * x + noise traces, so that coherence and transfer are non-trivial; zoom: correlated I/Q or one real trace"""
    x = uniform_noise(total, seed) + np.float32(0.1)
    if kind == "zoom_het":
        return [x]
    out = [x]
    h = [np.array([0.6, -0.3, 0.15]), np.array([0.2, 0.5]), np.array([-0.4, 0.1, 0.1, 0.05])]
    for c in range(1, {"csd": 2, "csm3": 3, "csm4": 4, "zoom_iq": 2}[kind]):
        y = np.convolve(x, h[c - 1])[:total] + 0.5 * uniform_noise(total, seed + 17 * c)
        out.append(y.astype(np.float32))
    return out


def group_args(kind):
    return {"csd": dict(kind=1), "csm3": dict(kind=2, channels=3), "csm4": dict(kind=2, channels=4),
            "zoom_iq": dict(kind=3, zoom_mode=0), "zoom_het": dict(kind=3, zoom_mode=1, ftw=FTW)}[kind]


def sequential(sp, kind, n, window, avg, det, hbf=1):
    kw = dict(window=window, hbf=sp.Hbf(hbf))
    if kind == "csd":
        c = sp.CsdCascade(n, **kw)
    elif kind.startswith("csm"):
        c = sp.CsmCascade(n, int(kind[3]), **kw)
    elif kind == "zoom_iq":
        c = sp.ZoomCascade.iq(n, **kw)
    else:
        c = sp.ZoomCascade.heterodyne(n, FTW, **kw)
    if avg is not None:
        c.set_avg(avg)
    c.set_detrend(sp.Detrend(det))
    return c


def readout(obj, kind):
    """-> (real rows, [(cross term, S_ii, S_jj)], breaks), for a group or a handle alike"""
    if kind == "csd":
        pxx, pyy, pxy, b = obj.csd()
        return [pxx, pyy], [(pxy, pxx, pyy)], b
    if kind.startswith("csm"):
        s, b = obj.csm()
        k = s.shape[0]
        d = [s[i, i].real for i in range(k)]
        assert all(np.all(s[i, i].imag == 0) for i in range(k))
        return d, [(s[i, j], d[i], d[j]) for i in range(k) for j in range(i + 1, k)], b
    pp, pn, b = obj.spectrum()
    return [pp, pn], [], b


def compare(got, want, det):
    """breaks field by field; real rows under the PSD group's rule; cross terms against sqrt(S_ii S_jj)"""
    rows, cross, b = got
    wrows, wcross, wb = want
    assert [breaks_tuple(v) for v in b] == [breaks_tuple(v) for v in wb]
    head = 2 if det >= 2 else 0
    for r, w in zip(rows, wrows):
        assert r.shape == w.shape
        np.testing.assert_allclose(r[head:], w[head:], rtol=3e-5, atol=1e-6 * float(np.median(w)))
    for (g, _, _), (s, sii, sjj) in zip(cross, wcross):
        sii, sjj = np.asarray(sii, np.float64), np.asarray(sjj, np.float64)
        tol = 3e-5 * np.sqrt(sii * sjj) + 1e-6 * float(np.median(sii))
        err = np.abs(g.astype(np.complex128) - s.astype(np.complex128))
        assert np.all(err[head:] <= tol[head:]), float(np.max((err - tol)[head:]))


def feed(sp, g, xs, how, devs):
    """host: the whole capture in one call; device: the same from CUDA tensors; ragged / ragged_dev: every rank in
    three calls of odd lengths (host arrays / tensors on the rank's device), so stream positions leave multiples of 4"""
    import torch
    if how == "host":
        g.time_process_all(*xs)
        return
    if how == "device":
        g.time_process_all(*[torch.from_numpy(x).cuda() for x in xs])
        return
    for r in range(g.n_ranks):
        c = g.time_chunk(r)
        a = c.feed_lo + (c.feed_hi - c.feed_lo) // 3 + 1
        m = a + (c.feed_hi - a) // 2 + 2
        for lo, hi in ((c.feed_lo, a), (a, m), (m, c.feed_hi)):
            parts = [x[lo:hi] for x in xs]
            if how == "ragged_dev":
                parts = [torch.from_numpy(p.copy()).to("cuda:%d" % devs[r]) for p in parts]
            g.time_process(r, *parts)


CASES = [
    # kind, n, total, world, n_local, avg, detrend, window, feed
    ("csd", 512, 2_000_017, 2, 2, None, 0, 1, "ragged"),
    ("csd", 4096, 12_000_000, 3, 1, None, 3, 1, "host"),
    ("csd", 256, 1_200_001, 1, 2, None, 1, 1, "host"),                      # one rank: the handle itself
    ("csm3", 512, 2_500_000, 4, 0, (999, 2 ** 32 - 2), 3, 1, "device"),    # the psd binary's preset, planner's n_local
    ("csm4", 1024, 3_000_001, 3, 2, (0, 64), 1, 1, "ragged"),
    ("csm4", 256, 1_500_000, 2, 2, None, 0, 0, "host"),                     # rectangular window
    ("zoom_iq", 512, 2_000_000, 2, 0, None, 2, 1, "ragged_dev"),
    ("zoom_iq", 64, 700_001, 1, 2, None, 0, 1, "host"),
    ("zoom_het", 512, 2_000_003, 3, 2, None, 0, 1, "ragged_dev"),
    ("zoom_het", 256, 1_800_000, 4, 2, (999, 2 ** 32 - 2), 3, 0, "device"),
    ("zoom_het", 4096, 9_000_000, 2, 1, (0, 64), 2, 1, "ragged"),
]


@pytest.mark.parametrize("kind,n,total,world,k,avg,det,window,how", CASES)
def test_cross_group_equals_sequential(sp, kind, n, total, world, k, avg, det, window, how):
    import torch
    xs = streams(kind, total, 300 + n)
    a = sp.AvgOpts(*avg) if avg else None
    seq = sequential(sp, kind, n, sp.Window(window), a, det)
    if kind.startswith("csm"):
        seq.process(xs)
    else:
        seq.process(*xs)
    want = readout(seq, kind)
    for devs in device_lists(world):
        g = sp.Group(n, devices=devs, mode=sp.ShardMode.TIME, window=sp.Window(window), **group_args(kind))
        if a is not None:
            g.set_avg(a)
        g.set_detrend(sp.Detrend(det))
        g.time_plan(total, k)
        assert all(g.time_chunk(r).feed_lo % 8 == 0 for r in range(world))
        feed(sp, g, xs, how, devs)
        g.time_finish()
        assert torch.cuda.current_device() == 0
        compare(readout(g, kind), want, det)


def test_heterodyne_ranks_mix_at_their_absolute_position(sp):
    """a tone between bins over weak noise: a rank whose mixer restarted at 0 would rotate its chunk by the constant
    phase (feed_lo ftw) mod 2^32, so the gathered stream of the deep stages, which resolve the tone, would jump in phase
    at every rank boundary and smear it"""
    n, total, world = 512, 3_000_000, 3
    f0 = FTW / 2.0 ** 32
    t = np.arange(total, dtype=np.float64)
    x = (np.cos(2 * np.pi * (f0 + 3.37 / (n * 64)) * t) + 1e-4 * uniform_noise(total, 9)).astype(np.float32)
    seq = sequential(sp, "zoom_het", n, sp.Window.HANN, None, 0)
    seq.process(x)
    want = readout(seq, "zoom_het")
    for devs in device_lists(world):
        g = sp.Group(n, devices=devs, mode=sp.ShardMode.TIME, **group_args("zoom_het"))
        g.time_plan(total, 1)
        feed(sp, g, [x], "ragged", devs)
        g.time_finish()
        got = readout(g, "zoom_het")
        compare(got, want, 0)
        # the comparison above is sensitive to the rotation: the tone's stage-0 bins carry most of the power
        assert float(np.max(got[0][0])) > 1e4 * float(np.median(got[0][0]))


@pytest.mark.parametrize("kind", ["csd", "csm3", "zoom_het"])
def test_cross_group_against_the_float64_model(sp, kind):
    """DESIGN.md section 4's per-bin rule against the float64 models, every merged bin"""
    n, total, world = 256, 600_000, 3
    xs = streams(kind, total, 41)
    g = sp.Group(n, devices=[0] * world, mode=sp.ShardMode.TIME, **group_args(kind))
    g.time_plan(total, 2)
    g.time_process_all(*xs)
    g.time_finish()
    rows, cross, b = readout(g, kind)
    if kind == "csd":
        tx, ty, txy, b64 = mcsd.merge_cross(mcsd.cross_cascade(xs[0], xs[1], n), n)
        assert_bins_close(rows[0], tx, "pxx")
        assert_bins_close(rows[1], ty, "pyy")
        assert_cross_close(cross[0][0], txy, tx, ty, "pxy")
    elif kind == "csm3":
        t, b64 = ocsm.f64_matrix(xs, n)
        d = [np.real(t[i, i]) for i in range(3)]
        for i in range(3):
            assert_bins_close(rows[i], d[i], "S%d%d" % (i, i))
        for (s, _, _), (i, j) in zip(cross, [(0, 1), (0, 2), (1, 2)]):
            assert_cross_close(s, t[i, j], d[i], d[j], "S%d%d" % (i, j))
    else:
        i, q = zbinding.heterodyne(xs[0], FTW)
        tp, tn, b64 = mz.merge_zoom(mz.zoom_cascade(i, q, n), n)
        assert_bins_close(rows[0], tp, "p_pos")
        assert_bins_close(rows[1], tn, "p_neg")
    assert [(v.count, v.bins.start, v.bins.stop, v.decimation) for v in b] == \
        [(d["count"], d["bins"][0], d["bins"][1], d["decimation"]) for d in b64]


@pytest.mark.parametrize("kind", ["csm4", "zoom_het"])
def test_deterministic_p2p_runs_are_bit_equal(sp, kind):
    total = 2_000_001
    xs = streams(kind, total, 5)
    outs = []
    for _ in range(2):
        g = sp.Group(512, devices=[0, 0, 0], mode=sp.ShardMode.TIME, deterministic=True, **group_args(kind))
        g.set_avg(sp.AvgOpts(999, 2 ** 32 - 2))
        g.time_plan(total, 2)
        g.time_process_all(*xs)
        g.time_finish()
        assert g.info()["reduce"] == "p2p"
        rows, cross, b = readout(g, kind)
        outs.append(([r.view(np.uint32).copy() for r in rows], [c[0].view(np.uint32).copy() for c in cross],
                     [breaks_tuple(v) for v in b]))
    assert outs[0][2] == outs[1][2]
    assert all(np.array_equal(a, c) for a, c in zip(outs[0][0] + outs[0][1], outs[1][0] + outs[1][1]))


def test_cross_group_errors_consume_nothing(sp):
    import ctypes as C
    import torch
    from stabilizer_stream_b200 import _lib as L
    lib = L.lib()
    with pytest.raises(L.SspsdError) as e:
        sp.Group(512, devices=[0, 0], mode=sp.ShardMode.CHANNELS, kind=sp.GroupKind.CSM, channels=3)
    assert e.value.status == L.EINVAL
    for n in (8192, 32):
        with pytest.raises(L.SspsdError) as e:
            sp.Group(n, devices=[0, 0], mode=sp.ShardMode.TIME, kind=sp.GroupKind.CSD)
        assert e.value.status == L.EINVAL
    total = 600_000
    xs = streams("csd", total, 3)
    g = sp.Group(512, devices=[0, 0], mode=sp.ShardMode.TIME, kind=sp.GroupKind.CSD)
    with pytest.raises(L.SspsdError):
        g.time_finish()                                   # no plan
    g.time_plan(total, 2)
    c0 = g.time_chunk(0)
    x0 = xs[0][c0.feed_lo:c0.feed_hi]
    # wrong-kind entry points: EINVAL, nothing consumed
    assert lib.sspsd_group_time_process_f32(g._h, 0, x0.ctypes.data, x0.size, L.MEM_HOST) == L.EINVAL
    assert lib.sspsd_group_time_process_all_f32(g._h, xs[0].ctypes.data, total) == L.EINVAL
    assert lib.sspsd_group_time_process_noise(g._h, 0, 1) == L.EINVAL
    with pytest.raises(ValueError):
        g.time_process(0, x0)                             # one stream for two
    with pytest.raises(ValueError):
        g.time_process_all(*xs, xs[0])                    # three for two
    g.time_process(0, *[x[c0.feed_lo:c0.feed_hi] for x in xs])
    with pytest.raises(L.SspsdError):
        g.time_finish()                                   # rank 1 not fed
    with pytest.raises(L.SspsdError):
        g.csd()                                           # not finished
    c1 = g.time_chunk(1)
    g.time_process(1, *[x[c1.feed_lo:c1.feed_hi] for x in xs])
    g.time_finish()
    pl, bl = C.c_size_t(16), C.c_size_t(16)
    p = np.zeros(16, np.float32)
    b = (L.BreakC * 16)()
    assert lib.sspsd_group_psd(g._h, 0, None, p.ctypes.data, C.byref(pl), b, C.byref(bl)) == L.EINVAL
    assert lib.sspsd_group_csm_read(g._h, None, p.ctypes.data, C.byref(pl), b, C.byref(bl)) == L.EINVAL
    assert lib.sspsd_group_zoom_read(g._h, None, p.ctypes.data, p.ctypes.data, C.byref(pl), b, C.byref(bl)) == L.EINVAL
    # capacity: ESHORT with the lengths needed, as sspsd_csd_read
    pl = C.c_size_t(1)
    assert lib.sspsd_group_csd_read(g._h, None, p.ctypes.data, p.ctypes.data, p.ctypes.data, C.byref(pl), b,
                                    C.byref(bl)) == L.ESHORT and pl.value > 1
    seq = sp.CsdCascade(512)
    seq.process(*xs)
    compare(readout(g, "csd"), readout(seq, "csd"), 0)    # the refused calls consumed nothing
    # a cross read on a PSD group
    gp = sp.Group(512, devices=[0, 0], mode=sp.ShardMode.TIME)
    gp.time_plan(total, 2)
    gp.time_process_all(xs[0])
    gp.time_finish()
    pl = C.c_size_t(16)
    assert lib.sspsd_group_csd_read(gp._h, None, p.ctypes.data, p.ctypes.data, p.ctypes.data, C.byref(pl), b,
                                    C.byref(bl)) == L.EINVAL
    k = L.GroupKindC()
    L.check(lib.sspsd_group_kind_of(g._h, C.byref(k)))
    assert (k.kind, k.channels) == (L.GROUP_CSD, 2)
    assert torch.cuda.current_device() == 0


def test_entry_points_keep_the_current_device(sp):
    """a cross group on the last GPU: torch's current device stays 0 through every entry point"""
    import torch
    torch.cuda.set_device(0)
    dev = torch.cuda.device_count() - 1
    total = 800_000
    xs = streams("zoom_het", total, 8)
    g = sp.Group(256, devices=[dev, dev], mode=sp.ShardMode.TIME, **group_args("zoom_het"))
    steps = [lambda: g.set_avg(sp.AvgOpts(999, 2 ** 32 - 2)), lambda: g.set_detrend(sp.Detrend.MEAN),
             lambda: g.time_plan(total, 2), lambda: g.time_process_all(*xs), lambda: g.sync(), lambda: g.time_finish(),
             lambda: g.spectrum(), lambda: g.info()]
    for s in steps:
        s()
        assert torch.cuda.current_device() == 0


@pytest.mark.skipif(bool(os.environ.get("SSPSD_LIB")), reason="already running against another build")
def test_bounds_build():
    """one case per kind on the bounds-checking build: no device-side assert fires"""
    if not os.path.exists(BOUNDS):
        pytest.skip("libsspsd_bounds.so not built")
    env = dict(os.environ, SSPSD_LIB=BOUNDS)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "tests"), env.get("PYTHONPATH", "")])
    r = subprocess.run([sys.executable, "-m", "pytest", "-m", "gpu", "-x", "-q", os.path.abspath(__file__), "-k",
                        "equals_sequential and (csd-512 or csm4-1024 or zoom_iq-512 or zoom_het-512)"],
                       env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and " passed" in r.stdout, r.stdout[-1500:] + r.stderr[-1500:]


def test_cpp_group_kinds_on_gpu():
    from test_abi_xgroup import build_cpp
    r = subprocess.run([build_cpp()], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "xgroup ok" in r.stdout, r.stdout + r.stderr


def test_one_process_per_gpu_csm_over_nccl():
    """ncclCommInitRank path for a cross kind: torchrun, 2 ranks, 2 GPUs (tools/group_rank.py --kind csm)"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29583", os.path.join(ROOT, "tools", "group_rank.py"), "--mode", "time", "--kind", "csm"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert out["ok"] and out["world"] == 2 and out["kind"] == "csm", out
