"""The default decimator (stage A read straight from the staged tile) against the TMA-staged kernel with the
de-interleaving round trip (SSPSD_K3=tma960): both compute every output with the same expression, so the decimated
stream, and everything downstream of it in deterministic mode, must be bit-identical.  The batch lists cover the
first batch with its drain, batches shorter than one 960-output tile, clipped lowest tiles and tiles that straddle the
carry / fresh boundary (every batch after the first), for both tap presets and N = 4096 and 512."""
import os

import numpy as np
import pytest

from conftest import uniform_noise

pytestmark = pytest.mark.gpu

# ragged batch lengths: a first batch that ends inside the drain, sub-tile batches (< 8 * 960 samples), lengths that
# are not multiples of 4 or 8, and batches of many tiles
BATCHES = [1000, 3, 5000, 7681, 7679, 64, 40001, 123457, 8, 7680 * 3 + 5, 250000, 17, 1 << 20]


@pytest.fixture(scope="module")
def sp():
    import torch
    assert torch.cuda.is_available()
    import stabilizer_stream_b200 as m
    return m


def make(factory, k3):
    """create a handle with SSPSD_K3 = k3 (None: the default), which the library reads at creation"""
    old = os.environ.pop("SSPSD_K3", None)
    try:
        if k3 is not None:
            os.environ["SSPSD_K3"] = k3
        return factory()
    finally:
        os.environ.pop("SSPSD_K3", None)
        if old is not None:
            os.environ["SSPSD_K3"] = old


def decimated(sp, n, hbf, batches, seed, device_input):
    import torch
    x = uniform_noise(sum(batches), seed) + np.float32(0.25)
    out = {}
    for k3 in (None, "tma960"):
        st = make(lambda: sp.Psd(n, hbf=hbf), k3)
        ys, pos = [], 0
        for b in batches:
            xb = x[pos:pos + b]
            pos += b
            ys.append(st.process(torch.from_numpy(xb).cuda() if device_input else xb))
        torch.cuda.synchronize()
        out[k3] = np.concatenate(ys)
    return out[None], out["tma960"]


@pytest.mark.parametrize("device_input", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("n", [4096, 512])
@pytest.mark.parametrize("preset", ["TAPS_140", "TAPS_98"])
def test_decimated_stream_bit_identical(sp, preset, n, device_input):
    got, ref = decimated(sp, n, sp.Hbf[preset], BATCHES, n + len(preset), device_input)
    assert got.size == ref.size and got.size > 150_000
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), \
        "first difference at %d of %d" % (int(np.argmax(got.view(np.uint32) != ref.view(np.uint32))), got.size)


@pytest.mark.parametrize("preset", ["TAPS_140", "TAPS_98"])
def test_single_sample_batches(sp, preset):
    """outputs trickle out one tile-clip at a time: every launch is one clipped lowest tile straddling the carry"""
    got, ref = decimated(sp, 512, sp.Hbf[preset], [8] * 300 + [7] * 100 + [1] * 50, 77, False)
    assert got.size > 250
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


@pytest.mark.parametrize("n,preset", [(4096, "TAPS_140"), (512, "TAPS_98"), (512, "TAPS_140")])
def test_cascade_deterministic_bit_identical(sp, n, preset):
    """a full cascade (stage 0 and the deep stages' decimators) in deterministic mode: same rows and breaks"""
    import torch
    x = uniform_noise(6_000_000 + 4321, 0xDEC + n)
    res = {}
    for k3 in (None, "tma960"):
        c = make(lambda: sp.PsdCascade(n, hbf=sp.Hbf[preset], deterministic=True), k3)
        pos = 0
        for i, b in enumerate((700_001, 3, 2_500_000, 64_000, x.size - 3_264_004)):
            c.process(torch.from_numpy(x[pos:pos + b]).cuda() if i % 2 else x[pos:pos + b])
            pos += b
        assert pos == x.size
        res[k3] = c.psd(sp.MergeOpts(keep_overlap=True, min_count=0, keep_transition_band=True))
    (p, b), (pr, br) = res[None], res["tma960"]
    assert [(k.count, k.pending, k.bins.start, k.bins.stop, k.decimation) for k in b] == \
        [(k.count, k.pending, k.bins.start, k.bins.stop, k.decimation) for k in br]
    assert len(b) >= 3
    assert np.array_equal(p.view(np.uint32), pr.view(np.uint32))
