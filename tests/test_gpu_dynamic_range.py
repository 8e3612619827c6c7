"""The device at high dynamic range: tones, a comb, a large offset, stop-band tones and red noise through every PSD
kernel (K2), every decimator (K3), deterministic accumulation and a time-chunked group, each stage held to the
budget of dynamic_range_cases.py against the float64 model.  Needs a B200 (115 s on one).

With DYNAMIC_RANGE_PROFILE=<file> the per-stage gamma of the device and of the f32 restatement of the reference
(and the decimated-sample errors) are written there as JSON lines."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import dynamic_range_cases as D

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
FULL = dict(keep_overlap=True, min_count=0, keep_transition_band=True)
DEFAULT_K3 = "decim8_tma_kernel"

_refs = {}
_samples = {}


@pytest.fixture(scope="module")
def sp():
    import torch
    assert torch.cuda.is_available()
    import stabilizer_stream_b200 as m
    return m


@pytest.fixture(scope="module")
def record():
    rows = []
    yield lambda **kw: rows.append(kw)
    path = os.environ.get("DYNAMIC_RANGE_PROFILE")
    if path:
        with open(path, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


@pytest.fixture(scope="module")
def signal_dir(tmp_path_factory):
    return tmp_path_factory.mktemp("dynamic_range")


def reference(case):
    """the float64 rows and the restatement's gammas, kept for the module without the input (268 MB for red noise
    at N = 4096): the tests regenerate that from the case's seed"""
    if case.id not in _refs:
        r = D.Reference(case)
        r.x = None
        _refs[case.id] = r
    return _refs[case.id]


def k2_kernel(case):
    if case.window == D.orc.WINDOW_RECT and case.n == 4096:
        return "psd_stage_kernel_r16"
    if case.window == D.orc.WINDOW_HANN and case.n in (512, 4096):
        return {512: "psd_stage_kernel_w16", 4096: "psd_stage_kernel_ring"}[case.n]
    return "psd_stage_kernel<%d>" % int(np.log2(case.n))


def check_spectra(case, path, rows, record):
    r = reference(case)
    gam = r.gamma(rows)
    bad = []
    for i, (gd, gr) in enumerate(zip(gam, r.gamma_ref)):
        b = D.budget(case, gr)
        record(case=case.id, path=path, stage=i, count=r.counts[i], gamma_dev=gd, gamma_ref=gr, budget=b)
        if not gd <= b:
            bad.append("stage %d: gamma %.3g > %.3g (reference %.3g)" % (i, gd, b, gr))
    assert not bad, "%s via %s: %s" % (case.id, path, "; ".join(bad))


def check_samples(case, path, y, record):
    if case.id not in _samples:
        x = case.signal()
        st = D.orc.Stage(case.n, D.orc.WINDOW_HANN, case.hbf)
        y_ref = st.process(x)
        y64 = D.decimated_truth(case, x, st.count())
        _samples[case.id] = (y64, D.sample_error(y_ref, y64), D.sample_allowed(D.sample_error(y_ref, y64), x))
    y64, err_ref, allowed = _samples[case.id]
    err = D.sample_error(y, y64)
    record(case=case.id, path=path, samples=int(y64.size), sample_err_dev=err, sample_err_ref=err_ref, allowed=allowed)
    assert err <= allowed, "%s via %s: max|y - y64| = %.3g > %.3g (reference %.3g)" % (case.id, path, err, allowed, err_ref)


def cascade_rows(sp, case, x, **kw):
    c = sp.PsdCascade(case.n, hbf=sp.Hbf(case.hbf), **kw)
    c.set_detrend(sp.Detrend(case.detrend))
    c.process(x)
    return D.merged_rows(*c.psd(sp.MergeOpts(**FULL)))


@pytest.mark.parametrize("case", D.cases(("tone", "comb", "offset", "hbf", "red")), ids=lambda c: c.id)
def test_default_kernels(sp, record, case):
    x = case.signal()
    check_spectra(case, "%s + %s" % (k2_kernel(case), DEFAULT_K3), cascade_rows(sp, case, x), record)


@pytest.mark.parametrize("case", D.cases(("rect",)), ids=lambda c: c.id)
def test_rectangular_window_single_stage(sp, record, case):
    r = reference(case)
    g = sp.Psd(case.n, sp.Window.RECTANGULAR, hbf=sp.Hbf(case.hbf))
    g.process(case.signal())
    assert g.count() == r.counts[0]
    row = g.spectrum().astype(np.float64) / D.stage_gain(case, 0, g.count())
    check_spectra(case, k2_kernel(case), [row], record)


@pytest.mark.parametrize("case", [c for c in D.cases(("hbf",)) if c.n == 4096], ids=lambda c: c.id)
def test_decimated_samples(sp, record, case):
    y = sp.Psd(case.n, hbf=sp.Hbf(case.hbf)).process(case.signal())
    check_samples(case, DEFAULT_K3, y, record)


# the K2 variants on the PSD cases at their size, the K3 variants on the stop-band and red-noise cases
VARIANTS = ([({"SSPSD_K2": v}, 4096) for v in ("r16", "r8", "ring1", "ring1x5")] + [({"SSPSD_K2": "r8"}, 512)] +
            [({"SSPSD_K3": v}, None) for v in ("tiled", "tma640", "tma768", "async960", "async640", "pf960", "pf640")])


@pytest.mark.parametrize("env,n", VARIANTS, ids=["%s=%s" % (*e.items(),)[0] + ("-n%d" % n if n else "") for e, n in VARIANTS])
def test_kernel_variants(record, signal_dir, tmp_path, env, n):
    cases = [c for c in D.cases(("tone", "comb", "offset")) if c.n == n] if n else D.cases(("hbf", "red"))
    for c in cases:
        f = signal_dir / (c.id + ".npy")
        if not f.exists():
            np.save(f, c.signal())
    out = tmp_path / "rows.npz"
    e = dict(os.environ)
    e.update(env)
    e["PYTHONPATH"] = os.pathsep.join([os.path.dirname(HERE), HERE, e.get("PYTHONPATH", "")])
    r = subprocess.run([sys.executable, os.path.join(HERE, "dynamic_range_check.py"), str(signal_dir), str(out)] +
                       [c.id for c in cases], env=e, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "dynamic range run ok" in r.stdout, r.stdout[-500:] + r.stderr[-1500:]
    res = np.load(out)
    path = " ".join("%s=%s" % kv for kv in env.items())
    failures = []
    for c in cases:
        rows = [res["%s:rows%d" % (c.id, i)] for i in range(len(reference(c).counts))]
        try:
            check_spectra(c, path, rows, record)
            if c.group == "hbf" and c.n == 4096:
                check_samples(c, path, res[c.id + ":samples"], record)
        except AssertionError as err:
            failures.append(str(err))
    assert not failures, "\n".join(failures)


@pytest.mark.parametrize("cid", ["comb-n512-0-h1-d0", "comb-n4096-0-h1-d0", "tone-n4096-2045p37-h1-d0",
                                 "offset-n4096-0-h1-d3", "offset-n512-0-h1-d2", "red-n512-2-h1-d0"])
def test_deterministic_accumulation(sp, record, cid):
    case = D.case_by_id(cid)
    rows = cascade_rows(sp, case, case.signal(), deterministic=True)
    check_spectra(case, "%s + reduce_partials_kernel" % k2_kernel(case), rows, record)


@pytest.mark.parametrize("cid", ["tone-n4096-512p37-h1-d0", "comb-n512-0-h1-d0", "tone-n1024-509p37-h1-d0",
                                 "offset-n512-0-h1-d3"])
def test_power_of_two_scale_is_exact(sp, cid):
    """x 2^+-30 scales every readout bin by exactly 2^+-60: no flush to zero and no overflow in the range the
    kernels use (deterministic accumulation, so the order of the sums is fixed)."""
    case = D.case_by_id(cid)
    x = case.signal()

    def readout(s):
        c = sp.PsdCascade(case.n, hbf=sp.Hbf(case.hbf), deterministic=True)
        c.set_detrend(sp.Detrend(case.detrend))
        c.process(x * np.float32(s))
        return np.concatenate(D.merged_rows(*c.psd(sp.MergeOpts(**FULL)))).astype(np.float32)

    p = readout(1.0)
    assert p.size and np.all(np.isfinite(p))
    for e in (30, -30):
        want = p * np.float32(2.0 ** (2 * e))
        got = readout(2.0 ** e)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (cid, e, np.max(np.abs(got / want - 1)))


@pytest.mark.parametrize("order", [1, 2])
def test_time_chunked_group_red_noise(sp, record, order):
    """three ranks on GPU 0, each starting its stages from a warm-up halo of the previous rank's range"""
    case = D.Case("red", 512, order)
    x = case.signal()
    g = sp.Group(case.n, devices=[0, 0, 0], mode=sp.ShardMode.TIME, hbf=sp.Hbf(case.hbf))
    g.time_plan(x.size, 3)
    g.time_process_all(x)
    g.time_finish()
    rows = D.merged_rows(*g.psd(0, sp.MergeOpts(**FULL)))
    check_spectra(case, "time-chunked group of 3", rows, record)


@pytest.mark.parametrize("n,detrend", [(64, 0), (64, 1), (512, 0), (512, 1)])
def test_large_offset_distribution(sp, record, n, detrend):
    """A 1e4 offset over 40 seeds.  The deep stages hold 1-5 segments, so one seed's gamma is one draw of the rounding;
    the device is held to the restatement's distribution instead: per stage its median gamma is within 1.6x of the
    restatement's (measured on a B200: at most 1.46x, N = 64 Midpoint stage 1) and its worst within GAMMA_OFFSET.
    The difference lives in the decimator: its samples' median error is within 1.25x of the restatement's (measured
    1.08x after one stage, 1.13x after two); the PSD kernel on the restatement's own stage-2 input is as accurate."""
    gd, gr, ed, er = [], [], [], []
    for seed in range(40):
        x = (1e4 + np.random.default_rng(1000 + seed).standard_normal(200 * n)).astype(np.float32)
        case = D.Case("offset", n, detrend=detrend)
        r = D.Reference(case, x)
        gr.append(r.gamma_ref)
        gd.append(r.gamma(cascade_rows(sp, case, x)))
        st = D.orc.Stage(n)
        y1 = st.process(x)
        y64 = D.decimated_truth(case, x, st.count())
        er.append(D.sample_error(y1, y64))
        ed.append(D.sample_error(sp.Psd(n).process(x), y64))
    gd, gr = np.array(gd), np.array(gr)
    for i in range(gd.shape[1]):
        record(case="offset-n%d-d%d-40seeds" % (n, detrend), path="default kernels", stage=i, gamma_dev_median=np.median(gd[:, i]),
               gamma_ref_median=np.median(gr[:, i]), gamma_dev_max=gd[:, i].max(), gamma_ref_max=gr[:, i].max())
    record(case="offset-n%d-d%d-40seeds" % (n, detrend), path=DEFAULT_K3, sample_err_dev_median=np.median(ed),
           sample_err_ref_median=np.median(er))
    assert np.all(gd.max(0) <= D.GAMMA_OFFSET), gd.max(0)
    assert np.all(np.median(gd, 0) <= 1.6 * np.median(gr, 0)), (np.median(gd, 0), np.median(gr, 0))
    assert np.median(ed) <= 1.25 * np.median(er), (np.median(ed), np.median(er))
