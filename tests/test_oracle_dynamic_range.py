"""The error budget of the high-dynamic-range parity tests, justified on the CPU: the f32 restatement of the
reference (oracle.Cascade, oracle.Stage) against the float64 model on the cases of dynamic_range_cases.py.  The
device is held to gamma = 1e-7 (tests/test_gpu_dynamic_range.py); the reference's own arithmetic needs at most
half of that here, and a dropped 140 dB decimator tap is far outside the decimated-sample bound."""
import numpy as np
import pytest

import dynamic_range_cases as D

SPECTRUM_CASES = [c for c in D.cases() if not c.large_offset]
HBF_CASES = [c for c in D.cases(("hbf",)) if c.n == 4096]


@pytest.mark.parametrize("case", SPECTRUM_CASES, ids=lambda c: c.id)
def test_restatement_meets_the_spectrum_budget(oracle, case):
    r = D.Reference(case)
    assert len(r.counts) == {"rect": 1, "red": 5}.get(case.group, 3), (case.id, r.counts)
    worst = max(r.gamma_ref)
    assert worst <= D.GAMMA, (case.id, r.gamma_ref)
    assert worst <= D.GAMMA_REF_MAX, (case.id, r.gamma_ref)


@pytest.mark.parametrize("detrend", [0, 1])
def test_restatement_offset_floor(oracle, detrend):
    """Under a 1e4 offset the deepest stage of N = 64 holds one segment, and one draw of the f32 rounding decides its
    gamma: over 40 seeds the restatement itself needs 0.9e-7 (None) and 1.4e-7 (Midpoint) there, so 1e-7 cannot be
    the offset floor."""
    worst = 0.0
    for seed in range(40):
        x = (1e4 + np.random.default_rng(1000 + seed).standard_normal(200 * 64)).astype(np.float32)
        r = D.Reference(D.Case("offset", 64, detrend=detrend), x)
        assert r.counts[-1] == 1
        worst = max(worst, max(r.gamma_ref))
    assert D.GAMMA / 2 < worst <= D.GAMMA_OFFSET / 2, worst


@pytest.mark.parametrize("case", HBF_CASES, ids=lambda c: c.id)
def test_restatement_decimated_samples(oracle, case):
    x = case.signal()
    st = oracle.Stage(case.n, oracle.WINDOW_HANN, case.hbf)
    y = st.process(x)
    y64 = D.decimated_truth(case, x, st.count())
    err = D.sample_error(y, y64)
    assert err <= D.SAMPLE_REF_MAX * float(np.max(np.abs(x))), (case.id, err)
    assert err <= D.sample_allowed(err, x)


@pytest.mark.parametrize("freq", [0.095, 0.05, 0.0])
def test_a_dropped_outer_tap_breaks_the_sample_bound(oracle, monkeypatch, freq):
    """The outermost tap of the 140 dB preset's lowest-rate half-band is 7.6e-7: dropping it moves white-noise
    output by ~1e-6, inside the old atol=3e-6, but puts a tone's decimated samples ~6e-6 off."""
    from oracle import model_f64 as m64
    case = D.Case("hbf", 4096, freq, hbf=oracle.HBF_140)
    x = case.signal()
    st = oracle.Stage(case.n, oracle.WINDOW_HANN, case.hbf)
    y = st.process(x)
    y64 = D.decimated_truth(case, x, st.count())
    allowed = D.sample_allowed(D.sample_error(y, y64), x)
    taps = [list(s) for s in m64.TAPS]
    taps[case.hbf] = [t.copy() for t in m64.TAPS[case.hbf]]
    taps[case.hbf][0][0] = 0.0
    monkeypatch.setattr(m64, "TAPS", taps)
    assert D.sample_error(D.decimated_truth(case, x, st.count()), y64) > 4 * allowed


def test_gamma_needed_is_the_tightest_budget():
    rng = np.random.default_rng(3)
    truth = 10.0 ** rng.uniform(-12, 0, 500)
    S = 50.0
    dev = truth * (1 + rng.uniform(-3e-4, 3e-4, truth.size)) + 1e-9
    g = D.gamma_needed(dev, truth, S)
    bound = lambda gam: D.RTOL * truth + gam * np.sqrt(truth * S) + gam * gam * S
    assert np.all(np.abs(dev - truth) <= bound(g) * (1 + 1e-12))
    assert not np.all(np.abs(dev - truth) <= bound(g * (1 - 1e-6)))
    assert D.gamma_needed(truth, truth, S) == 0.0


def test_case_table_covers_the_special_bins():
    ids = {c.id for c in D.cases()}
    assert len(ids) == len(D.cases())
    for n, ks in ((4096, (128, 384, 256, 2048, 2045.37)), (512, (8, 24, 248, 256)), (1024, (64, 128, 192))):
        for k in ks:
            assert D.Case("tone", n, float(k)).id in ids, (n, k)
    assert {c.detrend for c in D.cases(("offset",))} == {0, 1, 2, 3}
    assert {(c.hbf, c.param) for c in D.cases(("hbf",))} == {(h, f) for h in (0, 1) for f in D.HBF_FREQS}
