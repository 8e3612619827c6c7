"""High-dynamic-range cases and the error budget that scales with the signal (DESIGN.md section 4).

White noise hides the faults an FFT or FIR kernel is most likely to have (a twiddle or split constant a few ulp
off, a dropped or mis-indexed decimator tap): they move a white spectrum by ~1e-6 relative, far inside the 1e-4
per-bin rule.  A tone, a stop-band tone or red noise puts 100-150 dB between the loudest and the quietest bins, and
there the same faults stand out.  The per-bin 1e-4 rule cannot be used as it is at that range (the reference's own
f32 arithmetic breaks it in most bins of a deep stage), so each stage i is held to

    |dev_k - t_k| <= 1e-4 t_k + gamma sqrt(t_k S_i) + gamma^2 S_i                      for every bin k

with t the float64 row and S_i = count_i N sum(w^2) 64^i mean(x^2) the power the stage and the decimators before
it handled (each half-band has gain 2).  The middle term is the cross term of an f32 rounding error of relative
size gamma against the bin's own amplitude, the last one the floor it leaves in empty bins.

Every generator synthesises in float64 and rounds once to float32; seeds derive from the case id.
"""
import zlib
from dataclasses import dataclass

import numpy as np

from oracle import binding as orc
from oracle import model_f64 as m64

RTOL = 1e-4
GAMMA = 1e-7          # device budget for tones, combs, stop-band tones and red noise
GAMMA_REF_MAX = 5e-8  # what the f32 restatement of the reference needs on those cases (worst measured: 2.8e-8)
GAMMA_OFFSET = 4e-7   # floor of the large-offset cases.  Their deep stages hold 1-5 segments, so one draw of the rounding
#                       decides; over 40 seeds x N = 64, 512 x None, Midpoint the restatement needs up to 1.5e-7 and the
#                       device up to 3.1e-7 (profiles/r03_offset_seeds.jsonl): under a 1e4 offset the device decimator's
#                       samples are ~1.1x further from f64 than the restatement's (test_large_offset_distribution)
SAMPLE_REF_MAX = 1e-6  # max|y_ref - y64| / max|x| of the restatement's decimator on the hbf cases
NOISE = 1e-5          # white noise under the tones: ~100 dB below the tone per bin at N = 4096
SIZES = (64, 512, 1024, 4096, 8192)
HBF_FREQS = (0.38, 0.19, 0.095, 0.05, 0.025, 0.0)  # stop bands of half-bands A, B, C; transition band; passband
#                                                    edge 0.4 / 16; DC (fractions of the input rate)


def special_bins(n):
    """Bins that a kernel computes on a path of their own."""
    if n == 4096:  # ring / radix-16 kernels: thread 0 owns the multiples of 128, W_32 split of the odd ones
        return [128, 384, 640, 1152, 1920, 256, 768, 1280, 1792]
    if n == 512:   # warp kernel: lanes 0 and 8 are their own shuffle partners
        return [8, 24, 40, 120, 248]
    k = n // 8     # generic kernel: K = M / 4, the bins K / 2 and K use twN[K / 2], twN[K / 2 + K]
    return [k // 2, k, k // 2 + k]


def tone_bins(n):
    base = [1, 3, n // 8, n // 4, n // 2 - 3]
    ks = base + [k + 0.37 for k in base] + [n // 2] + special_bins(n)
    return sorted(set(float(k) for k in ks))


@dataclass(frozen=True)
class Case:
    group: str       # tone | rect | comb | offset | hbf | red
    n: int
    param: float = 0.0   # tone bin, hbf frequency (of the input rate), red-noise order
    hbf: int = orc.HBF_140
    detrend: int = orc.DETREND_NONE

    @property
    def id(self):
        p = ("%g" % self.param).replace(".", "p")
        return "%s-n%d-%s-h%d-d%d" % (self.group, self.n, p, self.hbf, self.detrend)

    @property
    def seed(self):
        return zlib.crc32(self.id.encode())

    @property
    def window(self):
        return orc.WINDOW_RECT if self.group == "rect" else orc.WINDOW_HANN

    @property
    def length(self):
        return 8 ** 4 * self.n * 4 if self.group == "red" else 200 * self.n

    @property
    def large_offset(self):
        return self.group == "offset"

    def signal(self):
        rng = np.random.default_rng(self.seed)
        n, L = self.n, self.length
        t = np.arange(L, dtype=np.float64)
        if self.group in ("tone", "rect"):
            x = np.cos(2 * np.pi * self.param / n * t + rng.uniform(0, 2 * np.pi)) + NOISE * rng.standard_normal(L)
        elif self.group == "comb":
            # unit tones at every k = 3 (mod 16), random phases; their split images fall on k = 13 (mod 16), which
            # stays empty.  On-bin tones are N-periodic: one period, tiled.
            spec = np.zeros(n // 2 + 1, np.complex128)
            ks = np.arange(3, n // 2, 16)
            spec[ks] = n / 2 * np.exp(1j * rng.uniform(0, 2 * np.pi, ks.size))
            x = np.tile(np.fft.irfft(spec, n), L // n) + NOISE * rng.standard_normal(L)
        elif self.group == "offset":
            x = 1e4 + rng.standard_normal(L)
        elif self.group == "hbf":
            phase = rng.uniform(0, 2 * np.pi) if self.param else 0.0
            x = np.cos(2 * np.pi * self.param * t + phase)
        elif self.group == "red":
            x = rng.standard_normal(L)
            for _ in range(int(self.param)):
                x = np.cumsum(x)
        else:
            raise ValueError(self.group)
        return x.astype(np.float32)


def cases(group=None):
    out = []
    for n in SIZES:
        out += [Case("tone", n, k) for k in tone_bins(n)]
        out.append(Case("comb", n))
        out += [Case("offset", n, detrend=d) for d in range(4)]
    for n in (512, 4096):
        out += [Case("rect", n, k) for k in (3.0, 3.37, n / 8, n / 8 + 0.37, n // 2 - 3, n // 2)]
        out += [Case("hbf", n, f, hbf=h) for h in (orc.HBF_98, orc.HBF_140) for f in HBF_FREQS]
        out += [Case("red", n, order) for order in (1, 2)]
    return [c for c in out if group is None or c.group in group]


def case_by_id(cid):
    for c in cases():
        if c.id == cid:
            return c
    raise KeyError(cid)


def stage_power(case, x, stage, count):
    """S_i in the units of the stage's raw accumulator row."""
    w = m64.window(case.n, case.window)[0]
    return count * case.n * float(np.sum(w * w)) * 64.0 ** stage * float(np.mean(np.asarray(x, np.float64) ** 2))


def stage_gain(case, stage, count):
    """The factor PsdCascade::psd divides the stage's row by (gain * decimation, src/psd.rs:516)."""
    _, power, nenbw, _ = m64.window(case.n, case.window)
    return (case.n // 2) * count * nenbw * power * 8.0 ** stage


def gamma_needed(dev, truth, S):
    """Smallest gamma for which every bin of `dev` meets the bound against the float64 row `truth`."""
    dev = np.asarray(dev, np.float64)
    truth = np.asarray(truth, np.float64)
    e = np.maximum(np.abs(dev - truth) - RTOL * truth, 0.0)
    a = np.sqrt(np.maximum(truth, 0.0) * S)
    return float(np.max(2 * e / (a + np.sqrt(a * a + 4 * S * e))))  # positive root of S g^2 + a g - e


def budget(case, gamma_ref):
    """gamma a device row must meet: the device is never worse than the reference's own arithmetic"""
    return max(GAMMA_OFFSET, gamma_ref) if case.large_offset else GAMMA


class Reference:
    """The float64 truth and the f32 restatement of the reference for one case, per stage in merged units
    (the row divided by gain_i 8^i, as PsdCascade::psd reads it out)."""

    def __init__(self, case, x=None):
        self.case = case
        self.x = case.signal() if x is None else x
        n = case.n
        if case.group == "rect":
            t = orc.CascadeF64(n, hbf=case.hbf, window=case.window, detrend=case.detrend, max_stages=1)
            o = orc.Stage(n, case.window, case.hbf)
            o.set_detrend(case.detrend)
            o.process(self.x)
            ref = [(o.spectrum(), o.count())]
        else:
            t = orc.CascadeF64(n, hbf=case.hbf, detrend=case.detrend)
            o = orc.Cascade(n, case.hbf)
            o.set_detrend(case.detrend)
            o.process(self.x)
            ref = [(o.stage_spectrum(i), o.stage_count(i)) for i in range(o.num_stages())]
        t.process(self.x)
        self.truth, self.S, self.counts, self.gamma_ref = [], [], [], []
        for i, (row, cnt) in enumerate(ref):
            t_row, t_cnt, _, _ = t.stage(i)
            assert t_cnt == cnt, (case.id, i, t_cnt, cnt)
            if cnt == 0:
                break
            g = stage_gain(case, i, cnt)
            self.counts.append(cnt)
            self.truth.append(t_row / g)
            self.S.append(stage_power(case, self.x, i, cnt) / g)
            self.gamma_ref.append(gamma_needed(row / g, self.truth[i], self.S[i]))

    def gamma(self, rows):
        """per-stage gamma a list of merged-unit rows (stage 0 first) needs"""
        assert len(rows) == len(self.truth), (self.case.id, len(rows), len(self.truth))
        return [gamma_needed(r, t, S) for r, t, S in zip(rows, self.truth, self.S)]


def merged_rows(p, breaks):
    """Per-stage rows (stage 0 first) of a readout taken with MergeOpts(keep_overlap=True, min_count=0,
    keep_transition_band=True); stages without a segment are left out."""
    rows = {}
    for b in breaks:
        if b.count:
            stage = int(round(np.log(b.decimation) / np.log(8)))
            rows[stage] = np.asarray(p[b.start:b.start + len(b.bins)], np.float64)
    return [rows[i] for i in range(len(rows))]


def decimated_truth(case, x, count):
    """model_f64.hbf8 over the samples the stage's `count` segments consumed, without the zero-state drain: what
    Psd(n).process(x) returns"""
    hop = case.n // 2
    d = case.n + (count - 1) * hop
    return m64.hbf8(x[:d], case.hbf)[m64.DRAIN[case.hbf]:]


def sample_error(y, y64):
    y = np.asarray(y, np.float64)
    assert y.shape == y64.shape, (y.shape, y64.shape)
    return float(np.max(np.abs(y - y64)))


def sample_allowed(err_ref, x):
    """max|y_dev - y64| <= 2 max|y_ref - y64| + 2^-24 max|x|"""
    return 2 * err_ref + 2.0 ** -24 * float(np.max(np.abs(x)))
