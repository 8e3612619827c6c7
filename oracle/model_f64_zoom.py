"""Independent float64 model of the two-sided cascaded spectrum of z = i + i q (TEST INFRASTRUCTURE ONLY).

model_f64.cascade() over the real and imaginary parts in lockstep: segments, window, detrend of each part and the
half-band decimators from model_f64 (stage(), hbf8(), window(), detrend(), merge()), with one numpy complex FFT of
z per segment and the rows P+[k] = sum g |Z[k]|^2, P-[k] = sum g |Z[N-k]|^2, k = 0 .. N/2.  The merge is
model_f64.merge() on each row, halved: the two-sided density (DESIGN.md section 3c).
"""
import numpy as np

from .model_f64 import DEPTH, DRAIN, detrend, hbf8, merge, stage, window


def zoom_stage(i, q, n, win_kind=1, det=0, avg=2 ** 32 - 1, preset=1):
    """stage() of i for the bookkeeping and i's decimation, with spectrum_pos / spectrum_neg of z and q's decimation"""
    i, q = np.asarray(i, dtype=np.float64), np.asarray(q, dtype=np.float64)
    st = stage(i, n, win_kind, det, avg, preset)
    w, _, _, overlap = window(n, win_kind)
    hop = n - overlap
    craw = st["count_raw"]
    spos, sneg = np.zeros(n // 2 + 1), np.zeros(n // 2 + 1)
    if craw:
        idx = np.arange(n)[None, :] + hop * np.arange(craw)[:, None]
        Z = np.fft.fft(detrend(i[idx], det) * w + 1j * (detrend(q[idx], det) * w), axis=-1)
        P = Z.real ** 2 + Z.imag ** 2
        k = np.arange(n // 2 + 1)
        Ppos, Pneg = P[:, k], P[:, (n - k) % n]
        if avg >= craw:
            spos, sneg = Ppos.sum(axis=0), Pneg.sum(axis=0)
        else:
            count = 0
            for s in range(craw):
                g = 1.0
                if count > avg:
                    g = np.float64(np.float32(avg) / np.float32(count))
                    count = avg
                count += 1
                spos, sneg = g * spos + Ppos[s], g * sneg + Pneg[s]
    D = n + (craw - 1) * hop if craw else 0
    st["spectrum"], st["spectrum_neg"] = spos, sneg
    st["decimated_q"] = hbf8(q[:D], preset)[DRAIN[preset]:] if D else np.zeros(0)
    return st


def zoom_cascade(i, q, n, det=0, avg_limit=2 ** 32 - 1, avg_count=2 ** 32 - 1, preset=1, win_kind=1):
    """per-stage dicts as model_f64.cascade() returns, with spectrum = P+ and spectrum_neg = P-"""
    out = []
    s, t = np.asarray(i, dtype=np.float64), np.asarray(q, dtype=np.float64)
    assert s.size == t.size
    k = 0
    while s.size > 0:
        avg = min(avg_count >> (DEPTH * k) if DEPTH * k < 32 else 0, avg_limit)
        st = zoom_stage(s, t, n, win_kind, det, avg, preset)
        st["avg"] = avg
        out.append(st)
        s, t = st["decimated"], st["decimated_q"]
        k += 1
    return out


def merge_zoom(stages, n, **opts):
    """merge() of both rows, halved: (p_pos, p_neg, breaks)"""
    pp, breaks = merge(stages, n, **opts)
    pn, _ = merge([dict(st, spectrum=st["spectrum_neg"]) for st in stages], n, **opts)
    return pp / 2, pn / 2, breaks


def mix(x, ftw, pos0=0):
    """the heterodyne mixer in float64 from the integer phase: (x cos, -x sin), see oracle/zbinding.py"""
    from .zbinding import heterodyne
    return heterodyne(x, ftw, pos0)
