"""Independent float64 model of the cascaded cross-spectral density (TEST INFRASTRUCTURE ONLY).

The reference has no CSD: this is model_f64.cascade() with |X|^2 replaced by conj(X) Y for the cross row
(Psd::process with |c|^2 replaced by conj(cx) cy, DESIGN.md section 3a).  Whole-stream numpy f64 rfft, reusing
model_f64's stage(), hbf8(), window(), detrend() and merge().
"""
import numpy as np

from .model_f64 import DEPTH, DRAIN, detrend, hbf8, merge, stage, window


def cross_stage(x, y, n, win_kind=1, det=0, avg=2 ** 32 - 1, preset=1):
    """stage() over two streams: the spectrum of x, and for the same segments sum g |Y|^2 and sum g conj(X) Y."""
    x, y = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    st = stage(x, n, win_kind, det, avg, preset)
    w, _, _, overlap = window(n, win_kind)
    hop = n - overlap
    craw = st["count_raw"]
    syy, sxy = np.zeros(n // 2 + 1), np.zeros(n // 2 + 1, np.complex128)
    if craw:
        idx = np.arange(n)[None, :] + hop * np.arange(craw)[:, None]
        X = np.fft.rfft(detrend(x[idx], det) * w, axis=-1)
        Y = np.fft.rfft(detrend(y[idx], det) * w, axis=-1)
        Pyy, Pxy = Y.real ** 2 + Y.imag ** 2, np.conj(X) * Y
        if avg >= craw:
            syy, sxy = Pyy.sum(axis=0), Pxy.sum(axis=0)
        else:
            count = 0
            for k in range(craw):
                g = 1.0
                if count > avg:
                    g = np.float64(np.float32(avg) / np.float32(count))
                    count = avg
                count += 1
                syy, sxy = g * syy + Pyy[k], g * sxy + Pxy[k]
    D = n + (craw - 1) * hop if craw else 0
    st["spectrum_yy"], st["spectrum_xy"] = syy, sxy
    st["decimated_y"] = hbf8(y[:D], preset)[DRAIN[preset]:] if D else np.zeros(0)
    return st


def cross_cascade(x, y, n, det=0, avg_limit=2 ** 32 - 1, avg_count=2 ** 32 - 1, preset=1, win_kind=1):
    """The cascaded cross-spectral density of x and y: per-stage dicts as model_f64.cascade() returns, with
    spectrum_yy and spectrum_xy (complex) beside the spectrum of x."""
    out = []
    s, t = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    assert s.size == t.size
    i = 0
    while s.size > 0:
        avg = min(avg_count >> (DEPTH * i) if DEPTH * i < 32 else 0, avg_limit)
        st = cross_stage(s, t, n, win_kind, det, avg, preset)
        st["avg"] = avg
        out.append(st)
        s, t = st["decimated"], st["decimated_y"]
        i += 1
    return out


def merge_cross(stages, n, **opts):
    """merge() of the three rows of cross_cascade(): (pxx, pyy, pxy, breaks)"""
    pxx, breaks = merge(stages, n, **opts)
    pyy, _ = merge([dict(st, spectrum=st["spectrum_yy"]) for st in stages], n, **opts)
    pxy, _ = merge([dict(st, spectrum=st["spectrum_xy"]) for st in stages], n, **opts)
    return pxx, pyy, pxy.astype(np.complex128), breaks
