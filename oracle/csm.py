"""The cross-spectral matrix of K streams, composed pairwise from the CSD references (no new C).

Row (i, j) of the f32 restatement is oracle.xbinding.XCascade(x_i, x_j): the oracle transforms each channel on its
own, so S_ii from the pair (i, j) is the same for every j.  The float64 truth is model_f64_csd.cross_cascade over
the same pairs."""
import itertools

import numpy as np

from oracle import model_f64_csd as mcsd
from oracle import xbinding


class CsmCascade:
    """K = 2 .. 4 streams through one pairwise XCascade per pair i < j; csm() -> (S complex [K, K, bins], breaks)"""

    def __init__(self, n, k, window=xbinding.WINDOW_HANN, hbf=xbinding.HBF_140):
        self.n, self.k = n, k
        self.pairs = {p: xbinding.XCascade(n, window=window, hbf=hbf) for p in itertools.combinations(range(k), 2)}

    def set_avg(self, limit, count):
        for c in self.pairs.values():
            c.set_avg(limit, count)

    def set_detrend(self, d):
        for c in self.pairs.values():
            c.set_detrend(d)

    def process(self, xs):
        assert len(xs) == self.k
        for (i, j), c in self.pairs.items():
            c.process(xs[i], xs[j])

    def num_stages(self):
        return self.pairs[(0, 1)].num_stages()

    def csm(self):
        rows = {p: c.csd() for p, c in self.pairs.items()}
        return _assemble(self.k, {p: r[:3] for p, r in rows.items()}, np.complex64), rows[(0, 1)][3]


def _assemble(k, rows, dtype):
    """{(i, j): (pxx, pyy, pxy)} -> S [k, k, bins]; the diagonal from the first pair holding the channel"""
    m = rows[(0, 1)][0].size
    s = np.zeros((k, k, m), dtype)
    done = set()
    for (i, j), (pxx, pyy, pxy) in rows.items():
        s[i, j] = pxy
        s[j, i] = np.conj(pxy)
        for c, p in ((i, pxx), (j, pyy)):
            if c not in done:
                s[c, c] = p
                done.add(c)
    return s


def f64_matrix(xs, n, det=0, preset=1, win_kind=1, avg_limit=2 ** 32 - 1, avg_count=2 ** 32 - 1):
    """-> (S complex128 [K, K, bins], breaks as model_f64_csd.merge_cross returns them)"""
    k = len(xs)
    rows, breaks = {}, None
    for i, j in itertools.combinations(range(k), 2):
        st = mcsd.cross_cascade(xs[i], xs[j], n, det, avg_limit=avg_limit, avg_count=avg_count, preset=preset,
                                win_kind=win_kind)
        pxx, pyy, pxy, b = mcsd.merge_cross(st, n)
        rows[(i, j)] = (pxx, pyy, pxy)
        breaks = breaks or b
    return _assemble(k, rows, np.complex128), breaks
