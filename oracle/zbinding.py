"""ctypes binding of the CPU restatement of the two-sided spectrum of z = i + i q, oracle/sspsd_zoracle.c (TEST
INFRASTRUCTURE ONLY; the reference has no two-sided spectrum, see DESIGN.md section 3c), and the heterodyne mixer's
model.

sspsd_zoracle.c (which includes sspsd_xoracle.c) is linked with sspsd_oracle.c into its own shared object, built and
placed as oracle/xbinding.py builds the CSD restatement.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from .binding import HBF_140, WINDOW_HANN, WINDOW_RECT, Break, _f32, _fp, _ptr  # noqa: F401
from .xbinding import CFLAGS

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = ("sspsd_zoracle.c", "sspsd_oracle.c", "sspsd_xoracle.c", "sspsd_oracle.h", "hbf_taps.h")
_lib = None


def lib_path():
    h = hashlib.sha1()
    try:
        with open("/proc/cpuinfo") as f:
            h.update(next((line for line in f if line.startswith("flags")), "").encode())
    except OSError:
        pass
    for name in _SOURCES:
        with open(os.path.join(_HERE, name), "rb") as f:
            h.update(f.read())
    key = h.hexdigest()[:12]
    build_dir = os.path.join(_HERE, "_build")
    out = os.path.join(build_dir, key, "libsspsd_zoracle.so")
    if os.path.exists(out) or os.access(build_dir if os.path.isdir(build_dir) else _HERE, os.W_OK):
        return out
    return os.path.join(tempfile.gettempdir(), "sspsd_oracle_%d" % os.getuid(), key, "libsspsd_zoracle.so")


def build():
    out = lib_path()
    if not os.path.exists(out):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        cc = os.environ.get("CC", "gcc")
        tmp = out + ".%d.tmp" % os.getpid()
        r = subprocess.run([cc] + CFLAGS + ["-shared", "-o", tmp] + [os.path.join(_HERE, s) for s in _SOURCES[:2]]
                           + ["-lm", "-lpthread"], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("two-sided oracle build failed:\n" + r.stdout + r.stderr)
        os.replace(tmp, out)
    return out


def lib():
    global _lib
    if _lib is not None:
        return _lib
    L = C.CDLL(build())
    vp = C.c_void_p
    sig = {
        "orc_xcascade_new": (vp, [C.c_int, C.c_int, C.c_int]),
        "orc_xcascade_free": (None, [vp]),
        "orc_xcascade_set_avg": (None, [vp, C.c_uint32, C.c_uint32]),
        "orc_xcascade_set_detrend": (None, [vp, C.c_int]),
        "orc_zcascade_process": (None, [vp, _fp, _fp, C.c_size_t]),
        "orc_xcascade_num_stages": (C.c_size_t, [vp]),
        "orc_xcascade_csd": (C.c_size_t, [vp, C.c_int, C.c_uint32, C.c_int, _fp, _fp, _fp, C.POINTER(Break),
                                         C.POINTER(C.c_size_t)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def phase_cos_sin(n, ftw):
    """(cos, sin) of 2 pi phi_n / 2^32 in float64, phi_n = (n ftw) mod 2^32 from the integer index n (uint64 array):
    the quadrant from phi's top two bits, the rest an exact argument below a quarter turn, so multiples of a quarter
    turn give exactly 0 and +-1"""
    n = np.asarray(n, dtype=np.uint64)
    phi = (n * np.uint64(ftw)) & np.uint64(0xFFFFFFFF)
    quad = (phi >> np.uint64(30)).astype(np.int64)
    a = (phi & np.uint64(0x3FFFFFFF)).astype(np.float64) * (np.pi / 2.0 ** 31)
    c, s = np.cos(a), np.sin(a)
    cs = [(c, s), (-s, c), (-c, -s), (s, -c)]
    cos = np.choose(quad, [v[0] for v in cs])
    sin = np.choose(quad, [v[1] for v in cs])
    return cos, sin


def heterodyne(x, ftw, pos0=0):
    """the mixer in float64: (x cos, -x sin) of the absolute phase, samples pos0 .. pos0 + len(x) - 1"""
    x = np.asarray(x, dtype=np.float64)
    c, s = phase_cos_sin(np.arange(x.size, dtype=np.uint64) + np.uint64(pos0), ftw)
    return x * c, -x * s


class ZCascade:
    """Two-sided spectrum of z = i + i q: P+ = sum g |Z[k]|^2 and P- = sum g |Z[N-k]|^2 per stage, merged like
    PsdCascade::psd and halved (the two-sided density).  ftw != None: heterodyne mode, process(x) mixes x in float64
    from the integer phase and rounds i and q to float32."""

    def __init__(self, n, window=WINDOW_HANN, hbf=HBF_140, ftw=None):
        self.n = n
        self.ftw = ftw
        self.pos = 0
        self._h = lib().orc_xcascade_new(n, window, hbf)
        if not self._h:
            raise ValueError("unsupported cascade configuration")

    def set_avg(self, limit, count):
        lib().orc_xcascade_set_avg(self._h, limit, count)

    def set_detrend(self, d):
        lib().orc_xcascade_set_detrend(self._h, d)

    def process(self, x, q=None):
        if self.ftw is not None:
            assert q is None
            i64, q64 = heterodyne(x, self.ftw, self.pos)
            self.pos += i64.size
            i, q = i64.astype(np.float32), q64.astype(np.float32)
        else:
            i, q = _f32(x), _f32(q)
        assert i.size == q.size
        lib().orc_zcascade_process(self._h, _ptr(i), _ptr(q), i.size)

    def num_stages(self):
        return lib().orc_xcascade_num_stages(self._h)

    def spectrum(self, keep_overlap=False, min_count=1, keep_transition_band=False):
        """-> (p_pos, p_neg, breaks)"""
        ns = max(self.num_stages(), 1)
        cap = ns * (self.n // 2 + 1)
        pp, pn, unused = np.zeros(cap, np.float32), np.zeros(cap, np.float32), np.zeros(2 * cap, np.float32)
        b = (Break * ns)()
        nb = C.c_size_t()
        n = lib().orc_xcascade_csd(self._h, int(keep_overlap), min_count, int(keep_transition_band), _ptr(pp),
                                   _ptr(pn), _ptr(unused), b, C.byref(nb))
        half = np.float32(0.5)
        return pp[:n] * half, pn[:n] * half, [b[i] for i in range(nb.value)]

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:  # (module globals vanish at interpreter exit)
            _lib.orc_xcascade_free(self._h)
            self._h = None
