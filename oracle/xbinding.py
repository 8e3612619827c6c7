"""ctypes binding of the CPU restatement of the cross-spectral density, oracle/sspsd_xoracle.c (TEST INFRASTRUCTURE
ONLY; the reference has no CSD, see DESIGN.md section 3a).

sspsd_xoracle.c is linked with sspsd_oracle.c into its own shared object, with the flags of oracle/Makefile, into a
directory keyed on the host CPU's feature flags and the sources (see binding.py for why), or into a per-user
temporary directory when the tree is read-only.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from .binding import HBF_140, WINDOW_HANN, WINDOW_RECT, Break, _f32, _fp, _ptr  # noqa: F401

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = ("sspsd_xoracle.c", "sspsd_oracle.c", "sspsd_oracle.h", "hbf_taps.h")
# oracle/Makefile's CFLAGS: -ffp-contract=off because rustc never contracts a*b+c into an FMA
CFLAGS = ["-O3", "-march=native", "-ffp-contract=off", "-fPIC", "-std=c11", "-Wall", "-Wextra", "-D_GNU_SOURCE"]
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
    out = os.path.join(build_dir, key, "libsspsd_xoracle.so")
    if os.path.exists(out) or os.access(build_dir if os.path.isdir(build_dir) else _HERE, os.W_OK):
        return out
    return os.path.join(tempfile.gettempdir(), "sspsd_oracle_%d" % os.getuid(), key, "libsspsd_xoracle.so")


def build():
    out = lib_path()
    if not os.path.exists(out):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        cc = os.environ.get("CC", "gcc")
        tmp = out + ".%d.tmp" % os.getpid()
        r = subprocess.run([cc] + CFLAGS + ["-shared", "-o", tmp] + [os.path.join(_HERE, s) for s in _SOURCES[:2]]
                           + ["-lm", "-lpthread"], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("cross-spectrum oracle build failed:\n" + r.stdout + r.stderr)
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
        "orc_xcascade_process": (None, [vp, _fp, _fp, C.c_size_t]),
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


class XCascade:
    """Cross-spectral density of two streams: Psd::process over x and y in lockstep with |c|^2 replaced by
    conj(cx) cy for the cross row, merged like PsdCascade::psd."""

    def __init__(self, n, window=WINDOW_HANN, hbf=HBF_140):
        self.n = n
        self._h = lib().orc_xcascade_new(n, window, hbf)
        if not self._h:
            raise ValueError("unsupported cascade configuration")

    def set_avg(self, limit, count):
        lib().orc_xcascade_set_avg(self._h, limit, count)

    def set_detrend(self, d):
        lib().orc_xcascade_set_detrend(self._h, d)

    def process(self, x, y):
        x, y = _f32(x), _f32(y)
        assert x.size == y.size
        lib().orc_xcascade_process(self._h, _ptr(x), _ptr(y), x.size)

    def num_stages(self):
        return lib().orc_xcascade_num_stages(self._h)

    def csd(self, keep_overlap=False, min_count=1, keep_transition_band=False):
        """-> (pxx, pyy, pxy complex64, breaks)"""
        ns = max(self.num_stages(), 1)
        cap = ns * (self.n // 2 + 1)
        pxx, pyy, pxy = np.zeros(cap, np.float32), np.zeros(cap, np.float32), np.zeros(2 * cap, np.float32)
        b = (Break * ns)()
        nb = C.c_size_t()
        n = lib().orc_xcascade_csd(self._h, int(keep_overlap), min_count, int(keep_transition_band), _ptr(pxx),
                                   _ptr(pyy), _ptr(pxy), b, C.byref(nb))
        return pxx[:n].copy(), pyy[:n].copy(), pxy[:2 * n].view(np.complex64).copy(), [b[i] for i in range(nb.value)]

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:  # (module globals vanish at interpreter exit)
            _lib.orc_xcascade_free(self._h)
            self._h = None
