"""ctypes binding of the CPU restatement of the plants, oracle/sspsd_poracle.c (TEST INFRASTRUCTURE ONLY; DESIGN.md
section 3d).

sspsd_poracle.c is linked with sspsd_oracle.c (whose orc_source_* give the noise inputs) into its own shared object,
built and placed as oracle/zbinding.py builds the two-sided restatement.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from .xbinding import CFLAGS

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = ("sspsd_poracle.c", "sspsd_oracle.c", "sspsd_oracle.h", "hbf_taps.h")
_lib = None
NOISE, TONE = 0, 1


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
    out = os.path.join(build_dir, key, "libsspsd_poracle.so")
    if os.path.exists(out) or os.access(build_dir if os.path.isdir(build_dir) else _HERE, os.W_OK):
        return out
    return os.path.join(tempfile.gettempdir(), "sspsd_oracle_%d" % os.getuid(), key, "libsspsd_poracle.so")


def build():
    out = lib_path()
    if not os.path.exists(out):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        cc = os.environ.get("CC", "gcc")
        tmp = out + ".%d.tmp" % os.getpid()
        r = subprocess.run([cc] + CFLAGS + ["-shared", "-o", tmp] + [os.path.join(_HERE, s) for s in _SOURCES[:2]]
                           + ["-lm", "-lpthread"], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("plant oracle build failed:\n" + r.stdout + r.stderr)
        os.replace(tmp, out)
    return out


def lib():
    global _lib
    if _lib is not None:
        return _lib
    L = C.CDLL(build())
    fp = C.POINTER(C.c_float)
    L.orc_plant_cos.restype = C.c_float
    L.orc_plant_cos.argtypes = [C.c_uint32]
    L.orc_plant_generate.restype = C.c_int
    L.orc_plant_generate.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, fp, C.POINTER(C.c_int32),
                                     C.POINTER(C.c_int64), C.POINTER(C.c_uint64), fp, C.c_uint64, C.c_size_t, fp]
    _lib = L
    return L


def plant_cos(phi):
    return lib().orc_plant_cos(int(phi) & 0xFFFFFFFF)


def plant(taps, inputs, n, pos=0):
    """positions [pos, pos + n) of every output, [K, n] float32.  inputs: objects with kind, param, seed, amplitude
    (stabilizer_stream_b200.PlantInput) or (kind, param, seed, amplitude) tuples.  The inputs are generated from
    position 0, so pos + n is what the run costs."""
    taps = np.ascontiguousarray(np.asarray(taps, np.float32))
    k, m, nt = taps.shape
    ins = [(u.kind, u.param, u.seed, u.amplitude) if hasattr(u, "kind") else tuple(u) for u in inputs]
    if len(ins) != m:
        raise ValueError("taps have %d inputs, %d given" % (m, len(ins)))
    kinds = (C.c_int32 * m)(*[int(u[0]) for u in ins])
    params = (C.c_int64 * m)(*[int(u[1]) for u in ins])
    seeds = (C.c_uint64 * m)(*[int(u[2]) & (2 ** 64 - 1) for u in ins])
    amps = (C.c_float * m)(*[float(u[3]) for u in ins])
    out = np.zeros((k, n), np.float32)
    fp = C.POINTER(C.c_float)
    rc = lib().orc_plant_generate(k, m, nt, taps.ctypes.data_as(fp), kinds, params, seeds, amps, pos, n,
                                  out.ctypes.data_as(fp))
    if rc == -1:
        raise ValueError("input kind or exponent the plant refuses")
    if rc:
        raise MemoryError("orc_plant_generate")
    return out
