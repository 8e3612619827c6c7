"""ctypes binding of the CPU oracle (TEST INFRASTRUCTURE ONLY).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg may
import this module.  The product package (stabilizer_stream_b200) never does.

The shared object is built on demand with `make -C oracle` into a directory keyed on the host
CPU's feature flags, because it is compiled with -march=native (mirroring the reference's
`-C target-cpu=native`, .cargo/config.toml:1-2) and the repo snapshot travels between hosts.
When the tree is read-only and holds no build for this host, it is built into a per-user
temporary directory instead.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

WINDOW_RECT, WINDOW_HANN = 0, 1
DETREND_NONE, DETREND_MIDPOINT, DETREND_SPAN, DETREND_MEAN, DETREND_LINEAR = range(5)
HBF_98, HBF_140 = 0, 1
OK, EHEADER, EFORMAT, ESIZE, EBATCHES, ESHORT = 0, 5, 6, 7, 8, 9


def _host_key():
    flags = ""
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("flags"):
                    flags = line
                    break
    except OSError:
        pass
    h = hashlib.sha1(flags.encode())
    for name in ("sspsd_oracle.c", "model_f64.c", "sspsd_oracle.h", "hbf_taps.h", "Makefile"):
        with open(os.path.join(_HERE, name), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:12]


def lib_path():
    key = _host_key()
    out = os.path.join(_HERE, "_build", key, "libsspsd_oracle.so")
    build_dir = os.path.join(_HERE, "_build")
    if os.path.exists(out) or os.access(build_dir if os.path.isdir(build_dir) else _HERE, os.W_OK):
        return out
    return os.path.join(tempfile.gettempdir(), "sspsd_oracle_%d" % os.getuid(), key, "libsspsd_oracle.so")


def build(verbose=False):
    out = lib_path()
    if not os.path.exists(out):
        r = subprocess.run(["make", "-C", _HERE, "OUT=" + out], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("oracle build failed:\n" + r.stdout + r.stderr)
        if verbose:
            print(r.stdout)
    return out


class Break(C.Structure):
    _fields_ = [("start", C.c_uint64), ("include", C.c_uint32), ("count", C.c_uint32),
                ("avg", C.c_uint32), ("_pad", C.c_uint32), ("bins_start", C.c_uint64),
                ("bins_end", C.c_uint64), ("fft_size", C.c_uint64), ("decimation", C.c_uint64),
                ("pending", C.c_uint64), ("processed", C.c_uint64)]

    def as_tuple(self):
        return (self.start, bool(self.include), self.count, self.avg, self.bins_start, self.bins_end,
                self.fft_size, self.decimation, self.pending, self.processed)


class Header(C.Structure):
    _fields_ = [("format", C.c_uint8), ("batches", C.c_uint8), ("seq", C.c_uint32)]


class LossC(C.Structure):
    _fields_ = [("received", C.c_uint64), ("dropped", C.c_uint64), ("seq", C.c_uint32),
                ("has_seq", C.c_uint8)]


_lib = None
_fp = C.POINTER(C.c_float)


def lib():
    global _lib
    if _lib is not None:
        return _lib
    L = C.CDLL(build())
    vp = C.c_void_p
    sig = {
        "orc_hbf8_new": (vp, [C.c_int]),
        "orc_hbf8_free": (None, [vp]),
        "orc_hbf8_block": (None, [vp, _fp, C.c_size_t, _fp]),
        "orc_hbf_response_length": (C.c_int, [C.c_int]),
        "orc_hbf_passband": (C.c_float, []),
        "orc_fft_forward": (None, [_fp, C.c_int]),
        "orc_stage_new": (vp, [C.c_int, C.c_int, C.c_int]),
        "orc_stage_clone": (vp, [vp]),
        "orc_stage_free": (None, [vp]),
        "orc_stage_set_avg": (None, [vp, C.c_uint32]),
        "orc_stage_set_detrend": (None, [vp, C.c_int]),
        "orc_stage_process": (C.c_size_t, [vp, _fp, C.c_size_t, _fp]),
        "orc_stage_spectrum": (_fp, [vp]),
        "orc_stage_count": (C.c_uint32, [vp]),
        "orc_stage_gain": (C.c_float, [vp]),
        "orc_stage_buf": (C.c_size_t, [vp, _fp]),
        "orc_window": (None, [C.c_int, C.c_int, _fp, _fp, _fp, C.POINTER(C.c_size_t)]),
        "orc_detrend_apply": (C.c_int, [C.c_int, _fp, _fp, C.c_int, _fp]),
        "orc_cascade_new": (vp, [C.c_int, C.c_int]),
        "orc_cascade_clone": (vp, [vp]),
        "orc_cascade_free": (None, [vp]),
        "orc_cascade_rbw": (C.c_float, [vp]),
        "orc_cascade_set_avg": (None, [vp, C.c_uint32, C.c_uint32]),
        "orc_cascade_set_detrend": (None, [vp, C.c_int]),
        "orc_cascade_process": (None, [vp, _fp, C.c_size_t]),
        "orc_cascade_num_stages": (C.c_size_t, [vp]),
        "orc_cascade_stage": (vp, [vp, C.c_size_t]),
        "orc_cascade_psd": (C.c_size_t, [vp, C.c_int, C.c_uint32, C.c_int, _fp, C.POINTER(Break),
                                        C.POINTER(C.c_size_t)]),
        "orc_break_frequencies": (C.c_size_t, [C.POINTER(Break), C.c_size_t, _fp]),
        "orc_frame_decode": (C.c_int, [C.c_char_p, C.c_size_t, C.POINTER(Header), C.POINTER(_fp),
                                       C.POINTER(C.c_size_t), C.POINTER(C.c_int)]),
        "orc_loss_update": (None, [C.POINTER(LossC), C.c_uint32, C.c_uint8]),
        "orc_loss_ratio": (C.c_float, [C.POINTER(LossC)]),
        "orc_var_eval": (C.c_float, [C.c_int, C.c_int, C.c_float, C.c_size_t, _fp, _fp, C.c_size_t,
                                     C.c_float]),
        "orc_trace_plot": (C.c_size_t, [C.c_float, C.c_float, C.c_float, C.c_int, _fp, _fp, C.c_size_t, _fp,
                                        C.POINTER(C.c_double)]),
        "orc_philox4x32_10": (None, [C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
        "orc_source_new": (vp, [C.c_int, C.c_int64, C.c_uint64]),
        "orc_source_free": (None, [vp]),
        "orc_source_get": (None, [vp, _fp, C.c_size_t]),
        "orc_dsm_input": (C.c_uint32, [C.c_uint64, C.c_uint32]),
        "f64_cascade_new": (vp, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_uint32, C.c_int]),
        "f64_cascade_free": (None, [vp]),
        "f64_cascade_process": (None, [vp, _fp, C.c_size_t]),
        "f64_cascade_num_stages": (C.c_int, [vp]),
        "f64_cascade_stage": (None, [vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_uint64),
                                     C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _ptr(a):
    return a.ctypes.data_as(_fp)


def fft_forward(c):
    """c: complex64 array -> forward unnormalised DFT (rustfft restatement)."""
    a = np.ascontiguousarray(c, dtype=np.complex64).copy()
    lib().orc_fft_forward(a.view(np.float32).ctypes.data_as(_fp), a.size)
    return a


def window(n, kind):
    w = np.zeros(n, np.float32)
    power, nenbw, ov = C.c_float(), C.c_float(), C.c_size_t()
    lib().orc_window(n, kind, _ptr(w), C.byref(power), C.byref(nenbw), C.byref(ov))
    return w, power.value, nenbw.value, ov.value


def detrend_apply(detrend, x, win):
    x, win = _f32(x), _f32(win)
    c = np.zeros(x.size, np.complex64)
    r = lib().orc_detrend_apply(detrend, _ptr(x), _ptr(win), x.size, c.view(np.float32).ctypes.data_as(_fp))
    if r != 0:
        raise NotImplementedError("Detrend::Linear")
    return c


class Hbf8:
    def __init__(self, preset=HBF_140):
        self._h = lib().orc_hbf8_new(preset)
        assert self._h

    def block(self, x):
        x = _f32(x)
        assert x.size % 8 == 0
        y = np.zeros(x.size // 8, np.float32)
        lib().orc_hbf8_block(self._h, _ptr(x), x.size // 8, _ptr(y))
        return y

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:  # (module globals vanish at interpreter exit)
            _lib.orc_hbf8_free(self._h)
            self._h = None


class Stage:
    """Psd<N> (reference src/psd.rs:123-288)."""

    def __init__(self, n, window=WINDOW_HANN, hbf=HBF_140, _h=None):
        self.n = n
        self._h = _h if _h is not None else lib().orc_stage_new(n, window, hbf)
        if not self._h:
            raise ValueError("unsupported stage configuration")

    def clone(self):
        return Stage(self.n, _h=lib().orc_stage_clone(self._h))

    def set_avg(self, avg):
        lib().orc_stage_set_avg(self._h, avg)

    def set_detrend(self, d):
        lib().orc_stage_set_detrend(self._h, d)

    def process(self, x):
        x = _f32(x)
        y = np.zeros(x.size // 8 + self.n // 8 + 8, np.float32)
        n = lib().orc_stage_process(self._h, _ptr(x), x.size, _ptr(y))
        return y[:n].copy()

    def spectrum(self):
        p = lib().orc_stage_spectrum(self._h)
        return np.ctypeslib.as_array(p, shape=(self.n // 2 + 1,)).copy()

    def count(self):
        return lib().orc_stage_count(self._h)

    def gain(self):
        return lib().orc_stage_gain(self._h)

    def buf(self):
        out = np.zeros(self.n, np.float32)
        n = lib().orc_stage_buf(self._h, _ptr(out))
        return out[:n]

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:  # (module globals vanish at interpreter exit)
            _lib.orc_stage_free(self._h)
            self._h = None


class Cascade:
    """PsdCascade<N> (reference src/psd.rs:399-544)."""

    def __init__(self, n, hbf=HBF_140, _h=None):
        self.n = n
        self._h = _h if _h is not None else lib().orc_cascade_new(n, hbf)
        if not self._h:
            raise ValueError("unsupported cascade configuration")

    def clone(self):
        return Cascade(self.n, _h=lib().orc_cascade_clone(self._h))

    def rbw(self):
        return lib().orc_cascade_rbw(self._h)

    def set_avg(self, limit, count):
        lib().orc_cascade_set_avg(self._h, limit, count)

    def set_detrend(self, d):
        lib().orc_cascade_set_detrend(self._h, d)

    def process(self, x):
        x = _f32(x)
        lib().orc_cascade_process(self._h, _ptr(x), x.size)

    def num_stages(self):
        return lib().orc_cascade_num_stages(self._h)

    def stage_spectrum(self, i):
        s = lib().orc_cascade_stage(self._h, i)
        p = lib().orc_stage_spectrum(s)
        return np.ctypeslib.as_array(p, shape=(self.n // 2 + 1,)).copy()

    def stage_count(self, i):
        return lib().orc_stage_count(lib().orc_cascade_stage(self._h, i))

    def psd(self, keep_overlap=False, min_count=1, keep_transition_band=False):
        ns = max(self.num_stages(), 1)
        p = np.zeros(ns * (self.n // 2 + 1), np.float32)
        b = (Break * ns)()
        nb = C.c_size_t()
        n = lib().orc_cascade_psd(self._h, int(keep_overlap), min_count, int(keep_transition_band),
                                  _ptr(p), b, C.byref(nb))
        return p[:n].copy(), [b[i] for i in range(nb.value)]

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:  # (module globals vanish at interpreter exit)
            _lib.orc_cascade_free(self._h)
            self._h = None


def break_frequencies(breaks):
    nb = len(breaks)
    arr = (Break * max(nb, 1))(*breaks)
    total = sum(int(b.bins_end - b.bins_start) for b in breaks if b.include)
    f = np.zeros(max(total, 1), np.float32)
    n = lib().orc_break_frequencies(arr, nb, _ptr(f))
    return f[:n].copy()


def frame_decode(buf):
    """Frame::from_bytes + traces(): returns (status, header, [traces])."""
    buf = bytes(buf)
    hdr = Header()
    cap = max(8 * 256, 1)
    tr = [np.zeros(cap, np.float32) for _ in range(4)]
    ptrs = (_fp * 4)(*[_ptr(t) for t in tr])
    ns, nt = C.c_size_t(), C.c_int()
    st = lib().orc_frame_decode(buf, len(buf), C.byref(hdr), ptrs, C.byref(ns), C.byref(nt))
    if st != OK:
        return st, None, []
    return st, hdr, [t[:ns.value].copy() for t in tr[:nt.value]]


class Loss:
    """Loss (reference src/loss.rs:4-38)."""

    def __init__(self):
        self.c = LossC()

    def update(self, seq, batches):
        lib().orc_loss_update(C.byref(self.c), seq, batches)

    @property
    def received(self):
        return self.c.received

    @property
    def dropped(self):
        return self.c.dropped

    @property
    def seq(self):
        return self.c.seq if self.c.has_seq else None

    def ratio(self):
        return lib().orc_loss_ratio(C.byref(self.c))


def var_eval(phase_psd, frequencies, tau, x_exp=-2, sinx_exp=4, clip=3.4028234663852886e38, dc_cut=2):
    p, f = _f32(phase_psd), _f32(frequencies)
    return lib().orc_var_eval(x_exp, sinx_exp, clip, dc_cut, _ptr(p), _ptr(f), min(p.size, f.size), tau)


def trace_plot(psd, frequencies, fs=1.0, integral_start=1e-6, integral_end=0.5, integrate=False):
    """Trace::plot (bin/psd.rs:125-157) -> (sqrt of the band integral, plot points [n, 2] float64)"""
    p, f = _f32(psd), _f32(frequencies)
    n = min(p.size, f.size)
    xy = np.zeros((max(n, 1), 2), np.float64)
    integ = C.c_float()
    m = lib().orc_trace_plot(fs, integral_start, integral_end, int(integrate), _ptr(p), _ptr(f), n, C.byref(integ),
                             xy.ctypes.data_as(C.POINTER(C.c_double)))
    return integ.value, xy[:m].copy()


SOURCE_NOISE, SOURCE_DSM = 0, 1


def philox4x32_10(ctr, key):
    c = (C.c_uint32 * 4)(*ctr)
    k = (C.c_uint32 * 2)(*key)
    o = (C.c_uint32 * 4)()
    lib().orc_philox4x32_10(c, k, o)
    return tuple(o)


class Source:
    """Data::Noise / Data::Dsm of source.rs:66-73, 104-134 (sequential f32 restatement)."""

    def __init__(self, kind, param, seed=0x7654321):
        self.h = lib().orc_source_new(kind, param, seed)
        if not self.h:
            raise ValueError("unsupported source")

    def __del__(self):
        if getattr(self, "h", None) and _lib is not None:  # (module globals vanish at interpreter exit)
            _lib.orc_source_free(self.h)
            self.h = None

    def get(self, n):
        out = np.empty(n, dtype=np.float32)
        lib().orc_source_get(self.h, _ptr(out), n)
        return out


def dsm_input(i, ftw):
    return lib().orc_dsm_input(i, ftw)


class CascadeF64:
    """Streaming float64 truth model (oracle/model_f64.c): same semantics as Cascade, f64 arithmetic,
    independent code structure.  max_stages=1 models a single Psd<N> stage."""

    def __init__(self, n, hbf=HBF_140, window=WINDOW_HANN, detrend=DETREND_NONE, avg_limit=0xFFFFFFFF,
                 avg_count=0xFFFFFFFF, max_stages=0):
        self.n = n
        self._h = lib().f64_cascade_new(n, window, hbf, detrend, avg_limit, avg_count, max_stages)
        if not self._h:
            raise ValueError("unsupported configuration")

    def process(self, x):
        x = _f32(x)
        lib().f64_cascade_process(self._h, _ptr(x), x.size)

    def num_stages(self):
        return lib().f64_cascade_num_stages(self._h)

    def stage(self, i):
        """(spectrum float64[N/2+1], effective count, segments, samples received)"""
        sp = np.zeros(self.n // 2 + 1, np.float64)
        cnt, craw, L = C.c_uint64(), C.c_uint64(), C.c_uint64()
        lib().f64_cascade_stage(self._h, i, sp.ctypes.data_as(C.POINTER(C.c_double)), C.byref(cnt), C.byref(craw),
                                C.byref(L))
        return sp, cnt.value, craw.value, L.value

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.f64_cascade_free(self._h)
            self._h = None
