"""Host-side mirror of the reference's PSD API (quartiq/stabilizer-stream src/psd.rs, src/de,
src/loss.rs, src/var.rs) on top of the C ABI of libsspsd.so.  Same names, same argument meaning,
same error behaviour; all arithmetic happens in the CUDA library (there is no CPU path here).

    PsdCascade(n).process(x); p, breaks = cascade.psd(MergeOpts()); f = Break.frequencies(breaks)

`x` may be a numpy float32 array (host memory) or a CUDA torch tensor (device memory, consumed in
stream order on the cascade's stream).
"""
import ctypes as C
import enum
from dataclasses import dataclass

import numpy as np

from . import _lib as L

DEPTH = 3  # src/psd.rs:117
HBF_PASSBAND = 0.4  # idsp::hbf::HBF_PASSBAND, src/psd.rs:601


class Detrend(enum.IntEnum):
    """enum Detrend, src/psd.rs:59-72"""
    NONE = 0
    MIDPOINT = 1
    SPAN = 2
    MEAN = 3
    LINEAR = 4


class Window(enum.IntEnum):
    """Window::rectangular / Window::hann, src/psd.rs:24-55"""
    RECTANGULAR = 0
    HANN = 1


class Hbf(enum.IntEnum):
    TAPS_98 = 0
    TAPS_140 = 1


@dataclass
class AvgOpts:
    """src/psd.rs:360-376"""
    limit: int = 0xFFFFFFFF
    count: int = 0xFFFFFFFF


@dataclass
class MergeOpts:
    """src/psd.rs:339-358"""
    keep_overlap: bool = False
    min_count: int = 1
    keep_transition_band: bool = False


@dataclass
class Break:
    """src/psd.rs:290-337"""
    start: int
    include: bool
    count: int
    avg: int
    bins: range
    fft_size: int
    decimation: int
    pending: int
    processed: int

    def effective_fft_size(self):
        return self.fft_size * self.decimation

    def rbw(self):
        return np.float32(1.0) / np.float32(self.effective_fft_size())

    @staticmethod
    def frequencies(breaks):
        """Break::frequencies, src/psd.rs:315-327 (computed by the library)."""
        arr = (L.BreakC * max(len(breaks), 1))()
        for i, b in enumerate(breaks):
            arr[i] = b._c()
        n = C.c_size_t(0)
        st = L.lib().sspsd_break_frequencies(arr, len(breaks), None, C.byref(n))
        if st not in (L.OK, L.ESHORT):
            L.check(st)
        f = np.zeros(max(n.value, 1), np.float32)
        n = C.c_size_t(f.size)
        L.check(L.lib().sspsd_break_frequencies(arr, len(breaks), f.ctypes.data, C.byref(n)))
        return f[:n.value]

    def _c(self):
        return L.BreakC(self.start, int(self.include), self.count, self.avg, 0, self.bins.start, self.bins.stop,
                        self.fft_size, self.decimation, self.pending, self.processed)

    @staticmethod
    def _from_c(b):
        return Break(b.start, bool(b.include), b.count, b.avg, range(b.bins_start, b.bins_end), b.fft_size,
                     b.decimation, b.pending, b.processed)


def _as_buffer(x):
    """-> (pointer, n, mem, keepalive)"""
    if isinstance(x, np.ndarray) or not hasattr(x, "data_ptr"):
        a = np.ascontiguousarray(x, dtype=np.float32)
        return a.ctypes.data, a.size, L.MEM_HOST, a
    import torch
    if x.dtype != torch.float32:
        raise TypeError("expected float32 samples")
    t = x.contiguous()
    mem = L.MEM_DEVICE if t.is_cuda else L.MEM_HOST
    return t.data_ptr(), t.numel(), mem, t


def _default_stream(device):
    """With torch in the process, order the handle's work on torch's current stream of that device (this
    initialises torch's CUDA context if it is not yet), so that device tensors handed to process() follow
    torch's usual stream-ordered lifetime rules.  Without torch: a private stream."""
    import sys
    torch = sys.modules.get("torch")
    if torch is None or not torch.cuda.is_available():
        return None
    h = torch.cuda.current_stream(device).cuda_stream
    # torch's default stream is the legacy NULL stream; a NULL cfg.stream means "private stream" in the
    # C ABI, so name the legacy stream explicitly (cudaStreamLegacy == (cudaStream_t)1)
    return h if h else 1


class _StreamOrdered:
    """Mixin of the handle classes that read CUDA tensors in place: SSPSD_MEM_DEVICE input is consumed
    asynchronously on the HANDLE's stream (include/sspsd.h), which need not be the stream torch is on when
    process() is called (a handle made before `with torch.cuda.stream(s)`, or one with a private stream).
    Before the call the handle's stream waits for torch's current stream (the producer of x); after it torch's
    current stream waits for the handle's stream (_release_device_input), so the caching allocator -- which reuses
    a freed block in the order of the stream it was allocated on -- cannot recycle a temporary (e.g. the
    .contiguous() copy) while the kernels still read it.  (Not Tensor.record_stream: the allocator would later
    record an event on the handle's stream, which may have been destroyed with the handle by then.)"""

    _hs = None

    def _stream_ptr(self):  # overridden where the C ABI exposes the handle's stream
        return None

    def _handle_stream(self, t):
        import torch
        if t.device.index != self.device:
            raise ValueError("tensor lives on cuda:%d, the handle on cuda:%d" % (t.device.index, self.device))
        if self._hs is None:
            ptr = self._stream_ptr()
            if ptr is None:
                return None, None
            self._hs = (torch.cuda.default_stream(t.device) if ptr in (0, 1)
                        else torch.cuda.ExternalStream(ptr, device=t.device))
        cur = torch.cuda.current_stream(t.device)
        if (cur.cuda_stream or 1) == (self._hs.cuda_stream or 1):
            return None, None
        return self._hs, cur

    def _order_device_input(self, t):
        hs, cur = self._handle_stream(t)
        if hs is not None:
            hs.wait_stream(cur)

    def _release_device_input(self, t):
        """after an ASYNCHRONOUS call that read (or wrote) t on the handle's stream"""
        hs, cur = self._handle_stream(t)
        if hs is not None:
            cur.wait_stream(hs)


def _config(n, window, hbf, device, stream, max_batch, host_stage, deep_defer=0, deterministic=False):
    if stream is None:
        stream = _default_stream(device)
    cfg = L.Config()
    L.check(L.lib().sspsd_config_default(n, C.byref(cfg)))
    cfg.window = int(window)
    cfg.hbf = int(hbf)
    cfg.device = int(device)
    cfg.stream = stream
    cfg.max_batch = max_batch
    cfg.host_stage = host_stage
    cfg.deep_defer = deep_defer
    cfg.flags = L.FLAG_DETERMINISTIC if deterministic else 0
    return cfg


class PsdCascade(_StreamOrdered):
    """PsdCascade<N>, src/psd.rs:399-544.  `PsdCascade(n)` is `PsdCascade::<N>::default()`."""

    def __init__(self, n=512, device=0, hbf=Hbf.TAPS_140, stream=None, max_batch=0, host_stage=0, deep_defer=0,
                 deterministic=False, _handle=None):
        self.n = n
        self.device = int(device)
        if _handle is not None:
            self._h = _handle
            return
        cfg = _config(n, Window.HANN, hbf, device, stream, max_batch, host_stage, deep_defer, deterministic)
        h = C.c_void_p()
        L.check(L.lib().sspsd_cascade_create(C.byref(cfg), C.byref(h)))
        self._h = h

    def clone(self):
        h = C.c_void_p()
        L.check(L.lib().sspsd_cascade_clone(self._h, C.byref(h)))
        return PsdCascade(self.n, device=self.device, _handle=h)

    def _stream_ptr(self):
        s = C.c_void_p()
        L.check(L.lib().sspsd_cascade_stream(self._h, C.byref(s)))
        return s.value or 0

    def reset(self):
        L.check(L.lib().sspsd_cascade_reset(self._h))

    def rbw(self):
        r = C.c_float()
        L.check(L.lib().sspsd_cascade_rbw(self._h, C.byref(r)))
        return r.value

    def set_avg(self, avg: AvgOpts):
        L.check(L.lib().sspsd_cascade_set_avg(self._h, L.AvgOptsC(avg.limit, avg.count)))

    def set_detrend(self, d: Detrend):
        L.check(L.lib().sspsd_cascade_set_detrend(self._h, int(d)))

    def process(self, x):
        ptr, n, mem, keep = _as_buffer(x)
        if mem == L.MEM_DEVICE:
            self._order_device_input(keep)
        L.check(L.lib().sspsd_cascade_process_f32(self._h, ptr, n, mem))
        if mem == L.MEM_DEVICE:
            self._release_device_input(keep)
        del keep

    def process_raw(self, ptr, n, mem):
        L.check(L.lib().sspsd_cascade_process_f32(self._h, ptr, n, mem))

    def process_source(self, source, n):
        """Feed the next n samples of a device-resident synthetic Source (no host memory involved);
        the loop of bin/stream_test.rs:52-58 with `--noise` / `--dsm`."""
        L.check(L.lib().sspsd_cascade_process_source(self._h, source._h, n))

    def flush(self):
        L.check(L.lib().sspsd_cascade_flush(self._h))

    def sync(self):
        L.check(L.lib().sspsd_cascade_sync(self._h))

    def num_stages(self):
        n = C.c_uint32()
        L.check(L.lib().sspsd_cascade_num_stages(self._h, C.byref(n)))
        return n.value

    def psd(self, opts: MergeOpts = None):
        opts = opts or MergeOpts()
        o = L.MergeOptsC(int(opts.keep_overlap), opts.min_count, int(opts.keep_transition_band))
        p = np.zeros(L.MAX_STAGES * (self.n // 2 + 1), np.float32)
        b = (L.BreakC * L.MAX_STAGES)()
        pl, bl = C.c_size_t(p.size), C.c_size_t(L.MAX_STAGES)
        L.check(L.lib().sspsd_cascade_psd(self._h, C.byref(o), p.ctypes.data, C.byref(pl), b, C.byref(bl)))
        return p[:pl.value].copy(), [Break._from_c(b[i]) for i in range(bl.value)]

    # ---- time-chunked processing of one stream by several handles (include/sspsd.h) ----
    def seek(self, pos):
        L.check(L.lib().sspsd_cascade_seek(self._h, pos))

    def set_window(self, own_lo, own_hi, n_local):
        L.check(L.lib().sspsd_cascade_set_window(self._h, own_lo, own_hi if own_hi is not None else 2 ** 64 - 1, n_local))

    def take_tail(self, j_lo, j_hi):
        """-> (first stream index, numpy array) of the exported stage-n_local input stream in [j_lo, j_hi)"""
        n = C.c_size_t(0)
        first = C.c_uint64(0)
        st = L.lib().sspsd_cascade_take_tail(self._h, j_lo, j_hi, None, C.byref(n), C.byref(first), L.MEM_HOST)
        if st not in (L.OK, L.ESHORT):
            L.check(st)
        out = np.zeros(max(n.value, 1), np.float32)
        n = C.c_size_t(out.size)
        L.check(L.lib().sspsd_cascade_take_tail(self._h, j_lo, j_hi, out.ctypes.data, C.byref(n), C.byref(first),
                                                L.MEM_HOST))
        return first.value, out[:n.value]

    def take_tail_device(self, j_lo, j_hi, out):
        """like take_tail, but into the CUDA float32 tensor `out` (no host round trip); -> (first, length)"""
        n = C.c_size_t(out.numel())
        first = C.c_uint64(0)
        L.check(L.lib().sspsd_cascade_take_tail(self._h, j_lo, j_hi, out.data_ptr(), C.byref(n), C.byref(first),
                                                L.MEM_DEVICE))
        return first.value, n.value

    def process_stage(self, stage, x):
        ptr, n, mem, keep = _as_buffer(x)
        if mem == L.MEM_DEVICE:
            # copied into the stage's own buffer on a library stream: make the producer's work visible first
            import torch
            torch.cuda.current_stream(keep.device).synchronize()
        L.check(L.lib().sspsd_cascade_process_stage(self._h, stage, ptr, n, mem))
        del keep

    def set_stream_state(self, stage, samples, segments):
        L.check(L.lib().sspsd_cascade_set_stream_state(self._h, stage, samples, segments))

    def profile_enable(self, on=True):
        L.check(L.lib().sspsd_cascade_profile_enable(self._h, int(on)))

    def profile_read(self):
        """-> dict(class -> (ms, launches, input samples)), total kernel launches since the last read"""
        out = L.ProfileC()
        L.check(L.lib().sspsd_cascade_profile_read(self._h, C.byref(out)))
        names = ("psd_stage0", "psd_deep", "decim_stage0", "decim_deep", "other")
        return {k: (out.ms[i], out.launches[i], out.units[i]) for i, k in enumerate(names)}, out.launches_total

    def partials(self):
        out = L.PartialsC()
        L.check(L.lib().sspsd_cascade_partials(self._h, C.byref(out)))
        return out

    def set_counts(self, counts):
        arr = (C.c_uint64 * len(counts))(*counts)
        L.check(L.lib().sspsd_cascade_set_counts(self._h, arr, len(counts)))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h and L is not None and getattr(L, "_lib", None) is not None:
            L._lib.sspsd_cascade_destroy(h)
            self._h = None


class CsdCascade(_StreamOrdered):
    """Cascaded cross-spectral density of two streams x and y (include/sspsd.h, sspsd_csd_*).  Both go through the
    same cascade as PsdCascade; every stage accumulates |X|^2, |Y|^2 and conj(X) Y (scipy.signal.csd's convention),
    so for y = h * x, pxy / pxx is the transfer function H and pxx is what a PsdCascade fed x alone returns.
    n = 64 .. 4096."""

    def __init__(self, n=512, window=Window.HANN, device=0, hbf=Hbf.TAPS_140, stream=None, max_batch=0, host_stage=0,
                 deep_defer=0, deterministic=False, _handle=None):
        self.n = n
        self.device = int(device)
        if _handle is not None:
            self._h = _handle
            return
        cfg = _config(n, window, hbf, device, stream, max_batch, host_stage, deep_defer, deterministic)
        h = C.c_void_p()
        L.check(L.lib().sspsd_csd_create(C.byref(cfg), C.byref(h)))
        self._h = h

    def clone(self):
        h = C.c_void_p()
        L.check(L.lib().sspsd_csd_clone(self._h, C.byref(h)))
        return CsdCascade(self.n, device=self.device, _handle=h)

    def _stream_ptr(self):
        s = C.c_void_p()
        L.check(L.lib().sspsd_csd_stream(self._h, C.byref(s)))
        return s.value or 0

    def reset(self):
        L.check(L.lib().sspsd_csd_reset(self._h))

    def rbw(self):
        r = C.c_float()
        L.check(L.lib().sspsd_csd_rbw(self._h, C.byref(r)))
        return r.value

    def set_avg(self, avg: AvgOpts):
        L.check(L.lib().sspsd_csd_set_avg(self._h, L.AvgOptsC(avg.limit, avg.count)))

    def set_detrend(self, d: Detrend):
        L.check(L.lib().sspsd_csd_set_detrend(self._h, int(d)))

    def process(self, x, y):
        """the next samples of both streams: equal-length float32 numpy arrays, or CUDA tensors (both)"""
        px, n, mem, kx = _as_buffer(x)
        py, ny, memy, ky = _as_buffer(y)
        if n != ny:
            raise ValueError("x and y must have the same length (%d != %d)" % (n, ny))
        if mem != memy:
            raise ValueError("x and y must both be host arrays or both be CUDA tensors")
        if mem == L.MEM_DEVICE:
            self._order_device_input(kx)
            self._order_device_input(ky)
        L.check(L.lib().sspsd_csd_process_f32(self._h, px, py, n, mem))
        if mem == L.MEM_DEVICE:
            self._release_device_input(kx)
        del kx, ky

    def flush(self):
        L.check(L.lib().sspsd_csd_flush(self._h))

    def sync(self):
        L.check(L.lib().sspsd_csd_sync(self._h))

    def num_stages(self):
        n = C.c_uint32()
        L.check(L.lib().sspsd_csd_num_stages(self._h, C.byref(n)))
        return n.value

    def csd(self, opts: MergeOpts = None):
        """-> (pxx, pyy, pxy (complex64), breaks), merged like PsdCascade.psd"""
        opts = opts or MergeOpts()
        o = L.MergeOptsC(int(opts.keep_overlap), opts.min_count, int(opts.keep_transition_band))
        cap = L.MAX_STAGES * (self.n // 2 + 1)
        pxx, pyy = np.zeros(cap, np.float32), np.zeros(cap, np.float32)
        pxy = np.zeros(2 * cap, np.float32)
        b = (L.BreakC * L.MAX_STAGES)()
        pl, bl = C.c_size_t(cap), C.c_size_t(L.MAX_STAGES)
        L.check(L.lib().sspsd_csd_read(self._h, C.byref(o), pxx.ctypes.data, pyy.ctypes.data, pxy.ctypes.data,
                                       C.byref(pl), b, C.byref(bl)))
        n = pl.value
        return (pxx[:n].copy(), pyy[:n].copy(), pxy[:2 * n].view(np.complex64).copy(),
                [Break._from_c(b[i]) for i in range(bl.value)])

    @staticmethod
    def coherence(pxx, pyy, pxy):
        """magnitude-squared coherence |pxy|^2 / (pxx pyy) per bin (0 where a power is 0)"""
        pxx, pyy = np.asarray(pxx, np.float64), np.asarray(pyy, np.float64)
        den = pxx * pyy
        return np.divide(np.abs(np.asarray(pxy, np.complex128)) ** 2, den, out=np.zeros_like(den), where=den > 0)

    @staticmethod
    def transfer(pxx, pxy):
        """transfer function estimate H = pxy / pxx per bin (0 where pxx is 0)"""
        pxx = np.asarray(pxx, np.float64)
        return np.divide(np.asarray(pxy, np.complex128), pxx, out=np.zeros(pxx.shape, np.complex128), where=pxx > 0)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h and L is not None and getattr(L, "_lib", None) is not None:
            L._lib.sspsd_csd_destroy(h)
            self._h = None


class CsmCascade(_StreamOrdered):
    """Cascaded cross-spectral matrix of K = 2, 3 or 4 streams (include/sspsd.h, sspsd_csm_*).  All go through one
    cascade and every stage accumulates S_ij = sum w conj(X_i) X_j, CsdCascade's convention: S[0, 1] is pxy of
    CsdCascade(x0, x1) and S[i, i] what a PsdCascade fed x_i alone returns.  Every transform is shared by all
    pairs: the matrix of K streams costs K FFTs and K decimations per segment.  n = 64 .. 4096."""

    def __init__(self, n=512, channels=4, window=Window.HANN, device=0, hbf=Hbf.TAPS_140, stream=None, max_batch=0,
                 host_stage=0, deep_defer=0, deterministic=False, _handle=None):
        self.n = n
        self.channels = int(channels)
        self.device = int(device)
        if _handle is not None:
            self._h = _handle
            return
        cfg = _config(n, window, hbf, device, stream, max_batch, host_stage, deep_defer, deterministic)
        h = C.c_void_p()
        L.check(L.lib().sspsd_csm_create(C.byref(cfg), self.channels, C.byref(h)))
        self._h = h

    def clone(self):
        h = C.c_void_p()
        L.check(L.lib().sspsd_csm_clone(self._h, C.byref(h)))
        return CsmCascade(self.n, self.channels, device=self.device, _handle=h)

    def _stream_ptr(self):
        s = C.c_void_p()
        L.check(L.lib().sspsd_csm_stream(self._h, C.byref(s)))
        return s.value or 0

    def reset(self):
        L.check(L.lib().sspsd_csm_reset(self._h))

    def rbw(self):
        r = C.c_float()
        L.check(L.lib().sspsd_csm_rbw(self._h, C.byref(r)))
        return r.value

    def set_avg(self, avg: AvgOpts):
        L.check(L.lib().sspsd_csm_set_avg(self._h, L.AvgOptsC(avg.limit, avg.count)))

    def set_detrend(self, d: Detrend):
        L.check(L.lib().sspsd_csm_set_detrend(self._h, int(d)))

    def process(self, xs):
        """the next samples of every stream: K equal-length float32 numpy arrays or CUDA tensors, or one (K, n)
        array or tensor"""
        if len(xs) != self.channels:
            raise ValueError("expected %d channels, got %d" % (self.channels, len(xs)))
        bufs = [_as_buffer(x) for x in xs]
        n, mem = bufs[0][1], bufs[0][2]
        if any(b[1] != n for b in bufs):
            raise ValueError("all channels must have the same length (%s)" % [b[1] for b in bufs])
        if any(b[2] != mem for b in bufs):
            raise ValueError("channels must all be host arrays or all be CUDA tensors")
        ptrs = (C.c_void_p * self.channels)(*[b[0] for b in bufs])
        if mem == L.MEM_DEVICE:
            for b in bufs:
                self._order_device_input(b[3])
        L.check(L.lib().sspsd_csm_process_f32(self._h, ptrs, n, mem))
        if mem == L.MEM_DEVICE:
            self._release_device_input(bufs[0][3])
        del bufs

    def flush(self):
        L.check(L.lib().sspsd_csm_flush(self._h))

    def sync(self):
        L.check(L.lib().sspsd_csm_sync(self._h))

    def num_stages(self):
        n = C.c_uint32()
        L.check(L.lib().sspsd_csm_num_stages(self._h, C.byref(n)))
        return n.value

    def csm(self, opts: MergeOpts = None):
        """-> (S complex64 [K, K, bins], breaks), every entry merged like PsdCascade.psd"""
        opts = opts or MergeOpts()
        o = L.MergeOptsC(int(opts.keep_overlap), opts.min_count, int(opts.keep_transition_band))
        k = self.channels
        cap = L.MAX_STAGES * (self.n // 2 + 1)
        s = np.zeros(2 * k * k * cap, np.float32)
        b = (L.BreakC * L.MAX_STAGES)()
        pl, bl = C.c_size_t(cap), C.c_size_t(L.MAX_STAGES)
        L.check(L.lib().sspsd_csm_read(self._h, C.byref(o), s.ctypes.data, C.byref(pl), b, C.byref(bl)))
        n = pl.value
        m = s[:2 * k * k * n].view(np.complex64).reshape(k, k, n).copy()
        return m, [Break._from_c(b[i]) for i in range(bl.value)]

    @staticmethod
    def coherence(S):
        """magnitude-squared coherence |S_ij|^2 / (S_ii S_jj) per bin, [K, K, bins] (0 where a power is 0)"""
        S = np.asarray(S, np.complex128)
        d = np.real(np.einsum("iib->ib", S))
        den = d[:, None, :] * d[None, :, :]
        return np.divide(np.abs(S) ** 2, den, out=np.zeros(den.shape), where=den > 0)

    @staticmethod
    def transfer(S, inputs, outputs):
        """MIMO transfer function estimate H [len(outputs), len(inputs), bins] with y_o = sum_i H[o, i] u_i:
        H = (S_uu^-1 S_uy)^T per bin, S_uu the inputs' block and S_uy the inputs-by-outputs block of S.  0 where
        S_uu is singular (det 0, or below 1e-12 of the product of its diagonal).  With one input this is
        CsdCascade.transfer."""
        S = np.asarray(S, np.complex128)
        inputs, outputs = list(inputs), list(outputs)
        suu = np.moveaxis(S[np.ix_(inputs, inputs)], -1, 0)    # [bins, ni, ni]
        suy = np.moveaxis(S[np.ix_(inputs, outputs)], -1, 0)   # [bins, ni, no]
        diag = np.prod(np.real(np.einsum("bii->bi", suu)), axis=1)
        det = np.linalg.det(suu)
        ok = (diag > 0) & (np.abs(det) > 1e-12 * np.where(diag > 0, diag, 0))
        h = np.zeros((S.shape[-1], len(inputs), len(outputs)), np.complex128)
        if np.any(ok):
            h[ok] = np.linalg.solve(suu[ok], suy[ok])
        return np.transpose(h, (2, 1, 0))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h and L is not None and getattr(L, "_lib", None) is not None:
            L._lib.sspsd_csm_destroy(h)
            self._h = None


class ZoomCascade(_StreamOrdered):
    """Two-sided cascaded spectrum of a complex stream z (include/sspsd.h, sspsd_zoom_*), in one of two modes:
    ZoomCascade.iq(n): z = i + i q of two real streams (a lock-in's BI / BQ); ZoomCascade.heterodyne(n, ftw):
    z = x exp(-2 pi i phi_n / 2^32), phi_n = (n ftw) mod 2^32, one real stream mixed down by the carrier
    f0 = ftw / 2^32 (units of the sample rate) on the device, so the cascade's fine low-frequency resolution lands
    around f0.  spectrum() returns both sides, p_pos at f0 + f and p_neg at f0 - f, with PsdCascade.psd's breaks and
    the two-sided density's scale (a real x fed as (x, 0) reads back psd(x) / 2 per side).  n = 64 .. 4096."""

    def __init__(self, n=512, mode=L.ZOOM_IQ, ftw=0, window=Window.HANN, device=0, hbf=Hbf.TAPS_140, stream=None,
                 max_batch=0, host_stage=0, deep_defer=0, deterministic=False, _handle=None):
        self.n = n
        self.mode = int(mode)
        self.ftw = int(ftw)
        self.device = int(device)
        if _handle is not None:
            self._h = _handle
            return
        cfg = _config(n, window, hbf, device, stream, max_batch, host_stage, deep_defer, deterministic)
        h = C.c_void_p()
        L.check(L.lib().sspsd_zoom_create(C.byref(cfg), self.mode, self.ftw, C.byref(h)))
        self._h = h

    @classmethod
    def iq(cls, n=512, **kw):
        """I/Q mode: process(i, q)"""
        return cls(n, L.ZOOM_IQ, 0, **kw)

    @classmethod
    def heterodyne(cls, n, ftw, **kw):
        """heterodyne mode around the carrier ftw / 2^32 (ftw: a 32-bit frequency tuning word, see ftw_of): process(x)"""
        if not 0 <= int(ftw) < 2 ** 32:
            raise ValueError("ftw must be a 32-bit frequency tuning word, got %d" % ftw)
        return cls(n, L.ZOOM_HETERODYNE, ftw, **kw)

    @staticmethod
    def ftw_of(f0):
        """the tuning word of the carrier f0 (units of the sample rate, any sign): round(f0 2^32) mod 2^32"""
        return int(round(float(f0) * 2.0 ** 32)) % 2 ** 32

    def clone(self):
        h = C.c_void_p()
        L.check(L.lib().sspsd_zoom_clone(self._h, C.byref(h)))
        return ZoomCascade(self.n, self.mode, self.ftw, device=self.device, _handle=h)

    def _stream_ptr(self):
        s = C.c_void_p()
        L.check(L.lib().sspsd_zoom_stream(self._h, C.byref(s)))
        return s.value or 0

    def reset(self):
        L.check(L.lib().sspsd_zoom_reset(self._h))

    def rbw(self):
        r = C.c_float()
        L.check(L.lib().sspsd_zoom_rbw(self._h, C.byref(r)))
        return r.value

    def carrier(self):
        """-> (mode, ftw) of the handle"""
        m, f = C.c_int32(), C.c_uint32()
        L.check(L.lib().sspsd_zoom_carrier(self._h, C.byref(m), C.byref(f)))
        return m.value, f.value

    def set_avg(self, avg: AvgOpts):
        L.check(L.lib().sspsd_zoom_set_avg(self._h, L.AvgOptsC(avg.limit, avg.count)))

    def set_detrend(self, d: Detrend):
        L.check(L.lib().sspsd_zoom_set_detrend(self._h, int(d)))

    def process(self, x, q=None):
        """the next samples: process(x) in heterodyne mode, process(i, q) in I/Q mode; float32 numpy arrays or CUDA
        tensors (both of a pair alike)"""
        if (q is None) != (self.mode == L.ZOOM_HETERODYNE):
            raise ValueError("heterodyne mode takes process(x), I/Q mode process(i, q)")
        px, n, mem, kx = _as_buffer(x)
        if q is None:
            if mem == L.MEM_DEVICE:
                self._order_device_input(kx)
            L.check(L.lib().sspsd_zoom_process_f32(self._h, px, n, mem))
        else:
            pq, nq, memq, kq = _as_buffer(q)
            if n != nq:
                raise ValueError("i and q must have the same length (%d != %d)" % (n, nq))
            if mem != memq:
                raise ValueError("i and q must both be host arrays or both be CUDA tensors")
            if mem == L.MEM_DEVICE:
                self._order_device_input(kx)
                self._order_device_input(kq)
            L.check(L.lib().sspsd_zoom_process_iq_f32(self._h, px, pq, n, mem))
        if mem == L.MEM_DEVICE:
            self._release_device_input(kx)

    def flush(self):
        L.check(L.lib().sspsd_zoom_flush(self._h))

    def sync(self):
        L.check(L.lib().sspsd_zoom_sync(self._h))

    def num_stages(self):
        n = C.c_uint32()
        L.check(L.lib().sspsd_zoom_num_stages(self._h, C.byref(n)))
        return n.value

    def spectrum(self, opts: MergeOpts = None):
        """-> (p_pos, p_neg, breaks): the densities at f0 + f and f0 - f, f = Break.frequencies(breaks) >= 0"""
        opts = opts or MergeOpts()
        o = L.MergeOptsC(int(opts.keep_overlap), opts.min_count, int(opts.keep_transition_band))
        cap = L.MAX_STAGES * (self.n // 2 + 1)
        pp, pn = np.zeros(cap, np.float32), np.zeros(cap, np.float32)
        b = (L.BreakC * L.MAX_STAGES)()
        pl, bl = C.c_size_t(cap), C.c_size_t(L.MAX_STAGES)
        L.check(L.lib().sspsd_zoom_read(self._h, C.byref(o), pp.ctypes.data, pn.ctypes.data, C.byref(pl), b,
                                        C.byref(bl)))
        n = pl.value
        return pp[:n].copy(), pn[:n].copy(), [Break._from_c(b[i]) for i in range(bl.value)]

    @staticmethod
    def two_sided(p_pos, p_neg, breaks, ftw=0):
        """-> (f, p) in ascending absolute frequency f = f0 -+ f_j (units of the sample rate, f0 = ftw / 2^32), the
        DC (f_j = 0) and Nyquist (f_j = 1/2) bins once: they are the same bin on both sides"""
        f = Break.frequencies(breaks).astype(np.float64)
        p_pos, p_neg = np.asarray(p_pos), np.asarray(p_neg)
        neg = (f > 0) & (f < 0.5)
        f0 = int(ftw) / 2.0 ** 32
        return (np.concatenate([f0 - f[neg][::-1], f0 + f]), np.concatenate([p_neg[neg][::-1], p_pos]))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h and L is not None and getattr(L, "_lib", None) is not None:
            L._lib.sspsd_zoom_destroy(h)
            self._h = None


class Psd(_StreamOrdered):
    """Psd<N> + trait PsdStage, src/psd.rs:119-288 (one stage, decimated output exposed)."""

    def __init__(self, n=512, window=Window.HANN, device=0, hbf=Hbf.TAPS_140, stream=None):
        self.n = n
        self.device = int(device)
        cfg = _config(n, window, hbf, device, stream, 0, 0)
        h = C.c_void_p()
        L.check(L.lib().sspsd_stage_create(C.byref(cfg), C.byref(h)))
        self._h = h

    def _stream_ptr(self):
        s = C.c_void_p()
        L.check(L.lib().sspsd_stage_stream(self._h, C.byref(s)))
        return s.value or 0

    def set_avg(self, avg: int):
        L.check(L.lib().sspsd_stage_set_avg(self._h, avg))

    def set_detrend(self, d: Detrend):
        L.check(L.lib().sspsd_stage_set_detrend(self._h, int(d)))

    def process(self, x, out=None):
        """PsdStage::process(x, y) -> y[..n].  Returns a numpy array, or a view of `out` (a CUDA float32
        tensor that receives the decimated items on the device) when given."""
        ptr, n, mem, keep = _as_buffer(x)
        if mem == L.MEM_DEVICE:
            self._order_device_input(keep)
        if out is not None:
            self._order_device_input(out)  # written on the handle's stream
            yl = C.c_size_t(out.numel())
            L.check(L.lib().sspsd_stage_process_f32(self._h, ptr, n, mem, out.data_ptr(), C.byref(yl), L.MEM_DEVICE))
            self._release_device_input(out)  # also orders the read of x, if that is a CUDA tensor
            return out[:yl.value]
        y = np.zeros(n // 8 + self.n // 8 + 16, np.float32)
        yl = C.c_size_t(y.size)
        L.check(L.lib().sspsd_stage_process_f32(self._h, ptr, n, mem, y.ctypes.data, C.byref(yl), L.MEM_HOST))
        del keep
        return y[:yl.value]

    def spectrum(self):
        out = np.zeros(self.n // 2 + 1, np.float32)
        ln = C.c_size_t(out.size)
        L.check(L.lib().sspsd_stage_spectrum(self._h, out.ctypes.data, C.byref(ln), L.MEM_HOST))
        return out

    def count(self):
        c = C.c_uint32()
        L.check(L.lib().sspsd_stage_count(self._h, C.byref(c)))
        return c.value

    def gain(self):
        g = C.c_float()
        L.check(L.lib().sspsd_stage_gain(self._h, C.byref(g)))
        return g.value

    def buf(self):
        out = np.zeros(self.n, np.float32)
        ln = C.c_size_t(out.size)
        L.check(L.lib().sspsd_stage_buf(self._h, out.ctypes.data, C.byref(ln), L.MEM_HOST))
        return out[:ln.value]

    def __del__(self):
        h = getattr(self, "_h", None)
        if h and L is not None and getattr(L, "_lib", None) is not None:
            L._lib.sspsd_stage_destroy(h)
            self._h = None


class Format(enum.IntEnum):
    """enum Format, src/de/mod.rs:9-17"""
    AdcDac = 1
    Fls = 2
    ThermostatEem = 3
    Mpll = 4


TRACE_NAMES = {  # src/de/data.rs:37,48,59,70 / 100,111,124,131 / 155 / 181,190,199
    Format.AdcDac: ("ADC0", "ADC1", "DAC0", "DAC1"),
    Format.Fls: ("AR", "AP", "BI", "BQ"),
    Format.ThermostatEem: ("T00", "T20", "I0", "I1"),
    Format.Mpll: ("phase (rad)", "frequency (kHz)", "amplitude (V/G10)"),
}


class DecodeError(Exception):
    """de::Error (src/de/mod.rs:19-27) plus the reference's panics, by status code."""

    def __init__(self, status, frames_ok):
        super().__init__("%s at frame %d" % (L.STATUS_NAMES.get(status, status), frames_ok))
        self.status = status
        self.frames_ok = frames_ok


class Loss:
    """struct Loss, src/loss.rs:4-38"""

    def __init__(self):
        self.c = L.LossC()

    received = property(lambda self: self.c.received)
    dropped = property(lambda self: self.c.dropped)
    seq = property(lambda self: self.c.seq if self.c.has_seq else None)

    def update(self, seq, batches):
        L.lib().sspsd_loss_update(C.byref(self.c), seq, batches)

    def ratio(self):
        return L.lib().sspsd_loss_ratio(C.byref(self.c))


def _trace_map(target, traces):
    """The trace indices a CsdCascade / CsmCascade / ZoomCascade target of process_frames / pump reads, one per channel
    (default 0 .. K-1; a heterodyne ZoomCascade reads one trace); None for a list of PsdCascades, which take trace t
    into target[t]."""
    if not isinstance(target, (CsdCascade, CsmCascade, ZoomCascade)):
        if traces is not None:
            raise ValueError("traces= applies to a CsdCascade, CsmCascade or ZoomCascade target")
        return None
    if isinstance(target, ZoomCascade):
        k = 1 if target.mode == L.ZOOM_HETERODYNE else 2
    else:
        k = 2 if isinstance(target, CsdCascade) else target.channels
    tmap = list(range(k)) if traces is None else [int(t) for t in traces]
    if len(tmap) != k:
        raise ValueError("expected %d trace indices (one per channel), got %d" % (k, len(tmap)))
    return tmap


class FrameDecoder(_StreamOrdered):
    """Batched Frame::from_bytes + Loss::update + Payload::traces (src/de/frame.rs:49-60,
    src/loss.rs:11-26, src/de/data.rs)."""

    def __init__(self, device=0, stream=None):
        # stream=None: a private stream of the decoder's own (NULL in the C ABI), not torch's current one -- the frames'
        # H2D copy of call c + 1 must not queue behind the cascades of call c, which usually sit on torch's stream;
        # CUDA tensors handed in are ordered against torch's stream by _order_device_input
        h = C.c_void_p()
        L.check(L.lib().sspsd_decoder_create(device, stream or None, C.byref(h)))
        self._h = h
        self.device = int(device)

    def _stream_ptr(self):
        s = C.c_void_p()
        L.check(L.lib().sspsd_decoder_stream(self._h, C.byref(s)))
        return s.value or 0

    def _frames(self, frames, frame_len, frame_stride):
        if hasattr(frames, "data_ptr"):
            t = frames.contiguous()
            if t.is_cuda:
                self._order_device_input(t)
            return t.data_ptr(), t.numel(), (L.MEM_DEVICE if t.is_cuda else L.MEM_HOST), t
        a = np.frombuffer(frames, dtype=np.uint8) if not isinstance(frames, np.ndarray) else np.ascontiguousarray(frames, np.uint8)
        return a.ctypes.data, a.size, L.MEM_HOST, a

    def decode(self, frames, frame_len, loss: Loss = None, frame_stride=None, n_frames=None):
        """-> (format, [(name, np.ndarray)], frames_ok).  Raises DecodeError on a malformed frame after
        having accounted (in `loss`) for the frames before it."""
        frame_stride = frame_stride or frame_len
        ptr, nbytes, mem, keep = self._frames(frames, frame_len, frame_stride)
        if n_frames is None:
            n_frames = 0 if nbytes < frame_len else 1 + (nbytes - frame_len) // frame_stride
        payload = max(frame_len - 8, 0)
        cap = max(n_frames * max(payload // 64 * 8, payload // 24), 1)
        tr = [np.zeros(cap, np.float32) for _ in range(L.MAX_TRACES)]
        ptrs = (C.c_void_p * L.MAX_TRACES)(*[t.ctypes.data for t in tr])
        info = L.DecodeInfoC()
        st = L.lib().sspsd_decode_frames(self._h, ptr, n_frames, frame_len, frame_stride, mem,
                                         C.byref(loss.c) if loss is not None else None, ptrs, cap, L.MEM_HOST,
                                         C.byref(info))
        del keep
        traces = []
        if info.frames_ok:
            names = TRACE_NAMES[Format(info.format)]
            traces = [(names[t], tr[t][:info.samples_per_trace]) for t in range(info.n_traces)]
        if st in (L.EHEADER, L.EFORMAT, L.ESIZE, L.EBATCHES, L.ESHORT) and info.frames_ok < n_frames:
            err = DecodeError(st, info.frames_ok)
            err.traces = traces
            err.format = info.format
            raise err
        L.check(st)
        return (Format(info.format) if info.frames_ok else None), traces, info.frames_ok

    def decode_device(self, frames, frame_len, out, loss: Loss = None, frame_stride=None, n_frames=None):
        """Like decode(), but the traces stay on the device: `out` is a list of 4 CUDA float32 tensors that
        receive them.  Returns the sspsd_decode_info (format, n_traces, samples_per_trace, frames_ok)."""
        frame_stride = frame_stride or frame_len
        ptr, nbytes, mem, keep = self._frames(frames, frame_len, frame_stride)
        if n_frames is None:
            n_frames = 0 if nbytes < frame_len else 1 + (nbytes - frame_len) // frame_stride
        for t in out:
            self._order_device_input(t)  # written on the decoder's stream
        ptrs = (C.c_void_p * L.MAX_TRACES)(*[t.data_ptr() for t in out])
        info = L.DecodeInfoC()
        st = L.lib().sspsd_decode_frames(self._h, ptr, n_frames, frame_len, frame_stride, mem,
                                         C.byref(loss.c) if loss is not None else None, ptrs,
                                         min(t.numel() for t in out), L.MEM_DEVICE, C.byref(info))
        del keep
        if st in (L.EHEADER, L.EFORMAT, L.ESIZE, L.EBATCHES, L.ESHORT) and info.frames_ok < n_frames:
            raise DecodeError(st, info.frames_ok)
        L.check(st)
        return info

    def process_frames(self, target, frames, frame_len, loss: Loss = None, frame_stride=None, n_frames=None,
                       traces=None):
        """Fused decode -> spectra.  `target` is a list of PsdCascades (trace t -> target[t], None drops a trace;
        src/bin/psd.rs:174-182), a CsdCascade (x, y <- traces, default (0, 1)), a CsmCascade (channel i <-
        traces[i], default range(K)) or a ZoomCascade (I/Q: i, q <- traces, default (0, 1), e.g. (2, 3) for Fls BI /
        BQ; heterodyne: x <- traces[0], default 0, mixed on the device).  Raises DecodeError on a malformed frame after having consumed the frames
        before it."""
        tmap = _trace_map(target, traces)
        frame_stride = frame_stride or frame_len
        ptr, nbytes, mem, keep = self._frames(frames, frame_len, frame_stride)
        if n_frames is None:
            n_frames = 0 if nbytes < frame_len else 1 + (nbytes - frame_len) // frame_stride
        info = L.DecodeInfoC()
        lp = C.byref(loss.c) if loss is not None else None
        if isinstance(target, CsmCascade):
            st = L.lib().sspsd_csm_process_frames(self._h, target._h, (C.c_uint32 * len(tmap))(*tmap), ptr, n_frames,
                                                  frame_len, frame_stride, mem, lp, C.byref(info))
        elif isinstance(target, ZoomCascade):
            st = L.lib().sspsd_zoom_process_frames(self._h, target._h, (C.c_uint32 * len(tmap))(*tmap), ptr, n_frames,
                                                   frame_len, frame_stride, mem, lp, C.byref(info))
        elif isinstance(target, CsdCascade):
            st = L.lib().sspsd_csd_process_frames(self._h, target._h, tmap[0], tmap[1], ptr, n_frames, frame_len,
                                                  frame_stride, mem, lp, C.byref(info))
        else:
            hs = (C.c_void_p * len(target))(*[(c._h if c is not None else None) for c in target])
            st = L.lib().sspsd_cascade_process_frames(self._h, hs, len(target), ptr, n_frames, frame_len,
                                                      frame_stride, mem, lp, C.byref(info))
        del keep
        if st in (L.EHEADER, L.EFORMAT, L.ESIZE, L.EBATCHES, L.ESHORT) and info.frames_ok < n_frames:
            raise DecodeError(st, info.frames_ok)
        L.check(st)
        return info

    def __del__(self):
        h = getattr(self, "_h", None)
        if h and L is not None and getattr(L, "_lib", None) is not None:
            L._lib.sspsd_decoder_destroy(h)
            self._h = None


@dataclass
class Var:
    """struct Var / VarBuilder defaults, src/var.rs:4-19"""
    x_exp: int = -2
    sinx_exp: int = 4
    clip: float = 3.4028234663852886e38
    dc_cut: int = 2

    def eval(self, phase_psd, frequencies, tau):
        """Var::eval, src/var.rs:26-45"""
        p = np.ascontiguousarray(phase_psd, np.float32)
        f = np.ascontiguousarray(frequencies, np.float32)
        v = L.VarC(self.x_exp, self.sinx_exp, self.clip, 0, self.dc_cut)
        return L.lib().sspsd_var_eval(C.byref(v), p.ctypes.data, f.ctypes.data, min(p.size, f.size), tau)


@dataclass
class Trace:
    """struct Trace of src/bin/psd.rs:118-157: a merged spectrum with its breaks and frequencies.
    plot() is Trace::plot: trapezoidal integration over the irregular frequency grid (struct Trapezoidal,
    bin/psd.rs:96-116) and the log-log plot points."""
    name: str
    breaks: list
    psd: np.ndarray
    frequencies: np.ndarray

    def plot(self, fs=1.0, integral_start=1e-6, integral_end=0.5, integrate=False):
        """-> (sqrt of the integral over [integral_start, integral_end], points [n, 2] float64)"""
        p = np.ascontiguousarray(self.psd, np.float32)
        f = np.ascontiguousarray(self.frequencies, np.float32)
        n = min(p.size, f.size)
        o = L.PlotOptsC(fs, integral_start, integral_end, int(integrate))
        xy = np.zeros((max(n, 1), 2), np.float64)
        integ = C.c_float()
        npts = C.c_size_t(xy.shape[0])
        L.check(L.lib().sspsd_trace_plot(C.byref(o), p.ctypes.data, f.ctypes.data, n, C.byref(integ), xy.ctypes.data,
                                         C.byref(npts)))
        return integ.value, xy[:npts.value].copy()


class SourceKind(enum.IntEnum):
    NOISE = 0
    DSM = 1


class Source:
    """Data::Noise / Data::Dsm of src/source.rs:66-79, 104-134, generated on the device.

    Source.noise(e): power-law noise with PSD ~ f^e (`--noise e`, source.rs:40-42);
    Source.dsm(ftw): MASH-1-1-1 modulated sine marker (`--dsm ftw`, source.rs:44-46)."""

    SEED = 0x7654321  # source.rs:69

    def __init__(self, kind, param, seed=SEED, device=0, stream=None):
        if stream is None:
            stream = _default_stream(device)
        h = C.c_void_p()
        L.check(L.lib().sspsd_source_create(int(kind), int(param), int(seed), device, stream, C.byref(h)))
        self._h = h
        self.device = device

    @classmethod
    def noise(cls, exponent, seed=SEED, device=0, stream=None):
        return cls(SourceKind.NOISE, exponent, seed, device, stream)

    @classmethod
    def dsm(cls, ftw, device=0, stream=None):
        return cls(SourceKind.DSM, ftw, 0, device, stream)

    def reset(self):
        L.check(L.lib().sspsd_source_reset(self._h))

    def position(self):
        p = C.c_uint64()
        L.check(L.lib().sspsd_source_position(self._h, C.byref(p)))
        return p.value

    def generate_raw(self, ptr, n):
        """next n samples into device memory at ptr (asynchronous on the source's stream)"""
        L.check(L.lib().sspsd_source_generate(self._h, ptr, n))

    def get(self, n, out=None):
        """Source::get with a caller-chosen block length: the next n samples as a device tensor"""
        import torch
        if out is None:
            out = torch.empty(n, dtype=torch.float32, device=f"cuda:{self.device}")
        assert out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and out.numel() >= n
        self.generate_raw(out.data_ptr(), n)
        return out[:n]

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and L is not None and L._lib is not None:
            L._lib.sspsd_source_destroy(h)


class Receiver:
    """Data::Udp of src/source.rs:81-93, 159-165: datagrams collected with recvmmsg into page-locked
    slots and handed on as runs of equally sized frames.

    Receiver(ip, port): SourceOpts::{ip, port} (source.rs:17-23).  `pinned=False` keeps the slots in
    plain host memory (hosts without a CUDA device)."""

    def __init__(self, ip="0.0.0.0", port=9293, slot_bytes=2048, n_slots=1024, pinned=True):
        h = C.c_void_p()
        L.check(L.lib().sspsd_receiver_create(ip.encode(), port, slot_bytes, n_slots, 0 if pinned else 1, C.byref(h)))
        self._h = h

    def _info(self):
        port, slot, n = C.c_uint16(), C.c_size_t(), C.c_uint64()
        L.check(L.lib().sspsd_receiver_info(self._h, C.byref(port), C.byref(slot), C.byref(n)))
        return port.value, slot.value, n.value

    @property
    def port(self):
        return self._info()[0]

    @property
    def slot_bytes(self):
        return self._info()[1]

    @property
    def datagrams(self):
        return self._info()[2]

    def recv(self, max_frames=1024, timeout_ms=1000):
        """-> (frames, frame_len): frames is a (n, slot_bytes) uint8 view of the slots (valid until the
        next call), the first frame_len bytes of each row are the datagram; n == 0 on timeout"""
        ptr, n, ln = C.c_void_p(), C.c_size_t(), C.c_size_t()
        L.check(L.lib().sspsd_receiver_recv(self._h, max_frames, timeout_ms, C.byref(ptr), C.byref(n), C.byref(ln)))
        slot = self.slot_bytes
        if n.value == 0:
            return np.empty((0, slot), np.uint8), 0
        buf = (C.c_uint8 * (n.value * slot)).from_address(ptr.value)
        return np.frombuffer(buf, np.uint8).reshape(n.value, slot), ln.value

    def pump(self, decoder, target, loss: "Loss" = None, max_frames=1024, timeout_ms=1000, traces=None):
        """recv + FrameDecoder.process_frames in one call (`target` and `traces` as there); returns the decode info
        (frames_ok == 0 on timeout).  Malformed datagrams raise DecodeError like process_frames."""
        tmap = _trace_map(target, traces)
        info = L.DecodeInfoC()
        lp = C.byref(loss.c) if loss is not None else None
        if isinstance(target, CsmCascade):
            st = L.lib().sspsd_receiver_pump_csm(self._h, decoder._h, target._h, (C.c_uint32 * len(tmap))(*tmap),
                                                 max_frames, timeout_ms, lp, C.byref(info))
        elif isinstance(target, ZoomCascade):
            st = L.lib().sspsd_receiver_pump_zoom(self._h, decoder._h, target._h, (C.c_uint32 * len(tmap))(*tmap),
                                                  max_frames, timeout_ms, lp, C.byref(info))
        elif isinstance(target, CsdCascade):
            st = L.lib().sspsd_receiver_pump_csd(self._h, decoder._h, target._h, tmap[0], tmap[1], max_frames,
                                                 timeout_ms, lp, C.byref(info))
        else:
            hs = (C.c_void_p * L.MAX_TRACES)()
            for t, c in enumerate(target[:L.MAX_TRACES]):
                hs[t] = c._h if c is not None else None
            st = L.lib().sspsd_receiver_pump(self._h, decoder._h, hs, min(len(target), L.MAX_TRACES), max_frames,
                                             timeout_ms, lp, C.byref(info))
        if L.EHEADER <= st <= L.ESHORT:
            raise DecodeError(st, info.frames_ok)
        L.check(st)
        return info

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and L is not None and getattr(L, "_lib", None) is not None:
            L._lib.sspsd_receiver_destroy(h)


class _BorrowedCascade(PsdCascade):
    """a cascade handle owned by a Group: never destroyed from Python"""

    def __del__(self):
        self._h = None


class ShardMode(enum.IntEnum):
    CHANNELS = 0
    TIME = 1


@dataclass
class TimeChunk:
    """sspsd_time_chunk: what one rank of a time-chunked group owns and is fed"""
    own_lo: int
    own_hi: object   # None for the last rank
    feed_lo: int
    feed_hi: int
    tail_lo: int
    tail_hi: object  # None: open
    n_local: int

    @staticmethod
    def _from_c(c):
        none = 2 ** 64 - 1
        return TimeChunk(c.own_lo, None if c.own_hi == none else c.own_hi, c.feed_lo, c.feed_hi, c.tail_lo,
                         None if c.tail_hi == none else c.tail_hi, c.n_local)


def time_plan(n_fft, total, n_ranks, rank, n_local=0, window=Window.HANN, hbf=Hbf.TAPS_140):
    """sspsd_time_plan: pure host planner of the time-chunked mode"""
    out = L.TimeChunkC()
    L.check(L.lib().sspsd_time_plan(n_fft, int(window), int(hbf), total, n_ranks, rank, n_local, C.byref(out)))
    return TimeChunk._from_c(out)


class Group:
    """sspsd_group: the reference's single-threaded loop over traces (src/bin/psd.rs:170-183) spread over GPUs,
    with the NCCL plumbing inside the library.

    Group(n, devices=[0, 1, ...])            all ranks in this process (ncclCommInitAll / peer loads)
    Group(n, rank=r, n_ranks=w, unique_id=b) one rank of a multi-process job (torchrun): unique_id from
                                             Group.unique_id() on rank 0, broadcast by the caller"""

    def __init__(self, n=512, devices=None, mode=ShardMode.CHANNELS, rank=None, n_ranks=None, unique_id=None, device=0,
                 hbf=Hbf.TAPS_140, max_batch=0, host_stage=0, stream=None):
        self.n = n
        cfg = _config(n, Window.HANN, hbf, device, 0, max_batch, host_stage)
        cfg.stream = stream  # one-rank-per-process groups only; None = private streams
        h = C.c_void_p()
        if rank is None:
            devices = list(devices if devices is not None else [0])
            arr = (C.c_int32 * len(devices))(*devices)
            L.check(L.lib().sspsd_group_create(C.byref(cfg), arr, len(devices), int(mode), C.byref(h)))
            self.n_ranks, self.rank = len(devices), 0
        else:
            buf = (C.c_uint8 * 128).from_buffer_copy(bytes(unique_id)) if unique_id is not None else None
            L.check(L.lib().sspsd_group_create_rank(C.byref(cfg), buf, rank, n_ranks, int(mode), C.byref(h)))
            self.n_ranks, self.rank = n_ranks, rank
        self._h = h
        self.mode = ShardMode(mode)

    @staticmethod
    def unique_id():
        buf = (C.c_uint8 * 128)()
        L.check(L.lib().sspsd_group_unique_id(buf))
        return bytes(buf)

    def info(self):
        a, b, c = C.c_uint32(), C.c_uint32(), C.c_uint32()
        m, r = C.c_int32(), C.c_int32()
        L.check(L.lib().sspsd_group_info(self._h, C.byref(a), C.byref(b), C.byref(c), C.byref(m), C.byref(r)))
        return dict(n_ranks=a.value, first_rank=b.value, n_local_ranks=c.value, mode=m.value,
                    reduce="nccl" if r.value == 0 else "p2p")

    def set_avg(self, avg: AvgOpts):
        L.check(L.lib().sspsd_group_set_avg(self._h, L.AvgOptsC(avg.limit, avg.count)))

    def set_detrend(self, d: Detrend):
        L.check(L.lib().sspsd_group_set_detrend(self._h, int(d)))

    def sync(self):
        L.check(L.lib().sspsd_group_sync(self._h))

    # ---- channels ----
    def process(self, channel, x):
        ptr, n, mem, keep = _as_buffer(x)
        if mem == L.MEM_DEVICE:
            import torch
            torch.cuda.current_stream(keep.device).synchronize()  # the group's handles own their streams
        L.check(L.lib().sspsd_group_process_f32(self._h, channel, ptr, n, mem))
        if mem == L.MEM_DEVICE:
            self.sync()  # the tensor is borrowed for the call only
        del keep

    def process_raw(self, channel, ptr, n, mem):
        L.check(L.lib().sspsd_group_process_f32(self._h, channel, ptr, n, mem))

    def channel_cascade(self, channel):
        """the PsdCascade of a channel this process owns (borrowed from the group), or None"""
        h = C.c_void_p()
        L.check(L.lib().sspsd_group_channel_handle(self._h, channel, C.byref(h)))
        if not h.value:
            return None
        c = PsdCascade.__new__(PsdCascade)
        c.n, c.device, c._h, c._borrowed = self.n, self.channel_device(channel)[0], h, self
        c.__class__ = _BorrowedCascade
        return c

    def channel_device(self, channel):
        d, r = C.c_int32(), C.c_uint32()
        L.check(L.lib().sspsd_group_channel_device(self._h, channel, C.byref(d), C.byref(r)))
        return d.value, r.value

    def psd(self, channel=0, opts: MergeOpts = None):
        opts = opts or MergeOpts()
        o = L.MergeOptsC(int(opts.keep_overlap), opts.min_count, int(opts.keep_transition_band))
        p = np.zeros(L.MAX_STAGES * (self.n // 2 + 1), np.float32)
        b = (L.BreakC * L.MAX_STAGES)()
        pl, bl = C.c_size_t(p.size), C.c_size_t(L.MAX_STAGES)
        L.check(L.lib().sspsd_group_psd(self._h, channel, C.byref(o), p.ctypes.data, C.byref(pl), b, C.byref(bl)))
        return p[:pl.value].copy(), [Break._from_c(b[i]) for i in range(bl.value)]

    def psd_all(self, n_channels, opts: MergeOpts = None):
        """-> [(p, breaks)] per channel on the process holding rank 0 (empty arrays elsewhere); a collective in
        a multi-process group"""
        opts = opts or MergeOpts()
        o = L.MergeOptsC(int(opts.keep_overlap), opts.min_count, int(opts.keep_transition_band))
        ps = L.MAX_STAGES * (self.n // 2 + 1)
        p = np.zeros((n_channels, ps), np.float32)
        b = (L.BreakC * (L.MAX_STAGES * n_channels))()
        pl = (C.c_size_t * n_channels)()
        bl = (C.c_size_t * n_channels)()
        L.check(L.lib().sspsd_group_psd_all(self._h, n_channels, C.byref(o), p.ctypes.data, ps, pl, b, L.MAX_STAGES, bl))
        return [(p[c, :pl[c]].copy(), [Break._from_c(b[c * L.MAX_STAGES + i]) for i in range(bl[c])])
                for c in range(n_channels)]

    # ---- time chunks of one stream ----
    def time_plan(self, total, n_local=0):
        L.check(L.lib().sspsd_group_time_plan(self._h, total, n_local))

    def time_chunk(self, rank):
        out = L.TimeChunkC()
        L.check(L.lib().sspsd_group_time_chunk(self._h, rank, C.byref(out)))
        return TimeChunk._from_c(out)

    def time_process(self, rank, x):
        ptr, n, mem, keep = _as_buffer(x)
        if mem == L.MEM_DEVICE:
            import torch
            torch.cuda.current_stream(keep.device).synchronize()
        L.check(L.lib().sspsd_group_time_process_f32(self._h, rank, ptr, n, mem))
        if mem == L.MEM_DEVICE:
            self.sync()
        del keep

    def time_process_all(self, x):
        a = np.ascontiguousarray(x, dtype=np.float32)
        L.check(L.lib().sspsd_group_time_process_all_f32(self._h, a.ctypes.data, a.size))

    def time_process_noise(self, exponent=0, seed=Source.SEED):
        L.check(L.lib().sspsd_group_time_process_noise(self._h, exponent, seed))

    def time_finish(self):
        L.check(L.lib().sspsd_group_time_finish(self._h))

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and L is not None and getattr(L, "_lib", None) is not None:
            L._lib.sspsd_group_destroy(h)
