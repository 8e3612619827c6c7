#!/usr/bin/env python3
"""Headless driver in the shape of the reference's `stream_test` binary (src/bin/stream_test.rs:35-76) on top
of the GPU cascade: read a source, feed one PsdCascade per trace, then log breaks, PSD and the FVAR sweep.

Sources (reference src/source.rs:16-48, 102-167):
  --raw FILE          native-endian f32 samples, no header (what stream_to_raw writes, stream_to_raw.rs:20-26)
  --file FILE         stabilizer frames of --frame-size bytes each (default 8 + 30*2*6*4 like source.rs:29-31)
  --noise N           synthetic power-law noise f^N generated on the device (|N| integrators/differentiators,
                      source.rs:104-118)
  --udp IP:PORT       live Stabilizer stream (source.rs:81-93, 159-165): recvmmsg batches into page-locked slots;
                      ends after --samples items per trace or 1 s without traffic
  --dsm FTW           MASH-1-1-1 modulated sine marker generated on the device (source.rs:119-130)
--repeat wraps files around; the run ends after --samples items per trace (files: at EOF without --repeat).
Host reads go through a pinned double buffer, so the H2D copy of block b+1 overlaps the kernels of block b.

--csm TRACES (with --file or --udp), e.g. 0,2 or 0,1,2,3: feed the listed traces of the frames to one CsmCascade
instead of one PsdCascade per trace, and report the diagonal PSD of --trace (one of TRACES, default the first) plus
the median coherence of every pair; --save FILE.npz writes the matrix S [K, K, bins], the frequencies and the breaks.

--iq I,Q (with --file or --udp), e.g. 2,3 for the BI / BQ of Fls frames: feed the two traces as z = I + i Q to a
ZoomCascade and report its two-sided spectrum.  --zoom FTW (with --file or --udp): mix trace --trace down by the
carrier FTW / 2^32 of the sample rate on the device (ZoomCascade.heterodyne) and report the two-sided spectrum around
it.  With either, --save FILE.npz writes p_pos, p_neg, the frequencies f >= 0 (p_pos at f0 + f, p_neg at f0 - f), the
absolute two-sided axis and spectrum, and the breaks.
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from stabilizer_stream_b200 import (Break, CsmCascade, Detrend, FrameDecoder, Loss, MergeOpts, PsdCascade, Receiver,
                                    Source, Var, ZoomCascade)  # noqa: E402

BREAK_FIELDS = ("start", "include", "count", "avg", "bins_start", "bins_end", "fft_size", "decimation", "pending",
                "processed")


def break_row(k):
    return [k.start, k.include, k.count, k.avg, k.bins.start, k.bins.stop, k.fft_size, k.decimation, k.pending,
            k.processed]


def parse_csm(ap, a):
    """--csm / --trace / --save checks, before any device work: -> the trace list or None"""
    if a.csm is None:
        if a.save and a.iq is None and a.zoom is None:
            ap.error("--save needs --csm, --iq or --zoom")
        return None
    try:
        traces = [int(t) for t in a.csm.split(",")]
    except ValueError:
        ap.error("--csm takes comma-separated trace indices, e.g. 0,2")
    if not 2 <= len(traces) <= 4:
        ap.error("--csm takes 2 to 4 trace indices (a CsmCascade has at most 4 channels)")
    if any(not 0 <= t < 4 for t in traces):
        ap.error("--csm trace indices are 0 .. 3")
    if not (a.file or a.udp):
        ap.error("--csm needs --file or --udp (frames carry the traces)")
    if a.trace is not None and a.trace not in traces:
        ap.error("--trace must be one of the --csm traces")
    return traces


def parse_zoom(ap, a):
    """--iq / --zoom checks, before any device work: -> the trace map of the ZoomCascade or None"""
    if sum(v is not None for v in (a.csm, a.iq, a.zoom)) > 1:
        ap.error("use one of --csm, --iq, --zoom")
    if a.iq is None and a.zoom is None:
        return None
    if not (a.file or a.udp):
        ap.error("--iq / --zoom need --file or --udp (frames carry the traces)")
    if a.iq is not None:
        try:
            traces = [int(t) for t in a.iq.split(",")]
        except ValueError:
            traces = []
        if len(traces) != 2:
            ap.error("--iq takes two trace indices I,Q, e.g. 2,3")
        if a.trace is not None:
            ap.error("--trace does not apply to --iq (the spectrum is of I + i Q)")
    else:
        if not 0 <= a.zoom < 2 ** 32:
            ap.error("--zoom takes a 32-bit frequency tuning word")
        traces = [0 if a.trace is None else a.trace]
    if any(not 0 <= t < 4 for t in traces):
        ap.error("--iq / --trace indices are 0 .. 3")
    return traces


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--raw")
    ap.add_argument("--file")
    ap.add_argument("--frame-size", type=int, default=8 + 30 * 2 * 6 * 4)
    ap.add_argument("--noise", type=int)
    ap.add_argument("--dsm", type=int)
    ap.add_argument("--udp")
    ap.add_argument("--repeat", action="store_true")
    ap.add_argument("--samples", type=float, default=0, help="stop after this many items per trace (0: until EOF)")
    ap.add_argument("--fft", type=int, default=512, help="FFT size N (the reference binaries use 512)")
    ap.add_argument("--detrend", default="midpoint", choices=["none", "midpoint", "span", "mean"])
    ap.add_argument("--trace", type=int, default=None, help="trace to report (default 0; with --csm the first of TRACES)")
    ap.add_argument("--csm", metavar="TRACES", help="comma-separated traces (2 to 4) into one CsmCascade")
    ap.add_argument("--iq", metavar="I,Q", help="two traces into one ZoomCascade as I + i Q (two-sided spectrum)")
    ap.add_argument("--zoom", metavar="FTW", type=int,
                    help="mix --trace down by the carrier FTW / 2^32 of the sample rate (two-sided spectrum around it)")
    ap.add_argument("--save", metavar="FILE.npz", help="with --csm, --iq or --zoom: write the spectra, frequencies and breaks")
    ap.add_argument("--block", type=int, default=1 << 24, help="items (or frames*64) read per block")
    ap.add_argument("--json", action="store_true")
    a = ap.parse_args()
    csm_traces = parse_csm(ap, a)
    zoom_traces = parse_zoom(ap, a)
    if zoom_traces:
        csm_traces = None
    if a.trace is None:
        a.trace = csm_traces[0] if csm_traces else 0
    dev = torch.device("cuda", 0)
    det = Detrend[a.detrend.upper()]
    limit = int(a.samples)
    cas, names, loss = [], [], Loss()
    total = 0
    t0 = time.perf_counter()

    def cascades(n):
        if zoom_traces:
            if not cas:
                z = ZoomCascade.iq(a.fft) if a.iq is not None else ZoomCascade.heterodyne(a.fft, a.zoom)
                z.set_detrend(det)
                cas.append(z)
            return
        if csm_traces:
            if not cas:
                m = CsmCascade(a.fft, len(csm_traces))
                m.set_detrend(det)
                cas.append(m)
            return
        while len(cas) < n:
            c = PsdCascade(a.fft)
            c.set_detrend(det)
            cas.append(c)

    def target():
        return cas[0] if (csm_traces or zoom_traces) else cas

    tmap = zoom_traces or csm_traces

    if a.noise is not None or a.dsm is not None:
        cascades(1)
        names = ["noise" if a.dsm is None else "dsm"]
        src = Source.noise(a.noise) if a.dsm is None else Source.dsm(a.dsm)
        if limit == 0:
            ap.error("--noise/--dsm need --samples")
        while total < limit:
            n = min(a.block, limit - total)
            cas[0].process_source(src, n)  # generated and consumed on the device
            total += n
    elif a.raw:
        cascades(1)
        names = ["raw"]
        pinned = [torch.empty(a.block, dtype=torch.float32, pin_memory=True) for _ in range(2)]
        with open(a.raw, "rb") as f:
            b = 0
            while True:
                buf = pinned[b & 1]
                got = f.readinto(memoryview(buf.numpy()).cast("B"))
                n = got // 4
                if n == 0:
                    if a.repeat and total:
                        f.seek(0)
                        continue
                    break
                if limit and total + n > limit:
                    n = limit - total
                cas[0].process(buf[:n])   # returns once the H2D copy is done; kernels keep running
                total += n
                b += 1
                if limit and total >= limit:
                    break
    elif a.file:
        dec = FrameDecoder()
        fpb = max(1, a.block * 2 // a.frame_size)
        with open(a.file, "rb") as f:
            while True:
                data = f.read(fpb * a.frame_size)
                nfr = len(data) // a.frame_size
                if nfr == 0:
                    if a.repeat and total:
                        f.seek(0)
                        continue
                    break
                cascades(4)
                info = dec.process_frames(target(), data[:nfr * a.frame_size], a.frame_size, loss, traces=tmap)
                if not names:
                    from stabilizer_stream_b200.psd import TRACE_NAMES, Format
                    names = list(TRACE_NAMES[Format(info.format)])
                total += info.samples_per_trace
                if limit and total >= limit:
                    break
    elif a.udp:
        ip, _, port = a.udp.rpartition(":")
        rx = Receiver(ip or "0.0.0.0", int(port))
        dec = FrameDecoder()
        cascades(4)
        while True:
            info = rx.pump(dec, target(), loss, max_frames=1024, timeout_ms=1000, traces=tmap)
            if info.frames_ok == 0:
                break
            if not names:
                from stabilizer_stream_b200.psd import TRACE_NAMES, Format
                names = list(TRACE_NAMES[Format(info.format)])
            total += info.samples_per_trace
            if limit and total >= limit:
                break
    else:
        ap.error("one of --raw, --file, --udp, --noise, --dsm is required")

    coherence = []
    zoom = None
    if zoom_traces:
        pp, pn, b = cas[0].spectrum(MergeOpts())
        dt = time.perf_counter() - t0
        ftw = a.zoom or 0
        fa, pa = ZoomCascade.two_sided(pp, pn, b, ftw)
        y = (pp + pn).astype(np.float32)  # both sides folded: what fdev of a real trace would see
        zoom = {"mode": "iq" if a.iq is not None else "heterodyne", "traces": zoom_traces, "ftw": ftw,
                "f0": ftw / 2.0 ** 32, "bins": int(pa.size),
                "peak": {"f": float(fa[np.argmax(pa)]), "p": float(np.max(pa))} if pa.size else None}
        if a.save:
            np.savez(a.save, p_pos=pp, p_neg=pn, frequencies=Break.frequencies(b), f_abs=fa, p_abs=pa,
                     traces=np.array(zoom_traces), ftw=np.uint32(ftw),
                     breaks=np.array([break_row(k_) for k_ in b], np.uint64).reshape(-1, len(BREAK_FIELDS)),
                     break_fields=np.array(BREAK_FIELDS))
    elif csm_traces:
        S, b = cas[0].csm(MergeOpts())
        dt = time.perf_counter() - t0
        y = np.real(S[csm_traces.index(a.trace), csm_traces.index(a.trace)]).astype(np.float32)
        coh = CsmCascade.coherence(S)
        k = len(csm_traces)
        for i in range(k):
            for j in range(i + 1, k):
                coherence.append({"traces": [csm_traces[i], csm_traces[j]],
                                  "median": float(np.median(coh[i, j])) if coh.shape[-1] else None})
        if a.save:
            np.savez(a.save, S=S, frequencies=Break.frequencies(b), traces=np.array(csm_traces),
                     breaks=np.array([break_row(k_) for k_ in b], np.uint64).reshape(-1, len(BREAK_FIELDS)),
                     break_fields=np.array(BREAK_FIELDS))
    else:
        c = cas[min(a.trace, len(cas) - 1)]
        y, b = c.psd(MergeOpts())
        dt = time.perf_counter() - t0
    f = Break.frequencies(b)
    fdev = []
    if b:
        var = Var(dc_cut=1, clip=1.0)          # stream_test.rs:62
        tau = 1.0
        while tau <= b[0].effective_fft_size() // 2:
            fdev.append((tau, float(np.sqrt(max(var.eval(y, f, tau), 0.0)))))
            tau *= 2.0
    out = {"trace": names[min(a.trace, len(names) - 1)] if names else None, "items_per_trace": int(total),
           "traces": len(csm_traces) if csm_traces else len(cas), "seconds": dt, "MSps_per_trace": total / dt / 1e6,
           "breaks": [{"start": k.start, "count": k.count, "bins": [k.bins.start, k.bins.stop], "decimation": k.decimation,
                       "pending": k.pending, "processed": k.processed, "include": k.include} for k in b],
           "psd_bins": int(y.size), "psd_median": float(np.median(y)) if y.size else None,
           "fdev": fdev[:8], "loss": {"received": loss.received, "dropped": loss.dropped}}
    if csm_traces:
        out["csm"] = {"traces": csm_traces, "coherence": coherence}
    if zoom:
        out["zoom"] = zoom
    if a.json:
        print(json.dumps(out))
    else:
        print("breaks:", out["breaks"])
        print("psd: %d bins, median %.6g" % (out["psd_bins"], out["psd_median"] or 0))
        print("fdev:", out["fdev"])
        if zoom and zoom["peak"]:
            print("two-sided: %d bins around f0 = %.9g, peak %.6g at %.9g" % (zoom["bins"], zoom["f0"], zoom["peak"]["p"],
                                                                          zoom["peak"]["f"]))
        for c_ in coherence:
            i, j = c_["traces"]
            print("coherence %s / %s: median %.4g over %d bins" % (names[i] if names else i, names[j] if names else j,
                                                                 c_["median"] or 0, y.size))
        if loss.received:
            print("Loss: %g %% (%d of %d)" % (100 * loss.ratio(), loss.dropped, loss.received + loss.dropped))
        print("%.1f MS/s per trace over %.2f s" % (out["MSps_per_trace"], dt))


if __name__ == "__main__":
    main()
