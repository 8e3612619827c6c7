#!/usr/bin/env python3
"""End-to-end rate of the cross-spectral matrix fed from Stabilizer frames in pinned host memory (BASELINE config 3's
shape: 2^20 AdcDac frames of 22 batches, 1416 bytes each, every 1009th frame lost, the sequence counter wrapping).

Arms, alternated in one process, each a full pass over the frames in calls of --chunk frames followed by the readout:
  frames_csm   FrameDecoder.process_frames(CsmCascade(N, 4), ...): sub-chunked H2D copy overlapped with decode + CSM
  manual_csm   the manual path: H2D copy, FrameDecoder.decode_device into four tensors, CsmCascade.process
  frames_psd4  FrameDecoder.process_frames into four PsdCascade(N)s (bench.py's e2e_frames path)
  copy         a bare pinned H2D copy of the same bytes: the ceiling
Prints and writes (--out) G trace-samples/s per arm (four traces per frame sample), each as a share of the copy's
rate, with the card's name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from stabilizer_stream_b200 import CsmCascade, FrameDecoder, Loss, MergeOpts, PsdCascade  # noqa: E402

BATCHES, N_FRAMES, DROP_EVERY = 22, 1 << 20, 1009
FLEN = 8 + 64 * BATCHES
ARMS = ("frames_csm", "manual_csm", "frames_psd4", "copy")


def gpu_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = q[0] if q else None
    except OSError:
        info["power_limit_and_max_sm_clock"] = None
    return info


def make_frames():
    """2^20 AdcDac frames in pinned memory; the sequence numbers of every DROP_EVERY-th frame are skipped and start
    just below 2^32, so the counter wraps within the first pass"""
    rng = np.random.default_rng(3)
    fr = np.empty((N_FRAMES, FLEN), np.uint8)
    fr[:, 0], fr[:, 1], fr[:, 2], fr[:, 3] = 0x7B, 0x05, 1, BATCHES
    idx = np.arange(N_FRAMES, dtype=np.uint64)
    slot = idx + idx // (DROP_EVERY - 1)  # frame f sits at stream slot f + (frames dropped before it)
    seq = ((slot * BATCHES + 0xFFFFF000) & 0xFFFFFFFF).astype(np.uint32)
    fr[:, 4:8] = seq.view(np.uint8).reshape(N_FRAMES, 4)
    base = rng.integers(0, 256, (1 << 16, FLEN - 8), dtype=np.uint8)  # ADC/DAC words, repeated every 2^16 frames
    for f0 in range(0, N_FRAMES, 1 << 16):
        fr[f0:f0 + (1 << 16), 8:] = base
    return torch.from_numpy(fr.reshape(-1)).pin_memory()


class Arm:
    def __init__(self, name, n, host, chunk):
        self.name, self.host, self.chunk = name, host, chunk
        self.dec = FrameDecoder(0)
        if name in ("frames_csm", "manual_csm"):
            self.target = CsmCascade(n, 4)
        elif name == "frames_psd4":
            self.target = [PsdCascade(n) for _ in range(4)]
        if name == "manual_csm":
            self.dframes = torch.empty(chunk * FLEN, dtype=torch.uint8, device="cuda")
            self.traces = [torch.empty(chunk * BATCHES * 8 + 64, dtype=torch.float32, device="cuda") for _ in range(4)]
        if name == "copy":
            self.dframes = torch.empty(N_FRAMES * FLEN, dtype=torch.uint8, device="cuda")

    def one_pass(self):
        loss = Loss()
        if self.name == "copy":
            self.dframes.copy_(self.host, non_blocking=True)
            return loss
        for f0 in range(0, N_FRAMES, self.chunk):
            part = self.host[f0 * FLEN:(f0 + self.chunk) * FLEN]
            if self.name == "manual_csm":
                d = self.dframes[:part.numel()]
                d.copy_(part, non_blocking=True)
                info = self.dec.decode_device(d, FLEN, self.traces, loss)
                self.target.process([t[:info.samples_per_trace] for t in self.traces])
            else:
                self.dec.process_frames(self.target, part, FLEN, loss)
        if isinstance(self.target, list):
            for c in self.target:
                c.psd(MergeOpts())
        else:
            self.target.csm(MergeOpts())
        return loss

    def timed(self):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loss = self.one_pass()
        torch.cuda.synchronize()
        return time.perf_counter() - t0, loss


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--sizes", default="4096,512")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--chunk", type=int, default=1 << 16, help="frames per call")
    ap.add_argument("--out", help="write the result JSON here")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    host = make_frames()
    samples = 4 * N_FRAMES * BATCHES * 8
    out = {"gpu": gpu_info(), "frames": N_FRAMES, "frame_bytes": FLEN, "frames_per_call": a.chunk,
           "h2d_bytes_per_pass": N_FRAMES * FLEN, "trace_samples_per_pass": samples, "rounds": a.rounds, "sizes": {}}
    for n in [int(v) for v in a.sizes.split(",")]:
        arms = [Arm(name, n, host, a.chunk) for name in ARMS]
        losses = {}
        for arm in arms:  # warm-up pass of every shape
            arm.timed()
        times = {arm.name: [] for arm in arms}
        for _ in range(a.rounds):
            for arm in arms:
                dt, loss = arm.timed()
                times[arm.name].append(dt)
                losses[arm.name] = (int(loss.received), int(loss.dropped))
        med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
        rate = {k: samples / v / 1e9 for k, v in med.items()}
        res = {k: {"G_trace_samples_per_s": rate[k], "share_of_copy": rate[k] / rate["copy"], "seconds": med[k],
                   "seconds_all": times[k]} for k in med}
        res["copy"]["GBps"] = N_FRAMES * FLEN / med["copy"] / 1e9
        res["loss"] = {k: v for k, v in losses.items() if k != "copy"}
        out["sizes"][str(n)] = res
        for k in ARMS:
            print("N=%d %-12s %6.2f G trace-samples/s  %5.1f %% of copy" % (n, k, rate[k], 100 * rate[k] / rate["copy"]),
                  flush=True)
        del arms
        torch.cuda.empty_cache()
    print(json.dumps(out))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
