#!/usr/bin/env python3
"""Throughput of the cross-spectral matrix (CsmCascade, 4 channels) against CsdCascades on the same data.

Four device-resident channels of 200e6 samples each are fed per step, at N = 512 and 4096, Hann window, default
options, one readout at the end of the timed window.  Reported: input samples per second with all four channels
counted once (the data a user has), for
  csm4   CsmCascade(N, 4).process(x)                the whole 4 x 4 matrix
  csd6   six CsdCascade(N), one per pair i < j       the same matrix, pair by pair
  csd2   two CsdCascade(N), pairs (0, 1) and (2, 3)  only the diagonal blocks
The setups alternate over `--rounds` rounds so that the spread shows.  CUDA events on the handles' shared stream.
Then one step of csm4 per size runs under torch.profiler (a separate, untimed pass) for the device time of
csd_stage_kernel against csm_cross_kernel.

    python tools/bench_csm.py --out profiles/r05_csm_bench.json
"""
import argparse
import itertools
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from stabilizer_stream_b200 import CsdCascade, CsmCascade, MergeOpts  # noqa: E402

SAMPLES = 200_000_000
SETUPS = ("csm4", "csd6", "csd2")


def gpu_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = q[0] if q else None
    except OSError:
        info["power_limit_and_max_sm_clock"] = None
    return info


def make(setup, n, stream):
    s = stream.cuda_stream or 1
    if setup == "csm4":
        return [((0, 1, 2, 3), CsmCascade(n, 4, stream=s))]
    pairs = itertools.combinations(range(4), 2) if setup == "csd6" else [(0, 1), (2, 3)]
    return [(p, CsdCascade(n, stream=s)) for p in pairs]


def step(handles, xs):
    for chans, h in handles:
        if isinstance(h, CsmCascade):
            h.process(xs)
        else:
            h.process(xs[chans[0]], xs[chans[1]])


def readout(handles):
    for _, h in handles:
        (h.csm if isinstance(h, CsmCascade) else h.csd)(MergeOpts())


def run(setup, n, xs, steps, warmup, stream):
    handles = make(setup, n, stream)
    for _ in range(warmup):
        step(handles, xs)
    readout(handles)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        step(handles, xs)
    readout(handles)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    return 4.0 * SAMPLES * steps / (ms * 1e-3)


def kernel_times(n, xs, stream):
    """device time (ms) per kernel name of one csm4 step, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    handles = make("csm4", n, stream)
    step(handles, xs)
    readout(handles)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step(handles, xs)
        readout(handles)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        for name in ("csd_stage_kernel", "csm_cross_kernel", "hbf", "decim"):
            if name in e.key and t > 0:
                out[name] = round(out.get(name, 0.0) + t / 1e3, 3)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--sizes", default="512,4096")
    ap.add_argument("--out", default=None, help="JSON file to write (default: print only)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_csm.py needs a CUDA device")
    stream = torch.cuda.current_stream()
    g = torch.Generator(device="cuda").manual_seed(1)
    base = (torch.rand(SAMPLES, device="cuda", generator=g) - 0.5) * (12 ** 0.5)
    xs = [(0.6 * base + (torch.rand(SAMPLES, device="cuda", generator=g) - 0.5) * (12 ** 0.5)).contiguous()
          for _ in range(4)]
    del base
    res = dict(gpu_info(), samples_per_channel_per_step=SAMPLES, channels=4, steps=a.steps, warmup=a.warmup,
               results={})
    for n in [int(v) for v in a.sizes.split(",")]:
        runs = {k: [] for k in SETUPS}
        for _ in range(a.rounds):
            for setup in runs:
                runs[setup].append(run(setup, n, xs, a.steps, a.warmup, stream))
        r = {k: {"input_samples_per_s_median": sorted(v)[len(v) // 2], "runs": v} for k, v in runs.items()}
        r["csm4_kernel_ms_one_step"] = kernel_times(n, xs, stream)
        res["results"][str(n)] = r
        print(json.dumps({"n": n, **{k: round(sorted(v)[len(v) // 2] / 1e9, 1) for k, v in runs.items()},
                          "kernel_ms": r["csm4_kernel_ms_one_step"]}), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
