#!/usr/bin/env python3
"""Throughput of the cross-spectral density (CsdCascade) against two PsdCascades on the same data.

Two device-resident channels of 200e6 samples each are fed per step (the size of bench.py's steps), at N = 512 and
4096, Hann window, default options, one readout at the end of the timed window.  Reported: input samples per second
with both channels counted, for
  csd      CsdCascade(N).process(x, y)
  psd2     two default PsdCascade(N) (ring / w16 kernels), x and y
  psd2_r8  two PsdCascade(N) created with SSPSD_K2=r8: the generic tiled kernel family the CSD kernel is built on
The setups alternate over `--rounds` rounds so that the spread shows.  CUDA events on the handles' shared stream.

    python tools/bench_csd.py --out profiles/r04_csd_bench.json
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from stabilizer_stream_b200 import CsdCascade, MergeOpts, PsdCascade  # noqa: E402

SAMPLES = 200_000_000


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
    if setup == "csd":
        return [CsdCascade(n, stream=s)]
    if setup == "psd2_r8":
        os.environ["SSPSD_K2"] = "r8"  # read when a handle is created
        try:
            return [PsdCascade(n, stream=s), PsdCascade(n, stream=s)]
        finally:
            del os.environ["SSPSD_K2"]
    return [PsdCascade(n, stream=s), PsdCascade(n, stream=s)]


def step(handles, x, y):
    if len(handles) == 1:
        handles[0].process(x, y)
    else:
        handles[0].process(x)
        handles[1].process(y)


def readout(handles):
    for h in handles:
        (h.csd if isinstance(h, CsdCascade) else h.psd)(MergeOpts())


def run(setup, n, x, y, steps, warmup, stream):
    handles = make(setup, n, stream)
    for _ in range(warmup):
        step(handles, x, y)
    readout(handles)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        step(handles, x, y)
    readout(handles)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    return 2.0 * SAMPLES * steps / (ms * 1e-3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--sizes", default="512,4096")
    ap.add_argument("--out", default=None, help="JSON file to write (default: print only)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_csd.py needs a CUDA device")
    stream = torch.cuda.current_stream()
    g = torch.Generator(device="cuda").manual_seed(1)
    x = (torch.rand(SAMPLES, device="cuda", generator=g) - 0.5) * (12 ** 0.5)
    y = (0.6 * x + (torch.rand(SAMPLES, device="cuda", generator=g) - 0.5) * (12 ** 0.5)).contiguous()
    res = dict(gpu_info(), samples_per_channel_per_step=SAMPLES, steps=a.steps, warmup=a.warmup, results={})
    for n in [int(v) for v in a.sizes.split(",")]:
        runs = {k: [] for k in ("csd", "psd2", "psd2_r8")}
        for _ in range(a.rounds):
            for setup in runs:
                runs[setup].append(run(setup, n, x, y, a.steps, a.warmup, stream))
        res["results"][str(n)] = {k: {"input_samples_per_s_median": sorted(v)[len(v) // 2], "runs": v}
                                  for k, v in runs.items()}
        print(json.dumps({"n": n, **{k: round(sorted(v)[len(v) // 2] / 1e9, 1) for k, v in runs.items()}}), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
