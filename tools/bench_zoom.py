#!/usr/bin/env python3
"""Throughput of the two-sided spectrum (ZoomCascade) against CsdCascade, the mixer's share in heterodyne mode, and the
image floor that a two-sided spectrum assembled from CsdCascade's rows reaches.

  iq          ZoomCascade.iq(N).process(i, q) on two device-resident 200e6-sample channels (both counted)
  csd         CsdCascade(N).process(i, q) on the same channels (the same transform with the CSD's epilogue)
  heterodyne  ZoomCascade.heterodyne(N, ftw).process(x) on one 200e6-sample channel (input samples counted)
N = 512 and 4096, Hann window, default options, one readout at the end of the timed window; the setups alternate over
`--rounds` rounds and the median is reported.  CUDA events on the handles' shared stream.  A separate pass under
torch.profiler gives the mixer kernel's share of the device time of one heterodyne step.

The image case is tests/test_gpu_zoom.py's: a unit complex exponential at +3.37 bins of stage 2 (N = 512) over white
noise at 1e-5, 2^21 samples.  For p_neg = |Z[N-k]|^2 from ZoomCascade and from CsdCascade's (pxx + pyy + 2 Im pxy) / 2
it records the largest deviation from the float64 model over the merged row, relative to the tone's peak.

    python tools/bench_zoom.py --out profiles/r07_zoom_bench.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from stabilizer_stream_b200 import CsdCascade, MergeOpts, ZoomCascade  # noqa: E402

SAMPLES = 200_000_000
FTW = 0x1F9ADD37


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
    if setup == "iq":
        return ZoomCascade.iq(n, stream=s)
    if setup == "csd":
        return CsdCascade(n, stream=s)
    return ZoomCascade.heterodyne(n, FTW, stream=s)


def step(h, setup, x, y):
    if setup == "heterodyne":
        h.process(x)
    else:
        h.process(x, y)


def readout(h):
    (h.csd if isinstance(h, CsdCascade) else h.spectrum)(MergeOpts())


def run(setup, n, x, y, steps, warmup, stream):
    h = make(setup, n, stream)
    for _ in range(warmup):
        step(h, setup, x, y)
    readout(h)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        step(h, setup, x, y)
    readout(h)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    return (1.0 if setup == "heterodyne" else 2.0) * SAMPLES * steps / (ms * 1e-3)


def mixer_share(n, x, stream):
    from torch.profiler import ProfilerActivity, profile
    h = make("heterodyne", n, stream)
    step(h, "heterodyne", x, None)
    h.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step(h, "heterodyne", x, None)
        h.sync()
    per = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t:
            per[e.key] = per.get(e.key, 0.0) + t
    total = sum(per.values())
    mix = sum(v for k, v in per.items() if "heterodyne_kernel" in k)
    top = sorted(per.items(), key=lambda kv: -kv[1])[:6]
    return {"mixer_us": mix, "device_us": total, "mixer_share": mix / total if total else None,
            "top_kernels_us": {k[:80]: v for k, v in top}}


def image_case():
    from oracle import model_f64_zoom as mz
    n, m = 512, 1 << 21
    t = np.arange(m, dtype=np.float64)
    z = np.exp(2j * np.pi * (3.37 / (n * 64)) * t)
    rng = np.random.default_rng(1)
    i = (z.real + 1e-5 * (rng.random(m) - 0.5) * 12 ** 0.5).astype(np.float32)
    q = (z.imag + 1e-5 * (rng.random(m) - 0.5) * 12 ** 0.5).astype(np.float32)
    c = ZoomCascade.iq(n)
    c.process(i, q)
    pp, pn, b = c.spectrum()
    d = CsdCascade(n)
    d.process(i, q)
    pxx, pyy, pxy, _ = d.csd()
    tp, tn, _ = mz.merge_zoom(mz.zoom_cascade(i, q, n), n)
    from_csd = (pxx.astype(np.float64) + pyy + 2 * pxy.imag) / 2
    peak = float(np.max(tp))
    out = {}
    for name, row in (("zoom_kernel", pn.astype(np.float64)), ("csd_rows", from_csd)):
        err = np.abs(row - tn)
        out[name] = {"max_abs_err_rel_peak_db": float(10 * np.log10(np.max(err) / peak)),
                     "median_abs_err_rel_peak_db": float(10 * np.log10(np.median(err) / peak + 1e-300))}
    out["truth_image_floor_rel_peak_db"] = float(10 * np.log10(np.median(tn) / peak))
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
        sys.exit("bench_zoom.py needs a CUDA device")
    stream = torch.cuda.current_stream()
    g = torch.Generator(device="cuda").manual_seed(1)
    x = (torch.rand(SAMPLES, device="cuda", generator=g) - 0.5) * (12 ** 0.5)
    y = (0.6 * x + (torch.rand(SAMPLES, device="cuda", generator=g) - 0.5) * (12 ** 0.5)).contiguous()
    res = dict(gpu_info(), samples_per_channel_per_step=SAMPLES, steps=a.steps, warmup=a.warmup, ftw=FTW,
               results={})
    for n in [int(v) for v in a.sizes.split(",")]:
        runs = {k: [] for k in ("iq", "csd", "heterodyne")}
        for _ in range(a.rounds):
            for setup in runs:
                runs[setup].append(run(setup, n, x, y, a.steps, a.warmup, stream))
        r = {k: {"input_samples_per_s_median": sorted(v)[len(v) // 2], "runs": v} for k, v in runs.items()}
        r["heterodyne_profile"] = mixer_share(n, x, stream)
        res["results"][str(n)] = r
        print(json.dumps({"n": n, **{k: round(sorted(v)[len(v) // 2] / 1e9, 1) for k, v in runs.items()},
                          "mixer_share": r["heterodyne_profile"]["mixer_share"]}), flush=True)
    res["image_case"] = image_case()
    print(json.dumps({"image_case": res["image_case"]}), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
