#!/usr/bin/env python3
"""Plants (sspsd_plant_*, DESIGN.md 3d): generation rate, the cost of feeding the cross-spectral handles from a plant
instead of from device-resident arrays, and time-chunked CSM groups fed by time_process_plant.

  (a) generate  Plant(K, M, L).generate into preallocated device buffers, (K, M, L) = (2, 2, 8), (4, 2, 32), (4, 4, 32):
                G positions/s, output bytes/s against a device-to-device copy of the same bytes, and the f64 FMA rate
                (K M L per position)
  (b) consumers CsdCascade(N), CsmCascade(N, 4), ZoomCascade I/Q and heterodyne at N = 512 and 4096, fed 2^30 positions
                by process_plant against the same handles fed the same positions from device arrays (generated before
                the clock starts, as r04 / r05 / r07 did); the plant's share of device time from torch.profiler in a
                separate pass
  (c) groups    CSM K = 4, N = 4096: a 4.8e9-sample capture generated inside the timed window by time_process_plant,
                wall time from plan to rank 0's csm(), on W ranks sharing GPU 0 and on W GPUs where the box has them
Rounds alternate the setups; the median of 3 is reported.  The card's name and power limit are read in the same run.

    python tools/bench_plant.py --out profiles/r09_plant_bench.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import stabilizer_stream_b200 as sp  # noqa: E402

FTW = 0x9E3779B9


def gpu_info():
    info = {"device": torch.cuda.get_device_name(0), "gpus": torch.cuda.device_count()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["name_power_limit_max_sm_clock"] = q
    except OSError:
        info["name_power_limit_max_sm_clock"] = None
    return info


def plant(k, m, nt):
    taps = np.random.default_rng(k * 100 + m * 10 + nt).standard_normal((k, m, nt)).astype(np.float32)
    return sp.Plant(taps, [sp.Plant.noise(q % 2, 1000 + q) for q in range(m)])


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def median(xs):
    return float(np.median(xs))


def bench_generate(rounds):
    n = 1 << 26
    out = torch.empty((4, n), dtype=torch.float32, device="cuda:0")
    src = torch.empty(4 * n, dtype=torch.float32, device="cuda:0")
    dst = torch.empty_like(src)
    shapes = [(2, 2, 8), (4, 2, 32), (4, 4, 32)]
    ps = {s: plant(*s) for s in shapes}
    for s in shapes:
        ps[s].generate(n, out=out[:s[0]])
    dst.copy_(src)
    times = {s: [] for s in shapes}
    copy = []
    reps = 8
    for _ in range(rounds):
        for s in shapes:
            times[s].append(timed(lambda: [ps[s].generate(n, out=out[:s[0]]) for _ in range(reps)]) / reps)
        copy.append(timed(lambda: [dst.copy_(src) for _ in range(reps)]) / reps)
    copy_bps = 2 * 4 * 4 * n / median(copy)   # read + write bytes of a device-to-device copy
    rows = []
    for s in shapes:
        t = median(times[s])
        k, m, nt = s
        rows.append({"K": k, "M": m, "L": nt, "G_positions_per_s": n / t / 1e9,
                     "output_GB_per_s": 4 * k * n / t / 1e9,
                     "output_share_of_copy_peak": 4 * k * n / t / copy_bps,
                     "f64_TFMA_per_s": k * m * nt * n / t / 1e12, "ms": 1e3 * t})
    return {"positions": n, "rows": rows, "copy_read_plus_write_GB_per_s": copy_bps / 1e9}


def handle(kind, n):
    if kind == "csd":
        return sp.CsdCascade(n), 2
    if kind == "csm4":
        return sp.CsmCascade(n, 4), 4
    if kind == "zoom_iq":
        return sp.ZoomCascade.iq(n), 2
    return sp.ZoomCascade.heterodyne(n, FTW), 1


def feed_arrays(h, kind, y):
    if kind == "csm4":
        h.process(list(y))
    elif y.shape[0] == 2:
        h.process(y[0], y[1])
    else:
        h.process(y[0])


def bench_consumers(rounds, total):
    rows = []
    for n in (512, 4096):
        for kind in ("csd", "csm4", "zoom_iq", "zoom_het"):
            _, k = handle(kind, n)
            p = plant(k, 2, 8)
            y = p.generate(total).clone()
            tp, ta = [], []
            for _ in range(rounds):
                h, _ = handle(kind, n)
                p.reset()
                tp.append(timed(lambda: (h.process_plant(p, total), h.sync())))
                h, _ = handle(kind, n)
                ta.append(timed(lambda: (feed_arrays(h, kind, y), h.sync())))
            del y
            share = plant_share(kind, n, k, total)
            rows.append({"kind": kind, "N": n, "K": k, "positions": total,
                         "plant_GS_per_s": total / median(tp) / 1e9, "arrays_GS_per_s": total / median(ta) / 1e9,
                         "plant_share_of_device_time": share})
            torch.cuda.empty_cache()
    return rows


def plant_share(kind, n, k, total):
    """torch.profiler pass of its own: plant_kernel's share of the CUDA kernel time of one process_plant"""
    from torch.profiler import ProfilerActivity, profile
    h, _ = handle(kind, n)
    p = plant(k, 2, 8)
    h.process_plant(p, 1 << 24)
    h.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        h.process_plant(p, total)
        h.sync()
    tot = mine = 0.0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
        tot += t
        if "plant_kernel" in e.key:
            mine += t
    return mine / tot if tot else None


def bench_groups(rounds, total):
    n = 4096
    p = plant(4, 2, 8)
    setups = [("shared", [0] * w) for w in (1, 2, 4)]
    g_avail = torch.cuda.device_count()
    for w in (2, 4, 8):
        if g_avail >= w:
            setups.append(("gpus", list(range(w))))
    times = {i: [] for i in range(len(setups))}
    groups = [sp.Group(n, devices=d, mode=sp.ShardMode.TIME, kind=sp.GroupKind.CSM, channels=4) for _, d in setups]
    for _ in range(rounds):
        for i, g in enumerate(groups):
            def run():
                g.time_plan(total)
                g.time_process_plant(p)
                g.time_finish()
                g.csm()
            times[i].append(timed(run))
    rows = [{"setup": s, "devices": d, "ranks": len(d), "seconds": median(times[i]),
             "GS_per_s": total / median(times[i]) / 1e9} for i, (s, d) in enumerate(setups)]
    for w in (2, 4, 8):
        if g_avail < w:
            rows.append({"setup": "gpus", "ranks": w, "seconds": "not measured (%d GPU(s) on the box)" % g_avail})
    return {"N": n, "K": 4, "samples": total, "rows": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--consumer-positions", type=int, default=1 << 30)
    ap.add_argument("--group-samples", type=float, default=4.8e9)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = {"gpu": gpu_info(), "rounds": a.rounds, "median_of": a.rounds}
    res["generate"] = bench_generate(a.rounds)
    print(json.dumps(res["generate"]), flush=True)
    res["consumers"] = bench_consumers(a.rounds, a.consumer_positions)
    print(json.dumps(res["consumers"]), flush=True)
    res["groups"] = bench_groups(a.rounds, int(a.group_samples))
    print(json.dumps(res["groups"]), flush=True)
    out = a.out or os.path.join(tempfile.gettempdir(), "r09_plant_bench.json")
    with open(out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", out)


if __name__ == "__main__":
    main()
