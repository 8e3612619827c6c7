#!/usr/bin/env python3
"""Time-chunked CSM groups (Group(kind=GroupKind.CSM)) against the plain CsmCascade on the same capture.

One capture of four device-resident channels of `--samples` samples each (default 1e9), N = 4096, Hann window, default
options.  Reported, as input samples per second with the four channels counted once, and as wall time from the first
sample fed to the readout available on rank 0:
  (a) handle   CsmCascade(N, 4).process(x) and one csm() readout
      group1   a one-rank group on the same GPU: plan, feed, time_finish, csm()
  (b) shared W W ranks on GPU 0 (the direct reduction): the halo's recompute and time_finish's own time
  (c) gpus W   W = 2, 4, 8 ranks on as many GPUs (NCCL), each rank's range resident on its GPU before the clock
               starts, all ranks fed asynchronously; "not measured" where the box has fewer GPUs
The halo overhead sum(feed_hi - feed_lo) / total comes from the group's plan.  Rounds alternate the setups so that
the spread shows; the median is reported.  The card's name and power limit are read in the same run.

    python tools/bench_xgroup.py --out profiles/r08_xgroup_bench.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import stabilizer_stream_b200 as sp  # noqa: E402
from stabilizer_stream_b200 import _lib as L  # noqa: E402

N, K = 4096, 4


def gpu_info():
    info = {"device": torch.cuda.get_device_name(0), "gpus": torch.cuda.device_count()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["name_power_limit_max_sm_clock"] = q
    except OSError:
        info["name_power_limit_max_sm_clock"] = None
    return info


def run_handle(xs):
    c = sp.CsmCascade(N, K)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    c.process(xs)
    s, _ = c.csm()
    return time.perf_counter() - t0, s


def run_group(xs_of_rank, devs, total):
    """xs_of_rank[r]: rank r's K streams [feed_lo, feed_hi) on devs[r] -> (wall s, time_finish s, S, halo ratio)"""
    g = sp.Group(N, devices=devs, mode=sp.ShardMode.TIME, kind=sp.GroupKind.CSM, channels=K)
    g.time_plan(total)
    chunks = [g.time_chunk(r) for r in range(len(devs))]
    halo = sum(c.feed_hi - c.feed_lo for c in chunks) / total
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for r, c in enumerate(chunks):
        xs = xs_of_rank(r, c)
        ptrs = (C.c_void_p * K)(*[x.data_ptr() for x in xs])
        # asynchronous on the rank's stream: the ranks of several GPUs run at once
        L.check(L.lib().sspsd_group_time_process_multi_f32(g._h, r, ptrs, c.feed_hi - c.feed_lo, L.MEM_DEVICE))
    g.sync()
    t1 = time.perf_counter()
    g.time_finish()
    s, _ = g.csm()
    t2 = time.perf_counter()
    return t2 - t0, t2 - t1, s, halo, chunks[0].n_local


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=float, default=1e9)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--shared", default="2,4,8")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    total = int(args.samples)
    ngpu = torch.cuda.device_count()
    g = torch.Generator(device="cuda:0").manual_seed(7)
    x0 = torch.rand(total, device="cuda:0", generator=g) - 0.5
    xs = [x0] + [(0.5 * x0 + torch.rand(total, device="cuda:0", generator=g) - 0.5) for _ in range(K - 1)]
    on0 = lambda r, c: [x[c.feed_lo:c.feed_hi] for x in xs]  # noqa: E731
    setups = {"group1": ([0], on0)}
    for w in [int(v) for v in args.shared.split(",") if v]:
        setups["shared%d" % w] = ([0] * w, on0)
    multi = {}
    for w in (2, 4, 8):
        if ngpu < w:
            multi["gpus%d" % w] = "not measured (the box has %d GPU%s)" % (ngpu, "s" if ngpu > 1 else "")
            continue
        # each rank's range copied to its GPU once, before any clock starts
        plan = [sp.time_plan(N, total, w, r) for r in range(w)]
        local = [[x[c.feed_lo:c.feed_hi].to("cuda:%d" % r) for x in xs] for r, c in enumerate(plan)]
        setups["gpus%d" % w] = (list(range(w)), lambda r, c, local=local: local[r])
    res = {k: {"wall_s": [], "finish_s": []} for k in ["handle"] + list(setups)}
    ref = None
    for _ in range(args.rounds):
        t, ref = run_handle(xs)
        res["handle"]["wall_s"].append(t)
        for name, (devs, fn) in setups.items():
            t, tf, s, halo, nl = run_group(fn, devs, total)
            r = res[name]
            r["wall_s"].append(t)
            r["finish_s"].append(tf)
            r["halo_ratio"], r["n_local"] = halo, nl
            d = np.real(np.einsum("iib->ib", ref)).astype(np.float64)
            scale = np.sqrt(d[:, None, :] * d[None, :, :])
            r["max_dev_vs_handle"] = float(np.max(np.abs(s.astype(np.complex128) - ref)[..., 2:] / scale[..., 2:]))
    out = {"what": "time-chunked CSM group vs CsmCascade", "n_fft": N, "channels": K, "samples_per_channel": total,
           "window": "hann", "input": "device-resident, torch.rand", "rounds": args.rounds, **gpu_info()}
    for name, r in res.items():
        w = float(np.median(r["wall_s"]))
        r["median_wall_s"] = w
        r["gsps_per_channel"] = total / w / 1e9
        if r["finish_s"]:
            r["median_finish_s"] = float(np.median(r["finish_s"]))
        else:
            del r["finish_s"]
        out[name] = r
    out.update(multi)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
