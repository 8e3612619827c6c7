#!/usr/bin/env python3
"""Benchmark of the cascaded-PSD hot path (BASELINE.json metric: sustained MS/s through the full
PSD cascade; % of HBM roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[1] -- default PsdCascade (N=4096 Hann, 50 % overlap,
divide-by-8 half-band cascade per stage) over one second of a 200 MS/s synthetic raw f32 stream.
A step = one pass of the whole cascade over 200e6 samples.  `value` times K back-to-back steps plus ONE
psd() readout at the end (SURVEY.md 8d: "process + final psd() readout, steady state"; the reference's GUI
reads out at frame rate, not per batch); `value_readout_every_step` is the same loop with a psd() readout
after every step, `sustained_2s` the same loop run for at least two seconds.  With N GPUs every
rank runs its own channel of the same shape (channels are independent cascades, reference
src/bin/psd.rs:174-182): weak scaling, no data-path collective, one NCCL gather of the merged
spectra at readout.

`value` is measured with the input resident in HBM (800 MB per step, far larger than the 126 MB L2,
so nothing is served from cache between steps); `e2e` is the same metric through the same C-ABI
call with the samples in pinned HOST memory (H2D inside the timed region) and the spectra read back.
`--impl reference` times the CPU restatement of the reference (oracle/, kind "port": the Rust
reference cannot be built offline) on the box's host cores.

`--dump-outputs DIR` writes, after all timed runs, the psd() readout that ends the headline loop as
the caller receives it, per channel c: `psd_ch<c>.npy` (float32 spectrum) and `breaks_ch<c>.npy`
(float64, one row per stage, columns BREAK_FIELDS).  The input is seeded, so two builds run with
the same arguments can be compared output for output.  The benchmark writes nothing into the tree.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only; leave no __pycache__ in it either

N_FFT = 4096
SAMPLES_PER_STEP = 200_000_000
BYTES_PER_SAMPLE = 4.0  # algorithmic: every raw f32 sample must cross HBM once (SURVEY.md 8d)
# measured DRAM traffic of the stage-0 PSD kernel: dram__bytes_read.sum + dram__bytes_write.sum = 270.96 MB +
# 3.82 MB for a 2^26-sample launch (ncu --set full, profiles/r02_ncu_final_k2ring_k3tma_metrics.csv)
TRAFFIC_BYTES_PER_SAMPLE = (270.964224e6 + 3.822336e6) / (1 << 26)
# FP32 lane operations the stage-0 PSD kernel executes per input sample (ncu instruction mix of the final kernel,
# profiles/r01_ncu_ring_packed_instruction_mix.csv: 2 x 43.41 M packed + 15.44 M scalar FP warp instructions for
# 2^26 samples): the roof that actually bounds it -- explanatory, next to the contract's HBM roofline
FP32_LANE_OPS_PER_SAMPLE = (2 * 43.41e6 + 15.44e6) * 32 / (1 << 26)
WORKLOAD = "PsdCascade N=4096 Hann 50% overlap, div-8 half-band per stage, 200e6-sample f32 stream per channel"
STAGE_COUNTS_PER_STEP = [97655, 12205, 1524, 189, 22, 1, 0]  # closed form (SURVEY.md a9) for one 200e6-sample step
PARITY_NOTE = ("idsp 0.20 hbf (taps, FIR phase, hbf_dec_response_length) is not on disk: decimator parity is against the "
               "restatement in oracle/, unpinned against the real crate; the CPU arm is that restatement (kind=port), not "
               "rustfft/idsp")


def config_dict(n):
    """Identical in both arms (the driver compares them): describes the workload only, no measured values."""
    return {"workload": WORKLOAD, "n_fft": N_FFT, "channels": n, "samples_per_step_per_gpu": SAMPLES_PER_STEP,
            "stage_counts_per_step": STAGE_COUNTS_PER_STEP,
            "readout": "one psd() readout at the end of the timed region"}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (NVML polled from a thread every
    ~2 ms; the timed region is tens of milliseconds, too short for `nvidia-smi -lms`)."""

    def __init__(self, index, power=False):
        self.index = index
        self.power = [] if power else None
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None
        self._err = None

    def _run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                     "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                     "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                nv.nvmlDeviceGetCurrentClocksThrottleReasons
            while not self._stop.is_set():
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                if self.power is not None:
                    self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
                r = get_reasons(h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
                time.sleep(0.002)
            nv.nvmlShutdown()
        except Exception as e:  # noqa: BLE001
            self._err = repr(e)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        time.sleep(0.01)

    def stop(self):
        self._stop.set()
        if self._t is not None:
            self._t.join(timeout=2.0)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["no samples: %s" % self._err]}
        sm = sorted(self.samples)
        out = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
               "samples": len(sm)}
        if self.power:
            out["sm_mhz_min"] = sm[0]
            out["power_w_max"] = max(self.power)
            out["power_w_median"] = sorted(self.power)[len(self.power) // 2]
        return out


def _cpu_feed(cas, block, samples):
    """feed exactly `samples` samples by cycling over a 2^22-sample block (ctypes releases the GIL)"""
    pos = 0
    while pos < samples:
        n = min(block.size, samples - pos)
        cas.process(block[:n])
        pos += n


def _cpu_block():
    import numpy as np
    rng = np.random.default_rng(0x7654321)
    return ((rng.random(1 << 22, dtype=np.float32) - np.float32(0.5)) * np.float32(12 ** 0.5)).astype(np.float32)


def cpu_run(samples_per_step, steps, warmup, threads=1, n_fft=N_FFT):
    """The CPU restatement (oracle) on this host: `threads` independent channels, one cascade per thread, each
    processing steps x samples_per_step samples + one psd() readout -- the same loop the GPU arm times."""
    from oracle import binding as orc
    orc.lib()
    block = _cpu_block()
    cas = [orc.Cascade(n_fft, orc.HBF_140) for _ in range(threads)]

    def work(i, k):
        for _ in range(k):
            _cpu_feed(cas[i], block, samples_per_step)
        cas[i].psd()

    def run(k):
        ths = [threading.Thread(target=work, args=(i, k)) for i in range(threads)]
        t0 = time.perf_counter()
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        return time.perf_counter() - t0

    if warmup:
        run(warmup)
    dt = run(steps)
    total = threads * steps * samples_per_step
    return {"value": total / dt / 1e6, "unit": "MS/s", "cores": threads, "kind": "port",
            "sample": "%d channel(s) x %d step(s) x %d samples (N=%d cascade, CPU restatement of src/psd.rs, gcc -O3 "
                      "-march=native; the Rust reference cannot be built offline; it publishes >200 MS/s/core at N=512)"
                      % (threads, steps, samples_per_step, n_fft), "seconds": dt}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = max(1, args.gpus)
    # the reference runs one cascade per trace on one receiver thread; with N channels it can use N threads
    threads = min(n, os.cpu_count() or 1)
    # (SSPSD_BENCH_CPU_SAMPLES shortens the step for the CPU-only smoke test of this arm; the driver never sets it)
    per_step = int(os.environ.get("SSPSD_BENCH_CPU_SAMPLES", SAMPLES_PER_STEP))
    cb = cpu_run(per_step, args.steps, min(args.warmup, 1), threads)
    v = cb["value"] * n / threads  # (threads == n unless the host has fewer cores than channels)
    cfg = config_dict(n)
    out = {"impl": "reference", "metric": "sustained MS/s through full PSD cascade", "value": v, "unit": "MS/s",
           "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": cb["seconds"] / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
           "cpu_baseline": cb, "parity_note": PARITY_NOTE,
           "e2e": {"value": v, "unit": "MS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)


def bind_to_gpu_numa_node(index):
    """Pin this rank's threads to the CPUs of its GPU's NUMA node BEFORE any pinned host buffer is allocated, so
    that the staging memory of the end-to-end path is first-touched next to the GPU's PCIe root (round 1: eight
    ranks allocating from one node shared 184 GB/s; VERDICT r01 weak #9).  Returns a description for the record."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        bus = nv.nvmlDeviceGetPciInfo(nv.nvmlDeviceGetHandleByIndex(index)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return {"numa_node": node, "bound": False, "why": "no NUMA information for the device"}
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if not allowed:
            return {"numa_node": node, "bound": False, "why": "node's CPUs are outside this process's cpuset"}
        os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "bound": True, "cpus": len(allowed)}
    except Exception as e:  # noqa: BLE001
        return {"bound": False, "why": repr(e)}


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from stabilizer_stream_b200 import Group, MergeOpts, ShardMode, _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa = bind_to_gpu_numa_node(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    stream = torch.cuda.current_stream(dev)

    # The multi-GPU plumbing lives in the library: every rank joins one sspsd_group (ncclCommInitRank inside
    # libsspsd.so; torch.distributed only hands the 128-byte id around and provides the barrier of the contract).
    def new_group(mode=ShardMode.CHANNELS):
        ids = [Group.unique_id() if (rank == 0 and world > 1) else None]  # a fresh NCCL id per communicator
        if world > 1:
            dist.broadcast_object_list(ids, src=0)
        return Group(N_FFT, rank=rank, n_ranks=world, unique_id=ids[0], device=local, mode=mode,
                     stream=stream.cuda_stream or 1)

    gen = torch.Generator(device=dev).manual_seed(0x7654321 + rank)
    x = (torch.rand(SAMPLES_PER_STEP, device=dev, generator=gen) - 0.5) * (12 ** 0.5)
    xh = torch.empty(SAMPLES_PER_STEP, dtype=torch.float32, pin_memory=True)
    xh.copy_(x)
    torch.cuda.synchronize(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    class Channel:
        """this rank's channel (= trace `rank` of the job) of a channel-sharded group"""

        def __init__(self):
            self.g = new_group()
            self.g.process_raw(rank, x.data_ptr(), 4 * N_FFT, _lib.MEM_DEVICE)  # creates the channel's cascade
            self.c = self.g.channel_cascade(rank)
            self.c.reset()

        def process(self, src):
            if src is x:
                self.g.process_raw(rank, x.data_ptr(), SAMPLES_PER_STEP, _lib.MEM_DEVICE)
            else:
                self.g.process_raw(rank, xh.data_ptr(), SAMPLES_PER_STEP, _lib.MEM_HOST)

        def readout(self):
            """psd() of every channel of the job on rank 0: ONE ncclAllGather of accumulator rows + bookkeeping"""
            return self.g.psd_all(world, MergeOpts())

    def timed(ch, src, steps, warmup):
        for _ in range(warmup):
            ch.process(src)
            ch.readout()
        ch.c.profile_read()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            ch.process(src)
            res = ch.readout()
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), res

    # ---- device-resident run (value) with per-kernel event timing and clock sampling ----
    # Timed region: K back-to-back process() calls on the resident 200e6-sample buffer + ONE final
    # psd() readout (SURVEY.md 8d: "process + final psd() readout, steady state"; the reference's GUI
    # reads out at frame rate, i.e. every few 1e6 samples of a 200 MS/s stream, not every batch).
    # `value_readout_every_step` repeats the measurement with a psd() readout after every step.
    def device_run(readout_every_step, profile=False):
        ch = Channel()
        ch.c.profile_enable(profile)
        for _ in range(args.warmup):
            ch.process(x)
            ch.readout()
        ch.c.profile_read()
        barrier()
        # clocks are sampled during the headline run; the NVML polling thread of 8 ranks costs the
        # readout-every-step loop 5-15 % (tools/readout_probe.py), so that run goes without it
        sampler = ClockSampler(local)
        if not readout_every_step:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            ch.process(x)
            if readout_every_step:
                res = ch.readout()
        if not readout_every_step:
            res = ch.readout()
        e1.record(stream)
        barrier()
        clocks = sampler.stop() if not readout_every_step else None
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        prof, launches = ch.c.profile_read()
        return float(ms.item()), prof, launches, clocks, res

    ms_rs, _, _, _, _ = device_run(True)
    ms, _, launches, clocks, readout = device_run(False)
    # the same loop once more with every kernel launch bracketed by CUDA events (per-kernel times for the roofline;
    # the event records cost a few percent, so the headline comes from the unprofiled run above)
    ms_prof, prof, _, _, _ = device_run(False, profile=True)
    value = world * SAMPLES_PER_STEP * args.steps / (ms * 1e-3) / 1e6
    value_rs = world * SAMPLES_PER_STEP * args.steps / (ms_rs * 1e-3) / 1e6

    # ---- sustained: the same loop for >= 2 s of device time (SURVEY.md 8d), clocks + power sampled throughout ----
    def sustained(seconds=2.0):
        c = Channel()
        for _ in range(3):
            c.process(x)
        c.readout()
        barrier()
        k = max(args.steps, int(seconds / (ms / args.steps * 1e-3)) + 1)
        sampler = ClockSampler(local, power=True)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(k):
            c.process(x)
            if i % 64 == 63:
                c.g.sync()  # bound the launch queue; a sync every 64 steps (56 ms) costs nothing measurable
        c.readout()
        e1.record(stream)
        barrier()
        ck = sampler.stop()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t = float(t.item())
        return {"value": world * SAMPLES_PER_STEP * k / (t * 1e-3) / 1e6, "unit": "MS/s", "steps": k, "seconds": t * 1e-3,
                "clocks": ck}

    sus = sustained()
    tc = timechunk_record(new_group, barrier, rank, world, dist, dev)

    # ---- end-to-end run: host pinned input, H2D inside the timed region, spectra read back ----
    c2 = Channel()
    e2e_steps = max(1, min(args.steps, 5))
    ms2, _ = timed(c2, xh, e2e_steps, min(args.warmup, 2))
    e2e_value = world * SAMPLES_PER_STEP * e2e_steps / (ms2 * 1e-3) / 1e6

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_kind = peaks()
    k_ms, k_launches, k_units = prof["psd_stage0"]
    achieved = (BYTES_PER_SAMPLE * k_units / (k_ms * 1e-3) / 1e9) if k_ms > 0 else 0.0
    roof = {"bound": "hbm", "kernel": "psd_stage_kernel_ring (stage 0, N=4096)", "achieved": achieved, "peak": peak,
            "peak_kind": peak_kind, "unit": "GB/s", "frac": achieved / peak,
            "traffic": TRAFFIC_BYTES_PER_SAMPLE * k_units / max(k_launches, 1),
            "traffic_source": "ncu --set full, profiles/r02_ncu_final_k2ring_k3tma_metrics.csv, scaled per sample",
            "fp32_pipe": {"lane_ops_per_sample": FP32_LANE_OPS_PER_SAMPLE,
                          "achieved_Tops": FP32_LANE_OPS_PER_SAMPLE * k_units / (k_ms * 1e-3) / 1e12 if k_ms > 0 else 0.0,
                          "peak_Tops": 148 * 128 * (clocks.get("sm_max_mhz") or 1965.0) * 1e6 / 1e12,
                          "note": "explanatory: the kernel is FP32 / latency bound, not HBM bound"},
            "launches": int(k_launches), "avg_launch_ms": (k_ms / k_launches) if k_launches else None,
            "algorithmic_bytes_per_launch": BYTES_PER_SAMPLE * k_units / max(k_launches, 1),
            "share_of_step": k_ms / ms_prof, "profiled_ms_per_step": ms_prof / args.steps,
            "other_kernels_ms": {k: v[0] for k, v in prof.items() if k != "psd_stage0"},
            "whole_step_frac": BYTES_PER_SAMPLE * SAMPLES_PER_STEP * args.steps / (ms * 1e-3) / 1e9 / peak}
    d2h = sum(len(k.bins) for k in readout[0][1] if k.include) * 4
    out = {"metric": "sustained MS/s through full PSD cascade", "value": value, "unit": "MS/s", "n_gpus": world,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": config_dict(world),
           "cache": "inputs (800 MB per step) larger than the 126 MB L2",
           "value_readout_every_step": value_rs, "sustained_2s": sus, "timechunk": tc,
           "readout_collective": "one ncclAllGather of accumulator rows + bookkeeping inside libsspsd.so (sspsd_group_psd_all)",
           "roofline": roof, "clocks": clocks, "gpu_launches": int(launches), "parity_note": PARITY_NOTE,
           "e2e": {"value": e2e_value, "unit": "MS/s", "h2d_bytes_per_step": SAMPLES_PER_STEP * 4 * world,
                   "d2h_bytes_per_step": d2h * world, "steps": e2e_steps, "ms_per_step": ms2 / e2e_steps,
                   "h2d_GBps_per_gpu": SAMPLES_PER_STEP * 4 / (ms2 / e2e_steps * 1e-3) / 1e9, "numa_rank0": numa}}
    if world == 1:
        # CPU arm beside it: one bounded step of the same workload on one host core, and the reference's own
        # in-tree size N=512 next to its published ">200 MS/s per core" (README.md:11, src/psd.rs:550)
        out["cpu_baseline"] = cpu_run(SAMPLES_PER_STEP, 8, 1, 1)
        n512 = cpu_run(100_000_000, 3, 1, 1, n_fft=512)
        n512["published"] = ">200 MS/s on one (Skylake) core at N=512 (reference README.md:11, src/psd.rs:550)"
        out["cpu_baseline_n512"] = n512
        out["e2e_small_calls"] = small_calls()
        out["e2e_frames"] = e2e_frames(local)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, readout)
    emit(out)
    if world > 1:
        dist.destroy_process_group()


BREAK_FIELDS = ("start", "include", "count", "avg", "bins_start", "bins_end", "fft_size", "decimation", "pending",
                "processed")


def dump_outputs(d, readout):
    """readout: psd_all()'s [(spectrum, breaks)] per channel; at most 16 stages x (N/2 + 1) bins per channel"""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    for c, (p, breaks) in enumerate(readout):
        rows = [(k.start, k.include, k.count, k.avg, k.bins.start, k.bins.stop, k.fft_size, k.decimation, k.pending,
                 k.processed) for k in breaks]
        np.save(os.path.join(d, "psd_ch%d.npy" % c), np.asarray(p, np.float32))
        np.save(os.path.join(d, "breaks_ch%d.npy" % c), np.array(rows, np.float64).reshape(-1, len(BREAK_FIELDS)))


def timechunk_record(new_group, barrier, rank, world, dist, dev):
    """BASELINE config 5 beside the headline: ONE 4.8e9-sample capture cut into `world` time chunks (strong scaling),
    every rank generating its range of the counter-based stream on its device; one NCCL sum-reduction of rows +
    counts + tail slices at readout, all inside the library (sspsd_group_time_*).  The merged spectrum is checked
    against the float64 truth rows committed in tests/golden/fullsize_c5_default.npz (tools/gen_golden_fullsize.py)."""
    import numpy as np
    import torch
    from stabilizer_stream_b200 import ShardMode
    total = 4_800_000_000
    g = new_group(ShardMode.TIME)
    times = []
    for it in range(3):
        g.time_plan(total)          # creates + positions the handles (allocations): outside the timed region
        barrier()
        t0 = time.perf_counter()
        g.time_process_noise(0, 0x7654321)
        g.time_finish()             # collective; synchronises
        p, b = g.psd(0)
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        times.append(float(t.item()))
    out = {"workload": "4.8e9-sample capture, N=4096, time-chunked over %d GPU(s) (strong scaling)" % world,
           "samples": total, "seconds": min(times), "value": total / min(times) / 1e6, "unit": "MS/s",
           "n_local_stages": g.time_chunk(0).n_local, "reduce": g.info()["reduce"] if world > 1 else "none",
           "timing": "host clock around process + exchange + psd(), max over ranks, best of 3 (input generated on the device)"}
    if rank == 0:
        out["stage_counts"] = [k.count for k in reversed(b)]
        gold = os.path.join(ROOT, "tests", "golden", "fullsize_c5_default.npz")
        if os.path.exists(gold):
            z = np.load(gold)
            rows64, counts = z["rows64"], z["counts"]
            truth = []
            for k in b:
                stage = 0
                while 8 ** stage < k.decimation:
                    stage += 1
                if k.include:
                    gain = (N_FFT // 2) * float(counts[stage]) * 1.5 * 0.25
                    truth.append(rows64[stage][k.bins.start:k.bins.stop] / (gain * k.decimation))
            truth = np.concatenate(truth)
            floor = 1e-5 * np.median(truth)
            out["max_rel_vs_f64"] = float(np.max(np.maximum(np.abs(p - truth) - floor, 0) / truth)) if truth.size == p.size else None
            out["counts_match_golden"] = [k.count for k in reversed(b)] == [int(c) for c in counts]
    return out


def e2e_frames(local, chunk=1 << 16):
    """BASELINE config 3 end to end: AdcDac frames (22 batches, 1416 bytes; header + i16 ADC/DAC words, reference
    src/de/data.rs:12-82) in pinned HOST memory -> H2D -> frame decode + loss accounting -> four cascades
    (one per trace, src/bin/psd.rs:174-182) -> psd() of each.  2.011 bytes cross PCIe per trace sample instead
    of 4, so the PCIe-bound end-to-end rate in trace samples is about twice that of the raw f32 stream."""
    import numpy as np
    import torch
    from stabilizer_stream_b200 import FrameDecoder, Loss, MergeOpts, PsdCascade
    batches, n_frames = 22, 1 << 20     # config 3's batch: 2^20 frames = 1.48 GB = 184.5e6 samples per trace
    flen = 8 + 64 * batches
    rng = np.random.default_rng(3)
    fr = np.empty((n_frames, flen), np.uint8)
    fr[:, 0], fr[:, 1], fr[:, 2], fr[:, 3] = 0x7B, 0x05, 1, batches
    seq = (np.arange(n_frames, dtype=np.uint64) * batches + 0xFFFFF000).astype(np.uint32)
    fr[:, 4:8] = seq.view(np.uint8).reshape(n_frames, 4)
    base = rng.integers(0, 256, (1 << 16, flen - 8), dtype=np.uint8)   # random ADC/DAC words, repeated every 2^16 frames
    for f0 in range(0, n_frames, 1 << 16):
        fr[f0:f0 + (1 << 16), 8:] = base
    host = torch.from_numpy(fr.reshape(-1)).pin_memory()
    dec = FrameDecoder(local)
    cas = [PsdCascade(N_FFT, device=local) for _ in range(4)]
    # chunk = frames per call: the call returns once its frames are decoded (Loss is returned by value), the cascades of
    # call c run while the frames of call c + 1 cross PCIe

    def one_pass():
        loss = Loss()
        for f0 in range(0, n_frames, chunk):
            dec.process_frames(cas, host[f0 * flen:(f0 + chunk) * flen], flen, loss)
        return [c.psd(MergeOpts()) for c in cas], loss

    one_pass()
    torch.cuda.synchronize()
    times = []
    for _ in range(3):
        t0 = time.perf_counter()
        res, loss = one_pass()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    dt = sorted(times)[len(times) // 2]   # median of 3 passes (host-clocked: the decode call synchronises per chunk)
    samples = 4 * n_frames * batches * 8
    return {"value": samples / dt / 1e6, "unit": "M trace-samples/s", "frames_per_step": n_frames, "frames_per_call": chunk,
            "frame_bytes": flen,
            "h2d_bytes_per_step": n_frames * flen, "h2d_GBps": n_frames * flen / dt / 1e9, "seconds_per_step": dt,
            "seconds_per_step_all": times, "bytes_per_trace_sample": n_frames * flen / samples, "loss_received": int(loss.received), "loss_dropped": int(loss.dropped),
            "stage0_count": res[0][1][-1].count}


def small_calls():
    """The reference's call pattern through the C ABI from plain C: 4096-sample pageable slices
    (reference src/source.rs:116, src/bin/psd.rs:170-183); tools/small_calls.c"""
    import subprocess
    exe = os.path.join(ROOT, "tools", "_build", "small_calls")
    if not os.path.exists(exe):
        return {"unavailable": "tools/_build/small_calls not built (run __graft_entry__.build())"}
    res = {}
    for name, argv in (("n4096_block4096", ["4096", "4096", "400000000"]), ("n512_block4096", ["512", "4096", "400000000"]),
                       ("n512_block176", ["512", "176", "100000000"])):
        try:
            r = subprocess.run([exe] + argv, capture_output=True, text=True, timeout=120)
            res[name] = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else {"error": r.stderr[-300:]}
        except Exception as e:  # noqa: BLE001
            res[name] = {"error": repr(e)}
    return res


_REAL_STDOUT = None


def emit(obj):
    """the ONE JSON line of the contract, on the process's real stdout"""
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


def main():
    # Libraries print to stdout behind our back (NCCL announces its version at the first communicator when
    # NCCL_DEBUG=VERSION/WARN is set in the environment): everything but the result line goes to stderr.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the headline loop's final psd() readout as .npy files")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
