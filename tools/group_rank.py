#!/usr/bin/env python3
"""One rank of a multi-process sspsd_group (ncclCommInitRank inside the library): launched by torchrun, checks
the group's result against the sequential cascade on rank 0 and prints one JSON line.

    torchrun --nproc-per-node N tools/group_rank.py --mode time|time_preset|channels [--total 6e6] [--n 512]
                                                    [--kind psd|csd|csm|zoom]

--kind csd / csm / zoom time-chunks one capture of 2 / 4 streams (zoom: one stream mixed down around a carrier) and
checks rank 0's readout against the matching sequential handle.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402


FTW = 0x9E3779B9


def cross_kind(sp, kind, n, total, rank, world, local, uid):
    """every process makes the same streams; each feeds its own rank's range; rank 0 checks the readout"""
    rng = np.random.default_rng(4321)
    x = (rng.random(total, dtype=np.float32) - np.float32(0.5)).astype(np.float32)
    xs = [x]
    if kind != "zoom":
        for c in range(1, 2 if kind == "csd" else 4):
            y = np.convolve(x, [0.5, -0.25 * c, 0.1])[:total] + 0.3 * (rng.random(total, dtype=np.float32) - 0.5)
            xs.append(y.astype(np.float32))
    args = {"csd": dict(kind=sp.GroupKind.CSD), "csm": dict(kind=sp.GroupKind.CSM, channels=4),
            "zoom": dict(kind=sp.GroupKind.ZOOM, zoom_mode=1, ftw=FTW)}[kind]
    g = sp.Group(n, rank=rank, n_ranks=world, unique_id=uid, device=local, mode=sp.ShardMode.TIME, **args)
    g.set_detrend(sp.Detrend.MEAN)
    g.set_avg(sp.AvgOpts(999, 2 ** 32 - 2))
    g.time_plan(total)
    c = g.time_chunk(rank)
    g.time_process(rank, *[v[c.feed_lo:c.feed_hi] for v in xs])
    g.time_finish()
    read = {"csd": lambda o: o.csd(), "csm": lambda o: o.csm(), "zoom": lambda o: o.spectrum()}[kind]
    got = read(g)
    if rank != 0:
        assert got[0].size == 0 and got[-1] == []
        return {}
    seq = {"csd": lambda: sp.CsdCascade(n, device=local), "csm": lambda: sp.CsmCascade(n, 4, device=local),
           "zoom": lambda: sp.ZoomCascade.heterodyne(n, FTW, device=local)}[kind]()
    seq.set_detrend(sp.Detrend.MEAN)
    seq.set_avg(sp.AvgOpts(999, 2 ** 32 - 2))
    seq.process(xs) if kind == "csm" else seq.process(*xs)
    want = read(seq)
    same = [(k.count, k.pending, k.processed, k.bins) for k in got[-1]] == \
        [(k.count, k.pending, k.processed, k.bins) for k in want[-1]]
    # every part of the readout relative to the largest diagonal entry of its bin (cross terms pass through zero)
    a = [np.asarray(v, np.complex128) for v in got[:-1]]
    b = [np.asarray(v, np.complex128) for v in want[:-1]]
    if kind == "csm":
        scale = np.max(np.abs(np.einsum("iib->ib", b[0])), axis=0)
    else:
        scale = np.max(np.abs(np.stack(b[:2])), axis=0)
    rel = max(float(np.max(np.abs(u - v)[..., 2:] / scale[2:])) for u, v in zip(a, b)) if a[0].shape == b[0].shape \
        else float("inf")
    return dict(breaks_equal=same, max_rel_diff_vs_sequential=rel, ok=bool(same and rel < 5e-5),
                reduce=g.info()["reduce"], n_local=c.n_local)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", default="time")
    ap.add_argument("--total", type=float, default=6e6)
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--kind", choices=["psd", "csd", "csm", "zoom"], default="psd")
    args = ap.parse_args()
    import stabilizer_stream_b200 as sp
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", "0"))
    dist.init_process_group("gloo")  # only to hand the 128-byte NCCL id around
    torch.cuda.set_device(local)
    ids = [sp.Group.unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    n, total = args.n, int(args.total)
    preset = args.mode == "time_preset"
    out = {"world": world, "mode": args.mode, "kind": args.kind}
    if args.kind != "psd":
        out.update(cross_kind(sp, args.kind, n, total, rank, world, local, ids[0]))
    elif args.mode.startswith("time"):
        g = sp.Group(n, rank=rank, n_ranks=world, unique_id=ids[0], device=local, mode=sp.ShardMode.TIME)
        if preset:
            g.set_detrend(sp.Detrend.MEAN)
            g.set_avg(sp.AvgOpts(999, 2 ** 32 - 2))
        g.time_plan(total)
        g.time_process_noise(0, sp.Source.SEED)
        g.time_finish()
        p, b = g.psd(0)
        if rank == 0:
            seq = sp.PsdCascade(n, device=local)
            if preset:
                seq.set_detrend(sp.Detrend.MEAN)
                seq.set_avg(sp.AvgOpts(999, 2 ** 32 - 2))
            src = sp.Source.noise(0, device=local)
            pos = 0
            while pos < total:
                m = min(1 << 26, total - pos)
                seq.process_source(src, m)
                pos += m
            ps, bs = seq.psd()
            same = [(k.count, k.pending, k.processed, k.bins) for k in b] == [(k.count, k.pending, k.processed, k.bins) for k in bs]
            head = 2 if preset else 0
            rel = float(np.max(np.abs(p[head:] - ps[head:]) / np.maximum(ps[head:], 1e-30))) if p.size == ps.size else float("inf")
            out.update(breaks_equal=same, max_rel_diff_vs_sequential=rel, ok=bool(same and rel < 5e-5), reduce=g.info()["reduce"],
                       n_local=g.time_chunk(0).n_local)
        else:
            assert p.size == 0 and b == []
    else:
        n_ch = 2 * world + 1
        g = sp.Group(n, rank=rank, n_ranks=world, unique_id=ids[0], device=local, mode=sp.ShardMode.CHANNELS)
        xs = []
        for c in range(n_ch):
            rng = np.random.default_rng(900 + c)
            xs.append(((rng.random(150 * n + 31 * c, dtype=np.float32) - np.float32(0.5)) * np.float32(1 + c)).astype(np.float32))
            g.process(c, xs[c])      # a no-op on the ranks that do not own channel c
        res = g.psd_all(n_ch)
        if rank == 0:
            ok = True
            for c in range(n_ch):
                seq = sp.PsdCascade(n, device=local)
                seq.process(xs[c])
                ps, bs = seq.psd()
                p, b = res[c]
                ok = ok and p.size == ps.size and [k.count for k in b] == [k.count for k in bs] and \
                    bool(np.max(np.abs(p - ps) / np.maximum(ps, 1e-30)) < 1e-5)
            out.update(ok=bool(ok), channels=n_ch)
        else:
            assert all(p.size == 0 for p, _ in res)
    if rank == 0:
        print(json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
