"""stabilizer-stream cascaded PSD hot path on B200 (sm_100a).

Host-side mirror of the reference API (src/psd.rs, src/de, src/loss.rs, src/var.rs) over the
C ABI in include/sspsd.h.  The CUDA library is the only implementation: importing `psd` symbols
works without a GPU, creating any handle does not.
"""
from .psd import (DEPTH, HBF_PASSBAND, AvgOpts, Break, CsdCascade, CsmCascade, DecodeError, Detrend, Format, FrameDecoder, Hbf, Loss,
                  MergeOpts, Plant, PlantInput, PlantSpec, Psd, PsdCascade, Receiver, ShardMode, Source, SourceKind, TimeChunk, Trace, Var, Window,
                  ZoomCascade, Group, GroupKind, time_plan)

__all__ = ["DEPTH", "HBF_PASSBAND", "AvgOpts", "Break", "CsdCascade", "CsmCascade", "DecodeError", "Detrend", "Format", "FrameDecoder", "Hbf",
           "Loss", "MergeOpts", "Plant", "PlantInput", "PlantSpec", "Psd", "PsdCascade", "Receiver", "ShardMode", "Source", "SourceKind", "TimeChunk", "Trace",
           "Var", "Window", "ZoomCascade", "Group", "GroupKind", "time_plan"]
