"""Loader and ctypes prototypes of the C ABI (include/sspsd.h) of libsspsd.so.

There is no CPU fallback: if the shared library has not been built (``python -c "import
__graft_entry__ as g; g.build()"`` or ``make -C stabilizer_stream_b200``) importing this module
raises, and every create call fails with SSPSD_ECUDA when no CUDA device is usable.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SSPSD_LIB selects another build of the same library (e.g. libsspsd_bounds.so, the bounds-checking build)
LIB_PATH = os.environ.get("SSPSD_LIB") or os.path.join(_HERE, "libsspsd.so")

OK, EINVAL, EUNIMPLEMENTED, ECUDA, ENOMEM, EHEADER, EFORMAT, ESIZE, EBATCHES, ESHORT, ENCCL, EIO = range(12)
MEM_HOST, MEM_DEVICE = 0, 1
ZOOM_IQ, ZOOM_HETERODYNE = 0, 1
FLAG_DETERMINISTIC = 1
MAX_STAGES = 16
MAX_TRACES = 4

STATUS_NAMES = {0: "OK", 1: "EINVAL", 2: "EUNIMPLEMENTED", 3: "ECUDA", 4: "ENOMEM", 5: "EHEADER", 6: "EFORMAT",
                7: "ESIZE", 8: "EBATCHES", 9: "ESHORT", 10: "ENCCL", 11: "EIO"}


class Config(C.Structure):
    _fields_ = [("n_fft", C.c_uint32), ("window", C.c_int32), ("hbf", C.c_int32), ("device", C.c_int32),
                ("stream", C.c_void_p), ("max_batch", C.c_uint64), ("host_stage", C.c_uint64),
                ("deep_defer", C.c_uint64), ("flags", C.c_uint32), ("_pad", C.c_uint32)]


class AvgOptsC(C.Structure):
    _fields_ = [("limit", C.c_uint32), ("count", C.c_uint32)]


class MergeOptsC(C.Structure):
    _fields_ = [("keep_overlap", C.c_uint32), ("min_count", C.c_uint32), ("keep_transition_band", C.c_uint32)]


class BreakC(C.Structure):
    _fields_ = [("start", C.c_uint64), ("include", C.c_uint32), ("count", C.c_uint32), ("avg", C.c_uint32),
                ("_pad", C.c_uint32), ("bins_start", C.c_uint64), ("bins_end", C.c_uint64),
                ("fft_size", C.c_uint64), ("decimation", C.c_uint64), ("pending", C.c_uint64),
                ("processed", C.c_uint64)]


class PartialsC(C.Structure):
    _fields_ = [("acc", C.c_void_p), ("acc_stride", C.c_uint64), ("n_stages", C.c_uint32), ("_pad", C.c_uint32),
                ("count_raw", C.c_uint64 * MAX_STAGES)]


class ProfileC(C.Structure):
    _fields_ = [("ms", C.c_double * 5), ("launches", C.c_uint64 * 5), ("units", C.c_uint64 * 5),
                ("launches_total", C.c_uint64)]


class LossC(C.Structure):
    _fields_ = [("received", C.c_uint64), ("dropped", C.c_uint64), ("seq", C.c_uint32), ("has_seq", C.c_uint32)]


class DecodeInfoC(C.Structure):
    _fields_ = [("format", C.c_uint32), ("n_traces", C.c_uint32), ("samples_per_trace", C.c_uint64),
                ("frames_ok", C.c_uint64)]


class PlotOptsC(C.Structure):
    _fields_ = [("fs", C.c_float), ("integral_start", C.c_float), ("integral_end", C.c_float),
                ("integrate", C.c_uint32)]


class TimeChunkC(C.Structure):
    _fields_ = [("own_lo", C.c_uint64), ("own_hi", C.c_uint64), ("feed_lo", C.c_uint64), ("feed_hi", C.c_uint64),
                ("tail_lo", C.c_uint64), ("tail_hi", C.c_uint64), ("n_local", C.c_uint32), ("_pad", C.c_uint32)]


class VarC(C.Structure):
    _fields_ = [("x_exp", C.c_int32), ("sinx_exp", C.c_int32), ("clip", C.c_float), ("_pad", C.c_uint32),
                ("dc_cut", C.c_uint64)]


_vp = C.c_void_p
_sz = C.c_size_t
_psz = C.POINTER(C.c_size_t)
_i32 = C.c_int32

# name -> (restype, argtypes); one entry per declaration in include/sspsd.h
PROTOTYPES = {
    "sspsd_last_error": (C.c_char_p, []),
    "sspsd_hbf_info": (_i32, [_i32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "sspsd_config_default": (_i32, [C.c_uint32, C.POINTER(Config)]),
    "sspsd_cascade_create": (_i32, [C.POINTER(Config), C.POINTER(_vp)]),
    "sspsd_cascade_destroy": (None, [_vp]),
    "sspsd_cascade_clone": (_i32, [_vp, C.POINTER(_vp)]),
    "sspsd_cascade_reset": (_i32, [_vp]),
    "sspsd_cascade_process_f32": (_i32, [_vp, _vp, _sz, _i32]),
    "sspsd_cascade_set_avg": (_i32, [_vp, AvgOptsC]),
    "sspsd_cascade_set_detrend": (_i32, [_vp, _i32]),
    "sspsd_cascade_rbw": (_i32, [_vp, C.POINTER(C.c_float)]),
    "sspsd_cascade_psd": (_i32, [_vp, C.POINTER(MergeOptsC), _vp, _psz, C.POINTER(BreakC), _psz]),
    "sspsd_cascade_num_stages": (_i32, [_vp, C.POINTER(C.c_uint32)]),
    "sspsd_cascade_stream": (_i32, [_vp, C.POINTER(_vp)]),
    "sspsd_cascade_flush": (_i32, [_vp]),
    "sspsd_cascade_sync": (_i32, [_vp]),
    "sspsd_break_frequencies": (_i32, [C.POINTER(BreakC), _sz, _vp, _psz]),
    "sspsd_csd_create": (_i32, [C.POINTER(Config), C.POINTER(_vp)]),
    "sspsd_csd_destroy": (None, [_vp]),
    "sspsd_csd_clone": (_i32, [_vp, C.POINTER(_vp)]),
    "sspsd_csd_reset": (_i32, [_vp]),
    "sspsd_csd_process_f32": (_i32, [_vp, _vp, _vp, _sz, _i32]),
    "sspsd_csd_set_avg": (_i32, [_vp, AvgOptsC]),
    "sspsd_csd_set_detrend": (_i32, [_vp, _i32]),
    "sspsd_csd_rbw": (_i32, [_vp, C.POINTER(C.c_float)]),
    "sspsd_csd_read": (_i32, [_vp, C.POINTER(MergeOptsC), _vp, _vp, _vp, _psz, C.POINTER(BreakC), _psz]),
    "sspsd_csd_num_stages": (_i32, [_vp, C.POINTER(C.c_uint32)]),
    "sspsd_csd_stream": (_i32, [_vp, C.POINTER(_vp)]),
    "sspsd_csd_flush": (_i32, [_vp]),
    "sspsd_csd_sync": (_i32, [_vp]),
    "sspsd_csm_create": (_i32, [C.POINTER(Config), _i32, C.POINTER(_vp)]),
    "sspsd_csm_destroy": (None, [_vp]),
    "sspsd_csm_clone": (_i32, [_vp, C.POINTER(_vp)]),
    "sspsd_csm_channels": (_i32, [_vp, C.POINTER(_i32)]),
    "sspsd_csm_reset": (_i32, [_vp]),
    "sspsd_csm_process_f32": (_i32, [_vp, _vp, _sz, _i32]),
    "sspsd_csm_set_avg": (_i32, [_vp, AvgOptsC]),
    "sspsd_csm_set_detrend": (_i32, [_vp, _i32]),
    "sspsd_csm_rbw": (_i32, [_vp, C.POINTER(C.c_float)]),
    "sspsd_csm_read": (_i32, [_vp, C.POINTER(MergeOptsC), _vp, _psz, C.POINTER(BreakC), _psz]),
    "sspsd_csm_num_stages": (_i32, [_vp, C.POINTER(C.c_uint32)]),
    "sspsd_csm_stream": (_i32, [_vp, C.POINTER(_vp)]),
    "sspsd_csm_flush": (_i32, [_vp]),
    "sspsd_csm_sync": (_i32, [_vp]),
    "sspsd_zoom_create": (_i32, [C.POINTER(Config), _i32, C.c_uint32, C.POINTER(_vp)]),
    "sspsd_zoom_destroy": (None, [_vp]),
    "sspsd_zoom_clone": (_i32, [_vp, C.POINTER(_vp)]),
    "sspsd_zoom_reset": (_i32, [_vp]),
    "sspsd_zoom_process_iq_f32": (_i32, [_vp, _vp, _vp, _sz, _i32]),
    "sspsd_zoom_process_f32": (_i32, [_vp, _vp, _sz, _i32]),
    "sspsd_zoom_set_avg": (_i32, [_vp, AvgOptsC]),
    "sspsd_zoom_set_detrend": (_i32, [_vp, _i32]),
    "sspsd_zoom_rbw": (_i32, [_vp, C.POINTER(C.c_float)]),
    "sspsd_zoom_read": (_i32, [_vp, C.POINTER(MergeOptsC), _vp, _vp, _psz, C.POINTER(BreakC), _psz]),
    "sspsd_zoom_carrier": (_i32, [_vp, C.POINTER(_i32), C.POINTER(C.c_uint32)]),
    "sspsd_zoom_num_stages": (_i32, [_vp, C.POINTER(C.c_uint32)]),
    "sspsd_zoom_stream": (_i32, [_vp, C.POINTER(_vp)]),
    "sspsd_zoom_flush": (_i32, [_vp]),
    "sspsd_zoom_sync": (_i32, [_vp]),
    "sspsd_heterodyne_f32": (_i32, [_vp, _vp, _sz, C.c_uint64, C.c_uint32, _vp, _vp]),
    "sspsd_cascade_partials": (_i32, [_vp, C.POINTER(PartialsC)]),
    "sspsd_cascade_set_counts": (_i32, [_vp, C.POINTER(C.c_uint64), C.c_uint32]),
    "sspsd_cascade_seek": (_i32, [_vp, C.c_uint64]),
    "sspsd_cascade_set_window": (_i32, [_vp, C.c_uint64, C.c_uint64, C.c_uint32]),
    "sspsd_cascade_take_tail": (_i32, [_vp, C.c_uint64, C.c_uint64, _vp, _psz, C.POINTER(C.c_uint64), _i32]),
    "sspsd_cascade_process_stage": (_i32, [_vp, C.c_uint32, _vp, _sz, _i32]),
    "sspsd_cascade_set_stream_state": (_i32, [_vp, C.c_uint32, C.c_uint64, C.c_uint64]),
    "sspsd_cascade_profile_enable": (_i32, [_vp, _i32]),
    "sspsd_cascade_profile_read": (_i32, [_vp, C.POINTER(ProfileC)]),
    "sspsd_stage_create": (_i32, [C.POINTER(Config), C.POINTER(_vp)]),
    "sspsd_stage_destroy": (None, [_vp]),
    "sspsd_stage_stream": (_i32, [_vp, C.POINTER(_vp)]),
    "sspsd_stage_set_avg": (_i32, [_vp, C.c_uint32]),
    "sspsd_stage_set_detrend": (_i32, [_vp, _i32]),
    "sspsd_stage_process_f32": (_i32, [_vp, _vp, _sz, _i32, _vp, _psz, _i32]),
    "sspsd_stage_spectrum": (_i32, [_vp, _vp, _psz, _i32]),
    "sspsd_stage_count": (_i32, [_vp, C.POINTER(C.c_uint32)]),
    "sspsd_stage_gain": (_i32, [_vp, C.POINTER(C.c_float)]),
    "sspsd_stage_buf": (_i32, [_vp, _vp, _psz, _i32]),
    "sspsd_decoder_create": (_i32, [_i32, _vp, C.POINTER(_vp)]),
    "sspsd_decoder_destroy": (None, [_vp]),
    "sspsd_decoder_stream": (_i32, [_vp, C.POINTER(_vp)]),
    "sspsd_decode_frames": (_i32, [_vp, _vp, _sz, _sz, _sz, _i32, C.POINTER(LossC), C.POINTER(_vp), _sz, _i32,
                                   C.POINTER(DecodeInfoC)]),
    "sspsd_cascade_process_frames": (_i32, [_vp, C.POINTER(_vp), C.c_uint32, _vp, _sz, _sz, _sz, _i32,
                                            C.POINTER(LossC), C.POINTER(DecodeInfoC)]),
    "sspsd_csm_process_frames": (_i32, [_vp, _vp, C.POINTER(C.c_uint32), _vp, _sz, _sz, _sz, _i32, C.POINTER(LossC),
                                        C.POINTER(DecodeInfoC)]),
    "sspsd_csd_process_frames": (_i32, [_vp, _vp, C.c_uint32, C.c_uint32, _vp, _sz, _sz, _sz, _i32, C.POINTER(LossC),
                                        C.POINTER(DecodeInfoC)]),
    "sspsd_zoom_process_frames": (_i32, [_vp, _vp, C.POINTER(C.c_uint32), _vp, _sz, _sz, _sz, _i32,
                                         C.POINTER(LossC), C.POINTER(DecodeInfoC)]),
    "sspsd_loss_update": (None, [C.POINTER(LossC), C.c_uint32, C.c_uint8]),
    "sspsd_loss_ratio": (C.c_float, [C.POINTER(LossC)]),
    "sspsd_var_eval": (C.c_float, [C.POINTER(VarC), _vp, _vp, _sz, C.c_float]),
    "sspsd_trace_plot": (_i32, [C.POINTER(PlotOptsC), _vp, _vp, _sz, C.POINTER(C.c_float), _vp, _psz]),
    "sspsd_source_create": (_i32, [_i32, C.c_int64, C.c_uint64, _i32, _vp, C.POINTER(_vp)]),
    "sspsd_source_destroy": (None, [_vp]),
    "sspsd_source_reset": (_i32, [_vp]),
    "sspsd_source_generate": (_i32, [_vp, _vp, _sz]),
    "sspsd_source_position": (_i32, [_vp, C.POINTER(C.c_uint64)]),
    "sspsd_cascade_process_source": (_i32, [_vp, _vp, _sz]),
    "sspsd_source_seek": (_i32, [_vp, C.c_uint64]),
    "sspsd_group_create": (_i32, [C.POINTER(Config), C.POINTER(_i32), C.c_uint32, _i32, C.POINTER(_vp)]),
    "sspsd_group_unique_id": (_i32, [_vp]),
    "sspsd_group_create_rank": (_i32, [C.POINTER(Config), _vp, C.c_uint32, C.c_uint32, _i32, C.POINTER(_vp)]),
    "sspsd_group_destroy": (None, [_vp]),
    "sspsd_group_info": (_i32, [_vp, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32),
                                C.POINTER(_i32), C.POINTER(_i32)]),
    "sspsd_group_set_avg": (_i32, [_vp, AvgOptsC]),
    "sspsd_group_set_detrend": (_i32, [_vp, _i32]),
    "sspsd_group_sync": (_i32, [_vp]),
    "sspsd_group_process_f32": (_i32, [_vp, C.c_uint32, _vp, _sz, _i32]),
    "sspsd_group_channel_device": (_i32, [_vp, C.c_uint32, C.POINTER(_i32), C.POINTER(C.c_uint32)]),
    "sspsd_group_channel_handle": (_i32, [_vp, C.c_uint32, C.POINTER(_vp)]),
    "sspsd_group_psd": (_i32, [_vp, C.c_uint32, C.POINTER(MergeOptsC), _vp, _psz, C.POINTER(BreakC), _psz]),
    "sspsd_group_psd_all": (_i32, [_vp, C.c_uint32, C.POINTER(MergeOptsC), _vp, _sz, _psz, C.POINTER(BreakC), _sz, _psz]),
    "sspsd_time_plan": (_i32, [C.c_uint32, _i32, _i32, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32,
                               C.POINTER(TimeChunkC)]),
    "sspsd_group_time_plan": (_i32, [_vp, C.c_uint64, C.c_uint32]),
    "sspsd_group_time_chunk": (_i32, [_vp, C.c_uint32, C.POINTER(TimeChunkC)]),
    "sspsd_group_time_process_f32": (_i32, [_vp, C.c_uint32, _vp, _sz, _i32]),
    "sspsd_group_time_process_all_f32": (_i32, [_vp, _vp, _sz]),
    "sspsd_group_time_process_noise": (_i32, [_vp, C.c_int64, C.c_uint64]),
    "sspsd_group_time_finish": (_i32, [_vp]),
    "sspsd_receiver_create": (_i32, [C.c_char_p, C.c_uint16, C.c_uint32, C.c_uint32, _i32, C.POINTER(_vp)]),
    "sspsd_receiver_destroy": (None, [_vp]),
    "sspsd_receiver_info": (_i32, [_vp, C.POINTER(C.c_uint16), _psz, C.POINTER(C.c_uint64)]),
    "sspsd_receiver_recv": (_i32, [_vp, C.c_uint32, _i32, C.POINTER(_vp), _psz, _psz]),
    "sspsd_receiver_pump": (_i32, [_vp, _vp, C.POINTER(_vp), C.c_uint32, C.c_uint32, _i32, C.POINTER(LossC),
                                   C.POINTER(DecodeInfoC)]),
    "sspsd_receiver_pump_csm": (_i32, [_vp, _vp, _vp, C.POINTER(C.c_uint32), C.c_uint32, _i32, C.POINTER(LossC),
                                       C.POINTER(DecodeInfoC)]),
    "sspsd_receiver_pump_csd": (_i32, [_vp, _vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, _i32, C.POINTER(LossC),
                                       C.POINTER(DecodeInfoC)]),
    "sspsd_receiver_pump_zoom": (_i32, [_vp, _vp, _vp, C.POINTER(C.c_uint32), C.c_uint32, _i32, C.POINTER(LossC),
                                        C.POINTER(DecodeInfoC)]),
}

_lib = None


class SspsdError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("%s (%d): %s" % (STATUS_NAMES.get(status, "?"), status, message))
        self.status = status


def lib():
    """Load libsspsd.so (raises if it has not been built -- there is no fallback path)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s not found: build the CUDA library first (__graft_entry__.build())" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(status):
    if status != OK:
        msg = lib().sspsd_last_error()
        raise SspsdError(status, msg.decode() if msg else "")
    return status
