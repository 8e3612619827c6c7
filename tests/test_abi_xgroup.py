"""CPU checks of the group kinds (sspsd_group_create_kind & co.): kind, mode and size errors that need no device, the
Python stream-count checks, the C++ overloads (tests/cpp/test_xgroup.cpp) and tools/group_rank.py's --kind option."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "cpp", "_build", "test_xgroup")


def test_bad_kinds_are_einval_before_any_device():
    from stabilizer_stream_b200 import _lib as L
    lib = L.lib()
    cfg = L.Config()
    L.check(lib.sspsd_config_default(512, C.byref(cfg)))
    devs = (C.c_int32 * 2)(0, 0)
    h = C.c_void_p(1)
    bad = [(L.GROUP_CSM, 4, 0, 0, 0),            # a cross kind in channel mode
           (L.GROUP_CSM, 5, 0, 0, 1), (L.GROUP_CSM, 1, 0, 0, 1), (L.GROUP_CSD, 3, 0, 0, 1),
           (L.GROUP_ZOOM, 2, 2, 0, 1), (L.GROUP_ZOOM, 2, L.ZOOM_IQ, 5, 1), (L.GROUP_PSD, 2, 0, 0, 1),
           (L.GROUP_CSD, 2, 0, 7, 1), (9, 2, 0, 0, 1)]
    for kind, ch, zm, ftw, mode in bad:
        k = L.GroupKindC(kind, ch, zm, ftw)
        assert lib.sspsd_group_create_kind(C.byref(cfg), C.byref(k), devs, 2, mode, C.byref(h)) == L.EINVAL
        assert not h.value
        h = C.c_void_p(1)
        assert lib.sspsd_group_create_kind_rank(C.byref(cfg), C.byref(k), None, 0, 1, mode, C.byref(h)) == L.EINVAL
        assert not h.value
    for n in (8192, 32):
        L.check(lib.sspsd_config_default(n, C.byref(cfg)))
        k = L.GroupKindC(L.GROUP_CSD, 2, 0, 0)
        assert lib.sspsd_group_create_kind(C.byref(cfg), C.byref(k), devs, 2, 1, C.byref(h)) == L.EINVAL
    assert lib.sspsd_group_create_kind(C.byref(cfg), None, devs, 2, 1, C.byref(h)) == L.EINVAL


def test_null_groups_are_einval():
    from stabilizer_stream_b200 import _lib as L
    lib = L.lib()
    x = np.zeros(4, np.float32)
    ptrs = (C.c_void_p * 1)(x.ctypes.data)
    n = C.c_size_t(0)
    for call in (lambda: lib.sspsd_group_kind_of(None, None),
                 lambda: lib.sspsd_group_time_process_multi_f32(None, 0, ptrs, 4, L.MEM_HOST),
                 lambda: lib.sspsd_group_time_process_all_multi_f32(None, ptrs, 4),
                 lambda: lib.sspsd_group_csd_read(None, None, None, None, None, C.byref(n), None, C.byref(n)),
                 lambda: lib.sspsd_group_csm_read(None, None, None, C.byref(n), None, C.byref(n)),
                 lambda: lib.sspsd_group_zoom_read(None, None, None, None, C.byref(n), None, C.byref(n))):
        assert call() == L.EINVAL


def test_python_stream_count_checks():
    """the wrong number of streams, or streams of different lengths or memory kinds, raise before any library call"""
    from stabilizer_stream_b200 import Group, GroupKind
    g = Group.__new__(Group)
    g._h, g.kind, g.n_inputs = None, GroupKind.CSM, 3
    x = np.zeros(8, np.float32)
    with pytest.raises(ValueError):
        g.time_process(0, x, x)
    with pytest.raises(ValueError):
        g.time_process(0, x, x, x[:4])
    with pytest.raises(ValueError):
        g.time_process_all(x, x, x, x)


def build_cpp():
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    lib = os.path.join(ROOT, "stabilizer_stream_b200")
    cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "test_xgroup.cpp"), "-o", EXE, "-L", lib, "-lsspsd", "-Wl,-rpath," + lib]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return EXE


def test_cpp_overloads_compile_and_refuse_without_gpu():
    """the kind checks of tests/cpp/test_xgroup.cpp run before any device is needed; then ECUDA (exit code 3)"""
    import torch
    exe = build_cpp()
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu test")
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 3, (r.returncode, r.stderr)


def test_group_rank_lists_kind():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "group_rank.py"), "--help"], capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0 and "--kind" in r.stdout
