"""CPU checks of ZoomCascade's interfaces (sspsd_zoom_*, sspsd_heterodyne_f32, the frame entry points): argument and
mode errors that need no device, the Python helpers, the C++ overloads (tests/cpp/test_zoom.cpp) and the --iq /
--zoom argument checks of tools/stream_psd.py."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "cpp", "_build", "test_zoom")
FRAME = bytes([0x7B, 0x05, 1, 1]) + bytes(4 + 64)


def test_null_handles_and_arguments_are_einval():
    from stabilizer_stream_b200 import _lib as L
    lib = L.lib()
    cfg = L.Config()
    L.check(lib.sspsd_config_default(512, C.byref(cfg)))
    h = C.c_void_p()
    assert lib.sspsd_zoom_create(None, L.ZOOM_IQ, 0, C.byref(h)) == L.EINVAL
    assert lib.sspsd_zoom_create(C.byref(cfg), L.ZOOM_IQ, 0, None) == L.EINVAL
    for call in (lambda: lib.sspsd_zoom_process_iq_f32(None, None, None, 0, L.MEM_HOST),
                 lambda: lib.sspsd_zoom_process_f32(None, None, 0, L.MEM_HOST),
                 lambda: lib.sspsd_zoom_reset(None), lambda: lib.sspsd_zoom_flush(None),
                 lambda: lib.sspsd_zoom_sync(None), lambda: lib.sspsd_zoom_num_stages(None, None),
                 lambda: lib.sspsd_zoom_carrier(None, None, None), lambda: lib.sspsd_zoom_stream(None, None),
                 lambda: lib.sspsd_zoom_rbw(None, None), lambda: lib.sspsd_zoom_clone(None, None),
                 lambda: lib.sspsd_zoom_read(None, None, None, None, None, None, None),
                 lambda: lib.sspsd_zoom_set_detrend(None, 0)):
        assert call() == L.EINVAL
    x = np.zeros(16, np.float32)
    assert lib.sspsd_heterodyne_f32(None, None, 16, 0, 1, x.ctypes.data, x.ctypes.data) == L.EINVAL
    assert lib.sspsd_heterodyne_f32(None, None, 0, 0, 1, None, None) == L.OK  # nothing to do
    buf = C.create_string_buffer(FRAME)
    loss = L.LossC()
    for traces in (None, (C.c_uint32 * 2)(0, 1), (C.c_uint32 * 2)(0, 9)):
        assert lib.sspsd_zoom_process_frames(None, None, traces, buf, 1, len(FRAME), len(FRAME), L.MEM_HOST,
                                             C.byref(loss), None) == L.EINVAL
        assert lib.sspsd_receiver_pump_zoom(None, None, None, traces, 16, 0, None, None) == L.EINVAL
    assert (loss.received, loss.dropped, loss.has_seq) == (0, 0, 0)


def test_python_mode_and_trace_map_checks():
    """the wrong call for the mode, a tuning word outside 32 bits or the wrong number of trace indices raise before
    any library call"""
    from stabilizer_stream_b200 import FrameDecoder, Loss, ZoomCascade
    from stabilizer_stream_b200 import _lib as L
    with pytest.raises(ValueError):
        ZoomCascade.heterodyne(512, 2 ** 32)
    with pytest.raises(ValueError):
        ZoomCascade.heterodyne(512, -1)
    iq = ZoomCascade.__new__(ZoomCascade)
    iq._h, iq.mode = None, L.ZOOM_IQ
    het = ZoomCascade.__new__(ZoomCascade)
    het._h, het.mode = None, L.ZOOM_HETERODYNE
    x = np.zeros(8, np.float32)
    with pytest.raises(ValueError):
        iq.process(x)
    with pytest.raises(ValueError):
        het.process(x, x)
    with pytest.raises(ValueError):
        iq.process(x, x[:4])
    dec = FrameDecoder.__new__(FrameDecoder)
    dec._h = None
    for target, traces in ((iq, (2,)), (iq, (0, 1, 2)), (het, (0, 1))):
        with pytest.raises(ValueError):
            dec.process_frames(target, FRAME, len(FRAME), Loss(), traces=traces)


def test_ftw_of_and_two_sided_axis():
    from stabilizer_stream_b200 import Break, ZoomCascade
    assert ZoomCascade.ftw_of(0.25) == 1 << 30
    assert ZoomCascade.ftw_of(-0.25) == 3 << 30
    assert ZoomCascade.ftw_of(1.0) == 0
    assert ZoomCascade.ftw_of(1 / 3) == 0x55555555
    # one stage of N = 8: bins 0 .. 4 at f = k / 8; DC and Nyquist once
    b = [Break(0, True, 1, 1, range(0, 5), 8, 1, 0, 8)]
    pp = np.arange(5, dtype=np.float32) + 10
    pn = np.arange(5, dtype=np.float32) + 20
    f, p = ZoomCascade.two_sided(pp, pn, b, ftw=1 << 30)
    np.testing.assert_allclose(f, 0.25 + np.array([-3, -2, -1, 0, 1, 2, 3, 4]) / 8)
    np.testing.assert_array_equal(p, [23, 22, 21, 10, 11, 12, 13, 14])


def build_cpp():
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    lib = os.path.join(ROOT, "stabilizer_stream_b200")
    cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "test_zoom.cpp"), "-o", EXE, "-L", lib, "-lsspsd", "-Wl,-rpath," + lib]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return EXE


def test_cpp_overloads_compile_and_refuse_without_gpu():
    import torch
    exe = build_cpp()
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu test")
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 3, (r.returncode, r.stderr)


@pytest.mark.gpu
def test_cpp_overloads_on_gpu():
    r = subprocess.run([build_cpp()], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "zoom ok" in r.stdout, r.stdout + r.stderr


def run_driver(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "tools", "stream_psd.py"), *args], capture_output=True,
                          text=True, timeout=300)


def test_driver_help_lists_iq_and_zoom():
    r = run_driver("--help")
    assert r.returncode == 0 and "--iq" in r.stdout and "--zoom" in r.stdout


@pytest.mark.parametrize("args,msg", [
    (("--file", "x.bin", "--iq", "2"), "two trace indices"),
    (("--file", "x.bin", "--iq", "2,4"), "0 .. 3"),
    (("--file", "x.bin", "--iq", "a,b"), "two trace indices"),
    (("--raw", "x.bin", "--iq", "2,3"), "--file or --udp"),
    (("--file", "x.bin", "--zoom", "99999999999"), "32-bit"),
    (("--file", "x.bin", "--zoom", "12", "--iq", "2,3"), "one of"),
    (("--file", "x.bin", "--zoom", "12", "--csm", "0,1"), "one of"),
    (("--file", "x.bin", "--iq", "2,3", "--trace", "1"), "--trace"),
])
def test_driver_argument_errors(args, msg):
    r = run_driver(*args)
    assert r.returncode == 2 and msg in r.stderr, r.stderr
