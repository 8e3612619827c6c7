"""CPU checks of the frame entry points of the cross-spectral cascades (sspsd_csd_process_frames,
sspsd_csm_process_frames, sspsd_receiver_pump_csd / _csm): argument errors that need no device, the C++ overloads,
and the --csm argument checks of tools/stream_psd.py."""
import ctypes as C
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "cpp", "_build", "test_frames_xspec")
FRAME = bytes([0x7B, 0x05, 1, 1]) + bytes(4 + 64)


def test_null_handles_and_trace_indices_are_einval():
    from stabilizer_stream_b200 import _lib as L
    lib = L.lib()
    buf = C.create_string_buffer(FRAME)
    for traces in (None, (C.c_uint32 * 4)(0, 1, 2, 3), (C.c_uint32 * 4)(0, 9, 2, 3)):
        assert lib.sspsd_csm_process_frames(None, None, traces, buf, 1, len(FRAME), len(FRAME), L.MEM_HOST, None,
                                            None) == L.EINVAL
        assert lib.sspsd_receiver_pump_csm(None, None, None, traces, 16, 0, None, None) == L.EINVAL
    for tx, ty in ((0, 1), (0, 4), (7, 1)):
        assert lib.sspsd_csd_process_frames(None, None, tx, ty, buf, 1, len(FRAME), len(FRAME), L.MEM_HOST, None,
                                            None) == L.EINVAL
        assert lib.sspsd_receiver_pump_csd(None, None, None, tx, ty, 16, 0, None, None) == L.EINVAL
    loss = L.LossC()
    assert lib.sspsd_csd_process_frames(None, None, 0, 1, buf, 1, len(FRAME), len(FRAME), L.MEM_HOST, C.byref(loss),
                                        None) == L.EINVAL
    assert (loss.received, loss.dropped, loss.has_seq) == (0, 0, 0)


def test_python_trace_maps_are_checked_before_the_library():
    """the wrong number of trace indices for the target, or traces= for PsdCascades, raise before any call"""
    from stabilizer_stream_b200 import CsdCascade, CsmCascade, FrameDecoder, Loss
    dec = FrameDecoder.__new__(FrameDecoder)
    dec._h = None
    m = CsmCascade.__new__(CsmCascade)
    m._h, m.channels = None, 3
    c = CsdCascade.__new__(CsdCascade)
    c._h = None
    for target, traces in ((m, (0, 1)), (m, (0, 1, 2, 3)), (c, (0,)), (c, (0, 1, 2)), ([None] * 4, (0, 1))):
        with pytest.raises(ValueError):
            dec.process_frames(target, FRAME, len(FRAME), Loss(), traces=traces)


def build_cpp():
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    lib = os.path.join(ROOT, "stabilizer_stream_b200")
    cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "test_frames_xspec.cpp"), "-o", EXE, "-L", lib, "-lsspsd",
           "-Wl,-rpath," + lib]
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
    assert r.returncode == 0 and "frames xspec ok" in r.stdout, r.stdout + r.stderr


def run_driver(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "tools", "stream_psd.py"), *args], capture_output=True,
                          text=True, timeout=300)


def test_driver_help_lists_csm():
    r = run_driver("--help")
    assert r.returncode == 0 and "--csm" in r.stdout and "--save" in r.stdout


@pytest.mark.parametrize("args,msg", [
    (("--file", "x.bin", "--csm", "0,1,2,3,0"), "2 to 4"),
    (("--file", "x.bin", "--csm", "0"), "2 to 4"),
    (("--file", "x.bin", "--csm", "0,4"), "0 .. 3"),
    (("--file", "x.bin", "--csm", "a,b"), "comma-separated"),
    (("--raw", "x.bin", "--csm", "0,1"), "--file or --udp"),
    (("--file", "x.bin", "--csm", "0,2", "--trace", "1"), "--trace"),
    (("--file", "x.bin", "--save", "s.npz"), "--save needs --csm"),
])
def test_driver_argument_errors(args, msg):
    r = run_driver(*args)
    assert r.returncode == 2 and msg in r.stderr, r.stderr
