"""CPU checks of the plant interfaces (sspsd_plant_*, the process_plant entry points, sspsd_group_time_process_plant):
spec and argument errors that need no device, the Python spec helpers, the C++ overloads (tests/cpp/test_plant.cpp)
and the --plant argument checks of tools/stream_psd.py."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "tests", "cpp", "_build", "test_plant")


def spec_c(k=1, m=1, nt=1, inputs=None, taps=True):
    from stabilizer_stream_b200 import _lib as L
    ins = inputs if inputs is not None else [(L.PLANT_NOISE, 0, 1, 0.0)] * m
    arr = (L.PlantInputC * max(len(ins), 1))(*[L.PlantInputC(a, 0, b, c, d, 0) for a, b, c, d in ins])
    t = np.ones(max(k * m * nt, 1), np.float32)
    s = L.PlantSpecC(k, m, nt, 0, t.ctypes.data_as(C.POINTER(C.c_float)) if taps else None, arr)
    return s, (arr, t)


@pytest.mark.parametrize("k,m,nt,inputs,taps,status", [
    (0, 1, 1, None, True, "EINVAL"),
    (5, 1, 1, None, True, "EINVAL"),
    (1, 0, 1, None, True, "EINVAL"),
    (1, 5, 1, None, True, "EINVAL"),
    (1, 1, 0, None, True, "EINVAL"),
    (1, 1, 33, None, True, "EINVAL"),
    (1, 1, 1, None, False, "EINVAL"),
    (1, 1, 1, [(7, 0, 0, 0.0)], True, "EINVAL"),               # unknown kind
    (1, 1, 1, [(1, 2 ** 32, 0, 1.0)], True, "EINVAL"),          # tone ftw past u32
    (1, 1, 1, [(1, -1, 0, 1.0)], True, "EINVAL"),
    (1, 1, 1, [(1, 5, 0, float("inf"))], True, "EINVAL"),       # amplitude not finite
    (1, 1, 1, [(0, -1, 0, 0.0)], True, "EUNIMPLEMENTED"),       # integrated noise carries state
    (1, 1, 1, [(0, 9, 0, 0.0)], True, "EUNIMPLEMENTED"),
    (1, 1, 1, None, True, "ECUDA"),                             # a valid spec: no device here
])
def test_create_checks_the_spec_before_the_device(k, m, nt, inputs, taps, status):
    import torch
    from stabilizer_stream_b200 import _lib as L
    if status == "ECUDA" and torch.cuda.is_available():
        pytest.skip("GPU present")
    s, keep = spec_c(k, m, nt, inputs, taps)
    h = C.c_void_p()
    assert L.lib().sspsd_plant_create(C.byref(s), 0, None, C.byref(h)) == getattr(L, status)
    assert not h.value
    del keep


def test_null_handles_and_arguments_are_einval():
    from stabilizer_stream_b200 import _lib as L
    lib = L.lib()
    s, keep = spec_c()
    assert lib.sspsd_plant_create(None, 0, None, C.byref(C.c_void_p())) == L.EINVAL
    assert lib.sspsd_plant_create(C.byref(s), 0, None, None) == L.EINVAL
    for call in (lambda: lib.sspsd_plant_reset(None), lambda: lib.sspsd_plant_seek(None, 5),
                 lambda: lib.sspsd_plant_position(None, None), lambda: lib.sspsd_plant_generate(None, None, 4),
                 lambda: lib.sspsd_cascade_process_plant(None, None, 4), lambda: lib.sspsd_csd_process_plant(None, None, 4),
                 lambda: lib.sspsd_csm_process_plant(None, None, 4), lambda: lib.sspsd_zoom_process_plant(None, None, 4),
                 lambda: lib.sspsd_group_time_process_plant(None, C.byref(s))):
        assert call() == L.EINVAL
    lib.sspsd_plant_destroy(None)
    del keep


def test_python_spec_checks():
    from stabilizer_stream_b200 import Plant, PlantSpec
    from stabilizer_stream_b200 import _lib as L
    with pytest.raises(ValueError):
        PlantSpec(np.ones((2, 2)), [Plant.noise()])                      # not [K, M, L]
    with pytest.raises(ValueError):
        PlantSpec(np.ones((2, 2, 3)), [Plant.noise()])                   # M = 2 taps, one input
    with pytest.raises(TypeError):
        PlantSpec(np.ones((1, 1, 1)), [(0, 0, 0, 0.0)])
    s = PlantSpec(np.arange(24).reshape(2, 3, 4), [Plant.noise(1, 5), Plant.tone(7, 0.5), Plant.noise(seed=2 ** 64 - 1)])
    assert (s.c.k, s.c.m, s.c.taps_len) == (2, 3, 4)
    assert [s.c.inputs[i].kind for i in range(3)] == [L.PLANT_NOISE, L.PLANT_TONE, L.PLANT_NOISE]
    assert (s.c.inputs[1].param, s.c.inputs[1].amplitude, s.c.inputs[2].seed) == (7, 0.5, 2 ** 64 - 1)
    assert [s.c.taps[i] for i in range(24)] == list(range(24))
    assert C.sizeof(L.PlantInputC) == 32 and C.sizeof(L.PlantSpecC) == 32


def test_expected_csm_of_white_noise_and_a_delay():
    """a unit-RMS white input reads 2 (the one-sided density); y1 = u delayed by one: S_01 = 2 e^(-2 pi i f)"""
    from stabilizer_stream_b200 import Plant
    p = Plant.__new__(Plant)
    from stabilizer_stream_b200.psd import PlantSpec
    p._spec = PlantSpec([[[1.0, 0.0]], [[0.0, 1.0]]], [Plant.noise(0)])
    p.k = 2
    f = np.linspace(0, 0.5, 11)
    S = p.expected_csm(f)
    np.testing.assert_allclose(S[0, 0], 2.0)
    np.testing.assert_allclose(S[1, 1], 2.0)
    np.testing.assert_allclose(S[0, 1], 2.0 * np.exp(-2j * np.pi * f), atol=1e-12)
    np.testing.assert_allclose(S[1, 0], np.conj(S[0, 1]))
    p._spec = PlantSpec([[[1.0]]], [Plant.noise(2), Plant.tone(5)][:1])
    p.k = 1
    np.testing.assert_allclose(p.expected_csm(f)[0, 0], 2.0 * (2 * np.sin(np.pi * f)) ** 4)
    p._h = None


def build_cpp():
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    lib = os.path.join(ROOT, "stabilizer_stream_b200")
    cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
           os.path.join(ROOT, "tests", "cpp", "test_plant.cpp"), "-o", EXE, "-L", lib, "-lsspsd", "-Wl,-rpath," + lib]
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
    assert r.returncode == 0 and "plant ok" in r.stdout, r.stdout + r.stderr


def run_driver(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "tools", "stream_psd.py"), *args], capture_output=True,
                          text=True, timeout=300)


def test_driver_help_lists_plant():
    r = run_driver("--help")
    assert r.returncode == 0 and "--plant" in r.stdout


def _write(tmp_path, obj):
    p = tmp_path / "plant.json"
    p.write_text(obj if isinstance(obj, str) else json.dumps(obj))
    return str(p)


GOOD = {"taps": [[[1.0, 0.5]], [[0.0, 1.0]]], "inputs": [{"noise": 0, "seed": 1}], "samples": 1000}


@pytest.mark.parametrize("spec,extra,msg", [
    ("{not json", (), "JSON"),
    ({"inputs": [{"noise": 0}], "samples": 10}, (), "taps"),
    ({"taps": [[[1.0]]], "inputs": [{"noise": 0}]}, (), "samples"),
    ({"taps": [[[1.0]]], "inputs": [{"dsm": 3}], "samples": 10}, (), "every input is"),
    ({"taps": [[[1.0]]], "inputs": [{"noise": 0}, {"noise": 1}], "samples": 10}, (), "[K, M, L]"),
    (GOOD, (), "--csm, --iq or --zoom"),                        # K = 2 with the PSD target
    (GOOD, ("--csm", "0,1,2"), "outputs"),                       # K = 2 into a 3-channel matrix
    (GOOD, ("--zoom", "12"), "outputs"),                         # heterodyne takes one
    (GOOD, ("--noise", "0"), "one of"),
])
def test_driver_plant_argument_errors(tmp_path, spec, extra, msg):
    r = run_driver("--plant", _write(tmp_path, spec), *extra)
    assert r.returncode == 2 and msg in r.stderr, r.stderr
