"""Every script the GPU box runs must at least compile here (no GPU needed): bench.py, __graft_entry__.py, tools/."""
import glob
import os
import py_compile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_scripts_compile(tmp_path):
    files = [os.path.join(ROOT, "bench.py"), os.path.join(ROOT, "__graft_entry__.py")]
    files += sorted(glob.glob(os.path.join(ROOT, "tools", "*.py")))
    files += sorted(glob.glob(os.path.join(ROOT, "stabilizer_stream_b200", "*.py")))
    assert len(files) > 8
    for f in files:
        py_compile.compile(f, cfile=str(tmp_path / (os.path.basename(f) + "c")), doraise=True)


def test_bench_reference_arm_contract_keys():
    """bench.py --impl reference and the default arm print the keys the driver reads (static check of the source)"""
    src = open(os.path.join(ROOT, "bench.py")).read()
    for key in ('"metric"', '"value"', '"unit"', '"n_gpus"', '"steps"', '"warmup"', '"ms_per_step"', '"higher_is_better"',
                '"scaling"', '"vs_baseline"', '"dtype"', '"data"', '"config"', '"roofline"', '"cpu_baseline"', '"clocks"',
                '"gpu_launches"', '"e2e"', '"h2d_bytes_per_step"', '"d2h_bytes_per_step"', '"impl"'):
        assert key in src, key


def test_reference_arm_runs_and_matches_the_gpu_arms_config():
    """the CPU arm on a tiny step count: same `config` as the GPU arm builds (VERDICT r01: same_config was false),
    one JSON line on stdout, sane scaling keys"""
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, env=dict(os.environ, SSPSD_BENCH_CPU_SAMPLES="4000000"))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    out = json.loads(lines[0])
    sys.path.insert(0, ROOT)
    import bench
    assert out["impl"] == "reference" and out["config"] == bench.config_dict(1)
    assert out["cpu_baseline"]["kind"] == "port" and out["cpu_baseline"]["cores"] == 1 and out["value"] > 1
    assert out["e2e"]["h2d_bytes_per_step"] == 0 and "parity_note" in out
    for key in ("sustained_2s", "timechunk", "e2e_small_calls", "e2e_frames", "cpu_baseline_n512", "value_readout_every_step"):
        assert '"%s"' % key in open(os.path.join(ROOT, "bench.py")).read()


def test_bench_dump_outputs_layout(tmp_path):
    """--dump-outputs: one float32 spectrum and one float64 break table per channel of the readout"""
    import sys

    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from stabilizer_stream_b200 import Break
    breaks = [Break(0, False, 0, 0, range(0, 0), 4096, 64, 10, 0),
              Break(0, True, 3, 0xFFFFFFFF, range(0, 1639), 4096, 8, 7, 1 << 40),
              Break(1639, True, 97655, 0xFFFFFFFF, range(205, 2049), 4096, 1, 2048, 200_000_000)]
    p = np.linspace(1, 2, 1639 + 1844, dtype=np.float32)
    bench.dump_outputs(str(tmp_path / "out"), [(p, breaks), (np.zeros(0, np.float32), [])])
    assert sorted(os.listdir(tmp_path / "out")) == ["breaks_ch0.npy", "breaks_ch1.npy", "psd_ch0.npy", "psd_ch1.npy"]
    got = np.load(tmp_path / "out" / "psd_ch0.npy")
    assert got.dtype == np.float32 and np.array_equal(got, p)
    b = np.load(tmp_path / "out" / "breaks_ch0.npy")
    assert b.dtype == np.float64 and b.shape == (3, len(bench.BREAK_FIELDS))
    assert b[1, -1] == 1 << 40
    assert b[2].tolist() == [1639, 1, 97655, 0xFFFFFFFF, 205, 2049, 4096, 1, 2048, 200_000_000]
    assert np.load(tmp_path / "out" / "breaks_ch1.npy").shape == (0, len(bench.BREAK_FIELDS))


def test_bench_rejects_bad_arguments():
    import subprocess
    import sys
    for argv in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "x"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and not r.stdout, (argv, r.stderr[-500:])
