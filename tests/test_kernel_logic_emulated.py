"""Kernel LOGIC in the GPU-less container: the parity tests of tests/test_gpu_parity.py and the driver tests of
tests/test_driver.py are re-run against tests/cuda_emu/libtfbs_emu.so, i.e. the product's own kernel sources compiled with g++ on
top of a CUDA-on-host shim (every CUDA thread is a fiber, see tests/cuda_emu/include/cuda_runtime.h).

This is test infrastructure, not a product path: nothing under find_tfbs_b200/ builds, links or loads the emulated library, it is
not built by __graft_entry__.build(), and libtfbs_b200.so still fails without a B200 (test_abi.py::test_no_gpu_fails_loudly).
What it buys: indexing / hashing / bookkeeping bugs in the kernels show up here, before any GPU time is spent; races, memory
ordering and speed are only visible to the `-m gpu` run on the B200."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "cuda_emu")


@pytest.fixture(scope="module")
def emu_env():
    subprocess.check_call(["make", "-C", EMU, "-j2"], stdout=subprocess.DEVNULL)
    env = dict(os.environ)
    env["TFBS_B200_LIB"] = os.path.join(EMU, "libtfbs_emu.so")
    env["TFBS_B200_DRIVER"] = os.path.join(EMU, "find-tfbs-emu")
    env["TFBS_TEST_SCALE"] = "0.004"  # the full-size property test shrinks to 40 regions under emulation
    return env


def run_marked_gpu_tests(env, path, select, workers=4):
    cmd = [sys.executable, "-m", "pytest", path, "-q", "-x", "-m", "gpu", "-p", "no:cacheprovider"]
    try:
        import xdist  # noqa: F401  (the emulation is single-threaded per process: spread the cases over a few processes)
        cmd += ["-n", str(workers)]
    except ImportError:
        pass
    if select:
        cmd += ["-k", select]
    r = subprocess.run(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-4000:]
    assert " passed" in r.stdout and "failed" not in r.stdout
    return r.stdout


def test_product_binding_never_loads_the_emulator():
    """The override is an environment variable read by the ctypes binding only; the product sources do not mention the emulator."""
    for dp, _, fs in os.walk(os.path.join(ROOT, "find_tfbs_b200")):
        for f in fs:
            if f.endswith((".py", ".cu", ".cpp", ".hpp", ".h")) or f == "Makefile":
                text = open(os.path.join(dp, f), errors="replace").read()
                assert "libtfbs_emu" not in text and "cuda_emu/include" not in text, os.path.join(dp, f)
    assert "cuda_emu" not in open(os.path.join(ROOT, "__graft_entry__.py")).read()


def test_emulator_selftest(tmp_path):
    """The shim itself: block barriers, full-warp and 8-lane-group shuffles with divergent trip counts, ballot with exited lanes,
    atomics, dynamic shared memory (tests/cuda_emu/selftest.cpp)."""
    exe = str(tmp_path / "emu_selftest")
    subprocess.check_call(["g++", "-O1", "-g", "-std=c++17", "-I", os.path.join(EMU, "include"), "-x", "c++", os.path.join(EMU, "selftest.cpp"), "-o", exe])
    r = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    assert r.returncode == 0 and "selftest ok" in r.stdout, r.stdout


def test_parity_suite_on_emulated_kernels(emu_env):
    """Every parity case except the two large ones (minutes under emulation): rows, hit lists, groupings and counters of the
    emulated kernels equal the oracle's, in both scan modes."""
    out = run_marked_gpu_tests(emu_env, "tests/test_gpu_parity.py", "not config2_slice and not config3_like and not config3_full")
    assert "23 passed" in out or " passed" in out


def test_driver_on_emulated_kernels(emu_env):
    """The C++ driver end to end on the CPU: the reference's two integration outputs (main.rs:548-568) and the synthetic file sets."""
    run_marked_gpu_tests(emu_env, "tests/test_driver.py", "", workers=2)
    run_marked_gpu_tests(emu_env, "tests/test_bcf_edge_cases.py", "", workers=2)
    run_marked_gpu_tests(emu_env, "tests/test_multi_gpu.py", "", workers=2)  # two processes, shared-memory arenas; --devices 0,0


CONTRACT_KEYS = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
                 "config", "roofline", "e2e", "gpu_launches", "clocks", "cpu_baseline")


def test_bench_control_flow_dry_run(emu_env, tmp_path):
    """bench.py end to end with torch.cuda stubbed and the emulated library (tests/cuda_emu/run_bench_emulated.py): the one JSON
    line carries every contract key and internally consistent counters: the north-star workload (configs[2], strong scaling), the
    shared-memory gather of the grouped rows, the sustained run, the configs[1] secondary object, and --dump-outputs writes the
    oracle's rows of the same seeded block.  The numbers themselves mean nothing."""
    import json
    import numpy as np
    import parity_helpers as hp
    from find_tfbs_b200 import binding, synth
    r = subprocess.run([sys.executable, os.path.join(EMU, "run_bench_emulated.py"), "--scale", "0.0004", "--steps", "2", "--warmup", "1",
                        "--cpu-seconds", "0.2", "--no-full-scan", "--sustain-seconds", "0.01", "--no-driver", "--dump-outputs", str(tmp_path)],
                       cwd=ROOT, env=emu_env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for k in CONTRACT_KEYS:
        assert k in d, k
    assert d["metric"] == "pwm_cells_per_s" and d["n_gpus"] == 1 and d["steps"] == 2 and d["higher_is_better"] is True
    assert d["scaling"] == "strong" and d["config"]["workload"].startswith("configs[2]") and d["config"]["samples"] == 2504
    rf = d["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic", "hbm"):
        assert k in rf, k
    assert rf["hbm"]["algorithmic_bytes_per_step"] > 0 and rf["cells_per_step"] == d["evaluated_cells_per_step"]
    assert d["nominal_cells_per_step"] >= d["executed_cells_per_step"] >= d["evaluated_cells_per_step"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["gpu_launches"] > 0
    assert d["e2e"]["gathered_on_rank0"]["rows_last_step"] == d["rows_per_step"]
    assert d["sustained"]["steps"] >= 2 and d["secondary"]["config"]["workload"].startswith("configs[1]")
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    dump = {f[:-len(".npy")]: np.load(str(tmp_path / f)) for f in os.listdir(str(tmp_path))}
    assert all(a.dtype in (np.float32, np.float64) for a in dump.values())
    assert sum(os.path.getsize(str(tmp_path / f)) for f in os.listdir(str(tmp_path))) <= 64 << 20
    pats, blk = synth.config3(scale=0.0004, seed=3)
    o = hp.run_oracle(binding.PatternSet(pats), blk)
    assert len(o["region"]) == d["rows_per_step"] > 0 and np.array_equal(dump["rows"], np.arange(len(o["region"])))
    for k in ("region", "inner", "pattern_id", "vmin", "vmax"):
        assert np.array_equal(dump[k], o[k]), k
    dense = dump["dense_rows"].astype(np.int64)
    assert np.array_equal(dump["left"], o["left"][dense]) and np.array_equal(dump["right"], o["right"][dense])
    assert len(dump["n_groups"]) == blk.n_regions and dump["n_groups"].min() >= 1


def test_bench_reference_arm():
    """`bench.py --impl reference` needs no GPU: the CPU restatement on the host cores, same metric / config keys, impl = reference."""
    import json
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--scale", "0.0004", "--steps", "1", "--warmup", "1",
                        "--ref-seconds-per-step", "0.2"], cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.strip()][-1])
    assert d["impl"] == "reference" and d["metric"] == "pwm_cells_per_s" and d["value"] > 0 and d["gpu_launches"] == 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"]


def test_bench_configs3_dry_run(emu_env):
    """`bench.py --workload configs3` (sample blocks, tfbs_merge_sample_blocks, roofline_k1) end to end on the emulated library with a
    tiny cohort: control flow and the contract keys only."""
    import json
    r = subprocess.run([sys.executable, os.path.join(EMU, "run_bench_emulated.py"), "--workload", "configs3", "--c3-regions", "2", "--c3-samples", "96",
                        "--c3-block", "48", "--steps", "1", "--warmup", "1", "--cpu-seconds", "0.2"], cwd=ROOT, env=emu_env,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for k in CONTRACT_KEYS:
        assert k in d, k
    assert d["config"]["workload"].startswith("configs[3]") and d["config"]["sample_blocks"] == 2
    k1 = d["roofline_k1"]
    assert k1["bound"] == "hbm" and k1["algorithmic_bytes_per_step"] > 0 and 0 < k1["frac"]
    assert d["e2e"]["rows_all_keys"] >= d["e2e"]["rows_kept"] == d["rows_per_step"] and d["e2e"]["d2h_bytes_per_step"] > 0
    assert d["nominal_cells_per_step"] >= d["executed_cells_per_step"] >= d["evaluated_cells_per_step"] > 0
