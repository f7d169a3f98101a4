"""The library's kernels executed on the CPU from their own CUDA source text: tests/host/build_emu.py compiles every
translation unit of infercnv_b200/csrc with g++ against a host emulation of the CUDA execution model
(tests/host/emu/cuda_runtime.h: the threads of a block are fibers; __syncthreads, warp shuffles / reductions and atomics
have their CUDA semantics; a divergent barrier or a live-lock aborts; fresh device and shared memory is poisoned), with
synchronous stand-ins for the few inline-PTX copy primitives (TMA bulk copy + mbarrier, cp.async), and
tests/host/run_emulated.py runs the SAME parity tests the B200 box runs (-m gpu) against that build in a subprocess.

Test infrastructure only: it exercises the kernels' index arithmetic, barriers, shared-memory hand-offs and memory
accesses without a GPU - the fused cell pipeline, both Viterbi kernels with the certificate / re-run logic, the median
filter, and the kernels of the widened rows.  It says nothing about performance, floating-point contraction differs
from nvcc's in the last bit (the tests' tolerances are unchanged), and the package never loads the emulated library
(tests/test_capi_symbols.py)."""
import os
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(shutil.which("g++") is None and not os.path.exists("/usr/bin/g++"), reason="no host compiler")
@pytest.mark.parametrize("order", ["forward", "reverse"])
def test_gpu_parity_tests_pass_under_the_host_emulation(order):
    """`order` = the order in which the emulation resumes the runnable threads of a block (EMU_ORDER; "random:<seed>"
    also exists): results that depend on it would mean a data race - a missing barrier or an unsynchronised hand-off
    through shared memory - in one of the kernels."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "host", "run_emulated.py")], capture_output=True, text=True,
                       timeout=1500, env=dict(os.environ, EMU_ORDER=order))
    tail = "\n".join(r.stdout.splitlines()[-25:]) + r.stderr[-2000:]
    assert r.returncode == 0, tail
    assert " passed" in r.stdout and "failed" not in r.stdout, tail


@pytest.mark.skipif(shutil.which("g++") is None and not os.path.exists("/usr/bin/g++"), reason="no host compiler")
@pytest.mark.parametrize("env", [{"ICNV_VFAST_WARPS": "24"}, {"ICNV_VFAST_WARPS": "20"}, {"ICNV_HMM_MODE": "2"},
                                 {"ICNV_CELL_PADQ": "0"}, {"ICNV_CELL_KERNEL": "4"}, {"ICNV_MF_KERNEL": "2"}, {"ICNV_MF_KERNEL": "5"}], ids=lambda e: "-".join(f"{k}={v}" for k, v in e.items()))
def test_kernel_variants_behind_the_tuning_switches_under_the_host_emulation(env):
    """The variants DESIGN.md section 8 lists (Viterbi occupancy variants, the single-precision first pass, the ping-pong layout of the two-buffer cell
    pipeline and the single-buffer v4 kernel at gene counts where v3 is the default) through the parity tests of the path
    they replace."""
    pick = "viterbi and not scale and not oligo and not device_resident" if ("ICNV_VFAST_WARPS" in env or "ICNV_HMM_MODE" in env) else \
        ("median_filter" if "ICNV_MF_KERNEL" in env else "golden or slow_paths or smooth_lengths or known or padded_q or benchmark_layout")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "host", "run_emulated.py"),
                        os.path.join(ROOT, "tests", "test_gpu_parity.py"), "-k", pick], capture_output=True, text=True, timeout=1500,
                       env=dict(os.environ, **env))
    tail = "\n".join(r.stdout.splitlines()[-25:]) + r.stderr[-2000:]
    assert r.returncode == 0, tail
    assert " passed" in r.stdout and "failed" not in r.stdout, tail


@pytest.mark.skipif(shutil.which("g++") is None and not os.path.exists("/usr/bin/g++"), reason="no host compiler")
def test_differential_fuzz_of_edge_shapes_under_the_host_emulation():
    """Random small shapes - single genes / cells, one-gene chromosomes, windows longer than a chromosome, constant and
    tie-dominated columns, groups of one - through smooth block, centring, both Viterbi arithmetics (cells and groups,
    i6 and i3), median filter and region calling, each against the oracle (tests/host/fuzz_emulated.py)."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "host", "fuzz_emulated.py"), "40", "20260923"],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "40 cases ok" in r.stdout, r.stdout[-1500:] + r.stderr[-1500:]


@pytest.mark.skipif(shutil.which("g++") is None and not os.path.exists("/usr/bin/g++"), reason="no host compiler")
@pytest.mark.parametrize("world", [1, 2])
def test_engine_and_multi_rank_path_under_the_host_emulation(world):
    """infercnv_b200/device.py (Engine) on CPU tensors against the emulated library: one rank against the oracle
    (smooth block, HMM, i3 mu/sigma, device-resident consensus and regions incl. a strided state matrix, median filter);
    two gloo ranks - the sharded smooth block with its all-gathered partial sums, the HMM, mu/sigma and the all-reduced
    region consensus - bitwise equal to the single-rank run (what tools/check_multigpu.py checks over NCCL)."""
    cmd = [sys.executable, os.path.join(ROOT, "tests", "host", "engine_emulated.py")] + (["--world", str(world)] if world > 1 else [])
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
    assert ("BITWISE EQUAL" in r.stdout) if world > 1 else ("equal to the oracle" in r.stdout), r.stdout[-1500:]


@pytest.mark.skipif(shutil.which("g++") is None and not os.path.exists("/usr/bin/g++"), reason="no host compiler")
@pytest.mark.parametrize("world,config", [(1, "c3"), (2, "c3"), (2, "c4")])
def test_bench_script_reaches_its_json_line_under_the_host_emulation(world, config, tmp_path):
    """bench.py itself (workload, warm-up + timed loop, e2e through the host ABI, max over ranks, JSON assembly, the
    --dump-outputs files) at a toy size on the CPU, for 1 rank and for 2 ranks launched the way torchrun launches them.
    The numbers are meaningless (emulation, wall clock); the contract keys and the multi-rank control flow are what is
    checked."""
    import json
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    dump = tmp_path / "outputs"
    args = ["--gpus", str(world), "--config", config, "--steps", "2", "--warmup", "3", "--ref-sample-cells", "16",
            "--dump-outputs", str(dump)] + \
        (["--cells", "64", "--genes", "1100"] if config == "c3" else ["--cells", "700", "--genes", "260"])
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), LOCAL_RANK=str(r), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1",
                   MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "host", "bench_emulated.py")] + args,
                                      stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env))
    outs = [p.communicate(timeout=900) for p in procs]
    assert all(p.returncode == 0 for p in procs), outs[0][1][-1500:] + outs[-1][1][-1500:]
    lines = [ln for ln in outs[0][0].splitlines() if ln.startswith("{")]
    assert len(lines) == 1 and all(not o[0].strip() for o in outs[1:])          # ONE JSON line, from rank 0
    j = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline"):
        assert key in j, key
    assert j["n_gpus"] == world and j["steps"] == 2 and j["warmup"] == 3 and j["value"] > 0 and j["gpu_launches"] > 0
    assert j["dtype"] == "f64" and j["scaling"] == "strong" and "workload" in j["config"] and "model" not in j["config"]
    assert j["config"]["cells"] == (64 if config == "c3" else 700) and j["config"]["config"] == config
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(j["roofline"]) and j["roofline"]["bound"] == "hbm"
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(j["e2e"]) and j["e2e"]["h2d_bytes_per_step"] > 0
    if world == 1:
        assert {"value", "unit", "cores", "kind", "sample"} <= set(j["cpu_baseline"])
    import numpy as np
    got = {f.name: np.load(f) for f in dump.iterdir()}
    assert set(got) == {"cells.npy", "smoothed.npy", "states.npy"} | ({"median_filtered.npy"} if config == "c4" else set())
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())
    n, G = j["config"]["cells"], j["config"]["genes"]
    assert np.array_equal(got["cells.npy"], np.arange(n))         # the toy sizes fit the dump budget whole
    assert all(v.shape == (n, G) for k, v in got.items() if k != "cells.npy")
    # every row against the oracle on the seeded workload at its global cell index (also checks the 2-rank gather order);
    # the HMM and the median filter are re-run on the dumped smoothed matrix, so only their own arithmetic is compared
    import bench
    from oracle import oracle as orc
    seed = bench.SEED0 + bench.CONFIGS[config]["index"]
    cs, cl = bench.chr_layout(G)
    refs = bench.ref_groups_global(n)
    want = orc.smooth_block(orc.synth(G, cs, cl, np.arange(n), n, seed), cs, cl, refs)
    S = np.asfortranarray(got["smoothed.npy"].T)
    assert float(np.max(np.abs(S - want) / np.abs(want))) < 1e-11
    if config == "c3":
        Pi, delta, mean, sd = bench.i6_model()
    else:
        Pi, delta, mean, sd = bench.i3_model(*orc.mean_sd_over_cells(S, np.concatenate(refs)))
    assert np.array_equal(got["states.npy"].T, orc.viterbi_matrix(S, cs, cl, Pi, delta, mean, sd))
    if config == "c4":
        lists = bench.subclusters_global(n, seed) + refs
        assert np.allclose(got["median_filtered.npy"].T, orc.median_filter(S, cs, cl, lists, 7), rtol=0, atol=1e-15)


def test_the_package_cannot_reach_the_emulated_library():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "infercnv_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".c", ".R")):
                src = open(os.path.join(dirpath, f), errors="replace").read()
                assert "_emu" not in src and "cuda_emu" not in src and "ICNV_EMU" not in src, f
