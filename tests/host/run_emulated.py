#!/usr/bin/env python
"""TEST INFRASTRUCTURE: run the GPU parity tests (the same test functions the B200 box runs with -m gpu) against
tests/host/_build/libinfercnv_b200_emu.so, i.e. against the kernels' own source text executed by the host emulation of
the CUDA execution model in tests/host/emu/cuda_runtime.h.  A separate process, because it points the ctypes loader at
the emulated library before anything is loaded; the package itself has no such switch.

    python tests/host/run_emulated.py [--full] [pytest args]

Default: the cell-pipeline launch map, the widened rows (tests/test_gpu_widen_*.py), the ops mirror and the hot-path
parity tests minus the four that take more than ten seconds each under emulation; --full adds those (about 2 minutes more).
Never run: tests that need torch device tensors (Engine) and the full-size property tests (10^7 - 10^8 cell-genes).
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import build_emu  # noqa: E402
import pytest  # noqa: E402

from infercnv_b200 import _lib  # noqa: E402

_lib.LIB_PATH = build_emu.build()
assert _lib._lib is None

full = "--full" in sys.argv
extra = [a for a in sys.argv[1:] if a != "--full"]
NEVER = ["test_device_resident_states_from_the_viterbi_kernel_to_regions", "test_full_size_round_trip_and_run_count",
         "test_engine_slab_pipelined_host_path_is_bit_identical", "test_engine_stage_flag_combinations",
         "test_engine_strided_misaligned_and_indexed_inputs_are_bitwise"]
SLOW = ["test_multi_slab_host_pipeline_and_fused_call", "test_oligodendroglioma_hmm_cells_and_samples",
        "test_oligodendroglioma_smooth_block_two_ref_groups", "test_viterbi_modes_agree_with_oracle_at_scale"]
files = ["test_gpu_cell_pipeline_map.py", "test_gpu_ops_mirror.py", "test_gpu_parity.py", "test_gpu_widen_denoise.py", "test_gpu_widen_elementwise.py",
         "test_gpu_widen_hmm_per_chr.py", "test_gpu_widen_ingest.py", "test_gpu_widen_regions.py"]
skip = NEVER + ([] if full else SLOW)
args = [os.path.join(ROOT, "tests", f) for f in files]
args += ["-m", "gpu", "-q", "-x", "-p", "no:cacheprovider", "-k", " and ".join("not " + d for d in skip)] + extra
sys.exit(pytest.main(args))
