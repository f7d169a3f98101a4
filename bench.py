#!/usr/bin/env python
"""bench.py - cells x genes / s through the smooth block + HMM (BASELINE.json metric).

    python bench.py [--config c2|c3|c4|c5] [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over the workload: run() steps 4, 8-12, 14 (fused smooth block) followed by
step 17 (per-cell Viterbi) on a synthetic depth-normalised matrix; c4 adds apply_median_filtering.

Configs are BASELINE.json's (SURVEY section 8d), seeds 20260922 + index:
  c2  10 000 cells x 10 000 genes, i6                      (the reference's CPU-runnable size)
  c3  100 000 x 10 000, i6   <- DEFAULT: the configuration the metric is quoted on; fits one B200 (8 GB in, 8 GB out)
  c4  100 000 x 10 000, i3 (mu / sigma from the reference cells) + apply_median_filtering over 50-500-cell subclusters
  c5  500 000 x 20 000, i6, 8 x B200; with fewer ranks the same shape at 62 500 cells per rank (labelled as such)
N > 1 (torchrun, one rank per GPU) STRONG-scales the configuration: the cells are cut into N shards, the only exchange
is one NCCL all-gather of reference chunk sums behind each of the two reference-mean steps (c4: plus the mu / sigma
pairs and the 4-cell halos of the reference groups for the median filter).  `--scaling weak` keeps the per-rank cells.
Inputs are far larger than the 126 MB L2 (>= 0.8 GB per pass), so consecutive timed steps cannot hit in cache.

Prints ONE JSON line (rank 0).  `value` = device-resident throughput (CUDA events, max over ranks); `e2e` = the same
metric through the host-pointer C ABI from PAGEABLE host memory (what an R matrix is), H2D and D2H inside the timed
region; `roofline` = the dominant kernel against measured HBM bandwidth; `cpu_baseline` = the C oracle port on the host
cores over a bounded sample.

`--impl reference` times the CPU restatement of the reference's algorithm (oracle/; the reference itself is interpreted
R: when `Rscript` is on the PATH and ICNV_REFERENCE_R_DIR names the reference's R/ directory the arm source()s its
sources instead, kind "reference-R") with
all host threads on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "cells x genes / s (smooth block + HMM)"
UNIT = "cell-genes/s"
CONFIGS = {
    "c2": {"index": 1, "cells": 10_000, "genes": 10_000, "hmm": "i6", "median_filter": False, "steps": 400,
           "what": "BASELINE configs[1]"},
    "c3": {"index": 2, "cells": 100_000, "genes": 10_000, "hmm": "i6", "median_filter": False, "steps": 40,
           "what": "BASELINE configs[2], the configuration the metric is quoted on"},
    "c4": {"index": 3, "cells": 100_000, "genes": 10_000, "hmm": "i3", "median_filter": True, "steps": 8,
           "what": "BASELINE configs[3]"},
    "c5": {"index": 4, "cells": 500_000, "genes": 20_000, "hmm": "i6", "median_filter": False, "steps": 8, "shards": 8,
           "what": "BASELINE configs[4]"},
}
CHR_TEMPLATE = [852, 615, 535, 288, 420, 453, 458, 297, 349, 363, 514, 472, 162, 301, 274, 397, 546, 126, 545, 239, 90,
                212]  # oligodendroglioma example, SURVEY section 8(d)
I6_MEAN = np.array([0.41234766, 0.84075773, 1.01693983, 1.12238786, 1.23842619, 1.44298781])
I6_SD = np.array([0.028893, 0.164549, 0.105553, 0.190574, 0.244093, 0.290072])
SEED0 = 20260922
SEED = SEED0 + 1          # c2 (tools/ and tests import this)
BYTES_MF = 16.0              # median filter: 8 read + 8 written
# algorithmic HBM bytes per cell-gene (SURVEY section 8d, FP64 parity mode)
BYTES_SMOOTH = 16.0          # + 16 per reference-cell gene for the two reference pre-passes
BYTES_HMM = 9.0              # 8 read + 1 state byte written


def chr_layout(G: int):
    t = np.array(CHR_TEMPLATE, dtype=np.float64)
    lens = np.floor(t * G / t.sum()).astype(np.int64)
    lens[0] += G - lens.sum()
    starts = np.concatenate([[0], np.cumsum(lens)[:-1]])
    return starts.astype(np.int32), lens.astype(np.int32)


def ref_groups_global(C_total: int):
    """first 10 % of the cells are reference cells in two groups (6 % / 4 %)."""
    a, b = int(round(0.06 * C_total)), int(round(0.10 * C_total))
    return [np.arange(0, a, dtype=np.int64), np.arange(a, b, dtype=np.int64)]


def ncu_traffic(kernel, config, world):
    """DRAM bytes per launch of `kernel` on `config` from the committed ncu --set full capture
    (profiles/r02_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one launch), or None."""
    if world != 1:
        return None
    try:
        return float(json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))[config][kernel]["dram_bytes_per_launch"])
    except Exception:
        return None


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Clock / throttle-reason sampling during the timed region (B200_PROFILING.md clocks line).

    Two sources run side by side from before the warm-up until after the timed region: an `nvidia-smi -lms 20`
    child writing CSV to a temp file, and an NVML polling thread in this process (pynvml, same counters).  Samples
    are selected by wall-clock stamp inside [t0, t1]; nvidia-smi rows win when any landed there, else the NVML
    thread's, else everything captured under the (identical) warm-up load - `window` / `source` say which."""

    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    NVML_BITS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, gpu_index: int):
        self.proc = None
        self.path = None
        self.gpu = gpu_index
        self.nvml_rows = []          # (stamp, sm_mhz, sm_max_mhz, reason mask)
        self._stop = None
        self._thread = None

    def _nvml_loop(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                getattr(pynvml, "nvmlDeviceGetCurrentClocksThrottleReasons")
            while not self._stop.is_set():
                try:
                    self.nvml_rows.append((time.time(), float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)), mx,
                                           int(reasons(h))))
                except Exception:
                    pass
                self._stop.wait(0.02)
        except Exception:
            return

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
        try:
            import threading
            self._stop = threading.Event()
            self._thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self._thread.start()
        except Exception:
            self._thread = None

    @staticmethod
    def _stamp(text):
        import datetime
        try:
            return datetime.datetime.strptime(text.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except ValueError:
            return None

    def stop(self, t0=None, t1=None):
        """t0 / t1: wall-clock bounds (time.time()) of the timed region.  The nvidia-smi child is left running for
        up to a second past t1 so that its stdio buffer holding the timed region's rows reaches the file before it
        is terminated."""
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if t1 is not None:
            time.sleep(max(0.0, min(1.0, t1 + 1.0 - time.time())))
        if self._thread is not None:
            self._stop.set()
            self._thread.join(timeout=2)
        smi = []                     # (stamp, sm, max, [reason names])
        if self.proc is not None:
            try:
                self.proc.terminate()      # exact PID we started
                self.proc.wait(timeout=5)
            except Exception:
                pass
            try:
                for line in open(self.path):
                    r = line.strip().split(", ")
                    if len(r) < 9:
                        continue
                    try:
                        smi.append((self._stamp(r[0]), float(r[1]), float(r[2]),
                                    [n for n, v in zip(self.NAMES, r[5:9]) if v.strip().lower().startswith("active")]))
                    except ValueError:
                        continue
                os.unlink(self.path)
            except Exception:
                pass
        nvml = [(t, sm, mx, [n for n, b in self.NVML_BITS.items() if mask & b]) for t, sm, mx, mask in self.nvml_rows]

        def inside(rows):
            if t0 is None or t1 is None:
                return rows
            return [r for r in rows if r[0] is not None and t0 <= r[0] <= t1]
        for rows, source, window in ((inside(smi), "nvidia-smi", "timed region"),
                                     (inside(nvml), "nvml", "timed region"),
                                     (smi, "nvidia-smi", "warm-up + timed region (no sample was stamped inside the timed region)"),
                                     (nvml, "nvml", "warm-up + timed region (no sample was stamped inside the timed region)")):
            if rows:
                out = {"sm_mhz": float(np.median([r[1] for r in rows])), "sm_max_mhz": float(max(r[2] for r in rows)),
                       "reasons": sorted({n for r in rows for n in r[3]}), "samples": len(rows), "window": window,
                       "source": source}
                break
        return out


# ---- workload -------------------------------------------------------------------------------------------------------
def resolve_config(args, world):
    """-> (cfg, G, C_total, seed, label).  Strong scaling keeps the configuration's cells; c5 below its 8 shards (and
    `--scaling weak`) keep the cells PER RANK instead and say so."""
    cfg = CONFIGS[args.config]
    G = args.genes or cfg["genes"]
    shards = cfg.get("shards", 1)
    per_rank = cfg["cells"] // shards
    note = ""
    if args.cells:
        C_total = args.cells
        note = f" (--cells {args.cells})"
    elif args.scaling == "weak":
        C_total = per_rank * world
        note = f" (weak scaling: {per_rank} cells per rank)"
    elif shards > 1 and world < shards:
        C_total = per_rank * world
        note = f" ({world} of the configuration's {shards} shards of {per_rank} cells: {cfg['cells']} cells need {shards} GPUs)"
    else:
        C_total = cfg["cells"]
    return cfg, G, C_total, SEED0 + cfg["index"], note


def subclusters_global(C_total: int, seed: int):
    """c4: the observation cells (behind the first 10 %) form 4 groups, each cut into subclusters of 50-500 cells listed
    in index order (SURVEY section 8d)."""
    rng = np.random.default_rng(seed)
    first = int(round(0.10 * C_total))
    edges = np.linspace(first, C_total, 5).astype(np.int64)
    out = []
    for a, b in zip(edges[:-1], edges[1:]):
        pos = int(a)
        while pos < b:
            n = int(rng.integers(50, 501))
            if b - (pos + n) < 50:      # no stub shorter than 50 cells at a group's end
                n = int(b - pos)
            out.append(np.arange(pos, pos + n, dtype=np.int64))
            pos += n
    return out


def workload_config(args, cfg, G, C_total, world, note):
    per = -(-C_total // world)
    return {"workload": f"{args.config}: synthetic {C_total} cells x {G} genes, 22 chromosomes, window 101, {cfg['hmm']} HMM per cell"
                        + (" + apply_median_filtering(window 7) over 50-500-cell subclusters and the reference groups" if cfg["median_filter"] else "")
                        + f" ({cfg['what']}){note}",
            "config": args.config, "cells": C_total, "cells_per_gpu": per, "genes": G, "window_length": 101,
            "hmm": f"{cfg['hmm']} per cell, t=1e-6" + (", mu / sigma from the reference cells, i3_p_val 0.05" if cfg["hmm"] == "i3" else ""),
            "reference_cells": "first 10 % in two groups (6 % / 4 %)", "sharding": f"cells over {world} GPU(s)",
            "l2": "inputs (%.2f GB/GPU/pass) exceed the 126 MB L2; no explicit flush" % (per * G * 8 / 1e9)}


def i6_model():
    from infercnv_b200.hmm import CNV_LEVELS, get_HMM
    Pi, delta, _, _ = get_HMM({k: {"mean": m, "sd": s} for k, m, s in zip(CNV_LEVELS, I6_MEAN, I6_SD)}, 1e-6)
    return Pi, delta, I6_MEAN, I6_SD


def i3_model(mu, sigma):
    from infercnv_b200.hmm import i3HMM_get_HMM, i3_mean_delta
    return i3HMM_get_HMM({"mu": mu, "sigma": sigma, "mean_delta": i3_mean_delta(sigma, 0.05), "KS_delta": None}, 1e-6)


# ---- CPU arm --------------------------------------------------------------------------------------------------------
def usable_cpus() -> int:
    """Host threads this process may really run at once: the affinity mask, cut by the container's CPU quota (cgroup v2
    cpu.max / v1 cfs quota).  omp_get_num_procs() alone over-reports inside a quota-limited container, and 2 x the quota
    in spinning OpenMP threads is many times slower than the quota itself; torchrun's OMP_NUM_THREADS=1 under-reports."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)


def pick_cpu_threads(cfg, G, C_total, seed, args):
    """All the host threads the port can USE: time one pass on a small sample at n, n/2 and n/4 threads (n = usable CPUs)
    and keep the fastest - SMT siblings and memory bandwidth make 'every logical CPU' the slowest choice on some boxes."""
    n = usable_cpus()
    cands = sorted({max(1, n), max(1, n // 2), max(1, n // 4)}, reverse=True)
    if len(cands) == 1:
        return cands[0], {cands[0]: None}
    X, cs, cl, ref_local, lists, _, _ = cpu_sample(args, cfg, G, C_total, seed, min(C_total, 8 * n), n)
    rates = {}
    for t in cands:
        step = cpu_step_fn(cfg, X, cs, cl, ref_local, lists, t)
        t0 = time.perf_counter()
        step()
        rates[t] = G * X.shape[1] / (time.perf_counter() - t0)
    best = max(rates, key=rates.get)
    return best, rates


def cpu_sample(args, cfg, G, C_total, seed, n_want, nt=None):
    """A bounded sample of the workload for the CPU arm: (X, reference groups, median-filter lists) in sample-local
    columns.  i6 configs: every stride-th cell.  c4: a 10 % slice of reference cells plus whole subclusters, so that the
    median filter sees real blocks.  The generator is the C twin of the device one (oracle/, no product library)."""
    from oracle import oracle as orc
    cs, cl = chr_layout(G)
    nt = nt or usable_cpus()
    refs_g = ref_groups_global(C_total)
    lists = None
    if not cfg["median_filter"]:
        stride = max(1, C_total // n_want)
        cells = np.arange(0, C_total, stride, dtype=np.int64)[:n_want]
        what = f"{len(cells)} cells (every {stride}th of {C_total})"
    else:
        n_ref = max(2, n_want // 10)
        a = max(1, int(round(n_ref * 0.6)))
        picked = [refs_g[0][:a], refs_g[1][:n_ref - a]]
        subs, tot = [], n_ref
        for s in subclusters_global(C_total, seed):
            if tot >= n_want:
                break
            subs.append(s)
            tot += len(s)
        cells = np.concatenate(picked + subs)
        what = f"{len(cells)} cells ({n_ref} reference cells + {len(subs)} whole subclusters of {C_total})"
    X = orc.synth(G, cs, cl, cells, C_total, seed, nthreads=nt)
    ref_local = [np.flatnonzero(np.isin(cells, g)).astype(np.int32) for g in refs_g]
    ref_local = [g for g in ref_local if len(g)]
    if cfg["median_filter"]:
        lists, pos = [], sum(len(p) for p in picked)
        for s in subs:
            lists.append(np.arange(pos, pos + len(s), dtype=np.int32))
            pos += len(s)
        lists += ref_local
    return X, cs, cl, ref_local, lists, what, nt


def cpu_step_fn(cfg, X, cs, cl, ref_local, lists, nt):
    from oracle import oracle as orc
    Pi6, delta6 = orc.hmm_params(6)

    def step():
        S = orc.smooth_block(X, cs, cl, ref_local, apply_log=True, threshold=3.0, window=101, nthreads=nt)
        if cfg["hmm"] == "i6":
            orc.viterbi_matrix(S, cs, cl, Pi6, delta6, I6_MEAN, I6_SD, nthreads=nt)
        else:
            mu, sg = orc.mean_sd_over_cells(S, np.concatenate(ref_local))
            Pi3, d3, m3, s3 = i3_model(mu, sg)
            orc.viterbi_matrix(S, cs, cl, Pi3, d3, m3, s3, nthreads=nt)
        if cfg["median_filter"]:
            orc.median_filter(S, cs, cl, lists, 7, nthreads=nt)
    return step


def rscript_reference(args, cfg, G, C_total, seed):
    """The real reference, when the caller provides it: `Rscript` plus the reference's R/ directory named by
    ICNV_REFERENCE_R_DIR.  tools/reference_arm.R source()s the hot-path functions and times them on a sample written to
    a temp file.  Returns the JSON dict it printed, or None (no Rscript, or ICNV_REFERENCE_R_DIR unset)."""
    import shutil
    rs = shutil.which("Rscript")
    rdir = os.environ.get("ICNV_REFERENCE_R_DIR")
    script = os.path.join(ROOT, "tools", "reference_arm.R")
    if not rs or not rdir or not os.path.isdir(rdir) or not os.path.exists(script):
        return None
    try:
        n = min(C_total, 200)   # interpreted R: ~0.3-0.5 s per cell for the Viterbi alone
        X, cs, cl, ref_local, lists, what, _ = cpu_sample(args, cfg, G, C_total, seed, n)
        with tempfile.TemporaryDirectory() as td:
            X.T.astype("<f8").tofile(os.path.join(td, "x.bin"))      # cells contiguous = R column-major G x n
            np.savetxt(os.path.join(td, "chr_len.txt"), cl, fmt="%d")
            np.savetxt(os.path.join(td, "i6_mean.txt"), I6_MEAN, fmt="%.17g")
            np.savetxt(os.path.join(td, "i6_sd.txt"), I6_SD, fmt="%.17g")
            wl = lambda f, ls: open(os.path.join(td, f), "w").write("\n".join(" ".join(str(int(i) + 1) for i in g) for g in ls) + "\n")  # noqa: E731
            wl("refs.txt", ref_local)
            wl("lists.txt", lists or [])
            open(os.path.join(td, "meta.txt"), "w").write("\n".join([f"G={int(G)}", f"C={int(X.shape[1])}", f"hmm={cfg['hmm']}",
                                                                     f"median_filter={1 if cfg['median_filter'] else 0}",
                                                                     f"steps={max(1, min(args.steps, 2))}", f"rdir={rdir}"]) + "\n")
            r = subprocess.run([rs, script, td], capture_output=True, text=True, timeout=3000)
            line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            if r.returncode == 0 and line:
                d = json.loads(line[-1])
                d["sample"] = what
                return d
    except Exception as e:  # pragma: no cover
        print(f"[bench] Rscript arm failed ({e}); using the C port", file=sys.stderr)
    return None


def run_reference(args):
    """CPU arm: the reference's algorithm on the host cores over a bounded sample of the configured workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc
    orc.build()
    world = max(1, args.gpus)
    cfg, G, C_total, seed, note = resolve_config(args, world)
    steps = args.steps or 10
    args.steps = steps
    base = {"impl": "reference", "metric": METRIC, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": args.scaling_label, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, cfg, G, C_total, world, note)}
    r = rscript_reference(args, cfg, G, C_total, seed)
    if r is not None:
        value = float(r["cell_genes_per_s"])
        base.update({"value": value, "ms_per_step": float(r["ms_per_step"]),
                     "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "reference-R", "sample": r["sample"]},
                     "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                     "note": "the reference's own R functions source()d from its R/ directory; this path ignores num_threads (1 core)"})
        print(json.dumps(base))
        return
    nt, rates = pick_cpu_threads(cfg, G, C_total, seed, args)
    n_want = min(C_total, max(args.ref_sample_cells, 32 * nt))   # >= 32 cells per thread keeps every core fed
    X, cs, cl, ref_local, lists, what, nt = cpu_sample(args, cfg, G, C_total, seed, n_want, nt)
    step = cpu_step_fn(cfg, X, cs, cl, ref_local, lists, nt)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    value = G * X.shape[1] / dt
    base.update({"value": value, "ms_per_step": dt * 1e3,
                 "cpu_baseline": {"value": value, "unit": UNIT, "cores": nt, "kind": "port", "sample": f"{what} x {G} genes per step",
                                  "usable_cpus": usable_cpus(), "thread_count_trial_cell_genes_per_s": {str(k): v for k, v in rates.items()}},
                 "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                 "note": "reference = interpreted R (no Rscript + reference sources on this box); this arm is the C restatement in "
                         "oracle/ with OpenMP over cells on every host core (thread count set explicitly, not from OMP_NUM_THREADS) "
                         "- a best-case CPU line, the R path itself is single-threaded"})
    print(json.dumps(base))


def cpu_baseline(args, cfg, G, C_total, seed):
    """Oracle port on the host cores over a bounded sample (rank 0, N = 1 only), ~10 s."""
    nt, rates = pick_cpu_threads(cfg, G, C_total, seed, args)
    n_want = min(C_total, max(args.ref_sample_cells, 32 * nt))
    X, cs, cl, ref_local, lists, what, nt = cpu_sample(args, cfg, G, C_total, seed, n_want, nt)
    step = cpu_step_fn(cfg, X, cs, cl, ref_local, lists, nt)
    step()
    reps, t_total = 0, 0.0
    while t_total < 10.0 and reps < 50:
        t0 = time.perf_counter()
        step()
        t_total += time.perf_counter() - t0
        reps += 1
    return {"value": reps * G * X.shape[1] / t_total, "unit": UNIT, "cores": nt, "kind": "port",
            "sample": f"{what} x {G} genes, {reps} passes, {t_total:.1f} s", "usable_cpus": usable_cpus(),
            "thread_count_trial_cell_genes_per_s": {str(k): v for k, v in rates.items()}}


# ---- GPU arm --------------------------------------------------------------------------------------------------------
DUMP_BYTES = 60 << 20        # --dump-outputs writes at most this many bytes of array data


def dump_outputs(out_dir, cells, C_total, G, Y, states, F, world, rank):
    """--dump-outputs: what the timed path computed in its last step - the smoothed matrix, the HMM states and (c4) the
    median-filtered matrix - for a sample of cells drawn with a fixed seed, rows in global cell order, so that two builds
    can be compared output for output.  Every rank contributes the sampled cells it holds; rank 0 writes."""
    import torch
    import torch.distributed as dist
    per_cell = 8 + G * (8 + 4 + (8 if F is not None else 0))
    n = min(C_total, max(1, DUMP_BYTES // per_cell))
    pick = np.sort(np.random.default_rng(SEED0).choice(C_total, n, replace=False))
    rows = np.flatnonzero(np.isin(cells, pick))
    idx = torch.as_tensor(rows, device=Y.device)
    part = {"cells": np.asarray(cells)[rows].astype(np.float64), "smoothed": Y[idx].cpu().numpy(),
            "states": states[idx].cpu().numpy().astype(np.float32)}
    if F is not None:
        part["median_filtered"] = F[idx].cpu().numpy()
    parts = [part]
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, part)
    if rank != 0:
        return
    out = {k: np.concatenate([p[k] for p in parts]) for k in part}
    order = np.argsort(out["cells"], kind="stable")
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v[order])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS))
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=0, help="default: per config, sized for a timed region of about a second")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--cells", type=int, default=0, help="total cells (default: the configuration's)")
    ap.add_argument("--genes", type=int, default=0)
    ap.add_argument("--ref-sample-cells", type=int, default=512)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's outputs for a fixed, seeded sample of cells to DIR/*.npy "
                         "(GPU arm only)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs; --impl reference has none to write")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    cfg0 = CONFIGS[args.config]
    args.scaling_label = "weak" if (args.scaling == "weak" or (cfg0.get("shards", 1) > max(world_env, args.gpus) and not args.cells)) else "strong"
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist

    from infercnv_b200 import api, dist as shard
    from infercnv_b200.device import Engine

    world = world_env
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU path); use --impl reference for the CPU arm")
    eng = Engine(local_rank)
    sampler = ClockSampler(local_rank)   # started now: nvidia-smi takes longer to come up than a short timed region lasts
    if rank == 0:
        sampler.start()
    cfg, G, C_total, seed, note = resolve_config(args, world)
    steps = args.steps or max(3, cfg["steps"] * world * (cfg["cells"] // cfg.get("shards", 1)) // max(1, C_total))
    cs, cl = chr_layout(G)
    refs_g = ref_groups_global(C_total)
    atoms = subclusters_global(C_total, seed) if cfg["median_filter"] else None
    plan = shard.plan_shards(C_total, refs_g, world, other_atoms=atoms)[rank]
    cells = plan.local_cells
    C_local = len(cells)
    X = eng.synth(G, cs, cl, cells, C_total, seed)
    ref_local = plan.local_ref_groups()
    n_ref_local = int(sum(len(g) for g in ref_local))
    MF_R = 4                                                     # window 7 -> radius (7 + 1) / 2
    n_scratch = 2 * MF_R * len(ref_local) if cfg["median_filter"] else 0
    Yext = torch.empty((C_local + n_scratch, G), dtype=torch.float64, device=X.device)
    Y = Yext[:C_local]
    states = torch.empty((C_local, G), dtype=torch.uint8, device=X.device)
    Fext = torch.empty_like(Yext) if cfg["median_filter"] else None
    sub_local = []
    if cfg["median_filter"]:
        oc = plan.other_cells
        for a in atoms:
            if len(oc) and oc[0] <= a[0] <= oc[-1]:
                p0 = n_ref_local + int(np.searchsorted(oc, a[0]))
                sub_local.append(np.arange(p0, p0 + len(a), dtype=np.int32))
    model6 = i6_model()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    flags = []

    def step(record=None):
        marks = [ev() for _ in range(4)] if record is not None else None
        if marks:
            marks[0].record()
        _, f1 = eng.smooth_block(X, cs, cl, ref_local, plan.ref_sizes, plan.max_chunks, apply_log=True, threshold=3.0,
                                 window=101, use_bounds=True, out=Y)
        if marks:
            marks[1].record()
        if cfg["hmm"] == "i6":
            Pi, delta, mean, sd = model6
        else:      # i3: mu / sigma over the reference cells' smoothed values, all ranks (R/inferCNV_i3HMM.R:17-30)
            mu, sg = eng.mean_sd(Y, ref_local)
            Pi, delta, mean, sd = i3_model(mu, sg)
        _, f2 = eng.viterbi(Y, cs, cl, Pi, delta, mean, sd, out=states)
        if marks:
            marks[2].record()
        if cfg["median_filter"]:
            eng.median_filter_sharded(Yext, C_local, sub_local, ref_local, cs, cl, 7, out=Fext)
        if marks:
            marks[3].record()
            record.append(marks)
        flags.append((f1, f2))

    for _ in range(args.warmup):
        step()
    barrier()
    launches0 = eng.launch_count()
    rec = []
    eng.timing = []
    barrier()
    wall0 = time.time()
    t_start, t_end = ev(), ev()
    t_start.record()
    for _ in range(steps):
        step(rec)
    t_end.record()
    barrier()
    wall1 = time.time()
    launches = eng.launch_count() - launches0
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    ms_step = t_start.elapsed_time(t_end) / steps
    ms_smooth = float(np.mean([m[0].elapsed_time(m[1]) for m in rec]))
    ms_hmm = float(np.mean([m[1].elapsed_time(m[2]) for m in rec]))
    ms_mf = float(np.mean([m[2].elapsed_time(m[3]) for m in rec]))
    ms_pass2 = float(np.mean([a.elapsed_time(b) for _, a, b in eng.timing]))
    eng.timing = None
    for f1, f2 in flags:
        if int(f1.item()) or int(f2.item()):
            raise SystemExit("non-finite / underflow flag raised during the benchmark")
    smin, smax = int(states.min().item()), int(states.max().item())
    assert 1 <= smin and smax <= (6 if cfg["hmm"] == "i6" else 3), (smin, smax)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, cells, C_total, G, Y, states, Fext[:C_local] if cfg["median_filter"] else None, world, rank)

    # ---- end to end through the host-facing API from PAGEABLE host memory, copies inside the timed region ----
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, cfg, eng, api, X, Yext, Fext, states, cs, cl, ref_local, sub_local, plan, model6, G, C_total, C_local, world,
                      barrier)

    # ---- max over ranks ----------------------------------------------------------------------------------------
    t = torch.tensor([ms_step, ms_smooth, ms_hmm, ms_pass2, ms_mf], dtype=torch.float64, device=X.device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step, ms_smooth, ms_hmm, ms_pass2, ms_mf = (float(v) for v in t.tolist())

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        n_listed = C_local
        hmm_bytes = BYTES_HMM * C_local * G
        smooth_bytes = BYTES_SMOOTH * C_local * G + 16.0 * n_ref_local * G
        pass2_bytes = BYTES_SMOOTH * C_local * G
        mf_bytes = BYTES_MF * n_listed * G
        parts = {"cell_pipeline pass 2": ms_pass2, "viterbi": ms_hmm, "median_filter": ms_mf}
        reruns = int(api.hmm_rerun_count())
        second_pass = int(api.hmm_second_pass_count())

        def roof(name, kernel, nbytes, ms, note, **extra):
            ach = nbytes / (ms * 1e-3) / 1e9
            d = {"kernel": f"{kernel} ({100 * ms / ms_step:.0f} % of the step)", "bound": "hbm", "achieved": ach, "peak": peak,
                 "unit": "GB/s", "frac": ach / peak, "traffic": ncu_traffic(name, args.config, world), "peak_source": peak_src,
                 "algorithmic_bytes_per_launch": nbytes, "ms_per_launch": ms, "note": note}
            d.update(extra)
            return d
        r_p2 = roof("cell_pipeline_pass2", "cell_pipeline kernel, pass 2 over all local cells", pass2_bytes, ms_pass2,
                    "16 B per cell-gene (one FP64 read, one FP64 write); see DESIGN.md section 3 K2")
        r_hmm = roof("viterbi_fast", (f"viterbi_fast32_kernel<{6 if cfg['hmm'] == 'i6' else 3}> + FP64 second pass + exact re-run list" if os.environ.get("ICNV_HMM_MODE", "1")[:1] == "2"
                      else f"viterbi_fast_kernel<{6 if cfg['hmm'] == 'i6' else 3}> + exact re-run list"), hmm_bytes, ms_hmm,
                     "9 B per cell-gene (8 read + 1 state byte); see DESIGN.md section 3 K3",
                     sequences_rerun_in_reference_order_arithmetic=reruns, sequences_second_pass_fp64=second_pass, sequences=int(C_local * len(cs)))
        r_mf = roof("median_filter", "median filter kernel (window 7: 9 x 9 taps)", mf_bytes, ms_mf,
                    "16 B per listed cell-gene; see DESIGN.md section 3 K4") if cfg["median_filter"] else None
        dominant = max(parts, key=parts.get)
        out = {
            "metric": METRIC, "value": G * C_total / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": args.scaling_label, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, cfg, G, C_total, world, note),
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": {"cell_pipeline pass 2": r_p2, "viterbi": r_hmm, "median_filter": r_mf}[dominant],
            "roofline_cell_pipeline": r_p2, "roofline_hmm": r_hmm,
            "roofline_smooth_block": {"kernels": "group partial sums + bounds + cell_pipeline pass 1 (reference cells) + pass 2",
                                      "bound": "hbm", "achieved": smooth_bytes / (ms_smooth * 1e-3) / 1e9, "peak": peak,
                                      "unit": "GB/s", "frac": smooth_bytes / (ms_smooth * 1e-3) / 1e9 / peak,
                                      "algorithmic_bytes_per_step": smooth_bytes, "ms_per_step": ms_smooth},
            "stage_ms": {"smooth_block": ms_smooth, "hmm": ms_hmm, "median_filter": ms_mf if cfg["median_filter"] else None},
        }
        if r_mf:
            out["roofline_median_filter"] = r_mf
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(args, cfg, G, C_total, seed)
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_e2e(args, cfg, eng, api, X, Yext, Fext, states, cs, cl, ref_local, sub_local, plan, model6, G, C_total, C_local, world, barrier):
    """The same step through the host-facing API with HOST buffers.  N = 1: the C ABI's host-pointer entry points on
    pageable NumPy arrays - exactly what an R matrix is - so the library's pinned staging ring and copy threads are inside
    the timed region.  N > 1: every rank moves its shard between pinned host tensors and its GPU around the device step."""
    import torch
    import torch.distributed as dist
    Y = Yext[:C_local]
    n_e2e = 2 if C_local * G > 4e8 else 5
    if world == 1:
        xn = np.empty((G, C_local), dtype=np.float64, order="F")      # pageable
        xn.T[...] = X.cpu().numpy()
        yn = np.empty((G, C_local), dtype=np.float64, order="F")
        sn = np.empty((G, C_local), dtype=np.uint8, order="F")
        fn = np.empty((G, C_local), dtype=np.float64, order="F") if cfg["median_filter"] else None
        Pi, delta, mean, sd = model6
        if cfg["hmm"] == "i6":
            def e2e_step():
                api.smooth_hmm(xn, cs, cl, ref_local, Pi, delta, mean, sd, out=yn, out_states=sn)
            label = "icnv_smooth_hmm_u8_f64: ONE fused call on pageable host memory (the call infercnvb200's fused R closure makes)"
            h2d = int(C_local * G * 8 * 1.1)
            d2h = C_local * G * 9
        else:
            ref_all = np.concatenate(ref_local)

            def e2e_step():
                api.smooth_block(xn, cs, cl, ref_local, apply_log=True, threshold=3.0, window_length=101, out=yn)
                mu, sg = api.mean_sd(yn, ref_all)
                P3, d3, m3, s3 = i3_model(mu, sg)
                api.viterbi(yn, cs, cl, P3, d3, m3, s3, out=sn)
                api.median_filter(yn, cs, cl, list(sub_local) + list(ref_local), 7, out=fn)
            label = ("icnv_smooth_block_f64 + icnv_mean_sd_f64 + icnv_viterbi_u8_f64 + icnv_median_filter_f64 on pageable host memory "
                     "(four calls, as the R wrappers make them)")
            h2d = int(C_local * G * 8 * (1.1 + 0.1 + 1 + 1))
            d2h = C_local * G * (8 + 1 + 8)
        e2e_step()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            e2e_step()
        dt = (time.perf_counter() - t0) / n_e2e
    else:
        hX = torch.empty((C_local, G), dtype=torch.float64, pin_memory=True)
        hX.copy_(X)
        hY = torch.empty((C_local, G), dtype=torch.float64, pin_memory=True)
        hS = torch.empty((C_local, G), dtype=torch.uint8, pin_memory=True)
        hF = torch.empty((C_local, G), dtype=torch.float64, pin_memory=True) if cfg["median_filter"] else None
        dX = torch.empty_like(X)
        torch.cuda.synchronize()
        Pi, delta, mean, sd = model6
        if cfg["hmm"] == "i6":
            def e2e_step():
                eng.smooth_hmm_host(hX, hY, hS, dX, Y, states, cs, cl, ref_local, plan.ref_sizes, plan.max_chunks, Pi, delta, mean, sd)
            label = "Engine.smooth_hmm_host: per-rank slab pipeline between pinned host tensors and the GPU (one rank per GPU)"
        else:
            def e2e_step():
                dX.copy_(hX, non_blocking=True)
                eng.smooth_block(dX, cs, cl, ref_local, plan.ref_sizes, plan.max_chunks, out=Y)
                mu, sg = eng.mean_sd(Y, ref_local)
                P3, d3, m3, s3 = i3_model(mu, sg)
                eng.viterbi(Y, cs, cl, P3, d3, m3, s3, out=states)
                eng.median_filter_sharded(Yext, C_local, sub_local, ref_local, cs, cl, 7, out=Fext)
                hY.copy_(Y, non_blocking=True)
                hS.copy_(states, non_blocking=True)
                hF.copy_(Fext[:C_local], non_blocking=True)
                torch.cuda.synchronize()
            label = "per rank: upload, Engine.smooth_block / mean_sd / viterbi / median_filter_sharded, download (pinned host tensors)"
        h2d = C_local * G * 8
        d2h = C_local * G * (9 + (8 if cfg["median_filter"] else 0))
        e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            e2e_step()
        torch.cuda.synchronize()
        dtt = torch.tensor([(time.perf_counter() - t0) / n_e2e], dtype=torch.float64, device=X.device)
        dist.all_reduce(dtt, op=dist.ReduceOp.MAX)
        dt = float(dtt.item())
    return {"value": G * C_total / dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "ms_per_step": dt * 1e3, "steps": n_e2e, "host_memory": "pageable (NumPy)" if world == 1 else "pinned (torch)", "api": label}


if __name__ == "__main__":
    main()
