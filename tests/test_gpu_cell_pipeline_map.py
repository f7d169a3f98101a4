"""Every compiled instantiation of the fused cell pipeline (icnv_dev_cell_pipeline_f64: cell_pipeline3_kernel and
cell_pipeline4_kernel) against the CPU oracle, each reached through the launcher's own selection and identified by the
test hook icnv_debug_cell_launch.  Needs a B200: run with `pytest -m gpu`.

The launch map (LAUNCH_MAP) follows the launcher's shared-memory arithmetic (smem_for / smem4) and build_segments:
gene count, chromosome layout and window select the thread count, the padded-Q or ping-pong layout of v3, v4 when v3's
two buffers do not fit, and the fully unrolled slice loops.  The tuning switches (ICNV_CELL_KERNEL / _NT / _PADQ / _LFIX)
are only used for what the default selection never picks.  Each case runs at least three cells per resident CTA, with
cell kinds mixed so that consecutive cells of one CTA take different median paths.
"""
import ctypes as ct
import re

import numpy as np
import pytest

import bench
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

# (version, threads, padded Q, fixed slice length, min CTAs per SM) of every kernel the launcher can launch
INSTANTIATIONS = {
    (3, 256, 1, 0, 1), (3, 512, 1, 0, 1), (3, 1024, 1, 0, 1), (3, 1024, 1, 11, 1),
    (3, 256, 0, 0, 1), (3, 512, 0, 0, 1), (3, 1024, 0, 0, 1),
    (4, 256, 0, 0, 4), (4, 256, 0, 0, 1), (4, 512, 0, 0, 2), (4, 512, 0, 21, 2), (4, 512, 0, 0, 1),
    (4, 1024, 0, 0, 1), (4, 1024, 0, 21, 1),
}

SWITCHES = ("ICNV_CELL_KERNEL", "ICNV_CELL_NT", "ICNV_CELL_PADQ", "ICNV_CELL_LFIX", "ICNV_SLAB_CELLS")

# name: (G, chromosomes (22 = the benchmark's layout, else a mixed layout with one-gene chromosomes and chromosomes shorter
# than the window), layout seed, window, switches, expected instantiation)
LAUNCH_MAP = {
    "v3_256_padq_oddG": (1501, 24, 1, 101, {}, (3, 256, 1, 0, 1)),
    "v3_512_padq_oddG": (4001, 30, 2, 3, {}, (3, 512, 1, 0, 1)),
    "v3_1024_padq": (8000, 22, 0, 201, {}, (3, 1024, 1, 0, 1)),
    "v3_1024_padq_lfix11_c2_c3": (10000, 22, 0, 101, {}, (3, 1024, 1, 11, 1)),
    "v3_256_pingpong": (2000, 150, 3, 201, {}, (3, 256, 0, 0, 1)),        # the padded Q does not fit: ping-pong on its own
    "v3_512_pingpong": (5000, 150, 4, 201, {}, (3, 512, 0, 0, 1)),
    "v3_1024_pingpong": (12600, 22, 0, 101, {}, (3, 1024, 0, 0, 1)),
    "v4_1024_lfix21_c5": (20000, 22, 0, 101, {}, (4, 1024, 0, 21, 1)),
    "v4_1024_largest_w101": (23861, 22, 0, 101, {}, (4, 1024, 0, 0, 1)),  # shared memory used to the last byte
    "v4_1024_lfix21_w51": (20000, 22, 0, 51, {}, (4, 1024, 0, 21, 1)),    # odd h: the chunk table needs 8 bytes of padding
    "v4_256x4_oddG": (3001, 24, 5, 101, {"ICNV_CELL_KERNEL": "4"}, (4, 256, 0, 0, 4)),
    "v4_256x1": (16000, 22, 0, 3, {"ICNV_CELL_KERNEL": "4", "ICNV_CELL_NT": "256"}, (4, 256, 0, 0, 1)),
    "v4_512x2_lfix21": (10000, 22, 0, 101, {"ICNV_CELL_KERNEL": "4"}, (4, 512, 0, 21, 2)),
    "v4_512x2": (8000, 22, 0, 101, {"ICNV_CELL_KERNEL": "4"}, (4, 512, 0, 0, 2)),
    "v4_512x1": (16000, 22, 0, 101, {"ICNV_CELL_KERNEL": "4", "ICNV_CELL_NT": "512"}, (4, 512, 0, 0, 1)),
    # more chromosomes than the gene count's thread count: the next larger CTA
    "k300_w3": (1500, 300, 6, 3, {}, (3, 512, 1, 0, 1)),
    "k300_w0": (1500, 300, 6, 0, {}, (3, 512, 1, 0, 1)),
    "k600_w3": (4000, 600, 7, 3, {}, (3, 1024, 1, 0, 1)),
    "k600_w0": (4000, 600, 7, 0, {}, (3, 1024, 1, 0, 1)),
}


@pytest.fixture(scope="module")
def api():
    from infercnv_b200 import api as a
    a.init(0)
    return a


def _hook():
    from infercnv_b200 import _lib
    lib = _lib.load()
    lib.icnv_debug_cell_launch.restype = ct.c_int
    lib.icnv_debug_cell_launch.argtypes = [ct.c_void_p]
    lib.icnv_debug_stats.restype = ct.c_int
    lib.icnv_debug_stats.argtypes = [ct.c_void_p, ct.c_int]
    return lib


def last_launch():
    """(version, threads, padded Q, fixed slice length, min CTAs per SM, segment length, grid, resident CTAs)"""
    from infercnv_b200 import _lib
    out = (ct.c_int * 8)()
    _lib.check(_hook().icnv_debug_cell_launch(ct.addressof(out)))
    return tuple(out)


def median_stats(reset=True):
    """{medians, histogram hits, bracketing exits (split / all equal / key space), gather exits} since the last reset"""
    from infercnv_b200 import _lib
    out = (ct.c_ulonglong * 16)()
    _lib.check(_hook().icnv_debug_stats(ct.addressof(out), int(reset)))
    return {"medians": out[1], "hist": out[10], "bracket": out[2], "gather": out[3]}


def switch(api, monkeypatch, env):
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    api.reinit()   # tuning switches are read once, at icnv_init


def layout(G, K, seed):
    if K == 22:
        return bench.chr_layout(G)
    rng = np.random.default_rng(seed)
    fixed = [1, 2, 40, 1, 150, 3]   # single-gene, two-gene and shorter-than-the-window chromosomes
    rest = G - sum(fixed)
    w = rng.random(K - len(fixed)) + 0.2
    lens = np.floor(w / w.sum() * rest).astype(np.int64)
    lens[0] += rest - lens.sum()
    lens = np.concatenate([lens[:len(lens) // 2], fixed, lens[len(lens) // 2:]]).astype(np.int32)
    assert lens.min() >= 1 and lens.sum() == G
    return np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int32), lens


N_REF = 5   # columns 0..2 and 3..4: two reference groups of identical cells, so the dead-band bounds are known values
KINDS = ("poisson", "lognormal", "zero", "constant", "two_valued", "three_valued", "bimodal", "heavy", "on_bounds", "minus_one")


def cells(G, C, grid, seed, minus_one=True):
    """Raw counts, G x C.  Cell j has kind KINDS[(j // grid + j) % n]: the cells one CTA processes back to back (j, j + grid,
    ...) differ in kind, and so in the path their median takes.  After log2(x + 1), the dead band and the clamp at 3:
    -1 -> -3 and 1e12 -> +3 exactly (constant, two- and three-valued cells: ties far beyond 64 in the middle bin), a
    reference group's own value -> exactly on a dead-band bound."""
    rng = np.random.default_rng(seed)
    lam = rng.lognormal(0.5, 1.0, size=G)
    a = rng.poisson(lam).astype(np.float64)
    b = rng.poisson(1.3 * lam).astype(np.float64)
    X = np.empty((G, C), dtype=np.float64, order="F")
    X[:, :3] = a[:, None]
    X[:, 3:N_REF] = b[:, None]
    kinds = [k for k in KINDS if minus_one or k not in ("constant", "two_valued", "three_valued", "minus_one")]
    for j in range(N_REF, C):
        kind = kinds[(j // grid + j) % len(kinds)]
        if kind == "poisson":
            x = rng.poisson(lam * rng.lognormal(0, 0.3)).astype(np.float64)
        elif kind == "lognormal":   # log2(x + 1) continuous and mostly above the dead band: no ties even unsmoothed
            x = np.exp2(3.0 + 0.7 * rng.standard_normal(G)) - 1.0
        elif kind == "zero":
            x = np.zeros(G)
        elif kind == "constant":
            x = np.full(G, -1.0 if j % 2 else 1e12)
        elif kind == "two_valued":
            x = np.where(rng.random(G) < 0.55, -1.0, 1e12)
        elif kind == "three_valued":
            x = rng.choice(np.array([-1.0, 1e12, 0.0]), size=G, p=[0.3, 0.3, 0.4])
            x[x == 0.0] = a[x == 0.0]
        elif kind == "bimodal":   # 70 % low, 30 % high: the median lies outside mean +- 0.35 sd
            x = np.where(rng.random(G) < 0.7, rng.poisson(0.3, size=G), rng.poisson(80.0, size=G)).astype(np.float64)
        elif kind == "heavy":
            x = np.exp(3.0 * rng.standard_normal(G))
        elif kind == "on_bounds":
            x = np.where(rng.random(G) < 0.5, a, b)
        else:   # minus_one: x + 1 == 0 at a tenth of the genes
            x = rng.poisson(lam).astype(np.float64)
            x[rng.random(G) < 0.1] = -1.0
        X[:, j] = x
    return X


def resident_ctas(api, X, cs, lens, window):
    """CTAs the launcher runs at once for this shape (a one-cell launch through the same selection)"""
    api.smooth(X[:, :1], cs, lens, window)
    return last_launch()[7]


def tolerance(lens, window, threshold=3.0):
    """1e-10 relative, or the rounding bound of the kernels' second-order prefix sums where that is larger: over a
    chromosome of n genes they reach ~ threshold * n^2 / 2, and a smoothed value is a difference of three of them divided
    by (h + 1)^2: with window 3 and 1 600-gene chromosomes up to ~1e-9, four orders of magnitude inside the 1e-5 of the
    north star."""
    if window < 2:
        return 1e-10
    h = (window - 1) // 2
    n = float(np.max(lens))
    return max(1e-10, 16 * np.finfo(np.float64).eps * threshold * n * n / 2 / (h + 1) ** 2)


def _rel(got, want):
    return float(np.max(np.abs(got - want) / np.abs(want)))


# ---- the launch map ---------------------------------------------------------------------------------------------------
def test_launch_map_covers_every_instantiation(api, monkeypatch):
    """Each LAUNCH_MAP row reaches the kernel it names; together they reach all 14.  A kernel added to the launcher and
    missing here fails this test."""
    seen = {}
    for name, (G, K, seed, w, env, want) in LAUNCH_MAP.items():
        switch(api, monkeypatch, env)
        cs, lens = layout(G, K, seed)
        api.smooth(np.ones((G, 1)), cs, lens, w)
        got = last_launch()
        assert got[:5] == want, (name, got)
        assert got[5] > 0 and got[6] == 1, (name, got)
        seen.setdefault(got[:5], name)
    switch(api, monkeypatch, {})
    print("\n" + "\n".join(f"  {k}: {v}" for k, v in sorted(seen.items())))
    assert set(seen) == INSTANTIATIONS


@pytest.mark.parametrize("name", list(LAUNCH_MAP))
def test_launch_map_case_against_the_oracle(api, monkeypatch, name):
    """The smooth block (steps 4, 8-12, 14) of the case's kernel: every value within 1e-10 relative of the oracle; the
    histogram median and at least one bracketing exit taken; the padded-Q and ping-pong layouts, and the unrolled and
    generic slice loops, bit for bit the same; v3 against v4 where both can run."""
    from infercnv_b200._lib import InfercnvB200Error
    G, K, seed, w, env, want = LAUNCH_MAP[name]
    cs, lens = layout(G, K, seed)
    one_slab = {"ICNV_SLAB_CELLS": "65536"}   # the whole matrix in one launch
    switch(api, monkeypatch, dict(env, **one_slab))
    resident = resident_ctas(api, np.ones((G, 1)), cs, lens, w)
    C = max(3 * resident, 3 * len(KINDS) + N_REF)
    X = cells(G, C, resident, seed=1000 + G)
    refs = [np.arange(0, 3), np.arange(3, N_REF)]

    median_stats(reset=True)
    got = api.smooth_block(X, cs, lens, refs, apply_log=True, threshold=3.0, window_length=w)
    launch = last_launch()
    st = median_stats(reset=True)
    assert launch[:5] == want and launch[6] == resident and C >= 3 * launch[6], launch
    assert st["medians"] == C + N_REF, st
    assert st["hist"] > 0 and st["bracket"] > 0, st
    want_y = orc.smooth_block(X, cs, lens, refs, window=w, nthreads=orc.max_threads())
    rel, tol = _rel(got, want_y), tolerance(lens, w)
    print(f"\n[{name}] {launch[:6]} C={C}: max rel err vs oracle {rel:.2e} (bound {tol:.1e}); medians {st}")
    assert np.all(np.isfinite(got)) and rel < tol

    def rerun(extra):
        switch(api, monkeypatch, dict(env, **one_slab, **extra))
        y = api.smooth_block(X, cs, lens, refs, apply_log=True, threshold=3.0, window_length=w)
        return y, last_launch()

    if want[0] == 3 and want[2] == 1:
        y, l = rerun({"ICNV_CELL_PADQ": "0"})
        assert l[:3] == (3, want[1], 0) and np.array_equal(y, got), l
    if want[3]:
        y, l = rerun({"ICNV_CELL_LFIX": "0"})
        assert l[:4] == want[:3] + (0,) and np.array_equal(y, got), l
    # v3 against v4 on the same shape, where the default selection and the switch give one of each
    other = None
    if want[0] == 3:
        try:
            other, l = rerun({"ICNV_CELL_KERNEL": "4"})
            assert l[0] == 4
        except InfercnvB200Error as e:   # v4's padded column holds 2h + 3 pads per chromosome: too long for some layouts
            assert e.code == -4 and "shared memory" in str(e)
    elif "ICNV_CELL_KERNEL" in env:
        y, l = rerun({k: v for k, v in env.items() if k not in ("ICNV_CELL_KERNEL", "ICNV_CELL_NT")})
        other = y if l[0] == 3 else None
    if other is not None:
        d = _rel(other, got)
        print(f"[{name}] v3 against v4: max rel difference {d:.2e}, {int(np.sum(other != got))} of {got.size} values differ")
        assert d < tol
    switch(api, monkeypatch, {})


def test_column_too_long_for_shared_memory_is_refused(api):
    """One gene more than v4_1024_largest_w101: error -4, and the message names the bytes the column needs and the limit."""
    from infercnv_b200._lib import InfercnvB200Error
    G = LAUNCH_MAP["v4_1024_largest_w101"][0] + 1
    cs, lens = bench.chr_layout(G)
    with pytest.raises(InfercnvB200Error) as e:
        api.smooth(np.ones((G, 2)), cs, lens, 101)
    assert e.value.code == -4
    m = re.search(r"needs (\d+) B of shared memory, more than the (\d+) B", str(e.value))
    assert m and int(m.group(1)) > int(m.group(2)), str(e.value)


def test_more_chromosomes_than_a_cta_has_threads_is_refused(api):
    """1025 one-gene chromosomes cannot be given a thread each: -4 with that reason."""
    from infercnv_b200._lib import InfercnvB200Error
    lens = np.ones(1025, dtype=np.int32)
    cs = np.arange(1025, dtype=np.int32)
    with pytest.raises(InfercnvB200Error) as e:
        api.smooth(np.ones((1025, 2)), cs, lens, 3)
    assert e.value.code == -4 and "1025 non-empty chromosomes need a thread each" in str(e.value), str(e.value)


def test_bench_configs_keep_their_kernels(api, monkeypatch):
    """bench.py's gene counts (c2 / c3: 10 000, c5: 20 000) in its chromosome layout, window 101, default switches."""
    switch(api, monkeypatch, {})
    for G, want in ((10000, (3, 1024, 1, 11, 1, 11)), (20000, (4, 1024, 0, 21, 1, 21))):
        cs, lens = bench.chr_layout(G)
        api.smooth(np.ones((G, 1)), cs, lens, 101)
        assert last_launch()[:6] == want, (G, last_launch())


# ---- the device ABI through Engine: stage flags, strided and misaligned inputs -------------------------------------------
ENGINE_SHAPES = {"v3_256": (2000, 24, 11, {}, (3, 256, 1, 0, 1)),
                 "v4_256x4": (2000, 24, 11, {"ICNV_CELL_KERNEL": "4"}, (4, 256, 0, 0, 4)),
                 "v3_1024_lfix11": (10000, 22, 0, {}, (3, 1024, 1, 11, 1))}


@pytest.fixture(scope="module")
def engine():
    import torch

    from infercnv_b200.device import Engine
    return Engine(0), torch


def _engine_case(api, monkeypatch, engine, shape, window=101, minus_one=True):
    eng, torch = engine
    G, K, seed, env, want = ENGINE_SHAPES[shape]
    switch(api, monkeypatch, env)
    cs, lens = layout(G, K, seed)
    resident = resident_ctas(api, np.ones((G, 1)), cs, lens, window)
    C = max(3 * resident, 3 * len(KINDS) + N_REF)
    X = cells(G, C, resident, seed=2000 + G, minus_one=minus_one)
    return eng, torch, G, C, cs, lens, X, want


def _reference(X, cs, lens, log, mode, b1, thr, window, center, b2, exp2):
    """The pipeline's stages composed from the oracle's step functions (dead band and mid subtraction written out)."""
    def subtract(x, b):
        lo, hi, mid = (v[:, None] for v in b)
        if mode == "bounds":
            return np.where(x > hi, x - hi, np.where(x < lo, x - lo, 0.0))
        return x - mid if mode == "mid" else x
    x = orc.log2xplus1(X) if log else X.copy(order="F")
    x = subtract(x, b1)
    if thr > 0:
        x = orc.apply_max_threshold_bounds(x, thr)
    x = orc.smooth_by_chromosome(x, cs, lens, window, nthreads=orc.max_threads())
    if center:
        x = orc.center_columns(x, "median" if center == 1 else "mean", nthreads=orc.max_threads())
    x = subtract(x, b2)
    return orc.invert_log2(x) if exp2 else x


@pytest.mark.parametrize("shape", ["v3_256", "v4_256x4"])
def test_engine_stage_flag_combinations(api, monkeypatch, engine, shape):
    """log on / off x bounds / mid / none x threshold 0 / 3 x centre none / median / mean x 2^x on / off through
    Engine.cell_pipeline: the fast grouped stage A / D loops (log + bounds + threshold, bounds + 2^x) and the generic ones,
    every column within 1e-10 of the oracle's column's largest magnitude (at least 1)."""
    eng, torch, G, C, cs, lens, X, want = _engine_case(api, monkeypatch, engine, shape, minus_one=False)
    rng = np.random.default_rng(3)
    m1 = 1.0 + 0.4 * rng.standard_normal((G, 2))
    m2 = 0.2 * rng.standard_normal((G, 2))
    b1 = (m1.min(1), m1.max(1), m1.mean(1))
    b2 = (m2.min(1), m2.max(1), m2.mean(1))
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(eng.tdev)   # noqa: E731
    dX, dXl = dev(X.T), dev(orc.log2xplus1(X).T)   # without the log step the input is already on the log scale
    db1, db2 = tuple(dev(v) for v in b1), tuple(dev(v) for v in b2)
    Y = torch.empty_like(dX)
    flag = torch.zeros(1, dtype=torch.int32, device=eng.tdev)
    worst = 0.0
    for log in (True, False):
        for mode in ("bounds", "mid", "none"):
            for thr in (0.0, 3.0):
                for center in (0, 1, 2):
                    for exp2 in (True, False):
                        eng.cell_pipeline(dX if log else dXl, None, Y, cs, lens, log, None if mode == "none" else db1, thr, 101, center,
                                          None if mode == "none" else db2, exp2, use_bounds=mode == "bounds", err_flag=flag)
                        got = Y.cpu().numpy().T
                        assert last_launch()[:5] == want
                        ref = _reference(X if log else orc.log2xplus1(X), cs, lens, log, mode, b1, thr, 101, center, b2, exp2)
                        # log-scale values: a unit floor under each column's scale, so that a column that is exactly
                        # zero in the oracle (an all-zero cell: the kernels' table-driven log2(1 + 0) is ~3e-18, not 0)
                        # is held to 1e-10 absolute
                        scale = np.maximum(np.max(np.abs(ref), axis=0), 1.0)
                        err = float(np.max(np.max(np.abs(got - ref), axis=0) / scale))
                        worst = max(worst, err)
                        assert err < 1e-10, (log, mode, thr, center, exp2, err)
    assert int(flag.item()) == 0
    print(f"\n[{shape}] 72 stage combinations, C={C}: worst column-relative error {worst:.2e}")
    switch(api, monkeypatch, {})


@pytest.mark.parametrize("shape", list(ENGINE_SHAPES))
def test_engine_strided_misaligned_and_indexed_inputs_are_bitwise(api, monkeypatch, engine, shape):
    """The same cells read through an odd ldx (the bulk copy and the element-wise fallback load alternate from cell to
    cell within a CTA), from an address one double off (every column misaligned), through a permuted index list with
    repeats, and written with ldy > G (the pad rows keep their sentinel): bit for bit the contiguous run.  And
    api.smooth_block (host pointers) equals Engine.smooth_block (device tensors) bit for bit."""
    eng, torch, G, C, cs, lens, X, want = _engine_case(api, monkeypatch, engine, shape)
    refs = [np.arange(0, 3), np.arange(3, N_REF)]
    dX = torch.from_numpy(np.ascontiguousarray(X.T)).to(eng.tdev)
    Y0, flag = eng.smooth_block(dX, cs, lens, refs)
    torch.cuda.synchronize()
    assert int(flag.item()) == 0 and last_launch()[:5] == want
    host = api.smooth_block(X, cs, lens, refs)
    assert np.array_equal(host, Y0.cpu().numpy().T)
    # the same pass-2 arguments as Engine.smooth_block's last launch, on differently laid out inputs
    b1, b2, _, _, _ = eng._reference_bounds(dX, cs, lens, refs, None, None, True, 3.0, 101, True, flag)

    def run(Xv, cols=None, out=None):
        n = Xv.shape[0] if cols is None else cols.numel()
        Y = torch.empty((n, G), dtype=torch.float64, device=eng.tdev) if out is None else out
        eng.cell_pipeline(Xv, cols, Y, cs, lens, True, b1, 3.0, 101, 1, b2, True, True, flag)
        return Y

    base = run(dX)
    torch.cuda.synchronize()
    ldx = G + 3   # G even, ldx odd: consecutive columns alternate between 16-byte aligned and not
    big = torch.full((C, ldx), np.nan, dtype=torch.float64, device=eng.tdev)
    big[:, :G] = dX
    assert torch.equal(run(big[:, :G]), base)
    flat = torch.empty(C * G + 1, dtype=torch.float64, device=eng.tdev)
    off = flat[1:].view(C, G)
    off.copy_(dX)
    assert off.data_ptr() % 16 == 8
    assert torch.equal(run(off), base)
    rng = np.random.default_rng(4)
    idx = np.concatenate([rng.permutation(C), rng.integers(0, C, size=C // 3)]).astype(np.int32)
    cols = torch.from_numpy(idx).to(eng.tdev)
    assert torch.equal(run(dX, cols), base[torch.from_numpy(idx.astype(np.int64)).to(eng.tdev)])
    sentinel = -12345.678
    ybig = torch.full((C, G + 5), sentinel, dtype=torch.float64, device=eng.tdev)
    run(big[:, :G], out=ybig[:, :G])
    torch.cuda.synchronize()
    assert torch.equal(ybig[:, :G], base)
    assert bool((ybig[:, G:] == sentinel).all())
    assert int(flag.item()) == 0
    switch(api, monkeypatch, {})
