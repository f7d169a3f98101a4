"""CNV region calling (SURVEY section 8(f) rank 1; R/inferCNV_HMM.R:706-1087) through the C ABI against the
oracle, the reference's bundled known answer, and size-independent properties at full size."""
import os

import numpy as np
import pytest

from oracle import regions as orr

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden", "cnv_regions_fixture.npz")


def _layout(lens):
    lens = np.asarray(lens, dtype=np.int32)
    return np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int32), lens


def _states(rng, G, C, p_noise=0.2, unassigned=0.0):
    """few distinct values in long runs (real HMM output) + salt noise -> ties and many boundaries"""
    base = np.repeat(rng.integers(1, 7, size=(G // 37 + 1, C)), 37, axis=0)[:G]
    S = np.where(rng.random((G, C)) < p_noise, rng.integers(0, 7, size=(G, C)), base).astype(np.uint8)
    if unassigned:
        S[:, rng.random(C) < unassigned] = 255
    return np.asfortranarray(S)


def _same_regions(got, want):
    for k in ("seq", "chr", "first_gene", "last_gene", "state", "start", "end"):
        assert got[k].shape == want[k].shape, (k, got[k].shape, want[k].shape)
        assert np.array_equal(got[k], want[k]), k


@pytest.mark.parametrize("G", [4613, 4612, 1027, 97])     # 4612: 32-bit load path; the others: byte path
def test_state_consensus_matches_the_oracle(G):
    from infercnv_b200 import api
    rng = np.random.default_rng(G)
    C = 700
    S = _states(rng, G, C, p_noise=0.5, unassigned=0.05)
    perm = rng.permutation(C)
    groups = [perm[:1], perm[1:3], perm[3:260], perm[260:520], np.sort(perm[100:700]), perm[::-1][:256], perm[:255]]
    got = api.state_consensus(S, groups)
    assert got.dtype == np.uint8 and got.shape == (G, len(groups))
    for k, g in enumerate(groups):
        assert np.array_equal(got[:, k], orr.state_consensus(S, g)), k
    # literal transcription of .get_state_consensus on a slice (table / order(decreasing=TRUE)[1])
    lit = orr.literal_state_consensus(S[:200][:, groups[3]])
    assert np.array_equal(np.where(lit < 0, 255, lit), got[:200, 3])


def test_consensus_ties_and_unassigned_order():
    from infercnv_b200 import api
    m = np.array([[2, 4, 4, 2], [6, 5, 6, 5], [3, 3, 3, 1], [255, 255, 1, 1], [0, 0, 6, 6]], dtype=np.uint8)
    assert api.state_consensus(m, [np.arange(4)])[:, 0].tolist() == [2, 5, 3, 255, 0]
    assert api.state_consensus(np.array(m, dtype=np.float64) * 0 + 3, [np.arange(4)])[:, 0].tolist() == [3] * 5


def test_invalid_state_byte_is_rejected():
    from infercnv_b200 import _lib, api
    m = np.full((40, 6), 3, dtype=np.uint8)
    m[17, 2] = 9
    with pytest.raises(_lib.InfercnvB200Error) as e:
        api.state_consensus(m, [np.arange(6)])
    assert e.value.code == -3


@pytest.mark.parametrize("lens", [[598, 615, 1, 2, 9, 1300, 1, 1, 475], [1024, 1024, 2048], [5, 1, 1], [3000]])
def test_region_calling_matches_the_oracle(lens):
    from infercnv_b200 import api
    rng = np.random.default_rng(sum(lens))
    cs, cl = _layout(lens)
    G, n_seq = int(cl.sum()), 9
    S = _states(rng, G, n_seq, p_noise=0.05, unassigned=0.15)
    gs = np.cumsum(rng.integers(1, 1000, size=G)).astype(np.float64)
    ge = gs + rng.integers(1, 50000, size=G)              # long genes: max(stop) is not the last gene's stop
    got = api.cnv_regions(S, cs, cl, gs, ge)
    want = orr.cnv_regions(S, cs, cl, gs, ge)
    _same_regions(got, want)
    # literal transcription of .define_cnv_gene_regions / .get_cnv_gene_region_bounds for one sequence
    codes = np.repeat(np.arange(len(cl)), cl)
    names = ["chr%d" % (k + 1) for k in range(len(cl))]
    col = np.where(S[:, 4] == 255, -1, S[:, 4].astype(np.int64))
    lit, _ = orr.literal_define_cnv_gene_regions(col, codes, names, 0)
    sel = got["seq"] == 4
    assert [(g[0], g[-1], st) for _, st, g in lit] == list(zip(got["first_gene"][sel], got["last_gene"][sel], got["state"][sel]))
    bounds = orr.literal_cnv_gene_region_bounds(lit, gs, ge)
    assert [(lo, hi) for _, _, lo, hi in bounds] == list(zip(got["start"][sel], got["end"][sel]))


def test_predicted_regions_consensus_and_cell_modes():
    from infercnv_b200 import api
    rng = np.random.default_rng(5)
    cs, cl = _layout([300, 1, 450, 2, 271])
    G, C = int(cl.sum()), 300
    S = _states(rng, G, C, p_noise=0.3)
    gs = np.arange(G, dtype=np.float64) * 100
    ge = gs + 250
    groups = [np.arange(0, 30), np.arange(30, 290), np.arange(290, 300)]
    reg, cons = api.predicted_cnv_regions(S, cs, cl, gs, ge, groups, want_consensus=True)
    want_cons = np.stack([orr.state_consensus(S, g) for g in groups], axis=1)
    assert np.array_equal(cons, want_cons)
    _same_regions(reg, orr.cnv_regions(want_cons, cs, cl, gs, ge))
    # by = "cell": single-cell groups in an arbitrary order read the state matrix directly
    order = rng.permutation(C)[:77]
    reg = api.predicted_cnv_regions(S, cs, cl, gs, ge, [np.array([i]) for i in order])
    _same_regions(reg, orr.cnv_regions(S[:, order], cs, cl, gs, ge))


def test_reference_bundled_known_answer_and_report_files(tmp_path):
    """data/HMM_states.rda -> generate_cnv_region_reports(by="subcluster") == what data/mcmc_obj.rda recorded of
    the reference's own run; the four files byte for byte against the oracle's write.table restatement."""
    from mirror import ops
    z = np.load(GOLD)
    codes = z["chr_codes"]
    levels = [str(s) for s in z["chr_levels"]]
    sub = z["subcluster_cells"] - 1
    obj = ops.Infercnv(expr_data=z["hmm_states"].astype(np.float64), gene_order_chr=codes,
                       reference_grouped_cell_indices={"normal": z["ref_idx"] - 1},
                       observation_grouped_cell_indices={"tumor": z["obs_idx"] - 1},
                       tumor_subclusters={"subclusters": {"tumor": {"tumor_s1": sub}}},
                       gene_names=[str(s) for s in z["gene_names"]], gene_order_start=z["gene_start"],
                       gene_order_stop=z["gene_stop"], cell_names=[str(s) for s in z["cell_names"]],
                       chr_names={i + 1: n for i, n in enumerate(levels)})
    regions = ops.get_predicted_CNV_regions(obj, by="subcluster")
    assert [g["cell_group_name"] for g in regions] == ["tumor.tumor_s1"]
    r, gr = regions[0]["cnv_ranges"], regions[0]["gene_regions"]
    got = [(n, a + 1, b + 1, b - a + 1) for n, st, a, b in zip(r["cnv_name"], r["state"], gr["first_gene"], gr["last_gene"])
           if st != 3]
    want = list(zip(z["region_names"].tolist(), z["region_first_gene"].tolist(), z["region_last_gene"].tolist(),
                    z["region_n_genes"].tolist()))
    assert got == want
    assert sorted(regions[0]["cells"]) == sorted(str(z["cell_names"][i - 1]) for i in z["region_cells"][0])

    starts = np.flatnonzero(np.concatenate([[True], codes[1:] != codes[:-1]]))
    lens = np.diff(np.concatenate([starts, [len(codes)]]))
    for by, neutral in (("subcluster", 3), ("consensus", 3), ("cell", None)):
        ops.generate_cnv_region_reports(obj, "17_HMM_pred." + by, str(tmp_path), ignore_neutral_state=neutral, by=by)
        ref = orr.predicted_cnv_regions(z["hmm_states"], starts, lens, levels, obj.gene_names, z["gene_start"],
                                        z["gene_stop"], obj.cell_names, obj.reference_grouped_cell_indices,
                                        obj.observation_grouped_cell_indices, obj.tumor_subclusters["subclusters"], by=by)
        text = orr.cnv_region_reports(ref, [levels[c - 1] for c in codes], obj.gene_names, z["gene_start"], z["gene_stop"],
                                      ignore_neutral_state=neutral)
        for suffix, want_text in text.items():
            with open(os.path.join(str(tmp_path), "17_HMM_pred.%s.%s" % (by, suffix))) as f:
                assert f.read() == want_text, (by, suffix)


def test_full_size_round_trip_and_run_count():
    """BASELINE configs[1] shape in by-cell mode (10 000 genes x 2 000 cells here): decoding the records (run-length
    expand) gives back the state matrix on every chromosome of >= 2 genes, and the record count equals the number
    of state changes + chromosome starts."""
    from infercnv_b200 import api
    rng = np.random.default_rng(11)
    t = np.array([852, 615, 535, 288, 420, 453, 458, 297, 349, 363, 514, 472, 162, 301, 274, 397, 546, 126, 545, 239, 90, 212])
    lens = np.floor(t * 10000 / t.sum()).astype(np.int64)
    lens[0] += 10000 - lens.sum() - 1
    lens = np.concatenate([lens, [1]])                      # one single-gene chromosome, never reported
    cs, cl = _layout(lens)
    G, C = 10000, 2000
    S = _states(rng, G, C, p_noise=0.01)
    gs = np.arange(G, dtype=np.float64)
    reg = api.predicted_cnv_regions(S, cs, cl, gs, gs + 1, [np.array([i]) for i in range(C)])
    valid = np.repeat(cl >= 2, cl)
    first = np.zeros(G, dtype=bool)
    first[cs] = True
    change = np.concatenate([np.ones((1, C), dtype=bool), S[1:] != S[:-1]], axis=0) | first[:, None]
    assert len(reg["seq"]) == int((change & valid[:, None]).sum())
    n = reg["last_gene"] - reg["first_gene"] + 1
    assert n.min() >= 1 and int(n.sum()) == int(valid.sum()) * C
    back = np.full((G, C), 200, dtype=np.uint8)
    back[np.concatenate([np.arange(a, b + 1) for a, b in zip(reg["first_gene"], reg["last_gene"])]),
         np.repeat(reg["seq"], n)] = np.repeat(reg["state"], n)
    assert np.array_equal(back[valid], S[valid])
    assert np.array_equal(reg["start"], reg["first_gene"]) and np.array_equal(reg["end"], reg["last_gene"] + 1.0)
    assert np.all(np.diff(reg["seq"].astype(np.int64) * G + reg["first_gene"]) > 0)      # (sequence, position) order


def test_device_resident_states_from_the_viterbi_kernel_to_regions():
    """Engine path: states stay on the GPU between the HMM and the region calls (no PCIe round trip of the matrix);
    a strided view (column stride > G) exercises lds != G."""
    import torch
    from infercnv_b200.device import Engine
    eng = Engine(0)
    rng = np.random.default_rng(3)
    cs, cl = _layout([700, 2, 1, 333])
    G, C = int(cl.sum()), 130
    S = _states(rng, G, C, p_noise=0.2, unassigned=0.1)
    gs = np.arange(G, dtype=np.float64) * 10
    ge = gs + 95
    wide = torch.zeros((C, G + 4), dtype=torch.uint8, device="cuda")
    wide[:, :G] = torch.from_numpy(np.ascontiguousarray(S.T)).cuda()
    groups = [np.arange(0, 100), np.arange(100, 130), np.array([7])]
    for dS in (wide[:, :G].contiguous(), wide[:, :G]):
        cons = eng.state_consensus(dS, groups)
        want = np.stack([orr.state_consensus(S, g) for g in groups], axis=0)
        assert np.array_equal(cons.cpu().numpy(), want)
        _same_regions(eng.cnv_regions(cons, cs, cl, gs, ge), orr.cnv_regions(want.T, cs, cl, gs, ge))
        cells = [5, 0, 129, 64]
        _same_regions(eng.cnv_regions(dS, cs, cl, gs, ge, cols=cells), orr.cnv_regions(S[:, cells], cs, cl, gs, ge))


def test_engine_slab_pipelined_host_path_is_bit_identical():
    """Engine.smooth_hmm_host (reference columns first, then H2D / pass 2 + Viterbi / D2H overlapped over cell slabs on three
    streams, pinned host tensors) against smooth_block + viterbi on the uploaded matrix: identical bits."""
    import torch
    from infercnv_b200.device import Engine
    from oracle import oracle as orc
    eng = Engine(0)
    cs, cl = _layout([700, 2, 1, 333, 1200, 90])
    G, C = int(cl.sum()), 700
    refs = [np.arange(0, 40), np.arange(40, 64)]
    X = eng.synth(G, cs, cl, np.arange(C), C, 20260923)
    Y, f1 = eng.smooth_block(X, cs, cl, refs)
    mean = np.array([0.41234766, 0.84075773, 1.01693983, 1.12238786, 1.23842619, 1.44298781])
    sd = np.array([0.028893, 0.164549, 0.105553, 0.190574, 0.244093, 0.290072])
    Pi, delta = orc.hmm_params(6)
    S, f2 = eng.viterbi(Y, cs, cl, Pi, delta, mean, sd)
    hX = torch.empty((C, G), dtype=torch.float64, pin_memory=True)
    hX.copy_(X)
    hY = torch.empty((C, G), dtype=torch.float64, pin_memory=True)
    hS = torch.empty((C, G), dtype=torch.uint8, pin_memory=True)
    for slab in (128, 333):
        hY.zero_()
        hS.zero_()
        flags = eng.smooth_hmm_host(hX, hY, hS, torch.empty_like(X), torch.empty_like(X), torch.empty_like(S), cs, cl, refs, None,
                                    None, Pi, delta, mean, sd, slab_cells=slab)
        assert all(int(f.item()) == 0 for f in flags) and int(f1.item()) == 0 and int(f2.item()) == 0
        assert torch.equal(hY, Y.cpu()) and torch.equal(hS, S.cpu())
