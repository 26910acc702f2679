"""Host side of local phasing from the reads (afc_wrapper(phase_from_reads=True)): the wave schedule, the region
layout handed to xg_local_phase, the per-region columns, the option conflict.  No GPU needed."""

import logging

import numpy as np
import pytest

import local_phase_cases as lpc
from xcltk_b200.baf.fc.phasing import csr_from_coo, phase_layout, phase_waves


def test_waves_chains_and_two_earlier_regions():
    lists = [[1, 2], [2, 3], [3, 4], [9], [4, 9], [1, 9], [20, 21], []]
    # r1 follows r0 (2), r2 follows r1 (3): a chain; r4 shares 4 with r2 (wave 2) and 9 with r3 (wave 0);
    # r5 shares 1 with r0 (wave 0) and 9 with r4 (wave 3); r6 and the empty r7 share nothing
    assert phase_waves(lists).tolist() == [0, 1, 2, 0, 3, 4, 0, 0]
    assert phase_waves([[5], [5], [5]]).tolist() == [0, 1, 2]
    assert phase_waves([]).tolist() == []


def test_waves_never_put_two_regions_with_a_shared_snp_together():
    rng = np.random.default_rng(3)
    lists = [sorted(set(rng.integers(0, 60, rng.integers(1, 8)).tolist())) for _ in range(200)]
    w = phase_waves(lists)
    for a in range(len(lists)):
        for b in range(a + 1, len(lists)):
            if set(lists[a]) & set(lists[b]):
                assert w[b] > w[a]
    # and as early as possible: a region after wave 0 shares a SNP with a region of the wave before it
    for b in range(len(lists)):
        if w[b] > 0:
            assert any(w[a] == w[b] - 1 and set(lists[a]) & set(lists[b]) for a in range(b))


def _dense_from_layout(lay, k, n_cells):
    """Region k's (AD, DP) over (its local cells, its slots), once from each order of the entries."""
    s0, s1 = lay["reg_snp_ptr"][k], lay["reg_snp_ptr"][k + 1]
    c0, c1 = lay["reg_cell_ptr"][k], lay["reg_cell_ptr"][k + 1]
    sm = np.zeros((2, c1 - c0, s1 - s0), dtype=np.int64)
    for j in range(s1 - s0):
        for e in range(lay["slot_ent_ptr"][s0 + j], lay["slot_ent_ptr"][s0 + j + 1]):
            sm[:, lay["sm_cell"][e], j] = lay["sm_ad"][e], lay["sm_dp"][e]
    cm = np.zeros_like(sm)
    for c in range(c1 - c0):
        snp = lay["cm_snp"][lay["cell_ent_ptr"][c0 + c]:lay["cell_ent_ptr"][c0 + c + 1]]
        assert np.all(np.diff(snp) > 0)
        for e in range(lay["cell_ent_ptr"][c0 + c], lay["cell_ent_ptr"][c0 + c + 1]):
            cm[:, c, lay["cm_snp"][e]] = lay["cm_ad"][e], lay["cm_dp"][e]
    return sm, cm


def test_layout_holds_each_region_in_both_orders():
    case = lpc.imbalanced(5, 40, 30, 0.2, 1000, n_regions=4, overlap=3)
    case.regions.append([])
    case.regions.append([0, 39])
    lay = phase_layout(case.regions, case.csr(), case.DP.shape[0])
    for k, ids in enumerate(case.regions):
        sm, cm = _dense_from_layout(lay, k, case.DP.shape[0])
        assert np.array_equal(sm, cm)
        live = case.DP[:, ids].sum(axis=1) > 0 if ids else np.zeros(case.DP.shape[0], bool)
        assert np.array_equal(sm[0], case.AD[np.ix_(live, ids)])
        assert np.array_equal(sm[1], case.DP[np.ix_(live, ids)])
        assert lay["reg_snp"][lay["reg_snp_ptr"][k]:lay["reg_snp_ptr"][k + 1]].tolist() == ids


def test_csr_drops_masked_cells_and_joins_ad_onto_dp():
    dp = (np.array([0, 0, 1, 2, 2]), np.array([0, 3, 1, 0, 2]), np.array([2, 1, 4, 3, 5]))
    ad = (np.array([0, 2, 2]), np.array([3, 0, 2]), np.array([1, 2, 5]))
    row_ptr, col, a, d = csr_from_coo(4, ad, dp, np.array([True, True, False, True]))
    assert row_ptr.tolist() == [0, 2, 3, 4, 4]
    assert col.tolist() == [0, 3, 1, 0]
    assert d.tolist() == [2, 1, 4, 3]
    assert a.tolist() == [0, 1, 0, 2]


@pytest.mark.parametrize("with_ref_cells", [False, True])
def test_region_columns_equal_the_cellsnp_path(with_ref_cells):
    """On the golden C2 inputs (SNP file sorted by position) a region's snp_list is exactly the cellsnp path's
    `cols`, and the layout gives each region the matrices afc_core hands reg_local_phasing."""
    case, cols, data, col_of = lpc.golden_c2(with_ref_cells)
    assert len(case.regions) == 65
    lay = phase_layout(case.regions, case.csr(), case.DP.shape[0], [sorted(x) for x in case.regions])
    ad_all, dp_all = data.AD.toarray(), data.DP.toarray()
    for k, (ids, c) in enumerate(zip(case.regions, cols)):
        assert col_of[ids].tolist() == c.tolist() == col_of[sorted(ids)].tolist()
        sm, _cm = _dense_from_layout(lay, k, case.DP.shape[0])
        live = dp_all[:, c].sum(axis=1) > 0
        assert np.array_equal(sm[0], ad_all[np.ix_(live, c)])
        assert np.array_equal(sm[1], dp_all[np.ix_(live, c)])


def test_unsorted_snp_file_pairs_file_order_counts_with_position_order_snps(tmp_path):
    """bch869's SNP file is not sorted by position: the cellsnp path's `cols` (cellSNP rows, file order) differ from
    snp_list (position order) in many regions, and are the region's SNP ids in file order, which is what the device
    layout counts with (row_lists)."""
    from test_gpu_snp_pileup import golden_inputs, oracle_dir
    r = golden_inputs("bch869_smartseq")
    oracle_dir(r, str(tmp_path / "csp"))
    case, cols, _data, col_of = lpc.cellsnp_case(r["features"], r["snps"], str(tmp_path / "csp"))
    assert col_of.tolist() == list(range(len(col_of)))
    assert sum(col_of[ids].tolist() != c.tolist() for ids, c in zip(case.regions, cols)) > 10
    for ids, c in zip(case.regions, cols):
        assert col_of[sorted(ids)].tolist() == c.tolist()
    lay = phase_layout(case.regions, case.csr(), case.DP.shape[0], [sorted(x) for x in case.regions])
    for k, ids in enumerate(case.regions):
        sm, _cm = _dense_from_layout(lay, k, case.DP.shape[0])
        live = case.DP[:, ids].sum(axis=1) > 0
        assert np.array_equal(sm[1], case.DP[np.ix_(live, sorted(ids))])
        assert lay["reg_snp"][lay["reg_snp_ptr"][k]:lay["reg_snp_ptr"][k + 1]].tolist() == ids


def test_phase_from_reads_with_cellsnp_dir_returns_minus_one(tmp_path, caplog):
    from xcltk_b200.baf.fc.main import afc_wrapper
    with caplog.at_level(logging.ERROR):
        rc = afc_wrapper(lpc.C1 + "/a.bam", lpc.C1 + "/barcodes.tsv", lpc.C1 + "/features.tsv",
                         lpc.C1 + "/snps.tsv", str(tmp_path / "out"), cellsnp_dir=lpc.C2 + "/cellsnp",
                         phase_from_reads=True)
    assert rc == -1
    assert "phase_from_reads" in caplog.text and "cellsnp_dir" in caplog.text


def test_config_uses_local_phasing_with_either_source():
    from xcltk_b200.baf.fc.config import Config
    conf = Config()
    assert not conf.use_local_phasing() and conf.phase_from_reads is False
    conf.phase_from_reads = True
    assert conf.use_local_phasing()
    conf.phase_from_reads, conf.cellsnp_dir = False, "x"
    assert conf.use_local_phasing()


class _AllTies(object):
    """Stands in for the device: reports every region as a tie (status 2), so that local_phasing_device decides
    each region with reg_local_phasing, one wave per call."""

    def __init__(self):
        self.calls = []

    def local_phase(self, pos, ref_idx, layout):
        n_slot, n_reg = len(layout["reg_snp"]), len(layout["reg_snp_ptr"]) - 1
        self.calls.append(n_reg)
        return np.ones(n_slot, np.uint8), np.zeros(n_slot, np.uint8), np.full(n_reg, 2, np.int8)

    def timing(self):
        return [0.0] * 16


def test_tie_regions_are_decided_by_the_reference_wave_by_wave():
    from xcltk_b200.baf.fc.phasing import local_phasing_device
    case = lpc.imbalanced(12, 300, 200, 0.1, 15000, 6, 10)
    host = lpc.host_run(case)
    snps = case.snps()
    regs = case.regs(snps)
    fake = _AllTies()
    flips, stats = local_phasing_device(fake, regs, snps, case.csr(), case.DP.shape[0])
    got = lpc._result(regs, snps, flips)
    for k in ("lists", "flips", "ref_idx", "alt_idx", "gt", "counters"):
        assert got[k] == host[k], k
    n_waves = int(phase_waves(case.regions).max()) + 1
    assert n_waves > 1 and len(fake.calls) == n_waves and fake.calls[0] == 6
    assert stats[9] == n_waves and stats[10] == 6
