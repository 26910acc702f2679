"""xg_local_phase against the host reference (reg_local_phasing region by region, in list order), and
afc_wrapper(phase_from_reads=True) against the pileup -> cellsnp_dir composition it replaces."""

import logging
import os
import re
import warnings

import numpy as np
import pytest

import local_phase_cases as lpc
from test_gpu_bam_index import library  # noqa: F401  (module fixture: the indexed synthetic library)

pytestmark = pytest.mark.gpu


def assert_same(ctx, case, expect_phased=None):
    host = lpc.host_run(case)
    dev = lpc.device_run(ctx, case)
    diff = [k for k, (a, b) in enumerate(zip(host["flips"], dev["flips"])) if a != b]
    assert not diff, (case.name, [(getattr(case, "names", {}).__getitem__(k) if hasattr(case, "names") else k,
                                   host["flips"][k], dev["flips"][k]) for k in diff[:5]])
    for k in ("lists", "flips", "ref_idx", "alt_idx", "gt", "counters"):
        assert dev[k] == host[k], (case.name, k)
    if expect_phased is not None:
        assert [f is not None for f in host["flips"]] == expect_phased, case.name
    return host, dev


@pytest.mark.parametrize("with_ref_cells", [False, True])
def test_golden_c2_regions(gpu_ctx, with_ref_cells):
    case, _cols, _data, _col_of = lpc.golden_c2(with_ref_cells)
    host, dev = assert_same(gpu_ctx, case)
    assert host["counters"][0] == 65 and host["counters"][3] > 0
    t = dev["timing"]
    assert t[3] == 65 and t[2] >= 1 and t[4] > 0


def test_bch869_regions(gpu_ctx, tmp_path):
    """The long regions of bch869_smartseq with the oracle's per-SNP counts: few cells, deep counts, and regions
    whose flips sit within rounding of a tie."""
    from test_gpu_snp_pileup import golden_inputs, oracle_dir
    r = golden_inputs("bch869_smartseq")
    oracle_dir(r, str(tmp_path / "csp"))
    case, _cols, _data, _col_of = lpc.cellsnp_case(r["features"], r["snps"], str(tmp_path / "csp"), name="bch869")
    host, dev = assert_same(gpu_ctx, case)
    assert host["counters"][0] == 70 and dev["timing"][10] >= 2


@pytest.mark.parametrize("args", [
    (11, 1000, 5000, 0.02, 5000, 1, 0),        # 1 000 SNPs x 5 000 cells in one region
    (12, 300, 2000, 0.05, 15000, 6, 10),       # overlapping regions: several waves
    (13, 120, 400, 0.1, 40000, 8, 5),
    (14, 60, 3000, 0.01, 100000, 3, 20),       # SNPs beyond each other's smoothing window
])
def test_seeded_imbalanced_regions(gpu_ctx, args):
    case = lpc.imbalanced(*args)
    host, dev = assert_same(gpu_ctx, case)
    assert all(f is not None for f in host["flips"])
    if args[5] > 1:
        assert dev["timing"][2] > 1


def _edge(name, AD, DP, spacing=100000, ref0=None):
    AD, DP = np.asarray(AD), np.asarray(DP)
    n = DP.shape[1]
    return lpc.Case(1000 + np.arange(n) * spacing, np.zeros(n, np.int64) if ref0 is None else ref0, AD, DP,
                    [list(range(n))], name)


def _imbalanced_block(n_cells, n_snps):
    """Depth 5 everywhere; AD 4 or 1 by cell parity, the other way round at SNP 0 (so no cell's BAF is 0.5 for
    3 SNPs or more)."""
    ad = np.where((np.arange(n_cells)[:, None] % 2 == 0) != (np.arange(n_snps)[None, :] == 0), 4, 1)
    return ad, np.full((n_cells, n_snps), 5)


class _Counts(object):
    """Counts the host reference's EM calls and iterations (phasing_em calls _loglik once per iteration + once)."""

    def __init__(self, mp):
        import xcltk_b200.baf.localphase as lp
        self.em, self.loglik = [], []
        real_em, real_ll = lp.phasing_em, lp._loglik

        def em(*a, **k):
            self.loglik.append(0)
            self.em.append(1)
            return real_em(*a, **k)

        def ll(*a, **k):
            self.loglik[-1] += 1
            return real_ll(*a, **k)
        mp.setattr(lp, "phasing_em", em)
        mp.setattr(lp, "_loglik", ll)


def test_nan_poisoned_round_and_the_1000_iteration_cap(gpu_ctx, monkeypatch):
    # SNP 4 is expressed by cell 0 only, whose BAF is 0.5: the filter removes it, SNP 4's starting Z is 0/0
    ad, dp = _imbalanced_block(6, 5)
    ad[:, 4] = dp[:, 4] = 0
    ad = np.vstack([np.zeros((1, 5), int), ad])
    dp = np.vstack([np.zeros((1, 5), int), dp])
    ad[0, 4], dp[0, 4] = 1, 2
    case = _edge("nan", ad, dp)
    from xcltk_b200.baf.localphase import phasing_em
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        Z, _th, ll = phasing_em(np.array([[3, 0], [0, 2], [0, 0]]), np.array([[3, 0], [0, 2], [0, 0]]), None)
    assert np.isnan(Z).all() and np.isnan(ll)          # one SNP without depth: everything NaN
    cnt = _Counts(monkeypatch)
    lpc.host_run(case)
    assert len(cnt.em) == 6 and max(cnt.loglik) == 1001      # rounds 0..5, each EM at its 1000-iteration cap
    monkeypatch.undo()
    host, dev = assert_same(gpu_ctx, case, [True])
    assert host["flips"] == [[0, 0, 0, 0, 0]] and dev["timing"][10] == 0


def test_no_cells_left_fails(gpu_ctx):
    dp = np.full((4, 3), 2)
    assert_same(gpu_ctx, _edge("no_cells", dp // 2, dp), [False])


def test_every_snp_unexpressed(gpu_ctx):
    z = np.zeros((5, 4), int)
    host, _dev = assert_same(gpu_ctx, _edge("unexpressed", z, z), [False])
    assert host["lists"] == [[]] and host["counters"] == (1, 1, 0, 0)


def test_some_snps_unexpressed_are_pruned(gpu_ctx):
    ad, dp = _imbalanced_block(8, 6)
    ad[:, [1, 4]] = dp[:, [1, 4]] = 0
    host, _dev = assert_same(gpu_ctx, _edge("pruned", ad, dp), [True])
    assert host["lists"] == [[0, 2, 3, 5]]


def test_one_cell(gpu_ctx):
    ad, dp = _imbalanced_block(1, 4)
    assert_same(gpu_ctx, _edge("one_cell", ad, dp), [True])


def test_cell_baf_exactly_at_the_bounds(gpu_ctx):
    ad, dp = _imbalanced_block(6, 4)
    extra_ad = np.array([[9, 0, 0, 0], [11, 0, 0, 0], [0, 9, 0, 0], [0, 0, 11, 0]])
    extra_dp = np.array([[20, 0, 0, 0], [20, 0, 0, 0], [0, 20, 0, 0], [0, 0, 20, 0]])
    assert_same(gpu_ctx, _edge("baf_bounds", np.vstack([ad, extra_ad]), np.vstack([dp, extra_dp])), [True])


def test_flip_mean_of_exactly_one_half_is_not_inverted(gpu_ctx):
    from xcltk_b200.baf.localphase import snp_local_phasing
    case = lpc.small_seeded(6)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        raw = snp_local_phasing(case.AD, case.DP, case.pos)
    assert raw is not None and np.mean(raw) == 0.5
    host, _dev = assert_same(gpu_ctx, case, [True])
    assert host["flips"][0] == raw.astype(int).tolist()


def test_the_50_round_cap(gpu_ctx):
    """A region whose rounds keep flipping a proper subset until the cap.  Such oscillation happens around a flip
    decision of |Z1 - Z0| ~ 1 ulp, so the device reports a tie and the reference decides; the result is the same."""
    case = lpc.small_seeded(24)
    with pytest.MonkeyPatch.context() as mp:
        cnt = _Counts(mp)
        lpc.host_run(case)
        assert len(cnt.em) == 50
    _host, dev = assert_same(gpu_ctx, case, [True])
    assert dev["timing"][10] == 1


def test_shared_snps_need_the_waves(gpu_ctx):
    """Two regions sharing six SNPs: with the waves the device equals the host; without them -- each region starting
    from the starting orientation, the flips combined afterwards -- the result differs."""
    from xcltk_b200.baf.fc.phasing import phase_layout
    case = lpc.imbalanced(0, 16, 30, 0.5, 100000, n_regions=2, overlap=6)
    host, dev = assert_same(gpu_ctx, case, [True, True])
    assert dev["timing"][2] == 2
    start = case.ref0.astype(np.uint8)
    ref = start.copy()
    for ids in case.regions:
        layout = phase_layout([ids], case.csr(), case.DP.shape[0])
        layout["wave_ptr"] = np.array([0, 1], dtype=np.int32)
        r = start.copy()
        _keep, _flip, status = gpu_ctx.local_phase(case.pos, r, layout)
        assert status.tolist() == [1]
        ref ^= r ^ start
    assert ref.tolist() != host["ref_idx"]


def test_two_runs_give_the_same_bytes(gpu_ctx):
    from xcltk_b200.baf.fc.phasing import phase_layout, phase_waves
    case = lpc.imbalanced(12, 300, 2000, 0.05, 15000, 6, 10)
    w = phase_waves(case.regions)
    order = np.argsort(w, kind="stable")
    layout = phase_layout([case.regions[i] for i in order], case.csr(), case.DP.shape[0])
    layout["wave_ptr"] = np.searchsorted(w[order], np.arange(w.max() + 2)).astype(np.int32)
    outs = []
    for _ in range(2):
        ref = case.ref0.astype(np.uint8)
        keep, flip, status = gpu_ctx.local_phase(case.pos, ref, layout)
        outs.append(b"".join(x.tobytes() for x in (keep, flip, status, ref)))
    assert outs[0] == outs[1]


# ---- end to end ----------------------------------------------------------------------------------------------------

PHASE_LINES = re.compile(r"^#(regions: total=\d+; local_phasing=.*|SNPs: local_phasing=.*)$")
AFC_FILES = ("xcltk.region.tsv", "xcltk.samples.tsv", "xcltk.AD.mtx", "xcltk.DP.mtx", "xcltk.OTH.mtx")


def _count_loads(mp):
    from xcltk_b200 import engine
    n = {"load_reads": 0, "load_reads_multi": 0, "load_reads_sharded": 0}
    for name in n:
        real = getattr(engine, name)

        def spy(*a, _real=real, _name=name, **kw):
            b = _real(*a, **kw)
            if b is not None:
                n[_name] += 1
            return b
        mp.setattr(engine, name, spy)
    return n


def _afc(caplog, out, inp, **kw):
    from xcltk_b200.baf.fc.main import afc_wrapper
    caplog.clear()
    with caplog.at_level(logging.INFO):
        assert afc_wrapper(inp["sam"], inp["barcodes"], inp["features"], inp["snps"], out, ncores=4,
                           output_all_reg=True, **inp["kw"], **kw) == 0
    lines = [r.getMessage() for r in caplog.records if PHASE_LINES.match(r.getMessage())]
    assert len(lines) == 2
    return {f: open(os.path.join(out, f), "rb").read() for f in AFC_FILES}, lines


def _end_to_end(inp, tmp_path, monkeypatch, caplog, ref_cell_fn=None):
    from xcltk_b200.baf.pileup import pileup_wrapper
    csd = str(tmp_path / "cellsnp")
    assert pileup_wrapper(inp["sam"], inp["barcodes"], inp["snps"], csd, ncores=4, **inp["kw"]) == 0
    exp, exp_lines = _afc(caplog, str(tmp_path / "two_step"), inp, cellsnp_dir=csd, ref_cell_fn=ref_cell_fn)
    assert int(re.search(r"local_phasing=(\d+)", exp_lines[0]).group(1)) > 0
    for mode in ("device", "host", "sharded"):
        with monkeypatch.context() as mp:
            if mode == "host":
                mp.setenv("XCLTK_B200_DEVICE_DECODE", "0")
            if mode == "sharded":
                mp.setenv("XCLTK_B200_GPUS", "2")
                mp.setenv("XCLTK_B200_EMULATE_SHARDS", "1")
            n = _count_loads(mp)
            got, lines = _afc(caplog, str(tmp_path / mode), inp, phase_from_reads=True, ref_cell_fn=ref_cell_fn)
        assert sum(n.values()) == 1, (mode, n)
        if mode == "sharded":
            assert n["load_reads_sharded"] + n["load_reads_multi"] == 1, n
        assert lines == exp_lines, mode
        assert got == exp, mode
    return exp


@pytest.mark.parametrize("ref_cells", [False, True])
def test_c1_chr22_10x_equals_the_two_step_composition(gpu_ctx, tmp_path, monkeypatch, caplog, ref_cells):
    from test_gpu_snp_pileup import golden_inputs
    inp = golden_inputs("c1_chr22_10x")
    exp = _end_to_end(inp, tmp_path, monkeypatch, caplog,
                      os.path.join(lpc.C2, "ref_cells.tsv") if ref_cells else None)
    assert exp["xcltk.DP.mtx"].count(b"\n") > 10


def test_bch869_smartseq_equals_the_two_step_composition(gpu_ctx, tmp_path, monkeypatch, caplog):
    from test_gpu_snp_pileup import golden_inputs
    _end_to_end(golden_inputs("bch869_smartseq"), tmp_path, monkeypatch, caplog)


def test_indexed_synthetic_library_equals_the_two_step_composition(gpu_ctx, library, tmp_path,  # noqa: F811
                                                                    monkeypatch, caplog):
    import bai
    from xcltk_b200 import synth
    bam = library["bams"][0]
    ft = str(tmp_path / "features.tsv")
    # long regions (>= 50 kb with SNPs >= 50 kb apart) that overlap each other, beside the library's features
    feats = [f for f in library["feats"] if f[0] in ("2", "22")]
    feats += [("2", b, b + 160000, "long%d" % b) for b in range(100000, 1500000, 90000)]
    feats.sort(key=lambda f: (int(f[0]), f[1]))
    synth.write_features(ft, [("chr" + c, s, e, n) for c, s, e, n in feats])
    bai.index_bam(bam)
    try:
        inp = dict(sam=bam, barcodes=library["barcodes"], features=ft, snps=library["snp_tsv"], kw={})
        _end_to_end(inp, tmp_path, monkeypatch, caplog)
    finally:
        os.remove(bam + ".bai")
