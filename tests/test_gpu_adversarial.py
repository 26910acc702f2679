"""Adversarial record / feature sets built directly as arrays (lib.ArrayReads) to force every
fallback of the counting kernels -- index slices that do not fit shared memory, stabbing
lists and CIGAR streams beyond the staging caps, the direct-insert path when the pair stage
overflows, reads with >= 255 CIGAR ops, tiles of exactly 1024 / 1025 records, features that
are duplicated, nested, empty or unfetchable -- each compared bit-exactly with the CPU oracle."""

import numpy as np
import pytest

from xcltk_b200 import engine, lib

pytestmark = pytest.mark.gpu

M, I, D, N, S = 0, 1, 2, 3, 4


class Conf(object):
    min_mapq, min_len, min_include = 0, 1, 0.5
    incl_flag, excl_flag, no_orphan = 0, 0, False

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def use_barcodes(self):
        return True

    def use_umi(self):
        return True


def build_reads(rng, n, contig_len, cigar_kind, n_cells, n_umis, ks, n_contigs=1, with_seq=False):
    """n reads per contig, sorted by pos; cigar_kind(rng, k) -> list of (op, len) or None = simple."""
    pos_end, fmq, cig_off, keys, cigar, runs = [], [], [0], [], [], []
    seq_off, seq = [], []
    def bc(c):
        return "".join("ACGT"[(c >> (2 * t)) & 3] for t in range(10)) + "-%d" % (c % 10)
    cells = [ks.encode(bc(c)) if c % 7 else ks.encode("cell_%d" % c) for c in range(n_cells + 3)]
    cell_keys = np.array(cells[:n_cells], dtype=np.uint64)
    for g in range(n_contigs):
        beg = len(fmq)
        ps = np.sort(rng.randint(0, contig_len, size=n))
        for k, p in enumerate(ps):
            ops = cigar_kind(rng, k)
            if ops is None:
                L = int(rng.randint(20, 120))
                end, ncw = p + L, 0
            else:
                rlen = sum(l for op, l in ops if op in (M, D, N, 7, 8))
                end = p + max(rlen, 1)
                if len(ops) >= 255:
                    cigar.append(len(ops))
                    ncw = 255
                else:
                    ncw = len(ops)
                cig_off[-1] = len(cigar)
                cigar.extend((l << 4) | op for op, l in ops)
            cig_off.append(len(cigar))
            pos_end.append((int(p), int(end)))
            flag = int(rng.choice([0, 16, 256, 1024, 99, 1]))
            fmq.append(flag | (int(rng.choice([0, 3, 20, 255])) << 16) | (ncw << 24))
            c = int(rng.randint(0, n_cells + 3))
            ck = cells[c] if rng.rand() > 0.03 else lib.XG_KEY_NONE
            r = rng.rand()
            uk = lib.XG_KEY_NONE if r < 0.03 else lib.XG_KEY_EMPTY if r < 0.05 else \
                ks.encode("".join("ACGT"[x] for x in rng.randint(0, 4, size=10)) if n_umis is None
                          else "UMI%d" % rng.randint(0, n_umis))
            keys.append((ck, uk))
        runs.append((0, g, beg, len(fmq)))
    # cig_off[i] must be the first word of read i: rebuild as a clean prefix array
    off = [0]
    ci = 0
    words = []
    rebuilt = []
    idx = 0
    for i, f in enumerate(fmq):
        ncw = f >> 24
        if ncw == 0:
            rebuilt.append(len(words))
            continue
        start = cig_off[i]
        if ncw == 255:
            cnt = cigar[start - 1]
            words.append(cnt)
            rebuilt.append(len(words))
            words.extend(cigar[start:start + cnt])
        else:
            rebuilt.append(len(words))
            words.extend(cigar[start:start + ncw])
    rebuilt.append(len(words))
    max_aln = 4096
    return lib.ArrayReads(np.array(pos_end, dtype=np.int32), np.array(fmq, dtype=np.uint32),
                          np.array(rebuilt, dtype=np.uint32), np.array(keys, dtype=np.uint64),
                          np.array(words, dtype=np.uint32), runs, max_aln_len=max_aln, max_span=1 << 20), cell_keys


def compare(ctx, reads, cell_keys, gid, beg, end, conf, n_cells):
    from oracle import oracle
    gid, beg, end = (np.asarray(a, dtype=np.int32) for a in (gid, beg, end))
    d = ctx.upload(reads)
    try:
        params = engine.make_params(conf, reads.max_aln_len, with_include=True)
        row, col, val, _ = ctx.basefc(d, gid, beg, end, cell_keys, n_cells, params)
        o = oracle.basefc(reads, gid, beg, end, cell_keys, n_cells, oracle.params(conf), 2)
    finally:
        d.close()
    assert np.array_equal(row, o[0]) and np.array_equal(col, o[1]) and np.array_equal(val, o[2])
    return len(val)


def simple(rng, k):
    return None


def spliced(rng, k):
    a = int(rng.randint(5, 60))
    return [(M, a), (N, int(rng.randint(50, 3000))), (M, int(rng.randint(5, 60))), (I, 2), (D, 3), (M, 7), (S, 4)]


def mixed(rng, k):
    r = rng.rand()
    if r < 0.5:
        return None
    if r < 0.9:
        return spliced(rng, k)
    if r < 0.95:
        return []                                      # no CIGAR at all (stored as one 0-length P)
    return [(M, 2), (I, 1)] * 150                      # 300 ops: count word before the stream


@pytest.mark.parametrize("n", [1, 1023, 1024, 1025, 2049])
def test_tile_boundaries(gpu_ctx, n):
    rng = np.random.RandomState(n)
    ks = lib.KeySpace()
    reads, ck = build_reads(rng, n, 20000, mixed, 20, 30, ks)
    feats = [(0, 0, 20000), (0, 5000, 5100), (0, 5050, 5060), (0, 100, 19000)]
    nnz = compare(gpu_ctx, reads, ck, *zip(*feats), Conf(), 20)
    assert nnz > 0 or n == 1


def test_many_tiny_features_exceed_the_staged_boundary_slice(gpu_ctx):
    """Far more than SB_MAX (128) boundaries under one tile window: global binary search path."""
    rng = np.random.RandomState(1)
    ks = lib.KeySpace()
    reads, ck = build_reads(rng, 3000, 60000, mixed, 50, None, ks)
    starts = np.arange(0, 60000, 40)
    feats = [(0, int(s), int(s) + int(rng.randint(5, 120))) for s in starts] + [(0, 0, 60000)]
    assert compare(gpu_ctx, reads, ck, *zip(*feats), Conf(min_include=0.2), 50) > 1000


def test_deep_nesting_exceeds_stab_and_pair_stage(gpu_ctx):
    """400 nested features over the same span: stabbing lists > 256 entries per segment and far
    more (read, feature) pairs than the pair stage holds -> direct-insert path."""
    rng = np.random.RandomState(2)
    ks = lib.KeySpace()
    reads, ck = build_reads(rng, 5000, 30000, mixed, 40, 200, ks)
    feats = [(0, 100 + 7 * k, 29000 - 5 * k) for k in range(400)]
    feats += [feats[3], feats[3]]                                        # duplicated rows
    assert compare(gpu_ctx, reads, ck, *zip(*feats), Conf(min_include=1), 40) > 10000


def test_all_spliced_exceeds_cigar_stage(gpu_ctx):
    """Every read carries 7 CIGAR ops: > 1024 words per tile -> CIGAR read from global memory."""
    rng = np.random.RandomState(3)
    ks = lib.KeySpace()
    reads, ck = build_reads(rng, 4000, 200000, spliced, 30, None, ks)
    feats = [(0, int(s), int(s) + 4000) for s in range(0, 200000, 3000)]
    for conf in (Conf(), Conf(min_include=30), Conf(min_include=0.95, min_len=40)):
        compare(gpu_ctx, reads, ck, *zip(*feats), conf, 30)


def test_unfetchable_and_empty_features_multi_contig(gpu_ctx):
    rng = np.random.RandomState(4)
    ks = lib.KeySpace()
    reads, ck = build_reads(rng, 2500, 50000, mixed, 10, 50, ks, n_contigs=3)
    feats = [(0, 0, 50000), (-1, 0, 100), (1, 100, 100), (1, 200, 150), (2, 49990, 60000), (5, 0, 10),
             (2, 0, 1), (1, 0, 50000), (0, 49999, 50000), (0, -5, 10)]
    gid, beg, end = (list(x) for x in zip(*feats))
    gid[9] = -1                                       # start <= 0 is resolved to "never fetched" by the host
    assert compare(gpu_ctx, reads, ck, gid, beg, end, Conf(), 10) > 0


@pytest.mark.parametrize("seed", range(6))
def test_random_small_cases(gpu_ctx, seed):
    rng = np.random.RandomState(100 + seed)
    ks = lib.KeySpace()
    n = int(rng.randint(1, 3000))
    L = int(rng.choice([500, 5000, 100000]))
    n_cells = int(rng.randint(1, 40))
    reads, ck = build_reads(rng, n, L, mixed, n_cells, int(rng.randint(1, 50)), ks, n_contigs=int(rng.randint(1, 4)))
    nf = int(rng.randint(1, 200))
    gid = rng.randint(-1, 4, size=nf)
    beg = rng.randint(0, L, size=nf)
    end = beg + rng.randint(-3, L // 2 + 2, size=nf)
    conf = Conf(min_include=float(rng.choice([0.0, 0.3, 0.9, 1.0, 25.0])), min_mapq=int(rng.choice([0, 3, 20])),
                min_len=int(rng.choice([1, 30])), excl_flag=int(rng.choice([0, 772, 1796])),
                no_orphan=bool(rng.randint(0, 2)), incl_flag=int(rng.choice([0, 0, 16])))
    if conf.min_include >= 1:
        conf.min_include = int(conf.min_include)
    compare(gpu_ctx, reads, ck, gid, beg, end, conf, n_cells)


# ------------------------------------------------------------------------------ baf
NT16 = "=ACMGRSVTWYHKDBN"


def add_sequences(rng, reads):
    """Random 4-bit sequences (incl. N, '=', IUPAC codes, and a few reads without SEQ)."""
    n = reads.n
    seq_off = np.zeros(n, dtype=np.uint32)
    words = []
    cig_off = reads._arrays["cig_off"]
    cigar = reads._arrays["cigar"]
    for i in range(n):
        f = int(reads.fmq[i])
        ncw = f >> 24
        if ncw == 0:
            qlen = int(reads.pos_end[i, 1] - reads.pos_end[i, 0])
        else:
            off = int(cig_off[i])
            cnt = int(cigar[off - 1]) if ncw == 255 else ncw
            qlen = sum(int(w >> 4) for w in cigar[off:off + cnt] if (int(w) & 15) in (0, 1, 4, 7, 8))
        if rng.rand() < 0.02 or qlen == 0:
            seq_off[i] = 0xFFFFFFFF
            continue
        codes = rng.choice([1, 2, 4, 8, 15, 0, 5, 10], p=[.23, .23, .23, .23, .03, .01, .02, .02], size=qlen)
        nb = (qlen + 1) // 2
        b = np.zeros(((nb + 3) // 4) * 4, dtype=np.uint8)
        b[:nb] = (np.pad(codes, (0, nb * 2 - qlen))[0::2] << 4) | np.pad(codes, (0, nb * 2 - qlen))[1::2]
        seq_off[i] = len(words)
        words.extend(b.view(np.uint32).tolist())
    a = reads._arrays
    return lib.ArrayReads(a["pos_end"].reshape(-1, 2), a["fmq"], a["cig_off"], a["keys"].reshape(-1, 2), a["cigar"],
                          reads.runs, seq_off, np.array(words if words else [0], dtype=np.uint32),
                          reads.max_aln_len, reads.max_span)


@pytest.mark.parametrize("seed", range(5))
def test_baf_random_cases(gpu_ctx, seed):
    from oracle import oracle
    rng = np.random.RandomState(500 + seed)
    ks = lib.KeySpace()
    n = int(rng.choice([1, 900, 1024, 1025, 4000]))
    L = int(rng.choice([300, 3000, 40000]))
    n_cells = int(rng.randint(1, 30))
    n_contigs = int(rng.randint(1, 3))
    reads, ck = build_reads(rng, n, L, mixed, n_cells, int(rng.randint(1, 40)), ks, n_contigs=n_contigs)
    reads = add_sequences(rng, reads)
    n_snps = int(rng.randint(1, 400))
    snp_gid = rng.randint(-1, n_contigs + 1, size=n_snps).astype(np.int32)
    snp_pos = rng.randint(0, L + 50, size=n_snps).astype(np.int32)
    if n_snps > 5:
        snp_pos[1], snp_gid[1] = snp_pos[0], snp_gid[0]                   # duplicate SNP rows are kept
    ref = rng.randint(0, 5, size=n_snps)
    alt = rng.randint(0, 5, size=n_snps)                                  # may equal ref, may be N
    letters = "ACGTN"
    ref_idx = rng.randint(0, 2, size=n_snps)
    n_reg = int(rng.randint(1, 60))
    reg = []
    for r in range(n_reg):                                                # overlapping regions share SNPs
        g = int(rng.randint(0, n_contigs))
        b = int(rng.randint(0, L))
        e = b + int(rng.randint(1, L))
        idx = np.nonzero((snp_gid == g) & (snp_pos >= b) & (snp_pos < e))[0]
        reg.append(idx[np.argsort(snp_pos[idx], kind="stable")])
    reg_ptr = np.concatenate([[0], np.cumsum([len(x) for x in reg])]).astype(np.int64)
    reg_snp = np.concatenate(reg + [np.zeros(0, np.int64)]).astype(np.int32)
    conf = Conf(min_include=0, min_mapq=int(rng.choice([0, 20])), min_len=int(rng.choice([1, 30])),
                excl_flag=int(rng.choice([0, 772])), no_orphan=bool(rng.randint(0, 2)))
    min_count, min_maf = int(rng.choice([1, 2, 4])), float(rng.choice([0, 0.1, 0.3]))
    no_dup = bool(rng.randint(0, 2))
    # hap table as SNP.gt = {ref: ref_idx, alt: alt_idx} gives it (ALT entry wins when ref == alt)
    hap = np.full((n_snps, 8), 2, dtype=np.uint8)
    ii = np.arange(n_snps)
    hap[ii, ref] = ref_idx
    hap[ii, alt] = 1 - ref_idx
    d = gpu_ctx.upload(reads)
    try:
        params = engine.make_params(conf, reads.max_aln_len, with_include=False)
        totals, st = gpu_ctx.baf_pileup(d, snp_gid, snp_pos, ck, n_cells, params)
        tot = totals.sum(axis=1)
        minor = np.minimum(totals[ii, ref], totals[ii, alt])
        keep = ((tot >= min_count) & ~(minor < tot * min_maf)).astype(np.uint8)
        got = gpu_ctx.baf_count(st, reg_ptr, reg_snp, hap, keep, no_dup)
        st.close()
    finally:
        d.close()
    exp = oracle.baf(reads, snp_gid, snp_pos, "".join(letters[x] for x in ref), "".join(letters[x] for x in alt),
                     ref_idx, 1 - ref_idx, reg_ptr, reg_snp, ck, n_cells, oracle.params(conf), min_count, min_maf,
                     no_dup, 2)
    for g, e in zip(got, exp):
        assert all(np.array_equal(np.asarray(a), b) for a, b in zip(g[:3], e))
