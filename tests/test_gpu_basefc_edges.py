"""basefc at the switches of its segment finalize, its cell and UMI limits and its input caches, every case against
oracle.basefc (oracle.baf for the SNP table).  Each GPU case also asserts that it reached the route it names, from
Context.basefc_finalize_stats() (heavy features, careful ranges, fast-range overflows, sub-partition doublings per
CTA size) or timing()[14] / [15] (features counted in segments / in sets).

  light / heavy   a feature with at most LIGHT pair words keeps them in registers: 1 638 in the ordinary CTA
                  (256 threads, 4 096-slot table), 6 553 in the big one (1 024 threads, 16 384 slots, taken by
                  features with more than 4 096 candidate reads)
  column ranges   a heavy feature is split by ranges of 2^wshift cells (wshift_of below); a range with more than CAP
                  words takes the careful path; 96 probes without a slot on the fast path redo the range carefully,
                  and a careful pass that overflows doubles the hash sub-partitions
  cells           big CTAs up to BIG_CTA_MAX_COLS columns; pair words (segments) up to 2^19; the set finalize's
                  histogram holds 40 960 cells per pass
  candidates      more than 2^22 candidate reads: the feature keeps a set
  UMI keys        a pair word holds interned ids below 2^39 and packed UMIs of up to 13 symbols
  caches          the barcode table, the feature index and the SNP table are reused only for equal inputs; the
                  crafted inputs below have the same 64-bit hash as the first one

The hash mirrors (pair_hash, set_home, barcode_home, the cache hashes) are checked on the CPU: the crafted inputs
really collide."""

import struct

import numpy as np
import pytest

from recsets import build, cell_keys, umi_keys
from xcltk_b200 import engine

gpu = pytest.mark.gpu

M64 = (1 << 64) - 1
GOLD = 0x9E3779B97F4A7C15
FNV_OFF, FNV_P = 1469598103934665603, 1099511628211

TBL_LOG2 = {"ordinary": 12, "big": 14}                     # FS_TBL_LOG2 / FS_BIG_TBL_LOG2 (basefc.cu)
CAP = {k: (1 << v) * 2 // 5 for k, v in TBL_LOG2.items()}   # words of a table pass: 1 638 / 6 553
LIGHT = {"ordinary": min(CAP["ordinary"], 7 * 256), "big": min(CAP["big"], 7 * 1024)}
SEG_BIG = 4096                                             # candidate reads above which a feature takes a big CTA
SEG_MAX = 1 << 22                                          # candidate reads above which a feature keeps a set
FS_RANGES = 1024
HIST_COLS = 40 * 1024
FS_SHARED_BYTES = 4256                                     # sizeof(FsShared)


def big_cta_max_cols():
    """The most columns with which the big CTA's shared memory fits (basefc_plan)."""
    n = 32
    while (10 << 14) + (2 * ((n + 1 + 31) // 32) + 1) * 4 + FS_SHARED_BYTES + 1280 <= 200 * 1024:
        n += 1
    return n


BIG_CTA_MAX_COLS = big_cta_max_cols()


def wshift_of(n, n_cols, cta):
    """Range width (log2 cells) of a heavy feature of n words: k_basefc_finalize_segs.  Also returns the width before
    the FS_RANGES widening."""
    t = TBL_LOG2[cta]
    w = 5
    while w < t - 2 and (n << (w + 1)) <= (CAP[cta] * 3 // 4) * n_cols:
        w += 1
    w0 = w
    while ((n_cols - 1) >> w) + 1 > FS_RANGES:
        w += 1
    return w, w0


class Conf(object):
    min_mapq, min_len, min_include = 20, 1, 1
    incl_flag, excl_flag, no_orphan = 0, 0, False
    barcodes = True

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def use_barcodes(self):
        return self.barcodes

    def use_umi(self):
        return True


# ---------------------------------------------------------------------------------------------- hash mirrors
def pair_hash(pw):
    with np.errstate(over="ignore"):
        h = np.asarray(pw, np.uint64) * np.uint64(GOLD)
        h ^= h >> np.uint64(29)
        return h * np.uint64(0xBF58476D1CE4E5B9)


def fs_slot(pw, log2):
    """Home slot of a pair word in a finalize table of 2^log2 slots (fs_insert / fs_insert_range)."""
    with np.errstate(over="ignore"):
        return (pair_hash(pw) * np.uint64(GOLD)) >> np.uint64(64 - log2)


def colliding_umis(col, log2, count):
    """Packed-form UMI keys whose pair words with cell `col` all have the table's last slot as home."""
    k = np.arange(1, 1 << 22, dtype=np.uint64)
    umi = (k << np.uint64(30)) | np.uint64(1 << 28)
    hit = umi[fs_slot(umi | np.uint64(col), log2) == np.uint64((1 << log2) - 1)]
    assert len(hit) >= count
    return hit[:count]


def mix64(x):
    with np.errstate(over="ignore"):
        x = np.asarray(x, np.uint64)
        x = x ^ (x >> np.uint64(33))
        x = x * np.uint64(0xff51afd7ed558ccd)
        x = x ^ (x >> np.uint64(33))
        x = x * np.uint64(0xc4ceb9fe1a85ec53)
        return x ^ (x >> np.uint64(33))


def set_home(umi, col, cap):
    """Home slot of (cell, UMI) in a feature's set of cap slots (the counting kernel's set_home)."""
    with np.errstate(over="ignore"):
        h = mix64(np.asarray(umi, np.uint64) ^ (np.uint64(col) * np.uint64(GOLD)))
        return ((h >> np.uint64(32)) * np.uint64(cap)) >> np.uint64(32)


def barcode_home(key, shift):
    key = np.asarray(key, np.uint64)
    x = (key & np.uint64(0xFFFFFFFF)) ^ (key >> np.uint64(32))
    return ((x * np.uint64(0x9E3779B1)) & np.uint64(0xFFFFFFFF)) >> np.uint64(shift)


def barcode_table_shift(n):
    cap, log2 = 16, 4
    while cap < 2 * n + 2:
        cap, log2 = cap * 2, log2 + 1
    return 32 - log2, cap


# The caches' input hashes: xg_mix_bytes chained over the arrays (features, SNPs, regions), and the barcode chain.
LANE_SEED = (0x9E3779B97F4A7C15, 0xBF58476D1CE4E5B9, 0x94D049BB133111EB, 0xD6E8FEB86659FD93)
LANE_SHIFT = (29, 31, 27, 30)


def _lane_step(s, w, lane):
    x = ((s ^ w) * FNV_P) & M64
    return x ^ (x >> LANE_SHIFT[lane])


def mix_bytes(h, data):
    data = bytes(data)
    nb = len(data) // 32
    words = np.frombuffer(data, "<u8", count=4 * nb).tolist() if nb else []
    lanes = [h ^ s for s in LANE_SEED]
    for k in range(nb):
        for L in range(4):
            lanes[L] = _lane_step(lanes[L], words[4 * k + L], L)
    a, b, c, d = lanes
    h = ((a * 3 + (b ^ ((b << 7) & M64))) & M64) ^ ((c * 5 + (d ^ (d >> 11))) & M64)
    for byte in data[32 * nb:]:
        h = ((h ^ byte) * FNV_P) & M64
    h = ((h ^ len(data)) * FNV_P) & M64
    return h ^ (h >> 32)


def input_hash(arrays):
    h = FNV_OFF
    for a in arrays:
        h = mix_bytes(h, np.ascontiguousarray(a).tobytes())
    return h


def lane_collide(h, data, blk, lane, new_word):
    """`data` with 64-bit word `lane` of 32-byte block `blk` set to new_word and the same lane's word of the next block
    chosen so that mix_bytes(h, .) does not change."""
    data = bytes(data)
    words = np.frombuffer(data, "<u8", count=4 * (blk + 2)).tolist()
    s = h ^ LANE_SEED[lane]
    for k in range(blk):
        s = _lane_step(s, words[4 * k + lane], lane)
    old, new = _lane_step(s, words[4 * blk + lane], lane), _lane_step(s, new_word, lane)
    out = bytearray(data)
    struct.pack_into("<Q", out, 8 * (4 * blk + lane), new_word)
    struct.pack_into("<Q", out, 8 * (4 * blk + 4 + lane), words[4 * blk + 4 + lane] ^ old ^ new)
    return bytes(out)


def barcode_chain(keys, n=None):
    """The barcode table's hash (xg_build_barcode_table); n: the list's length, if keys is only its beginning."""
    h = FNV_OFF ^ (len(keys) if n is None else n)
    for k in np.asarray(keys, np.uint64).tolist():
        x = ((h ^ k) * FNV_P) & M64
        h = x ^ (x >> 29)
    return h


def barcode_collide(keys, j, new_key):
    """keys with keys[j] = new_key and keys[j + 1] chosen so that barcode_chain does not change."""
    keys = np.array(keys, np.uint64)
    h = barcode_chain(keys[:j], len(keys))                       # the chain's state after j keys
    step = lambda s, k: (lambda x: x ^ (x >> 29))(((s ^ k) * FNV_P) & M64)
    old, new = step(h, int(keys[j])), step(h, int(new_key))
    keys[j + 1] = np.uint64(int(keys[j + 1]) ^ old ^ new)
    keys[j] = np.uint64(new_key)
    return keys


def feature_collision():
    """Feature sets A and B (gid, beg, end) with equal cache hashes: B moves feature 10's end off its reads, and the
    same lane of the next 32-byte block (the ends of features 18 and 19) compensates."""
    n = 64
    gid = np.zeros(n, np.int32)
    beg = (np.arange(n) * 1000).astype(np.int32)
    end = beg + 600
    h = input_hash([np.int32(1), np.int32(n), gid, beg])
    blk, lane = 1, 1                                               # ends 10, 11 / 18, 19
    w = np.array([beg[10] + 20, end[11]], np.int32).view("<u8")[0]
    end_b = np.frombuffer(lane_collide(h, end.tobytes(), blk, lane, int(w)), np.int32).copy()
    return gid, beg, end, end_b


def snp_collision(snp_pos):
    """SNP position list B with the cache hash of A: SNP 2 moves to A's position of SNP 3, and the lane's next word
    (SNPs 10, 11) compensates."""
    n = len(snp_pos)
    gid = np.zeros(n, np.int32)
    h = input_hash([np.int32(1), np.int32(n), gid])
    pos = np.asarray(snp_pos, np.int32)
    w = np.array([pos[3], pos[3]], np.int32).view("<u8")[0]
    return np.frombuffer(lane_collide(h, pos.tobytes(), 0, 1, int(w)), np.int32).copy()


# ------------------------------------------------------------------------------------------- batches and calls
def feature_reads(feats, n_bad=0, seed=0):
    """feats: [(cells, umis)] per feature, in record order.  Feature f covers [10^6 f, 10^6 f + 9 * 10^5) and its
    reads lie inside it.  Plus n_bad reads per feature, at random places, that fail the mapq filter: candidates, never
    words."""
    rng = np.random.RandomState(seed)
    pos, cell, umi, mapq = [], [], [], []
    for f, (c, u) in enumerate(feats):
        c, u = np.asarray(c, np.int64), np.asarray(u, np.uint64)
        q = np.full(len(c), 60)
        if n_bad:
            at = np.sort(rng.randint(0, len(c) + 1, n_bad))
            c = np.insert(c, at, rng.randint(0, c.max() + 1, n_bad))
            u = np.insert(u, at, umi_keys(n_bad, salt=1 << 20))
            q = np.insert(q, at, 0)
        pos.append(10 ** 6 * f + 1000 + np.arange(len(c)) // 4)
        cell.append(c)
        umi.append(u)
        mapq.append(q)
    pos = np.concatenate(pos)
    return pos, np.concatenate(cell), np.concatenate(umi), np.concatenate(mapq).astype(np.uint32)


def with_tile_dups(cells, umis, n_dup):
    """The first n_dup pairs once more, at least a tile (1 024 records) after the first copy: each copy is a word."""
    assert len(cells) - n_dup >= 1024
    return np.concatenate([cells, cells[:n_dup]]), np.concatenate([umis, umis[:n_dup]])


def run(ctx, feats, n_cols, conf=None, n_bad=0, read_keys=None):
    """basefc on the batch of feature_reads(feats) == oracle.basefc; read_keys: the cell key of each cell index of the
    reads (default: the n_cols listed cells).  Returns (result, timing(), finalize stats)."""
    pos, cell, umi, mapq = feature_reads(feats, n_bad)
    ck = cell_keys(n_cols) if read_keys is None else read_keys[:n_cols]
    rk = ck if read_keys is None else read_keys
    reads = build(pos, rk[cell], umi, [(0, 0, 0, len(pos))], end=pos + 50, mapq=mapq)
    nf = len(feats)
    gid = np.zeros(nf, np.int32)
    beg = (np.arange(nf) * 10 ** 6).astype(np.int32)
    return call(ctx, reads, gid, beg, beg + 900000, ck, n_cols, conf)


def call(ctx, reads, gid, beg, end, ck, n_cols, conf=None):
    from oracle import oracle
    conf = conf or Conf()
    p = engine.make_params(conf, reads.max_aln_len, True)
    d = ctx.upload(reads)
    try:
        got = [np.asarray(x) for x in ctx.basefc(d, gid, beg, end, ck, n_cols, p)[:3]]
        t, st = ctx.timing(), ctx.basefc_finalize_stats()
    finally:
        d.close()
    exp = oracle.basefc(reads, gid, beg, end, ck, n_cols, oracle.params(conf), 8)
    for a, b in zip(got, exp):
        assert np.array_equal(a, b)
    assert len(got[2]) > 0
    return got, t, st


def spread(n, cells, rng, salt=0):
    """n distinct (cell, UMI) pairs over the given cells."""
    return np.asarray(cells, np.int64)[rng.randint(0, len(cells), n)], umi_keys(n, salt=salt)


# ------------------------------------------------------------------------------------------------ CPU: mirrors
def test_crafted_pair_words_collide_in_the_finalize_tables():
    for log2 in (12, 14):
        u = colliding_umis(7, log2, 120)
        assert len(set(u.tolist())) == 120
        assert np.all(fs_slot(u | np.uint64(7), log2) == (1 << log2) - 1)
        for small in (9, 10, log2):             # careful / light tables of 2^small slots: the last slot again
            assert np.all(fs_slot(u | np.uint64(7), small) == (1 << small) - 1)


def test_set_and_barcode_homes():
    u = umi_keys(1 << 20)
    s = set_home(u, 0, 508)
    assert s.max() == 507 and np.sum(s == 507) > 300
    shift, cap = barcode_table_shift(64)
    assert (shift, cap) == (24, 256)
    k = (np.arange(1, 1 << 18, dtype=np.uint64) << np.uint64(24)) | np.uint64(5)
    assert np.sum(barcode_home(k, shift) == cap - 1) > 100


def test_crafted_cache_inputs_collide():
    keys = cell_keys(50)
    kb = barcode_collide(keys, 48, 0x123456789ABCDEF)
    assert not np.array_equal(keys, kb) and barcode_chain(keys) == barcode_chain(kb)
    assert len(set(kb.tolist())) == 50
    gid, beg, end, end_b = feature_collision()
    assert np.sum(end != end_b) >= 2 and end_b[10] == beg[10] + 20
    assert input_hash([np.int32(1), np.int32(64), gid, beg, end]) == \
        input_hash([np.int32(1), np.int32(64), gid, beg, end_b])
    pos = (1000 + 7 * np.arange(40)).astype(np.int32)
    pos_b = snp_collision(pos)
    assert pos_b[2] == pos[3] and np.sum(pos != pos_b) >= 3
    g = np.zeros(40, np.int32)
    assert input_hash([np.int32(1), np.int32(40), g, pos]) == input_hash([np.int32(1), np.int32(40), g, pos_b])


def test_range_width_helper():
    assert wshift_of(2000, 32, "ordinary") == (5, 5)
    assert wshift_of(2000, 4097, "ordinary")[0] == 10
    assert wshift_of(700000, BIG_CTA_MAX_COLS + 1, "ordinary") == (8, 7)       # widened by FS_RANGES
    assert wshift_of(SEG_MAX, 40000, "big") == (6, 5)
    assert BIG_CTA_MAX_COLS == 141664


# ------------------------------------------------------------------------------------------ light / heavy
@gpu
@pytest.mark.parametrize("cta,words", [("ordinary", 1638), ("ordinary", 1639), ("big", 6553), ("big", 6554)])
def test_light_heavy_boundary(gpu_ctx, cta, words):
    rng = np.random.RandomState(words)
    c, u = spread(words - 300, range(3000), rng)
    c, u = with_tile_dups(c, u, 300)
    _, t, st = run(gpu_ctx, [(c, u)], 3000, n_bad=200)
    other = "big" if cta == "ordinary" else "ordinary"
    assert st[cta]["heavy"] == int(words > LIGHT[cta]) and st[other]["heavy"] == 0
    assert t[14] == 1


# ------------------------------------------------------------------------------------------ column ranges
@gpu
@pytest.mark.parametrize("n_cols", [32, 33, 4097])
def test_range_edges(gpu_ctx, n_cols):
    """A heavy feature in the ordinary CTA with words in the cells on both sides of every range edge."""
    rng = np.random.RandomState(n_cols)
    n = 2000
    w, _ = wshift_of(n, n_cols, "ordinary")
    edges = [c for k in range(1, ((n_cols - 1) >> w) + 1) for c in ((k << w) - 1, k << w)] + [0, n_cols - 1]
    c, u = spread(n - 300 - 10 * len(edges), range(n_cols), rng)
    c = np.concatenate([np.repeat(edges, 10), c])
    u = np.concatenate([umi_keys(10 * len(edges), salt=1 << 16), u])
    c, u = with_tile_dups(c, u, 300)
    (row, col, val), _, st = run(gpu_ctx, [(c, u)], n_cols)
    assert set(edges) <= set(col.tolist())
    assert st["ordinary"]["heavy"] == 1
    assert st["ordinary"]["careful"] == np.sum(np.bincount(c >> w) > CAP["ordinary"])
    assert (n_cols == 4097) == (st["ordinary"]["careful"] == 0)


# ------------------------------------------------------------------------------------------ careful path from skew
@gpu
@pytest.mark.parametrize("cta,deep", [("ordinary", 1638), ("ordinary", 1639), ("big", 6553), ("big", 6554)])
def test_careful_path_from_one_deep_cell(gpu_ctx, monkeypatch, cta, deep):
    """Cell 0 holds `deep` distinct UMIs alone in its column range; the other words are in later ranges."""
    rng = np.random.RandomState(deep)
    n_other = 3000                                             # candidates > 4 096 in both cases
    if cta == "ordinary":
        monkeypatch.setenv("XG_SEG_BIG", str(1 << 40))           # every feature in the ordinary CTA
    n_cols = 3000
    w, _ = wshift_of(deep + n_other, n_cols, cta)
    c, u = spread(n_other, range(1 << w, n_cols), rng, salt=1 << 20)
    c = np.concatenate([np.zeros(deep, np.int64), c])
    u = np.concatenate([umi_keys(deep), u])
    (row, col, val), _, st = run(gpu_ctx, [(c, u)], n_cols)
    assert val[col == 0].tolist() == [deep]
    assert st[cta]["heavy"] == 1 and st[cta]["careful"] == int(deep > CAP[cta])


@gpu
def test_bin_like_deep_cell(gpu_ctx):
    """A 1 Mb bin: one cell with 10^5 UMIs (some read twice) among 3 000 ordinary cells."""
    rng = np.random.RandomState(5)
    c, u = spread(90000, range(1, 3000), rng, salt=1 << 21)
    c = np.concatenate([np.zeros(100000, np.int64), c])
    u = np.concatenate([umi_keys(100000), u])
    c, u = with_tile_dups(c, u, 20000)
    (row, col, val), _, st = run(gpu_ctx, [(c, u)], 3000)
    assert val[col == 0].tolist() == [100000]
    assert st["big"]["heavy"] == 1 and st["big"]["careful"] >= 1


# ------------------------------------------------------------------------------------------ crafted collisions
@gpu
@pytest.mark.parametrize("cta", ["ordinary", "big"])
def test_crafted_collisions_overflow_and_double(gpu_ctx, cta):
    """Feature 0 (heavy): 120 words of cell 0 share the table's last slot as home, in a range of far fewer than CAP
    words: the fast pass overflows after 96 probes, the careful pass (a smaller table, the same last slot) overflows
    at one sub-partition and doubles.  Feature 1 (light): 200 words with the last slot as home, wrapping around."""
    rng = np.random.RandomState(3)
    log2 = TBL_LOG2[cta]
    hot = colliding_umis(0, log2, 120)
    n_cols, n_other = (20000, 7000) if cta == "big" else (3000, 1600)
    w, _ = wshift_of(120 + n_other, n_cols, cta)
    c, u = spread(n_other, range(1 << w, n_cols), rng, salt=1 << 20)
    heavy = (np.concatenate([np.zeros(120, np.int64), c]), np.concatenate([hot, u]))
    light = (np.zeros(200, np.int64), colliding_umis(0, 9, 200))    # light table: 512 slots
    (row, col, val), _, st = run(gpu_ctx, [heavy, light], n_cols)
    assert val[(row == 0) & (col == 0)].tolist() == [120] and val[row == 1].tolist() == [200]
    assert st[cta]["heavy"] == 1
    assert st[cta]["fast_overflow"] >= 1 and st[cta]["doubled"] >= 1


@gpu
def test_crafted_set_collisions(gpu_ctx, monkeypatch):
    """Sets only (XG_SEG_MODE=0): 300 (cell 0, UMI) elements whose home is the set's last slot wrap around."""
    monkeypatch.setenv("XG_SEG_MODE", "0")
    cand = 400
    cap = cand + cand // 4 + 8
    u = umi_keys(1 << 20)
    hot = u[set_home(u, 0, cap) == cap - 1][:300]
    rng = np.random.RandomState(4)
    c, v = spread(cand - 300, range(1, 50), rng, salt=1 << 21)
    (row, col, val), t, _ = run(gpu_ctx, [(np.concatenate([np.zeros(300, np.int64), c]), np.concatenate([hot, v]))],
                                50)
    assert val[col == 0].tolist() == [300]
    assert t[14] == 0 and t[15] == 1


@gpu
def test_barcode_cluster_wraps(gpu_ctx):
    """64 listed cells, 40 of them with the barcode table's last slot as home; reads of 20 unlisted cells with that
    home walk the cluster and are dropped."""
    shift, cap = barcode_table_shift(64)
    k = (np.arange(1, 1 << 18, dtype=np.uint64) << np.uint64(24)) | np.uint64(5)
    hot = k[barcode_home(k, shift) == cap - 1]
    listed = np.concatenate([hot[:40], cell_keys(24, salt=1 << 30)])
    keys = np.concatenate([listed, hot[40:60]])                 # column 64.. : unlisted
    rng = np.random.RandomState(6)
    c, u = spread(3000, range(84), rng)
    (row, col, val), _, _ = run(gpu_ctx, [(c, u)], 64, read_keys=keys)
    assert set(col.tolist()) == set(np.unique(c[c < 64]).tolist()) and col.max() < 64
    assert val.sum() == np.sum(c < 64)


# ------------------------------------------------------------------------------------------ cell-count regimes
@gpu
@pytest.mark.parametrize("n_cols", [BIG_CTA_MAX_COLS, BIG_CTA_MAX_COLS + 1],
                         ids=["%d-big-on" % BIG_CTA_MAX_COLS, "%d-big-off" % (BIG_CTA_MAX_COLS + 1)])
def test_big_cta_column_limit(gpu_ctx, n_cols):
    """A heavy feature of 700 000 words over every cell (ranges widened for FS_RANGES in the ordinary CTA) and a light
    one."""
    rng = np.random.RandomState(1)
    n = 700000
    c = np.tile(np.arange(n // 2, dtype=np.int64) % n_cols, 2)   # every pair twice, 350 000 records apart
    u = np.tile(umi_keys(n // 2), 2)
    lc, lu = spread(300, range(n_cols), rng, salt=1 << 22)
    (row, col, val), _, st = run(gpu_ctx, [(c, u), (lc, lu)], n_cols)
    on = n_cols <= BIG_CTA_MAX_COLS
    assert st["big"]["heavy"] == int(on) and st["ordinary"]["heavy"] == int(not on)
    w, w0 = wshift_of(n, n_cols, "big" if on else "ordinary")
    assert (w > w0) == (not on)
    assert col[row == 0].max() == n_cols - 1


@gpu
@pytest.mark.parametrize("n_cols", [1 << 19, (1 << 19) + 1], ids=["2^19", "2^19+1"])
def test_segment_mode_column_limit(gpu_ctx, n_cols):
    """40 features over the same 600 reads of one tile (the tile filter expresses 2^(24 - 19) = 32 of them; repeated
    (cell, UMI) pairs of the others reach the finalize) and a heavy feature."""
    rng = np.random.RandomState(2)
    n_small = 600
    sc = np.array([0, 1, n_cols - 1])[rng.randint(0, 3, n_small)]
    su = umi_keys(5)[rng.randint(0, 5, n_small)]
    hc, hu = spread(3000, range(n_cols), rng, salt=1 << 20)
    pos = np.concatenate([1000 + np.arange(n_small) // 8, 10 ** 6 + 1000 + np.arange(3000) // 4])
    ck = cell_keys(n_cols)
    cells = np.concatenate([sc, hc])
    reads = build(pos, ck[cells], np.concatenate([su, hu]), [(0, 0, 0, len(pos))], end=pos + 50)
    beg = np.concatenate([np.full(40, 900), [10 ** 6]]).astype(np.int32)
    end = np.concatenate([1200 + np.arange(40), [10 ** 6 + 900000]]).astype(np.int32)
    (row, col, val), t, st = call(gpu_ctx, reads, np.zeros(41, np.int32), beg, end, ck, n_cols)
    assert np.all(np.bincount(row, minlength=41) > 0)
    if n_cols <= 1 << 19:
        assert t[14] == 41 and t[15] == 0 and st["ordinary"]["heavy"] == 1
    else:
        assert t[14] == 0 and t[15] == 41 and sum(st["ordinary"].values()) == 0


@gpu
@pytest.mark.parametrize("n_cols", [HIST_COLS, HIST_COLS + 1])
def test_set_finalize_histogram_passes(gpu_ctx, monkeypatch, n_cols):
    """Sets only: one histogram pass at 40 960 cells, two at 40 961; a row with entries on both sides of the edge."""
    monkeypatch.setenv("XG_SEG_MODE", "0")
    rng = np.random.RandomState(n_cols)
    c, u = spread(5000, range(n_cols), rng)
    c[:40] = np.repeat([HIST_COLS - 1, min(HIST_COLS, n_cols - 1)], 20)
    (row, col, val), t, _ = run(gpu_ctx, [(c, u)], n_cols)
    assert {HIST_COLS - 1, n_cols - 1} <= set(col.tolist())
    assert t[14] == 0 and t[15] == 1


# ------------------------------------------------------------------------------------------ seg_max
@gpu
def test_segment_candidate_limit(gpu_ctx):
    """2^22 + 1 reads on one contig; feature A ends before the last one (2^22 candidates: a segment in a big CTA, its
    ranges widened for FS_RANGES and reduced carefully), feature B includes it (2^22 + 1: a set)."""
    n, n_cols = SEG_MAX + 1, 40000
    i = np.arange(n, dtype=np.int64)
    pos = 1000 + i // 32
    pos[-1] = pos[-2] + 100
    c = i % n_cols
    u = (((i // 80000) + 1).astype(np.uint64) << np.uint64(30)) | np.uint64(1 << 28)   # each pair twice, tiles apart
    ck = cell_keys(n_cols)
    reads = build(pos, ck[c], u, [(0, 0, 0, n)], end=pos + 50)
    beg = np.array([500, 500], np.int32)
    end = np.array([pos[-1], pos[-1] + 1], np.int32)
    (row, col, val), t, st = call(gpu_ctx, reads, np.zeros(2, np.int32), beg, end, ck, n_cols)
    assert t[14] == 1 and t[15] == 1
    w, w0 = wshift_of(SEG_MAX, n_cols, "big")
    assert w > w0
    assert st["big"]["heavy"] == 1 and st["big"]["careful"] >= 1
    assert val[row == 1].sum() == val[row == 0].sum() + 1


# ------------------------------------------------------------------------------------------ UMI keys
@gpu
@pytest.mark.parametrize("case", ["interned-2^39-1", "interned-2^39", "packed-13", "packed-14"])
def test_umi_key_limits(gpu_ctx, case):
    """Interned ids (bit 63 set) below 2^39 and packed UMIs with their low 24 bits free fit a pair word; others make
    the call redo itself with sets, and the batch remembers.  Ids 0 and 2^39 (one cell): a wrong shift merges them."""
    from oracle import oracle
    rng = np.random.RandomState(7)
    n, n_cols = 3000, 100
    top = np.uint64(1 << 63)
    if case.startswith("interned"):
        big = (1 << 39) - 1 if case.endswith("-1") else 1 << 39
        u = top | np.arange(n, dtype=np.uint64)
        u[:2] = [top | np.uint64(0), top | np.uint64(big)]
        u[2] = top | np.uint64((1 << 39) - 1)
    else:
        u = (np.arange(1, n + 1, dtype=np.uint64) << np.uint64(40)) | np.uint64(1 << 24)
        if case == "packed-14":
            u[5:] |= np.uint64(1 << 21)
    c = rng.randint(0, n_cols, n)
    c[:3] = 0
    fits = case in ("interned-2^39-1", "packed-13")
    pos = 1000 + np.arange(n) // 4
    ck = cell_keys(n_cols)
    reads = build(pos, ck[c], u, [(0, 0, 0, n)], end=pos + 50)
    gid, beg, end = np.zeros(1, np.int32), np.array([500], np.int32), np.array([900000], np.int32)
    conf = Conf()
    p = engine.make_params(conf, reads.max_aln_len, True)
    d = gpu_ctx.upload(reads)
    try:
        exp = oracle.basefc(reads, gid, beg, end, ck, n_cols, oracle.params(conf), 8)
        for _ in range(2):
            got = gpu_ctx.basefc(d, gid, beg, end, ck, n_cols, p)[:3]
            t = gpu_ctx.timing()
            assert all(np.array_equal(np.asarray(a), b) for a, b in zip(got, exp))
            assert (t[14], t[15]) == ((1, 0) if fits else (0, 1))
    finally:
        d.close()


# ------------------------------------------------------------------------------------------ input caches
@gpu
def test_barcode_cache_compares_the_keys(gpu_ctx):
    """Cell lists A and B differ in their last two keys and have the same hash: B gets a table of its own."""
    n = 50
    a = cell_keys(n)
    b = barcode_collide(a, n - 2, 0x0123456789ABCD05)
    assert barcode_chain(a) == barcode_chain(b)
    keys = np.concatenate([a, b[-2:]])                          # columns n, n + 1 of the reads: B's new keys
    rng = np.random.RandomState(8)
    c, u = spread(4000, range(n + 2), rng)
    c[:300] = n + np.arange(300) % 2
    pos, cell, umi, mapq = feature_reads([(c, u)])
    reads = build(pos, keys[cell], umi, [(0, 0, 0, len(pos))], end=pos + 50, mapq=mapq)
    gid, beg, end = np.zeros(1, np.int32), np.array([0], np.int32), np.array([900000], np.int32)
    ra = call(gpu_ctx, reads, gid, beg, end, a, n)[0]
    rb = call(gpu_ctx, reads, gid, beg, end, b, n)[0]
    assert not all(np.array_equal(x, y) for x, y in zip(ra, rb))


@gpu
def test_feature_cache_compares_the_features(gpu_ctx):
    """Feature sets A and B with the same hash (B: feature 10 ends before its reads, features 18 and 19 get other
    ends); A again reuses its index."""
    gid, beg, end, end_b = feature_collision()
    rng = np.random.RandomState(9)
    n = 200
    pos = np.sort(np.concatenate([beg[k] + 100 + rng.randint(0, 400, n) for k in range(len(beg))]))
    c = rng.randint(0, 20, len(pos))
    ck = cell_keys(20)
    reads = build(pos, ck[c], umi_keys(len(pos)), [(0, 0, 0, len(pos))], end=pos + 50)
    ra, t1, _ = call(gpu_ctx, reads, gid, beg, end, ck, 20)
    rb = call(gpu_ctx, reads, gid, beg, end_b, ck, 20)[0]
    assert 10 not in rb[0].tolist() and 10 in ra[0].tolist()
    # reuse: a large feature set, built once, then found again
    big = 200000
    g2 = np.zeros(big, np.int32)
    b2 = (np.arange(big) * 50).astype(np.int32)
    call(gpu_ctx, reads, g2, b2, b2 + 300, ck, 20)
    t_build = gpu_ctx.timing()[8]
    call(gpu_ctx, reads, g2, b2, b2 + 300, ck, 20)
    t_hit = gpu_ctx.timing()[8]
    assert t_hit * 3 < t_build, (t_hit, t_build)


@gpu
def test_snp_cache_compares_the_snps(gpu_ctx):
    """SNP lists A and B with the same hash (B: SNP 2 at SNP 3's position, SNPs 10 and 11 elsewhere): baf_pileup
    sorts B's table instead of reusing A's."""
    from oracle import oracle
    rng = np.random.RandomState(10)
    n_snp, n_cols, L = 40, 30, 60
    pos_a = (1000 + 7 * np.arange(n_snp)).astype(np.int32)
    pos_b = snp_collision(pos_a)
    n = 6000
    rpos = np.sort(rng.randint(900, 1300, n))
    seq = rng.choice([1, 2, 4, 8], size=(n, L)).astype(np.uint8)
    ck = cell_keys(n_cols)
    reads = build(rpos, ck[rng.randint(0, n_cols, n)], umi_keys(n), [(0, 0, 0, n)], end=rpos + L, seq=seq)
    conf = Conf(min_mapq=0, min_include=0)
    params = engine.make_params(conf, reads.max_aln_len, with_include=False)
    ref = rng.randint(0, 4, n_snp)
    alt = (ref + 1) % 4
    hap = np.full((n_snp, 8), 2, np.uint8)
    hap[np.arange(n_snp), ref] = 0
    hap[np.arange(n_snp), alt] = 1
    reg_ptr, reg_snp = np.arange(n_snp + 1, dtype=np.int64), np.arange(n_snp, dtype=np.int32)
    d = gpu_ctx.upload(reads)
    out = []
    try:
        for sp in (pos_a, pos_b):
            exp = oracle.baf(reads, np.zeros(n_snp, np.int32), sp, "".join("ACGT"[x] for x in ref),
                             "".join("ACGT"[x] for x in alt), np.zeros(n_snp), np.ones(n_snp), reg_ptr, reg_snp, ck,
                             n_cols, oracle.params(conf), 1, 0.0, True, 4)
            got = gpu_ctx.baf_fc(d, np.zeros(n_snp, np.int32), sp, ck, n_cols, params, ref, alt, 1, 0.0, reg_ptr,
                                 reg_snp, hap, True)
            for g, e in zip(got, exp):
                for k in range(3):
                    assert np.array_equal(np.asarray(g[k]), e[k])
            out.append(exp)
    finally:
        d.close()
    assert not all(np.array_equal(x, y) for x, y in zip(out[0][1], out[1][1]))
