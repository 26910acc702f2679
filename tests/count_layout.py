"""What the host (build_feat_index) and k_tile_desc decide for every tile of a basefc call, modelled in Python, so
that a test of k_basefc_count can check that its input lands on the switch it targets: the interval index of the
valid features, each tile's window in it (bx, by, st_n, c_lo / c_hi, jmin), the three staged flags and the bits of a
column index.  Constants and names follow basefc.cu."""

import numpy as np

from xcltk_b200 import lib

SB_MAX, STAB_CAP, CIG_CAP, INCL_CAP, WPAIR_CAP, FILT_BITS = 128, 128, 1024, 256, 96, 11


class Index(object):
    """build_feat_index: features sorted by (gid, beg, end, row) after dropping the ones never fetched; per contig
    the sorted distinct boundaries; per segment [bnd[k], bnd[k+1]) its stabbing list (features with beg <= bnd[k]
    and end >= bnd[k + 1], in sorted order); per boundary the first sorted feature with beg >= bnd[k] (fb)."""

    def __init__(self, gid, beg, end, n_gid):
        gid, beg, end = (np.asarray(a, dtype=np.int64) for a in (gid, beg, end))
        ok = [i for i in range(len(gid)) if 0 <= gid[i] < n_gid and beg[i] >= 0 and end[i] > beg[i]]
        order = sorted(ok, key=lambda i: (gid[i], beg[i], end[i], i))
        self.sf_row = np.array(order, dtype=np.int64)
        self.sf_beg = beg[self.sf_row] if order else np.zeros(0, np.int64)
        self.sf_end = end[self.sf_row] if order else np.zeros(0, np.int64)
        sf_gid = gid[self.sf_row] if order else np.zeros(0, np.int64)
        self.sf_goff = np.searchsorted(sf_gid, np.arange(n_gid + 1))
        self.bnd, self.bnd_goff, self.stab_off, self.stab = [], [0], [], []
        for g in range(n_gid):
            j0, j1 = self.sf_goff[g], self.sf_goff[g + 1]
            b = np.unique(np.concatenate([self.sf_beg[j0:j1], self.sf_end[j0:j1]]))
            lists = [[] for _ in b]
            for j, lo, hi in zip(range(j0, j1), np.searchsorted(b, self.sf_beg[j0:j1]),
                                 np.searchsorted(b, self.sf_end[j0:j1])):
                for k in range(lo, hi):
                    lists[k].append(j)
            for lst in lists:
                self.stab_off.append(len(self.stab))
                self.stab += lst
            self.bnd += b.tolist()
            self.bnd_goff.append(len(self.bnd))
        self.stab_off.append(len(self.stab))
        self.bnd = np.array(self.bnd, dtype=np.int64)
        self.stab_off = np.array(self.stab_off, dtype=np.int64)
        self.stab = np.array(self.stab, dtype=np.int64)
        self.fb = np.zeros(len(self.bnd) + 1, dtype=np.int64)
        for g in range(n_gid):
            k0, k1, j0, j1 = self.bnd_goff[g], self.bnd_goff[g + 1], self.sf_goff[g], self.sf_goff[g + 1]
            self.fb[k0:k1] = j0 + np.searchsorted(self.sf_beg[j0:j1], self.bnd[k0:k1], side="left")
        self.fb[len(self.bnd)] = len(self.sf_row)

    def stabbing(self, k):
        """sorted features of the stabbing list of segment k (global boundary index)"""
        return self.stab[self.stab_off[k]:self.stab_off[k + 1]]


class Tile(object):
    __slots__ = ("rec_beg", "n_rec", "run", "gid", "col", "first_pos", "max_end", "bx", "by", "st_lo", "st_n",
                 "c_lo", "c_hi", "jmin", "b0", "b1")

    @property
    def live(self):
        return self.bx >= 0

    @property
    def staged(self):
        return self.by - (self.bx & ~3) <= SB_MAX

    @property
    def stab_staged(self):
        return self.staged and self.st_n <= STAB_CAP

    @property
    def c_al(self):
        return self.c_lo & ~3

    @property
    def cig_staged(self):
        return self.c_hi - self.c_al <= CIG_CAP


def tiles(reads):
    """ArrayReads' tiles: every run cut into chunks of XG_TILE records -> [(rec_beg, n_rec, run index)]"""
    out = []
    for k, (_, _, rb, re_) in enumerate(reads.runs):
        for s in range(rb, re_, lib.XG_TILE):
            out.append((s, min(s + lib.XG_TILE, re_) - s, k))
    return out


def tile_descs(reads, ix):
    """k_tile_desc for every tile of the batch (cig_off of the batch: the device call's CIGAR ranges, which the
    streamed call's k_tile_cig computes alike)."""
    cig_off = reads._arrays["cig_off"]
    pe = reads.pos_end
    n_gid = len(ix.bnd_goff) - 1
    out = []
    for rec_beg, n_rec, run in tiles(reads):
        bam, gid = reads.runs[run][0], reads.runs[run][1]
        d = Tile()
        d.rec_beg, d.n_rec, d.run, d.gid, d.col = rec_beg, n_rec, run, gid, bam
        d.first_pos = int(pe[rec_beg, 0])
        d.max_end = int(pe[rec_beg:rec_beg + n_rec, 1].max())
        c_first = int(cig_off[rec_beg])
        d.c_lo = c_first - 1 if c_first else 0
        d.c_hi = int(cig_off[rec_beg + n_rec])
        d.bx = d.by = -1
        d.st_lo = d.st_n = d.jmin = d.b0 = d.b1 = 0
        if 0 <= gid < n_gid and ix.sf_goff[gid] != ix.sf_goff[gid + 1]:
            b0, b1 = ix.bnd_goff[gid], ix.bnd_goff[gid + 1]
            bnd = ix.bnd
            lo = b0 + int(np.searchsorted(bnd[b0:b1], d.first_pos, side="right"))
            x = max(b0, lo - 1)
            y = max(x, lo + int(np.searchsorted(bnd[lo:b1], d.max_end, side="left")))
            y_seg = min(y + 1, b1)
            if ix.stab_off[y_seg] > ix.stab_off[x] or ix.fb[y] > ix.fb[min(x + 1, y)]:
                d.bx, d.by, d.b0, d.b1 = x, y, b0, b1
                d.st_lo = int(ix.stab_off[x])
                d.st_n = int(ix.stab_off[y]) - d.st_lo
                d.jmin = int(ix.stab[ix.stab_off[x]]) if ix.stab_off[x + 1] > ix.stab_off[x] else \
                    int(ix.fb[min(x + 1, b1)])
        out.append(d)
    return out


def first_bnd_above(ix, d, pos):
    """count_record's `ub`: the first boundary of the tile's contig > pos (global index)"""
    return d.b0 + int(np.searchsorted(ix.bnd[d.b0:d.b1], pos, side="right"))


def col_bits(n_cols):
    b = 1
    while (1 << b) < n_cols:
        b += 1
    return b


def filter_bound(n_cols):
    """local feature indices j - jmin below this go through the tile's duplicate filter"""
    return 1 << (24 - col_bits(n_cols))


def filter_slot(fk):
    """the filter slot of a 64-bit key (emit_pair)"""
    fk = np.asarray(fk, dtype=np.uint64)
    lo = (fk & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    hi = (fk >> np.uint64(32)).astype(np.uint32)
    with np.errstate(over="ignore"):
        h = ((lo * np.uint32(0x85EBCA6B)) ^ hi) * np.uint32(0x9E3779B1)
    return h >> np.uint32(32 - FILT_BITS)


def umi_compact(umi):
    """the UMI key with its low 24 bits free, as seg_mode stores it (None: it does not fit)"""
    umi = int(umi)
    if umi >> 63:
        i = umi & ((1 << 63) - 1)
        return None if i >> 39 else (1 << 63) | (i << 24)
    return None if umi & 0xFFFFFF else umi
