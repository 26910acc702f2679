"""Record batches (lib.ArrayReads) built from numpy arrays, for tests that need to place reads, CIGARs,
bases, cells and UMIs exactly: tens of thousands to millions of reads without a per-read Python loop
for the common case (one M block per read, or one CIGAR shape for all reads)."""

import numpy as np

from xcltk_b200 import lib

M, I, D, N, S, H, P, EQ, X = 0, 1, 2, 3, 4, 5, 6, 7, 8
NT16 = "=ACMGRSVTWYHKDBN"
CODE = {b: k for k, b in enumerate(NT16)}          # base letter -> 4-bit code


def cell_keys(n, salt=0):
    """n distinct cell keys (bits 60..62 clear, so they never equal a synthetic barcode)."""
    return ((np.arange(n, dtype=np.uint64) + np.uint64(1 + salt)) << np.uint64(24)) | np.uint64(0x5)


def umi_keys(n, salt=0):
    """n distinct UMI keys with the low 24 bits clear (the form a packed 8-symbol UMI has)."""
    return ((np.arange(n, dtype=np.uint64) + np.uint64(1 + salt)) << np.uint64(30)) | np.uint64(1 << 28)


def ref_len(ops):
    return sum(l for op, l in ops if op in (M, D, N, EQ, X))


def query_len(ops):
    return sum(l for op, l in ops if op in (M, I, S, EQ, X))


def aligned_len(ops):
    return sum(l for op, l in ops if op in (M, EQ, X))


def _pack_seq(codes_list):
    """[array of 4-bit codes per read, or None for a record without SEQ] -> (seq_off, words)."""
    n = len(codes_list)
    seq_off = np.full(n, 0xFFFFFFFF, dtype=np.uint32)
    parts, at = [], 0
    for i, c in enumerate(codes_list):
        if c is None:
            continue
        c = np.asarray(c, dtype=np.uint8)
        if len(c) % 2:
            c = np.append(c, np.uint8(0))
        b = (c[0::2] << 4) | c[1::2]
        b = np.pad(b, (0, (-len(b)) % 4))
        seq_off[i] = at
        parts.append(b.view(np.uint32))
        at += len(b) // 4
    words = np.concatenate(parts) if parts else np.zeros(1, np.uint32)
    return seq_off, words


def _pack_seq_uniform(codes):
    """codes: (n, L) uint8, the same query length for every read."""
    n, L = codes.shape
    c = np.pad(codes.astype(np.uint8), ((0, 0), (0, L % 2)))
    b = (c[:, 0::2] << 4) | c[:, 1::2]
    b = np.pad(b, ((0, 0), (0, (-b.shape[1]) % 4)))
    w = np.ascontiguousarray(b).view(np.uint32)
    return (np.arange(n, dtype=np.uint32) * np.uint32(w.shape[1])), w.reshape(-1)


def build(pos, cell, umi, runs, end=None, ops=None, flag=0, mapq=60, seq=None):
    """One batch.  pos: 0-based starts, sorted inside every run; runs: [(bam_idx, gid, rec_beg, rec_end)].
    ops: None (every read one M block over [pos, end)), a list with one [(op, len)] per read (None = simple),
    or one [(op, len)] shared by every read.  A read with a CIGAR ends at pos + its reference length; end is
    needed for the simple reads only.
    seq: None (no sequences), an (n, L) array of 4-bit codes, or a list of code arrays / None per read.
    flag / mapq: scalars or arrays."""
    pos = np.asarray(pos, dtype=np.int64)
    n = len(pos)
    shared = ops is not None and len(ops) > 0 and isinstance(ops[0], tuple)
    if ops is None or shared:
        if ops is None:
            ncw = np.zeros(n, dtype=np.uint32)
            cig_off = np.zeros(n + 1, dtype=np.uint32)
            cigar = np.zeros(1, dtype=np.uint32)
            rl = None
            aln = None
        else:
            wds = np.array([(l << 4) | op for op, l in ops], dtype=np.uint32)
            k = len(wds)
            head = 1 if k >= 255 else 0
            per = np.concatenate([[k] if head else [], wds]).astype(np.uint32)
            cigar = np.tile(per, n)
            cig_off = (np.arange(n + 1, dtype=np.int64) * len(per) + head).astype(np.uint32)
            cig_off[-1] = len(cigar)
            ncw = np.full(n, 255 if head else k, dtype=np.uint32)
            rl, aln = ref_len(ops), aligned_len(ops)
        if end is None:
            end = pos + max(rl, 1)
        max_aln = int(np.max(np.asarray(end) - pos)) if aln is None else aln
    else:
        assert len(ops) == n
        words, offs, ncws, ends, alns = [], [], [], [], []
        for i, o in enumerate(ops):
            if o is None:
                offs.append(len(words))
                ncws.append(0)
                ends.append(int(end[i]))
                alns.append(int(end[i]) - int(pos[i]))
                continue
            k = len(o)
            if k >= 255:
                words.append(k)
            offs.append(len(words))
            words.extend((l << 4) | op for op, l in o)
            ncws.append(255 if k >= 255 else k)
            ends.append(int(pos[i]) + max(ref_len(o), 1))
            alns.append(aligned_len(o))
        cig_off = np.array(offs + [len(words)], dtype=np.uint32)
        cigar = np.array(words if words else [0], dtype=np.uint32)
        ncw = np.array(ncws, dtype=np.uint32)
        end = np.array(ends)
        max_aln = max(alns) if alns else 1
    end = np.asarray(end, dtype=np.int64)
    flag = np.broadcast_to(np.asarray(flag, dtype=np.uint32), (n,))
    mapq = np.broadcast_to(np.asarray(mapq, dtype=np.uint32), (n,))
    fmq = flag | (mapq << np.uint32(16)) | (ncw << np.uint32(24))
    keys = np.stack([np.broadcast_to(np.asarray(cell, dtype=np.uint64), (n,)),
                     np.broadcast_to(np.asarray(umi, dtype=np.uint64), (n,))], axis=1)
    pos_end = np.stack([pos, end], axis=1).astype(np.int32)
    seq_off = words = None
    if seq is not None:
        seq_off, words = _pack_seq_uniform(seq) if isinstance(seq, np.ndarray) else _pack_seq(seq)
    max_span = int((end - pos).max()) if n else 1
    return lib.ArrayReads(pos_end, fmq, cig_off, keys, cigar, runs, seq_off, words,
                          max_aln_len=max(1, max_aln), max_span=max(1, max_span))


# ---- a hand-built panel of reads with every CIGAR operator (one read per cell, distinct UMIs) ------------------
# label: (pos, CIGAR, query sequence); query sequence letters are 4-bit codes of NT16
CIGAR_PANEL = [
    ("R0", 100, [(S, 5), (M, 10), (I, 3), (M, 10)], "CCCCC" "AAAAAAAAAT" "CCC" "GAAAAAAAAA"),
    ("R1", 100, [(H, 4), (S, 3), (EQ, 6), (X, 2), (D, 4), (M, 8), (H, 2)], "TTT" "AAAAAC" "GT" "CAAAAAAA"),
    ("R2", 100, [(M, 10), (P, 2), (I, 3), (M, 0), (M, 10)], "AAAAAAAAAG" "TTT" "CAAAAAAAAA"),
    ("R3", 102, [(M, 0), (EQ, 5), (N, 100), (X, 5), (S, 5)], "ACGTA" "CCCCG" "TTTTT"),
    ("R5", 104, None, "ACN=RGTACG"),
    ("R4", 105, [(M, 3), (I, 2), (X, 4), (D, 1), (EQ, 5)], "ACG" "TT" "CAGA" "GTCAT"),
]


def cigar_panel(rows=CIGAR_PANEL):
    """(reads, cell keys): the rows (CIGAR_PANEL) in record order, read k in column k, one run on contig 0."""
    pos = [p for _, p, _, _ in rows]
    ops = [o for _, _, o, _ in rows]
    end = [p + (ref_len(o) if o is not None else len(s)) for _, p, o, s in rows]
    seq = [np.array([CODE[b] for b in s], dtype=np.uint8) for _, _, _, s in rows]
    n = len(rows)
    ck = cell_keys(n)
    return build(pos, ck, umi_keys(n), [(0, 0, 0, n)], end=end, ops=ops, seq=seq), ck
