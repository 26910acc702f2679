"""Region-wise local phasing before the counting (xcltk/baf/fc/phasing.py:13-78).

reg_local_phasing: one region on the host (numpy), from the cellsnp-lite counts of `afc_wrapper(cellsnp_dir=...)`.
local_phasing_device: every long region at once on the device (xg_local_phase), from SNP x cell counts of the call's
own reads (`afc_wrapper(phase_from_reads=True)`), with the same effect on the SNP objects and region lists."""

from logging import warning as warn

import numpy as np

from ..localphase import snp_local_phasing


def reg_local_phasing(reg, AD, DP):
    """AD, DP: cell x SNP count arrays of the cellsnp-lite SNPs inside `reg`, columns in the order of
    reg.snp_list.  SNPs nobody expresses leave the region's list; the SNPs the EM flips swap their haplotype
    indices (the SNP objects are shared by every region that holds them).  Returns (reg, flip) with flip = None
    when the phasing could not be done."""
    cell_idx = DP.sum(axis=1) > 0
    snp_idx = DP.sum(axis=0) > 0
    AD, DP = AD[np.ix_(cell_idx, snp_idx)], DP[np.ix_(cell_idx, snp_idx)]
    reg.snp_list = [s for keep, s in zip(snp_idx, reg.snp_list) if keep]
    BD = DP - AD
    flip = np.array([snp.ref_idx == 1 for snp in reg.snp_list])
    AD_ref_phased = AD * (1 - flip.T) + BD * flip.T          # ALT counts -> counts of haplotype 1
    flip = snp_local_phasing(AD_ref_phased, DP, np.array([s.pos for s in reg.snp_list]))
    if flip is None:
        warn("local phasing for region '%s' failed!" % reg.name)
        return reg, None
    flip = (1 - flip if np.mean(flip) > 0.5 else flip + 0).astype(int)     # as few changes as possible
    assert len(reg.snp_list) == len(flip)
    for snp, f in zip(reg.snp_list, flip):
        if f == 1:
            snp.ref_idx, snp.alt_idx = 1 - snp.ref_idx, 1 - snp.alt_idx
            snp.gt = {snp.ref: snp.ref_idx, snp.alt: snp.alt_idx}
    return reg, flip


def is_long_region(conf, reg):
    """The regions afc_core phases locally (baf/fc/main.py:107-149): >= rlp_min_len bp, >= rlp_min_n_snps SNPs,
    SNP span >= rlp_min_gap."""
    if reg.end - reg.start < conf.rlp_min_len:
        return False
    if reg.snp_list is None or len(reg.snp_list) < max(1, conf.rlp_min_n_snps):
        return False
    return reg.snp_list[-1].pos - reg.snp_list[0].pos + 1 >= conf.rlp_min_gap


def phase_waves(snp_lists):
    """Wave (0-based) of every region, in list order: 1 + the largest wave of the earlier regions that share a SNP
    with it (0 without such a region).  A region's starting orientation is what the earlier regions left on its SNPs,
    so it runs after all of them; regions of one wave share no SNP and can run together."""
    last = {}
    waves = np.zeros(len(snp_lists), dtype=np.int64)
    for r, ids in enumerate(snp_lists):
        w = 1 + max((last.get(i, -1) for i in ids), default=-1)
        waves[r] = w
        for i in ids:
            last[i] = w
    return waves


def phase_layout(snp_lists, csr, n_cells, row_lists=None):
    """xg_phase_regions arrays (without wave_ptr) of the regions `snp_lists` (SNP ids, in the order they run).
    csr = (row_ptr, col, ad, dp): SNP x cell counts over the cells that take part, DP > 0 only, columns ascending.
    Slot k of a region counts with CSR row row_lists[r][k] (default: snp_lists[r][k]).  A region's entries are those
    rows, SNP-major as given and cell-major by (cell, slot); its local cells are their cells in ascending order."""
    row_ptr, col, ad, dp = (np.asarray(x) for x in csr)
    rows = np.concatenate([np.asarray(x, dtype=np.int64) for x in (row_lists if row_lists is not None else snp_lists)]
                          + [np.zeros(0, np.int64)])
    n_reg = len(snp_lists)
    m = np.array([len(x) for x in snp_lists], dtype=np.int64)
    reg_snp_ptr = np.zeros(n_reg + 1, dtype=np.int64)
    np.cumsum(m, out=reg_snp_ptr[1:])
    reg_snp = np.concatenate([np.asarray(x, dtype=np.int64) for x in snp_lists] + [np.zeros(0, np.int64)])
    slot_j = np.arange(len(reg_snp), dtype=np.int64) - np.repeat(reg_snp_ptr[:-1], m)
    ln = row_ptr[rows + 1] - row_ptr[rows]
    slot_ent_ptr = np.zeros(len(reg_snp) + 1, dtype=np.int64)
    np.cumsum(ln, out=slot_ent_ptr[1:])
    n_ent = int(slot_ent_ptr[-1])
    src = np.repeat(row_ptr[rows] - slot_ent_ptr[:-1], ln) + np.arange(n_ent, dtype=np.int64)
    cell = col[src].astype(np.int64)
    ent_reg = np.repeat(np.repeat(np.arange(n_reg, dtype=np.int64), m), ln)
    order = np.argsort(ent_reg * max(int(n_cells), 1) + cell, kind="stable")
    key = (ent_reg * max(int(n_cells), 1) + cell)[order]
    first = np.ones(n_ent, dtype=bool)
    first[1:] = key[1:] != key[:-1]
    reg_cell_ptr = np.zeros(n_reg + 1, dtype=np.int64)
    np.cumsum(np.bincount(ent_reg[order][first], minlength=n_reg), out=reg_cell_ptr[1:])
    seq = np.cumsum(first) - 1                                   # cell slot of every cell-major entry
    sm_cell = np.empty(n_ent, dtype=np.int32)
    sm_cell[order] = seq - reg_cell_ptr[ent_reg[order]]
    ent_ad, ent_dp = ad[src], dp[src]
    return {"reg_snp_ptr": reg_snp_ptr, "reg_snp": reg_snp, "slot_ent_ptr": slot_ent_ptr, "sm_cell": sm_cell,
            "sm_ad": ent_ad, "sm_dp": ent_dp, "reg_cell_ptr": reg_cell_ptr,
            "cell_ent_ptr": np.append(np.flatnonzero(first), n_ent).astype(np.int64),
            "cm_snp": np.repeat(slot_j, ln)[order], "cm_ad": ent_ad[order], "cm_dp": ent_dp[order]}


def csr_from_coo(n_snps, ad, dp, cell_mask):
    """(row_ptr, col, ad, dp) over SNP ids x cells from the (row, col, val) of AD and DP (AD's support lies in DP's),
    the cells with cell_mask False left out."""
    r, c, v = (np.asarray(x, dtype=np.int64) for x in dp[:3])
    live = np.asarray(cell_mask, dtype=bool)[c] & (v > 0)
    r, c, v = r[live], c[live], v[live]
    o = np.lexsort((c, r))
    r, c, v = r[o], c[o], v[o]
    n_cells = len(cell_mask)
    a = np.zeros(len(r), dtype=np.int64)
    ar, ac, av = (np.asarray(x, dtype=np.int64) for x in ad[:3])
    if len(ar):
        k = r * n_cells + c
        ak = ar * n_cells + ac
        at = np.searchsorted(k, ak)
        hit = (at < len(k)) & (k[np.minimum(at, max(len(k) - 1, 0))] == ak)
        a[at[hit]] = av[hit]
    row_ptr = np.zeros(n_snps + 1, dtype=np.int64)
    np.cumsum(np.bincount(r, minlength=n_snps), out=row_ptr[1:])
    return row_ptr, c.astype(np.int32), a.astype(np.int32), v.astype(np.int32)


def _dense(csr, ids, n_cells):
    """AD, DP (cells x ids) of the CSR rows `ids`: the matrices afc_core's cellsnp path hands reg_local_phasing."""
    row_ptr, col, ad, dp = csr
    AD = np.zeros((n_cells, len(ids)), dtype=np.int64)
    DP = np.zeros((n_cells, len(ids)), dtype=np.int64)
    for j, g in enumerate(ids):
        a, b = row_ptr[g], row_ptr[g + 1]
        AD[col[a:b], j] = ad[a:b]
        DP[col[a:b], j] = dp[a:b]
    return AD, DP


def local_phasing_device(ctx, regs, snps, csr, n_cells):
    """reg_local_phasing of every region of `regs` (list order), on the device in waves (xg_local_phase).
    snps: all SNP objects (SNP.index = position in the SNP file); csr: csr_from_coo over them, n_cells its columns.
    As the cellsnp path pairs `data.AD[:, cols]` (the region's SNPs in file order, the cellSNP row order) with
    reg.snp_list (sorted by position), the k-th SNP of snp_list -- its position, orientation, pruning and flip --
    counts with the k-th of the region's SNPs in file order; with a SNP file sorted by position that is itself.
    Applies what reg_local_phasing applies: the pruned snp_list, the swapped ref_idx / alt_idx / gt of the flipped
    SNPs.
    A region the device reports as a tie (status 2: a flip or convergence test within rounding of its threshold) is
    decided by reg_local_phasing itself, on the same matrices, and the later waves run again from there.
    Returns (flips, stats): per region the flip array over its pruned list, or None when the phasing failed; stats
    = the device timing of the first call (xg_last_timing), with [9] = device calls and [10] = tie regions."""
    lists = [[s.index for s in reg.snp_list] for reg in regs]
    rows = [sorted(x) for x in lists]
    waves = phase_waves(lists)
    order = np.argsort(waves, kind="stable")
    pos = np.array([s.pos for s in snps], dtype=np.int64)
    if len(pos) and (pos.min() < 0 or pos.max() >= 2 ** 31):
        raise ValueError("SNP positions out of the int32 range")
    flips = [None] * len(regs)
    stats, n_calls, n_ties = None, 0, 0
    while len(order):
        w = waves[order]
        layout = phase_layout([lists[i] for i in order], csr, n_cells, [rows[i] for i in order])
        layout["wave_ptr"] = np.searchsorted(w, np.arange(w[0], w[-1] + 2)).astype(np.int32)
        ref_idx = np.array([s.ref_idx == 1 for s in snps], dtype=np.uint8)
        keep, flip, status = ctx.local_phase(pos, ref_idx, layout)
        n_calls += 1
        if stats is None:
            stats = ctx.timing()
        tie = np.flatnonzero(status == 2)
        stop = w[tie[0]] if len(tie) else w[-1] + 1           # accept every wave before the first tie's
        ptr = layout["reg_snp_ptr"]
        for k, r in enumerate(order):
            if w[k] > stop:
                break
            reg = regs[r]
            if status[k] == 2:
                AD, DP = _dense(csr, rows[r], n_cells)
                _reg, f = reg_local_phasing(reg, AD, DP)
                flips[r] = None if f is None else np.asarray(f)
                n_ties += 1
                continue
            kp = keep[ptr[k]:ptr[k + 1]].astype(bool)
            reg.snp_list = [s for s, x in zip(reg.snp_list, kp) if x]
            if not status[k]:
                warn("local phasing for region '%s' failed!" % reg.name)
                continue
            f = flip[ptr[k]:ptr[k + 1]][kp].astype(int)
            for snp, x in zip(reg.snp_list, f):
                if x == 1:
                    snp.ref_idx, snp.alt_idx = 1 - snp.ref_idx, 1 - snp.alt_idx
                    snp.gt = {snp.ref: snp.ref_idx, snp.alt: snp.alt_idx}
            flips[r] = f
        order = order[w > stop]
    stats = list(stats) if stats is not None else [0.0] * 16
    stats[9], stats[10] = n_calls, n_ties
    return flips, stats
