// baf.cu -- feature-level allele counting at phased heterozygous SNPs (AD / DP / OTH matrices).
//
// Reference being replaced (xcltk v0.5.2):
//   plp_snp                  xcltk/baf/fc/core.py:198-247   pileup of one SNP over all BAMs
//   SCount.push_read         xcltk/baf/fc/mcount.py:109-127 first read per (SNP, cell, UMI) wins
//   UCount.push_read         xcltk/baf/fc/mcount.py:39-60   + get_query_bases utils/sam.py:4-40
//   SCount.stat/MCount.stat  xcltk/baf/fc/mcount.py:140-150,250-256  A/C/G/T/N totals per SNP
//   fc_fet1                  xcltk/baf/fc/core.py:143-194   region-level UMI set algebra
//
// Phase 1 (xg_baf_pileup): stream the reads once; a tile whose window holds no SNP is skipped
// without touching its records; a read overlapping SNPs emits (SNP, cell, UMI, ordinal, base)
// pairs.  First-read-wins = atomicMin of the record ordinal per (SNP, cell, UMI) key in a
// 128-bit-CAS hash table -- decided BEFORE looking at the base, so a read that skips the SNP
// (N / D) still claims the UMI (SURVEY.md A.2 B5).  Winners with a base add to the SNP totals.
// The caller applies the min_count / min_maf filter in Python (float exactness, B8).
// Phase 2 (xg_baf_count): winners of kept SNPs OR a 3-bit haplotype mask into
// (region, cell, UMI); the masks reduce to ref / alt / shared / other UMI counts per
// (region, cell) and then to AD / DP / OTH (B9, B10).
#include <algorithm>
#include <chrono>
#include <cstring>

#include "compact.cuh"

struct xg_baf_state {
    int64_t n_pairs = 0;
    int32_t n_snps = 0, n_cols = 0;
    uint32_t *pr_snp = nullptr;      // SNP index (caller's order)
    uint32_t *pr_colal = nullptr;    // col | base code << 24 | winner << 31
    uint64_t *pr_umi = nullptr;
};

namespace {

enum { CODE_NONE = 6, CODE_OTHER = 5 };

struct BafScanDev {
    const int2 *pos_end;
    const uint32_t *fmq, *cig_off, *cigar, *seq_off, *seq;
    const ulonglong2 *keys;
    const xg_run *runs;
    const xg_tile *tiles;
    int32_t n_gid;
    const int32_t *snp_goff;    // per gid range in the (gid, pos)-sorted SNP arrays
    const int32_t *snp_pos;
    const int32_t *snp_idx;     // caller's SNP index
    BarcodeTable bc;
    FilterParams fp;
    // pair output
    uint32_t *pr_snp, *pr_colal;
    uint64_t *pr_umi, *pr_ord;
    unsigned long long *n_pairs;
    unsigned long long cap_pairs;
};

// base code at reference position sp: 0..3 ACGT, 4 N, 5 other (=, IUPAC), 6 not covered (None)
__device__ __forceinline__ uint32_t base_at(const BafScanDev &P, int64_t i, int32_t pos, int32_t end,
                                            uint32_t n_ops, const uint32_t *cig, int32_t sp) {
    int32_t q = -1;
    if (n_ops == 0) {
        q = sp - pos;          // single M block covering [pos, end)
    } else {
        int32_t p = pos, qi = 0;
        for (uint32_t k = 0; k < n_ops; k++) {
            uint32_t w = __ldg(&cig[k]), op = w & 15u;
            int32_t l = (int32_t)(w >> 4);
            if (cig_aligned(op)) {
                if (sp >= p && sp < p + l) {
                    q = qi + (sp - p);
                    break;
                }
                p += l;
                qi += l;
            } else if (cig_skips_ref(op)) {
                p += l;
            } else if (op == 1 || op == 4) {
                qi += l;
            }
        }
    }
    if (q < 0) return CODE_NONE;
    uint32_t so = P.seq_off[i];
    if (so == 0xFFFFFFFFu) return CODE_NONE;   // record without sequence
    uint32_t byte = (uint32_t)q >> 1;
    uint32_t w = __ldg(&P.seq[so + (byte >> 2)]);
    uint32_t nib = (w >> (8 * (byte & 3u) + ((q & 1) ? 0u : 4u))) & 15u;
    switch (nib) {
        case 1: return 0;
        case 2: return 1;
        case 4: return 2;
        case 8: return 3;
        case 15: return 4;
        default: return CODE_OTHER;
    }
}

// Per tile: the SNPs inside its window [first_pos, max_end) -- two binary searches over the contig's sorted SNP
// positions, one thread per tile, so that the scan CTAs find their range with one load (and tiles over no SNP are
// passed over without touching their records).
__global__ void k_baf_tile_snps(const xg_tile *tiles, const xg_run *runs, int32_t n_tiles, int32_t n_gid,
                                const int32_t *snp_goff, const int32_t *snp_pos, int2 *out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    const xg_tile tile = tiles[t];
    const int32_t gid = runs[tile.run].gid;
    int2 r = make_int2(0, 0);
    if (gid >= 0 && gid < n_gid) {
        const int32_t g0 = snp_goff[gid], g1 = snp_goff[gid + 1];
        int32_t lo = g0, hi = g1;
        while (lo < hi) {
            int32_t mid = (lo + hi) >> 1;
            if (snp_pos[mid] < tile.first_pos) lo = mid + 1; else hi = mid;
        }
        r.x = lo;
        hi = g1;
        while (lo < hi) {
            int32_t mid = (lo + hi) >> 1;
            if (snp_pos[mid] < tile.max_end) lo = mid + 1; else hi = mid;
        }
        r.y = lo;
    }
    out[t] = r;
}

#define SCAN_SNP_CAP 256      // SNP positions of a tile staged in shared memory
#define SCAN_RPT (XG_TILE / 256)

// Persistent CTAs, two phases.
//   Phase 1 streams the CTA's tiles (static stride): a tile's SNP positions are staged in shared memory, every
//   thread loads its four records' (pos, end) up front (coalesced 8-byte loads) and finds the first SNP at or after
//   pos among the staged positions.  A read that covers a SNP (about one in twenty) is only NOTED -- (tile, record,
//   first SNP) appended to the CTA's own candidate list through a shared-memory cursor -- so that the stream never
//   waits for the dependent flag / key / barcode / CIGAR / sequence loads of the few.
//   Phase 2 takes the candidates 256 at a time, one per thread, so that those loads are in flight for all of them
//   at once; the (read, SNP) pairs of a batch reserve their place in the pair list with one atomic.
struct ScanCand {
    uint32_t rec;         // tile * XG_TILE + record of the tile
    int32_t snp;          // first sorted SNP at or after the read's pos
};

__global__ void __launch_bounds__(256) k_baf_scan(const __grid_constant__ BafScanDev P, const int2 *tile_snp,
                                                  int32_t n_tiles, ScanCand *cand_all, uint32_t cand_cap) {
    __shared__ int32_t s_snp[2][SCAN_SNP_CAP];
    __shared__ uint32_t s_warp[8];
    __shared__ unsigned long long s_base;
    __shared__ uint32_t s_ncand;
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    ScanCand *cand = cand_all + (size_t)blockIdx.x * cand_cap;       // this CTA's list (cand_cap = its tiles x XG_TILE)
    if (threadIdx.x == 0) s_ncand = 0;
    int buf = 0;
    // ---- phase 1
    for (int32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const int2 rg = tile_snp[t];
        if (rg.x >= rg.y) continue;       // no SNP under this tile: its records are never read
        const int32_t sa = rg.x, ns = rg.y - rg.x;
        const xg_tile tile = P.tiles[t];
        const bool staged = ns <= SCAN_SNP_CAP;
        int2 pe[SCAN_RPT];
#pragma unroll
        for (int r = 0; r < SCAN_RPT; r++) {
            const int32_t k = threadIdx.x + r * 256;
            pe[r] = k < tile.n_rec ? P.pos_end[tile.rec_beg + k] : make_int2(0, 0);
        }
        int32_t *sn = s_snp[buf];
        if (staged)
            for (int k = threadIdx.x; k < ns; k += 256) sn[k] = __ldg(&P.snp_pos[sa + k]);
        buf ^= 1;
        __syncthreads();                  // staged; and the other buffer is free again
#pragma unroll
        for (int r = 0; r < SCAN_RPT; r++) {
            const int32_t k = threadIdx.x + r * 256;
            // first SNP with pos >= read.pos (fetch(chrom, pos-1, pos): pos0 in [read.pos, read.end))
            int32_t lo = 0;
            bool hit = false;
            if (k < tile.n_rec) {
                if (staged) {
                    if (ns <= 8) {
                        for (int q = 0; q < ns; q++) lo += sn[q] < pe[r].x;
                    } else {
                        int32_t hi = ns;
                        while (lo < hi) {
                            int32_t mid = (lo + hi) >> 1;
                            if (sn[mid] < pe[r].x) lo = mid + 1; else hi = mid;
                        }
                    }
                    hit = lo < ns && sn[lo] < pe[r].y;
                } else {
                    int32_t hi = ns;
                    while (lo < hi) {
                        int32_t mid = (lo + hi) >> 1;
                        if (__ldg(&P.snp_pos[sa + mid]) < pe[r].x) lo = mid + 1; else hi = mid;
                    }
                    hit = lo < ns && __ldg(&P.snp_pos[sa + lo]) < pe[r].y;
                }
            }
            const unsigned m = __ballot_sync(0xffffffffu, hit);
            if (m) {
                uint32_t base = 0;
                if (lane == 0) base = atomicAdd(&s_ncand, (uint32_t)__popc(m));
                base = __shfl_sync(0xffffffffu, base, 0);
                if (hit) {
                    ScanCand c;
                    c.rec = (uint32_t)t * XG_TILE + (uint32_t)k;
                    c.snp = sa + lo;
                    cand[base + __popc(m & ((1u << lane) - 1u))] = c;
                }
            }
        }
    }
    __syncthreads();
    const uint32_t n_cand = s_ncand;
    // ---- phase 2: one candidate per thread
    for (uint32_t c0 = 0; c0 < n_cand; c0 += 256) {
        const uint32_t ci = c0 + threadIdx.x;
        uint32_t cnt = 0, col = 0, n_ops = 0;
        int32_t lo = 0, sb = 0;
        int64_t i = 0;
        int2 pe = make_int2(0, 0);
        uint64_t umi = 0;
        const uint32_t *cig = nullptr;
        do {
            if (ci >= n_cand) break;
            const ScanCand c = cand[ci];
            const uint32_t t = c.rec / XG_TILE;
            const xg_tile tile = P.tiles[t];
            i = tile.rec_beg + (c.rec % XG_TILE);
            lo = c.snp;
            sb = tile_snp[t].y;
            pe = P.pos_end[i];
            const uint32_t fmq = P.fmq[i];
            if (!read_passes_flags(P.fp, fmq)) break;
            const ulonglong2 ky = P.keys[i];
            umi = ky.y;
            if (umi == XG_KEY_NONE || umi == XG_KEY_EMPTY) break;
            if (P.fp.use_cell_tag) {
                if (ky.x == XG_KEY_NONE) break;
                int32_t cc = barcode_lookup(P.bc, ky.x);
                if (cc < 0) break;
                col = (uint32_t)cc;
            } else {
                col = (uint32_t)P.runs[tile.run].bam_idx;
            }
            n_ops = fmq >> 24;
            int32_t aln;
            if (n_ops == 0) {
                aln = pe.y - pe.x;
            } else {
                cig = P.cigar + P.cig_off[i];
                if (n_ops == 255) n_ops = __ldg(cig - 1);
                aln = 0;
                for (uint32_t q = 0; q < n_ops; q++) {
                    uint32_t w = __ldg(&cig[q]);
                    if (cig_aligned(w & 15u)) aln += (int32_t)(w >> 4);
                }
            }
            if (aln < P.fp.min_len) break;
            for (int32_t s = lo; s < sb && __ldg(&P.snp_pos[s]) < pe.y; s++) cnt++;
        } while (false);
        // the batch's pairs reserve their place: block-wide exclusive prefix sum, one atomic
        uint32_t incl = cnt;
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += y;
        }
        __syncthreads();                  // s_warp / s_base of the previous batch have been read
        if (lane == 31) s_warp[wp] = incl;
        __syncthreads();
        uint32_t before = 0, total = 0;
        for (int q = 0; q < 8; q++) {
            const uint32_t x = s_warp[q];
            if (q < wp) before += x;
            total += x;
        }
        if (total == 0) continue;         // uniform: every thread sees the same total
        if (threadIdx.x == 0) s_base = atomicAdd(P.n_pairs, (unsigned long long)total);
        __syncthreads();
        unsigned long long o = s_base + before + (incl - cnt);
        for (uint32_t q = 0; q < cnt; q++, o++) {
            const int32_t s = lo + (int32_t)q;
            const uint32_t code = base_at(P, i, pe.x, pe.y, n_ops, cig, __ldg(&P.snp_pos[s]));
            if (o < P.cap_pairs) {
                P.pr_snp[o] = (uint32_t)__ldg(&P.snp_idx[s]);
                P.pr_colal[o] = col | (code << 24);
                P.pr_umi[o] = umi;
                P.pr_ord[o] = (uint64_t)i;
            }
        }
    }
}

// find-or-insert of a 128-bit key; returns the slot
__device__ __forceinline__ uint32_t table_slot(xg_e128 *tbl, uint32_t cap, xg_e128 want) {
    uint32_t s = hash_to_range(mix64(want.a ^ (want.b * 0x9E3779B97F4A7C15ULL)), cap);
    while (true) {
        xg_e128 cur = ld128_relaxed(&tbl[s]);
        if (cur.b == 0) {
            xg_e128 empty;
            empty.a = 0;
            empty.b = 0;
            cur = cas128(&tbl[s], empty, want);
            if (cur.b == 0) return s;
        }
        if (cur.a == want.a && cur.b == want.b) return s;
        s = (s + 1 == cap) ? 0 : s + 1;
    }
}

__global__ void k_baf_first(int64_t n, const uint32_t *pr_snp, const uint32_t *pr_colal,
                            const uint64_t *pr_umi, const uint64_t *pr_ord, xg_e128 *tbl, uint32_t cap,
                            unsigned long long *min_ord, uint32_t *pr_slot) {
    int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    xg_e128 want;
    want.a = pr_umi[p];
    want.b = ((unsigned long long)(pr_colal[p] & 0xFFFFFFu) << 32) | ((unsigned long long)pr_snp[p] + 1ull);
    uint32_t s = table_slot(tbl, cap, want);
    pr_slot[p] = s;
    atomicMin(&min_ord[s], (unsigned long long)pr_ord[p]);
}

__global__ void k_baf_resolve(int64_t n, const uint32_t *pr_snp, uint32_t *pr_colal,
                              const uint64_t *pr_ord, const unsigned long long *min_ord,
                              const uint32_t *pr_slot, unsigned long long *totals) {
    int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    if (min_ord[pr_slot[p]] != pr_ord[p]) return;
    uint32_t ca = pr_colal[p];
    pr_colal[p] = ca | 0x80000000u;              // winner: the first read of this (SNP, cell, UMI)
    uint32_t code = (ca >> 24) & 0x7u;
    if (code == CODE_NONE) return;               // allele None: claims the UMI, counts nowhere
    uint32_t bucket = code < 4 ? code : 4;       // non-ACGT -> "N" bucket (mcount.py:145-149)
    atomicAdd(&totals[(size_t)pr_snp[p] * 5 + bucket], 1ull);
}

struct BafRegDev {
    int64_t n_pairs;
    const uint32_t *pr_snp, *pr_colal;
    const uint64_t *pr_umi;
    const int64_t *snp_reg_ptr;
    const int32_t *snp_reg;
    const uint8_t *hap_of, *keep;
    xg_e128 *tbl;
    uint32_t cap;
    uint32_t *mask;
};

// upper bound of the (region, cell, UMI) elements of every region: one per (winner, region)
__global__ void k_baf_count_combos(BafRegDev P, int32_t *reg_cnt) {
    int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P.n_pairs) return;
    uint32_t ca = P.pr_colal[p], snp = P.pr_snp[p];
    if (!(ca & 0x80000000u) || ((ca >> 24) & 7u) == CODE_NONE || !P.keep[snp]) return;
    for (int64_t k = P.snp_reg_ptr[snp]; k < P.snp_reg_ptr[snp + 1]; k++) atomicAdd(&reg_cnt[P.snp_reg[k]], 1);
}

// find-or-insert of a 128-bit key; returns the slot and whether it was created by this call
__device__ __forceinline__ uint32_t table_slot_new(xg_e128 *tbl, uint32_t cap, xg_e128 want, bool *is_new) {
    uint32_t s = hash_to_range(mix64(want.a ^ (want.b * 0x9E3779B97F4A7C15ULL)), cap);
    *is_new = false;
    while (true) {
        xg_e128 cur = ld128_relaxed(&tbl[s]);
        if (cur.b == 0) {
            xg_e128 empty;
            empty.a = 0;
            empty.b = 0;
            cur = cas128(&tbl[s], empty, want);
            if (cur.b == 0) {
                *is_new = true;
                return s;
            }
        }
        if (cur.a == want.a && cur.b == want.b) return s;
        s = (s + 1 == cap) ? 0 : s + 1;
    }
}

// winners of kept SNPs OR their haplotype bit into (region, cell, UMI); a new element is
// appended to its region's log so that the region can be reduced from its own elements only
__global__ void k_baf_region_masks(BafRegDev P, const int64_t *reg_log_off, int32_t *reg_cur, uint32_t *reg_log) {
    int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P.n_pairs) return;
    uint32_t ca = P.pr_colal[p], snp = P.pr_snp[p];
    uint32_t code = (ca >> 24) & 7u;
    if (!(ca & 0x80000000u) || code == CODE_NONE || !P.keep[snp]) return;
    uint32_t bit = 1u << min((uint32_t)P.hap_of[(size_t)snp * 8 + code], 2u);     // 1 ref-hap, 2 alt-hap, 4 other
    uint32_t col = ca & 0xFFFFFFu;
    uint64_t umi = P.pr_umi[p];
    for (int64_t k = P.snp_reg_ptr[snp]; k < P.snp_reg_ptr[snp + 1]; k++) {
        const int32_t r = P.snp_reg[k];
        xg_e128 want;
        want.a = umi;
        want.b = ((unsigned long long)col << 32) | ((unsigned long long)r + 1ull);
        bool is_new;
        uint32_t s = table_slot_new(P.tbl, P.cap, want, &is_new);
        atomicOr(&P.mask[s], bit);
        if (is_new) reg_log[reg_log_off[r] + atomicAdd(&reg_cur[r], 1)] = s;
    }
}

// Reduce one region to its rows of AD / DP / OTH (baf/fc/core.py:156-192 + emit :84-101):
// per UMI mask m (bit0 ref-hap, bit1 alt-hap, bit2 other):
//   no_dup_hap:  AD += alt - both,  DP += ref + alt - 2*both      (both = ref & alt)
//   otherwise:   AD += alt,         DP += ref + alt
//   OTH += other & !(ref | alt)
// Histograms over cells + a bitmap of touched cells in shared memory; the set bits walked in
// order give the rows in column order.  Persistent CTAs, work counter, staging + cursors per
// matrix; column-range passes when 3 histograms of all cells do not fit.
__global__ void __launch_bounds__(256) k_baf_finalize(const xg_e128 *tbl, const uint32_t *mask,
                                                      const int64_t *reg_log_off, const int32_t *reg_cur,
                                                      const uint32_t *reg_log, int32_t n_regions, int32_t n_cols,
                                                      int32_t hist_cols, int32_t no_dup, unsigned int *work,
                                                      unsigned long long *cursor /* [3] */,
                                                      int64_t *seg_base /* [3][n_regions] */,
                                                      int32_t *seg_nnz /* [3][n_regions] */,
                                                      int32_t *st_col /* [3][cap] */, int32_t *st_val, int64_t st_cap) {
    extern __shared__ uint32_t smem[];
    uint32_t *hist = smem;                                   // [3][hist_cols]
    uint32_t *bitmap = smem + 3 * (size_t)hist_cols;         // (hist_cols + 31) / 32
    __shared__ int warp_tot[8];
    __shared__ long long base_s;
    __shared__ int r_s;
    const int nwm = (hist_cols + 31) >> 5;
    for (int c = threadIdx.x; c < 3 * hist_cols; c += blockDim.x) hist[c] = 0;
    for (int c = threadIdx.x; c < nwm; c += blockDim.x) bitmap[c] = 0;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int n_pass = (n_cols + hist_cols - 1) / hist_cols;
    while (true) {
        __syncthreads();
        if (threadIdx.x == 0) r_s = (int)atomicAdd(work, 1u);
        __syncthreads();
        const int r = r_s;
        if (r >= n_regions) break;
        const int n_el = reg_cur[r];
        if (n_el == 0) continue;
        const uint32_t *log = reg_log + reg_log_off[r];
        long long base[3] = {0, 0, 0};
        // stage 0 (only when n_pass > 1): count; stage 1: write
        for (int stage = (n_pass > 1 ? 0 : 1); stage < 2; stage++) {
            int total_nz[3] = {0, 0, 0};
            for (int pass = 0; pass < n_pass; pass++) {
                const uint32_t c_lo = (uint32_t)pass * (uint32_t)hist_cols;
                const int nc = min(hist_cols, n_cols - (int)c_lo);
                const int nw = (nc + 31) >> 5;
                for (int k = threadIdx.x; k < n_el; k += blockDim.x) {
                    const uint32_t s = log[k];
                    const uint32_t col = (uint32_t)(tbl[s].b >> 32) - c_lo;
                    if (col >= (uint32_t)nc) continue;
                    const uint32_t m = mask[s];
                    const int ref = m & 1, alt = (m >> 1) & 1, both = ref & alt;
                    const int ad_c = no_dup ? alt - both : alt;
                    const int dp_c = no_dup ? ref + alt - 2 * both : ref + alt;
                    const int ot_c = ((m & 4u) && !(m & 3u)) ? 1 : 0;
                    if (ad_c) atomicAdd(&hist[col], (uint32_t)ad_c);
                    if (dp_c) atomicAdd(&hist[hist_cols + col], (uint32_t)dp_c);
                    if (ot_c) atomicAdd(&hist[2 * hist_cols + col], 1u);
                    if (ad_c | dp_c | ot_c) atomicOr(&bitmap[col >> 5], 1u << (col & 31));
                }
                __syncthreads();
                const bool writing = (stage == 1);
                for (int wh = 0; wh < 3; wh++) {
                    const uint32_t *hw = hist + (size_t)wh * hist_cols;
                    if (!writing || n_pass == 1) {            // non-zero cells of this range
                        int nz = 0;
                        for (int k = threadIdx.x; k < nw; k += blockDim.x) {
                            uint32_t bits = bitmap[k];
                            while (bits) {
                                const int bpos = __ffs(bits) - 1;
                                bits &= bits - 1;
                                nz += hw[(k << 5) + bpos] != 0;
                            }
                        }
                        for (int d = 16; d > 0; d >>= 1) nz += __shfl_xor_sync(0xffffffffu, nz, d);
                        if (lane == 0) warp_tot[w] = nz;
                        __syncthreads();
                        for (int k = 0; k < 8; k++) total_nz[wh] += warp_tot[k];
                        __syncthreads();
                    }
                    if (writing && n_pass == 1) {             // single range: reserve now
                        if (threadIdx.x == 0) {
                            long long b = total_nz[wh] ? (long long)atomicAdd(&cursor[wh], (unsigned long long)total_nz[wh]) : 0;
                            seg_base[(size_t)wh * n_regions + r] = b;
                            seg_nnz[(size_t)wh * n_regions + r] = total_nz[wh];
                            base_s = b;
                        }
                        __syncthreads();
                        base[wh] = base_s;
                    }
                    if (!writing) continue;
                    for (int k0 = 0; k0 < nw; k0 += blockDim.x) {     // ordered walk over the bitmap
                        const int k = k0 + threadIdx.x;
                        uint32_t bits = k < nw ? bitmap[k] : 0u;
                        int cnt = 0;
                        for (uint32_t bb = bits; bb; bb &= bb - 1) cnt += hw[(k << 5) + __ffs(bb) - 1] != 0;
                        int incl = cnt;
                        for (int d = 1; d < 32; d <<= 1) {
                            int y = __shfl_up_sync(0xffffffffu, incl, d);
                            if (lane >= d) incl += y;
                        }
                        if (lane == 31) warp_tot[w] = incl;
                        __syncthreads();
                        int before = 0, tot = 0;
                        for (int q = 0; q < 8; q++) {
                            const int x = warp_tot[q];
                            if (q < w) before += x;
                            tot += x;
                        }
                        long long o = base[wh] + before + (incl - cnt);
                        while (bits) {
                            const int bpos = __ffs(bits) - 1;
                            bits &= bits - 1;
                            const int c = (k << 5) + bpos;
                            const uint32_t v = hw[c];
                            if (v) {
                                st_col[(size_t)wh * st_cap + o] = (int32_t)(c_lo + (uint32_t)c);
                                st_val[(size_t)wh * st_cap + o] = (int32_t)v;
                                o++;
                            }
                        }
                        base[wh] += tot;
                        __syncthreads();
                    }
                }
                // clear what this range touched
                for (int k = threadIdx.x; k < nw; k += blockDim.x) {
                    uint32_t bits = bitmap[k];
                    while (bits) {
                        const int c = (k << 5) + __ffs(bits) - 1;
                        bits &= bits - 1;
                        hist[c] = 0;
                        hist[hist_cols + c] = 0;
                        hist[2 * hist_cols + c] = 0;
                    }
                    bitmap[k] = 0;
                }
                __syncthreads();
            }
            if (stage == 0) {                                 // multi-range: reserve after counting
                for (int wh = 0; wh < 3; wh++) {
                    if (threadIdx.x == 0) {
                        long long b = total_nz[wh] ? (long long)atomicAdd(&cursor[wh], (unsigned long long)total_nz[wh]) : 0;
                        seg_base[(size_t)wh * n_regions + r] = b;
                        seg_nnz[(size_t)wh * n_regions + r] = total_nz[wh];
                        base_s = b;
                    }
                    __syncthreads();
                    base[wh] = base_s;
                    __syncthreads();
                }
            }
        }
    }
}

template <class T>
int upload_arr(xg_ctx *ctx, const T *src, size_t n, const char *name, const T **out) {
    T *d = (T *)ctx->get(name, sizeof(T) * (n + 1));
    if (!d) return XG_E_CUDA;
    if (n) XG_CUDA(cudaMemcpyAsync(d, src, sizeof(T) * n, cudaMemcpyHostToDevice, ctx->stream));
    *out = d;
    return XG_OK;
}

}  // namespace

extern "C" void xg_baf_state_free(xg_ctx *ctx, xg_baf_state *st) {
    if (!st) return;
    if (ctx) cudaSetDevice(ctx->device);
    for (void *p : {(void *)st->pr_snp, (void *)st->pr_colal, (void *)st->pr_umi})
        if (p) {
            if (ctx) ctx->dev_put(p); else cudaFree(p);
        }
    delete st;
}

extern "C" int xg_baf_pileup(xg_ctx *ctx, const xg_dreads *rd, const xg_snps *snps,
                             const xg_barcodes *cells, const xg_params *par, int64_t *totals,
                             xg_baf_state **state) {
    if (!ctx || !ctx->stream) return ctx ? ctx->fail(XG_E_CUDA, "context has no device") : XG_E_ARG;
    if (!rd || !snps || !cells || !par || !state)          // totals == NULL: they stay on the device (xg_baf_fc)
        return ctx->fail(XG_E_ARG, "xg_baf_pileup: null argument");
    if (!rd->seq || !rd->seq_off) return ctx->fail(XG_E_ARG, "xg_baf_pileup: reads were decoded without sequences");
    if (cells->n_samples <= 0 || cells->n_samples >= (1 << 24))
        return ctx->fail(XG_E_ARG, "xg_baf_pileup: number of cells must be in [1, 2^24)");
    if (par->use_cell_tag && cells->n != cells->n_samples)
        return ctx->fail(XG_E_ARG, "xg_baf_pileup: barcode mode needs one key per column");
    XG_CUDA(cudaSetDevice(ctx->device));
    for (double &t : ctx->timing) t = 0;
    int launches = 0;
    const auto t_call = std::chrono::steady_clock::now();
    auto ms_since = [](std::chrono::steady_clock::time_point a) {
        return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - a).count();
    };

    int32_t n_gid = 0;
    for (auto &r : rd->h_runs) n_gid = std::max(n_gid, r.gid + 1);
    if (!par->use_cell_tag)
        for (auto &r : rd->h_runs)
            if (r.bam_idx >= cells->n_samples) return ctx->fail(XG_E_ARG, "more BAMs than sample columns");
    // SNPs sorted by (gid, pos); pos < 0 (1-based pos <= 0) can never be fetched.  The sorted
    // table depends on the SNP list only: it is kept on the device while the caller passes
    // the same list (hash of the arrays).
    const size_t sb = sizeof(int32_t) * (size_t)snps->n;
    const std::initializer_list<xg_input_key::Span> in = {
        {&n_gid, sizeof n_gid}, {&snps->n, sizeof snps->n}, {snps->gid, sb}, {snps->pos, sb}};
    const uint64_t sh = xg_input_key::hash_of(in);
    const bool snp_cached = ctx->bf_snp_valid && ctx->bf_snp_key.matches(sh, in);
    if (!snp_cached) {
        ctx->bf_snp_valid = false;
        std::vector<int32_t> ord;
        for (int32_t i = 0; i < snps->n; i++)
            if (snps->gid[i] >= 0 && snps->gid[i] < n_gid && snps->pos[i] >= 0) ord.push_back(i);
        std::sort(ord.begin(), ord.end(), [&](int32_t a, int32_t b) {
            if (snps->gid[a] != snps->gid[b]) return snps->gid[a] < snps->gid[b];
            if (snps->pos[a] != snps->pos[b]) return snps->pos[a] < snps->pos[b];
            return a < b;
        });
        std::vector<int32_t> goff((size_t)n_gid + 1, 0), spos(ord.size()), sidx(ord.size());
        for (size_t k = 0; k < ord.size(); k++) {
            goff[(size_t)snps->gid[ord[k]] + 1]++;
            spos[k] = snps->pos[ord[k]];
            sidx[k] = ord[k];
        }
        for (int32_t g = 0; g < n_gid; g++) goff[(size_t)g + 1] += goff[(size_t)g];
        const int32_t *dummy = nullptr;
        int rc0;
        if ((rc0 = upload_arr(ctx, goff.data(), goff.size(), "bf_goff", &dummy))) return rc0;
        if ((rc0 = upload_arr(ctx, spos.data(), spos.size(), "bf_spos", &dummy))) return rc0;
        if ((rc0 = upload_arr(ctx, sidx.data(), sidx.size(), "bf_sidx", &dummy))) return rc0;
        XG_CUDA(cudaStreamSynchronize(ctx->stream));
        ctx->bf_snp_key.assign(sh, in);
        ctx->bf_snp_sorted = (int64_t)ord.size();
        ctx->bf_snp_valid = true;
    }
    const bool any_snp = ctx->bf_snp_sorted > 0;

    BafScanDev P;
    memset(&P, 0, sizeof(P));
    P.pos_end = rd->pos_end;
    P.fmq = rd->fmq;
    P.cig_off = rd->cig_off;
    P.cigar = rd->cigar;
    P.seq_off = rd->seq_off;
    P.seq = rd->seq;
    P.keys = rd->keys;
    P.runs = rd->runs;
    P.tiles = rd->tiles;
    P.n_gid = n_gid;
    int rc;
    P.snp_goff = (const int32_t *)ctx->scratch["bf_goff"].p;
    P.snp_pos = (const int32_t *)ctx->scratch["bf_spos"].p;
    P.snp_idx = (const int32_t *)ctx->scratch["bf_sidx"].p;
    P.fp.min_mapq = par->min_mapq;
    P.fp.min_len = par->min_len;
    P.fp.incl_flag = par->incl_flag;
    P.fp.excl_flag = par->excl_flag;
    P.fp.no_orphan = par->no_orphan;
    P.fp.use_cell_tag = par->use_cell_tag;
    P.fp.need_umi_tag = par->need_umi_tag;
    if (par->use_cell_tag && (rc = xg_build_barcode_table(ctx, cells, &P.bc))) return rc;
    XG_GET(d_tile_snp, int2, "bf_tile_snp", rd->n_tiles + 1);
    // candidate lists of the scan CTAs: room for every record of the tiles a CTA walks
    const int scan_grid = std::max(1, std::min(rd->n_tiles, 148 * 8));
    const uint32_t cand_cap = (uint32_t)((rd->n_tiles + scan_grid - 1) / scan_grid) * XG_TILE;
    if ((uint64_t)rd->n_tiles * XG_TILE >= (1ull << 32))
        return ctx->fail(XG_E_LIMIT, "xg_baf_pileup: more than 2^32 record slots in one batch");
    XG_GET(d_cand, ScanCand, "bf_cand", (size_t)scan_grid * cand_cap + 1);
    XG_GET(d_npairs, unsigned long long, "bf_npairs", 2);
    XG_GET(d_totals, unsigned long long, "bf_totals", (size_t)snps->n * 5 + 1);
    ctx->timing[8] = ms_since(t_call);          // host: SNP table (cached), barcode table, buffers (nothing to wait for)

    cudaEventRecord(ctx->ev[0], ctx->stream);
    if (rd->n_tiles > 0 && any_snp) {
        k_baf_tile_snps<<<(rd->n_tiles + 255) / 256, 256, 0, ctx->stream>>>(rd->tiles, rd->runs, rd->n_tiles, n_gid,
                                                                          P.snp_goff, P.snp_pos, d_tile_snp);
        launches++;
    }
    // scan; the pair buffer grows and the scan is repeated in the (rare) overflow case
    unsigned long long cap_pairs = std::max<unsigned long long>(1ull << 16, (unsigned long long)rd->n_reads / 4);
    unsigned long long n_pairs = 0;
    float t_scan = 0;
    for (int attempt = 0; attempt < 8; attempt++) {
        XG_GET(pr_snp, uint32_t, "bf_pr_snp", cap_pairs);
        XG_GET(pr_colal, uint32_t, "bf_pr_colal", cap_pairs);
        XG_GET(pr_umi, uint64_t, "bf_pr_umi", cap_pairs);
        XG_GET(pr_ord, uint64_t, "bf_pr_ord", cap_pairs);
        P.pr_snp = pr_snp;
        P.pr_colal = pr_colal;
        P.pr_umi = pr_umi;
        P.pr_ord = pr_ord;
        P.n_pairs = d_npairs;
        P.cap_pairs = cap_pairs;
        XG_CUDA(cudaMemsetAsync(d_npairs, 0, 16, ctx->stream));
        cudaEventRecord(ctx->ev[1], ctx->stream);
        if (rd->n_tiles > 0 && any_snp) {
            k_baf_scan<<<scan_grid, 256, 0, ctx->stream>>>(P, d_tile_snp, rd->n_tiles, d_cand, cand_cap);
            launches++;
            XG_CUDA(cudaGetLastError());
        }
        cudaEventRecord(ctx->ev[2], ctx->stream);
        XG_CUDA(cudaMemcpyAsync(&n_pairs, d_npairs, 8, cudaMemcpyDeviceToHost, ctx->stream));
        XG_CUDA(cudaStreamSynchronize(ctx->stream));
        cudaEventElapsedTime(&t_scan, ctx->ev[1], ctx->ev[2]);
        if (n_pairs <= cap_pairs) break;
        cap_pairs = n_pairs + n_pairs / 8 + 1024;
    }
    if (n_pairs > cap_pairs) return ctx->fail(XG_E_LIMIT, "pair buffer overflow");
    if (n_pairs >= (1ull << 31)) return ctx->fail(XG_E_LIMIT, "more than 2^31 (read, SNP) pairs in one batch");

    XG_CUDA(cudaMemsetAsync(d_totals, 0, sizeof(unsigned long long) * ((size_t)snps->n * 5 + 1), ctx->stream));
    xg_baf_state *st = new xg_baf_state();
    st->n_pairs = (int64_t)n_pairs;
    st->n_snps = snps->n;
    st->n_cols = cells->n_samples;
    if (n_pairs > 0) {
        const uint64_t cap64 = 2ull * n_pairs + 16ull;         // slots are 32-bit indices
        if (cap64 > 0xFFFFFFFFull) {
            xg_baf_state_free(ctx, st);
            return ctx->fail(XG_E_LIMIT, "(SNP, cell, UMI) table exceeds 2^32 slots");
        }
        const uint32_t cap = (uint32_t)cap64;
        XG_GET(tbl, xg_e128, "bf_tbl1", cap);
        XG_GET(min_ord, unsigned long long, "bf_minord", cap);
        XG_GET(pr_slot, uint32_t, "bf_pr_slot", n_pairs);
        XG_CUDA(cudaMemsetAsync(tbl, 0, sizeof(xg_e128) * cap, ctx->stream));
        XG_CUDA(cudaMemsetAsync(min_ord, 0xFF, sizeof(unsigned long long) * cap, ctx->stream));
        unsigned grid = (unsigned)((n_pairs + 255) / 256);
        k_baf_first<<<grid, 256, 0, ctx->stream>>>((int64_t)n_pairs, P.pr_snp, P.pr_colal, P.pr_umi,
                                                   P.pr_ord, tbl, cap, min_ord, pr_slot);
        k_baf_resolve<<<grid, 256, 0, ctx->stream>>>((int64_t)n_pairs, P.pr_snp, P.pr_colal, P.pr_ord,
                                                     min_ord, pr_slot, d_totals);
        launches += 4;
        XG_CUDA(cudaGetLastError());
        // the state keeps its own copy of the pairs (scratch buffers are reused by later calls)
        st->pr_snp = (uint32_t *)ctx->dev_get(n_pairs * 4);
        st->pr_colal = (uint32_t *)ctx->dev_get(n_pairs * 4);
        st->pr_umi = (uint64_t *)ctx->dev_get(n_pairs * 8);
        if (!st->pr_snp || !st->pr_colal || !st->pr_umi) {
            xg_baf_state_free(ctx, st);
            return ctx->fail(XG_E_CUDA, "out of device memory for the pileup state");
        }
        cudaMemcpyAsync(st->pr_snp, P.pr_snp, n_pairs * 4, cudaMemcpyDeviceToDevice, ctx->stream);
        cudaMemcpyAsync(st->pr_colal, P.pr_colal, n_pairs * 4, cudaMemcpyDeviceToDevice, ctx->stream);
        cudaMemcpyAsync(st->pr_umi, P.pr_umi, n_pairs * 8, cudaMemcpyDeviceToDevice, ctx->stream);
    }
    cudaEventRecord(ctx->ev[3], ctx->stream);
    unsigned long long *h_tot = nullptr;
    if (totals) {
        h_tot = (unsigned long long *)ctx->pinned_get(sizeof(unsigned long long) * ((size_t)snps->n * 5 + 1));
        if (!h_tot) {
            xg_baf_state_free(ctx, st);
            return ctx->fail(XG_E_NOMEM, "out of pinned host memory");
        }
    }
    cudaEventRecord(ctx->ev[4], ctx->stream);
    if (totals)
        cudaMemcpyAsync(h_tot, d_totals, sizeof(unsigned long long) * (size_t)snps->n * 5, cudaMemcpyDeviceToHost,
                        ctx->stream);
    cudaEventRecord(ctx->ev[5], ctx->stream);
    if (!totals) {
        // xg_baf_fc: the totals stay on the device and the count follows on the same stream -- nothing to wait for
        // here (a call that has a short kernel's worth of work pays every synchronisation in full when another
        // context keeps the GPU busy); the caller reads the scan's time from ev[1] / ev[2] at its end
        ctx->timing[2] = launches;
        ctx->timing[6] = (double)n_pairs;
        ctx->timing[9] = ctx->timing[10] = ms_since(t_call);
        *state = st;
        return XG_OK;
    }
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        if (h_tot) ctx->pinned_put(h_tot);
        xg_baf_state_free(ctx, st);
        return ctx->fail(XG_E_CUDA, std::string("baf pileup: ") + cudaGetErrorString(e));
    }
    ctx->timing[9] = ms_since(t_call);          // ... + kernels + totals on the host
    if (totals) {
        memcpy(totals, h_tot, sizeof(int64_t) * (size_t)snps->n * 5);   // counts < 2^31: the same bits as int64
        ctx->pinned_put(h_tot);
    }
    ctx->timing[10] = ms_since(t_call);         // ... + copy into the caller's array
    float t_all = 0, t_d2h = 0;
    cudaEventElapsedTime(&t_all, ctx->ev[0], ctx->ev[3]);
    cudaEventElapsedTime(&t_d2h, ctx->ev[4], ctx->ev[5]);
    ctx->timing[0] = t_all;
    ctx->timing[1] = t_scan;
    ctx->timing[2] = launches;
    ctx->timing[4] = t_d2h;
    ctx->timing[6] = (double)n_pairs;
    *state = st;
    return XG_OK;
}

// keep: the caller's SNP filter (host array) -- or keep_dev: the one k_baf_snp_filter left on the device
static int baf_count_impl(xg_ctx *ctx, xg_baf_state *st, int32_t n_regions, const int64_t *reg_ptr,
                          const int32_t *reg_snp, const uint8_t *hap_of, const uint8_t *keep, const uint8_t *keep_dev,
                          int32_t no_dup_hap, xg_coo **ad, xg_coo **dp, xg_coo **oth) {
    if (!ctx || !ctx->stream) return ctx ? ctx->fail(XG_E_CUDA, "context has no device") : XG_E_ARG;
    if (!st || n_regions < 0 || !reg_ptr || !hap_of || (!keep && !keep_dev) || !ad || !dp || !oth)
        return ctx->fail(XG_E_ARG, "xg_baf_count: bad argument");
    XG_CUDA(cudaSetDevice(ctx->device));
    for (double &t : ctx->timing) t = 0;
    int launches = 0;
    const auto t_call = std::chrono::steady_clock::now();
    auto ms_since = [](std::chrono::steady_clock::time_point a) {
        return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - a).count();
    };
    const int32_t n_cols = st->n_cols, n_snps = st->n_snps;
    // invert region -> SNP lists (cached on the device while the caller passes the same lists)
    const int64_t n_mem = reg_ptr[n_regions];
    const std::initializer_list<xg_input_key::Span> in = {{&n_snps, sizeof n_snps},
                                                          {&n_regions, sizeof n_regions},
                                                          {reg_ptr, sizeof(int64_t) * ((size_t)n_regions + 1)},
                                                          {reg_snp, sizeof(int32_t) * (size_t)n_mem}};
    const uint64_t sh = xg_input_key::hash_of(in);
    const bool sr_cached = ctx->bf_sr_valid && ctx->bf_sr_key.matches(sh, in);
    if (!sr_cached) {
        ctx->bf_sr_valid = false;
        std::vector<int64_t> sr_ptr((size_t)n_snps + 1, 0);
        for (int64_t k = 0; k < n_mem; k++) {
            if (reg_snp[k] < 0 || reg_snp[k] >= n_snps) return ctx->fail(XG_E_ARG, "reg_snp out of range");
            sr_ptr[(size_t)reg_snp[k] + 1]++;
        }
        for (int32_t s2 = 0; s2 < n_snps; s2++) sr_ptr[(size_t)s2 + 1] += sr_ptr[(size_t)s2];
        std::vector<int32_t> sr((size_t)n_mem);
        {
            std::vector<int64_t> cur(sr_ptr.begin(), sr_ptr.end() - 1);
            for (int32_t r = 0; r < n_regions; r++)
                for (int64_t k = reg_ptr[r]; k < reg_ptr[r + 1]; k++) sr[(size_t)cur[(size_t)reg_snp[k]]++] = r;
        }
        const int64_t *d64 = nullptr;
        const int32_t *d32 = nullptr;
        int rc0;
        if ((rc0 = upload_arr(ctx, sr_ptr.data(), sr_ptr.size(), "bf_sr_ptr", &d64))) return rc0;
        if ((rc0 = upload_arr(ctx, sr.data(), sr.size(), "bf_sr", &d32))) return rc0;
        XG_CUDA(cudaStreamSynchronize(ctx->stream));
        ctx->bf_sr_key.assign(sh, in);
        ctx->bf_sr_valid = true;
    }

    BafRegDev R;
    memset(&R, 0, sizeof(R));
    R.n_pairs = st->n_pairs;
    R.pr_snp = st->pr_snp;
    R.pr_colal = st->pr_colal;
    R.pr_umi = st->pr_umi;
    int rc;
    R.snp_reg_ptr = (const int64_t *)ctx->scratch["bf_sr_ptr"].p;
    R.snp_reg = (const int32_t *)ctx->scratch["bf_sr"].p;
    if ((rc = upload_arr(ctx, hap_of, (size_t)n_snps * 8, "bf_hap_of", &R.hap_of))) return rc;
    if (keep_dev)
        R.keep = keep_dev;
    else if ((rc = upload_arr(ctx, keep, (size_t)n_snps, "bf_keep", &R.keep)))
        return rc;
    XG_GET(reg_cnt, int32_t, "bf_reg_cnt", n_regions + 1);
    XG_GET(reg_cur, int32_t, "bf_reg_cur", n_regions + 1);
    XG_GET(reg_log_off, int64_t, "bf_reg_log_off", n_regions + 2);
    XG_GET(cursor, unsigned long long, "bf_cursor", 4);
    XG_GET(work, unsigned int, "bf_work", 4);
    XG_GET(seg_base, int64_t, "bf_seg_base", 3 * (size_t)n_regions + 1);
    XG_GET(seg_nnz, int32_t, "bf_seg_nnz", 3 * (size_t)n_regions + 1);
    ctx->timing[8] = ms_since(t_call);          // host: region lists (cached), hap / keep upload, buffers (nothing to wait for)

    cudaEventRecord(ctx->ev[0], ctx->stream);
    unsigned grid = (unsigned)((st->n_pairs + 255) / 256);
    XG_CUDA(cudaMemsetAsync(reg_cnt, 0, sizeof(int32_t) * (size_t)(n_regions + 1), ctx->stream));
    XG_CUDA(cudaMemsetAsync(reg_cur, 0, sizeof(int32_t) * (size_t)(n_regions + 1), ctx->stream));
    XG_CUDA(cudaMemsetAsync(cursor, 0, 32, ctx->stream));
    XG_CUDA(cudaMemsetAsync(work, 0, 16, ctx->stream));
    XG_CUDA(cudaMemsetAsync(seg_base, 0, sizeof(int64_t) * (3 * (size_t)n_regions + 1), ctx->stream));
    XG_CUDA(cudaMemsetAsync(seg_nnz, 0, sizeof(int32_t) * (3 * (size_t)n_regions + 1), ctx->stream));
    if (st->n_pairs > 0) {
        k_baf_count_combos<<<grid, 256, 0, ctx->stream>>>(R, reg_cnt);
        launches++;
    }
    k_exclusive_scan<<<1, 1024, 0, ctx->stream>>>(reg_cnt, reg_log_off, n_regions);
    launches++;
    long long combos = 0;
    XG_CUDA(cudaMemcpyAsync(&combos, reg_log_off + n_regions, 8, cudaMemcpyDeviceToHost, ctx->stream));
    XG_CUDA(cudaStreamSynchronize(ctx->stream));
    if (combos >= (1ll << 31)) return ctx->fail(XG_E_LIMIT, "more than 2^31 (region, cell, UMI) candidates");
    const uint64_t cap64 = 2ull * (uint64_t)combos + 16ull;   // slots are 32-bit indices
    if (cap64 > 0xFFFFFFFFull) return ctx->fail(XG_E_LIMIT, "(region, cell, UMI) table exceeds 2^32 slots");
    const uint32_t cap = (uint32_t)cap64;
    XG_GET(tbl, xg_e128, "bf_tbl2", cap);
    XG_GET(mask, uint32_t, "bf_mask", cap);
    XG_GET(reg_log, uint32_t, "bf_reg_log", combos + 1);
    XG_GET(st_col, int32_t, "bf_st_col", 3 * (size_t)combos + 1);
    XG_GET(st_val, int32_t, "bf_st_val", 3 * (size_t)combos + 1);
    XG_CUDA(cudaMemsetAsync(tbl, 0, sizeof(xg_e128) * cap, ctx->stream));
    XG_CUDA(cudaMemsetAsync(mask, 0, sizeof(uint32_t) * cap, ctx->stream));
    R.tbl = tbl;
    R.cap = cap;
    R.mask = mask;
    if (combos > 0) {
        k_baf_region_masks<<<grid, 256, 0, ctx->stream>>>(R, reg_log_off, reg_cur, reg_log);
        launches++;
        // three histograms over the cells (+ bitmap) in shared memory; column ranges if too many
        const int32_t hist_cols = std::min(n_cols, 14 * 1024);
        const size_t smem = (size_t)hist_cols * 12 + (size_t)((hist_cols + 31) / 32) * 4;
        XG_CUDA(cudaFuncSetAttribute(k_baf_finalize, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const int per_sm = std::max(1, std::min(8, (int)(200 * 1024 / (smem + 1024))));
        k_baf_finalize<<<std::min(n_regions, 148 * per_sm), 256, smem, ctx->stream>>>(
            tbl, mask, reg_log_off, reg_cur, reg_log, n_regions, n_cols, hist_cols, no_dup_hap, work, cursor,
            seg_base, seg_nnz, st_col, st_val, (int64_t)combos);
        launches++;
        XG_CUDA(cudaGetLastError());
    }
    const double ms_kernels = ms_since(t_call);
    xg_coo **outs[3] = {ad, dp, oth};
    if ((rc = xg_staging_to_coo3(ctx, "bf3", n_regions, n_cols, seg_base, seg_nnz, st_col, st_val, (int64_t)combos, outs,
                                 &launches)))
        return rc;
    float t_all = 0;
    cudaEventElapsedTime(&t_all, ctx->ev[0], ctx->ev[3]);
    ctx->timing[0] = t_all;
    ctx->timing[2] = launches;
    ctx->timing[6] = (double)combos;
    ctx->timing[9] = ms_kernels;                // ... + kernels queued (one sync for the candidate count)
    ctx->timing[10] = ms_since(t_call);         // ... + the three results on the host
    return XG_OK;
}

extern "C" int xg_baf_count(xg_ctx *ctx, xg_baf_state *st, int32_t n_regions, const int64_t *reg_ptr,
                            const int32_t *reg_snp, const uint8_t *hap_of, const uint8_t *keep,
                            int32_t no_dup_hap, xg_coo **ad, xg_coo **dp, xg_coo **oth) {
    if (ctx && !keep) return ctx->fail(XG_E_ARG, "xg_baf_count: bad argument");
    return baf_count_impl(ctx, st, n_regions, reg_ptr, reg_snp, hap_of, keep, nullptr, no_dup_hap, ad, dp, oth);
}

// plp_snp's filter (baf/fc/core.py:238-246) on the device totals: skip iff `snp_cnt < min_count` or
// `min(ref_cnt, alt_cnt) < snp_cnt * min_maf` -- Python's int-with-float arithmetic is IEEE double on values
// < 2^53, which is what is evaluated here (one rounded multiply, no contraction).
static __global__ void k_baf_snp_filter(const unsigned long long *tot, const uint8_t *ref_i, const uint8_t *alt_i,
                                        int32_t n, double min_count, double min_maf, uint8_t *keep) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long *t = tot + (size_t)i * 5;
    const unsigned long long cnt = t[0] + t[1] + t[2] + t[3] + t[4];
    const unsigned long long minor = min(t[ref_i[i]], t[alt_i[i]]);
    const bool skip = ((double)cnt < min_count) || ((double)minor < __dmul_rn((double)cnt, min_maf));
    keep[i] = skip ? 0 : 1;
}

static int snp_filter_check(xg_ctx *ctx, const xg_snps *snps, const xg_snp_filter *filt, const char *fn) {
    if (!ctx || !ctx->stream) return ctx ? ctx->fail(XG_E_CUDA, "context has no device") : XG_E_ARG;
    if (!snps || !filt || !filt->ref_idx || !filt->alt_idx) return ctx->fail(XG_E_ARG, std::string(fn) + ": null argument");
    for (int32_t i = 0; i < snps->n; i++)
        if (filt->ref_idx[i] > 4 || filt->alt_idx[i] > 4)
            return ctx->fail(XG_E_ARG, std::string(fn) + ": allele index out of range");
    return XG_OK;
}

// plp_snp's filter on the totals the last xg_baf_pileup left on the device -> d_keep (scratch "bf_keep"), and the
// allele indices on the device (scratch "bf_ref_i" / "bf_alt_i"); keep_out (may be NULL) receives the filter
static int snp_filter_launch(xg_ctx *ctx, const xg_snps *snps, const xg_snp_filter *filt, uint8_t *keep_out,
                             const uint8_t **d_keep_out, const uint8_t **d_ref, const uint8_t **d_alt, const char *fn) {
    uint8_t *d_keep = (uint8_t *)ctx->get("bf_keep", (size_t)snps->n + 16);
    if (!d_keep || upload_arr(ctx, filt->ref_idx, (size_t)snps->n, "bf_ref_i", d_ref) ||
        upload_arr(ctx, filt->alt_idx, (size_t)snps->n, "bf_alt_i", d_alt))
        return ctx->fail(XG_E_CUDA, std::string(fn) + ": out of device memory");
    if (snps->n > 0)
        k_baf_snp_filter<<<(snps->n + 255) / 256, 256, 0, ctx->stream>>>(
            (const unsigned long long *)ctx->scratch["bf_totals"].p, *d_ref, *d_alt, snps->n, filt->min_count, filt->min_maf,
            d_keep);
    if (keep_out && snps->n > 0)          // pageable destination: the copy has landed when the call returns
        cudaMemcpyAsync(keep_out, d_keep, (size_t)snps->n, cudaMemcpyDeviceToHost, ctx->stream);
    *d_keep_out = d_keep;
    return XG_OK;
}

extern "C" int xg_baf_fc(xg_ctx *ctx, const xg_dreads *rd, const xg_snps *snps, const xg_barcodes *cells,
                         const xg_params *par, const xg_snp_filter *filt, int32_t n_regions, const int64_t *reg_ptr,
                         const int32_t *reg_snp, const uint8_t *hap_of, int32_t no_dup_hap, int64_t *totals,
                         uint8_t *keep_out, xg_coo **ad, xg_coo **dp, xg_coo **oth) {
    int rc = snp_filter_check(ctx, snps, filt, "xg_baf_fc");
    if (rc) return rc;
    const auto t_call = std::chrono::steady_clock::now();
    auto ms_since = [](std::chrono::steady_clock::time_point a) {
        return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - a).count();
    };
    xg_baf_state *st = nullptr;
    XG_CUDA(cudaSetDevice(ctx->device));
    cudaEventRecord(ctx->ev[6], ctx->stream);
    rc = xg_baf_pileup(ctx, rd, snps, cells, par, totals, &st);
    if (rc) return rc;
    double tp[16];
    for (int k = 0; k < 16; k++) tp[k] = ctx->timing[k];
    const double ms_pileup = ms_since(t_call);
    const uint8_t *d_ref = nullptr, *d_alt = nullptr, *d_keep = nullptr;
    if ((rc = snp_filter_launch(ctx, snps, filt, keep_out, &d_keep, &d_ref, &d_alt, "xg_baf_fc"))) {
        xg_baf_state_free(ctx, st);
        return rc;
    }
    rc = baf_count_impl(ctx, st, n_regions, reg_ptr, reg_snp, hap_of, nullptr, d_keep, no_dup_hap, ad, dp, oth);
    xg_baf_state_free(ctx, st);
    if (rc) return rc;
    // timing of the fused call: device ms and launches of both halves; [8] / [9] / [10] = host ms at the end of the
    // pileup / when the count kernels were queued / at the end
    const double tc9 = ctx->timing[9];
    ctx->timing[7] = ctx->timing[6];            // (region, cell, UMI) candidates
    ctx->timing[6] = tp[6];                     // (read, SNP) pairs
    if (totals) {
        ctx->timing[0] += tp[0];
        ctx->timing[1] = tp[1];
    } else {                                    // the pileup did not wait: its events have passed by now
        float t_all = 0, t_scan = 0;
        cudaEventElapsedTime(&t_all, ctx->ev[6], ctx->ev[3]);
        cudaEventElapsedTime(&t_scan, ctx->ev[1], ctx->ev[2]);
        ctx->timing[0] = t_all;
        ctx->timing[1] = t_scan;
    }
    ctx->timing[2] += tp[2] + 1;
    ctx->timing[4] += tp[4];
    ctx->timing[8] = ms_pileup;
    ctx->timing[9] = ms_pileup + tc9;
    ctx->timing[10] = ms_since(t_call);
    return XG_OK;
}

// ---- SNP-level counting (xg_snp_pileup): the winners of the pileup reduced straight into SNP x cell AD / DP / OTH.
// One SNP is a region of one SNP with GT 0|1 (baf/fc/core.py:143-194 with ref_idx 0, alt_idx 1): a winning UMI whose
// allele is not None is ALT (its base is the SNP's ALT; checked first, so REF == ALT counts as ALT), REF, or OTH.
// AD = ALT UMIs, DP = REF + ALT UMIs, OTH = the others; no_dup_hap cannot matter, a UMI has one allele at one SNP.
#define SNP_WARP_MAX 128      // a SNP with at most this many winners is reduced by one warp, more by the whole CTA
#define SNP_HIST_COLS 4096    // cells per column range of the CTA path's shared-memory histograms
#define SNP_BATCH 8           // SNPs a CTA takes from the work counter at a time: one per warp

namespace {

enum { CLS_REF = 0, CLS_ALT = 1, CLS_OTH = 2 };

// winners of kept SNPs with an allele: one count per SNP
__global__ void k_snp_hist(int64_t n, const uint32_t *pr_snp, const uint32_t *pr_colal, const uint8_t *keep,
                           int32_t *cnt) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const uint32_t ca = pr_colal[p], snp = pr_snp[p];
    if (!(ca & 0x80000000u) || ((ca >> 24) & 7u) == CODE_NONE || !keep[snp]) return;
    atomicAdd(&cnt[snp], 1);
}

// the same winners, one word each (col << 2 | class) in their SNP's segment [off[snp], off[snp + 1])
__global__ void k_snp_scatter(int64_t n, const uint32_t *pr_snp, const uint32_t *pr_colal, const uint8_t *keep,
                              const uint8_t *ref_i, const uint8_t *alt_i, const int64_t *off, int32_t *cur,
                              uint32_t *words) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const uint32_t ca = pr_colal[p], snp = pr_snp[p], code = (ca >> 24) & 7u;
    if (!(ca & 0x80000000u) || code == CODE_NONE || !keep[snp]) return;
    const uint32_t cls = code == alt_i[snp] ? CLS_ALT : code == ref_i[snp] ? CLS_REF : CLS_OTH;
    words[off[snp] + atomicAdd(&cur[snp], 1)] = (ca & 0xFFFFFFu) << 2 | cls;
}

__device__ __forceinline__ void snp_emit(int wh, int32_t v, uint32_t col, int64_t o, int32_t *st_col, int32_t *st_val,
                                         int64_t st_stride) {
    st_col[(size_t)wh * st_stride + o] = (int32_t)col;
    st_val[(size_t)wh * st_stride + o] = v;
}

// Rows of the SNPs, in column order.  A SNP's rows go to the staging areas at its own word segment (a row has at most
// as many entries as the SNP has winners), so no cursor is needed: seg_base = off[snp] in all three matrices.
//   warp path (n <= SNP_WARP_MAX): the words are rank-sorted in shared memory; the first word of a column run counts
//     the run's classes and emits the column's entries, placed by ballots;
//   CTA path: three histograms (REF / ALT / OTH) over a range of SNP_HIST_COLS cells + a bitmap of touched cells,
//     one range after another; the set bits walked in order give the entries (as k_baf_finalize).
__global__ void __launch_bounds__(256) k_snp_finalize(const int64_t *off, const uint32_t *words, int32_t n_snps,
                                                      int32_t n_cols, int32_t hist_cols, unsigned int *work,
                                                      unsigned long long *paths /* [2] */, int64_t *seg_base,
                                                      int32_t *seg_nnz, int32_t *st_col, int32_t *st_val,
                                                      int64_t st_stride) {
    extern __shared__ uint32_t smem[];
    uint32_t *hist = smem;                                   // [3][hist_cols]
    uint32_t *bitmap = smem + 3 * (size_t)hist_cols;         // (hist_cols + 31) / 32
    __shared__ uint32_t s_words[SNP_BATCH][2 * SNP_WARP_MAX];
    __shared__ int warp_tot[3][8];
    __shared__ int s_first;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const unsigned lt = (1u << lane) - 1u;
    const int nwm = (hist_cols + 31) >> 5;
    for (int c = threadIdx.x; c < 3 * hist_cols; c += blockDim.x) hist[c] = 0;
    for (int c = threadIdx.x; c < nwm; c += blockDim.x) bitmap[c] = 0;
    unsigned long long n_warp = 0, n_cta = 0;
    while (true) {
        __syncthreads();
        if (threadIdx.x == 0) s_first = (int)atomicAdd(work, (unsigned)SNP_BATCH);
        __syncthreads();
        const int first = s_first;
        if (first >= n_snps) break;
        // ---- warp path: SNP first + w
        const int s = first + w;
        if (s < n_snps) {
            const int64_t beg = off[s];
            const int n = (int)min(off[s + 1] - beg, (int64_t)SNP_WARP_MAX + 1);
            if (n > 0 && n <= SNP_WARP_MAX) {
                uint32_t *sw = s_words[w], *ss = sw + SNP_WARP_MAX;
                for (int i = lane; i < n; i += 32) sw[i] = words[beg + i];
                __syncwarp();
                for (int i = lane; i < n; i += 32) {             // rank sort; equal words keep their order
                    const uint32_t x = sw[i];
                    int r = 0;
                    for (int j = 0; j < n; j++) {
                        const uint32_t y = sw[j];
                        r += (y < x) || (y == x && j < i);
                    }
                    ss[r] = x;
                }
                __syncwarp();
                int o[3] = {0, 0, 0};
                for (int i0 = 0; i0 < n; i0 += 32) {
                    const int i = i0 + lane;
                    const uint32_t col = i < n ? ss[i] >> 2 : 0u;
                    const bool start = i < n && (i == 0 || (ss[i - 1] >> 2) != col);
                    int cr = 0, ca = 0, co = 0;
                    if (start)
                        for (int j = i; j < n && (ss[j] >> 2) == col; j++) {
                            const uint32_t cls = ss[j] & 3u;
                            cr += cls == CLS_REF;
                            ca += cls == CLS_ALT;
                            co += cls == CLS_OTH;
                        }
                    const int v[3] = {ca, cr + ca, co};                  // AD, DP, OTH
#pragma unroll
                    for (int wh = 0; wh < 3; wh++) {
                        const unsigned m = __ballot_sync(0xffffffffu, v[wh] > 0);
                        if (v[wh] > 0) snp_emit(wh, v[wh], col, beg + o[wh] + __popc(m & lt), st_col, st_val, st_stride);
                        o[wh] += __popc(m);
                    }
                }
                if (lane == 0) {
#pragma unroll
                    for (int wh = 0; wh < 3; wh++) {
                        seg_base[(size_t)wh * n_snps + s] = beg;
                        seg_nnz[(size_t)wh * n_snps + s] = o[wh];
                    }
                    n_warp++;
                }
            }
        }
        // ---- CTA path: the batch's SNPs with more winners, one after the other (the test is uniform over the CTA)
        for (int k = 0; k < SNP_BATCH && first + k < n_snps; k++) {
            const int sc = first + k;
            const int64_t beg = off[sc], n = off[sc + 1] - beg;
            if (n <= SNP_WARP_MAX) continue;
            int o[3] = {0, 0, 0};
            for (int c_lo = 0; c_lo < n_cols; c_lo += hist_cols) {
                const int nc = min(hist_cols, n_cols - c_lo), nw = (nc + 31) >> 5;
                for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
                    const uint32_t x = words[beg + i], col = (x >> 2) - (uint32_t)c_lo;
                    if (col >= (uint32_t)nc) continue;
                    atomicAdd(&hist[(x & 3u) * hist_cols + col], 1u);
                    atomicOr(&bitmap[col >> 5], 1u << (col & 31));
                }
                __syncthreads();
                for (int k0 = 0; k0 < nw; k0 += blockDim.x) {          // ordered walk over the bitmap
                    const int kw = k0 + threadIdx.x;
                    const uint32_t bits = kw < nw ? bitmap[kw] : 0u;
                    int cnt[3] = {0, 0, 0};
                    for (uint32_t bb = bits; bb; bb &= bb - 1) {
                        const int c = (kw << 5) + __ffs(bb) - 1;
                        const uint32_t r = hist[CLS_REF * hist_cols + c], a = hist[CLS_ALT * hist_cols + c];
                        cnt[0] += a != 0;
                        cnt[1] += (r + a) != 0;
                        cnt[2] += hist[CLS_OTH * hist_cols + c] != 0;
                    }
                    int incl[3], before[3] = {0, 0, 0}, tot[3] = {0, 0, 0};
#pragma unroll
                    for (int wh = 0; wh < 3; wh++) {
                        incl[wh] = cnt[wh];
                        for (int d = 1; d < 32; d <<= 1) {
                            const int y = __shfl_up_sync(0xffffffffu, incl[wh], d);
                            if (lane >= d) incl[wh] += y;
                        }
                        if (lane == 31) warp_tot[wh][w] = incl[wh];
                    }
                    __syncthreads();
#pragma unroll
                    for (int wh = 0; wh < 3; wh++)
                        for (int q = 0; q < 8; q++) {
                            const int x = warp_tot[wh][q];
                            if (q < w) before[wh] += x;
                            tot[wh] += x;
                        }
                    int64_t e[3];
#pragma unroll
                    for (int wh = 0; wh < 3; wh++) e[wh] = beg + o[wh] + before[wh] + (incl[wh] - cnt[wh]);
                    for (uint32_t bb = bits; bb; bb &= bb - 1) {
                        const int c = (kw << 5) + __ffs(bb) - 1;
                        const uint32_t r = hist[CLS_REF * hist_cols + c], a = hist[CLS_ALT * hist_cols + c],
                                       t = hist[CLS_OTH * hist_cols + c], col = (uint32_t)(c_lo + c);
                        if (a) snp_emit(0, (int32_t)a, col, e[0]++, st_col, st_val, st_stride);
                        if (r + a) snp_emit(1, (int32_t)(r + a), col, e[1]++, st_col, st_val, st_stride);
                        if (t) snp_emit(2, (int32_t)t, col, e[2]++, st_col, st_val, st_stride);
                    }
#pragma unroll
                    for (int wh = 0; wh < 3; wh++) o[wh] += tot[wh];
                    __syncthreads();                          // warp_tot is rewritten by the next chunk
                }
                for (int kw = threadIdx.x; kw < nw; kw += blockDim.x) {   // clear what this range touched
                    for (uint32_t bb = bitmap[kw]; bb; bb &= bb - 1) {
                        const int c = (kw << 5) + __ffs(bb) - 1;
                        hist[c] = 0;
                        hist[hist_cols + c] = 0;
                        hist[2 * hist_cols + c] = 0;
                    }
                    bitmap[kw] = 0;
                }
                __syncthreads();
            }
            if (threadIdx.x == 0) {
#pragma unroll
                for (int wh = 0; wh < 3; wh++) {
                    seg_base[(size_t)wh * n_snps + sc] = beg;
                    seg_nnz[(size_t)wh * n_snps + sc] = o[wh];
                }
                n_cta++;
            }
        }
    }
    if (n_warp) atomicAdd(&paths[0], n_warp);
    if (n_cta) atomicAdd(&paths[1], n_cta);
}

}  // namespace

extern "C" int xg_snp_pileup(xg_ctx *ctx, const xg_dreads *rd, const xg_snps *snps, const xg_barcodes *cells,
                             const xg_params *par, const xg_snp_filter *filt, int64_t *totals, uint8_t *keep_out,
                             xg_coo **ad, xg_coo **dp, xg_coo **oth) {
    int rc = snp_filter_check(ctx, snps, filt, "xg_snp_pileup");
    if (rc) return rc;
    if (!ad || !dp || !oth) return ctx->fail(XG_E_ARG, "xg_snp_pileup: null argument");
    if (cells && cells->n_samples >= (1 << 24))       // col << 2 | class must fit 32 bits
        return ctx->fail(XG_E_LIMIT, "xg_snp_pileup: more than 2^24 columns");
    const auto t_call = std::chrono::steady_clock::now();
    auto ms_since = [](std::chrono::steady_clock::time_point a) {
        return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - a).count();
    };
    xg_baf_state *st = nullptr;
    XG_CUDA(cudaSetDevice(ctx->device));
    cudaEventRecord(ctx->ev[6], ctx->stream);
    if ((rc = xg_baf_pileup(ctx, rd, snps, cells, par, totals, &st))) return rc;
    const double tp2 = ctx->timing[2], ms_pileup = ms_since(t_call);
    const int64_t n_pairs = st->n_pairs;
    const int32_t n_snps = snps->n, n_cols = st->n_cols;
    const uint8_t *d_ref = nullptr, *d_alt = nullptr, *d_keep = nullptr;
    // one free of the state on every path out; the scratch buffers below do not depend on it
    struct StateGuard {
        xg_ctx *c;
        xg_baf_state *s;
        ~StateGuard() { xg_baf_state_free(c, s); }
    } guard{ctx, st};
    if ((rc = snp_filter_launch(ctx, snps, filt, keep_out, &d_keep, &d_ref, &d_alt, "xg_snp_pileup"))) return rc;
    int launches = 1;
    // capacities: the winners of one SNP never exceed the batch's pairs (< 2^31, checked by the pileup)
    const size_t cap = (size_t)n_pairs + 1;
    XG_GET(cnt, int32_t, "sp_cnt", (size_t)n_snps + 1);
    XG_GET(cur, int32_t, "sp_cur", (size_t)n_snps + 1);
    XG_GET(off, int64_t, "sp_off", (size_t)n_snps + 2);
    XG_GET(words, uint32_t, "sp_words", cap);
    XG_GET(work, unsigned int, "sp_work", 4);
    XG_GET(paths, unsigned long long, "sp_paths", 2);
    XG_GET(seg_base, int64_t, "sp_seg_base", 3 * (size_t)n_snps + 1);
    XG_GET(seg_nnz, int32_t, "sp_seg_nnz", 3 * (size_t)n_snps + 1);
    XG_GET(st_col, int32_t, "sp_st_col", 3 * cap);
    XG_GET(st_val, int32_t, "sp_st_val", 3 * cap);
    XG_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int32_t) * ((size_t)n_snps + 1), ctx->stream));
    XG_CUDA(cudaMemsetAsync(cur, 0, sizeof(int32_t) * ((size_t)n_snps + 1), ctx->stream));
    XG_CUDA(cudaMemsetAsync(work, 0, 16, ctx->stream));
    XG_CUDA(cudaMemsetAsync(paths, 0, 16, ctx->stream));
    XG_CUDA(cudaMemsetAsync(seg_base, 0, sizeof(int64_t) * (3 * (size_t)n_snps + 1), ctx->stream));
    XG_CUDA(cudaMemsetAsync(seg_nnz, 0, sizeof(int32_t) * (3 * (size_t)n_snps + 1), ctx->stream));
    const unsigned grid = (unsigned)((n_pairs + 255) / 256);
    if (n_pairs > 0) {
        k_snp_hist<<<grid, 256, 0, ctx->stream>>>(n_pairs, st->pr_snp, st->pr_colal, d_keep, cnt);
        launches++;
    }
    k_exclusive_scan<<<1, 1024, 0, ctx->stream>>>(cnt, off, n_snps);
    launches++;
    if (n_pairs > 0 && n_snps > 0) {
        k_snp_scatter<<<grid, 256, 0, ctx->stream>>>(n_pairs, st->pr_snp, st->pr_colal, d_keep, d_ref, d_alt, off, cur,
                                                     words);
        const int32_t hist_cols = std::min(n_cols, SNP_HIST_COLS);
        const size_t smem = (size_t)hist_cols * 12 + (size_t)((hist_cols + 31) / 32) * 4;
        XG_CUDA(cudaFuncSetAttribute(k_snp_finalize, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const int per_sm = std::max(1, std::min(8, (int)(200 * 1024 / (smem + 8 * 1024 + 1024))));
        const int n_batches = (n_snps + SNP_BATCH - 1) / SNP_BATCH;
        k_snp_finalize<<<std::min(n_batches, 148 * per_sm), 256, smem, ctx->stream>>>(
            off, words, n_snps, n_cols, hist_cols, work, paths, seg_base, seg_nnz, st_col, st_val, (int64_t)cap);
        launches += 2;
    }
    XG_CUDA(cudaGetLastError());
    const double ms_kernels = ms_since(t_call);
    xg_coo **outs[3] = {ad, dp, oth};
    if ((rc = xg_staging_to_coo3(ctx, "sp3", n_snps, n_cols, seg_base, seg_nnz, st_col, st_val, (int64_t)cap, outs,
                                 &launches)))
        return rc;
    // the stream is idle now: the winner count and the path counters cost one short copy
    long long stats[3] = {0, 0, 0};
    XG_CUDA(cudaMemcpyAsync(&stats[0], off + n_snps, 8, cudaMemcpyDeviceToHost, ctx->stream));
    XG_CUDA(cudaMemcpyAsync(&stats[1], paths, 16, cudaMemcpyDeviceToHost, ctx->stream));
    XG_CUDA(cudaStreamSynchronize(ctx->stream));
    float t_all = 0, t_scan = 0;
    cudaEventElapsedTime(&t_all, ctx->ev[6], ctx->ev[3]);
    cudaEventElapsedTime(&t_scan, ctx->ev[1], ctx->ev[2]);
    const double t_d2h = ctx->timing[4];       // the pileup's totals (if copied out) + the results
    for (double &t : ctx->timing) t = 0;
    ctx->timing[0] = t_all;
    ctx->timing[1] = t_scan;
    ctx->timing[2] = tp2 + launches;
    ctx->timing[4] = t_d2h;
    ctx->timing[6] = (double)n_pairs;
    ctx->timing[7] = (double)stats[0];
    ctx->timing[8] = ms_pileup;
    ctx->timing[9] = ms_kernels;
    ctx->timing[10] = ms_since(t_call);
    ctx->timing[14] = (double)stats[1];
    ctx->timing[15] = (double)stats[2];
    return XG_OK;
}
