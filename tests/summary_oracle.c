/* summary_oracle.c -- CPU oracle of basefc's read-assignment summary (xg_basefc_summary).  TEST INFRASTRUCTURE ONLY.
 *
 * The contract restated record by record, with a brute-force loop over the features of the record's contig (no
 * interval index): a record is in range iff some feature that fetch() would query (gid >= 0, beg >= 0, end > beg)
 * satisfies pos < end && bam_endpos > beg.  Row: the listed column of its cell key, else n_samples (__no_cell); in
 * sample-ID mode the BAM's column.  Fate, in check_read's order (rdr/fc/core.py:46-62): 0 mapq, 1 flags / orphan,
 * 2 UMI tag missing or empty (when UMIs are counted), 3 len(read.positions) < min_len, then the include test of
 * rdr/fc/core.py:160-165 with the reference's float expression (m / float(n) < min_include, as orc_basefc evaluates
 * it; not the device's integer table) for every overlapping feature: 4 none passes, 5 one, 6 two or more.
 * The helpers of the basefc oracle (barcode dict, read.positions) are used as they are by including it.
 */
#include "../oracle/xg_oracle.c"

#define ORC_FATES 7

/* own: NULL or {gid_lo, pos_lo, gid_hi, pos_hi}: only records whose (gid, pos) lies in [lo, hi) count.
 * out: (n_samples + 1) x ORC_FATES counters, zeroed here. */
int orc_basefc_summary(const xg_reads *r, int32_t n_feat, const int32_t *gid, const int32_t *beg, const int32_t *end,
                       int32_t n_bc, const uint64_t *bc_keys, int32_t n_samples, const orc_params *c,
                       const int32_t *own, int32_t n_threads, int64_t *out) {
    const size_t n_out = ((size_t)n_samples + 1) * ORC_FATES;
    memset(out, 0, n_out * sizeof(int64_t));
    bc_dict bc;
    memset(&bc, 0, sizeof(bc));
    if (c->use_cell_tag && bc_build(&bc, n_bc, bc_keys)) return -1;
    /* the fetchable features of every contig, in input order */
    int32_t n_gid = 0;
    for (int32_t ri = 0; ri < r->n_runs; ri++)
        if (r->runs[ri].gid + 1 > n_gid) n_gid = r->runs[ri].gid + 1;
    int32_t *goff = (int32_t *)calloc((size_t)n_gid + 1, 4);
    int32_t *feat = (int32_t *)malloc((size_t)(n_feat > 0 ? n_feat : 1) * 4);
    if (!goff || !feat) return -1;
    for (int32_t f = 0; f < n_feat; f++)
        if (gid[f] >= 0 && gid[f] < n_gid && beg[f] >= 0 && end[f] > beg[f]) goff[gid[f] + 1]++;
    for (int32_t g = 0; g < n_gid; g++) goff[g + 1] += goff[g];
    {
        int32_t *cur = (int32_t *)malloc(((size_t)n_gid + 1) * 4);
        if (!cur) return -1;
        memcpy(cur, goff, ((size_t)n_gid + 1) * 4);
        for (int32_t f = 0; f < n_feat; f++)
            if (gid[f] >= 0 && gid[f] < n_gid && beg[f] >= 0 && end[f] > beg[f]) feat[cur[gid[f]]++] = f;
        free(cur);
    }
    int err = 0;
    (void)n_threads;
#ifdef _OPENMP
#pragma omp parallel num_threads(n_threads > 0 ? n_threads : 1)
#endif
    {
        int64_t *mine = (int64_t *)calloc(n_out, sizeof(int64_t));
        int32_t *posbuf = NULL, poscap = 0;
        if (!mine) err = 1;
        for (int32_t ri = 0; ri < r->n_runs; ri++) {  /* every thread meets every worksharing loop */
            const xg_run *run = &r->runs[ri];
            const int32_t g = run->gid;
            if (g < 0) continue;
#ifdef _OPENMP
#pragma omp for schedule(dynamic, 4096)
#endif
            for (int64_t i = run->rec_beg; i < run->rec_end; i++) {
                const int32_t pos = r->pos_end[2 * i], rend = r->pos_end[2 * i + 1];
                if (own && (g < own[0] || (g == own[0] && pos < own[1]) || g > own[2] || (g == own[2] && pos >= own[3])))
                    continue;
                int in_range = 0;
                for (int32_t k = goff[g]; k < goff[g + 1] && !in_range; k++)
                    in_range = pos < end[feat[k]] && rend > beg[feat[k]];
                if (!in_range) continue;
                int32_t row = run->bam_idx;
                if (c->use_cell_tag) {
                    const uint64_t ck = r->keys[2 * i];
                    const int32_t col = ck == XG_KEY_NONE ? -1 : bc_get(&bc, ck);
                    row = col < 0 ? n_samples : col;
                }
                const uint32_t flag = rd_flag(r, i);
                const uint64_t umi = r->keys[2 * i + 1];
                int fate;
                if ((double)rd_mapq(r, i) < c->min_mapq) {
                    fate = 0;
                } else if ((c->excl_flag && (flag & c->excl_flag)) || (c->incl_flag && !(flag & c->incl_flag)) ||
                           (c->no_orphan && (flag & 1u) && !(flag & 2u))) {
                    fate = 1;
                } else if (c->need_umi_tag && (umi == XG_KEY_NONE || umi == XG_KEY_EMPTY)) {
                    fate = 2;
                } else {
                    const int32_t n = rd_positions(r, i, &posbuf, &poscap);
                    if (n < c->min_len) {
                        fate = 3;
                    } else {
                        int n_pass = 0;
                        for (int32_t k = goff[g]; k < goff[g + 1]; k++) {
                            const int32_t f = feat[k];
                            if (!(pos < end[f] && rend > beg[f])) continue;
                            const int32_t s = beg[f], e = end[f] - 1;
                            int32_t m = 0;
                            for (int32_t q = 0; q < n; q++) m += s <= posbuf[q] && posbuf[q] <= e;
                            int pass;
                            if (0 < c->min_include && c->min_include < 1)
                                pass = n > 0 && !((double)m / (double)n < c->min_include);
                            else
                                pass = !((double)m < c->min_include);
                            n_pass += pass;
                        }
                        fate = 4 + (n_pass > 2 ? 2 : n_pass);
                    }
                }
                if (mine) mine[(size_t)row * ORC_FATES + (size_t)fate]++;
            }
        }
#ifdef _OPENMP
#pragma omp critical
#endif
        {
            if (mine)
                for (size_t k = 0; k < n_out; k++) out[k] += mine[k];
        }
        free(mine);
        free(posbuf);
    }
    free(goff);
    free(feat);
    free(bc.keys);
    free(bc.cols);
    return err ? -1 : 0;
}
