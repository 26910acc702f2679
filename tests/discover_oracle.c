/* discover_oracle.c -- CPU oracle of SNP discovery (xg_snp_discover).  TEST INFRASTRUCTURE ONLY.
 *
 * A brute force over every target position that some read's [pos, end) covers: at each such position p it runs
 * plp_snp (xcltk/baf/fc/core.py:198-247) exactly as orc_baf does -- check_read, listed cell (or the BAM's column),
 * a UMI key, the first read per (cell, UMI) in file order wins even when its allele is None, winners with an allele
 * count into base_idx buckets -- and then the allele inference and the filter of the discovery contract:
 * REF = the A..T bucket with the largest count, ALT = the second largest (ties to the lower index; N never),
 * kept iff ALT >= 1, sum >= min_count and ALT >= sum * min_maf (double compares).  It does NOT use the GPU's raw
 * pre-filter: the device's pruning is tested against this, not restated in it.
 *
 * The helpers of the baf oracle (check_read_head, the barcode dict, fetch_begin, base_idx, SEQ_NT16) are used as
 * they are by including oracle/xg_oracle.c.  The allele of a read at p is read_allele's (the idx-th M/=/X base,
 * query positions advanced by S and I), found with a CIGAR cursor that moves with p instead of rebuilding
 * read.positions at every position, so that a library of a few million reads is checked in seconds.
 */
#include "../oracle/xg_oracle.c"

typedef struct {
    int64_t n, cap;
    int32_t *gid, *pos;
    uint8_t *ref, *alt;
    int64_t *tot;
} orc_sites;

void orc_sites_free(orc_sites *s) {
    free(s->gid);
    free(s->pos);
    free(s->ref);
    free(s->alt);
    free(s->tot);
    memset(s, 0, sizeof(*s));
}

static int sites_push(orc_sites *s, int32_t g, int32_t p, int r, int a, const int64_t *tc) {
    if (s->n == s->cap) {
        int64_t nc = s->cap ? s->cap * 2 : 256;
        int32_t *g2 = (int32_t *)realloc(s->gid, (size_t)nc * 4);
        if (g2) s->gid = g2;
        int32_t *p2 = (int32_t *)realloc(s->pos, (size_t)nc * 4);
        if (p2) s->pos = p2;
        uint8_t *r2 = (uint8_t *)realloc(s->ref, (size_t)nc);
        if (r2) s->ref = r2;
        uint8_t *a2 = (uint8_t *)realloc(s->alt, (size_t)nc);
        if (a2) s->alt = a2;
        int64_t *t2 = (int64_t *)realloc(s->tot, (size_t)nc * 40);
        if (t2) s->tot = t2;
        if (!g2 || !p2 || !r2 || !a2 || !t2) return -1;
        s->cap = nc;
    }
    s->gid[s->n] = g;
    s->pos[s->n] = p;
    s->ref[s->n] = (uint8_t)r;
    s->alt[s->n] = (uint8_t)a;
    memcpy(s->tot + s->n * 5, tc, 40);
    s->n++;
    return 0;
}

/* a passing read that covers the current position, with its CIGAR cursor */
typedef struct {
    int64_t i;
    int32_t rend, col;
    uint64_t umi;
    const uint32_t *w;      /* NULL: one M op of length rend - pos (a "simple" record) */
    uint32_t one, nops, k;
    int32_t rp, qp;         /* reference / query position at the start of op k */
} act_t;

static uint32_t act_op(const act_t *a, uint32_t k) { return a->w ? a->w[k] : a->one; }

/* read_allele(): the base letter at p, or 0 for None; p never decreases between calls */
static char act_allele(const xg_reads *r, act_t *a, int32_t p) {
    while (a->k < a->nops) {
        uint32_t w = act_op(a, a->k), op = w & 15u;
        int32_t l = (int32_t)(w >> 4);
        if (op == 0 || op == 7 || op == 8) {
            if (p < a->rp + l) break;
            a->rp += l;
            a->qp += l;
        } else if (op == 2 || op == 3) {
            if (p < a->rp + l) break;
            a->rp += l;
        } else if (op == 1 || op == 4) {
            a->qp += l;
        }
        a->k++;
    }
    if (a->k >= a->nops) return 0;
    uint32_t op = act_op(a, a->k) & 15u;
    if (!(op == 0 || op == 7 || op == 8) || p < a->rp) return 0;
    if (r->seq_off[a->i] == 0xFFFFFFFFu) return 0;
    int32_t qi = a->qp + (p - a->rp);
    const uint8_t *seq = (const uint8_t *)(r->seq + r->seq_off[a->i]);
    uint8_t b = seq[qi >> 1];
    return SEQ_NT16[(qi & 1) ? (b & 15) : (b >> 4)];
}

/* (cell, UMI) set of one position: slots are valid while their stamp equals the position's epoch */
typedef struct {
    uint64_t *key;
    int32_t *cell;
    uint32_t *stamp;
    uint32_t cap, n, epoch;
} umiset;

static int us_init(umiset *u, uint32_t cap) {
    u->key = (uint64_t *)malloc((size_t)cap * 8);
    u->cell = (int32_t *)malloc((size_t)cap * 4);
    u->stamp = (uint32_t *)calloc(cap, 4);
    u->cap = cap;
    u->n = 0;
    u->epoch = 1;
    return (u->key && u->cell && u->stamp) ? 0 : -1;
}
static void us_free(umiset *u) {
    free(u->key);
    free(u->cell);
    free(u->stamp);
}
static void us_next(umiset *u) {
    u->n = 0;
    if (++u->epoch == 0) {
        memset(u->stamp, 0, (size_t)u->cap * 4);
        u->epoch = 1;
    }
}
/* 1 if (cell, key) was not in the set (and is now) */
static int us_insert(umiset *u, int32_t cell, uint64_t key) {
    if ((uint64_t)(u->n + 1) * 2 > u->cap) {      /* grow: keep this epoch's entries */
        umiset o = *u;
        if (us_init(u, o.cap * 2)) return -1;
        u->epoch = 1;
        for (uint32_t s = 0; s < o.cap; s++)
            if (o.stamp[s] == o.epoch) us_insert(u, o.cell[s], o.key[s]);
        us_free(&o);
    }
    uint32_t s = (uint32_t)hash64(key ^ ((uint64_t)(uint32_t)cell << 40)) & (u->cap - 1);
    while (u->stamp[s] == u->epoch) {
        if (u->cell[s] == cell && u->key[s] == key) return 0;
        s = (s + 1) & (u->cap - 1);
    }
    u->stamp[s] = u->epoch;
    u->cell[s] = cell;
    u->key[s] = key;
    u->n++;
    return 1;
}

/* check_read + min_len + cell + UMI of orc_baf's plp_snp loop; col = the read's column */
static int read_passes(const xg_reads *r, const xg_run *run, int64_t i, const orc_params *c, const bc_dict *bc,
                       int32_t *col) {
    if (check_read_head(r, i, c) < 0) return 0;
    const uint32_t *w;
    uint32_t one, n = rd_cigar(r, i, &w, &one);
    int32_t aln = 0;
    for (uint32_t q = 0; q < n; q++) {
        uint32_t op = w[q] & 15u;
        if (op == 0 || op == 7 || op == 8) aln += (int32_t)(w[q] >> 4);
    }
    if (aln < c->min_len) return 0;
    if (c->use_cell_tag) {
        *col = bc_get(bc, r->keys[2 * i]);
        if (*col < 0) return 0;
    } else {
        *col = run->bam_idx;
    }
    uint64_t umi = r->keys[2 * i + 1];
    return umi != XG_KEY_EMPTY && umi != XG_KEY_NONE;
}

#define ORC_CHUNK 65536

/* positions [cb, ce) of contig g */
static int discover_chunk(const xg_reads *r, int32_t g, int32_t cb, int32_t ce, const orc_params *c,
                          const bc_dict *bc, double min_count, double min_maf, orc_sites *out) {
    int32_t nr = 0;
    for (int32_t k = 0; k < r->n_runs; k++) nr += r->runs[k].gid == g;
    if (!nr) return 0;
    int32_t *runs = (int32_t *)malloc((size_t)nr * 4);
    int64_t *nxt = (int64_t *)malloc((size_t)nr * 8);
    act_t **act = (act_t **)calloc((size_t)nr, sizeof(act_t *));
    int64_t *na = (int64_t *)calloc((size_t)nr, 8), *ca = (int64_t *)calloc((size_t)nr, 8);
    umiset us;
    int err = (!runs || !nxt || !act || !na || !ca || us_init(&us, 1024)) ? -1 : 0;
    nr = 0;
    for (int32_t k = 0; k < r->n_runs && !err; k++)
        if (r->runs[k].gid == g) {
            runs[nr] = k;
            nxt[nr] = fetch_begin(r, &r->runs[k], cb);
            nr++;
        }
    int32_t p = cb;
    while (!err && p < ce) {
        int64_t live = 0;
        for (int32_t k = 0; k < nr; k++) {              /* reads that start at or before p enter */
            const xg_run *run = &r->runs[runs[k]];
            for (; nxt[k] < run->rec_end && r->pos_end[2 * nxt[k]] <= p; nxt[k]++) {
                int64_t i = nxt[k];
                int32_t col;
                if (r->pos_end[2 * i + 1] <= p || !read_passes(r, run, i, c, bc, &col)) continue;
                if (na[k] == ca[k]) {
                    ca[k] = ca[k] ? ca[k] * 2 : 64;
                    act_t *x = (act_t *)realloc(act[k], (size_t)ca[k] * sizeof(act_t));
                    if (!x) {
                        err = -1;
                        break;
                    }
                    act[k] = x;
                }
                act_t *a = &act[k][na[k]++];
                a->i = i;
                a->rend = r->pos_end[2 * i + 1];
                a->col = col;
                a->umi = r->keys[2 * i + 1];
                a->nops = rd_cigar(r, i, &a->w, &a->one);
                if (a->w == &a->one) a->w = NULL;
                a->k = 0;
                a->rp = r->pos_end[2 * i];
                a->qp = 0;
            }
            live += na[k];
        }
        if (err) break;
        if (!live) {                                    /* jump to the next read's start */
            int32_t nx = ce;
            for (int32_t k = 0; k < nr; k++)
                if (nxt[k] < r->runs[runs[k]].rec_end && r->pos_end[2 * nxt[k]] < nx) nx = r->pos_end[2 * nxt[k]];
            p = nx > p ? nx : p + 1;
            continue;
        }
        us_next(&us);
        int64_t tc[5] = {0, 0, 0, 0, 0};
        for (int32_t k = 0; k < nr; k++) {              /* file order: runs in index order, records in order */
            int64_t m = 0;
            for (int64_t j = 0; j < na[k]; j++) {
                act_t *a = &act[k][j];
                if (a->rend <= p) continue;            /* left behind: removed */
                act[k][m++] = *a;
                a = &act[k][m - 1];
                int nw = us_insert(&us, a->col, a->umi);
                if (nw < 0) err = -1;
                char al = act_allele(r, a, p);
                if (nw == 1 && al) tc[base_idx(al)]++;  /* first read wins, even if None */
            }
            na[k] = m;
        }
        int ri = 0;
        for (int b = 1; b < 4; b++)
            if (tc[b] > tc[ri]) ri = b;
        int ai = ri == 0 ? 1 : 0;
        for (int b = ai + 1; b < 4; b++)
            if (b != ri && tc[b] > tc[ai]) ai = b;
        int64_t sum = tc[0] + tc[1] + tc[2] + tc[3] + tc[4];
        if (tc[ai] >= 1 && !((double)sum < min_count) && !((double)tc[ai] < (double)sum * min_maf))
            if (sites_push(out, g, p, ri, ai, tc)) err = -1;
        p++;
    }
    for (int32_t k = 0; k < nr && act; k++) free(act[k]);
    free(act);
    free(na);
    free(ca);
    free(runs);
    free(nxt);
    us_free(&us);
    return err;
}

/* targets in caller order ({gid, beg, end}; gid < 0 or end <= beg: skipped); sites in target order, then by
 * position.  Returns 0, or -1 when out of memory. */
int orc_snp_discover(const xg_reads *r, int32_t n_tg, const int32_t *tg_gid, const int32_t *tg_beg,
                     const int32_t *tg_end, int32_t n_bc, const uint64_t *bc_keys, const orc_params *c,
                     double min_count, double min_maf, int32_t n_threads, orc_sites *out) {
    memset(out, 0, sizeof(*out));
    bc_dict bc;
    memset(&bc, 0, sizeof(bc));
    if (c->use_cell_tag && bc_build(&bc, n_bc, bc_keys)) return -1;
    int64_t n_ch = 0;
    for (int32_t t = 0; t < n_tg; t++)
        if (tg_gid[t] >= 0 && tg_end[t] > tg_beg[t])
            n_ch += ((int64_t)tg_end[t] - tg_beg[t] + ORC_CHUNK - 1) / ORC_CHUNK;
    int32_t *ch_g = (int32_t *)malloc((size_t)(n_ch + 1) * 4), *ch_b = (int32_t *)malloc((size_t)(n_ch + 1) * 4),
            *ch_e = (int32_t *)malloc((size_t)(n_ch + 1) * 4);
    orc_sites *parts = (orc_sites *)calloc((size_t)n_ch + 1, sizeof(orc_sites));
    int err = (!ch_g || !ch_b || !ch_e || !parts) ? -1 : 0;
    int64_t q = 0;
    for (int32_t t = 0; t < n_tg && !err; t++) {
        if (tg_gid[t] < 0 || tg_end[t] <= tg_beg[t]) continue;
        for (int64_t b = tg_beg[t]; b < tg_end[t]; b += ORC_CHUNK) {
            ch_g[q] = tg_gid[t];
            ch_b[q] = (int32_t)b;
            ch_e[q] = (int32_t)(b + ORC_CHUNK < tg_end[t] ? b + ORC_CHUNK : tg_end[t]);
            q++;
        }
    }
    (void)n_threads;
#ifdef _OPENMP
#pragma omp parallel for schedule(dynamic, 1) num_threads(n_threads > 0 ? n_threads : 1)
#endif
    for (int64_t k = 0; k < (err ? 0 : n_ch); k++)
        if (discover_chunk(r, ch_g[k], ch_b[k], ch_e[k], c, &bc, min_count, min_maf, &parts[k])) {
#ifdef _OPENMP
#pragma omp atomic write
#endif
            err = -1;
        }
    for (int64_t k = 0; k < n_ch && !err; k++)
        for (int64_t s = 0; s < parts[k].n && !err; s++)
            if (sites_push(out, parts[k].gid[s], parts[k].pos[s], parts[k].ref[s], parts[k].alt[s],
                           parts[k].tot + s * 5))
                err = -1;
    for (int64_t k = 0; parts && k < n_ch; k++) orc_sites_free(&parts[k]);
    free(parts);
    free(ch_g);
    free(ch_b);
    free(ch_e);
    free(bc.keys);
    free(bc.cols);
    if (err) orc_sites_free(out);
    return err;
}

/* ============================== raw scan mirror ===========================================
 * orc_disc_raw: the counters the device's raw scan (k_disc_route / k_disc_hist) reports, restated per read on the
 * CPU so that a test can compare them exactly -- timing()[5] covered windows, [6] positions scanned, [13] (read,
 * window) entries, [7] raw candidates.  Separate from orc_snp_discover on purpose: that oracle defines the sites
 * without any pre-filter; this one pins what the pre-filter looks at, so that over-counting (a read routed twice,
 * a histogram left over from a CTA's previous window) and under-counting show even where no site changes.
 *
 * The contract it follows (discover.cu):
 *   a read counts   check_read's flags, a stored SEQ, a UMI key that is neither none nor empty, a listed cell in
 *                   barcode mode, aligned length >= min_len
 *   a read enters   its [pos, end) meets a live target of its contig (live: 0 <= gid < 1 + the largest gid of a
 *                   run, beg >= 0, end > beg); an unmapped read has end = pos + 1 but all its blocks are walked
 *   windows         DISC_W positions from each live target's beg, numbered in caller order; a read adds one entry
 *                   per distinct window its aligned (M / = / X) blocks touch
 *   counters        covered = windows with an entry; scanned = their lengths inside their targets; a position of a
 *                   covered window is a candidate iff raw A+C+G+T+N >= t_sum and the second largest of A..T >= t_alt,
 *                   the raw count being the entering reads with an aligned base there (code 1/2/4/8 A/C/G/T, else N)
 *   thresholds      t_sum = ceil(min_count), t_alt = max(1, ceil(min_count * min_maf)) with the product in double
 * out[4] = {covered windows, positions scanned, entries, raw candidates}.  Returns 0, -1 (out of memory) or -2
 * (overlapping live targets of one contig, or reads without sequences: the device rejects both). */
#define ORC_DISC_W 2048

static uint64_t orc_ceil_count(double v) {
    if (!(v > 0)) return 0;
    if (v >= 1e18) return 1000000000000000000ull;
    uint64_t c = (uint64_t)v;
    return (double)c < v ? c + 1 : c;
}

typedef struct {
    int32_t beg, end, win0;
} orc_tg;

static int orc_tg_cmp(const void *a, const void *b) {
    const orc_tg *x = (const orc_tg *)a, *y = (const orc_tg *)b;
    return x->beg < y->beg ? -1 : x->beg > y->beg;
}

int orc_disc_raw(const xg_reads *r, int32_t n_tg, const int32_t *tg_gid, const int32_t *tg_beg, const int32_t *tg_end,
                 int32_t n_bc, const uint64_t *bc_keys, const orc_params *c, double min_count, double min_maf,
                 int64_t *out) {
    memset(out, 0, 4 * sizeof(int64_t));
    if (!r->seq_off || !r->seq) return -2;
    int32_t n_gid = 0;
    for (int32_t k = 0; k < r->n_runs; k++)
        if (r->runs[k].gid + 1 > n_gid) n_gid = r->runs[k].gid + 1;
    /* live targets: windows in caller order, then per contig sorted by beg */
    int64_t n_win = 0;
    int32_t *cnt = (int32_t *)calloc((size_t)n_gid + 1, 4);
    orc_tg *all = (orc_tg *)malloc(((size_t)n_tg + 1) * sizeof(orc_tg));
    int32_t *gof = (int32_t *)calloc((size_t)n_gid + 2, 4);
    if (!cnt || !all || !gof) {
        free(cnt), free(all), free(gof);
        return -1;
    }
    for (int32_t t = 0; t < n_tg; t++) {
        int32_t g = tg_gid[t], b = tg_beg[t], e = tg_end[t];
        if (!(g >= 0 && g < n_gid && b >= 0 && e > b)) continue;
        cnt[g]++;
        n_win += ((int64_t)e - b + ORC_DISC_W - 1) / ORC_DISC_W;
    }
    for (int32_t g = 0; g < n_gid; g++) gof[g + 1] = gof[g] + cnt[g];
    memset(cnt, 0, (size_t)n_gid * 4);
    int64_t w_at = 0;
    for (int32_t t = 0; t < n_tg; t++) {
        int32_t g = tg_gid[t], b = tg_beg[t], e = tg_end[t];
        if (!(g >= 0 && g < n_gid && b >= 0 && e > b)) continue;
        orc_tg *x = &all[gof[g] + cnt[g]++];
        x->beg = b;
        x->end = e;
        x->win0 = (int32_t)w_at;
        w_at += ((int64_t)e - b + ORC_DISC_W - 1) / ORC_DISC_W;
    }
    int err = 0;
    for (int32_t g = 0; g < n_gid; g++) {
        qsort(all + gof[g], (size_t)(gof[g + 1] - gof[g]), sizeof(orc_tg), orc_tg_cmp);
        for (int32_t k = gof[g] + 1; k < gof[g + 1]; k++)
            if (all[k - 1].end > all[k].beg) err = -2;
    }
    int64_t *entries = (int64_t *)calloc((size_t)n_win + 1, 8);
    uint32_t **hist = (uint32_t **)calloc((size_t)n_win + 1, sizeof(uint32_t *));
    int32_t *wbeg = (int32_t *)malloc(((size_t)n_win + 1) * 4), *wlen = (int32_t *)malloc(((size_t)n_win + 1) * 4);
    bc_dict bc;
    memset(&bc, 0, sizeof(bc));
    if (!entries || !hist || !wbeg || !wlen || (c->use_cell_tag && bc_build(&bc, n_bc, bc_keys))) err = err ? err : -1;
    for (int32_t k = 0; k < gof[n_gid] && !err; k++)
        for (int32_t w = 0; (int64_t)all[k].beg + (int64_t)w * ORC_DISC_W < all[k].end; w++) {
            int32_t s = all[k].beg + w * ORC_DISC_W;
            wbeg[all[k].win0 + w] = s;
            wlen[all[k].win0 + w] = (all[k].end - s < ORC_DISC_W) ? all[k].end - s : ORC_DISC_W;
        }
    for (int32_t k = 0; k < r->n_runs && !err; k++) {
        const xg_run *run = &r->runs[k];
        int32_t g = run->gid;
        if (g < 0 || g >= n_gid || gof[g] == gof[g + 1]) continue;
        const orc_tg *T = all + gof[g];
        int32_t nt = gof[g + 1] - gof[g];
        for (int64_t i = run->rec_beg; i < run->rec_end && !err; i++) {
            int32_t pos = r->pos_end[2 * i], rend = r->pos_end[2 * i + 1];
            int32_t t0 = 0;
            while (t0 < nt && T[t0].end <= pos) t0++;
            if (t0 >= nt || T[t0].beg >= rend) continue;                 /* meets no live target */
            if (check_read_head(r, i, c) < 0 || r->seq_off[i] == 0xFFFFFFFFu) continue;
            uint64_t umi = r->keys[2 * i + 1];
            if (umi == XG_KEY_NONE || umi == XG_KEY_EMPTY) continue;
            if (c->use_cell_tag && bc_get(&bc, r->keys[2 * i]) < 0) continue;
            const uint32_t *wd;
            uint32_t one, nops = rd_cigar(r, i, &wd, &one);
            int32_t aln = 0;
            for (uint32_t q = 0; q < nops; q++) {
                uint32_t op = wd[q] & 15u;
                if (op == 0 || op == 7 || op == 8) aln += (int32_t)(wd[q] >> 4);
            }
            if (aln < c->min_len) continue;
            const uint8_t *seq = (const uint8_t *)(r->seq + r->seq_off[i]);
            int32_t rp = pos, qp = 0;
            int64_t last = -1;
            for (uint32_t q = 0; q < nops && !err; q++) {
                uint32_t op = wd[q] & 15u;
                int32_t l = (int32_t)(wd[q] >> 4);
                if (op == 0 || op == 7 || op == 8) {
                    for (int32_t p = rp; p < rp + l; p++) {             /* every aligned base, one at a time */
                        int32_t t = t0;
                        while (t < nt && T[t].end <= p) t++;
                        if (t >= nt || T[t].beg > p) continue;
                        int64_t w = T[t].win0 + (p - T[t].beg) / ORC_DISC_W;
                        if (w != last) {
                            entries[w]++;
                            last = w;
                        }
                        if (!hist[w] && !(hist[w] = (uint32_t *)calloc(5 * ORC_DISC_W, 4))) {
                            err = -1;
                            break;
                        }
                        int32_t qi = qp + (p - rp);
                        uint8_t b = seq[qi >> 1], nib = (qi & 1) ? (b & 15) : (b >> 4);
                        int bk = nib == 1 ? 0 : nib == 2 ? 1 : nib == 4 ? 2 : nib == 8 ? 3 : 4;
                        hist[w][bk * ORC_DISC_W + (p - wbeg[w])]++;
                    }
                    rp += l;
                    qp += l;
                } else if (op == 2 || op == 3) {
                    rp += l;
                } else if (op == 1 || op == 4) {
                    qp += l;
                }
            }
        }
    }
    uint64_t t_sum = orc_ceil_count(min_count);
    double prod = (min_count > 0 && min_maf > 0) ? min_count * min_maf : 0.0;
    uint64_t t_alt = orc_ceil_count(prod);
    if (t_alt < 1) t_alt = 1;
    for (int64_t w = 0; w < n_win && !err; w++) {
        if (!entries[w]) continue;
        out[0]++;
        out[1] += wlen[w];
        out[2] += entries[w];
        for (int32_t b = 0; b < wlen[w]; b++) {
            uint64_t v[5], sum = 0;
            for (int k = 0; k < 5; k++) sum += v[k] = hist[w][k * ORC_DISC_W + b];
            uint64_t m1 = 0, m2 = 0;                                      /* largest and second largest of A..T */
            for (int k = 0; k < 4; k++) {
                if (v[k] > m1) {
                    m2 = m1;
                    m1 = v[k];
                } else if (v[k] > m2) {
                    m2 = v[k];
                }
            }
            out[3] += sum >= t_sum && m2 >= t_alt;
        }
    }
    for (int64_t w = 0; hist && w < n_win; w++) free(hist[w]);
    free(hist);
    free(entries);
    free(wbeg);
    free(wlen);
    free(cnt);
    free(all);
    free(gof);
    free(bc.keys);
    free(bc.cols);
    return err;
}
