// discover.cu -- SNP discovery: heterozygous sites called from the reads themselves when no candidate list is given
// (cellsnp-lite's second mode; no counterpart in the reference, whose plp_snp pileup defines the counts).
//
// A site is a 0-based position p of a target contig.  Its totals are exactly what plp_snp (xcltk/baf/fc/core.py:
// 198-247) gives a SNP at p, i.e. what xg_baf_pileup writes: check_read, listed cell (or the BAM in sample mode), a
// UMI key, the first read per (cell, UMI) in file order wins even when its allele is None, and the winners with an
// allele count into A / C / G / T / N.  REF is the A..T bucket with the largest count, ALT the second largest (ties
// to the lower index, N never), and the site is kept iff ALT >= 1, sum >= min_count and ALT >= sum * min_maf.
//
// Two stages:
//   raw scan   every aligned base (M / = / X) of every passing read is counted at its position, without the UMI
//              collapse, in shared-memory histograms over windows of DISC_W positions.  A read is handed to every
//              window its aligned blocks touch (count / scan / scatter), so an N gap is never walked.  A winner with
//              base b at p is a distinct passing read with base b at p, so each deduplicated bucket is at most its
//              raw count: a kept site has raw sum >= min_count and two A..T buckets of raw count >= max(1, min_count
//              * min_maf).  Positions failing that test are dropped, nothing else; the survivors are compacted in
//              position order after a counting pass sized the output.
//   exact      xg_baf_pileup on the candidates (sliced if a slice exceeds one of its limits), then the allele
//              inference and the filter on its device totals, and the kept sites compacted in order.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "compact.cuh"

#define DISC_W 2048                 // positions per window: 5 x 32-bit histograms = 40 KB of shared memory
#define DISC_WORDS (DISC_W / 32)    // pass bitmap words of a window

namespace {

struct DiscDev {
    const int2 *pos_end;
    const uint32_t *fmq, *cig_off, *cigar, *seq_off, *seq;
    const ulonglong2 *keys;
    const xg_run *runs;
    const xg_tile *tiles;
    BarcodeTable bc;
    FilterParams fp;
    int32_t n_gid;
    const int32_t *tg_goff;     // [n_gid + 1]: range of each contig in tg
    const int4 *tg;             // targets sorted by (gid, beg): beg, end, first window, caller index
};

// check_read + UMI key + listed cell -- the filters of the pileup's scan (k_baf_scan phase 2) -- and a stored
// sequence (a read without bases has only None alleles: it counts nowhere)
__device__ __forceinline__ bool disc_read_passes(const DiscDev &P, int64_t i, int2 pe, uint32_t *n_ops_out,
                                                 const uint32_t **cig_out) {
    const uint32_t fmq = P.fmq[i];
    if (!read_passes_flags(P.fp, fmq)) return false;
    if (P.seq_off[i] == 0xFFFFFFFFu) return false;
    const ulonglong2 ky = P.keys[i];
    if (ky.y == XG_KEY_NONE || ky.y == XG_KEY_EMPTY) return false;
    if (P.fp.use_cell_tag && (ky.x == XG_KEY_NONE || barcode_lookup(P.bc, ky.x) < 0)) return false;
    uint32_t n_ops = fmq >> 24;
    const uint32_t *cig = nullptr;
    int32_t aln;
    if (n_ops == 0) {
        aln = pe.y - pe.x;
    } else {
        cig = P.cigar + P.cig_off[i];
        if (n_ops == 255) n_ops = __ldg(cig - 1);
        aln = 0;
        for (uint32_t q = 0; q < n_ops; q++) {
            const uint32_t w = __ldg(&cig[q]);
            if (cig_aligned(w & 15u)) aln += (int32_t)(w >> 4);
        }
    }
    if (aln < P.fp.min_len) return false;
    *n_ops_out = n_ops;
    *cig_out = cig;
    return true;
}

// f(w) once for every window the read's aligned blocks touch; t0 = first target of the contig whose end > pos
template <class F>
__device__ __forceinline__ void disc_windows(const DiscDev &P, int2 pe, uint32_t n_ops, const uint32_t *cig,
                                             int32_t t0, int32_t t1, F &&f) {
    int32_t ti = t0, last = -1;
    auto block = [&](int32_t b0, int32_t b1) {
        if (b0 >= b1) return;
        while (ti < t1 && P.tg[ti].y <= b0) ti++;
        for (int32_t t = ti; t < t1; t++) {
            const int4 g = P.tg[t];
            if (g.x >= b1) break;
            const int32_t lo = max(b0, g.x), hi = min(b1, g.y);
            const int32_t w0 = g.z + (lo - g.x) / DISC_W, w1 = g.z + (hi - 1 - g.x) / DISC_W;
            for (int32_t w = w0; w <= w1; w++)
                if (w != last) f(w);        // blocks ascend: only a block's first window can repeat the last one
            last = w1;
        }
    };
    if (n_ops == 0) {
        block(pe.x, pe.y);
        return;
    }
    int32_t p = pe.x;
    for (uint32_t k = 0; k < n_ops; k++) {
        const uint32_t w = __ldg(&cig[k]), op = w & 15u;
        const int32_t l = (int32_t)(w >> 4);
        if (cig_aligned(op)) {
            block(p, p + l);
            p += l;
        } else if (cig_skips_ref(op)) {
            p += l;
        }
    }
}

// One CTA per tile.  SCATTER = false: reads per window; true: the read indices into their windows' lists.
template <bool SCATTER>
__global__ void __launch_bounds__(256) k_disc_route(const __grid_constant__ DiscDev P, int32_t *win_cnt,
                                                    const int64_t *win_off, int32_t *win_cur, uint32_t *win_reads) {
    const xg_tile tile = P.tiles[blockIdx.x];
    const int32_t gid = P.runs[tile.run].gid;
    if (gid < 0 || gid >= P.n_gid) return;
    const int32_t g0 = P.tg_goff[gid], g1 = P.tg_goff[gid + 1];
    if (g0 >= g1) return;
    for (int32_t k = threadIdx.x; k < tile.n_rec; k += 256) {
        const int64_t i = tile.rec_beg + k;
        const int2 pe = P.pos_end[i];
        int32_t lo = g0, hi = g1;
        while (lo < hi) {
            const int32_t mid = (lo + hi) >> 1;
            if (P.tg[mid].y <= pe.x) lo = mid + 1; else hi = mid;
        }
        if (lo >= g1 || P.tg[lo].x >= pe.y) continue;      // [pos, end) meets no target: nothing else is loaded
        uint32_t n_ops = 0;
        const uint32_t *cig = nullptr;
        if (!disc_read_passes(P, i, pe, &n_ops, &cig)) continue;
        disc_windows(P, pe, n_ops, cig, lo, g1, [&](int32_t w) {
            if (SCATTER)
                win_reads[win_off[w] + atomicAdd(&win_cur[w], 1)] = (uint32_t)i;
            else
                atomicAdd(&win_cnt[w], 1);
        });
    }
}

// windows that received reads, in no particular order
__global__ void k_disc_covered(int32_t n_win, const int64_t *win_off, int32_t *cov, unsigned int *n_cov) {
    const int32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n_win || win_off[w + 1] == win_off[w]) return;
    cov[atomicAdd(n_cov, 1u)] = w;
}

// target (caller order) of window w: the last target whose first window is <= w (targets without windows share
// their first window with the next target)
__device__ __forceinline__ int4 disc_target_of(const int4 *tc, int32_t n_tg, int32_t w) {
    int32_t lo = 0, hi = n_tg;
    while (hi - lo > 1) {
        const int32_t mid = (lo + hi) >> 1;
        if (tc[mid].z <= w) lo = mid; else hi = mid;
    }
    return tc[lo];
}

// base class of query position q: 0..3 A C G T, 4 anything else (N, '=', IUPAC: the N bucket, mcount.py:145-149)
__device__ __forceinline__ uint32_t disc_bucket(const uint32_t *seq, uint32_t so, int32_t q) {
    const uint32_t byte = (uint32_t)q >> 1;
    const uint32_t w = __ldg(&seq[so + (byte >> 2)]);
    const uint32_t nib = (w >> (8 * (byte & 3u) + ((q & 1) ? 0u : 4u))) & 15u;
    switch (nib) {
        case 1: return 0;
        case 2: return 1;
        case 4: return 2;
        case 8: return 3;
        default: return 4;
    }
}

// Persistent CTAs over the covered windows: raw A/C/G/T/N counts of the window in shared memory (one read per
// warp, only its aligned bases inside the window), then the pre-filter per position into the window's pass
// bitmap (one ballot per 32 positions) and the window's candidate count.
__global__ void __launch_bounds__(256) k_disc_hist(const __grid_constant__ DiscDev P, const int32_t *cov, int32_t n_cov,
                                                   const int64_t *win_off, const uint32_t *win_reads, const int4 *tc,
                                                   int32_t n_tg, unsigned long long t_sum, uint32_t t_alt,
                                                   uint32_t *bits, int32_t *win_ncand, unsigned long long *scanned,
                                                   unsigned int *work) {
    __shared__ uint32_t h[5 * DISC_W];
    __shared__ int32_t s_c;
    __shared__ uint32_t s_n;
    const int lane = threadIdx.x & 31;
    unsigned long long n_scanned = 0;
    while (true) {
        if (threadIdx.x == 0) {
            s_c = (int32_t)atomicAdd(work, 1u);
            s_n = 0;
        }
        for (int k = threadIdx.x; k < 5 * DISC_W; k += 256) h[k] = 0;
        __syncthreads();
        const int32_t c = s_c;
        if (c >= n_cov) break;
        const int32_t w = cov[c];
        const int4 g = disc_target_of(tc, n_tg, w);
        const int32_t ws = g.x + (w - g.z) * DISC_W, we = min(g.y, ws + DISC_W);
        // one read per warp, the lanes over its aligned positions in the window
        for (int64_t r = win_off[w] + (threadIdx.x >> 5); r < win_off[w + 1]; r += 8) {
            const uint32_t i = win_reads[r];
            const int2 pe = P.pos_end[i];
            const uint32_t so = P.seq_off[i];
            uint32_t n_ops = P.fmq[i] >> 24;
            const uint32_t *cig = nullptr;
            if (n_ops != 0) {
                cig = P.cigar + P.cig_off[i];
                if (n_ops == 255) n_ops = __ldg(cig - 1);
            }
            int32_t rp = pe.x, qp = 0;
            for (uint32_t k = 0; k < (n_ops ? n_ops : 1u); k++) {
                uint32_t op = 0;
                int32_t l = pe.y - pe.x;
                if (n_ops) {
                    const uint32_t cw = __ldg(&cig[k]);
                    op = cw & 15u;
                    l = (int32_t)(cw >> 4);
                }
                if (cig_aligned(op)) {
                    const int32_t a = max(rp, ws), b = min(rp + l, we);
                    for (int32_t p = a + lane; p < b; p += 32)
                        atomicAdd(&h[disc_bucket(P.seq, so, qp + (p - rp)) * DISC_W + (p - ws)], 1u);
                    rp += l;
                    qp += l;
                    if (rp >= we) break;
                } else if (cig_skips_ref(op)) {
                    rp += l;
                    if (rp >= we) break;
                } else if (op == 1 || op == 4) {
                    qp += l;
                }
            }
        }
        __syncthreads();
        uint32_t n_pass = 0;
        for (int32_t b = threadIdx.x; b < DISC_W; b += 256) {
            bool pass = false;
            if (b < we - ws) {
                const uint32_t a = h[b], cc = h[DISC_W + b], gg = h[2 * DISC_W + b], t = h[3 * DISC_W + b];
                const unsigned long long sum =
                    (unsigned long long)a + cc + gg + t + h[4 * DISC_W + b];
                const uint32_t m1 = max(a, cc), m2 = min(a, cc), x1 = max(gg, t), x2 = min(gg, t);
                const uint32_t second = max(min(m1, x1), max(m2, x2));       // second largest of A, C, G, T
                pass = sum >= t_sum && second >= t_alt;
            }
            const unsigned m = __ballot_sync(0xffffffffu, pass);
            if (lane == 0) bits[(size_t)c * DISC_WORDS + (b >> 5)] = m;
            n_pass += pass;
        }
        for (int d = 16; d > 0; d >>= 1) n_pass += __shfl_xor_sync(0xffffffffu, n_pass, d);
        if (lane == 0 && n_pass) atomicAdd(&s_n, n_pass);
        if (threadIdx.x == 0) n_scanned += (unsigned long long)(we - ws);
        __syncthreads();
        if (threadIdx.x == 0) win_ncand[w] = (int32_t)s_n;
        __syncthreads();
    }
    if (threadIdx.x == 0 && n_scanned) atomicAdd(scanned, n_scanned);
}

// One warp per covered window: its passing positions written in position order at the window's offset
__global__ void k_disc_emit(const int32_t *cov, int32_t n_cov, const uint32_t *bits, const int64_t *cand_off,
                            const int4 *tc, int32_t n_tg, int32_t *cand_gid, int32_t *cand_pos) {
    const int32_t c = (int32_t)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (c >= n_cov) return;
    const int32_t w = cov[c];
    const int4 g = disc_target_of(tc, n_tg, w);
    const int32_t ws = g.x + (w - g.z) * DISC_W;
    int64_t o = cand_off[w];
    for (int k0 = 0; k0 < DISC_WORDS; k0 += 32) {
        uint32_t m = bits[(size_t)c * DISC_WORDS + k0 + lane];
        const uint32_t pc = __popc(m);
        uint32_t incl = pc;
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += y;
        }
        int64_t at = o + (incl - pc);
        while (m) {
            const int b = __ffs(m) - 1;
            m &= m - 1;
            cand_gid[at] = g.w;
            cand_pos[at] = ws + (k0 + lane) * 32 + b;
            at++;
        }
        o += __shfl_sync(0xffffffffu, incl, 31);
    }
}

// REF / ALT from the deduplicated totals and plp_snp's filter (baf/fc/core.py:238-246, IEEE double as Python
// evaluates int-with-float) with minor = ALT; false if the site is not kept
__device__ __forceinline__ bool disc_infer(const unsigned long long *t, double min_count, double min_maf, int *ref,
                                           int *alt) {
    int r = 0;
    for (int k = 1; k < 4; k++)
        if (t[k] > t[r]) r = k;
    int a = r == 0 ? 1 : 0;
    for (int k = a + 1; k < 4; k++)
        if (k != r && t[k] > t[a]) a = k;
    *ref = r;
    *alt = a;
    const unsigned long long sum = t[0] + t[1] + t[2] + t[3] + t[4];
    if (t[a] < 1) return false;
    if ((double)sum < min_count) return false;
    return !((double)t[a] < __dmul_rn((double)sum, min_maf));
}

// The kept sites of a slice, order-preserving: WRITE = false counts per CTA, WRITE = true writes at the CTA's offset
template <bool WRITE>
__global__ void __launch_bounds__(256) k_disc_keep(int32_t n, const unsigned long long *tot, double min_count,
                                                   double min_maf, int32_t *blk_cnt, const int64_t *blk_off,
                                                   const int32_t *c_gid, const int32_t *c_pos, int64_t base,
                                                   int32_t *o_gid, int32_t *o_pos, uint8_t *o_ref, uint8_t *o_alt,
                                                   int64_t *o_tot) {
    __shared__ uint32_t s_warp[8];
    const int32_t i = blockIdx.x * 256 + threadIdx.x;
    int r = 0, a = 0;
    const bool keep = i < n && disc_infer(tot + (size_t)i * 5, min_count, min_maf, &r, &a);
    if (!WRITE) {
        const int k = __syncthreads_count(keep);
        if (threadIdx.x == 0) blk_cnt[blockIdx.x] = k;
        return;
    }
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) s_warp[wp] = __popc(m);
    __syncthreads();
    if (!keep) return;
    int64_t o = base + blk_off[blockIdx.x] + __popc(m & ((1u << lane) - 1u));
    for (int q = 0; q < wp; q++) o += s_warp[q];
    o_gid[o] = c_gid[i];
    o_pos[o] = c_pos[i];
    o_ref[o] = (uint8_t)r;
    o_alt[o] = (uint8_t)a;
    for (int k = 0; k < 5; k++) o_tot[o * 5 + k] = (int64_t)tot[(size_t)i * 5 + k];
}

// a non-negative double threshold as an integer count: the smallest integer x with x >= v (saturating)
unsigned long long ceil_count(double v) {
    if (!(v > 0)) return 0;
    if (v >= 1e18) return 1000000000000000000ull;
    return (unsigned long long)std::ceil(v);
}

struct EventGuard {
    cudaEvent_t e[3] = {};
    ~EventGuard() {
        for (auto x : e)
            if (x) cudaEventDestroy(x);
    }
};

}  // namespace

extern "C" void xg_sites_free(xg_sites *s) { free(s); }

extern "C" int xg_snp_discover(xg_ctx *ctx, const xg_dreads *rd, const xg_features *targets, const xg_barcodes *cells,
                               const xg_params *par, const xg_discover_filter *filt, xg_sites **out) {
    if (!ctx || !ctx->stream) return ctx ? ctx->fail(XG_E_CUDA, "context has no device") : XG_E_ARG;
    if (!rd || !targets || !cells || !par || !filt || !out) return ctx->fail(XG_E_ARG, "xg_snp_discover: null argument");
    *out = nullptr;
    if (targets->n < 0 || (targets->n > 0 && (!targets->gid || !targets->beg || !targets->end)))
        return ctx->fail(XG_E_ARG, "xg_snp_discover: bad target arrays");
    if (!rd->seq || !rd->seq_off) return ctx->fail(XG_E_ARG, "xg_snp_discover: reads were decoded without sequences");
    if (cells->n_samples <= 0 || cells->n_samples >= (1 << 24))
        return ctx->fail(XG_E_ARG, "xg_snp_discover: number of cells must be in [1, 2^24)");
    if (par->use_cell_tag && cells->n != cells->n_samples)
        return ctx->fail(XG_E_ARG, "xg_snp_discover: barcode mode needs one key per column");
    if ((uint64_t)rd->n_tiles * XG_TILE >= (1ull << 32))
        return ctx->fail(XG_E_LIMIT, "xg_snp_discover: more than 2^32 record slots in one batch");
    XG_CUDA(cudaSetDevice(ctx->device));
    const auto t_call = std::chrono::steady_clock::now();
    int32_t n_gid = 0;
    for (auto &r : rd->h_runs) n_gid = std::max(n_gid, r.gid + 1);
    if (!par->use_cell_tag)
        for (auto &r : rd->h_runs)
            if (r.bam_idx >= cells->n_samples) return ctx->fail(XG_E_ARG, "more BAMs than sample columns");

    // targets: windows numbered in caller order; the device looks them up sorted by (gid, beg)
    const int32_t n_tg = targets->n;
    std::vector<int4> tc((size_t)n_tg + 1);
    std::vector<int32_t> ord;
    int64_t n_win = 0;
    for (int32_t t = 0; t < n_tg; t++) {
        const int32_t g = targets->gid[t], b = targets->beg[t], e = targets->end[t];
        const bool live = g >= 0 && g < n_gid && b >= 0 && e > b;
        tc[t] = make_int4(b, e, (int32_t)std::min<int64_t>(n_win, INT32_MAX), g);
        if (!live) continue;
        ord.push_back(t);
        n_win += ((int64_t)e - b + DISC_W - 1) / DISC_W;
    }
    if (n_win >= INT32_MAX) return ctx->fail(XG_E_LIMIT, "xg_snp_discover: more than 2^31 windows");
    tc[n_tg] = make_int4(0, 0, (int32_t)n_win, -1);
    std::sort(ord.begin(), ord.end(), [&](int32_t a, int32_t b) {
        if (targets->gid[a] != targets->gid[b]) return targets->gid[a] < targets->gid[b];
        return targets->beg[a] < targets->beg[b];
    });
    std::vector<int4> tg(ord.size() + 1);
    std::vector<int32_t> goff((size_t)n_gid + 1, 0);
    for (size_t k = 0; k < ord.size(); k++) {
        const int32_t t = ord[k];
        if (k > 0 && targets->gid[ord[k - 1]] == targets->gid[t] && targets->end[ord[k - 1]] > targets->beg[t])
            return ctx->fail(XG_E_ARG, "xg_snp_discover: targets of one contig overlap");
        tg[k] = make_int4(targets->beg[t], targets->end[t], tc[t].z, t);
        goff[(size_t)targets->gid[t] + 1]++;
    }
    for (int32_t g = 0; g < n_gid; g++) goff[(size_t)g + 1] += goff[(size_t)g];

    DiscDev P;
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
    P.fp.min_mapq = par->min_mapq;
    P.fp.min_len = par->min_len;
    P.fp.incl_flag = par->incl_flag;
    P.fp.excl_flag = par->excl_flag;
    P.fp.no_orphan = par->no_orphan;
    P.fp.use_cell_tag = par->use_cell_tag;
    P.fp.need_umi_tag = par->need_umi_tag;
    int rc;
    if (par->use_cell_tag && (rc = xg_build_barcode_table(ctx, cells, &P.bc))) return rc;
    XG_GET(d_tg, int4, "sd_tg", tg.size());
    XG_GET(d_tc, int4, "sd_tc", tc.size());
    XG_GET(d_goff, int32_t, "sd_goff", goff.size());
    XG_GET(win_cnt, int32_t, "sd_win_cnt", n_win + 1);
    XG_GET(win_cur, int32_t, "sd_win_cur", n_win + 1);
    XG_GET(win_ncand, int32_t, "sd_win_ncand", n_win + 1);
    XG_GET(win_off, int64_t, "sd_win_off", n_win + 2);
    XG_GET(cand_off, int64_t, "sd_cand_off", n_win + 2);
    XG_GET(cov, int32_t, "sd_cov", n_win + 1);
    XG_GET(ctr, unsigned long long, "sd_ctr", 4);      // [0] covered windows, [1] work counter, [2] positions scanned
    XG_CUDA(cudaMemcpyAsync(d_tg, tg.data(), sizeof(int4) * tg.size(), cudaMemcpyHostToDevice, ctx->stream));
    XG_CUDA(cudaMemcpyAsync(d_tc, tc.data(), sizeof(int4) * tc.size(), cudaMemcpyHostToDevice, ctx->stream));
    XG_CUDA(cudaMemcpyAsync(d_goff, goff.data(), sizeof(int32_t) * goff.size(), cudaMemcpyHostToDevice, ctx->stream));
    P.tg = d_tg;
    P.tg_goff = d_goff;
    EventGuard ev;
    for (auto &e : ev.e) XG_CUDA(cudaEventCreate(&e));
    int launches = 0;

    // ---- raw scan
    cudaEventRecord(ev.e[0], ctx->stream);
    XG_CUDA(cudaMemsetAsync(win_cnt, 0, sizeof(int32_t) * (n_win + 1), ctx->stream));
    XG_CUDA(cudaMemsetAsync(win_cur, 0, sizeof(int32_t) * (n_win + 1), ctx->stream));
    XG_CUDA(cudaMemsetAsync(win_ncand, 0, sizeof(int32_t) * (n_win + 1), ctx->stream));
    XG_CUDA(cudaMemsetAsync(ctr, 0, 32, ctx->stream));
    const bool any = rd->n_tiles > 0 && n_win > 0;
    if (any) {
        k_disc_route<false><<<rd->n_tiles, 256, 0, ctx->stream>>>(P, win_cnt, nullptr, nullptr, nullptr);
        launches++;
    }
    k_exclusive_scan<<<1, 1024, 0, ctx->stream>>>(win_cnt, win_off, (int32_t)n_win);
    launches++;
    if (n_win > 0) {
        k_disc_covered<<<(unsigned)((n_win + 255) / 256), 256, 0, ctx->stream>>>((int32_t)n_win, win_off, cov,
                                                                                   (unsigned int *)&ctr[0]);
        launches++;
    }
    XG_CUDA(cudaGetLastError());
    long long h_entries = 0;
    unsigned long long h_ctr[4] = {0, 0, 0, 0};
    XG_CUDA(cudaMemcpyAsync(&h_entries, win_off + n_win, 8, cudaMemcpyDeviceToHost, ctx->stream));
    XG_CUDA(cudaMemcpyAsync(h_ctr, ctr, 8, cudaMemcpyDeviceToHost, ctx->stream));
    XG_CUDA(cudaStreamSynchronize(ctx->stream));
    const int32_t n_cov = (int32_t)(h_ctr[0] & 0xFFFFFFFFull);
    XG_GET(win_reads, uint32_t, "sd_win_reads", h_entries + 1);
    XG_GET(bits, uint32_t, "sd_bits", (size_t)n_cov * DISC_WORDS + 1);
    const unsigned long long t_sum = ceil_count(filt->min_count);
    const double prod = (filt->min_count > 0 && filt->min_maf > 0) ? filt->min_count * filt->min_maf : 0.0;
    const unsigned long long t_alt64 = std::max<unsigned long long>(1ull, ceil_count(prod));
    const uint32_t t_alt = (uint32_t)std::min<unsigned long long>(t_alt64, 0xFFFFFFFFull);
    if (h_entries > 0) {
        k_disc_route<true><<<rd->n_tiles, 256, 0, ctx->stream>>>(P, nullptr, win_off, win_cur, win_reads);
        const int grid = std::min(n_cov, 148 * 5);
        k_disc_hist<<<grid, 256, 0, ctx->stream>>>(P, cov, n_cov, win_off, win_reads, d_tc, n_tg, t_sum, t_alt, bits,
                                                    win_ncand, &ctr[2], (unsigned int *)&ctr[1]);
        launches += 2;
    }
    k_exclusive_scan<<<1, 1024, 0, ctx->stream>>>(win_ncand, cand_off, (int32_t)n_win);
    launches++;
    XG_CUDA(cudaGetLastError());
    long long n_cand = 0;
    XG_CUDA(cudaMemcpyAsync(&n_cand, cand_off + n_win, 8, cudaMemcpyDeviceToHost, ctx->stream));
    XG_CUDA(cudaMemcpyAsync(h_ctr, ctr, 32, cudaMemcpyDeviceToHost, ctx->stream));
    XG_CUDA(cudaStreamSynchronize(ctx->stream));
    if (n_cand >= INT32_MAX) return ctx->fail(XG_E_LIMIT, "xg_snp_discover: more than 2^31 raw candidates");
    XG_GET(cand_gid, int32_t, "sd_cand_gid", n_cand + 1);
    XG_GET(cand_pos, int32_t, "sd_cand_pos", n_cand + 1);
    std::vector<int32_t> h_gid((size_t)n_cand), h_pos((size_t)n_cand);
    if (n_cand > 0) {
        k_disc_emit<<<(unsigned)((n_cov + 7) / 8), 256, 0, ctx->stream>>>(cov, n_cov, bits, cand_off, d_tc, n_tg,
                                                                           cand_gid, cand_pos);
        launches++;
        XG_CUDA(cudaGetLastError());
        XG_CUDA(cudaMemcpyAsync(h_gid.data(), cand_gid, 4 * (size_t)n_cand, cudaMemcpyDeviceToHost, ctx->stream));
        XG_CUDA(cudaMemcpyAsync(h_pos.data(), cand_pos, 4 * (size_t)n_cand, cudaMemcpyDeviceToHost, ctx->stream));
    }
    cudaEventRecord(ev.e[1], ctx->stream);
    XG_CUDA(cudaStreamSynchronize(ctx->stream));

    // ---- exact stage: the pileup on the candidates, slice by slice
    XG_GET(o_gid, int32_t, "sd_o_gid", n_cand + 1);
    XG_GET(o_pos, int32_t, "sd_o_pos", n_cand + 1);
    XG_GET(o_ref, uint8_t, "sd_o_ref", n_cand + 1);
    XG_GET(o_alt, uint8_t, "sd_o_alt", n_cand + 1);
    XG_GET(o_tot, int64_t, "sd_o_tot", 5 * (n_cand + 1));
    int64_t slice = ctx->discover_slice > 0 ? ctx->discover_slice : (1ll << 22);
    int64_t n_kept = 0, n_slices = 0;
    for (int64_t s0 = 0; s0 < n_cand;) {
        const int32_t n = (int32_t)std::min<int64_t>(slice, n_cand - s0);
        xg_snps snps;
        snps.n = n;
        snps.gid = h_gid.data() + s0;
        snps.pos = h_pos.data() + s0;
        xg_baf_state *st = nullptr;
        rc = xg_baf_pileup(ctx, rd, &snps, cells, par, nullptr, &st);
        if (rc == XG_E_LIMIT && n > 1) {          // too many (read, site) pairs for one pileup: smaller slices
            slice = n / 2;
            continue;
        }
        if (rc) return rc;
        launches += (int)ctx->timing[2];
        xg_baf_state_free(ctx, st);
        const unsigned long long *tot = (const unsigned long long *)ctx->scratch["bf_totals"].p;
        const int32_t n_blk = (n + 255) / 256;
        XG_GET(blk_cnt, int32_t, "sd_blk_cnt", n_blk + 1);
        XG_GET(blk_off, int64_t, "sd_blk_off", n_blk + 2);
        k_disc_keep<false><<<n_blk, 256, 0, ctx->stream>>>(n, tot, filt->min_count, filt->min_maf, blk_cnt, nullptr,
                                                            nullptr, nullptr, 0, nullptr, nullptr, nullptr, nullptr,
                                                            nullptr);
        k_exclusive_scan<<<1, 1024, 0, ctx->stream>>>(blk_cnt, blk_off, n_blk);
        k_disc_keep<true><<<n_blk, 256, 0, ctx->stream>>>(n, tot, filt->min_count, filt->min_maf, nullptr, blk_off,
                                                           cand_gid + s0, cand_pos + s0, n_kept, o_gid, o_pos, o_ref,
                                                           o_alt, o_tot);
        launches += 3;
        XG_CUDA(cudaGetLastError());
        long long k = 0;
        XG_CUDA(cudaMemcpyAsync(&k, blk_off + n_blk, 8, cudaMemcpyDeviceToHost, ctx->stream));
        XG_CUDA(cudaStreamSynchronize(ctx->stream));
        n_kept += k;
        s0 += n;
        n_slices++;
    }
    cudaEventRecord(ev.e[2], ctx->stream);

    // ---- result in library-owned host memory (one block: header, totals, gid, pos, ref, alt)
    const size_t n = (size_t)n_kept;
    xg_sites *res = (xg_sites *)malloc(sizeof(xg_sites) + n * (40 + 4 + 4 + 1 + 1) + 16);
    if (!res) return ctx->fail(XG_E_NOMEM, "xg_snp_discover: out of host memory");
    uint8_t *base = (uint8_t *)(res + 1);
    int64_t *h_tot = (int64_t *)base;
    int32_t *r_gid = (int32_t *)(base + n * 40);
    int32_t *r_pos = r_gid + n;
    uint8_t *r_ref = (uint8_t *)(r_pos + n);
    uint8_t *r_alt = r_ref + n;
    if (n) {
        cudaMemcpyAsync(h_tot, o_tot, n * 40, cudaMemcpyDeviceToHost, ctx->stream);
        cudaMemcpyAsync(r_gid, o_gid, n * 4, cudaMemcpyDeviceToHost, ctx->stream);
        cudaMemcpyAsync(r_pos, o_pos, n * 4, cudaMemcpyDeviceToHost, ctx->stream);
        cudaMemcpyAsync(r_ref, o_ref, n, cudaMemcpyDeviceToHost, ctx->stream);
        cudaMemcpyAsync(r_alt, o_alt, n, cudaMemcpyDeviceToHost, ctx->stream);
    }
    const cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        free(res);
        return ctx->fail(XG_E_CUDA, std::string("snp discover: ") + cudaGetErrorString(e));
    }
    res->n = n_kept;
    res->gid = r_gid;
    res->pos = r_pos;
    res->ref = r_ref;
    res->alt = r_alt;
    res->totals = h_tot;
    *out = res;
    float t_all = 0, t_raw = 0, t_exact = 0;
    cudaEventElapsedTime(&t_all, ev.e[0], ev.e[2]);
    cudaEventElapsedTime(&t_raw, ev.e[0], ev.e[1]);
    cudaEventElapsedTime(&t_exact, ev.e[1], ev.e[2]);
    for (double &t : ctx->timing) t = 0;
    ctx->timing[0] = t_all;
    ctx->timing[1] = t_raw;
    ctx->timing[2] = launches;
    ctx->timing[3] = t_exact;
    ctx->timing[5] = (double)n_cov;
    ctx->timing[6] = (double)h_ctr[2];
    ctx->timing[7] = (double)n_cand;
    ctx->timing[11] = (double)n_slices;
    ctx->timing[12] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_call).count();
    ctx->timing[13] = (double)h_entries;
    ctx->timing[14] = (double)n_kept;
    return XG_OK;
}
