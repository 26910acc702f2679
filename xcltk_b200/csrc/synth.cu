// synth.cu -- synthetic 10x-style read records generated directly in HBM (bench / tests).
//
// No reference counterpart (the reference ships no benchmark; SURVEY.md 8(d) C1-C3 define the
// distribution).  Every field of read i is a pure function of (i, seed), so the array comes out
// coordinate sorted without a sort: read i sits in stratum i of the concatenated span space.
//   CIGAR mix: 78% LM, 15% aM gN bM (g in 80..5000), 4% soft clip, 3% aM 2D bM 3I
//   flags: strand; 4% secondary, 5% duplicate, 1% supplementary; MAPQ 255 (85%) else {0,1,3}
//   molecules: groups of 96 consecutive reads hold 32 molecules of 3 reads each, interleaved
//   (same cell + UMI, ~32 reads apart); 10% of the reads are singletons instead;
//   5% of molecules carry an unlisted barcode, 1% of reads lack CB, 1% lack UB, 0.5% empty UB.
#include <algorithm>
#include <cstring>
#include <string>

#include "compact.cuh"
#include "keys.hpp"

namespace {

struct SynthDev {
    int64_t n_reads;       // reads of this batch: reads [i_base, i_base + n_reads) of a library of n_total
    int64_t i_base, n_total;
    uint64_t G;            // total span length
    uint64_t seed;
    int32_t n_cells, n_cells_all, read_len, want_seq, seq_words;
    int32_t n_spans;
    const int32_t *span_gid, *span_beg;
    const uint64_t *span_pre;   // n_spans + 1 prefix lengths
    int32_t n_snps;
    const int32_t *snp_goff;    // per gid offsets into the sorted SNP arrays
    const int32_t *snp_pos;
    const uint8_t *snp_ref, *snp_alt, *snp_ref_hap;
    int32_t n_gid;
    int32_t pseudo_ref;              // bases of aligned query positions follow a pseudo-reference ...
    uint32_t ref_err_ppm;            // ... except this many per million, which get another base
    // outputs
    int2 *pos_end;
    uint32_t *fmq, *cig_off, *cigar, *seq_off, *seq;
    ulonglong2 *keys;
    const int64_t *chunk_cig_base;   // exclusive scan of per-chunk cigar words
    int32_t *maxes;                  // [0] max_aln_len [1] max_span
};

__host__ __device__ inline uint64_t hsh(uint64_t seed, uint64_t i, uint64_t salt) {
    return mix64(i * 0x9E3779B97F4A7C15ULL + salt * 0xD1B54A32D192ED03ULL + seed);
}

// position of read i in the concatenated span space (monotone non-decreasing in i)
__host__ __device__ inline uint64_t span_coord(uint64_t seed, uint64_t i, uint64_t G, uint64_t N) {
    return (i * G + hsh(seed, i, 1) % G) / N;
}

// packed key of "[ACGT]{16}-1" for cell index k (see keys.hpp for the bit layout)
__host__ __device__ inline uint64_t cell_key(uint64_t seed, uint32_t k) {
    uint32_t x = k ^ (uint32_t)hsh(seed, 0, 77);
    uint64_t key = 0;
    int bits = 0;
    for (int t = 0; t < 16; t++) {
        uint64_t code = ((x >> (2 * t)) & 3u) + 1u;
        key |= code << (63 - bits - 3);
        bits += 3;
    }
    key |= 6ull << (63 - bits - 3);
    bits += 3;
    key |= (uint64_t)((7 << 4) | 1) << (63 - bits - 7);
    return key;
}

__host__ __device__ inline uint64_t umi_key(uint64_t h) {
    uint64_t key = 0;
    int bits = 0;
    for (int t = 0; t < 12; t++) {
        uint64_t code = ((h >> (2 * t)) & 3u) + 1u;
        key |= code << (63 - bits - 3);
        bits += 3;
    }
    return key;
}

struct CigarPlan {
    uint32_t w[4];
    int n;          // words stored (0 = simple)
    int32_t rlen;   // reference length
};

__host__ __device__ inline CigarPlan plan_cigar(uint64_t seed, uint64_t i, int32_t L) {
    CigarPlan c;
    c.n = 0;
    c.rlen = L;
    uint64_t h = hsh(seed, i, 2);
    uint32_t r = (uint32_t)(h % 100);
    uint32_t a = 5 + (uint32_t)((h >> 8) % (uint32_t)(L - 15));    // 5 .. L-11
    if (r < 78) return c;
    if (r < 93) {
        uint32_t g = 80 + (uint32_t)((h >> 24) % 4921);
        c.w[0] = (a << 4) | 0;
        c.w[1] = (g << 4) | 3;
        c.w[2] = ((uint32_t)L - a) << 4 | 0;
        c.n = 3;
        c.rlen = L + (int32_t)g;
    } else if (r < 97) {
        uint32_t s = 1 + (uint32_t)((h >> 8) % (uint32_t)(L / 2));
        if ((h >> 40) & 1) {
            c.w[0] = (s << 4) | 4;
            c.w[1] = ((uint32_t)L - s) << 4 | 0;
        } else {
            c.w[0] = ((uint32_t)L - s) << 4 | 0;
            c.w[1] = (s << 4) | 4;
        }
        c.n = 2;
        c.rlen = L - (int32_t)s;
    } else {
        c.w[0] = (a << 4) | 0;
        c.w[1] = (2u << 4) | 2;
        c.w[2] = ((uint32_t)L - a - 3) << 4 | 0;
        c.w[3] = (3u << 4) | 1;
        c.n = 4;
        c.rlen = L - 3 + 2;
    }
    return c;
}

#define SYNTH_CHUNK 1024

__global__ void __launch_bounds__(256) k_synth_count(uint64_t seed, int64_t n, int64_t i_base, int32_t L,
                                                     int32_t *chunk_words) {
    int64_t c = blockIdx.x;
    int cnt = 0;
    for (int k = threadIdx.x; k < SYNTH_CHUNK; k += blockDim.x) {
        int64_t i = c * SYNTH_CHUNK + k;
        if (i < n) cnt += plan_cigar(seed, (uint64_t)(i_base + i), L).n;
    }
    __shared__ int s[256];
    s[threadIdx.x] = cnt;
    __syncthreads();
    for (int d = 128; d > 0; d >>= 1) {
        if (threadIdx.x < d) s[threadIdx.x] += s[threadIdx.x + d];
        __syncthreads();
    }
    if (threadIdx.x == 0) chunk_words[c] = s[0];
}

__global__ void __launch_bounds__(1024) k_synth_fill(const __grid_constant__ SynthDev P) {
    __shared__ int scan[SYNTH_CHUNK];
    const int64_t i = (int64_t)blockIdx.x * SYNTH_CHUNK + threadIdx.x;
    const bool live = i < P.n_reads;
    CigarPlan cp;
    cp.n = 0;
    cp.rlen = P.read_len;
    const uint64_t gi = (uint64_t)(P.i_base + i);      // the read's index in the whole library
    if (live) cp = plan_cigar(P.seed, gi, P.read_len);
    // in-chunk exclusive scan of cigar words (Hillis-Steele; 1024 threads)
    scan[threadIdx.x] = live ? cp.n : 0;
    __syncthreads();
    for (int d = 1; d < SYNTH_CHUNK; d <<= 1) {
        int v = threadIdx.x >= d ? scan[threadIdx.x - d] : 0;
        __syncthreads();
        scan[threadIdx.x] += v;
        __syncthreads();
    }
    if (!live) return;
    const uint32_t coff = (uint32_t)(P.chunk_cig_base[blockIdx.x] + scan[threadIdx.x] - cp.n);

    // position
    uint64_t u = span_coord(P.seed, gi, P.G, (uint64_t)P.n_total);
    int lo = 0, hi = P.n_spans;             // last span with pre <= u
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (P.span_pre[mid] <= u) lo = mid; else hi = mid;
    }
    const int32_t gid = P.span_gid[lo];
    const int32_t pos = P.span_beg[lo] + (int32_t)(u - P.span_pre[lo]);
    const int32_t end = pos + cp.rlen;
    P.pos_end[i] = make_int2(pos, end);
    int32_t aln = 0;
    if (cp.n == 0) aln = cp.rlen;
    for (int k = 0; k < cp.n; k++) {
        P.cigar[coff + k] = cp.w[k];
        uint32_t op = cp.w[k] & 15u;
        if (op == 0) aln += (int32_t)(cp.w[k] >> 4);
    }
    P.cig_off[i] = coff;
    atomicMax(&P.maxes[0], aln);
    atomicMax(&P.maxes[1], end - pos);

    // flags / mapq
    uint64_t h = hsh(P.seed, gi, 3);
    uint32_t flag = (h & 1) ? 16u : 0u;
    uint32_t r = (uint32_t)((h >> 8) % 100);
    if (r < 4) flag |= 256u;
    else if (r < 9) flag |= 1024u;
    else if (r < 10) flag |= 2048u;
    uint32_t mq = ((h >> 20) % 100) < 85 ? 255u : (uint32_t)((0x030100u >> (8 * ((h >> 32) % 3))) & 0xffu);
    P.fmq[i] = flag | (mq << 16) | ((uint32_t)cp.n << 24);

    // molecule -> cell, UMI
    const uint64_t grp = gi / 96, w = gi % 96;
    uint64_t mol = grp * 32 + (w & 31);
    if (hsh(P.seed, gi, 4) % 10 == 0) mol = (uint64_t)P.n_total + gi;   // singleton
    const uint64_t hm = hsh(P.seed, mol, 5);
    const uint32_t cell = (uint32_t)(hm % (uint64_t)P.n_cells_all);
    uint64_t ck = cell_key(P.seed, cell), uk = umi_key(hm >> 20);
    const uint32_t tg = (uint32_t)(hsh(P.seed, gi, 6) % 1000);
    if (tg < 10) ck = XG_KEY_NONE;
    else if (tg < 20) uk = XG_KEY_NONE;
    else if (tg < 25) uk = XG_KEY_EMPTY;
    P.keys[i] = make_ulonglong2(ck, uk);

    if (P.want_seq) {
        const uint32_t so = (uint32_t)((uint64_t)i * (uint64_t)P.seq_words);
        P.seq_off[i] = so;
        uint32_t *sq = P.seq + so;
        for (int wd = 0; wd < P.seq_words; wd++) {
            uint64_t hb = hsh(P.seed, gi * 16 + (uint64_t)wd, 7);
            uint32_t word = 0;
            for (int b = 0; b < 8; b++) word |= (1u << ((hb >> (2 * b)) & 3u)) << (4 * b);
            sq[wd] = word;
        }
        // pseudo-reference: an aligned base at (gid, p) is the library's base there, or with probability
        // ref_err_ppm / 10^6 one of the other three; the SNP table below overrides its positions
        if (P.pseudo_ref) {
            int32_t p = pos, qi = 0;
            for (int k = 0; k < (cp.n ? cp.n : 1); k++) {
                uint32_t op = 0;
                int32_t l = cp.rlen;
                if (cp.n) {
                    op = cp.w[k] & 15u;
                    l = (int32_t)(cp.w[k] >> 4);
                }
                if (op == 0) {
                    for (int32_t t = 0; t < l; t++) {
                        const int32_t q = qi + t;
                        uint32_t base = (uint32_t)hsh(P.seed, ((uint64_t)(uint32_t)gid << 32) | (uint32_t)(p + t), 10) & 3u;
                        const uint64_t he = hsh(P.seed, gi * 4096 + (uint64_t)q, 11);
                        if (he % 1000000u < P.ref_err_ppm) base = (base + 1u + (uint32_t)((he >> 32) % 3u)) & 3u;
                        const uint32_t byte = (uint32_t)q >> 1, shift = 8 * (byte & 3u) + ((q & 1) ? 0u : 4u);
                        sq[byte >> 2] = (sq[byte >> 2] & ~(15u << shift)) | ((1u << base) << shift);
                    }
                    p += l;
                    qi += l;
                } else if (op == 2 || op == 3) {
                    p += l;
                } else if (op == 1 || op == 4) {
                    qi += l;
                }
            }
        }
        // haplotype-consistent bases at SNPs covered by aligned blocks
        if (P.n_snps > 0 && gid < P.n_gid) {
            const int32_t s0 = P.snp_goff[gid], s1 = P.snp_goff[gid + 1];
            int a = s0, b = s1;
            while (a < b) {
                int mid = (a + b) >> 1;
                if (P.snp_pos[mid] < pos) a = mid + 1; else b = mid;
            }
            const uint32_t hap = (uint32_t)(hsh(P.seed, mol, 8) & 1);
            for (int s = a; s < s1 && P.snp_pos[s] < end; s++) {
                const int32_t sp = P.snp_pos[s];
                // query index of reference position sp (or -1)
                int32_t q = -1, p = pos, qi = 0;
                if (cp.n == 0) {
                    q = sp - pos;
                } else {
                    for (int k = 0; k < cp.n && q < 0; k++) {
                        uint32_t op = cp.w[k] & 15u;
                        int32_t l = (int32_t)(cp.w[k] >> 4);
                        if (op == 0) {
                            if (sp >= p && sp < p + l) q = qi + (sp - p);
                            p += l;
                            qi += l;
                        } else if (op == 2 || op == 3) {
                            p += l;
                        } else if (op == 1 || op == 4) {
                            qi += l;
                        }
                    }
                }
                if (q < 0) continue;
                uint64_t hs = hsh(P.seed, gi * 64 + (uint64_t)(s - a), 9);
                uint32_t rr = (uint32_t)(hs % 100);
                uint32_t code;
                if (rr < 2) {
                    code = (rr == 0 && ((hs >> 8) & 1)) ? 15u : (1u << ((hs >> 10) & 3u));
                } else {
                    uint32_t hh = rr < 3 ? 1u - hap : hap;
                    uint32_t base = (P.snp_ref_hap[s] == hh) ? P.snp_ref[s] : P.snp_alt[s];
                    code = 1u << base;
                }
                // BAM packing: byte q>>1, high nibble for even q
                uint32_t byte = (uint32_t)q >> 1, shift = 8 * (byte & 3u) + ((q & 1) ? 0u : 4u);
                uint32_t wv = sq[byte >> 2];
                wv = (wv & ~(15u << shift)) | (code << shift);
                sq[byte >> 2] = wv;
            }
        }
    }
}

__global__ void k_tile_index(const int2 *pos_end, xg_tile *tiles, int32_t n_tiles) {
    int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (t >= n_tiles) return;
    int lane = threadIdx.x & 31;
    xg_tile tl = tiles[t];
    int32_t m = INT32_MIN;
    for (int k = lane; k < tl.n_rec; k += 32) m = max(m, pos_end[tl.rec_beg + k].y);
    for (int d = 16; d > 0; d >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, d));
    if (lane == 0) {
        tiles[t].first_pos = pos_end[tl.rec_beg].x;
        tiles[t].max_end = m;
    }
}

}  // namespace

extern "C" int xg_synth_reads(xg_ctx *ctx, const xg_synth_params *sp, xg_dreads **out,
                              uint64_t *barcode_keys) {
    if (!ctx || !ctx->stream) return ctx ? ctx->fail(XG_E_CUDA, "context has no device") : XG_E_ARG;
    if (!sp || !out || sp->n_reads <= 0 || sp->n_spans <= 0 || sp->n_cells <= 0 || sp->read_len < 32)
        return ctx->fail(XG_E_ARG, "xg_synth_reads: bad parameters");
    XG_CUDA(cudaSetDevice(ctx->device));
    const int64_t N = sp->n_reads;
    const int64_t NT = sp->total_reads > 0 ? sp->total_reads : N, I0 = sp->total_reads > 0 ? sp->first_read : 0;
    if (I0 < 0 || I0 + N > NT) return ctx->fail(XG_E_ARG, "xg_synth_reads: slice outside the library");
    // span prefix + per-gid boundaries
    std::vector<uint64_t> pre((size_t)sp->n_spans + 1, 0);
    int32_t n_gid = 0;
    for (int32_t s = 0; s < sp->n_spans; s++) {
        if (sp->span_end[s] <= sp->span_beg[s]) return ctx->fail(XG_E_ARG, "empty span");
        if (s > 0 && (sp->span_gid[s] < sp->span_gid[s - 1] ||
                      (sp->span_gid[s] == sp->span_gid[s - 1] && sp->span_beg[s] < sp->span_end[s - 1])))
            return ctx->fail(XG_E_ARG, "spans must be sorted and disjoint");
        pre[(size_t)s + 1] = pre[(size_t)s] + (uint64_t)(sp->span_end[s] - sp->span_beg[s]);
        n_gid = std::max(n_gid, sp->span_gid[s] + 1);
    }
    const uint64_t G = pre.back();
    if ((double)G * (double)NT > 9.0e18) return ctx->fail(XG_E_LIMIT, "n_reads * span length overflows");
    const int32_t seq_words = sp->want_seq ? ((sp->read_len + 1) / 2 + 3) / 4 : 0;
    if ((double)N * seq_words >= 4294967296.0) return ctx->fail(XG_E_LIMIT, "sequence stream exceeds 2^32 words");

    // runs: reads of each gid are contiguous; first read with coord >= boundary (pure function)
    xg_dreads *d = new xg_dreads();
    auto first_at_least = [&](uint64_t bound) -> int64_t {       // in this batch's own numbering
        int64_t lo = 0, hi = NT;
        while (lo < hi) {
            int64_t mid = (lo + hi) / 2;
            if (span_coord(sp->seed, (uint64_t)mid, G, (uint64_t)NT) >= bound) hi = mid; else lo = mid + 1;
        }
        return std::min(std::max(lo, I0), I0 + N) - I0;
    };
    {
        int32_t s = 0;
        while (s < sp->n_spans) {
            int32_t g = sp->span_gid[s], e = s;
            while (e < sp->n_spans && sp->span_gid[e] == g) e++;
            int64_t rb = first_at_least(pre[(size_t)s]), re = first_at_least(pre[(size_t)e]);
            if (re > rb) d->h_runs.push_back(xg_run{0, g, rb, re});
            s = e;
        }
    }
    for (size_t r = 0; r < d->h_runs.size(); r++)
        for (int64_t b = d->h_runs[r].rec_beg; b < d->h_runs[r].rec_end; b += XG_TILE) {
            xg_tile t;
            t.rec_beg = b;
            t.n_rec = (int32_t)std::min<int64_t>(XG_TILE, d->h_runs[r].rec_end - b);
            t.run = (int32_t)r;
            t.first_pos = 0;
            t.max_end = 0;
            d->h_tiles.push_back(t);
        }
    d->n_reads = N;
    d->n_runs = (int32_t)d->h_runs.size();
    d->n_tiles = (int32_t)d->h_tiles.size();

    // SNP table sorted by (gid, pos)
    std::vector<int32_t> snp_goff((size_t)n_gid + 1, 0), snp_pos;
    std::vector<uint8_t> snp_ref, snp_alt, snp_rh;
    if (sp->n_snps > 0) {
        std::vector<int32_t> ord((size_t)sp->n_snps);
        for (int32_t i = 0; i < sp->n_snps; i++) ord[(size_t)i] = i;
        std::sort(ord.begin(), ord.end(), [&](int32_t a, int32_t b) {
            if (sp->snp_gid[a] != sp->snp_gid[b]) return sp->snp_gid[a] < sp->snp_gid[b];
            return sp->snp_pos[a] < sp->snp_pos[b];
        });
        for (int32_t i : ord) {
            int32_t g = sp->snp_gid[i];
            if (g < 0 || g >= n_gid) continue;
            snp_goff[(size_t)g + 1]++;
            snp_pos.push_back(sp->snp_pos[i]);
            snp_ref.push_back(sp->snp_ref[i]);
            snp_alt.push_back(sp->snp_alt[i]);
            snp_rh.push_back(sp->snp_ref_hap[i]);
        }
        for (int32_t g = 0; g < n_gid; g++) snp_goff[(size_t)g + 1] += snp_goff[(size_t)g];
    }

    const int64_t n_chunks = (N + SYNTH_CHUNK - 1) / SYNTH_CHUNK;
    auto fail_free = [&](int code, const std::string &msg) {
        xg_dreads_free(ctx, d);
        return ctx->fail(code, msg);
    };
#define SYN_MALLOC(ptr, bytes)                                                        \
    if (cudaMalloc((void **)&(ptr), (bytes) + 64) != cudaSuccess) {                   \
        cudaGetLastError();                                                           \
        return fail_free(XG_E_CUDA, "cudaMalloc failed in xg_synth_reads");           \
    }
    SYN_MALLOC(d->pos_end, (size_t)N * 8);
    SYN_MALLOC(d->fmq, (size_t)N * 4);
    SYN_MALLOC(d->cig_off, ((size_t)N + 1) * 4);
    SYN_MALLOC(d->keys, (size_t)N * 16);
    if (sp->want_seq) {
        SYN_MALLOC(d->seq_off, (size_t)N * 4);
        SYN_MALLOC(d->seq, (size_t)N * (size_t)seq_words * 4);
        d->n_seq_words = N * seq_words;
    }
    SYN_MALLOC(d->runs, d->h_runs.size() * sizeof(xg_run));
    SYN_MALLOC(d->tiles, d->h_tiles.size() * sizeof(xg_tile));

    int32_t *chunk_words = (int32_t *)ctx->get("syn_chunk_words", sizeof(int32_t) * (size_t)(n_chunks + 1));
    int64_t *chunk_base = (int64_t *)ctx->get("syn_chunk_base", sizeof(int64_t) * (size_t)(n_chunks + 1));
    int32_t *maxes = (int32_t *)ctx->get("syn_maxes", 16);
    int32_t *d_span_gid = (int32_t *)ctx->get("syn_span_gid", 4 * (size_t)sp->n_spans);
    int32_t *d_span_beg = (int32_t *)ctx->get("syn_span_beg", 4 * (size_t)sp->n_spans);
    uint64_t *d_span_pre = (uint64_t *)ctx->get("syn_span_pre", 8 * ((size_t)sp->n_spans + 1));
    int32_t *d_snp_goff = (int32_t *)ctx->get("syn_snp_goff", 4 * ((size_t)n_gid + 1));
    int32_t *d_snp_pos = (int32_t *)ctx->get("syn_snp_pos", 4 * (snp_pos.size() + 1));
    uint8_t *d_snp_ref = (uint8_t *)ctx->get("syn_snp_ref", snp_pos.size() + 1);
    uint8_t *d_snp_alt = (uint8_t *)ctx->get("syn_snp_alt", snp_pos.size() + 1);
    uint8_t *d_snp_rh = (uint8_t *)ctx->get("syn_snp_rh", snp_pos.size() + 1);
    if (!chunk_words || !chunk_base || !maxes || !d_span_gid || !d_span_beg || !d_span_pre ||
        !d_snp_goff || !d_snp_pos || !d_snp_ref || !d_snp_alt || !d_snp_rh)
        return fail_free(XG_E_CUDA, ctx->err);
    cudaStream_t st = ctx->stream;
    cudaMemcpyAsync(d_span_gid, sp->span_gid, 4 * (size_t)sp->n_spans, cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(d_span_beg, sp->span_beg, 4 * (size_t)sp->n_spans, cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(d_span_pre, pre.data(), 8 * pre.size(), cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(d_snp_goff, snp_goff.data(), 4 * snp_goff.size(), cudaMemcpyHostToDevice, st);
    if (!snp_pos.empty()) {
        cudaMemcpyAsync(d_snp_pos, snp_pos.data(), 4 * snp_pos.size(), cudaMemcpyHostToDevice, st);
        cudaMemcpyAsync(d_snp_ref, snp_ref.data(), snp_ref.size(), cudaMemcpyHostToDevice, st);
        cudaMemcpyAsync(d_snp_alt, snp_alt.data(), snp_alt.size(), cudaMemcpyHostToDevice, st);
        cudaMemcpyAsync(d_snp_rh, snp_rh.data(), snp_rh.size(), cudaMemcpyHostToDevice, st);
    }
    cudaMemcpyAsync(d->runs, d->h_runs.data(), d->h_runs.size() * sizeof(xg_run), cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(d->tiles, d->h_tiles.data(), d->h_tiles.size() * sizeof(xg_tile), cudaMemcpyHostToDevice, st);
    cudaMemsetAsync(maxes, 0, 16, st);

    k_synth_count<<<(unsigned)n_chunks, 256, 0, st>>>(sp->seed, N, I0, sp->read_len, chunk_words);
    k_exclusive_scan<<<1, 1024, 0, st>>>(chunk_words, chunk_base, (int32_t)n_chunks);
    int64_t n_cig = 0;
    cudaMemcpyAsync(&n_cig, chunk_base + n_chunks, 8, cudaMemcpyDeviceToHost, st);
    if (cudaStreamSynchronize(st) != cudaSuccess)
        return fail_free(XG_E_CUDA, std::string("synth count: ") + cudaGetErrorString(cudaGetLastError()));
    if (n_cig >= (1LL << 32)) return fail_free(XG_E_LIMIT, "CIGAR stream exceeds 2^32 words");
    SYN_MALLOC(d->cigar, (size_t)n_cig * 4);
    d->n_cigar = n_cig;

    {
        uint32_t sentinel = (uint32_t)n_cig;
        cudaMemcpyAsync(d->cig_off + N, &sentinel, 4, cudaMemcpyHostToDevice, st);
        cudaStreamSynchronize(st);
    }
    SynthDev P;
    memset(&P, 0, sizeof(P));
    P.n_reads = N;
    P.i_base = I0;
    P.n_total = NT;
    P.G = G;
    P.seed = sp->seed;
    P.n_cells = sp->n_cells;
    P.n_cells_all = sp->n_cells + std::max(1, sp->n_cells / 20);
    P.read_len = sp->read_len;
    P.want_seq = sp->want_seq;
    P.seq_words = seq_words;
    P.n_spans = sp->n_spans;
    P.span_gid = d_span_gid;
    P.span_beg = d_span_beg;
    P.span_pre = d_span_pre;
    P.n_snps = (int32_t)snp_pos.size();
    P.snp_goff = d_snp_goff;
    P.snp_pos = d_snp_pos;
    P.snp_ref = d_snp_ref;
    P.snp_alt = d_snp_alt;
    P.snp_ref_hap = d_snp_rh;
    P.n_gid = n_gid;
    P.pseudo_ref = sp->pseudo_ref;
    P.ref_err_ppm = (uint32_t)std::min(1e6, std::max(0.0, sp->ref_error * 1e6 + 0.5));
    P.pos_end = d->pos_end;
    P.fmq = d->fmq;
    P.cig_off = d->cig_off;
    P.cigar = d->cigar;
    P.seq_off = d->seq_off;
    P.seq = d->seq;
    P.keys = d->keys;
    P.chunk_cig_base = chunk_base;
    P.maxes = maxes;
    k_synth_fill<<<(unsigned)n_chunks, SYNTH_CHUNK, 0, st>>>(P);
    if (d->n_tiles > 0) k_tile_index<<<(d->n_tiles + 7) / 8, 256, 0, st>>>(d->pos_end, d->tiles, d->n_tiles);
    int32_t h_max[4] = {0, 0, 0, 0};
    cudaMemcpyAsync(h_max, maxes, 16, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(d->h_tiles.data(), d->tiles, d->h_tiles.size() * sizeof(xg_tile), cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail_free(XG_E_CUDA, std::string("synth fill: ") + cudaGetErrorString(e));
    d->max_aln_len = h_max[0];
    d->max_span = h_max[1];
    {
        int rc = xg_make_tile_pmax(ctx, d);
        if (rc) {
            xg_dreads_free(ctx, d);
            return rc;
        }
    }
    d->bytes = N * 32 + n_cig * 4 + d->n_seq_words * 4 + (sp->want_seq ? N * 4 : 0);

    // barcode keys in column order = sorted barcode strings (rdr/fc/main.py:346)
    if (barcode_keys) {
        std::vector<std::pair<std::string, uint64_t>> bc((size_t)sp->n_cells);
        for (int32_t k = 0; k < sp->n_cells; k++) {
            uint64_t key = cell_key(sp->seed, (uint32_t)k);
            char buf[32];
            int64_t n = xg::key_unpack(key, buf, 32);
            bc[(size_t)k] = {std::string(buf, (size_t)n), key};
        }
        std::sort(bc.begin(), bc.end());
        for (int32_t k = 0; k < sp->n_cells; k++) barcode_keys[k] = bc[(size_t)k].second;
    }
    *out = d;
    return XG_OK;
}

// First read of the library p describes (p->n_reads reads in all; first_read / total_reads ignored) that lies at
// or after position `pos` of contig `gid` -- how a caller cuts the library into genomic chunks.
extern "C" int64_t xg_synth_read_index(const xg_synth_params *sp, int32_t gid, int32_t pos) {
    if (!sp || sp->n_reads <= 0 || sp->n_spans <= 0) return -1;
    std::vector<uint64_t> pre((size_t)sp->n_spans + 1, 0);
    for (int32_t s = 0; s < sp->n_spans; s++)
        pre[(size_t)s + 1] = pre[(size_t)s] + (uint64_t)(sp->span_end[s] - sp->span_beg[s]);
    // coordinate of (gid, pos) in the concatenated span space: a position in a gap counts as the next span's start
    uint64_t bound = pre.back();
    for (int32_t s = 0; s < sp->n_spans; s++) {
        if (sp->span_gid[s] < gid || (sp->span_gid[s] == gid && sp->span_end[s] <= pos)) continue;
        bound = pre[(size_t)s];
        if (sp->span_gid[s] == gid && pos > sp->span_beg[s]) bound += (uint64_t)(pos - sp->span_beg[s]);
        break;
    }
    const uint64_t G = pre.back(), N = (uint64_t)sp->n_reads;
    int64_t lo = 0, hi = sp->n_reads;
    while (lo < hi) {
        int64_t mid = (lo + hi) / 2;
        if (span_coord(sp->seed, (uint64_t)mid, G, N) >= bound) hi = mid; else lo = mid + 1;
    }
    return lo;
}
