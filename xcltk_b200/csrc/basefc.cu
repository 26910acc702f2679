// basefc.cu -- per-feature, per-cell distinct-UMI counting (the RDR total-depth matrix).
//
// Reference being replaced (xcltk v0.5.2):
//   fc_features / fc_fet1      xcltk/rdr/fc/core.py:69-178   for feature: fetch reads, filter, count
//   check_read                 xcltk/rdr/fc/core.py:46-62
//   __get_include_frac/_len    xcltk/rdr/fc/core.py:32-43, used :160-165
//   MCount/SCount.push_read    xcltk/rdr/fc/mcount.py:34-43,102-132 (cell lookup, UMI set)
//   sam_fetch                  xcltk/utils/sam.py:85-118  (reads overlapping the feature)
//
// The reference walks features and re-fetches the reads of each one.  Here the reads are streamed ONCE in file
// order by persistent CTAs (tiles of <= 1024 records from a work counter; tile descriptors, the slice of the interval
// index under the tile and its CIGAR words staged in shared memory by bulk copies); each read finds the features it
// overlaps through a per-contig interval index (sorted boundaries + per-segment stabbing lists + start-sorted
// features) and evaluates the include test arithmetically on its CIGAR.  A passing (feature, cell, UMI) is one 64-bit
// pair word `umi | cell`: it goes through a tile-local duplicate filter and is APPENDED to the feature's segment of a
// pool; when the last read that can touch a feature has been streamed, one CTA deduplicates the segment in shared
// memory and writes the row's non-zeros in column order.  What does not fit a pair word (or a segment) keeps an
// open-addressing (cell, UMI) set in global memory (128-bit CAS).  Features are counted independently (a read
// overlapping k features is evaluated k times), exactly as the reference does (SURVEY.md A.1 R9).
#include <fcntl.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <iterator>
#include <map>
#include <thread>

#include "compact.cuh"

// XG_DEBUG_SYNC=1: synchronise and report after every launch (locates a faulting / hanging kernel)
#define XG_DBG(name)                                                                          \
    do {                                                                                      \
        if (c.dbg_sync) {                                                                     \
            cudaError_t e_ = cudaDeviceSynchronize();                                         \
            fprintf(stderr, "[xg] %s: %s\n", name, cudaGetErrorString(e_));                   \
        }                                                                                     \
    } while (0)

namespace {

struct FeatIndexHost {
    int32_t n_gid = 0;
    std::vector<int32_t> sf_goff, sf_beg, sf_end, sf_row;
    std::vector<int32_t> bnd_goff, bnd, stab_off, stab;
    std::vector<int32_t> fb;   // per boundary: first sorted feature with beg >= bnd[k] (+ terminator)
};

// Interval index over the valid features of every contig.
int build_feat_index(xg_ctx *ctx, const xg_features *f, int32_t n_gid, FeatIndexHost &ix) {
    ix.n_gid = n_gid;
    std::vector<int32_t> order;
    order.reserve((size_t)f->n);
    for (int32_t i = 0; i < f->n; i++) {
        // never fetched: unknown contig, start <= 0 (fetch raises), empty interval
        if (f->gid[i] < 0 || f->gid[i] >= n_gid || f->beg[i] < 0 || f->end[i] <= f->beg[i]) continue;
        order.push_back(i);
    }
    std::sort(order.begin(), order.end(), [&](int32_t a, int32_t b) {
        if (f->gid[a] != f->gid[b]) return f->gid[a] < f->gid[b];
        if (f->beg[a] != f->beg[b]) return f->beg[a] < f->beg[b];
        if (f->end[a] != f->end[b]) return f->end[a] < f->end[b];
        return a < b;
    });
    size_t m = order.size();
    ix.sf_beg.resize(m);
    ix.sf_end.resize(m);
    ix.sf_row.resize(m);
    ix.sf_goff.assign((size_t)n_gid + 1, 0);
    for (size_t j = 0; j < m; j++) {
        int32_t i = order[j];
        ix.sf_beg[j] = f->beg[i];
        ix.sf_end[j] = f->end[i];
        ix.sf_row[j] = i;
        ix.sf_goff[(size_t)f->gid[i] + 1]++;
    }
    for (int32_t g = 0; g < n_gid; g++) ix.sf_goff[g + 1] += ix.sf_goff[g];
    ix.bnd_goff.assign((size_t)n_gid + 1, 0);
    ix.stab_off.clear();
    for (int32_t g = 0; g < n_gid; g++) {
        int32_t j0 = ix.sf_goff[g], j1 = ix.sf_goff[g + 1];
        std::vector<int32_t> b;
        b.reserve(2 * (size_t)(j1 - j0));
        for (int32_t j = j0; j < j1; j++) {
            b.push_back(ix.sf_beg[j]);
            b.push_back(ix.sf_end[j]);
        }
        std::sort(b.begin(), b.end());
        b.erase(std::unique(b.begin(), b.end()), b.end());
        size_t nb = b.size();
        // stabbing list of segment k = [b[k], b[k+1]): features with beg <= b[k] and end >= b[k+1]
        std::vector<int32_t> cnt(nb + 1, 0);
        std::vector<std::pair<int32_t, int32_t>> span((size_t)(j1 - j0));
        int64_t total = 0;
        for (int32_t j = j0; j < j1; j++) {
            int32_t lo = (int32_t)(std::lower_bound(b.begin(), b.end(), ix.sf_beg[j]) - b.begin());
            int32_t hi = (int32_t)(std::lower_bound(b.begin(), b.end(), ix.sf_end[j]) - b.begin());
            span[(size_t)(j - j0)] = {lo, hi};
            for (int32_t k = lo; k < hi; k++) cnt[(size_t)k]++;
            total += hi - lo;
        }
        if ((int64_t)ix.stab.size() + total > (1LL << 30))
            return ctx->fail(XG_E_LIMIT, "feature overlap structure too large (stabbing lists > 2^30)");
        size_t base_seg = ix.bnd.size();
        size_t base_stab = ix.stab.size();
        ix.bnd.insert(ix.bnd.end(), b.begin(), b.end());
        std::vector<int32_t> off(nb + 1, 0);
        for (size_t k = 0; k < nb; k++) off[k + 1] = off[k] + cnt[k];
        ix.stab.resize(base_stab + (size_t)total);
        std::vector<int32_t> cur(off.begin(), off.end() - 1);
        for (int32_t j = j0; j < j1; j++) {
            auto sp = span[(size_t)(j - j0)];
            for (int32_t k = sp.first; k < sp.second; k++) ix.stab[base_stab + (size_t)cur[(size_t)k]++] = j;
        }
        for (size_t k = 0; k < nb; k++) ix.stab_off.push_back((int32_t)(base_stab + (size_t)off[k]));
        (void)base_seg;
        ix.bnd_goff[(size_t)g + 1] = (int32_t)ix.bnd.size();
    }
    ix.stab_off.push_back((int32_t)ix.stab.size());
    // features beginning exactly at boundary k are the sorted features [fb[k], fb[k+1])
    ix.fb.resize(ix.bnd.size() + 1);
    for (int32_t g = 0; g < n_gid; g++) {
        int32_t j = ix.sf_goff[g];
        for (int32_t k = ix.bnd_goff[g]; k < ix.bnd_goff[(size_t)g + 1]; k++) {
            while (j < ix.sf_goff[(size_t)g + 1] && ix.sf_beg[(size_t)j] < ix.bnd[(size_t)k]) j++;
            ix.fb[(size_t)k] = j;
        }
    }
    ix.fb[ix.bnd.size()] = (int32_t)m;
    return XG_OK;
}

// Per (feature, run of its contig): the tiles that can hold an overlapping read -- tiles with
// prefix-max(end) > beg and first_pos < end (two binary searches over the tile index) --
// tightened to records: from the first record of the first tile whose end > beg to the first
// record of the last tile whose pos >= end.  One warp per (feature, run).  Outputs per feature:
// candidate-read count (capacity of its set), first / last tile (its lifetime).
struct WinJob {
    int32_t j0, j1;          // sorted features [j0, j1) of the run's contig
    int32_t t0, t1;          // tiles [t0, t1) of the run
    int64_t warp0;           // first warp of the job (prefix of j1 - j0)
};
__global__ void __launch_bounds__(256) k_feature_windows(const WinJob *jobs, int32_t n_jobs, int64_t n_warps,
                                                         const xg_tile *tiles, const int32_t *pmax,
                                                         const int2 *pos_end, int32_t refine,
                                                         const int32_t *sf_beg, const int32_t *sf_end,
                                                         unsigned long long *cand, int32_t *tlo, int32_t *thi) {
    const int64_t w = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (w >= n_warps) return;
    int a = 0, b = n_jobs;                  // last job with warp0 <= w
    while (b - a > 1) {
        int mid = (a + b) >> 1;
        if (jobs[mid].warp0 <= w) a = mid; else b = mid;
    }
    const WinJob job = jobs[a];
    const int32_t j = job.j0 + (int32_t)(w - job.warp0);
    const int32_t beg = sf_beg[j], end = sf_end[j];
    int32_t lo = job.t0, hi = job.t1;
    while (lo < hi) {                       // first tile with pmax > beg
        int32_t mid = (lo + hi) >> 1;
        if (pmax[mid] > beg) hi = mid; else lo = mid + 1;
    }
    const int32_t t_lo = lo;
    hi = job.t1;
    while (lo < hi) {                       // first tile with first_pos >= end
        int32_t mid = (lo + hi) >> 1;
        if (tiles[mid].first_pos >= end) hi = mid; else lo = mid + 1;
    }
    const int32_t t_hi = lo;
    if (t_hi <= t_lo) return;
    const xg_tile L = tiles[t_lo], H = tiles[t_hi - 1];
    int64_t first = L.rec_beg, last = H.rec_beg + H.n_rec;
    if (refine) {
        first = L.rec_beg + L.n_rec;
        for (int base = 0; base < L.n_rec; base += 32) {
            int k = base + lane;
            unsigned msk = __ballot_sync(0xffffffffu, k < L.n_rec && pos_end[L.rec_beg + k].y > beg);
            if (msk) {
                first = L.rec_beg + base + (__ffs(msk) - 1);
                break;
            }
        }
        for (int base = 0; base < H.n_rec; base += 32) {
            int k = base + lane;
            unsigned msk = __ballot_sync(0xffffffffu, k < H.n_rec && pos_end[H.rec_beg + k].x >= end);
            if (msk) {
                last = H.rec_beg + base + (__ffs(msk) - 1);
                break;
            }
        }
    }
    if (lane == 0) {
        if (last > first) atomicAdd(&cand[j], (unsigned long long)(last - first));
        atomicMin(&tlo[j], t_lo);
        atomicMax(&thi[j], t_hi);
    }
}

// ---- epoch plan ------------------------------------------------------------------------
// The read stream is cut into epochs of `epoch_tiles` tiles.  A feature owns a block of the
// pool (its (cell, UMI) set) from the first epoch that can hold one of its reads to the last;
// the block is zeroed just before the first, reduced to the row's non-zeros just after the
// last, and then reused by later features.  The pool therefore stays about as large as the
// state of the features under the current genomic window, so that it can live in the 126 MB
// L2 instead of streaming through HBM.
// cap > 0: a set (slots, cursor, log); cap == 0: a segment of log_cap 8-byte pair words
#define SEG_TBL_SLOTS 4096                         // dedup table of the finalize CTAs (64-bit words)
#define SEG_PART_WORDS (SEG_TBL_SLOTS * 2 / 5)     // a segment with more words is split by hash first
__host__ __device__ __forceinline__ uint64_t plan_blk_bytes(uint32_t cap, uint32_t log_cap) {
    // a segment that may have to be split carries a scratch half of the same size
    if (!cap) return ((((uint64_t)log_cap * 8) + 15) & ~15ull) * (log_cap > SEG_PART_WORDS ? 2 : 1);
    return (uint64_t)cap * 16 + 16 + ((((uint64_t)log_cap * 4) + 15) & ~15ull);
}

// ---- the counting kernel ------------------------------------------------------------------
#define CNT_THREADS 256
#define CNT_WARPS 8
#define CHUNK 32         // records per warp iteration: one per lane
#define SB_MAX 128       // boundaries of a tile's window staged in shared memory
#define STAB_CAP 128     // stabbing-list entries of those boundaries staged in shared memory
#define CIG_CAP 1024     // CIGAR words of the tile staged in shared memory
#define WPAIR_CAP 96     // (feature, cell, UMI) pairs a warp stages before it appends them
#define FILT_BITS 10     // tile-local duplicate filter: 2^FILT_BITS direct-mapped 64-bit entries, one per index stage
#define INCL_CAP 256     // include-threshold table entries kept in shared memory
#define LEGACY_BIT 0x80000000u
#define NO_SEG 0xFFFFFFFFu

// per sorted feature: where its state lives in the pool.
//   cap > 0  : "set" feature -- [ set: cap x 16 B ][ cursor: 16 B ][ log: log_cap x 4 B ]; the log
//              receives the cell of every NEW (cell, UMI) element (heavy features, and every
//              feature of a batch whose UMI keys do not leave their low 24 bits free)
//   cap == 0 : "segment" feature -- log_cap x 8 B of appended pair words `umi | cell`, deduplicated
//              by the finalize CTA in shared memory (log_cap = candidate reads = upper bound)
struct __align__(16) FeatDesc {
    unsigned long long blk_off;
    uint32_t cap, log_cap;
};

// ---- the epoch planner (device) ---------------------------------------------------------------
// From every sorted feature's candidate reads and tile window (k_feature_windows) the planner decides, without a
// round trip to the host: set or segment (big or not), the feature's block in the pool, and the per-epoch lists
// of features to zero and to finalize.  Lists are counting sorts over one histogram of keys
//   [kind k][last epoch e][32 - floor(log2 candidates)]   kind 0 segments, 1 sets, 2 big segments
//   [first epoch e]                                       sets to zero before their first epoch
// so that the finalize list of (k, e) is one range of a single array, heaviest rows first (the persistent finalize
// CTAs end closer together); order inside a key is whatever the atomics made it.  Blocks: a feature that lives in
// one or two epochs takes its block from the arena of its first epoch -- three arenas in rotation, each as large
// as the busiest epoch, since zero(e) / count(e) are ordered after finalize(e-2) -- and the few that live longer
// get a place of their own behind the arenas.  The host reads the summary only.
#define PLAN_KEYS 33                               // log2 buckets of an epoch
#define PLAN_SCAN_THREADS 1024
struct PlanSummary {
    unsigned long long pool_bytes, staging_cap;    // staging_cap = sum of min(candidates, columns)
    unsigned long long n_seg_feat, n_set_feat, n_big_feat;
    unsigned int err;                              // bit 0: a window of >= 2^32 reads; bit 1: segment pool >= 64 GiB
    unsigned int pad;
};
struct PlanAcc {                                   // the planner's state of a call, zeroed before it starts
    PlanSummary sum;
    unsigned long long long_bytes, arena;
};

// atomicAdd(p, v) of the lanes with `on`, one atomic per distinct address of the warp; returns what a plain
// atomicAdd would have returned in some order of the lanes.  Whole warp.
template <class T>
__device__ __forceinline__ T warp_add(bool on, T *p, T v) {
    const unsigned act = __ballot_sync(0xffffffffu, on);
    if (!on) return 0;
    const unsigned peers = __match_any_sync(act, (unsigned long long)p);
    const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
    T pre = 0, tot = 0;
    for (unsigned q = peers; q; q &= q - 1) {
        const int l = __ffs(q) - 1;
        const T x = __shfl_sync(peers, v, l);
        if (l < lane) pre += x;
        tot += x;
    }
    T base = 0;
    if (lane == leader) base = atomicAdd(p, tot);
    return __shfl_sync(peers, base, leader) + pre;
}

// What the plan's rules make of one feature.
struct PlanFeat {
    bool on, set;                 // has candidates (and fits); keeps a set
    uint32_t cap, log_cap;        // FeatDesc
    int32_t fe, le;               // first / last epoch
    int64_t fin_key;              // histogram key of its finalize
};
__device__ __forceinline__ PlanFeat plan_feat(unsigned long long c, int32_t tlo, int32_t thi, int32_t epoch_tiles,
                                              int32_t n_epochs, uint64_t seg_max, uint64_t seg_big) {
    PlanFeat f;
    const unsigned long long cap = c + c / 4 + 8;
    f.on = c != 0 && cap < (1ull << 32);
    f.set = f.on && c > seg_max;
    f.cap = f.set ? (uint32_t)cap : 0u;
    f.log_cap = f.on ? (uint32_t)c : 0u;
    f.fe = f.on ? tlo / epoch_tiles : 0;
    f.le = f.on ? (thi - 1) / epoch_tiles : 0;
    const int bk = f.on ? min(63 - __clzll((long long)c), 32) : 0;
    const int kind = f.set ? 1 : c > seg_big ? 2 : 0;
    f.fin_key = ((int64_t)kind * n_epochs + f.le) * PLAN_KEYS + (32 - bk);
    return f;
}

// per feature: classify, count into the histogram, take a block of its first epoch's arena or of the long region
__global__ void __launch_bounds__(256) k_plan_features(const unsigned long long *cand, const int32_t *tlo,
                                                       const int32_t *thi, int32_t m, int32_t n_cols,
                                                       int32_t epoch_tiles, int32_t n_epochs, uint64_t seg_max,
                                                       uint64_t seg_big, PlanAcc *acc,
                                                       unsigned long long *epoch_bytes, int32_t *hist,
                                                       FeatDesc *fdesc, uint32_t *segoff16) {
    const int32_t j = blockIdx.x * blockDim.x + threadIdx.x;         // no early exit: warp_add takes whole warps
    const unsigned long long c = j < m ? cand[j] : 0ull;
    const PlanFeat f = plan_feat(c, j < m ? tlo[j] : 0, j < m ? thi[j] : 0, epoch_tiles, n_epochs, seg_max, seg_big);
    if (c != 0 && !f.on) atomicOr(&acc->sum.err, 1u);
    typedef unsigned long long u64;
    warp_add<u64>(f.on, &acc->sum.staging_cap, c < (u64)n_cols ? c : (u64)n_cols);
    warp_add<u64>(f.on && !f.set, &acc->sum.n_seg_feat, 1ull);
    warp_add<u64>(f.set, &acc->sum.n_set_feat, 1ull);
    warp_add<u64>(f.on && !f.set && c > seg_big, &acc->sum.n_big_feat, 1ull);
    warp_add<int32_t>(f.on, &hist[f.fin_key], 1);
    warp_add<int32_t>(f.set, &hist[(int64_t)3 * n_epochs * PLAN_KEYS + f.fe], 1);
    const u64 need = f.on ? plan_blk_bytes(f.cap, f.log_cap) : 0ull;
    // offset inside the arena or the long region, for now
    const u64 at = warp_add<u64>(f.on, f.le <= f.fe + 1 ? &epoch_bytes[f.fe] : &acc->long_bytes, need);
    if (j < m) {
        fdesc[j] = FeatDesc{at, f.cap, f.log_cap};
        segoff16[j] = NO_SEG;
    }
}

// Exclusive prefix sums over [0, n) in one CTA of PLAN_SCAN_THREADS threads: store(i, sum of load(0 .. i-1)).
// Returns the total to every thread.
template <class T, class Load, class Store>
__device__ T cta_scan(int64_t n, Load load, Store store) {
    __shared__ T wsum[PLAN_SCAN_THREADS / 32];
    __shared__ T carry_s;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    T carry = 0;
    for (int64_t b = 0; b < n; b += PLAN_SCAN_THREADS) {
        const int64_t i = b + threadIdx.x;
        const T v = i < n ? load(i) : (T)0;
        T s = v;
        for (int d = 1; d < 32; d <<= 1) {
            const T y = __shfl_up_sync(0xffffffffu, s, d);
            if (lane >= d) s += y;
        }
        if (lane == 31) wsum[w] = s;
        __syncthreads();
        if (w == 0) {
            T t = wsum[lane];
            for (int d = 1; d < 32; d <<= 1) {
                const T y = __shfl_up_sync(0xffffffffu, t, d);
                if (lane >= d) t += y;
            }
            wsum[lane] = t;
        }
        __syncthreads();
        const T before = carry + (w ? wsum[w - 1] : (T)0) + s - v;
        if (i < n) store(i, before);
        if (threadIdx.x == PLAN_SCAN_THREADS - 1) carry_s = before + v;
        __syncthreads();
        carry = carry_s;
        __syncthreads();
    }
    return carry;
}

// one CTA: the arena size and the pool's; the histogram becomes the lists' offsets (hist[n_hist] = total), and
// a copy of them the scatter cursors
__global__ void __launch_bounds__(PLAN_SCAN_THREADS) k_plan_offsets(PlanAcc *acc, const unsigned long long *epoch_bytes,
                                                                    int32_t n_epochs, int32_t *hist, int64_t n_hist,
                                                                    int32_t *cur) {
    __shared__ unsigned long long wmax[PLAN_SCAN_THREADS / 32];
    unsigned long long mx = 0;
    for (int32_t e = threadIdx.x; e < n_epochs; e += PLAN_SCAN_THREADS) mx = max(mx, epoch_bytes[e]);
    for (int d = 16; d > 0; d >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, d));
    if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = mx;
    __syncthreads();
    const int32_t total = cta_scan<int32_t>(
        n_hist, [&](int64_t i) { return hist[i]; },
        [&](int64_t i, int32_t v) {
            hist[i] = v;
            cur[i] = v;
        });
    if (threadIdx.x == 0) {
        hist[n_hist] = total;
        for (int k = 0; k < PLAN_SCAN_THREADS / 32; k++) mx = max(mx, wmax[k]);
        const unsigned long long arena = (mx + 255) & ~255ull;
        acc->arena = arena;
        acc->sum.pool_bytes = arena * (unsigned long long)min(3, n_epochs) + acc->long_bytes;
    }
}

// per feature: its final block offset, and its places in the finalize list and (a set) in the zero list
__global__ void __launch_bounds__(256) k_plan_place(const unsigned long long *cand, const int32_t *tlo,
                                                    const int32_t *thi, int32_t m, int32_t epoch_tiles,
                                                    int32_t n_epochs, uint64_t seg_max, uint64_t seg_big,
                                                    PlanAcc *acc, int32_t *cur, int32_t *list, FeatDesc *fdesc,
                                                    uint32_t *segoff16) {
    const int32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    const PlanFeat f = plan_feat(j < m ? cand[j] : 0ull, j < m ? tlo[j] : 0, j < m ? thi[j] : 0, epoch_tiles,
                                 n_epochs, seg_max, seg_big);
    if (f.on) {
        const unsigned long long arena = acc->arena;
        const int n_arenas = min(3, n_epochs);
        const unsigned long long off =
            fdesc[j].blk_off + arena * (unsigned long long)(f.le <= f.fe + 1 ? f.fe % n_arenas : n_arenas);
        fdesc[j].blk_off = off;
        if (!f.set) {
            if (off / 16 >= 0xFFFFFFFFull) atomicOr(&acc->sum.err, 2u);
            segoff16[j] = (uint32_t)(off / 16);
        }
    }
    const int32_t pf = warp_add<int32_t>(f.on, &cur[f.fin_key], 1);
    if (f.on) list[pf] = j;
    const int32_t pz = warp_add<int32_t>(f.set, &cur[(int64_t)3 * n_epochs * PLAN_KEYS + f.fe], 1);
    if (f.set) list[pz] = j;
}

// one CTA: byte prefix of the zero list (set + cursor of each), so that k_zero_segments spreads an epoch's bytes
// evenly over its CTAs
__global__ void __launch_bounds__(PLAN_SCAN_THREADS) k_plan_zero_prefix(const int32_t *zero_lo, const int32_t *zero_hi,
                                                                        const int32_t *list, const FeatDesc *fdesc,
                                                                        unsigned long long *zpre) {
    const int32_t z0 = *zero_lo, z1 = *zero_hi;
    const unsigned long long total = cta_scan<unsigned long long>(
        z1 - z0, [&](int64_t i) { return (unsigned long long)fdesc[list[z0 + i]].cap * 16 + 16; },
        [&](int64_t i, unsigned long long v) { zpre[z0 + i] = v; });
    if (threadIdx.x == 0) zpre[z1] = total;
}

// What a context keeps between calls: the interval index of the last feature set (valid while the caller passes the
// same one), the window jobs of the last call and the pinned slot the plan's summary comes back to.
struct FeatCache {
    bool valid = false;
    xg_input_key key;
    FeatIndexHost ix;
    std::vector<WinJob> jobs;
    PlanSummary *h_sum = nullptr;
};

// Everything the counting kernel needs to know about a tile, in one 64-byte line that the CTA
// fetches two tiles ahead with a bulk copy.
struct __align__(16) TileDesc {
    int64_t rec_beg;
    int32_t n_rec;
    int32_t col;          // sample-ID mode: the column of the tile's BAM
    int32_t bx, by;       // boundaries [bx, by) under the tile's window; bx < 0: no feature, skip
    int32_t st_lo, st_n;  // stabbing entries of the segments [bx, by)
    uint32_t c_lo, c_hi;  // CIGAR words of the tile's records (c_lo one word back: a >=255-op count)
    int32_t jmin;         // smallest sorted-feature index a record of the tile can meet
    int32_t b0, b1;       // boundary range of the contig (windows too wide to stage)
    int32_t pad[3];
};
static_assert(sizeof(TileDesc) == 64, "TileDesc is one 64-byte line");

struct BasefcDev {
    const int2 *pos_end;
    const uint32_t *fmq, *cig_off, *cigar;
    const ulonglong2 *keys;
    const TileDesc *tdesc;
    const int32_t *sf_end, *bnd, *stab_off, *fb;
    const int4 *stab4;            // stabbing lists: {sorted feature, beg, end, segment offset / 16 or NO_SEG}
    const uint32_t *segoff16;     // per sorted feature: the same offset (features met through `fb`)
    uint32_t *seg_cur;            // per sorted feature: pairs appended so far
    uint8_t *pool;
    const FeatDesc *fdesc;
    unsigned int *work;           // tile counter of this launch
    unsigned int *flags;          // bit 0: a UMI key did not fit the pair word (the call is redone with sets)
    int32_t tile0, tile1;         // tiles [tile0, tile1) of this launch (epoch)
    int32_t seg_mode;             // 1: pair words + duplicate filter; 0: every feature is a set
    int32_t col_bits;             // bits of a column index (pair word: umi | col, filter: umi | local feature | col)
    BarcodeTable bc;
    FilterParams fp;
    const int32_t *incl_tab;
    int32_t incl_tab_len, incl_len;
};

struct __align__(16) PairEnt {
    unsigned long long a;         // segment: pair word; set: UMI key
    uint32_t j;                   // sorted feature (| LEGACY_BIT: a set feature)
    uint32_t b;                   // segment: pool offset / 16; set: column
};

struct IdxStage {                 // the slice of the interval index under one tile (bulk-copied) and its filter
    unsigned long long filt[1 << FILT_BITS];       // the tile's duplicate filter (written by the warps)
    int4 stab4[STAB_CAP];
    uint32_t cigar[CIG_CAP + 4];
    int32_t bnd[SB_MAX + 4];
    int32_t stab_off[SB_MAX + 8];
};

struct CountSmem {
    IdxStage idx[2];
    TileDesc desc[4];
    PairEnt pairs[CNT_WARPS][WPAIR_CAP];
    unsigned long long bar_idx[2], bar_desc[4];
    unsigned long long bar_done[2];                // tile k done (every warp, and its buffers freed): bar_done[k & 1]
    int32_t incl[INCL_CAP];
    int t_ring[4];
    int np[CNT_WARPS];
    int chunk_ctr[2];             // next chunk of tile k: chunk_ctr[k & 1] (warps claim chunks)
    int n_done[2];                // warps done with tile k: n_done[k & 1] (the last one frees the buffers)
    int t_pend;                   // the elected lane's pipeline state lives here, not in everybody's registers:
    uint32_t n_issued;            // the tile of the next descriptor to issue; index slices issued so far
};

// ---- mbarrier / bulk-copy (TMA) primitives
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, uint32_t parity) {
    const uint32_t a = smem_u32(bar);
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(a), "r"(parity)
            : "memory");
    } while (!done);
}
// global -> shared bulk copy (16-byte aligned, size a multiple of 16) completing on `bar`
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// Tile descriptors: window of the tile in the interval index (two binary searches), the slice of
// stabbing entries and CIGAR words under it, the smallest feature index it can meet.
__global__ void k_tile_desc(const xg_tile *tiles, const xg_run *runs, int32_t n_tiles, int32_t n_gid,
                            const int32_t *sf_goff, const int32_t *bnd_goff, const int32_t *bnd,
                            const int32_t *stab_off, const int4 *stab4, const int32_t *fb,
                            const uint32_t *cig_off, TileDesc *out) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    const xg_tile tl = tiles[t];
    const xg_run run = runs[tl.run];
    const int32_t gid = run.gid;
    TileDesc d;
    memset(&d, 0, sizeof(d));
    d.rec_beg = tl.rec_beg;
    d.n_rec = tl.n_rec;
    d.col = run.bam_idx;
    d.bx = d.by = -1;
    if (cig_off) {
        const uint32_t c_first = cig_off[tl.rec_beg];
        d.c_lo = c_first ? c_first - 1 : 0;
        d.c_hi = cig_off[tl.rec_beg + tl.n_rec];
    }
    if (gid >= 0 && gid < n_gid && sf_goff[gid] != sf_goff[gid + 1] && bnd_goff[gid] != bnd_goff[gid + 1]) {
        const int32_t b0 = bnd_goff[gid], b1 = bnd_goff[gid + 1];
        int32_t lo = b0, hi = b1;
        while (lo < hi) {              // upper_bound(first_pos)
            int32_t mid = (lo + hi) >> 1;
            if (bnd[mid] <= tl.first_pos) lo = mid + 1; else hi = mid;
        }
        const int32_t x = max(b0, lo - 1);
        hi = b1;
        while (lo < hi) {              // lower_bound(max_end)
            int32_t mid = (lo + hi) >> 1;
            if (bnd[mid] < tl.max_end) lo = mid + 1; else hi = mid;
        }
        const int32_t y = max(x, lo);
        // features that a record of this tile can overlap: those stabbing a segment in [x, y] or
        // beginning at a boundary in (x, y).  None (e.g. another GPU's genomic chunk): skip the tile.
        const int32_t y_seg = min(y + 1, b1);
        const bool any = stab_off[y_seg] > stab_off[x] || fb[y] > fb[min(x + 1, y)];
        if (any) {
            d.bx = x;
            d.by = y;
            d.st_lo = stab_off[x];
            d.st_n = stab_off[y] - d.st_lo;
            d.b0 = b0;
            d.b1 = b1;
            d.jmin = stab_off[x + 1] > stab_off[x] ? stab4[stab_off[x]].x : fb[min(x + 1, b1)];
        }
    }
    out[t] = d;
}

// streaming calls: the CIGAR range of a tile is known once its records are in HBM
__global__ void k_tile_cig(const xg_tile *tiles, int32_t t0, int32_t t1, const uint32_t *cig_off, TileDesc *out) {
    int t = t0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= t1) return;
    const xg_tile tl = tiles[t];
    const uint32_t c_first = cig_off[tl.rec_beg];
    out[t].c_lo = c_first ? c_first - 1 : 0;
    out[t].c_hi = cig_off[tl.rec_beg + tl.n_rec];
}

// per call: the segment offsets of the plan go into the stabbing entries
__global__ void k_patch_stab(int4 *stab4, int32_t n, const uint32_t *segoff16) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) stab4[k].w = (int32_t)segoff16[stab4[k].x];
}

__device__ __forceinline__ uint32_t set_home(uint64_t umi, uint32_t col, uint32_t cap) {
    return hash_to_range(mix64(umi ^ ((uint64_t)col * 0x9E3779B97F4A7C15ULL)), cap);
}

// (cell, UMI) -> the feature's set, starting at slot s whose content `cur` was already loaded.
// Empty slot: b == 0.  Returns true when the element is new.
__device__ __forceinline__ bool set_insert_from(xg_e128 *tbl, uint32_t cap, uint32_t s, xg_e128 cur,
                                                xg_e128 want) {
    for (uint32_t probe = 0; probe < cap; probe++) {
        if (cur.b == 0) {
            xg_e128 empty;
            empty.a = 0;
            empty.b = 0;
            cur = cas128(&tbl[s], empty, want);
            if (cur.b == 0) return true;
        }
        if (cur.a == want.a && cur.b == want.b) return false;
        s = (s + 1 == cap) ? 0 : s + 1;
        cur = ld128_relaxed(&tbl[s]);
    }
    return false;
}

// Append the cell of a new element to the feature's log.  Lanes of the warp that append to
// the same feature are grouped with match_any: one cursor atomic per group.  Whole warp.
__device__ __forceinline__ void log_append(xg_e128 *tbl, uint32_t cap, bool is_new, uint32_t col) {
    const unsigned active = __ballot_sync(0xffffffffu, is_new);
    if (!is_new) return;
    const unsigned peers = __match_any_sync(active, (unsigned long long)tbl);
    const int leader = __ffs(peers) - 1, lane = threadIdx.x & 31;
    uint32_t *cursor = (uint32_t *)(tbl + cap);
    uint32_t base = 0;
    if (lane == leader) base = atomicAdd(cursor, (uint32_t)__popc(peers));
    base = __shfl_sync(peers, base, leader);
    uint32_t *log = cursor + 4;
    log[base + __popc(peers & ((1u << lane) - 1u))] = col;
}

__device__ __forceinline__ void set_insert_direct(const BasefcDev &P, uint32_t j, uint64_t umi, uint32_t col) {
    const FeatDesc fd = P.fdesc[j];
    if (!fd.cap) return;
    xg_e128 want;
    want.a = umi;
    want.b = (unsigned long long)col + 1ull;
    xg_e128 *tbl = (xg_e128 *)(P.pool + fd.blk_off);
    const uint32_t s = set_home(umi, col, fd.cap);
    if (set_insert_from(tbl, fd.cap, s, ld128_relaxed(&tbl[s]), want)) {
        uint32_t *cursor = (uint32_t *)(tbl + fd.cap);
        cursor[4 + atomicAdd(cursor, 1u)] = col;
    }
}

// m = number of aligned (M/=/X) reference positions p of the read with s0 <= p < e0
// (== len([x for x in read.positions if s <= x <= e]), rdr/fc/core.py:40-43)
__device__ __forceinline__ int32_t included_len(const uint32_t *cig, uint32_t n_ops, int32_t pos,
                                                 int32_t s0, int32_t e0) {
    int32_t m = 0, p = pos;
    for (uint32_t k = 0; k < n_ops; k++) {
        uint32_t w = cig[k], op = w & 15u;
        int32_t l = (int32_t)(w >> 4);
        if (cig_aligned(op)) {
            int32_t a = max(p, s0), b = min(p + l, e0);
            if (b > a) m += b - a;
            p += l;
        } else if (cig_skips_ref(op)) {
            p += l;
        }
    }
    return m;
}

// what a lane knows about the record it is working on
struct RecCtx {
    int32_t pos, end, aln, need;
    const uint32_t *cig;
    uint32_t n_ops, col;
    uint64_t umi;         // the UMI key as stored
    uint64_t umi_c;       // ... with its low 24 bits free (seg_mode)
};

// The warp's staged pairs go to their features: a segment pair is appended at a cursor position
// reserved once per (warp, feature) group (match_any); a set pair is inserted with a 128-bit CAS.
__device__ __forceinline__ void flush_warp(const BasefcDev &P, CountSmem &S, int w, int lane) {
    __syncwarp();
    const int np = min(__shfl_sync(0xffffffffu, S.np[w], 0), WPAIR_CAP);     // one value for the whole warp
    for (int p0 = 0; p0 < np; p0 += 32) {
        const int p = p0 + lane;
        const bool act = p < np;
        PairEnt e;
        e.a = 0;
        e.j = 0;
        e.b = 0;
        if (act) e = S.pairs[w][p];
        const bool seg = act && !(e.j & LEGACY_BIT);
        const unsigned segm = __ballot_sync(0xffffffffu, seg);
        if (seg) {
            const unsigned peers = __match_any_sync(segm, e.j);
            const int leader = __ffs(peers) - 1;
            uint32_t base = 0;
            if (lane == leader) base = atomicAdd(&P.seg_cur[e.j], (uint32_t)__popc(peers));
            base = __shfl_sync(peers, base, leader);
            const uint32_t at = base + (uint32_t)__popc(peers & ((1u << lane) - 1u));
            *(unsigned long long *)(P.pool + (uint64_t)e.b * 16 + (uint64_t)at * 8) = e.a;
        }
        const bool leg = act && !seg;
        if (__ballot_sync(0xffffffffu, leg)) {
            xg_e128 *tbl = nullptr;
            uint32_t cap = 0;
            bool is_new = false;
            if (leg) {
                const FeatDesc fd = P.fdesc[e.j & ~LEGACY_BIT];
                if (fd.cap) {
                    cap = fd.cap;
                    tbl = (xg_e128 *)(P.pool + fd.blk_off);
                    xg_e128 want;
                    want.a = e.a;
                    want.b = (unsigned long long)e.b + 1ull;
                    const uint32_t s = set_home(e.a, e.b, cap);
                    is_new = set_insert_from(tbl, cap, s, ld128_relaxed(&tbl[s]), want);
                }
            }
            log_append(tbl, cap, is_new, e.b);
        }
    }
    __syncwarp();
    if (lane == 0) S.np[w] = 0;
    __syncwarp();
}

// include test of one (read, feature) pair; a passing pair that the tile has not seen yet is staged
__device__ __forceinline__ void emit_pair(const BasefcDev &P, CountSmem &S, unsigned long long *filt, int32_t jmin,
                                          int w, const RecCtx &r, int32_t j, int32_t s0, int32_t e0, uint32_t segoff) {
    int32_t m;
    if (r.n_ops == 0) {
        int32_t a = max(r.pos, s0), b = min(r.end, e0);
        m = b > a ? b - a : 0;
    } else if (s0 <= r.pos && r.end <= e0) {
        m = r.aln;                // the read lies inside the feature: every aligned position counts
    } else {
        m = included_len(r.cig, r.n_ops, r.pos, s0, e0);
    }
    if (m < r.need) return;
    if (P.seg_mode) {
        // duplicate filter: (UMI, feature, cell) fits 64 bits when the feature is numbered from the
        // tile's first one.  A hit means that the same triple went out earlier in this tile; a miss
        // (or a triple the filter cannot express) is passed on -- the features' own dedup is exact.
        const uint32_t jl = (uint32_t)(j - jmin);
        if (jl < (1u << (24 - P.col_bits))) {
            const unsigned long long fk = r.umi_c | ((unsigned long long)jl << P.col_bits) | r.col;
            const uint32_t h = ((((uint32_t)fk * 0x85EBCA6Bu) ^ (uint32_t)(fk >> 32)) * 0x9E3779B1u) >> (32 - FILT_BITS);
            if (filt[h] == fk) return;
            filt[h] = fk;
        }
    }
    const bool seg = segoff != NO_SEG;
    // the counter is the warp's own: only lanes of this warp contend for it
    const int slot = atomicAdd(&S.np[w], 1);
    if (slot < WPAIR_CAP) {
        PairEnt e;
        if (seg) {
            e.a = r.umi_c | r.col;
            e.j = (uint32_t)j;
            e.b = segoff;
        } else {
            e.a = r.umi;
            e.j = (uint32_t)j | LEGACY_BIT;
            e.b = r.col;
        }
        S.pairs[w][slot] = e;
    } else if (seg) {              // stage full (very deep feature overlap): append right away
        const uint32_t at = atomicAdd(&P.seg_cur[j], 1u);
        *(unsigned long long *)(P.pool + (uint64_t)segoff * 16 + (uint64_t)at * 8) = r.umi_c | r.col;
    } else {
        set_insert_direct(P, (uint32_t)j, r.umi, r.col);
    }
}

// the tile's fields the record path needs, read once per tile into registers
struct TileRegs {
    int32_t bx, by, b0, st_lo, jmin;
    const TileDesc *td;           // the rest stays in shared memory (the contig's last boundary: wide windows only)
    uint32_t c_al;
    bool staged, stab_staged, cig_staged;
};

// One record: filters (check_read), the features it overlaps, include test per feature.
__device__ __forceinline__ void count_record(const BasefcDev &P, CountSmem &S, const TileRegs &T, IdxStage &X,
                                             int w, int2 pe, uint32_t fmq, uint32_t co, uint64_t umi,
                                             int32_t colv) {
    if (umi == XG_KEY_NONE || umi == XG_KEY_EMPTY) return;       // has_tag / `if umi:`
    if (!read_passes_flags(P.fp, fmq)) return;
    if (colv < 0) return;                                         // cell tag absent or not listed
    RecCtx r;
    r.umi = umi;
    r.umi_c = umi;
    r.col = (uint32_t)colv;
    if (P.seg_mode) {
        if (umi >> 63) {                                          // interned id: moved above the column bits
            const unsigned long long id = umi & 0x7fffffffffffffffULL;
            if (id >> 39) {
                atomicOr(P.flags, 1u);
                return;
            }
            r.umi_c = (1ULL << 63) | (id << 24);
        } else if (umi & 0xffffffULL) {                           // packed string longer than 13 symbols
            atomicOr(P.flags, 1u);
            return;
        }
    }
    r.pos = pe.x;
    r.end = pe.y;
    r.n_ops = fmq >> 24;                      // aligned length = len(read.positions)
    r.cig = nullptr;
    if (r.n_ops == 0) {
        r.aln = r.end - r.pos;
    } else {
        r.cig = T.cig_staged ? &X.cigar[co - T.c_al] : P.cigar + co;
        if (r.n_ops == 255) r.n_ops = r.cig[-1];
        int32_t aln = 0;
        for (uint32_t q = 0; q < r.n_ops; q++) {
            const uint32_t cw = r.cig[q];
            if (cig_aligned(cw & 15u)) aln += (int32_t)(cw >> 4);
        }
        r.aln = aln;
    }
    if (r.aln < P.fp.min_len) return;
    if (P.incl_tab) {
        const int32_t k = min(r.aln, P.incl_tab_len - 1);
        r.need = k < INCL_CAP ? S.incl[k] : __ldg(&P.incl_tab[k]);
    } else {
        r.need = P.incl_len;
    }

    // first boundary > pos (global index)
    const int32_t nb = T.by - T.bx;
    int32_t ub;
    if (T.staged) {
        const int32_t *sb = X.bnd + (T.bx - (T.bx & ~3));
        int32_t lo = 0;
        if (nb <= 8) {                         // few boundaries under the tile: branch-free count
            for (int k = 0; k < nb; k++) lo += sb[k] <= r.pos;
        } else {
            int32_t hi = nb;
            while (lo < hi) {
                int32_t mid = (lo + hi) >> 1;
                if (sb[mid] <= r.pos) lo = mid + 1; else hi = mid;
            }
        }
        ub = T.bx + lo;
    } else {
        int32_t lo = T.b0, hi = T.td->b1;
        while (lo < hi) {
            int32_t mid = (lo + hi) >> 1;
            if (__ldg(&P.bnd[mid]) <= r.pos) lo = mid + 1; else hi = mid;
        }
        ub = lo;
    }
    // (1) features covering `pos`: stabbing list of the segment [bnd[ub-1], bnd[ub])
    if (ub > T.b0) {
        int32_t s0i, s1i;
        if (T.staged && ub > T.bx) {
            s0i = X.stab_off[ub - 1 - (T.bx & ~3)];
            s1i = X.stab_off[ub - (T.bx & ~3)];
        } else {
            s0i = __ldg(&P.stab_off[ub - 1]);
            s1i = __ldg(&P.stab_off[ub]);
        }
        for (int32_t s = s0i; s < s1i; s++) {
            const int4 f = (T.stab_staged && s >= T.st_lo) ? X.stab4[s - T.st_lo] : __ldg(&P.stab4[s]);
            emit_pair(P, S, X.filt, T.jmin, w, r, f.x, f.y, f.z, (uint32_t)f.w);
        }
    }
    // (2) features beginning at a boundary inside (pos, end); every boundary from `by` on is
    // >= the tile's max end, so a staged tile never looks past its staged range
    const int32_t kb_end = T.staged ? T.by : T.td->b1;
    for (int32_t kb = ub; kb < kb_end; kb++) {
        const int32_t bv = T.staged ? X.bnd[kb - (T.bx & ~3)] : __ldg(&P.bnd[kb]);
        if (bv >= r.end) break;
        const int32_t j1 = __ldg(&P.fb[kb + 1]);
        for (int32_t j = __ldg(&P.fb[kb]); j < j1; j++)
            emit_pair(P, S, X.filt, T.jmin, w, r, j, bv, __ldg(&P.sf_end[j]), __ldg(&P.segoff16[j]));
    }
}

// Persistent CTAs take tiles from a work counter.  Inside a tile the warps work on their own: 32-record chunks
// claimed from a counter, the record loads issued one chunk ahead, pairs staged per warp and appended per warp.
// There is no CTA barrier: the state of a tile is double-buffered -- its chunk counter by the tile's parity, its
// index stage and duplicate filter by the parity of the live tiles counted so far -- and a warp that runs out of
// chunks in tile k goes on to tile k+1 as soon as tile k-1 has freed its buffers: warps are at most one tile apart.
// A warp arrives on tile k's "done" mbarrier when it has flushed its pairs of the tile; the last of them first
// clears the tile's filter and chunk counter for their next user and moves the staging pipeline on (elected lane: tile k+4's index fetched from the counter, tile k+3's descriptor and
// tile k+2's slice of the interval index -- boundaries, stabbing lists, CIGAR words -- brought into shared memory by
// bulk copies completing on mbarriers), then arrives: the phase completes only when the buffers are free.
template <int MIN_CTAS>
__global__ void __launch_bounds__(CNT_THREADS, MIN_CTAS) k_basefc_count(const __grid_constant__ BasefcDev P) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    CountSmem &S = *reinterpret_cast<CountSmem *>(smem_raw);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int32_t n_launch = P.tile1 - P.tile0;

    if (threadIdx.x == 0) {
        for (int k = 0; k < 2; k++) mbar_init(&S.bar_idx[k], 1);
        for (int k = 0; k < 4; k++) mbar_init(&S.bar_desc[k], 1);
        for (int k = 0; k < 2; k++) mbar_init(&S.bar_done[k], CNT_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (threadIdx.x < CNT_WARPS) S.np[threadIdx.x] = 0;
    if (threadIdx.x < 2) S.chunk_ctr[threadIdx.x] = S.n_done[threadIdx.x] = 0;
    if (P.seg_mode)                  // both filters start empty; afterwards the last user of a stage clears it
        for (int q = threadIdx.x; q < 2 << FILT_BITS; q += CNT_THREADS) S.idx[q >> FILT_BITS].filt[q & ((1 << FILT_BITS) - 1)] = 0;
    if (P.incl_tab)
        for (int k = threadIdx.x; k < INCL_CAP && k < P.incl_tab_len; k += CNT_THREADS) S.incl[k] = __ldg(&P.incl_tab[k]);

    // ---- elected lane: state of the staging pipeline
    // S.t_pend: the tile of the next descriptor to issue; S.n_issued: index slices issued so far (buffer = n & 1,
    // parity = (n >> 1) & 1)
    auto fetch_tile = [&]() -> int {
        const unsigned int v = atomicAdd(P.work, 1u);
        return v < (unsigned int)n_launch ? P.tile0 + (int)v : -1;
    };
    auto issue_desc = [&](int k, int t) {         // descriptor of tile t -> ring slot k & 3
        S.t_ring[k & 3] = t;
        if (t < 0) return;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx(&S.bar_desc[k & 3], (uint32_t)sizeof(TileDesc));
        bulk_g2s(&S.desc[k & 3], &P.tdesc[t], (uint32_t)sizeof(TileDesc), &S.bar_desc[k & 3]);
    };
    auto issue_idx = [&](int k) {                 // the slice of the index under tile k (if live) -> next buffer
        if (S.t_ring[k & 3] < 0) return;
        mbar_wait(&S.bar_desc[k & 3], (uint32_t)(k >> 2) & 1u);
        const TileDesc &d = S.desc[k & 3];
        if (d.bx < 0) return;
        IdxStage &X = S.idx[S.n_issued & 1];
        unsigned long long *bar = &S.bar_idx[S.n_issued & 1];
        S.n_issued++;
        const int32_t bx_al = d.bx & ~3;
        const uint32_t c_al = d.c_lo & ~3u;
        uint32_t n_bnd = 0, n_so = 0, n_st = 0, n_cg = 0;
        if (d.by - bx_al <= SB_MAX) {
            n_bnd = (uint32_t)((d.by - bx_al + 3) & ~3) * 4u;
            n_so = (uint32_t)((d.by + 1 - bx_al + 3) & ~3) * 4u;
            if (d.st_n <= STAB_CAP) n_st = (uint32_t)d.st_n * 16u;
        }
        if (d.c_hi - c_al <= CIG_CAP) n_cg = ((d.c_hi - c_al + 3u) & ~3u) * 4u;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx(bar, n_bnd + n_so + n_st + n_cg);
        if (n_bnd) bulk_g2s(X.bnd, P.bnd + bx_al, n_bnd, bar);
        if (n_so) bulk_g2s(X.stab_off, P.stab_off + bx_al, n_so, bar);
        if (n_st) bulk_g2s(X.stab4, P.stab4 + d.st_lo, n_st, bar);
        if (n_cg) bulk_g2s(X.cigar, P.cigar + c_al, n_cg, bar);
    };
    if (threadIdx.x == 0) {
        S.n_issued = 0;
        for (int k = 0; k < 3; k++) issue_desc(k, fetch_tile());
        S.t_pend = fetch_tile();
        issue_idx(0);
        issue_idx(1);
    }
    __syncthreads();                 // the only CTA barrier: initial state and the pipeline's first stages

    uint32_t n_used = 0;             // index slices consumed so far (every thread counts alike)
    // Warp done with tile k (its pairs flushed).  The last warp of the tile frees the tile's buffers -- nobody touches
    // its filter, chunk counter or index stage any more -- before it arrives.
    auto tile_done = [&](int k) {
        const int s = k & 1;
        __syncwarp();
        int last = 0;
        if (lane == 0) {
            __threadfence_block();
            last = atomicAdd(&S.n_done[s], 1) == CNT_WARPS - 1;
            __threadfence_block();
        }
        if (__shfl_sync(0xffffffffu, last, 0)) {
            __syncwarp();
            if (S.desc[k & 3].bx >= 0 && P.seg_mode) {     // a live tile's filter is its stage's: (n_used - 1) & 1
                uint4 *f4 = reinterpret_cast<uint4 *>(S.idx[(n_used - 1) & 1].filt);
                for (int q = lane; q < (1 << FILT_BITS) / 2; q += 32) f4[q] = make_uint4(0, 0, 0, 0);
            }
            if (lane == 0) {
                S.chunk_ctr[s] = 0;
                S.n_done[s] = 0;
                const int t = S.t_pend;
                S.t_pend = t >= 0 ? fetch_tile() : -1;
                issue_desc(k + 3, t);
                issue_idx(k + 2);
            }
            __syncwarp();
        }
        if (lane == 0) mbar_arrive(&S.bar_done[s]);
    };
    // tile k's parity is free once tile k-2 is done with it
    auto wait_parity = [&](int k) {
        if (k >= 2) mbar_wait(&S.bar_done[k & 1], (uint32_t)((k - 2) >> 1) & 1u);
    };

    // A warp that runs out of chunks in tile k claims its first chunk of tile k+1 and issues that chunk's record
    // loads before it flushes its pairs of tile k: the loads' DRAM latency passes under the flush.
    int pre_c = -1;
    int2 pe_n = make_int2(0, 0);
    uint32_t fq_n = 0, co_n = 0;
    ulonglong2 ky_n = make_ulonglong2(XG_KEY_NONE, XG_KEY_NONE);

    for (int k = 0;; k++) {
        if (S.t_ring[k & 3] < 0) break;
        wait_parity(k);
        mbar_wait(&S.bar_desc[k & 3], (uint32_t)(k >> 2) & 1u);
        const TileDesc &td = S.desc[k & 3];          // stays put until tile k+1 is done with
        if (td.bx >= 0) {                  // no feature under a dead tile's window: its records are never read
            IdxStage &X = S.idx[n_used & 1];
            mbar_wait(&S.bar_idx[n_used & 1], (n_used >> 1) & 1u);
            n_used++;

            TileRegs T;
            T.bx = td.bx;
            T.by = td.by;
            T.b0 = td.b0;
            T.td = &td;
            T.st_lo = td.st_lo;
            T.jmin = td.jmin;
            T.c_al = td.c_lo & ~3u;
            T.staged = T.by - (T.bx & ~3) <= SB_MAX;
            T.stab_staged = T.staged && td.st_n <= STAB_CAP;
            T.cig_staged = td.c_hi - T.c_al <= CIG_CAP;
            const int64_t rec_beg = td.rec_beg;
            const int32_t n_rec = td.n_rec, tile_col = td.col;
            const int n_chunks = (n_rec + CHUNK - 1) / CHUNK;

            // ---- the warp's chunks, claimed from the tile's counter one ahead: the records of the next
            // chunk are on their way (coalesced 8 / 4 / 4 / 16-byte loads) while this one is counted.  (A third
            // stage that also kept the next chunk's barcode slot in flight was measured slower: the registers
            // it needs spill.)
            auto claim = [&]() -> int {
                int c = 0;
                if (lane == 0) c = atomicAdd(&S.chunk_ctr[k & 1], 1);
                return __shfl_sync(0xffffffffu, c, 0);
            };
            auto load_from = [&](int64_t beg, int32_t n, int c) {
                const int r = c * CHUNK + lane;
                ky_n = make_ulonglong2(XG_KEY_NONE, XG_KEY_NONE);            // an absent UMI drops the record
                if (r < n) {
                    const int64_t i = beg + r;
                    pe_n = __ldcs(&P.pos_end[i]);                             // streamed once: evict-first
                    fq_n = __ldcs(&P.fmq[i]);
                    co_n = __ldcs(&P.cig_off[i]);
                    ky_n = __ldcs(&P.keys[i]);
                }
            };
            auto load_chunk = [&](int c) { load_from(rec_beg, n_rec, c); };
            int c = pre_c;
            if (c < 0) {             // nothing claimed at the end of the previous tile
                c = claim();
                if (c < n_chunks) load_chunk(c);
            }
            pre_c = -1;
            while (c < n_chunks) {
                const int2 pe = pe_n;
                const uint32_t fq = fq_n, co = co_n;
                const ulonglong2 ky = ky_n;
                const int cn = claim();
                if (cn < n_chunks) load_chunk(cn);
                // cell lookup
                int32_t colv = tile_col;
                if (P.fp.use_cell_tag) {
                    colv = -1;
                    if (ky.x != XG_KEY_NONE) {
                        uint32_t sl = barcode_home(ky.x, P.bc.shift);
                        while (true) {
                            const ulonglong2 e = __ldg(&P.bc.slots[sl]);
                            if (e.x == ky.x) {
                                colv = (int32_t)e.y;
                                break;
                            }
                            if (e.x == XG_KEY_NONE) break;
                            sl = (sl + 1) & P.bc.mask;
                        }
                    }
                }
                count_record(P, S, T, X, w, pe, fq, co, ky.y, colv);
                __syncwarp();
                // Append the staged pairs when the stage is more than half full (32 at a time keep the lanes
                // busy).  The decision is lane 0's: a lane reading the counter for itself could see it already
                // raised by lanes that went on to the next record, and part ways with them.
                if (__shfl_sync(0xffffffffu, S.np[w], 0) > WPAIR_CAP / 2) flush_warp(P, S, w, lane);
                c = cn;
            }
            // the first chunk of the next tile (its descriptor arrived two tiles ago; its parity's counter is reset
            // once tile k-1 is done)
            if (S.t_ring[(k + 1) & 3] >= 0) {
                wait_parity(k + 1);
                mbar_wait(&S.bar_desc[(k + 1) & 3], (uint32_t)((k + 1) >> 2) & 1u);
                const TileDesc &nd = S.desc[(k + 1) & 3];
                if (nd.bx >= 0) {
                    int cx = 0;
                    if (lane == 0) cx = atomicAdd(&S.chunk_ctr[(k + 1) & 1], 1);
                    pre_c = __shfl_sync(0xffffffffu, cx, 0);
                    if (pre_c * CHUNK < nd.n_rec) load_from(nd.rec_beg, nd.n_rec, pre_c);
                }
            }
            flush_warp(P, S, w, lane);
        }
        tile_done(k);
    }
}

// "narrow" result entries: column | count << 16; a count that does not fit goes to the side list
__global__ void k_pack_rows(const int32_t *col, const int32_t *val, uint32_t *packed, long long from, long long to,
                            long long *over_idx, int32_t *over_val, unsigned int *over_n, unsigned int over_cap) {
    const long long i = from + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= to) return;
    const uint32_t c = (uint32_t)col[i], v = (uint32_t)val[i];
    uint32_t v16 = v;
    if (v >= 0xffffu) {
        v16 = 0xffffu;
        const unsigned int k = atomicAdd(over_n, 1u);
        if (k < over_cap) {
            over_idx[k] = i;
            over_val[k] = (int32_t)v;
        }
    }
    packed[i] = c | (v16 << 16);
}

// "tiny" result entries (XG_LAYOUT_ROWS_TINY): 16 bits each -- (column - previous column of the row - 1) << 4 | count.
// An entry that does not fit (the first of its row, a gap of more than 4095 columns, a count above 15) is the word
// 0 and goes to the side list with its column and count.  A quarter of the bytes of (col, val) pairs.
__global__ void k_mark_row_starts(const int64_t *seg_base, const int32_t *seg_nnz, int32_t n_rows, uint32_t *bits) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows || seg_nnz[r] <= 0) return;
    const int64_t i = seg_base[r];
    atomicOr(&bits[i >> 5], 1u << (i & 31));
}
__global__ void k_pack_rows_tiny(const int32_t *col, const int32_t *val, const uint32_t *row_start, uint16_t *tiny,
                                 long long from, long long to, long long *over_idx, int32_t *over_col, int32_t *over_val,
                                 unsigned int *over_n, unsigned int over_cap) {
    const long long i = from + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= to) return;
    const uint32_t c = (uint32_t)col[i], v = (uint32_t)val[i];
    const bool first = (row_start[i >> 5] >> (i & 31)) & 1u;
    const uint32_t d = first ? 0xFFFFFFFFu : c - (uint32_t)col[i - 1] - 1u;     // columns ascend within a row
    uint32_t w = 0;
    if (d <= 4094u && v >= 1u && v <= 15u) {
        w = (d << 4) | v;
    } else {
        const unsigned int k = atomicAdd(over_n, 1u);
        if (k < over_cap) {
            over_idx[k] = i;
            over_col[k] = (int32_t)c;
            over_val[k] = (int32_t)v;
        }
    }
    tiny[i] = (uint16_t)w;
}

__global__ void k_snapshot_cursor(const unsigned long long *cursor, unsigned long long *host_slot) {
    *host_slot = *cursor;
    __threadfence_system();
}

// Zero the sets of the features that become active in this epoch: the zero list's entries [*lo, *hi), laid end to
// end in a virtual byte space (pre = byte prefix of the list, k_plan_zero_prefix).  CTAs stride over its chunks.
#define ZERO_CHUNK 16384
__global__ void __launch_bounds__(256) k_zero_segments(uint8_t *pool, const FeatDesc *fdesc, const int32_t *list,
                                                       const unsigned long long *pre, const int32_t *lo_p,
                                                       const int32_t *hi_p) {
    const int32_t lo = *lo_p, hi = *hi_p;
    if (hi <= lo) return;
    const uint64_t base = pre[lo], total = pre[hi] - base;
    const uint4 z = make_uint4(0, 0, 0, 0);
    for (uint64_t c0 = (uint64_t)blockIdx.x * ZERO_CHUNK; c0 < total; c0 += (uint64_t)gridDim.x * ZERO_CHUNK) {
        int32_t a = lo, b = hi;          // last entry with pre <= c0
        while (b - a > 1) {
            int32_t mid = (a + b) >> 1;
            if (pre[mid] - base <= c0) a = mid; else b = mid;
        }
        int32_t s = a;
        uint64_t s_beg = pre[s] - base, s_end = pre[s + 1] - base;
        uint8_t *blk = pool + fdesc[list[s]].blk_off;
        for (uint64_t p = c0 + (uint64_t)threadIdx.x * 16; p < c0 + ZERO_CHUNK && p < total;
             p += (uint64_t)blockDim.x * 16) {
            while (p >= s_end) {
                s++;
                s_beg = s_end;
                s_end = pre[s + 1] - base;
                blk = pool + fdesc[list[s]].blk_off;
            }
            *(uint4 *)(blk + (p - s_beg)) = z;
        }
    }
}

// ---- finalize: a feature whose last epoch just finished becomes its row of the matrix -----------------
// The non-zeros of a row leave in column order (the reference's emit loop, rdr/fc/core.py:109-117), to a
// staging area at an atomically reserved offset; k_gather_rows puts the rows in input order.  Persistent
// CTAs take features from a work counter.
//
// Segment features (k_basefc_finalize_segs).  The feature's pair words (umi | cell; duplicates across
// tiles are still in) are reduced in shared memory by small CTAs, five to an SM, so that one feature's
// latencies hide behind another's:
//   phase 1  every word sets the bit of its cell in a bitmap over all cells; the prefix popcounts of the
//            bitmap give the row's size (reserved right away) and every cell's rank in the row;
//   phase 2  the words go into an open-addressing table (64-bit CAS); every NEW word adds one to a counter
//            indexed by its cell's rank;
//   output   cell / counter pairs in rank order.
// A light feature (<= FS_CAP words) keeps its words in registers between the phases.  A heavy one is first
// split by column range into the scratch half of its block (count, prefix, scatter: two sweeps from L2), so
// that a range's words fit the table and its cells the counters; ranges go through phase 2 one after
// the other.  A range that still holds too many words (skewed cells) is swept once per hash sub-partition,
// with twice the sub-partitions after a table overflow.
#define FS_THREADS 256                // CTA of the features of ordinary size, four or five to an SM
#define FS_BIG_THREADS 1024           // CTA of a big feature (its passes are bound by the loads one CTA keeps in flight,
                                      // and by a barrier + a memory round trip per column range)
#define FS_TBL SEG_TBL_SLOTS          // table slots (64-bit)
#define FS_CAP SEG_PART_WORDS         // words a table pass should hold (40 % load); also the rank counters
#define FS_REG 7                      // words a thread keeps in registers (FS_REG * FS_THREADS >= FS_CAP)
#define FS_RANGES 1024                // column ranges of a heavy feature (counters live in the idle table)
#define FS_TBL_LOG2 12                // ordinary CTAs: 4096-slot table (FS_TBL)
#define FS_BIG_TBL_LOG2 14            // big CTAs: 16384 slots -- a quarter of the ranges, each a barrier and a round trip
#define FS_STATS 8                    // route counters of the two instantiations (xg_basefc_finalize_stats)
static_assert((1 << FS_TBL_LOG2) == FS_TBL, "table size");

__device__ __forceinline__ uint64_t pair_hash(unsigned long long pw) {
    uint64_t h = pw * 0x9E3779B97F4A7C15ULL;
    h ^= h >> 29;
    h *= 0xBF58476D1CE4E5B9ULL;
    return h;
}

struct FsShared {
    uint32_t warp_tot[32];
    long long base_s;
    int ovf_s;
    int ovf_b[2];                     // ... of the fast range passes, one per counter bank
    int f_s[2];                       // this / the next work item (fetched one ahead)
    uint32_t range_off[FS_RANGES + 1];
};

// table of a pass over n words: a power of two >= 2.5 n, 64 .. FS_TBL slots
__device__ __forceinline__ uint32_t fs_table_size(uint32_t n, uint32_t tbl_max = FS_TBL) {
    uint32_t tsz = 64;
    while (tsz < tbl_max && tsz * 2 < n * 5) tsz <<= 1;
    return tsz;
}

// rank of cell `col` in the row: set bits below it
__device__ __forceinline__ uint32_t fs_rank(const uint32_t *bitmap, const uint32_t *pre, uint32_t col) {
    return pre[col >> 5] + (uint32_t)__popc(bitmap[col >> 5] & ((1u << (col & 31)) - 1u));
}

// one word into the table; a NEW word counts for its cell.  false: the table is too full
__device__ __forceinline__ bool fs_insert(unsigned long long *tbl, uint32_t tsz, int shift, unsigned long long pw,
                                          uint64_t h, uint32_t *cnt, uint32_t r, uint32_t probe_max) {
    uint32_t slot = (uint32_t)((h * 0x9E3779B97F4A7C15ULL) >> shift);
    for (uint32_t probe = 0; probe < probe_max; probe++) {
        const unsigned long long old = atomicCAS(&tbl[slot], 0ULL, pw);
        if (old == 0ULL) {
            atomicAdd(&cnt[r], 1u);
            return true;
        }
        if (old == pw) return true;
        slot = (slot + 1) & (tsz - 1);
    }
    return false;
}

// The same for the ranges of a heavy feature, which go through the table one after the other WITHOUT clearing it:
// every word carries its range in the upper bits of its cell, so an entry of an earlier range is as good as an
// empty slot and is overwritten in place.  (The table is cleared once per feature.)
template <int TBL_LOG2>
__device__ __forceinline__ bool fs_insert_range(unsigned long long *tbl, unsigned long long pw, uint64_t h, uint32_t rg,
                                                int wshift, uint32_t *cnt, uint32_t r) {
    constexpr uint32_t TBL = 1u << TBL_LOG2;
    uint32_t slot = (uint32_t)((h * 0x9E3779B97F4A7C15ULL) >> (64 - TBL_LOG2));
    for (uint32_t probe = 0; probe < 96;) {
        const unsigned long long old = *(volatile unsigned long long *)&tbl[slot];
        if (old == pw) return true;
        if (old != 0ULL && (((uint32_t)old & 0xffffffu) >> wshift) == rg) {     // a word of this range: next slot
            slot = (slot + 1) & (TBL - 1);
            probe++;
            continue;
        }
        if (atomicCAS(&tbl[slot], old, pw) == old) {
            atomicAdd(&cnt[r], 1u);
            return true;
        }
        // lost the slot to another word of this range (or to this very word): look at it again
    }
    return false;
}

// 48 registers: five ordinary CTAs fit an SM, and an SM that holds a big CTA has room for an ordinary one
template <int THREADS, int TBL_LOG2>
__global__ void __maxnreg__(48) k_basefc_finalize_segs(
    const uint8_t *pool, const FeatDesc *fdesc, const uint32_t *seg_cur, const int32_t *sf_row,
    const int32_t *fin_list, const int32_t *fin_lo, const int32_t *fin_hi, int32_t n_cols, unsigned int *work,
    unsigned long long *cursor, int64_t *seg_base, int32_t *seg_nnz, int32_t *st_col, int32_t *st_val,
    unsigned long long *stats) {
    extern __shared__ __align__(16) uint8_t fin_smem[];
    // the epoch's features: a range of the plan's finalize list (surplus CTAs of the fixed grid leave at once)
    const int32_t *fin_feat = fin_list + *fin_lo;
    const int32_t n_fin = *fin_hi - *fin_lo;
    // table slots; words a table pass should hold (40 % load: the light / heavy limit); cells of a range on the fast
    // path = one counter bank; the counters (a light feature uses both banks as one)
    constexpr uint32_t TBL = 1u << TBL_LOG2, CAP = TBL * 2 / 5, RCELLS = TBL / 4, CNT = 2 * RCELLS;
    constexpr uint32_t LIGHT = CAP < FS_REG * THREADS ? CAP : FS_REG * THREADS;     // words a CTA keeps in registers
    static_assert(LIGHT >= SEG_PART_WORDS, "a feature without a scratch half must be light");
    // xg_basefc_finalize_stats: heavy features, careful ranges, fast-range overflows, sub-partition doublings
    if (THREADS == FS_BIG_THREADS) stats += FS_STATS / 2;
    const int bm_words = (n_cols + 31) >> 5;
    unsigned long long *tbl = reinterpret_cast<unsigned long long *>(fin_smem);      // TBL
    uint32_t *cnt = reinterpret_cast<uint32_t *>(tbl + TBL);                       // CNT rank counters
    uint32_t *bitmap = cnt + CNT;                                                  // bm_words
    uint32_t *pre = bitmap + bm_words;                                                // bm_words + 1
    __shared__ FsShared F;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        F.ovf_s = 0;
        F.ovf_b[0] = F.ovf_b[1] = 0;
        F.f_s[0] = (int)atomicAdd(work, 1u);
    }
    for (int c = threadIdx.x; c < bm_words; c += THREADS) bitmap[c] = 0;
    for (int c = threadIdx.x; c < CNT; c += THREADS) cnt[c] = 0;

    for (int it = 0;; it++) {
        __syncthreads();             // the previous feature is out; bitmap and counters are clean
        const int f = F.f_s[it & 1];
        if (f >= n_fin) break;
        if (threadIdx.x == 0) F.f_s[(it + 1) & 1] = (int)atomicAdd(work, 1u);     // consumed after the next barrier
        const int32_t j = fin_feat[f];
        const FeatDesc fd = fdesc[j];
        const uint32_t n = seg_cur[j];
        const unsigned long long *seg = (const unsigned long long *)(pool + fd.blk_off);
        const bool light = n <= LIGHT;

        // range width of a heavy feature: a power of two (>= 32 cells) with about 3/4 CAP expected words
        int wshift = 5;
        uint32_t n_rng = 1;
        uint32_t *rc = reinterpret_cast<uint32_t *>(tbl);             // the table is idle: counters, then cursors
        if (!light) {
            if (threadIdx.x == 0) atomicAdd(&stats[0], 1ull);
            while (wshift < TBL_LOG2 - 2 && ((uint64_t)n << (wshift + 1)) <= (uint64_t)(CAP * 3 / 4) * (uint64_t)n_cols) wshift++;
            while (((n_cols - 1) >> wshift) + 1 > FS_RANGES) wshift++;      // very many cells: wider ranges, rank windows
            n_rng = (uint32_t)((n_cols - 1) >> wshift) + 1;
            for (uint32_t q = threadIdx.x; q < n_rng; q += THREADS) rc[q] = 0;
            __syncthreads();
        }

        // ---- phase 1: bitmap of the row's cells.  A light feature's words stay in registers; a heavy one
        // counts its words per column range in the same sweep.
        unsigned long long pw[FS_REG];
        if (light) {
#pragma unroll
            for (int q = 0; q < FS_REG; q++) {
                const uint32_t s = threadIdx.x + (uint32_t)q * THREADS;
                pw[q] = s < n ? seg[s] : 0ULL;
            }
            const uint32_t tsz0 = fs_table_size(n, TBL);
            for (uint32_t s = threadIdx.x; s < tsz0; s += THREADS) tbl[s] = 0ULL;
#pragma unroll
            for (int q = 0; q < FS_REG; q++)
                if (pw[q]) {
                    const uint32_t col = (uint32_t)(pw[q] & 0xffffffULL);
                    atomicOr(&bitmap[col >> 5], 1u << (col & 31));
                }
        } else {
            for (uint32_t s0 = threadIdx.x; s0 < n; s0 += THREADS * 4) {
                unsigned long long v[4];
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const uint32_t s = s0 + (uint32_t)q * THREADS;
                    v[q] = s < n ? seg[s] : 0ULL;
                }
#pragma unroll
                for (int q = 0; q < 4; q++)
                    if (v[q]) {
                        const uint32_t col = (uint32_t)(v[q] & 0xffffffULL);
                        atomicOr(&bitmap[col >> 5], 1u << (col & 31));
                        atomicAdd(&rc[col >> wshift], 1u);
                    }
            }
        }
        __syncthreads();
        // ---- prefix popcounts: pre[k] = set bits in words [0, k); the row's size; its place in the staging area
        {
            const int per = (bm_words + THREADS - 1) / THREADS;
            const int k0 = threadIdx.x * per, k1 = min(bm_words, k0 + per);
            uint32_t mine = 0;
            for (int k = k0; k < k1; k++) mine += (uint32_t)__popc(bitmap[k]);
            uint32_t incl = mine;
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl += y;
            }
            if (lane == 31) F.warp_tot[w] = incl;
            __syncthreads();
            uint32_t run = incl - mine;
            for (int q = 0; q < w; q++) run += F.warp_tot[q];
            for (int k = k0; k < k1; k++) {
                pre[k] = run;
                run += (uint32_t)__popc(bitmap[k]);
            }
            if (threadIdx.x == THREADS - 1) {
                pre[bm_words] = run;
                const int32_t row = sf_row[j];
                const long long b = run ? (long long)atomicAdd(cursor, (unsigned long long)run) : 0;
                seg_base[row] = b;
                seg_nnz[row] = (int32_t)run;
                F.base_s = b;
            }
        }
        __syncthreads();
        const long long base = F.base_s;

        if (light) {
            // ---- phase 2 from the registers, then the row
            const uint32_t tsz = fs_table_size(n, TBL);
            const int shift = 64 - (31 - __clz((int)tsz));
            // the table is at most 40 % full: with the whole table as probe limit an insert cannot fail
#pragma unroll
            for (int q = 0; q < FS_REG; q++)
                if (pw[q]) {
                    const uint32_t col = (uint32_t)(pw[q] & 0xffffffULL);
                    fs_insert(tbl, tsz, shift, pw[q], pair_hash(pw[q]), cnt, fs_rank(bitmap, pre, col), tsz);
                }
            __syncthreads();
            for (int k = threadIdx.x; k < bm_words; k += THREADS) {
                uint32_t bits = bitmap[k];
                if (!bits) continue;
                uint32_t r = pre[k];
                bitmap[k] = 0;
                while (bits) {
                    const int bpos = __ffs(bits) - 1;
                    bits &= bits - 1;
                    st_col[base + r] = (k << 5) + bpos;
                    st_val[base + r] = (int32_t)cnt[r];
                    cnt[r] = 0;
                    r++;
                }
            }
            continue;
        }

        // ---- heavy feature: split by column range into the scratch half of the block
        {   // exclusive prefix over the n_rng counters (F.warp_tot was read before the last barrier)
            const int per = (int)((n_rng + THREADS - 1) / THREADS);
            const uint32_t k0 = threadIdx.x * (uint32_t)per, k1 = min(n_rng, k0 + (uint32_t)per);
            uint32_t mine = 0;
            for (uint32_t k = k0; k < k1; k++) mine += rc[k];
            uint32_t incl = mine;
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl += y;
            }
            if (lane == 31) F.warp_tot[w] = incl;
            __syncthreads();
            uint32_t run = incl - mine;
            for (int q = 0; q < w; q++) run += F.warp_tot[q];
            for (uint32_t k = k0; k < k1; k++) {
                const uint32_t c = rc[k];
                F.range_off[k] = run;
                rc[k] = run;
                run += c;
            }
            if (threadIdx.x == THREADS - 1) F.range_off[n_rng] = n;
        }
        __syncthreads();
        unsigned long long *scr = const_cast<unsigned long long *>(seg) + ((((size_t)fd.log_cap) + 1) & ~(size_t)1);
        for (uint32_t s0 = threadIdx.x; s0 < n; s0 += THREADS * 4) {
            unsigned long long v[4];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const uint32_t s = s0 + (uint32_t)q * THREADS;
                v[q] = s < n ? seg[s] : 0ULL;
            }
#pragma unroll
            for (int q = 0; q < 4; q++)
                if (v[q]) scr[atomicAdd(&rc[(uint32_t)(v[q] & 0xffffffULL) >> wshift], 1u)] = v[q];
        }
        __syncthreads();
        // ---- the table (it held the range cursors) is cleared once; the row's cells go out in the same breath
        for (uint32_t s2 = threadIdx.x; s2 < TBL; s2 += THREADS) tbl[s2] = 0ULL;
        for (int k = threadIdx.x; k < bm_words; k += THREADS) {
            uint32_t bits = bitmap[k];
            uint32_t r = pre[k];
            while (bits) {
                const int bpos = __ffs(bits) - 1;
                bits &= bits - 1;
                st_col[base + r] = (k << 5) + bpos;
                r++;
            }
        }
        __syncthreads();
        // ---- the ranges, one after the other.  Fast path (the range's words fit a table pass, its cells a counter
        // bank): [insert into bank b] sync [bank b -> the row's counts, coalesced, and back to zero]; the next
        // range inserts into the other bank meanwhile, so a range costs ONE barrier.
        uint32_t bank = 0;
        for (uint32_t rg = 0; rg < n_rng; rg++) {
            const uint32_t p0 = F.range_off[rg], m = F.range_off[rg + 1] - p0;
            if (m == 0) continue;
            const uint32_t c0 = rg << wshift, c1 = min((uint32_t)n_cols, c0 + (1u << wshift));
            const uint32_t k_lo = c0 >> 5, k_hi = (c1 + 31) >> 5;
            const uint32_t rank0 = pre[k_lo];
            const uint32_t nz_r = pre[k_hi] - rank0;
            bool slow = m > CAP || nz_r > RCELLS;
            if (!slow) {
                uint32_t *cb = cnt + bank * RCELLS;
                for (uint32_t s0 = threadIdx.x; s0 < m; s0 += THREADS * 4) {
                    unsigned long long v[4];
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        const uint32_t s2 = s0 + (uint32_t)q * THREADS;
                        v[q] = s2 < m ? scr[p0 + s2] : 0ULL;
                    }
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        if (!v[q]) continue;
                        const uint32_t r = fs_rank(bitmap, pre, (uint32_t)(v[q] & 0xffffffULL)) - rank0;
                        if (!fs_insert_range<TBL_LOG2>(tbl, v[q], pair_hash(v[q]), rg, wshift, cb, r)) F.ovf_b[bank] = 1;
                    }
                }
                __syncthreads();
                if (!F.ovf_b[bank]) {       // (the flag of the OTHER bank may already be written by the next range)
                    for (uint32_t r = threadIdx.x; r < nz_r; r += THREADS) {
                        st_val[base + rank0 + r] = (int32_t)cb[r];
                        cb[r] = 0;
                    }
                    bank ^= 1;
                    continue;
                }
                // 96 probes were not enough (never with a sane hash): forget the attempt, take the careful path
                __syncthreads();
                for (uint32_t r = threadIdx.x; r < RCELLS; r += THREADS) cb[r] = 0;
                if (threadIdx.x == 0) {
                    F.ovf_b[bank] = 0;
                    atomicAdd(&stats[2], 1ull);
                }
                slow = true;
            }
            // ---- careful path: [clear table] sync [insert] sync per hash sub-partition, rank windows of CAP cells
            __syncthreads();                 // both banks are idle from here on
            if (threadIdx.x == 0) atomicAdd(&stats[1], 1ull);
            for (uint32_t win = 0; win < nz_r; win += CAP) {
                uint32_t n_sub = (m + CAP - 1) / CAP;
                while (true) {
                    const uint32_t tsz = fs_table_size(m / n_sub + 1, TBL);
                    const int shift = 64 - (31 - __clz((int)tsz));
                    for (uint32_t sub = 0; sub < n_sub; sub++) {
                        __syncthreads();             // the previous pass (or the previous window's row part) is done
                        for (uint32_t s2 = threadIdx.x; s2 < tsz; s2 += THREADS) tbl[s2] = 0ULL;
                        __syncthreads();
                        for (uint32_t s0 = threadIdx.x; s0 < m; s0 += THREADS * 4) {
                            unsigned long long v[4];
#pragma unroll
                            for (int q = 0; q < 4; q++) {
                                const uint32_t s2 = s0 + (uint32_t)q * THREADS;
                                v[q] = s2 < m ? scr[p0 + s2] : 0ULL;
                            }
#pragma unroll
                            for (int q = 0; q < 4; q++) {
                                if (!v[q]) continue;
                                const uint64_t h = pair_hash(v[q]);
                                if (n_sub > 1 && (uint32_t)(((h & 0xffffffffULL) * n_sub) >> 32) != sub) continue;
                                const uint32_t r = fs_rank(bitmap, pre, (uint32_t)(v[q] & 0xffffffULL)) - rank0 - win;
                                if (r >= CAP) continue;                       // another window of this range
                                if (!fs_insert(tbl, tsz, shift, v[q], h, cnt, r, min(tsz, 96u))) F.ovf_s = 1;
                            }
                        }
                    }
                    __syncthreads();
                    if (!F.ovf_s) break;
                    // a pass overflowed the table: forget the window's counts, sweep again with finer sub-partitions
                    __syncthreads();
                    for (uint32_t c = threadIdx.x; c < CAP; c += THREADS) cnt[c] = 0;
                    if (threadIdx.x == 0) {
                        F.ovf_s = 0;
                        atomicAdd(&stats[3], 1ull);
                    }
                    n_sub *= 2;
                }
                // the window's counts; the counters go back to zero as they are read
                const uint32_t n_w = min(nz_r - win, (uint32_t)CAP);
                for (uint32_t r = threadIdx.x; r < n_w; r += THREADS) {
                    st_val[base + rank0 + win + r] = (int32_t)cnt[r];
                    cnt[r] = 0;
                }
            }
            // the table holds what the last pass left: the fast path must not take those entries for duplicates of a
            // later range's words -- they carry THIS range's number, which no later range has; nothing to do.
            __syncthreads();
            bank = 0;
        }
        __syncthreads();
        for (int k = threadIdx.x; k < bm_words; k += THREADS) bitmap[k] = 0;
    }
}

// Set features (and every feature of a batch whose UMI keys do not fit the pair word): the feature's
// new-element log holds one cell index per distinct (cell, UMI); it is reduced through a shared-memory
// histogram over the cells plus a bitmap of the touched cells, cleared while they are read so that the next
// feature starts clean.  When the cells do not fit the histogram (n_cols > hist_cols) the log is read once
// per column range, first to count, then to write.
#define FIN_THREADS 512
#define FIN_WARPS (FIN_THREADS / 32)

__global__ void __launch_bounds__(FIN_THREADS) k_basefc_finalize_sets(
    const uint8_t *pool, const FeatDesc *fdesc, const int32_t *sf_row, const int32_t *fin_list,
    const int32_t *fin_lo, const int32_t *fin_hi, int32_t n_cols, int32_t hist_cols, unsigned int *work,
    unsigned long long *cursor, int64_t *seg_base, int32_t *seg_nnz, int32_t *st_col, int32_t *st_val) {
    extern __shared__ __align__(16) uint8_t fin_smem[];
    const int32_t *fin_feat = fin_list + *fin_lo;      // the epoch's features (as in k_basefc_finalize_segs)
    const int32_t n_fin = *fin_hi - *fin_lo;
    uint32_t *hist = reinterpret_cast<uint32_t *>(fin_smem);                          // hist_cols
    uint32_t *bitmap = hist + hist_cols;                                              // (hist_cols + 31) / 32
    __shared__ int warp_tot[FIN_WARPS];
    __shared__ long long base_s;
    __shared__ int f_s;
    const int n_words_max = (hist_cols + 31) >> 5;
    for (int c = threadIdx.x; c < hist_cols; c += FIN_THREADS) hist[c] = 0;
    for (int c = threadIdx.x; c < n_words_max; c += FIN_THREADS) bitmap[c] = 0;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int n_pass = (n_cols + hist_cols - 1) / hist_cols;

    while (true) {
        __syncthreads();
        if (threadIdx.x == 0) f_s = (int)atomicAdd(work, 1u);
        __syncthreads();
        const int f = f_s;
        if (f >= n_fin) break;
        const int32_t j = fin_feat[f];
        const FeatDesc fd = fdesc[j];
        const uint32_t *cur_p = (const uint32_t *)(pool + fd.blk_off + (size_t)fd.cap * 16);
        const uint32_t n_new = cur_p[0];
        const uint32_t *log = cur_p + 4;
        long long base = 0;
        // stage 0 (only when n_pass > 1): count; stage 1: write
        for (int stage = (n_pass > 1 ? 0 : 1); stage < 2; stage++) {
            int total_nz = 0;
            for (int pass = 0; pass < n_pass; pass++) {
                const uint32_t c_lo = (uint32_t)pass * (uint32_t)hist_cols;
                const int nc = min(hist_cols, n_cols - (int)c_lo);
                const int nw = (nc + 31) >> 5;
                for (uint32_t s = threadIdx.x; s < n_new; s += FIN_THREADS) {
                    const uint32_t col = log[s] - c_lo;
                    if (col < (uint32_t)nc && atomicAdd(&hist[col], 1u) == 0)
                        atomicOr(&bitmap[col >> 5], 1u << (col & 31));
                }
                __syncthreads();
                const bool writing = (stage == 1);
                if (!writing || n_pass == 1) {            // non-zero cells of this range
                    int nz = 0;
                    for (int k = threadIdx.x; k < nw; k += FIN_THREADS) nz += __popc(bitmap[k]);
                    for (int d = 16; d > 0; d >>= 1) nz += __shfl_xor_sync(0xffffffffu, nz, d);
                    if (lane == 0) warp_tot[w] = nz;
                    __syncthreads();
                    for (int k = 0; k < FIN_WARPS; k++) total_nz += warp_tot[k];
                    __syncthreads();
                }
                if (writing && n_pass == 1) {             // single range: reserve now
                    if (threadIdx.x == 0) {
                        const int32_t row = sf_row[j];
                        long long b = total_nz ? (long long)atomicAdd(cursor, (unsigned long long)total_nz) : 0;
                        seg_base[row] = b;
                        seg_nnz[row] = total_nz;
                        base_s = b;
                    }
                    __syncthreads();
                    base = base_s;
                }
                // ordered walk over the bitmap words; clears histogram and bitmap as it goes
                for (int k0 = 0; k0 < nw; k0 += FIN_THREADS) {
                    const int k = k0 + threadIdx.x;
                    uint32_t bits = k < nw ? bitmap[k] : 0u;
                    int cnt = __popc(bits), incl = cnt;
                    for (int d = 1; d < 32; d <<= 1) {
                        int y = __shfl_up_sync(0xffffffffu, incl, d);
                        if (lane >= d) incl += y;
                    }
                    if (lane == 31) warp_tot[w] = incl;
                    __syncthreads();
                    int before = 0, tot = 0;
                    for (int q = 0; q < FIN_WARPS; q++) {
                        const int x = warp_tot[q];
                        if (q < w) before += x;
                        tot += x;
                    }
                    long long o = base + before + (incl - cnt);
                    while (bits) {
                        const int bpos = __ffs(bits) - 1;
                        bits &= bits - 1;
                        const int c = (k << 5) + bpos;
                        if (writing) {
                            st_col[o] = (int32_t)(c_lo + (uint32_t)c);
                            st_val[o] = (int32_t)hist[c];
                            o++;
                        }
                        hist[c] = 0;
                    }
                    if (k < nw) bitmap[k] = 0;
                    base += tot;
                    __syncthreads();
                }
            }
            if (stage == 0) {                             // multi-range: reserve after counting
                if (threadIdx.x == 0) {
                    const int32_t row = sf_row[j];
                    long long b = total_nz ? (long long)atomicAdd(cursor, (unsigned long long)total_nz) : 0;
                    seg_base[row] = b;
                    seg_nnz[row] = total_nz;
                    base_s = b;
                }
                __syncthreads();
                base = base_s;
            }
        }
    }
}

}  // namespace

template <class T>
static int upload_vec(xg_ctx *ctx, const std::vector<T> &v, const char *name, const T **out) {
    T *d = (T *)ctx->get(name, sizeof(T) * (v.size() + 1));
    if (!d) return XG_E_CUDA;
    if (!v.empty())
        XG_CUDA(cudaMemcpyAsync(d, v.data(), sizeof(T) * v.size(), cudaMemcpyHostToDevice, ctx->stream));
    *out = d;
    return XG_OK;
}

static double ms_since(std::chrono::steady_clock::time_point a) {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - a).count();
}

// One basefc call: what its phases (params -> windows -> plan -> epochs -> result) hand on to one another.
struct BasefcCall {
    xg_ctx *ctx = nullptr;
    const xg_dreads *rd = nullptr;
    // != nullptr: the records of `rd` are not in HBM yet -- its device arrays are allocated but empty, and every
    // epoch's slice is copied from this pinned host batch on a copy stream just ahead of the epoch that counts it
    const xg_reads *src = nullptr;
    int32_t n_rows = 0, n_cols = 0;
    bool dbg_sync = false;
    int launches = 0;
    FeatCache *fc = nullptr;          // interval index and window jobs (kept by the context)
    size_t m = 0;                     // sorted features of the interval index
    BasefcDev P;
    const int32_t *d_sf_row = nullptr;
    TileDesc *d_tdesc = nullptr;
    const unsigned long long *d_cand = nullptr;     // per sorted feature: candidate reads, first / end tile
    const int32_t *d_tlo = nullptr, *d_thi = nullptr;
    bool seg_mode = false;
    int32_t n_epochs = 0, epoch_tiles = 0;
    PlanSummary plan;                 // the part of the device plan the host needs
    const int32_t *d_off = nullptr;   // the plan's list offsets (k_plan_offsets)
    const int32_t *d_list = nullptr;  // finalize lists, then the zero list
    const unsigned long long *d_zpre = nullptr;
    int64_t *seg_base = nullptr;      // staging area: first entry and entries of every row, the entries
    int32_t *seg_nnz = nullptr, *st_col = nullptr, *st_val = nullptr;
    unsigned long long *cursor = nullptr;
    unsigned int *fin_work = nullptr;
    uint32_t *seg_cur = nullptr;
    unsigned long long *fs_stats = nullptr;   // route counters of the segment finalize (xg_basefc_finalize_stats)
    unsigned long long *h_cur = nullptr;    // rows layouts: the staging cursor after every epoch (mapped host memory)
    int64_t h2d_bytes = 0;
    double ms_index = 0, ms_windows = 0, ms_alloc = 0, ms_upload = 0;
    // per-epoch events: 0 count start, 1 count end, 2 epoch end, 3 H2D, 4 big finalize end
    cudaEvent_t ev(int kind, int32_t e) const { return ctx->ev_pool[(size_t)5 * e + kind]; }
    cudaEvent_t ev_init() const { return ctx->ev_pool[(size_t)5 * n_epochs]; }
    // offsets of the finalize list of kind k (0 segments, 1 sets, 2 big segments) / of the zero list, epoch e
    const int32_t *fin_off(int k, int32_t e) const { return d_off + ((int64_t)k * n_epochs + e) * PLAN_KEYS; }
    const int32_t *zero_off(int32_t e) const { return d_off + (int64_t)3 * n_epochs * PLAN_KEYS + e; }
};

// The filters of the call and the cell-barcode table on the device.
static int basefc_params(BasefcCall &c, const xg_barcodes *cells, const xg_params *par) {
    xg_ctx *ctx = c.ctx;
    BasefcDev &P = c.P;
    auto t_ph = std::chrono::steady_clock::now();
    if (par->min_incl_tab) {
        if (par->min_incl_tab_len <= c.rd->max_aln_len)
            return ctx->fail(XG_E_ARG, "min_incl_tab shorter than max aligned length + 1");
        XG_GET(d_incl, int32_t, "fx_incl_tab", par->min_incl_tab_len + 1);
        // the caller's table outlives the call, which ends in a synchronisation
        XG_CUDA(cudaMemcpyAsync(d_incl, par->min_incl_tab, sizeof(int32_t) * (size_t)par->min_incl_tab_len,
                                cudaMemcpyHostToDevice, ctx->stream));
        P.incl_tab = d_incl;
        P.incl_tab_len = par->min_incl_tab_len;
    }
    P.incl_len = par->min_incl_len;
    P.col_bits = 1;
    while ((1 << P.col_bits) < c.n_cols) P.col_bits++;
    P.fp.min_mapq = par->min_mapq;
    P.fp.min_len = par->min_len;
    P.fp.incl_flag = par->incl_flag;
    P.fp.excl_flag = par->excl_flag;
    P.fp.no_orphan = par->no_orphan;
    P.fp.use_cell_tag = par->use_cell_tag;
    P.fp.need_umi_tag = par->need_umi_tag;
    int rc = XG_OK;
    if (par->use_cell_tag && (rc = xg_build_barcode_table(ctx, cells, &P.bc))) return rc;
    c.ms_upload = ms_since(t_ph);
    return XG_OK;
}

// The context's interval index of `feats` (FeatCache).  It depends on the features only: it is rebuilt only when the
// caller passes another set (host copy in the cache; device arrays in the named scratch buffers "fx_*", uploaded by
// feat_index_upload).  *cached: the index was the last call's.
static int feat_index(xg_ctx *ctx, const xg_features *feats, int32_t n_gid, FeatCache **out, bool *cached) {
    const size_t fb = sizeof(int32_t) * (size_t)feats->n;
    const std::initializer_list<xg_input_key::Span> in = {
        {&n_gid, sizeof n_gid}, {&feats->n, sizeof feats->n}, {feats->gid, fb}, {feats->beg, fb}, {feats->end, fb}};
    const uint64_t fh = xg_input_key::hash_of(in);
    FeatCache *fc = (FeatCache *)ctx->fx_cache;
    if (!fc) {
        fc = new FeatCache();
        ctx->fx_cache = fc;
        ctx->fx_cache_free = [](void *p) { delete (FeatCache *)p; };
    }
    *out = fc;
    *cached = fc->valid && fc->key.matches(fh, in);
    if (!*cached) {
        fc->valid = false;
        fc->ix = FeatIndexHost();
        int rc = build_feat_index(ctx, feats, n_gid, fc->ix);
        if (rc) return rc;
        fc->key.assign(fh, in);
    }
    return XG_OK;
}

// The index's device arrays (stabbing entries with their segment offsets zeroed); the cache is valid afterwards.
static int feat_index_upload(xg_ctx *ctx, FeatCache *fc) {
    const FeatIndexHost &ix = fc->ix;
    std::vector<int4> stab4(ix.stab.size());
    for (size_t k = 0; k < ix.stab.size(); k++) {
        const int32_t j = ix.stab[k];
        stab4[k] = make_int4(j, ix.sf_beg[(size_t)j], ix.sf_end[(size_t)j], 0);
    }
    const int4 *d_stab4 = nullptr;
    const int32_t *d = nullptr;
    int rc = XG_OK;
    if ((rc = upload_vec(ctx, ix.sf_goff, "fx_sf_goff", &d))) return rc;
    if ((rc = upload_vec(ctx, ix.sf_beg, "fx_sf_beg", &d))) return rc;
    if ((rc = upload_vec(ctx, ix.sf_end, "fx_sf_end", &d))) return rc;
    if ((rc = upload_vec(ctx, ix.sf_row, "fx_sf_row", &d))) return rc;
    if ((rc = upload_vec(ctx, ix.bnd_goff, "fx_bnd_goff", &d))) return rc;
    if ((rc = upload_vec(ctx, ix.bnd, "fx_bnd", &d))) return rc;
    if ((rc = upload_vec(ctx, ix.stab_off, "fx_stab_off", &d))) return rc;
    if ((rc = upload_vec(ctx, stab4, "fx_stab4", &d_stab4))) return rc;
    if ((rc = upload_vec(ctx, ix.fb, "fx_fb", &d))) return rc;
    XG_CUDA(cudaStreamSynchronize(ctx->stream));
    fc->valid = true;
    return XG_OK;
}

// Interval index of the features (host) and every feature's tile window and exact candidate count (device).
static int basefc_windows(BasefcCall &c, const xg_features *feats, int32_t n_gid) {
    xg_ctx *ctx = c.ctx;
    const xg_dreads *rd = c.rd;
    auto t_ph = std::chrono::steady_clock::now();
    FeatCache *fc = nullptr;
    bool index_cached = false;
    int rc = feat_index(ctx, feats, n_gid, &fc, &index_cached);
    if (rc) return rc;
    c.fc = fc;
    if (!fc->h_sum && !(fc->h_sum = (PlanSummary *)ctx->pinned_get(sizeof(PlanSummary))))
        return ctx->fail(XG_E_NOMEM, "out of pinned host memory");
    const FeatIndexHost &ix = fc->ix;
    const size_t m = c.m = ix.sf_beg.size();
    c.ms_index = ms_since(t_ph);
    t_ph = std::chrono::steady_clock::now();
    BasefcDev &P = c.P;
    P.pos_end = rd->pos_end;
    P.fmq = rd->fmq;
    P.cig_off = rd->cig_off;
    P.cigar = rd->cigar;
    P.keys = rd->keys;
    if (((uintptr_t)rd->pos_end | (uintptr_t)rd->fmq | (uintptr_t)rd->cig_off | (uintptr_t)rd->keys |
         (uintptr_t)rd->cigar) & 15)
        return ctx->fail(XG_E_ARG, "xg_basefc: record arrays must be 16-byte aligned");
    if (!index_cached && (rc = feat_index_upload(ctx, fc))) return rc;
    // the named scratch buffers keep their addresses between calls
    const int32_t *d_sf_goff = (const int32_t *)ctx->scratch["fx_sf_goff"].p;
    const int32_t *d_sf_beg = (const int32_t *)ctx->scratch["fx_sf_beg"].p;
    P.sf_end = (const int32_t *)ctx->scratch["fx_sf_end"].p;
    c.d_sf_row = (const int32_t *)ctx->scratch["fx_sf_row"].p;
    const int32_t *d_bnd_goff = (const int32_t *)ctx->scratch["fx_bnd_goff"].p;
    P.bnd = (const int32_t *)ctx->scratch["fx_bnd"].p;
    P.stab_off = (const int32_t *)ctx->scratch["fx_stab_off"].p;
    P.stab4 = (const int4 *)ctx->scratch["fx_stab4"].p;
    P.fb = (const int32_t *)ctx->scratch["fx_fb"].p;
    // feature windows on the device: one job per stretch of tiles of a run whose contig has features
    std::vector<WinJob> &jobs = fc->jobs;      // kept: the copy may still read it when this function returns
    jobs.clear();
    int64_t n_warps = 0;
    for (const int3 &rt : rd->h_run_tiles) {
        const int32_t g = rd->h_runs[(size_t)rt.x].gid;
        if (g >= 0 && g < n_gid && ix.sf_goff[(size_t)g + 1] > ix.sf_goff[(size_t)g]) {
            jobs.push_back(WinJob{ix.sf_goff[(size_t)g], ix.sf_goff[(size_t)g + 1], rt.y, rt.z, n_warps});
            n_warps += ix.sf_goff[(size_t)g + 1] - ix.sf_goff[(size_t)g];
        }
    }
    const WinJob *d_jobs = nullptr;
    if ((rc = upload_vec(ctx, jobs, "fx_jobs", &d_jobs))) return rc;
    XG_GET(d_cand, unsigned long long, "fx_cand", m + 1);
    XG_GET(d_tlo, int32_t, "fx_tlo", m + 1);
    XG_GET(d_thi, int32_t, "fx_thi", m + 1);
    XG_GET(d_tdesc, TileDesc, "fx_tdesc", rd->n_tiles + 1);
    P.tdesc = c.d_tdesc = d_tdesc;
    c.d_cand = d_cand;
    c.d_tlo = d_tlo;
    c.d_thi = d_thi;
    cudaEventRecord(ctx->ev[0], ctx->stream);
    XG_CUDA(cudaMemsetAsync(d_cand, 0, sizeof(unsigned long long) * (m + 1), ctx->stream));
    XG_CUDA(cudaMemsetAsync(d_tlo, 0x7f, sizeof(int32_t) * (m + 1), ctx->stream));
    XG_CUDA(cudaMemsetAsync(d_thi, 0xff, sizeof(int32_t) * (m + 1), ctx->stream));
    if (n_warps > 0) {
        k_feature_windows<<<(unsigned)((n_warps + 7) / 8), 256, 0, ctx->stream>>>(
            d_jobs, (int32_t)jobs.size(), n_warps, rd->tiles, rd->tile_pmax, rd->pos_end, c.src ? 0 : 1, d_sf_beg,
            P.sf_end, d_cand, d_tlo, d_thi);
        c.launches++;
        XG_DBG("k_feature_windows");
    }
    if (rd->n_tiles > 0) {
        // streaming call: the records (and with them the tiles' CIGAR ranges) arrive epoch by epoch
        k_tile_desc<<<(rd->n_tiles + 255) / 256, 256, 0, ctx->stream>>>(
            rd->tiles, rd->runs, rd->n_tiles, n_gid, d_sf_goff, d_bnd_goff, P.bnd, P.stab_off, P.stab4, P.fb,
            c.src ? nullptr : rd->cig_off, d_tdesc);
        c.launches++;
        XG_DBG("k_tile_desc");
    }
    c.ms_windows = ms_since(t_ph);
    return XG_OK;
}

// The epoch plan, on the device where the windows are (k_plan_*): pool layout, which features each epoch zeroes
// and finalizes.  Its summary is the call's one wait before the epochs: it sizes the pool and the staging area.
static int basefc_plan(BasefcCall &c, bool force_sets) {
    xg_ctx *ctx = c.ctx;
    const xg_dreads *rd = c.rd;
    FeatCache *fc = c.fc;
    const size_t m = c.m;
    const int32_t n_cols = c.n_cols;
    BasefcDev &P = c.P;
    auto t_ph = std::chrono::steady_clock::now();
    int32_t epoch_tiles = c.src ? 8192 : 65536;     // streaming: finer epochs = finer H2D / kernel overlap
    if (const char *e = getenv(c.src ? "XG_EPOCH_TILES_HOST" : "XG_EPOCH_TILES")) {
        epoch_tiles = std::max(1, atoi(e));
    } else if (!c.src && rd->n_tiles > 0) {
        // equal epochs: a short last epoch costs its launches, its drain and its finalize like a full one
        const int32_t n_ep = (rd->n_tiles + epoch_tiles - 1) / epoch_tiles;
        epoch_tiles = (rd->n_tiles + n_ep - 1) / n_ep;
    }
    c.epoch_tiles = epoch_tiles;
    c.n_epochs = std::max(1, (rd->n_tiles + epoch_tiles - 1) / epoch_tiles);
    const int32_t ne = c.n_epochs;
    // Pair-word mode: a (cell, UMI) pair is one 64-bit word `umi | cell` (every UMI key of the batch leaves
    // its low 24 bits free: packed strings of up to 13 symbols, interned ids below 2^39), features collect
    // their words in segments.  The kernel verifies the keys it meets; a key that does not fit raises a
    // flag and the call is redone with a set per feature (and the batch remembers it).
    bool seg_mode = !force_sets && n_cols <= (1 << 19) && rd->umi_compact != 0;      // cell bitmap + ranks in shared memory
    if (const char *e = getenv("XG_SEG_MODE")) seg_mode = seg_mode && atoi(e) != 0;
    c.seg_mode = seg_mode;
    P.seg_mode = seg_mode ? 1 : 0;
    // seg_max: features with at most this many candidate reads collect pair words in a segment (0: every feature
    // keeps a set); heavier features keep a set in global memory
    uint64_t seg_max = 1ull << 22;
    if (const char *e = getenv("XG_SEG_MAX")) seg_max = (uint64_t)atoll(e);
    if (!seg_mode) seg_max = 0;
    // The reduction of a feature is one CTA's work and its passes are bound by the loads that CTA keeps in flight:
    // the few features with very many reads (a long tail in expression data) would be the critical path of their
    // epoch.  They get CTAs of 1024 threads, launched beside the ordinary ones.
    uint64_t seg_big = 4096;                  // candidate reads; about 1 600 words, the light / heavy limit of the ordinary CTAs
    if (const char *e = getenv("XG_SEG_BIG")) seg_big = (uint64_t)atoll(e);
    if (((size_t)10 << FS_BIG_TBL_LOG2) + (size_t)(2 * ((n_cols + 31) / 32) + 1) * 4 + sizeof(FsShared) + 1280 > 200 * 1024)
        seg_big = ~0ull;                      // so many cells that the big CTA's shared memory does not fit: no big CTAs
    // histogram / offsets: [3 kinds][epochs][PLAN_KEYS], then [epochs] of the zero list, then the total
    const int64_t n_hist = (int64_t)3 * ne * PLAN_KEYS + ne;
    XG_GET(fdesc, FeatDesc, "fx_fdesc", m + 1);
    XG_GET(segoff16, uint32_t, "fx_segoff16", m + 1);
    XG_GET(list, int32_t, "fx_plan_list", 2 * m + 1);
    XG_GET(zpre, unsigned long long, "fx_plan_zpre", 2 * m + 2);
    XG_GET(cur, int32_t, "fx_plan_cur", n_hist + 1);
    const size_t acc_bytes = sizeof(PlanAcc) + sizeof(unsigned long long) * (size_t)ne + sizeof(int32_t) * (size_t)(n_hist + 1);
    XG_GET(acc_raw, uint8_t, "fx_plan_acc", acc_bytes);
    PlanAcc *acc = (PlanAcc *)acc_raw;
    unsigned long long *epoch_bytes = (unsigned long long *)(acc + 1);
    int32_t *hist = (int32_t *)(epoch_bytes + ne);
    P.fdesc = fdesc;
    P.segoff16 = segoff16;
    c.d_off = hist;
    c.d_list = list;
    c.d_zpre = zpre;
    cudaStream_t st = ctx->stream;
    XG_CUDA(cudaMemsetAsync(acc_raw, 0, acc_bytes, st));
    const unsigned plan_grid = (unsigned)((m + 255) / 256);
    if (m) {
        k_plan_features<<<plan_grid, 256, 0, st>>>(c.d_cand, c.d_tlo, c.d_thi, (int32_t)m, n_cols, epoch_tiles, ne, seg_max,
                                                   seg_big, acc, epoch_bytes, hist, fdesc, segoff16);
        c.launches++;
        XG_DBG("k_plan_features");
    }
    k_plan_offsets<<<1, PLAN_SCAN_THREADS, 0, st>>>(acc, epoch_bytes, ne, hist, n_hist, cur);
    c.launches++;
    XG_DBG("k_plan_offsets");
    if (m) {
        k_plan_place<<<plan_grid, 256, 0, st>>>(c.d_cand, c.d_tlo, c.d_thi, (int32_t)m, epoch_tiles, ne, seg_max, seg_big,
                                                acc, cur, list, fdesc, segoff16);
        c.launches++;
        XG_DBG("k_plan_place");
    }
    k_plan_zero_prefix<<<1, PLAN_SCAN_THREADS, 0, st>>>(c.zero_off(0), c.zero_off(ne), list, fdesc, zpre);
    c.launches++;
    XG_DBG("k_plan_zero_prefix");
    const size_t n_stab = fc->ix.stab.size();
    if (n_stab) {      // the segment offsets of the plan go into the stabbing entries
        k_patch_stab<<<(unsigned)((n_stab + 255) / 256), 256, 0, st>>>((int4 *)P.stab4, (int32_t)n_stab, segoff16);
        c.launches++;
        XG_DBG("k_patch_stab");
    }
    XG_CUDA(cudaMemcpyAsync(fc->h_sum, &acc->sum, sizeof(PlanSummary), cudaMemcpyDeviceToHost, st));
    XG_CUDA(cudaStreamSynchronize(st));
    c.plan = *fc->h_sum;
    c.ms_windows += ms_since(t_ph);
    if (c.plan.err & 1u) return ctx->fail(XG_E_LIMIT, "feature window exceeds 2^32 reads");
    if (c.plan.err & 2u) return ctx->fail(XG_E_LIMIT, "segment pool exceeds 64 GiB; use smaller epochs (XG_EPOCH_TILES)");
    t_ph = std::chrono::steady_clock::now();
    XG_GET(pool, uint8_t, "fx_pool", c.plan.pool_bytes + 16);
    XG_GET(seg_base, int64_t, "fx_seg_base", c.n_rows + 1);
    XG_GET(seg_nnz, int32_t, "fx_seg_nnz", c.n_rows + 1);
    XG_GET(st_col, int32_t, "fx_st_col", c.plan.staging_cap + 1);
    XG_GET(st_val, int32_t, "fx_st_val", c.plan.staging_cap + 1);
    XG_GET(cursor, unsigned long long, "fx_cursor", 2);
    // per epoch: work counters of the ordinary finalize, counting, set finalize and big finalize launches; flags
    XG_GET(fin_work, unsigned int, "fx_fin_work", 4 * (ne + 1) + 4);
    XG_GET(seg_cur, uint32_t, "fx_seg_cur", m + 1);
    c.seg_base = seg_base;
    c.seg_nnz = seg_nnz;
    c.st_col = st_col;
    c.st_val = st_val;
    c.cursor = cursor;
    c.fin_work = fin_work;
    c.seg_cur = seg_cur;
    P.pool = pool;
    P.seg_cur = seg_cur;
    P.flags = fin_work + 4 * (ne + 1);
    c.ms_alloc = ms_since(t_ph);
    return XG_OK;
}

// The epochs on the device: zero(e) -> count(e) -> finalize(e), one after another on the context's stream.  The
// counting kernel is persistent and fills the GPU by itself; only the big-segment finalize runs beside the
// ordinary one, and (xg_basefc_host) the copy of the next epoch's records beside the kernels.  How many features
// an epoch zeroes and finalizes is known on the device only: those kernels get a fixed grid and read their
// epoch's range of the plan's lists.
static int basefc_epochs(BasefcCall &c, bool rows) {
    xg_ctx *ctx = c.ctx;
    const xg_dreads *rd = c.rd;
    const PlanSummary &pl = c.plan;
    const int32_t n_rows = c.n_rows, n_cols = c.n_cols, ne = c.n_epochs;
    const size_t m = c.m;
    BasefcDev &P = c.P;
    // shared memory of the finalize kernels.  Segments: dedup table, rank counters, bitmap over the cells and
    // its prefix popcounts.  Sets: histogram (+ bitmap) over the cells -- all cells if they fit.
    const int bm_words = (n_cols + 31) / 32;
    auto segs_smem = [&](int tbl_log2) {
        return ((size_t)8 << tbl_log2) + ((size_t)2 << tbl_log2) + (size_t)(2 * bm_words + 1) * 4;    // table, counters, bitmap + prefix
    };
    const size_t segs_bytes = segs_smem(FS_TBL_LOG2), big_bytes = segs_smem(FS_BIG_TBL_LOG2);
    // only segment features use these kernels, and only in seg_mode (n_cols <= 2^19) does their bitmap fit: with
    // more columns the attribute would be refused and the call fail although no segment kernel runs
    if (c.seg_mode)
        XG_CUDA(cudaFuncSetAttribute(k_basefc_finalize_segs<FS_THREADS, FS_TBL_LOG2>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)segs_bytes));
    // big CTAs need the large table; with so many cells that it does not fit, big features go the ordinary way
    const bool big_ok = big_bytes + sizeof(FsShared) + 1280 <= 200 * 1024;
    if (c.seg_mode && big_ok)
        XG_CUDA(cudaFuncSetAttribute(k_basefc_finalize_segs<FS_BIG_THREADS, FS_BIG_TBL_LOG2>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)big_bytes));
    const int segs_ctas_per_sm = std::max(1, std::min(8, (int)(224 * 1024 / (segs_bytes + sizeof(FsShared) + 1280))));
    int32_t hist_cols = std::min(n_cols, 40 * 1024);
    if (const char *e = getenv("XG_HIST_COLS")) hist_cols = std::max(32, std::min(n_cols, atoi(e)));
    const size_t hist_bytes = (size_t)hist_cols * 4 + (size_t)((hist_cols + 31) / 32) * 4;
    XG_CUDA(cudaFuncSetAttribute(k_basefc_finalize_sets, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hist_bytes));
    const int fin_ctas_per_sm = std::max(1, std::min(4, (int)(220 * 1024 / (hist_bytes + 2048))));
    XG_CUDA(cudaFuncSetAttribute(k_basefc_count<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CountSmem)));
    // fixed grids: the most CTAs that fit the GPU, fewer when the whole call has fewer features of the kind
    const int64_t n_seg = (int64_t)(pl.n_seg_feat - pl.n_big_feat), n_big = (int64_t)pl.n_big_feat,
                  n_set = (int64_t)pl.n_set_feat;
    const int segs_grid = (int)std::min<int64_t>(n_seg, 148 * segs_ctas_per_sm);
    const int big_grid = (int)std::min<int64_t>(n_big, 148);
    const int sets_grid = (int)std::min<int64_t>(n_set, 148 * fin_ctas_per_sm);
    const unsigned zero_grid = 148 * 8;

    if (n_big > 0 && !ctx->big_stream) XG_CUDA(cudaStreamCreateWithFlags(&ctx->big_stream, cudaStreamNonBlocking));
    if (c.src && !ctx->copy_stream) XG_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    while ((int32_t)ctx->ev_pool.size() < 5 * ne + 1) {
        cudaEvent_t ev;
        XG_CUDA(cudaEventCreate(&ev));
        ctx->ev_pool.push_back(ev);
    }
    unsigned int *cnt_work = c.fin_work + ne + 1;          // tile counters of the counting launches
    unsigned int *set_work = c.fin_work + 2 * (ne + 1);    // work counters of the set finalize launches
    unsigned int *big_work = c.fin_work + 3 * (ne + 1);    // ... of the big-segment finalize launches
    cudaStream_t st = ctx->stream;
    XG_CUDA(cudaMemsetAsync(c.seg_nnz, 0, sizeof(int32_t) * (size_t)(n_rows + 1), st));
    XG_CUDA(cudaMemsetAsync(c.seg_base, 0, sizeof(int64_t) * (size_t)(n_rows + 1), st));
    XG_CUDA(cudaMemsetAsync(c.cursor, 0, 16, st));
    XG_CUDA(cudaMemsetAsync(c.fin_work, 0, sizeof(unsigned int) * (size_t)(4 * (ne + 1) + 4), st));
    XG_CUDA(cudaMemsetAsync(c.seg_cur, 0, sizeof(uint32_t) * (m + 1), st));
    c.launches += 6;
    cudaEventRecord(c.ev_init(), st);
    if (c.src) cudaStreamWaitEvent(ctx->copy_stream, c.ev_init(), 0);
    // rows layouts: the rows stay in the order they were completed; after every epoch the staging cursor is
    // snapshotted so that the host can copy that epoch's rows out while the later epochs are still being counted
    unsigned long long *d_cur = nullptr;
    if (rows) {
        if (!ctx->d2h_stream) XG_CUDA(cudaStreamCreateWithFlags(&ctx->d2h_stream, cudaStreamNonBlocking));
        c.h_cur = (unsigned long long *)ctx->pinned_get(sizeof(unsigned long long) * (size_t)(ne + 1));
        if (!c.h_cur) return ctx->fail(XG_E_NOMEM, "out of pinned host memory");
        if (cudaHostGetDevicePointer((void **)&d_cur, c.h_cur, 0) != cudaSuccess) {
            cudaGetLastError();
            ctx->pinned_put(c.h_cur);
            c.h_cur = nullptr;
            return ctx->fail(XG_E_CUDA, "pinned host memory is not mapped for the device");
        }
    }
    for (int32_t e = 0; e < ne; e++) {
        const int32_t t0 = e * c.epoch_tiles, t1 = std::min(rd->n_tiles, t0 + c.epoch_tiles);
        if (c.src) {      // this epoch's records: host -> HBM on the copy stream
            const xg_reads *src = c.src;
            if (t1 > t0) {
                const int64_t ra = rd->h_tiles[(size_t)t0].rec_beg;
                const int64_t rb = rd->h_tiles[(size_t)t1 - 1].rec_beg + rd->h_tiles[(size_t)t1 - 1].n_rec;
                const size_t nr = (size_t)(rb - ra);
                const uint32_t ca = src->cig_off[ra], cb = src->cig_off[rb];
                cudaStream_t cs = ctx->copy_stream;
                cudaMemcpyAsync(rd->pos_end + ra, src->pos_end + 2 * ra, nr * 8, cudaMemcpyHostToDevice, cs);
                cudaMemcpyAsync(rd->fmq + ra, src->fmq + ra, nr * 4, cudaMemcpyHostToDevice, cs);
                cudaMemcpyAsync(rd->cig_off + ra, src->cig_off + ra, (nr + 1) * 4, cudaMemcpyHostToDevice, cs);
                cudaMemcpyAsync(rd->keys + ra, src->keys + 2 * ra, nr * 16, cudaMemcpyHostToDevice, cs);
                const uint32_t ca1 = ca ? ca - 1 : 0;      // one word back: a >=255-op count word
                if (cb > ca1)
                    cudaMemcpyAsync(rd->cigar + ca1, src->cigar + ca1, (size_t)(cb - ca1) * 4, cudaMemcpyHostToDevice, cs);
                c.h2d_bytes += (int64_t)(nr * 32 + 4 + (size_t)(cb - ca1) * 4);
            }
            cudaEventRecord(c.ev(3, e), ctx->copy_stream);
            cudaStreamWaitEvent(st, c.ev(3, e), 0);
        }
        if (n_set > 0) {
            k_zero_segments<<<zero_grid, 256, 0, st>>>(P.pool, P.fdesc, c.d_list, c.d_zpre, c.zero_off(e), c.zero_off(e + 1));
            c.launches++;
            XG_DBG("k_zero_segments");
        }
        if (c.src && t1 > t0) {      // the CIGAR ranges of the tiles whose records have just arrived
            k_tile_cig<<<(t1 - t0 + 255) / 256, 256, 0, st>>>(rd->tiles, t0, t1, rd->cig_off, c.d_tdesc);
            c.launches++;
            XG_DBG("k_tile_cig");
        }
        cudaEventRecord(c.ev(0, e), st);
        if (t1 > t0 && m > 0) {
            P.tile0 = t0;
            P.tile1 = t1;
            P.work = cnt_work + e;
            k_basefc_count<4><<<std::min(t1 - t0, 148 * 4), CNT_THREADS, sizeof(CountSmem), st>>>(P);
            c.launches++;
            XG_DBG("k_basefc_count");
        }
        cudaEventRecord(c.ev(1, e), st);
        // big segments first, on a stream of their own: their few large CTAs take their SMs before the ordinary
        // finalize CTAs fill the rest, and both kernels run side by side
        if (n_big > 0) {
            cudaStreamWaitEvent(ctx->big_stream, c.ev(1, e), 0);
            k_basefc_finalize_segs<FS_BIG_THREADS, FS_BIG_TBL_LOG2><<<big_grid, FS_BIG_THREADS, big_bytes, ctx->big_stream>>>(
                P.pool, P.fdesc, c.seg_cur, c.d_sf_row, c.d_list, c.fin_off(2, e), c.fin_off(2, e + 1), n_cols,
                big_work + e, c.cursor, c.seg_base, c.seg_nnz, c.st_col, c.st_val, c.fs_stats);
            c.launches++;
            XG_DBG("k_basefc_finalize_segs<big>");
            cudaEventRecord(c.ev(4, e), ctx->big_stream);
        }
        if (n_seg > 0) {
            k_basefc_finalize_segs<FS_THREADS, FS_TBL_LOG2><<<segs_grid, FS_THREADS, segs_bytes, st>>>(
                P.pool, P.fdesc, c.seg_cur, c.d_sf_row, c.d_list, c.fin_off(0, e), c.fin_off(0, e + 1), n_cols,
                c.fin_work + e, c.cursor, c.seg_base, c.seg_nnz, c.st_col, c.st_val, c.fs_stats);
            c.launches++;
            XG_DBG("k_basefc_finalize_segs");
        }
        if (n_set > 0) {
            k_basefc_finalize_sets<<<sets_grid, FIN_THREADS, hist_bytes, st>>>(
                P.pool, P.fdesc, c.d_sf_row, c.d_list, c.fin_off(1, e), c.fin_off(1, e + 1), n_cols, hist_cols,
                set_work + e, c.cursor, c.seg_base, c.seg_nnz, c.st_col, c.st_val);
            c.launches++;
            XG_DBG("k_basefc_finalize_sets");
        }
        // the snapshot is a store into mapped host memory, not a copy: a D2H of 8 bytes would queue
        // behind the result copies on the copy engine and stall the finalize stream with them
        if (n_big > 0) cudaStreamWaitEvent(st, c.ev(4, e), 0);      // join: the epoch's rows are all reserved
        if (d_cur) k_snapshot_cursor<<<1, 1, 0, st>>>(c.cursor, d_cur + e);
        cudaEventRecord(c.ev(2, e), st);
    }
    XG_CUDA(cudaGetLastError());
    return XG_OK;
}

// Rows layouts: every epoch's rows go to pinned host memory as soon as the epoch has finished, while the later
// epochs are counted -- as they are, or packed on the way (16-bit column | 16-bit count, or the 16-bit words of
// XG_LAYOUT_ROWS_TINY) with a side list for the entries that do not fit.  The first call has no size hint and
// copies everything at the end.
static int basefc_collect_rows(BasefcCall &c, int32_t layout, xg_coo **out) {
    xg_ctx *ctx = c.ctx;
    const int64_t staging_cap = (int64_t)c.plan.staging_cap;
    const int32_t n_rows = c.n_rows, n_cols = c.n_cols;
    const int32_t *st_col = c.st_col, *st_val = c.st_val;
    const auto t_tail = std::chrono::steady_clock::now();
    xg_coo_owner *o = new xg_coo_owner();
    memset(&o->m, 0, sizeof(o->m));
    o->ctx = ctx;
    auto give_up = [&](int code, const std::string &msg) {
        cudaStreamSynchronize(ctx->d2h_stream);
        cudaStreamSynchronize(ctx->stream);
        for (void *q : o->bufs) ctx->pinned_put(q);
        ctx->pinned_put(c.h_cur);
        delete o;
        return ctx->fail(code, msg);
    };
    int64_t cap = ctx->fx_nnz_hint > 0 ? ctx->fx_nnz_hint + ctx->fx_nnz_hint / 8 + 1024 : 0;
    cap = std::min<int64_t>(cap, staging_cap + 1);
    // The entry format: narrow entries need 16-bit columns, and a packed format whose side list overflows falls
    // back to plain entries (below) -- the only two places it is chosen.
    int32_t fmt = layout == XG_LAYOUT_ROWS_NARROW && n_cols > 65536 ? XG_LAYOUT_ROWS : layout;
    const bool narrow = fmt == XG_LAYOUT_ROWS_NARROW, tiny = fmt == XG_LAYOUT_ROWS_TINY;    // device buffers
    const int64_t OVER_CAP = tiny ? (1 << 23) : (1 << 20);
    uint32_t *d_packed = nullptr;
    uint16_t *d_tiny = nullptr;
    uint32_t *d_row_start = nullptr;
    long long *d_over_idx = nullptr;
    int32_t *d_over_val = nullptr, *d_over_col = nullptr;
    unsigned int *d_over_n = nullptr;
    const size_t row_start_words = (size_t)(staging_cap + 32) / 32 + 1;
    if (narrow || tiny) {
        if (narrow) d_packed = (uint32_t *)ctx->get("fx_packed", sizeof(uint32_t) * (size_t)(staging_cap + 1));
        if (tiny) {
            d_tiny = (uint16_t *)ctx->get("fx_tiny", sizeof(uint16_t) * (size_t)(staging_cap + 2));
            d_row_start = (uint32_t *)ctx->get("fx_row_start", sizeof(uint32_t) * row_start_words);
            d_over_col = (int32_t *)ctx->get("fx_over_col", sizeof(int32_t) * (size_t)OVER_CAP);
        }
        d_over_idx = (long long *)ctx->get("fx_over_idx", sizeof(long long) * (size_t)OVER_CAP);
        d_over_val = (int32_t *)ctx->get("fx_over_val", sizeof(int32_t) * (size_t)OVER_CAP);
        d_over_n = (unsigned int *)ctx->get("fx_over_n", 16);
        if ((narrow && !d_packed) || (tiny && (!d_tiny || !d_row_start || !d_over_col)) || !d_over_idx || !d_over_val ||
            !d_over_n)
            return give_up(XG_E_CUDA, ctx->err);
        cudaMemsetAsync(d_over_n, 0, 4, ctx->d2h_stream);
        if (tiny) cudaMemsetAsync(d_row_start, 0, sizeof(uint32_t) * row_start_words, ctx->d2h_stream);
    }
    int32_t *h_col = nullptr, *h_val = nullptr;
    uint32_t *h_packed = nullptr;
    uint16_t *h_tiny = nullptr;
    auto host_buffers = [&](int64_t n_cap) {
        for (void *q : o->bufs) ctx->pinned_put(q);
        o->bufs.clear();
        h_col = h_val = nullptr;
        h_packed = nullptr;
        h_tiny = nullptr;
        switch (fmt) {
        case XG_LAYOUT_ROWS_TINY:
            if ((h_tiny = (uint16_t *)ctx->pinned_get((size_t)n_cap * 2 + 16))) o->bufs.push_back(h_tiny);
            return h_tiny != nullptr;
        case XG_LAYOUT_ROWS_NARROW:
            if ((h_packed = (uint32_t *)ctx->pinned_get((size_t)n_cap * 4))) o->bufs.push_back(h_packed);
            return h_packed != nullptr;
        default:
            if ((h_col = (int32_t *)ctx->pinned_get((size_t)n_cap * 4))) o->bufs.push_back(h_col);
            if ((h_val = (int32_t *)ctx->pinned_get((size_t)n_cap * 4))) o->bufs.push_back(h_val);
            return h_col && h_val;
        }
    };
    auto queue_rows = [&](int64_t from, int64_t to) {       // staging entries [from, to) -> host
        const size_t n = (size_t)(to - from);
        switch (fmt) {
        case XG_LAYOUT_ROWS_TINY:
            // the rows finished so far have their places (seg_base / seg_nnz): mark their first entries
            k_mark_row_starts<<<(n_rows + 255) / 256, 256, 0, ctx->d2h_stream>>>(c.seg_base, c.seg_nnz, n_rows, d_row_start);
            k_pack_rows_tiny<<<(unsigned)((n + 255) / 256), 256, 0, ctx->d2h_stream>>>(
                st_col, st_val, d_row_start, d_tiny, from, to, d_over_idx, d_over_col, d_over_val, d_over_n,
                (unsigned int)OVER_CAP);
            cudaMemcpyAsync(h_tiny + from, d_tiny + from, n * 2, cudaMemcpyDeviceToHost, ctx->d2h_stream);
            break;
        case XG_LAYOUT_ROWS_NARROW:
            k_pack_rows<<<(unsigned)((n + 255) / 256), 256, 0, ctx->d2h_stream>>>(st_col, st_val, d_packed, from, to, d_over_idx,
                                                                                d_over_val, d_over_n, (unsigned int)OVER_CAP);
            cudaMemcpyAsync(h_packed + from, d_packed + from, n * 4, cudaMemcpyDeviceToHost, ctx->d2h_stream);
            break;
        default:
            cudaMemcpyAsync(h_col + from, st_col + from, n * 4, cudaMemcpyDeviceToHost, ctx->d2h_stream);
            cudaMemcpyAsync(h_val + from, st_val + from, n * 4, cudaMemcpyDeviceToHost, ctx->d2h_stream);
        }
    };
    if (cap > 0 && !host_buffers(cap)) return give_up(XG_E_NOMEM, "out of pinned host memory for the result");
    int64_t done = 0;            // entries already queued for the host
    bool fits = cap > 0;
    for (int32_t e = 0; e < c.n_epochs && fits; e++) {
        cudaError_t ce = cudaEventSynchronize(c.ev(2, e));
        if (ce != cudaSuccess) return give_up(XG_E_CUDA, std::string("basefc: ") + cudaGetErrorString(ce));
        const int64_t cur = (int64_t)c.h_cur[e];
        if (cur > cap) {
            fits = false;        // more rows than the last call: finish with one copy at the end
            break;
        }
        if (cur > done) {
            queue_rows(done, cur);
            done = cur;
        }
    }
    cudaError_t ce = cudaStreamSynchronize(ctx->stream);      // every epoch has finished
    if (ce != cudaSuccess) return give_up(XG_E_CUDA, std::string("basefc: ") + cudaGetErrorString(ce));
    unsigned long long nnz_u = 0;
    XG_CUDA(cudaMemcpy(&nnz_u, c.cursor, 8, cudaMemcpyDeviceToHost));
    const int64_t nnz = (int64_t)nnz_u;
    if (!fits || nnz > cap) {
        cudaStreamSynchronize(ctx->d2h_stream);
        cap = nnz + nnz / 8 + 1024;
        if (!host_buffers(cap)) return give_up(XG_E_NOMEM, "out of pinned host memory for the result");
        if (fmt != XG_LAYOUT_ROWS) cudaMemsetAsync(d_over_n, 0, 4, ctx->d2h_stream);
        done = 0;
    }
    if (nnz > done) queue_rows(done, nnz);
    unsigned int n_over = 0;
    if (fmt != XG_LAYOUT_ROWS) {
        cudaMemcpyAsync(&n_over, d_over_n, 4, cudaMemcpyDeviceToHost, ctx->d2h_stream);
        ce = cudaStreamSynchronize(ctx->d2h_stream);
        if (ce != cudaSuccess) return give_up(XG_E_CUDA, std::string("result D2H: ") + cudaGetErrorString(ce));
        if ((int64_t)n_over > OVER_CAP) {       // too many entries for the side list: plain 32-bit columns
            fmt = XG_LAYOUT_ROWS;
            if (!host_buffers(cap)) return give_up(XG_E_NOMEM, "out of pinned host memory for the result");
            if (nnz > 0) queue_rows(0, nnz);
            n_over = 0;
        }
    }
    long long *h_over_idx = nullptr;
    int32_t *h_over_val = nullptr, *h_over_col = nullptr;
    if (fmt != XG_LAYOUT_ROWS) {
        h_over_idx = (long long *)ctx->pinned_get(((size_t)n_over + 1) * 8);
        h_over_val = (int32_t *)ctx->pinned_get(((size_t)n_over + 1) * 4);
        if (h_over_idx) o->bufs.push_back(h_over_idx);
        if (h_over_val) o->bufs.push_back(h_over_val);
        if (fmt == XG_LAYOUT_ROWS_TINY) {
            h_over_col = (int32_t *)ctx->pinned_get(((size_t)n_over + 1) * 4);
            if (h_over_col) o->bufs.push_back(h_over_col);
        }
        if (!h_over_idx || !h_over_val || (fmt == XG_LAYOUT_ROWS_TINY && !h_over_col))
            return give_up(XG_E_NOMEM, "out of pinned host memory for the result");
        if (n_over) {
            cudaMemcpyAsync(h_over_idx, d_over_idx, (size_t)n_over * 8, cudaMemcpyDeviceToHost, ctx->d2h_stream);
            cudaMemcpyAsync(h_over_val, d_over_val, (size_t)n_over * 4, cudaMemcpyDeviceToHost, ctx->d2h_stream);
            if (h_over_col) cudaMemcpyAsync(h_over_col, d_over_col, (size_t)n_over * 4, cudaMemcpyDeviceToHost, ctx->d2h_stream);
        }
    }
    int64_t *h_beg = (int64_t *)ctx->pinned_get((size_t)(n_rows + 1) * 8);
    int32_t *h_cnt = (int32_t *)ctx->pinned_get((size_t)(n_rows + 1) * 4);
    if (h_beg) o->bufs.push_back(h_beg);
    if (h_cnt) o->bufs.push_back(h_cnt);
    if (!h_beg || !h_cnt) return give_up(XG_E_NOMEM, "out of pinned host memory for the result");
    cudaMemcpyAsync(h_beg, c.seg_base, (size_t)n_rows * 8, cudaMemcpyDeviceToHost, ctx->d2h_stream);
    cudaMemcpyAsync(h_cnt, c.seg_nnz, (size_t)n_rows * 4, cudaMemcpyDeviceToHost, ctx->d2h_stream);
    cudaEventRecord(ctx->ev[3], ctx->stream);
    ce = cudaStreamSynchronize(ctx->d2h_stream);
    if (ce != cudaSuccess) return give_up(XG_E_CUDA, std::string("result D2H: ") + cudaGetErrorString(ce));
    cudaEventSynchronize(ctx->ev[3]);
    ctx->pinned_put(c.h_cur);
    ctx->fx_nnz_hint = nnz;
    ctx->fx_res_valid = true;
    ctx->fx_res_nnz = nnz;
    ctx->fx_res_rows = n_rows;
    ctx->fx_res_cols = n_cols;
    ctx->timing[4] = ms_since(t_tail);
    o->m.nnz = nnz;
    o->m.n_rows = n_rows;
    o->m.n_cols = n_cols;
    o->m.col = h_col;
    o->m.val = h_val;
    o->m.colval16 = h_packed;
    o->m.n_over = (int64_t)n_over;
    o->m.over_idx = (const int64_t *)h_over_idx;
    o->m.over_val = h_over_val;
    o->m.coldelta16 = h_tiny;
    o->m.over_col = h_over_col;
    o->m.row_beg = h_beg;
    o->m.row_cnt = h_cnt;
    *out = &o->m;
    return XG_OK;
}

// xg_last_timing of the call (include/xcltk_b200.h); [4], the result copy, is set by the result phase.
static void basefc_timing(const BasefcCall &c, std::chrono::steady_clock::time_point t_call) {
    xg_ctx *ctx = c.ctx;
    float t_all = 0, t_span = 0;
    double t_cnt = 0;
    cudaEventElapsedTime(&t_all, ctx->ev[0], ctx->ev[3]);
    for (int32_t e = 0; e < c.n_epochs; e++) {
        float t = 0;
        cudaEventElapsedTime(&t, c.ev(0, e), c.ev(1, e));
        t_cnt += t;
    }
    cudaEventElapsedTime(&t_span, c.ev_init(), ctx->ev[3]);
    ctx->timing[0] = t_all;      // device time of the call: planning kernels, zero, count, finalize, gather
    ctx->timing[1] = t_cnt;      // sum over epochs of the counting kernel
    ctx->timing[2] = c.launches;
    ctx->timing[3] = t_span;     // epochs + scan + gather (no host planning in between)
    ctx->timing[5] = c.n_epochs;
    ctx->timing[6] = (double)c.plan.pool_bytes;
    ctx->timing[7] = (double)c.plan.staging_cap;
    ctx->timing[8] = c.ms_index;
    ctx->timing[9] = c.ms_windows;
    ctx->timing[10] = c.ms_alloc;
    ctx->timing[11] = c.ms_upload;
    ctx->timing[12] = ms_since(t_call);
    ctx->timing[13] = (double)c.h2d_bytes;
    ctx->timing[14] = (double)c.plan.n_seg_feat;
    ctx->timing[15] = (double)c.plan.n_set_feat;
}

// `src` != nullptr: the records of `rd` are copied from the pinned host batch `src` epoch by epoch (BasefcCall).
static int basefc_run(xg_ctx *ctx, const xg_dreads *rd, const xg_reads *src, const xg_features *feats,
                      const xg_barcodes *cells, const xg_params *par, int32_t layout, xg_coo **out,
                      bool force_sets = false) {
    if (!ctx || !ctx->stream) return ctx ? ctx->fail(XG_E_CUDA, "context has no device") : XG_E_ARG;
    if (!rd || !feats || !cells || !par || !out) return ctx->fail(XG_E_ARG, "xg_basefc: null argument");
    if (layout < XG_LAYOUT_CSR || layout > XG_LAYOUT_ROWS_TINY) return ctx->fail(XG_E_ARG, "xg_basefc: unknown layout");
    if (feats->n < 0 || cells->n_samples <= 0) return ctx->fail(XG_E_ARG, "xg_basefc: empty sample list");
    if (par->use_cell_tag && cells->n != cells->n_samples)
        return ctx->fail(XG_E_ARG, "xg_basefc: barcode mode needs one key per column");
    if (rd->mapped) return ctx->fail(XG_E_ARG, "xg_basefc: needs an uploaded batch (xg_upload_reads), not xg_map_reads");
    XG_CUDA(cudaSetDevice(ctx->device));
    ctx->fx_res_valid = false;
    for (double &t : ctx->timing) t = 0;
    BasefcCall c;
    memset(&c.P, 0, sizeof(c.P));
    c.ctx = ctx;
    c.rd = rd;
    c.src = src;
    c.n_rows = feats->n;
    c.n_cols = cells->n_samples;
    c.dbg_sync = getenv("XG_DEBUG_SYNC") && atoi(getenv("XG_DEBUG_SYNC")) != 0;
    int32_t n_gid = 0;
    for (auto &r : rd->h_runs) n_gid = std::max(n_gid, r.gid + 1);
    if (!par->use_cell_tag)
        for (auto &r : rd->h_runs)
            if (r.bam_idx >= c.n_cols) return ctx->fail(XG_E_ARG, "more BAMs than sample columns");
    const auto t_call = std::chrono::steady_clock::now();
    c.fs_stats = (unsigned long long *)ctx->get("fx_fs_stats", sizeof(unsigned long long) * FS_STATS);
    if (!c.fs_stats) return XG_E_CUDA;
    // a call redone with sets keeps the counts of its first attempt, whose segments were reduced
    if (!force_sets) XG_CUDA(cudaMemsetAsync(c.fs_stats, 0, sizeof(unsigned long long) * FS_STATS, ctx->stream));
    int rc = XG_OK;
    if ((rc = basefc_params(c, cells, par)) || (rc = basefc_windows(c, feats, n_gid)) ||
        (rc = basefc_plan(c, force_sets)) || (rc = basefc_epochs(c, layout != XG_LAYOUT_CSR)))
        return rc;
    if (layout != XG_LAYOUT_CSR)
        rc = basefc_collect_rows(c, layout, out);
    else
        rc = xg_staging_to_coo(ctx, "fx", c.n_rows, c.n_cols, c.seg_base, c.seg_nnz, c.st_col, c.st_val, out, &c.launches);
    if (rc) return rc;
    basefc_timing(c, t_call);
    if (c.seg_mode) {             // did every UMI key fit the pair word?
        unsigned int h_flags = 0;
        XG_CUDA(cudaMemcpy(&h_flags, c.P.flags, sizeof(h_flags), cudaMemcpyDeviceToHost));
        if (h_flags & 1u) {
            xg_coo_free(*out);
            *out = nullptr;
            const_cast<xg_dreads *>(rd)->umi_compact = 0;
            return basefc_run(ctx, rd, src, feats, cells, par, layout, out, true);
        }
    }
    return XG_OK;
}

extern "C" int xg_basefc(xg_ctx *ctx, const xg_dreads *rd, const xg_features *feats,
                         const xg_barcodes *cells, const xg_params *par, int32_t layout, xg_coo **out) {
    return basefc_run(ctx, rd, nullptr, feats, cells, par, layout, out);
}

extern "C" int xg_basefc_host(xg_ctx *ctx, const xg_reads *h, const xg_features *feats,
                              const xg_barcodes *cells, const xg_params *par, int32_t layout, xg_coo **out) {
    if (!ctx || !ctx->stream) return ctx ? ctx->fail(XG_E_CUDA, "context has no device") : XG_E_ARG;
    if (!h) return ctx->fail(XG_E_ARG, "xg_basefc_host: null argument");
    XG_CUDA(cudaSetDevice(ctx->device));
    cudaPointerAttributes at;
    if (h->n_reads > 0 && (cudaPointerGetAttributes(&at, h->pos_end) != cudaSuccess || at.type != cudaMemoryTypeHost)) {
        cudaGetLastError();
        return ctx->fail(XG_E_ARG, "xg_basefc_host: record arrays must be pinned host memory");
    }
    xg_dreads *d = xg_dreads_new(h);
    const size_t n = (size_t)h->n_reads;
    d->pos_end = (int2 *)ctx->dev_get(n * 8 + 64);
    d->fmq = (uint32_t *)ctx->dev_get(n * 4 + 64);
    d->cig_off = (uint32_t *)ctx->dev_get((n + 1) * 4 + 64);
    d->keys = (ulonglong2 *)ctx->dev_get(n * 16 + 64);
    d->cigar = (uint32_t *)ctx->dev_get((size_t)h->n_cigar * 4 + 64);
    d->runs = (xg_run *)ctx->dev_get((size_t)h->n_runs * sizeof(xg_run) + 16);
    d->tiles = (xg_tile *)ctx->dev_get((size_t)h->n_tiles * sizeof(xg_tile) + 16);
    int rc = XG_OK;
    if (!d->pos_end || !d->fmq || !d->cig_off || !d->keys || !d->cigar || !d->runs || !d->tiles) {
        rc = ctx->fail(XG_E_CUDA, "out of device memory for the read batch");
    } else {
        cudaMemcpyAsync(d->runs, h->runs, (size_t)h->n_runs * sizeof(xg_run), cudaMemcpyHostToDevice, ctx->stream);
        cudaMemcpyAsync(d->tiles, h->tiles, (size_t)h->n_tiles * sizeof(xg_tile), cudaMemcpyHostToDevice, ctx->stream);
        rc = xg_make_tile_pmax(ctx, d);
        if (!rc) rc = basefc_run(ctx, d, h, feats, cells, par, layout, out);
    }
    cudaStreamSynchronize(ctx->stream);
    xg_dreads_free(ctx, d);
    return rc;
}

// ---- Matrix-Market text on the device (SURVEY.md 8f N2) ----------------------------------------------------------
// Replaces merge_mtx (rdr/fc/utils.py:54-94) for the rows of the last xg_basefc call with a rows layout, which are
// still in the staging area: one warp per row sizes its lines ("<output row>\t<column + 1>\t<count>\n"), a scan
// places the rows in input order, one warp per row writes its lines, and the text leaves through a ring of pinned
// buffers that writer threads pwrite() at their offsets (several at a time: the page cache takes them in parallel).
namespace {
__device__ __forceinline__ int mtx_digits(uint32_t v) {
    return v < 10u ? 1 : v < 100u ? 2 : v < 1000u ? 3 : v < 10000u ? 4 : v < 100000u ? 5 : v < 1000000u ? 6
           : v < 10000000u ? 7 : v < 100000000u ? 8 : v < 1000000000u ? 9 : 10;
}
__device__ __forceinline__ char *mtx_put(char *p, uint32_t v, int nd) {
    for (int k = nd - 1; k >= 0; k--) {
        p[k] = (char)('0' + v % 10u);
        v /= 10u;
    }
    return p + nd;
}
__global__ void k_mtx_row_bytes(int32_t n_rows, const int64_t *seg_base, const int32_t *seg_nnz, const int32_t *st_col,
                                const int32_t *st_val, const int32_t *out_row, int32_t *row_bytes) {
    const int r = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (r >= n_rows) return;
    const int32_t n = seg_nnz[r], orow = out_row[r];
    int bytes = 0;
    if (n > 0 && orow > 0) {
        const int64_t b = seg_base[r];
        const int dr = mtx_digits((uint32_t)orow) + 3;
        for (int k = lane; k < n; k += 32) bytes += dr + mtx_digits((uint32_t)st_col[b + k] + 1u) + mtx_digits((uint32_t)st_val[b + k]);
    }
    for (int d = 16; d > 0; d >>= 1) bytes += __shfl_xor_sync(0xffffffffu, bytes, d);
    if (lane == 0) row_bytes[r] = bytes;
}
__global__ void k_mtx_write(int32_t n_rows, const int64_t *seg_base, const int32_t *seg_nnz, const int32_t *st_col,
                            const int32_t *st_val, const int32_t *out_row, const int64_t *row_off, char *text) {
    const int r = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (r >= n_rows) return;
    const int32_t n = seg_nnz[r], orow = out_row[r];
    if (n <= 0 || orow <= 0) return;
    const int64_t b = seg_base[r];
    const int dr = mtx_digits((uint32_t)orow);
    int64_t at = row_off[r];
    for (int k0 = 0; k0 < n; k0 += 32) {
        const int k = k0 + lane;
        uint32_t c = 0, v = 0;
        int dc = 0, dv = 0, len = 0;
        if (k < n) {
            c = (uint32_t)st_col[b + k] + 1u;
            v = (uint32_t)st_val[b + k];
            dc = mtx_digits(c);
            dv = mtx_digits(v);
            len = dr + dc + dv + 3;
        }
        int incl = len;
        for (int d = 1; d < 32; d <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += y;
        }
        if (k < n) {
            char *p = text + at + (incl - len);
            p = mtx_put(p, (uint32_t)orow, dr);
            *p++ = '\t';
            p = mtx_put(p, c, dc);
            *p++ = '\t';
            p = mtx_put(p, v, dv);
            *p = '\n';
        }
        at += __shfl_sync(0xffffffffu, incl, 31);
    }
}
}  // namespace

extern "C" int xg_basefc_write_mtx_device(xg_ctx *ctx, const char *path, int32_t n_rows_in, const int32_t *out_row,
                                          int32_t n_rows_out, int32_t n_threads) {
    if (!ctx || !ctx->stream) return ctx ? ctx->fail(XG_E_CUDA, "context has no device") : XG_E_ARG;
    if (!path || !out_row || n_rows_in < 0) return ctx->fail(XG_E_ARG, "xg_basefc_write_mtx_device: bad argument");
    if (!ctx->fx_res_valid || ctx->fx_res_rows != n_rows_in)
        return ctx->fail(XG_E_ARG, "xg_basefc_write_mtx_device: the last basefc call of this context did not produce a rows layout of that many rows");
    XG_CUDA(cudaSetDevice(ctx->device));
    const int32_t n_rows = n_rows_in;
    const int64_t *seg_base = (const int64_t *)ctx->scratch["fx_seg_base"].p;
    const int32_t *seg_nnz = (const int32_t *)ctx->scratch["fx_seg_nnz"].p;
    const int32_t *st_col = (const int32_t *)ctx->scratch["fx_st_col"].p;
    const int32_t *st_val = (const int32_t *)ctx->scratch["fx_st_val"].p;
    XG_GET(d_out_row, int32_t, "mx_out_row", n_rows + 1);
    XG_GET(d_row_bytes, int32_t, "mx_row_bytes", n_rows + 1);
    XG_GET(d_row_off, int64_t, "mx_row_off", n_rows + 2);
    for (int32_t r = 0; r < n_rows; r++)
        if (out_row[r] < 0 || out_row[r] > n_rows_out) return ctx->fail(XG_E_ARG, "xg_basefc_write_mtx_device: output row out of range");
    XG_CUDA(cudaMemcpyAsync(d_out_row, out_row, sizeof(int32_t) * (size_t)n_rows, cudaMemcpyHostToDevice, ctx->stream));
    long long total = 0;
    const unsigned grid = (unsigned)(((unsigned long long)n_rows * 32 + 255) / 256);
    if (n_rows > 0) {
        k_mtx_row_bytes<<<grid, 256, 0, ctx->stream>>>(n_rows, seg_base, seg_nnz, st_col, st_val, d_out_row, d_row_bytes);
        k_exclusive_scan<<<1, 1024, 0, ctx->stream>>>(d_row_bytes, d_row_off, n_rows);
        XG_CUDA(cudaMemcpyAsync(&total, d_row_off + n_rows, 8, cudaMemcpyDeviceToHost, ctx->stream));
    }
    XG_CUDA(cudaStreamSynchronize(ctx->stream));
    char *d_text = (char *)ctx->get("mx_text", (size_t)total + 64);
    if (!d_text) return XG_E_CUDA;
    if (total > 0) k_mtx_write<<<grid, 256, 0, ctx->stream>>>(n_rows, seg_base, seg_nnz, st_col, st_val, d_out_row, d_row_off, d_text);
    XG_CUDA(cudaGetLastError());
    // every staged entry of an emitted row is a line: a row with entries but no output row would be lost
    char header[160];
    // (the count of lines = entries of the rows that have an output row; checked against the result's nnz by the caller)
    std::vector<int32_t> h_cnt((size_t)n_rows + 1);
    XG_CUDA(cudaMemcpyAsync(h_cnt.data(), seg_nnz, sizeof(int32_t) * (size_t)n_rows, cudaMemcpyDeviceToHost, ctx->stream));
    XG_CUDA(cudaStreamSynchronize(ctx->stream));
    long long lines = 0;
    for (int32_t r = 0; r < n_rows; r++) {
        if (h_cnt[(size_t)r] > 0 && out_row[r] <= 0) return ctx->fail(XG_E_ARG, "xg_write_mtx: non-empty row without an output row");
        lines += h_cnt[(size_t)r];
    }
    const int hl = snprintf(header, sizeof header, "%%%%MatrixMarket matrix coordinate integer general\n%%%%\n%d\t%d\t%lld\n",
                            n_rows_out, ctx->fx_res_cols, lines);
    const int fd = open(path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (fd < 0) return ctx->fail(XG_E_IO, std::string("cannot write '") + path + "'");
    bool ok = write(fd, header, (size_t)hl) == hl;
    // ring of pinned buffers: the copy of chunk c + 1 runs while the writers of the chunks before it pwrite()
    // (a small matrix takes one small buffer: pinning memory costs more than writing it)
    const size_t CHUNK_B = std::min<size_t>((size_t)32 << 20, ((size_t)std::max<long long>(total, 1) + 4095) & ~(size_t)4095);
    const int n_buf = (int)std::max<long long>(1, std::min<long long>(std::min(n_threads > 0 ? n_threads : 4, 8),
                                                                     (total + (long long)CHUNK_B - 1) / (long long)CHUNK_B));
    std::vector<char *> buf((size_t)n_buf, nullptr);
    std::vector<std::thread> wr((size_t)n_buf);
    std::vector<char> failed((size_t)n_buf, 0);
    for (int k = 0; k < n_buf; k++)
        if (!(buf[(size_t)k] = (char *)ctx->pinned_get(CHUNK_B))) ok = false;
    int c = 0;
    for (long long off = 0; ok && off < total; off += (long long)CHUNK_B, c++) {
        const int k = c % n_buf;
        if (wr[(size_t)k].joinable()) wr[(size_t)k].join();
        const size_t len = (size_t)std::min<long long>((long long)CHUNK_B, total - off);
        if (cudaMemcpyAsync(buf[(size_t)k], d_text + off, len, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
            cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
            ok = false;
            break;
        }
        char *src = buf[(size_t)k];
        char *flag = &failed[(size_t)k];
        const long long file_off = (long long)hl + off;
        wr[(size_t)k] = std::thread([fd, src, len, file_off, flag] {
            size_t done = 0;
            while (done < len) {
                const ssize_t w = pwrite(fd, src + done, len - done, (off_t)(file_off + (long long)done));
                if (w <= 0) {
                    *flag = 1;
                    return;
                }
                done += (size_t)w;
            }
        });
    }
    for (auto &t : wr)
        if (t.joinable()) t.join();
    for (int k = 0; k < n_buf; k++) {
        if (buf[(size_t)k]) ctx->pinned_put(buf[(size_t)k]);
        if (failed[(size_t)k]) ok = false;
    }
    if (close(fd) != 0) ok = false;
    if (!ok) {
        cudaGetLastError();
        return ctx->fail(XG_E_IO, std::string("short write on '") + path + "'");
    }
    return XG_OK;
}

extern "C" int xg_basefc_finalize_stats(xg_ctx *ctx, int64_t out[8]) {
    if (!ctx || !ctx->stream) return ctx ? ctx->fail(XG_E_CUDA, "context has no device") : XG_E_ARG;
    if (!out) return ctx->fail(XG_E_ARG, "xg_basefc_finalize_stats: null argument");
    XG_CUDA(cudaSetDevice(ctx->device));
    static_assert(FS_STATS == 8, "xg_basefc_finalize_stats reports 8 counters");
    unsigned long long h[FS_STATS] = {};
    auto it = ctx->scratch.find("fx_fs_stats");
    if (it != ctx->scratch.end() && it->second.p) {
        XG_CUDA(cudaStreamSynchronize(ctx->stream));
        XG_CUDA(cudaMemcpy(h, it->second.p, sizeof h, cudaMemcpyDeviceToHost));
    }
    for (int k = 0; k < FS_STATS; k++) out[k] = (int64_t)h[k];
    return XG_OK;
}

// ---- read-assignment summary (xg_basefc_summary) -----------------------------------------------------------------
// One CTA per tile, a thread per record.  Phase 1 reads pos / end only (coalesced) and finds, through the interval
// index of the features, whether the record overlaps one: the features covering `pos` (the stabbing list of its
// segment) or beginning in (pos, end).  Only the records in range go on to their flags, keys and CIGAR: their fate is
// the first of check_read's tests (rdr/fc/core.py:46-62) that fails, else how many features pass the include test
// (rdr/fc/core.py:160-165, as k_basefc_count applies it), counted up to two.  The warp adds its counts per counter
// (match_any on the address) before the global atomics.
namespace {
#define SUM_FATES 7
#define SUM_THREADS 256

struct SummaryDev {
    const int2 *pos_end;
    const uint32_t *fmq, *cig_off, *cigar;
    const ulonglong2 *keys;
    const xg_tile *tiles;
    const xg_run *runs;
    const int32_t *bnd_goff, *bnd, *stab_off, *fb, *sf_end;
    const int4 *stab4;            // {sorted feature, beg, end, -}
    int32_t n_gid, n_samples;
    int32_t own_g0, own_p0, own_g1, own_p1;   // records with (gid, pos) in [(g0, p0), (g1, p1))
    BarcodeTable bc;
    FilterParams fp;
    const int32_t *incl_tab;
    int32_t incl_tab_len, incl_len;
    unsigned long long *out;      // (n_samples + 1) x SUM_FATES
};

// m of the include test for feature [s0, e0) (emit_pair)
__device__ __forceinline__ int32_t summary_m(const uint32_t *cig, uint32_t n_ops, int32_t pos, int32_t end, int32_t aln,
                                             int32_t s0, int32_t e0) {
    if (n_ops == 0) {
        const int32_t a = max(pos, s0), b = min(end, e0);
        return b > a ? b - a : 0;
    }
    if (s0 <= pos && end <= e0) return aln;
    return included_len(cig, n_ops, pos, s0, e0);
}

__global__ void __launch_bounds__(SUM_THREADS) k_basefc_summary(const __grid_constant__ SummaryDev P) {
    __shared__ int32_t s_win[2];  // the tile's window of boundaries [lo, hi) for the search of every record
    const xg_tile tl = P.tiles[blockIdx.x];
    const int32_t gid = P.runs[tl.run].gid;
    if (gid < 0 || gid >= P.n_gid) return;
    const int32_t b0 = P.bnd_goff[gid], b1 = P.bnd_goff[gid + 1];
    if (b0 == b1) return;                                     // a contig without features
    if (gid < P.own_g0 || gid > P.own_g1 || (gid == P.own_g1 && tl.first_pos >= P.own_p1)) return;
    if (threadIdx.x == 0) {
        // every record's pos is >= first_pos: its first boundary > pos is >= the first one > first_pos, and (when
        // pos < max_end) <= the first one >= max_end
        int32_t lo = b0, hi = b1;
        while (lo < hi) {
            const int32_t mid = (lo + hi) >> 1;
            if (P.bnd[mid] <= tl.first_pos) lo = mid + 1; else hi = mid;
        }
        int32_t a = lo;
        hi = b1;
        while (a < hi) {
            const int32_t mid = (a + hi) >> 1;
            if (P.bnd[mid] < tl.max_end) a = mid + 1; else hi = mid;
        }
        s_win[0] = lo;
        s_win[1] = a;
    }
    __syncthreads();
    const int32_t w_lo = s_win[0], w_hi = s_win[1];
    const int32_t col_tile = P.runs[tl.run].bam_idx;
    for (int32_t base = 0; base < tl.n_rec; base += SUM_THREADS) {    // the same trip count for every thread
        const int32_t k = base + (int32_t)threadIdx.x;
        bool on = false;
        int32_t row = 0, fate = 0;
        if (k < tl.n_rec) {
            const int64_t i = tl.rec_beg + k;
            const int2 pe = __ldcs(&P.pos_end[i]);
            const bool own = (gid > P.own_g0 || (gid == P.own_g0 && pe.x >= P.own_p0)) &&
                             (gid < P.own_g1 || (gid == P.own_g1 && pe.x < P.own_p1));
            int32_t ub = w_hi, s0i = 0, s1i = 0;
            if (own) {
                int32_t lo = w_lo, hi = pe.x < tl.max_end ? w_hi : b1;
                while (lo < hi) {                             // first boundary > pos
                    const int32_t mid = (lo + hi) >> 1;
                    if (__ldg(&P.bnd[mid]) <= pe.x) lo = mid + 1; else hi = mid;
                }
                ub = lo;
                if (ub > b0) {
                    s0i = __ldg(&P.stab_off[ub - 1]);
                    s1i = __ldg(&P.stab_off[ub]);
                }
                // phase 1: in range iff some feature overlaps [pos, end) (pos < f.end && end > f.beg)
                for (int32_t s = s0i; s < s1i && !on; s++) {
                    const int4 f = __ldg(&P.stab4[s]);
                    on = pe.x < f.z && pe.y > f.y;
                }
                for (int32_t kb = ub; kb < b1 && !on; kb++) {  // features beginning at a boundary in (pos, end)
                    if (__ldg(&P.bnd[kb]) >= pe.y) break;
                    on = __ldg(&P.fb[kb + 1]) > __ldg(&P.fb[kb]);
                }
            }
            if (on) {
                const uint32_t fmq = P.fmq[i];
                if (P.fp.use_cell_tag) {
                    const uint64_t ck = P.keys[i].x;
                    const int32_t c = ck == XG_KEY_NONE ? -1 : barcode_lookup(P.bc, ck);
                    row = c < 0 ? P.n_samples : c;
                } else {
                    row = col_tile;
                }
                if ((int32_t)((fmq >> 16) & 0xffu) < P.fp.min_mapq) {
                    fate = 0;
                } else if (!read_passes_flags(P.fp, fmq)) {           // the mapq test passed: a flag test failed
                    fate = 1;
                } else if (P.fp.need_umi_tag && (P.keys[i].y == XG_KEY_NONE || P.keys[i].y == XG_KEY_EMPTY)) {
                    fate = 2;
                } else {
                    uint32_t n_ops = fmq >> 24;
                    const uint32_t *cig = nullptr;
                    int32_t aln;
                    if (n_ops == 0) {
                        aln = pe.y - pe.x;
                    } else {
                        const uint32_t co = P.cig_off[i];
                        cig = P.cigar + co;
                        if (n_ops == 255) n_ops = cig[-1];
                        aln = 0;
                        for (uint32_t q = 0; q < n_ops; q++) {
                            const uint32_t cw = cig[q];
                            if (cig_aligned(cw & 15u)) aln += (int32_t)(cw >> 4);
                        }
                    }
                    if (aln < P.fp.min_len) {
                        fate = 3;
                    } else {
                        const int32_t need =
                            P.incl_tab ? __ldg(&P.incl_tab[min(aln, P.incl_tab_len - 1)]) : P.incl_len;
                        int n_pass = 0;
                        for (int32_t s = s0i; s < s1i && n_pass < 2; s++) {
                            const int4 f = __ldg(&P.stab4[s]);
                            if (pe.x < f.z && pe.y > f.y)
                                n_pass += summary_m(cig, n_ops, pe.x, pe.y, aln, f.y, f.z) >= need;
                        }
                        for (int32_t kb = ub; kb < b1 && n_pass < 2; kb++) {
                            const int32_t bv = __ldg(&P.bnd[kb]);
                            if (bv >= pe.y) break;
                            const int32_t j1 = __ldg(&P.fb[kb + 1]);
                            for (int32_t j = __ldg(&P.fb[kb]); j < j1 && n_pass < 2; j++)
                                n_pass += summary_m(cig, n_ops, pe.x, pe.y, aln, bv, __ldg(&P.sf_end[j])) >= need;
                        }
                        fate = 4 + n_pass;
                    }
                }
            }
        }
        warp_add<unsigned long long>(on, &P.out[(int64_t)row * SUM_FATES + fate], 1ull);
    }
}
}  // namespace

extern "C" int xg_basefc_summary(xg_ctx *ctx, const xg_dreads *rd, const xg_features *feats, const xg_barcodes *cells,
                                 const xg_params *par, const int32_t *own, int64_t *out) {
    if (!ctx || !ctx->stream) return ctx ? ctx->fail(XG_E_CUDA, "context has no device") : XG_E_ARG;
    if (!rd || !feats || !cells || !par || !out) return ctx->fail(XG_E_ARG, "xg_basefc_summary: null argument");
    if (feats->n < 0 || cells->n_samples <= 0) return ctx->fail(XG_E_ARG, "xg_basefc_summary: empty sample list");
    if (par->use_cell_tag && cells->n != cells->n_samples)
        return ctx->fail(XG_E_ARG, "xg_basefc_summary: barcode mode needs one key per column");
    if (par->min_incl_tab && par->min_incl_tab_len <= rd->max_aln_len)
        return ctx->fail(XG_E_ARG, "min_incl_tab shorter than max aligned length + 1");
    // the kernel's loads: keys as 16-byte pairs, pos / end as 8-byte pairs, the rest as 32-bit words
    if (((uintptr_t)rd->keys & 15) | ((uintptr_t)rd->pos_end & 7) |
        (((uintptr_t)rd->fmq | (uintptr_t)rd->cig_off | (uintptr_t)rd->cigar) & 3))
        return ctx->fail(XG_E_ARG, "xg_basefc_summary: record arrays are not aligned to their element pairs / words");
    XG_CUDA(cudaSetDevice(ctx->device));
    int32_t n_gid = 0;
    for (auto &r : rd->h_runs) n_gid = std::max(n_gid, r.gid + 1);
    if (!par->use_cell_tag)
        for (auto &r : rd->h_runs)
            if (r.bam_idx >= cells->n_samples) return ctx->fail(XG_E_ARG, "more BAMs than sample columns");
    for (double &t : ctx->timing) t = 0;
    const auto t_call = std::chrono::steady_clock::now();
    FeatCache *fc = nullptr;
    bool cached = false;
    int rc = feat_index(ctx, feats, n_gid, &fc, &cached);
    if (!rc && !cached) rc = feat_index_upload(ctx, fc);
    if (rc) return rc;
    SummaryDev P;
    memset(&P, 0, sizeof(P));
    P.pos_end = rd->pos_end;
    P.fmq = rd->fmq;
    P.cig_off = rd->cig_off;
    P.cigar = rd->cigar;
    P.keys = rd->keys;
    P.tiles = rd->tiles;
    P.runs = rd->runs;
    P.bnd_goff = (const int32_t *)ctx->scratch["fx_bnd_goff"].p;
    P.bnd = (const int32_t *)ctx->scratch["fx_bnd"].p;
    P.stab_off = (const int32_t *)ctx->scratch["fx_stab_off"].p;
    P.fb = (const int32_t *)ctx->scratch["fx_fb"].p;
    P.sf_end = (const int32_t *)ctx->scratch["fx_sf_end"].p;
    P.stab4 = (const int4 *)ctx->scratch["fx_stab4"].p;
    P.n_gid = n_gid;
    P.n_samples = cells->n_samples;
    P.own_g0 = own ? own[0] : INT32_MIN;
    P.own_p0 = own ? own[1] : INT32_MIN;
    P.own_g1 = own ? own[2] : INT32_MAX;
    P.own_p1 = own ? own[3] : INT32_MAX;
    P.fp.min_mapq = par->min_mapq;
    P.fp.min_len = par->min_len;
    P.fp.incl_flag = par->incl_flag;
    P.fp.excl_flag = par->excl_flag;
    P.fp.no_orphan = par->no_orphan;
    P.fp.use_cell_tag = par->use_cell_tag;
    P.fp.need_umi_tag = par->need_umi_tag;
    P.incl_len = par->min_incl_len;
    if (par->min_incl_tab) {
        XG_GET(d_incl, int32_t, "sm_incl_tab", par->min_incl_tab_len + 1);
        XG_CUDA(cudaMemcpyAsync(d_incl, par->min_incl_tab, sizeof(int32_t) * (size_t)par->min_incl_tab_len,
                                cudaMemcpyHostToDevice, ctx->stream));
        P.incl_tab = d_incl;
        P.incl_tab_len = par->min_incl_tab_len;
    }
    if (par->use_cell_tag && (rc = xg_build_barcode_table(ctx, cells, &P.bc))) return rc;
    const size_t n_out = ((size_t)cells->n_samples + 1) * SUM_FATES;
    XG_GET(d_out, unsigned long long, "sm_out", n_out);
    P.out = d_out;
    XG_CUDA(cudaMemsetAsync(d_out, 0, sizeof(unsigned long long) * n_out, ctx->stream));
    cudaEventRecord(ctx->ev[0], ctx->stream);
    if (rd->n_tiles > 0 && n_gid > 0) k_basefc_summary<<<(unsigned)rd->n_tiles, SUM_THREADS, 0, ctx->stream>>>(P);
    XG_CUDA(cudaGetLastError());
    cudaEventRecord(ctx->ev[1], ctx->stream);
    static_assert(sizeof(unsigned long long) == sizeof(int64_t), "counters are 64-bit");
    XG_CUDA(cudaMemcpyAsync(out, d_out, sizeof(int64_t) * n_out, cudaMemcpyDeviceToHost, ctx->stream));
    XG_CUDA(cudaStreamSynchronize(ctx->stream));
    float t_k = 0;
    cudaEventElapsedTime(&t_k, ctx->ev[0], ctx->ev[1]);
    ctx->timing[0] = t_k;
    ctx->timing[1] = t_k;
    ctx->timing[2] = rd->n_tiles > 0 && n_gid > 0 ? 1 : 0;
    ctx->timing[12] = ms_since(t_call);
    return XG_OK;
}
