// gpu_decode.cu -- BAM -> read batch on the device: BGZF inflate + record parse.
//
// Same result, array for array, as the host decoder (decode.cpp: xg_decode_bams followed by
// xg_upload_reads); replaces what the reference gets from pysam/htslib on its counting paths
// (pysam.AlignmentFile + fetch(), xcltk/rdr/fc/core.py:75,100; xcltk/baf/fc/core.py:60,99).
// The compressed file crosses PCIe once (~55 B/read), every BGZF block is inflated and
// CRC-checked by one warp (inflate.cuh), and the records are parsed where they land, window by
// window, into the batch arrays.
//
// Block-parallel parsing needs every BGZF block to start at a record boundary.  htslib
// writes BAM that way (bam_write1 flushes the block before a record that does not fit, and
// the header ends with a flush), so files from samtools / cellranger / STARsolo qualify; the
// walk kernel verifies it and any other layout returns XG_E_UNSUPPORTED so that the caller
// uses xg_decode_bams + xg_upload_reads instead.  Cell / UMI values that do not pack into 63
// bits are gathered here and interned by the host keyspace.  Both decoders are decoders:
// neither counts anything, and the counting kernels stay device-only.
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <thread>

#include "bamfile.hpp"
#include "common.cuh"
#include "inflate.cuh"
#include "keys.hpp"
#include "owner.hpp"

namespace {


// ---- unaligned little-endian loads (buffers are padded by 8 bytes) --------------------------
__device__ __forceinline__ uint32_t ld32u(const uint8_t *p) {
    const uintptr_t a = (uintptr_t)p;
    const uint32_t *w = (const uint32_t *)(a & ~(uintptr_t)3);
    const uint32_t sh = (uint32_t)(a & 3) * 8;
    const uint32_t lo = w[0];
    if (sh == 0) return lo;
    return __funnelshift_r(lo, w[1], sh);
}
__device__ __forceinline__ uint32_t ld16u(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }

struct BlkInfo {
    uint32_t n_all;      // records in the block
    uint32_t n_kept;     // ... on a contig the caller asked for
    uint32_t cig;        // cigar words the kept records store
    uint32_t seq;        // sequence words
    unsigned long long first_key, last_key;   // (tid, pos) of the first / last record; unplaced sort last
    uint32_t status;     // 0 ok, 1 block does not hold whole records, 2 corrupt record, 3 unsorted
    uint32_t n_starts;   // run-start entries the block will emit (first kept record + tid changes)
};

// One group of S lanes per BGZF block (inflate.cuh); INFLATE_THREADS / S blocks per CTA.
constexpr int INFLATE_THREADS = 128;
template <int S>
__global__ void __launch_bounds__(INFLATE_THREADS) k_inflate(const uint8_t *comp, const BgzfBlockDev *blocks,
                                                             int32_t n_blocks, int *n_bad) {
    extern __shared__ __align__(16) unsigned char inflate_smem[];
    xg_inflate::GroupSmem *gs = reinterpret_cast<xg_inflate::GroupSmem *>(inflate_smem);
    const int grp = threadIdx.x / S;
    const int b = blockIdx.x * (INFLATE_THREADS / S) + grp;
    if (b >= n_blocks) return;
    const BgzfBlockDev bk = blocks[b];
    if (bk.isize == 0) return;
    const int n = xg_inflate::inflate_group<S>(gs[grp], comp + bk.coff, bk.clen, bk.uptr, bk.isize);
    bool bad = n != (int)bk.isize;
    if (S == 32 && !bad) {
        __syncwarp();                                  // the block's bytes, written by all lanes; the tables are idle now
        xg_inflate::crc_build_table(gs[grp].lut);
        __syncwarp();
        bad = xg_inflate::crc32_warp(gs[grp].lut, bk.uptr, bk.isize) != bk.crc;    // gzip trailer, as htslib checks
    }
    if ((threadIdx.x & (S - 1)) == 0 && bad) atomicAdd(n_bad, 1);
}

template <int S>
void launch_inflate_s(cudaStream_t st, const uint8_t *comp, const BgzfBlockDev *blocks, int32_t n_blocks, int *n_bad) {
    constexpr int per_cta = INFLATE_THREADS / S;
    const size_t smem = per_cta * sizeof(xg_inflate::GroupSmem);
    static bool attr_set = false;
    if (!attr_set) {
        cudaFuncSetAttribute(k_inflate<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        attr_set = true;
    }
    k_inflate<S><<<(unsigned)((n_blocks + per_cta - 1) / per_cta), INFLATE_THREADS, smem, st>>>(comp, blocks, n_blocks,
                                                                                              n_bad);
}

// One warp per BGZF block.  Sub-warp groups (2-8 blocks per warp, inflate_group<16/8/4>) were measured
// slower: 102 / 156 / 267 ms against 76 ms on the same file -- divergent decoders serialise.
inline void launch_inflate(cudaStream_t st, const uint8_t *comp, const BgzfBlockDev *blocks, int32_t n_blocks,
                           int *n_bad) {
    if (n_blocks <= 0) return;
    launch_inflate_s<32>(st, comp, blocks, n_blocks, n_bad);
}

__device__ __forceinline__ unsigned long long sort_key(int32_t tid, int32_t pos) {
    if (tid < 0) return 0x7fffffff00000000ull;
    return ((unsigned long long)(uint32_t)tid << 32) | (uint32_t)pos;
}

struct RecGeom {
    int32_t pos, end, aln;
    uint32_t fmq, n_words, seq_words, n_cig, l_name, l_seq;
    bool ok;
};

// decode.cpp: rec_info()
__device__ __forceinline__ RecGeom rec_geom(const uint8_t *r, uint32_t bs, bool want_seq) {
    RecGeom o;
    o.pos = (int32_t)ld32u(r + 8);
    const uint32_t w12 = ld32u(r + 12), w16 = ld32u(r + 16);
    o.l_name = w12 & 0xff;
    const uint32_t mapq = (w12 >> 8) & 0xff;
    o.n_cig = w16 & 0xffff;
    const uint32_t flag = w16 >> 16;
    o.l_seq = ld32u(r + 20);
    const unsigned long long need = 36ull + o.l_name + 4ull * o.n_cig + ((unsigned long long)o.l_seq + 1) / 2 + o.l_seq;
    o.ok = need <= (unsigned long long)bs + 4ull && o.l_seq < 0x40000000u;
    if (!o.ok) return o;
    const uint8_t *cig = r + 36 + o.l_name;
    long long rlen = 0, aln = 0;
    uint32_t first_op = 15;
    for (uint32_t i = 0; i < o.n_cig; i++) {
        const uint32_t w = ld32u(cig + 4 * i), op = w & 15, l = w >> 4;
        if (i == 0) first_op = op;
        if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) rlen += l;
        if (op == 0 || op == 7 || op == 8) aln += l;
    }
    if (flag & 4) rlen = 0;
    if (rlen == 0) rlen = 1;
    o.end = (int32_t)(o.pos + rlen);
    o.aln = (int32_t)aln;
    const bool simple = o.n_cig == 1 && (first_op == 0 || first_op == 7 || first_op == 8) && aln == rlen && !(flag & 4);
    uint32_t ncw;
    if (simple) {
        ncw = 0;
        o.n_words = 0;
    } else if (o.n_cig == 0) {
        ncw = 1;
        o.n_words = 1;
    } else if (o.n_cig < 255) {
        ncw = o.n_cig;
        o.n_words = o.n_cig;
    } else {
        ncw = 255;
        o.n_words = o.n_cig + 1;
    }
    o.fmq = flag | (mapq << 16) | (ncw << 24);
    o.seq_words = want_seq ? (((o.l_seq + 1) / 2 + 3) / 4) : 0;
    return o;
}

// One thread per BGZF block: check that the block holds whole records in coordinate order and
// size what the kept ones will store.
__global__ void k_walk(const BgzfBlockDev *blocks, int32_t n_blocks, unsigned long long hdr_end,
                       const int32_t *tid_map, int32_t n_ref, int want_seq, BlkInfo *info, int *maxes) {
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_blocks) return;
    const BgzfBlockDev bk = blocks[b];
    BlkInfo bi;
    bi.n_all = bi.n_kept = bi.cig = bi.seq = 0;
    bi.first_key = ~0ull;
    bi.last_key = 0;
    bi.status = 0;
    bi.n_starts = 0;
    if (bk.uoff + bk.isize <= hdr_end) {
        info[b] = bi;
        return;
    }
    uint32_t off = bk.uoff < hdr_end ? (uint32_t)(hdr_end - bk.uoff) : 0u;      // offsets within the block
    const uint32_t end = bk.isize;
    int32_t max_aln = 0, max_span = 0, prev_kept_tid = -2;
    while (off < end) {
        if (off + 4 > end) {
            bi.status = 1;
            break;
        }
        const uint8_t *r = bk.uptr + off;
        const uint32_t bs = ld32u(r);
        if (bs < 32) {
            bi.status = 2;
            break;
        }
        if ((unsigned long long)off + 4ull + bs > end) {
            bi.status = 1;
            break;
        }
        const int32_t tid = (int32_t)ld32u(r + 4), pos = (int32_t)ld32u(r + 8);
        if (tid >= n_ref) {
            bi.status = 2;
            break;
        }
        const unsigned long long key = sort_key(tid, pos);
        if (bi.n_all == 0) bi.first_key = key;
        else if (key < bi.last_key) bi.status = 3;
        bi.last_key = key;
        bi.n_all++;
        if (tid >= 0 && tid_map[tid] >= 0) {
            const RecGeom g = rec_geom(r, bs, want_seq != 0);
            if (!g.ok) {
                bi.status = 2;
                break;
            }
            bi.n_kept++;
            bi.cig += g.n_words;
            bi.seq += g.seq_words;
            max_aln = max(max_aln, g.aln);
            max_span = max(max_span, g.end - g.pos);
            if (tid != prev_kept_tid) bi.n_starts++;
            prev_kept_tid = tid;
        }
        off += 4u + bs;
    }
    info[b] = bi;
    if (max_aln > 0) atomicMax(&maxes[0], max_aln);
    if (max_span > 0) atomicMax(&maxes[1], max_span);
}

// keys.hpp: key_pack().  Returns false when the string needs the host's intern table.
__device__ __forceinline__ bool pack_key(const uint8_t *s, const uint8_t *end, bool nul_terminated, int n_fixed,
                                         unsigned long long *out) {
    unsigned long long k = 0;
    int bits = 0;
    for (int i = 0; nul_terminated ? (s + i < end) : (i < n_fixed); i++) {
        const uint32_t c = s[i];
        if (nul_terminated && c == 0) break;
        int code;
        switch (c) {
            case 'A': code = 1; break;
            case 'C': code = 2; break;
            case 'G': code = 3; break;
            case 'T': code = 4; break;
            case 'N': code = 5; break;
            case '-': code = 6; break;
            default: code = (c >= '0' && c <= '9') ? 7 : -1;
        }
        if (code < 0) return false;
        if (code < 7) {
            if (bits + 3 > 63) return false;
            k |= (unsigned long long)code << (63 - bits - 3);
            bits += 3;
        } else {
            if (bits + 7 > 63) return false;
            k |= (unsigned long long)((7u << 4) | (c - '0')) << (63 - bits - 7);
            bits += 7;
        }
    }
    *out = k;
    return true;
}

// What a cell / UMI value turns into.  status 0: `key` is final (packed, NONE, EMPTY, NOMATCH);
// 1: the value needs the host's intern table -- the string [s, s + n), or for an integer UMI tag
// the spelling "\x01<decimal>" of decode.cpp's tag_key() (n counts its bytes); 2: a value this
// decoder does not spell (float UMI tag).
struct KeyRef {
    int status;
    unsigned long long key;
    const uint8_t *s;
    uint32_t n;
    long long iv;
    bool is_int;
};

__device__ __forceinline__ uint32_t dec_digits(unsigned long long v) {
    uint32_t d = 1;
    while (v >= 10) {
        v /= 10;
        d++;
    }
    return d;
}

// decode.cpp: tag_key() for the value at `t` (type byte first)
__device__ __forceinline__ KeyRef key_ref_tag(const uint8_t *t, const uint8_t *end, bool is_cell) {
    KeyRef k;
    k.status = 0;
    k.key = XG_KEY_NOMATCH;
    k.s = nullptr;
    k.n = 0;
    k.iv = 0;
    k.is_int = false;
    const uint32_t typ = t[0];
    const uint8_t *v = t + 1;
    if (typ == 'Z' || typ == 'H' || typ == 'A') {
        uint32_t n = 1;
        if (typ != 'A') {
            n = 0;
            while (v + n < end && v[n]) n++;
        }
        if (pack_key(v, end, false, (int)n, &k.key)) return k;
        k.status = 1;
        k.s = v;
        k.n = n;
        return k;
    }
    if (is_cell) return k;                      // not a string: never equals a barcode
    switch (typ) {
        case 'c': k.iv = (signed char)v[0]; break;
        case 'C': k.iv = v[0]; break;
        case 's': k.iv = (short)ld16u(v); break;
        case 'S': k.iv = (long long)ld16u(v); break;
        case 'i': k.iv = (int)ld32u(v); break;
        case 'I': k.iv = (long long)ld32u(v); break;
        case 'f':
            if (ld32u(v) == 0u || ld32u(v) == 0x80000000u) k.key = XG_KEY_EMPTY;      // 0.0f / -0.0f: falsy
            else k.status = 2;
            return k;
        default: return k;                      // NOMATCH
    }
    if (k.iv == 0) {
        k.key = XG_KEY_EMPTY;                   // `if umi:` -- a zero is falsy
        return k;
    }
    k.status = 1;
    k.is_int = true;
    k.n = 1 + (k.iv < 0 ? 1u : 0u) + dec_digits(k.iv < 0 ? (unsigned long long)(-k.iv) : (unsigned long long)k.iv);
    return k;
}

__device__ __forceinline__ KeyRef key_ref_name(const uint8_t *r, const uint8_t *end, uint32_t l_name) {
    KeyRef k;
    k.status = 0;
    k.s = r + 36;
    k.n = l_name ? l_name - 1 : 0;
    k.iv = 0;
    k.is_int = false;
    if (!pack_key(k.s, end, false, (int)k.n, &k.key)) k.status = 1;
    return k;
}

__device__ __forceinline__ void key_ref_write(const KeyRef &k, uint8_t *dst) {
    if (!k.is_int) {
        for (uint32_t i = 0; i < k.n; i++) dst[i] = k.s[i];
        return;
    }
    dst[0] = 1;                                 // "\x01%lld"
    uint32_t at = k.n;
    unsigned long long v = k.iv < 0 ? (unsigned long long)(-k.iv) : (unsigned long long)k.iv;
    do {
        dst[--at] = (uint8_t)('0' + v % 10);
        v /= 10;
    } while (v);
    if (k.iv < 0) dst[--at] = '-';
}

struct RunStart {
    long long rec;      // global record index
    int32_t tid;
    int32_t bam;
};

struct ExtractArgs {
    const BgzfBlockDev *blocks;
    const BlkInfo *info;
    const unsigned long long *rec_base;   // per block: global index of its first kept record
    const unsigned long long *cig_base;
    const unsigned long long *seq_base;
    const int32_t *tid_map;
    int32_t n_blocks, bam_idx;
    unsigned long long hdr_end;
    int want_seq, has_cell, has_umi;
    uint32_t cell_tag, umi_tag;           // two characters, little endian
    int2 *pos_end;
    uint32_t *fmq, *cig_off, *seq_off, *cigar, *seq;
    ulonglong2 *keys;
    RunStart *starts;
    int *n_starts;
    int *n_need_host;                     // values for the host's intern table
    int *n_unspelled;                     // values this decoder cannot hand over (float UMI tags)
    uint2 *hk;                            // per block: such values, bytes of their strings
};

// one pass over the aux fields finds both tags (first occurrence wins, as bam_aux_get)
__device__ __forceinline__ void find_tags(const ExtractArgs &a, const uint8_t *p, const uint8_t *rend,
                                          const uint8_t **t_cell_out, const uint8_t **t_umi_out) {
    const uint8_t *t_cell = nullptr, *t_umi = nullptr;
    int want = (a.has_cell ? 1 : 0) + (a.has_umi ? 1 : 0);
    while (want > 0 && p + 3 <= rend) {
        const uint32_t tag = ld16u(p), typ = p[2];
        if (a.has_cell && !t_cell && tag == a.cell_tag) {
            t_cell = p + 2;
            want--;
        }
        // host order: the cell tag is looked up first, then the UMI tag, each from the start;
        // identical tags resolve to the same field
        if (a.has_umi && !t_umi && tag == a.umi_tag) {
            t_umi = p + 2;
            want--;
        }
        const uint8_t *v = p + 3;
        unsigned long long sz;
        if (typ == 'A' || typ == 'c' || typ == 'C') sz = 1;
        else if (typ == 's' || typ == 'S') sz = 2;
        else if (typ == 'i' || typ == 'I' || typ == 'f') sz = 4;
        else if (typ == 'Z' || typ == 'H') {
            const uint8_t *z = v;
            while (z < rend && *z) z++;
            if (z >= rend) break;
            sz = (unsigned long long)(z - v) + 1;
        } else if (typ == 'B') {
            if (v + 5 > rend) break;
            const uint32_t st = v[0], cnt = ld32u(v + 1);
            const unsigned long long es = (st == 'c' || st == 'C') ? 1 : (st == 's' || st == 'S') ? 2 : 4;
            sz = 5 + es * cnt;
        } else break;
        p = v + sz;
    }
    *t_cell_out = t_cell;
    *t_umi_out = t_umi;
}

// the two keys of a record
__device__ __forceinline__ void record_keys(const ExtractArgs &a, const uint8_t *r, uint32_t bs, const RecGeom &q,
                                            KeyRef *ck, KeyRef *uk) {
    const uint8_t *sq = r + 36 + q.l_name + 4ull * q.n_cig;
    const uint8_t *p = sq + (q.l_seq + 1) / 2 + q.l_seq, *rend = r + 4 + bs;
    const uint8_t *t_cell, *t_umi;
    find_tags(a, p, rend, &t_cell, &t_umi);
    ck->status = uk->status = 0;
    ck->key = uk->key = XG_KEY_NONE;
    if (t_cell) *ck = key_ref_tag(t_cell, rend, true);
    if (a.has_umi) {
        if (t_umi) *uk = key_ref_tag(t_umi, rend, false);
    } else {
        *uk = key_ref_name(r, rend, q.l_name);
    }
}

// One WARP per BGZF block.  The record starts are a chain (each record gives the next one's offset): the warp walks
// 32 links with uniform loads -- one transaction each -- and lane i keeps link i; then every lane takes ITS record:
// geometry, a warp prefix sum places its CIGAR / sequence words and its record slot behind the block's base offsets
// (exactly what k_walk counted), the fixed-size fields of 32 consecutive records leave as coalesced stores, and the
// aux fields of 32 records are parsed side by side instead of one after the other.
#define EXTRACT_THREADS 128
__global__ void __launch_bounds__(EXTRACT_THREADS) k_extract(const ExtractArgs a) {
    const int lane = threadIdx.x & 31;
    const int b = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);
    if (b >= a.n_blocks) return;
    const BlkInfo bi = a.info[b];
    if (bi.n_kept == 0) {
        if (lane == 0) a.hk[b] = make_uint2(0u, 0u);
        return;
    }
    const BgzfBlockDev bk = a.blocks[b];
    uint32_t off = bk.uoff < a.hdr_end ? (uint32_t)(a.hdr_end - bk.uoff) : 0u;      // uniform: the next link
    const uint32_t end = bk.isize;
    unsigned long long g0 = a.rec_base[b], co0 = a.cig_base[b], so0 = a.seq_base[b];
    int32_t prev_tid = -2;                 // contig of the last kept record before this batch
    uint32_t hk_n = 0, hk_bytes = 0;
    int unspelled = 0;
    const uint32_t lt = (1u << lane) - 1u;
    while (off < end) {
        uint32_t my_off = 0xFFFFFFFFu;
        for (int i = 0; i < 32 && off < end; i++) {
            if (lane == i) my_off = off;
            off += 4u + ld32u(bk.uptr + off);          // k_walk has checked every link of the chain
        }
        const bool valid = my_off != 0xFFFFFFFFu;
        const uint8_t *r = bk.uptr + (valid ? my_off : 0u);
        uint32_t bs = 0;
        int32_t tid = -1;
        if (valid) {
            bs = ld32u(r);
            tid = (int32_t)ld32u(r + 4);
        }
        const bool kept = valid && tid >= 0 && a.tid_map[tid] >= 0;
        RecGeom q;
        q.n_words = q.seq_words = 0;
        if (kept) q = rec_geom(r, bs, a.want_seq != 0);
        const uint32_t kmask = __ballot_sync(0xffffffffu, kept);
        // inclusive warp scans of the CIGAR and sequence words
        uint32_t ci = kept ? q.n_words : 0u, si = kept ? q.seq_words : 0u;
        const uint32_t my_c = ci, my_s = si;
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t yc = __shfl_up_sync(0xffffffffu, ci, d), ys = __shfl_up_sync(0xffffffffu, si, d);
            if (lane >= d) {
                ci += yc;
                si += ys;
            }
        }
        const uint32_t tot_c = __shfl_sync(0xffffffffu, ci, 31), tot_s = __shfl_sync(0xffffffffu, si, 31);
        // contig of the kept record before mine (run starts)
        const uint32_t below = kmask & lt;
        const int src = below ? 31 - __clz((int)below) : 0;
        const int32_t tid_before = __shfl_sync(0xffffffffu, tid, src);
        const int32_t my_prev = below ? tid_before : prev_tid;
        if (kmask) prev_tid = __shfl_sync(0xffffffffu, tid, 31 - __clz((int)kmask));
        if (kept) {
            const unsigned long long g = g0 + (unsigned long long)__popc(below);
            unsigned long long co = co0 + (ci - my_c), so = so0 + (si - my_s);
            a.pos_end[g] = make_int2(q.pos, q.end);
            a.fmq[g] = q.fmq;
            const uint8_t *cig = r + 36 + q.l_name;
            const uint32_t ncw = q.fmq >> 24;
            if (ncw == 0) {
                a.cig_off[g] = (uint32_t)co;
            } else if (q.n_cig == 0) {
                a.cig_off[g] = (uint32_t)co;
                a.cigar[co++] = 6;
            } else {
                if (ncw == 255) a.cigar[co++] = q.n_cig;
                a.cig_off[g] = (uint32_t)co;
                for (uint32_t i = 0; i < q.n_cig; i++) a.cigar[co++] = ld32u(cig + 4 * i);
            }
            const uint8_t *sq = cig + 4ull * q.n_cig;
            const uint32_t seq_bytes = (q.l_seq + 1) / 2;
            if (a.want_seq) {
                a.seq_off[g] = q.seq_words ? (uint32_t)so : 0xFFFFFFFFu;
                for (uint32_t w = 0; w < q.seq_words; w++) {
                    uint32_t v = ld32u(sq + 4 * w);
                    const uint32_t left = seq_bytes - 4 * w;
                    if (left < 4) v &= (1u << (8 * left)) - 1u;
                    a.seq[so++] = v;
                }
            }
            KeyRef ck, uk;
            record_keys(a, r, bs, q, &ck, &uk);
            for (const KeyRef *k : {&ck, &uk}) {
                if (k->status == 1) {
                    hk_n++;
                    hk_bytes += k->n;
                } else if (k->status == 2) {
                    unspelled++;
                }
            }
            a.keys[g] = make_ulonglong2(ck.key, uk.key);      // a key still to come from the host holds a placeholder
            if (tid != my_prev) {
                const int s2 = atomicAdd(a.n_starts, 1);
                a.starts[s2] = RunStart{(long long)g, tid, a.bam_idx};
            }
        }
        g0 += (unsigned long long)__popc(kmask);
        co0 += tot_c;
        so0 += tot_s;
    }
    for (int d = 16; d > 0; d >>= 1) {
        hk_n += __shfl_xor_sync(0xffffffffu, hk_n, d);
        hk_bytes += __shfl_xor_sync(0xffffffffu, hk_bytes, d);
        unspelled += __shfl_xor_sync(0xffffffffu, unspelled, d);
    }
    if (lane == 0) {
        a.hk[b] = make_uint2(hk_n, hk_bytes);
        if (hk_n) atomicMax(a.n_need_host, 1);
        if (unspelled) atomicMax(a.n_unspelled, 1);
    }
}

// Values for the host's intern table: which key of which record, and the string.
struct KeyReq {
    long long rec;
    unsigned long long off;  // into the string buffer
    unsigned int len, which; // which: 0 cell, 1 UMI
};

__global__ void k_keys_gather(const ExtractArgs a, const unsigned long long *req_base, const unsigned long long *str_base,
                              KeyReq *reqs, uint8_t *strs) {
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.n_blocks) return;
    if (a.hk[b].x == 0) return;
    const BgzfBlockDev bk = a.blocks[b];
    uint32_t off = bk.uoff < a.hdr_end ? (uint32_t)(a.hdr_end - bk.uoff) : 0u;
    const uint32_t end = bk.isize;
    unsigned long long g = a.rec_base[b], ri = req_base[b], so = str_base[b];
    while (off < end) {
        const uint8_t *r = bk.uptr + off;
        const uint32_t bs = ld32u(r);
        const int32_t tid = (int32_t)ld32u(r + 4);
        off += 4u + bs;
        if (tid < 0 || a.tid_map[tid] < 0) continue;
        const RecGeom q = rec_geom(r, bs, false);
        KeyRef ck, uk;
        record_keys(a, r, bs, q, &ck, &uk);
        if (ck.status == 1) {
            reqs[ri++] = KeyReq{(long long)g, so, ck.n, 0u};
            key_ref_write(ck, strs + so);
            so += ck.n;
        }
        if (uk.status == 1) {
            reqs[ri++] = KeyReq{(long long)g, so, uk.n, 1u};
            key_ref_write(uk, strs + so);
            so += uk.n;
        }
        g++;
    }
}

// Equal strings of a window are interned once: hash every string, then elect a representative
// per distinct string in an open-addressing table of request indices (a slot holds index + 1;
// hashes and bytes are complete before the election starts, so a loser can compare at once).
__global__ void k_keys_hash(const KeyReq *reqs, const uint8_t *strs, long long n, unsigned long long *hash) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const KeyReq q = reqs[i];
    unsigned long long h = 1469598103934665603ull ^ q.len;
    for (unsigned int k = 0; k < q.len; k++) h = (h ^ strs[q.off + k]) * 1099511628211ull;
    hash[i] = mix64(h);
}

__global__ void k_keys_elect(const KeyReq *reqs, const uint8_t *strs, const unsigned long long *hash, long long n,
                             unsigned int *slots, unsigned int cap, unsigned int *rep) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const KeyReq q = reqs[i];
    const unsigned long long h = hash[i];
    unsigned int s = hash_to_range(h, cap);
    while (true) {
        unsigned int cur = slots[s];
        if (cur == 0) cur = atomicCAS(&slots[s], 0u, (unsigned int)i + 1u);
        if (cur == 0) {
            rep[i] = (unsigned int)i;
            return;
        }
        const unsigned int r = cur - 1u;
        if (hash[r] == h) {
            const KeyReq qr = reqs[r];
            bool same = qr.len == q.len;
            for (unsigned int k = 0; same && k < q.len; k++) same = strs[qr.off + k] == strs[q.off + k];
            if (same) {
                rep[i] = r;
                return;
            }
        }
        s = s + 1 == cap ? 0 : s + 1;
    }
}

__global__ void k_keys_patch(const KeyReq *reqs, const unsigned long long *vals, long long n, ulonglong2 *keys) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const KeyReq q = reqs[i];
    if (q.which) keys[q.rec].y = vals[i];
    else keys[q.rec].x = vals[i];
}

__global__ void k_tile_index2(const int2 *pos_end, xg_tile *tiles, int32_t n_tiles) {
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

double now_ms();
bool g_lap_on = false;          // XG_DECODE_TIMING: host-side phase times on stderr
double g_lap_t = 0;
void lap(const char *what) {
    if (!g_lap_on) return;
    const double t = now_ms();
    fprintf(stderr, "[device decode] %-14s %8.2f ms\n", what, t - g_lap_t);
    g_lap_t = t;
}

double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// ---- file -> HBM -> inflated -> records, in windows -----------------------------------------------
// The compressed file is read straight into two pinned staging buffers (several pread threads
// per chunk) and copied to the device chunk by chunk on the copy stream; the file is never held
// in host memory.  The BGZF block index is built from each chunk while it is staged (the
// unscanned tail of a chunk -- a block cut by the chunk boundary, < 64 KiB + header -- is carried
// in front of the next one), and the blocks that are complete are inflated on the compute
// stream as soon as their chunk has landed: disk read, PCIe copy and inflate overlap.
// A window is a run of chunks whose compressed and inflated bytes fit the window buffers (sized
// from the free device memory); at the end of a window its blocks are walked and their records are
// appended to the batch, and the buffers are reused.  Device memory is therefore bounded by the
// window plus the batch itself, whatever the size of the BAM.
constexpr size_t STAGE_HEAD = 128u << 10;
size_t env_bytes(const char *name, size_t dflt) {
    const char *e = getenv(name);
    return e ? (size_t)atoll(e) : dflt;
}
size_t stage_bytes() {          // XG_STAGE_BYTES / XG_DECODE_WINDOW: tests use small values to exercise the carry / windows
    return std::max<size_t>(env_bytes("XG_STAGE_BYTES", 64u << 20), STAGE_HEAD) & ~(size_t)4095;
}

bool pread_all(int fd, uint8_t *dst, size_t len, uint64_t off) {
    while (len) {
        ssize_t got = pread(fd, dst, len, (off_t)off);
        if (got <= 0) return false;
        dst += got;
        off += (uint64_t)got;
        len -= (size_t)got;
    }
    return true;
}

bool pread_parallel(int fd, uint8_t *dst, size_t len, uint64_t off, int n_threads) {
    if (len < (4u << 20) || n_threads <= 1) return pread_all(fd, dst, len, off);
    std::atomic<bool> ok(true);
    std::vector<std::thread> th;
    const size_t slice = ((len + n_threads - 1) / n_threads + 4095) & ~(size_t)4095;
    for (size_t b = 0; b < len; b += slice)
        th.emplace_back([=, &ok] {
            if (!pread_all(fd, dst + b, std::min(slice, len - b), off + b)) ok = false;
        });
    for (auto &t : th) t.join();
    return ok;
}

struct Decoder {
    xg_ctx *ctx = nullptr;
    int want_seq = 0;
    const char *cell_tag = nullptr, *umi_tag = nullptr;
    xg_keyspace *ks = nullptr;                // interns the values that do not pack into 63 bits
    int *cnt = nullptr;                       // device counters: [0] bad blocks, [2] max aln, [3] max span, [4] starts,
                                              // [5] values for the host's intern table, [6] values not spelled here
    uint2 *hk = nullptr;                      // per block of the window: such values, bytes of their strings
    int64_t n_interned = 0, n_distinct = 0;  // values handed to the host / strings it had to intern
    double t_keys = 0;
    // window buffers, shared by all BAMs of the call
    uint8_t *comp = nullptr, *slab = nullptr;
    size_t comp_cap = 0, slab_cap = 0, blk_cap = 0, tid_cap = 0;
    BgzfBlockDev *blocks = nullptr;
    BlkInfo *info = nullptr;
    unsigned long long *bases = nullptr;      // 3 x blk_cap
    int32_t *d_tid_map = nullptr;
    cudaEvent_t ev_win = nullptr;             // the window buffers are free again
    cudaStream_t ist2 = nullptr;              // every other chunk is inflated here: a launch is about one wave of CTAs,
    cudaEvent_t ev_i2 = nullptr;              // two streams let the tail of one overlap the head of the next
    // the batch under construction (capacities in elements)
    int2 *pos_end = nullptr;
    uint32_t *fmq = nullptr, *cig_off = nullptr, *seq_off = nullptr, *cigar = nullptr, *seq = nullptr;
    ulonglong2 *keys = nullptr;
    size_t cap_n = 0, cap_cig = 0, cap_seq = 0;
    int64_t n_total = 0, cig_total = 0, seq_total = 0, n_seen = 0;
    int32_t max_aln = 0, max_span = 0;
    std::vector<RunStart> starts;
    uint64_t comp_all = 0, comp_done = 0;     // compressed bytes of all BAMs / consumed so far (sizes the batch)
    double t_read = 0, t_stream = 0, t_walk = 0, t_extract = 0, t_alloc = 0;
    int n_windows = 0;

    template <class T>
    bool regrow(T *&p, size_t used, size_t want) {      // new buffer of `want` elements holding the first `used`
        T *q = (T *)ctx->dev_get(want * sizeof(T) + 64);
        if (!q) return false;
        if (p && used) cudaMemcpyAsync(q, p, used * sizeof(T), cudaMemcpyDeviceToDevice, ctx->stream);
        if (p) {
            cudaStreamSynchronize(ctx->stream);          // the old buffer goes back to the pool
            ctx->dev_put(p);
        }
        p = q;
        return true;
    }
    // room for the records of the window that is about to be extracted
    bool reserve(int64_t n_need, int64_t cig_need, int64_t seq_need) {
        const double t0 = now_ms();
        const double scale = comp_done ? std::max(1.0, (double)comp_all / (double)comp_done) : 1.0;
        auto target = [&](int64_t need) {
            // exact when everything has been seen, else what the rest of the input would add (+10 %)
            return scale <= 1.0 ? (size_t)need + 1 : (size_t)((double)need * scale * 1.1) + 4096;
        };
        bool ok = true;
        if ((size_t)n_need + 1 > cap_n) {
            const size_t want = target(n_need);
            ok = ok && regrow(pos_end, (size_t)n_total, want) && regrow(fmq, (size_t)n_total, want) &&
                 regrow(cig_off, (size_t)n_total, want + 1) && regrow(keys, (size_t)n_total, want);
            if (want_seq) ok = ok && regrow(seq_off, (size_t)n_total, want);
            if (ok) cap_n = want;
        }
        if (ok && (size_t)cig_need + 1 > cap_cig) {
            const size_t want = target(cig_need);
            ok = regrow(cigar, (size_t)cig_total, want);
            if (ok) cap_cig = want;
        }
        if (ok && want_seq && (size_t)seq_need + 1 > cap_seq) {
            const size_t want = target(seq_need);
            ok = regrow(seq, (size_t)seq_total, want);
            if (ok) cap_seq = want;
        }
        t_alloc += now_ms() - t0;
        return ok;
    }
    void release_window_buffers() {
        ctx->dev_put(comp);
        ctx->dev_put(slab);
        ctx->dev_put(blocks);
        ctx->dev_put(info);
        ctx->dev_put(bases);
        ctx->dev_put(d_tid_map);
        ctx->dev_put(hk);
        comp = slab = nullptr;
        blocks = nullptr;
        info = nullptr;
        bases = nullptr;
        hk = nullptr;
        d_tid_map = nullptr;
        if (ev_win) cudaEventDestroy(ev_win);
        if (ev_i2) cudaEventDestroy(ev_i2);
        ev_win = ev_i2 = nullptr;
    }
    void release_batch() {
        void *ps[] = {pos_end, fmq, cig_off, keys, seq_off, cigar, seq};
        for (void *p : ps) ctx->dev_put(p);
        pos_end = nullptr;
        fmq = cig_off = seq_off = cigar = seq = nullptr;
        keys = nullptr;
    }
};

struct BamState {                       // per BAM, across its windows
    const char *path;
    int32_t bam_idx, n_ref = 0;
    uint64_t hdr_end = 0;
    unsigned long long last_key = 0;
};

// The values of the window that do not pack into 63 bits: their strings are gathered on the
// device, interned by the host's keyspace (several threads; the keyspace is sharded) and the
// keys patched into the batch.  Query-name UMIs (`--UMItag None`) take this path for every read.
int intern_keys(Decoder &D, const ExtractArgs &a, int32_t nb) {
    xg_ctx *ctx = D.ctx;
    cudaStream_t st = ctx->stream;
    const double t0 = now_ms();
    std::vector<uint2> hk((size_t)nb);
    cudaError_t e = cudaMemcpy(hk.data(), D.hk, (size_t)nb * sizeof(uint2), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return ctx->fail(XG_E_CUDA, std::string("device decode: ") + cudaGetErrorString(e));
    std::vector<unsigned long long> base(2 * (size_t)nb);
    unsigned long long n_req = 0, n_bytes = 0;
    for (int32_t b = 0; b < nb; b++) {
        base[(size_t)b] = n_req;
        base[(size_t)nb + b] = n_bytes;
        n_req += hk[(size_t)b].x;
        n_bytes += hk[(size_t)b].y;
    }
    unsigned long long *d_base = (unsigned long long *)ctx->dev_get(2 * (size_t)nb * 8 + 16);
    KeyReq *d_reqs = (KeyReq *)ctx->dev_get((size_t)n_req * sizeof(KeyReq) + 16);
    uint8_t *d_strs = (uint8_t *)ctx->dev_get((size_t)n_bytes + 16);
    unsigned long long *d_vals = (unsigned long long *)ctx->dev_get((size_t)n_req * 8 + 16);
    auto done = [&](int code, const std::string &msg) {
        cudaStreamSynchronize(st);
        ctx->dev_put(d_base);
        ctx->dev_put(d_reqs);
        ctx->dev_put(d_strs);
        ctx->dev_put(d_vals);
        return code ? ctx->fail(code, msg) : XG_OK;
    };
    if (!d_base || !d_reqs || !d_strs || !d_vals) return done(XG_E_UNSUPPORTED, "the key strings do not fit the device");
    cudaMemcpyAsync(d_base, base.data(), 2 * (size_t)nb * 8, cudaMemcpyHostToDevice, st);
    k_keys_gather<<<(unsigned)((nb + 63) / 64), 64, 0, st>>>(a, d_base, d_base + nb, d_reqs, d_strs);
    // one representative per distinct string (requests are indexed with 32 bits here)
    if (n_req >= 0xffffffffull) return done(XG_E_UNSUPPORTED, "too many values for the intern table in one window");
    const unsigned int cap = (unsigned int)std::min<unsigned long long>(2 * n_req + 16, 0xfffffff0ull);
    unsigned long long *d_hash = d_vals;            // the hashes are done with before the values arrive
    unsigned int *d_slots = (unsigned int *)ctx->dev_get((size_t)cap * 4 + 16);
    unsigned int *d_rep = (unsigned int *)ctx->dev_get((size_t)n_req * 4 + 16);
    if (!d_slots || !d_rep) {
        ctx->dev_put(d_slots);
        ctx->dev_put(d_rep);
        return done(XG_E_UNSUPPORTED, "the key strings do not fit the device");
    }
    cudaMemsetAsync(d_slots, 0, (size_t)cap * 4, st);
    k_keys_hash<<<(unsigned)((n_req + 255) / 256), 256, 0, st>>>(d_reqs, d_strs, (long long)n_req, d_hash);
    k_keys_elect<<<(unsigned)((n_req + 255) / 256), 256, 0, st>>>(d_reqs, d_strs, d_hash, (long long)n_req, d_slots, cap,
                                                                d_rep);
    std::vector<KeyReq> reqs((size_t)n_req);
    std::vector<uint8_t> strs((size_t)n_bytes + 1);
    std::vector<unsigned int> rep((size_t)n_req);
    cudaMemcpyAsync(reqs.data(), d_reqs, (size_t)n_req * sizeof(KeyReq), cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(strs.data(), d_strs, (size_t)n_bytes, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(rep.data(), d_rep, (size_t)n_req * 4, cudaMemcpyDeviceToHost, st);
    e = cudaStreamSynchronize(st);
    ctx->dev_put(d_slots);
    ctx->dev_put(d_rep);
    if (e != cudaSuccess) return done(XG_E_CUDA, std::string("device decode: ") + cudaGetErrorString(e));
    std::vector<unsigned long long> vals((size_t)n_req);
    {
        const int n_threads = (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
        const size_t per = ((size_t)n_req + n_threads - 1) / n_threads;
        auto over_slices = [&](auto body) {
            std::vector<std::thread> th;
            for (int t = 0; t < n_threads; t++) {
                const size_t lo = std::min((size_t)n_req, per * t), hi = std::min((size_t)n_req, per * (t + 1));
                if (lo < hi) th.emplace_back([=] { body(lo, hi); });
            }
            for (auto &t : th) t.join();
        };
        std::atomic<long long> n_distinct(0);
        over_slices([&](size_t lo, size_t hi) {           // representatives go through the keyspace ...
            long long nd = 0;
            for (size_t i = lo; i < hi; i++)
                if (rep[i] == (unsigned int)i) {
                    vals[i] = D.ks->encode((const char *)strs.data() + reqs[i].off, (int64_t)reqs[i].len);
                    nd++;
                }
            n_distinct += nd;
        });
        over_slices([&](size_t lo, size_t hi) {           // ... the others take their representative's key
            for (size_t i = lo; i < hi; i++)
                if (rep[i] != (unsigned int)i) vals[i] = vals[rep[i]];
        });
        D.n_distinct += n_distinct;
    }
    cudaMemcpyAsync(d_vals, vals.data(), (size_t)n_req * 8, cudaMemcpyHostToDevice, st);
    if (n_req) k_keys_patch<<<(unsigned)((n_req + 255) / 256), 256, 0, st>>>(d_reqs, d_vals, (long long)n_req, D.keys);
    D.n_interned += (int64_t)n_req;
    int rc = done(XG_OK, "");
    D.t_keys += now_ms() - t0;
    return rc;
}

// Walk the window's blocks, append their records to the batch.
int flush_window(Decoder &D, BamState &B, int32_t nb) {
    xg_ctx *ctx = D.ctx;
    cudaStream_t st = ctx->stream;
    if (nb <= 0) return XG_OK;
    D.n_windows++;
    if (D.ist2) cudaStreamWaitEvent(st, D.ev_i2, 0);        // the chunks inflated on the second stream
    cudaEventRecord(ctx->ev[0], st);
    k_walk<<<(unsigned)((nb + 63) / 64), 64, 0, st>>>(D.blocks, nb, B.hdr_end, D.d_tid_map, B.n_ref, D.want_seq, D.info,
                                                      D.cnt + 2);
    cudaEventRecord(ctx->ev[1], st);
    std::vector<BlkInfo> h_info((size_t)nb);
    int h_cnt[8];
    cudaMemcpyAsync(h_cnt, D.cnt, sizeof(h_cnt), cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(h_info.data(), D.info, (size_t)nb * sizeof(BlkInfo), cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return ctx->fail(XG_E_CUDA, std::string("device inflate: ") + cudaGetErrorString(e));
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
    D.t_walk += ms;
    if (h_cnt[0])
        return ctx->fail(XG_E_FORMAT, std::string("BGZF inflate failed (corrupt block or CRC mismatch) in '") + B.path + "'");
    std::vector<unsigned long long> bases(3 * (size_t)nb);
    int64_t kept = 0, cig = 0, seq = 0, n_all = 0, n_starts = 0;
    for (int32_t b = 0; b < nb; b++) {
        const BlkInfo &bi = h_info[(size_t)b];
        if (bi.status == 2) return ctx->fail(XG_E_FORMAT, std::string("corrupt BAM record in '") + B.path + "'");
        if (bi.status == 3) return ctx->fail(XG_E_FORMAT, std::string("'") + B.path + "' is not coordinate sorted");
        if (bi.status == 1)
            return ctx->fail(XG_E_UNSUPPORTED, std::string("records of '") + B.path + "' cross BGZF block boundaries");
        if (bi.n_all) {
            if (bi.first_key < B.last_key) return ctx->fail(XG_E_FORMAT, std::string("'") + B.path + "' is not coordinate sorted");
            B.last_key = bi.last_key;
        }
        bases[(size_t)b] = (unsigned long long)(D.n_total + kept);
        bases[(size_t)nb + b] = (unsigned long long)(D.cig_total + cig);
        bases[2 * (size_t)nb + b] = (unsigned long long)(D.seq_total + seq);
        n_all += bi.n_all;
        kept += bi.n_kept;
        cig += bi.cig;
        seq += bi.seq;
        n_starts += bi.n_starts;
    }
    D.max_aln = std::max(D.max_aln, h_cnt[2]);
    D.max_span = std::max(D.max_span, h_cnt[3]);
    D.n_seen += n_all;
    if (D.cig_total + cig >= (1LL << 32) || D.seq_total + seq >= (1LL << 32))
        return ctx->fail(XG_E_LIMIT, "batch too large for 32-bit stream offsets; decode fewer reads per batch");
    if (kept > 0) {
        if (!D.reserve(D.n_total + kept, D.cig_total + cig, D.seq_total + seq))
            return ctx->fail(XG_E_UNSUPPORTED, "the read batch does not fit the device");
        RunStart *d_starts = (RunStart *)ctx->dev_get(((size_t)n_starts + 1) * sizeof(RunStart));
        if (!d_starts) return ctx->fail(XG_E_CUDA, "out of device memory");
        cudaMemcpyAsync(D.bases, bases.data(), 3 * (size_t)nb * 8, cudaMemcpyHostToDevice, st);
        cudaMemsetAsync(D.cnt + 4, 0, sizeof(int), st);
        ExtractArgs a;
        a.blocks = D.blocks;
        a.info = D.info;
        a.rec_base = D.bases;
        a.cig_base = D.bases + nb;
        a.seq_base = D.bases + 2 * (size_t)nb;
        a.tid_map = D.d_tid_map;
        a.n_blocks = nb;
        a.bam_idx = B.bam_idx;
        a.hdr_end = B.hdr_end;
        a.want_seq = D.want_seq;
        a.has_cell = D.cell_tag != nullptr;
        a.has_umi = D.umi_tag != nullptr;
        a.cell_tag = D.cell_tag ? ((uint32_t)(uint8_t)D.cell_tag[0] | ((uint32_t)(uint8_t)D.cell_tag[1] << 8)) : 0;
        a.umi_tag = D.umi_tag ? ((uint32_t)(uint8_t)D.umi_tag[0] | ((uint32_t)(uint8_t)D.umi_tag[1] << 8)) : 0;
        a.pos_end = D.pos_end;
        a.fmq = D.fmq;
        a.cig_off = D.cig_off;
        a.seq_off = D.seq_off;
        a.cigar = D.cigar;
        a.seq = D.seq;
        a.keys = D.keys;
        a.starts = d_starts;
        a.n_starts = D.cnt + 4;
        a.n_need_host = D.cnt + 5;
        a.n_unspelled = D.cnt + 6;
        a.hk = D.hk;
        cudaMemsetAsync(D.cnt + 5, 0, 2 * sizeof(int), st);
        cudaEventRecord(ctx->ev[0], st);
        k_extract<<<(unsigned)(((unsigned long long)nb * 32 + EXTRACT_THREADS - 1) / EXTRACT_THREADS), EXTRACT_THREADS, 0, st>>>(a);
        cudaEventRecord(ctx->ev[1], st);
        const size_t s0 = D.starts.size();
        D.starts.resize(s0 + (size_t)n_starts);
        cudaMemcpyAsync(h_cnt, D.cnt, sizeof(h_cnt), cudaMemcpyDeviceToHost, st);
        if (n_starts) cudaMemcpyAsync(D.starts.data() + s0, d_starts, (size_t)n_starts * sizeof(RunStart), cudaMemcpyDeviceToHost, st);
        e = cudaStreamSynchronize(st);
        ctx->dev_put(d_starts);
        if (e != cudaSuccess) return ctx->fail(XG_E_CUDA, std::string("device decode: ") + cudaGetErrorString(e));
        cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
        D.t_extract += ms;
        if (h_cnt[4] != (int)n_starts) return ctx->fail(XG_E_CUDA, "device decode: run starts do not add up");
        if (h_cnt[6])
            return ctx->fail(XG_E_UNSUPPORTED, "float-typed UMI tags are left to the host decoder");
        if (h_cnt[5]) {
            if (!D.ks)
                return ctx->fail(XG_E_UNSUPPORTED, "cell / UMI values need the host intern table (not short "
                                                   "ACGTN-/digit strings) and no keyspace was given");
            int rc = intern_keys(D, a, nb);
            if (rc) return rc;
        }
        D.n_total += kept;
        D.cig_total += cig;
        D.seq_total += seq;
    }
    cudaEventRecord(D.ev_win, st);
    return XG_OK;
}

// Stream one BAM through the window buffers.
// range_lo / range_hi (range_hi > 0): only the BGZF blocks in [range_lo, range_hi) of the file -- both must be block
// starts (or the file's end), and the block at range_lo must begin with a record (htslib's layout; the caller takes
// the offsets from xg_bgzf_block_index / xg_bam_block_probe).  The header is still read from the file's beginning.
int decode_bam(Decoder &D, const char *path, int32_t bam_idx, const int32_t *tid_map, int32_t tid_map_len,
               int64_t range_lo = 0, int64_t range_hi = 0) {
    xg_ctx *ctx = D.ctx;
    const int fd = open(path, O_RDONLY);
    struct stat stt;
    if (fd < 0 || fstat(fd, &stt) != 0) {
        if (fd >= 0) close(fd);
        return ctx->fail(XG_E_IO, std::string("cannot open '") + path + "'");
    }
    const uint64_t fsize = (uint64_t)stt.st_size;
    const bool ranged = range_hi > 0;
    if (ranged && (range_lo < 0 || range_lo > range_hi || (uint64_t)range_hi > fsize)) {
        close(fd);
        return ctx->fail(XG_E_ARG, "xg_decode_bams_device_range: byte range outside the file");
    }
    const uint64_t csize = ranged ? (uint64_t)range_hi : fsize;     // the streaming loop ends here
    const size_t STAGE_BYTES = stage_bytes();
    uint8_t *stage[2] = {(uint8_t *)ctx->pinned_get(STAGE_HEAD + STAGE_BYTES), (uint8_t *)ctx->pinned_get(STAGE_HEAD + STAGE_BYTES)};
    // the chunk's block descriptors travel through pinned memory too: a copy from pageable memory
    // synchronises the stream first, i.e. waits for the chunk's own bytes to arrive
    constexpr size_t DESC_STAGE = 1u << 20;
    BgzfBlockDev *desc_stage[2] = {(BgzfBlockDev *)ctx->pinned_get(DESC_STAGE), (BgzfBlockDev *)ctx->pinned_get(DESC_STAGE)};
    cudaEvent_t done[2] = {nullptr, nullptr};
    auto finish = [&](int code, const std::string &msg) {
        cudaStreamSynchronize(ctx->copy_stream);       // staging buffers may still be in flight
        if (D.ist2) cudaStreamSynchronize(D.ist2);
        cudaStreamSynchronize(ctx->stream);
        for (int k = 0; k < 2; k++) {
            if (desc_stage[k]) ctx->pinned_put(desc_stage[k]);
            if (stage[k]) ctx->pinned_put(stage[k]);
            if (done[k]) cudaEventDestroy(done[k]);
        }
        close(fd);
        return code ? ctx->fail(code, msg) : XG_OK;
    };
    if (!stage[0] || !stage[1] || !desc_stage[0] || !desc_stage[1])
        return finish(XG_E_NOMEM, "out of pinned host memory for the staging buffers");
    cudaEventCreateWithFlags(&done[0], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&done[1], cudaEventDisableTiming);
    if (csize == 0) return finish(XG_E_FORMAT, std::string("'") + path + "' is not BGZF (empty file)");
    const int n_threads = (int)std::max(1u, std::min(8u, std::thread::hardware_concurrency()));
    BamState B;
    B.path = path;
    B.bam_idx = bam_idx;
    uint64_t next_off = 0, uoff = 0;
    const uint8_t *prev_data = nullptr;
    size_t prev_len = 0;
    bool header_done = false;
    xg_dec::Header hdr;
    std::vector<xg_dec::BgzfBlock> hb;            // the blocks completed by the current chunk
    std::vector<BgzfBlockDev> dv;
    // the window being filled
    uint64_t win_base = 0;                         // file offset of comp[0]
    size_t win_infl = 0;
    int32_t win_blocks = 0;
    bool win_open = false;
    const double t_loop = now_ms();
    uint64_t c_begin = 0;
    if (ranged && range_lo > 0) {
        // the header comes from the file's first blocks (host inflate); the stream then starts at range_lo
        const size_t len = (size_t)std::min<uint64_t>(STAGE_BYTES, fsize);
        uint8_t *data = stage[0] + STAGE_HEAD;
        if (!pread_parallel(fd, data, len, 0, n_threads)) return finish(XG_E_IO, std::string("short read on '") + path + "'");
        uint64_t off = 0, uo = 0;
        while (off < len) {
            uint32_t total = 0, hl = 0;
            int rc = xg_dec::bgzf_block_header(data + off, len - off, &total, &hl);
            if (rc != 0 || off + total > len) break;
            xg_dec::BgzfBlock b;
            b.coff = off + hl;
            b.clen = total - hl - 8;
            memcpy(&b.isize, data + off + total - 4, 4);
            memcpy(&b.crc, data + off + total - 8, 4);
            b.uoff = uo;
            uo += b.isize;
            hb.push_back(b);
            off += total;
        }
        size_t nb = 1;
        while (true) {
            if (hb.empty()) return finish(XG_E_FORMAT, std::string("'") + path + "' is not BGZF (bad block header)");
            const size_t take = std::min(nb, hb.size());
            xg_dec::Bytes u;
            int rc = xg_dec::inflate_blocks(data, 0, hb.data(), take, u, 1);
            if (rc) return finish(rc, xg_host_last_error());
            rc = xg_dec::parse_header(u, hdr, path);
            if (rc == XG_OK) break;
            if (rc != XG_E_LIMIT) return finish(rc, xg_host_last_error());
            if (take >= hb.size())
                return finish(XG_E_UNSUPPORTED, std::string("BAM header of '") + path + "' does not end within the first staged chunk");
            nb *= 2;
        }
        hb.clear();
        header_done = true;
        B.hdr_end = hdr.end_off;
        B.n_ref = (int32_t)hdr.names.size();
        if (tid_map_len < B.n_ref) return finish(XG_E_ARG, "tid_map shorter than the BAM's contig list");
        if ((size_t)B.n_ref + 1 > D.tid_cap) {
            ctx->dev_put(D.d_tid_map);
            D.tid_cap = (size_t)B.n_ref + 1;
            D.d_tid_map = (int32_t *)ctx->dev_get(D.tid_cap * 4);
            if (!D.d_tid_map) return finish(XG_E_CUDA, "out of device memory");
        }
        cudaMemcpyAsync(D.d_tid_map, tid_map, (size_t)B.n_ref * 4, cudaMemcpyHostToDevice, ctx->stream);
        cudaStreamSynchronize(ctx->stream);          // stage[0] is about to be reused
        c_begin = next_off = (uint64_t)range_lo;
        uoff = hdr.end_off;                           // every block of the range lies behind the header
    }
    uint64_t k = 0;
    for (uint64_t c0 = c_begin; c0 < csize; c0 += STAGE_BYTES, k++) {
        const int si = (int)(k & 1);
        const size_t len = (size_t)std::min<uint64_t>(STAGE_BYTES, csize - c0);
        if (k >= 2) cudaEventSynchronize(done[si]);
        uint8_t *data = stage[si] + STAGE_HEAD;
        const size_t carry = (size_t)(c0 - next_off);
        if (carry) memcpy(data - carry, prev_data + prev_len - carry, carry);
        const double t0 = now_ms();
        if (!pread_parallel(fd, data, len, c0, n_threads)) return finish(XG_E_IO, std::string("short read on '") + path + "'");
        D.t_read += now_ms() - t0;
        const uint64_t view_beg = next_off, view_end = c0 + len;
        hb.clear();
        size_t chunk_infl = 0;
        while (next_off < view_end) {
            const uint8_t *p = data - (c0 - next_off);      // next_off >= c0 - carry
            uint32_t total = 0, hl = 0;
            int rc = xg_dec::bgzf_block_header(p, view_end - next_off, &total, &hl);
            if (rc == 0 && next_off + total > view_end) rc = 1;
            if (rc == 1) {
                if (view_end == csize) return finish(XG_E_FORMAT, std::string("truncated BGZF block in '") + path + "'");
                break;
            }
            if (rc < 0) return finish(XG_E_FORMAT, std::string("'") + path + "' is not BGZF (bad block header)");
            xg_dec::BgzfBlock b;
            b.coff = next_off + hl;
            b.clen = total - hl - 8;
            memcpy(&b.isize, p + total - 4, 4);
            memcpy(&b.crc, p + total - 8, 4);
            b.uoff = uoff;
            if (b.isize > 65536) return finish(XG_E_FORMAT, "BGZF block larger than 64 KiB");
            uoff += b.isize;
            chunk_infl += b.isize;
            hb.push_back(b);
            next_off += total;
        }
        if (view_end - next_off > STAGE_HEAD) return finish(XG_E_FORMAT, "BGZF block larger than 64 KiB");
        if (!header_done) {
            // the BAM header: inflate leading blocks on the host until it parses
            size_t nb = 1;
            while (true) {
                const size_t take = std::min(nb, hb.size());
                xg_dec::Bytes u;
                int rc = xg_dec::inflate_blocks(data, c0, hb.data(), take, u, 1);
                if (rc) return finish(rc, xg_host_last_error());
                rc = xg_dec::parse_header(u, hdr, path);
                if (rc == XG_OK) break;
                if (rc != XG_E_LIMIT) return finish(rc, xg_host_last_error());
                if (take >= hb.size())
                    return finish(view_end == csize ? XG_E_FORMAT : XG_E_UNSUPPORTED,
                                  std::string("BAM header of '") + path + "' does not end within the first staged chunk");
                nb *= 2;
            }
            header_done = true;
            B.hdr_end = hdr.end_off;
            B.n_ref = (int32_t)hdr.names.size();
            if (tid_map_len < B.n_ref) return finish(XG_E_ARG, "tid_map shorter than the BAM's contig list");
            if ((size_t)B.n_ref + 1 > D.tid_cap) {
                ctx->dev_put(D.d_tid_map);
                D.tid_cap = (size_t)B.n_ref + 1;
                D.d_tid_map = (int32_t *)ctx->dev_get(D.tid_cap * 4);
                if (!D.d_tid_map) return finish(XG_E_CUDA, "out of device memory");
            }
            cudaMemcpyAsync(D.d_tid_map, tid_map, (size_t)B.n_ref * 4, cudaMemcpyHostToDevice, ctx->stream);
        }
        // does the chunk fit the open window?
        if (win_open && ((size_t)(view_end - win_base) > D.comp_cap || win_infl + chunk_infl + 16 > D.slab_cap ||
                         (size_t)win_blocks + hb.size() > D.blk_cap)) {
            int rc = flush_window(D, B, win_blocks);
            if (rc) return finish(rc, ctx->err);
            win_open = false;
        }
        if (!win_open) {
            // an empty window takes any chunk: grow the buffers if this one alone is too large
            if (chunk_infl + 16 > D.slab_cap || hb.size() > D.blk_cap) {
                cudaStreamSynchronize(ctx->stream);
                if (chunk_infl + 16 > D.slab_cap) {
                    ctx->dev_put(D.slab);
                    D.slab_cap = chunk_infl + chunk_infl / 4 + 16;
                    D.slab = (uint8_t *)ctx->dev_get(D.slab_cap);
                }
                if (hb.size() > D.blk_cap) {
                    ctx->dev_put(D.blocks);
                    ctx->dev_put(D.info);
                    ctx->dev_put(D.bases);
                    D.blk_cap = hb.size() + hb.size() / 4;
                    ctx->dev_put(D.hk);
                    D.blocks = (BgzfBlockDev *)ctx->dev_get((D.blk_cap + 1) * sizeof(BgzfBlockDev));
                    D.info = (BlkInfo *)ctx->dev_get((D.blk_cap + 1) * sizeof(BlkInfo));
                    D.bases = (unsigned long long *)ctx->dev_get((3 * D.blk_cap + 1) * 8);
                    D.hk = (uint2 *)ctx->dev_get((D.blk_cap + 1) * sizeof(uint2));
                }
                if (!D.slab || !D.blocks || !D.info || !D.bases || !D.hk)
                    return finish(XG_E_UNSUPPORTED, "the inflate window does not fit the device");
            }
            win_open = true;
            win_base = view_beg;       // a fresh window starts at the carried bytes of the cut block
            win_infl = 0;
            win_blocks = 0;
            cudaStreamWaitEvent(ctx->copy_stream, D.ev_win, 0);     // the previous window has left the buffers
        }
        const uint64_t up_off = win_blocks == 0 && win_infl == 0 && win_base == view_beg ? view_beg : c0;
        cudaMemcpyAsync(D.comp + (up_off - win_base), data - (c0 - up_off), (size_t)(view_end - up_off),
                        cudaMemcpyHostToDevice, ctx->copy_stream);
        dv.resize(hb.size());
        for (size_t i = 0; i < hb.size(); i++) {
            dv[i].coff = hb[i].coff - win_base;
            dv[i].clen = hb[i].clen;
            dv[i].isize = hb[i].isize;
            dv[i].uoff = hb[i].uoff;
            dv[i].uptr = D.slab + win_infl;
            dv[i].crc = hb[i].crc;
            dv[i].pad_ = 0;
            win_infl += hb[i].isize;
        }
        if (!dv.empty()) {
            const BgzfBlockDev *src = dv.data();
            if (dv.size() * sizeof(BgzfBlockDev) <= DESC_STAGE) {
                memcpy(desc_stage[si], dv.data(), dv.size() * sizeof(BgzfBlockDev));
                src = desc_stage[si];
            }
            cudaMemcpyAsync(D.blocks + win_blocks, src, dv.size() * sizeof(BgzfBlockDev), cudaMemcpyHostToDevice,
                            ctx->copy_stream);
        }
        cudaEventRecord(done[si], ctx->copy_stream);
        cudaStream_t ist = (k & 1) && D.ist2 ? D.ist2 : ctx->stream;
        cudaStreamWaitEvent(ist, done[si], 0);
        launch_inflate(ist, D.comp, D.blocks + win_blocks, (int32_t)dv.size(), D.cnt + 0);
        if (ist != ctx->stream) cudaEventRecord(D.ev_i2, ist);
        win_blocks += (int32_t)hb.size();
        D.comp_done += len;
        prev_data = data;
        prev_len = len;
    }
    D.t_stream += now_ms() - t_loop;
    if (win_open) {
        int rc = flush_window(D, B, win_blocks);
        if (rc) return finish(rc, ctx->err);
    }
    return finish(XG_OK, "");
}

}  // namespace

extern "C" {

// Testing / validation entry: inflate a whole BGZF file on the device, return the bytes.
int xg_bgzf_inflate_device(xg_ctx *ctx, const char *path, uint8_t *out, int64_t cap, int64_t *n_out) {
    if (!ctx || !ctx->stream) return ctx ? ctx->fail(XG_E_CUDA, "context has no device") : XG_E_ARG;
    if (!path || !n_out) return ctx->fail(XG_E_ARG, "xg_bgzf_inflate_device: null argument");
    XG_CUDA(cudaSetDevice(ctx->device));
    xg_dec::Bytes f;
    std::vector<xg_dec::BgzfBlock> blocks;
    int rc = xg_dec::read_file(path, f);
    if (!rc) rc = xg_dec::scan_bgzf(f, blocks, path);
    if (rc) return ctx->fail(rc, xg_host_last_error());
    const uint64_t usize = blocks.empty() ? 0 : blocks.back().uoff + blocks.back().isize;
    *n_out = (int64_t)usize;
    if (!out || cap < (int64_t)usize) return XG_OK;      // size query
    uint8_t *comp = nullptr, *ubuf = nullptr;
    BgzfBlockDev *dblk = nullptr;
    XG_GET(cnt, int, "gd_counters", 8);
    if (cudaMalloc(&comp, f.size() + 4096) != cudaSuccess || cudaMalloc(&ubuf, usize + 16) != cudaSuccess ||     // a corrupt last block may be read a batch of symbols past its end
        cudaMalloc(&dblk, (blocks.size() + 1) * sizeof(BgzfBlockDev)) != cudaSuccess) {
        cudaGetLastError();
        cudaFree(comp);
        cudaFree(ubuf);
        cudaFree(dblk);
        return ctx->fail(XG_E_CUDA, "out of device memory");
    }
    cudaStream_t st = ctx->stream;
    cudaMemcpyAsync(comp, f.data(), f.size(), cudaMemcpyHostToDevice, st);
    std::vector<BgzfBlockDev> dv(blocks.size());
    for (size_t i = 0; i < blocks.size(); i++) {
        dv[i].coff = blocks[i].coff;
        dv[i].clen = blocks[i].clen;
        dv[i].isize = blocks[i].isize;
        dv[i].uoff = blocks[i].uoff;
        dv[i].uptr = ubuf + blocks[i].uoff;
        dv[i].crc = blocks[i].crc;
        dv[i].pad_ = 0;
    }
    cudaMemcpyAsync(dblk, dv.data(), dv.size() * sizeof(BgzfBlockDev), cudaMemcpyHostToDevice, st);
    cudaMemsetAsync(cnt, 0, 8 * sizeof(int), st);
    cudaEventRecord(ctx->ev[0], st);
    launch_inflate(st, comp, dblk, (int32_t)blocks.size(), cnt);
    cudaEventRecord(ctx->ev[1], st);
    int bad = 0;
    cudaMemcpyAsync(&bad, cnt, 4, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(out, ubuf, usize, cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaStreamSynchronize(st);
    float ms = 0;
    if (e == cudaSuccess) cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
    ctx->timing[0] = ms;
    cudaFree(comp);
    cudaFree(ubuf);
    cudaFree(dblk);
    if (e != cudaSuccess) return ctx->fail(XG_E_CUDA, std::string("device inflate: ") + cudaGetErrorString(e));
    if (bad) return ctx->fail(XG_E_FORMAT, "BGZF inflate failed (corrupt block or CRC mismatch)");
    return XG_OK;
}

static int decode_bams_device_impl(xg_ctx *ctx, int32_t n_bams, const char *const *paths, const int32_t *const *tid_map,
                                   const int32_t *tid_map_len, const char *cell_tag, const char *umi_tag,
                                   int32_t want_seq, xg_keyspace *ks, xg_dreads **out, int64_t *n_records_seen,
                                   const int64_t *range_lo, const int64_t *range_hi);

// no C++ exception crosses the C boundary (host vectors of the block index, the key strings ...)
int xg_decode_bams_device_range(xg_ctx *ctx, int32_t n_bams, const char *const *paths, const int32_t *const *tid_map,
                                const int32_t *tid_map_len, const char *cell_tag, const char *umi_tag, int32_t want_seq,
                                xg_keyspace *ks, const int64_t *range_lo, const int64_t *range_hi, xg_dreads **out,
                                int64_t *n_records_seen) {
    try {
        return decode_bams_device_impl(ctx, n_bams, paths, tid_map, tid_map_len, cell_tag, umi_tag, want_seq, ks, out,
                                       n_records_seen, range_lo, range_hi);
    } catch (const std::exception &e) {
        if (ctx && ctx->stream) {
            cudaStreamSynchronize(ctx->stream);
            if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
        }
        return ctx ? ctx->fail(XG_E_NOMEM, std::string("device decode: ") + e.what()) : XG_E_NOMEM;
    }
}

int xg_decode_bams_device(xg_ctx *ctx, int32_t n_bams, const char *const *paths, const int32_t *const *tid_map,
                          const int32_t *tid_map_len, const char *cell_tag, const char *umi_tag, int32_t want_seq,
                          xg_keyspace *ks, xg_dreads **out, int64_t *n_records_seen) {
    try {
        return decode_bams_device_impl(ctx, n_bams, paths, tid_map, tid_map_len, cell_tag, umi_tag, want_seq, ks, out,
                                       n_records_seen, nullptr, nullptr);
    } catch (const std::exception &e) {
        if (ctx && ctx->stream) {
            cudaStreamSynchronize(ctx->stream);
            if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
        }
        return ctx ? ctx->fail(XG_E_NOMEM, std::string("device decode: ") + e.what()) : XG_E_NOMEM;
    }
}

static int decode_bams_device_impl(xg_ctx *ctx, int32_t n_bams, const char *const *paths, const int32_t *const *tid_map,
                                   const int32_t *tid_map_len, const char *cell_tag, const char *umi_tag,
                                   int32_t want_seq, xg_keyspace *ks, xg_dreads **out, int64_t *n_records_seen,
                                   const int64_t *range_lo, const int64_t *range_hi) {
    if (!ctx || !ctx->stream) return ctx ? ctx->fail(XG_E_CUDA, "context has no device") : XG_E_ARG;
    if (n_bams < 0 || !out) return ctx->fail(XG_E_ARG, "xg_decode_bams_device: bad argument");
    if (cell_tag && strlen(cell_tag) != 2) return ctx->fail(XG_E_ARG, "cell tag must have 2 characters");
    if (umi_tag && strlen(umi_tag) != 2) return ctx->fail(XG_E_ARG, "UMI tag must have 2 characters");
    XG_CUDA(cudaSetDevice(ctx->device));
    const double t_begin = now_ms();
    for (double &t : ctx->timing) t = 0;
    g_lap_on = getenv("XG_DECODE_TIMING") != nullptr;
    g_lap_t = t_begin;
    if (!ctx->copy_stream) XG_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    Decoder D;
    D.ctx = ctx;
    D.want_seq = want_seq;
    D.cell_tag = cell_tag;
    D.umi_tag = umi_tag;
    D.ks = ks;
    D.cnt = (int *)ctx->get("gd_counters", 8 * sizeof(int));
    if (!D.cnt) return XG_E_CUDA;
    // window buffers: as large as the largest BAM needs, at most XG_DECODE_WINDOW compressed bytes
    uint64_t max_csize = 0;
    for (int32_t b = 0; b < n_bams; b++) {
        struct stat stt;
        if (stat(paths[b], &stt) != 0) return ctx->fail(XG_E_IO, std::string("cannot open '") + paths[b] + "'");
        const uint64_t part = range_hi && range_hi[b] > 0 ? (uint64_t)(range_hi[b] - range_lo[b]) : (uint64_t)stt.st_size;
        D.comp_all += part;
        max_csize = std::max<uint64_t>(max_csize, part);
    }
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    const size_t avail = free_b + ctx->dev_idle_bytes();
    // window: a tenth of the free memory in compressed bytes (the inflated window takes up to 6x that, the
    // batch the rest), so a BAM up to ~17 GB goes through in one window on an empty B200
    const size_t stage = stage_bytes();
    const size_t window = std::max<size_t>(env_bytes("XG_DECODE_WINDOW", std::max<size_t>((size_t)2 << 30, avail / 10)), stage);
    D.comp_cap = std::max<size_t>(std::min<size_t>((size_t)max_csize, window), stage) + STAGE_HEAD + 16;
    D.slab_cap = std::max<size_t>(std::min<size_t>(D.comp_cap * 6, avail / 3), 1u << 20);
    D.blk_cap = D.comp_cap / 1024 + 4096;
    D.comp = (uint8_t *)ctx->dev_get(D.comp_cap);
    D.slab = (uint8_t *)ctx->dev_get(D.slab_cap);
    D.blocks = (BgzfBlockDev *)ctx->dev_get((D.blk_cap + 1) * sizeof(BgzfBlockDev));
    D.info = (BlkInfo *)ctx->dev_get((D.blk_cap + 1) * sizeof(BlkInfo));
    D.bases = (unsigned long long *)ctx->dev_get((3 * D.blk_cap + 1) * 8);
    D.hk = (uint2 *)ctx->dev_get((D.blk_cap + 1) * sizeof(uint2));
    auto bail = [&](int code, const std::string &msg) {
        cudaStreamSynchronize(ctx->copy_stream);
        cudaStreamSynchronize(ctx->stream);
        D.release_window_buffers();
        D.release_batch();
        return ctx->fail(code, msg);
    };
    if (!D.comp || !D.slab || !D.blocks || !D.info || !D.bases || !D.hk)
        return bail(XG_E_UNSUPPORTED, "the inflate window does not fit the device");
    if (cudaEventCreateWithFlags(&D.ev_win, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&D.ev_i2, cudaEventDisableTiming) != cudaSuccess)
        return bail(XG_E_CUDA, "cudaEventCreate");
    if (!ctx->inflate_stream && cudaStreamCreateWithFlags(&ctx->inflate_stream, cudaStreamNonBlocking) != cudaSuccess)
        return bail(XG_E_CUDA, "cudaStreamCreate");
    if (!getenv("XG_INFLATE_ONE_STREAM")) D.ist2 = ctx->inflate_stream;
    cudaStream_t st = ctx->stream;
    cudaMemsetAsync(D.cnt, 0, 8 * sizeof(int), st);
    cudaEventRecord(ctx->ev[2], st);
    cudaEventRecord(D.ev_win, st);
    cudaEventRecord(D.ev_i2, st);
    lap("setup");
    std::vector<int64_t> bam_end((size_t)n_bams, 0);
    for (int32_t b = 0; b < n_bams; b++) {
        int rc = decode_bam(D, paths[b], b, tid_map[b], tid_map_len[b], range_lo ? range_lo[b] : 0,
                            range_hi ? range_hi[b] : 0);
        if (rc) {
            const std::string msg = ctx->err;
            return bail(rc, msg);
        }
        bam_end[(size_t)b] = D.n_total;
    }
    lap("bams");
    D.release_window_buffers();
    const int64_t n_total = D.n_total;
    if (!D.reserve(n_total, D.cig_total, D.seq_total)) return bail(XG_E_UNSUPPORTED, "the read batch does not fit the device");
    xg_dreads *d = new xg_dreads();
    d->pooled = true;
    d->n_reads = n_total;
    d->n_cigar = D.cig_total;
    d->n_seq_words = D.seq_total;
    d->max_aln_len = D.max_aln;
    d->max_span = D.max_span;
    d->pos_end = D.pos_end;
    d->fmq = D.fmq;
    d->cig_off = D.cig_off;
    d->keys = D.keys;
    d->cigar = D.cigar;
    d->seq_off = D.seq_off;
    d->seq = D.seq;
    auto fail_free = [&](int code, const std::string &msg) {
        cudaStreamSynchronize(ctx->stream);
        xg_dreads_free(ctx, d);
        return ctx->fail(code, msg);
    };
    const uint32_t sentinel = (uint32_t)D.cig_total;
    cudaMemcpyAsync(d->cig_off + n_total, &sentinel, 4, cudaMemcpyHostToDevice, st);
    std::vector<RunStart> &starts = D.starts;
    std::sort(starts.begin(), starts.end(), [](const RunStart &x, const RunStart &y) { return x.rec < y.rec; });
    // runs: maximal stretches of kept records of one contig of one BAM (decode.cpp's run_tid)
    size_t si = 0;
    for (int32_t b = 0; b < n_bams; b++) {
        int32_t run_tid = -2;
        for (; si < starts.size() && starts[si].rec < bam_end[(size_t)b]; si++) {
            if (starts[si].tid == run_tid) continue;
            run_tid = starts[si].tid;
            if (!d->h_runs.empty() && d->h_runs.back().rec_end < 0) d->h_runs.back().rec_end = starts[si].rec;
            xg_run r;
            r.bam_idx = b;
            r.gid = tid_map[b][run_tid];
            r.rec_beg = starts[si].rec;
            r.rec_end = -1;
            d->h_runs.push_back(r);
        }
        if (!d->h_runs.empty() && d->h_runs.back().rec_end < 0) d->h_runs.back().rec_end = bam_end[(size_t)b];
    }
    for (size_t r = 0; r < d->h_runs.size(); r++)
        for (int64_t s = d->h_runs[r].rec_beg; s < d->h_runs[r].rec_end; s += XG_TILE) {
            xg_tile tl;
            tl.rec_beg = s;
            tl.n_rec = (int32_t)std::min<int64_t>(XG_TILE, d->h_runs[r].rec_end - s);
            tl.run = (int32_t)r;
            tl.first_pos = 0;
            tl.max_end = 0;
            d->h_tiles.push_back(tl);
        }
    d->n_runs = (int32_t)d->h_runs.size();
    d->n_tiles = (int32_t)d->h_tiles.size();
    d->runs = (xg_run *)ctx->dev_get((size_t)d->n_runs * sizeof(xg_run) + 16);
    d->tiles = (xg_tile *)ctx->dev_get((size_t)d->n_tiles * sizeof(xg_tile) + 16);
    if (!d->runs || !d->tiles) return fail_free(XG_E_CUDA, "out of device memory for the tile index");
    cudaMemcpyAsync(d->runs, d->h_runs.data(), (size_t)d->n_runs * sizeof(xg_run), cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(d->tiles, d->h_tiles.data(), (size_t)d->n_tiles * sizeof(xg_tile), cudaMemcpyHostToDevice, st);
    if (d->n_tiles) {
        k_tile_index2<<<(d->n_tiles + 7) / 8, 256, 0, st>>>(d->pos_end, d->tiles, d->n_tiles);
        cudaMemcpyAsync(d->h_tiles.data(), d->tiles, (size_t)d->n_tiles * sizeof(xg_tile), cudaMemcpyDeviceToHost, st);
    }
    cudaEventRecord(ctx->ev[3], st);
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail_free(XG_E_CUDA, std::string("device decode: ") + cudaGetErrorString(e));
    lap("runs+tiles");
    int rc = xg_make_tile_pmax(ctx, d);
    if (rc) {
        xg_dreads_free(ctx, d);
        return rc;
    }
    lap("pmax");
    const size_t n = (size_t)n_total;
    d->bytes = (int64_t)(n * 32 + (size_t)D.cig_total * 4 + (size_t)D.seq_total * 4 + (want_seq ? n * 4 : 0));
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[3]);
    ctx->timing[0] = ms;                    // device span of the call
    ctx->timing[2] = D.t_walk;              // walk kernels
    ctx->timing[3] = D.t_extract;           // extract kernels
    ctx->timing[4] = D.t_stream;            // file read + H2D + inflate (pipelined) incl. the windows' walk / extract
    ctx->timing[5] = D.n_windows;
    ctx->timing[8] = D.t_read;              // time inside pread
    ctx->timing[9] = D.t_alloc;             // growing the batch
    ctx->timing[6] = (double)D.n_interned;  // values interned by the host's keyspace
    ctx->timing[7] = D.t_keys;              // ... and the time that took
    ctx->timing[11] = (double)D.n_distinct; // ... distinct strings per window among them
    {
        const double t_f0 = now_ms();
        ctx->dev_trim(8ull << 30);          // keep small inputs' buffers for the next call, give the rest back
        ctx->timing[10] = now_ms() - t_f0;
    }
    ctx->timing[12] = now_ms() - t_begin;   // whole call
    if (n_records_seen) *n_records_seen = D.n_seen;
    *out = d;
    return XG_OK;
}

}  // extern "C"
