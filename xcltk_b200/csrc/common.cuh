// common.cuh -- shared device helpers and the context object (sm_100a only).
#pragma once
#include <cstring>
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <initializer_list>
#include <map>
#include <string>
#include <vector>

#include "../../include/xcltk_b200.h"

#define XG_CUDA(call)                                                                  \
    do {                                                                               \
        cudaError_t e_ = (call);                                                       \
        if (e_ != cudaSuccess) {                                                       \
            return ctx->fail(XG_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
        }                                                                              \
    } while (0)

// Device-resident read batch: same arrays as xg_reads (include/xcltk_b200.h).
struct xg_dreads {
    int64_t n_reads = 0, n_cigar = 0, n_seq_words = 0;
    int32_t n_runs = 0, n_tiles = 0, max_aln_len = 0, max_span = 0;
    int2 *pos_end = nullptr;
    uint32_t *fmq = nullptr;
    uint32_t *cig_off = nullptr;
    ulonglong2 *keys = nullptr;
    uint32_t *seq_off = nullptr;
    uint32_t *cigar = nullptr;
    uint32_t *seq = nullptr;
    xg_run *runs = nullptr;      // device
    xg_tile *tiles = nullptr;    // device
    int32_t *tile_pmax = nullptr;   // device: per run, prefix max of tile.max_end (window planning)
    std::vector<xg_run> h_runs;  // host copies for the planners
    std::vector<xg_tile> h_tiles;
    std::vector<int3> h_run_tiles;  // maximal stretches of tiles of one run: {run, first tile, end tile}
    double h2d_ms = 0;
    int64_t bytes = 0;
    bool pooled = false;         // buffers came from xg_ctx::dev_get
    bool mapped = false;         // xg_map_reads: only pos_end / runs / tiles are device copies
    int8_t umi_compact = -1;     // 0: a UMI key of the batch does not fit a pair word (learnt by xg_basefc)
};

// Hash of an input array (are these the features / SNPs / regions of the last call?): four independent
// multiply-xorshift lanes over 32-byte blocks -- the dependent chain of a single lane is what bounds a
// word-wise FNV (1.6 MB of SNP arrays: 0.2 ms -> 0.06 ms per call).
static inline void xg_mix_bytes(uint64_t &h, const void *p, size_t n) {
    const uint8_t *q = (const uint8_t *)p;
    uint64_t a = h ^ 0x9E3779B97F4A7C15ull, b = h ^ 0xBF58476D1CE4E5B9ull, c = h ^ 0x94D049BB133111EBull, d = h ^ 0xD6E8FEB86659FD93ull;
    size_t k = 0;
    for (; k + 32 <= n; k += 32) {
        uint64_t w[4];
        memcpy(w, q + k, 32);
        a = (a ^ w[0]) * 1099511628211ull;
        b = (b ^ w[1]) * 1099511628211ull;
        c = (c ^ w[2]) * 1099511628211ull;
        d = (d ^ w[3]) * 1099511628211ull;
        a ^= a >> 29;
        b ^= b >> 31;
        c ^= c >> 27;
        d ^= d >> 30;
    }
    h = (a * 3 + (b ^ (b << 7))) ^ (c * 5 + (d ^ (d >> 11)));
    for (; k < n; k++) h = (h ^ q[k]) * 1099511628211ull;
    h = (h ^ (uint64_t)n) * 1099511628211ull;
    h ^= h >> 32;
}

// The input a device-side cache was built from (the features, SNPs, regions or barcodes of the last call).  The hash
// is the quick test; inputs with equal hashes are easy to build (every step of xg_mix_bytes can be inverted), so a hit
// also compares the bytes, of which the key keeps a copy.
struct xg_input_key {
    struct Span {
        const void *p;
        size_t n;
    };
    uint64_t hash = 0;
    std::vector<uint8_t> bytes;
    static uint64_t hash_of(std::initializer_list<Span> in) {
        uint64_t h = 1469598103934665603ull;
        for (const Span &s : in) xg_mix_bytes(h, s.p, s.n);
        return h;
    }
    bool matches(uint64_t h, std::initializer_list<Span> in) const {
        if (h != hash) return false;
        size_t at = 0;
        for (const Span &s : in) {
            if (s.n > bytes.size() - at || (s.n && memcmp(bytes.data() + at, s.p, s.n) != 0)) return false;
            at += s.n;
        }
        return at == bytes.size();
    }
    void assign(uint64_t h, std::initializer_list<Span> in) {
        hash = h;
        bytes.clear();
        for (const Span &s : in)
            if (s.n) bytes.insert(bytes.end(), (const uint8_t *)s.p, (const uint8_t *)s.p + s.n);
    }
};

struct xg_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;    // xg_basefc_host: H2D of the next epoch
    cudaStream_t d2h_stream = nullptr;     // basefc rows layouts: result rows copied out while later epochs run
    int64_t fx_nnz_hint = 0;
    int64_t discover_slice = 0;            // xg_snp_discover: candidates per pileup slice (0: the default)               // nnz of the last basefc call (sizes the pinned result up front)
    // the rows of the last basefc call with a rows layout are still in the staging area (scratch "fx_st_col" /
    // "fx_st_val", places in "fx_seg_base" / "fx_seg_nnz") until the next call: xg_basefc_write_mtx_device formats them
    bool fx_res_valid = false;
    int64_t fx_res_nnz = 0;
    int32_t fx_res_rows = 0, fx_res_cols = 0;
    cudaStream_t big_stream = nullptr;     // basefc: big-segment finalize beside the ordinary one
    cudaStream_t inflate_stream = nullptr; // device decoder: second inflate stream
    cudaEvent_t ev[8] = {};
    std::vector<cudaEvent_t> ev_pool;     // per-epoch timing events
    std::string err;
    double timing[16] = {};
    // growable named scratch buffers (avoid cudaMalloc/cudaFree on every call)
    struct Buf {
        void *p = nullptr;
        size_t cap = 0;
    };
    std::map<std::string, Buf> scratch;

    // pinned host buffers of results are recycled (cudaHostAlloc of GBs costs ~100 ms/GB)
    struct Pinned {
        void *p;
        size_t cap;
        bool used;
    };
    std::vector<Pinned> pinned;
    void *pinned_get(size_t bytes) {
        size_t best = pinned.size();
        for (size_t k = 0; k < pinned.size(); k++)
            if (!pinned[k].used && pinned[k].cap >= bytes && (best == pinned.size() || pinned[k].cap < pinned[best].cap))
                best = k;
        if (best < pinned.size()) {
            pinned[best].used = true;
            return pinned[best].p;
        }
        void *p = nullptr;
        size_t want = bytes + bytes / 8 + 4096;
        if (cudaHostAlloc(&p, want, cudaHostAllocDefault) != cudaSuccess) {
            cudaGetLastError();
            for (auto it = pinned.begin(); it != pinned.end();)      // drop idle buffers and retry
                if (!it->used) {
                    cudaFreeHost(it->p);
                    it = pinned.erase(it);
                } else {
                    ++it;
                }
            want = bytes ? bytes : 4096;
            if (cudaHostAlloc(&p, want, cudaHostAllocDefault) != cudaSuccess) {
                cudaGetLastError();
                return nullptr;
            }
        }
        pinned.push_back(Pinned{p, want, true});
        return p;
    }
    void pinned_put(void *p) {
        for (auto &b : pinned)
            if (b.p == p) {
                b.used = false;
                return;
            }
        cudaFreeHost(p);
    }

    // device buffers with caller-visible lifetime (uploaded read batches, baf state) are
    // recycled the same way: cudaMalloc / cudaFree of GBs per call is slow and synchronises
    std::vector<Pinned> devbufs;
    void *dev_get(size_t bytes) {
        size_t best = devbufs.size();
        for (size_t k = 0; k < devbufs.size(); k++)
            if (!devbufs[k].used && devbufs[k].cap >= bytes && devbufs[k].cap <= bytes + bytes / 2 + (1 << 20) &&
                (best == devbufs.size() || devbufs[k].cap < devbufs[best].cap))
                best = k;
        if (best < devbufs.size()) {
            devbufs[best].used = true;
            return devbufs[best].p;
        }
        void *p = nullptr;
        size_t want = bytes ? bytes : 256;
        if (cudaMalloc(&p, want) != cudaSuccess) {
            cudaGetLastError();
            for (auto it = devbufs.begin(); it != devbufs.end();)     // drop idle buffers and retry
                if (!it->used) {
                    cudaFree(it->p);
                    it = devbufs.erase(it);
                } else {
                    ++it;
                }
            if (cudaMalloc(&p, want) != cudaSuccess) {
                cudaGetLastError();
                return nullptr;
            }
        }
        devbufs.push_back(Pinned{p, want, true});
        return p;
    }
    size_t dev_idle_bytes() const {
        size_t n = 0;
        for (auto &b : devbufs)
            if (!b.used) n += b.cap;
        return n;
    }
    // free idle buffers (largest first) until at most `keep` bytes stay pooled
    void dev_trim(size_t keep) {
        while (dev_idle_bytes() > keep) {
            size_t big = devbufs.size();
            for (size_t k = 0; k < devbufs.size(); k++)
                if (!devbufs[k].used && (big == devbufs.size() || devbufs[k].cap > devbufs[big].cap)) big = k;
            if (big == devbufs.size()) break;
            cudaFree(devbufs[big].p);
            devbufs.erase(devbufs.begin() + (long)big);
        }
    }
    void dev_put(void *p) {
        if (!p) return;
        for (auto &b : devbufs)
            if (b.p == p) {
                b.used = false;
                return;
            }
        cudaFree(p);
    }
    // cache of the last sorted SNP table of xg_baf_pileup (device arrays in scratch "bf_*")
    bool bf_snp_valid = false;
    xg_input_key bf_snp_key;
    int64_t bf_snp_sorted = 0;
    bool bf_sr_valid = false;              // ... and of the inverted region -> SNP lists of xg_baf_count
    xg_input_key bf_sr_key;
    // the two most recent barcode tables (basefc and baf alternate with different cell lists): scratch "bc_slots0/1"
    struct BcCache {
        bool valid = false;
        xg_input_key key;
        uint64_t used = 0;
        const void *slots = nullptr;
        uint32_t mask = 0, shift = 0;
    } bc_cache[2];
    uint64_t bc_clock = 0;
    // cache of the last interval index built by xg_basefc (owned by basefc.cu)
    void *fx_cache = nullptr;
    void (*fx_cache_free)(void *) = nullptr;

    int fail(int code, const std::string &msg) {
        err = msg;
        return code;
    }
    // Returns nullptr on failure (err set).
    void *get(const char *name, size_t bytes) {
        Buf &b = scratch[name];
        if (b.cap >= bytes && b.p) return b.p;
        if (b.p) cudaFree(b.p);
        b.p = nullptr;
        b.cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&b.p, want);
        if (e != cudaSuccess) {
            cudaGetLastError();
            dev_trim(0);                     // idle pooled buffers give way to scratch
            e = cudaMalloc(&b.p, bytes ? bytes : 256);
            want = bytes ? bytes : 256;
        }
        if (e != cudaSuccess) {
            err = std::string("cudaMalloc(") + name + ", " + std::to_string(bytes) + " B): " +
                  cudaGetErrorString(e);
            b.p = nullptr;
            return nullptr;
        }
        b.cap = want;
        return b.p;
    }
};

#define XG_GET(ptr, type, name, count)                                      \
    type *ptr = (type *)ctx->get(name, sizeof(type) * (size_t)(count));     \
    if (!ptr) return XG_E_CUDA;

// ---- device helpers -----------------------------------------------------------------
struct __align__(16) xg_e128 {
    unsigned long long a, b;
};

__device__ __forceinline__ xg_e128 ld128_relaxed(const xg_e128 *addr) {
    xg_e128 v;
    asm volatile(
        "{\n\t.reg .b128 t;\n\tld.relaxed.gpu.global.b128 t, [%2];\n\tmov.b128 {%0, %1}, t;\n\t}"
        : "=l"(v.a), "=l"(v.b)
        : "l"(addr)
        : "memory");
    return v;
}

__device__ __forceinline__ xg_e128 cas128(xg_e128 *addr, xg_e128 cmp, xg_e128 val) {
    xg_e128 old;
    asm volatile(
        "{\n\t.reg .b128 c, v, o;\n\t"
        "mov.b128 c, {%2, %3};\n\t"
        "mov.b128 v, {%4, %5};\n\t"
        "atom.relaxed.gpu.global.cas.b128 o, [%6], c, v;\n\t"
        "mov.b128 {%0, %1}, o;\n\t}"
        : "=l"(old.a), "=l"(old.b)
        : "l"(cmp.a), "l"(cmp.b), "l"(val.a), "l"(val.b), "l"(addr)
        : "memory");
    return old;
}

__host__ __device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 33;
    x *= 0xff51afd7ed558ccdULL;
    x ^= x >> 33;
    x *= 0xc4ceb9fe1a85ec53ULL;
    x ^= x >> 33;
    return x;
}

// slot in [0, cap) from a 64-bit hash without a division
__host__ __device__ __forceinline__ uint32_t hash_to_range(uint64_t h, uint32_t cap) {
    return (uint32_t)(((h >> 32) * (uint64_t)cap) >> 32);
}

__device__ __forceinline__ bool cig_aligned(uint32_t op) { return (0x181u >> op) & 1u; }       // M, =, X
__device__ __forceinline__ bool cig_skips_ref(uint32_t op) { return op == 2 || op == 3; }

// Cell-barcode lookup table (open addressing, linear probing; empty = XG_KEY_NONE).
// One 16-byte entry {key, column} per slot: a probe is a single 128-bit load.
struct BarcodeTable {
    const ulonglong2 *slots;
    uint32_t mask;
    uint32_t shift;      // 32 - log2(slots)
};
// home slot: the two halves of the key folded, one 32-bit multiply, top bits (a 64-bit mix costs
// four times the instructions and the packed barcode strings spread their entropy over both halves)
__host__ __device__ __forceinline__ uint32_t barcode_home(uint64_t key, uint32_t shift) {
    return (((uint32_t)key ^ (uint32_t)(key >> 32)) * 0x9E3779B1u) >> shift;
}
__device__ __forceinline__ int32_t barcode_lookup(const BarcodeTable &t, uint64_t key) {
    uint32_t s = barcode_home(key, t.shift);
    while (true) {
        const ulonglong2 e = __ldg(&t.slots[s]);
        if (e.x == key) return (int32_t)e.y;
        if (e.x == XG_KEY_NONE) return -1;
        s = (s + 1) & t.mask;
    }
}

// check_read(): xcltk/rdr/fc/core.py:46-62 (mapq, flags, orphan, tag presence); the
// min_len test needs the aligned length and is done by the caller.
struct FilterParams {
    int32_t min_mapq, min_len;
    uint32_t incl_flag, excl_flag;
    int32_t no_orphan, use_cell_tag, need_umi_tag;
};
__device__ __forceinline__ bool read_passes_flags(const FilterParams &f, uint32_t fmq) {
    uint32_t flag = fmq & 0xffffu, mapq = (fmq >> 16) & 0xffu;
    if ((int32_t)mapq < f.min_mapq) return false;
    if (f.excl_flag && (flag & f.excl_flag)) return false;
    if (f.incl_flag && !(flag & f.incl_flag)) return false;
    if (f.no_orphan && (flag & 1u) && !(flag & 2u)) return false;
    return true;
}

int xg_build_barcode_table(xg_ctx *ctx, const xg_barcodes *cells, BarcodeTable *out);
int xg_make_tile_pmax(xg_ctx *ctx, xg_dreads *d);
// A pooled batch with the counts and the host run / tile index of `h`, and no device arrays yet.
xg_dreads *xg_dreads_new(const xg_reads *h);
