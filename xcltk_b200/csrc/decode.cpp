// decode.cpp -- host side: BGZF inflate + BAM record parse -> flat structure-of-arrays.
//
// Replaces what the reference gets from pysam/htslib on its two counting paths
// (pysam.AlignmentFile / AlignedSegment; call sites in SURVEY.md section 8c):
//   pos, bam_endpos (fetch overlap rule), flag, mapq, CIGAR words, 4-bit sequence, the
//   cell / UMI tag strings (or the query name when no UMI tag is used).
// Semantics restated from the SAM/BAM specification (SAMv1 section 4.2) and SURVEY.md A.3.
// Inflate and field extraction are multi-threaded; nothing here touches the GPU except the
// (optional) pinned allocator installed by the CUDA translation unit.
#include <sys/stat.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "bamfile.hpp"
#include "keys.hpp"
#include "owner.hpp"

namespace {
thread_local std::string g_err;
}

namespace xg_dec {
int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
}  // namespace xg_dec

namespace {
using namespace xg_dec;

void *default_alloc(size_t n) {
    void *p = nullptr;
    if (posix_memalign(&p, 256, n ? n : 256) != 0) return nullptr;
    return p;
}
void default_free(void *p) { free(p); }
void *(*g_alloc)(size_t) = default_alloc;
void (*g_free)(void *) = default_free;

inline uint32_t rd32(const uint8_t *p) {
    uint32_t v;
    memcpy(&v, p, 4);
    return v;
}
inline uint16_t rd16(const uint8_t *p) {
    uint16_t v;
    memcpy(&v, p, 2);
    return v;
}

template <class F>
void parallel_for(int64_t n, int n_threads, F f) {
    // f(thread_index, begin, end) over a static partition of [0, n)
    if (n_threads < 1) n_threads = 1;
    if (n < 4096) n_threads = 1;
    std::vector<std::thread> th;
    for (int t = 0; t < n_threads; t++) {
        int64_t b = n * t / n_threads, e = n * (t + 1) / n_threads;
        if (t == n_threads - 1) {
            f(t, b, e);
        } else {
            th.emplace_back([=] { f(t, b, e); });
        }
    }
    for (auto &x : th) x.join();
}

}  // namespace

namespace xg_dec {

int read_file(const char *path, Bytes &buf, int64_t max_bytes) {
    FILE *fp = fopen(path, "rb");
    if (!fp) return fail(XG_E_IO, std::string("cannot open '") + path + "'");
    fseek(fp, 0, SEEK_END);
    long n = ftell(fp);
    fseek(fp, 0, SEEK_SET);
    if (max_bytes >= 0 && n > max_bytes) n = (long)max_bytes;
    buf.resize((size_t)n);
    size_t got = n ? fread(buf.data(), 1, (size_t)n, fp) : 0;
    fclose(fp);
    if ((long)got != n) return fail(XG_E_IO, std::string("short read on '") + path + "'");
    return XG_OK;
}

// One BGZF block header at p (RFC 1952 member with a 'BC' extra subfield, SAMv1 4.1).
// Returns 0 and the block's total / header sizes, 1 when fewer than the needed bytes are
// available (the caller supplies more), or a negative XG_E_* code.
int bgzf_block_header(const uint8_t *p, uint64_t avail, uint32_t *total, uint32_t *hdr_len) {
    if (avail < 18) return 1;
    if (p[0] != 31 || p[1] != 139 || p[2] != 8 || !(p[3] & 4)) return XG_E_FORMAT;
    const uint32_t xlen = rd16(p + 10);
    if (avail < 12ull + xlen) return 1;
    int64_t bsize = -1;
    uint64_t x = 12, xend = 12ull + xlen;
    while (x + 4 <= xend) {
        const uint32_t slen = rd16(p + x + 2);
        if (p[x] == 66 && p[x + 1] == 67 && slen == 2 && x + 6 <= xend) bsize = rd16(p + x + 4);
        x += 4 + slen;
    }
    if (bsize < 0) return XG_E_FORMAT;
    *total = (uint32_t)bsize + 1;
    *hdr_len = 12 + xlen;
    if (*total < *hdr_len + 8) return XG_E_FORMAT;
    return 0;
}

// Walk the BGZF blocks of a buffer.  allow_partial_tail: the buffer is a prefix of the file;
// stop quietly at the first block that is cut off.
int scan_bgzf(const Bytes &f, std::vector<BgzfBlock> &blocks, const char *path, bool allow_partial_tail) {
    uint64_t off = 0, uoff = 0, n = f.size();
    while (off < n) {
        uint32_t total = 0, hdr = 0;
        int rc = bgzf_block_header(&f[off], n - off, &total, &hdr);
        if (rc == 0 && off + total > n) rc = 1;
        if (rc == 1) {
            if (allow_partial_tail) break;
            return fail(XG_E_FORMAT, std::string("truncated BGZF block in '") + path + "'");
        }
        if (rc < 0) return fail(XG_E_FORMAT, std::string("'") + path + "' is not BGZF (bad block header)");
        BgzfBlock b;
        b.coff = off + hdr;
        b.clen = total - hdr - 8;
        b.isize = rd32(&f[off + total - 4]);
        b.crc = rd32(&f[off + total - 8]);
        b.uoff = uoff;
        if (b.isize > 65536) return fail(XG_E_FORMAT, "BGZF block larger than 64 KiB");
        uoff += b.isize;
        blocks.push_back(b);
        off += total;
    }
    return XG_OK;
}

// f_base: file offset of f[0] (block descriptors hold file offsets)
int inflate_blocks(const uint8_t *f, uint64_t f_base, const BgzfBlock *blocks, size_t n_blocks, Bytes &out,
                   int n_threads) {
    uint64_t base = n_blocks ? blocks[0].uoff : 0;
    uint64_t total = n_blocks ? blocks[n_blocks - 1].uoff + blocks[n_blocks - 1].isize - base : 0;
    out.resize(total);
    std::atomic<int> bad(0);
    parallel_for((int64_t)n_blocks, n_threads, [&](int, int64_t b, int64_t e) {
        z_stream zs;
        memset(&zs, 0, sizeof(zs));
        if (inflateInit2(&zs, -15) != Z_OK) {
            bad = 1;
            return;
        }
        for (int64_t i = b; i < e; i++) {
            const BgzfBlock &bk = blocks[i];
            if (bk.isize == 0) continue;
            inflateReset(&zs);
            zs.next_in = const_cast<Bytef *>(f + (bk.coff - f_base));
            zs.avail_in = bk.clen;
            zs.next_out = &out[bk.uoff - base];
            zs.avail_out = bk.isize;
            int rc = inflate(&zs, Z_FINISH);
            if (rc != Z_STREAM_END || zs.avail_out != 0 ||
                (uint32_t)crc32(crc32(0L, Z_NULL, 0), &out[bk.uoff - base], bk.isize) != bk.crc) {     // as htslib checks
                bad = 1;
                break;
            }
        }
        inflateEnd(&zs);
    });
    if (bad) return fail(XG_E_FORMAT, "BGZF inflate failed (corrupt block or CRC mismatch)");
    return XG_OK;
}

// XG_E_LIMIT: the buffer ends inside the header (the caller inflates more blocks and retries)
int parse_header(const Bytes &u, Header &h, const char *path) {
    uint64_t n = u.size();
    if (n >= 4 && memcmp(u.data(), "BAM\1", 4) != 0)
        return fail(XG_E_IO, std::string("'") + path + "' is not a BAM file (bad magic)");
    if (n < 12) return fail(XG_E_LIMIT, "truncated BAM header");
    uint64_t off = 8 + (uint64_t)(int32_t)rd32(&u[4]);
    if (off + 4 > n) return fail(XG_E_LIMIT, "truncated BAM header");
    int32_t n_ref = (int32_t)rd32(&u[off]);
    off += 4;
    h.names.clear();
    h.lens.clear();
    for (int32_t i = 0; i < n_ref; i++) {
        if (off + 4 > n) return fail(XG_E_LIMIT, "truncated BAM header");
        uint32_t l = rd32(&u[off]);
        off += 4;
        if (l == 0) return fail(XG_E_FORMAT, "corrupt BAM header (empty contig name)");
        if (off + l + 4 > n) return fail(XG_E_LIMIT, "truncated BAM header");
        h.names.emplace_back((const char *)&u[off], l - 1);
        off += l;
        h.lens.push_back((int64_t)(int32_t)rd32(&u[off]));
        off += 4;
    }
    h.end_off = off;
    return XG_OK;
}

// Read (a prefix of) the file, index its blocks and parse the header, inflating only as many
// leading blocks as the header spans.  header_only reads a growing prefix instead of the file.
int open_bam(const char *path, BamFile &bf, bool header_only) {
    int64_t prefix = header_only ? (1 << 20) : -1;
    while (true) {
        bf.blocks.clear();
        int rc = read_file(path, bf.f, prefix);
        if (rc) return rc;
        bool partial = prefix >= 0 && (int64_t)bf.f.size() >= prefix;
        rc = scan_bgzf(bf.f, bf.blocks, path, partial);
        if (rc) return rc;
        size_t nb = 1;
        while (true) {
            size_t take = std::min(nb, bf.blocks.size());
            Bytes u;
            rc = inflate_blocks(bf.f.data(), 0, bf.blocks.data(), take, u, 1);
            if (rc) return rc;
            rc = parse_header(u, bf.h, path);
            if (rc != XG_E_LIMIT) return rc;
            if (take >= bf.blocks.size()) break;
            nb *= 2;
        }
        if (!partial) return fail(XG_E_FORMAT, std::string("truncated BAM header in '") + path + "'");
        prefix *= 8;          // header longer than the prefix: read more of the file
    }
}

}  // namespace xg_dec

namespace {

struct Bam {
    Bytes u;
    Header h;
    std::vector<uint64_t> rec;      // offset of block_size of each kept record
    struct Run {
        int32_t gid;
        int64_t beg, end;           // into rec
    };
    std::vector<Run> runs;
    int64_t n_seen = 0;
};

inline bool op_aligned(uint32_t op) { return op == 0 || op == 7 || op == 8; }
inline bool op_ref(uint32_t op) { return op == 0 || op == 2 || op == 3 || op == 7 || op == 8; }

struct RecInfo {
    int32_t pos, end;
    uint32_t fmq;
    uint32_t n_words;      // cigar words stored (incl. overflow count word)
    uint32_t seq_words;
    int32_t aln_len;
};

inline RecInfo rec_info(const uint8_t *r, bool want_seq) {
    RecInfo o;
    int32_t pos = (int32_t)rd32(r + 8);
    uint32_t l_name = r[12], mapq = r[13];
    uint32_t n_cig = rd16(r + 16), flag = rd16(r + 18), l_seq = rd32(r + 20);
    const uint8_t *cig = r + 36 + l_name;
    int64_t rlen = 0, aln = 0;
    for (uint32_t i = 0; i < n_cig; i++) {
        uint32_t w = rd32(cig + 4 * i), op = w & 15, l = w >> 4;
        if (op_ref(op)) rlen += l;
        if (op_aligned(op)) aln += l;
    }
    if (flag & 4) rlen = 0;          // htslib bam_endpos(): FUNMAP => rlen 0 => 1
    if (rlen == 0) rlen = 1;
    o.pos = pos;
    o.end = (int32_t)(pos + rlen);
    o.aln_len = (int32_t)aln;
    bool simple = n_cig == 1 && op_aligned(rd32(cig) & 15) && aln == rlen && !(flag & 4);
    uint32_t ncw;
    if (simple) {
        ncw = 0;
        o.n_words = 0;
    } else if (n_cig == 0) {
        ncw = 1;
        o.n_words = 1;
    } else if (n_cig < 255) {
        ncw = n_cig;
        o.n_words = n_cig;
    } else {
        ncw = 255;
        o.n_words = n_cig + 1;
    }
    o.fmq = flag | (mapq << 16) | (ncw << 24);
    o.seq_words = want_seq ? (((l_seq + 1) / 2 + 3) / 4) : 0;
    return o;
}

// Locate an aux tag; returns pointer to its type byte or nullptr. First match wins (bam_aux_get).
const uint8_t *find_tag(const uint8_t *aux, const uint8_t *end, const char *tag) {
    const uint8_t *p = aux;
    while (p + 3 <= end) {
        bool hit = p[0] == (uint8_t)tag[0] && p[1] == (uint8_t)tag[1];
        uint8_t t = p[2];
        const uint8_t *v = p + 3;
        size_t sz;
        switch (t) {
            case 'A': case 'c': case 'C': sz = 1; break;
            case 's': case 'S': sz = 2; break;
            case 'i': case 'I': case 'f': sz = 4; break;
            case 'Z': case 'H': {
                const uint8_t *q = (const uint8_t *)memchr(v, 0, (size_t)(end - v));
                if (!q) return nullptr;
                sz = (size_t)(q - v) + 1;
                break;
            }
            case 'B': {
                if (v + 5 > end) return nullptr;
                uint8_t st = v[0];
                uint32_t cnt = rd32(v + 1);
                size_t es = (st == 'c' || st == 'C') ? 1 : (st == 's' || st == 'S') ? 2 : 4;
                sz = 5 + es * cnt;
                break;
            }
            default: return nullptr;
        }
        if (sz > (size_t)(end - v)) return nullptr;      // truncated value: the tag does not exist
        if (hit) return p + 2;
        p = v + sz;
    }
    return nullptr;
}

// Key of a tag value as Python would see it through pysam get_tag():
// Z/H/A -> str; integer / float types are not strings: they never equal a barcode
// (cell) and are interned under a type-tagged spelling (UMI; falsy 0 -> EMPTY).
uint64_t tag_key(const uint8_t *t, const uint8_t *end, xg_keyspace *ks, bool is_cell) {
    uint8_t typ = t[0];
    const uint8_t *v = t + 1;
    if (typ == 'Z' || typ == 'H') {
        const uint8_t *q = (const uint8_t *)memchr(v, 0, (size_t)(end - v));
        int64_t n = q ? (int64_t)(q - v) : (int64_t)(end - v);
        return ks->encode((const char *)v, n);
    }
    if (typ == 'A') return ks->encode((const char *)v, 1);
    if (is_cell) return XG_KEY_NOMATCH;
    char buf[48];
    long long iv = 0;
    switch (typ) {
        case 'c': iv = (int8_t)v[0]; break;
        case 'C': iv = v[0]; break;
        case 's': iv = (int16_t)rd16(v); break;
        case 'S': iv = rd16(v); break;
        case 'i': iv = (int32_t)rd32(v); break;
        case 'I': iv = rd32(v); break;
        case 'f': {
            float fv;
            memcpy(&fv, v, 4);
            if (fv == 0.0f) return XG_KEY_EMPTY;
            int n = snprintf(buf, sizeof buf, "\x02%a", (double)fv);
            return ks->intern(buf, n);
        }
        default: return XG_KEY_NOMATCH;
    }
    if (iv == 0) return XG_KEY_EMPTY;
    int n = snprintf(buf, sizeof buf, "\x01%lld", iv);
    return ks->intern(buf, n);
}

}  // namespace

struct xg_bam_header {
    Header h;
};

extern "C" {

void xg_set_host_alloc(void *(*a)(size_t), void (*f)(void *)) {
    g_alloc = a ? a : default_alloc;
    g_free = f ? f : default_free;
}

const char *xg_host_last_error(void) { return g_err.c_str(); }

xg_keyspace *xg_keyspace_create(void) { return new (std::nothrow) xg_keyspace(); }
void xg_keyspace_destroy(xg_keyspace *ks) { delete ks; }
uint64_t xg_key_encode(xg_keyspace *ks, const char *s, int64_t len) { return ks->encode(s, len); }
int64_t xg_key_decode(xg_keyspace *ks, uint64_t key, char *buf, int64_t cap) {
    return ks->decode(key, buf, cap);
}
int64_t xg_keyspace_n_interned(xg_keyspace *ks) { return ks->n_interned(); }

int xg_bam_header_read(const char *path, xg_bam_header **out) {
    BamFile bf;
    int rc = open_bam(path, bf, true);
    if (rc) return rc;
    xg_bam_header *bh = new xg_bam_header();
    bh->h = std::move(bf.h);
    *out = bh;
    return XG_OK;
}
int32_t xg_bam_header_n_ref(const xg_bam_header *h) { return (int32_t)h->h.names.size(); }
const char *xg_bam_header_ref_name(const xg_bam_header *h, int32_t tid) {
    return (tid >= 0 && tid < (int32_t)h->h.names.size()) ? h->h.names[tid].c_str() : nullptr;
}
int64_t xg_bam_header_ref_len(const xg_bam_header *h, int32_t tid) {
    return (tid >= 0 && tid < (int32_t)h->h.lens.size()) ? h->h.lens[tid] : -1;
}
void xg_bam_header_free(xg_bam_header *h) { delete h; }

void xg_reads_free(xg_reads *r) {
    if (!r) return;
    xg_reads_owner *o = reinterpret_cast<xg_reads_owner *>(r);
    for (void *p : o->bufs) (o->free_fn ? o->free_fn : default_free)(p);
    delete o;
}

static int decode_bams_impl(int32_t n_bams, const char *const *paths, const int32_t *const *tid_map,
                            const int32_t *tid_map_len, const char *cell_tag, const char *umi_tag,
                            int32_t want_seq, int32_t n_threads, xg_keyspace *ks, xg_reads **out);

// no C++ exception crosses the C boundary
int xg_decode_bams(int32_t n_bams, const char *const *paths, const int32_t *const *tid_map,
                   const int32_t *tid_map_len, const char *cell_tag, const char *umi_tag,
                   int32_t want_seq, int32_t n_threads, xg_keyspace *ks, xg_reads **out) {
    try {
        return decode_bams_impl(n_bams, paths, tid_map, tid_map_len, cell_tag, umi_tag, want_seq, n_threads, ks, out);
    } catch (const std::bad_alloc &) {
        return fail(XG_E_NOMEM, "out of host memory while decoding");
    } catch (const std::exception &e) {
        return fail(XG_E_IO, std::string("decode failed: ") + e.what());
    }
}

static int decode_bams_impl(int32_t n_bams, const char *const *paths, const int32_t *const *tid_map,
                            const int32_t *tid_map_len, const char *cell_tag, const char *umi_tag,
                            int32_t want_seq, int32_t n_threads, xg_keyspace *ks, xg_reads **out) {
    if (n_bams < 0 || !out || !ks) return fail(XG_E_ARG, "xg_decode_bams: bad argument");
    if (cell_tag && strlen(cell_tag) != 2) return fail(XG_E_ARG, "cell tag must have 2 characters");
    if (umi_tag && strlen(umi_tag) != 2) return fail(XG_E_ARG, "UMI tag must have 2 characters");
    if (n_threads <= 0) n_threads = (int)std::thread::hardware_concurrency();
    if (n_threads <= 0) n_threads = 1;

    const bool timing = getenv("XG_DECODE_TIMING") != nullptr;
    auto tnow = [] { return std::chrono::steady_clock::now(); };
    auto tprev = tnow();
    auto lap = [&](const char *what) {
        if (!timing) return;
        auto t = tnow();
        fprintf(stderr, "[decode] %-10s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(t - tprev).count());
        tprev = t;
    };
    std::vector<Bam> bams((size_t)n_bams);
    int64_t n_total = 0, n_seen = 0;
    for (int32_t b = 0; b < n_bams; b++) {
        Bam &bm = bams[b];
        {
            Bytes f;
            int rc = read_file(paths[b], f);
            if (rc) return rc;
            lap("read");
            std::vector<BgzfBlock> blocks;
            rc = scan_bgzf(f, blocks, paths[b]);
            if (rc) return rc;
            lap("scan");
            rc = inflate_blocks(f.data(), 0, blocks.data(), blocks.size(), bm.u, n_threads);
            if (rc) return rc;
            lap("inflate");
        }
        int rc = parse_header(bm.u, bm.h, paths[b]);
        if (rc) return rc == XG_E_LIMIT ? XG_E_FORMAT : rc;
        int32_t n_ref = (int32_t)bm.h.names.size();
        if (tid_map_len[b] < n_ref) return fail(XG_E_ARG, "tid_map shorter than the BAM's contig list");
        const int32_t *map = tid_map[b];
        // sequential walk over record boundaries; sortedness check (the reference needs a
        // coordinate-sorted, indexed BAM for fetch()).
        uint64_t off = bm.h.end_off, n = bm.u.size();
        int32_t last_tid = -2, last_pos = -1, run_tid = -2;
        bool seen_unplaced = false;
        while (off + 4 <= n) {
            uint32_t bs = rd32(&bm.u[off]);
            if (bs < 32 || off + 4 + bs > n)
                return fail(XG_E_FORMAT, std::string("corrupt BAM record in '") + paths[b] + "'");
            int32_t tid = (int32_t)rd32(&bm.u[off + 4]);
            int32_t pos = (int32_t)rd32(&bm.u[off + 8]);
            bm.n_seen++;
            if (tid >= n_ref) return fail(XG_E_FORMAT, "record refers to an unknown contig");
            if (tid < 0) {
                seen_unplaced = true;
            } else {
                if (seen_unplaced || tid < last_tid || (tid == last_tid && pos < last_pos))
                    return fail(XG_E_FORMAT,
                                std::string("'") + paths[b] + "' is not coordinate sorted");
                if (map[tid] >= 0) {
                    // geometry of a kept record (same test as the device decoder's rec_geom): name, CIGAR,
                    // sequence and qualities must lie inside the record, or the passes below would read
                    // past it; and pos + reference length must stay an int32
                    const uint8_t *r = &bm.u[off + 4];
                    const uint64_t l_name = r[8], n_cig = rd16(r + 12), l_seq = rd32(r + 16);
                    const uint64_t need = 32 + l_name + 4 * n_cig + (l_seq + 1) / 2 + l_seq;
                    if (need > bs || l_seq >= 0x40000000u)
                        return fail(XG_E_FORMAT, std::string("corrupt BAM record in '") + paths[b] + "'");
                    int64_t rlen = 0;
                    for (uint64_t k = 0; k < n_cig; k++) {
                        const uint32_t cw = rd32(r + 32 + l_name + 4 * k);
                        if (op_ref(cw & 15)) rlen += cw >> 4;
                    }
                    if ((int64_t)pos + std::max<int64_t>(rlen, 1) > INT32_MAX)
                        return fail(XG_E_FORMAT, std::string("record ends beyond 2^31 in '") + paths[b] + "'");
                    if (tid != run_tid) {
                        bm.runs.push_back({map[tid], (int64_t)bm.rec.size(), (int64_t)bm.rec.size()});
                        run_tid = tid;
                    }
                    bm.rec.push_back(off);
                    bm.runs.back().end = (int64_t)bm.rec.size();
                }
                last_tid = tid;
                last_pos = pos;
            }
            off += 4 + bs;
        }
        if (off != n) return fail(XG_E_FORMAT, std::string("trailing bytes in '") + paths[b] + "'");
        lap("walk");
        n_total += (int64_t)bm.rec.size();
        n_seen += bm.n_seen;
    }

    // pass A: sizes of the streams (per thread partial sums over a global record numbering)
    struct Part {
        int64_t cig = 0, seq = 0;
        int32_t max_aln = 0, max_span = 0;
    };
    std::vector<int64_t> bam_base((size_t)n_bams + 1, 0);
    for (int32_t b = 0; b < n_bams; b++) bam_base[b + 1] = bam_base[b] + (int64_t)bams[b].rec.size();
    std::vector<std::vector<Part>> parts((size_t)n_bams);
    int64_t cig_total = 0, seq_total = 0;
    int32_t max_aln = 0, max_span = 0;
    std::vector<std::vector<int64_t>> cig_base((size_t)n_bams), seq_base((size_t)n_bams);
    for (int32_t b = 0; b < n_bams; b++) {
        Bam &bm = bams[b];
        parts[b].assign((size_t)n_threads, Part());
        parallel_for((int64_t)bm.rec.size(), n_threads, [&](int t, int64_t lo, int64_t hi) {
            Part p;
            for (int64_t i = lo; i < hi; i++) {
                RecInfo ri = rec_info(&bm.u[bm.rec[i]], want_seq != 0);
                p.cig += ri.n_words;
                p.seq += ri.seq_words;
                p.max_aln = std::max(p.max_aln, ri.aln_len);
                p.max_span = std::max(p.max_span, ri.end - ri.pos);
            }
            parts[b][t] = p;
        });
        cig_base[b].assign((size_t)n_threads, 0);
        seq_base[b].assign((size_t)n_threads, 0);
        for (int t = 0; t < n_threads; t++) {
            cig_base[b][t] = cig_total;
            seq_base[b][t] = seq_total;
            cig_total += parts[b][t].cig;
            seq_total += parts[b][t].seq;
            max_aln = std::max(max_aln, parts[b][t].max_aln);
            max_span = std::max(max_span, parts[b][t].max_span);
        }
    }
    lap("passA");
    if (cig_total >= (1LL << 32) || seq_total >= (1LL << 32))
        return fail(XG_E_LIMIT, "batch too large for 32-bit stream offsets; decode fewer reads per batch");

    xg_reads_owner *own = new xg_reads_owner();
    memset(&own->r, 0, sizeof(own->r));
    own->free_fn = g_free;
    auto alloc = [&](size_t bytes) -> void * {
        void *p = g_alloc(bytes);
        if (p) own->bufs.push_back(p);
        return p;
    };
    int32_t n_runs = 0;
    for (auto &bm : bams) n_runs += (int32_t)bm.runs.size();
    int64_t n_tiles = 0;
    for (auto &bm : bams)
        for (auto &r : bm.runs) n_tiles += (r.end - r.beg + XG_TILE - 1) / XG_TILE;
    int32_t *pos_end = (int32_t *)alloc(sizeof(int32_t) * 2 * (size_t)n_total);
    uint32_t *fmq = (uint32_t *)alloc(sizeof(uint32_t) * (size_t)n_total);
    uint32_t *cig_off = (uint32_t *)alloc(sizeof(uint32_t) * ((size_t)n_total + 1));
    uint64_t *keys = (uint64_t *)alloc(sizeof(uint64_t) * 2 * (size_t)n_total);
    uint32_t *seq_off = want_seq ? (uint32_t *)alloc(sizeof(uint32_t) * (size_t)n_total) : nullptr;
    uint32_t *cigar = (uint32_t *)alloc(sizeof(uint32_t) * (size_t)cig_total);
    uint32_t *seq = want_seq ? (uint32_t *)alloc(sizeof(uint32_t) * (size_t)seq_total) : nullptr;
    xg_run *runs = (xg_run *)alloc(sizeof(xg_run) * (size_t)n_runs);
    xg_tile *tiles = (xg_tile *)alloc(sizeof(xg_tile) * (size_t)n_tiles);
    if (!pos_end || !fmq || !cig_off || !keys || !cigar || !runs || !tiles ||
        (want_seq && (!seq_off || !seq))) {
        xg_reads_free(&own->r);
        return fail(XG_E_NOMEM, "out of host memory");
    }

    lap("alloc");
    // pass B: fill
    for (int32_t b = 0; b < n_bams; b++) {
        Bam &bm = bams[b];
        int64_t base = bam_base[b];
        parallel_for((int64_t)bm.rec.size(), n_threads, [&](int t, int64_t lo, int64_t hi) {
            int64_t co = cig_base[b][t], so = seq_base[b][t];
            for (int64_t i = lo; i < hi; i++) {
                const uint8_t *r = &bm.u[bm.rec[i]];
                RecInfo ri = rec_info(r, want_seq != 0);
                int64_t g = base + i;
                pos_end[2 * g] = ri.pos;
                pos_end[2 * g + 1] = ri.end;
                fmq[g] = ri.fmq;
                uint32_t l_name = r[12], n_cig = rd16(r + 16), l_seq = rd32(r + 20);
                uint32_t bs = rd32(r);
                const uint8_t *cig = r + 36 + l_name;
                uint32_t ncw = ri.fmq >> 24;
                if (ncw == 0) {
                    cig_off[g] = (uint32_t)co;
                } else if (n_cig == 0) {
                    cig_off[g] = (uint32_t)co;
                    cigar[co++] = 6;    // 0-length P op: consumes nothing
                } else {
                    if (ncw == 255) cigar[co++] = n_cig;
                    cig_off[g] = (uint32_t)co;
                    memcpy(&cigar[co], cig, 4 * (size_t)n_cig);
                    co += n_cig;
                }
                const uint8_t *sq = cig + 4 * (size_t)n_cig;
                if (want_seq) {
                    // a record without sequence (l_seq == 0: query_sequence is None) is marked
                    seq_off[g] = ri.seq_words ? (uint32_t)so : 0xFFFFFFFFu;
                    if (ri.seq_words) {
                        seq[so + ri.seq_words - 1] = 0;
                        memcpy(&seq[so], sq, (l_seq + 1) / 2);
                        so += ri.seq_words;
                    }
                }
                const uint8_t *aux = sq + (l_seq + 1) / 2 + l_seq;
                const uint8_t *end = r + 4 + bs;
                uint64_t ck = XG_KEY_NONE, uk = XG_KEY_NONE;
                if (cell_tag) {
                    const uint8_t *t = find_tag(aux, end, cell_tag);
                    if (t) ck = tag_key(t, end, ks, true);
                }
                if (umi_tag) {
                    const uint8_t *t = find_tag(aux, end, umi_tag);
                    if (t) uk = tag_key(t, end, ks, false);
                } else {
                    uk = ks->encode((const char *)(r + 36), l_name ? (int64_t)l_name - 1 : 0);
                }
                keys[2 * g] = ck;
                keys[2 * g + 1] = uk;
            }
        });
    }

    cig_off[n_total] = (uint32_t)cig_total;    // sentinel: end of the last read's words
    lap("passB");

    // runs + tile index
    int32_t ri = 0;
    int64_t ti = 0;
    for (int32_t b = 0; b < n_bams; b++) {
        for (auto &r : bams[b].runs) {
            runs[ri].bam_idx = b;
            runs[ri].gid = r.gid;
            runs[ri].rec_beg = bam_base[b] + r.beg;
            runs[ri].rec_end = bam_base[b] + r.end;
            for (int64_t s = runs[ri].rec_beg; s < runs[ri].rec_end; s += XG_TILE) {
                int64_t e = std::min<int64_t>(s + XG_TILE, runs[ri].rec_end);
                xg_tile &tl = tiles[ti++];
                tl.rec_beg = s;
                tl.n_rec = (int32_t)(e - s);
                tl.run = ri;
                tl.first_pos = pos_end[2 * s];
                tl.max_end = 0;
            }
            ri++;
        }
    }
    parallel_for(n_tiles, n_threads, [&](int, int64_t lo, int64_t hi) {
        for (int64_t t = lo; t < hi; t++) {
            int32_t m = INT32_MIN;
            for (int64_t i = tiles[t].rec_beg; i < tiles[t].rec_beg + tiles[t].n_rec; i++)
                m = std::max(m, pos_end[2 * i + 1]);
            tiles[t].max_end = m;
        }
    });

    lap("tiles");
    xg_reads &o = own->r;
    o.n_reads = n_total;
    o.n_cigar = cig_total;
    o.n_seq_words = seq_total;
    o.n_runs = n_runs;
    o.n_tiles = (int32_t)n_tiles;
    o.max_aln_len = max_aln;
    o.max_span = max_span;
    o.n_records_seen = n_seen;
    o.pos_end = pos_end;
    o.fmq = fmq;
    o.cig_off = cig_off;
    o.keys = keys;
    o.seq_off = seq_off;
    o.cigar = cigar;
    o.seq = seq;
    o.runs = runs;
    o.tiles = tiles;
    *out = &own->r;
    return XG_OK;
}

}  // extern "C"

// ---- Matrix-Market writer ---------------------------------------------------------------
// Text exactly as merge_mtx produces it (xcltk/rdr/fc/utils.py:54-94 == baf/fc/utils.py:204-245):
//   "%%MatrixMarket matrix coordinate integer general\n%%\n<nrow>\t<ncol>\t<nnz>\n" then one
//   "<row>\t<col>\t<val>\n" per non-zero, 1-based, rows renumbered over the EMITTED features.
// Input is the CSR result of the counting call over all input rows; out_row[r] is the 1-based
// output row of input row r (0 = row not emitted; such a row must be empty).  Rows are
// formatted by a pool of threads in slabs and written in order.
namespace {
inline char *put_int(char *p, uint32_t v) {
    char tmp[12];
    int n = 0;
    do {
        tmp[n++] = (char)('0' + v % 10);
        v /= 10;
    } while (v);
    while (n) *p++ = tmp[--n];
    return p;
}
}  // namespace

namespace {
// entry(k, &col, &val): column (0-based) and count of entry k
template <class Entry>
int write_rows_impl(const char *path, int32_t n_rows_in, const int64_t *row_beg, const int32_t *row_cnt,
                    const int32_t *out_row, int32_t n_rows_out, int32_t n_cols, Entry entry, int32_t n_threads) {
    if (!path || !row_beg || !row_cnt || !out_row || n_rows_in < 0)
        return fail(XG_E_ARG, "xg_write_mtx: bad argument");
    if (n_threads <= 0) n_threads = (int)std::thread::hardware_concurrency();
    if (n_threads <= 0) n_threads = 1;
    int64_t nnz = 0;
    for (int32_t r = 0; r < n_rows_in; r++) {
        int64_t c = row_cnt[r];
        if (c && out_row[r] <= 0) return fail(XG_E_ARG, "xg_write_mtx: non-empty row without an output row");
        nnz += c;
    }
    FILE *fp = fopen(path, "wb");
    if (!fp) return fail(XG_E_IO, std::string("cannot write '") + path + "'");
    fprintf(fp, "%%%%MatrixMarket matrix coordinate integer general\n%%%%\n%d\t%d\t%lld\n", n_rows_out, n_cols,
            (long long)nnz);
    // slabs of consecutive rows holding about `slab` non-zeros each: a few per thread, so that
    // small matrices still use every thread and large ones keep the buffers modest
    const int64_t slab = std::max<int64_t>(1 << 15, std::min<int64_t>(1 << 21, nnz / (4 * (int64_t)n_threads) + 1));
    std::vector<int32_t> cut{0};
    {
        int64_t acc = 0;
        for (int32_t r = 0; r < n_rows_in; r++) {
            acc += row_cnt[r];
            if (acc >= slab) {
                cut.push_back(r + 1);
                acc = 0;
            }
        }
        if (cut.back() != n_rows_in) cut.push_back(n_rows_in);
    }
    const size_t n_slabs = cut.size() - 1;
    std::atomic<bool> ok(true);
    struct Text {
        std::unique_ptr<char[]> p;      // not value-initialised: 36 bytes per entry are reserved
        size_t n = 0;
    };
    std::thread writer;                 // writes group g while group g + 1 is being formatted
    for (size_t s0 = 0; s0 < n_slabs && ok; s0 += (size_t)n_threads) {
        const size_t s1 = std::min(n_slabs, s0 + (size_t)n_threads);
        auto bufs = std::make_shared<std::vector<Text>>(s1 - s0);
        std::vector<std::thread> th;
        for (size_t s = s0; s < s1; s++)
            th.emplace_back([&, s] {
                const int32_t r0 = cut[s], r1 = cut[s + 1];
                Text &b = (*bufs)[s - s0];
                int64_t n_ent = 0;
                for (int32_t r = r0; r < r1; r++) n_ent += row_cnt[r];
                b.p.reset(new (std::nothrow) char[(size_t)n_ent * 36 + 16]);      // no exception may leave a worker thread
                if (!b.p) {
                    ok = false;
                    return;
                }
                char *p = b.p.get();
                Entry ent = entry;              // the thread's own copy: an entry reader may carry state along a row
                for (int32_t r = r0; r < r1; r++)
                    for (int64_t k = row_beg[r]; k < row_beg[r] + row_cnt[r]; k++) {
                        uint32_t c = 0, v = 0;
                        ent(k, k == row_beg[r], &c, &v);
                        p = put_int(p, (uint32_t)out_row[r]);
                        *p++ = '\t';
                        p = put_int(p, c + 1u);
                        *p++ = '\t';
                        p = put_int(p, v);
                        *p++ = '\n';
                    }
                b.n = (size_t)(p - b.p.get());
            });
        for (auto &t : th) t.join();
        if (writer.joinable()) writer.join();
        writer = std::thread([fp, bufs, &ok] {
            for (auto &b : *bufs)
                if (b.n && fwrite(b.p.get(), 1, b.n, fp) != b.n) ok = false;
        });
    }
    if (writer.joinable()) writer.join();
    if (fclose(fp) != 0) ok = false;
    if (!ok) return fail(XG_E_IO, std::string("short write on '") + path + "'");
    return XG_OK;
}
}  // namespace

extern "C" int xg_write_mtx_rows(const char *path, int32_t n_rows_in, const int64_t *row_beg, const int32_t *row_cnt,
                                 const int32_t *out_row, int32_t n_rows_out, int32_t n_cols, const int32_t *col,
                                 const int32_t *val, int32_t n_threads) {
    if (!col || !val) return fail(XG_E_ARG, "xg_write_mtx: bad argument");
    try {
        return write_rows_impl(path, n_rows_in, row_beg, row_cnt, out_row, n_rows_out, n_cols,
                               [=](int64_t k, bool, uint32_t *c, uint32_t *v) {
                                   *c = (uint32_t)col[k];
                                   *v = (uint32_t)val[k];
                               },
                               n_threads);
    } catch (const std::exception &e) {
        return fail(XG_E_NOMEM, std::string("xg_write_mtx: ") + e.what());
    }
}

extern "C" int xg_write_mtx_rows16(const char *path, int32_t n_rows_in, const int64_t *row_beg, const int32_t *row_cnt,
                                   const int32_t *out_row, int32_t n_rows_out, int32_t n_cols, const uint32_t *colval16,
                                   int64_t n_over, const int64_t *over_idx, const int32_t *over_val,
                                   int32_t n_threads) {
    if (!colval16 || n_over < 0 || (n_over && (!over_idx || !over_val))) return fail(XG_E_ARG, "xg_write_mtx: bad argument");
    try {
    std::unordered_map<int64_t, uint32_t> over;
    for (int64_t i = 0; i < n_over; i++) over[over_idx[i]] = (uint32_t)over_val[i];
    const std::unordered_map<int64_t, uint32_t> *ov = &over;
    return write_rows_impl(path, n_rows_in, row_beg, row_cnt, out_row, n_rows_out, n_cols,
                           [=](int64_t k, bool, uint32_t *c, uint32_t *v) {
                               const uint32_t w = colval16[k];
                               *c = w & 0xffffu;
                               *v = w >> 16;
                               if (*v == 0xffffu) {
                                   auto it = ov->find(k);
                                   if (it != ov->end()) *v = it->second;      // (an entry missing from the list keeps 65535)
                               }
                           },
                           n_threads);
    } catch (const std::exception &e) {
        return fail(XG_E_NOMEM, std::string("xg_write_mtx: ") + e.what());
    }
}

// ... and from the 16-bit layout (XG_LAYOUT_ROWS_TINY): entry k = (column - previous column of the row - 1) << 4 | count,
// the word 0 = look the entry up in the side list (every row's first entry is there).  The side list is sorted by
// entry index once; a reader walks a row with a cursor into it.
namespace {
struct TinyReader {
    const uint16_t *w;
    const int64_t *idx;
    const int32_t *col, *val;      // side list sorted by idx
    int64_t n;
    int64_t cur = 0;
    uint32_t prev = 0;
    bool bad = false;
    void operator()(int64_t k, bool first, uint32_t *c, uint32_t *v) {
        const uint32_t x = w[k];
        if (x) {
            prev += (x >> 4) + 1u;
            *c = prev;
            *v = x & 15u;
            return;
        }
        if (first || cur >= n || idx[cur] != k) cur = std::lower_bound(idx, idx + n, k) - idx;
        if (cur < n && idx[cur] == k) {
            prev = (uint32_t)col[cur];
            *v = (uint32_t)val[cur];
            cur++;
        } else {
            bad = true;             // (an entry missing from the list: the device list overflowed)
            *v = 0;
        }
        *c = prev;
    }
};
}  // namespace

extern "C" int xg_write_mtx_rows_tiny(const char *path, int32_t n_rows_in, const int64_t *row_beg, const int32_t *row_cnt,
                                      const int32_t *out_row, int32_t n_rows_out, int32_t n_cols, const uint16_t *coldelta16,
                                      int64_t n_over, const int64_t *over_idx, const int32_t *over_col,
                                      const int32_t *over_val, int32_t n_threads) {
    if (!coldelta16 || n_over < 0 || (n_over && (!over_idx || !over_col || !over_val)))
        return fail(XG_E_ARG, "xg_write_mtx: bad argument");
    try {
        std::vector<int64_t> ord((size_t)n_over);
        for (int64_t i = 0; i < n_over; i++) ord[(size_t)i] = i;
        std::sort(ord.begin(), ord.end(), [&](int64_t a, int64_t b) { return over_idx[a] < over_idx[b]; });
        std::vector<int64_t> s_idx((size_t)n_over);
        std::vector<int32_t> s_col((size_t)n_over), s_val((size_t)n_over);
        for (int64_t i = 0; i < n_over; i++) {
            s_idx[(size_t)i] = over_idx[ord[(size_t)i]];
            s_col[(size_t)i] = over_col[ord[(size_t)i]];
            s_val[(size_t)i] = over_val[ord[(size_t)i]];
        }
        TinyReader rd{coldelta16, s_idx.data(), s_col.data(), s_val.data(), n_over};
        return write_rows_impl(path, n_rows_in, row_beg, row_cnt, out_row, n_rows_out, n_cols, rd, n_threads);
    } catch (const std::exception &e) {
        return fail(XG_E_NOMEM, std::string("xg_write_mtx: ") + e.what());
    }
}

extern "C" int xg_write_mtx(const char *path, int32_t n_rows_in, const int64_t *row_ptr, const int32_t *out_row,
                            int32_t n_rows_out, int32_t n_cols, const int32_t *col, const int32_t *val,
                            int32_t n_threads) {
    if (!path || !row_ptr || !out_row || n_rows_in < 0) return fail(XG_E_ARG, "xg_write_mtx: bad argument");
    std::vector<int32_t> cnt((size_t)n_rows_in);
    for (int32_t r = 0; r < n_rows_in; r++) cnt[(size_t)r] = (int32_t)(row_ptr[r + 1] - row_ptr[r]);
    return xg_write_mtx_rows(path, n_rows_in, row_ptr, cnt.data(), out_row, n_rows_out, n_cols, col, val, n_threads);
}

// ---- BAM writer for a record batch (bench / tests) -------------------------------------------------
// The inverse of the decoders: a coordinate-sorted BAM whose records carry exactly what the batch holds --
// pos, flag, mapq, CIGAR (a "simple" read gets its one M operation back), the 4-bit sequence when the batch has
// one (else pseudo-random bases of the CIGAR's query length), constant qualities, CB:Z / UB:Z tags spelled from
// the keys (absent key: no tag), query name "r<record index>" -- or, with name_from_umi, the text of the record's
// UMI key, so that records of one molecule share their name the way mates do (SMART-seq style input, counted
// with --UMItag None).  Blocks are laid out as htslib lays them out
// (whole records per BGZF block, the header in blocks of its own) and compressed by a pool of threads.
// No reference counterpart: it exists so that the file-to-matrix measurement and the decoder tests can start
// from a file of the very records whose matrix is known.
extern "C" int xg_write_bam(const char *path, const xg_reads *r, int32_t n_gid, const char *const *gid_names,
                            const int64_t *gid_lens, xg_keyspace *ks, const char *cell_tag, const char *umi_tag,
                            int32_t name_from_umi, int32_t level, int32_t n_threads) {
    if (!path || !r || n_gid <= 0 || !gid_names || !gid_lens) return fail(XG_E_ARG, "xg_write_bam: bad argument");
    if (n_threads <= 0) n_threads = (int)std::thread::hardware_concurrency();
    if (n_threads <= 0) n_threads = 1;
    if (level < 0 || level > 9) level = 1;
    for (int32_t k = 0; k < r->n_runs; k++) {
        if (r->runs[k].bam_idx != 0) return fail(XG_E_ARG, "xg_write_bam: batch holds more than one BAM");
        if (r->runs[k].gid < 0 || r->runs[k].gid >= n_gid) return fail(XG_E_ARG, "xg_write_bam: run on an unnamed contig");
        if (k && r->runs[k].gid <= r->runs[k - 1].gid) return fail(XG_E_ARG, "xg_write_bam: runs not in contig order");
    }
    const int64_t n = r->n_reads;
    std::vector<int32_t> tid_of((size_t)n_gid, -1);
    // header: the contigs in gid order (tid = gid)
    std::string text = "@HD\tVN:1.6\tSO:coordinate\n";
    for (int32_t g = 0; g < n_gid; g++) text += std::string("@SQ\tSN:") + gid_names[g] + "\tLN:" + std::to_string(gid_lens[g]) + "\n";
    std::string head = std::string("BAM\1", 4);
    auto put32 = [](std::string &s, uint32_t v) { s.append((const char *)&v, 4); };
    put32(head, (uint32_t)text.size());
    head += text;
    put32(head, (uint32_t)n_gid);
    for (int32_t g = 0; g < n_gid; g++) {
        std::string nm = std::string(gid_names[g]) + '\0';
        put32(head, (uint32_t)nm.size());
        head += nm;
        put32(head, (uint32_t)gid_lens[g]);
    }
    // per record: contig (from the runs) and byte size
    std::vector<int32_t> rec_gid((size_t)n, 0);
    for (int32_t k = 0; k < r->n_runs; k++)
        for (int64_t i = r->runs[k].rec_beg; i < r->runs[k].rec_end; i++) rec_gid[(size_t)i] = r->runs[k].gid;
    const bool has_seq = r->seq_off && r->seq;
    auto cigar_of = [&](int64_t i, uint32_t *one, const uint32_t **cg) -> uint32_t {
        const uint32_t ncw = r->fmq[i] >> 24;
        if (ncw == 0) {
            *one = (uint32_t)(r->pos_end[2 * i + 1] - r->pos_end[2 * i]) << 4;
            *cg = one;
            return 1;
        }
        *cg = r->cigar + r->cig_off[i];
        return ncw == 255 ? r->cigar[r->cig_off[i] - 1] : ncw;
    };
    auto qlen_of = [](const uint32_t *cg, uint32_t nc) {
        uint32_t q = 0;
        for (uint32_t k = 0; k < nc; k++) {
            const uint32_t op = cg[k] & 15;
            if (op == 0 || op == 1 || op == 4 || op == 7 || op == 8) q += cg[k] >> 4;
        }
        return q;
    };
    auto key_text = [&](uint64_t key, char *buf) -> int64_t {       // -1: no tag
        if (key == XG_KEY_NONE || key == XG_KEY_NOMATCH) return -1;
        if (key == XG_KEY_EMPTY) return 0;
        if (!(key >> 63)) return xg::key_unpack(key, buf, 64);
        return ks ? ks->decode(key, buf, 256) : -1;
    };
    std::vector<uint32_t> rec_len((size_t)n);
    auto size_range = [&](int64_t a, int64_t b) {
        char buf[260];
        for (int64_t i = a; i < b; i++) {
            uint32_t one;
            const uint32_t *cg;
            const uint32_t nc = cigar_of(i, &one, &cg), q = qlen_of(cg, nc);
            uint32_t l_name = 12;                                       // "r%010lld\0"
            if (name_from_umi) {
                const int64_t m = key_text(r->keys[2 * i + 1], buf);
                if (m > 0 && m < 250) l_name = (uint32_t)m + 1;
            }
            uint32_t len = 36 + l_name + 4 * nc + (q + 1) / 2 + q;      // fixed part, name, CIGAR, SEQ, QUAL
            if (cell_tag) {
                const int64_t m = key_text(r->keys[2 * i], buf);
                if (m >= 0) len += 3 + (uint32_t)m + 1;
            }
            if (umi_tag) {
                const int64_t m = key_text(r->keys[2 * i + 1], buf);
                if (m >= 0) len += 3 + (uint32_t)m + 1;
            }
            rec_len[(size_t)i] = len;
        }
    };
    {
        std::vector<std::thread> th;
        for (int t = 0; t < n_threads; t++)
            th.emplace_back(size_range, n * t / n_threads, n * (t + 1) / n_threads);
        for (auto &x : th) x.join();
    }
    // blocks: as many whole records as fit 0xff00 bytes
    const uint32_t PAYLOAD = 0xff00;
    std::vector<int64_t> blk_first{0};
    {
        uint32_t acc = 0;
        for (int64_t i = 0; i < n; i++) {
            if (rec_len[(size_t)i] > PAYLOAD) return fail(XG_E_LIMIT, "xg_write_bam: record larger than a BGZF block");
            if (acc + rec_len[(size_t)i] > PAYLOAD) {
                blk_first.push_back(i);
                acc = 0;
            }
            acc += rec_len[(size_t)i];
        }
        blk_first.push_back(n);
    }
    const size_t n_blk = blk_first.size() - 1;
    auto bgzf = [&](const uint8_t *src, uint32_t len, std::vector<uint8_t> &out) -> bool {
        uint8_t comp[0x10200];
        z_stream zs;
        memset(&zs, 0, sizeof zs);
        if (deflateInit2(&zs, level, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) return false;
        zs.next_in = const_cast<uint8_t *>(src);
        zs.avail_in = len;
        zs.next_out = comp;
        zs.avail_out = sizeof comp;
        const int rc = deflate(&zs, Z_FINISH);
        const uint32_t clen = (uint32_t)zs.total_out;
        deflateEnd(&zs);
        if (rc != Z_STREAM_END || clen + 26 > 0x10000) return false;
        const uint8_t hdr[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
        out.insert(out.end(), hdr, hdr + 16);
        const uint16_t bsize = (uint16_t)(clen + 25);
        out.push_back((uint8_t)(bsize & 0xff));
        out.push_back((uint8_t)(bsize >> 8));
        out.insert(out.end(), comp, comp + clen);
        const uint32_t crc = (uint32_t)crc32(crc32(0L, Z_NULL, 0), src, len);
        for (int k = 0; k < 4; k++) out.push_back((uint8_t)(crc >> (8 * k)));
        for (int k = 0; k < 4; k++) out.push_back((uint8_t)(len >> (8 * k)));
        return true;
    };
    FILE *fp = fopen(path, "wb");
    if (!fp) return fail(XG_E_IO, std::string("cannot write '") + path + "'");
    std::atomic<bool> ok(true);
    {
        std::vector<uint8_t> hb;
        for (size_t off = 0; off < head.size() && ok; off += PAYLOAD)      // the header in blocks of its own (bam_hdr_write flushes)
            if (!bgzf((const uint8_t *)head.data() + off, (uint32_t)std::min<size_t>(PAYLOAD, head.size() - off), hb)) ok = false;
        if (ok && fwrite(hb.data(), 1, hb.size(), fp) != hb.size()) ok = false;
    }
    auto build_block = [&](size_t b, std::vector<uint8_t> &raw) {
        raw.clear();
        char buf[260];
        for (int64_t i = blk_first[b]; i < blk_first[b + 1]; i++) {
            uint32_t one;
            const uint32_t *cg;
            const uint32_t nc = cigar_of(i, &one, &cg), q = qlen_of(cg, nc);
            const size_t at = raw.size();
            raw.resize(at + rec_len[(size_t)i]);
            uint8_t *p = raw.data() + at;
            auto w32 = [&](size_t o, uint32_t v) { memcpy(p + o, &v, 4); };
            auto w16 = [&](size_t o, uint16_t v) { memcpy(p + o, &v, 2); };
            uint32_t l_name = 12;
            int64_t name_len = -1;
            if (name_from_umi) {
                name_len = key_text(r->keys[2 * i + 1], buf);
                if (name_len > 0 && name_len < 250) l_name = (uint32_t)name_len + 1; else name_len = -1;
            }
            w32(0, rec_len[(size_t)i] - 4);
            w32(4, (uint32_t)rec_gid[(size_t)i]);
            w32(8, (uint32_t)r->pos_end[2 * i]);
            p[12] = (uint8_t)l_name;                          // l_read_name incl. NUL
            p[13] = (uint8_t)((r->fmq[i] >> 16) & 0xff);
            w16(14, 4680);                                    // bin: not used by sequential readers
            w16(16, (uint16_t)std::min<uint32_t>(nc, 65535));
            w16(18, (uint16_t)(r->fmq[i] & 0xffff));
            w32(20, q);
            w32(24, 0xffffffffu);
            w32(28, 0xffffffffu);
            w32(32, 0);
            if (name_len > 0) {
                memcpy(p + 36, buf, (size_t)name_len);
                p[36 + name_len] = 0;
            } else {
                snprintf((char *)p + 36, 12, "r%010lld", (long long)i);
            }
            size_t o = 36 + l_name;
            memcpy(p + o, cg, 4 * (size_t)nc);
            o += 4 * (size_t)nc;
            const size_t nb = (q + 1) / 2;
            if (has_seq) {
                memcpy(p + o, (const uint8_t *)(r->seq + r->seq_off[i]), nb);
            } else {
                uint64_t h = (uint64_t)i * 0x9E3779B97F4A7C15ULL + 12345;
                for (size_t k = 0; k < nb; k++) {
                    h ^= h >> 29;
                    h *= 0xBF58476D1CE4E5B9ULL;
                    p[o + k] = (uint8_t)(((1u << (h & 3)) << 4) | (1u << ((h >> 2) & 3)));
                }
                if (q & 1) p[o + nb - 1] &= 0xf0;
            }
            o += nb;
            memset(p + o, 0xff, q);
            o += q;
            const char *tags[2] = {cell_tag, umi_tag};
            for (int t = 0; t < 2; t++) {
                if (!tags[t]) continue;
                const int64_t m = key_text(r->keys[2 * i + t], buf);
                if (m < 0) continue;
                p[o] = (uint8_t)tags[t][0];
                p[o + 1] = (uint8_t)tags[t][1];
                p[o + 2] = 'Z';
                memcpy(p + o + 3, buf, (size_t)m);
                p[o + 3 + m] = 0;
                o += 4 + (size_t)m;
            }
        }
    };
    // groups of blocks: compressed by the pool, written in order
    const size_t GROUP = (size_t)n_threads * 64;
    std::vector<std::vector<uint8_t>> out(GROUP);
    for (size_t b0 = 0; b0 < n_blk && ok; b0 += GROUP) {
        const size_t b1 = std::min(n_blk, b0 + GROUP);
        std::atomic<size_t> next(b0);
        std::vector<std::thread> th;
        for (int t = 0; t < n_threads; t++)
            th.emplace_back([&]() {
                std::vector<uint8_t> raw;
                raw.reserve(0x10000);
                for (;;) {
                    const size_t b = next.fetch_add(1);
                    if (b >= b1 || !ok) break;
                    build_block(b, raw);
                    out[b - b0].clear();
                    if (!bgzf(raw.data(), (uint32_t)raw.size(), out[b - b0])) ok = false;
                }
            });
        for (auto &x : th) x.join();
        for (size_t b = b0; b < b1 && ok; b++)
            if (fwrite(out[b - b0].data(), 1, out[b - b0].size(), fp) != out[b - b0].size()) ok = false;
    }
    static const uint8_t eof_block[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0,
                                          0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    if (ok && fwrite(eof_block, 1, 28, fp) != 28) ok = false;
    if (fclose(fp) != 0) ok = false;
    if (!ok) return fail(XG_E_IO, std::string("writing '") + path + "' failed");
    return XG_OK;
}

// ---- splitting a BAM between GPUs (host side) --------------------------------------------------------
// Offsets of the BGZF blocks of a file: the chain of block sizes is followed with one small read per block
// (nothing is inflated).  *offsets (n + 1 entries, the last one = file size) is malloc'ed: xg_free_array().
// *first_record_block: the block in which the first alignment record starts, and *aligned = 1 when it starts
// exactly at that block's beginning (htslib flushes after the header), else 0.
extern "C" int xg_bgzf_block_index(const char *path, int64_t **offsets, int64_t *n_blocks, int64_t *first_record_block,
                                   int32_t *aligned) {
    if (!path || !offsets || !n_blocks) return fail(XG_E_ARG, "xg_bgzf_block_index: null argument");
    xg_dec::BamFile bf;
    int rc = xg_dec::open_bam(path, bf, true);       // header only
    if (rc) return rc;
    const uint64_t hdr_usize = bf.h.end_off;
    FILE *fp = fopen(path, "rb");
    if (!fp) return fail(XG_E_IO, std::string("cannot open '") + path + "'");
    std::vector<int64_t> off;
    int64_t at = 0, first_blk = -1;
    int32_t is_aligned = 0;
    uint64_t usize = 0;
    uint8_t h[18];
    while (true) {
        if (fseeko(fp, (off_t)at, SEEK_SET) != 0) break;
        const size_t got = fread(h, 1, 18, fp);
        if (got == 0) break;
        uint32_t total = 0, hl = 0;
        if (got < 18 || xg_dec::bgzf_block_header(h, 1u << 20, &total, &hl) < 0 || total < 26) {
            fclose(fp);
            return fail(XG_E_FORMAT, std::string("'") + path + "' is not BGZF (bad block header)");
        }
        if (first_blk < 0) {                        // still inside the header: this block's inflated size
            uint8_t t4[4];
            if (fseeko(fp, (off_t)(at + total - 4), SEEK_SET) != 0 || fread(t4, 1, 4, fp) != 4) {
                fclose(fp);
                return fail(XG_E_FORMAT, std::string("truncated BGZF block in '") + path + "'");
            }
            const uint32_t isize = rd32(t4);
            if (usize + isize > hdr_usize || (usize == hdr_usize && isize > 0)) {
                first_blk = (int64_t)off.size();
                is_aligned = usize == hdr_usize ? 1 : 0;
            }
            usize += isize;
        }
        off.push_back(at);
        at += total;
    }
    fclose(fp);
    off.push_back(at);
    if (first_blk < 0) first_blk = (int64_t)off.size() - 1;       // no record at all
    int64_t *o = (int64_t *)malloc(off.size() * sizeof(int64_t));
    if (!o) return fail(XG_E_NOMEM, "out of memory");
    memcpy(o, off.data(), off.size() * sizeof(int64_t));
    *offsets = o;
    *n_blocks = (int64_t)off.size() - 1;
    if (first_record_block) *first_record_block = first_blk;
    if (aligned) *aligned = is_aligned;
    return XG_OK;
}

extern "C" void xg_free_array(void *p) { free(p); }

// (tid, pos) of the record at the beginning of the block at `offset` (htslib writes whole records per block): one
// block is read and inflated.  tid = -2: the block is empty (the EOF marker) or too short for a record header.
extern "C" int xg_bam_block_probe(const char *path, int64_t offset, int32_t *tid, int32_t *pos) {
    if (!path || !tid || !pos) return fail(XG_E_ARG, "xg_bam_block_probe: null argument");
    *tid = -2;
    *pos = -1;
    FILE *fp = fopen(path, "rb");
    if (!fp) return fail(XG_E_IO, std::string("cannot open '") + path + "'");
    std::vector<uint8_t> buf(0x10000 + 64);
    if (fseeko(fp, (off_t)offset, SEEK_SET) != 0) {
        fclose(fp);
        return fail(XG_E_IO, "seek failed");
    }
    const size_t got = fread(buf.data(), 1, buf.size(), fp);
    fclose(fp);
    uint32_t total = 0, hl = 0;
    if (got < 26 || xg_dec::bgzf_block_header(buf.data(), got, &total, &hl) != 0 || total > got)
        return fail(XG_E_FORMAT, std::string("no BGZF block at the given offset of '") + path + "'");
    xg_dec::BgzfBlock b;
    b.coff = hl;
    b.clen = total - hl - 8;
    memcpy(&b.isize, buf.data() + total - 4, 4);
    memcpy(&b.crc, buf.data() + total - 8, 4);
    b.uoff = 0;
    xg_dec::Bytes u;
    int rc = xg_dec::inflate_blocks(buf.data(), 0, &b, 1, u, 1);
    if (rc) return rc;
    if (u.size() < 12) return XG_OK;
    *tid = (int32_t)rd32(&u[4]);
    *pos = (int32_t)rd32(&u[8]);
    return XG_OK;
}

// ---- the BAM index (.bai, SAMv1 section 5.2) -------------------------------------------------------------
// Which blocks hold the records of a set of intervals, the way htslib's bam_itr_queryi finds them: the chunks of the
// bins that overlap an interval (reg2bins), less those that end before the linear index's offset of the interval's
// 16 kb window.  The chunks are then widened to whole BGZF blocks and merged, so that the device decoder can stage
// them: a range starts at the block of its first chunk and ends at the block after its last chunk's end.
struct xg_bam_index {
    struct Ref {
        std::vector<uint32_t> bins;          // ascending
        std::vector<int64_t> bin_ptr;        // bins.size() + 1 entries into chunks (pairs)
        std::vector<uint64_t> chunks;        // (beg, end) virtual offsets, per bin as the index lists them
        std::vector<uint64_t> linear;        // 16 kb windows
    };
    std::string bam_path;
    uint64_t bam_size = 0;
    std::vector<Ref> refs;
};

namespace {

constexpr uint32_t BAI_PSEUDO_BIN = 37450;

int bai_fail(const std::string &bai, const std::string &why) {
    return fail(XG_E_FORMAT, std::string("index '") + bai + "' is not used: " + why);
}

int bai_parse(const Bytes &f, const std::string &bai, xg_bam_index &idx) {
    const uint64_t n = f.size();
    uint64_t o = 0;
    auto need = [&](uint64_t k) { return o + k <= n; };
    if (!need(8) || memcmp(f.data(), "BAI\1", 4) != 0) return bai_fail(bai, "not a BAI file");
    const int32_t n_ref = (int32_t)rd32(&f[4]);
    o = 8;
    if (n_ref < 0) return bai_fail(bai, "negative n_ref");
    idx.refs.resize((size_t)n_ref);
    for (int32_t t = 0; t < n_ref; t++) {
        xg_bam_index::Ref &R = idx.refs[(size_t)t];
        if (!need(4)) return bai_fail(bai, "truncated");
        const int32_t n_bin = (int32_t)rd32(&f[o]);
        o += 4;
        if (n_bin < 0) return bai_fail(bai, "negative n_bin");
        std::vector<std::pair<uint32_t, std::pair<uint64_t, uint64_t>>> all;     // (bin, chunk); stable by bin below
        for (int32_t b = 0; b < n_bin; b++) {
            if (!need(8)) return bai_fail(bai, "truncated");
            const uint32_t bin = rd32(&f[o]);
            const int32_t n_chunk = (int32_t)rd32(&f[o + 4]);
            o += 8;
            if (n_chunk < 0 || !need(16ull * (uint64_t)n_chunk)) return bai_fail(bai, "truncated");
            for (int32_t c = 0; c < n_chunk; c++, o += 16) {
                uint64_t cb, ce;
                memcpy(&cb, &f[o], 8);
                memcpy(&ce, &f[o + 8], 8);
                if (bin == BAI_PSEUDO_BIN) continue;          // (ref_beg, ref_end), (n_mapped, n_unmapped)
                if (bin > BAI_PSEUDO_BIN) return bai_fail(bai, "bin number out of range");
                all.push_back({bin, {cb, ce}});
            }
        }
        std::stable_sort(all.begin(), all.end(), [](const auto &x, const auto &y) { return x.first < y.first; });
        for (const auto &e : all) {
            if (R.bins.empty() || R.bins.back() != e.first) {
                R.bins.push_back(e.first);
                R.bin_ptr.push_back((int64_t)R.chunks.size() / 2);
            }
            R.chunks.push_back(e.second.first);
            R.chunks.push_back(e.second.second);
        }
        R.bin_ptr.push_back((int64_t)R.chunks.size() / 2);
        if (!need(4)) return bai_fail(bai, "truncated");
        const int32_t n_intv = (int32_t)rd32(&f[o]);
        o += 4;
        if (n_intv < 0 || !need(8ull * (uint64_t)n_intv)) return bai_fail(bai, "truncated");
        R.linear.resize((size_t)n_intv);
        if (n_intv) memcpy(R.linear.data(), &f[o], 8ull * (uint64_t)n_intv);
        o += 8ull * (uint64_t)n_intv;
    }
    // an optional n_no_coor may follow
    return XG_OK;
}

// The BGZF block at file offset `coff`: its total and inflated sizes; false when no block header is there.
bool block_at(FILE *fp, uint64_t coff, uint32_t *total, uint32_t *isize) {
    uint8_t h[18], t4[4];
    if (fseeko(fp, (off_t)coff, SEEK_SET) != 0 || fread(h, 1, 18, fp) != 18) return false;
    uint32_t hl = 0;
    if (bgzf_block_header(h, 18, total, &hl) != 0) return false;
    if (fseeko(fp, (off_t)(coff + *total - 4), SEEK_SET) != 0 || fread(t4, 1, 4, fp) != 4) return false;
    *isize = rd32(t4);
    return true;
}

}  // namespace

extern "C" int xg_bam_index_open(const char *bam_path, xg_bam_index **out) {
    if (!bam_path || !out) return fail(XG_E_ARG, "xg_bam_index_open: null argument");
    *out = nullptr;
    std::string bam(bam_path), bai = bam + ".bai";
    struct stat st_bai, st_bam;
    if (stat(bai.c_str(), &st_bai) != 0) {
        if (bam.size() > 4 && bam.compare(bam.size() - 4, 4, ".bam") == 0) bai = bam.substr(0, bam.size() - 4) + ".bai";
        if (stat(bai.c_str(), &st_bai) != 0) return XG_OK;     // no index: the caller reads the whole file
    }
    if (stat(bam_path, &st_bam) != 0) return fail(XG_E_IO, std::string("cannot open '") + bam + "'");
    if (st_bai.st_mtime < st_bam.st_mtime) return bai_fail(bai, "it is older than the BAM");
    std::unique_ptr<xg_bam_index> idx(new (std::nothrow) xg_bam_index());
    if (!idx) return fail(XG_E_NOMEM, "out of memory");
    idx->bam_path = bam;
    idx->bam_size = (uint64_t)st_bam.st_size;
    {
        Bytes f;
        int rc = read_file(bai.c_str(), f);
        if (rc) return rc;
        try {
            rc = bai_parse(f, bai, *idx);
        } catch (const std::exception &e) {
            return fail(XG_E_NOMEM, std::string("reading '") + bai + "': " + e.what());
        }
        if (rc) return rc;
    }
    BamFile bf;
    int rc = open_bam(bam_path, bf, true);
    if (rc) return rc;
    if (bf.h.names.size() != idx->refs.size())
        return bai_fail(bai, "it lists " + std::to_string(idx->refs.size()) + " contigs, the BAM header " +
                                 std::to_string(bf.h.names.size()));
    for (const auto &R : idx->refs) {
        for (uint64_t v : R.chunks)
            if ((v >> 16) >= idx->bam_size) return bai_fail(bai, "an offset lies beyond the end of the BAM");
        for (uint64_t v : R.linear)
            if ((v >> 16) >= idx->bam_size) return bai_fail(bai, "an offset lies beyond the end of the BAM");
    }
    *out = idx.release();
    return XG_OK;
}

extern "C" void xg_bam_index_free(xg_bam_index *idx) { delete idx; }

extern "C" int32_t xg_bam_index_n_ref(const xg_bam_index *idx) { return idx ? (int32_t)idx->refs.size() : 0; }

extern "C" int xg_bam_index_ref(const xg_bam_index *idx, int32_t tid, int64_t *n_bins, const uint32_t **bins,
                                const int64_t **bin_ptr, const uint64_t **chunks, int64_t *n_intv,
                                const uint64_t **linear) {
    if (!idx || tid < 0 || tid >= (int32_t)idx->refs.size()) return fail(XG_E_ARG, "xg_bam_index_ref: no such contig");
    const xg_bam_index::Ref &R = idx->refs[(size_t)tid];
    *n_bins = (int64_t)R.bins.size();
    *bins = R.bins.data();
    *bin_ptr = R.bin_ptr.data();
    *chunks = R.chunks.data();
    *n_intv = (int64_t)R.linear.size();
    *linear = R.linear.data();
    return XG_OK;
}

static int bam_index_ranges_impl(const xg_bam_index *idx, int64_t n, const int32_t *tid, const int64_t *beg,
                                 const int64_t *end, int64_t **ranges, int64_t *n_ranges) {
    // (tid, bin) -> the smallest linear-index offset among the intervals that visit the bin
    std::unordered_map<uint64_t, uint64_t> visit;
    for (int64_t i = 0; i < n; i++) {
        if (tid[i] < 0 || tid[i] >= (int32_t)idx->refs.size()) continue;
        const int64_t b = std::max<int64_t>(0, beg[i]), e = std::min<int64_t>(end[i], (int64_t)1 << 29);
        if (e <= b) continue;
        const xg_bam_index::Ref &R = idx->refs[(size_t)tid[i]];
        if (R.bins.empty()) continue;
        const uint64_t w = (uint64_t)b >> 14;
        const uint64_t min_off = w < R.linear.size() ? R.linear[w] : 0;
        const int64_t last = e - 1;
        const int shifts[6] = {29, 26, 23, 20, 17, 14};
        const uint32_t firsts[6] = {0, 1, 9, 73, 585, 4681};
        for (int l = 0; l < 6; l++)
            for (uint32_t k = firsts[l] + (uint32_t)(b >> shifts[l]); k <= firsts[l] + (uint32_t)(last >> shifts[l]); k++) {
                if (!std::binary_search(R.bins.begin(), R.bins.end(), k)) continue;
                const uint64_t key = ((uint64_t)(uint32_t)tid[i] << 32) | k;
                auto it = visit.find(key);
                if (it == visit.end()) visit.emplace(key, min_off);
                else it->second = std::min(it->second, min_off);
            }
    }
    std::vector<std::pair<uint64_t, uint64_t>> ch;
    for (const auto &kv : visit) {
        const xg_bam_index::Ref &R = idx->refs[(size_t)(kv.first >> 32)];
        const size_t j = (size_t)(std::lower_bound(R.bins.begin(), R.bins.end(), (uint32_t)kv.first) - R.bins.begin());
        for (int64_t c = R.bin_ptr[j]; c < R.bin_ptr[j + 1]; c++) {
            const uint64_t cb = R.chunks[2 * (size_t)c], ce = R.chunks[2 * (size_t)c + 1];
            if (ce > kv.second && ce > cb) ch.push_back({cb, ce});
        }
    }
    std::sort(ch.begin(), ch.end());
    std::vector<std::pair<uint64_t, uint64_t>> vm;              // merged in virtual offsets
    for (const auto &c : ch) {
        if (!vm.empty() && c.first <= vm.back().second) vm.back().second = std::max(vm.back().second, c.second);
        else vm.push_back(c);
    }
    std::vector<int64_t> out;
    FILE *fp = vm.empty() ? nullptr : fopen(idx->bam_path.c_str(), "rb");
    if (!vm.empty() && !fp) return fail(XG_E_IO, "cannot open '" + idx->bam_path + "'");
    auto bad = [&](const std::string &why) {
        fclose(fp);
        return fail(XG_E_FORMAT, "index of '" + idx->bam_path + "' is not used: " + why);
    };
    for (const auto &c : vm) {
        const uint64_t lo = c.first >> 16, last = c.second >> 16;
        uint32_t total = 0, isize = 0;
        uint64_t hi = last;
        if (c.second & 0xffff) {                                // the last chunk ends inside block `last`
            if (!block_at(fp, last, &total, &isize)) return bad("offset " + std::to_string(last) + " is not a BGZF block start");
            hi = last + total;
        }
        if (hi > idx->bam_size) return bad("an offset lies beyond the end of the BAM");
        if (hi <= lo) continue;
        if (!out.empty() && (int64_t)lo <= out.back() + XG_BAM_INDEX_MERGE_GAP) {     // close enough: read the gap too
            out.back() = std::max<int64_t>(out.back(), (int64_t)hi);
            continue;
        }
        if (!block_at(fp, lo, &total, &isize)) return bad("offset " + std::to_string(lo) + " is not a BGZF block start");
        if ((c.first & 0xffff) >= isize) return bad("a record offset lies beyond its block");
        out.push_back((int64_t)c.first);                        // the virtual offset of the range's first record
        out.push_back((int64_t)hi);
    }
    if (fp) fclose(fp);
    int64_t *o = (int64_t *)malloc(std::max<size_t>(1, out.size()) * sizeof(int64_t));
    if (!o) return fail(XG_E_NOMEM, "out of memory");
    if (!out.empty()) memcpy(o, out.data(), out.size() * sizeof(int64_t));
    *ranges = o;
    *n_ranges = (int64_t)out.size() / 2;
    return XG_OK;
}

extern "C" int xg_bam_index_ranges(const xg_bam_index *idx, int64_t n, const int32_t *tid, const int64_t *beg,
                                   const int64_t *end, int64_t **ranges, int64_t *n_ranges) {
    if (!idx || n < 0 || (n && (!tid || !beg || !end)) || !ranges || !n_ranges)
        return fail(XG_E_ARG, "xg_bam_index_ranges: bad argument");
    try {
        return bam_index_ranges_impl(idx, n, tid, beg, end, ranges, n_ranges);
    } catch (const std::exception &e) {
        return fail(XG_E_NOMEM, std::string("xg_bam_index_ranges: ") + e.what());
    }
}
