#include <cstdint>
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <vector>
#include <zlib.h>
#define __device__
#define __forceinline__ inline
#define __noinline__
#define __constant__
struct TI { unsigned x; } threadIdx = {0};
static inline unsigned __brev(unsigned v) { unsigned r = 0; for (int i = 0; i < 32; i++) if (v & (1u << i)) r |= 1u << (31 - i); return r; }
static inline int __ffs(int v) { return __builtin_ffs(v); }
template <class T> T __shfl_sync(unsigned, T v, int, int = 32) { return v; }
template <class T> T __shfl_up_sync(unsigned, T v, int, int) { return v; }
static inline unsigned __ballot_sync(unsigned, bool p) { return p ? 1u : 0u; }
static inline void __syncwarp(unsigned) {}
static inline bool __any_sync(unsigned, bool p) { return p; }
static inline unsigned __funnelshift_r(unsigned lo, unsigned hi, unsigned sh) {
    return (unsigned)(((((unsigned long long)hi) << 32) | lo) >> (sh & 31));
}
static inline unsigned __reduce_or_sync(unsigned, unsigned v) { return v; }
static inline int __popc(unsigned v) { return __builtin_popcount(v); }
using std::min;
#include "../xcltk_b200/csrc/inflate.cuh"
// harness FILE [-r]: every block against zlib; with -r also each block's inflate_group<1> return code
int main(int argc, char **argv) {
    FILE *fp = fopen(argv[1], "rb");
    const bool print_rc = argc > 2 && !strcmp(argv[2], "-r");
    std::vector<uint8_t> f;
    uint8_t tmp[65536];
    size_t n;
    while ((n = fread(tmp, 1, sizeof tmp, fp)) > 0) f.insert(f.end(), tmp, tmp + n);
    f.resize(f.size() + 64);
    size_t off = 0, fsz = f.size() - 64;
    int bi = 0, bad = 0;
    static xg_inflate::GroupSmem g;
    while (off < fsz) {
        unsigned xlen = f[off + 10] | (f[off + 11] << 8);
        unsigned bsize = (f[off + 16] | (f[off + 17] << 8)) + 1;
        unsigned clen = bsize - 12 - xlen - 8;
        unsigned isize; memcpy(&isize, &f[off + bsize - 4], 4);
        std::vector<uint8_t> exp(isize + 1), got(isize + 64);
        z_stream zs; memset(&zs, 0, sizeof zs); inflateInit2(&zs, -15);
        zs.next_in = &f[off + 12 + xlen]; zs.avail_in = clen; zs.next_out = exp.data(); zs.avail_out = isize;
        inflate(&zs, Z_FINISH); inflateEnd(&zs);
        int r = isize ? xg_inflate::inflate_group<1>(g, &f[off + 12 + xlen], clen, got.data(), isize) : 0;
        if (print_rc) printf("block %d: rc %d\n", bi, r);
        // the lane-parallel CRC's arithmetic: 32 chunk CRCs combined must give the block's CRC32
        {
            const unsigned chunk = (isize + 31u) / 32u;
            unsigned total = 0;
            for (unsigned lane = 0; lane < 32; lane++) {
                const unsigned beg = std::min(isize, lane * chunk), end = std::min(isize, beg + chunk);
                if (end == beg) continue;
                const unsigned ci = (unsigned)crc32(crc32(0L, Z_NULL, 0), exp.data() + beg, end - beg);
                total ^= xg_inflate::crc_multmodp(xg_inflate::crc_x8n(isize - end), ci);
            }
            unsigned trailer;
            memcpy(&trailer, &f[off + bsize - 8], 4);
            if (isize && (total != trailer || total != (unsigned)crc32(crc32(0L, Z_NULL, 0), exp.data(), isize))) {
                printf("block %d: combined CRC %08x, trailer %08x\n", bi, total, trailer);
                bad++;
            }
        }
        if (r != (int)isize || memcmp(got.data(), exp.data(), isize)) {
            if (bad < 5) {
                size_t k = 0; while (k < isize && got[k] == exp[k]) k++;
                printf("block %d: r=%d isize=%u first diff at %zu\n", bi, r, isize, k);
            }
            bad++;
        }
        off += bsize; bi++;
    }
    printf("%d blocks, %d bad\n", bi, bad);
}
