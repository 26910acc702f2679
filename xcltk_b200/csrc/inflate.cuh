// inflate.cuh -- DEFLATE (RFC 1951) decoder for BGZF blocks on the device.
//
// BGZF (SAMv1 section 4.1) is a series of independent gzip members of <= 64 KiB payload, so a
// BAM file inflates block-parallel: the reference reaches the same bytes through
// pysam/htslib's bgzf reader (`pysam.AlignmentFile`, xcltk/rdr/fc/core.py:75).  Written from the
// RFC.  One group of S lanes (S = 32: a warp) owns one BGZF block:
//   * lane 0 runs the serial part -- block headers, code tables, Huffman decoding -- against
//     lookup tables in shared memory (2^10 literal/length entries, 2^8 distance entries, each
//     entry carrying code length, extra-bit count and base value; longer codes take the
//     canonical count/symbol walk) and queues up to S symbols;
//   * all S lanes then write the batch: a prefix sum over the symbols' output lengths places
//     them, literals are stored side by side, each LZ77 match is copied by the whole group
//     (period-d indexing, so a match never reads its own output), stored blocks are copied
//     coalesced.
// The per-symbol instruction count of lane 0 bounds the kernel (issue-bound, not HBM-bound).
#pragma once
#include <cstdint>

struct BgzfBlockDev {
    unsigned long long coff;   // offset of the deflate payload in the compressed buffer
    unsigned int clen;         // payload bytes
    unsigned int isize;        // uncompressed bytes
    unsigned long long uoff;   // offset in the uncompressed stream
    unsigned char *uptr;       // where the block is inflated to (slabs: blocks are contiguous within one)
    unsigned int crc;          // CRC32 of the uncompressed bytes (gzip trailer)
    unsigned int skip;         // leading bytes the record walk leaves out (the head of a range's first block)
};

namespace xg_inflate {

constexpr int LB = 10;     // literal/length table bits
constexpr int DB = 8;      // distance table bits
constexpr uint32_t KIND_LIT = 0, KIND_LEN = 1, KIND_EOB = 2, KIND_BAD = 3;

struct GroupSmem {
    uint32_t lut[1 << LB];
    uint32_t dlut[1 << DB];
    uint32_t queue[32];
    uint32_t cllut[128];          // code-length code table (7 bits)
    uint16_t lsym[288], lcount[16];
    uint16_t dsym[32], dcount[16];
    uint16_t offs[16], next[16];
    uint8_t lens[320];
    uint8_t cl_lens[32];
};

// entry: [0:3] code length, [4:7] extra bits, [8:23] base value, [28:31] kind; 0 = not in table
__device__ __forceinline__ uint32_t lit_entry(int s, int l) {
    if (s < 256) return (uint32_t)l | ((uint32_t)s << 8);
    if (s == 256) return (uint32_t)l | (KIND_EOB << 28);
    if (s > 285) return (uint32_t)l | (KIND_BAD << 28);
    const int idx = s - 257;
    int ex = 0, base;
    if (idx < 8) base = 3 + idx;
    else if (idx == 28) base = 258;
    else {
        ex = (idx >> 2) - 1;
        base = ((4 + (idx & 3)) << ex) + 3;
    }
    return (uint32_t)l | ((uint32_t)ex << 4) | ((uint32_t)base << 8) | (KIND_LEN << 28);
}
__device__ __forceinline__ uint32_t dist_entry(int s, int l) {
    if (s > 29) return (uint32_t)l | (KIND_BAD << 28);
    int ex = 0, base;
    if (s < 4) base = 1 + s;
    else {
        ex = (s >> 1) - 1;
        base = ((2 + (s & 1)) << ex) + 1;
    }
    return (uint32_t)l | ((uint32_t)ex << 4) | ((uint32_t)base << 8);
}
__device__ __forceinline__ uint32_t cl_entry(int s, int l) { return (uint32_t)l | ((uint32_t)s << 8); }

// Canonical code from code lengths: per-length counts + symbols ordered by (length, symbol) for
// the long-code walk, and the 2^tbits lookup table (already zeroed) indexed by the next tbits
// input bits (LSB first, so codes are bit-reversed).  mode 0 literal/length, 1 distance,
// 2 code-length code.  Returns 0 ok, -1 over-subscribed, 1 incomplete.
__device__ int build_table(GroupSmem &g, const uint8_t *lens, int n, uint32_t *lut, int tbits, uint16_t *symarr,
                           uint16_t *count, int mode) {
    for (int l = 0; l < 16; l++) count[l] = 0;
    for (int s = 0; s < n; s++) count[lens[s]]++;
    if (count[0] == n) return 0;
    int left = 1;
    for (int l = 1; l < 16; l++) {
        left = (left << 1) - count[l];
        if (left < 0) return -1;
    }
    g.offs[1] = 0;
    for (int l = 1; l < 15; l++) g.offs[l + 1] = g.offs[l] + count[l];
    uint32_t code = 0;
    for (int l = 1; l < 16; l++) {
        code = (code + (l > 1 ? count[l - 1] : 0)) << 1;
        g.next[l] = (uint16_t)code;
    }
    for (int s = 0; s < n; s++) {
        const int l = lens[s];
        if (!l) continue;
        if (symarr) symarr[g.offs[l]++] = (uint16_t)s;
        const uint32_t c = g.next[l]++;
        if (l <= tbits) {
            const uint32_t e = mode == 0 ? lit_entry(s, l) : mode == 1 ? dist_entry(s, l) : cl_entry(s, l);
            for (uint32_t i = __brev(c) >> (32 - l); i < (1u << tbits); i += 1u << l) lut[i] = e;
        }
    }
    return left > 0 ? 1 : 0;
}

// code longer than the table: walk the lengths on the peeked bits
__device__ __noinline__ int slow_decode(uint32_t buf, const uint16_t *count, const uint16_t *symarr, int *len) {
    int code = 0, first = 0, index = 0;
    for (int l = 1; l < 16; l++) {
        code |= (int)((buf >> (l - 1)) & 1u);
        const int c = count[l];
        if (code - c < first) {
            *len = l;
            return symarr[index + (code - first)];
        }
        index += c;
        first = (first + c) << 1;
        code <<= 1;
    }
    return -1;
}

// Bit window over the compressed stream: two consecutive little-endian words and the bit
// offset into the first; peek() is one funnel shift, skip() refills at most once (n <= 32).
// The words are read aligned, so up to 3 bytes before the stream and 11 after it are touched
// (both inside the compressed buffer: neighbouring blocks / its padding).
struct BitReader {
    const uint32_t *wp;     // next word to load
    uint32_t w0, w1, pos;   // pos in [0, 32)
    __device__ __forceinline__ void init(const uint8_t *p) {
        const uintptr_t a = (uintptr_t)p;
        wp = (const uint32_t *)(a & ~(uintptr_t)3);
        pos = (uint32_t)(a & 3) * 8;
        w0 = wp[0];
        w1 = wp[1];
        wp += 2;
    }
    __device__ __forceinline__ uint32_t peek() const { return __funnelshift_r(w0, w1, pos); }
    __device__ __forceinline__ void skip(uint32_t n) {
        pos += n;
        if (pos >= 32) {
            w0 = w1;
            w1 = *wp++;
            pos -= 32;
        }
    }
    __device__ __forceinline__ uint32_t take(uint32_t n) {   // n <= 16
        const uint32_t v = peek() & ((1u << n) - 1u);
        skip(n);
        return v;
    }
    __device__ __forceinline__ void align_byte() { skip((8 - (pos & 7)) & 7); }
    __device__ __forceinline__ const uint8_t *byte_pos() const { return (const uint8_t *)(wp - 2) + (pos >> 3); }
};

__device__ __constant__ const unsigned char CL_ORDER[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

// Inflate one raw DEFLATE stream with a group of S lanes (S a power of two <= 32; all lanes of
// the group call with the same arguments).  Returns bytes produced or a negative error.
template <int S>
__device__ int inflate_group(GroupSmem &g, const uint8_t *in, uint32_t n_in, uint8_t *out, uint32_t cap) {
    const unsigned lane_w = threadIdx.x & 31u, lane = lane_w & (S - 1), gbase = lane_w & ~(unsigned)(S - 1);
    const unsigned gmask = (S == 32) ? 0xffffffffu : (((1u << S) - 1u) << gbase);
    BitReader br;
    const uint8_t *in_end = in + n_in;
    if (lane == 0) br.init(in);
    uint32_t o = 0;            // bytes written (uniform over the group)
    int last = 0;
    while (!last) {
        // ---- block header (lane 0) ----
        int type = 0, err = 0;
        uint32_t stored_len = 0;
        const uint8_t *stored_src = nullptr;
        int hlit = 0, hdist = 0;
        if (lane == 0) {
            last = (int)br.take(1);
            type = (int)br.take(2);
            if ((const uint8_t *)br.wp > in_end + 16) err = -20;
            if (type == 0) {
                br.align_byte();
                const uint32_t len = br.take(16), nlen = br.take(16);
                if ((len ^ 0xffffu) != nlen) err = -2;
                stored_len = len;
                stored_src = br.byte_pos();
                if (stored_src + len > in_end) err = -2;
            } else if (type == 1) {
                int s = 0;
                for (; s < 144; s++) g.lens[s] = 8;
                for (; s < 256; s++) g.lens[s] = 9;
                for (; s < 280; s++) g.lens[s] = 7;
                for (; s < 288; s++) g.lens[s] = 8;
                for (; s < 320; s++) g.lens[s] = 5;
                hlit = 288;
                hdist = 30;
            } else if (type == 2) {
                hlit = (int)br.take(5) + 257;
                hdist = (int)br.take(5) + 1;
                const int hclen = (int)br.take(4) + 4;
                if (hlit > 286 || hdist > 30) err = -5;
                for (int k = 0; k < 19; k++) g.cl_lens[k] = 0;
                for (int k = 0; k < hclen; k++) g.cl_lens[CL_ORDER[k]] = (uint8_t)br.take(3);
                for (int k = 0; k < 128; k++) g.cllut[k] = 0;
                if (!err && build_table(g, g.cl_lens, 19, g.cllut, 7, nullptr, g.lcount, 2) != 0) err = -6;
                int idx = 0;
                while (!err && idx < hlit + hdist) {
                    const uint32_t e = g.cllut[br.peek() & 127u];
                    const uint32_t l = e & 15u;
                    if (!l) {
                        err = -7;
                        break;
                    }
                    br.skip(l);
                    const int sym = (int)(e >> 8);
                    if (sym < 16) {
                        g.lens[idx++] = (uint8_t)sym;
                    } else {
                        int prev = 0, rep;
                        if (sym == 16) {
                            if (idx == 0) {
                                err = -8;
                                break;
                            }
                            prev = g.lens[idx - 1];
                            rep = 3 + (int)br.take(2);
                        } else if (sym == 17) {
                            rep = 3 + (int)br.take(3);
                        } else {
                            rep = 11 + (int)br.take(7);
                        }
                        if (idx + rep > hlit + hdist) {
                            err = -9;
                            break;
                        }
                        while (rep--) g.lens[idx++] = (uint8_t)prev;
                    }
                }
                if (!err && g.lens[256] == 0) err = -10;
            } else {
                err = -4;
            }
        }
        err = __shfl_sync(gmask, err, 0, S);
        if (err) return err;
        last = __shfl_sync(gmask, last, 0, S);
        type = __shfl_sync(gmask, type, 0, S);
        if (type == 0) {
            stored_len = __shfl_sync(gmask, stored_len, 0, S);
            stored_src = (const uint8_t *)__shfl_sync(gmask, (unsigned long long)stored_src, 0, S);
            if (o + stored_len > cap) return -3;
            for (uint32_t k = lane; k < stored_len; k += S) out[o + k] = stored_src[k];
            o += stored_len;
            if (lane == 0) br.init(stored_src + stored_len);
            __syncwarp(gmask);
            continue;
        }
        // ---- code tables ----
        for (int k = (int)lane; k < (1 << LB); k += S) g.lut[k] = 0;
        for (int k = (int)lane; k < (1 << DB); k += S) g.dlut[k] = 0;
        __syncwarp(gmask);
        if (lane == 0) {
            // an incomplete code is legal only as one code of one bit (RFC 1951 3.2.7; zlib's inflate_table)
            int e1 = build_table(g, g.lens, hlit, g.lut, LB, g.lsym, g.lcount, 0);
            if (type == 2 && (e1 < 0 || (e1 > 0 && (hlit - g.lcount[0] != 1 || g.lcount[1] != 1)))) err = -11;
            int e2 = build_table(g, g.lens + hlit, hdist, g.dlut, DB, g.dsym, g.dcount, 1);
            if (type == 2 && (e2 < 0 || (e2 > 0 && (hdist - g.dcount[0] != 1 || g.dcount[1] != 1)))) err = -12;   // fixed distance code: 30 of 32
        }
        err = __shfl_sync(gmask, err, 0, S);
        if (err) return err;
        // ---- symbols: lane 0 decodes a batch, the group writes it ----
        int eob = 0;
        while (!eob) {
            int n = 0;
            if (lane == 0) {
                // queue entries: a literal keeps its table entry (byte in bits 8..15, bit 31 clear),
                // a match is 1<<31 | length << 16 | distance; offsets are validated by the group
                uint32_t bad = 0;
                while (n < S) {
                    const uint32_t bits = br.peek();
                    uint32_t e = g.lut[bits & ((1u << LB) - 1u)];
                    if ((e & 15u) == 0) {
                        int l = 0;
                        const int sym = slow_decode(bits, g.lcount, g.lsym, &l);
                        if (sym < 0) {
                            err = -13;
                            break;
                        }
                        e = lit_entry(sym, l);
                    }
                    const uint32_t l = e & 15u;
                    if (e < (1u << 28)) {                 // literal
                        br.skip(l);
                        g.queue[n++] = e;
                        continue;
                    }
                    if ((e >> 28) != KIND_LEN) {
                        if ((e >> 28) == KIND_EOB) {
                            br.skip(l);
                            eob = 1;
                        } else {
                            err = -14;
                        }
                        break;
                    }
                    const uint32_t ex = (e >> 4) & 15u;
                    const uint32_t len = ((e >> 8) & 0xffffu) + ((bits >> l) & ~(0xffffffffu << ex));
                    br.skip(l + ex);
                    const uint32_t dbits = br.peek();
                    uint32_t de = g.dlut[dbits & ((1u << DB) - 1u)];
                    if ((de & 15u) == 0) {
                        int dl = 0;
                        const int sym = slow_decode(dbits, g.dcount, g.dsym, &dl);
                        if (sym < 0) {
                            err = -15;
                            break;
                        }
                        de = dist_entry(sym, dl);
                    }
                    bad |= de >> 28;
                    const uint32_t dl = de & 15u, dx = (de >> 4) & 15u;
                    const uint32_t d = ((de >> 8) & 0xffffu) + ((dbits >> dl) & ~(0xffffffffu << dx));
                    br.skip(dl + dx);
                    g.queue[n++] = 0x80000000u | (len << 16) | d;
                }
                if (bad) err = -15;
                if ((const uint8_t *)br.wp > in_end + 16) err = -20;
            }
            __syncwarp(gmask);
            err = __shfl_sync(gmask, err, 0, S);
            if (err) return err;
            n = __shfl_sync(gmask, n, 0, S);
            eob = __shfl_sync(gmask, eob, 0, S);
            const uint32_t q = (int)lane < n ? g.queue[lane] : 0u;
            const bool is_match = (q >> 31) != 0;
            const uint32_t mylen = (int)lane < n ? (is_match ? ((q >> 16) & 0x1ffu) : 1u) : 0u;
            uint32_t incl = mylen;
#pragma unroll
            for (int dlt = 1; dlt < S; dlt <<= 1) {
                const uint32_t v = __shfl_up_sync(gmask, incl, dlt, S);
                if ((int)lane >= dlt) incl += v;
            }
            const uint32_t myoff = o + incl - mylen;
            const uint32_t total = __shfl_sync(gmask, incl, S - 1, S);
            // a distance reaching before the start of the output, or output past the block's size
            if (__any_sync(gmask, (is_match && (q & 0xffffu) > myoff) || o + total > cap)) return -16;
            uint32_t mm;
            if constexpr (S == 32) {
                // Every output byte of the batch is produced by the lane at its position: 32 bytes per
                // round, the owning symbol found from a bitmap of the symbols' start offsets.  A match
                // that reads bytes of this very batch (distance shorter than its offset into the batch)
                // is left to the ordered loop below; BAM matches mostly reach back whole records.
                const bool valid = (int)lane < n;
                const uint32_t d_i = q & 0xffffu;
                const bool dep_i = valid && is_match && (myoff - d_i + min(mylen, d_i) > o);
                const uint32_t offv = valid ? myoff : 0xffffffffu;
                const uint32_t end = o + total;
                for (uint32_t base = o; base < end; base += 32) {
                    const uint32_t sym_before = __popc(__ballot_sync(0xffffffffu, offv < base));
                    const uint32_t rel = offv - base;
                    const uint32_t starts = __reduce_or_sync(0xffffffffu, rel < 32u ? (1u << rel) : 0u);
                    const uint32_t p = base + lane;
                    const int idx = (int)(sym_before + __popc(starts & (0xffffffffu >> (31 - lane)))) - 1;
                    const uint32_t sq = __shfl_sync(0xffffffffu, q, idx), soff = __shfl_sync(0xffffffffu, myoff, idx);
                    if (p < end) {
                        if (sq >> 31) {
                            const uint32_t d = sq & 0xffffu, len = (sq >> 16) & 0x1ffu;
                            if (soff - d + min(len, d) <= o) out[p] = out[d >= len ? p - d : soff - d + ((p - soff) % d)];
                        } else {
                            out[p] = (uint8_t)(sq >> 8);
                        }
                    }
                }
                mm = __ballot_sync(0xffffffffu, dep_i);
            } else {
                if ((int)lane < n && !is_match) out[myoff] = (uint8_t)(q >> 8);
                mm = (__ballot_sync(gmask, is_match) >> gbase) & ((1u << S) - 1u);
            }
            if (mm) {
                __syncwarp(gmask);
                while (mm) {
                    const int src = __ffs((int)mm) - 1;
                    mm &= mm - 1;
                    const uint32_t len = __shfl_sync(gmask, mylen, src, S);
                    const uint32_t d = __shfl_sync(gmask, q & 0xffffu, src, S);
                    const uint32_t dst = __shfl_sync(gmask, myoff, src, S);
                    if (d >= len) {
                        for (uint32_t k = lane; k < len; k += S) out[dst + k] = out[dst - d + k];
                    } else {
                        for (uint32_t k = lane; k < len; k += S) out[dst + k] = out[dst - d + (k % d)];
                    }
                    __syncwarp(gmask);
                }
            }
            o += total;
            __syncwarp(gmask);
        }
    }
    return (int)o;
}

// ---- CRC32 of the inflated block (gzip trailer check, as htslib does) -------------------------
// Lane-parallel: every lane takes 1/32 of the block through the byte-wise table algorithm, the 32
// CRCs are combined with crc(A||B) = crc(A) * x^(8|B|) mod P  xor  crc(B) (reflected polynomial
// 0xEDB88320, the arithmetic zlib's crc32_combine uses).
constexpr unsigned int CRC_POLY = 0xedb88320u;

__device__ __forceinline__ unsigned int crc_multmodp(unsigned int a, unsigned int b) {
    unsigned int m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = (b & 1u) ? (b >> 1) ^ CRC_POLY : b >> 1;
    }
    return p;
}

// x^(8 n) mod P
__device__ __forceinline__ unsigned int crc_x8n(unsigned int n) {
    unsigned int p = 1u << 31;               // x^0
    unsigned int sq = 1u << 23;              // x^8
    while (n) {
        if (n & 1u) p = crc_multmodp(sq, p);
        n >>= 1;
        if (n) sq = crc_multmodp(sq, sq);
    }
    return p;
}

// table[i] for the byte-wise update; every warp builds its own copy (in its idle Huffman table)
__device__ __forceinline__ void crc_build_table(unsigned int *table) {
    for (unsigned int i = threadIdx.x & 31u; i < 256; i += 32) {
        unsigned int c = i;
        for (int k = 0; k < 8; k++) c = (c & 1u) ? (c >> 1) ^ CRC_POLY : c >> 1;
        table[i] = c;
    }
}

#ifdef __CUDACC__
// CRC32 of out[0, n) by one warp (all lanes call; the result is uniform).
__device__ __forceinline__ unsigned int crc32_warp(const unsigned int *table, const uint8_t *out, unsigned int n) {
    const unsigned int lane = threadIdx.x & 31u;
    const unsigned int chunk = (n + 31u) / 32u;
    const unsigned int beg = min(n, lane * chunk), end = min(n, beg + chunk);
    unsigned int c = 0xffffffffu;
    {
        // 16-byte loads over the aligned body of the chunk (a byte load per step would make the
        // 32 lanes' strided accesses the bottleneck), single bytes at its ragged ends
        const uint8_t *p = out + beg, *pe = out + end;
        while (p < pe && ((uintptr_t)p & 15)) c = table[(c ^ *p++) & 0xffu] ^ (c >> 8);
        for (; p + 16 <= pe; p += 16) {
            const uint4 v = *reinterpret_cast<const uint4 *>(p);
            const unsigned int w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int j = 0; j < 4; j++) {
                c ^= w[j];
#pragma unroll
                for (int b = 0; b < 4; b++) c = table[c & 0xffu] ^ (c >> 8);
            }
        }
        while (p < pe) c = table[(c ^ *p++) & 0xffu] ^ (c >> 8);
    }
    c ^= 0xffffffffu;                         // the CRC of this lane's chunk (of the empty string: 0)
    // crc(A|B|C) = crc(A) x^(8(|B|+|C|)) + crc(B) x^(8|C|) + crc(C): every lane shifts its own CRC
    // past the bytes that follow its chunk, the terms are xor-ed together
    const unsigned int term = end > beg ? crc_multmodp(crc_x8n(n - end), c) : 0u;
    const unsigned int total = __reduce_xor_sync(0xffffffffu, term);
    return total;
}
#endif

}  // namespace xg_inflate
