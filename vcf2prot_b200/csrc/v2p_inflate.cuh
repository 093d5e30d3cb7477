// v2p_inflate.cuh -- BGZF blocks -> text on the device (v2p_vcf_load_bgzf in v2p_vcf.cu; the format is stated in
// include/v2p_vcf.h).  The host walks the block headers and hands k_inflate a table of blocks; the kernel inflates them.
//
// k_inflate: one warp per BGZF block, the grid sized to the resident warps, blocks taken in a grid stride.  A block's
// DEFLATE stream is serial, so one lane (lane 0) reads the bits; the other 31 work on everything that is not serial:
//   tables   each Huffman code is built warp-parallel in shared memory: a primary table on the first kLitBits /
//            kDistBits bits, and for the rare longer codes the canonical (count, sorted symbol) form, walked a bit at a
//            time.  Over-subscribed / incomplete sets are refused as zlib's inftrees.c refuses them.
//   tokens   lane 0 decodes up to kRing symbols into a shared ring: literals and (length, distance) pairs, each with
//            its output offset.  The warp then writes every literal of the batch (a byte per lane), and copies the
//            matches in order, 32 bytes a step: a distance d >= 32 reads 32 bytes written before the step; d < 32 reads
//            the d bytes in front of the match once and writes the period out[p + i] = out[p - d + (i mod d)] from
//            registers.  Match sources are bytes this warp wrote, so they are read with plain loads (never .nc).
//   stored   a stored block is copied a byte per lane.
//   CRC-32   each lane takes a 1/32 slice of the block's output; the slices combine with gf_mul (v2p_crc32.cuh).
// No write leaves [out_off, out_off + isize) whatever the stream says: writes past ISIZE are dropped, and the decode
// goes on to the end of the stream so that a DEFLATE error past ISIZE still ranks above the size error.
// The first bad block, (block << 3) | class, is published with a 64-bit atomicMin, so the lowest block wins whatever
// the warp timing.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "v2p_crc32.cuh"

namespace {

struct BgzfBlock {     // one BGZF member, from the host's header walk
    uint64_t c_off;    // first byte of its raw DEFLATE data in the compressed buffer
    uint64_t out_off;  // first byte of its text: exclusive sum of ISIZE
    uint32_t c_len;    // bytes of DEFLATE data (BSIZE + 1 - header - trailer)
    uint32_t isize;
    uint32_t crc;
    uint32_t pad;
};
static_assert(sizeof(BgzfBlock) == 32, "block table entries are 32 bytes");

enum { BGZF_HEADER = 1, BGZF_DEFLATE = 2, BGZF_SIZE = 3, BGZF_CRC = 4 };  // precedence within one block

constexpr int kInfWarps = 8;  // warps per CTA
constexpr int kLitBits = 10, kDistBits = 8, kClBits = 7;
constexpr int kRing = 64;
constexpr uint32_t kMatch = 0x80000000u;  // token: literal = byte, match = kMatch | len | dist << 9

__constant__ uint16_t c_len_base[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31,
                                        35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t c_len_extra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint16_t c_dist_base[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769,
                                         1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
__constant__ uint8_t c_dist_extra[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
__constant__ uint8_t c_cl_perm[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

struct InflateSmem {             // one warp's tables and token ring: 4 KiB
    uint16_t lit[1 << kLitBits];   // primary tables: symbol | length << 9; 0 = longer code or no code
    uint16_t dist[1 << kDistBits]; // also the code-length code's table while a dynamic header is read
    uint16_t lsym[288], dsym[32];  // symbols sorted by (length, value)
    uint16_t lcount[16], dcount[16];
    uint32_t next[16], cmo[16];    // build scratch: next free slot per length, canonical code - slot per length
    uint32_t tpos[kRing], tval[kRing];
    uint8_t lens[320];             // HLIT + HDIST code lengths
    uint8_t cll[20];               // code-length code lengths
};

// Lane 0's view of the DEFLATE data.  Bytes past c_len read as zero; over() tells when the stream used them.
struct BitReader {
    const uint8_t* __restrict__ in;
    uint32_t clen, bp;  // bp: next byte to load
    uint64_t buf;
    int nb;             // valid bits in buf
    __device__ __forceinline__ void refill() {
        if (nb > 56) return;
        const int take = (64 - nb) >> 3;
        uint64_t w = 0;
        if (bp + 8 <= clen) {
#pragma unroll
            for (int k = 0; k < 8; ++k) w |= (uint64_t)in[bp + k] << (8 * k);
        } else {
            for (int k = 0; k < take; ++k) w |= (uint64_t)(bp + k < clen ? in[bp + k] : 0u) << (8 * k);
        }
        buf |= w << nb;
        bp += take, nb += 8 * take;
        if (nb < 64) buf &= (1ull << nb) - 1;
    }
    __device__ __forceinline__ uint32_t get(int n) {  // n <= 32
        if (nb < n) refill();
        const uint32_t v = (uint32_t)(buf & ((1ull << n) - 1));
        buf >>= n, nb -= n;
        return v;
    }
    __device__ __forceinline__ void drop(int n) { buf >>= n, nb -= n; }
    __device__ __forceinline__ bool over() const { return (uint64_t)bp * 8 - (uint64_t)nb > (uint64_t)clen * 8; }
};

// Huffman code from lens[0, n) into a primary table of `bits` bits plus count / sorted symbols.  Warp-wide; lens must be
// visible to every lane on entry (the caller's __syncwarp), the tables are on return.  Returns false for a set zlib
// refuses: over-subscribed, or incomplete unless it is a lit/len or distance set whose longest code has length 1; an
// empty set is accepted except for the code-length code (a code from it is then an invalid code).
__device__ bool build_code(const uint8_t* lens, int n, int bits, uint16_t* tab, uint16_t* count, uint16_t* sym, bool cl_code,
                           InflateSmem& s, uint32_t lane) {
    if (lane < 16) s.next[lane] = 0;
    for (int e = lane; e < (1 << bits); e += 32) tab[e] = 0;
    __syncwarp();
    for (int i = lane; i < n; i += 32)
        if (lens[i]) atomicAdd(&s.next[lens[i]], 1u);
    __syncwarp();
    int ok = 1;
    if (lane == 0) {
        int left = 1, max = 0;
        uint32_t slot = 0, code = 0;
        for (int l = 1; l < 16; ++l) {
            const uint32_t c = s.next[l];
            left = (left << 1) - (int)c;
            if (left < 0) ok = 0;
            if (c) max = l;
            count[l] = (uint16_t)c;
            s.cmo[l] = code - slot;  // canonical code of the slot-th symbol of length l = slot + cmo[l]
            s.next[l] = slot;
            slot += c, code = (code + c) << 1;
        }
        count[0] = 0;
        if (max == 0 && cl_code) ok = 0;
        if (left > 0 && max > 0 && (cl_code || max != 1)) ok = 0;
    }
    ok = __shfl_sync(0xffffffffu, ok, 0);
    __syncwarp();
    if (!ok) return false;
    for (int base = 0; base < n; base += 32) {
        const int i = base + (int)lane;
        const uint32_t l = i < n ? lens[i] : 0u;
        const uint32_t peers = __match_any_sync(0xffffffffu, l);
        const uint32_t rank = __popc(peers & ((1u << lane) - 1));
        if (l) {
            const uint32_t slot = s.next[l] + rank;
            sym[slot] = (uint16_t)i;
            if ((int)l <= bits) {
                const uint32_t rev = __brev(slot + s.cmo[l]) >> (32 - l);
                const uint16_t ent = (uint16_t)(i | (l << 9));
                for (uint32_t e = rev; e < (1u << bits); e += 1u << l) tab[e] = ent;
            }
        }
        __syncwarp();
        if (l && rank == 0) s.next[l] += __popc(peers);
        __syncwarp();
    }
    return true;
}

// Lane 0: next symbol of the code (>= 15 bits in the reader), -1 for a bit pattern that is no code.
__device__ __forceinline__ int decode_sym(BitReader& br, const uint16_t* tab, int bits, const uint16_t* count, const uint16_t* sym) {
    const uint32_t e = tab[br.buf & ((1u << bits) - 1)];
    if (e) {
        br.drop(e >> 9);
        return (int)(e & 511u);
    }
    int code = 0, first = 0, index = 0;
    for (int l = 1; l < 16; ++l) {
        code |= (int)((br.buf >> (l - 1)) & 1u);
        const int c = count[l];
        if (code - c < first) {
            br.drop(l);
            return sym[index + (code - first)];
        }
        index += c, first = (first + c) << 1, code <<= 1;
    }
    return -1;
}

// out[p, p + len) = the match at distance d (1 <= d <= p), dropped past isize.  Warp-wide.
__device__ __forceinline__ void copy_match(uint8_t* out, uint32_t isize, uint32_t p, uint32_t len, uint32_t d, uint32_t lane) {
    if (p >= isize) return;
    const uint32_t end = min(p + len, isize);
    if (d >= 32) {
        for (uint32_t q = p; q < end; q += 32) {
            const uint32_t i = q + lane;
            if (i < end) out[i] = out[i - d];
            __syncwarp();
        }
    } else {
        const uint32_t pat = lane < d ? out[p - d + lane] : 0u;
        uint32_t off = lane % d;
        const uint32_t step = 32 % d;
        for (uint32_t q = p; q < end; q += 32) {
            const uint32_t b = __shfl_sync(0xffffffffu, pat, off);
            if (q + lane < end) out[q + lane] = (uint8_t)b;
            off += step;
            if (off >= d) off -= d;
        }
        __syncwarp();
    }
}

// One BGZF block's DEFLATE data -> out[0, isize).  Warp-wide; returns 0, BGZF_DEFLATE or BGZF_SIZE.
__device__ int inflate_block(const uint8_t* __restrict__ in, uint32_t clen, uint8_t* out, uint32_t isize, InflateSmem& s,
                             uint32_t lane) {
    const unsigned FULL = 0xffffffffu;
    BitReader br{in, clen, 0, 0, 0};
    uint32_t pos = 0;  // bytes produced (lane 0's count, broadcast where the warp needs it)
    bool last = false;
    int fixed = 0;     // the tables hold the fixed code
    while (!last) {
        int hdr = 0;
        if (lane == 0) {
            br.refill();
            hdr = (int)br.get(3);
        }
        hdr = __shfl_sync(FULL, hdr, 0);
        last = hdr & 1;
        const int type = hdr >> 1;
        if (type == 3) return BGZF_DEFLATE;
        if (type == 0) {  // stored: LEN, NLEN on the next byte boundary, then LEN bytes
            uint32_t src = 0, len = 0;
            int bad = 0;
            if (lane == 0) {
                br.drop(br.nb & 7);
                br.bp -= (uint32_t)(br.nb >> 3);
                br.buf = 0, br.nb = 0;
                if (br.bp + 4 > clen) {
                    bad = 1;
                } else {
                    len = in[br.bp] | (uint32_t)in[br.bp + 1] << 8;
                    const uint32_t nlen = in[br.bp + 2] | (uint32_t)in[br.bp + 3] << 8;
                    src = br.bp + 4;
                    bad = (len != (~nlen & 0xffffu)) || src + len > clen;
                    br.bp = src + len;
                }
            }
            bad = __shfl_sync(FULL, bad, 0);
            if (bad) return BGZF_DEFLATE;
            src = __shfl_sync(FULL, src, 0), len = __shfl_sync(FULL, len, 0), pos = __shfl_sync(FULL, pos, 0);
            for (uint32_t i = lane; i < len; i += 32)
                if (pos + i < isize) out[pos + i] = in[src + i];
            pos += len;
            __syncwarp();
            continue;
        }
        if (type == 1) {
            if (!fixed) {
                for (int i = lane; i < 320; i += 32) s.lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : i < 288 ? 8 : 5;
                __syncwarp();
                build_code(s.lens, 288, kLitBits, s.lit, s.lcount, s.lsym, false, s, lane);
                build_code(s.lens + 288, 32, kDistBits, s.dist, s.dcount, s.dsym, false, s, lane);
                fixed = 1;
            }
        } else {  // dynamic: HLIT, HDIST, HCLEN, the code-length code, then the code lengths it codes
            fixed = 0;
            int bad = 0, hlit = 0, hdist = 0;
            if (lane == 0) {
                br.refill();
                hlit = (int)br.get(5) + 257, hdist = (int)br.get(5) + 1;
                const int hclen = (int)br.get(4) + 4;
                bad = hlit > 286 || hdist > 30;
                for (int i = 0; i < 19; ++i) s.cll[i] = 0;
                for (int i = 0; i < hclen; ++i) s.cll[c_cl_perm[i]] = (uint8_t)br.get(3);
            }
            bad = __shfl_sync(FULL, bad, 0);
            if (bad) return BGZF_DEFLATE;
            __syncwarp();
            if (!build_code(s.cll, 19, kClBits, s.dist, s.dcount, s.dsym, true, s, lane)) return BGZF_DEFLATE;
            if (lane == 0) {
                const int n = hlit + hdist;
                for (int i = 0; i < n && !bad;) {
                    if (br.nb < 16) br.refill();
                    const int sym = decode_sym(br, s.dist, kClBits, s.dcount, s.dsym);
                    int rep = 0;
                    uint8_t val = 0;
                    if (sym < 0) {
                        bad = 1;
                    } else if (sym < 16) {
                        rep = 1, val = (uint8_t)sym;
                    } else if (sym == 16) {
                        if (i == 0) bad = 1;
                        else rep = 3 + (int)br.get(2), val = s.lens[i - 1];
                    } else {
                        rep = sym == 17 ? 3 + (int)br.get(3) : 11 + (int)br.get(7);
                    }
                    if (i + rep > n) bad = 1;
                    for (int k = 0; k < rep && !bad; ++k) s.lens[i++] = val;
                    if (br.over()) bad = 1;
                }
                if (!bad && s.lens[256] == 0) bad = 1;
            }
            hlit = __shfl_sync(FULL, hlit, 0), hdist = __shfl_sync(FULL, hdist, 0);
            bad = __shfl_sync(FULL, bad, 0);
            __syncwarp();
            if (bad) return BGZF_DEFLATE;
            if (!build_code(s.lens, hlit, kLitBits, s.lit, s.lcount, s.lsym, false, s, lane)) return BGZF_DEFLATE;
            if (!build_code(s.lens + hlit, hdist, kDistBits, s.dist, s.dcount, s.dsym, false, s, lane)) return BGZF_DEFLATE;
        }
        // symbols until the end of the block, kRing tokens a batch
        for (;;) {
            int ntok = 0, state = 0;  // state: 0 ring full, 1 end of block, 2 invalid stream
            if (lane == 0) {
                while (ntok < kRing) {
                    br.refill();  // >= 57 bits: a length and a distance with their extra bits take at most 48
                    if (br.over()) {
                        state = 2;
                        break;
                    }
                    const int sym = decode_sym(br, s.lit, kLitBits, s.lcount, s.lsym);
                    if (sym < 256) {
                        if (sym < 0) {
                            state = 2;
                            break;
                        }
                        s.tpos[ntok] = pos, s.tval[ntok] = (uint32_t)sym;
                        ++ntok, ++pos;
                        continue;
                    }
                    if (sym == 256) {
                        state = br.over() ? 2 : 1;
                        break;
                    }
                    if (sym > 285) {
                        state = 2;
                        break;
                    }
                    const uint32_t len = c_len_base[sym - 257] + br.get(c_len_extra[sym - 257]);
                    const int ds = decode_sym(br, s.dist, kDistBits, s.dcount, s.dsym);
                    if (ds < 0 || ds > 29) {
                        state = 2;
                        break;
                    }
                    const uint32_t dist = c_dist_base[ds] + br.get(c_dist_extra[ds]);
                    if (dist > pos) {  // before the start of the block: blocks are independent
                        state = 2;
                        break;
                    }
                    s.tpos[ntok] = pos, s.tval[ntok] = kMatch | len | dist << 9;
                    ++ntok, pos += len;
                }
            }
            ntok = __shfl_sync(FULL, ntok, 0), state = __shfl_sync(FULL, state, 0);
            if (state == 2) return BGZF_DEFLATE;
            __syncwarp();
            for (int t = lane; t < ntok; t += 32) {
                const uint32_t v = s.tval[t], p = s.tpos[t];
                if (!(v & kMatch) && p < isize) out[p] = (uint8_t)v;
            }
            __syncwarp();
            for (int base = 0; base < ntok; base += 32) {
                const int t = base + (int)lane;
                for (uint32_t m = __ballot_sync(FULL, t < ntok && (s.tval[t] & kMatch)); m; m &= m - 1) {
                    const int k = base + __ffs(m) - 1;
                    const uint32_t v = s.tval[k];
                    copy_match(out, isize, s.tpos[k], v & 511u, (v >> 9) & 0xffffu, lane);
                }
            }
            __syncwarp();
            if (state == 1) break;
        }
    }
    pos = __shfl_sync(FULL, pos, 0);
    return pos == isize ? 0 : BGZF_SIZE;
}

// CRC-32 of out[0, n), a slice per lane combined in GF(2).  Warp-wide; the result is in every lane.
__device__ uint32_t warp_crc32(const uint8_t* out, uint32_t n, const uint32_t (*tab)[256], uint32_t lane) {
    const uint32_t per = ((n + 31) / 32 + 3) & ~3u;
    const uint32_t lo = min(lane * per, n), hi = min(lo + per, n);
    uint32_t crc = 0xFFFFFFFFu, p = lo;
    for (; p < hi && ((uintptr_t)(out + p) & 3); ++p) crc = tab[0][(crc ^ out[p]) & 255u] ^ (crc >> 8);
    for (; p + 4 <= hi; p += 4) {
        crc ^= *reinterpret_cast<const uint32_t*>(out + p);
        crc = tab[3][crc & 255u] ^ tab[2][(crc >> 8) & 255u] ^ tab[1][(crc >> 16) & 255u] ^ tab[0][crc >> 24];
    }
    for (; p < hi; ++p) crc = tab[0][(crc ^ out[p]) & 255u] ^ (crc >> 8);
    crc = ~crc;
    uint32_t part = gf_mul(x_pow_8n(n - hi), crc);  // moved past the slices after this one (an empty slice's CRC is 0)
#pragma unroll
    for (int d = 16; d; d >>= 1) part ^= __shfl_xor_sync(0xffffffffu, part, d);
    return part;
}

// `text` is written here and read back (matches, CRC): no const / __restrict__, so no non-coherent loads.
__global__ void __launch_bounds__(kInfWarps * 32) k_inflate(const uint8_t* __restrict__ comp, const BgzfBlock* __restrict__ blk,
                                                            uint64_t n_blk, uint8_t* text, unsigned long long* err) {
    __shared__ uint32_t s_tab[4][256];
    __shared__ InflateSmem s_w[kInfWarps];
    for (int i = threadIdx.x; i < 4 * 256; i += blockDim.x) s_tab[i >> 8][i & 255] = g_crc_tab[i >> 8][i & 255];
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31;
    InflateSmem& s = s_w[threadIdx.x >> 5];
    const uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * (uint64_t)blockDim.x) >> 5;
    for (uint64_t b = warp; b < n_blk; b += n_warps) {
        const BgzfBlock B = blk[b];
        uint8_t* out = text + B.out_off;
        int cls = inflate_block(comp + B.c_off, B.c_len, out, B.isize, s, lane);
        if (!cls && warp_crc32(out, B.isize, s_tab, lane) != B.crc) cls = BGZF_CRC;
        if (cls && lane == 0) atomicMin(err, (unsigned long long)(b << 3 | (uint64_t)cls));
        __syncwarp();
    }
}

}  // namespace
