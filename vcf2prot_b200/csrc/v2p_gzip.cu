// v2p_gzip.cu -- gzip file images on the device (include/v2p_gzip.h; SURVEY 8f rank 4).
//
// Replaces GzEncoder::new(file, Compression::best()) of personalized_genome.rs:87-101 / :135-170 for the FASTA image
// the engine leaves in HBM.  Two streaming passes over the input, one CTA per 16 KiB chunk:
//   k_gz_plan    histogram -> length-limited Huffman code lengths -> exact compressed size; CRC-32 of the chunk
//   (CUB scan)   chunk sizes (+ the file's header / trailer bytes) -> output offsets
//   k_gz_files   per file: CRC-32 of the file from the chunk CRCs (GF(2) algebra), header and trailer
//   k_gz_encode  canonical codes from the saved lengths, bits packed in shared memory, stored to the final offset
// The format decisions (tie-breaks, header run-length rules, stored fallback) are stated once more, in Python, in
// oracle/gzip_twin.py; the GPU tests compare the two byte for byte and inflate the result with zlib.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cub/device/device_scan.cuh>
#include <new>
#include <string>
#include <vector>

#include "v2p_crc32.cuh"
#include "v2p_gzip.h"
#include "v2p_mapped.cuh"

namespace {

constexpr int CH = V2P_GZIP_CHUNK;
constexpr int NT = 256;
constexpr int PIECE = CH / NT;  // bytes of a chunk one thread owns
constexpr int LENS_STRIDE = 272;  // 257 code lengths, [260] = 1 when the chunk is a stored block
static_assert(PIECE == 64, "piece = 16 words");

// code-length alphabet: fixed complete code, thirteen 4-bit + six 5-bit symbols; codes are canonical, bit-reversed
__constant__ uint8_t c_cl_len[19] = {4, 5, 5, 5, 4, 4, 4, 4, 4, 4, 4, 4, 4, 5, 5, 5, 4, 4, 4};
__constant__ uint8_t c_cl_code[19] = {0, 11, 27, 7, 8, 4, 12, 2, 10, 6, 14, 1, 9, 23, 15, 31, 5, 13, 3};
__constant__ uint8_t c_cl_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

struct GzArgs {
    const uint8_t* in;        // base such that file bytes are in[file_begin[f] ..)
    uint64_t in_lo, in_hi;    // valid byte range of `in` (for the vector loads)
    const uint64_t* file_begin;
    const uint64_t* chunk_first;
    uint64_t n_files, n_chunks;
    uint8_t* lens;
    uint64_t* csize;          // pass 1 out: bytes the chunk (and the file framing it carries) occupies
    uint32_t* ccrc;
    const uint64_t* coff;     // scan of csize
    uint8_t* out;
    uint64_t* out_begin;      // device copy
    unsigned long long* n_stored;
};

struct ChunkPos {
    uint64_t file, idx, begin;
    uint32_t n, first, last;
};

__device__ __forceinline__ ChunkPos locate(const GzArgs& a, uint64_t c) {
    uint64_t lo = 0, hi = a.n_files;  // last f with chunk_first[f] <= c
    while (hi - lo > 1) {
        const uint64_t mid = (lo + hi) >> 1;
        if (a.chunk_first[mid] <= c) lo = mid;
        else hi = mid;
    }
    ChunkPos p;
    p.file = lo, p.idx = c - a.chunk_first[lo];
    const uint64_t fb = a.file_begin[lo], fe = a.file_begin[lo + 1];
    p.begin = fb + p.idx * CH;
    p.n = (uint32_t)min((uint64_t)CH, fe - min(fe, p.begin));
    p.first = p.idx == 0, p.last = c + 1 == a.chunk_first[lo + 1];
    return p;
}

// chunk bytes -> shared memory (chunk-relative), 16-byte global loads realigned with a funnel shift
__device__ __forceinline__ void load_chunk(uint32_t* s_in, const GzArgs& a, uint64_t begin, uint32_t n) {
    const uint8_t* src = a.in + begin;
    const uint32_t ph = (uint32_t)((uintptr_t)src & 15u);
    const uint4* base = reinterpret_cast<const uint4*>(src - ph);
    const uint8_t* lo = a.in + a.in_lo;
    const uint8_t* hi = a.in + a.in_hi;
    if (n == CH && src - ph >= lo && src + CH + 16 <= hi) {  // whole chunk inside the buffer: all loads in flight at once
        const uint32_t wsh = ph >> 2, bsh = (ph & 3u) * 8;
        uint4 x[CH / 16 / NT], y[CH / 16 / NT];
#pragma unroll
        for (int u = 0; u < CH / 16 / NT; ++u) {
            x[u] = __ldcs(base + threadIdx.x + u * NT);
            y[u] = __ldcs(base + threadIdx.x + u * NT + 1);
        }
#pragma unroll
        for (int u = 0; u < CH / 16 / NT; ++u) {
            const uint32_t q[8] = {x[u].x, x[u].y, x[u].z, x[u].w, y[u].x, y[u].y, y[u].z, y[u].w};
            uint32_t w[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                uint32_t a0 = 0, a1 = 0;
#pragma unroll
                for (int m = 0; m < 4; ++m)
                    if (wsh == (uint32_t)m) a0 = q[k + m], a1 = q[k + m + 1 < 8 ? k + m + 1 : 7];
                w[k] = __funnelshift_r(a0, a1, bsh);
            }
            *reinterpret_cast<uint4*>(s_in + (threadIdx.x + u * NT) * 4) = make_uint4(w[0], w[1], w[2], w[3]);
        }
        return;
    }
    for (uint32_t v = threadIdx.x; v * 16 < n; v += NT) {
        const uint8_t* g0 = reinterpret_cast<const uint8_t*>(base + v);
        uint32_t w[4];
        if (g0 >= lo && g0 + 32 <= hi) {
            const uint4 x = __ldcs(base + v), y = ph ? __ldcs(base + v + 1) : x;
            const uint32_t q[8] = {x.x, x.y, x.z, x.w, y.x, y.y, y.z, y.w};
            const uint32_t wsh = ph >> 2, bsh = (ph & 3u) * 8;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                uint32_t a0 = 0, a1 = 0;
#pragma unroll
                for (int m = 0; m < 4; ++m)  // select without dynamic register indexing
                    if (wsh == (uint32_t)m) a0 = q[k + m], a1 = q[k + m + 1 < 8 ? k + m + 1 : 7];
                w[k] = __funnelshift_r(a0, a1, bsh);
            }
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                uint32_t x = 0;
                for (int b = 0; b < 4; ++b) {
                    const uint32_t i = v * 16 + k * 4 + b;
                    if (i < n) x |= (uint32_t)src[i] << (8 * b);
                }
                w[k] = x;
            }
        }
        *reinterpret_cast<uint4*>(s_in + v * 4) = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

struct Tree {
    uint32_t w[2 * 257];
    uint16_t parent[2 * 257];
    uint16_t sym[260];
    uint32_t num[16];
    int n;
};

// Length-limited Huffman lengths, by one warp.  Leaves are sorted by (frequency, symbol); two-queue merge, leaf first
// on ties (lane 0, queue heads kept in registers); leaf depths by walking up, one leaf per lane; depths above 15 folded
// back by the Kraft-sum repair; the rarest symbols get the longest lengths.
__device__ void build_lengths(Tree& t, uint8_t* lens, int lane) {
    const int n = t.n;
    if (n == 1) {
        if (lane == 0) lens[t.sym[0]] = 1;
        return;
    }
    if (lane == 0) {
        constexpr uint32_t NONE = 0xFFFFFFFFu;
        int li = 0, ii = n;
        uint32_t wl = t.w[0], wl2 = n > 1 ? t.w[1] : NONE, wi = NONE;
        for (int k = n; k < 2 * n - 1; ++k) {
            uint32_t sum = 0;
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                if (li < n && (ii >= k || wl <= wi)) {
                    sum += wl;
                    t.parent[li++] = (uint16_t)k;
                    wl = wl2;
                    wl2 = li + 1 < n ? t.w[li + 1] : NONE;
                } else {
                    sum += wi;
                    t.parent[ii++] = (uint16_t)k;
                    wi = ii < k ? t.w[ii] : NONE;
                }
            }
            t.w[k] = sum;
            if (ii == k) wi = sum;  // the new node is the head of the (otherwise empty) internal queue
        }
    }
    if (lane < 16) t.num[lane] = 0;
    __syncwarp();
    const int root = 2 * n - 2;
    for (int i = lane; i < n; i += 32) {
        int d = 0;
        for (int k = i; k != root; k = t.parent[k]) ++d;
        atomicAdd(&t.num[min(d, 15)], 1u);
    }
    __syncwarp();
    if (lane == 0) {
        uint32_t total = 0;
        for (int l = 1; l <= 15; ++l) total += t.num[l] << (15 - l);
        while (total > (1u << 15)) {
            t.num[15]--;
            for (int l = 14; l >= 1; --l)
                if (t.num[l]) {
                    t.num[l]--;
                    t.num[l + 1] += 2;
                    break;
                }
            --total;
        }
    }
    __syncwarp();
    for (int i = lane; i < n; i += 32) {  // leaf i (ascending frequency): lengths are handed out longest first
        uint32_t acc = 0;
        int l = 15;
        for (; l > 1; --l) {
            acc += t.num[l];
            if ((uint32_t)i < acc) break;
        }
        lens[t.sym[i]] = (uint8_t)l;
    }
}

// ---- block header ---------------------------------------------------------------------------------------------------
// After the 3 block-type bits: HLIT=257, HDIST=1, HCLEN=19, the fixed code-length code (74 bits so far), then the code
// lengths as code-length symbols: the 256 byte values run-length coded -- one thread per run, so both the size and
// the bits come out of a block-wide scan instead of a serial walk -- then the end-of-block length and the single
// (unused, zero) distance length as two plain symbols.
constexpr uint32_t HDR_FIXED_BITS = 3 + 5 + 5 + 4 + 19 * 3;

struct BitSink {
    uint32_t* words;
    uint32_t pos;
    __device__ __forceinline__ void put(uint32_t v, uint32_t nbits) {
        const uint32_t w = pos >> 5, sh = pos & 31;
        const uint64_t x = (uint64_t)v << sh;
        atomicOr(&words[w], (uint32_t)x);
        if (sh + nbits > 32) atomicOr(&words[w + 1], (uint32_t)(x >> 32));
        pos += nbits;
    }
    __device__ __forceinline__ void cl(uint32_t s, uint32_t xv, uint32_t xb) {
        put(c_cl_code[s] | xv << c_cl_len[s], c_cl_len[s] + xb);
    }
};

__device__ __forceinline__ uint32_t run_bits(uint32_t v, uint32_t r) {
    if (v == 0) {
        const uint32_t k = r / 138, rem = r % 138;
        return k * (c_cl_len[18] + 7u) + (rem >= 11 ? c_cl_len[18] + 7u : rem >= 3 ? c_cl_len[17] + 3u : rem * c_cl_len[0]);
    }
    const uint32_t q = r - 1, k = q / 6, rem = q % 6, lv = c_cl_len[v];
    return lv + k * (c_cl_len[16] + 2u) + (rem >= 3 ? c_cl_len[16] + 2u : rem * lv);
}

__device__ void emit_run(BitSink& o, uint32_t v, uint32_t r) {
    if (v == 0) {
        while (r >= 11) {
            const uint32_t t = min(r, 138u);
            o.cl(18, t - 11, 7);
            r -= t;
        }
        if (r >= 3) {
            o.cl(17, r - 3, 3);
            r = 0;
        }
        for (; r > 0; --r) o.cl(0, 0, 0);
    } else {
        o.cl(v, 0, 0);
        --r;
        while (r >= 3) {
            const uint32_t t = min(r, 6u);
            o.cl(16, t - 3, 2);
            r -= t;
        }
        for (; r > 0; --r) o.cl(v, 0, 0);
    }
}

// thread t < 256 looks at byte value t: is it the first of a run of equal code lengths, and how long is the run.
// s_mask[8] must hold the ballots of `start` (one word per warp) and be visible (barrier) before the call.
__device__ __forceinline__ uint32_t run_length(const uint32_t* s_mask, int t) {
    int w = t >> 5;
    const int lane = t & 31;
    uint32_t m = lane == 31 ? 0u : s_mask[w] & (~0u << (lane + 1));
    while (!m && ++w < NT / 32) m = s_mask[w];
    return (m ? w * 32 + __ffs(m) - 1 : 256) - t;
}

// block-wide exclusive scan of one value per thread (NT threads); two barriers; *total = sum over the block
__device__ __forceinline__ uint32_t block_scan(uint32_t v, uint32_t* s_scan, uint32_t* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += o;
    }
    __syncthreads();  // s_scan free
    if (lane == 31) s_scan[warp] = incl;
    __syncthreads();
    uint32_t before = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < NT / 32; ++w) {
        const uint32_t x = s_scan[w];
        before += w < warp ? x : 0u;
        tot += x;
    }
    *total = tot;
    return before + incl - v;
}

// ---- pass 1 ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT, 6) k_gz_plan(GzArgs a) {
    __shared__ __align__(16) uint32_t s_in[CH / 4 + 8];
    __shared__ uint32_t s_hist[NT / 32][260];
    __shared__ uint32_t s_tab[4][256];
    __shared__ uint32_t s_used[260];
    __shared__ uint8_t s_lens[LENS_STRIDE];
    __shared__ Tree s_tree;
    __shared__ ChunkPos s_pos;
    __shared__ uint32_t s_red[NT / 32], s_mask[NT / 32], s_cnt[NT / 32], s_scan[NT / 32];
    __shared__ uint32_t s_last_crc;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    for (int k = 0; k < 4; ++k) s_tab[k][t] = g_crc_tab[k][t];

    for (uint64_t c = blockIdx.x; c < a.n_chunks; c += gridDim.x) {
        __syncthreads();  // previous iteration done with shared memory
        if (t == 0) s_pos = locate(a, c);
        for (int i = t; i < (NT / 32) * 260; i += NT) (&s_hist[0][0])[i] = 0;
        for (int i = t; i < LENS_STRIDE; i += NT) s_lens[i] = 0;
        __syncthreads();
        const ChunkPos p = s_pos;
        const uint64_t framing = (p.first ? 10 : 0) + (p.last ? 10 : 0);
        if (p.n == 0) {  // an empty file: framing only
            if (t == 0) a.csize[c] = framing, a.ccrc[c] = 0;
            for (int i = t; i < LENS_STRIDE; i += NT) a.lens[c * LENS_STRIDE + i] = 0;
            continue;
        }
        load_chunk(s_in, a, p.begin, p.n);
        __syncthreads();

        // my piece: histogram + CRC-32; the chunk CRC is  x^(8m) * XOR_t x^(8*64*(np-2-t)) * crc_t  ^  crc_last
        // (np pieces, the last one m bytes long): one GF(2) multiplication per thread
        const int np = (int)(p.n + PIECE - 1) / PIECE, my = max(0, min(PIECE, (int)p.n - t * PIECE));
        uint32_t crc = 0xFFFFFFFFu;
        uint32_t* hist = s_hist[warp];
        if (my == PIECE) {  // whole piece: 16-byte shared loads, four bytes of CRC per step
            const uint4* pv = reinterpret_cast<const uint4*>(s_in + t * (PIECE / 4));
#pragma unroll
            for (int q = 0; q < PIECE / 16; ++q) {
                const uint4 v = pv[q];
                const uint32_t wds[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint32_t wd = wds[k];
                    atomicAdd(&hist[wd & 255u], 1u);
                    atomicAdd(&hist[(wd >> 8) & 255u], 1u);
                    atomicAdd(&hist[(wd >> 16) & 255u], 1u);
                    atomicAdd(&hist[wd >> 24], 1u);
                    crc ^= wd;
                    crc = s_tab[3][crc & 255u] ^ s_tab[2][(crc >> 8) & 255u] ^ s_tab[1][(crc >> 16) & 255u] ^ s_tab[0][crc >> 24];
                }
            }
        } else {
            for (int k = 0; k * 4 < my; ++k) {
                uint32_t wd = s_in[t * (PIECE / 4) + k];
                const int nb = min(4, my - k * 4);
                for (int b = 0; b < nb; ++b, wd >>= 8) {
                    const uint32_t byte = wd & 255u;
                    atomicAdd(&hist[byte], 1u);
                    crc = s_tab[0][(crc ^ byte) & 255u] ^ (crc >> 8);
                }
            }
        }
        crc = ~crc;
        uint32_t part = t < np - 1 ? gf_mul(g_x64[np - 2 - t], crc) : 0u;
        if (t == np - 1) s_last_crc = crc;
#pragma unroll
        for (int d = 16; d; d >>= 1) part ^= __shfl_xor_sync(0xffffffffu, part, d);
        if (lane == 0) s_red[warp] = part;
        __syncthreads();

        // frequencies; the used symbols compacted (symbol 256, end of block, occurs once and goes last)
        uint32_t f = 0;
#pragma unroll
        for (int w = 0; w < NT / 32; ++w) f += s_hist[w][t];
        const uint32_t key = f << 9 | (uint32_t)t;  // sort key (frequency, symbol)
        const uint32_t um = __ballot_sync(0xffffffffu, f != 0);
        if (lane == 0) s_cnt[warp] = __popc(um);
        __syncthreads();
        int n_used = 1, at = 0;
#pragma unroll
        for (int w = 0; w < NT / 32; ++w) {
            const int x = (int)s_cnt[w];
            at += w < warp ? x : 0;
            n_used += x;
        }
        if (f) s_used[at + __popc(um & ((1u << lane) - 1u))] = key;
        if (t == 0) s_used[n_used - 1] = 1u << 9 | 256u;
        __syncthreads();
        {  // rank among the used symbols = position in the sorted leaf list
            const uint32_t eob = 1u << 9 | 256u;
            int rank = 0, rank_eob = 0;
            for (int j = 0; j < n_used; ++j) {
                const uint32_t k = s_used[j];
                rank += k < key;
                rank_eob += k < eob;
            }
            if (f) s_tree.sym[rank] = (uint16_t)t, s_tree.w[rank] = f;
            if (t == 0) s_tree.sym[rank_eob] = 256, s_tree.w[rank_eob] = 1, s_tree.n = n_used;
        }
        __syncthreads();
        if (warp == 0) build_lengths(s_tree, s_lens, lane);
        if (t == 32) {
            uint32_t c32 = 0;
#pragma unroll
            for (int w = 0; w < NT / 32; ++w) c32 ^= s_red[w];
            const uint32_t m = p.n - (uint32_t)(np - 1) * PIECE;
            a.ccrc[c] = gf_mul(g_xb[m], c32) ^ s_last_crc;
        }
        __syncthreads();
        // header bits (one thread per run of equal lengths) + payload bits, reduced over the block
        const uint32_t mylen = s_lens[t];
        const bool start = t == 0 || s_lens[t - 1] != mylen;
        const uint32_t sm = __ballot_sync(0xffffffffu, start);
        if (lane == 0) s_mask[warp] = sm;
        __syncthreads();
        uint32_t bits = f * mylen + (start ? run_bits(mylen, run_length(s_mask, t)) : 0u);
#pragma unroll
        for (int d = 16; d; d >>= 1) bits += __shfl_xor_sync(0xffffffffu, bits, d);
        if (lane == 0) s_scan[warp] = bits;
        __syncthreads();
        if (t == 0) {
            uint32_t tot = HDR_FIXED_BITS + c_cl_len[s_lens[256]] + c_cl_len[0] + s_lens[256];
#pragma unroll
            for (int w = 0; w < NT / 32; ++w) tot += s_scan[w];
            const uint32_t dyn = (tot + 3 + 7) / 8 + 4;  // + empty stored block header, aligned, 00 00 FF FF
            const bool stored = dyn >= p.n + 5;
            s_lens[260] = stored;
            a.csize[c] = (stored ? p.n + 5 : dyn) + framing;
            if (stored) atomicAdd(a.n_stored, 1ull);
        }
        __syncthreads();
        for (int i = t; i < LENS_STRIDE; i += NT) a.lens[c * LENS_STRIDE + i] = s_lens[i];
    }
}

// ---- per file: CRC of the whole file, gzip header and trailer --------------------------------------------------------
__global__ void __launch_bounds__(128) k_gz_files(GzArgs a) {
    const uint64_t f = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f > a.n_files) return;
    if (f == a.n_files) {
        a.out_begin[f] = a.coff[a.n_chunks];
        return;
    }
    const uint64_t c0 = a.chunk_first[f], c1 = a.chunk_first[f + 1];
    const uint64_t flen = a.file_begin[f + 1] - a.file_begin[f];
    const uint32_t full = x_pow_8n(CH);
    uint32_t crc = 0;
    for (uint64_t c = c0; c < c1; ++c) {
        const uint64_t n = min((uint64_t)CH, flen - (c - c0) * CH);
        crc = gf_mul(n == CH ? full : x_pow_8n(n), crc) ^ a.ccrc[c];
    }
    uint8_t* o = a.out + a.coff[c0];
    const uint8_t hdr[10] = {0x1F, 0x8B, 8, 0, 0, 0, 0, 0, 2, 0xFF};  // deflate, no flags, mtime 0, XFL = best, OS unknown
    for (int i = 0; i < 10; ++i) o[i] = hdr[i];
    uint8_t* e = a.out + a.coff[c1] - 10;
    e[0] = 0x03, e[1] = 0x00;  // final block: fixed Huffman, end-of-block only
    for (int i = 0; i < 4; ++i) e[2 + i] = (uint8_t)(crc >> (8 * i)), e[6 + i] = (uint8_t)((uint32_t)flen >> (8 * i));
    a.out_begin[f] = a.coff[c0];
}

// ---- pass 2 ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT, 5) k_gz_encode(GzArgs a) {
    __shared__ __align__(16) uint32_t s_in[CH / 4 + 8];
    __shared__ uint32_t s_out[CH / 4 + 16];
    __shared__ uint32_t s_code[260];  // reversed code | length << 16
    __shared__ uint8_t s_lens[LENS_STRIDE];
    __shared__ uint16_t s_usym[260];
    __shared__ uint32_t s_next[16], s_lcnt[16];
    __shared__ uint32_t s_scan[NT / 32], s_mask[NT / 32], s_cnt[NT / 32];
    __shared__ ChunkPos s_pos;
    __shared__ uint32_t s_bytes;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;

    for (uint64_t c = blockIdx.x; c < a.n_chunks; c += gridDim.x) {
        __syncthreads();
        if (t == 0) s_pos = locate(a, c);
        for (int i = t; i < LENS_STRIDE; i += NT) s_lens[i] = a.lens[c * LENS_STRIDE + i];
        for (int i = t; i < CH / 4 + 16; i += NT) s_out[i] = 0;
        if (t < 16) s_lcnt[t] = 0;
        __syncthreads();
        const ChunkPos p = s_pos;
        if (p.n == 0) continue;
        uint8_t* dst = a.out + a.coff[c] + (p.first ? 10 : 0);
        load_chunk(s_in, a, p.begin, p.n);
        if (s_lens[260]) {  // stored block: 00 | LEN | ~LEN | bytes
            __syncthreads();
            if (t < 5) {
                const uint32_t n = p.n, h[5] = {0u, n & 255u, n >> 8, ~n & 255u, (~n >> 8) & 255u};
                dst[t] = (uint8_t)h[t];
            }
            const uint8_t* sb = reinterpret_cast<const uint8_t*>(s_in);
            for (uint32_t i = t; i < p.n; i += NT) dst[5 + i] = sb[i];
            continue;
        }
        const uint32_t dph = (uint32_t)((uintptr_t)dst & 3u);  // s_out word 0 <-> the aligned word holding dst[0]
        const uint32_t mylen = s_lens[t], eoblen = s_lens[256];
        const bool start = t == 0 || s_lens[t - 1] != mylen;
        const uint32_t sm = __ballot_sync(0xffffffffu, start), um = __ballot_sync(0xffffffffu, mylen != 0);
        if (lane == 0) s_mask[warp] = sm, s_cnt[warp] = __popc(um);
        if (mylen) atomicAdd(&s_lcnt[mylen], 1u);
        if (t == 0) atomicAdd(&s_lcnt[eoblen], 1u);
        __syncthreads();
        // used byte values in symbol order (for the canonical codes); first code of every length (RFC 1951 3.2.2)
        int n_used = 1, at = 0;
#pragma unroll
        for (int w = 0; w < NT / 32; ++w) {
            const int x = (int)s_cnt[w];
            at += w < warp ? x : 0;
            n_used += x;
        }
        at += __popc(um & ((1u << lane) - 1u));
        if (mylen) s_usym[at] = (uint16_t)t;
        if (t == 0) {
            uint32_t code = 0;
            for (int l = 1; l < 16; ++l) {
                code = (code + (l > 1 ? s_lcnt[l - 1] : 0u)) << 1;
                s_next[l] = code;
            }
        }
        const uint32_t run = start ? run_length(s_mask, t) : 0u;
        uint32_t hdr_total;
        const uint32_t hdr_at = block_scan(start ? run_bits(mylen, run) : 0u, s_scan, &hdr_total);  // barriers inside
        const uint32_t hdr0 = dph * 8;
        if (start) {
            BitSink o{s_out, hdr0 + HDR_FIXED_BITS + hdr_at};
            emit_run(o, mylen, run);
        }
        if (t == 32) {
            BitSink o{s_out, hdr0};
            o.put(0u | 2u << 1, 3);               // not final, dynamic Huffman
            o.put(0u | 0u << 5 | 15u << 10, 14);  // HLIT - 257, HDIST - 1, HCLEN - 4
            for (int i = 0; i < 19; ++i) o.put(c_cl_len[c_cl_order[i]], 3);
            o.pos = hdr0 + HDR_FIXED_BITS + hdr_total;
            o.cl(eoblen, 0, 0);
            o.cl(0, 0, 0);
        }
        const uint32_t data0 = hdr0 + HDR_FIXED_BITS + hdr_total + c_cl_len[eoblen] + c_cl_len[0];
        if (mylen) {
            uint32_t before = 0;
            for (int j = 0; j < at; ++j) before += s_lens[s_usym[j]] == mylen;
            s_code[t] = (__brev(s_next[mylen] + before) >> (32 - mylen)) | mylen << 16;
        } else {
            s_code[t] = 0;
        }
        if (t == 0) {  // end of block is the last symbol of its length
            uint32_t before = 0;
            for (int j = 0; j < n_used - 1; ++j) before += s_lens[s_usym[j]] == eoblen;
            s_code[256] = (__brev(s_next[eoblen] + before) >> (32 - eoblen)) | eoblen << 16;
        }
        __syncthreads();
        // bits of my piece, block-wide exclusive scan, then pack
        const int my = max(0, min(PIECE, (int)p.n - t * PIECE));
        uint32_t bits = 0;
        const uint4* pv = reinterpret_cast<const uint4*>(s_in + t * (PIECE / 4));
        if (my == PIECE) {
#pragma unroll
            for (int q = 0; q < PIECE / 16; ++q) {
                const uint4 v = pv[q];
                const uint32_t wds[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    bits += (s_code[wds[k] & 255u] >> 16) + (s_code[(wds[k] >> 8) & 255u] >> 16) +
                            (s_code[(wds[k] >> 16) & 255u] >> 16) + (s_code[wds[k] >> 24] >> 16);
            }
        } else {
            for (int k = 0; k * 4 < my; ++k) {
                const uint32_t wd = s_in[t * (PIECE / 4) + k];
                const int nb = min(4, my - k * 4);
                for (int b = 0; b < nb; ++b) bits += s_code[(wd >> (8 * b)) & 255u] >> 16;
            }
        }
        uint32_t total;
        uint32_t pos = data0 + block_scan(bits, s_scan, &total);
        {
            uint64_t acc = 0;
            uint32_t have = pos & 31, word = pos >> 5;  // acc holds `have` bits below the next code
            if (my == PIECE) {
#pragma unroll
                for (int q = 0; q < PIECE / 16; ++q) {
                    const uint4 v = pv[q];
                    const uint32_t wds[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
#pragma unroll
                        for (int h = 0; h < 2; ++h) {  // two codes (<= 30 bits) per 64-bit insert
                            const uint32_t c0 = s_code[(wds[k] >> (16 * h)) & 255u], c1 = s_code[(wds[k] >> (16 * h + 8)) & 255u];
                            const uint32_t l0 = c0 >> 16;
                            acc |= (uint64_t)((c0 & 0xFFFFu) | (c1 & 0xFFFFu) << l0) << have;
                            have += l0 + (c1 >> 16);
                            if (have >= 32) {
                                atomicOr(&s_out[word++], (uint32_t)acc);
                                acc >>= 32, have -= 32;
                            }
                        }
                    }
                }
            } else {
                for (int k = 0; k * 4 < my; ++k) {
                    const uint32_t wd = s_in[t * (PIECE / 4) + k];
                    const int nb = min(4, my - k * 4);
                    for (int b = 0; b < nb; ++b) {
                        const uint32_t cl = s_code[(wd >> (8 * b)) & 255u];
                        acc |= (uint64_t)(cl & 0xFFFFu) << have;
                        have += cl >> 16;
                        if (have >= 32) {
                            atomicOr(&s_out[word++], (uint32_t)acc);
                            acc >>= 32, have -= 32;
                        }
                    }
                }
            }
            if (acc) atomicOr(&s_out[word], (uint32_t)acc);
        }
        if (t == 0) {  // end of block, empty stored block (3 zero bits), pad to a byte, 00 00 FF FF
            BitSink o{s_out, data0 + total};
            o.put(s_code[256] & 0xFFFFu, s_code[256] >> 16);
            o.pos = (o.pos + 3 + 7) & ~7u;
            o.pos += 16;
            o.put(0xFFFFu, 16);
            s_bytes = o.pos / 8 - dph;  // bytes of the chunk
        }
        __syncthreads();
        const uint32_t T = s_bytes;
        uint32_t* g0 = reinterpret_cast<uint32_t*>(dst - dph);
        const uint8_t* sb = reinterpret_cast<const uint8_t*>(s_out);
        for (uint32_t i = t; i * 4 < dph + T; i += NT) {
            if (i * 4 >= dph && i * 4 + 4 <= dph + T) g0[i] = s_out[i];
            else
                for (uint32_t b = i * 4; b < i * 4 + 4; ++b)
                    if (b >= dph && b < dph + T) reinterpret_cast<uint8_t*>(g0)[b] = sb[b];
        }
    }
}

struct Buf {
    void* p = nullptr;
    size_t cap = 0;
};

}  // namespace

struct v2p_gzip {
    int device = 0, sms = 148;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string err;
    Buf file_begin, chunk_first, lens, csize, ccrc, coff, out_begin, ctr, cub_tmp, in_stage, out_stage;
    v2p::MappedBuf pub;  // totals and per-file offsets come back through mapped pinned memory (v2p_mapped.cuh)
};

namespace {

int zfail(v2p_gzip* z, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (z) z->err = buf;
    return code;
}
#define ZCU(z, call)                                                                                                  \
    do {                                                                                                              \
        cudaError_t _st = (call);                                                                                     \
        if (_st != cudaSuccess) return zfail((z), V2P_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_st), \
                                             __FILE__, __LINE__);                                                      \
    } while (0)

int zneed(v2p_gzip* z, Buf& b, size_t bytes) {
    bytes = bytes < 256 ? 256 : bytes;
    if (b.cap >= bytes) return V2P_OK;
    if (b.p) ZCU(z, cudaFree(b.p));
    b.p = nullptr, b.cap = 0;
    ZCU(z, cudaMalloc(&b.p, bytes + bytes / 8));
    b.cap = bytes + bytes / 8;
    return V2P_OK;
}

}  // namespace

extern "C" {

int v2p_gzip_create(int cuda_device, v2p_gzip** out) {
    if (!out) return V2P_ERR_INVALID_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || cuda_device < 0 || cuda_device >= n) return V2P_ERR_CUDA;  // no CPU fallback
    v2p_gzip* z = new (std::nothrow) v2p_gzip;
    if (!z) return V2P_ERR_CUDA;
    z->device = cuda_device;
    if (cudaSetDevice(cuda_device) != cudaSuccess || cudaStreamCreateWithFlags(&z->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&z->ev0) != cudaSuccess || cudaEventCreate(&z->ev1) != cudaSuccess) {
        delete z;
        return V2P_ERR_CUDA;
    }
    cudaDeviceGetAttribute(&z->sms, cudaDevAttrMultiProcessorCount, cuda_device);
    k_crc32_init<<<1, 256, 0, z->stream>>>();
    if (cudaStreamSynchronize(z->stream) != cudaSuccess) {
        v2p_gzip_destroy(z);
        return V2P_ERR_CUDA;
    }
    *out = z;
    return V2P_OK;
}

void v2p_gzip_destroy(v2p_gzip* z) {
    if (!z) return;
    cudaSetDevice(z->device);
    cudaStreamSynchronize(z->stream);
    Buf* all[] = {&z->file_begin, &z->chunk_first, &z->lens, &z->csize, &z->ccrc, &z->coff, &z->out_begin, &z->ctr, &z->cub_tmp,
                  &z->in_stage, &z->out_stage};
    for (Buf* b : all)
        if (b->p) cudaFree(b->p);
    z->pub.release();
    if (z->ev0) cudaEventDestroy(z->ev0);
    if (z->ev1) cudaEventDestroy(z->ev1);
    if (z->stream) cudaStreamDestroy(z->stream);
    delete z;
}

const char* v2p_gzip_last_error(v2p_gzip* z) { return z ? z->err.c_str() : "gzip context is NULL"; }

uint64_t v2p_gzip_bound(uint64_t in_bytes, uint64_t n_files) {
    return in_bytes + (in_bytes / CH + n_files + 1) * 5 + n_files * 20 + 64;  // worst case: every chunk stored
}

int v2p_gzip_files(v2p_gzip* z, const uint8_t* in, const uint64_t* file_begin, uint64_t n_files, uint8_t* out,
                   uint64_t out_capacity, uint64_t* out_begin, uint32_t flags, v2p_gzip_result* res) {
    if (!z || !file_begin || !out_begin) return V2P_ERR_INVALID_ARG;
    z->err.clear();
    if (res) memset(res, 0, sizeof *res);
    for (uint64_t f = 0; f < n_files; ++f)
        if (file_begin[f + 1] < file_begin[f]) return zfail(z, V2P_ERR_INVALID_ARG, "file_begin not ascending at file %llu", (unsigned long long)f);
    const uint64_t lo = file_begin[0], hi = file_begin[n_files], in_bytes = hi - lo;
    if ((in_bytes && !in) || (n_files && !out)) return zfail(z, V2P_ERR_INVALID_ARG, "in / out is NULL");
    out_begin[0] = 0;
    if (!n_files) return V2P_OK;
    ZCU(z, cudaSetDevice(z->device));
    cudaStream_t st = z->stream;
    std::vector<uint64_t> chunk_first(n_files + 1);
    chunk_first[0] = 0;
    for (uint64_t f = 0; f < n_files; ++f) {
        const uint64_t len = file_begin[f + 1] - file_begin[f];
        chunk_first[f + 1] = chunk_first[f] + std::max<uint64_t>(1, (len + CH - 1) / CH);
    }
    const uint64_t n_chunks = chunk_first[n_files];
    int rc;
    if ((rc = zneed(z, z->file_begin, (n_files + 1) * 8)) || (rc = zneed(z, z->chunk_first, (n_files + 1) * 8)) ||
        (rc = zneed(z, z->out_begin, (n_files + 1) * 8)) || (rc = zneed(z, z->lens, n_chunks * LENS_STRIDE)) ||
        (rc = zneed(z, z->csize, (n_chunks + 1) * 8)) || (rc = zneed(z, z->coff, (n_chunks + 1) * 8)) ||
        (rc = zneed(z, z->ccrc, n_chunks * 4)) || (rc = zneed(z, z->ctr, 64)))
        return rc;
    const bool dev = flags & V2P_FLAG_DEVICE_PTRS;
    ZCU(z, cudaEventRecord(z->ev0, st));
    GzArgs a{};
    if (dev) {
        a.in = in, a.in_lo = lo, a.in_hi = hi;
    } else {
        if ((rc = zneed(z, z->in_stage, in_bytes + 16))) return rc;
        if (in_bytes) ZCU(z, cudaMemcpyAsync(z->in_stage.p, in + lo, in_bytes, cudaMemcpyHostToDevice, st));
        a.in = (const uint8_t*)z->in_stage.p - lo, a.in_lo = lo, a.in_hi = hi;  // only in[lo..hi) is ever dereferenced
    }
    ZCU(z, cudaMemcpyAsync(z->file_begin.p, file_begin, (n_files + 1) * 8, cudaMemcpyHostToDevice, st));
    ZCU(z, cudaMemcpyAsync(z->chunk_first.p, chunk_first.data(), (n_files + 1) * 8, cudaMemcpyHostToDevice, st));
    ZCU(z, cudaMemsetAsync(z->ctr.p, 0, 64, st));
    ZCU(z, cudaMemsetAsync((char*)z->csize.p + n_chunks * 8, 0, 8, st));
    a.file_begin = (const uint64_t*)z->file_begin.p, a.chunk_first = (const uint64_t*)z->chunk_first.p;
    a.n_files = n_files, a.n_chunks = n_chunks;
    a.lens = (uint8_t*)z->lens.p, a.csize = (uint64_t*)z->csize.p, a.ccrc = (uint32_t*)z->ccrc.p;
    a.coff = (const uint64_t*)z->coff.p, a.out_begin = (uint64_t*)z->out_begin.p, a.n_stored = (unsigned long long*)z->ctr.p;
    const unsigned grid = (unsigned)std::min<uint64_t>(n_chunks, (uint64_t)z->sms * 16);
    k_gz_plan<<<grid, NT, 0, st>>>(a);
    ZCU(z, cudaGetLastError());
    size_t tmp = 0;
    ZCU(z, cub::DeviceScan::ExclusiveSum(nullptr, tmp, a.csize, (uint64_t*)z->coff.p, (int64_t)(n_chunks + 1), st));
    if ((rc = zneed(z, z->cub_tmp, tmp))) return rc;
    ZCU(z, cub::DeviceScan::ExclusiveSum(z->cub_tmp.p, tmp, a.csize, (uint64_t*)z->coff.p, (int64_t)(n_chunks + 1), st));
    ZCU(z, z->pub.reserve(n_files + 1 + 8));
    {
        v2p::PubList pl{};
        pl.src[0] = (const unsigned long long*)z->coff.p + n_chunks, pl.src[1] = (const unsigned long long*)z->ctr.p, pl.n = 2;
        v2p::k_publish_list<<<1, 32, 0, st>>>(z->pub.p, pl);
    }
    ZCU(z, cudaStreamSynchronize(st));
    const uint64_t total = z->pub.p[0];
    const unsigned long long n_stored = z->pub.p[1];
    if (total > out_capacity)
        return zfail(z, V2P_ERR_RES_OOB, "output needs %llu bytes, capacity is %llu (v2p_gzip_bound gives a safe size)",
                     (unsigned long long)total, (unsigned long long)out_capacity);
    if (dev) {
        a.out = out;
    } else {
        if ((rc = zneed(z, z->out_stage, total + 16))) return rc;
        a.out = (uint8_t*)z->out_stage.p;
    }
    k_gz_files<<<(unsigned)((n_files + 1 + 127) / 128), 128, 0, st>>>(a);
    k_gz_encode<<<grid, NT, 0, st>>>(a);
    ZCU(z, cudaGetLastError());
    ZCU(z, v2p::publish_words(z->pub.p + 8, z->out_begin.p, n_files + 1, st));
    if (!dev && total) ZCU(z, cudaMemcpyAsync(out, a.out, total, cudaMemcpyDeviceToHost, st));
    ZCU(z, cudaEventRecord(z->ev1, st));
    ZCU(z, cudaStreamSynchronize(st));
    memcpy(out_begin, z->pub.p + 8, (n_files + 1) * 8);
    float ms = 0;
    ZCU(z, cudaEventElapsedTime(&ms, z->ev0, z->ev1));
    if (res) res->in_bytes = in_bytes, res->out_bytes = total, res->n_chunks = n_chunks, res->n_stored_chunks = n_stored, res->ms = ms;
    return V2P_OK;
}

}  // extern "C"
