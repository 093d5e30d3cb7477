// v2p_vcf.cu -- VCF sample columns -> FORMAT/BCSQ mask matrix on the device (include/v2p_vcf.h).
//
// Index (v2p_vcf_load), every byte of the text read twice:
//   nl_count    16 KB tiles, 16-byte loads, SWAR byte compares: newlines per tile
//   (scan)      CUB exclusive sum over the tiles
//   nl_emit     the same tiles again: a block scan of the per-thread counts puts every line start in file order
//   classify    one thread per line: end ('\r' stripped), empty / '#' / data, the first "#CHROM" line
//   (scan)      data-line ordinals; compact: line_begin / line_end / file line number of every data line
//   find_cells  one warp per data line: where its 9th tab ends (only columns 1-9 are read)
//   header_tabs the #CHROM line's tabs -> n_samples
// Parse (v2p_vcf_parse_masks), every byte of the selected cells read twice:
//   rec_segs    the selected lines cut into 512-byte segments (one warp, one 16-byte chunk per lane), so a few
//               600 KB lines and many 15 KB lines both spread over the whole GPU; (scan) -> segment ranges
//   pass 1      per segment: tabs (-> first sample column after a scan), the widest mask, the first malformed cell
//   (scan)      tabs per segment -> sample column of every segment's first cell
//   check       cell counts per line and the first error in file order (lowest line, then sample column)
//   pass 2      every cell is parsed by the lane holding the tab in front of it (cell 0: the line's first lane),
//               reading past the segment as far as the cell goes, and writes its zero-padded words
// BGZF input (v2p_vcf_load_bgzf): the host walks the block headers while the compressed bytes upload, k_inflate
// (v2p_inflate.cuh) writes the text, then the same index runs on it, and
//   fixed_len   one thread per data line: bytes of columns 1-9; (scan) -> fixed_begin
//   fixed       one warp per data line, 16-byte loads: columns 1-9 of every data line, concatenated, for the host
// Small results come back through mapped memory (v2p_mapped.cuh), not the copy engine: load waits for the line count
// (to size the line arrays) and for the header counters before it copies the line tables back; parse waits once, for the
// matrix width and the first error.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <cub/block/block_scan.cuh>
#include <cub/device/device_scan.cuh>
#include <new>
#include <string>
#include <vector>

#include "v2p_hostres.cuh"
#include "v2p_inflate.cuh"
#include "v2p_mapped.cuh"
#include "v2p_vcf.h"
#include "v2p_vcf_bgzf.h"

using namespace v2p;

namespace {

constexpr int kThreads = 256;
constexpr int kChunksPerThread = 4;                                          // 16-byte chunks, contiguous per thread
constexpr uint64_t kTile = (uint64_t)kThreads * kChunksPerThread * 16;      // 16 KB of text per block (newline passes)
constexpr uint64_t kSeg = 32 * 16;                                           // parse segment: a warp, a chunk per lane
constexpr uint32_t kNoErr = 0xffffffffu;
constexpr unsigned long long kNone = ~0ull;

enum { E_BAD_CHAR = 1, E_EMPTY = 2, E_OVERFLOW = 3, E_COUNT = 4 };  // tie order at one (line, sample column)

// bit 7 of every byte of x that equals the byte replicated in c4 (exact: no borrow between bytes)
__device__ __forceinline__ uint32_t eq_bytes(uint32_t x, uint32_t c4) {
    const uint32_t y = x ^ c4;
    return ~(((y & 0x7f7f7f7fu) + 0x7f7f7f7fu) | y | 0x7f7f7f7fu);
}

// 16-bit mask of the chunk's bytes equal to c (bit k = byte k)
__device__ __forceinline__ uint32_t chunk_eq(const uint4& v, uint32_t c4) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t m = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        uint32_t t = eq_bytes(w[i], c4) >> 7;  // bits 0, 8, 16, 24
        t = (t | (t >> 7) | (t >> 14) | (t >> 21)) & 0xfu;
        m |= t << (4 * i);
    }
    return m;
}

__device__ __forceinline__ uint64_t umin(uint64_t a, uint64_t b) { return a < b ? a : b; }

// bytes of the chunk at offset o that fall inside [lo, hi)
__device__ __forceinline__ uint32_t range_bits(uint64_t o, uint64_t lo, uint64_t hi) {
    const uint32_t a = lo <= o ? 0u : (uint32_t)umin(lo - o, 16);
    const uint32_t b = hi <= o ? 0u : (uint32_t)umin(hi - o, 16);
    return ((1u << b) - 1u) & ~((1u << a) - 1u);
}

__device__ __forceinline__ uint4 load16(const uint8_t* text, uint64_t o) { return __ldg(reinterpret_cast<const uint4*>(text + o)); }

__device__ __forceinline__ uint32_t byte_of(const uint4& v, uint32_t k) {
    const uint32_t w = k < 8 ? (k < 4 ? v.x : v.y) : (k < 12 ? v.z : v.w);
    return (w >> (8 * (k & 3))) & 0xffu;
}

constexpr uint32_t kNL4 = 0x0a0a0a0au, kTab4 = 0x09090909u;

// ---------------------------------------------------------------------------------------------------------- index
// newlines at positions [0, n-1): each one starts a line (the last byte never does)
__device__ __forceinline__ uint32_t thread_nl(const uint8_t* text, uint64_t n, uint64_t o, uint32_t (&m)[kChunksPerThread]) {
    uint32_t c = 0;
#pragma unroll
    for (int j = 0; j < kChunksPerThread; ++j) {
        const uint64_t oj = o + 16 * j;
        m[j] = oj + 1 < n ? chunk_eq(load16(text, oj), kNL4) & range_bits(oj, 0, n - 1) : 0u;
        c += __popc(m[j]);
    }
    return c;
}

__global__ void __launch_bounds__(kThreads) k_nl_count(const uint8_t* __restrict__ text, uint64_t n, uint64_t* __restrict__ tile_cnt,
                                                       uint64_t n_tiles) {
    __shared__ uint32_t s;
    if (threadIdx.x == 0) s = 0;
    __syncthreads();
    uint32_t m[kChunksPerThread];
    uint32_t c = thread_nl(text, n, blockIdx.x * kTile + threadIdx.x * (16 * kChunksPerThread), m);
#pragma unroll
    for (int d = 16; d; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s, c);
    __syncthreads();
    if (threadIdx.x == 0) {
        tile_cnt[blockIdx.x] = s;
        if (blockIdx.x == 0) tile_cnt[n_tiles] = 0;
    }
}

__global__ void __launch_bounds__(kThreads) k_nl_emit(const uint8_t* __restrict__ text, uint64_t n, const uint64_t* __restrict__ tile_x,
                                                      uint64_t* __restrict__ starts) {
    using Scan = cub::BlockScan<uint32_t, kThreads>;
    __shared__ typename Scan::TempStorage tmp;
    const uint64_t o = blockIdx.x * kTile + threadIdx.x * (16 * kChunksPerThread);
    uint32_t m[kChunksPerThread];
    const uint32_t c = thread_nl(text, n, o, m);
    uint32_t off;
    Scan(tmp).ExclusiveSum(c, off);
    uint64_t* dst = starts + 1 + tile_x[blockIdx.x] + off;
    if (blockIdx.x == 0 && threadIdx.x == 0) starts[0] = 0;
#pragma unroll
    for (int j = 0; j < kChunksPerThread; ++j)
        for (uint32_t b = m[j]; b; b &= b - 1) *dst++ = o + 16 * j + (__ffs(b) - 1) + 1;
}

struct LoadCtr {              // published to the host after the index pass
    unsigned long long n_data;
    unsigned long long chrom;  // first #CHROM line (line ordinal), kNone = none
    unsigned long long hb, he;
    unsigned long long tabs;   // tabs of the #CHROM line
};

__global__ void k_classify(const uint8_t* __restrict__ text, uint64_t n, const uint64_t* __restrict__ starts, uint64_t n_raw,
                           uint64_t* __restrict__ is_data, uint64_t* __restrict__ ends, LoadCtr* ctr) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i == n_raw) is_data[n_raw] = 0;
    if (i >= n_raw) return;
    const uint64_t b = starts[i];
    uint64_t e = i + 1 < n_raw ? starts[i + 1] - 1 : (text[n - 1] == '\n' ? n - 1 : n);
    if (e > b && text[e - 1] == '\r') --e;
    ends[i] = e;
    const bool hash = e > b && text[b] == '#';
    is_data[i] = (e > b && !hash) ? 1 : 0;
    if (hash && e - b >= 6 && text[b + 1] == 'C' && text[b + 2] == 'H' && text[b + 3] == 'R' && text[b + 4] == 'O' && text[b + 5] == 'M')
        atomicMin(&ctr->chrom, (unsigned long long)i);
}

__global__ void k_header_range(const uint64_t* __restrict__ starts, const uint64_t* __restrict__ ends, LoadCtr* ctr) {
    if (ctr->chrom != kNone) ctr->hb = starts[ctr->chrom], ctr->he = ends[ctr->chrom];
}

__global__ void k_header_tabs(const uint8_t* __restrict__ text, LoadCtr* ctr) {
    const uint64_t hb = ctr->hb, he = ctr->he;
    uint32_t c = 0;
    for (uint64_t o = (hb & ~15ull) + 16 * (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x); o < he; o += 16ull * gridDim.x * blockDim.x)
        c += __popc(chunk_eq(load16(text, o), kTab4) & range_bits(o, hb, he));
#pragma unroll
    for (int d = 16; d; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&ctr->tabs, (unsigned long long)c);
}

__global__ void k_compact(const uint64_t* __restrict__ starts, const uint64_t* __restrict__ ends, const uint64_t* __restrict__ is_data,
                          const uint64_t* __restrict__ data_x, uint64_t n_raw, uint64_t* __restrict__ line_begin,
                          uint64_t* __restrict__ line_end, uint32_t* __restrict__ line_no, LoadCtr* ctr) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i == 0) ctr->n_data = data_x[n_raw];
    if (i >= n_raw || !is_data[i]) return;
    const uint64_t j = data_x[i];
    line_begin[j] = starts[i], line_end[j] = ends[i], line_no[j] = (uint32_t)i;
}

// one warp per data line: offset after its 9th tab (has_cells = 1), or the line end (has_cells = 0)
__global__ void k_find_cells(const uint8_t* __restrict__ text, const uint64_t* __restrict__ line_begin, const uint64_t* __restrict__ line_end,
                             const LoadCtr* __restrict__ ctr, uint64_t* __restrict__ cells_begin, uint8_t* __restrict__ has_cells) {
    const uint64_t n_lines = ctr->n_data;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * (uint64_t)blockDim.x) >> 5;
    for (uint64_t l = warp; l < n_lines; l += n_warps) {
        const uint64_t b = line_begin[l], e = line_end[l];
        uint32_t seen = 0;  // tabs before this step
        uint64_t at = kNone;
        for (uint64_t base = b & ~15ull; base < e && at == kNone; base += kSeg) {
            const uint64_t o = base + 16 * lane;
            const uint32_t m = o < e ? chunk_eq(load16(text, o), kTab4) & range_bits(o, b, e) : 0u;
            const uint32_t c = __popc(m);
            uint32_t incl = c;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= (uint32_t)d) incl += t;
            }
            const uint32_t excl = incl - c;
            const bool mine = seen + excl < 9 && seen + incl >= 9;
            uint64_t pos = 0;
            if (mine) {
                uint32_t mm = m;
                for (uint32_t k = seen + excl + 1; k < 9; ++k) mm &= mm - 1;
                pos = o + (__ffs(mm) - 1);
            }
            const uint32_t who = __ballot_sync(0xffffffffu, mine);
            if (who) at = __shfl_sync(0xffffffffu, pos, __ffs(who) - 1);
            seen += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) {
            cells_begin[l] = at == kNone ? e : at + 1;
            has_cells[l] = at == kNone ? 0 : 1;
        }
    }
}

// columns 1-9 of every data line, concatenated in file order (BGZF input: the host has no text of its own)
__global__ void k_fixed_len(const uint64_t* __restrict__ line_begin, const uint64_t* __restrict__ cells_begin, uint64_t n,
                            uint64_t* __restrict__ len) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i == n) len[n] = 0;
    if (i < n) len[i] = cells_begin[i] - line_begin[i];
}

__global__ void k_fixed(const uint8_t* __restrict__ text, const uint64_t* __restrict__ line_begin, const uint64_t* __restrict__ cells_begin,
                        const uint64_t* __restrict__ fixed_x, uint64_t n_lines, uint8_t* __restrict__ fixed) {
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * (uint64_t)blockDim.x) >> 5;
    for (uint64_t l = warp; l < n_lines; l += n_warps) {
        const uint64_t b = line_begin[l], e = cells_begin[l], x = fixed_x[l];
        for (uint64_t o = (b & ~15ull) + 16 * lane; o < e; o += kSeg) {
            const uint4 v = load16(text, o);
            for (uint32_t m = range_bits(o, b, e); m; m &= m - 1) {
                const uint32_t k = __ffs(m) - 1;
                fixed[x + (o + k - b)] = (uint8_t)byte_of(v, k);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------- parse
struct ParseArgs {
    const uint8_t* text;
    const uint64_t* rec_line;
    const uint64_t* cells_begin;
    const uint64_t* line_end;
    const uint8_t* has_cells;
    const uint32_t* line_no;
    const uint64_t* seg_begin;  // n_rec+1: segments of record r = [seg_begin[r], seg_begin[r+1])
    uint64_t n_rec;
    uint64_t n_samples;
    uint64_t* seg_tabs;         // pass 1: tabs per segment (+1 trailing 0), scanned into seg_tab_x
    const uint64_t* seg_tab_x;
    uint32_t* seg_err;          // pass 1: min (local cell ordinal << 3 | class), kNoErr = none
    uint32_t* seg_rec;          // pass 1: record of the segment
    unsigned long long* ctr;    // [0] widest mask (words), [1] first error key
    uint32_t* masks;            // pass 2
    uint32_t W;
};

__global__ void k_rec_segs(const uint64_t* __restrict__ rec_line, uint64_t n_rec, const uint64_t* __restrict__ cells_begin,
                           const uint64_t* __restrict__ line_end, uint64_t* __restrict__ n_seg) {
    const uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (r == n_rec) n_seg[n_rec] = 0;
    if (r >= n_rec) return;
    const uint64_t l = rec_line[r], a0 = cells_begin[l] & ~15ull, e = line_end[l];
    n_seg[r] = e > a0 ? (e - a0 + kSeg - 1) / kSeg : 1;
}

// Reads the bytes of one cell, from its first byte to the next tab or the line end, keeping one 16-byte chunk in
// registers.  The mask is the last ':'-field: a ':' restarts the field (WRITE: the words already stored are overwritten
// by the next field's, which is never wider than W).  Returns the last field's word count; *err = the class of its
// first malformed word (0 = none).
template <bool WRITE>
__device__ uint32_t parse_cell(const uint8_t* __restrict__ text, uint64_t p, uint64_t e, uint64_t& co, uint4& v, uint32_t* out,
                               uint32_t W, uint32_t* err) {
    uint32_t nw = 0, ferr = 0;
    uint64_t val = 0;
    bool empty = true, bad = false;
    for (;; ++p) {
        uint32_t c = '\t';
        if (p < e) {
            if (p >= co + 16) co = p & ~15ull, v = load16(text, co);
            c = byte_of(v, (uint32_t)(p - co));
        }
        const uint32_t d = c - '0';
        if (d < 10) {
            val = val * 10 + d;
            if (val > 0xffffffffull) val = 0x100000000ull;  // overflowed; stays above 2^32-1
            empty = false;
        } else if (c == ',' || c == '\t') {
            const uint32_t cls = empty ? E_EMPTY : bad ? E_BAD_CHAR : val > 0xffffffffull ? E_OVERFLOW : 0;
            if (!ferr) ferr = cls;
            if (WRITE && nw < W) out[nw] = (uint32_t)val;
            ++nw;
            val = 0, empty = true, bad = false;
            if (c == '\t') break;
        } else if (c == ':') {
            nw = 0, ferr = 0, val = 0, empty = true, bad = false;
        } else {
            bad = true, empty = false;
        }
    }
    if (WRITE)
        for (uint32_t k = nw; k < W; ++k) out[k] = 0;
    *err = ferr;
    return nw;
}

template <bool WRITE>
__global__ void __launch_bounds__(kThreads) k_parse(ParseArgs a) {
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * (uint64_t)blockDim.x) >> 5;
    const uint64_t total = a.seg_begin[a.n_rec];
    const uint64_t per = (total + n_warps - 1) / n_warps, g0 = warp * per, g1 = umin(total, g0 + per);
    if (g0 >= g1) return;
    uint64_t lo = 0, hi = a.n_rec;  // last r with seg_begin[r] <= g0
    while (hi - lo > 1) {
        const uint64_t mid = (lo + hi) >> 1;
        if (a.seg_begin[mid] <= g0) lo = mid;
        else hi = mid;
    }
    uint64_t r = lo, sb = a.seg_begin[r], se = a.seg_begin[r + 1];
    uint64_t l = a.rec_line[r], cb = a.cells_begin[l], e = a.line_end[l];
    bool hc = a.has_cells[l];
    uint32_t widest = 0;
    for (uint64_t g = g0; g < g1; ++g) {
        if (g >= se) {
            while (a.seg_begin[r + 1] <= g) ++r;
            sb = a.seg_begin[r], se = a.seg_begin[r + 1];
            l = a.rec_line[r], cb = a.cells_begin[l], e = a.line_end[l], hc = a.has_cells[l];
        }
        const uint64_t o = (cb & ~15ull) + (g - sb) * kSeg + 16 * lane;
        uint4 v = make_uint4(0, 0, 0, 0);
        uint32_t tabs = 0;
        if (o < e) {
            v = load16(a.text, o);
            tabs = chunk_eq(v, kTab4) & range_bits(o, cb, e);
        }
        const uint32_t c = __popc(tabs);
        uint32_t incl = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= (uint32_t)d) incl += t;
        }
        // this lane's cells: local ordinal k (sample column = tabs of the line before the segment + k)
        uint32_t k = incl - c + 1;
        uint32_t lerr = kNoErr;
        const bool first = g == sb && lane == 0 && hc;  // cell 0 starts at cells_begin
        uint64_t base = 0;
        if (WRITE) base = a.seg_tab_x[g] - a.seg_tab_x[sb];
        uint64_t co = o;
        for (int it = first ? -1 : 0; it < 0 || tabs; ++it) {
            uint64_t p;
            uint32_t ord;
            if (it < 0) {
                p = cb, ord = 0;
            } else {
                p = o + (__ffs(tabs) - 1) + 1, ord = k++;
                tabs &= tabs - 1;
            }
            uint32_t cerr;
            if (WRITE) {
                const uint64_t col = base + ord;
                if (col < a.n_samples) parse_cell<true>(a.text, p, e, co, v, a.masks + (r * a.n_samples + col) * a.W, a.W, &cerr);
            } else {
                widest = max(widest, parse_cell<false>(a.text, p, e, co, v, nullptr, 0, &cerr));
                if (cerr && lerr == kNoErr) lerr = (ord << 3) | cerr;
            }
        }
        if (!WRITE) {
            uint32_t m = lerr;
#pragma unroll
            for (int d = 16; d; d >>= 1) m = min(m, __shfl_xor_sync(0xffffffffu, m, d));
            if (lane == 31) a.seg_tabs[g] = incl;
            if (lane == 0) a.seg_err[g] = m, a.seg_rec[g] = (uint32_t)r;
        }
    }
    if (!WRITE) {
#pragma unroll
        for (int d = 16; d; d >>= 1) widest = max(widest, __shfl_xor_sync(0xffffffffu, widest, d));
        if (lane == 0 && widest) atomicMax(&a.ctr[0], (unsigned long long)widest);
    }
}

__device__ __forceinline__ unsigned long long err_key(uint32_t line_no, uint64_t col, uint32_t cls) {
    return ((unsigned long long)line_no << 32) | (umin(col, (1ull << 29) - 1) << 3) | cls;
}

// cell counts per selected line and the first error in file order
__global__ void k_check(ParseArgs a) {
    const uint64_t total = a.seg_begin[a.n_rec];
    for (uint64_t g = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; g < total; g += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t r = a.seg_rec[g];
        const uint64_t sb = a.seg_begin[r], tb = a.seg_tab_x[sb], l = a.rec_line[r];
        if (g == sb) {
            const uint64_t n_cells = a.has_cells[l] ? a.seg_tab_x[a.seg_begin[r + 1]] - tb + 1 : 0;
            if (n_cells != a.n_samples) atomicMin(&a.ctr[1], err_key(a.line_no[l], umin(n_cells, a.n_samples), E_COUNT));
        }
        const uint32_t se = a.seg_err[g];
        if (se != kNoErr) atomicMin(&a.ctr[1], err_key(a.line_no[l], a.seg_tab_x[g] - tb + (se >> 3), se & 7));
    }
}

}  // namespace

struct v2p_vcf {
    int device = 0;
    int sms = 148;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[7] = {};
    std::string err;
    MappedBuf pub;
    // the loaded text and its index
    bool loaded = false;
    const uint8_t* text = nullptr;  // owned copy (buf_text) or the caller's device text
    uint64_t n_bytes = 0, n_lines = 0, n_samples = 0;
    DevBuf buf_text, tile_cnt, tile_x, starts, ends, is_data, data_x, line_begin, line_end, line_no, cells_begin, has_cells, ctr, cub_tmp;
    std::vector<uint64_t> h_line_begin, h_cells_begin;
    // BGZF input: compressed bytes, block table; columns 1-9 for the host
    DevBuf comp, blocks, fixed_len, fixed_x, fixed;
    std::vector<BgzfBlock> h_blocks;
    PinnedBuf h_head, h_fixed, h_fixed_begin;
    // parse
    DevBuf rec_line, n_seg, seg_begin, seg_tabs, seg_tab_x, seg_err, seg_rec, masks;
};

namespace {

// device words -> mapped host memory -> dst, after everything queued so far
int fetch(v2p_vcf* v, const void* src, uint64_t n_words, void* dst) {
    CU(v->err, v->pub.reserve(n_words));
    CU(v->err, v2p::publish_words(v->pub.p, src, n_words, v->stream));
    CU(v->err, cudaStreamSynchronize(v->stream));
    memcpy(dst, v->pub.p, n_words * 8);
    return V2P_OK;
}

// Index of v->text[0, n): line tables on the device, their host copies, n_lines / n_samples; the index kernels end
// with `done` recorded.  h = the counters of the #CHROM line.
int index_text(v2p_vcf* v, uint64_t n, cudaEvent_t done, LoadCtr& h) {
    cudaStream_t st = v->stream;
    int rc;
    const uint64_t n_tiles = (n + kTile - 1) / kTile;
    h = LoadCtr{0, kNone, 0, 0, 0};
    CU(v->err, v->ctr.need(sizeof(LoadCtr)));
    CU(v->err, v->tile_cnt.need((n_tiles + 1) * 8));
    CU(v->err, v->tile_x.need((n_tiles + 1) * 8));
    LoadCtr* ctr = (LoadCtr*)v->ctr.p;
    CU(v->err, cudaMemcpyAsync(ctr, &h, sizeof h, cudaMemcpyHostToDevice, st));
    uint64_t n_nl = 0;
    if (n) {
        k_nl_count<<<(unsigned)n_tiles, kThreads, 0, st>>>(v->text, n, (uint64_t*)v->tile_cnt.p, n_tiles);
        if ((rc = exclusive_sum(v->err, v->cub_tmp, (const uint64_t*)v->tile_cnt.p, (uint64_t*)v->tile_x.p, n_tiles + 1, st))) return rc;
        if ((rc = fetch(v, (const uint64_t*)v->tile_x.p + n_tiles, 1, &n_nl))) return rc;
    }
    const uint64_t n_raw = n ? n_nl + 1 : 0;
    if (n_raw >> 32) return fail(v->err, V2P_ERR_INVALID_ARG, "more than 2^32 lines");
    CU(v->err, v->starts.need((n_raw + 1) * 8));
    CU(v->err, v->ends.need((n_raw + 1) * 8));
    CU(v->err, v->is_data.need((n_raw + 1) * 8));
    CU(v->err, v->data_x.need((n_raw + 1) * 8));
    CU(v->err, v->line_begin.need(n_raw * 8));
    CU(v->err, v->line_end.need(n_raw * 8));
    CU(v->err, v->line_no.need(n_raw * 4));
    CU(v->err, v->cells_begin.need(n_raw * 8));
    CU(v->err, v->has_cells.need(n_raw));
    if (n) {
        const uint64_t* starts = (const uint64_t*)v->starts.p;
        k_nl_emit<<<(unsigned)n_tiles, kThreads, 0, st>>>(v->text, n, (const uint64_t*)v->tile_x.p, (uint64_t*)v->starts.p);
        k_classify<<<blocks(n_raw + 1), 256, 0, st>>>(v->text, n, starts, n_raw, (uint64_t*)v->is_data.p, (uint64_t*)v->ends.p, ctr);
        k_header_range<<<1, 1, 0, st>>>(starts, (const uint64_t*)v->ends.p, ctr);
        k_header_tabs<<<(unsigned)v->sms, 256, 0, st>>>(v->text, ctr);
        if ((rc = exclusive_sum(v->err, v->cub_tmp, (const uint64_t*)v->is_data.p, (uint64_t*)v->data_x.p, n_raw + 1, st))) return rc;
        k_compact<<<blocks(n_raw), 256, 0, st>>>(starts, (const uint64_t*)v->ends.p, (const uint64_t*)v->is_data.p,
                                                 (const uint64_t*)v->data_x.p, n_raw, (uint64_t*)v->line_begin.p,
                                                 (uint64_t*)v->line_end.p, (uint32_t*)v->line_no.p, ctr);
        // the grid is sized by the line count, the kernel reads the data-line count k_compact left in ctr
        k_find_cells<<<(unsigned)std::min<uint64_t>((n_raw + 7) / 8, (uint64_t)v->sms * 32), 256, 0, st>>>(
            v->text, (const uint64_t*)v->line_begin.p, (const uint64_t*)v->line_end.p, ctr, (uint64_t*)v->cells_begin.p,
            (uint8_t*)v->has_cells.p);
        CU(v->err, cudaGetLastError());
    }
    CU(v->err, cudaEventRecord(done, st));
    static_assert(sizeof(LoadCtr) == 40, "LoadCtr is published as five 8-byte words");
    if ((rc = fetch(v, ctr, 5, &h))) return rc;
    if (h.chrom == kNone) return fail(v->err, V2P_ERR_VCF_PARSE, "no #CHROM line: the number of samples is unknown");
    v->n_lines = h.n_data, v->n_bytes = n, v->n_samples = h.tabs >= 9 ? h.tabs - 8 : 0;
    v->h_line_begin.resize(v->n_lines), v->h_cells_begin.resize(v->n_lines);
    if (v->n_lines) {
        CU(v->err, cudaMemcpyAsync(v->h_line_begin.data(), v->line_begin.p, v->n_lines * 8, cudaMemcpyDeviceToHost, st));
        CU(v->err, cudaMemcpyAsync(v->h_cells_begin.data(), v->cells_begin.p, v->n_lines * 8, cudaMemcpyDeviceToHost, st));
    }
    CU(v->err, cudaStreamSynchronize(st));
    return V2P_OK;
}

void fill_lines(const v2p_vcf* v, const LoadCtr& h, v2p_vcf_lines* out) {
    out->n_samples = v->n_samples, out->header_begin = h.hb, out->header_end = h.he, out->n_lines = v->n_lines;
    out->line_begin = v->h_line_begin.data(), out->cells_begin = v->h_cells_begin.data();
}

constexpr uint64_t kBgzfMaxIsize = 65536;
const char* const kBgzfWhat[] = {"", "bad BGZF block header", "invalid DEFLATE data",
                                 "inflated size differs from the trailer's ISIZE", "CRC-32 differs from the trailer's"};

inline uint32_t le16(const uint8_t* p) { return p[0] | (uint32_t)p[1] << 8; }
inline uint32_t le32(const uint8_t* p) { return le16(p) | le16(p + 2) << 16; }

// SAM spec 4.1 block headers from `d`: the block table (out_off = exclusive sum of ISIZE) and each block's file offset.
// Stops at the first bad header: returns false with `why` set and its offset last in `at`; the blocks before it are in
// the table.
bool walk_bgzf(const uint8_t* d, uint64_t n, std::vector<BgzfBlock>& tab, std::vector<uint64_t>& at, uint64_t& text_bytes,
               char* why, size_t why_len) {
    tab.clear(), at.clear();
    text_bytes = 0;
    for (uint64_t o = 0; o < n;) {
        const uint64_t left = n - o;
        const uint8_t* h = d + o;
        at.push_back(o);
        if (left < 18) return snprintf(why, why_len, "%llu bytes left, a header takes 18", (unsigned long long)left), false;
        if (h[0] != 31 || h[1] != 139 || h[2] != 8 || h[3] != 4)
            return snprintf(why, why_len, "no gzip header with FEXTRA alone (not BGZF: recompress with bgzip)"), false;
        const uint32_t xlen = le16(h + 10);
        if (xlen < 6 || 12 + (uint64_t)xlen > left) return snprintf(why, why_len, "XLEN %u", xlen), false;
        int64_t bsize = -1;
        for (uint32_t x = 0; x + 4 <= xlen;) {
            const uint32_t slen = le16(h + 12 + x + 2);
            if (x + 4 + slen > xlen) break;
            if (h[12 + x] == 'B' && h[12 + x + 1] == 'C' && slen == 2) bsize = le16(h + 12 + x + 4);
            x += 4 + slen;
        }
        if (bsize < 0) return snprintf(why, why_len, "no BC subfield (not BGZF: recompress with bgzip)"), false;
        const uint64_t total = (uint64_t)bsize + 1;
        if (total < 12 + (uint64_t)xlen + 8 || total > left)
            return snprintf(why, why_len, "BSIZE %lld with %llu bytes left", (long long)bsize, (unsigned long long)left), false;
        const uint32_t isize = le32(h + total - 4);
        if (isize > kBgzfMaxIsize) return snprintf(why, why_len, "ISIZE %u > 65536", isize), false;
        BgzfBlock b{};
        b.c_off = o + 12 + xlen, b.c_len = (uint32_t)(total - 12 - xlen - 8), b.out_off = text_bytes, b.isize = isize;
        b.crc = le32(h + total - 8);
        tab.push_back(b);
        text_bytes += isize, o += total;
    }
    return true;
}

}  // namespace

extern "C" {

int v2p_vcf_create(int cuda_device, v2p_vcf** out) {
    if (!out) return V2P_ERR_INVALID_ARG;
    *out = nullptr;
    v2p_vcf* v = new (std::nothrow) v2p_vcf();
    if (!v) return V2P_ERR_INVALID_ARG;
    v->device = cuda_device;
    bool ok = cudaSetDevice(cuda_device) == cudaSuccess && cudaStreamCreateWithFlags(&v->stream, cudaStreamNonBlocking) == cudaSuccess &&
              cudaDeviceGetAttribute(&v->sms, cudaDevAttrMultiProcessorCount, cuda_device) == cudaSuccess;
    for (cudaEvent_t& e : v->ev) ok = ok && cudaEventCreate(&e) == cudaSuccess;
    if (ok) {
        k_crc32_init<<<1, 256, 0, v->stream>>>();
        ok = cudaStreamSynchronize(v->stream) == cudaSuccess;
    }
    if (!ok) {
        v2p_vcf_destroy(v);
        return V2P_ERR_CUDA;
    }
    *out = v;
    return V2P_OK;
}

void v2p_vcf_destroy(v2p_vcf* v) {
    if (!v) return;
    cudaSetDevice(v->device);
    if (v->stream) cudaStreamSynchronize(v->stream);
    for (cudaEvent_t e : v->ev)
        if (e) cudaEventDestroy(e);
    if (v->stream) cudaStreamDestroy(v->stream);
    delete v;  // frees every buffer
}

const char* v2p_vcf_last_error(v2p_vcf* v) { return v ? v->err.c_str() : "vcf object is NULL"; }

int v2p_vcf_load(v2p_vcf* v, const uint8_t* text, uint64_t n_bytes, uint32_t flags, v2p_vcf_lines* out) {
    if (!v || !out) return V2P_ERR_INVALID_ARG;
    memset(out, 0, sizeof *out);
    v->err.clear();
    v->loaded = false;
    if (flags & ~V2P_FLAG_DEVICE_PTRS) return fail(v->err, V2P_ERR_INVALID_ARG, "unknown flags 0x%x", flags);
    if (n_bytes && !text) return fail(v->err, V2P_ERR_INVALID_ARG, "text is NULL");
    const bool dev = flags & V2P_FLAG_DEVICE_PTRS;
    if (dev && ((uintptr_t)text & 15)) return fail(v->err, V2P_ERR_INVALID_ARG, "device text must be 16-byte aligned");
    CU(v->err, cudaSetDevice(v->device));
    cudaStream_t st = v->stream;
    int rc;
    CU(v->err, cudaEventRecord(v->ev[0], st));
    if (dev) {
        v->text = text;
    } else {
        CU(v->err, upload(v->buf_text, text, n_bytes, st));
        v->text = (const uint8_t*)v->buf_text.p;
    }
    CU(v->err, cudaEventRecord(v->ev[1], st));
    LoadCtr h;
    if ((rc = index_text(v, n_bytes, v->ev[2], h))) return rc;
    float h2d = 0, idx = 0;
    CU(v->err, cudaEventElapsedTime(&h2d, v->ev[0], v->ev[1]));
    CU(v->err, cudaEventElapsedTime(&idx, v->ev[1], v->ev[2]));
    fill_lines(v, h, out);
    out->h2d_bytes = dev ? 0 : n_bytes, out->h2d_ms = h2d, out->index_ms = idx;
    v->loaded = true;
    return V2P_OK;
}

int v2p_vcf_load_bgzf(v2p_vcf* v, const uint8_t* data, uint64_t n_bytes, uint32_t flags, v2p_vcf_lines* out, v2p_vcf_bgzf* bz) {
    if (!v || !out || !bz) return V2P_ERR_INVALID_ARG;
    memset(out, 0, sizeof *out);
    memset(bz, 0, sizeof *bz);
    v->err.clear();
    v->loaded = false;
    if (flags & V2P_FLAG_DEVICE_PTRS) return fail(v->err, V2P_ERR_INVALID_ARG, "BGZF input must be host memory (V2P_FLAG_DEVICE_PTRS)");
    if (flags) return fail(v->err, V2P_ERR_INVALID_ARG, "unknown flags 0x%x", flags);
    if (n_bytes && !data) return fail(v->err, V2P_ERR_INVALID_ARG, "data is NULL");
    CU(v->err, cudaSetDevice(v->device));
    cudaStream_t st = v->stream;
    int rc;
    // the upload runs while the host walks the block headers
    CU(v->err, cudaEventRecord(v->ev[0], st));
    CU(v->err, upload(v->comp, data, n_bytes, st));
    CU(v->err, cudaEventRecord(v->ev[1], st));
    std::vector<uint64_t> at;
    uint64_t text_bytes = 0;
    char why[160] = "";
    const bool walked = walk_bgzf(data, n_bytes, v->h_blocks, at, text_bytes, why, sizeof why);
    const uint64_t n_blk = v->h_blocks.size();
    CU(v->err, v->blocks.need(n_blk * sizeof(BgzfBlock)));
    CU(v->err, v->buf_text.need(text_bytes + 16));
    CU(v->err, v->ctr.need(sizeof(LoadCtr)));
    if (n_blk) CU(v->err, cudaMemcpyAsync(v->blocks.p, v->h_blocks.data(), n_blk * sizeof(BgzfBlock), cudaMemcpyHostToDevice, st));
    unsigned long long* ekey = (unsigned long long*)v->ctr.p;
    CU(v->err, cudaMemsetAsync(ekey, 0xff, 8, st));
    v->text = (const uint8_t*)v->buf_text.p;
    CU(v->err, cudaEventRecord(v->ev[2], st));
    if (n_blk) {
        int per_sm = 1;
        CU(v->err, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_inflate, kInfWarps * 32, 0));
        const uint64_t grid = std::min<uint64_t>((uint64_t)v->sms * std::max(per_sm, 1), (n_blk + kInfWarps - 1) / kInfWarps);
        k_inflate<<<(unsigned)grid, kInfWarps * 32, 0, st>>>((const uint8_t*)v->comp.p, (const BgzfBlock*)v->blocks.p, n_blk,
                                                             (uint8_t*)v->buf_text.p, ekey);
        CU(v->err, cudaGetLastError());
    }
    CU(v->err, cudaEventRecord(v->ev[3], st));
    unsigned long long key = kNone;
    if ((rc = fetch(v, ekey, 1, &key))) return rc;
    // blocks before a bad header were inflated: a bad one among them comes first in file order
    if (key != kNone || !walked) {
        const uint64_t b = key != kNone ? key >> 3 : n_blk;
        const unsigned cls = key != kNone ? (unsigned)(key & 7) : (unsigned)BGZF_HEADER;
        const unsigned long long off = at[b];
        if (cls == BGZF_HEADER)
            return fail(v->err, V2P_ERR_BGZF, "BGZF block %llu at byte %llu: %s (%s)", (unsigned long long)b, off, kBgzfWhat[cls], why);
        return fail(v->err, V2P_ERR_BGZF, "BGZF block %llu at byte %llu: %s", (unsigned long long)b, off, kBgzfWhat[cls]);
    }
    CU(v->err, cudaEventRecord(v->ev[4], st));
    LoadCtr h;
    if ((rc = index_text(v, text_bytes, v->ev[5], h))) return rc;
    // columns 1-9 of every data line and the header lines back to the host
    const uint64_t nl = v->n_lines;
    uint64_t n_fixed = 0;
    for (uint64_t l = 0; l < nl; ++l) n_fixed += v->h_cells_begin[l] - v->h_line_begin[l];
    CU(v->err, v->fixed_len.need((nl + 1) * 8));
    CU(v->err, v->fixed_x.need((nl + 1) * 8));
    CU(v->err, v->fixed.need(n_fixed));
    CU(v->err, v->h_fixed_begin.need((nl + 1) * 8));
    CU(v->err, v->h_fixed.need(n_fixed));
    CU(v->err, v->h_head.need(h.he));
    const uint64_t* lb = (const uint64_t*)v->line_begin.p;
    const uint64_t* cb = (const uint64_t*)v->cells_begin.p;
    k_fixed_len<<<blocks(nl + 1), 256, 0, st>>>(lb, cb, nl, (uint64_t*)v->fixed_len.p);
    if ((rc = exclusive_sum(v->err, v->cub_tmp, (const uint64_t*)v->fixed_len.p, (uint64_t*)v->fixed_x.p, nl + 1, st))) return rc;
    if (nl)
        k_fixed<<<(unsigned)std::min<uint64_t>((nl + 7) / 8, (uint64_t)v->sms * 32), 256, 0, st>>>(v->text, lb, cb, (const uint64_t*)v->fixed_x.p,
                                                                                                   nl, (uint8_t*)v->fixed.p);
    CU(v->err, cudaGetLastError());
    CU(v->err, cudaMemcpyAsync(v->h_fixed_begin.p, v->fixed_x.p, (nl + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (n_fixed) CU(v->err, cudaMemcpyAsync(v->h_fixed.p, v->fixed.p, n_fixed, cudaMemcpyDeviceToHost, st));
    if (h.he) CU(v->err, cudaMemcpyAsync(v->h_head.p, v->text, h.he, cudaMemcpyDeviceToHost, st));
    CU(v->err, cudaEventRecord(v->ev[6], st));
    CU(v->err, cudaStreamSynchronize(st));
    float h2d = 0, inf = 0, idx = 0, fix = 0;
    CU(v->err, cudaEventElapsedTime(&h2d, v->ev[0], v->ev[1]));
    CU(v->err, cudaEventElapsedTime(&inf, v->ev[2], v->ev[3]));
    CU(v->err, cudaEventElapsedTime(&idx, v->ev[4], v->ev[5]));
    CU(v->err, cudaEventElapsedTime(&fix, v->ev[5], v->ev[6]));
    fill_lines(v, h, out);
    out->h2d_bytes = n_bytes, out->h2d_ms = h2d, out->index_ms = idx;
    bz->n_blocks = n_blk, bz->text_bytes = text_bytes, bz->text = v->text;
    bz->head = (const uint8_t*)v->h_head.p, bz->fixed = (const uint8_t*)v->h_fixed.p, bz->fixed_begin = (const uint64_t*)v->h_fixed_begin.p;
    bz->inflate_ms = inf, bz->fixed_ms = fix;
    v->loaded = true;
    return V2P_OK;
}

int v2p_vcf_parse_masks(v2p_vcf* v, uint64_t n_records, const uint64_t* rec_line, uint32_t flags, v2p_vcf_masks* out) {
    if (!v || !out) return V2P_ERR_INVALID_ARG;
    memset(out, 0, sizeof *out);
    v->err.clear();
    if (!v->loaded) return fail(v->err, V2P_ERR_INVALID_ARG, "no text loaded (v2p_vcf_load failed or was not called)");
    if (flags) return fail(v->err, V2P_ERR_INVALID_ARG, "unknown flags 0x%x", flags);
    if (n_records && !rec_line) return fail(v->err, V2P_ERR_INVALID_ARG, "rec_line is NULL");
    for (uint64_t r = 0; r < n_records; ++r)
        if (rec_line[r] >= v->n_lines)
            return fail(v->err, V2P_ERR_INVALID_ARG, "rec_line[%llu] = %llu: the text has %llu data lines", (unsigned long long)r,
                        (unsigned long long)rec_line[r], (unsigned long long)v->n_lines);
    if (n_records >> 32) return fail(v->err, V2P_ERR_INVALID_ARG, "more than 2^32 records");
    CU(v->err, cudaSetDevice(v->device));
    cudaStream_t st = v->stream;
    int rc;
    CU(v->err, cudaEventRecord(v->ev[0], st));
    CU(v->err, v->rec_line.need(n_records * 8));
    CU(v->err, v->n_seg.need((n_records + 1) * 8));
    CU(v->err, v->seg_begin.need((n_records + 1) * 8));
    CU(v->err, v->ctr.need(16));
    if (n_records) CU(v->err, cudaMemcpyAsync(v->rec_line.p, rec_line, n_records * 8, cudaMemcpyHostToDevice, st));
    // segments: at most one per 512 bytes of each selected line (from its 16-byte block of cells_begin) plus one
    uint64_t seg_cap = 0;
    for (uint64_t r = 0; r < n_records; ++r) {
        const uint64_t l = rec_line[r], a0 = v->h_cells_begin[l] & ~15ull;
        const uint64_t e = l + 1 < v->n_lines ? v->h_line_begin[l + 1] : v->n_bytes;  // >= the line's end
        seg_cap += e > a0 ? (e - a0 + kSeg - 1) / kSeg : 1;
    }
    CU(v->err, v->seg_tabs.need((seg_cap + 1) * 8));
    CU(v->err, v->seg_tab_x.need((seg_cap + 1) * 8));
    CU(v->err, v->seg_err.need(seg_cap * 4));
    CU(v->err, v->seg_rec.need(seg_cap * 4));
    unsigned long long* ctr = (unsigned long long*)v->ctr.p;
    CU(v->err, cudaMemsetAsync(ctr, 0, 8, st));
    CU(v->err, cudaMemsetAsync(ctr + 1, 0xff, 8, st));
    ParseArgs a{};
    a.text = v->text, a.rec_line = (const uint64_t*)v->rec_line.p, a.cells_begin = (const uint64_t*)v->cells_begin.p;
    a.line_end = (const uint64_t*)v->line_end.p, a.has_cells = (const uint8_t*)v->has_cells.p, a.line_no = (const uint32_t*)v->line_no.p;
    a.seg_begin = (const uint64_t*)v->seg_begin.p, a.n_rec = n_records, a.n_samples = v->n_samples;
    a.seg_tabs = (uint64_t*)v->seg_tabs.p, a.seg_tab_x = (const uint64_t*)v->seg_tab_x.p, a.seg_err = (uint32_t*)v->seg_err.p;
    a.seg_rec = (uint32_t*)v->seg_rec.p, a.ctr = ctr;
    // k_parse hands every warp an equal run of segments; one resident wave of blocks
    int per_sm = 1;
    CU(v->err, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_parse<false>, kThreads, 0));
    const unsigned grid = (unsigned)(v->sms * std::max(per_sm, 1));
    unsigned long long hc[2] = {0, kNone};
    if (n_records) {
        k_rec_segs<<<blocks(n_records + 1), 256, 0, st>>>(a.rec_line, n_records, a.cells_begin, a.line_end, (uint64_t*)v->n_seg.p);
        if ((rc = exclusive_sum(v->err, v->cub_tmp, (const uint64_t*)v->n_seg.p, (uint64_t*)v->seg_begin.p, n_records + 1, st))) return rc;
        k_parse<false><<<grid, kThreads, 0, st>>>(a);
        // entries past the segment total are not written; the scan values up to the total do not depend on them
        if ((rc = exclusive_sum(v->err, v->cub_tmp, (const uint64_t*)a.seg_tabs, (uint64_t*)v->seg_tab_x.p, seg_cap + 1, st))) return rc;
        k_check<<<grid, 256, 0, st>>>(a);
        CU(v->err, cudaGetLastError());
        if ((rc = fetch(v, ctr, 2, hc))) return rc;
    }
    if (hc[1] != kNone) {
        static const char* what[] = {"", "a mask word with a character other than a decimal digit", "an empty mask word",
                                     "a mask word above 2^32-1", "a number of sample cells other than the #CHROM line's"};
        const uint64_t col = (hc[1] >> 3) & ((1ull << 29) - 1);
        const unsigned cls = (unsigned)(hc[1] & 7);
        return fail(v->err, V2P_ERR_VCF_PARSE, "VCF line %llu, sample column %llu: %s", (unsigned long long)(hc[1] >> 32) + 1,
                    (unsigned long long)col + 1, cls <= E_COUNT ? what[cls] : "?");
    }
    const uint32_t W = hc[0] ? (uint32_t)hc[0] : 1;
    const uint64_t n_words = n_records * v->n_samples * W;
    if (n_records && v->n_samples && n_words / n_records / v->n_samples != W) return fail(v->err, V2P_ERR_INVALID_ARG, "matrix size overflows");
    CU(v->err, v->masks.need(n_words * 4));
    a.masks = (uint32_t*)v->masks.p, a.W = W;
    if (n_records && v->n_samples) k_parse<true><<<grid, kThreads, 0, st>>>(a);
    CU(v->err, cudaGetLastError());
    CU(v->err, cudaEventRecord(v->ev[1], st));
    CU(v->err, cudaStreamSynchronize(st));
    float ms = 0;
    CU(v->err, cudaEventElapsedTime(&ms, v->ev[0], v->ev[1]));
    out->masks = (const uint32_t*)v->masks.p, out->n_records = n_records, out->n_samples = v->n_samples, out->words_per_cell = W;
    out->parse_ms = ms;
    return V2P_OK;
}

}  // extern "C"
