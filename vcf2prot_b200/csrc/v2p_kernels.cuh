// v2p_kernels.cuh -- sm_100a kernels of the sequence-generation engine.
//
// The work is the reference's Task::execute (task.rs:38-50) looped as GIR::execute (gir.rs:230-234):
//   res[dst .. dst+len] <- (stream==0 ? ref : alt)[src .. src+len]   for every task, '.' elsewhere.
// It is byte-granular gather into a contiguous output stream: HBM/L2 bound, no flops, no tensor cores.
//
// Design (output-stationary, one warp per output tile):
//   plan   k_plan_haps / k_plan_tasks   validate every task where the reference would panic, and build
//                                       lb[k] = first task whose global dst >= k*TILE (one u32 per tile)
//   copy   k_copy_tiles<TILE>           each warp owns TILE output bytes staged in shared memory:
//            A. one lane per overlapping task: head/tail bytes (partial 16-B vectors) -> st.shared.u8,
//               and lead[v0] = lane for the first fully covered vector of the task
//            B. warp max-scan over lead[] -> owner task of every fully covered 16-B vector
//            C. one lane per vector: 2 aligned 16-B loads + funnel-shift realign -> st.shared.v4
//            D. one elected lane: TMA bulk store (cp.async.bulk.global.shared::cta) of the whole tile
//          => every output byte is written exactly once with full-width stores, '.' gaps come for free
//             from the tile prefill, and cost per byte is independent of task-length skew.
//   serial k_serial                     tasks that are NOT sorted/non-overlapping by dst keep the
//                                       reference's in-order semantics (later task wins) on the GPU.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "v2p_engine.h"

namespace v2p {

constexpr int kWarpsPerCta = 8;
constexpr uint32_t kTileHasGap = 0x80000000u;
constexpr int kThreads = kWarpsPerCta * 32;

// Device-side status block, written by the plan kernels with atomics.
struct DevStatus {
    unsigned long long err_key;     // min over ((global task idx << 8) | V2P_ERR_*) of slice errors; ~0 = none
    unsigned long long gap_key;     // min global task idx violating gir.rs:208 contiguity (VALIDATE); ~0 = none
    unsigned long long stream_key;  // min global task idx whose stream code is not 0/1; ~0 = none.  Kept apart from
                                    // err_key: the reference panics on it while the Task array is BUILT
                                    // (haplotype_instruction.rs:154), before any validator or copy runs, so it wins
                                    // over a slice error or a gap at a smaller index
    unsigned int unsorted;          // number of haplotypes whose tasks are not sorted / overlap (hap_flags[h] = 1):
                                    // those take the serial-order kernel, everybody else the tile kernel
    unsigned int bad_args;          // base arrays not monotone / totals inconsistent
};

struct KParams {
    const v2p_task16* tasks;     // tasks[t - task_origin]
    const uint64_t* task_begin;  // n_hap+1 (absolute task numbers)
    const uint8_t* ref;
    const uint64_t* ref_base;  // n_hap+1 or nullptr
    const uint8_t* ref_rep;    // 16 byte-shifted replicas of the registered reference (tma_mode 1) or nullptr
    uint64_t rep_stride;       // bytes between replicas; replica r stores ref[x] at ref_rep + r*rep_stride + x + r
    int tma_mode;              // 0: register path only; 1: TMA bulk copies from the replicas
    const uint8_t* alt;        // alt[a - alt_origin]
    const uint64_t* alt_base;  // n_hap+1 (absolute)
    uint8_t* out;              // out[o - out_origin], 16-byte aligned
    const uint64_t* out_base;  // n_hap+1 (absolute)
    uint64_t n_hap, n_tasks, n_ref, n_alt, n_out;  // totals of THIS launch (relative sizes)
    uint64_t task_origin, ref_origin, alt_origin, out_origin;
    uint32_t* lb;        // n_tiles+1
    uint32_t* tile_hap;  // n_tiles: haplotype owning the tile's first byte; bit 31 (kTileHasGap) = some byte of the tile is
                         // covered by no task of the tile kernel (a '.' gap, or a haplotype left to k_serial): prefill it
    uint32_t* chunk_hap;  // haplotype of the first task of every k_plan_tasks warp (kPlanWarpTasks tasks each)
    uint32_t* hap_flags;  // n_hap: 1 = this haplotype's tasks are unsorted / overlapping (reference order semantics:
                          // the tile kernel skips its tasks, k_serial applies them in array order afterwards)
    uint32_t* ser_list;   // the flagged haplotypes, compacted by k_plan_fix (ser_list[0 .. status->unsorted))
    // Tile processing order (see k_copy_tiles): order_hdr[0] = s_max = most tile GROUPS (2^order_gshift consecutive
    // tiles) any haplotype owns (k_plan_haps); order[((g * n_hap + h) << gshift) + i] = tile i of group g of haplotype h,
    // or ~0 (k_plan_tiles).  When that does not fit order_cap (wildly uneven haplotypes) order[] is the identity.
    uint32_t* order_hdr;
    uint32_t* order;
    uint64_t order_cap;
    uint32_t order_gshift;
    uint64_t n_tiles;
    uint32_t tile_bytes;
    uint32_t tile_shift;  // log2(tile_bytes)
    uint32_t fill_word;  // 0x2E2E2E2E for 1-byte residues, 0x0000002E for UTF-32 units
    int keep_out;        // 1: uncovered bytes keep the caller's content (soa call without FILL_DOT)
    int validate;        // V2P_FLAG_VALIDATE
    DevStatus* status;
    unsigned long long* warp_ns;  // profiling (v2p_engine_profile_warps): wall time of every warp of the copy grid, or nullptr
};

// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t upper_bound_u64(const uint64_t* __restrict__ a, uint64_t lo, uint64_t hi,
                                                    uint64_t key) {
    // first index in [lo,hi) with a[idx] > key
    while (lo < hi) {
        uint64_t mid = (lo + hi) >> 1;
        if (__ldg(a + mid) <= key)
            lo = mid + 1;
        else
            hi = mid;
    }
    return lo;
}

// haplotype owning absolute task number t: largest h with task_begin[h] <= t (skips empty haplotypes)
__device__ __forceinline__ uint64_t hap_of_task(const KParams& p, uint64_t t, uint64_t hint) {
    if (hint < p.n_hap && __ldg(p.task_begin + hint) <= t && t < __ldg(p.task_begin + hint + 1)) return hint;
    return upper_bound_u64(p.task_begin, 0, p.n_hap + 1, t) - 1;
}

__global__ void k_init_status(DevStatus* s) {
    s->err_key = ~0ull;
    s->gap_key = ~0ull;
    s->stream_key = ~0ull;
    s->unsorted = 0;
    s->bad_args = 0;
}

// One thread per haplotype: base-array sanity (monotone, consistent with the totals the caller passed).
__global__ void k_plan_haps(KParams p) {
    uint64_t h = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (h >= p.n_hap) return;
    uint64_t o0 = p.out_base[h], o1 = p.out_base[h + 1];
    uint64_t t0 = p.task_begin[h], t1 = p.task_begin[h + 1];
    uint64_t a0 = p.alt_base[h], a1 = p.alt_base[h + 1];
    bool bad = o1 < o0 || t1 < t0 || a1 < a0;
    if (p.ref_base) bad |= p.ref_base[h + 1] < p.ref_base[h];
    if (h == 0) {
        bad |= o0 != p.out_origin || t0 != p.task_origin || a0 != p.alt_origin;
        if (p.ref_base) bad |= p.ref_base[0] != p.ref_origin;
    }
    if (h == p.n_hap - 1) {
        bad |= o1 - p.out_origin != p.n_out || t1 - p.task_origin != p.n_tasks || a1 - p.alt_origin != p.n_alt;
        if (p.ref_base) bad |= p.ref_base[h + 1] - p.ref_origin != p.n_ref;
    }
    if (bad) atomicExch(&p.status->bad_args, 1u);
    // tiles whose first byte lies in this haplotype's tape: ceil(o1/T) - ceil(o0/T), in groups; the maximum sizes the order
    const uint64_t T1 = (uint64_t)p.tile_bytes - 1;
    const uint64_t nt = bad ? 0 : ((o1 - p.out_origin + T1) >> p.tile_shift) - ((o0 - p.out_origin + T1) >> p.tile_shift);
    uint32_t s = (uint32_t)((nt + (1u << p.order_gshift) - 1) >> p.order_gshift);
    s = __reduce_max_sync(__activemask(), s);
    if ((threadIdx.x & 31) == 0 && s) atomicMax(p.order_hdr, s);
}

// slots of the haplotype-interleaved tile order, or 0 when it does not fit (then order[] is the identity over n_tiles)
__device__ __forceinline__ uint64_t tile_order_slots(const KParams& p, uint32_t s_max) {
    const uint64_t n = ((uint64_t)s_max * p.n_hap) << p.order_gshift;
    return (p.n_hap > 1 && n <= p.order_cap) ? n : 0;
}

// One lane per task; every warp owns kPlanWarpTasks CONSECUTIVE tasks: everything the reference would panic on, plus
// lb[] (tile -> first task).  All task arithmetic is launch-relative and 32-bit (n_tasks < 2^32-2, checked by the host;
// a tile index fits 32 bits for any tape that fits HBM).  The owning haplotype's bases are warp-uniform registers that
// advance with the warp's position (a haplotype is ~20k tasks; the haplotype of every warp's first task comes from
// k_plan_tiles, so no warp starts with a dependent-load binary search); only a sub-iteration that straddles a
// haplotype boundary or the end of the range takes the per-lane lookup.  The previous task's (dst, len, tile) reaches
// a lane by ONE rotate shuffle per value: lane 31 contributes what it held in the previous sub-iteration.
__device__ __forceinline__ void prefetch_l2(const void* gptr) { asm volatile("prefetch.global.L2 [%0];" ::"l"(gptr)); }
constexpr int kPlanU = 4;                       // sub-iterations whose loads are issued together
constexpr int kPlanWarpTasks = 32 * 16;         // consecutive tasks per warp
constexpr int kPlanChunk = kPlanWarpTasks * 8;  // ... per 256-thread CTA

struct PlanHap {  // bases of one haplotype, launch-relative
    uint32_t h;         // its index
    uint32_t tb0, tb1;  // its tasks [tb0, tb1)
    uint64_t orel;      // start of its result tape
    uint32_t otile, orem;  // ... as tile number and offset inside that tile (32-bit tile arithmetic for the hot loop)
    uint64_t n_res, n_alt, n_ref;
};

__device__ __forceinline__ PlanHap plan_hap_load(const KParams& p, uint64_t h) {
    PlanHap c;
    c.h = (uint32_t)h;
    c.tb0 = (uint32_t)(__ldg(p.task_begin + h) - p.task_origin);
    c.tb1 = (uint32_t)min(__ldg(p.task_begin + h + 1) - p.task_origin, p.n_tasks);
    const uint64_t o0 = __ldg(p.out_base + h);
    c.orel = o0 - p.out_origin;
    c.otile = (uint32_t)(c.orel >> p.tile_shift), c.orem = (uint32_t)c.orel & (p.tile_bytes - 1u);
    c.n_res = __ldg(p.out_base + h + 1) - o0;
    c.n_alt = __ldg(p.alt_base + h + 1) - __ldg(p.alt_base + h);
    c.n_ref = p.ref_base ? __ldg(p.ref_base + h + 1) - __ldg(p.ref_base + h) : p.n_ref;
    return c;
}
__device__ __forceinline__ PlanHap plan_hap_of(const KParams& p, uint32_t tr) {
    return plan_hap_load(p, upper_bound_u64(p.task_begin, 0, p.n_hap + 1, tr + p.task_origin) - 1);
}

// One thread per output tile: the haplotype that owns the tile's first byte (binary search over out_base);
// and one thread per k_plan_tasks warp: the haplotype of its first task (binary search over task_begin).
__global__ void k_plan_tiles(KParams p) {
    const uint64_t k = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (k < p.n_tiles) {
        const uint64_t x = (k << p.tile_shift) + p.out_origin;
        uint64_t h = upper_bound_u64(p.out_base, 0, p.n_hap + 1, x);  // first h with out_base[h] > x
        h = h ? h - 1 : 0;
        if (h >= p.n_hap) h = p.n_hap - 1;
        p.tile_hap[k] = (uint32_t)h;
        if (tile_order_slots(p, p.order_hdr[0])) {  // slot of this tile in the haplotype-interleaved order
            const uint64_t first = (__ldg(p.out_base + h) - p.out_origin + p.tile_bytes - 1) >> p.tile_shift;
            const uint64_t c = k - first, gm = (1u << p.order_gshift) - 1;
            const uint64_t idx = (((c >> p.order_gshift) * p.n_hap + h) << p.order_gshift) + (c & gm);
            if (idx < p.order_cap) p.order[idx] = (uint32_t)k;  // (always, unless the base arrays are inconsistent)
        } else if (k < p.order_cap) {
            p.order[k] = (uint32_t)k;
        }
    }
    const uint64_t t = k * kPlanWarpTasks;
    if (t < p.n_tasks) {
        uint64_t h = upper_bound_u64(p.task_begin, 0, p.n_hap + 1, t + p.task_origin);
        h = h ? h - 1 : 0;  // task_begin[0] > origin is reported by k_plan_haps (bad_args)
        if (h >= p.n_hap) h = p.n_hap - 1;
        p.chunk_hap[k] = (uint32_t)h;
    }
}

// tile in which haplotype-relative offset dst of haplotype m starts, clamped to n_tiles (a rejected task's garbage
// offset must not index lb[] out of range), in 32-bit arithmetic that cannot overflow
__device__ __forceinline__ uint32_t plan_tile_of(const KParams& p, const PlanHap& m, const uint32_t dst) {
    const uint32_t k = m.otile + (dst >> p.tile_shift) + (((dst & (p.tile_bytes - 1u)) + m.orem) >> p.tile_shift);
    return min(k, (uint32_t)p.n_tiles);
}

// One task of the plan (lane-private): m = bases of its haplotype; (kprev, p_dst, p_len) = the task in front of it.
__device__ __forceinline__ void plan_one(const KParams& p, const PlanHap& m, const uint4 raw, const uint32_t tr,
                                         const uint32_t kt, const uint32_t kprev, const uint32_t p_dst,
                                         const uint32_t p_len) {
    const uint32_t src = raw.x, len = raw.y, dst = raw.z, stream = raw.w;
    // every reference panic, one predicate each (error paths are cold)
    const bool bad_stream = stream > 1u;                                           // haplotype_instruction.rs:154
    const bool bad_res = (uint64_t)dst + len > m.n_res;                            // task.rs:44/48 (result slice)
    const bool bad_src = (uint64_t)src + len > (stream == 0 ? m.n_ref : m.n_alt);  // task.rs:44/48 (source slice)
    // gir.rs:208 contiguity (VALIDATE): the validator sees the whole Task array before any task runs, so a task that
    // does not start where the previous one ended is reported as such, whether it leaves a gap, goes back or has a bad slice
    if (p.validate && tr != m.tb0 && dst != (uint64_t)p_dst + p_len) atomicMin(&p.status->gap_key, (unsigned long long)tr);
    if (bad_stream | bad_res | bad_src) {
        if (bad_stream) atomicMin(&p.status->stream_key, (unsigned long long)tr);
        else atomicMin(&p.status->err_key, ((unsigned long long)tr << 8) | (bad_res ? V2P_ERR_RES_OOB : V2P_ERR_SRC_OOB));
        return;
    }
    // bytes no task covers read '.' (haplotype_instruction.rs:78): the tiles that hold any are marked, and only those
    // are prefilled by the copy kernel (everywhere else every byte of the tile is written by some task)
    auto mark_gap = [&](uint64_t a, uint64_t b) {  // launch-relative byte range [a, b)
        for (uint64_t k = a >> p.tile_shift; k <= ((b - 1) >> p.tile_shift) && k < p.n_tiles; ++k) atomicOr(p.tile_hap + k, kTileHasGap);
    };
    if (tr != m.tb0) {  // previous task is in the same haplotype: sortedness
        const uint64_t pend = (uint64_t)p_dst + p_len;
        if (dst < pend) {  // this haplotype needs the reference's order semantics (later task wins): k_serial
            if (atomicExch(p.hap_flags + m.h, 1u) == 0u) atomicAdd(&p.status->unsorted, 1u);
            return;
        }
        if (dst != pend) mark_gap(m.orel + pend, m.orel + dst);
    } else if (dst != 0u) {
        mark_gap(m.orel, m.orel + dst);  // in front of the haplotype's first task
    }
    if (tr + 1u == m.tb1 && (uint64_t)dst + len < m.n_res) mark_gap(m.orel + dst + len, m.orel + m.n_res);  // behind its last
    // Only tasks that start a new tile (or follow whole tiles of '.') write lb[].  kt and kprev are clamped to
    // n_tiles by the caller (the task in FRONT of this one may be a rejected one with a garbage dst -- the launch
    // then fails with its status, but lb[] must not be written out of range meanwhile); valid sorted input has
    // kt >= kprev, and kprev == ~0 (task 0) wraps to tile 0.
    if (kprev == 0xFFFFFFFFu || kt > kprev) {
        p.lb[kprev + 1u] = tr;
        for (uint32_t k = kprev + 2u; k <= kt; ++k) p.lb[k] = tr;
    }
}

#ifndef V2P_PLAN_MINB
#define V2P_PLAN_MINB 4
#endif
__global__ void __launch_bounds__(256, V2P_PLAN_MINB) k_plan_tasks(KParams p) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t wid = (uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const uint64_t first64 = wid * kPlanWarpTasks;
    if (first64 >= p.n_tasks) return;
    if (p.status->bad_args) return;
    const uint32_t first = (uint32_t)first64;
    const uint32_t end = (uint32_t)min(first64 + kPlanWarpTasks, p.n_tasks);
    const uint4* __restrict__ tk = reinterpret_cast<const uint4*>(p.tasks);
    const uint32_t rot = (lane + 31u) & 31u;

    uint4 raw[kPlanU];
#pragma unroll
    for (int u = 0; u < kPlanU; ++u) {  // the first loads go out before the haplotype bases are known
        const uint32_t tr = first + 32 * u + lane;
        raw[u] = tr < end ? __ldg(tk + tr) : make_uint4(0u, 0u, 0u, 0u);
    }
    PlanHap c = plan_hap_load(p, __ldg(p.chunk_hap + wid));  // warp-uniform
    // what lane 31 "held before": the task in front of this warp's range (its tile, dst, len)
    uint32_t o_kt = 0xFFFFFFFFu, o_dst = 0u, o_len = 0u;  // first == 0: lb[0 .. tile of task 0] = 0
    if (first > 0) {
        const uint4 pt = __ldg(tk + first - 1);
        o_kt = first - 1 >= c.tb0 ? plan_tile_of(p, c, pt.z) : plan_tile_of(p, plan_hap_of(p, first - 1), pt.z);
        o_dst = pt.z, o_len = pt.y;
    }

    for (uint32_t base = first; base < end; base += 32 * kPlanU) {
        if (base != first) {
#pragma unroll
            for (int u = 0; u < kPlanU; ++u) {
                const uint32_t tr = base + 32 * u + lane;
                raw[u] = tr < end ? __ldg(tk + tr) : make_uint4(0u, 0u, 0u, 0u);
            }
        }
#pragma unroll
        for (int u = 0; u < kPlanU; ++u) {
            const uint32_t t0 = base + 32 * u;  // warp-uniform
            if (t0 >= end) break;
            if (t0 >= c.tb1) c = plan_hap_of(p, t0);  // the warp moved into another haplotype
            const uint32_t tr = t0 + lane;
            const uint32_t len = raw[u].y, dst = raw[u].z;
            const bool whole = t0 + 32u <= min(c.tb1, end);  // warp-uniform: all 32 tasks exist and belong to c
            if (whole) {
                const uint32_t kt = plan_tile_of(p, c, dst);  // tile in which this task starts
                const uint32_t kprev = __shfl_sync(0xffffffffu, lane == 31u ? o_kt : kt, rot);
                const uint32_t p_dst = __shfl_sync(0xffffffffu, lane == 31u ? o_dst : dst, rot);
                const uint32_t p_len = __shfl_sync(0xffffffffu, lane == 31u ? o_len : len, rot);
                o_kt = kt, o_dst = dst, o_len = len;
                plan_one(p, c, raw[u], tr, kt, kprev, p_dst, p_len);
            } else {  // a haplotype boundary or the end of the range inside these 32 tasks: per-lane bases
                PlanHap m = c;
                if (tr >= c.tb1 && tr < end) m = plan_hap_of(p, tr);
                const uint32_t kt = plan_tile_of(p, m, dst);
                const uint32_t kprev = __shfl_sync(0xffffffffu, lane == 31u ? o_kt : kt, rot);
                const uint32_t p_dst = __shfl_sync(0xffffffffu, lane == 31u ? o_dst : dst, rot);
                const uint32_t p_len = __shfl_sync(0xffffffffu, lane == 31u ? o_len : len, rot);
                o_kt = kt, o_dst = dst, o_len = len;
                if (tr < end) plan_one(p, m, raw[u], tr, kt, kprev, p_dst, p_len);
            }
        }
    }
}

// One thread per haplotype, after k_plan_tasks: haplotypes flagged as unsorted / overlapping are compacted into
// ser_list[] (the work list of k_serial) and taken out of the tile kernel's view.  Their tasks wrote lb[] entries that
// mean nothing (lb[] is "first task at or after this tile" only for sorted input), and the tile kernel walks
// [lb[k]-1, lb[k+1]) -- so every tile boundary inside the haplotype's tape gets the entry it would have if the
// haplotype had no tasks at all: the first task BEHIND it.  (Its tasks wrote only entries of tiles in its own tape --
// plan_one writes (kprev, kt] and both are tiles of validated destinations of this haplotype -- so nothing outside
// needs repair.)  Two flagged neighbours may both write a shared boundary entry; either value is a valid bound.
__global__ void k_plan_fix(KParams p, unsigned int* ser_count) {
    const uint64_t h = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (h >= p.n_hap) return;
    const uint64_t o0 = p.out_base[h] - p.out_origin, o1 = p.out_base[h + 1] - p.out_origin;
    const bool flagged = p.hap_flags[h] != 0u;
    // a haplotype without tasks is all '.', one in serial order is left to the prefill by the tile kernel: every tile
    // that holds a byte of it needs the prefill
    if (o1 > o0 && (flagged || p.task_begin[h + 1] == p.task_begin[h]))
        for (uint64_t k = o0 >> p.tile_shift; k <= ((o1 - 1) >> p.tile_shift) && k < p.n_tiles; ++k) atomicOr(p.tile_hap + k, kTileHasGap);
    if (!flagged) return;
    p.ser_list[atomicAdd(ser_count, 1u)] = (uint32_t)h;
    const uint32_t tb1 = (uint32_t)min(p.task_begin[h + 1] - p.task_origin, p.n_tasks);
    const uint64_t k0 = (o0 + p.tile_bytes - 1) >> p.tile_shift, k1 = min(o1 >> p.tile_shift, p.n_tiles);
    for (uint64_t k = k0; k <= k1; ++k) p.lb[k] = tb1;
}

// ------------------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_addr(const void* ptr) { return (uint32_t)__cvta_generic_to_shared(ptr); }
// L2 policies: the result stream is written once and never re-read (evict_first), the reference tape / replicas are
// re-read by every haplotype (evict_last) -- keeps the proteome resident in the 126 MB L2 under a multi-GB write stream.
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void bulk_store_s2g(void* gdst, const void* ssrc, uint32_t bytes, uint64_t pol) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(gdst),
                 "r"(smem_addr(ssrc)), "r"(bytes), "l"(pol)
                 : "memory");
}
__device__ __forceinline__ void bulk_store_s2g_nohint(void* gdst, const void* ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_addr(ssrc)),
                 "r"(bytes)
                 : "memory");
}
// classic cp.async (LDGSTS): global -> shared without a destination register, completion by commit/wait groups
__device__ __forceinline__ void cp_async16(void* sdst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_addr(sdst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async8(void* sdst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_addr(sdst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async4(void* sdst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_addr(sdst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait0() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t mbar, uint32_t bytes) {
    asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t mbar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(mbar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
            : "=r"(ok)
            : "r"(mbar), "r"(parity)
            : "memory");
    } while (!ok);
}
// TMA bulk copy global -> shared, completion counted in bytes on an mbarrier (16-byte aligned both sides)
__device__ __forceinline__ void bulk_load_g2s(void* sdst, const void* gsrc, uint32_t bytes, uint32_t mbar, uint64_t pol) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_addr(sdst)),
        "l"(gsrc), "r"(bytes), "r"(mbar), "l"(pol)
        : "memory");
}
__device__ __forceinline__ void bulk_load_g2s_nohint(void* sdst, const void* gsrc, uint32_t bytes, uint32_t mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_addr(sdst)),
                 "l"(gsrc), "r"(bytes), "r"(mbar)
                 : "memory");
}
// dst = *p if pred (one byte, zero-extended), else dst keeps its value.  A predicated load INTO the caller's register:
// nothing consumes the loaded value here, so the warp does not wait for it (a C++ `if (c) x = __ldg(p)` that the
// compiler turns into load-to-temporary + move stalls on the move for the whole memory latency).
__device__ __forceinline__ void ldg_u8_if(uint32_t& dst, const uint8_t* p, bool pred) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q ld.global.nc.u8 %0, [%1];\n\t}" : "+r"(dst) : "l"(p), "r"((uint32_t)pred));
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// bytes [sh, sh+16) of the 32-byte little-endian concatenation A||B  (sh in [0,16))
__device__ __forceinline__ uint4 realign16(const uint4 A, const uint4 B, const uint32_t sh) {
    const bool k2 = (sh & 8u) != 0, k1 = (sh & 4u) != 0;
    const uint32_t x0 = k2 ? A.z : A.x, x1 = k2 ? A.w : A.y, x2 = k2 ? B.x : A.z, x3 = k2 ? B.y : A.w,
                   x4 = k2 ? B.z : B.x, x5 = k2 ? B.w : B.y;
    const uint32_t y0 = k1 ? x1 : x0, y1 = k1 ? x2 : x1, y2 = k1 ? x3 : x2, y3 = k1 ? x4 : x3, y4 = k1 ? x5 : x4;
    const uint32_t s = (sh & 3u) * 8u;
    uint4 r;
    r.x = __funnelshift_r(y0, y1, s);
    r.y = __funnelshift_r(y1, y2, s);
    r.z = __funnelshift_r(y2, y3, s);
    r.w = __funnelshift_r(y3, y4, s);
    return r;
}

// inclusive max-scan of the 4 bytes of a word (byte 0 = lowest address)
__device__ __forceinline__ uint32_t bytescan_max(uint32_t x) {
    x = __vmaxu4(x, x << 8);
    x = __vmaxu4(x, x << 16);
    return x;
}

// ------------------------------------------------------------------------------------------------ copy kernel
// Partial 16-byte vectors ("pieces") of a task.  Tasks are disjoint and sorted, so in any output vector at most one
// piece starts at byte 0 and ends inside (T: the tail of a task that came in from the left), at most one starts inside
// and ends at byte 16 (H: the head of a task that continues to the right), and any number lie strictly inside (M).
// T and H pieces are merged as whole vectors: source fetched with (at most) two aligned 16-byte loads, realigned in
// registers, then  new = (old & ~mask) | (val & mask)  on the shared-memory tile; the two classes run in separate
// warp-synchronous passes so no two lanes ever read-modify-write the same vector at once.  M pieces (a 1-residue
// missense patch, typically) are byte copies after both passes.
struct Piece {
    uint4 A, B;
    uint32_t sh;
};
// bytes [a,b) of tile vector vx come from p0 + 16*vx + [a,b)
__device__ __forceinline__ Piece piece_load(const long long p0, const int vx, const int a, const int b, const bool on) {
    Piece pc;
    const unsigned long long sa = (unsigned long long)(p0 + (long long)vx * 16);
    pc.sh = (uint32_t)sa & 15u;
    const uint4* ap = reinterpret_cast<const uint4*>(sa - pc.sh);
    pc.A = make_uint4(0u, 0u, 0u, 0u);
    pc.B = pc.A;
    if (on && a < 16 - (int)pc.sh) pc.A = __ldg(ap);      // some valid byte lives in the first aligned chunk
    if (on && b > 16 - (int)pc.sh) pc.B = __ldg(ap + 1);  // ... in the second one (implies sh != 0)
    return pc;
}
// lo16[x] = 16-byte mask whose first x bytes are 0xFF (x = 0..16), staged in shared memory
__device__ __forceinline__ void piece_merge(uint8_t* __restrict__ tile, const uint4* __restrict__ lo16, const uint4 r,
                                            const int vx, const int nlow, const bool keep_low) {
    // r: the piece's source vector, realigned; keep_low: the piece is [nlow,16) (H) -> old bytes below nlow are kept;
    // else the piece is [0,nlow) (T)
    const uint4 m = lo16[nlow];
    uint4* dst = reinterpret_cast<uint4*>(tile) + vx;
    const uint4 o = *dst;
    uint4 n;
    if (keep_low) {
        n.x = (o.x & m.x) | (r.x & ~m.x), n.y = (o.y & m.y) | (r.y & ~m.y);
        n.z = (o.z & m.z) | (r.z & ~m.z), n.w = (o.w & m.w) | (r.w & ~m.w);
    } else {
        n.x = (r.x & m.x) | (o.x & ~m.x), n.y = (r.y & m.y) | (o.y & ~m.y);
        n.z = (r.z & m.z) | (o.z & ~m.z), n.w = (r.w & m.w) | (o.w & ~m.w);
    }
    *dst = n;
}

// ---- the register path of the copy kernel, out of line.  With a registered reference tape (TMA mode) these run for
// out-of-phase alteration payloads only; kept out of the tile loop's body they do not count against its register
// budget (80 registers at 3 CTAs/SM, and every spilled value there costs a local-memory round trip per tile).

// The short out-of-phase runs of a batch (alteration payloads of up to kLaneRunBytes, typically), copied by the WHOLE
// warp: lane i brings its run's vectors [v0, v1) (none: v0 == v1); a warp scan numbers all vectors of all runs, and
// every round 32 of them are fetched by 32 lanes -- each finds the run its vector belongs to by a 5-step binary search
// over the scanned counts (shuffles), then two aligned loads, funnel-shift realign, one 16-byte store.  (Round 1 had
// every lane copy its own run: a 400-byte frameshift tail kept one lane busy for seven dependent load rounds while 31
// waited -- on the skew stress that serial tail cost more than everything else in the tile.)
__device__ __noinline__ void coop_run_copy(uint8_t* __restrict__ tile, const long long p0, const int v0, const int v1, const int lane) {
    const uint32_t full = 0xffffffffu;
    const uint32_t cnt = (uint32_t)(v1 - v0);
    uint32_t incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(full, incl, d);
        if (lane >= d) incl += o;
    }
    const uint32_t total = __shfl_sync(full, incl, 31), excl = incl - cnt;
    const uint32_t p0lo = (uint32_t)(unsigned long long)p0, p0hi = (uint32_t)((unsigned long long)p0 >> 32);
    uint4* const tv = reinterpret_cast<uint4*>(tile);
    for (uint32_t j0 = 0; j0 < total; j0 += 64) {  // two vectors per lane and round: four loads in flight
        uint4 A[2], B[2];
        uint32_t shv[2];
        int vv[2];
        bool on[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const uint32_t j = j0 + 32u * u + (uint32_t)lane;
            uint32_t o = 0;  // smallest lane whose inclusive count exceeds j = the run vector j belongs to
#pragma unroll
            for (int step = 16; step; step >>= 1) {
                const uint32_t probe = __shfl_sync(full, incl, (int)(o + step - 1));
                if (probe <= j) o += step;
            }
            o = min(o, 31u);
            const uint32_t oex = __shfl_sync(full, excl, (int)o), ov0 = __shfl_sync(full, (uint32_t)v0, (int)o);
            const uint32_t qlo = __shfl_sync(full, p0lo, (int)o), qhi = __shfl_sync(full, p0hi, (int)o);
            on[u] = j < total;
            vv[u] = (int)(ov0 + (j - oex));
            const unsigned long long sa = (((unsigned long long)qhi << 32) | qlo) + (unsigned long long)((long long)vv[u] * 16);
            shv[u] = (uint32_t)sa & 15u;
            const uint4* ap = reinterpret_cast<const uint4*>(sa - shv[u]);
            A[u] = make_uint4(0u, 0u, 0u, 0u);
            if (on[u]) A[u] = __ldg(ap);
            B[u] = A[u];
            if (on[u] && shv[u]) B[u] = __ldg(ap + 1);
        }
#pragma unroll
        for (int u = 0; u < 2; ++u)
            if (on[u]) tv[vv[u]] = realign16(A[u], B[u], shv[u]);
    }
}

// B: owner of every vector = last task (of this batch) whose covered range started at or before it (warp max-scan over
// lead[]); C: one lane per fully covered 16-byte vector, loads of G vectors issued before any is used.  Whole warp.
template <int TILE, int G>
__device__ __noinline__ void owner_scan_copy(uint8_t* __restrict__ tile, uint8_t* __restrict__ lead, const long long p0,
                                             const uint32_t v1, const int lane) {
    constexpr int NV = TILE / 16, LWW = NV / 32 / 4;
    {
        uint32_t wv[LWW];
        uint32_t top = 0;
#pragma unroll
        for (int w = 0; w < LWW; ++w) {  // inclusive max-scan over this lane's LW owner bytes
            wv[w] = bytescan_max(reinterpret_cast<uint32_t*>(lead)[lane * LWW + w]);
            wv[w] = __vmaxu4(wv[w], top * 0x01010101u);
            top = wv[w] >> 24;
        }
        uint32_t incl = top;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t o = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl = max(incl, o);
        }
        uint32_t excl = __shfl_up_sync(0xffffffffu, incl, 1);
        if (lane == 0) excl = 0;
        const uint32_t bc = excl * 0x01010101u;
#pragma unroll
        for (int w = 0; w < LWW; ++w) reinterpret_cast<uint32_t*>(lead)[lane * LWW + w] = __vmaxu4(wv[w], bc);
    }
    __syncwarp();
    const uint32_t p0lo = (uint32_t)(unsigned long long)p0, p0hi = (uint32_t)((unsigned long long)p0 >> 32);
#pragma unroll
    for (int r0 = 0; r0 < NV / 32; r0 += G) {
        uint4 A[G], B[G];
        uint32_t shv[G];
        bool on[G];
#pragma unroll
        for (int i = 0; i < G; ++i) {
            const int v = lane + 32 * (r0 + i);
            const uint32_t owner = lead[v];
            const int srcl = (int)((owner - 1u) & 31u);
            const uint32_t qlo = __shfl_sync(0xffffffffu, p0lo, srcl);
            const uint32_t qhi = __shfl_sync(0xffffffffu, p0hi, srcl);
            const uint32_t qv1 = __shfl_sync(0xffffffffu, v1, srcl);
            on[i] = owner != 0u && (uint32_t)v < qv1;
            const unsigned long long sa = (((unsigned long long)qhi << 32) | qlo) + (unsigned long long)(v * 16);
            shv[i] = (uint32_t)sa & 15u;
            const uint4* ap = reinterpret_cast<const uint4*>(sa - shv[i]);
            A[i] = make_uint4(0u, 0u, 0u, 0u);
            if (on[i]) A[i] = __ldg(ap);
            B[i] = A[i];
            if (on[i] && shv[i]) B[i] = __ldg(ap + 1);
        }
#pragma unroll
        for (int i = 0; i < G; ++i) {
            const int v = lane + 32 * (r0 + i);
            if (on[i]) reinterpret_cast<uint4*>(tile)[v] = realign16(A[i], B[i], shv[i]);
        }
    }
}

constexpr int kLaneRunBytes = 512;  // out-of-phase runs up to this many fully covered bytes go to coop_run_copy (longer: owner scan)
constexpr int kTileScratch = 16 + 576 + 64 + 16;  // per warp, behind tile | lead[]: mbarrier | staged tasks (32 x 16 B) + bases /
                                                  // flag (8 x 8 B) | metadata ring (4 x {tile, lb[k], lb[k+1], tile_hap[k]}) |
                                                  // slot scheduler state (4 x u32)
constexpr uint32_t kSlotEmpty = 0xFFFFFFFFu, kSlotEnd = 0xFFFFFFFEu;  // ring sentinels: no tile in this slot / no slot left
constexpr uint32_t kDynBlock = 8;      // most slots claimed per atomic in the dynamic tail
constexpr uint32_t kStaticNum = 3, kStaticDen = 4;  // share of the slots handed out statically (round-robin)

// TILE: output bytes per warp-tile; G: vectors per lane whose loads are issued back to back (memory-level
// parallelism); MINB: CTAs per SM the register allocation is held to.
// FLAGS: 1 = L2 cache-policy hints; 2 = haplotype-interleaved tile order (see below).
template <int TILE, int G, int MINB, int FLAGS>
__global__ void __launch_bounds__(kThreads, MINB) k_copy_tiles(const KParams p) {
    constexpr bool kHints = (FLAGS & 1) != 0;
    constexpr bool kOrder = (FLAGS & 2) != 0;
    constexpr int NV = TILE / 16;   // 16-byte vectors per tile
    constexpr int LW = NV / 32;     // lead[] bytes per lane in the scan (4, 8 or 16)
    constexpr int LWW = LW / 4;     // ... as 32-bit words
    constexpr int STRIDE = TILE + NV + kTileScratch;
    static_assert(LW == 4 || LW == 8 || LW == 16, "TILE must be 2048, 4096 or 8192");
    extern __shared__ __align__(128) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t* const tile = smem + warp * STRIDE;
    uint8_t* const lead = tile + TILE;
    const uint32_t mbar = smem_addr(tile + TILE + NV);
    uint32_t mbar_phase = 0;
    uint4* const st_tasks = reinterpret_cast<uint4*>(tile + TILE + NV + 16);
    uint64_t* const st_bases = reinterpret_cast<uint64_t*>(tile + TILE + NV + 16 + 512);
    uint32_t* const st_meta = reinterpret_cast<uint32_t*>(tile + TILE + NV + 16 + 576);
    uint4* const lo16 = reinterpret_cast<uint4*>(smem + kWarpsPerCta * STRIDE);  // 17 masks, shared by the CTA
    if (threadIdx.x < 17 * 4) {
        const int x = threadIdx.x >> 2, w = threadIdx.x & 3, nb = min(max(x - 4 * w, 0), 4);
        reinterpret_cast<uint32_t*>(lo16)[threadIdx.x] = nb == 4 ? 0xFFFFFFFFu : ((1u << (8 * nb)) - 1u);
    }
    __syncthreads();

    if (p.status->bad_args || p.status->err_key != ~0ull || p.status->gap_key != ~0ull || p.status->stream_key != ~0ull)
        return;
    if (lane == 0) mbar_init(mbar, 1);
    if (p.warp_ns && lane == 0) {  // load-balance evidence (SURVEY 8d C4): when did this warp start (kept in shared memory)
        unsigned long long t;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
        st_bases[6] = t;
    }
    __syncwarp();

    const uint32_t n_warps = gridDim.x * kWarpsPerCta;
    const uint64_t pol_stream = l2_policy_evict_first(), pol_keep = l2_policy_evict_last();
    const uint4 fillv = make_uint4(p.fill_word, p.fill_word, p.fill_word, p.fill_word);

    // Processing order (FLAGS & 2).  A warp's successive tiles are NOT neighbours on the tape: slot
    // ((g * n_hap + h) << gshift) + i is tile i of group g of haplotype h, so the ~3.5k warps in flight sit at the same
    // relative position of ~3.5k different haplotypes.  Every haplotype's tape follows the proteome's transcript order,
    // so at any moment the whole GPU reads one narrow band of the proteome (times 16 replicas) -- it stays in L2 however
    // large the replica set is -- instead of sweeping all 171 MB of it once per ~9 haplotypes.  Slots without a tile
    // (shorter haplotypes) hold ~0.  Without the flag, slots are tiles in tape order (phase-aligned layouts, whose
    // runs come from the one plain tape, gain nothing from the interleave).
    // (tiles and order slots of one launch stay below 2^32 - 2^20: checked by the host).  The slot count lives in this
    // warp's shared-memory scratch, not in a register: the tile loop is out of registers, and a spilled loop bound is
    // reloaded from LOCAL memory behind the queue of cp.async requests (8 % of all stall samples before this).
    {
        uint32_t ns32 = (uint32_t)p.n_tiles;
        if constexpr (kOrder) {
            const uint64_t ns = tile_order_slots(p, __ldg(p.order_hdr));
            if (ns) ns32 = (uint32_t)ns;  // else order[] is the identity over n_tiles
        }
        if (lane == 0) *reinterpret_cast<uint32_t*>(st_bases + 7) = ns32;
        __syncwarp();
    }
    const volatile uint32_t* const n_slots_p = reinterpret_cast<const volatile uint32_t*>(st_bases + 7);
#define n_slots (*n_slots_p)
    // Software pipeline over this warp's slots, three dependent fetches deep, all of them cp.async into a 4-entry ring
    // in shared memory (no register is carried from tile to tile, and nobody waits on a load it issued for later):
    //   iteration i   waits for everything issued at i-1, then issues
    //     stage(i+1)       first 32 tasks + the owning haplotype's bases / serial flag   <- needs meta(i+1)
    //     fetch_meta(i+2)  lb[k], lb[k+1], tile_hap[k]                                   <- needs tile(i+2)
    //     fetch_tile(i+3)  order[slot]  (interleaved order; tape order: slot itself)
    // A ring entry is {tile (~0: none), lb[k], lb[k+1], tile_hap[k]}.
    const uint32_t n_tasks32 = (uint32_t)p.n_tasks;  // < 2^32 - 1 (checked by the host)
    auto first_task = [&](uint32_t lo) -> uint32_t {
        const uint32_t t = min(lo, n_tasks32);
        return t > 0u ? t - 1u : 0u;  // the task before may extend into the tile
    };
    auto ring = [&](uint32_t it) -> uint32_t* { return st_meta + ((it & 3u) << 2); };
    // Which slot comes next for this warp.  The first 3/4 of the slots go round-robin over the warps (slot = warp + i *
    // n_warps: at any moment the whole grid works on one band of the slot order, which is what keeps the proteome band
    // in L2); the rest is claimed kDynBlock slots at a time from a global counter.  Without the dynamic tail the grid
    // finished ragged -- the warp schedulers favour the older CTAs of an SM, whose warps were done 8 % before the
    // youngest CTA's, which then ran the tail at a third of the occupancy (profiles/dev/warp_time_probe.py).
    // State (lane 0 only, in the warp's scratch): {next static slot, next claimed slot, claimed slots left, n_static}.
    volatile uint32_t* const sched = reinterpret_cast<volatile uint32_t*>(tile + TILE + NV + 16 + 576 + 64);
    if (lane == 0) {
        const uint32_t ns = n_slots;
        sched[0] = blockIdx.x * kWarpsPerCta + warp;
        sched[1] = 0u, sched[2] = 0u;
        sched[3] = (uint32_t)((uint64_t)ns * kStaticNum / kStaticDen / n_warps) * n_warps;
    }
    auto fetch_tile = [&](uint32_t it) {
        if (lane == 0) {
            uint32_t* m = ring(it);
            uint32_t slot = sched[0];
            const uint32_t n_static = sched[3];
            if (slot < n_static) {
                sched[0] = slot + n_warps;
            } else {
                uint32_t left = sched[2];
                slot = sched[1];
                if (left == 0u) {  // (the counter only grows past n_slots by one block per warp: no wrap)
                    // block size: kDynBlock when every warp can expect several blocks, down to single slots for a small
                    // launch (a 100 MB batch is three tiles per warp: an 8-slot claim would triple one warp's share)
                    const uint32_t ns = n_slots;
                    const uint32_t blk = max(1u, min(kDynBlock, (ns - n_static) / (4u * n_warps)));
                    slot = n_static + atomicAdd(p.order_hdr + 1, blk);
                    left = blk;
                    if (slot >= ns) left = 0xFFFFFFFFu;  // nothing left anywhere: stop asking
                }
                sched[1] = slot + 1u, sched[2] = left - 1u;
            }
            if (slot >= n_slots) m[0] = kSlotEnd;
            else if constexpr (kOrder) cp_async4(m, p.order + slot);
            else m[0] = slot;
        }
    };
    auto fetch_meta = [&](uint32_t it) {
        uint32_t* m = ring(it);
        const uint32_t t = m[0];
        if (lane < 3) {
            if (t >= kSlotEnd) m[1 + lane] = 0u;
            else cp_async4(m + 1 + lane, lane == 2 ? p.tile_hap + t : p.lb + t + lane);
        }
    };
    auto stage = [&](uint32_t it) {
        const uint32_t* m = ring(it);
        if (m[0] >= kSlotEnd) return;
        const uint32_t lo = m[1], hi = m[2], hp = m[3] & ~kTileHasGap;
        const uint32_t tr = first_task(lo) + lane;
        if (tr < min(hi, n_tasks32)) cp_async16(st_tasks + lane, reinterpret_cast<const uint4*>(p.tasks) + tr);
        // lanes 0-5: the owning haplotype's bases task_begin[h], task_begin[h+1], out_base[h], alt_base[h], ref_base[h]
        // and its serial-order flag (spelled out per lane: a lane-dependent array pointer kept in registers across the
        // tile loop is what used to spill)
        if (lane == 0) cp_async8(st_bases + 0, p.task_begin + hp);
        if (lane == 1) cp_async8(st_bases + 1, p.task_begin + hp + 1);
        if (lane == 2) cp_async8(st_bases + 2, p.out_base + hp);
        if (lane == 3) cp_async8(st_bases + 3, p.alt_base + hp);
        if (lane == 4 && p.ref_base) cp_async8(st_bases + 4, p.ref_base + hp);
        if (lane == 5) cp_async4(st_bases + 5, p.hap_flags + hp);  // 1: the haplotype is left to k_serial
    };
    __syncwarp();
    fetch_tile(0), fetch_tile(1), fetch_tile(2);
    cp_async_commit();
    cp_async_wait0();
    __syncwarp();
    fetch_meta(0), fetch_meta(1);
    cp_async_commit();
    cp_async_wait0();
    __syncwarp();
    stage(0);
    cp_async_commit();
    for (uint32_t it = 0;; ++it) {
        // this tile's tasks and bases were staged while the previous tile was being assembled
        cp_async_wait0();
        __syncwarp();
        const uint32_t* const mc = ring(it);
        const uint32_t tile_no = mc[0];  // kSlotEmpty = an empty slot of the interleaved order
        if (tile_no == kSlotEnd) break;  // (nothing is in flight: the ring entries behind an end marker are end markers)
        const uint32_t c_lo = mc[1], c_hi = mc[2];
        const bool has_gap = (mc[3] & kTileHasGap) != 0u;  // some byte of the tile is written by nobody: prefill it
        const uint4 raw0 = st_tasks[lane];
        // warp-uniform bases of the haplotype that owns the tile's first byte (the common case for every task here)
        // (launch-relative 32-bit task numbers; the tape bases folded into what a task needs: where the haplotype's
        // result tape starts relative to this tile, and where its two source tapes start)
        const uint32_t hb_t0 = (uint32_t)(st_bases[0] - p.task_origin), hb_t1 = (uint32_t)min(st_bases[1] - p.task_origin, p.n_tasks);
        const uint64_t hb_out = st_bases[2];
        const uint8_t* const hb_altp = p.alt + (st_bases[3] - p.alt_origin);
        const uint8_t* const hb_refp = p.ref + ((p.ref_base ? st_bases[4] : p.ref_origin) - p.ref_origin);
        const bool hb_serial = *reinterpret_cast<const uint32_t*>(st_bases + 5) != 0u;
        __syncwarp();
        stage(it + 1);
        fetch_meta(it + 2);
        fetch_tile(it + 3);
        cp_async_commit();
        if (tile_no == kSlotEmpty) continue;
        const uint64_t tile_start = (uint64_t)tile_no * (uint64_t)TILE;
        const uint32_t tile_len = (uint32_t)min((uint64_t)TILE, p.n_out - tile_start);
        uint8_t* const gout = p.out + tile_start;
        const long long hb_rel = (long long)(hb_out - p.out_origin) - (long long)tile_start;  // tape start - tile start
        const uint32_t t_lo = first_task(c_lo);
        const uint32_t t_hi = min(c_hi, n_tasks32);
        // the second batch of tasks (tiles of more than 32) is requested now and consumed after the first batch
        const uint4 raw1 = t_lo + 32u + lane < t_hi ? __ldg(reinterpret_cast<const uint4*>(p.tasks) + t_lo + 32u + lane)
                                                    : make_uint4(0u, 0u, 0u, 0u);

        // the previous tile's bulk store must have finished READING shared memory before we overwrite it
        if (lane == 0) bulk_wait_read0();
        __syncwarp();

        // prefill: '.' (haplotype_instruction.rs:78) -- only where the plan found a byte that no task covers (round 2: a
        // third of the tile's shared-memory traffic for nothing otherwise) -- or the caller's current content
        if (!p.keep_out) {
            if (has_gap) {
#pragma unroll
                for (int i = 0; i < NV / 32; ++i) reinterpret_cast<uint4*>(tile)[lane + 32 * i] = fillv;
            }
        } else {
#pragma unroll
            for (int i = 0; i < NV / 32; ++i) {
                int v = lane + 32 * i;
                if ((uint32_t)(v * 16 + 16) <= tile_len) {
                    reinterpret_cast<uint4*>(tile)[v] = *reinterpret_cast<const uint4*>(gout + v * 16);
                } else {
                    for (int b = 0; b < 16; ++b)
                        if ((uint32_t)(v * 16 + b) < tile_len) tile[v * 16 + b] = gout[v * 16 + b];
                }
            }
        }
#pragma unroll
        for (int w = 0; w < LWW; ++w) reinterpret_cast<uint32_t*>(lead)[lane * LWW + w] = 0u;
        fence_async_smem();  // the prefill must be ordered before TMA loads land in the same bytes
        __syncwarp();
        bool tma_used = false;
        // 1-residue patches of fused chains (below), first / second batch of the tile: bit 31 of pd = armed, low bits =
        // tile offset; pv = the byte.  They are applied after the chain's TMA load has landed (phase D).
        uint32_t pv0 = 0, pd0 = 0, pv1 = 0, pd1 = 0;

        for (uint32_t tb = t_lo; tb < t_hi; tb += 32) {
            // ---- A: one lane per task: partial head/tail vectors, and the start of its fully covered vector range
            const uint32_t tr = tb + lane;
            long long p0 = 0;   // source address of tile byte 0 for this task (may point before the segment)
            uint32_t v1 = 0;    // end (exclusive) of the fully covered vector range, in vectors
            uint32_t tma_bytes = 0, tma_dst = 0;  // fully covered range served by a TMA bulk copy from a replica
            const uint8_t* tma_src = nullptr;
            bool tma_alt = false;  // alteration payloads are read once (evict_first), reference runs are re-read (evict_last)
            bool has_lead = false, onT = false, onH = false, onM = false;
            int lane_v0 = 0, lane_v1 = 0;  // fully covered vectors of a short out-of-phase run, copied by this lane
            int pvh = 0, pvt = 0, pa1 = 0, pb2 = 16;
            uint4 raw = make_uint4(0u, 0u, 0u, 0u);
            int s = 0, e = 0;       // this task clipped to the tile; e > s: something to do
            bool main_hap = false;  // the task belongs to the haplotype that owns the tile's first byte
            if (tr < t_hi) {
                raw = tb == t_lo ? raw0 : tb == t_lo + 32u ? raw1 : __ldg(reinterpret_cast<const uint4*>(p.tasks) + tr);
                long long rel = hb_rel;
                const uint8_t *altp = hb_altp, *refp = hb_refp;
                bool serial = hb_serial;
                main_hap = tr >= hb_t0 && tr < hb_t1;
                if (!main_hap) {  // another haplotype (tile spans a haplotype boundary)
                    const uint64_t h = upper_bound_u64(p.task_begin, 0, p.n_hap + 1, tr + p.task_origin) - 1;
                    rel = (long long)(__ldg(p.out_base + h) - p.out_origin) - (long long)tile_start;
                    altp = p.alt + (__ldg(p.alt_base + h) - p.alt_origin);
                    refp = p.ref + ((p.ref_base ? __ldg(p.ref_base + h) : p.ref_origin) - p.ref_origin);
                    serial = __ldg(p.hap_flags + h) != 0u;
                }
                const long long g = rel + raw.z;
                const long long ge = g + raw.y;
                s = (int)max(g, 0ll), e = (int)min(ge, (long long)tile_len);
                if (e > s && !serial) {  // (a haplotype in serial order keeps its prefill here; k_serial paints it)
                    p0 = (long long)((raw.w ? altp : refp) + raw.x) - g;
                } else {
                    s = e = 0;
                }
            }
            // ---- A': chain fusion.  `R A R` -- two reference runs with the same (source - destination) offset and a
            // 1-residue alteration exactly filling the hole between them (a missense patch, transcript_instructions.rs
            // :654-663) -- is one reference run with one byte replaced afterwards.  The reference lanes of such a chain
            // (lanes i, i+2, i+4, ... of this batch) collapse into its first lane, whose extent grows to the end of the
            // last one; the patch lanes keep one byte each for phase D.  Fewer, longer bulk copies and no partial-vector
            // work around the patches.  (First two batches of a tile only: the patch registers are per batch.)
            if (tb - t_lo < 64u) {
                const uint32_t full = 0xffffffffu;
                const bool ok = e > s && main_hap;
                const uint32_t prev_end = __shfl_up_sync(full, raw.z + raw.y, 1);
                const uint32_t delta = raw.x - raw.z, delta2 = __shfl_up_sync(full, delta, 2);
                const uint32_t Bref = __ballot_sync(full, ok && raw.w == 0u);
                const uint32_t Bpat = __ballot_sync(full, ok && raw.w == 1u && raw.y == 1u);
                const uint32_t Bc = __ballot_sync(full, lane > 0 && raw.z == prev_end);  // starts where the lane before ends
                const uint32_t Bb = __ballot_sync(full, raw.x < raw.z);                  // (33rd bit of source - destination)
                const uint32_t Bd = __ballot_sync(full, lane > 1 && delta == delta2);
                const uint32_t link = Bref & (Bref << 2) & (Bpat << 1) & Bc & (Bc << 1) & ~(Bb ^ (Bb << 2)) & Bd;
                if (link) {  // (warp-uniform)
                    const bool cont = (link >> lane) & 1u;                           // linked to the reference lane two below
                    const bool patch = lane < 31 && ((link >> (lane + 1)) & 1u);   // the byte between two linked runs
                    uint32_t tail = lane;
                    if (lane < 30 && !cont) tail = lane + (uint32_t)__ffs((int)~((link >> (lane + 2)) | 0xAAAAAAAAu)) - 1u;
                    const int e_tail = __shfl_sync(full, e, tail);
                    const bool first = tb == t_lo;
                    const uint8_t* sp = reinterpret_cast<const uint8_t*>(p0 + s);
                    ldg_u8_if(pv0, sp, patch && first);
                    ldg_u8_if(pv1, sp, patch && !first);
                    if (patch && first) pd0 = 0x80000000u | (uint32_t)s;
                    if (patch && !first) pd1 = 0x80000000u | (uint32_t)s;
                    if (cont || patch) s = e = 0;  // nothing else to do for these lanes
                    else if (e > s) e = e_tail;
                }
            }
            if (e > s) {
                // Source in phase with the destination: the tape itself, or for an out-of-phase reference run with a
                // registered tape the replica r = (-q) mod 16 that holds it at the output's 16-byte phase; then the
                // fully covered vectors are ONE TMA bulk copy and the partial ones single aligned loads.
                if ((p0 & 15) != 0 && p.tma_mode && raw.w == 0u) {
                    const long long q = p0 - (long long)p.ref;  // ref offset of tile byte 0
                    const uint32_t r = (uint32_t)(-q) & 15u;
                    p0 = (long long)(p.ref_rep + (uint64_t)r * p.rep_stride + r) + q;
                }
                const int vh = s >> 4, vt = (e - 1) >> 4;
                const int v0b = (s + 15) & ~15, v1b = e & ~15;
                if (v1b > v0b) {
                    if ((p0 & 15) == 0) {
                        tma_src = reinterpret_cast<const uint8_t*>(p0 + v0b);
                        tma_alt = raw.w != 0u;
                        tma_dst = (uint32_t)v0b;
                        tma_bytes = (uint32_t)(v1b - v0b);
                    } else if (v1b - v0b <= kLaneRunBytes) {
                        // a short out-of-phase run (an alteration payload, typically): all such runs of the batch are
                        // copied by the warp together, below -- cheaper than the whole-tile owner scan for a few vectors
                        lane_v0 = v0b >> 4, lane_v1 = v1b >> 4;
                    } else {
                        lead[v0b >> 4] = (uint8_t)(lane + 1);
                        v1 = (uint32_t)(v1b >> 4);
                        has_lead = true;
                    }
                }
                // classify the partial vectors (see Piece): H = [a1,16) of vh, T = [0,b2) of vt, M = [a1,b1) of vh
                pvh = vh, pvt = vt;
                pa1 = s & 15, pb2 = e - (vt << 4);
                if (vt > vh) {
                    onH = pa1 != 0;
                    onT = pb2 != 16;
                } else if (pa1 != 0 || pb2 != 16) {  // the whole (clipped) task sits inside one vector
                    if (pa1 == 0) onT = true;
                    else if (pb2 == 16) onH = true;
                    else onM = true;
                }
            }
            // The loads of the partial vectors go out first, so that their latency runs under the (serial, one elected
            // lane at a time) issue of the TMA bulk loads; nothing consumes them before that loop is through.
            const Piece pcT = piece_load(p0, pvt, 0, pb2, onT), pcH = piece_load(p0, pvh, pa1, 16, onH);
            uint32_t m_first = 0;  // first byte of a piece strictly inside one vector (a 1-residue task, typically)
            ldg_u8_if(m_first, reinterpret_cast<const uint8_t*>(p0) + (pvh << 4) + pa1, onM);
            {
                const uint32_t total = __reduce_add_sync(0xffffffffu, tma_bytes);
                if (total) {
                    if (lane == 0) mbar_expect_tx(mbar, total);
                    __syncwarp();
                    if (tma_bytes) {
                        if (kHints)
                            bulk_load_g2s(tile + tma_dst, tma_src, tma_bytes, mbar, tma_alt ? pol_stream : pol_keep);
                        else
                            bulk_load_g2s_nohint(tile + tma_dst, tma_src, tma_bytes, mbar);
                    }
                    tma_used = true;
                }
            }
            {
                // (with a registered tape every reference piece comes from the in-phase replica: shift 0, nothing to realign)
                const bool shifted = __any_sync(0xffffffffu, (onT && pcT.sh != 0u) || (onH && pcH.sh != 0u));
                if (onT) piece_merge(tile, lo16, shifted ? realign16(pcT.A, pcT.B, pcT.sh) : pcT.A, pvt, pb2, false);
                __syncwarp();
                if (onH) piece_merge(tile, lo16, shifted ? realign16(pcH.A, pcH.B, pcH.sh) : pcH.A, pvh, pa1, true);
                __syncwarp();
                if (onM) {
                    const uint8_t* __restrict__ sp = reinterpret_cast<const uint8_t*>(p0) + (pvh << 4);
                    uint8_t* d = tile + (pvh << 4);
                    d[pa1] = (uint8_t)m_first;
                    for (int j = pa1 + 1; j < pb2; ++j) d[j] = __ldg(sp + j);
                }
            }
            if (__any_sync(0xffffffffu, lane_v1 > lane_v0)) coop_run_copy(tile, p0, lane_v0, lane_v1, lane);  // (warp-uniform)
            __syncwarp();  // orders this batch's tile stores before the next batch's read-modify-writes
            if (!__any_sync(0xffffffffu, has_lead)) continue;  // nothing for the register path in this batch

            // ---- B, C: owner scan over lead[], then one lane per fully covered vector (register path, out of line)
            owner_scan_copy<TILE, G>(tile, lead, p0, v1, lane);
            __syncwarp();
            if (tb + 32u < t_hi) {  // another batch follows: reset lead[]
#pragma unroll
                for (int w = 0; w < LWW; ++w) reinterpret_cast<uint32_t*>(lead)[lane * LWW + w] = 0u;
                __syncwarp();
            }
        }

        // ---- D: publish the tile (after every TMA load of this tile has landed)
        if (tma_used) {
            if (lane == 0) mbar_arrive(mbar);
            mbar_wait(mbar, mbar_phase);
            mbar_phase ^= 1u;
        }
        if (pd0 >> 31) tile[pd0 & 0xFFFFu] = (uint8_t)pv0;  // the patches of fused chains, over the landed reference bytes
        if (pd1 >> 31) tile[pd1 & 0xFFFFu] = (uint8_t)pv1;
        fence_async_smem();
        __syncwarp();
        const uint32_t bulk = tile_len & ~15u;
        if (lane == 0 && bulk) {
            if (kHints)
                bulk_store_s2g(gout, tile, bulk, pol_stream);
            else
                bulk_store_s2g_nohint(gout, tile, bulk);
            bulk_commit();
        }
        if (bulk + lane < tile_len) gout[bulk + lane] = tile[bulk + lane];  // < 16 trailing bytes of the whole output
    }
    if (lane == 0) bulk_wait0();
    if (p.warp_ns && lane == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
        p.warp_ns[blockIdx.x * kWarpsPerCta + warp] = t - st_bases[6];
    }
#undef n_slots
}

// ------------------------------------------------------------------------------------------------ serial order
// Reference order semantics (gir.rs:233: tasks applied strictly in array order, a later task overwrites an earlier
// one) for the haplotypes the plan flagged as unsorted / overlapping -- and only for those; everybody else was
// written by the tile kernel.  Output-stationary like the tile kernel, so one odd haplotype is spread over the
// whole GPU instead of one CTA: a work item is a kSerialSpan-byte span of one flagged haplotype's result tape.  The
// CTA prefills its span, then walks ALL of the haplotype's tasks in array order (kSerialThreads per step, one
// coalesced load; the next window is in flight while this one is judged) and applies the ones that overlap the
// span, clipped to it, one after the other.  Every byte therefore sees its writers in array order, with no
// inter-CTA ordering needed; the price is that every span re-reads the haplotype's task array (L2-resident, ~20k
// tasks), which is why this is not the main path.
// Launched by the host only after the plan reported `unsorted` and no error, when the call is waited -- possibly after
// later asynchronous launches on the same stream have reused the engine's scratch.  So nothing here is read from that
// scratch: the count is passed by value, and ser_list belongs to the launch (its event, or its single-haplotype slot).
constexpr int kSerialThreads = 512;
constexpr uint32_t kSerialSpan = 16384;
__global__ void __launch_bounds__(kSerialThreads) k_serial(const KParams p, const uint32_t n_ser) {
    __shared__ uint32_t s_cnt[kSerialThreads / 32];
    __shared__ const uint8_t* s_src[kSerialThreads];
    __shared__ uint32_t s_dst[kSerialThreads], s_len[kSerialThreads];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    for (uint32_t i = 0; i < n_ser; ++i) {
        const uint64_t h = p.ser_list[i];
        const uint64_t o0 = p.out_base[h] - p.out_origin, n_res = p.out_base[h + 1] - p.out_base[h];
        uint8_t* const res = p.out + o0;
        const uint8_t* const ref = p.ref + (p.ref_base ? p.ref_base[h] - p.ref_origin : 0ull);
        const uint8_t* const alt = p.alt + (p.alt_base[h] - p.alt_origin);
        const uint64_t t0 = p.task_begin[h] - p.task_origin, t1 = p.task_begin[h + 1] - p.task_origin;
        const uint64_t n_spans = (n_res + kSerialSpan - 1) / kSerialSpan;
        const uint4* __restrict__ tk = reinterpret_cast<const uint4*>(p.tasks);
        for (uint64_t j = blockIdx.x; j < n_spans; j += gridDim.x) {
            const uint64_t r0 = j * kSerialSpan, r1 = min(r0 + kSerialSpan, n_res);
            if (!p.keep_out)
                for (uint64_t x = r0 + tid; x < r1; x += kSerialThreads)
                    res[x] = (uint8_t)(p.fill_word >> (8u * (uint32_t)((o0 + x) & 3u)));
            uint4 nxt = t0 + tid < t1 ? __ldg(tk + t0 + tid) : make_uint4(0u, 0u, 0u, 0u);
            for (uint64_t t = t0; t < t1; t += kSerialThreads) {
                const uint4 raw = nxt;
                const uint64_t tn = t + kSerialThreads + tid;
                nxt = tn < t1 ? __ldg(tk + tn) : make_uint4(0u, 0u, 0u, 0u);
                // overlap of [dst, dst+len) with [r0, r1)   (lanes past t1 hold len == 0)
                const uint64_t d0 = max((uint64_t)raw.z, r0), d1 = min((uint64_t)raw.z + raw.y, r1);
                const bool hit = d1 > d0;
                if (!__syncthreads_or(hit)) continue;  // (also orders the prefill / the previous window's copies)
                const uint32_t bal = __ballot_sync(0xffffffffu, hit);
                if (lane == 0) s_cnt[warp] = __popc(bal);
                __syncthreads();
                uint32_t before = 0, total = 0;
                for (uint32_t w = 0; w < kSerialThreads / 32; ++w) {
                    const uint32_t c = s_cnt[w];
                    before += w < warp ? c : 0u;
                    total += c;
                }
                if (hit) {
                    const uint32_t q = before + __popc(bal & ((1u << lane) - 1u));
                    s_src[q] = (raw.w ? alt : ref) + raw.x + (d0 - raw.z);
                    s_dst[q] = (uint32_t)(d0 - r0);
                    s_len[q] = (uint32_t)(d1 - d0);
                }
                __syncthreads();
                for (uint32_t q = 0; q < total; ++q) {  // array order; a barrier between two writers of a byte
                    const uint8_t* __restrict__ src = s_src[q];
                    uint8_t* dst = res + r0 + s_dst[q];
                    for (uint32_t x = tid; x < s_len[q]; x += kSerialThreads) dst[x] = src[x];
                    __syncthreads();
                }
            }
            __syncthreads();
        }
    }
}

// ------------------------------------------------------------------------------------------------ replicas
// rep[r*stride + x + r] = ref[x] for r in 0..15: whatever (dst - src) mod 16 a run has, one replica holds it at
// the output's 16-byte phase, so its fully covered vectors are plain aligned TMA bulk copies.
// `ref` may be replica 0 itself (already in place): then only replicas 1..15 are written.
__global__ void k_build_replicas(const uint8_t* ref, uint64_t n_ref, uint8_t* rep, uint64_t stride) {
    const uint64_t x = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (x >= n_ref) return;
    const uint8_t v = ref[x];
    for (int r = (ref == rep) ? 1 : 0; r < 16; ++r) rep[(uint64_t)r * stride + x + r] = v;
}

// ------------------------------------------------------------------------------------------------ SoA hand-off
// gir.rs:283-299 shape (four usize arrays) -> packed tasks in BYTES of `unit`-byte residues.
// All reference panics are decided here on the ORIGINAL 64-bit values (before the u32 packing):
// stream code (haplotype_instruction.rs:154), contiguity (gir.rs:208, when `validate`), slices (task.rs:44/48).
__global__ void k_soa_pack(uint64_t n, const uint64_t* __restrict__ code, const uint64_t* __restrict__ sp,
                           const uint64_t* __restrict__ len, const uint64_t* __restrict__ spr, uint64_t n_ref,
                           uint64_t n_alt, uint64_t n_res, uint32_t unit, int validate, v2p_task16* __restrict__ out,
                           DevStatus* status) {
    uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t >= n) return;
    const uint64_t c = code[t], s = sp[t], l = len[t], d = spr[t];
    unsigned long long key = (unsigned long long)t << 8;
    v2p_task16 o = {0u, 0u, 0u, 0u};
    if (validate && t > 0 && d != spr[t - 1] + len[t - 1]) atomicMin(&status->gap_key, (unsigned long long)t);
    if (c > 1) {
        atomicMin(&status->stream_key, (unsigned long long)t);
    } else if (d + l < d || d + l > n_res) {
        atomicMin(&status->err_key, key | V2P_ERR_RES_OOB);
    } else if (s + l < s || s + l > (c == 0 ? n_ref : n_alt)) {
        atomicMin(&status->err_key, key | V2P_ERR_SRC_OOB);
    } else {
        o.src_off = (uint32_t)(s * unit);
        o.len = (uint32_t)(l * unit);
        o.dst_off = (uint32_t)(d * unit);
        o.stream = (uint32_t)c;
    }
    out[t] = o;
}

}  // namespace v2p
