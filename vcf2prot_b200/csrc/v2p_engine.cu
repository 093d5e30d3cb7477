// v2p_engine.cu -- C ABI (include/v2p_engine.h) over the sm_100a kernels in v2p_kernels.cuh.
//
// Replaces the `Engine::GPU` arm of GIR::execute (/root/reference/src/data_structures/InternalRep/gir.rs:236-239)
// and adds the batched native entry the host pipeline uses.  No CPU fallback exists in this file: every
// result byte is produced by a CUDA kernel or the call fails.
//
// Streams: device-pointer batches and the SoA call run on the engine stream (or the caller's, v2p_engine_set_stream).
// Host-pointer batches rotate over kSlots staging slots, each with its own stream and device staging, so that with
// V2P_FLAG_ASYNC chunk i's copy-back (D2H) overlaps chunk i+1's upload (H2D) and kernels -- the per-GPU pinned
// staging / async copy-back pipeline of BASELINE.json:north_star.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "v2p_engine.h"
#include "v2p_hostres.cuh"
#include "v2p_kernels.cuh"
#include "v2p_mapped.cuh"

using namespace v2p;

namespace {

struct Scratch {  // per-stream planning scratch: used only by the kernels of the launch group itself
    DevBuf lb, tile_hap, chunk_hap, order, status, hap_flags;
};

constexpr int kSlots = 3;

struct Slot {  // one in-flight host-pointer batch
    cudaStream_t stream = nullptr;
    Scratch sc;
    DevBuf d_tasks, d_task_begin, d_ref, d_ref_base, d_alt, d_alt_base, d_out, d_out_base;
    bool busy = false;
};

constexpr int kSoaSlots = 16;  // concurrent v2p_execute_soa / v2p_gir_execute callers (rayon workers, parts/exec.rs:36-39)

struct SoaSlot {  // everything one in-flight single-haplotype call needs: nobody else touches it until the call returns
    cudaStream_t stream = nullptr;
    Scratch sc;
    DevBuf d_soa[4], tasks, ref, alt, out, bases, ser_list;
    MappedBuf h_status;  // one DevStatus
    PinnedBuf h_stage;   // staging of the 1-byte tapes (ref | alt | res), grown on demand
    bool busy = false;
};

}  // namespace

struct v2p_event {
    cudaEvent_t ev_start = nullptr, ev_stop = nullptr, ev_done = nullptr, ev_copy = nullptr;
    MappedBuf h_status;             // one DevStatus, published right behind the launch group
    KParams kp;                     // for the deferred serial fallback
    DevBuf ser_list;                // kp.ser_list: k_serial reads it at the wait, after any later launch's plan
    cudaStream_t stream = nullptr;
    Slot* slot = nullptr;  // host-pointer mode
    uint8_t* h_out = nullptr;
    size_t out_bytes = 0;
    const uint64_t* h_task_begin = nullptr;  // borrowed until the wait (host-pointer mode)
};

struct v2p_engine {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    std::mutex mu;
    std::atomic<uint64_t> launches{0};
    int variant = -1;     // -1 = auto: 8 KiB tiles on the TMA path, 4 KiB tiles on the register path
    int ctas_per_sm = 0;  // 0 = the variant's default
    Scratch sc;           // for e->stream
    Slot slots[kSlots];
    int next_slot = 0;
    std::vector<v2p_event*> event_pool;  // CUDA events + pinned status blocks are recycled (no per-call alloc/free)
    // the single-haplotype entry: per-caller slots, handed out under soa_mu (held only for the hand-out)
    SoaSlot soa[kSoaSlots];
    std::mutex soa_mu;
    std::condition_variable soa_cv;
    // registered reference: replica r (0..15) at ref_rep + r*rep_stride, holding ref[x] at offset x + r
    DevBuf ref_rep;
    uint64_t rep_stride = 0, reg_n_ref = 0;
    bool has_ref = false;
    int ref_tma_mode = 0;  // 1: 16 replicas + TMA bulk copies (default), 0: register path only
    int order_gshift = 2;  // interleave groups of 2^2 consecutive tiles (measured best: profiles/r1);
                           // env V2P_TILE_ORDER=tape: tiles in tape order; =gN: groups of 2^N tiles (A/B knobs)
    bool tape_order = false;
    // profiling: per-warp wall time of the copy grid of the last launch group on e->stream (v2p_engine_profile_warps)
    bool profile_warps = false;
    DevBuf warp_ns;
    uint32_t warp_ns_n = 0;
};

namespace {

// The message of the last failed call is per host THREAD: the engine is called concurrently (one haplotype per rayon
// worker in the reference, parts/exec.rs:36-39), and a shared string could be overwritten under the reader's eyes.
thread_local std::string t_err;

// Copy-kernel variants selectable through v2p_engine_set_tuning (profiling sweeps); 0 is the shipped default.
struct CopyVariant {
    int tile;
    int ctas_per_sm;
    void (*fn)(const KParams);     // tiles in tape order
    void (*fn_il)(const KParams);  // haplotype-interleaved tile order (FLAGS | 2)
};
#define V2P_VARIANT(T, G, M, F) k_copy_tiles<T, G, M, F>, k_copy_tiles<T, G, M, (F) | 2>
const CopyVariant kVariants[] = {
    {4096, 4, V2P_VARIANT(4096, 2, 4, 1)},  // 0: 4 KiB tiles, 4 CTAs/SM (64 regs), L2 hints  [default without replicas]
    {4096, 4, V2P_VARIANT(4096, 2, 4, 0)},  // 1: no L2 hints
    {4096, 4, V2P_VARIANT(4096, 1, 4, 1)},  // 2: one vector in flight per lane
    {4096, 5, V2P_VARIANT(4096, 2, 5, 1)},  // 3: 5 CTAs/SM (48 regs)
    {4096, 6, V2P_VARIANT(4096, 1, 6, 1)},  // 4: 6 CTAs/SM (40 regs)
    {4096, 3, V2P_VARIANT(4096, 4, 3, 1)},  // 5: 3 CTAs/SM (80 regs), 4 vectors in flight
    {2048, 6, V2P_VARIANT(2048, 2, 6, 1)},  // 6: 2 KiB tiles, 6 CTAs/SM
    {2048, 8, V2P_VARIANT(2048, 1, 8, 1)},  // 7: 2 KiB tiles, 8 CTAs/SM (32 regs)
    {8192, 3, V2P_VARIANT(8192, 2, 3, 1)},  // 8: 8 KiB tiles, 3 CTAs/SM (80 regs)  [default with replicas]
    {8192, 2, V2P_VARIANT(8192, 4, 2, 1)},  // 9: 8 KiB tiles, 2 CTAs/SM
};
constexpr int kNumVariants = (int)(sizeof(kVariants) / sizeof(kVariants[0]));
constexpr int kAutoTma = 8, kAutoPlain = 0;  // measured best per path (profiles/r1)

// plan + copy on stream s.  kp.{lb,tile_hap,status,n_tiles,tile_bytes} are filled here.
// ser_list is the launch's own (k_serial may read it long after the launch group, see k_serial).
int launch_group(v2p_engine* e, cudaStream_t s, Scratch& sc, DevBuf& ser_list, KParams& kp, cudaEvent_t ev_start,
                 cudaEvent_t ev_stop, DevStatus* h_status, bool init_status, cudaEvent_t ev_copy, bool aligned_layout) {
    const CopyVariant& cv = kVariants[e->variant >= 0 ? e->variant : (kp.tma_mode ? kAutoTma : kAutoPlain)];
    const int T = cv.tile;
    kp.tile_bytes = (uint32_t)T;
    kp.tile_shift = T == 8192 ? 13u : T == 4096 ? 12u : 11u;
    kp.n_tiles = (kp.n_out + T - 1) / T;
    if (kp.n_tasks >= 0xFFFFFFFEull) return fail(t_err, V2P_ERR_INVALID_ARG, "more than 2^32-2 tasks in one launch");
    if (kp.n_hap >= 0x80000000ull) return fail(t_err, V2P_ERR_INVALID_ARG, "more than 2^31 haplotypes in one launch");  // bit 31 of tile_hap[] is a flag
    CU(t_err, sc.lb.need((kp.n_tiles + 1) * sizeof(uint32_t)));
    CU(t_err, sc.tile_hap.need(std::max<uint64_t>(kp.n_tiles, 1) * sizeof(uint32_t)));
    CU(t_err, sc.status.need(sizeof(DevStatus)));
    const uint64_t n_chunks = (kp.n_tasks + kPlanWarpTasks - 1) / kPlanWarpTasks;
    CU(t_err, sc.chunk_hap.need(std::max<uint64_t>(n_chunks, 1) * sizeof(uint32_t)));
    kp.chunk_hap = (uint32_t*)sc.chunk_hap.p;
    // per-haplotype "needs serial order" flags (+ one counter word behind them) and the compacted list of those
    CU(t_err, sc.hap_flags.need((kp.n_hap + 1) * sizeof(uint32_t)));
    CU(t_err, ser_list.need(std::max<uint64_t>(kp.n_hap, 1) * sizeof(uint32_t)));
    kp.hap_flags = (uint32_t*)sc.hap_flags.p;
    kp.ser_list = (uint32_t*)ser_list.p;
    // tile order: 16-byte header (s_max) + one slot per (tile rank within its haplotype, haplotype)
    if (kp.n_tiles >= 0xFFF00000ull) return fail(t_err, V2P_ERR_INVALID_ARG, "more than 2^32 tiles in one launch");
    // tape order = identity over n_tiles (n_hap "1"): the cap then only has to hold the identity
    // Tile order: haplotype-interleaved (DESIGN.md section 4) unless the caller says the layout is phase-aligned
    // (V2P_FLAG_ALIGNED_LAYOUT: every run then comes from the one plain tape and tape order is ~3 % faster).
    const bool interleave = !aligned_layout && !e->tape_order && kp.n_hap > 1;
    kp.order_gshift = (uint32_t)e->order_gshift;
    const uint64_t order_cap =
        interleave ? std::min<uint64_t>(2 * kp.n_tiles + ((kp.n_hap + 64) << kp.order_gshift), 0xFFF00000ull) : 0;
    CU(t_err, sc.order.need(16 + order_cap * sizeof(uint32_t)));
    kp.order_hdr = (uint32_t*)sc.order.p;
    kp.order = kp.order_hdr + 4;
    kp.order_cap = order_cap;
    kp.lb = (uint32_t*)sc.lb.p;
    kp.tile_hap = (uint32_t*)sc.tile_hap.p;
    kp.status = (DevStatus*)sc.status.p;
    if (ev_start) CU(t_err, cudaEventRecord(ev_start, s));
    CU(t_err, cudaMemsetAsync(kp.lb, 0xFF, (kp.n_tiles + 1) * sizeof(uint32_t), s));
    CU(t_err, cudaMemsetAsync(kp.order_hdr, 0, 16, s));
    CU(t_err, cudaMemsetAsync(kp.hap_flags, 0, (kp.n_hap + 1) * sizeof(uint32_t), s));
    if (order_cap) CU(t_err, cudaMemsetAsync(kp.order, 0xFF, order_cap * sizeof(uint32_t), s));
    if (init_status) {
        k_init_status<<<1, 1, 0, s>>>(kp.status);
        e->launches++;
    }
    if (kp.n_hap) {
        k_plan_haps<<<(unsigned)((kp.n_hap + 255) / 256), 256, 0, s>>>(kp);
        e->launches++;
        if (kp.n_tiles || n_chunks) {
            k_plan_tiles<<<(unsigned)((std::max(kp.n_tiles, n_chunks) + 255) / 256), 256, 0, s>>>(kp);
            e->launches++;
        }
    }
    if (kp.n_tasks) {
        k_plan_tasks<<<(unsigned)((kp.n_tasks + kPlanChunk - 1) / kPlanChunk), 256, 0, s>>>(kp);
        e->launches++;
    }
    if (kp.n_hap) {  // (also without any task: a haplotype that has none is all '.', and k_plan_fix is who marks its tiles)
        k_plan_fix<<<(unsigned)((kp.n_hap + 255) / 256), 256, 0, s>>>(kp, kp.hap_flags + kp.n_hap);
        e->launches++;
    }
    if (ev_copy) CU(t_err, cudaEventRecord(ev_copy, s));
    if (kp.n_tiles) {
        const int per_sm = e->ctas_per_sm > 0 ? e->ctas_per_sm : cv.ctas_per_sm;
        uint64_t want = (kp.n_tiles + kWarpsPerCta - 1) / kWarpsPerCta;
        unsigned grid = (unsigned)std::min<uint64_t>(want, (uint64_t)e->sm_count * per_sm);
        size_t smem = (size_t)kWarpsPerCta * (cv.tile + cv.tile / 16 + kTileScratch) + 17 * 16;
        kp.warp_ns = nullptr;
        if (e->profile_warps && s == e->stream) {
            CU(t_err, e->warp_ns.need((size_t)grid * kWarpsPerCta * sizeof(unsigned long long)));
            kp.warp_ns = (unsigned long long*)e->warp_ns.p;
            e->warp_ns_n = grid * kWarpsPerCta;
        }
        void (*fn)(const KParams) = interleave ? cv.fn_il : cv.fn;
        if (smem > 48 * 1024) CU(t_err, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        fn<<<grid, kThreads, smem, s>>>(kp);
        e->launches++;
    }
    if (ev_stop) CU(t_err, cudaEventRecord(ev_stop, s));
    CU(t_err, cudaGetLastError());
    // status rides the stream right behind the kernels, so a later launch cannot overwrite it first; it is stored
    // into mapped pinned memory by a kernel (v2p_mapped.cuh) so it never queues behind a result tape on the copy engine
    static_assert(sizeof(DevStatus) == 32, "DevStatus is published as four 8-byte words");
    CU(t_err, publish_words(reinterpret_cast<unsigned long long*>(h_status), kp.status, 4, s));
    e->launches++;
    return V2P_OK;
}

void decode_status(const DevStatus& st, const uint64_t* task_begin_host, uint64_t n_hap, uint64_t task_origin,
                   v2p_result* res) {
    res->status = V2P_OK;
    res->bad_hap = 0;
    res->bad_task = 0;
    if (st.bad_args) {
        res->status = V2P_ERR_INVALID_ARG;
        return;
    }
    // The reference handles one haplotype after the other (personalized_genome.rs:64-65, parts/exec.rs:34-40), and
    // inside one haplotype in this order: a bad stream code panics while the Task array is built
    // (haplotype_instruction.rs:154), then the contiguity validator runs (gir.rs:203-229), then slices panic
    // during execution (task.rs:44/48).  So: the lowest haplotype with any finding wins; inside it, that precedence.
    struct Finding {
        int status;
        uint64_t task;  // launch-relative global index
        uint64_t hap;
    } f[3] = {{V2P_ERR_BAD_STREAM, st.stream_key, 0},
              {V2P_ERR_NOT_CONTIGUOUS, st.gap_key, 0},
              {st.err_key != ~0ull ? (int)(st.err_key & 0xFF) : 0, st.err_key != ~0ull ? st.err_key >> 8 : ~0ull, 0}};
    const bool have_tb = task_begin_host && n_hap;
    const Finding* best = nullptr;
    for (Finding& c : f) {
        if (c.task == ~0ull) continue;
        if (have_tb) {
            size_t h = std::upper_bound(task_begin_host, task_begin_host + n_hap + 1, c.task + task_origin) - task_begin_host;
            h = h ? h - 1 : 0;
            c.hap = h >= n_hap ? n_hap - 1 : h;
        }
        if (!best || c.hap < best->hap) best = &c;  // (ties keep the earlier class)
    }
    if (!best) return;
    res->status = best->status;
    res->bad_task = best->task;  // launch-relative global index unless task_begin is known on the host
    if (have_tb) {
        res->bad_hap = best->hap;
        res->bad_task = best->task + task_origin - task_begin_host[best->hap];
    }
}

bool needs_serial(const DevStatus& st) {
    return !st.bad_args && st.err_key == ~0ull && st.gap_key == ~0ull && st.stream_key == ~0ull && st.unsorted;
}

// serial-order kernel over the n_ser haplotypes the plan flagged (unsorted / overlapping tasks); everybody else
// was written by the tile kernel of the same launch group
int launch_serial(v2p_engine* e, cudaStream_t s, const KParams& kp, uint32_t n_ser) {
    unsigned grid = (unsigned)e->sm_count * 4;
    k_serial<<<grid, kSerialThreads, 0, s>>>(kp, n_ser);
    e->launches++;
    CU(t_err, cudaGetLastError());
    return V2P_OK;
}

void free_event(v2p_event* ev) {
    if (ev->ev_start) cudaEventDestroy(ev->ev_start);
    if (ev->ev_stop) cudaEventDestroy(ev->ev_stop);
    if (ev->ev_done) cudaEventDestroy(ev->ev_done);
    if (ev->ev_copy) cudaEventDestroy(ev->ev_copy);
    delete ev;
}

// returns the event object to the engine's pool (its slot becomes free again)
void destroy_event(v2p_engine* e, v2p_event* ev) {
    if (ev->slot) ev->slot->busy = false;
    ev->slot = nullptr;
    ev->h_out = nullptr;
    ev->out_bytes = 0;
    ev->h_task_begin = nullptr;
    e->event_pool.push_back(ev);
}

v2p_event* acquire_event(v2p_engine* e) {
    if (!e->event_pool.empty()) {
        v2p_event* ev = e->event_pool.back();
        e->event_pool.pop_back();
        return ev;
    }
    v2p_event* ev = new (std::nothrow) v2p_event();
    if (!ev) return nullptr;
    if (cudaEventCreate(&ev->ev_start) != cudaSuccess || cudaEventCreate(&ev->ev_stop) != cudaSuccess ||
        cudaEventCreate(&ev->ev_copy) != cudaSuccess ||
        cudaEventCreateWithFlags(&ev->ev_done, cudaEventDisableTiming) != cudaSuccess ||
        ev->h_status.reserve(4) != cudaSuccess) {
        free_event(ev);
        return nullptr;
    }
    return ev;
}

// Completes a launch group: status, serial fallback (+ repeated copy-back in host mode); destroys the event.
int wait_locked(v2p_engine* e, v2p_event* ev, v2p_result* res) {
    v2p_result local;
    memset(&local, 0, sizeof local);
    auto finish = [&](int code) {
        destroy_event(e, ev);
        if (res) *res = local;
        return code;
    };
    cudaSetDevice(e->device);
    if (cudaEventSynchronize(ev->ev_done) != cudaSuccess)
        return finish(fail(t_err, V2P_ERR_CUDA, "launch group failed: %s", cudaGetErrorString(cudaGetLastError())));
    const DevStatus& st = *reinterpret_cast<const DevStatus*>(ev->h_status.p);
    if (needs_serial(st)) {
        int rc = launch_serial(e, ev->stream, ev->kp, st.unsorted);
        if (rc) return finish(rc);
        if (ev->slot && ev->out_bytes &&
            cudaMemcpyAsync(ev->h_out, ev->kp.out, ev->out_bytes, cudaMemcpyDeviceToHost, ev->stream) != cudaSuccess)
            return finish(fail(t_err, V2P_ERR_CUDA, "D2H failed: %s", cudaGetErrorString(cudaGetLastError())));
        if (cudaStreamSynchronize(ev->stream) != cudaSuccess)
            return finish(fail(t_err, V2P_ERR_CUDA, "serial-order kernel failed: %s", cudaGetErrorString(cudaGetLastError())));
    }
    std::vector<uint64_t> tb_copy;
    const uint64_t* tb = ev->h_task_begin;
    if (!tb && ev->kp.n_hap && (st.err_key != ~0ull || st.gap_key != ~0ull || st.stream_key != ~0ull)) {  // error path only: fetch task_begin
        tb_copy.resize(ev->kp.n_hap + 1);
        if (cudaMemcpy(tb_copy.data(), ev->kp.task_begin, tb_copy.size() * sizeof(uint64_t), cudaMemcpyDeviceToHost) ==
            cudaSuccess)
            tb = tb_copy.data();
    }
    decode_status(st, tb, ev->kp.n_hap, ev->kp.task_origin, &local);
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ev->ev_start, ev->ev_stop) == cudaSuccess) local.kernel_ms = ms;
    if (cudaEventElapsedTime(&ms, ev->ev_copy, ev->ev_stop) == cudaSuccess) local.copy_ms = ms;
    if (local.status != V2P_OK)
        fail(t_err, local.status, "haplotype %llu task %llu rejected with status %d", (unsigned long long)local.bad_hap,
             (unsigned long long)local.bad_task, local.status);
    return finish(local.status);
}

}  // namespace

// ------------------------------------------------------------------------------------------------ ABI
extern "C" {

int v2p_abi_version(void) { return V2P_ABI_VERSION; }

int v2p_engine_device(v2p_engine* e) { return e ? e->device : -1; }

int v2p_engine_from_str(const char* s, int* engine_kind) {
    if (!s || !engine_kind) return V2P_ERR_INVALID_ARG;
    if (!strcmp(s, "st") || !strcmp(s, "ST")) return *engine_kind = V2P_ENGINE_ST, V2P_OK;
    if (!strcmp(s, "mt") || !strcmp(s, "MT")) return *engine_kind = V2P_ENGINE_MT, V2P_OK;
    if (!strcmp(s, "gpu") || !strcmp(s, "GPU")) return *engine_kind = V2P_ENGINE_GPU, V2P_OK;
    return V2P_ERR_BAD_ENGINE;
}

int v2p_engine_create(int cuda_device, v2p_engine** out) {
    if (!out) return V2P_ERR_INVALID_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0 || cuda_device < 0 || cuda_device >= n) return V2P_ERR_CUDA;
    v2p_engine* e = new (std::nothrow) v2p_engine();
    if (!e) return V2P_ERR_INVALID_ARG;
    e->device = cuda_device;
    cudaDeviceProp prop;
    bool ok = cudaSetDevice(cuda_device) == cudaSuccess && cudaGetDeviceProperties(&prop, cuda_device) == cudaSuccess &&
              cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; ok && i < kSlots; ++i)
        ok = cudaStreamCreateWithFlags(&e->slots[i].stream, cudaStreamNonBlocking) == cudaSuccess;
    if (!ok) {
        v2p_engine_destroy(e);
        return V2P_ERR_CUDA;
    }
    e->sm_count = prop.multiProcessorCount;
    const char* ord = getenv("V2P_TILE_ORDER");
    e->tape_order = ord && !strcmp(ord, "tape");
    if (ord && ord[0] == 'g' && ord[1] >= '0' && ord[1] <= '6') e->order_gshift = ord[1] - '0';
    *out = e;
    return V2P_OK;
}

void v2p_engine_destroy(v2p_engine* e) {
    if (!e) return;
    cudaSetDevice(e->device);
    cudaDeviceSynchronize();
    for (SoaSlot& sl : e->soa)
        if (sl.stream) cudaStreamDestroy(sl.stream);
    for (Slot& sl : e->slots)
        if (sl.stream) cudaStreamDestroy(sl.stream);
    for (v2p_event* ev : e->event_pool) free_event(ev);
    if (e->own_stream && e->stream) cudaStreamDestroy(e->stream);
    delete e;  // frees every buffer
}

const char* v2p_last_error(v2p_engine* e) { return e ? t_err.c_str() : "engine is NULL"; }

int v2p_host_alloc(void** ptr, size_t bytes) {
    if (!ptr) return V2P_ERR_INVALID_ARG;
    return cudaMallocHost(ptr, std::max<size_t>(bytes, 16)) == cudaSuccess ? V2P_OK : V2P_ERR_CUDA;
}
int v2p_host_free(void* ptr) { return cudaFreeHost(ptr) == cudaSuccess ? V2P_OK : V2P_ERR_CUDA; }

uint64_t v2p_kernel_launch_count(v2p_engine* e) { return e ? e->launches.load() : 0; }

int v2p_engine_set_tuning(v2p_engine* e, int variant, int ctas_per_sm) {
    if (!e || variant < -1 || variant >= kNumVariants || ctas_per_sm < 0 || ctas_per_sm > 32) return V2P_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    e->variant = variant;
    e->ctas_per_sm = ctas_per_sm;
    return V2P_OK;
}

int v2p_engine_profile_warps(v2p_engine* e, int on) {
    if (!e) return V2P_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    e->profile_warps = on != 0;
    return V2P_OK;
}

int v2p_engine_read_warp_ns(v2p_engine* e, uint64_t* ns_out, uint64_t cap, uint64_t* n_warps) {
    if (!e || !n_warps) return V2P_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    *n_warps = e->warp_ns_n;
    if (!ns_out || cap < e->warp_ns_n || !e->warp_ns_n) return e->warp_ns_n && ns_out ? V2P_ERR_INVALID_ARG : V2P_OK;
    CU(t_err, cudaSetDevice(e->device));
    CU(t_err, cudaStreamSynchronize(e->stream));
    CU(t_err, cudaMemcpy(ns_out, e->warp_ns.p, (size_t)e->warp_ns_n * 8, cudaMemcpyDeviceToHost));
    return V2P_OK;
}

int v2p_engine_set_stream(v2p_engine* e, void* cuda_stream) {
    if (!e) return V2P_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    cudaSetDevice(e->device);
    cudaStreamSynchronize(e->stream);
    if (e->own_stream && e->stream) cudaStreamDestroy(e->stream);
    if (cuda_stream) {
        e->stream = (cudaStream_t)cuda_stream;
        e->own_stream = false;
    } else {
        if (cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) return V2P_ERR_CUDA;
        e->own_stream = true;
    }
    return V2P_OK;
}

int v2p_engine_set_reference(v2p_engine* e, const uint8_t* ref, uint64_t n_ref, uint32_t flags) {
    if (!e || (n_ref && !ref)) return V2P_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    t_err.clear();
    CU(t_err, cudaSetDevice(e->device));
    CU(t_err, cudaDeviceSynchronize());  // nothing in flight may still read the previous tape
    e->has_ref = false;
    const bool replicas = (flags & V2P_REF_NO_TMA) == 0;
    const uint64_t stride = (n_ref + 64 + 255) & ~255ull;
    const uint64_t bytes = (replicas ? 16 : 1) * stride + 256;
    CU(t_err, e->ref_rep.need(bytes));
    uint8_t* rep = (uint8_t*)e->ref_rep.p;
    CU(t_err, cudaMemsetAsync(rep, 0, bytes, e->stream));
    if (n_ref) {
        CU(t_err, cudaMemcpyAsync(rep, ref, n_ref,
                                    (flags & V2P_FLAG_DEVICE_PTRS) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice,
                                    e->stream));
        if (replicas) {
            k_build_replicas<<<(unsigned)((n_ref + 255) / 256), 256, 0, e->stream>>>(rep, n_ref, rep, stride);
            e->launches++;
            CU(t_err, cudaGetLastError());
        }
    }
    CU(t_err, cudaStreamSynchronize(e->stream));
    e->ref_tma_mode = replicas ? 1 : 0;
    e->rep_stride = stride;
    e->reg_n_ref = n_ref;
    e->has_ref = true;
    return V2P_OK;
}

// ---- batched native call -------------------------------------------------------------------------
int v2p_execute_batch(v2p_engine* e, const v2p_batch* b, uint32_t flags, v2p_result* res, v2p_event** done) {
    if (!e) return V2P_ERR_INVALID_ARG;
    std::lock_guard<std::mutex> g(e->mu);
    t_err.clear();
    if (!b) return fail(t_err, V2P_ERR_INVALID_ARG, "batch is NULL");
    if (b->n_hap && (!b->task_begin || !b->alt_base || !b->out_base))
        return fail(t_err, V2P_ERR_INVALID_ARG, "task_begin/alt_base/out_base must not be NULL");
    const bool async = (flags & V2P_FLAG_ASYNC) != 0;
    if (async && !done) return fail(t_err, V2P_ERR_INVALID_ARG, "ASYNC needs an event out-pointer");
    if (!async && !res) return fail(t_err, V2P_ERR_INVALID_ARG, "synchronous call needs a result out-pointer");
    CU(t_err, cudaSetDevice(e->device));
    if (res) memset(res, 0, sizeof *res);
    const bool use_reg_ref = b->ref == nullptr && b->ref_base == nullptr;
    if (use_reg_ref && !e->has_ref)
        return fail(t_err, V2P_ERR_INVALID_ARG, "ref == NULL but no reference was registered (v2p_engine_set_reference)");

    v2p_event* ev = acquire_event(e);
    if (!ev) return fail(t_err, V2P_ERR_CUDA, "event/pinned allocation failed");
    auto bail = [&](int code) {
        destroy_event(e, ev);
        return code;
    };

    KParams kp;
    memset(&kp, 0, sizeof kp);
    kp.n_hap = b->n_hap;
    kp.fill_word = 0x2E2E2E2Eu;
    kp.validate = (flags & V2P_FLAG_VALIDATE) ? 1 : 0;
    cudaStream_t s = e->stream;
    Scratch* sc = &e->sc;
    int rc;

    if (flags & V2P_FLAG_DEVICE_PTRS) {
        if (((uintptr_t)b->out & 15u) != 0) return bail(fail(t_err, V2P_ERR_INVALID_ARG, "out must be 16-byte aligned"));
        kp.tasks = b->tasks;
        kp.task_begin = b->task_begin;
        kp.ref = b->ref;
        kp.ref_base = b->ref_base;
        kp.alt = b->alt;
        kp.alt_base = b->alt_base;
        kp.out = b->out;
        kp.out_base = b->out_base;
        kp.n_tasks = b->n_tasks;
        kp.n_ref = b->n_ref;
        kp.n_alt = b->n_alt;
        kp.n_out = b->n_out;  // origins stay 0: device-pointer batches are self-contained
    } else {
        // host pointers: stage through the next slot's device buffers on that slot's stream
        Slot* sl = &e->slots[e->next_slot];
        if (sl->busy)
            return bail(fail(t_err, V2P_ERR_INVALID_ARG,
                             "%d host-pointer batches already in flight: wait for the oldest event first", kSlots));
        const uint64_t H = b->n_hap;
        const uint64_t t0 = H ? b->task_begin[0] : 0, t1 = H ? b->task_begin[H] : 0;
        const uint64_t a0 = H ? b->alt_base[0] : 0, a1 = H ? b->alt_base[H] : 0;
        const uint64_t o0 = H ? b->out_base[0] : 0, o1 = H ? b->out_base[H] : 0;
        uint64_t r0 = 0, r1 = use_reg_ref ? 0 : b->n_ref;
        if (b->ref_base && H) r0 = b->ref_base[0], r1 = b->ref_base[H];
        if (t1 < t0 || a1 < a0 || o1 < o0 || r1 < r0) return bail(fail(t_err, V2P_ERR_INVALID_ARG, "base arrays not monotone"));
        kp.n_tasks = t1 - t0;
        kp.n_alt = a1 - a0;
        kp.n_out = o1 - o0;
        kp.n_ref = r1 - r0;
        kp.task_origin = t0;
        kp.alt_origin = a0;
        kp.out_origin = o0;
        kp.ref_origin = r0;
        if ((kp.n_tasks && !b->tasks) || (kp.n_out && !b->out) || (kp.n_ref && !b->ref) || (kp.n_alt && !b->alt))
            return bail(fail(t_err, V2P_ERR_INVALID_ARG, "NULL data pointer"));
        const size_t nb = (H + 1) * sizeof(uint64_t);
        auto stage = [&]() -> int {
            CU(t_err, sl->d_tasks.need(kp.n_tasks * sizeof(v2p_task16)));
            CU(t_err, sl->d_task_begin.need(nb));
            CU(t_err, sl->d_ref.need(kp.n_ref + 32));
            CU(t_err, sl->d_ref_base.need(nb));
            CU(t_err, sl->d_alt.need(kp.n_alt + 32));
            CU(t_err, sl->d_alt_base.need(nb));
            CU(t_err, sl->d_out.need(kp.n_out + 32));
            CU(t_err, sl->d_out_base.need(nb));
            return V2P_OK;
        };
        if ((rc = stage())) return bail(rc);
        s = sl->stream;
        sc = &sl->sc;
        auto h2d = [&](void* d, const void* h, size_t n) {
            return (n && H) ? cudaMemcpyAsync(d, h, n, cudaMemcpyHostToDevice, s) : cudaSuccess;
        };
        if (h2d(sl->d_tasks.p, b->tasks + t0, kp.n_tasks * sizeof(v2p_task16)) != cudaSuccess ||
            h2d(sl->d_task_begin.p, b->task_begin, nb) != cudaSuccess ||
            h2d(sl->d_ref.p, b->ref + r0, kp.n_ref) != cudaSuccess ||
            (b->ref_base && h2d(sl->d_ref_base.p, b->ref_base, nb) != cudaSuccess) ||
            h2d(sl->d_alt.p, b->alt + a0, kp.n_alt) != cudaSuccess || h2d(sl->d_alt_base.p, b->alt_base, nb) != cudaSuccess ||
            h2d(sl->d_out_base.p, b->out_base, nb) != cudaSuccess)
            return bail(fail(t_err, V2P_ERR_CUDA, "H2D failed: %s", cudaGetErrorString(cudaGetLastError())));
        kp.tasks = (const v2p_task16*)sl->d_tasks.p;
        kp.task_begin = (const uint64_t*)sl->d_task_begin.p;
        kp.ref = (const uint8_t*)sl->d_ref.p;
        kp.ref_base = b->ref_base ? (const uint64_t*)sl->d_ref_base.p : nullptr;
        kp.alt = (const uint8_t*)sl->d_alt.p;
        kp.alt_base = (const uint64_t*)sl->d_alt_base.p;
        kp.out = (uint8_t*)sl->d_out.p;
        kp.out_base = (const uint64_t*)sl->d_out_base.p;
        ev->slot = sl;
        sl->busy = true;
        e->next_slot = (e->next_slot + 1) % kSlots;
        ev->h_out = H ? b->out + o0 : nullptr;
        ev->out_bytes = kp.n_out;
        ev->h_task_begin = b->task_begin;
    }
    if (use_reg_ref) {
        kp.ref = (const uint8_t*)e->ref_rep.p;  // replica 0 is the plain tape
        kp.ref_base = nullptr;
        kp.ref_origin = 0;
        kp.n_ref = e->reg_n_ref;
        kp.ref_rep = (const uint8_t*)e->ref_rep.p;
        kp.rep_stride = e->rep_stride;
        kp.tma_mode = e->ref_tma_mode;
    }
    ev->stream = s;
    rc = launch_group(e, s, *sc, ev->ser_list, kp, ev->ev_start, ev->ev_stop, reinterpret_cast<DevStatus*>(ev->h_status.p),
                      true, ev->ev_copy, (flags & V2P_FLAG_ALIGNED_LAYOUT) != 0);
    if (rc) return bail(rc);
    // host mode: the copy-back is enqueued right away (a batch that needs the serial-order kernel repeats it later)
    if (ev->slot && ev->out_bytes &&
        cudaMemcpyAsync(ev->h_out, kp.out, ev->out_bytes, cudaMemcpyDeviceToHost, s) != cudaSuccess)
        return bail(fail(t_err, V2P_ERR_CUDA, "D2H failed: %s", cudaGetErrorString(cudaGetLastError())));
    if (cudaEventRecord(ev->ev_done, s) != cudaSuccess)
        return bail(fail(t_err, V2P_ERR_CUDA, "event record failed: %s", cudaGetErrorString(cudaGetLastError())));
    ev->kp = kp;
    if (async) {
        *done = ev;
        return V2P_OK;
    }
    return wait_locked(e, ev, res);
}

int v2p_event_wait(v2p_engine* e, v2p_event* ev, v2p_result* res) {
    if (!e || !ev) return V2P_ERR_INVALID_ARG;
    // block on the caller's own event BEFORE taking the engine lock: other threads keep submitting meanwhile
    cudaSetDevice(e->device);
    cudaEventSynchronize(ev->ev_done);
    std::lock_guard<std::mutex> g(e->mu);
    return wait_locked(e, ev, res);
}

// ---- reference-faithful single-haplotype call ------------------------------------------------------
// Called concurrently, one haplotype per rayon worker (parts/exec.rs:36-39 -> personalized_genome.rs:64-65 ->
// gir.rs:236-239).  Every caller gets its own slot (stream, device buffers, pinned staging, status block) for the
// duration of the call; the engine lock is not taken, so uploads, kernels and copy-backs of different callers overlap.
// When every residue of the three tapes is a code point below 256 (always, for protein FASTA) the tapes cross PCIe
// and are processed as 1-byte residues: narrowed into the slot's pinned staging on the way up, widened into the
// caller's `char` tape on the way back -- a quarter of the bytes of the UTF-32 path, same result.
namespace {

SoaSlot* soa_acquire(v2p_engine* e) {
    std::unique_lock<std::mutex> g(e->soa_mu);
    for (;;) {
        for (SoaSlot& sl : e->soa)
            if (!sl.busy) {
                sl.busy = true;
                return &sl;
            }
        e->soa_cv.wait(g);
    }
}
void soa_release(v2p_engine* e, SoaSlot* sl) {
    {
        std::lock_guard<std::mutex> g(e->soa_mu);
        sl->busy = false;
    }
    e->soa_cv.notify_one();
}

// dst[i] = (uint8_t)src[i]; returns the OR of all units (> 0xFF: some residue does not fit a byte)
uint32_t narrow_u32(const uint32_t* __restrict__ src, uint8_t* __restrict__ dst, size_t n) {
    uint32_t acc = 0;
    for (size_t i = 0; i < n; ++i) {
        acc |= src[i];
        dst[i] = (uint8_t)src[i];
    }
    return acc;
}
void widen_u8(const uint8_t* __restrict__ src, uint32_t* __restrict__ dst, size_t n) {
    for (size_t i = 0; i < n; ++i) dst[i] = src[i];
}

int soa_run(v2p_engine* e, SoaSlot* sl, size_t n_tasks, const uint64_t* exec_code, const uint64_t* start_pos,
            const uint64_t* length, const uint64_t* start_pos_res, const uint32_t* ref_utf32, size_t n_ref,
            const uint32_t* alt_utf32, size_t n_alt, uint32_t* res_utf32, size_t n_res, uint32_t flags, uint64_t* bad_index) {
    CU(t_err, cudaSetDevice(e->device));
    if (!sl->stream) CU(t_err, cudaStreamCreateWithFlags(&sl->stream, cudaStreamNonBlocking));
    CU(t_err, sl->h_status.reserve(4));
    DevStatus* const h_status = reinterpret_cast<DevStatus*>(sl->h_status.p);
    cudaStream_t s = sl->stream;
    const bool keep = !(flags & V2P_FLAG_FILL_DOT);
    int rc;
    // ---- narrow the tapes into pinned staging (ref | alt | res), unless a residue needs more than a byte
    CU(t_err, sl->h_stage.need(n_ref + n_alt + n_res + 64));
    uint8_t* const h_ref = (uint8_t*)sl->h_stage.p;
    uint8_t* const h_alt = h_ref + n_ref;
    uint8_t* const h_res = h_alt + n_alt;
    uint32_t wide = narrow_u32(ref_utf32, h_ref, n_ref) | narrow_u32(alt_utf32, h_alt, n_alt);
    if (keep) wide |= narrow_u32(res_utf32, h_res, n_res);
    const uint32_t unit = wide > 0xFFu ? 4u : 1u;  // bytes per residue on the device
    const size_t tb = n_tasks * sizeof(uint64_t);
    for (int i = 0; i < 4; ++i) CU(t_err, sl->d_soa[i].need(tb));
    CU(t_err, sl->tasks.need(n_tasks * sizeof(v2p_task16)));
    CU(t_err, sl->ref.need(n_ref * unit + 32));
    CU(t_err, sl->alt.need(n_alt * unit + 32));
    CU(t_err, sl->out.need(n_res * unit + 32));
    CU(t_err, sl->bases.need(64));
    CU(t_err, sl->sc.status.need(sizeof(DevStatus)));
    const uint64_t* soa[4] = {exec_code, start_pos, length, start_pos_res};
    for (int i = 0; i < 4; ++i)
        if (tb) CU(t_err, cudaMemcpyAsync(sl->d_soa[i].p, soa[i], tb, cudaMemcpyHostToDevice, s));
    if (unit == 1) {
        if (n_ref) CU(t_err, cudaMemcpyAsync(sl->ref.p, h_ref, n_ref, cudaMemcpyHostToDevice, s));
        if (n_alt) CU(t_err, cudaMemcpyAsync(sl->alt.p, h_alt, n_alt, cudaMemcpyHostToDevice, s));
        if (keep && n_res) CU(t_err, cudaMemcpyAsync(sl->out.p, h_res, n_res, cudaMemcpyHostToDevice, s));
    } else {
        if (n_ref) CU(t_err, cudaMemcpyAsync(sl->ref.p, ref_utf32, n_ref * 4, cudaMemcpyHostToDevice, s));
        if (n_alt) CU(t_err, cudaMemcpyAsync(sl->alt.p, alt_utf32, n_alt * 4, cudaMemcpyHostToDevice, s));
        if (keep && n_res) CU(t_err, cudaMemcpyAsync(sl->out.p, res_utf32, n_res * 4, cudaMemcpyHostToDevice, s));
    }
    // task_begin | alt_base | out_base, two entries each (staged in the pinned status block's neighbourhood is not
    // worth it: 48 bytes from the stack, consumed before this frame returns because the call is synchronous)
    const uint64_t bases[6] = {0, n_tasks, 0, n_alt * unit, 0, n_res * unit};
    CU(t_err, cudaMemcpyAsync(sl->bases.p, bases, sizeof bases, cudaMemcpyHostToDevice, s));

    KParams kp;
    memset(&kp, 0, sizeof kp);
    const uint64_t* db = (const uint64_t*)sl->bases.p;
    kp.tasks = (const v2p_task16*)sl->tasks.p;
    kp.task_begin = db;
    kp.ref = (const uint8_t*)sl->ref.p;
    kp.alt = (const uint8_t*)sl->alt.p;
    kp.alt_base = db + 2;
    kp.out = (uint8_t*)sl->out.p;
    kp.out_base = db + 4;
    kp.n_hap = 1;
    kp.n_tasks = n_tasks;
    kp.n_ref = n_ref * unit;
    kp.n_alt = n_alt * unit;
    kp.n_out = n_res * unit;
    kp.fill_word = unit == 1 ? 0x2E2E2E2Eu : 0x0000002Eu;  // '.' per byte, or as one UTF-32 unit
    kp.keep_out = keep ? 1 : 0;
    // kp.validate stays 0: k_soa_pack judges contiguity on the caller's 64-bit values, and the packed tasks it hands
    // to the plan have every rejected task zeroed, which the plan would take for a contiguity break of its own
    const int validate = (flags & V2P_FLAG_VALIDATE) ? 1 : 0;

    // pack (and judge every reference panic on the original 64-bit values), then plan + copy
    kp.status = (DevStatus*)sl->sc.status.p;
    k_init_status<<<1, 1, 0, s>>>(kp.status);
    e->launches++;
    if (n_tasks) {
        k_soa_pack<<<(unsigned)((n_tasks + 255) / 256), 256, 0, s>>>(
            n_tasks, (const uint64_t*)sl->d_soa[0].p, (const uint64_t*)sl->d_soa[1].p, (const uint64_t*)sl->d_soa[2].p,
            (const uint64_t*)sl->d_soa[3].p, n_ref, n_alt, n_res, unit, validate, (v2p_task16*)sl->tasks.p, kp.status);
        e->launches++;
    }
    rc = launch_group(e, s, sl->sc, sl->ser_list, kp, nullptr, nullptr, h_status, /*init_status=*/false, nullptr, false);
    if (rc) return rc;
    CU(t_err, cudaStreamSynchronize(s));
    if (needs_serial(*h_status)) {
        if ((rc = launch_serial(e, s, kp, h_status->unsorted))) return rc;
        CU(t_err, cudaStreamSynchronize(s));
    }
    v2p_result r;
    memset(&r, 0, sizeof r);
    decode_status(*h_status, nullptr, 0, 0, &r);
    if (r.status != V2P_OK) {
        if (bad_index) *bad_index = r.bad_task;
        return fail(t_err, r.status, "task %llu rejected with status %d", (unsigned long long)r.bad_task, r.status);
    }
    if (n_res) {
        if (unit == 1) {
            CU(t_err, cudaMemcpyAsync(h_res, sl->out.p, n_res, cudaMemcpyDeviceToHost, s));
            CU(t_err, cudaStreamSynchronize(s));
            widen_u8(h_res, res_utf32, n_res);
        } else {
            CU(t_err, cudaMemcpyAsync(res_utf32, sl->out.p, n_res * 4, cudaMemcpyDeviceToHost, s));
            CU(t_err, cudaStreamSynchronize(s));
        }
    }
    return V2P_OK;
}

}  // namespace

int v2p_execute_soa(v2p_engine* e, size_t n_tasks, const uint64_t* exec_code, const uint64_t* start_pos,
                    const uint64_t* length, const uint64_t* start_pos_res, const uint32_t* ref_utf32, size_t n_ref,
                    const uint32_t* alt_utf32, size_t n_alt, uint32_t* res_utf32, size_t n_res, uint32_t flags,
                    uint64_t* bad_index) {
    if (!e) return V2P_ERR_INVALID_ARG;
    t_err.clear();
    if (bad_index) *bad_index = 0;
    if (n_tasks && (!exec_code || !start_pos || !length || !start_pos_res))
        return fail(t_err, V2P_ERR_INVALID_ARG, "NULL task array");
    if ((n_ref && !ref_utf32) || (n_alt && !alt_utf32) || (n_res && !res_utf32))
        return fail(t_err, V2P_ERR_INVALID_ARG, "NULL tape");
    const uint64_t lim = 0xFFFFFFFFull / 4;
    if (n_ref > lim || n_alt > lim || n_res > lim)
        return fail(t_err, V2P_ERR_INVALID_ARG, "tape longer than 2^30 residues: use v2p_execute_batch");
    SoaSlot* sl = soa_acquire(e);
    const int rc = soa_run(e, sl, n_tasks, exec_code, start_pos, length, start_pos_res, ref_utf32, n_ref, alt_utf32, n_alt,
                           res_utf32, n_res, flags, bad_index);
    if (rc != V2P_OK && sl->stream) cudaStreamSynchronize(sl->stream);  // nothing of a failed call may still be in flight
    soa_release(e, sl);
    return rc;
}

int v2p_gir_execute(v2p_engine* e, int engine_kind, size_t n_tasks, const uint64_t* exec_code, const uint64_t* start_pos,
                    const uint64_t* length, const uint64_t* start_pos_res, const uint32_t* ref_utf32, size_t n_ref,
                    const uint32_t* alt_utf32, size_t n_alt, uint32_t* res_utf32, size_t n_res, uint32_t flags,
                    uint64_t* bad_index) {
    if (engine_kind != V2P_ENGINE_GPU)
        return fail(t_err, V2P_ERR_NOT_GPU_ENGINE, "engine kind %d is executed by the caller (gir.rs:201-235)", engine_kind);
    return v2p_execute_soa(e, n_tasks, exec_code, start_pos, length, start_pos_res, ref_utf32, n_ref, alt_utf32, n_alt,
                           res_utf32, n_res, flags, bad_index);
}

}  // extern "C"
