/*
 * v2p_engine.h -- C ABI of the B200-native sequence-generation engine for vcf2prot.
 *
 * This is the drop-in boundary for ONE path of the reference: the `Engine::GPU` arm of
 * `GIR::execute` (/root/reference/src/data_structures/InternalRep/gir.rs:197-241, GPU arm :236-239),
 * i.e. executing a haplotype's concatenated `Vec<Task>` (task.rs:2-9, task.rs:38-50) against the
 * reference tape, the alteration tape and the '.'-prefilled result tape
 * (haplotype_instruction.rs:75-137).  VCF parsing, csq decoding, instruction generation and FASTA
 * writing stay in the caller (INTEGRATION.md shows the Rust `extern "C"` block and the three-line
 * replacement of gir.rs:236-239).
 *
 * Conventions
 *   - C linkage, no exceptions cross the boundary, every function returns an int status (V2P_OK == 0).
 *   - All pointers are borrowed for the duration of the call (or until v2p_event_wait for ASYNC);
 *     the caller owns every buffer; the library never frees caller memory.
 *   - Contexts are thread-safe: concurrent calls on one context are serialised per stream slot, which
 *     matches the reference calling GIR::execute from many rayon workers (parts/exec.rs:36-39).
 *   - There is NO CPU fallback: without a CUDA device v2p_engine_create fails with V2P_ERR_CUDA.
 */
#ifndef V2P_ENGINE_H
#define V2P_ENGINE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define V2P_ABI_VERSION 1

/* ---- status codes ------------------------------------------------------------------------------ */
enum {
    V2P_OK = 0,
    V2P_ERR_INVALID_ARG = 1,    /* NULL / misaligned / inconsistent arguments                           */
    V2P_ERR_CUDA = 2,           /* CUDA runtime failure (see v2p_last_error)                            */
    V2P_ERR_BAD_ENGINE = 3,     /* engines.rs:28  "<s> is not a supported engine"                       */
    V2P_ERR_BAD_STREAM = 4,     /* exe_code not in {0,1}: haplotype_instruction.rs:154 panics           */
    V2P_ERR_RES_OOB = 5,        /* start_pos_res+length beyond the result tape: task.rs:44/48 panics    */
    V2P_ERR_SRC_OOB = 6,        /* start_pos+length beyond the ref/alt tape:    task.rs:44/48 panics    */
    V2P_ERR_NOT_CONTIGUOUS = 7, /* V2P_FLAG_VALIDATE: gir.rs:208-225 (DEBUG_CPU_EXEC / DEBUG_GPU) check */
    /* 8 is reserved (UTF-32 tapes are executed natively as 4-byte units, any code point is fine)       */
    V2P_ERR_NOT_GPU_ENGINE = 9, /* v2p_gir_execute called with ST/MT: those stay in the caller          */
    V2P_ERR_TASKGEN = 10,       /* device task generation: the reference aborts on this transcript (usize
                                   underflow in add_till_next_ins / add_last_instruction, negative result size) */
    V2P_ERR_VCF_PARSE = 11,     /* VCF text outside the dialect of include/v2p_vcf.h (message: line, sample)  */
    V2P_ERR_BGZF = 12           /* input that is not valid BGZF (include/v2p_vcf.h; message: block, byte, class) */
};

/* ---- engine selection (engines.rs:15-30) ------------------------------------------------------- */
enum { V2P_ENGINE_ST = 0, V2P_ENGINE_MT = 1, V2P_ENGINE_GPU = 2 };

/* Engine::from_str (engines.rs:20-29): exactly "st"|"ST" -> ST, "mt"|"MT" -> MT, "gpu"|"GPU" -> GPU;
 * anything else (including "Gpu") -> V2P_ERR_BAD_ENGINE. */
int v2p_engine_from_str(const char* s, int* engine_kind);

/* ---- flags ------------------------------------------------------------------------------------- */
#define V2P_FLAG_FILL_DOT 0x1u    /* library pre-fills the result tape with '.' (haplotype_instruction.rs:78);
                                     without it uncovered result units keep the caller's content (soa only) */
#define V2P_FLAG_VALIDATE 0x2u    /* run the gir.rs:203-229 contiguity check; report first bad index, copy nothing */
#define V2P_FLAG_DEVICE_PTRS 0x4u /* batch call: every data pointer is device memory on the engine's GPU  */
#define V2P_FLAG_ASYNC 0x8u       /* batch call: enqueue and return; completion + status via v2p_event_wait */
#define V2P_FLAG_ALIGNED_LAYOUT 0x10u /* batch call, performance hint only (results never depend on it): the producer
                                     placed every transcript's result in phase (mod 16) with its source in the
                                     reference tape (v2p::HaplotypeBatch aligned layout, V2P_GEN_ALIGNED), so tiles
                                     are processed in tape order instead of the haplotype-interleaved order that keeps
                                     the replicas of the reference resident in L2 for the reference's own layout */

/* ---- lifecycle --------------------------------------------------------------------------------- */
typedef struct v2p_engine v2p_engine;
typedef struct v2p_event v2p_event;

/* One context per GPU; usable from any host thread.  Replaces nothing in the reference (its GPU build
 * is not in the tree, README.md:225-267); corresponds to process start-up of `-g gpu` (cli.rs:57-71). */
int v2p_engine_create(int cuda_device, v2p_engine** out);
void v2p_engine_destroy(v2p_engine* e);
/* Message of the last failure on this context ("" if none).  Valid until the next call on `e`. */
const char* v2p_last_error(v2p_engine* e);
int v2p_abi_version(void);
/* CUDA device ordinal the context was created on. */
int v2p_engine_device(v2p_engine* e);

/* Pinned host memory for tapes / task arrays so H2D/D2H run at PCIe rate (optional helper). */
int v2p_host_alloc(void** ptr, size_t bytes);
int v2p_host_free(void* ptr);

/* Register the reference proteome (the reference keeps it in a HashMap<String,String>, readers.rs:58-98; here it is
 * one concatenated residue tape).  The tape is copied into HBM once together with 16 byte-shifted replicas, so that
 * whatever (destination - source) phase a reference run has, one replica holds it at the output's 16-byte phase and
 * its fully covered vectors are plain aligned TMA bulk copies into the shared-memory output tile (TMA cannot start at
 * an arbitrary byte: a tensor load with a coordinate that is not 16-byte aligned faults, profiles/dev/tma_probe.cu).
 * Batches that pass ref == NULL and ref_base == NULL index this tape (Task.start_pos = transcript offset in the tape
 * + position).  flags: V2P_FLAG_DEVICE_PTRS if `ref` is device memory, optionally V2P_REF_NO_TMA.               */
#define V2P_REF_NO_TMA 0x200u /* keep one copy only; every run takes the register path (2 aligned loads + funnel shift) */
int v2p_engine_set_reference(v2p_engine* e, const uint8_t* ref, uint64_t n_ref, uint32_t flags);

/* ---- (i) reference-faithful single-haplotype call == GIR::execute(Engine::GPU) ------------------- */
/* Replaces gir.rs:236-239.  The SoA shape is the reference's own hand-off,
 * GIR::consume_and_produce_produce_content (gir.rs:283-299): four `usize` arrays (exe_code widened,
 * start_pos, length, start_pos_res) and three UTF-32 `char` tapes.  Host pointers only.
 *   - res_utf32 is in/out: with V2P_FLAG_FILL_DOT it is overwritten entirely ('.' where no task writes),
 *     otherwise units not covered by any task are left untouched (task.rs:118-144 relies on this).
 *   - tasks are applied in array order (later tasks win on overlap), exactly like gir.rs:233.
 *   - on any error nothing is guaranteed about res_utf32 (the reference aborts the process there);
 *     *bad_index (may be NULL) receives the offending task index.
 */
int v2p_execute_soa(v2p_engine* e, size_t n_tasks, const uint64_t* exec_code, const uint64_t* start_pos,
                    const uint64_t* length, const uint64_t* start_pos_res, const uint32_t* ref_utf32, size_t n_ref,
                    const uint32_t* alt_utf32, size_t n_alt, uint32_t* res_utf32, size_t n_res, uint32_t flags,
                    uint64_t* bad_index);

/* Same call through the engine selector: engine_kind must be V2P_ENGINE_GPU (ST/MT stay in the caller,
 * gir.rs:201-235) -> V2P_ERR_NOT_GPU_ENGINE otherwise. */
int v2p_gir_execute(v2p_engine* e, int engine_kind, size_t n_tasks, const uint64_t* exec_code,
                    const uint64_t* start_pos, const uint64_t* length, const uint64_t* start_pos_res,
                    const uint32_t* ref_utf32, size_t n_ref, const uint32_t* alt_utf32, size_t n_alt,
                    uint32_t* res_utf32, size_t n_res, uint32_t flags, uint64_t* bad_index);

/* ---- (ii) native batched call: many haplotypes, 1-byte residues, packed tasks -------------------- */
/* One Task (task.rs:2-9) packed to 16 bytes.  Offsets are relative to the owning haplotype's tape bases. */
typedef struct {
    uint32_t src_off; /* Task::start_pos      (in the ref tape if stream==0, else in the alt tape) */
    uint32_t len;     /* Task::length                                                              */
    uint32_t dst_off; /* Task::start_pos_res  (authoritative: gaps stay '.')                       */
    uint32_t stream;  /* Task::exe_code: 0 = reference tape, 1 = alteration tape; other -> error   */
} v2p_task16;

typedef struct {
    const uint64_t* task_begin; /* n_hap+1: tasks of haplotype h are tasks[task_begin[h] .. task_begin[h+1])    */
    const v2p_task16* tasks;    /* task_begin[n_hap] entries                                                  */
    const uint8_t* ref;         /* reference residues; NULL (with ref_base NULL) = the registered reference   */
    const uint64_t* ref_base;   /* n_hap+1 per-haplotype ref-tape bounds, or NULL: all haplotypes share the   */
    uint64_t n_ref;             /*   whole tape ref[0..n_ref) (the proteome; tasks then carry global offsets) */
    const uint8_t* alt;         /* concatenated alteration tapes                                              */
    const uint64_t* alt_base;   /* n_hap+1                                                                    */
    uint8_t* out;               /* concatenated result tapes, out_base[n_hap] bytes; 16-byte aligned          */
    const uint64_t* out_base;   /* n_hap+1, non-decreasing                                                    */
    uint64_t n_hap;
    /* Totals == last entries of the base arrays.  REQUIRED with V2P_FLAG_DEVICE_PTRS (the host cannot read  */
    /* device arrays without a sync; the plan kernel cross-checks them); ignored for host pointers.          */
    uint64_t n_tasks; /* task_begin[n_hap] */
    uint64_t n_alt;   /* alt_base[n_hap]   */
    uint64_t n_out;   /* out_base[n_hap]   */
} v2p_batch;

typedef struct {
    int status;        /* V2P_OK or the first error class found                          */
    uint64_t bad_hap;  /* haplotype of the lowest offending task (when status != V2P_OK) */
    uint64_t bad_task; /* its index within that haplotype                                */
    float kernel_ms;   /* device time of the launch group (plan + copy), CUDA events     */
    float copy_ms;     /* device time of the dominant kernel alone (k_copy_tiles)        */
} v2p_result;

/* Executes every haplotype of the batch == n_hap calls of GIR::execute (gir.rs:197-241), one launch group.
 * Result tapes are always '.'-prefilled (V2P_FLAG_FILL_DOT is implied: the batch owns `out`).
 * Fast path requires each haplotype's tasks sorted by dst_off and non-overlapping -- the invariant
 * haplotype_instruction.rs:94-133 produces; any other order is still executed on the GPU with the
 * reference's serial semantics (later task wins), only slower.
 * Without V2P_FLAG_DEVICE_PTRS all pointers are host memory (pinned recommended) and the call performs
 * H2D of tasks/tapes and D2H of `out` on the engine's streams.
 * With V2P_FLAG_ASYNC `*done` receives an event; result via v2p_event_wait.  Otherwise `res` is filled. */
int v2p_execute_batch(v2p_engine* e, const v2p_batch* batch, uint32_t flags, v2p_result* res, v2p_event** done);
int v2p_event_wait(v2p_engine* e, v2p_event* ev, v2p_result* res); /* also releases the event */

/* Launch-level introspection for bench.py: kernels launched by this context since creation. */
uint64_t v2p_kernel_launch_count(v2p_engine* e);
/* Load-balance evidence (SURVEY.md 8d, skew stress): with profiling on, every warp of the copy kernel's persistent
 * grid records its wall time (ns, %globaltimer) for device-pointer batches on the engine stream;
 * v2p_engine_read_warp_ns returns the last launch's values (n_warps entries; call with ns_out == NULL to size it).
 * max / mean of them is what a skewed Task array would push up if a long segment pinned one worker. */
int v2p_engine_profile_warps(v2p_engine* e, int on);
int v2p_engine_read_warp_ns(v2p_engine* e, uint64_t* ns_out, uint64_t cap, uint64_t* n_warps);

/* Kernel tunables for profiling sweeps: copy-kernel variant (-1 = automatic choice, the default) and CTAs per SM
 * (0 = the variant's own). */
int v2p_engine_set_tuning(v2p_engine* e, int variant, int ctas_per_sm);
/* Run on a caller-owned CUDA stream (a cudaStream_t / CUstream handle, e.g. torch's current stream) so the
 * caller's own events bracket the kernels; NULL restores the engine's private non-blocking stream. */
int v2p_engine_set_stream(v2p_engine* e, void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* V2P_ENGINE_H */
