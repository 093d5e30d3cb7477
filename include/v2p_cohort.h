/*
 * v2p_cohort.h -- one process, all the GPUs of the box: a cohort's site lists in, every sample's .fasta / .fasta.gz
 * file image out, the samples split into contiguous ranges over the devices.
 *
 * What it stands for in the reference: parts/exec.rs:34-40 -- ONE process fans the probands out over a rayon pool
 * (`vec_int_repr.into_par_iter().map(...)`) -- and parts/io.rs:45-57, where the same pool writes one file per
 * proband.  Here the pool is one host thread per GPU, each with its own engine (proteome registered), catalogue
 * lanes, pinned staging ring and v2p_pipeline (include/v2p_pipeline.h); GPU g owns a contiguous sample range
 * (BASELINE.json north_star: "each GPU owning a contiguous sample range with its own pinned host staging and async
 * copy-back to the FASTA writer"), ranges balanced by the number of variant sites the samples carry (the size of a
 * sample's result tape is, to within a percent, proportional to it; the tapes themselves only exist on the devices).
 * There is no collective and no peer traffic: haplotypes are independent and the proteome is replicated.
 * A caller that links this library needs no torchrun / MPI launcher to use every GPU.
 *
 * The same device may be named more than once (two workers share one GPU: useful on a one-GPU box and in tests).
 */
#ifndef V2P_COHORT_H
#define V2P_COHORT_H

#include <stddef.h>
#include <stdint.h>

#include "v2p_pipeline.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct v2p_cohort v2p_cohort;

#define V2P_COHORT_MAX_DEVICES 16

/* The inputs every device needs (host pointers, copied / uploaded during create):
 *   proteome[n_proteome]      the reference tape (v2p_engine_set_reference on every device)
 *   tx_offsets[n_tx+1]        offset of every transcript in it
 *   name_off[n_tx+1], names   transcript names of the FASTA headers (v2p_catalogue_set_names)
 * and ONE of the two catalogue forms of include/v2p_taskgen.h:
 *   general == 0: the seven-class tables   (arguments of v2p_catalogue_create;     ins_* unused)
 *   general != 0: reference Instructions   (arguments of v2p_catalogue_create_ins; site_pos/cls/rlen unused)        */
typedef struct {
    const uint8_t* proteome;
    uint64_t n_proteome;
    uint64_t n_tx;
    const uint64_t* tx_offsets;
    const uint64_t* name_off;
    const uint8_t* names;
    int general;
    uint64_t n_sites;
    const uint32_t* site_tx;
    const uint32_t* site_pos;   /* seven-class */
    const uint8_t* site_cls;    /* seven-class */
    const uint32_t* site_rlen;  /* seven-class */
    const uint8_t* ins_code;    /* general */
    const uint8_t* ins_flags;   /* general */
    const uint32_t* ins_pos_ref;
    const uint32_t* ins_pos_res;
    const uint32_t* ins_len;
    const uint64_t* site_doff;  /* both */
    const uint32_t* site_dlen;  /* both */
    const uint8_t* pool;
    uint64_t n_pool;
} v2p_cohort_inputs;

/* devices[n_devices]: CUDA ordinals, one worker each (1..V2P_COHORT_MAX_DEVICES).  lanes_per_device: chunks in flight
 * per worker (1..V2P_PIPE_MAX_LANES; 0 = 2).  Fails with V2P_ERR_CUDA when a device is missing -- no CPU fallback. */
int v2p_cohort_create(const int* devices, uint32_t n_devices, const v2p_cohort_inputs* in, uint32_t lanes_per_device,
                      v2p_cohort** out);
void v2p_cohort_destroy(v2p_cohort* c);
const char* v2p_cohort_last_error(v2p_cohort* c);

typedef struct {
    uint32_t n_devices;
    v2p_pipeline_result total;                              /* counters summed over the workers; wall_s = the whole call */
    v2p_pipeline_result per_device[V2P_COHORT_MAX_DEVICES]; /* each worker's own counters and wall clock                 */
    uint64_t first_sample[V2P_COHORT_MAX_DEVICES + 1];      /* worker g ran samples [first_sample[g], first_sample[g+1]) */
} v2p_cohort_result;

#define V2P_COHORT_CONCURRENT_SINK 0x100u /* the sink is thread-safe: workers call it concurrently (v2p_dir_writer_sink
                                           * is); without the flag calls are serialised by a lock                        */

/* Prepares V2P_PIPE_ALL_RECORDS (the reference's `-a`, personalized_genome.rs:120-210) on every worker:
 * v2p_pipeline_enable_all_records with the proteome, transcript offsets and names of `in` (the same arrays create got;
 * the catalogue fields are not read).  The workers do it in parallel. */
int v2p_cohort_enable_all_records(v2p_cohort* c, const v2p_cohort_inputs* in);

/* site_begin[2*n_samples+1] / sites: the whole cohort's CSR lists (host pointers), haplotype h = 2*sample + (hap-1).
 * flags: V2P_PIPE_GZIP, V2P_PIPE_SKIP_ABORTS, V2P_PIPE_ALL_RECORDS (include/v2p_pipeline.h), V2P_COHORT_CONCURRENT_SINK.
 * The sink is called per chunk with cohort-wide sample numbers; inside one worker's range chunks arrive in sample
 * order, chunks of different workers interleave (the reference writes its files from a parallel pool too).
 * The first failing worker's status is returned (its message in v2p_cohort_last_error); the others finish their
 * chunk in flight and stop. */
int v2p_cohort_run_lists(v2p_cohort* c, uint64_t n_samples, const uint64_t* site_begin, const uint32_t* sites,
                         uint32_t chunk_samples, uint32_t flags, v2p_file_sink sink, void* user, v2p_cohort_result* res);

#define V2P_COHORT_DEVICE_MASKS 0x200u /* v2p_cohort_run_masks: `masks` is device memory on the FIRST worker's device (e.g.
                                        * v2p_vcf_parse_masks, include/v2p_vcf.h); it is decoded there without an upload */

/* Same from the FORMAT/BCSQ mask matrix (host memory, or with V2P_COHORT_DEVICE_MASKS device memory on the first
 * worker's device; arguments as v2p_sites_from_masks, include/v2p_taskgen.h).
 * The matrix is decoded ONCE, on the first worker's device (the decode reads every record of every sample exactly once
 * and is a fraction of a percent of the job); its CSR lists -- 4 bytes per carried site -- come back to the host, are
 * split by the rule above and each worker uploads its own range.  res->total.decode_ms includes the decode, and
 * h2d_bytes the matrix upload (none with V2P_COHORT_DEVICE_MASKS). */
int v2p_cohort_run_masks(v2p_cohort* c, uint64_t n_records, uint64_t n_samples, uint32_t words_per_cell,
                         const uint32_t* masks, const uint64_t* csq_begin, const int32_t* csq_site, uint32_t chunk_samples,
                         uint32_t flags, v2p_file_sink sink, void* user, v2p_cohort_result* res);

/* Kernel launches of all workers' engines since create (v2p_kernel_launch_count summed). */
uint64_t v2p_cohort_launch_count(v2p_cohort* c);

#ifdef __cplusplus
}
#endif
#endif /* V2P_COHORT_H */
