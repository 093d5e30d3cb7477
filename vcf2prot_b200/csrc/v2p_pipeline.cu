// v2p_pipeline.cu -- site lists / bit-masks -> per-sample .fasta(.gz) file images in host memory (include/v2p_pipeline.h).
//
// Host-side sequencing only: every byte is produced by the kernels behind v2p_generate_tasks (V2P_GEN_FASTA),
// v2p_execute_batch and v2p_gzip_files; this file chains them per chunk of samples through the public C ABI and
// overlaps each chunk's copy-back with the next chunk's kernels (one copy stream + one event per lane).  It stands
// where the reference loops over probands on rayon threads (parts/exec.rs:27-41) and writes one file per proband
// (parts/io.rs:45-57, personalized_genome.rs:72-117).  No CPU fallback: any stage that fails fails the call.
#include <cuda_runtime.h>
#include <fcntl.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <mutex>
#include <thread>
#include <chrono>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "v2p_allrecords.cuh"
#include "v2p_hostres.cuh"
#include "v2p_mapped.cuh"
#include "v2p_pipeline.h"

using namespace v2p;

namespace {

struct Lane {
    v2p_catalogue* cat = nullptr;  // borrowed
    v2p_gzip* gz = nullptr;        // owned
    cudaStream_t copy = nullptr;
    cudaEvent_t landed = nullptr;
    DevBuf d_gz;      // compressed chunk
    DevBuf d_begin;   // rebased site_begin of the chunk (mask entry point)
    MappedBuf pub;    // out_base of the chunk, published by a kernel (v2p_mapped.cuh)
    PinnedBuf h_buf;  // staging (sink mode)
    // `-a` expansion of the chunk (V2P_PIPE_ALL_RECORDS, v2p_allrecords.cuh): scratch, the merged Task array, its tape
    DevBuf ar[12];
    // the chunk in flight
    bool pending = false;
    uint64_t first_sample = 0, n = 0;
    const uint8_t* h_data = nullptr;
    std::vector<uint64_t> fb_rel;
};

}  // namespace

struct v2p_pipeline {
    v2p_engine* eng = nullptr;
    int device = 0;
    uint32_t n_lanes = 0;
    cudaStream_t aux = nullptr;  // small kernels of the pipeline itself (never behind a copy-back)
    Lane lanes[V2P_PIPE_MAX_LANES];
    std::string err;
    // `-a`: tables of the extended reference tape (v2p_pipeline_enable_all_records)
    bool all_on = false;
    v2p_ar::Tables tab{};
    DevBuf d_tab[4];
    uint64_t n_proteome = 0;
};

namespace {

double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// the chunk's bytes have landed: hand them to the sink (chunks retire in sample order, lanes rotate)
int retire(v2p_pipeline* p, Lane& l, v2p_file_sink sink, void* user, v2p_pipeline_result* res) {
    if (!l.pending) return V2P_OK;
    l.pending = false;
    const double t0 = now_s();
    CU(p->err, cudaEventSynchronize(l.landed));
    const double t1 = now_s();
    res->wait_wall_s += t1 - t0;
    const int stop = sink ? sink(user, l.first_sample, l.n, l.h_data, l.fb_rel.data()) : 0;
    res->sink_wall_s += now_s() - t1;
    if (stop != 0)
        return fail(p->err, V2P_ERR_INVALID_ARG, "the file sink stopped the run at sample %llu", (unsigned long long)l.first_sample);
    return V2P_OK;
}

// `-a`: the generated chunk's Task array with three reference-stream segments per unaltered transcript appended to
// every haplotype (v2p_allrecords.cuh).  -> *xb, a device-pointer batch whose arrays live in the lane; *n_extra_records.
int expand_all_records(v2p_pipeline* p, Lane& l, const v2p_generated& g, v2p_batch* xb, uint64_t* n_extra_records) {
    using namespace v2p_ar;
    const uint64_t nh = g.batch.n_hap, nr = g.n_rows, nt = g.batch.n_tasks;
    cudaStream_t st = p->aux;
    int rc;
    for (int i : {0, 3, 4, 5, 6, 7, 8}) CU(p->err, l.ar[i].need((nh + 1) * 8));  // per haplotype
    for (int i : {1, 2}) CU(p->err, l.ar[i].need((nr + 1) * 8));                 // per annotation row
    Chunk c{};
    c.n_hap = nh, c.n_rows = nr, c.n_tasks = nt;
    c.ann_hap = g.ann_hap, c.ann_tx = g.ann_tx, c.task_begin = g.batch.task_begin, c.out_base = g.batch.out_base, c.tasks = g.batch.tasks;
    c.row_begin = (uint64_t*)l.ar[0].p, c.row_bytes = (uint64_t*)l.ar[1].p, c.row_x = (uint64_t*)l.ar[2].p;
    c.ut = (uint64_t*)l.ar[3].p, c.ut_x = (uint64_t*)l.ar[4].p, c.ub = (uint64_t*)l.ar[5].p, c.ub_x = (uint64_t*)l.ar[6].p;
    c.new_tb = (uint64_t*)l.ar[7].p, c.new_ob = (uint64_t*)l.ar[8].p;
    k_ar_rows<<<blocks(std::max(nh, nr) + 1), 256, 0, st>>>(c, p->tab);
    if ((rc = exclusive_sum(p->err, l.ar[9], (const uint64_t*)c.row_bytes, c.row_x, nr + 1, st))) return rc;
    k_ar_hap<<<blocks(nh + 1), 256, 0, st>>>(c, p->tab);
    if ((rc = exclusive_sum(p->err, l.ar[9], (const uint64_t*)c.ut, c.ut_x, nh + 1, st)) ||
        (rc = exclusive_sum(p->err, l.ar[9], (const uint64_t*)c.ub, c.ub_x, nh + 1, st)))
        return rc;
    k_ar_bases<<<blocks(nh + 1), 256, 0, st>>>(c);
    CU(p->err, l.pub.reserve(64));
    v2p::PubList pl{};
    pl.src[0] = (const unsigned long long*)(c.ut_x + nh), pl.src[1] = (const unsigned long long*)(c.ub_x + nh), pl.n = 2;
    v2p::k_publish_list<<<1, 32, 0, st>>>(l.pub.p, pl);
    CU(p->err, cudaStreamSynchronize(st));
    const uint64_t extra_tasks = l.pub.p[0], extra_bytes = l.pub.p[1];
    const uint64_t n_tasks = nt + extra_tasks, n_out = g.batch.n_out + extra_bytes;
    CU(p->err, l.ar[10].need((n_tasks + 1) * sizeof(v2p_task16)));
    CU(p->err, l.ar[11].need(n_out + 64));
    c.new_tasks = (v2p_task16*)l.ar[10].p;
    if (nt) k_ar_move<<<blocks(nt), 256, 0, st>>>(c);
    if (nh && p->tab.n_tx) k_ar_emit<<<blocks(nh * p->tab.n_tx), 256, 0, st>>>(c, p->tab, p->n_proteome);
    CU(p->err, cudaGetLastError());
    CU(p->err, cudaStreamSynchronize(st));
    *xb = g.batch;
    xb->task_begin = c.new_tb, xb->tasks = c.new_tasks, xb->out = (uint8_t*)l.ar[11].p, xb->out_base = c.new_ob;
    xb->n_tasks = n_tasks, xb->n_out = n_out;
    *n_extra_records = extra_tasks / 3;
    return V2P_OK;
}

// What differs between the two entry points: how chunk [h0,h1) gets its Task batch.
struct ListSource {
    const uint64_t* site_begin;  // host, n_hap+1 (absolute indices into `sites`)
    const uint32_t* h_sites;     // host lists, or
    const uint32_t* d_sites;     // device lists (mask entry point)
};

int run(v2p_pipeline* p, uint64_t n_samples, const ListSource& src, uint32_t chunk_samples, uint32_t flags, uint8_t* out,
        uint64_t out_capacity, uint64_t* file_begin, v2p_file_sink sink, void* user, v2p_pipeline_result* res) {
    if (!out && !sink) return fail(p->err, V2P_ERR_INVALID_ARG, "neither an output buffer nor a sink was given");
    if (out && !file_begin) return fail(p->err, V2P_ERR_INVALID_ARG, "file_begin is NULL");
    if (!chunk_samples) chunk_samples = 128;
    const bool gzip = (flags & V2P_PIPE_GZIP) != 0, all_records = (flags & V2P_PIPE_ALL_RECORDS) != 0;
    if (all_records && !p->all_on)
        return fail(p->err, V2P_ERR_INVALID_ARG, "V2P_PIPE_ALL_RECORDS needs v2p_pipeline_enable_all_records first");
    const uint32_t gen_flags = V2P_GEN_FASTA | ((flags & V2P_PIPE_SKIP_ABORTS) ? V2P_GEN_SKIP_ABORTS : 0u);
    CU(p->err, cudaSetDevice(p->device));
    for (uint32_t i = 0; i < p->n_lanes; ++i) p->lanes[i].pending = false;
    uint64_t total = 0;
    if (file_begin) file_begin[0] = 0;
    std::vector<uint64_t> sb;
    uint64_t ci = 0;
    int rc = V2P_OK;
    for (uint64_t s0 = 0; s0 < n_samples && rc == V2P_OK; s0 += chunk_samples, ++ci) {
        const uint64_t ns = std::min<uint64_t>(chunk_samples, n_samples - s0), h0 = 2 * s0, nh = 2 * ns;
        Lane& l = p->lanes[ci % p->n_lanes];
        if ((rc = retire(p, l, sink, user, res))) break;
        // ---- Task batch of the chunk, generated on the device with the record framing in it
        sb.resize(nh + 1);
        for (uint64_t h = 0; h <= nh; ++h) sb[h] = src.site_begin[h0 + h] - src.site_begin[h0];
        v2p_generated g;
        const double t_gen0 = now_s();
        if (src.h_sites) {
            rc = v2p_generate_tasks(l.cat, nh, sb.data(), src.h_sites + src.site_begin[h0], gen_flags, &g);
            res->h2d_bytes += sb[nh] * 4 + (nh + 1) * 8;
        } else {
            CU_BREAK(p->err, rc, l.d_begin.need((nh + 1) * 8));
            CU_BREAK(p->err, rc, cudaMemcpy(l.d_begin.p, sb.data(), (nh + 1) * 8, cudaMemcpyHostToDevice));
            v2p_site_lists lists;
            memset(&lists, 0, sizeof lists);
            lists.n_hap = nh, lists.n_sites = sb[nh];
            lists.site_begin = (const uint64_t*)l.d_begin.p, lists.sites = src.d_sites + src.site_begin[h0];
            rc = v2p_generate_tasks_from_lists(l.cat, &lists, gen_flags, &g);
            res->h2d_bytes += (nh + 1) * 8;
        }
        if (rc) {
            fail(p->err, rc, "task generation failed at sample %llu: %s", (unsigned long long)s0, v2p_catalogue_last_error(l.cat));
            break;
        }
        // ---- `-a`: the unaltered transcripts' records behind every haplotype's altered ones (write_all)
        v2p_batch xb = g.batch;
        uint64_t extra_records = 0;
        if (all_records && (rc = expand_all_records(p, l, g, &xb, &extra_records))) break;
        const double t_exec0 = now_s();
        res->gen_wall_s += t_exec0 - t_gen0;
        // ---- the hot path: every haplotype's result tape == its FASTA text
        v2p_result er;
        if ((rc = v2p_execute_batch(p->eng, &xb, V2P_FLAG_DEVICE_PTRS, &er, nullptr))) {
            fail(p->err, rc, "execution failed at sample %llu (haplotype %llu task %llu): %s", (unsigned long long)s0,
                 (unsigned long long)er.bad_hap, (unsigned long long)er.bad_task, v2p_last_error(p->eng));
            break;
        }
        res->exec_wall_s += now_s() - t_exec0;
        // ---- file bounds: sample s owns haplotypes 2s, 2s+1
        CU_BREAK(p->err, rc, l.pub.reserve(nh + 1));
        CU_BREAK(p->err, rc, v2p::publish_words(l.pub.p, xb.out_base, nh + 1, p->aux));
        CU_BREAK(p->err, rc, cudaStreamSynchronize(p->aux));
        l.fb_rel.resize(ns + 1);
        for (uint64_t s = 0; s <= ns; ++s) l.fb_rel[s] = l.pub.p[2 * s];
        const uint8_t* d_src = xb.out;
        uint64_t bytes = xb.n_out;
        if (gzip) {
            const uint64_t cap = v2p_gzip_bound(xb.n_out, ns);
            CU_BREAK(p->err, rc, l.d_gz.need(cap));
            std::vector<uint64_t> fb_abs(l.fb_rel);
            v2p_gzip_result zr;
            if ((rc = v2p_gzip_files(l.gz, xb.out, fb_abs.data(), ns, (uint8_t*)l.d_gz.p, cap, l.fb_rel.data(),
                                     V2P_FLAG_DEVICE_PTRS, &zr))) {
                fail(p->err, rc, "gzip failed at sample %llu: %s", (unsigned long long)s0, v2p_gzip_last_error(l.gz));
                break;
            }
            res->gzip_ms += zr.ms;
            res->gzip_wall_s += zr.ms * 1e-3;
            d_src = (const uint8_t*)l.d_gz.p;
            bytes = l.fb_rel[ns];
        }
        // ---- copy-back on the lane's own stream: overlaps the next chunk's kernels
        uint8_t* h_dst;
        if (out) {
            if (total + bytes > out_capacity) {
                rc = fail(p->err, V2P_ERR_RES_OOB, "output needs more than %llu bytes (at sample %llu)", (unsigned long long)out_capacity,
                          (unsigned long long)s0);
                break;
            }
            h_dst = out + total;
        } else {
            CU_BREAK(p->err, rc, l.h_buf.need(bytes));
            h_dst = (uint8_t*)l.h_buf.p;
        }
        if (bytes) CU_BREAK(p->err, rc, cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, l.copy));
        CU_BREAK(p->err, rc, cudaEventRecord(l.landed, l.copy));
        l.pending = true, l.first_sample = s0, l.n = ns, l.h_data = h_dst;
        if (file_begin)
            for (uint64_t s = 1; s <= ns; ++s) file_begin[s0 + s] = total + l.fb_rel[s];
        total += bytes;
        res->n_sites += g.n_sites, res->n_tasks += xb.n_tasks, res->n_records += g.n_rows + extra_records;
        res->image_bytes += xb.n_out, res->out_bytes += bytes;
        res->gen_ms += g.gen_ms, res->exec_ms += er.kernel_ms;
        res->n_skipped += g.n_skipped, res->n_aborted += g.n_aborted;
        res->n_chunks++;
    }
    // drain in order: the oldest chunk sits in the lane the next chunk would have taken
    for (uint32_t k = 0; k < p->n_lanes; ++k) {
        Lane& l = p->lanes[(ci + k) % p->n_lanes];
        if (rc == V2P_OK) rc = retire(p, l, sink, user, res);
        else if (l.pending) cudaEventSynchronize(l.landed), l.pending = false;
    }
    return rc;
}

}  // namespace

extern "C" {

int v2p_pipeline_create(v2p_engine* e, v2p_catalogue* const* lanes, uint32_t n_lanes, v2p_pipeline** out) {
    if (!out) return V2P_ERR_INVALID_ARG;
    *out = nullptr;
    if (!e || !lanes || n_lanes < 1 || n_lanes > V2P_PIPE_MAX_LANES) return V2P_ERR_INVALID_ARG;
    for (uint32_t i = 0; i < n_lanes; ++i) {
        if (!lanes[i]) return V2P_ERR_INVALID_ARG;
        for (uint32_t k = 0; k < i; ++k)
            if (lanes[k] == lanes[i]) return V2P_ERR_INVALID_ARG;  // a lane owns the buffers of a chunk in flight
    }
    v2p_pipeline* p = new (std::nothrow) v2p_pipeline();
    if (!p) return V2P_ERR_INVALID_ARG;
    p->eng = e;
    p->device = v2p_engine_device(e);
    p->n_lanes = n_lanes;
    bool ok = cudaSetDevice(p->device) == cudaSuccess && cudaStreamCreateWithFlags(&p->aux, cudaStreamNonBlocking) == cudaSuccess;
    for (uint32_t i = 0; ok && i < n_lanes; ++i) {
        Lane& l = p->lanes[i];
        l.cat = lanes[i];
        ok = v2p_gzip_create(p->device, &l.gz) == V2P_OK &&
             cudaStreamCreateWithFlags(&l.copy, cudaStreamNonBlocking) == cudaSuccess &&
             cudaEventCreateWithFlags(&l.landed, cudaEventDisableTiming) == cudaSuccess;
    }
    if (!ok) {
        v2p_pipeline_destroy(p);
        return V2P_ERR_CUDA;
    }
    *out = p;
    return V2P_OK;
}

void v2p_pipeline_destroy(v2p_pipeline* p) {
    if (!p) return;
    cudaSetDevice(p->device);
    for (uint32_t i = 0; i < p->n_lanes; ++i) {
        Lane& l = p->lanes[i];
        if (l.copy) cudaStreamSynchronize(l.copy), cudaStreamDestroy(l.copy);
        if (l.landed) cudaEventDestroy(l.landed);
        if (l.gz) v2p_gzip_destroy(l.gz);
    }
    if (p->aux) cudaStreamDestroy(p->aux);
    delete p;  // frees every buffer
}

int v2p_pipeline_enable_all_records(v2p_pipeline* p, const uint8_t* proteome, uint64_t n_proteome, uint64_t n_tx,
                                    const uint64_t* tx_offsets, const uint64_t* name_off, const uint8_t* names) {
    if (!p) return V2P_ERR_INVALID_ARG;
    p->err.clear();
    if (!tx_offsets || !name_off || (n_proteome && !proteome) || (n_tx && name_off[n_tx] && !names))
        return fail(p->err, V2P_ERR_INVALID_ARG, "NULL argument");
    if (tx_offsets[n_tx] > n_proteome) return fail(p->err, V2P_ERR_INVALID_ARG, "tx_offsets run past the proteome tape");
    // extended tape: proteome | for every transcript ">{name}_1\n" ">{name}_2\n"
    std::vector<uint8_t> ext(proteome, proteome + n_proteome);
    std::vector<uint64_t> hdr(n_tx), rec_x(n_tx + 1, 0);
    std::vector<uint32_t> nlen(n_tx);
    for (uint64_t t = 0; t < n_tx; ++t) {
        if (name_off[t + 1] < name_off[t] || tx_offsets[t + 1] < tx_offsets[t]) return fail(p->err, V2P_ERR_INVALID_ARG, "offsets not monotone");
        const uint64_t nl = name_off[t + 1] - name_off[t];
        nlen[t] = (uint32_t)nl;
        hdr[t] = ext.size();
        for (int k = 1; k <= 2; ++k) {
            ext.push_back('>');
            ext.insert(ext.end(), names + name_off[t], names + name_off[t + 1]);
            ext.push_back('_');
            ext.push_back((uint8_t)('0' + k));
            ext.push_back('\n');
        }
        rec_x[t + 1] = rec_x[t] + nl + 5 + (tx_offsets[t + 1] - tx_offsets[t]);
    }
    if (ext.size() >> 32) return fail(p->err, V2P_ERR_INVALID_ARG, "extended reference tape exceeds 4 GiB");
    int rc = v2p_engine_set_reference(p->eng, ext.data(), ext.size(), 0);
    if (rc) return fail(p->err, rc, "registering the extended reference tape failed: %s", v2p_last_error(p->eng));
    CU(p->err, cudaSetDevice(p->device));
    const void* src[4] = {tx_offsets, hdr.data(), nlen.data(), rec_x.data()};
    const size_t bytes[4] = {(n_tx + 1) * 8, n_tx * 8, n_tx * 4, (n_tx + 1) * 8};
    for (int i = 0; i < 4; ++i) {
        CU(p->err, p->d_tab[i].need(bytes[i] + 16));
        CU(p->err, cudaMemcpy(p->d_tab[i].p, src[i], bytes[i], cudaMemcpyHostToDevice));
    }
    p->tab = v2p_ar::Tables{n_tx, (const uint64_t*)p->d_tab[0].p, (const uint64_t*)p->d_tab[1].p, (const uint32_t*)p->d_tab[2].p,
                            (const uint64_t*)p->d_tab[3].p};
    p->n_proteome = n_proteome;
    p->all_on = true;
    return V2P_OK;
}

const char* v2p_pipeline_last_error(v2p_pipeline* p) { return p ? p->err.c_str() : "pipeline is NULL"; }

int v2p_pipeline_run_lists(v2p_pipeline* p, uint64_t n_samples, const uint64_t* site_begin, const uint32_t* sites,
                           uint32_t chunk_samples, uint32_t flags, uint8_t* out, uint64_t out_capacity, uint64_t* file_begin,
                           v2p_file_sink sink, void* user, v2p_pipeline_result* res) {
    if (!p) return V2P_ERR_INVALID_ARG;
    p->err.clear();
    v2p_pipeline_result local;
    memset(&local, 0, sizeof local);
    if (res) *res = local;  // (also on the argument errors below)
    if (!site_begin || site_begin[0] != 0) return fail(p->err, V2P_ERR_INVALID_ARG, "site_begin is NULL or does not start at 0");
    for (uint64_t h = 0; h < 2 * n_samples; ++h)
        if (site_begin[h + 1] < site_begin[h]) return fail(p->err, V2P_ERR_INVALID_ARG, "site_begin not monotone at haplotype %llu", (unsigned long long)h);
    if (site_begin[2 * n_samples] && !sites) return fail(p->err, V2P_ERR_INVALID_ARG, "sites is NULL");
    const auto t0 = std::chrono::steady_clock::now();
    local.n_samples = n_samples;
    ListSource src{site_begin, sites ? sites : reinterpret_cast<const uint32_t*>(site_begin), nullptr};
    const int rc = run(p, n_samples, src, chunk_samples, flags, out, out_capacity, file_begin, sink, user, &local);
    local.wall_s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    if (res) *res = local;
    return rc;
}

int v2p_pipeline_run_masks(v2p_pipeline* p, uint64_t n_records, uint64_t n_samples, uint32_t words_per_cell,
                           const uint32_t* masks, const uint64_t* csq_begin, const int32_t* csq_site, uint32_t mask_flags,
                           uint32_t chunk_samples, uint32_t flags, uint8_t* out, uint64_t out_capacity, uint64_t* file_begin,
                           v2p_file_sink sink, void* user, v2p_pipeline_result* res) {
    if (!p) return V2P_ERR_INVALID_ARG;
    p->err.clear();
    v2p_pipeline_result local;
    memset(&local, 0, sizeof local);
    const auto t0 = std::chrono::steady_clock::now();
    local.n_samples = n_samples;
    // the whole matrix is decoded once, by the last lane's catalogue object (the lists live in its md_* buffers, which no
    // generation touches); the chunks read them in place
    v2p_catalogue* dec = p->lanes[p->n_lanes - 1].cat;
    v2p_site_lists lists;
    int rc = v2p_sites_from_masks(dec, n_records, n_samples, words_per_cell, masks, csq_begin, csq_site, mask_flags, &lists);
    if (rc) {
        fail(p->err, rc, "mask decode failed: %s", v2p_catalogue_last_error(dec));
    } else {
        local.decode_ms = lists.decode_ms;
        if (!(mask_flags & V2P_FLAG_DEVICE_PTRS)) local.h2d_bytes += n_records * n_samples * words_per_cell * 4;
        std::vector<uint64_t> sb(2 * n_samples + 1);
        cudaError_t st = cudaSetDevice(p->device);
        if (st == cudaSuccess) st = cudaMemcpy(sb.data(), lists.site_begin, sb.size() * 8, cudaMemcpyDeviceToHost);
        if (st != cudaSuccess) {
            rc = fail(p->err, V2P_ERR_CUDA, "reading the decoded list bounds failed: %s", cudaGetErrorString(st));
        } else {
            ListSource src{sb.data(), nullptr, lists.sites};
            rc = run(p, n_samples, src, chunk_samples, flags, out, out_capacity, file_begin, sink, user, &local);
        }
    }
    local.wall_s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    if (res) *res = local;
    return rc;
}

// ---- directory writer (parts/io.rs:35-57, personalized_genome.rs:74-84) ----------------------------------------------
struct v2p_dir_writer {
    std::string dir, suffix, err;
    std::vector<std::string> names;
    unsigned threads = 4;
    std::atomic<uint64_t> bytes{0}, files{0};
    std::mutex mu;
};

int v2p_dir_writer_create(const char* out_dir, const char* const* proband_names, uint64_t n_probands, int compressed,
                          uint32_t threads, v2p_dir_writer** out) {
    if (!out) return V2P_ERR_INVALID_ARG;
    *out = nullptr;
    if (!out_dir || (n_probands && !proband_names)) return V2P_ERR_INVALID_ARG;
    v2p_dir_writer* w = new (std::nothrow) v2p_dir_writer();
    if (!w) return V2P_ERR_INVALID_ARG;
    w->dir = out_dir;
    w->suffix = compressed ? ".fasta.gz" : ".fasta";
    w->threads = std::max<uint32_t>(1, std::min<uint32_t>(threads ? threads : 4, 64));
    for (uint64_t i = 0; i < n_probands; ++i) {
        if (!proband_names[i]) {
            delete w;
            return V2P_ERR_INVALID_ARG;
        }
        w->names.emplace_back(proband_names[i]);
    }
    *out = w;
    return V2P_OK;
}

int v2p_dir_writer_sink(void* writer, uint64_t first_sample, uint64_t n_samples, const uint8_t* data, const uint64_t* file_begin) {
    v2p_dir_writer* w = static_cast<v2p_dir_writer*>(writer);
    if (!w || !file_begin || first_sample + n_samples > w->names.size()) {
        if (w) {
            std::lock_guard<std::mutex> g(w->mu);
            w->err = "chunk beyond the proband list";
        }
        return 1;
    }
    std::atomic<int> failed{0};
    auto work = [&](unsigned k, unsigned stride) {
        for (uint64_t i = k; i < n_samples && !failed.load(std::memory_order_relaxed); i += stride) {
            const std::string path = w->dir + "/" + w->names[first_sample + i] + w->suffix;
            const int fd = ::open(path.c_str(), O_CREAT | O_TRUNC | O_WRONLY, 0644);
            const uint8_t* ptr = data + file_begin[i];
            uint64_t left = file_begin[i + 1] - file_begin[i];
            bool ok = fd >= 0;
            while (ok && left) {
                const ssize_t n = ::write(fd, ptr, (size_t)std::min<uint64_t>(left, 1u << 30));
                if (n < 0 && errno == EINTR) continue;
                if (n <= 0) ok = false;
                else ptr += n, left -= (uint64_t)n;
            }
            if (fd >= 0 && ::close(fd) != 0) ok = false;
            if (!ok) {
                std::lock_guard<std::mutex> g(w->mu);
                w->err = "could not create/write " + path + ": " + std::strerror(errno);
                failed.store(1);
                return;
            }
            w->bytes += file_begin[i + 1] - file_begin[i];
            w->files += 1;
        }
    };
    const unsigned T = (unsigned)std::min<uint64_t>(w->threads, std::max<uint64_t>(n_samples, 1));
    std::vector<std::thread> pool;
    for (unsigned k = 1; k < T; ++k) pool.emplace_back(work, k, T);
    work(0, T);
    for (std::thread& t : pool) t.join();
    return failed.load();
}

uint64_t v2p_dir_writer_bytes(v2p_dir_writer* w) { return w ? w->bytes.load() : 0; }
uint64_t v2p_dir_writer_files(v2p_dir_writer* w) { return w ? w->files.load() : 0; }
const char* v2p_dir_writer_last_error(v2p_dir_writer* w) { return w ? w->err.c_str() : "writer is NULL"; }
void v2p_dir_writer_destroy(v2p_dir_writer* w) { delete w; }

}  // extern "C"
