// v2p_cohort.cu -- one process, every GPU of the box (include/v2p_cohort.h): the proband loop of parts/exec.rs:34-40
// and the per-proband writer of parts/io.rs:45-57, with one host thread + engine + pipeline per device and the samples
// split into contiguous ranges.  Sequencing over the public ABI of this library only; no kernels of its own.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "v2p_cohort.h"
#include "v2p_taskgen.h"

namespace {

struct Worker {
    int device = 0;
    v2p_engine* eng = nullptr;
    v2p_catalogue* lanes[V2P_PIPE_MAX_LANES] = {nullptr, nullptr, nullptr, nullptr};
    v2p_pipeline* pipe = nullptr;
};

}  // namespace

struct v2p_cohort {
    uint32_t n_dev = 0, n_lanes = 2;
    Worker w[V2P_COHORT_MAX_DEVICES];
    std::string err;
    std::mutex err_mu;
};

namespace {

int cofail(v2p_cohort* c, int code, const char* fmt, ...) {
    char buf[768];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) {
        std::lock_guard<std::mutex> g(c->err_mu);
        if (c->err.empty()) c->err = buf;  // the first failure is the one reported
    }
    return code;
}

int make_catalogue(int dev, const v2p_cohort_inputs* in, v2p_catalogue** out) {
    int rc = in->general
                 ? v2p_catalogue_create_ins(dev, in->n_tx, in->tx_offsets, in->n_sites, in->site_tx, in->ins_code, in->ins_flags,
                                            in->ins_pos_ref, in->ins_pos_res, in->ins_len, in->site_doff, in->site_dlen, in->pool,
                                            in->n_pool, out)
                 : v2p_catalogue_create(dev, in->n_tx, in->tx_offsets, in->n_sites, in->site_tx, in->site_pos, in->site_cls,
                                        in->site_rlen, in->site_doff, in->site_dlen, in->pool, in->n_pool, out);
    if (rc == V2P_OK) rc = v2p_catalogue_set_names(*out, in->name_off, in->names);
    return rc;
}

// Contiguous sample ranges with (nearly) equal numbers of variant sites: first[g] = first sample of worker g.
void split_by_sites(uint64_t n_samples, const uint64_t* site_begin, uint32_t n_dev, uint64_t* first) {
    const uint64_t total = site_begin[2 * n_samples];
    first[0] = 0;
    for (uint32_t g = 1; g < n_dev; ++g) {
        const uint64_t target = total / n_dev * g + total % n_dev * g / n_dev;
        // first sample s with site_begin[2 s] >= target (binary search over the even entries)
        uint64_t lo = first[g - 1], hi = n_samples;
        while (lo < hi) {
            const uint64_t mid = (lo + hi) / 2;
            if (site_begin[2 * mid] < target) lo = mid + 1;
            else hi = mid;
        }
        first[g] = lo;
    }
    first[n_dev] = n_samples;
    if (total == 0)  // nothing to weigh: equal counts
        for (uint32_t g = 1; g < n_dev; ++g) first[g] = n_samples * g / n_dev;
}

struct SinkShim {
    v2p_file_sink sink;
    void* user;
    uint64_t first;      // first sample of this worker's range
    std::mutex* serial;  // nullptr: the sink is thread-safe
    std::atomic<int>* stop;
};

int shim_sink(void* p, uint64_t first_sample, uint64_t n, const uint8_t* data, const uint64_t* file_begin) {
    SinkShim* s = (SinkShim*)p;
    if (s->stop->load(std::memory_order_relaxed)) return 1;  // another worker failed: stop after the chunk in flight
    if (!s->sink) return 0;
    if (s->serial) {
        std::lock_guard<std::mutex> g(*s->serial);
        return s->sink(s->user, s->first + first_sample, n, data, file_begin);
    }
    return s->sink(s->user, s->first + first_sample, n, data, file_begin);
}

void add(v2p_pipeline_result& t, const v2p_pipeline_result& r) {
    t.n_samples += r.n_samples, t.n_chunks += r.n_chunks, t.n_sites += r.n_sites, t.n_tasks += r.n_tasks;
    t.n_records += r.n_records, t.image_bytes += r.image_bytes, t.out_bytes += r.out_bytes, t.h2d_bytes += r.h2d_bytes;
    t.decode_ms += r.decode_ms, t.gen_ms += r.gen_ms, t.exec_ms += r.exec_ms, t.gzip_ms += r.gzip_ms;
    t.n_skipped += r.n_skipped, t.n_aborted += r.n_aborted;
    t.gen_wall_s += r.gen_wall_s, t.exec_wall_s += r.exec_wall_s, t.gzip_wall_s += r.gzip_wall_s;
    t.wait_wall_s += r.wait_wall_s, t.sink_wall_s += r.sink_wall_s;
}

}  // namespace

extern "C" {

int v2p_cohort_create(const int* devices, uint32_t n_devices, const v2p_cohort_inputs* in, uint32_t lanes_per_device,
                      v2p_cohort** out) {
    if (!out) return V2P_ERR_INVALID_ARG;
    *out = nullptr;
    if (!devices || !in || n_devices < 1 || n_devices > V2P_COHORT_MAX_DEVICES || lanes_per_device > V2P_PIPE_MAX_LANES)
        return V2P_ERR_INVALID_ARG;
    if (!in->tx_offsets || !in->name_off || (in->n_proteome && !in->proteome)) return V2P_ERR_INVALID_ARG;
    v2p_cohort* c = new (std::nothrow) v2p_cohort();
    if (!c) return V2P_ERR_INVALID_ARG;
    c->n_dev = n_devices;
    c->n_lanes = lanes_per_device ? lanes_per_device : 2;
    // the devices are set up in parallel: replicas of the proteome, catalogue uploads, streams (hundreds of ms each)
    std::vector<int> rcs(n_devices, V2P_OK);
    std::vector<std::thread> th;
    for (uint32_t g = 0; g < n_devices; ++g) {
        c->w[g].device = devices[g];
        th.emplace_back([c, g, in, &rcs] {
            Worker& w = c->w[g];
            int rc = v2p_engine_create(w.device, &w.eng);
            if (rc == V2P_OK) rc = v2p_engine_set_reference(w.eng, in->proteome, in->n_proteome, 0);
            for (uint32_t l = 0; rc == V2P_OK && l < c->n_lanes; ++l) rc = make_catalogue(w.device, in, &w.lanes[l]);
            if (rc == V2P_OK) rc = v2p_pipeline_create(w.eng, w.lanes, c->n_lanes, &w.pipe);
            rcs[g] = rc;
        });
    }
    for (auto& t : th) t.join();
    for (uint32_t g = 0; g < n_devices; ++g)
        if (rcs[g] != V2P_OK) {
            const int rc = rcs[g];
            v2p_cohort_destroy(c);
            return rc;
        }
    *out = c;
    return V2P_OK;
}

void v2p_cohort_destroy(v2p_cohort* c) {
    if (!c) return;
    for (uint32_t g = 0; g < c->n_dev; ++g) {
        Worker& w = c->w[g];
        if (w.pipe) v2p_pipeline_destroy(w.pipe);
        for (v2p_catalogue* l : w.lanes)
            if (l) v2p_catalogue_destroy(l);
        if (w.eng) v2p_engine_destroy(w.eng);
    }
    delete c;
}

const char* v2p_cohort_last_error(v2p_cohort* c) { return c ? c->err.c_str() : "cohort is NULL"; }

int v2p_cohort_enable_all_records(v2p_cohort* c, const v2p_cohort_inputs* in) {
    if (!c) return V2P_ERR_INVALID_ARG;
    {
        std::lock_guard<std::mutex> g(c->err_mu);
        c->err.clear();
    }
    if (!in || !in->tx_offsets || !in->name_off || (in->n_proteome && !in->proteome))
        return cofail(c, V2P_ERR_INVALID_ARG, "enable_all_records: proteome / tx_offsets / name_off missing");
    std::vector<int> rcs(c->n_dev, V2P_OK);
    std::vector<std::thread> th;
    for (uint32_t g = 0; g < c->n_dev; ++g)
        th.emplace_back([c, g, in, &rcs] {
            rcs[g] = v2p_pipeline_enable_all_records(c->w[g].pipe, in->proteome, in->n_proteome, in->n_tx, in->tx_offsets,
                                                     in->name_off, in->names);
        });
    for (auto& t : th) t.join();
    for (uint32_t g = 0; g < c->n_dev; ++g)
        if (rcs[g] != V2P_OK)
            return cofail(c, rcs[g], "device %d: %s", c->w[g].device, v2p_pipeline_last_error(c->w[g].pipe));
    return V2P_OK;
}

uint64_t v2p_cohort_launch_count(v2p_cohort* c) {
    uint64_t n = 0;
    if (c)
        for (uint32_t g = 0; g < c->n_dev; ++g) n += v2p_kernel_launch_count(c->w[g].eng);
    return n;
}

int v2p_cohort_run_lists(v2p_cohort* c, uint64_t n_samples, const uint64_t* site_begin, const uint32_t* sites,
                         uint32_t chunk_samples, uint32_t flags, v2p_file_sink sink, void* user, v2p_cohort_result* res) {
    if (!c) return V2P_ERR_INVALID_ARG;
    {
        std::lock_guard<std::mutex> g(c->err_mu);
        c->err.clear();
    }
    if (!site_begin || site_begin[0] != 0) return cofail(c, V2P_ERR_INVALID_ARG, "site_begin is NULL or does not start at 0");
    for (uint64_t h = 0; h < 2 * n_samples; ++h)
        if (site_begin[h + 1] < site_begin[h])
            return cofail(c, V2P_ERR_INVALID_ARG, "site_begin not monotone at haplotype %llu", (unsigned long long)h);
    if (site_begin[2 * n_samples] && !sites) return cofail(c, V2P_ERR_INVALID_ARG, "sites is NULL");
    v2p_cohort_result local;
    memset(&local, 0, sizeof local);
    local.n_devices = c->n_dev;
    split_by_sites(n_samples, site_begin, c->n_dev, local.first_sample);
    const auto t0 = std::chrono::steady_clock::now();
    std::mutex serial;
    std::atomic<int> stop{0};
    std::vector<int> rcs(c->n_dev, V2P_OK);
    std::vector<std::thread> th;
    for (uint32_t g = 0; g < c->n_dev; ++g) {
        th.emplace_back([&, g] {
            const uint64_t s0 = local.first_sample[g], ns = local.first_sample[g + 1] - s0;
            if (!ns) return;
            // this worker's slice of the lists, rebased to start at 0 (the pipeline wants site_begin[0] == 0)
            std::vector<uint64_t> sb(2 * ns + 1);
            const uint64_t base = site_begin[2 * s0];
            for (uint64_t h = 0; h <= 2 * ns; ++h) sb[h] = site_begin[2 * s0 + h] - base;
            SinkShim shim{sink, user, s0, (flags & V2P_COHORT_CONCURRENT_SINK) ? nullptr : &serial, &stop};
            const int rc = v2p_pipeline_run_lists(c->w[g].pipe, ns, sb.data(), sites ? sites + base : nullptr, chunk_samples,
                                                  flags & (V2P_PIPE_GZIP | V2P_PIPE_SKIP_ABORTS | V2P_PIPE_ALL_RECORDS),
                                                  nullptr, 0, nullptr, shim_sink,
                                                  &shim, &local.per_device[g]);
            if (rc != V2P_OK && !stop.exchange(1)) {
                rcs[g] = rc;
                cofail(c, rc, "device %d (samples %llu..%llu): %s", c->w[g].device, (unsigned long long)s0,
                       (unsigned long long)(s0 + ns), v2p_pipeline_last_error(c->w[g].pipe));
            }
        });
    }
    for (auto& t : th) t.join();
    for (uint32_t g = 0; g < c->n_dev; ++g) add(local.total, local.per_device[g]);
    local.total.wall_s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    if (res) *res = local;
    for (uint32_t g = 0; g < c->n_dev; ++g)
        if (rcs[g] != V2P_OK) return rcs[g];
    return V2P_OK;
}

int v2p_cohort_run_masks(v2p_cohort* c, uint64_t n_records, uint64_t n_samples, uint32_t words_per_cell, const uint32_t* masks,
                         const uint64_t* csq_begin, const int32_t* csq_site, uint32_t chunk_samples, uint32_t flags,
                         v2p_file_sink sink, void* user, v2p_cohort_result* res) {
    if (!c) return V2P_ERR_INVALID_ARG;
    {
        std::lock_guard<std::mutex> g(c->err_mu);
        c->err.clear();
    }
    Worker& w0 = c->w[0];
    if (cudaSetDevice(w0.device) != cudaSuccess) return cofail(c, V2P_ERR_CUDA, "cudaSetDevice(%d) failed", w0.device);
    v2p_site_lists lists;
    memset(&lists, 0, sizeof lists);
    const bool dev = flags & V2P_COHORT_DEVICE_MASKS;
    int rc = v2p_sites_from_masks(w0.lanes[0], n_records, n_samples, words_per_cell, masks, csq_begin, csq_site,
                                  dev ? V2P_FLAG_DEVICE_PTRS : 0u, &lists);
    if (rc != V2P_OK) return cofail(c, rc, "mask decode on device %d: %s", w0.device, v2p_catalogue_last_error(w0.lanes[0]));
    std::vector<uint64_t> sb(2 * n_samples + 1, 0);
    std::vector<uint32_t> sites(lists.n_sites);
    rc = v2p_device_read(sb.data(), lists.site_begin, sb.size() * sizeof(uint64_t));
    if (rc == V2P_OK && lists.n_sites) rc = v2p_device_read(sites.data(), lists.sites, sites.size() * sizeof(uint32_t));
    if (rc != V2P_OK) return cofail(c, rc, "reading the decoded lists back from device %d failed", w0.device);
    v2p_cohort_result local;
    memset(&local, 0, sizeof local);
    rc = v2p_cohort_run_lists(c, n_samples, sb.data(), sites.data(), chunk_samples, flags & ~V2P_COHORT_DEVICE_MASKS, sink, user, &local);
    local.total.decode_ms += lists.decode_ms, local.per_device[0].decode_ms += lists.decode_ms;
    const uint64_t up = dev ? 0 : n_records * n_samples * (uint64_t)words_per_cell * sizeof(uint32_t);
    local.total.h2d_bytes += up, local.per_device[0].h2d_bytes += up;
    if (res) *res = local;
    return rc;
}

}  // extern "C"
