// v2p_taskgen.cu -- device-side Task generation (include/v2p_taskgen.h): per-haplotype site lists -> packed batch.
//
// Bit-exact twin of the host producer vcf2prot_b200/cohort.py::build_batch (global proteome tape; packed or aligned
// layout), i.e. of the reference's emission rules for the seven synthetic-cohort classes
// (transcript_instructions.rs:452-780) and its concatenate/re-index loop (haplotype_instruction.rs:94-158):
//
//   classify   one thread per selected site: group (haplotype, transcript) membership, the "nothing after a
//              truncating variant" rule, how many tasks / result residues / alt bytes the site emits
//   scans      CUB exclusive sums turn those counts into task slots, result offsets, alt offsets, group ids
//   groups     per transcript-on-haplotype: result length, (aligned) slot; scan -> start on the result tape
//   emit       one thread per site writes its <= 3 tasks (base copy, mutation, follow-up copy) and its alt bytes
//
// Everything is integer work on HBM-resident arrays; no floating point, no host round trip except four 8-byte totals.
#include <cuda_runtime.h>

#include <cstring>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <new>
#include <string>

#include "v2p_hostres.cuh"
#include "v2p_mapped.cuh"
#include "v2p_taskgen.h"
#include "v2p_taskgen_rules.cuh"

using namespace v2p;

namespace {

struct Cat {  // device views
    const uint64_t* tx_off;
    const uint32_t *tx, *pos, *rlen, *dlen;
    const uint8_t* cls;
    const uint64_t* doff;
    const uint8_t* pool;
    const uint64_t* name_off;  // FASTA framing (V2P_GEN_FASTA): transcript names, name_off[n_tx+1] into `names`
    const uint8_t* names;
};

struct Sel {  // one generation
    uint64_t n_sel, n_hap;
    const uint32_t* sites;       // catalogue index of selected site j
    const uint64_t* site_begin;  // n_hap+1
    uint32_t* site_hap;          // haplotype of j
    uint64_t n_cat;              // catalogue sites (every list entry must be below it)
    unsigned long long* bad;     // min list position j whose entry is not a catalogue site or not ascending; ~0 = none
    uint8_t* flags;              // bit0 keep, bit1 newg, bit2 lastg, bit3 long payload
    uint64_t *cnt, *slen, *acon, *newg, *shortc, *slotl;              // scan inputs  (n_sel+1, last = 0)
    uint64_t *task_x, *l_x, *a_x, *g_x, *sh_x, *sl_x;                  // exclusive scans
    int aligned;
    int fasta;  // V2P_GEN_FASTA: `>{name}_{1|2}\n` / `\n` segments around every transcript (packed layout); shortc/sh_x then
                // carry the name-tape entry lengths (len(name)+5 per record) instead of the short-payload sizes
};

__device__ __forceinline__ bool is_trunc(uint8_t c) { return c == V2P_CLS_F || c == V2P_CLS_G || c == V2P_CLS_L || c == V2P_CLS_0; }

__global__ void k_tg_site_hap(Sel s) {
    uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (j >= s.n_sel) return;
    uint64_t lo = 0, hi = s.n_hap + 1;  // first h with site_begin[h] > j
    while (lo < hi) {
        uint64_t mid = (lo + hi) >> 1;
        if (s.site_begin[mid] <= j) lo = mid + 1; else hi = mid;
    }
    s.site_hap[j] = (uint32_t)(lo - 1);
    // the lists index the catalogue tables in every later kernel: reject what is not a site, and lists that are not
    // strictly ascending inside a haplotype (ascending in a (transcript, position)-sorted catalogue = grouped by transcript)
    const uint32_t si = s.sites[j];
    if (si >= s.n_cat || (j > s.site_begin[lo - 1] && s.sites[j - 1] >= si)) atomicMin(s.bad, (unsigned long long)j);
}

// what one kept site emits (transcript_instructions.rs:654-780 per class, :508-651 for the follow-up copy)
struct SiteTasks {
    bool has_base, has_mut, has_fol;
    uint64_t base_len, mut_len, fol_start, fol_len, acontrib;
};

__device__ __forceinline__ SiteTasks site_tasks(const Cat& c, uint32_t si, bool newg, bool lastg, uint64_t p_next) {
    SiteTasks o;
    const uint8_t cls = c.cls[si];
    const uint64_t p = c.pos[si], rlen = c.rlen[si], dlen = c.dlen[si];
    o.has_base = newg && cls != V2P_CLS_0;  // build_base_instruction :713-736 (start_lost: empty GIR :338-343)
    o.base_len = p;
    o.has_mut = cls == V2P_CLS_M || cls == V2P_CLS_I || cls == V2P_CLS_D || cls == V2P_CLS_F || cls == V2P_CLS_L;
    o.mut_len = (cls == V2P_CLS_M || cls == V2P_CLS_D) ? 1 : dlen;
    o.has_fol = cls == V2P_CLS_M || cls == V2P_CLS_I || cls == V2P_CLS_D;
    o.fol_start = cls == V2P_CLS_D ? p + rlen : p + 1;  // D: pos_ref + len + 1 with len = rlen - 1 (:514-548, :637-642)
    o.fol_len = p_next - o.fol_start;
    if (cls == V2P_CLS_D && !lastg && p + rlen - 1 == p_next) o.has_fol = false;  // phi rule of add_till_next_ins
    o.acontrib = cls == V2P_CLS_M ? 2 : dlen;  // missense pushes its residue twice (:659-660)
    return o;
}

__global__ void k_tg_classify(Sel s, Cat c) {
    uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (j >= s.n_sel) return;
    if (*s.bad != ~0ull) return;  // a bad list entry (k_tg_site_hap): the host reports it at its next hand-off
    const uint32_t h = s.site_hap[j];
    const uint64_t j0 = s.site_begin[h], j1 = s.site_begin[h + 1];
    const uint32_t si = s.sites[j];
    const uint32_t t = c.tx[si];
    // group start and truncating sites before me (groups are a handful of sites)
    uint64_t g0 = j;
    int truncs = 0;
    while (g0 > j0 && c.tx[s.sites[g0 - 1]] == t) {
        --g0;
        truncs += is_trunc(c.cls[s.sites[g0]]);
    }
    const bool keep = truncs == 0, newg = g0 == j;
    uint8_t fl = 0;
    uint64_t cnt = 0, slen = 0, acon = 0, shortc = 0;
    if (keep) {
        const bool next_in_group = j + 1 < j1 && c.tx[s.sites[j + 1]] == t;
        const bool lastg = !next_in_group || is_trunc(c.cls[si]);
        const uint64_t Lr = c.tx_off[t + 1] - c.tx_off[t];
        const uint64_t p_next = lastg ? Lr : c.pos[s.sites[j + 1]];
        const SiteTasks k = site_tasks(c, si, newg, lastg, p_next);
        cnt = (uint64_t)k.has_base + k.has_mut + k.has_fol;
        slen = (k.has_base ? k.base_len : 0) + (k.has_mut ? k.mut_len : 0) + (k.has_fol ? k.fol_len : 0);
        acon = k.acontrib;
        const bool is_long = s.aligned && k.has_mut && acon >= 32;
        shortc = is_long ? 0 : acon;
        if (s.fasta) {  // record framing (personalized_genome.rs:97,107): header before the first task, '\n' after the last
            const uint64_t nlen = c.name_off[t + 1] - c.name_off[t];
            cnt += (newg ? 1 : 0) + (lastg ? 1 : 0);
            slen += (newg ? nlen + 4 : 0) + (lastg ? 1 : 0);
            shortc = newg ? nlen + 5 : 0;
        }
        fl = 1u | (newg ? 2u : 0u) | (lastg ? 4u : 0u) | (is_long ? 8u : 0u);
    }
    s.flags[j] = fl;
    s.cnt[j] = cnt;
    s.slen[j] = slen;
    s.acon[j] = acon;
    s.newg[j] = (keep && newg) ? 1 : 0;
    s.shortc[j] = shortc;
}

struct Grp {
    uint64_t n_groups;
    uint64_t *g_first, *g_len, *g_slot, *g_slot_x;
    uint32_t *g_hap, *g_tx;
    uint64_t *ann_start, *ann_end;
};

__global__ void k_tg_groups(Sel s, Cat c, Grp g) {
    uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (j == 0) g.g_first[g.n_groups] = s.n_sel;
    if (j >= s.n_sel || !(s.flags[j] & 2u)) return;
    const uint64_t gi = s.g_x[j];
    g.g_first[gi] = j;
    g.g_hap[gi] = s.site_hap[j];
    g.g_tx[gi] = c.tx[s.sites[j]];
}

__global__ void k_tg_group_sizes(Sel s, Cat c, Grp g) {
    uint64_t gi = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (gi == 0) g.g_slot[g.n_groups] = 0;
    if (gi >= g.n_groups) return;
    const uint64_t len = s.l_x[g.g_first[gi + 1]] - s.l_x[g.g_first[gi]];
    const uint64_t c16 = c.tx_off[g.g_tx[gi]] & 15u;
    g.g_len[gi] = len;
    g.g_slot[gi] = s.aligned ? (len ? ((c16 + len + 15u) & ~uint64_t(15)) : 0) : len;
}

struct Out {
    v2p_task16* tasks;
    uint64_t *task_begin, *alt_base, *out_base;
    uint64_t *alt_per_hap, *short_tot;  // aligned alt layout
    uint64_t* mut_dst;                  // per site
    uint8_t* alt;
};

__global__ void k_tg_hap_bases(Sel s, Grp g, Out o) {
    uint64_t h = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (h > s.n_hap) return;
    const uint64_t j = s.site_begin[h];
    o.task_begin[h] = s.task_x[j];
    o.out_base[h] = g.g_slot_x[s.g_x[j]];
    if (!s.aligned) o.alt_base[h] = s.a_x[j] + (s.fasta ? s.sh_x[j] : 0);  // FASTA: + the name-tape entries before
}

__global__ void k_tg_emit_tasks(Sel s, Cat c, Grp g, Out o) {
    uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (j >= s.n_sel) return;
    const uint8_t fl = s.flags[j];
    s.slotl[j] = 0;
    if (!(fl & 1u)) return;
    const bool newg = fl & 2u, lastg = fl & 4u;
    const uint32_t h = s.site_hap[j], si = s.sites[j], t = c.tx[si];
    const uint64_t gi = newg ? s.g_x[j] : s.g_x[j] - 1;
    const uint64_t G0 = s.g_x[s.site_begin[h]];
    const uint64_t c16tx = c.tx_off[t] & 15u;
    const uint64_t g_start = g.g_slot_x[gi] - g.g_slot_x[G0] + ((s.aligned && g.g_len[gi]) ? c16tx : 0);
    // FASTA framing: this record's entry `>{name}_{1|2}\n\n` on the name tape behind the haplotype's alteration bytes
    const uint64_t nlen = s.fasta ? c.name_off[t + 1] - c.name_off[t] : 0;
    uint64_t name_src = 0;
    if (s.fasta) {
        const uint64_t j0 = s.site_begin[h], j1 = s.site_begin[h + 1];
        name_src = (s.a_x[j1] - s.a_x[j0]) + (s.sh_x[g.g_first[gi]] - s.sh_x[j0]);
    }
    if (newg) {
        g.ann_start[gi] = g_start + (s.fasta ? nlen + 4 : 0);
        g.ann_end[gi] = g_start + g.g_len[gi] - (s.fasta ? 1 : 0);
    }
    const uint64_t Lr = c.tx_off[t + 1] - c.tx_off[t];
    const uint64_t p_next = lastg ? Lr : c.pos[s.sites[j + 1]];
    const SiteTasks k = site_tasks(c, si, newg, lastg, p_next);
    uint64_t dst = g_start + (s.l_x[j] - s.l_x[g.g_first[gi]]);
    uint64_t slot = s.task_x[j];
    const uint64_t ref0 = c.tx_off[t];
    if (s.fasta && newg) {
        o.tasks[slot++] = v2p_task16{(uint32_t)name_src, (uint32_t)(nlen + 4), (uint32_t)dst, 1u};
        dst += nlen + 4;
    }
    if (k.has_base) {
        o.tasks[slot++] = v2p_task16{(uint32_t)ref0, (uint32_t)k.base_len, (uint32_t)dst, 0u};
        dst += k.base_len;
    }
    if (k.has_mut) {
        o.tasks[slot++] = v2p_task16{0u, (uint32_t)k.mut_len, (uint32_t)dst, 1u};  // src filled by k_tg_emit_alt
        o.mut_dst[j] = dst;
        if (fl & 8u) s.slotl[j] = ((dst & 15u) + k.acontrib + 15u) & ~uint64_t(15);
        dst += k.mut_len;
    }
    if (k.has_fol) {
        o.tasks[slot++] = v2p_task16{(uint32_t)(ref0 + k.fol_start), (uint32_t)k.fol_len, (uint32_t)dst, 0u};
        dst += k.fol_len;
    }
    if (s.fasta && lastg) o.tasks[slot] = v2p_task16{(uint32_t)(name_src + nlen + 4), 1u, (uint32_t)dst, 1u};
}

__global__ void k_tg_alt_sizes(Sel s, Out o) {  // aligned layout: [short payloads | pad to 16 | long slots] per haplotype
    uint64_t h = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (h > s.n_hap) return;
    if (h == s.n_hap) {
        o.alt_per_hap[h] = 0;
        return;
    }
    const uint64_t j0 = s.site_begin[h], j1 = s.site_begin[h + 1];
    const uint64_t st = s.sh_x[j1] - s.sh_x[j0];
    o.short_tot[h] = st;
    o.alt_per_hap[h] = ((st + 15u) & ~uint64_t(15)) + (s.sl_x[j1] - s.sl_x[j0]);
}

__global__ void k_tg_emit_alt(Sel s, Cat c, Out o) {
    uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (j >= s.n_sel) return;
    const uint8_t fl = s.flags[j];
    if (!(fl & 1u)) return;
    const uint64_t acon = s.acon[j];
    const uint32_t h = s.site_hap[j], si = s.sites[j];
    const uint64_t j0 = s.site_begin[h];
    if (s.fasta && (fl & 2u)) {  // the record's name-tape entry: '>' name '_' {1|2} '\n' '\n'
        const uint32_t t = c.tx[si];
        const uint64_t n0 = c.name_off[t], nlen = c.name_off[t + 1] - n0;
        uint8_t* d = o.alt + o.alt_base[h] + (s.a_x[s.site_begin[h + 1]] - s.a_x[j0]) + (s.sh_x[j] - s.sh_x[j0]);
        d[0] = '>';
        for (uint64_t w = 0; w < nlen; ++w) d[1 + w] = c.names[n0 + w];
        d[1 + nlen] = '_';
        d[2 + nlen] = (uint8_t)('1' + (h & 1u));
        d[3 + nlen] = '\n';
        d[4 + nlen] = '\n';
    }
    if (!acon) return;
    const uint8_t cls = c.cls[si];
    uint64_t a_new;
    if (!s.aligned) a_new = s.a_x[j] - s.a_x[j0];
    else if (fl & 8u) a_new = ((o.short_tot[h] + 15u) & ~uint64_t(15)) + (s.sl_x[j] - s.sl_x[j0]) + (o.mut_dst[j] & 15u);
    else a_new = s.sh_x[j] - s.sh_x[j0];
    // the mutation task is the site's first task, or its second when the site also emits the base copy
    const bool has_mut = cls == V2P_CLS_M || cls == V2P_CLS_I || cls == V2P_CLS_D || cls == V2P_CLS_F || cls == V2P_CLS_L;
    if (has_mut) {
        const bool has_base = (fl & 2u) && cls != V2P_CLS_0;
        const uint64_t slot = s.task_x[j] + (has_base ? 1 : 0) + ((s.fasta && (fl & 2u)) ? 1 : 0);
        o.tasks[slot].src_off = (uint32_t)(a_new + (cls == V2P_CLS_M ? 1 : 0));
    }
    uint8_t* dst = o.alt + o.alt_base[h] + a_new;
    const uint8_t* src = c.pool + c.doff[si];
    for (uint64_t w = 0; w < acon; ++w) dst[w] = src[cls == V2P_CLS_M ? 0 : w];
}


// ---------------------------------------------------------------------------------------------------------------------
// General catalogue (v2p_catalogue_create_ins): every instruction code, the reference's own outcomes.  One thread per
// transcript-on-haplotype runs csrc/v2p_taskgen_rules.cuh twice: a counting pass (sizes, task and alteration-byte counts,
// outcome), scans over the groups, then the emitting pass.
struct InsCat {
    const uint64_t* tx_off;
    const uint32_t* tx;
    const uint8_t *code, *flags;
    const uint32_t *pos_ref, *pos_res, *len, *dlen;
    const uint64_t* doff;
    const uint8_t* pool;
    const uint64_t* name_off;
    const uint8_t* names;
};

struct InsGen {
    uint64_t n_sel, n_hap, n_groups;
    const uint32_t* sites;
    const uint64_t* site_begin;
    const uint32_t* site_hap;
    uint64_t *newg, *g_x;  // per site (+ sentinel)
    const unsigned long long* bad_site;  // k_tg_site_hap's verdict on the lists (~0 = fine)
    // per group (+ sentinel)
    uint64_t *g_first, *g_size;
    uint32_t *g_hap, *g_tx, *g_nsites;
    uint8_t* g_status;
    uint64_t *c_tasks, *c_alt, *c_name, *c_adv, *c_tape, *c_rows, *c_skip;  // scan inputs
    uint64_t *x_tasks, *x_alt, *x_name, *x_adv, *x_tape, *x_rows, *x_skip;  // exclusive scans
    unsigned long long* err;  // [0] min group index the reference aborts on, [1] how many such groups
    int fasta, skip_aborts;
};

__global__ void k_ti_mark(InsGen g, InsCat c) {
    uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (j > g.n_sel) return;
    if (j == g.n_sel) {
        g.newg[j] = 0;
        return;
    }
    if (*g.bad_site != ~0ull) {
        g.newg[j] = 0;
        return;
    }
    const uint32_t h = g.site_hap[j];
    g.newg[j] = (j == g.site_begin[h] || c.tx[g.sites[j - 1]] != c.tx[g.sites[j]]) ? 1 : 0;
}

struct InsGet {
    const InsCat* c;
    const uint32_t* sites;
    uint64_t j0;
    __device__ __forceinline__ v2p_rules::TgIns operator()(int i) const {
        const uint32_t si = sites[j0 + i];
        v2p_rules::TgIns t;
        t.code = c->code[si], t.flags = c->flags[si];
        t.pos_ref = c->pos_ref[si], t.pos_res = c->pos_res[si], t.len = c->len[si], t.dlen = c->dlen[si];
        t.doff = c->doff[si];
        return t;
    }
};

__global__ void k_ti_count(InsGen g, InsCat c) {
    uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (j == 0) {  // sentinels of the per-group scans
        const uint64_t G = g.n_groups;
        g.c_tasks[G] = g.c_alt[G] = g.c_name[G] = g.c_adv[G] = g.c_tape[G] = g.c_rows[G] = g.c_skip[G] = 0;
        g.g_first[G] = g.n_sel;
    }
    if (j >= g.n_sel || !g.newg[j]) return;
    const uint64_t gi = g.g_x[j];
    const uint32_t h = g.site_hap[j], t = c.tx[g.sites[j]];
    const uint64_t j1 = g.site_begin[h + 1];
    uint64_t je = j + 1;
    while (je < j1 && c.tx[g.sites[je]] == t) ++je;
    const InsGet get{&c, g.sites, j};
    v2p_rules::NullSink null;
    v2p_rules::TgSummary s = v2p_rules::tg_transcript(get, (int)(je - j), c.tx_off[t + 1] - c.tx_off[t], null);
    if (s.status == v2p_rules::TG_PANIC) {
        atomicMin(g.err, (unsigned long long)gi);
        atomicAdd(g.err + 1, 1ull);
        if (g.skip_aborts) s = v2p_rules::TgSummary{v2p_rules::TG_ABSENT, 0, 0, 0};  // V2P_GEN_SKIP_ABORTS
    }
    const bool row = s.status == v2p_rules::TG_OK || s.status == v2p_rules::TG_EMPTY;
    const uint64_t adv = s.status == v2p_rules::TG_OK ? s.size : 0;
    const uint64_t nlen = g.fasta ? c.name_off[t + 1] - c.name_off[t] : 0;
    g.g_first[gi] = j, g.g_nsites[gi] = (uint32_t)(je - j), g.g_hap[gi] = h, g.g_tx[gi] = t;
    g.g_status[gi] = (uint8_t)s.status, g.g_size[gi] = s.size;
    g.c_tasks[gi] = s.n_tasks + ((g.fasta && row) ? 2 : 0);
    g.c_alt[gi] = s.n_alt;
    g.c_name[gi] = (g.fasta && row) ? nlen + 5 : 0;
    g.c_rows[gi] = row ? 1 : 0;
    g.c_skip[gi] = s.status == v2p_rules::TG_SKIPPED ? 1 : 0;
    if (g.fasta) {  // a file image holds records only: header + sequence + newline per annotation row
        g.c_adv[gi] = g.c_tape[gi] = row ? nlen + 4 + adv + 1 : 0;
    } else {  // the tape was sized from every instruction set before any transcript could fail (haplotype_instruction.rs:78)
        g.c_adv[gi] = adv;
        g.c_tape[gi] = s.status == v2p_rules::TG_ABSENT ? 0 : s.size;
    }
}

struct InsOut {
    v2p_task16* tasks;
    uint64_t *task_begin, *alt_base, *out_base;
    uint8_t* alt;
    uint32_t *ann_hap, *ann_tx;
    uint64_t *ann_start, *ann_end;
};

__global__ void k_ti_hap_bases(InsGen g, InsOut o) {
    uint64_t h = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (h > g.n_hap) return;
    const uint64_t G0 = g.g_x[g.site_begin[h]];
    o.task_begin[h] = g.x_tasks[G0];
    o.alt_base[h] = g.x_alt[G0] + g.x_name[G0];
    o.out_base[h] = g.x_tape[G0];
}

struct EmitSink {  // the rules' sink: writes tasks and alteration bytes in place
    v2p_task16* tasks;     // next task slot
    uint8_t* alt_bytes;    // next alteration byte of this transcript
    const uint8_t* pool;
    uint64_t ref0, alt0, dst0;  // proteome offset of the transcript; haplotype-relative offsets of its alt bytes / result
    __device__ __forceinline__ void task(uint32_t stream, uint64_t src, uint64_t len, uint64_t dst) {
        *tasks++ = v2p_task16{(uint32_t)((stream ? alt0 : ref0) + src), (uint32_t)len, (uint32_t)(dst0 + dst), stream};
    }
    __device__ __forceinline__ void alt(uint64_t doff, uint32_t dlen) {
        for (uint32_t w = 0; w < dlen; ++w) alt_bytes[w] = pool[doff + w];
        alt_bytes += dlen;
    }
};

__global__ void k_ti_emit(InsGen g, InsCat c, InsOut o) {
    uint64_t gi = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (gi >= g.n_groups) return;
    const int status = g.g_status[gi];
    if (status != v2p_rules::TG_OK && status != v2p_rules::TG_EMPTY) return;
    const uint32_t h = g.g_hap[gi], t = g.g_tx[gi];
    const uint64_t G0 = g.g_x[g.site_begin[h]], G1 = g.g_x[g.site_begin[h + 1]];
    const uint64_t g_start = g.x_adv[gi] - g.x_adv[G0];
    const uint64_t size = status == v2p_rules::TG_OK ? g.g_size[gi] : 0;
    const uint64_t nlen = g.fasta ? c.name_off[t + 1] - c.name_off[t] : 0, hdr = g.fasta ? nlen + 4 : 0;
    const uint64_t row = g.x_rows[gi];
    o.ann_hap[row] = h, o.ann_tx[row] = t;
    o.ann_start[row] = g_start + hdr, o.ann_end[row] = g_start + hdr + size;
    v2p_task16* tk = o.tasks + g.x_tasks[gi];
    const uint64_t alt_local = g.x_alt[gi] - g.x_alt[G0];
    if (g.fasta) {  // `>{name}_{1|2}\n` before, `\n` after, both read from the name tape behind the alteration bytes
        const uint64_t name_src = (g.x_alt[G1] - g.x_alt[G0]) + (g.x_name[gi] - g.x_name[G0]);
        *tk++ = v2p_task16{(uint32_t)name_src, (uint32_t)hdr, (uint32_t)g_start, 1u};
        o.tasks[g.x_tasks[gi + 1] - 1] = v2p_task16{(uint32_t)(name_src + hdr), 1u, (uint32_t)(g_start + hdr + size), 1u};
        uint8_t* d = o.alt + o.alt_base[h] + name_src;
        const uint64_t n0 = c.name_off[t];
        d[0] = '>';
        for (uint64_t w = 0; w < nlen; ++w) d[1 + w] = c.names[n0 + w];
        d[1 + nlen] = '_';
        d[2 + nlen] = (uint8_t)('1' + (h & 1u));
        d[3 + nlen] = '\n';
        d[4 + nlen] = '\n';
    }
    if (status != v2p_rules::TG_OK) return;
    EmitSink sink{tk, o.alt + o.alt_base[h] + alt_local, c.pool, c.tx_off[t], alt_local, g_start + hdr};
    const InsGet get{&c, g.sites, g.g_first[gi]};
    v2p_rules::tg_transcript(get, (int)g.g_nsites[gi], c.tx_off[t + 1] - c.tx_off[t], sink);
}

// ---------------------------------------------------------------------------------------------------------------------
// Genotype bit-masks -> per-haplotype site lists (MaskDecoder.rs:95-153 + the transpose of vcf_ds.rs:126-295).
// The mask matrix is streamed twice (population count to size the key buffer, then the emit); everything after that
// works on the set bits only: 64-bit keys (haplotype << site_bits | site), one radix sort over the significant bits,
// duplicate drop, and a binary search per haplotype for the CSR offsets.
struct MdCtr {
    unsigned long long n_bits, cursor, bad_record, n_unique;
};

__device__ __forceinline__ uint4 md_load4(const uint32_t* m, uint64_t j, uint64_t n_words) {
    if (j + 4 <= n_words) return __ldcs(reinterpret_cast<const uint4*>(m + j));
    uint4 v = make_uint4(0, 0, 0, 0);
    if (j < n_words) v.x = m[j];
    if (j + 1 < n_words) v.y = m[j + 1];
    if (j + 2 < n_words) v.z = m[j + 2];
    return v;
}

__global__ void __launch_bounds__(256) k_md_count(const uint32_t* __restrict__ masks, uint64_t n_words, MdCtr* ctr) {
    unsigned long long n = 0;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x * 4;
    for (uint64_t j = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; j < n_words; j += stride) {
        const uint4 v = md_load4(masks, j, n_words);
        n += __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
    }
    n = __reduce_add_sync(0xffffffffu, (unsigned)n);  // <= 32 lanes * a few thousand words * 32 bits: fits 32 bits
    if ((threadIdx.x & 31) == 0 && n) atomicAdd(&ctr->n_bits, n);
}

struct MdArgs {
    const uint32_t* masks;
    uint64_t n_words, n_samples;
    uint32_t W, site_bits;
    const uint64_t* csq_begin;
    const int32_t* csq_site;
    uint64_t* keys;
    MdCtr* ctr;
};

// one word of one cell: set bit b -> csq 15*w + (b >> 1) of the record, haplotype 2*sample + (b & 1)
__device__ __forceinline__ unsigned md_word(const MdArgs& a, uint32_t word, uint64_t j, uint64_t* dst, bool write) {
    if (!word) return 0;
    const uint64_t cell = j / a.W;
    const uint32_t w = (uint32_t)(j - cell * a.W);
    const uint64_t r = cell / a.n_samples, smp = cell - r * a.n_samples;
    const uint64_t c0 = a.csq_begin[r], nc = a.csq_begin[r + 1] - c0;
    unsigned n = 0;
    while (word) {
        const int b = __ffs(word) - 1;
        word &= word - 1;
        const uint64_t k = 15ull * w + (b >> 1);
        if (k >= nc) {
            atomicMin(&a.ctr->bad_record, (unsigned long long)r);
            continue;
        }
        const int32_t site = a.csq_site[c0 + k];
        if (site < 0) continue;  // a consequence class the tool does not support: dropped, vcf_ds.rs:249,262
        if (write) dst[n] = ((2 * smp + (b & 1)) << a.site_bits) | (uint32_t)site;
        ++n;
    }
    return n;
}

__global__ void __launch_bounds__(256) k_md_emit(MdArgs a) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x * 4;
    const unsigned lane = threadIdx.x & 31;
    // uniform trip count so the warp-wide scan below is always converged
    const uint64_t first = (uint64_t)blockIdx.x * blockDim.x * 4;
    for (uint64_t base = first; base < a.n_words; base += stride) {
        const uint64_t j = base + (uint64_t)threadIdx.x * 4;
        const uint4 v = md_load4(a.masks, j, a.n_words);
        const bool any = (v.x | v.y | v.z | v.w) != 0;
        if (!__any_sync(0xffffffffu, any)) continue;
        unsigned n = 0;
        if (any)
            n = md_word(a, v.x, j, nullptr, false) + md_word(a, v.y, j + 1, nullptr, false) +
                md_word(a, v.z, j + 2, nullptr, false) + md_word(a, v.w, j + 3, nullptr, false);
        unsigned incl = n;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= (unsigned)d) incl += t;
        }
        const unsigned tot = __shfl_sync(0xffffffffu, incl, 31);
        if (!tot) continue;
        unsigned long long wb = 0;
        if (lane == 31) wb = atomicAdd(&a.ctr->cursor, (unsigned long long)tot);
        wb = __shfl_sync(0xffffffffu, wb, 31);
        if (n) {
            uint64_t* dst = a.keys + wb + (incl - n);
            dst += md_word(a, v.x, j, dst, true);
            dst += md_word(a, v.y, j + 1, dst, true);
            dst += md_word(a, v.z, j + 2, dst, true);
            md_word(a, v.w, j + 3, dst, true);
        }
    }
}

__global__ void __launch_bounds__(256) k_md_csr(const uint64_t* __restrict__ keys, const MdCtr* ctr, uint64_t n_hap,
                                                uint32_t site_bits, uint64_t* site_begin, uint32_t* sites) {
    const uint64_t n = ctr->n_unique;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) sites[i] = (uint32_t)(keys[i] & ((1ull << site_bits) - 1));
    if (i <= n_hap) {  // first key of haplotype >= i
        const uint64_t want = i << site_bits;
        uint64_t lo = 0, hi = n;
        while (lo < hi) {
            const uint64_t mid = (lo + hi) >> 1;
            if (keys[mid] < want) lo = mid + 1;
            else hi = mid;
        }
        site_begin[i] = lo;
    }
}

}  // namespace

struct v2p_catalogue {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string err;
    uint64_t n_tx = 0, n_sites = 0;
    DevBuf tx_off, tx, pos, rlen, dlen, cls, doff, pool;
    bool is_ins = false;  // created by v2p_catalogue_create_ins (general rules) rather than the seven-class tables
    DevBuf i_code, i_flags, i_pos_ref, i_pos_res, i_len;  // (+ tx, doff, dlen, pool shared with the class tables)
    DevBuf gi_newg, gi_gx, gi_first, gi_size, gi_hap, gi_tx, gi_nsites, gi_status, gi_c[7], gi_x[7], gi_err;
    v2p::MappedBuf pub;   // totals come back through mapped pinned memory, not the copy engine (v2p_mapped.cuh)
    DevBuf name_off, names;  // v2p_catalogue_set_names
    bool has_names = false;
    // per-generation buffers
    DevBuf sites, site_begin, site_hap, flags, scan_in[6], scan_out[6], cub_tmp, totals, sel_err;
    DevBuf g_first, g_len, g_slot, g_slot_x, g_hap, g_tx, ann_start, ann_end;
    DevBuf tasks, task_begin, alt_base, out_base, alt_per_hap, short_tot, mut_dst, alt, out;
    // mask decode (v2p_sites_from_masks)
    DevBuf md_masks, md_csq_begin, md_csq_site, md_keys[2], md_uniq, md_begin, md_sites, md_ctr;
};

namespace {

int generate_on_device(v2p_catalogue* c, uint64_t n_hap, uint64_t n_sel, const uint64_t* d_site_begin, const uint32_t* d_sites,
                       uint32_t flags, v2p_generated* out);
int generate_ins_on_device(v2p_catalogue* c, uint64_t n_hap, uint64_t n_sel, const uint64_t* d_site_begin,
                           const uint32_t* d_sites, uint32_t flags, v2p_generated* out);

}  // namespace

extern "C" {

int v2p_catalogue_create(int cuda_device, uint64_t n_tx, const uint64_t* tx_offsets, uint64_t n_sites,
                         const uint32_t* site_tx, const uint32_t* site_pos, const uint8_t* site_cls,
                         const uint32_t* site_rlen, const uint64_t* site_doff, const uint32_t* site_dlen,
                         const uint8_t* pool, uint64_t n_pool, v2p_catalogue** out) {
    if (!out || !tx_offsets || (n_sites && (!site_tx || !site_pos || !site_cls || !site_rlen || !site_doff || !site_dlen)))
        return V2P_ERR_INVALID_ARG;
    *out = nullptr;
    for (uint64_t i = 0; i < n_sites; ++i)  // the kernels index tx_offsets[] and pool[] with these
        if (site_tx[i] >= n_tx || site_cls[i] > V2P_CLS_0 || site_doff[i] + site_dlen[i] > n_pool ||
            (i && (site_tx[i] < site_tx[i - 1] || (site_tx[i] == site_tx[i - 1] && site_pos[i] < site_pos[i - 1]))))
            return V2P_ERR_INVALID_ARG;
    v2p_catalogue* c = new (std::nothrow) v2p_catalogue();
    if (!c) return V2P_ERR_INVALID_ARG;
    c->device = cuda_device;
    c->n_tx = n_tx, c->n_sites = n_sites;
    cudaStream_t& st = c->stream;
    if (cudaSetDevice(cuda_device) || cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) || cudaEventCreate(&c->ev0) ||
        cudaEventCreate(&c->ev1) || upload(c->tx_off, tx_offsets, (n_tx + 1) * 8, st) || upload(c->tx, site_tx, n_sites * 4, st) ||
        upload(c->pos, site_pos, n_sites * 4, st) || upload(c->cls, site_cls, n_sites, st) ||
        upload(c->rlen, site_rlen, n_sites * 4, st) || upload(c->doff, site_doff, n_sites * 8, st) ||
        upload(c->dlen, site_dlen, n_sites * 4, st) || upload(c->pool, pool, n_pool, st) || cudaStreamSynchronize(st)) {
        v2p_catalogue_destroy(c);
        return V2P_ERR_CUDA;
    }
    *out = c;
    return V2P_OK;
}

int v2p_catalogue_create_ins(int cuda_device, uint64_t n_tx, const uint64_t* tx_offsets, uint64_t n_sites,
                             const uint32_t* site_tx, const uint8_t* ins_code, const uint8_t* ins_flags,
                             const uint32_t* ins_pos_ref, const uint32_t* ins_pos_res, const uint32_t* ins_len,
                             const uint64_t* ins_doff, const uint32_t* ins_dlen, const uint8_t* pool, uint64_t n_pool,
                             v2p_catalogue** out) {
    if (!out || !tx_offsets ||
        (n_sites && (!site_tx || !ins_code || !ins_flags || !ins_pos_ref || !ins_pos_res || !ins_len || !ins_doff || !ins_dlen)))
        return V2P_ERR_INVALID_ARG;
    *out = nullptr;
    for (uint64_t i = 0; i < n_sites; ++i)
        if (site_tx[i] >= n_tx || ins_doff[i] + ins_dlen[i] > n_pool || (i && site_tx[i] < site_tx[i - 1])) return V2P_ERR_INVALID_ARG;
    v2p_catalogue* c = new (std::nothrow) v2p_catalogue();
    if (!c) return V2P_ERR_INVALID_ARG;
    c->device = cuda_device;
    c->is_ins = true;
    c->n_tx = n_tx, c->n_sites = n_sites;
    cudaStream_t& st = c->stream;
    if (cudaSetDevice(cuda_device) || cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) || cudaEventCreate(&c->ev0) ||
        cudaEventCreate(&c->ev1) || upload(c->tx_off, tx_offsets, (n_tx + 1) * 8, st) || upload(c->tx, site_tx, n_sites * 4, st) ||
        upload(c->i_code, ins_code, n_sites, st) || upload(c->i_flags, ins_flags, n_sites, st) ||
        upload(c->i_pos_ref, ins_pos_ref, n_sites * 4, st) || upload(c->i_pos_res, ins_pos_res, n_sites * 4, st) ||
        upload(c->i_len, ins_len, n_sites * 4, st) || upload(c->doff, ins_doff, n_sites * 8, st) ||
        upload(c->dlen, ins_dlen, n_sites * 4, st) || upload(c->pool, pool, n_pool, st) || cudaStreamSynchronize(st)) {
        v2p_catalogue_destroy(c);
        return V2P_ERR_CUDA;
    }
    *out = c;
    return V2P_OK;
}

void v2p_catalogue_destroy(v2p_catalogue* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;  // frees every buffer
}

const char* v2p_catalogue_last_error(v2p_catalogue* c) { return c ? c->err.c_str() : "catalogue is NULL"; }

int v2p_catalogue_set_names(v2p_catalogue* c, const uint64_t* name_off, const uint8_t* names) {
    if (!c || !name_off) return V2P_ERR_INVALID_ARG;
    c->err.clear();
    c->has_names = false;
    if (name_off[0] != 0) return fail(c->err, V2P_ERR_INVALID_ARG, "name_off[0] must be 0");
    for (uint64_t t = 0; t < c->n_tx; ++t)
        if (name_off[t + 1] < name_off[t]) return fail(c->err, V2P_ERR_INVALID_ARG, "name_off not monotone");
    if (name_off[c->n_tx] && !names) return fail(c->err, V2P_ERR_INVALID_ARG, "names is NULL");
    CU(c->err, cudaSetDevice(c->device));
    CU(c->err, upload(c->name_off, name_off, (c->n_tx + 1) * 8, c->stream));
    CU(c->err, upload(c->names, names, name_off[c->n_tx], c->stream));
    CU(c->err, cudaStreamSynchronize(c->stream));
    c->has_names = true;
    return V2P_OK;
}

int v2p_device_read(void* host_dst, const void* dev_src, size_t bytes) {
    if (!bytes) return V2P_OK;
    return cudaMemcpy(host_dst, dev_src, bytes, cudaMemcpyDeviceToHost) == cudaSuccess ? V2P_OK : V2P_ERR_CUDA;
}

int v2p_generate_tasks(v2p_catalogue* c, uint64_t n_hap, const uint64_t* site_begin, const uint32_t* sites, uint32_t flags,
                       v2p_generated* out) {
    if (!c || !out || !site_begin || site_begin[0] != 0) return V2P_ERR_INVALID_ARG;
    memset(out, 0, sizeof *out);
    c->err.clear();
    CU(c->err, cudaSetDevice(c->device));
    const uint64_t n_sel = site_begin[n_hap];
    if (n_sel && !sites) return fail(c->err, V2P_ERR_INVALID_ARG, "sites is NULL");
    for (uint64_t h = 0; h < n_hap; ++h)
        if (site_begin[h + 1] < site_begin[h]) return fail(c->err, V2P_ERR_INVALID_ARG, "site_begin not monotone");
    CU(c->err, cudaEventRecord(c->ev0, c->stream));
    CU(c->err, upload(c->sites, sites, n_sel * 4, c->stream));
    CU(c->err, upload(c->site_begin, site_begin, (n_hap + 1) * 8, c->stream));
    return generate_on_device(c, n_hap, n_sel, (const uint64_t*)c->site_begin.p, (const uint32_t*)c->sites.p, flags, out);
}

int v2p_sites_from_masks(v2p_catalogue* c, uint64_t n_records, uint64_t n_samples, uint32_t words_per_cell,
                         const uint32_t* masks, const uint64_t* csq_begin, const int32_t* csq_site, uint32_t flags,
                         v2p_site_lists* out) {
    if (!c || !out || !csq_begin || !words_per_cell || csq_begin[0] != 0) return V2P_ERR_INVALID_ARG;
    memset(out, 0, sizeof *out);
    c->err.clear();
    const uint64_t n_words = n_records * n_samples * words_per_cell, n_hap = 2 * n_samples, n_csq = csq_begin[n_records];
    if ((n_words && !masks) || (n_csq && !csq_site)) return fail(c->err, V2P_ERR_INVALID_ARG, "masks / csq_site is NULL");
    if (n_hap >> 31) return fail(c->err, V2P_ERR_INVALID_ARG, "more than 2^30 samples");
    for (uint64_t r = 0; r < n_records; ++r)
        if (csq_begin[r + 1] < csq_begin[r]) return fail(c->err, V2P_ERR_INVALID_ARG, "csq_begin not monotone");
    for (uint64_t k = 0; k < n_csq; ++k)
        if (csq_site[k] >= 0 && (uint64_t)csq_site[k] >= c->n_sites)
            return fail(c->err, V2P_ERR_INVALID_ARG, "csq_site[%llu] = %d is not a catalogue site", (unsigned long long)k, csq_site[k]);
    CU(c->err, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    CU(c->err, cudaEventRecord(c->ev0, st));
    const uint32_t* d_masks = masks;
    if (!(flags & V2P_FLAG_DEVICE_PTRS)) {
        CU(c->err, upload(c->md_masks, masks, n_words * 4, st));
        d_masks = (const uint32_t*)c->md_masks.p;
    } else if ((uintptr_t)masks & 15) {
        return fail(c->err, V2P_ERR_INVALID_ARG, "device mask matrix must be 16-byte aligned");
    }
    CU(c->err, upload(c->md_csq_begin, csq_begin, (n_records + 1) * 8, st));
    CU(c->err, upload(c->md_csq_site, csq_site, n_csq * 4, st));
    CU(c->err, c->md_ctr.need(sizeof(MdCtr)));
    CU(c->err, c->md_begin.need((n_hap + 1) * 8));
    MdCtr* ctr = (MdCtr*)c->md_ctr.p;
    MdCtr h{0, 0, ~0ull, 0};
    CU(c->err, cudaMemcpyAsync(ctr, &h, sizeof h, cudaMemcpyHostToDevice, st));
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device);
    const unsigned grid = (unsigned)std::min<uint64_t>((n_words + 1023) / 1024 + 1, (uint64_t)sms * 16);
    if (n_words) k_md_count<<<grid, 256, 0, st>>>(d_masks, n_words, ctr);
    static_assert(sizeof(MdCtr) == 32, "MdCtr is published as four 8-byte words");
    CU(c->err, c->pub.reserve(64));
    auto fetch_ctr = [&]() -> cudaError_t {  // counters -> mapped pinned memory -> h
        cudaError_t e1 = v2p::publish_words(c->pub.p, ctr, 4, st);
        if (e1 != cudaSuccess) return e1;
        e1 = cudaStreamSynchronize(st);
        memcpy(&h, c->pub.p, sizeof h);
        return e1;
    };
    CU(c->err, fetch_ctr());
    const uint64_t cap = h.n_bits;  // upper bound of the keys: every set bit
    uint32_t site_bits = 1, hap_bits = 1;
    while ((1ull << site_bits) < c->n_sites) ++site_bits;
    while ((1ull << hap_bits) < n_hap + 1) ++hap_bits;
    CU(c->err, c->md_keys[0].need(cap * 8 + 16));
    CU(c->err, c->md_keys[1].need(cap * 8 + 16));
    CU(c->err, c->md_uniq.need(cap * 8 + 16));
    CU(c->err, c->md_sites.need(cap * 4 + 16));
    uint64_t n_unique = 0;
    if (cap) {
        MdArgs a{d_masks, n_words, n_samples, words_per_cell, site_bits, (const uint64_t*)c->md_csq_begin.p,
                 (const int32_t*)c->md_csq_site.p, (uint64_t*)c->md_keys[0].p, ctr};
        k_md_emit<<<grid, 256, 0, st>>>(a);
        CU(c->err, fetch_ctr());
        if (h.bad_record != ~0ull)
            return fail(c->err, V2P_ERR_SRC_OOB, "record %llu: a mask bit selects a consequence beyond the record's %llu (vcf_ds.rs:287)",
                        h.bad_record, (unsigned long long)(csq_begin[h.bad_record + 1] - csq_begin[h.bad_record]));
        const uint64_t n_keys = h.cursor;
        if (n_keys) {
            cub::DoubleBuffer<uint64_t> db((uint64_t*)c->md_keys[0].p, (uint64_t*)c->md_keys[1].p);
            size_t tmp = 0;
            CU(c->err, cub::DeviceRadixSort::SortKeys(nullptr, tmp, db, (int64_t)n_keys, 0, (int)(site_bits + hap_bits), st));
            CU(c->err, c->cub_tmp.need(tmp));
            CU(c->err, cub::DeviceRadixSort::SortKeys(c->cub_tmp.p, tmp, db, (int64_t)n_keys, 0, (int)(site_bits + hap_bits), st));
            CU(c->err, cub::DeviceSelect::Unique(nullptr, tmp, db.Current(), (uint64_t*)c->md_uniq.p, &ctr->n_unique, (int64_t)n_keys, st));
            CU(c->err, c->cub_tmp.need(tmp));
            CU(c->err, cub::DeviceSelect::Unique(c->cub_tmp.p, tmp, db.Current(), (uint64_t*)c->md_uniq.p, &ctr->n_unique, (int64_t)n_keys, st));
            CU(c->err, fetch_ctr());
            n_unique = h.n_unique;
        }
    }
    k_md_csr<<<blocks(std::max<uint64_t>(n_unique, n_hap + 1)), 256, 0, st>>>((const uint64_t*)c->md_uniq.p, ctr, n_hap, site_bits,
                                                                             (uint64_t*)c->md_begin.p, (uint32_t*)c->md_sites.p);
    CU(c->err, cudaGetLastError());
    CU(c->err, cudaEventRecord(c->ev1, st));
    CU(c->err, cudaStreamSynchronize(st));
    float ms = 0;
    CU(c->err, cudaEventElapsedTime(&ms, c->ev0, c->ev1));
    out->n_hap = n_hap, out->n_sites = n_unique;
    out->site_begin = (const uint64_t*)c->md_begin.p, out->sites = (const uint32_t*)c->md_sites.p;
    out->decode_ms = ms;
    return V2P_OK;
}

int v2p_generate_tasks_from_lists(v2p_catalogue* c, const v2p_site_lists* lists, uint32_t flags, v2p_generated* out) {
    if (!c || !out || !lists || (lists->n_hap && !lists->site_begin)) return V2P_ERR_INVALID_ARG;
    memset(out, 0, sizeof *out);
    c->err.clear();
    CU(c->err, cudaSetDevice(c->device));
    CU(c->err, cudaEventRecord(c->ev0, c->stream));
    return generate_on_device(c, lists->n_hap, lists->n_sites, lists->site_begin, lists->sites, flags, out);
}

}  // extern "C"

namespace {

// site_begin / sites are device pointers here; c->ev0 has been recorded by the caller
int generate_on_device(v2p_catalogue* c, uint64_t n_hap, uint64_t n_sel, const uint64_t* d_site_begin, const uint32_t* d_sites,
                       uint32_t flags, v2p_generated* out) {
    if (c->is_ins) return generate_ins_on_device(c, n_hap, n_sel, d_site_begin, d_sites, flags, out);
    cudaStream_t st = c->stream;
    int rc;
    CU(c->err, c->site_hap.need(n_sel * 4 + 16));
    CU(c->err, c->flags.need(n_sel + 16));
    CU(c->err, c->mut_dst.need(n_sel * 8 + 16));
    CU(c->err, c->totals.need(64));
    CU(c->err, c->sel_err.need(16));
    for (int i = 0; i < 6; ++i) {
        CU(c->err, c->scan_in[i].need((n_sel + 1) * 8));
        CU(c->err, c->scan_out[i].need((n_sel + 1) * 8));
    }
    const bool fasta = (flags & V2P_GEN_FASTA) != 0;
    if (fasta && (flags & V2P_GEN_ALIGNED))
        return fail(c->err, V2P_ERR_INVALID_ARG, "V2P_GEN_FASTA needs the packed layout (a file image cannot contain pad bytes)");
    if (fasta && !c->has_names) return fail(c->err, V2P_ERR_INVALID_ARG, "V2P_GEN_FASTA needs v2p_catalogue_set_names first");
    Cat cat{(const uint64_t*)c->tx_off.p, (const uint32_t*)c->tx.p, (const uint32_t*)c->pos.p, (const uint32_t*)c->rlen.p,
            (const uint32_t*)c->dlen.p, (const uint8_t*)c->cls.p, (const uint64_t*)c->doff.p, (const uint8_t*)c->pool.p,
            (const uint64_t*)c->name_off.p, (const uint8_t*)c->names.p};
    Sel s{};
    s.n_sel = n_sel, s.n_hap = n_hap;
    s.sites = d_sites, s.site_begin = d_site_begin;
    s.site_hap = (uint32_t*)c->site_hap.p, s.flags = (uint8_t*)c->flags.p;
    s.n_cat = c->n_sites, s.bad = (unsigned long long*)c->sel_err.p;
    CU(c->err, cudaMemsetAsync(s.bad, 0xFF, 8, st));
    uint64_t** ins[6] = {&s.cnt, &s.slen, &s.acon, &s.newg, &s.shortc, &s.slotl};
    uint64_t** outs[6] = {&s.task_x, &s.l_x, &s.a_x, &s.g_x, &s.sh_x, &s.sl_x};
    for (int i = 0; i < 6; ++i) *ins[i] = (uint64_t*)c->scan_in[i].p, *outs[i] = (uint64_t*)c->scan_out[i].p;
    s.aligned = (flags & V2P_GEN_ALIGNED) ? 1 : 0;
    s.fasta = fasta ? 1 : 0;

    for (int i = 0; i < 6; ++i)  // sentinel entry [n_sel] of every scan input
        CU(c->err, cudaMemsetAsync((char*)c->scan_in[i].p + n_sel * 8, 0, 8, st));
    if (n_sel) {
        k_tg_site_hap<<<blocks(n_sel), 256, 0, st>>>(s);
        k_tg_classify<<<blocks(n_sel), 256, 0, st>>>(s, cat);
    }
    for (int i = 0; i < 5; ++i)
        if ((rc = exclusive_sum(c->err, c->cub_tmp, (const uint64_t*)*ins[i], *outs[i], n_sel + 1, st))) return rc;
    // totals: n_tasks, n_groups
    CU(c->err, c->pub.reserve(64));
    {
        v2p::PubList pl{};
        pl.src[0] = (const unsigned long long*)(s.task_x + n_sel), pl.src[1] = (const unsigned long long*)(s.g_x + n_sel);
        pl.src[2] = s.bad, pl.n = 3;
        v2p::k_publish_list<<<1, 32, 0, st>>>(c->pub.p, pl);
    }
    CU(c->err, cudaStreamSynchronize(st));
    const uint64_t n_tasks = c->pub.p[0], n_groups = c->pub.p[1];
    if (c->pub.p[2] != ~0ull)
        return fail(c->err, V2P_ERR_INVALID_ARG, "site list entry %llu is not a catalogue site (< %llu) in strictly ascending order "
                    "inside its haplotype", c->pub.p[2], (unsigned long long)c->n_sites);

    Grp g{};
    g.n_groups = n_groups;
    CU(c->err, c->g_first.need((n_groups + 1) * 8));
    CU(c->err, c->g_len.need((n_groups + 1) * 8));
    CU(c->err, c->g_slot.need((n_groups + 1) * 8));
    CU(c->err, c->g_slot_x.need((n_groups + 1) * 8));
    CU(c->err, c->g_hap.need((n_groups + 1) * 4));
    CU(c->err, c->g_tx.need((n_groups + 1) * 4));
    CU(c->err, c->ann_start.need((n_groups + 1) * 8));
    CU(c->err, c->ann_end.need((n_groups + 1) * 8));
    CU(c->err, c->tasks.need((n_tasks + 1) * sizeof(v2p_task16)));
    CU(c->err, c->task_begin.need((n_hap + 1) * 8));
    CU(c->err, c->alt_base.need((n_hap + 1) * 8));
    CU(c->err, c->out_base.need((n_hap + 1) * 8));
    CU(c->err, c->alt_per_hap.need((n_hap + 1) * 8));
    CU(c->err, c->short_tot.need((n_hap + 1) * 8));
    g.g_first = (uint64_t*)c->g_first.p, g.g_len = (uint64_t*)c->g_len.p, g.g_slot = (uint64_t*)c->g_slot.p;
    g.g_slot_x = (uint64_t*)c->g_slot_x.p, g.g_hap = (uint32_t*)c->g_hap.p, g.g_tx = (uint32_t*)c->g_tx.p;
    g.ann_start = (uint64_t*)c->ann_start.p, g.ann_end = (uint64_t*)c->ann_end.p;
    Out o{};
    o.tasks = (v2p_task16*)c->tasks.p, o.task_begin = (uint64_t*)c->task_begin.p, o.alt_base = (uint64_t*)c->alt_base.p;
    o.out_base = (uint64_t*)c->out_base.p, o.alt_per_hap = (uint64_t*)c->alt_per_hap.p, o.short_tot = (uint64_t*)c->short_tot.p;
    o.mut_dst = (uint64_t*)c->mut_dst.p;

    k_tg_groups<<<blocks(n_sel + 1), 256, 0, st>>>(s, cat, g);
    k_tg_group_sizes<<<blocks(n_groups + 1), 256, 0, st>>>(s, cat, g);
    if ((rc = exclusive_sum(c->err, c->cub_tmp, (const uint64_t*)g.g_slot, g.g_slot_x, n_groups + 1, st))) return rc;
    k_tg_hap_bases<<<blocks(n_hap + 1), 256, 0, st>>>(s, g, o);
    if (n_sel) k_tg_emit_tasks<<<blocks(n_sel), 256, 0, st>>>(s, cat, g, o);
    v2p::PubList pl{};
    if (s.aligned) {
        if ((rc = exclusive_sum(c->err, c->cub_tmp, (const uint64_t*)s.slotl, s.sl_x, n_sel + 1, st))) return rc;
        k_tg_alt_sizes<<<blocks(n_hap + 1), 256, 0, st>>>(s, o);
        if ((rc = exclusive_sum(c->err, c->cub_tmp, (const uint64_t*)o.alt_per_hap, o.alt_base, n_hap + 1, st))) return rc;
        pl.src[0] = (const unsigned long long*)(o.alt_base + n_hap);
    } else {
        pl.src[0] = (const unsigned long long*)(s.a_x + n_sel);
    }
    pl.src[1] = (const unsigned long long*)(g.g_slot_x + n_groups);
    pl.src[2] = (const unsigned long long*)(s.sh_x + n_sel);  // FASTA: bytes of the name tape
    pl.n = 3;
    v2p::k_publish_list<<<1, 32, 0, st>>>(c->pub.p, pl);
    CU(c->err, cudaStreamSynchronize(st));
    const uint64_t n_out = c->pub.p[1], n_alt = c->pub.p[0] + (fasta ? c->pub.p[2] : 0);
    CU(c->err, c->alt.need(n_alt + 64));
    CU(c->err, c->out.need(n_out + 64));
    o.alt = (uint8_t*)c->alt.p;
    CU(c->err, cudaMemsetAsync(o.alt, '.', n_alt + 16, st));
    if (n_sel) k_tg_emit_alt<<<blocks(n_sel), 256, 0, st>>>(s, cat, o);
    CU(c->err, cudaEventRecord(c->ev1, st));
    CU(c->err, cudaGetLastError());
    CU(c->err, cudaStreamSynchronize(st));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, c->ev0, c->ev1);

    out->batch.task_begin = o.task_begin;
    out->batch.tasks = o.tasks;
    out->batch.ref = nullptr;  // the proteome registered with v2p_engine_set_reference
    out->batch.ref_base = nullptr;
    out->batch.alt = o.alt;
    out->batch.alt_base = o.alt_base;
    out->batch.out = (uint8_t*)c->out.p;
    out->batch.out_base = o.out_base;
    out->batch.n_hap = n_hap;
    out->batch.n_tasks = n_tasks;
    out->batch.n_alt = n_alt;
    out->batch.n_out = n_out;
    out->n_rows = n_groups;
    out->ann_hap = g.g_hap;
    out->ann_tx = g.g_tx;
    out->ann_start = g.ann_start;
    out->ann_end = g.ann_end;
    out->n_sites = n_sel;
    out->gen_ms = ms;
    return V2P_OK;
}

// General catalogue: site_begin / sites are device pointers; c->ev0 has been recorded by the caller.
int generate_ins_on_device(v2p_catalogue* c, uint64_t n_hap, uint64_t n_sel, const uint64_t* d_site_begin,
                           const uint32_t* d_sites, uint32_t flags, v2p_generated* out) {
    cudaStream_t st = c->stream;
    const bool fasta = (flags & V2P_GEN_FASTA) != 0;
    if (flags & V2P_GEN_ALIGNED)
        return fail(c->err, V2P_ERR_INVALID_ARG, "the general catalogue generates the reference's packed layout only (no V2P_GEN_ALIGNED)");
    if (fasta && !c->has_names) return fail(c->err, V2P_ERR_INVALID_ARG, "V2P_GEN_FASTA needs v2p_catalogue_set_names first");
    int rc;
    CU(c->err, c->site_hap.need(n_sel * 4 + 16));
    CU(c->err, c->gi_newg.need((n_sel + 1) * 8));
    CU(c->err, c->gi_gx.need((n_sel + 1) * 8));
    CU(c->err, c->gi_err.need(16));
    CU(c->err, c->sel_err.need(16));
    CU(c->err, c->task_begin.need((n_hap + 1) * 8));
    CU(c->err, c->alt_base.need((n_hap + 1) * 8));
    CU(c->err, c->out_base.need((n_hap + 1) * 8));
    CU(c->err, c->pub.reserve(64));
    InsCat cat{(const uint64_t*)c->tx_off.p, (const uint32_t*)c->tx.p, (const uint8_t*)c->i_code.p, (const uint8_t*)c->i_flags.p,
               (const uint32_t*)c->i_pos_ref.p, (const uint32_t*)c->i_pos_res.p, (const uint32_t*)c->i_len.p,
               (const uint32_t*)c->dlen.p, (const uint64_t*)c->doff.p, (const uint8_t*)c->pool.p,
               (const uint64_t*)c->name_off.p, (const uint8_t*)c->names.p};
    InsGen g{};
    g.n_sel = n_sel, g.n_hap = n_hap, g.sites = d_sites, g.site_begin = d_site_begin;
    g.site_hap = (const uint32_t*)c->site_hap.p;
    g.newg = (uint64_t*)c->gi_newg.p, g.g_x = (uint64_t*)c->gi_gx.p;
    g.err = (unsigned long long*)c->gi_err.p;
    g.fasta = fasta ? 1 : 0;
    g.skip_aborts = (flags & V2P_GEN_SKIP_ABORTS) ? 1 : 0;
    CU(c->err, cudaMemsetAsync(g.err, 0xFF, 8, st));
    CU(c->err, cudaMemsetAsync(g.err + 1, 0, 8, st));
    g.bad_site = (const unsigned long long*)c->sel_err.p;
    CU(c->err, cudaMemsetAsync(c->sel_err.p, 0xFF, 8, st));
    if (n_sel) {
        Sel sh{};
        sh.n_sel = n_sel, sh.n_hap = n_hap, sh.site_begin = d_site_begin, sh.site_hap = (uint32_t*)c->site_hap.p;
        sh.sites = d_sites, sh.n_cat = c->n_sites, sh.bad = (unsigned long long*)c->sel_err.p;
        k_tg_site_hap<<<blocks(n_sel), 256, 0, st>>>(sh);
    }
    k_ti_mark<<<blocks(n_sel + 1), 256, 0, st>>>(g, cat);
    if ((rc = exclusive_sum(c->err, c->cub_tmp, (const uint64_t*)g.newg, g.g_x, n_sel + 1, st))) return rc;
    {
        v2p::PubList pl{};
        pl.src[0] = (const unsigned long long*)(g.g_x + n_sel), pl.src[1] = g.bad_site, pl.n = 2;
        v2p::k_publish_list<<<1, 32, 0, st>>>(c->pub.p, pl);
    }
    CU(c->err, cudaStreamSynchronize(st));
    const uint64_t G = c->pub.p[0];
    if (c->pub.p[1] != ~0ull)
        return fail(c->err, V2P_ERR_INVALID_ARG, "site list entry %llu is not a catalogue site (< %llu) in strictly ascending order "
                    "inside its haplotype", c->pub.p[1], (unsigned long long)c->n_sites);
    g.n_groups = G;
    CU(c->err, c->gi_first.need((G + 1) * 8));
    CU(c->err, c->gi_size.need((G + 1) * 8));
    CU(c->err, c->gi_hap.need((G + 1) * 4));
    CU(c->err, c->gi_tx.need((G + 1) * 4));
    CU(c->err, c->gi_nsites.need((G + 1) * 4));
    CU(c->err, c->gi_status.need(G + 1));
    for (int i = 0; i < 7; ++i) {
        CU(c->err, c->gi_c[i].need((G + 1) * 8));
        CU(c->err, c->gi_x[i].need((G + 1) * 8));
    }
    g.g_first = (uint64_t*)c->gi_first.p, g.g_size = (uint64_t*)c->gi_size.p, g.g_hap = (uint32_t*)c->gi_hap.p;
    g.g_tx = (uint32_t*)c->gi_tx.p, g.g_nsites = (uint32_t*)c->gi_nsites.p, g.g_status = (uint8_t*)c->gi_status.p;
    uint64_t** cin[7] = {&g.c_tasks, &g.c_alt, &g.c_name, &g.c_adv, &g.c_tape, &g.c_rows, &g.c_skip};
    uint64_t** cx[7] = {&g.x_tasks, &g.x_alt, &g.x_name, &g.x_adv, &g.x_tape, &g.x_rows, &g.x_skip};
    for (int i = 0; i < 7; ++i) *cin[i] = (uint64_t*)c->gi_c[i].p, *cx[i] = (uint64_t*)c->gi_x[i].p;
    k_ti_count<<<blocks(n_sel + 1), 256, 0, st>>>(g, cat);
    for (int i = 0; i < 7; ++i)
        if ((rc = exclusive_sum(c->err, c->cub_tmp, (const uint64_t*)*cin[i], *cx[i], G + 1, st))) return rc;
    {
        v2p::PubList pl{};
        const uint64_t* tot[8] = {g.x_tasks + G, g.x_alt + G, g.x_name + G, g.x_tape + G, g.x_rows + G, g.x_skip + G,
                                  (const uint64_t*)g.err, (const uint64_t*)(g.err + 1)};
        for (int i = 0; i < 8; ++i) pl.src[i] = (const unsigned long long*)tot[i];
        pl.n = 8;
        v2p::k_publish_list<<<1, 32, 0, st>>>(c->pub.p, pl);
    }
    CU(c->err, cudaGetLastError());
    CU(c->err, cudaStreamSynchronize(st));
    const uint64_t n_tasks = c->pub.p[0], n_alt = c->pub.p[1] + c->pub.p[2], n_out = c->pub.p[3], n_rows = c->pub.p[4],
                   n_skip = c->pub.p[5], bad = c->pub.p[6], n_abort = c->pub.p[7];
    if (bad != ~0ull && !g.skip_aborts) {  // name the transcript the reference aborts on
        uint32_t hh = 0, tt = 0;
        cudaMemcpy(&hh, g.g_hap + bad, 4, cudaMemcpyDeviceToHost);
        cudaMemcpy(&tt, g.g_tx + bad, 4, cudaMemcpyDeviceToHost);
        return fail(c->err, V2P_ERR_TASKGEN,
                    "haplotype %u transcript %u: the reference aborts while generating its tasks (usize underflow in "
                    "add_till_next_ins / add_last_instruction, or a negative result size)", hh, tt);
    }
    CU(c->err, c->tasks.need((n_tasks + 1) * sizeof(v2p_task16)));
    CU(c->err, c->alt.need(n_alt + 64));
    CU(c->err, c->out.need(n_out + 64));
    CU(c->err, c->g_hap.need((n_rows + 1) * 4));
    CU(c->err, c->g_tx.need((n_rows + 1) * 4));
    CU(c->err, c->ann_start.need((n_rows + 1) * 8));
    CU(c->err, c->ann_end.need((n_rows + 1) * 8));
    InsOut o{(v2p_task16*)c->tasks.p, (uint64_t*)c->task_begin.p, (uint64_t*)c->alt_base.p, (uint64_t*)c->out_base.p,
             (uint8_t*)c->alt.p, (uint32_t*)c->g_hap.p, (uint32_t*)c->g_tx.p, (uint64_t*)c->ann_start.p, (uint64_t*)c->ann_end.p};
    k_ti_hap_bases<<<blocks(n_hap + 1), 256, 0, st>>>(g, o);
    if (G) k_ti_emit<<<blocks(G), 256, 0, st>>>(g, cat, o);
    CU(c->err, cudaEventRecord(c->ev1, st));
    CU(c->err, cudaGetLastError());
    CU(c->err, cudaStreamSynchronize(st));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, c->ev0, c->ev1);
    out->batch.task_begin = o.task_begin, out->batch.tasks = o.tasks;
    out->batch.ref = nullptr, out->batch.ref_base = nullptr;
    out->batch.alt = o.alt, out->batch.alt_base = o.alt_base;
    out->batch.out = (uint8_t*)c->out.p, out->batch.out_base = o.out_base;
    out->batch.n_hap = n_hap, out->batch.n_tasks = n_tasks, out->batch.n_alt = n_alt, out->batch.n_out = n_out;
    out->n_rows = n_rows;
    out->ann_hap = o.ann_hap, out->ann_tx = o.ann_tx, out->ann_start = o.ann_start, out->ann_end = o.ann_end;
    out->n_sites = n_sel, out->gen_ms = ms, out->n_skipped = n_skip, out->n_aborted = n_abort;
    return V2P_OK;
}

}  // namespace
