// v2p_host.hpp -- C++17 host-side mirror of the reference's engine interface, over the C ABI (v2p_engine.h).
//
// The reference's host is Rust; its toolchain is not available in this image, so this header is what the host side
// above the boundary looks like in a compiled language, with the reference's own names and argument meaning:
//
//   v2p::Engine / Engine::from_str     src/data_structures/InternalRep/engines.rs:15-30
//   v2p::Task                          .../task.rs:2-19                 {exe_code, start_pos, length, start_pos_res}
//   v2p::GIR  / GIR::execute(Engine)   .../gir.rs:15-46, :197-241       consumes the representation, returns
//                                                                       (res_array, annotation); GPU arm -> C ABI
//   v2p::HaplotypeBatch                .../haplotype_instruction.rs:75-158  get_g_rep's concat + re-index loop
//                                      (update_task :140-158), generalised to MANY haplotypes per launch and to the
//                                      B200 layouts (shared proteome tape, phase-aligned result slots)
//   v2p::Instruction / InstructionCatalogue   .../instruction.rs:6-16   the host's Instruction values, uploaded once;
//                                      Task generation then happens on the device (include/v2p_taskgen.h)
//   v2p::Pipeline / v2p::DirWriter     parts/exec.rs:27-41 + parts/io.rs:35-57: every proband's haplotypes executed and
//                                      written as {out_dir}/{proband}.fasta[.gz] (include/v2p_pipeline.h)
//
// Errors: where the reference panics (task.rs:44/48, haplotype_instruction.rs:154, gir.rs:223) this throws
// v2p::EngineError carrying the ABI status and the offending haplotype/task.  ST and MT are the caller's CPU engines
// (gir.rs:201-235): GIR::execute refuses them, it never computes on the host.
#ifndef V2P_HOST_HPP
#define V2P_HOST_HPP

#include <cstdint>
#include <map>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "v2p_engine.h"
#include "v2p_cohort.h"
#include "v2p_pipeline.h"
#include "v2p_vcf.h"
#include "v2p_vcf_bgzf.h"

namespace v2p {

struct EngineError : std::runtime_error {
    int status;
    uint64_t bad_hap, bad_task;
    EngineError(int st, const std::string& msg, uint64_t h = 0, uint64_t t = 0)
        : std::runtime_error(msg + " (status " + std::to_string(st) + ")"), status(st), bad_hap(h), bad_task(t) {}
};

// engines.rs:15
enum class Engine { ST = V2P_ENGINE_ST, MT = V2P_ENGINE_MT, GPU = V2P_ENGINE_GPU };

// engines.rs:17-30 -- Err(format!("{} is not a supported engine", name)) becomes an exception
inline Engine engine_from_str(const std::string& name) {
    int kind = -1;
    if (v2p_engine_from_str(name.c_str(), &kind) != V2P_OK) throw EngineError(V2P_ERR_BAD_ENGINE, name + " is not a supported engine");
    return static_cast<Engine>(kind);
}

// task.rs:2-9
struct Task {
    uint8_t exe_code;
    uint64_t start_pos, length, start_pos_res;
    Task(uint8_t c, uint64_t sp, uint64_t len, uint64_t spr) : exe_code(c), start_pos(sp), length(len), start_pos_res(spr) {}
    uint64_t get_length() const { return length; }
    uint64_t get_start_pos_res() const { return start_pos_res; }
    uint8_t get_stream() const { return exe_code; }
    void shift_start_pos_stream(uint64_t n) { start_pos += n; }  // task.rs:103-107
    void shift_start_pos_res(uint64_t n) { start_pos_res += n; }  // task.rs:108-112
};

using Annotation = std::map<std::string, std::pair<uint64_t, uint64_t>>;  // HashMap<String,(usize,usize)>

// One engine context (one per GPU); RAII over v2p_engine_create / v2p_engine_destroy.
class Context {
public:
    explicit Context(int cuda_device = 0) {
        if (v2p_engine_create(cuda_device, &e_) != V2P_OK)
            throw EngineError(V2P_ERR_CUDA, "no usable CUDA device: the GPU engine has no CPU fallback");
    }
    ~Context() { v2p_engine_destroy(e_); }
    Context(const Context&) = delete;
    Context& operator=(const Context&) = delete;
    v2p_engine* get() const { return e_; }
    std::string last_error() const { return v2p_last_error(e_); }
    void set_reference(const std::string& proteome_tape, uint32_t flags = 0) {
        int st = v2p_engine_set_reference(e_, reinterpret_cast<const uint8_t*>(proteome_tape.data()), proteome_tape.size(), flags);
        if (st != V2P_OK) throw EngineError(st, last_error());
    }

private:
    v2p_engine* e_ = nullptr;
};

// gir.rs:15-23.  Tapes are UTF-32 (Rust `char`) like the reference's Vec<char>.
class GIR {
public:
    GIR(std::vector<Task> g_rep, Annotation annotation, std::u32string alt_stream, std::u32string ref_stream,
        std::u32string res_array)
        : g_rep_(std::move(g_rep)), annotation_(std::move(annotation)), alt_(std::move(alt_stream)),
          ref_(std::move(ref_stream)), res_(std::move(res_array)) {}
    const std::vector<Task>& get_tasks() const { return g_rep_; }
    const Annotation& get_annotation() const { return annotation_; }
    uint64_t get_results_max() const {  // gir.rs:157-168
        uint64_t m = 0;
        for (const auto& kv : annotation_) m = kv.second.second > m ? kv.second.second : m;
        return m;
    }
    // gir.rs:197-241: consumes self; `validate` is the DEBUG_GPU / DEBUG_CPU_EXEC contiguity check (gir.rs:203-229)
    std::pair<std::u32string, Annotation> execute(Engine engine, Context& ctx, bool validate = false) && {
        if (engine != Engine::GPU)
            throw EngineError(V2P_ERR_NOT_GPU_ENGINE, "ST/MT engines are the caller's CPU path (gir.rs:201-235)");
        // gir.rs:283-299 consume_and_produce_produce_content: four usize arrays + three char tapes
        const size_t n = g_rep_.size();
        std::vector<uint64_t> code(n), sp(n), len(n), spr(n);
        for (size_t i = 0; i < n; ++i) {
            code[i] = g_rep_[i].exe_code, sp[i] = g_rep_[i].start_pos, len[i] = g_rep_[i].length, spr[i] = g_rep_[i].start_pos_res;
        }
        uint64_t bad = 0;
        int st = v2p_gir_execute(ctx.get(), V2P_ENGINE_GPU, n, code.data(), sp.data(), len.data(), spr.data(),
                                 reinterpret_cast<const uint32_t*>(ref_.data()), ref_.size(),
                                 reinterpret_cast<const uint32_t*>(alt_.data()), alt_.size(),
                                 reinterpret_cast<uint32_t*>(&res_[0]), res_.size(), validate ? V2P_FLAG_VALIDATE : 0u, &bad);
        if (st != V2P_OK) throw EngineError(st, ctx.last_error(), 0, bad);
        return {std::move(res_), std::move(annotation_)};
    }

private:
    std::vector<Task> g_rep_;
    Annotation annotation_;
    std::u32string alt_, ref_, res_;
};

// Many haplotypes per launch: HaplotypeInstruction::get_g_rep's concat loop (haplotype_instruction.rs:94-133),
// writing straight into the packed batch layout of v2p_execute_batch.
class HaplotypeBatch {
public:
    enum class RefLayout { PerHaplotype, SharedProteome };  // haplotype_instruction.rs:118  vs  registered tape
    explicit HaplotypeBatch(RefLayout layout = RefLayout::PerHaplotype, bool aligned_slots = false)
        : layout_(layout), aligned_(aligned_slots) {
        if (aligned_ && layout_ != RefLayout::SharedProteome) throw std::invalid_argument("aligned slots need the shared proteome tape");
    }

    void begin_haplotype() {  // ref_counter = alt_counter = res_counter = 0  (haplotype_instruction.rs:91)
        task_begin_.push_back(tasks_.size());
        alt_base_.push_back(alt_.size());
        out_base_.push_back(out_size_);
        ref_base_.push_back(ref_.size());
        annotations_.emplace_back();
        ref_counter_ = alt_counter_ = res_counter_ = 0;
    }

    // One transcript's GIR (TranscriptInstruction::get_g_rep output): tasks relative to the transcript, its alt
    // stream, its reference sequence (PerHaplotype) or its offset in the registered proteome (SharedProteome),
    // and the size of its result array (compute_expected_results_array_size).
    void add_transcript(const std::string& name, const std::vector<Task>& tasks, const std::string& alt_stream,
                        const std::string& ref_stream, uint64_t proteome_offset, uint64_t res_len) {
        if (task_begin_.empty()) throw std::logic_error("begin_haplotype() first");
        uint64_t res_start = res_counter_, slot = res_len;
        if (aligned_ && res_len) {  // result in phase with the proteome tape inside a 16-byte-multiple slot
            const uint64_t c = proteome_offset & 15u;  // res_counter_ is a multiple of 16 here by construction
            res_start = res_counter_ + c;
            slot = (c + res_len + 15u) & ~uint64_t(15);
        }
        const uint64_t ref_shift = layout_ == RefLayout::PerHaplotype ? ref_counter_ : proteome_offset;
        for (const Task& t : tasks) {  // update_task, haplotype_instruction.rs:140-158
            uint64_t src;
            if (t.exe_code == 0) src = t.start_pos + ref_shift;
            else if (t.exe_code == 1) src = t.start_pos + alt_counter_;
            else throw EngineError(V2P_ERR_BAD_STREAM, "Unsupported Stream code", task_begin_.size() - 1, tasks_.size() - task_begin_.back());
            const uint64_t dst = t.start_pos_res + res_start;
            if (src > 0xFFFFFFFFull || dst > 0xFFFFFFFFull || t.length > 0xFFFFFFFFull)
                throw std::length_error("haplotype tape beyond 4 GiB");
            tasks_.push_back(v2p_task16{(uint32_t)src, (uint32_t)t.length, (uint32_t)dst, (uint32_t)t.exe_code});
        }
        alt_.append(alt_stream);
        if (layout_ == RefLayout::PerHaplotype) ref_.append(ref_stream);
        annotations_.back()[name] = {res_start, res_start + res_len};  // haplotype_instruction.rs:120-125
        ref_counter_ += ref_stream.size();
        alt_counter_ += alt_stream.size();
        res_counter_ += slot;
        out_size_ += slot;
    }

    size_t n_haplotypes() const { return task_begin_.size(); }
    const std::vector<v2p_task16>& tasks() const { return tasks_; }
    const Annotation& annotation(size_t h) const { return annotations_[h]; }

    // Executes every haplotype (n_hap x GIR::execute in one launch group); returns the concatenated result tapes.
    // result(h) = out.substr(out_base(h), out_base(h+1)-out_base(h)); slice it by annotation(h) like SequenceTape::get_seq.
    std::string execute(Engine engine, Context& ctx, bool validate = false) {
        if (engine != Engine::GPU)
            throw EngineError(V2P_ERR_NOT_GPU_ENGINE, "ST/MT engines are the caller's CPU path (gir.rs:201-235)");
        const size_t H = task_begin_.size();
        std::vector<uint64_t> tb(task_begin_), ab(alt_base_), ob(out_base_), rb(ref_base_);
        tb.push_back(tasks_.size()), ab.push_back(alt_.size()), ob.push_back(out_size_), rb.push_back(ref_.size());
        std::string out(out_size_, '\0');
        v2p_batch b{};
        b.task_begin = tb.data(), b.tasks = tasks_.data();
        if (layout_ == RefLayout::PerHaplotype) {
            b.ref = reinterpret_cast<const uint8_t*>(ref_.data());
            b.ref_base = rb.data();
            b.n_ref = ref_.size();
        }  // SharedProteome: ref == NULL -> the tape registered with Context::set_reference
        b.alt = reinterpret_cast<const uint8_t*>(alt_.data()), b.alt_base = ab.data();
        b.out = reinterpret_cast<uint8_t*>(&out[0]), b.out_base = ob.data();
        b.n_hap = H;
        v2p_result r{};
        int st = v2p_execute_batch(ctx.get(), &b, validate ? V2P_FLAG_VALIDATE : 0u, &r, nullptr);
        if (st != V2P_OK) throw EngineError(st, ctx.last_error(), r.bad_hap, r.bad_task);
        out_base_final_ = ob;
        return out;
    }
    uint64_t out_base(size_t h) const { return out_base_final_.at(h); }

private:
    RefLayout layout_;
    bool aligned_;
    std::vector<v2p_task16> tasks_;
    std::vector<uint64_t> task_begin_, alt_base_, out_base_, ref_base_, out_base_final_;
    std::string alt_, ref_;
    std::vector<Annotation> annotations_;
    uint64_t ref_counter_ = 0, alt_counter_ = 0, res_counter_ = 0, out_size_ = 0;
};

// sequence_tape.rs:9-117 -- the consumer of a haplotype's result tape: sequences annotated head to tail on one string.
// The engine never sees it; it is here so that a C++ host slices results exactly as the reference does.
class SequenceTape {
public:
    // sequence_tape.rs:33-41: Err("Bad Tape Encountered ...") when an annotation ends beyond the tape
    SequenceTape(std::string seq_str, Annotation annotations) : seq_(std::move(seq_str)), ann_(std::move(annotations)) {
        const uint64_t mx = get_max_index(ann_);
        if (mx > seq_.size())
            throw std::invalid_argument("Bad Tape Encountered, the provided maximum index is " + std::to_string(mx) +
                                        " while tape length is " + std::to_string(seq_.size()));
    }
    const Annotation& get_annotation() const { return ann_; }
    // sequence_tape.rs:77-89
    std::string get_seq(const std::string& seq_name) const {
        auto it = ann_.find(seq_name);
        if (it == ann_.end()) throw std::out_of_range("The provided sequence name: " + seq_name + ", is not defined in the current table");
        return seq_.substr(it->second.first, it->second.second - it->second.first);
    }
    // sequence_tape.rs:105-116
    static uint64_t get_max_index(const Annotation& a) {
        uint64_t m = 0;
        for (const auto& kv : a) m = kv.second.second > m ? kv.second.second : m;
        return m;
    }
    // personalized_genome.rs:97,107: the records of one haplotype, `>{name}_{1|2}\n{seq}\n`
    std::string fasta_text(int hap_label) const {
        std::string out;
        for (const auto& kv : ann_) out += ">" + kv.first + "_" + std::to_string(hap_label) + "\n" + get_seq(kv.first) + "\n";
        return out;
    }

private:
    std::string seq_;
    Annotation ann_;
};

// instruction.rs:6-16, as Instruction::from_mutation builds it with validate_s_state taken as true, plus the two facts
// the device needs to redo that validation per haplotype (include/v2p_taskgen.h).
struct Instruction {
    uint32_t transcript;  // index into the proteome's transcript table
    char code;
    bool star;         // the consequence class is '*'-prefixed
    bool invalidates;  // stop_gained / frameshift / *stop_gained / inframe ins-del whose mutated field is or ends in '*'
    uint32_t pos_ref, pos_res, len;
    std::string data;
};

// The general catalogue on one GPU: instructions sorted by (transcript, mutated position), transcript names for the
// FASTA headers.  RAII over v2p_catalogue_create_ins / v2p_catalogue_destroy.
class InstructionCatalogue {
public:
    InstructionCatalogue(int cuda_device, const std::vector<uint64_t>& tx_offsets, const std::vector<std::string>& tx_names,
                         const std::vector<Instruction>& ins) {
        std::vector<uint32_t> tx, pr, ps, ln, dl;
        std::vector<uint8_t> code, flags;
        std::vector<uint64_t> doff, name_off(1, 0);
        std::string pool, names;
        for (const Instruction& i : ins) {
            tx.push_back(i.transcript), code.push_back((uint8_t)i.code);
            flags.push_back((i.star ? V2P_INS_STAR : 0u) | (i.invalidates ? V2P_INS_INVALIDATES : 0u));
            pr.push_back(i.pos_ref), ps.push_back(i.pos_res), ln.push_back(i.len);
            doff.push_back(pool.size()), dl.push_back((uint32_t)i.data.size());
            pool += i.data;
        }
        for (const std::string& n : tx_names) names += n, name_off.push_back(names.size());
        int st = v2p_catalogue_create_ins(cuda_device, tx_offsets.size() - 1, tx_offsets.data(), ins.size(), tx.data(), code.data(),
                                          flags.data(), pr.data(), ps.data(), ln.data(), doff.data(), dl.data(),
                                          reinterpret_cast<const uint8_t*>(pool.data()), pool.size(), &c_);
        if (st != V2P_OK) throw EngineError(st, "v2p_catalogue_create_ins failed");
        st = v2p_catalogue_set_names(c_, name_off.data(), reinterpret_cast<const uint8_t*>(names.data()));
        if (st != V2P_OK) {
            const std::string msg = v2p_catalogue_last_error(c_);
            v2p_catalogue_destroy(c_);
            throw EngineError(st, msg);
        }
    }
    ~InstructionCatalogue() { v2p_catalogue_destroy(c_); }
    InstructionCatalogue(const InstructionCatalogue&) = delete;
    InstructionCatalogue& operator=(const InstructionCatalogue&) = delete;
    v2p_catalogue* get() const { return c_; }

private:
    v2p_catalogue* c_ = nullptr;
};

// parts/io.rs:35-57: {out_dir}/{proband}.fasta or .fasta.gz, one file per proband.
class DirWriter {
public:
    DirWriter(const std::string& out_dir, const std::vector<std::string>& probands, bool write_compressed, unsigned threads = 4) {
        std::vector<const char*> names;
        for (const std::string& p : probands) names.push_back(p.c_str());
        if (v2p_dir_writer_create(out_dir.c_str(), names.data(), names.size(), write_compressed ? 1 : 0, threads, &w_) != V2P_OK)
            throw EngineError(V2P_ERR_INVALID_ARG, "v2p_dir_writer_create failed");
    }
    ~DirWriter() { v2p_dir_writer_destroy(w_); }
    DirWriter(const DirWriter&) = delete;
    DirWriter& operator=(const DirWriter&) = delete;
    v2p_dir_writer* get() const { return w_; }
    uint64_t files_written() const { return v2p_dir_writer_files(w_); }
    uint64_t bytes_written() const { return v2p_dir_writer_bytes(w_); }

private:
    v2p_dir_writer* w_ = nullptr;
};

// parts/exec.rs:27-41 for Engine::GPU: every proband's two haplotypes, from their mutation lists to files.
// `lanes`: one catalogue object per chunk in flight, built from the same instructions.
class Pipeline {
public:
    Pipeline(Context& ctx, const std::vector<InstructionCatalogue*>& lanes) {
        std::vector<v2p_catalogue*> raw;
        for (InstructionCatalogue* c : lanes) raw.push_back(c->get());
        if (v2p_pipeline_create(ctx.get(), raw.data(), (uint32_t)raw.size(), &p_) != V2P_OK)
            throw EngineError(V2P_ERR_INVALID_ARG, "v2p_pipeline_create failed");
    }
    ~Pipeline() { v2p_pipeline_destroy(p_); }
    Pipeline(const Pipeline&) = delete;
    Pipeline& operator=(const Pipeline&) = delete;

    // The reference's `-a` flag (write_all, personalized_genome.rs:120-210): call once, then pass write_all = true.
    void enable_write_all(const std::string& proteome, const std::vector<uint64_t>& tx_offsets, const std::vector<std::string>& tx_names) {
        std::vector<uint64_t> name_off(1, 0);
        std::string names;
        for (const std::string& n : tx_names) names += n, name_off.push_back(names.size());
        const int st = v2p_pipeline_enable_all_records(p_, reinterpret_cast<const uint8_t*>(proteome.data()), proteome.size(),
                                                       tx_offsets.size() - 1, tx_offsets.data(), name_off.data(),
                                                       reinterpret_cast<const uint8_t*>(names.data()));
        if (st != V2P_OK) throw EngineError(st, v2p_pipeline_last_error(p_));
    }

    // per_haplotype[2 * proband + (hap - 1)] = ascending catalogue indices of the mutations that haplotype carries
    v2p_pipeline_result write(const std::vector<std::vector<uint32_t>>& per_haplotype, DirWriter& writer, bool write_compressed,
                              uint32_t chunk_probands = 128, bool write_all = false) {
        std::vector<uint64_t> begin(1, 0);
        std::vector<uint32_t> sites;
        for (const auto& l : per_haplotype) {
            sites.insert(sites.end(), l.begin(), l.end());
            begin.push_back(sites.size());
        }
        v2p_pipeline_result r{};
        const int st = v2p_pipeline_run_lists(p_, per_haplotype.size() / 2, begin.data(), sites.data(), chunk_probands,
                                              (write_compressed ? V2P_PIPE_GZIP : 0u) | (write_all ? V2P_PIPE_ALL_RECORDS : 0u), nullptr,
                                              0, nullptr, v2p_dir_writer_sink, writer.get(), &r);
        if (st != V2P_OK) throw EngineError(st, v2p_pipeline_last_error(p_));
        return r;
    }

private:
    v2p_pipeline* p_ = nullptr;
};

// parts/exec.rs:34-40 + parts/io.rs:45-57 over EVERY GPU named, from this one process: a worker (host thread, engine
// with the proteome registered, catalogue lanes, pinned ring, pipeline) per device, contiguous proband ranges, the
// directory writer as the common sink.  RAII over v2p_cohort_create / v2p_cohort_destroy (include/v2p_cohort.h).
class Cohort {
public:
    Cohort(const std::vector<int>& cuda_devices, const std::string& proteome, const std::vector<uint64_t>& tx_offsets,
           const std::vector<std::string>& tx_names, const std::vector<Instruction>& ins, unsigned lanes_per_device = 2) {
        std::vector<uint32_t> tx, pr, ps, ln, dl;
        std::vector<uint8_t> code, flags;
        std::vector<uint64_t> doff, name_off(1, 0);
        std::string pool, names;
        for (const Instruction& i : ins) {
            tx.push_back(i.transcript), code.push_back((uint8_t)i.code);
            flags.push_back((i.star ? V2P_INS_STAR : 0u) | (i.invalidates ? V2P_INS_INVALIDATES : 0u));
            pr.push_back(i.pos_ref), ps.push_back(i.pos_res), ln.push_back(i.len);
            doff.push_back(pool.size()), dl.push_back((uint32_t)i.data.size());
            pool += i.data;
        }
        for (const std::string& n : tx_names) names += n, name_off.push_back(names.size());
        v2p_cohort_inputs in{};
        in.proteome = reinterpret_cast<const uint8_t*>(proteome.data()), in.n_proteome = proteome.size();
        in.n_tx = tx_offsets.size() - 1, in.tx_offsets = tx_offsets.data();
        in.name_off = name_off.data(), in.names = reinterpret_cast<const uint8_t*>(names.data());
        in.general = 1, in.n_sites = ins.size(), in.site_tx = tx.data();
        in.ins_code = code.data(), in.ins_flags = flags.data(), in.ins_pos_ref = pr.data(), in.ins_pos_res = ps.data(), in.ins_len = ln.data();
        in.site_doff = doff.data(), in.site_dlen = dl.data(), in.pool = reinterpret_cast<const uint8_t*>(pool.data()), in.n_pool = pool.size();
        const int st = v2p_cohort_create(cuda_devices.data(), (uint32_t)cuda_devices.size(), &in, lanes_per_device, &c_);
        if (st != V2P_OK) throw EngineError(st, "v2p_cohort_create failed (a device is missing? there is no CPU fallback)");
    }
    ~Cohort() { v2p_cohort_destroy(c_); }
    Cohort(const Cohort&) = delete;
    Cohort& operator=(const Cohort&) = delete;

    // The reference's `-a` flag on every device (v2p_cohort_enable_all_records): call once, then pass write_all = true.
    void enable_write_all(const std::string& proteome, const std::vector<uint64_t>& tx_offsets, const std::vector<std::string>& tx_names) {
        std::vector<uint64_t> name_off(1, 0);
        std::string names;
        for (const std::string& n : tx_names) names += n, name_off.push_back(names.size());
        v2p_cohort_inputs in{};
        in.proteome = reinterpret_cast<const uint8_t*>(proteome.data()), in.n_proteome = proteome.size();
        in.n_tx = tx_offsets.size() - 1, in.tx_offsets = tx_offsets.data();
        in.name_off = name_off.data(), in.names = reinterpret_cast<const uint8_t*>(names.data());
        const int st = v2p_cohort_enable_all_records(c_, &in);
        if (st != V2P_OK) throw EngineError(st, v2p_cohort_last_error(c_));
    }

    v2p_cohort_result write(const std::vector<std::vector<uint32_t>>& per_haplotype, DirWriter& writer, bool write_compressed,
                            uint32_t chunk_probands = 128, bool write_all = false) {
        std::vector<uint64_t> begin(1, 0);
        std::vector<uint32_t> sites;
        for (const auto& l : per_haplotype) {
            sites.insert(sites.end(), l.begin(), l.end());
            begin.push_back(sites.size());
        }
        v2p_cohort_result r{};
        const int st = v2p_cohort_run_lists(c_, per_haplotype.size() / 2, begin.data(), sites.data(), chunk_probands,
                                            (write_compressed ? V2P_PIPE_GZIP : 0u) | (write_all ? V2P_PIPE_ALL_RECORDS : 0u) | V2P_COHORT_CONCURRENT_SINK,
                                            v2p_dir_writer_sink,
                                            writer.get(), &r);
        if (st != V2P_OK) throw EngineError(st, v2p_cohort_last_error(c_));
        return r;
    }

private:
    v2p_cohort* c_ = nullptr;
};

// VCF sample columns on the device (include/v2p_vcf.h): the text is loaded and indexed once; the host reads columns 1-9
// of the records it wants (text[line_begin, cells_begin)) and parses their sample cells into the FORMAT/BCSQ mask
// matrix, which stays on the device for v2p_pipeline_run_masks / v2p_cohort_run_masks.  RAII over v2p_vcf_create.
class VcfText {
public:
    explicit VcfText(int cuda_device = 0) {
        if (v2p_vcf_create(cuda_device, &v_) != V2P_OK) throw EngineError(V2P_ERR_CUDA, "v2p_vcf_create failed (no such device?)");
    }
    ~VcfText() { v2p_vcf_destroy(v_); }
    VcfText(const VcfText&) = delete;
    VcfText& operator=(const VcfText&) = delete;

    // Host text (pinned memory uploads at the full PCIe rate), or device text on this object's device (16-byte aligned,
    // alive until the next load).  The tables in the result are owned by this object until the next load.
    const v2p_vcf_lines& load(const uint8_t* text, uint64_t n_bytes, bool device_text = false) {
        const int st = v2p_vcf_load(v_, text, n_bytes, device_text ? V2P_FLAG_DEVICE_PTRS : 0u, &lines_);
        if (st != V2P_OK) throw EngineError(st, v2p_vcf_last_error(v_));
        bgzf_ = v2p_vcf_bgzf{};
        set_names(device_text ? nullptr : text);
        return lines_;
    }
    const v2p_vcf_lines& load(const std::string& text) { return load(reinterpret_cast<const uint8_t*>(text.data()), text.size()); }

    // A bgzip'd file (host memory; pinned uploads at the full PCIe rate), inflated and indexed on the device.  Offsets
    // in the result are into the inflated text; the host reads columns 1-9 from bgzf().fixed (sliced by fixed_begin)
    // and the header lines from bgzf().head.  Both are owned by this object until the next load.
    const v2p_vcf_lines& load_bgzf(const uint8_t* data, uint64_t n_bytes) {
        const int st = v2p_vcf_load_bgzf(v_, data, n_bytes, 0, &lines_, &bgzf_);
        if (st != V2P_OK) throw EngineError(st, v2p_vcf_last_error(v_));
        set_names(bgzf_.head);
        return lines_;
    }
    const v2p_vcf_lines& load_bgzf(const std::string& data) { return load_bgzf(reinterpret_cast<const uint8_t*>(data.data()), data.size()); }

    // What the last load_bgzf found (zeroed after a plain load).
    const v2p_vcf_bgzf& bgzf() const { return bgzf_; }

    // Columns 1-9 of data line l after load_bgzf.
    std::string fixed(uint64_t l) const {
        return std::string(reinterpret_cast<const char*>(bgzf_.fixed) + bgzf_.fixed_begin[l], bgzf_.fixed_begin[l + 1] - bgzf_.fixed_begin[l]);
    }

    // Sample names of the #CHROM line (host text or BGZF input).
    const std::vector<std::string>& sample_names() const { return names_; }

    // Row r of the matrix = data line rec_line[r].  The matrix is device memory owned by this object until the next call.
    v2p_vcf_masks parse_masks(const std::vector<uint64_t>& rec_line) {
        v2p_vcf_masks m{};
        const int st = v2p_vcf_parse_masks(v_, rec_line.size(), rec_line.data(), 0, &m);
        if (st != V2P_OK) throw EngineError(st, v2p_vcf_last_error(v_));
        return m;
    }

    // Device -> host copy of a matrix (tests, debugging).
    static std::vector<uint32_t> read(const v2p_vcf_masks& m) {
        std::vector<uint32_t> out(m.n_records * m.n_samples * m.words_per_cell);
        if (!out.empty() && v2p_device_read(out.data(), m.masks, out.size() * sizeof(uint32_t)) != V2P_OK)
            throw EngineError(V2P_ERR_CUDA, "v2p_device_read failed");
        return out;
    }

    v2p_vcf* get() { return v_; }

private:
    void set_names(const uint8_t* text) {  // text[header_begin, header_end) is the #CHROM line
        names_.clear();
        if (!text || !lines_.n_samples) return;
        const std::string hdr(reinterpret_cast<const char*>(text) + lines_.header_begin, lines_.header_end - lines_.header_begin);
        size_t col = 0, at = 0;
        for (size_t tab = hdr.find('\t'); ; tab = hdr.find('\t', at)) {
            if (col++ >= 9) names_.push_back(hdr.substr(at, tab == std::string::npos ? std::string::npos : tab - at));
            if (tab == std::string::npos) break;
            at = tab + 1;
        }
    }

    v2p_vcf* v_ = nullptr;
    v2p_vcf_lines lines_{};
    v2p_vcf_bgzf bgzf_{};
    std::vector<std::string> names_;
};

}  // namespace v2p
#endif  // V2P_HOST_HPP
