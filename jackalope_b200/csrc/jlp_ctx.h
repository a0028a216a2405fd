// Internal to the library, not installed: the context and device types behind the C ABI (include/jlp_b200.h) and the
// helpers its drivers share.  jlp_api.cu defines the functions declared here; the drivers are jlp_run_illumina.cu,
// jlp_run_pacbio.cu, jlp_run_vcf.cu, jlp_run_haps.cu and jlp_run_vcf_read.cu.
#pragma once

#include "../../include/jlp_b200.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdint>
#include <exception>
#include <functional>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "jlp_host.h"
#include "jlp_kernels.cuh"
#include "jlp_output.h"
#include "jlp_pacbio.h"

namespace jlp {

// Bytes of padding in front of and behind every sequence allocation: the read kernel
// fetches template bases as aligned words and may touch a few bytes outside a chromosome.
constexpr size_t kPad = 64;

// A failed call is reported once: the thread's last error is reset, so that a failure a caller recovers from (a
// cudaMalloc too large) is not reported again by the next kernel launch's cudaGetLastError().
#define CK(call)                                                                          \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) {                                                          \
            cudaGetLastError();                                                           \
            throw CudaErr(std::string(#call) + ": " + cudaGetErrorString(e_));            \
        }                                                                                 \
    } while (0)

template <typename T> struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    void ensure(size_t count) {
        if (count <= n) return;
        if (p) cudaFree(p);
        p = nullptr; n = 0;
        CK(cudaMalloc(reinterpret_cast<void**>(&p), std::max<size_t>(count, 1) * sizeof(T)));
        n = count;
    }
    void upload(const std::vector<T>& v, cudaStream_t s) {
        ensure(v.size());
        if (!v.empty()) CK(cudaMemcpyAsync(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, s));
    }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
    ~DevBuf() { release(); }
};

template <typename T> struct PinBuf {
    T* p = nullptr;
    size_t n = 0;
    void ensure(size_t count) {
        if (count <= n) return;
        if (p) cudaFreeHost(p);
        p = nullptr; n = 0;
        CK(cudaMallocHost(reinterpret_cast<void**>(&p), std::max<size_t>(count, 1) * sizeof(T)));
        n = count;
    }
    ~PinBuf() { if (p) cudaFreeHost(p); }
};

// AllMutations of one haplotype chromosome (src/hap_classes.h:100-104) as the library keeps them on the host:
// a haplotype chromosome is materialised on a device only when a run's pair range touches it (SURVEY.md 8e:
// "each GPU needs only the haplotypes its range touches"), so the records outlive jlp_add_haplotype.
struct HapChromHost {
    uint64_t size = 0;                                   // mutated chromosome size
    uint64_t n_muts = 0;
    // one array, one upload: old_pos[n] | new_pos[n] | nuc_off[n] | size_modifier[n] (src/hap_classes.h:314-333) | the
    // nucleotide pool, padded to whole words
    std::vector<uint64_t> packed;
    uint64_t pool_bytes = 0;
};
struct HapStore {
    std::string name;
    std::vector<HapChromHost> chrom;
};

// Device memory of the materialised haplotype chromosomes: carved out of a few large slabs (one cudaMalloc per GiB,
// not one per chromosome -- 96 haplotypes x 20 chromosomes would be 1920 allocations); freed together.
struct HapArena {
    std::vector<uint8_t*> slabs;
    size_t used = 0, cap = 0;
    uint8_t* alloc(size_t n);
    void release() { for (uint8_t* p : slabs) cudaFree(p); slabs.clear(); used = cap = 0; }
    ~HapArena() { release(); }
};

// inline, as the other members of these types: the library exports the C ABI only
inline uint8_t* HapArena::alloc(size_t n) {
    n = (n + 255) & ~(size_t)255;
    if (slabs.empty() || used + n > cap) {
        const size_t want = std::max<size_t>(n, (size_t)1 << 30);
        uint8_t* p = nullptr;
        CK(cudaMalloc(reinterpret_cast<void**>(&p), want));
        slabs.push_back(p);
        used = 0; cap = want;
    }
    uint8_t* r = slabs.back() + used;
    used += n;
    return r;
}

// The device BGZF coder's buffers for one or two files: per file one 64 KiB slot per block, the members' sizes and
// offsets, and the contiguous compressed image (`out`, what the D2H copy moves); the codes of the batch.
struct Bgzf {
    DevBuf<uint8_t> slots[2], out[2], code;
    DevBuf<uint32_t> zlen[2];
    DevBuf<uint64_t> zoff[2];
    int files = 1;
    // room per file for nblk blocks holding in_bytes: a member never exceeds its input plus 64 bytes (a block that does
    // not compress is stored)
    void ensure(uint32_t nblk, uint64_t in_bytes, int n_files) {
        files = n_files;
        for (int e = 0; e < n_files; e++) {
            slots[e].ensure((size_t)nblk * kBgzfSlot);
            out[e].ensure(in_bytes + (size_t)nblk * 64 + 64);
            zlen[e].ensure(nblk);
            zoff[e].ensure(nblk);
        }
        code.ensure(kBgzfCodeBytes);
    }
    // launch_bgzf on the files of the last ensure(); with one file, totals[1] must be 0: the second file's buffers alias
    // the first's.  Levels 4 and above also search for matches.
    cudaError_t launch(const uint8_t* in0, const uint8_t* in1, uint64_t* totals, uint32_t nblk, int level, cudaStream_t s) {
        const int f = files - 1;
        return launch_bgzf(in0, in1, totals, nblk, level >= 4, slots[0].p, slots[f].p, zlen[0].p, zlen[f].p, zoff[0].p, zoff[f].p,
                           out[0].p, out[f].p, code.p, s);
    }
};

struct Slot {
    DevBuf<uint8_t> out[2];
    DevBuf<EndPlan> plan;
    DevBuf<uint32_t> rec_len, rec_local;
    DevBuf<uint64_t> block_tot, block_base, totals;
    PinBuf<uint8_t> h_out[2];
    PinBuf<uint64_t> h_totals;
    Bgzf z;                       // device BGZF
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // start, placed, scanned, reads done, copied, all kernels done
    uint32_t pairs = 0;
    uint64_t tot[2] = {0, 0};     // FASTQ bytes of the batch per file (read back from the device)
    uint64_t ztot[2] = {0, 0};    // compressed bytes of the batch per file (device BGZF)
    bool busy = false;
    HostBatch host;               // h_out on its way into the files
};

// Everything a context keeps on one GPU.  A device listed twice in jlp_ctx_create_multi gets two of these.
struct Device {
    int id = 0;
    int n_sm = 148;
    cudaStream_t s_compute = nullptr, s_copy = nullptr;
    cudaStream_t s_upload = nullptr;            // genome H2D, chromosome by chromosome
    // genome
    DevBuf<uint8_t> genome;
    std::vector<cudaEvent_t> chrom_ev;          // chromosome c is resident once chrom_ev[c] has fired
    bool upload_pending = false;                // some chromosome is not resident yet (or its copy not waited for)
    const char* upload_src = nullptr;           // host bases of a deferred upload (jlp_set_genome_async), else NULL
    std::vector<char> chrom_resident;           // 1: the chromosome's H2D copy has been issued
    // haplotypes: hap_seq[h][c] is chromosome c of haplotype h on this device; it aliases the reference when
    // unmutated; NULL = not materialised yet
    std::vector<std::vector<const uint8_t*>> hap_seq;
    HapArena hap_mem;
    // profiles
    DevBuf<uint32_t> d_meta[2];
    DevBuf<uint64_t> d_coin[2], d_mis[2], d_entry64[2];
    // run-scoped device data
    DevBuf<uint64_t> d_frag, d_group_off;
    DevBuf<uint32_t> d_frag_guide;
    DevBuf<GroupDev> d_groups;
    DevBuf<uint8_t> d_strpool;
    DevBuf<uint32_t> d_status;
    Slot slot[3];                               // compute | D2H copy | delivery to the sink, one batch each
    WriterPool writers;
    cudaEvent_t ev_run[2] = {nullptr, nullptr};
    uint64_t h2d_bytes = 0;
    // PacBio driver: the per-read plan of a batch (its other buffers are those of the slots)
    DevBuf<PbRead> pb_reads;
    // materialisation: the records of the next chromosomes are uploaded (s_upload) while k_materialize works on the
    // ones before (s_compute); kMatBufs scratch buffers in turn
    static constexpr int kMatBufs = 3;
    DevBuf<uint64_t> m_pack[kMatBufs];
    cudaEvent_t m_up[kMatBufs] = {nullptr, nullptr, nullptr}, m_done[kMatBufs] = {nullptr, nullptr, nullptr};
    uint64_t m_next = 0;

    void free_haps() {
        hap_seq.clear();
        hap_mem.release();
    }
    ~Device() {
        cudaSetDevice(id);
        cudaDeviceSynchronize();
        free_haps();
        for (Slot& s : slot) for (cudaEvent_t ev : s.ev) if (ev) cudaEventDestroy(ev);
        for (cudaEvent_t ev : ev_run) if (ev) cudaEventDestroy(ev);
        if (s_compute) cudaStreamDestroy(s_compute);
        if (s_copy) cudaStreamDestroy(s_copy);
        if (s_upload) cudaStreamDestroy(s_upload);
        for (int k = 0; k < kMatBufs; k++) { if (m_up[k]) cudaEventDestroy(m_up[k]); if (m_done[k]) cudaEventDestroy(m_done[k]); }
        for (cudaEvent_t ev : chrom_ev) cudaEventDestroy(ev);
        writers.stop();
    }
};

}  // namespace jlp

// What a context keeps once on the host, and its devices (one, or several for jlp_ctx_create_multi).
struct jlp_ctx {
    std::string err;
    // genome
    std::vector<uint64_t> chrom_off;
    std::vector<std::string> chrom_names;
    std::string genome_name;
    std::vector<std::shared_ptr<jlp::HapStore>> haps;
    // profiles
    jlp::EndTables tab[2];
    bool have_prof[2] = {false, false};
    // PacBioPassSampler's outlier thresholds (one chi-squared quantile per read length up to chi2_params_n[2]) of the last call
    std::shared_ptr<std::atomic<double>[]> pb_qcache;
    double pb_qcache_key[3] = {0, 0, 0};
    size_t pb_qcache_n = 0;
    std::vector<std::unique_ptr<jlp::Device>> dev;
};

// The library exports the C ABI only, so what follows is hidden.  The types above are not: jlp_ctx, which the C ABI's
// functions take, holds them.
#pragma GCC visibility push(hidden)

namespace jlp {

// ------------------------------------------------------------------------------------------ errors and devices ---

int fail(jlp_ctx* c, int code, const std::string& msg);

template <typename F> int guarded(jlp_ctx* c, F f) {
    try {
        if (c && c->dev.size() == 1) CK(cudaSetDevice(c->dev[0]->id));
        f();
        return JLP_OK;
    } catch (const ArgErr& e) { return fail(c, JLP_ERR_ARG, e.what());
    } catch (const CudaErr& e) { return fail(c, JLP_ERR_CUDA, e.what());
    } catch (const IoErr& e) { return fail(c, JLP_ERR_IO, e.what());
    } catch (const Unsupported& e) { return fail(c, JLP_ERR_UNSUPPORTED, e.what());
    } catch (const Aborted& e) { return fail(c, JLP_ERR_ABORTED, e.what());
    } catch (const std::exception& e) { return fail(c, JLP_ERR_ARG, e.what()); }
}

Device& device0(jlp_ctx* c);

// f(d) for every device d of the context, made current: on the calling thread for one device, else on one host thread
// per device while the calling thread runs `wait` every 20 ms (if given).  The first error other than Aborted is
// rethrown with its type (CUDA errors name their device), else Aborted if a device was aborted.
template <typename F> void on_each_device(jlp_ctx* c, F f, const std::function<void()>& wait = nullptr) {
    const size_t N = c->dev.size();
    if (N == 1) {
        CK(cudaSetDevice(c->dev[0]->id));
        f(*c->dev[0]);
        return;
    }
    std::vector<std::exception_ptr> errs(N);
    std::atomic<size_t> left{N};
    std::vector<std::thread> th;
    for (size_t r = 0; r < N; r++)
        th.emplace_back([&, r]() {
            Device& d = *c->dev[r];
            try {
                CK(cudaSetDevice(d.id));
                f(d);
            } catch (const CudaErr& e) {
                errs[r] = std::make_exception_ptr(CudaErr("device " + std::to_string(d.id) + ": " + e.what()));
            } catch (...) {
                errs[r] = std::current_exception();
            }
            left.fetch_sub(1);
        });
    while (wait && left.load() != 0) {
        std::this_thread::sleep_for(std::chrono::milliseconds(20));
        wait();
    }
    for (std::thread& t : th) t.join();
    for (const std::exception_ptr& e : errs)
        if (e) try { std::rethrow_exception(e); } catch (const Aborted&) {}
    for (const std::exception_ptr& e : errs)
        if (e) std::rethrow_exception(e);
}

// ------------------------------------------------------------------------------------ genome and haplotypes ---

void clear_haps(jlp_ctx* c);
void issue_upload(const jlp_ctx* c, Device& d, size_t first, size_t last);
void finish_upload(const jlp_ctx* c, Device& d);
int claim_mat_buf(Device& d);
void ensure_hap_chrom(const jlp_ctx* c, Device& d, size_t h, size_t ci);
void attach_hap(jlp_ctx* c, const std::shared_ptr<HapStore>& S);

// the reference's chromosome lengths, JLP_ERR_ARG if one has 2^32 bases or more
std::vector<uint64_t> chrom_lengths(const jlp_ctx* c);

// Haplotypes made on the first device, one region per (haplotype, chromosome), r = haplotype * chromosomes + chromosome:
// its records in the HapChromHost::packed layout at src[r] (device memory; unread when n[r] == 0), their pool bytes and
// the chromosome's size.
struct HapRegions {
    std::vector<std::string> names;
    std::vector<const uint64_t*> src;
    std::vector<uint64_t> n, pool, size;
};
// the regions copied into one HapStore per haplotype by up to `threads` host threads (one when there are few records);
// the stores replace the context's haplotypes
void store_haps(jlp_ctx* c, const HapRegions& G, unsigned threads);

// ------------------------------------------------------------------------------------------------------ layout ---

struct Job {
    uint64_t lo, hi;          // pair-instance range
    std::string file_prefix;  // <prefix> or <prefix>_<hap>
};

void shard_range(uint64_t job_lo, uint64_t job_hi, uint32_t si, uint32_t S, uint64_t& lo, uint64_t& hi);

// What a run's groups and jobs depend on besides the context, from the parameters of either driver (which name these
// fields alike); Illumina adds its barcodes.
struct LayoutSpec {
    uint64_t seed;
    uint64_t n_units;                          // pairs (Illumina: floor(n_reads / n_ends)) or reads (PacBio)
    bool use_haps;                             // the haplotypes, else the reference
    const double* hap_probs;
    const char* const* barcodes = nullptr;     // one per haplotype (one for the reference), or NULL
    uint32_t read_len = 0;                     // a barcode must be shorter than the read
    bool sep_files;                            // one job per haplotype
    const char* prefix;
    template <typename Params> LayoutSpec(bool haps, const Params* P, uint64_t units)
        : seed(P->seed), n_units(units), use_haps(haps), hap_probs(P->haplotype_probs), sep_files(P->sep_files != 0),
          prefix(P->out_prefix) {}
};

// The (haplotype, chromosome) groups of a run in the order the reference exhausts them (hap-major, chrom-major:
// src/hts_illumina.cpp:199-201, :505-528), their pair-index prefix offsets, ID-line prefixes and barcodes, and the
// jobs (= sets of output files).  A pure function of the parameters and of the sizes the context knows: a multi-GPU
// run builds it once for all its devices.
struct Layout {
    uint64_t n_pairs = 0;
    std::vector<uint64_t> group_off;      // [n_groups + 1]
    std::vector<GroupDev> groups;         // seq is filled in per device
    std::vector<uint32_t> group_hap, group_chrom;
    std::vector<uint8_t> strpool;
    std::vector<Job> jobs;
};

Layout make_layout(const jlp_ctx* c, const LayoutSpec& S);
std::vector<std::vector<uint64_t>> apportion(const jlp_ctx* c, const LayoutSpec& S);
std::string file_name(const Job& job, int e, bool gz, const jlp_illumina_params* P);

// ------------------------------------------------------------------------------------------------------ output ---

void check_compression(int compress, const char* comp_method, int comp_engine);
Compression file_compression(int compress, const char* comp_method, uint64_t n_threads, int comp_engine, SinkKind kind);

// If a run ends by an exception, nothing of it may stay in flight: kernels and copies still use the slots, writer
// tasks still hold the file descriptors the caller's Output is about to close.  Files the run extends itself are cut
// back to the last completely written batch (an extended, never filled tail would otherwise stay behind as zero bytes).
struct Quiesce {
    Device& d;
    Output* out;
    bool armed = true;
    ~Quiesce() {
        if (!armed) return;
        cudaStreamSynchronize(d.s_compute);
        cudaStreamSynchronize(d.s_copy);
        HostBatch* b[3];
        for (int k = 0; k < 3; k++) { d.slot[k].busy = false; b[k] = &d.slot[k].host; }
        out->abandon(b, 3);
    }
};

void hand_over(Device& d, Output& sink, uint64_t& n_batch, const uint8_t* src, uint64_t nb, uint64_t job, uint64_t cap);

// ------------------------------------------------------------------------------------- host threads and timing ---

unsigned host_threads(uint64_t items);
float elapsed_ms(cudaEvent_t a, cudaEvent_t b);

}  // namespace jlp

#pragma GCC visibility pop
