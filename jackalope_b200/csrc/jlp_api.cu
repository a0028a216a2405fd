// C ABI (include/jlp_b200.h): context, genome / haplotype / profile upload, and
// the batch pipeline that stands in for write_reads_cpp_ / write_reads_cpp_sep_files_
// / write_reads_one_filetype_ (/root/reference/src/hts.h:323-552).
#include "../../include/jlp_b200.h"

#include <cuda_runtime.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <sys/statvfs.h>
#include <unistd.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <cctype>
#include <cerrno>
#include <chrono>
#include <cmath>
#include <deque>
#include <exception>
#include <functional>
#include <thread>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "jlp_deflate.h"
#include "jlp_draws.h"
#include "jlp_host.h"
#include "jlp_kernels.cuh"
#include "jlp_output.h"
#include "jlp_pacbio.h"

using namespace jlp;

namespace {

std::string g_create_error;

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

}  // namespace

// What a context keeps once on the host, and its devices (one, or several for jlp_ctx_create_multi).
struct jlp_ctx {
    std::string err;
    // genome
    std::vector<uint64_t> chrom_off;
    std::vector<std::string> chrom_names;
    std::string genome_name;
    std::vector<std::shared_ptr<HapStore>> haps;
    // profiles
    EndTables tab[2];
    bool have_prof[2] = {false, false};
    // PacBioPassSampler's outlier thresholds (one chi-squared quantile per read length up to chi2_params_n[2]) of the last call
    std::shared_ptr<std::atomic<double>[]> pb_qcache;
    double pb_qcache_key[3] = {0, 0, 0};
    size_t pb_qcache_n = 0;
    std::vector<std::unique_ptr<Device>> dev;
};

namespace {

uint8_t* HapArena::alloc(size_t n) {
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

int fail(jlp_ctx* c, int code, const std::string& msg) {
    if (c) c->err = msg; else g_create_error = msg;
    return code;
}

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

// The device of the calls that use only the first one (PacBio, create_haplotypes, ...), made current.
Device& device0(jlp_ctx* c) {
    CK(cudaSetDevice(c->dev[0]->id));
    return *c->dev[0];
}

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

void clear_haps(jlp_ctx* c) {
    c->haps.clear();
    on_each_device(c, [](Device& d) { d.free_haps(); });
}

// Issue the H2D copies of chromosomes [first, last] of a deferred genome upload (those not
// issued yet); every copy is followed by its chromosome's event.
void issue_upload(const jlp_ctx* c, Device& d, size_t first, size_t last) {
    if (!d.upload_src) return;
    for (size_t i = first; i <= last && i < d.chrom_resident.size(); i++) {
        if (d.chrom_resident[i]) continue;
        const uint64_t len = c->chrom_off[i + 1] - c->chrom_off[i];
        if (len) CK(cudaMemcpyAsync(d.genome.p + kPad + c->chrom_off[i], d.upload_src + c->chrom_off[i], len, cudaMemcpyHostToDevice, d.s_upload));
        CK(cudaEventRecord(d.chrom_ev[i], d.s_upload));
        d.chrom_resident[i] = 1;
        d.h2d_bytes += len;
    }
}
// Make the whole genome resident and wait for it.
void finish_upload(const jlp_ctx* c, Device& d) {
    if (!d.upload_pending) return;
    if (!d.chrom_resident.empty()) issue_upload(c, d, 0, d.chrom_resident.size() - 1);
    CK(cudaStreamSynchronize(d.s_upload));
    d.upload_pending = false;
    d.upload_src = nullptr;
}

// What the genome setters share: drop the genome and the haplotypes, give every device a buffer for the new genome,
// record its chromosomes once all devices have one, then fill(d) on every device.  If any of it fails, the context
// is left without a genome, as a fresh context is.
template <typename F> void replace_genome(jlp_ctx* c, const std::vector<uint64_t>& off, const std::vector<std::string>& names,
                                          const char* genome_name, F fill) {
    try {
        c->chrom_off.clear();
        c->chrom_names.clear();
        c->haps.clear();
        on_each_device(c, [&](Device& d) {
            d.free_haps();
            if (d.upload_pending) {      // a deferred upload that never ran is simply dropped
                d.upload_pending = false;
                d.upload_src = nullptr;
                CK(cudaStreamSynchronize(d.s_upload));
            }
            d.genome.ensure(off.back() + 2 * kPad);
        });
        c->chrom_off = off;
        c->chrom_names = names;
        c->genome_name = genome_name ? genome_name : "REF";
        on_each_device(c, fill);
    } catch (...) {
        c->chrom_off.clear();
        c->chrom_names.clear();
        for (auto& d : c->dev) { d->upload_pending = false; d->upload_src = nullptr; }    // the caller's bases are not read again
        throw;
    }
}

// ---------------------------------------------------------------- the run ---

struct Job {
    uint64_t lo, hi;          // pair-instance range
    std::string file_prefix;  // <prefix> or <prefix>_<hap>
};


// Contiguous, near-equal split of a job's pair-index range over shards (the even split of
// split_int, src/util.h:245-258, applied to GPUs instead of threads).
void shard_range(uint64_t job_lo, uint64_t job_hi, uint32_t si, uint32_t S, uint64_t& lo, uint64_t& hi) {
    const uint64_t nj = job_hi - job_lo;
    lo = job_lo + nj / S * si + std::min<uint64_t>(si, nj % S);
    hi = lo + nj / S + (si < nj % S ? 1 : 0);
}

// Pairs per (haplotype, chromosome): threads -> haplotypes -> chromosomes
// (write_reads_one_filetype_ src/hts.h:334-353, add_n_reads src/hts_illumina.h:410-418 and :620-644,
//  write_reads_cpp_sep_files_ src/hts.h:527-529).  One "thread"; n_pairs = floor(n_reads / n_ends).
// A reference run has one pseudo-haplotype.  Both the pooled and the sep_files haplotype paths first
// split pairs over haplotypes by haplotype_probs, then each haplotype's pairs over its chromosomes
// by size, so one routine serves both.
std::vector<std::vector<uint64_t>> apportion_sizes(uint64_t seed, uint64_t n_pairs, uint64_t n_haps, uint64_t n_chroms,
                                                   const double* hap_probs, const uint64_t* sizes) {
    uint64_t sub_seed = seed * 0x9E3779B97F4A7C15ull + 0x1234567ull;
    auto next_seed = [&]() { sub_seed = sub_seed * 6364136223846793005ull + 1442695040888963407ull; return sub_seed; };
    std::vector<std::vector<uint64_t>> out;
    if (!hap_probs) {
        std::vector<double> w(n_chroms);
        for (uint64_t i = 0; i < n_chroms; i++) w[i] = (double)sizes[i];
        out.push_back(reads_per_group(n_pairs, w, next_seed()));
        return out;
    }
    std::vector<double> hp(hap_probs, hap_probs + n_haps);
    bool any = false;
    for (double v : hp) { if (!(v >= 0)) throw ArgErr("haplotype_probs must be >= 0"); any |= v > 0; }
    if (!any) throw ArgErr("haplotype_probs must have at least one value > 0");
    std::vector<uint64_t> hap_pairs = reads_per_group(n_pairs, hp, next_seed());
    for (uint64_t h = 0; h < n_haps; h++) {
        std::vector<double> w(n_chroms);
        for (uint64_t i = 0; i < n_chroms; i++) w[i] = (double)sizes[h * n_chroms + i];
        out.push_back(reads_per_group(hap_pairs[h], w, next_seed()));
    }
    return out;
}

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

std::vector<std::vector<uint64_t>> apportion(const jlp_ctx* c, const LayoutSpec& S) {
    if (c->chrom_off.size() < 2) throw ArgErr("no reference genome has been set");
    if (S.use_haps && c->haps.empty()) throw ArgErr("no haplotypes have been added");
    const uint64_t n_chroms = c->chrom_off.size() - 1;
    std::vector<uint64_t> sizes;
    if (!S.use_haps) {
        for (uint64_t i = 0; i < n_chroms; i++) sizes.push_back(c->chrom_off[i + 1] - c->chrom_off[i]);
        return apportion_sizes(S.seed, S.n_units, 1, n_chroms, nullptr, sizes.data());
    }
    if (!S.hap_probs) throw ArgErr("haplotype_probs is NULL");
    for (const auto& h : c->haps)
        for (const HapChromHost& M : h->chrom) sizes.push_back(M.size);
    return apportion_sizes(S.seed, S.n_units, c->haps.size(), n_chroms, S.hap_probs, sizes.data());
}

// How a run's compressed output is produced (write_reads_cpp_, src/hts.h:441-500): compressed + one thread -> the
// method asked for; compressed + several threads -> always bgzip (the reference writes plain files first and bgzips
// them afterwards; here the batches are compressed on their way to the file).  comp_engine picks who compresses:
// the device coder (BGZF members of one dynamic-Huffman block each, jlp_bgzf.cu; only compressed bytes cross PCIe)
// or zlib on the writer threads at the level asked for.  AUTO uses the device coder only where the reference itself
// would write BGZF (comp_method "bgzip", or several threads) at levels 1..6; a gzip request with one thread is a
// gzip stream from zlib (FileGZ, src/io.h:140-236).  Memory and stream sinks receive compressed bytes only when the
// device coder is asked for explicitly.
Compression compression_of(const jlp_illumina_params* P, SinkKind kind) {
    Compression z;
    if (P->compress <= 0) return z;
    const std::string m = P->comp_method ? P->comp_method : "";
    const bool bgzip = P->n_threads > 1 || m == "bgzip";
    z.want_gz = true;
    z.dev_z = P->comp_engine == JLP_COMP_DEVICE || (P->comp_engine == JLP_COMP_AUTO && P->compress <= 6 && kind == SINK_FILES && bgzip);
    if (!z.dev_z) z.zmethod = bgzip ? DEFLATE_BGZF : DEFLATE_GZIP;
    return z;
}

// The compression arguments of every driver.  A level <= 0 is no compression, and the method is then not looked at.
void check_compression(int compress, const char* comp_method, int comp_engine) {
    const std::string m = comp_method ? comp_method : "";
    if (compress > 0 && m != "gzip" && m != "bgzip") throw ArgErr("\nUnrecognized compression method.");  // src/hts.h:470
    if (compress > 9) throw ArgErr("\nInvalid bgzip compress level of " + std::to_string(compress) +
                                   ". It must be in range [0,9].");                                      // src/io.h:113-117
    if (comp_engine < JLP_COMP_AUTO || comp_engine > JLP_COMP_DEVICE) throw ArgErr("comp_engine must be 0 (auto), 1 (host) or 2 (device)");
}

// the argument checks the C++ layer of the reference performs, plus the ranges of the additions
void check_params(const jlp_ctx* c, bool use_haps, const jlp_illumina_params* P, SinkKind kind) {
    if (!P) throw ArgErr("params is NULL");
    const int n_ends = P->paired || P->matepair ? 2 : 1;
    if (c->chrom_off.size() < 2) throw ArgErr("no reference genome has been set");
    if (use_haps && c->haps.empty()) throw ArgErr("no haplotypes have been added");
    if (!c->have_prof[0]) throw ArgErr("no quality profile for read 1");
    if (n_ends == 2) {
        if (!c->have_prof[1]) throw ArgErr("no quality profile for read 2");
        if (c->tab[0].L != c->tab[1].L)   // src/hts_illumina.h:348-352
            throw ArgErr("In IlluminaOneGenome constr., read lengths for R1 and R2 don't match.");
    }
    check_compression(P->compress, P->comp_method, P->comp_engine);
    if (!(P->prob_dup >= 0 && P->prob_dup <= 1)) throw ArgErr("prob_dup must be in [0,1]");
    const double insp[2] = {P->ins_prob1, P->ins_prob2}, delp[2] = {P->del_prob1, P->del_prob2};
    for (int e = 0; e < n_ends; e++)
        if (!(insp[e] >= 0 && insp[e] <= 1 && delp[e] >= 0 && delp[e] <= 1))
            throw ArgErr("insertion / deletion probabilities must be in [0,1]");
    if (P->frag_len_min < 1 || P->frag_len_min > P->frag_len_max)
        throw ArgErr("frag_len_min must be >= 1 and <= frag_len_max");
    if (!(P->frag_len_shape > 0 && P->frag_len_scale > 0)) throw ArgErr("fragment Gamma shape and scale must be > 0");
    if (P->read_pool_size < 1) throw ArgErr("read_pool_size must be >= 1");
    if (kind == SINK_FILES && (!P->out_prefix || !*P->out_prefix)) throw ArgErr("out_prefix is empty");
    if (use_haps && !P->haplotype_probs) throw ArgErr("haplotype_probs is NULL");
    if (P->shard_count > 1 && P->shard_index >= P->shard_count) throw ArgErr("shard_index >= shard_count");
}

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

Layout make_layout(const jlp_ctx* c, const LayoutSpec& S) {
    Layout Y;
    const uint64_t n_haps = c->haps.size(), n_chroms = c->chrom_off.size() - 1;
    const bool use_haps = S.use_haps, sep = use_haps && S.sep_files;
    // --- barcodes (T/C/A/G only, R/hts_illumina.R:385-391)
    std::vector<std::string> barcodes(use_haps ? n_haps : 1);
    if (S.barcodes)
        for (size_t i = 0; i < barcodes.size(); i++) {
            barcodes[i] = S.barcodes[i] ? S.barcodes[i] : "";
            for (char ch : barcodes[i])
                if (ch != 'T' && ch != 'C' && ch != 'A' && ch != 'G') throw ArgErr("barcodes may only contain T, C, A, G");
            if (barcodes[i].size() >= S.read_len) throw ArgErr("a barcode is as long as the read");
        }
    // --- apportion pairs: threads -> haplotypes -> chromosomes
    //     (write_reads_one_filetype_ src/hts.h:334-353, add_n_reads src/hts_illumina.h:410-418, :620-644,
    //      write_reads_cpp_sep_files_ src/hts.h:527-529; PacBioOneGenome::add_n_reads, src/hts_pacbio.h); one "thread"
    Y.n_pairs = S.n_units;
    const std::vector<std::vector<uint64_t>> counts = apportion(c, S);
    Y.group_off.assign(1, 0);
    auto add_group = [&](const std::string& gname, uint32_t hap, uint64_t chrom, uint64_t len, const std::string& bc, uint64_t count) {
        GroupDev g;
        std::string pre = "@" + gname + "-" + c->chrom_names[chrom] + "-";
        g.seq = nullptr; g.len = len;
        g.prefix_off = (uint32_t)Y.strpool.size(); g.prefix_len = (uint32_t)pre.size();
        Y.strpool.insert(Y.strpool.end(), pre.begin(), pre.end());
        g.bc_off = (uint32_t)Y.strpool.size(); g.bc_len = (uint32_t)bc.size();
        Y.strpool.insert(Y.strpool.end(), bc.begin(), bc.end());
        Y.groups.push_back(g);
        Y.group_hap.push_back(hap); Y.group_chrom.push_back((uint32_t)chrom);
        Y.group_off.push_back(Y.group_off.back() + count);
        if (count > 0 && len == 0) throw ArgErr("a chromosome of length 0 was given reads");
    };
    const std::string prefix = S.prefix ? S.prefix : "";
    if (!use_haps) {
        for (uint64_t i = 0; i < n_chroms; i++)
            add_group(c->genome_name, 0, i, c->chrom_off[i + 1] - c->chrom_off[i], barcodes[0], counts[0][i]);
        Y.jobs.push_back(Job{0, Y.n_pairs, prefix});
    } else {
        for (uint64_t h = 0; h < n_haps; h++) {
            const HapStore& H = *c->haps[h];
            uint64_t lo = Y.group_off.back();
            for (uint64_t i = 0; i < n_chroms; i++) add_group(H.name, (uint32_t)h, i, H.chrom[i].size, barcodes[h], counts[h][i]);
            if (sep) Y.jobs.push_back(Job{lo, Y.group_off.back(), prefix + "_" + H.name});
        }
        if (!sep) Y.jobs.push_back(Job{0, Y.group_off.back(), prefix});
    }
    if (Y.group_off.back() != Y.n_pairs) throw std::runtime_error("internal: apportioning does not add up");
    return Y;
}

LayoutSpec illumina_spec(const jlp_ctx* c, bool use_haps, const jlp_illumina_params* P) {
    LayoutSpec S(use_haps, P, P->n_reads / (P->paired || P->matepair ? 2 : 1));
    S.barcodes = P->barcodes;
    S.read_len = (uint32_t)c->tab[0].L;
    return S;
}

// name of output file `e` of a job (src/hts.h:344; ".gz" appended by FileGZ / FileBGZF, src/io.h:126,217).
// A process that generates one shard of a run (shard_count > 1, one process per GPU) writes its own files,
// <prefix>[_<hap>]_R<k>.fq[.gz].shard<i>of<n>: concatenated in shard order they are the unsharded run's file.
std::string file_name(const Job& job, int e, bool gz, const jlp_illumina_params* P) {
    std::string n = job.file_prefix + "_R" + std::to_string(e + 1) + ".fq";
    if (gz) n += ".gz";
    if (P && P->shard_count > 1) n += ".shard" + std::to_string(P->shard_index) + "of" + std::to_string(P->shard_count);
    return n;
}

// The next of materialisation's buffers, free: the kernels that read it last, whose end the caller records in m_done,
// must be done before the buffer can grow (cudaFree) or be written again.  An event never recorded is complete.
int claim_mat_buf(Device& d) {
    const int k = (int)(d.m_next++ % Device::kMatBufs);
    CK(cudaEventSynchronize(d.m_done[k]));
    return k;
}

// Materialise haplotype chromosome (h, ci) on device d if it is not resident yet
// (HapChrom::get_chrom_full, src/hap_classes.cpp:80-116).
void ensure_hap_chrom(const jlp_ctx* c, Device& d, size_t h, size_t ci) {
    const uint8_t*& seq = d.hap_seq[h][ci];
    if (seq) return;
    const HapChromHost& M = c->haps[h]->chrom[ci];
    const uint64_t ref_size = c->chrom_off[ci + 1] - c->chrom_off[ci];
    const uint8_t* ref = d.genome.p + kPad + c->chrom_off[ci];
    const int k = claim_mat_buf(d);
    d.m_pack[k].upload(M.packed, d.s_upload);
    CK(cudaEventRecord(d.m_up[k], d.s_upload));
    d.h2d_bytes += M.n_muts * 32 + M.pool_bytes;
    uint8_t* out = d.hap_mem.alloc(M.size + 2 * kPad);
    const uint64_t* w = d.m_pack[k].p;
    const uint64_t n = M.n_muts;
    CK(cudaStreamWaitEvent(d.s_compute, d.m_up[k], 0));
    CK(launch_materialize(ref, ref_size, n, w, w + n, reinterpret_cast<const int64_t*>(w + 3 * n), w + 2 * n,
                          reinterpret_cast<const uint8_t*>(w + 4 * n), M.size, out + kPad, d.s_compute));
    CK(cudaEventRecord(d.m_done[k], d.s_compute));
    seq = out + kPad;       // valid in stream order: everything that reads it runs on s_compute
}

typedef std::vector<std::pair<uint64_t, uint64_t>> Ranges;
typedef std::vector<std::array<uint64_t, 2>> PerJobBytes;

// What a multi-GPU run tells each of its devices (jlp_ctx_create_multi); a plain call leaves everything empty.
struct RunExtras {
    const Ranges* ranges = nullptr;       // [jobs] the pair range of every job this call generates (else: the shard of P)
    PerJobBytes* sizes_out = nullptr;     // size pass: only count the FASTQ bytes per job and end of those ranges
    const PerJobBytes* base = nullptr;    // [jobs] where this call's bytes start in each job's files / in the memory sink
    bool shared_files = false;            // the files exist, created and sized by the caller: open without truncating, no EOF block
    // [jobs] compressed multi-GPU runs: this call writes <name><suffix>, joined by the caller, who appends the BGZF
    // end-of-file block
    const std::vector<std::string>* job_suffix = nullptr;
    PerJobBytes* zsizes_out = nullptr;    // the compressed bytes per job and end this call produced (device coder)
    bool dry_files = false;               // generate and compress as for files, deliver nothing (sink NONE): the compressed size pass
};

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

// One Illumina run on device d, with the run's Layout (make_layout) and parameters checked (check_params) by the caller.
void run(const jlp_ctx* c, Device& d, bool use_haps, const jlp_illumina_params* P, Layout Y, Output& sink, jlp_run_stats* stats,
         const RunExtras& X = RunExtras()) {
    const int n_ends = P->paired || P->matepair ? 2 : 1;
    const bool matepair = P->matepair != 0;
    if (use_haps) finish_upload(c, d);
    const uint64_t h2d_before = d.h2d_bytes;
    const Compression Z = compression_of(P, X.dry_files ? SINK_FILES : sink.kind);
    const bool dev_z = Z.dev_z;
    const bool sizes_only = X.sizes_out != nullptr;
    if (X.zsizes_out) X.zsizes_out->assign(X.ranges ? X.ranges->size() : 0, std::array<uint64_t, 2>{0, 0});
    const double insp[2] = {P->ins_prob1, P->ins_prob2}, delp[2] = {P->del_prob1, P->del_prob2};
    const uint32_t L = (uint32_t)c->tab[0].L;

    const std::vector<uint64_t>& group_off = Y.group_off;
    std::vector<GroupDev>& groups = Y.groups;
    const std::vector<Job>& jobs = Y.jobs;

    // --- the pair range of every job this call generates
    Ranges ranges;
    if (X.ranges) ranges = *X.ranges;
    else {
        const uint32_t S = P->shard_count > 1 ? P->shard_count : 1, si = P->shard_count > 1 ? P->shard_index : 0;
        for (const Job& j : jobs) { uint64_t lo, hi; shard_range(j.lo, j.hi, si, S, lo, hi); ranges.emplace_back(lo, hi); }
    }
    if (ranges.size() != jobs.size()) throw std::runtime_error("internal: one range per job");
    const uint64_t pool_pairs = (P->read_pool_size + n_ends - 1) / n_ends;   // pool closes at >= read_pool_size reads
    // groups a range reads: those of its pairs, and through a duplicate chain's leader possibly the one before
    // (a leader lies at most pool_pairs - 1 pairs before its duplicate, never before the job's start)
    auto groups_of = [&](const Job& job, uint64_t lo, uint64_t hi, size_t& g_lo, size_t& g_hi) {
        const uint64_t first_pair = lo - std::min<uint64_t>(lo - job.lo, pool_pairs - 1);
        g_lo = (size_t)(std::upper_bound(group_off.begin(), group_off.end(), first_pair) - group_off.begin()) - 1;
        g_hi = (size_t)(std::upper_bound(group_off.begin(), group_off.end(), hi - 1) - group_off.begin()) - 1;
        g_hi = std::min(g_hi, groups.size() - 1);
        g_lo = std::min(g_lo, g_hi);
    };
    // --- sequences: the reference's chromosomes, or the haplotype chromosomes the ranges touch (materialised now)
    if (!use_haps) {
        for (size_t g = 0; g < groups.size(); g++) groups[g].seq = d.genome.p + kPad + c->chrom_off[g];
    } else {
        for (size_t k = 0; k < jobs.size(); k++) {
            if (ranges[k].second <= ranges[k].first) continue;
            size_t g_lo, g_hi;
            groups_of(jobs[k], ranges[k].first, ranges[k].second, g_lo, g_hi);
            for (size_t g = g_lo; g <= g_hi; g++) ensure_hap_chrom(c, d, Y.group_hap[g], Y.group_chrom[g]);
        }
        for (size_t g = 0; g < groups.size(); g++) groups[g].seq = d.hap_seq[Y.group_hap[g]][Y.group_chrom[g]];
    }

    // --- thresholds
    GenParams gp;
    std::memset(&gp, 0, sizeof gp);
    gp.seed = P->seed;
    philox_round_keys(P->seed, gp.rk);
    gp.n_ends = n_ends; gp.L = L; gp.matepair = matepair;
    gp.pool_pairs = pool_pairs;
    Thr td = thr_double_lt(P->prob_dup);
    gp.c_dup = td.thr; gp.dup_never = td.thr == 0;
    gp.c_rev = thr_ld_lt(0.5).thr;
    for (int e = 0; e < n_ends; e++) {
        EndDev& E = gp.end[e];
        E.meta = d.d_meta[e].p; E.entry64 = d.d_entry64[e].p; E.coin = d.d_coin[e].p;
        E.mis = d.d_mis[e].p;
        E.entry_n = (uint32_t)c->tab[e].entry64.size();
        Thr ta = thr_double_le(insp[e] + delp[e]);   // u > ins + del  <=>  x >= tA
        Thr ti = thr_double_le(insp[e]);             // u > ins        <=>  x >= tI
        E.tA = ta.thr; E.tA_all = ta.all; E.tI = ti.thr; E.tI_all = ti.all;
        E.hA = ta.all ? 0x10000u : (uint32_t)(ta.thr >> 48);
    }
    CK(cudaEventRecord(d.ev_run[0], d.s_compute));
    std::vector<uint64_t> frag = frag_table(P->frag_len_shape, P->frag_len_scale, P->frag_len_min, P->frag_len_max);
    std::vector<uint32_t> guide = frag_guide(frag);
    d.d_frag.upload(frag, d.s_compute);
    d.d_frag_guide.upload(guide, d.s_compute);
    d.d_group_off.upload(group_off, d.s_compute);
    d.d_groups.upload(groups, d.s_compute);
    d.d_strpool.upload(Y.strpool, d.s_compute);
    d.d_status.ensure(1);
    CK(cudaMemsetAsync(d.d_status.p, 0, sizeof(uint32_t), d.s_compute));
    d.h2d_bytes += frag.size() * 8 + group_off.size() * 8 + groups.size() * sizeof(GroupDev) + Y.strpool.size();
    gp.frag_cdf = d.d_frag.p; gp.frag_guide = d.d_frag_guide.p; gp.frag_n = (uint32_t)frag.size(); gp.frag_min = P->frag_len_min;
    gp.group_off = d.d_group_off.p; gp.n_groups = (uint32_t)groups.size();
    gp.groups = d.d_groups.p; gp.strpool = d.d_strpool.p; gp.status = d.d_status.p;

    // --- batch buffers
    uint64_t max_range = 0;
    for (const auto& r : ranges) max_range = std::max(max_range, r.second - r.first);
    uint64_t B = P->batch_pairs ? P->batch_pairs : (1ull << 20);
    B = std::max<uint64_t>(1, std::min(B, max_range));
    uint32_t max_prefix = 0;
    for (const GroupDev& g : groups) max_prefix = std::max(max_prefix, g.prefix_len);
    const uint64_t max_rec = (uint64_t)max_prefix + 20 + 5 + 2ull * L + 4;
    B = std::max<uint64_t>(1, std::min<uint64_t>(B, 0xfff00000ull / max_rec));     // offsets inside a batch's output are 32 bits wide in k_reads
    gp.rec_buf = (uint32_t)((max_rec + 32 + 15) & ~15ull);   // a record at any 16-byte phase, and the 16 bytes the carry reads behind it
    gp.tpl_buf = (L + 50u + 15u) & ~15u;        // the template, 16..31 bytes in front of it, 16 behind, the word over-read
    gp.cod_buf = (L + 40u + 15u) & ~15u;        // base codes of a read's template (up to 2 more than the read with deletions), rounded up to the 16 of a lane
    if (!sizes_only && !reads_fits(gp)) throw Unsupported("read_length " + std::to_string(L) + " (with these chromosome names) needs more shared memory per "
                                                          "read pair than one SM has: the read kernel cannot hold such a record");
    const uint64_t n_rec_max = B * n_ends;
    const uint32_t nsb_max = (uint32_t)((B + kScanBlock - 1) / kScanBlock);
    const bool need_host = sink.kind != SINK_NONE && !sizes_only;
    const uint32_t nblk = (uint32_t)((B * max_rec + kBgzfIn - 1) / kBgzfIn) + 1;
    for (Slot& s : d.slot) {
        s.plan.ensure(n_rec_max);
        s.rec_len.ensure(n_rec_max);
        s.rec_local.ensure(n_rec_max);
        s.block_tot.ensure((size_t)nsb_max * 2);
        s.block_base.ensure((size_t)nsb_max * 2);
        s.totals.ensure(4);
        s.h_totals.ensure(4);
        CK(cudaMemsetAsync(s.totals.p, 0, 4 * sizeof(uint64_t), d.s_compute));
        for (int e = 0; e < n_ends && !sizes_only; e++) {
            s.out[e].ensure(B * max_rec + 64);
            // compressed bytes of a batch never exceed its FASTQ bytes plus the members' framing (an incompressible block is stored)
            // (the same size with and without compression: pinning a gigabyte again for the first compressed call took seconds)
            if (need_host) s.h_out[e].ensure(B * max_rec + (size_t)nblk * 64 + 64);
        }
        if (dev_z && !sizes_only) s.z.ensure(nblk, B * max_rec, n_ends);
        s.busy = false;
    }

    jlp_run_stats st;
    std::memset(&st, 0, sizeof st);

    sink.begin(Z, P->compress, P->n_threads, d.writers);
    Quiesce quiesce{d, &sink};
    uint64_t job_index = 0;
    // stage 2 of a batch: its kernels are done -> statistics, then its FASTQ starts its way to the host
    // (queued right behind the previous batch's copy, so the bus never idles)
    auto issue_copy = [&](Slot& s) {
        CK(cudaEventSynchronize(s.ev[5]));
        float ms_place = 0, ms_all = 0, ms_reads = 0, ms_z = 0;
        CK(cudaEventElapsedTime(&ms_place, s.ev[0], s.ev[1]));
        CK(cudaEventElapsedTime(&ms_reads, s.ev[2], s.ev[3]));
        CK(cudaEventElapsedTime(&ms_z, s.ev[3], s.ev[5]));
        CK(cudaEventElapsedTime(&ms_all, s.ev[0], s.ev[5]));
        st.place_ms += ms_place; st.reads_ms += ms_reads; st.device_ms += ms_all;
        if (dev_z) st.bgzf_ms += ms_z;
        for (int e = 0; e < n_ends; e++) {
            s.tot[e] = s.h_totals.p[e]; st.bytes_out[e] += s.tot[e];
            s.ztot[e] = dev_z ? s.h_totals.p[2 + e] : 0; st.z_bytes[e] += s.ztot[e];
            if (X.zsizes_out && job_index < X.zsizes_out->size()) (*X.zsizes_out)[job_index][e] += s.ztot[e];
        }
        st.pairs += s.pairs;
        st.batches++;
        if (!need_host) return;
        sink.settle(s.host);                    // the pinned buffers of this slot are free again
        for (int e = 0; e < n_ends; e++) {
            const uint64_t nb = dev_z ? s.ztot[e] : s.tot[e];
            CK(cudaMemcpyAsync(s.h_out[e].p, dev_z ? s.z.out[e].p : s.out[e].p, nb, cudaMemcpyDeviceToHost, d.s_copy));
            st.d2h_bytes += nb;
        }
        CK(cudaEventRecord(s.ev[4], d.s_copy));
    };
    // stage 3: the copy has landed -> hand the batch to the sink
    auto deliver = [&](Slot& s) {
        if (need_host) {
            CK(cudaEventSynchronize(s.ev[4]));
            const uint8_t* data[2] = {s.h_out[0].p, s.h_out[1].p};
            const uint64_t n[2] = {dev_z ? s.ztot[0] : s.tot[0], dev_z ? s.ztot[1] : s.tot[1]};
            sink.deliver(s.host, data, n, job_index, n_ends);
        }
        if (P->progress_cb) P->progress_cb(P->cb_user, (uint64_t)s.pairs * n_ends);
        s.busy = false;
    };

    std::vector<char> chrom_waited(d.chrom_ev.size(), 0);
    if (sizes_only) X.sizes_out->assign(jobs.size(), std::array<uint64_t, 2>{0, 0});

    for (size_t jk = 0; jk < jobs.size(); jk++) {
        const Job& job = jobs[jk];
        const uint64_t lo = ranges[jk].first, hi = ranges[jk].second;
        if (P->abort_cb && P->abort_cb(P->cb_user)) throw Aborted();   // src/hts.h:536
        if (X.ranges && hi <= lo) { job_index++; continue; }             // a multi-GPU device with no part in this job's files
        if (!sizes_only) {
            std::string names[2];
            for (int e = 0; e < n_ends; e++)
                names[e] = file_name(job, e, Z.want_gz, P) + (X.job_suffix ? (*X.job_suffix)[jk] : "");
            sink.open_job(names, n_ends, X.base ? (*X.base)[jk].data() : nullptr, X.shared_files);
        }
        if (sizes_only) {
            // size pass: placement and scan only; the totals come back batch by batch (a few hundred microseconds each)
            for (uint64_t b0 = lo; b0 < hi; b0 += B) {
                Slot& s = d.slot[0];
                const uint32_t np = (uint32_t)std::min<uint64_t>(B, hi - b0);
                gp.job_lo = job.lo; gp.job_hi = job.hi; gp.batch_lo = b0; gp.batch_pairs = np;
                gp.plan = s.plan.p; gp.rec_len = s.rec_len.p; gp.rec_local = s.rec_local.p; gp.block_base = s.block_base.p;
                gp.n_scan_blocks = (np + kScanBlock - 1) / kScanBlock;
                CK(launch_place(gp, d.s_compute));
                CK(launch_scan(s.rec_len.p, np * n_ends, n_ends, s.rec_local.p, s.block_tot.p, s.block_base.p, s.totals.p, d.s_compute));
                CK(cudaMemcpyAsync(s.h_totals.p, s.totals.p, 4 * sizeof(uint64_t), cudaMemcpyDeviceToHost, d.s_compute));
                CK(cudaStreamSynchronize(d.s_compute));
                for (int e = 0; e < n_ends; e++) (*X.sizes_out)[jk][e] += s.h_totals.p[e];
                st.kernel_launches += 3; st.pairs += np; st.batches++;
            }
            job_index++;
            continue;
        }
        // three batches in flight: batch b computes while b-1 crosses PCIe and b-2 is handed to the sink
        std::deque<Slot*> computing, copying;
        auto drain_one = [&]() {
            if (!copying.empty() && (computing.empty() || copying.size() >= 2)) { deliver(*copying.front()); copying.pop_front(); }
            else if (!computing.empty()) { issue_copy(*computing.front()); copying.push_back(computing.front()); computing.pop_front(); }
        };
        uint64_t bi = 0;
        for (uint64_t b0 = lo; b0 < hi; b0 += B, bi++) {
            Slot& s = d.slot[bi % 3];
            while (s.busy) drain_one();
            const uint32_t np = (uint32_t)std::min<uint64_t>(B, hi - b0);
            if (d.upload_pending && !use_haps) {
                // make the compute stream wait for exactly the uploads of the chromosomes this batch reads
                size_t g_lo, g_hi;
                groups_of(job, b0, b0 + np, g_lo, g_hi);
                g_hi = std::min(g_hi, d.chrom_ev.size() - 1);
                g_lo = std::min(g_lo, g_hi);
                if (b0 == lo) {
                    // first batch of this call's part of the job: a deferred upload copies, in the order the part
                    // will read them, all the chromosomes it reads and nothing else (with N GPUs each needs about
                    // 1/N of the genome); the rest stays on the host until some run asks for it
                    size_t g_end = (size_t)(std::upper_bound(group_off.begin(), group_off.end(), hi - 1) - group_off.begin()) - 1;
                    issue_upload(c, d, g_lo, std::min(g_end, d.chrom_ev.size() - 1));
                }
                issue_upload(c, d, g_lo, g_hi);
                for (size_t g = g_lo; g <= g_hi; g++)
                    if (!chrom_waited[g]) { CK(cudaStreamWaitEvent(d.s_compute, d.chrom_ev[g], 0)); chrom_waited[g] = 1; }
            }
            gp.job_lo = job.lo; gp.job_hi = job.hi; gp.batch_lo = b0; gp.batch_pairs = np;
            const uint32_t n_rec = np * n_ends;
            const uint32_t nsb = (np + kScanBlock - 1) / kScanBlock;
            gp.plan = s.plan.p; gp.rec_len = s.rec_len.p; gp.rec_local = s.rec_local.p; gp.block_base = s.block_base.p;
            gp.n_scan_blocks = nsb; gp.out[0] = s.out[0].p; gp.out[1] = s.out[1].p;
            CK(cudaEventRecord(s.ev[0], d.s_compute));
            CK(launch_place(gp, d.s_compute));
            CK(cudaEventRecord(s.ev[1], d.s_compute));
            CK(launch_scan(s.rec_len.p, n_rec, n_ends, s.rec_local.p, s.block_tot.p, s.block_base.p, s.totals.p,
                           d.s_compute));
            CK(cudaEventRecord(s.ev[2], d.s_compute));
            CK(launch_reads(gp, d.n_sm, d.s_compute));
            CK(cudaEventRecord(s.ev[3], d.s_compute));
            if (dev_z) {
                CK(s.z.launch(s.out[0].p, s.out[1].p, s.totals.p, nblk, P->compress, d.s_compute));
                st.kernel_launches += kBgzfLaunches;
            }
            CK(cudaMemcpyAsync(s.h_totals.p, s.totals.p, 4 * sizeof(uint64_t), cudaMemcpyDeviceToHost, d.s_compute));
            CK(cudaEventRecord(s.ev[5], d.s_compute));
            st.kernel_launches += 4;
            s.pairs = np; s.busy = true;
            computing.push_back(&s);
            // the previous batch's copy is queued before the one in flight is waited for
            if (computing.size() > 1) { issue_copy(*computing.front()); copying.push_back(computing.front()); computing.pop_front(); }
            if (copying.size() > 1) { deliver(*copying.front()); copying.pop_front(); }
            if (P->abort_cb && P->abort_cb(P->cb_user)) throw Aborted();   // Quiesce settles what is in flight
        }
        while (!computing.empty() || !copying.empty()) drain_one();
        for (Slot& s : d.slot) sink.settle(s.host);
        // a multi-GPU run appends the end-of-file block once, after joining the parts
        sink.end_job(job_index, n_ends, !X.shared_files && !X.job_suffix);
        job_index++;
    }
    CK(cudaEventRecord(d.ev_run[1], d.s_compute));
    CK(cudaEventSynchronize(d.ev_run[1]));
    {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, d.ev_run[0], d.ev_run[1]));
        st.run_ms = ms;
    }
    if (d.upload_pending) {
        // the copies this run issued are done before the caller gets control back; chromosomes no
        // shard of this run touched remain on the host (upload_src must stay valid, see the header)
        CK(cudaStreamSynchronize(d.s_upload));
        if (std::find(d.chrom_resident.begin(), d.chrom_resident.end(), 0) == d.chrom_resident.end()) {
            d.upload_pending = false;
            d.upload_src = nullptr;
        }
    }
    uint32_t status = 0;
    CK(cudaMemcpy(&status, d.d_status.p, sizeof status, cudaMemcpyDeviceToHost));
    if (status & 1u) throw ArgErr("a barcode is at least as long as a read's template (fragment or chromosome too short)");
    st.h2d_bytes = d.h2d_bytes - h2d_before;      // of this call (a deferred genome upload it performed included)
    if (stats) *stats = st;
    quiesce.armed = false;
}

// ------------------------------------------------- one call, several GPUs ---
//
// The reference splits a run over its threads and keeps ONE ordered set of files inside one call
// (write_reads_one_filetype_, src/hts.h:334-353 split, :401-416 both pools written together;
// write_reads_cpp_sep_files_, :512-552).  A multi-GPU context does the same over devices: the run's pair-index
// space [0, n_pairs) is cut into near-equal contiguous pieces, one per device (a piece may cover several
// haplotypes' jobs with sep_files, and a job may have several writers); every device runs the three-stage batch
// pipeline of run() on its piece from its own host thread.  No data moves between the devices (no collective):
//   plain FASTQ   a size pass (placement + scan only, a few hundred microseconds per batch) tells every device how
//                 many bytes it will write per job and file, so the devices write into disjoint ranges of the
//                 same, pre-sized R1 / R2 files (or of the caller's memory buffers) -- R1 and R2 stay aligned;
//   compressed    by the device coder: the devices first generate and compress their pieces without delivering them
//                 (a dry run: they are some fifty times faster than any sink), which gives every piece's compressed
//                 size; then the files are pre-sized and every device writes its BGZF members straight to their
//                 final place.  By zlib on the host (levels 7-9): the job's first device writes the file, device r
//                 writes <file>.part<r>, the parts are moved in behind it and the EOF block is appended once.
// Only the haplotype chromosomes a device's piece touches are materialised there (ensure_hap_chrom).
// Callbacks run on the calling thread only (R is single-threaded): the device threads count progress in an atomic
// and poll an abort flag; the calling thread polls both while it waits.

struct MultiShared {
    std::atomic<uint64_t> progress{0};
    std::atomic<int> abort{0};
};
int multi_abort_cb(void* u) { return static_cast<MultiShared*>(u)->abort.load(std::memory_order_relaxed); }
void multi_progress_cb(void* u, uint64_t reads) { static_cast<MultiShared*>(u)->progress.fetch_add(reads, std::memory_order_relaxed); }

void run_multi(jlp_ctx* c, bool use_haps, const jlp_illumina_params* P, Output& sink, jlp_run_stats* stats) {
    if (sink.kind == SINK_STREAM)
        throw Unsupported("jlp_illumina_stream on a multi-GPU context: batches of several devices have no single order; "
                          "use files / memory, or one context per device with shard_index / shard_count");
    if (P->shard_count > 1) throw ArgErr("shard_index / shard_count do not combine with a multi-GPU context");
    const size_t N = c->dev.size();
    const Layout Y = make_layout(c, illumina_spec(c, use_haps, P));
    const size_t nj = Y.jobs.size();
    const int n_ends = P->paired || P->matepair ? 2 : 1;
    const Compression Z = compression_of(P, sink.kind);
    if (Z.want_gz && Z.dev_z && sink.kind == SINK_MEMORY)
        throw Unsupported("compressed output into memory on a multi-GPU context");
    const bool sized = sink.kind == SINK_MEMORY || (sink.kind == SINK_FILES && !Z.want_gz);   // plain bytes at known offsets
    // compressed by the device coder: the sizes come from a dry run (the devices generate and compress everything once
    // without delivering it -- they are some fifty times faster than any sink), then every device writes its members
    // straight to their final place; compressed by zlib on the host: part files, joined afterwards
    const bool zsized = sink.kind == SINK_FILES && Z.want_gz && Z.dev_z;
    const bool parts = sink.kind == SINK_FILES && Z.want_gz && !Z.dev_z;

    // --- the devices' pieces of the pair-index space, per job
    std::vector<Ranges> ranges(N, Ranges(nj));
    for (size_t r = 0; r < N; r++) {
        uint64_t glo, ghi;
        shard_range(0, Y.n_pairs, (uint32_t)r, (uint32_t)N, glo, ghi);
        for (size_t k = 0; k < nj; k++) {
            const uint64_t lo = std::min(std::max(glo, Y.jobs[k].lo), Y.jobs[k].hi), hi = std::min(std::max(ghi, Y.jobs[k].lo), Y.jobs[k].hi);
            ranges[r][k] = {lo, std::max(lo, hi)};
        }
    }

    MultiShared shared;
    jlp_illumina_params Pk = *P;
    Pk.shard_index = 0; Pk.shard_count = 0;
    Pk.abort_cb = multi_abort_cb; Pk.progress_cb = multi_progress_cb; Pk.cb_user = &shared;
    Pk.n_threads = P->n_threads <= 1 ? 1 : std::max<uint64_t>(2, (P->n_threads + N - 1) / N);   // host writer threads per device

    std::vector<jlp_run_stats> st(N);
    auto serve_callbacks = [&]() {
        const uint64_t n = shared.progress.exchange(0);
        if (n && P->progress_cb) P->progress_cb(P->cb_user, n);
        if (P->abort_cb && !shared.abort.load() && P->abort_cb(P->cb_user)) shared.abort.store(2);
    };
    // run f(d, r) for every device d (the r-th); the calling thread serves the callbacks meanwhile
    auto on_devices = [&](const std::function<void(Device&, size_t)>& f, bool with_callbacks) {
        on_each_device(c, [&](Device& d) {
            size_t r = 0;
            while (c->dev[r].get() != &d) r++;
            try {
                f(d, r);
            } catch (...) {                   // the others stop at their next batch
                int none = 0;
                shared.abort.compare_exchange_strong(none, 1);
                throw;
            }
        }, with_callbacks ? std::function<void()>(serve_callbacks) : nullptr);
        const uint64_t n = shared.progress.exchange(0);
        if (n && P->progress_cb && with_callbacks) P->progress_cb(P->cb_user, n);
        if (shared.abort.load() == 2) throw Aborted();
    };

    // a shared output file is created with its final size at once (no pages yet; pages are reserved slice by slice by the
    // devices' writer threads, see Output::deliver), its last `tail` bytes written now; a file system that cannot hold
    // everything the run will write is reported here rather than half-way through
    uint64_t need_bytes = 0;
    auto create_sized = [&](const std::string& name, uint64_t size, const uint8_t* tail, uint64_t tail_len) {
        const int fd = ::open(name.c_str(), O_RDWR | O_CREAT | O_TRUNC, 0644);
        if (fd < 0) throw IoErr("Unable to open file " + name + ".\n");      // src/io.h:288-290
        need_bytes += size;
        struct statvfs vfs;
        const int rc = ::fstatvfs(fd, &vfs) == 0 && (uint64_t)vfs.f_bavail * vfs.f_frsize < need_bytes ? ENOSPC
                       : ::ftruncate(fd, (off_t)size) == 0 ? 0 : errno;
        const std::string w = rc ? std::strerror(rc) : pwrite_all(fd, tail, tail_len, size - tail_len);
        ::close(fd);
        if (!w.empty()) throw IoErr("Error writing to file " + name + ": " + w);
    };

    // --- size pass
    std::vector<PerJobBytes> sizes(N), base(N, PerJobBytes(nj, std::array<uint64_t, 2>{0, 0}));
    std::vector<std::array<uint64_t, 2>> job_total(nj, std::array<uint64_t, 2>{0, 0});
    uint64_t launches = 0;
    if (sized) {
        on_devices([&](Device& d, size_t r) {
            Output none;
            RunExtras X;
            X.ranges = &ranges[r]; X.sizes_out = &sizes[r];
            run(c, d, use_haps, &Pk, Y, none, &st[r], X);
        }, false);
        uint64_t mem_off[2] = {0, 0};
        for (size_t k = 0; k < nj; k++)
            for (int e = 0; e < n_ends; e++) {
                uint64_t o = sink.kind == SINK_MEMORY ? mem_off[e] : 0;      // memory: the jobs' outputs are concatenated
                for (size_t r = 0; r < N; r++) { base[r][k][e] = o; o += sizes[r][k][e]; }
                job_total[k][e] = o - (sink.kind == SINK_MEMORY ? mem_off[e] : 0);
                mem_off[e] += job_total[k][e];
            }
        for (size_t r = 0; r < N; r++) launches += st[r].kernel_launches;
        if (sink.kind == SINK_FILES)
            for (size_t k = 0; k < nj; k++)
                for (int e = 0; e < n_ends; e++) create_sized(file_name(Y.jobs[k], e, false, P), job_total[k][e], nullptr, 0);
        if (sink.kind == SINK_MEMORY) { sink.len[0] = mem_off[0]; sink.len[1] = mem_off[1]; }
    }

    // --- compressed size pass (device coder)
    std::vector<PerJobBytes> zsizes(N), zcheck(N);
    if (zsized) {
        jlp_illumina_params Pdry = Pk;
        Pdry.progress_cb = nullptr;
        on_devices([&](Device& d, size_t r) {
            Output none;
            RunExtras X;
            X.ranges = &ranges[r]; X.zsizes_out = &zsizes[r]; X.dry_files = true;
            run(c, d, use_haps, &Pdry, Y, none, &st[r], X);
        }, true);
        for (size_t r = 0; r < N; r++) launches += st[r].kernel_launches;
        for (size_t k = 0; k < nj; k++)
            for (int e = 0; e < n_ends; e++) {
                uint64_t o = 0;
                for (size_t r = 0; r < N; r++) { base[r][k][e] = o; o += zsizes[r][k][e]; }
                job_total[k][e] = o;
                // bgzf_close: one empty block ends the file
                create_sized(file_name(Y.jobs[k], e, true, P), o + sizeof kBgzfEof, kBgzfEof, sizeof kBgzfEof);
            }
    }

    // --- the run proper
    struct Cleanup {       // part files never outlive the call
        std::vector<std::string> names;
        ~Cleanup() { for (const std::string& n : names) ::unlink(n.c_str()); }
    } cleanup;
    // compressed: for every job the first device with a part in it writes the file itself, the others write parts
    std::vector<size_t> first_dev(nj, N);
    for (size_t k = 0; k < nj; k++)
        for (size_t r = N; r-- > 0;) if (ranges[r][k].second > ranges[r][k].first) first_dev[k] = r;
    if (parts)
        for (size_t r = 0; r < N; r++)
            for (size_t k = 0; k < nj; k++)
                if (ranges[r][k].second > ranges[r][k].first && r != first_dev[k])
                    for (int e = 0; e < n_ends; e++) cleanup.names.push_back(file_name(Y.jobs[k], e, true, P) + ".part" + std::to_string(r));
    on_devices([&](Device& d, size_t r) {
        Output sk(sink.kind);
        for (int e = 0; e < 2; e++) { sk.mem[e] = sink.mem[e]; sk.cap[e] = sink.cap[e]; }
        RunExtras X;
        X.ranges = &ranges[r];
        if (sized) { X.base = &base[r]; X.shared_files = sink.kind == SINK_FILES; }
        if (zsized) { X.base = &base[r]; X.shared_files = true; X.zsizes_out = &zcheck[r]; }
        std::vector<std::string> suffix;
        if (parts) {
            // per job: the job's first device writes <name> itself (no EOF block yet), every other one <name>.part<r>
            X.job_suffix = &suffix;
            for (size_t k = 0; k < nj; k++) suffix.push_back(r == first_dev[k] ? std::string() : ".part" + std::to_string(r));
        }
        run(c, d, use_haps, &Pk, Y, sk, &st[r], X);
    }, true);

    if (zsized)         // the coder is deterministic; a difference between the two passes would have put members in the wrong place
        for (size_t r = 0; r < N; r++)
            if (zcheck[r] != zsizes[r]) throw std::runtime_error("internal: compressed sizes differ between the size pass and the run");

    // --- compressed: the parts move behind the first device's bytes in device order (their offsets are known now),
    //     slices of them copied by several threads at once; one end-of-file block per file
    if (parts) {
        struct CopyTask { int in_fd, out_fd; uint64_t in_off, out_off, len; };
        std::vector<CopyTask> tasks;
        std::vector<int> fds;
        struct CloseAll { std::vector<int>& f; ~CloseAll() { for (int x : f) ::close(x); } } close_all{fds};
        const bool eof = Z.dev_z || Z.zmethod == DEFLATE_BGZF;
        for (size_t k = 0; k < nj; k++)
            for (int e = 0; e < n_ends; e++) {
                const std::string name = file_name(Y.jobs[k], e, true, P);
                const int fd = ::open(name.c_str(), first_dev[k] < N ? O_RDWR : (O_RDWR | O_CREAT | O_TRUNC), 0644);
                if (fd < 0) throw IoErr("Unable to open file " + name + ".\n");
                fds.push_back(fd);
                struct stat sb;
                if (::fstat(fd, &sb) != 0) throw IoErr("Error writing to file " + name + ": " + std::strerror(errno));
                uint64_t pos = (uint64_t)sb.st_size;
                for (size_t r = 0; r < N; r++) {
                    if (ranges[r][k].second <= ranges[r][k].first || r == first_dev[k]) continue;
                    const std::string part = name + ".part" + std::to_string(r);
                    const int in = ::open(part.c_str(), O_RDONLY);
                    if (in < 0 || ::fstat(in, &sb) != 0) { if (in >= 0) ::close(in); throw IoErr("cannot read " + part); }
                    fds.push_back(in);
                    const uint64_t slice = 64ull << 20;
                    for (uint64_t o = 0; o < (uint64_t)sb.st_size; o += slice)
                        tasks.push_back(CopyTask{in, fd, o, pos + o, std::min<uint64_t>(slice, (uint64_t)sb.st_size - o)});
                    pos += (uint64_t)sb.st_size;
                }
                if (::ftruncate(fd, (off_t)(pos + (eof ? sizeof kBgzfEof : 0))) != 0)
                    throw IoErr("Error writing to file " + name + ": " + std::strerror(errno));
                if (eof) {
                    const std::string w = pwrite_all(fd, kBgzfEof, sizeof kBgzfEof, pos);
                    if (!w.empty()) throw IoErr("Error writing to file " + name + ": " + w);
                }
            }
        // a slice is copied through mappings of both files where that works (threads writing one file through
        // write() / copy_file_range queue on its inode lock; page-cache pages filled through a mapping do not), else by
        // copy_range; the writer threads of the first device do the copying
        WriterPool& writers = c->dev[0]->writers;
        std::atomic<int> pending{0};
        writers.start(std::min<size_t>(std::max<size_t>(tasks.size(), 1), std::min<uint64_t>(std::max<uint64_t>(P->n_threads, 4), 32)));
        for (const CopyTask& t : tasks)
            writers.submit(&pending, [t]() {
                Mapping mo, mi;
                std::string w;
                if (map_range(t.out_fd, t.out_off, t.len, mo) && map_range(t.in_fd, t.in_off, t.len, mi, true))
                    std::memcpy(mo.at, mi.at, t.len);
                else
                    w = copy_range(t.out_fd, t.out_off, t.in_fd, t.in_off, t.len);
                mi.unmap();
                mo.unmap();
                return w;
            });
        const std::string w = writers.wait(pending);
        if (!w.empty()) { writers.clear_error(); throw IoErr("Error joining the devices' parts: " + w); }
    }

    jlp_run_stats tot;
    std::memset(&tot, 0, sizeof tot);
    for (size_t r = 0; r < N; r++) {
        tot.pairs += st[r].pairs; tot.batches += st[r].batches; tot.kernel_launches += st[r].kernel_launches;
        for (int e = 0; e < 2; e++) { tot.bytes_out[e] += st[r].bytes_out[e]; tot.z_bytes[e] += st[r].z_bytes[e]; }
        tot.d2h_bytes += st[r].d2h_bytes; tot.h2d_bytes += st[r].h2d_bytes;
        // device time: the slowest device's (they work side by side)
        tot.device_ms = std::max(tot.device_ms, st[r].device_ms); tot.place_ms = std::max(tot.place_ms, st[r].place_ms);
        tot.reads_ms = std::max(tot.reads_ms, st[r].reads_ms); tot.bgzf_ms = std::max(tot.bgzf_ms, st[r].bgzf_ms);
        tot.run_ms = std::max(tot.run_ms, st[r].run_ms);
    }
    tot.kernel_launches += launches;
    if (stats) *stats = tot;
}

}  // namespace

// ------------------------------------------------------------------ C ABI ---

extern "C" {

// A context over devices[0..n_devices) (NULL: devices 0..n_devices-1; n_devices == 0: every visible device).
static int create_ctx(int n_devices, const int* devices, jlp_ctx** out) {
    if (!out) return fail(nullptr, JLP_ERR_ARG, "out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(nullptr, JLP_ERR_NO_DEVICE,
                    std::string("no CUDA device available (") + cudaGetErrorString(e) +
                        "); this library has no CPU fallback");
    if (n_devices < 0 || n_devices > 64) return fail(nullptr, JLP_ERR_ARG, "n_devices must be 0 (all visible devices) .. 64");
    if (n_devices == 0) { n_devices = n; devices = nullptr; }
    std::unique_ptr<jlp_ctx> c(new jlp_ctx);
    int rc = guarded(c.get(), [&]() {
        for (int i = 0; i < n_devices; i++) {
            const int id = devices ? devices[i] : i;
            if (id < 0 || id >= n) throw ArgErr("device index out of range");
            c->dev.emplace_back(new Device);
            Device& d = *c->dev.back();
            d.id = id;
            CK(cudaSetDevice(id));
            CK(cudaDeviceGetAttribute(&d.n_sm, cudaDevAttrMultiProcessorCount, id));
            CK(cudaStreamCreateWithFlags(&d.s_compute, cudaStreamNonBlocking));
            CK(cudaStreamCreateWithFlags(&d.s_copy, cudaStreamNonBlocking));
            CK(cudaStreamCreateWithFlags(&d.s_upload, cudaStreamNonBlocking));
            for (Slot& s : d.slot) for (cudaEvent_t& ev : s.ev) CK(cudaEventCreate(&ev));
            for (cudaEvent_t& ev : d.ev_run) CK(cudaEventCreate(&ev));
            for (int k = 0; k < Device::kMatBufs; k++) {
                CK(cudaEventCreateWithFlags(&d.m_up[k], cudaEventDisableTiming));
                CK(cudaEventCreateWithFlags(&d.m_done[k], cudaEventDisableTiming));
            }
            CK(bgzf_init());
        }
    });
    if (rc != JLP_OK) { g_create_error = c->err; return rc; }
    *out = c.release();
    return JLP_OK;
}

int jlp_ctx_create(int device, jlp_ctx** out) { return create_ctx(1, &device, out); }

int jlp_ctx_create_multi(int n_devices, const int* devices, jlp_ctx** out) { return create_ctx(n_devices, devices, out); }

int jlp_ctx_n_devices(const jlp_ctx* c) { return c ? (int)c->dev.size() : 0; }

void jlp_ctx_destroy(jlp_ctx* c) { delete c; }

const char* jlp_last_error(const jlp_ctx* c) { return c ? c->err.c_str() : g_create_error.c_str(); }

static int set_genome_impl(jlp_ctx* c, const char* bases, const uint64_t* chrom_off, uint64_t n_chroms,
                           const char* const* chrom_names, const char* genome_name, bool wait) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        if (!bases || !chrom_off || !chrom_names || n_chroms == 0) throw ArgErr("empty genome");
        for (uint64_t i = 0; i < n_chroms; i++)
            if (chrom_off[i + 1] < chrom_off[i]) throw ArgErr("chrom_off must be non-decreasing");
        if (chrom_off[0] != 0) throw ArgErr("chrom_off[0] must be 0");
        std::vector<std::string> names;
        for (uint64_t i = 0; i < n_chroms; i++) names.push_back(chrom_names[i] ? chrom_names[i] : "");
        // one copy and one event per chromosome: generation starts as soon as the chromosomes a batch
        // reads are resident, the rest of the genome follows underneath (PCIe is full duplex, the
        // FASTQ flows the other way).  The asynchronous form defers the copies to the next run, which
        // starts them at the first chromosome its shard reads (with several devices: each device's piece).
        replace_genome(c, std::vector<uint64_t>(chrom_off, chrom_off + n_chroms + 1), names, genome_name, [&](Device& d) {
            while (d.chrom_ev.size() < n_chroms) {
                cudaEvent_t ev;
                CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
                d.chrom_ev.push_back(ev);
            }
            d.upload_src = bases;
            d.upload_pending = true;
            d.chrom_resident.assign(n_chroms, 0);
            if (wait) finish_upload(c, d);
        });
    });
}

int jlp_set_genome(jlp_ctx* c, const char* bases, const uint64_t* chrom_off, uint64_t n_chroms,
                   const char* const* chrom_names, const char* genome_name) {
    return set_genome_impl(c, bases, chrom_off, n_chroms, chrom_names, genome_name, true);
}

int jlp_set_genome_async(jlp_ctx* c, const char* bases, const uint64_t* chrom_off, uint64_t n_chroms,
                         const char* const* chrom_names, const char* genome_name) {
    return set_genome_impl(c, bases, chrom_off, n_chroms, chrom_names, genome_name, false);
}

int jlp_genome_sync(jlp_ctx* c) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() { on_each_device(c, [&](Device& d) { finish_upload(c, d); }); });
}

int jlp_create_genome(jlp_ctx* c, uint64_t n_chroms, const uint64_t* lens, const double* pi_tcag, uint64_t seed,
                      const char* const* chrom_names, const char* genome_name) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        if (!lens || !pi_tcag || n_chroms == 0) throw ArgErr("empty genome");
        double tot = 0;
        for (int k = 0; k < 4; k++) { if (!(pi_tcag[k] >= 0)) throw ArgErr("pi_tcag must be >= 0"); tot += pi_tcag[k]; }
        if (!(tot > 0)) throw ArgErr("pi_tcag must have at least one value > 0");
        std::vector<uint64_t> off(1, 0);
        std::vector<std::string> names;
        for (uint64_t i = 0; i < n_chroms; i++) {
            if (lens[i] == 0) throw ArgErr("chromosome lengths must be >= 1");       // "never returns empty chromosomes"
            off.push_back(off.back() + lens[i]);
            names.push_back(chrom_names && chrom_names[i] ? chrom_names[i] : "chrom" + std::to_string(i));   // src/create_sequences.cpp:178-181
        }
        // AliasSampler(pi_tcag), src/alias_sampler.h:68-106
        double Prob[4];
        uint64_t Alias[4];
        alias_build(pi_tcag, 4, Prob, Alias);
        GenomeTables t;
        for (int k = 0; k < 4; k++) {
            Thr th = thr_double_lt(Prob[k]);
            t.thr[k] = th.thr; t.thr16[k] = (uint32_t)(th.thr >> 48); t.alias[k] = (uint32_t)Alias[k];
        }
        // the same seed gives every device the same genome: generated in place everywhere, nothing copied
        replace_genome(c, off, names, genome_name, [&](Device& d) {
            d.chrom_resident.assign(n_chroms, 1);
            for (uint64_t i = 0; i < n_chroms; i++)
                CK(launch_create_chrom(d.genome.p + kPad + off[i], lens[i], (uint32_t)i, seed, t, d.s_compute));
            CK(cudaStreamSynchronize(d.s_compute));
        });
    });
}

int jlp_get_genome(jlp_ctx* c, char* out, uint64_t cap, uint64_t* len) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        if (c->chrom_off.size() < 2) throw ArgErr("no reference genome has been set");
        Device& d = device0(c);
        finish_upload(c, d);
        const uint64_t n = c->chrom_off.back();
        if (len) *len = n;
        if (!out) return;
        if (n > cap) throw ArgErr("output buffer too small");
        CK(cudaMemcpy(out, d.genome.p + kPad, n, cudaMemcpyDeviceToHost));
    });
}

int jlp_clear_haplotypes(jlp_ctx* c) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() { clear_haps(c); });
}

// the host-side store of one haplotype: a copy of the caller's AllMutations arrays + size_modifier per record, one packed
// array per chromosome, built by a few threads (one chromosome at a time each)
static std::shared_ptr<HapStore> make_hap_store(const jlp_ctx* c, const char* name, const uint64_t* n_muts, const uint64_t* const* old_pos,
                                                const uint64_t* const* new_pos, const uint64_t* const* nuc_off,
                                                const char* const* nuc_pool, const uint64_t* nuc_pool_len, const uint64_t* chrom_sizes) {
    if (c->chrom_off.size() < 2) throw ArgErr("set the reference genome first");
    if (!n_muts || !chrom_sizes) throw ArgErr("n_muts / chrom_sizes is NULL");
    const uint64_t nc = c->chrom_off.size() - 1;
    auto S = std::make_shared<HapStore>();
    S->name = name ? name : "";
    S->chrom.resize(nc);
    uint64_t total = 0;
    for (uint64_t ci = 0; ci < nc; ci++) total += n_muts[ci];
    const unsigned nt = total < (1u << 16) ? 1u : (unsigned)std::min<uint64_t>(std::min<uint64_t>(nc, 16), std::max(1u, std::thread::hardware_concurrency()));
    parallel_for(nc, nt, [&](uint64_t ci) {
        const uint64_t M = n_muts[ci];
        const uint64_t ref_size = c->chrom_off[ci + 1] - c->chrom_off[ci];
        HapChromHost& H = S->chrom[ci];
        H.size = chrom_sizes[ci];
        if (M == 0) {   // get_chrom_full returns the reference string (src/hap_classes.cpp:82)
            if (chrom_sizes[ci] != ref_size) throw ArgErr("chromosome without mutations must keep the reference size");
            return;
        }
        if (!old_pos || !new_pos || !nuc_off || !nuc_pool || !nuc_pool_len || !old_pos[ci] || !new_pos[ci] || !nuc_off[ci])
            throw ArgErr("mutation arrays are NULL");
        const uint64_t pb = nuc_pool_len[ci];
        H.n_muts = M; H.pool_bytes = pb;
        H.packed.resize(4 * M + (pb + 7) / 8);
        uint64_t* w = H.packed.data();
        std::memcpy(w, old_pos[ci], M * 8);
        std::memcpy(w + M, new_pos[ci], M * 8);
        std::memcpy(w + 2 * M, nuc_off[ci], M * 8);
        // size_modifier per record, src/hap_classes.h:314-333
        int64_t* sm = reinterpret_cast<int64_t*>(w + 3 * M);
        for (uint64_t i = 0; i < M; i++) {
            if (i && new_pos[ci][i] < new_pos[ci][i - 1]) throw ArgErr("mutations must be sorted by new_pos");
            const int64_t s = (i + 1 < M) ? (int64_t)(new_pos[ci][i + 1] - old_pos[ci][i + 1]) : (int64_t)(chrom_sizes[ci] - ref_size);
            sm[i] = s + (int64_t)(old_pos[ci][i] - new_pos[ci][i]);
        }
        if (pb) std::memcpy(w + 4 * M, nuc_pool[ci], pb);
    });
    return S;
}

// attach a haplotype to a context: unmutated chromosomes alias the reference, the others wait for a run to touch them
static void attach_hap(jlp_ctx* c, const std::shared_ptr<HapStore>& S) {
    c->haps.push_back(S);
    for (auto& d : c->dev) {
        std::vector<const uint8_t*> seq;
        for (size_t ci = 0; ci < S->chrom.size(); ci++)
            seq.push_back(S->chrom[ci].n_muts == 0 ? d->genome.p + kPad + c->chrom_off[ci] : nullptr);
        d->hap_seq.push_back(std::move(seq));
    }
}

int jlp_add_haplotype(jlp_ctx* c, const char* name, const uint64_t* n_muts, const uint64_t* const* old_pos,
                      const uint64_t* const* new_pos, const uint64_t* const* nuc_off,
                      const char* const* nuc_pool, const uint64_t* nuc_pool_len,
                      const uint64_t* chrom_sizes, uint64_t* hap_index) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        std::shared_ptr<HapStore> S = make_hap_store(c, name, n_muts, old_pos, new_pos, nuc_off, nuc_pool, nuc_pool_len, chrom_sizes);
        if (hap_index) *hap_index = c->haps.size();
        attach_hap(c, S);
    });
}

int jlp_materialize_haplotypes(jlp_ctx* c) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        on_each_device(c, [&](Device& d) {
            finish_upload(c, d);
            for (size_t h = 0; h < d.hap_seq.size(); h++)
                for (size_t ci = 0; ci < d.hap_seq[h].size(); ci++) ensure_hap_chrom(c, d, h, ci);
            CK(cudaStreamSynchronize(d.s_compute));
        });
    });
}

int jlp_get_haplotype_chrom(jlp_ctx* c, uint64_t hap, uint64_t chrom, char* out, uint64_t cap, uint64_t* len) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        if (hap >= c->haps.size() || chrom >= c->haps[hap]->chrom.size()) throw ArgErr("haplotype / chromosome index out of range");
        uint64_t n = c->haps[hap]->chrom[chrom].size;
        if (len) *len = n;
        if (n > cap) throw ArgErr("output buffer too small");
        Device& d = device0(c);
        finish_upload(c, d);
        ensure_hap_chrom(c, d, hap, chrom);
        CK(cudaStreamSynchronize(d.s_compute));
        if (n) CK(cudaMemcpy(out, d.hap_seq[hap][chrom], n, cudaMemcpyDeviceToHost));
    });
}

int jlp_get_haplotype_muts(jlp_ctx* c, uint64_t hap, uint64_t chrom, uint64_t* old_pos, uint64_t* new_pos,
                           uint64_t* nuc_off, char* pool, uint64_t cap_muts, uint64_t cap_pool, uint64_t* n_muts,
                           uint64_t* pool_len, uint64_t* chrom_size) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        if (hap >= c->haps.size() || chrom >= c->haps[hap]->chrom.size()) throw ArgErr("haplotype / chromosome index out of range");
        const HapChromHost& H = c->haps[hap]->chrom[chrom];
        const uint64_t M = H.n_muts;
        if (n_muts) *n_muts = M;
        if (pool_len) *pool_len = H.pool_bytes;
        if (chrom_size) *chrom_size = H.size;
        if (!old_pos) return;
        if (M > cap_muts || H.pool_bytes > cap_pool) throw ArgErr("output arrays too small");
        if (M && (!new_pos || !nuc_off)) throw ArgErr("new_pos / nuc_off is NULL");
        if (H.pool_bytes && !pool) throw ArgErr("pool is NULL");
        const uint64_t* w = H.packed.data();
        if (M) {
            std::memcpy(old_pos, w, M * 8);
            std::memcpy(new_pos, w + M, M * 8);
            std::memcpy(nuc_off, w + 2 * M, M * 8);
        }
        if (H.pool_bytes) std::memcpy(pool, w + 4 * M, H.pool_bytes);
    });
}

// ---------------------------------------------------------------- create_haplotypes ---

namespace {

// The visiting order of one tree and the node-state slots (k_mutate): preorder with the child of fewer tips first, a
// parent's slot freed when its last child is visited (before that child takes one), so at most about log2(tips) + 2
// slots are live.  Childless nodes that are not tips are left out.  tab: the node's first row after the tree's.
std::vector<MutNode> mut_schedule(const GeneTree& T, uint32_t n_cat, uint32_t& max_slots) {
    const uint32_t n = (uint32_t)T.parent.size();
    std::vector<int32_t> tip_of(n, -1);
    for (uint32_t t = 0; t < T.tip_node.size(); t++) tip_of[T.tip_node[t]] = (int32_t)t;
    std::vector<std::vector<uint32_t>> kids(n);
    for (uint32_t i = 1; i < n; i++) kids[T.parent[i]].push_back(i);
    std::vector<uint64_t> tips(n, 0);
    for (uint32_t i = n; i-- > 0;) {
        if (kids[i].empty()) tips[i] = tip_of[i] >= 0 ? 1 : 0;
        if (i) tips[T.parent[i]] += tips[i];
    }
    for (auto& k : kids) std::stable_sort(k.begin(), k.end(), [&](uint32_t a, uint32_t b) { return tips[a] < tips[b]; });
    std::vector<uint32_t> left(n), slot(n, 0), free_slots;
    for (uint32_t i = 0; i < n; i++) left[i] = (uint32_t)kids[i].size();
    for (uint32_t s = kMutSlots; s-- > 1;) free_slots.push_back((uint32_t)s);
    max_slots = 1;
    std::vector<MutNode> out;
    std::vector<uint32_t> stack(kids[0].rbegin(), kids[0].rend());
    while (!stack.empty()) {
        const uint32_t v = stack.back();
        stack.pop_back();
        const uint32_t par = (uint32_t)T.parent[v];
        MutNode m;
        m.node = v;
        m.tab = v * n_cat * 4;
        m.tip = tip_of[v];
        m.pslot = (uint16_t)slot[par];
        m.slot = 0;
        if (--left[par] == 0) free_slots.push_back(slot[par]);
        if (!kids[v].empty()) {
            if (free_slots.empty()) throw ArgErr("tree too deep for the node-state slots");
            slot[v] = free_slots.back();
            free_slots.pop_back();
            m.slot = (uint16_t)slot[v];
            max_slots = std::max<uint32_t>(max_slots, kMutSlots - (uint32_t)free_slots.size());
            for (auto it = kids[v].rbegin(); it != kids[v].rend(); ++it) stack.push_back(*it);
        }
        if (!kids[v].empty() || m.tip >= 0) out.push_back(m);
    }
    return out;
}

struct EventSet {
    cudaEvent_t e[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    EventSet() { for (cudaEvent_t& x : e) CK(cudaEventCreate(&x)); }
    ~EventSet() { for (cudaEvent_t x : e) if (x) cudaEventDestroy(x); }
    float ms(int a, int b) const { float t = 0; cudaEventElapsedTime(&t, e[a], e[b]); return t; }
};

constexpr uint64_t kTableBudget = 1ull << 30;       // default bytes of threshold tables per window

// Device buffers of the threshold tables: the items of a window, the flagged items, the tables.
struct TableBufs {
    DevBuf<TabItem> items;
    DevBuf<uint32_t> flag;
    std::vector<uint32_t> h_flag;
    std::vector<uint4> h_rows;
};

// The tables of `items` built on the device (k_mut_tables); the items it flags are recomputed here with the host's
// transition_matrix + row_thresholds and copied over theirs (and over P_out's, when given).  Returns their count.
uint64_t device_tables(cudaStream_t s, const double Q[16], const std::vector<TabItem>& items, TableBufs& B, uint4* hi,
                       uint4* lo, double* P_out) {
    if (items.empty()) return 0;
    if (items.size() >> 32) throw ArgErr("2^32 or more transition matrices in one window");
    TabQ q;
    std::memcpy(q.q, Q, sizeof q.q);
    B.items.upload(items, s);
    B.flag.ensure(items.size() + 1);
    CK(cudaMemsetAsync(B.flag.p, 0, 4, s));
    CK(launch_mut_tables(B.items.p, (uint32_t)items.size(), q, hi, lo, P_out, B.flag.p, B.flag.p + 1, s));
    uint32_t nf = 0;
    CK(cudaMemcpyAsync(&nf, B.flag.p, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (nf == 0) return 0;
    B.h_flag.resize(nf);
    CK(cudaMemcpyAsync(B.h_flag.data(), B.flag.p + 1, (size_t)nf * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    B.h_rows.resize((size_t)nf * 8);
    std::vector<double> Ps(P_out ? (size_t)nf * 16 : 0);
    for (uint32_t f = 0; f < nf; f++) {
        const TabItem& it = items[B.h_flag[f]];
        double P[16];
        transition_matrix(Q, it.t, P);
        if (P_out) std::memcpy(&Ps[16 * (size_t)f], P, sizeof P);
        for (uint32_t a = 0; a < 4; a++) {
            uint64_t t[3];
            row_thresholds(P + 4 * a, t);
            B.h_rows[8 * (size_t)f + a] = make_uint4((uint32_t)(t[0] >> 32), (uint32_t)(t[1] >> 32), (uint32_t)(t[2] >> 32), 0);
            B.h_rows[8 * (size_t)f + 4 + a] = make_uint4((uint32_t)t[0], (uint32_t)t[1], (uint32_t)t[2], 0);
        }
        CK(cudaMemcpyAsync(hi + it.row, &B.h_rows[8 * (size_t)f], 4 * sizeof(uint4), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(lo + it.row, &B.h_rows[8 * (size_t)f + 4], 4 * sizeof(uint4), cudaMemcpyHostToDevice, s));
        if (P_out)
            CK(cudaMemcpyAsync(P_out + 16 * (size_t)B.h_flag[f], &Ps[16 * (size_t)f], 16 * sizeof(double),
                               cudaMemcpyHostToDevice, s));
    }
    CK(cudaStreamSynchronize(s));
    return nf;
}

void check_model(const jlp_ctx* c, const jlp_mutation_params* p) {
    if (c->chrom_off.size() < 2) throw ArgErr("set the reference genome first");
    for (int i = 0; i < 16; i++)
        if (i % 5 && !(std::isfinite(p->Q[i]) && p->Q[i] >= 0)) throw ArgErr("the off-diagonal rates of Q must be finite and >= 0");
    if (!(p->invariant >= 0 && p->invariant < 1)) throw ArgErr("invariant must be >= 0 and < 1");
    if (p->n_rates < 1 || p->n_rates > 255 || !p->rates) throw ArgErr("n_rates must be 1..255 (rates not NULL)");
    for (uint32_t k = 0; k < p->n_rates; k++)
        if (!(std::isfinite(p->rates[k]) && p->rates[k] >= 0)) throw ArgErr("category rates must be finite and >= 0");
    if (p->n_tips < 1 || p->n_tips > kMutMaxTips)
        throw ArgErr("a tree of " + std::to_string(p->n_tips) + " tips: 1 to " + std::to_string(kMutMaxTips) + " tips are supported");
    if (!p->tip_names) throw ArgErr("tip_node / tip_names is NULL");
    for (uint32_t t = 0; t < p->n_tips; t++)
        if (!p->tip_names[t]) throw ArgErr("tip name is NULL");
}

// the tree of p as the one tree of the genome: one region per (non-empty) chromosome
GeneTrees one_tree(const jlp_ctx* c, const jlp_mutation_params* p) {
    const uint32_t n = p->n_nodes;
    if (n < 2 || n > kMutMaxNodes || !p->parent || !p->branch_len)
        throw ArgErr("the tree needs 2 to " + std::to_string(kMutMaxNodes) + " nodes (parent / branch_len not NULL)");
    if (p->parent[0] != -1) throw ArgErr("parent[0] must be -1 (the root comes first)");
    std::vector<char> has_kid(n, 0);
    for (uint32_t i = 1; i < n; i++) {
        if (p->parent[i] < 0 || (uint32_t)p->parent[i] >= i) throw ArgErr("the tree must be in preorder: 0 <= parent[i] < i");
        if (!(std::isfinite(p->branch_len[i]) && p->branch_len[i] >= 0)) throw ArgErr("branch lengths must be finite and >= 0");
        has_kid[p->parent[i]] = 1;
    }
    if (!p->tip_node) throw ArgErr("tip_node / tip_names is NULL");
    std::vector<char> is_tip(n, 0);
    for (uint32_t t = 0; t < p->n_tips; t++) {
        const uint32_t v = p->tip_node[t];
        if (v >= n || has_kid[v] || is_tip[v]) throw ArgErr("tip_node must list distinct childless nodes");
        is_tip[v] = 1;
    }
    GeneTrees g;
    g.trees.resize(1);
    g.trees[0].parent.assign(p->parent, p->parent + n);
    g.trees[0].branch_len.assign(p->branch_len, p->branch_len + n);
    g.trees[0].tip_node.assign(p->tip_node, p->tip_node + p->n_tips);
    const uint64_t nc = c->chrom_off.size() - 1;
    g.regions.resize(nc);
    for (uint64_t ci = 0; ci < nc; ci++) {
        const uint64_t len = c->chrom_off[ci + 1] - c->chrom_off[ci];
        if (len >> 32) throw ArgErr("chromosomes of 2^32 bases or more are not supported");
        if (len) g.regions[ci].push_back(TreeRegion{0, (uint32_t)len, 0});
    }
    return g;
}

unsigned host_threads(uint64_t items) {
    return (unsigned)std::min<uint64_t>(std::min<uint64_t>(items, 16), std::max(1u, std::thread::hardware_concurrency()));
}

}  // namespace

// The whole call: the trees and every chromosome's regions (one tree for the genome: one region per chromosome);
// im == nullptr: substitutions only, otherwise the indel model (ins_pi: the inserted columns' birth distribution) and
// its stats (one tree only).  table_budget: bytes of threshold tables per window (0: the default).
static void create_haps(jlp_ctx* c, const jlp_mutation_params* p, const GeneTrees& G, uint64_t table_budget,
                        const IndelModel* im, const double* ins_pi, jlp_mutation_stats* stats, jlp_indel_stats* istats,
                        jlp_gtree_stats* gstats) {
    const auto t0 = std::chrono::steady_clock::now();
    const uint32_t n = p->n_nodes;           // the one tree's nodes (indels only)
    const uint64_t nc = c->chrom_off.size() - 1;
    const uint32_t K = p->n_rates, n_tips = p->n_tips;
    const size_t n_items = (size_t)n_tips * nc;
    const uint64_t n_trees = G.trees.size();

    // the trees' schedules, one after the other (trees no region uses get none)
    std::vector<char> used(n_trees, 0);
    for (const auto& rs : G.regions)
        for (const TreeRegion& r : rs) used[r.tree] = 1;
    std::vector<std::vector<MutNode>> scheds(n_trees);
    std::vector<uint32_t> slots(n_trees, 0);
    parallel_for(n_trees, host_threads(n_trees / 64 + 1), [&](uint64_t i) {
        if (used[i]) scheds[i] = mut_schedule(G.trees[i], K, slots[i]);
    });
    std::vector<uint64_t> sched0(n_trees + 1, 0);
    for (uint64_t i = 0; i < n_trees; i++) sched0[i + 1] = sched0[i] + scheds[i].size();
    if (sched0[n_trees] >> 32) throw ArgErr("2^32 or more tree nodes in all");
    std::vector<MutNode> sched(sched0[n_trees]);
    for (uint64_t i = 0; i < n_trees; i++) std::copy(scheds[i].begin(), scheds[i].end(), sched.begin() + sched0[i]);
    const uint32_t max_slots = n_trees ? *std::max_element(slots.begin(), slots.end()) : 0;

    // tiles: per region from its start rounded down to a multiple of 4, kMutTile sites apart
    std::vector<uint32_t> tile0(nc + 1, 0);
    std::vector<MutTile> tiles;
    std::vector<uint32_t> tile_tree;
    for (uint64_t ci = 0; ci < nc; ci++) {
        tile0[ci] = (uint32_t)tiles.size();
        for (const TreeRegion& r : G.regions[ci])
            for (uint64_t f = r.start & ~3u; f < r.end; f += kMutTile) {
                tiles.push_back(MutTile{(uint32_t)ci, (uint32_t)f, r.start, r.end, (uint32_t)sched0[r.tree],
                                        (uint32_t)(sched0[r.tree + 1] - sched0[r.tree]), 0, 0});
                tile_tree.push_back(r.tree);
            }
        if (tiles.size() >> 32) throw ArgErr("genome too large");
    }
    tile0[nc] = (uint32_t)tiles.size();
    const uint32_t n_tiles = tile0[nc];

    // windows: contiguous tile ranges whose trees' tables fit the budget (a window holds at least one tree)
    struct Window { uint32_t t0, t1; uint64_t rows; std::vector<uint32_t> trees; };
    std::vector<Window> win;
    {
        const uint64_t budget = table_budget ? table_budget : kTableBudget;
        const uint64_t max_rows = std::min<uint64_t>(budget / (2 * sizeof(uint4)), 1ull << 31);
        std::vector<uint64_t> stamp(n_trees, UINT64_MAX), base(n_trees, 0);
        for (uint32_t tl = 0; tl < n_tiles; tl++) {
            const uint32_t tr = tile_tree[tl];
            if (win.empty() || stamp[tr] != win.size() - 1) {
                const uint64_t rows = (uint64_t)G.trees[tr].parent.size() * K * 4;
                if (win.empty() || (win.back().rows && win.back().rows + rows > max_rows)) {
                    if (!win.empty()) win.back().t1 = tl;
                    win.push_back(Window{tl, tl, 0, {}});
                }
                stamp[tr] = win.size() - 1;
                base[tr] = win.back().rows;
                win.back().rows += rows;
                win.back().trees.push_back(tr);
            }
            tiles[tl].tab0 = (uint32_t)base[tr];
        }
        if (!win.empty()) win.back().t1 = n_tiles;
    }
    uint64_t max_win_rows = 0, table_bytes = 0;
    for (const Window& w : win) {
        max_win_rows = std::max(max_win_rows, w.rows);
        table_bytes += w.rows * 2 * sizeof(uint4);
    }

    // indels: the event pass, chromosomes on up to 16 host threads; then the tips' records in one array (region
    // tip * nc + chromosome), each tile's first record, and the inserted columns with their places in the pools
    std::vector<IndelChrom> ich(im ? nc : 0);
    std::vector<IndelRec> irec;
    std::vector<uint64_t> ir_start;
    std::vector<uint32_t> icur;
    std::vector<int32_t> tip_of(im ? n : 0, -1);
    double event_ms = 0;
    if (im) {
        for (uint32_t t = 0; t < n_tips; t++) tip_of[p->tip_node[t]] = (int32_t)t;
        const auto te = std::chrono::steady_clock::now();
        parallel_for(nc, host_threads(nc), [&](uint64_t ci) {
            indel_events(p->seed, (uint32_t)ci, c->chrom_off[ci + 1] - c->chrom_off[ci], n, p->parent, p->branch_len,
                         tip_of.data(), n_tips, *im, ich[ci]);
        });
        ir_start.resize(n_items + 1);
        for (size_t r = 0; r < n_items; r++) {
            ir_start[r] = irec.size();
            const std::vector<IndelRec>& v = ich[r % nc].tip[r / nc].recs;
            irec.insert(irec.end(), v.begin(), v.end());
        }
        ir_start[n_items] = irec.size();
        if (irec.size() >> 32) throw ArgErr("2^32 or more insertion and deletion records are not supported");
        icur.resize((size_t)n_tips * n_tiles);
        for (size_t r = 0; r < n_items; r++) {
            const uint64_t ci = r % nc;
            uint64_t j = ir_start[r];
            for (uint32_t tl = tile0[ci]; tl < tile0[ci + 1]; tl++) {
                while (j < ir_start[r + 1] && irec[j].old_pos < tiles[tl].first) j++;
                icur[(r / nc) * n_tiles + tl] = (uint32_t)j;
            }
        }
        event_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - te).count();
    }

    // the inserted columns: birth node -> its schedule index and the end of its subtree's interval; per column the
    // (tip, record, byte) it fills, tips in schedule order
    std::vector<InsCol> cols;
    std::vector<InsEnt> ents;
    if (im) {
        std::vector<int64_t> spos(n, -1);
        std::vector<uint32_t> scount(n, 0);
        for (size_t i = 0; i < sched.size(); i++) spos[sched[i].node] = (int64_t)i;
        for (uint32_t i = n; i-- > 1;) {
            scount[i] += spos[i] >= 0;
            scount[p->parent[i]] += scount[i];
        }
        std::vector<uint64_t> col_base(nc + 1, 0);
        for (uint64_t ci = 0; ci < nc; ci++) col_base[ci + 1] = col_base[ci] + ich[ci].birth.size();
        if (col_base[nc] >> 32) throw ArgErr("2^32 or more inserted columns are not supported");
        cols.resize(col_base[nc]);
        std::vector<uint64_t> ecount(cols.size() + 1, 0);
        for (int pass = 0; pass < 2; pass++) {
            for (size_t si = 0; si < sched.size(); si++) {
                if (sched[si].tip < 0) continue;
                const uint32_t t = (uint32_t)sched[si].tip;
                for (uint64_t ci = 0; ci < nc; ci++) {
                    const IndelTip& T = ich[ci].tip[t];
                    const size_t r = (size_t)t * nc + ci;
                    for (size_t j = 0; j < T.recs.size(); j++)
                        for (uint64_t q = T.ids_off[j]; q < T.ids_off[j + 1]; q++) {
                            const uint64_t g = col_base[ci] + T.ids[q];
                            if (pass == 0) { ecount[g + 1]++; continue; }
                            const uint32_t k = (uint32_t)(q - T.ids_off[j]) + (T.recs[j].kind == kAnchorRec);
                            ents[cols[g].e1++] = InsEnt{(uint32_t)si, k, r, ir_start[r] + j};
                        }
                }
            }
            if (pass == 0) {
                for (size_t g = 0; g < cols.size(); g++) ecount[g + 1] += ecount[g];
                ents.resize(ecount.back());
                for (uint64_t ci = 0; ci < nc; ci++)
                    for (uint32_t id = 0; id < ich[ci].birth.size(); id++) {
                        const uint64_t g = col_base[ci] + id;
                        const uint32_t u = ich[ci].birth[id];
                        InsCol& col = cols[g];
                        col.chrom = (uint32_t)ci; col.id = id;
                        col.n0 = spos[u] >= 0 ? (uint32_t)spos[u] : 0;
                        col.n1 = spos[u] >= 0 ? (uint32_t)spos[u] + scount[u] : 0;
                        col.e0 = col.e1 = ecount[g];
                    }
            }
        }
    }
    std::vector<uint64_t> cat_thr(K);
    cat_thr[0] = prob_threshold(p->invariant);
    for (uint32_t j = 1; j < K; j++) cat_thr[j] = prob_threshold(p->invariant + j * (1 - p->invariant) / K);

    Device& d = device0(c);
    finish_upload(c, d);
    cudaStream_t s = d.s_compute;
    DevBuf<uint64_t> d_off, d_cat, d_region, d_region_n, d_out, d_ir_start, d_ir_nuc;
    DevBuf<uint32_t> d_tile0, d_cnt, d_icur;
    DevBuf<MutTile> d_tiles;
    DevBuf<IndelRec> d_irec;
    DevBuf<InsCol> d_cols;
    DevBuf<InsEnt> d_ents;
    DevBuf<MutNode> d_sched;
    DevBuf<uint4> d_hi, d_lo;
    TableBufs tb;
    d_off.upload(c->chrom_off, s);
    d_tile0.upload(tile0, s);
    d_tiles.upload(tiles, s);
    d_sched.upload(sched, s);
    d_cat.upload(cat_thr, s);
    d_hi.ensure(max_win_rows);
    d_lo.ensure(max_win_rows);
    if (max_win_rows) {                      // rows no node uses (the root's) are staged too: defined, never read
        CK(cudaMemsetAsync(d_hi.p, 0, max_win_rows * sizeof(uint4), s));
        CK(cudaMemsetAsync(d_lo.p, 0, max_win_rows * sizeof(uint4), s));
    }
    const size_t n_cnt = (size_t)n_tips * n_tiles;
    d_cnt.ensure(n_cnt);
    if (n_cnt) CK(cudaMemsetAsync(d_cnt.p, 0, n_cnt * 4, s));
    d_region_n.ensure((size_t)n_tips * nc);
    MutParams mp{};
    mp.seed = p->seed;
    mp.genome = d.genome.p + kPad;
    mp.chrom_off = d_off.p;
    mp.tile0 = d_tile0.p;
    mp.tiles = d_tiles.p;
    mp.n_chroms = (uint32_t)nc; mp.n_tiles = n_tiles; mp.n_tips = n_tips; mp.n_sched = (uint32_t)sched.size();
    mp.sched = d_sched.p;
    mp.n_cat = K;
    mp.cat_thr = d_cat.p;
    mp.thr_hi = d_hi.p; mp.thr_lo = d_lo.p;
    mp.cnt = d_cnt.p;
    if (im) {
        d_irec.upload(irec, s);
        d_ir_start.upload(ir_start, s);
        d_icur.upload(icur, s);
        d_ir_nuc.ensure(irec.size());
        mp.irec = d_irec.p; mp.ir_start = d_ir_start.p; mp.icur = d_icur.p; mp.ir_nuc = d_ir_nuc.p;
    }

    // a window's tables: one item per (tree, scheduled node, category)
    double table_ms = 0;
    std::vector<TabItem> titems;
    auto build_tables = [&](const Window& w) {
        const auto tt = std::chrono::steady_clock::now();
        titems.clear();
        uint64_t base = 0;
        for (uint32_t tr : w.trees) {
            const double* bl = G.trees[tr].branch_len.data();
            for (const MutNode& m : scheds[tr])
                for (uint32_t k = 0; k < K; k++)
                    titems.push_back(TabItem{p->rates[k] * bl[m.node], (uint32_t)(base + m.tab + 4ull * k), 0});
            base += (uint64_t)G.trees[tr].parent.size() * K * 4;
        }
        device_tables(s, p->Q, titems, tb, d_hi.p, d_lo.p, nullptr);
        table_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tt).count();
    };
    bool all_smem = true;
    auto set_window = [&](const Window& w) {
        mp.tile_begin = w.t0; mp.tile_end = w.t1;
        mp.tab_rows = (uint32_t)w.rows;
        mp.tab_smem = w.trees.size() == 1 && mut_smem_bytes((uint32_t)w.rows) <= (64u << 10);
        all_smem &= mp.tab_smem != 0;
    };
    EventSet ev;
    float count_ms = 0, write_ms = 0;
    for (const Window& w : win) {
        build_tables(w);
        set_window(w);
        CK(cudaEventRecord(ev.e[0], s));
        CK(launch_mutate(mp, false, im != nullptr, gstats != nullptr, s));
        CK(cudaEventRecord(ev.e[1], s));
        CK(cudaEventSynchronize(ev.e[1]));
        count_ms += ev.ms(0, 1);
    }
    CK(cudaEventRecord(ev.e[1], s));
    CK(launch_mut_scan(mp, d_region_n.p, s));
    CK(cudaEventRecord(ev.e[2], s));
    std::vector<uint64_t> region_n((size_t)n_tips * nc), region((size_t)n_tips * nc);
    CK(cudaMemcpyAsync(region_n.data(), d_region_n.p, region_n.size() * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    const float scan_ms = ev.ms(1, 2);
    // with indels region_n becomes substitution + indel records, pool the substitutions' bytes + the indel records'
    std::vector<uint64_t> pool(region_n);
    if (im)
        for (size_t r = 0; r < region.size(); r++) {
            const uint64_t a = ir_start[r], b = ir_start[r + 1];
            region_n[r] += b - a;
            if (b > a) pool[r] += irec[b - 1].pool_before + indel_pool_len(irec[b - 1]);
        }
    uint64_t words = 0, records = 0;
    for (size_t r = 0; r < region.size(); r++) {
        region[r] = words;
        words += 4 * region_n[r] + (pool[r] + 7) / 8;
        records += region_n[r];
    }
    d_region.upload(region, s);
    if (im) {
        d_region_n.upload(region_n, s);
        d_icur.upload(icur, s);
    }
    mp.region = d_region.p;
    mp.region_n = d_region_n.p;              // k_mut_scan left the totals there
    d_out.ensure(words);
    if (words) CK(cudaMemsetAsync(d_out.p, 0, words * 8, s));
    mp.out = d_out.p;
    if (records)
        for (const Window& w : win) {
            if (win.size() > 1) build_tables(w);
            set_window(w);
            CK(cudaEventRecord(ev.e[3], s));
            CK(launch_mutate(mp, true, im != nullptr, gstats != nullptr, s));
            CK(cudaEventRecord(ev.e[4], s));
            CK(cudaEventSynchronize(ev.e[4]));
            write_ms += ev.ms(3, 4);
        }
    if (im && !cols.empty()) {               // one tree: one window, whose tables are still in place
        d_cols.upload(cols, s);
        d_ents.upload(ents, s);
        InsParams ip{};
        ip.seed = p->seed;
        if (cols.size() >> 32) throw ArgErr("2^32 or more inserted columns are not supported");
        ip.n_cols = (uint32_t)cols.size();
        ip.n_cat = K;
        ip.cols = d_cols.p; ip.ent = d_ents.p; ip.sched = d_sched.p; ip.cat_thr = d_cat.p;
        row_thresholds(ins_pi, ip.pi_thr);
        ip.thr_hi = d_hi.p; ip.thr_lo = d_lo.p;
        ip.out = d_out.p; ip.region = d_region.p; ip.region_n = d_region_n.p; ip.ir_nuc = d_ir_nuc.p;
        CK(cudaEventRecord(ev.e[3], s));
        CK(launch_ins_walk(ip, s));
        CK(cudaEventRecord(ev.e[4], s));
        CK(cudaEventSynchronize(ev.e[4]));
        write_ms += ev.ms(3, 4);
    }
    CK(cudaStreamSynchronize(s));
    const auto t_gen = std::chrono::steady_clock::now();

    // the records into one HapStore per tip, copied straight into the packed arrays by a few host threads
    std::vector<std::shared_ptr<HapStore>> stores(n_tips);
    for (uint32_t t = 0; t < n_tips; t++) {
        stores[t] = std::make_shared<HapStore>();
        stores[t]->name = p->tip_names[t];
        stores[t]->chrom.resize(nc);
    }
    const unsigned nt = records < (1u << 16) ? 1u : host_threads(n_items);
    parallel_for(n_items, nt, [&](uint64_t r) {
        HapChromHost& H = stores[r / nc]->chrom[r % nc];
        const uint64_t M = region_n[r];
        H.size = im ? ich[r % nc].tip[r / nc].size : c->chrom_off[r % nc + 1] - c->chrom_off[r % nc];
        H.n_muts = M;
        H.pool_bytes = pool[r];
        if (!M) return;
        H.packed.resize(4 * M + (pool[r] + 7) / 8);
        CK(cudaSetDevice(d.id));
        CK(cudaMemcpy(H.packed.data(), d_out.p + region[r], H.packed.size() * 8, cudaMemcpyDeviceToHost));
    });

    clear_haps(c);
    for (const auto& S : stores) attach_hap(c, S);
    if (stats) {
        const auto t1 = std::chrono::steady_clock::now();
        stats->count_ms = count_ms;
        stats->scan_ms = scan_ms;
        stats->write_ms = write_ms;
        stats->store_ms = std::chrono::duration<double, std::milli>(t1 - t_gen).count();
        stats->total_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
        stats->records = records;
        stats->d2h_bytes = words * 8;
        stats->table_bytes = table_bytes;
        stats->table_in_smem = (int)(all_smem && !win.empty());
        stats->max_slots = max_slots;
    }
    if (istats) {
        *istats = jlp_indel_stats{};
        for (const IndelChrom& x : ich) {
            istats->insertions += x.insertions;
            istats->deletions += x.deletions;
            istats->inserted_bases += x.inserted_bases;
            istats->steps += x.steps;
        }
        istats->indel_records = irec.size();
        istats->event_ms = event_ms;
    }
    if (gstats) {
        gstats->n_trees = n_trees;
        gstats->n_regions = 0;
        for (const auto& rs : G.regions) gstats->n_regions += rs.size();
        gstats->windows = win.size();
        gstats->table_ms = table_ms;
    }
}

int jlp_create_haplotypes(jlp_ctx* c, const jlp_mutation_params* p, jlp_mutation_stats* stats) {
    if (!c || !p) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        check_model(c, p);
        create_haps(c, p, one_tree(c, p), 0, nullptr, nullptr, stats, nullptr, nullptr);
    });
}

int jlp_create_haplotypes_indels(jlp_ctx* c, const jlp_mutation_params* p, const jlp_indel_params* ip,
                                 jlp_mutation_stats* stats, jlp_indel_stats* istats) {
    if (!c || !p || !ip) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        auto rate_ok = [](double x) { return std::isfinite(x) && x >= 0; };
        if (!rate_ok(ip->rate_ins) || !rate_ok(ip->rate_del)) throw ArgErr("indel rates must be finite and >= 0");
        const double R = ip->rate_ins + ip->rate_del;
        if (R == 0) {
            check_model(c, p);
            create_haps(c, p, one_tree(c, p), 0, nullptr, nullptr, stats, nullptr, nullptr);
            if (istats) *istats = jlp_indel_stats{};
            return;
        }
        if (!(std::isfinite(ip->epsilon) && ip->epsilon > 0))
            throw ArgErr("epsilon must be > 0 when an indel rate is > 0");
        auto weights_ok = [&](double rate, uint32_t nw, const double* w) {
            if (rate == 0) return;
            if (nw < 1 || !w) throw ArgErr("an indel kind with a rate > 0 needs length weights (n >= 1, not NULL)");
            double sum = 0;
            for (uint32_t u = 0; u < nw; u++) {
                if (!rate_ok(w[u])) throw ArgErr("indel length weights must be finite and >= 0");
                sum += w[u];
            }
            if (!(sum > 0)) throw ArgErr("indel length weights need one weight > 0");
        };
        weights_ok(ip->rate_ins, ip->n_ins, ip->w_ins);
        weights_ok(ip->rate_del, ip->n_del, ip->w_del);
        double pis = 0;
        for (double x : ip->pi) {
            if (!rate_ok(x)) throw ArgErr("pi must be finite and >= 0");
            pis += x;
        }
        if (!(pis > 0)) throw ArgErr("pi needs one value > 0");
        // a kind of rate 0 has no lengths
        const uint32_t n_ins = ip->rate_ins > 0 ? ip->n_ins : 0, n_del = ip->rate_del > 0 ? ip->n_del : 0;
        IndelModel im;
        im.rate_ins = ip->rate_ins; im.rate_del = ip->rate_del; im.epsilon = ip->epsilon;
        im.n_ins = n_ins;
        im.kl_thr = indel_thresholds(ip->rate_ins, ip->w_ins, n_ins, ip->rate_del, ip->w_del, n_del);
        check_model(c, p);
        create_haps(c, p, one_tree(c, p), 0, &im, ip->pi, stats, istats, nullptr);
    });
}

int jlp_create_haplotypes_gtrees(jlp_ctx* c, const jlp_mutation_params* p, const jlp_gtree_params* g,
                                 jlp_mutation_stats* stats, jlp_gtree_stats* gstats) {
    if (!c || !p || !g) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        check_model(c, p);
        if (p->n_nodes || p->parent || p->branch_len || p->tip_node)
            throw ArgErr("with gene trees the trees come from the ms text: n_nodes, parent, branch_len and tip_node must be 0 / NULL");
        if (!g->text && g->text_len) throw ArgErr("the ms text is NULL");
        const uint64_t nc = c->chrom_off.size() - 1;
        std::vector<uint64_t> len(nc);
        for (uint64_t ci = 0; ci < nc; ci++) {
            len[ci] = c->chrom_off[ci + 1] - c->chrom_off[ci];
            if (len[ci] >> 32) throw ArgErr("chromosomes of 2^32 bases or more are not supported");
        }
        const auto t0 = std::chrono::steady_clock::now();
        GeneTrees G;
        parse_ms(g->text, g->text_len, len, p->tip_names, p->n_tips, kMutMaxNodes,
                 std::max(1u, std::thread::hardware_concurrency()), G);
        const double parse_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        jlp_gtree_stats gs{};
        create_haps(c, p, G, g->table_budget, nullptr, nullptr, stats, nullptr, &gs);
        gs.parse_ms = parse_ms;
        if (stats) stats->total_ms += parse_ms;
        if (gstats) *gstats = gs;
    });
}

int jlp_ms_regions(const char* text, uint64_t text_len, const uint64_t* chrom_len, uint64_t n_chroms,
                   const char* const* tip_names, uint32_t n_tips, uint64_t* reg, uint64_t cap, uint64_t* n_regions,
                   uint64_t* n_trees, char* err, uint64_t err_cap) {
    try {
        if ((!text && text_len) || (!chrom_len && n_chroms) || (!tip_names && n_tips)) throw ArgErr("NULL argument");
        GeneTrees G;
        parse_ms(text, text_len, std::vector<uint64_t>(chrom_len, chrom_len + n_chroms), tip_names, n_tips, kMutMaxNodes,
                 std::max(1u, std::thread::hardware_concurrency()), G);
        uint64_t k = 0;
        for (uint64_t ci = 0; ci < n_chroms; ci++)
            for (const TreeRegion& r : G.regions[ci]) {
                if (reg && k < cap) { reg[4 * k] = ci; reg[4 * k + 1] = r.start; reg[4 * k + 2] = r.end; reg[4 * k + 3] = r.tree; }
                k++;
            }
        if (n_regions) *n_regions = k;
        if (n_trees) *n_trees = G.trees.size();
        return JLP_OK;
    } catch (const std::exception& e) {
        if (err && err_cap) { std::strncpy(err, e.what(), err_cap - 1); err[err_cap - 1] = 0; }
        return JLP_ERR_ARG;
    }
}

int jlp_transition_tables(jlp_ctx* c, const double Q[16], const double* t, uint64_t n, double* P, uint64_t* thr,
                          uint64_t* n_host) {
    if (!c || !Q || (n && (!t || !P || !thr))) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        if (n >> 28) throw ArgErr("n must be below 2^28");
        std::vector<TabItem> items(n);
        for (uint64_t i = 0; i < n; i++) items[i] = TabItem{t[i], (uint32_t)(4 * i), 0};
        Device& d = device0(c);
        cudaStream_t s = d.s_compute;
        DevBuf<uint4> hi, lo;
        DevBuf<double> dP;
        TableBufs tb;
        hi.ensure(4 * n); lo.ensure(4 * n); dP.ensure(16 * n);
        const uint64_t nh = device_tables(s, Q, items, tb, hi.p, lo.p, dP.p);
        std::vector<uint4> h(4 * n), l(4 * n);
        if (n) {
            CK(cudaMemcpyAsync(h.data(), hi.p, 4 * n * sizeof(uint4), cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(l.data(), lo.p, 4 * n * sizeof(uint4), cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(P, dP.p, 16 * n * sizeof(double), cudaMemcpyDeviceToHost, s));
        }
        CK(cudaStreamSynchronize(s));
        for (uint64_t r = 0; r < 4 * n; r++) {
            thr[3 * r] = (uint64_t)h[r].x << 32 | l[r].x;
            thr[3 * r + 1] = (uint64_t)h[r].y << 32 | l[r].y;
            thr[3 * r + 2] = (uint64_t)h[r].z << 32 | l[r].z;
        }
        if (n_host) *n_host = nh;
    });
}

int jlp_set_profile(jlp_ctx* c, int end, uint64_t read_length, const uint32_t* nq, const double* probs,
                    const uint8_t* quals) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        if (end < 0 || end > 1) throw ArgErr("end must be 0 or 1");
        if (!nq || !probs || !quals) throw ArgErr("profile arrays are NULL");
        if (read_length >= 65536) throw ArgErr("read_length too large");
        build_end_tables(read_length, nq, probs, quals, c->tab[end]);
        const EndTables& t = c->tab[end];
        on_each_device(c, [&](Device& d) {
            d.d_meta[end].upload(t.meta, d.s_compute);
            d.d_entry64[end].upload(t.entry64, d.s_compute);
            d.d_coin[end].upload(t.coin, d.s_compute);
            d.d_mis[end].upload(t.mis, d.s_compute);
            CK(cudaStreamSynchronize(d.s_compute));
            d.h2d_bytes += t.meta.size() * 4 + t.entry64.size() * 16 + 256 * 8;
        });
        c->have_prof[end] = true;
    });
}

static void run_any(jlp_ctx* c, bool use_haps, const jlp_illumina_params* p, Output& s, jlp_run_stats* stats) {
    check_params(c, use_haps, p, s.kind);
    if (c->dev.size() == 1) run(c, *c->dev[0], use_haps, p, make_layout(c, illumina_spec(c, use_haps, p)), s, stats);
    else run_multi(c, use_haps, p, s, stats);
}

int jlp_illumina_ref(jlp_ctx* c, const jlp_illumina_params* p, jlp_run_stats* stats) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() { Output s(SINK_FILES); run_any(c, false, p, s, stats); });
}
int jlp_illumina_hap(jlp_ctx* c, const jlp_illumina_params* p, jlp_run_stats* stats) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() { Output s(SINK_FILES); run_any(c, true, p, s, stats); });
}

int jlp_illumina_to_memory(jlp_ctx* c, int use_haplotypes, const jlp_illumina_params* p, char* out1, uint64_t cap1,
                           uint64_t* len1, char* out2, uint64_t cap2, uint64_t* len2, jlp_run_stats* stats) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        Output s(SINK_MEMORY);
        s.mem[0] = out1; s.cap[0] = out1 ? cap1 : 0;
        s.mem[1] = out2; s.cap[1] = out2 ? cap2 : 0;
        run_any(c, use_haplotypes != 0, p, s, stats);
        if (len1) *len1 = s.len[0];
        if (len2) *len2 = s.len[1];
        if (s.len[0] > s.cap[0] || s.len[1] > s.cap[1]) throw ArgErr("output buffer too small");
    });
}

int jlp_illumina_stream(jlp_ctx* c, int use_haplotypes, const jlp_illumina_params* p, jlp_chunk_cb cb, void* user,
                        jlp_run_stats* stats) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        if (!cb) throw ArgErr("chunk callback is NULL");
        Output s(SINK_STREAM);
        s.chunk_cb = cb; s.chunk_user = user;
        run_any(c, use_haplotypes != 0, p, s, stats);
    });
}

int jlp_illumina_device_only(jlp_ctx* c, int use_haplotypes, const jlp_illumina_params* p, jlp_run_stats* stats) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() { Output s; run_any(c, use_haplotypes != 0, p, s, stats); });
}

int jlp_illumina_group_counts(jlp_ctx* c, int use_haplotypes, const jlp_illumina_params* p, uint64_t* counts,
                              uint64_t cap, uint64_t* n_groups) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        if (!p) throw ArgErr("params is NULL");
        std::vector<std::vector<uint64_t>> cnt = apportion(c, illumina_spec(c, use_haplotypes != 0, p));
        uint64_t n = 0;
        for (const auto& v : cnt) n += v.size();
        if (n_groups) *n_groups = n;
        if (n > cap) throw ArgErr("counts buffer too small");
        uint64_t k = 0;
        for (const auto& v : cnt) for (uint64_t x : v) counts[k++] = x;
    });
}

// ---- PacBio ----

namespace {

void pb_model_from(const jlp_pacbio_params* P, PbModel& m) {
    if (!P) throw ArgErr("params is NULL");
    m.scale = P->scale; m.sigma = P->sigma; m.loc = P->loc; m.min_read_len = P->min_read_len;
    if (P->n_custom) {
        if (!P->read_probs || !P->read_lens) throw ArgErr("custom read lengths are NULL");
        m.read_probs.assign(P->read_probs, P->read_probs + P->n_custom);
        m.read_lens.assign(P->read_lens, P->read_lens + P->n_custom);
    }
    m.max_passes = P->max_passes;
    std::copy(P->chi2_params_n, P->chi2_params_n + 3, m.chi2_n);
    std::copy(P->chi2_params_s, P->chi2_params_s + 5, m.chi2_s);
    std::copy(P->sqrt_params, P->sqrt_params + 2, m.sqrt_params);
    std::copy(P->norm_params, P->norm_params + 2, m.norm_params);
    m.prob_thresh = P->prob_thresh; m.prob_ins = P->prob_ins; m.prob_del = P->prob_del; m.prob_subst = P->prob_subst;
    if (!(m.sigma > 0) || !(m.scale > 0) || m.max_passes < 1 || !(m.norm_params[1] > 0)) throw ArgErr("invalid PacBio model parameters");
    try { pb_prepare(m); } catch (const std::exception& e) { throw ArgErr(e.what()); }
}

// The compression rule of the drivers that write one file per job (PacBio, VCF): unlike compression_of(), AUTO takes the
// device coder at levels 1..6 whatever the method and thread count; compressed output goes to files only.
Compression file_compression(int compress, const char* comp_method, uint64_t n_threads, int comp_engine, SinkKind kind) {
    Compression z;
    if (compress <= 0) return z;
    z.want_gz = true;
    if (kind != SINK_FILES) return z;
    z.dev_z = comp_engine == JLP_COMP_DEVICE || (comp_engine == JLP_COMP_AUTO && compress <= 6);
    if (!z.dev_z) z.zmethod = n_threads > 1 || std::string(comp_method) == "bgzip" ? DEFLATE_BGZF : DEFLATE_GZIP;
    return z;
}

// One batch of the drivers that write one file per job (PacBio, VCF), its stream synchronised: nb bytes at src on the
// device go through the pinned buffer of slot n_batch & 1 (free once the batch before last is settled; grown to
// max(nb, cap) + 64 bytes when it holds less than nb + 64) to the sink, which writes them while the next batch is made.
void hand_over(Device& d, Output& sink, uint64_t& n_batch, const uint8_t* src, uint64_t nb, uint64_t job, uint64_t cap) {
    Slot& hs = d.slot[n_batch++ & 1];
    sink.settle(hs.host);
    PinBuf<uint8_t>& h = hs.h_out[0];
    if (h.n < nb + 64) h.ensure(std::max(nb, cap) + 64);
    CK(cudaMemcpy(h.p, src, nb, cudaMemcpyDeviceToHost));
    const uint8_t* data[2] = {h.p, nullptr};
    const uint64_t len[2] = {nb, 0};
    sink.deliver(hs.host, data, len, job, 1);
}

// The driver: per batch the per-read quantities are prepared on the host (batch k + 1 on a helper thread while batch k
// is on the device), then plan upload, k_pb_plan, scan, k_pb_reads, optional BGZF, copy, and the write of batch k
// overlaps the next batch.  Callbacks are called on the calling thread between batches.
void run_pacbio(jlp_ctx* c, Device& d, bool use_haps, const jlp_pacbio_params* P, Output& sink, jlp_run_stats* stats) {
    PbModel model;
    pb_model_from(P, model);
    // the quantiles computed by earlier calls with the same pass-sampler parameters are kept (each costs a bisection on
    // the incomplete gamma function; a fresh table made the first thousands of reads of every call slow)
    if (c->pb_qcache && c->pb_qcache_n == model.qchisq_n && std::equal(model.chi2_n, model.chi2_n + 3, c->pb_qcache_key))
        model.qchisq_cache = c->pb_qcache;
    else {
        c->pb_qcache = model.qchisq_cache; c->pb_qcache_n = model.qchisq_n;
        std::copy(model.chi2_n, model.chi2_n + 3, c->pb_qcache_key);
    }
    if (!(P->prob_dup >= 0 && P->prob_dup <= 1)) throw ArgErr("prob_dup must be in [0,1]");
    if (P->read_pool_size < 1) throw ArgErr("read_pool_size must be >= 1");
    const Thr t_dup = thr_double_lt(P->prob_dup);
    const bool dups = t_dup.thr != 0 || t_dup.all;
    if (dups && P->read_pool_size > 65536) throw Unsupported("prob_dup > 0 with read_pool_size > 65536");
    if (P->compress < 0) throw ArgErr("\nInvalid bgzip compress level. It must be in range [0,9].");
    check_compression(P->compress, P->comp_method, P->comp_engine);
    if (P->shard_count > 1 && P->shard_index >= P->shard_count) throw ArgErr("shard_index >= shard_count");
    finish_upload(c, d);
    Layout G = make_layout(c, LayoutSpec(use_haps, P, P->n_reads));
    for (size_t g = 0; g < G.groups.size(); g++) {
        const uint32_t h = G.group_hap[g], ci = G.group_chrom[g];
        if (use_haps && G.group_off[g + 1] > G.group_off[g]) ensure_hap_chrom(c, d, h, ci);   // materialised when first read from
        G.groups[g].seq = use_haps ? d.hap_seq[h][ci] : d.genome.p + kPad + c->chrom_off[ci];
    }
    const Compression Z = file_compression(P->compress, P->comp_method, P->n_threads, P->comp_engine, sink.kind);
    const bool dev_z = Z.dev_z;
    // the slots' buffers (pinning a gigabyte of host memory on every call cost more than generating the reads, and a dozen
    // device allocations and frees per call several milliseconds): the device arrays of slot 0; hand_over's pinned buffers
    Slot& S0 = d.slot[0];
    cudaEvent_t* ev = S0.ev;
    uint64_t n_batch = 0;
    sink.begin(Z, P->compress, P->n_threads, d.writers);
    Quiesce quiesce{d, &sink};
    d.d_groups.upload(G.groups, d.s_compute);
    d.d_strpool.upload(G.strpool, d.s_compute);
    S0.totals.ensure(4);
    CK(cudaMemsetAsync(S0.totals.p, 0, 4 * sizeof(uint64_t), d.s_compute));
    uint64_t B = P->batch_reads ? P->batch_reads : 32768;
    // a chain of duplicates never leaves its pool (src/hts.h:266-267): batches are whole pools, so a duplicate's leader is in
    // its batch
    if (dups) B = std::max<uint64_t>(P->read_pool_size, B / P->read_pool_size * P->read_pool_size);
    uint32_t max_prefix = 0;
    for (const GroupDev& g : G.groups) max_prefix = std::max(max_prefix, g.prefix_len);
    const uint64_t c_rev = thr_ld_lt(0.5).thr;
    jlp_run_stats st;
    std::memset(&st, 0, sizeof st);
    for (size_t jk = 0; jk < G.jobs.size(); jk++) {
        const Job& job = G.jobs[jk];
        const std::string names[2] = {file_name(job, 0, Z.want_gz, nullptr)};     // PacBio's files have no shard suffix
        sink.open_job(names, 1, nullptr, false);
        // this shard's part of the job: whole pools, so that chains of duplicates stay inside it
        uint64_t s_lo = job.lo, s_hi = job.hi;
        if (P->shard_count > 1) {
            const uint64_t pool = std::max<uint64_t>(P->read_pool_size, 1), n_pools = (job.hi - job.lo + pool - 1) / pool;
            uint64_t p_lo, p_hi;
            shard_range(0, n_pools, P->shard_index, P->shard_count, p_lo, p_hi);
            s_lo = std::min(job.hi, job.lo + p_lo * pool);
            s_hi = std::min(job.hi, job.lo + p_hi * pool);
        }
        // ---- per-read quantities on the host (read length, passes, error probabilities, thresholds): batch k + 1 is
        //      prepared by a helper thread (which spreads the reads over n_threads workers) while the device
        //      generates batch k and the sink takes it; bound: the FASTQ bytes of the batch at most
        struct Prepared { std::vector<PbRead> plan; uint64_t bound = 0; std::exception_ptr err; };
        auto prepare = [&](uint64_t b0, uint32_t n, Prepared& out) {
            try {
                out.plan.resize(n);
                const uint64_t len = pb_plan(model, P->seed, b0, n, job.lo, P->read_pool_size, t_dup, G.group_off, G.groups.data(),
                                             P->n_threads, out.plan.data(), nullptr);
                out.bound = (uint64_t)n * (max_prefix + 24 + 5) + 2 * len;
            } catch (...) { out.err = std::current_exception(); }
        };
        Prepared prep[2];
        std::thread prep_thread;
        struct JoinPrep { std::thread& t; ~JoinPrep() { if (t.joinable()) t.join(); } } join_prep{prep_thread};
        // JLP_TRACE=1: where the host side of the call spends its time (stderr, one line per job)
        const bool trace = std::getenv("JLP_TRACE") != nullptr;
        double t_first = 0, t_join = 0, t_alloc = 0, t_sync = 0;
        auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
        const double t_job = now();
        // with the default batch size the first batches are small (8192 reads, doubling): the first preparation is the
        // one nothing overlaps, so the device should not wait for a full batch of it
        auto batch_size = [&](uint64_t k) -> uint64_t {
            if (P->batch_reads) return B;
            uint64_t b = std::min<uint64_t>(B, 8192ull << std::min<uint64_t>(k, 8));
            if (dups) b = std::max<uint64_t>(P->read_pool_size, b / P->read_pool_size * P->read_pool_size);
            return b;
        };
        {   // the per-read device arrays once, for the largest batch of the job (growing them batch by batch would
            // free and allocate -- and synchronise -- at every step of the ramp)
            const uint64_t n_max = std::min<uint64_t>(B, s_hi - s_lo);
            d.pb_reads.ensure(n_max); S0.rec_len.ensure(n_max); S0.rec_local.ensure(n_max);
            const uint64_t nsb_max = (n_max + kScanBlock - 1) / kScanBlock;
            S0.block_tot.ensure(nsb_max); S0.block_base.ensure(nsb_max);
        }
        // batches differ in size: the output buffers grow with slack, and at once to what a full batch will need (pinning
        // is slow)
        auto grow_to = [&](uint64_t need, uint32_t n) {
            const uint64_t want = std::max(need, n ? need / n * std::min<uint64_t>(B, s_hi - s_lo) : need);
            return want + want / 4;
        };
        uint64_t n_next = std::min<uint64_t>(batch_size(0), s_hi - s_lo), b0_next = s_lo;
        if (s_lo < s_hi) prepare(s_lo, (uint32_t)n_next, prep[0]);
        t_first = now() - t_job;
        uint64_t bk = 0;
        for (uint64_t b0 = s_lo; b0 < s_hi; b0 = b0_next, bk++) {
            const uint32_t n = (uint32_t)n_next;
            double t0 = now();
            if (prep_thread.joinable()) prep_thread.join();
            t_join += now() - t0;
            Prepared& cur = prep[bk & 1];
            if (cur.err) std::rethrow_exception(cur.err);
            if (P->abort_cb && P->abort_cb(P->cb_user)) throw Aborted();      // Progress::check_abort, src/hts.h:396-399
            b0_next = b0 + n;
            if (b0_next < s_hi) {
                Prepared* nxt = &prep[(bk + 1) & 1];
                const uint64_t nb0 = b0_next;
                n_next = std::min<uint64_t>(batch_size(bk + 1), s_hi - nb0);
                const uint32_t nn = (uint32_t)n_next;
                prep_thread = std::thread([&prepare, nb0, nn, nxt]() { prepare(nb0, nn, *nxt); });
            }
            std::vector<PbRead>& plan = cur.plan;
            const uint64_t bound = cur.bound;
            t0 = now();
            d.pb_reads.ensure(n);
            S0.rec_len.ensure(n); S0.rec_local.ensure(n);
            const uint32_t nsb = (n + kScanBlock - 1) / kScanBlock;
            S0.block_tot.ensure(nsb); S0.block_base.ensure(nsb);
            if (S0.out[0].n < bound + 64) S0.out[0].ensure(grow_to(bound, n) + 64);
            t_alloc += now() - t0;
            CK(cudaMemcpyAsync(d.pb_reads.p, plan.data(), n * sizeof(PbRead), cudaMemcpyHostToDevice, d.s_compute));
            st.h2d_bytes += n * sizeof(PbRead);
            CK(cudaEventRecord(ev[0], d.s_compute));
            CK(launch_pb_plan(d.pb_reads.p, n, b0, P->seed, d.d_groups.p, c_rev, S0.rec_len.p, d.s_compute));
            if (dups) { CK(launch_pb_dups(d.pb_reads.p, n, b0, P->seed, d.d_groups.p, S0.rec_len.p, d.s_compute)); st.kernel_launches++; }
            CK(launch_scan(S0.rec_len.p, n, 1, S0.rec_local.p, S0.block_tot.p, S0.block_base.p, S0.totals.p, d.s_compute));
            CK(launch_pb_reads(d.pb_reads.p, n, b0, P->seed, d.d_groups.p, d.d_strpool.p, S0.rec_local.p, S0.block_base.p, S0.out[0].p,
                               d.s_compute));
            CK(cudaEventRecord(ev[1], d.s_compute));
            st.kernel_launches += 4;
            const uint32_t nblk = (uint32_t)((bound + kBgzfIn - 1) / kBgzfIn) + 1;
            if (dev_z) {
                S0.z.ensure(nblk, bound, 1);
                CK(S0.z.launch(S0.out[0].p, S0.out[0].p, S0.totals.p, nblk, P->compress, d.s_compute));
                st.kernel_launches += kBgzfLaunches;
            }
            CK(cudaEventRecord(ev[2], d.s_compute));
            uint64_t tot[4];
            CK(cudaMemcpyAsync(tot, S0.totals.p, sizeof tot, cudaMemcpyDeviceToHost, d.s_compute));
            t0 = now();
            CK(cudaStreamSynchronize(d.s_compute));
            t_sync += now() - t0;
            if (tot[0] > bound) throw std::runtime_error("internal: PacBio batch larger than its bound");
            float ms = 0;
            CK(cudaEventElapsedTime(&ms, ev[0], ev[1])); st.reads_ms += ms; st.device_ms += ms;
            CK(cudaEventElapsedTime(&ms, ev[1], ev[2])); if (dev_z) { st.bgzf_ms += ms; st.device_ms += ms; }
            st.pairs += n; st.batches++; st.bytes_out[0] += tot[0];
            if (dev_z) st.z_bytes[0] += tot[2];
            if (sink.kind == SINK_NONE) { if (P->progress_cb) P->progress_cb(P->cb_user, n); continue; }
            const uint64_t nb = dev_z ? tot[2] : tot[0];
            hand_over(d, sink, n_batch, dev_z ? S0.z.out[0].p : S0.out[0].p, nb, jk, grow_to(nb, n));
            st.d2h_bytes += nb;
            if (P->progress_cb) P->progress_cb(P->cb_user, n);                  // Progress::increment, src/hts.h:414
        }
        if (prep_thread.joinable()) prep_thread.join();
        sink.settle(d.slot[0].host); sink.settle(d.slot[1].host);
        if (trace)
            std::fprintf(stderr, "[jlp trace] pacbio job %llu reads: %.4f s (first prepare %.4f, waiting for later ones %.4f, "
                         "device allocations %.4f, waiting for the device %.4f)\n", (unsigned long long)(s_hi - s_lo), now() - t_job,
                         t_first, t_join, t_alloc, t_sync);
        sink.end_job(jk, 1, true);
    }
    if (stats) *stats = st;
    quiesce.armed = false;
}

// ---- VCF (DESIGN.md section 11) ----

// The VCF of the context's haplotypes on device d, chromosome by chromosome: the included haplotypes' records are
// uploaded (the next chromosome's while this one's kernels run), grouped into lines and sized on the device; the host
// cuts the lines into batches of about batch_bytes of text, each written on the device at its final offsets, optionally
// compressed there, copied into the slots' pinned buffers and handed to the sink.  The header opens the first batch.
void write_vcf(jlp_ctx* c, Device& d, const jlp_vcf_params* P, jlp_vcf_stats* stats) {
    const auto t_call = std::chrono::steady_clock::now();
    if (!P) throw ArgErr("params is NULL");
    if (!P->path || !*P->path) throw ArgErr("path is empty");
    if (c->chrom_off.size() < 2) throw ArgErr("no reference genome has been set");
    if (c->haps.empty()) throw ArgErr("no haplotypes have been added");
    if (P->n_samples < 1 || P->ploidy < 1 || !P->sample_haps) throw ArgErr("the sample matrix is empty");
    if (P->n_samples * P->ploidy >= 0xffffffffull) throw ArgErr("the sample matrix has 2^32 slots or more");
    if (!P->sample_names || !P->file_date) throw ArgErr("sample_names / file_date is NULL");
    if (P->compress < 0) throw ArgErr("\nInvalid bgzip compress level. It must be in range [0,9].");
    check_compression(P->compress, P->comp_method, P->comp_engine);
    if (P->n_threads < 1 || P->n_threads > 64) throw ArgErr("n_threads must be in 1..64");
    const uint64_t n_haps = c->haps.size(), n_chroms = c->chrom_off.size() - 1, n_slots = P->n_samples * P->ploidy;
    for (const std::string& n : c->chrom_names)
        for (char ch : n)
            if (std::isspace((unsigned char)ch)) throw ArgErr("chromosome name \"" + n + "\" contains whitespace");
    for (uint64_t i = 0; i < P->n_samples; i++) {
        if (!P->sample_names[i]) throw ArgErr("a sample name is NULL");
        if (std::strpbrk(P->sample_names[i], "\t\r\n")) throw ArgErr("a sample name contains a tab, CR or LF");
    }
    // the included haplotypes in index order, each slot's included haplotype, their first slots and slot counts
    std::vector<uint32_t> local(n_haps, 0xffffffffu), slot_hap(n_slots), inc, first_slot, slots_of;
    for (uint64_t k = 0; k < n_slots; k++)
        if (P->sample_haps[k] >= n_haps) throw ArgErr("sample_haps: haplotype index out of range");
    for (uint64_t k = 0; k < n_slots; k++) local[P->sample_haps[k]] = 0;
    for (uint64_t h = 0; h < n_haps; h++)
        if (local[h] == 0) { local[h] = (uint32_t)inc.size(); inc.push_back((uint32_t)h); }
    first_slot.assign(inc.size(), 0xffffffffu);
    slots_of.assign(inc.size(), 0);
    for (uint64_t k = 0; k < n_slots; k++) {
        const uint32_t u = local[P->sample_haps[k]];
        slot_hap[k] = u;
        first_slot[u] = std::min(first_slot[u], (uint32_t)k);
        slots_of[u]++;
    }
    const uint32_t n_inc = (uint32_t)inc.size();
    std::vector<uint64_t> n_rec(n_chroms, 0);
    uint64_t n_max = 1;
    for (uint64_t ci = 0; ci < n_chroms; ci++) {
        for (uint32_t h : inc) n_rec[ci] += c->haps[h]->chrom[ci].n_muts;
        if (n_rec[ci] >= 0xffffffffull) throw ArgErr("2^32 records or more on one chromosome");
        n_max = std::max(n_max, n_rec[ci]);
    }
    std::string hdr = "##fileformat=VCFv4.3\n##fileDate=" + std::string(P->file_date) + "\n##source=jackalope_b200\n";
    std::vector<uint8_t> names;
    std::vector<uint64_t> name_off;
    for (uint64_t ci = 0; ci < n_chroms; ci++) {
        hdr += "##contig=<ID=" + c->chrom_names[ci] + ",length=" + std::to_string(c->chrom_off[ci + 1] - c->chrom_off[ci]) + ">\n";
        name_off.push_back(names.size());
        names.insert(names.end(), c->chrom_names[ci].begin(), c->chrom_names[ci].end());
    }
    hdr += "##ALT=<ID=DEL,Description=\"The haplotype has no bases over this line\">\n"
           "##FORMAT=<ID=GT,Number=1,Type=String,Description=\"Genotype\">\n"
           "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT";
    for (uint64_t i = 0; i < P->n_samples; i++) hdr += std::string("\t") + P->sample_names[i];
    hdr += "\n";

    finish_upload(c, d);
    const cudaStream_t s = d.s_compute;
    const Compression Z = file_compression(P->compress, P->comp_method, P->n_threads, P->comp_engine, SINK_FILES);
    Output sink(SINK_FILES);
    sink.begin(Z, P->compress, P->n_threads, d.writers);
    const std::string files[2] = {P->path, ""};
    sink.open_job(files, 1, nullptr, false);
    Quiesce quiesce{d, &sink};
    Slot& S0 = d.slot[0];
    cudaEvent_t* ev = S0.ev;
    // device scratch for the largest chromosome
    DevBuf<uint64_t> b_start, b_end, b_start_s, b_end_s, b_maxend, b_key2, b_key2_s, b_line_s, b_line_e, b_line_len, b_line_end;
    DevBuf<uint32_t> b_rec_hap, b_val, b_order, b_flag, b_lid, b_car_pos, b_cls_car, b_cls_slot, b_cls_rank, b_alt_car, b_line_first,
        b_n_car, b_n_alt, b_slot_hap, b_first_slot, b_slots_of, b_hidx;
    DevBuf<VcfCar> b_car;
    DevBuf<VcfHap> b_hap;
    DevBuf<uint8_t> b_cub, b_names;
    for (DevBuf<uint64_t>* b : {&b_start, &b_end, &b_start_s, &b_end_s, &b_maxend, &b_key2, &b_key2_s, &b_line_s, &b_line_e, &b_line_len,
                                &b_line_end})
        b->ensure(n_max + 1);
    for (DevBuf<uint32_t>* b : {&b_rec_hap, &b_val, &b_order, &b_flag, &b_lid, &b_car_pos, &b_cls_car, &b_cls_slot, &b_cls_rank,
                                &b_alt_car, &b_line_first, &b_n_car, &b_n_alt})
        b->ensure(n_max + 1);
    b_car.ensure(n_max);
    b_cub.ensure(vcf_cub_bytes((uint32_t)n_max));
    const uint64_t hidx_n = (uint64_t)vcf_line_blocks(~0ull >> 8, d.n_sm) * 8 * n_inc;
    b_hidx.ensure(hidx_n);
    CK(cudaMemsetAsync(b_hidx.p, 0, hidx_n * sizeof(uint32_t), s));
    b_slot_hap.upload(slot_hap, s);
    b_first_slot.upload(first_slot, s);
    b_slots_of.upload(slots_of, s);
    b_names.upload(names, s);
    PinBuf<uint64_t> h_line_end, h_small;
    h_line_end.ensure(n_max);
    h_small.ensure(4);
    const uint64_t B = P->batch_bytes ? P->batch_bytes : (256ull << 20);
    const bool dev_z = Z.dev_z;
    jlp_vcf_stats st;
    std::memset(&st, 0, sizeof st);
    bool hdr_done = false;
    uint64_t n_batch = 0;
    auto elapsed = [&](cudaEvent_t a, cudaEvent_t b) { float ms = 0; CK(cudaEventElapsedTime(&ms, a, b)); return (double)ms; };
    // one batch: the header if it has not been written, then the text of lines [l0, l1) of v
    auto emit = [&](const VcfChrom* v, uint32_t l0, uint32_t l1, uint64_t text_n) {
        const uint64_t hn = hdr_done ? 0 : hdr.size(), total = hn + text_n;
        S0.out[0].ensure(std::max(total, B) + 64);
        if (hn) CK(cudaMemcpyAsync(S0.out[0].p, hdr.data(), hn, cudaMemcpyHostToDevice, s));
        CK(cudaEventRecord(ev[0], s));
        if (v) CK(launch_vcf_text(*v, l0, l1, S0.out[0].p, hn, d.n_sm, s));
        CK(cudaEventRecord(ev[1], s));
        if (dev_z) {
            const uint32_t nblk = (uint32_t)(total / kBgzfIn) + 1;
            S0.z.ensure(nblk, total, 1); S0.totals.ensure(4);
            h_small.p[0] = total; h_small.p[1] = 0;
            CK(cudaMemcpyAsync(S0.totals.p, h_small.p, 2 * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
            CK(S0.z.launch(S0.out[0].p, S0.out[0].p, S0.totals.p, nblk, P->compress, s));
            CK(cudaMemcpyAsync(h_small.p, S0.totals.p, 4 * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        }
        CK(cudaEventRecord(ev[2], s));
        CK(cudaStreamSynchronize(s));
        st.text_ms += elapsed(ev[0], ev[1]);
        if (dev_z) st.bgzf_ms += elapsed(ev[1], ev[2]);
        hand_over(d, sink, n_batch, dev_z ? S0.z.out[0].p : S0.out[0].p, dev_z ? h_small.p[2] : total, 0, B);
        st.batches++;
        st.text_bytes += total;
        hdr_done = true;
    };
    // the records of chromosome ci, each included haplotype's packed array once, on the upload stream into the next of
    // materialisation's buffers
    std::vector<VcfHap> hap_tab;
    auto upload = [&](uint64_t ci) {
        const int k = claim_mat_buf(d);
        uint64_t words = 0;
        for (uint32_t h : inc) words += c->haps[h]->chrom[ci].packed.size();
        d.m_pack[k].ensure(words);
        words = 0;
        for (uint32_t h : inc) {
            const HapChromHost& M = c->haps[h]->chrom[ci];
            if (!M.packed.empty())
                CK(cudaMemcpyAsync(d.m_pack[k].p + words, M.packed.data(), M.packed.size() * 8, cudaMemcpyHostToDevice, d.s_upload));
            words += M.packed.size();
            d.h2d_bytes += M.packed.size() * 8;
        }
        CK(cudaEventRecord(d.m_up[k], d.s_upload));
        return k;
    };
    int k_cur = n_rec[0] ? upload(0) : -1;
    for (uint64_t ci = 0; ci < n_chroms; ci++) {
        const int k = k_cur;
        k_cur = -1;
        if (n_rec[ci] == 0) {
            if (ci + 1 < n_chroms && n_rec[ci + 1]) k_cur = upload(ci + 1);
            continue;
        }
        hap_tab.clear();
        uint64_t woff = 0, r0 = 0;
        for (uint32_t h : inc) {
            const HapChromHost& M = c->haps[h]->chrom[ci];
            hap_tab.push_back(VcfHap{woff, (uint32_t)M.n_muts, (uint32_t)r0});
            woff += M.packed.size();
            r0 += M.n_muts;
        }
        hap_tab.push_back(VcfHap{woff, 0, (uint32_t)r0});
        b_hap.upload(hap_tab, s);
        VcfChrom v;
        v.recs = d.m_pack[k].p; v.hap = b_hap.p; v.n_hap = n_inc; v.n_rec = (uint32_t)n_rec[ci];
        v.ref = d.genome.p + kPad + c->chrom_off[ci]; v.L = c->chrom_off[ci + 1] - c->chrom_off[ci];
        v.name = b_names.p + name_off[ci]; v.name_len = (uint32_t)c->chrom_names[ci].size();
        v.ploidy = P->ploidy; v.n_samples = (uint32_t)P->n_samples;
        v.slot_hap = b_slot_hap.p; v.first_slot = b_first_slot.p; v.n_slots = b_slots_of.p;
        v.start = b_start.p; v.end = b_end.p; v.start_sorted = b_start_s.p; v.end_sorted = b_end_s.p; v.maxend = b_maxend.p;
        v.key2 = b_key2.p; v.key2_sorted = b_key2_s.p;
        v.rec_hap = b_rec_hap.p; v.val = b_val.p; v.order = b_order.p; v.flag = b_flag.p; v.lid = b_lid.p;
        v.car = b_car.p; v.car_pos = b_car_pos.p; v.cls_car = b_cls_car.p; v.cls_slot = b_cls_slot.p; v.cls_rank = b_cls_rank.p;
        v.alt_car = b_alt_car.p;
        v.line_first = b_line_first.p; v.n_car = b_n_car.p; v.n_alt = b_n_alt.p;
        v.line_s = b_line_s.p; v.line_e = b_line_e.p; v.line_len = b_line_len.p; v.line_end = b_line_end.p;
        v.hidx = b_hidx.p; v.cub_tmp = b_cub.p; v.cub_bytes = b_cub.n;
        CK(cudaStreamWaitEvent(s, d.m_up[k], 0));
        CK(cudaEventRecord(ev[3], s));
        CK(launch_vcf_spans(v, s));
        if (ci + 1 < n_chroms && n_rec[ci + 1]) k_cur = upload(ci + 1);      // overlaps this chromosome's kernels
        CK(cudaMemcpyAsync(h_small.p + 3, v.lid + v.n_rec - 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        const uint32_t n_lines = *reinterpret_cast<const uint32_t*>(h_small.p + 3);
        CK(launch_vcf_size(v, n_lines, d.n_sm, s));
        CK(cudaEventRecord(ev[4], s));
        CK(cudaMemcpyAsync(h_line_end.p, v.line_end, n_lines * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        st.span_ms += elapsed(ev[3], ev[4]);
        st.records += v.n_rec;
        const uint64_t* le = h_line_end.p;
        for (uint32_t l = 0; l < n_lines; l++) st.lines += le[l] > (l ? le[l - 1] : 0);
        for (uint32_t l0 = 0; l0 < n_lines;) {
            const uint64_t b0 = l0 ? le[l0 - 1] : 0, hn = hdr_done ? 0 : hdr.size();
            const uint64_t budget = B > hn ? B - hn : 0;
            uint32_t l1 = (uint32_t)(std::upper_bound(le + l0, le + n_lines, b0 + budget) - le);
            if (l1 == l0) l1 = l0 + 1;
            if (le[l1 - 1] > b0 || hn) emit(&v, l0, l1, le[l1 - 1] - b0);
            l0 = l1;
        }
        CK(cudaEventRecord(d.m_done[k], s));
    }
    if (!hdr_done) emit(nullptr, 0, 0, 0);
    sink.settle(d.slot[0].host); sink.settle(d.slot[1].host);
    sink.end_job(0, 1, true);
    quiesce.armed = false;
    struct stat sb;
    if (::stat(P->path, &sb) == 0) st.file_bytes = (uint64_t)sb.st_size;
    st.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_call).count();
    if (stats) *stats = st;
}

}  // namespace

int jlp_write_vcf(jlp_ctx* c, const jlp_vcf_params* p, jlp_vcf_stats* stats) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() { write_vcf(c, device0(c), p, stats); });
}

int jlp_pacbio(jlp_ctx* c, int use_haplotypes, const jlp_pacbio_params* p, jlp_run_stats* stats) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        if (!p || !p->out_prefix || !*p->out_prefix) throw ArgErr("out_prefix is empty");
        Output out(SINK_FILES);
        run_pacbio(c, device0(c), use_haplotypes != 0, p, out, stats);
    });
}

int jlp_pacbio_to_memory(jlp_ctx* c, int use_haplotypes, const jlp_pacbio_params* p, char* out, uint64_t cap, uint64_t* len,
                         jlp_run_stats* stats) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        Output sink(out ? SINK_MEMORY : SINK_NONE);
        sink.mem[0] = out; sink.cap[0] = out ? cap : 0;
        run_pacbio(c, device0(c), use_haplotypes != 0, p, sink, stats);
        if (len) *len = sink.len[0];
        if (out && sink.len[0] > cap) throw ArgErr("output buffer too small");
    });
}

int jlp_pacbio_read_plan(jlp_ctx* c, int use_haplotypes, const jlp_pacbio_params* p, uint64_t* group, uint64_t* read_len,
                         uint64_t* split_pos, double* passes_left, double* passes_right) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        PbModel model;
        pb_model_from(p, model);
        const Layout G = make_layout(c, LayoutSpec(use_haplotypes != 0, p, p->n_reads));
        const Thr t_dup = thr_double_lt(p->prob_dup);
        // chunks of whole pools, as the driver's batches
        const uint64_t pool = std::max<uint64_t>(p->read_pool_size, 1), B = std::max<uint64_t>(pool, 32768 / pool * pool);
        std::vector<PbRead> plan;
        std::vector<PbSample> smp;
        for (const Job& job : G.jobs)
            for (uint64_t b0 = job.lo; b0 < job.hi; b0 += B) {
                const uint32_t n = (uint32_t)std::min(B, job.hi - b0);
                plan.resize(n);
                smp.resize(n);
                pb_plan(model, p->seed, b0, n, job.lo, pool, t_dup, G.group_off, G.groups.data(), p->n_threads, plan.data(), smp.data());
                for (uint32_t i = 0; i < n; i++) {
                    const uint64_t j = b0 + i;
                    if (group) group[j] = plan[i].group;
                    if (read_len) read_len[j] = smp[i].read_length;
                    if (split_pos) split_pos[j] = smp[i].split_pos;
                    if (passes_left) passes_left[j] = smp[i].passes_left;
                    if (passes_right) passes_right[j] = smp[i].passes_right;
                }
            }
    });
}

int jlp_pacbio_sample(const jlp_pacbio_params* p, uint64_t n, uint64_t chrom_len, uint64_t* read_len, uint64_t* split_pos,
                      double* passes_left, double* passes_right) {
    try {
        PbModel model;
        pb_model_from(p, model);
        for (uint64_t j = 0; j < n; j++) {
            const PbSample s = pb_sample(model, p->seed, j, chrom_len);
            if (read_len) read_len[j] = s.read_length;
            if (split_pos) split_pos[j] = s.split_pos;
            if (passes_left) passes_left[j] = s.passes_left;
            if (passes_right) passes_right[j] = s.passes_right;
        }
    } catch (const std::exception& e) { return fail(nullptr, JLP_ERR_ARG, e.what()); }
    return JLP_OK;
}

// ---- host-side pieces (no device) ----

int jlp_deflate(int bgzf, int level, const void* in, uint64_t n, void* out, uint64_t cap, uint64_t* len) {
    if ((!in && n) || !len) return JLP_ERR_ARG;
    std::vector<uint8_t> v;
    std::string e = deflate_members(bgzf ? DEFLATE_BGZF : DEFLATE_GZIP, level, static_cast<const uint8_t*>(in), n, v);
    if (!e.empty()) return JLP_ERR_ARG;
    if (bgzf) v.insert(v.end(), kBgzfEof, kBgzfEof + sizeof kBgzfEof);
    *len = v.size();
    if (!out) return JLP_OK;                 // size query
    if (v.size() > cap) return JLP_ERR_ARG;
    std::memcpy(out, v.data(), v.size());
    return JLP_OK;
}

int jlp_bgzf_device(jlp_ctx* c, int level, const void* in, uint64_t n, void* out, uint64_t cap, uint64_t* len) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        if ((n && !in) || !len) throw ArgErr("NULL argument");
        Device& d = device0(c);
        const uint32_t nblk = (uint32_t)((n + kBgzfIn - 1) / kBgzfIn);
        DevBuf<uint8_t> d_in;
        DevBuf<uint64_t> d_tot;
        Bgzf z;
        d_in.ensure(n + 64); d_tot.ensure(4); z.ensure(nblk, n, 1);
        const uint64_t tot[4] = {n, 0, 0, 0};
        if (n) CK(cudaMemcpyAsync(d_in.p, in, n, cudaMemcpyHostToDevice, d.s_compute));
        CK(cudaMemcpyAsync(d_tot.p, tot, sizeof tot, cudaMemcpyHostToDevice, d.s_compute));
        CK(z.launch(d_in.p, d_in.p, d_tot.p, nblk, level, d.s_compute));
        uint64_t back[4];
        CK(cudaMemcpyAsync(back, d_tot.p, sizeof back, cudaMemcpyDeviceToHost, d.s_compute));
        CK(cudaStreamSynchronize(d.s_compute));
        *len = back[2] + sizeof kBgzfEof;
        if (!out) return;
        if (cap < *len) throw ArgErr("output buffer too small");
        if (back[2]) CK(cudaMemcpy(out, z.out[0].p, back[2], cudaMemcpyDeviceToHost));
        std::memcpy(static_cast<uint8_t*>(out) + back[2], kBgzfEof, sizeof kBgzfEof);
    });
}

int jlp_shard_range(uint64_t job_lo, uint64_t job_hi, uint32_t shard_index, uint32_t shard_count, uint64_t* lo,
                    uint64_t* hi) {
    if (!lo || !hi || job_hi < job_lo || shard_count == 0 || shard_index >= shard_count) return JLP_ERR_ARG;
    shard_range(job_lo, job_hi, shard_index, shard_count, *lo, *hi);
    return JLP_OK;
}

int jlp_apportion(uint64_t seed, uint64_t n_pairs, uint64_t n_haps, uint64_t n_chroms, const double* hap_probs,
                  const uint64_t* sizes, uint64_t* counts) {
    if (!sizes || !counts || n_chroms == 0 || (hap_probs && n_haps == 0)) return JLP_ERR_ARG;
    try {
        std::vector<std::vector<uint64_t>> cnt = apportion_sizes(seed, n_pairs, n_haps, n_chroms, hap_probs, sizes);
        uint64_t k = 0;
        for (const auto& v : cnt) for (uint64_t x : v) counts[k++] = x;
    } catch (const std::exception&) { return JLP_ERR_ARG; }
    return JLP_OK;
}

int jlp_reads_per_group(uint64_t n_reads, const double* probs, uint64_t n, uint64_t seed, uint64_t* out) {
    if (!probs || !out) return JLP_ERR_ARG;
    std::vector<uint64_t> r = reads_per_group(n_reads, std::vector<double>(probs, probs + n), seed);
    std::copy(r.begin(), r.end(), out);
    return JLP_OK;
}
int jlp_transition_matrix(const double Q[16], double t, double P[16]) {
    if (!Q || !P || !(t >= 0) || !std::isfinite(t)) return JLP_ERR_ARG;
    transition_matrix(Q, t, P);
    return JLP_OK;
}
int jlp_alias_build(const double* probs, uint64_t n, double* prob_out, uint64_t* alias_out) {
    if (!probs || !prob_out || !alias_out) return JLP_ERR_ARG;
    alias_build(probs, n, prob_out, alias_out);
    return JLP_OK;
}
int jlp_threshold(int kind, double p, uint64_t* thr, int* all) {
    Thr t;
    if (kind == 1) t = thr_double_lt(p);
    else if (kind == 2) t = thr_double_le(p);
    else if (kind == 3) t = thr_ld_lt(p);
    else if (kind == 11) t = thr_double_lt_x87(p);
    else if (kind == 12) t = thr_double_le_x87(p);
    else if (kind == 13) t = thr_ld_lt_x87(p);
    else return JLP_ERR_ARG;
    if (thr) *thr = t.thr;
    if (all) *all = t.all;
    return JLP_OK;
}
uint64_t jlp_unif_expr(int kind, uint64_t x, double p, uint64_t n) {
    (void)p;
    switch (kind) {
    case 0: return mul_floor_x87(x, n);
    case 4: return nqual_x87(x);
    case 5: {
        double u = (x == ~0ull) ? 1.0 : (double)(x + 1) * 5.421010862427522170037e-20;
        return (uint64_t)(u * (double)n);
    }
    case 6: return ins_base_index(x);
    }
    return 0;
}
int jlp_frag_table(double shape, double scale, uint64_t frag_min, uint64_t frag_max, uint64_t* cdf, uint64_t cap,
                   uint64_t* n) {
    std::vector<uint64_t> t = frag_table(shape, scale, frag_min, frag_max);
    if (n) *n = t.size();
    if (t.size() > cap) return JLP_ERR_ARG;
    if (cdf) std::copy(t.begin(), t.end(), cdf);
    return JLP_OK;
}
void jlp_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
    U4 w = philox4x32_10(ctr[0], ctr[1], ctr[2], ctr[3], key[0], key[1]);
    out[0] = w.w0; out[1] = w.w1; out[2] = w.w2; out[3] = w.w3;
}
uint64_t jlp_draw_pos(uint64_t seed, uint64_t j, uint32_t end, uint32_t purpose, uint32_t pos) {
    if (high_bits(purpose) == 0) return slow64(seed, j, end, purpose, pos);
    U4 w = purpose == PU_INDEL ? draw_block(seed, j, pos >> 3, PL_INDEL, end) : draw_block(seed, j, pos >> 1, PL_QUAL, end);
    return full_draw(high_of(w, purpose, pos), seed, j, end, purpose, pos);
}
uint64_t jlp_genome_draw(uint64_t seed, uint32_t chrom, uint64_t pos, int which) {
    return genome_draw(seed, chrom, pos, (uint32_t)which);
}
uint64_t jlp_draw_pair(uint64_t seed, uint64_t j, int which) {
    U4 w = draw_block(seed, j, (uint32_t)(which >> 1), PL_PAIR, 0);
    return (which & 1) ? hi64(w) : lo64(w);
}

const char* jlp_version(void) { return "jackalope-b200 0.1 (sm_100a)"; }

}  // extern "C"
