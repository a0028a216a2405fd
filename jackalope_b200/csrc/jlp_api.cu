// C ABI (include/jlp_b200.h): context, genome / haplotype / profile upload, and
// the batch pipeline that stands in for write_reads_cpp_ / write_reads_cpp_sep_files_
// / write_reads_one_filetype_ (/root/reference/src/hts.h:323-552).
#include "../../include/jlp_b200.h"

#include <cuda_runtime.h>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/statvfs.h>
#include <unistd.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <cerrno>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <deque>
#include <functional>
#include <mutex>
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
#include "jlp_pacbio.h"

using namespace jlp;

namespace {

std::string g_create_error;

// Bytes of padding in front of and behind every sequence allocation: the read kernel
// fetches template bases as aligned words and may touch a few bytes outside a chromosome.
constexpr size_t kPad = 64;

struct CudaErr : std::runtime_error {
    explicit CudaErr(const std::string& m) : std::runtime_error(m) {}
};
struct ArgErr : std::runtime_error {
    explicit ArgErr(const std::string& m) : std::runtime_error(m) {}
};
struct IoErr : std::runtime_error {
    explicit IoErr(const std::string& m) : std::runtime_error(m) {}
};
struct Unsupported : std::runtime_error {
    explicit Unsupported(const std::string& m) : std::runtime_error(m) {}
};
struct Aborted : std::runtime_error {
    Aborted() : std::runtime_error("aborted by user") {}
};

#define CK(call)                                                                          \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess)                                                            \
            throw CudaErr(std::string(#call) + ": " + cudaGetErrorString(e_));            \
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

// Host writer threads: the FASTQ of a batch sits in a pinned buffer; its slices are written
// with pwrite() at their final file offsets while the GPU generates and copies the next
// batch (the reference's threads serialise on one omp critical per pool instead,
// src/hts.h:401-416).
class WriterPool {
public:
    // a task returns an error text (empty = fine); `pending` counts the tasks of one batch slot
    struct Task { std::function<std::string()> run; std::atomic<int>* pending; };
    ~WriterPool() { stop(); }
    void start(size_t n_threads) {
        if (th.size() == n_threads) return;
        stop();
        quit = false;
        for (size_t i = 0; i < n_threads; i++) th.emplace_back([this]() { loop(); });
    }
    void stop() {
        { std::lock_guard<std::mutex> l(m); quit = true; }
        cv.notify_all();
        for (std::thread& t : th) t.join();
        th.clear();
    }
    void submit(std::atomic<int>* pending, std::function<std::string()> f) {
        pending->fetch_add(1);
        { std::lock_guard<std::mutex> l(m); q.push_back(Task{std::move(f), pending}); }
        cv.notify_one();
    }
    // wait until every task counted by `pending` is done; returns the first error text (empty = none)
    std::string wait(std::atomic<int>& pending) {
        std::unique_lock<std::mutex> l(m);
        cv_done.wait(l, [&]() { return pending.load() == 0; });
        return err;
    }
    void clear_error() { std::lock_guard<std::mutex> l(m); err.clear(); }
private:
    void loop() {
        for (;;) {
            Task t;
            {
                std::unique_lock<std::mutex> l(m);
                cv.wait(l, [&]() { return quit || !q.empty(); });
                if (q.empty()) return;
                t = std::move(q.front()); q.pop_front();
            }
            std::string e = t.run();
            {
                std::lock_guard<std::mutex> l(m);
                if (!e.empty() && err.empty()) err = e;
                t.pending->fetch_sub(1);
            }
            cv_done.notify_all();
        }
    }
    std::vector<std::thread> th;
    std::mutex m;
    std::condition_variable cv, cv_done;
    std::deque<Task> q;
    std::string err;
    bool quit = false;
};

std::string pwrite_all(int fd, const uint8_t* p, uint64_t n, uint64_t off) {
    while (n) {
        ssize_t w = ::pwrite(fd, p, n > (1u << 30) ? (1u << 30) : n, (off_t)off);
        if (w < 0) { if (errno == EINTR) continue; return std::strerror(errno); }
        p += w; n -= (uint64_t)w; off += (uint64_t)w;
    }
    return std::string();
}

// Files are also written through shared mappings: the main thread extends the file by a batch and maps the new
// range once, the writer threads copy their slices into the mapping (page-cache pages are allocated and filled by
// the copying thread, so the threads do not queue on the inode lock that serialises write() calls on one file;
// measured on the B200 box's tmpfs: 7.4 GB/s with pwrite from any number of threads, 14 GB/s with 16 threads
// copying into mappings, tools/write_probe.cpp), and the range is unmapped when the batch's slices are done --
// one munmap per batch and file, not one TLB shoot-down per slice.
struct Mapping {
    void* base = nullptr;
    size_t len = 0;
    uint8_t* at = nullptr;      // where the batch's first byte goes
    void unmap() { if (base) ::munmap(base, len); base = nullptr; len = 0; at = nullptr; }
};
bool map_range(int fd, uint64_t off, uint64_t n, Mapping& m) {
    static const uint64_t page = (uint64_t)sysconf(_SC_PAGESIZE);
    const uint64_t a0 = off / page * page;
    void* p = ::mmap(nullptr, (size_t)(off + n - a0), PROT_READ | PROT_WRITE, MAP_SHARED, fd, (off_t)a0);
    if (p == MAP_FAILED) return false;
    m.base = p; m.len = (size_t)(off + n - a0); m.at = static_cast<uint8_t*>(p) + (off - a0);
    return true;
}

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
struct HapDev {
    std::shared_ptr<HapStore> store;    // shared by the devices of a multi-GPU context
    std::vector<const uint8_t*> seq;    // per chromosome; aliases the reference when unmutated; NULL = not materialised yet
    std::vector<uint64_t> len;
    const std::string& name() const { return store->name; }
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

struct Slot {
    DevBuf<uint8_t> out[2];
    DevBuf<EndPlan> plan;
    DevBuf<uint32_t> rec_len, rec_local;
    DevBuf<uint64_t> block_tot, block_base, totals;
    PinBuf<uint8_t> h_out[2];
    PinBuf<uint64_t> h_totals;
    // device BGZF: one 64 KiB slot per block, the members' sizes and offsets, the contiguous compressed batch
    DevBuf<uint8_t> zslots[2], zdev[2];
    DevBuf<uint32_t> zlen[2];
    DevBuf<uint64_t> zoff[2];
    DevBuf<uint8_t> zcode;        // launch_bgzf's scratch (the codes of the batch)
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // start, placed, scanned, reads done, copied, all kernels done
    uint32_t pairs = 0;
    uint64_t tot[2] = {0, 0};     // FASTQ bytes of the batch per file (read back from the device)
    uint64_t ztot[2] = {0, 0};    // compressed bytes of the batch per file (device BGZF)
    bool busy = false;
    std::atomic<int> writes{0};   // slices of h_out still being written to / compressed for the files
    std::vector<std::vector<uint8_t>> zout[2];   // compressed slices of the batch, in file order
    Mapping map[2];               // the file ranges this batch is being copied into
    uint64_t file_end[2] = {0, 0};  // where this batch ends in the files (plain FASTQ)
};

}  // namespace

struct jlp_ctx {
    int device = 0;
    // a multi-GPU context (jlp_ctx_create_multi) owns one child context per device and no device state of its own:
    // it keeps the genome / haplotype metadata (names, sizes) and fans every call out to its children
    std::vector<jlp_ctx*> kids;
    std::string err;
    cudaStream_t s_compute = nullptr, s_copy = nullptr;
    // genome
    DevBuf<uint8_t> genome;
    std::vector<uint64_t> chrom_off;
    std::vector<std::string> chrom_names;
    std::string genome_name;
    std::vector<HapDev> haps;
    // profiles
    EndTables tab[2];
    bool have_prof[2] = {false, false};
    DevBuf<uint32_t> d_meta[2];
    DevBuf<uint64_t> d_coin[2], d_mis[2], d_entry64[2];
    int n_sm = 148;
    // run-scoped device data
    DevBuf<uint64_t> d_frag, d_group_off;
    DevBuf<uint32_t> d_frag_guide;
    DevBuf<GroupDev> d_groups;
    DevBuf<uint8_t> d_strpool;
    DevBuf<uint32_t> d_status;
    Slot slot[3];                               // compute | D2H copy | delivery to the sink, one batch each
    WriterPool writers;
    cudaStream_t s_upload = nullptr;            // genome H2D, chromosome by chromosome
    std::vector<cudaEvent_t> chrom_ev;          // chromosome c is resident once chrom_ev[c] has fired
    bool upload_pending = false;                // some chromosome is not resident yet (or its copy not waited for)
    const char* upload_src = nullptr;           // host bases of a deferred upload (jlp_set_genome_async), else NULL
    std::vector<char> chrom_resident;           // 1: the chromosome's H2D copy has been issued
    cudaEvent_t ev_run[2] = {nullptr, nullptr};
    uint64_t h2d_bytes = 0;
    // scratch of the haplotype materialisation (mutation records of one chromosome)
    HapArena hap_mem;
    // PacBio driver: FASTQ of a batch on the device, its compressed form, and the two pinned host buffers batches alternate between
    DevBuf<uint8_t> pb_out, pb_zslots, pb_zout, pb_strpool, pb_zcode;
    DevBuf<PbRead> pb_reads;
    DevBuf<GroupDev> pb_groups;
    DevBuf<uint32_t> pb_rec_len, pb_rec_local, pb_zlen;
    DevBuf<uint64_t> pb_block_tot, pb_block_base, pb_totals, pb_zoff;
    PinBuf<uint8_t> pb_h_buf[2];
    // PacBioPassSampler's outlier thresholds (one chi-squared quantile per read length up to chi2_params_n[2]) of the last call
    std::shared_ptr<std::atomic<double>[]> pb_qcache;
    double pb_qcache_key[3] = {0, 0, 0};
    size_t pb_qcache_n = 0;
    // materialisation: the records of the next chromosomes are uploaded (s_upload) while k_materialize works on the
    // ones before (s_compute); kMatBufs scratch buffers in turn
    static constexpr int kMatBufs = 3;
    DevBuf<uint64_t> m_pack[kMatBufs];
    cudaEvent_t m_up[kMatBufs] = {nullptr, nullptr, nullptr}, m_done[kMatBufs] = {nullptr, nullptr, nullptr};
    bool m_busy[kMatBufs] = {false, false, false};
    uint64_t m_next = 0;
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

void free_haps(jlp_ctx* c) {
    c->haps.clear();
    c->hap_mem.release();
}

int fail(jlp_ctx* c, int code, const std::string& msg) {
    if (c) c->err = msg; else g_create_error = msg;
    return code;
}

template <typename F> int guarded(jlp_ctx* c, F f) {
    try {
        if (c && c->kids.empty()) CK(cudaSetDevice(c->device));
        f();
        return JLP_OK;
    } catch (const ArgErr& e) { return fail(c, JLP_ERR_ARG, e.what());
    } catch (const CudaErr& e) { return fail(c, JLP_ERR_CUDA, e.what());
    } catch (const IoErr& e) { return fail(c, JLP_ERR_IO, e.what());
    } catch (const Unsupported& e) { return fail(c, JLP_ERR_UNSUPPORTED, e.what());
    } catch (const Aborted& e) { return fail(c, JLP_ERR_ABORTED, e.what());
    } catch (const std::exception& e) { return fail(c, JLP_ERR_ARG, e.what()); }
}

// the context itself, or the first child of a multi-GPU context (made current): calls that do not spread over devices
jlp_ctx* first_device(jlp_ctx* c) {
    if (c->kids.empty()) return c;
    CK(cudaSetDevice(c->kids[0]->device));
    return c->kids[0];
}
// f(device context) for the context itself, or for every child of a multi-GPU context (current device set)
template <typename F> void for_each_device(jlp_ctx* c, F f) {
    if (c->kids.empty()) { f(c); return; }
    for (jlp_ctx* k : c->kids) { CK(cudaSetDevice(k->device)); f(k); }
}
// the same, one host thread per device; the first error (if any) is rethrown as a runtime_error of its text
template <typename F> void for_each_device_parallel(jlp_ctx* c, F f) {
    if (c->kids.size() <= 1) { for_each_device(c, f); return; }
    std::vector<std::string> errs(c->kids.size());
    std::vector<std::thread> th;
    for (size_t r = 0; r < c->kids.size(); r++)
        th.emplace_back([&, r]() {
            try { CK(cudaSetDevice(c->kids[r]->device)); f(c->kids[r]); } catch (const std::exception& e) { errs[r] = e.what(); if (errs[r].empty()) errs[r] = "error"; }
        });
    for (std::thread& t : th) t.join();
    for (const std::string& e : errs) if (!e.empty()) throw CudaErr(e);
}

// Issue the H2D copies of chromosomes [first, last] of a deferred genome upload (those not
// issued yet); every copy is followed by its chromosome's event.
void issue_upload(jlp_ctx* c, size_t first, size_t last) {
    if (!c->upload_src) return;
    for (size_t i = first; i <= last && i < c->chrom_resident.size(); i++) {
        if (c->chrom_resident[i]) continue;
        const uint64_t len = c->chrom_off[i + 1] - c->chrom_off[i];
        if (len) CK(cudaMemcpyAsync(c->genome.p + kPad + c->chrom_off[i], c->upload_src + c->chrom_off[i], len, cudaMemcpyHostToDevice, c->s_upload));
        CK(cudaEventRecord(c->chrom_ev[i], c->s_upload));
        c->chrom_resident[i] = 1;
        c->h2d_bytes += len;
    }
}
// Make the whole genome resident and wait for it.
void finish_upload(jlp_ctx* c) {
    if (!c->upload_pending) return;
    if (!c->chrom_resident.empty()) issue_upload(c, 0, c->chrom_resident.size() - 1);
    CK(cudaStreamSynchronize(c->s_upload));
    c->upload_pending = false;
    c->upload_src = nullptr;
}

// ---------------------------------------------------------------- the run ---

enum SinkKind { SINK_FILES, SINK_MEMORY, SINK_STREAM, SINK_NONE };

struct Sink {
    SinkKind kind = SINK_NONE;
    // memory
    char* mem[2] = {nullptr, nullptr};
    uint64_t cap[2] = {0, 0}, len[2] = {0, 0};
    // stream
    jlp_chunk_cb chunk_cb = nullptr;
    void* chunk_user = nullptr;
    // files
    int fd[2] = {-1, -1};
    uint64_t pos[2] = {0, 0};        // where the next batch goes
    uint64_t done[2] = {0, 0};       // end of the last batch known to be completely written (error paths truncate back to it)
    bool own_size[2] = {false, false};   // this call extends the file itself (not a pre-sized file shared with other devices)
    std::string names[2];
    void close_files() {
        for (int e = 0; e < 2; e++) if (fd[e] >= 0) { ::close(fd[e]); fd[e] = -1; }
    }
    ~Sink() { close_files(); }
};

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

// needs only the sizes: works on a multi-GPU parent context (metadata, no device state) as well
std::vector<std::vector<uint64_t>> apportion(const jlp_ctx* c, bool use_haps, const jlp_illumina_params* P, uint64_t n_pairs) {
    const uint64_t n_chroms = c->chrom_off.size() - 1;
    std::vector<uint64_t> sizes;
    if (!use_haps) {
        for (uint64_t i = 0; i < n_chroms; i++) sizes.push_back(c->chrom_off[i + 1] - c->chrom_off[i]);
        return apportion_sizes(P->seed, n_pairs, 1, n_chroms, nullptr, sizes.data());
    }
    if (!P->haplotype_probs) throw ArgErr("haplotype_probs is NULL");
    for (const HapDev& h : c->haps) sizes.insert(sizes.end(), h.len.begin(), h.len.end());
    return apportion_sizes(P->seed, n_pairs, c->haps.size(), n_chroms, P->haplotype_probs, sizes.data());
}

// How a run's compressed output is produced (write_reads_cpp_, src/hts.h:441-500): compressed + one thread -> the
// method asked for; compressed + several threads -> always bgzip (the reference writes plain files first and bgzips
// them afterwards; here the batches are compressed on their way to the file).  comp_engine picks who compresses:
// the device coder (BGZF members of one dynamic-Huffman block each, jlp_bgzf.cu; only compressed bytes cross PCIe)
// or zlib on the writer threads at the level asked for.  AUTO uses the device coder only where the reference itself
// would write BGZF (comp_method "bgzip", or several threads) at levels 1..6; a gzip request with one thread is a
// gzip stream from zlib (FileGZ, src/io.h:140-236).  Memory and stream sinks receive compressed bytes only when the
// device coder is asked for explicitly.
struct Compression {
    bool dev_z = false;       // BGZF on the device
    int zmethod = -1;         // host zlib: DEFLATE_BGZF / DEFLATE_GZIP; -1 = none
    bool want_gz = false;     // file names get ".gz"
};
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
    if (P->compress > 0) {
        std::string m = P->comp_method ? P->comp_method : "";
        if (m != "gzip" && m != "bgzip") throw ArgErr("\nUnrecognized compression method.");  // src/hts.h:470
        if (P->compress > 9) throw ArgErr("\nInvalid bgzip compress level of " + std::to_string(P->compress) +
                                          ". It must be in range [0,9].");                   // src/io.h:113-117
    }
    if (P->comp_engine < JLP_COMP_AUTO || P->comp_engine > JLP_COMP_DEVICE) throw ArgErr("comp_engine must be 0 (auto), 1 (host) or 2 (device)");
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
// jobs (= sets of output files).  A pure function of the parameters and of the sizes the context knows, so every
// device of a multi-GPU run builds the same one.
struct Layout {
    int n_ends = 1;
    uint64_t n_pairs = 0;
    std::vector<uint64_t> group_off;      // [n_groups + 1]
    std::vector<GroupDev> groups;         // seq is filled in per device
    std::vector<uint32_t> group_hap, group_chrom;
    std::vector<uint8_t> strpool;
    std::vector<Job> jobs;
};

Layout make_layout(const jlp_ctx* c, bool use_haps, const jlp_illumina_params* P) {
    Layout Y;
    Y.n_ends = P->paired || P->matepair ? 2 : 1;
    const uint32_t L = (uint32_t)c->tab[0].L;
    const uint64_t n_haps = c->haps.size(), n_chroms = c->chrom_off.size() - 1;
    const bool sep = use_haps && P->sep_files;
    // --- barcodes (T/C/A/G only, R/hts_illumina.R:385-391)
    std::vector<std::string> barcodes(use_haps ? n_haps : 1);
    if (P->barcodes)
        for (size_t i = 0; i < barcodes.size(); i++) barcodes[i] = P->barcodes[i] ? P->barcodes[i] : "";
    for (const std::string& bcs : barcodes) {
        for (char ch : bcs)
            if (ch != 'T' && ch != 'C' && ch != 'A' && ch != 'G') throw ArgErr("barcodes may only contain T, C, A, G");
        if (bcs.size() >= L) throw ArgErr("a barcode is as long as the read");
    }
    // --- apportion pairs: threads -> haplotypes -> chromosomes
    //     (write_reads_one_filetype_ src/hts.h:334-353, add_n_reads src/hts_illumina.h:410-418, :620-644,
    //      write_reads_cpp_sep_files_ src/hts.h:527-529); one "thread", n_pairs = floor(n_reads / n_ends)
    Y.n_pairs = P->n_reads / Y.n_ends;
    const std::vector<std::vector<uint64_t>> counts = apportion(c, use_haps, P, Y.n_pairs);
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
    const std::string prefix = P->out_prefix ? P->out_prefix : "";
    if (!use_haps) {
        for (uint64_t i = 0; i < n_chroms; i++)
            add_group(c->genome_name, 0, i, c->chrom_off[i + 1] - c->chrom_off[i], barcodes[0], counts[0][i]);
        Y.jobs.push_back(Job{0, Y.n_pairs, prefix});
    } else {
        for (uint64_t h = 0; h < n_haps; h++) {
            const HapDev& H = c->haps[h];
            uint64_t lo = Y.group_off.back();
            for (uint64_t i = 0; i < n_chroms; i++) add_group(H.name(), (uint32_t)h, i, H.len[i], barcodes[h], counts[h][i]);
            if (sep) Y.jobs.push_back(Job{lo, Y.group_off.back(), prefix + "_" + H.name()});
        }
        if (!sep) Y.jobs.push_back(Job{0, Y.group_off.back(), prefix});
    }
    if (Y.group_off.back() != Y.n_pairs) throw std::runtime_error("internal: apportioning does not add up");
    return Y;
}

// name of output file `e` of a job (src/hts.h:344; ".gz" appended by FileGZ / FileBGZF, src/io.h:126,217).
// A process that generates one shard of a run (shard_count > 1, one process per GPU) writes its own files,
// <prefix>[_<hap>]_R<k>.fq[.gz].shard<i>of<n>: concatenated in shard order they are the unsharded run's file.
std::string file_name(const Job& job, int e, bool gz, const jlp_illumina_params* P) {
    std::string n = job.file_prefix + "_R" + std::to_string(e + 1) + ".fq";
    if (gz) n += ".gz";
    if (P->shard_count > 1) n += ".shard" + std::to_string(P->shard_index) + "of" + std::to_string(P->shard_count);
    return n;
}

// Materialise haplotype chromosome (h, ci) on this context's device if it is not resident yet
// (HapChrom::get_chrom_full, src/hap_classes.cpp:80-116).
void ensure_hap_chrom(jlp_ctx* c, size_t h, size_t ci) {
    HapDev& H = c->haps[h];
    if (H.seq[ci]) return;
    const HapChromHost& M = H.store->chrom[ci];
    const uint64_t ref_size = c->chrom_off[ci + 1] - c->chrom_off[ci];
    const uint8_t* ref = c->genome.p + kPad + c->chrom_off[ci];
    const int k = (int)(c->m_next++ % jlp_ctx::kMatBufs);
    if (!c->m_up[k]) {
        CK(cudaEventCreateWithFlags(&c->m_up[k], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&c->m_done[k], cudaEventDisableTiming));
    }
    // the kernel that read this buffer last must be done before the buffer can grow (cudaFree) or be written again
    if (c->m_busy[k]) CK(cudaEventSynchronize(c->m_done[k]));
    c->m_pack[k].upload(M.packed, c->s_upload);
    CK(cudaEventRecord(c->m_up[k], c->s_upload));
    c->h2d_bytes += M.n_muts * 32 + M.pool_bytes;
    uint8_t* out = c->hap_mem.alloc(M.size + 2 * kPad);
    const uint64_t* w = c->m_pack[k].p;
    const uint64_t n = M.n_muts;
    CK(cudaStreamWaitEvent(c->s_compute, c->m_up[k], 0));
    CK(launch_materialize(ref, ref_size, n, w, w + n, reinterpret_cast<const int64_t*>(w + 3 * n), w + 2 * n,
                          reinterpret_cast<const uint8_t*>(w + 4 * n), M.size, out + kPad, c->s_compute));
    CK(cudaEventRecord(c->m_done[k], c->s_compute));
    c->m_busy[k] = true;
    H.seq[ci] = out + kPad;       // valid in stream order: everything that reads it runs on s_compute
}

typedef std::vector<std::pair<uint64_t, uint64_t>> Ranges;
typedef std::vector<std::array<uint64_t, 2>> PerJobBytes;

// What a multi-GPU run tells each of its devices (jlp_ctx_create_multi); a plain call leaves everything empty.
struct RunExtras {
    const Ranges* ranges = nullptr;       // [jobs] the pair range of every job this call generates (else: the shard of P)
    PerJobBytes* sizes_out = nullptr;     // size pass: only count the FASTQ bytes per job and end of those ranges
    const PerJobBytes* base = nullptr;    // [jobs] where this call's bytes start in each job's files / in the memory sink
    bool shared_files = false;            // the files exist, created and sized by the caller: open without truncating, no EOF block
    std::string part_suffix;              // compressed multi-GPU runs: this call writes <name><suffix>, joined by the caller
    bool no_eof = false;                  // ... and the caller appends the BGZF end-of-file block
    const std::vector<std::string>* job_suffix = nullptr;   // [jobs] the same per job (overrides part_suffix)
    PerJobBytes* zsizes_out = nullptr;    // the compressed bytes per job and end this call produced (device coder)
    bool dry_files = false;               // generate and compress as for files, deliver nothing (sink NONE): the compressed size pass
};

void run(jlp_ctx* c, bool use_haps, const jlp_illumina_params* P, Sink& sink, jlp_run_stats* stats, const RunExtras& X = RunExtras()) {
    check_params(c, use_haps, P, sink.kind);
    const int n_ends = P->paired || P->matepair ? 2 : 1;
    const bool matepair = P->matepair != 0;
    if (use_haps) finish_upload(c);
    const uint64_t h2d_before = c->h2d_bytes;
    const Compression Z = compression_of(P, X.dry_files ? SINK_FILES : sink.kind);
    const bool dev_z = Z.dev_z, want_gz = Z.want_gz;
    const int zmethod = Z.zmethod;
    const bool sizes_only = X.sizes_out != nullptr;
    if (X.zsizes_out) X.zsizes_out->assign(X.ranges ? X.ranges->size() : 0, std::array<uint64_t, 2>{0, 0});
    const double insp[2] = {P->ins_prob1, P->ins_prob2}, delp[2] = {P->del_prob1, P->del_prob2};
    const uint32_t L = (uint32_t)c->tab[0].L;

    Layout Y = make_layout(c, use_haps, P);
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
        for (size_t g = 0; g < groups.size(); g++) groups[g].seq = c->genome.p + kPad + c->chrom_off[g];
    } else {
        for (size_t k = 0; k < jobs.size(); k++) {
            if (ranges[k].second <= ranges[k].first) continue;
            size_t g_lo, g_hi;
            groups_of(jobs[k], ranges[k].first, ranges[k].second, g_lo, g_hi);
            for (size_t g = g_lo; g <= g_hi; g++) ensure_hap_chrom(c, Y.group_hap[g], Y.group_chrom[g]);
        }
        for (size_t g = 0; g < groups.size(); g++) groups[g].seq = c->haps[Y.group_hap[g]].seq[Y.group_chrom[g]];
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
        E.meta = c->d_meta[e].p; E.entry64 = c->d_entry64[e].p; E.coin = c->d_coin[e].p;
        E.mis = c->d_mis[e].p;
        E.entry_n = (uint32_t)c->tab[e].entry64.size();
        Thr ta = thr_double_le(insp[e] + delp[e]);   // u > ins + del  <=>  x >= tA
        Thr ti = thr_double_le(insp[e]);             // u > ins        <=>  x >= tI
        E.tA = ta.thr; E.tA_all = ta.all; E.tI = ti.thr; E.tI_all = ti.all;
        E.hA = ta.all ? 0x10000u : (uint32_t)(ta.thr >> 48);
    }
    for (cudaEvent_t& ev : c->ev_run) if (!ev) CK(cudaEventCreate(&ev));
    CK(cudaEventRecord(c->ev_run[0], c->s_compute));
    std::vector<uint64_t> frag = frag_table(P->frag_len_shape, P->frag_len_scale, P->frag_len_min, P->frag_len_max);
    std::vector<uint32_t> guide = frag_guide(frag);
    c->d_frag.upload(frag, c->s_compute);
    c->d_frag_guide.upload(guide, c->s_compute);
    c->d_group_off.upload(group_off, c->s_compute);
    c->d_groups.upload(groups, c->s_compute);
    c->d_strpool.upload(Y.strpool, c->s_compute);
    c->d_status.ensure(1);
    CK(cudaMemsetAsync(c->d_status.p, 0, sizeof(uint32_t), c->s_compute));
    c->h2d_bytes += frag.size() * 8 + group_off.size() * 8 + groups.size() * sizeof(GroupDev) + Y.strpool.size();
    gp.frag_cdf = c->d_frag.p; gp.frag_guide = c->d_frag_guide.p; gp.frag_n = (uint32_t)frag.size(); gp.frag_min = P->frag_len_min;
    gp.group_off = c->d_group_off.p; gp.n_groups = (uint32_t)groups.size();
    gp.groups = c->d_groups.p; gp.strpool = c->d_strpool.p; gp.status = c->d_status.p;

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
    const uint32_t nblk_all = (uint32_t)((B * max_rec + kBgzfIn - 1) / kBgzfIn) + 1;
    const uint32_t nblk_max = dev_z && !sizes_only ? nblk_all : 0;
    for (Slot& s : c->slot) {
        s.plan.ensure(n_rec_max);
        s.rec_len.ensure(n_rec_max);
        s.rec_local.ensure(n_rec_max);
        s.block_tot.ensure((size_t)nsb_max * 2);
        s.block_base.ensure((size_t)nsb_max * 2);
        s.totals.ensure(4);
        s.h_totals.ensure(4);
        CK(cudaMemsetAsync(s.totals.p, 0, 4 * sizeof(uint64_t), c->s_compute));
        for (int e = 0; e < n_ends && !sizes_only; e++) {
            s.out[e].ensure(B * max_rec + 64);
            // compressed bytes of a batch never exceed its FASTQ bytes plus the members' framing (an incompressible block is stored)
            // (the same size with and without compression: pinning a gigabyte again for the first compressed call took seconds)
            if (need_host) s.h_out[e].ensure(B * max_rec + (size_t)nblk_all * 64 + 64);
        }
        if (dev_z && !sizes_only)
            for (int e = 0; e < 2; e++) {
                s.zslots[e].ensure((size_t)nblk_max * kBgzfSlot);
                s.zdev[e].ensure(B * max_rec + (size_t)nblk_max * 64 + 64);
                s.zlen[e].ensure(nblk_max);
                s.zoff[e].ensure(nblk_max);
                s.zcode.ensure(kBgzfCodeBytes);
            }
        for (cudaEvent_t& ev : s.ev) if (!ev) CK(cudaEventCreate(&ev));
        s.busy = false;
    }

    jlp_run_stats st;
    std::memset(&st, 0, sizeof st);

    // If the run ends by an exception, nothing of it may stay in flight: kernels and copies still use the
    // slots, writer tasks still hold the file descriptors the caller's Sink is about to close.  Files this call
    // extends itself are cut back to the last completely written batch (an extended, never filled tail would
    // otherwise stay behind as zero bytes).
    struct Quiesce {
        jlp_ctx* c;
        Sink* sink;
        bool armed = true;
        ~Quiesce() {
            if (!armed) return;
            cudaStreamSynchronize(c->s_compute);
            cudaStreamSynchronize(c->s_copy);
            for (Slot& s : c->slot) {
                c->writers.wait(s.writes);
                for (Mapping& m : s.map) m.unmap();
                s.busy = false;
                s.zout[0].clear(); s.zout[1].clear();
            }
            c->writers.clear_error();
            if (sink->kind == SINK_FILES)
                for (int e = 0; e < 2; e++)
                    if (sink->fd[e] >= 0 && sink->own_size[e] && ::ftruncate(sink->fd[e], (off_t)sink->done[e]) != 0) { /* best effort */ }
        }
    } quiesce{c, &sink};

    auto wait_writes = [&](Slot& s) {
        if (sink.kind != SINK_FILES) return;
        std::string e = c->writers.wait(s.writes);
        for (Mapping& m : s.map) m.unmap();
        if (!e.empty()) { c->writers.clear_error(); throw IoErr("Error writing to file " + sink.names[0] + " / " + sink.names[1] + ": " + e); }
        // compressed slices of the slot's batch go to the files in order
        for (int k = 0; k < n_ends; k++) {
            for (std::vector<uint8_t>& v : s.zout[k]) {
                std::string w = pwrite_all(sink.fd[k], v.data(), v.size(), sink.pos[k]);
                if (!w.empty()) throw IoErr("Error writing to file " + sink.names[k] + ": " + w);
                sink.pos[k] += v.size();
            }
            s.zout[k].clear();
            if (s.file_end[k] > sink.done[k]) sink.done[k] = s.file_end[k];
            if (zmethod >= 0) sink.done[k] = sink.pos[k];
        }
    };
    if (sink.kind == SINK_FILES && !sizes_only) c->writers.start((size_t)std::min<uint64_t>(std::max<uint64_t>(P->n_threads, 1), 64));
    uint64_t job_index = 0;
    Slot* z_pending = nullptr;      // the batch whose compressed slices are not in the files yet
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
        if (z_pending == &s) { wait_writes(s); z_pending = nullptr; }
        wait_writes(s);                         // the pinned buffers of this slot are free again
        for (int e = 0; e < n_ends; e++) {
            const uint64_t nb = dev_z ? s.ztot[e] : s.tot[e];
            CK(cudaMemcpyAsync(s.h_out[e].p, dev_z ? s.zdev[e].p : s.out[e].p, nb, cudaMemcpyDeviceToHost, c->s_copy));
            st.d2h_bytes += nb;
        }
        CK(cudaEventRecord(s.ev[4], c->s_copy));
    };
    // stage 3: the copy has landed -> hand the batch to the sink
    auto deliver = [&](Slot& s) {
        if (need_host) {
            CK(cudaEventSynchronize(s.ev[4]));
            if (zmethod >= 0 && z_pending) { wait_writes(*z_pending); z_pending = nullptr; }   // files stay in batch order
            for (int e = 0; e < n_ends; e++) {
                const uint64_t n = dev_z ? s.ztot[e] : s.tot[e];
                s.file_end[e] = 0;
                if (sink.kind == SINK_FILES && zmethod < 0) {
                    // R1 and R2 stay record-aligned: both files receive the same batches in the same order.
                    // With several writer threads the file is extended and the batch's range mapped; ONE task per file
                    // reserves the range's pages (posix_fallocate: a full file system is an error in that task, not a
                    // SIGBUS later) and then hands the 8 MiB slices to the pool, which copies them into the mapping.
                    // Page allocation is what the kernel serialises per file and it costs more than the copy, so it
                    // must neither sit on the driver thread nor be fought over by all the writers (tools/fill_probe.cpp,
                    // tools/files_probe.py; tmpfs, 16 threads: reserved by the driver thread 11.1 GB/s, by every writer
                    // for its own slice 8.5, by page faults in the copies 9.2, this way 13.3).
                    // With one thread, or when the range cannot be mapped, plain pwrite.
                    bool mapped = P->n_threads > 1 && n > 0;
                    if (mapped) {
                        if (sink.own_size[e]) mapped = ::ftruncate(sink.fd[e], (off_t)(sink.pos[e] + n)) == 0;
                        mapped = mapped && map_range(sink.fd[e], sink.pos[e], n, s.map[e]);
                    }
                    const uint64_t slice = 8ull << 20;
                    if (mapped) {
                        const int fd = sink.fd[e];
                        const uint8_t* src0 = s.h_out[e].p;
                        uint8_t* dst0 = s.map[e].at;
                        const uint64_t off0 = sink.pos[e];
                        WriterPool* pool = &c->writers;
                        std::atomic<int>* pend = &s.writes;
                        c->writers.submit(&s.writes, [fd, src0, dst0, off0, n, slice, pool, pend]() {
                            const int rc = ::posix_fallocate(fd, (off_t)off0, (off_t)n);
                            if (rc != 0 && rc != EOPNOTSUPP && rc != EINVAL) return std::string(std::strerror(rc));
                            for (uint64_t o = 0; o < n; o += slice) {
                                uint8_t* dst = dst0 + o;
                                const uint8_t* src = src0 + o;
                                const uint64_t len = std::min(slice, n - o);
                                pool->submit(pend, [dst, src, len]() { std::memcpy(dst, src, len); return std::string(); });
                            }
                            return std::string();
                        });
                    } else {
                        for (uint64_t o = 0; o < n; o += slice) {
                            const int fd = sink.fd[e];
                            const uint8_t* src = s.h_out[e].p + o;
                            const uint64_t len = std::min(slice, n - o), off = sink.pos[e] + o;
                            c->writers.submit(&s.writes, [fd, src, len, off]() { return pwrite_all(fd, src, len, off); });
                        }
                    }
                    sink.pos[e] += n;
                    s.file_end[e] = sink.pos[e];
                } else if (sink.kind == SINK_FILES) {
                    // compressed: the writer threads deflate slices of whole members; their output is
                    // written in order once the batch is done (wait_writes)
                    const uint64_t unit = zmethod == DEFLATE_BGZF ? 0xff00ull : (1ull << 20);
                    const uint64_t slice = unit * (zmethod == DEFLATE_BGZF ? 64 : 4);
                    const size_t n_slices = (size_t)((n + slice - 1) / slice);
                    s.zout[e].assign(n_slices, std::vector<uint8_t>());
                    for (size_t k = 0; k < n_slices; k++) {
                        const uint8_t* src = s.h_out[e].p + k * slice;
                        const uint64_t len = std::min<uint64_t>(slice, n - k * slice);
                        std::vector<uint8_t>* dst = &s.zout[e][k];
                        const int lvl = P->compress;
                        c->writers.submit(&s.writes, [zmethod, lvl, src, len, dst]() { return deflate_members(zmethod, lvl, src, len, *dst); });
                    }
                    z_pending = &s;
                } else if (sink.kind == SINK_STREAM) {
                    if (sink.chunk_cb(sink.chunk_user, job_index, e, reinterpret_cast<const char*>(s.h_out[e].p), n))
                        throw IoErr("the chunk callback reported an error");
                } else {
                    if (sink.len[e] + n <= sink.cap[e]) std::memcpy(sink.mem[e] + sink.len[e], s.h_out[e].p, n);
                    sink.len[e] += n;
                }
            }
        }
        if (P->progress_cb) P->progress_cb(P->cb_user, (uint64_t)s.pairs * n_ends);
        s.busy = false;
    };

    std::vector<char> chrom_waited(c->chrom_ev.size(), 0);
    if (sizes_only) X.sizes_out->assign(jobs.size(), std::array<uint64_t, 2>{0, 0});

    for (size_t jk = 0; jk < jobs.size(); jk++) {
        const Job& job = jobs[jk];
        const uint64_t lo = ranges[jk].first, hi = ranges[jk].second;
        if (P->abort_cb && P->abort_cb(P->cb_user)) throw Aborted();   // src/hts.h:536
        if (X.ranges && hi <= lo) { job_index++; continue; }             // a multi-GPU device with no part in this job's files
        if (sink.kind == SINK_FILES && !sizes_only) {
            for (Slot& s : c->slot) wait_writes(s);
            sink.close_files();
            for (int e = 0; e < n_ends; e++) {
                sink.names[e] = file_name(job, e, want_gz, P) + (X.job_suffix ? (*X.job_suffix)[jk] : X.part_suffix);
                sink.pos[e] = sink.done[e] = X.base ? (*X.base)[jk][e] : 0;
                sink.own_size[e] = !X.shared_files;
                sink.fd[e] = ::open(sink.names[e].c_str(), X.shared_files ? O_RDWR : (O_RDWR | O_CREAT | O_TRUNC), 0644);
                if (sink.fd[e] < 0) throw IoErr("Unable to open file " + sink.names[e] + ".\n");  // src/io.h:288-290
            }
        }
        if (sink.kind == SINK_MEMORY && X.base) for (int e = 0; e < n_ends; e++) sink.len[e] = (*X.base)[jk][e];
        if (sizes_only) {
            // size pass: placement and scan only; the totals come back batch by batch (a few hundred microseconds each)
            for (uint64_t b0 = lo; b0 < hi; b0 += B) {
                Slot& s = c->slot[0];
                const uint32_t np = (uint32_t)std::min<uint64_t>(B, hi - b0);
                gp.job_lo = job.lo; gp.job_hi = job.hi; gp.batch_lo = b0; gp.batch_pairs = np;
                gp.plan = s.plan.p; gp.rec_len = s.rec_len.p; gp.rec_local = s.rec_local.p; gp.block_base = s.block_base.p;
                gp.n_scan_blocks = (np + kScanBlock - 1) / kScanBlock;
                CK(launch_place(gp, c->s_compute));
                CK(launch_scan(s.rec_len.p, np * n_ends, n_ends, s.rec_local.p, s.block_tot.p, s.block_base.p, s.totals.p, c->s_compute));
                CK(cudaMemcpyAsync(s.h_totals.p, s.totals.p, 4 * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->s_compute));
                CK(cudaStreamSynchronize(c->s_compute));
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
            Slot& s = c->slot[bi % 3];
            while (s.busy) drain_one();
            const uint32_t np = (uint32_t)std::min<uint64_t>(B, hi - b0);
            if (c->upload_pending && !use_haps) {
                // make the compute stream wait for exactly the uploads of the chromosomes this batch reads
                size_t g_lo, g_hi;
                groups_of(job, b0, b0 + np, g_lo, g_hi);
                g_hi = std::min(g_hi, c->chrom_ev.size() - 1);
                g_lo = std::min(g_lo, g_hi);
                if (b0 == lo) {
                    // first batch of this call's part of the job: a deferred upload copies, in the order the part
                    // will read them, all the chromosomes it reads and nothing else (with N GPUs each needs about
                    // 1/N of the genome); the rest stays on the host until some run asks for it
                    size_t g_end = (size_t)(std::upper_bound(group_off.begin(), group_off.end(), hi - 1) - group_off.begin()) - 1;
                    issue_upload(c, g_lo, std::min(g_end, c->chrom_ev.size() - 1));
                }
                issue_upload(c, g_lo, g_hi);
                for (size_t g = g_lo; g <= g_hi; g++)
                    if (!chrom_waited[g]) { CK(cudaStreamWaitEvent(c->s_compute, c->chrom_ev[g], 0)); chrom_waited[g] = 1; }
            }
            gp.job_lo = job.lo; gp.job_hi = job.hi; gp.batch_lo = b0; gp.batch_pairs = np;
            const uint32_t n_rec = np * n_ends;
            const uint32_t nsb = (np + kScanBlock - 1) / kScanBlock;
            gp.plan = s.plan.p; gp.rec_len = s.rec_len.p; gp.rec_local = s.rec_local.p; gp.block_base = s.block_base.p;
            gp.n_scan_blocks = nsb; gp.out[0] = s.out[0].p; gp.out[1] = s.out[1].p;
            CK(cudaEventRecord(s.ev[0], c->s_compute));
            CK(launch_place(gp, c->s_compute));
            CK(cudaEventRecord(s.ev[1], c->s_compute));
            CK(launch_scan(s.rec_len.p, n_rec, n_ends, s.rec_local.p, s.block_tot.p, s.block_base.p, s.totals.p,
                           c->s_compute));
            CK(cudaEventRecord(s.ev[2], c->s_compute));
            CK(launch_reads(gp, c->n_sm, c->s_compute));
            CK(cudaEventRecord(s.ev[3], c->s_compute));
            if (dev_z) {
                CK(launch_bgzf(s.out[0].p, s.out[1].p, s.totals.p, nblk_max, P->compress >= 4, s.zslots[0].p, s.zslots[1].p, s.zlen[0].p,
                               s.zlen[1].p, s.zoff[0].p, s.zoff[1].p, s.zdev[0].p, s.zdev[1].p, s.zcode.p, c->s_compute));
                st.kernel_launches += kBgzfLaunches;
            }
            CK(cudaMemcpyAsync(s.h_totals.p, s.totals.p, 4 * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->s_compute));
            CK(cudaEventRecord(s.ev[5], c->s_compute));
            st.kernel_launches += 4;
            s.pairs = np; s.busy = true;
            computing.push_back(&s);
            // the previous batch's copy is queued before the one in flight is waited for
            if (computing.size() > 1) { issue_copy(*computing.front()); copying.push_back(computing.front()); computing.pop_front(); }
            if (copying.size() > 1) { deliver(*copying.front()); copying.pop_front(); }
            if (P->abort_cb && P->abort_cb(P->cb_user)) throw Aborted();   // Quiesce settles what is in flight
        }
        while (!computing.empty() || !copying.empty()) drain_one();
        if (z_pending) { wait_writes(*z_pending); z_pending = nullptr; }
        for (Slot& s : c->slot) wait_writes(s);
        const bool eof_block = !X.shared_files && X.part_suffix.empty() && !X.no_eof;      // a multi-GPU run appends it once, after joining the parts
        if (sink.kind == SINK_FILES && (zmethod == DEFLATE_BGZF || dev_z) && eof_block)
            for (int e = 0; e < n_ends; e++) {   // bgzf_close appends the empty end-of-file block
                std::string w = pwrite_all(sink.fd[e], kBgzfEof, sizeof kBgzfEof, sink.pos[e]);
                if (!w.empty()) throw IoErr("Error writing to file " + sink.names[e] + ": " + w);
                sink.pos[e] += sizeof kBgzfEof;
                sink.done[e] = sink.pos[e];
            }
        if (dev_z && sink.kind == SINK_STREAM)
            for (int e = 0; e < n_ends; e++)
                if (sink.chunk_cb(sink.chunk_user, job_index, e, reinterpret_cast<const char*>(kBgzfEof), sizeof kBgzfEof))
                    throw IoErr("the chunk callback reported an error");
        if (dev_z && sink.kind == SINK_MEMORY)
            for (int e = 0; e < n_ends; e++) {
                if (sink.len[e] + sizeof kBgzfEof <= sink.cap[e]) std::memcpy(sink.mem[e] + sink.len[e], kBgzfEof, sizeof kBgzfEof);
                sink.len[e] += sizeof kBgzfEof;
            }
        job_index++;
    }
    CK(cudaEventRecord(c->ev_run[1], c->s_compute));
    CK(cudaEventSynchronize(c->ev_run[1]));
    {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, c->ev_run[0], c->ev_run[1]));
        st.run_ms = ms;
    }
    sink.close_files();
    if (c->upload_pending) {
        // the copies this run issued are done before the caller gets control back; chromosomes no
        // shard of this run touched remain on the host (upload_src must stay valid, see the header)
        CK(cudaStreamSynchronize(c->s_upload));
        if (std::find(c->chrom_resident.begin(), c->chrom_resident.end(), 0) == c->chrom_resident.end()) {
            c->upload_pending = false;
            c->upload_src = nullptr;
        }
    }
    uint32_t status = 0;
    CK(cudaMemcpy(&status, c->d_status.p, sizeof status, cudaMemcpyDeviceToHost));
    if (status & 1u) throw ArgErr("a barcode is at least as long as a read's template (fragment or chromosome too short)");
    st.h2d_bytes = c->h2d_bytes - h2d_before;      // of this call (a deferred genome upload it performed included)
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

// n bytes from in_fd at in_off to out_fd at out_off (both files on any file system)
std::string copy_range(int out_fd, uint64_t out_off, int in_fd, uint64_t in_off, uint64_t n) {
    std::vector<uint8_t> buf;
    bool use_cfr = true;
    while (n) {
        if (use_cfr) {
            off_t oi = (off_t)in_off, oo = (off_t)out_off;
            const ssize_t w = ::copy_file_range(in_fd, &oi, out_fd, &oo, (size_t)std::min<uint64_t>(n, 1ull << 30), 0);
            if (w > 0) { n -= (uint64_t)w; in_off += (uint64_t)w; out_off += (uint64_t)w; continue; }
            if (w < 0 && errno == EINTR) continue;
            if (w == 0) return "unexpected end of a part file";
            if (errno != EXDEV && errno != EINVAL && errno != ENOSYS && errno != EOPNOTSUPP) return std::strerror(errno);
            use_cfr = false;                                  // file systems without copy_file_range: read + write
        }
        buf.resize(8u << 20);
        const ssize_t r = ::pread(in_fd, buf.data(), (size_t)std::min<uint64_t>(n, buf.size()), (off_t)in_off);
        if (r < 0) { if (errno == EINTR) continue; return std::strerror(errno); }
        if (r == 0) return "unexpected end of a part file";
        const std::string w = pwrite_all(out_fd, buf.data(), (uint64_t)r, out_off);
        if (!w.empty()) return w;
        n -= (uint64_t)r; in_off += (uint64_t)r; out_off += (uint64_t)r;
    }
    return std::string();
}

void run_multi(jlp_ctx* c, bool use_haps, const jlp_illumina_params* P, Sink& sink, jlp_run_stats* stats) {
    check_params(c, use_haps, P, sink.kind);
    if (sink.kind == SINK_STREAM)
        throw Unsupported("jlp_illumina_stream on a multi-GPU context: batches of several devices have no single order; "
                          "use files / memory, or one context per device with shard_index / shard_count");
    if (P->shard_count > 1) throw ArgErr("shard_index / shard_count do not combine with a multi-GPU context");
    const size_t N = c->kids.size();
    const Layout Y = make_layout(c, use_haps, P);
    const size_t nj = Y.jobs.size();
    const int n_ends = Y.n_ends;
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

    std::vector<std::string> errs(N);
    std::vector<int> codes(N, JLP_OK);
    std::vector<jlp_run_stats> st(N);
    // run f(r) for every device on its own thread; the calling thread serves the callbacks meanwhile
    auto on_devices = [&](const std::function<void(size_t)>& f, bool with_callbacks) {
        std::atomic<size_t> left{N};
        std::vector<std::thread> th;
        for (size_t r = 0; r < N; r++)
            th.emplace_back([&, r]() {
                codes[r] = guarded(c->kids[r], [&]() { f(r); });
                if (codes[r] != JLP_OK) {                     // the others stop at their next batch
                    errs[r] = c->kids[r]->err;
                    int none = 0;
                    shared.abort.compare_exchange_strong(none, 1);
                }
                left.fetch_sub(1);
            });
        while (left.load() != 0) {
            std::this_thread::sleep_for(std::chrono::milliseconds(with_callbacks ? 20 : 2));
            if (!with_callbacks) continue;
            const uint64_t d = shared.progress.exchange(0);
            if (d && P->progress_cb) P->progress_cb(P->cb_user, d);
            if (P->abort_cb && !shared.abort.load() && P->abort_cb(P->cb_user)) shared.abort.store(2);
        }
        for (std::thread& t : th) t.join();
        const uint64_t d = shared.progress.exchange(0);
        if (d && P->progress_cb && with_callbacks) P->progress_cb(P->cb_user, d);
        if (shared.abort.load() == 2) throw Aborted();
        for (size_t r = 0; r < N; r++) {
            if (codes[r] == JLP_OK || codes[r] == JLP_ERR_ABORTED) continue;      // a device aborted because another failed
            const std::string m = "device " + std::to_string(c->kids[r]->device) + ": " + errs[r];
            switch (codes[r]) {
            case JLP_ERR_ARG: throw ArgErr(errs[r]);
            case JLP_ERR_IO: throw IoErr(errs[r]);
            case JLP_ERR_UNSUPPORTED: throw Unsupported(errs[r]);
            default: throw CudaErr(m);
            }
        }
    };

    // a shared output file gets its final size at once (no pages yet); a file system that cannot hold everything the
    // run will write is reported here rather than half-way through
    uint64_t need_bytes = 0;
    auto presize = [](int fd, uint64_t size, uint64_t& need) -> int {
        need += size;
        struct statvfs vfs;
        if (::fstatvfs(fd, &vfs) == 0 && (uint64_t)vfs.f_bavail * vfs.f_frsize < need) return ENOSPC;
        return ::ftruncate(fd, (off_t)size) == 0 ? 0 : errno;
    };

    // --- size pass
    std::vector<PerJobBytes> sizes(N), base(N, PerJobBytes(nj, std::array<uint64_t, 2>{0, 0}));
    std::vector<std::array<uint64_t, 2>> job_total(nj, std::array<uint64_t, 2>{0, 0});
    uint64_t launches = 0;
    if (sized) {
        on_devices([&](size_t r) {
            Sink none;
            RunExtras X;
            X.ranges = &ranges[r]; X.sizes_out = &sizes[r];
            run(c->kids[r], use_haps, &Pk, none, &st[r], X);
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
                for (int e = 0; e < n_ends; e++) {
                    const std::string name = file_name(Y.jobs[k], e, false, P);
                    const int fd = ::open(name.c_str(), O_RDWR | O_CREAT | O_TRUNC, 0644);
                    if (fd < 0) throw IoErr("Unable to open file " + name + ".\n");      // src/io.h:288-290
                    // sized now, pages reserved slice by slice by the devices' writer threads (see deliver() in run())
                    const int rc = presize(fd, job_total[k][e], need_bytes);
                    ::close(fd);
                    if (rc != 0) throw IoErr("Error writing to file " + name + ": " + std::strerror(rc));
                }
        if (sink.kind == SINK_MEMORY) { sink.len[0] = mem_off[0]; sink.len[1] = mem_off[1]; }
    }

    // --- compressed size pass (device coder)
    std::vector<PerJobBytes> zsizes(N), zcheck(N);
    if (zsized) {
        jlp_illumina_params Pdry = Pk;
        Pdry.progress_cb = nullptr;
        on_devices([&](size_t r) {
            Sink none;
            RunExtras X;
            X.ranges = &ranges[r]; X.zsizes_out = &zsizes[r]; X.dry_files = true;
            run(c->kids[r], use_haps, &Pdry, none, &st[r], X);
        }, true);
        for (size_t r = 0; r < N; r++) launches += st[r].kernel_launches;
        for (size_t k = 0; k < nj; k++)
            for (int e = 0; e < n_ends; e++) {
                uint64_t o = 0;
                for (size_t r = 0; r < N; r++) { base[r][k][e] = o; o += zsizes[r][k][e]; }
                job_total[k][e] = o;
                const std::string name = file_name(Y.jobs[k], e, true, P);
                const int fd = ::open(name.c_str(), O_RDWR | O_CREAT | O_TRUNC, 0644);
                if (fd < 0) throw IoErr("Unable to open file " + name + ".\n");      // src/io.h:288-290
                const uint64_t size = o + sizeof kBgzfEof;                            // bgzf_close: one empty block ends the file
                const int rc = presize(fd, size, need_bytes);
                std::string w;
                if (rc == 0) w = pwrite_all(fd, kBgzfEof, sizeof kBgzfEof, o);
                ::close(fd);
                if (rc != 0) throw IoErr("Error writing to file " + name + ": " + std::strerror(rc));
                if (!w.empty()) throw IoErr("Error writing to file " + name + ": " + w);
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
    on_devices([&](size_t r) {
        Sink sk;
        sk.kind = sink.kind;
        for (int e = 0; e < 2; e++) { sk.mem[e] = sink.mem[e]; sk.cap[e] = sink.cap[e]; }
        RunExtras X;
        X.ranges = &ranges[r];
        if (sized) { X.base = &base[r]; X.shared_files = sink.kind == SINK_FILES; }
        if (zsized) { X.base = &base[r]; X.shared_files = true; X.zsizes_out = &zcheck[r]; }
        std::vector<std::string> suffix;
        if (parts) {
            // per job: the job's first device writes <name> itself (no EOF block yet), every other one <name>.part<r>
            X.no_eof = true;
            X.job_suffix = &suffix;
            for (size_t k = 0; k < nj; k++) suffix.push_back(r == first_dev[k] ? std::string() : ".part" + std::to_string(r));
        }
        run(c->kids[r], use_haps, &Pk, sk, &st[r], X);
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
        std::atomic<size_t> next{0};
        std::mutex em;
        std::string first_err;
        // a slice is copied through mappings of both files where that works (threads writing one file through
        // write() / copy_file_range queue on its inode lock; page-cache pages filled through a mapping do not), else by copy_range
        auto worker = [&]() {
            static const uint64_t page = (uint64_t)sysconf(_SC_PAGESIZE);
            for (size_t i = next.fetch_add(1); i < tasks.size(); i = next.fetch_add(1)) {
                const CopyTask& t = tasks[i];
                std::string w;
                const uint64_t o0 = t.out_off / page * page, i0 = t.in_off / page * page;
                void* mo = ::mmap(nullptr, (size_t)(t.out_off + t.len - o0), PROT_READ | PROT_WRITE, MAP_SHARED, t.out_fd, (off_t)o0);
                void* mi = mo == MAP_FAILED ? MAP_FAILED : ::mmap(nullptr, (size_t)(t.in_off + t.len - i0), PROT_READ, MAP_SHARED, t.in_fd, (off_t)i0);
                if (mo != MAP_FAILED && mi != MAP_FAILED)
                    std::memcpy(static_cast<uint8_t*>(mo) + (t.out_off - o0), static_cast<const uint8_t*>(mi) + (t.in_off - i0), t.len);
                else
                    w = copy_range(t.out_fd, t.out_off, t.in_fd, t.in_off, t.len);
                if (mi != MAP_FAILED) ::munmap(mi, (size_t)(t.in_off + t.len - i0));
                if (mo != MAP_FAILED) ::munmap(mo, (size_t)(t.out_off + t.len - o0));
                if (!w.empty()) { std::lock_guard<std::mutex> l(em); if (first_err.empty()) first_err = w; }
            }
        };
        const size_t nth = std::min<size_t>(std::max<size_t>(tasks.size(), 1), std::min<uint64_t>(std::max<uint64_t>(P->n_threads, 4), 32));
        std::vector<std::thread> th;
        for (size_t i = 1; i < nth; i++) th.emplace_back(worker);
        worker();
        for (std::thread& t : th) t.join();
        if (!first_err.empty()) throw IoErr("Error joining the devices' parts: " + first_err);
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

int jlp_ctx_create(int device, jlp_ctx** out) {
    if (!out) return fail(nullptr, JLP_ERR_ARG, "out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(nullptr, JLP_ERR_NO_DEVICE,
                    std::string("no CUDA device available (") + cudaGetErrorString(e) +
                        "); this library has no CPU fallback");
    if (device < 0 || device >= n) return fail(nullptr, JLP_ERR_ARG, "device index out of range");
    std::unique_ptr<jlp_ctx> c(new jlp_ctx);
    c->device = device;
    int rc = guarded(c.get(), [&]() {
        CK(cudaDeviceGetAttribute(&c->n_sm, cudaDevAttrMultiProcessorCount, device));
        CK(cudaStreamCreateWithFlags(&c->s_compute, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&c->s_copy, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&c->s_upload, cudaStreamNonBlocking));
        CK(bgzf_init());
    });
    if (rc != JLP_OK) { g_create_error = c->err; return rc; }
    *out = c.release();
    return JLP_OK;
}

int jlp_ctx_create_multi(int n_devices, const int* devices, jlp_ctx** out) {
    if (!out) return fail(nullptr, JLP_ERR_ARG, "out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(nullptr, JLP_ERR_NO_DEVICE, std::string("no CUDA device available (") + cudaGetErrorString(e) +
                                                    "); this library has no CPU fallback");
    if (n_devices < 0 || n_devices > 64) return fail(nullptr, JLP_ERR_ARG, "n_devices must be 0 (all visible devices) .. 64");
    if (n_devices == 0) { n_devices = n; devices = nullptr; }
    std::unique_ptr<jlp_ctx> c(new jlp_ctx);
    c->device = -1;
    for (int i = 0; i < n_devices; i++) {
        const int d = devices ? devices[i] : i;
        jlp_ctx* k = nullptr;
        const int rc = jlp_ctx_create(d, &k);
        if (rc != JLP_OK) { for (jlp_ctx* q : c->kids) jlp_ctx_destroy(q); return rc; }
        c->kids.push_back(k);
    }
    *out = c.release();
    return JLP_OK;
}

int jlp_ctx_n_devices(const jlp_ctx* c) { return c ? (c->kids.empty() ? 1 : (int)c->kids.size()) : 0; }

void jlp_ctx_destroy(jlp_ctx* c) {
    if (!c) return;
    if (!c->kids.empty()) {
        for (jlp_ctx* k : c->kids) jlp_ctx_destroy(k);
        delete c;
        return;
    }
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    free_haps(c);
    for (Slot& s : c->slot) for (cudaEvent_t ev : s.ev) if (ev) cudaEventDestroy(ev);
    for (cudaEvent_t ev : c->ev_run) if (ev) cudaEventDestroy(ev);
    if (c->s_compute) cudaStreamDestroy(c->s_compute);
    if (c->s_copy) cudaStreamDestroy(c->s_copy);
    if (c->s_upload) cudaStreamDestroy(c->s_upload);
    for (int k = 0; k < jlp_ctx::kMatBufs; k++) { if (c->m_up[k]) cudaEventDestroy(c->m_up[k]); if (c->m_done[k]) cudaEventDestroy(c->m_done[k]); }
    for (cudaEvent_t ev : c->chrom_ev) cudaEventDestroy(ev);
    c->writers.stop();
    delete c;
}

const char* jlp_last_error(const jlp_ctx* c) { return c ? c->err.c_str() : g_create_error.c_str(); }

static int set_genome_impl(jlp_ctx* c, const char* bases, const uint64_t* chrom_off, uint64_t n_chroms,
                           const char* const* chrom_names, const char* genome_name, bool wait) {
    if (!c) return JLP_ERR_ARG;
    if (!c->kids.empty()) {
        // every device gets a deferred upload (a run copies only the chromosomes the device's piece reads); the
        // synchronous form then makes the whole genome resident everywhere, one host thread per device
        return guarded(c, [&]() {
            for (jlp_ctx* k : c->kids) {
                const int rc = set_genome_impl(k, bases, chrom_off, n_chroms, chrom_names, genome_name, false);
                if (rc != JLP_OK) throw ArgErr(k->err);
            }
            c->haps.clear();
            c->chrom_off = c->kids[0]->chrom_off; c->chrom_names = c->kids[0]->chrom_names; c->genome_name = c->kids[0]->genome_name;
            if (wait) for_each_device_parallel(c, [](jlp_ctx* d) { finish_upload(d); });
        });
    }
    return guarded(c, [&]() {
        if (!bases || !chrom_off || !chrom_names || n_chroms == 0) throw ArgErr("empty genome");
        for (uint64_t i = 0; i < n_chroms; i++)
            if (chrom_off[i + 1] < chrom_off[i]) throw ArgErr("chrom_off must be non-decreasing");
        if (chrom_off[0] != 0) throw ArgErr("chrom_off[0] must be 0");
        if (c->upload_pending) {      // a deferred upload that never ran is simply dropped
            c->upload_src = nullptr;
            CK(cudaStreamSynchronize(c->s_upload));
            c->upload_pending = false;
        }
        free_haps(c);
        c->chrom_off.assign(chrom_off, chrom_off + n_chroms + 1);
        c->chrom_names.clear();
        for (uint64_t i = 0; i < n_chroms; i++) c->chrom_names.push_back(chrom_names[i] ? chrom_names[i] : "");
        c->genome_name = genome_name ? genome_name : "REF";
        uint64_t total = chrom_off[n_chroms];
        c->genome.ensure(total + 2 * kPad);
        while (c->chrom_ev.size() < n_chroms) {
            cudaEvent_t ev;
            CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            c->chrom_ev.push_back(ev);
        }
        // one copy and one event per chromosome: generation starts as soon as the chromosomes a batch
        // reads are resident, the rest of the genome follows underneath (PCIe is full duplex, the
        // FASTQ flows the other way).  The asynchronous form defers the copies to the next run, which
        // starts them at the first chromosome its shard reads.
        c->upload_src = bases;
        c->upload_pending = true;
        c->chrom_resident.assign(n_chroms, 0);
        if (wait) finish_upload(c);
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
    return guarded(c, [&]() {
        for_each_device_parallel(c, [](jlp_ctx* d) { finish_upload(d); });
    });
}

int jlp_create_genome(jlp_ctx* c, uint64_t n_chroms, const uint64_t* lens, const double* pi_tcag, uint64_t seed,
                      const char* const* chrom_names, const char* genome_name) {
    if (!c) return JLP_ERR_ARG;
    if (!c->kids.empty())        // the same seed gives every device the same genome: generated in place everywhere, nothing copied
        return guarded(c, [&]() {
            for (jlp_ctx* k : c->kids) {
                const int rc = jlp_create_genome(k, n_chroms, lens, pi_tcag, seed, chrom_names, genome_name);
                if (rc != JLP_OK) throw ArgErr(k->err);
            }
            c->haps.clear();
            c->chrom_off = c->kids[0]->chrom_off; c->chrom_names = c->kids[0]->chrom_names; c->genome_name = c->kids[0]->genome_name;
        });
    return guarded(c, [&]() {
        if (!lens || !pi_tcag || n_chroms == 0) throw ArgErr("empty genome");
        double tot = 0;
        for (int k = 0; k < 4; k++) { if (!(pi_tcag[k] >= 0)) throw ArgErr("pi_tcag must be >= 0"); tot += pi_tcag[k]; }
        if (!(tot > 0)) throw ArgErr("pi_tcag must have at least one value > 0");
        if (c->upload_pending) { c->upload_src = nullptr; CK(cudaStreamSynchronize(c->s_upload)); c->upload_pending = false; }
        free_haps(c);
        c->chrom_off.assign(1, 0);
        c->chrom_names.clear();
        for (uint64_t i = 0; i < n_chroms; i++) {
            if (lens[i] == 0) throw ArgErr("chromosome lengths must be >= 1");       // "never returns empty chromosomes"
            c->chrom_off.push_back(c->chrom_off.back() + lens[i]);
            c->chrom_names.push_back(chrom_names && chrom_names[i] ? chrom_names[i] : "chrom" + std::to_string(i));   // src/create_sequences.cpp:178-181
        }
        c->genome_name = genome_name ? genome_name : "REF";
        c->chrom_resident.assign(n_chroms, 1);
        c->genome.ensure(c->chrom_off.back() + 2 * kPad);
        // AliasSampler(pi_tcag), src/alias_sampler.h:68-106
        double Prob[4];
        uint64_t Alias[4];
        alias_build(pi_tcag, 4, Prob, Alias);
        GenomeTables t;
        for (int k = 0; k < 4; k++) {
            Thr th = thr_double_lt(Prob[k]);
            t.thr[k] = th.thr; t.thr16[k] = (uint32_t)(th.thr >> 48); t.alias[k] = (uint32_t)Alias[k];
        }
        for (uint64_t i = 0; i < n_chroms; i++)
            CK(launch_create_chrom(c->genome.p + kPad + c->chrom_off[i], lens[i], (uint32_t)i, seed, t, c->s_compute));
        CK(cudaStreamSynchronize(c->s_compute));
    });
}

int jlp_get_genome(jlp_ctx* c, char* out, uint64_t cap, uint64_t* len) {
    if (!c) return JLP_ERR_ARG;
    if (!c->kids.empty()) {
        const int rc = jlp_get_genome(c->kids[0], out, cap, len);
        if (rc != JLP_OK) c->err = c->kids[0]->err;
        return rc;
    }
    return guarded(c, [&]() {
        if (c->chrom_off.size() < 2) throw ArgErr("no reference genome has been set");
        finish_upload(c);
        const uint64_t n = c->chrom_off.back();
        if (len) *len = n;
        if (!out) return;
        if (n > cap) throw ArgErr("output buffer too small");
        CK(cudaMemcpy(out, c->genome.p + kPad, n, cudaMemcpyDeviceToHost));
    });
}

int jlp_clear_haplotypes(jlp_ctx* c) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        for_each_device(c, [](jlp_ctx* d) { free_haps(d); });
        c->haps.clear();
    });
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
    std::atomic<uint64_t> next{0};
    std::mutex err_mu;
    std::string err;
    auto work = [&]() {
        for (uint64_t ci; (ci = next.fetch_add(1)) < nc;) {
            const char* bad = nullptr;
            const uint64_t M = n_muts[ci];
            const uint64_t ref_size = c->chrom_off[ci + 1] - c->chrom_off[ci];
            HapChromHost& H = S->chrom[ci];
            H.size = chrom_sizes[ci];
            if (M == 0) {   // get_chrom_full returns the reference string (src/hap_classes.cpp:82)
                if (chrom_sizes[ci] != ref_size) bad = "chromosome without mutations must keep the reference size";
            } else if (!old_pos || !new_pos || !nuc_off || !nuc_pool || !nuc_pool_len || !old_pos[ci] || !new_pos[ci] || !nuc_off[ci]) {
                bad = "mutation arrays are NULL";
            } else {
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
                    if (i && new_pos[ci][i] < new_pos[ci][i - 1]) { bad = "mutations must be sorted by new_pos"; break; }
                    const int64_t s = (i + 1 < M) ? (int64_t)(new_pos[ci][i + 1] - old_pos[ci][i + 1]) : (int64_t)(chrom_sizes[ci] - ref_size);
                    sm[i] = s + (int64_t)(old_pos[ci][i] - new_pos[ci][i]);
                }
                if (pb) std::memcpy(w + 4 * M, nuc_pool[ci], pb);
            }
            if (bad) { std::lock_guard<std::mutex> g(err_mu); if (err.empty()) err = bad; }
        }
    };
    uint64_t total = 0;
    for (uint64_t ci = 0; ci < nc; ci++) total += n_muts[ci];
    const unsigned nt = total < (1u << 16) ? 1u : (unsigned)std::min<uint64_t>(std::min<uint64_t>(nc, 16), std::max(1u, std::thread::hardware_concurrency()));
    std::vector<std::thread> th;
    for (unsigned i = 1; i < nt; i++) th.emplace_back(work);
    work();
    for (std::thread& t : th) t.join();
    if (!err.empty()) throw ArgErr(err);
    return S;
}

// attach a haplotype to a context: unmutated chromosomes alias the reference, the others wait for a run to touch them
static void attach_hap(jlp_ctx* c, const std::shared_ptr<HapStore>& S) {
    HapDev H;
    H.store = S;
    const bool device = c->kids.empty();
    for (size_t ci = 0; ci < S->chrom.size(); ci++) {
        const HapChromHost& M = S->chrom[ci];
        H.len.push_back(M.size);
        H.seq.push_back(device && M.n_muts == 0 ? c->genome.p + kPad + c->chrom_off[ci] : nullptr);
    }
    c->haps.push_back(std::move(H));
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
        for (jlp_ctx* k : c->kids) attach_hap(k, S);
    });
}

int jlp_materialize_haplotypes(jlp_ctx* c) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        for_each_device(c, [&](jlp_ctx* d) {
            finish_upload(d);
            for (size_t h = 0; h < d->haps.size(); h++)
                for (size_t ci = 0; ci < d->haps[h].seq.size(); ci++) ensure_hap_chrom(d, h, ci);
            CK(cudaStreamSynchronize(d->s_compute));
        });
    });
}

int jlp_get_haplotype_chrom(jlp_ctx* c, uint64_t hap, uint64_t chrom, char* out, uint64_t cap, uint64_t* len) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        jlp_ctx* d = c->kids.empty() ? c : c->kids[0];
        if (!c->kids.empty()) CK(cudaSetDevice(d->device));
        if (hap >= d->haps.size() || chrom >= d->haps[hap].seq.size()) throw ArgErr("haplotype / chromosome index out of range");
        uint64_t n = d->haps[hap].len[chrom];
        if (len) *len = n;
        if (n > cap) throw ArgErr("output buffer too small");
        finish_upload(d);
        ensure_hap_chrom(d, hap, chrom);
        CK(cudaStreamSynchronize(d->s_compute));
        if (n) CK(cudaMemcpy(out, d->haps[hap].seq[chrom], n, cudaMemcpyDeviceToHost));
    });
}

int jlp_get_haplotype_muts(jlp_ctx* c, uint64_t hap, uint64_t chrom, uint64_t* old_pos, uint64_t* new_pos,
                           uint64_t* nuc_off, char* pool, uint64_t cap_muts, uint64_t cap_pool, uint64_t* n_muts,
                           uint64_t* pool_len, uint64_t* chrom_size) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        if (hap >= c->haps.size() || chrom >= c->haps[hap].store->chrom.size()) throw ArgErr("haplotype / chromosome index out of range");
        const HapChromHost& H = c->haps[hap].store->chrom[chrom];
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

// The visiting order of the tree and the node-state slots (k_mutate): preorder with the child of fewer tips first, a
// parent's slot freed when its last child is visited (before that child takes one), so at most about log2(tips) + 2
// slots are live.  Childless nodes that are not tips are left out.
std::vector<MutNode> mut_schedule(const jlp_mutation_params* p, const std::vector<int32_t>& tip_of, uint32_t n_cat,
                                  uint32_t& max_slots) {
    const uint32_t n = p->n_nodes;
    std::vector<std::vector<uint32_t>> kids(n);
    for (uint32_t i = 1; i < n; i++) kids[p->parent[i]].push_back(i);
    std::vector<uint64_t> tips(n, 0);
    for (uint32_t i = n; i-- > 0;) {
        if (kids[i].empty()) tips[i] = tip_of[i] >= 0 ? 1 : 0;
        if (i) tips[p->parent[i]] += tips[i];
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
        const uint32_t par = (uint32_t)p->parent[v];
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

}  // namespace

int jlp_create_haplotypes(jlp_ctx* c, const jlp_mutation_params* p, jlp_mutation_stats* stats) {
    if (!c || !p) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        const auto t0 = std::chrono::steady_clock::now();
        if (c->chrom_off.size() < 2) throw ArgErr("set the reference genome first");
        for (int i = 0; i < 16; i++)
            if (i % 5 && !(std::isfinite(p->Q[i]) && p->Q[i] >= 0)) throw ArgErr("the off-diagonal rates of Q must be finite and >= 0");
        if (!(p->invariant >= 0 && p->invariant < 1)) throw ArgErr("invariant must be >= 0 and < 1");
        if (p->n_rates < 1 || p->n_rates > 255 || !p->rates) throw ArgErr("n_rates must be 1..255 (rates not NULL)");
        for (uint32_t k = 0; k < p->n_rates; k++)
            if (!(std::isfinite(p->rates[k]) && p->rates[k] >= 0)) throw ArgErr("category rates must be finite and >= 0");
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
        if (p->n_tips < 1 || p->n_tips > kMutMaxTips)
            throw ArgErr("a tree of " + std::to_string(p->n_tips) + " tips: 1 to " + std::to_string(kMutMaxTips) + " tips are supported");
        if (!p->tip_node || !p->tip_names) throw ArgErr("tip_node / tip_names is NULL");
        std::vector<int32_t> tip_of(n, -1);
        for (uint32_t t = 0; t < p->n_tips; t++) {
            const uint32_t v = p->tip_node[t];
            if (v >= n || has_kid[v] || tip_of[v] >= 0) throw ArgErr("tip_node must list distinct childless nodes");
            if (!p->tip_names[t]) throw ArgErr("tip name is NULL");
            tip_of[v] = (int32_t)t;
        }
        const uint64_t nc = c->chrom_off.size() - 1;
        std::vector<uint32_t> tile0(nc + 1, 0);
        for (uint64_t ci = 0; ci < nc; ci++) {
            const uint64_t len = c->chrom_off[ci + 1] - c->chrom_off[ci];
            if (len >> 32) throw ArgErr("chromosomes of 2^32 bases or more are not supported");
            const uint64_t t = tile0[ci] + (len + kMutTile - 1) / kMutTile;
            if (t >> 32) throw ArgErr("genome too large");
            tile0[ci + 1] = (uint32_t)t;
        }
        const uint32_t K = p->n_rates, n_tips = p->n_tips, n_tiles = tile0[nc];

        // host tables: the schedule, per (node, category, parent state) the row thresholds, the category thresholds
        uint32_t max_slots = 0;
        const std::vector<MutNode> sched = mut_schedule(p, tip_of, K, max_slots);
        const uint64_t rows = (uint64_t)n * K * 4;
        std::vector<uint4> thr_hi(rows, make_uint4(0, 0, 0, 0)), thr_lo(rows, make_uint4(0, 0, 0, 0));
        for (const MutNode& m : sched)
            for (uint32_t k = 0; k < K; k++) {
                double P[16];
                transition_matrix(p->Q, p->rates[k] * p->branch_len[m.node], P);
                for (uint32_t a = 0; a < 4; a++) {
                    uint64_t t[3];
                    row_thresholds(P + 4 * a, t);
                    const uint64_t r = m.tab + 4ull * k + a;
                    thr_hi[r] = make_uint4((uint32_t)(t[0] >> 32), (uint32_t)(t[1] >> 32), (uint32_t)(t[2] >> 32), 0);
                    thr_lo[r] = make_uint4((uint32_t)t[0], (uint32_t)t[1], (uint32_t)t[2], 0);
                }
            }
        std::vector<uint64_t> cat_thr(K);
        cat_thr[0] = prob_threshold(p->invariant);
        for (uint32_t j = 1; j < K; j++) cat_thr[j] = prob_threshold(p->invariant + j * (1 - p->invariant) / K);

        jlp_ctx* d = first_device(c);
        finish_upload(d);
        cudaStream_t s = d->s_compute;
        DevBuf<uint64_t> d_off, d_cat, d_region, d_region_n, d_out;
        DevBuf<uint32_t> d_tile0, d_cnt;
        DevBuf<MutNode> d_sched;
        DevBuf<uint4> d_hi, d_lo;
        d_off.upload(d->chrom_off, s);
        d_tile0.upload(tile0, s);
        d_sched.upload(sched, s);
        d_cat.upload(cat_thr, s);
        d_hi.upload(thr_hi, s);
        d_lo.upload(thr_lo, s);
        const size_t n_cnt = (size_t)n_tips * n_tiles;
        d_cnt.ensure(n_cnt);
        if (n_cnt) CK(cudaMemsetAsync(d_cnt.p, 0, n_cnt * 4, s));
        d_region_n.ensure((size_t)n_tips * nc);
        MutParams mp{};
        mp.seed = p->seed;
        mp.genome = d->genome.p + kPad;
        mp.chrom_off = d_off.p;
        mp.tile0 = d_tile0.p;
        mp.n_chroms = (uint32_t)nc; mp.n_tiles = n_tiles; mp.n_tips = n_tips; mp.n_sched = (uint32_t)sched.size();
        mp.sched = d_sched.p;
        mp.n_cat = K;
        mp.cat_thr = d_cat.p;
        mp.thr_hi = d_hi.p; mp.thr_lo = d_lo.p;
        mp.tab_rows = (uint32_t)rows;
        mp.tab_smem = mut_smem_bytes((uint32_t)rows) <= (64u << 10);
        mp.cnt = d_cnt.p;
        EventSet ev;
        CK(cudaEventRecord(ev.e[0], s));
        CK(launch_mutate(mp, false, s));
        CK(cudaEventRecord(ev.e[1], s));
        CK(launch_mut_scan(mp, d_region_n.p, s));
        CK(cudaEventRecord(ev.e[2], s));
        std::vector<uint64_t> region_n((size_t)n_tips * nc), region((size_t)n_tips * nc);
        CK(cudaMemcpyAsync(region_n.data(), d_region_n.p, region_n.size() * 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        uint64_t words = 0, records = 0;
        for (size_t r = 0; r < region.size(); r++) {
            region[r] = words;
            words += 4 * region_n[r] + (region_n[r] + 7) / 8;
            records += region_n[r];
        }
        d_region.upload(region, s);
        mp.region = d_region.p;
        mp.region_n = d_region_n.p;              // k_mut_scan left the totals there
        d_out.ensure(words);
        if (words) CK(cudaMemsetAsync(d_out.p, 0, words * 8, s));
        mp.out = d_out.p;
        CK(cudaEventRecord(ev.e[3], s));
        if (records) CK(launch_mutate(mp, true, s));
        CK(cudaEventRecord(ev.e[4], s));
        CK(cudaStreamSynchronize(s));
        const float count_ms = ev.ms(0, 1), scan_ms = ev.ms(1, 2), write_ms = ev.ms(3, 4);
        const auto t_gen = std::chrono::steady_clock::now();

        // the records into one HapStore per tip, copied straight into the packed arrays by a few host threads
        std::vector<std::shared_ptr<HapStore>> stores(n_tips);
        for (uint32_t t = 0; t < n_tips; t++) {
            stores[t] = std::make_shared<HapStore>();
            stores[t]->name = p->tip_names[t];
            stores[t]->chrom.resize(nc);
        }
        const size_t n_items = (size_t)n_tips * nc;
        std::atomic<size_t> next{0};
        std::mutex err_mu;
        std::string err;
        const int dev = d->device;
        auto work = [&]() {
            try {
                CK(cudaSetDevice(dev));
                for (size_t r; (r = next.fetch_add(1)) < n_items;) {
                    HapChromHost& H = stores[r / nc]->chrom[r % nc];
                    const uint64_t M = region_n[r];
                    H.size = c->chrom_off[r % nc + 1] - c->chrom_off[r % nc];
                    H.n_muts = M;
                    H.pool_bytes = M;
                    if (!M) continue;
                    H.packed.resize(4 * M + (M + 7) / 8);
                    CK(cudaMemcpy(H.packed.data(), d_out.p + region[r], H.packed.size() * 8, cudaMemcpyDeviceToHost));
                }
            } catch (const std::exception& e) { std::lock_guard<std::mutex> g(err_mu); if (err.empty()) err = e.what(); }
        };
        const unsigned nt = records < (1u << 16) ? 1u
                            : (unsigned)std::min<uint64_t>(std::min<uint64_t>(n_items, 16), std::max(1u, std::thread::hardware_concurrency()));
        std::vector<std::thread> th;
        for (unsigned i = 1; i < nt; i++) th.emplace_back(work);
        work();
        for (std::thread& t : th) t.join();
        if (!err.empty()) throw CudaErr(err);
        CK(cudaSetDevice(dev));

        for_each_device(c, [](jlp_ctx* k) { free_haps(k); });
        c->haps.clear();
        for (const auto& S : stores) {
            attach_hap(c, S);
            for (jlp_ctx* k : c->kids) attach_hap(k, S);
        }
        if (stats) {
            const auto t1 = std::chrono::steady_clock::now();
            stats->count_ms = count_ms;
            stats->scan_ms = scan_ms;
            stats->write_ms = write_ms;
            stats->store_ms = std::chrono::duration<double, std::milli>(t1 - t_gen).count();
            stats->total_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
            stats->records = records;
            stats->d2h_bytes = words * 8;
            stats->table_bytes = rows * 2 * sizeof(uint4);
            stats->table_in_smem = (int)mp.tab_smem;
            stats->max_slots = max_slots;
        }
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
        if (!c->kids.empty()) {        // the parent keeps the host tables (read length, checks); every device gets its copy
            for (jlp_ctx* k : c->kids) {
                const int rc = jlp_set_profile(k, end, read_length, nq, probs, quals);
                if (rc != JLP_OK) throw ArgErr(k->err);
            }
            c->have_prof[end] = true;
            return;
        }
        const EndTables& t = c->tab[end];
        c->d_meta[end].upload(t.meta, c->s_compute);
        c->d_entry64[end].upload(t.entry64, c->s_compute);
        c->d_coin[end].upload(t.coin, c->s_compute);
        c->d_mis[end].upload(t.mis, c->s_compute);
        CK(cudaStreamSynchronize(c->s_compute));
        c->h2d_bytes += t.meta.size() * 4 + t.entry64.size() * 16 + 256 * 8;
        c->have_prof[end] = true;
    });
}

static void run_any(jlp_ctx* c, bool use_haps, const jlp_illumina_params* p, Sink& s, jlp_run_stats* stats) {
    if (c->kids.empty()) run(c, use_haps, p, s, stats);
    else run_multi(c, use_haps, p, s, stats);
}

int jlp_illumina_ref(jlp_ctx* c, const jlp_illumina_params* p, jlp_run_stats* stats) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() { Sink s; s.kind = SINK_FILES; run_any(c, false, p, s, stats); });
}
int jlp_illumina_hap(jlp_ctx* c, const jlp_illumina_params* p, jlp_run_stats* stats) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() { Sink s; s.kind = SINK_FILES; run_any(c, true, p, s, stats); });
}

int jlp_illumina_to_memory(jlp_ctx* c, int use_haplotypes, const jlp_illumina_params* p, char* out1, uint64_t cap1,
                           uint64_t* len1, char* out2, uint64_t cap2, uint64_t* len2, jlp_run_stats* stats) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        Sink s;
        s.kind = SINK_MEMORY;
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
        Sink s;
        s.kind = SINK_STREAM; s.chunk_cb = cb; s.chunk_user = user;
        run_any(c, use_haplotypes != 0, p, s, stats);
    });
}

int jlp_illumina_device_only(jlp_ctx* c, int use_haplotypes, const jlp_illumina_params* p, jlp_run_stats* stats) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() { Sink s; s.kind = SINK_NONE; run_any(c, use_haplotypes != 0, p, s, stats); });
}

int jlp_illumina_group_counts(jlp_ctx* c, int use_haplotypes, const jlp_illumina_params* p, uint64_t* counts,
                              uint64_t cap, uint64_t* n_groups) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        if (!p) throw ArgErr("params is NULL");
        if (c->chrom_off.size() < 2) throw ArgErr("no reference genome has been set");
        if (use_haplotypes && c->haps.empty()) throw ArgErr("no haplotypes have been added");
        const int n_ends = p->paired || p->matepair ? 2 : 1;
        std::vector<std::vector<uint64_t>> cnt = apportion(c, use_haplotypes != 0, p, p->n_reads / n_ends);
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

struct PbGroups {
    std::vector<uint64_t> group_off;      // read-index prefix offsets
    std::vector<GroupDev> groups;
    std::vector<uint8_t> strpool;
    std::vector<Job> jobs;
};

// reads -> haplotypes -> chromosomes, as for Illumina with one "end" (PacBioOneGenome::add_n_reads, src/hts_pacbio.h)
PbGroups pb_groups(jlp_ctx* c, bool use_haps, const jlp_pacbio_params* P) {
    if (c->chrom_off.size() < 2) throw ArgErr("no reference genome has been set");
    if (use_haps && c->haps.empty()) throw ArgErr("no haplotypes have been added");
    if (use_haps) finish_upload(c);
    const uint64_t n_chroms = c->chrom_off.size() - 1, n_haps = c->haps.size();
    std::vector<uint64_t> sizes;
    std::vector<std::vector<uint64_t>> counts;
    if (!use_haps) {
        for (uint64_t i = 0; i < n_chroms; i++) sizes.push_back(c->chrom_off[i + 1] - c->chrom_off[i]);
        counts = apportion_sizes(P->seed, P->n_reads, 1, n_chroms, nullptr, sizes.data());
    } else {
        if (!P->haplotype_probs) throw ArgErr("haplotype_probs is NULL");
        for (const HapDev& h : c->haps) sizes.insert(sizes.end(), h.len.begin(), h.len.end());
        counts = apportion_sizes(P->seed, P->n_reads, n_haps, n_chroms, P->haplotype_probs, sizes.data());
    }
    PbGroups G;
    G.group_off.push_back(0);
    const std::string prefix = P->out_prefix ? P->out_prefix : "";
    auto add = [&](const std::string& gname, uint64_t chrom, const uint8_t* seq, uint64_t len, uint64_t count) {
        GroupDev g;
        const std::string pre = "@" + gname + "-" + c->chrom_names[chrom] + "-";
        g.seq = seq; g.len = len;
        g.prefix_off = (uint32_t)G.strpool.size(); g.prefix_len = (uint32_t)pre.size();
        G.strpool.insert(G.strpool.end(), pre.begin(), pre.end());
        g.bc_off = 0; g.bc_len = 0;
        G.groups.push_back(g);
        G.group_off.push_back(G.group_off.back() + count);
        if (count > 0 && len == 0) throw ArgErr("a chromosome of length 0 was given reads");
    };
    if (!use_haps) {
        for (uint64_t i = 0; i < n_chroms; i++) add(c->genome_name, i, c->genome.p + kPad + c->chrom_off[i], sizes[i], counts[0][i]);
        G.jobs.push_back(Job{0, P->n_reads, prefix});
    } else {
        for (uint64_t h = 0; h < n_haps; h++) {
            const uint64_t lo = G.group_off.back();
            for (uint64_t i = 0; i < n_chroms; i++) {
                if (counts[h][i]) ensure_hap_chrom(c, h, i);        // materialised when first read from
                add(c->haps[h].name(), i, c->haps[h].seq[i], c->haps[h].len[i], counts[h][i]);
            }
            if (P->sep_files) G.jobs.push_back(Job{lo, G.group_off.back(), prefix + "_" + c->haps[h].name()});
        }
        if (!P->sep_files) G.jobs.push_back(Job{0, G.group_off.back(), prefix});
    }
    return G;
}

// The driver: per batch the per-read quantities are prepared on the host (batch k + 1 on a helper thread while batch k
// is on the device), then plan upload, k_pb_plan, scan, k_pb_reads, optional BGZF, copy, and the write of batch k
// overlaps the next batch.  Callbacks are called on the calling thread between batches.
void run_pacbio(jlp_ctx* c, bool use_haps, const jlp_pacbio_params* P, int sink_kind, char* mem, uint64_t cap, uint64_t* mem_len,
                jlp_run_stats* stats) {
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
    if (P->compress < 0 || P->compress > 9) throw ArgErr("\nInvalid bgzip compress level. It must be in range [0,9].");
    if (P->compress > 0) {
        const std::string m = P->comp_method ? P->comp_method : "";
        if (m != "gzip" && m != "bgzip") throw ArgErr("\nUnrecognized compression method.");
    }
    finish_upload(c);
    const PbGroups G = pb_groups(c, use_haps, P);
    const bool dev_z = P->compress > 0 && sink_kind == SINK_FILES &&
                       (P->comp_engine == JLP_COMP_DEVICE || (P->comp_engine == JLP_COMP_AUTO && P->compress <= 6));
    const int zmethod = P->compress <= 0 || dev_z || sink_kind != SINK_FILES ? -1
                        : (P->n_threads > 1 || std::string(P->comp_method) == "bgzip") ? DEFLATE_BGZF : DEFLATE_GZIP;
    // every buffer belongs to the context: pinning (and unpinning) a gigabyte of host memory on every call cost more than
    // generating the reads, and a dozen device allocations and frees per call several milliseconds
    DevBuf<GroupDev>& d_groups = c->pb_groups;
    DevBuf<uint8_t>&d_strpool = c->pb_strpool, &d_out = c->pb_out, &d_zslots = c->pb_zslots, &d_zout = c->pb_zout, &d_zcode = c->pb_zcode;
    DevBuf<PbRead>& d_reads = c->pb_reads;
    DevBuf<uint32_t>&d_rec_len = c->pb_rec_len, &d_rec_local = c->pb_rec_local, &d_zlen = c->pb_zlen;
    DevBuf<uint64_t>&d_block_tot = c->pb_block_tot, &d_block_base = c->pb_block_base, &d_totals = c->pb_totals, &d_zoff = c->pb_zoff;
    // two host buffers: the writer threads copy batch k into the file while batch k + 1 is prepared, generated and copied
    PinBuf<uint8_t>* h_buf = c->pb_h_buf;
    Mapping h_map[2];
    std::atomic<int> h_pending[2];
    h_pending[0] = 0; h_pending[1] = 0;
    uint64_t n_batch = 0;
    auto settle = [&](int k) { c->writers.wait(h_pending[k]); h_map[k].unmap(); };
    struct Settle { decltype(settle)& f; ~Settle() { f(0); f(1); } } settle_all{settle};       // also on error paths, before fd closes
    d_groups.upload(G.groups, c->s_compute);
    d_strpool.upload(G.strpool, c->s_compute);
    d_totals.ensure(4);
    CK(cudaMemsetAsync(d_totals.p, 0, 4 * sizeof(uint64_t), c->s_compute));
    uint64_t B = P->batch_reads ? P->batch_reads : 32768;
    // a chain of duplicates never leaves its pool (src/hts.h:266-267): batches are whole pools, so a duplicate's leader is in
    // its batch
    if (dups) B = std::max<uint64_t>(P->read_pool_size, B / P->read_pool_size * P->read_pool_size);
    uint32_t max_prefix = 0;
    for (const GroupDev& g : G.groups) max_prefix = std::max(max_prefix, g.prefix_len);
    const uint64_t c_rev = thr_ld_lt(0.5).thr;
    jlp_run_stats st;
    std::memset(&st, 0, sizeof st);
    uint64_t mem_used = 0;
    cudaEvent_t ev[3];
    for (cudaEvent_t& e : ev) CK(cudaEventCreate(&e));
    for (const Job& job : G.jobs) {
        int fd = -1;
        uint64_t fpos = 0;
        std::string fname;
        if (sink_kind == SINK_FILES) {
            fname = job.file_prefix + "_R1.fq" + (P->compress > 0 ? ".gz" : "");        // write_reads_one_filetype_, src/hts.h:344
            fd = ::open(fname.c_str(), O_RDWR | O_CREAT | O_TRUNC, 0644);
            if (fd < 0) throw IoErr("Unable to open file " + fname + ".\n");
        }
        try {
            // this shard's part of the job: whole pools, so that chains of duplicates stay inside it
            uint64_t s_lo = job.lo, s_hi = job.hi;
            if (P->shard_count > 1) {
                if (P->shard_index >= P->shard_count) throw ArgErr("shard_index >= shard_count");
                const uint64_t pool = std::max<uint64_t>(P->read_pool_size, 1), n_pools = (job.hi - job.lo + pool - 1) / pool;
                uint64_t p_lo, p_hi;
                shard_range(0, n_pools, P->shard_index, P->shard_count, p_lo, p_hi);
                s_lo = std::min(job.hi, job.lo + p_lo * pool);
                s_hi = std::min(job.hi, job.lo + p_hi * pool);
            }
            // ---- per-read quantities on the host (read length, passes, error probabilities, thresholds): batch k + 1 is
            //      prepared by a helper thread (which spreads the reads over n_threads workers) while the device
            //      generates batch k and the sink takes it
            struct Prepared { std::vector<PbRead> plan; uint64_t bound = 0; std::string err; };
            auto prepare = [&](uint64_t b0, uint32_t n, Prepared& out) {
                try {
                    std::vector<PbRead>& plan = out.plan;
                    plan.resize(n);
                    // chains of duplicates: read i re-reads iff the draw made after read i - 1 says so and i does not open a pool
                    std::vector<uint32_t> lead(n, kPbNoLeader);
                    if (dups)
                        for (uint32_t i = 1; i < n; i++)
                            if ((b0 + i - job.lo) % P->read_pool_size != 0 && (t_dup.all || pb_dup_draw(P->seed, b0 + i - 1) < t_dup.thr))
                                lead[i] = lead[i - 1] == kPbNoLeader ? i - 1 : lead[i - 1];
                    // the reads are independent given their leaders: split over the host threads (n_threads, at most 64),
                    // first the leaders, then the duplicates (which take their leader's chromosome and length)
                    const uint32_t nt = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(P->n_threads, 1), 64);
                    std::vector<uint64_t> part(nt, 0);
                    std::vector<std::string> errs(nt);
                    for (int pass = 0; pass < (dups ? 2 : 1); pass++) {
                        auto work = [&](uint32_t k) {
                            try {
                                for (uint32_t i = k; i < n; i += nt) {
                                    if ((lead[i] != kPbNoLeader) != (pass == 1)) continue;
                                    const uint64_t j = b0 + i;
                                    PbSample smp;
                                    size_t g;
                                    if (pass == 0) {
                                        g = (size_t)(std::upper_bound(G.group_off.begin(), G.group_off.end(), j) - G.group_off.begin()) - 1;
                                        smp = pb_sample(model, P->seed, j, G.groups[g].len);
                                    } else {
                                        g = plan[lead[i]].group;
                                        smp = pb_sample_passes(model, P->seed, j, plan[lead[i]].read_length);
                                    }
                                    std::memset(&plan[i], 0, sizeof(PbRead));
                                    pb_read_model(model, P->seed, j, smp, plan[i]);
                                    plan[i].group = (uint32_t)g;
                                    plan[i].leader = lead[i];
                                    part[k] += max_prefix + 24 + 2 * smp.read_length + 5;
                                }
                            } catch (const std::exception& e) { errs[k] = e.what(); }
                        };
                        std::vector<std::thread> th;
                        for (uint32_t k = 1; k < nt; k++) th.emplace_back(work, k);
                        work(0);
                        for (std::thread& t : th) t.join();
                    }
                    for (const std::string& e : errs) if (!e.empty()) { out.err = e; return; }
                    out.bound = 0;
                    for (uint64_t v : part) out.bound += v;
                } catch (const std::exception& e) { out.err = e.what(); }
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
                d_reads.ensure(n_max); d_rec_len.ensure(n_max); d_rec_local.ensure(n_max);
                const uint64_t nsb_max = (n_max + kScanBlock - 1) / kScanBlock;
                d_block_tot.ensure(nsb_max); d_block_base.ensure(nsb_max);
            }
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
                if (!cur.err.empty()) throw ArgErr(cur.err);
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
                d_reads.ensure(n);
                d_rec_len.ensure(n); d_rec_local.ensure(n);
                const uint32_t nsb = (n + kScanBlock - 1) / kScanBlock;
                d_block_tot.ensure(nsb); d_block_base.ensure(nsb);
                if (bound + 64 > d_out.n) {      // batches differ in size: grow with slack, and at once to what a full batch will need
                    const uint64_t full = n ? bound / n * std::min<uint64_t>(B, s_hi - s_lo) : bound;
                    const uint64_t want = std::max(bound, full);
                    d_out.ensure(want + want / 4 + 64);
                }
                t_alloc += now() - t0;
                CK(cudaMemcpyAsync(d_reads.p, plan.data(), n * sizeof(PbRead), cudaMemcpyHostToDevice, c->s_compute));
                st.h2d_bytes += n * sizeof(PbRead);
                CK(cudaEventRecord(ev[0], c->s_compute));
                CK(launch_pb_plan(d_reads.p, n, b0, P->seed, d_groups.p, c_rev, d_rec_len.p, c->s_compute));
                if (dups) { CK(launch_pb_dups(d_reads.p, n, b0, P->seed, d_groups.p, d_rec_len.p, c->s_compute)); st.kernel_launches++; }
                CK(launch_scan(d_rec_len.p, n, 1, d_rec_local.p, d_block_tot.p, d_block_base.p, d_totals.p, c->s_compute));
                CK(launch_pb_reads(d_reads.p, n, b0, P->seed, d_groups.p, d_strpool.p, d_rec_local.p, d_block_base.p, d_out.p,
                                   c->s_compute));
                CK(cudaEventRecord(ev[1], c->s_compute));
                st.kernel_launches += 4;
                const uint32_t nblk = (uint32_t)((bound + kBgzfIn - 1) / kBgzfIn) + 1;
                if (dev_z) {
                    d_zslots.ensure((size_t)nblk * kBgzfSlot); d_zout.ensure((size_t)nblk * kBgzfSlot);
                    d_zlen.ensure(2 * nblk); d_zoff.ensure(2 * nblk); d_zcode.ensure(kBgzfCodeBytes);
                    CK(launch_bgzf(d_out.p, d_out.p, d_totals.p, nblk, P->compress >= 4, d_zslots.p, d_zslots.p, d_zlen.p, d_zlen.p + nblk,
                                   d_zoff.p, d_zoff.p + nblk, d_zout.p, d_zout.p, d_zcode.p, c->s_compute));
                    st.kernel_launches += kBgzfLaunches;
                }
                CK(cudaEventRecord(ev[2], c->s_compute));
                uint64_t tot[4];
                CK(cudaMemcpyAsync(tot, d_totals.p, sizeof tot, cudaMemcpyDeviceToHost, c->s_compute));
                t0 = now();
                CK(cudaStreamSynchronize(c->s_compute));
                t_sync += now() - t0;
                if (tot[0] > bound) throw std::runtime_error("internal: PacBio batch larger than its bound");
                float ms = 0;
                CK(cudaEventElapsedTime(&ms, ev[0], ev[1])); st.reads_ms += ms; st.device_ms += ms;
                CK(cudaEventElapsedTime(&ms, ev[1], ev[2])); if (dev_z) { st.bgzf_ms += ms; st.device_ms += ms; }
                st.pairs += n; st.batches++; st.bytes_out[0] += tot[0];
                if (dev_z) st.z_bytes[0] += tot[2];
                if (sink_kind == SINK_NONE) { if (P->progress_cb) P->progress_cb(P->cb_user, n); continue; }
                const uint64_t nb = dev_z ? tot[2] : tot[0];
                const int hk = (int)(n_batch++ & 1);
                settle(hk);                                     // the slices of the batch before last are in the file
                PinBuf<uint8_t>& h_out = h_buf[hk];
                if (nb + 64 > h_out.n) {          // like d_out: at once to what a full batch will need (pinning is slow)
                    const uint64_t full = n ? nb / n * std::min<uint64_t>(B, s_hi - s_lo) : nb;
                    const uint64_t want = std::max(nb, full);
                    h_out.ensure(want + want / 4 + 64);
                }
                CK(cudaMemcpy(h_out.p, dev_z ? d_zout.p : d_out.p, nb, cudaMemcpyDeviceToHost));
                st.d2h_bytes += nb;
                if (sink_kind == SINK_MEMORY) {
                    if (mem && mem_used + nb <= cap) std::memcpy(mem + mem_used, h_out.p, nb);
                    mem_used += nb;
                } else {
                    const uint8_t* src = h_out.p;
                    uint64_t len = nb;
                    std::vector<uint8_t> z;
                    if (zmethod >= 0) {
                        const std::string e = deflate_members(zmethod, P->compress, h_out.p, nb, z);
                        if (!e.empty()) throw IoErr(e);
                        src = z.data(); len = z.size();
                    }
                    // several writer threads: the file is extended and the batch copied into a mapping of the new range
                    // in parallel (see Mapping) while the next batch is on its way; otherwise one pwrite
                    struct statvfs vfs;
                    if (zmethod < 0 && P->n_threads > 1 && len > (8u << 20) && ::fstatvfs(fd, &vfs) == 0 &&
                        (uint64_t)vfs.f_bavail * vfs.f_frsize > 2 * len + (64ull << 20) && ::ftruncate(fd, (off_t)(fpos + len)) == 0 &&
                        map_range(fd, fpos, len, h_map[hk])) {
                        c->writers.start((size_t)std::min<uint64_t>(P->n_threads, 64));
                        const uint64_t slice = 8ull << 20;
                        for (uint64_t o = 0; o < len; o += slice) {
                            uint8_t* dst = h_map[hk].at + o;
                            const uint8_t* from = src + o;
                            const uint64_t nb2 = std::min(slice, len - o);
                            c->writers.submit(&h_pending[hk], [dst, from, nb2]() { std::memcpy(dst, from, nb2); return std::string(); });
                        }
                    } else {
                        const std::string w = pwrite_all(fd, src, len, fpos);
                        if (!w.empty()) throw IoErr("Error writing to file " + fname + ": " + w);
                    }
                    fpos += len;
                }
                if (P->progress_cb) P->progress_cb(P->cb_user, n);                  // Progress::increment, src/hts.h:414
            }
            if (prep_thread.joinable()) prep_thread.join();
            settle(0); settle(1);
            if (trace)
                std::fprintf(stderr, "[jlp trace] pacbio job %llu reads: %.4f s (first prepare %.4f, waiting for later ones %.4f, "
                             "device allocations %.4f, waiting for the device %.4f)\n", (unsigned long long)(s_hi - s_lo), now() - t_job,
                             t_first, t_join, t_alloc, t_sync);
            if (fd >= 0 && (dev_z || zmethod == DEFLATE_BGZF)) {
                const std::string w = pwrite_all(fd, kBgzfEof, sizeof kBgzfEof, fpos);
                if (!w.empty()) throw IoErr("Error writing to file " + fname + ": " + w);
            }
        } catch (...) {
            settle(0); settle(1);
            if (fd >= 0) ::close(fd);
            for (cudaEvent_t& e : ev) cudaEventDestroy(e);
            throw;
        }
        if (fd >= 0) ::close(fd);
    }
    for (cudaEvent_t& e : ev) cudaEventDestroy(e);
    if (mem_len) *mem_len = mem_used;
    if (stats) *stats = st;
}

}  // namespace

int jlp_pacbio(jlp_ctx* c, int use_haplotypes, const jlp_pacbio_params* p, jlp_run_stats* stats) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        if (!p || !p->out_prefix || !*p->out_prefix) throw ArgErr("out_prefix is empty");
        jlp_ctx* d = first_device(c);
        run_pacbio(d, use_haplotypes != 0, p, SINK_FILES, nullptr, 0, nullptr, stats);
    });
}

int jlp_pacbio_to_memory(jlp_ctx* c, int use_haplotypes, const jlp_pacbio_params* p, char* out, uint64_t cap, uint64_t* len,
                         jlp_run_stats* stats) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        uint64_t need = 0;
        jlp_ctx* d = first_device(c);
        run_pacbio(d, use_haplotypes != 0, p, out ? SINK_MEMORY : SINK_NONE, out, cap, &need, stats);
        if (len) *len = need;
        if (out && need > cap) throw ArgErr("output buffer too small");
    });
}

int jlp_pacbio_read_plan(jlp_ctx* c, int use_haplotypes, const jlp_pacbio_params* p, uint64_t* group, uint64_t* read_len,
                         uint64_t* split_pos, double* passes_left, double* passes_right) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() {
        PbModel model;
        pb_model_from(p, model);
        const PbGroups G = pb_groups(first_device(c), use_haplotypes != 0, p);
        const Thr t_dup = thr_double_lt(p->prob_dup);
        const bool dups = t_dup.thr != 0 || t_dup.all;
        for (const Job& job : G.jobs) {
            uint64_t leader = job.lo;
            PbSample ls{};
            size_t lg = 0;
            for (uint64_t j = job.lo; j < job.hi; j++) {
                const bool dup = dups && j > job.lo && (j - job.lo) % std::max<uint64_t>(p->read_pool_size, 1) != 0 &&
                                 (t_dup.all || pb_dup_draw(p->seed, j - 1) < t_dup.thr);
                PbSample s;
                if (!dup) {
                    leader = j;
                    lg = (size_t)(std::upper_bound(G.group_off.begin(), G.group_off.end(), j) - G.group_off.begin()) - 1;
                    s = ls = pb_sample(model, p->seed, j, G.groups[lg].len);
                } else {
                    s = pb_sample_passes(model, p->seed, j, ls.read_length);
                }
                (void)leader;
                if (group) group[j] = lg;
                if (read_len) read_len[j] = s.read_length;
                if (split_pos) split_pos[j] = s.split_pos;
                if (passes_left) passes_left[j] = s.passes_left;
                if (passes_right) passes_right[j] = s.passes_right;
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
        c = first_device(c);
        const uint32_t nblk = (uint32_t)((n + kBgzfIn - 1) / kBgzfIn);
        DevBuf<uint8_t> d_in, d_slots, d_out, d_code;
        DevBuf<uint32_t> d_zlen;
        DevBuf<uint64_t> d_zoff, d_tot;
        d_in.ensure(n + 64); d_slots.ensure((size_t)nblk * kBgzfSlot); d_out.ensure((size_t)nblk * kBgzfSlot);
        d_zlen.ensure(nblk); d_zoff.ensure(nblk); d_tot.ensure(4); d_code.ensure(kBgzfCodeBytes);
        const uint64_t tot[4] = {n, 0, 0, 0};
        if (n) CK(cudaMemcpyAsync(d_in.p, in, n, cudaMemcpyHostToDevice, c->s_compute));
        CK(cudaMemcpyAsync(d_tot.p, tot, sizeof tot, cudaMemcpyHostToDevice, c->s_compute));
        CK(launch_bgzf(d_in.p, d_in.p, d_tot.p, nblk, level >= 4, d_slots.p, d_slots.p, d_zlen.p, d_zlen.p, d_zoff.p, d_zoff.p, d_out.p,
                       d_out.p, d_code.p, c->s_compute));
        uint64_t back[4];
        CK(cudaMemcpyAsync(back, d_tot.p, sizeof back, cudaMemcpyDeviceToHost, c->s_compute));
        CK(cudaStreamSynchronize(c->s_compute));
        *len = back[2] + sizeof kBgzfEof;
        if (!out) return;
        if (cap < *len) throw ArgErr("output buffer too small");
        if (back[2]) CK(cudaMemcpy(out, d_out.p, back[2], cudaMemcpyDeviceToHost));
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
