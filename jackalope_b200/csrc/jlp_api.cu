// C ABI (include/jlp_b200.h): the context, genome, haplotype and profile calls, the stateless helpers, and the
// definitions behind jlp_ctx.h.  The drivers are jlp_run_illumina.cu, jlp_run_pacbio.cu, jlp_run_vcf.cu,
// jlp_run_haps.cu and jlp_run_vcf_read.cu.
#include "jlp_ctx.h"

#include <cmath>
#include <cstring>

#include "jlp_deflate.h"
#include "jlp_draws.h"

using namespace jlp;

namespace {

std::string g_create_error;

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

}  // namespace

namespace jlp {

int fail(jlp_ctx* c, int code, const std::string& msg) {
    if (c) c->err = msg; else g_create_error = msg;
    return code;
}

// The device of the calls that use only the first one (PacBio, create_haplotypes, ...), made current.
Device& device0(jlp_ctx* c) {
    CK(cudaSetDevice(c->dev[0]->id));
    return *c->dev[0];
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

// Contiguous, near-equal split of a job's pair-index range over shards (the even split of
// split_int, src/util.h:245-258, applied to GPUs instead of threads).
void shard_range(uint64_t job_lo, uint64_t job_hi, uint32_t si, uint32_t S, uint64_t& lo, uint64_t& hi) {
    const uint64_t nj = job_hi - job_lo;
    lo = job_lo + nj / S * si + std::min<uint64_t>(si, nj % S);
    hi = lo + nj / S + (si < nj % S ? 1 : 0);
}

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

// The compression arguments of every driver.  A level <= 0 is no compression, and the method is then not looked at.
void check_compression(int compress, const char* comp_method, int comp_engine) {
    const std::string m = comp_method ? comp_method : "";
    if (compress > 0 && m != "gzip" && m != "bgzip") throw ArgErr("\nUnrecognized compression method.");  // src/hts.h:470
    if (compress > 9) throw ArgErr("\nInvalid bgzip compress level of " + std::to_string(compress) +
                                   ". It must be in range [0,9].");                                      // src/io.h:113-117
    if (comp_engine < JLP_COMP_AUTO || comp_engine > JLP_COMP_DEVICE) throw ArgErr("comp_engine must be 0 (auto), 1 (host) or 2 (device)");
}

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

// attach a haplotype to a context: unmutated chromosomes alias the reference, the others wait for a run to touch them
void attach_hap(jlp_ctx* c, const std::shared_ptr<HapStore>& S) {
    c->haps.push_back(S);
    for (auto& d : c->dev) {
        std::vector<const uint8_t*> seq;
        for (size_t ci = 0; ci < S->chrom.size(); ci++)
            seq.push_back(S->chrom[ci].n_muts == 0 ? d->genome.p + kPad + c->chrom_off[ci] : nullptr);
        d->hap_seq.push_back(std::move(seq));
    }
}

// the reference's chromosome lengths; positions in a chromosome are 32 bits wide (TreeRegion, MutTile, VrLine)
std::vector<uint64_t> chrom_lengths(const jlp_ctx* c) {
    const uint64_t nc = c->chrom_off.size() - 1;
    std::vector<uint64_t> len(nc);
    for (uint64_t ci = 0; ci < nc; ci++) {
        len[ci] = c->chrom_off[ci + 1] - c->chrom_off[ci];
        if (len[ci] >> 32) throw ArgErr("chromosomes of 2^32 bases or more are not supported");
    }
    return len;
}

void store_haps(jlp_ctx* c, const HapRegions& G, unsigned threads) {
    const uint64_t nc = c->chrom_off.size() - 1;
    const size_t n_haps = G.names.size(), n_items = n_haps * nc;
    const int dev = c->dev[0]->id;
    std::vector<std::shared_ptr<HapStore>> stores(n_haps);
    uint64_t records = 0;
    for (size_t h = 0; h < n_haps; h++) {
        stores[h] = std::make_shared<HapStore>();
        stores[h]->name = G.names[h];
        stores[h]->chrom.resize(nc);
    }
    for (size_t r = 0; r < n_items; r++) records += G.n[r];
    const unsigned nt = records < (1u << 16) ? 1u : threads;
    parallel_for(n_items, nt, [&](uint64_t r) {
        HapChromHost& H = stores[r / nc]->chrom[r % nc];
        const uint64_t M = G.n[r];
        H.size = G.size[r];
        H.n_muts = M;
        H.pool_bytes = G.pool[r];
        if (!M) return;
        H.packed.resize(4 * M + (G.pool[r] + 7) / 8);
        CK(cudaSetDevice(dev));
        CK(cudaMemcpy(H.packed.data(), G.src[r], H.packed.size() * 8, cudaMemcpyDeviceToHost));
    });

    clear_haps(c);
    for (const auto& S : stores) attach_hap(c, S);
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

// host threads for `items` independent pieces of work: at most 16, and no more than the machine runs at once
unsigned host_threads(uint64_t items) {
    return (unsigned)std::min<uint64_t>(std::min<uint64_t>(items, 16), std::max(1u, std::thread::hardware_concurrency()));
}

// milliseconds between two recorded events
float elapsed_ms(cudaEvent_t a, cudaEvent_t b) {
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, a, b));
    return ms;
}

}  // namespace jlp

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
    const unsigned nt = total < (1u << 16) ? 1u : host_threads(nc);
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
