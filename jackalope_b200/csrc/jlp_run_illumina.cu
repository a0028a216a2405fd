// The Illumina driver (jlp_illumina_*): the batch pipeline that stands in for write_reads_cpp_ /
// write_reads_cpp_sep_files_ / write_reads_one_filetype_ (/root/reference/src/hts.h:323-552), on one device or on
// several (jlp_ctx_create_multi).
#include "jlp_ctx.h"

#include <fcntl.h>
#include <sys/stat.h>
#include <sys/statvfs.h>
#include <unistd.h>

#include <array>
#include <cerrno>
#include <cstring>
#include <deque>

#include "jlp_deflate.h"
#include "jlp_draws.h"

using namespace jlp;

namespace {

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

int ends_of(const jlp_illumina_params* P) { return P->paired || P->matepair ? 2 : 1; }
// pairs of a duplicate pool: the pool closes at >= read_pool_size reads
uint64_t pool_pairs(const jlp_illumina_params* P) { return (P->read_pool_size + ends_of(P) - 1) / ends_of(P); }

// the argument checks the C++ layer of the reference performs, plus the ranges of the additions
void check_params(const jlp_ctx* c, bool use_haps, const jlp_illumina_params* P, SinkKind kind) {
    if (!P) throw ArgErr("params is NULL");
    const int n_ends = ends_of(P);
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

LayoutSpec illumina_spec(const jlp_ctx* c, bool use_haps, const jlp_illumina_params* P) {
    LayoutSpec S(use_haps, P, P->n_reads / ends_of(P));
    S.barcodes = P->barcodes;
    S.read_len = (uint32_t)c->tab[0].L;
    return S;
}

typedef std::vector<std::pair<uint64_t, uint64_t>> Ranges;
typedef std::vector<std::array<uint64_t, 2>> PerJobBytes;

// What a multi-GPU run tells each of its devices (jlp_ctx_create_multi); a plain call leaves everything empty.
struct Piece {
    const Ranges* ranges = nullptr;       // [jobs] the pair range of every job this call generates (else: the shard of P)
    const PerJobBytes* base = nullptr;    // [jobs] where this call's bytes start in each job's files / in the memory sink
    bool shared_files = false;            // the files exist, created and sized by the caller: open without truncating, no EOF block
    const std::vector<std::string>* suffix = nullptr;   // [jobs] zlib: this call writes <name><suffix>, the caller joins them
};

// the first and last group the pairs [lo, hi) of job read: those of the pairs, and through a duplicate chain's leader
// possibly the one before (a leader lies at most pool_pairs - 1 pairs before its duplicate, never before the job's start)
std::pair<size_t, size_t> groups_of(const Layout& Y, const jlp_illumina_params* P, const Job& job, uint64_t lo, uint64_t hi) {
    const uint64_t first_pair = lo - std::min<uint64_t>(lo - job.lo, pool_pairs(P) - 1);
    const size_t g_lo = (size_t)(std::upper_bound(Y.group_off.begin(), Y.group_off.end(), first_pair) - Y.group_off.begin()) - 1;
    const size_t g_hi = std::min((size_t)(std::upper_bound(Y.group_off.begin(), Y.group_off.end(), hi - 1) - Y.group_off.begin()) - 1,
                                 Y.groups.size() - 1);
    return {std::min(g_lo, g_hi), g_hi};
}

// The groups' sequences on d: the reference's chromosomes, or the haplotype chromosomes the ranges touch (materialised now).
void bind_sequences(const jlp_ctx* c, Device& d, bool use_haps, const jlp_illumina_params* P, Layout& Y, const Ranges& ranges) {
    if (ranges.size() != Y.jobs.size()) throw std::runtime_error("internal: one range per job");
    for (size_t k = 0; k < Y.jobs.size() && use_haps; k++) {
        if (ranges[k].second <= ranges[k].first) continue;
        const auto [g_lo, g_hi] = groups_of(Y, P, Y.jobs[k], ranges[k].first, ranges[k].second);
        for (size_t g = g_lo; g <= g_hi; g++) ensure_hap_chrom(c, d, Y.group_hap[g], Y.group_chrom[g]);
    }
    for (size_t g = 0; g < Y.groups.size(); g++)
        Y.groups[g].seq = use_haps ? d.hap_seq[Y.group_hap[g]][Y.group_chrom[g]] : d.genome.p + kPad + c->chrom_off[g];
}

// The kernels' parameters, with the fragment table, the groups, the string pool and a cleared status word uploaded to d
GenParams gen_params(const jlp_ctx* c, Device& d, const jlp_illumina_params* P, const Layout& Y) {
    const int n_ends = ends_of(P);
    const double insp[2] = {P->ins_prob1, P->ins_prob2}, delp[2] = {P->del_prob1, P->del_prob2};
    GenParams gp;
    std::memset(&gp, 0, sizeof gp);
    gp.seed = P->seed;
    philox_round_keys(P->seed, gp.rk);
    gp.n_ends = n_ends; gp.L = (uint32_t)c->tab[0].L; gp.matepair = P->matepair != 0;
    gp.pool_pairs = pool_pairs(P);
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
    d.d_group_off.upload(Y.group_off, d.s_compute);
    d.d_groups.upload(Y.groups, d.s_compute);
    d.d_strpool.upload(Y.strpool, d.s_compute);
    d.d_status.ensure(1);
    CK(cudaMemsetAsync(d.d_status.p, 0, sizeof(uint32_t), d.s_compute));
    d.h2d_bytes += frag.size() * 8 + Y.group_off.size() * 8 + Y.groups.size() * sizeof(GroupDev) + Y.strpool.size();
    gp.frag_cdf = d.d_frag.p; gp.frag_guide = d.d_frag_guide.p; gp.frag_n = (uint32_t)frag.size(); gp.frag_min = P->frag_len_min;
    gp.group_off = d.d_group_off.p; gp.n_groups = (uint32_t)Y.groups.size();
    gp.groups = d.d_groups.p; gp.strpool = d.d_strpool.p; gp.status = d.d_status.p;
    return gp;
}

struct Batches { uint64_t B; uint32_t nblk; };   // pairs per batch, BGZF blocks of a file's batch

// The pairs per batch, the read kernel's record buffers in gp, and every slot's buffers: placement and scan; FASTQ for
// n_out files (none: no read kernel runs), pinned host copies of it (need_host); the device coder's (dev_z).
Batches size_batches(Device& d, GenParams& gp, const Layout& Y, const Ranges& ranges, const jlp_illumina_params* P, int n_out,
                     bool need_host, bool dev_z) {
    uint64_t max_range = 0;
    for (const auto& r : ranges) max_range = std::max(max_range, r.second - r.first);
    uint64_t B = P->batch_pairs ? P->batch_pairs : (1ull << 20);
    B = std::max<uint64_t>(1, std::min(B, max_range));
    uint32_t max_prefix = 0;
    for (const GroupDev& g : Y.groups) max_prefix = std::max(max_prefix, g.prefix_len);
    const uint64_t max_rec = (uint64_t)max_prefix + 20 + 5 + 2ull * gp.L + 4;
    B = std::max<uint64_t>(1, std::min<uint64_t>(B, 0xfff00000ull / max_rec));     // offsets inside a batch's output are 32 bits wide in k_reads
    gp.rec_buf = (uint32_t)((max_rec + 32 + 15) & ~15ull);   // a record at any 16-byte phase, and the 16 bytes the carry reads behind it
    gp.tpl_buf = (gp.L + 50u + 15u) & ~15u;     // the template, 16..31 bytes in front of it, 16 behind, the word over-read
    gp.cod_buf = (gp.L + 40u + 15u) & ~15u;     // base codes of a read's template (up to 2 more than the read with deletions), rounded up to the 16 of a lane
    if (n_out && !reads_fits(gp)) throw Unsupported("read_length " + std::to_string(gp.L) + " (with these chromosome names) needs more shared memory per "
                                                    "read pair than one SM has: the read kernel cannot hold such a record");
    const uint64_t n_rec_max = B * ends_of(P);
    const uint32_t nsb_max = (uint32_t)((B + kScanBlock - 1) / kScanBlock);
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
        for (int e = 0; e < n_out; e++) {
            s.out[e].ensure(B * max_rec + 64);
            // compressed bytes of a batch never exceed its FASTQ bytes plus the members' framing (an incompressible block is stored)
            // (the same size with and without compression: pinning a gigabyte again for the first compressed call took seconds)
            if (need_host) s.h_out[e].ensure(B * max_rec + (size_t)nblk * 64 + 64);
        }
        if (dev_z) s.z.ensure(nblk, B * max_rec, ends_of(P));
        s.busy = false;
    }
    return Batches{B, nblk};
}

// A deferred genome upload: the compute stream waits for exactly the uploads of the chromosomes the batch [b0, b1) reads.
// The first batch of this call's part [lo, hi) of the job copies, in the order the part reads them, all its chromosomes and
// nothing else (with N GPUs each needs about 1/N of the genome); the rest stays on the host until some run asks for it.
void wait_chromosomes(const jlp_ctx* c, Device& d, const Layout& Y, const jlp_illumina_params* P, const Job& job, uint64_t lo,
                      uint64_t hi, uint64_t b0, uint64_t b1, std::vector<char>& waited) {
    auto [g_lo, g_hi] = groups_of(Y, P, job, b0, b1);
    g_hi = std::min(g_hi, d.chrom_ev.size() - 1);
    g_lo = std::min(g_lo, g_hi);
    if (b0 == lo) issue_upload(c, d, g_lo, std::min(groups_of(Y, P, job, lo, hi).second, d.chrom_ev.size() - 1));
    issue_upload(c, d, g_lo, g_hi);
    for (size_t g = g_lo; g <= g_hi; g++)
        if (!waited[g]) { CK(cudaStreamWaitEvent(d.s_compute, d.chrom_ev[g], 0)); waited[g] = 1; }
}

// After a run's last batch: its time, the deferred upload's bookkeeping, the device's status word and the statistics.
void finish(Device& d, jlp_run_stats& st, uint64_t h2d_before, jlp_run_stats* stats) {
    CK(cudaEventRecord(d.ev_run[1], d.s_compute));
    CK(cudaEventSynchronize(d.ev_run[1]));
    st.run_ms = elapsed_ms(d.ev_run[0], d.ev_run[1]);
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
}

// One Illumina run on device d, with the run's Layout (make_layout) and parameters checked (check_params) by the caller.
// Returns the device coder's bytes per job and file: into SINK_NONE with the files' Compression Z, a dry run sizes them.
PerJobBytes run(const jlp_ctx* c, Device& d, bool use_haps, const jlp_illumina_params* P, const Compression& Z, Layout Y,
                Output& sink, jlp_run_stats* stats, const Piece& piece = Piece()) {
    const int n_ends = ends_of(P);
    const bool dev_z = Z.dev_z, need_host = sink.kind != SINK_NONE;
    if (use_haps) finish_upload(c, d);
    const uint64_t h2d_before = d.h2d_bytes;
    Ranges ranges;
    if (piece.ranges) ranges = *piece.ranges;
    else {
        const uint32_t S = P->shard_count > 1 ? P->shard_count : 1, si = P->shard_count > 1 ? P->shard_index : 0;
        for (const Job& j : Y.jobs) { uint64_t lo, hi; shard_range(j.lo, j.hi, si, S, lo, hi); ranges.emplace_back(lo, hi); }
    }
    bind_sequences(c, d, use_haps, P, Y, ranges);
    GenParams gp = gen_params(c, d, P, Y);
    const Batches b = size_batches(d, gp, Y, ranges, P, n_ends, need_host, dev_z);
    jlp_run_stats st{};
    PerJobBytes zbytes(Y.jobs.size());
    sink.begin(Z, P->compress, P->n_threads, d.writers);
    Quiesce quiesce{d, &sink};
    size_t jk = 0;
    // stage 2 of a batch: its kernels are done -> statistics, then its FASTQ starts its way to the host
    // (queued right behind the previous batch's copy, so the bus never idles)
    auto issue_copy = [&](Slot& s) {
        CK(cudaEventSynchronize(s.ev[5]));
        const float ms_place = elapsed_ms(s.ev[0], s.ev[1]), ms_reads = elapsed_ms(s.ev[2], s.ev[3]);
        const float ms_z = elapsed_ms(s.ev[3], s.ev[5]), ms_all = elapsed_ms(s.ev[0], s.ev[5]);
        st.place_ms += ms_place; st.reads_ms += ms_reads; st.device_ms += ms_all;
        if (dev_z) st.bgzf_ms += ms_z;
        for (int e = 0; e < n_ends; e++) {
            s.tot[e] = s.h_totals.p[e]; st.bytes_out[e] += s.tot[e];
            s.ztot[e] = dev_z ? s.h_totals.p[2 + e] : 0; st.z_bytes[e] += s.ztot[e];
            zbytes[jk][e] += s.ztot[e];
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
            sink.deliver(s.host, data, n, jk, n_ends);
        }
        if (P->progress_cb) P->progress_cb(P->cb_user, (uint64_t)s.pairs * n_ends);
        s.busy = false;
    };

    std::vector<char> chrom_waited(d.chrom_ev.size(), 0);
    for (jk = 0; jk < Y.jobs.size(); jk++) {
        const Job& job = Y.jobs[jk];
        const uint64_t lo = ranges[jk].first, hi = ranges[jk].second;
        if (P->abort_cb && P->abort_cb(P->cb_user)) throw Aborted();   // src/hts.h:536
        if (piece.ranges && hi <= lo) continue;                         // a multi-GPU device with no part in this job's files
        std::string names[2];
        for (int e = 0; e < n_ends; e++) names[e] = file_name(job, e, Z.want_gz, P) + (piece.suffix ? (*piece.suffix)[jk] : "");
        sink.open_job(names, n_ends, piece.base ? (*piece.base)[jk].data() : nullptr, piece.shared_files);
        // three batches in flight: batch b computes while b-1 crosses PCIe and b-2 is handed to the sink
        std::deque<Slot*> computing, copying;
        auto drain_one = [&]() {
            if (!copying.empty() && (computing.empty() || copying.size() >= 2)) { deliver(*copying.front()); copying.pop_front(); }
            else if (!computing.empty()) { issue_copy(*computing.front()); copying.push_back(computing.front()); computing.pop_front(); }
        };
        uint64_t bi = 0;
        for (uint64_t b0 = lo; b0 < hi; b0 += b.B, bi++) {
            Slot& s = d.slot[bi % 3];
            while (s.busy) drain_one();
            const uint32_t np = (uint32_t)std::min<uint64_t>(b.B, hi - b0);
            if (d.upload_pending && !use_haps) wait_chromosomes(c, d, Y, P, job, lo, hi, b0, b0 + np, chrom_waited);
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
                CK(s.z.launch(s.out[0].p, s.out[1].p, s.totals.p, b.nblk, P->compress, d.s_compute));
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
        sink.end_job(jk, n_ends, !piece.shared_files && !piece.suffix);
    }
    finish(d, st, h2d_before, stats);
    quiesce.armed = false;
    return zbytes;
}

// The FASTQ bytes per job and file that run() writes on device d for the given ranges: placement and scan only, the
// totals come back batch by batch (a few hundred microseconds each).
PerJobBytes count_bytes(const jlp_ctx* c, Device& d, bool use_haps, const jlp_illumina_params* P, Layout Y, const Ranges& ranges,
                        jlp_run_stats* stats) {
    const int n_ends = ends_of(P);
    if (use_haps) finish_upload(c, d);
    const uint64_t h2d_before = d.h2d_bytes;
    bind_sequences(c, d, use_haps, P, Y, ranges);
    GenParams gp = gen_params(c, d, P, Y);
    const Batches b = size_batches(d, gp, Y, ranges, P, 0, false, false);
    jlp_run_stats st{};
    PerJobBytes bytes(Y.jobs.size());
    Output none;
    none.begin(Compression(), P->compress, P->n_threads, d.writers);
    Quiesce quiesce{d, &none};
    Slot& s = d.slot[0];
    for (size_t jk = 0; jk < Y.jobs.size(); jk++) {
        if (P->abort_cb && P->abort_cb(P->cb_user)) throw Aborted();
        for (uint64_t b0 = ranges[jk].first; b0 < ranges[jk].second; b0 += b.B) {
            const uint32_t np = (uint32_t)std::min<uint64_t>(b.B, ranges[jk].second - b0);
            gp.job_lo = Y.jobs[jk].lo; gp.job_hi = Y.jobs[jk].hi; gp.batch_lo = b0; gp.batch_pairs = np;
            gp.plan = s.plan.p; gp.rec_len = s.rec_len.p; gp.rec_local = s.rec_local.p; gp.block_base = s.block_base.p;
            gp.n_scan_blocks = (np + kScanBlock - 1) / kScanBlock;
            CK(launch_place(gp, d.s_compute));
            CK(launch_scan(s.rec_len.p, np * n_ends, n_ends, s.rec_local.p, s.block_tot.p, s.block_base.p, s.totals.p, d.s_compute));
            CK(cudaMemcpyAsync(s.h_totals.p, s.totals.p, 4 * sizeof(uint64_t), cudaMemcpyDeviceToHost, d.s_compute));
            CK(cudaStreamSynchronize(d.s_compute));
            for (int e = 0; e < n_ends; e++) bytes[jk][e] += s.h_totals.p[e];
            st.kernel_launches += 3; st.pairs += np; st.batches++;
        }
    }
    finish(d, st, h2d_before, stats);
    quiesce.armed = false;
    return bytes;
}

// ------------------------------------------------- one call, several GPUs ---
//
// The reference splits a run over its threads and keeps ONE ordered set of files inside one call
// (write_reads_one_filetype_, src/hts.h:334-353 split, :401-416 both pools written together;
// write_reads_cpp_sep_files_, :512-552).  A multi-GPU context does the same over devices: the run's pair-index
// space [0, n_pairs) is cut into near-equal contiguous pieces, one per device (a piece may cover several
// haplotypes' jobs with sep_files, and a job may have several writers); every device runs the three-stage batch
// pipeline of run() on its piece from its own host thread.  No data moves between the devices (no collective):
//   plain FASTQ   a size pass (count_bytes) tells every device how many bytes it will write per job and file, so the
//                 devices write into disjoint ranges of the same, pre-sized R1 / R2 files (or of the caller's memory
//                 buffers) -- R1 and R2 stay aligned;
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

// Where each device's bytes start in each job's output, the devices in order, every job from 0 (files) or behind the one
// before (concat: memory), from the bytes every device produces per job.  Returns where each job's bytes end.
PerJobBytes offsets(const std::vector<PerJobBytes>& sizes, bool concat, std::vector<PerJobBytes>& base) {
    const size_t nj = sizes[0].size();
    base.assign(sizes.size(), PerJobBytes(nj));
    PerJobBytes end(nj);
    for (size_t k = 0; k < nj; k++)
        for (int e = 0; e < 2; e++) {
            uint64_t o = concat && k ? end[k - 1][e] : 0;
            for (size_t r = 0; r < sizes.size(); r++) { base[r][k][e] = o; o += sizes[r][k][e]; }
            end[k][e] = o;
        }
    return end;
}

// Every job's shared files created with their final size at once (no pages yet; pages are reserved slice by slice by the
// devices' writer threads, see Output::deliver), bgzf_close's empty end-of-file block written now (gz); a file system
// that cannot hold everything the run will write is reported here rather than half-way through.
void create_sized(const Layout& Y, const jlp_illumina_params* P, const PerJobBytes& bytes, bool gz) {
    const uint64_t tail = gz ? sizeof kBgzfEof : 0;
    uint64_t need_bytes = 0;
    for (size_t k = 0; k < Y.jobs.size(); k++)
        for (int e = 0; e < ends_of(P); e++) {
            const std::string name = file_name(Y.jobs[k], e, gz, P);
            const uint64_t size = bytes[k][e] + tail;
            const int fd = ::open(name.c_str(), O_RDWR | O_CREAT | O_TRUNC, 0644);
            if (fd < 0) throw IoErr("Unable to open file " + name + ".\n");      // src/io.h:288-290
            need_bytes += size;
            struct statvfs vfs;
            const int rc = ::fstatvfs(fd, &vfs) == 0 && (uint64_t)vfs.f_bavail * vfs.f_frsize < need_bytes ? ENOSPC
                           : ::ftruncate(fd, (off_t)size) == 0 ? 0 : errno;
            const std::string w = rc ? std::strerror(rc) : pwrite_all(fd, kBgzfEof, tail, size - tail);
            ::close(fd);
            if (!w.empty()) throw IoErr("Error writing to file " + name + ": " + w);
        }
}

// zlib output: the parts move behind the first device's bytes in device order (their offsets are known now), slices of
// them copied by several threads at once; one end-of-file block per file (eof)
void join_parts(jlp_ctx* c, const Layout& Y, const jlp_illumina_params* P, bool eof, const std::vector<Ranges>& ranges,
                const std::vector<size_t>& first_dev) {
    const size_t N = ranges.size();
    struct CopyTask { int in_fd, out_fd; uint64_t in_off, out_off, len; };
    std::vector<CopyTask> tasks;
    std::vector<int> fds;
    struct CloseAll { std::vector<int>& f; ~CloseAll() { for (int x : f) ::close(x); } } close_all{fds};
    for (size_t k = 0; k < Y.jobs.size(); k++)
        for (int e = 0; e < ends_of(P); e++) {
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
            const std::string w = pwrite_all(fd, kBgzfEof, eof ? sizeof kBgzfEof : 0, pos);
            if (!w.empty()) throw IoErr("Error writing to file " + name + ": " + w);
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

void run_multi(jlp_ctx* c, bool use_haps, const jlp_illumina_params* P, Output& sink, jlp_run_stats* stats) {
    if (sink.kind == SINK_STREAM)
        throw Unsupported("jlp_illumina_stream on a multi-GPU context: batches of several devices have no single order; "
                          "use files / memory, or one context per device with shard_index / shard_count");
    if (P->shard_count > 1) throw ArgErr("shard_index / shard_count do not combine with a multi-GPU context");
    const size_t N = c->dev.size();
    const Layout Y = make_layout(c, illumina_spec(c, use_haps, P));
    const size_t nj = Y.jobs.size();
    const Compression Z = compression_of(P, sink.kind);
    if (Z.want_gz && Z.dev_z && sink.kind == SINK_MEMORY)
        throw Unsupported("compressed output into memory on a multi-GPU context");
    const bool sized = sink.kind == SINK_MEMORY || (sink.kind == SINK_FILES && !Z.want_gz);   // plain bytes at known offsets
    const bool zsized = sink.kind == SINK_FILES && Z.want_gz && Z.dev_z;   // device coder: sized by a dry run
    const bool parts = sink.kind == SINK_FILES && Z.want_gz && !Z.dev_z;   // zlib on the host: part files, joined afterwards

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

    std::vector<jlp_run_stats> st(N), pre(N);   // the run's, the size pass's (of which only the launches are reported)
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

    // --- plain size pass
    std::vector<PerJobBytes> base;
    if (sized) {
        std::vector<PerJobBytes> sizes(N);
        on_devices([&](Device& d, size_t r) { sizes[r] = count_bytes(c, d, use_haps, &Pk, Y, ranges[r], &pre[r]); }, false);
        const PerJobBytes end = offsets(sizes, sink.kind == SINK_MEMORY, base);    // memory: the jobs' outputs are concatenated
        if (sink.kind == SINK_FILES) create_sized(Y, P, end, false);
        if (sink.kind == SINK_MEMORY) { sink.len[0] = end.back()[0]; sink.len[1] = end.back()[1]; }
    }

    // --- device-BGZF dry run
    std::vector<PerJobBytes> zsizes(N), zcheck(N);
    if (zsized) {
        jlp_illumina_params Pdry = Pk;
        Pdry.progress_cb = nullptr;
        on_devices([&](Device& d, size_t r) {
            Output none;
            zsizes[r] = run(c, d, use_haps, &Pdry, Z, Y, none, &pre[r], Piece{&ranges[r]});
        }, true);
        create_sized(Y, P, offsets(zsizes, false, base), true);
    }

    // --- the run proper
    struct Cleanup {       // part files never outlive the call
        std::vector<std::string> names;
        ~Cleanup() { for (const std::string& n : names) ::unlink(n.c_str()); }
    } cleanup;
    // zlib: for every job the first device with a part in it writes <name> itself (no EOF block yet), device r <name>.part<r>
    std::vector<size_t> first_dev(nj, N);
    for (size_t k = 0; k < nj; k++)
        for (size_t r = N; r-- > 0;) if (ranges[r][k].second > ranges[r][k].first) first_dev[k] = r;
    if (parts)
        for (size_t r = 0; r < N; r++)
            for (size_t k = 0; k < nj; k++)
                if (ranges[r][k].second > ranges[r][k].first && r != first_dev[k])
                    for (int e = 0; e < ends_of(P); e++) cleanup.names.push_back(file_name(Y.jobs[k], e, true, P) + ".part" + std::to_string(r));
    on_devices([&](Device& d, size_t r) {
        Output sk(sink.kind);
        for (int e = 0; e < 2; e++) { sk.mem[e] = sink.mem[e]; sk.cap[e] = sink.cap[e]; }
        std::vector<std::string> suffix;
        for (size_t k = 0; k < nj && parts; k++) suffix.push_back(r == first_dev[k] ? std::string() : ".part" + std::to_string(r));
        const Piece piece{&ranges[r], sized || zsized ? &base[r] : nullptr, sink.kind == SINK_FILES && (sized || zsized),
                          parts ? &suffix : nullptr};
        zcheck[r] = run(c, d, use_haps, &Pk, Z, Y, sk, &st[r], piece);
    }, true);

    if (zsized)         // the coder is deterministic; a difference between the two passes would have put members in the wrong place
        for (size_t r = 0; r < N; r++)
            if (zcheck[r] != zsizes[r]) throw std::runtime_error("internal: compressed sizes differ between the size pass and the run");
    if (parts) join_parts(c, Y, P, Z.zmethod == DEFLATE_BGZF, ranges, first_dev);

    // --- the devices' statistics summed, their device times the slowest device's (they work side by side)
    jlp_run_stats tot{};
    for (size_t r = 0; r < N; r++) {
        const jlp_run_stats& s = st[r];
        tot.pairs += s.pairs; tot.batches += s.batches; tot.kernel_launches += pre[r].kernel_launches + s.kernel_launches;
        for (int e = 0; e < 2; e++) { tot.bytes_out[e] += s.bytes_out[e]; tot.z_bytes[e] += s.z_bytes[e]; }
        tot.d2h_bytes += s.d2h_bytes; tot.h2d_bytes += s.h2d_bytes;
        tot.device_ms = std::max(tot.device_ms, s.device_ms); tot.place_ms = std::max(tot.place_ms, s.place_ms);
        tot.reads_ms = std::max(tot.reads_ms, s.reads_ms); tot.bgzf_ms = std::max(tot.bgzf_ms, s.bgzf_ms);
        tot.run_ms = std::max(tot.run_ms, s.run_ms);
    }
    if (stats) *stats = tot;
}

}  // namespace

extern "C" {

static void run_any(jlp_ctx* c, bool use_haps, const jlp_illumina_params* p, Output& s, jlp_run_stats* stats) {
    check_params(c, use_haps, p, s.kind);
    if (c->dev.size() == 1) run(c, *c->dev[0], use_haps, p, compression_of(p, s.kind), make_layout(c, illumina_spec(c, use_haps, p)), s, stats);
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

}  // extern "C"
