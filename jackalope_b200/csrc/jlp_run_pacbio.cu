// The PacBio driver (jlp_pacbio*): per batch the per-read plan on the host, reads and optional BGZF on the first device
// of the context.
#include "jlp_ctx.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>

using namespace jlp;

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
            const float ms_reads = elapsed_ms(ev[0], ev[1]), ms_z = elapsed_ms(ev[1], ev[2]);
            st.reads_ms += ms_reads; st.device_ms += ms_reads;
            if (dev_z) { st.bgzf_ms += ms_z; st.device_ms += ms_z; }
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

}  // namespace

extern "C" {

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

}  // extern "C"
