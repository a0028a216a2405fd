// The VCF writer (jlp_write_vcf, DESIGN.md section 11), on the first device of the context.
#include "jlp_ctx.h"

#include <sys/stat.h>

#include <cctype>
#include <cstring>

using namespace jlp;

namespace {

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
        st.text_ms += elapsed_ms(ev[0], ev[1]);
        if (dev_z) st.bgzf_ms += elapsed_ms(ev[1], ev[2]);
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
        st.span_ms += elapsed_ms(ev[3], ev[4]);
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

extern "C" {

int jlp_write_vcf(jlp_ctx* c, const jlp_vcf_params* p, jlp_vcf_stats* stats) {
    if (!c) return JLP_ERR_ARG;
    return guarded(c, [&]() { write_vcf(c, device0(c), p, stats); });
}

}  // extern "C"
