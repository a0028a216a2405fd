// Shared pieces of the Rcpp glue (integration/hts_illumina_b200.cpp, integration/hts_pacbio_b200.cpp): the context
// holder, and the flattening of jackalope's RefGenome / HapSet into the plain arrays of include/jlp_b200.h.
// Only jackalope's own types are read, through const access, as the original code does (XPtr<RefGenome> /
// XPtr<HapSet> are borrowed, never freed: src/hts_illumina.h:307,513).
#ifndef JLP_B200_GLUE_H
#define JLP_B200_GLUE_H

#include <RcppArmadillo.h>

#include <string>
#include <vector>

#include "jackalope_types.h"  // uint64, uint8
#include "ref_classes.h"      // RefGenome, RefChrom   (src/ref_classes.h:36-140)
#include "hap_classes.h"      // HapSet, HapGenome, HapChrom, AllMutations (src/hap_classes.h:100-104,287-296,537-)
#include "jlp_b200.h"

namespace jlp_glue {

using namespace Rcpp;

struct Ctx {                       // destroys the context on every exit path, Rcpp::stop included
    jlp_ctx* p = nullptr;
    std::string bases;             // the flattened genome: the library reads it during the run (deferred upload)
    // every GPU the process can see (CUDA_VISIBLE_DEVICES selects them): one call, one ordered set of files,
    // as the reference's n_threads share one set (src/hts.h:334-353); no CPU fallback
    Ctx() {
        if (jlp_ctx_create_multi(0, nullptr, &p) != JLP_OK) stop(jlp_last_error(nullptr));
    }
    ~Ctx() { jlp_ctx_destroy(p); }
    void check(int rc) { if (rc != JLP_OK) stop(std::string(jlp_last_error(p))); }
};

// RefGenome -> one contiguous byte array + offsets.  The upload is deferred: the run copies, chromosome by
// chromosome underneath the first batches, what each device's piece of the run reads (haplotype runs: everything).
inline void set_genome(Ctx& ctx, const RefGenome& ref) {
    ctx.bases.clear();
    ctx.bases.reserve(ref.total_size);
    std::vector<uint64_t> off(1, 0);
    std::vector<const char*> names;
    for (uint64 i = 0; i < ref.size(); i++) {
        ctx.bases += ref[i].nucleos;
        off.push_back(ctx.bases.size());
        names.push_back(ref[i].name.c_str());
    }
    ctx.check(jlp_set_genome_async(ctx.p, ctx.bases.data(), off.data(), names.size(), names.data(), ref.name.c_str()));
}

// one haplotype: AllMutations of every chromosome as flat arrays
inline void add_haplotype(Ctx& ctx, const HapGenome& hap) {
    const uint64 nc = hap.size();
    std::vector<std::vector<uint64_t>> old_pos(nc), new_pos(nc), nuc_off(nc);
    std::vector<std::string> pools(nc);
    std::vector<uint64_t> n_muts(nc), pool_len(nc), sizes(nc);
    std::vector<const uint64_t*> p_old(nc), p_new(nc), p_off(nc);
    std::vector<const char*> p_pool(nc);
    for (uint64 c = 0; c < nc; c++) {
        const AllMutations& m = hap[c].mutations;
        n_muts[c] = m.size();
        sizes[c] = hap[c].size();
        old_pos[c].assign(m.old_pos.begin(), m.old_pos.end());
        new_pos[c].assign(m.new_pos.begin(), m.new_pos.end());
        for (uint64 i = 0; i < m.size(); i++) {
            nuc_off[c].push_back(pools[c].size());
            if (m.nucleos[i] != nullptr) pools[c] += m.nucleos[i];     // nullptr = deletion
        }
        pool_len[c] = pools[c].size();
        p_old[c] = old_pos[c].data(); p_new[c] = new_pos[c].data(); p_off[c] = nuc_off[c].data();
        p_pool[c] = pools[c].data();
    }
    uint64_t idx = 0;
    ctx.check(jlp_add_haplotype(ctx.p, hap.name.c_str(), n_muts.data(), p_old.data(), p_new.data(), p_off.data(),
                                p_pool.data(), pool_len.data(), sizes.data(), &idx));
}

inline uint64_t seed_from_r() {           // as mt_seeds does: 32-bit values from R's RNG, so set.seed() governs the run (src/pcg.h:37-46)
    std::vector<uint64> s = as<std::vector<uint64>>(Rcpp::runif(2, 0, 4294967296.0));
    return (static_cast<uint64_t>(s[0]) << 32) | static_cast<uint64_t>(s[1]);
}

}  // namespace jlp_glue
#endif
