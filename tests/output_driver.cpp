// Feeds seeded batches through jlp::Output (jackalope_b200/csrc/jlp_output.cpp) the way the Illumina and PacBio drivers
// do, without a GPU; tests/test_output_host.py compiles it with g++ and checks what it wrote.
//   output_driver <case> <dir>
// writes <dir>/out_R<e>.fq (what Output produced) and <dir>/expect_R<e>.fq (what it must be), and prints one line of
// facts the test checks (sizes, lengths).
#include <fcntl.h>
#include <unistd.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "jlp_deflate.h"
#include "jlp_output.h"

using namespace jlp;

namespace {

// sizes that cross the plain (8 MiB), BGZF (64 x 0xff00) and gzip (4 MiB) slices, an empty batch and a one-byte one
const std::vector<uint64_t> kSizes = {9437201, 300000, 0, 8355845, 1, 4194304};

std::vector<uint8_t> batch(size_t k, int e) {
    std::vector<uint8_t> v(kSizes[k] >> e);          // end 1 gets batches of half the size
    uint64_t x = 0x9E3779B97F4A7C15ull * (2 * k + e + 1);
    for (size_t i = 0; i < v.size(); i++) {
        x = x * 6364136223846793005ull + 1442695040888963407ull;
        v[i] = i % 61 == 60 ? '\n' : "ACGT"[(x >> 62) & 3];
    }
    return v;
}

void save(const std::string& name, const std::vector<uint8_t>& v) {
    FILE* f = std::fopen(name.c_str(), "wb");
    if (!f || std::fwrite(v.data(), 1, v.size(), f) != v.size()) { std::perror(name.c_str()); std::exit(2); }
    std::fclose(f);
}

struct Log { std::string dir; std::vector<std::string> calls; std::vector<uint8_t> data[2][2]; };
int on_chunk(void* user, uint64_t job, int end, const char* p, uint64_t n) {
    Log* L = static_cast<Log*>(user);
    L->calls.push_back(std::to_string(job) + ":" + std::to_string(end) + ":" + std::to_string(n));
    L->data[job][end].insert(L->data[job][end].end(), p, p + n);
    return 0;
}

}  // namespace

int main(int argc, char** argv) {
    if (argc != 3) return 2;
    const std::string c = argv[1], dir = argv[2];
    const std::string out[2] = {dir + "/out_R1.fq", dir + "/out_R2.fq"};
    std::vector<std::vector<uint8_t>> b[2];
    std::vector<uint8_t> plain[2];
    for (size_t k = 0; k < kSizes.size(); k++)
        for (int e = 0; e < 2; e++) {
            b[e].push_back(batch(k, e));
            plain[e].insert(plain[e].end(), b[e][k].begin(), b[e][k].end());
        }
    WriterPool pool;
    HostBatch hb[3];
    bool mapped = false;      // some batch went into a mapping of the file (else: pwrite)
    auto put = [&](Output& o, HostBatch& h, size_t k, int n_ends, uint64_t job) {
        const uint8_t* data[2] = {b[0][k].data(), b[1][k].data()};
        const uint64_t n[2] = {b[0][k].size(), b[1][k].size()};
        o.deliver(h, data, n, job, n_ends);
        mapped |= h.map[0].base != nullptr;
    };
    // batch k is delivered from hb[k % 3] once the batch that used it before is settled, as run() does
    auto feed = [&](Output& o, size_t n_batches, int n_ends, uint64_t job) {
        for (size_t k = 0; k < n_batches; k++) {
            o.settle(hb[k % 3]);
            put(o, hb[k % 3], k, n_ends, job);
        }
    };
    auto settle_all = [&](Output& o) { for (HostBatch& h : hb) o.settle(h); };

    if (c == "plain1" || c == "plain4" || c == "bgzf" || c == "gzip") {
        Compression z;
        if (c == "bgzf" || c == "gzip") { z.want_gz = true; z.zmethod = c == "bgzf" ? DEFLATE_BGZF : DEFLATE_GZIP; }
        Output o(SINK_FILES);
        o.begin(z, 6, c == "plain1" || c == "gzip" ? 1 : 4, pool);
        o.open_job(out, 2, nullptr, false);
        feed(o, kSizes.size(), 2, 0);
        settle_all(o);
        o.end_job(0, 2, true);
        for (int e = 0; e < 2; e++) {
            std::vector<uint8_t> want;            // zlib: what PacBio wrote before, deflate_members over each whole batch
            if (z.zmethod < 0) want = plain[e];
            else
                for (const std::vector<uint8_t>& v : b[e])
                    if (!deflate_members(z.zmethod, 6, v.data(), v.size(), want).empty()) return 3;
            if (z.zmethod == DEFLATE_BGZF) want.insert(want.end(), kBgzfEof, kBgzfEof + sizeof kBgzfEof);
            save(dir + "/expect_R" + std::to_string(e + 1) + ".fq", want);
            save(dir + "/plain_R" + std::to_string(e + 1) + ".fq", plain[e]);
        }
        std::printf("mapped=%d\n", (int)mapped);
    } else if (c == "memory") {
        const uint64_t cap = kSizes[0] + kSizes[1] + 100;          // the first two batches fit, the third (empty) too
        std::vector<char> mem(cap + 4096, 'x');
        Output o(SINK_MEMORY);
        o.mem[0] = mem.data(); o.cap[0] = cap;
        Compression z;
        z.dev_z = true;                                            // the device coder's output ends with the EOF block
        o.begin(z, 6, 4, pool);
        o.open_job(out, 1, nullptr, false);
        feed(o, kSizes.size(), 1, 0);
        settle_all(o);
        o.end_job(0, 1, true);
        save(dir + "/out_R1.fq", std::vector<uint8_t>(mem.begin(), mem.end()));
        std::vector<uint8_t> want = plain[0];
        want.insert(want.end(), kBgzfEof, kBgzfEof + sizeof kBgzfEof);
        save(dir + "/expect_R1.fq", want);
        std::printf("%llu %llu\n", (unsigned long long)o.len[0], (unsigned long long)cap);
    } else if (c == "stream") {
        Log L;
        Output o(SINK_STREAM);
        o.chunk_cb = on_chunk; o.chunk_user = &L;
        Compression z;
        z.dev_z = true;
        o.begin(z, 6, 4, pool);
        for (uint64_t job = 0; job < 2; job++) {
            o.open_job(out, 2, nullptr, false);
            feed(o, job ? 2 : kSizes.size(), 2, job);
            settle_all(o);
            o.end_job(job, 2, true);
        }
        for (int j = 0; j < 2; j++)
            for (int e = 0; e < 2; e++) save(dir + "/stream_" + std::to_string(j) + "_" + std::to_string(e), L.data[j][e]);
        for (int e = 0; e < 2; e++) save(dir + "/plain_R" + std::to_string(e + 1) + ".fq", plain[e]);
        for (const std::string& s : L.calls) std::printf("%s ", s.c_str());
        std::printf("\n");
    } else if (c == "shared") {
        // a file created and sized by the caller (a multi-GPU run): this call's bytes go to [base, base + n)
        const uint64_t base = 12345, tail = 777;
        std::vector<uint8_t> want(base, 'x');
        want.insert(want.end(), plain[0].begin(), plain[0].end());
        want.insert(want.end(), tail, 'x');
        save(out[0], std::vector<uint8_t>(want.size(), 'x'));
        save(dir + "/expect_R1.fq", want);
        Output o(SINK_FILES);
        Compression z;
        z.dev_z = true;
        o.begin(z, 6, 4, pool);
        const uint64_t at[2] = {base, 0};
        o.open_job(out, 1, at, true);
        feed(o, kSizes.size(), 1, 0);
        settle_all(o);
        o.end_job(0, 1, false);
        std::printf("ok\n");
    } else if (c == "abandon1" || c == "abandon4") {
        // batches 0 and 1 settled, batch 3 (8 MB) delivered, then an error: the file is cut back to batches 0 and 1
        Output o(SINK_FILES);
        o.begin(Compression(), 6, c == "abandon1" ? 1 : 4, pool);
        o.open_job(out, 1, nullptr, false);
        feed(o, 2, 1, 0);
        o.settle(hb[0]); o.settle(hb[1]);
        put(o, hb[2], 3, 1, 0);
        HostBatch* all[3] = {&hb[0], &hb[1], &hb[2]};
        o.abandon(all, 3);
        o.close_files();
        std::vector<uint8_t> want(b[0][0]);
        want.insert(want.end(), b[0][1].begin(), b[0][1].end());
        save(dir + "/expect_R1.fq", want);
        std::printf("mapped=%d\n", (int)mapped);
    } else {
        return 2;
    }
    return 0;
}
