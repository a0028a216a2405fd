// Runs jlp::parallel_for (jackalope_b200/csrc/jlp_host.h) without a GPU; tests/test_parallel_host.py compiles it with
// g++ and checks the one line it prints.
//   parallel_driver count <n> <n_threads>   "runs=<items that ran exactly once> threads=<distinct threads used>"
//   parallel_driver throws <n> <n_threads>  items 3 and 7 throw different types, item 3 after item 7:
//                                           "caught=<type> what=<message> ran=<items run>"
//   parallel_driver serial <n>              n_threads = 1: "caller_only=<1 if every item ran on the calling thread>"
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <set>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "jlp_host.h"

using jlp::parallel_for;

int main(int argc, char** argv) {
    if (argc < 3) return 2;
    const std::string c = argv[1];
    const uint64_t n = std::strtoull(argv[2], nullptr, 10);
    const unsigned nt = argc > 3 ? (unsigned)std::strtoul(argv[3], nullptr, 10) : 1;
    std::vector<std::atomic<int>> hits(n);
    std::mutex mu;
    std::set<std::thread::id> ids;
    auto count = [&](uint64_t i) {
        hits[i].fetch_add(1);
        std::lock_guard<std::mutex> g(mu);
        ids.insert(std::this_thread::get_id());
    };
    uint64_t once = 0;
    if (c == "count") {
        parallel_for(n, nt, [&](uint64_t i) {
            count(i);
            std::this_thread::sleep_for(std::chrono::microseconds(200));      // so that every thread gets items
        });
        for (auto& h : hits) once += h.load() == 1;
        std::printf("runs=%llu threads=%zu\n", (unsigned long long)once, ids.size());
    } else if (c == "throws") {
        try {
            parallel_for(n, nt, [&](uint64_t i) {
                count(i);
                if (i == 3) {
                    std::this_thread::sleep_for(std::chrono::milliseconds(100));
                    throw std::invalid_argument("three");
                }
                if (i == 7) throw std::out_of_range("seven");
            });
            std::printf("caught=none\n");
        } catch (const std::invalid_argument& e) {
            for (auto& h : hits) once += h.load() == 1;
            std::printf("caught=invalid_argument what=%s ran=%llu\n", e.what(), (unsigned long long)once);
        } catch (const std::exception& e) {
            std::printf("caught=other what=%s\n", e.what());
        }
    } else if (c == "serial") {
        parallel_for(n, 1, count);
        std::printf("caller_only=%d\n", (int)(ids.size() == 1 && *ids.begin() == std::this_thread::get_id()));
    } else {
        return 2;
    }
    return 0;
}
