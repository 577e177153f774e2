// Drives the KV page allocator (fastllm_b200/csrc/kv_pool.hpp, no CUDA) for test_kv_pool_cpu.py.  One command per stdin line:
//   init B P N | reserve slot tokens [slot tokens ...] | release slot | release_all | fork src dst len
// After each command it flushes the table updates and prints one JSON line: the command's result and the allocator's whole state.
#include <cstdio>
#include <iostream>
#include <sstream>
#include <string>

#include "../fastllm_b200/csrc/kv_pool.hpp"

int main() {
    fl::KvPool pool;
    std::string line;
    while (std::getline(std::cin, line)) {
        std::istringstream in(line);
        std::string cmd;
        if (!(in >> cmd)) continue;
        bool ok = true;
        std::pair<int, int> copy{-1, -1};
        if (cmd == "init") {
            int b, p, n;
            in >> b >> p >> n;
            pool.init(b, p, n);
        } else if (cmd == "reserve") {
            std::vector<std::pair<int, int64_t>> req;
            int s;
            long long t;
            while (in >> s >> t) req.push_back({s, (int64_t)t});
            ok = pool.reserve(req);
        } else if (cmd == "release") {
            int s;
            in >> s;
            pool.release(s);
        } else if (cmd == "release_all") {
            pool.release_all();
        } else if (cmd == "fork") {
            int src, dst;
            long long len;
            in >> src >> dst >> len;
            ok = pool.fork(src, dst, len, &copy);
        } else {
            std::fprintf(stderr, "unknown command %s\n", cmd.c_str());
            return 2;
        }
        const auto upd = pool.flush();
        std::printf("{\"ok\": %d, \"copy\": [%d, %d], \"free\": %d, \"total\": %d, \"ref\": [", (int)ok, copy.first, copy.second,
                    pool.free_pages(), pool.total_pages());
        for (int i = 0; i < pool.total_pages(); ++i) std::printf("%s%d", i ? ", " : "", pool.refcount(i));
        std::printf("], \"pages\": [");
        for (int s = 0; s < pool.max_batch(); ++s) {
            std::printf("%s[", s ? ", " : "");
            const auto& v = pool.slot_pages(s);
            for (size_t i = 0; i < v.size(); ++i) std::printf("%s%d", i ? ", " : "", v[i]);
            std::printf("]");
        }
        std::printf("], \"table\": [");
        for (size_t i = 0; i < pool.table().size(); ++i) std::printf("%s%d", i ? ", " : "", pool.table()[i]);
        std::printf("], \"flush\": [");
        for (size_t i = 0; i < upd.size(); ++i) std::printf("%s[%d, %d]", i ? ", " : "", upd[i].first, upd[i].second);
        std::printf("]}\n");
    }
    return 0;
}
