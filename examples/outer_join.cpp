// The reference's test_join data (tests/test_pair_rdd.rs:39-82) through a left outer join:
// col1.left_outer_join(col2, 4), String payloads replaced by indices into the tables below.
// Expected 7 rows: keys 1,1,2,2,3,3 matched, and key 4 once with no right value:
// (4, ((G,H), None)).
#include <algorithm>
#include <cstdio>

#include "vega_b200.hpp"

int main()
{
    try {
        auto sc = vega::Context::create();
        const char *t1[] = {"(A,B)", "(C,D)", "(E,F)", "(G,H)"};
        const char *t2[] = {"A1", "A2", "B1", "B2", "C1", "C2"};
        std::vector<std::pair<int32_t, uint64_t>> col1 = {{1, 0}, {2, 1}, {3, 2}, {4, 3}};
        std::vector<std::pair<int32_t, uint64_t>> col2 = {{1, 0}, {1, 1}, {2, 2}, {2, 3}, {3, 4}, {3, 5}};
        auto r1 = sc->parallelize(col1, 4);
        auto r2 = sc->parallelize(col2, 4);
        auto res = r1.left_outer_join(r2, 4);
        std::sort(res.begin(), res.end());
        size_t unmatched = 0;
        std::printf("result: [");
        for (size_t i = 0; i < res.size(); ++i) {
            const auto &v = res[i].second.first;
            const auto &w = res[i].second.second;
            std::printf("%s(%d, (%s, %s))", i ? ", " : "", res[i].first, v ? t1[*v] : "None", w ? t2[*w] : "None");
            unmatched += !w;
        }
        std::printf("]\n");
        return res.size() == 7 && unmatched == 1 ? 0 : 1;
    } catch (const vega::Error &e) {
        std::fprintf(stderr, "%s\n", e.what());
        return 2;
    }
}
