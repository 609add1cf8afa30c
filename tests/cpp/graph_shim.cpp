// Test shim (CPU tests only): the score graph's host/device scorer (hmk_score_with_shift of hammock_b200/csrc/hmk_common.h)
// and the C++ host's score_graph.tsv writer (hammock_host.hpp), compiled with plain g++ and exported with C linkage so
// that tests/test_score_graph.py can compare them with the oracle and the Python writer.  Never linked into the product.
#include "../../hammock_b200/csrc/hmk_common.h"
#include "../../hammock_b200/host_cpp/hammock_host.hpp"

using namespace hammock;

extern "C" {
int32_t shim_score_with_shift(const uint8_t* s1, int l1, const uint8_t* s2, int l2, const int32_t* M, int X, int P, int* shift) {
    return hmk_score_with_shift(s1, l1, s2, l2, M, X, P, shift);
}
// sequences: n strings joined by '\n'; edges: n_edges x (seq, partner, score, shift)
int shim_save_score_graph(const char* sequences, const int32_t* edges, int64_t n_edges, const char* path) {
    std::vector<UniqueSequence> seqs;
    std::string_view all(sequences);
    for (size_t i = 0; i <= all.size();) {
        size_t j = all.find('\n', i);
        if (j == std::string_view::npos) j = all.size();
        seqs.emplace_back(std::string(all.substr(i, j - i)), std::vector<std::pair<std::string, int32_t>>{{"x", 1}});
        i = j + 1;
    }
    std::vector<hmk_graph_edge> e((size_t)n_edges);
    for (int64_t k = 0; k < n_edges; k++) e[k] = hmk_graph_edge{edges[4 * k], edges[4 * k + 1], edges[4 * k + 2], edges[4 * k + 3]};
    TsvWriter w(path);
    writeScoreGraphHeader(w);
    writeScoreGraphEdges(w, seqs, e.data(), e.size());
    return 0;
}
}
