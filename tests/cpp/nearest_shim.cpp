// Test shim (CPU tests only): the C++ host's nearest_partners.tsv writer (hammock_host.hpp), compiled with plain g++ and
// exported with C linkage so that tests/test_nearest.py can compare it with the Python writer.  Never linked into the
// product.
#include "../../hammock_b200/host_cpp/hammock_host.hpp"

using namespace hammock;

extern "C" {
// sequences: n strings joined by '\n'; partner / score / shift: n x k, count: n.  Rows are written in two calls
// (rows [0, split) and [split, n)), as the driver writes row ranges.
int shim_save_nearest(const char* sequences, int32_t k, const int32_t* partner, const int32_t* score, const int32_t* shift,
                      const int32_t* count, int32_t split, const char* path) {
    std::vector<UniqueSequence> seqs;
    std::string_view all(sequences);
    for (size_t i = 0; i <= all.size();) {
        size_t j = all.find('\n', i);
        if (j == std::string_view::npos) j = all.size();
        seqs.emplace_back(std::string(all.substr(i, j - i)), std::vector<std::pair<std::string, int32_t>>{{"x", 1}});
        i = j + 1;
    }
    const int32_t n = (int32_t)seqs.size();
    TsvWriter w(path);
    writeNearestHeader(w);
    writeNearestRows(w, seqs, 0, split, k, partner, score, shift, count);
    const size_t e = (size_t)split * k;
    writeNearestRows(w, seqs, split, n - split, k, partner + e, score + e, shift + e, count + split);
    return 0;
}
}
