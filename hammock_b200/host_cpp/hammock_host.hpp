// hammock_host.hpp -- C++ host side above the C ABI (include/hammock_b200.h).
//
// The reference is compiled code (Java) whose toolchain is absent from this image, so the host
// layer that a Hammock maintainer would keep in Java is mirrored here in C++ for the greedy path:
// same names, argument meaning and error behaviour as the reference classes (file:line cited,
// relative to /root/reference/src/cz/krejciadam/hammock/).  Parsing, ordering, automatic
// parameters and the result files live here; all scoring and clustering happens on the GPU
// behind hmk_greedy_cluster().  There is no CPU fallback.
#pragma once
#include <algorithm>
#include <cctype>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <map>
#include <sstream>
#include <stdexcept>
#include <string>
#include <string_view>
#include <unordered_map>
#include <vector>

#include "../../include/hammock_b200.h"

namespace hammock {

struct HammockException : std::runtime_error { using std::runtime_error::runtime_error; };      // HammockException.java
struct DataException : HammockException { using HammockException::HammockException; };          // DataException.java
struct FileFormatException : HammockException { using HammockException::HammockException; };    // FileFormatException.java
struct CLIException : HammockException { using HammockException::HammockException; };           // CLIException.java
struct NullPointerException : HammockException {   // LimitedGreedySequenceClusterer.java:104,108 (SURVEY.md 3.2)
    int step;
    explicit NullPointerException(int s)
        : HammockException("NullPointerException in greedy phase 1, step " + std::to_string(s)), step(s) {}
};
struct CudaException : HammockException { using HammockException::HammockException; };
struct UnsupportedInput : HammockException { using HammockException::HammockException; };   // HMK_STATUS_UNSUPPORTED (clinkage entry)

static const char* const ALPHABET = "ARNDCQEGHILKMFPSTWYVBZX*";   // UniqueSequence.java:23-26

inline int32_t wrap_add(int32_t a, int32_t b) { return (int32_t)((uint32_t)a + (uint32_t)b); }   // Java int

// ---------------------------------------------------------------- Java collection semantics
inline int32_t java_string_hash(const std::string& s) {   // String.hashCode
    uint32_t h = 0;
    for (unsigned char c : s) h = 31u * h + c;
    return (int32_t)h;
}

// Iteration order of a java.util.HashMap<String, ?> (Java 8+: tail insertion, order-preserving
// resize) filled with `keys` in this order.  Bins are assumed not to treeify (< 8 collisions).
inline std::vector<std::string> java_hashmap_order(const std::vector<std::string>& keys) {
    size_t cap = 16;
    while (keys.size() > cap * 3 / 4) cap *= 2;
    std::vector<std::vector<std::string>> bins(cap);
    for (const auto& k : keys) {
        uint32_t h = (uint32_t)java_string_hash(k);
        h ^= h >> 16;
        bins[h & (cap - 1)].push_back(k);
    }
    std::vector<std::string> out;
    for (auto& b : bins) out.insert(out.end(), b.begin(), b.end());
    return out;
}

struct JavaRandom {   // java.util.Random
    uint64_t seed;
    explicit JavaRandom(int64_t s) : seed(((uint64_t)s ^ 0x5DEECE66DULL) & ((1ULL << 48) - 1)) {}
    int32_t next(int bits) {
        seed = (seed * 0x5DEECE66DULL + 0xBULL) & ((1ULL << 48) - 1);
        return (int32_t)(int64_t)(seed >> (48 - bits));
    }
    int32_t nextInt(int32_t bound) {
        int32_t r = next(31), m = bound - 1;
        if ((bound & m) == 0) return (int32_t)(((int64_t)bound * (int64_t)r) >> 31);
        for (int32_t u = r; (int32_t)((uint32_t)u - (uint32_t)(r = u % bound) + (uint32_t)m) < 0; u = next(31)) {}
        return r;
    }
};

// ---------------------------------------------------------------- data model
// letter -> code 0..23, -1 = not in the alphabet (lower case folds to upper case, UniqueSequence.java:44)
struct ResidueTable {
    int8_t code[256];
    ResidueTable() {
        std::memset(code, -1, sizeof code);
        for (int i = 0; ALPHABET[i]; i++) {
            code[(unsigned char)ALPHABET[i]] = (int8_t)i;
            code[(unsigned char)std::tolower((unsigned char)ALPHABET[i])] = (int8_t)i;
        }
    }
};
inline const ResidueTable& residue_table() { static const ResidueTable t; return t; }

struct UniqueSequence {   // UniqueSequence.java:19-57, 81-109
    std::string sequence;                                  // upper-case letters (getSequenceString)
    std::vector<std::pair<std::string, int32_t>> labels;   // labelsMap (insertion order kept for determinism)

    UniqueSequence(std::string s, std::vector<std::pair<std::string, int32_t>> lab) : sequence(std::move(s)), labels(std::move(lab)) {
        const ResidueTable& t = residue_table();
        for (char& c : sequence) {
            const int8_t k = t.code[(unsigned char)c];
            if (k < 0) throw FileFormatException(std::string("Error, character ") + c +
                                                 " is not a valid letter from the amino acid alphabet code.");   // :51-54
            c = ALPHABET[k];
        }
    }
    size_t length() const { return sequence.size(); }
    uint8_t code(size_t i) const { return (uint8_t)residue_table().code[(unsigned char)sequence[i]]; }   // getSequence()[i]
    int32_t size() const {   // :81-88
        int32_t s = 0;
        for (auto& kv : labels) s = wrap_add(s, kv.second);
        return s;
    }
    int32_t count(const std::string& label) const {
        for (auto& kv : labels) if (kv.first == label) return kv.second;
        return 0;
    }
    bool has(const std::string& label) const {
        for (auto& kv : labels) if (kv.first == label) return true;
        return false;
    }
};

struct Cluster {   // Cluster.java:21-74, 113-123, 156-158
    int32_t id = 0;
    int32_t sizeSum = 0;
    std::vector<int> members;   // indices into the clustering-ordered sequence vector, insertion order
    int32_t getId() const { return id; }
    int32_t size() const { return sizeSum; }
    size_t getUniqueSize() const { return members.size(); }
};

// ---------------------------------------------------------------- loaders
inline bool java_ws(unsigned char c) { return c == ' ' || c == '\t' || c == '\n' || c == 0x0B || c == '\f' || c == '\r'; }

inline std::string read_file(const std::string& path) {
    std::FILE* f = std::fopen(path.c_str(), "rb");
    if (!f) throw HammockException("cannot open " + path);
    std::string text;
    char buf[1 << 16];
    if (std::fseek(f, 0, SEEK_END) == 0) {
        const long n = std::ftell(f);
        if (n > 0) text.reserve((size_t)n);
        std::rewind(f);
    }
    for (size_t got; (got = std::fread(buf, 1, sizeof buf, f)) > 0;) text.append(buf, got);
    std::fclose(f);
    return text;
}

// BufferedReader.readLine over a whole file held in memory: fn(line) per line, terminator (and a '\r' before it) stripped
template <class Fn>
inline void for_each_line(const std::string& text, Fn&& fn) {
    size_t i = 0;
    while (i < text.size()) {
        const void* nl = std::memchr(text.data() + i, '\n', text.size() - i);
        size_t j = nl ? (size_t)((const char*)nl - text.data()) : text.size();
        size_t e = j;
        if (e > i && text[e - 1] == '\r') e--;
        fn(std::string_view(text.data() + i, e - i));
        i = j + 1;
    }
}

inline std::vector<std::string> read_lines(const std::string& path) {
    const std::string text = read_file(path);
    std::vector<std::string> lines;
    for_each_line(text, [&](std::string_view l) { lines.emplace_back(l); });
    return lines;
}

inline int32_t parse_int(const std::string& tok) {   // Integer.parseInt
    size_t i = 0;
    bool neg = false;
    if (!tok.empty() && (tok[0] == '-' || tok[0] == '+')) { neg = tok[0] == '-'; i = 1; }
    if (i >= tok.size()) throw FileFormatException("NumberFormatException: For input string: \"" + tok + "\"");
    int64_t v = 0;
    for (; i < tok.size(); i++) {
        if (tok[i] < '0' || tok[i] > '9') throw FileFormatException("NumberFormatException: For input string: \"" + tok + "\"");
        v = v * 10 + (tok[i] - '0');
        if (v > (int64_t)INT32_MAX + 1) throw FileFormatException("NumberFormatException: For input string: \"" + tok + "\"");
    }
    if (neg) v = -v;
    if (v > INT32_MAX || v < INT32_MIN) throw FileFormatException("NumberFormatException: For input string: \"" + tok + "\"");
    return (int32_t)v;
}

inline int32_t decode_int(const std::string& tok) {   // Integer.decode
    std::string s = tok;
    bool neg = false;
    if (!s.empty() && s[0] == '-') { neg = true; s.erase(0, 1); } else if (!s.empty() && s[0] == '+') s.erase(0, 1);
    int radix = 10;
    if (s.size() >= 2 && s[0] == '0' && (s[1] == 'x' || s[1] == 'X')) { radix = 16; s.erase(0, 2); }
    else if (!s.empty() && s[0] == '#') { radix = 16; s.erase(0, 1); }
    else if (s.size() > 1 && s[0] == '0') { radix = 8; s.erase(0, 1); }
    if (s.empty()) throw FileFormatException("NumberFormatException: For input string: \"" + tok + "\"");
    int64_t v = 0;
    for (char c : s) {
        int d = (c >= '0' && c <= '9') ? c - '0' : (c >= 'a' && c <= 'f') ? c - 'a' + 10 : (c >= 'A' && c <= 'F') ? c - 'A' + 10 : 99;
        if (d >= radix) throw FileFormatException("NumberFormatException: For input string: \"" + tok + "\"");
        v = v * radix + d;
        if (v > (int64_t)INT32_MAX + 1) throw FileFormatException("NumberFormatException: For input string: \"" + tok + "\"");
    }
    if (neg) v = -v;
    if (v > INT32_MAX || v < INT32_MIN) throw FileFormatException("NumberFormatException: For input string: \"" + tok + "\"");
    return (int32_t)v;
}

inline std::string_view java_trim(std::string_view s) {   // String.trim
    size_t i = 0, j = s.size();
    while (i < j && (unsigned char)s[i] <= ' ') i++;
    while (j > i && (unsigned char)s[j - 1] <= ' ') j--;
    return s.substr(i, j - i);
}

inline int32_t decode_int(std::string_view tok) {   // Integer.decode; plain short decimals (no sign, no radix prefix) directly
    if (!tok.empty() && tok.size() <= 9 && tok[0] >= '1' && tok[0] <= '9') {
        int32_t v = 0;
        size_t i = 0;
        for (; i < tok.size() && tok[i] >= '0' && tok[i] <= '9'; i++) v = v * 10 + (tok[i] - '0');
        if (i == tok.size()) return v;
    }
    return decode_int(std::string(tok));
}
inline int32_t decode_int(const char* tok) { return decode_int(std::string(tok)); }

// String.split(sep) for a one-character separator: trailing empty strings are dropped (an all-empty result keeps one)
inline void java_split(std::string_view s, char sep, std::vector<std::string_view>& parts) {
    parts.clear();
    size_t i = 0;
    for (;;) {
        const size_t j = s.find(sep, i);
        parts.push_back(s.substr(i, j == std::string_view::npos ? std::string_view::npos : j - i));
        if (j == std::string_view::npos) break;
        i = j + 1;
    }
    while (parts.size() > 1 && parts.back().empty()) parts.pop_back();
}

// FileIOManager.loadScoringMatrix (FileIOManager.java:46-81), quirks included (rows in file order,
// dead header check, exactly 25 whitespace tokens per data line, > 24 rows is an error)
inline std::vector<int32_t> loadScoringMatrix(const std::string& path) {
    std::vector<int32_t> M(576, 0);
    int row = 0;
    for (const std::string& line : read_lines(path)) {
        if (!line.empty() && (line[0] == '#' || line[0] == ' ' || line[0] == '\t')) continue;
        std::vector<std::string> toks;
        if (line.empty()) toks.push_back("");
        else {
            if (java_ws((unsigned char)line[0])) toks.push_back("");
            size_t i = 0;
            while (i < line.size()) {
                while (i < line.size() && java_ws((unsigned char)line[i])) i++;
                if (i >= line.size()) break;
                size_t j = i;
                while (j < line.size() && !java_ws((unsigned char)line[j])) j++;
                toks.push_back(line.substr(i, j - i));
                i = j;
            }
        }
        if (toks.size() != 25)
            throw FileFormatException("Error in scoring matrix file: " + path +
                                      ". Scoring matrix should always have 24 columns (plus 1 column describing AAs).");
        if (row >= 24)
            throw FileFormatException("Error in scoring matrix file: " + path +
                                      ". Scoring matrix should always have 24 rows (plus 1 column describing AAs).");
        for (int c = 1; c < 25; c++) M[row * 24 + c - 1] = parse_int(toks[c]);
        row++;
    }
    return M;
}

// LinkedHashMap<String, Map<String, Integer>> of the fasta loader: first-occurrence order of the sequences, an open-
// addressing index over the entries (no node per key)
struct SequenceTable {
    struct Entry { std::string sequence; std::vector<std::pair<std::string, int32_t>> labels; };
    std::vector<Entry> entries;
    std::vector<uint32_t> slots;    // entry index + 1, 0 = free
    std::vector<uint64_t> hashes;   // per entry
    explicit SequenceTable(size_t expected) {
        size_t cap = 1024;
        while (cap < 2 * expected) cap *= 2;
        slots.assign(cap, 0);
        entries.reserve(expected);
        hashes.reserve(expected);
    }
    static uint64_t hash(std::string_view s) {
        uint64_t h = 0xcbf29ce484222325ull;
        for (unsigned char c : s) { h ^= c; h *= 0x100000001b3ull; }
        return h ^ (h >> 29);
    }
    void grow() {
        std::vector<uint32_t> bigger(slots.size() * 2, 0);
        for (size_t e = 0; e < entries.size(); e++) {
            size_t i = hashes[e] & (bigger.size() - 1);
            while (bigger[i]) i = (i + 1) & (bigger.size() - 1);
            bigger[i] = (uint32_t)e + 1;
        }
        slots.swap(bigger);
    }
    void add(std::string_view sequence, std::string_view label, int32_t count) {
        const uint64_t h = hash(sequence);
        size_t i = h & (slots.size() - 1);
        for (; slots[i]; i = (i + 1) & (slots.size() - 1)) {
            const uint32_t e = slots[i] - 1;
            if (hashes[e] != h || entries[e].sequence != sequence) continue;
            for (auto& kv : entries[e].labels)
                if (kv.first == label) { kv.second = wrap_add(kv.second, count); return; }
            entries[e].labels.emplace_back(std::string(label), count);
            return;
        }
        slots[i] = (uint32_t)entries.size() + 1;
        entries.push_back(Entry{std::string(sequence), {{std::string(label), count}}});
        hashes.push_back(h);
        if (2 * entries.size() > slots.size()) grow();
    }
};

// FileIOManager.loadUniqueSequencesFromFasta (FileIOManager.java:159-216)
inline std::vector<UniqueSequence> loadUniqueSequencesFromFasta(const std::string& path) {
    const std::string text = read_file(path);
    SequenceTable table(text.size() / 24);
    std::string sequence, label;
    std::vector<std::string_view> parts;
    int32_t count = 0;
    bool have = false;
    for_each_line(text, [&](std::string_view line) {
        if (!line.empty() && line[0] == '>') {
            if (!sequence.empty()) { table.add(sequence, label, count); sequence.clear(); }
            java_split(java_trim(line).substr(1), '|', parts);
            if (parts.size() >= 2) {
                count = decode_int(java_trim(parts[1]));
                if (count < 1) throw FileFormatException("Error while loading input file. Fasta header defines sequence count lower than 1.");
            } else count = 1;
            if (parts.size() >= 3) label.assign(parts[2]); else label = "no_label";
            have = true;
        } else {
            if (!have) throw FileFormatException("Error. Incorrect fasta format. Maybe header or sequence line missing?");
            sequence += java_trim(line);
        }
    });
    if (!have) throw FileFormatException("Error. Incorrect fasta format. Maybe header or sequence line missing?");
    table.add(sequence, label, count);
    std::vector<UniqueSequence> out;
    out.reserve(table.entries.size());
    for (auto& e : table.entries) out.emplace_back(std::move(e.sequence), std::move(e.labels));
    return out;
}

// FileIOManager.loadUniqueSequencesFromTable (FileIOManager.java:227-255)
inline std::vector<UniqueSequence> loadUniqueSequencesFromTable(const std::string& path) {
    const std::string text = read_file(path);
    std::vector<std::string> header;
    std::vector<std::string_view> parts;
    std::vector<UniqueSequence> out;
    bool first = true;
    for_each_line(text, [&](std::string_view line) {
        java_split(line, '\t', parts);
        if (first) { for (auto p : parts) header.emplace_back(p); first = false; return; }
        std::vector<std::pair<std::string, int32_t>> lab;
        for (size_t i = 1; i < parts.size(); i++) {
            const int32_t v = decode_int(parts[i]);
            if (v != 0) lab.emplace_back(header.at(i), v);
        }
        out.emplace_back(std::string(parts[0]), std::move(lab));
    });
    if (first) throw FileFormatException("empty table");
    return out;
}

// ---------------------------------------------------------------- labels, ordering, defaults
// Hammock.getSortedLabels (Hammock.java:1586-1605): TreeMap with ValueComparator
// (FileIOManager.java:1464-1480, never returns 0) filled from a HashMap: count descending, equal
// counts in REVERSE HashMap iteration order.
inline std::vector<std::string> getSortedLabels(const std::vector<UniqueSequence>& seqs) {
    std::vector<std::string> keys;
    std::unordered_map<std::string, int32_t> cnt;
    for (auto& s : seqs)
        for (auto& kv : s.labels) {
            if (!cnt.count(kv.first)) { keys.push_back(kv.first); cnt[kv.first] = 0; }
            cnt[kv.first] = wrap_add(cnt[kv.first], kv.second);
        }
    std::vector<std::string> sorted;   // in-order content of the TreeMap
    for (auto& k : java_hashmap_order(keys)) {
        size_t pos = 0;                // after everything strictly larger, before everything <= (compare: a >= b -> -1)
        while (pos < sorted.size() && cnt[sorted[pos]] > cnt[k]) pos++;
        sorted.insert(sorted.begin() + pos, k);
    }
    return sorted;
}

// UniqueSequence.sortSequences (UniqueSequence.java:176-203).  Sorted through an index array with the abundances computed
// once and the first eight letters as an integer (most comparisons never touch the strings); `permutation`, if given,
// receives for every new position the position the sequence had before (the reference keeps a copy of the list instead,
// Hammock.java:800).
inline void sortSequences(std::vector<UniqueSequence>& v, const std::string& order, const std::vector<std::string>& labels,
                          int64_t seed, std::vector<int>* permutation = nullptr) {
    struct Key { int32_t count, size; uint64_t prefix; int idx; };
    std::vector<Key> keys(v.size());
    for (size_t i = 0; i < v.size(); i++) {
        uint64_t p = 0;
        for (size_t k = 0; k < 8; k++) p = (p << 8) | (k < v[i].sequence.size() ? (unsigned char)v[i].sequence[k] : 0);
        keys[i] = Key{0, v[i].size(), p, (int)i};
    }
    auto alpha_desc = [&](const Key& a, const Key& b) {       // reverseOrder(String.compareTo), strict
        if (a.prefix != b.prefix) return a.prefix > b.prefix;
        return v[a.idx].sequence > v[b.idx].sequence;
    };
    auto size_alpha_desc = [&](const Key& a, const Key& b) {  // reverseOrder(SizeAlphabetic)
        if (a.size != b.size) return a.size > b.size;
        return alpha_desc(a, b);
    };
    if (order == "size") std::stable_sort(keys.begin(), keys.end(), size_alpha_desc);
    else if (order == "alphabetic") std::stable_sort(keys.begin(), keys.end(), alpha_desc);
    else if (order == "random") {   // Collections.shuffle(list, new Random(seed))
        JavaRandom rnd(seed);
        for (size_t i = keys.size(); i > 1; i--) std::swap(keys[i - 1], keys[(size_t)rnd.nextInt((int32_t)i)]);
    } else if (order == "input") {
    } else {                        // two stable sorts in the reference: by size/alphabet, then by the label's count
        if (std::find(labels.begin(), labels.end(), order) == labels.end())
            throw DataException("Incorrect sequence order defined. Use one of: size, alphabetic, random, input, or a label");
        for (auto& k : keys) k.count = v[k.idx].count(order);
        std::stable_sort(keys.begin(), keys.end(), [&](const Key& a, const Key& b) {
            if (a.count != b.count) return a.count > b.count;
            return size_alpha_desc(a, b);
        });
    }
    std::vector<UniqueSequence> sorted;
    sorted.reserve(v.size());
    for (auto& k : keys) sorted.push_back(std::move(v[k.idx]));
    v.swap(sorted);
    if (permutation) {
        permutation->resize(keys.size());
        for (size_t i = 0; i < keys.size(); i++) (*permutation)[i] = keys[i].idx;
    }
}

inline int32_t java_round(double x) { return (int32_t)std::floor(x + 0.5); }
inline double getMeanSequenceLength(const std::vector<UniqueSequence>& s) {   // Hammock.java:1554-1563
    int64_t sum = 0;
    for (auto& q : s) sum += (int64_t)q.length();
    return (double)sum / (double)s.size();
}
inline int32_t setGreedyThreshold(const std::vector<UniqueSequence>& s) { return java_round(getMeanSequenceLength(s) * 1.7); }   // :1409-1413
inline int32_t setClinkageThreshold(const std::vector<UniqueSequence>& s) { return java_round(getMeanSequenceLength(s) * 1.7); } // :1415-1419
inline int32_t checkMaxShift(const std::vector<UniqueSequence>& s, int32_t maxShift) {   // :1421-1427
    int32_t mn = INT32_MAX;
    for (auto& q : s) mn = std::min<int32_t>(mn, (int32_t)q.length());
    return std::min(maxShift, mn - 1);
}
inline int32_t getMaxShift(const std::vector<UniqueSequence>& s) { return checkMaxShift(s, java_round(getMeanSequenceLength(s) / 4)); }   // :1429-1434
inline int32_t initialClustersLimit(const std::vector<UniqueSequence>& s) { return java_round((double)s.size() * 0.025); }   // :398-401

// ---------------------------------------------------------------- the clusterer (SequenceClusterer seam)
// List<Cluster> from the arrays of the C ABI: members by rank, clusters in result order
// (ids: greedy 0 .. n-1 = the founder's index; clinkage 1 .. 2n+1 = Cluster ids in creation order)
inline std::vector<Cluster> rebuildClusters(int32_t n, const int32_t* cid, const int32_t* rank, const int32_t* order, int32_t nResult,
                                            const int32_t* abundance) {
    int32_t maxId = 0;
    for (int32_t i = 0; i < n; i++) {
        if (cid[i] < 0) throw HammockException("negative cluster id");
        maxId = std::max(maxId, cid[i]);
    }
    std::vector<int> start((size_t)maxId + 2, 0);
    for (int32_t i = 0; i < n; i++) start[cid[i] + 1]++;
    for (int32_t i = 0; i <= maxId; i++) start[i + 1] += start[i];
    std::vector<int> byRank(n);
    for (int32_t i = 0; i < n; i++) byRank[start[cid[i]] + rank[i]] = i;
    std::vector<Cluster> result;
    result.reserve(nResult);
    for (int32_t k = 0; k < nResult; k++) {
        Cluster c;
        c.id = order[k];
        c.members.assign(byRank.begin() + start[c.id], byRank.begin() + start[c.id + 1]);
        for (int m : c.members) c.sizeSum = wrap_add(c.sizeSum, abundance[m]);
        result.push_back(std::move(c));
    }
    return result;
}

// == new LimitedGreedySequenceClusterer(new ShiftedScorer(matrix, shiftPenalty, maxShift), threshold,
//    maxClusters).cluster(sequences)   (Hammock.java:402-409)
// the arrays of hmk_greedy_in for a sequence list in the caller's order
struct PackedSequences {
    std::vector<uint8_t> res;
    std::vector<int32_t> off, ab;
    explicit PackedSequences(const std::vector<UniqueSequence>& seqs) : off(seqs.size() + 1, 0), ab(seqs.size()) {
        size_t total = 0;
        for (auto& q : seqs) total += q.length();
        res.reserve(total + 1);
        for (size_t i = 0; i < seqs.size(); i++) {
            for (size_t k = 0; k < seqs[i].length(); k++) res.push_back(seqs[i].code(k));
            off[i + 1] = (int32_t)res.size();
            ab[i] = seqs[i].size();
        }
        if (res.empty()) res.push_back(0);
    }
};

struct GpuGreedySequenceClusterer {
    std::vector<int32_t> matrix;
    int32_t shiftPenalty, maxShift, threshold, maxClusters;
    int device = 0;

    std::vector<Cluster> cluster(const std::vector<UniqueSequence>& seqs) const {
        const int32_t n = (int32_t)seqs.size();
        std::vector<int32_t> cid(std::max(n, 1)), rank(std::max(n, 1)), order(std::max(n, 1));
        const PackedSequences packed(seqs);
        const std::vector<uint8_t>& res = packed.res;
        const std::vector<int32_t>&off = packed.off, &ab = packed.ab;
        hmk_greedy_in in{n, res.data(), off.data(), ab.data(), matrix.data(), threshold, maxShift, shiftPenalty, maxClusters};
        hmk_greedy_out out{cid.data(), rank.data(), order.data(), 0, 0, -1};
        char err[512] = {0};
        int rc = hmk_greedy_cluster(&in, &out, device, err, sizeof err);
        if (rc == HMK_STATUS_SHIFT_TOO_BIG) throw DataException(err);
        if (rc == HMK_STATUS_NULL_CLUSTER) throw NullPointerException(out.error_step);
        if (rc == HMK_STATUS_BAD_RESIDUE) throw FileFormatException(err);
        if (rc != HMK_STATUS_OK) throw CudaException(std::string("hammock_b200: ") + err);
        return rebuildClusters(n, cid.data(), rank.data(), order.data(), out.n_result, ab.data());
    }
};

// == new ClinkageSequenceClusterer(new ShiftedScorer(matrix, shiftPenalty, maxShift), threshold).cluster(sequences)
//    (Hammock.java:457-462): sequences in the caller's order (runClinkageClustering does not sort)
struct GpuClinkageSequenceClusterer {
    std::vector<int32_t> matrix;
    int32_t shiftPenalty, maxShift, threshold;
    int device = 0;

    std::vector<Cluster> cluster(const std::vector<UniqueSequence>& seqs) const {
        const int32_t n = (int32_t)seqs.size();
        std::vector<int32_t> cid(std::max(n, 1)), rank(std::max(n, 1)), order(std::max(n, 1));
        const PackedSequences packed(seqs);
        hmk_greedy_in in{n, packed.res.data(), packed.off.data(), packed.ab.data(), matrix.data(), threshold, maxShift, shiftPenalty, 0};
        hmk_greedy_out out{cid.data(), rank.data(), order.data(), 0, 0, -1};
        char err[512] = {0};
        int rc = hmk_clinkage_cluster(&in, &out, device, err, sizeof err);
        if (rc == HMK_STATUS_SHIFT_TOO_BIG) throw DataException(err);
        if (rc == HMK_STATUS_BAD_RESIDUE) throw FileFormatException(err);
        if (rc == HMK_STATUS_UNSUPPORTED) throw UnsupportedInput(err);
        if (rc != HMK_STATUS_OK) throw CudaException(std::string("hammock_b200: ") + err);
        return rebuildClusters(n, cid.data(), rank.data(), order.data(), out.n_result, packed.ab.data());
    }
};

// The score graph of `seqs` in the caller's order (hmk_score_graph on a context of its own): every pair i < j with
// scoreWithShift(seq j, seq i) >= threshold, handed to fn(edges, count) one page of at most `page` edges at a time, in
// graph order.  Returns the number of edges.
struct GpuScoreGraph {
    std::vector<int32_t> matrix;
    int32_t shiftPenalty, maxShift, threshold;
    int device = 0;

    template <class Fn>
    int64_t pull(const std::vector<UniqueSequence>& seqs, Fn&& fn, int64_t page = 1 << 20) const {
        const int32_t n = (int32_t)seqs.size();
        const PackedSequences packed(seqs);
        hmk_greedy_in in{n, packed.res.data(), packed.off.data(), packed.ab.data(), matrix.data(), threshold, maxShift, shiftPenalty, 0};
        char err[512] = {0};
        auto check = [&](int rc) {
            if (rc == HMK_STATUS_SHIFT_TOO_BIG) throw DataException(err);
            if (rc == HMK_STATUS_BAD_RESIDUE) throw FileFormatException(err);
            if (rc != HMK_STATUS_OK) throw CudaException(std::string("hammock_b200: ") + err);
        };
        hmk_ctx* ctx = nullptr;
        check(hmk_create(&ctx, device, err, sizeof err));
        struct Destroy { hmk_ctx* c; ~Destroy() { hmk_destroy(c); } } destroy{ctx};
        check(hmk_upload(ctx, &in, err, sizeof err));
        std::vector<hmk_graph_edge> buf((size_t)page);
        int64_t cursor[2] = {0, 0}, total = 0;
        while (cursor[0] != n || cursor[1] != 0) {
            int64_t got = 0;
            check(hmk_score_graph(ctx, cursor, buf.data(), page, &got, err, sizeof err));
            fn(buf.data(), (size_t)got);
            total += got;
        }
        return total;
    }
};

// The k nearest partners of every sequence of `seqs` in the caller's order (hmk_nearest on a context of its own): for
// each i, the sequences j != i with scoreWithShift(seq j, seq i) >= threshold, best first under (score desc, size desc,
// j asc).  Handed to fn(row_begin, n_rows, partner, score, shift, count, more) `rows` rows at a time (partner, score,
// shift: [n_rows][k]), so that host memory stays bounded.  Returns the number of entries.
struct GpuNearestPartners {
    std::vector<int32_t> matrix;
    int32_t shiftPenalty, maxShift, threshold, k;
    int device = 0;

    template <class Fn>
    int64_t pull(const std::vector<UniqueSequence>& seqs, Fn&& fn, int32_t rows = 1 << 16) const {
        const int32_t n = (int32_t)seqs.size();
        const PackedSequences packed(seqs);
        hmk_greedy_in in{n, packed.res.data(), packed.off.data(), packed.ab.data(), matrix.data(), threshold, maxShift, shiftPenalty, 0};
        char err[512] = {0};
        auto check = [&](int rc) {
            if (rc == HMK_STATUS_SHIFT_TOO_BIG) throw DataException(err);
            if (rc == HMK_STATUS_BAD_RESIDUE) throw FileFormatException(err);
            if (rc != HMK_STATUS_OK) throw CudaException(std::string("hammock_b200: ") + err);
        };
        hmk_ctx* ctx = nullptr;
        check(hmk_create(&ctx, device, err, sizeof err));
        struct Destroy { hmk_ctx* c; ~Destroy() { hmk_destroy(c); } } destroy{ctx};
        check(hmk_upload(ctx, &in, err, sizeof err));
        const size_t cap = (size_t)std::min(rows, std::max(n, 1));
        std::vector<int32_t> partner(cap * std::max(k, 1)), score(partner.size()), shift(partner.size()), count(cap), more(cap);
        int64_t total = 0;
        for (int32_t r0 = 0; r0 < n; r0 += (int32_t)cap) {
            const int32_t m = std::min<int32_t>((int32_t)cap, n - r0);
            check(hmk_nearest(ctx, k, r0, m, partner.data(), score.data(), shift.data(), count.data(), more.data(), err, sizeof err));
            fn(r0, m, partner.data(), score.data(), shift.data(), count.data(), more.data());
            for (int32_t t = 0; t < m; t++) total += count[t];
        }
        return total;
    }
};

// ---------------------------------------------------------------- result files (FileIOManager.java)
static const char SEP = '\t';   // Hammock.CSV_SEPARATOR (Hammock.java:35)

// Cluster.compareTo reversed (Cluster.java:197-204): size descending, then id descending; stable
inline std::vector<const Cluster*> clustersLargestFirst(const std::vector<Cluster>& clusters) {
    struct Key { int32_t size, id; const Cluster* c; };
    std::vector<Key> keys;
    keys.reserve(clusters.size());
    for (auto& c : clusters) keys.push_back(Key{c.size(), c.id, &c});
    std::stable_sort(keys.begin(), keys.end(), [](const Key& a, const Key& b) {
        if (a.size != b.size) return a.size > b.size;
        return a.id > b.id;
    });
    std::vector<const Cluster*> v;
    v.reserve(keys.size());
    for (auto& k : keys) v.push_back(k.c);
    return v;
}

// BufferedWriter: rows are formatted into one buffer and written in 1 MB pieces
class TsvWriter {
    std::FILE* f_;
    std::string buf_;
public:
    explicit TsvWriter(const std::string& path) : f_(std::fopen(path.c_str(), "wb")) {
        if (!f_) throw HammockException("cannot write " + path);
        buf_.reserve((1 << 20) + 4096);
    }
    TsvWriter(const TsvWriter&) = delete;
    TsvWriter& operator=(const TsvWriter&) = delete;
    ~TsvWriter() { flush(); std::fclose(f_); }
    void flush() { if (!buf_.empty()) { std::fwrite(buf_.data(), 1, buf_.size(), f_); buf_.clear(); } }
    TsvWriter& operator<<(std::string_view s) { buf_.append(s); if (buf_.size() > (1u << 20)) flush(); return *this; }
    TsvWriter& operator<<(const char* s) { return *this << std::string_view(s); }
    TsvWriter& operator<<(const std::string& s) { return *this << std::string_view(s); }
    TsvWriter& operator<<(char c) { buf_.push_back(c); return *this; }
    TsvWriter& operator<<(int32_t v) {   // Integer.toString
        char tmp[12];
        int n = 0;
        uint32_t u = v < 0 ? 0u - (uint32_t)v : (uint32_t)v;
        do { tmp[n++] = (char)('0' + u % 10); u /= 10; } while (u);
        if (v < 0) tmp[n++] = '-';
        while (n) buf_.push_back(tmp[--n]);
        return *this;
    }
};

inline std::vector<int32_t> sequenceSizes(const std::vector<UniqueSequence>& seqs) {
    std::vector<int32_t> sizes(seqs.size());
    for (size_t i = 0; i < seqs.size(); i++) sizes[i] = seqs[i].size();
    return sizes;
}

inline void writeHeader(TsvWriter& w, const char* second, const char* third, const std::vector<std::string>& labels) {
    w << "cluster_id" << SEP << second << SEP;
    if (third) w << third << SEP;
    w << "sum";
    for (auto& l : labels) w << SEP << l;
    w << '\n';
}

// one row of the *_sequences files; clusterId < 0 = "NA"
inline void writeRow(TsvWriter& w, int32_t clusterId, const UniqueSequence& s, int32_t size, bool alone,
                     const std::vector<std::string>& labels) {
    if (clusterId < 0) w << "NA"; else w << clusterId;
    w << SEP << s.sequence << SEP << (alone ? std::string_view(s.sequence) : std::string_view("NA")) << SEP << size;
    for (auto& l : labels) w << SEP << s.count(l);
    w << '\n';
}

// saveClusterSequencesToCsv (FileIOManager.java:398-404, 594-638): one row per sequence, clusters largest
// first, inside a cluster abundance desc then string desc.  The `alignment` column is the sequence
// itself for one-member clusters (Cluster.getFastaString) and "NA" for multi-member clusters: the
// reference fills it from the Clustal-Omega MSA it builds next (Hammock.java:414-426), which is outside
// this path; `cluster` mode accepts NA and rebuilds the MSAs (FileIOManager.java:351-357).
inline void saveClusterSequencesToCsv(const std::vector<Cluster>& clusters, const std::vector<UniqueSequence>& seqs,
                                      const std::string& path, const std::vector<std::string>& labels) {
    const std::vector<int32_t> sizes = sequenceSizes(seqs);
    TsvWriter w(path);
    writeHeader(w, "sequence", "alignment", labels);
    std::vector<int> m;
    for (const Cluster* c : clustersLargestFirst(clusters)) {
        m = c->members;
        std::stable_sort(m.begin(), m.end(), [&](int a, int b) {
            if (sizes[a] != sizes[b]) return sizes[a] > sizes[b];
            return seqs[a].sequence > seqs[b].sequence;
        });
        for (int i : m) writeRow(w, c->id, seqs[i], sizes[i], m.size() == 1, labels);
    }
}

// saveClusterSequencesToCsvOrdered (FileIOManager.java:371-374): same rows in the given sequence order; a sequence that
// is in no cluster gets NA (:625-627)
inline void saveClusterSequencesToCsvOrdered(const std::vector<Cluster>& clusters, const std::vector<UniqueSequence>& seqs,
                                             const std::vector<int>& sequenceOrder, const std::string& path,
                                             const std::vector<std::string>& labels) {
    std::vector<const Cluster*> of(seqs.size(), nullptr);
    for (auto& c : clusters) for (int i : c.members) of[i] = &c;
    TsvWriter w(path);
    writeHeader(w, "sequence", "alignment", labels);
    for (int i : sequenceOrder) {
        const Cluster* c = of[i];
        writeRow(w, c ? c->id : -1, seqs[i], seqs[i].size(), c && c->members.size() == 1, labels);
    }
}

// SaveClustersToCsv (FileIOManager.java:649-676): main_sequence = most abundant member, ties alphabetically FIRST
inline void SaveClustersToCsv(const std::vector<Cluster>& clusters, const std::vector<UniqueSequence>& seqs,
                              const std::string& path, const std::vector<std::string>& labels) {
    const std::vector<int32_t> sizes = sequenceSizes(seqs);
    TsvWriter w(path);
    writeHeader(w, "main_sequence", nullptr, labels);
    for (const Cluster* c : clustersLargestFirst(clusters)) {
        int best = c->members[0];
        for (int i : c->members)   // first element of sort(reverseOrder(UniqueSequence.compareTo)); stable
            if (sizes[i] > sizes[best] || (sizes[i] == sizes[best] && seqs[i].sequence < seqs[best].sequence)) best = i;
        w << c->id << SEP << seqs[best].sequence << SEP << c->size();
        for (auto& l : labels) {
            int32_t sum = 0;
            for (int i : c->members) sum = wrap_add(sum, seqs[i].count(l));
            w << SEP << sum;
        }
        w << '\n';
    }
}

// score_graph.tsv (graph mode): the header, then one row per edge as sequence strings -- the same bytes as the Python
// host's save_score_graph
inline void writeScoreGraphHeader(TsvWriter& w) { w << "sequence" << SEP << "partner" << SEP << "score" << SEP << "shift" << '\n'; }
inline void writeScoreGraphEdges(TsvWriter& w, const std::vector<UniqueSequence>& seqs, const hmk_graph_edge* e, size_t count) {
    for (size_t k = 0; k < count; k++)
        w << seqs[e[k].seq].sequence << SEP << seqs[e[k].partner].sequence << SEP << e[k].score << SEP << e[k].shift << '\n';
}

// nearest_partners.tsv (nearest mode): the header, then for each row its entries rank 1 .. count as sequence strings --
// the same bytes as the Python host's save_nearest_partners
inline void writeNearestHeader(TsvWriter& w) {
    w << "sequence" << SEP << "rank" << SEP << "partner" << SEP << "score" << SEP << "shift" << '\n';
}
inline void writeNearestRows(TsvWriter& w, const std::vector<UniqueSequence>& seqs, int32_t row_begin, int32_t n_rows, int32_t k,
                             const int32_t* partner, const int32_t* score, const int32_t* shift, const int32_t* count) {
    for (int32_t t = 0; t < n_rows; t++)
        for (int32_t r = 0; r < count[t]; r++) {
            const size_t e = (size_t)t * k + r;
            w << seqs[row_begin + t].sequence << SEP << (r + 1) << SEP << seqs[partner[e]].sequence << SEP << score[e] << SEP
              << shift[e] << '\n';
        }
}

// saveInputStatistics (FileIOManager.java:709-729); no newline after the last line
inline void saveInputStatistics(const std::vector<UniqueSequence>& seqs, const std::vector<std::string>& labels, const std::string& path) {
    TsvWriter w(path);
    for (auto& l : labels) w << SEP << l;
    w << '\n' << "total_count";
    for (auto& l : labels) { int32_t t = 0; for (auto& s : seqs) t = wrap_add(t, s.count(l)); w << SEP << t; }
    w << '\n' << "unique_count";
    for (auto& l : labels) { int32_t u = 0; for (auto& s : seqs) u += s.has(l) ? 1 : 0; w << SEP << u; }
}

}  // namespace hammock
