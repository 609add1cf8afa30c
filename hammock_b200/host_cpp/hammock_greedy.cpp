// hammock_greedy -- native driver of the `greedy` mode of Hammock (Hammock.java:217-234, 392-437) on
// top of libhammock_b200: fasta/tab input -> ordering + automatic parameters -> GPU greedy clustering
// -> initial_clusters*.tsv in the reference's format, so that the unchanged Java `cluster` mode
// (`java -jar Hammock.jar cluster -i <outdir>/initial_clusters_sequences.tsv`) can take over.
// `hammock_greedy clinkage ...` is the `clinkage` mode (Hammock.java:236-252, 449-489): the exact complete-linkage
// clusterer on the sequences in INPUT order (no sorting, no cluster limit), same result files.
// `hammock_greedy graph ...` writes the score graph both clusterings are built from: every pair of sequences (input order,
// clinkage's automatic threshold and max shift) scoring >= threshold with its score and shift, to score_graph.tsv.
// `hammock_greedy nearest ... [-k n]` writes, on the same sequences and parameters, the n (default 8) best-scoring
// partners of every sequence with score and shift to nearest_partners.tsv, pulling rows in ranges.
// Flags keep the reference's names (Hammock.java:824-970).  Multiple alignments are NOT built here
// (that is the Clustal-Omega stage, outside this path): the alignment column is "NA" for multi-member
// clusters, which `cluster` mode accepts.
#include <chrono>
#include <iostream>

#include "hammock_host.hpp"

using namespace hammock;

static void usage() {
    std::cerr << "usage: hammock_greedy [greedy|clinkage|graph|nearest] -i <input.fa> -d <outdir> [-f fasta|tab] [-m <matrix.txt>] [-g <threshold>] [-x <max_shift>]\n"
                 "                      [-p <gap_penalty>] [--initial_clusters_limit <n>] [-R size|alphabetic|random|input|<label>]\n"
                 "                      [-S <seed>] [-l label1,label2,...] [-k <partners>] [--device <n>] [--dump-prepared]\n";
}

int main(int argc, char** argv) {
    std::string input, outdir, format = "fasta", matrixPath, order = "size";
    bool haveT = false, haveX = false, haveK = false, dump = false, haveLabels = false, timeHost = false, hostOnly = false;
    bool clinkage = false, graph = false, nearest = false;   // graph, nearest: input order and clinkage's automatic parameters
    int32_t nearestK = 8;
    int32_t threshold = 0, maxShift = 0, shiftPenalty = 0, limit = 0;   // shiftPenalty default 0 (Hammock.java:82)
    int64_t seed = 42;                                                   // Hammock.java:67
    int device = 0;
    std::vector<std::string> labels;
    try {
        for (int i = 1; i < argc; i++) {
            std::string a = argv[i];
            auto next = [&]() -> std::string {
                if (i + 1 >= argc) throw CLIException("Error. Parameter " + a + " needs a value.");
                return argv[++i];
            };
            if (a == "greedy") continue;
            else if (a == "clinkage" && i == 1) clinkage = true;
            else if (a == "graph" && i == 1) clinkage = graph = true;
            else if (a == "nearest" && i == 1) clinkage = nearest = true;
            else if (a == "-k" && nearest) nearestK = decode_int(next());
            else if (a == "-i" || a == "--input") input = next();
            else if (a == "-d" || a == "--outputDirectory") outdir = next();
            else if (a == "-f" || a == "--file_format") format = next();
            else if (a == "-m" || a == "--matrix") matrixPath = next();
            else if (a == "-g" || a == "--greedy_threshold" || a == "--alignment_threshold" || a == "--clinkage_threshold") {
                threshold = decode_int(next()); haveT = true;
            }
            else if (a == "-x" || a == "--max_shift") { maxShift = decode_int(next()); haveX = true; }
            else if (a == "-p" || a == "--gap_penalty") shiftPenalty = decode_int(next());
            else if (a == "--initial_clusters_limit") { limit = decode_int(next()); haveK = true; }
            else if (a == "-R" || a == "--order") order = next();
            else if (a == "-S" || a == "--seed") seed = decode_int(next());
            else if (a == "-t" || a == "--threads") next();   // accepted for compatibility; the GPU does the work
            else if (a == "--device") device = decode_int(next());
            else if (a == "--dump-prepared") dump = true;
            else if (a == "--time-host") timeHost = true;       // stage timings of the host side on stderr
            else if (a == "--host-only") hostOnly = true;       // stop before the GPU call (with --time-host: SURVEY.md 8f N4)
            else if (a == "-l" || a == "--labels") {
                std::string v = next(), cur;
                for (char c : v) { if (c == ',') { labels.push_back(cur); cur.clear(); } else cur.push_back(c); }
                labels.push_back(cur);
                haveLabels = true;
            } else if (a == "-h" || a == "--help") { usage(); return 0; }
            else throw CLIException("Error. Unknown parameter: " + a);
        }
        if (nearest && (nearestK < 1 || nearestK > HMK_NEAREST_MAX_K)) throw CLIException("Error. Parameter -k must be between 1 and 31.");
        if (input.empty()) throw CLIException("Error. Parameter input file (-i) missing with no default.");
        if (matrixPath.empty() && !dump) throw CLIException("Error. Parameter matrix (-m) missing (e.g. matrices/blosum62.txt of the Hammock distribution).");
        if (format != "fasta" && format != "tab") throw CLIException("Error. Wrong input file format. Use \"fasta\" or \"tab\"");

        auto tick = std::chrono::steady_clock::now();
        auto lap = [&](const char* what) {
            auto now = std::chrono::steady_clock::now();
            if (timeHost) std::cerr << "host time " << what << ": " << std::chrono::duration<double, std::milli>(now - tick).count() << " ms\n";
            tick = now;
        };
        // loadInputSequences (Hammock.java:749-787)
        std::vector<UniqueSequence> sequences = format == "fasta" ? loadUniqueSequencesFromFasta(input) : loadUniqueSequencesFromTable(input);
        lap("load + de-duplicate");
        if (haveLabels) {   // filterSequencesForLabels (Hammock.java:1661-1675): keep sequences having any listed label
            std::vector<UniqueSequence> kept;
            for (auto& s : sequences) {
                std::vector<std::pair<std::string, int32_t>> lab;
                for (auto& kv : s.labels) if (std::find(labels.begin(), labels.end(), kv.first) != labels.end()) lab.push_back(kv);
                if (!lab.empty()) kept.emplace_back(s.sequence, lab);
            }
            sequences.swap(kept);
        }
        if (sequences.empty()) throw FileFormatException("Error. No sequences (with specified labels) to cluster.");
        // prepareSequenceClustering (Hammock.java:795-817)
        if (!haveLabels) labels = getSortedLabels(sequences);
        if (!haveX) maxShift = getMaxShift(sequences); else maxShift = checkMaxShift(sequences, maxShift);
        if (!haveT) threshold = clinkage ? setClinkageThreshold(sequences) : setGreedyThreshold(sequences);   // Hammock.java:394-397, 452-455
        if (!haveK) limit = initialClustersLimit(sequences);              // :398-401
        lap("labels + automatic parameters");
        std::vector<int> cameFrom;                                        // input position of every sorted sequence
        // greedy: :407 (the reference copies the list instead, :800); clinkage clusters the list as loaded (:449-462)
        sortSequences(sequences, clinkage ? "input" : order, labels, seed, &cameFrom);
        lap("sortSequences");
        if (hostOnly) return 0;

        if (dump) {   // host-side state right before clusterer.cluster(sequences): used by the CPU tests
            std::cout << "threshold\t" << threshold << "\nmax_shift\t" << maxShift << "\nlimit\t" << limit << "\nlabels";
            for (auto& l : labels) std::cout << '\t' << l;
            std::cout << '\n';
            if (nearest) std::cout << "k\t" << nearestK << '\n';
            for (auto& s : sequences) std::cout << s.sequence << '\t' << s.size() << '\n';
            return 0;
        }

        const std::vector<int32_t> matrix = loadScoringMatrix(matrixPath);
        if (graph) {
            if (outdir.empty()) throw CLIException("Error. Parameter output directory (-d) missing: graph mode writes score_graph.tsv.");
            std::string d = outdir;
            if (d.back() != '/') d.push_back('/');
            std::cerr << "Score graph... (" << sequences.size() << " unique sequences, threshold " << threshold << ", max shift " << maxShift << ")\n";
            auto t0 = std::chrono::steady_clock::now();
            int64_t edges = 0;
            {
                TsvWriter w(d + "score_graph.tsv");
                writeScoreGraphHeader(w);
                edges = GpuScoreGraph{matrix, shiftPenalty, maxShift, threshold, device}.pull(
                    sequences, [&](const hmk_graph_edge* e, size_t count) { writeScoreGraphEdges(w, sequences, e, count); });
            }
            auto ms = std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - t0).count();
            std::cerr << "Ready. Time: " << ms << "\nEdges: " << edges << "\nScore graph in: " << d << "score_graph.tsv\n";
            return 0;
        }
        if (nearest) {
            if (outdir.empty()) throw CLIException("Error. Parameter output directory (-d) missing: nearest mode writes nearest_partners.tsv.");
            std::string d = outdir;
            if (d.back() != '/') d.push_back('/');
            std::cerr << "Nearest partners... (" << sequences.size() << " unique sequences, k " << nearestK << ", threshold " << threshold
                      << ", max shift " << maxShift << ")\n";
            auto t0 = std::chrono::steady_clock::now();
            int64_t entries = 0;
            {
                TsvWriter w(d + "nearest_partners.tsv");
                writeNearestHeader(w);
                entries = GpuNearestPartners{matrix, shiftPenalty, maxShift, threshold, nearestK, device}.pull(
                    sequences, [&](int32_t r0, int32_t m, const int32_t* partner, const int32_t* score, const int32_t* shift,
                                   const int32_t* count, const int32_t*) {
                        writeNearestRows(w, sequences, r0, m, nearestK, partner, score, shift, count);
                    });
            }
            auto ms = std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - t0).count();
            std::cerr << "Ready. Time: " << ms << "\nEntries: " << entries << "\nNearest partners in: " << d << "nearest_partners.tsv\n";
            return 0;
        }
        std::cerr << (clinkage ? "Clinkage" : "Greedy") << " clustering... (" << sequences.size() << " unique sequences, threshold " << threshold
                  << ", max shift " << maxShift;
        if (!clinkage) std::cerr << ", clusters limit " << limit;
        std::cerr << ")\n";
        auto t0 = std::chrono::steady_clock::now();
        std::vector<Cluster> clusters = clinkage ? GpuClinkageSequenceClusterer{matrix, shiftPenalty, maxShift, threshold, device}.cluster(sequences)
                                                 : GpuGreedySequenceClusterer{matrix, shiftPenalty, maxShift, threshold, limit, device}.cluster(sequences);
        auto ms = std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now() - t0).count();
        std::cerr << "Ready. Clustering time: " << ms << "\nResulting clusers: " << clusters.size() << "\n";   // Hammock.java:411-412

        if (!outdir.empty()) {
            std::string d = outdir;
            if (d.back() != '/') d.push_back('/');
            std::vector<int> inputOrder(sequences.size());   // clustering-order index of every input-order sequence
            for (size_t i = 0; i < cameFrom.size(); i++) inputOrder[cameFrom[i]] = (int)i;
            saveInputStatistics(sequences, labels, d + "input_statistics.tsv");   // sums: the order does not matter
            saveClusterSequencesToCsv(clusters, sequences, d + "initial_clusters_sequences.tsv", labels);
            saveClusterSequencesToCsvOrdered(clusters, sequences, inputOrder, d + "initial_clusters_sequences_original_order.tsv", labels);
            SaveClustersToCsv(clusters, sequences, d + "initial_clusters.tsv", labels);
            std::cerr << (clinkage ? "Clinkage" : "Greedy") << " clustering results in: " << d << "initial_clusters.tsv\nand: " << d
                      << "initial_clusters_sequences.tsv\n";
        }
        hmk_release_cached();
        return 0;
    } catch (const CLIException& e) {
        std::cerr << e.what() << "\n";
        usage();
        return 2;
    } catch (const HammockException& e) {
        std::cerr << "Error: " << e.what() << "\n";
        return 1;
    }
}
