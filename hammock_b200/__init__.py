"""hammock_b200 -- B200-native greedy initial clustering stage of Hammock.

The product is libhammock_b200.so (hand-written CUDA for sm_100a, C ABI in
include/hammock_b200.h).  This package is the host-side mirror of the reference's interface
for that path (host.py) plus the build script and the synthetic workload generator.
"""
from .host import (ALPHABET, Cluster, CudaError, DataException, FileFormatException, GreedyContext,  # noqa: F401
                   GreedyResult, HammockException, LimitedGreedySequenceClusterer, NullClusterError, ShiftedScorer,
                   UniqueSequence, check_max_shift, get_max_shift, greedy_cluster_arrays, initial_clusters_limit,
                   load_scoring_matrix, load_unique_sequences_from_fasta, load_unique_sequences_from_table,
                   pack_sequences, rebuild_clusters, run_greedy_clustering, set_greedy_threshold, sort_sequences,
                   get_sorted_labels, java_hashmap_order, save_cluster_sequences_to_csv,
                   save_cluster_sequences_to_csv_ordered, save_clusters_to_csv, save_input_statistics, result_digest, ClinkageSequenceClusterer, UnsupportedInput,
                   clinkage_cluster_arrays, run_clinkage_clustering, set_clinkage_threshold, EDGE_DTYPE, score_graph,
                   save_score_graph, nearest_partners, save_nearest_partners)

__all__ = [n for n in dir() if not n.startswith("_")]
