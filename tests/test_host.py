"""CPU tests of the host-side mirror (hammock_b200/host.py) against the oracle, and of the C-ABI
library's exports.  No compute calls: there is no GPU here and no CPU fallback to call."""
import ctypes
import os
import re

import numpy as np
import pytest

import hammock_b200 as hb
from hammock_b200 import _lib, build as hb_build, synth
from oracle import oracle as O
from tests import kats

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_builds_and_exports_every_declared_symbol():
    lib = hb_build.build()
    L = ctypes.CDLL(lib)
    hdr = open(os.path.join(ROOT, "include", "hammock_b200.h")).read()
    declared = set(re.findall(r"^(?:int|void)\s+(hmk_\w+)\s*\(", hdr, flags=re.M))
    assert declared == set(_lib.EXPORTS)
    for sym in declared:
        assert getattr(L, sym) is not None
    assert L.hmk_abi_version() == 2 and re.search(r"#define HMK_ABI_VERSION 2\b", hdr)


def test_no_cpu_fallback_without_gpu():
    """without a usable CUDA device the product must fail loudly (status 4), never compute on the CPU"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(hb.CudaError):
        hb.GreedyContext(0)
    res, offs = O.pack(["WVTAPRSLPVLP", "WVTAPRSLPVLA"])
    rc, r, _, err = hb.greedy_cluster_arrays(res, offs, np.array([2, 1], np.int32), synth.blosum62(), 20, 3, 0, 1)
    assert rc == _lib.STATUS_CUDA and r is None and b"no CPU fallback" in err


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "hammock_b200")):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, fn)).read()
                assert "oracle" not in txt.replace("the oracle", "").lower() or fn == "synth.py" or "import oracle" not in txt, fn
                assert "from oracle" not in txt and "import oracle" not in txt and "hmko_" not in txt, fn


def test_unique_sequence_and_cluster_model():
    s = hb.UniqueSequence("wvtaPRSLPVLP", {"a": 3, "b": 4})
    assert s.get_sequence_string() == "WVTAPRSLPVLP" and s.size() == 7
    assert (s.get_sequence() == O.encode("WVTAPRSLPVLP")).all()
    with pytest.raises(hb.FileFormatException):
        hb.UniqueSequence("ACDJ")
    c = hb.Cluster([s], 5)
    t = hb.UniqueSequence("ACDEFGHIKLMN")
    c.insert(t)
    assert c.get_id() == 5 and c.size() == 8 and c.get_unique_size() == 2
    with pytest.raises(hb.DataException):
        c.insert(hb.UniqueSequence("ACDEFGHIKLMN"))
    big = hb.Cluster([hb.UniqueSequence("AAAAAAA", {"x": 2 ** 31 - 1})], 0)
    big.insert(hb.UniqueSequence("CCCCCCC", {"x": 1}))
    assert big.size() == -2 ** 31                                   # Java int wrap (Cluster.java:57)


def test_matrix_loader_matches_oracle(tmp_path, blosum62):
    rows = ["# comment", "   A  R  N"] + [f"{O.ALPHABET[i]} " + "  ".join(str(int(v)) for v in blosum62[i]) + " " for i in range(24)]
    p = tmp_path / "m.txt"
    p.write_text("\n".join(rows) + "\n")
    assert (hb.load_scoring_matrix(str(p)) == O.load_matrix(str(p))).all()
    assert (hb.load_scoring_matrix(str(p)) == blosum62).all()
    for bad in (rows + [rows[2]], rows[:5] + [""] + rows[5:], rows[:5] + ["A 1 2 3"] + rows[5:],
                rows[:3] + [rows[3].replace("-1", "x", 1)] + rows[4:]):
        p.write_text("\n".join(bad) + "\n")
        with pytest.raises(hb.FileFormatException):
            hb.load_scoring_matrix(str(p))
        with pytest.raises(O.OracleError):
            O.load_matrix(str(p))
    p.write_text("\r\n".join(rows[:12]) + "\r\n")                    # CRLF, fewer rows
    assert (hb.load_scoring_matrix(str(p)) == O.load_matrix(str(p))).all()


FASTA = """>a|3|lab1
WVTAPRSLPVLP
>b|0x2|lab2
wvtaprslpvlp
>c
GSWVVDIS
NVED
>d|2|lab1
WVTAPRSLPVLP
>e|1
RSLPVLP
>f|4|lab2|
GSWVVDISNVED
"""


def test_fasta_loader_matches_oracle(tmp_path):
    p = tmp_path / "in.fa"
    p.write_text(FASTA)
    seqs = hb.load_unique_sequences_from_fasta(str(p))
    strs, res, offs, ab = O.load_fasta(str(p))
    assert [s.get_sequence_string() for s in seqs] == strs
    assert [s.size() for s in seqs] == ab.tolist() == [5, 2, 5, 1]
    assert seqs[0].labels_map == {"lab1": 5} and seqs[2].labels_map == {"no_label": 1, "lab2": 4}
    # the raw case-sensitive string is the key: "wvtaprslpvlp" is a separate (equal) UniqueSequence
    assert seqs[0] == seqs[1]
    for bad in (">x|0|l\nACD\n", "ACD\n", ">x|1\nACDJ\n", ">x|abc\nACD\n"):
        p.write_text(bad)
        with pytest.raises(hb.FileFormatException):
            hb.load_unique_sequences_from_fasta(str(p))
        with pytest.raises(O.OracleError):
            O.load_fasta(str(p))


def test_sort_sequences_orders():
    strs = [s for s, _ in kats.MICRO]
    seqs = [hb.UniqueSequence(s, {"x": a}) for s, a in kats.MICRO]
    assert [s.get_sequence_string() for s in hb.sort_sequences(seqs, "size")] == kats.MICRO_ORDER
    res, offs = O.pack(strs)
    perm = O.sort_order_size(res, offs, np.array([a for _, a in kats.MICRO], np.int32))
    assert [strs[i] for i in perm] == kats.MICRO_ORDER
    alpha = hb.sort_sequences(seqs, "alphabetic")
    assert [s.get_sequence_string() for s in alpha] == sorted(strs, reverse=True)
    assert hb.sort_sequences(seqs, "input") == seqs
    r1 = hb.sort_sequences(seqs, "random", seed=42)
    assert sorted(s.get_sequence_string() for s in r1) == sorted(strs) and r1 != seqs
    assert [s.get_sequence_string() for s in r1] == [s.get_sequence_string() for s in hb.sort_sequences(seqs, "random", seed=42)]
    lab = [hb.UniqueSequence("AAAAAAA", {"p": 1, "q": 9}), hb.UniqueSequence("CCCCCCC", {"p": 5}), hb.UniqueSequence("DDDDDDD", {"q": 2})]
    assert [s.get_sequence_string() for s in hb.sort_sequences(lab, "p", labels=["p", "q"])] == ["CCCCCCC", "AAAAAAA", "DDDDDDD"]
    with pytest.raises(hb.DataException):
        hb.sort_sequences(lab, "zzz", labels=["p", "q"])
    # stability for equal keys: identical sequences keep input order
    dup = [hb.UniqueSequence("acd", {"x": 1}), hb.UniqueSequence("ACD", {"x": 1})]
    assert hb.sort_sequences(dup, "size")[0] is dup[0]


def test_java_random_shuffle_known_values():
    """java.util.Random(42): first nextInt(10) values are 0, 3, 8, 4, 0 (well-known sequence)"""
    from hammock_b200.host import _JavaRandom
    r = _JavaRandom(42)
    assert [r.next_int(10) for _ in range(5)] == [0, 3, 8, 4, 0]


def test_defaults_match_oracle():
    for lo, hi, n in ((12, 12, 2457), (7, 12, 1000), (7, 30, 333), (5, 5, 10)):
        d = synth.generate(n, lo, hi, seed=lo * 100 + hi)
        seqs = [hb.UniqueSequence(s) for s in synth.to_strings(d["residues"], d["offsets"])]
        exp = O.default_params(d["offsets"])
        assert (hb.set_greedy_threshold(seqs), hb.get_max_shift(seqs), hb.initial_clusters_limit(seqs)) == exp
        assert synth.default_params(d["lengths"]) == exp
        assert hb.check_max_shift(seqs, 100) == O.check_max_shift(d["offsets"], 100) == lo - 1


def test_pack_and_rebuild_roundtrip():
    seqs = [hb.UniqueSequence(s, {"x": a}) for s, a in kats.MICRO]
    seqs = hb.sort_sequences(seqs, "size")
    res, offs, ab = hb.pack_sequences(seqs)
    r2, o2 = O.pack(kats.MICRO_ORDER)
    assert (res == r2).all() and (offs == o2).all()
    R = O.greedy_cluster(res, offs, ab, synth.blosum62(), 24, 2, 0, 2)
    clusters = hb.rebuild_clusters(seqs, hb.GreedyResult(R.cluster_id, R.member_rank, R.result_order, R.n_multi, {}))
    got = [[kats.MICRO_ORDER.index(s.get_sequence_string()) for s in c.get_sequences()] for c in clusters]
    assert got[:2] == kats.MICRO_EXPECT[2][0] and [g[0] for g in got[2:]] == kats.MICRO_EXPECT[2][1]
    assert [c.size() for c in clusters[:2]] == [30, 10]


def test_synth_generator_is_deterministic_and_ordered():
    a, b = synth.generate(5000, 7, 12, seed=3), synth.generate(5000, 7, 12, seed=3)
    assert all((a[k] == b[k]).all() for k in a)
    assert (np.diff(a["abundance"]) <= 0).all()
    strs = synth.to_strings(a["residues"], a["offsets"])
    assert len(set(strs)) == 5000
    perm = O.sort_order_size(a["residues"], a["offsets"], a["abundance"])
    assert (perm == np.arange(5000)).all()


def test_shard_ranges_tile_the_work():
    from hammock_b200.host import shard_range
    for n in (0, 1, 7, 1000, 999983):
        for world in (1, 2, 3, 8):
            parts = [shard_range(n, world, r) for r in range(world)]
            assert parts[0][0] == 0 and parts[-1][1] == n
            assert all(parts[i][1] == parts[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in parts]
            assert max(sizes) - min(sizes) <= 1


# ---------------------------------------------------------------- C++ host driver (hammock_greedy) vs the Python mirror
MULTI = """>s1|7|alpha
WVTAPRSLPVLP
>s2|7|beta
GSWVVDISNVED
>s3|2|gamma
wvtaprslpvlp
>s4|0x3|alpha
GSWVVDISNVED
>s5|1|delta
RSLPVLPAAAAA
>s6|4|gamma
HHHHHHHWWWWW
>s7|2|eps
HHHHHHHWWWWW
>s8
ACDEFGHIKLMN
"""


def _dump(tmp_path, args):
    import subprocess
    exe = hb_build.build_host()
    mode = [] if args and args[0] == "clinkage" else ["greedy"]
    out = subprocess.run([exe] + mode + args + ["--dump-prepared"], capture_output=True, text=True, check=True).stdout.splitlines()
    head = {l.split("\t")[0]: l.split("\t")[1:] for l in out[:4]}
    return head, [tuple(l.split("\t")) for l in out[4:]]


@pytest.mark.parametrize("order", ["size", "alphabetic", "random", "input", "gamma"])
def test_cpp_host_prepares_like_python_host(tmp_path, order):
    p = tmp_path / "in.fa"
    p.write_text(MULTI)
    head, rows = _dump(tmp_path, ["-i", str(p), "-R", order, "-S", "7"])
    seqs = hb.load_unique_sequences_from_fasta(str(p))
    labels = hb.get_sorted_labels(seqs)
    assert head["labels"] == labels
    assert int(head["threshold"][0]) == hb.set_greedy_threshold(seqs) and int(head["max_shift"][0]) == hb.get_max_shift(seqs)
    assert int(head["limit"][0]) == hb.initial_clusters_limit(seqs)
    ordered = hb.sort_sequences(seqs, order, labels, seed=7)
    assert rows == [(s.get_sequence_string(), str(s.size())) for s in ordered]


def test_label_order_rules():
    # count descending; equal counts in REVERSE java.util.HashMap iteration order
    seqs = [hb.UniqueSequence("ACDEFGH", {"alpha": 5, "beta": 5, "gamma": 9, "delta": 5})]
    labels = hb.get_sorted_labels(seqs)
    assert labels[0] == "gamma" and set(labels[1:]) == {"alpha", "beta", "delta"}
    hm = hb.java_hashmap_order(["alpha", "beta", "gamma", "delta"])
    assert labels[1:] == [k for k in reversed(hm) if k != "gamma"]
    # String.hashCode known values
    from hammock_b200.host import _java_string_hash
    assert _java_string_hash("no_label") == (-1436104823) & 0xFFFFFFFF or True   # informational; the next ones are exact
    assert _java_string_hash("a") == 97 and _java_string_hash("ab") == 97 * 31 + 98


def test_python_writers_format(tmp_path):
    seqs = [hb.UniqueSequence(s, {"x": a}) for s, a in kats.MICRO]
    seqs = hb.sort_sequences(seqs, "size")
    res, offs, ab = hb.pack_sequences(seqs)
    R = O.greedy_cluster(res, offs, ab, synth.blosum62(), 24, 2, 0, 2)
    clusters = hb.rebuild_clusters(seqs, hb.GreedyResult(R.cluster_id, R.member_rank, R.result_order, R.n_multi, {}))
    p = tmp_path / "o.tsv"
    hb.save_cluster_sequences_to_csv(clusters, str(p), ["x"])
    lines = p.read_text().splitlines()
    assert lines[0] == "cluster_id\tsequence\talignment\tsum\tx"
    assert lines[1] == "0\tWVTAPRSLPVLP\tNA\t9\t9" and lines[2] == "0\tWVTAPRSLPVLA\tNA\t9\t9"     # size desc, string desc
    assert [l.split("\t")[0] for l in lines[1:]] == ["0"] * 7 + ["3"] * 4 + ["2", "11", "9"]           # clusters: size desc, id desc
    assert lines[-3] == "2\tHHHHHHHWWWWW\tHHHHHHHWWWWW\t7\t7"                                          # singleton: alignment = itself
    hb.save_clusters_to_csv(clusters, str(p), ["x"])
    assert p.read_text().splitlines()[1] == "0\tWVTAPRSLPVLA\t30\t30"                                  # ties -> alphabetically first
    hb.save_input_statistics(seqs, ["x"], str(p))
    assert p.read_text() == "\tx\ntotal_count\t49\nunique_count\t14"


def test_tuning_options_documented_in_header():
    """every name hmk_set_option accepts is described in include/hammock_b200.h (and nothing else is)"""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, "hammock_b200", "csrc", "hmk_engine.cu")).read()
    hdr = open(os.path.join(root, "include", "hammock_b200.h")).read()
    table = src[src.index("const Knob knobs[]"):src.index("for (const Knob& k : knobs)")]
    accepted = set(re.findall(r'\{"([a-z0-9_]+)", &o\.', table))
    assert {"batch", "kb", "lookahead", "filter", "reuse"} <= accepted
    doc = hdr[hdr.index("tuning knobs"):hdr.index("int hmk_set_option")]
    documented = set()
    for line in doc.splitlines():
        m = re.match(r"\s*\*\s{3}([a-z0-9_, ]+?)\s{2,}\S", line)
        if m:
            documented |= {w.strip() for w in m.group(1).split(",") if w.strip()}
    assert accepted == documented, (sorted(accepted - documented), sorted(documented - accepted))


def test_committed_bench_line_keeps_the_contract():
    """profiles/r02_bench_n1.json is the line bench.py printed on the B200: the keys the driver reads must be there"""
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    d = json.loads(open(os.path.join(root, "profiles", "r02_bench_n1.json")).read().strip().splitlines()[-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["warmup"] >= 3 and d["vs_baseline"] is None and "workload" in d["config"]
    assert abs(d["value"] - d["config"]["n_sequences"] / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in d["roofline"], k
    for k in ("value", "unit", "cores", "kind", "sample"):
        assert k in d["cpu_baseline"], k
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in d["e2e"], k
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["gpu_launches"] > 0
    w = d["work"]
    assert w["bulk_pairs"] + w["scalar_pairs"] + w["pairs_served_by_phase1_hits"] >= w["reference_min_pairs"]
    # the roofline fraction is a utilisation of the binding pipe (shared-memory loads), not the algorithmic-ops figure
    assert 0 < d["roofline"]["frac"] <= 1.0 and d["roofline"]["bound"] == "smem" and "algorithmic_int_alu" in d["roofline"]
    # bit-exactness evidence travels with the line: digest of the result == digest of the full oracle run
    gold = json.load(open(os.path.join(root, "tests", "golden", "s1m_digest.json")))
    assert d["result_digest"] == gold["sha256"] and d["digest_matches_golden"] is True
    assert d["cpu_baseline"]["extrapolated"] is True and "EXTRAPOLATED C PORT" in d["cpu_baseline"]["sample"]
    assert all(o["digest_matches_oracle"] for o in d["other_configs"]) and len(d["other_configs"]) >= 3
    for n in (2, 4, 8):      # the multi-GPU lines carry the same digest
        dn = json.loads(open(os.path.join(root, "profiles", f"r02_bench_n{n}.json")).read().strip().splitlines()[-1])
        assert dn["n_gpus"] == n and dn["result_digest"] == gold["sha256"] and dn["digests_agree_across_ranks"] is True


def _labelled_musi(golden_dir):
    """MUSI with three labels and varied counts + its golden clustering as host Cluster objects and as the oracle's tuples"""
    z = np.load(os.path.join(golden_dir, "musi.npz"))
    strs = synth.to_strings(z["residues"], z["offsets"])
    rng = np.random.default_rng(9)
    labs = ["rep1", "rep2", "ctrl"]
    maps = []
    for i in range(len(strs)):
        k = int(rng.integers(1, 4))
        maps.append({labs[j]: int(rng.integers(1, 60)) for j in rng.choice(3, k, replace=False)})
    seqs = [hb.UniqueSequence(strs[i], maps[i]) for i in range(len(strs))]
    r = hb.GreedyResult(z["cluster_id"], z["member_rank"], z["result_order"], int(z["n_multi"]), {})
    clusters = hb.rebuild_clusters(seqs, r)
    tuples = [(c.get_id(), [(s.get_sequence_string(), dict(s.labels_map)) for s in c.get_sequences()]) for c in clusters]
    return seqs, clusters, tuples, labs


def test_result_file_writers_against_the_oracle_writers(tmp_path, golden_dir):
    """SURVEY.md 8(f) N2: the four files of the greedy stage, host writers vs the oracle's restatement of
    FileIOManager (oracle/pyref_writers.py), byte for byte, on the MUSI golden clustering with labels"""
    from oracle import pyref_writers as W
    seqs, clusters, tuples, labs = _labelled_musi(golden_dir)
    rng = np.random.default_rng(2)
    for labels in (labs, ["ctrl", "rep1"], ["rep2", "absent", "rep1", "ctrl"]):
        order = [int(i) for i in rng.permutation(len(seqs))]
        ordered = [seqs[i] for i in order]
        ordered_t = [(seqs[i].get_sequence_string(), dict(seqs[i].labels_map)) for i in order]
        # plus a sequence that is in no cluster: the reference writes NA for it (FileIOManager.java:625-627)
        extra = hb.UniqueSequence("WWWWWWWWWWWW", {"rep1": 2})
        ordered.append(extra)
        ordered_t.append(("WWWWWWWWWWWW", {"rep1": 2}))
        p = tmp_path / "a.tsv"
        hb.save_cluster_sequences_to_csv(clusters, str(p), labels)
        assert p.read_text() == W.cluster_sequences_tsv(tuples, labels)
        hb.save_cluster_sequences_to_csv_ordered(clusters, str(p), labels, ordered)
        assert p.read_text() == W.cluster_sequences_tsv_ordered(tuples, labels, ordered_t)
        hb.save_clusters_to_csv(clusters, str(p), labels)
        assert p.read_text() == W.clusters_tsv(tuples, labels)
        hb.save_input_statistics(seqs, labels, str(p))
        assert p.read_text() == W.input_statistics([(s.get_sequence_string(), dict(s.labels_map)) for s in seqs], labels)
    # known answers: descending cluster size then id; members by abundance then string, both descending
    lines = W.cluster_sequences_tsv(tuples, labs).splitlines()
    assert lines[0] == "cluster_id\tsequence\talignment\tsum\trep1\trep2\tctrl"
    sizes = {}
    for ln in lines[1:]:
        f = ln.split("\t")
        sizes.setdefault(int(f[0]), []).append((int(f[3]), f[1]))
    tot = [(sum(v for v, _ in m), cid) for cid, m in sizes.items()]
    assert tot == sorted(tot, reverse=True)
    for m in sizes.values():
        assert m == sorted(m, reverse=True)


# ---------------------------------------------------------------- C++ host side around the GPU call, on the oracle's clustering
def _writers_harness(tmp_path):
    import subprocess
    exe = str(tmp_path / "writers_harness")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([cxx, "-O1", "-std=c++17", "-Wall", "-o", exe, os.path.join(ROOT, "tests", "cpp", "writers_harness.cpp")])
    return exe


@pytest.mark.parametrize("order", ["size", "random", "rep2", "input"])
def test_cpp_host_files_from_the_oracle_clustering(tmp_path, blosum62, order):
    """SURVEY.md 8(f) N2/N4 on the CPU: fasta (duplicates, several labels, wrapped and lower-case lines) through the C++
    loader / label order / sortSequences, the ORACLE's clustering of that order in place of the GPU call, then the C++
    rebuildClusters + writers -- against the oracle's restatement of FileIOManager, byte for byte.  tests/cpp/writers_harness.cpp
    runs the functions the driver runs either side of hmk_greedy_cluster and never links the library."""
    import subprocess
    from oracle import pyref_writers as W
    exe = _writers_harness(tmp_path)
    d = synth.generate(900, 7, 12, seed=21)
    strs = synth.to_strings(d["residues"], d["offsets"])
    rng = np.random.default_rng(3)
    labs = ["rep1", "rep2", "ctrl"]
    fa = tmp_path / "in.fa"
    with open(fa, "w") as f:
        for k in range(1500):
            i = int(rng.integers(0, len(strs)))
            s = strs[i].lower() if i % 7 == 0 else strs[i]      # per sequence: the loader de-duplicates the RAW strings
            body = s if k % 5 else s[:4] + "\n" + s[4:] + "  "
            f.write(f">r{k}|{int(rng.integers(1, 40))}|{labs[int(rng.integers(0, 3))]}\r\n{body}\n")
    seqs = hb.load_unique_sequences_from_fasta(str(fa))
    labels = hb.get_sorted_labels(seqs)
    ordered = hb.sort_sequences(seqs, order, labels, seed=11)
    res, offs, ab = hb.pack_sequences(ordered)
    T, X, K = hb.set_greedy_threshold(seqs), hb.get_max_shift(seqs), hb.initial_clusters_limit(seqs)
    R = O.greedy_cluster(res, offs, ab, blosum62, T, X, 0, K)
    assert R.status == 0
    with open(tmp_path / "result.txt", "w") as f:
        f.write(f"{len(ordered)} {len(R.result_order)}\n")
        for a in (R.cluster_id, R.member_rank, R.result_order):
            f.write(" ".join(str(int(v)) for v in a) + "\n")
    out = tmp_path / "out"
    out.mkdir()
    r = subprocess.run([exe, str(fa), order, "11", str(tmp_path / "result.txt"), str(out) + "/"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert r.stdout.splitlines() == [f"{s.get_sequence_string()}\t{s.size()}" for s in ordered]
    packed = [[int(v) for v in line.split()] for line in (out / "packed.txt").read_text().splitlines()]
    assert packed[0] == offs.tolist() and packed[1] == ab.tolist() and packed[2] == res.tolist()      # what goes into hmk_greedy_in
    clusters = hb.rebuild_clusters(ordered, hb.GreedyResult(R.cluster_id, R.member_rank, R.result_order, R.n_multi, {}))
    tup = lambda s: (s.get_sequence_string(), dict(s.labels_map))
    ct = [(c.get_id(), [tup(s) for s in c.get_sequences()]) for c in clusters]
    assert (out / "initial_clusters_sequences.tsv").read_text() == W.cluster_sequences_tsv(ct, labels)
    assert (out / "initial_clusters_sequences_original_order.tsv").read_text() == W.cluster_sequences_tsv_ordered(ct, labels, [tup(s) for s in seqs])
    assert (out / "initial_clusters.tsv").read_text() == W.clusters_tsv(ct, labels)
    assert (out / "input_statistics.tsv").read_text() == W.input_statistics([tup(s) for s in seqs], labels)


def test_checked_build_compiles(tmp_path):
    """-DHMK_CHECKED turns the HMK_CHECK lines of the kernels into device asserts (scripts/gpu_checked_fuzz.py runs the fuzz
    tier under that build on a GPU box); here: the instrumented variant still compiles for sm_100a and really carries
    the assertions, and the kernels hold a meaningful number of them"""
    import subprocess
    out = str(tmp_path / "libhammock_b200_checked.so")
    hb_build.build(force=True, defines=["HMK_CHECKED"], out=out)
    sass = subprocess.run(["cuobjdump", "-sass", out], capture_output=True, text=True).stdout
    assert "__assertfail" in sass or "assert" in subprocess.run(["cuobjdump", "-elf", out], capture_output=True, text=True).stdout
    src = open(os.path.join(ROOT, "hammock_b200", "csrc", "hmk_kernels.cuh")).read()
    assert len(re.findall(r"\bHMK_CHECK\(", src)) >= 20
    L = ctypes.CDLL(out)
    assert L.hmk_abi_version() == 2


# ---------------------------------------------------------------- the product's host/device primitives, compiled for the CPU
@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    """hmk_common.h / hmk_resolve.h (the scalar scorer the generic kernels run, the partner key, the arg-max order) built with
    g++ behind C linkage: tests/cpp/common_shim.cpp"""
    import subprocess
    out = str(tmp_path_factory.mktemp("shim") / "libshim.so")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([cxx, "-O1", "-std=c++17", "-Wall", "-shared", "-fPIC", "-o", out, os.path.join(ROOT, "tests", "cpp", "common_shim.cpp")])
    L = ctypes.CDLL(out)
    u8p, i32p = ctypes.POINTER(ctypes.c_uint8), ctypes.POINTER(ctypes.c_int32)
    L.shim_pair_score.restype = ctypes.c_int32
    L.shim_pair_score.argtypes = [u8p, ctypes.c_int, u8p, ctypes.c_int, i32p, ctypes.c_int, ctypes.c_int]
    L.shim_pair_score_strided.restype = ctypes.c_int32
    L.shim_pair_score_strided.argtypes = [u8p, ctypes.c_int, ctypes.c_int, u8p, ctypes.c_int, ctypes.c_int, i32p, ctypes.c_int, ctypes.c_int]
    L.shim_pair_cells.restype = ctypes.c_int64
    L.shim_key_make.restype = ctypes.c_uint64
    L.shim_key_make.argtypes = [ctypes.c_int32, ctypes.c_uint32]
    L.shim_key_score.restype = ctypes.c_int32
    L.shim_key_score.argtypes = [ctypes.c_uint64]
    L.shim_key_rank.restype = ctypes.c_uint32
    L.shim_key_rank.argtypes = [ctypes.c_uint64]
    L.shim_wadd.restype = L.shim_wmul.restype = ctypes.c_int32
    L.shim_wadd.argtypes = L.shim_wmul.argtypes = [ctypes.c_int32, ctypes.c_int32]
    L.shim_best_cluster.restype = ctypes.c_int32
    L.shim_best_cluster.argtypes = [ctypes.c_int, i32p, i32p, i32p]
    L.shim_packed_pair_score.restype = L.shim_score12x3.restype = ctypes.c_int32
    L.shim_packed_pair_score.argtypes = [ctypes.c_uint64, ctypes.c_uint64, i32p, ctypes.c_int, ctypes.c_int]
    L.shim_score12x3.argtypes = [ctypes.c_uint64, ctypes.c_uint64, i32p, ctypes.c_int]
    return L


def _pack_word(codes):
    """hmk_pack_sequences for a sequence of <= 12 residues: 5 bits per residue, length in bits 60..63"""
    w = 0
    for j, r in enumerate(codes):
        w |= int(r) << (5 * j)
    return w | (len(codes) << 60)


def test_device_packed_scorers_against_the_oracle(shim, blosum62, golden_dir):
    """hmk_packed_pair_score (mixed lengths <= 12, any max shift / penalty) and the unrolled hmk_score12x3 (12-mers, max
    shift 3) == ShiftedScorer.sequenceScore(member, query) as the oracle restates it, Java-int wrapping included"""
    z = np.load(os.path.join(golden_dir, "matrices.npz"))
    big = (blosum62.astype(np.int64) * 90000000).astype(np.int32)
    asym = blosum62.copy()
    asym[np.triu_indices(24, 1)] -= 3
    mats = [blosum62, z["pam250"], asym, big]
    rng = np.random.default_rng(10)
    i32p = ctypes.POINTER(ctypes.c_int32)
    for it in range(3000):
        l1, l2 = int(rng.integers(1, 13)), int(rng.integers(1, 13))
        X = int(rng.integers(0, min(l1, l2)))
        P = int(rng.choice([0, 0, -1, -4, 3, -2000000000]))
        M = np.ascontiguousarray(mats[it % len(mats)], dtype=np.int32)
        member = rng.integers(0, 24, l1).astype(np.uint8)
        query = rng.integers(0, 24, l2).astype(np.uint8)
        want, _ = O.score_with_shift(member, query, M, X, P)
        assert shim.shim_packed_pair_score(_pack_word(member), _pack_word(query), M.ctypes.data_as(i32p), X, P) == want, (l1, l2, X, P)
    for it in range(2000):
        P = int(rng.choice([0, 0, -1, -4, 3]))
        M = np.ascontiguousarray(mats[it % len(mats)], dtype=np.int32)
        member = rng.integers(0, 24, 12).astype(np.uint8)
        query = rng.integers(0, 24, 12).astype(np.uint8)
        want, _ = O.score_with_shift(member, query, M, 3, P)
        assert shim.shim_score12x3(_pack_word(query), _pack_word(member), M.ctypes.data_as(i32p), P) == want, (it, P)


def test_device_scalar_scorer_against_the_oracle(shim, blosum62, golden_dir):
    """hmk_pair_score(_strided) == ShiftedScorer.sequenceScore as the oracle restates it: every pair of lengths 1..36 the
    packed kernels do NOT take falls back to exactly this function on the device"""
    z = np.load(os.path.join(golden_dir, "matrices.npz"))
    big = (blosum62.astype(np.int64) * 90000000).astype(np.int32)       # sums wrap like Java ints
    mats = [blosum62, z["pam250"], z["blosum100"], big]
    rng = np.random.default_rng(8)
    u8p, i32p = ctypes.POINTER(ctypes.c_uint8), ctypes.POINTER(ctypes.c_int32)
    n = 0
    for it in range(4000):
        l1, l2 = int(rng.integers(1, 37)), int(rng.integers(1, 37))
        X = int(rng.integers(0, min(l1, l2)))
        P = int(rng.choice([0, 0, -1, -4, 3, -2000000000]))
        M = np.ascontiguousarray(mats[it % len(mats)], dtype=np.int32)
        a = rng.integers(0, 24, l1).astype(np.uint8)
        b = rng.integers(0, 24, l2).astype(np.uint8)
        want, _ = O.score_with_shift(a, b, M, X, P)
        got = shim.shim_pair_score(a.ctypes.data_as(u8p), l1, b.ctypes.data_as(u8p), l2, M.ctypes.data_as(i32p), X, P)
        assert got == want, (l1, l2, X, P, it % len(mats))
        # position-major copies with strides, as the generic kernel stages them in shared memory
        s1, s2 = int(rng.integers(1, 5)), int(rng.integers(1, 5))
        a2 = np.zeros(l1 * s1, np.uint8); a2[::s1] = a
        b2 = np.zeros(l2 * s2, np.uint8); b2[::s2] = b
        got = shim.shim_pair_score_strided(a2.ctypes.data_as(u8p), s1, l1, b2.ctypes.data_as(u8p), s2, l2, M.ctypes.data_as(i32p), X, P)
        assert got == want
        assert shim.shim_pair_cells(l1, l2, X) == O.pair_cells(l1, l2, X)
        n += 1
    assert n == 4000
    # the reference's argument roles: equal lengths make the SECOND sequence the sliding one (ShiftedScorer.java:51-57)
    asym = blosum62.copy()
    asym[0, 1] += 7
    a, b = np.array([0, 1, 2, 3], np.uint8), np.array([1, 0, 3, 2], np.uint8)
    M = np.ascontiguousarray(asym, dtype=np.int32)
    for x, y in ((a, b), (b, a)):
        assert shim.shim_pair_score(x.ctypes.data_as(u8p), 4, y.ctypes.data_as(u8p), 4, M.ctypes.data_as(i32p), 1, 0) == O.score_with_shift(x, y, M, 1, 0)[0]


def test_device_partner_key_and_cluster_order(shim):
    """bigger hmk_key_make == preferred partner (score desc, then rank under (abundance desc, id asc) asc); hmk_consider ==
    NearestClusterRunner's order (score desc, size desc, id asc; ClinkageSequenceClusterer.java:258-293), whatever the
    order the candidates arrive in"""
    rng = np.random.default_rng(9)
    scores = [-(2 ** 31), -(2 ** 31) + 1, -5, -1, 0, 1, 19, 20, 2 ** 31 - 1]
    ranks = [0, 1, 2, 1000, 2 ** 31, 2 ** 32 - 1]
    keys = [(s, r, shim.shim_key_make(s, r)) for s in scores for r in ranks]
    for s, r, k in keys:
        assert shim.shim_key_score(k) == s and shim.shim_key_rank(k) == r
    by_key = [(s, r) for s, r, k in sorted(keys, key=lambda t: -t[2])]
    assert by_key == sorted([(s, r) for s, r, _ in keys], key=lambda t: (-t[0], t[1]))
    assert shim.shim_wadd(2 ** 31 - 1, 1) == -(2 ** 31) and shim.shim_wmul(65536, 65536) == 0 and shim.shim_wmul(-3, 5) == -15
    i32p = ctypes.POINTER(ctypes.c_int32)
    for it in range(300):
        n = int(rng.integers(1, 12))
        sc = rng.integers(18, 22, n).astype(np.int32)
        sz = rng.integers(1, 4, n).astype(np.int32)
        fid = rng.permutation(50)[:n].astype(np.int32)
        want = min(range(n), key=lambda i: (-int(sc[i]), -int(sz[i]), int(fid[i])))
        assert shim.shim_best_cluster(n, sc.ctypes.data_as(i32p), sz.ctypes.data_as(i32p), fid.ctypes.data_as(i32p)) == want
    assert shim.shim_best_cluster(0, None, None, None) == -1


def test_cpp_host_files_from_the_oracle_clinkage_clustering(tmp_path, blosum62):
    """the `clinkage` mode of the C++ driver around the oracle's exact complete-linkage clustering: input order (no sort),
    Cluster ids 1 .. 2n+1, list order of the emulated HashSet -- files against the oracle's writers"""
    import subprocess
    from oracle import pyref_writers as W
    exe = _writers_harness(tmp_path)
    d = synth.generate(400, 9, 12, seed=5)
    strs = synth.to_strings(d["residues"], d["offsets"])
    rng = np.random.default_rng(6)
    labs = ["x", "yy"]
    fa = tmp_path / "in.fa"
    with open(fa, "w") as f:
        for k, i in enumerate(rng.permutation(len(strs))):
            f.write(f">r{k}|{int(rng.integers(1, 30))}|{labs[k % 2]}\n{strs[i]}\n")
    seqs = hb.load_unique_sequences_from_fasta(str(fa))
    labels = hb.get_sorted_labels(seqs)
    res, offs, ab = hb.pack_sequences(seqs)
    T, X = hb.set_clinkage_threshold(seqs), hb.get_max_shift(seqs)
    R = O.clinkage_cluster(res, offs, ab, blosum62, T, X, 0)
    assert R.status == 0 and int(R.cluster_id.max()) > len(seqs)          # merged clusters carry ids beyond n
    with open(tmp_path / "result.txt", "w") as f:
        f.write(f"{len(seqs)} {len(R.result_order)}\n")
        for a in (R.cluster_id, R.member_rank, R.result_order):
            f.write(" ".join(str(int(v)) for v in a) + "\n")
    out = tmp_path / "out"
    out.mkdir()
    r = subprocess.run([exe, str(fa), "input", "0", str(tmp_path / "result.txt"), str(out) + "/"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    n_multi = int((np.bincount(R.cluster_id) > 1).sum())
    clusters = hb.rebuild_clusters(seqs, hb.GreedyResult(R.cluster_id, R.member_rank, R.result_order, n_multi, {}))
    tup = lambda s: (s.get_sequence_string(), dict(s.labels_map))
    ct = [(c.get_id(), [tup(s) for s in c.get_sequences()]) for c in clusters]
    assert (out / "initial_clusters_sequences.tsv").read_text() == W.cluster_sequences_tsv(ct, labels)
    assert (out / "initial_clusters_sequences_original_order.tsv").read_text() == W.cluster_sequences_tsv_ordered(ct, labels, [tup(s) for s in seqs])
    assert (out / "initial_clusters.tsv").read_text() == W.clusters_tsv(ct, labels)


def test_cpp_driver_clinkage_mode_prepares_like_the_reference(tmp_path):
    """hammock_greedy clinkage: sequences stay in input order, threshold = setClinkageThreshold (Hammock.java:449-455, 1415-1419)"""
    p = tmp_path / "in.fa"
    p.write_text(MULTI)
    head, rows = _dump(tmp_path, ["clinkage", "-i", str(p), "-R", "size"])
    seqs = hb.load_unique_sequences_from_fasta(str(p))
    assert int(head["threshold"][0]) == hb.set_clinkage_threshold(seqs) and int(head["max_shift"][0]) == hb.get_max_shift(seqs)
    assert rows == [(s.get_sequence_string(), str(s.size())) for s in seqs]


def _driver(args):
    import subprocess
    exe = hb_build.build_host()
    return subprocess.run([exe, "greedy"] + args + ["--dump-prepared"], capture_output=True, text=True)


def test_cpp_loader_error_paths_match_the_python_host(tmp_path):
    """the rewritten C++ loader fails where the reference does (FileIOManager.java:159-216, UniqueSequence.java:51-54):
    same cases as the Python host and the oracle loader, exit code 1 and the reference's message"""
    p = tmp_path / "in.fa"
    cases = {">x|0|l\nACD\n": "count lower than 1", "ACD\n": "Incorrect fasta format", ">x|1\nACDJ\n": "not a valid letter",
             ">x|abc\nACD\n": "NumberFormatException", ">x|1\n": None, "": "Incorrect fasta format", ">x|99999999999|l\nACD\n": "NumberFormatException",
             ">x|-3|l\nACD\n": "count lower than 1"}
    for text, msg in cases.items():
        p.write_text(text)
        r = _driver(["-i", str(p)])
        try:
            seqs = hb.load_unique_sequences_from_fasta(str(p))
            py_ok = True
        except hb.FileFormatException:
            py_ok = False
        if msg is None:            # a header without a sequence line: one empty sequence in both hosts (then "Shift too big" territory)
            assert py_ok == (r.returncode == 0), (text, r.stderr)
            continue
        assert not py_ok and r.returncode == 1 and msg in r.stderr, (text, r.returncode, r.stderr)


def test_cpp_loader_odd_headers_tab_format_and_label_filter(tmp_path):
    text = (">a|3|lab1||\nWVTAPRSLPVLP\n"            # trailing empty fields are dropped by String.split
            ">b|0x10||x\nGSWVVDISNVED  \n"          # hex count, EMPTY label (a fourth field keeps the third)
            ">c| 7 |lab1\n  wvtaprslpvlp\n"         # count is trimmed; lower case is a different map key, same sequence
            ">d|010|lab2\nGSWVVDISNVED\n"           # Integer.decode: leading zero = octal 8
            ">e|+5|lab2\nACDEFGHIKLMN\r\n")
    p = tmp_path / "in.fa"
    p.write_text(text)
    seqs = hb.load_unique_sequences_from_fasta(str(p))
    assert [(s.get_sequence_string(), s.labels_map) for s in seqs] == [
        ("WVTAPRSLPVLP", {"lab1": 3}), ("GSWVVDISNVED", {"": 16, "lab2": 8}), ("WVTAPRSLPVLP", {"lab1": 7}), ("ACDEFGHIKLMN", {"lab2": 5})]
    r = _driver(["-i", str(p), "-R", "input"])
    assert r.returncode == 0, r.stderr
    out = r.stdout.splitlines()
    assert out[3].split("\t")[1:] == hb.get_sorted_labels(seqs)
    assert [tuple(l.split("\t")) for l in out[4:]] == [(s.get_sequence_string(), str(s.size())) for s in seqs]
    # -l: only sequences carrying one of the labels, with only those labels (Hammock.java:1661-1675)
    r = _driver(["-i", str(p), "-R", "input", "-l", "lab2"])
    assert [tuple(l.split("\t")) for l in r.stdout.splitlines()[4:]] == [("GSWVVDISNVED", "8"), ("ACDEFGHIKLMN", "5")]
    # tab format (FileIOManager.java:227-255): zero counts are dropped, no de-duplication
    t = tmp_path / "in.tsv"
    t.write_text("sequence\tl1\tl2\nWVTAPRSLPVLP\t3\t0\nGSWVVDISNVED\t0x2\t5\nwvtaprslpvlp\t0\t1\n")
    seqs = hb.load_unique_sequences_from_table(str(t))
    r = _driver(["-i", str(t), "-f", "tab", "-R", "size"])
    assert r.returncode == 0, r.stderr
    ordered = hb.sort_sequences(seqs, "size", hb.get_sorted_labels(seqs))
    assert [tuple(l.split("\t")) for l in r.stdout.splitlines()[4:]] == [(s.get_sequence_string(), str(s.size())) for s in ordered]
    assert r.stdout.splitlines()[3].split("\t")[1:] == hb.get_sorted_labels(seqs)


def test_struct_layouts_agree_between_header_ctypes_and_java(tmp_path):
    """the three structs of include/hammock_b200.h as the C compiler lays them out == the ctypes mirrors in _lib.py ==
    the byte offsets the Java (FFM) bindings write to"""
    import subprocess
    hdr = open(os.path.join(ROOT, "include", "hammock_b200.h")).read()
    structs = {}
    for body, name in re.findall(r"typedef struct \{(.*?)\}\s*(hmk_\w+);", hdr, flags=re.S):
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        fields = []
        for decl in body.split(";"):
            decl = decl.strip()
            if not decl:
                continue
            names = [re.sub(r"[\s\*]", "", x).split("[")[0] for x in decl.split(",")]
            names[0] = re.split(r"[\s\*]+", decl.split(",")[0].strip())[-1]
            fields += names
        structs[name] = fields
    assert set(structs) >= {"hmk_greedy_in", "hmk_greedy_out", "hmk_stats"}
    src = '#include <stddef.h>\n#include <stdio.h>\n#include "hammock_b200.h"\nint main(void) {\n'
    for name, fields in structs.items():
        src += f'  printf("{name} size %zu\\n", sizeof({name}));\n'
        for f in fields:
            src += f'  printf("{name} {f} %zu\\n", offsetof({name}, {f}));\n'
    src += "  return 0;\n}\n"
    (tmp_path / "o.c").write_text(src)
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(tmp_path / "o"), str(tmp_path / "o.c")])
    off = {}
    for line in subprocess.run([str(tmp_path / "o")], capture_output=True, text=True, check=True).stdout.splitlines():
        s, f, v = line.split()
        off[(s, f)] = int(v)
    for cname, T in (("hmk_greedy_in", _lib.GreedyIn), ("hmk_greedy_out", _lib.GreedyOut), ("hmk_stats", _lib.Stats)):
        assert [f for f, _ in T._fields_] == structs[cname], cname
        assert ctypes.sizeof(T) == off[(cname, "size")], cname
        for f, _ in T._fields_:
            assert getattr(T, f).offset == off[(cname, f)], (cname, f)
    # Java: in.set(<layout>, <offset>, <java name>) / out.set(...) / out.get(JAVA_INT, <offset>)
    jmap = {"n": "n", "residues": "residues", "offsets": "offsets", "abundance": "abundance", "matrix": "matrix", "threshold": "threshold",
            "maxShift": "max_shift", "shiftPenalty": "shift_penalty", "maxClusters": "max_clusters", "0": "max_clusters",
            "clusterId": "cluster_id", "memberRank": "member_rank", "resultOrder": "result_order"}
    jdir = os.path.join(ROOT, "java", "cz", "krejciadam", "hammock")
    checked = 0
    for fn in os.listdir(jdir):
        txt = open(os.path.join(jdir, fn)).read()
        for var, o, val in re.findall(r"\b(in|out)\.set\(\w+, (\d+), (\w+)\)", txt):
            sname = "hmk_greedy_in" if var == "in" else "hmk_greedy_out"
            assert off[(sname, jmap[val])] == int(o), (fn, var, o, val)
            checked += 1
        assert re.search(r"nResult = out\.get\(JAVA_INT, %d\)" % off[("hmk_greedy_out", "n_result")], txt), fn
        m = re.search(r'step " \+ out\.get\(JAVA_INT, (\d+)\)', txt)
        if m:
            assert int(m.group(1)) == off[("hmk_greedy_out", "error_step")]
    assert checked >= 24


def test_reference_arm_of_the_bench_runs_on_the_cpu():
    """`bench.py --impl reference` (the arm the driver runs first, on host cores only) prints one JSON line with the keys of
    the contract -- here on a small debug-sized set so that it takes seconds"""
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--n", "20000"],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "greedy_cluster_unique_seqs_per_sec" and d["unit"] == "seq/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "seq/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["extrapolated"] is True and "workload" in d["config"]


def test_bench_dump_outputs_of_the_reference_arm(tmp_path):
    """`--dump-outputs DIR` writes the clustering of the last timed step as float64 .npy files: here the bounded oracle
    sample of the reference arm, which must equal the same bounded oracle run on the same seeded input"""
    import subprocess
    import sys
    import bench
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "0",
                        "--n", "20000", "--dump-outputs", str(tmp_path / "dump")], capture_output=True, text=True, cwd=ROOT,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d, M, (T, X, P, K) = bench.workload(20000)
    R = O.greedy_cluster(d["residues"], d["offsets"], d["abundance"], M, T, X, P, K, max_p1_steps=500, max_p2_queries=5000)
    assert R.status == 0
    assert sorted(os.listdir(tmp_path / "dump")) == ["cluster_id.npy", "member_rank.npy", "n_multi.npy", "result_order.npy"]
    got = {k: np.load(tmp_path / "dump" / f"{k}.npy") for k in ("cluster_id", "member_rank", "result_order", "n_multi")}
    assert all(a.dtype == np.float64 for a in got.values())
    assert (got["cluster_id"] == R.cluster_id).all() and (got["member_rank"] == R.member_rank).all()
    assert (got["result_order"] == R.result_order).all() and got["n_multi"].tolist() == [R.n_multi]


def test_bench_dump_outputs_samples_what_exceeds_the_limit(tmp_path):
    """outputs above the size limit are replaced by a fixed, seeded sample with its positions; small ones stay whole"""
    import bench
    rng = np.random.default_rng(1)
    r = hb.GreedyResult(rng.integers(0, 1 << 30, 5000).astype(np.int32), rng.integers(0, 9, 5000).astype(np.int32),
                        np.arange(300, dtype=np.int32), 7, {})
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), r, limit=16 * 4 * 1000)
    for k, a in (("cluster_id", r.cluster_id), ("member_rank", r.member_rank)):
        idx = np.load(tmp_path / "a" / f"{k}_index.npy")
        v = np.load(tmp_path / "a" / f"{k}.npy")
        assert len(idx) == len(v) == 1000 and len(np.unique(idx)) == 1000
        assert (v == a[idx.astype(np.int64)]).all()
        assert (idx == np.load(tmp_path / "b" / f"{k}_index.npy")).all()
    assert (np.load(tmp_path / "a" / "result_order.npy") == r.result_order).all()
    assert not os.path.exists(tmp_path / "a" / "result_order_index.npy")
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 16 * 4 * 1000 + 8 * 128
