"""Host-side mirror of the reference's interface for the greedy initial clustering path.

Same names, argument meaning and error behaviour as the Java classes it stands in for
(reference: /root/reference/src/cz/krejciadam/hammock/, cited per item), so that the parity
tests read like tests of the reference.  All scoring and clustering happens in
libhammock_b200.so (CUDA, sm_100a) through the C ABI of include/hammock_b200.h; this module
only parses, orders, packs and rebuilds objects.  No CPU fallback exists.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Iterable, List, Optional, Sequence

import numpy as np

from . import _lib

ALPHABET = "ARNDCQEGHILKMFPSTWYVBZX*"  # UniqueSequence.java:23-26
_CODE = {ch: i for i, ch in enumerate(ALPHABET)}


# ---------------------------------------------------------------- exceptions (reference names)
class HammockException(Exception):
    """HammockException.java"""


class DataException(HammockException):
    """DataException.java"""


class FileFormatException(HammockException):
    """FileFormatException.java"""


class NullClusterError(HammockException):
    """The NullPointerException the reference throws at LimitedGreedySequenceClusterer.java:104/108
    when a query has neither a cluster nor a partner while one of the two candidate collections
    is empty (SURVEY.md 3.2).  `step` is the phase-1 step index."""

    def __init__(self, step):
        super().__init__(f"NullPointerException at phase-1 step {step} (nearest-cluster object without a cluster)")
        self.step = step


class CudaError(HammockException):
    """CUDA / NCCL failure inside libhammock_b200 (status 4); there is no CPU fallback."""


# ---------------------------------------------------------------- data model
class UniqueSequence:
    """UniqueSequence.java:19-57, 81-109."""

    __slots__ = ("sequence", "labels_map")

    def __init__(self, sequence: str, labels_map: Optional[Dict[str, int]] = None):
        up = sequence.upper()                                   # :49
        codes = np.empty(len(up), dtype=np.uint8)
        for i, ch in enumerate(up):
            k = _CODE.get(ch)
            if k is None:                                       # :52-54
                raise FileFormatException(
                    f"Error, character {sequence[i]} is not a valid letter from the amino acid alphabet code.")
            codes[i] = k
        self.sequence = codes
        self.labels_map = {"no_label": 1} if labels_map is None else labels_map   # :65-68

    def size(self) -> int:                                      # :81-88 (Java int)
        s = 0
        for v in self.labels_map.values():
            s = _i32(s + v)
        return s

    def get_sequence(self) -> np.ndarray:
        return self.sequence

    def get_sequence_string(self) -> str:                       # :103-109
        return "".join(ALPHABET[c] for c in self.sequence)

    def get_labels_map(self) -> Dict[str, int]:
        return self.labels_map

    def __eq__(self, other):                                    # :143-153
        return isinstance(other, UniqueSequence) and np.array_equal(self.sequence, other.sequence)

    def __hash__(self):
        return hash(self.sequence.tobytes())

    def __repr__(self):
        return f"UniqueSequence({self.get_sequence_string()!r}, size={self.size()})"


def _i32(x: int) -> int:
    return ((int(x) + 2 ** 31) % 2 ** 32) - 2 ** 31


class Cluster:
    """Cluster.java:21-74, 113-123, 156-158."""

    def __init__(self, sequences: Iterable[UniqueSequence], id: int):
        self._sequences: List[UniqueSequence] = list(sequences)
        self._id = id
        self._size = 0
        for s in self._sequences:
            self._size = _i32(self._size + s.size())

    def insert(self, sequence: UniqueSequence) -> None:         # :50-63
        if sequence in self._sequences:
            raise DataException(
                f"Trying to insert unique sequence {sequence.get_sequence_string()} into cluster "
                f"{self._id}, which already contains this sequence. ")
        self._sequences.append(sequence)
        self._size = _i32(self._size + sequence.size())

    def insert_all(self, sequences: Iterable[UniqueSequence]) -> None:   # :70-74
        for s in sequences:
            self.insert(s)

    def get_unique_size(self) -> int:
        return len(self._sequences)

    def get_sequences(self) -> List[UniqueSequence]:
        return self._sequences

    def get_id(self) -> int:
        return self._id

    def size(self) -> int:
        return self._size

    def __eq__(self, other):                                    # :185-195 identity by id
        return isinstance(other, Cluster) and other._id == self._id

    def __hash__(self):
        return 79 * 7 + self._id                                # :179-183

    def __repr__(self):
        return f"Cluster(id={self._id}, unique={len(self._sequences)}, size={self._size})"


# ---------------------------------------------------------------- loaders
_JAVA_WS = " \t\n\x0b\f\r"


def load_scoring_matrix(path: str) -> np.ndarray:
    """FileIOManager.loadScoringMatrix (FileIOManager.java:46-81), quirks included: rows in file
    order with no label check, lines starting with '#', ' ' or TAB skipped, every other line
    (also an empty one) needs exactly 25 whitespace-separated tokens, more than 24 rows is an
    error, fewer leave zeros."""
    M = np.zeros((24, 24), dtype=np.int32)
    row = 0
    with open(path, "r", newline="") as f:
        text = f.read()
    lines = text.split("\n")
    if lines and lines[-1] == "":
        lines.pop()
    for line in lines:
        if line.endswith("\r"):
            line = line[:-1]
        if line[:1] in ("#", " ", "\t"):
            continue
        toks = _java_split_ws(line)
        if len(toks) != 25:
            raise FileFormatException(
                f"Error in scoring matrix file: {path}. Scoring matrix should always have 24 columns "
                "(plus 1 column describing AAs).")
        if row >= 24:
            raise FileFormatException(
                f"Error in scoring matrix file: {path}. Scoring matrix should always have 24 rows "
                "(plus 1 column describing AAs).")
        for c in range(1, 25):
            M[row, c - 1] = _parse_int(toks[c])
        row += 1
    return M


def _java_split_ws(line: str) -> List[str]:
    """String.split("\\\\s+"): keeps a leading empty token, drops trailing empty ones."""
    if line == "":
        return [""]
    toks, cur, i, n = [], [], 0, len(line)
    if line[0] in _JAVA_WS:
        toks.append("")
    while i < n:
        while i < n and line[i] in _JAVA_WS:
            i += 1
        if i >= n:
            break
        j = i
        while j < n and line[j] not in _JAVA_WS:
            j += 1
        toks.append(line[i:j])
        i = j
    return toks


def _parse_int(tok: str) -> int:
    """Integer.parseInt"""
    body = tok[1:] if tok[:1] in "+-" else tok
    if not body or not body.isascii() or not body.isdigit():
        raise FileFormatException(f"NumberFormatException: For input string: \"{tok}\"")
    v = int(tok)
    if not -2 ** 31 <= v < 2 ** 31:
        raise FileFormatException(f"NumberFormatException: For input string: \"{tok}\"")
    return v


def _decode_int(tok: str) -> int:
    """Integer.decode"""
    s, neg = tok, False
    if s[:1] == "-":
        neg, s = True, s[1:]
    elif s[:1] == "+":
        s = s[1:]
    radix = 10
    if s[:2] in ("0x", "0X"):
        radix, s = 16, s[2:]
    elif s[:1] == "#":
        radix, s = 16, s[1:]
    elif len(s) > 1 and s[0] == "0":
        radix, s = 8, s[1:]
    try:
        if not s or s[0] in "+-":
            raise ValueError
        v = int(s, radix)
    except ValueError:
        raise FileFormatException(f"NumberFormatException: For input string: \"{tok}\"") from None
    v = -v if neg else v
    if not -2 ** 31 <= v < 2 ** 31:
        raise FileFormatException(f"NumberFormatException: For input string: \"{tok}\"")
    return v


def _java_trim(s: str) -> str:
    i, j = 0, len(s)
    while i < j and s[i] <= " ":
        i += 1
    while j > i and s[j - 1] <= " ":
        j -= 1
    return s[i:j]


def load_unique_sequences_from_fasta(path: str) -> List[UniqueSequence]:
    """FileIOManager.loadUniqueSequencesFromFasta (FileIOManager.java:159-216): headers
    `>id|count|label`, multi-line sequences concatenated, repeated sequences accumulate per label,
    first-occurrence order, the map key is the raw (case-sensitive) string."""
    seq_map: Dict[str, Dict[str, int]] = {}
    sequence, label, count = "", None, None

    def flush():
        m = seq_map.get(sequence)
        if m is None:
            seq_map[sequence] = {label: count}
        else:
            m[label] = _i32(m.get(label, 0) + count)

    with open(path, "r", newline="") as f:
        text = f.read()
    lines = text.split("\n")
    if lines and lines[-1] == "":
        lines.pop()
    for line in lines:
        if line.endswith("\r"):
            line = line[:-1]
        if line.startswith(">"):
            if len(sequence) > 0:
                flush()
                sequence = ""
            parts = _java_trim(line)[1:].split("|")
            while len(parts) > 1 and parts[-1] == "":
                parts.pop()
            if len(parts) >= 2:
                count = _decode_int(_java_trim(parts[1]))
                if count < 1:
                    raise FileFormatException(
                        "Error while loading input file. Fasta header defines sequence count lower than 1.")
            else:
                count = 1
            label = parts[2] if len(parts) >= 3 else "no_label"
        else:
            if label is None or count is None:
                raise FileFormatException("Error. Incorrect fasta format. Maybe header or sequence line missing?")
            sequence += _java_trim(line)
    if label is None:
        raise FileFormatException("Error. Incorrect fasta format. Maybe header or sequence line missing?")
    flush()
    return [UniqueSequence(k, v) for k, v in seq_map.items()]


def load_unique_sequences_from_table(path: str, separator: str = "\t") -> List[UniqueSequence]:
    """FileIOManager.loadUniqueSequencesFromTable (FileIOManager.java:227-255)."""
    out = []
    with open(path, "r") as f:
        header = f.readline().rstrip("\r\n").split(separator)
        labels = header[1:]
        for line in f:
            parts = line.rstrip("\r\n").split(separator)
            m = {}
            for i, tok in enumerate(parts[1:]):
                v = _decode_int(tok)
                if v != 0:
                    m[labels[i]] = v
            out.append(UniqueSequence(parts[0], m))
    return out


# ---------------------------------------------------------------- ordering + defaults
class _JavaRandom:
    """java.util.Random (LCG), enough for Collections.shuffle."""

    def __init__(self, seed: int):
        self.seed = (seed ^ 0x5DEECE66D) & ((1 << 48) - 1)

    def _next(self, bits: int) -> int:
        self.seed = (self.seed * 0x5DEECE66D + 0xB) & ((1 << 48) - 1)
        return _i32(self.seed >> (48 - bits))

    def next_int(self, bound: int) -> int:
        r = self._next(31)
        m = bound - 1
        if bound & m == 0:
            return _i32((bound * r) >> 31)
        u = r
        r = u % bound
        while _i32(u - r + m) < 0:
            u = self._next(31)
            r = u % bound
        return r


def sort_sequences(sequences: List[UniqueSequence], order: str = "size", labels: Optional[Sequence[str]] = None,
                   seed: int = 42) -> List[UniqueSequence]:
    """UniqueSequence.sortSequences (UniqueSequence.java:176-203): stable sorts with reversed
    comparators.  "random" assumes a fresh java.util.Random(seed) (Hammock.java:1252)."""
    def size_alpha(seqs):
        return sorted(seqs, key=lambda s: (s.size(), s.get_sequence_string()), reverse=True)

    if order == "size":
        return size_alpha(sequences)
    if order == "alphabetic":
        return sorted(sequences, key=lambda s: s.get_sequence_string(), reverse=True)
    if order == "random":                                        # Collections.shuffle(list, rnd)
        out = list(sequences)
        rnd = _JavaRandom(seed)
        for i in range(len(out), 1, -1):
            j = rnd.next_int(i)
            out[i - 1], out[j] = out[j], out[i - 1]
        return out
    if order == "input":
        return list(sequences)
    if labels is None or order not in labels:
        raise DataException("Incorrect sequence order defined. Use one of: size, alphabetic, random, input, or a label")
    return sorted(size_alpha(sequences), key=lambda s: s.labels_map.get(order, 0), reverse=True)


def _java_round(x: float) -> int:
    import math
    return int(math.floor(x + 0.5))


def get_mean_sequence_length(sequences) -> float:              # Hammock.java:1554-1563
    return sum(len(s.sequence) for s in sequences) / len(sequences)


def set_greedy_threshold(sequences) -> int:                    # Hammock.java:1409-1413
    return _java_round(get_mean_sequence_length(sequences) * 1.7)


def check_max_shift(sequences, max_shift: int) -> int:         # Hammock.java:1421-1427
    return min(max_shift, min(len(s.sequence) for s in sequences) - 1)


def get_max_shift(sequences) -> int:                           # Hammock.java:1429-1434
    return check_max_shift(sequences, _java_round(get_mean_sequence_length(sequences) / 4))


def initial_clusters_limit(sequences) -> int:                  # Hammock.java:398-401
    return _java_round(len(sequences) * 0.025)


# ---------------------------------------------------------------- labels + result files
def _java_string_hash(s: str) -> int:
    h = 0
    for ch in s:                          # String.hashCode (labels are ASCII here)
        h = (31 * h + ord(ch)) & 0xFFFFFFFF
    return h


def java_hashmap_order(keys: Sequence[str]) -> List[str]:
    """Iteration order of a java.util.HashMap<String, ?> (Java 8+: tail insertion, order-preserving resize,
    bins assumed not to treeify) that received `keys` in this order."""
    cap = 16
    while len(keys) > cap * 3 // 4:
        cap *= 2
    bins: List[List[str]] = [[] for _ in range(cap)]
    for k in keys:
        h = _java_string_hash(k)
        h ^= h >> 16
        bins[h & (cap - 1)].append(k)
    return [k for b in bins for k in b]


def get_sorted_labels(sequences: Sequence[UniqueSequence]) -> List[str]:
    """Hammock.getSortedLabels (Hammock.java:1586-1605): TreeMap with ValueComparator (FileIOManager.java:1464-1480,
    never returns 0) filled from a HashMap -> count descending, equal counts in reverse HashMap iteration order."""
    cnt: Dict[str, int] = {}
    for s in sequences:
        for k, v in s.labels_map.items():
            cnt[k] = _i32(cnt.get(k, 0) + v)
    out: List[str] = []
    for k in java_hashmap_order(list(cnt.keys())):
        pos = 0
        while pos < len(out) and cnt[out[pos]] > cnt[k]:
            pos += 1
        out.insert(pos, k)
    return out


def _clusters_largest_first(clusters: Sequence[Cluster]) -> List[Cluster]:
    """Collections.sort(list, reverseOrder()) with Cluster.compareTo (Cluster.java:197-204): size desc, id desc"""
    return sorted(clusters, key=lambda c: (c.size(), c.get_id()), reverse=True)


def _row(cluster_id, s: UniqueSequence, alignment: str, labels) -> str:
    return "\t".join([str(cluster_id), s.get_sequence_string(), alignment, str(s.size())] +
                     [str(s.labels_map.get(lab, 0)) for lab in labels]) + "\n"


def save_cluster_sequences_to_csv(clusters: Sequence[Cluster], path: str, labels: Sequence[str]) -> None:
    """FileIOManager.saveClusterSequencesToCsv (FileIOManager.java:398-404, 594-638).  The alignment column is the
    sequence for one-member clusters and "NA" for multi-member clusters (the reference fills it from the Clustal-Omega
    MSA it builds after the greedy stage, Hammock.java:414-426 -- outside this path; `cluster` mode accepts NA)."""
    with open(path, "w") as w:
        w.write("\t".join(["cluster_id", "sequence", "alignment", "sum"] + list(labels)) + "\n")
        for c in _clusters_largest_first(clusters):
            members = sorted(c.get_sequences(), key=lambda s: (s.size(), s.get_sequence_string()), reverse=True)
            for s in members:
                w.write(_row(c.get_id(), s, s.get_sequence_string() if len(members) == 1 else "NA", labels))


def save_cluster_sequences_to_csv_ordered(clusters: Sequence[Cluster], path: str, labels: Sequence[str],
                                          ordered_sequences: Sequence[UniqueSequence]) -> None:
    """FileIOManager.saveClusterSequencesToCsvOrdered (FileIOManager.java:371-374)"""
    of = {}
    for c in clusters:
        for s in c.get_sequences():
            of[s.get_sequence_string()] = c
    with open(path, "w") as w:
        w.write("\t".join(["cluster_id", "sequence", "alignment", "sum"] + list(labels)) + "\n")
        for s in ordered_sequences:
            c = of.get(s.get_sequence_string())
            if c is None:
                w.write(_row("NA", s, "NA", labels))
            else:
                w.write(_row(c.get_id(), s, s.get_sequence_string() if c.get_unique_size() == 1 else "NA", labels))


def save_clusters_to_csv(clusters: Sequence[Cluster], path: str, labels: Sequence[str]) -> None:
    """FileIOManager.SaveClustersToCsv (FileIOManager.java:649-676): main_sequence = most abundant member, ties
    alphabetically first."""
    with open(path, "w") as w:
        w.write("\t".join(["cluster_id", "main_sequence", "sum"] + list(labels)) + "\n")
        for c in _clusters_largest_first(clusters):
            seqs = c.get_sequences()
            top = max(s.size() for s in seqs)
            main = min(s.get_sequence_string() for s in seqs if s.size() == top)
            sums = []
            for lab in labels:
                t = 0
                for s in seqs:
                    t = _i32(t + s.labels_map.get(lab, 0))
                sums.append(str(t))
            w.write("\t".join([str(c.get_id()), main, str(c.size())] + sums) + "\n")


def save_input_statistics(sequences: Sequence[UniqueSequence], labels: Sequence[str], path: str) -> None:
    """FileIOManager.saveInputStatistics (FileIOManager.java:709-729)"""
    with open(path, "w") as w:
        w.write("".join("\t" + lab for lab in labels) + "\n")
        w.write("total_count" + "".join("\t" + str(_i32(sum(s.labels_map.get(lab, 0) for s in sequences))) for lab in labels) + "\n")
        w.write("unique_count" + "".join("\t" + str(sum(1 for s in sequences if lab in s.labels_map)) for lab in labels))


# ---------------------------------------------------------------- packing + C ABI
def shard_range(n: int, world: int, rank: int):
    """Contiguous share [lo, hi) of n work items for `rank` of `world` (same split as the library's
    hmk_shard_range: sizes differ by at most one)."""
    lo = (n * rank) // world
    hi = (n * (rank + 1)) // world
    return lo, hi


def pack_sequences(sequences: Sequence[UniqueSequence]):
    n = len(sequences)
    offs = np.zeros(n + 1, dtype=np.int32)
    if n:
        offs[1:] = np.cumsum([len(s.sequence) for s in sequences], dtype=np.int64)
    res = np.concatenate([s.sequence for s in sequences]).astype(np.uint8) if n else np.zeros(0, np.uint8)
    ab = np.array([s.size() for s in sequences], dtype=np.int32)
    return np.ascontiguousarray(res), offs, ab


def _ptr(a: np.ndarray, t):
    return a.ctypes.data_as(C.POINTER(t))


def _raise_status(rc: int, err: bytes, step: int = -1):
    msg = err.decode(errors="replace")
    if rc == _lib.STATUS_SHIFT_TOO_BIG:
        raise DataException(msg or "Shift too big")
    if rc == _lib.STATUS_NULL_CLUSTER:
        raise NullClusterError(step)
    if rc == _lib.STATUS_BAD_RESIDUE:
        raise FileFormatException(msg)
    if rc == _lib.STATUS_BAD_ARG:
        raise ValueError(msg or "bad argument")
    raise CudaError(msg or f"status {rc}")


# one score-graph edge, laid out as hmk_graph_edge
EDGE_DTYPE = np.dtype([("seq", "<i4"), ("partner", "<i4"), ("score", "<i4"), ("shift", "<i4")])


class GreedyResult:
    def __init__(self, cluster_id, member_rank, result_order, n_multi, stats):
        self.cluster_id, self.member_rank, self.result_order = cluster_id, member_rank, result_order
        self.n_multi, self.stats = n_multi, stats


class GreedyContext:
    """Handle API (hmk_create / upload / run / download): keeps sequences resident on the GPU."""

    def __init__(self, device: int = 0, **options):
        self._L = _lib.load()
        self._h = C.c_void_p()
        err = C.create_string_buffer(512)
        rc = self._L.hmk_create(C.byref(self._h), device, err, 512)
        if rc:
            _raise_status(rc, err.value)
        self._keep = None
        self.n = 0
        self._kb = 8        # option kb (the engine's default): row length of bulk_probe's key lists
        self._capq = 256    # option capq (the engine's default): rows of batch_probe's candidate arrays
        for k, v in options.items():
            self.set_option(k, v)

    def set_option(self, name: str, value: int):
        if self._L.hmk_set_option(self._h, name.encode(), int(value)):
            raise ValueError(f"unknown option {name}")
        if name == "kb":
            self._kb = int(value)
        if name == "capq":
            self._capq = int(value)

    def close(self):
        if self._h:
            self._L.hmk_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def upload(self, residues, offsets, abundance, matrix, threshold, max_shift, shift_penalty, max_clusters):
        residues = np.ascontiguousarray(residues, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.int32)
        abundance = np.ascontiguousarray(abundance, dtype=np.int32)
        matrix = np.ascontiguousarray(matrix, dtype=np.int32).reshape(-1)
        if matrix.size != 576:
            raise ValueError("matrix must be 24x24")
        self._keep = (residues, offsets, abundance, matrix)
        self.n = len(abundance)
        gin = _lib.GreedyIn(self.n, _ptr(residues, C.c_uint8), _ptr(offsets, C.c_int32), _ptr(abundance, C.c_int32),
                            _ptr(matrix, C.c_int32), int(threshold), int(max_shift), int(shift_penalty),
                            int(max_clusters))
        err = C.create_string_buffer(512)
        rc = self._L.hmk_upload(self._h, C.byref(gin), err, 512)
        if rc:
            _raise_status(rc, err.value)

    def run(self):
        err = C.create_string_buffer(512)
        rc = self._L.hmk_run(self._h, err, 512)
        if rc:
            _raise_status(rc, err.value, self.stats().get("error_step", -1))

    def run_status(self):
        """Like run() but returns (status, phase-1 step) instead of raising."""
        err = C.create_string_buffer(512)
        rc = self._L.hmk_run(self._h, err, 512)
        return rc, err.value.decode(errors="replace")

    def download(self) -> GreedyResult:
        n = self.n
        cid = np.empty(max(n, 1), dtype=np.int32)
        rank = np.empty(max(n, 1), dtype=np.int32)
        order = np.empty(max(n, 1), dtype=np.int32)
        out = _lib.GreedyOut(_ptr(cid, C.c_int32), _ptr(rank, C.c_int32), _ptr(order, C.c_int32), 0, 0, -1)
        err = C.create_string_buffer(512)
        rc = self._L.hmk_download(self._h, C.byref(out), err, 512)
        if rc:
            _raise_status(rc, err.value)
        return GreedyResult(cid[:n], rank[:n], order[:out.n_result].copy(), int(out.n_multi), self.stats())

    def stats(self) -> dict:
        st = _lib.Stats()
        self._L.hmk_get_stats(self._h, C.byref(st))
        return st.as_dict()

    def init_distributed(self, dist, rank: int, world: int):
        """Join an NCCL communicator of `world` ranks.  `dist` is an initialised torch.distributed
        (any backend): it is only used to hand rank 0's 128-byte NCCL id to the other ranks."""
        from . import distributed
        uid = distributed.exchange_unique_id(dist, rank, nccl_unique_id)
        buf = (C.c_char * 128).from_buffer_copy(uid)
        err = C.create_string_buffer(512)
        rc = self._L.hmk_init_distributed(self._h, int(rank), int(world), buf, err, 512)
        if rc:
            _raise_status(rc, err.value)

    def timer_begin(self):
        self._L.hmk_timer_begin(self._h)

    def timer_end(self) -> float:
        ms = C.c_double(0)
        self._L.hmk_timer_end(self._h, C.byref(ms))
        return float(ms.value)

    def measure_peaks(self) -> dict:
        buf = (C.c_double * 4)()
        err = C.create_string_buffer(512)
        rc = self._L.hmk_measure_peaks(self._h, buf, err, 512)
        if rc:
            _raise_status(rc, err.value)
        return {"int32_iadd3_per_s": buf[0], "int32_mix_per_s": buf[1], "smem_lds_bytes_per_s": buf[2],
                "sm_count": int(buf[3])}

    def section_ms(self) -> dict:
        buf = (C.c_double * len(_lib.SECTIONS))()
        self._L.hmk_get_section_ms(self._h, buf, len(_lib.SECTIONS))
        return {k: float(buf[i]) for i, k in enumerate(_lib.SECTIONS)}

    def clinkage(self, residues, offsets, abundance, matrix, threshold, max_shift, shift_penalty):
        """hmk_clinkage_run: the exact complete-linkage clustering of clinkage_cluster_arrays on this context, so that its
        options apply and stats() / section_ms() report the call (section slots 0, 1, 2 = scoring, sparse row build,
        chain) -> (status, GreedyResult | None, message).  Replaces the uploaded sequences."""
        residues = np.ascontiguousarray(residues, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.int32)
        abundance = np.ascontiguousarray(abundance, dtype=np.int32)
        matrix = np.ascontiguousarray(matrix, dtype=np.int32).reshape(-1)
        self._keep = (residues, offsets, abundance, matrix)
        n = self.n = len(abundance)
        cid = np.empty(max(n, 1), dtype=np.int32)
        rank = np.empty(max(n, 1), dtype=np.int32)
        order = np.empty(max(n, 1), dtype=np.int32)
        gin = _lib.GreedyIn(n, _ptr(residues, C.c_uint8), _ptr(offsets, C.c_int32), _ptr(abundance, C.c_int32),
                            _ptr(matrix, C.c_int32), int(threshold), int(max_shift), int(shift_penalty), 0)
        out = _lib.GreedyOut(_ptr(cid, C.c_int32), _ptr(rank, C.c_int32), _ptr(order, C.c_int32), 0, 0, -1)
        err = C.create_string_buffer(512)
        rc = self._L.hmk_clinkage_run(self._h, C.byref(gin), C.byref(out), err, 512)
        if rc:
            return rc, None, err.value
        return 0, GreedyResult(cid[:n], rank[:n], order[:out.n_result].copy(), int(out.n_multi), self.stats()), b""

    def score_block(self, first_ids, second_ids) -> np.ndarray:
        """scores[a, b] = ShiftedScorer.sequenceScore(seq1 = first_ids[a], seq2 = second_ids[b])."""
        f = np.ascontiguousarray(first_ids, dtype=np.int32)
        s = np.ascontiguousarray(second_ids, dtype=np.int32)
        out = np.empty((len(f), len(s)), dtype=np.int32)
        err = C.create_string_buffer(512)
        rc = self._L.hmk_score_block(self._h, _ptr(f, C.c_int32), len(f), _ptr(s, C.c_int32), len(s),
                                     _ptr(out, C.c_int32), err, 512)
        if rc:
            _raise_status(rc, err.value)
        return out

    def graph_page(self, cursor, cap: int):
        """hmk_score_graph: at most `cap` edges of the score graph from `cursor` = (row, edges of the row already taken)
        -> (EDGE_DTYPE array, next cursor); the cursor (n, 0) means done."""
        cur = (C.c_int64 * 2)(int(cursor[0]), int(cursor[1]))
        out = np.empty(max(int(cap), 1), dtype=EDGE_DTYPE)
        got = C.c_int64(0)
        err = C.create_string_buffer(512)
        rc = self._L.hmk_score_graph(self._h, cur, out.ctypes.data_as(C.c_void_p), int(cap), C.byref(got), err, 512)
        if rc:
            _raise_status(rc, err.value)
        return out[:got.value], (int(cur[0]), int(cur[1]))

    def score_graph(self, chunk: int = 1 << 22):
        """Yields the score graph of the uploaded sequences as EDGE_DTYPE arrays of at most `chunk` edges, in graph order
        (seq, then partner): every pair seq < partner with ShiftedScorer.scoreWithShift(partner, seq) >= threshold."""
        cursor = (0, 0)
        while cursor != (self.n, 0):
            edges, cursor = self.graph_page(cursor, chunk)
            if len(edges):
                yield edges

    def score_pairs(self, seq1_ids, seq2_ids):
        """hmk_score_pairs: ShiftedScorer.scoreWithShift(seq1 = seq1_ids[e], seq2 = seq2_ids[e]) -> (scores, shifts)."""
        a = np.ascontiguousarray(seq1_ids, dtype=np.int32)
        b = np.ascontiguousarray(seq2_ids, dtype=np.int32)
        if a.shape != b.shape:
            raise ValueError("seq1_ids and seq2_ids differ in length")
        scores = np.empty(max(len(a), 1), dtype=np.int32)
        shifts = np.empty(max(len(a), 1), dtype=np.int32)
        err = C.create_string_buffer(512)
        rc = self._L.hmk_score_pairs(self._h, _ptr(a, C.c_int32), _ptr(b, C.c_int32), len(a), _ptr(scores, C.c_int32),
                                     _ptr(shifts, C.c_int32), err, 512)
        if rc:
            _raise_status(rc, err.value)
        return scores[:len(a)], shifts[:len(a)]

    def nearest(self, k: int, rows=None):
        """hmk_nearest: the k best-scoring partners of every row in `rows` = (begin, end) (default: all uploaded
        sequences) -> (partner, score, shift) [rows, k] and (count, more) [rows], all int32.  Row i's entries are the
        sequences j != i with ShiftedScorer.scoreWithShift(seq1 = j, seq2 = i) >= threshold, best first under (score
        desc, abundance[j] desc, j asc); slots past count[i] hold partner -1.  more = 1: more than k qualify."""
        begin, end = (0, self.n) if rows is None else (int(rows[0]), int(rows[1]))
        m = max(end - begin, 0)
        partner = np.empty((m, max(int(k), 0)), dtype=np.int32)
        score, shift = np.empty_like(partner), np.empty_like(partner)
        count, more = np.empty(m, dtype=np.int32), np.empty(m, dtype=np.int32)
        err = C.create_string_buffer(512)
        rc = self._L.hmk_nearest(self._h, int(k), begin, end - begin, _ptr(partner, C.c_int32), _ptr(score, C.c_int32),
                                 _ptr(shift, C.c_int32), _ptr(count, C.c_int32), _ptr(more, C.c_int32), err, 512)
        if rc:
            _raise_status(rc, err.value)
        return partner, score, shift, count, more

    _KERNELS = {-1: "none", 0: "generic", 1: "fast", 2: "filter", 3: "long"}

    def bulk_probe(self, mode: int, query_ids, db=None, db_range=None, clustered=None, hit_cap: int = 0):
        """hmk_bulk_probe: one bulk launch (the kernel tests' hook).  The thread side is the id list `db` or the id range
        `db_range` = (begin, count); `clustered` (optional, bool per uploaded sequence) skips those items.
        -> dict with "hits" (int32 [k, 3]: query id (mode 0) or query index (mode 1), thread-side
        id, score), "hit_count" (what the kernel found; may exceed hit_cap), "kernel" (kind, filter_lt, nw, lane_bits,
        persistent) and, in mode 0, "keys" (uint64 [nq, kb]), "cnt", "ovf"."""
        q = np.ascontiguousarray(query_ids, dtype=np.int32)
        nq = len(q)
        if (db is None) == (db_range is None):
            raise ValueError("give exactly one of db and db_range")
        if db is not None:
            dbi = np.ascontiguousarray(db, dtype=np.int32)
            dbp, begin, ndb = _ptr(dbi, C.c_int32), 0, len(dbi)
        else:
            dbi = None
            dbp, (begin, ndb) = None, (int(db_range[0]), int(db_range[1]))
        cl = None if clustered is None else np.ascontiguousarray(clustered, dtype=np.uint8)
        keys = np.zeros((max(nq, 1), self._kb), dtype=np.uint64)
        cnt = np.zeros(max(nq, 1), dtype=np.int32)
        ovf = np.zeros(max(nq, 1), dtype=np.int32)
        hits = np.zeros((max(hit_cap, 1), 3), dtype=np.int32)
        hcount = C.c_int64(0)
        kern = np.zeros(5, dtype=np.int32)
        err = C.create_string_buffer(512)
        rc = self._L.hmk_bulk_probe(self._h, int(mode), _ptr(q, C.c_int32), nq, dbp, begin, ndb,
                                    None if cl is None else _ptr(cl, C.c_uint8), _ptr(keys, C.c_uint64),
                                    _ptr(cnt, C.c_int32), _ptr(ovf, C.c_int32), _ptr(hits, C.c_int32), int(hit_cap),
                                    C.byref(hcount), _ptr(kern, C.c_int32), err, 512)
        if rc:
            _raise_status(rc, err.value)
        out = {"hits": hits[:min(hcount.value, hit_cap)], "hit_count": int(hcount.value),
               "kernel": {"kind": self._KERNELS[int(kern[0])], "filter_lt": int(kern[1]), "nw": int(kern[2]),
                          "lane_bits": int(kern[3]), "persistent": int(kern[4])}}
        if mode == 0:
            out.update(keys=keys[:nq], cnt=cnt[:nq], ovf=ovf[:nq])
        return out

    def batch_probe(self, clusters, cur: int, nq: int, capq: int = 0, tail_stream: bool = False, fhit_cap: int = 1 << 20):
        """hmk_batch_probe: phase 1's per-batch inputs of the resolver on the clustering state `clusters` (a list of member
        id lists in chain order, founder first; everything else is a singleton), batch = the first nq singletons with id
        >= cur (the kernel tests' hook).  -> dict with "qid", "keys" (uint64 [nq, kb]), "cnt", "ovf", "ib" [nq, nq],
        "ibm", "ibm2" (uint32 [nq, nw]), "pcand" [nq, kb], "pd" [nq, nq * kb], "fhits" (int32 [k, 3]: query index,
        founder id, score), "fhit_count", "ac_cnt", "ac_slot", "ac_score" [nq, capq], "ac_best" [nq, 4] and "kernel"."""
        off = np.zeros(len(clusters) + 1, dtype=np.int32)
        off[1:] = np.cumsum([len(c) for c in clusters])
        mem = np.ascontiguousarray(np.concatenate([np.asarray(c, dtype=np.int32) for c in clusters]) if clusters
                                   else np.zeros(1, dtype=np.int32), dtype=np.int32)
        kb, nw = self._kb, (nq + 31) // 32
        cq = capq if capq > 0 else self._capq
        a = dict(qid=np.zeros(nq, np.int32), keys=np.zeros((nq, kb), np.uint64), cnt=np.zeros(nq, np.int32),
                 ovf=np.zeros(nq, np.int32), ib=np.zeros((nq, nq), np.int32), ibm=np.zeros((nq, nw), np.uint32),
                 ibm2=np.zeros((nq, nw), np.uint32), pcand=np.zeros((nq, kb), np.int32), pd=np.zeros((nq, nq * kb), np.int32),
                 fhits=np.zeros((max(fhit_cap, 1), 3), np.int32), ac_cnt=np.zeros(nq, np.int32),
                 ac_slot=np.zeros((nq, cq), np.int32), ac_score=np.zeros((nq, cq), np.int32),
                 ac_best=np.zeros((nq, 4), np.int32))
        i32, u32 = C.c_int32, C.c_uint32
        o = _lib.BatchProbeOut(0, _ptr(a["qid"], i32), _ptr(a["keys"], C.c_uint64), _ptr(a["cnt"], i32), _ptr(a["ovf"], i32),
                               _ptr(a["ib"], i32), _ptr(a["ibm"], u32), _ptr(a["ibm2"], u32), _ptr(a["pcand"], i32),
                               _ptr(a["pd"], i32), _ptr(a["fhits"], i32), int(fhit_cap), 0, _ptr(a["ac_cnt"], i32),
                               _ptr(a["ac_slot"], i32), _ptr(a["ac_score"], i32), _ptr(a["ac_best"], i32))
        err = C.create_string_buffer(512)
        rc = self._L.hmk_batch_probe(self._h, _ptr(off, i32), _ptr(mem, i32), len(clusters), int(cur), int(nq), int(capq),
                                     int(bool(tail_stream)), C.byref(o), err, 512)
        if rc:
            _raise_status(rc, err.value)
        n = o.nq_out
        out = {k: v[:n] for k, v in a.items() if k != "fhits"}
        out["ib"] = a["ib"].reshape(-1)[:n * n].reshape(n, n)
        nwn = (n + 31) // 32
        out["ibm"], out["ibm2"] = (a[k].reshape(-1)[:n * nwn].reshape(n, nwn) for k in ("ibm", "ibm2"))
        out["pd"] = a["pd"].reshape(-1)[:n * n * kb].reshape(n, n * kb)
        out["fhits"] = a["fhits"][:min(o.fhit_count, fhit_cap)]
        out["fhit_count"] = int(o.fhit_count)
        k = list(o.kernel)
        out["kernel"] = {"kind": self._KERNELS[k[0]], "filter_lt": k[1], "nw": k[2], "lane_bits": k[3], "persistent": k[4],
                         "search_launches": k[5], "tables": "dense_packed" if k[6] == -1 else self._KERNELS[k[6]],
                         "table_launches": k[7], "founder": self._KERNELS[k[8]], "founder_launches": k[9],
                         "member_check": {-1: "none", 0: "state", 1: "packed", 2: "score12x3"}[k[10]]}
        return out


def nccl_unique_id() -> bytes:
    L = _lib.load()
    buf = (C.c_char * 128)()
    err = C.create_string_buffer(512)
    rc = L.hmk_nccl_unique_id(buf, err, 512)
    if rc:
        _raise_status(rc, err.value)
    return bytes(buf)


def result_digest(cluster_id, member_rank, result_order) -> str:
    """sha256 over cluster_id || member_rank || result_order as little-endian int32 -- the three arrays from which the
    host rebuilds the List<Cluster> the reference returns (members, their order, the order of the list).  The golden
    digests under tests/golden/*_digest.json hash the same bytes of a full CPU-oracle run."""
    import hashlib
    h = hashlib.sha256()
    for a in (cluster_id, member_rank, result_order):
        h.update(np.ascontiguousarray(a, dtype="<i4").tobytes())
    return h.hexdigest()


def greedy_cluster_arrays(residues, offsets, abundance, matrix, threshold, max_shift, shift_penalty, max_clusters,
                          device: int = 0, devices: Optional[Sequence[int]] = None):
    """One blocking hmk_greedy_cluster call on host arrays -> (status, GreedyResult | None, error_step, message).
    `devices`: run hmk_greedy_cluster_multi on these GPUs of this process instead (one worker thread per device
    inside the library)."""
    L = _lib.load()
    residues = np.ascontiguousarray(residues, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.int32)
    abundance = np.ascontiguousarray(abundance, dtype=np.int32)
    matrix = np.ascontiguousarray(matrix, dtype=np.int32).reshape(-1)
    n = len(abundance)
    cid = np.empty(max(n, 1), dtype=np.int32)
    rank = np.empty(max(n, 1), dtype=np.int32)
    order = np.empty(max(n, 1), dtype=np.int32)
    gin = _lib.GreedyIn(n, _ptr(residues, C.c_uint8), _ptr(offsets, C.c_int32), _ptr(abundance, C.c_int32),
                        _ptr(matrix, C.c_int32), int(threshold), int(max_shift), int(shift_penalty), int(max_clusters))
    out = _lib.GreedyOut(_ptr(cid, C.c_int32), _ptr(rank, C.c_int32), _ptr(order, C.c_int32), 0, 0, -1)
    err = C.create_string_buffer(512)
    if devices is not None:
        devs = np.ascontiguousarray(devices, dtype=np.int32)
        rc = L.hmk_greedy_cluster_multi(C.byref(gin), C.byref(out), _ptr(devs, C.c_int32), len(devs), err, 512)
    else:
        rc = L.hmk_greedy_cluster(C.byref(gin), C.byref(out), device, err, 512)
    if rc:
        return rc, None, int(out.error_step), err.value
    return 0, GreedyResult(cid[:n], rank[:n], order[:out.n_result].copy(), int(out.n_multi), {}), -1, b""


def clinkage_cluster_arrays(residues, offsets, abundance, matrix, threshold, max_shift, shift_penalty, device: int = 0):
    """One blocking hmk_clinkage_cluster call on host arrays (sequences in the caller's order)
    -> (status, GreedyResult | None, message).  cluster_id holds Cluster.getId() (1-based, merged clusters n + 2, ...)."""
    L = _lib.load()
    residues = np.ascontiguousarray(residues, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.int32)
    abundance = np.ascontiguousarray(abundance, dtype=np.int32)
    matrix = np.ascontiguousarray(matrix, dtype=np.int32).reshape(-1)
    n = len(abundance)
    cid = np.empty(max(n, 1), dtype=np.int32)
    rank = np.empty(max(n, 1), dtype=np.int32)
    order = np.empty(max(n, 1), dtype=np.int32)
    gin = _lib.GreedyIn(n, _ptr(residues, C.c_uint8), _ptr(offsets, C.c_int32), _ptr(abundance, C.c_int32),
                        _ptr(matrix, C.c_int32), int(threshold), int(max_shift), int(shift_penalty), 0)
    out = _lib.GreedyOut(_ptr(cid, C.c_int32), _ptr(rank, C.c_int32), _ptr(order, C.c_int32), 0, 0, -1)
    err = C.create_string_buffer(512)
    rc = L.hmk_clinkage_cluster(C.byref(gin), C.byref(out), device, err, 512)
    if rc:
        return rc, None, err.value
    return 0, GreedyResult(cid[:n], rank[:n], order[:out.n_result].copy(), int(out.n_multi), {}), b""


# ---------------------------------------------------------------- scorer / clusterer seam
class ShiftedScorer:
    """ShiftedScorer.java:12-32 (constructor arguments) -- the scoring itself runs on the GPU."""

    def __init__(self, scoring_matrix, shift_penalty: int, max_shift: int, device: int = 0):
        self.scoring_matrix = np.ascontiguousarray(scoring_matrix, dtype=np.int32).reshape(24, 24)
        self.shift_penalty, self.max_shift, self.device = int(shift_penalty), int(max_shift), device

    def sequence_score(self, seq1: UniqueSequence, seq2: UniqueSequence) -> int:
        """ShiftedScorer.sequenceScore (ShiftedScorer.java:97-100)."""
        return int(self.score_block([seq1], [seq2])[0, 0])

    def score_with_shift(self, seq1: UniqueSequence, seq2: UniqueSequence):
        """AligningSequenceScorer.scoreWithShift (ShiftedScorer.java:48-95) -> (score, shift), the AligningScorerResult."""
        res, offs, ab = pack_sequences([seq1, seq2])
        ctx = GreedyContext(self.device)
        try:
            ctx.upload(res, offs, ab, self.scoring_matrix, 0, self.max_shift, self.shift_penalty, 0)
            scores, shifts = ctx.score_pairs([0], [1])
            return int(scores[0]), int(shifts[0])
        finally:
            ctx.close()

    def score_block(self, firsts: Sequence[UniqueSequence], seconds: Sequence[UniqueSequence]) -> np.ndarray:
        seqs = list(firsts) + list(seconds)
        if min(len(s.sequence) for s in seqs) <= self.max_shift:        # ShiftedScorer.java:59-62
            raise DataException("Shift too big")
        res, offs, ab = pack_sequences(seqs)
        ctx = GreedyContext(self.device)
        try:
            ctx.upload(res, offs, ab, self.scoring_matrix, 0, self.max_shift, self.shift_penalty, 0)
            return ctx.score_block(np.arange(len(firsts)), np.arange(len(firsts), len(seqs)))
        finally:
            ctx.close()


class LimitedGreedySequenceClusterer:
    """LimitedGreedySequenceClusterer.java:17-30 + SequenceClusterer.java:15-26."""

    def __init__(self, sequence_scorer: ShiftedScorer, threshold: int, max_clusters: int):
        self.sequence_scorer, self.threshold, self.max_clusters = sequence_scorer, int(threshold), int(max_clusters)
        self.last_stats: dict = {}

    def cluster(self, sequences: List[UniqueSequence]) -> List[Cluster]:
        """cluster(List<UniqueSequence>) -> List<Cluster> (LimitedGreedySequenceClusterer.java:39-69).
        `sequences` must already be in clustering order (Hammock.java:407)."""
        sc = self.sequence_scorer
        res, offs, ab = pack_sequences(sequences)
        rc, r, step, err = greedy_cluster_arrays(res, offs, ab, sc.scoring_matrix, self.threshold, sc.max_shift,
                                                 sc.shift_penalty, self.max_clusters, sc.device)
        if rc:
            _raise_status(rc, err, step)
        return rebuild_clusters(sequences, r)


class UnsupportedInput(HammockException):
    """hmk_clinkage_cluster: asymmetric matrix, valid pairs beyond the free device memory, or a treeified java.util.HashMap
    bin"""


class ClinkageSequenceClusterer:
    """ClinkageSequenceClusterer.java:22-39 + SequenceClusterer.java:15-26 -- the exact complete-linkage clusterer
    (nearest-neighbour chain), Hammock's default initial stage for up to 10 000 unique sequences (Hammock.java:371-373)."""

    def __init__(self, sequence_scorer: ShiftedScorer, threshold: int, size_limit: int = 1):
        # size_limit only decides which cluster scores the reference caches (CachedClusterScorer.java:38-41); the
        # cached values equal the recomputed ones, so it does not change the result
        self.sequence_scorer, self.threshold, self.size_limit = sequence_scorer, int(threshold), int(size_limit)

    def cluster(self, sequences: List[UniqueSequence]) -> List[Cluster]:
        """cluster(List<UniqueSequence>) -> List<Cluster> (ClinkageSequenceClusterer.java:43-124), in the order of the
        list the reference returns (java.util.HashSet iteration order, OpenJDK 8+)."""
        sc = self.sequence_scorer
        res, offs, ab = pack_sequences(sequences)
        rc, r, err = clinkage_cluster_arrays(res, offs, ab, sc.scoring_matrix, self.threshold, sc.max_shift, sc.shift_penalty, sc.device)
        if rc == _lib.STATUS_UNSUPPORTED:
            raise UnsupportedInput(err.decode(errors="replace"))
        if rc:
            _raise_status(rc, err)
        return rebuild_clusters(sequences, r)


def set_clinkage_threshold(sequences: Sequence[UniqueSequence]) -> int:
    """Hammock.setClinkageThreshold (Hammock.java:1415-1419)"""
    return _java_round(get_mean_sequence_length(sequences) * 1.7)


def run_clinkage_clustering(sequences: List[UniqueSequence], scoring_matrix, threshold: Optional[int] = None,
                            max_shift: Optional[int] = None, shift_penalty: int = 0, device: int = 0) -> List[Cluster]:
    """The clustering part of Hammock.runClinkageClustering (Hammock.java:449-462): automatic parameters, NO sorting."""
    if not sequences:
        raise FileFormatException("Error. No sequences (with specified labels) to cluster.")   # Hammock.java:783-785
    max_shift = get_max_shift(sequences) if max_shift is None else check_max_shift(sequences, max_shift)
    if threshold is None:
        threshold = set_clinkage_threshold(sequences)
    return ClinkageSequenceClusterer(ShiftedScorer(scoring_matrix, shift_penalty, max_shift, device), threshold).cluster(list(sequences))


def score_graph(sequences: Sequence[UniqueSequence], scoring_matrix, threshold: Optional[int] = None,
                max_shift: Optional[int] = None, shift_penalty: int = 0, device: int = 0) -> np.ndarray:
    """The score graph both initial clusterings are built from: every pair i < j of `sequences` (input order, as
    run_clinkage_clustering) with ShiftedScorer.scoreWithShift(seq j, seq i) >= threshold, as an EDGE_DTYPE array
    ordered by i, then j.  Defaults: setClinkageThreshold and getMaxShift.  GreedyContext.score_graph streams it."""
    if len(sequences) == 0:
        return np.zeros(0, dtype=EDGE_DTYPE)
    max_shift = get_max_shift(sequences) if max_shift is None else check_max_shift(sequences, max_shift)
    if threshold is None:
        threshold = set_clinkage_threshold(sequences)
    res, offs, ab = pack_sequences(sequences)
    ctx = GreedyContext(device)
    try:
        ctx.upload(res, offs, ab, scoring_matrix, threshold, max_shift, shift_penalty, 0)
        parts = list(ctx.score_graph())
    finally:
        ctx.close()
    return np.concatenate(parts) if parts else np.zeros(0, dtype=EDGE_DTYPE)


def save_score_graph(sequences: Sequence[UniqueSequence], edges, path: str) -> None:
    """score_graph.tsv: header `sequence, partner, score, shift`, one row per edge in the order given, sequences as
    strings.  `edges`: one EDGE_DTYPE array or an iterable of them (GreedyContext.score_graph)."""
    strs = [s.get_sequence_string() for s in sequences]
    chunks = [edges] if isinstance(edges, np.ndarray) else edges
    with open(path, "w", newline="") as w:
        w.write("sequence\tpartner\tscore\tshift\n")
        for e in chunks:
            w.write("".join(f"{strs[i]}\t{strs[j]}\t{s}\t{k}\n"
                            for i, j, s, k in zip(e["seq"].tolist(), e["partner"].tolist(), e["score"].tolist(),
                                                  e["shift"].tolist())))


def nearest_partners(sequences: Sequence[UniqueSequence], scoring_matrix, k: int = 8, threshold: Optional[int] = None,
                     max_shift: Optional[int] = None, shift_penalty: int = 0, device: int = 0):
    """The k nearest partners of every sequence of `sequences` (input order, as score_graph): the sequences j != i with
    ShiftedScorer.scoreWithShift(seq j, seq i) >= threshold, best first under (score desc, size desc, j asc) ->
    (partner, score, shift) [n, k] and (count, more) [n] as GreedyContext.nearest returns them.  Defaults:
    setClinkageThreshold and getMaxShift."""
    if len(sequences) == 0:
        z = np.zeros((0, k), dtype=np.int32)
        return z, z.copy(), z.copy(), np.zeros(0, np.int32), np.zeros(0, np.int32)
    max_shift = get_max_shift(sequences) if max_shift is None else check_max_shift(sequences, max_shift)
    if threshold is None:
        threshold = set_clinkage_threshold(sequences)
    res, offs, ab = pack_sequences(sequences)
    ctx = GreedyContext(device)
    try:
        ctx.upload(res, offs, ab, scoring_matrix, threshold, max_shift, shift_penalty, 0)
        return ctx.nearest(k)
    finally:
        ctx.close()


def save_nearest_partners(sequences: Sequence[UniqueSequence], nearest, path: str) -> None:
    """nearest_partners.tsv: header `sequence, rank, partner, score, shift`, then for every sequence in input order its
    entries rank 1 .. count, sequences as strings.  `nearest`: what nearest_partners returns, for all sequences."""
    partner, score, shift, count = (np.asarray(a) for a in nearest[:4])
    strs = [s.get_sequence_string() for s in sequences]
    with open(path, "w", newline="") as w:
        w.write("sequence\trank\tpartner\tscore\tshift\n")
        for i, c in enumerate(count.tolist()):
            w.write("".join(f"{strs[i]}\t{r + 1}\t{strs[j]}\t{s}\t{h}\n"
                            for r, (j, s, h) in enumerate(zip(partner[i, :c].tolist(), score[i, :c].tolist(),
                                                              shift[i, :c].tolist()))))


def rebuild_clusters(sequences: Sequence[UniqueSequence], r: GreedyResult) -> List[Cluster]:
    """cluster_id / member_rank / result_order -> the List<Cluster> the reference returns."""
    members: Dict[int, List] = {}
    for i, (c, k) in enumerate(zip(r.cluster_id.tolist(), r.member_rank.tolist())):
        members.setdefault(c, []).append((k, i))
    out = []
    for c in r.result_order.tolist():
        ms = sorted(members[c])
        cl = Cluster([sequences[ms[0][1]]], c)
        for _, i in ms[1:]:
            cl.insert(sequences[i])      # raises DataException on a duplicate member (Cluster.java:51-55)
        out.append(cl)
    return out


def run_greedy_clustering(sequences: List[UniqueSequence], scoring_matrix, threshold: Optional[int] = None,
                          max_shift: Optional[int] = None, shift_penalty: int = 0,
                          initial_clusters_limit_: Optional[int] = None, order: str = "size",
                          labels: Optional[Sequence[str]] = None, seed: int = 42, device: int = 0) -> List[Cluster]:
    """The clustering part of Hammock.runGreedyClustering (Hammock.java:392-411) with its
    automatic parameters (:394-401, 803-812)."""
    if not sequences:
        raise FileFormatException("Error. No sequences (with specified labels) to cluster.")   # Hammock.java:783-785
    if max_shift is None:
        max_shift = get_max_shift(sequences)
    else:
        max_shift = check_max_shift(sequences, max_shift)
    if threshold is None:
        threshold = set_greedy_threshold(sequences)
    if initial_clusters_limit_ is None:
        initial_clusters_limit_ = initial_clusters_limit(sequences)
    scorer = ShiftedScorer(scoring_matrix, shift_penalty, max_shift, device)
    clusterer = LimitedGreedySequenceClusterer(scorer, threshold, initial_clusters_limit_)
    ordered = sort_sequences(list(sequences), order, labels, seed)
    return clusterer.cluster(ordered)
