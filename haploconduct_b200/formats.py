"""Host-side containers and file formats of the path (numpy only, no device code).

Mirrors, for the Python tests / bench harness, what the reference keeps in
``FastqStorage`` (src/FastqStorage.h:58-98, src/FastqStorage.cpp:92-235) and ``Overlap``
(src/Overlap.h:20-59): reads in ``m_read_vec`` order (singles first, then pairs), and the
13-column overlaps text format ``ID1 ID2 POS1 POS2 ORD ORI1 ORI2 PERC1 PERC2 LEN1 LEN2 TYPE1 TYPE2``
(scripts/sfo2overlaps.py:153).  The numpy dtypes below are byte-for-byte the C structs of
``include/hc_b200.h``.
"""
from __future__ import annotations

import os
from dataclasses import dataclass, field
from typing import Dict, Iterable, List, Optional, Tuple

import numpy as np

# ---- C-ABI mirrors (include/hc_b200.h) -------------------------------------------------------
READ_DESC = np.dtype([("seq_off", "<u8", (2,)), ("seq_len", "<u4", (2,))])
CANDIDATE = np.dtype(
    [
        ("idx1", "<u4"), ("idx2", "<u4"), ("pos1", "<u4"), ("pos2", "<u4"), ("len1", "<u4"), ("len2", "<u4"),
        ("perc1", "u1"), ("perc2", "u1"), ("ord", "u1"), ("ori1", "u1"), ("ori2", "u1"),
        ("type1", "u1"), ("type2", "u1"), ("reserved", "u1"),
    ]
)
CANDIDATE_COMPACT = np.dtype([("idx1", "<u4"), ("idx2", "<u4"), ("pos1_flags", "<u4"), ("pos2", "<u4")])


def compact_candidates(c: np.ndarray) -> np.ndarray:
    """hc_candidate -> hc_candidate_compact (POS1 must fit 28 bits)."""
    out = np.zeros(len(c), dtype=CANDIDATE_COMPACT)
    out["idx1"], out["idx2"], out["pos2"] = c["idx1"], c["idx2"], c["pos2"]
    assert (c["pos1"] < (1 << 28)).all()
    ordc = np.where(c["ord"] == ord("1"), 1, np.where(c["ord"] == ord("2"), 2, 0)).astype(np.uint32)
    out["pos1_flags"] = c["pos1"] | ((c["ori1"] != 0).astype(np.uint32) << 28) | ((c["ori2"] != 0).astype(np.uint32) << 29) | (ordc << 30)
    return out


CANDIDATE_SHORT = np.dtype([("idx1", "<u4"), ("idx2", "<u4"), ("pos", "<u4")])
assert CANDIDATE_SHORT.itemsize == 12


def short_candidates(c: np.ndarray) -> np.ndarray:
    """hc_candidate -> hc_candidate_short (POS1 and POS2 must be below 2^14)."""
    if len(c) and (int(c["pos1"].max()) >= (1 << 14) or int(c["pos2"].max()) >= (1 << 14)):
        raise ValueError("positions do not fit the 12-byte candidate record")
    out = np.zeros(len(c), dtype=CANDIDATE_SHORT)
    out["idx1"], out["idx2"] = c["idx1"], c["idx2"]
    ordc = np.where(c["ord"] == ord("1"), 1, np.where(c["ord"] == ord("2"), 2, 0)).astype(np.uint32)
    out["pos"] = (c["pos1"] | (c["pos2"].astype(np.uint32) << 14) | ((c["ori1"] != 0).astype(np.uint32) << 28)
                  | ((c["ori2"] != 0).astype(np.uint32) << 29) | (ordc << 30))
    return out


CANDIDATE_ENTRY = np.dtype([("other", "<u4"), ("pos", "<u4")])
assert CANDIDATE_ENTRY.itemsize == 8


def run_encode(c: np.ndarray):
    """hc_candidate -> (run_anchor uint32[n_runs], run_start uint64[n_runs + 1], hc_candidate_entry[n]) for
    hc_score_batch_runs.  A run is a stretch of consecutive candidates that share one read; two vectorised cuts are
    tried (runs of equal ID1, runs of equal min(ID1, ID2) -- the sort key of scripts/sfo2overlaps.py:52) and the one with
    fewer runs is kept.  The candidate order is not changed."""
    n = len(c)
    if n == 0:
        return np.zeros(0, np.uint32), np.zeros(1, np.uint64), np.zeros(0, CANDIDATE_ENTRY)
    sc = short_candidates(c)
    i1, i2 = sc["idx1"], sc["idx2"]
    if int(max(i1.max(), i2.max())) >= (1 << 31):
        raise ValueError("read indices do not fit the 8-byte candidate record")
    best = None
    for key in (i1, np.minimum(i1, i2)):
        cut = np.flatnonzero(np.concatenate(([True], key[1:] != key[:-1])))
        if best is None or len(cut) < len(best[0]):
            best = (cut, key)
    cut, key = best
    start = np.concatenate((cut, [n])).astype(np.uint64)
    anchor = key[cut].astype(np.uint32)
    per_cand_anchor = key
    out = np.zeros(n, dtype=CANDIDATE_ENTRY)
    is1 = i1 == per_cand_anchor                      # the anchor is ID1 -> store ID2, flag 0
    out["other"] = np.where(is1, i2, i1 | np.uint32(1 << 31))
    out["pos"] = sc["pos"]
    return anchor, start, out


def entries6(en: np.ndarray) -> np.ndarray:
    """hc_candidate_entry (8 bytes) -> hc_candidate_entry6 (6 bytes, uint8[n, 6]): a 48-bit little-endian number, bits 0-24
    other read, 25 anchor-is-ID2, 26 ORI1 '+', 27 ORI2 '+', 28-29 ORD, 30-38 POS1, 39-47 POS2 (reads shorter than 512 bases,
    at most 2^25 reads)."""
    other = (en["other"] & np.uint32(0x7fffffff)).astype(np.uint64)
    role = (en["other"] >> np.uint32(31)).astype(np.uint64)
    pos = en["pos"].astype(np.uint64)
    p1, p2 = pos & np.uint64(0x3fff), (pos >> np.uint64(14)) & np.uint64(0x3fff)
    flags = (pos >> np.uint64(28)) & np.uint64(0xf)                     # ORI1, ORI2, ORD (2 bits)
    if len(en) and (int(other.max()) >= (1 << 25) or int(p1.max()) >= 512 or int(p2.max()) >= 512):
        raise ValueError("records do not fit the 6-byte candidate entry")
    v = other | (role << np.uint64(25)) | (flags << np.uint64(26)) | (p1 << np.uint64(30)) | (p2 << np.uint64(39))
    return np.ascontiguousarray(v.astype("<u8").view(np.uint8).reshape(-1, 8)[:, :6])


PARAMS = np.dtype(
    [
        ("edge_threshold", "<f8"), ("ov_threshold", "<f8"), ("merge_contigs", "<f8"), ("mismatch", "<f8"),
        ("min_read_len", "<u4"), ("flags", "<u4"),
    ]
)
RESULT = np.dtype(
    [
        ("score", "<f8"), ("mismatch_rate", "<f8"), ("pos3", "<i4"), ("pos4", "<i4"),
        ("mismatches", "<u4", (2,)), ("compared", "<u4", (2,)),
        ("cls", "u1"), ("status", "u1", (2,)), ("exact", "u1"), ("indel_count", "<u4"),
    ]
)
EDGE = np.dtype([("cand", "<u8"), ("score", "<f8"), ("mismatch_rate", "<f8"), ("pos3", "<i4"), ("pos4", "<i4"),
                 ("mean_log", "<f8", (2,))])
EDGE_SMALL = np.dtype([("cand", "<u4"), ("mismatches", "<u2", (2,)), ("compared", "<u2", (2,)), ("flags", "<u4"), ("score", "<f8")])
EDGE_SMALL_EXACT = np.dtype([("cand", "<u4"), ("mismatches", "<u2", (2,)), ("compared", "<u2", (2,)), ("flags", "<u4"),
                             ("mean_log", "<f8", (2,))])
EDGE_BOTH, EDGE_TWO, EDGE_EXACT, EDGE_OVERFLOW = 1, 2, 4, 8
assert EDGE_SMALL.itemsize == 24 and EDGE_SMALL_EXACT.itemsize == 32
BATCH_STATS = np.dtype(
    [
        ("n_candidates", "<u8"), ("n_edges", "<u8"), ("n_nonedges", "<u8"), ("n_exact", "<u8"),
        ("n_windows", "<u8"), ("n_positions", "<u8"), ("algorithmic_bytes", "<u8"),
        ("kernel_ms", "<f4"), ("total_ms", "<f4"), ("kernel_launches", "<u4"), ("score_kernel_ms", "<f4"),
    ]
)
assert READ_DESC.itemsize == 24 and CANDIDATE.itemsize == 32 and PARAMS.itemsize == 40
assert RESULT.itemsize == 48 and EDGE.itemsize == 48 and BATCH_STATS.itemsize == 72

# FindNextOverlaps (FNO1) records
FNO_EDGE = np.dtype([("u", "<u4"), ("v", "<u4"), ("pos1", "<i4"), ("pos2", "<i4"), ("perc", "<i4"), ("len1", "<i4"),
                     ("len2", "<i4"), ("ord", "u1"), ("ori1", "u1"), ("ori2", "u1"), ("nonedge", "u1")])
FNO_READ = np.dtype([("id", "<u8"), ("len1", "<u4"), ("len2", "<u4")])
FNO_SUBREAD = np.dtype([("index1", "<i4"), ("index2", "<i4"), ("startpos1", "<i4"), ("startpos2", "<i4")])
FNO_OVERLAP = np.dtype([("id1", "<u8"), ("id2", "<u8"), ("pos1", "<i4"), ("pos2", "<i4"), ("perc", "<i4"), ("len1", "<i4"),
                        ("len2", "<i4"), ("ord", "u1"), ("ori1", "u1"), ("ori2", "u1"), ("type1", "u1"), ("type2", "u1"),
                        ("reserved", "u1", (3,)), ("perc2", "<i4")])
FNO3_POS = np.dtype([("index1", "<i4"), ("index2", "<i4")])
DEDUP_EDGE = np.dtype([("vertex1", "<u4"), ("vertex2", "<u4"), ("score", "<f8"), ("mismatch_rate", "<f8"), ("pos1", "<i4"),
                       ("pos2", "<i4"), ("pos3", "<i4"), ("overlap_len", "<i4"), ("perc", "<i4"), ("ori1", "u1"), ("ori2", "u1"),
                       ("reserved", "u1", (2,))])
assert DEDUP_EDGE.itemsize == 48
INGEST_PARAMS = np.dtype([("max_overlaps", "<u8"), ("min_overlap_len", "<u4"), ("min_overlap_perc", "<u4"), ("relax_PE_edges", "u1"),
                          ("allow_spaces", "u1"), ("reserved", "u1", (6,))])
OVERLAP_REC = np.dtype([("id1", "<u8"), ("id2", "<u8"), ("pos1", "<u4"), ("pos2", "<u4"), ("perc1", "<u4"), ("perc2", "<u4"),
                        ("len1", "<u4"), ("len2", "<u4"), ("ord", "u1"), ("ori1", "u1"), ("ori2", "u1"), ("type1", "u1"),
                        ("type2", "u1"), ("reserved", "u1", (3,))])
INGEST_STATS = np.dtype([("n_lines", "<u8"), ("n_scored", "<u8"), ("n_filtered", "<u8"), ("n_skipped", "<u8"), ("n_dropped", "<u8"),
                         ("first_error_line", "<u8"), ("first_error_offset", "<u8"), ("first_error_length", "<u8"),
                         ("first_error_status", "<u4"), ("device_ms", "<f4")])
assert INGEST_PARAMS.itemsize == 24 and OVERLAP_REC.itemsize == 48 and INGEST_STATS.itemsize == 72
INGEST_SCORE_STATS = np.dtype([("ingest", INGEST_STATS), ("score", BATCH_STATS), ("n_kept", "<u8")])   # hc_ingest_score_stats
assert INGEST_SCORE_STATS.itemsize == 152
FNO_NONEDGE_STATS = np.dtype([("n_lines", "<u8"), ("n_nonedges", "<u8"), ("n_stream", "<u8"), ("first_error_line", "<u8"),
                              ("first_error_offset", "<u8"), ("first_error_length", "<u8"), ("first_error_status", "<u4"),
                              ("device_ms", "<f4")])   # hc_fno_nonedge_stats
assert FNO_NONEDGE_STATS.itemsize == 56
CONS_SEQ = np.dtype([("read", "<u4"), ("mate", "u1"), ("rc", "u1"), ("reserved", "<u2"), ("pos", "<i4")])
CONS_PROBLEM = np.dtype([("seq_begin", "<u8"), ("seq_end", "<u8"), ("out_offset", "<u8"), ("total_len", "<i4"),
                         ("subreads_needed", "u1"), ("error_correction", "u1"), ("reserved", "u1", (2,))])
CONS_RESULT = np.dtype([("ret", "<i4"), ("length", "<i4")])
assert CONS_SEQ.itemsize == 12 and CONS_PROBLEM.itemsize == 32 and CONS_RESULT.itemsize == 8


def consensus_arrays(problems) -> tuple:
    """List of dicts (total_len, subreads_needed, error_correction, entries [(read, mate, rc, pos)]) -> (CONS_PROBLEM, CONS_SEQ)
    with the outputs laid out back to back."""
    n_seq = sum(len(p["entries"]) for p in problems)
    P = np.zeros(len(problems), dtype=CONS_PROBLEM)
    S = np.zeros(n_seq, dtype=CONS_SEQ)
    k = off = 0
    for i, p in enumerate(problems):
        P[i]["seq_begin"], P[i]["seq_end"] = k, k + len(p["entries"])
        P[i]["out_offset"], P[i]["total_len"] = off, p["total_len"]
        P[i]["subreads_needed"], P[i]["error_correction"] = int(p["subreads_needed"]), int(p["error_correction"])
        for read, mate, rc, pos in p["entries"]:
            S[k] = (read, mate, int(rc), 0, pos)
            k += 1
        off += p["total_len"]
    return P, S


LINE_SCORE, LINE_NONEDGE, LINE_DROPPED, LINE_SKIPPED, LINE_ERROR, LINE_UNKNOWN_ID = 1, 2, 3, 4, 5, 6


def make_ingest_params(min_overlap_len: int, min_overlap_perc: int = 0, relax_PE_edges: bool = False, allow_spaces: bool = False,
                       max_overlaps: int = 2 ** 64 - 1) -> np.ndarray:
    p = np.zeros(1, dtype=INGEST_PARAMS)
    p["max_overlaps"], p["min_overlap_len"], p["min_overlap_perc"] = max_overlaps, min_overlap_len, min_overlap_perc
    p["relax_PE_edges"], p["allow_spaces"] = int(relax_PE_edges), int(allow_spaces)
    return p


def overlap_rec_lines(recs: np.ndarray) -> list:
    """Overlap::get_overlap_line (src/Overlap.h:234-237) of OVERLAP_REC records, without the newline."""
    return ["%d\t%d\t%d\t%d\t%s\t%s\t%s\t%d\t%d\t%d\t%d\t%s\t%s" % (
        int(r["id1"]), int(r["id2"]), int(r["pos1"]), int(r["pos2"]), chr(r["ord"]), chr(r["ori1"]), chr(r["ori2"]), int(r["perc1"]),
        int(r["perc2"]), int(r["len1"]), int(r["len2"]), chr(r["type1"]), chr(r["type2"])) for r in recs]


def candidate_lines(cands: np.ndarray, ids: np.ndarray) -> list:
    """The same line for CANDIDATE records (ids through the store's id table)."""
    return ["%d\t%d\t%d\t%d\t%s\t%s\t%s\t%d\t%d\t%d\t%d\t%s\t%s" % (
        int(ids[c["idx1"]]), int(ids[c["idx2"]]), int(c["pos1"]), int(c["pos2"]), chr(c["ord"]), "+" if c["ori1"] else "-",
        "+" if c["ori2"] else "-", int(c["perc1"]), int(c["perc2"]), int(c["len1"]), int(c["len2"]), chr(c["type1"]), chr(c["type2"]))
        for c in cands]
assert FNO_EDGE.itemsize == 32 and FNO_READ.itemsize == 16 and FNO_SUBREAD.itemsize == 16 and FNO_OVERLAP.itemsize == 48

CLASS_DISCARD, CLASS_EDGE, CLASS_NONEDGE = 0, 1, 2
FLAG_EXACT_EDGE_SCORES = 1


def make_params(edge_threshold=0.99, ov_threshold=0.9, merge_contigs=0.0, mismatch=0.0, min_read_len=0, flags=0):
    """Defaults are the option-table defaults of src/ViralQuasispecies.cpp:63-64,81,83,88."""
    p = np.zeros(1, dtype=PARAMS)
    p["edge_threshold"] = edge_threshold
    p["ov_threshold"] = ov_threshold
    p["merge_contigs"] = merge_contigs
    p["mismatch"] = mismatch
    p["min_read_len"] = min_read_len
    p["flags"] = flags
    return p


# ---- reads -------------------------------------------------------------------------------------
@dataclass
class ReadSet:
    """Reads in m_read_vec order: ``n_single`` singles, then pairs (src/FastqStorage.h:88-97)."""

    ids: np.ndarray          # uint64 read IDs as used in the overlaps file
    descs: np.ndarray        # READ_DESC per read
    bases: np.ndarray        # uint8 ASCII blob
    quals: np.ndarray        # uint8 ASCII blob (raw FASTQ characters)
    n_single: int
    _id_to_index: Optional[Dict[int, int]] = field(default=None, repr=False)

    @property
    def n_reads(self) -> int:
        return int(self.descs.shape[0])

    def id_to_index(self) -> Dict[int, int]:
        if self._id_to_index is None:
            self._id_to_index = {int(v): i for i, v in enumerate(self.ids)}
        return self._id_to_index

    def seq(self, idx: int, mate: int = 0) -> str:
        d = self.descs[idx]
        o, n = int(d["seq_off"][mate]), int(d["seq_len"][mate])
        return self.bases[o:o + n].tobytes().decode()

    def qual(self, idx: int, mate: int = 0) -> str:
        d = self.descs[idx]
        o, n = int(d["seq_off"][mate]), int(d["seq_len"][mate])
        return self.quals[o:o + n].tobytes().decode()

    def is_paired(self, idx: int) -> bool:
        return int(self.descs[idx]["seq_len"][1]) > 0

    @staticmethod
    def from_lists(singles: List[Tuple[int, str, str]], pairs: List[Tuple[int, str, str, str, str]]) -> "ReadSet":
        """singles: (id, seq, qual); pairs: (id, seq1, qual1, seq2, qual2)."""
        n = len(singles) + len(pairs)
        descs = np.zeros(n, dtype=READ_DESC)
        ids = np.zeros(n, dtype=np.uint64)
        chunks_b: List[bytes] = []
        chunks_q: List[bytes] = []
        off = 0
        for i, (rid, s, q) in enumerate(singles):
            assert len(s) == len(q) and len(s) > 0
            ids[i] = rid
            descs[i]["seq_off"][0] = off
            descs[i]["seq_len"][0] = len(s)
            chunks_b.append(s.encode())
            chunks_q.append(q.encode())
            off += len(s)
        for j, (rid, s1, q1, s2, q2) in enumerate(pairs):
            i = len(singles) + j
            assert len(s1) == len(q1) and len(s2) == len(q2) and len(s1) > 0 and len(s2) > 0
            ids[i] = rid
            descs[i]["seq_off"][0] = off
            descs[i]["seq_len"][0] = len(s1)
            off += len(s1)
            descs[i]["seq_off"][1] = off
            descs[i]["seq_len"][1] = len(s2)
            off += len(s2)
            chunks_b += [s1.encode(), s2.encode()]
            chunks_q += [q1.encode(), q2.encode()]
        bases = np.frombuffer(b"".join(chunks_b), dtype=np.uint8).copy()
        quals = np.frombuffer(b"".join(chunks_q), dtype=np.uint8).copy()
        return ReadSet(ids=ids, descs=descs, bases=bases, quals=quals, n_single=len(singles))

    def subset(self, keep: Iterable[int]) -> "ReadSet":
        keep = sorted(set(int(k) for k in keep))
        singles = [(int(self.ids[i]), self.seq(i), self.qual(i)) for i in keep if not self.is_paired(i)]
        pairs = [
            (int(self.ids[i]), self.seq(i, 0), self.qual(i, 0), self.seq(i, 1), self.qual(i, 1))
            for i in keep if self.is_paired(i)
        ]
        return ReadSet.from_lists(singles, pairs)


def _read_fastq_records(path: str) -> List[Tuple[str, str, str]]:
    out = []
    with open(path, "r") as f:
        lines = f.read().split("\n")
    if lines and lines[-1] == "":
        lines.pop()
    for k in range(0, len(lines) - 3, 4):
        if not lines[k].startswith("@"):
            raise ValueError("Read ID does not start with @")
        name = lines[k][1:].split()[0] if lines[k][1:].split() else ""
        out.append((name, lines[k + 1], lines[k + 3]))
    return out


def _parse_id(s: str) -> int:
    """str_to_read_id = strtoul(s, NULL, 0) (src/Types.h:99-102): base auto-detection."""
    s = s.strip()
    try:
        return int(s, 0)
    except ValueError:
        # strtoul parses the longest valid prefix, 0 if none
        digits = ""
        for ch in s:
            if ch.isdigit():
                digits += ch
            else:
                break
        return int(digits) if digits else 0


def load_fastq_set(singles: Optional[str], paired1: Optional[str], paired2: Optional[str]) -> ReadSet:
    """FastqStorage semantics: singles are upper-cased (src/FastqStorage.cpp:123), pairs are taken
    verbatim (:196-197); empty sequences are an error (:143-146,:222-225)."""
    s_list: List[Tuple[int, str, str]] = []
    p_list: List[Tuple[int, str, str, str, str]] = []
    if singles and singles != "None":
        for name, s, q in _read_fastq_records(singles):
            if len(s) == 0:
                raise ValueError("single read with an empty sequence")
            s_list.append((_parse_id(name), s.upper(), q))
    if paired1 and paired1 != "None":
        r1 = _read_fastq_records(paired1)
        r2 = _read_fastq_records(paired2)
        for (n1, s1, q1), (n2, s2, q2) in zip(r1, r2):
            if n1 != n2:
                raise ValueError("Fastq files /1 /2 are not ordered identically")
            if len(s1) == 0 or len(s2) == 0:
                raise ValueError("paired read with an empty sequence")
            p_list.append((_parse_id(n1), s1, q1, s2, q2))
    return ReadSet.from_lists(s_list, p_list)


def write_fastq_set(rs: ReadSet, singles: str, paired1: str, paired2: str) -> None:
    with open(singles, "w") as fs, open(paired1, "w") as f1, open(paired2, "w") as f2:
        for i in range(rs.n_reads):
            rid = int(rs.ids[i])
            if not rs.is_paired(i):
                fs.write("@%d\n%s\n+\n%s\n" % (rid, rs.seq(i), rs.qual(i)))
            else:
                f1.write("@%d\n%s\n+\n%s\n" % (rid, rs.seq(i, 0), rs.qual(i, 0)))
                f2.write("@%d\n%s\n+\n%s\n" % (rid, rs.seq(i, 1), rs.qual(i, 1)))


# ---- overlaps file -------------------------------------------------------------------------------
def candidates_to_lines(cands: np.ndarray, ids: np.ndarray) -> List[str]:
    """Overlap::get_overlap_line (src/Overlap.h:234-237): every numeric field printed, '-' never
    re-emitted for POS2/PERC2/LEN2 (they were folded to 0 by the constructor, :55-59)."""
    out = []
    for c in cands:
        out.append(
            "%d\t%d\t%d\t%d\t%s\t%s\t%s\t%d\t%d\t%d\t%d\t%s\t%s\n"
            % (
                int(ids[c["idx1"]]), int(ids[c["idx2"]]), c["pos1"], c["pos2"], chr(c["ord"]),
                "+" if c["ori1"] else "-", "+" if c["ori2"] else "-", c["perc1"], c["perc2"], c["len1"], c["len2"],
                chr(c["type1"]), chr(c["type2"]),
            )
        )
    return out


def write_overlaps(path: str, cands: np.ndarray, ids: np.ndarray, dash_for_single: bool = True) -> None:
    """Writes the producer-side format (scripts/sfo2overlaps.py:153,186-199): S-S lines carry '-' in
    POS2/PERC2/LEN2."""
    with open(path, "w") as f:
        for c in cands:
            ss = dash_for_single and c["type1"] == ord("s") and c["type2"] == ord("s")
            f.write(
                "%d\t%d\t%d\t%s\t%s\t%s\t%s\t%d\t%s\t%d\t%s\t%s\t%s\n"
                % (
                    int(ids[c["idx1"]]), int(ids[c["idx2"]]), c["pos1"], "-" if ss else str(int(c["pos2"])),
                    chr(c["ord"]), "+" if c["ori1"] else "-", "+" if c["ori2"] else "-", c["perc1"],
                    "-" if ss else str(int(c["perc2"])), c["len1"], "-" if ss else str(int(c["len2"])),
                    chr(c["type1"]), chr(c["type2"]),
                )
            )


def _atoi(s: str) -> int:
    s = s.strip()
    sign = 1
    k = 0
    if k < len(s) and s[k] in "+-":
        sign = -1 if s[k] == "-" else 1
        k += 1
    v = 0
    while k < len(s) and s[k].isdigit():
        v = v * 10 + ord(s[k]) - 48
        k += 1
    return sign * v


def parse_overlaps(path: str, id_to_index: Dict[int, int], max_overlaps: int = 100000000) -> Tuple[np.ndarray, np.ndarray]:
    """The parsing half of EdgeCalculator::construct_edges (src/EdgeCalculator.cpp:581-607, tab-split
    branch) + Overlap's constructor (src/Overlap.h:39-73).  Returns (candidates, 1-based line numbers);
    self-overlaps and lines without exactly 13 fields are skipped like the reference does."""
    recs = []
    lines_no = []
    with open(path, "r") as f:
        for i, line in enumerate(f, start=1):
            if i > max_overlaps:
                break
            t = line.rstrip("\n").strip("\t ")
            fld = t.split("\t")
            if len(fld) != 13:
                continue
            id1, id2 = _parse_id(fld[0]), _parse_id(fld[1])
            if id1 == id2:
                continue
            pos2, perc2, len2 = _atoi(fld[3]), _atoi(fld[8]), _atoi(fld[10])
            if fld[3] == "-":
                pos2 = perc2 = len2 = 0
            recs.append(
                (
                    id_to_index[id1], id_to_index[id2], _atoi(fld[2]), pos2, _atoi(fld[9]), len2, _atoi(fld[7]), perc2,
                    ord(fld[4].replace(" ", "")[0]), 1 if fld[5].strip() == "+" else 0, 1 if fld[6].strip() == "+" else 0,
                    ord(fld[11].strip()[0]), ord(fld[12].strip()[0]), 0,
                )
            )
            lines_no.append(i)
    return np.array(recs, dtype=CANDIDATE), np.array(lines_no, dtype=np.int64)


def prefilter(cands: np.ndarray, min_overlap_len: int, min_overlap_perc: int = 0, relax_PE_edges: bool = False) -> np.ndarray:
    """Vectorised src/EdgeCalculator.cpp:605-635.  Returns int8: 1 = scored, 0 = filtered non-edge
    (written back to nonedge_overlaps.txt, :633-635,:654-660), -1 = silently dropped."""
    c = cands
    perc = np.where(c["perc2"] > 0, (0.5 * (c["perc1"].astype(np.float64) + c["perc2"])).astype(np.uint32), c["perc1"])
    anyp = (c["type1"] == ord("p")) | (c["type2"] == ord("p"))
    ss = (c["type1"] == ord("s")) & (c["type2"] == ord("s"))
    b1 = (c["len1"] >= min_overlap_len) & ss
    b2 = ~b1 & (c["len1"] >= 0.5 * min_overlap_len) & (c["len2"] >= 0.5 * min_overlap_len) & anyp
    b3 = ~b1 & ~b2 & bool(relax_PE_edges) & ((c["len1"].astype(np.int64) + c["len2"]) >= min_overlap_len) & anyp
    inb = b1 | b2 | b3
    out = np.zeros(len(c), dtype=np.int8)
    out[inb & (perc >= min_overlap_perc)] = 1
    out[inb & (perc < min_overlap_perc)] = -1
    out[c["idx1"] == c["idx2"]] = -1
    return out


# ---- FindNextOverlaps -------------------------------------------------------------------------------
@dataclass
class FnoInput:
    """Array form of what SRBuilder::findNextOverlaps reads (src/FindNextOverlaps.cpp:890-913)."""

    visited: np.ndarray       # uint8 [V]
    label: np.ndarray         # uint8 [V]
    vertex_read: np.ndarray   # FNO_READ [V]
    sr_off: np.ndarray        # uint64 [V+1]
    sr_idx: np.ndarray        # uint32
    sr_sub: np.ndarray        # FNO_SUBREAD
    superread: np.ndarray     # FNO_READ
    resolve_orientations: int
    no_inclusions: int
    edges: np.ndarray         # FNO_EDGE, processing order


def fno_lines(ov: np.ndarray) -> List[str]:
    """The reference's overlap line (src/FindNextOverlaps.cpp:122-148): PERC2 is the literal 0."""
    return ["%d\t%d\t%d\t%d\t%s\t%s\t%s\t%d\t%d\t%d\t%d\t%s\t%s" % (
        o["id1"], o["id2"], o["pos1"], o["pos2"], chr(o["ord"]), chr(o["ori1"]), chr(o["ori2"]), o["perc"], o["perc2"], o["len1"],
        o["len2"], chr(o["type1"]), chr(o["type2"])) for o in ov]


def fno_output_file(ov: np.ndarray) -> List[str]:
    """overlaps.txt = std::set<std::string> of the lines: unique, byte-lexicographic (:918,:946-948)."""
    return sorted(set(fno_lines(ov)), key=lambda s: s.encode())


@dataclass
class Fno3Input:
    """Array form of what findNextOverlaps3 reads: per original read (in the reference's iteration
    order) the new reads containing it and its position inside each (src/FindNextOverlaps3.cpp:26-76)."""

    off: np.ndarray        # uint64 [n_originals + 1]
    sr_idx: np.ndarray     # uint32
    sr_pos: np.ndarray     # FNO3_POS
    reads: np.ndarray      # FNO_READ (super-reads, then trivial reads)
    no_inclusions: int
