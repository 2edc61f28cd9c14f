"""Seeded synthetic reads and candidate-overlap producers (host side, numpy).

The reference gets its candidates from rust-overlaps / bwa via scripts/sfo2overlaps.py and
scripts/sam2overlaps.py, none of which is available offline, so the parity tests and the bench
produce the same 13-column records here:

* ``seed_candidates``      exact k-mer seed enumeration on real FASTQ input (savage/example,
                           polyte/example) -- SURVEY Appendix A, extended to all read types and
                           orientations through the window table of src/EdgeCalculator.cpp:199-351.
* ``synth_readset`` + ``geometry_candidates``   reads simulated from known genome coordinates, every
                           TYPE x ORI x ORD case, plus deliberately broken candidates (shifted
                           positions, positions past the read end, N runs, Q=0 bases).
LEN/PERC follow scripts/sfo2overlaps.py:161,190-195.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from .formats import CANDIDATE, ReadSet

_COMP = np.zeros(256, dtype=np.uint8)
for _a, _b in zip(b"ACGTN", b"TGCAN"):
    _COMP[_a] = _b


def revcomp_bytes(a: np.ndarray) -> np.ndarray:
    return _COMP[a[::-1]]


def revcomp(s: str) -> str:
    return revcomp_bytes(np.frombuffer(s.encode(), dtype=np.uint8)).tobytes().decode()


# A "view" = (read index, mate slot, rc flag): one oriented sequence as overlap_score sees it.
View = Tuple[int, int, int]


def window_views(paired1: bool, paired2: bool, ori1: int, ori2: int, ord_: str, r1: int, r2: int):
    """The window table of EdgeCalculator::compute_overlap (src/EdgeCalculator.cpp:199-351):
    returns [(A_view, B_view, 'pos1'|'pos2'), ...] for one candidate."""
    rc1, rc2 = int(not ori1), int(not ori2)
    if not paired1 and not paired2:                       # S-S :199-233
        return [((r1, 0, rc1), (r2, 0, rc2), "pos1")]
    f2, s2 = (0, 1) if ori2 else (1, 0)
    f1, s1 = (0, 1) if ori1 else (1, 0)
    if not paired1 and paired2:                           # S-P :238-253
        return [((r1, 0, rc1), (r2, f2, rc2), "pos1"), ((r1, 0, rc1), (r2, s2, rc2), "pos2")]
    if paired1 and not paired2:                           # P-S :276-291
        return [((r1, f1, rc1), (r2, 0, rc2), "pos1"), ((r2, 0, rc2), (r1, s1, rc1), "pos2")]
    w1 = ((r1, f1, rc1), (r2, f2, rc2), "pos1")          # P-P :316-351
    if ord_ == "1":
        return [w1, ((r1, s1, rc1), (r2, s2, rc2), "pos2")]
    return [w1, ((r2, s2, rc2), (r1, s1, rc1), "pos2")]


def _view_bytes(rs: ReadSet, v: View) -> np.ndarray:
    d = rs.descs[v[0]]
    o, n = int(d["seq_off"][v[1]]), int(d["seq_len"][v[1]])
    a = rs.bases[o:o + n]
    return revcomp_bytes(a) if v[2] else a


def _sfo_len_perc(lenA: int, lenB: int, pos: int) -> Tuple[int, int]:
    ol = min(lenA - pos, lenB)
    perc = min(int(round(100.0 * ol / min(lenA, lenB))), 100)
    return ol, perc


def _mk(r1, r2, pos1, pos2, ord_, ori1, ori2, p1, p2, l1, l2, t1, t2):
    return (r1, r2, pos1, pos2, l1, l2, p1, p2, ord(ord_), ori1, ori2, ord(t1), ord(t2), 0)


def seed_candidates(rs: ReadSet, k: int = 24, max_cands: Optional[int] = None, seed: int = 1,
                    orientations: Sequence[Tuple[int, int]] = ((1, 1), (1, 0), (0, 1), (0, 0))) -> np.ndarray:
    """Every (A_view, B_view, p) with B_view[:k] == A_view[p:p+k], assembled into candidates of all
    read types.  Deterministic given (rs, k, seed)."""
    code = np.full(256, 4, dtype=np.int64)
    for i, ch in enumerate(b"ACGT"):
        code[ch] = i
    views: List[View] = []
    for r in range(rs.n_reads):
        for m in range(2 if rs.is_paired(r) else 1):
            views += [(r, m, 0), (r, m, 1)]
    # prefix k-mer of every view
    prefix: Dict[int, List[int]] = {}
    seqs = []
    for vi, v in enumerate(views):
        a = _view_bytes(rs, v)
        seqs.append(a)
        if len(a) < k:
            continue
        c = code[a[:k]]
        if (c == 4).any():
            continue
        h = 0
        for x in c:
            h = h * 4 + int(x)
        prefix.setdefault(h, []).append(vi)
    keys = np.array(sorted(prefix.keys()), dtype=np.int64)
    hits: Dict[Tuple[View, View], List[int]] = {}
    mask = (1 << (2 * k)) - 1
    for ai, v in enumerate(views):
        a = seqs[ai]
        n = len(a)
        if n < k:
            continue
        c = code[a]
        # rolling 2-bit hash, positions containing N are invalidated
        h = np.zeros(n - k + 1, dtype=np.int64)
        cur = 0
        bad = 0
        for i in range(n):
            x = int(c[i])
            if x == 4:
                bad = k
                x = 0
            cur = ((cur << 2) | x) & mask
            if bad > 0:
                bad -= 1
            if i >= k - 1:
                h[i - k + 1] = cur if bad == 0 else -1
        pos = np.searchsorted(keys, h)
        pos[pos >= len(keys)] = len(keys) - 1
        ok = keys[pos] == h
        for p in np.nonzero(ok)[0]:
            for bi in prefix[int(h[p])]:
                if views[bi][0] == v[0]:
                    continue
                hits.setdefault((v, views[bi]), []).append(int(p))
    rng = np.random.RandomState(seed)
    pairs = sorted({(a[0], b[0]) for (a, b) in hits.keys()})
    out = []
    for (r1, r2) in pairs:
        p1, p2 = rs.is_paired(r1), rs.is_paired(r2)
        for (o1, o2) in orientations:
            for ord_ in (("1", "2") if (p1 and p2) else ("-",)):
                wins = window_views(p1, p2, o1, o2, ord_, r1, r2)
                pos_lists = [hits.get((w[0], w[1])) for w in wins]
                if any(pl is None for pl in pos_lists):
                    continue
                pos1 = pos_lists[0][0]
                if pos1 == 0 and not (p1 or p2) and r1 > r2:
                    continue  # p == 0 pairs once, smaller index first (SURVEY Appendix A)
                lens = []
                for w, pl in zip(wins, pos_lists):
                    la = int(rs.descs[w[0][0]]["seq_len"][w[0][1]])
                    lb = int(rs.descs[w[1][0]]["seq_len"][w[1][1]])
                    lens.append(_sfo_len_perc(la, lb, pl[0]))
                t1, t2 = ("p" if p1 else "s"), ("p" if p2 else "s")
                if len(wins) == 1:
                    out.append(_mk(r1, r2, pos1, 0, "-", o1, o2, lens[0][1], 0, lens[0][0], 0, t1, t2))
                else:
                    out.append(_mk(r1, r2, pos1, pos_lists[1][0], ord_, o1, o2, lens[0][1], lens[1][1], lens[0][0],
                                   lens[1][0], t1, t2))
    c = np.array(out, dtype=CANDIDATE) if out else np.zeros(0, dtype=CANDIDATE)
    if max_cands is not None and len(c) > max_cands:
        keep = np.sort(rng.choice(len(c), size=max_cands, replace=False))
        c = c[keep]
    return c


# ---- simulated reads with known coordinates ---------------------------------------------------------
def _mutate(genome: np.ndarray, rate: float, rng) -> np.ndarray:
    g = genome.copy()
    m = rng.random_sample(len(g)) < rate
    g[m] = (g[m] + rng.randint(1, 4, size=int(m.sum()))) % 4
    return g


def quality_profile(length: int, rng, qmax: int = 41, qset: Optional[Sequence[int]] = None) -> np.ndarray:
    """Position dependent Illumina-like qualities: mean ~36 at the start falling to ~28, values in
    {2, 11..qmax} (SURVEY 8d, C3)."""
    pos = np.arange(length)
    mean = 36.0 - 8.0 * pos / max(length - 1, 1)
    q = np.rint(rng.normal(mean, 4.0)).astype(np.int64)
    q = np.clip(q, 11, qmax)
    low = rng.random_sample(length) < 0.01
    q[low] = 2
    if qset is not None:
        qs = np.array(sorted(qset))
        q = qs[np.abs(qs[None, :] - q[:, None]).argmin(axis=1)]
    return q


_B = np.frombuffer(b"ACGT", dtype=np.uint8)


def _emit(seg: np.ndarray, rng, qmax: int, n_rate: float, qset=None, q_lo: Optional[int] = None) -> Tuple[str, str]:
    """Sequencing model: substitution errors at 10^(-Q/10), N with Q=0 ('!') at n_rate."""
    L = len(seg)
    if q_lo is None:
        q = quality_profile(L, rng, qmax, qset)
    else:
        q = rng.randint(q_lo, qmax + 1, size=L)
    err = rng.random_sample(L) < 10.0 ** (-q / 10.0)
    s = seg.copy()
    s[err] = (s[err] + rng.randint(1, 4, size=int(err.sum()))) % 4
    b = _B[s].copy()
    nn = rng.random_sample(L) < n_rate
    b[nn] = ord("N")
    q = q.copy()
    q[nn] = 0
    return b.tobytes().decode(), (q + 33).astype(np.uint8).tobytes().decode()


class SynthSet:
    """Reads + the genome coordinates they were drawn from (per read: strain, strand of the stored
    sequence(s), [start,end) of mate 0 / mate 1 on the forward genome strand)."""

    def __init__(self, rs: ReadSet, strain, strand, seg0, seg1):
        self.rs = rs
        self.strain = strain
        self.strand = strand
        self.seg0 = seg0
        self.seg1 = seg1


def synth_readset(n_single: int, n_pairs: int, genome_len: int = 3000, n_strains: int = 3, read_len=(120, 260),
                  pair_len=(100, 151), insert=(280, 40), divergence=(0.0, 0.01, 0.03, 0.06), qmax: int = 41,
                  n_rate: float = 0.0005, flip_fraction: float = 0.3, seed: int = 7, qset=None,
                  q_lo: Optional[int] = None) -> SynthSet:
    rng = np.random.RandomState(seed)
    base = rng.randint(0, 4, size=genome_len)
    strains = [base] + [_mutate(base, divergence[min(i, len(divergence) - 1)], rng) for i in range(1, n_strains)]
    singles, pairs = [], []
    strain_a, strand_a, seg0, seg1 = [], [], [], []
    rid = 0
    for _ in range(n_single):
        L = rng.randint(read_len[0], read_len[1] + 1)
        st = rng.randint(0, genome_len - L + 1)
        k = rng.randint(0, n_strains)
        seg = strains[k][st:st + L]
        flip = rng.random_sample() < flip_fraction
        s, q = _emit(seg, rng, qmax, n_rate, qset, q_lo)
        if flip:
            s, q = revcomp(s), q[::-1]
        singles.append((rid, s, q))
        rid += 1
        strain_a.append(k); strand_a.append(-1 if flip else 1); seg0.append((st, st + L)); seg1.append((0, 0))
    for _ in range(n_pairs):
        L1 = rng.randint(pair_len[0], pair_len[1] + 1)
        L2 = rng.randint(pair_len[0], pair_len[1] + 1)
        ins = max(int(rng.normal(insert[0], insert[1])), max(L1, L2))
        ins = min(ins, genome_len)
        st = rng.randint(0, genome_len - ins + 1)
        k = rng.randint(0, n_strains)
        a = strains[k][st:st + L1]
        b = strains[k][st + ins - L2:st + ins]
        flip = rng.random_sample() < flip_fraction
        s1, q1 = _emit(a, rng, qmax, n_rate, qset, q_lo)
        s2, q2 = _emit(b, rng, qmax, n_rate, qset, q_lo)
        if flip:  # the whole fragment seen from the other strand: /1 = rc(right), /2 = rc(left)
            s1, q1, s2, q2 = revcomp(s2), q2[::-1], revcomp(s1), q1[::-1]
            segs = ((st + ins - L2, st + ins), (st, st + L1))
        else:
            segs = ((st, st + L1), (st + ins - L2, st + ins))
        pairs.append((rid, s1, q1, s2, q2))
        rid += 1
        strain_a.append(k); strand_a.append(-1 if flip else 1); seg0.append(segs[0]); seg1.append(segs[1])
    rs = ReadSet.from_lists(singles, pairs)
    return SynthSet(rs, np.array(strain_a), np.array(strand_a), np.array(seg0), np.array(seg1))


def _oriented_segments(ss: SynthSet, r: int, ori: int):
    """Segments of read r in orientation ori, in reading order, with the genome strand they are read
    along: returns (dir, [(mate_slot, gstart, gend), ...]) where dir=+1 reads along increasing
    genome coordinates."""
    d = ss.strand[r] * (1 if ori else -1)
    paired = ss.rs.is_paired(r)
    if not paired:
        return d, [(0, int(ss.seg0[r][0]), int(ss.seg0[r][1]))]
    first, second = (0, 1) if ori else (1, 0)
    segs = {0: ss.seg0[r], 1: ss.seg1[r]}
    return d, [(first, int(segs[first][0]), int(segs[first][1])), (second, int(segs[second][0]), int(segs[second][1]))]


def _offset(d: int, A, B) -> int:
    """pos such that B's first base lies on A[pos] when both are read along direction d."""
    return (B[1] - A[1]) if d > 0 else (A[2] - B[2])


def geometry_candidates(ss: SynthSet, n_target: int = 4000, seed: int = 11, junk_fraction: float = 0.15,
                        min_ov: int = 20) -> np.ndarray:
    """Candidates from true coordinates covering S-S / S-P / P-S / P-P x 4 orientations x ord, then a
    share of perturbed ones (shifted pos, pos past the end)."""
    rng = np.random.RandomState(seed)
    rs = ss.rs
    n = rs.n_reads
    centre = np.array([(min(ss.seg0[r][0], ss.seg1[r][0] if rs.is_paired(r) else ss.seg0[r][0])) for r in range(n)])
    order = np.argsort(centre, kind="stable")
    rank = np.empty(n, dtype=np.int64)
    rank[order] = np.arange(n)
    out = []
    tries = 0
    while len(out) < n_target and tries < 60 * n_target:
        tries += 1
        r1 = int(rng.randint(0, n))
        j = int(rank[r1]) + int(rng.randint(-40, 41))
        if j < 0 or j >= n:
            continue
        r2 = int(order[j])
        if r1 == r2:
            continue
        o1, o2 = int(rng.randint(0, 2)), int(rng.randint(0, 2))
        d1, segs1 = _oriented_segments(ss, r1, o1)
        d2, segs2 = _oriented_segments(ss, r2, o2)
        if d1 != d2:
            o2 = 1 - o2
            d2, segs2 = _oriented_segments(ss, r2, o2)
        p1, p2 = rs.is_paired(r1), rs.is_paired(r2)
        t1, t2 = ("p" if p1 else "s"), ("p" if p2 else "s")

        def lenp(A, B, pos):
            return _sfo_len_perc(A[2] - A[1], B[2] - B[1], pos)

        if not p1 and not p2:
            pos1 = _offset(d1, segs1[0], segs2[0])
            if pos1 < 0 or pos1 > (segs1[0][2] - segs1[0][1]) - min_ov:
                continue
            l, pc = lenp(segs1[0], segs2[0], pos1)
            cand = _mk(r1, r2, pos1, 0, "-", o1, o2, pc, 0, l, 0, t1, t2)
        elif not p1 and p2:
            pos1 = _offset(d1, segs1[0], segs2[0])
            pos2 = _offset(d1, segs1[0], segs2[1])
            LA = segs1[0][2] - segs1[0][1]
            if pos1 < 0 or pos2 < 0 or pos1 > LA - min_ov or pos2 > LA - min_ov:
                continue
            l1, pc1 = lenp(segs1[0], segs2[0], pos1)
            l2, pc2 = lenp(segs1[0], segs2[1], pos2)
            cand = _mk(r1, r2, pos1, pos2, "-", o1, o2, pc1, pc2, l1, l2, t1, t2)
        elif p1 and not p2:
            pos1 = _offset(d1, segs1[0], segs2[0])
            pos2 = _offset(d1, segs2[0], segs1[1])
            if pos1 < 0 or pos2 < 0 or pos1 > (segs1[0][2] - segs1[0][1]) - min_ov or pos2 > (segs2[0][2] - segs2[0][1]) - min_ov:
                continue
            l1, pc1 = lenp(segs1[0], segs2[0], pos1)
            l2, pc2 = lenp(segs2[0], segs1[1], pos2)
            cand = _mk(r1, r2, pos1, pos2, "-", o1, o2, pc1, pc2, l1, l2, t1, t2)
        else:
            pos1 = _offset(d1, segs1[0], segs2[0])
            if pos1 < 0 or pos1 > (segs1[0][2] - segs1[0][1]) - min_ov:
                continue
            pos2 = _offset(d1, segs1[1], segs2[1])
            if pos2 >= 0:
                ord_ = "1"
                if pos2 > (segs1[1][2] - segs1[1][1]) - min_ov:
                    continue
                l2, pc2 = lenp(segs1[1], segs2[1], pos2)
            else:
                ord_ = "2"
                pos2 = -pos2
                if pos2 > (segs2[1][2] - segs2[1][1]) - min_ov:
                    continue
                l2, pc2 = lenp(segs2[1], segs1[1], pos2)
            l1, pc1 = lenp(segs1[0], segs2[0], pos1)
            cand = _mk(r1, r2, pos1, pos2, ord_, o1, o2, pc1, pc2, l1, l2, t1, t2)
        if rng.random_sample() < junk_fraction:
            c = list(cand)
            kind = rng.randint(0, 4)
            if kind == 0:
                c[2] = max(0, c[2] + int(rng.randint(-3, 4)))          # shifted pos1: low score
            elif kind == 1:
                c[3] = c[3] + int(rng.randint(1, 5)) if (p1 or p2) else 0  # shifted pos2
            elif kind == 2:
                c[2] = c[2] + 100000                                     # pos1 past the end: early out
            else:
                c[2], c[3] = int(rng.randint(0, 90)), (int(rng.randint(0, 90)) if (p1 or p2) else 0)
            cand = tuple(c)
        out.append(cand)
    return np.array(out, dtype=CANDIDATE)


# ---- irregular overlaps-file text (ingestion tests) ---------------------------------------------------
def fuzz_overlap_text(cands: np.ndarray, ids: np.ndarray, seed: int = 5, allow_spaces: bool = False, junk: bool = True,
                      self_fraction: float = 0.03) -> bytes:
    """The candidates as overlaps-file lines in every spelling the reference's parser accepts
    (src/Overlap.h:39-73 over strtoul(s, NULL, 0) / atoi): hex / octal / signed / space-padded ids, zero-padded
    numbers, numbers with trailing junk, empty numeric fields for 0, '-' for POS2/PERC2/LEN2, space-decorated
    ORD/ORI/TYPE, outer tabs and spaces; plus lines the loop skips (blank, 12 or 14 fields) and self overlaps.
    No line makes the reference exit."""
    rng = np.random.RandomState(seed)

    def ident(v: int) -> str:
        k = rng.randint(0, 8)
        if allow_spaces:
            k = k if k not in (3, 4) else 0
        if k == 1:
            return hex(v)
        if k == 2:
            return "0" + oct(v)[2:] if v else "0"
        if k == 3:
            return " " + str(v)
        if k == 4:
            return str(v) + " x"
        if k == 5:
            return "+" + str(v)
        if k == 6:
            return "0X%X" % v
        return str(v)

    def num(v: int, may_empty: bool = True) -> str:
        k = rng.randint(0, 8)
        if allow_spaces:
            k = k if k not in (2, 5) else 0
        if k == 1:
            return "00" + str(v)
        if k == 2:
            return " " + str(v)
        if k == 3:
            return str(v) + "abc"
        if k == 4:
            return "+" + str(v)
        if k == 5 and v == 0 and may_empty:
            return ""
        if k == 6:
            return str(v) + ".7"
        return str(v)

    def ch(c: str) -> str:
        if allow_spaces:
            return c
        return [c, c, c, " " + c, c + " ", " " + c + "  "][rng.randint(0, 6)]

    out = []
    for c in cands:
        i1, i2 = int(ids[c["idx1"]]), int(ids[c["idx2"]])
        if rng.rand() < self_fraction:
            i2 = i1
        ss = c["type1"] == ord("s") and c["type2"] == ord("s")
        dash = ss and int(c["pos2"]) == 0 and rng.rand() < 0.6
        f = [ident(i1), ident(i2), num(int(c["pos1"]), False), "-" if dash else num(int(c["pos2"])), ch(chr(c["ord"])),
             ch("+" if c["ori1"] else "-"), ch("+" if c["ori2"] else "-"), num(int(c["perc1"])),
             (["-", "7", "55"][rng.randint(0, 3)] if dash else num(int(c["perc2"]))), num(int(c["len1"])),
             (["-", "9", "120"][rng.randint(0, 3)] if dash else num(int(c["len2"]))), ch(chr(c["type1"])), ch(chr(c["type2"]))]
        if allow_spaces:
            f = [x if x != "" else "0" for x in f]
            seps = ["\t", " ", "  ", "\t\t", " \t "]
            line = f[0]
            for x in f[1:]:
                line += seps[rng.randint(0, len(seps))] + x
        else:
            line = "\t".join(f)
        k = rng.randint(0, 10)
        if k == 0:
            line = "\t" + line
        elif k == 1:
            line = "  " + line + " \t"
        elif k == 2:
            line = line + "\t\t"
        out.append(line)
        if junk:
            k = rng.randint(0, 40)
            if k == 0:
                out.append("")
            elif k == 1:
                out.append(" \t ")
            elif k == 2:
                out.append("\t".join(f[:12]))
            elif k == 3:
                out.append("\t".join(f + ["x"]))
            elif k == 4:
                out.append("# comment")
    text = "\n".join(out)
    if rng.rand() < 0.5:
        text += "\n"
    return text.encode()


# ---- consensus problems (SRBuilder::consensus inputs) -------------------------------------------------
def consensus_problems(seed: int = 1, n_problems: int = 200, read_len=(40, 160), qmax: int = 41, n_rate: float = 0.01):
    """Pile-ups as SRBuilder::sort_vertices hands them to consensus(): a read set (singles and pairs) and, per problem,
    entries (read, mate, rc, pos) with pos ascending from 0, total_len, subreads_needed, error_correction.  Reads
    are error-laden copies of a per-problem template, so most columns agree; some problems have gaps, Q0 / N
    columns, equal positions, a single read, or too little support for error correction."""
    rng = np.random.RandomState(seed)
    singles, pairs, problems = [], [], []

    def emit(seq: str, qual: str) -> tuple:
        """stores the sequence (forward or as its reverse complement) as a single or as a mate; returns (read, mate, rc)"""
        rc = bool(rng.rand() < 0.4)
        s, q = (revcomp(seq), qual[::-1]) if rc else (seq, qual)
        if rng.rand() < 0.3:
            other_len = int(rng.randint(read_len[0], read_len[1]))
            o_s = "".join("ACGT"[k] for k in rng.randint(0, 4, other_len))
            o_q = "".join(chr(33 + k) for k in rng.randint(2, qmax + 1, other_len))
            mate = int(rng.randint(0, 2))
            pairs.append((0, s, q, o_s, o_q) if mate == 0 else (0, o_s, o_q, s, q))
            return ("p", len(pairs) - 1, mate, rc)
        singles.append((0, s, q))
        return ("s", len(singles) - 1, 0, rc)

    for pi in range(n_problems):
        kind = pi % 10
        n = 1 if kind == 7 else int(rng.randint(2, 14))
        T = int(rng.randint(150, 600))
        tmpl = rng.randint(0, 4, T + 400 + 16 * read_len[1] + 900)
        pos, entries = 0, []
        total = 0
        for j in range(n):
            L = int(rng.randint(read_len[0], read_len[1]))
            if j > 0:
                step = 0 if rng.rand() < 0.15 else int(rng.randint(0, 60))
                if kind == 5 and j == n // 2:
                    step += 300                                  # a gap nobody covers
                pos += step
            q = np.clip(np.round(rng.normal(33, 7, L)), 2, qmax).astype(int)
            if kind == 3:
                q[rng.rand(L) < 0.1] = 0                         # Q0 ('!')
            err = rng.rand(L) < 10.0 ** (-q / 10.0)
            b = tmpl[pos:pos + L].copy()
            b[err] = (b[err] + rng.randint(1, 4, int(err.sum()))) % 4
            seq = np.array(list("ACGT"))[b]
            seq[rng.rand(L) < n_rate] = "N"
            entries.append((emit("".join(seq), "".join(chr(33 + int(x)) for x in q)), pos))
            total = max(total, pos + L)
        if kind == 6:
            total += 25                                          # total_len beyond every read
        problems.append(dict(total_len=total, subreads_needed=bool(kind == 8), error_correction=bool(pi % 3 != 0), entries=entries))
    # ids / indices: singles first, then pairs
    singles = [(i, s, q) for i, (_, s, q) in enumerate(singles)]
    pairs = [(len(singles) + i, a, b, c, d) for i, (_, a, b, c, d) in enumerate(pairs)]
    rs = ReadSet.from_lists(singles, pairs)
    for p in problems:
        p["entries"] = [((idx if t == "s" else len(singles) + idx), mate, rc, pos) for (t, idx, mate, rc), pos in p["entries"]]
    return rs, problems


def consensus_problem_text(rs, problems) -> str:
    """The problems as the '--consensus' input of oracle/ref_driver (strings exactly as sort_vertices would pass them)."""
    out = []
    for p in problems:
        out.append("P %d %d %d %d" % (p["total_len"], p["subreads_needed"], p["error_correction"], len(p["entries"])))
        for read, mate, rc, pos in p["entries"]:
            s, q = rs.seq(read, mate), rs.qual(read, mate)
            if rc:
                s, q = revcomp(s), q[::-1]
            out.append("%d %s %s" % (pos, s, q))
    return "\n".join(out) + "\n"


def _render_int(v: np.ndarray, zeros: np.ndarray, plus: np.ndarray) -> np.ndarray:
    """Decimal text of v, right-aligned in a uint8 matrix (one row per value, 0 = no byte): `zeros` leading zeros and a
    '+' before non-negative values where `plus` is set."""
    mag = np.abs(v).astype(np.int64)
    nd = np.ones(len(v), dtype=np.int64)
    t = mag // 10
    while t.any():
        nd += t > 0
        t //= 10
    shown = nd + zeros
    width = int(shown.max(initial=1)) + 1
    m = np.zeros((len(v), width), dtype=np.uint8)
    p10 = np.ones(len(v), dtype=np.int64)
    for j in range(width):                                # j = position from the right
        col = width - 1 - j
        m[:, col] = np.where(j < shown, ord("0") + (mag // p10) % 10, 0)
        sign = np.where(v < 0, ord("-"), np.where(plus, ord("+"), 0))
        m[:, col] = np.where(j == shown, sign, m[:, col])
        if j < 18:
            p10 = p10 * 10
    return m


def make_sfo_text(seed: int, num_singles: int, num_pairs: int, n_lines: int, irregular: bool = False,
                  dup_fraction: float = 0.05, chunk: int = 1 << 20) -> bytes:
    """Seeded SFO text ("idA idB ori OHA OHB OLA OLB K" per line, the overlapper's output that lib/hc_sfo2overlaps reads),
    built with numpy a chunk of lines at a time (oracle/make_golden_sfo.make_sfo writes one line at a time and is meant
    for small fixtures).  Per chunk: overlaps of two paired-end reads as the two lines of their ends (consistent, so that
    the converter matches most of them), single-paired and single-single overlaps (num_singles > 0), a few
    self-overlaps; both orientations, overhangs of either sign, either id first (flipped lines); dup_fraction of the
    lines repeated elsewhere in the chunk.  irregular: separators of spaces and tabs, leading whitespace, '+' signs,
    leading zeros and CRLF line ends, chosen per line."""
    ss = np.random.SeedSequence(seed)
    parts = []
    left = n_lines
    for child in ss.spawn(max(1, (n_lines + chunk - 1) // chunk)):
        if left <= 0:
            break
        c = min(chunk, left)
        left -= c
        parts.append(_sfo_chunk(np.random.default_rng(child), num_singles, num_pairs, c, irregular, dup_fraction))
    return b"".join(parts)


def _sfo_chunk(rng, ns: int, npairs: int, n: int, irregular: bool, dup_fraction: float) -> bytes:
    m = max(1, int(round(n * (1 - dup_fraction))))
    ev = (m + 1) // 2                                      # overlap events of two lines each
    kind = rng.random(ev)
    if npairs == 0:
        kind[:] = 0.95
    elif ns == 0:
        kind[:] = 0.0
    a = rng.integers(0, max(npairs, 1), ev)
    b = (a + 1 + rng.integers(0, max(min(npairs, 200) - 1, 1), ev)) % max(npairs, 1)
    s1 = rng.integers(0, max(ns, 1), ev)
    s2 = (s1 + 1 + rng.integers(0, max(min(ns, 200) - 1, 1), ev)) % max(ns, 1)
    isN = rng.random(ev) < 0.6
    end = np.stack([np.zeros(ev, np.int64), np.ones(ev, np.int64)], 1)                 # (ev, 2): the two lines
    mateB = np.where(isN[:, None], end, 1 - end)
    pp = (ns + a[:, None] + end * npairs, ns + b[:, None] + mateB * npairs)
    sp = (np.repeat(s1[:, None], 2, 1), ns + a[:, None] + end * npairs)
    s_s = (np.stack([s1, s2], 1), np.stack([s2, s1], 1))
    self_ = (np.repeat((ns + a)[:, None], 2, 1), ns + a[:, None] + end * npairs)
    sel = np.select([kind < 0.7, kind < 0.85, kind < 0.99], [0, 1, 2], 3)[:, None]
    idA = np.choose(sel, [pp[0], sp[0], s_s[0], self_[0]]).ravel()[:m]
    idB = np.choose(sel, [pp[1], sp[1], s_s[1], self_[1]]).ravel()[:m]
    if npairs == 0:
        idA, idB = np.stack([s1, s2], 1).ravel()[:m], np.stack([s2, s1], 1).ravel()[:m]
    ori = np.repeat(np.where(isN, ord("N"), ord("I")), 2)[:m].astype(np.uint8)
    oha = rng.integers(-60, 61, m)
    ohb = rng.integers(-60, 61, m)
    ola = rng.integers(20, 151, m)
    olb = ola + rng.integers(-3, 4, m)
    k = rng.integers(0, 4, m)
    swap = rng.random(m) < 0.5                             # the same overlap seen from the other read
    isI = ori == ord("I")
    idA, idB = np.where(swap, idB, idA), np.where(swap, idA, idB)
    oha, ohb = np.where(swap, np.where(isI, ohb, -oha), oha), np.where(swap, np.where(isI, oha, -ohb), ohb)
    ola, olb = np.where(swap, olb, ola), np.where(swap, ola, olb)
    idx = np.concatenate([np.arange(m), rng.integers(0, m, n - m)])
    idx = idx[rng.permutation(n)]
    f = [a_[idx] for a_ in (idA, idB, ori, oha, ohb, ola, olb, k)]
    nf = len(f)
    if irregular:
        zeros = rng.integers(0, 3, (nf, n)) * (rng.random((nf, n)) < 0.1)
        plus = rng.random((nf, n)) < 0.1
        sep_kind = rng.integers(0, 4, (nf, n)) * (rng.random((nf, n)) < 0.3)     # 0 tab, 1 space, 2 two spaces, 3 space tab
        lead = np.where(rng.random(n) < 0.05, ord(" "), 0).astype(np.uint8)
        crlf = rng.random(n) < 0.2
    else:
        zeros = np.zeros((nf, n), np.int64)
        plus = np.zeros((nf, n), bool)
        sep_kind = np.zeros((nf, n), np.int64)
        lead = np.zeros(n, np.uint8)
        crlf = np.zeros(n, bool)
    sep_tab = np.array([[9, 0], [32, 0], [32, 32], [32, 9]], dtype=np.uint8)
    cols = [lead[:, None]]
    for j in range(nf):
        if j:
            cols.append(sep_tab[sep_kind[j]])
        cols.append(f[j][:, None] if j == 2 else _render_int(f[j], zeros[j], plus[j]))
    cols.append(np.where(crlf, 13, 0).astype(np.uint8)[:, None])
    cols.append(np.full((n, 1), 10, np.uint8))
    mat = np.concatenate(cols, axis=1).ravel()
    return mat[mat != 0].tobytes()


def make_sam_text(seed: int, n_single: int, n_pairs: int, refs: Sequence[Tuple[str, int]], irregular: bool = False,
                  chunk: int = 1 << 18) -> Tuple[bytes, bytes, bytes]:
    """Seeded (FASTA, single-end SAM, interleaved paired-end SAM) text of alignments to `refs` ((name, length) pairs),
    what lib/hc_sam2overlaps reads, built with numpy a chunk of lines at a time (oracle/make_golden_sam.make_case writes
    one line at a time and is meant for small fixtures).  The same cases as make_case: soft and hard clips, insertions,
    deletions, reverse strands, unmapped singles and unmapped first ends, pair ends of different orientation, mismatched
    pair ids (q<i>), several references, single-end positions up to 40 past the reference end.  irregular: CRLF line ends,
    multi-character CIGAR operations ("MM", "SS", "=" runs) and alignments further past the reference end, chosen per line.
    (A doubled hard clip, "HH", would count as reference bases but not as read length: overlaps of negative length, on
    which the converter exits.)  Both SAM texts start with an @SQ / @PG header."""
    ss = np.random.SeedSequence(seed)
    r_fa, r_s, r_p = (np.random.default_rng(c) for c in ss.spawn(3))
    fasta = b"".join(b">%s description\n" % n.encode() + _fasta_seq(r_fa, L) for n, L in refs)
    header = b"".join(b"@SQ\tSN:%s\tLN:%d\n" % (n.encode(), L) for n, L in refs) + b"@PG\tID:x\n"
    names = [n.encode() for n, _ in refs]
    lens = np.array([L for _, L in refs], dtype=np.int64)
    out_s, out_p = [header], [header]
    for c0 in range(0, n_single, chunk):
        c = min(chunk, n_single - c0)
        ref = r_s.integers(0, len(refs), c)
        flag = np.array([0, 16, 4])[r_s.choice(3, c, p=[0.55, 0.35, 0.1])]
        pos = r_s.integers(1, lens[ref] + 40)
        if irregular:
            pos = np.where(r_s.random(c) < 0.02, lens[ref] + r_s.integers(0, 400, c), pos)
        out_s.append(_sam_lines(r_s, b"s", np.arange(c0, c0 + c), np.zeros(c, bool), flag, ref, pos, names, irregular))
    for c0 in range(0, n_pairs, chunk):
        c = min(chunk, n_pairs - c0)
        ref = r_p.integers(0, len(refs), c)
        p1 = r_p.integers(1, lens[ref])
        p2 = p1 + r_p.integers(-20, 200, c)
        r = r_p.random(c)
        both_rev = (r >= 0.45) & (r < 0.8)
        f1 = np.select([r < 0.45, r < 0.8, r < 0.9], [0, 16, 0], 4)
        f2 = np.select([r < 0.45, r < 0.8, r < 0.9], [0, 16, 16], 0)
        p1, p2 = np.where(both_rev, np.maximum(p1, p2), p1), np.where(both_rev, np.minimum(p1, p2), p2)
        q = r_p.random(c) <= 0.03
        num = np.repeat(np.arange(c0, c0 + c), 2)
        mism = np.stack([np.zeros(c, bool), q], 1).ravel()
        flag = np.stack([f1, f2], 1).ravel()
        pos = np.maximum(np.stack([p1, p2], 1).ravel(), 1)
        out_p.append(_sam_lines(r_p, b"p", num, mism, flag, np.repeat(ref, 2), pos, names, irregular))
    return fasta, b"".join(out_s), b"".join(out_p)


def _fasta_seq(rng, L: int) -> bytes:
    seq = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, L)]
    rows = [seq[o:o + 70].tobytes() for o in range(0, L, 70)]
    return b"\n".join(rows) + b"\n"


def _text_col(words: Sequence[bytes], pick: np.ndarray) -> np.ndarray:
    """Rows of a uint8 matrix spelling words[pick[i]], 0 = no byte."""
    w = max(1, max(len(x) for x in words))
    tab = np.zeros((len(words), w), dtype=np.uint8)
    for i, x in enumerate(words):
        tab[i, :len(x)] = np.frombuffer(x, dtype=np.uint8)
    return tab[pick]


def _sam_lines(rng, prefix: bytes, num: np.ndarray, mism: np.ndarray, flag: np.ndarray, ref: np.ndarray, pos: np.ndarray,
               names: List[bytes], irregular: bool) -> bytes:
    n = len(num)
    qlen = rng.integers(60, 151, n)
    kind = rng.integers(0, 8, n)
    clip = rng.integers(1, 8, n)
    pre_s, pre_h, post_h = kind == 1, kind == 2, kind == 3
    core = qlen - np.where(pre_s, clip, 0)
    ins = (np.isin(kind, (4, 6)) & (core > 30))
    dl = (np.isin(kind, (5, 7)) & (core > 30))
    a = rng.integers(5, np.maximum(core - 10, 6))
    k_id = np.where(ins, rng.integers(1, 4, n), rng.integers(1, 5, n))
    rest = np.where(ins, core - a - k_id, core - a)
    first = np.where(ins | dl, a, core)
    none = np.zeros(n, np.int64)

    def num_col(v, keep):
        m = _render_int(v, none, np.zeros(n, bool))
        m[~keep] = 0
        return m

    op_m = np.zeros(n, np.int64)                     # 0 "M", 1 "MM", 2 "=", indices into the words below
    op_clip = np.zeros(n, np.int64)                  # 1: a soft clip spelled "SS"
    crlf = np.zeros(n, bool)
    if irregular:
        op_m = np.where(rng.random(n) < 0.05, rng.integers(1, 3, n), 0)
        op_clip = (rng.random(n) < 0.2).astype(np.int64)
        crlf = rng.random(n) < 0.2
    mid = np.where(ins, 0, np.where(dl, 1, 2))       # "I", "D", none
    cols = [
        np.full((n, 1), prefix[0], np.uint8), _text_col([b"", b"q"], mism.astype(np.int64)), num_col(num, np.ones(n, bool)),
        np.full((n, 1), 9, np.uint8), num_col(flag, np.ones(n, bool)), np.full((n, 1), 9, np.uint8),
        _text_col(names, ref), np.full((n, 1), 9, np.uint8), num_col(pos, np.ones(n, bool)), _text_col([b"\t60\t"], none),
        num_col(clip, pre_s | pre_h), _text_col([b"", b"S", b"H", b"SS"], np.where(pre_s, 1 + 2 * op_clip, np.where(pre_h, 2, 0))),
        num_col(first, np.ones(n, bool)), _text_col([b"M", b"MM", b"="], op_m),
        num_col(k_id, ins | dl), _text_col([b"I", b"D", b""], mid),
        num_col(rest, ins | dl), _text_col([b"M", b"MM", b"="], np.where(ins | dl, op_m, 0)) * (ins | dl)[:, None],
        num_col(clip, post_h), _text_col([b"", b"H"], post_h.astype(np.int64)),
        _text_col([b"\t=\t0\t0\t"], none),
    ]
    seq = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, (n, 150), dtype=np.uint8)]
    inside = np.arange(150)[None, :] < qlen[:, None]
    cols.append(np.where(inside, seq, 0).astype(np.uint8))
    cols.append(np.full((n, 1), 9, np.uint8))
    cols.append(np.where(inside, ord("I"), 0).astype(np.uint8))
    cols.append(np.where(crlf, 13, 0).astype(np.uint8)[:, None])
    cols.append(np.full((n, 1), 10, np.uint8))
    mat = np.concatenate(cols, axis=1).ravel()
    return mat[mat != 0].tobytes()
