"""GPU suite: hc_consensus at the decisions its kernel hands to the host, and on the paths random pile-ups miss.

cons_sums (hc_consensus.cu) adds the four column scores bit for bit as the reference does, then evaluates :349-401 of
SRBuilder::consensus_pos with the device's pow / log10.  It marks every column whose outcome could differ from the
host libm's, and hc_cons_final_pos decides the marked columns again on the host.  The marks:

* keep = 1 - p_inc within 64 ulp (EPS) of min_qual, when more than one sequence covers the column;
* p_inc within 1e-3 relative of the kernel's 10^-9.3 (LIM);
* x = -10 log10(p_inc) within 4.35 EPS / p_inc + 1e-9 of a half-integer;
* mx < -290 (the powers approach or reach the subnormal range).

Random pile-ups almost never come near these boundaries, so the columns below sit on them.  They were found by a
deterministic search over columns of 2-4 sequences and are hard-coded.  Cases: the rounding boundary, 10^-9.3,
min_qual (with one sequence, and with one base plus one N), underflow, exact ties, more marked columns than the
kernel's list holds (cols / 64 + 4096) and exactly as many, and the tile-to-problem lookup across empty problems at
1, 255, 256, 257 and 513 columns, with columns covered by more than 65535 sequences (the 16-bit count saturates).

Every GPU case asserts three things: the results equal the pinned restatement (oracle/consensus_oracle.py); they
equal the results under HC_CONS_HOST_ALL=1; and certain <= K <= possible, where K is the number of columns that
hc_consensus reports (HC_CONS_VERBOSE) as re-evaluated on the host.  Both bounds come from host values and the
kernel's criteria: `certain` counts the columns inside half a window, and every column with mx < -290 (exact, as the
scores are); `possible` counts the columns inside twice a window.  test_edge_columns_hit_their_boundaries (no GPU)
checks that every hard-coded column still lies where its case says.
"""
import math
import re

import numpy as np
import pytest

from haploconduct_b200 import capi, formats as F
from haploconduct_b200.workloads import revcomp
from oracle import consensus_oracle as CO
from util import consensus_oracle_results

EPS = 64 * 2.220446049250313e-16        # cons_sums: bound on the relative error of max / total
LIM = 5.011872336272715e-10             # cons_sums: its 10^-9.3 (glibc's pow(10, -9.3) is one ulp lower)
VERBOSE = re.compile(r"hc_consensus: (\d+) of (\d+) columns re-evaluated on the host")


@pytest.fixture(autouse=True, params=["packed", "planar"])
def layout(request, monkeypatch):
    if request.param == "planar":
        monkeypatch.setenv("HC_STORE_LAYOUT", "planar")
    return request.param


# ---- the hard-coded columns: (bases, Phred values), one pair per covering sequence, in list order ------------------
# x = -10 log10(p_inc) within half the kernel's window of a half-integer; x from 81.4999960 to 92.5000312, rounding
# down (x just below .5) and up (just above)
HALF_COLUMNS = [
    ("AAC", (2, 93, 14)), ("AAAC", (20, 40, 44, 29)), ("AAAC", (19, 34, 44, 20)), ("AAAC", (20, 39, 48, 29)),
    ("AAAC", (20, 39, 49, 29)), ("AAAC", (20, 39, 50, 29)), ("AAA", (3, 23, 58)), ("AAAC", (20, 45, 46, 30)),
    ("AAAA", (5, 15, 23, 35)), ("AAAC", (20, 39, 51, 29)), ("AAAC", (20, 36, 54, 28)), ("AAA", (3, 23, 59)),
    ("AAAC", (20, 44, 48, 30)), ("AAA", (21, 30, 31)), ("AAAC", (20, 45, 47, 30)), ("AAAC", (20, 46, 46, 30)),
    ("AAAC", (17, 39, 41, 15)), ("AAAC", (20, 39, 52, 29)), ("AAAC", (20, 23, 58, 18)), ("AAAC", (20, 43, 50, 30)),
    ("AAAC", (20, 36, 55, 28)), ("AAA", (3, 23, 60)), ("AAAC", (20, 44, 49, 30)), ("AAAC", (17, 38, 43, 15)),
    ("AAAC", (20, 45, 48, 30)), ("AAAC", (20, 46, 47, 30)), ("AAAC", (20, 39, 53, 29)),
]
# p_inc within half the kernel's window of 10^-9.3: five above it (x is computed), five below (Phred 93 directly).
# None can lie between glibc's pow(10, -9.3) and LIM: p_inc = 1 - max / total is a multiple of 2^-53 there, and no
# multiple of 2^-53 lies in that one-ulp interval (test_edge_columns_hit_their_boundaries checks this too).
LIM_COLUMNS = [
    ("AAAA", (4, 8, 11, 59)), ("AAAA", (6, 21, 24, 29)), ("AAAC", (10, 16, 59, 2)), ("AAAC", (9, 30, 60, 15)),
    ("AAC", (6, 88, 5)),
    ("AAC", (28, 68, 8)), ("AAAC", (3, 29, 59, 5)), ("AAAC", (2, 28, 60, 3)), ("AAAA", (3, 13, 18, 48)),
    ("AAC", (18, 77, 7)),
]
# called with min_qual = keep and one ulp to either side; the last two: one sequence only (the min_qual test does
# not apply), and one base plus one N (it does: N counts toward the sequences covering the column)
MINQ_COLUMNS = [("AC", (30, 10)), ("AAC", (20, 25, 12)), ("AAAC", (30, 30, 30, 20)), ("GT", (13, 7)), ("A", (20,)),
                ("AN", (25, 25))]
# Phred-93 reads split between A and C (interleaved or in two blocks), and Phred-0 reads: mx in [-308, -290);
# mx in [-324, -308), where the largest power is subnormal; mx < -324, where every power is 0; all four sums -inf;
# exactly one sum -inf
UNDERFLOW_COLUMNS = [
    ("AC" * 30, (93,) * 60), ("A" * 31 + "C" * 31, (93,) * 62), ("A" * 30 + "C" * 32, (93,) * 62),
    ("AC" * 32, (93,) * 64), ("A" * 33 + "C" * 33, (93,) * 66),
    ("AC" * 34, (93,) * 68), ("A" * 34 + "C" * 34, (93,) * 68),
    ("ACGT", (0, 0, 0, 0)),
    ("AC", (0, 30)), ("GAA", (0, 20, 20)),
]
# exact maxima: A=C, T=C (twice), C=G, A=T=C=G (twice); the reference picks the first of A, T, C, G
TIE_COLUMNS = [("AC", (20, 20)), ("CT", (20, 20)), ("TC", (33, 33)), ("GC", (35, 35)), ("ACGT", (30, 30, 30, 30)),
               ("GTCA", (30, 30, 30, 30))]


def column_scores(pairs):
    """{base: score} as cons_sums and SRBuilder::consensus_pos add them: in list order, N contributing nothing."""
    s = dict.fromkeys("ACTG", 0.0)
    for b, Q in pairs:
        if b == "N":
            continue
        p = CO.phred_to_prob(Q)
        hit, miss = (math.log10(1 - p) if p < 1 else float("-inf")), math.log10(p / 3.0)
        for k in s:
            s[k] += hit if k == b else miss
    return s


def host_terms(pairs):
    """(mx, p_inc, x) with the host libm; p_inc None when no base contributed or the powers sum to 0, x None when
    p_inc is not positive."""
    s = column_scores(pairs)
    mx = max(s["A"], s["T"], s["C"], s["G"])
    total = math.pow(10.0, s["A"]) + math.pow(10.0, s["T"]) + math.pow(10.0, s["C"]) + math.pow(10.0, s["G"])
    if mx == 0 or total == 0.0:
        return mx, None, None
    p_inc = 1 - math.pow(10.0, mx) / total
    return mx, p_inc, (-10 * math.log10(p_inc) if p_inc > 0 else None)


def in_windows(pairs, min_qual, f):
    """Whether the column lies within f times one of cons_sums's windows (mx < -290 is exact and counts for any f)."""
    mx, p, x = host_terms(pairs)
    if mx == 0:
        return False
    if mx < -290.0:
        return True
    near_q = len(pairs) > 1 and abs((1 - p) - min_qual) <= f * EPS
    near_lim = abs(p - LIM) <= f * 1e-3 * LIM
    near_half = x is not None and abs(x - math.floor(x) - 0.5) <= f * (4.35 * EPS / p + 1e-9)
    if f <= 1:
        # the last two tests are certain only where every evaluation reaches them: keep clearly >= min_qual, p_inc
        # clearly >= 10^-9.3 for the half-integer test
        past_q = len(pairs) <= 1 or (1 - p) - min_qual > EPS
        return near_q or (past_q and (near_lim or (near_half and p > LIM * 1.001)))
    return near_q or near_lim or near_half


def half_window(pairs):
    mx, p, x = host_terms(pairs)
    return abs(x - math.floor(x) - 0.5) / (4.35 * EPS / p + 1e-9)


# ---- pile-ups ----------------------------------------------------------------------------------------------------
class Pileups:
    """A read set and consensus problems.  Read j of a problem is a single, mate 0 or mate 1 of a pair (j % 4: 0 and 1
    single, 2 mate 0, 3 mate 1), and stored as its reverse complement with reversed qualities when j % 3 == 1, so the
    device reads the reverse-strand slot.  The other mate of a pair repeats the read's qualities over 'A's, which
    adds no quality value to the store."""

    def __init__(self):
        self.singles, self.pairs, self.problems = [], [], []

    def _emit(self, j, seq, qual):
        rc = j % 3 == 1
        s, q = (revcomp(seq), qual[::-1]) if rc else (seq, qual)
        if j % 4 < 2:
            self.singles.append((s, q))
            return ("s", len(self.singles) - 1, 0, rc)
        mate = j % 4 - 2
        other = ("A" * len(q), q)
        self.pairs.append((s, q) + other if mate == 0 else other + (s, q))
        return ("p", len(self.pairs) - 1, mate, rc)

    def add_problem(self, reads, total_len, error_correction=False, subreads_needed=False):
        """reads: [(pos, bases, Phred values)], pos ascending from 0."""
        ent = [self._emit(j, b, "".join(chr(33 + q) for q in qs)) + (pos,) for j, (pos, b, qs) in enumerate(reads)]
        self.problems.append(dict(total_len=total_len, subreads_needed=subreads_needed, error_correction=error_correction,
                                  entries=ent))

    def add_columns(self, columns, **kw):
        """One problem per number of covering sequences k: k reads of length L at column 0, read j carrying the j-th
        pair of each of the problem's L columns."""
        by_k = {}
        for bases, quals in columns:
            by_k.setdefault(len(bases), []).append((bases, quals))
        for k, cols in by_k.items():
            reads = [(0, "".join(c[0][j] for c in cols), [c[1][j] for c in cols]) for j in range(k)]
            self.add_problem(reads, len(cols), **kw)

    def build(self):
        ns = len(self.singles)
        rs = F.ReadSet.from_lists([(i, s, q) for i, (s, q) in enumerate(self.singles)],
                                  [(ns + i,) + p for i, p in enumerate(self.pairs)])
        probs = [dict(p, entries=[((i if t == "s" else ns + i), m, rc, pos) for t, i, m, rc, pos in p["entries"]])
                 for p in self.problems]
        return rs, probs


def pileup(columns, **kw):
    b = Pileups()
    b.add_columns(columns, **kw)
    return b.build()


def device_columns(rs, problems):
    """Every column cons_sums evaluates, as the (base, Phred) pairs of the sequences covering it in list order."""
    for p in problems:
        seqs = []
        for read, mate, rc, pos in p["entries"]:
            s, q = rs.seq(read, mate), rs.qual(read, mate)
            seqs.append((pos, revcomp(s) if rc else s, q[::-1] if rc else q))
        for c in range(p["total_len"]):
            yield [(s[c - pos], ord(q[c - pos]) - 33) for pos, s, q in seqs if pos <= c < pos + len(s)]


def mark_bounds(rs, problems, min_qual):
    lo = hi = 0
    for pairs in device_columns(rs, problems):
        lo += in_windows(pairs, min_qual, 0.5)
        hi += in_windows(pairs, min_qual, 2.0)
    return lo, hi


def check_call(st, rs, problems, min_clique_size, min_qual, capfd, monkeypatch):
    """hc_consensus against the restatement and against HC_CONS_HOST_ALL; K within the bounds.  Returns (K, N).

    hc_consensus reports the columns the host decided: the marked ones while the list of N / 64 + 4096 holds them
    all, every column (K = N) once there are more marks than that."""
    want = consensus_oracle_results(rs, problems, min_clique_size, min_qual)
    lo, hi = mark_bounds(rs, problems, min_qual)
    monkeypatch.setenv("HC_CONS_VERBOSE", "1")
    capfd.readouterr()
    got = st.consensus(problems, min_clique_size, min_qual)
    lines = VERBOSE.findall(capfd.readouterr().err)
    monkeypatch.setenv("HC_CONS_HOST_ALL", "1")
    host = st.consensus(problems, min_clique_size, min_qual)
    monkeypatch.delenv("HC_CONS_HOST_ALL")
    assert got == want
    assert host == want
    assert len(lines) == 1, lines
    K, N = int(lines[0][0]), int(lines[0][1])
    assert N == sum(p["total_len"] for p in problems)
    cap = N // 64 + 4096
    if lo > cap:                       # more certain marks than the list holds
        assert K == N, (lo, K, N)
    elif hi <= cap:                    # the list holds every possible mark
        assert lo <= K <= hi, (lo, K, hi)
        if lo == hi:                   # every column certain or clearly outside all windows
            assert K == lo
    else:
        assert lo <= K <= hi or K == N, (lo, K, hi, N)
    return K, N


# ---- layout and overflow pile-ups ----------------------------------------------------------------------------------
CAP_COLS = 8192                       # marked-list capacity cols / 64 + 4096 = 4224 at 8192 columns, 4225 at 8256
FILL_COLS = 64


def overflow_pileups():
    """Problem 0: 62 Phred-93 reads over 8192 columns, 4225 of them with mx in [-308, -290) (certain marks, and not
    'N' on the host), spread over the problem; the others all one base (p_inc = 0, outside every window).
    Problem 1: 64 columns of two agreeing Phred-93 reads, outside every window."""
    n_marked = CAP_COLS // 64 + 4096 + 1
    kinds = ["AC" * 31, "A" * 31 + "C" * 31, "A" * 30 + "C" * 32]
    cols = []
    for i in range(CAP_COLS):
        if (i * n_marked) % CAP_COLS < n_marked:      # n_marked is odd: exactly n_marked columns
            cols.append((kinds[i % 3], (93,) * 62))
        else:
            cols.append(("ACGT"[i % 4] * 62, (93,) * 62))
    b = Pileups()
    b.add_columns(cols)
    b.add_columns([("ACGT"[i % 4] * 2, (93, 93)) for i in range(FILL_COLS)])
    return b.build(), n_marked


def layout_pileups(error_correction):
    """Problems of 1, 255, 256, 257 and 513 columns between problems of none (with and without sequences), each
    covered from column 0 to its end by a first read, with five more reads at seeded positions.  The two one-column
    problems are covered by 70000 and by 65536 reads of length 1: the 16-bit count saturates at 65535 (a count that
    wrapped would give 4464 and 0, the second 'nobody covers the column')."""
    rng = np.random.RandomState(7)
    b = Pileups()

    def rnd(n):
        bases = "".join("ACGTN"[k] for k in rng.choice(5, n, p=[0.24, 0.24, 0.24, 0.24, 0.04]))
        return bases, [int(q) for q in rng.randint(2, 41, n)]

    def covered(total, **kw):
        reads = [(0,) + rnd(total)]
        for pos in sorted(rng.randint(0, total, 5)):
            reads.append((int(pos),) + rnd(int(rng.randint(1, total - pos + 1))))
        b.add_problem(reads, total, error_correction=error_correction, **kw)

    def deep(n, base):
        b.add_problem([(0, "N" if j % 7 == 3 else base, [40]) for j in range(n)], 1, error_correction=error_correction)

    b.add_problem([], 0, error_correction=error_correction)
    deep(70000, "A")
    b.add_problem([], 0, error_correction=error_correction)
    covered(255)
    covered(256)
    b.add_problem([(0, "ACG", [20, 20, 20])], 0, error_correction=error_correction)
    covered(257, subreads_needed=True)
    deep(65536, "G")
    b.add_problem([], 0, error_correction=error_correction)
    covered(513)
    b.add_problem([], 0, error_correction=error_correction)
    return b.build()


# ---- GPU cases -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_rounding_boundary(built_lib, capfd, monkeypatch):
    rs, probs = pileup(HALF_COLUMNS)
    with capi.Store(rs) as st:
        K, _ = check_call(st, rs, probs, 1, 0.5, capfd, monkeypatch)
    assert K == len(HALF_COLUMNS)


@pytest.mark.gpu
def test_near_ten_to_minus_9_3(built_lib, capfd, monkeypatch):
    rs, probs = pileup(LIM_COLUMNS)
    with capi.Store(rs) as st:
        K, _ = check_call(st, rs, probs, 1, 0.5, capfd, monkeypatch)
    assert K == len(LIM_COLUMNS)


@pytest.mark.gpu
def test_min_qual_boundary(built_lib, capfd, monkeypatch):
    """min_qual = the host's 1 - p_inc of one column and one ulp to either side; the 'N' decision flips where the
    restatement's does (test_edge_columns_hit_their_boundaries: between keep and the ulp above, more than one
    sequence only)."""
    rs, probs = pileup(MINQ_COLUMNS)
    with capi.Store(rs) as st:
        for bases, quals in MINQ_COLUMNS:
            keep = 1 - host_terms(list(zip(bases, quals)))[1]
            for mq in (math.nextafter(keep, 0.0), keep, math.nextafter(keep, 1.0)):
                check_call(st, rs, probs, 1, mq, capfd, monkeypatch)


@pytest.mark.gpu
def test_underflow(built_lib, capfd, monkeypatch):
    rs, probs = pileup(UNDERFLOW_COLUMNS)
    with capi.Store(rs) as st:
        check_call(st, rs, probs, 1, 0.5, capfd, monkeypatch)


@pytest.mark.gpu
def test_ties(built_lib, capfd, monkeypatch):
    rs, probs = pileup(TIE_COLUMNS)
    with capi.Store(rs) as st:
        check_call(st, rs, probs, 1, 0.0, capfd, monkeypatch)


@pytest.mark.gpu
def test_marked_list_overflow(built_lib, capfd, monkeypatch):
    """One marked column more than the list holds: every column goes back to the host (K = N).  Exactly as many (the
    64-column problem raises the capacity by one): the list holds them all (K = the capacity)."""
    (rs, probs), n_marked = overflow_pileups()
    assert [p["total_len"] for p in probs] == [CAP_COLS, FILL_COLS]
    with capi.Store(rs) as st:
        K, N = check_call(st, rs, probs[:1], 1, 0.5, capfd, monkeypatch)
        assert n_marked == N // 64 + 4096 + 1 and K == N
        K, N = check_call(st, rs, probs, 1, 0.5, capfd, monkeypatch)
        assert K == n_marked == N // 64 + 4096


@pytest.mark.gpu
@pytest.mark.parametrize("error_correction", [False, True])
def test_tile_lookup_and_saturated_count(built_lib, capfd, monkeypatch, error_correction):
    rs, probs = layout_pileups(error_correction)
    with capi.Store(rs) as st:
        check_call(st, rs, probs, 3, 0.9, capfd, monkeypatch)


# ---- the cases still reach their boundaries (no GPU) ---------------------------------------------------------------
def _pairs(col):
    return list(zip(*col))


def test_edge_columns_hit_their_boundaries():
    # LIM is one ulp above glibc's pow(10, -9.3), and no multiple of 2^-53 (the grid of p_inc there) lies between them
    glibc = math.pow(10.0, -9.3)
    assert math.nextafter(glibc, 1.0) == LIM
    assert math.floor(LIM * 2.0 ** 53) < glibc * 2.0 ** 53

    for col in HALF_COLUMNS:
        assert half_window(_pairs(col)) <= 0.5, col
        assert in_windows(_pairs(col), 0.5, 0.5) and host_terms(_pairs(col))[1] > LIM * 1.001, col
    xs = [host_terms(_pairs(c))[2] for c in HALF_COLUMNS]
    assert len(set(round(x, 6) for x in xs)) == len(HALF_COLUMNS) >= 20
    assert any(x % 1 < 0.5 for x in xs) and any(x % 1 > 0.5 for x in xs)

    above = 0
    for col in LIM_COLUMNS:
        p = host_terms(_pairs(col))[1]
        assert abs(p - LIM) <= 0.5e-3 * LIM, col
        above += p >= LIM
    assert above == 5 and len(LIM_COLUMNS) - above == 5

    for bases, quals in MINQ_COLUMNS:
        q = "".join(chr(33 + x) for x in quals)
        keep = 1 - host_terms(_pairs((bases, quals)))[1]
        got = [CO.consensus_pos(bases, q, mq)[1] for mq in (math.nextafter(keep, 0.0), keep, math.nextafter(keep, 1.0))]
        flips = len(bases) > 1
        assert got[0] != "N" and got[1] != "N" and (got[2] == "N") == flips, (bases, got)
    assert [len(b) for b, _ in MINQ_COLUMNS[-2:]] == [1, 2] and MINQ_COLUMNS[-1][0][1] == "N"

    mxs = [host_terms(_pairs(c))[0] for c in UNDERFLOW_COLUMNS]
    assert sum(-308 <= mx < -290 for mx in mxs) == 3
    assert sum(-324 <= mx < -308 for mx in mxs) == 2
    assert sum(mx < -324 for mx in mxs) == 3                       # two splits, and the four -inf sums
    for bases, quals in UNDERFLOW_COLUMNS:
        s = column_scores(_pairs((bases, quals)))
        n_inf = sum(v == float("-inf") for v in s.values())
        mx = max(s.values())
        res = CO.consensus_pos(bases, "".join(chr(33 + x) for x in quals), 0.5)
        if mx < -324:
            assert res == (True, "N", "$"), bases
        elif mx < -290:
            assert res[0] and res[1] != "N", bases                 # the host decides a base: the mark matters
        else:
            assert n_inf == 1, bases
        if set(quals) == {0} and len(bases) == 4:
            assert n_inf == 4
    assert sum(sum(v == float("-inf") for v in column_scores(_pairs(c)).values()) == 1 for c in UNDERFLOW_COLUMNS) == 2

    for bases, quals in TIE_COLUMNS:
        s = column_scores(_pairs((bases, quals)))
        mx = max(s.values())
        tied = [b for b in "ATCG" if s[b] == mx]
        assert len(tied) == len(set(bases)) >= 2, (bases, s)
        assert CO.consensus_pos(bases, "".join(chr(33 + x) for x in quals), 0.0)[1] == tied[0]
    tie_sets = [frozenset(b for b in "ATCG" if column_scores(_pairs(c))[b] == max(column_scores(_pairs(c)).values()))
                for c in TIE_COLUMNS]
    assert {frozenset("AC"), frozenset("TC"), frozenset("CG"), frozenset("ATCG")} <= set(tie_sets)

    # the packed layout holds at most 63 quality values: every case's store must fit it
    for cols in (HALF_COLUMNS, LIM_COLUMNS, MINQ_COLUMNS, UNDERFLOW_COLUMNS, TIE_COLUMNS):
        assert len({q for _, qs in cols for q in qs}) <= 63

    # overflow: exactly one more certain mark than the list holds at 8192 columns, none possible elsewhere
    (rs, probs), n_marked = overflow_pileups()
    assert n_marked == CAP_COLS // 64 + 4096 + 1
    assert mark_bounds(rs, probs[:1], 0.5) == (n_marked, n_marked)
    assert mark_bounds(rs, probs[1:], 0.5) == (0, 0)
    assert n_marked == (CAP_COLS + FILL_COLS) // 64 + 4096

    # layout: problem sizes, empty problems between them, column depths above 65535
    rs, probs = layout_pileups(False)
    assert [p["total_len"] for p in probs] == [0, 1, 0, 255, 256, 0, 257, 1, 0, 513, 0]
    assert [len(p["entries"]) for p in probs if p["total_len"] == 1] == [70000, 65536]
    assert len(np.unique(rs.quals)) <= 63
