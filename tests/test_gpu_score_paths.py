"""GPU suite: the shapes of hc_score_kernel the other files do not reach, against the plain-C oracle.

* whole-warp walks of big candidates (>= HC_BIG_CHUNKS = 64 lane-chunks of 32 positions) and the lane-chunk rounds
  (at most HC_PARTMAX = 512 lane-chunks per round, so a tile with more takes several), in the packed layout too;
* N, void and the largest fixed-point addends inside long windows;
* void decided differently in the two orders of a quality pair (the reference-order pass decides);
* the switch between the packed (<= 63 quality values) and the three-plane layout;
* the 16-bit counts of the small edge records (HC_EDGE_OVERFLOW);
* both modes of the reference-order pass on long windows;
* the cases in the order of an overlaps file (sorted by read), as plain and as run-encoded records.

Every read set is cut from a seeded random genome, so each window's length and content is known by construction.
test_cases_hit_their_shapes (no GPU) checks from geometry and oracle output alone that every case still reaches the
shape it is named for.  Bar: that of test_gpu_parity._against_oracle (classes, lists in input order, pos3/pos4,
counts, statuses and mismatch rates bit-exact, scores within 1e-6); with HC_FLAG_EXACT_EDGE_SCORES every accepted edge
is re-added in the reference's order and matches the oracle's score within 1e-14 (the device exp).
"""
import functools
import math

import numpy as np
import pytest

from haploconduct_b200 import capi, formats as F
from oracle import oracle as O
from util import assert_results_match

BIG_CHUNKS, PARTMAX = 64, 512          # HC_BIG_CHUNKS, HC_PARTMAX (hc_kernels.cuh)
FX_SCALE = 2.0 ** 22                   # HC_FX_SCALE
# reference-order pass on a B200 (148 SMs): queued candidates below which every launch configuration of hc_exact_kernel
# gives each one a warp, and above which every one gives each a thread
WARP_MODE_MAX = 148 * 256 // 32
THREAD_MODE_MIN = 148 * 8 * 128 // 32


@pytest.fixture(autouse=True, params=["packed", "planar"])
def store_layout(request, monkeypatch):
    """Every test runs on both device layouts: the packed one (one byte per base, used when the store
    has <= 63 distinct quality values) and the three-plane one (forced through HC_STORE_LAYOUT)."""
    monkeypatch.setenv("HC_STORE_LAYOUT", "planar" if request.param == "planar" else "auto")
    return request.param


# ---- read sets cut from a genome -----------------------------------------------------------------------
_BASES = np.frombuffer(b"ACGTN", dtype=np.uint8)
_COMP = str.maketrans("ACGTN", "TGCAN")


def _text(codes):
    return _BASES[np.asarray(codes)].tobytes().decode()


def _qtext(q):
    return (np.asarray(q) + 33).astype(np.uint8).tobytes().decode()


def _rc(codes):
    out = np.asarray(codes)[::-1].copy()
    m = out < 4
    out[m] = 3 - out[m]
    return out


def _chunks(L):
    return (np.asarray(L) + 31) // 32


class Case:
    def __init__(self, name, rs, cands, params, **meta):
        self.name, self.rs, self.cands, self.params, self.meta = name, rs, cands, params, meta


class _Builder:
    """Reads given by their views in the candidate's orientation (stored reverse-complemented for orientation '-'), and
    S-S / P-P candidates between them.  Codes 0-3 = ACGT, 4 = N."""

    def __init__(self, seed, genome_len):
        self.rng = np.random.RandomState(seed)
        self.genome = self.rng.randint(0, 4, size=genome_len).astype(np.uint8)
        self.singles, self.pairs, self.cands = [], [], []

    def cut(self, start, n, mut=0.0):
        s = self.genome[start:start + n].copy()
        assert len(s) == n and start >= 0
        if mut:
            m = self.rng.random_sample(n) < mut
            s[m] = (s[m] + 1 + self.rng.randint(0, 3, size=int(m.sum()))) % 4
        return s

    def qual(self, n, lo=20, hi=42):
        return self.rng.randint(lo, hi, size=n)

    def start(self, n):
        return int(self.rng.randint(0, len(self.genome) - n + 1))

    def single(self, seq, q, rc=False):
        if rc:
            seq, q = _rc(seq), np.asarray(q)[::-1]
        self.singles.append((_text(seq), _qtext(q)))
        return ("s", len(self.singles) - 1, 0 if rc else 1)

    def pair(self, first, qf, second, qs, rc=False):
        """views (first, second) of a paired read in orientation '+', or '-' when rc"""
        if rc:
            m0, q0, m1, q1 = _rc(second), np.asarray(qs)[::-1], _rc(first), np.asarray(qf)[::-1]
        else:
            m0, q0, m1, q1 = first, qf, second, qs
        self.pairs.append((_text(m0), _qtext(q0), _text(m1), _qtext(q1)))
        return ("p", len(self.pairs) - 1, 0 if rc else 1)

    def cand(self, r1, r2, pos1, pos2=0, ord_="-"):
        self.cands.append((r1, r2, pos1, pos2, ord_))

    def _views(self, L, pos, extra, mut, q):
        """A (pos + L + extra) and B (L) cut so that A[pos + i] lies over B[i]: a window of exactly L positions"""
        s = self.start(pos + L + extra)
        A, B = self.cut(s, pos + L + extra, mut), self.cut(s + pos, L, mut)
        return A, self.qual(len(A), *q), B, self.qual(L, *q)

    def ss(self, L, pos=0, extra=0, rc=(False, False), mut=0.002, q=(20, 42), nA=(), nB=()):
        """S-S candidate with one window of L positions; nA / nB: N at these window positions on the A / B side"""
        A, qa, B, qb = self._views(L, pos, extra, mut, q)
        for p in nA:
            A[pos + p] = 4
        for p in nB:
            B[p] = 4
        self.cand(self.single(A, qa, rc[0]), self.single(B, qb, rc[1]), pos)

    def pp(self, L0, L1, pos=(0, 0), ord_="1", rc=(False, False), mut=0.002, q=(20, 42)):
        """P-P candidate with windows of L0 and L1 positions"""
        a0, qa0, b0, qb0 = self._views(L0, pos[0], int(self.rng.randint(0, 20)), mut, q)
        a1, qa1, b1, qb1 = self._views(L1, pos[1], int(self.rng.randint(0, 20)), mut, q)
        if ord_ == "1":            # window 2: second of read 1 over second of read 2
            r1, r2 = self.pair(a0, qa0, a1, qa1, rc[0]), self.pair(b0, qb0, b1, qb1, rc[1])
        else:                      # ord 2: second of read 2 over second of read 1
            r1, r2 = self.pair(a0, qa0, b1, qb1, rc[0]), self.pair(b0, qb0, a1, qa1, rc[1])
        self.cand(r1, r2, pos[0], pos[1], ord_)

    def oor(self, lenA=300):
        """pos >= len(A): HC_WIN_POS_OOR, no lane-chunks"""
        A = self.cut(self.start(lenA), lenA)
        B = self.cut(self.start(100), 100)
        self.cand(self.single(A, self.qual(lenA)), self.single(B, self.qual(100)), lenA + int(self.rng.randint(0, 40)))

    def finish(self, name, params, **meta):
        ns = len(self.singles)
        rs = F.ReadSet.from_lists([(i, s, q) for i, (s, q) in enumerate(self.singles)],
                                  [(ns + j,) + p for j, p in enumerate(self.pairs)])
        c = np.zeros(len(self.cands), dtype=F.CANDIDATE)
        idx = lambda r: r[1] if r[0] == "s" else ns + r[1]
        for k, (r1, r2, p1, p2, od) in enumerate(self.cands):
            c[k] = (idx(r1), idx(r2), p1, p2, 1, 0, 50, 0, ord(od), r1[2], r2[2], ord(r1[0]), ord(r2[0]), 0)
        return Case(name, rs, c, params, **meta)


def _views(rs, c):
    """[(A, qA, B, qB, pos)] per window of an S-S or P-P candidate, laid out like src/EdgeCalculator.cpp:199-351"""
    def view(i, mate, rc):
        s, q = rs.seq(i, mate), rs.qual(i, mate)
        return (s.translate(_COMP)[::-1], q[::-1]) if rc else (s, q)
    i1, i2, o1, o2 = int(c["idx1"]), int(c["idx2"]), int(c["ori1"]) != 0, int(c["ori2"]) != 0
    if not rs.is_paired(i1) and not rs.is_paired(i2):
        return [view(i1, 0, not o1) + view(i2, 0, not o2) + (int(c["pos1"]),)]
    assert rs.is_paired(i1) and rs.is_paired(i2)
    f1, s1 = view(i1, 0 if o1 else 1, not o1), view(i1, 1 if o1 else 0, not o1)
    f2, s2 = view(i2, 0 if o2 else 1, not o2), view(i2, 1 if o2 else 0, not o2)
    return [f1 + f2 + (int(c["pos1"]),), (s1 + s2 if c["ord"] == ord("1") else s2 + s1) + (int(c["pos2"]),)]


def _window_lengths(rs, cands):
    """[n, 2] window lengths (src/EdgeCalculator.cpp:86-88; 0 for pos >= len(A) and for an unused second window)"""
    out = np.zeros((len(cands), 2), dtype=np.int64)
    for k, c in enumerate(cands):
        for w, (A, _, B, _, pos) in enumerate(_views(rs, c)):
            out[k, w] = min(len(A) - pos, len(B)) if pos < len(A) else 0
    return out


def _n_positions(rs, c):
    """per window: (window positions with N on the A side, ... on the B side)"""
    out = []
    for A, _, B, _, pos in _views(rs, c):
        L = min(len(A) - pos, len(B)) if pos < len(A) else 0
        a = np.frombuffer(A[pos:pos + L].encode(), dtype=np.uint8)
        b = np.frombuffer(B[:L].encode(), dtype=np.uint8)
        out.append((set(np.nonzero(a == ord("N"))[0].tolist()), set(np.nonzero(b == ord("N"))[0].tolist())))
    return out


def _tile_chunks(rs, cands):
    """per tile of 32 candidates: (lane-chunks per candidate, lane-chunks the rounds deal out = those of candidates
    below HC_BIG_CHUNKS)"""
    ct = _chunks(_window_lengths(rs, cands)).sum(axis=1)
    out = []
    for t in range(0, len(ct), 32):
        x = ct[t:t + 32]
        out.append((x, int(x[(x > 0) & (x < BIG_CHUNKS)].sum())))
    return out


def _p_mismatch(qa, qb):
    """p of a mismatch with quality qa on the A side and qb on the B side: the reference's expression (src/EdgeCalculator.cpp:44),
    which is not bit-symmetric"""
    p1, p2 = O.lib().hco_phred_to_prob(qa), O.lib().hco_phred_to_prob(qb)
    return p1 * (1 - p2) / 3.0 + p2 * (1 - p1) / 3.0 + (2 / 9.0) * p1 * p2


# ---- the cases ---------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def case_big_boundary():
    """Single windows of 63, 64 and 65 lane-chunks at every A-side offset mod 32, and paired candidates whose two windows
    hold 63-65 lane-chunks together but fewer than 64 each."""
    b = _Builder(101, 20000)
    lens = (2015, 2016, 2017, 2047, 2048, 2049)
    for L in lens:
        for off in range(32):
            b.ss(L, pos=off + 32 * (off % 3), extra=int(b.rng.randint(0, 40)) * (off % 2), rc=(off % 4 >= 2, off % 3 == 1))
    combos = ((31, 32), (32, 32), (33, 32), (62, 1), (63, 1), (63, 2), (1, 62), (1, 63), (40, 24), (40, 25))
    for k, (c0, c1) in enumerate(combos):
        for j in range(4):
            L0 = 32 * c0 - (0 if j == 0 else int(b.rng.randint(0, 32)))
            L1 = 32 * c1 - (0 if j == 1 else int(b.rng.randint(0, 32)))
            b.pp(L0, L1, pos=(int(b.rng.randint(0, 64)), int(b.rng.randint(0, 64))), ord_="12"[j % 2], rc=(j >= 2, (j + k) % 2 == 1))
    return b.finish("big_boundary", [F.make_params(edge_threshold=0.975, ov_threshold=0.96), F.make_params(edge_threshold=0.9, merge_contigs=0.002)],
                    lens=lens, combos=combos)


def _tile(b, items):
    """One tile: an int c = S-S window of c lane-chunks; ("pp", c0, c1); ("oor",); ("empty", c) = a window of c lane-chunks
    whose B side is all N"""
    for it in items:
        if isinstance(it, (int, np.integer)):
            b.ss(32 * int(it) - int(b.rng.randint(0, 32)), pos=int(b.rng.randint(0, 40)), rc=(bool(b.rng.randint(2)), bool(b.rng.randint(2))))
        elif it[0] == "pp":
            b.pp(32 * it[1] - int(b.rng.randint(0, 32)), 32 * it[2] - int(b.rng.randint(0, 32)), pos=(int(b.rng.randint(0, 40)), int(b.rng.randint(0, 40))),
                 ord_="12"[int(b.rng.randint(2))], rc=(bool(b.rng.randint(2)), bool(b.rng.randint(2))))
        elif it[0] == "oor":
            b.oor()
        else:
            b.ss(32 * it[1] - 5, pos=3, nB=range(32 * it[1] - 5))


@functools.lru_cache(maxsize=None)
def case_multi_round():
    """Tiles whose rounds take 512, 513, ~1000 and ~2000 lane-chunks, a tile whose first lane holds 63, 64 windows in one
    round, tiles that mix big, small, out-of-range and all-N windows, and a last tile of 13 candidates with a big one."""
    b = _Builder(202, 30000)
    r = b.rng
    tiles = [
        [16] * 32,                                                          # exactly one round
        [16] * 31 + [17],                                                   # one lane-chunk into a second round
        [int(x) for x in r.randint(16, 48, size=32)],                       # ~1000: two rounds
        [int(x) for x in r.permutation([62] * 16 + [63] * 16)],             # 2000: four rounds
        [63] + [int(x) for x in r.randint(1, 41, size=31)],                 # the first lane alone holds 63
        [("pp", int(x), int(y)) for x, y in zip(r.randint(1, 9, size=32), r.randint(1, 9, size=32))],   # 64 windows
        [("pp", 30, 33), ("pp", 33, 33), 64, ("oor",), ("empty", 70), 5, 70, ("empty", 3), ("oor",), 63, 1, 100,
         ("pp", 2, 2), 40, ("empty", 64), 64, 31, 32, 33, ("oor",), 65, 20, ("pp", 63, 1), 12, 90, 7, ("empty", 20), 60, 61, 62, 2, 66],
        [70, 5, ("oor",), 63, 64, ("empty", 10)] + [int(x) for x in r.randint(20, 64, size=26)],
        [9, ("oor",), 33, 63, ("pp", 50, 20), 12, ("empty", 66), 2, 40, 17, 80, 3, 55],    # last tile: 13 candidates
    ]
    for t in tiles:
        _tile(b, t)
    return b.finish("multi_round", [F.make_params(edge_threshold=0.99), F.make_params(edge_threshold=0.98, ov_threshold=0.6, merge_contigs=0.001)])


@functools.lru_cache(maxsize=None)
def case_n_and_void():
    """N at window positions 31/32 and 2047/2048 on either side and on both at once, reads with 1, 2 and 3 N (three: not in
    the device's two-entry N list), and with ps.mismatch > 0 one void mismatch deep inside a big window next to low-quality
    mismatches that do not void."""
    b = _Builder(303, 30000)
    places = ((31,), (32,), (31, 32), (2047,), (2048,), (2047, 2048), (31, 2048), (32, 2047, 2048), (0, 31, 32))
    for L in (2049, 2100, 2400):
        for k, ns in enumerate(places):
            ns = [p for p in ns if p < L]
            rc = (k % 2 == 1, k % 3 == 2)
            b.ss(L, pos=k, rc=rc, nA=ns)
            b.ss(L, pos=k + 7, rc=rc, nB=ns)
            b.ss(L, pos=k + 13, rc=rc, nA=ns, nB=ns)                    # N in both reads at the same position
            b.ss(L, pos=k + 20, rc=rc, nA=ns[:1], nB=ns[1:])
    for L in (1500, 1900, 2016):                                         # the same in windows the rounds take
        for k, ns in enumerate(((31,), (31, 32), (32, 1023, 1024), (0,))):
            b.ss(L, pos=k, rc=(k % 2 == 1, False), nA=ns)
            b.ss(L, pos=k, rc=(False, k % 2 == 0), nB=ns, nA=ns[:1])
    # void: exactly one Q30 mismatch at window position 1500 of a big window; Q2/Q2 mismatches elsewhere (p = 0.24, not void)
    void = []
    for L, rc in ((2100, (False, False)), (2600, (True, False)), (3000, (False, True)), (1800, (True, True))):
        for kind in ("void", "low"):
            A, _, B, _ = b._views(L, 5, 0, 0.0, (30, 31))
            qa, qb = np.full(len(A), 30), np.full(L, 30)
            if kind == "void":
                B[1500] = (B[1500] + 1) % 4
            else:
                for p in (100, 1500, L - 1):
                    B[p] = (B[p] + 2) % 4
                    qa[5 + p] = qb[p] = 2
            void.append(len(b.cands))
            b.cand(b.single(A, qa, rc[0]), b.single(B, qb, rc[1]), 5)
    return b.finish("n_and_void", [F.make_params(edge_threshold=0.97), F.make_params(edge_threshold=0.98, mismatch=0.02)],
                    places=places, void=void)


@functools.lru_cache(maxsize=None)
def case_fixed_point_extremes():
    """Windows that mismatch at every position with Phred 93 (the largest addend) or Phred 0 on both sides: 10^4 positions
    (big), 2016 (63 lane-chunks, rounds) and 1000, at several A-side offsets."""
    b = _Builder(404, 30000)
    for qv in (93, 0):
        for L in (10000, 2016, 1000):
            for k, pos in enumerate((0, 1, 17, 31)):
                A, _, B, _ = b._views(L, pos, 3 * k, 0.0, (20, 21))
                B = (B + 1 + b.rng.randint(0, 3, size=L)) % 4
                b.cand(b.single(A, np.full(len(A), qv), k % 2 == 1), b.single(B, np.full(L, qv), k >= 2), pos)
    # and a few ordinary windows, so that the alphabet holds more than the two extremes
    for k in range(6):
        b.ss(int(b.rng.randint(500, 4000)), pos=k)
    return b.finish("fixed_point_extremes", [F.make_params(edge_threshold=0.99), F.make_params(edge_threshold=0.0, ov_threshold=-1.0)])


@functools.lru_cache(maxsize=None)
def case_one_order_void():
    """Windows whose only mismatches pair Phred 2 with Phred 5, with Q2 on the A side (x) or on the B side (y), and windows
    whose only mismatches are Q5 against Q5 (z); long (big branch) and short (rounds), on both strands.  All other positions
    are Q30 matches."""
    b = _Builder(505, 20000)
    kinds = []
    for L in (2100, 100, 700):
        for kind, (q_a, q_b) in (("x", (2, 5)), ("y", (5, 2)), ("z", (5, 5))):
            for rc in ((False, False), (True, False), (False, True)):
                A, _, B, _ = b._views(L, 9, 4, 0.0, (30, 31))
                qa, qb = np.full(len(A), 30), np.full(L, 30)
                for p in sorted(set(int(x) for x in b.rng.randint(0, L, size=3))):
                    B[p] = (B[p] + 1) % 4
                    qa[9 + p], qb[p] = q_a, q_b
                kinds.append(kind)
                b.cand(b.single(A, qa, rc[0]), b.single(B, qb, rc[1]), 9)
    p25, p52, p55 = _p_mismatch(2, 5), _p_mismatch(5, 2), _p_mismatch(5, 5)
    params = [F.make_params(mismatch=max(p25, p52)), F.make_params(mismatch=p55), F.make_params(mismatch=float(np.nextafter(p55, 1.0)))]
    return b.finish("one_order_void", params, kinds=np.array(kinds))


def _alphabet(n_values):
    """63 values: Phred 0, 93 and 2..62; 64: and Phred 1"""
    return np.array([0, 93] + list(range(2, 63)) + ([1] if n_values == 64 else []))


@functools.lru_cache(maxsize=None)
def case_alphabet(n_values):
    """The same reads with 63 and with 64 distinct quality values, every value equally often (the frequency ranking of the
    codes then falls back to its tie rule)."""
    b = _Builder(606, 12000)
    lens = [3024] * 4 + [1008] * 4                                    # 16128 = 63 * 256 = 64 * 252 positions
    starts = [0, 900, 1700, 2600, 800, 1500, 2300, 3100]
    seqs = [b.cut(s, L, 0.003) for s, L in zip(starts, lens)]
    qv = _alphabet(n_values)
    q = b.rng.permutation(np.repeat(qv, sum(lens) // len(qv)))
    quals = np.split(q, np.cumsum(lens)[:-1])
    h = [b.single(s, qq, rc=k % 3 == 2) for k, (s, qq) in enumerate(zip(seqs, quals))]
    for i in range(len(lens)):
        for j in range(len(lens)):
            if i != j and starts[i] <= starts[j] < starts[i] + lens[i] - 50:
                b.cand(h[i], h[j], starts[j] - starts[i])
                b.cand(h[i], h[j], starts[j] - starts[i] + 1)
    return b.finish("alphabet_%d" % n_values, [F.make_params(edge_threshold=0.9, ov_threshold=0.5), F.make_params(edge_threshold=0.3, ov_threshold=0.1)])


@functools.lru_cache(maxsize=None)
def case_overflow():
    """Windows of 65535, 65536 and 65537 compared positions (positions below 2^14: the 12-byte and run-encoded records
    hold them), and one of 65537 positions with two N (compared = 65535)."""
    b = _Builder(707, 80000)
    A = b.cut(0, 70000, 0.00002)
    qa = b.qual(70000, 38, 42)
    ha = b.single(A, qa)
    An = A.copy()
    An[[5000, 40000]] = 4
    han = b.single(An, qa)
    def suffix(pos):                                   # A[pos:] with three mismatches
        s = A[pos:].copy()
        for p in b.rng.randint(0, len(s), size=3):
            s[p] = (s[p] + 1) % 4
        return b.single(s, qa[pos:].copy())
    for L in (65535, 65536, 65537):
        b.cand(ha, suffix(70000 - L), 70000 - L)
    b.cand(han, suffix(70000 - 65537), 70000 - 65537)
    b.cand(b.single(b.cut(100, 3000, 0.0005), b.qual(3000, 38, 42)), b.single(b.cut(1100, 2000, 0.0005), b.qual(2000, 38, 42)), 1000)   # an ordinary edge
    return b.finish("overflow", [F.make_params(edge_threshold=0.99)])


@functools.lru_cache(maxsize=None)
def case_exact_modes():
    """Thousands of reads of 600-3000 bases cut from a 30 kb genome: candidates between overlapping reads, most of them
    edges over long windows."""
    b = _Builder(808, 30000)
    n = 420
    lens = b.rng.randint(600, 3001, size=n)
    starts = np.array([b.start(int(L)) for L in lens])
    h = []
    for k in range(n):
        s = b.cut(int(starts[k]), int(lens[k]), 0.001)
        if k % 25 == 0:
            s[b.rng.randint(0, lens[k], size=1 + k % 3)] = 4
        h.append(b.single(s, b.qual(int(lens[k])), rc=k % 2 == 1))
    for i in range(n):
        for j in range(n):
            if i != j and starts[i] <= starts[j] < starts[i] + lens[i] - 400:
                b.cand(h[i], h[j], int(starts[j] - starts[i]))
    return b.finish("exact_modes", [F.make_params(edge_threshold=0.9, ov_threshold=0.5, flags=F.FLAG_EXACT_EDGE_SCORES)])


# ---- checks ------------------------------------------------------------------------------------------------
_REF = {}


def _oracle(case, p):
    q = p.copy()
    q["flags"] = 0                                     # the oracle has no flags
    key = (case.name, q.tobytes())
    if key not in _REF:
        _REF[key] = O.score_batch(case.rs, q, case.cands)[0]
    return _REF[key]


def _against(st, case, p, order=None, exact=False):
    """The parity bar of test_gpu_parity._against_oracle on the case's candidates (permuted by `order`); with exact, the
    same under HC_FLAG_EXACT_EDGE_SCORES and every accepted edge re-added in the reference's order."""
    p = p.copy()
    if exact:
        p["flags"] |= F.FLAG_EXACT_EDGE_SCORES
    cands = case.cands if order is None else case.cands[order]
    ref = _oracle(case, p) if order is None else _oracle(case, p)[order]
    edges, nonedge, per, stats = st.score_batch(p, cands)
    assert_results_match(per, ref["score"], ref["mismatch_rate"], ref["pos3"], ref["pos4"], ref["cls"], what=case.name)
    assert np.array_equal(per["mismatches"], ref["mismatches"]), case.name
    assert np.array_equal(per["compared"], ref["compared"]), case.name
    assert np.array_equal(per["status"], ref["status"]), case.name
    ei = np.nonzero(per["cls"] == F.CLASS_EDGE)[0]
    assert np.array_equal(edges["cand"], ei.astype(np.uint64))
    assert np.array_equal(nonedge, np.nonzero(per["cls"] == F.CLASS_NONEDGE)[0].astype(np.uint64))
    assert np.array_equal(edges["score"], per["score"][ei]) and np.array_equal(edges["mismatch_rate"], per["mismatch_rate"][ei])
    assert np.array_equal(edges["pos3"], per["pos3"][ei]) and np.array_equal(edges["pos4"], per["pos4"][ei])
    assert int(stats["n_candidates"]) == len(cands)
    assert int(stats["n_edges"]) == len(edges) and int(stats["n_nonedges"]) == len(nonedge)
    assert int(stats["n_positions"]) == int(O.window_lengths(ref).sum())
    if p["flags"][0] & F.FLAG_EXACT_EDGE_SCORES:
        e = ref["cls"] == F.CLASS_EDGE
        assert (per["exact"][e] == 1).all()
        assert np.allclose(per["score"][e], ref["score"][e], rtol=1e-14, atol=0)
    return per, ref, stats


def _by_read(c):
    """the order of a list sorted by read, like an overlaps file"""
    return np.lexsort((np.maximum(c["idx1"], c["idx2"]), np.minimum(c["idx1"], c["idx2"])))


CORE = {"big_boundary": case_big_boundary, "multi_round": case_multi_round, "n_and_void": case_n_and_void,
        "fixed_point_extremes": case_fixed_point_extremes}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CORE))
def test_score_paths_against_oracle(built_lib, name):
    case = CORE[name]()
    with capi.Store(case.rs) as st:
        assert st.quality_alphabet <= 63
        for p in case.params:
            _against(st, case, p)
            _against(st, case, p, exact=True)


@pytest.mark.gpu
def test_void_in_one_order_only(built_lib):
    """ps.mismatch between p(2,5) and p(5,2): the symmetric fixed-point table voids both orders, the reference-order pass
    keeps the one the reference keeps.  ps.mismatch = p(5,5) does not void a Q5/Q5 mismatch; one ulp above it does."""
    case = case_one_order_void()
    with capi.Store(case.rs) as st:
        for k, p in enumerate(case.params):
            per, ref, stats = _against(st, case, p)
            if k == 0:
                assert int(stats["n_exact"]) >= 1
            _against(st, case, p, exact=True)


@pytest.mark.gpu
@pytest.mark.parametrize("n_values", [63, 64])
def test_quality_alphabet_boundary(built_lib, monkeypatch, store_layout, n_values):
    """63 quality values are packed (one byte per base), 64 are not: the store takes as many device bytes as a forced
    three-plane store of the same reads exactly when it is not packed."""
    case = case_alphabet(n_values)
    with capi.Store(case.rs) as st:
        assert st.quality_alphabet == n_values
        own = st.device_bytes
        for p in case.params:
            _against(st, case, p)
            _against(st, case, p, exact=True)
    monkeypatch.setenv("HC_STORE_LAYOUT", "planar")
    with capi.Store(case.rs) as st:
        planar = st.device_bytes
    if store_layout == "packed" and n_values == 63:
        assert own < planar
    else:
        assert own == planar


@pytest.mark.gpu
def test_phred_93_is_accepted_and_94_rejected(built_lib):
    with capi.Store(F.ReadSet.from_lists([(0, "ACGT", "!~I~"), (1, "ACGT", "IIII")], [])) as st:
        assert st.quality_alphabet == 3
    with pytest.raises(capi.HcError):
        capi.Store(F.ReadSet.from_lists([(0, "ACGT", "II" + chr(127) + "I"), (1, "ACGT", "IIII")], []))


@pytest.mark.gpu
@pytest.mark.parametrize("exact", [False, True])
def test_small_records_flag_16bit_overflow(built_lib, exact):
    """hc_edge_small(_exact) holds 16-bit counts: HC_EDGE_OVERFLOW is set on exactly the edges with a window of more than
    65535 compared positions (N positions are not compared); every other count equals the full output's."""
    case = case_overflow()
    p = case.params[0]
    with capi.Store(case.rs) as st:
        per, ref, _ = _against(st, case, p, exact=exact)
        if exact:
            p = p.copy()
            p["flags"] |= F.FLAG_EXACT_EDGE_SCORES
        edges, _, _, _ = st.score_batch(p, case.cands)
        assert len(edges) == len(case.cands)
        for runs in (True, False):
            se, nonedge, _ = st.score_batch_small(p, case.cands, runs=runs)
            assert np.array_equal(se["cand"].astype(np.uint64), edges["cand"]) and not nonedge.any()
            cmp, mm = per["compared"][se["cand"]], per["mismatches"][se["cand"]]
            over = (cmp > 0xffff).any(axis=1)
            assert np.array_equal((se["flags"] & F.EDGE_OVERFLOW) != 0, over), runs
            assert over.sum() == 2
            assert np.array_equal(se["compared"][~over], cmp[~over]) and np.array_equal(se["mismatches"][~over], mm[~over])
            assert np.array_equal(se["compared"][over], np.minimum(cmp[over], 0xffff))


@pytest.mark.gpu
def test_reference_order_pass_modes_on_long_windows(built_lib):
    """Every accepted edge queued (HC_FLAG_EXACT_EDGE_SCORES) on windows of up to 3000 positions: thousands of them (one
    thread each; the wide table in the packed layout) and a few hundred (one warp each)."""
    case = case_exact_modes()
    p = case.params[0]
    with capi.Store(case.rs) as st:
        per, ref, stats = _against(st, case, p)
        assert (ref["cls"] == F.CLASS_EDGE).sum() > THREAD_MODE_MIN and int(stats["n_exact"]) > THREAD_MODE_MIN
        few = np.arange(len(case.cands)) < 500
        per2, ref2, stats2 = _against(st, case, p, order=np.nonzero(few)[0])
        assert 0 < int(stats2["n_exact"]) < WARP_MODE_MAX
        assert per2.tobytes() == per[few].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("exact", [False, True])
@pytest.mark.parametrize("name", sorted(CORE))
def test_by_read_order_against_oracle(built_lib, name, exact):
    """The cases sorted by read, as an overlaps file lists them, against the oracle, with the records with and without run
    information; with exact, every accepted edge is also re-added in the reference's order."""
    case = CORE[name]()
    order = _by_read(case.cands)
    with capi.Store(case.rs) as st:
        for p in case.params:
            if exact:                  # set here so that the run-encoded call below scores under the same flags
                p = p.copy()
                p["flags"] |= F.FLAG_EXACT_EDGE_SCORES
            per, _, _ = _against(st, case, p, order=order)
            _, _, per_runs, _ = st.score_batch(p, case.cands[order], compact="runs")
            assert per_runs.tobytes() == per.tobytes()


# ---- the cases reach their shapes (no GPU) ---------------------------------------------------------------------
def test_cases_hit_their_shapes():
    # a. single windows of 63/64/65 lane-chunks at every offset mod 32; paired totals of 63-65 below 64 per window
    a = case_big_boundary()
    wl = _window_lengths(a.rs, a.cands)
    ck = _chunks(wl)
    single = wl[:, 1] == 0
    assert sorted(set(wl[single, 0].tolist())) == list(a.meta["lens"])
    for c in (63, 64, 65):
        offs = {int(x) % 32 for x in a.cands["pos1"][single & (ck[:, 0] == c)]}
        assert offs == set(range(32)), c
    pt = ck[~single]
    assert set(pt.sum(axis=1).tolist()) == {63, 64, 65} and pt.max() < BIG_CHUNKS
    assert {tuple(x) for x in pt.tolist()} == set(a.meta["combos"])
    # b. rounds of 512, 513, ~1000, ~2000 lane-chunks; first lane 63; 64 windows in one round; mixed tiles; partial last tile
    b = case_multi_round()
    tiles = _tile_chunks(b.rs, b.cands)
    rounds = [r for _, r in tiles]
    assert rounds[0] == PARTMAX and rounds[1] == PARTMAX + 1 and 900 <= rounds[2] <= 1100 and rounds[3] == 2000
    assert tiles[4][0][0] == 63 and rounds[4] > PARTMAX
    assert (_window_lengths(b.rs, b.cands[160:192]) > 0).all() and rounds[5] <= PARTMAX
    rb = _oracle(b, b.params[0])
    st = rb["status"].reshape(-1)
    assert set(np.unique(st).tolist()) >= {0, 1, 2, 5}
    for t in (6, 7, 8):
        x = tiles[t][0]
        s = rb["status"][32 * t:32 * t + 32]
        assert (x >= BIG_CHUNKS).any() and ((x > 0) & (x < BIG_CHUNKS)).any(), t
        assert (s == 2).any() and (s == 5).any(), t
    assert len(b.cands) % 32 == 13 and (tiles[-1][0] >= BIG_CHUNKS).any()
    # c. N at window positions 31/32/2047/2048 on the A side, the B side and both; reads with 1, 2 and 3 N; one void window
    c = case_n_and_void()
    seen = {"A": set(), "B": set(), "both": set()}
    for x in c.cands:
        for nA, nB in _n_positions(c.rs, x):
            seen["A"] |= nA
            seen["B"] |= nB
            seen["both"] |= nA & nB
    for side in seen.values():
        assert {31, 32, 2047, 2048} <= side
    ncount = [s.count("N") for s in [c.rs.seq(i) for i in range(c.rs.n_reads)]]
    assert {1, 2, 3} <= set(ncount)
    rv = _oracle(c, c.params[1])
    vd = np.array(c.meta["void"])
    assert (rv["status"][vd[0::2], 0] == 4).all() and (rv["status"][vd[1::2], 0] == 1).all()
    ck = _chunks(_window_lengths(c.rs, c.cands[vd]))[:, 0]
    assert (ck[:6] >= BIG_CHUNKS).all() and (ck[6:] < BIG_CHUNKS).all()        # big windows, and one the rounds take
    assert (_oracle(c, c.params[0])["status"][vd] == [1, 0]).all()
    # d. every position mismatches; at Phred 93 one lane-chunk sums to more than 2.9e9 in units of 2^-22, below 2^32
    d = case_fixed_point_extremes()
    rd = _oracle(d, d.params[0])
    full = (rd["compared"][:, 0] > 0) & (rd["mismatches"][:, 0] == rd["compared"][:, 0])
    assert full.sum() == 24 and 10000 in set(rd["compared"][full, 0].tolist())
    top = -math.log(_p_mismatch(93, 93)) * FX_SCALE
    assert 2.9e9 < 32 * round(top) < 2 ** 32
    # e. p(2,5) != p(5,2): under max of the two, Q2 on the A side voids and Q5 on the A side does not
    e = case_one_order_void()
    assert _p_mismatch(2, 5) != _p_mismatch(5, 2)
    kinds = e.meta["kinds"]
    st0, st1, st2 = (_oracle(e, p)["status"][:, 0] for p in e.params)
    lo_first = _p_mismatch(2, 5) < _p_mismatch(5, 2)
    assert (st0[kinds == ("x" if lo_first else "y")] == 4).all() and (st0[kinds == ("y" if lo_first else "x")] == 1).all()
    assert (st1[kinds == "z"] == 1).all() and (st2[kinds == "z"] == 4).all()
    # f. 63 / 64 values, 0 and 93 among them, all equally frequent
    for nv in (63, 64):
        f = case_alphabet(nv)
        vals, cnt = np.unique(f.rs.quals, return_counts=True)
        assert len(vals) == nv and {33, 33 + 93} <= set(vals.tolist()) and len(set(cnt.tolist())) == 1
    assert case_alphabet(63).rs.bases.tobytes() == case_alphabet(64).rs.bases.tobytes()
    # g. compared counts 65535 / 65536 / 65537, and a 65537-position window with two N, all of them edges
    g = case_overflow()
    rg = _oracle(g, g.params[0])
    assert rg["compared"][:4, 0].tolist() == [65535, 65536, 65537, 65535] and O.window_lengths(rg)[3] == 65537
    assert (rg["cls"] == F.CLASS_EDGE).all() and (g.cands["pos1"] < (1 << 14)).all()
    # h. thousands of edges over long windows (thread mode), the first 500 candidates a few hundred (warp mode)
    h = case_exact_modes()
    rh = _oracle(h, h.params[0])
    assert (rh["cls"] == 1).sum() > THREAD_MODE_MIN and 0 < (rh["cls"][:500] == 1).sum() < WARP_MODE_MAX - 100
    assert O.window_lengths(rh).max() > 2500
