"""The compressed candidate records at the limits of their fields, and run-encoded lists cut by hand through the host
pipeline's steps and device shards.

Field limits.  Each record form is pinned bit for bit to the small encoder below (CPU), and scored on a store built so
that every field reaches its top bit and its all-ones value:
  * a store of exactly 2^25 reads, mostly 4-base fillers, with real reads where the 25-bit read field of the 6-byte run
    entry changes its top bits, at POS 0/255/256/511: 6-, 8-, 12-, 16- and 32-byte records;
  * reads of 16.5-17 kb at POS 8191/8192/16383: 12- and 8-byte records, full and small outputs;
  * one read of 2^28 + 2000 bases at POS1 2^27 - 1 / 2^27 / 2^28 - 1: 16-byte records.
Run bookkeeping.  hc_score_batch_runs, _runs_small and _runs6_small get hand-made (anchor, start, entries) arrays: one run
per candidate, one run for the whole batch, runs of 31-65 candidates starting at every offset mod 32 and exactly at and
one past the pipeline's step boundaries, a run split in two with the same anchor, runs anchored on ID2; under steps of
64, 1024 and 4160 candidates, whole-shard and two-slot mode, pageable and pinned record buffers.

The reference is the oracle on the equivalent 32-byte records, with the bar of test_gpu_parity._against_oracle: classes,
lists, pos3/pos4, counts, statuses and mismatch rates bit-exact, scores within 1e-6 (1e-14 for the edges re-added in the
reference's order under HC_FLAG_EXACT_EDGE_SCORES).  Every form is also compared with hc_score_batch on the 32-byte
records: per-candidate results and edge records byte for byte, or, for the small outputs, every field of the small edge
records and the whole non-edge bit map.  Each case runs in both store layouts, with and without
HC_FLAG_EXACT_EDGE_SCORES, and once with thresholds placed exactly on oracle scores, which sends candidates through the
reference-order pass (hc_exact_kernel), the second place that decodes a record.
"""
import contextlib
import ctypes
import os

import numpy as np
import pytest

from haploconduct_b200 import capi, formats as F, workloads as W
from oracle import oracle as O
from util import assert_results_match

ORD_CODE = {ord("-"): 0, ord("1"): 1, ord("2"): 2}
SENTINEL = np.uint64(0xDEADBEEFDEADBEEF)
PARAM_KINDS = ["plain", "exact", "boundary"]

# field layouts (first bit, width) of the record forms, include/hc_b200.h
COMPACT_FIELDS = {"idx1": (0, 32), "idx2": (32, 32), "pos1": (64, 28), "ori1": (92, 1), "ori2": (93, 1), "ord": (94, 2),
                  "pos2": (96, 32)}
SHORT_FIELDS = {"idx1": (0, 32), "idx2": (32, 32), "pos1": (64, 14), "pos2": (78, 14), "ori1": (92, 1), "ori2": (93, 1),
                "ord": (94, 2)}
ENTRY_FIELDS = {"other": (0, 31), "role": (31, 1), "pos1": (32, 14), "pos2": (46, 14), "ori1": (60, 1), "ori2": (61, 1),
                "ord": (62, 2)}
ENTRY6_FIELDS = {"other": (0, 25), "role": (25, 1), "ori1": (26, 1), "ori2": (27, 1), "ord": (28, 2), "pos1": (30, 9),
                 "pos2": (39, 9)}


# ---- an independent encoder / decoder, one bit at a time ------------------------------------------------------------
def _pack(layout, values, nbytes):
    v, used = 0, 0
    for name, (off, width) in layout.items():
        x = int(values[name])
        if not 0 <= x < (1 << width):
            raise ValueError("%s = %d does not fit %d bits" % (name, x, width))
        for b in range(width):
            bit = 1 << (off + b)
            assert not used & bit
            used |= bit
            if (x >> b) & 1:
                v |= bit
    assert used == (1 << (8 * nbytes)) - 1
    return v.to_bytes(nbytes, "little")


def _cand_fields(c):
    return {"idx1": c["idx1"], "idx2": c["idx2"], "pos1": c["pos1"], "pos2": c["pos2"], "ori1": int(c["ori1"] != 0),
            "ori2": int(c["ori2"] != 0), "ord": ORD_CODE.get(int(c["ord"]), 0)}


def _entry_fields(c, anchor):
    f = _cand_fields(c)
    assert anchor in (int(c["idx1"]), int(c["idx2"]))
    role = int(int(c["idx1"]) != anchor)          # 1: the anchor is ID2, the record names ID1
    f.update(other=int(c["idx1"]) if role else int(c["idx2"]), role=role)
    return f


def _enc(layout, nbytes, rows):
    return b"".join(_pack(layout, r, nbytes) for r in rows)


def _unpack(raw, layout):
    """uint8 [n, nbytes] records -> {field: uint64 values}, bit by bit."""
    raw = np.asarray(raw, dtype=np.uint8)
    out = {}
    for name, (off, width) in layout.items():
        v = np.zeros(len(raw), dtype=np.uint64)
        for b in range(width):
            k = off + b
            v |= ((raw[:, k // 8] >> np.uint8(k % 8)) & np.uint8(1)).astype(np.uint64) << np.uint64(b)
        out[name] = v
    return out


def _raw(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint8).reshape(len(a), -1)


def _assert_hits(vals, layout, names):
    """Every named field has its top bit set somewhere, and takes its all-ones value somewhere."""
    for name in names:
        w = layout[name][1]
        v = vals[name]
        assert ((v >> np.uint64(w - 1)) & np.uint64(1)).any(), name + ": top bit never set"
        assert (v == np.uint64((1 << w) - 1)).any(), name + ": never all ones"


# ---- candidates, runs and calls ------------------------------------------------------------------------------------
def _mk(rows):
    """rows of (idx1, idx2, pos1, pos2, ord char, ori1, ori2, type1, type2) -> CANDIDATE records."""
    c = np.zeros(len(rows), dtype=F.CANDIDATE)
    for k, name in enumerate(("idx1", "idx2", "pos1", "pos2")):
        c[name] = [r[k] for r in rows]
    c["ord"] = [ord(r[4]) for r in rows]
    c["ori1"], c["ori2"] = [r[5] for r in rows], [r[6] for r in rows]
    c["type1"], c["type2"] = [ord(r[7]) for r in rows], [ord(r[8]) for r in rows]
    c["len1"], c["perc1"] = 1, 50
    return c


def _runs_by_anchor(c, anchor_of):
    """Candidates sorted (stably) by the anchor each one was given; runs = stretches of equal anchor."""
    order = np.argsort(anchor_of, kind="stable")
    c, a = c[order], np.asarray(anchor_of)[order]
    cut = np.flatnonzero(np.r_[True, a[1:] != a[:-1]])
    return c, a[cut].astype(np.uint32), np.r_[cut, len(c)].astype(np.uint64)


def _per_cand_anchor(anchor, start):
    return np.repeat(anchor, np.diff(start.astype(np.int64)))


def _entries(c, anchor, start):
    """hc_candidate_entry records of explicit runs (the anchor is ID2 when it is not ID1)."""
    a = _per_cand_anchor(anchor, start)
    assert ((c["idx1"] == a) | (c["idx2"] == a)).all()
    role = c["idx1"] != a
    e = np.zeros(len(c), dtype=F.CANDIDATE_ENTRY)
    e["other"] = np.where(role, c["idx1"], c["idx2"]).astype(np.uint32) | (role.astype(np.uint32) << np.uint32(31))
    e["pos"] = F.short_candidates(c)["pos"]
    return e


@contextlib.contextmanager
def _env(**kw):
    old = {k: os.environ.get(k) for k in kw}
    try:
        for k, v in kw.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _store(rs, layout, **kw):
    with _env(HC_STORE_LAYOUT="planar" if layout == "planar" else "auto"):
        return capi.Store(rs, **kw)


def _call_runs(st, params, anchor, start, entries):
    """hc_score_batch_runs with explicit run arrays -> (per_cand, edges, nonedge list, stats)."""
    n = len(entries)
    per = np.zeros(max(n, 1), dtype=F.RESULT)
    edges = np.zeros(max(n, 1), dtype=F.EDGE)
    nonedge = np.zeros(max(n, 1), dtype=np.uint64)
    ne, nn = ctypes.c_uint64(0), ctypes.c_uint64(0)
    stats = np.zeros(1, dtype=F.BATCH_STATS)
    capi._check(capi.lib().hc_score_batch_runs(st.handle, params.ctypes.data, anchor.ctypes.data, start.ctypes.data, len(anchor),
                                               entries.ctypes.data, n, per.ctypes.data, edges.ctypes.data, n, ctypes.byref(ne),
                                               nonedge.ctypes.data, n, ctypes.byref(nn), stats.ctypes.data))
    return per[:n], edges[:ne.value], nonedge[:nn.value], stats[0]


def _call_small(st, params, kind, records, anchor=None, start=None):
    """hc_score_batch_short_small ("short"), _runs_small ("runs") or _runs6_small ("runs6") on a bit map pre-filled with
    a sentinel one word past what the call owns -> (small edges, the owned words, n_nonedges, stats)."""
    L = capi.lib()
    exact = bool(int(params["flags"][0]) & F.FLAG_EXACT_EDGE_SCORES)
    n = len(records)
    edges = np.zeros(max(n, 1), dtype=F.EDGE_SMALL_EXACT if exact else F.EDGE_SMALL)
    words = (n + 63) // 64
    bits = np.full(words + 1, SENTINEL, dtype=np.uint64)
    ne, nn = ctypes.c_uint64(0), ctypes.c_uint64(0)
    stats = np.zeros(1, dtype=F.BATCH_STATS)
    tail = (edges.ctypes.data, n, ctypes.byref(ne), bits.ctypes.data, ctypes.byref(nn), stats.ctypes.data)
    if kind == "short":
        rc = L.hc_score_batch_short_small(st.handle, params.ctypes.data, records.ctypes.data, n, *tail)
    else:
        fn = L.hc_score_batch_runs6_small if kind == "runs6" else L.hc_score_batch_runs_small
        rc = fn(st.handle, params.ctypes.data, anchor.ctypes.data, start.ctypes.data, len(anchor), records.ctypes.data, n, *tail)
    capi._check(rc)
    assert bits[words] == SENTINEL, "the call wrote past the words it owns"
    return edges[:ne.value], bits[:words], int(nn.value), stats[0]


def _check_parity(per, edges, nonedge, stats, ref, params, means):
    """The bar of test_gpu_parity._against_oracle, plus, under HC_FLAG_EXACT_EDGE_SCORES, the 1e-14 bar of the re-added
    edges and their mean logs bit for bit with the oracle's (means: its per-window mean logs)."""
    assert_results_match(per, ref["score"], ref["mismatch_rate"], ref["pos3"], ref["pos4"], ref["cls"], what="vs oracle")
    assert np.array_equal(per["mismatches"], ref["mismatches"])
    assert np.array_equal(per["compared"], ref["compared"])
    assert np.array_equal(per["status"], ref["status"])
    ei = np.nonzero(per["cls"] == F.CLASS_EDGE)[0]
    assert np.array_equal(edges["cand"], ei.astype(np.uint64))
    assert np.array_equal(nonedge, np.nonzero(per["cls"] == F.CLASS_NONEDGE)[0].astype(np.uint64))
    assert np.array_equal(edges["score"], per["score"][ei]) and np.array_equal(edges["mismatch_rate"], per["mismatch_rate"][ei])
    assert np.array_equal(edges["pos3"], per["pos3"][ei]) and np.array_equal(edges["pos4"], per["pos4"][ei])
    assert int(stats["n_candidates"]) == len(per) and int(stats["n_edges"]) == len(edges)
    assert int(stats["n_nonedges"]) == len(nonedge)
    assert int(stats["n_positions"]) == int(O.window_lengths(ref).sum())
    if int(params["flags"][0]) & F.FLAG_EXACT_EDGE_SCORES:
        assert (per["exact"][ei] == 1).all()
        assert np.allclose(per["score"][ei], ref["score"][ei], rtol=1e-14, atol=0)
        scored = ref["status"][ei] == 1                                     # HC_WIN_SCORED; other windows carry NaN
        assert edges["mean_log"][scored].tobytes() == means[ei][scored].tobytes()
        assert np.isnan(edges["mean_log"][~scored]).all()


def _batch(st, params, c, **kw):
    """Store.score_batch reordered as (per_cand, edges, nonedge list, stats)."""
    edges, nonedge, per, stats = st.score_batch(params, c, **kw)
    return per, edges, nonedge, stats


def _check_same_full(got, full):
    per, edges, nonedge = got[:3]
    assert per.tobytes() == full[0].tobytes()
    assert edges.tobytes() == full[1].tobytes() and np.array_equal(nonedge, full[2])


def _check_small(got, full, params):
    se, words, nn, stats = got
    per, edges, nonedge = full[:3]
    want = np.zeros(64 * len(words), dtype=bool)          # bits past n stay 0
    want[nonedge.astype(np.int64)] = True
    assert np.array_equal(words, np.packbits(want, bitorder="little").view(np.uint64)), "non-edge bit map"
    assert nn == len(nonedge) and int(stats["n_nonedges"]) == nn and int(stats["n_edges"]) == len(edges)
    ec = edges["cand"].astype(np.int64)
    assert np.array_equal(se["cand"], ec.astype(np.uint32))
    assert np.array_equal(se["mismatches"], per["mismatches"][ec].astype(np.uint16))
    assert np.array_equal(se["compared"], per["compared"][ec].astype(np.uint16))
    assert np.array_equal((se["flags"] & F.EDGE_TWO) != 0, per["status"][ec, 1] != 0)
    if int(params["flags"][0]) & F.FLAG_EXACT_EDGE_SCORES:
        a, b = se["mean_log"], edges["mean_log"]
        assert np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~np.isnan(a)], b[~np.isnan(b)])
        assert (se["flags"] & F.EDGE_EXACT).all()
    else:
        assert np.array_equal(se["score"], edges["score"])


_PLAIN = dict(edge_threshold=0.95, ov_threshold=0.8)


def _params(kind, rs, c, cache):
    """plain / exact / boundary: thresholds ON oracle scores of these candidates (the edge threshold on the median, the
    overlap threshold on the lower quartile of the scores in (0.5, 0.9999))."""
    if kind not in cache:
        if kind == "boundary":
            ref = O.score_batch(rs, F.make_params(**_PLAIN), c)[0]
            s = np.sort(ref["score"][(ref["score"] > 0.5) & (ref["score"] < 0.9999)])
            assert len(s) >= 2
            cache[kind] = F.make_params(edge_threshold=float(s[len(s) // 2]), ov_threshold=float(s[len(s) // 4]))
        else:
            cache[kind] = F.make_params(flags=F.FLAG_EXACT_EDGE_SCORES if kind == "exact" else 0, **_PLAIN)
    return cache[kind]


def _score_forms(st, rs, params, c, anchor, start, forms, ref=None):
    """c scored through hc_score_batch (checked against the oracle) and through each named form (checked against it)."""
    if ref is None:
        ref = O.score_batch(rs, params, c)
    ref, means = ref
    e0, n0, p0, s0 = st.score_batch(params, c)
    _check_parity(p0, e0, n0, s0, ref, params, means)
    full = (p0, e0, n0)
    if params["edge_threshold"][0] in ref["score"]:
        assert p0["exact"].any()               # the boundary candidates went through the reference-order pass
    smalls = []
    for form in forms:
        if form == "compact":
            _check_same_full(_batch(st, params, c, compact=True), full)
        elif form == "short":
            _check_same_full(_batch(st, params, c, compact="short"), full)
            smalls.append(_call_small(st, params, "short", np.ascontiguousarray(F.short_candidates(c))))
        elif form == "runs":
            entries = _entries(c, anchor, start)
            _check_same_full(_call_runs(st, params, anchor, start, entries), full)
            smalls.append(_call_small(st, params, "runs", entries, anchor, start))
        elif form == "runs6":
            entries = _entries(c, anchor, start)
            smalls.append(_call_small(st, params, "runs6", F.entries6(entries), anchor, start))
    for got in smalls:
        _check_small(got, full, params)
        assert got[0].tobytes() == smalls[0][0].tobytes() and np.array_equal(got[1], smalls[0][1])
    return p0, ref


class _Fixture:
    """Host read set and candidates of one case, with its stores (one per layout) made on first use."""

    def __init__(self, rs, c, anchor, start):
        self.rs, self.c, self.anchor, self.start = rs, c, anchor, start
        self.stores, self.params, self.refs = {}, {}, {}

    def store(self, layout):
        if layout not in self.stores:
            self.stores[layout] = _store(self.rs, layout)
        return self.stores[layout]

    def ref(self, kind):
        if kind not in self.refs:
            self.refs[kind] = O.score_batch(self.rs, _params(kind, self.rs, self.c, self.params), self.c)
        return self.refs[kind]

    def close(self):
        for st in self.stores.values():
            st.close()
        self.stores = {}


def _substitute(seg, rng, rate=0.002):
    s = seg.copy()
    m = rng.random_sample(len(s)) < rate
    s[m] = (s[m] + rng.randint(1, 4, size=int(m.sum()))) % 4
    return s


_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


# ---- 1a. the wide-index store: exactly 2^25 reads ---------------------------------------------------------------------
WIDE_N = 1 << 25
STARTS9 = (0, 256, 511, 767)       # genome offsets of the real reads: their differences are 255, 256 and 511
POS9 = (0, 255, 256, 511)


def _wide_layout(n_reads):
    """{index: (genome offset, length of mate 0, length of mate 1)} of the real reads, the filler indices used in
    candidates, and n_single.  Singles at 0, 1, 2^16 - 1, 2^16, 2^24 - 1, 2^24 and just below the 8 pairs on top."""
    rng = np.random.RandomState(25)
    singles = [0, 1, (1 << 16) - 1, 1 << 16, (1 << 24) - 1, 1 << 24] + list(range(n_reads - 14, n_reads - 8))
    pairs = list(range(n_reads - 8, n_reads))
    real = {}
    for k, i in enumerate(singles + pairs):
        real[i] = (STARTS9[k % 4], int(rng.randint(600, 901)), int(rng.randint(600, 901)) if i in pairs else 0)
    return real, [2, (1 << 24) + 1, n_reads - 15], n_reads - 8


def _wide_readset(n_reads):
    real, _, n_single = _wide_layout(n_reads)
    rng = np.random.RandomState(26)
    genome = rng.randint(0, 4, size=3000)
    lens = np.zeros((n_reads, 2), dtype=np.uint32)
    lens[:, 0] = 4
    for i, (_, l0, l1) in real.items():
        lens[i] = (l0, l1)
    tot = lens.astype(np.uint64).sum(axis=1)
    off = np.zeros(n_reads, dtype=np.uint64)
    np.cumsum(tot[:-1], out=off[1:])
    descs = np.zeros(n_reads, dtype=F.READ_DESC)
    descs["seq_len"] = lens
    descs["seq_off"][:, 0] = off
    descs["seq_off"][:, 1] = np.where(lens[:, 1] > 0, off + lens[:, 0], 0)
    total = int(tot.sum())
    bases = np.resize(_ACGT, total)
    quals = np.full(total, 33 + 30, dtype=np.uint8)        # a value of the real reads' alphabet: the store stays packed
    for i, (s, l0, l1) in sorted(real.items()):
        o = int(off[i])
        for seg in ((s, l0), (s + 1000, l1)) if l1 else ((s, l0),):
            bases[o:o + seg[1]] = _ACGT[_substitute(genome[seg[0]:seg[0] + seg[1]], rng)]
            quals[o:o + seg[1]] = 33 + rng.randint(20, 42, size=seg[1])
            o += seg[1]
    return F.ReadSet(ids=np.arange(n_reads, dtype=np.uint64), descs=descs, bases=bases, quals=quals, n_single=n_single)


def _wide_cands():
    """S-S, S-P, P-S and P-P candidates between the real reads (both index orders, four ori, POS1 x POS2 in POS9, ORD 1
    and 2), fillers as A at POS 511 (POS_OOR), as B, and against each other; in runs anchored on the lower index for
    every other candidate and on the higher one otherwise."""
    real, fillers, _ = _wide_layout(WIDE_N)
    idx = sorted(real)
    rows, k = [], 0
    for a in idx:
        for b in idx:
            if a == b:
                continue
            ta, tb = "p" if real[a][2] else "s", "p" if real[b][2] else "s"
            for o1 in (0, 1):
                for o2 in (0, 1):
                    for p1 in POS9:
                        for p2 in POS9:
                            rows.append((a, b, p1, p2, "12"[k % 2] if ta + tb == "pp" else "-12"[k % 3], o1, o2, ta, tb))
                            k += 1
    for f in fillers:
        for b in idx[::3]:
            tb = "p" if real[b][2] else "s"
            rows += [(f, b, 511, 511, "-", 1, 1, "s", tb), (b, f, 511, 511, "1", 1, 0, tb, "s"), (f, b, 0, 0, "2", 0, 1, "s", tb)]
    rows.append((fillers[0], fillers[1], 511, 511, "-", 1, 1, "s", "s"))
    c = _mk(rows)
    lo, hi = np.minimum(c["idx1"], c["idx2"]), np.maximum(c["idx1"], c["idx2"])
    return _runs_by_anchor(c, np.where(np.arange(len(c)) % 2 == 0, lo, hi))


@pytest.fixture(scope="module")
def wide():
    c, anchor, start = _wide_cands()
    fx = _Fixture(_wide_readset(WIDE_N), c, anchor, start)
    yield fx
    fx.close()


def test_wide_store_records_hit_their_limits():
    c, anchor, start = _wide_cands()
    e8 = _entries(c, anchor, start)
    v6 = _unpack(_raw(F.entries6(e8)), ENTRY6_FIELDS)
    _assert_hits(v6, ENTRY6_FIELDS, ("other", "role", "ori1", "ori2", "pos1", "pos2"))
    assert set(v6["ord"].tolist()) == {0, 1, 2}
    assert (v6["role"] == 0).any() and ((v6["other"] >> np.uint64(24)) == 0).any()
    v8 = _unpack(_raw(e8), ENTRY_FIELDS)
    assert (v8["other"] == np.uint64(WIDE_N - 1)).any() and ((v8["other"] >> np.uint64(24)) & np.uint64(1)).any()
    assert (v8["pos1"] == 511).any() and (v8["pos2"] == 511).any() and set(v8["role"].tolist()) == {0, 1}
    real, fillers, n_single = _wide_layout(WIDE_N)
    assert max(real) == WIDE_N - 1 and n_single == WIDE_N - 8
    # every type, both index orders, every ori, ORD 1 and 2 of P-P, every POS pair
    t = {(chr(a), chr(b)) for a, b in zip(c["type1"], c["type2"])}
    assert t == {("s", "s"), ("s", "p"), ("p", "s"), ("p", "p")}
    assert (c["idx1"] < c["idx2"]).any() and (c["idx1"] > c["idx2"]).any()
    assert {(int(a), int(b)) for a, b in zip(c["ori1"], c["ori2"])} == {(0, 0), (0, 1), (1, 0), (1, 1)}
    pp = (c["type1"] == ord("p")) & (c["type2"] == ord("p"))
    assert set(c["ord"][pp].tolist()) == {ord("1"), ord("2")}
    assert {(int(a), int(b)) for a, b in zip(c["pos1"], c["pos2"])} >= {(p, q) for p in POS9 for q in POS9}
    # POS at the field maximum past the end of A (4-base fillers)
    lens = np.array([real[int(i)][1] if int(i) in real else 4 for i in c["idx1"]])
    assert ((c["pos1"] == 511) & (lens <= 511)).sum() >= 3


@pytest.mark.gpu
@pytest.mark.parametrize("kind", PARAM_KINDS)
@pytest.mark.parametrize("layout", ["packed", "planar"])
def test_wide_store_at_the_record_limits(built_lib, wide, layout, kind):
    """2^25 reads: read indices with bits 16, 24 and all 25 bits set, POS with bit 8 set, through the 6-, 8-, 12-, 16- and
    32-byte records."""
    st = wide.store(layout)
    params = _params(kind, wide.rs, wide.c, wide.params)
    per, ref = _score_forms(st, wide.rs, params, wide.c, wide.anchor, wide.start, ("compact", "short", "runs", "runs6"),
                            ref=wide.ref(kind))
    real = _wide_layout(WIDE_N)[0]
    oor = (wide.c["pos1"] == 511) & ~np.isin(wide.c["idx1"], list(real))
    assert oor.sum() >= 3 and (per["status"][oor, 0] == 2).all()                  # HC_WIN_POS_OOR
    assert (per["cls"] == F.CLASS_EDGE).sum() >= 10
    print("2^25-read store (%s): %d bytes on the device" % (layout, st.device_bytes))


@pytest.mark.gpu
def test_runs6_store_size_limit(built_lib, wide):
    """hc_score_batch_runs6_small takes a store of 2^25 reads and rejects one of 2^25 + 1."""
    c, anchor, start = _runs_by_anchor(wide.c[::97], np.minimum(wide.c["idx1"][::97], wide.c["idx2"][::97]))
    e6 = F.entries6(_entries(c, anchor, start))
    assert (_unpack(_raw(e6), ENTRY6_FIELDS)["other"] == np.uint64(WIDE_N - 1)).any()
    _call_small(wide.store("packed"), F.make_params(), "runs6", e6, anchor, start)
    wide.close()
    big = _wide_readset(WIDE_N + 1)
    with capi.Store(big) as st1:
        with pytest.raises(capi.HcError) as ei:
            _call_small(st1, F.make_params(), "runs6", e6, anchor, start)
        assert ei.value.code == -1 and "2^25" in str(ei.value)


# ---- 1b. 14-bit positions ---------------------------------------------------------------------------------------------
STARTS14 = (0, 8191, 8192, 16383)  # differences 8191, 8192 and 16383
POS14 = (8191, 8192, 16383)


def _long_fixture_data():
    rng = np.random.RandomState(14)
    genome = rng.randint(0, 4, size=16383 + 20000 + 17001)
    singles, pairs = [], []
    for k, s in enumerate(STARTS14):
        l0, l1 = int(rng.randint(16500, 17001)), int(rng.randint(16500, 17001))
        q = lambda L: (33 + rng.randint(20, 42, size=L)).astype(np.uint8).tobytes().decode()
        sq = lambda a, L: _ACGT[_substitute(genome[a:a + L], rng)].tobytes().decode()
        singles.append((k, sq(s, l0), q(l0)))
        pairs.append((10 + k, sq(s, l0), q(l0), sq(s + 20000, l1), q(l1)))
    rs = F.ReadSet.from_lists(singles, pairs)
    rows, k = [], 0
    for group, t in ((range(0, 4), "s"), (range(4, 8), "p")):
        for a in group:
            for b in group:
                if a == b:
                    continue
                for o1 in (0, 1):
                    for o2 in (0, 1):
                        for p1 in POS14:
                            for p2 in POS14:
                                rows.append((a, b, p1, p2, "12"[k % 2] if t == "p" else "-12"[k % 3], o1, o2, t, t))
                                k += 1
    c = _mk(rows)
    lo, hi = np.minimum(c["idx1"], c["idx2"]), np.maximum(c["idx1"], c["idx2"])
    return (rs,) + _runs_by_anchor(c, np.where(np.arange(len(c)) % 2 == 0, lo, hi))


@pytest.fixture(scope="module")
def long_reads():
    fx = _Fixture(*_long_fixture_data())
    yield fx
    fx.close()


def test_long_read_records_hit_their_limits():
    rs, c, anchor, start = _long_fixture_data()
    assert int(rs.descs["seq_len"][:, 0].min()) >= 16500 and int(rs.descs["seq_len"].max()) <= 17000
    e8 = _entries(c, anchor, start)
    for raw, layout in ((_raw(F.short_candidates(c)), SHORT_FIELDS), (_raw(e8), ENTRY_FIELDS)):
        v = _unpack(raw, layout)
        _assert_hits(v, layout, ("pos1", "pos2", "ori1", "ori2"))
        assert ((v["pos1"] >> np.uint64(13)) == 0).any()
    assert set(_unpack(_raw(e8), ENTRY_FIELDS)["role"].tolist()) == {0, 1}
    assert {(chr(a), chr(b)) for a, b in zip(c["type1"], c["type2"])} == {("s", "s"), ("p", "p")}


@pytest.mark.gpu
@pytest.mark.parametrize("kind", PARAM_KINDS)
@pytest.mark.parametrize("layout", ["packed", "planar"])
def test_long_reads_at_the_14_bit_limits(built_lib, long_reads, layout, kind):
    """POS 8191 / 8192 / 16383 on 16.5-17 kb reads through the 12- and 8-byte records, full and small outputs."""
    fx = long_reads
    params = _params(kind, fx.rs, fx.c, fx.params)
    per, _ = _score_forms(fx.store(layout), fx.rs, params, fx.c, fx.anchor, fx.start, ("short", "runs"), ref=fx.ref(kind))
    assert (per["cls"] == F.CLASS_EDGE).sum() >= 5 and (per["status"][:, 0] == 1).all()


# ---- 1c. 28-bit POS1 ---------------------------------------------------------------------------------------------------
BIG = (1 << 28) + 2000
POS28 = ((1 << 27) - 1, 1 << 27, (1 << 28) - 1)


def _pos28_cands():
    """Read 0 is the long single, 1-3 singles copied from it at POS28, 4-5 pairs whose mate 0 lies at POS28[0] / [2]
    and mate 1 3000 bases earlier.  Every B at every POS28 in four ori, and one short A at 2^28 - 1 (POS_OOR)."""
    pos2 = {4: POS28[0] - 3000, 5: POS28[2] - 3000}
    rows = []
    for b in range(1, 6):
        t = "p" if b >= 4 else "s"
        for p1 in POS28:
            for o1 in (0, 1):
                for o2 in (0, 1):
                    rows.append((0, b, p1, pos2.get(b, 0), "-", o1, o2, "s", t))
    rows.append((1, 0, POS28[2], 0, "-", 1, 1, "s", "s"))
    c = _mk(rows)
    return _runs_by_anchor(c, np.minimum(c["idx1"], c["idx2"]))


def _pos28_readset():
    rng = np.random.RandomState(28)
    codes = rng.randint(0, 4, size=BIG, dtype=np.uint8)
    big = _ACGT[codes]
    bigq = rng.randint(33 + 20, 33 + 42, size=BIG, dtype=np.uint8)
    segs = [(0, BIG)] + [(p, int(rng.randint(600, 901))) for p in POS28]
    segs += [(POS28[0], 800), (POS28[0] - 3000, 700), (POS28[2], 900), (POS28[2] - 3000, 650)]
    bases = [big]
    quals = [bigq]
    for p, L in segs[1:]:
        bases.append(_ACGT[_substitute(codes[p:p + L], rng)])
        quals.append((33 + rng.randint(20, 42, size=L)).astype(np.uint8))
    lens = [L for _, L in segs]
    descs = np.zeros(6, dtype=F.READ_DESC)
    off = np.r_[0, np.cumsum(lens)].astype(np.uint64)
    for i in range(4):
        descs[i]["seq_off"][0], descs[i]["seq_len"][0] = off[i], lens[i]
    for j, i in enumerate((4, 5)):
        k = 4 + 2 * j
        descs[i]["seq_off"] = (off[k], off[k + 1])
        descs[i]["seq_len"] = (lens[k], lens[k + 1])
    return F.ReadSet(ids=np.arange(6, dtype=np.uint64), descs=descs, bases=np.concatenate(bases), quals=np.concatenate(quals),
                     n_single=4)


@pytest.fixture(scope="module")
def pos28():
    fx = _Fixture(_pos28_readset(), *_pos28_cands())
    yield fx
    fx.close()


def test_pos28_records_hit_their_limits():
    c, _, _ = _pos28_cands()
    v = _unpack(_raw(F.compact_candidates(c)), COMPACT_FIELDS)
    _assert_hits(v, COMPACT_FIELDS, ("pos1", "ori1", "ori2"))
    assert ((v["pos1"] >> np.uint64(27)) == 0).any() and (v["pos2"] > (1 << 27)).any()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", PARAM_KINDS)
@pytest.mark.parametrize("layout", ["packed", "planar"])
def test_pos28_through_the_16_byte_record(built_lib, pos28, layout, kind):
    """POS1 2^27 - 1, 2^27 and 2^28 - 1 on a read of 2^28 + 2000 bases through the 16-byte record."""
    fx = pos28
    params = _params(kind, fx.rs, fx.c, fx.params)
    per, _ = _score_forms(fx.store(layout), fx.rs, params, fx.c, fx.anchor, fx.start, ("compact",), ref=fx.ref(kind))
    assert (per["cls"] == F.CLASS_EDGE).any() and (per["status"][fx.c["idx1"] == 1, 0] == 2).all()


# ---- encoders ---------------------------------------------------------------------------------------------------------
def _random_cands(n, seed, max_idx, max_pos1, max_pos2):
    rng = np.random.RandomState(seed)
    c = np.zeros(n, dtype=F.CANDIDATE)
    c["idx1"] = rng.randint(0, 40, size=n)                 # few distinct anchors: runs form when sorted
    c["idx2"] = rng.randint(0, max_idx + 1, size=n, dtype=np.int64)
    c["idx2"][:4] = (max_idx, max_idx - 1, 1 << 24, 0)
    c["pos1"] = rng.randint(0, max_pos1 + 1, size=n, dtype=np.int64)
    c["pos2"] = rng.randint(0, max_pos2 + 1, size=n, dtype=np.int64)
    c["pos1"][:2], c["pos2"][:2] = max_pos1, max_pos2
    c["ori1"], c["ori2"] = rng.randint(0, 2, size=n), rng.randint(0, 2, size=n)
    c["ord"] = np.array([ord(x) for x in "-12"])[rng.randint(0, 3, size=n)]
    c = c[np.argsort(c["idx1"], kind="stable")]
    return c[c["idx1"] != c["idx2"]]


@pytest.mark.parametrize("seed", [1, 2])
def test_encoders_match_a_bit_by_bit_encoder(seed):
    c = _random_cands(3000, seed, (1 << 25) - 1, 511, 511)
    rows = [_cand_fields(x) for x in c]
    assert _raw(F.compact_candidates(c)).tobytes() == _enc(COMPACT_FIELDS, 16, rows)
    assert _raw(F.short_candidates(c)).tobytes() == _enc(SHORT_FIELDS, 12, rows)
    anchor, start, e8 = F.run_encode(c)
    assert start[0] == 0 and start[-1] == len(c) and (np.diff(start.astype(np.int64)) > 0).all() and len(anchor) < len(c) // 4
    erows = [_entry_fields(x, int(a)) for x, a in zip(c, _per_cand_anchor(anchor, start))]
    assert _raw(e8).tobytes() == _enc(ENTRY_FIELDS, 8, erows)
    assert F.entries6(e8).tobytes() == _enc(ENTRY6_FIELDS, 6, erows)
    # the decoder reads back what the encoder wrote
    v = _unpack(_raw(F.entries6(e8)), ENTRY6_FIELDS)
    assert np.array_equal(v["other"], np.array([r["other"] for r in erows], dtype=np.uint64))
    # 28-bit POS1, 32-bit POS2 and 14-bit positions at their maxima
    cw = _random_cands(500, seed + 10, (1 << 31) - 1, (1 << 28) - 1, (1 << 32) - 1)
    assert _raw(F.compact_candidates(cw)).tobytes() == _enc(COMPACT_FIELDS, 16, [_cand_fields(x) for x in cw])
    cs = _random_cands(500, seed + 20, (1 << 31) - 1, (1 << 14) - 1, (1 << 14) - 1)
    srows = [_cand_fields(x) for x in cs]
    assert _raw(F.short_candidates(cs)).tobytes() == _enc(SHORT_FIELDS, 12, srows)
    anchor, start, e8 = F.run_encode(cs)
    assert _raw(e8).tobytes() == _enc(ENTRY_FIELDS, 8, [_entry_fields(x, int(a)) for x, a in zip(cs, _per_cand_anchor(anchor, start))])


def _one(idx1=5, idx2=9, pos1=0, pos2=0):
    return _mk([(idx1, idx2, pos1, pos2, "1", 1, 0, "p", "p")])


@pytest.mark.parametrize("encode, ok, bad", [
    ("entries6", dict(pos1=511), dict(pos1=512)),
    ("entries6", dict(pos2=511), dict(pos2=512)),
    ("entries6", dict(idx2=(1 << 25) - 1), dict(idx2=1 << 25)),
    ("short", dict(pos1=(1 << 14) - 1), dict(pos1=1 << 14)),
    ("short", dict(pos2=(1 << 14) - 1), dict(pos2=1 << 14)),
    ("compact", dict(pos1=(1 << 28) - 1), dict(pos1=1 << 28)),
    ("runs", dict(idx2=(1 << 31) - 1), dict(idx2=1 << 31)),
])
def test_encoders_reject_the_first_value_out_of_range(encode, ok, bad):
    fn = {"entries6": lambda c: F.entries6(F.run_encode(c)[2]), "short": F.short_candidates, "compact": F.compact_candidates,
          "runs": lambda c: F.run_encode(c)[2]}[encode]
    layout = {"entries6": ENTRY6_FIELDS, "short": SHORT_FIELDS, "compact": COMPACT_FIELDS, "runs": ENTRY_FIELDS}[encode]
    v = _unpack(_raw(fn(_one(**ok))), layout)
    want = dict(ok)
    if "idx2" in want:
        want = {"other": want["idx2"]}
    for name, x in want.items():
        assert int(v[name][0]) == x
    with pytest.raises(ValueError):
        fn(_one(**bad))


# ---- 2. hand-made runs through the host pipeline -----------------------------------------------------------------------
N_BIG = 100003
STEP_EDGES = (64, 65, 128, 129, 1024, 1025, 2048, 2049, 4160, 4161, 8320, 8321)   # step starts (64, 1024, 4160) and one past


def _run_pool():
    ss = W.synth_readset(150, 150, seed=31, n_rate=0.002)
    c = W.geometry_candidates(ss, 6000, seed=32, junk_fraction=0.1)
    return ss.rs, c[(c["pos1"] < 512) & (c["pos2"] < 512)]


def _sample_runs(rng, pool, lens, id2_only=False):
    """One run per length: a read with candidates and that many of them (with repeats), anchored on that read."""
    role_of = [pool["idx2"]] if id2_only else [pool["idx1"], pool["idx2"]]
    reads = np.unique(np.concatenate(role_of))
    parts, anchor = [], []
    for L in lens:
        r = int(rng.choice(reads))
        mine = np.flatnonzero(np.any([x == r for x in role_of], axis=0))
        parts.append(pool[rng.choice(mine, size=L)])
        anchor.append(r)
    start = np.r_[0, np.cumsum(lens)].astype(np.uint64)
    return np.concatenate(parts), np.array(anchor, dtype=np.uint32), start


def _lens_through(rng, n, choices, forced=()):
    """Run lengths drawn from `choices` whose starts include every position of `forced`."""
    starts, pos = {0}, 0
    while pos < n:
        pos += int(rng.choice(choices))
        starts.add(min(pos, n))
    starts |= {x for x in forced if x < n}
    return np.diff(np.array(sorted(starts | {n})))


def _run_shapes():
    rs, pool = _run_pool()
    rng = np.random.RandomState(33)
    shapes = {}
    sel = pool[rng.randint(0, len(pool), size=N_BIG)]                     # every candidate its own run, anchors alternate
    own = np.where(np.arange(N_BIG) % 2 == 0, sel["idx1"], sel["idx2"]).astype(np.uint32)
    shapes["own"] = (sel, own, np.arange(N_BIG + 1, dtype=np.uint64))
    for n in (1, 31, 32, 33, N_BIG):                                         # one run holds the whole batch
        shapes["whole%d" % n] = _sample_runs(rng, pool, [n])
    mixed = _lens_through(rng, N_BIG, (31, 32, 33, 63, 64, 65), STEP_EDGES)
    shapes["mixed"] = _sample_runs(rng, pool, mixed)
    c, anchor, start = _sample_runs(rng, pool, _lens_through(rng, 30011, (31, 32, 33, 63, 64, 65, 200)))
    cuts = np.array([rng.randint(int(start[k]) + 1, int(start[k + 1])) for k in range(0, len(anchor), 3) if start[k + 1] - start[k] > 1])
    k = np.searchsorted(start, cuts, side="right") - 1                      # split those runs in two with the same anchor
    shapes["split"] = (c, np.insert(anchor, k + 1, anchor[k]), np.unique(np.r_[start, cuts]).astype(np.uint64))
    shapes["id2"] = _sample_runs(rng, pool, _lens_through(rng, 30011, tuple(range(1, 201))), id2_only=True)
    return rs, pool, shapes


@pytest.fixture(scope="module")
def runs_data():
    rs, pool, shapes = _run_shapes()
    fx = _Fixture(rs, pool, None, None)
    fx.shapes = {name: (c, a, s, _entries(c, a, s)) for name, (c, a, s) in shapes.items()}
    fx.pinned = {}
    fx.full = {}
    yield fx
    fx.close()


def test_run_shapes_hit_their_limits():
    rs, pool, shapes = _run_shapes()
    for name, (c, anchor, start) in shapes.items():
        n = len(c)
        assert start[0] == 0 and start[-1] == n and (np.diff(start.astype(np.int64)) > 0).all(), name
        e = _entries(c, anchor, start)                                       # every candidate holds its run's anchor
        assert n % 32 != 0 or name == "whole32", name
        if name == "id2":
            assert (e["other"] >> 31 == 1).all()
    assert len(shapes["own"][1]) == N_BIG and set((_entries(*shapes["own"])["other"] >> 31).tolist()) == {0, 1}
    assert len(shapes["whole%d" % N_BIG][1]) == 1
    st = shapes["mixed"][2].astype(np.int64)
    assert set((st % 32).tolist()) == set(range(32)) and set(STEP_EDGES) <= set(st.tolist())
    assert set(np.diff(st).tolist()) >= {1, 31, 32, 33, 63, 64, 65}
    c, anchor, start = shapes["split"]
    assert (anchor[1:] == anchor[:-1]).sum() >= 50                          # adjacent runs with the same anchor
    assert max(np.diff(shapes["id2"][2].astype(np.int64))) > 3 * 64 and (pool["pos1"] < 512).all()


def _pinned_copy(fx, key, a):
    if key not in fx.pinned:
        buf = capi.host_alloc(max(a.nbytes, 1))
        buf[:a.nbytes] = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
        fx.pinned[key] = buf[:a.nbytes].view(a.dtype).reshape(a.shape)
    return fx.pinned[key]


def _runs_store(fx, layout):
    """The store of the run tests.  Its first call scores one run per candidate in two-slot mode with steps of 4160, so
    tile t < 130 of both slots of the run scratch holds run index 32 t of that call before any other call uses it.

    Why: a step that starts d candidates into a run relies on the host clipping that run's start to 0.  Unclipped, the
    start wraps; for d >= 32 hc_tile_runs then writes none of the run's tiles, and its candidates walk from whatever
    run index an earlier step left in the slot (for d < 32 the wrap lands on tile 0 and the tiles come out right).
    Tile 0 always holds run 0, the right start for any step, but tiles 1, 2, ... hold run indices > 0 after a
    one-run-per-candidate step.  In every test below the "own" shape runs first, so the whole-batch run of 100003 that
    follows meets such tiles in slot 1 at every step size in two-slot mode, and takes wrong anchors if the clip is
    missing; the "split" and "id2" shapes do too, at every step size, and "mixed" with steps of 64.  Seeding the store first keeps those stale values run indices of an earlier call (inside the run arrays'
    buffers) rather than uninitialised memory."""
    if layout not in fx.stores:
        st = fx.store(layout)
        c, anchor, start, e = fx.shapes["own"]
        with _env(HC_HOST_CHUNK="4160", HC_HOST_WHOLE_MAX="0"):
            _call_runs(st, F.make_params(), anchor, start, e)
    return fx.stores[layout]


@pytest.mark.gpu
@pytest.mark.parametrize("buffer", ["pageable", "pinned"])
@pytest.mark.parametrize("mode", ["whole", "two_slot"])
@pytest.mark.parametrize("chunk", [64, 1000, 4160])
@pytest.mark.parametrize("kind", PARAM_KINDS)
@pytest.mark.parametrize("layout", ["packed", "planar"])
def test_hand_made_runs_through_the_pipeline(built_lib, runs_data, layout, kind, chunk, mode, buffer):
    """Every run shape through hc_score_batch_runs, _runs_small and _runs6_small, with steps of 64, 1024 (HC_HOST_CHUNK=1000
    rounded up to a multiple of 64) and 4160 candidates that cut runs mid-run, exactly at a run start and one past it."""
    fx = runs_data
    st = _runs_store(fx, layout)
    params = _params(kind, fx.rs, fx.c, fx.params)
    with _env(HC_HOST_CHUNK=None, HC_HOST_WHOLE_MAX=None):
        for name, (c, anchor, start, e8) in fx.shapes.items():
            key = (layout, kind, name)
            if key not in fx.full:                                          # hc_score_batch on 32-byte records, one step
                ref, means = O.score_batch(fx.rs, params, c)
                e0, n0, p0, s0 = st.score_batch(params, c)
                _check_parity(p0, e0, n0, s0, ref, params, means)
                fx.full[key] = (p0, e0, n0)
    full_of = {name: fx.full[(layout, kind, name)] for name in fx.shapes}
    with _env(HC_HOST_CHUNK=str(chunk), HC_HOST_WHOLE_MAX="0" if mode == "two_slot" else None):
        for name, (c, anchor, start, e8) in fx.shapes.items():
            e6 = F.entries6(e8)
            if buffer == "pinned":
                e8, e6 = _pinned_copy(fx, (name, 8), e8), _pinned_copy(fx, (name, 6), e6)
            full = full_of[name]
            got = _call_runs(st, params, anchor, start, e8)
            _check_same_full(got, full)
            s8 = _call_small(st, params, "runs", e8, anchor, start)
            s6 = _call_small(st, params, "runs6", e6, anchor, start)
            for s in (s8, s6):
                _check_small(s, full, params)
            assert s8[0].tobytes() == s6[0].tobytes()
            if kind == "boundary" and name == "mixed":
                assert int(got[3]["n_exact"]) >= 1 and int(s6[3]["n_exact"]) >= 1


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["whole", "two_slot"])
@pytest.mark.parametrize("kind", PARAM_KINDS)
@pytest.mark.parametrize("layout", ["packed", "planar"])
def test_runs_across_two_devices(built_lib, runs_data, layout, kind, mode):
    """Two devices: the shard cut (a multiple of 64) inside a run, and batches of fewer than 64 x 2 candidates, where the
    first shard is empty.  One device's hc_score_batch on the 32-byte records is checked against the oracle, and the
    two devices' run entry points against it."""
    if capi.device_count() < 2:
        pytest.skip("needs two GPUs")
    fx = runs_data
    params = _params(kind, fx.rs, fx.c, fx.params)
    c, _, _, _ = fx.shapes["mixed"]
    n = len(c)
    cut = (n // 2) & ~63                                                     # where hc_score_batch cuts two shards
    rng = np.random.RandomState(34)
    lens = np.r_[_lens_through(rng, cut - 900, (31, 63, 65)), 2000, _lens_through(rng, n - cut - 1100, (31, 63, 65, 4000))]
    cases = [_sample_runs(rng, fx.c, lens)] + [_sample_runs(rng, fx.c, [n]) for n in (1, 33, 100)]
    cases.append(_sample_runs(rng, fx.c, [40, 7, 80]))
    with _store(fx.rs, layout) as one, _store(fx.rs, layout, n_devices=2) as two:
        fulls = []
        for c, _, _ in cases:
            fulls.append(_batch(one, params, c))
            ref, means = O.score_batch(fx.rs, params, c)
            _check_parity(*fulls[-1], ref, params, means)
        for chunk in (None, "64", "1000"):
            with _env(HC_HOST_CHUNK=chunk, HC_HOST_WHOLE_MAX="0" if mode == "two_slot" else None):
                for (c, anchor, start), full in zip(cases, fulls):
                    e8 = _entries(c, anchor, start)
                    _check_same_full(_call_runs(two, params, anchor, start, e8), full)
                    _check_small(_call_small(two, params, "runs", e8, anchor, start), full, params)
                    _check_small(_call_small(two, params, "runs6", F.entries6(e8), anchor, start), full, params)


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["runs", "runs_small", "runs6_small"])
def test_bad_run_starts_are_rejected(built_lib, runs_data, entry):
    """The three malformed run_start arrays of test_gpu_parity's hc_score_batch_runs check, and n_runs = 0 for n > 0, at
    every run entry point."""
    fx = runs_data
    c, anchor, start, _ = fx.shapes["mixed"]
    first = start[start < 200]
    c, anchor, start = c[:200], anchor[:len(first)], np.r_[first, 200].astype(np.uint64)
    e8 = _entries(c, anchor, start)
    rec = F.entries6(e8) if entry == "runs6_small" else e8
    L = capi.lib()
    st = _runs_store(fx, "packed")
    n = len(c)
    ne, nn = ctypes.c_uint64(0), ctypes.c_uint64(0)
    edges = np.zeros(n, dtype=F.EDGE)
    out = np.zeros(n, dtype=np.uint64)
    p = F.make_params()

    def call(a, s, n_runs):
        if entry == "runs":
            return L.hc_score_batch_runs(st.handle, p.ctypes.data, a.ctypes.data, s.ctypes.data, n_runs, rec.ctypes.data, n, None,
                                         edges.ctypes.data, n, ctypes.byref(ne), out.ctypes.data, n, ctypes.byref(nn), None)
        fn = L.hc_score_batch_runs6_small if entry == "runs6_small" else L.hc_score_batch_runs_small
        return fn(st.handle, p.ctypes.data, a.ctypes.data, s.ctypes.data, n_runs, rec.ctypes.data, n, edges.ctypes.data, n,
                  ctypes.byref(ne), out.ctypes.data, ctypes.byref(nn), None)

    assert call(anchor, start, len(anchor)) == 0
    for bad in (start[::-1].copy(), np.concatenate((start[:1], start[:-1])), start + 1):
        assert call(anchor, bad, len(anchor)) == -1 and "run_start must begin at 0 and end at n" in capi.last_error()
    empty = np.r_[start[:2], start[1:]].astype(np.uint64)                   # begins at 0, ends at n, one empty run
    assert call(np.r_[anchor[:1], anchor].astype(np.uint32), empty, len(anchor) + 1) == -1
    assert "strictly increasing" in capi.last_error()
    assert call(anchor, start, 0) == -1 and "run arrays" in capi.last_error()
