"""GPU suite (-m gpu): the CUDA path, called through the C ABI, against
  * the golden fixtures (outputs of the UNMODIFIED reference C++), and
  * the plain-C oracle on fresh seeded inputs and on hand-made edge cases.
Bar: classes, accepted-edge list and its order, non-edge list, pos3/pos4, mismatch counts and
mismatch rates bit-exact; scores within 1e-6 relative (tolerance stated in util.assert_results_match).
"""
import numpy as np
import pytest

from haploconduct_b200 import capi, formats as F, workloads as W
from oracle import oracle as O
from util import assert_results_match, golden_names, load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, params=["packed", "planar"])
def store_layout(request, monkeypatch):
    """Every test runs on both device layouts: the packed one (one byte per base, used when the store
    has <= 63 distinct quality values) and the three-plane one (forced through HC_STORE_LAYOUT)."""
    monkeypatch.setenv("HC_STORE_LAYOUT", "planar" if request.param == "planar" else "auto")
    return request.param


def _check_lists(edges, nonedge, per, n):
    """edges / non-edges are exactly the class-1 / class-2 candidates, in input order."""
    ei = np.nonzero(per["cls"] == F.CLASS_EDGE)[0]
    ni = np.nonzero(per["cls"] == F.CLASS_NONEDGE)[0]
    assert np.array_equal(edges["cand"], ei.astype(np.uint64))
    assert np.array_equal(nonedge, ni.astype(np.uint64))
    assert np.array_equal(edges["score"], per["score"][ei])
    assert np.array_equal(edges["mismatch_rate"], per["mismatch_rate"][ei])
    assert np.array_equal(edges["pos3"], per["pos3"][ei]) and np.array_equal(edges["pos4"], per["pos4"][ei])


def _against_oracle(rs, params, cands, store=None, rel=1e-6):
    own = store is None
    st = store or capi.Store(rs)
    try:
        edges, nonedge, per, stats = st.score_batch(params, cands)
    finally:
        if own:
            st.close()
    ref, _ = O.score_batch(rs, params, cands)
    assert_results_match(per, ref["score"], ref["mismatch_rate"], ref["pos3"], ref["pos4"], ref["cls"], rel=rel, what="vs oracle")
    assert np.array_equal(per["mismatches"], ref["mismatches"])
    assert np.array_equal(per["compared"], ref["compared"])
    assert np.array_equal(per["status"], ref["status"])
    _check_lists(edges, nonedge, per, len(cands))
    assert int(stats["n_candidates"]) == len(cands)
    assert int(stats["n_edges"]) == len(edges) and int(stats["n_nonedges"]) == len(nonedge)
    assert int(stats["n_positions"]) == int(O.window_lengths(ref).sum())
    return per, ref, stats


@pytest.mark.parametrize("name", golden_names())
def test_golden_reference_outputs(built_lib, name):
    g = load_golden(name)
    cands = g.scored()
    with capi.Store(g.rs) as st:
        edges, nonedge, per, stats = st.score_batch(g.params(), cands)
    ref = g.ref_cands
    assert_results_match(per, ref["score"], ref["mismatch_rate"], ref["pos3"], ref["pos4"], ref["cls"], what=name)
    _check_lists(edges, nonedge, per, len(cands))
    # the candidates the reference wrote to nonedge_overlaps.txt (scored ones come first, src/EdgeCalculator.cpp:546-555)
    lines = F.candidates_to_lines(cands[nonedge.astype(np.int64)], g.rs.ids)
    assert [l.rstrip("\n") for l in lines] == g.ref_nonedge[: len(lines)]


@pytest.mark.parametrize("name", golden_names())
def test_golden_exact_edge_scores(built_lib, name):
    """HC_FLAG_EXACT_EDGE_SCORES: accepted edges are re-summed in the reference's order; what is left
    is the device exp() against glibc's (<= 2 ulp)."""
    g = load_golden(name)
    cands = g.scored()
    with capi.Store(g.rs) as st:
        edges, nonedge, per, stats = st.score_batch(g.params(flags=F.FLAG_EXACT_EDGE_SCORES), cands)
    ref = g.ref_cands
    assert_results_match(per, ref["score"], ref["mismatch_rate"], ref["pos3"], ref["pos4"], ref["cls"], what=name)
    e = ref["cls"] == F.CLASS_EDGE
    assert (per["exact"][e] == 1).all()
    assert np.allclose(per["score"][e], ref["score"][e], rtol=1e-15, atol=0)


def test_reference_order_pass_many_and_few(built_lib):
    """The reference-order pass runs one warp per queued candidate when few are queued and one thread each when many
    are (every accepted edge under HC_FLAG_EXACT_EDGE_SCORES): both give the oracle's sums (scores to 1e-14: device exp)."""
    ss = W.synth_readset(400, 400, seed=777, n_rate=0.002)
    c = W.geometry_candidates(ss, 40000, seed=778)
    px = F.make_params(edge_threshold=0.9, mismatch=0.0, flags=F.FLAG_EXACT_EDGE_SCORES)
    per, ref, stats = _against_oracle(ss.rs, px, c)
    edges = ref["cls"] == F.CLASS_EDGE
    assert edges.sum() > 6000 and (per["exact"][edges] == 1).all()          # more than 148*8*128/32 queued: thread mode
    assert np.allclose(per["score"][edges], ref["score"][edges], rtol=1e-14, atol=0)
    per2, ref2, _ = _against_oracle(ss.rs, px, c[:3000])                      # few queued: warp mode
    e2 = ref2["cls"] == F.CLASS_EDGE
    assert 0 < e2.sum() < 4000 and (per2["exact"][e2] == 1).all()
    assert np.allclose(per2["score"][e2], ref2["score"][e2], rtol=1e-14, atol=0)
    assert per2.tobytes() == per[:3000].tobytes()
    # the same with void quality pairs (p < mismatch) and a high N rate: the wide-table thread mode decides neither per position
    ss3 = W.synth_readset(400, 400, seed=779, n_rate=0.02)
    c3 = W.geometry_candidates(ss3, 40000, seed=780)
    for kw in (dict(edge_threshold=0.8, mismatch=0.02), dict(edge_threshold=0.5, ov_threshold=0.3, mismatch=0.0)):
        per3, ref3, _ = _against_oracle(ss3.rs, F.make_params(flags=F.FLAG_EXACT_EDGE_SCORES, **kw), c3)
        e3 = ref3["cls"] == F.CLASS_EDGE
        assert e3.sum() > 4000 and (per3["exact"][e3] == 1).all()
        assert np.allclose(per3["score"][e3], ref3["score"][e3], rtol=1e-14, atol=0)


def test_fresh_inputs_all_types(built_lib):
    ss = W.synth_readset(400, 400, seed=4242, n_rate=0.002)
    c = W.geometry_candidates(ss, 20000, seed=4243)
    for kw in (dict(edge_threshold=0.97), dict(edge_threshold=0.9, ov_threshold=0.6, merge_contigs=0.02, min_read_len=130),
               dict(edge_threshold=1.0), dict(edge_threshold=0.99, mismatch=0.02)):
        _against_oracle(ss.rs, F.make_params(**kw), c)


def test_threshold_boundaries_are_decided_like_the_reference(built_lib):
    """Thresholds placed exactly ON reference scores: 'score > threshold' must flip at the same
    candidates as in the reference.  These go through the reference-order pass (exact == 1)."""
    g = load_golden("synth_all_types")
    cands = g.scored()
    ref = g.ref_cands
    order = np.argsort(ref["score"])
    picks = [i for i in order[len(order) // 3::97] if 0.5 < ref["score"][i] < 0.9999][:12]
    assert len(picks) >= 6
    flips = []
    with capi.Store(g.rs) as st:
        for i in picks:
            s = float(ref["score"][i])
            for thr in (s, float(np.nextafter(s, 0.0)), float(np.nextafter(s, 1.0))):
                p = F.make_params(edge_threshold=thr, ov_threshold=min(0.5, thr))
                edges, nonedge, per, stats = st.score_batch(p, cands)
                oref, _ = O.score_batch(g.rs, p, cands)
                assert np.array_equal(per["cls"], oref["cls"]), (i, thr)
                assert int(stats["n_exact"]) >= 1
                flips.append(int(per["cls"][i]))
    assert 0 in flips or 2 in flips
    assert 1 in flips   # listed boundary cases: decided identically on both sides of the threshold


def _mk_cand(i1, i2, pos1, pos2=0, ord_="-", o1=1, o2=1, t1="s", t2="s", l1=1, l2=0):
    c = np.zeros(1, dtype=F.CANDIDATE)
    c["idx1"], c["idx2"], c["pos1"], c["pos2"], c["len1"], c["len2"] = i1, i2, pos1, pos2, l1, l2
    c["ord"], c["ori1"], c["ori2"], c["type1"], c["type2"] = ord(ord_), o1, o2, ord(t1), ord(t2)
    c["perc1"] = 50
    return c


def test_ragged_windows_and_chunk_boundaries(built_lib):
    rng = np.random.RandomState(5)
    def rnd(n):
        return "".join("ACGT"[k] for k in rng.randint(0, 4, size=n))
    def q(n):
        return "".join(chr(33 + k) for k in rng.randint(0, 42, size=n))
    base = rnd(400)
    singles = []
    lens = [1, 2, 15, 16, 17, 31, 32, 33, 47, 48, 49, 63, 64, 65, 100, 127, 128, 129, 255, 256, 257, 400]
    for k, L in enumerate(lens):
        singles.append((k, base[:L], q(L)))
    n0 = len(singles)
    for k, L in enumerate(lens):       # suffixes, so that reverse windows are unaligned in every way
        singles.append((n0 + k, base[400 - L:], q(L)))
    singles.append((2 * n0, "N" * 40, "!" * 40))
    singles.append((2 * n0 + 1, base[:20] + "N" * 5 + base[25:60], q(60)))
    rs = F.ReadSet.from_lists(singles, [])
    cs = []
    n = rs.n_reads
    for a in range(n):
        for b in range(n):
            if a == b:
                continue
            la = int(rs.descs[a]["seq_len"][0])
            for pos in sorted({0, 1, 3, la // 2, max(la - 17, 0), max(la - 16, 0), max(la - 1, 0), la, la + 5}):
                for o1, o2 in ((1, 1), (0, 1), (1, 0), (0, 0)):
                    cs.append(_mk_cand(a, b, pos, o1=o1, o2=o2))
    c = np.concatenate(cs)
    per, ref, stats = _against_oracle(rs, F.make_params(edge_threshold=0.9, ov_threshold=0.3), c)
    assert set(np.unique(per["status"][:, 0])) >= {1, 2, 5}   # scored, pos out of range, empty (all N)


@pytest.mark.parametrize("n_quals", [94, 63])
def test_long_contigs_and_wide_quality_alphabet(built_lib, n_quals):
    """1-10 kb contigs (config 5): warp-cooperative path, windows far longer than one warp round,
    94 distinct quality values (7-bit codes, the largest score table) or 63 including Phred 0 and 93 (the most the
    packed layout holds: every code bit in use)."""
    qset = np.arange(94) if n_quals == 94 else np.array([0, 93] + list(range(2, 63)))
    rng = np.random.RandomState(9)
    genome = rng.randint(0, 4, size=30000)
    singles = []
    segs = []
    for k in range(60):
        L = int(np.exp(rng.uniform(np.log(1000), np.log(10000))))
        st = int(rng.randint(0, 30000 - L))
        seg = genome[st:st + L].copy()
        mut = rng.random_sample(L) < (0.0 if k % 3 else 0.004)
        seg[mut] = (seg[mut] + 1) % 4
        s = "".join("ACGT"[x] for x in seg)
        qv = qset[rng.randint(0, len(qset), size=L)]
        singles.append((k, s, "".join(chr(33 + x) for x in qv)))
        segs.append((st, st + L))
    rs = F.ReadSet.from_lists(singles, [])
    cs = []
    for a in range(60):
        for b in range(60):
            if a != b and segs[a][0] <= segs[b][0] < segs[a][1] - 50:
                cs.append(_mk_cand(a, b, segs[b][0] - segs[a][0], l1=min(segs[a][1], segs[b][1]) - segs[b][0]))
                cs.append(_mk_cand(a, b, segs[b][0] - segs[a][0] + 1))
    c = np.concatenate(cs)
    with capi.Store(rs) as st:
        assert st.quality_alphabet == n_quals
        per, ref, stats = _against_oracle(rs, F.make_params(edge_threshold=0.995, min_read_len=100), c, store=st)
    assert int(O.window_lengths(ref).max()) > 4096
    assert not per["indel_count"].any()            # the path compares gaplessly: no indels (SURVEY 8a)


def test_empty_single_and_capacity(built_lib):
    g = load_golden("c2_polyte_example_it1")
    cands = g.scored()
    with capi.Store(g.rs) as st:
        e, n, per, stats = st.score_batch(g.params(), cands[:0])
        assert len(e) == 0 and len(n) == 0 and int(stats["n_candidates"]) == 0
        e1, n1, per1, _ = st.score_batch(g.params(), cands[:1])
        ref, _ = O.score_batch(g.rs, g.params(), cands[:1])
        assert per1["cls"][0] == ref["cls"][0]
        efull, nfull, _, _ = st.score_batch(g.params(), cands)
        assert len(efull) > 2
        with pytest.raises(capi.HcError) as ei:
            st.score_batch(g.params(), cands, edges_cap=2)
        assert ei.value.code == -5 and ei.value.required == (len(efull), len(nfull))
        bad = cands[:4].copy()
        bad["idx2"][2] = g.rs.n_reads + 7
        with pytest.raises(capi.HcError) as ei:
            st.score_batch(g.params(), bad)
        assert ei.value.code == -1
        # the store is still usable afterwards
        e2, n2, _, _ = st.score_batch(g.params(), cands)
        assert e2.tobytes() == efull.tobytes() and np.array_equal(n2, nfull)   # bytes: mean_log of an unused window is NaN


def test_invalid_input_is_rejected_like_the_reference(built_lib):
    with pytest.raises(capi.HcError):
        capi.Store(F.ReadSet.from_lists([(0, "ACGU", "IIII"), (1, "ACGT", "IIII")], []))     # assert in score(), :29-30
    with pytest.raises(capi.HcError):
        capi.Store(F.ReadSet.from_lists([], [(0, "acgt", "IIII", "ACGT", "IIII")]))          # pairs are not upper-cased
    with pytest.raises(capi.HcError):
        capi.Store(F.ReadSet.from_lists([(0, "ACGT", "II I"), (1, "ACGT", "IIII")], []))     # Q < 0


def test_overlap_score_primitive(built_lib):
    p = F.make_params()
    rng = np.random.RandomState(3)
    for _ in range(5):
        a = "".join("ACGT"[k] for k in rng.randint(0, 4, size=120))
        b = a[40:] + "ACGTACGT"
        qa = "".join(chr(33 + k) for k in rng.randint(2, 42, size=len(a)))
        qb = "".join(chr(33 + k) for k in rng.randint(2, 42, size=len(b)))
        s, mm = capi.overlap_score(a, b, qa, qb, 40, p)
        so, mmo = O.overlap_score(a, b, qa, qb, 40, p)
        assert mm == mmo and abs(s - so) <= 1e-6 * so
    s, mm = capi.overlap_score("ACGT", "ACGT", "IIII", "IIII", 4, p)
    assert s == 0.0 and mm == 1.0


def test_larger_random_batch_and_determinism(built_lib):
    ss = W.synth_readset(0, 1500, seed=77, n_rate=0.0005, pair_len=(150, 150), genome_len=4000)
    c = W.geometry_candidates(ss, 30000, seed=78, junk_fraction=0.05)
    c = np.tile(c, 8)
    p = F.make_params(edge_threshold=0.97)
    with capi.Store(ss.rs) as st:
        per, ref, stats = _against_oracle(ss.rs, p, c, store=st)
        e1, n1, per1, _ = st.score_batch(p, c)
        e2, n2, per2, _ = st.score_batch(p, c[::-1].copy())
    # integer sums: the result of a candidate does not depend on its position in the batch
    assert np.array_equal(per1, per) and np.array_equal(per2[::-1], per1)


@pytest.mark.parametrize("whole_max", ["0", ""])
@pytest.mark.parametrize("chunk", ["777", "100000000"])
def test_chunked_pipeline_and_compact_records(built_lib, monkeypatch, chunk, whole_max):
    """hc_score_batch streams the batch through the device in steps (3 streams; the records either all copied ahead into
    one buffer -- the default up to 2 GB -- or through two slots, forced here with HC_HOST_WHOLE_MAX=0); the step
    size must not change anything, and the 16-byte compact records give the same results."""
    if whole_max:
        monkeypatch.setenv("HC_HOST_WHOLE_MAX", whole_max)
    g = load_golden("synth_all_types")
    cands = np.tile(g.scored(), 3)
    p = g.params()
    with capi.Store(g.rs) as st:
        monkeypatch.setenv("HC_HOST_CHUNK", "100000000")
        e0, n0, per0, s0 = st.score_batch(p, cands)
        monkeypatch.setenv("HC_HOST_CHUNK", chunk)
        e1, n1, per1, s1 = st.score_batch(p, cands)
        e2, n2, per2, s2 = st.score_batch(p, cands, compact=True)
        e3, n3, _, _ = st.score_batch(p, cands, per_candidate=False, compact=True, edges_cap=len(e0), nonedge_cap=len(n0))
        fits = (cands["pos1"] < (1 << 14)) & (cands["pos2"] < (1 << 14))      # the 12-byte records hold 14-bit positions
        e4, n4, per4, s4 = st.score_batch(p, cands[fits], compact="short")
        e5, n5, per5, s5 = st.score_batch(p, cands[fits])
    assert fits.sum() > 0.9 * len(cands) and not fits.all()
    with pytest.raises(ValueError):
        F.short_candidates(cands)
    assert e4.tobytes() == e5.tobytes() and np.array_equal(n4, n5) and per4.tobytes() == per5.tobytes()
    assert per4.tobytes() == per0[fits].tobytes()
    for e, n, per, s in ((e1, n1, per1, s1), (e2, n2, per2, s2)):
        assert e.tobytes() == e0.tobytes() and np.array_equal(n, n0) and per.tobytes() == per0.tobytes()
        assert int(s["n_positions"]) == int(s0["n_positions"]) and int(s["n_edges"]) == len(e0)
    assert e3.tobytes() == e0.tobytes() and np.array_equal(n3, n0)
    ref = np.tile(g.ref_cands, 3)
    assert np.array_equal(per1["cls"], ref["cls"])


@pytest.mark.parametrize("whole_max", ["0", ""])
@pytest.mark.parametrize("chunk", ["33", "777", "100000000"])
@pytest.mark.parametrize("order", ["file", "by_read", "by_min_id"])
def test_run_encoded_records(built_lib, monkeypatch, chunk, order, whole_max):
    """hc_score_batch_runs (8-byte records, the shared read of a run held once): same edges, non-edge indices and
    per-candidate results as the 12-byte records, whatever the order of the list (long runs when it is sorted by
    read, runs of length 1 otherwise) and wherever the pipeline cuts it."""
    if whole_max:
        monkeypatch.setenv("HC_HOST_WHOLE_MAX", whole_max)
    g = load_golden("synth_all_types")
    cands = np.tile(g.scored(), 3)
    cands = cands[(cands["pos1"] < (1 << 14)) & (cands["pos2"] < (1 << 14))]
    if order == "by_read":
        cands = cands[np.argsort(cands["idx1"], kind="stable")]
    elif order == "by_min_id":
        lo, hi = np.minimum(cands["idx1"], cands["idx2"]), np.maximum(cands["idx1"], cands["idx2"])
        cands = cands[np.lexsort((hi, lo))]
    anchor, start, entries = F.run_encode(cands)
    assert start[0] == 0 and start[-1] == len(cands) and (np.diff(start.astype(np.int64)) > 0).all()
    if order != "file":
        assert len(anchor) < len(cands) // 2
    other = entries["other"] & 0x7fffffff
    flip = (entries["other"] >> 31).astype(bool)
    per_anchor = np.repeat(anchor, np.diff(start.astype(np.int64)))
    assert np.array_equal(np.where(flip, other, per_anchor), cands["idx1"]) and np.array_equal(np.where(flip, per_anchor, other), cands["idx2"])
    p = g.params()
    with capi.Store(g.rs) as st:
        monkeypatch.setenv("HC_HOST_CHUNK", "100000000")
        e0, n0, per0, s0 = st.score_batch(p, cands, compact="short")
        monkeypatch.setenv("HC_HOST_CHUNK", chunk)
        e1, n1, per1, s1 = st.score_batch(p, cands, compact="runs")
        e2, n2, _, _ = st.score_batch(p, cands, compact="runs", per_candidate=False)
        ez, nz, _, _ = st.score_batch(p, cands[:0], compact="runs")
    assert e1.tobytes() == e0.tobytes() and np.array_equal(n1, n0) and per1.tobytes() == per0.tobytes()
    assert e2.tobytes() == e0.tobytes() and np.array_equal(n2, n0)
    assert int(s1["n_positions"]) == int(s0["n_positions"]) and len(ez) == 0 and len(nz) == 0


def test_run_encoded_records_bad_runs(built_lib):
    g = load_golden("synth_all_types")
    cands = g.scored()[:50]
    cands = cands[(cands["pos1"] < (1 << 14)) & (cands["pos2"] < (1 << 14))]
    anchor, start, entries = F.run_encode(cands)
    L = capi.lib()
    import ctypes
    with capi.Store(g.rs) as st:
        ne, nn = ctypes.c_uint64(0), ctypes.c_uint64(0)
        edges = np.zeros(len(cands), dtype=F.EDGE); nonedge = np.zeros(len(cands), dtype=np.uint64)
        p = g.params()
        for bad in (start[::-1].copy(), np.concatenate((start[:1], start[:-1])), start + 1):
            rc = L.hc_score_batch_runs(st._h, p.ctypes.data, anchor.ctypes.data, bad.ctypes.data, len(anchor), entries.ctypes.data,
                                       len(entries), None, edges.ctypes.data, len(edges), ctypes.byref(ne), nonedge.ctypes.data,
                                       len(nonedge), ctypes.byref(nn), None)
            assert rc == -1 and "run_start" in capi.last_error()


def test_overlap_score_multi_self_overlap_scan(built_lib):
    """The scan of SRBuilder::merge_self_overlap (src/SRBuilder.cpp:880-888): seq2 slid over seq1 from
    pos = len1-15 downwards; first position whose score exceeds 0.99 -- same position as the oracle's loop."""
    rng = np.random.RandomState(21)
    left = "".join("ACGT"[k] for k in rng.randint(0, 4, size=180))
    right = left[120:] + "".join("ACGT"[k] for k in rng.randint(0, 4, size=140))     # true overlap starts at 120
    q1 = "".join(chr(33 + k) for k in rng.randint(25, 42, size=len(left)))
    q2 = "".join(chr(33 + k) for k in rng.randint(25, 42, size=len(right)))
    p = F.make_params(edge_threshold=0.99)
    pos = np.array([len(left) - 15 - k for k in range(len(left) - 15)], dtype=np.uint32)
    sc, mm, above = capi.overlap_score_multi(left, right, q1, q2, pos, p)
    want = [O.overlap_score(left, right, q1, q2, int(x), p) for x in pos]
    assert np.array_equal(mm, np.array([w[1] for w in want]))
    assert np.allclose(sc, np.array([w[0] for w in want]), rtol=1e-6, atol=0)
    assert np.array_equal(above, np.array([w[0] > 0.99 for w in want]))
    first = int(pos[np.nonzero(above)[0][0]])
    assert first == 120
