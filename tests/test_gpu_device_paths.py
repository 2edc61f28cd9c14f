"""GPU suite: the HBM-resident entry points on one GPU -- hc_score_batch_device (the call the throughput benchmark times)
and hc_ingest_overlaps_device -- against the goldens, the oracles and the host-buffer calls, which run the same kernels and
so must give the same bytes.  Every output buffer is filled with a sentinel byte first: what a call writes is compared,
and everything past it must still be the sentinel."""
import numpy as np
import pytest
import torch

from haploconduct_b200 import capi, formats as F, workloads as W, workloads_torch as WT
from oracle import ingest_oracle as IO, oracle as O
from util import IngestGolden, assert_results_match, golden_names, ingest_golden_names, load_golden

pytestmark = pytest.mark.gpu

SENT = 0xAB
PAD = 64                      # sentinel bytes behind every output buffer
NO_ERROR = 2 ** 64 - 1
INGEST_FIELDS = ("n_lines", "n_scored", "n_filtered", "n_skipped", "n_dropped", "first_error_line", "first_error_offset",
                 "first_error_length", "first_error_status")
TAIL_SIZES = (1, 31, 32, 33, 4095, 4096, 4097, 3 * 4096 + 5)     # 32-candidate tiles, 4096-candidate compaction blocks


@pytest.fixture(autouse=True, params=["packed", "planar"])
def store_layout(request, monkeypatch):
    """Every test runs on both device layouts (HC_STORE_LAYOUT=planar forces the three-plane one)."""
    monkeypatch.setenv("HC_STORE_LAYOUT", "planar" if request.param == "planar" else "auto")
    return request.param


def _ready():
    """torch fills tensors on its own stream; the library's calls run on others."""
    torch.cuda.synchronize()


def _dev(nbytes):
    return torch.full((nbytes + PAD,), SENT, dtype=torch.uint8, device="cuda")


def _written(buf, nbytes):
    """The first nbytes of a sentinel-filled device buffer; every byte behind them must still be the sentinel."""
    h = buf.cpu().numpy()
    assert (h[nbytes:] == SENT).all(), "bytes written past the first %d" % nbytes
    return h[:nbytes].tobytes()


def _to_dev(cands, offset=0):
    """hc_candidate records in a device tensor, starting `offset` records into it: (tensor, pointer to the first record)."""
    raw = np.zeros((offset + len(cands)) * 32 + PAD, dtype=np.uint8)
    raw[offset * 32:(offset + len(cands)) * 32] = np.ascontiguousarray(cands).view(np.uint8)
    t = torch.from_numpy(raw).cuda()
    return t, t.data_ptr() + 32 * offset


class DevOut:
    """The device outputs of one hc_score_batch_device call, sentinel-filled."""

    def __init__(self, n, edges_cap=None, nonedge_cap=None, per_cand=True):
        self.n = n
        self.ecap = n if edges_cap is None else edges_cap
        self.ncap = n if nonedge_cap is None else nonedge_cap
        self.per = _dev(48 * n) if per_cand else None
        self.edges = _dev(48 * self.ecap)
        self.nonedge = _dev(8 * self.ncap)
        self.counts = _dev(32)

    def call(self, st, p, d_cand, stream=None, stats=False):
        return st.score_batch_device(0, stream.cuda_stream if stream is not None else 0, p, d_cand, self.n,
                                     self.per.data_ptr() if self.per is not None else 0, self.edges.data_ptr(), self.ecap,
                                     self.nonedge.data_ptr(), self.ncap, self.counts.data_ptr(), stats)

    def read(self):
        """(counts, edges, non-edge indices, per-candidate results) as the call wrote them."""
        torch.cuda.synchronize()
        counts = np.frombuffer(_written(self.counts, 32), dtype=np.uint64)
        ne, nn = min(int(counts[0]), self.ecap), min(int(counts[1]), self.ncap)
        edges = np.frombuffer(_written(self.edges, 48 * ne), dtype=F.EDGE)
        nonedge = np.frombuffer(_written(self.nonedge, 8 * nn), dtype=np.uint64)
        per = np.frombuffer(_written(self.per, 48 * self.n), dtype=F.RESULT) if self.per is not None else None
        return counts, edges, nonedge, per


def _score_dev(st, p, d_cand, n, **kw):
    out = DevOut(n)
    _ready()
    out.call(st, p, d_cand, **kw)
    return out.read()


def _same_bytes(a, b):
    return all((x is None and y is None) or x.tobytes() == y.tobytes() for x, y in zip(a, b))


def _assert_same_as_host(got, host):
    counts, edges, nonedge, per = got
    he, hn, hp, hs = host
    assert counts.tolist() == [len(he), len(hn), int(hs["n_exact"]), 0]
    assert edges.tobytes() == he.tobytes(), "edge records differ from the host path"
    assert nonedge.tobytes() == hn.tobytes(), "non-edge indices differ from the host path"
    if per is not None:
        assert per.tobytes() == hp.tobytes(), "per-candidate results differ from the host path"


def _assert_matches_oracle(per, ref, exact=False, what=""):
    assert_results_match(per, ref["score"], ref["mismatch_rate"], ref["pos3"], ref["pos4"], ref["cls"], what=what)
    assert np.array_equal(per["mismatches"], ref["mismatches"]) and np.array_equal(per["compared"], ref["compared"])
    assert np.array_equal(per["status"], ref["status"])
    if exact:
        e = ref["cls"] == F.CLASS_EDGE
        assert (per["exact"][e] == 1).all()
        assert np.allclose(per["score"][e], ref["score"][e], rtol=1e-14, atol=0)


@pytest.fixture(scope="module")
def bench_shaped():
    """The benchmark's workload at a test size: 2x150 pairs, P-P candidates with D = 140 partners, generated and kept in HBM
    (about 2 M candidates)."""
    pr = WT.make_paired_reads(16_000, read_len=150, genome_len=4_000, seed=20261018, device="cuda")
    rec = WT.make_pp_candidates(pr, D=140, max_cands=2_000_000)
    torch.cuda.synchronize()
    return pr.readset(), rec


@pytest.fixture(scope="module")
def mixed():
    """Singles and pairs, every read-type combination, N bases: 20000 candidates."""
    ss = W.synth_readset(400, 400, seed=4242, n_rate=0.002)
    return ss.rs, W.geometry_candidates(ss, 20000, seed=4243)


BENCH_PARAMS = dict(edge_threshold=0.97, ov_threshold=0.9, merge_contigs=0.0, mismatch=0.0, min_read_len=0)


# ---- hc_score_batch_device ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", golden_names())
@pytest.mark.parametrize("exact", [False, True])
def test_goldens(built_lib, name, exact):
    g = load_golden(name)
    cands = g.scored()
    p = g.params(flags=F.FLAG_EXACT_EDGE_SCORES if exact else 0)
    with capi.Store(g.rs) as st:
        t, ptr = _to_dev(cands)
        got = _score_dev(st, p, ptr, len(cands))
        host = st.score_batch(p, cands)
    _assert_same_as_host(got, host)
    per, ref = got[3], g.ref_cands
    assert_results_match(per, ref["score"], ref["mismatch_rate"], ref["pos3"], ref["pos4"], ref["cls"], what=name)
    if exact:
        e = ref["cls"] == F.CLASS_EDGE
        assert (per["exact"][e] == 1).all()
        assert np.allclose(per["score"][e], ref["score"][e], rtol=1e-14, atol=0)


def test_bench_shaped_workload(built_lib, bench_shaped):
    rs, rec = bench_shaped
    n = rec.shape[0]
    assert n >= 1_500_000
    p = F.make_params(**BENCH_PARAMS)
    cands = WT.candidates_as_numpy(rec)          # for the host path and the oracle only: the device call reads `rec` in HBM
    with capi.Store(rs) as st:
        got = _score_dev(st, p, rec.data_ptr(), n)
        host = st.score_batch(p, cands)
    _assert_same_as_host(got, host)
    counts, edges, nonedge, per = got
    assert 0 < len(edges) < n and 0 < len(nonedge) < n
    pick = np.sort(np.random.RandomState(1).choice(n, size=40_000, replace=False))
    ref, _ = O.score_batch(rs, p, cands[pick])
    _assert_matches_oracle(per[pick], ref, what="sample")


def test_batch_tails_and_offsets(built_lib, mixed):
    """Batches of every tail size, at record offsets inside a larger tensor (as bench.py --device-chunk launches them): the
    matching slice of the whole batch's results, with indices relative to the call."""
    rs, c = mixed
    N = len(c)
    p = F.make_params(edge_threshold=0.97)
    offsets = (0, 1, 777)
    assert N >= max(offsets) + max(TAIL_SIZES)
    with capi.Store(rs) as st:
        t, base = _to_dev(c)
        whole = _score_dev(st, p, base, N)
        _assert_same_as_host(whole, st.score_batch(p, c))
        _, we, wn, wp = whole
        for o in offsets:
            for n in TAIL_SIZES:
                counts, e, ne, per = _score_dev(st, p, base + 32 * o, n)
                want_e = we[(we["cand"] >= o) & (we["cand"] < o + n)].copy()
                want_e["cand"] -= np.uint64(o)
                want_n = wn[(wn >= o) & (wn < o + n)] - np.uint64(o)
                assert per.tobytes() == wp[o:o + n].tobytes(), (o, n)
                assert e.tobytes() == want_e.tobytes() and ne.tobytes() == want_n.tobytes(), (o, n)
                assert int(counts[0]) == len(want_e) and int(counts[1]) == len(want_n) and int(counts[3]) == 0, (o, n)


def test_caller_streams_and_stats(built_lib, mixed):
    """A caller's stream, the NULL stream and the synchronous form with stats give the same bytes as the host path."""
    rs, c = mixed
    p = F.make_params(edge_threshold=0.9, ov_threshold=0.6, merge_contigs=0.02, min_read_len=130)
    with capi.Store(rs) as st:
        host = st.score_batch(p, c)
        t, ptr = _to_dev(c)
        for how in ("stream", "null", "stats"):
            s = torch.cuda.Stream() if how == "stream" else None
            out = DevOut(len(c))
            _ready()
            stats = out.call(st, p, ptr, stream=s, stats=how == "stats")
            _assert_same_as_host(out.read(), host)
            if how == "stats":
                for f in ("n_candidates", "n_edges", "n_nonedges", "n_positions"):
                    assert int(stats[f]) == int(host[3][f]), f
            else:
                assert stats is None


def test_capacities_truncate_the_lists(built_lib, mixed):
    """Capacities below the counts: HC_OK, full counts, exactly the first `cap` records written."""
    rs, c = mixed
    p = F.make_params(edge_threshold=0.97)
    with capi.Store(rs) as st:
        he, hn, _, hs = st.score_batch(p, c)
        ne, nn = len(he), len(hn)
        assert ne > 2 and nn > 2
        t, ptr = _to_dev(c)
        full = [ne, nn, int(hs["n_exact"]), 0]
        for ecap, ncap in ((0, nn), (1, nn), (ne - 1, nn), (ne, 0), (ne, 1), (ne, nn - 1), (0, 0), (1, 1)):
            out = DevOut(len(c), ecap, ncap, per_cand=False)
            _ready()
            out.call(st, p, ptr)                  # raises unless HC_OK
            counts, e, nonedge, _ = out.read()
            assert counts.tolist() == full, (ecap, ncap)
            assert e.tobytes() == he[:ecap].tobytes() and nonedge.tobytes() == hn[:ncap].tobytes(), (ecap, ncap)
        # NULL outputs with capacity 0: a counts-only call
        counts = _dev(32)
        _ready()
        st.score_batch_device(0, 0, p, ptr, len(c), 0, 0, 0, 0, 0, counts.data_ptr(), False)
        torch.cuda.synchronize()
        assert np.frombuffer(_written(counts, 32), dtype=np.uint64).tolist() == full


def test_invalid_candidates_and_empty_batch(built_lib):
    g = load_golden("synth_all_types")
    c = g.scored()
    p = g.params()
    paired = np.nonzero(g.rs.descs["seq_len"][:, 1] > 0)[0]
    bad = c[:3].copy()
    bad["idx2"][0] = g.rs.n_reads + 7                                  # read index outside the store
    bad["idx2"][1] = bad["idx1"][1]                                     # self overlap
    bad["idx1"][2], bad["idx2"][2], bad["ord"][2] = paired[0], paired[1], ord("-")   # P-P with ORD '-'
    is_bad = np.zeros(len(c) + 3, dtype=bool)
    is_bad[[5, 101, len(c) // 2]] = True
    mix = np.zeros(len(c) + 3, dtype=F.CANDIDATE)
    mix[is_bad], mix[~is_bad] = bad, c
    good_at = np.nonzero(~is_bad)[0].astype(np.uint64)                 # index in `mix` of every valid candidate
    with capi.Store(g.rs) as st:
        he, hn, hp, hs = host = st.score_batch(p, c)
        t, ptr = _to_dev(mix)
        counts, e, ne, per = _score_dev(st, p, ptr, len(mix))           # stats == NULL: HC_OK, the count in d_counts[3]
        assert counts.tolist() == [len(he), len(hn), int(hs["n_exact"]), 3]
        assert per[~is_bad].tobytes() == hp.tobytes()
        assert (per["cls"][is_bad] == F.CLASS_DISCARD).all()
        want_e = he.copy()
        want_e["cand"] = good_at[he["cand"].astype(np.int64)]
        assert e.tobytes() == want_e.tobytes() and np.array_equal(ne, good_at[hn.astype(np.int64)])
        out = DevOut(len(mix))
        _ready()
        with pytest.raises(capi.HcError) as ei:                         # with stats: HC_ERR_ARG
            out.call(st, p, ptr, stats=True)
        assert ei.value.code == -1
        torch.cuda.synchronize()
        empty = DevOut(0)
        _ready()
        empty.call(st, p, ptr)
        assert empty.read()[0].tolist() == [0, 0, 0, 0]
        t2, ptr2 = _to_dev(c)
        _assert_same_as_host(_score_dev(st, p, ptr2, len(c)), host)      # the store is still right afterwards


def test_argument_errors(built_lib):
    """NULL arguments, a device without a replica and misaligned pointers return HC_ERR_ARG before anything is enqueued
    (the counts buffer keeps its sentinel); the misaligned cases use n = 0, where no kernel touches the pointers."""
    g = load_golden("synth_mismatch_void")
    c = g.scored()
    p = g.params()
    n = len(c)
    L = capi.lib()
    with capi.Store(g.rs) as st:
        host = st.score_batch(p, c)
        t, ptr = _to_dev(c)
        out = DevOut(n)
        _ready()
        ok = [st.handle, 0, None, p.ctypes.data, ptr, n, out.per.data_ptr(), out.edges.data_ptr(), n, out.nonedge.data_ptr(), n,
              out.counts.data_ptr(), None]
        cases = {"store": (0, None), "params": (3, None), "d_counts": (11, None), "d_cand": (4, None),
                 "device": (1, capi.device_count())}
        for what, (k, v) in cases.items():
            a = list(ok)
            a[k] = v
            assert L.hc_score_batch_device(*a) == -1, what
        for what, k, shift in (("d_cand", 4, 8), ("d_cand", 4, 1), ("d_per_cand", 6, 4), ("d_edges", 7, 4), ("d_nonedge_idx", 9, 4),
                               ("d_counts", 11, 4)):
            a = list(ok)
            a[5] = 0
            a[k] = a[k] + shift
            assert L.hc_score_batch_device(*a) == -1, what
            assert "aligned" in capi.last_error(), what
        torch.cuda.synchronize()
        assert out.counts.cpu().numpy().tolist() == [SENT] * (32 + PAD)
        _assert_same_as_host(_score_dev(st, p, ptr, n), host)


def test_calls_sharing_the_workspace(built_lib, bench_shaped):
    """Calls on different streams with no synchronisation between them, and a device call followed by a host-buffer call:
    each gives the bytes it gives on its own.  The first call sizes the workspace for 2n, the overlapping calls take n
    candidates each and n-record outputs (so every index the kernels compute stays inside the allocations)."""
    rs, rec = bench_shaped
    n = rec.shape[0] // 2
    X, Y = rec.data_ptr(), rec.data_ptr() + 32 * n
    y_host = WT.candidates_as_numpy(rec[n:2 * n])
    p0 = F.make_params(**BENCH_PARAMS)
    px = F.make_params(flags=F.FLAG_EXACT_EDGE_SCORES, **BENCH_PARAMS)
    pm = F.make_params(**dict(BENCH_PARAMS, mismatch=0.02))
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    with capi.Store(rs) as st:
        warm = DevOut(2 * n, per_cand=False)
        _ready()
        warm.call(st, p0, X, stats=True)
        # each call on its own; the last one leaves the tables of mismatch 0 in place, so that in (c) the call on stream B
        # rebuilds them while the one on stream A may still run
        y_mm = _score_dev(st, pm, Y, n)
        y_ex = _score_dev(st, px, Y, n)
        h_alone = st.score_batch(p0, y_host)
        x_0 = _score_dev(st, p0, X, n)
        assert not _same_bytes(y_mm, y_ex)
        for second in ("exact on B", "host buffers", "new tables on B"):
            a = DevOut(n)
            b = DevOut(n) if second != "host buffers" else None
            _ready()
            a.call(st, p0, X, stream=sa)
            if second == "exact on B":
                b.call(st, px, Y, stream=sb)
            elif second == "new tables on B":
                b.call(st, pm, Y, stream=sb)
            else:
                h = st.score_batch(p0, y_host)
            assert _same_bytes(a.read(), x_0), second
            if b is None:
                assert all(x.tobytes() == y.tobytes() for x, y in zip(h[:3], h_alone[:3])), second
            else:
                assert _same_bytes(b.read(), y_ex if second == "exact on B" else y_mm), second


# ---- hc_ingest_overlaps_device --------------------------------------------------------------------------------------
def _ingest_dev(m, text, ip, offset, cand_cap=None, filtered_cap=None):
    """hc_ingest_overlaps_device on a caller's stream, the text `offset` bytes past a 16-byte boundary.
    Returns (rc, stats, candidates, their lines, filtered records, their lines); the outputs are those the call wrote."""
    n = len(text)
    buf = torch.full((offset + n + PAD,), 0x0a, dtype=torch.uint8, device="cuda")      # newlines around it: a read past
    assert buf.data_ptr() % 16 == 0                                                      # the text would show up as lines
    if n:
        buf[offset:offset + n].copy_(torch.from_numpy(np.frombuffer(text, dtype=np.uint8).copy()))
    guess = text.count(b"\n") + 1
    ccap = guess if cand_cap is None else cand_cap
    fcap = guess if filtered_cap is None else filtered_cap
    d_cand, d_cl, d_filt, d_fl = _dev(32 * ccap), _dev(8 * ccap), _dev(48 * fcap), _dev(8 * fcap)
    st = np.zeros(1, dtype=F.INGEST_STATS)
    s = torch.cuda.Stream()
    _ready()
    rc = capi.lib().hc_ingest_overlaps_device(m.handle, s.cuda_stream, buf.data_ptr() + offset, n, ip.ctypes.data, d_cand.data_ptr(),
                                              d_cl.data_ptr(), ccap, d_filt.data_ptr(), d_fl.data_ptr(), fcap, st.ctypes.data)
    torch.cuda.synchronize()
    ns, nf = (int(st[0]["n_scored"]), int(st[0]["n_filtered"])) if rc == 0 else (0, 0)
    out = (np.frombuffer(_written(d_cand, 32 * ns), dtype=F.CANDIDATE), np.frombuffer(_written(d_cl, 8 * ns), dtype=np.uint64),
           np.frombuffer(_written(d_filt, 48 * nf), dtype=F.OVERLAP_REC), np.frombuffer(_written(d_fl, 8 * nf), dtype=np.uint64))
    return (rc, st[0]) + out


def _id_to_index(ids):
    d = {}
    for i, v in enumerate(ids):
        d.setdefault(int(v), i)              # std::map::insert keeps the first (src/FastqStorage.h:90-93)
    return d


def _assert_ingest_matches_oracle(text, ids, kw, st, cand, cl, filt, fl):
    status, scored, filtered = IO.ingest(text, _id_to_index(ids), **kw)
    assert F.candidate_lines(cand, ids) == [IO.rec_line(r[1]) for r in scored]
    assert cand["idx1"].tolist() == [r[2] for r in scored] and cand["idx2"].tolist() == [r[3] for r in scored]
    assert cl.tolist() == [r[0] for r in scored]
    assert F.overlap_rec_lines(filt) == [IO.rec_line(r[1]) for r in filtered]
    assert fl.tolist() == [r[0] for r in filtered]
    assert [int(st["n_lines"]), int(st["n_skipped"]), int(st["n_dropped"])] == [len(status), status.count(IO.SKIPPED),
                                                                                 status.count(IO.DROPPED)]
    errs = [i for i, s in enumerate(status) if s in (IO.ERROR, IO.UNKNOWN_ID)]
    if errs:
        assert int(st["first_error_line"]) == errs[0] and int(st["first_error_status"]) == status[errs[0]]
        off, ln = int(st["first_error_offset"]), int(st["first_error_length"])
        assert text[off:off + ln] == IO.split_lines(text)[errs[0]]
    else:
        assert int(st["first_error_line"]) == NO_ERROR


def _ingest_cases():
    """(name, text, ids, ingest keywords): the ingest goldens, fuzzed texts and texts cut at awkward lengths."""
    out = []
    for name in ingest_golden_names():
        g = IngestGolden(name)
        out.append((name, g.text, g.ids, g.kw()))
    g = load_golden("synth_all_types")
    ids = g.rs.ids
    t11 = W.fuzz_overlap_text(g.cands[:2000], ids, seed=11)
    kw = dict(min_overlap_len=80, min_overlap_perc=20)
    out.append(("tabs", t11, ids, kw))
    out.append(("spaces", W.fuzz_overlap_text(g.cands[:2000], ids, seed=12, allow_spaces=True), ids, dict(kw, allow_spaces=True)))
    v = load_golden("synth_mismatch_void")
    sparse = v.rs.ids * np.uint64(2 ** 40 + 12345) + np.uint64(7)                       # the hash table, not the direct one
    out.append(("sparse ids", W.fuzz_overlap_text(v.cands, sparse, seed=13), sparse, dict(kw, relax_PE_edges=True)))
    out.append(("max_overlaps", t11, ids, dict(min_overlap_len=80, max_overlaps=1000)))
    out.append(("unknown ids", t11, ids[: len(ids) // 2], dict(min_overlap_len=80)))
    lines = t11.split(b"\n")
    lines[len(lines) // 2] = b"1\t2\t-1\t-\t-\t+\t+\t50\t-\t100\t-\ts\ts"             # a line the reference exits on
    out.append(("error line", b"\n".join(lines), ids, kw))
    head = t11[: t11.rfind(b"\n", 0, 4000) + 1]
    for total, nl in ((4096, True), (4096, False), (4095, False), (4097, True)):
        body = head + b"#" * (total - len(head) - (1 if nl else 0)) + (b"\n" if nl else b"")
        assert len(body) == total
        out.append(("%d bytes%s" % (total, "" if nl else ", no newline"), body, ids, kw))
    cut = t11[:9001].rstrip(b"\n")                                                     # ends inside a line, 9001 % 16 != 0
    out.append(("unterminated", cut, ids, kw))
    out.append(("one line", t11[: t11.find(b"\n")], ids, kw))
    out.append(("empty", b"", ids, kw))
    return out


def test_ingest_device(built_lib):
    """Every text on a caller's stream at byte offsets 0..15 from a 16-byte boundary (the newline index reads unaligned
    text byte by byte): the oracle's records, lines, counts and first error, and the host call's bytes."""
    for name, text, ids, kw in _ingest_cases():
        ip = F.make_ingest_params(**kw)
        m = capi.IdMap(ids)
        hc, hcl, hf, hfl, hst = m.ingest(text, ip)
        _assert_ingest_matches_oracle(text, ids, kw, hst, hc, hcl, hf, hfl)
        for off in range(16):
            rc, st, cand, cl, filt, fl = _ingest_dev(m, text, ip, off)
            assert rc == 0, (name, off, capi.last_error())
            assert [int(st[f]) for f in INGEST_FIELDS] == [int(hst[f]) for f in INGEST_FIELDS], (name, off)
            assert cand.tobytes() == hc.tobytes() and cl.tobytes() == hcl.tobytes(), (name, off)
            assert filt.tobytes() == hf.tobytes() and fl.tobytes() == hfl.tobytes(), (name, off)
        m.close()


def test_ingest_device_capacity_and_null_arguments(built_lib):
    g = load_golden("synth_all_types")
    ids = g.rs.ids
    text = W.fuzz_overlap_text(g.cands[:1500], ids, seed=21)
    ip = F.make_ingest_params(80, 20)
    m = capi.IdMap(ids)
    rc, st, *_ = _ingest_dev(m, text, ip, 3)
    need = (int(st["n_scored"]), int(st["n_filtered"]))
    assert rc == 0 and min(need) > 1
    for caps in ((need[0] - 1, need[1]), (need[0], need[1] - 1), (0, 0)):
        rc, st, cand, cl, filt, fl = _ingest_dev(m, text, ip, 5, *caps)                # asserts every output byte unchanged
        assert rc == -5 and (int(st["n_scored"]), int(st["n_filtered"])) == need, caps
    L = capi.lib()
    buf = torch.zeros(64, dtype=torch.uint8, device="cuda")
    st = np.zeros(1, dtype=F.INGEST_STATS)
    ok = [m.handle, None, buf.data_ptr(), 16, ip.ctypes.data, None, None, 0, None, None, 0, st.ctypes.data]
    for k in (0, 2, 4, 11):
        a = list(ok)
        a[k] = None
        assert L.hc_ingest_overlaps_device(*a) == -1, k
        assert "NULL argument" in capi.last_error()
    m.close()


@pytest.mark.parametrize("name", golden_names())
def test_ingest_then_score_in_hbm(built_lib, name):
    """hc_ingest_overlaps_device, then hc_score_batch_device on its d_cand: the oracle chain (ingest restatement, then the
    scoring oracle) and the host chain (hc_ingest_overlaps, then hc_score_batch)."""
    g = load_golden(name)
    ids = g.rs.ids
    text = W.fuzz_overlap_text(g.cands[:6000], ids, seed=61)
    kw = dict(min_overlap_len=int(g.ps.get("min_overlap_len", 150)), min_overlap_perc=int(g.ps.get("min_overlap_perc", 0)),
              relax_PE_edges=bool(g.ps.get("relax_PE_edges", 0)))
    ip = F.make_ingest_params(**kw)
    p = g.params()
    m = capi.IdMap(ids)
    with capi.Store(g.rs) as st:
        n_text = len(text)
        d_text = torch.from_numpy(np.frombuffer(text, dtype=np.uint8).copy()).cuda()
        cap = text.count(b"\n") + 1
        d_cand, d_filt = _dev(32 * cap), _dev(48 * cap)
        ist = np.zeros(1, dtype=F.INGEST_STATS)
        s = torch.cuda.Stream()
        _ready()
        rc = capi.lib().hc_ingest_overlaps_device(m.handle, s.cuda_stream, d_text.data_ptr(), n_text, ip.ctypes.data, d_cand.data_ptr(),
                                                  None, cap, d_filt.data_ptr(), None, cap, ist.ctypes.data)
        assert rc == 0, capi.last_error()
        n = int(ist[0]["n_scored"])
        assert n > 0
        out = DevOut(n)
        out.call(st, p, d_cand.data_ptr(), stream=s)            # same stream: ordered after the ingest, no host round trip
        got = out.read()
        hc, _, _, _, _ = m.ingest(text, ip)
        host = st.score_batch(p, hc)
    assert d_cand.cpu().numpy()[: 32 * n].tobytes() == hc.tobytes()
    _assert_same_as_host(got, host)
    status, scored, _ = IO.ingest(text, _id_to_index(ids), **kw)
    c = np.zeros(len(scored), dtype=F.CANDIDATE)
    for k, (_, r, i1, i2) in enumerate(scored):
        c[k] = (i1, i2, r[2], r[3], r[9], r[10], r[7], r[8], r[4], int(r[5] == ord("+")), int(r[6] == ord("+")), r[11], r[12], 0)
    assert F.candidate_lines(c, ids) == F.candidate_lines(hc, ids)
    ref, _ = O.score_batch(g.rs, p, c)
    _assert_matches_oracle(got[3], ref, what=name)
    m.close()
