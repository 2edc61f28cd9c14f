"""GPU suite: hc_ingest_score_overlaps (overlaps-file text in; kept candidates, edge records and pre-filtered overlaps out)
against the reference's own outputs on the scoring goldens, against the two-call path (hc_ingest_overlaps followed by
hc_score_batch*) on fuzzed text, across piece boundaries, at the edges of its input and on its errors; and the host
mirror's --gpu_parse path that calls it on reads of 16384+ bases."""
import ctypes
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

from haploconduct_b200 import build as B, capi, formats as F, workloads as W
from test_gpu_score_paths import case_overflow
from util import assert_results_match, golden_names, load_golden

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NO_ERROR = 2 ** 64 - 1
INGEST_FIELDS = ("n_lines", "n_scored", "n_filtered", "n_skipped", "n_dropped", "first_error_line", "first_error_offset",
                 "first_error_length", "first_error_status")
SCORE_FIELDS = ("n_candidates", "n_edges", "n_nonedges", "n_exact", "n_windows", "n_positions", "algorithmic_bytes")


def _text(cands, ids, tmp_path):
    path = str(tmp_path / "ov.txt")
    F.write_overlaps(path, cands, ids)
    with open(path, "rb") as f:
        return f.read()


def _ingest_params(g, **kw):
    return F.make_ingest_params(int(g.ps.get("min_overlap_len", 150)), int(g.ps.get("min_overlap_perc", 0)),
                                bool(g.ps.get("relax_PE_edges", 0)), **kw)


def _rate(mm, tl, two):
    r = np.where(tl == 0, 1.0, np.where(mm == 0, 0.0, mm.astype(np.float32).astype(np.float64) / np.maximum(tl, 1)))
    return np.where(two, np.maximum(r[:, 0], r[:, 1]), r[:, 0])


def _edge_fields(rs, kept, edges, p):
    """The Edge fields as the header comment derives them: from kept[cand] and the edge record (host libm exp())."""
    lens = rs.descs["seq_len"]
    c = kept[edges["cand"].astype(np.int64)]
    two = (edges["flags"] & F.EDGE_TWO) != 0
    res = np.zeros(len(edges), dtype=[("cls", "u1"), ("score", "<f8"), ("mismatch_rate", "<f8"), ("pos3", "<i4"), ("pos4", "<i4")])
    res["cls"] = F.CLASS_EDGE
    res["mismatch_rate"] = _rate(edges["mismatches"], edges["compared"], two)
    thr = float(p["edge_threshold"][0])
    p3, p4 = ctypes.c_int32(0), ctypes.c_int32(0)
    for k in range(len(edges)):
        l1, l2 = lens[int(c["idx1"][k])], lens[int(c["idx2"][k])]
        capi.lib().hc_edge_extra_pos(int(c["pos1"][k]), int(c["pos2"][k]), bytes([int(c["ord"][k])]), int(l1[0]), int(l1[1]), int(l2[0]),
                                     int(l2[1]), ctypes.byref(p3), ctypes.byref(p4))
        res["pos3"][k], res["pos4"][k] = p3.value, p4.value
        if "mean_log" in edges.dtype.names:
            cmp, ml = edges["compared"][k], edges["mean_log"][k]
            o1 = math.exp(ml[0]) if cmp[0] else 0.0
            if two[k]:
                o2 = math.exp(ml[1]) if cmp[1] else 0.0
                res["score"][k] = 0.5 * (o1 + o2) if (o1 > thr and o2 > thr) else min(o1, o2)
            else:
                res["score"][k] = o1
        else:
            res["score"][k] = edges["score"][k]
    return res


@pytest.mark.parametrize("name", golden_names())
@pytest.mark.parametrize("exact", [False, True])
def test_against_reference(built_lib, tmp_path, name, exact):
    g = load_golden(name)
    ids = g.rs.ids
    p = g.params(flags=F.FLAG_EXACT_EDGE_SCORES if exact else 0)
    with capi.Store(g.rs) as st:
        kept, kl, kc, edges, filt, fl, stats = st.ingest_score(capi.IdMap(ids), _text(g.cands, ids, tmp_path), _ingest_params(g), p)
    ref = g.ref_cands
    keep = ref["cls"] != F.CLASS_DISCARD
    scored_lines = np.nonzero(g.prefilter() == 1)[0]
    assert kc.tolist() == ref["cls"][keep].tolist()
    assert kl.tolist() == scored_lines[keep].tolist()
    assert F.candidate_lines(kept, ids) == F.candidate_lines(g.scored()[keep], ids)
    assert np.array_equal(edges["cand"], np.nonzero(kc == F.CLASS_EDGE)[0].astype(np.uint32))
    re = ref[ref["cls"] == F.CLASS_EDGE]
    res = _edge_fields(g.rs, kept, edges, p)
    assert_results_match(res, re["score"], re["mismatch_rate"], re["pos3"], re["pos4"], re["cls"], rel=0.0 if exact else 1e-6, what=name)
    assert F.candidate_lines(kept[kc == F.CLASS_NONEDGE], ids) + F.overlap_rec_lines(filt) == g.ref_nonedge
    assert int(stats["n_kept"]) == len(kept) == int(stats["score"]["n_edges"]) + int(stats["score"]["n_nonedges"])
    assert int(stats["ingest"]["first_error_line"]) == NO_ERROR


def _clamped(cand):
    """The 12-byte records hold positions below 2^14; the fuzzed files also name larger ones, which lie beyond every read of
    these stores, so that 2^14 - 1 gives the same window status (position out of range, score 0)."""
    c = cand.copy()
    c["pos1"], c["pos2"] = np.minimum(c["pos1"], (1 << 14) - 1), np.minimum(c["pos2"], (1 << 14) - 1)
    return c


def _two_call(st, m, text, ip, p):
    """hc_ingest_overlaps, then hc_score_batch_short_small / hc_score_batch on its candidates; the results in the form of
    hc_ingest_score_overlaps (edge records' cand remapped to the kept list)."""
    cand, cl, filt, fl, ist = m.ingest(text, ip)
    se, flags, bst = st.score_batch_small(p, _clamped(cand), runs=False)
    full_e, full_n, _, _ = st.score_batch(p, cand, per_candidate=False)
    assert len(full_e) == int(bst["n_edges"]) and len(full_n) == int(bst["n_nonedges"])
    cls = np.zeros(len(cand), dtype=np.uint8)
    cls[flags] = F.CLASS_NONEDGE
    cls[se["cand"].astype(np.int64)] = F.CLASS_EDGE
    keep = np.nonzero(cls)[0]
    e = se.copy()
    e["cand"] = np.searchsorted(keep, se["cand"].astype(np.int64))
    return cand[keep], cl[keep], cls[keep], e, filt, fl, ist, bst


def _assert_same_as_two_call(st, m, text, ip, p):
    kept, kl, kc, edges, filt, fl, s = st.ingest_score(m, text, ip, p)
    k2, kl2, kc2, e2, f2, fl2, ist, bst = _two_call(st, m, text, ip, p)
    assert kept.tobytes() == k2.tobytes() and kl.tolist() == kl2.tolist() and kc.tolist() == kc2.tolist()
    assert edges.tobytes() == e2.tobytes()
    assert filt.tobytes() == f2.tobytes() and fl.tolist() == fl2.tolist()
    assert [int(s["ingest"][f]) for f in INGEST_FIELDS] == [int(ist[f]) for f in INGEST_FIELDS]
    assert [int(s["score"][f]) for f in SCORE_FIELDS] == [int(bst[f]) for f in SCORE_FIELDS]
    assert int(s["n_kept"]) == len(kept)
    return kept, kl, kc, edges, filt, fl, s


def _all(r):
    """Every output of one call as bytes (stats without the times)."""
    kept, kl, kc, edges, filt, fl, s = r
    return (kept.tobytes(), kl.tobytes(), kc.tobytes(), edges.tobytes(), filt.tobytes(), fl.tobytes(),
            [int(s["ingest"][f]) for f in INGEST_FIELDS], [int(s["score"][f]) for f in SCORE_FIELDS], int(s["n_kept"]))


@pytest.mark.parametrize("seed,allow_spaces,exact", [(11, False, False), (12, True, True), (13, False, False), (13, False, True)])
def test_against_two_call_path(built_lib, seed, allow_spaces, exact):
    g = load_golden("synth_all_types" if seed != 13 else "synth_mismatch_void")
    ids = g.rs.ids * np.uint64(2 ** 40 + 12345) + np.uint64(7) if seed == 13 else g.rs.ids       # sparse ids: the hash table
    text = W.fuzz_overlap_text(g.cands, ids, seed=seed, allow_spaces=allow_spaces)
    p = g.params(flags=F.FLAG_EXACT_EDGE_SCORES if exact else 0)
    with capi.Store(g.rs) as st:
        m = capi.IdMap(ids)
        r = _assert_same_as_two_call(st, m, text, F.make_ingest_params(80, 20, seed == 13, allow_spaces), p)
        assert len(r[0]) > 100 and len(r[3]) > 10 and (r[2] == F.CLASS_NONEDGE).any()
        _assert_same_as_two_call(st, m, text, F.make_ingest_params(80, allow_spaces=allow_spaces, max_overlaps=1000), p)
        r = _assert_same_as_two_call(st, capi.IdMap(ids[: len(ids) // 2]), text, F.make_ingest_params(80, allow_spaces=allow_spaces), p)
        assert int(r[6]["ingest"]["first_error_line"]) != NO_ERROR       # unknown ids: reported, the other lines still scored
        assert len(r[0]) > 0


def test_piece_boundaries(built_lib, monkeypatch):
    """The text cut into pieces of 700, 5000 and 100000 bytes gives what one piece gives: max_overlaps ending inside a
    piece, unknown ids in the middle, an error line in the middle, a last line longer than a piece without a newline, and
    pieces that score nothing or only discard, between pieces that keep candidates."""
    g = load_golden("synth_all_types")
    ids = g.rs.ids
    p = g.params()
    ip = F.make_ingest_params(80, 20)
    with capi.Store(g.rs) as st:
        m = capi.IdMap(ids)
        base = W.fuzz_overlap_text(np.tile(g.cands, 2), ids, seed=31)
        _, cl, _, _, _ = m.ingest(base, ip)
        # blocks of lines: only pre-filtered / dropped lines, and only candidates the scorer discards
        cand_all, _, _, _, _ = m.ingest(W.fuzz_overlap_text(g.cands, ids, seed=32, junk=False), ip)
        se, flags, _ = st.score_batch_small(p, _clamped(cand_all), runs=False)
        disc = np.ones(len(cand_all), dtype=bool)
        disc[flags] = False
        disc[se["cand"].astype(np.int64)] = False
        pre = F.prefilter(g.cands, 80, 20)
        assert disc.any()
        discarded = np.resize(cand_all[disc], 400)                                            # 400 lines, repeated if need be
        discarded["perc1"], discarded["perc2"] = 100, 100
        filtered_only = F.candidates_to_lines(g.cands[pre != 1][:400], ids)
        disc_text = "".join(F.candidates_to_lines(discarded, ids)).encode()
        assert len(disc_text) > 2 * 5000 and len("".join(filtered_only)) > 2 * 5000
        keepers = base[: len(base) // 4]
        keepers = keepers[: keepers.rfind(b"\n") + 1]
        lines = base.split(b"\n")
        lines[len(lines) // 2] = b"1\t2\t-1\t-\t-\t+\t+\t50\t-\t100\t-\ts\ts"             # a line the reference exits on
        cases = [(base, ip, m), (base, F.make_ingest_params(80, max_overlaps=3333), m), (base, ip, capi.IdMap(ids[: len(ids) // 2])),
                 (b"\n".join(lines), ip, m), (base + b"x" * 3000, ip, m),
                 (keepers + "".join(filtered_only).encode() + b"\n\n" + disc_text + keepers, ip, m)]
        for text, ipp, mm in cases:
            monkeypatch.delenv("HC_INGEST_PIECE", raising=False)
            one = st.ingest_score(mm, text, ipp, p)
            assert int(one[6]["n_kept"]) > 0
            _assert_same_as_two_call(st, mm, text, ipp, p)
            for piece in ("700", "5000", "100000"):
                monkeypatch.setenv("HC_INGEST_PIECE", piece)
                assert _all(st.ingest_score(mm, text, ipp, p)) == _all(one), piece


def test_edges_of_the_input(built_lib, tmp_path):
    g = load_golden("synth_all_types")
    ids = g.rs.ids
    p = g.params()
    with capi.Store(g.rs) as st:
        m = capi.IdMap(ids)
        kept, kl, kc, edges, filt, fl, s = st.ingest_score(m, b"", F.make_ingest_params(60), p)
        assert len(kept) == len(edges) == len(filt) == 0 and int(s["ingest"]["n_lines"]) == 0
        assert int(s["ingest"]["first_error_line"]) == NO_ERROR
        # every line pre-filtered, self overlaps dropped, blank and 12-field lines skipped
        pre = F.prefilter(g.cands, 60)
        c = g.cands[pre != 1][:300].copy()
        text = _text(c, ids, tmp_path) + b"7\t7\t0\t-\t-\t+\t+\t90\t-\t300\t-\ts\ts\n\n1\t2\t3\n"
        kept, kl, kc, edges, filt, fl, s = _assert_same_as_two_call(st, m, text, F.make_ingest_params(60), p)
        assert len(kept) == len(edges) == 0 and len(filt) == int((F.prefilter(c, 60) == 0).sum()) > 0
        assert int(s["ingest"]["n_skipped"]) == 2 and int(s["ingest"]["n_dropped"]) >= 1
        # pinned text (hc_host_alloc) and pageable text give the same bytes
        text = W.fuzz_overlap_text(g.cands, ids, seed=41)
        pinned = capi.host_alloc(len(text))
        pinned[:] = np.frombuffer(text, dtype=np.uint8)
        a = _all(st.ingest_score(m, text, F.make_ingest_params(60), p))
        b = _all(st.ingest_score(m, pinned, F.make_ingest_params(60), p))
        assert a == b
        capi.lib().hc_host_free(pinned.ctypes.data)


@pytest.mark.parametrize("exact", [False, True])
def test_long_reads_and_16bit_overflow(built_lib, tmp_path, exact):
    """Reads of 70000 bases (no 16384-base limit) and windows of 65535-65537 compared positions: HC_EDGE_OVERFLOW is set
    as hc_score_batch_short_small sets it."""
    case = case_overflow()
    p = case.params[0].copy()
    if exact:
        p["flags"] |= F.FLAG_EXACT_EDGE_SCORES
    assert int(case.rs.descs["seq_len"].max()) >= 16384
    with capi.Store(case.rs) as st:
        text = _text(case.cands, case.rs.ids, tmp_path)
        kept, kl, kc, edges, filt, fl, s = _assert_same_as_two_call(st, capi.IdMap(case.rs.ids), text, F.make_ingest_params(0), p)
    assert len(edges) == len(case.cands) and ((edges["flags"] & F.EDGE_OVERFLOW) != 0).sum() == 2


def test_capacities(built_lib):
    g = load_golden("synth_mismatch_void")
    text = W.fuzz_overlap_text(g.cands, g.rs.ids, seed=51)
    ip, p = F.make_ingest_params(120, relax_PE_edges=True), g.params()
    with capi.Store(g.rs) as st:
        m = capi.IdMap(g.rs.ids)
        full = st.ingest_score(m, text, ip, p)
        need = (len(full[0]), len(full[3]), len(full[4]))
        assert min(need) > 1
        for k in range(3):
            caps = [None, None, None]
            caps[k] = need[k] - 1
            with pytest.raises(capi.HcError) as e:
                st.ingest_score(m, text, ip, p, kept_cap=caps[0], edges_cap=caps[1], filtered_cap=caps[2])
            assert e.value.code == -5 and e.value.required == need
            r = st.ingest_score(m, text, ip, p, kept_cap=need[0], edges_cap=need[1], filtered_cap=need[2])
            assert _all(r) == _all(full)


def test_rejected_candidates_and_null_arguments(built_lib):
    g = load_golden("synth_all_types")
    ids = g.rs.ids
    pairs = np.nonzero(g.rs.descs["seq_len"][:, 1] > 0)[0]
    a, b = int(ids[pairs[0]]), int(ids[pairs[1]])
    # typed s/s with ORD '-' in the file, but both reads are paired in the store: a P-P candidate with ORD '-'
    line = ("%d\t%d\t5\t-\t-\t+\t+\t90\t-\t200\t-\ts\ts\n" % (a, b)).encode()
    p = g.params()
    with capi.Store(g.rs) as st:
        m = capi.IdMap(ids)
        cand, _, _, _, _ = m.ingest(line, F.make_ingest_params(60))
        assert len(cand) == 1
        with pytest.raises(capi.HcError) as e1:
            st.score_batch(p, cand)
        with pytest.raises(capi.HcError) as e2:
            st.ingest_score(m, line, F.make_ingest_params(60), p)
        assert e2.value.code == e1.value.code == -1 and str(e2.value) == str(e1.value)
        # an id map that knows more reads than the store: an index outside the store
        big = capi.IdMap(np.concatenate([ids, np.array([10 ** 12], dtype=np.uint64)]))
        bad = ("%d\t%d\t5\t-\t-\t+\t+\t90\t-\t200\t-\ts\ts\n" % (int(ids[0]), 10 ** 12)).encode()
        with pytest.raises(capi.HcError) as e3:
            st.ingest_score(big, bad, F.make_ingest_params(60), p)
        assert e3.value.code == -1 and str(e3.value) == str(e1.value)
        L = capi.lib()
        ip = F.make_ingest_params(60)
        st_buf = np.zeros(1, dtype=F.INGEST_SCORE_STATS)
        buf = np.frombuffer(line, dtype=np.uint8)
        kept = np.zeros(4, dtype=F.CANDIDATE)
        kc = np.zeros(4, dtype=np.uint8)
        edges = np.zeros(4, dtype=F.EDGE_SMALL)
        filt = np.zeros(4, dtype=F.OVERLAP_REC)
        args = [st.handle, m.handle, buf.ctypes.data, len(buf), ip.ctypes.data, p.ctypes.data, kept.ctypes.data, None, kc.ctypes.data, 4,
                edges.ctypes.data, 4, filt.ctypes.data, None, 4, st_buf.ctypes.data]
        for k in (0, 1, 2, 4, 5, 6, 8, 10, 12, 15):
            a2 = list(args)
            a2[k] = None
            assert L.hc_ingest_score_overlaps(*a2) == -1, k
            assert "NULL argument" in capi.last_error()


@pytest.mark.skipif(capi.device_count() < 2 if os.path.exists(capi.LIB_PATH) else True, reason="needs two GPUs")
def test_id_map_without_store_replica(built_lib):
    g = load_golden("synth_all_types")
    with capi.Store(g.rs, first_device=0, n_devices=1) as st:
        with pytest.raises(capi.HcError) as e:
            st.ingest_score(capi.IdMap(g.rs.ids, device=1), W.fuzz_overlap_text(g.cands, g.rs.ids, seed=3), F.make_ingest_params(60), g.params())
    assert e.value.code == -1 and "no replica" in str(e.value)


def test_stats_struct_size_matches_header(tmp_path):
    gcc = shutil.which("gcc")
    if not gcc:
        pytest.skip("no gcc on this box")
    src = tmp_path / "size.c"
    src.write_text('#include <stdio.h>\n#include "hc_b200.h"\nint main(void) { printf("%d\\n", (int)sizeof(hc_ingest_score_stats)); return 0; }\n')
    exe = str(tmp_path / "size")
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe], check=True)
    assert int(subprocess.run([exe], check=True, stdout=subprocess.PIPE, text=True).stdout) == F.INGEST_SCORE_STATS.itemsize == 152


def _mirror(d, rs, cands, gpu_parse):
    """hc_edgecalc on the reads and overlaps of a case: (adjacency dump, nonedge_overlaps.txt, stderr)."""
    out = os.path.join(d, "parse" if gpu_parse else "host")
    os.makedirs(out, exist_ok=True)
    F.write_fastq_set(rs, d + "/s.fastq", d + "/p1.fastq", d + "/p2.fastq")
    F.write_overlaps(d + "/ov.txt", cands, rs.ids)
    cmd = [os.path.join(B.LIBDIR, "hc_edgecalc"), "--overlaps", d + "/ov.txt", "--dump-graph", out + "/graph.tsv", "--edge_threshold", "0.99",
           "--min_overlap_len", "0", "--gpu_parse=" + ("true" if gpu_parse else "false")]
    if rs.n_single:
        cmd += ["--singles", d + "/s.fastq"]
    if rs.n_reads > rs.n_single:
        cmd += ["--paired1", d + "/p1.fastq", "--paired2", d + "/p2.fastq"]
    r = subprocess.run(cmd, cwd=out, check=True, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=dict(os.environ, HC_MIRROR_TIMING="1"))
    with open(out + "/graph.tsv", "rb") as f:
        graph = f.read()
    with open(out + "/nonedge_overlaps.txt", "rb") as f:
        nonedge = f.read()
    return graph, nonedge, r.stderr


def test_mirror_long_contigs(built_lib, tmp_path):
    """hc_edgecalc --gpu_parse=true on contigs of 70000 bases: the one-call path when no window reaches 65536 positions,
    the batch path when one does; both byte-identical to --gpu_parse=false."""
    case = case_overflow()
    with capi.Store(case.rs) as st:
        _, _, per, _ = st.score_batch(case.params[0], case.cands)
    short = np.nonzero(per["compared"].max(axis=1) <= 0xffff)[0]
    assert 0 < len(short) < len(case.cands)
    for cands, one_call in ((case.cands[short], True), (case.cands, False)):
        d = str(tmp_path / ("short" if one_call else "all"))
        os.makedirs(d)
        g1, n1, err = _mirror(d, case.rs, cands, True)
        g0, n0, _ = _mirror(d, case.rs, cands, False)
        assert g1 == g0 and n1 == n0 and len(g1) > 0
        assert ("hc_ingest_score_overlaps" in err) == one_call, err
