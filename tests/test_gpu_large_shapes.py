"""GPU suite: the library's calls at the sizes where their scans carry between the passes of a single-block loop -- more
than 1024 compaction blocks of 4096 candidates in one scoring launch (hc_compact_scan), more than 4,194,304 inputs to
hc_scan::exclusive_u32 (FNO1 / FNO3 counts, overlaps.txt line offsets, adjacency offsets) and more than 4 MB of FASTQ text
in one file (scan_counts of the newline index).  The benchmark and multi-million-edge runs use these sizes; every check
is against a reference that does not run the loop under test: the per-candidate classes of the host pipeline in 1 M
steps, the C and numpy oracles, Python-formatted files, an array-built store.  test_cases_cross_their_boundaries (no
GPU) checks that the planned sizes still cross; each GPU test asserts the size it reached."""
import numpy as np
import pytest

from haploconduct_b200 import capi, formats as F
from oracle import oracle as O
from util import assert_results_match, random_fno_input

SCAN_CARRY = 1024 * 4096                 # hc_scan / hc_compact_scan: 1024 threads x 4096-entry blocks
COMPACT_BLOCK = 4096                     # candidates per compaction block of the scoring launch
TEXT_CARRY = 1024 * 4096                 # scan_counts: 1024 threads x 4096-byte text tiles
SCORE_SIZES = [SCAN_CARRY, SCAN_CARRY + 1, 3 * SCAN_CARRY + 1234]
HOST_STEP = 6_000_000                    # HC_HOST_CHUNK of the large-step pipeline runs
REF_STEP = 1_000_000                     # HC_HOST_CHUNK of the reference run, and the device chunk size
ADJ_VERTICES = [SCAN_CARRY - 1, SCAN_CARRY]
FNO1_EDGES = 8_000_000
FNO3_ORIGINALS = SCAN_CARRY + 4321
FASTQ_PAIRS = 15_000
BENCH_PARAMS = dict(edge_threshold=0.97, ov_threshold=0.9, merge_contigs=0.0, mismatch=0.0, min_read_len=0)
SENT, PAD = 0xAB, 64


def compaction_blocks(n):
    return (n + COMPACT_BLOCK - 1) // COMPACT_BLOCK


def test_cases_cross_their_boundaries():
    blocks = [compaction_blocks(n) for n in SCORE_SIZES]
    assert blocks == [1024, 1025, 3073]                          # one full pass of hc_compact_scan, then two and four
    assert 1024 < compaction_blocks(HOST_STEP) < 2048 and compaction_blocks(REF_STEP) < 1024
    assert [v + 1 - SCAN_CARRY for v in ADJ_VERTICES] == [0, 1]  # V + 1 offsets: on the boundary and one past it
    assert FNO1_EDGES > SCAN_CARRY and FNO3_ORIGINALS > SCAN_CARRY
    assert FASTQ_PAIRS * (2 * 150 + 12) > TEXT_CARRY             # each mate file: > 1024 newline tiles


# ---- scoring compaction ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def big_batch():
    """The benchmark's shape (2x150 pairs, P-P candidates with D = 140 partners) generated in HBM, 12.6 M candidates, and
    the per-candidate results of the host pipeline in 1 M steps (245 compaction blocks a launch: no carry)."""
    import torch
    from haploconduct_b200 import workloads_torch as WT

    pr = WT.make_paired_reads(150_000, read_len=150, genome_len=37_500, seed=20261022, device="cuda")
    rec = WT.make_pp_candidates(pr, D=140, max_cands=max(SCORE_SIZES))
    torch.cuda.synchronize()
    assert rec.shape[0] == max(SCORE_SIZES)
    rs = pr.readset()
    cands = WT.candidates_as_numpy(rec)
    p = F.make_params(**BENCH_PARAMS)
    mp = pytest.MonkeyPatch()
    mp.setenv("HC_HOST_CHUNK", str(REF_STEP))
    try:
        with capi.Store(rs) as st:
            ref = st.score_batch(p, cands, per_candidate=True)
    finally:
        mp.undo()
    return rs, rec, cands, p, ref


def _dev(nbytes):
    import torch

    return torch.full((nbytes + PAD,), SENT, dtype=torch.uint8, device="cuda")


def _written(buf, nbytes):
    h = buf.cpu().numpy()
    assert (h[nbytes:] == SENT).all(), "bytes written past the first %d" % nbytes
    return h[:nbytes]


def _score_device(st, p, ptr, n):
    """One hc_score_batch_device call with n-record, sentinel-filled outputs: (counts, edges, non-edge indices)."""
    import torch

    edges, nonedge, counts = _dev(48 * n), _dev(8 * n), _dev(32)
    torch.cuda.synchronize()
    st.score_batch_device(0, 0, p, ptr, n, 0, edges.data_ptr(), n, nonedge.data_ptr(), n, counts.data_ptr(), False)
    torch.cuda.synchronize()
    c = _written(counts, 32).view(np.uint64)
    ne, nn = int(c[0]), int(c[1])
    assert ne <= n and nn <= n
    return c, _written(edges, 48 * ne).view(F.EDGE), _written(nonedge, 8 * nn).view(np.uint64)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["packed", "planar"])
@pytest.mark.parametrize("n", SCORE_SIZES)
def test_device_call_compaction(built_lib, big_batch, monkeypatch, layout, n):
    """hc_score_batch_device on n candidates in one launch (the benchmark's call): the edge and non-edge lists are exactly
    the candidates the reference classed so, in input order, with the records of chunked calls of <= 1 M candidates."""
    monkeypatch.setenv("HC_STORE_LAYOUT", layout if layout == "planar" else "auto")
    rs, rec, cands, p, ref = big_batch
    assert compaction_blocks(n) > 1023
    re, rn, rper, _ = ref
    cls = rper["cls"][:n]
    want_e, want_n = np.flatnonzero(cls == F.CLASS_EDGE), np.flatnonzero(cls == F.CLASS_NONEDGE)
    assert len(want_e) > 1000 and len(want_n) > 1000
    with capi.Store(rs) as st:
        counts, edges, nonedge = _score_device(st, p, rec.data_ptr(), n)
        assert [int(counts[0]), int(counts[1]), int(counts[3])] == [len(want_e), len(want_n), 0]
        assert np.array_equal(edges["cand"], want_e.astype(np.uint64))
        assert np.array_equal(nonedge, want_n.astype(np.uint64))
        parts_e, parts_n = [], []
        for lo in range(0, n, REF_STEP):
            m = min(REF_STEP, n - lo)
            _, e, ne = _score_device(st, p, rec.data_ptr() + 32 * lo, m)
            e = e.copy()
            e["cand"] += np.uint64(lo)
            parts_e.append(e)
            parts_n.append(ne + np.uint64(lo))
    assert np.concatenate(parts_e).tobytes() == edges.tobytes()
    assert np.array_equal(np.concatenate(parts_n), nonedge)
    assert edges.tobytes() == re[re["cand"] < n].tobytes()


@pytest.mark.gpu
def test_reference_sample_against_oracle(built_lib, big_batch):
    """The per-candidate reference itself, on a random sample, against the scoring oracle."""
    rs, rec, cands, p, ref = big_batch
    rper = ref[2]
    pick = np.sort(np.random.RandomState(3).choice(len(cands), size=40_000, replace=False))
    oref, _ = O.score_batch(rs, p, cands[pick])
    assert_results_match(rper[pick], oref["score"], oref["mismatch_rate"], oref["pos3"], oref["pos4"], oref["cls"], what="sample")


# (HC_HOST_CHUNK, HC_HOST_WHOLE_MAX, candidates in the largest step): steps of 6 M; the default schedule, whose largest
# step for 12.6 M candidates is 4.7 M; two copy slots with uniform 8 M steps
HOST_SCHEDULES = {"6M_steps": ("6000000", None, HOST_STEP), "tapered": (None, None, 4_719_232), "8M_slots": (None, "0", 8 << 20)}


@pytest.mark.gpu
@pytest.mark.parametrize("schedule", sorted(HOST_SCHEDULES))
def test_host_pipeline_compaction(built_lib, big_batch, monkeypatch, schedule):
    """hc_score_batch and the benchmark's end-to-end form hc_score_batch_runs6_small on host buffers, with pipeline steps
    of more than 1024 compaction blocks: the lists of the 1 M-step run and the per-candidate classes."""
    chunk, whole_max, largest = HOST_SCHEDULES[schedule]
    for var, v in (("HC_HOST_CHUNK", chunk), ("HC_HOST_WHOLE_MAX", whole_max)):
        if v is None:
            monkeypatch.delenv(var, raising=False)
        else:
            monkeypatch.setenv(var, v)
    rs, rec, cands, p, ref = big_batch
    assert compaction_blocks(largest) > 1024
    re, rn, rper, rstats = ref
    assert np.array_equal(re["cand"], np.flatnonzero(rper["cls"] == F.CLASS_EDGE).astype(np.uint64))
    assert np.array_equal(rn, np.flatnonzero(rper["cls"] == F.CLASS_NONEDGE).astype(np.uint64))
    with capi.Store(rs) as st:
        e, ne, _, stats = st.score_batch(p, cands, per_candidate=False)
        assert e.tobytes() == re.tobytes() and np.array_equal(ne, rn)
        assert (int(stats["n_edges"]), int(stats["n_nonedges"])) == (len(re), len(rn))
        se, flags, sstats = st.score_batch_small(p, cands, runs=6)
    assert np.array_equal(se["cand"].astype(np.uint64), re["cand"])
    assert np.array_equal(se["score"], re["score"])
    assert np.array_equal(np.flatnonzero(flags).astype(np.uint64), rn)
    assert (int(sstats["n_edges"]), int(sstats["n_nonedges"])) == (len(re), len(rn))


# ---- FindNextOverlaps -----------------------------------------------------------------------------------------------
def random_fno3_input(seed, n_originals, n_reads=50_000):
    """util.random_fno3_input without the per-original loop: 1-3 distinct new reads per original (k-th at s + k * t mod
    n_reads, t < n_reads / 3), most originals in one read only, so that the output stays below a million lines."""
    rng = np.random.default_rng(seed)
    reads = np.zeros(n_reads, dtype=F.FNO_READ)
    reads["id"] = rng.permutation(n_reads)
    reads["len1"] = rng.integers(80, 600, n_reads)
    reads["len2"] = np.where(rng.random(n_reads) < 0.4, rng.integers(80, 600, n_reads), 0)
    c = rng.choice([1, 2, 3], size=n_originals, p=[0.8, 0.15, 0.05])
    off = np.zeros(n_originals + 1, dtype=np.uint64)
    off[1:] = np.cumsum(c)
    m = int(off[-1])
    k = np.arange(m) - np.repeat(off[:-1].astype(np.int64), c)
    s = np.repeat(rng.integers(0, n_reads, n_originals), c)
    t = np.repeat(rng.integers(1, n_reads // 3, n_originals), c)
    pos = np.zeros(m, dtype=F.FNO3_POS)
    pos["index1"], pos["index2"] = rng.integers(-20, 500, m), rng.integers(-20, 500, m)
    return F.Fno3Input(off=off, sr_idx=((s + k * t) % n_reads).astype(np.uint32), sr_pos=pos, reads=reads, no_inclusions=seed % 2)


def fno_lines_bytes(ov):
    """formats.fno_lines of many records, each line as bytes (column lists instead of per-record field access)."""
    cols = [ov[f].tolist() for f in ("id1", "id2", "pos1", "pos2", "ord", "ori1", "ori2", "perc", "perc2", "len1", "len2", "type1", "type2")]
    return [b"%d\t%d\t%d\t%d\t%c\t%c\t%c\t%d\t%d\t%d\t%d\t%c\t%c" % r for r in zip(*cols)]


@pytest.fixture(scope="module")
def fno1_big():
    # util.random_fno_input loops over vertices only; the edges are drawn as arrays
    fi = random_fno_input(31, n_vertices=20_000, n_sr=3_000, n_edges=FNO1_EDGES)
    return fi, O.fno1(fi)


@pytest.mark.gpu
@pytest.mark.parametrize("small", [False, True])
def test_fno1_records(built_lib, fno1_big, small):
    fi, ref = fno1_big
    assert len(fi.edges) > SCAN_CARRY and len(ref) > SCAN_CARRY
    assert capi.fno1(fi, small=small).tobytes() == ref.tobytes()


@pytest.mark.gpu
def test_fno1_text(built_lib, fno1_big):
    """overlaps.txt: the lines unique and in byte order (np.unique of an S array), more than 4,194,304 of them."""
    fi, ref = fno1_big
    lines = np.unique(np.array(fno_lines_bytes(ref), dtype="S"))
    assert len(lines) > SCAN_CARRY
    got = capi.fno1_text(fi)
    assert got == b"\n".join(lines.tolist()) + b"\n"


@pytest.mark.gpu
def test_fno3_records_and_text(built_lib):
    fi = random_fno3_input(32, FNO3_ORIGINALS)
    assert len(fi.off) - 1 > SCAN_CARRY
    ref = O.fno3(fi)
    assert len(ref) > 100_000
    for small in (False, True):
        assert capi.fno3(fi, small=small).tobytes() == ref.tobytes(), small
    assert capi.fno3_text(fi) == b"".join(l + b"\n" for l in fno_lines_bytes(ref))


# ---- adjacency ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("V", ADJ_VERTICES)
def test_adjacency_offsets_past_the_scan(built_lib, V):
    """hc_build_adjacency with V + 1 = 4,194,304 and 4,194,305 offsets, 8 M edges with hubs and many equal keys, against
    oracle.sort_edges (numpy)."""
    rng = np.random.default_rng(V)
    n = 8_000_000
    g = np.zeros(n, dtype=O.REF_EDGE)
    hub = rng.random(n) < 0.05
    g["v1"] = np.where(hub, rng.integers(0, 16, n), rng.integers(0, V, n))
    g["v1"][-3:] = V - 1                                                   # the last vertex's offsets too
    g["v2"] = np.where(rng.random(n) < 0.05, rng.integers(0, 16, n), rng.integers(0, V, n))
    g["len1"] = rng.integers(10, 13, n)
    read_len = rng.integers(100, 103, V).astype(np.int64)
    order = np.argsort(g["v1"], kind="stable")
    ref_sorted, (rv, ro, rsrc), ties_long = O.sort_edges(g[order], read_len)
    e = np.zeros(n, dtype=capi.ADJ_EDGE)
    e["vertex1"], e["vertex2"] = g["v1"], g["v2"]
    e["nonoverlap_len"] = (read_len[g["v1"].astype(np.int64)] + read_len[g["v2"].astype(np.int64)] - 2 * g["len1"].astype(np.int64)) & 0xffffffff
    out_off, perm, in_off, in_src, ties = capi.build_adjacency(e, V, sort=True)
    assert len(out_off) == V + 1 and len(out_off) >= SCAN_CARRY
    want_off = np.concatenate([[0], np.cumsum(np.bincount(g["v1"].astype(np.int64), minlength=V))]).astype(np.uint64)
    assert np.array_equal(out_off, want_off)
    assert g[perm].tobytes() == ref_sorted.tobytes()
    assert int(ties.sum()) == ties_long and ties_long > 0
    want_in = np.concatenate([[0], np.cumsum(np.bincount(g["v2"].astype(np.int64), minlength=V))]).astype(np.uint64)
    assert np.array_equal(in_off, want_in)
    deg = np.diff(in_off.astype(np.int64))
    vs = np.nonzero(deg)[0]
    assert np.array_equal(vs, rv) and np.array_equal(np.append(in_off.astype(np.int64)[vs], n), ro)
    assert np.array_equal(in_src.astype(np.int64), rsrc)


# ---- FASTQ text > 4 MB per file -------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_fastq_files_past_the_tile_scan(built_lib, tmp_path):
    """2x150 pairs as FASTQ text of more than 4 MB per mate file, through hc_store_create_fastq and the streamed
    hc_store_create_fastq_files (default ring): the ids of the array-built store, and byte-identical scoring."""
    import torch
    from haploconduct_b200 import workloads_torch as WT

    pr = WT.make_paired_reads(FASTQ_PAIRS, read_len=150, genome_len=3_000, seed=20261023, device="cuda")
    rs = pr.readset()
    rec = WT.make_pp_candidates(pr, D=40, max_cands=300_000)
    torch.cuda.synchronize()
    cands = WT.candidates_as_numpy(rec)
    assert rs.n_single == 0 and len(cands) > 100_000
    texts = []
    for mate in (0, 1):
        texts.append("".join("@%d\n%s\n+\n%s\n" % (int(rs.ids[i]), rs.seq(i, mate), rs.qual(i, mate)) for i in range(rs.n_reads)).encode())
    assert min(len(t) for t in texts) > TEXT_CARRY
    paths = []
    for k, t in enumerate(texts):
        f = tmp_path / ("p%d.fastq" % (k + 1))
        f.write_bytes(t)
        paths.append(str(f))
    p = F.make_params(**BENCH_PARAMS)
    with capi.Store(rs) as st:
        want = st.score_batch(p, cands)
    assert len(want[0]) > 0
    for make in (lambda: capi.Store.from_fastq(b"", texts[0], texts[1]), lambda: capi.Store.from_fastq_files(None, *paths)):
        with make() as st:
            ids, lens = st.read_ids()
            assert np.array_equal(ids, rs.ids) and np.array_equal(lens, rs.descs["seq_len"])
            got = st.score_batch(p, cands)
        assert got[0].tobytes() == want[0].tobytes() and np.array_equal(got[1], want[1]) and got[2].tobytes() == want[2].tobytes()
