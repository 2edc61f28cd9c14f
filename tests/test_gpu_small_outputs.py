"""GPU suite: the small-output entry points (hc_score_batch_runs_small / hc_score_batch_short_small) against the full
outputs of hc_score_batch on the same candidates -- same accepted edges in the same order, the same non-edge set,
scores / mean logs / counts bit for bit -- and, on lists sorted by read, the run-encoded records of hc_score_batch_runs
against the plain hc_candidate records (every output must be byte-identical)."""
import ctypes

import numpy as np
import pytest

from haploconduct_b200 import capi, formats as F, workloads as W
from util import golden_names, load_golden

pytestmark = pytest.mark.gpu


def _rate(mm, tl, two):
    r = np.where(tl == 0, 1.0, np.where(mm == 0, 0.0, mm.astype(np.float32).astype(np.float64) / np.maximum(tl, 1)))
    return np.where(two, np.maximum(r[:, 0], r[:, 1]), r[:, 0])


@pytest.mark.parametrize("name", golden_names())
@pytest.mark.parametrize("exact", [False, True])
@pytest.mark.parametrize("chunk", [0, 1000])
def test_small_outputs_equal_full_outputs(built_lib, monkeypatch, name, exact, chunk):
    if chunk:
        monkeypatch.setenv("HC_HOST_CHUNK", str(chunk))
    g = load_golden(name)
    cands = g.scored()
    fits = (cands["pos1"] < (1 << 14)) & (cands["pos2"] < (1 << 14))
    cands = cands[fits]
    p = g.params(flags=F.FLAG_EXACT_EDGE_SCORES if exact else 0)
    with capi.Store(g.rs) as st:
        edges, nonedge, per, _ = st.score_batch(p, cands)
        small6 = g.rs.n_reads < (1 << 25) and int(g.rs.descs["seq_len"].max()) < 512
        for runs in (True, False) + ((6,) if small6 else ()):
            se, flags, stats = st.score_batch_small(p, cands, runs=runs)
            assert np.array_equal(np.nonzero(flags)[0].astype(np.uint64), nonedge)
            assert np.array_equal(se["cand"].astype(np.uint64), edges["cand"])
            two = (se["flags"] & F.EDGE_TWO) != 0
            assert np.array_equal(_rate(se["mismatches"], se["compared"], two), edges["mismatch_rate"])
            assert np.array_equal(se["mismatches"], per["mismatches"][edges["cand"].astype(np.int64)])
            assert np.array_equal(se["compared"], per["compared"][edges["cand"].astype(np.int64)])
            if exact:
                a, b = se["mean_log"], edges["mean_log"]
                assert np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~np.isnan(a)], b[~np.isnan(b)])
                assert np.all(se["flags"] & F.EDGE_EXACT)
            else:
                assert np.array_equal(se["score"], edges["score"])
            assert int(stats["n_edges"]) == len(edges) and int(stats["n_nonedges"]) == len(nonedge)
        # pos3 / pos4 from the candidate alone
        lens = g.rs.descs["seq_len"]
        p3, p4 = ctypes.c_int32(0), ctypes.c_int32(0)
        for k in range(min(len(edges), 200)):
            c = cands[int(edges["cand"][k])]
            l1, l2 = lens[int(c["idx1"])], lens[int(c["idx2"])]
            capi.lib().hc_edge_extra_pos(int(c["pos1"]), int(c["pos2"]), bytes([int(c["ord"])]), int(l1[0]), int(l1[1]), int(l2[0]), int(l2[1]),
                                         ctypes.byref(p3), ctypes.byref(p4))
            assert (p3.value, p4.value) == (int(edges["pos3"][k]), int(edges["pos4"][k]))


def test_small_outputs_capacity_and_empty(built_lib):
    g = load_golden(golden_names()[0])
    cands = g.scored()
    with capi.Store(g.rs) as st:
        e, f, _ = st.score_batch_small(g.params(), cands[:0])
        assert len(e) == 0 and len(f) == 0
        full, _, _ = st.score_batch_small(g.params(), cands)
        assert len(full) > 1
        with pytest.raises(capi.HcError) as ei:
            st.score_batch_small(g.params(), cands, edges_cap=len(full) - 1)
        assert ei.value.code == -5 and ei.value.required[0] == len(full)


@pytest.mark.parametrize("seed", [11, 12, 13])
@pytest.mark.parametrize("exact", [False, True])
def test_run_records_equal_candidate_records(built_lib, seed, exact):
    rng = np.random.RandomState(seed)
    ss = W.synth_readset(int(rng.randint(20, 120)), int(rng.randint(20, 120)), genome_len=int(rng.randint(800, 4000)), read_len=(60, 400),
                         qmax=41, q_lo=int(rng.choice([2, 20])), seed=seed, n_rate=float(rng.choice([0.0, 0.002])), flip_fraction=0.3)
    c = W.geometry_candidates(ss, 6000, seed=seed + 1, junk_fraction=0.1, min_ov=20)
    c = c[(c["pos1"] < (1 << 14)) & (c["pos2"] < (1 << 14))]                                   # (junk candidates carry any position)
    c = c[np.lexsort((np.maximum(c["idx1"], c["idx2"]), np.minimum(c["idx1"], c["idx2"])))]     # sorted by read, like an overlaps file
    p = F.make_params(edge_threshold=0.95, ov_threshold=0.9, mismatch=float(rng.choice([0.0, 0.05])),
                      flags=F.FLAG_EXACT_EDGE_SCORES if exact else 0)
    with capi.Store(ss.rs) as st:
        e0, n0, p0, _ = st.score_batch(p, c)
        e1, n1, p1, _ = st.score_batch(p, c, compact="runs")
    assert p1.tobytes() == p0.tobytes() and e1.tobytes() == e0.tobytes() and np.array_equal(n1, n0)
