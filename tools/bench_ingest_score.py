#!/usr/bin/env python
"""Overlaps-file text -> kept candidates and edges on one B200, two ways, alternated in one process:

  (a) hc_ingest_overlaps -> run encoding on the host -> hc_score_batch_runs_small   (every scored line comes back as a
      32-byte record and goes in again as an 8-byte run record)
  (b) hc_ingest_score_overlaps                                                      (only the candidates scored as edges
      or non-edges come back)

    python tools/bench_ingest_score.py [--pairs 3000000] [--rounds 3]

The input is built as tools/bench_pipeline.py builds it (paired 2x150 bp reads, real P-P overlaps between them), so the
kept fraction is that of a real overlaps file; it is printed next to the times.  Each of (a) and (b) runs from pageable
and from pinned (hc_host_alloc) text; output buffers are pageable numpy arrays, allocated once.  Prints one JSON line.
Benchmark tool, not product code."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_pipeline import write_inputs  # noqa: E402
from haploconduct_b200 import capi, formats as F  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             check=True, stdout=subprocess.PIPE, text=True).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:          # the numbers are only worth something with the card they were taken on
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=3_000_000)
    ap.add_argument("--partners", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seed", type=int, default=7)
    a = ap.parse_args()
    L = capi.lib()
    d = tempfile.mkdtemp(prefix="hc_ingest_score_")
    write_inputs(d, a.pairs, 150, a.partners, a.seed)
    with open(os.path.join(d, "ov.txt"), "rb") as f:
        text = f.read()
    n_lines = text.count(b"\n") + 1
    st = capi.Store.from_fastq_files(paired1=os.path.join(d, "p1.fastq"), paired2=os.path.join(d, "p2.fastq"))
    ids, _ = st.read_ids()
    m = capi.IdMap(ids)
    ip = F.make_ingest_params(150)                      # bench_pipeline's --min_overlap_len / --edge_threshold
    p = F.make_params(edge_threshold=0.97)
    erec = F.EDGE_SMALL.itemsize
    pageable = np.frombuffer(text, dtype=np.uint8)
    pinned = capi.host_alloc(len(text))
    pinned[:] = pageable
    # output buffers, allocated (and touched) once
    cand = np.zeros(n_lines, dtype=F.CANDIDATE)
    filt = np.zeros(n_lines, dtype=F.OVERLAP_REC)
    ist = np.zeros(1, dtype=F.INGEST_STATS)
    bst = np.zeros(1, dtype=F.BATCH_STATS)
    edges_a = np.zeros(n_lines, dtype=F.EDGE_SMALL)
    bits = np.zeros(n_lines // 64 + 2, dtype=np.uint64)
    kept = np.zeros(n_lines, dtype=F.CANDIDATE)
    kc = np.zeros(n_lines, dtype=np.uint8)
    edges_b = np.zeros(n_lines, dtype=F.EDGE_SMALL)
    sst = np.zeros(1, dtype=F.INGEST_SCORE_STATS)
    ne, nn = ctypes.c_uint64(0), ctypes.c_uint64(0)

    def run_a(buf):
        t0 = time.perf_counter()
        rc = L.hc_ingest_overlaps(m.handle, buf.ctypes.data, len(buf), ip.ctypes.data, cand.ctypes.data, None, n_lines, filt.ctypes.data,
                                  None, n_lines, ist.ctypes.data)
        assert rc == 0, capi.last_error()
        t1 = time.perf_counter()
        n = int(ist[0]["n_scored"])
        anchor, start, entries = F.run_encode(cand[:n])
        t2 = time.perf_counter()
        rc = L.hc_score_batch_runs_small(st.handle, p.ctypes.data, anchor.ctypes.data, start.ctypes.data, len(anchor), entries.ctypes.data, n,
                                         edges_a.ctypes.data, n_lines, ctypes.byref(ne), bits.ctypes.data, ctypes.byref(nn), bst.ctypes.data)
        assert rc == 0, capi.last_error()
        t3 = time.perf_counter()
        e, nf = int(ne.value), int(ist[0]["n_filtered"])
        return {"wall_ms": (t3 - t0) * 1e3, "ingest_wall_ms": (t1 - t0) * 1e3, "run_encoding_ms": (t2 - t1) * 1e3, "score_wall_ms": (t3 - t2) * 1e3,
                "ingest_device_ms": float(ist[0]["device_ms"]), "score_device_ms": float(bst[0]["total_ms"]),
                "h2d_bytes": len(buf) + n * 8 + len(anchor) * 8 + 8,
                "d2h_bytes": n * 32 + nf * 48 + e * erec + ((n + 63) // 64) * 8}

    def run_b(buf):
        t0 = time.perf_counter()
        rc = L.hc_ingest_score_overlaps(st.handle, m.handle, buf.ctypes.data, len(buf), ip.ctypes.data, p.ctypes.data, kept.ctypes.data, None,
                                        kc.ctypes.data, n_lines, edges_b.ctypes.data, n_lines, filt.ctypes.data, None, n_lines, sst.ctypes.data)
        assert rc == 0, capi.last_error()
        t1 = time.perf_counter()
        s = sst[0]
        k, e, nf = int(s["n_kept"]), int(s["score"]["n_edges"]), int(s["ingest"]["n_filtered"])
        return {"wall_ms": (t1 - t0) * 1e3, "ingest_device_ms": float(s["ingest"]["device_ms"]), "score_device_ms": float(s["score"]["kernel_ms"]),
                "h2d_bytes": len(buf), "d2h_bytes": k * (32 + 1) + nf * 48 + e * erec}

    def same():
        """(a) and (b) keep the same candidates, classify them alike and emit the same edge records (cand remapped)."""
        n = int(ist[0]["n_scored"])
        cls = np.zeros(n, dtype=np.uint8)
        flags = np.unpackbits(bits[: (n + 63) // 64].view(np.uint8), bitorder="little")[:n].astype(bool)
        cls[flags] = F.CLASS_NONEDGE
        ea = edges_a[: int(ne.value)].copy()
        cls[ea["cand"].astype(np.int64)] = F.CLASS_EDGE
        keep = np.nonzero(cls)[0]
        ea["cand"] = np.searchsorted(keep, ea["cand"].astype(np.int64))
        k = int(sst[0]["n_kept"])
        return bool(k == len(keep) and cand[keep].tobytes() == kept[:k].tobytes() and cls[keep].tobytes() == kc[:k].tobytes()
                    and ea.tobytes() == edges_b[: int(sst[0]["score"]["n_edges"])].tobytes())

    for buf in (pageable, pinned):      # warm-up: contexts, workspaces, tables
        run_a(buf)
        run_b(buf)
    res = {"metric": "overlaps-file text -> kept candidates + edge records, wall ms per call", "gpu": gpu_info(), "pairs": a.pairs,
           "overlaps_file_bytes": len(text), "lines": n_lines - 1}
    for name, buf in (("pageable", pageable), ("pinned", pinned)):
        ra, rb, eq = [], [], []
        for _ in range(a.rounds):
            ra.append(run_a(buf))
            rb.append(run_b(buf))
            eq.append(same())
        res[name] = {"a_ingest_encode_score": ra, "b_ingest_score": rb, "same_outputs": all(eq),
                     "a_wall_ms_range": [min(r["wall_ms"] for r in ra), max(r["wall_ms"] for r in ra)],
                     "b_wall_ms_range": [min(r["wall_ms"] for r in rb), max(r["wall_ms"] for r in rb)]}
    n, k = int(ist[0]["n_scored"]), int(sst[0]["n_kept"])
    res["scored"], res["kept"], res["edges"], res["filtered"] = n, k, int(sst[0]["score"]["n_edges"]), int(sst[0]["ingest"]["n_filtered"])
    res["kept_fraction_of_scored"] = k / max(n, 1)
    res["note"] = ("score_device_ms: (a) CUDA events around the whole hc_score_batch_runs_small call, copies included; (b) the scoring "
                   "and compaction kernels summed over the pieces.  ingest_device_ms: the ingestion kernels in both.  run_encoding_ms: "
                   "formats.run_encode (numpy), not the host mirror's OpenMP loop.  Bytes are computed from the counts.")
    L.hc_host_free(pinned.ctypes.data)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
