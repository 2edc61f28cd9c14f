#!/usr/bin/env python
"""Throughput of FindNextOverlaps 1 on one B200 (hc_fno1, host buffers in and out) next to the pinned C restatement
of the reference's sequential walk (oracle/fno_oracle.c, one host core) on the same input.

The "text" leg times hc_fno1_text (overlaps.txt formatted, sorted and de-duplicated on the device) into a pinned and
into a pageable buffer, checks its bytes once against the Python statement of the reference's std::set<std::string>,
and times, on the same records, the host step it replaces (snprintf + std::set<std::string> + concatenation, as the
C++ binding did it), compiled here with the build's host compiler.

    python tools/bench_fno.py [--edges 10000000] [--vertices 1000000] [--steps 5]
Prints one JSON line."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from haploconduct_b200 import build as B, capi, formats as F  # noqa: E402

HOST_FORMAT = r"""
#include <chrono>
#include <cstdio>
#include <set>
#include <string>
#include "hc_b200.h"
// the host step of the C++ binding before hc_fno1_text: one snprintf per record into a std::set<std::string>, then the
// set's lines concatenated with '\n'
extern "C" double host_format(const hc_fno_overlap* o, unsigned long long n, unsigned long long* bytes, unsigned long long* lines) {
    const auto t0 = std::chrono::steady_clock::now();
    std::set<std::string> set;
    std::string line;
    char buf[160];
    for (unsigned long long k = 0; k < n; k++) {
        const int m = std::snprintf(buf, sizeof(buf), "%lu\t%lu\t%d\t%d\t%c\t%c\t%c\t%d\t%d\t%d\t%d\t%c\t%c", (unsigned long)o[k].id1,
                                    (unsigned long)o[k].id2, o[k].pos1, o[k].pos2, o[k].ord, o[k].ori1, o[k].ori2, o[k].perc, o[k].perc2,
                                    o[k].len1, o[k].len2, o[k].type1, o[k].type2);
        line.assign(buf, (size_t)m);
        set.insert(line);
    }
    std::string out;
    for (const std::string& l : set) { out.append(l); out.push_back('\n'); }
    *bytes = out.size();
    *lines = set.size();
    return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}
"""


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             check=True, stdout=subprocess.PIPE, text=True).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:          # the numbers are only worth something with the card they were taken on
        return {"error": str(e)}


def host_format_seconds(records: np.ndarray):
    """(seconds, bytes, lines) of the replaced host step on `records` (formats.FNO_OVERLAP), built in a temporary directory."""
    import ctypes
    with tempfile.TemporaryDirectory() as d:
        src, so = os.path.join(d, "host_format.cpp"), os.path.join(d, "host_format.so")
        with open(src, "w") as f:
            f.write(HOST_FORMAT)
        subprocess.check_call([B.HOST_CXX, "-O2", "-std=c++14", "-shared", "-fPIC", "-I" + os.path.join(ROOT, "include"), src, "-o", so])
        L = ctypes.CDLL(so)
    L.host_format.restype = ctypes.c_double
    L.host_format.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)]
    rec = np.ascontiguousarray(records)
    nb, nl = ctypes.c_uint64(0), ctypes.c_uint64(0)
    dt = L.host_format(rec.ctypes.data, len(rec), ctypes.byref(nb), ctypes.byref(nl))
    return dt, nb.value, nl.value


def text_leg(fi: F.FnoInput, records: np.ndarray, steps: int) -> dict:
    import ctypes
    L = capi.lib()
    st, keep = capi._fno_input_c(fi)
    edges = np.ascontiguousarray(fi.edges)
    text = capi.fno1_text(fi)                                      # warm-up; sizes the buffers
    n = len(text)
    pinned = capi.host_alloc(n)
    pageable = np.empty(n, dtype=np.uint8)
    pageable[:] = 0                                                # touched once: no page faults inside the timed calls
    nb, nl, nr = ctypes.c_uint64(0), ctypes.c_uint64(0), ctypes.c_uint64(0)
    t = {"pinned": [], "pageable": []}
    for _ in range(steps):
        for kind, buf in (("pinned", pinned), ("pageable", pageable)):
            t0 = time.perf_counter()
            rc = L.hc_fno1_text(ctypes.byref(st), edges.ctypes.data, len(edges), buf.ctypes.data, n, ctypes.byref(nb), ctypes.byref(nl),
                                ctypes.byref(nr), 0)
            t[kind].append(time.perf_counter() - t0)
            assert rc == 0 and nb.value == n
    assert pinned[:n].tobytes() == text and pageable.tobytes() == text
    ref = sorted(set(F.fno_lines(records)), key=lambda s: s.encode())
    identical = text == "".join(l + "\n" for l in ref).encode()
    del ref
    host_s, host_bytes, host_lines = host_format_seconds(records)
    return {"ms_pinned": statistics.median(t["pinned"]) * 1e3, "ms_pageable": statistics.median(t["pageable"]) * 1e3,
            "bytes": n, "lines": int(nl.value), "records": int(nr.value), "identical_to_sorted_set_of_lines": bool(identical),
            "host_step_replaced": {"what": "snprintf + std::set<std::string> + concatenation, one host core, same records",
                                   "s": host_s, "bytes": int(host_bytes), "lines": int(host_lines)}}


def make_input(V: int, n_sr: int, n_edges: int, seed: int = 3, paired_fraction: float = 0.4) -> F.FnoInput:
    """The dense random input of tests/util.random_fno_input, vectorised for 1e6+ vertices."""
    rng = np.random.RandomState(seed)
    visited = (rng.random_sample(V) < 0.6).astype(np.uint8)
    label = rng.randint(0, 2, size=V).astype(np.uint8)
    vr = np.zeros(V, dtype=F.FNO_READ)
    vr["id"] = rng.permutation(V) + n_sr
    vr["len1"] = rng.randint(60, 300, size=V)
    vr["len2"] = np.where(rng.random_sample(V) < paired_fraction, rng.randint(60, 300, size=V), 0)
    sr = np.zeros(n_sr, dtype=F.FNO_READ)
    sr["id"] = np.arange(n_sr)
    sr["len1"] = rng.randint(100, 900, size=n_sr)
    sr["len2"] = np.where(rng.random_sample(n_sr) < paired_fraction, rng.randint(100, 900, size=n_sr), 0)
    k = np.where(visited > 0, rng.randint(0, 5, size=V), 0)
    off = np.zeros(V + 1, dtype=np.uint64)
    off[1:] = np.cumsum(k)
    n_ent = int(off[-1])
    owner = np.repeat(np.arange(V), k)
    j = np.arange(n_ent) - off[:-1][owner].astype(np.int64)
    start = rng.randint(0, n_sr, size=V)[owner]
    idx = ((start + j * 7919) % n_sr).astype(np.uint32)           # distinct super-reads within one vertex
    sub = np.zeros(n_ent, dtype=F.FNO_SUBREAD)
    i1, i2 = rng.randint(0, 400, size=n_ent), rng.randint(0, 400, size=n_ent)
    names = sub.dtype.names
    sub[names[0]], sub[names[1]] = i1, i2
    sub[names[2]] = np.where((i1 > 0) & (rng.random_sample(n_ent) < 0.8), 0, rng.randint(0, 30, size=n_ent))
    sub[names[3]] = np.where((i2 > 0) & (rng.random_sample(n_ent) < 0.8), 0, rng.randint(0, 30, size=n_ent))
    e = np.zeros(n_edges, dtype=F.FNO_EDGE)
    e["u"] = rng.randint(0, V, size=n_edges)
    e["v"] = (e["u"] + rng.randint(1, V, size=n_edges)) % V
    e["pos1"], e["pos2"] = rng.randint(0, 250, size=n_edges), rng.randint(0, 250, size=n_edges)
    e["perc"] = rng.randint(20, 101, size=n_edges)
    e["len1"], e["len2"] = rng.randint(30, 250, size=n_edges), rng.randint(0, 250, size=n_edges)
    pu, pv = vr["len2"][e["u"]] > 0, vr["len2"][e["v"]] > 0
    e["ord"] = np.where(pu & pv, np.where(rng.random_sample(n_edges) < 0.5, ord("1"), ord("2")), ord("-"))
    e["ori1"], e["ori2"] = rng.randint(0, 2, size=n_edges), rng.randint(0, 2, size=n_edges)
    e["nonedge"] = rng.random_sample(n_edges) < 0.5
    return F.FnoInput(visited=visited, label=label, vertex_read=vr, sr_off=off, sr_idx=idx, sr_sub=sub, superread=sr,
                      resolve_orientations=1, no_inclusions=0, edges=e)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--edges", type=int, default=10_000_000)
    ap.add_argument("--vertices", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--cpu-edges", type=int, default=2_000_000)
    ap.add_argument("--no-text", action="store_true", help="skip the text leg")
    a = ap.parse_args()
    fi = make_input(a.vertices, a.vertices // 3, a.edges)
    import ctypes
    out = capi.fno1(fi)                                            # warm-up (also sizes the output)
    L = capi.lib()
    keep = [np.ascontiguousarray(x) for x in (fi.visited, fi.label, fi.vertex_read, fi.sr_off, fi.sr_idx, fi.sr_sub, fi.superread)]
    st = capi._FnoInputC(len(fi.visited), *[k.ctypes.data for k in keep[:6]], len(fi.superread), keep[6].ctypes.data,
                         fi.resolve_orientations, fi.no_inclusions)
    edges = np.ascontiguousarray(fi.edges)
    buf = np.zeros(len(out) + 16, dtype=F.FNO_OVERLAP)              # touched once: no page faults inside the timed calls
    bufs = np.zeros(len(out) + 16, dtype=capi.FNO_OVERLAP_SMALL)
    n = ctypes.c_uint64(0)
    t, ts = [], []
    for _ in range(a.steps):
        t0 = time.perf_counter()
        rc = L.hc_fno1(ctypes.byref(st), edges.ctypes.data, len(edges), buf.ctypes.data, len(buf), ctypes.byref(n), 0)
        t.append(time.perf_counter() - t0)
        assert rc == 0 and n.value == len(out)
        t0 = time.perf_counter()
        rc = L.hc_fno1_small(ctypes.byref(st), edges.ctypes.data, len(edges), bufs.ctypes.data, len(bufs), ctypes.byref(n), 0)
        ts.append(time.perf_counter() - t0)
        assert rc == 0 and n.value == len(out)
    assert buf[: len(out)].tobytes() == out.tobytes()
    assert capi.fno_small_to_overlaps(bufs[: len(out)]).tobytes() == out.tobytes()
    best = min(ts)
    res = {"metric": "FNO1 edges processed per second (host buffers, incl. all copies and allocations)", "unit": "edges/s",
           "edges": a.edges, "vertices": a.vertices, "overlaps_out": int(len(out)), "ms": best * 1e3, "value": a.edges / best,
           "records": "hc_fno1_small: 24-byte result records (the call of the C++ binding hcb::SRBuilder)",
           "ms_48_byte_records": min(t) * 1e3,
           "bytes_in": int(fi.edges.nbytes + fi.sr_sub.nbytes + fi.sr_idx.nbytes + fi.vertex_read.nbytes + fi.superread.nbytes),
           "bytes_out": int(len(out) * 24), "bytes_out_48": int(out.nbytes), "gpu": gpu_info()}
    if not a.no_text:
        res["text"] = text_leg(fi, out, a.steps)
    try:
        from oracle import oracle as O
        import copy
        small = copy.copy(fi)
        small.edges = fi.edges[: a.cpu_edges]
        t0 = time.perf_counter()
        ref = O.fno1(small)
        dt = time.perf_counter() - t0
        mine = capi.fno1(small)
        res["cpu_baseline"] = {"kind": "port", "cores": 1, "edges": int(len(small.edges)), "value": len(small.edges) / dt,
                               "identical_output": bool(mine.tobytes() == ref.tobytes())}
    except Exception as ex:      # the oracle is test infrastructure; its absence only removes the baseline
        res["cpu_baseline"] = {"unavailable": str(ex)[:200]}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
