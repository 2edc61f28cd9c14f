#!/usr/bin/env python
"""FindNextOverlaps 1 with the non-edge file parsed on the host (the loop of hcb_fno.cpp, src/FindNextOverlaps.cpp:635-697)
and on the device (lib/hc_fno --gpu_parse=true, hc_fno1_text_nonedges), alternated on one B200:

    python tools/bench_fno_nonedge.py [--reads 2000000] [--adjacency 2500000] [--nonedge 10000000] [--rounds 3] [--out f.json]

Inputs are generated into a temporary directory from a seed: single-end FASTQ reads (ids 0..n-1, so vertex i is read i),
a state file with --adjacency adjacency edges (one in ten a non-edge overlap, score 0) and no merged reads, and a
nonedge_overlaps.txt of --nonedge lines, a fifth of them on an adjacency pair (in either direction), the rest on random
pairs.  Every round runs lib/hc_fno once each way; the two overlaps.txt files must be byte-identical.  Prints one JSON
line: per run the findNextOverlaps wall time (t_stream_s + t_device_s + t_format_s of hc_fno's summary), t_stream_s (the
host part of the stream) and nonedge_device_ms, with the GPU's name, power limit and clocks.  Benchmark tool, not product
code."""
import argparse
import filecmp
import json
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "haploconduct_b200", "lib", "hc_fno")


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader", "-i", "0"],
                             check=True, stdout=subprocess.PIPE, text=True).stdout.strip()
        name, power, clock, cur = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock, "sm_clock_at_start": cur}
    except Exception as e:          # the numbers are only worth something with the card they were taken on
        return {"error": str(e)}


def _cols_to_lines(cols):
    return "\n".join(map("\t".join, zip(*[c.astype(str).tolist() if isinstance(c, np.ndarray) else c for c in cols]))) + "\n"


def write_inputs(d, n_reads, n_adj, n_nonedge, seed):
    rng = np.random.RandomState(seed)
    read_len = 100
    seq, qual = "ACGT" * (read_len // 4), "I" * read_len
    with open(os.path.join(d, "s.fastq"), "w") as f:
        for b in range(0, n_reads, 1 << 20):
            f.write("".join("@%d\n%s\n+\n%s\n" % (i, seq, qual) for i in range(b, min(n_reads, b + (1 << 20)))))
    # adjacency lists in vertex order; A records: list vertex1 vertex2 pos1 pos2 ord ori1 ori2 score perc len1 len2
    u = np.sort(rng.randint(0, n_reads, size=n_adj))
    v = (u + rng.randint(1, n_reads, size=n_adj)) % n_reads
    pos1 = rng.randint(1, 60, size=n_adj)
    score = np.where(rng.random_sample(n_adj) < 0.1, "0", "0.995")
    n = n_adj
    with open(os.path.join(d, "state.txt"), "w") as f:
        f.write("P\t1\t0\t0\t0.99\t%d\n" % n_reads)
        ids = np.arange(n_reads)
        f.write(_cols_to_lines([np.full(n_reads, "V"), ids, np.zeros(n_reads, dtype=np.int64), ids, np.ones(n_reads, dtype=np.int64)]))
        f.write(_cols_to_lines([np.full(n, "A"), u, u, v, pos1, np.zeros(n, dtype=np.int64), np.full(n, "-"),
                                rng.randint(0, 2, size=n), rng.randint(0, 2, size=n), score, rng.randint(40, 100, size=n),
                                read_len - pos1, np.zeros(n, dtype=np.int64)]))
    # non-edge lines: ID1 ID2 POS1 POS2 ORD ORI1 ORI2 PERC1 PERC2 LEN1 LEN2 TYPE1 TYPE2
    m = n_nonedge
    on_adj = rng.random_sample(m) < 0.2
    k = rng.randint(0, n_adj, size=m)
    rev = rng.random_sample(m) < 0.5
    a = np.where(on_adj, np.where(rev, v[k], u[k]), rng.randint(0, n_reads, size=m))
    b = np.where(on_adj, np.where(rev, u[k], v[k]), rng.randint(0, n_reads, size=m))
    p1 = rng.randint(1, 80, size=m)
    with open(os.path.join(d, "nonedge_overlaps.txt"), "w") as f:
        for s in range(0, m, 1 << 21):
            e = slice(s, min(m, s + (1 << 21)))
            c = e.stop - e.start
            f.write(_cols_to_lines([a[e], b[e], p1[e], np.zeros(c, dtype=np.int64), np.full(c, "-"),
                                    np.where(rng.random_sample(c) < 0.5, "+", "-"), np.where(rng.random_sample(c) < 0.5, "+", "-"),
                                    rng.randint(20, 100, size=c), np.zeros(c, dtype=np.int64), read_len - p1[e],
                                    np.zeros(c, dtype=np.int64), np.full(c, "s"), np.full(c, "s")]))


def run(d, gpu_parse):
    out = os.path.join(d, "out_gpu" if gpu_parse else "out_host") + "/"
    os.makedirs(out, exist_ok=True)
    shutil.copy(os.path.join(d, "nonedge_overlaps.txt"), out)
    p = subprocess.run([EXE, "--state", os.path.join(d, "state.txt"), "--output", out, "--FNO", "1",
                        "--singles", os.path.join(d, "s.fastq"), "--gpu_parse=" + ("true" if gpu_parse else "false")],
                       check=True, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    s = json.loads([l for l in p.stdout.split("\n") if l.startswith("{")][-1])
    s["fno_wall_s"] = s["t_stream_s"] + s["t_device_s"] + s["t_format_s"]
    return out + "overlaps.txt", s


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=2_000_000)
    ap.add_argument("--adjacency", type=int, default=2_500_000)
    ap.add_argument("--nonedge", type=int, default=10_000_000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    d = tempfile.mkdtemp(prefix="bench_fno_nonedge_")
    try:
        write_inputs(d, a.reads, a.adjacency, a.nonedge, a.seed)
        res = {"metric": "FindNextOverlaps 1, non-edge file parsed on the host vs on the device (lib/hc_fno), seconds",
               "gpu": gpu_info(), "reads": a.reads, "adjacency_edges": a.adjacency, "nonedge_lines": a.nonedge,
               "nonedge_bytes": os.path.getsize(os.path.join(d, "nonedge_overlaps.txt")), "host": [], "device": []}
        for r in range(a.rounds):
            order = (True, False) if r % 2 == 0 else (False, True)
            files = {}
            for g in order:
                files[g], s = run(d, g)
                if s["nonedge_on_device"] != int(g):
                    raise SystemExit("hc_fno --gpu_parse=%s did not take the path it was asked for" % ("true" if g else "false"))
                res["device" if g else "host"].append({k: s[k] for k in ("fno_wall_s", "t_stream_s", "t_device_s", "t_format_s",
                                                                          "nonedge_lines", "nonedge_kept", "nonedge_on_device",
                                                                          "nonedge_device_ms",
                                                                          "stream", "lines")})
            if not filecmp.cmp(files[True], files[False], shallow=False):
                raise SystemExit("overlaps.txt differs between the host and the device non-edge parse")
        res["identical_overlaps_txt"] = True
        res["overlaps_txt_bytes"] = os.path.getsize(files[True])
        line = json.dumps(res)
        print(line)
        if a.out:
            with open(a.out, "w") as f:
                f.write(line + "\n")
    finally:
        shutil.rmtree(d, ignore_errors=True)


if __name__ == "__main__":
    main()
