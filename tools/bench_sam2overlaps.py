#!/usr/bin/env python
"""lib/hc_sam2overlaps next to the reference's scripts/sam2overlaps.py (run from the temporary Python-3 copy that
oracle/make_golden_sam.py makes; build container only) on seeded SAM files.   python tools/bench_sam2overlaps.py [--reads 20000]

--gpu: the device leg instead, at each of --sizes (READS:REF_LEN, READS single-end reads and READS pairs, so 3 x READS
alignments, over one reference of REF_LEN bases) from workloads.make_sam_text: the host converter's wall time on all host threads, the wall time of
the same binary with --gpu=true, the hc_sam2overlaps call itself split into copy in, device and copy out, and whether the
outputs are byte-identical; with the GPU's name, power limit and max SM clock.  One JSON line per size.  Files go to a
temporary directory."""
import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
from haploconduct_b200 import build as B  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], check=True,
                           stdout=subprocess.PIPE, text=True).stdout.splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(","))
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except (OSError, subprocess.CalledProcessError, IndexError, ValueError):
        return {"gpu": "unknown"}


def sha(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for block in iter(lambda: f.read(1 << 24), b""):
            h.update(block)
    return h.hexdigest()


def device_leg(sizes, min_ov):
    from haploconduct_b200 import capi, workloads as W
    info = gpu_info()
    exe = os.path.join(B.LIBDIR, "hc_sam2overlaps")
    for reads, ref_len in sizes:
        d = tempfile.mkdtemp(prefix="hc_sam_bench_")
        try:
            fasta, sam_s, sam_p = W.make_sam_text(21, reads, reads, [("refA", ref_len)])
            for fn, text in (("ref.fasta", fasta), ("s.sam", sam_s), ("p.sam", sam_p)):
                with open(os.path.join(d, fn), "wb") as f:
                    f.write(text)
            args = [exe, "--ref", "ref.fasta", "--sam_s", "s.sam", "--sam_p", "p.sam", "--min_overlap_len", str(min_ov)]
            t0 = time.perf_counter()
            subprocess.run(args + ["--out", "host.txt"], cwd=d, check=True, stdout=subprocess.DEVNULL)
            t_host = time.perf_counter() - t0
            t0 = time.perf_counter()
            subprocess.run(args + ["--out", "gpu.txt", "--gpu=true"], cwd=d, check=True, stdout=subprocess.DEVNULL)
            t_gpu = time.perf_counter() - t0
            host_sha = sha(os.path.join(d, "host.txt"))
            same_cli = sha(os.path.join(d, "gpu.txt")) == host_sha
            os.remove(os.path.join(d, "gpu.txt"))
            capi.sam2overlaps(b"s\t0\tr\t1\t0\t4M\t=\t0\t0\tACGT\tIIII\n", None, {"r": 0}, [10], 0)   # context and module load
            t0 = time.perf_counter()
            out, st, _ = capi.sam2overlaps(sam_s, sam_p, {"refA": 0}, [ref_len], min_ov)
            t_call = time.perf_counter() - t0
            same_call = hashlib.sha256(out).hexdigest() == host_sha
            res = {"metric": "sam2overlaps wall time", "alignments": 3 * reads, "sam_bytes": len(sam_s) + len(sam_p), "ref_len": ref_len,
                   "min_overlap_len": min_ov, "out_lines": int(st["n_out_lines"]), "out_bytes": len(out),
                   "host_threads": int(os.environ.get("OMP_NUM_THREADS", os.cpu_count())), "host_cli_s": t_host, "gpu_cli_s": t_gpu,
                   "cli_speedup": t_host / t_gpu, "call_s": t_call, "call_copy_in_ms": float(st["h2d_ms"]),
                   "call_device_ms": float(st["device_ms"]), "call_copy_out_ms": float(st["d2h_ms"]),
                   "identical_output": same_cli and same_call, **info}
            print(json.dumps(res), flush=True)
        finally:
            shutil.rmtree(d, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=20000)
    ap.add_argument("--gpu", action="store_true", help="the device leg (needs a B200)")
    ap.add_argument("--sizes", default="20000:9000,333333:150000", help="--gpu: READS:REF_LEN, comma-separated")
    ap.add_argument("--min_overlap_len", type=int, default=50)
    a = ap.parse_args()
    if a.gpu:
        device_leg([tuple(int(v) for v in x.split(":")) for x in a.sizes.split(",")], a.min_overlap_len)
        return
    import make_golden_sam as G
    d = tempfile.mkdtemp(prefix="hc_sam_bench_")
    fasta, sam_s, sam_p = G.make_case(21, a.reads, a.reads, [("refA", 9000)])
    for fn, text in (("ref.fasta", fasta), ("s.sam", sam_s), ("p.sam", sam_p)):
        open(os.path.join(d, fn), "w").write(text)
    args = ["--ref", "ref.fasta", "--sam_s", "s.sam", "--sam_p", "p.sam", "--min_overlap_len", "50"]
    t0 = time.perf_counter()
    subprocess.run([os.path.join(B.LIBDIR, "hc_sam2overlaps")] + args + ["--out", "mine.txt"], cwd=d, check=True, stdout=subprocess.DEVNULL)
    t_mine = time.perf_counter() - t0
    res = {"metric": "sam2overlaps wall time", "alignments": 3 * a.reads, "threads": os.cpu_count(), "hc_sam2overlaps_s": t_mine,
           "overlap_lines": sum(1 for _ in open(os.path.join(d, "mine.txt")))}
    if os.path.exists(G.REF_SCRIPT):
        script = G.py3_copy(d)
        t0 = time.perf_counter()
        subprocess.run([sys.executable, script] + args + ["--out", "ref.txt"], cwd=d, check=True, stdout=subprocess.DEVNULL)
        res["reference_script_s"] = time.perf_counter() - t0
        res["speedup"] = res["reference_script_s"] / t_mine
        res["identical_output"] = open(os.path.join(d, "mine.txt"), "rb").read() == open(os.path.join(d, "ref.txt"), "rb").read()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
