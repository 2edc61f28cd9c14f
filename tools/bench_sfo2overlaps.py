#!/usr/bin/env python
"""lib/hc_sfo2overlaps next to the reference's scripts/sfo2overlaps.py (run from the temporary Python-3 copy that
oracle/make_golden_sfo.py makes; build container only) on a seeded SFO file.   python tools/bench_sfo2overlaps.py [--lines 400000]

--gpu: the device leg instead, at each of --sizes lines of workloads.make_sfo_text: the host converter's wall time on all
host threads, the wall time of the same binary with --gpu=true, the hc_sfo2overlaps call itself split into copy in,
device and copy out, and whether the two outputs are byte-identical; with the GPU's name, power limit and max SM clock.
One JSON line per size.  Files go to a temporary directory."""
import argparse
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


def device_leg(sizes, ns, npairs):
    from haploconduct_b200 import capi, workloads as W
    info = gpu_info()
    exe = os.path.join(B.LIBDIR, "hc_sfo2overlaps")
    for n in sizes:
        d = tempfile.mkdtemp(prefix="hc_sfo_bench_")
        try:
            text = W.make_sfo_text(17, ns, npairs, n, irregular=False)
            with open(os.path.join(d, "in.sfo"), "wb") as f:
                f.write(text)
            args = [exe, "--in", "in.sfo", "--num_singles", str(ns), "--num_pairs", str(npairs)]
            t0 = time.perf_counter()
            subprocess.run(args + ["--out", "host.txt"], cwd=d, check=True, stdout=subprocess.DEVNULL)
            t_host = time.perf_counter() - t0
            t0 = time.perf_counter()
            subprocess.run(args + ["--out", "gpu.txt", "--gpu=true"], cwd=d, check=True, stdout=subprocess.DEVNULL)
            t_gpu = time.perf_counter() - t0
            with open(os.path.join(d, "host.txt"), "rb") as f:
                host = f.read()
            with open(os.path.join(d, "gpu.txt"), "rb") as f:
                same_cli = f.read() == host
            capi.sfo2overlaps(b"1\t2\tN\t3\t4\t50\t50\t0\n", 5, 0)          # context and module load outside the timed call
            t0 = time.perf_counter()
            out, st = capi.sfo2overlaps(text, ns, npairs)
            t_call = time.perf_counter() - t0
            res = {"metric": "sfo2overlaps wall time", "sfo_lines": n, "sfo_bytes": len(text), "out_lines": int(st["n_out_lines"]),
                   "host_threads": int(os.environ.get("OMP_NUM_THREADS", os.cpu_count())), "host_cli_s": t_host, "gpu_cli_s": t_gpu,
                   "cli_speedup": t_host / t_gpu, "call_s": t_call, "call_copy_in_ms": float(st["h2d_ms"]),
                   "call_device_ms": float(st["device_ms"]), "call_copy_out_ms": float(st["d2h_ms"]),
                   "identical_output": same_cli and out == host, **info}
            print(json.dumps(res), flush=True)
        finally:
            shutil.rmtree(d, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lines", type=int, default=400000)
    ap.add_argument("--gpu", action="store_true", help="the device leg (needs a B200)")
    ap.add_argument("--sizes", default="1000000,50000000", help="--gpu: SFO lines per run, comma-separated")
    a = ap.parse_args()
    if a.gpu:
        device_leg([int(x) for x in a.sizes.split(",")], 200000, 1500000)
        return
    import make_golden_sfo as G
    d = tempfile.mkdtemp(prefix="hc_sfo_bench_")
    ns, npairs = 20000, 60000
    text = G.make_sfo(11, ns, npairs, a.lines)
    open(os.path.join(d, "in.sfo"), "w").write(text)
    args = ["--in", "in.sfo", "--num_singles", str(ns), "--num_pairs", str(npairs)]
    t0 = time.perf_counter()
    subprocess.run([os.path.join(B.LIBDIR, "hc_sfo2overlaps")] + args + ["--out", "mine.txt"], cwd=d, check=True, stdout=subprocess.DEVNULL)
    t_mine = time.perf_counter() - t0
    res = {"metric": "sfo2overlaps wall time", "sfo_lines": text.count("\n"), "threads": os.cpu_count(), "hc_sfo2overlaps_s": t_mine}
    if os.path.exists(G.REF_SCRIPT):
        script = G.py3_copy(d)
        t0 = time.perf_counter()
        subprocess.run([sys.executable, script] + args + ["--out", "ref.txt"], cwd=d, env=dict(os.environ, LC_ALL="C"), check=True, stdout=subprocess.DEVNULL)
        res["reference_script_s"] = time.perf_counter() - t0
        res["speedup"] = res["reference_script_s"] / t_mine
        res["identical_output"] = open(os.path.join(d, "mine.txt"), "rb").read() == open(os.path.join(d, "ref.txt"), "rb").read()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
