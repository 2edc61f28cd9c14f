#!/usr/bin/env python
"""bench.py -- candidate overlaps scored per second on config 4 of BASELINE.json.

Workload (config.workload): synthetic 10 M 2x150 bp pairs replicated in each GPU's HBM, ~1e9 P-P
candidate overlaps sharded in 8 contiguous ranges; every GPU scores one shard of 1.25e8 candidates
per step ("weak" scaling: N GPUs score N shards; N = 8 is the whole list).

  value     candidates/s with the candidate records already resident in HBM (CUDA events on the
            launching stream, barrier + synchronize on both sides, max over ranks)
  e2e       the same step through hc_score_batch_runs() on HOST buffers: pinned host candidates (run-encoded 8-byte
            records; --e2e-records short|compact for the 12- / 16-byte ones) -> device, kernels, accepted edges +
            non-edge indices -> host, inside the timed region
  roofline  hc_score_kernel: algorithmic bytes per launch / its CUDA-event duration vs the measured
            HBM copy bandwidth of MEASURED_PEAKS.json
  cpu_baseline  the UNMODIFIED reference's scoring region (oracle/_ref/ref_driver --time-scoring,
            OpenMP over all host cores) on a bounded sample of the same candidates
  --impl reference   only that CPU measurement, as the driver's reference arm.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "candidate_overlaps_scored_per_sec"
UNIT = "candidates/s"
N_SHARDS = 8
PARAMS = dict(edge_threshold=0.97, ov_threshold=0.9, merge_contigs=0.0, mismatch=0.0, min_read_len=0)   # SAVAGE stage a
MIN_OVERLAP_LEN = 150


# stdout carries exactly one JSON line: everything libraries print to file descriptor 1 (NCCL prints its version
# there when NCCL_DEBUG=VERSION) is sent to stderr, the line itself goes to the saved descriptor.
_REAL_STDOUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line: dict) -> None:
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def workload_name(args) -> str:
    return ("C4 synthetic %d 2x%dbp pairs (store replicated per GPU), P-P candidates, shard r of %d of the ~%.2g-candidate "
            "list: %d candidates per GPU per step%s" % (args.pairs, args.read_len, N_SHARDS, args.pairs * 100.0, args.cands,
                                                         " [diagnostic: 4-bin qualities]" if getattr(args, "binned_qualities", False) else ""))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for t, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9 or not (t0 - 0.05 <= t <= t1 + 0.15):
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            for t, line in self.rows[-3:]:
                f = [x.strip() for x in line.split(",")]
                try:
                    sm.append(float(f[1])); smax.append(float(f[2]))
                except Exception:
                    pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def kernel_source_sha() -> str:
    import hashlib
    h = hashlib.sha256()
    for f in ("hc_kernels.cu", "hc_kernels.cuh", "hc_layout.h"):
        with open(os.path.join(ROOT, "haploconduct_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def measured_traffic(n_candidates: int, default_config: bool):
    """dram__bytes_read.sum + dram__bytes_write.sum of hc_score_kernel per launch, from the committed ncu --set full
    capture of this same configuration (bench.py cannot run under a profiler itself).  The capture names the kernel
    sources it was taken with; if they have changed since, the number is withheld rather than repeated."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            t = json.load(f)
        if not default_config:
            return None, "not the captured configuration"
        if t.get("kernel_source_sha") != kernel_source_sha():
            return None, "stale: %s was captured with kernel sources %s, these are %s" % (t["source"], t.get("kernel_source_sha"), kernel_source_sha())
        return float(t["dram_bytes_per_candidate"]) * n_candidates, t["source"]
    except Exception as ex:
        return None, "unavailable: %r" % (ex,)


def bind_to_gpu_numa_node(gpu_index: int):
    """Pin this process (and so its first-touch / pinned host allocations) to the CPUs of the NUMA node the GPU hangs
    off: at 8 ranks the host-side copies otherwise cross the socket interconnect."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        with open("/sys/bus/pci/devices/%s/numa_node" % bus) as f:
            node = int(f.read().strip())
        if node < 0:
            return {"node": node, "bound": False, "why": "no NUMA information for the device"}
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if not allowed:
            return {"node": node, "bound": False, "why": "none of the node's CPUs is available to this process"}
        os.sched_setaffinity(0, allowed)
        return {"node": node, "bound": True, "cpus": len(allowed)}
    except Exception as ex:
        return {"bound": False, "why": repr(ex)}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---- CPU arm: the unmodified reference's scoring region on a bounded sample -------------------------
def write_sample_files(d: str, rs_bases: np.ndarray, rs_quals: np.ndarray, read_len: int, cands: np.ndarray):
    """FASTQ pair + overlaps file for the reads the sampled candidates touch (ids renumbered densely)."""
    from haploconduct_b200 import formats as F

    used = np.unique(np.concatenate([cands["idx1"], cands["idx2"]]))
    L = read_len
    with open(os.path.join(d, "p1.fastq"), "w") as f1, open(os.path.join(d, "p2.fastq"), "w") as f2:
        for new, old in enumerate(used):
            o = int(old) * 2 * L
            f1.write("@%d\n%s\n+\n%s\n" % (new, rs_bases[o:o + L].tobytes().decode(), rs_quals[o:o + L].tobytes().decode()))
            f2.write("@%d\n%s\n+\n%s\n" % (new, rs_bases[o + L:o + 2 * L].tobytes().decode(),
                                           rs_quals[o + L:o + 2 * L].tobytes().decode()))
    c = cands.copy()
    c["idx1"] = np.searchsorted(used, cands["idx1"]).astype(np.uint32)
    c["idx2"] = np.searchsorted(used, cands["idx2"]).astype(np.uint32)
    F.write_overlaps(os.path.join(d, "ov.txt"), c, np.arange(len(used), dtype=np.uint64))
    return len(used)


def run_cpu_reference(bases: np.ndarray, quals: np.ndarray, read_len: int, cands: np.ndarray, reps: int, threads: int):
    from oracle import oracle as O

    if not O.have_ref():
        raise RuntimeError("oracle/_ref/ref_driver is missing (it is built by __graft_entry__.build() where /root/reference exists)")
    d = tempfile.mkdtemp(prefix="hc_cpu_")
    n_reads = write_sample_files(d, bases, quals, read_len, cands)
    out = O.run_ref(d, os.path.join(d, "ov.txt"), None, os.path.join(d, "p1.fastq"), os.path.join(d, "p2.fastq"), threads=threads,
                    time_scoring=True, reps=reps, edge_threshold=PARAMS["edge_threshold"], min_overlap_len=MIN_OVERLAP_LEN)
    assert out["scored"] == len(cands), (out["scored"], len(cands))
    return out, n_reads


def cpu_model() -> str:
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


DUMP_SAMPLE = 1 << 19     # candidates in the --dump-outputs sample: at most 2 + 9 float64 values each, 44 MB in all
DUMP_SEED = 1


def dump_outputs(out_dir: str, n: int, d_edges, d_nonedge, d_counts) -> None:
    """Writes what a step of hc_score_batch_device handed back (hc_edge records, non-edge indices, counts) as float64 .npy
    files of finite values, so that two builds run with the same arguments can be compared output for output: counts.npy
    whole; for a fixed seeded sample of the step's candidates cand.npy (index) and cls.npy (0 discarded, 1 edge, 2 non-edge);
    for the sampled candidates that are edges, in the same order, the hc_edge fields edge_cand, edge_score,
    edge_mismatch_rate, edge_pos3, edge_pos4, edge_mean_log (0 for a window that was not scored, where the record holds NaN)
    and edge_window_scored (1 where it was)."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    counts = d_counts.cpu()
    ne, nn = int(counts[0]), int(counts[1])
    pick = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=min(n, DUMP_SAMPLE), replace=False))
    k = torch.from_numpy(pick).to(d_edges.device)

    def find(sorted_idx):      # position of each sampled candidate in an input-ordered index list, and whether it is there
        if len(sorted_idx) == 0:
            return torch.zeros_like(k), torch.zeros_like(k, dtype=torch.bool)
        at = torch.searchsorted(sorted_idx, k).clamp_(max=len(sorted_idx) - 1)
        return at, sorted_idx[at] == k

    edges = d_edges[:ne]
    at, is_edge = find(edges.view(torch.int64)[:, 0].contiguous())
    _, is_non = find(d_nonedge[:nn])
    rec = edges[at[is_edge]]
    f64, i32 = rec.view(torch.float64), rec.view(torch.int32)
    mean_log = f64[:, 4:6]
    scored = ~torch.isnan(mean_log)
    cls = torch.where(is_edge, 1, torch.where(is_non, 2, 0))
    out = {"counts": counts.double().numpy(), "cand": pick.astype(np.float64), "cls": cls.double().cpu().numpy(),
           "edge_cand": rec.view(torch.int64)[:, 0].double(), "edge_score": f64[:, 1], "edge_mismatch_rate": f64[:, 2],
           "edge_pos3": i32[:, 6].double(), "edge_pos4": i32[:, 7].double(), "edge_mean_log": torch.where(scored, mean_log, 0.0),
           "edge_window_scored": scored.double()}
    for name, v in out.items():
        v = v.cpu().numpy() if torch.is_tensor(v) else v
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(v))


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs", type=int, default=10_000_000)
    ap.add_argument("--read-len", type=int, default=150)
    ap.add_argument("--cands", type=int, default=125_000_000, help="candidates per GPU per step")
    ap.add_argument("--partners", type=int, default=140, help="D: rank window of candidate partners")
    ap.add_argument("--cpu-sample", type=int, default=400_000, help="candidates in the CPU-baseline sample")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--binned-qualities", action="store_true",
                    help="diagnostic workload: qualities quantised to the four bins of current Illumina instruments")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true", help="skip the files-in -> graph-out leg (tools/bench_pipeline.py, about 20 s)")
    ap.add_argument("--e2e-no-output", action="store_true",
                    help="diagnostic: the e2e leg with zero output capacity (nothing is copied back; INVALID as an e2e number)")
    ap.add_argument("--dma-load", action="store_true",
                    help="diagnostic: run the device-resident steps while both copy engines are busy (1 GB in, 0.8 GB out per step)")
    ap.add_argument("--device-chunk", type=int, default=0,
                    help="diagnostic: split the device-resident step into launches of this many candidates (what the host pipeline's "
                         "steps cost without any copies)")
    ap.add_argument("--e2e-records", default="runs6", choices=["runs6", "runs", "short", "compact"],
                    help="host record of the e2e leg: run-encoded 6-byte hc_candidate_entry6 (reads < 512 bases, <= 2^25 reads), run-encoded "
                         "8-byte hc_candidate_entry, 12-byte hc_candidate_short (both: reads < 16384 bases) or 16-byte hc_candidate_compact")
    ap.add_argument("--e2e-output", default="small", choices=["small", "full"],
                    help="what the e2e leg brings back: hc_edge_small records + one bit per candidate (hc_score_batch_runs_small), "
                         "or 48-byte hc_edge records + 8-byte non-edge indices (hc_score_batch_runs)")
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "nccl"],
                    help="N > 1: how the accepted-edge lists are gathered: one-sided puts over NVLink peer memory on the copy engines (peer), "
                         "NCCL all-gather (nccl), or peer where it can be set up (auto)")
    ap.add_argument("--no-exchange", action="store_true", help="N > 1: leave the all-gather of the accepted edges out of the timed region")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin the process to the GPU's NUMA node")
    ap.add_argument("--seed", type=int, default=20261018)
    ap.add_argument("--exact-edge-scores", action="store_true",
                    help="HC_FLAG_EXACT_EDGE_SCORES: re-sum every accepted edge in the reference's order (diagnostic)")
    ap.add_argument("--position-sorted-ids", action="store_true",
                    help="diagnostic only: number the reads in genome order (cache-friendly, NOT the benchmark layout)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0: counts, the class of a fixed seeded sample of "
                         "its candidates and the edge fields of the sampled edges) to DIR/<name>.npy as float64, to compare two builds "
                         "output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.device_chunk):
        ap.error("--dump-outputs writes the outputs of the device-resident step of --impl ours, without --device-chunk")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    import torch
    from haploconduct_b200 import formats as F, workloads_torch as WT

    # ------------------------------------------------------------------ reference arm (CPU only)
    if args.impl == "reference":
        if rank != 0:
            return
        t0 = time.time()
        if torch.cuda.is_available():
            # the very workload of the GPU arm (torch generates it on the device: plumbing, none of this repo's kernels), and of
            # it the same prefix of shard 0 the GPU arm's cpu_baseline leg scores
            torch.cuda.set_device(local_rank)
            pr = WT.make_paired_reads(args.pairs, read_len=args.read_len, seed=args.seed, device="cuda:%d" % local_rank)
            rec = WT.make_pp_candidates(pr, D=args.partners, shard=0, n_shards=N_SHARDS, max_cands=args.cands)
            cands = WT.candidates_as_numpy(rec[: args.cpu_sample])
            del rec
            torch.cuda.empty_cache()
            what = "the first %d candidates of shard 0 of this workload" % len(cands)
        else:
            n_pairs_s = min(args.pairs, 400_000)
            genome_s = max(1000, 100_000 * n_pairs_s // max(args.pairs, 1))   # same coverage as the full configuration
            pr = WT.make_paired_reads(n_pairs_s, read_len=args.read_len, genome_len=genome_s, seed=args.seed, device="cpu")
            rec = WT.make_pp_candidates(pr, D=args.partners, shard=0, n_shards=N_SHARDS, max_cands=args.cpu_sample)
            cands = WT.candidates_as_numpy(rec)
            what = "%d candidates of the same generator at the same coverage (%d pairs on a %d bp genome; no GPU to generate the full read set)" % (
                len(cands), n_pairs_s, genome_s)
        threads = os.cpu_count() or 1
        out, n_reads = run_cpu_reference(pr.bases.numpy(), pr.quals.numpy(), args.read_len, cands, args.warmup + args.steps, threads)
        times = out["rep_times_s"][args.warmup:]
        ms = 1e3 * float(np.mean(times))
        v = len(cands) / (ms / 1e3)
        sample = "%s (%d read pairs), scoring region src/EdgeCalculator.cpp:395-423 of the unmodified reference only, per step" % (what, n_reads)
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic", "config": {"workload": workload_name(args), "sample": sample},
                "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "reference", "sample": sample,
                                 "cpu": cpu_model()},
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
                "setup_s": round(time.time() - t0, 1)}
        emit(line)
        return

    # ------------------------------------------------------------------ our arm
    import torch.distributed as dist
    from haploconduct_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    numa = {"bound": False, "why": "--no-numa-bind"} if args.no_numa_bind else bind_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    t_setup = time.time()
    pr = WT.make_paired_reads(args.pairs, read_len=args.read_len, seed=args.seed, device=str(dev),
                              position_sorted_ids=args.position_sorted_ids, binned_qualities=args.binned_qualities)
    torch.cuda.synchronize()
    log("[rank %d] reads generated in %.1fs" % (rank, time.time() - t_setup))
    rs = pr.readset()
    t1 = time.time()
    store = capi.Store(rs, first_device=local_rank, n_devices=1)
    store_build_s = time.time() - t1
    log("[rank %d] store packed + uploaded in %.1fs (%.2f GB on device, %d quality codes)" %
        (rank, time.time() - t1, store.device_bytes / 1e9, store.quality_alphabet))
    t1 = time.time()
    shard = rank % N_SHARDS
    rec = WT.make_pp_candidates(pr, D=args.partners, shard=shard, n_shards=N_SHARDS, max_cands=args.cands)
    n = rec.shape[0]
    torch.cuda.synchronize()
    log("[rank %d] %d candidates (shard %d/%d) generated in %.1fs" % (rank, n, shard, N_SHARDS, time.time() - t1))
    params = F.make_params(flags=F.FLAG_EXACT_EDGE_SCORES if args.exact_edge_scores else 0, **PARAMS)
    d_edges = torch.empty((n, 48), dtype=torch.uint8, device=dev)
    d_nonedge = torch.empty(n, dtype=torch.int64, device=dev)
    d_counts = torch.zeros(4, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream(dev)

    def step(want_stats=False):
        if args.device_chunk and not want_stats:   # diagnostic: the same work as launches of `device_chunk` candidates
            for i0 in range(0, n, args.device_chunk):
                m = min(args.device_chunk, n - i0)
                store.score_batch_device(local_rank, stream.cuda_stream, params, rec[i0:i0 + m].data_ptr(), m, 0, d_edges.data_ptr(), n,
                                         d_nonedge.data_ptr(), n, d_counts.data_ptr(), False)
            return None
        return store.score_batch_device(local_rank, stream.cuda_stream, params, rec.data_ptr(), n, 0, d_edges.data_ptr(), n,
                                        d_nonedge.data_ptr(), n, d_counts.data_ptr(), want_stats)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # N > 1: the accepted-edge lists of all ranks are concatenated in rank order (= input order) by an NCCL all-gather of the
    # device-resident lists, on a side stream so that the gather of step k runs next to the kernels of step k + 1
    exchange = None
    exchange_kind = None
    if world > 1 and not args.no_exchange:
        from haploconduct_b200 import dist as HD
        step()
        torch.cuda.synchronize()
        cap_t = torch.tensor([int(int(d_counts[0].item()) * 1.02) + 1024], dtype=torch.int64, device=dev)
        dist.all_reduce(cap_t, op=dist.ReduceOp.MAX)      # the lists are padded to ONE length: the longest rank's
        cap_e = int(cap_t.item())
        if args.exchange == "nccl":
            gather, exchange_kind = HD.DeviceGather(48, cap_e, dev), "nccl"
        else:
            gather, exchange_kind = HD.make_device_gather(48, cap_e, dev)
            if args.exchange == "peer" and exchange_kind != "peer":
                raise RuntimeError("--exchange peer: peer memory could not be set up on this box")
        log("[rank %d] accepted-edge gather: %s, lists padded to %d records" % (rank, exchange_kind, cap_e))
        xs = torch.cuda.Stream(dev)
        x_done = torch.cuda.Event()
        k_done = torch.cuda.Event()
        d_edges_x = torch.empty((cap_e, 48), dtype=torch.uint8, device=dev)       # the list being gathered (step k) while step k+1 writes d_edges
        d_cnt_x = torch.zeros(1, dtype=torch.int64, device=dev)

        def exchange():
            stream.wait_event(x_done)                       # the previous gather has read its snapshot
            d_edges_x.copy_(d_edges[:cap_e], non_blocking=True)
            d_cnt_x.copy_(d_counts[:1], non_blocking=True)
            k_done.record(stream)
            with torch.cuda.stream(xs):
                xs.wait_event(k_done)
                gather.gather(d_edges_x, d_cnt_x)
                x_done.record(xs)

    def full_step():
        step()
        if exchange:
            exchange()

    for _ in range(args.warmup):
        full_step()
    if exchange:
        stream.wait_event(x_done)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if args.dma_load:   # diagnostic: the device step while the copy engines move what an e2e step moves (1 GB in, 0.6 GB out)
        s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        h_in = torch.empty(1 << 28, dtype=torch.int32, pin_memory=True); d_in = torch.empty(1 << 28, dtype=torch.int32, device=dev)
        h_out = torch.empty(3 << 26, dtype=torch.int32, pin_memory=True); d_out = torch.empty(3 << 26, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        ci0, ci1, co0, co1 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
        with torch.cuda.stream(s_in):
            ci0.record(s_in)
            for _ in range(args.steps):
                d_in.copy_(h_in, non_blocking=True)
            ci1.record(s_in)
        with torch.cuda.stream(s_out):
            co0.record(s_out)
            for _ in range(args.steps):
                h_out.copy_(d_out, non_blocking=True)
            co1.record(s_out)
    tw0 = time.time()
    e0.record(stream)
    for _ in range(args.steps):
        full_step()
    if exchange:
        stream.wait_event(x_done)                           # the last gather ends inside the timed region
    e1.record(stream)
    barrier()
    tw1 = time.time()
    ms_total = e0.elapsed_time(e1)
    if args.dma_load:
        log("[dma-load] host->device %.1f GB/s, device->host %.1f GB/s while the kernels ran" %
            (args.steps * h_in.numel() * 4 / ci0.elapsed_time(ci1) / 1e6, args.steps * h_out.numel() * 4 / co0.elapsed_time(co1) / 1e6))
    clocks = sampler.stop(tw0, tw1) if rank == 0 else None
    if args.dump_outputs and rank == 0:     # before the legs below reuse d_edges (the exact-scores leg writes other scores)
        dump_outputs(args.dump_outputs, n, d_edges, d_nonedge, d_counts)
    # dominant-kernel duration, measured live with CUDA events around hc_score_kernel on its stream
    kms, stats = [], None
    for _ in range(3):
        stats = step(want_stats=True)
        kms.append(float(stats["score_kernel_ms"]))
    score_ms = float(np.mean(kms))
    counts = d_counts.cpu().numpy()

    # ---- e2e through the host-buffer entry point
    e2e = None
    e2e_pageable = None
    if not args.no_e2e:
        # the host-facing call on the smallest record the reads allow: 12 bytes (idx1, idx2, pos1|pos2|ori|ord) when every
        # position is below 2^14, else the 16-byte compact record (idx1, idx2, pos1|ori|ord, pos2)
        r32 = rec.view(torch.int32).reshape(-1, 8)
        ordc = torch.where(((r32[:, 6] >> 16) & 0xff) == ord("1"), 1, 2)
        runs6 = args.e2e_records == "runs6" and args.read_len < 512 and args.pairs <= (1 << 25) and args.e2e_output == "small"
        if args.e2e_records == "runs6" and not runs6:
            args.e2e_records = "runs"
        short = args.e2e_records in ("short", "runs", "runs6") and args.read_len < (1 << 14)
        use_runs = short and args.e2e_records in ("runs", "runs6")
        rec_bytes = 6 if runs6 else (8 if use_runs else (12 if short else 16))
        cc = torch.empty((n, 2 if use_runs else rec_bytes // 4), dtype=torch.int32, device=dev)
        run_bytes = 0
        if use_runs:
            # run-encoded 8-byte records (hc_score_batch_runs): the list is sorted by (min id, max id), so the candidates of
            # one read-pair form a run; the run holds that read, the record the other one (+ bit 31 when the anchor is ID2)
            i1, i2 = r32[:, 0], r32[:, 1]
            key = torch.minimum(i1, i2)
            first = torch.ones(n, dtype=torch.bool, device=dev)
            first[1:] = key[1:] != key[:-1]
            cut = torch.nonzero(first).flatten()
            h_anchor = torch.empty(len(cut), dtype=torch.int32, pin_memory=True)
            h_anchor.copy_(key[cut])
            h_start = torch.empty(len(cut) + 1, dtype=torch.int64, pin_memory=True)
            h_start[:-1].copy_(cut)
            h_start[-1] = n
            cc[:, 0] = torch.where(i1 == key, i2, i1 | (-(1 << 31)))
            cc[:, 1] = r32[:, 2] | (r32[:, 3] << 14) | (3 << 28) | (ordc << 30).to(torch.int32)
            run_bytes = len(cut) * 4 + (len(cut) + 1) * 4      # what the library sends per step: anchors + relative starts
            del i1, i2, key, first, cut
        else:
            cc[:, 0] = r32[:, 0]; cc[:, 1] = r32[:, 1]
        if use_runs:
            pass
        elif short:
            cc[:, 2] = r32[:, 2] | (r32[:, 3] << 14) | (3 << 28) | (ordc << 30).to(torch.int32)   # POS1 | POS2 | ORI '+','+' | ORD
        else:
            cc[:, 3] = r32[:, 3]
            cc[:, 2] = r32[:, 2] | (3 << 28) | (ordc << 30).to(torch.int32)      # POS1 | ORI1 '+' | ORI2 '+' | ORD
        if runs6:     # the 8-byte entry squeezed into 48 bits: other (25) | anchor-is-ID2 | ORI1 | ORI2 | ORD (2) | POS1 (9) | POS2 (9)
            other = (cc[:, 0] & 0x7fffffff).to(torch.int64)
            role = ((cc[:, 0] >> 31) & 1).to(torch.int64)
            pw = cc[:, 1].to(torch.int64) & 0xffffffff
            v = other | (role << 25) | (((pw >> 28) & 0xf) << 26) | ((pw & 0x3fff) << 30) | (((pw >> 14) & 0x3fff) << 39)
            c6 = v.view(torch.uint8).reshape(n, 8)[:, :6].contiguous()
            if os.environ.get("HC_BENCH_WC"):      # experiment: the records in write-combined pinned memory (the host only writes them)
                h_cand = torch.from_numpy(capi.host_alloc(n * 6, write_combined=True)).reshape(n, 6)
            else:
                h_cand = torch.empty((n, 6), dtype=torch.uint8, pin_memory=True)
            h_cand.copy_(c6)
            del other, role, pw, v, c6
        else:
            h_cand = torch.empty((n, rec_bytes // 4), dtype=torch.int32, pin_memory=True)
            h_cand.copy_(cc)
        del cc
        ne, nn = int(counts[0]), int(counts[1])
        small = use_runs and args.e2e_output == "small"
        erec = (32 if args.exact_edge_scores else 24) if small else 48
        h_edges = torch.empty((max(ne, 1) + 1024, erec), dtype=torch.uint8, pin_memory=True)
        h_nonedge = torch.empty(((n + 63) // 64 + 1) if small else (max(nn, 1) + 1024), dtype=torch.int64, pin_memory=True)
        import ctypes
        L = capi.lib()
        c_ne, c_nn = ctypes.c_uint64(0), ctypes.c_uint64(0)

        def e2e_step():
            if small:     # hc_edge_small records + one bit per candidate
                fn_small = L.hc_score_batch_runs6_small if runs6 else L.hc_score_batch_runs_small
                rc = fn_small(store.handle, params.ctypes.data, h_anchor.data_ptr(), h_start.data_ptr(), h_anchor.shape[0],
                                                 h_cand.data_ptr(), n, h_edges.data_ptr(), h_edges.shape[0], ctypes.byref(c_ne),
                                                 h_nonedge.data_ptr(), ctypes.byref(c_nn), None)
                if rc != 0:
                    raise RuntimeError(capi.last_error())
                return
            if use_runs:
                ecap, ncap = (0, 0) if args.e2e_no_output else (h_edges.shape[0], h_nonedge.shape[0])
                rc = L.hc_score_batch_runs(store.handle, params.ctypes.data, h_anchor.data_ptr(), h_start.data_ptr(), h_anchor.shape[0],
                                           h_cand.data_ptr(), n, None, h_edges.data_ptr(), ecap, ctypes.byref(c_ne),
                                           h_nonedge.data_ptr(), ncap, ctypes.byref(c_nn), None)
                if rc != 0 and not (args.e2e_no_output and rc == -5):
                    raise RuntimeError(capi.last_error())
                return
            fn = L.hc_score_batch_short if short else L.hc_score_batch_compact
            rc = fn(store.handle, params.ctypes.data, h_cand.data_ptr(), n, None, h_edges.data_ptr(),
                                  h_edges.shape[0], ctypes.byref(c_ne), h_nonedge.data_ptr(), h_nonedge.shape[0],
                                  ctypes.byref(c_nn), None)
            if rc != 0:
                raise RuntimeError(capi.last_error())

        for _ in range(max(args.warmup, 3)):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()
        barrier()
        e2e_ms = 1e3 * (time.perf_counter() - t0) / args.steps
        assert c_ne.value == ne and c_nn.value == nn
        # the same call on PAGEABLE buffers (what a std::vector / numpy caller hands over): the library stages the records
        # through its ring of pinned buffers; reported next to the pinned number
        e2e_pageable = None
        if small and not os.environ.get("HC_BENCH_WC"):   # (the leg copies the records back out of h_cand: not out of write-combined memory)
            try:
                p_cand = np.empty(h_cand.shape, dtype=np.uint8 if runs6 else np.int32)
                p_cand[...] = h_cand.numpy()
                p_edges = np.empty(h_edges.shape, dtype=np.uint8)
                p_bits = np.empty(h_nonedge.shape, dtype=np.int64)
                p_anchor, p_start = h_anchor.numpy().copy(), h_start.numpy().copy()

                def pg_step():
                    rc = fn_small(store.handle, params.ctypes.data, p_anchor.ctypes.data, p_start.ctypes.data, p_anchor.shape[0], p_cand.ctypes.data, n,
                                  p_edges.ctypes.data, p_edges.shape[0], ctypes.byref(c_ne), p_bits.ctypes.data, ctypes.byref(c_nn), None)
                    if rc != 0:
                        raise RuntimeError(capi.last_error())
                fn_small = L.hc_score_batch_runs6_small if runs6 else L.hc_score_batch_runs_small
                for _ in range(2):
                    pg_step()
                barrier()
                tp0 = time.perf_counter()
                for _ in range(3):
                    pg_step()
                barrier()
                pg_ms = 1e3 * (time.perf_counter() - tp0) / 3
                assert c_ne.value == ne and c_nn.value == nn and p_edges[:ne].tobytes() == h_edges[:ne].numpy().tobytes()
                e2e_pageable = {"ms_per_step": pg_ms, "value_per_gpu": n / (pg_ms * 1e-3), "unit": UNIT,
                                "note": "same call, pageable host buffers (numpy): records and results staged through the library's ring of pinned buffers by up to 16 of the %d host threads" % (os.cpu_count() or 1)}
                del p_cand, p_edges, p_bits
            except Exception as ex:
                e2e_pageable = {"failed": repr(ex)}
        if small:      # the bit map really says what the index list says
            bits = h_nonedge[: (n + 63) // 64].numpy().view(np.uint8)
            assert int(np.unpackbits(bits).sum()) == nn
        e2e = (e2e_ms, n * rec_bytes + run_bytes, (ne * erec + ((n + 63) // 64) * 8 + 64) if small else (ne * 48 + nn * 8 + 64),
               ("hc_candidate_entry6 (6 B, run-encoded)" if runs6 else "hc_candidate_entry (8 B, run-encoded)" if use_runs else ("hc_candidate_short (12 B)" if short else "hc_candidate_compact (16 B)"))
               + (" in; hc_edge_small (%d B) + 1 bit per candidate out" % erec if small else " in; hc_edge (48 B) + 8-byte non-edge indices out"))

    # the mode the drop-in host mirror runs in (HC_FLAG_EXACT_EDGE_SCORES: every accepted edge re-summed in the reference's
    # order), as an extra number next to the default line
    exact_ms = None
    if not args.exact_edge_scores:
        px = F.make_params(flags=F.FLAG_EXACT_EDGE_SCORES, **PARAMS)
        for _ in range(2):
            store.score_batch_device(local_rank, stream.cuda_stream, px, rec.data_ptr(), n, 0, d_edges.data_ptr(), n, d_nonedge.data_ptr(), n,
                                     d_counts.data_ptr(), False)
        x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        x0.record(stream)
        for _ in range(3):
            store.score_batch_device(local_rank, stream.cuda_stream, px, rec.data_ptr(), n, 0, d_edges.data_ptr(), n, d_nonedge.data_ptr(), n,
                                     d_counts.data_ptr(), False)
        x1.record(stream)
        torch.cuda.synchronize()
        exact_ms = x0.elapsed_time(x1) / 3

    ms_step = ms_total / args.steps
    tvals = torch.tensor([ms_step, e2e[0] if e2e else 0.0], dtype=torch.float64, device=dev)
    tot = torch.tensor([n], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(tvals, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_step, e2e_ms = float(tvals[0]), float(tvals[1])
    total_cands = int(tot[0])

    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        alg = int(stats["algorithmic_bytes"])
        achieved = alg / (score_ms * 1e-3) / 1e9
        default_cfg = args.pairs == 10_000_000 and args.read_len == 150 and args.partners == 140 and not args.position_sorted_ids and not args.binned_qualities
        traffic, traffic_src = measured_traffic(n, default_cfg)
        line = {
            "metric": METRIC, "value": total_cands / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32 fixed-point (2^-22) sums + f64 reference-order pass at threshold boundaries", "data": "synthetic",
            "config": {"workload": workload_name(args), "l2": "inputs larger than L2: %.1f GB candidate stream + %.1f GB read store "
                       "per step, no flush needed" % (n * 32 / 1e9, store.device_bytes / 1e9),
                       "params": PARAMS, "candidates_per_gpu": n, "seed": args.seed},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "kernel": "hc_score_kernel", "kernel_ms": score_ms,
                         "algorithmic_bytes_per_launch": alg, "peak_source": peak_src,
                         "positions_per_launch": int(stats["n_positions"]), "all_kernels_ms": float(stats["kernel_ms"])},
            "gpu_launches": int(stats["kernel_launches"]) * args.steps,
            "clocks": clocks,
            "results": {"edges": int(counts[0]), "nonedges": int(counts[1]), "reference_order_pass": int(counts[2])},
            "exchange": ((("one-sided puts over NVLink peer memory (copy engines; device-side barriers before and after) of every rank's accepted "
                           "edges into every peer's buffer" if exchange_kind == "peer" else
                           "NCCL all-gather (counts, then lists padded to the longest) of every rank's accepted edges") +
                          ", 48-byte records, inside the timed region on a side stream; rank order = input order") if exchange else
                         ("none (one rank)" if world == 1 else "left out (--no-exchange)")),
            "exact_edge_scores": (None if exact_ms is None else {"ms_per_step": exact_ms, "value": n / (exact_ms * 1e-3), "unit": UNIT + " per GPU",
                                                                 "note": "HC_FLAG_EXACT_EDGE_SCORES: the mode of the drop-in host mirror"}),
            "numa": numa,
            "setup_s": round(time.time() - t_setup, 1), "store_build_s": round(store_build_s, 2),
        }
        if e2e:
            line["e2e"] = {"value": total_cands / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": e2e[1],
                           "d2h_bytes_per_step": e2e[2], "ms_per_step": e2e_ms, "records": e2e[3]}
        if e2e and e2e_pageable is not None:
            line["e2e"]["pageable"] = e2e_pageable
        if world == 1 and not args.no_cpu:
            try:
                cs = WT.candidates_as_numpy(rec[: args.cpu_sample])
                threads = os.cpu_count() or 1
                out, n_reads = run_cpu_reference(pr.bases.numpy(), pr.quals.numpy(), args.read_len, cs, 3, threads)
                t = float(np.mean(out["rep_times_s"][1:]))
                t1 = None
                try:
                    out1, _ = run_cpu_reference(pr.bases.numpy(), pr.quals.numpy(), args.read_len, cs[: max(len(cs) // 16, 1)], 1, 1)
                    t1 = (max(len(cs) // 16, 1)) / float(out1["rep_times_s"][0])
                except Exception:
                    pass
                line["cpu_baseline"] = {"value": len(cs) / t, "unit": UNIT, "cores": threads, "kind": "reference",
                                        "sample": "first %d candidates of this rank's shard (%d read pairs), 3 repetitions of the "
                                                  "OpenMP scoring region src/EdgeCalculator.cpp:395-423 of the unmodified reference"
                                                  % (len(cs), n_reads), "one_thread_value": t1, "cpu": cpu_model()}
            except Exception as ex:   # the baseline is a reported number, never a reason to lose the GPU line
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": "failed: %r" % (ex,)}
        if world == 1 and not args.no_cpu and not args.no_pipeline:
            # files in -> overlap graph out through the reference's own interface (construct_edges of the unmodified reference on
            # all host threads next to the host mirror over the C ABI, same files, graphs compared): tools/bench_pipeline.py
            try:
                import subprocess
                pr_out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_pipeline.py"), "--pairs", "300000", "--partners", "20",
                                         "--one-thread-limit", "0", "--skip-host-parsers"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                                        text=True, timeout=300).stdout
                pj = json.loads([l for l in pr_out.split("\n") if l.startswith("{")][-1])
                m, r, b = pj.get("mirror_device_ingest", {}), pj.get("reference", {}), pj.get("breakdown", {})
                line["files_to_graph"] = {
                    "workload": "%d read pairs, %d candidates, %.0f MB overlaps file + FASTQ files on disk" % (pj["pairs"], pj["candidates"], pj["overlaps_file_bytes"] / 1e6),
                    "reference_construct_edges_s": r.get("t_construct_edges_s"), "reference_threads": r.get("threads"), "reference_wall_s": r.get("wall_s"),
                    "mirror_construct_edges_s": m.get("t_construct_edges_s"), "mirror_wall_s": m.get("wall_s"), "mirror_cuda_context_s": m.get("t_cuda_init_s"),
                    "speedup_construct_edges": b.get("speedup_construct_edges_vs_reference"), "speedup_wall": b.get("speedup_wall_vs_reference"),
                    "same_edges_as_reference": m.get("same_edges_as_reference"), "mirror_phases_s": b.get("phases_s")}
            except Exception as ex:
                line["files_to_graph"] = {"failed": repr(ex)[:200]}
        emit(line)
    store.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
