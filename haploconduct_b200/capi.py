"""ctypes binding of the C ABI in include/hc_b200.h (haploconduct_b200/lib/libhc_b200.so).

The binding is deliberately thin: every call goes through the exported ``extern "C"`` symbols, the
same ones a cgo/JNI/C++ host would bind.  There is no Python or CPU fallback: if the shared
library is missing or no sm_100 device is present the calls raise.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional, Tuple

import numpy as np

from . import formats as F

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HC_B200_LIB") or os.path.join(HERE, "lib", "libhc_b200.so")   # override: kernel experiments only

# every symbol include/hc_b200.h declares
EXPORTED = [
    "hc_store_create", "hc_store_destroy", "hc_store_n_reads", "hc_store_n_single", "hc_store_n_devices",
    "hc_store_device_bytes", "hc_store_quality_alphabet", "hc_score_batch", "hc_score_batch_compact", "hc_score_batch_short", "hc_score_batch_runs", "hc_score_batch_runs_small", "hc_score_batch_runs6_small", "hc_score_batch_short_small", "hc_edge_extra_pos", "hc_score_batch_device",
    "hc_overlap_score", "hc_overlap_score_multi",
    "hc_phred_to_prob", "hc_exp_threshold", "hc_device_count", "hc_warm_up", "hc_last_error", "hc_version", "hc_fno1", "hc_fno3", "hc_fno1_small", "hc_fno3_small", "hc_fno1_text", "hc_fno3_text", "hc_build_adjacency", "hc_subread_info", "hc_host_alloc", "hc_host_free",
    "hc_store_create_fastq", "hc_store_create_fastq_files", "hc_store_read_ids", "hc_consensus", "hc_dedup_edges", "hc_idmap_create", "hc_idmap_destroy", "hc_ingest_overlaps", "hc_ingest_overlaps_device",
    "hc_ingest_score_overlaps", "hc_fno1_text_nonedges",
]

_lib: Optional[ctypes.CDLL] = None


class HcError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("hc_b200 error %d: %s" % (code, msg))
        self.code = code


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "%s is missing: build it with `python -m haploconduct_b200.build` (there is no CPU fallback)" % LIB_PATH
            )
        L = ctypes.CDLL(LIB_PATH)
        vp, u64, i32, u32, dbl = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int, ctypes.c_uint32, ctypes.c_double
        L.hc_store_create.restype = vp
        L.hc_store_create.argtypes = [vp, u64, u64, vp, vp, i32, i32]
        L.hc_store_create_fastq.restype = vp
        L.hc_store_create_fastq.argtypes = [vp, u64, vp, u64, vp, u64, u64, i32, i32]
        L.hc_store_create_fastq_files.restype = vp
        L.hc_store_create_fastq_files.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, u64, i32, i32]
        L.hc_store_read_ids.restype = i32
        L.hc_store_read_ids.argtypes = [vp, vp, vp]
        L.hc_consensus.restype = i32
        L.hc_consensus.argtypes = [vp, vp, u64, vp, u64, u32, dbl, vp, vp, u64, vp]
        L.hc_store_destroy.restype = None
        L.hc_store_destroy.argtypes = [vp]
        for name in ("hc_store_n_reads", "hc_store_n_single", "hc_store_device_bytes"):
            getattr(L, name).restype = u64
            getattr(L, name).argtypes = [vp]
        for name in ("hc_store_n_devices", "hc_store_quality_alphabet"):
            getattr(L, name).restype = i32
            getattr(L, name).argtypes = [vp]
        L.hc_score_batch.restype = i32
        L.hc_score_batch.argtypes = [vp, vp, vp, u64, vp, vp, u64, vp, vp, u64, vp, vp]
        L.hc_score_batch_compact.restype = i32
        L.hc_score_batch_compact.argtypes = [vp, vp, vp, u64, vp, vp, u64, vp, vp, u64, vp, vp]
        L.hc_score_batch_short.restype = i32
        L.hc_score_batch_short.argtypes = [vp, vp, vp, u64, vp, vp, u64, vp, vp, u64, vp, vp]
        L.hc_score_batch_runs.restype = i32
        L.hc_score_batch_runs.argtypes = [vp, vp, vp, vp, u64, vp, u64, vp, vp, u64, vp, vp, u64, vp, vp]
        L.hc_score_batch_runs_small.restype = i32
        L.hc_score_batch_runs_small.argtypes = [vp, vp, vp, vp, u64, vp, u64, vp, u64, vp, vp, vp, vp]
        L.hc_score_batch_runs6_small.restype = i32
        L.hc_score_batch_runs6_small.argtypes = [vp, vp, vp, vp, u64, vp, u64, vp, u64, vp, vp, vp, vp]
        L.hc_score_batch_short_small.restype = i32
        L.hc_score_batch_short_small.argtypes = [vp, vp, vp, u64, vp, u64, vp, vp, vp, vp]
        L.hc_edge_extra_pos.restype = None
        L.hc_edge_extra_pos.argtypes = [u32, u32, ctypes.c_char, u32, u32, u32, u32, vp, vp]
        L.hc_score_batch_device.restype = i32
        L.hc_score_batch_device.argtypes = [vp, i32, vp, vp, vp, u64, vp, vp, u64, vp, u64, vp, vp]
        L.hc_overlap_score.restype = dbl
        L.hc_overlap_score.argtypes = [ctypes.c_char_p, u32, ctypes.c_char_p, u32, ctypes.c_char_p, ctypes.c_char_p, u32, vp,
                                       ctypes.POINTER(dbl)]
        L.hc_overlap_score_multi.restype = i32
        L.hc_overlap_score_multi.argtypes = [ctypes.c_char_p, u32, ctypes.c_char_p, u32, ctypes.c_char_p, ctypes.c_char_p, vp, u32, vp,
                                             vp, vp, vp]
        L.hc_phred_to_prob.restype = dbl
        L.hc_phred_to_prob.argtypes = [i32]
        L.hc_exp_threshold.restype = dbl
        L.hc_exp_threshold.argtypes = [dbl]
        L.hc_device_count.restype = i32
        L.hc_device_count.argtypes = []
        L.hc_fno1.restype = i32
        L.hc_fno1.argtypes = [vp, vp, u64, vp, u64, ctypes.POINTER(u64), i32]
        L.hc_fno3.restype = i32
        L.hc_fno3.argtypes = [u64, vp, vp, vp, u64, vp, i32, vp, u64, ctypes.POINTER(u64), i32]
        L.hc_build_adjacency.restype = i32
        L.hc_build_adjacency.argtypes = [vp, u64, vp, u64, i32, vp, vp, vp, vp, vp, ctypes.POINTER(u64), i32]
        L.hc_host_alloc.restype = vp
        L.hc_host_alloc.argtypes = [u64, i32]
        L.hc_host_free.restype = None
        L.hc_host_free.argtypes = [vp]
        L.hc_subread_info.restype = i32
        L.hc_subread_info.argtypes = [vp, u64, vp, vp, u64, vp, vp, i32]
        L.hc_fno1_small.restype = i32
        L.hc_fno1_small.argtypes = L.hc_fno1.argtypes
        L.hc_fno3_small.restype = i32
        L.hc_fno3_small.argtypes = L.hc_fno3.argtypes
        L.hc_fno1_text.restype = i32
        L.hc_fno1_text.argtypes = [vp, vp, u64, vp, u64, ctypes.POINTER(u64), ctypes.POINTER(u64), ctypes.POINTER(u64), i32]
        L.hc_fno3_text.restype = i32
        L.hc_fno3_text.argtypes = [u64, vp, vp, vp, u64, vp, i32, vp, u64, ctypes.POINTER(u64), ctypes.POINTER(u64), i32]
        L.hc_dedup_edges.restype = i32
        L.hc_dedup_edges.argtypes = [vp, u64, i32, vp, vp, u64, vp, i32]
        L.hc_idmap_create.restype = vp
        L.hc_idmap_create.argtypes = [vp, u64, i32]
        L.hc_idmap_destroy.restype = None
        L.hc_idmap_destroy.argtypes = [vp]
        L.hc_ingest_overlaps.restype = i32
        L.hc_ingest_overlaps.argtypes = [vp, vp, u64, vp, vp, vp, u64, vp, vp, u64, vp]
        L.hc_ingest_overlaps_device.restype = i32
        L.hc_ingest_overlaps_device.argtypes = [vp, vp, vp, u64, vp, vp, vp, u64, vp, vp, u64, vp]
        L.hc_ingest_score_overlaps.restype = i32
        L.hc_ingest_score_overlaps.argtypes = [vp, vp, vp, u64, vp, vp, vp, vp, vp, u64, vp, u64, vp, vp, u64, vp]
        L.hc_fno1_text_nonedges.restype = i32
        L.hc_fno1_text_nonedges.argtypes = [vp, vp, vp, u64, u64, vp, u64, vp, u64, vp, u64, ctypes.POINTER(u64), ctypes.POINTER(u64),
                                            ctypes.POINTER(u64), vp, i32]
        L.hc_last_error.restype = ctypes.c_char_p
        L.hc_version.restype = ctypes.c_char_p
        _lib = L
    return _lib


def last_error() -> str:
    return lib().hc_last_error().decode()


def _check(rc: int) -> None:
    if rc != 0:
        raise HcError(rc, last_error())


class Store:
    """Device-resident read store (hc_store_create / hc_store_destroy)."""

    def __init__(self, rs: F.ReadSet, first_device: int = 0, n_devices: int = 1):
        L = lib()
        descs = np.ascontiguousarray(rs.descs)
        self._h = L.hc_store_create(descs.ctypes.data, rs.n_reads, rs.n_single, rs.bases.ctypes.data, rs.quals.ctypes.data,
                                    first_device, n_devices)
        if not self._h:
            raise HcError(-1, last_error())
        self.first_device = first_device
        self.n_devices = n_devices

    @classmethod
    def from_fastq(cls, singles: bytes = b"", paired1: bytes = b"", paired2: bytes = b"", max_reads: int = 2 ** 62,
                   first_device: int = 0, n_devices: int = 1) -> "Store":
        """hc_store_create_fastq: the store straight from the text of the FASTQ files."""
        L = lib()
        bufs = [np.frombuffer(t, dtype=np.uint8) if len(t) else None for t in (singles, paired1, paired2)]
        self = cls.__new__(cls)
        self._h = L.hc_store_create_fastq(*[x for b in bufs for x in ((b.ctypes.data, len(b)) if b is not None else (None, 0))],
                                          max_reads, first_device, n_devices)
        if not self._h:
            raise HcError(-4, last_error())
        self.first_device, self.n_devices = first_device, n_devices
        return self

    @classmethod
    def from_fastq_files(cls, singles: Optional[str] = None, paired1: Optional[str] = None, paired2: Optional[str] = None,
                         max_reads: int = 2 ** 62, first_device: int = 0, n_devices: int = 1) -> "Store":
        """hc_store_create_fastq_files: the store from the FASTQ files themselves, streamed to the device."""
        L = lib()
        self = cls.__new__(cls)
        enc = [p.encode() if p else None for p in (singles, paired1, paired2)]
        self._h = L.hc_store_create_fastq_files(enc[0], enc[1], enc[2], max_reads, first_device, n_devices)
        if not self._h:
            raise HcError(-4, last_error())
        self.first_device, self.n_devices = first_device, n_devices
        return self

    def consensus(self, problems, min_clique_size: int, min_qual: float):
        """hc_consensus on a list of problem dicts (formats.consensus_arrays).  Returns [(ret, cons_seq, cons_qual)]."""
        P, S = F.consensus_arrays(problems)
        total = int(P["total_len"].sum()) if len(P) else 0
        cs = np.zeros(max(total, 1), dtype=np.uint8)
        cq = np.zeros(max(total, 1), dtype=np.uint8)
        res = np.zeros(max(len(P), 1), dtype=F.CONS_RESULT)
        _check(lib().hc_consensus(self._h, P.ctypes.data if len(P) else None, len(P), S.ctypes.data if len(S) else None, len(S),
                                  min_clique_size, min_qual, cs.ctypes.data, cq.ctypes.data, total, res.ctypes.data))
        out = []
        for i in range(len(P)):
            o, n = int(P[i]["out_offset"]), int(res[i]["length"])
            out.append((int(res[i]["ret"]), cs[o:o + n].tobytes().decode(), cq[o:o + n].tobytes().decode()))
        return out

    def read_ids(self):
        """(ids, mate lengths [n, 2]) of a store built from FASTQ text."""
        n = int(lib().hc_store_n_reads(self._h))
        ids = np.zeros(n, dtype=np.uint64)
        lens = np.zeros((n, 2), dtype=np.uint32)
        _check(lib().hc_store_read_ids(self._h, ids.ctypes.data, lens.ctypes.data))
        return ids, lens

    @property
    def handle(self):
        return self._h

    def close(self) -> None:
        if getattr(self, "_h", None):
            lib().hc_store_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def device_bytes(self) -> int:
        return int(lib().hc_store_device_bytes(self._h))

    @property
    def quality_alphabet(self) -> int:
        return int(lib().hc_store_quality_alphabet(self._h))

    def score_batch(self, params: np.ndarray, cands: np.ndarray, per_candidate: bool = True, edges_cap: Optional[int] = None,
                    nonedge_cap: Optional[int] = None, compact: bool = False):
        """hc_score_batch on HOST buffers; compact=True -> hc_score_batch_compact (16-byte records), compact="short" ->
        hc_score_batch_short (12-byte records), compact="runs" -> hc_score_batch_runs (run-encoded 8-byte records).
        Returns (edges, nonedge_idx, per_cand or None, stats)."""
        L = lib()
        if compact == "runs":
            anchor, start, entries = F.run_encode(cands)
            n = len(entries)
            ecap = n if edges_cap is None else edges_cap
            ncap = n if nonedge_cap is None else nonedge_cap
            edges = np.zeros(max(ecap, 1), dtype=F.EDGE)
            nonedge = np.zeros(max(ncap, 1), dtype=np.uint64)
            per = np.zeros(n, dtype=F.RESULT) if per_candidate else None
            ne, nn = ctypes.c_uint64(0), ctypes.c_uint64(0)
            stats = np.zeros(1, dtype=F.BATCH_STATS)
            rc = L.hc_score_batch_runs(self._h, params.ctypes.data, anchor.ctypes.data if n else None, start.ctypes.data, len(anchor),
                                       entries.ctypes.data if n else None, n, per.ctypes.data if per is not None and n else None,
                                       edges.ctypes.data, ecap, ctypes.byref(ne), nonedge.ctypes.data, ncap, ctypes.byref(nn),
                                       stats.ctypes.data)
            if rc != 0:
                err = HcError(rc, last_error())
                err.required = (int(ne.value), int(nn.value))
                raise err
            return edges[: ne.value], nonedge[: nn.value], per, stats[0]
        if compact == "short":
            cands = F.short_candidates(cands)
        elif compact:
            cands = F.compact_candidates(cands)
        cands = np.ascontiguousarray(cands)
        n = len(cands)
        ecap = n if edges_cap is None else edges_cap
        ncap = n if nonedge_cap is None else nonedge_cap
        edges = np.zeros(max(ecap, 1), dtype=F.EDGE)
        nonedge = np.zeros(max(ncap, 1), dtype=np.uint64)
        per = np.zeros(n, dtype=F.RESULT) if per_candidate else None
        ne, nn = ctypes.c_uint64(0), ctypes.c_uint64(0)
        stats = np.zeros(1, dtype=F.BATCH_STATS)
        fn = L.hc_score_batch_short if compact == "short" else (L.hc_score_batch_compact if compact else L.hc_score_batch)
        rc = fn(self._h, params.ctypes.data, cands.ctypes.data if n else None, n,
                              per.ctypes.data if per is not None and n else None, edges.ctypes.data, ecap, ctypes.byref(ne),
                              nonedge.ctypes.data, ncap, ctypes.byref(nn), stats.ctypes.data)
        if rc != 0:
            err = HcError(rc, last_error())
            err.required = (int(ne.value), int(nn.value))
            raise err
        return edges[: ne.value], nonedge[: nn.value], per, stats[0]

    def score_batch_small(self, params: np.ndarray, cands: np.ndarray, runs: bool = True, edges_cap: Optional[int] = None):
        """hc_score_batch_runs_small / hc_score_batch_short_small: small outputs.  Returns (edges as EDGE_SMALL or
        EDGE_SMALL_EXACT records, non-edge flags as a bool array over the candidates, stats)."""
        L = lib()
        exact = bool(int(params["flags"][0]) & F.FLAG_EXACT_EDGE_SCORES)
        dt = F.EDGE_SMALL_EXACT if exact else F.EDGE_SMALL
        ne, nn = ctypes.c_uint64(0), ctypes.c_uint64(0)
        stats = np.zeros(1, dtype=F.BATCH_STATS)
        if runs:
            anchor, start, entries = F.run_encode(cands)
            n = len(entries)
            if runs == 6:
                entries = F.entries6(entries)
        else:
            entries = np.ascontiguousarray(F.short_candidates(cands))
            n = len(entries)
        ecap = n if edges_cap is None else edges_cap
        edges = np.zeros(max(ecap, 1), dtype=dt)
        bits = np.full((n + 63) // 64 + 1, 0xdeadbeefdeadbeef, dtype=np.uint64)     # the call must write every word it owns
        if runs == 6:
            rc = L.hc_score_batch_runs6_small(self._h, params.ctypes.data, anchor.ctypes.data if n else None, start.ctypes.data, len(anchor),
                                              entries.ctypes.data if n else None, n, edges.ctypes.data, ecap, ctypes.byref(ne),
                                              bits.ctypes.data, ctypes.byref(nn), stats.ctypes.data)
        elif runs:
            rc = L.hc_score_batch_runs_small(self._h, params.ctypes.data, anchor.ctypes.data if n else None, start.ctypes.data, len(anchor),
                                             entries.ctypes.data if n else None, n, edges.ctypes.data, ecap, ctypes.byref(ne),
                                             bits.ctypes.data, ctypes.byref(nn), stats.ctypes.data)
        else:
            rc = L.hc_score_batch_short_small(self._h, params.ctypes.data, entries.ctypes.data if n else None, n, edges.ctypes.data, ecap,
                                              ctypes.byref(ne), bits.ctypes.data, ctypes.byref(nn), stats.ctypes.data)
        if rc != 0:
            err = HcError(rc, last_error())
            err.required = (int(ne.value), int(nn.value))
            raise err
        flags = np.unpackbits(bits[: (n + 63) // 64].view(np.uint8), bitorder="little")[:n].astype(bool)
        assert int(flags.sum()) == int(nn.value)
        return edges[: ne.value], flags, stats[0]

    def ingest_score(self, idmap: "IdMap", text, ingest_params: np.ndarray, params: np.ndarray, kept_cap: Optional[int] = None,
                     edges_cap: Optional[int] = None, filtered_cap: Optional[int] = None):
        """hc_ingest_score_overlaps: overlaps-file text (bytes or a uint8 array, e.g. from host_alloc) parsed and scored on
        the id map's device.  Returns (kept CANDIDATE records, their line numbers, their classes, edges as EDGE_SMALL or
        EDGE_SMALL_EXACT records whose `cand` indexes kept, filtered OVERLAP_REC records, their line numbers, stats)."""
        buf = text if isinstance(text, np.ndarray) else (np.frombuffer(text, dtype=np.uint8) if len(text) else np.zeros(0, dtype=np.uint8))
        exact = bool(int(params["flags"][0]) & F.FLAG_EXACT_EDGE_SCORES)
        guess = int(np.count_nonzero(buf == 10)) + 1
        kcap = guess if kept_cap is None else kept_cap
        ecap = guess if edges_cap is None else edges_cap
        fcap = guess if filtered_cap is None else filtered_cap
        kept = np.zeros(max(kcap, 1), dtype=F.CANDIDATE)
        kl = np.zeros(max(kcap, 1), dtype=np.uint64)
        kc = np.zeros(max(kcap, 1), dtype=np.uint8)
        edges = np.zeros(max(ecap, 1), dtype=F.EDGE_SMALL_EXACT if exact else F.EDGE_SMALL)
        filt = np.zeros(max(fcap, 1), dtype=F.OVERLAP_REC)
        fl = np.zeros(max(fcap, 1), dtype=np.uint64)
        st = np.zeros(1, dtype=F.INGEST_SCORE_STATS)
        rc = lib().hc_ingest_score_overlaps(self._h, idmap.handle, buf.ctypes.data if len(buf) else None, len(buf),
                                            ingest_params.ctypes.data, params.ctypes.data, kept.ctypes.data, kl.ctypes.data,
                                            kc.ctypes.data, kcap, edges.ctypes.data, ecap, filt.ctypes.data, fl.ctypes.data, fcap,
                                            st.ctypes.data)
        s = st[0]
        if rc != 0:
            err = HcError(rc, last_error())
            err.required = (int(s["n_kept"]), int(s["score"]["n_edges"]), int(s["ingest"]["n_filtered"]))
            raise err
        nk, ne, nf = int(s["n_kept"]), int(s["score"]["n_edges"]), int(s["ingest"]["n_filtered"])
        return kept[:nk], kl[:nk], kc[:nk], edges[:ne], filt[:nf], fl[:nf], s

    def score_batch_device(self, device: int, stream: int, params: np.ndarray, d_cand: int, n: int, d_per_cand: int,
                           d_edges: int, edges_cap: int, d_nonedge: int, nonedge_cap: int, d_counts: int, want_stats: bool):
        """hc_score_batch_device on raw DEVICE pointers (e.g. torch tensors' data_ptr())."""
        stats = np.zeros(1, dtype=F.BATCH_STATS) if want_stats else None
        rc = lib().hc_score_batch_device(self._h, device, stream or None, params.ctypes.data, d_cand or None, n,
                                         d_per_cand or None, d_edges, edges_cap, d_nonedge, nonedge_cap, d_counts,
                                         stats.ctypes.data if want_stats else None)
        _check(rc)
        return stats[0] if want_stats else None


def overlap_score(seq1: str, seq2: str, q1: str, q2: str, pos: int, params: np.ndarray) -> Tuple[float, float]:
    mm = ctypes.c_double(0)
    s = lib().hc_overlap_score(seq1.encode(), len(seq1), seq2.encode(), len(seq2), q1.encode(), q2.encode(), pos,
                               params.ctypes.data, ctypes.byref(mm))
    if s < 0:
        raise HcError(-1, last_error())
    return s, mm.value


def overlap_score_multi(seq1: str, seq2: str, q1: str, q2: str, pos, params: np.ndarray):
    """hc_overlap_score_multi: (scores, mismatch_rates, above_threshold) for many start positions."""
    pos = np.ascontiguousarray(pos, dtype=np.uint32)
    sc = np.zeros(len(pos)); mm = np.zeros(len(pos)); ab = np.zeros(len(pos), dtype=np.uint8)
    _check(lib().hc_overlap_score_multi(seq1.encode(), len(seq1), seq2.encode(), len(seq2), q1.encode(), q2.encode(),
                                        pos.ctypes.data, len(pos), params.ctypes.data, sc.ctypes.data, mm.ctypes.data, ab.ctypes.data))
    return sc, mm, ab.astype(bool)


def phred_to_prob(q: int) -> float:
    return lib().hc_phred_to_prob(q)


def exp_threshold(thr: float) -> float:
    return lib().hc_exp_threshold(thr)


def device_count() -> int:
    return lib().hc_device_count()


class _FnoInputC(ctypes.Structure):     # hc_fno_input
    _fields_ = [("n_vertices", ctypes.c_uint64), ("visited", ctypes.c_void_p), ("label", ctypes.c_void_p),
                ("vertex_read", ctypes.c_void_p), ("sr_off", ctypes.c_void_p), ("sr_idx", ctypes.c_void_p),
                ("sr_sub", ctypes.c_void_p), ("n_superreads", ctypes.c_uint64), ("superread", ctypes.c_void_p),
                ("resolve_orientations", ctypes.c_uint8), ("no_inclusions", ctypes.c_uint8)]


FNO_OVERLAP_SMALL = np.dtype([("id1", "<u4"), ("id2", "<u4"), ("pos1_perc", "<u4"), ("pos2_perc2", "<u4"), ("len1_flags", "<u4"),
                              ("len2", "<u4")])     # hc_fno_overlap_small, 24 bytes


def fno_small_to_overlaps(r: np.ndarray) -> np.ndarray:
    """hc_fno_overlap_small records -> formats.FNO_OVERLAP (what hc_fno1 / hc_fno3 return)."""
    o = np.zeros(len(r), dtype=F.FNO_OVERLAP)
    fl = r["len1_flags"] >> 24
    o["id1"], o["id2"] = r["id1"], r["id2"]
    o["pos1"], o["perc"] = r["pos1_perc"] & 0xffffff, r["pos1_perc"] >> 24
    o["pos2"], o["perc2"] = r["pos2_perc2"] & 0xffffff, r["pos2_perc2"] >> 24
    o["len1"], o["len2"] = r["len1_flags"] & 0xffffff, r["len2"] & 0xffffff
    o["ord"] = np.where((fl & 3) == 1, ord("1"), np.where((fl & 3) == 2, ord("2"), ord("-")))
    o["ori1"] = np.where(fl & 4, ord("+"), ord("-"))
    o["ori2"] = np.where(fl & 8, ord("+"), ord("-"))
    o["type1"] = np.where(fl & 16, ord("p"), ord("s"))
    o["type2"] = np.where(fl & 32, ord("p"), ord("s"))
    return o


def _fno_input_c(fi: "F.FnoInput"):
    """hc_fno_input for fi, and the arrays it points into (keep them alive while it is used)."""
    keep = [np.ascontiguousarray(a) for a in (fi.visited, fi.label, fi.vertex_read, fi.sr_off, fi.sr_idx, fi.sr_sub, fi.superread)]
    st = _FnoInputC(len(fi.visited), keep[0].ctypes.data, keep[1].ctypes.data, keep[2].ctypes.data, keep[3].ctypes.data,
                    keep[4].ctypes.data, keep[5].ctypes.data, len(fi.superread), keep[6].ctypes.data, fi.resolve_orientations,
                    fi.no_inclusions)
    return st, keep


def fno1(fi: "F.FnoInput", device: int = 0, small: bool = False) -> np.ndarray:
    """hc_fno1 (small: hc_fno1_small, decoded): next-iteration overlaps derived on the GPU, in processing order
    (formats.FNO_OVERLAP)."""
    st, keep = _fno_input_c(fi)
    edges = np.ascontiguousarray(fi.edges)
    cap = max(2 * len(edges), 1024)
    fn = lib().hc_fno1_small if small else lib().hc_fno1
    while True:
        out = np.zeros(cap, dtype=FNO_OVERLAP_SMALL if small else F.FNO_OVERLAP)
        n = ctypes.c_uint64(0)
        rc = fn(ctypes.byref(st), edges.ctypes.data if len(edges) else None, len(edges), out.ctypes.data, cap, ctypes.byref(n), device)
        if rc == 0:
            return fno_small_to_overlaps(out[: n.value]) if small else out[: n.value]
        if rc != -5:
            raise HcError(rc, last_error())
        cap = int(n.value)


def fno3(fi: "F.Fno3Input", device: int = 0, small: bool = False) -> np.ndarray:
    """hc_fno3 (small: hc_fno3_small, decoded): overlaps between new reads sharing an original read, in discovery order."""
    off, idx, pos, reads = (np.ascontiguousarray(a) for a in (fi.off, fi.sr_idx, fi.sr_pos, fi.reads))
    cap = 4096
    fn = lib().hc_fno3_small if small else lib().hc_fno3
    while True:
        out = np.zeros(cap, dtype=FNO_OVERLAP_SMALL if small else F.FNO_OVERLAP)
        n = ctypes.c_uint64(0)
        rc = fn(len(off) - 1, off.ctypes.data, idx.ctypes.data, pos.ctypes.data, len(reads), reads.ctypes.data,
                fi.no_inclusions, out.ctypes.data, cap, ctypes.byref(n), device)
        if rc == 0:
            return fno_small_to_overlaps(out[: n.value]) if small else out[: n.value]
        if rc != -5:
            raise HcError(rc, last_error())
        cap = int(n.value)


def _text_call(call, cap: int) -> bytes:
    while True:
        out = np.empty(max(cap, 1), dtype=np.uint8)
        nb, nl = ctypes.c_uint64(0), ctypes.c_uint64(0)
        rc = call(out.ctypes.data, cap, ctypes.byref(nb), ctypes.byref(nl))
        if rc == 0:
            return out[: nb.value].tobytes()
        if rc != -5:
            raise HcError(rc, last_error())
        cap = int(nb.value)


def fno1_text(fi: "F.FnoInput", device: int = 0) -> bytes:
    """hc_fno1_text: the reference's overlaps.txt (unique lines in byte order, each ending in a newline), built on the GPU."""
    st, keep = _fno_input_c(fi)
    edges = np.ascontiguousarray(fi.edges)
    return _text_call(lambda p, cap, nb, nl: lib().hc_fno1_text(ctypes.byref(st), edges.ctypes.data if len(edges) else None, len(edges),
                                                                 p, cap, nb, nl, None, device), max(96 * len(edges), 4096))


def fno1_text_nonedges(fi: "F.FnoInput", idmap: "IdMap", head: np.ndarray, n_adjacency: int, nonedge_text, tail: np.ndarray,
                       device: int = 0, text_cap: Optional[int] = None):
    """hc_fno1_text_nonedges: overlaps.txt of the stream head ++ (lines of nonedge_text that are not an edge of
    head[:n_adjacency]) ++ tail, the non-edge lines parsed on the GPU (fi.edges is not read).  nonedge_text: bytes or a
    uint8 array (e.g. a slice of host_alloc memory).  Returns (rc, text, n_lines, n_records, stats of formats.FNO_NONEDGE_STATS);
    with text_cap one call with that capacity (rc may be HC_ERR_CAPACITY), else the capacity is grown until the text fits.
    Argument and input errors are returned in rc, not raised."""
    st, keep = _fno_input_c(fi)
    head = np.ascontiguousarray(head, dtype=F.FNO_EDGE)
    tail = np.ascontiguousarray(tail, dtype=F.FNO_EDGE)
    buf = np.frombuffer(nonedge_text, dtype=np.uint8) if isinstance(nonedge_text, (bytes, bytearray)) else nonedge_text
    cap = max(96 * (len(head) + len(tail) + len(buf) // 40), 4096) if text_cap is None else text_cap
    stats = np.zeros(1, dtype=F.FNO_NONEDGE_STATS)
    while True:
        out = np.empty(max(cap, 1), dtype=np.uint8)
        nb, nl, nr = ctypes.c_uint64(0), ctypes.c_uint64(0), ctypes.c_uint64(0)
        rc = lib().hc_fno1_text_nonedges(ctypes.byref(st), idmap.handle, head.ctypes.data if len(head) else None, len(head), n_adjacency,
                                         buf.ctypes.data if len(buf) else None, len(buf), tail.ctypes.data if len(tail) else None,
                                         len(tail), out.ctypes.data if cap else None, cap, ctypes.byref(nb), ctypes.byref(nl),
                                         ctypes.byref(nr), stats.ctypes.data, device)
        if rc == -5 and text_cap is None:
            cap = int(nb.value)
            continue
        return rc, out[: nb.value].tobytes() if rc == 0 else b"", int(nl.value), int(nr.value), stats[0]


def fno3_text(fi: "F.Fno3Input", device: int = 0) -> bytes:
    """hc_fno3_text: the lines of hc_fno3's overlaps in discovery order, each ending in a newline, built on the GPU."""
    off, idx, pos, reads = (np.ascontiguousarray(a) for a in (fi.off, fi.sr_idx, fi.sr_pos, fi.reads))
    return _text_call(lambda p, cap, nb, nl: lib().hc_fno3_text(len(off) - 1, off.ctypes.data, idx.ctypes.data, pos.ctypes.data,
                                                                 len(reads), reads.ctypes.data, fi.no_inclusions, p, cap, nb, nl,
                                                                 device), 1 << 16)


ADJ_EDGE = np.dtype([("vertex1", "<u4"), ("vertex2", "<u4"), ("nonoverlap_len", "<u4"), ("reserved", "<u4")])   # hc_adj_edge


def build_adjacency(edges: np.ndarray, n_vertices: int, keep: Optional[np.ndarray] = None, sort: bool = False, device: int = 0):
    """hc_build_adjacency: (out_off, out_perm, in_off, in_src, ties) -- adjacency lists in insertion order or, sort=True,
    in the order of OverlapGraph::sortEdges, and the adj_in lists that walk produces."""
    edges = np.ascontiguousarray(edges, dtype=ADJ_EDGE)
    n = len(edges)
    k = None if keep is None else np.ascontiguousarray(keep, dtype=np.uint8)
    out_off = np.zeros(n_vertices + 1, dtype=np.uint64)
    in_off = np.zeros(n_vertices + 1, dtype=np.uint64)
    out_perm = np.zeros(max(n, 1), dtype=np.uint32)
    in_src = np.zeros(max(n, 1), dtype=np.uint32)
    ties = np.zeros(max(n_vertices, 1), dtype=np.uint8)
    kept = ctypes.c_uint64(0)
    _check(lib().hc_build_adjacency(edges.ctypes.data if n else None, n, k.ctypes.data if k is not None else None, n_vertices, int(sort),
                                    out_off.ctypes.data, out_perm.ctypes.data, in_off.ctypes.data, in_src.ctypes.data, ties.ctypes.data,
                                    ctypes.byref(kept), device))
    m = int(kept.value)
    return out_off, out_perm[:m], in_off, in_src[:m], ties[:n_vertices]


SUBREAD_PROBLEM = np.dtype([("begin1", "<u8"), ("end1", "<u8"), ("begin2", "<u8"), ("end2", "<u8"), ("trim_pos1", "<i4"), ("trim_pos2", "<i4")])


def subread_info(problems: np.ndarray, pos: np.ndarray, vertex: np.ndarray, device: int = 0):
    """hc_subread_info: (info [n_entries] of formats.FNO_SUBREAD, first [n_entries])."""
    P = np.ascontiguousarray(problems, dtype=SUBREAD_PROBLEM)
    pos = np.ascontiguousarray(pos, dtype=np.int32)
    vertex = np.ascontiguousarray(vertex, dtype=np.uint32)
    n = len(pos)
    info = np.zeros(max(n, 1), dtype=F.FNO_SUBREAD)
    first = np.zeros(max(n, 1), dtype=np.uint8)
    _check(lib().hc_subread_info(P.ctypes.data if len(P) else None, len(P), pos.ctypes.data if n else None, vertex.ctypes.data if n else None, n,
                                 info.ctypes.data, first.ctypes.data, device))
    return info[:n], first[:n]


def host_alloc(nbytes: int, write_combined: bool = False) -> np.ndarray:
    """hc_host_alloc as a uint8 numpy array (pinned; the memory lives until the process ends or hc_host_free on its address)."""
    p = lib().hc_host_alloc(nbytes, int(write_combined))
    if not p:
        raise HcError(-3, "hc_host_alloc failed")
    return np.ctypeslib.as_array((ctypes.c_uint8 * nbytes).from_address(p))


def dedup_edges(edges: np.ndarray, n_vertices: int, ignore_inclusions: bool = False, inclusions: Optional[np.ndarray] = None,
                device: int = 0):
    """hc_dedup_edges: (winner flags, inclusions marks, dup_count, inclusion_count) of the graph insert."""
    edges = np.ascontiguousarray(edges, dtype=F.DEDUP_EDGE)
    win = np.zeros(max(len(edges), 1), dtype=np.uint8)
    inc = np.zeros(max(n_vertices, 1), dtype=np.uint8) if inclusions is None else np.ascontiguousarray(inclusions, dtype=np.uint8).copy()
    counts = np.zeros(2, dtype=np.uint64)
    _check(lib().hc_dedup_edges(edges.ctypes.data if len(edges) else None, len(edges), int(ignore_inclusions), win.ctypes.data,
                                inc.ctypes.data, n_vertices, counts.ctypes.data, device))
    return win[: len(edges)].astype(bool), inc[:n_vertices], int(counts[0]), int(counts[1])


class IdMap:
    """hc_idmap: read id -> store index on the device (FastqStorage::m_ID_to_index)."""

    def __init__(self, ids: np.ndarray, device: int = 0):
        ids = np.ascontiguousarray(ids, dtype=np.uint64)
        self._h = lib().hc_idmap_create(ids.ctypes.data if len(ids) else None, len(ids), device)
        if not self._h:
            raise HcError(-1, last_error())

    @property
    def handle(self):
        return self._h

    def close(self) -> None:
        if getattr(self, "_h", None):
            lib().hc_idmap_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def ingest(self, text: bytes, params: np.ndarray, cand_cap: Optional[int] = None, filtered_cap: Optional[int] = None):
        """hc_ingest_overlaps on a host buffer of complete lines.
        Returns (candidates, candidate line numbers, filtered OVERLAP_REC, their line numbers, stats)."""
        buf = np.frombuffer(text, dtype=np.uint8) if len(text) else np.zeros(0, dtype=np.uint8)
        guess = int(np.count_nonzero(buf == 10)) + 1
        ccap = guess if cand_cap is None else cand_cap
        fcap = guess if filtered_cap is None else filtered_cap
        cand = np.zeros(max(ccap, 1), dtype=F.CANDIDATE)
        cl = np.zeros(max(ccap, 1), dtype=np.uint64)
        filt = np.zeros(max(fcap, 1), dtype=F.OVERLAP_REC)
        fl = np.zeros(max(fcap, 1), dtype=np.uint64)
        st = np.zeros(1, dtype=F.INGEST_STATS)
        rc = lib().hc_ingest_overlaps(self._h, buf.ctypes.data if len(buf) else None, len(buf), params.ctypes.data, cand.ctypes.data,
                                      cl.ctypes.data, ccap, filt.ctypes.data, fl.ctypes.data, fcap, st.ctypes.data)
        if rc != 0:
            err = HcError(rc, last_error())
            err.required = (int(st[0]["n_scored"]), int(st[0]["n_filtered"]))
            raise err
        ns, nf = int(st[0]["n_scored"]), int(st[0]["n_filtered"])
        return cand[:ns], cl[:ns], filt[:nf], fl[:nf], st[0]
