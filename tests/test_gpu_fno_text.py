"""GPU suite: hc_fno1_text / hc_fno3_text, the bytes of overlaps.txt built on the device -- against the reference's own
files (golden), against the oracle's records formatted, sorted and de-duplicated in Python, on inputs whose ids and
values make byte order and numeric order disagree, and at the capacity and argument edges of the C ABI."""
import ctypes

import numpy as np
import pytest

from haploconduct_b200 import capi, formats as F
from oracle import oracle as O
from util import fno3_golden_names, fno_golden_names, load_fno3_golden, load_fno_golden, random_fno3_input, random_fno_input

pytestmark = pytest.mark.gpu


def as_file(lines):
    return "".join(l + "\n" for l in lines).encode()


@pytest.mark.parametrize("name", fno_golden_names())
def test_fno1_text_is_the_reference_file(built_lib, name):
    fi, ref = load_fno_golden(name)
    assert capi.fno1_text(fi) == as_file(ref)


@pytest.mark.parametrize("name", fno3_golden_names())
def test_fno3_text_is_the_reference_file(built_lib, name):
    fi, ref = load_fno3_golden(name)
    assert capi.fno3_text(fi) == as_file(ref)


@pytest.mark.parametrize("stage48", [False, True])
def test_text_of_dense_random_inputs(built_lib, monkeypatch, stage48):
    """Both record forms: 24-byte records, and (HC_FNO_STAGE48, many first-found-wins partitions) 48-byte ones."""
    if stage48:
        monkeypatch.setenv("HC_FNO_STAGE48", "1")
        monkeypatch.setenv("HC_FNO_PART", "700")
    for seed in (1, 2, 3):
        fi = random_fno_input(seed, n_vertices=500, n_sr=150, n_edges=60000)
        ref = F.fno_output_file(O.fno1(fi))
        assert len(ref) > 1000
        assert capi.fno1_text(fi) == as_file(ref)
        fi3 = random_fno3_input(seed, n_originals=30000, n_reads=2000)
        ref3 = F.fno_lines(O.fno3(fi3))
        assert len(ref3) > 1000
        assert capi.fno3_text(fi3) == as_file(ref3)


def copies_input(ids, edges):
    """Unmerged vertices only: every edge is copied to one line between the vertices' new ids (:46-72)."""
    V = len(ids)
    vr = np.zeros(V, dtype=F.FNO_READ)
    vr["id"] = ids
    vr["len1"] = 100
    e = np.zeros(len(edges), dtype=F.FNO_EDGE)
    for name in edges.dtype.names:
        e[name] = edges[name]
    return F.FnoInput(visited=np.zeros(V, np.uint8), label=np.ones(V, np.uint8), vertex_read=vr,
                      sr_off=np.zeros(V + 1, np.uint64), sr_idx=np.zeros(0, np.uint32), sr_sub=np.zeros(0, dtype=F.FNO_SUBREAD),
                      superread=np.zeros(0, dtype=F.FNO_READ), resolve_orientations=1, no_inclusions=0, edges=e)


def random_edges(rng, n, V):
    e = np.zeros(n, dtype=F.FNO_EDGE)
    e["u"] = rng.randint(0, V, size=n)
    e["v"] = (e["u"] + rng.randint(1, V, size=n)) % V
    e["pos1"], e["pos2"] = rng.randint(0, 3000, size=n), rng.randint(0, 30, size=n)
    e["perc"], e["len1"], e["len2"] = rng.randint(0, 101, size=n), rng.randint(0, 2000, size=n), rng.randint(0, 2000, size=n)
    e["ord"] = rng.choice([ord("1"), ord("2"), ord("-")], size=n)
    e["ori1"], e["ori2"], e["nonedge"] = rng.randint(0, 2, size=n), rng.randint(0, 2, size=n), rng.randint(0, 2, size=n)
    return e


def test_byte_order_is_not_numeric_order(built_lib):
    """Ids of every digit count, with shared prefixes ("1" < "10" < "100" < "2"): every radix digit varies."""
    rng = np.random.RandomState(5)
    pool = [0, 1, 2, 9, 10, 11, 19, 100, 1000000000, 4294967294]
    for d in range(1, 11):
        pool += [int(x) for x in rng.randint(10 ** (d - 1), min(10 ** d, 2 ** 32 - 1), size=4, dtype=np.int64)]
    ids = np.array(sorted(set(pool)), dtype=np.uint64)
    rng.shuffle(ids)
    fi = copies_input(ids, random_edges(rng, 20000, len(ids)))
    got = capi.fno1_text(fi)
    lines = F.fno_lines(O.fno1(fi))
    assert got == as_file(sorted(set(lines), key=lambda s: s.encode()))
    assert got != as_file(sorted(set(lines), key=lambda s: [int(x) if x.lstrip("-").isdigit() else x for x in s.split("\t")]))


@pytest.mark.parametrize("negative", [False, True])
def test_long_runs_of_one_pair_and_repeats(built_lib, negative):
    """More than 32 lines between the same two new reads (the heap-sort branch of the run sort), exact repeats among
    them; with negative and extreme %d values the records take the 48-byte form."""
    rng = np.random.RandomState(7)
    ids = np.array([10, 9, 100, 1, 4294967294], dtype=np.uint64)
    e = random_edges(rng, 3000, len(ids))
    e["u"][:400], e["v"][:400] = 0, 1
    e["u"][400:440], e["v"][400:440] = 3, 2                             # a second run, in the other id order
    special = [-1, -10, -2, 0, 10, 5, 2 ** 31 - 1, -2 ** 31] if negative else [0, 1, 10, 2, 100, 9, 2 ** 24 - 1, 19]
    e["pos1"][:400] = np.resize(special, 400)
    if negative:
        e["len1"][:400:3] = np.resize([-5, -50, -2 ** 31, 2 ** 31 - 1], len(e["len1"][:400:3]))
        e["pos2"][400:440] = np.resize([-3, 3, -30, 30], 40)
    e[200:400] = e[0:200]                                               # exact repeats
    fi = copies_input(ids, e)
    lines = F.fno_lines(O.fno1(fi))
    ref = sorted(set(lines), key=lambda s: s.encode())
    assert len(ref) < len(lines)
    assert capi.fno1_text(fi) == as_file(ref)
    if negative:
        with pytest.raises(capi.HcError):                              # the values really need the 48-byte record
            capi.fno1(fi, small=True)


def fno1_text_raw(fi, text, cap):
    st, keep = capi._fno_input_c(fi)
    edges = np.ascontiguousarray(fi.edges)
    nb, nl, nr = ctypes.c_uint64(7), ctypes.c_uint64(7), ctypes.c_uint64(7)
    rc = capi.lib().hc_fno1_text(ctypes.byref(st), edges.ctypes.data if len(edges) else None, len(edges), text, cap,
                                 ctypes.byref(nb), ctypes.byref(nl), ctypes.byref(nr), 0)
    return rc, nb.value, nl.value, nr.value


def fno3_text_raw(fi, text, cap):
    off, idx, pos, reads = (np.ascontiguousarray(a) for a in (fi.off, fi.sr_idx, fi.sr_pos, fi.reads))
    nb, nl = ctypes.c_uint64(7), ctypes.c_uint64(7)
    rc = capi.lib().hc_fno3_text(len(off) - 1, off.ctypes.data, idx.ctypes.data, pos.ctypes.data, len(reads), reads.ctypes.data,
                                 fi.no_inclusions, text, cap, ctypes.byref(nb), ctypes.byref(nl), 0)
    return rc, nb.value, nl.value


def test_capacity_query_then_exact_buffer(built_lib):
    fi = random_fno_input(4, n_vertices=500, n_sr=150, n_edges=60000)
    records = O.fno1(fi)
    ref = as_file(F.fno_output_file(records))
    rc, nb, nl, nr = fno1_text_raw(fi, None, 0)
    assert (rc, nb, nl, nr) == (-5, len(ref), ref.count(b"\n"), len(records))
    buf = np.empty(nb, np.uint8)
    rc, nb2, nl2, nr2 = fno1_text_raw(fi, buf.ctypes.data, nb)
    assert (rc, nb2, nl2, nr2) == (0, nb, nl, nr)
    assert buf.tobytes() == ref
    rc, _, _, _ = fno1_text_raw(fi, buf.ctypes.data, nb - 1)
    assert rc == -5

    fi3 = random_fno3_input(4, n_originals=30000, n_reads=2000)
    ref3 = as_file(F.fno_lines(O.fno3(fi3)))
    rc, nb, nl = fno3_text_raw(fi3, None, 0)
    assert (rc, nb, nl) == (-5, len(ref3), ref3.count(b"\n"))
    buf = np.empty(nb, np.uint8)
    assert fno3_text_raw(fi3, buf.ctypes.data, nb) == (0, nb, nl)
    assert buf.tobytes() == ref3


def test_empty_outputs(built_lib):
    fi = random_fno_input(9, n_edges=10)
    fi.edges = fi.edges[:0]
    assert fno1_text_raw(fi, None, 0) == (0, 0, 0, 0)
    fi = random_fno_input(9, n_edges=3000)
    fi.visited[:] = 1                                                   # every edge goes through super-reads ...
    fi.sr_off = np.arange(len(fi.visited) + 1, dtype=np.uint64)         # ... one per vertex ...
    fi.sr_idx = (np.arange(len(fi.visited)) % len(fi.superread)).astype(np.uint32)
    fi.sr_sub = np.zeros(len(fi.visited), dtype=F.FNO_SUBREAD)
    fi.edges["pos1"] = 10 ** 6                                          # ... and every derivation fails (pos1 beyond the reads)
    assert len(O.fno1(fi)) == 0
    assert fno1_text_raw(fi, None, 0) == (0, 0, 0, 0)
    assert capi.fno1_text(fi) == b""
    fi3 = random_fno3_input(9, n_originals=200)
    fi3.off = np.arange(len(fi3.off), dtype=np.uint64)                  # one new read per original: no pair at all
    fi3.sr_idx, fi3.sr_pos = fi3.sr_idx[:len(fi3.off) - 1], fi3.sr_pos[:len(fi3.off) - 1]
    assert fno3_text_raw(fi3, None, 0) == (0, 0, 0)
    assert capi.fno3_text(fi3) == b""


def test_argument_errors(built_lib):
    fi = random_fno_input(9, n_edges=10)
    fi.edges["u"][3] = 10 ** 6
    with pytest.raises(capi.HcError):
        capi.fno1_text(fi)
    fi = random_fno_input(9, n_edges=10)
    v = int(np.nonzero(fi.visited == 0)[0][0])
    fi.vertex_read["id"][v] = 2 ** 32
    with pytest.raises(capi.HcError):
        capi.fno1_text(fi)
    fi3 = random_fno3_input(9, n_originals=50)
    fi3.sr_idx = fi3.sr_idx.copy()
    fi3.sr_idx[0] = len(fi3.reads)
    with pytest.raises(capi.HcError):
        capi.fno3_text(fi3)
    fi3 = random_fno3_input(9, n_originals=50)
    fi3.reads["id"][0] = 2 ** 32
    with pytest.raises(capi.HcError):
        capi.fno3_text(fi3)
