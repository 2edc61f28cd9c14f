"""hc_fno1_text_nonedges: FindNextOverlaps 1 with nonedge_overlaps.txt parsed, checked against the adjacency lists and put
into the edge stream on the device (the loop of src/FindNextOverlaps.cpp:635-697, hcb_fno.cpp's append_nonedges).

The oracle is a Python restatement of that loop (getline, trim, tab split, Overlap::from_fields, the id map, checkEdge);
hc_fno1_text on the stream it builds must give the same text, line and record counts.  On the reference fixtures the
restatement must reproduce the reference's own stream, and lib/hc_fno --gpu_parse=true the reference's overlaps.txt."""
import glob
import json
import os
import subprocess

import numpy as np
import pytest

from haploconduct_b200 import build as B, capi, formats as F
from util import GOLDEN, load_fno_golden, random_fno_input

EXE = os.path.join(B.LIBDIR, "hc_fno")
HC_ERR_ARG, HC_ERR_INPUT, HC_ERR_CAPACITY = -1, -4, -5
SKIPPED, ERROR, UNKNOWN_ID = 4, 5, 6
ULONG_MAX = (1 << 64) - 1


# ---- the host loop, restated --------------------------------------------------------------------------------------------
def _strtol_like(s, base0):
    """strtoul(s, NULL, 0) (base0) or strtol(s, NULL, 10), C semantics on the leading part of s."""
    if s.isascii() and s.isdigit() and len(s) < 19 and not (base0 and len(s) > 1 and s[0] == "0"):
        return int(s)
    i, n = 0, len(s)
    while i < n and s[i] in " \t\n\v\f\r":
        i += 1
    neg = False
    if i < n and s[i] in "+-":
        neg = s[i] == "-"
        i += 1
    base = 10
    if base0:
        if s[i:i + 2] in ("0x", "0X") and i + 2 < n and s[i + 2] in "0123456789abcdefABCDEF":
            base, i = 16, i + 2
        elif s[i:i + 1] == "0":
            base = 8
    digits = "0123456789abcdef"[:base]
    v = 0
    while i < n and s[i].lower() in digits:
        v = v * base + digits.index(s[i].lower())
        i += 1
    if base0:
        if v > ULONG_MAX:
            return ULONG_MAX
        return (-v) & ULONG_MAX if neg else v
    lim = (1 << 63) - (0 if neg else 1)
    v = min(v, lim)
    return -v if neg else v


def _atoi_u32(s):
    """(unsigned int)atoi(s)"""
    return _strtol_like(s, False) & 0xffffffff


def _i32(x):
    return x - (1 << 32) if x >= 1 << 31 else x


def _char_field(f, strip):
    if len(f) == 1:
        return f
    return "".join(c for c in f if c not in strip)


def parse_overlap(fields):
    """Overlap::from_fields (hcb_host.cpp) -> dict, or None where the constructor dies."""
    if len(fields) != 13:
        return None
    pos1, pos2, perc1, perc2 = (_atoi_u32(fields[k]) for k in (2, 3, 7, 8))
    len1, len2 = _atoi_u32(fields[9]), _atoi_u32(fields[10])
    if fields[3] == "-":
        pos2 = perc2 = len2 = 0
    if _i32(pos1) < 0 or _i32(pos2) < 0:
        return None
    ori1, ori2 = _char_field(fields[5], " "), _char_field(fields[6], " ")
    if ori1 not in ("+", "-") or ori2 not in ("+", "-"):
        return None
    if any(_i32(p) < 0 or _i32(p) > 100 for p in (perc1, perc2)) or _i32(len1) < 0 or _i32(len2) < 0:
        return None
    t1, t2 = _char_field(fields[11], "\n\t "), _char_field(fields[12], "\n\t ")
    if t1 not in ("s", "p") or t2 not in ("s", "p"):
        return None
    o = _char_field(fields[4], " ")
    ok = o in ("1", "2", "-") and (o == "-" if "s" in (t1, t2) else o in ("1", "2"))
    if not ok:
        return None
    perc = int(0.5 * (perc1 + perc2)) if perc2 > 0 else perc1
    return dict(id1=_strtol_like(fields[0], True), id2=_strtol_like(fields[1], True), pos1=pos1, pos2=pos2, ord=ord(o),
                ori1=int(ori1 == "+"), ori2=int(ori2 == "+"), perc=perc, len1=len1, len2=len2)


def host_nonedges(text, read_ids, adjacency):
    """The stream's middle segment of hcb_fno.cpp's loop: (FNO_EDGE records, n_lines, first error (line, offset, length,
    status) or None).  read_ids[i] = id of read i = vertex i; adjacency = the adj_out lists in order (FNO_EDGE).
    A line of more than 13 fields is an error here, as in hc_fno1_text_nonedges; the host loop reads its first 13 and the
    device call leaves such a file to it."""
    index = {}
    for i, r in enumerate(read_ids.tolist()):
        index.setdefault(r, i)                          # std::map::insert keeps the first
    first = {}
    for e in adjacency[["u", "v", "nonedge"]].tolist():
        first.setdefault((e[0], e[1]), e[2])
    lines = text.split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()                                     # getline: no line after a final newline
    out, off = [], 0
    for k, raw in enumerate(lines):
        line = raw.decode("latin-1").strip("\t ")
        fields = line.split("\t") if line else []
        o = parse_overlap(fields)
        status = SKIPPED if len(fields) != 13 else ERROR
        if o is not None:
            if o["id1"] not in index or o["id2"] not in index:
                o, status = None, UNKNOWN_ID
        if o is None:
            return None, len(lines), (k, off, len(raw), status)
        v1, v2 = index[o["id1"]], index[o["id2"]]
        ne = first.get((v1, v2), first.get((v2, v1)))   # checkEdge(v1, v2, true): the first v1 -> v2, else the first v2 -> v1
        off += len(raw) + 1
        if ne is not None and ne == 0:
            continue                                    # an edge: score > 0
        out.append((v1, v2, o["pos1"], o["pos2"], o["perc"], o["len1"], o["len2"], o["ord"], o["ori1"], o["ori2"], 1))
    rec = np.zeros(len(out), dtype=F.FNO_EDGE)
    if out:
        a = np.array(out, dtype=np.int64)
        for j, name in enumerate(F.FNO_EDGE.names):
            rec[name] = a[:, j].astype(F.FNO_EDGE[name]) if name not in ("pos1", "pos2", "len1", "len2") else \
                (a[:, j] & 0xffffffff).astype(np.uint32).view(np.int32)
    return rec, len(lines), None


# ---- fixtures -------------------------------------------------------------------------------------------------------------
def fno1_state_names():
    return sorted(os.path.basename(p)[len("fnostate_"):-4] for p in glob.glob(os.path.join(GOLDEN, "fnostate_fno1_*.npz")))


def fixture_segments(name):
    """(FnoInput, ref lines, read ids, head, n_adjacency, non-edge text, tail, middle of the reference's stream)"""
    z = np.load(os.path.join(GOLDEN, "fnostate_" + name + ".npz"))
    fi, ref = load_fno_golden(name)
    kinds = [l.split(b"\t", 1)[0] for l in z["state"].tobytes().split(b"\n")]
    n_adj, n_head = kinds.count(b"A"), kinds.count(b"A") + kinds.count(b"B")
    text = z["nonedge"].tobytes()
    mid, _, err = host_nonedges(text, z["ids"], fi.edges[:n_adj])
    assert err is None
    return fi, ref, z["ids"], fi.edges[:n_head], n_adj, text, fi.edges[n_head + len(mid):], mid


@pytest.mark.parametrize("name", fno1_state_names())
def test_restatement_builds_the_reference_stream(name):
    fi, _, _, head, _, _, tail, mid = fixture_segments(name)
    got = np.concatenate([head, mid, tail])
    assert len(got) == len(fi.edges) and got.tobytes() == fi.edges.tobytes(), name


def setup_fixture(d, name, extra_nonedge=b""):
    z = np.load(os.path.join(GOLDEN, "fnostate_" + name + ".npz"))
    rs = F.ReadSet(ids=z["ids"], descs=z["descs"], bases=z["bases"], quals=z["quals"], n_single=int(z["n_single"]))
    F.write_fastq_set(rs, d + "/s.fastq", d + "/p1.fastq", d + "/p2.fastq")
    with open(d + "/state.txt", "wb") as f:
        f.write(z["state"].tobytes())
    with open(d + "/nonedge_overlaps.txt", "wb") as f:
        f.write(z["nonedge"].tobytes() + extra_nonedge)
    cmd = [EXE, "--state", d + "/state.txt", "--output", d + "/", "--FNO", "1"]
    if rs.n_single:
        cmd += ["--singles", d + "/s.fastq"]
    if rs.n_reads > rs.n_single:
        cmd += ["--paired1", d + "/p1.fastq", "--paired2", d + "/p2.fastq"]
    return cmd


@pytest.mark.gpu
@pytest.mark.parametrize("name", fno1_state_names())
def test_hc_fno_gpu_parse_writes_the_reference_file(built_lib, tmp_path, name):
    d = str(tmp_path)
    cmd = setup_fixture(d, name)
    ref = [str(x) for x in np.load(os.path.join(GOLDEN, name + ".npz"))["ref_lines"]]
    summaries = []
    for flag in ("--gpu_parse=true", "--gpu_parse=false"):
        out = subprocess.run(cmd + [flag], cwd=d, check=True, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True).stdout
        summaries.append(json.loads([l for l in out.split("\n") if l.startswith("{")][-1]))
        with open(d + "/overlaps.txt") as f:
            assert f.read().split("\n")[:-1] == ref, (name, flag)
    dev, host = summaries
    for k in ("lines", "stream", "device_overlaps", "nonedge_lines", "nonedge_kept"):
        assert dev[k] == host[k], k
    assert dev["nonedge_on_device"] == 1 and dev["nonedge_device_ms"] > 0      # the device branch ran, not the host loop
    assert host["nonedge_on_device"] == 0 and host["nonedge_device_ms"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", fno1_state_names())
def test_fixture_stream_equals_hc_fno1_text(built_lib, name):
    fi, ref, ids, head, n_adj, text, tail, mid = fixture_segments(name)
    _, n_text_lines, _ = host_nonedges(text, ids, head[:n_adj])
    m = capi.IdMap(ids)
    rc, got, n_lines, n_rec, st = capi.fno1_text_nonedges(fi, m, head, n_adj, text, tail)
    assert rc == 0, capi.last_error()
    assert got.decode().split("\n")[:-1] == ref
    assert int(st["n_nonedges"]) == len(mid) and int(st["n_stream"]) == len(fi.edges)
    assert int(st["n_lines"]) == n_text_lines
    assert int(st["first_error_line"]) == ULONG_MAX
    assert got == capi.fno1_text(fi) and n_lines == len(ref)


# ---- synthetic inputs -----------------------------------------------------------------------------------------------------
def _line(rng, a, b, types=None, pad=False, dash=False):
    t1, t2 = types or (("s", "p")[rng.randint(2)], ("s", "p")[rng.randint(2)])
    o = "-" if "s" in (t1, t2) else "12"[rng.randint(2)]
    f = [str(a), str(b), str(rng.randint(0, 300)), "-" if dash else str(rng.randint(0, 300)), o, "+-"[rng.randint(2)],
         "+-"[rng.randint(2)], str(rng.randint(0, 101)), str(rng.randint(0, 101)), str(rng.randint(0, 300)), str(rng.randint(0, 300)), t1, t2]
    s = "\t".join(f)
    if pad:
        s = " \t " + s + "\t  "
    return s


def synthetic(seed, V=300, n_lines=4000, n_adj=3000, n_branch=200, n_tail=150):
    """(FnoInput, read ids, head, n_adjacency, text, tail): adjacency lists with duplicate and conflicting entries, branching
    edges on adjacency pairs, lines on forward / reverse / both-way / absent pairs, self-overlaps, padding, '-' in POS2 and
    all four read-type pairs."""
    rng = np.random.RandomState(seed)
    fi = random_fno_input(seed, n_vertices=V, n_edges=n_adj + n_branch + n_tail)
    e = fi.edges
    adj = np.sort(e[:n_adj], order=["u"], kind="stable")
    dup = rng.choice(n_adj, size=n_adj // 10)
    h = len(dup) // 2
    for f in ("u", "v"):
        adj[f][dup[:h]] = adj[f][dup[h:2 * h]]          # repeated pairs, with their own non-edge flags
    adj = np.sort(adj, order=["u"], kind="stable")
    branch = e[n_adj:n_adj + n_branch].copy()
    for f in ("u", "v"):
        branch[f][: n_branch // 2] = adj[f][: n_branch // 2]
    branch["nonedge"][: n_branch // 2] = 0
    tail = e[n_adj + n_branch:]
    ids = (rng.permutation(V).astype(np.uint64) * 7 + 1000)
    lines = []
    for _ in range(n_lines):
        r = rng.randint(6)
        if r < 2:
            k = rng.randint(n_adj)
            a, b = (adj[k]["u"], adj[k]["v"]) if r == 0 else (adj[k]["v"], adj[k]["u"])
        elif r == 2:
            k = rng.randint(n_branch)
            a, b = branch[k]["u"], branch[k]["v"]
        elif r == 3:
            a = b = rng.randint(V)
        else:
            a, b = rng.randint(V), rng.randint(V)
        lines.append(_line(rng, ids[a], ids[b], pad=rng.randint(8) == 0, dash=rng.randint(8) == 0))
    text = ("\n".join(lines) + "\n").encode()
    return fi, ids, np.concatenate([adj, branch]), n_adj, text, tail


def expected(fi, ids, head, n_adj, text, tail):
    mid, n_lines, err = host_nonedges(text, ids, head[:n_adj])
    assert err is None
    fi.edges = np.concatenate([head, mid, tail])
    return capi.fno1_text(fi), len(mid), n_lines


def check(fi, ids, head, n_adj, text, tail, buf=None):
    want, n_mid, n_lines = expected(fi, ids, head, n_adj, text, tail)
    m = capi.IdMap(ids)
    rc, got, nl, nr, st = capi.fno1_text_nonedges(fi, m, head, n_adj, text if buf is None else buf, tail)
    assert rc == 0, capi.last_error()
    assert got == want
    assert nl == want.count(b"\n") and int(st["n_nonedges"]) == n_mid and int(st["n_lines"]) == n_lines
    assert int(st["n_stream"]) == len(head) + n_mid + len(tail)
    n = ctypes_records(fi)
    assert nr == n
    return st


def ctypes_records(fi):
    """*n_records of hc_fno1_text on fi.edges"""
    import ctypes
    st, keep = capi._fno_input_c(fi)
    nb, nl, nr = ctypes.c_uint64(0), ctypes.c_uint64(0), ctypes.c_uint64(0)
    e = np.ascontiguousarray(fi.edges)
    rc = capi.lib().hc_fno1_text(ctypes.byref(st), e.ctypes.data if len(e) else None, len(e), None, 0, ctypes.byref(nb), ctypes.byref(nl),
                                 ctypes.byref(nr), 0)
    assert rc in (0, HC_ERR_CAPACITY)
    return int(nr.value)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 2])
def test_synthetic_streams(built_lib, seed):
    st = check(*synthetic(seed))
    assert 0 < int(st["n_nonedges"]) < int(st["n_lines"])


@pytest.mark.gpu
def test_million_lines_in_many_pieces(built_lib, monkeypatch):
    fi, ids, head, n_adj, text, tail = synthetic(7, V=2000, n_lines=1_000_000, n_adj=20000, n_branch=500, n_tail=300)
    monkeypatch.setenv("HC_INGEST_PIECE", "3000000")
    assert len(text) > 10 * 3000000
    st = check(fi, ids, head, n_adj, text, tail)
    assert int(st["n_lines"]) == 1_000_000 and st["device_ms"] > 0


@pytest.mark.gpu
def test_byte_offsets_pinned_and_unterminated(built_lib, monkeypatch):
    fi, ids, head, n_adj, text, tail = synthetic(3, n_lines=600)
    monkeypatch.setenv("HC_INGEST_PIECE", "2500")
    for k in range(16):
        buf = np.zeros(len(text) + 32, dtype=np.uint8)
        buf[k:k + len(text)] = np.frombuffer(text, dtype=np.uint8)
        check(fi, ids, head, n_adj, text, tail, buf[k:k + len(text)])
    pinned = capi.host_alloc(len(text) + 32)
    pinned[5:5 + len(text)] = np.frombuffer(text, dtype=np.uint8)
    check(fi, ids, head, n_adj, text, tail, pinned[5:5 + len(text)])
    check(fi, ids, head, n_adj, text[:-1], tail)                 # no newline after the last line
    check(fi, ids, head, n_adj, b"", tail)                        # == hc_fno1_text(head ++ tail)
    fi.edges = np.concatenate([head, tail])
    rc, got, _, _, st = capi.fno1_text_nonedges(fi, capi.IdMap(ids), head, n_adj, b"", tail)
    assert rc == 0 and got == capi.fno1_text(fi) and int(st["n_lines"]) == 0


def _edge(u, v, nonedge):
    e = np.zeros(1, dtype=F.FNO_EDGE)
    e["u"], e["v"], e["pos1"], e["perc"], e["len1"], e["ord"], e["nonedge"] = u, v, 10, 90, 100, ord("-"), nonedge
    return e


@pytest.mark.gpu
def test_which_lines_join_the_stream(built_lib):
    """checkEdge(v1, v2, true) > 0 decided by the first adjacency entry of (v1, v2), else of (v2, v1); branching edges and
    the tail are not in the graph."""
    fi = random_fno_input(11, n_vertices=20, n_edges=1)
    ids = np.arange(20, dtype=np.uint64) + 100
    adj = np.concatenate([_edge(1, 2, 0),                      # forward edge only
                          _edge(3, 4, 1), _edge(3, 4, 0),      # first match a non-edge, later an edge: kept
                          _edge(5, 6, 0), _edge(5, 6, 1),      # first match an edge: dropped
                          _edge(7, 8, 0), _edge(8, 7, 1),      # both ways: the forward one decides
                          _edge(10, 9, 1), _edge(10, 11, 0),
                          _edge(12, 12, 0)])                   # a self pair
    branch = _edge(13, 14, 0)                                  # not in the graph
    tail = _edge(15, 16, 0)
    head = np.concatenate([adj, branch])
    rows = [(1, 2, True), (2, 1, True), (3, 4, False), (5, 6, True), (6, 5, True), (7, 8, True), (8, 7, False), (9, 10, False),
            (11, 10, True), (12, 12, True), (13, 14, False), (15, 16, False), (17, 18, False), (19, 19, False)]
    rng = np.random.RandomState(0)
    text = "".join(_line(rng, 100 + a, 100 + b, types=t) + "\n" for a, b, _ in rows for t in (("s", "s"), ("s", "p"), ("p", "s"), ("p", "p")))
    text = text.encode()
    mid, _, err = host_nonedges(text, ids, adj)
    assert err is None
    want_pairs = [(a, b) for a, b, dropped in rows for _ in range(4) if not dropped]
    assert list(zip(mid["u"].tolist(), mid["v"].tolist())) == want_pairs
    check(fi, ids, head, len(adj), text, tail)


# ---- errors ---------------------------------------------------------------------------------------------------------------
SENTINEL = 0xA5


def call_raw(fi, m, head, n_adj, text, tail, cap, device=0):
    import ctypes
    st, keep = capi._fno_input_c(fi)
    head = np.ascontiguousarray(head, dtype=F.FNO_EDGE)
    tail = np.ascontiguousarray(tail, dtype=F.FNO_EDGE)
    buf = np.frombuffer(text, dtype=np.uint8)
    out = np.full(max(cap, 1) + 64, SENTINEL, dtype=np.uint8)
    stats = np.zeros(1, dtype=F.FNO_NONEDGE_STATS)
    nb, nl, nr = ctypes.c_uint64(7), ctypes.c_uint64(7), ctypes.c_uint64(7)
    rc = capi.lib().hc_fno1_text_nonedges(ctypes.byref(st), m.handle, head.ctypes.data if len(head) else None, len(head), n_adj,
                                          buf.ctypes.data if len(buf) else None, len(buf), tail.ctypes.data if len(tail) else None,
                                          len(tail), out.ctypes.data if cap else None, cap, ctypes.byref(nb), ctypes.byref(nl),
                                          ctypes.byref(nr), stats.ctypes.data, device)
    return rc, out, int(nb.value), int(nl.value), stats[0]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["fields12", "bad_ori", "cr", "unknown_id", "empty_line", "fields14"])
def test_bad_line_is_reported_and_nothing_written(built_lib, monkeypatch, kind):
    fi, ids, head, n_adj, text, tail = synthetic(5, n_lines=3000)
    monkeypatch.setenv("HC_INGEST_PIECE", "20000")
    lines = text.split(b"\n")[:-1]
    k = 2345
    f = lines[k].split(b"\t")
    bad = {"fields12": b"\t".join(f[:12]), "bad_ori": b"\t".join(f[:5] + [b"x"] + f[6:]), "cr": lines[k] + b"\r",
           "unknown_id": b"\t".join([b"999999999"] + f[1:]), "empty_line": b"", "fields14": lines[k] + b"\tp"}[kind]
    lines[k] = bad
    text = b"\n".join(lines) + b"\n"
    offset = sum(len(l) + 1 for l in lines[:k])
    _, _, err = host_nonedges(text, ids, head[:n_adj])
    status = {"fields12": SKIPPED, "empty_line": SKIPPED, "fields14": SKIPPED, "unknown_id": UNKNOWN_ID}.get(kind, ERROR)
    assert err == (k, offset, len(bad), status)
    cap = 1 << 22
    rc, out, nb, nl, st = call_raw(fi, capi.IdMap(ids), head, n_adj, text, tail, cap)
    assert rc == HC_ERR_INPUT, capi.last_error()
    assert (int(st["first_error_line"]), int(st["first_error_offset"]), int(st["first_error_length"]),
            int(st["first_error_status"])) == (k, offset, len(bad), status)
    assert np.all(out == SENTINEL) and nb == 0 and nl == 0


@pytest.mark.gpu
def test_argument_errors(built_lib):
    fi, ids, head, n_adj, text, tail = synthetic(4, n_lines=50)
    m = capi.IdMap(ids)
    assert call_raw(fi, m, head, n_adj, text, tail, 0, device=1)[0] == HC_ERR_ARG           # m lives on device 0
    assert call_raw(fi, capi.IdMap(ids[:-1]), head, n_adj, text, tail, 0)[0] == HC_ERR_ARG  # one read per vertex
    assert call_raw(fi, m, head, len(head) + 1, text, tail, 0)[0] == HC_ERR_ARG               # n_adjacency > n_head
    h = head.copy()
    h[[5, n_adj - 5]] = h[[n_adj - 5, 5]]
    assert call_raw(fi, m, h, n_adj, text, tail, 0)[0] == HC_ERR_ARG                          # adjacency not in vertex order
    h = head.copy()
    h["v"][-1] = len(ids)
    assert call_raw(fi, m, h, n_adj, text, tail, 0)[0] == HC_ERR_ARG                          # a branching edge out of range
    t = tail.copy()
    t["u"][0] = len(ids) + 3
    assert call_raw(fi, m, head, n_adj, text, t, 0)[0] == HC_ERR_ARG
    bad = random_fno_input(4, n_vertices=len(ids), n_edges=1)
    bad.superread["id"][0] = 1 << 33                                                          # a check of hc_fno1_text
    assert call_raw(bad, m, head, n_adj, text, tail, 0)[0] == HC_ERR_ARG
    assert call_raw(fi, m, head, len(head) + 1, text + b"1\t2\n", tail, 0)[0] == HC_ERR_ARG   # arguments before input


@pytest.mark.gpu
def test_capacity_protocol(built_lib):
    fi, ids, head, n_adj, text, tail = synthetic(6, n_lines=800)
    want, _, _ = expected(fi, ids, head, n_adj, text, tail)
    m = capi.IdMap(ids)
    rc, _, nb, nl, _ = call_raw(fi, m, head, n_adj, text, tail, 0)
    assert rc == HC_ERR_CAPACITY and nb == len(want) and nl == want.count(b"\n")
    rc, out, nb, _, _ = call_raw(fi, m, head, n_adj, text, tail, len(want) - 1)
    assert rc == HC_ERR_CAPACITY and nb == len(want) and np.all(out == SENTINEL)
    rc, out, nb, nl, st = call_raw(fi, m, head, n_adj, text, tail, len(want))
    assert rc == 0 and out[:nb].tobytes() == want and np.all(out[nb:] == SENTINEL)


@pytest.mark.gpu
def test_hc_fno_falls_back_to_the_host_loop_on_a_bad_line(built_lib, tmp_path):
    name = "fno1_synth_paired_0"
    d = str(tmp_path / "clean")
    os.makedirs(d)
    out = subprocess.run(setup_fixture(d, name) + ["--gpu_parse=true"], cwd=d, check=True, stdout=subprocess.PIPE, text=True).stdout
    assert json.loads([l for l in out.split("\n") if l.startswith("{")][-1])["nonedge_on_device"] == 1   # without the bad line
    res = []
    for flag in ("--gpu_parse=true", "--gpu_parse=false"):
        d = str(tmp_path / flag[2:].replace("=", "_"))
        os.makedirs(d)
        cmd = setup_fixture(d, name, extra_nonedge=b"0\t1\t5\t5\t-\t+\t*\t90\t0\t100\t0\ts\ts\n")
        p = subprocess.run(cmd + [flag], cwd=d, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        res.append((p.returncode, p.stderr))
        assert not os.path.exists(d + "/overlaps.txt")
    assert res[0] == res[1] and res[0][0] != 0
    assert "m_ori" in res[0][1]
