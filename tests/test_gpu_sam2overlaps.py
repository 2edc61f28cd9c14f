"""hc_sam2overlaps (the overlaps file of the reference-guided mode built on the GPU from SAM alignments) and
lib/hc_sam2overlaps --gpu=true against what the reference script wrote (tests/golden/sam_*.npz) and against the host
converter, which tests/test_sam2overlaps.py pins on the same fixtures and which is the specification for any other input."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from haploconduct_b200 import build as B, capi, formats as F, workloads as W
from util import GOLDEN

NAMES = sorted(f[len("sam_"):-4] for f in os.listdir(GOLDEN) if f.startswith("sam_"))
EXE = os.path.join(B.LIBDIR, "hc_sam2overlaps")


def fasta_table(fasta):
    """The converter's FASTA reading (:258-283): {name: index} (the last duplicate wins) and the lengths."""
    names, lens, ident, seq, have = {}, [], None, 0, False
    for line in fasta.split(b"\n")[:-1] if fasta.endswith(b"\n") else fasta.split(b"\n"):
        if line.startswith(b">"):
            if have and ident:
                lens.append(seq)
                names[ident] = len(lens) - 1
                seq, have = 0, False
            ident = line.split()[0][1:] if line.split() else b""
        else:
            seq += len(line)
            have = have or len(line) > 0
    lens.append(seq)
    names[ident] = len(lens) - 1
    return names, lens


def expected_stdout(st, rs, use_s, use_p, verbose):
    """What the converter prints for these counts."""
    out = b""
    if verbose and use_s:
        out += b"Number of singles unmapped:  %d\nNumber of singles reversed:  %d\n" % (st["unmapped_s"], st["reverse_s"])
    if verbose and use_p:
        out += (b"Number of read ends discarded:  %d\nNumber of read ends unmapped:  %d\nNumber of reverse complements considered:  %d\n"
                % (st["discarded"], st["unmapped_p"], st["reverse_p"]))
    for r in rs:
        if not verbose or r["n_alignments"] == 0:
            continue
        out += b"Total number of alignments:  %d\n... of which singles:  %d\n... of which paired:  %d\n" % (
            r["n_alignments"], r["n_singles"], r["n_paired"])
        if r["problems"]:
            out += b"# cases where overlap_pos2 < 0:  %d\n" % r["problems"]
        out += (b"Total number of overlaps found:  %d\n... of which ++:  %d\n... of which +-:  %d\n... of which -+:  %d\n"
                b"... of which --:  %d\n" % (r["n_overlaps"], *[int(x) for x in r["types"]]))
    if st["total_alns"] == 0:
        out += b"\n\nERROR: No reads could be aligned to reference. Exiting.\n"
    return out


def run_cli(tmp_path, fasta, sam_s, sam_p, min_ov, verbose, gpu, env=None, name="x"):
    """(exit status, output file bytes or None, stdout, stderr) of the converter."""
    d = tmp_path / (name + ("_gpu" if gpu else "_host"))
    d.mkdir(exist_ok=True)
    (d / "ref.fasta").write_bytes(fasta)
    cmd = [EXE, "--ref", "ref.fasta", "--out", "out.txt", "--min_overlap_len", str(min_ov)]
    for fn, t, flag in (("s.sam", sam_s, "--sam_s"), ("p.sam", sam_p, "--sam_p")):
        if t is not None:
            (d / fn).write_bytes(t)
            cmd += [flag, fn]
    if verbose:
        cmd.append("--verbose")
    if gpu:
        cmd.append("--gpu=true")
    if (d / "out.txt").exists():
        (d / "out.txt").unlink()
    r = subprocess.run(cmd, cwd=str(d), env=dict(os.environ, **(env or {})), stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    out = (d / "out.txt").read_bytes() if (d / "out.txt").exists() else None
    return r.returncode, out, r.stdout, r.stderr


def check_against_host(tmp_path, fasta, sam_s, sam_p, min_ov, verbose=True, name="x"):
    """The ABI and the --gpu=true CLI against the host CLI: file, stdout, exit status."""
    host = run_cli(tmp_path, fasta, sam_s, sam_p, min_ov, verbose, gpu=False, name=name)
    assert host[0] in (0, 1) and host[1] is not None and host[3] == b"", host[3]         # 1: nothing aligned
    names, lens = fasta_table(fasta)
    got, st, rs = capi.sam2overlaps(sam_s, sam_p, names, lens, min_ov)
    assert got == host[1]
    assert expected_stdout(st, rs, sam_s is not None, sam_p is not None, verbose) == host[2]
    assert int(st["n_out_lines"]) == host[1].count(b"\n")
    gpu = run_cli(tmp_path, fasta, sam_s, sam_p, min_ov, verbose, gpu=True, name=name)
    assert gpu == host
    return st, rs


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_goldens_abi_and_cli(built_lib, tmp_path, name):
    z = np.load(os.path.join(GOLDEN, "sam_" + name + ".npz"))
    fasta = z["fasta"].tobytes()
    sam_s = z["sam_s"].tobytes() if int(z["use_s"]) else None
    sam_p = z["sam_p"].tobytes() if int(z["use_p"]) else None
    min_ov, verbose = int(z["min_overlap_len"]), bool(int(z["verbose"]))
    names, lens = fasta_table(fasta)
    got, st, rs = capi.sam2overlaps(sam_s, sam_p, names, lens, min_ov)
    assert got == z["overlaps"].tobytes()
    assert expected_stdout(st, rs, sam_s is not None, sam_p is not None, verbose) == z["stdout"].tobytes()
    rc, out, stdout, err = run_cli(tmp_path, fasta, sam_s, sam_p, min_ov, verbose, gpu=True)
    assert rc == 0, err
    assert out == z["overlaps"].tobytes() and stdout == z["stdout"].tobytes()


SHAPES = [   # seed, singles, pairs, references, min_overlap_len, irregular
    (1, 3000, 0, [("refA", 4000)], 30, False),                       # singles only
    (2, 0, 3000, [("refA", 5000)], 40, False),                       # pairs only
    (3, 2000, 2000, [("refA", 3000), ("refB", 2500), ("refC", 900)], 20, False),
    (4, 1500, 1500, [("refA", 2000)], 0, True),                      # CRLF, "MM" / "SS" / "=" operations, past the end
    (5, 1500, 1500, [("refA", 2000), ("refB", 700)], 140, True),     # min_overlap_len above most reads
    (6, 400, 400, [("chr 1", 600)], -3, False),                      # a negative min_overlap_len
]


@pytest.mark.gpu
@pytest.mark.parametrize("seed,ns,npairs,refs,min_ov,irregular", SHAPES)
def test_random_against_host(built_lib, tmp_path, seed, ns, npairs, refs, min_ov, irregular):
    fasta, sam_s, sam_p = W.make_sam_text(seed, ns, npairs, refs, irregular=irregular)
    if refs[0][0] == "chr 1":                 # the FASTA id ends at whitespace: the SAM says "chr"
        sam_s, sam_p = (t.replace(b"\tchr 1\t", b"\tchr\t") for t in (sam_s, sam_p))
    check_against_host(tmp_path, fasta, sam_s if ns else None, sam_p if npairs else None, min_ov)


@pytest.mark.gpu
def test_references_unused_and_named_twice(built_lib, tmp_path):
    """A reference without alignments, a FASTA name given twice (the later sequence's index wins) and one more after."""
    fasta, sam_s, sam_p = W.make_sam_text(7, 800, 800, [("refA", 1500), ("refB", 1200)])
    fasta += b">refA again\n" + b"ACGT" * 300 + b"\n>empty1\nAC\n>refZ\n" + b"A" * 3000 + b"\n"
    check_against_host(tmp_path, fasta, sam_s, sam_p, 25)


def sam(name, flag, ref, pos, cigar, seq_len, crlf=False):
    return b"%s\t%d\t%s\t%d\t60\t%s\t=\t0\t0\t%s\t%s%s\n" % (name, flag, ref, pos, cigar, b"A" * seq_len, b"I" * seq_len, b"\r" if crlf else b"")


FA = b">r\n" + b"ACGT" * 100 + b"\n"
HEAD = b"@SQ\tSN:r\tLN:400\n"

EDGE = {   # name: (sam_s, sam_p, min_ov)
    # singles and pairs at equal positions: singles first; runs of three and four equal ids; unmapped lines between mates
    "ties_runs_unmapped": (HEAD + sam(b"s1", 0, b"r", 50, b"100M", 100) + sam(b"s2", 16, b"r", 50, b"3S97M", 100)
                           + sam(b"s3", 0, b"r", 80, b"60M", 60),
                           HEAD + sam(b"a", 0, b"r", 50, b"100M", 100) + sam(b"a", 0, b"r", 120, b"90M", 90)
                           + sam(b"a", 0, b"r", 60, b"90M", 90)
                           + sam(b"b", 16, b"r", 90, b"80M", 80) + sam(b"u", 4, b"*", 0, b"*", 10) + sam(b"b", 16, b"r", 50, b"70M", 70)
                           + sam(b"b", 0, b"r", 55, b"70M", 70) + sam(b"b", 0, b"r", 100, b"70M", 70)
                           + sam(b"c", 0, b"r", 50, b"5H80M", 80) + sam(b"c", 0, b"r", 51, b"80M4H", 80)
                           + sam(b"d", 16, b"r", 50, b"80M", 80) + sam(b"d", 16, b"r", 50, b"2I78M", 80) + sam(b"e", 0, b"r", 70, b"80M", 80), 0),
    # pairs whose second ends lie left of a later single's (problems), and both directions of the paired-paired walk
    "problems_and_ord": (HEAD + sam(b"s1", 0, b"r", 60, b"100M", 100) + sam(b"s2", 0, b"r", 200, b"100M", 100),
                         HEAD + sam(b"p", 16, b"r", 70, b"100M", 100) + sam(b"p", 16, b"r", 50, b"100M", 100)
                         + sam(b"q", 0, b"r", 52, b"100M", 100) + sam(b"q", 0, b"r", 100, b"10M2D80M", 90)
                         + sam(b"t", 0, b"r", 55, b"100M", 100) + sam(b"t", 0, b"r", 60, b"100M", 100), 10),
    # records past the reference end (only the first of them is processed), CRLF
    "past_the_end": (HEAD + sam(b"s1", 0, b"r", 300, b"100M", 100, True) + sam(b"s2", 0, b"r", 399, b"50M", 50, True)
                     + sam(b"s3", 0, b"r", 401, b"80M", 80, True) + sam(b"s4", 0, b"r", 402, b"80M", 80, True), None, 0),
    # multi-character operations: "SS" is no soft clip, "MM" / "II" count as reference bases, "HH" adds nothing
    "odd_operations": (HEAD + sam(b"s1", 0, b"r", 40, b"5SS95MM", 100) + sam(b"s2", 0, b"r", 50, b"50M2II48M", 100)
                       + sam(b"s3", 0, b"r", 60, b"90M3HH", 90) + sam(b"s4", 0, b"r", 70, b"40=1X40M", 81), None, 0),
    # a defect on an unmapped line is no error; an unterminated last line counts
    "unmapped_defects": (HEAD + sam(b"s1", 0, b"r", 40, b"100M", 100) + b"s2\t4\tr\tx\ty\t*\t=\tz\tw\t\t\n"
                         + sam(b"s3", 0, b"r", 60, b"90M", 90)[:-1], None, 0),
    # no header, empty texts
    "no_header": (sam(b"s1", 0, b"r", 40, b"100M", 100) + sam(b"s2", 0, b"r", 45, b"100M", 100), b"", 0),
    "nothing_aligned": (HEAD + sam(b"s1", 4, b"r", 40, b"100M", 100), None, 0),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(EDGE))
def test_edge_cases(built_lib, tmp_path, case):
    sam_s, sam_p, min_ov = EDGE[case]
    check_against_host(tmp_path, FA, sam_s, sam_p, min_ov)


@pytest.mark.gpu
def test_large_input(built_lib, tmp_path):
    """10^6 alignments: several radix passes, more than 2^16 records with partners, a pile-up of 3000 alignments at
    one place (a record with thousands of partners), three references."""
    refs = [("chrA", 3_000_000), ("chrB", 2_000_000), ("chrC", 1_000_000)]
    fasta, sam_s, sam_p = W.make_sam_text(11, 500_000, 250_000, refs, irregular=True)
    pile = b"".join(sam(b"pile%d" % i, 16 * (i % 2), b"chrC", 20_000 + i % 7, b"100M", 100) for i in range(3000))
    sam_s += pile
    st, rs = check_against_host(tmp_path, fasta, sam_s, sam_p, 30)
    assert int(st["total_alns"]) > 2 ** 16 and int(st["n_out_lines"]) > 10 ** 6


ERRORS = {   # name: (sam_s, sam_p, min_ov, status, file, line)
    "ten_fields": (HEAD + sam(b"s1", 0, b"r", 40, b"100M", 100) + b"s2\t0\tr\t5\t60\t10M\t=\t0\t0\tAAAAAAAAAA\n", None, 0, F.SAM_DIES, 0, 2),
    "empty_line": (HEAD + sam(b"s1", 0, b"r", 40, b"100M", 100) + b"\n", None, 0, F.SAM_DIES, 0, 2),
    "empty_line_in_header": (HEAD + b"\n" + sam(b"s1", 0, b"r", 40, b"100M", 100), None, 0, F.SAM_DIES, 0, 1),
    "bad_flag": (None, HEAD + b"p\t4x\t*\t0\t0\t*\t=\t0\t0\tA\tI\n", 0, F.SAM_DIES, 1, 1),
    "bad_pos": (HEAD + b"s1\t0\tr\t4a\t60\t10M\t=\t0\t0\tAAAAAAAAAA\tIIIIIIIIII\n", None, 0, F.SAM_DIES, 0, 1),
    "bad_tlen": (HEAD + b"s1\t0\tr\t4\t60\t10M\t=\t0\t-\tAAAAAAAAAA\tIIIIIIIIII\n", None, 0, F.SAM_DIES, 0, 1),
    "one_cigar_run": (HEAD + sam(b"s1", 0, b"r", 40, b"*", 100), None, 0, F.SAM_DIES, 0, 1),
    "unknown_ref": (HEAD + sam(b"s1", 0, b"r", 40, b"100M", 100) + sam(b"s2", 0, b"x", 40, b"100M", 100), None, 0, F.SAM_DIES, 0, 2),
    "unknown_ref_pair": (None, HEAD + sam(b"p", 0, b"x", 40, b"100M", 100) + sam(b"p", 0, b"r", 60, b"100M", 100), 0, F.SAM_DIES, 1, 1),
    "odd_cigar_walked": (HEAD + sam(b"s1", 0, b"r", 40, b"100M", 100) + sam(b"s2", 0, b"r", 50, b"90M5", 90), None, 0, F.SAM_DIES, 0, 2),
    "zero_run_walked_back": (HEAD + sam(b"s1", 0, b"r", 40, b"100M", 100) + sam(b"s2", 0, b"r", 50, b"0M90M", 90), None, 0, F.SAM_DIES, 0, 2),
    "empty_seq_walked": (HEAD + sam(b"s1", 0, b"r", 40, b"100M", 100) + sam(b"s2", 0, b"r", 50, b"90M", 0), None, -5, F.SAM_DIES, 0, 2),
    # the second end of a pair is walked only when the pair is: its defect kills there
    "defect_in_second_end": (HEAD + sam(b"s1", 0, b"r", 40, b"100M", 100),
                             HEAD + sam(b"p", 0, b"r", 45, b"100M", 100) + sam(b"p", 0, b"r", 60, b"M90", 90), 0, F.SAM_DIES, 1, 2),
    "nineteen_digits": (HEAD + b"s1\t0\tr\t4\t0000000000000000060\t10M\t=\t0\t0\tAAAAAAAAAA\tIIIIIIIIII\n", None, 0, F.SAM_DECLINED, 0, 1),
    "pos_2_to_40": (HEAD + sam(b"s1", 0, b"r", 2 ** 40, b"100M", 100), None, 0, F.SAM_DECLINED, 0, 1),
    "cigar_run_2_to_40": (HEAD + sam(b"s1", 0, b"r", 40, b"%dS100M" % 2 ** 40, 100), None, 0, F.SAM_DECLINED, 0, 1),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(ERRORS))
def test_errors_and_declines(built_lib, tmp_path, case):
    sam_s, sam_p, min_ov, status, f, line = ERRORS[case]
    names, lens = fasta_table(FA)
    with pytest.raises(capi.HcError) as e:
        capi.sam2overlaps(sam_s, sam_p, names, lens, min_ov)
    st = e.value.stats
    assert e.value.code == -4 and int(st["first_error_status"]) == status
    assert (int(st["first_error_file"]), int(st["first_error_line"])) == (f, line)
    text = (sam_s, sam_p)[f]
    off, ln = int(st["first_error_offset"]), int(st["first_error_length"])
    assert text.split(b"\n")[line] + b"\n" == text[off:off + ln]
    for verbose in (False, True):
        host = run_cli(tmp_path, FA, sam_s, sam_p, min_ov, verbose, gpu=False)
        gpu = run_cli(tmp_path, FA, sam_s, sam_p, min_ov, verbose, gpu=True)
        assert gpu[:3] == host[:3]
        extra = gpu[3][:len(gpu[3]) - len(host[3])]        # one line saying why the host converts, then the host's own messages
        assert gpu[3].endswith(host[3]) and extra.count(b"\n") == 1 and b"converting on the host" in extra
        assert (host[0] == 1) == (status == F.SAM_DIES)


def test_gpu_flag_without_a_device_is_an_error(built_lib, tmp_path):
    rc, out, stdout, err = run_cli(tmp_path, FA, HEAD + sam(b"s1", 0, b"r", 40, b"100M", 100), None, 0, True, gpu=True,
                                   env={"CUDA_VISIBLE_DEVICES": ""})
    assert rc == 1 and out is None and stdout == b"" and err.strip()


@pytest.mark.gpu
def test_capacity(built_lib):
    z = np.load(os.path.join(GOLDEN, "sam_mixed_two_refs.npz"))
    sam_s, sam_p = z["sam_s"].tobytes(), z["sam_p"].tobytes()
    names, lens = fasta_table(z["fasta"].tobytes())
    want = z["overlaps"].tobytes()
    nm = [n for n in names]
    blob = b"".join(nm)
    off = np.concatenate([[0], np.cumsum([len(n) for n in nm])]).astype(np.uint64)
    idx = np.array([names[n] for n in nm], dtype=np.uint32)
    rl = np.array(lens, dtype=np.int64)
    L = capi.lib()
    st = np.zeros(1, dtype=F.SAM_STATS)
    nb = ctypes.c_uint64(0)

    def call(buf, cap):
        return L.hc_sam2overlaps(sam_s, len(sam_s), sam_p, len(sam_p), blob, off.ctypes.data, idx.ctypes.data, len(idx), rl.ctypes.data,
                                 len(rl), int(z["min_overlap_len"]), buf, cap, ctypes.byref(nb), None, st.ctypes.data, 0)
    assert call(None, 0) == -5 and nb.value == len(want)
    buf = np.full(len(want) + 8, 0x5a, dtype=np.uint8)
    assert call(buf.ctypes.data, len(want) - 1) == -5
    assert nb.value == len(want) and (buf == 0x5a).all()
    assert call(buf.ctypes.data, len(want)) == 0
    assert nb.value == len(want) and buf[:len(want)].tobytes() == want and (buf[len(want):] == 0x5a).all()
