"""hc_sfo2overlaps (the overlaps file built on the GPU from the overlapper's SFO lines) and lib/hc_sfo2overlaps --gpu=true
against what the reference script wrote (tests/golden/sfo_*.npz) and against the host converter, which
tests/test_sfo2overlaps.py pins on the same fixtures and which is the specification for any other input."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from haploconduct_b200 import build as B, capi, formats as F, workloads as W
from util import GOLDEN

NAMES = sorted(f[len("sfo_"):-4] for f in os.listdir(GOLDEN) if f.startswith("sfo_"))
EXE = os.path.join(B.LIBDIR, "hc_sfo2overlaps")
STDOUT = b"total overlap count: %d\nof which single-single: %d\n"


def run_cli(tmp_path, text, ns, npairs, gpu, env=None, name="x"):
    """(exit status, output file bytes or None, stdout, stderr) of the converter on `text`."""
    d = tmp_path / (name + ("_gpu" if gpu else "_host"))
    d.mkdir(exist_ok=True)
    (d / "in.sfo").write_bytes(text)
    if (d / "out.txt").exists():
        (d / "out.txt").unlink()
    args = [EXE, "--in", "in.sfo", "--out", "out.txt", "--num_singles", str(ns), "--num_pairs", str(npairs)] + (["--gpu=true"] if gpu else [])
    r = subprocess.run(args, cwd=str(d), env=dict(os.environ, **(env or {})), stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    out = (d / "out.txt").read_bytes() if (d / "out.txt").exists() else None
    return r.returncode, out, r.stdout, r.stderr


def check_against_host(tmp_path, text, ns, npairs, name="x"):
    rc, ref, stdout, err = run_cli(tmp_path, text, ns, npairs, gpu=False, name=name)
    assert rc == 0, err
    got, st = capi.sfo2overlaps(text, ns, npairs)
    assert got == ref
    assert STDOUT % (int(st["s_s_count"]) + int(st["p_count"]), int(st["s_s_count"])) == stdout
    assert int(st["n_lines"]) == text.count(b"\n") + (1 if text and not text.endswith(b"\n") else 0)
    assert int(st["n_out_lines"]) == ref.count(b"\n")
    return st


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_goldens_abi_and_cli(built_lib, tmp_path, name):
    z = np.load(os.path.join(GOLDEN, "sfo_" + name + ".npz"))
    text, ns, npairs = z["sfo"].tobytes(), int(z["num_singles"]), int(z["num_pairs"])
    got, st = capi.sfo2overlaps(text, ns, npairs)
    assert got == z["overlaps"].tobytes()
    assert STDOUT % (int(st["s_s_count"]) + int(st["p_count"]), int(st["s_s_count"])) == z["stdout"].tobytes()
    rc, out, stdout, err = run_cli(tmp_path, text, ns, npairs, gpu=True)
    assert rc == 0, err
    assert out == z["overlaps"].tobytes() and stdout == z["stdout"].tobytes()


SHAPES = [   # seed, num_singles, num_pairs, lines, irregular spelling
    (1, 300, 0, 2000, False),            # no pairs: single-single lines only
    (2, 0, 400, 5000, False),            # no singles
    (3, 500, 1000, 20000, False),
    (4, 20, 30, 20000, True),            # dense: few reads, large groups, many repeats
    (5, 20000, 60000, 100000, True),
    (6, 10, 10, 1, False),
    (7, 10, 10, 37, True),
    (8, 4, 6, 3000, False),              # dense, canonical spelling
]


@pytest.mark.gpu
@pytest.mark.parametrize("seed,ns,npairs,n,irregular", SHAPES)
def test_random_against_host(built_lib, tmp_path, seed, ns, npairs, n, irregular):
    check_against_host(tmp_path, W.make_sfo_text(seed, ns, npairs, n, irregular=irregular), ns, npairs)


@pytest.mark.gpu
def test_large_input(built_lib, tmp_path):
    """5 * 10^6 lines: many radix tiles, ids that vary in every byte of the key (every digit pass), more than 2^16
    groups, a group of 6000 lines, a run of 40 lines with equal keys and different text, identical lines far apart."""
    ns, npairs = 1000, 2 ** 31 - 1000
    rng = np.random.default_rng(9)
    big = [W.make_sfo_text(31, ns, npairs, 5_000_000 - 6000 - 40 - 2, irregular=True)]
    a, b = ns + 5, ns + 6                                  # one group: the two reads' four end pairs, 6000 distinct lines
    grp = []
    for i in range(6000):
        ea, eb = rng.integers(0, 2, 2)
        grp.append(b"%d\t%d\t%s\t%d\t%d\t%d\t%d\t%d" % (a + ea * npairs, b + eb * npairs, b"NI"[i % 2:i % 2 + 1], rng.integers(-50, 50),
                                                       rng.integers(-50, 50), rng.integers(30, 90), rng.integers(30, 90), i))
    run = []                                               # equal keys (7, 9, 7, 9), different text
    for i in range(40):
        sa = (b"+7", b"7", b"007")[i % 3]
        sep = (b"\t", b" ", b"  ")[i // 3 % 3]
        run.append(sa + sep + b"9\tN\t%d\t4\t50\t50\t%d" % (3 + i % 2, i % 5))
    same = b"11\t12\tN\t3\t-4\t60\t61\t2"
    text = same + b"\n" + b"\n".join(grp[:3000]) + b"\n" + big[0] + b"\n".join(run + grp[3000:]) + b"\n" + same + b"\n"
    st = check_against_host(tmp_path, text, ns, npairs)
    assert int(st["n_lines"]) == 5_000_000
    assert paired_groups(text, ns, npairs) > 2 ** 16


def paired_groups(text, ns, npairs):
    """The host converter's groups in `text`: distinct (idA, idB) of original ids, idA != idB, one of them paired."""
    sfo = np.array([int(x) for line in text.splitlines() for x in line.split(None, 2)[:2]], dtype=np.int64).reshape(-1, 2)
    orig = np.where(sfo < ns + npairs, sfo, sfo - npairs)
    a, b = orig.min(axis=1), orig.max(axis=1)
    keep = (a != b) & (b >= ns)
    return len(np.unique(a[keep] << 32 | b[keep]))


EDGE = {
    "empty": (b"", 5, 5),
    "no_trailing_newline": (b"1\t2\tN\t3\t4\t50\t50\t0\n2\t1\tN\t-3\t4\t51\t50\t0", 5, 0),
    "single_line": (b"1\t2\tN\t3\t4\t50\t50\t0\n", 5, 0),
    "self_overlaps_only": (b"6\t6\tN\t3\t4\t50\t50\t0\n5\t9\tN\t3\t4\t50\t50\t0\n1\t1\tI\t0\t0\t10\t10\t1\n", 3, 4),
    # the pairs of (3, 4) are the last group: never matched; the single-single line still comes out
    "last_group_unmatched": (b"3\t4\tN\t5\t6\t50\t50\t0\n5\t6\tN\t7\t8\t50\t50\t0\n0\t1\tN\t2\t2\t40\t40\t0\n", 3, 2),
    # (ns 2, np 4: sfo 6..9 are the second ends of reads 2..5) one-line groups around a matched group, then a last group
    "one_line_groups": (b"2\t3\tN\t5\t6\t50\t50\t0\n2\t4\tN\t5\t6\t50\t50\t0\n6\t8\tN\t7\t8\t50\t50\t0\n"
                        b"3\t5\tI\t1\t2\t30\t30\t0\n0\t1\tN\t1\t1\t20\t20\t0\n4\t5\tN\t1\t1\t20\t20\t0\n", 2, 4),
    # idA > idB: flip_N negates the overhangs, flip_I swaps them as strings
    "flipped_N_and_I": (b"6\t3\tN\t+5\t-06\t50\t49\t0\n8\t5\tN\t7\t-8\t50\t48\t1\n6\t4\tI\t+2\t03\t40\t41\t0\n8\t2\tI\t1\t+5\t40\t39\t0\n"
                        b"2\t1\tN\t-2\t3\t30\t30\t0\n3\t6\tN\t-5\t6\t49\t50\t0\n", 10, 0),
    "flipped_paired": (b"7\t4\tN\t+5\t-06\t50\t49\t0\n3\t0\tN\t7\t-8\t50\t48\t1\n4\t3\tI\t+2\t03\t40\t41\t0\n0\t7\tI\t1\t+5\t40\t39\t0\n"
                       b"5\t2\tN\t-2\t3\t30\t30\t0\n", 0, 4),
    "crlf": (b"1\t2\tN\t3\t4\t50\t50\t0\r\n2\t1\tI\t-3\t4\t51\t50\t0\r\n1\t2\tN\t3\t4\t50\t50\t0\n", 5, 0),
    # minlen == 0 in the last group (4, 5): the host never computes it; the group (3, 4) before it is matched
    "minlen0_last_group": (b"3\t4\tN\t0\t5\t50\t50\t0\n6\t7\tN\t1\t5\t50\t50\t0\n4\t5\tN\t0\t5\t0\t10\t0\n7\t8\tN\t0\t5\t0\t10\t0\n", 3, 3),
    # minlen == 0 in a group whose pair does not match (different ori), followed by another group
    "minlen0_unmatched_pair": (b"3\t4\tN\t0\t5\t0\t10\t0\n6\t7\tI\t0\t5\t50\t50\t0\n3\t5\tN\t1\t1\t20\t20\t0\n", 3, 3),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(EDGE))
def test_edge_cases(built_lib, tmp_path, case):
    text, ns, npairs = EDGE[case]
    check_against_host(tmp_path, text, ns, npairs)


@pytest.mark.gpu
def test_golden_with_crlf_line_ends(built_lib, tmp_path):
    z = np.load(os.path.join(GOLDEN, "sfo_mixed_dense.npz"))
    text = z["sfo"].tobytes().replace(b"\n", b"\r\n")
    check_against_host(tmp_path, text, int(z["num_singles"]), int(z["num_pairs"]))


ERRORS = {   # name: (text, ns, np, the status hc_sfo2overlaps reports)
    "seven_fields": (b"1\t2\tN\t3\t4\t50\t50\n", 5, 0, F.SFO_DIES),
    "empty_line": (b"1\t2\tN\t3\t4\t50\t50\t0\n\n1\t3\tN\t3\t4\t50\t50\t0\n", 5, 0, F.SFO_DIES),
    "bad_id": (b"1\tx2\tN\t3\t4\t50\t50\t0\n", 5, 0, F.SFO_DIES),
    "bad_number": (b"1\t2\tN\t3\t4\t5a\t50\t0\n", 5, 0, F.SFO_DIES),
    "lone_sign": (b"1\t2\tN\t-\t4\t50\t50\t0\n", 5, 0, F.SFO_DIES),
    "id_out_of_range": (b"1\t99\tN\t3\t4\t50\t50\t0\n", 5, 2, F.SFO_DIES),
    "negative_id_paired": (b"-1\t3\tN\t3\t4\t50\t50\t0\n", 5, 2, F.SFO_DIES),
    "minlen0_single_single": (b"1\t2\tN\t3\t4\t50\t50\t0\n1\t3\tN\t0\t5\t0\t10\t0\n", 5, 0, F.SFO_DIES),
    "minlen0_matched_pair": (b"0\t1\tN\t0\t5\t0\t10\t0\n4\t5\tN\t1\t5\t10\t10\t0\n2\t3\tN\t1\t1\t20\t20\t0\n", 0, 4, F.SFO_DIES),
    "nineteen_digits": (b"1\t2\tN\t0000000000000000003\t4\t50\t50\t0\n", 5, 0, F.SFO_DECLINED),
    "id_2_to_32": (b"4294967296\t2\tN\t3\t4\t50\t50\t0\n", 5, 0, F.SFO_DECLINED),
    "negative_id_single": (b"-3\t2\tN\t3\t4\t50\t50\t0\n", 5, 0, F.SFO_DECLINED),
    "overhang_2_to_40": (b"1\t2\tN\t1099511627776\t4\t50\t50\t0\n", 5, 0, F.SFO_DECLINED),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(ERRORS))
def test_errors_and_declines(built_lib, tmp_path, case):
    text, ns, npairs, status = ERRORS[case]
    with pytest.raises(capi.HcError) as e:
        capi.sfo2overlaps(text, ns, npairs)
    assert e.value.code == -4 and int(e.value.stats["first_error_status"]) == status
    line = int(e.value.stats["first_error_line"])
    off, ln = int(e.value.stats["first_error_offset"]), int(e.value.stats["first_error_length"])
    assert text.split(b"\n")[line] + b"\n" == text[off:off + ln]
    host = run_cli(tmp_path, text, ns, npairs, gpu=False)
    gpu = run_cli(tmp_path, text, ns, npairs, gpu=True)
    assert gpu[0] == host[0] and gpu[1] == host[1] and gpu[2] == host[2]
    extra = gpu[3][:len(gpu[3]) - len(host[3])]            # one line saying why the host converts, then the host's own messages
    assert gpu[3].endswith(host[3]) and extra.count(b"\n") == 1 and b"converting on the host" in extra
    assert (host[0] == 1) == (status == F.SFO_DIES)


def test_gpu_flag_without_a_device_is_an_error(built_lib, tmp_path):
    rc, out, stdout, err = run_cli(tmp_path, b"1\t2\tN\t3\t4\t50\t50\t0\n", 5, 0, gpu=True, env={"CUDA_VISIBLE_DEVICES": ""})
    assert rc == 1 and out is None and stdout == b"" and err.strip()


@pytest.mark.gpu
def test_capacity(built_lib):
    z = np.load(os.path.join(GOLDEN, "sfo_mixed.npz"))
    text, ns, npairs = z["sfo"].tobytes(), int(z["num_singles"]), int(z["num_pairs"])
    want = z["overlaps"].tobytes()
    L = capi.lib()
    st = np.zeros(1, dtype=F.SFO_STATS)
    nb = ctypes.c_uint64(0)
    assert L.hc_sfo2overlaps(text, len(text), ns, npairs, None, 0, ctypes.byref(nb), st.ctypes.data, 0) == -5
    assert nb.value == len(want)
    buf = np.full(len(want) + 8, 0x5a, dtype=np.uint8)
    assert L.hc_sfo2overlaps(text, len(text), ns, npairs, buf.ctypes.data, len(want) - 1, ctypes.byref(nb), st.ctypes.data, 0) == -5
    assert nb.value == len(want) and (buf == 0x5a).all()
    assert L.hc_sfo2overlaps(text, len(text), ns, npairs, buf.ctypes.data, len(want), ctypes.byref(nb), st.ctypes.data, 0) == 0
    assert nb.value == len(want) and buf[:len(want)].tobytes() == want and (buf[len(want):] == 0x5a).all()
