"""CPU: the C++ drop-in boundary (include/interface + libb200jpg.so).

* the tag-list methods behave like the reference's (same transcript as the same test program linked to the reference),
* a client written against the interface compiles against BOTH header sets,
* that client, linked to the reference, reproduces the golden pixels (so the client itself is right),
* against this repository it parses and reports, and fails loudly for want of a GPU instead of falling back.
"""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLIENT = os.path.join(ROOT, "tests", "client")
GOLDEN = os.path.join(ROOT, "tests", "golden")
# stripe_client.cpp compiled against the reference's headers and library by oracle/Makefile (where a reference build exists)
STRIPE_REF = os.path.join(ROOT, "oracle", "_ref", "stripe_ref")


def build_b200(src, out):
    lib_dir = os.path.join(ROOT, "libjpeg_b200")
    subprocess.run(["g++", "-O1", "-I" + os.path.join(ROOT, "include"), os.path.join(CLIENT, src), "-L" + lib_dir, "-lb200jpg",
                    "-Wl,-rpath," + lib_dir, "-o", out], check=True)


def read_pnm(path):
    data = open(path, "rb").read()
    magic, dims, maxv, rest = data.split(b"\n", 3)
    w, h = map(int, dims.split())
    c = 3 if magic == b"P6" else 1
    return np.frombuffer(rest, dtype=np.uint8).reshape(h, w, c)


def test_tagitem_methods_match_reference(built, tmp_path):
    mine = str(tmp_path / "tag_b200")
    build_b200("tagitem_check.cpp", mine)
    a = subprocess.run([mine], capture_output=True, text=True, check=True).stdout
    assert "walk: 80000201=640 80000202=480 80000201=641 80000203=3 80000204=8" in a
    assert "filter count" in a and "sizeof item 16" in a
    # the same program linked against the reference library (tests/golden/make_reference_decodes.py)
    assert a == open(os.path.join(GOLDEN, "tagitem_transcript.txt")).read()


@pytest.mark.parametrize("name", ["c420_50x38_z4_q75", "c444_17x9_q95", "g_40x24_z2_q75", "c422_100x60_z5_q80"])
def test_client_against_reference_reproduces_golden(built, tmp_path, name):
    if not os.path.exists(STRIPE_REF):
        pytest.skip("oracle/_ref/stripe_ref is built where the reference build exists (oracle/Makefile)")
    out = str(tmp_path / "o.pnm")
    subprocess.run([STRIPE_REF, os.path.join(GOLDEN, name + ".jpg"), out], check=True, capture_output=True)
    golden = np.load(os.path.join(GOLDEN, "golden_pixels.npz"))[name]
    assert np.array_equal(read_pnm(out), golden)


def test_client_against_b200_parses_and_fails_loudly_without_gpu(built, tmp_path):
    import torch
    exe = str(tmp_path / "stripe_b200")
    build_b200("stripe_client.cpp", exe)
    r = subprocess.run([exe, os.path.join(GOLDEN, "c420_50x38_z4_q75.jpg"), str(tmp_path / "o.pnm")], capture_output=True, text=True)
    if torch.cuda.is_available():
        assert r.returncode == 0
    else:
        assert r.returncode == 1
        assert "-8193" in r.stderr  # B200JPG_ERR_NO_DEVICE: no silent CPU detour
    assert r.stdout.startswith("50 38 3")  # Read + GetInformation work on the host
    assert "subx=1,2 suby=1,2" in r.stdout
