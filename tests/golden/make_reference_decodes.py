"""Regenerates tests/golden/reference_decodes.json: shape and SHA-256 of the pixels of what the UNMODIFIED reference (oracle/_ref/refharness, oracle/_ref/jpeg)
makes of the streams tests/test_oracle.py builds -- the repo generator's streams (plain, DC quantiser patched, restart
markers damaged, stream variants, four components, a ZRL that steps over position 63), streams of the reference's own
encoder with other sampling factors (the streams stored as well, tests/golden/reference_encoded/<key>.jpg), and `jpeg -c`
decodes without colour transformation. A stream the reference refuses is stored as "refused". Also writes
tests/golden/tagitem_transcript.txt, the output of tests/client/tagitem_check.cpp linked against the reference library.

Run where the reference build exists (`make -C oracle ref`), REF naming the reference's source tree:
    REF=<libjpeg sources> python tests/golden/make_reference_decodes.py
"""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from tests import oracle_binding  # noqa: E402
from tests import test_oracle as t  # noqa: E402


def read_pnm(path):
    magic, dims, maxv, rest = open(path, "rb").read().split(b"\n", 3)
    w, h = map(int, dims.split())
    return np.frombuffer(rest, dtype=np.uint8).reshape(h, w, 3 if magic == b"P6" else 1)


def main():
    from libjpeg_b200 import synth
    out = {}
    os.makedirs(os.path.join(HERE, "reference_encoded"), exist_ok=True)
    with tempfile.TemporaryDirectory() as tmp:
        jpg, raw = os.path.join(tmp, "s.jpg"), os.path.join(tmp, "s.raw")

        def decode(kind, params, data):
            open(jpg, "wb").write(data)
            key = t.reference_key(kind, params)
            px = oracle_binding.reference_decode(jpg, raw)
            out[key] = "refused" if px is None else t.pixel_digest(px)
            print(key, "refused" if px is None else px.shape)

        for p in t.SYNTHETIC:
            decode("synthetic", p, t.synthetic_stream(*p))
        for p in t.HOT:
            decode("hot", p, t.hot_stream(*p))
        for p in oracle_binding.RESTART_DAMAGES:
            decode("damage", p, t.damaged_stream(p))
        for p in t.VARIANTS:
            decode("variant", p, t.variant_stream(*p))
        for p in t.FOUR_COMPONENT:
            decode("four", p, t.four_component_stream(*p))
        decode("zrl", (), oracle_binding.zrl_overrun_stream())
        ppm = os.path.join(tmp, "in.ppm")
        open(ppm, "wb").write(b"P6\n%d %d\n255\n" % (75, 61) + synth.source_image(75, 61, 17).tobytes())
        for sub in t.OTHER_SUBSAMPLING:
            subprocess.run([oracle_binding.REF_CLI, "-q", "80", "-bl", "-s", sub, "-z", "3", ppm, jpg], check=True, capture_output=True)
            data = open(jpg, "rb").read()
            open(os.path.join(HERE, "reference_encoded", t.reference_key("subsampling", sub) + ".jpg"), "wb").write(data)
            decode("subsampling", sub, data)
        for name in t.NO_COLOR_TRANSFORM:
            pnm = os.path.join(tmp, "o.ppm")
            subprocess.run([oracle_binding.REF_CLI, "-c", os.path.join(HERE, name + ".jpg"), pnm], check=True, capture_output=True)
            out[t.reference_key("nocolor", name)] = t.pixel_digest(read_pnm(pnm))
        exe = os.path.join(tmp, "tag_ref")
        subprocess.run(["g++", "-O1", "-w", "-DUSE_AUTOCONF", "-I" + os.path.join(ROOT, "oracle", "ref_config"),
                        "-I" + os.environ["REF"], os.path.join(ROOT, "tests", "client", "tagitem_check.cpp"),
                        os.path.join(ROOT, "oracle", "_ref", "libjpegref.a"), "-o", exe], check=True)
        transcript = subprocess.run([exe], capture_output=True, text=True, check=True).stdout
        open(os.path.join(HERE, "tagitem_transcript.txt"), "w").write(transcript)
    json.dump(out, open(os.path.join(HERE, "reference_decodes.json"), "w"), indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
