"""CPU: pins the oracle (oracle/jpeg_oracle.c) against what the unmodified reference made of the same streams -- the
golden vectors (tests/golden/make_golden.py ...) and the streams built below, whose reference decodes are stored as shape
and SHA-256 of the pixels in tests/golden/reference_decodes.json (tests/golden/make_reference_decodes.py)."""
import glob
import hashlib
import json
import os
import re

import numpy as np
import pytest

from tests import oracle_binding

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NAMES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.jpg")))


@pytest.fixture(scope="module")
def golden_pixels():
    return np.load(os.path.join(GOLDEN, "golden_pixels.npz"))


REFERENCE_DECODES = os.path.join(GOLDEN, "reference_decodes.json")
REFERENCE_ENCODED = os.path.join(GOLDEN, "reference_encoded")


def reference_key(kind, params):
    """Name of a case in reference_decodes.json: (72, 40, (2, 2), 3, 60) -> '<kind>__72_40_2_2_3_60'."""
    return kind + "__" + "_".join(re.findall(r"[0-9A-Za-z]+", str(params)))


def pixel_digest(px):
    return {"shape": list(px.shape), "sha256": hashlib.sha256(np.ascontiguousarray(px).tobytes()).hexdigest()}


def reference_decode(kind, params):
    """Shape and SHA-256 of the reference's pixels for a case, None where the reference refused the stream."""
    ref = json.load(open(REFERENCE_DECODES))[reference_key(kind, params)]
    return None if ref == "refused" else ref


def same_pixels(px, ref):
    return px.dtype == np.uint8 and pixel_digest(px) == ref


def synthetic_stream(w, h, sub, z, q):
    from libjpeg_b200 import synth
    return synth.encode(synth.source_image(w, h, 7 * w + h), q, sub, z).tobytes()


def hot_stream(w, h, sub, z, dcq):
    from libjpeg_b200 import synth
    return oracle_binding.with_dc_quantiser(synth.encode(synth.source_image(w, h, 5), 75, sub, z), dcq)


def damaged_stream(damage):
    from libjpeg_b200 import synth
    return oracle_binding.with_restart_damage(synth.encode(synth.source_image(200, 136, 3), 75, (2, 2), 2), damage)


def variant_stream(flags, w, h, sub, z):
    from libjpeg_b200 import synth
    return synth.encode(synth.source_image(w, h, 5), 80, sub, z, flags).tobytes()


def four_component_stream(w, h, sub, z):
    from libjpeg_b200 import synth
    return oracle_binding.with_fourth_component(synth.encode(synth.source_image(w, h, 5), 80, sub, z, 1))


SYNTHETIC = [(72, 40, (2, 2), 3, 60), (31, 47, (2, 2), 0, 85), (64, 32, (1, 1), 8, 92), (90, 33, (2, 1), 2, 70), (45, 90, (1, 2), 6, 70)]
HOT = [(96, 80, (2, 2), 3, 255), (200, 120, (2, 1), 0, 160), (64, 64, (1, 1), 4, 255), (130, 70, (1, 2), 2, 200)]
# sampling factors the reference encoder's -s takes; the streams it wrote are stored beside its decodes
OTHER_SUBSAMPLING = ["1x1,4x1,4x1", "1x1,3x2,3x2", "1x1,2x3,2x3", "1x1,1x4,1x4", "1x1,3x4,3x4", "1x1,4x3,4x3", "1x1,2x1,4x2"]
VARIANTS = [(1, 70, 50, (2, 2), 5), (1, 64, 48, (1, 1), 0), (2, 40, 40, (2, 2), 3), (6, 40, 40, (2, 1), 0), (7, 33, 47, (1, 2), 4)]
FOUR_COMPONENT = [(64, 48, (1, 1), 4), (70, 50, (2, 2), 5), (100, 37, (2, 1), 0), (33, 90, (1, 2), 3)]
NO_COLOR_TRANSFORM = ["c420_96x80_z6_q75", "c444_64x64_z16_q90", "c422_100x60_z5_q80"]


@pytest.mark.parametrize("name", NAMES)
def test_oracle_matches_golden(oracle, golden_pixels, name):
    data = open(os.path.join(GOLDEN, name + ".jpg"), "rb").read()
    rc, px = oracle.decode(data)
    assert rc == 0
    ref = golden_pixels[name]
    assert px.shape == ref.shape
    assert np.array_equal(px, ref), "oracle differs from the reference's pixels in %d bytes" % int((px != ref).sum())


def test_golden_covers_all_vectors(golden_pixels):
    assert sorted(golden_pixels.files) == NAMES and len(NAMES) >= 12


@pytest.mark.parametrize("w,h,sub,z,q", SYNTHETIC)
def test_oracle_matches_reference_on_synthetic_streams(oracle, built, w, h, sub, z, q):
    """Streams from the repo's own generator, decoded by the real reference and by the oracle."""
    ref = reference_decode("synthetic", (w, h, sub, z, q))
    assert ref is not None
    rc, px = oracle.decode(synthetic_stream(w, h, sub, z, q))
    assert rc == 0 and same_pixels(px, ref)


@pytest.mark.parametrize("w,h,sub,z,dcq", HOT)
def test_oracle_matches_reference_beyond_the_usual_sample_range(oracle, built, w, h, sub, z, dcq):
    """DC quantiser patched to a large value: IDCT samples leave int16 and the 32-bit colour range (the reference
    computes the colour matrix in 64 bits); the oracle must follow the reference there too."""
    ref = reference_decode("hot", (w, h, sub, z, dcq))
    assert ref is not None
    rc, px = oracle.decode(hot_stream(w, h, sub, z, dcq))
    assert rc == 0 and same_pixels(px, ref)


def test_oracle_idct_dc_only(oracle):
    """DC-only block: every sample = ((dc*q*16 + 128*128) * 512 + 256 >> 9) * 512 + 2048 >> 12 (idct.cpp:233-334)."""
    blk = np.zeros(64, dtype=np.int32)
    blk[0] = 5
    q = np.full(64, 16, dtype=np.uint16)
    out = oracle.idct(blk, q)
    t = 5 * 16 * 16 + 128 * 128
    p1 = (t * 512 + 256) >> 9
    assert np.all(out == ((p1 * 512 + 2048) >> 12))


def test_oracle_rejects_lossless_and_garbage(oracle):
    data = bytearray(open(os.path.join(GOLDEN, NAMES[0] + ".jpg"), "rb").read())
    i = data.find(b"\xff\xc0")
    data[i + 1] = 0xC3
    rc, _ = oracle.decode(bytes(data))
    assert rc == -1034  # NOT_IMPLEMENTED
    rc, _ = oracle.decode(b"\x00\x01\x02\x03")
    assert rc == -1038  # MALFORMED_STREAM


PROGRESSIVE = os.path.join(GOLDEN, "progressive")
PNAMES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(PROGRESSIVE, "*.jpg")))


@pytest.mark.parametrize("name", PNAMES)
def test_oracle_matches_progressive_golden(oracle, name):
    """SURVEY 8f2 groundwork: SOF2 streams of the reference encoder (DC first, AC bands, DC and AC refinement scans, with
    and without restart markers) decode to the reference's pixels (codestream/sequentialscan.cpp first passes,
    codestream/refinementscan.cpp)."""
    want = np.load(os.path.join(PROGRESSIVE, "progressive_pixels.npz"))[name]
    rc, px = oracle.decode(open(os.path.join(PROGRESSIVE, name + ".jpg"), "rb").read())
    assert rc == 0
    assert np.array_equal(px.reshape(want.shape), want)


SUBSAMPLING = os.path.join(GOLDEN, "subsampling")
SNAMES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(SUBSAMPLING, "*.jpg")))


@pytest.mark.parametrize("name", SNAMES)
def test_oracle_matches_3x_4x_subsampling_golden(oracle, name):
    """SURVEY 8f4 groundwork: chroma subsampled by 3 and 4 (4:1:1, 4:1:0, 3x3 ...) -- the reference's filter cores for those
    factors (upsampling/upsampler.cpp:171-268, 310-386), including their in-place store order."""
    want = np.load(os.path.join(SUBSAMPLING, "subsampling_pixels.npz"))[name]
    rc, px = oracle.decode(open(os.path.join(SUBSAMPLING, name + ".jpg"), "rb").read())
    assert rc == 0
    assert np.array_equal(px.reshape(want.shape), want)


@pytest.mark.parametrize("sub", OTHER_SUBSAMPLING)
def test_oracle_matches_reference_on_other_subsampling(oracle, sub):
    """Streams of the reference's encoder (its CLI takes the sampling factors: `jpeg -q 80 -bl -s <sub> -z 3` on S(75, 61, 17)),
    decoded by reference and oracle."""
    ref = reference_decode("subsampling", sub)
    rc, px = oracle.decode(open(os.path.join(REFERENCE_ENCODED, reference_key("subsampling", sub) + ".jpg"), "rb").read())
    assert rc == 0 and same_pixels(px, ref)


DAMAGED = os.path.join(GOLDEN, "damaged")
DNAMES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(DAMAGED, "*.jpg")))


@pytest.mark.parametrize("name", DNAMES)
def test_oracle_matches_damaged_golden(oracle, name):
    """Streams that end where a restart marker should stand: the reference's resynchronisation (entropyparser.cpp:137-199)
    marks the remaining intervals invalid and their MCUs stay cleared; the fixtures hold the reference's pixels."""
    want = np.load(os.path.join(DAMAGED, "damaged_pixels.npz"))[name]
    rc, px = oracle.decode(open(os.path.join(DAMAGED, name + ".jpg"), "rb").read())
    assert rc == 0
    assert np.array_equal(px.reshape(want.shape), want)


@pytest.mark.parametrize("damage", oracle_binding.RESTART_DAMAGES)
def test_oracle_resynchronises_like_the_reference(oracle, built, damage):
    """Restart markers out of sequence, missing, duplicated, buried in garbage: same verdict and same pixels as the reference."""
    ref = reference_decode("damage", damage)
    rc, px = oracle.decode(damaged_stream(damage))
    if ref is None:
        assert rc != 0
    else:
        assert rc == 0 and same_pixels(px, ref)


DEEP12 = os.path.join(GOLDEN, "deep12")
D12NAMES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(DEEP12, "*.jpg")))


@pytest.mark.parametrize("name", D12NAMES)
def test_oracle_matches_12bit_golden(oracle, name):
    """SURVEY 8f4 groundwork: 12-bit frames (SOF1 and SOF2) into 16-bit samples, level shift 2048, clamp 4095."""
    want = np.load(os.path.join(DEEP12, "deep12_pixels.npz"))[name]
    data = open(os.path.join(DEEP12, name + ".jpg"), "rb").read()
    rc, px = oracle.decode16(data)
    assert rc == 0 and px.dtype == np.uint16
    assert np.array_equal(px, want)
    rc8, _ = oracle.decode(data)   # one byte per sample cannot hold a 12-bit frame
    assert rc8 == -1024


def test_oracle_16bit_output_of_8bit_frames(oracle, golden_pixels):
    for name in NAMES[:4]:
        rc, px = oracle.decode16(open(os.path.join(GOLDEN, name + ".jpg"), "rb").read())
        assert rc == 0 and np.array_equal(px.reshape(golden_pixels[name].shape), golden_pixels[name].astype(np.uint16))


def test_progressive_golden_is_complete():
    assert len(PNAMES) >= 7
    assert set(np.load(os.path.join(PROGRESSIVE, "progressive_pixels.npz")).files) == set(PNAMES)


@pytest.mark.parametrize("flags,w,h,sub,z", VARIANTS)
def test_oracle_matches_reference_on_stream_variants(oracle, built, flags, w, h, sub, z):
    """One scan per component (flag 1), SOF1 header (2), 16-bit DQT (4): accepted by the reference, same pixels."""
    ref = reference_decode("variant", (flags, w, h, sub, z))
    assert ref is not None
    rc, px = oracle.decode(variant_stream(flags, w, h, sub, z))
    assert rc == 0 and same_pixels(px, ref)


NOEOI = os.path.join(GOLDEN, "noeoi")
NENAMES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(NOEOI, "*.jpg")))


@pytest.mark.parametrize("name", NENAMES)
def test_oracle_matches_reference_on_streams_without_eoi(oracle, name):
    """Streams cut off at the end (no EOI, possibly inside the entropy coded data): the reference only warns when nothing but
    the tail of the LAST restart interval is missing (Frame::ParseTrailer marker/frame.cpp:1089, zero bits behind the end of
    the data io/bitstream.cpp:103-105) and fails with UNEXPECTED_EOF when a restart marker it needs is gone
    (entropyparser.cpp:141-147). The fixtures hold the reference's verdict and pixels (make_noeoi.py)."""
    import json
    status = json.load(open(os.path.join(NOEOI, "noeoi_status.json")))[name]
    rc, px = oracle.decode(open(os.path.join(NOEOI, name + ".jpg"), "rb").read())
    assert rc == status
    if status == 0:
        want = np.load(os.path.join(NOEOI, "noeoi_pixels.npz"))[name]
        assert np.array_equal(px.reshape(want.shape), want)


def test_noeoi_fixtures_cover_both_verdicts():
    import json
    status = json.load(open(os.path.join(NOEOI, "noeoi_status.json")))
    assert sorted(status) == NENAMES and 0 in status.values() and -1025 in status.values()


def test_zrl_that_steps_over_position_63_ends_the_block_silently(oracle):
    """sequentialscan.cpp:717-719: after a ZRL the reference re-tests k <= 63 and leaves the block without an error."""
    ref = reference_decode("zrl", ())
    assert ref is not None
    rc, px = oracle.decode(oracle_binding.zrl_overrun_stream())
    assert rc == 0 and same_pixels(px, ref)


DNL = os.path.join(GOLDEN, "dnl")
DNLNAMES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(DNL, "*.jpg")))


@pytest.mark.parametrize("name", DNLNAMES)
def test_oracle_reads_the_height_from_the_dnl_marker(oracle, name):
    """SOF height 0 + DNL behind the first scan (entropyparser.cpp:204-249): the pixels the reference delivers for the same
    image with the height in the SOF; the reference's own decode of the DNL stream differs from that in its last pixel row
    only (its upsampler is sized before the DNL arrives -- make_dnl.py), which is not restated."""
    px = np.load(os.path.join(DNL, "dnl_pixels.npz"))
    rc, got = oracle.decode(open(os.path.join(DNL, name + ".jpg"), "rb").read())
    assert rc == 0 and np.array_equal(got, px[name])
    assert np.array_equal(got[:-1], px[name + "__ref_dnl"][:-1])


@pytest.mark.parametrize("w,h,sub,z", FOUR_COMPONENT)
def test_oracle_matches_reference_on_four_component_streams(oracle, built, w, h, sub, z):
    ref = reference_decode("four", (w, h, sub, z))
    assert ref is not None and ref["shape"][2] == 4
    rc, px = oracle.decode(four_component_stream(w, h, sub, z))
    assert rc == 0 and same_pixels(px, ref)


@pytest.mark.parametrize("name", NO_COLOR_TRANSFORM)
def test_oracle_without_color_transform_matches_reference_cli(oracle, name):
    """JPGTAG_MATRIX_LTRAFO = none (`jpeg -c` on decoding, cmd/main.cpp / reconstruct.cpp:336): Y, Cb, Cr upsampled, untransformed."""
    ref = reference_decode("nocolor", name)
    rc, px = oracle.decode_without_color_transform(open(os.path.join(GOLDEN, name + ".jpg"), "rb").read())
    assert rc == 0 and same_pixels(px, ref)


def test_oracle_planes_match_reference_without_upsampling(oracle):
    """JPGTAG_DECODER_UPSAMPLE = false (bitmapctrl.cpp:273-293, blockbitmaprequester.cpp:1013-1074): every component as a plane
    at its own resolution == what `oracle/_ref/jpeg -U -c` wrote (tests/golden/planes.npz, make_planes.py)."""
    fx = np.load(os.path.join(GOLDEN, "planes.npz"))
    names = sorted({k.rsplit("__", 1)[0] for k in fx.files})
    assert len(names) >= 12
    for name in names:
        data = open(os.path.join(GOLDEN, name.replace("__", "/") + ".jpg"), "rb").read()
        rc, planes = oracle.decode_planes(data)
        assert rc == 0
        for c, p in enumerate(planes):
            assert np.array_equal(p, fx["%s__%d" % (name, c)]), (name, c)


XT = os.path.join(GOLDEN, "xt")
XTNAMES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(XT, "*.jpg")))


def test_xt_fixture_set():
    assert len([n for n in XTNAMES if not n.endswith("__nimpl")]) >= 8 and len([n for n in XTNAMES if n.endswith("__nimpl")]) >= 3


@pytest.mark.parametrize("name", XTNAMES)
def test_oracle_merges_the_xt_residual_layer(oracle, name):
    """SURVEY 8f3 / VERDICT r1 #9, oracle first: JPEG XT streams with a residual codestream (RESI box) and a merging
    specification (SPEC box), written and decoded by the reference (tests/golden/xt, make_xt.py): base image + residual image
    through YCbCrTrafo::YCbCr2RGB's merge (colortrafo/ycbcrtrafo.cpp:747-880) == the reference's pixels; profiles outside the
    restated one (lossless residual, 12-bit residual, refinement scans) are NOT_IMPLEMENTED, never decoded as plain JPEG."""
    data = open(os.path.join(XT, name + ".jpg"), "rb").read()
    assert oracle.lib.jpgo_has_xt_layer(bytes(data), len(data)) == 1
    rc, px = oracle.decode(data)
    if name.endswith("__nimpl"):
        assert rc == -1034
        return
    want = np.load(os.path.join(XT, "xt_pixels.npz"))[name]
    assert rc == 0 and np.array_equal(px.reshape(want.shape), want)
    # the base layer alone (what a legacy decoder shows) is a different image: the merge is not a no-op
    base = bytearray(data)
    at = base.find(b"SPEC")
    base[at:at + 4] = b"free"
    at = base.find(b"RESI")
    while at >= 0:
        base[at:at + 4] = b"free"
        at = base.find(b"RESI", at)
    rc2, legacy = oracle.decode(bytes(base))
    assert rc2 == -1034 or not np.array_equal(legacy.reshape(want.shape), want)


def test_plain_streams_have_no_xt_layer(oracle):
    for name in NAMES[:3]:
        data = open(os.path.join(GOLDEN, name + ".jpg"), "rb").read()
        assert oracle.lib.jpgo_has_xt_layer(data, len(data)) == 0
