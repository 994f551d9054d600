"""GPU: the CUDA path (through the C ABI) against the golden vectors, the oracle, and size-independent
properties at the benchmark's frame sizes."""
import glob
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
NAMES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.jpg")))


def gpu_decode(built, frames, **kw):
    import torch
    dec = built.BatchDecoder(frames, **kw)
    out = dec.new_output()
    out.fill_(0x5A)
    dec.upload()
    dec.decode(out)
    torch.cuda.synchronize()
    return dec, out


@pytest.fixture(scope="module")
def golden_pixels():
    return np.load(os.path.join(GOLDEN, "golden_pixels.npz"))


@pytest.mark.parametrize("name", NAMES)
def test_golden_vector_bit_exact(built, golden_pixels, name):
    data = open(os.path.join(GOLDEN, name + ".jpg"), "rb").read()
    dec, out = gpu_decode(built, [data])
    assert dec.status(0) == 0
    px = dec.frame_view(out, 0).cpu().numpy()
    ref = golden_pixels[name]
    assert px.shape == ref.shape
    assert np.array_equal(px, ref), "%d differing bytes" % int((px != ref).sum())


def test_golden_vectors_as_one_heterogeneous_batch(built, golden_pixels):
    """All fixtures in ONE batch: different geometries, samplings and tables -> several launch classes."""
    datas = [open(os.path.join(GOLDEN, n + ".jpg"), "rb").read() for n in NAMES]
    dec, out = gpu_decode(built, datas)
    for i, n in enumerate(NAMES):
        assert dec.status(i) == 0
        assert np.array_equal(dec.frame_view(out, i).cpu().numpy(), golden_pixels[n]), n


@pytest.mark.parametrize("name", ["c420_96x80_z6_q75", "c444_64x64_z16_q90", "c420_130x70_z9_q98", "g_40x24_z2_q75"])
def test_coefficients_match_oracle(built, oracle, name):
    """Stage (a) alone: dequantised int16 coefficients == oracle's quantised coefficients * delta."""
    import torch
    data = open(os.path.join(GOLDEN, name + ".jpg"), "rb").read()
    dec = built.BatchDecoder([data])
    dec.upload()
    dec.decode_entropy()
    torch.cuda.synchronize()
    assert dec.status(0) == 0
    rc, s, planes = oracle.coefficients(data)
    assert rc == 0
    for c in range(s.ncomp):
        q = np.array(s.quant[s.tq[c]], dtype=np.int32).reshape(8, 8)
        want = planes[c] * q
        got = dec.coefficients(0, c).astype(np.int32)
        assert np.array_equal(got, want), "component %d" % c


@pytest.mark.parametrize("w,h,sub,z,q", [(1920, 1080, (2, 2), 120, 75), (3840, 2160, (2, 2), 240, 75), (512, 512, (1, 1), 256, 90),
                                          (641, 479, (2, 2), 13, 75), (333, 200, (2, 1), 0, 60)])
def test_synthetic_frames_match_oracle(built, oracle, w, h, sub, z, q):
    """Benchmark-sized frames (cfg2/cfg3 geometry) from the in-repo generator: GPU pixels == oracle pixels."""
    from libjpeg_b200 import synth
    data = synth.encode(synth.source_image(w, h, 11), q, sub, z)
    dec, out = gpu_decode(built, [data])
    assert dec.status(0) == 0
    rc, ref = oracle.decode(data.tobytes())
    assert rc == 0
    assert np.array_equal(dec.frame_view(out, 0).cpu().numpy(), ref)


def test_batch_of_identical_geometry_is_frame_independent(built, oracle):
    """Checksum-of-checksums property at batch scale: every copy of a frame decodes to the same bytes, and
    distinct frames to their own oracle result, whatever their position in the batch."""
    import torch
    from libjpeg_b200 import synth
    base = [synth.encode(synth.source_image(320, 176, s), 75, (2, 2), 20) for s in (1, 2, 3)]
    frames = [base[i % 3] for i in range(96)]
    dec, out = gpu_decode(built, frames)
    refs = [oracle.decode(b.tobytes())[1] for b in base]
    for i in range(96):
        assert dec.status(i) == 0
        assert np.array_equal(dec.frame_view(out, i).cpu().numpy(), refs[i % 3]), i
    # and decode is idempotent: a second run over the same batch gives the same buffer
    out2 = dec.new_output()
    dec.decode(out2)
    torch.cuda.synchronize()
    for i in range(96):
        assert torch.equal(dec.frame_view(out, i), dec.frame_view(out2, i))


@pytest.mark.parametrize("w,h,sub,z,dcq,copies", [(96, 80, (2, 2), 3, 255, 1), (200, 120, (2, 1), 0, 160, 1), (64, 64, (1, 1), 4, 255, 1),
                                                   (130, 70, (1, 2), 2, 200, 1), (320, 176, (2, 2), 20, 255, 5), (640, 360, (2, 2), 40, 160, 3)])
def test_samples_beyond_the_fast_ranges_match_oracle(built, oracle, w, h, sub, z, dcq, copies):
    """DC quantiser 255 on a full-range image: chroma samples beyond int16 (narrow planes) and luma / chroma beyond
    +-65535 (32-bit colour arithmetic) -- the exact paths (int32 planes, 64-bit colour) must give the reference's
    pixels; ordinary frames in the same batch must be unaffected."""
    from libjpeg_b200 import synth
    normal = synth.encode(synth.source_image(w, h, 5), 75, sub, z)
    from tests import oracle_binding
    hot = oracle_binding.with_dc_quantiser(normal, dcq)
    frames = []
    for _ in range(copies):
        frames += [normal, hot]
    dec, out = gpu_decode(built, frames)
    rc_n, ref_n = oracle.decode(normal.tobytes())
    rc_h, ref_h = oracle.decode(hot)
    assert rc_n == 0 and rc_h == 0
    assert not np.array_equal(ref_n, ref_h)
    for i, fr in enumerate(frames):
        assert dec.status(i) == 0
        assert np.array_equal(dec.frame_view(out, i).cpu().numpy(), ref_h if i & 1 else ref_n), i


def _damaged_fixtures():
    d = os.path.join(GOLDEN, "damaged")
    px = np.load(os.path.join(d, "damaged_pixels.npz"))
    return [(n, open(os.path.join(d, n + ".jpg"), "rb").read(), px[n]) for n in sorted(px.files)]


def test_truncated_streams_match_reference_fixtures(built):
    """Streams that end where a restart marker should stand: the reference marks the remaining intervals invalid and
    clears their MCUs (entropyparser.cpp:137-199, sequentialscan.cpp:415-419); the fixtures hold ITS pixels (the oracle
    only restates the in-sequence case)."""
    fx = _damaged_fixtures()
    dec, out = gpu_decode(built, [f[1] for f in fx])
    for i, (name, _, want) in enumerate(fx):
        assert dec.status(i) == 0, name
        got = dec.frame_view(out, i).cpu().numpy()
        assert np.array_equal(got.reshape(want.shape), want), name


def test_device_restart_index_equals_host_index(built, oracle, monkeypatch):
    """SURVEY 8f1: the restart index built by restart_index_kernel (default for interleaved scans with restart markers)
    against the host memchr walk (B200JPG_HOST_INDEX=1), the oracle and the reference's fixtures -- plain streams, fill
    bytes in front of markers, truncated streams, trailing bytes behind EOI, restart ids out of sequence."""
    import torch
    from libjpeg_b200 import synth
    from tests import oracle_binding
    a = synth.encode(synth.source_image(200, 136, 3), 75, (2, 2), 2)          # 59 intervals, ids wrap around
    b_ = synth.encode(synth.source_image(96, 80, 5), 80, (2, 1), 3).tobytes()
    c = synth.encode(synth.source_image(640, 360, 9), 75, (2, 2), 40).tobytes()   # intervals of several KB
    valid = [a.tobytes(), oracle_binding.with_fill_bytes(a, 2, 1), oracle_binding.with_fill_bytes(a, 3, 7), b_, c,
             a.tobytes() + b"\x00\x11\x22" * 5]
    fx = _damaged_fixtures()
    frames = valid + [f[1] for f in fx]
    dec, out = gpu_decode(built, frames, tolerate_bad=True)
    monkeypatch.setenv("B200JPG_HOST_INDEX", "1")
    dec_h, out_h = gpu_decode(built, frames, tolerate_bad=True)
    monkeypatch.delenv("B200JPG_HOST_INDEX")
    torch.cuda.synchronize()
    for i, fr in enumerate(frames):
        if i < len(valid):
            rc, want = oracle.decode(fr)
            assert rc == 0
        else:
            want = fx[i - len(valid)][2]
        assert dec.status(i) == 0 and dec_h.status(i) == 0, i
        assert np.array_equal(dec.frame_view(out, i).cpu().numpy().reshape(want.shape), want), i
        assert torch.equal(dec.frame_view(out, i), dec_h.frame_view(out_h, i)), i


def test_restart_marker_resynchronisation_matches_oracle(built, oracle, monkeypatch):
    """VERDICT r1 1(d): restart markers out of sequence, missing, duplicated, buried in garbage, streams cut inside an interval
    -- the reference resynchronises (entropyparser.cpp:137-199; the oracle restates it and is pinned on the reference for
    exactly these damages in tests/test_oracle.py). Device-side index (one thread replays the marker sequence) and host-side
    index: the oracle's verdict and the oracle's pixels."""
    import torch
    from libjpeg_b200 import synth
    from tests import oracle_binding
    srcs = [synth.encode(synth.source_image(200, 136, 3), 75, (2, 2), 2), synth.encode(synth.source_image(96, 80, 5), 80, (2, 1), 3),
            synth.encode(synth.source_image(64, 64, 6), 90, (1, 1), 4, 1)]  # the last one: one scan per component (host index)
    frames, labels = [], []
    for si, src in enumerate(srcs):
        for damage in oracle_binding.RESTART_DAMAGES:
            frames.append(oracle_binding.with_restart_damage(src, damage))
            labels.append((si, damage))
    # a stream with more restart markers than intervals AND ids out of sequence is beyond the marker list the index kernel
    # keeps: not part of this list (documented deviation, DESIGN.md)
    dec, out = gpu_decode(built, frames, tolerate_bad=True)
    monkeypatch.setenv("B200JPG_HOST_INDEX", "1")
    dec_h, out_h = gpu_decode(built, frames, tolerate_bad=True)
    monkeypatch.delenv("B200JPG_HOST_INDEX")
    torch.cuda.synchronize()
    verdicts = set()
    for i, fr in enumerate(frames):
        rc, want = oracle.decode(fr)
        verdicts.add(rc)
        assert dec.status(i) == rc and dec_h.status(i) == rc, (labels[i], rc, dec.status(i), dec_h.status(i))
        if rc == 0:
            assert np.array_equal(dec.frame_view(out, i).cpu().numpy(), want), labels[i]
            assert np.array_equal(dec_h.frame_view(out_h, i).cpu().numpy(), want), labels[i]
    assert 0 in verdicts and -1025 in verdicts


PROGRESSIVE = os.path.join(GOLDEN, "progressive")
PNAMES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(PROGRESSIVE, "*.jpg")))


@pytest.mark.parametrize("name", PNAMES)
def test_progressive_golden_vector_bit_exact(built, name):
    """SURVEY 8f2: SOF2 streams of the reference encoder (DC first, AC bands, DC / AC refinement) through the progressive
    scan kernels + dequantisation + the same stage b: the reference's pixels."""
    want = np.load(os.path.join(PROGRESSIVE, "progressive_pixels.npz"))[name]
    dec, out = gpu_decode(built, [open(os.path.join(PROGRESSIVE, name + ".jpg"), "rb").read()])
    assert dec.status(0) == 0
    assert np.array_equal(dec.frame_view(out, 0).cpu().numpy().reshape(want.shape), want)


def test_progressive_coefficients_and_mixed_batch(built, oracle, golden_pixels):
    """Quantised levels after all scans x quantiser == the oracle's planes; progressive and sequential frames share a batch."""
    prog = [open(os.path.join(PROGRESSIVE, n + ".jpg"), "rb").read() for n in PNAMES]
    base = [open(os.path.join(GOLDEN, n + ".jpg"), "rb").read() for n in NAMES[:5]]
    frames = [prog[0], base[0], prog[3], base[1], prog[1], base[2], prog[5], base[3], prog[6], base[4], prog[2], prog[4]]
    dec, out = gpu_decode(built, frames)
    px = np.load(os.path.join(PROGRESSIVE, "progressive_pixels.npz"))
    order = [("p", 0), ("b", 0), ("p", 3), ("b", 1), ("p", 1), ("b", 2), ("p", 5), ("b", 3), ("p", 6), ("b", 4), ("p", 2), ("p", 4)]
    for i, (kind, j) in enumerate(order):
        want = px[PNAMES[j]] if kind == "p" else golden_pixels[NAMES[j]]
        assert dec.status(i) == 0, i
        assert np.array_equal(dec.frame_view(out, i).cpu().numpy().reshape(want.shape), want), (i, kind, j)
    rc, s, planes = oracle.coefficients(prog[0])
    assert rc == 0
    for c in range(s.ncomp):
        q = np.array(s.quant[s.tq[c]], dtype=np.int32).reshape(8, 8)
        assert np.array_equal(dec.coefficients(0, c).astype(np.int32), planes[c] * q), "component %d" % c


def test_corrupt_stream_is_reported_not_crashing(built):
    from libjpeg_b200 import synth
    good = synth.encode(synth.source_image(128, 64, 5), 75, (2, 2), 8)
    bad = bytearray(good.tobytes())
    i = bad.find(b"\xff\xda") + 14
    for k in range(i + 40, i + 400):
        if bad[k] != 0xFF and bad[k - 1] != 0xFF:
            bad[k] = 0xF7  # mostly-ones bytes: runs the decoder into invalid / overlong codes
    dec, out = gpu_decode(built, [good.tobytes(), bytes(bad)])
    assert dec.status(0) == 0
    assert dec.status(1) in (0, -1038, -1025)  # reported per frame; the good frame is untouched


def test_truncated_stream_zero_fills_missing_intervals(built, oracle):
    """A stream that ends early: intervals the file does not contain decode as zero blocks (the reference
    greys out an invalid segment, sequentialscan.cpp:415-419) and the intervals before stay bit-exact."""
    from libjpeg_b200 import synth
    good = synth.encode(synth.source_image(128, 128, 9), 75, (2, 2), 8).tobytes()
    rc, ref = oracle.decode(good)
    cut = good.rfind(b"\xff\xd3")  # drop everything from the 4th restart marker on
    trunc = good[:cut] + b"\xff\xd9"
    dec, out = gpu_decode(built, [trunc])
    assert dec.status(0) == 0
    px = dec.frame_view(out, 0).cpu().numpy()
    assert np.array_equal(px[:48], ref[:48])  # 4 intervals of one 16-row MCU row each, minus the filter halo row


def test_dropin_client_through_cpp_interface(built, golden_pixels, tmp_path):
    """The reference-style stripe client (tests/client/stripe_client.cpp), compiled against include/interface and
    linked to libb200jpg.so: JPEG::Read / GetInformation / DisplayRectangle in 8-row stripes via the BitMapHook."""
    import subprocess
    lib_dir = os.path.join(ROOT, "libjpeg_b200")
    exe = str(tmp_path / "stripe_b200")
    subprocess.run(["g++", "-O1", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "client", "stripe_client.cpp"),
                    "-L" + lib_dir, "-lb200jpg", "-Wl,-rpath," + lib_dir, "-o", exe], check=True)
    for name in NAMES:
        if name.startswith("cfg1"):
            continue
        out = str(tmp_path / (name + ".pnm"))
        r = subprocess.run([exe, os.path.join(GOLDEN, name + ".jpg"), out], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        data = open(out, "rb").read()
        magic, dims, maxv, rest = data.split(b"\n", 3)
        w, h = map(int, dims.split())
        px = np.frombuffer(rest, dtype=np.uint8).reshape(h, w, 3 if magic == b"P6" else 1)
        assert np.array_equal(px, golden_pixels[name]), name
        depth = px.shape[2]
        stripes = (h + 7) // 8
        assert "requests=%d releases=%d" % (stripes * depth, stripes * depth) in r.stdout


@pytest.mark.parametrize("flags,w,h,sub,z", [(1, 70, 50, (2, 2), 5), (1, 64, 48, (1, 1), 0), (2, 40, 40, (2, 2), 3), (6, 40, 40, (2, 1), 0),
                                            (7, 33, 47, (1, 2), 4), (1, 1920, 1080, (2, 2), 40)])
def test_stream_variants_match_oracle(built, oracle, flags, w, h, sub, z):
    """Non-interleaved scans (each component its own scan and restart index), SOF1 headers, 16-bit quantisation tables."""
    from libjpeg_b200 import synth
    data = synth.encode(synth.source_image(w, h, 5), 80, sub, z, flags)
    dec, out = gpu_decode(built, [data])
    assert dec.status(0) == 0
    assert dec.info(0).nscans == (3 if flags & 1 else 1)
    rc, ref = oracle.decode(data.tobytes())
    assert rc == 0
    assert np.array_equal(dec.frame_view(out, 0).cpu().numpy(), ref)


def test_streams_without_eoi_match_reference_fixtures(built):
    """tests/golden/noeoi (make_noeoi.py): the tail of the stream is cut off. The reference's verdict -- pixels when only
    the tail of the last restart interval is gone (zero bits behind the end of the data), UNEXPECTED_EOF when a restart
    marker it needs is gone -- and its pixels, through the CUDA path."""
    import json
    d = os.path.join(GOLDEN, "noeoi")
    status = json.load(open(os.path.join(d, "noeoi_status.json")))
    px = np.load(os.path.join(d, "noeoi_pixels.npz"))
    names = sorted(status)
    dec, out = gpu_decode(built, [open(os.path.join(d, n + ".jpg"), "rb").read() for n in names], tolerate_bad=True)
    for i, n in enumerate(names):
        assert dec.status(i) == status[n], n
        if status[n] == 0:
            want = px[n]
            assert np.array_equal(dec.frame_view(out, i).cpu().numpy().reshape(want.shape), want), n


def test_zrl_that_steps_over_position_63_ends_the_block_silently(built, oracle):
    """sequentialscan.cpp:717-719 (ADVICE r1): no error, the block just ends; a coefficient whose run leaves the block is
    still MALFORMED_STREAM (:764-766)."""
    from tests import oracle_binding
    good = oracle_binding.zrl_overrun_stream()
    # DC +1, AC (0/1) at k = 1, three ZRLs (k = 50), twelve times run 0 size 1 (k = 62), then run 2 size 1: k = 64 leaves the block
    bad = oracle_binding.handmade_grey_stream("10" + "1" + "110" + "1" + "000" + ("110" + "1") * 12 + "1110" + "1")
    dec, out = gpu_decode(built, [good, bad], tolerate_bad=True)
    rc, want = oracle.decode(good)
    assert rc == 0 and dec.status(0) == 0
    assert np.array_equal(dec.frame_view(out, 0).cpu().numpy(), want)
    rc_bad, _ = oracle.decode(bad)
    assert rc_bad == -1038 and dec.status(1) == -1038


def _bench_frames(workload, distinct):
    from tools import bench_inputs
    if (bench_inputs.WORKLOADS[workload][5] or workload in bench_inputs.EXTRA_ARGS) and not bench_inputs.have_reference_encoder():
        pytest.skip("these inputs need the reference encoder (oracle/_ref/jpeg)")
    return bench_inputs.make_frames(workload, distinct, workers=min(16, os.cpu_count() or 1))


@pytest.mark.parametrize("workload,distinct", [("cfg3", 64), ("cfg2", 16), ("cfg1", 4)])
def test_every_distinct_bench_frame_matches_oracle(built, oracle, workload, distinct):
    """VERDICT r1 1(a,b): the benchmark's own inputs -- S(w,h,seed), seeds 1..distinct, written by the REFERENCE ENCODER
    (tools/bench_inputs.py; the repo's generator only where oracle/_ref/jpeg is absent) -- every one of them: GPU pixels ==
    oracle pixels, bit for bit."""
    frames = _bench_frames(workload, distinct)
    dec, out = gpu_decode(built, frames)
    for i, f in enumerate(frames):
        assert dec.status(i) == 0, i
        rc, want = oracle.decode(f)
        assert rc == 0
        got = dec.frame_view(out, i).cpu().numpy()
        assert np.array_equal(got, want), "%s frame %d (seed %d): %d differing bytes" % (workload, i, i + 1, int((got != want).sum()))


def test_xt_8k_bench_frame_matches_oracle(built, oracle):
    """BASELINE configs[4] geometry: one 8192x8192 frame of bench.py's cfg5 workload (4:2:0 q75 base with restart markers + 4:4:4
    q90 residual codestream in RESI boxes spread over hundreds of APP11 markers), pixels == oracle."""
    frames = _bench_frames("cfg5", 1)
    dec, out = gpu_decode(built, frames)
    assert dec.status(0) == 0
    rc, want = oracle.decode(frames[0])
    assert rc == 0 and want.shape == (8192, 8192, 3)
    got = dec.frame_view(out, 0).cpu().numpy()
    assert np.array_equal(got, want), "%d differing bytes" % int((got != want).sum())


def test_progressive_4k_frames_match_oracle(built, oracle):
    """VERDICT r1 1(c): BASELINE configs[3] geometry -- 3840x2160 4:2:0 q75 SOF2 streams of the reference encoder (ten scans,
    DRI 240), pixels and dequantised coefficients == oracle."""
    frames = _bench_frames("cfg4", 3)
    dec, out = gpu_decode(built, frames)
    for i, f in enumerate(frames):
        assert dec.status(i) == 0 and dec.info(i).nscans >= 8
        rc, want = oracle.decode(f)
        assert rc == 0
        assert np.array_equal(dec.frame_view(out, i).cpu().numpy(), want), i
    rc, s, planes = oracle.coefficients(frames[0])
    assert rc == 0
    for c in range(s.ncomp):
        q = np.array(s.quant[s.tq[c]], dtype=np.int32).reshape(8, 8)
        assert np.array_equal(dec.coefficients(0, c).astype(np.int32), planes[c] * q), "component %d" % c


def test_reference_cli_linked_against_the_b200_library(built, golden_pixels, tmp_path):
    """SURVEY 8b's acceptance test: the reference's OWN command line client (cmd/main.cpp, reconstruct.cpp, bitmaphook.cpp,
    filehook.cpp -- compiled unmodified by oracle/Makefile) linked against libb200jpg.so instead of the reference library:
    `jpeg_b200 in.jpg out.ppm` = Read with DECODER_STOP flags, PeekMarker, GetInformation, 8-row DisplayRectangle stripes
    with the reference's BitMapHook. Its output files must hold the reference's pixels."""
    import subprocess
    exe = os.path.join(ROOT, "oracle", "_ref", "jpeg_b200")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/jpeg_b200 is built where the reference build exists (oracle/Makefile)")
    for name in NAMES:
        out = str(tmp_path / (name + ".pnm"))
        r = subprocess.run([exe, os.path.join(GOLDEN, name + ".jpg"), out], capture_output=True, text=True)
        assert r.returncode == 0 and "failed" not in r.stdout + r.stderr, (name, r.stdout[-300:], r.stderr[-300:])
        data = open(out, "rb").read()
        magic, dims, maxv, rest = data.split(b"\n", 3)
        w, h = map(int, dims.split())
        px = np.frombuffer(rest, dtype=np.uint8).reshape(h, w, 3 if magic == b"P6" else 1)
        want = golden_pixels[name]
        assert np.array_equal(px.reshape(want.shape), want), name


def test_region_client_matches_reference_fixtures(built, tmp_path):
    """VERDICT r1 #10: horizontal crops (DECODER_MINX / MAXX), planar client bitmaps (BytesPerPixel = 1) and a BitMapHook that
    returns an error, through tests/client/region_client.cpp linked against libb200jpg.so -- byte for byte the canvas, and the
    same report line (ok flag, LastError code, number of hook requests), that the same client got from the unmodified
    reference (tests/golden/regions.npz, make_regions.py)."""
    import subprocess
    import sys
    sys.path.insert(0, GOLDEN)
    import make_regions
    fx = np.load(os.path.join(GOLDEN, "regions.npz"))
    lib_dir = os.path.join(ROOT, "libjpeg_b200")
    exe = str(tmp_path / "region_b200")
    subprocess.run(["g++", "-O1", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "client", "region_client.cpp"),
                    "-L" + lib_dir, "-lb200jpg", "-Wl,-rpath," + lib_dir, "-o", exe], check=True)
    for key, name, args in make_regions.CASES:
        raw = str(tmp_path / "o.raw")
        r = subprocess.run([exe, os.path.join(GOLDEN, name + ".jpg"), raw] + args, capture_output=True, text=True)
        assert r.returncode == 0, (key, r.stderr)
        assert r.stdout.strip() == bytes(fx[key + "__report"]).decode(), key
        assert np.array_equal(np.fromfile(raw, dtype=np.uint8), fx[key]), key


@pytest.mark.parametrize("workload,distinct", [("cfg2n", 6), ("cfg3n", 4)])
def test_restartless_reference_encoded_frames_match_oracle(built, oracle, workload, distinct):
    """VERDICT r1 #6: 1080p / 4K 4:2:0 frames of the reference encoder WITHOUT -z (no restart markers): the scan is cut at
    synchronisation points found on the device (spec_sync_kernel) and decoded one work item per lane. Pixels == oracle."""
    frames = _bench_frames(workload, distinct)
    dec, out = gpu_decode(built, frames)
    for i, f in enumerate(frames):
        assert dec.info(i).restart_interval == 0 and dec.info(i).n_intervals == 1
        assert dec.status(i) == 0, i
        rc, want = oracle.decode(f)
        assert rc == 0
        got = dec.frame_view(out, i).cpu().numpy()
        assert np.array_equal(got, want), "%s frame %d: %d differing bytes" % (workload, i, int((got != want).sum()))


def test_restartless_variants_match_oracle(built, oracle, monkeypatch):
    """Restart-less scans of every supported sampling, odd sizes, one scan per component, a stream cut short (with and
    without EOI) and the single-work-item path (B200JPG_NO_SPEC) for comparison -- all in one heterogeneous batch."""
    import torch
    from libjpeg_b200 import synth
    cases = [(640, 360, (2, 2), 75, 0), (333, 201, (2, 1), 60, 0), (512, 512, (1, 1), 90, 0), (97, 161, (1, 2), 98, 0), (1000, 300, (2, 2), 30, 0),
             (400, 300, (2, 2), 85, 1), (256, 256, (1, 1), 95, 1)]
    frames = [synth.encode(synth.source_image(w, h, 3 + i), q, sub, 0, fl).tobytes() for i, (w, h, sub, q, fl) in enumerate(cases)]
    big = frames[0]
    frames.append(big[:len(big) * 2 // 3] + b"\xff\xd9")  # cut inside the entropy coded data, EOI appended
    frames.append(big[:len(big) * 2 // 3])                # ... and without
    dec, out = gpu_decode(built, frames, tolerate_bad=True)
    monkeypatch.setenv("B200JPG_NO_SPEC", "1")
    dec1, out1 = gpu_decode(built, frames, tolerate_bad=True)
    monkeypatch.delenv("B200JPG_NO_SPEC")
    torch.cuda.synchronize()
    for i, f in enumerate(frames):
        rc, want = oracle.decode(f)
        assert dec.status(i) == rc and dec1.status(i) == rc, (i, rc, dec.status(i), dec1.status(i))
        if rc == 0:
            assert np.array_equal(dec.frame_view(out, i).cpu().numpy(), want), i
            assert np.array_equal(dec1.frame_view(out1, i).cpu().numpy(), want), i


def test_dnl_streams_match_reference_fixtures(built):
    """SURVEY 8f4: frame height in a DNL marker behind the first scan (tests/golden/dnl, make_dnl.py)."""
    d = os.path.join(GOLDEN, "dnl")
    px = np.load(os.path.join(d, "dnl_pixels.npz"))
    names = sorted(n for n in px.files if not n.endswith("__ref_dnl"))
    dec, out = gpu_decode(built, [open(os.path.join(d, n + ".jpg"), "rb").read() for n in names])
    for i, n in enumerate(names):
        assert dec.status(i) == 0, n
        got = dec.frame_view(out, i).cpu().numpy()
        assert np.array_equal(got, px[n]), n
        assert np.array_equal(got[:-1], px[n + "__ref_dnl"][:-1]), n


def test_fused_420_reconstruction_matches_oracle(built, oracle, golden_pixels, monkeypatch):
    """The single-kernel reconstruction of 4:2:0 frames (B200JPG_FUSED=1: chroma IDCT into a shared-memory ring, no sample
    planes) on the 4:2:0 goldens, odd sizes, frames whose samples leave the int16 / 32-bit colour ranges, and benchmark frames."""
    from libjpeg_b200 import synth
    from tests import oracle_binding
    monkeypatch.setenv("B200JPG_FUSED", "1")
    names = [n for n in NAMES if n.startswith("c420")]
    frames = [open(os.path.join(GOLDEN, n + ".jpg"), "rb").read() for n in names]
    want = [golden_pixels[n] for n in names]
    for (w, h, z, dcq) in [(641, 479, 13, 0), (96, 80, 3, 255), (640, 360, 40, 160), (1920, 1080, 120, 0), (3840, 2160, 240, 0), (260, 20, 0, 0)]:
        f = synth.encode(synth.source_image(w, h, 5), 75, (2, 2), z)
        f = oracle_binding.with_dc_quantiser(f, dcq) if dcq else f.tobytes()
        rc, px = oracle.decode(f)
        assert rc == 0
        frames.append(f)
        want.append(px)
    dec, out = gpu_decode(built, frames)
    for i in range(len(frames)):
        assert dec.status(i) == 0, i
        assert np.array_equal(dec.frame_view(out, i).cpu().numpy().reshape(want[i].shape), want[i]), i


def test_progressive_scan_by_scan_path_matches_fixtures(built, monkeypatch):
    """The progressive goldens again with the component-fused kernels switched off (B200JPG_NO_PFUSE): the scan-by-scan kernels
    of progressive_sm100.cu serve scan scripts the fused path does not take, and stay pinned on the same reference pixels."""
    monkeypatch.setenv("B200JPG_NO_PFUSE", "1")
    px = np.load(os.path.join(PROGRESSIVE, "progressive_pixels.npz"))
    dec, out = gpu_decode(built, [open(os.path.join(PROGRESSIVE, n + ".jpg"), "rb").read() for n in PNAMES])
    for i, n in enumerate(PNAMES):
        assert dec.status(i) == 0, n
        assert np.array_equal(dec.frame_view(out, i).cpu().numpy().reshape(px[n].shape), px[n]), n


SUBSAMPLING = os.path.join(GOLDEN, "subsampling")
SNAMES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(SUBSAMPLING, "*.jpg")))


def test_unusual_subsampling_matches_reference_fixtures(built):
    """SURVEY 8f4: chroma factors 3 and 4, components with different factors, 4:1:1 / 4:1:0 (upsampler.cpp:171-268,310-386) --
    streams of the reference encoder, pixels of the reference decoder (tests/golden/subsampling, make_subsampling.py), through
    the generic reconstruction kernels; all of them in one batch next to an ordinary 4:2:0 frame."""
    want = np.load(os.path.join(SUBSAMPLING, "subsampling_pixels.npz"))
    frames = [open(os.path.join(SUBSAMPLING, n + ".jpg"), "rb").read() for n in SNAMES]
    frames.append(open(os.path.join(GOLDEN, "c420_96x80_z6_q75.jpg"), "rb").read())
    dec, out = gpu_decode(built, frames)
    assert len(SNAMES) >= 7
    for i, n in enumerate(SNAMES):
        assert dec.status(i) == 0, n
        got = dec.frame_view(out, i).cpu().numpy()
        assert np.array_equal(got.reshape(want[n].shape), want[n]), n
    assert np.array_equal(dec.frame_view(out, len(SNAMES)).cpu().numpy(), np.load(os.path.join(GOLDEN, "golden_pixels.npz"))["c420_96x80_z6_q75"])


@pytest.mark.parametrize("w,h,sub,z", [(64, 48, (1, 1), 4), (70, 50, (2, 2), 5), (100, 37, (2, 1), 0), (33, 90, (1, 2), 3)])
def test_four_component_frames_match_oracle(built, oracle, w, h, sub, z):
    """SURVEY 8f4: four components (no colour transformation, ycbcrtrafo.cpp:834-892). The streams are three-component ones
    with the third component's scan duplicated under a fourth id (oracle_binding.with_fourth_component; the oracle is pinned on
    the reference for exactly these in tests/test_oracle.py)."""
    from libjpeg_b200 import synth
    from tests import oracle_binding
    data = oracle_binding.with_fourth_component(synth.encode(synth.source_image(w, h, 5), 80, sub, z, 1))
    dec, out = gpu_decode(built, [data])
    assert dec.status(0) == 0 and dec.info(0).ncomp == 4
    rc, px = oracle.decode(data)
    assert rc == 0 and px.shape[2] == 4
    assert np.array_equal(dec.frame_view(out, 0).cpu().numpy(), px)


def test_color_transform_can_be_switched_off(built, oracle):
    """JPGTAG_MATRIX_LTRAFO = ..._NONE (rectanglerequest.cpp:150-152) through the request flags of the C ABI: YCbCr frames come
    out as upsampled Y, Cb, Cr (the oracle's untransformed reconstruction, pinned on `jpeg -c` in tests/test_oracle.py)."""
    names = ["c420_96x80_z6_q75", "c444_64x64_z16_q90", "c422_100x60_z5_q80", "c440_100x61_z3_q80", "c420_127x255_z7_q30"]
    frames = [open(os.path.join(GOLDEN, n + ".jpg"), "rb").read() for n in names]
    dec, out = gpu_decode(built, frames, color_transform=False)
    for i, f in enumerate(frames):
        rc, want = oracle.decode_without_color_transform(f)
        assert rc == 0 and dec.status(i) == 0
        assert np.array_equal(dec.frame_view(out, i).cpu().numpy(), want), names[i]


DEEP12 = os.path.join(GOLDEN, "deep12")
D12NAMES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(DEEP12, "*.jpg")))


@pytest.mark.parametrize("name", D12NAMES)
def test_12bit_frames_match_reference_pixels(built, oracle, name):
    """SURVEY 8f4 / VERDICT r1 #7: 12-bit frames (SOF1 and SOF2; tables.cpp:1877-1891 -- the same LONG IDCT, level shift 2048,
    clamp 4095) through the CUDA path into native-endian 16-bit samples == what the reference wrote for CTYP_UWORD bitmaps
    (tests/golden/deep12, reference-made)."""
    want = np.load(os.path.join(DEEP12, "deep12_pixels.npz"))[name]
    data = open(os.path.join(DEEP12, name + ".jpg"), "rb").read()
    dec, out = gpu_decode(built, [data, data])
    assert dec.status(0) == 0 and dec.status(1) == 0 and dec.info(0).precision == 12
    for i in range(2):
        got = dec.frame_view(out, i).cpu().numpy().view(np.uint16)
        assert np.array_equal(got.reshape(want.shape), want), (name, i)
    rc, px = oracle.decode16(data)
    assert rc == 0 and np.array_equal(px.reshape(want.shape), want)


def test_12bit_and_8bit_frames_share_a_batch(built, golden_pixels):
    """A 12-bit frame between 8-bit ones: every frame at its own offset and sample size."""
    d12 = open(os.path.join(DEEP12, D12NAMES[0] + ".jpg"), "rb").read()
    want12 = np.load(os.path.join(DEEP12, "deep12_pixels.npz"))[D12NAMES[0]]
    d8 = open(os.path.join(GOLDEN, NAMES[0] + ".jpg"), "rb").read()
    dec, out = gpu_decode(built, [d8, d12, d8])
    assert [dec.status(i) for i in range(3)] == [0, 0, 0]
    assert np.array_equal(dec.frame_view(out, 1).cpu().numpy().view(np.uint16).reshape(want12.shape), want12)
    for i in (0, 2):
        assert np.array_equal(dec.frame_view(out, i).cpu().numpy().reshape(golden_pixels[NAMES[0]].shape), golden_pixels[NAMES[0]])


def test_reference_cli_writes_12bit_frames_through_the_b200_library(built, tmp_path):
    """The reference's own client asks for CTYP_UWORD bitmaps when the frame is deeper than 8 bits (cmd/reconstruct.cpp) and
    writes a 16-bit PNM: same samples as the reference-made vectors."""
    import subprocess
    exe = os.path.join(ROOT, "oracle", "_ref", "jpeg_b200")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/jpeg_b200 is built where the reference build exists (oracle/Makefile)")
    wants = np.load(os.path.join(DEEP12, "deep12_pixels.npz"))
    for name in D12NAMES:
        out = str(tmp_path / (name + ".pnm"))
        r = subprocess.run([exe, os.path.join(DEEP12, name + ".jpg"), out], capture_output=True, text=True)
        assert r.returncode == 0 and "failed" not in r.stdout + r.stderr, (name, r.stdout[-300:], r.stderr[-300:])
        magic, dims, maxv, rest = open(out, "rb").read().split(b"\n", 3)
        w, h = map(int, dims.split())
        assert int(maxv) == 4095
        px = np.frombuffer(rest, dtype=">u2").reshape(h, w, 3 if magic == b"P6" else 1)
        assert np.array_equal(px.reshape(wants[name].shape), wants[name]), name


def _plane_fixtures():
    fx = np.load(os.path.join(GOLDEN, "planes.npz"))
    return fx, sorted({k.rsplit("__", 1)[0] for k in fx.files})


def test_planes_without_upsampling_match_reference(built):
    """SURVEY 8f4 / VERDICT r1 #7: JPGTAG_DECODER_UPSAMPLE = false (bitmapctrl.cpp:273-293, blockbitmaprequester.cpp:1013-1074)
    through the batch API (B200JPG_FLAG_NO_UPSAMPLE): every component as a plane at its own resolution == what the reference's
    client wrote with `-U -c` (tests/golden/planes.npz): baseline, progressive, 3x / 4x factors, 12-bit."""
    fx, names = _plane_fixtures()
    datas = [open(os.path.join(GOLDEN, n.replace("__", "/") + ".jpg"), "rb").read() for n in names]
    dec, out = gpu_decode(built, datas, upsample=False)
    for i, name in enumerate(names):
        assert dec.status(i) == 0, name
        deep = dec.info(i).precision > 8
        for c, p in enumerate(dec.plane_views(out, i)):
            got = p.cpu().numpy()
            got = got.view(np.uint16) if deep else got.astype(np.uint16)
            assert np.array_equal(got, fx["%s__%d" % (name, c)]), (name, c)


def test_reference_cli_without_upsampling_through_the_b200_library(built, tmp_path):
    """`jpeg_b200 -U -c in.jpg out`: the reference's own client asks component by component, in stripes of 8 * suby lines, with
    JPGTAG_DECODER_UPSAMPLE = false (cmd/reconstruct.cpp:268-301) and writes one raw plane per component."""
    import subprocess
    exe = os.path.join(ROOT, "oracle", "_ref", "jpeg_b200")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/jpeg_b200 is built where the reference build exists (oracle/Makefile)")
    fx, names = _plane_fixtures()
    for name in names:
        out = str(tmp_path / "o")
        r = subprocess.run([exe, "-U", "-c", os.path.join(GOLDEN, name.replace("__", "/") + ".jpg"), out], capture_output=True, text=True)
        assert r.returncode == 0 and "failed" not in r.stdout + r.stderr, (name, r.stdout[-300:], r.stderr[-300:])
        c = 0
        while ("%s__%d" % (name, c)) in fx.files:
            want = fx["%s__%d" % (name, c)]
            f = open("%s_%d.h" % (out, c)).read().split()
            raw = np.fromfile("%s_%d.raw" % (out, c), dtype=np.uint8 if int(f[2]) <= 8 else ">u2").reshape(int(f[4]), int(f[3]))
            assert np.array_equal(raw.astype(np.uint16), want), (name, c)
            os.remove("%s_%d.raw" % (out, c))
            c += 1
        assert c > 0


XT = os.path.join(GOLDEN, "xt")
XTNAMES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(XT, "*.jpg")))


def test_xt_residual_layer_matches_reference(built, oracle):
    """SURVEY 8f3 / VERDICT r1 #9: JPEG XT streams of the 8-bit integer profile (`jpeg -r -q .. -Q ..`): the residual codestream of
    the RESI box runs through the same entropy / IDCT kernels as one more frame of the batch, the frame's reconstruction merges
    the two images (YCbCrTrafo::YCbCr2RGB colortrafo/ycbcrtrafo.cpp:747-880) == the reference's pixels (tests/golden/xt) ==
    the oracle's; plain frames in the same batch are untouched."""
    fx = np.load(os.path.join(XT, "xt_pixels.npz"))
    names = [n for n in XTNAMES if not n.endswith("__nimpl")]
    plain = open(os.path.join(GOLDEN, NAMES[0] + ".jpg"), "rb").read()
    datas = [open(os.path.join(XT, n + ".jpg"), "rb").read() for n in names]
    dec, out = gpu_decode(built, datas[:3] + [plain] + datas[3:])
    views = [dec.frame_view(out, i).cpu().numpy() for i in range(len(datas) + 1)]
    assert all(dec.status(i) == 0 for i in range(len(datas) + 1))
    rc, want_plain = oracle.decode(plain)
    assert np.array_equal(views.pop(3).reshape(want_plain.shape), want_plain)
    for name, data, got in zip(names, datas, views):
        assert np.array_equal(got.reshape(fx[name].shape), fx[name]), name
        rc, px = oracle.decode(data)
        assert rc == 0 and np.array_equal(px.reshape(fx[name].shape), fx[name]), name


@pytest.mark.parametrize("name", [n for n in XTNAMES if n.endswith("__nimpl")])
def test_xt_profiles_outside_the_path_are_refused(built, name):
    """Lossless / 12-bit residuals and refinement scans: NOT_IMPLEMENTED, never the base image passed off as the frame."""
    from libjpeg_b200 import NativeError
    data = open(os.path.join(XT, name + ".jpg"), "rb").read()
    with pytest.raises(NativeError) as e:
        built.BatchDecoder([data])
    assert e.value.code == -1034
    good = open(os.path.join(XT, [n for n in XTNAMES if not n.endswith("__nimpl")][0] + ".jpg"), "rb").read()
    dec = built.BatchDecoder([good, data], tolerate_bad=True)
    assert dec.status(1) == -1034 and dec.status(0) == 0


def test_reference_cli_decodes_xt_through_the_b200_library(built, tmp_path):
    import subprocess
    exe = os.path.join(ROOT, "oracle", "_ref", "jpeg_b200")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/jpeg_b200 is built where the reference build exists (oracle/Makefile)")
    fx = np.load(os.path.join(XT, "xt_pixels.npz"))
    for name in [n for n in XTNAMES if not n.endswith("__nimpl")]:
        out = str(tmp_path / (name + ".pnm"))
        r = subprocess.run([exe, os.path.join(XT, name + ".jpg"), out], capture_output=True, text=True)
        assert r.returncode == 0 and "failed" not in r.stdout + r.stderr, (name, r.stdout[-300:], r.stderr[-300:])
        magic, dims, maxv, rest = open(out, "rb").read().split(b"\n", 3)
        w, h = map(int, dims.split())
        px = np.frombuffer(rest, dtype=np.uint8).reshape(h, w, 3 if magic == b"P6" else 1)
        assert np.array_equal(px.reshape(fx[name].shape), fx[name]), name


def test_device_bitmap_client_never_leaves_the_gpu(built, golden_pixels, tmp_path):
    """SURVEY 5 / VERDICT r1 #5: a client of the C++ interface whose BitMapHook hands out CUDA DEVICE pointers (tag
    JPGTAG_B200_DEVICE_BITMAPS on DisplayRectangle, tests/client/device_client.cpp): the frame is decoded and copied rectangle
    by rectangle on the device; what the client copies back at the end is the reference's pixels."""
    import subprocess
    lib_dir = os.path.join(ROOT, "libjpeg_b200")
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    exe = str(tmp_path / "device_client")
    subprocess.run(["g++", "-O1", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(cuda, "include"),
                    os.path.join(ROOT, "tests", "client", "device_client.cpp"), "-L" + lib_dir, "-lb200jpg", "-L" + os.path.join(cuda, "lib64"), "-lcudart",
                    "-Wl,-rpath," + lib_dir, "-Wl,-rpath," + os.path.join(cuda, "lib64"), "-o", exe], check=True)
    for name in ["c420_96x80_z6_q75", "c420_127x255_z7_q30", "c444_17x9_q95", "g_40x24_z2_q75", "c422_100x60_z5_q80"]:
        raw = str(tmp_path / "o.raw")
        r = subprocess.run([exe, os.path.join(GOLDEN, name + ".jpg"), raw], capture_output=True, text=True)
        assert r.returncode == 0 and "ok=1" in r.stdout, (name, r.stdout, r.stderr)
        w, h, d = (int(v) for v in r.stdout.split()[:3])
        want = golden_pixels[name].reshape(h, w, d)
        got = np.fromfile(raw, dtype=np.uint8).reshape(-1, w, d)
        assert np.array_equal(got[:h], want), name
        assert (got[h:] == 0x5A).all(), name  # rows of the canvas below the image stay untouched
