"""ctypes binding of oracle/_ref/libjpgoracle.so (the plain-C restatement of the reference). TEST-ONLY."""
import ctypes
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIB = os.path.join(ORACLE_DIR, "_ref", "libjpgoracle.so")
REF_HARNESS = os.path.join(ORACLE_DIR, "_ref", "refharness")
REF_CLI = os.path.join(ORACLE_DIR, "_ref", "jpeg")


class ScanStruct(ctypes.Structure):
    _fields_ = [("ns", ctypes.c_int), ("comp", ctypes.c_int * 4), ("td", ctypes.c_int * 4), ("ta", ctypes.c_int * 4),
                ("restart_interval", ctypes.c_int), ("ecs_offset", ctypes.c_size_t), ("ecs_end", ctypes.c_size_t),
                ("mcu_cols", ctypes.c_int), ("mcu_rows", ctypes.c_int), ("ss", ctypes.c_int), ("se", ctypes.c_int),
                ("ah", ctypes.c_int), ("al", ctypes.c_int)]


class InfoStruct(ctypes.Structure):
    _fields_ = [("width", ctypes.c_int), ("height", ctypes.c_int), ("ncomp", ctypes.c_int), ("precision", ctypes.c_int),
                ("frame_type", ctypes.c_int), ("cid", ctypes.c_int * 4), ("hs", ctypes.c_int * 4), ("vs", ctypes.c_int * 4),
                ("tq", ctypes.c_int * 4), ("hmax", ctypes.c_int), ("vmax", ctypes.c_int), ("subx", ctypes.c_int * 4),
                ("suby", ctypes.c_int * 4), ("mcu_cols", ctypes.c_int), ("mcu_rows", ctypes.c_int), ("bw", ctypes.c_int * 4),
                ("bh", ctypes.c_int * 4), ("sbw", ctypes.c_int * 4), ("sbh", ctypes.c_int * 4), ("ycbcr", ctypes.c_int),
                ("nscans", ctypes.c_int), ("scan", ScanStruct * 16), ("quant", (ctypes.c_uint16 * 64) * 4),
                ("quant_defined", ctypes.c_int * 4)]


class Oracle:
    def __init__(self, lib):
        self.lib = lib
        lib.jpgo_read_info.restype = ctypes.c_int
        lib.jpgo_read_info.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(InfoStruct)]
        lib.jpgo_decode.restype = ctypes.c_int
        lib.jpgo_decode.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(InfoStruct)]
        lib.jpgo_decode16.restype = ctypes.c_int
        lib.jpgo_decode16.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(InfoStruct)]
        lib.jpgo_decode_coefficients.restype = ctypes.c_int
        lib.jpgo_decode_coefficients.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(InfoStruct), ctypes.POINTER(ctypes.c_void_p)]
        lib.jpgo_idct_block.restype = None
        lib.jpgo_idct_block.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32]

    def info(self, data):
        data = np.ascontiguousarray(np.frombuffer(bytes(data), dtype=np.uint8))
        s = InfoStruct()
        rc = self.lib.jpgo_read_info(data.ctypes.data, data.size, ctypes.byref(s))
        return rc, s

    def decode(self, data):
        """-> (rc, pixels [H,W,C] uint8 or None)"""
        data = np.ascontiguousarray(np.frombuffer(bytes(data), dtype=np.uint8))
        rc, s = self.info(data)
        if rc != 0:
            return rc, None
        out = np.zeros((s.height, s.width, s.ncomp), dtype=np.uint8)
        rc = self.lib.jpgo_decode(data.ctypes.data, data.size, out.ctypes.data, out.size, ctypes.byref(s))
        return rc, (out if rc == 0 else None)

    def decode16(self, data):
        """-> (rc, pixels [H,W,C] uint16 or None): 8- and 12-bit frames, what a CTYP_UWORD client bitmap receives"""
        data = np.ascontiguousarray(np.frombuffer(bytes(data), dtype=np.uint8))
        rc, s = self.info(data)
        if rc != 0:
            return rc, None
        out = np.zeros((s.height, s.width, s.ncomp), dtype=np.uint16)
        rc = self.lib.jpgo_decode16(data.ctypes.data, data.size, out.ctypes.data, out.size, ctypes.byref(s))
        return rc, (out if rc == 0 else None)

    def decode_planes(self, data):
        """-> (rc, [plane of component c: [ceil(H/suby), ceil(W/subx)] uint16] or None): JPGTAG_DECODER_UPSAMPLE = false"""
        data = np.ascontiguousarray(np.frombuffer(bytes(data), dtype=np.uint8))
        rc, s = self.info(data)
        if rc != 0:
            return rc, None
        dims = [((s.height + s.suby[c] - 1) // s.suby[c], (s.width + s.subx[c] - 1) // s.subx[c]) for c in range(s.ncomp)]
        out = np.zeros(sum(h * w for h, w in dims), dtype=np.uint16)
        self.lib.jpgo_decode_planes16.restype = ctypes.c_int
        self.lib.jpgo_decode_planes16.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(InfoStruct)]
        rc = self.lib.jpgo_decode_planes16(data.ctypes.data, data.size, out.ctypes.data, out.size, ctypes.byref(s))
        if rc != 0:
            return rc, None
        planes, at = [], 0
        for h, w in dims:
            planes.append(out[at:at + h * w].reshape(h, w))
            at += h * w
        return rc, planes

    def coefficients(self, data):
        """-> (rc, info, [per component int32 [bh,bw,8,8] QUANTIZED raster-order coefficients])"""
        data = np.ascontiguousarray(np.frombuffer(bytes(data), dtype=np.uint8))
        rc, s = self.info(data)
        if rc != 0:
            return rc, s, None
        planes = [np.zeros((s.bh[c], s.bw[c], 8, 8), dtype=np.int32) for c in range(s.ncomp)]
        ptrs = (ctypes.c_void_p * 4)(*[p.ctypes.data for p in planes] + [None] * (4 - s.ncomp))
        rc = self.lib.jpgo_decode_coefficients(data.ctypes.data, data.size, ctypes.byref(s), ptrs)
        return rc, s, planes

    def decode_without_color_transform(self, data):
        """-> (rc, pixels): the components upsampled and delivered as they are (JPGTAG_MATRIX_LTRAFO = none)"""
        rc, s, planes = self.coefficients(data)
        if rc != 0:
            return rc, None
        s.ycbcr = 0
        out = np.zeros((s.height, s.width, s.ncomp), dtype=np.uint8)
        ptrs = (ctypes.c_void_p * 4)(*[p.ctypes.data for p in planes] + [None] * (4 - s.ncomp))
        self.lib.jpgo_reconstruct.restype = ctypes.c_int
        self.lib.jpgo_reconstruct.argtypes = [ctypes.POINTER(InfoStruct), ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p]
        rc = self.lib.jpgo_reconstruct(ctypes.byref(s), ptrs, out.ctypes.data)
        return rc, (out if rc == 0 else None)

    def idct(self, block_raster_int32, delta_raster_u16, dcoffset=128):
        src = np.ascontiguousarray(block_raster_int32, dtype=np.int32)
        q = np.ascontiguousarray(delta_raster_u16, dtype=np.uint16)
        out = np.zeros(64, dtype=np.int32)
        self.lib.jpgo_idct_block(out.ctypes.data, src.ctypes.data, q.ctypes.data, dcoffset)
        return out.reshape(8, 8)


def build():
    """Compiles the C restatement (always) and, where the reference sources exist, the reference itself."""
    subprocess.run(["make", "-s", "-C", ORACLE_DIR, "all"], check=True)


def load():
    if not os.path.exists(LIB):
        build()
    return Oracle(ctypes.CDLL(LIB))


def reference_decode(jpg_path, tmp_raw):
    r = subprocess.run([REF_HARNESS, "decode", jpg_path, tmp_raw], capture_output=True, text=True)
    if r.returncode != 0:
        return None
    fields = r.stdout.split()
    w, h, d = map(int, fields[:3])
    wide = len(fields) > 3  # "16": native-endian 16-bit samples (precision above 8)
    return np.fromfile(tmp_raw, dtype=np.uint16 if wide else np.uint8).reshape(h, w, d)


def with_dc_quantiser(data, value):
    """The same codestream with the DC entry of every 8-bit quantisation table replaced: the coefficients stay within
    int16, but the IDCT samples leave the ranges the GPU fast paths are built for (int16 planes, 32-bit colour)."""
    b = bytearray(data.tobytes() if hasattr(data, "tobytes") else data)
    i = 2
    while i + 4 <= len(b) and b[i] == 0xFF and b[i + 1] != 0xDA:
        seglen = (b[i + 2] << 8) | b[i + 3]
        if b[i + 1] == 0xDB:
            j = i + 4
            while j < i + 2 + seglen:
                assert b[j] >> 4 == 0, "8-bit tables expected"
                b[j + 1] = value
                j += 65
        i += 2 + seglen
    return bytes(b)


def with_fill_bytes(data, every=2, count=1):
    """The same codestream with `count` fill bytes (0xFF) in front of every `every`-th restart marker / EOI of the
    entropy coded segment (legal: entropyparser.cpp:121-125, tables.cpp:1371-1373)."""
    b = bytes(data.tobytes() if hasattr(data, "tobytes") else data)
    sos = b.find(b"\xff\xda")
    start = sos + 2 + ((b[sos + 2] << 8) | b[sos + 3])
    out, n, i = bytearray(b[:start]), 0, start
    while i < len(b):
        if b[i] == 0xFF and i + 1 < len(b) and (0xD0 <= b[i + 1] <= 0xD7 or b[i + 1] == 0xD9):
            if n % every == 0:
                out += b"\xff" * count
            n += 1
            out += b[i:i + 2]
            i += 2
        else:
            out.append(b[i])
            i += 1
    return bytes(out)


def with_swapped_restart_ids(data, first=1):
    """The same codestream with the ids of restart markers number `first` and `first + 1` exchanged (out of sequence)."""
    b = bytearray(data.tobytes() if hasattr(data, "tobytes") else data)
    sos = bytes(b).find(b"\xff\xda")
    i, at = sos + 2 + ((b[sos + 2] << 8) | b[sos + 3]), []
    while i + 1 < len(b):
        if b[i] == 0xFF and 0xD0 <= b[i + 1] <= 0xD7:
            at.append(i + 1)
            i += 2
        else:
            i += 1
    b[at[first]], b[at[first + 1]] = b[at[first + 1]], b[at[first]]
    return bytes(b)


def handmade_grey_stream(blocks_bits, width=8, height=8, dri=0):
    """A tiny grey SOF0 codestream with hand-picked Huffman tables, for cases an encoder never writes:
    DC table: category 0 = '0', category 1 = '10'; AC table: ZRL (0xF0) = '0', EOB (0x00) = '10', 0/1 (0x01) = '110',
    2/1 (0x21) = '1110'.
    `blocks_bits` is the bit string of the whole entropy coded segment ('0'/'1'), padded with ones to a byte boundary."""
    bits = blocks_bits + "1" * (-len(blocks_bits) % 8)
    ecs = bytearray()
    for i in range(0, len(bits), 8):
        v = int(bits[i:i + 8], 2)
        ecs.append(v)
        if v == 0xFF:
            ecs.append(0)
    seg = lambda marker, payload: bytes([0xFF, marker]) + (len(payload) + 2).to_bytes(2, "big") + bytes(payload)
    dqt = seg(0xDB, [0] + [16] * 64)
    sof = seg(0xC0, [8] + list(height.to_bytes(2, "big")) + list(width.to_bytes(2, "big")) + [1, 1, 0x11, 0])
    dht_dc = [0x00] + [1, 1] + [0] * 14 + [0, 1]
    dht_ac = [0x10] + [1, 1, 1, 1] + [0] * 12 + [0xF0, 0x00, 0x01, 0x21]
    dht = seg(0xC4, dht_dc + dht_ac)
    drim = seg(0xDD, list(dri.to_bytes(2, "big"))) if dri else b""
    sos = seg(0xDA, [1, 1, 0x00, 0, 63, 0])
    return b"\xff\xd8" + dqt + sof + dht + drim + sos + bytes(ecs) + b"\xff\xd9"


def zrl_overrun_stream():
    """One 8x8 block: DC category 1 (value +1), one AC coefficient at k = 1, then four ZRLs -- the fourth steps from k = 50
    over position 63. The reference re-tests k <= 63 after a ZRL and silently ends the block (sequentialscan.cpp:717-719)."""
    return handmade_grey_stream("10" + "1" + "110" + "1" + "0000")


RESTART_DAMAGES = ["swap", "drop_marker", "drop_interval", "duplicate", "id_plus_4", "id_plus_2", "id_minus_1", "garbage",
                   "cut_mid_interval", "no_eoi"]


def with_restart_damage(data, damage):
    """The codestream with its restart markers damaged: ids exchanged / shifted, a marker or a whole interval dropped, a
    marker duplicated, garbage in front of a marker, the stream cut inside an interval (with and without a closing EOI)."""
    a = bytes(data.tobytes() if hasattr(data, "tobytes") else data)
    sos = a.find(b"\xff\xda")
    i, at = sos + 2 + ((a[sos + 2] << 8) | a[sos + 3]), []
    while i + 1 < len(a):
        if a[i] == 0xFF and 0xD0 <= a[i + 1] <= 0xD7:
            at.append(i)
            i += 2
        else:
            i += 1
    b = bytearray(a)
    if damage == "swap":
        b[at[2] + 1], b[at[3] + 1] = b[at[3] + 1], b[at[2] + 1]
    elif damage == "drop_marker":
        del b[at[3]:at[3] + 2]
    elif damage == "drop_interval":
        del b[at[3]:at[4]]
    elif damage == "duplicate":
        b[at[2]:at[2]] = a[at[2]:at[2] + 2]
    elif damage.startswith("id_"):
        delta = {"id_plus_4": 4, "id_plus_2": 2, "id_minus_1": 7}[damage]
        b[at[1] + 1] = 0xD0 + ((b[at[1] + 1] - 0xD0 + delta) & 7)
    elif damage == "garbage":
        b[at[2]:at[2]] = b"\x12\x34\xff\x00\x56"
    elif damage == "cut_mid_interval":
        b = bytearray(a[:at[3] + 20] + b"\xff\xd9")
    elif damage == "no_eoi":
        b = bytearray(a[:at[3] + 20])
    else:
        raise ValueError(damage)
    return bytes(b)


def with_fourth_component(data):
    """A four-component codestream made from a three-component one whose components are coded in separate scans
    (synth.NON_INTERLEAVED): the third component's frame entry and scan are duplicated under a new component id. Four
    components have no colour transformation in the reference (identity, colortrafo/ycbcrtrafo.cpp:834-892)."""
    b = bytes(data.tobytes() if hasattr(data, "tobytes") else data)
    sof = b.find(b"\xff\xc0")
    seglen = (b[sof + 2] << 8) | b[sof + 3]
    assert b[sof + 9] == 3
    last = b[sof + 10 + 6:sof + 10 + 9]  # (id, HV, Tq) of the third component
    new_id = max(b[sof + 10], b[sof + 13], b[sof + 16]) + 1
    sof_new = b[sof:sof + 2] + (seglen + 3).to_bytes(2, "big") + b[sof + 4:sof + 9] + bytes([4]) + b[sof + 10:sof + 2 + seglen] + bytes([new_id]) + last[1:]
    head = b[:sof] + sof_new
    rest = b[sof + 2 + seglen:]
    # the last SOS (third component) up to EOI
    pos, sos_at = 0, []
    while True:
        i = rest.find(b"\xff\xda", pos)
        if i < 0:
            break
        sos_at.append(i)
        pos = i + 2
    assert len(sos_at) == 3
    eoi = rest.rfind(b"\xff\xd9")
    scan3 = bytearray(rest[sos_at[2]:eoi])
    assert scan3[4] == 1  # one component in the scan
    scan3[5] = new_id
    return head + rest[:eoi] + bytes(scan3) + b"\xff\xd9"
