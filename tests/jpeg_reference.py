"""A plain numpy restatement of the device JPEG encoder (csrc/jpeg_encode.cu) and a small baseline decoder.

Forward: libjpeg's integer stages (jccolor.c's 16-bit fixed-point RGB -> YCbCr, edges replicated up to a whole 16x16
MCU, h2v2_downsample with its 1, 2 rounding bias), an fp64 DCT-II and round-half-away-from-zero quantisation with the
Annex K.1 tables at the IJG quality scaling.  Entropy coding: the Annex K.3 Huffman tables, a restart marker every
RESTART_MCUS MCUs, 1-bit padding and 0xFF stuffing.  The decoder parses a baseline 4:2:0 file with restarts and returns
its quantised coefficients, so a file can be compared coefficient by coefficient and re-encoded byte for byte.

Coefficients are int arrays [n_mcus, 6, 64] in zigzag order, blocks Y00 Y01 Y10 Y11 Cb Cr of each MCU in raster order.
"""
from __future__ import annotations

import struct
from typing import Dict, Tuple

import numpy as np

RESTART_MCUS = 4  # KP_JPEG_RESTART_MCUS

NATURAL = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,
                    7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31,
                    39, 46, 53, 60, 61, 54, 47, 55, 62, 63])  # zigzag position -> natural (row-major) index

STD_QUANT = np.array([
    [16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56,
     14, 17, 22, 29, 51, 87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92,
     49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99],
    [17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99,
     47, 66, 99, 99] + [99] * 36])  # Annex K.1, natural order

DC_LUM_BITS = [0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0]
DC_CHR_BITS = [0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0]
DC_VALS = list(range(12))
AC_LUM_BITS = [0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7D]
AC_LUM_VALS = [
    0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14,
    0x32, 0x81, 0x91, 0xA1, 0x08, 0x23, 0x42, 0xB1, 0xC1, 0x15, 0x52, 0xD1, 0xF0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09,
    0x0A, 0x16, 0x17, 0x18, 0x19, 0x1A, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2A, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3A,
    0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4A, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5A, 0x63, 0x64, 0x65,
    0x66, 0x67, 0x68, 0x69, 0x6A, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7A, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88,
    0x89, 0x8A, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9A, 0xA2, 0xA3, 0xA4, 0xA5, 0xA6, 0xA7, 0xA8, 0xA9,
    0xAA, 0xB2, 0xB3, 0xB4, 0xB5, 0xB6, 0xB7, 0xB8, 0xB9, 0xBA, 0xC2, 0xC3, 0xC4, 0xC5, 0xC6, 0xC7, 0xC8, 0xC9, 0xCA,
    0xD2, 0xD3, 0xD4, 0xD5, 0xD6, 0xD7, 0xD8, 0xD9, 0xDA, 0xE1, 0xE2, 0xE3, 0xE4, 0xE5, 0xE6, 0xE7, 0xE8, 0xE9, 0xEA,
    0xF1, 0xF2, 0xF3, 0xF4, 0xF5, 0xF6, 0xF7, 0xF8, 0xF9, 0xFA]
AC_CHR_BITS = [0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77]
AC_CHR_VALS = [
    0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32,
    0x81, 0x08, 0x14, 0x42, 0x91, 0xA1, 0xB1, 0xC1, 0x09, 0x23, 0x33, 0x52, 0xF0, 0x15, 0x62, 0x72, 0xD1, 0x0A, 0x16,
    0x24, 0x34, 0xE1, 0x25, 0xF1, 0x17, 0x18, 0x19, 0x1A, 0x26, 0x27, 0x28, 0x29, 0x2A, 0x35, 0x36, 0x37, 0x38, 0x39,
    0x3A, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4A, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5A, 0x63, 0x64,
    0x65, 0x66, 0x67, 0x68, 0x69, 0x6A, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7A, 0x82, 0x83, 0x84, 0x85, 0x86,
    0x87, 0x88, 0x89, 0x8A, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9A, 0xA2, 0xA3, 0xA4, 0xA5, 0xA6, 0xA7,
    0xA8, 0xA9, 0xAA, 0xB2, 0xB3, 0xB4, 0xB5, 0xB6, 0xB7, 0xB8, 0xB9, 0xBA, 0xC2, 0xC3, 0xC4, 0xC5, 0xC6, 0xC7, 0xC8,
    0xC9, 0xCA, 0xD2, 0xD3, 0xD4, 0xD5, 0xD6, 0xD7, 0xD8, 0xD9, 0xDA, 0xE2, 0xE3, 0xE4, 0xE5, 0xE6, 0xE7, 0xE8, 0xE9,
    0xEA, 0xF2, 0xF3, 0xF4, 0xF5, 0xF6, 0xF7, 0xF8, 0xF9, 0xFA]
# (class, id) -> (BITS, HUFFVAL): class 0 = DC, 1 = AC; id 0 = luminance, 1 = chrominance
HUFF = {(0, 0): (DC_LUM_BITS, DC_VALS), (1, 0): (AC_LUM_BITS, AC_LUM_VALS),
        (0, 1): (DC_CHR_BITS, DC_VALS), (1, 1): (AC_CHR_BITS, AC_CHR_VALS)}
TABLE_OF_BLOCK = (0, 0, 0, 0, 1, 1)  # quantisation / Huffman table id of each block of an MCU


def quant_tables(quality: int) -> np.ndarray:
    """The K.1 tables at the IJG quality scaling (jcparam.c jpeg_quality_scaling + jpeg_add_quant_table, baseline):
    int [2, 64], natural order."""
    scale = 5000 // quality if quality < 50 else 200 - 2 * quality
    return np.clip((STD_QUANT * scale + 50) // 100, 1, 255)


def huffman_codes(bits, vals) -> Dict[int, Tuple[int, int]]:
    """symbol -> (code, length), T.81 Annex C."""
    codes, code, k = {}, 0, 0
    for length in range(1, 17):
        for _ in range(bits[length - 1]):
            codes[vals[k]] = (code, length)
            k += 1
            code += 1
        code <<= 1
    return codes


CODES = {key: huffman_codes(*tab) for key, tab in HUFF.items()}


def _fix(x: float) -> int:
    return int(x * 65536 + 0.5)


def rgb_to_ycc(img: np.ndarray) -> np.ndarray:
    """jccolor.c rgb_ycc_convert: uint8 [..., 3] -> int64 [..., 3] (Y, Cb, Cr)."""
    r, g, b = (img[..., i].astype(np.int64) for i in range(3))
    half, off = 1 << 15, 128 << 16
    y = (_fix(0.29900) * r + _fix(0.58700) * g + _fix(0.11400) * b + half) >> 16
    cb = (-_fix(0.16874) * r - _fix(0.33126) * g + _fix(0.5) * b + off + half - 1) >> 16
    cr = (_fix(0.5) * r - _fix(0.41869) * g - _fix(0.08131) * b + off + half - 1) >> 16
    return np.stack([y, cb, cr], -1)


def downsample_h2v2(c: np.ndarray) -> np.ndarray:
    """jcsample.c h2v2_downsample of an even-sized plane: the 2x2 sum plus a bias 1, 2, 1, 2, ... along each row, >> 2."""
    bias = 1 + (np.arange(c.shape[1] // 2) & 1)
    return (c[0::2, 0::2] + c[0::2, 1::2] + c[1::2, 0::2] + c[1::2, 1::2] + bias) >> 2


def mcu_samples(img: np.ndarray) -> np.ndarray:
    """uint8 [H, W, 3] -> the level-shifted samples int64 [n_mcus, 6, 8, 8] of every block."""
    h, w = img.shape[:2]
    my, mx = -(-h // 16), -(-w // 16)
    padded = np.pad(img, ((0, 16 * my - h), (0, 16 * mx - w), (0, 0)), mode="edge")
    ycc = rgb_to_ycc(padded)
    y = ycc[..., 0].reshape(my, 2, 8, mx, 2, 8).transpose(0, 3, 1, 4, 2, 5).reshape(my * mx, 4, 8, 8)
    cb, cr = (downsample_h2v2(ycc[..., i]).reshape(my, 8, mx, 8).transpose(0, 2, 1, 3).reshape(my * mx, 1, 8, 8)
              for i in (1, 2))
    return np.concatenate([y, cb, cr], 1) - 128


def dct_matrix() -> np.ndarray:
    u, x = np.meshgrid(np.arange(8), np.arange(8), indexing="ij")
    c = np.cos((2 * x + 1) * u * np.pi / 16) * 0.5
    c[0] = np.sqrt(1 / 8)
    return c


def forward(img: np.ndarray, quality: int) -> Tuple[np.ndarray, np.ndarray]:
    """uint8 [H, W, 3] -> (quantised coefficients int64 [n_mcus, 6, 64], coef / Q in fp64 [n_mcus, 6, 64]), zigzag."""
    c = dct_matrix()
    coef = np.einsum("ux,nbxy,vy->nbuv", c, mcu_samples(img).astype(np.float64), c).reshape(-1, 6, 64)
    q = quant_tables(quality)[list(TABLE_OF_BLOCK)]  # [6, 64] natural
    ratio = (coef / q)[..., NATURAL]
    return (np.sign(ratio) * np.floor(np.abs(ratio) + 0.5)).astype(np.int64), ratio


def header(h: int, w: int, quality: int) -> bytes:
    """SOI, APP0 (JFIF 1.01), DQT, SOF0 (4:2:0), DHT (the four K.3 tables), DRI, SOS."""
    seg = lambda marker, body: struct.pack(">HH", marker, len(body) + 2) + body  # noqa: E731
    q = quant_tables(quality)
    dqt = b"".join(bytes([t]) + bytes(int(v) for v in q[t][NATURAL]) for t in range(2))
    dht = b"".join(bytes([cls << 4 | tid]) + bytes(HUFF[(cls, tid)][0]) + bytes(HUFF[(cls, tid)][1])
                   for tid, cls in ((0, 0), (0, 1), (1, 0), (1, 1)))
    return (b"\xff\xd8" + seg(0xFFE0, b"JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00") + seg(0xFFDB, dqt)
            + seg(0xFFC0, struct.pack(">BHHB", 8, h, w, 3) + bytes([1, 0x22, 0, 2, 0x11, 1, 3, 0x11, 1]))
            + seg(0xFFC4, dht) + seg(0xFFDD, struct.pack(">H", RESTART_MCUS))
            + seg(0xFFDA, bytes([3, 1, 0x00, 2, 0x11, 3, 0x11, 0, 63, 0])))


def _category(v: int) -> int:
    return abs(int(v)).bit_length()


def _magnitude(v: int, s: int) -> int:
    return (v - 1 if v < 0 else v) & ((1 << s) - 1)


class _BitWriter:
    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0

    def put(self, v: int, n: int) -> None:
        self.acc = self.acc << n | v
        self.n += n
        while self.n >= 8:
            self.n -= 8
            byte = (self.acc >> self.n) & 0xFF
            self.out.append(byte)
            if byte == 0xFF:
                self.out.append(0)  # stuffing
        self.acc &= (1 << self.n) - 1

    def flush(self) -> None:
        if self.n:
            self.put((1 << (8 - self.n)) - 1, 8 - self.n)  # pad with 1-bits


def entropy_code(coefs: np.ndarray) -> bytes:
    """coefficients int [n_mcus, 6, 64] (zigzag) -> the scan's bytes: restarts every RESTART_MCUS MCUs (RSTm, m
    cycling 0..7, DC predictors reset), 1-bit padding before each marker, 0xFF stuffing."""
    coefs = np.asarray(coefs)
    bw = _BitWriter()
    n = len(coefs)
    for seg, m0 in enumerate(range(0, n, RESTART_MCUS)):
        pred = [0, 0, 0]
        for mcu in coefs[m0:m0 + RESTART_MCUS].tolist():
            for b, zz in enumerate(mcu):
                comp = 0 if b < 4 else b - 3  # 0 Y, 1 Cb, 2 Cr
                tid = TABLE_OF_BLOCK[b]
                diff = zz[0] - pred[comp]
                pred[comp] = zz[0]
                s = _category(diff)
                bw.put(*CODES[(0, tid)][s])
                if s:
                    bw.put(_magnitude(diff, s), s)
                ac = CODES[(1, tid)]
                run = 0
                for v in zz[1:]:
                    if v == 0:
                        run += 1
                        continue
                    while run >= 16:
                        bw.put(*ac[0xF0])
                        run -= 16
                    s = _category(v)
                    bw.put(*ac[run << 4 | s])
                    bw.put(_magnitude(v, s), s)
                    run = 0
                if run:
                    bw.put(*ac[0x00])
        bw.flush()
        if m0 + RESTART_MCUS < n:
            bw.out += bytes([0xFF, 0xD0 + (seg & 7)])
    return bytes(bw.out)


def encode(coefs: np.ndarray, h: int, w: int, quality: int) -> bytes:
    """The whole file of the given coefficients."""
    return header(h, w, quality) + entropy_code(coefs) + b"\xff\xd9"


def encode_image(img: np.ndarray, quality: int) -> bytes:
    return encode(forward(img, quality)[0], img.shape[0], img.shape[1], quality)


# ---- decoder ----
def _lut(bits, vals) -> np.ndarray:
    """16-bit peek -> symbol << 8 | code length (0: no code)."""
    lut = np.zeros(1 << 16, dtype=np.int64)
    for sym, (code, length) in huffman_codes(bits, vals).items():
        lut[code << (16 - length):(code + 1) << (16 - length)] = sym << 8 | length
    return lut


def decode(data: bytes) -> dict:
    """A baseline file with 4:2:0 sampling (Y 2x2, Cb 1x1, Cr 1x1, one interleaved scan, restarts allowed) ->
    {"height", "width", "quant": {id: natural-order int [64]}, "restart", "coefs": int [n_mcus, 6, 64] zigzag}.
    Raises ValueError on anything else or on a malformed scan."""
    if data[:2] != b"\xff\xd8":
        raise ValueError("no SOI")
    pos, quant, huff, restart, comps, h = 2, {}, {}, 0, None, None
    while True:
        if data[pos] != 0xFF:
            raise ValueError(f"marker expected at {pos}")
        marker = data[pos + 1]
        length = struct.unpack(">H", data[pos + 2:pos + 4])[0]
        body = data[pos + 4:pos + 2 + length]
        pos += 2 + length
        if marker == 0xDB:
            i = 0
            while i < len(body):
                if body[i] >> 4:
                    raise ValueError("16-bit quantisation table")
                quant[body[i] & 15] = np.array(list(body[i + 1:i + 65]))[np.argsort(NATURAL)]
                i += 65
        elif marker == 0xC4:
            i = 0
            while i < len(body):
                bits = list(body[i + 1:i + 17])
                vals = list(body[i + 17:i + 17 + sum(bits)])
                huff[(body[i] >> 4, body[i] & 15)] = _lut(bits, vals)
                i += 17 + sum(bits)
        elif marker == 0xC0:
            p, h, w, nf = struct.unpack(">BHHB", body[:6])
            comps = [tuple(body[6 + 3 * k:9 + 3 * k]) for k in range(nf)]
            if p != 8 or [c[1] for c in comps] != [0x22, 0x11, 0x11]:
                raise ValueError(f"not 8-bit 4:2:0: {comps}")
        elif marker == 0xDD:
            restart = struct.unpack(">H", body)[0]
        elif marker == 0xDA:
            tabs = [(body[2 + 2 * k] >> 4, body[2 + 2 * k] & 15) for k in range(body[0])]
            break
        elif marker in (0xC1, 0xC2, 0xC3) or 0xC5 <= marker <= 0xCF:
            raise ValueError(f"not baseline: SOF{marker - 0xC0}")
    if comps is None:
        raise ValueError("no SOF0")
    n_mcus = -(-h // 16) * -(-w // 16)
    end = data.rindex(b"\xff\xd9")
    scan = data[pos:end]
    # split at RSTm (0xFF 0xD0..0xD7; a stuffed 0xFF is followed by 0x00), then unstuff
    segments, start, m = [], 0, 0
    i = scan.find(b"\xff")
    while i >= 0:
        nxt = scan[i + 1]
        if 0xD0 <= nxt <= 0xD7:
            if nxt != 0xD0 + (m & 7):
                raise ValueError(f"restart marker {nxt - 0xD0} out of order (expected {m & 7})")
            segments.append(scan[start:i])
            start, m = i + 2, m + 1
        elif nxt != 0x00:
            raise ValueError(f"unexpected marker 0xFF{nxt:02X} in the scan")
        i = scan.find(b"\xff", i + 2)
    segments.append(scan[start:])
    per = restart or n_mcus
    if len(segments) != -(-n_mcus // per):
        raise ValueError(f"{len(segments)} scan segments for {n_mcus} MCUs at restart interval {per}")
    coefs = np.zeros((n_mcus, 6, 64), dtype=np.int64)
    for s, seg in enumerate(segments):
        buf = seg.replace(b"\xff\x00", b"\xff") + b"\xff\xff\xff\xff"
        nbits = 8 * (len(buf) - 4)
        p = 0
        pred = [0, 0, 0]

        def bits(n):
            nonlocal p
            i = p >> 3
            v = (int.from_bytes(buf[i:i + 4], "big") >> (32 - (p & 7) - n)) & ((1 << n) - 1)
            p += n
            return v

        def symbol(lut):
            nonlocal p
            i = p >> 3
            e = int(lut[(int.from_bytes(buf[i:i + 4], "big") >> (16 - (p & 7))) & 0xFFFF])
            if e == 0:
                raise ValueError(f"invalid Huffman code in segment {s} at bit {p}")
            p += e & 0xFF
            return e >> 8

        def extend(v, t):
            return v - (1 << t) + 1 if t and v < (1 << (t - 1)) else v

        for mcu in range(s * per, min((s + 1) * per, n_mcus)):
            for b in range(6):
                comp = 0 if b < 4 else b - 3
                dc_t, ac_t = tabs[comp]
                t = symbol(huff[(0, dc_t)])
                pred[comp] += extend(bits(t), t) if t else 0
                zz = coefs[mcu, b]
                zz[0] = pred[comp]
                k = 1
                while k < 64:
                    rs = symbol(huff[(1, ac_t)])
                    r, t = rs >> 4, rs & 15
                    if t == 0:
                        if r == 15:
                            k += 16
                            continue
                        break  # EOB
                    k += r
                    if k > 63:
                        raise ValueError(f"AC run past the block in segment {s}")
                    zz[k] = extend(bits(t), t)
                    k += 1
        left = nbits - p
        if not 0 <= left < 8:
            raise ValueError(f"segment {s}: {left} bits left after its MCUs")
        if left and bits(left) != (1 << left) - 1:
            raise ValueError(f"segment {s}: the padding is not 1-bits")
    return {"height": h, "width": w, "quant": quant, "restart": restart, "coefs": coefs}
