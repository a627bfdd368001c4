"""Host-side members of the interface (no GPU): file quantizer, weight re-tiling, tokenizer, preprocess, image decoders -- each
checked bit-exactly against what the reference returned for the same inputs (tests/golden, recorded from oracle/_ref)."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import binding as bd
import synth_gguf as sg
from _util import FTYPES, GOLDEN, check_sha, golden, model_file

HOST = json.load(open(os.path.join(GOLDEN, "host_ops.json")))


def _sha(data):
    return hashlib.sha256(data).hexdigest()


def _reference_runs():
    """What the reference returned for this module's inputs beyond host_ops.json and jpeg/ (tests/golden/make_ref_golden.py)."""
    with open(os.path.join(GOLDEN, "reference_runs.json")) as f:
        return json.load(f)


class _ReferenceDecodes:
    """What the reference's clip_image_load_from_file returned for each file a decoder test writes, in the order the test writes them
    (sha256 of the pixels; of the file too where the encoder is lossy).  tests/golden/make_ref_golden.py records them by running the
    same test with the reference library in place of this class."""

    def __init__(self, test, pin_files=False):
        self.test, self.want, self.n, self.pin_files = test, _reference_runs()["decodes"][test], 0, pin_files

    def check(self, path, got):
        assert self.n < len(self.want), (self.test, "more files than the recording")
        file_sha, pix_sha = self.want[self.n]
        if self.pin_files:
            assert _sha(open(path, "rb").read()) == file_sha, (self.test, self.n, "the encoder wrote other bytes than when recorded")
        assert got is not None and _sha(got.tobytes()) == pix_sha, (self.test, self.n)
        self.n += 1

    def done(self):
        assert self.n == len(self.want), (self.test, self.n, len(self.want))


def _reference_decodes(test, pin_files=False):
    return _ReferenceDecodes(test, pin_files)


@pytest.mark.parametrize("ft", ["q4_0", "q4_1", "q5_0", "q5_1", "q8_0"])
def test_quantize_is_byte_identical_to_reference(prod, ft):
    """clip_model_quantize (clip.cpp:1661-1844): the sha256 in the fixture is of the file the REFERENCE's quantizer wrote."""
    g = golden("tiny")
    path = sg.model_path("tiny", 1234, ft) + ".check"
    assert prod.quantize(model_file("tiny", "f16", prod), path, FTYPES[ft])
    try:
        check_sha(path, g["sha_" + ft])
    finally:
        os.remove(path)


def test_quantize_rejects_bad_arguments(prod):
    assert not prod.quantize(model_file("tiny", "f16", prod), "/tmp/x.gguf", 5)       # unknown type
    assert not prod.quantize("/nonexistent.gguf", "/tmp/x.gguf", 2)
    assert not prod.quantize(model_file("tiny", "q4_0", prod), "/tmp/x.gguf", 2)      # already quantized


@pytest.mark.parametrize("ft", ["q4_0", "q4_1", "q5_0", "q5_1", "q8_0"])
def test_weight_retiling_is_lossless(prod, ft):
    """wpack.h: the TMA-friendly re-tiling keeps every quant and every fp16 scale bit (round trip on random blocks)."""
    import oracle as orc
    rng = np.random.default_rng(5)
    N, K = 256, 192
    raw = orc.quantize_rows(FTYPES[ft], (rng.standard_normal((N, K)) * 0.1).astype(np.float32))
    buf = np.frombuffer(raw, np.uint8)
    assert prod.lib.clip_b200_debug_repack_roundtrip(FTYPES[ft], buf.ctypes.data, N, K) == 0
    assert prod.lib.clip_b200_debug_repack_roundtrip(FTYPES[ft], buf.ctypes.data, 100, K) != 0     # N % 128 != 0 is refused


def _tokenize(prod, model, text):
    out = (C.c_int32 * 512)()
    n = prod.lib.clip_b200_debug_tokenize(model.encode(), text.encode("latin1"), out, 512)
    assert n >= 2
    return [int(out[i]) for i in range(n)]


def test_tokenizer_matches_reference_golden(prod):
    model = model_file("tiny", "f16", prod)
    check_sha(model, HOST["model_sha"])
    for text, ids in HOST["tokens"].items():
        assert _tokenize(prod, model, text) == ids, repr(text)


def _synth_u8(nx, ny, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    base = rng.integers(0, 256, size=(ny // 8 + 2, nx // 8 + 2, 3)).astype(np.float32)
    img = np.kron(base, np.ones((8, 8, 1), np.float32))[:ny, :nx]
    img += rng.normal(0, 12, size=img.shape).astype(np.float32)
    return np.clip(img, 0, 255).astype(np.uint8)


def _preprocess(prod, u8, S=64):
    mean = np.array([0.48145466, 0.4578275, 0.40821073], np.float32)
    std = np.array([0.26862954, 0.26130258, 0.27577711], np.float32)
    out = np.empty((S, S, 3), np.float32)
    fp = C.POINTER(C.c_float)
    rc = prod.lib.clip_b200_debug_preprocess(u8.ctypes.data_as(C.POINTER(C.c_uint8)), u8.shape[1], u8.shape[0], S,
                                             mean.ctypes.data_as(fp), std.ctypes.data_as(fp), out.ctypes.data_as(fp))
    assert rc == 0
    return out


def test_preprocess_matches_reference_golden_bit_exactly(prod):
    for e in HOST["preprocess"]:
        out = _preprocess(prod, _synth_u8(e["nx"], e["ny"], e["seed"]))
        assert hashlib.sha256(out.tobytes()).hexdigest() == e["sha256"], e


LIVE_TEXTS = ["the red apple isn't a dog", "  double  spaces and 42 numbers!!", "mixed'case I'LL"]
LIVE_IMAGE = (123, 77, 99)      # nx, ny, seed of _synth_u8


def test_tokenizer_and_preprocess_match_live_reference(prod):
    """Texts and an image outside host_ops.json, against the reference's tokens and preprocessed floats (tests/golden/reference_runs.json)."""
    want = _reference_runs()["tokenize_preprocess"]
    model = model_file("tiny", "f16", prod)
    check_sha(model, want["model_sha"])
    for t, ids in zip(LIVE_TEXTS, want["tokens"], strict=True):
        assert _tokenize(prod, model, t) == ids
    assert _sha(_preprocess(prod, _synth_u8(*LIVE_IMAGE)).tobytes()) == want["preprocess_sha256"]


def test_scoring_helpers_match_reference_arithmetic(prod):
    """clip_similarity_score (clip.cpp:1525-1532) and softmax_with_sorting (clip.cpp:1591-1622: no max subtraction, +1e-9)."""
    fp = C.POINTER(C.c_float)
    rng = np.random.default_rng(3)
    a, b = rng.standard_normal(512).astype(np.float32), rng.standard_normal(512).astype(np.float32)
    acc = np.float32(0)
    for x, y in zip(a, b):
        acc = np.float32(acc + np.float32(x * y))
    assert prod.lib.clip_similarity_score(a.ctypes.data_as(fp), b.ctypes.data_as(fp), 512) == pytest.approx(float(acc), rel=1e-6)
    s = rng.standard_normal(10).astype(np.float32)
    arr, scores, idx = s.copy(), np.empty(10, np.float32), np.empty(10, np.int32)
    assert prod.lib.softmax_with_sorting(arr.ctypes.data_as(fp), 10, scores.ctypes.data_as(fp), idx.ctypes.data_as(C.POINTER(C.c_int)))
    e = (np.exp(s.astype(np.float64)) + 1e-9).astype(np.float32)
    p = (e / e.astype(np.float64).sum()).astype(np.float32)
    assert np.array_equal(idx, np.argsort(-p, kind="stable"))
    assert np.allclose(scores, p[idx], rtol=1e-6)
    assert not prod.lib.softmax_with_sorting(arr.ctypes.data_as(fp), 0, scores.ctypes.data_as(fp), idx.ctypes.data_as(C.POINTER(C.c_int)))


def _load_file(lib, path):
    lib.lib.clip_image_load_from_file.restype = C.c_bool
    lib.lib.clip_image_load_from_file.argtypes = [C.c_char_p, C.POINTER(bd.clip_image_u8)]
    im = bd.clip_image_u8()
    if not lib.lib.clip_image_load_from_file(path.encode(), C.byref(im)):
        return None
    return np.ctypeslib.as_array(im.data, shape=(im.ny, im.nx, 3)).copy()


def test_png_decode_matches_pil_and_rejects_unknown_formats(prod, tmp_path):
    """clip_image_load_from_file (clip.cpp:709-726): PNG of every colour type decodes to the 3-channel pixels stb_image / PIL give;
    a format without a decoder here (TIFF) is refused with an explicit message instead of garbage."""
    Image = pytest.importorskip("PIL.Image")
    rng = np.random.default_rng(0)
    rgb = rng.integers(0, 256, (37, 53, 3), dtype=np.uint8)
    files = {"rgb.png": Image.fromarray(rgb), "rgba.png": Image.fromarray(rng.integers(0, 256, (20, 31, 4), dtype=np.uint8), "RGBA"),
             "gray.png": Image.fromarray(rng.integers(0, 256, (20, 31), dtype=np.uint8), "L"),
             "pal.png": Image.fromarray(rgb).convert("P", palette=Image.ADAPTIVE)}
    for name, im in files.items():
        p = str(tmp_path / name)
        im.save(p, optimize=(name == "rgb.png"))
        got = _load_file(prod, p)
        assert got is not None, (name, prod.last_error())
        assert np.array_equal(got, np.array(Image.open(p).convert("RGB"))), name
    g = str(tmp_path / "x.tif")
    Image.fromarray(rgb).save(g)
    assert _load_file(prod, g) is None and b"supported formats" in prod.lib.clip_b200_last_error()


def test_png_decode_matches_live_reference(prod, tmp_path):
    Image = pytest.importorskip("PIL.Image")
    rng = np.random.default_rng(1)
    ref = _reference_decodes("png_pil")
    ims = {"g16.png": Image.fromarray(rng.integers(0, 65536, (11, 13), dtype=np.uint16)),
           "la.png": Image.fromarray(rng.integers(0, 256, (20, 31, 2), dtype=np.uint8), "LA"),
           "rgb.png": Image.fromarray(rng.integers(0, 256, (64, 48, 3), dtype=np.uint8))}
    for name, im in ims.items():
        p = str(tmp_path / name)
        im.save(p)
        ref.check(p, _load_file(prod, p))
    ref.done()


def _write_png(path, arr, ctype, depth, interlace=False, palette=None):
    """Minimal PNG writer for the decoder tests (PIL cannot write interlaced files or pick bit depths): every colour type / bit depth,
    Adam7, and a different filter type on every row so all five predictors run."""
    import struct
    import zlib
    arr = np.asarray(arr)
    h, w = arr.shape[:2]
    ch = {0: 1, 2: 3, 3: 1, 4: 2, 6: 4}[ctype]
    a = arr.reshape(h, w, ch).astype(np.uint32)
    bpp = max(1, depth * ch // 8)

    def pack(sub):                                          # (ph, pw, ch) samples -> list of packed row byte strings
        rows = []
        for r in sub:
            flat = r.reshape(-1)
            if depth == 16:
                rows.append(b"".join(struct.pack(">H", int(v)) for v in flat))
            elif depth == 8:
                rows.append(bytes(int(v) for v in flat))
            else:
                bits = "".join(format(int(v), "0%db" % depth) for v in flat)
                bits += "0" * (-len(bits) % 8)
                rows.append(bytes(int(bits[i:i + 8], 2) for i in range(0, len(bits), 8)))
        return rows

    def filt(rows):
        out, prev = bytearray(), bytes(len(rows[0])) if rows else b""
        for y, cur in enumerate(rows):
            t = y % 5
            line = bytearray()
            for i, v in enumerate(cur):
                left = cur[i - bpp] if i >= bpp else 0
                up = prev[i]
                ul = prev[i - bpp] if i >= bpp else 0
                if t == 0:
                    pred = 0
                elif t == 1:
                    pred = left
                elif t == 2:
                    pred = up
                elif t == 3:
                    pred = (left + up) >> 1
                else:
                    pa, pb, pc = abs(up - ul), abs(left - ul), abs(left + up - 2 * ul)
                    pred = left if (pa <= pb and pa <= pc) else (up if pb <= pc else ul)
                line.append((v - pred) & 255)
            out += bytes([t]) + line
            prev = cur
        return bytes(out)

    if interlace:
        raw = b""
        for x0, y0, dx, dy in zip((0, 4, 0, 2, 0, 1, 0), (0, 0, 4, 0, 2, 0, 1), (8, 8, 4, 4, 2, 2, 1), (8, 8, 8, 4, 4, 2, 2)):
            sub = a[y0::dy, x0::dx]
            if sub.size:
                raw += filt(pack(sub))
    else:
        raw = filt(pack(a))

    def chunk(tag, body):
        return struct.pack(">I", len(body)) + tag + body + struct.pack(">I", zlib.crc32(tag + body) & 0xffffffff)

    data = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, depth, ctype, 0, 0, 1 if interlace else 0))
    if palette is not None:
        data += chunk(b"PLTE", bytes(np.asarray(palette, np.uint8).reshape(-1)))
    blob = zlib.compress(raw, 6)
    data += chunk(b"IDAT", blob[:len(blob) // 2]) + chunk(b"IDAT", blob[len(blob) // 2:]) + chunk(b"IEND", b"")
    open(path, "wb").write(data)


def _png_expected(arr, ctype, depth, palette=None):
    """What stb_image returns for 3 requested channels: grey replicated (and scaled up when packed), high byte of 16-bit samples, alpha dropped."""
    a = np.asarray(arr).astype(np.uint32)
    if ctype == 3:
        return np.asarray(palette, np.uint8)[a]
    if depth == 16:
        a = a >> 8
    elif depth < 8:
        a = a * (255 // ((1 << depth) - 1))
    a = a.astype(np.uint8)
    if ctype == 0:
        return np.repeat(a[..., None], 3, -1)
    if ctype == 4:
        return np.repeat(a[..., :1], 3, -1)
    return a[..., :3]


def test_png_every_colour_type_depth_and_interlace(prod, tmp_path):
    """clip_image_load_from_file on PNGs PIL cannot write: packed 1/2/4-bit grey and palette, 16-bit, Adam7 -- against the pixel rule of
    stb_image (computed here) and against what the reference library returned for each file."""
    rng = np.random.default_rng(11)
    ref = _reference_decodes("png_modes")
    pal = rng.integers(0, 256, (256, 3), dtype=np.uint8)
    n = 0
    for (w, h) in [(1, 1), (3, 2), (7, 9), (8, 8), (13, 5), (33, 17)]:
        for interlace in (False, True):
            cases = [(0, d, rng.integers(0, 1 << d, (h, w))) for d in (1, 2, 4, 8, 16)]
            cases += [(3, d, rng.integers(0, 1 << d, (h, w))) for d in (1, 2, 4, 8)]
            cases += [(2, d, rng.integers(0, 1 << d, (h, w, 3))) for d in (8, 16)]
            cases += [(4, d, rng.integers(0, 1 << d, (h, w, 2))) for d in (8, 16)]
            cases += [(6, d, rng.integers(0, 1 << d, (h, w, 4))) for d in (8, 16)]
            for ctype, depth, arr in cases:
                p = str(tmp_path / "t.png")
                _write_png(p, arr, ctype, depth, interlace, pal if ctype == 3 else None)
                got = _load_file(prod, p)
                assert got is not None, (w, h, ctype, depth, interlace, prod.last_error())
                assert np.array_equal(got, _png_expected(arr, ctype, depth, pal)), (w, h, ctype, depth, interlace)
                ref.check(p, got)
                n += 1
    assert n == 6 * 2 * 15
    ref.done()


def _bmp(w, h, bpp, row_fn, hsz=40, comp=0, masks=None, palette=None, topdown=False):
    """BMP writer for the decoder tests: OS/2 (12) and Windows (40 / 108 / 124) headers, palettes, BI_BITFIELDS, both row orders."""
    import struct
    pal = b"" if palette is None else b"".join(bytes([p[2], p[1], p[0]]) + (b"" if hsz == 12 else b"\0") for p in palette)
    extra = b""
    if hsz == 12:
        hdr = struct.pack("<IHHHH", 12, w, h, 1, bpp)
    else:
        hdr = struct.pack("<IiiHHIIiiII", hsz, w, -h if topdown else h, 1, bpp, comp, 0, 2835, 2835, 0, 0)
        if hsz == 40 and comp == 3:
            extra = struct.pack("<III", *masks)
        if hsz >= 108:
            m = masks or (0, 0, 0)
            hdr += struct.pack("<IIII", m[0], m[1], m[2], 0) + b"\0" * (hsz - 56)
    stride = ((w * bpp + 31) // 32) * 4
    rows = [row_fn(y) for y in (range(h) if topdown else range(h - 1, -1, -1))]
    offs = 14 + len(hdr) + len(extra) + len(pal)
    return b"BM" + struct.pack("<IHHI", offs + stride * h, 0, 0, offs) + hdr + extra + pal + b"".join(r + b"\0" * (stride - len(r)) for r in rows)


def _field(v, mask):
    """BI_BITFIELDS: the masked field, widened to 8 bits by repeating its bits (what stb_image does)."""
    n = bin(mask).count("1")
    lo = (mask & -mask).bit_length() - 1
    f = (int(v) & mask) >> lo
    bits = format(f, "0%db" % n) * 8
    return int(bits[:8], 2)


def test_bmp_and_pnm_variants(prod, tmp_path):
    """clip_image_load_from_file on BMP (palettes of 1/4/8 bits, 16-bit 555 / 565 / 444, 24-bit, 32-bit, V3/V4/V5 and OS/2 headers,
    top-down rows) and binary PGM / PPM: against the rule computed here and what the reference library returned for each file."""
    rng = np.random.default_rng(21)
    ref = _reference_decodes("bmp_pnm")
    p = str(tmp_path / "t.bin")

    def check(data, want, vs_ref=True):
        open(p, "wb").write(data)
        got = _load_file(prod, p)
        assert got is not None, prod.last_error()
        assert np.array_equal(got, want)
        if vs_ref:
            ref.check(p, got)

    for (w, h) in [(1, 1), (5, 3), (13, 7), (33, 10)]:
        for topdown in (False, True):
            px = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
            check(_bmp(w, h, 24, lambda y: bytes(px[y, :, 2::-1].reshape(-1)), topdown=topdown), px[..., :3])
            for hsz in (40, 108, 124):
                check(_bmp(w, h, 32, lambda y: bytes(px[y][:, [2, 1, 0, 3]].reshape(-1)), hsz=hsz, topdown=topdown), px[..., :3])
                v16 = rng.integers(0, 65536, (h, w), dtype=np.uint16)
                for comp, masks in ((0, (0x7C00, 0x03E0, 0x001F)), (3, (0xF800, 0x07E0, 0x001F)), (3, (0x0F00, 0x00F0, 0x000F))):
                    want = np.array([[[_field(v, m) for m in masks] for v in r] for r in v16], np.uint8)
                    check(_bmp(w, h, 16, lambda y: v16[y].astype("<u2").tobytes(), hsz=hsz, comp=comp, masks=masks, topdown=topdown), want)
            for bpp in (1, 4, 8):
                pal = rng.integers(0, 256, (1 << bpp, 3), dtype=np.uint8)
                idx = rng.integers(0, 1 << bpp, (h, w))

                def row(y):
                    bits = "".join(format(int(v), "0%db" % bpp) for v in idx[y])
                    bits += "0" * (-len(bits) % 8)
                    return bytes(int(bits[i:i + 8], 2) for i in range(0, len(bits), 8))
                check(_bmp(w, h, bpp, row, palette=pal, topdown=topdown), pal[idx])
                if not topdown:     # OS/2 header: the reference reads part of the palette from uninitialised memory -- rule only
                    check(_bmp(w, h, bpp, row, hsz=12, palette=pal), pal[idx], vs_ref=False)
    g = rng.integers(0, 256, (5, 7), dtype=np.uint8)
    c = rng.integers(0, 256, (5, 7, 3), dtype=np.uint8)
    check(b"P5\n# comment\n7 5\n255\n" + g.tobytes(), np.repeat(g[..., None], 3, -1))
    check(b"P5 7 5 15\n" + (g & 15).tobytes(), np.repeat((g & 15)[..., None], 3, -1))
    check(b"P6\n#a\n7\n#b\n5\n255\n" + c.tobytes(), c)
    open(p, "wb").write(b"P6 7 5 65535\n" + bytes(7 * 5 * 6))
    assert _load_file(prod, p) is None
    rle = bytearray(_bmp(4, 4, 8, lambda y: bytes(4), palette=rng.integers(0, 256, (256, 3), dtype=np.uint8)))
    rle[30] = 1                                                    # BI_RLE8: refused, as in the reference
    open(p, "wb").write(bytes(rle))
    assert _load_file(prod, p) is None
    ref.done()


def _gif_lzw(indices, min_bits, grow=True):
    """GIF LZW.  grow=False: a clear code before the code width would change (fixed-width stream); grow=True: a real dictionary coder."""
    clear, eoi = 1 << min_bits, (1 << min_bits) + 1
    out, state = bytearray(), [0, 0]

    def emit(code, width):
        state[0] |= code << state[1]
        state[1] += width
        while state[1] >= 8:
            out.append(state[0] & 255)
            state[0] >>= 8
            state[1] -= 8
    width = min_bits + 1
    emit(clear, width)
    if not grow:
        for i, v in enumerate(indices):
            if i and i % (clear - 2) == 0:
                emit(clear, width)
            emit(int(v), width)
    else:
        table, nxt, cur = {(i,): i for i in range(clear)}, eoi + 1, ()
        for v in indices:
            k = cur + (int(v),)
            if k in table:
                cur = k
                continue
            emit(table[cur], width)
            table[k] = nxt
            nxt += 1
            if nxt > (1 << width) and width < 12:
                width += 1
            if nxt >= 4095:
                emit(clear, width)
                table, nxt, width = {(i,): i for i in range(clear)}, eoi + 1, min_bits + 1
            cur = (int(v),)
        if cur:
            emit(table[cur], width)
    emit(eoi, width)
    if state[1]:
        out.append(state[0] & 255)
    return bytes([min_bits]) + b"".join(bytes([len(out[i:i + 255])]) + bytes(out[i:i + 255]) for i in range(0, len(out), 255)) + b"\0"


def _gif(W, H, gpal, frame, x0=0, y0=0, bg=0, transparent=None, interlace=False, lpal=None, grow=True):
    import struct
    h, w = frame.shape

    def table(p):
        n = max(1, int(np.ceil(np.log2(max(len(p), 2)))))
        return n, bytes(np.asarray(p, np.uint8).reshape(-1)) + b"\0" * (3 * ((1 << n) - len(p)))
    d = b"GIF89a"
    if gpal is not None:
        n, t = table(gpal)
        d += struct.pack("<HHBBB", W, H, 0x80 | (n - 1), bg, 0) + t
    else:
        d += struct.pack("<HHBBB", W, H, 0, bg, 0)
    d += b"\x21\xFE\x05hello\0"
    if transparent is not None:
        d += b"\x21\xF9\x04" + bytes([1, 0, 0, transparent]) + b"\0"
    rows = list(range(h))
    if interlace:
        rows = list(range(0, h, 8)) + list(range(4, h, 8)) + list(range(2, h, 4)) + list(range(1, h, 2))
    ncol = len(lpal) if lpal is not None else len(gpal)
    lf = 0x40 if interlace else 0
    if lpal is not None:
        n, t = table(lpal)
        d += b"\x2C" + struct.pack("<HHHHB", x0, y0, w, h, lf | 0x80 | (n - 1)) + t
    else:
        d += b"\x2C" + struct.pack("<HHHHB", x0, y0, w, h, lf)
    return d + _gif_lzw(frame[rows].reshape(-1), max(2, int(np.ceil(np.log2(max(ncol, 2))))), grow) + b"\x3B"


def test_gif_first_frame(prod, tmp_path):
    """clip_image_load_from_file on GIF: the first frame as stb_image composes it (transparent pixels black, uncovered canvas = background
    colour when its index is non-zero -- with red and blue swapped, a quirk of the reference that is kept), interlaced rows, local
    colour tables, both LZW styles; against the rule computed here and what the reference library returned for each file."""
    rng = np.random.default_rng(31)
    ref = _reference_decodes("gif")
    p = str(tmp_path / "t.gif")

    def check(data, want):
        open(p, "wb").write(data)
        got = _load_file(prod, p)
        assert got is not None, prod.last_error()
        assert np.array_equal(got, want)
        ref.check(p, got)

    for (W, H) in [(1, 1), (7, 5), (33, 21), (120, 90)]:
        for ncol in (2, 16, 200, 256):
            pal = rng.integers(0, 256, (ncol, 3), dtype=np.uint8)
            lp = rng.integers(0, 256, (ncol, 3), dtype=np.uint8)
            fr = rng.integers(0, ncol, (H, W))
            smooth = (np.add.outer(np.arange(H), np.arange(W)) // 3) % ncol
            for grow in (False, True):
                for il in (False, True):
                    check(_gif(W, H, pal, fr, interlace=il, grow=grow), pal[fr])
                    check(_gif(W, H, pal, smooth, interlace=il, grow=grow), pal[smooth])
            want = pal[fr].copy()
            want[fr == 1] = 0
            check(_gif(W, H, pal, fr, transparent=1), want)
            check(_gif(W, H, None, fr, lpal=lp), lp[fr])
            if W > 4 and H > 3:
                sub = fr[1:H - 1, 2:W - 1]
                for bg in (0, ncol - 1):
                    want = np.zeros((H, W, 3), np.uint8)
                    if bg:
                        want[:] = pal[bg][::-1]
                    want[1:H - 1, 2:W - 1] = pal[sub]
                    check(_gif(W, H, pal, sub, x0=2, y0=1, bg=bg, interlace=True), want)
    open(p, "wb").write(b"GIF89a" + bytes(7) + b"\x3B")
    assert _load_file(prod, p) is None
    ref.done()


JPEG_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "jpeg")


def test_jpeg_decode_matches_reference_golden(prod):
    """JPEG files decode to exactly the pixels the reference's loader (stb_image, clip.cpp:709-726) produces: baseline and progressive,
    every sampling layout, restart intervals, grey / RGB / CMYK / YCCK.  tests/golden/jpeg/manifest.json holds the sha256 of the
    reference's output for each committed file (tests/golden/make_jpeg_golden.py)."""
    import hashlib
    import json
    files = json.load(open(os.path.join(JPEG_GOLDEN, "manifest.json")))["files"]
    assert len(files) >= 30
    for name, want in sorted(files.items()):
        got = _load_file(prod, os.path.join(JPEG_GOLDEN, name + ".jpg"))
        assert got is not None, (name, prod.last_error())
        assert got.shape == (want["ny"], want["nx"], 3), name
        assert hashlib.sha256(got.tobytes()).hexdigest() == want["sha256"], (name, float(got.mean()), want["mean"])


def test_jpeg_decode_matches_live_reference(prod, tmp_path):
    """Same comparison on files PIL writes here (sizes x sampling x mode x quality), against what the reference library returned for
    them, and on the two sample JPEGs the reference ships (tests/golden/jpeg/ref_*.jpg)."""
    Image = pytest.importorskip("PIL.Image")
    rng = np.random.default_rng(5)
    ref = _reference_decodes("jpeg_pil", pin_files=True)
    p = str(tmp_path / "t.jpg")
    n = 0
    for (w, h) in [(1, 1), (8, 8), (15, 9), (33, 17), (100, 75), (224, 224), (1234, 901)]:       # the last one is > 1 MP: threaded IDCT / colour rows
        y, x = np.mgrid[0:h, 0:w]
        pics = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8),
                np.stack([np.sin(x / 3.0) * 127 + 128, np.cos(y / 5.0) * 127 + 128, ((x // 4 + y // 4) % 2) * 255], -1).astype(np.uint8)]
        for pic in pics:
            for sub in ("4:4:4", "4:2:2", "4:2:0"):
                for prog in (False, True):
                    q = int(rng.integers(5, 100))
                    Image.fromarray(pic).save(p, quality=q, subsampling=sub, progressive=prog, optimize=bool(n & 1))
                    ref.check(p, _load_file(prod, p))
                    n += 1
    for name in ("ref_red_apple", "ref_white"):
        f = os.path.join(JPEG_GOLDEN, name + ".jpg")
        ref.check(f, _load_file(prod, f))
    ref.done()


def test_jpeg_decoder_survives_corrupt_files(prod, tmp_path):
    """Truncated and bit-flipped JPEGs are refused or decoded to *something* of the declared size -- never a crash or an out-of-bounds
    read (the decoder was also run under ASan/UBSan over 18k such files)."""
    rng = np.random.default_rng(9)
    p = str(tmp_path / "c.jpg")
    for name in ("pil_420_prog", "pil_rst_base", "enc_420_noninterleaved_dri", "pil_cmyk_prog_420"):
        blob = open(os.path.join(JPEG_GOLDEN, name + ".jpg"), "rb").read()
        for it in range(150):
            m = bytearray(blob)
            if it % 3 == 0:
                m = m[:int(rng.integers(0, len(m)))]
            else:
                for _ in range(int(rng.integers(1, 4 if it % 3 == 1 else 40))):
                    m[int(rng.integers(0, len(m)))] = int(rng.integers(0, 256))
            open(p, "wb").write(bytes(m))
            got = _load_file(prod, p)
            assert got is None or got.ndim == 3


def test_gguf_parser_survives_corrupt_files(prod, tmp_path):
    """ADVICE r1: hostile / corrupt GGUF input must be refused, never read out of bounds.  The parser is shared by clip_model_load and
    clip_model_quantize; the quantizer runs it without a GPU."""
    src = model_file("tiny", "f16", prod)
    blob = bytearray(open(src, "rb").read())
    out = str(tmp_path / "out.gguf")

    def attempt(data, name):
        p = str(tmp_path / name)
        with open(p, "wb") as f:
            f.write(data)
        return prod.quantize(p, out, 2)

    assert attempt(bytes(blob), "ok.gguf")                                        # the unmodified file converts
    for cut in (0, 3, 11, 24, 200, 5000, len(blob) // 2, len(blob) - 7):            # truncations: header, kv area, tensor infos, data
        assert not attempt(bytes(blob[:cut]), "cut%d.gguf" % cut)
    bad = bytearray(blob); bad[0:4] = b"XXXX"
    assert not attempt(bytes(bad), "magic.gguf")
    bad = bytearray(blob); bad[8:16] = (2 ** 40).to_bytes(8, "little")             # absurd tensor count
    assert not attempt(bytes(bad), "ntensors.gguf")
    bad = bytearray(blob); bad[16:24] = (2 ** 40).to_bytes(8, "little")            # absurd kv count
    assert not attempt(bytes(bad), "nkv.gguf")
    # corrupt single bytes all over the metadata: any outcome but a crash is acceptable (most flips are refused, some are harmless)
    rng = np.random.default_rng(0)
    meta_end = blob.find(b"v.blk.0.attn_q.weight")
    for k in range(60):
        bad = bytearray(blob)
        pos = int(rng.integers(24, meta_end + 4000))
        bad[pos] ^= int(rng.integers(1, 256))
        attempt(bytes(bad), "flip.gguf")


def test_reference_examples_link_unchanged_and_fail_loudly_without_a_gpu(prod):
    """oracle/Makefile `examples`: the reference's examples/{simple.c,main.cpp,zsl.cpp,extract.cpp} compile and link against
    include/clip.h + libclip_b200.so as they are (the drop-in claim at the source level).  On a box without a GPU the resulting program
    must stop at clip_model_load with the library's message -- there is no CPU path to fall into."""
    import subprocess
    from _util import ROOT
    bins = [os.path.join(ROOT, "oracle", "_ref", b) for b in ("ex_simple_b200", "ex_main_b200", "ex_zsl_b200", "ex_extract_b200")]
    if not all(os.path.exists(b) for b in bins):
        pytest.skip("oracle/_ref/ex_*_b200 not built (needs /root/reference: make -C oracle examples)")
    if prod.lib.clip_b200_cuda_device_count() > 0:
        pytest.skip("a GPU is present: tests/test_gpu_zz_examples.py runs the programs for real")
    model = model_file("tiny", "f16", prod)
    r = subprocess.run([bins[1], "-m", model, "--text", "apple", "--image", os.path.join(JPEG_GOLDEN, "pil_444_base.jpg")],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and "no CUDA device" in (r.stdout + r.stderr), (r.returncode, r.stdout[-300:], r.stderr[-300:])


def test_jpeg_portable_loops_give_the_same_bytes():
    """csrc/jpeg.cpp picks AVX2 kernels for the inverse DCT and the colour rows at run time; CLIP_B200_JPEG_SIMD=0 keeps the portable
    loops.  Both must produce the reference's pixels: the golden-hash test is run again in a process with the switch set."""
    import subprocess
    import sys
    env = dict(os.environ, CLIP_B200_JPEG_SIMD="0")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-p", "no:cacheprovider", os.path.abspath(__file__) + "::test_jpeg_decode_matches_reference_golden"],
                       capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0 and "1 passed" in r.stdout, r.stdout[-800:] + r.stderr[-400:]
