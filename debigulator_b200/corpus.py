"""Synthetic corpora of the shapes BASELINE.json names (SURVEY.md 8d).

Pure Python / numpy / zlib: usable on the GPU box, independent of the oracle.
gzip members are hand-framed (10-byte header, FLG=0, deflate stream, CRC32,
ISIZE); PNGs are written here with a fixed-Huffman zlib stream (the shape
stb_image_write produces: one IDAT, filter forced or adaptive), so the decoder
under test never sees its own encoder.
"""
import ctypes
import struct
import zlib

import numpy as np

_TOOLS = None


def _tools():
    """Builds (gcc, once) and loads the corpus tools: the single-block fixed-Huffman encoder."""
    global _TOOLS
    if _TOOLS is None:
        from .build import build_corpus_tools
        L = ctypes.CDLL(build_corpus_tools())
        L.dbg_fixed_deflate.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t]
        L.dbg_fixed_deflate.restype = ctypes.c_size_t
        _TOOLS = L
    return _TOOLS


def fixed_block_deflate(data):
    """Raw DEFLATE of `data` as ONE final fixed-Huffman block (the shape stb_image_write emits)."""
    data = bytes(data)
    cap = len(data) + len(data) // 4 + 64
    out = ctypes.create_string_buffer(cap)
    n = _tools().dbg_fixed_deflate(data, len(data), out, cap)
    assert n <= cap
    return out.raw[:n]

_STB = None


def stb_available():
    from .build import build_tools
    return build_tools() is not None


def _stb():
    """The reference's vendored stb_image_write (tools/stb_gen.c, compiled against /root/reference/src/stb_write.h)."""
    global _STB
    if _STB is None:
        from .build import build_tools
        path = build_tools()
        if path is None:
            raise RuntimeError("tools/libstbgen.so is missing and /root/reference is not here to build it")
        L = ctypes.CDLL(path)
        L.stbgen_png.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
        L.stbgen_png.restype = ctypes.c_void_p
        L.stbgen_zlib.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
        L.stbgen_zlib.restype = ctypes.c_void_p
        L.stbgen_free.argtypes = [ctypes.c_void_p]
        L.stbgen_free.restype = None
        _STB = L
    return _STB


def stb_png(pixels, w, h, comp=4, filt=-1):
    """PNG bytes written by stb_image_write (stb_write.h:1128): one IDAT, one fixed-Huffman block."""
    L = _stb()
    n = ctypes.c_int(0)
    px = np.ascontiguousarray(np.frombuffer(pixels, np.uint8) if isinstance(pixels, (bytes, bytearray)) else pixels)
    assert px.size == w * h * comp
    p = L.stbgen_png(px.ctypes.data, w, h, comp, filt, ctypes.byref(n))
    out = ctypes.string_at(p, n.value)
    L.stbgen_free(p)
    return out


def stb_zlib(data, quality=8):
    L = _stb()
    n = ctypes.c_int(0)
    buf = ctypes.create_string_buffer(bytes(data), len(data))
    p = L.stbgen_zlib(buf, len(data), quality, ctypes.byref(n))
    out = ctypes.string_at(p, n.value)
    L.stbgen_free(p)
    return out


GZ_SEED_BASE = 0x64620000


def _rng(seed):
    return np.random.default_rng(seed)


def word_salad(n, seed, vocab=3000):
    """n bytes of space-separated pseudo-words drawn uniformly from a 3000-word
    vocabulary: deflate ratio ~1.9 with the fixed code, ~2.4 dynamic (SURVEY.md 8d)."""
    r = _rng(seed)
    lens = r.integers(2, 10, size=vocab)
    words = [bytes(r.integers(97, 123, size=int(l), dtype=np.uint8)) + b" " for l in lens]
    out = bytearray()
    while len(out) < n:
        idx = r.integers(0, vocab, size=20000)
        out += b"".join(words[i] for i in idx)
    return bytes(out[:n])


def low_entropy(n, seed, alphabet=4):
    r = _rng(seed)
    return bytes(r.integers(97, 97 + alphabet, size=n, dtype=np.uint8))


def periodic(n, seed, period):
    r = _rng(seed)
    base = bytes(r.integers(0, 256, size=period, dtype=np.uint8))
    return (base * (n // period + 1))[:n]


def runs(n, seed):
    r = _rng(seed)
    out = bytearray()
    while len(out) < n:
        out += bytes([int(r.integers(0, 256))]) * int(r.integers(200, 60000))
    return bytes(out[:n])


def raw_deflate(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    return c.compress(data) + c.flush()


def mixed_deflate(data, seed):
    """3-9 segments (stored / fixed / dynamic), all but the last closed with
    Z_FULL_FLUSH, in ONE raw deflate stream (SURVEY.md 8d cfg2 class 3)."""
    r = _rng(seed)
    nseg = int(r.integers(3, 10))
    cuts = sorted(set(int(x) for x in r.integers(1, max(2, len(data) - 1), size=nseg - 1)))
    bounds = [0] + cuts + [len(data)]
    out = b""
    for k in range(len(bounds) - 1):
        seg = data[bounds[k]:bounds[k + 1]]
        mode = int(r.integers(0, 3))
        level, strat = [(0, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_FIXED), (int(r.choice([1, 6, 9])), zlib.Z_DEFAULT_STRATEGY)][mode]
        c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strat)
        last = k == len(bounds) - 2
        body = c.compress(seg) + (c.flush(zlib.Z_FINISH) if last else c.flush(zlib.Z_FULL_FLUSH))
        if not last:
            pass  # Z_FULL_FLUSH leaves BFINAL=0 on every block and ends byte-aligned
        out += body
    return out


def gzip_frame(deflate, data, fname=None):
    flg = 8 if fname else 0
    hdr = bytes([31, 139, 8, flg, 0, 0, 0, 0, 0, 255])
    if fname:
        hdr += fname + b"\0"
    return hdr + deflate + struct.pack("<II", zlib.crc32(data) & 0xFFFFFFFF, len(data) & 0xFFFFFFFF)


def gz_member_cfg2(i, size=1 << 20):
    """BASELINE config 2 member i: class i%4 = stored / fixed / dynamic / mixed.
    Returns (gzip bytes, payload bytes)."""
    seed = GZ_SEED_BASE + i
    cls = i % 4
    if cls == 0:
        data = bytes(_rng(seed).integers(0, 256, size=size, dtype=np.uint8))
        d = raw_deflate(data, 0)
    elif cls == 1:
        data = word_salad(size, seed)
        d = raw_deflate(data, 6, zlib.Z_FIXED)
    elif cls == 2:
        data = word_salad(size, seed)
        d = raw_deflate(data, 6)
    else:
        data = word_salad(size, seed)
        d = mixed_deflate(data, seed)
    return gzip_frame(d, data), data


def gz_member_cfg5(i, size):
    """BASELINE config 5 member i: compressibility sweep by i%8."""
    seed = GZ_SEED_BASE + 0x50000 + i
    cls = i % 8
    if cls == 0:
        data = bytes(_rng(seed).integers(0, 256, size=size, dtype=np.uint8)); d = raw_deflate(data, 0)
    elif cls == 1:
        data = word_salad(size, seed); d = raw_deflate(data, 6)
    elif cls == 2:
        data = word_salad(size, seed); d = raw_deflate(data, 1)
    elif cls == 3:
        data = low_entropy(size, seed, 6); d = raw_deflate(data, 6, zlib.Z_HUFFMAN_ONLY)
    elif cls == 4:
        data = periodic(size, seed, 20000 + (i * 37) % 12000); d = raw_deflate(data, 6)
    elif cls == 5:
        data = periodic(size, seed, 32000); d = raw_deflate(data, 9)
    elif cls == 6:
        data = runs(size, seed); d = raw_deflate(data, 6)
    else:
        data = bytes(size); d = raw_deflate(data, 9)
    return gzip_frame(d, data), data


# ------------------------------------------------------------------- PNG --------
def gradient_noise_rgba(w, h, seed, amp=6):
    """Smooth gradient + low-amplitude noise (never pure noise: see SURVEY.md Q12)."""
    r = _rng(seed)
    y, x = np.mgrid[0:h, 0:w]
    img = np.empty((h, w, 4), dtype=np.uint8)
    img[..., 0] = (x * 255 // max(w - 1, 1)).astype(np.uint8)
    img[..., 1] = (y * 255 // max(h - 1, 1)).astype(np.uint8)
    img[..., 2] = ((x + y) * 255 // max(w + h - 2, 1)).astype(np.uint8)
    img[..., 3] = 255 - (x // 8 % 64).astype(np.uint8)
    noise = r.integers(0, amp, size=(h, w, 4), dtype=np.uint8)
    return (img + noise).astype(np.uint8)


def _paeth(a, b, c):
    a = a.astype(np.int16); b = b.astype(np.int16); c = c.astype(np.int16)
    p = a + b - c
    pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
    return np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c)).astype(np.uint8)


def png_filter_rows(img, filt):
    """img: (h, w, bpp) uint8. filt 0..4 forced, -1 = per-row minimum-sum choice, a sequence = one filter type per row."""
    h, w, bpp = img.shape
    raw = img.reshape(h, w * bpp)
    left = np.zeros_like(raw); left[:, bpp:] = raw[:, :-bpp]
    up = np.zeros_like(raw); up[1:] = raw[:-1]
    ul = np.zeros_like(raw); ul[1:, bpp:] = raw[:-1, :-bpp]
    cands = [raw, raw - left, raw - up,
             raw - ((left.astype(np.uint16) + up.astype(np.uint16)) >> 1).astype(np.uint8),
             raw - _paeth(left, up, ul)]
    out = np.empty((h, w * bpp + 1), dtype=np.uint8)
    if not np.isscalar(filt):
        best = np.asarray(filt, dtype=np.int64)
        out[:, 0] = best
        out[:, 1:] = np.stack(cands)[best, np.arange(h)]
    elif filt >= 0:
        out[:, 0] = filt
        out[:, 1:] = cands[filt]
    else:
        cost = np.stack([np.abs(c.astype(np.int8).astype(np.int32)).sum(axis=1) for c in cands])
        best = cost.argmin(axis=0)
        out[:, 0] = best
        allc = np.stack(cands)
        out[:, 1:] = allc[best, np.arange(h)]
    return out.tobytes()


def _chunk(tag, data):
    return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data) & 0xFFFFFFFF)


def write_png(img, filt=-1, level=6, strategy=zlib.Z_FIXED, idat_split=0, color_type=None, palette=None, extra_chunks=(),
              single_block=False):
    """Minimal PNG writer: 8-bit, colour type from the channel count (4 -> 6, 3 -> 2, 1 -> 3).
    single_block=True writes the zlib stream the way stb_image_write does: header 78 5E, one final
    fixed-Huffman block, Adler-32."""
    h, w, bpp = img.shape
    ct = color_type if color_type is not None else {4: 6, 3: 2, 1: 3}[bpp]
    rows = png_filter_rows(img, filt)
    if single_block:
        stream = b"\x78\x5e" + fixed_block_deflate(rows) + struct.pack(">I", zlib.adler32(rows) & 0xFFFFFFFF)
    else:
        z = zlib.compressobj(level, zlib.DEFLATED, 15, 8, strategy)
        stream = z.compress(rows) + z.flush()
    out = b"\x89PNG\r\n\x1a\n" + _chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, ct, 0, 0, 0))
    if ct == 3:
        out += _chunk(b"PLTE", bytes(palette))
    for tag, data in extra_chunks:
        out += _chunk(tag, data)
    if idat_split:
        for k in range(0, len(stream), idat_split):
            out += _chunk(b"IDAT", stream[k:k + idat_split])
    else:
        out += _chunk(b"IDAT", stream)
    return out + _chunk(b"IEND", b"")


def png_cfg3(i, w=1024, h=1024, filt=None):
    """BASELINE config 3 image i: filter forced to i%6-1 (-1 = adaptive) unless `filt` says otherwise. Returns (png bytes,
    rgba bytes). Written by this module's own encoder (tools/fixed_deflate.c): the stream shape stb writes, not stb itself."""
    img = gradient_noise_rgba(w, h, 0x706E6700 + i)
    return write_png(img, filt=(i % 6 - 1) if filt is None else filt, single_block=True), img.tobytes()


def png_bench(i, w=1024, h=1024, filt=None):
    """BASELINE config 3 / 4 image i as the benchmark times it: written by stb_image_write when that tooling is built
    (png_stb), else by this module's own encoder of the same stream shape (png_cfg3). Same pixels either way."""
    return (png_stb if stb_available() else png_cfg3)(i, w, h, filt)


def png_stb(i, w=1024, h=1024, filt=None):
    """BASELINE config 3 / 4 image i written by stb_image_write itself (SURVEY.md 8d): smooth gradient + low-amplitude
    noise, filter forced to i%6-1 (-1 = adaptive) unless `filt` says otherwise. Returns (png bytes, rgba bytes)."""
    img = gradient_noise_rgba(w, h, 0x706E6700 + i)
    return stb_png(img, w, h, 4, (i % 6 - 1) if filt is None else filt), img.tobytes()


def bmp_file(rgba: bytes, w: int, h: int, bottom_up: bool = False, v4: bool = False, pad: int = 0,
             bf_size: int = None, planes: int = 1, bpp: int = 32, dib_size: int = None, magic: bytes = b"BM") -> bytes:
    """A 32-bit BMP holding the RGBA image `rgba` (w*h*4 bytes, top row first). `pad` extra bytes sit between the
    headers and the pixels (moves image_offset, e.g. to an odd address); the remaining arguments let tests break
    individual header fields (decode_bmp.c:120-221)."""
    import struct
    assert len(rgba) == w * h * 4
    px = np.frombuffer(rgba, np.uint8).reshape(h, w, 4) if w * h else np.zeros((0, 0, 4), np.uint8)
    bgra = px[:, :, [2, 1, 0, 3]]
    if bottom_up:
        bgra = bgra[::-1]
    dib = 108 if v4 else 40
    offset = 14 + dib + pad
    body = bgra.tobytes()
    total = offset + len(body)
    hdr = magic + struct.pack("<IHHI", total if bf_size is None else bf_size, 0, 0, offset)
    info = struct.pack("<IiiHHIIIIII", dib if dib_size is None else dib_size, w, h if bottom_up else -h, planes, bpp,
                       3 if v4 else 0, len(body), 0, 0, 0, 0)
    if v4:
        info += struct.pack("<IIII", 0x00ff0000, 0x0000ff00, 0x000000ff, 0xff000000) + b"BGRs" + bytes(48)
    return hdr + info + bytes(pad) + body
