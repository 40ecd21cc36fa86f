"""Chunk-level PNG writer and a model of what the reference's decode_png() makes of a file, for the adversarial PNG tests.

The writer puts chunks in any order, with any length field, type bytes, payload and stored CRC (right, flipped, absent,
or solved in GF(2) so that the four bytes the walk reads as the CRC equal the CRC it computes). The zlib stream of the
scanlines (any per-row filter bytes, bpp 1, 3 or 4) may be cut into IDATs anywhere.

`model(data, rgba_size)` restates the reference's chunk walk (decode_png.c:755-1357, oracle/debig_oracle.c:314-458,
png_scan_warp in csrc/png_core.h) with its quirks -- Q11's optimistic `left`, the signed `char > 'Z'` ancillary test, IHDR
always 13 bytes, IEND not stepping over its payload, the inflate point at the first non-IDAT chunk after an IDAT -- and
returns the verdict, the device status and the RGBA a plain un-filter gives. RGB follows the spec (the reference is wrong
there, defect D3); palette indices at or past the palette's size give (0, 0, 0, 255). Where Q11 makes the reference read
outside the file the verdict is "ub": the reference is not called there, and every decoder must fail."""
import struct
import zlib

import numpy as np

from debigulator_b200 import corpus
from oracle import portlib

SIG = b"\x89PNG\r\n\x1a\n"
ST_OK, ST_INPUT_TOO_SMALL, ST_TOO_LARGE, ST_CONTAINER, ST_PNG_CRC, ST_PNG_FILTER, ST_PNG_SHORT = 0, 2, 3, 12, 13, 14, 15
INFLATE = "inflate"  # status of a stream the inflate kernels reject: one of the decoder's own statuses 1..11
SCAN_SEG = 65536     # csrc/png_core.h: chunks with 4 + length above this are CRC'd by segment tasks


def be32(v):
    return struct.pack(">I", v & 0xFFFFFFFF)


def _crc_solve(tag, payload, at):
    """payload with bytes [at, at + 4) replaced so that they hold, big-endian, CRC-32(tag + payload). The CRC is affine
    in those 32 bits: solve (M + I) x = CRC(x = 0) over GF(2), changing a spare byte of the payload if M + I is
    singular and the system has no solution."""
    p = bytearray(payload)
    spare_at = len(p) - 1 if len(p) > at + 4 else at - 1
    for spare in range(256):
        if spare and spare_at < 0:
            break
        if spare:
            p[spare_at] = spare
        def f(x):
            p[at:at + 4] = be32(x)
            return zlib.crc32(bytes(tag) + bytes(p)) & 0xFFFFFFFF
        c0 = f(0)
        rows = [(f(1 << i) ^ c0) ^ (1 << i) for i in range(32)]  # column i of M + I, as a 32-bit word
        # Gaussian elimination on the columns: basis[bit] = (column combination, mask of x bits used)
        basis = {}
        for i, col in enumerate(rows):
            m = 1 << i
            for b in sorted(basis, reverse=True):
                if col >> b & 1:
                    col ^= basis[b][0]
                    m ^= basis[b][1]
            if col:
                basis[col.bit_length() - 1] = (col, m)
        t, x = c0, 0
        for b in sorted(basis, reverse=True):
            if t >> b & 1:
                t ^= basis[b][0]
                x ^= basis[b][1]
        if t == 0:
            f(x)
            assert struct.unpack(">I", bytes(p[at:at + 4]))[0] == zlib.crc32(bytes(tag) + bytes(p)) & 0xFFFFFFFF
            return bytes(p)
    raise ValueError("no self-CRC solution")


def chunk(tag, payload=b"", length=None, crc="ok", solve_at=None):
    """One chunk. length: the length field (default: the payload's). crc: "ok", "flip" (bit 0 of the last byte of the
    right CRC flipped), "none" (no CRC field) or an int. solve_at: payload bytes [solve_at, solve_at + 4) are made
    equal to the chunk's CRC (over the type and the whole payload); the byte after them, or else the one before, is
    changed too if that is what it takes."""
    tag = bytes(tag)
    payload = bytes(payload)
    if solve_at is not None:
        payload = _crc_solve(tag, payload, solve_at)
    c = zlib.crc32(tag + payload) & 0xFFFFFFFF
    if crc == "flip":
        c ^= 1
    tail = b"" if crc == "none" else be32(c if isinstance(crc, str) else crc)
    return be32(len(payload) if length is None else length) + tag + payload + tail


def ihdr(w, h, ct, depth=8, filt=0):
    return chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, depth, ct, 0, filt, 0))


def scanlines(img, filt):
    """Filtered scanlines (corpus.png_filter_rows); filter bytes > 4 are written over the chosen rows' filter bytes."""
    h = img.shape[0]
    f = np.asarray(filt if not np.isscalar(filt) else [filt] * h, np.int64)
    rows = bytearray(corpus.png_filter_rows(img, np.where(f > 4, 0, f)))
    stride = img.shape[1] * img.shape[2] + 1
    for r in np.nonzero(f > 4)[0]:
        rows[r * stride] = int(f[r])
    return bytes(rows)


def zstream(raw, stb=True):
    """zlib stream of `raw`: stb-shaped (78 5E, one final fixed-Huffman block, Adler-32) or zlib's default."""
    if stb:
        return b"\x78\x5e" + corpus.fixed_block_deflate(raw) + be32(zlib.adler32(raw))
    return zlib.compress(raw, 6)


def split(stream, sizes):
    """IDAT chunks of the given payload sizes, the last one taking what is left (sizes may be 0)."""
    out, at = [], 0
    for s in sizes:
        out.append(chunk(b"IDAT", stream[at:at + s]))
        at += s
    if at < len(stream):
        out.append(chunk(b"IDAT", stream[at:]))
    return out


def pad_chunk(at, mod=16, want=0, tag=b"pAdd"):
    """An ancillary chunk for file offset `at` after which the next chunk's payload + `want` lands on 0 mod `mod`."""
    n = (-(at + 12 + 8 + want)) % mod
    return chunk(tag, bytes(n))


def png(chunks, sig=SIG):
    return sig + b"".join(chunks)


# ---------------------------------------------------------------------------------------------------------- model ----
def unfilter(scan, w, h, bpp):
    """Plain reconstruction (PNG spec 9.2; unknown filter types give a zero row, decode_png.c:528-540)."""
    stride = w * bpp
    prev = [0] * stride
    out = np.zeros((h, stride), np.uint8)
    for r in range(h):
        row = scan[r * (stride + 1):(r + 1) * (stride + 1)]
        ft, x = row[0], row[1:]
        if ft == 0:
            cur = list(x)
        elif ft == 2:
            cur = [(v + u) & 255 for v, u in zip(x, prev)]
        elif ft in (1, 3, 4):
            cur = [0] * stride
            for i in range(stride):
                a = cur[i - bpp] if i >= bpp else 0
                b = prev[i]
                if ft == 1:
                    p = a
                elif ft == 3:
                    p = (a + b) >> 1
                else:
                    c = prev[i - bpp] if i >= bpp else 0
                    pa, pb, pc = abs(b - c), abs(a - c), abs(a + b - 2 * c)
                    p = a if pa <= pb and pa <= pc else (b if pb <= pc else c)
                cur[i] = (x[i] + p) & 255
        else:
            cur = [0] * stride
        out[r] = cur
        prev = cur
    return out


def to_rgba(pix, w, h, bpp, plte):
    """RGB -> alpha 255 (the spec, not the reference's D3); palette: entries past the palette's size are black."""
    if bpp == 4:
        return pix.tobytes()
    alpha = np.full((h, w, 1), 255, np.uint8)
    if bpp == 3:
        return np.concatenate([pix.reshape(h, w, 3), alpha], axis=2).tobytes()
    n = len(plte) // 3
    table = np.zeros((256, 3), np.uint8)
    k = min(n, 256)
    table[:k] = np.frombuffer(plte[:3 * k], np.uint8).reshape(k, 3)
    return np.concatenate([table[pix.reshape(h, w)], alpha], axis=2).tobytes()


def model(data, rgba_size=None):
    """What the reference does with `data` when the caller's RGBA size is `rgba_size` (default: from the IHDR at the
    fixed offset 16, as decode_png_get_width_height reads it). Returns dict(verdict "good" / "fail" / "ub", status,
    rgba, w, h, bpp, n_idat, zrun)."""
    size = len(data)
    if rgba_size is None:
        rgba_size = int.from_bytes(data[16:20], "big") * int.from_bytes(data[20:24], "big") * 4 if size >= 24 else 0
    res = dict(verdict="fail", status=ST_CONTAINER, rgba=None, w=0, h=0, bpp=0, n_idat=0, zrun=0)

    def fail(st, ub=False):
        res.update(status=st, verdict="ub" if ub else "fail")
        return res

    if size < 8 or data[1:4] != b"PNG":
        return fail(ST_CONTAINER)
    pos, left = 8, size - 8
    found_idat = ran = found_ihdr = found_iend = False
    zlen = zrun = 0
    w = h = ct = 0
    plte = b""
    z = bytearray()
    while left >= 8 and not found_iend:
        if pos + 8 > size:
            return fail(ST_CONTAINER, ub=True)
        length = int.from_bytes(data[pos:pos + 4], "big")
        typ = data[pos + 4:pos + 8]
        pos += 8
        left -= 8
        is_idat = typ == b"IDAT"
        if not is_idat and found_idat:
            ran, zrun = True, zlen
        if length >= left:
            return fail(ST_CONTAINER)
        if pos + length + 4 > size:
            return fail(ST_CONTAINER, ub=True)
        crc = zlib.crc32(typ + data[pos:pos + length]) & 0xFFFFFFFF
        if typ == b"PLTE":
            if not found_ihdr or length % 3:
                return fail(ST_CONTAINER)
            plte = data[pos:pos + length]
            pos += length
        elif typ == b"IHDR":
            found_ihdr = True
            if pos + 13 > size:
                return fail(ST_CONTAINER, ub=True)
            b = data[pos:pos + 13]
            pos += 13
            w, h = int.from_bytes(b[0:4], "big"), int.from_bytes(b[4:8], "big")
            ct = b[9]
            if w * h * 4 != rgba_size:
                return fail(ST_CONTAINER)
            if w * h * 4 + h + 1 >= 1 << 32:
                return fail(ST_TOO_LARGE)
            if ct not in (2, 3, 6) or w < 1 or h < 1 or b[8] != 8 or b[11] != 0 or left < 4:
                return fail(ST_CONTAINER)
        elif is_idat:
            if not found_ihdr:
                return fail(ST_CONTAINER)
            payload = data[pos:pos + length]
            if not found_idat:
                found_idat = True
                if length < 2:
                    return fail(ST_CONTAINER)
                cmf, flg = payload[0], payload[1]
                payload = payload[2:]
                pos += 2
                chk = (cmf << 8) | flg
                if (cmf & 15) != 8 or chk == 0 or chk % 31 or (flg >> 5) & 1:
                    return fail(ST_CONTAINER)
            z += payload
            res["n_idat"] += 1
            zlen += len(payload)
            pos += len(payload)
            left -= len(payload)
        elif typ == b"IEND":
            found_iend = True
        elif typ[0] < 0x80 and typ[0] > ord("Z"):      # (signed char) type[0] > 'Z'
            pos += length
            left -= length
        else:
            return fail(ST_CONTAINER)
        if left < 4:
            return fail(ST_CONTAINER)
        if pos + 4 > size:
            return fail(ST_CONTAINER, ub=True)
        stored = int.from_bytes(data[pos:pos + 4], "big")
        pos += 4
        left -= 4
        if stored != crc:
            return fail(ST_PNG_CRC)
    res["zrun"] = zrun
    if not ran:
        return fail(ST_CONTAINER)
    if zrun < 4 + 5:
        return fail(ST_CONTAINER if zrun < 4 else ST_INPUT_TOO_SMALL)
    est = w * h * 4 + h + 1
    g, scan = portlib.inflate(bytes(z[:zrun - 4]), est)
    if not g:
        return fail(INFLATE)
    bpp = {6: 4, 2: 3, 3: 1}[ct]
    res.update(w=w, h=h, bpp=bpp)
    if not scan:
        return fail(None)          # (the filter byte the decoders test is stale memory then)
    if scan[0] > 4:
        return fail(ST_PNG_FILTER)
    if len(scan) < h * (w * bpp + 1):
        return fail(ST_PNG_SHORT)
    res.update(verdict="good", status=ST_OK, rgba=to_rgba(unfilter(scan, w, h, bpp), w, h, bpp, plte))
    return res


def status_ok(want, st):
    """A decoder's status against the model's."""
    if want == INFLATE:
        return 1 <= st <= 11
    if want is None:
        return st != ST_OK
    return st == want


# ------------------------------------------------------------------------------------------------------ catalogue ----
def _img(w, h, bpp, seed, amp=6):
    """A smooth image of w x h pixels and bpp channels; bpp 1 is a palette index ramp that uses every index."""
    if bpp == 1:
        y, x = np.mgrid[0:h, 0:w]
        return ((x * 7 + y * 3 + seed) % 256).astype(np.uint8)[..., None]
    return corpus.gradient_noise_rgba(w, h, seed, amp)[..., :bpp].copy()


def _pal(n, seed):
    return np.random.default_rng(seed).integers(0, 256, 3 * n, dtype=np.uint8).tobytes()


def image_file(w, h, bpp, filt, seed, stb=True, idat=None, before=(), after=(), pal_n=256, amp=6):
    """(file, image) of one image: IHDR, PLTE (bpp 1), `before`, the IDATs (payload sizes `idat`), `after`, IEND."""
    img = _img(w, h, bpp, seed, amp)
    ct = {4: 6, 3: 2, 1: 3}[bpp]
    z = zstream(scanlines(img, filt), stb)
    head = [ihdr(w, h, ct)] + ([chunk(b"PLTE", _pal(pal_n, seed))] if bpp == 1 else []) + list(before)
    return png(head + split(z, idat or []) + list(after) + [chunk(b"IEND")]), img


def _case(cases, fam, name, data, **kw):
    cases.append(dict(name="%s %s" % (fam, name), data=data, **kw))


def catalogue(big=False):
    """Families A-F. Small cases run through the emulator; `big` adds the sizes that need the GPU (large chunks are in both:
    they are what the segment tasks handle)."""
    cases = []
    S = 40 if big else 9          # image side for the walk families
    base, _ = image_file(S, S - 3, 4, 2, 1, amp=1)
    ih = ihdr(S, S - 3, 6)
    rows = scanlines(_img(S, S - 3, 4, 1, amp=1), 2)
    z = zstream(rows)
    tail = split(z, []) + [chunk(b"IEND")]

    # A: signature and walk
    _case(cases, "A", "well-formed", base)
    for b0 in (0x00, 0x41, 0xFF):
        _case(cases, "A", "signature byte 0 = %#x" % b0, bytes([b0]) + base[1:])
    for k in (1, 2, 3):
        _case(cases, "A", "signature byte %d wrong" % k, base[:k] + b"Q" + base[k + 1:])
    for t0 in (0x5B, 0x60, 0x7F, 0x80, 0xC1, ord("Q")):
        _case(cases, "A", "chunk type byte 0 = %#x" % t0, png([ih, chunk(bytes([t0]) + b"xYz", b"abc")] + tail))
    _case(cases, "A", "uppercase unknown chunk", png([ih, chunk(b"ZZZZ", b"")] + tail))
    at = len(SIG) + len(ih)
    left = len(base) - 8 - len(ih) - 8
    _case(cases, "A", "length = left", base[:at] + be32(left) + base[at + 4:])
    _case(cases, "A", "length = left - 1", base[:at] + be32(left - 1) + base[at + 4:])
    _case(cases, "A", "length with bit 31", png([ih, chunk(b"tEXt", b"hi", length=0x80000002)] + tail))
    b13 = struct.pack(">IIBBBBB", S, S - 3, 8, 6, 0, 0, 0)
    _case(cases, "A", "IHDR length 12, CRC after 13 bytes",
          png([be32(12) + b"IHDR" + b13 + be32(zlib.crc32(b"IHDR" + b13[:12]))] + tail))
    _case(cases, "A", "IHDR length 14", png([chunk(b"IHDR", b13 + b"\0")] + tail))
    _case(cases, "A", "IHDR length 17, CRC read inside the payload",
          png([chunk(b"IHDR", b13 + bytes(4), crc="none", solve_at=13)] + tail))
    _case(cases, "A", "IHDR length 17", png([chunk(b"IHDR", b13 + bytes(4))] + tail))
    idats = split(z, [])
    _case(cases, "A", "IEND length 4, solved CRC", png([ih] + idats + [chunk(b"IEND", bytes(4), solve_at=0)]))
    _case(cases, "A", "IEND length 6, solved CRC, no CRC field", png([ih] + idats + [chunk(b"IEND", bytes(6), crc="none", solve_at=0)]))
    _case(cases, "A", "IEND length 4, unsolved", png([ih] + idats + [chunk(b"IEND", b"\1\2\3\4")]))
    _case(cases, "A", "no IEND", png([ih] + idats))
    _case(cases, "A", "no IEND, ancillary after", png([ih] + idats + [chunk(b"tEXt", b"k\0v")]))
    _case(cases, "A", "no IEND, 7 trailing bytes", png([ih] + idats) + b"\0" * 7)
    _case(cases, "A", "trailing bytes after IEND", base + b"garbage after the end")
    _case(cases, "A", "truncated in the IEND CRC", base[:-2])
    _case(cases, "A", "IDAT CRC flipped", png([ih, chunk(b"IDAT", z, crc="flip"), chunk(b"IEND")]))

    # B: IHDR / PLTE
    Wb, Hb = (64, 16) if not big else (256, 64)
    swapped_img = _img(Hb, Wb, 4, 3)
    zs_ = zstream(scanlines(swapped_img, 1))
    _case(cases, "B", "two IHDRs, same", png([ihdr(Wb, Hb, 6), ihdr(Wb, Hb, 6)] + split(zstream(scanlines(_img(Wb, Hb, 4, 3), 1)), []) + [chunk(b"IEND")]))
    _case(cases, "B", "two IHDRs, swapped (%dx%d then %dx%d)" % (Wb, Hb, Hb, Wb),
          png([ihdr(Wb, Hb, 6), ihdr(Hb, Wb, 6)] + split(zs_, []) + [chunk(b"IEND")]), item4=True)
    _case(cases, "B", "two IHDRs, swapped, palette",
          png([ihdr(Wb, Hb, 6), ihdr(Hb, Wb, 3), chunk(b"PLTE", _pal(256, 4))]
              + split(zstream(scanlines(_img(Hb, Wb, 1, 4), 3)), []) + [chunk(b"IEND")]), item4=True)
    pw, ph = (13, 11) if not big else (45, 70)
    pimg = _img(pw, ph, 1, 5)
    pz = zstream(scanlines(pimg, [r % 5 for r in range(ph)]))
    pih = ihdr(pw, ph, 3)
    pend = split(pz, []) + [chunk(b"IEND")]
    _case(cases, "B", "PLTE before IHDR", png([chunk(b"PLTE", _pal(256, 5)), pih] + pend))
    _case(cases, "B", "PLTE length 7", png([pih, chunk(b"PLTE", _pal(256, 5)[:7])] + pend))
    for n in (0, 1, 237, 256, 300):
        _case(cases, "B", "PLTE of %d entries" % n, png([pih, chunk(b"PLTE", _pal(n, 6))] + pend))
    _case(cases, "B", "PLTE twice", png([pih, chunk(b"PLTE", _pal(256, 7)), chunk(b"PLTE", _pal(200, 8))] + pend))
    _case(cases, "B", "PLTE after the IDATs", png([pih] + split(pz, []) + [chunk(b"PLTE", _pal(256, 9)), chunk(b"IEND")]))
    _case(cases, "B", "no PLTE", png([pih] + pend))
    rimg = _img(pw, ph, 3, 10)
    _case(cases, "B", "PLTE on an RGB image", png([ihdr(pw, ph, 2), chunk(b"PLTE", _pal(16, 10))]
                                                   + split(zstream(scanlines(rimg, [r % 5 for r in range(ph)])), []) + [chunk(b"IEND")]))
    _case(cases, "B", "PLTE on an RGBA image", png([ih, chunk(b"PLTE", _pal(16, 11))] + tail))

    # C: IDAT gathering
    for first in (0, 1, 2):
        _case(cases, "C", "first IDAT of %d bytes" % first, png([ih] + split(z, [first]) + [chunk(b"IEND")]))
    _case(cases, "C", "0-length IDATs in the middle", png([ih] + split(z, [7, 0, 0, 5, 0]) + [chunk(b"IEND")]))
    _case(cases, "C", "IDAT of 1 byte each", png([ih] + split(z, [1] * 40) + [chunk(b"IEND")]))
    _case(cases, "C", "zlib header alone", png([ih] + split(z, [2]) + [chunk(b"IEND")]))
    _case(cases, "C", "Adler-32 alone in the last IDAT", png([ih] + split(z, [len(z) - 4]) + [chunk(b"IEND")]))
    _case(cases, "C", "Adler-32 split over two IDATs", png([ih] + split(z, [len(z) - 2]) + [chunk(b"IEND")]))
    # Every non-IDAT chunk after an IDAT moves the inflate point (the reference inflates there, again and again: Q14),
    # so the last one -- IEND at the latest -- sees every IDAT byte before it
    half = len(z) // 2
    _case(cases, "C", "IDAT-tEXt-IDAT, stream cut at the tEXt",
          png([ih] + split(z[:half], []) + [chunk(b"tEXt", b"k\0v")] + split(z[half:], []) + [chunk(b"IEND")]))
    _case(cases, "C", "IDAT-tEXt-IDAT, whole stream before the tEXt",
          png([ih] + split(z, []) + [chunk(b"tEXt", b"k\0v")] + split(bytes(range(37)), []) + [chunk(b"IEND")]))
    _case(cases, "C", "IDAT-IEND-IDAT", png([ih] + split(z[:half], []) + [chunk(b"IEND")] + split(z[half:], [])))
    for zr in (3, 4, 8, 9):
        # zr bytes after the zlib header when the walk reaches its inflate point
        _case(cases, "C", "zlen_at_run %d" % zr, png([ih] + split(z[:2 + zr], []) + [chunk(b"tEXt", b""), chunk(b"IEND")]))

    # C / D: large chunks -- segment tasks for the CRC and the copies (in both families: only they reach that code)
    cw, chh = 512, 200        # a 300 KB stream (Sub rows of a noisy image): IDATs of more than 2 x 64 KiB
    cimg = _img(cw, chh, 4, 12)
    cz = zstream(scanlines(cimg, 1))
    assert 131077 + 65537 + 65531 + 1000 < len(cz) < cw * chh * 4
    cih = ihdr(cw, chh, 6)
    off = len(SIG) + len(cih)
    for sizes in ((65531, 65537), (65537 + 2, 5000), (131077 + 2, 100), (65531, 131077, 65537)):
        # first IDAT payload (after the zlib header) 16-byte aligned in the file: copies take the 16-byte branch there
        pad = pad_chunk(off, want=2)
        _case(cases, "C", "IDATs of %s bytes" % "/".join(map(str, sizes)),
              png([cih, pad] + split(cz, list(sizes)) + [chunk(b"IEND")]), large=True)
    _case(cases, "C", "IDATs of 65537/65537, unaligned", png([cih] + split(cz, [65537, 65537]) + [chunk(b"IEND")]), large=True)

    dimg = _img(S, S - 3, 4, 13)
    dz = zstream(scanlines(dimg, 2))
    dih = ihdr(S, S - 3, 6)
    rng = np.random.default_rng(14)
    for n in (65535, 65536, 65537, 8192 * 9, 8192 * 9 + 1, 8192 * 9 - 1, 3 * 65536 + 5):
        payload = rng.integers(0, 256, n - 4, dtype=np.uint8).tobytes()
        _case(cases, "D", "ancillary chunk of 4+length = %d" % n,
              png([dih, chunk(b"zBig", payload)] + split(dz, []) + [chunk(b"IEND")]), large=n > SCAN_SEG)
    big_payload = rng.integers(0, 256, 3 * 65536 + 5 - 4, dtype=np.uint8).tobytes()
    three = lambda p1, crc="ok": png([cih, chunk(b"aBig", p1, crc=crc)] + split(cz, []) + [chunk(b"zAft", big_payload[:70000]), chunk(b"IEND")])
    _case(cases, "D", "large chunks before, in and after the IDAT", three(big_payload), large=True)
    for seg in range(4):
        for end in (0, 1):
            b = (seg * SCAN_SEG - 4 if seg else 0) if not end else min((seg + 1) * SCAN_SEG, len(big_payload) + 4) - 4 - 1
            p = bytearray(big_payload)
            p[b] ^= 0x40
            _case(cases, "D", "large ancillary chunk, byte %d of its payload flipped" % b, three(bytes(p), crc=zlib.crc32(b"aBig" + big_payload)),
                  large=True)
    _case(cases, "D", "large IDAT, stored CRC flipped", png([cih, chunk(b"IDAT", cz, crc="flip"), chunk(b"IEND")]), large=True)
    _case(cases, "D", "large IDAT, payload byte flipped under the right CRC",
          png([cih, chunk(b"IDAT", cz[:-9] + bytes([cz[-9] ^ 1]) + cz[-8:], crc=zlib.crc32(b"IDAT" + cz))] + [chunk(b"IEND")]), large=True)

    # E: the generic un-filter (palette and RGB)
    sizes = [(1, 1), (2, 31), (31, 32), (32, 33), (33, 1), (63, 65), (64, 2), (65, 31), (97, 32)] if not big else \
        [(1, 4300), (33, 4200), (97, 65), (300, 40), (2000, 33)]
    mixes = [(0,), (1,), (2,), (3,), (4,), (0, 1, 2, 3, 4), (1, 3), (2, 4)]
    for k, (w, h) in enumerate(sizes):
        for bpp in (1, 3):
            for j, fs in enumerate(mixes if not big or w * h < 200000 else mixes[4:6]):
                if not big and (k + j + bpp) % 3:
                    continue
                r = np.random.default_rng(100 + 10 * k + j)
                filt = r.choice(fs, size=h)
                f, _ = image_file(w, h, bpp, filt, 20 + k + j, stb=(k + j) % 2 == 0, pal_n=(237, 256, 300)[j % 3])
                _case(cases, "E", "bpp %d %dx%d filters %s" % (bpp, w, h, "".join(map(str, fs))), f)
    ew, eh = (13, 40) if not big else (77, 300)
    for bpp in (1, 3):
        filt = [1, 2, 3, 4] * (eh // 4)
        filt[5], filt[eh - 1] = 7, 255
        f, _ = image_file(ew, eh, bpp, filt, 30 + bpp)
        _case(cases, "E", "bpp %d filter > 4 on later rows" % bpp, f)
        f, _ = image_file(ew, eh, bpp, [5] + filt[1:], 31 + bpp)
        _case(cases, "E", "bpp %d filter 5 on row 0" % bpp, f)
        raw = scanlines(_img(ew, eh, bpp, 32 + bpp), 2)
        ct = {1: 3, 3: 2}[bpp]
        hd = [ihdr(ew, eh, ct)] + ([chunk(b"PLTE", _pal(256, 3))] if bpp == 1 else [])
        _case(cases, "E", "bpp %d scanlines exactly need" % bpp, png(hd + split(zstream(raw), []) + [chunk(b"IEND")]))
        _case(cases, "E", "bpp %d scanlines need - 1" % bpp, png(hd + split(zstream(raw[:-1]), []) + [chunk(b"IEND")]))
    return cases


def stb_shaped(data):
    """dbg_api.cu png_all_stb_shaped for one file: the files of a batch that takes the hinted packed route."""
    if len(data) < 8 + 25 + 12 + 3:
        return False
    w, h = int.from_bytes(data[16:20], "big"), int.from_bytes(data[20:24], "big")
    if w == 0 or h == 0 or w * h * 4 + h + 1 >= 1 << 32:
        return False
    pos = 8
    for _ in range(64):
        if pos + 12 > len(data):
            break
        length = int.from_bytes(data[pos:pos + 4], "big")
        if data[pos + 4:pos + 8] == b"IDAT":
            return length >= 3 and pos + 11 <= len(data) and (data[pos + 10] & 7) == 3
        pos += 12 + length
    return False
