"""The checker tests, smoke() and bench.py's CPU legs use: the unmodified
reference (oracle/_ref/libref.so, kind "reference") when it is available, else
the plain-C restatement (oracle/liboracle.so, kind "port"), which
tests/test_oracle.py pins to the reference's own outputs in tests/golden.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).
"""
from . import reflib

try:
    from . import portlib
except Exception:  # pragma: no cover
    portlib = None


def kind() -> str:
    return "reference" if reflib.available() else "port"


def _impl():
    if reflib.available():
        return reflib
    if portlib is None or not portlib.available():
        raise RuntimeError("no CPU checker available: build oracle/ (make -C oracle)")
    return portlib


def inflate(data: bytes, cap: int):
    return _impl().inflate(data, cap)


def decode_gz(data: bytes, cap: int):
    return _impl().decode_gz(data, cap)


def decode_png(data: bytes):
    return _impl().decode_png(data)


def decode_bmp(data: bytes, out_size: int = None):
    return _impl().decode_bmp(data, out_size)


def encode_bmp(rgba: bytes, w: int, h: int):
    return _impl().encode_bmp(rgba, w, h)


def stb_png(pixels: bytes, w: int, h: int, comp: int = 4, filt: int = -1) -> bytes:
    """A PNG of the shape stb_write.h writes (one IDAT, zlib header 78 5E, one final fixed-Huffman block): the
    reference's own stb_write.h when it is available, else the corpus's encoder (debigulator_b200/tools/fixed_deflate.c)."""
    if reflib.available():
        return reflib.stb_png(pixels, w, h, comp, filt)
    import numpy as np
    from debigulator_b200 import corpus
    img = np.frombuffer(bytes(pixels), np.uint8).reshape(h, w, comp)
    return corpus.write_png(img, filt=filt, single_block=True)


def stb_zlib(data: bytes, quality: int = 8) -> bytes:
    """A zlib stream of the shape stb_write.h writes (78 5E, one final fixed-Huffman block, Adler-32); see stb_png."""
    if reflib.available():
        return reflib.stb_zlib(data, quality)
    import struct
    import zlib
    from debigulator_b200 import corpus
    return b"\x78\x5e" + corpus.fixed_block_deflate(data) + struct.pack(">I", zlib.adler32(bytes(data)) & 0xFFFFFFFF)


class TimedRunner:
    """bench.py's CPU legs: decodes a fixed list of items over and over with everything allocated up front, so that
    what is timed is the checker's C entry point and nothing else (no Python allocation, no copies of the results).

        r = TimedRunner("gz" | "png", blobs, caps);  seconds, out_bytes = r.run()
    """

    def __init__(self, what, blobs, caps):
        import ctypes as C
        self.C = C
        self.what = what
        self.impl = _impl()
        self.L = self.impl.lib()
        self.ref = self.impl is reflib
        self.items = [(C.create_string_buffer(bytes(b) + bytes(64), len(b) + 64), len(b), int(c)) for b, c in zip(blobs, caps)]
        self.out = C.create_string_buffer(max(int(c) for c in caps) + 4096)
        self.n = C.c_uint64(0)
        self.g32 = C.c_uint32(0)
        self.g8 = C.c_uint8(0)

    def run(self):
        import time
        C, L = self.C, self.L
        total = 0
        t0 = time.perf_counter()
        for ib, size, cap in self.items:
            if self.what == "gz":
                if self.ref:
                    L.ref_decode_gz(ib, size, self.out, cap, C.byref(self.n), C.byref(self.g32))
                else:
                    L.oracle_decode_gz(ib, size, self.out, cap, C.byref(self.n), C.byref(self.g32))
                ok, produced = self.g32.value, self.n.value
            else:
                if self.ref:
                    L.ref_decode_png(ib, size, self.out, cap, C.byref(self.g8))
                else:
                    L.oracle_decode_png(ib, size, self.out, cap, 1, C.byref(self.g8))
                ok, produced = self.g8.value, cap
            if not ok:
                raise RuntimeError("CPU checker failed on a benchmark item")
            total += produced
        return time.perf_counter() - t0, total
