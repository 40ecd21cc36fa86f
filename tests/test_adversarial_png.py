"""CPU suite: hand-built PNG files (tests/png_writer.py) through the emulated device source of the PNG container path --
png_scan_warp with and without the segment queues of large chunks, the segment tasks and the CRC verdict of
png_tasks_kernel / png_verify_kernel, inflate and the un-filter -- in both lane orders, against the writer's model of the
reference.

Defined behaviour: the modelled status and RGBA. Where the reference reads outside the file (Q11, verdict "ub") every
path must fail, and the plain-C restatement must fail too."""
import ctypes as C
import os
import subprocess
import zlib

import pytest

import png_writer as W
from oracle import portlib

HERE = os.path.dirname(os.path.abspath(__file__))
EMU_DIR = os.path.join(HERE, "simt_emu")
CSRC = os.path.join(os.path.dirname(HERE), "debigulator_b200", "csrc")


@pytest.fixture(scope="module")
def emu():
    so = os.path.join(EMU_DIR, "libsimt_emu.so")
    srcs = [os.path.join(EMU_DIR, "emu.cpp")] + [os.path.join(CSRC, f) for f in ("simt.h", "inflate_core.h", "png_core.h", "bsplit_core.h", "fx_core.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", srcs[0], "-o", so])
    L = C.CDLL(so)
    L.emu_png_decode_queued.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_uint32, C.c_uint32,
                                        C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    L.emu_png_decode_queued.restype = C.c_uint32
    L.emu_png_decode.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_int]
    L.emu_png_decode.restype = C.c_uint32
    return L


@pytest.fixture(scope="module")
def small():
    return W.catalogue(big=False)


def run(L, data, rgba_size, queued, mis, rev, task_cap=0):
    """(status, rgba, tasks enqueued, large chunks) of the emulated device source."""
    ib = C.create_string_buffer(data, len(data))
    ob = C.create_string_buffer(rgba_size + 64)
    nt, nb = C.c_uint32(0), C.c_uint32(0)
    if queued:
        st = L.emu_png_decode_queued(ib, len(data), ob, rgba_size, mis, rev, task_cap, 0, C.byref(nt), C.byref(nb))
    else:
        st = L.emu_png_decode(ib, len(data), ob, rgba_size, rev)
    return st, ob.raw[:rgba_size], nt.value, nb.value


def rgba_size(data):
    return int.from_bytes(data[16:20], "big") * int.from_bytes(data[20:24], "big") * 4 if len(data) >= 24 else 0


def expect(case, ref):
    """The model's verdict, confirmed by the plain-C restatement (spec RGB expansion) everywhere and by the reference
    where its behaviour is defined."""
    m = W.model(case["data"])
    assert m["verdict"] in ("good", "fail", "ub"), case["name"]
    g, _, _, o = portlib.decode_png(case["data"], rgb_as_reference=False)
    assert (g, o) == ((1, m["rgba"]) if m["verdict"] == "good" else (0, b"")), case["name"]
    if m["verdict"] != "ub":
        g, _, _, o = ref.decode_png(case["data"])
        assert g == (m["verdict"] == "good"), case["name"]
        if g and m["bpp"] != 3:  # (RGB: the reference's expansion is defect D3)
            assert o == m["rgba"], case["name"]
    return m


def check(name, m, st, out):
    assert st < 0x1000, (name, hex(st))                 # the lanes agree
    if m["verdict"] == "good":
        assert st == 0 and out == m["rgba"], (name, st)
    elif m["verdict"] == "ub":
        assert st != 0, name
    else:
        assert W.status_ok(m["status"], st), (name, m["status"], st)


# ------------------------------------------------------------------------------------------- writer self-checks ----
def test_writer_and_model(small, ref):
    """Every catalogued file gets the modelled verdict and RGBA from the plain-C restatement and from the reference; the
    writer's CRCs are zlib's; the solved CRCs are what the walk reads; the families reach what they are named for."""
    names = set()
    for case in small:
        expect(case, ref)
        names.add(case["name"])
    assert len(names) == len(small)
    assert W.chunk(b"tEXt", b"abc")[-4:] == zlib.crc32(b"tEXtabc").to_bytes(4, "big")
    p = W.chunk(b"IEND", bytes(4), solve_at=0)[8:12]
    assert p == zlib.crc32(b"IEND" + p).to_bytes(4, "big")
    by = {c["name"]: W.model(c["data"]) for c in small}
    assert by["A IEND length 4, solved CRC"]["verdict"] == "good"
    assert by["A IEND length 4, unsolved"]["status"] == W.ST_PNG_CRC
    assert by["A IHDR length 17, CRC read inside the payload"]["verdict"] == "good"
    assert by["A chunk type byte 0 = 0x5b"]["verdict"] == by["A chunk type byte 0 = 0x60"]["verdict"] == "good"
    assert by["A chunk type byte 0 = 0x80"]["status"] == by["A chunk type byte 0 = 0xc1"]["status"] == W.ST_CONTAINER
    assert [by["C zlen_at_run %d" % z]["zrun"] for z in (3, 4, 8, 9)] == [3, 4, 8, 9]
    assert [by["C zlen_at_run %d" % z]["status"] for z in (3, 4, 8)] == [W.ST_CONTAINER, W.ST_INPUT_TOO_SMALL, W.ST_INPUT_TOO_SMALL]
    assert by["C zlen_at_run 9"]["status"] not in (W.ST_CONTAINER, W.ST_INPUT_TOO_SMALL)
    assert by["C IDAT-tEXt-IDAT, stream cut at the tEXt"]["verdict"] == "good"
    assert by["C IDAT-IEND-IDAT"]["verdict"] == "fail"
    assert by["E bpp 1 filter 5 on row 0"]["status"] == W.ST_PNG_FILTER
    assert by["E bpp 3 scanlines need - 1"]["status"] == W.ST_PNG_SHORT
    # no IEND: Q11 leaves `left` at least 15 bytes (IHDR, zlib header) above what the file holds, so the walk always
    # runs past the end of such a file -- undefined in the reference
    assert all(m["verdict"] == "ub" for n, m in by.items() if "no IEND" in n)


# ------------------------------------------------------------------------------------------ the device source ----
def test_families_through_the_emulated_device(emu, small, ref):
    """Every small case through the emulated device source: the walk with the large chunks deferred to segment tasks
    (run in queue order and in reverse) and without, in both lane orders, the file at several alignments."""
    queued_large = 0
    for k, case in enumerate(small):
        m = expect(case, ref)
        n = rgba_size(case["data"])
        if n >= 1 << 26:          # no IHDR at offset 16: the files of this kind fail on any RGBA size
            assert m["verdict"] != "good"
            n, m = 0, W.model(case["data"], 0)
        configs = [(0, 0, k & 1), (1, (5 * k) % 16, (k + 1) & 1)]
        if case.get("large"):
            configs += [(1, 0, k & 1), (1, 0, (k + 1) & 1)]
        for queued, mis, rev in configs:
            st, out, nt, nb = run(emu, case["data"], n, queued, mis, rev)
            check((case["name"], queued, mis, rev), m, st, out)
            if queued and case.get("large"):
                assert nt >= 2 and nb >= 1, (case["name"], nt, nb)
                queued_large += 1
    assert queued_large >= 40


def test_large_chunk_crc_only_the_segment_tasks_see(emu, small):
    """A flipped byte at the first and last byte of every 64 KiB segment of a large ancillary chunk, and a flipped
    stored CRC of a large IDAT: nothing but the recombined CRC can tell, and the verdict is exactly 13 on both routes."""
    cases = [c for c in small if c["name"].startswith(("D large ancillary chunk, byte", "D large IDAT"))]
    assert len(cases) == 10
    for k, c in enumerate(cases):
        for queued in (0, 1):
            st, _, nt, nb = run(emu, c["data"], rgba_size(c["data"]), queued, 0, k & 1)
            assert st == W.ST_PNG_CRC, (c["name"], queued, st)
            assert not queued or nb >= 1, c["name"]


def test_full_task_queue_falls_back_to_the_walk(emu):
    """A file of nothing but IDATs just over 64 KiB: the queue of png_task_cap takes every segment; with one slot too
    few, the walk does the chunk's work itself and marks the slots it leaves empty. Same pixels every time."""
    img = W._img(512, 200, 4, 12)
    data = W.png([W.ihdr(512, 200, 6)] + W.split(W.zstream(W.scanlines(img, 1)), [65537] * 4) + [W.chunk(b"IEND")])
    n = 512 * 200 * 4
    st, out, nt, nb = run(emu, data, n, 1, 0, 0)
    cap = 4 * (len(data) // W.SCAN_SEG) + 64
    assert st == 0 and out == img.tobytes() and nt <= cap and nb == 4, (st, nt, nb)
    for task_cap in (nt, nt - 1, nt - 3, 1):
        st, out, _, _ = run(emu, data, n, 1, 0, task_cap & 1, task_cap=task_cap)
        assert st == 0 and out == img.tobytes(), (task_cap, st)
