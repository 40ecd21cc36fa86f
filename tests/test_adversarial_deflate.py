"""CPU suite: hand-built DEFLATE streams (tests/deflate_writer.py) through every inflate path of the device source, run by
the SIMT emulator -- the warp-per-stream decoder with and without its lane-parallel rounds, the lane-serial fixed-block
path and the block-split path with and without pieces -- at the reference's quirks (Q2, Q3, Q5, BTYPE 3, repeat codes
across the litlen/dist boundary), the ends of both alphabets, incomplete and over-subscribed codes, expansion edges,
domain boundaries and the end of the stream.

Defined behaviour: status and bytes equal the reference's and the writer's intended output. Undefined behaviour in the
reference (over-subscribed codes, litlen 286/287, a repeat with no predecessor, output overflow): every path fails, the
plain-C restatement fails too, and the reference itself is not called."""
import ctypes as C
import os
import subprocess
import zlib

import numpy as np
import pytest

import deflate_writer as W
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
    L.emu_inflate.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.c_int, C.c_int]
    L.emu_inflate.restype = C.c_uint32
    L.emu_fx_inflate.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.c_int, C.c_int, C.c_uint32,
                                 C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    L.emu_fx_inflate.restype = C.c_uint32
    L.emu_bsplit_inflate_pieces.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.c_int, C.c_int,
                                            C.c_uint32, C.POINTER(C.c_uint32), C.c_uint32, C.c_int, C.c_uint32]
    L.emu_bsplit_inflate_pieces.restype = C.c_uint32
    L.emu_lane_block_stats.argtypes = [C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.c_int]
    return L


@pytest.fixture(scope="module")
def small():
    return W.catalogue(big=False)


def lane_rounds(L, reset=False):
    tried, done = C.c_uint32(0), C.c_uint32(0)
    L.emu_lane_block_stats(C.byref(tried), C.byref(done), int(reset))
    return done.value


def run_walk(L, data, cap, mis, rev):
    ib = C.create_string_buffer(data, max(len(data), 1))
    ob = C.create_string_buffer(cap + 64)
    n = C.c_uint64(0)
    st = L.emu_inflate(ib, len(data), ob, cap, C.byref(n), mis, rev)
    return st, ob.raw[: n.value]


def run_fx(L, data, cap, mis, rev, chunk, group):
    ib = C.create_string_buffer(data, len(data))
    ob = C.create_string_buffer(cap + 64)
    n, ms, nc = C.c_uint64(0), C.c_uint32(0), C.c_uint32(0)
    st = L.emu_fx_inflate(ib, len(data), ob, cap, C.byref(n), mis, rev, chunk, group, C.byref(ms), C.byref(nc))
    return st, ob.raw[: n.value], nc.value


def run_bsplit(L, data, cap, mis, rev, region, pieces):
    ib = C.create_string_buffer(data, len(data))
    ob = C.create_string_buffer(cap + 64)
    n, nch = C.c_uint64(0), C.c_uint32(0)
    st = L.emu_bsplit_inflate_pieces(ib, len(data), ob, cap, C.byref(n), mis, rev, region, C.byref(nch), 4, 1, pieces)
    return st, ob.raw[: n.value], nch.value


def reference(case, ref):
    """(verdict, bytes) the checks compare with: the writer's model, confirmed by the reference where it is defined and
    by the plain-C restatement everywhere."""
    verdict, want = case["want"]
    assert verdict in ("good", "fail", "ub"), case["name"]
    g, o = portlib.inflate(case["data"], case["cap"])
    assert (g, o) == ((1, want) if verdict == "good" else (0, b"")), case["name"]
    if verdict != "ub":
        g, o = ref.inflate(case["data"], case["cap"])
        assert (g, o) == ((1, want) if verdict == "good" else (0, b"")), case["name"]
    return verdict, want


def check(name, verdict, want, st, out):
    assert st < 0x1000, (name, hex(st))
    if verdict == "good":
        assert st == 0 and out == want, (name, st, len(out), len(want))
    else:
        assert st != 0, (name, verdict)


# ------------------------------------------------------------------------------------------- writer self-checks ----
def test_writer_against_zlib_and_reference(small, ref):
    """Random spec-valid streams (any mix of stored / fixed / dynamic blocks, explicit 258 encodings, code lengths from
    frequencies) decode with zlib to what the writer intended; every catalogued stream gets the intended verdict and
    bytes from the reference (defined behaviour) and from the plain-C restatement (all)."""
    rng = np.random.default_rng(5)
    for t in range(40):
        blocks, pos = [], 0
        for b in range(int(rng.integers(1, 6))):
            kind = int(rng.integers(0, 3))
            if kind == 0:
                d = rng.integers(0, 256, int(rng.integers(0, 3000)), dtype=np.uint8).tobytes()
                blocks.append(W.stored(d))
                pos += len(d)
                continue
            tok = W.filler(int(rng.integers(10, 20000)), rng, start_pos=pos, max_dist=int(rng.choice([4, 300, 32768])))
            if pos >= 1:
                tok = W.cat(tok, W.match(258, 1, lsym=284, lx=31), W.match(258, 1))
            blocks.append(W.fixed(tok) if kind == 1 else W.dynamic(tok))
            pos += int(W.token_out_len(tok).sum())
        blocks[-1].final = True
        s = W.write(blocks)
        assert s.spec_valid, t
        verdict, want = s.expect()
        assert verdict == "good" and zlib.decompress(s.data, -15) == want, t
        assert len(s.offsets) == sum(1 for bk in blocks if bk.btype in (1, 2))
    names = set()
    for case in small:
        reference(case, ref)
        names.add(case["name"])
        s = case["stream"]
        if s.spec_valid and case["want"][0] == "good" and case["data"] == s.data:
            assert zlib.decompress(s.data, -15) == case["want"][1], case["name"]
    assert len(names) == len(small)


def test_writer_packs_a_mebibyte_stream():
    """A stream of more than 1 MiB from 1.5 M tokens: the vectorised packing decodes with zlib to the intended output."""
    rng = np.random.default_rng(8)
    s = W.write([W.dynamic(W.filler(6_000_000, rng), final=True)])
    assert len(s.data) > 1 << 20
    assert zlib.decompress(s.data, -15) == s.output


# --------------------------------------------------------------------------------------------- through every path --
def test_families_warp_per_stream(emu, small, ref):
    """Every small case through inflate_warp, lane-parallel rounds on and off (bit 4 of the misalignment argument),
    both lane orders, several input misalignments."""
    lane_rounds(emu, reset=True)
    for k, case in enumerate(small):
        verdict, want = reference(case, ref)
        for rounds_off, rev in ((0, k & 1), (16, (k + 1) & 1), (0, (k + 1) & 1)):
            if rounds_off and case["path"] != "walk" and k % 2:
                continue
            if rounds_off == 0 and rev != k & 1 and case["name"].startswith(("I Q2", "F odd")):
                continue        # (one lane order with rounds is enough for these many variants of one stream)
            st, out = run_walk(emu, case["data"], case["cap"], ((5 * k + 3 * rev) % 16) | rounds_off, rev)
            check((case["name"], rounds_off, rev), verdict, want, st, out)
    assert lane_rounds(emu) >= 100


@pytest.mark.parametrize("fam", "DGHI")
def test_families_lane_serial_fixed(emu, small, ref, fam):
    """The single-fixed-block cases through the lane-serial path: chunks of 2 and 4 KiB, groups of 1-4 chunks."""
    ran = 0
    one_block = [c for c in small if c["name"][0] == fam and (c["data"][0] & 7) == 3 and len(c["data"]) >= 4096]
    for k, case in enumerate(one_block):
        verdict, want = reference(case, ref)
        for chunk, group in ((2048, 1), (2048, 3), (4096, 2), (4096, 4))[: 2 if "Q2" in case["name"] else 4]:
            st, out, nc = run_fx(emu, case["data"], case["cap"], (k + chunk // 1024) % 16, (k + group) & 1, chunk, group)
            assert st != 0x2000, case["name"]
            assert nc >= 2 or len(case["data"]) < 2 * chunk or (st and verdict != "good"), (case["name"], nc)
            check((case["name"], chunk, group), verdict, want, st, out)
            ran += 1
    assert ran >= 4


@pytest.mark.parametrize("fam", "FHI")
def test_families_block_split(emu, small, ref, fam):
    """The many-block cases through the block-split path, whole chunks and pieces, regions of 2-4 KiB. The streams with
    one odd block 60 % of the way in put that block's table or symbol into a chunk well after the first."""
    ran = expanded = 0
    for k, case in enumerate(c for c in small if c["path"] == "bsplit" and c["name"][0] == fam):
        verdict, want = reference(case, ref)
        configs = ((2048, 1), (4096, 1), (4096, 5), (2048, 16))
        for region, pieces in configs[1::2] if "odd block" in case["name"] or "after the final" in case["name"] else configs:
            st, out, nch = run_bsplit(emu, case["data"], case["cap"], (3 * k + region // 1024) % 16, (k + pieces) & 1, region, pieces)
            assert st != 0x4000, (case["name"], region)           # the chain of hinted chunks closed
            check((case["name"], region, pieces), verdict, want, st, out)
            if verdict == "good":
                assert (nch & 0xFFFF) >= 2, (case["name"], nch)   # hinted chunks really carried the stream
            expanded += nch >> 16
            ran += 1
    assert ran >= 4 and expanded >= 4                             # and some were expanded from tokens


def test_q2_drops_a_symbol_that_starts_in_the_last_byte(small):
    """The writer's rule-Q2 model: of the 16 placements of the last symbol, the ones that start inside the last byte
    are not decoded."""
    for last in ("literal", "match", "48-bit"):
        dropped = [len(c["want"][1]) < c["stream"].max_out for c in small if c["name"].startswith("I Q2 %s +" % last)]
        assert len(dropped) == 16 and 0 < sum(dropped) < 16, (last, dropped)
