"""GPU suite: the large hand-built DEFLATE streams of tests/deflate_writer.py through every inflate path of the product,
one context per path (created under the DBG_* switches that force it), against the reference and the writer's intended
output. Each context asserts from its own statistics that the path it stands for really ran."""
import gzip
import os
import struct
import zlib

import numpy as np
import pytest

import deflate_writer as W
from oracle import portlib

pytestmark = pytest.mark.gpu

CONTEXTS = {
    "default": {},
    # (the lane-serial and block-split paths off, so that every stream meets the warp-per-stream kernel's variant)
    "walk": {"DBG_ROUNDS": "0", "DBG_FX": "0", "DBG_BSPLIT": "0"},
    "short rounds": {"DBG_ROUND_BITS": "8192", "DBG_FX": "0", "DBG_BSPLIT": "0"},
    "fx small chunks": {"DBG_FX_CHUNK": "2048", "DBG_FX_GROUP": "4096"},
    "bsplit": {"DBG_BSPLIT": "1", "DBG_BSPLIT_ALL": "1", "DBG_BSPLIT_REGION": "8192", "DBG_BSPLIT_REGION_MIN": "4096",
               "DBG_BSPLIT_MIN_BYTES": "65536", "DBG_BS_PIECES": "0"},
    "bsplit pieces": {"DBG_BSPLIT": "1", "DBG_BSPLIT_ALL": "1", "DBG_BSPLIT_REGION": "8192", "DBG_BSPLIT_REGION_MIN": "4096",
                      "DBG_BSPLIT_MIN_BYTES": "65536", "DBG_BS_PIECES": "1"},
}


def make_ctx(env):
    import debigulator_b200 as dbg
    old = {k: os.environ.get(k) for k in env}
    try:
        os.environ.update(env)
        return dbg.Context(0)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.fixture(scope="module")
def large(ref):
    cases = W.catalogue(big=True)
    for c in cases:
        verdict, want = c["want"]
        assert verdict in ("good", "fail", "ub"), c["name"]
        assert portlib.inflate(c["data"], c["cap"]) == ((1, want) if verdict == "good" else (0, b"")), c["name"]
        if verdict != "ub":
            assert ref.inflate(c["data"], c["cap"]) == ((1, want) if verdict == "good" else (0, b"")), c["name"]
    return cases


def _check(cases, got, what):
    for c, (g, o) in zip(cases, got):
        verdict, want = c["want"]
        if verdict == "good":
            assert g == 1 and o == want, (what, c["name"], g, len(o), len(want))
        else:
            assert g == 0, (what, c["name"], verdict)


def _one_fixed_block(c):
    return (c["data"][0] & 7) == 3 and len(c["data"]) >= 8192 and c["cap"] >= len(c["data"])


def _counters(ctx):
    """(lane-serial streams, handed back), (block-split streams, handed back), chunks expanded from tokens, rounds of the
    warp-per-stream kernel."""
    fx = ctx.fx_stats()
    lane = ctx.lane_stats()
    return np.array([fx[0], fx[1], *ctx.bsplit_stats(), lane[3], lane[5]], np.int64)


@pytest.mark.parametrize("which", list(CONTEXTS))
def test_large_families_on_every_path(large, which):
    """Every large case on its own (so that the path statistics are the case's own): verdict and bytes, and for every
    case that targets the context's path and decodes, that the path took it and did not hand it back."""
    ctx = make_ctx(CONTEXTS[which])
    try:
        expanded = 0
        for c in large:
            before = _counters(ctx)
            _check([c], ctx.inflate_batch([c["data"]], [c["cap"]]), which)
            fx, fx_back, bs, bs_back, exp, rounds = _counters(ctx) - before
            expanded += exp
            good = c["want"][0] == "good"
            if which == "walk":
                assert fx == bs == rounds == 0, (c["name"], fx, bs, rounds)
            elif which == "short rounds":
                assert fx == bs == 0, c["name"]
                if good and c["path"] == "walk" and len(c["data"]) >= 16384:
                    assert rounds >= 1, c["name"]                   # 1 KiB rounds: every such stream has some
            elif which in ("default", "fx small chunks"):
                if good and _one_fixed_block(c):
                    assert (fx, fx_back) == (1, 0), (c["name"], fx, fx_back)
            elif good and c["path"] == "bsplit":
                assert (bs, bs_back) == (1, 0), (c["name"], bs, bs_back)
        if which.startswith("bsplit"):
            assert expanded > 0                                     # chunks (or pieces) expanded from tokens
    finally:
        ctx.close()


def test_device_entry_point_at_every_output_alignment(ctx, large):
    """Families G and I through inflate_device, each stream at every output offset mod 16."""
    import torch
    dev = torch.device("cuda", 0)
    items = [(c, a) for c in large if c["name"][0] in "GI" for a in range(16)]
    offs, total = [], 16
    for c, _ in items:
        offs.append(total)
        total += len(c["data"]) + 16
    arena = np.zeros((total + 64 + 15) // 16 * 16, np.uint8)
    for o, (c, _) in zip(offs, items):
        arena[o:o + len(c["data"])] = np.frombuffer(c["data"], np.uint8)
    out_off, pos = [], 0
    for c, a in items:
        pos = (pos + 15) // 16 * 16 + a
        out_off.append(pos)
        pos += c["cap"] + 1
    i64 = lambda a: torch.from_numpy(np.asarray(a, np.uint64).view(np.int64)).to(dev)
    d_in = torch.from_numpy(arena).to(dev)
    d_out = torch.zeros(pos + 64, dtype=torch.uint8, device=dev)
    d_size = torch.zeros(len(items), dtype=torch.int64, device=dev)
    d_st = torch.full((len(items),), -1, dtype=torch.int32, device=dev)
    ctx.inflate_device(d_in, i64(offs), i64([len(c["data"]) for c, _ in items]), d_out, i64(out_off),
                       i64([c["cap"] for c, _ in items]), d_size, d_st)
    torch.cuda.synchronize()
    out, st, sz = d_out.cpu().numpy(), d_st.cpu().numpy(), d_size.cpu().numpy()
    for i, (c, a) in enumerate(items):
        verdict, want = c["want"]
        if verdict == "good":
            assert st[i] == 0 and int(sz[i]) == len(want), (c["name"], a, st[i])
            assert out[out_off[i]:out_off[i] + len(want)].tobytes() == want, (c["name"], a)
        else:
            assert 1 <= st[i] <= 12, (c["name"], a, st[i])              # one of the decoder's own error statuses


def test_gzip_framed_stream_ends(ctx, large):
    """Large cases framed as gzip members: rule Q2 sees the deflate data's size (the member less its 8-byte trailer)
    while the trailer behind it is readable."""
    cases = [c for c in large if c["name"].startswith(("I Q2 48-bit", "I capacity exact (", "F tiny", "G dist"))]
    members = []
    for c in cases:
        hdr = b"\x1f\x8b\x08\x00" + bytes(4) + b"\x00\xff"
        want = c["want"][1]
        members.append(hdr + c["data"] + struct.pack("<II", zlib.crc32(want), len(want) & 0xFFFFFFFF))
    got = ctx.decode_gz_batch(members, [c["cap"] for c in cases])
    for c, m, (g, o) in zip(cases, members, got):
        rg, ro = portlib.decode_gz(m, c["cap"])
        verdict, want = c["want"]
        assert (rg, ro) == ((1, want) if verdict == "good" else (0, b"")), c["name"]
        assert (g, o) == (rg, ro), c["name"]
        if verdict == "good" and c["data"] == c["stream"].data and c["stream"].spec_valid:
            assert gzip.decompress(m) == want, c["name"]
