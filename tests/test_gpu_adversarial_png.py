"""GPU suite: the hand-built PNG files of tests/png_writer.py, large sizes, through every PNG route of the product -- the
read-back batch, the packed batch with and without the stb-shaped hints, and the device entry point at every input
alignment -- against the writer's model of the reference."""
import numpy as np
import pytest

import png_writer as W
from oracle import portlib

pytestmark = pytest.mark.gpu


def rgba_size(data):
    n = int.from_bytes(data[16:20], "big") * int.from_bytes(data[20:24], "big") * 4 if len(data) >= 24 else 0
    return n if n < 1 << 26 else 0      # (no IHDR at offset 16: such files fail on any size)


def scheduling_batch():
    """Family F: many one-band images and one very tall palette image, so that png_bands_kernel issues the un-filter
    work items in image order (its rule restated here)."""
    files = [W.image_file(40, 20 + k % 13, 4 if k % 3 else 1, k % 5, 200 + k, amp=1)[0] for k in range(300)]
    files.append(W.image_file(5, 45000, 1, [r % 5 for r in range(45000)], 7)[0])
    nb = [(int.from_bytes(f[20:24], "big") + 31) // 32 for f in files]
    fetches, carry = len(files) * max(nb), sum(nb)
    assert not fetches <= 8 * carry + 4096        # not band-major
    return files


@pytest.fixture(scope="module")
def large(ref):
    cases = W.catalogue(big=True)
    cases += [dict(name="F scheduling %d" % k, data=f) for k, f in enumerate(scheduling_batch())]
    for c in cases:
        c["rgba_size"] = rgba_size(c["data"])
        c["m"] = m = W.model(c["data"], c["rgba_size"])
        g, _, _, o = portlib.decode_png(c["data"], rgb_as_reference=False)
        if c["rgba_size"]:
            assert (g, o) == ((1, m["rgba"]) if m["verdict"] == "good" else (0, b"")), c["name"]
    return cases


def _check(c, st, out, what):
    m = c["m"]
    if m["verdict"] == "good":
        assert st == 0 and out == m["rgba"], (what, c["name"], st)
    elif m["verdict"] == "ub":
        assert st != 0, (what, c["name"])
    else:
        assert W.status_ok(m["status"], st), (what, c["name"], m["status"], st)


def _pack(files, caps):
    in_off, pos = [], 0
    for f in files:
        in_off.append(pos)
        pos += (len(f) + 15) // 16 * 16
    h_in = np.zeros(pos + 64, np.uint8)
    for o, f in zip(in_off, files):
        h_in[o:o + len(f)] = np.frombuffer(f, np.uint8)
    out_off = np.concatenate([[0], np.cumsum([(c + 15) // 16 * 16 for c in caps])[:-1]]).astype(np.uint64)
    h_out = np.zeros(int(sum((c + 15) // 16 * 16 for c in caps)) + 64, np.uint8)
    return h_in, np.array(in_off, np.uint64), np.array([len(f) for f in files], np.uint64), h_out, out_off, np.array(caps, np.uint64)


def _packed(ctx, cases, what):
    import debigulator_b200 as dbg
    h_in, in_off, in_size, h_out, out_off, out_cap = _pack([c["data"] for c in cases], [c["rgba_size"] for c in cases])
    _, st = ctx.decode_packed(dbg.api.KIND_PNG, h_in, in_off, in_size, h_out, out_off, out_cap)
    for i, c in enumerate(cases):
        o = int(out_off[i])
        _check(c, int(st[i]), h_out[o:o + c["rgba_size"]].tobytes(), what)


def test_read_back_route(ctx, large):
    """dbg_decode_png_batch (sizes from decode_png_get_width_height): verdict and RGBA of every case."""
    cases = [c for c in large if c["rgba_size"]]
    for c, (g, _, _, rgba) in zip(cases, ctx.decode_png_batch([c["data"] for c in cases])):
        want = c["m"]["verdict"] == "good"
        assert g == want and (not want or rgba == c["m"]["rgba"]), (c["name"], g)


def test_packed_routes(ctx, large, monkeypatch):
    """dbg_decode_batch_packed: the stb-shaped cases on their own (the hinted route, in waves), then every case in one
    mixed batch (the read-back route)."""
    import debigulator_b200 as dbg
    stb = [c for c in large if W.stb_shaped(c["data"])]
    assert len(stb) >= 60 and any(c.get("item4") for c in stb)
    monkeypatch.setenv("DBG_PNG_WAVES", "8")
    c8 = dbg.Context(0)
    try:
        fx0 = c8.fx_stats()[0]
        _packed(c8, stb, "hinted")
        assert c8.fx_stats()[0] > fx0                # the lane-serial path took the hinted streams
    finally:
        c8.close()
    _packed(ctx, large, "mixed")


def test_device_entry_point_at_every_input_alignment(ctx, large):
    """dbg_decode_png_batch_device, every case at every input offset mod 16 (the segment tasks' 16-byte copies and
    the un-filter's word loads see every alignment): the modelled status and RGBA."""
    import torch
    dev = torch.device("cuda", 0)
    items = [(c, a) for c in large if not c["name"].startswith("F") for a in range(16)]
    offs, total = [], 0
    for c, a in items:
        total = (total + 15) // 16 * 16 + a
        offs.append(total)
        total += len(c["data"])
    arena = np.zeros(total + 64, np.uint8)
    for o, (c, _) in zip(offs, items):
        arena[o:o + len(c["data"])] = np.frombuffer(c["data"], np.uint8)
    out_off, pos = [], 0
    for c, _ in items:
        out_off.append(pos)
        pos += (c["rgba_size"] + 15) // 16 * 16
    i64 = lambda a: torch.from_numpy(np.asarray(a, np.uint64).view(np.int64)).to(dev)
    d_out = torch.zeros(pos + 64, dtype=torch.uint8, device=dev)
    d_st = torch.full((len(items),), -1, dtype=torch.int32, device=dev)
    caps = [c["rgba_size"] for c, _ in items]
    ctx.png_device(torch.from_numpy(arena).to(dev), i64(offs), i64([len(c["data"]) for c, _ in items]), d_out, i64(out_off),
                   i64(caps), d_st, total, sum(caps))
    torch.cuda.synchronize()
    out, st = d_out.cpu().numpy(), d_st.cpu().numpy()
    for i, (c, a) in enumerate(items):
        _check(c, int(st[i]), out[out_off[i]:out_off[i] + caps[i]].tobytes(), ("device", a))


def test_crc_corruptions_in_a_64_image_batch(ctx):
    """64 images, each with a large ancillary chunk before its IDAT and a large one after; a byte of one of the two is
    flipped in a known third of them: exactly those get 13, every other one is byte-exact."""
    import torch
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(21)
    files, want, bad = [], [], set()
    for k in range(64):
        img = W._img(120 + k, 50, 4, 300 + k, amp=3)
        p1 = rng.integers(0, 256, 70000 + 977 * k, dtype=np.uint8).tobytes()
        p2 = rng.integers(0, 256, 140000 - 613 * k, dtype=np.uint8).tobytes()
        c1, c2 = W.chunk(b"bEfo", p1), W.chunk(b"aFtr", p2)
        if k % 3 == 1:
            bad.add(k)
            which = bytearray(c1 if k % 2 else c2)
            which[8 + int(rng.integers(0, len(which) - 12))] ^= 1 << (k % 8)
            c1, c2 = (bytes(which), c2) if k % 2 else (c1, bytes(which))
        z = W.zstream(W.scanlines(img, 1 + k % 4))
        files.append(W.png([W.ihdr(120 + k, 50, 6), c1] + W.split(z, []) + [c2, W.chunk(b"IEND")]))
        want.append(img.tobytes())
        m = W.model(files[-1])
        assert (m["status"], m["rgba"]) == ((W.ST_PNG_CRC, None) if k in bad else (W.ST_OK, want[-1])), k
    offs = np.concatenate([[0], np.cumsum([(len(f) + 15) // 16 * 16 for f in files])[:-1]])
    arena = np.zeros(int(offs[-1]) + len(files[-1]) + 64, np.uint8)
    for o, f in zip(offs, files):
        arena[o:o + len(f)] = np.frombuffer(f, np.uint8)
    caps = [len(w) for w in want]
    out_off = np.concatenate([[0], np.cumsum(caps)[:-1]])
    i64 = lambda a: torch.from_numpy(np.asarray(a, np.uint64).view(np.int64)).to(dev)
    d_out = torch.zeros(sum(caps) + 64, dtype=torch.uint8, device=dev)
    d_st = torch.full((64,), -1, dtype=torch.int32, device=dev)
    ctx.png_device(torch.from_numpy(arena).to(dev), i64(offs), i64([len(f) for f in files]), d_out, i64(out_off), i64(caps), d_st,
                   arena.size, sum(caps))
    torch.cuda.synchronize()
    out, st = d_out.cpu().numpy(), d_st.cpu().numpy()
    for k in range(64):
        if k in bad:
            assert st[k] == W.ST_PNG_CRC, (k, st[k])
        else:
            assert st[k] == 0 and out[out_off[k]:out_off[k] + caps[k]].tobytes() == want[k], (k, st[k])
