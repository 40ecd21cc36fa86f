"""BMP decode / encode (SURVEY.md 8(f) rank 4; decode_bmp.c:53-372).

CPU part: the plain-C restatement against the reference's own outputs (tests/golden/bmp_manifest.json,
made by make_golden_bmp.py from the unmodified decode_bmp.c) and against the reference live when it is
available. GPU part (-m gpu): the product through the C-ABI -- host batches, the device-resident
entry points and the drop-in decode_bmp.h functions -- against the same vectors and the checker."""
import base64
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

from debigulator_b200 import corpus
from oracle import checker, portlib, reflib

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sha = lambda b: hashlib.sha256(b).hexdigest()


@pytest.fixture(scope="module")
def bmp_manifest():
    with open(os.path.join(GOLDEN, "bmp_manifest.json")) as f:
        return json.load(f)


def _cases(m):
    for name, e in m["fixtures"].items():
        yield name, open(os.path.join(GOLDEN, name), "rb").read(), e
    for name, e in m["synthetic"].items():
        yield name, base64.b64decode(e["b64"]), e


def _random_bmps(seed, count):
    rng = np.random.default_rng(seed)
    for t in range(count):
        w, h = int(rng.integers(1, 300)), int(rng.integers(1, 40))
        if t % 7 == 0:
            w, h = int(rng.integers(4097, 9000)), int(rng.integers(1, 4))  # rows wider than one tile
        rgba = rng.integers(0, 256, w * h * 4, dtype=np.uint8).tobytes()
        yield rgba, w, h, corpus.bmp_file(rgba, w, h, bottom_up=bool(t & 1), v4=bool(t & 2), pad=int(rng.integers(0, 4)))


# ------------------------------------------------------------------ CPU: oracle --
def test_port_matches_golden(bmp_manifest):
    for name, data, e in _cases(bmp_manifest):
        g, w, h, rgba = portlib.decode_bmp(data)
        assert g == e["good"], name
        assert portlib.bmp_dims(data)[0] == e["dims_good"], name
        if g:
            assert (w, h) == (e["w"], e["h"]) and sha(rgba) == e["rgba_sha256"], name
            n, enc = portlib.encode_bmp(rgba, w, h)
            assert n == e["encode_size"] and sha(enc) == e["encode_sha256"], name


@pytest.mark.skipif(not reflib.available(), reason="needs the reference sources (oracle/_ref)")
def test_port_matches_reference_random():
    for rgba, w, h, data in _random_bmps(11, 40):
        r = reflib.decode_bmp(data)
        assert r == portlib.decode_bmp(data) and r[0] == 1 and r[3] == rgba
        assert reflib.encode_bmp(rgba, w, h) == portlib.encode_bmp(rgba, w, h)


def test_round_trip_property():
    # encode -> decode is the identity (the encoder writes a top-down file)
    for rgba, w, h, _ in _random_bmps(12, 10):
        n, enc = portlib.encode_bmp(rgba, w, h)
        assert n == 54 + len(rgba) + 1
        assert portlib.decode_bmp(enc)[3] == rgba


# ------------------------------------------------------------------ GPU: product --
@pytest.mark.gpu
def test_gpu_decode_golden(ctx, bmp_manifest):
    cases = list(_cases(bmp_manifest))
    got = ctx.decode_bmp_batch([c[1] for c in cases])
    for (name, data, e), (g, w, h, rgba) in zip(cases, got):
        assert g == e["good"], name
        if g:
            assert (w, h) == (e["w"], e["h"]) and sha(rgba) == e["rgba_sha256"], name


@pytest.mark.gpu
def test_gpu_encode_golden(ctx, bmp_manifest):
    cases = [c for c in _cases(bmp_manifest) if c[2]["good"]]
    imgs = []
    for name, data, e in cases:
        g, w, h, rgba = checker.decode_bmp(data)
        imgs.append((rgba, w, h))
    for (name, data, e), (st, n, enc) in zip(cases, ctx.encode_bmp_batch(imgs)):
        assert st == 0 and n == e["encode_size"] and sha(enc) == e["encode_sha256"], name


@pytest.mark.gpu
def test_gpu_random_parity_and_round_trip(ctx):
    items = list(_random_bmps(21, 60))
    got = ctx.decode_bmp_batch([it[3] for it in items])
    for (rgba, w, h, data), (g, gw, gh, out) in zip(items, got):
        assert (g, gw, gh) == (1, w, h) and out == rgba == checker.decode_bmp(data)[3]
    enc = ctx.encode_bmp_batch([(it[0], it[1], it[2]) for it in items])
    for (rgba, w, h, _), (st, n, out) in zip(items, enc):
        assert st == 0 and (n, out) == checker.encode_bmp(rgba, w, h)
    back = ctx.decode_bmp_batch([e[2] + b"\0" for e in enc])
    assert [b[3] for b in back] == [it[0] for it in items]


@pytest.mark.gpu
def test_gpu_out_of_bounds_inputs_are_rejected(ctx):
    rgba = bytes(range(256)) * 4
    good = corpus.bmp_file(rgba, 16, 16)
    # pixel data past the end of the file, output smaller than w*h*4, negative width, header cut short
    import struct
    neg = bytearray(good)
    struct.pack_into("<i", neg, 18, -16)
    res = ctx.decode_bmp_batch([good[:-8], good, bytes(neg), good[:40], good], caps=[1024, 1000, 1024, 1024, 2048])
    assert [r[0] for r in res] == [0, 0, 0, 0, 1]
    assert res[4][3] == rgba  # a larger output buffer is fine (decode_bmp.c:188-202 has no effect)
    enc = ctx.encode_bmp_batch([(rgba, 16, 16), (rgba[:1022], 16, 16), (rgba, 16, 16)], caps=[54 + 1024, 54 + 1023, 54 + 1025])
    assert [e[0] != 0 for e in enc] == [True, True, False]


@pytest.mark.gpu
def test_gpu_scalar_bmp_api(ctx, bmp_manifest):
    import debigulator_b200 as dbg
    L = dbg.load_library()
    L.decode_BMP.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_int64, C.POINTER(C.c_uint8)]
    L.decode_BMP.restype = None
    L.encode_BMP.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p, C.POINTER(C.c_uint32), C.c_int64]
    L.encode_BMP.restype = None
    data = open(os.path.join(GOLDEN, "fs_psychologist.bmp"), "rb").read()
    e = bmp_manifest["fixtures"]["fs_psychologist.bmp"]
    assert dbg.api.bmp_get_width_height(data) == (1, e["w"], e["h"])
    assert dbg.api.bmp_get_width_height(b"BA" + data[2:])[0] == 0
    n = e["w"] * e["h"] * 4
    ib = C.create_string_buffer(data, len(data))
    ob = C.create_string_buffer(n)
    g = C.c_uint8(7)
    L.decode_BMP(ib, len(data), ob, n, C.byref(g))
    assert g.value == 1 and sha(ob.raw) == e["rgba_sha256"]
    rb = C.create_string_buffer(54 + n + 1)
    rs = C.c_uint32(0)
    L.encode_BMP(ob, n, e["w"], e["h"], rb, C.byref(rs), 54 + n + 1)
    assert rs.value == e["encode_size"] and sha(rb.raw[: rs.value - 1]) == e["encode_sha256"]
    L.decode_BMP(ib, 20, ob, n, C.byref(g))
    assert g.value == 0


@pytest.mark.gpu
def test_gpu_device_api_misaligned(ctx):
    """Device-resident batch with files at odd offsets and outputs at 2-byte offsets (every alignment path)."""
    import torch
    items = list(_random_bmps(31, 24))
    dev = torch.device("cuda", 0)
    in_off, out_off, pos, opos = [], [], 1, 0
    for k, it in enumerate(items):
        in_off.append(pos)
        pos += len(it[3]) + (k % 4) + 1
        out_off.append(opos)
        opos += len(it[0]) + (0, 2, 4, 1)[k % 4]
    h_in = np.zeros(pos + 16, np.uint8)
    for o, it in zip(in_off, items):
        h_in[o:o + len(it[3])] = np.frombuffer(it[3], np.uint8)
    i64 = lambda a: torch.from_numpy(np.asarray(a, np.uint64).view(np.int64)).to(dev)
    d_in = torch.from_numpy(h_in).to(dev)
    d_out = torch.zeros(opos + 16, dtype=torch.uint8, device=dev)
    n = len(items)
    osz = torch.zeros(n, dtype=torch.int64, device=dev)
    st = torch.full((n,), 99, dtype=torch.int32, device=dev)
    wd = torch.zeros(n, dtype=torch.int32, device=dev)
    ht = torch.zeros(n, dtype=torch.int32, device=dev)
    ctx.bmp_decode_device(d_in, i64(in_off), i64([len(it[3]) for it in items]), d_out, i64(out_off),
                          i64([len(it[0]) for it in items]), osz, st, wd, ht)
    ctx.synchronize()
    out = d_out.cpu().numpy()
    assert st.tolist() == [0] * n
    for k, it in enumerate(items):
        assert (wd[k].item(), ht[k].item(), osz[k].item()) == (it[1], it[2], len(it[0]))
        assert out[out_off[k]:out_off[k] + len(it[0])].tobytes() == it[0], k
    # encode from the (mis)aligned RGBA we just produced
    e_off, epos = [], 3
    for it in items:
        e_off.append(epos)
        epos += 54 + len(it[0]) + 1 + 3
    d_enc = torch.zeros(epos + 16, dtype=torch.uint8, device=dev)
    esz = torch.zeros(n, dtype=torch.int64, device=dev)
    est = torch.full((n,), 99, dtype=torch.int32, device=dev)
    ctx.bmp_encode_device(d_out, i64(out_off), i64([len(it[0]) for it in items]), wd, ht, d_enc, i64(e_off),
                          i64([54 + len(it[0]) + 1 for it in items]), esz, est)
    ctx.synchronize()
    enc = d_enc.cpu().numpy()
    assert est.tolist() == [0] * n
    for k, it in enumerate(items):
        size, want = checker.encode_bmp(it[0], it[1], it[2])
        assert esz[k].item() == size
        assert enc[e_off[k]:e_off[k] + size - 1].tobytes() == want, k


def _sheet(images, w, h, cols):
    n = len(images)
    rows = (n + cols - 1) // cols
    sheet = np.zeros((rows * h, cols * w, 4), np.uint8)
    for i, im in enumerate(images):
        r, c = divmod(i, cols)
        sheet[r * h:(r + 1) * h, c * w:(c + 1) * w] = np.frombuffer(im, np.uint8).reshape(h, w, 4)
    return sheet.tobytes(), rows


@pytest.mark.gpu
def test_sprite_sheet_tiling(ctx):
    """dbg_tile_sprites / dbg_tile_sprites_device (the intent of the reference's concat_pngs.c:81-100, whose
    concatenate_images() is not defined anywhere in the reference tree): decoded images become the cells of a row-major
    grid, empty cells transparent black. Host and device forms, tile widths that do and do not allow 16-byte accesses,
    the default square-ish grid and a caller-given number of columns -- against a numpy tiling; the device form on the
    output of the PNG decoder."""
    import torch
    from debigulator_b200 import corpus
    for n, w, h, cols in ((7, 96, 64, 0), (3, 33, 17, 0), (10, 64, 8, 4), (1, 5, 5, 0), (5, 40, 30, 5)):
        images = [corpus.gradient_noise_rgba(w, h, 40 + i).tobytes() for i in range(n)]
        got, r, c = ctx.tile_sprites(images, w, h, cols)
        want_c = cols or next(k for k in range(1, n + 2) if k * k >= n)
        want, want_r = _sheet(images, w, h, min(want_c, n))
        assert (r, c) == (want_r, min(want_c, n)), (n, w, h, cols, r, c)
        assert got == want, (n, w, h, cols)
    # device form, fed by the PNG decoder's output arena
    n, w, h = 6, 128, 96
    files, pix = zip(*[corpus.png_cfg3(6 * i + 5, w, h) for i in range(n)])  # forced Paeth (a None-filtered tile this small trips rule Q12)
    dev = torch.device("cuda", 0)
    in_off = np.concatenate([[0], np.cumsum([(len(f) + 31) // 16 * 16 for f in files[:-1]])]).astype(np.int64)
    h_in = np.zeros(int(in_off[-1]) + len(files[-1]) + 64, np.uint8)
    for f, o in zip(files, in_off):
        h_in[o:o + len(f)] = np.frombuffer(f, np.uint8)
    rgba = w * h * 4
    d_in = torch.from_numpy(h_in).to(dev)
    d_out = torch.zeros(n * rgba, dtype=torch.uint8, device=dev)
    t64 = lambda a: torch.from_numpy(np.asarray(a, np.int64)).to(dev)
    o_off = t64(np.arange(n) * rgba)
    st = torch.zeros(n, dtype=torch.int32, device=dev)
    ctx.png_device(d_in, t64(in_off), t64([len(f) for f in files]), d_out, o_off, t64([rgba] * n), st, int(sum(len(f) for f in files)), n * rgba)
    d_sheet = torch.zeros(3 * w * 2 * h * 4, dtype=torch.uint8, device=dev)
    r, c = ctx.tile_sprites_device(d_out, o_off, n, w, h, 0, True, d_sheet)
    torch.cuda.synchronize()
    assert int(st.abs().sum()) == 0, st.tolist()
    assert (r, c) == (2, 3)
    assert d_sheet.cpu().numpy().tobytes() == _sheet(pix, w, h, 3)[0]
    with pytest.raises(Exception):
        ctx.tile_sprites_device(d_out, o_off, n, w, h, 0, True, d_sheet[:100])
