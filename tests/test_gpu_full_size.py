"""GPU parity at the sizes and with the generator BASELINE.json states (VERDICT r01, item 1): the batches bench.py
times -- config 3 (2048 x 1024^2, stb_write, six filter modes), config 4 (8192 x 8192, stb_write, forced Paeth),
configs 2 and 5 (every unique member) -- compared with the UNMODIFIED reference (oracle/_ref/libref.so) item by item.
Where the reference sources are not at hand (they are not part of the repository), the images come from the corpus's
own encoder of the same stream shape (corpus.png_bench) and every item is compared with the plain-C restatement,
which tests/test_oracle.py pins to the reference's stored outputs (the `ref` fixture, oracle/checker.py)."""
import hashlib
import multiprocessing as mp
import os

import numpy as np
import pytest

import debigulator_b200 as dbg
from debigulator_b200 import corpus

pytestmark = pytest.mark.gpu


def sha(b):
    return hashlib.sha256(b).hexdigest()


def _stb(spec):
    return corpus.png_bench(*spec)


def _pool(fn, args):
    with mp.get_context("fork").Pool(min(len(args), len(os.sched_getaffinity(0)))) as p:
        return p.map(fn, args, chunksize=1)


def _ref_png_sha(png):
    from oracle import checker
    good, w, h, rgba = checker.decode_png(png)
    return good, sha(rgba)


def _ref_gz(args):
    from oracle import checker
    g, cap = args
    good, out = checker.decode_gz(g, cap)
    return good, len(out), sha(out)


def test_cfg3_full_batch_stb_vs_reference(ctx, ref):
    """BASELINE config 3 as stated: 2048 PNGs of 1024x1024 RGBA written by stbi_write_png_to_mem (else by the corpus's
    encoder, one fixed-Huffman block as well), forced filter i % 6 - 1 (adaptive, None, Sub, Up, Avg, Paeth), 24 unique
    images cycled; every decoded image of the batch against `ref`'s decode_png of its file (decode_png.c:683)."""
    import torch
    uniq = _pool(_stb, [(i, 1024, 1024, None) for i in range(24)])
    want = _pool(_ref_png_sha, [u[0] for u in uniq])
    assert all(g == 1 for g, _ in want)
    for (p, rgba), (_, s) in zip(uniq, want):
        assert sha(rgba) == s              # the checker round-trips the writer's output
        assert p[8 + 8 + 13 + 4 + 8 + 2] & 7 == 3   # one final fixed-Huffman block behind the zlib header
    n, rgba = 2048, 1024 * 1024 * 4
    dev = torch.device("cuda", 0)
    offs, total = [], 0
    for i in range(n):
        offs.append(total)
        total += (len(uniq[i % 24][0]) + 31) // 16 * 16
    h = np.zeros(total + 64, np.uint8)
    for i in range(n):
        b = uniq[i % 24][0]
        h[offs[i]:offs[i] + len(b)] = np.frombuffer(b, np.uint8)
    i64 = lambda a: torch.from_numpy(np.asarray(a, np.uint64).view(np.int64)).to(dev)
    sizes = [len(uniq[i % 24][0]) for i in range(n)]
    d_in = torch.from_numpy(h).to(dev)
    d_out = torch.zeros(n * rgba, dtype=torch.uint8, device=dev)
    st = torch.full((n,), 99, dtype=torch.int32, device=dev)
    fx0 = ctx.fx_stats()
    ctx.png_device(d_in, i64(offs), i64(sizes), d_out, i64(np.arange(n, dtype=np.uint64) * np.uint64(rgba)), i64(np.full(n, rgba, np.uint64)),
                   st, sum(sizes), n * rgba)
    torch.cuda.synchronize()
    assert int(st.abs().sum().item()) == 0
    assert ctx.fx_stats()[0] - fx0[0] == n and ctx.fx_stats()[1] == fx0[1]
    got = d_out.view(n, rgba)
    exp = torch.stack([torch.from_numpy(np.frombuffer(u[1], np.uint8).copy()) for u in uniq]).to(dev)
    idx = torch.arange(n, device=dev) % 24
    for s in range(0, n, 64):
        assert torch.equal(got[s:s + 64], exp[idx[s:s + 64]]), s
    for k in (0, 5, 23, 1000, 2047):      # and byte-for-byte on the host for a few
        assert sha(got[k].cpu().numpy().tobytes()) == want[k % 24][1]
    del d_in, d_out
    ctx.trim()
    torch.cuda.empty_cache()


def test_cfg4_8192_stb_paeth_vs_reference_both_paths(ref, monkeypatch):
    """BASELINE config 4 at its own size and generator: stb-written (else corpus-written) 8192x8192 forced-Paeth RGBA
    PNGs (151 MB each from stb, one fixed-Huffman block of ~65 M symbols) through the lane-serial path AND, with that
    path switched off, through one warp per stream; both byte-compared with `ref`'s decode_png."""
    uniq = _pool(_stb, [(100 + i, 8192, 8192, 4) for i in range(2)])
    want = _pool(_ref_png_sha, [u[0] for u in uniq])
    for (p, rgba), (g, s) in zip(uniq, want):
        assert g == 1 and sha(rgba) == s and len(p) > 100_000_000
    files = [u[0] for u in uniq]
    c = dbg.Context(0)
    fx0 = c.fx_stats()
    res = c.decode_png_batch(files + files + files[:1])  # five items: through the packed path, not the batch-of-one route
    assert c.fx_stats()[0] - fx0[0] == 5
    for k, (good, w, h, rgba) in enumerate(res):
        assert good == 1 and (w, h) == (8192, 8192)
        assert sha(rgba) == want[k % 2][1], k
    del res
    c.close()
    monkeypatch.setenv("DBG_FX", "0")
    c = dbg.Context(0)
    (good, w, h, rgba), = c.decode_png_batch(files[:1])
    assert good == 1 and sha(rgba) == want[0][1]
    assert c.fx_stats()[0] == 0
    c.close()


def test_cfg2_and_cfg5_every_unique_member_vs_reference(ctx, ref):
    """Every unique member of the config-2 batch (64: 16 per class) and of the config-5-shape batch (64, 64 KiB-16 MiB,
    eight classes, including the ones the reference's rule Q2 cuts short) that bench.py cycles: status, size and
    payload hash against `ref`."""
    import bench
    cfg2 = [corpus.gz_member_cfg2(i, 1 << 20) for i in range(64)]
    cfg5 = _pool(bench._gen_cfg5, list(range(64)))
    members = [g for g, _ in cfg2] + [g for g, _, _ in cfg5]
    caps = [len(d) + len(g) + 64 for g, d in cfg2] + [(m + len(g) + 64 + 15) // 16 * 16 for g, m, _ in cfg5]
    want = _pool(_ref_gz, list(zip(members, caps)))
    got = ctx.decode_gz_batch(members, caps)
    short = 0
    for k, ((good, out), (rgood, rlen, rsha)) in enumerate(zip(got, want)):
        assert good == rgood == 1, k
        assert len(out) == rlen and sha(out) == rsha, k
        if k >= 64 and rlen != cfg5[k - 64][1]:
            short += 1
    assert short >= 1                      # the rule-Q2 members are really in there
