#!/usr/bin/env python
"""bench.py -- headline benchmark of the batched inflate / gzip / PNG decode path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python bench.py --strong cfg4|cfg5 --gpus N        (one batch over N GPUs through dbg_decode_batch_packed_multi)

One "step" = one pass of the hot path over one batch of synthetic input. The headline workload is BASELINE.json
config 2: a batch of 4096 synthetic 1 MiB gzip members per GPU (classes stored / fixed / dynamic / mixed by i % 4,
SURVEY.md 8d), decoded to their payloads. Weak scaling: every rank decodes its own batch; no collective is needed on
the data path (NCCL carries the barrier and the max-over-ranks reduction only).

  value         decompressed GB/s, whole job, inputs resident in HBM, CUDA events on the launching stream, max over ranks
  e2e           the same metric through the public C-ABI with pinned HOST buffers: H2D + kernels + D2H inside the call
  roofline      algorithmic bytes (C + U) per launch / event-timed duration of the dominant kernel, over the measured HBM peak
  cpu_baseline  the reference C on this box's host cores: one process per core, a bounded sample, plus one thread alone
  png, png_cfg4 BASELINE configs 3 and 4 (PNG half of the metric, Mpixels/s) with the same four objects each; the
                images are written by the reference's own stb_write.h (debigulator_b200/tools/stb_gen.c)
  cfg5_shape, bmp, cfg1   secondary lines (DESIGN.md "Measurement")

`--impl reference` times the reference's own CPU implementation (oracle/_ref, the unmodified C sources; else the
oracle port) on all host cores, on a bounded sample of the same workload. Pool, input distribution and buffers are
set up before the clock starts; each worker times nothing but its calls of the reference entry point.
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# the packed host API runs up to 16 waves on streams of their own; with the default 8 hardware queues waves on one
# queue wait for each other (INTEGRATION.md). Must be set before torch creates the CUDA context.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

MEMBER_BYTES = 1 << 20
N_MEMBERS = 4096
N_UNIQUE = 64
PNG_N, PNG_W, PNG_H, PNG_UNIQUE = 2048, 1024, 1024, 24
PNG4_N, PNG4_W, PNG4_H, PNG4_UNIQUE = 32, 8192, 8192, 8
METRIC = "inflate_output_GBps"
UNIT = "GB/s"


def _gen_gz(i):
    from debigulator_b200 import corpus
    return corpus.gz_member_cfg2(i, MEMBER_BYTES)


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def pool_map(fn, args, workers=None):
    workers = max(1, min(workers or host_cores(), len(args)))
    if workers == 1:
        return [fn(a) for a in args]
    with mp.get_context("fork").Pool(workers) as pool:
        return pool.map(fn, args, chunksize=1)


def make_unique(gen, count):
    return pool_map(gen, list(range(count)))


def pack(items, n, align=16, pad=16):
    """Cycles `items` (compressed bytes) to n entries inside one arena."""
    offs, sizes, total = [], [], 0
    for i in range(n):
        b = items[i % len(items)]
        offs.append(total)
        sizes.append(len(b))
        total += (len(b) + pad + align - 1) // align * align
    return offs, sizes, total


# ---------------------------------------------------------------- CPU baseline --
_CPU_JOB = None  # (what, blobs, caps): set in the parent before the workers are forked, so nothing is pickled


def _cpu_worker(w, procs, steps, warmup, barrier, q):
    try:
        from oracle import checker
        what, blobs, caps = _CPU_JOB
        runner = checker.TimedRunner(what, blobs[w::procs], caps[w::procs])
        for _ in range(warmup):
            runner.run()
        times, nbytes = [], 0
        for _ in range(steps):
            barrier.wait()
            dt, nbytes = runner.run()
            times.append(dt)
        q.put((w, times, nbytes, None))
    except Exception as e:  # pragma: no cover
        try:
            barrier.abort()
        except Exception:
            pass
        q.put((w, [], 0, repr(e)))


def cpu_throughput(what, blobs, caps, procs, steps=1, warmup=1):
    """One process per core on the reference C (slot 0 each, own working memory), static partition. Everything is
    set up before the clock: the workers are forked with their shards in place, allocate their buffers, run `warmup`
    untimed passes and then time only their calls. A step's duration is the slowest worker's. Returns
    (bytes per step, [seconds of every step])."""
    global _CPU_JOB
    procs = max(1, min(procs, len(blobs)))
    _CPU_JOB = (what, blobs, caps)
    if procs == 1:
        from oracle import checker
        runner = checker.TimedRunner(what, blobs, caps)
        for _ in range(warmup):
            runner.run()
        out = [runner.run() for _ in range(steps)]
        return out[0][1], [o[0] for o in out]
    ctx = mp.get_context("fork")
    barrier, q = ctx.Barrier(procs), ctx.Queue()
    ps = [ctx.Process(target=_cpu_worker, args=(w, procs, steps, warmup, barrier, q)) for w in range(procs)]
    for p in ps:
        p.start()
    res = [q.get() for _ in ps]
    for p in ps:
        p.join()
    err = [r[3] for r in res if r[3]]
    if err:
        raise RuntimeError("CPU baseline worker failed: " + err[0])
    return sum(r[2] for r in res), [max(r[1][k] for r in res) for k in range(steps)]


# ------------------------------------------------------------------- clocks -----
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------ reference ---
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import checker
    cores = host_cores()
    uniq = make_unique(_gen_gz, N_UNIQUE)
    per_step = cores * 32  # members per step: a bounded sample of the 4096-member batch, 8 of every class per core
    blobs = [uniq[i % N_UNIQUE][0] for i in range(per_step)]
    caps = [MEMBER_BYTES + len(b) for b in blobs]
    step_bytes, step_s = cpu_throughput("gz", blobs, caps, cores, steps=args.steps, warmup=max(1, min(args.warmup, 2)))
    b1, s1 = cpu_throughput("gz", blobs[:32], caps[:32], 1, steps=1, warmup=1)
    tot_s = sum(step_s)
    val = step_bytes * args.steps / tot_s / 1e9
    sample = (f"{per_step} of {N_MEMBERS} members per step ({per_step * MEMBER_BYTES >> 20} MiB out), one process per core, "
              "pool and buffers set up before the clock, each worker times only its reference calls, step = slowest worker")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": tot_s / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "cfg2: 4096 x 1 MiB gzip members (stored/fixed/dynamic/mixed by i%4)", "sample": sample},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": checker.kind(), "sample": sample,
                         "single_thread": {"value": b1 / s1[0] / 1e9, "unit": UNIT, "sample": "32 members (8 per class)"},
                         "parallel_efficiency": val / (b1 / s1[0] / 1e9 * cores)},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------ PNG ---
def _gen_png(spec):
    """spec = (index, w, h, forced filter or None). stb_write when the tooling is there, else the own encoder."""
    from debigulator_b200 import corpus
    return corpus.png_bench(*spec)


def png_corpus(w, h, n_unique, filt, share_tag=None, rank=0, world=1, barrier=None):
    """n_unique images. Large ones are written once per box (rank 0, all cores) and handed to the other ranks through
    /dev/shm."""
    specs = [(i, w, h, filt) for i in range(n_unique)]
    if share_tag is None or world == 1:
        return pool_map(_gen_png, specs)
    path = f"/dev/shm/dbg_bench_{share_tag}_{os.environ.get('MASTER_PORT', '0')}"
    if rank == 0:
        uniq = pool_map(_gen_png, specs)
        for k, (p, r) in enumerate(uniq):
            with open(f"{path}_{k}.png", "wb") as f:
                f.write(p)
            with open(f"{path}_{k}.rgba", "wb") as f:
                f.write(r)
    barrier()
    if rank != 0:
        uniq = [(open(f"{path}_{k}.png", "rb").read(), open(f"{path}_{k}.rgba", "rb").read()) for k in range(n_unique)]
    barrier()
    if rank == 0:
        for k in range(n_unique):
            os.unlink(f"{path}_{k}.png")
            os.unlink(f"{path}_{k}.rgba")
    return uniq


def bench_png(ctx, dbg, dev, torch, name, n, w, h, uniq, peak, steps, e2e=True, cpu=True, world=1, max_over_ranks=lambda x: x,
              barrier=lambda: None, e2e_images=None):
    from debigulator_b200 import corpus
    n_unique = len(uniq)
    offs, sizes, in_total = pack([u[0] for u in uniq], n)
    rgba = w * h * 4
    ne = min(n, e2e_images or n)  # images of the end-to-end leg (all of them unless host memory is short at N > 1)
    pinned = e2e
    h_in_t = torch.empty(in_total + 64, dtype=torch.uint8)
    if pinned:
        h_in_t = h_in_t.pin_memory()
    h_in = h_in_t.numpy()
    h_in[:] = 0
    for i in range(n):
        b = uniq[i % n_unique][0]
        h_in[offs[i]:offs[i] + len(b)] = np.frombuffer(b, np.uint8)
    d_in = h_in_t.to(dev)
    d_out = torch.zeros(n * rgba, dtype=torch.uint8, device=dev)
    i64 = lambda a: torch.from_numpy(np.asarray(a, dtype=np.uint64).view(np.int64)).to(dev)
    in_off, in_size = np.asarray(offs, np.uint64), np.asarray(sizes, np.uint64)
    out_off, out_cap = np.arange(n, dtype=np.uint64) * np.uint64(rgba), np.full(n, rgba, dtype=np.uint64)
    d_in_off, d_in_size, d_out_off, d_out_cap = i64(in_off), i64(in_size), i64(out_off), i64(out_cap)
    d_status = torch.zeros(n, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    tot_in = int(in_size.sum())

    def step():
        ctx.png_device(d_in, d_in_off, d_in_size, d_out, d_out_off, d_out_cap, d_status, tot_in, n * rgba, stream=stream)

    exp = torch.stack([torch.from_numpy(np.frombuffer(u[1], np.uint8).copy()) for u in uniq]).to(dev)
    idx = torch.arange(n, device=dev) % n_unique
    step_chk = max(1, (1 << 28) // rgba)

    def verify(buf):
        got = buf.view(n, rgba)
        for s in range(0, n, step_chk):
            assert torch.equal(got[s:s + step_chk], exp[idx[s:s + step_chk]]), f"{name}: pixel mismatch"

    fx0 = ctx.fx_stats()
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    assert int(d_status.abs().sum().item()) == 0, f"{name}: decode failures"
    verify(d_out)
    d_out.zero_()
    barrier()
    ctx.profile_enable(True)
    launches0 = ctx.kernel_launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / steps
    launches = (ctx.kernel_launches - launches0) // steps
    groups = {}
    for tag, gname in ((ctx.PROF_PNG_SCAN, "chunk walk + CRC-32"), (ctx.PROF_FX_SIZES, "inflate: head + sizes + chain"),
                       (ctx.PROF_FX_EXPAND, "inflate: tokens + expansion + resolve"), (ctx.PROF_INFLATE, "inflate: warp per stream"),
                       (ctx.PROF_PNG_UNFILTER, "un-filter")):
        t, k = ctx.profile_read_tag(tag)
        if k:
            groups[gname] = t / steps
    ctx.profile_enable(False)
    verify(d_out)
    fx1 = ctx.fx_stats()
    alg = tot_in + n * rgba                      # F + 4wh per image (SURVEY.md 8d)
    scan = n * (rgba + h + 1)                    # S: the filtered scanlines in between
    dom = max(groups, key=groups.get)
    value = world * n * w * h / (ms / 1e3) / 1e6
    out = {"metric": "png_decode_Mpixels_per_s", "value": value, "unit": "Mpix/s", "rgba_GBps": world * n * rgba / (ms / 1e3) / 1e9,
           "ms_per_step": ms, "steps": steps, "n_gpus": world, "gpu_launches": int(launches),
           "config": {"workload": f"{name}: {n} x {w}x{h} RGBA8 PNGs per GPU, written by "
                                  + ("the reference's stb_write.h (stbi_write_png_to_mem: one IDAT, one fixed-Huffman block)"
                                     if corpus.stb_available() else "tools/fixed_deflate.c (stb stream shape; stb_write.h tooling not built)"),
                      "unique_images": n_unique, "png_bytes_per_gpu": tot_in, "rgba_bytes_per_gpu": n * rgba,
                      "lane_serial_streams_per_step": (fx1[0] - fx0[0]) // (steps + 2), "handed_back": fx1[1] - fx0[1],
                      "l2": "inputs+outputs per step (%.1f GB) exceed the 126 MB L2; no explicit flush" % (alg / 1e9)},
           "roofline": {"bound": "hbm", "achieved": alg / (groups[dom] / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": alg / (groups[dom] / 1e3) / 1e9 / peak, "traffic": None, "kernel": dom, "avg_launch_ms": groups[dom],
                        "algorithmic_bytes_per_launch": alg, "whole_step_achieved": alg / (ms / 1e3) / 1e9,
                        "whole_step_frac": alg / (ms / 1e3) / 1e9 / peak,
                        "implementation_bytes_floor": tot_in * 3 + scan * 6 + n * rgba,
                        "implementation_note": "F read by CRC, sizes and token passes; S: 2 B cells written + read, bytes written, read by "
                                               "the un-filter (+ 8 B per symbol of tokens, not counted); 4wh written",
                        "kernel_groups_ms": groups}}
    if e2e:
        h_out_t = torch.empty(ne * rgba, dtype=torch.uint8).pin_memory()
        h_out = h_out_t.numpy()
        e_in = offs[ne] if ne < n else in_total
        a4 = (in_off[:ne], in_size[:ne], out_off[:ne], out_cap[:ne])
        ctx.decode_packed(dbg.api.KIND_PNG, h_in, a4[0], a4[1], h_out, a4[2], a4[3])
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            osz, st = ctx.decode_packed(dbg.api.KIND_PNG, h_in, a4[0], a4[1], h_out, a4[2], a4[3])
        torch.cuda.synchronize()
        dt1 = max_over_ranks(time.perf_counter() - t0) / steps
        assert int(st.sum()) == 0 and int(osz.sum()) == ne * rgba, f"{name}: e2e failures"
        for k in (0, 1, ne // 2, ne - 1):
            assert h_out[k * rgba:(k + 1) * rgba].tobytes() == uniq[k % n_unique][1], f"{name}: e2e pixel mismatch"
        # two calls in flight (dbg_pipe_*): the batch as two sub-batches, one's ramp under the other's downloads
        ctx.trim()
        h_out[:] = 0
        dt, osz, st, pipe_launches = e2e_pipelined(dbg, dev.index, dbg.api.KIND_PNG, h_in, a4[0], a4[1], h_out, a4[2], a4[3], steps,
                                                   barrier, max_over_ranks)
        assert int(st.sum()) == 0 and int(osz.sum()) == ne * rgba, f"{name}: pipelined e2e failures"
        for k in (0, 1, ne // 2 - 1, ne // 2, ne - 1):
            assert h_out[k * rgba:(k + 1) * rgba].tobytes() == uniq[k % n_unique][1], f"{name}: pipelined e2e pixel mismatch"
        # link ceiling: the same arenas copied up and down at once, nothing else running (all ranks together)
        s_up, s_dn = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        barrier()
        t0 = time.perf_counter()
        with torch.cuda.stream(s_up):
            d_in[:e_in].copy_(h_in_t[:e_in], non_blocking=True)
        with torch.cuda.stream(s_dn):
            h_out_t.copy_(d_out[:ne * rgba], non_blocking=True)
        torch.cuda.synchronize()
        ct = max_over_ranks(time.perf_counter() - t0)
        out["e2e"] = {"value": world * ne * w * h / dt / 1e6, "unit": "Mpix/s", "rgba_GBps": world * ne * rgba / dt / 1e9,
                      "ms_per_step": dt * 1e3, "images_per_gpu": ne, "h2d_bytes_per_step": int(e_in), "d2h_bytes_per_step": int(ne * rgba),
                      "steps": steps, "calls_in_flight": 2,
                      "api": "dbg_pipe_submit / dbg_pipe_wait (kind=PNG): every step's batch as two packed sub-batches of the same "
                             "pinned host arenas, two in flight",
                      "single_call": {"value": world * ne * w * h / dt1 / 1e6, "unit": "Mpix/s", "ms_per_step": dt1 * 1e3,
                                      "api": "dbg_decode_batch_packed(kind=PNG), one blocking call per step", "frac_of_ceiling": ct / dt1},
                      "kernel_launches_per_step": pipe_launches,
                      "link_ceiling": {"h2d_plus_d2h_s": ct, "Mpix_s_if_copies_only": world * ne * w * h / ct / 1e6,
                                       "ranks_copying_at_once": world, "per_rank_h2d_GBps": e_in / ct / 1e9,
                                       "per_rank_d2h_GBps": ne * rgba / ct / 1e9, "frac_of_ceiling": ct / dt}}
        del h_out_t
    if cpu:
        from oracle import checker
        cores = host_cores()
        per_core = 8 if rgba <= (1 << 24) else 1
        m = min(n, cores * per_core) if per_core > 1 else min(cores, n_unique, 8)
        blobs = [uniq[i % n_unique][0] for i in range(m)]
        caps = [rgba] * m
        procs = min(cores, m)
        sb, ss = cpu_throughput("png", blobs, caps, procs, steps=1, warmup=0 if per_core == 1 else 1)
        b1, s1 = cpu_throughput("png", blobs[:1], caps[:1], 1, steps=1, warmup=0)
        out["cpu_baseline"] = {"value": sb / 4 / ss[0] / 1e6, "unit": "Mpix/s", "cores": procs, "kind": checker.kind(),
                               "sample": f"{m} of {n} images, one process per core (reference decode_png, decode_png.c:683)",
                               "single_thread": {"value": b1 / 4 / s1[0] / 1e6, "unit": "Mpix/s", "sample": "1 image"}}
    return out


def e2e_pipelined(dbg, dev_index, kind, h_in_np, in_off, in_size, h_out_np, out_off, out_cap, steps, barrier, max_over_ranks,
                  parts=2, depth=2):
    """The packed host API with `depth` calls in flight (dbg_pipe_*): every step's batch goes through the pipe as `parts`
    consecutive sub-batches of the same pinned arenas, so one sub-batch's ramp (first upload, first kernels) runs under the
    previous one's downloads. Every step still uploads all of its inputs and downloads all of its outputs.
    Returns (seconds per step, out_size, status, kernel launches per step)."""
    n = len(in_off)
    cuts = [n * k // parts for k in range(parts + 1)]
    pipe = dbg.Pipe(dev_index, depth)

    def submit_step():
        return [pipe.submit(kind, h_in_np, in_off[a:b], in_size[a:b], h_out_np, out_off[a:b], out_cap[a:b])
                for a, b in zip(cuts, cuts[1:])]

    for t in submit_step():  # warm-up: the contexts size their arenas and scratch
        pipe.wait(t)
    l0 = pipe.kernel_launches()
    barrier()
    t0 = time.perf_counter()
    tickets = []
    for _ in range(steps):
        tickets += submit_step()  # blocks while `depth` sub-batches are in flight
    res = [pipe.wait(t) for t in tickets]
    dt = max_over_ranks(time.perf_counter() - t0) / steps
    osz = np.concatenate([r[0] for r in res[-parts:]])
    st = np.concatenate([r[1] for r in res[-parts:]])
    launches = (pipe.kernel_launches() - l0) / steps
    pipe.close()
    return dt, osz, st, launches


DUMP_SAMPLE = 1 << 22  # decoded bytes kept by --dump-outputs: 16 MiB as float32
DUMP_SEED = 20240601


def dump_outputs(out_dir, torch, d_out, d_out_size, d_status, n, size, stride):
    """What a caller of the device-resident gzip path receives from one call, as float arrays: every member's status
    and output size, and the decoded bytes at a fixed, seeded sample of positions of the n x `size` payloads (the whole
    output is n x 1 MiB). The positions are written too, so that two dumps can be compared position by position."""
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(DUMP_SEED)
    pos = np.sort(rng.choice(n * size, size=min(DUMP_SAMPLE, n * size), replace=False)).astype(np.int64)
    flat = torch.from_numpy((pos // size) * stride + pos % size).to(d_out.device)
    arrays = {"status": d_status.cpu().numpy().astype(np.float64),
              "out_size": d_out_size.cpu().numpy().astype(np.float64),
              "payload_sample": d_out[flat].cpu().numpy().astype(np.float32),
              "payload_sample_pos": pos.astype(np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------- ours ---
def run_ours(args):
    import torch
    import torch.distributed as dist
    import debigulator_b200 as dbg
    from debigulator_b200.build import build_library, build_tools

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    build_library()
    build_tools()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    ctx = dbg.Context(local)
    n, size = args.members, MEMBER_BYTES
    tstream = torch.cuda.Stream(device=dev)  # a real (non-default) stream: kernels, events and checks all live on it
    torch.cuda.set_stream(tstream)

    # ---- corpus: N_UNIQUE distinct members (16 per class), cycled to n, every copy at its own address
    uniq = make_unique(_gen_gz, N_UNIQUE) if (rank == 0 or world == 1) else None
    if world > 1:
        box = [uniq]
        dist.broadcast_object_list(box, src=0)
        uniq = box[0]
    offs, sizes, in_total = pack([u[0] for u in uniq], n)
    h_in = torch.empty(in_total + 64, dtype=torch.uint8).pin_memory()
    h_in.zero_()
    hv = h_in.numpy()
    for i in range(n):
        b = uniq[i % N_UNIQUE][0]
        hv[offs[i]:offs[i] + len(b)] = np.frombuffer(b, np.uint8)
    # inflate() requires recipient_size >= compressed_input_size (inflate.c:826); stored members are
    # slightly larger than their payload, so every output slot carries 4 KiB of slack
    stride = size + 4096
    out_total = n * size
    out_span = n * stride
    h_out = torch.empty(out_span, dtype=torch.uint8).pin_memory()
    in_off = np.array(offs, dtype=np.uint64)
    in_size = np.array(sizes, dtype=np.uint64)
    out_off = (np.arange(n, dtype=np.uint64) * np.uint64(stride))
    out_cap = np.full(n, stride, dtype=np.uint64)
    comp_bytes = int(in_size.sum())

    d_in = h_in.to(dev, non_blocking=False)
    d_out = torch.zeros(out_span, dtype=torch.uint8, device=dev)
    t_i64 = lambda a: torch.from_numpy(a.view(np.int64)).to(dev)
    d_in_off, d_in_size, d_out_off, d_out_cap = t_i64(in_off), t_i64(in_size), t_i64(out_off), t_i64(out_cap)
    d_out_size = torch.zeros(n, dtype=torch.int64, device=dev)
    d_status = torch.zeros(n, dtype=torch.int32, device=dev)
    # scheduling hint (any caller can compute it from the first deflate byte): longest-processing-time first,
    # where a member that starts with a stored block counts as 1/16 of its size
    first = np.array([uniq[i % N_UNIQUE][0][10] & 6 for i in range(n)])
    weight = np.where(first == 0, in_size // 16, in_size).astype(np.int64)
    order = np.argsort(-weight, kind="stable").astype(np.uint32)
    d_order = torch.from_numpy(order.view(np.int32)).to(dev)
    stream = torch.cuda.current_stream().cuda_stream

    def step_device():
        ctx.inflate_device(d_in, d_in_off, d_in_size, d_out, d_out_off, d_out_cap, d_out_size, d_status, d_order,
                           stream=stream, gz=True)

    def verify():
        torch.cuda.synchronize()
        bad = torch.nonzero(d_status).flatten()
        assert bad.numel() == 0, f"device decode reported failures: {[(int(i), int(d_status[i])) for i in bad[:8]]}"
        assert bool((d_out_size == size).all().item()), "wrong output sizes"
        exp = torch.stack([torch.from_numpy(np.frombuffer(u[1], np.uint8).copy()) for u in uniq]).to(dev)
        got = d_out.view(n, stride)
        idx = torch.arange(n, device=dev) % N_UNIQUE
        for s in range(0, n, 256):
            assert torch.equal(got[s:s + 256, :size], exp[idx[s:s + 256]]), "payload mismatch"

    # ---- device-resident timing
    for _ in range(args.warmup):
        step_device()
    barrier()
    if args.warmup:
        verify()
    d_out.zero_()
    launches0 = ctx.kernel_launches
    ctx.profile_enable(True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        step_device()
    ev1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    dev_ms = max_over_ranks(ev0.elapsed_time(ev1))
    kern_ms, kern_n = ctx.profile_read()
    ctx.profile_enable(False)
    launches = ctx.kernel_launches - launches0
    verify()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch, d_out, d_out_size, d_status, n, size, stride)
    value = world * n * size * args.steps / (dev_ms / 1e3) / 1e9

    # ---- end to end through the packed host API (pinned host arenas)
    hin_np, hout_np = h_in.numpy(), h_out.numpy()
    ctx.decode_packed(dbg.api.KIND_GZ, hin_np, in_off, in_size, hout_np, out_off, out_cap)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        osz, st = ctx.decode_packed(dbg.api.KIND_GZ, hin_np, in_off, in_size, hout_np, out_off, out_cap)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    assert int(st.sum()) == 0 and int(osz.sum()) == out_total
    for k in (0, 1, 2, 3, n - 1):
        assert hout_np[k * stride:k * stride + size].tobytes() == uniq[k % N_UNIQUE][1], "e2e payload mismatch"
    e2e_single = world * out_total * args.steps / e2e_s / 1e9
    # the same with two calls in flight (dbg_pipe_*: the batch as two sub-batches, one's ramp under the other's downloads)
    ctx.trim()
    hout_np[:] = 0
    pdt, osz, st, pipe_launches = e2e_pipelined(dbg, local, dbg.api.KIND_GZ, hin_np, in_off, in_size, hout_np, out_off, out_cap,
                                                args.steps, barrier, max_over_ranks)
    assert int(st.sum()) == 0 and int(osz.sum()) == out_total
    for k in (0, 1, 2, 3, n // 2 - 1, n // 2, n - 1):
        assert hout_np[k * stride:k * stride + size].tobytes() == uniq[k % N_UNIQUE][1], "pipelined e2e payload mismatch"
    e2e_val = world * out_total / pdt / 1e9
    # the link ceiling of that path: the same pinned arenas copied H2D and D2H at once, nothing else running -- on
    # every rank at the same time, so that at N > 1 it is the box's ceiling (host memory / PCIe fabric), not one link's
    s_up, s_dn = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    barrier()
    t0 = time.perf_counter()
    for _ in range(2):
        with torch.cuda.stream(s_up):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s_dn):
            h_out.copy_(d_out, non_blocking=True)
    torch.cuda.synchronize()
    own_dt = (time.perf_counter() - t0) / 2
    dt = max_over_ranks(own_dt)
    pcie = {"h2d_plus_d2h_s": dt, "output_GBps_if_copies_only": world * out_total / dt / 1e9, "ranks_copying_at_once": world,
            "per_rank_h2d_GBps": in_total / dt / 1e9, "per_rank_d2h_GBps": out_span / dt / 1e9,
            "e2e_frac_of_ceiling": (e2e_val / (world * out_total / dt / 1e9)),
            "single_call_frac_of_ceiling": (e2e_single / (world * out_total / dt / 1e9))}
    del h_out, hout_np
    torch.cuda.empty_cache()

    # ---- PNG half of the metric: BASELINE config 3 (every rank its own batch) and config 4
    png = png_large = None
    if args.png:
        uniq3 = png_corpus(PNG_W, PNG_H, PNG_UNIQUE, None, "cfg3" if world > 1 else None, rank, world, barrier)
        # the end-to-end leg pins ~7.5 MB of host memory per image and rank: all images when the box has room for every
        # rank's arenas, else half / a quarter of the batch (rank 0 decides for everybody)
        e2e_n = args.png_images
        if world > 1:
            box = [None]
            if rank == 0:
                import psutil
                avail = psutil.virtual_memory().available * 0.7
                per_image = 4 * PNG_W * PNG_H * 1.85
                while e2e_n > 256 and world * e2e_n * per_image > avail:
                    e2e_n //= 2
                box = [e2e_n]
            dist.broadcast_object_list(box, src=0)
            e2e_n = box[0]
        png = bench_png(ctx, dbg, dev, torch, "cfg3", args.png_images, PNG_W, PNG_H, uniq3, peak, args.steps, e2e=True,
                        cpu=(rank == 0 and world == 1 and not args.no_cpu), world=world, max_over_ranks=max_over_ranks, barrier=barrier,
                        e2e_images=e2e_n)
        del uniq3
    if args.png_large:
        uniq4 = png_corpus(PNG4_W, PNG4_H, min(PNG4_UNIQUE, args.png_large), 4, "cfg4" if world > 1 else None, rank, world, barrier)
        ctx.trim()
        torch.cuda.empty_cache()
        png_large = bench_png(ctx, dbg, dev, torch, "cfg4 (forced Paeth)", args.png_large, PNG4_W, PNG4_H, uniq4, peak, args.steps, e2e=(world == 1),
                              cpu=(rank == 0 and world == 1 and not args.no_cpu), world=world, max_over_ranks=max_over_ranks, barrier=barrier)
        del uniq4
        ctx.trim()
        torch.cuda.empty_cache()
    bmp = cfg5 = cfg1 = None
    if args.bmp and rank == 0 and world == 1:
        bmp = bench_bmp(ctx, dev, torch, args.bmp, args.steps)
        bmp["sprite_sheet"] = bench_sprites(ctx, dev, torch, args.steps)
    if args.cfg5 and rank == 0 and world == 1:
        cfg5 = bench_cfg5(ctx, dev, torch, args.cfg5, args.steps)
    if args.cfg1 and rank == 0 and world == 1:
        cfg1 = bench_cfg1(ctx, args.steps, no_cpu=args.no_cpu)

    # ---- CPU baseline: the reference C on this box's host cores (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import checker
        cores = host_cores()
        per = cores * 32
        blobs = [uniq[i % N_UNIQUE][0] for i in range(per)]
        caps = [size + len(b) for b in blobs]
        b1, s1 = cpu_throughput("gz", blobs[:32], caps[:32], 1, steps=1, warmup=1)
        bn, sn = cpu_throughput("gz", blobs, caps, cores, steps=3, warmup=1)
        v1, vn = b1 / s1[0] / 1e9, bn * 3 / sum(sn) / 1e9
        cpu = {"value": vn, "unit": UNIT, "cores": cores, "kind": checker.kind(),
               "sample": f"{per} of {n} members per pass ({per} MiB out), 3 passes, one process per core, setup outside the clock",
               "single_thread": {"value": v1, "unit": UNIT, "sample": "32 members (8 per class)"},
               "parallel_efficiency": vn / (v1 * cores)}

    if rank == 0:
        alg_bytes = comp_bytes + out_total  # C + U per launch (SURVEY.md 8d)
        # dram read + write of one inflate launch from the committed `ncu --set full` capture; reported only while the
        # kernel's sources still hash to what was captured (scripts/make_traffic_json.py)
        traffic, traffic_src = None, None
        try:
            sys.path.insert(0, os.path.join(ROOT, "scripts"))
            from make_traffic_json import kernel_hash
            tj = json.load(open(os.path.join(ROOT, "profiles", "r02", "inflate_traffic.json")))
            if n != N_MEMBERS or int(tj["algorithmic_bytes_per_launch"]) != int(alg_bytes):
                traffic_src = "no capture of this workload"
            elif tj["kernel_sources_sha256_16"] != kernel_hash():
                traffic_src = "stale: kernel sources changed since profiles/r02/inflate_traffic.json was captured"
            else:
                traffic = float(tj["traffic_bytes_per_launch"])
                traffic_src = "profiles/r02/inflate_traffic.json (ncu --set full; kernel source hash %s matches)" % tj["kernel_sources_sha256_16"]
        except Exception as e:
            traffic_src = "unavailable: %r" % (e,)
        avg_kern_ms = kern_ms / max(kern_n, 1)
        achieved = alg_bytes / (avg_kern_ms / 1e3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": f"cfg2: {n} x 1 MiB gzip members per GPU (stored/fixed/dynamic/mixed by i%4)",
                       "unique_members": N_UNIQUE, "compressed_bytes_per_gpu": comp_bytes, "output_bytes_per_gpu": out_total,
                       "l2": "inputs+outputs per step (%.1f GB) exceed the 126 MB L2; no explicit flush" % ((comp_bytes + out_total) / 1e9),
                       "parallelism": f"{world} independent shard(s), no collective"},
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(in_total + 64), "d2h_bytes_per_step": int(out_span),
                    "steps": args.steps, "ms_per_step": pdt * 1e3, "calls_in_flight": 2,
                    "api": "dbg_pipe_submit / dbg_pipe_wait (kind=gzip): every step's batch as two packed sub-batches of the same "
                           "pinned host arenas, two in flight",
                    "single_call": {"value": e2e_single, "unit": UNIT, "ms_per_step": e2e_s / args.steps * 1e3, "steps": args.steps,
                                    "api": "dbg_decode_batch_packed(kind=gzip), one blocking call per step"},
                    "kernel_launches_per_step": pipe_launches,
                    "link_ceiling": pcie},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "inflate_batch_kernel", "avg_launch_ms": avg_kern_ms, "launches": kern_n,
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s"},
            "cpu_baseline": cpu, "clocks": clocks,
        }
        if png:
            line["png"] = png
        if png_large:
            line["png_cfg4"] = png_large
        if cfg5:
            line["cfg5_shape"] = cfg5
        if cfg1:
            line["cfg1"] = cfg1
        if bmp:
            bmp["roofline"]["peak"] = peak
            bmp["roofline"]["frac"] = bmp["roofline"]["achieved"] / peak
            bmp["sprite_sheet"]["roofline"]["peak"] = peak
            bmp["sprite_sheet"]["roofline"]["frac"] = bmp["sprite_sheet"]["roofline"]["achieved"] / peak
            line["bmp"] = bmp
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def bench_cfg1(ctx, steps, no_cpu=False):
    """BASELINE config 1: the two bundled files as batches of one through the scalar-sized path (wall clock,
    host buffers in, host buffers out), next to the reference C on one core."""
    gold = os.path.join(ROOT, "tests", "golden")
    png = open(os.path.join(gold, "gimp_test.png"), "rb").read()
    gz = open(os.path.join(gold, "gzipsample.gz"), "rb").read()
    out = {}
    for name, fn in (("gimp_test.png", lambda: ctx.decode_png_batch([png])), ("gzipsample.gz", lambda: ctx.decode_gz_batch([gz], [600000]))):
        for _ in range(3):
            r = fn()
        assert r[0][0] == 1
        ts = []
        for _ in range(steps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        out[name] = {"gpu_ms_median": float(np.median(ts)) * 1e3, "gpu_ms_best": min(ts) * 1e3}
    if not no_cpu:
        from oracle import checker
        for name, what, blob, cap in (("gimp_test.png", "png", png, 1024 * 1024 * 4), ("gzipsample.gz", "gz", gz, 600000)):
            r = checker.TimedRunner(what, [blob], [cap])
            r.run()
            out[name]["reference_ms_one_core"] = min(r.run()[0] for _ in range(5)) * 1e3
    out["note"] = "batch of one: dbg_decode_png_batch / dbg_decode_gz_batch with n = 1, pageable host buffers, wall clock"
    return out


def _gen_cfg5(i):
    from debigulator_b200 import corpus
    size = int(65536 * (256.0 ** (((i * 2654435761) % 1000) / 999.0)))  # log-uniform in [64 KiB, 16 MiB]
    g, d = corpus.gz_member_cfg5(i, size)
    return g, len(d), zlib.crc32(d)


def bench_cfg5(ctx, dev, torch, n, steps, n_unique=64):
    """BASELINE config 5 shape, scaled to one GPU: gzip members of 64 KiB-16 MiB (log-uniform), eight
    compressibility classes, device-resident. The long members take the block-split path (DESIGN.md 4.3)."""
    uniq = pool_map(_gen_cfg5, list(range(n_unique)))
    offs, sizes, caps, total = [], [], [], 0
    for i in range(n):
        g, m, _ = uniq[i % n_unique]
        offs.append(total)
        sizes.append(len(g))
        caps.append((m + len(g) + 64 + 15) // 16 * 16)
        total += (len(g) + 31) // 16 * 16
    h = np.zeros(total + 64, np.uint8)
    for i in range(n):
        g = uniq[i % n_unique][0]
        h[offs[i]:offs[i] + len(g)] = np.frombuffer(g, np.uint8)
    out_off = np.concatenate([[0], np.cumsum(caps[:-1])]).astype(np.uint64)
    i64 = lambda a: torch.from_numpy(np.asarray(a, np.uint64).view(np.int64)).to(dev)
    d_in = torch.from_numpy(h).to(dev)
    d_out = torch.zeros(int(sum(caps)), dtype=torch.uint8, device=dev)
    d_size = torch.zeros(n, dtype=torch.int64, device=dev)
    d_st = torch.zeros(n, dtype=torch.int32, device=dev)
    a_off, a_sz, o_off, o_cap = i64(offs), i64(sizes), i64(out_off), i64(caps)
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        ctx.inflate_device(d_in, a_off, a_sz, d_out, o_off, o_cap, d_size, d_st, None, stream=stream, gz=True)

    before = ctx.bsplit_stats()
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    assert int(d_st.abs().sum().item()) == 0, "cfg5 decode failures"
    got = d_size.cpu().numpy()
    # every unique member whose size is the spec's (the reference's rule Q2 cuts some low-entropy members short;
    # tests/test_gpu_parity.py compares those with the reference): CRC-32 of the decoded payload against the source's
    checked = 0
    for k in range(min(n, n_unique)):
        if int(got[k]) == uniq[k][1]:
            data = d_out[int(out_off[k]):int(out_off[k]) + int(got[k])].cpu().numpy().tobytes()
            assert zlib.crc32(data) == uniq[k][2], f"cfg5 payload mismatch in member {k}"
            checked += 1
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    after = ctx.bsplit_stats()
    out_bytes = int(got.sum())
    return {"metric": "inflate_output_GBps", "value": out_bytes / ms / 1e6, "unit": "GB/s", "ms_per_step": ms,
            "config": {"workload": f"cfg5 shape: {n} gzip members, 64 KiB-16 MiB log-uniform, 8 compressibility classes "
                                   "(stored / text / Huffman-only / period ~32 kB / runs / zeros)",
                       "unique_members": n_unique, "output_bytes": out_bytes, "compressed_bytes": int(sum(sizes)),
                       "members_with_spec_size": int(sum(int(got[i]) == uniq[i % n_unique][1] for i in range(n))),
                       "unique_members_crc_checked": checked},
            "block_split_streams_per_step": (after[0] - before[0]) // (steps + 2), "block_split_fallbacks": after[1] - before[1]}


def bench_bmp(ctx, dev, torch, n, steps, w=2048, h=2048):
    """decode_BMP / encode_BMP on n bottom-up w x h files (SURVEY.md 8(f) rank 4): the one kernel of the
    library that is plain HBM traffic (every pixel read once, written once)."""
    from debigulator_b200 import corpus
    rng = np.random.default_rng(7)
    rgba = rng.integers(0, 256, w * h * 4, dtype=np.uint8).tobytes()
    file = corpus.bmp_file(rgba, w, h, bottom_up=True)
    fsz, osz = len(file), w * h * 4
    stride = (fsz + 255) // 256 * 256
    one = torch.from_numpy(np.frombuffer(file + bytes(stride - fsz), np.uint8).copy()).to(dev)
    d_in = one.repeat(n)
    d_out = torch.zeros(n * osz, dtype=torch.uint8, device=dev)
    i64 = lambda a: torch.from_numpy(np.asarray(a, dtype=np.uint64).view(np.int64)).to(dev)
    in_off, in_size = i64(np.arange(n, dtype=np.uint64) * np.uint64(stride)), i64(np.full(n, fsz, dtype=np.uint64))
    out_off, out_cap = i64(np.arange(n, dtype=np.uint64) * np.uint64(osz)), i64(np.full(n, osz, dtype=np.uint64))
    out_size = torch.zeros(n, dtype=torch.int64, device=dev)
    st = torch.zeros(n, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    # encode target: the decoded images back into BMP files
    estride = (54 + osz + 1 + 255) // 256 * 256
    d_enc = torch.zeros(n * estride, dtype=torch.uint8, device=dev)
    e_off, e_cap = i64(np.arange(n, dtype=np.uint64) * np.uint64(estride)), i64(np.full(n, estride, dtype=np.uint64))
    e_size = torch.zeros(n, dtype=torch.int64, device=dev)
    e_st = torch.zeros(n, dtype=torch.int32, device=dev)
    wd = torch.full((n,), w, dtype=torch.int32, device=dev)
    ht = torch.full((n,), h, dtype=torch.int32, device=dev)

    def dec():
        ctx.bmp_decode_device(d_in, in_off, in_size, d_out, out_off, out_cap, out_size, st, stream=stream)

    def enc():
        ctx.bmp_encode_device(d_out, out_off, out_cap, wd, ht, d_enc, e_off, e_cap, e_size, e_st, stream=stream)

    res = {}
    for name, fn in (("decode", dec), ("encode", enc)):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        res[name] = e0.elapsed_time(e1) / steps
    assert int(st.abs().sum().item()) == 0 and int(e_st.abs().sum().item()) == 0, "bmp failures"
    exp = torch.from_numpy(np.frombuffer(rgba, np.uint8).copy()).to(dev)
    assert torch.equal(d_out.view(n, osz)[0], exp) and torch.equal(d_out.view(n, osz)[n - 1], exp), "bmp pixel mismatch"
    # the encoder's output is checked without the oracle (bench.py may only time it, in the CPU legs): 54 header
    # bytes as decode_bmp.c:313-358 writes them, then the pixels as BGRA, and 54 + size + 1 reported
    import struct
    size = 54 + osz + 1
    got = d_enc.view(n, estride)[n - 1][: size - 1].cpu().numpy().tobytes()
    hdr = b"BM" + struct.pack("<IHHI", (w * h * 4 + 54) & 0xffffffff, 0, 0, 54) + struct.pack(
        "<IiiHHIIIIII", 40, w, -h, 1, 32, 0, w * h * 4, 0, 0, 0, 0)
    bgra = np.frombuffer(rgba, np.uint8).reshape(-1, 4)[:, [2, 1, 0, 3]].tobytes()
    assert got == hdr + bgra and int(e_size[0].item()) == size, "bmp encode mismatch"
    alg = 2 * n * osz  # pixels read once + written once
    ach = alg / (res["decode"] / 1e3) / 1e9
    return {"metric": "bmp_decode_Mpixels_per_s", "value": n * w * h / (res["decode"] / 1e3) / 1e6, "unit": "Mpix/s",
            "ms_per_step": res["decode"], "encode_Mpixels_per_s": n * w * h / (res["encode"] / 1e3) / 1e6,
            "encode_ms_per_step": res["encode"],
            "config": {"workload": f"{n} x {w}x{h} 32-bit bottom-up BMP files (rows flipped), then re-encoded", "unique_images": 1},
            "roofline": {"bound": "hbm", "achieved": ach, "unit": "GB/s", "kernel": "bmp_swizzle_kernel",
                         "algorithmic_bytes_per_launch": alg, "encode_achieved": alg / (res["encode"] / 1e3) / 1e9}}


def bench_sprites(ctx, dev, torch, steps, n=1000, w=512, h=512):
    """Sprite-sheet tiling (SURVEY.md 8(f) rank 4, intent of concat_pngs.c:81-100): n decoded w x h RGBA8 images into one
    sheet of ceil(sqrt(n)) columns; plain HBM traffic (every image pixel read once, every sheet pixel written once)."""
    rgba = w * h * 4
    g = torch.Generator(device=dev)
    g.manual_seed(5)
    d_img = torch.randint(0, 256, (n * rgba,), dtype=torch.uint8, device=dev, generator=g)
    off = torch.arange(n, dtype=torch.int64, device=dev) * rgba
    cols = next(c for c in range(1, n + 2) if c * c >= n)
    rows = (n + cols - 1) // cols
    d_sheet = torch.zeros(cols * w * rows * h * 4, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    for _ in range(3):
        r, c = ctx.tile_sprites_device(d_img, off, n, w, h, 0, True, d_sheet, stream=stream)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        ctx.tile_sprites_device(d_img, off, n, w, h, 0, True, d_sheet, stream=stream)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    sheet = d_sheet.view(rows * h, cols * w * 4)
    for i in (0, 1, cols, n - 1):  # spot check: tile i against its image
        rr, cc = divmod(i, cols)
        tile = sheet[rr * h:(rr + 1) * h, cc * w * 4:(cc + 1) * w * 4]
        assert torch.equal(tile.reshape(-1), d_img[i * rgba:(i + 1) * rgba]), "sprite sheet mismatch"
    assert (r, c) == (rows, cols)
    alg = n * rgba + d_sheet.numel()
    return {"metric": "sprite_sheet_Mpixels_per_s", "value": n * w * h / (ms / 1e3) / 1e6, "unit": "Mpix/s", "ms_per_step": ms,
            "config": {"workload": f"{n} x {w}x{h} RGBA8 images into one {cols} x {rows} sheet, device-resident"},
            "roofline": {"bound": "hbm", "achieved": alg / (ms / 1e3) / 1e9, "unit": "GB/s", "kernel": "sprite_tile_kernel",
                         "algorithmic_bytes_per_launch": alg}}


# -------------------------------------------------------------------- strong ----
def run_strong(args):
    """ONE batch over N GPUs of the box through dbg_decode_batch_packed_multi (one process, one host thread and one
    stream set per device): BASELINE config 4 as stated (256 x 8192^2 at N = 8; 32 x N images otherwise unless
    --images says so) or config 5 (2048 x N members). Host arenas in, host arenas out; wall clock."""
    import torch
    import debigulator_b200 as dbg
    from debigulator_b200.build import build_library, build_tools
    build_library()
    build_tools()
    ngpu = args.gpus
    m = dbg.MultiContext(ngpu)
    if args.strong == "cfg4":
        n = args.images or 32 * ngpu  # 256 at N = 8, as BASELINE config 4 states it
        uniq = pool_map(_gen_png, [(i, PNG4_W, PNG4_H, 4) for i in range(min(PNG4_UNIQUE, n))])
        kind, w, h = dbg.api.KIND_PNG, PNG4_W, PNG4_H
        caps = [w * h * 4] * n
        unit, per_item = "Mpix/s", w * h / 1e6
        name = f"cfg4: {n} x {w}x{h} RGBA8 PNGs (stb_write, forced Paeth), one batch"
    else:
        n = args.images or 2048 * ngpu  # 16,384 at N = 8
        uniq = [(g, None) for g, _, _ in pool_map(_gen_cfg5, list(range(64)))]
        sizes_out = [int(65536 * (256.0 ** (((i * 2654435761) % 1000) / 999.0))) for i in range(64)]
        kind = dbg.api.KIND_GZ
        caps = [(sizes_out[i % 64] + len(uniq[i % 64][0]) + 64 + 15) // 16 * 16 for i in range(n)]
        unit, per_item = "GB/s", None
        name = f"cfg5: {n} gzip members 64 KiB-16 MiB, one batch"
    offs, sizes, in_total = pack([u[0] for u in uniq], n)
    h_in_t = torch.empty(in_total + 64, dtype=torch.uint8).pin_memory()
    h_in = h_in_t.numpy()
    h_in[:] = 0
    for i in range(n):
        b = uniq[i % len(uniq)][0]
        h_in[offs[i]:offs[i] + len(b)] = np.frombuffer(b, np.uint8)
    out_off = np.concatenate([[0], np.cumsum(caps[:-1])]).astype(np.uint64)
    h_out_t = torch.empty(int(sum(caps)) + 64, dtype=torch.uint8).pin_memory()
    h_out = h_out_t.numpy()
    in_off, in_size, out_cap = np.asarray(offs, np.uint64), np.asarray(sizes, np.uint64), np.asarray(caps, np.uint64)
    res = []
    for rep in range(1 + args.steps):
        t0 = time.perf_counter()
        osz, st, devs = m.decode_packed(kind, h_in, in_off, in_size, h_out, out_off, out_cap)
        res.append(time.perf_counter() - t0)
    assert int(st.sum()) == 0, "strong-scaling batch: decode failures"
    if kind == dbg.api.KIND_PNG:
        for k in (0, 1, n // 2, n - 1):
            o = int(out_off[k])
            assert h_out[o:o + caps[k]].tobytes() == uniq[k % len(uniq)][1], "pixel mismatch"
        total_units = n * per_item
    else:
        total_units = float(osz.sum()) / 1e9
    dt = float(np.median(res[1:]))
    print(json.dumps({"metric": "png_decode_Mpixels_per_s" if kind == dbg.api.KIND_PNG else METRIC, "value": total_units / dt, "unit": unit,
                      "n_gpus": ngpu, "steps": args.steps, "warmup": 1, "ms_per_step": dt * 1e3, "higher_is_better": True,
                      "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "impl": "ours",
                      "config": {"workload": name, "unique_items": len(uniq), "api": "dbg_decode_batch_packed_multi, pinned host arenas, wall clock",
                                 "items_per_device": [int((devs == d).sum()) for d in range(ngpu)],
                                 "h2d_bytes_per_step": int(in_total), "d2h_bytes_per_step": int(sum(caps))},
                      "e2e": {"value": total_units / dt, "unit": unit, "h2d_bytes_per_step": int(in_total), "d2h_bytes_per_step": int(sum(caps))}}))
    m.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed steps of every GPU measurement (device-resident, end-to-end, secondary lines)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--members", type=int, default=N_MEMBERS)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--png", type=int, default=1)
    ap.add_argument("--png-images", type=int, default=PNG_N)
    ap.add_argument("--png-large", type=int, default=PNG4_N, help="8192x8192 images per GPU in the config-4 line (0 = skip)")
    ap.add_argument("--cfg5", type=int, default=2048, help="members of the config-5-shape line (0 = skip)")
    ap.add_argument("--cfg1", type=int, default=1, help="batch-of-one latency of the two bundled files (0 = skip)")
    ap.add_argument("--bmp", type=int, default=64, help="number of 2048x2048 BMP files in the BMP line (0 = skip)")
    ap.add_argument("--strong", default=None, choices=["cfg4", "cfg5"], help="one batch over --gpus devices (dbg_multi_*)")
    ap.add_argument("--images", type=int, default=0, help="--strong: items in the batch")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step of the headline workload returned to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.strong):
        ap.error("--dump-outputs writes the outputs of the headline GPU workload: not with --impl reference or --strong")
    if args.impl == "reference":
        run_reference(args)
    elif args.strong:
        run_strong(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
