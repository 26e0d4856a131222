#!/usr/bin/env python
"""bench.py -- HIMG encode+decode throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[3] "batch of 4096 1920x1080 RGB images encode+decode
sharded across 1/2/4/8 B200" -- STRONG scaling: the job is always the 4096 images with seeds 1..4096 at
quality 50; rank r of N codes the contiguous shard of 4096/N images (all 4096 on one GPU at N=1).  A "step"
is one pass of the hot path over the rank's shard: encode every image to a .himg bitstream, then decode
every bitstream back to pixels.

Printed JSON (one line, rank 0):
  value        megapixels (W*H, channels not counted) through encode AND decode per second, whole job, inputs
               resident in HBM, CUDA events, max over ranks
  e2e          the same through the host-buffer C-ABI calls (pinned host memory, H2D and D2H inside the timed
               region)
  roofline     K-fwd (k_forward: colour map + low-res subtract + WHT + quantise + map) and K-inv, algorithmic
               bytes = 2*nch per pixel, duration from CUDA events around every launch of the timed region,
               peak = MEASURED_PEAKS.json hbm_gbs
  parity_checked / multi_gpu_parity
               inside the run, before timing: every rank compares the FNV-1a-64 of the first and last
               bitstream and decoded image of its shard with the hashes recorded from the unmodified
               reference (tests/golden/golden_c4_shards.json); with N > 1 rank 0 additionally re-encodes a
               sample of every other rank's images on its own GPU and compares bitstreams byte for byte
  c2 / c3 / c5 sub-records of the other BASELINE.json configurations (N=1 only)
  cpu_baseline the unmodified reference (oracle/_ref) on the host cores, bounded sample

--dump-outputs DIR (e.g. bench_outputs) writes what the last timed step computed, see dump_outputs().
"""
from __future__ import annotations

import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, NCH, QUALITY = 1920, 1080, 3, 50
TOTAL_IMAGES = 4096
WORKLOAD = "c4: batch of 4096 1920x1080 RGB images (seeds 1..4096), quality 50, YCbCr, encode+decode, sharded by image"


# ------------------------------------------------------------------------------------------------
# CPU side: the reference's own implementation on the host cores (oracle/_ref, else the port)
# ------------------------------------------------------------------------------------------------
_CPU = {}


def _cpu_init(kind, w, h, nch, quality):
    """Pool initialiser: import the checker and keep the implementation around (outside the timed region)."""
    import oracle

    port = oracle.port()
    _CPU.update(port=port, impl=oracle.ref() if kind == "reference" else port, kind=kind, shape=(w, h, nch), quality=quality)


def _cpu_prepare(seeds):
    w, h, nch = _CPU["shape"]
    _CPU["images"] = [_CPU["port"].synth(w, h, nch, s, 6) for s in seeds]
    return len(seeds)


def _cpu_work(_):
    impl, kind, q = _CPU["impl"], _CPU["kind"], _CPU["quality"]
    t_enc = t_dec = 0.0
    for img in _CPU["images"]:
        t0 = time.perf_counter()
        packed = impl.encode(img, q, True)
        t1 = time.perf_counter()
        dec = impl.decode(packed, 1) if kind == "reference" else impl.decode(packed)
        t2 = time.perf_counter()
        assert dec is not None
        t_enc += t1 - t0
        t_dec += t2 - t1
    return t_enc, t_dec, len(_CPU["images"])


class CpuReference:
    """One reference Encoder/Decoder(1 thread) per host core over disjoint images (the reference encoder is
    single threaded, encoder.cpp:59-109).  The pool is forked and the images are synthesised BEFORE the
    timed region; only encode + decode are timed."""

    def __init__(self, images_per_core: int, shape=(W, H, NCH), quality=QUALITY):
        import multiprocessing as mp

        import oracle

        self.kind = "reference" if oracle.ref_available() else "port"
        self.cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        self.per = images_per_core
        self.shape = shape
        self.pool = mp.get_context("fork").Pool(self.cores, initializer=_cpu_init, initargs=(self.kind, *shape, quality))
        seeds = [[1 + c * images_per_core + i for i in range(images_per_core)] for c in range(self.cores)]
        # chunksize 1 + as many tasks as workers: every worker prepares (and later codes) its own images
        self.pool.map(_cpu_prepare, seeds, chunksize=1)

    def step(self):
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_work, range(self.cores), chunksize=1)
        wall = time.perf_counter() - t0
        n = sum(r[2] for r in res)
        mp_total = n * self.shape[0] * self.shape[1] / 1e6
        enc_core = mp_total / sum(r[0] for r in res)  # MP/s of one core while all cores are busy
        dec_core = mp_total / sum(r[1] for r in res)
        value = self.cores / (1.0 / enc_core + 1.0 / dec_core)
        sample = (f"{n} {self.shape[0]}x{self.shape[1]}x{self.shape[2]} q{QUALITY} images encode+decode, {self.per} per core on "
                  f"{self.cores} processes (pool and images prepared before timing); per-core encode {enc_core:.1f} MP/s, "
                  f"decode {dec_core:.1f} MP/s; value = cores / (1/enc + 1/dec); wall-clock {mp_total / wall:.1f} MP/s")
        return value, wall, sample

    def close(self):
        self.pool.close()
        self.pool.join()


# ------------------------------------------------------------------------------------------------
def start_clock_sampler(path):
    q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    try:
        return subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                stdout=open(path, "w"), stderr=subprocess.DEVNULL)
    except OSError:
        return None


def summarize_clocks(path, gpu_index):
    sm, mx, reasons = [], [], set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    try:
        for line in open(path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9 or not f[0].isdigit() or int(f[0]) != gpu_index:
                continue
            sm.append(float(f[1]))
            mx.append(float(f[2]))
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
    except (OSError, ValueError):
        pass
    if not sm:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
    # median over the busier half of the samples (= under load)
    busy = sorted(sm)[len(sm) // 2:]
    return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def load_golden():
    table = {}
    for name in ("golden_c4_shards.json", "golden_hashes.json"):
        try:
            for c in json.load(open(os.path.join(ROOT, "tests", "golden", name))):
                if (c["w"], c["h"], c["nch"], c["quality"], c.get("amp", 6), c.get("ycbcr", 1)) == (W, H, NCH, QUALITY, 6, 1) \
                        and c.get("pixel_hash"):
                    table[c["seed"]] = (c["himg_size"], c["himg_hash"], c["pixel_hash"])
        except (OSError, ValueError, KeyError):
            pass
    return table


def driver_times(args_list):
    """Min / average ms printed by the C++ `benchmark` driver (himg::Encoder / himg::Decoder, 30 iterations)."""
    exe = os.path.join(ROOT, "himg_b200", "_lib", "benchmark")
    try:
        out = subprocess.run([exe] + args_list, capture_output=True, text=True, timeout=300).stdout
        mn = re.search(r"Min: ([0-9.eE+-]+) ms", out)
        av = re.search(r"Average: ([0-9.eE+-]+) ms", out)
        return (float(mn.group(1)), float(av.group(1))) if mn and av else None
    except (OSError, subprocess.SubprocessError, ValueError):
        return None


DUMP_IMAGES = 8                # images of the shard whose outputs --dump-outputs writes
DUMP_PIXELS_PER_IMAGE = 1 << 19
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, first, out, sizes, table, decoded, status):
    """--dump-outputs: what the timed step returned in its last step, as float arrays, so that two builds can
    be compared output for output.  The whole size / offset table of the job and the decode status of every
    image of the shard; for a fixed, seeded sample of the shard's images (always its first and last) their
    whole bitstreams (-1 past the end) and their decoded pixels at a fixed, seeded set of positions (flat
    indices into H x W x NCH, the same in every image).  About 50 MB."""
    import numpy as np
    import torch

    B = sizes.numel()
    rng = np.random.default_rng(20261020)
    idx = sorted({0, B - 1} | {int(i) for i in rng.choice(B, min(B, DUMP_IMAGES - 2), replace=False)})
    pos = np.sort(rng.choice(H * W * NCH, min(H * W * NCH, DUMP_PIXELS_PER_IMAGE), replace=False))
    sizes_h = sizes.cpu().numpy()
    streams = np.full((len(idx), int(sizes_h[idx].max())), -1, np.float32)
    for k, i in enumerate(idx):
        streams[k, : sizes_h[i]] = out[i, : int(sizes_h[i])].cpu().numpy()
    sel = torch.tensor(idx, device=decoded.device)
    pixels = decoded[sel].reshape(len(idx), -1)[:, torch.from_numpy(pos).to(decoded.device)].cpu().numpy()
    arrays = {
        "sizes": table[0].cpu().numpy().astype(np.float64),
        "offsets": table[1].cpu().numpy().astype(np.float64),
        "status": status.cpu().numpy().astype(np.float64),
        "sample_images": np.asarray(idx, np.float64) + first,
        "sample_bitstreams": streams,
        "sample_pixel_positions": pos.astype(np.float64),
        "sample_pixels": pixels.astype(np.float32),
    }
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_LIMIT_BYTES
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--images", type=int, default=TOTAL_IMAGES, help="images of the whole job (strong scaling)")
    ap.add_argument("--e2e-images", type=int, default=512, help="images per GPU and step of the host-buffer leg (at most the shard)")
    ap.add_argument("--cpu-images-per-core", type=int, default=24)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-subrecords", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    # ---- reference arm: the reference's CPU implementation, rank 0 only --------------------------
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of --impl b200")
        if rank != 0:
            return 0
        per = max(1, min(args.cpu_images_per_core, 12))  # bounded sample per step
        cpu = CpuReference(per)
        for _ in range(args.warmup):
            cpu.step()
        vals, t0 = [], time.perf_counter()
        for _ in range(args.steps):
            vals.append(cpu.step())
        wall = time.perf_counter() - t0
        cpu.close()
        mps = sum(v[0] for v in vals) / len(vals)
        sample = vals[-1][2]
        print(json.dumps({
            "impl": "reference", "metric": "encode+decode megapixels/sec", "value": mps, "unit": "MP/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": wall / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "int16", "data": "synthetic",
            "config": {"workload": WORKLOAD, "quality": QUALITY, "sample_images_per_step": per * cpu.cores,
                       "same_config": False,
                       "note": "the CPU arm codes a bounded sample of the same image stream (seeds 1..), not all 4096 images"},
            "cpu_baseline": {"value": mps, "unit": "MP/s", "cores": cpu.cores, "kind": cpu.kind, "sample": sample},
            "e2e": {"value": mps, "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return 0

    # ---- CPU baseline first (fork before CUDA is initialised), rank 0 at N=1 only ---------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = CpuReference(max(1, args.cpu_images_per_core))
        cpu.step()  # warm-up pass (page faults, frequency ramp)
        value, wall, sample = cpu.step()
        cpu.close()
        cpu_baseline = {"value": value, "unit": "MP/s", "cores": cpu.cores, "kind": cpu.kind, "sample": sample,
                        "same_config": False}

    import numpy as np
    import torch
    import torch.distributed as dist

    import himg_b200
    from himg_b200 import sharding
    from himg_b200.synth import synth_images

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ctx = himg_b200.Context(local_rank)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream)
    # one launch of every kernel per step even for the 4096-image shard of N=1 (the default workspace limit
    # of 24 GB would split it into two sub-batches): the roofline figures are per launch
    ctx.set_option("max_workspace_bytes", 48 << 30)

    total_images = args.images
    first, B = sharding.shard_range(total_images, world, rank)  # contiguous image ranges per GPU
    pixels = synth_images(B, W, H, NCH, seed0=1 + first, amp=6, device=dev)
    out, sizes = ctx.encode_batch(pixels, QUALITY, True)
    offsets = torch.arange(B, dtype=torch.int64, device=dev) * out.stride(0)
    decoded, status = ctx.decode_batch(out.reshape(-1), offsets, sizes, W, H, NCH)
    torch.cuda.synchronize()
    ctx.encode_status()
    assert int(status.abs().sum()) == 0 and int((sizes == 0).sum()) == 0

    # ---- parity inside the run: recorded reference hashes of the shard's first and last image -----
    golden = load_golden()
    sizes_h = sizes.cpu().numpy()
    checked = []
    for i in sorted({0, B - 1}):
        seed = 1 + first + i
        if seed not in golden:
            continue
        want_size, want_himg, want_px = golden[seed]
        got = out[i, : int(sizes_h[i])].cpu().numpy()
        assert got.size == want_size, f"image seed {seed}: bitstream size {got.size}, reference {want_size}"
        assert f"{himg_b200.fnv1a64(got):016x}" == want_himg, f"image seed {seed}: bitstream differs from the reference"
        assert f"{himg_b200.fnv1a64(decoded[i].cpu().numpy()):016x}" == want_px, f"image seed {seed}: decoded pixels differ from the reference"
        checked.append(seed)
    parity_local = len(checked)

    # ---- multi-GPU parity: rank 0 re-encodes a sample of every rank's images on its own GPU --------
    multi_gpu_parity = "n/a (1 GPU)"
    if world > 1:
        sample_idx = sorted({0, B // 2, B - 1})
        smax = int(sizes_h.max())
        pack = torch.zeros((len(sample_idx), smax), dtype=torch.uint8, device=dev)
        meta = torch.zeros((len(sample_idx), 3), dtype=torch.int64, device=dev)  # seed, size, pixel hash
        for k, i in enumerate(sample_idx):
            pack[k, : int(sizes_h[i])] = out[i, : int(sizes_h[i])]
            ph = himg_b200.fnv1a64(decoded[i].cpu().numpy())
            meta[k] = torch.tensor([1 + first + i, int(sizes_h[i]), ph - (1 << 64) if ph >= (1 << 63) else ph], dtype=torch.int64)
        smax_t = torch.tensor([smax], dtype=torch.int64, device=dev)
        dist.all_reduce(smax_t, op=dist.ReduceOp.MAX)
        wide = torch.zeros((len(sample_idx), int(smax_t.item())), dtype=torch.uint8, device=dev)
        wide[:, :smax] = pack
        all_pack = [torch.zeros_like(wide) for _ in range(world)]
        all_meta = [torch.zeros_like(meta) for _ in range(world)]
        dist.all_gather(all_pack, wide)
        dist.all_gather(all_meta, meta)
        if rank == 0:
            bad = []
            for r in range(world):
                for k in range(len(sample_idx)):
                    seed, size, ph = (int(x) for x in all_meta[r][k].tolist())
                    img = synth_images(1, W, H, NCH, seed0=seed, amp=6, device=dev)
                    o1, s1 = ctx.encode_batch(img, QUALITY, True)
                    d1, st1 = ctx.decode_batch(o1.reshape(-1), torch.zeros(1, dtype=torch.int64, device=dev), s1, W, H, NCH)
                    torch.cuda.synchronize()
                    same = int(s1[0]) == size and torch.equal(o1[0, :size], all_pack[r][k, :size]) and int(st1[0]) == 0
                    ph1 = himg_b200.fnv1a64(d1[0].cpu().numpy())
                    same = same and (ph1 - (1 << 64) if ph1 >= (1 << 63) else ph1) == ph
                    if not same:
                        bad.append((r, seed))
            multi_gpu_parity = "ok" if not bad else f"MISMATCH {bad}"
            assert not bad, f"multi-GPU parity: {bad}"
        pc = torch.tensor([parity_local], dtype=torch.int64, device=dev)
        dist.all_reduce(pc, op=dist.ReduceOp.SUM)
        parity_total = int(pc.item())
        del all_pack, wide, pack
    else:
        parity_total = parity_local

    def step():
        ctx.encode_batch(pixels, QUALITY, True, out=out, sizes=sizes)
        # the only collective of the job: per-image bitstream sizes -> global offset table
        table = sharding.gather_sizes(sizes, world)
        ctx.decode_batch(out.reshape(-1), offsets, sizes, W, H, NCH, out=decoded, status=status)
        return table

    for _ in range(warmup):
        step()
    barrier()

    clk_path = os.path.join(tempfile.gettempdir(), f"himg_clocks_{os.getpid()}.csv")
    sampler = start_clock_sampler(clk_path) if rank == 0 else None
    ctx.profile(True)
    ctx.profile_reset()
    launches0 = ctx.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    barrier()
    ev[0].record(stream)
    for _ in range(args.steps):
        table = step()
    ev[1].record(stream)
    barrier()
    ms = ev[0].elapsed_time(ev[1])
    launches = ctx.launch_count() - launches0
    prof = ctx.profile_results()
    ctx.profile(False)
    ctx.encode_status()
    assert int(status.abs().sum()) == 0 and int(table[0].numel()) == total_images
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, first, out, sizes, table, decoded, status)

    # encode-only / decode-only splits (device resident), same timing discipline
    def timed(fn, reps):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(reps):
            fn()
        b.record(stream)
        barrier()
        return a.elapsed_time(b) / reps

    enc_ms = timed(lambda: ctx.encode_batch(pixels, QUALITY, True, out=out, sizes=sizes), max(2, args.steps // 2))
    dec_ms = timed(lambda: ctx.decode_batch(out.reshape(-1), offsets, sizes, W, H, NCH, out=decoded, status=status),
                   max(2, args.steps // 2))

    # ---- e2e: host buffers through the C ABI, H2D/D2H inside the timed region ---------------------
    Be = min(args.e2e_images, B)
    h_pixels = torch.empty((Be, H, W, NCH), dtype=torch.uint8, pin_memory=True)
    h_pixels.copy_(pixels[:Be])
    bound = himg_b200.encode_bound(W, H, NCH)
    h_out = torch.empty((Be * bound,), dtype=torch.uint8, pin_memory=True)
    h_dec = torch.empty((Be, H, W, NCH), dtype=torch.uint8, pin_memory=True)
    h_off = np.zeros(Be + 1, np.uint64)
    h_sizes = np.zeros(Be, np.uint32)
    h_status = np.zeros(Be, np.int32)

    def e2e_step():
        ctx.encode_batch_host(h_pixels, QUALITY, True, out=h_out, offsets=h_off, sizes=h_sizes)
        ctx.decode_batch_host(h_out, h_off, h_sizes, W, H, NCH, out=h_dec, status=h_status)

    def wall(fn, reps):
        barrier()
        t0 = time.perf_counter()
        fn(reps)
        barrier()
        return (time.perf_counter() - t0) * 1e3 / reps

    for _ in range(2):
        e2e_step()
    assert int(np.abs(h_status).sum()) == 0
    assert torch.equal(h_dec[Be - 1], decoded[Be - 1].cpu()), "e2e leg decoded different pixels"
    e2e_steps = max(2, min(args.steps, 5))
    e2e_serial_ms = wall(lambda reps: [e2e_step() for _ in range(reps)], e2e_steps)

    # Pipelined steps: encode is H2D-heavy and decode D2H-heavy, so one host thread encodes step k+1 (its
    # own context) while another decodes step k: both PCIe directions stay busy.  Same public calls,
    # same bytes per step inside the timed region.
    import queue
    import threading

    dev_index = dev.index if dev.index is not None else 0
    ctx_e, ctx_d = himg_b200.Context(dev_index), himg_b200.Context(dev_index)
    h_out2 = [h_out, torch.empty(h_out.shape, dtype=torch.uint8, pin_memory=True)]
    h_off2 = [h_off, np.zeros(Be + 1, np.uint64)]
    h_sizes2 = [h_sizes, np.zeros(Be, np.uint32)]

    def e2e_pipelined(reps):
        ready, free = queue.SimpleQueue(), [threading.Semaphore(1), threading.Semaphore(1)]
        stop = threading.Event()

        def encode_leg():
            try:
                for k in range(reps):
                    b = k & 1
                    free[b].acquire()
                    if stop.is_set():
                        return
                    ctx_e.encode_batch_host(h_pixels, QUALITY, True, out=h_out2[b], offsets=h_off2[b], sizes=h_sizes2[b])
                    ready.put(b)
            except Exception as e:  # surface in the main thread
                ready.put(e)

        th = threading.Thread(target=encode_leg, daemon=True)
        th.start()
        try:
            for _ in range(reps):
                b = ready.get(timeout=300)
                if isinstance(b, Exception):
                    raise b
                ctx_d.decode_batch_host(h_out2[b], h_off2[b], h_sizes2[b], W, H, NCH, out=h_dec, status=h_status)
                free[b].release()
        finally:  # never leave the encode leg parked on a semaphore
            stop.set()
            for sem in free:
                sem.release()
            th.join(timeout=300)

    h_dec.zero_()
    e2e_pipelined(2)
    assert int(np.abs(h_status).sum()) == 0
    assert torch.equal(h_dec[Be - 1], decoded[Be - 1].cpu()), "pipelined e2e leg decoded different pixels"
    e2e_pipe_steps = max(e2e_steps, 24)  # the first encode and the last decode run alone (1 / 25 of the time)
    e2e_ms = wall(e2e_pipelined, e2e_pipe_steps)
    ctx_e.close()
    ctx_d.close()
    packed_bytes = int(h_off[Be])
    h2d = Be * W * H * NCH + packed_bytes
    d2h = packed_bytes + Be * W * H * NCH
    del h_out2, h_pixels, h_dec, h_out

    if sampler is not None:
        sampler.terminate()
        sampler.wait()

    # ---- the other BASELINE.json configurations (N = 1): c2, c3 single images, c5 quality sweep ------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md 6.65 TB/s)"
    sub = {}
    if rank == 0 and world == 1 and not args.no_subrecords:
        del decoded
        torch.cuda.empty_cache()

        def single(name, w, h, nch):
            img = synth_images(1, w, h, nch, seed0=1, amp=6, device=dev)
            yc = nch >= 3
            o, s = ctx.encode_batch(img, QUALITY, yc)
            off = torch.zeros(1, dtype=torch.int64, device=dev)
            d, st = ctx.decode_batch(o.reshape(-1), off, s, w, h, nch)
            torch.cuda.synchronize()
            assert int(st[0]) == 0
            rec = {"shape": [w, h, nch], "quality": QUALITY, "himg_bytes": int(s[0])}
            try:  # recorded reference hashes of this configuration
                for c in json.load(open(os.path.join(ROOT, "tests", "golden", "golden_hashes.json"))):
                    if (c["w"], c["h"], c["nch"], c["quality"], c["seed"]) == (w, h, nch, QUALITY, 1):
                        ok = (int(s[0]) == c["himg_size"] and f"{himg_b200.fnv1a64(o[0, : int(s[0])].cpu().numpy()):016x}" == c["himg_hash"]
                              and f"{himg_b200.fnv1a64(d[0].cpu().numpy()):016x}" == c["pixel_hash"])
                        assert ok, f"{name}: output differs from the reference"
                        rec["parity_checked"] = True
            except (OSError, ValueError, KeyError):
                pass
            reps = 20
            rec["device_encode_ms"] = timed(lambda: ctx.encode_batch(img, QUALITY, yc, out=o, sizes=s), reps)
            rec["device_decode_ms"] = timed(lambda: ctx.decode_batch(o.reshape(-1), off, s, w, h, nch, out=d, status=st), reps)
            ctx.profile(True)
            ctx.profile_reset()
            for _ in range(reps):
                ctx.encode_batch(img, QUALITY, yc, out=o, sizes=s)
                ctx.decode_batch(o.reshape(-1), off, s, w, h, nch, out=d, status=st)
            pr = ctx.profile_results()
            ctx.profile(False)
            alg = 2 * nch * w * h
            for key, kn in (("k_forward", "k_fwd"), ("k_inverse", "k_inv")):
                t_ms, cnt = pr.get(key, (0.0, 0))
                if cnt:
                    us = t_ms / cnt * 1e3
                    rec[kn + "_us"] = us
                    rec[kn + "_frac"] = alg / (us * 1e-6) / 1e9 / peak
            rec["roofline_floor_us"] = alg / (peak * 1e9) * 1e6
            # the drop-in C++ classes (himg::Encoder / himg::Decoder over the C ABI, host buffers): the
            # `benchmark` driver, 30 iterations like the reference's
            tmp = os.path.join(tempfile.gettempdir(), f"himg_bench_{os.getpid()}_{name}.himg")
            with open(tmp, "wb") as f:
                f.write(o[0, : int(s[0])].cpu().numpy().tobytes())
            e = driver_times(["-e", f"synthetic:{w}x{h}x{nch}:1:6"])
            dd = driver_times(["-d", tmp])
            os.unlink(tmp)
            if e:
                rec["host_api_encode_ms"] = {"min": e[0], "avg": e[1]}
            if dd:
                rec["host_api_decode_ms"] = {"min": dd[0], "avg": dd[1]}
            rec["pcie_ms_of_its_bytes_at_55GBs"] = (w * h * nch + int(s[0])) / 55e9 * 1e3
            del img, o, d
            torch.cuda.empty_cache()
            return rec

        sub["c2"] = single("c2", 3840, 2160, 3)
        sub["c3"] = single("c3", 8192, 8192, 1)
        # c5: quality sweep on a 256-image slice of the resident batch (decode in lenient mode where the
        # reference decoder refuses its own encoder's stream: q0 / q10 for this generator)
        n5 = min(256, B)
        sweep = {}
        px5 = pixels[:n5]
        for q in (0, 50, 100):
            o5, s5 = ctx.encode_batch(px5, q, True)
            off5 = torch.arange(n5, dtype=torch.int64, device=dev) * o5.stride(0)
            d5, st5 = ctx.decode_batch(o5.reshape(-1), off5, s5, W, H, NCH, flags=himg_b200.LENIENT)
            torch.cuda.synchronize()
            assert int(st5.abs().sum()) == 0
            t_e = timed(lambda: ctx.encode_batch(px5, q, True, out=o5, sizes=s5), 3)
            t_d = timed(lambda: ctx.decode_batch(o5.reshape(-1), off5, s5, W, H, NCH, flags=himg_b200.LENIENT, out=d5, status=st5), 3)
            mp5 = n5 * W * H / 1e6
            sweep[f"q{q}"] = {"images": n5, "encode_mps": mp5 / (t_e / 1e3), "decode_mps": mp5 / (t_d / 1e3),
                              "bits_per_pixel": 8.0 * float(s5.sum().item()) / (n5 * W * H)}
            del o5, d5
            torch.cuda.empty_cache()
        sub["c5"] = sweep

    # ---- max over ranks -------------------------------------------------------------------------
    def rmax(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def rsum(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    ms, enc_ms, dec_ms, e2e_ms, e2e_serial_ms = rmax(ms), rmax(enc_ms), rmax(dec_ms), rmax(e2e_ms), rmax(e2e_serial_ms)
    launches = int(rsum(launches))
    e2e_images_total = int(rsum(Be))
    mp_per_step = total_images * W * H / 1e6
    value = mp_per_step * args.steps / (ms / 1e3)

    if rank == 0:
        fwd_ms, fwd_n = prof.get("k_forward", (0.0, 0))
        inv_ms, inv_n = prof.get("k_inverse", (0.0, 0))
        # per launch: nch read + nch written per pixel (a shard larger than the workspace limit is coded in
        # sub-batches: average over the launches)
        alg_total = 2 * NCH * W * H * B * args.steps
        fwd_gbs = alg_total / (fwd_ms / 1e3) / 1e9 if fwd_n else 0.0
        inv_gbs = alg_total / (inv_ms / 1e3) / 1e9 if inv_n else 0.0
        traffic = None  # DRAM bytes per launch from the committed ncu capture of this exact configuration
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "r2_final_traffic.json")))
            if tr["config"] == {"images": B, "width": W, "height": H, "channels": NCH, "quality": QUALITY}:
                traffic = tr["k_forward"]["traffic"]
        except (OSError, ValueError, KeyError):
            pass
        step_kernel_ms = sum(v[0] for v in prof.values()) / args.steps
        shares = {k: round(v[0] / args.steps / step_kernel_ms, 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}
        res = {
            "metric": "encode+decode megapixels/sec",
            "value": value,
            "unit": "MP/s",
            "n_gpus": world,
            "steps": args.steps,
            "warmup": warmup,
            "ms_per_step": ms / args.steps,
            "higher_is_better": True,
            "scaling": "strong",
            "vs_baseline": None,
            "dtype": "int16",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "images_per_gpu": B, "total_images": total_images, "quality": QUALITY,
                       "l2_policy": f"inputs larger than L2 ({B * W * H * NCH / 1e9:.1f} GB of pixels per GPU per step)",
                       "parallelism": f"image-sharded x{world}, NCCL all_gather of bitstream sizes only"},
            "parity_checked": parity_total > 0,
            "parity_images_checked_against_reference_hashes": parity_total,
            "multi_gpu_parity": multi_gpu_parity,
            "encode_mps": mp_per_step / (enc_ms / 1e3),
            "decode_mps": mp_per_step / (dec_ms / 1e3),
            "e2e": {"value": e2e_images_total * W * H / 1e6 / (e2e_ms / 1e3), "unit": "MP/s",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "images_per_gpu": Be,
                    "steps": e2e_pipe_steps, "serial_value": e2e_images_total * W * H / 1e6 / (e2e_serial_ms / 1e3),
                    "serial_steps": e2e_steps,
                    "api": "himgcu_encode_batch_host + himgcu_decode_batch_host on pinned host buffers (each call pipelines "
                           "H2D / coding lanes / D2H over sub-batches); value = consecutive steps pipelined by two host "
                           "threads (encode of step k+1 overlaps decode of step k: both PCIe directions busy); "
                           "serial_value = the two calls back to back, one step at a time; a step of this leg is "
                           "images_per_gpu images of the shard (bytes per step are per GPU)"},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": "k_forward", "achieved": fwd_gbs, "peak": peak, "unit": "GB/s",
                         "frac": fwd_gbs / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_step": alg_total // args.steps, "launches": fwd_n,
                         "avg_launch_ms": fwd_ms / fwd_n if fwd_n else None,
                         "k_inverse": {"achieved": inv_gbs, "frac": inv_gbs / peak, "launches": inv_n,
                                       "avg_launch_ms": inv_ms / inv_n if inv_n else None}},
            "kernel_time_shares": shares,
            "kernel_ms_per_step": step_kernel_ms,
            "cpu_baseline": cpu_baseline,
            "clocks": summarize_clocks(clk_path, local_rank),
            "packed_bits_per_pixel": 8.0 * packed_bytes / (Be * W * H),
        }
        res.update(sub)
        print(json.dumps(res))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
