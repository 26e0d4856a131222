"""Region decode of mixed-shape batches against the calls a caller had before it, alternated in one process (numbers for
DESIGN.md section 7).

    python tools/mixed_region_bench.py [--reps 20] [--json OUT]

Case 1: 512 RGB q50 images of seeded random sizes (sides 256-1024), 224x224 crops at seeded random valid origins.
decode_batch_region_mixed (one call) against one decode_batch_region call per distinct shape and against one
single-image device call (decode_batch_region with n = 1, what himgcu_decode_region does after its copies) per image.
Case 2: the uniform batch of 512 1080p RGB q50 images with 224x224 crops, decode_batch_region_mixed against
decode_batch_region: the cost of the generic inverse kernel and of grids sized by the bounding shape.  Outputs of all
arms are compared byte for byte before timing.  Times are CUDA event times per call (median over --reps repetitions
after warm-up, the arms alternating); per-kernel times come from Context.profile in a separate pass."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import himg_b200  # noqa: E402
from himg_b200.synth import synth_images  # noqa: E402


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # (the numbers stand without it, but say so)
        return f"unknown ({e})"


def alternate(fns, reps):
    """Median event time (ms) of each function, called in turn."""
    for _ in range(3):
        for f in fns:
            f()
    torch.cuda.synchronize()
    ev = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in fns] for _ in range(reps)]
    for rep in ev:
        for f, (a, b) in zip(fns, rep):
            a.record()
            f()
            b.record()
    torch.cuda.synchronize()
    return [float(np.median([rep[k][0].elapsed_time(rep[k][1]) for rep in ev])) for k in range(len(fns))]


def kernels(ctx, fn, calls=5):
    ctx.profile(True)
    ctx.profile_reset()
    for _ in range(calls):
        fn()
    ctx.synchronize()
    out = {k: round(v[0] / calls * 1e3, 1) for k, v in sorted(ctx.profile_results().items(), key=lambda kv: -kv[1][0])}
    ctx.profile(False)
    return out


def pack(streams):
    """One device buffer of the streams (16-byte aligned), their offsets and sizes."""
    lens = [int(s.numel()) for s in streams]
    offs = np.cumsum([0] + [(n + 15) & ~15 for n in lens])
    buf = torch.zeros(int(offs[-1]) + 64, dtype=torch.uint8, device="cuda")
    for o, s in zip(offs, streams):
        buf[int(o): int(o) + s.numel()] = s
    return (buf, torch.from_numpy(offs[:-1].astype(np.int64)).cuda(), torch.tensor(lens, dtype=torch.int32, device="cuda"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    ctx = himg_b200.Context(0)
    res = {"card": card(), "reps": args.reps}
    print("card:", res["card"])
    rng = np.random.default_rng(7)
    B, nch, rw, rh = 512, 3, 224, 224

    # ---- case 1: 512 random shapes
    dims = np.stack([rng.integers(256, 1025, B), rng.integers(256, 1025, B)], 1).astype(np.int32)
    streams = []
    for k, (w, h) in enumerate(dims):
        out, sizes = ctx.encode_batch(synth_images(1, int(w), int(h), nch, 100 + k, 6), 50, True)
        streams.append(out[0, : int(sizes[0])].clone())
    himg, offs, sizes = pack(streams)
    del streams
    org_np = np.stack([rng.integers(0, dims[:, 0] - rw + 1), rng.integers(0, dims[:, 1] - rh + 1)], 1).astype(np.int32)
    d_dims, org = torch.from_numpy(dims).cuda(), torch.from_numpy(org_np).cuda()
    max_w, max_h = int(dims[:, 0].max()), int(dims[:, 1].max())
    mixed, mst = ctx.decode_batch_region_mixed(himg, offs, sizes, d_dims, nch, org, rw, rh, max_w, max_h)
    # one call per distinct shape
    groups = {}
    for k, (w, h) in enumerate(dims):
        groups.setdefault((int(w), int(h)), []).append(k)
    per_shape = []
    for (w, h), ks in groups.items():
        idx = torch.tensor(ks, dtype=torch.int64, device="cuda")
        o, s, g = offs[idx].contiguous(), sizes[idx].contiguous(), org[idx].contiguous()
        px, st = ctx.decode_batch_region(himg, o, s, w, h, nch, g, rw, rh)
        per_shape.append((w, h, o, s, g, px, st, idx))
    # one single-image device call per image
    single = []
    for k, (w, h) in enumerate(dims):
        px, st = ctx.decode_batch_region(himg, offs[k: k + 1], sizes[k: k + 1], int(w), int(h), nch, org[k: k + 1], rw, rh)
        single.append((int(w), int(h), offs[k: k + 1], sizes[k: k + 1], org[k: k + 1], px, st))
    torch.cuda.synchronize()
    assert int(mst.abs().sum()) == 0
    for (w, h, o, s, g, px, st, idx) in per_shape:
        assert int(st.abs().sum()) == 0 and torch.equal(px, mixed[idx]), f"per-shape call {w}x{h} differs"
    for k, (w, h, o, s, g, px, st) in enumerate(single):
        assert int(st[0]) == 0 and torch.equal(px[0], mixed[k]), f"single call {k} differs"

    def run_mixed():
        ctx.decode_batch_region_mixed(himg, offs, sizes, d_dims, nch, org, rw, rh, max_w, max_h, out=mixed, status=mst)

    def run_per_shape():
        for (w, h, o, s, g, px, st, _) in per_shape:
            ctx.decode_batch_region(himg, o, s, w, h, nch, g, rw, rh, out=px, status=st)

    def run_single():
        for (w, h, o, s, g, px, st) in single:
            ctx.decode_batch_region(himg, o, s, w, h, nch, g, rw, rh, out=px, status=st)

    t_mixed, t_shape, t_single = alternate([run_mixed, run_per_shape, run_single], args.reps)
    r = {"images": B, "distinct_shapes": len(groups), "bounds": [max_w, max_h],
         "stream_mb": round(float(sizes.sum()) / 1e6, 1), "mixed_ms": round(t_mixed, 3), "per_shape_ms": round(t_shape, 3),
         "per_image_ms": round(t_single, 3), "kernels_us_mixed": kernels(ctx, run_mixed)}
    res["random_shapes"] = r
    print(f"512 random shapes (sides 256-1024, {len(groups)} distinct) q50, 224^2 crops: mixed {t_mixed:.3f} ms, "
          f"per-shape calls {t_shape:.3f} ms, per-image calls {t_single:.3f} ms")
    print("   kernels mixed (us/call):", r["kernels_us_mixed"])
    del mixed, per_shape, single, himg

    # ---- case 2: 512 x 1080p, one shape
    w, h = 1920, 1080
    px = synth_images(B, w, h, nch, 1, 6)
    out, sizes = ctx.encode_batch(px, 50, True)
    del px
    himg = out.reshape(-1)
    offs = torch.arange(B, dtype=torch.int64, device="cuda") * out.stride(0)
    org = torch.from_numpy(np.stack([rng.integers(0, w - rw + 1, B), rng.integers(0, h - rh + 1, B)], 1).astype(np.int32)).cuda()
    d_dims = torch.tensor([[w, h]] * B, dtype=torch.int32, device="cuda")
    reg, rst = ctx.decode_batch_region(himg, offs, sizes, w, h, nch, org, rw, rh)
    mixed, mst = ctx.decode_batch_region_mixed(himg, offs, sizes, d_dims, nch, org, rw, rh, w, h)
    torch.cuda.synchronize()
    assert int(rst.abs().sum()) == 0 and torch.equal(mst, rst) and torch.equal(mixed, reg)

    def run_region():
        ctx.decode_batch_region(himg, offs, sizes, w, h, nch, org, rw, rh, out=reg, status=rst)

    def run_mixed2():
        ctx.decode_batch_region_mixed(himg, offs, sizes, d_dims, nch, org, rw, rh, w, h, out=mixed, status=mst)

    t_reg, t_mix = alternate([run_region, run_mixed2], args.reps)
    r = {"region_ms": round(t_reg, 3), "mixed_ms": round(t_mix, 3), "ratio": round(t_mix / t_reg, 3),
         "kernels_us_region": kernels(ctx, run_region), "kernels_us_mixed": kernels(ctx, run_mixed2)}
    res["uniform_1080p"] = r
    print(f"512 x 1080p q50, 224^2 crops: decode_batch_region {t_reg:.3f} ms, mixed {t_mix:.3f} ms")
    print("   kernels region (us/call):", r["kernels_us_region"])
    print("   kernels mixed  (us/call):", r["kernels_us_mixed"])
    if args.json:
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
