"""Region decode against whole-image decode, alternated in one process (numbers for DESIGN.md section 7).

    python tools/region_bench.py [--reps 20] [--json OUT]

Cases: a batch of 512 1080p RGB images at q50 (encoded once), decode_batch against decode_batch_region with seeded
random origins for 224x224 and 512x512 crops and for the whole frame at (0, 0); one 8192^2 gray image (c3) and one
3840x2160 RGB image (c2), decode against a 1024^2 tile at a seeded position.  Times are CUDA event times per call
(median over --reps repetitions after warm-up, the two variants alternating); the single images are also timed
through the host calls (decode / decode_region, wall clock, copies included).  Per-kernel times come from
Context.profile in a separate pass."""
import argparse
import json
import os
import subprocess
import sys
import time

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


def alternate(fa, fb, reps):
    """Median event time (ms) of fa and of fb, called alternately."""
    for _ in range(3):
        fa()
        fb()
    torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(reps)]
    for e in ev:
        e[0].record()
        fa()
        e[1].record()
        e[2].record()
        fb()
        e[3].record()
    torch.cuda.synchronize()
    return (float(np.median([e[0].elapsed_time(e[1]) for e in ev])), float(np.median([e[2].elapsed_time(e[3]) for e in ev])))


def kernels(ctx, fn, calls=5):
    ctx.profile(True)
    ctx.profile_reset()
    for _ in range(calls):
        fn()
    ctx.synchronize()
    out = {k: round(v[0] / calls * 1e3, 1) for k, v in sorted(ctx.profile_results().items(), key=lambda kv: -kv[1][0])}
    ctx.profile(False)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    ctx = himg_b200.Context(0)
    res = {"card": card(), "reps": args.reps, "batch": {}, "single": {}}
    print("card:", res["card"])
    rng = np.random.default_rng(7)

    # ---- 512 x 1080p RGB q50
    w, h, n, B = 1920, 1080, 3, 512
    px = synth_images(B, w, h, n, 1, 6)
    out, sizes = ctx.encode_batch(px, 50, True)
    del px
    himg = out.reshape(-1)
    offs = torch.arange(B, dtype=torch.int64, device="cuda") * out.stride(0)
    full, st = ctx.decode_batch(himg, offs, sizes, w, h, n)
    torch.cuda.synchronize()
    assert int(st.abs().sum()) == 0
    for name, (cw, chh) in {"224x224": (224, 224), "512x512": (512, 512), "whole_frame": (w, h)}.items():
        if name == "whole_frame":
            org = torch.zeros((B, 2), dtype=torch.int32, device="cuda")
        else:
            org = torch.from_numpy(np.stack([rng.integers(0, w - cw + 1, B), rng.integers(0, h - chh + 1, B)], 1).astype(np.int32)).cuda()
        reg, rst = ctx.decode_batch_region(himg, offs, sizes, w, h, n, org, cw, chh)
        torch.cuda.synchronize()
        assert int(rst.abs().sum()) == 0
        o = org.cpu().numpy()
        for k in (0, B - 1):  # spot check against the whole decode
            x, y = o[k]
            assert torch.equal(reg[k], full[k, y: y + chh, x: x + cw]), f"{name}: image {k} differs from the crop"
        t_full, t_reg = alternate(lambda: ctx.decode_batch(himg, offs, sizes, w, h, n, out=full, status=st),
                                  lambda: ctx.decode_batch_region(himg, offs, sizes, w, h, n, org, cw, chh, out=reg, status=rst),
                                  args.reps)
        r = {"decode_batch_ms": round(t_full, 3), "decode_batch_region_ms": round(t_reg, 3), "ratio": round(t_reg / t_full, 3),
             "kernels_us_full": kernels(ctx, lambda: ctx.decode_batch(himg, offs, sizes, w, h, n, out=full, status=st)),
             "kernels_us_region": kernels(ctx, lambda: ctx.decode_batch_region(himg, offs, sizes, w, h, n, org, cw, chh, out=reg,
                                                                               status=rst))}
        res["batch"][name] = r
        print(f"512 x 1080p q50, {name}: decode_batch {t_full:.3f} ms, decode_batch_region {t_reg:.3f} ms")
        print("   kernels full  (us/call):", r["kernels_us_full"])
        print("   kernels region(us/call):", r["kernels_us_region"])
        del reg
    del full, out, himg

    # ---- single images, 1024^2 tile
    for name, (w, h, n) in {"c3_8192x8192x1": (8192, 8192, 1), "c2_3840x2160x3": (3840, 2160, 3)}.items():
        px = synth_images(1, w, h, n, 1, 6)
        out, sizes = ctx.encode_batch(px, 50, True)
        offs = torch.zeros(1, dtype=torch.int64, device="cuda")
        x, y = int(rng.integers(0, w - 1024 + 1)), int(rng.integers(0, h - 1024 + 1))
        org = torch.tensor([[x, y]], dtype=torch.int32, device="cuda")
        himg = out.reshape(-1)
        full, st = ctx.decode_batch(himg, offs, sizes, w, h, n)
        reg, rst = ctx.decode_batch_region(himg, offs, sizes, w, h, n, org, 1024, 1024)
        torch.cuda.synchronize()
        assert int(st[0]) == 0 and int(rst[0]) == 0 and torch.equal(reg[0], full[0, y: y + 1024, x: x + 1024])
        t_full, t_reg = alternate(lambda: ctx.decode_batch(himg, offs, sizes, w, h, n, out=full, status=st),
                                  lambda: ctx.decode_batch_region(himg, offs, sizes, w, h, n, org, 1024, 1024, out=reg, status=rst),
                                  args.reps)
        packed = bytes(out[0, : int(sizes[0])].cpu().numpy())
        host = {"decode": [], "decode_region": []}
        for i in range(args.reps + 2):
            t0 = time.perf_counter()
            ctx.decode(packed)
            t1 = time.perf_counter()
            ctx.decode_region(packed, x, y, 1024, 1024)
            t2 = time.perf_counter()
            if i >= 2:
                host["decode"].append((t1 - t0) * 1e3)
                host["decode_region"].append((t2 - t1) * 1e3)
        r = {"tile_origin": [x, y], "device_decode_ms": round(t_full, 3), "device_region_ms": round(t_reg, 3),
             "host_decode_ms": round(float(np.median(host["decode"])), 3),
             "host_decode_region_ms": round(float(np.median(host["decode_region"])), 3),
             "kernels_us_full": kernels(ctx, lambda: ctx.decode_batch(himg, offs, sizes, w, h, n, out=full, status=st)),
             "kernels_us_region": kernels(ctx, lambda: ctx.decode_batch_region(himg, offs, sizes, w, h, n, org, 1024, 1024, out=reg,
                                                                               status=rst))}
        res["single"][name] = r
        print(f"{name}, 1024^2 tile at {(x, y)}: device {t_full:.3f} -> {t_reg:.3f} ms, host call {r['host_decode_ms']:.3f} -> "
              f"{r['host_decode_region_ms']:.3f} ms")
        print("   kernels full  (us/call):", r["kernels_us_full"])
        print("   kernels region(us/call):", r["kernels_us_region"])
        del full, reg, out, himg, px
    if args.json:
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
