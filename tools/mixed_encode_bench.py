"""Encode of mixed-shape batches against the calls a caller had before it, alternated in one process (numbers for
DESIGN.md section 7).

    python tools/mixed_encode_bench.py [--reps 20] [--json OUT]

Case 1: the seeded batch of tools/mixed_region_bench.py, 512 RGB q50 images with sides 256-1024, in one flat device
buffer.  encode_batch_mixed (one call) against one encode_batch call with n = 1 per image.
Case 2: 512 1080p RGB q50 images (one shape), encode_batch_mixed against encode_batch: the cost of the generic
k_lowres_avg / k_forward against the lane-pair k_lowres_avg2 / k_forward3, and of grids sized by the bounding shape.
Outputs of all arms are compared byte for byte before timing.  Times are CUDA event times per call (median over --reps
repetitions after warm-up, the arms alternating); per-kernel times come from Context.profile in a separate pass."""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import himg_b200  # noqa: E402
from himg_b200.synth import synth_images  # noqa: E402
from mixed_region_bench import alternate, card, kernels  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    ctx = himg_b200.Context(0)
    res = {"card": card(), "reps": args.reps}
    print("card:", res["card"])
    rng = np.random.default_rng(7)
    B, nch, q = 512, 3, 50

    # ---- case 1: 512 random shapes (the dims and pixels of tools/mixed_region_bench.py)
    dims = np.stack([rng.integers(256, 1025, B), rng.integers(256, 1025, B)], 1).astype(np.int32)
    nbytes = [int(w) * int(h) * nch for (w, h) in dims]
    offs_np = np.cumsum([0] + nbytes)
    pixels = torch.empty(int(offs_np[-1]), dtype=torch.uint8, device="cuda")
    singles = []
    for k, (w, h) in enumerate(dims):
        img = synth_images(1, int(w), int(h), nch, 100 + k, 6)
        pixels[int(offs_np[k]): int(offs_np[k + 1])] = img.reshape(-1)
        singles.append(pixels[int(offs_np[k]): int(offs_np[k + 1])].view(1, int(h), int(w), nch))
    offs = torch.from_numpy(offs_np[:-1].astype(np.int64)).cuda()
    d_dims = torch.from_numpy(dims).cuda()
    max_w, max_h = int(dims[:, 0].max()), int(dims[:, 1].max())
    mixed, msz = ctx.encode_batch_mixed(pixels, offs, d_dims, nch, max_w, max_h, q)
    single = [ctx.encode_batch(px, q) for px in singles]
    torch.cuda.synchronize()
    ctx.encode_status()
    for k, (o, s) in enumerate(single):
        n = int(s[0])
        assert n > 0 and n == int(msz[k]) and torch.equal(o[0, :n], mixed[k, :n]), f"single call {k} differs"

    def run_mixed():
        ctx.encode_batch_mixed(pixels, offs, d_dims, nch, max_w, max_h, q, out=mixed, sizes=msz)

    def run_single():
        for px, (o, s) in zip(singles, single):
            ctx.encode_batch(px, q, out=o, sizes=s)

    t_mixed, t_single = alternate([run_mixed, run_single], args.reps)
    mp = float(sum(int(w) * int(h) for (w, h) in dims)) / 1e6
    r = {"images": B, "bounds": [max_w, max_h], "megapixels": round(mp, 1), "stream_mb": round(float(msz.sum()) / 1e6, 1),
         "mixed_ms": round(t_mixed, 3), "per_image_ms": round(t_single, 3), "kernels_us_mixed": kernels(ctx, run_mixed)}
    res["random_shapes"] = r
    print(f"512 random shapes (sides 256-1024, {mp:.0f} MP) q50: mixed {t_mixed:.3f} ms, per-image calls {t_single:.3f} ms")
    print("   kernels mixed (us/call):", r["kernels_us_mixed"])
    del mixed, single, singles, pixels

    # ---- case 2: 512 x 1080p, one shape
    w, h = 1920, 1080
    px = synth_images(B, w, h, nch, 1, 6)
    flat = px.reshape(-1)
    offs = torch.arange(B, dtype=torch.int64, device="cuda") * (w * h * nch)
    d_dims = torch.tensor([[w, h]] * B, dtype=torch.int32, device="cuda")
    ref, rsz = ctx.encode_batch(px, q)
    mixed, msz = ctx.encode_batch_mixed(flat, offs, d_dims, nch, w, h, q)
    torch.cuda.synchronize()
    ctx.encode_status()
    assert int(rsz.min()) > 0 and torch.equal(msz, rsz)
    for k in range(B):
        n = int(rsz[k])
        assert torch.equal(ref[k, :n], mixed[k, :n]), f"image {k} differs"

    def run_batch():
        ctx.encode_batch(px, q, out=ref, sizes=rsz)

    def run_mixed2():
        ctx.encode_batch_mixed(flat, offs, d_dims, nch, w, h, q, out=mixed, sizes=msz)

    t_b, t_m = alternate([run_batch, run_mixed2], args.reps)
    r = {"batch_ms": round(t_b, 3), "mixed_ms": round(t_m, 3), "ratio": round(t_m / t_b, 3),
         "kernels_us_batch": kernels(ctx, run_batch), "kernels_us_mixed": kernels(ctx, run_mixed2)}
    res["uniform_1080p"] = r
    print(f"512 x 1080p q50: encode_batch {t_b:.3f} ms, mixed {t_m:.3f} ms")
    print("   kernels batch (us/call):", r["kernels_us_batch"])
    print("   kernels mixed (us/call):", r["kernels_us_mixed"])
    if args.json:
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
