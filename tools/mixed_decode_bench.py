"""Whole-image decode of mixed-shape batches against the calls a caller had before it, alternated in one process
(numbers for DESIGN.md section 7).

    python tools/mixed_decode_bench.py [--reps 20] [--json OUT]

Case 1: 512 RGB q50 images of seeded random sizes (sides 256-1024, the sizes of tools/mixed_region_bench.py).
decode_batch_mixed (one call) against one decode_batch call per image.
Case 2: the uniform batch of 512 1080p RGB q50 images, decode_batch_mixed against decode_batch: the cost of the
generic inverse kernel (decode_batch takes the lane-pair k_inverse4 there) and of the separate segment-table walk.
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
from mixed_region_bench import alternate, card, kernels, pack  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    ctx = himg_b200.Context(0)
    res = {"card": card(), "reps": args.reps}
    print("card:", res["card"])
    rng = np.random.default_rng(7)
    B, nch = 512, 3

    # ---- case 1: 512 random shapes
    dims = np.stack([rng.integers(256, 1025, B), rng.integers(256, 1025, B)], 1).astype(np.int32)
    streams = []
    for k, (w, h) in enumerate(dims):
        out, sizes = ctx.encode_batch(synth_images(1, int(w), int(h), nch, 100 + k, 6), 50, True)
        streams.append(out[0, : int(sizes[0])].clone())
    himg, offs, sizes = pack(streams)
    del streams
    d_dims = torch.from_numpy(dims).cuda()
    max_w, max_h = int(dims[:, 0].max()), int(dims[:, 1].max())
    mixed, px_off, mst = ctx.decode_batch_mixed(himg, offs, sizes, d_dims, nch, max_w, max_h)
    spans = dims[:, 0].astype(np.int64) * dims[:, 1] * nch
    starts = np.cumsum(spans) - spans
    ref = torch.empty_like(mixed)
    rst = torch.empty((B,), dtype=torch.int32, device="cuda")
    single = [(int(w), int(h), offs[k: k + 1], sizes[k: k + 1], ref[int(starts[k]): int(starts[k] + spans[k])], rst[k: k + 1])
              for k, (w, h) in enumerate(dims)]

    def run_single():
        for (w, h, o, s, px, st) in single:
            ctx.decode_batch(himg, o, s, w, h, nch, out=px, status=st)

    def run_mixed():
        ctx.decode_batch_mixed(himg, offs, sizes, d_dims, nch, max_w, max_h, out=mixed, pixel_offsets=px_off, status=mst)

    run_single()
    torch.cuda.synchronize()
    assert int(mst.abs().sum()) == 0 and int(rst.abs().sum()) == 0
    assert torch.equal(px_off.cpu(), torch.from_numpy(starts)) and torch.equal(mixed, ref), "per-image calls differ"
    t_mixed, t_single = alternate([run_mixed, run_single], args.reps)
    r = {"images": B, "bounds": [max_w, max_h], "megapixels": round(float(spans.sum()) / nch / 1e6, 1),
         "stream_mb": round(float(sizes.sum()) / 1e6, 1), "mixed_ms": round(t_mixed, 3), "per_image_ms": round(t_single, 3),
         "kernels_us_mixed": kernels(ctx, run_mixed)}
    res["random_shapes"] = r
    print(f"512 random shapes (sides 256-1024) q50: mixed {t_mixed:.3f} ms, per-image decode_batch calls {t_single:.3f} ms")
    print("   kernels mixed (us/call):", r["kernels_us_mixed"])
    del mixed, ref, single, himg

    # ---- case 2: 512 x 1080p, one shape
    w, h = 1920, 1080
    px = synth_images(B, w, h, nch, 1, 6)
    out, sizes = ctx.encode_batch(px, 50, True)
    del px
    himg = out.reshape(-1)
    offs = torch.arange(B, dtype=torch.int64, device="cuda") * out.stride(0)
    d_dims = torch.tensor([[w, h]] * B, dtype=torch.int32, device="cuda")
    uni, ust = ctx.decode_batch(himg, offs, sizes, w, h, nch)
    mixed, px_off, mst = ctx.decode_batch_mixed(himg, offs, sizes, d_dims, nch, w, h)
    torch.cuda.synchronize()
    assert int(ust.abs().sum()) == 0 and torch.equal(mst, ust) and torch.equal(mixed, uni.reshape(-1))

    def run_batch():
        ctx.decode_batch(himg, offs, sizes, w, h, nch, out=uni, status=ust)

    def run_mixed2():
        ctx.decode_batch_mixed(himg, offs, sizes, d_dims, nch, w, h, out=mixed, pixel_offsets=px_off, status=mst)

    t_uni, t_mix = alternate([run_batch, run_mixed2], args.reps)
    r = {"batch_ms": round(t_uni, 3), "mixed_ms": round(t_mix, 3), "ratio": round(t_mix / t_uni, 3),
         "kernels_us_batch": kernels(ctx, run_batch), "kernels_us_mixed": kernels(ctx, run_mixed2)}
    res["uniform_1080p"] = r
    print(f"512 x 1080p q50: decode_batch {t_uni:.3f} ms, mixed {t_mix:.3f} ms")
    print("   kernels batch (us/call):", r["kernels_us_batch"])
    print("   kernels mixed (us/call):", r["kernels_us_mixed"])
    if args.json:
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
