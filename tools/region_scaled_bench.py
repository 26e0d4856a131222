"""Scaled region decode against the calls a caller had before it, alternated in one process (numbers for DESIGN.md
section 7).

    python tools/region_scaled_bench.py [--reps 20] [--json OUT]

Case 1: 512 x 1080p RGB q50, one 224 x 224 crop per image of the image scaled by f = 2 and 4, at seeded random origins.
decode_batch_region_scaled (lane-pair kernel, and with force_generic the generic kernel) against decode_batch_region of
the (224 f)^2 source rectangle followed by integer pooling in torch, and against decode_batch_scaled followed by a crop
(one gather).
Case 2: 512 RGB q50 images of seeded random sizes (sides 256-1024, the streams of tools/mixed_region_bench.py), 112 x 112
crops at f = 2.  decode_batch_region_mixed_scaled against decode_batch_region_mixed at 224 x 224 plus pooling (origins
are drawn so that the 224 x 224 source rectangle lies inside the image).
Case 3: one 8192 x 8192 gray q50 image, a 1024 x 1024 tile at f = 4 through the single-image host call (the viewer
case), against decode_region of the 4096 x 4096 source rectangle plus numpy pooling, and decode_scaled plus a crop.
Outputs of all arms are compared byte for byte before timing.  Device times are CUDA event times per call, host-call
times host clock times (the calls return after their device-to-host copy); medians over --reps repetitions after
warm-up, the arms alternating.  Per-kernel times come from Context.profile in a separate pass."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import himg_b200  # noqa: E402
from himg_b200.synth import synth_images  # noqa: E402
from mixed_region_bench import alternate, card, kernels, pack  # noqa: E402
from scaled_decode_bench import pool_uniform  # noqa: E402


def crop_gather(px, org, cw, ch):
    """[n][h][w][c] -> [n][ch][cw][c]: the crop of image i at org[i] = (x, y), in one gather."""
    n = px.shape[0]
    rows = org[:, 1:2] + torch.arange(ch, device=px.device)
    cols = org[:, 0:1] + torch.arange(cw, device=px.device)
    return px[torch.arange(n, device=px.device)[:, None, None], rows[:, :, None].long(), cols[:, None, :].long()]


def alternate_host(fns, reps):
    """Median host time (ms) of each synchronous function, called in turn."""
    for _ in range(2):
        for f in fns:
            f()
    t = [[] for _ in fns]
    for _ in range(reps):
        for k, f in enumerate(fns):
            t0 = time.perf_counter()
            f()
            t[k].append((time.perf_counter() - t0) * 1e3)
    return [float(np.median(x)) for x in t]


def pool_np(img, f):
    h, w, c = img.shape
    s = img.reshape(h // f, f, w // f, f, c).sum(axis=(1, 3), dtype=np.int32)
    return ((s + f * f // 2) // (f * f)).astype(np.uint8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    ctx = himg_b200.Context(0)
    gen = himg_b200.Context(0)
    gen.set_option("force_generic", 1)
    res = {"card": card(), "reps": args.reps}
    print("card:", res["card"])
    B, nch = 512, 3
    rng = np.random.default_rng(7)

    # ---- case 1: 512 x 1080p, 224^2 crops at f = 2 and 4
    w, h, crop = 1920, 1080, 224
    px = synth_images(B, w, h, nch, 1, 6)
    out, sizes = ctx.encode_batch(px, 50, True)
    del px
    himg = out.reshape(-1)
    offs = torch.arange(B, dtype=torch.int64, device="cuda") * out.stride(0)
    res["uniform_1080p"] = {}
    for f in (2, 4):
        sw, sh = w // f, h // f
        org = torch.from_numpy(np.stack([rng.integers(0, sw - crop + 1, B), rng.integers(0, sh - crop + 1, B)], 1)
                               .astype(np.int32)).cuda()
        src_org = org * f
        a, sa = ctx.decode_batch_region_scaled(himg, offs, sizes, w, h, nch, f, org, crop, crop)
        g, sg = gen.decode_batch_region_scaled(himg, offs, sizes, w, h, nch, f, org, crop, crop)
        rg, srg = ctx.decode_batch_region(himg, offs, sizes, w, h, nch, src_org, f * crop, f * crop)
        sc, ssc = ctx.decode_batch_scaled(himg, offs, sizes, w, h, nch, f)
        torch.cuda.synchronize()
        assert int(sa.abs().sum()) == 0 and torch.equal(sa, sg) and torch.equal(sa, srg) and torch.equal(sa, ssc)
        assert torch.equal(a, g), f"f {f}: lane-pair and generic kernels differ"
        assert torch.equal(a, pool_uniform(rg, f)) and torch.equal(a, crop_gather(sc, org, crop, crop)), f"f {f}: outputs differ"

        def run_region_pool():
            ctx.decode_batch_region(himg, offs, sizes, w, h, nch, src_org, f * crop, f * crop, out=rg, status=srg)
            return pool_uniform(rg, f)

        def run_scaled_crop():
            ctx.decode_batch_scaled(himg, offs, sizes, w, h, nch, f, out=sc, status=ssc)
            return crop_gather(sc, org, crop, crop)

        def run_fused():
            ctx.decode_batch_region_scaled(himg, offs, sizes, w, h, nch, f, org, crop, crop, out=a, status=sa)

        def run_fused_generic():
            gen.decode_batch_region_scaled(himg, offs, sizes, w, h, nch, f, org, crop, crop, out=g, status=sg)

        t = alternate([run_region_pool, run_scaled_crop, run_fused, run_fused_generic], args.reps)
        r = {"region_then_pool_ms": round(t[0], 3), "scaled_then_crop_ms": round(t[1], 3), "region_scaled_ms": round(t[2], 3),
             "region_scaled_generic_ms": round(t[3], 3),
             "kernels_us_region_scaled": kernels(ctx, run_fused),
             "kernels_us_region_scaled_generic": kernels(gen, run_fused_generic)}
        res["uniform_1080p"][f] = r
        print(f"512 x 1080p q50, 224^2 crops at f {f}: decode_batch_region {f * crop}^2 + pooling {t[0]:.3f} ms, "
              f"decode_batch_scaled + crop {t[1]:.3f} ms, decode_batch_region_scaled {t[2]:.3f} ms "
              f"(force_generic {t[3]:.3f} ms)")
        print("   kernels region_scaled         (us/call):", r["kernels_us_region_scaled"])
        print("   kernels region_scaled generic (us/call):", r["kernels_us_region_scaled_generic"])
        del a, g, rg, sc
    del himg, out
    torch.cuda.empty_cache()

    # ---- case 2: 512 random shapes, 112^2 crops at f = 2
    f, crop = 2, 112
    rng = np.random.default_rng(7)
    dims = np.stack([rng.integers(256, 1025, B), rng.integers(256, 1025, B)], 1).astype(np.int32)
    streams = []
    for k, (iw, ih) in enumerate(dims):
        o, s = ctx.encode_batch(synth_images(1, int(iw), int(ih), nch, 100 + k, 6), 50, True)
        streams.append(o[0, : int(s[0])].clone())
    himg, offs, sizes = pack(streams)
    del streams
    d_dims = torch.from_numpy(dims).cuda()
    max_w, max_h = int(dims[:, 0].max()), int(dims[:, 1].max())
    org_np = np.stack([rng.integers(0, (dims[:, 0] - f * crop) // f + 1), rng.integers(0, (dims[:, 1] - f * crop) // f + 1)],
                      1).astype(np.int32)
    org = torch.from_numpy(org_np).cuda()
    src_org = org * f
    a, sa = ctx.decode_batch_region_mixed_scaled(himg, offs, sizes, d_dims, nch, f, org, crop, crop, max_w, max_h)
    rg, srg = ctx.decode_batch_region_mixed(himg, offs, sizes, d_dims, nch, src_org, f * crop, f * crop, max_w, max_h)
    torch.cuda.synchronize()
    assert int(sa.abs().sum()) == 0 and torch.equal(sa, srg) and torch.equal(a, pool_uniform(rg, f)), "random shapes differ"

    def run_mixed_pool():
        ctx.decode_batch_region_mixed(himg, offs, sizes, d_dims, nch, src_org, f * crop, f * crop, max_w, max_h, out=rg,
                                      status=srg)
        return pool_uniform(rg, f)

    def run_mixed_fused():
        ctx.decode_batch_region_mixed_scaled(himg, offs, sizes, d_dims, nch, f, org, crop, crop, max_w, max_h, out=a, status=sa)

    t = alternate([run_mixed_pool, run_mixed_fused], args.reps)
    res["random_shapes"] = {"images": B, "bounds": [max_w, max_h], "region_mixed_then_pool_ms": round(t[0], 3),
                            "region_mixed_scaled_ms": round(t[1], 3), "kernels_us_region_mixed_scaled": kernels(ctx, run_mixed_fused)}
    print(f"512 random shapes q50, 112^2 crops at f 2: decode_batch_region_mixed 224^2 + pooling {t[0]:.3f} ms, "
          f"decode_batch_region_mixed_scaled {t[1]:.3f} ms")
    print("   kernels (us/call):", res["random_shapes"]["kernels_us_region_mixed_scaled"])
    del a, rg, himg
    torch.cuda.empty_cache()

    # ---- case 3: one 8192^2 gray image, a 1024^2 tile at f = 4 through the host call
    f, tile, W = 4, 1024, 8192
    o, s = ctx.encode_batch(synth_images(1, W, W, 1, 3, 6), 50, True)
    data = o[0, : int(s[0])].cpu().numpy().tobytes()
    x, y = 700, 900  # (scaled coordinates, inside the 2048^2 scaled image)
    fused = ctx.decode_region_scaled(data, f, x, y, tile, tile)
    src = ctx.decode_region(data, f * x, f * y, f * tile, f * tile)
    whole = ctx.decode_scaled(data, f)
    assert np.array_equal(fused, pool_np(src, f)) and np.array_equal(fused, whole[y: y + tile, x: x + tile]), "tile differs"
    t = alternate_host([lambda: pool_np(ctx.decode_region(data, f * x, f * y, f * tile, f * tile), f),
                        lambda: np.ascontiguousarray(ctx.decode_scaled(data, f)[y: y + tile, x: x + tile]),
                        lambda: ctx.decode_region_scaled(data, f, x, y, tile, tile)], args.reps)
    res["viewer_8192_gray"] = {"region_then_pool_ms": round(t[0], 3), "scaled_then_crop_ms": round(t[1], 3),
                               "region_scaled_ms": round(t[2], 3),
                               "kernels_us_region_scaled": kernels(ctx, lambda: ctx.decode_region_scaled(data, f, x, y, tile, tile))}
    print(f"8192^2 gray q50, 1024^2 tile at f 4 (host call): decode_region 4096^2 + numpy pooling {t[0]:.3f} ms, "
          f"decode_scaled + crop {t[1]:.3f} ms, decode_region_scaled {t[2]:.3f} ms")
    print("   kernels (us/call):", res["viewer_8192_gray"]["kernels_us_region_scaled"])
    if args.json:
        with open(args.json, "w") as fh:
            json.dump(res, fh, indent=1)
    gen.close()
    ctx.close()


if __name__ == "__main__":
    main()
