"""Scaled decode (1/2, 1/4, 1/8 size) against a full decode followed by the pooling a caller would write in torch,
alternated in one process (numbers for DESIGN.md section 7).

    python tools/scaled_decode_bench.py [--reps 20] [--json OUT]

Uniform case: 512 x 1080p RGB q50.  decode_batch followed by an int32 sum over the reshaped f x f windows and
(S + f^2 / 2) // f^2 (exact: 1920 and 1080 are multiples of 8), against decode_batch_scaled.
Random case: 512 RGB q50 images of seeded random sizes (sides 256-1024, the streams of tools/mixed_region_bench.py).
decode_batch_mixed followed by the same pooling per image (edge windows clipped, each divided by its own pixel count),
against decode_batch_mixed_scaled.
Outputs of both arms are compared byte for byte before timing.  Times are CUDA event times per call (median over --reps
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


def pool_uniform(px, f):
    """[n][h][w][c] uint8 with h, w multiples of f -> rounded box averages."""
    n, h, w, c = px.shape
    s = px.view(n, h // f, f, w // f, f, c).to(torch.int32).sum(dim=(2, 4))
    return torch.div(s + f * f // 2, f * f, rounding_mode="floor").to(torch.uint8)


_counts = {}


def pool_clipped(img, f):
    """[h][w][c] uint8 of any size -> rounded box averages, windows clipped at the right and bottom edges."""
    h, w, c = img.shape
    oh, ow = -(-h // f), -(-w // f)
    key = (h, w, f)
    if key not in _counts:  # (pixels per window: a caller computes these once per shape)
        ny = torch.clamp(h - f * torch.arange(oh, device=img.device), max=f)
        nx = torch.clamp(w - f * torch.arange(ow, device=img.device), max=f)
        _counts[key] = (ny.view(oh, 1, 1) * nx.view(1, ow, 1)).to(torch.int32)
    n = _counts[key]
    p = torch.nn.functional.pad(img.permute(2, 0, 1).to(torch.int32), (0, ow * f - w, 0, oh * f - h)).permute(1, 2, 0)
    s = p.reshape(oh, f, ow, f, c).sum(dim=(1, 3))
    return torch.div(s + n // 2, n, rounding_mode="floor").to(torch.uint8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    ctx = himg_b200.Context(0)
    res = {"card": card(), "reps": args.reps}
    print("card:", res["card"])
    B, nch = 512, 3

    # ---- uniform case: 512 x 1080p
    w, h = 1920, 1080
    px = synth_images(B, w, h, nch, 1, 6)
    out, sizes = ctx.encode_batch(px, 50, True)
    del px
    himg = out.reshape(-1)
    offs = torch.arange(B, dtype=torch.int64, device="cuda") * out.stride(0)
    full, fst = ctx.decode_batch(himg, offs, sizes, w, h, nch)
    res["uniform_1080p"] = {}
    for f in (2, 4, 8):
        ref = pool_uniform(full, f)
        sc, sst = ctx.decode_batch_scaled(himg, offs, sizes, w, h, nch, f)
        torch.cuda.synchronize()
        assert int(fst.abs().sum()) == 0 and torch.equal(sst, fst) and torch.equal(sc, ref), f"f {f}: outputs differ"
        del ref

        def run_pool():
            ctx.decode_batch(himg, offs, sizes, w, h, nch, out=full, status=fst)
            return pool_uniform(full, f)

        def run_scaled():
            ctx.decode_batch_scaled(himg, offs, sizes, w, h, nch, f, out=sc, status=sst)

        t_pool, t_sc = alternate([run_pool, run_scaled], args.reps)
        r = {"decode_then_pool_ms": round(t_pool, 3), "scaled_ms": round(t_sc, 3), "speedup": round(t_pool / t_sc, 3),
             "kernels_us_decode_batch": kernels(ctx, lambda: ctx.decode_batch(himg, offs, sizes, w, h, nch, out=full, status=fst)),
             "kernels_us_scaled": kernels(ctx, run_scaled)}
        res["uniform_1080p"][f] = r
        print(f"512 x 1080p q50, f {f}: decode_batch + torch pooling {t_pool:.3f} ms, decode_batch_scaled {t_sc:.3f} ms")
        print("   kernels decode_batch (us/call):", r["kernels_us_decode_batch"])
        print("   kernels scaled       (us/call):", r["kernels_us_scaled"])
        del sc
    del full, himg, out
    torch.cuda.empty_cache()

    # ---- random case: 512 random shapes
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
    full, fpx_off, fst = ctx.decode_batch_mixed(himg, offs, sizes, d_dims, nch, max_w, max_h)
    spans = dims[:, 0].astype(np.int64) * dims[:, 1] * nch
    starts = [int(x) for x in np.cumsum(spans) - spans]
    views = [full[s0: s0 + int(sp)].view(int(ih), int(iw), nch) for s0, sp, (iw, ih) in zip(starts, spans, dims)]
    res["random_shapes"] = {"images": B, "bounds": [max_w, max_h], "megapixels": round(float(spans.sum()) / nch / 1e6, 1)}
    for f in (2, 4, 8):
        sc, spx_off, sst = ctx.decode_batch_mixed_scaled(himg, offs, sizes, d_dims, nch, max_w, max_h, f)
        ref = torch.cat([pool_clipped(v, f).reshape(-1) for v in views])
        torch.cuda.synchronize()
        assert int(fst.abs().sum()) == 0 and torch.equal(sst, fst) and torch.equal(sc, ref), f"f {f}: outputs differ"
        del ref

        def run_pool():
            ctx.decode_batch_mixed(himg, offs, sizes, d_dims, nch, max_w, max_h, out=full, pixel_offsets=fpx_off, status=fst)
            return [pool_clipped(v, f) for v in views]

        def run_scaled():
            ctx.decode_batch_mixed_scaled(himg, offs, sizes, d_dims, nch, max_w, max_h, f, out=sc, pixel_offsets=spx_off,
                                          status=sst)

        t_pool, t_sc = alternate([run_pool, run_scaled], args.reps)
        r = {"decode_then_pool_ms": round(t_pool, 3), "scaled_ms": round(t_sc, 3), "speedup": round(t_pool / t_sc, 3),
             "kernels_us_decode_batch_mixed": kernels(ctx, lambda: ctx.decode_batch_mixed(
                 himg, offs, sizes, d_dims, nch, max_w, max_h, out=full, pixel_offsets=fpx_off, status=fst)),
             "kernels_us_scaled": kernels(ctx, run_scaled)}
        res["random_shapes"][f] = r
        print(f"512 random shapes q50, f {f}: decode_batch_mixed + per-image torch pooling {t_pool:.3f} ms, "
              f"decode_batch_mixed_scaled {t_sc:.3f} ms")
        print("   kernels mixed        (us/call):", r["kernels_us_decode_batch_mixed"])
        print("   kernels mixed scaled (us/call):", r["kernels_us_scaled"])
        del sc
    if args.json:
        with open(args.json, "w") as fh:
            json.dump(res, fh, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
