"""Launch trace of libhimgcu.so's host code, for checking that a host-side change leaves every launch as it was.

Runs a fixed matrix of calls that reaches every routing branch of the library (whole-image, scaled and region decodes,
uniform and mixed batches, encodes, the host-buffer pipelines, every stage entry point, and the options that change the
routing) and writes one record per call to OUT/trace.jsonl:

- "trace": the kernel, memcpy and memset records of each stream as torch.profiler (CUDA activities) reports them:
  name with template arguments, grid, block, dynamic shared memory, bytes.  Streams are listed as a sorted list of
  their sequences, so that stream numbering does not matter; for calls that run several coding lanes each sequence is
  sorted as well (which lane codes which sub-batch is timing-dependent).
- "profile" / "launches": from a separate pass with Context.profile(True), the names and counts of
  profile_results() and the launch_count() of the call.

Every call runs once untraced first, so the trace is of the steady state.  Two libraries with the same launch
sequences give identical files:

    python tools/launch_trace.py --out DIR_A --lib path/to/parent/libhimgcu.so
    python tools/launch_trace.py --out DIR_B
    python tools/launch_trace.py --compare DIR_A DIR_B
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def compare(a, b):
    """Compares the records of the calls both files have.  A call of the first file missing from the second fails, as a
    mismatch does; calls only the second file has (new entry points) are listed."""
    ra = {r["call"]: r for r in map(json.loads, open(os.path.join(a, "trace.jsonl")))}
    rb = {r["call"]: r for r in map(json.loads, open(os.path.join(b, "trace.jsonl")))}
    both = [k for k in ra if k in rb]
    bad = [k for k in both if ra[k] != rb[k]]
    print(json.dumps({"calls": len(both), "mismatches": bad, "only_a": [k for k in ra if k not in rb],
                      "only_b": [k for k in rb if k not in ra]}))
    return 1 if bad or any(k not in rb for k in ra) else 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="output directory")
    ap.add_argument("--lib", help="libhimgcu.so to load instead of the tree's")
    ap.add_argument("--compare", nargs=2, metavar="DIR")
    args = ap.parse_args()
    if args.compare:
        return compare(*args.compare)

    import torch
    from torch.profiler import ProfilerActivity, profile

    from himg_b200 import _native

    if args.lib:
        _native.LIB_PATH = os.path.abspath(args.lib)
    import himg_b200
    from himg_b200.synth import synth_images

    dev = "cuda"
    os.makedirs(args.out, exist_ok=True)

    # ---- inputs ---------------------------------------------------------------------------------
    maker = himg_b200.Context(0)
    maker.set_stream(torch.cuda.current_stream().cuda_stream)
    shapes = {"1080p": (1920, 1080, 3), "gray1024": (1024, 1024, 1), "rgba512": (512, 512, 4), "odd": (333, 207, 3),
              "ch5": (96, 64, 5), "4k": (3840, 2160, 3), "8kgray": (8192, 8192, 1), "oddw": (1922, 1080, 3), "rgb512": (512, 512, 3)}
    px, packed = {}, {}
    for k, (w, h, c) in shapes.items():
        n = 64 if k == "1080p" else 2
        px[k] = synth_images(n, w, h, c, 1, 6)
        if k in ("8kgray",):
            continue
        out, sizes = maker.encode_batch(px[k], 50, True)
        packed[k] = (out, sizes)
    torch.cuda.synchronize()

    streams = {k: out[0, : int(sizes[0])].cpu().numpy().tobytes() for k, (out, sizes) in packed.items()}
    host_img = {k: v[0].cpu().numpy() for k, v in px.items()}

    def batch(k, n):
        out, sizes = packed[k]
        offs = torch.arange(n, dtype=torch.int64, device=dev) * out.stride(0)
        return out.reshape(-1), offs, sizes[:n].contiguous()

    def out_at(nbytes, off):  # a flat output buffer whose data starts `off` bytes past a 256-byte boundary
        return torch.empty(nbytes + 256, dtype=torch.uint8, device=dev)[off: off + nbytes]

    mixed_dims = [(1920, 1080), (1000, 700), (333, 207), (1920, 1080), (64, 48)]
    mparts = [synth_images(1, w, h, 3, 7 + i, 6).reshape(-1) for i, (w, h) in enumerate(mixed_dims)]
    mpx = torch.cat(mparts)
    moffs = torch.tensor(np.cumsum([0] + [p.numel() for p in mparts[:-1]]), dtype=torch.int64, device=dev)
    mdims = torch.tensor(mixed_dims, dtype=torch.int32, device=dev)
    mout, msizes = maker.encode_batch_mixed(mpx, moffs, mdims, 3, 1920, 1080)
    mhimg = mout.reshape(-1)
    mhoffs = torch.arange(len(mixed_dims), dtype=torch.int64, device=dev) * mout.stride(0)
    torch.cuda.synchronize()

    rng = np.random.RandomState(5)
    huff_data = torch.from_numpy(rng.randint(0, 12, size=(2, 256 << 10)).astype(np.uint8)).to(dev)
    sl, sc = np.full(64, 2, np.uint8), np.full(64, 3, np.uint8)
    unmap = (np.arange(256) - 128).astype(np.int16)
    huff_packed = {bs: maker.stage_huff_compress(huff_data, bs) for bs in (0, 4096)}
    torch.cuda.synchronize()

    # ---- the matrix: (name, options, call(ctx)) -----------------------------------------------------
    calls = []

    def add(name, fn, opts=()):
        calls.append((name, dict(opts), fn))

    for k in ("1080p", "gray1024", "rgba512", "odd", "ch5"):
        w, h, c = shapes[k]
        add(f"decode/{k}", lambda ctx, k=k: ctx.decode(streams[k]))
        for f in (2, 4, 8):
            add(f"decode_scaled/{k}/f{f}", lambda ctx, k=k, f=f: ctx.decode_scaled(streams[k], f))
        add(f"decode_region/{k}", lambda ctx, k=k, w=w, h=h: ctx.decode_region(streams[k], w // 5, h // 7, w // 2, h // 3))
        for f in (1, 2, 4, 8):
            sw, sh = -(-w // f), -(-h // f)
            add(f"decode_region_scaled/{k}/f{f}", lambda ctx, k=k, f=f, sw=sw, sh=sh: ctx.decode_region_scaled(
                streams[k], f, sw // 5, sh // 7, max(1, sw // 2), max(1, sh // 3)))
        add(f"encode/{k}", lambda ctx, k=k: ctx.encode(host_img[k], 50, True))

    def decode_batch(ctx, k, n, f=None, off=0):
        w, h, c = shapes[k]
        himg, offs, sizes = batch(k, n)
        if f is None:
            o = out_at(n * w * h * c, off).view(n, h, w, c)
            return ctx.decode_batch(himg, offs, sizes, w, h, c, out=o)
        o = out_at(n * (-(-w // f)) * (-(-h // f)) * c, off).view(n, -(-h // f), -(-w // f), c)
        return ctx.decode_batch_scaled(himg, offs, sizes, w, h, c, f, out=o)

    for k in ("1080p", "gray1024", "rgba512", "odd", "ch5"):
        for n in ((64, 2) if k == "1080p" else (2,)):
            add(f"decode_batch/{k}/n{n}", lambda ctx, k=k, n=n: decode_batch(ctx, k, n))
            for f in (1, 2, 4, 8):
                add(f"decode_batch_scaled/{k}/n{n}/f{f}", lambda ctx, k=k, n=n, f=f: decode_batch(ctx, k, n, f))
    for off in (8, 1):
        add(f"decode_batch/1080p/n2/off{off}", lambda ctx, off=off: decode_batch(ctx, "1080p", 2, None, off))
    for f in (2, 4, 8):
        for off in (16 // f, 8, 1):
            add(f"decode_batch_scaled/1080p/n2/f{f}/off{off}", lambda ctx, f=f, off=off: decode_batch(ctx, "1080p", 2, f, off))

    def decode_mixed(ctx, f=None):
        if f is None:
            return ctx.decode_batch_mixed(mhimg, mhoffs, msizes, mdims, 3, 1920, 1080)
        return ctx.decode_batch_mixed_scaled(mhimg, mhoffs, msizes, mdims, 3, 1920, 1080, f)

    add("decode_batch_mixed", lambda ctx: decode_mixed(ctx))
    for f in (1, 2, 4, 8):
        add(f"decode_batch_mixed_scaled/f{f}", lambda ctx, f=f: decode_mixed(ctx, f))

    def region_batch(ctx, k, n, f=None):
        w, h, c = shapes[k]
        if f is not None:  # (a rectangle of the image scaled by f)
            w, h = -(-w // f), -(-h // f)
        cw, ch = min(224, w // 2), min(224, h // 2)
        himg, offs, sizes = batch(k, n)
        org = torch.tensor([[(37 * i) % (w - cw + 1), (23 * i) % (h - ch + 1)] for i in range(n)], dtype=torch.int32, device=dev)
        if f is not None:
            return ctx.decode_batch_region_scaled(himg, offs, sizes, *shapes[k], f, org, cw, ch)
        return ctx.decode_batch_region(himg, offs, sizes, w, h, c, org, cw, ch)

    for k, n in (("1080p", 64), ("1080p", 2), ("gray1024", 2), ("rgba512", 2), ("odd", 2), ("ch5", 2)):
        add(f"decode_batch_region/{k}/n{n}", lambda ctx, k=k, n=n: region_batch(ctx, k, n))
    add("decode_batch_region_mixed", lambda ctx: ctx.decode_batch_region_mixed(
        mhimg, mhoffs, msizes, mdims, 3, torch.zeros((len(mixed_dims), 2), dtype=torch.int32, device=dev), 64, 48, 1920, 1080))
    for f in (1, 2, 4, 8):
        for k, n in (("1080p", 64), ("1080p", 2), ("gray1024", 2), ("rgba512", 2), ("odd", 2), ("ch5", 2)):
            add(f"decode_batch_region_scaled/{k}/n{n}/f{f}", lambda ctx, k=k, n=n, f=f: region_batch(ctx, k, n, f))
        add(f"decode_batch_region_mixed_scaled/f{f}", lambda ctx, f=f: ctx.decode_batch_region_mixed_scaled(
            mhimg, mhoffs, msizes, mdims, 3, f, torch.zeros((len(mixed_dims), 2), dtype=torch.int32, device=dev), 64 // f, 48 // f,
            1920, 1080))

    for k, n in (("1080p", 64), ("1080p", 2), ("4k", 2), ("8kgray", 1), ("oddw", 2), ("odd", 2), ("ch5", 2), ("rgba512", 2),
                 ("gray1024", 2), ("rgb512", 2)):
        add(f"encode_batch/{k}/n{n}", lambda ctx, k=k, n=n: ctx.encode_batch(px[k][:n].contiguous(), 50, True))
    add("encode_batch/1080p/n2/rgb", lambda ctx: ctx.encode_batch(px["1080p"][:2].contiguous(), 50, False))
    add("encode_batch_mixed", lambda ctx: ctx.encode_batch_mixed(mpx, moffs, mdims, 3, 1920, 1080))

    host_px = px["1080p"][:24].cpu().numpy()
    host_packed = {}

    def enc_host(ctx):
        out, offsets, sizes = ctx.encode_batch_host(host_px, 50, True)
        host_packed["v"] = (out, offsets, sizes)
        return out

    def dec_host(ctx):
        out, offsets, sizes = host_packed["v"]
        return ctx.decode_batch_host(out, offsets, sizes, 1920, 1080, 3)

    for lanes in (1, 3):
        opts = {"host_lanes": lanes, "host_sub_batch_bytes": 24 << 20}
        add(f"encode_batch_host/lanes{lanes}", enc_host, opts)
        add(f"decode_batch_host/lanes{lanes}", dec_host, opts)

    # stages
    for k in ("1080p", "rgba512", "odd", "ch5"):
        w, h, c = shapes[k]
        rows, cols = (h + 7) >> 3, (w + 7) >> 3
        add(f"stage_lowres/{k}", lambda ctx, k=k: ctx.stage_lowres(px[k][:2].contiguous(), True))
        add(f"stage_lres_encode/{k}", lambda ctx, k=k, w=w, h=h: ctx.stage_lres_encode(ctx.stage_lowres(px[k][:2].contiguous()),
                                                                                        w, h, 50))
        add(f"stage_forward/{k}", lambda ctx, k=k: ctx.stage_forward(px[k][:2].contiguous(), ctx.stage_lowres(px[k][:2].contiguous()),
                                                                     50, True))
        add(f"stage_lres_decode/{k}", lambda ctx, k=k, w=w, h=h, c=c: ctx.stage_lres_decode(
            ctx.stage_lres_encode(ctx.stage_lowres(px[k][:2].contiguous()), w, h, 50)[0], w, h, c, unmap))
        add(f"stage_inverse/{k}", lambda ctx, w=w, h=h, c=c, rows=rows, cols=cols: ctx.stage_inverse(
            torch.zeros((2, rows * cols * 64 * c), dtype=torch.uint8, device=dev),
            torch.zeros((2, c, rows, cols), dtype=torch.uint8, device=dev), w, h, c, True, sl, sc, unmap))
    for bs in (0, 4096):
        add(f"stage_huff_compress/bs{bs}", lambda ctx, bs=bs: ctx.stage_huff_compress(huff_data, bs))
        add(f"stage_huff_uncompress/bs{bs}", lambda ctx, bs=bs: ctx.stage_huff_uncompress(
            *huff_packed[bs], huff_data.shape[1], bs))

    # options that change the routing, over the calls they route
    core = [c for c in calls if c[0] in (
        "decode/1080p", "decode/gray1024", "decode_scaled/1080p/f2", "decode_region/1080p", "encode/1080p", "encode/gray1024",
        "decode_batch/1080p/n64", "decode_batch/1080p/n2", "decode_batch_scaled/1080p/n64/f2", "decode_batch/rgba512/n2",
        "decode_batch_region/1080p/n64", "decode_batch_region/1080p/n2", "decode_batch_mixed", "decode_batch_region_mixed",
        "decode_region_scaled/1080p/f2", "decode_batch_region_scaled/1080p/n64/f2", "decode_batch_region_scaled/gray1024/n2/f4",
        "decode_batch_region_mixed_scaled/f2",
        "encode_batch/1080p/n64", "encode_batch/1080p/n2", "encode_batch/4k/n2", "encode_batch/8kgray/n1", "encode_batch_mixed",
        "stage_lowres/1080p", "stage_forward/1080p", "stage_inverse/1080p", "stage_huff_compress/bs4096",
        "stage_huff_uncompress/bs0", "stage_huff_uncompress/bs4096")]
    for opts in ({"force_generic": 1}, {"xform_variant": 1}, {"xform_variant": 4}, {"huff_warp_teams": 0}, {"huff_warp_teams": 2},
                 {"item_lists": 0}, {"max_workspace_bytes": 64 << 20}):
        tag = ",".join(f"{a}={b}" for a, b in opts.items())
        for name, o, fn in core:
            calls.append((f"{name}[{tag}]", {**o, **opts}, fn))

    # ---- tracing ----------------------------------------------------------------------------------
    def context(opts):
        ctx = himg_b200.Context(0)
        for a, b in opts.items():
            ctx.set_option(a, b)
        return ctx

    def finish(ctx):
        ctx.synchronize()
        torch.cuda.synchronize()

    def trace_of(events, multiset):
        streams = {}
        device = [e for e in events if e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset")]
        for e in sorted(device, key=lambda e: e["ts"]):
            a = e.get("args", {})
            rec = [e["cat"], e["name"], a.get("grid"), a.get("block"), a.get("shared memory"), a.get("bytes")]
            streams.setdefault(a.get("stream"), []).append(rec)
        seqs = [sorted(s, key=json.dumps) if multiset else s for s in streams.values()]
        return sorted(seqs, key=json.dumps)

    records = []
    for name, opts, fn in calls:
        ctx = context(opts)
        fn(ctx)  # warm-up: workspace, cached tables, lanes
        finish(ctx)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn(ctx)
            finish(ctx)
        with tempfile.NamedTemporaryFile(suffix=".json") as tmp:
            prof.export_chrome_trace(tmp.name)
            events = json.load(open(tmp.name))["traceEvents"]
        lanes = opts.get("host_lanes", 1) > 1
        records.append({"call": name, "trace": trace_of(events, lanes)})
        ctx.close()
    for rec, (name, opts, fn) in zip(records, calls):
        ctx = context(opts)
        ctx.profile(True)
        fn(ctx)
        finish(ctx)
        ctx.profile_reset()
        before = ctx.launch_count()
        fn(ctx)
        finish(ctx)
        rec["launches"] = ctx.launch_count() - before
        rec["profile"] = sorted((k, v[1]) for k, v in ctx.profile_results().items())
        ctx.close()
    with open(os.path.join(args.out, "trace.jsonl"), "w") as f:
        for rec in records:
            f.write(json.dumps(rec) + "\n")
    kernels = sum(len(s) for r in records for s in r["trace"])
    print(json.dumps({"calls": len(records), "records": kernels, "lib": _native.LIB_PATH}))
    return 0


if __name__ == "__main__":
    sys.exit(main())
