"""GPU JPEG decode (csrc/jpeg.cu) against Pillow on seeded synthetic camera frames.

    python tools/bench_jpeg.py [--frames 64] [--iters 5] [--out profiles/r3_bench_jpeg.json]

Frames: smooth noise fields encoded by Pillow at 1920x1080 and 4032x3024, 4:2:0 q95 and 4:4:4 q90.  Per class:
  * gpu_ms_per_frame: ma_jpeg_decode over a batch of `--frames` different frames (the blobs already on the device), CUDA
    events, steady state; the batch's coefficients + planes + RGB outputs exceed the 126 MB L2 for every class;
  * parse_ms_per_frame: ma_jpeg_parse on the host (one thread);
  * pillow_ms_per_frame: np.asarray(PIL.Image.open(f).convert("RGB")) on one thread;
  * load_images_s: wall time of load_images on a folder of `--frames` such files, through the GPU route and with the
    GPU route disabled (every file through Pillow, as before), same process.
Prints one JSON object and writes it to --out.  Needs a CUDA device; reads the card name and power limit itself.
"""
from __future__ import annotations

import argparse
import ctypes as C
import io
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "map-anything_b200")]


def frame(W, H, seed):
    rng = np.random.default_rng(seed)
    lo = rng.normal(0, 1, (H // 16 + 2, W // 16 + 2, 3)).astype(np.float32)
    import torch

    up = torch.nn.functional.interpolate(torch.from_numpy(lo).permute(2, 0, 1)[None], size=(H, W), mode="bicubic",
                                         align_corners=False)[0].permute(1, 2, 0).numpy()
    img = 128 + 60 * up + rng.normal(0, 6, (H, W, 3))
    return np.clip(img, 0, 255).astype(np.uint8)


def encode(a, subsampling, q):
    import PIL.Image

    b = io.BytesIO()
    PIL.Image.fromarray(a).save(b, "JPEG", quality=q, subsampling=subsampling)
    return b.getvalue()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import PIL.Image
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_jpeg.py needs a CUDA device")
    from mapanything_b200 import _lib, image as MI

    lib = _lib.load()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    res = {"gpu": smi[0] if smi else "unknown", "frames": args.frames, "classes": []}
    base = {}
    for W, H in ((1920, 1080), (4032, 3024)):
        base[(W, H)] = [frame(W, H, s) for s in range(4)]
    for (W, H), (ss, q, name) in [(wh, c) for wh in base for c in ((2, 95, "420_q95"), (0, 90, "444_q90"))]:
        # 4 distinct fields, each shifted per frame so that every one of the frames is a different stream
        files = [encode(np.roll(base[(W, H)][i % 4], 7 * i, axis=1), ss, q) for i in range(args.frames)]
        t0 = time.perf_counter()
        parsed = [MI.jpeg_parse(f) for f in files]
        parse_ms = (time.perf_counter() - t0) * 1e3 / len(files)
        n = len(files)
        offs = np.cumsum([0] + [p[1].size for p in parsed])
        d_blobs = torch.from_numpy(np.concatenate([p[1] for p in parsed])).cuda()
        infos = (_lib.JpegInfo * n)(*[p[0] for p in parsed])
        outs = torch.empty(n, H, W, 3, dtype=torch.uint8, device="cuda")
        ws = C.c_int64(0)
        _lib.check(lib.ma_jpeg_workspace(infos, n, C.byref(ws)), "ma_jpeg_workspace")
        work = torch.empty(ws.value, dtype=torch.uint8, device="cuda")
        status = torch.empty(n, dtype=torch.int32, device="cuda")
        args_c = (d_blobs.data_ptr(), (C.c_int64 * n)(*[int(x) for x in offs[:-1]]), infos, n,
                  (C.c_void_p * n)(*[outs[i].data_ptr() for i in range(n)]), (C.c_int32 * n)(*([1] * n)),
                  work.data_ptr(), ws.value, status.data_ptr())

        def run():
            _lib.check(lib.ma_jpeg_decode(*args_c, torch.cuda.current_stream().cuda_stream), "ma_jpeg_decode")

        run()
        torch.cuda.synchronize()
        ok = int((status == 0).sum())
        ref0 = np.asarray(PIL.Image.open(io.BytesIO(files[0])).convert("RGB"))
        exact = bool(np.array_equal(outs[0].cpu().numpy(), ref0))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        times = []
        for _ in range(args.iters):
            e0.record()
            run()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / n)
        t0 = time.perf_counter()
        k = min(n, 8)
        for f in files[:k]:
            np.asarray(PIL.Image.open(io.BytesIO(f)).convert("RGB"))
        pil_ms = (time.perf_counter() - t0) * 1e3 / k
        # load_images on a folder of these files, both routes
        with tempfile.TemporaryDirectory() as d:
            for i, f in enumerate(files):
                Path(d, f"{i:03d}.jpg").write_bytes(f)
            MI.load_images(d)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            MI.load_images(d)
            torch.cuda.synchronize()
            t_gpu = time.perf_counter() - t0
            keep = MI._open_for_gpu
            MI._open_for_gpu = lambda p: None
            try:
                t0 = time.perf_counter()
                MI.load_images(d)
                torch.cuda.synchronize()
                t_pil = time.perf_counter() - t0
            finally:
                MI._open_for_gpu = keep
        cls = dict(name=f"{W}x{H}_{name}", mean_file_bytes=int(np.mean([len(f) for f in files])),
                   workspace_bytes=ws.value, frames_decoded=ok, first_frame_equals_pillow=exact,
                   gpu_ms_per_frame=round(float(np.median(times)), 4), gpu_ms_per_frame_all=[round(t, 4) for t in times],
                   parse_ms_per_frame=round(parse_ms, 3), pillow_ms_per_frame=round(pil_ms, 3),
                   load_images_gpu_route_s=round(t_gpu, 3), load_images_pillow_route_s=round(t_pil, 3))
        print(json.dumps(cls), flush=True)
        res["classes"].append(cls)
        del work, outs, d_blobs
        torch.cuda.empty_cache()
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
