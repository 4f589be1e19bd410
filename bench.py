#!/usr/bin/env python
"""Benchmark of the MapAnything feed-forward inference hot path (BASELINE.json metric: views/sec @518 px).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--views V] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one forward pass over one synthetic V-view 518x518 image-only scene (random-init ViT-L + 24-layer
alternating attention + DPT + pose/scale heads), inputs resident in HBM -> per-view output dicts resident in HBM.
N = 1 runs BASELINE config[1] (8 views, bf16, 1xB200).  N > 1 (one process per GPU under torchrun): ONE scene of 8*N
views sharded by view (8 views per GPU); the 12 global-attention blocks all-gather K/V over NCCL, overlapped with the
attention over the local keys (SURVEY 8e).  Per-GPU view count is fixed ("weak"), but the algorithmic work per view
grows with the scene (global attention is quadratic): config.tflop_per_view and roofline.step_frac carry the
FLOP-normalised picture.  `--multi replicas` runs N independent 8-view scenes instead.  Rank 0 prints ONE JSON line.

  value     views/sec of `model.forward` (device-resident inputs), CUDA events, max over ranks
  e2e       views/sec of `model.infer` from pinned HOST images (H2D inside the timed region, GPU post-processing,
            D2H of pts3d / conf / mask / poses / intrinsics / scale)
  roofline  dominant kernel family = the tcgen05 GEMM (every Linear + implicit-GEMM conv): ALGORITHMIC FLOPs (2MNK of the
            reference layer: unpadded, unsplit K) / its summed launch durations, both taken live with CUDA events around
            each launch on the launching stream inside an instrumented pass of the same step; `kernel` = the kernel that
            took most of that time; peak = MEASURED_PEAKS.json; traffic = DRAM bytes of the dominant launch read from the
            committed ncu summary (profiles/), null when the file is absent
  cpu_baseline  the fp32 CPU oracle (a "port": the reference's uniception dependency is not installable) on the SAME
            scene (all V views when V <= 8), one forward, all host threads
  gpu_eager_baseline  the same oracle moved to the GPU, bf16 autocast + F.scaled_dot_product_attention: what PyTorch's own
            libraries (cuBLASLt, cuDNN) do for this model on this box -- the "kernel to beat" (SURVEY 8d); forward
            (CUDA events) and infer-style end to end (host images in, host numpy post-processing like the reference)
  N > 1     sharded_vs_single_rel (the sharded scene against the same scene run on each GPU alone, before timing; the run
            fails above 1e-2) and `strong` (the fixed 100-view scene of BASELINE config[3] timed on N GPUs and on one)
`--impl reference` times the CPU oracle alone on the same scene (N = 1: the V views of the config), same metric/config.
`--dump-outputs DIR` writes what the last timed forward step returned (see dump_outputs), so that two builds can be compared
output for output on the same arm: an arm's inputs and weights are seeded, identical from run to run.  The two arms are not
comparable this way: the repo arm keeps the constructors' default init, the reference arm draws init_reference_style
weights.  The stream-K GEMM tail adds partial sums in arrival order, so the repo arm's outputs repeat to rounding only
(amplified through the bf16 layers); MA_GEMM_STREAMK=0 makes them repeat bit for bit.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT / "map-anything_b200"))
sys.path.insert(0, str(ROOT))

IMG = 518
METRIC = "views_per_sec_518px"
_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line of the run, on the real stdout (see main())."""
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()

# Algorithmic GFLOP per view (SURVEY.md section 8d / BASELINE.md section 3), D = 768, regressor hidden 128
F_ENC, F_IS_LIN, F_FRAME, F_GLOBAL_PER_VIEW, F_DPT, F_POSE = 1013.6, 467.3, 69.1, 69.1, 308.9, 35.5


def ncu_gemm_traffic():
    """DRAM bytes (read + write) of ONE launch of the dominant GEMM (10960 x 4096 x 1024, bf16 out) from the committed ncu
    summary of this round, or (None, why)."""
    import csv

    for name in ("r2_gemm_raster_ncu.csv", "r1_gemm_2cta_tma_epilogue_ncu.csv"):
        f = ROOT / "profiles" / name
        if not f.exists():
            continue
        rows = list(csv.reader(f.open()))
        hdr = rows[0]
        rd = next(i for i, h in enumerate(hdr) if h.startswith("dram__bytes_read.sum"))
        wr = next(i for i, h in enumerate(hdr) if h.startswith("dram__bytes_write.sum"))
        unit = 1e6 if "Mbyte" in hdr[rd] else 1e9 if "Gbyte" in hdr[rd] else 1e3 if "Kbyte" in hdr[rd] else 1.0
        r = rows[1]
        return (float(r[rd]) + float(r[wr])) * unit, (f"dram bytes read + written by the first launch in profiles/{name} (gemm 10960x4096x1024, ncu "
                                                      f"--set full); algorithmic 120.6 MB (X 22.4 + W 8.4 + Y 89.8)")
    return None, "no ncu summary under profiles/"


def gflop_per_view(v: int) -> float:
    return F_ENC + F_IS_LIN + F_FRAME + F_GLOBAL_PER_VIEW * v + F_DPT + F_POSE


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d.get("bf16_tflops_sustained", 1401.9), d.get("hbm_gbs", 6542.7), "measured"
    return 1400.0, 6650.0, "fallback"  # B200_PROFILING.md fallback (sustained figure)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, pw, mx, reasons = [], [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                pw.append(float(r[2]))
                mx = max(mx, float(r[1]))
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None, "sm_max_mhz": mx or None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


def make_host_views(v: int, seed: int, pin: bool = True):
    import torch

    pin = pin and torch.cuda.is_available()

    g = torch.Generator().manual_seed(seed)
    mean = torch.tensor([0.485, 0.456, 0.406]).view(1, 3, 1, 1)
    std = torch.tensor([0.229, 0.224, 0.225]).view(1, 3, 1, 1)
    out = [((torch.rand(1, 3, IMG, IMG, generator=g) - mean) / std) for _ in range(v)]
    return [x.pin_memory() for x in out] if pin else out


def make_host_geometry(v: int, seed: int, first_view_identity: bool = True, pin: bool = True):
    """SURVEY 8d config C3 inputs per view: pinhole intrinsics (f ~ U[400,600], c = 259), depth_z ~ U[1,4] m,
    cam2world pose (view 0 identity), metric scale.  Pinned host tensors."""
    import torch

    g = torch.Generator().manual_seed(seed)
    out = []
    for i in range(v):
        f = float(torch.empty(1).uniform_(400, 600, generator=g))
        k = torch.tensor([[[f, 0, 259.0], [0, f, 259.0], [0, 0, 1.0]]])
        d = torch.empty(1, IMG, IMG, 1).uniform_(1.0, 4.0, generator=g)
        q = torch.randn(4, generator=g) * 0.2 + torch.tensor([0.0, 0.0, 0.0, 1.0])
        t = torch.randn(3, generator=g)
        if i == 0 and first_view_identity:
            q, t = torch.tensor([0.0, 0.0, 0.0, 1.0]), torch.zeros(3)
        x, y, z, w = (q / q.norm()).tolist()
        pose = torch.eye(4)
        pose[:3, :3] = torch.tensor([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])
        pose[:3, 3] = t
        e = {"intrinsics": k, "depth_z": d, "camera_poses": pose[None], "is_metric_scale": torch.tensor([True])}
        out.append({n: x.pin_memory() for n, x in e.items()} if pin and torch.cuda.is_available() else e)
    return out


DUMP_BYTES = 64 << 20  # all arrays of one --dump-outputs together


def dump_outputs(preds, out_dir: str) -> None:
    """Writes the per-view output dicts of one forward step as <out_dir>/<key>.npy in float32, views stacked on axis 0
    (masks as 0 / 1).  When everything would exceed DUMP_BYTES, the per-pixel maps keep one fixed, seeded sample of pixel
    positions (the same for every view and key, in raster order); per-view vectors are always written whole."""
    import numpy as np
    import torch

    arrays = {k: torch.cat([p[k] for p in preds]).float().cpu().numpy() for k in preds[0]}
    dense = [k for k, a in arrays.items() if a.shape[1:3] == (IMG, IMG)]
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        per_pixel = sum(arrays[k].nbytes for k in dense) // (IMG * IMG)
        keep = (DUMP_BYTES - (total - per_pixel * IMG * IMG)) // per_pixel
        pix = np.sort(np.random.default_rng(0).choice(IMG * IMG, size=keep, replace=False))
        for k in dense:
            a = arrays[k]
            arrays[k] = a.reshape(a.shape[0], IMG * IMG, *a.shape[3:])[:, pix]
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for k, a in arrays.items():
        np.save(out / f"{k}.npy", a)


def bench_config(v: int, gpus: int, multi: str, multimodal: bool, shard: bool):
    """The `config` object: identical for both arms of the same invocation."""
    v_scene = v * gpus if shard else v
    return {"workload": workload_name(v, gpus, multi, multimodal), "views": v * gpus, "views_per_gpu": v,
            "scene_views": v_scene, "tflop_per_view": gflop_per_view(v_scene) / 1e3, "image": IMG, "weights": "random-init",
            "parallelism": "single" if gpus == 1 else (f"view-shard x{gpus} + K/V all-gather" if shard else f"replicas x{gpus}"),
            "l2": "per-step activations (>1 GB) exceed the 126 MB L2; no explicit flush"}


def build_oracle():
    from oracle.config import mapanything_config
    from oracle.model import MapAnythingOracle
    from oracle.weights import init_reference_style

    return init_reference_style(MapAnythingOracle(**mapanything_config()).eval(), 0)


def run_reference(args):
    """The reference arm: the fp32 CPU oracle of the path on the host cores, all threads, on the SAME scene as the repo arm
    at N = 1 (all args.views views; the warm-up shrinks to fit a time budget, the timed steps are --steps).  For N > 1 the
    repo arm's scene has views x N views; the CPU arm runs the first `args.views` of them and says so."""
    import torch

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    scene = args.views * args.gpus if args.multi == "shard" else args.views
    sample_views = args.views
    model = build_oracle()
    imgs = make_host_views(sample_views, 1234)
    extra = make_host_geometry(sample_views, 4321) if args.multimodal else [{} for _ in range(sample_views)]
    if args.multimodal:
        from oracle import inference as OI

        views = OI.preprocess_views([{"img": im, "data_norm_type": ["dinov2"], **e} for im, e in zip(imgs, extra)])
        model.geometric_input_config.update({"overall_prob": 1.0, "dropout_prob": 0.0, "ray_dirs_prob": 1.0, "depth_prob": 1.0,
                                             "cam_prob": 1.0})
    else:
        views = [{"img": im, "data_norm_type": ["dinov2"]} for im in imgs]
    preds = []   # --dump-outputs: what the latest step returned

    def step():
        preds.clear()
        t0 = time.perf_counter()
        with torch.no_grad():
            out = model(views)
        t = time.perf_counter() - t0
        if args.dump_outputs:
            preds.append(out)
        return t

    t_first = step()  # warm-up (also sizes the rest of the warm-up: a CPU step takes tens of seconds)
    budget = 200.0
    warm = max(0, min(args.warmup - 1, int(0.25 * budget / max(t_first, 1e-3))))
    for _ in range(warm):
        step()
    steps = args.steps
    times = [step() for _ in range(steps)]
    if preds:
        dump_outputs(preds.pop(), args.dump_outputs)
    t = sum(times) / len(times)
    vps = sample_views / t
    same = sample_views == scene
    sample = (f"{'all ' if same else 'the first '}{sample_views} of the {scene} views of the scene (518x518, full ViT-L + 24-layer "
              f"info sharing + DPT), fp32, {steps} timed step(s) of {t:.2f} s")
    line = {
        "impl": "reference", "metric": METRIC, "value": vps, "unit": "views/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warm + 1, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": bench_config(args.views, args.gpus, args.multi, args.multimodal, args.gpus > 1 and args.multi == "shard"),
        "same_scene_as_repo_arm": same,
        "cpu_baseline": {"value": vps, "unit": "views/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": vps, "unit": "views/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def workload_name(v: int, gpus: int, multi: str = "shard", multimodal: bool = False) -> str:
    if multimodal:
        return (f"MapAnything multi-modal (images+intrinsics+poses+depth), {v * gpus} views 518x518 bf16 on {gpus}xB200"
                + (" (BASELINE config[2])" if v * gpus == 24 else ""))
    if gpus == 1:
        return f"MapAnything image-only, {v} views 518x518 bf16 on 1xB200 (BASELINE config[1])" if v == 8 else \
            f"MapAnything image-only, {v} views 518x518 bf16 on 1xB200"
    if multi == "replicas":
        return f"MapAnything image-only, {v} views 518x518 bf16 per GPU, {gpus} independent scenes on {gpus}xB200"
    return (f"MapAnything image-only, ONE scene of {v * gpus} views 518x518 bf16 sharded by view over {gpus}xB200 "
            f"({v} views per GPU; global attention = local queries x all-gathered K/V over NCCL); algorithmic work per view "
            f"grows with the scene: {gflop_per_view(v * gpus) / 1e3:.2f} TFLOP/view vs {gflop_per_view(v) / 1e3:.2f} at {v} views")


def rel_err(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm().clamp(min=1e-12)).item()


def sharded_vs_single(model, dev, rank, world, V):
    """Correctness of the sharded path, visible to the driver: every rank runs the WHOLE 8*N-view scene alone on its GPU
    (view sharding off) and compares its own views' outputs of the sharded pass with it.  Max over keys / views / ranks."""
    import torch
    import torch.distributed as dist

    full_views = [{"img": im.to(dev), "data_norm_type": ["dinov2"]} for r in range(world) for im in make_host_views(V, 1234 + r)]
    model.disable_view_sharding()
    full = model(full_views)
    model.enable_view_sharding(views_per_rank=[V] * world)
    part = model(full_views[rank * V:(rank + 1) * V])
    worst = 0.0
    for i, p in enumerate(part):
        f = full[rank * V + i]
        for k in ("pts3d", "depth_along_ray", "ray_directions", "conf", "cam_trans", "cam_quats", "metric_scaling_factor"):
            worst = max(worst, rel_err(p[k], f[k]))
    t = torch.tensor([worst], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    del full, part, full_views
    torch.cuda.empty_cache()
    return t.item()


def strong_scaling_record(model, dev, rank, world, timed, peak_tf, scene=100, steps=3):
    """BASELINE config[3]: ONE fixed 100-view scene on N GPUs (13,13,...,12 views per rank) against the same scene on one
    GPU of the same box, both timed here; plus the time the compute stream spent blocked on the K/V all-gather."""
    import torch
    import torch.distributed as dist

    from mapanything_b200.sharding import partition_views

    counts = partition_views(scene, world)
    lo = sum(counts[:rank])
    g = torch.Generator().manual_seed(777)
    mean = torch.tensor([0.485, 0.456, 0.406]).view(1, 3, 1, 1)
    std = torch.tensor([0.229, 0.224, 0.225]).view(1, 3, 1, 1)
    imgs = [((torch.rand(1, 3, IMG, IMG, generator=g) - mean) / std) for _ in range(scene)]  # same scene on every rank
    mine = [{"img": im.to(dev), "data_norm_type": ["dinov2"]} for im in imgs[lo:lo + counts[rank]]]
    model.enable_view_sharding(views_per_rank=counts)
    eng = model.engine()
    for _ in range(2):
        model(mine)
    eng.ag_wait_events = []
    ms_n = timed(lambda: model(mine), steps) / steps
    torch.cuda.synchronize()
    waits = [a.elapsed_time(b) for a, b in eng.ag_wait_events]
    eng.ag_wait_events = None
    exposed = torch.tensor([sum(waits) / max(len(waits), 1)], device=dev)
    exposed_min = exposed.clone()
    dist.all_reduce(exposed, op=dist.ReduceOp.MAX)
    dist.all_reduce(exposed_min, op=dist.ReduceOp.MIN)
    # end to end: infer() from pinned host images, every rank reads its views' point maps / masks / poses back
    host = [im.pin_memory() for im in imgs[lo:lo + counts[rank]]]

    host_out = []   # pinned result buffers, allocated by the first call

    def e2e():
        preds = model.infer([{"img": im, "data_norm_type": ["dinov2"]} for im in host])
        srcs = [p[k] for p in preds for k in ("pts3d", "conf", "mask", "camera_poses", "intrinsics")]
        if not host_out:
            host_out.extend(torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in srcs)
        for dst, src in zip(host_out, srcs):
            dst.copy_(src, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return host_out

    e2e()
    ms_e2e = timed(e2e, 2) / 2
    # the same scene on ONE GPU of this box (rank 0; the other ranks idle at the barrier)
    model.disable_view_sharding()
    ms_1 = torch.zeros(1, device=dev)
    if rank == 0:
        allv = [{"img": im.to(dev), "data_norm_type": ["dinov2"]} for im in imgs]
        model(allv)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(2):
            model(allv)
        e.record()
        torch.cuda.synchronize()
        ms_1[0] = s.elapsed_time(e) / 2
        del allv
    dist.broadcast(ms_1, src=0)
    torch.cuda.empty_cache()
    tf_scene = scene * gflop_per_view(scene) * 1e9 / 1e12  # TFLOP per scene
    return {
        "scene_views": scene, "views_per_rank": counts, "steps": steps,
        "ms_per_step": ms_n, "views_per_s": scene / (ms_n * 1e-3),
        "e2e_ms_per_step": ms_e2e, "e2e_views_per_s": scene / (ms_e2e * 1e-3),
        "single_gpu_ms_per_step": ms_1.item(), "single_gpu_views_per_s": scene / (ms_1.item() * 1e-3),
        "speedup_vs_single_gpu": ms_1.item() / ms_n, "efficiency": ms_1.item() / ms_n / world,
        "per_gpu_step_frac": tf_scene / world / (ms_n * 1e-3) / peak_tf,
        "single_gpu_step_frac": tf_scene / (ms_1.item() * 1e-3) / peak_tf,
        "allgather_exposed_ms_per_global_layer": exposed_min.item(),
        "allgather_wait_ms_per_global_layer_max_over_ranks": exposed.item(),
        "load_balance_bound": scene / (max(counts) * world),
        "allgather_note": "time the compute stream waited for the NCCL K/V all-gather after finishing the local-key attention "
                          "(CUDA events around work.wait(), mean over 12 layers x steps).  The all-gather is a collective: a rank "
                          "with fewer views (12 instead of 13) reaches it early and waits for the others, so the MIN over ranks "
                          "(the slowest rank's wait) is the exposed communication and the MAX is mostly load imbalance; "
                          "tools/bench_allgather.py measures the same exchange in isolation (8 GPUs, 13 views per rank: 0.68 ms "
                          "alone, 0.003 ms exposed behind the 1.34 ms local attention)",
    }


def gpu_eager_baseline(oracle_model, dev, host_imgs, host_extra, d2h_keys, multimodal, steps=3):
    """What PyTorch's own libraries do for this model on this GPU: the oracle under torch.autocast(bf16) (the reference's
    infer(use_amp=True, amp_dtype="bf16") wiring, model.py:2092-2095) with F.scaled_dot_product_attention, cuBLASLt GEMMs
    and cuDNN convolutions.  Forward: device-resident inputs, CUDA events.  e2e: oracle.infer() from host images incl.
    its host-side (numpy) post-processing, as the reference does it, and the same D2H reads as the repo arm."""
    import torch

    import oracle.vit as ov
    from oracle import inference as OI

    ov.USE_SDPA = True
    try:
        m = oracle_model.to(dev)
        views = [{"img": im.to(dev), "data_norm_type": ["dinov2"], **{k: x.to(dev) for k, x in e.items()}}
                 for im, e in zip(host_imgs, host_extra)]
        if multimodal:
            views = OI.preprocess_views(views)
            m.geometric_input_config.update({"overall_prob": 1.0, "dropout_prob": 0.0, "ray_dirs_prob": 1.0, "depth_prob": 1.0,
                                             "cam_prob": 1.0})
        with torch.no_grad():
            for _ in range(2):
                m(views, amp_bf16=True)
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(steps):
                m(views, amp_bf16=True)
            e.record()
            torch.cuda.synchronize()
            ms = s.elapsed_time(e) / steps

            def e2e():
                hv = [{"img": im, "data_norm_type": ["dinov2"], **ex} for im, ex in zip(host_imgs, host_extra)]
                preds = m.infer(hv)
                outs = [p[k].to("cpu") for p in preds for k in d2h_keys]
                torch.cuda.synchronize()
                return outs

            e2e()
            t0 = time.perf_counter()
            for _ in range(steps):
                e2e()
            ms_e2e = (time.perf_counter() - t0) / steps * 1e3
        v = len(host_imgs)
        return {"value": v / (ms * 1e-3), "unit": "views/s", "ms_per_step": ms,
                "e2e": {"value": v / (ms_e2e * 1e-3), "unit": "views/s", "ms_per_step": ms_e2e},
                "what": "oracle (PyTorch modules) on cuda, torch.autocast(bf16) over encoder + info sharing, heads fp32/TF32-off as "
                        "the reference, F.scaled_dot_product_attention; same views; e2e = oracle.infer from host images with "
                        "the reference's host-side numpy post-processing", "steps": steps}
    finally:
        ov.USE_SDPA = False
        oracle_model.to("cpu")
        torch.cuda.empty_cache()


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from mapanything_b200 import MapAnything, mapanything_config, ops
    from mapanything_b200 import _lib

    _lib.load()  # fail loudly if the CUDA library is missing
    torch.manual_seed(0)
    model = MapAnything(**mapanything_config()).to(dev).eval()  # random-init weights of the architecture
    V = args.views  # views per GPU
    shard = world > 1 and args.multi == "shard"
    v_scene = V * world if shard else V  # views of the scene each forward pass works on
    host_imgs = make_host_views(V, 1234 + rank)
    host_extra = make_host_geometry(V, 4321 + rank, first_view_identity=(rank == 0)) if args.multimodal else [{} for _ in range(V)]
    dev_views = [{"img": im.to(dev), "data_norm_type": ["dinov2"]} for im in host_imgs]
    if args.multimodal:
        # forward() takes the model's internal keys: preprocess once (device resident), enable the geometric inputs
        from mapanything_b200.preprocess import preprocess_input_views_for_inference

        dev_views = preprocess_input_views_for_inference(
            [{**v, **{k: x.to(dev) for k, x in e.items()}} for v, e in zip(dev_views, host_extra)])
        model.geometric_input_config.update({"overall_prob": 1.0, "dropout_prob": 0.0, "ray_dirs_prob": 1.0, "depth_prob": 1.0,
                                             "cam_prob": 1.0})
    model.engine()
    if args.cuda_graph and world == 1:
        model.enable_cuda_graphs()
    sharded_rel = None
    if shard:
        sharded_rel = sharded_vs_single(model, dev, rank, world, V)   # leaves view sharding enabled
        if sharded_rel > 1e-2:
            if rank == 0:
                emit({"error": "sharded scene deviates from the single-GPU scene", "sharded_vs_single_rel": sharded_rel})
            dist.barrier()
            dist.destroy_process_group()
            sys.exit(3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def fwd_step():
        return model(dev_views)

    kept = []   # --dump-outputs: what the latest timed forward step returned

    def fwd_step_kept():
        kept.clear()   # the previous step's outputs are freed before this step runs, as with fwd_step
        kept.append(fwd_step())

    d2h_keys = ("pts3d", "conf", "mask", "camera_poses", "intrinsics", "metric_scaling_factor")

    host_out = []   # pinned result buffers, allocated on the first step and reused (what a serving loop does)

    def e2e_step():
        views = [{"img": im, "data_norm_type": ["dinov2"], **e} for im, e in zip(host_imgs, host_extra)]  # pinned HOST tensors
        preds = model.infer(views)
        srcs = [p[k] for p in preds for k in d2h_keys]
        if not host_out:
            host_out.extend(torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in srcs)
        for dst, src in zip(host_out, srcs):
            dst.copy_(src, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return host_out

    def timed(fn, steps):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            fn()
        e.record()
        barrier()
        ms = s.elapsed_time(e)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    if args.profile_mode:  # short, un-reported run for ncu: one warm-up step, one step, nothing else
        fwd_step()
        torch.cuda.synchronize()
        fwd_step()
        torch.cuda.synchronize()
        if rank == 0:
            emit({"profile_mode": True, "views": V, "launches_per_step": ops.LAUNCHES // 2})
        return
    for _ in range(max(args.warmup, 3)):
        fwd_step()
    with ClockSampler(local_rank) as clocks:
        launches0 = ops.LAUNCHES
        ms_fwd = timed(fwd_step_kept if args.dump_outputs else fwd_step, args.steps)
        launches = ops.LAUNCHES - launches0
        # instrumented pass of the same step for the per-kernel roofline (events around every GEMM launch)
        # (single stream for this pass: with the encoder's two view groups on two streams the kernels overlap and the
        # per-launch event times would count the time spent waiting for SMs)
        eng = model.engine()
        n_streams, eng.encoder_streams = eng.encoder_streams, 1
        graphs, model._graphs = model._graphs, None   # the instrumented pass launches kernel by kernel
        ops.PROFILE = []
        barrier()
        fwd_step()
        torch.cuda.synchronize()
        prof, ops.PROFILE = ops.PROFILE, None
        model._graphs = graphs
        eng.encoder_streams = n_streams
        for _ in range(2):
            e2e_step()
        ms_e2e = timed(e2e_step, args.steps)
    if kept and rank == 0:
        dump_outputs(kept[0], args.dump_outputs)
    kept.clear()
    ms_step = ms_fwd / args.steps
    vps = world * V / (ms_step * 1e-3)
    e2e_ms_step = ms_e2e / args.steps
    e2e_vps = world * V / (e2e_ms_step * 1e-3)

    peak_tf, peak_hbm, peak_src = measured_peaks()
    if os.environ.get("MA_BENCH_DUMP") and rank == 0:  # per-launch list (family, algorithmic flops, ms) for offline analysis
        Path(os.environ["MA_BENCH_DUMP"]).write_text(json.dumps([[n, f, s.elapsed_time(e), t] for n, f, s, e, t in prof]))
    fam = {}
    for name, flops, s, e, _tag in prof:
        d = fam.setdefault(name, [0.0, 0.0, 0])
        d[0] += flops
        d[1] += s.elapsed_time(e)
        d[2] += 1
    gemm = [a + b for a, b in zip(fam.get("gemm", [0.0, 1e-9, 0]), fam.get("conv3x3", [0.0, 0.0, 0]))]  # one kernel family
    achieved = gemm[0] / (gemm[1] * 1e-3) / 1e12
    by_kernel = {}
    for name, flops, s, e, tag in prof:
        if name in ("gemm", "conv3x3") and "|" in tag:
            d = by_kernel.setdefault(tag.split("|")[1], [0.0, 0.0, 0])
            d[0] += flops
            d[1] += s.elapsed_time(e)
            d[2] += 1
    top_kernel = max(by_kernel.items(), key=lambda kv: kv[1][1]) if by_kernel else ("gemm_bf16_2cta_kernel<256>", [0.0, 1e-9, 0])
    traffic, traffic_note = ncu_gemm_traffic()
    step_tf = V * gflop_per_view(v_scene) * 1e9 / (ms_step * 1e-3) / 1e12  # per GPU

    outs = e2e_step()  # every rank: the sharded step is collective
    d2h = sum(o.numel() * o.element_size() for o in outs) * world
    h2d = (sum(im.numel() * 4 for im in host_imgs)
           + sum(x.numel() * x.element_size() for e in host_extra for x in e.values())) * world
    strong = None
    if shard and not args.multimodal and not args.no_strong:
        strong = strong_scaling_record(model, dev, rank, world, timed, peak_tf)
        model.enable_view_sharding(views_per_rank=[V] * world)
    cpu = eager = None
    if rank == 0 and world == 1 and not args.no_cpu:  # host + GPU-library baselines are reported at N = 1 only
        oracle_model = build_oracle()
        cpu = cpu_baseline(V, oracle_model, args.multimodal)
        if not args.no_eager:
            eager = gpu_eager_baseline(oracle_model, dev, host_imgs, host_extra, d2h_keys, args.multimodal)
        del oracle_model
    if rank == 0:
        line = {
            "metric": METRIC, "value": vps, "unit": "views/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": bench_config(V, world, args.multi, args.multimodal, shard),
            "roofline": {
                "bound": "tensor", "kernel": top_kernel[0], "achieved": achieved, "peak": peak_tf,
                "unit": "TFLOP/s", "frac": achieved / peak_tf, "traffic": traffic, "traffic_note": traffic_note,
                "peak_source": peak_src, "flops": "algorithmic: 2*M*N*K of the reference layers (unpadded, unsplit K)",
                "family": "every tcgen05 GEMM / implicit-GEMM conv launch of the step (one kernel template, two tile forms)",
                "launches": gemm[2], "kernel_ms_per_step": gemm[1], "gemm_share_of_step": gemm[1] / ms_step,
                "top_kernel": {"name": top_kernel[0], "launches": top_kernel[1][2], "ms_per_step": top_kernel[1][1],
                               "achieved": top_kernel[1][0] / (top_kernel[1][1] * 1e-3) / 1e12},
                "attention": ({"achieved": fam["attention"][0] / (fam["attention"][1] * 1e-3) / 1e12,
                               "frac": fam["attention"][0] / (fam["attention"][1] * 1e-3) / 1e12 / peak_tf,
                               "ms_per_step": fam["attention"][1]} if "attention" in fam else None),
                "step_achieved_tflops": step_tf, "step_frac": step_tf / peak_tf,
                "families_ms": {k: round(v[1], 3) for k, v in fam.items()},
            },
            "cpu_baseline": cpu,
            "gpu_eager_baseline": eager,
            "sharded_vs_single_rel": sharded_rel,
            "strong": strong,
            "e2e": {"value": e2e_vps, "unit": "views/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms_step},
            "gpu_launches": launches,
            "clocks": clocks.summary(),
            "cuda_graph": bool(args.cuda_graph and world == 1),
        }
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def cpu_baseline(v: int, model, multimodal: bool):
    """fp32 CPU oracle on the same scene (all v views for v <= 8, else the first 8): one forward, all host threads."""
    import torch

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    n = min(v, 8)
    imgs = make_host_views(n, 1234)
    if multimodal:
        from oracle import inference as OI

        views = OI.preprocess_views([{"img": im, "data_norm_type": ["dinov2"], **e} for im, e in zip(imgs, make_host_geometry(n, 4321))])
        model.geometric_input_config.update({"overall_prob": 1.0, "dropout_prob": 0.0, "ray_dirs_prob": 1.0, "depth_prob": 1.0,
                                             "cam_prob": 1.0})
    else:
        views = [{"img": im, "data_norm_type": ["dinov2"]} for im in imgs]
    t0 = time.perf_counter()
    with torch.no_grad():
        model(views)
    t = time.perf_counter() - t0
    return {"value": n / t, "unit": "views/s", "cores": cores, "kind": "port",
            "sample": f"{'all ' if n == v else 'the first '}{n} of the {v} views, one fp32 forward of the full model on the host ({t:.1f} s)"}


def main():
    # rank 0 prints exactly ONE line on stdout
    # ... and everything else any library writes to fd 1 (NCCL's banner and INFO lines among them) goes to stderr: the
    # process-wide stdout is re-pointed at stderr and the JSON line is written to a private duplicate of the real stdout
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":   # keep NCCL's init lines (transports, NVLS) visible
        os.environ["NCCL_DEBUG"] = "INFO"
        os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--views", type=int, default=8, help="views per GPU")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--multimodal", action="store_true",
                    help="BASELINE config[2]: every view also carries intrinsics, depth and a camera pose (use with --views 24)")
    ap.add_argument("--multi", default="shard", choices=["shard", "replicas"],
                    help="N > 1: one scene of views*N views sharded by view (default) or N independent scenes")
    ap.add_argument("--no-eager", action="store_true", help="skip the GPU-eager (PyTorch library) baseline leg")
    ap.add_argument("--no-cpu", action="store_true", help="A/B runs only: skip the CPU baseline leg too (cpu_baseline: null)")
    ap.add_argument("--cuda-graph", action="store_true",
                    help="N = 1: replay the step as one captured CUDA graph (model.enable_cuda_graphs(); small scenes are launch-bound)")
    ap.add_argument("--no-strong", action="store_true", help="N > 1: skip the fixed 100-view strong-scaling record")
    ap.add_argument("--profile-mode", action="store_true", help="1 warm-up + 1 step only, for ncu captures (prints no bench line)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed forward step (rank 0's views) as DIR/<key>.npy, float32, "
                         f"at most {DUMP_BYTES >> 20} MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.profile_mode:
        ap.error("--profile-mode times nothing: there are no outputs for --dump-outputs")
    if args.impl == "reference":
        # torchrun exports OMP_NUM_THREADS=1; the reference arm gets every host core (set before torch is imported)
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
        os.environ["MKL_NUM_THREADS"] = str(os.cpu_count() or 1)
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
