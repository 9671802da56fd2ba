#!/usr/bin/env python
"""Cost of the surface distances (btpost_surface_distance, PostConfig.with_surface_dist) on the synthetic workload.

    python scripts/surface_timing.py [--reps 3]

1. Kernel time of btpost_surface_distance on 64 synthetic projector masks (the mask stage's seg_mask of the synthetic
   batch, whose edges are dense) against their GT masks, at 640^2 and 1024^2: CUDA events around 50 back-to-back calls,
   then one torch.profiler pass for the split over the four kernels.
2. Step time at 64 x 640^2 with and without with_surface_dist, alternated: serial (PostProcessor.run back to back on one
   stream) and pipelined (Pipeline, 4 batches in flight, captured steps).
Prints the card's name and power limit first, then one JSON line per measurement."""
import argparse, ctypes as C, json, subprocess, sys
from pathlib import Path
ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "multitask-bonetumor-yolo_b200")]
import torch
from btpost import Pipeline, PostConfig, PostProcessor, _lib, synth

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=3)
args = ap.parse_args()
dev = torch.device("cuda:0")
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip(), flush=True)
L = _lib.load()
B, N = 64, 50


def synthetic(S):
    b = synth.make_batch_device(synth.SynthConfig(batch=B, img_size=S, seed=20262), dev)
    return b


def masks_of(b, S):
    pp = PostProcessor(PostConfig(batch=B, img_size=S, with_seg_mask=True, gt_mode=1), dev)
    out = pp.run(b["head"], b["protos"], b["det_boxes_gt"], b["masks_gt"], b["proj_weight"], b["proj_bias"])
    torch.cuda.synchronize()
    return out["seg_mask"].clone(), b["masks_gt"].contiguous()


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


for S in (640, 1024):
    b = synthetic(S)
    pred, gt = masks_of(b, S)
    nb = C.c_size_t()
    _lib.check(L.btpost_surface_bytes(B, S, C.byref(nb)), "btpost_surface_bytes")
    scratch = torch.empty(nb.value, dtype=torch.uint8, device=dev)
    outs = [torch.empty(B, dtype=torch.float32, device=dev) for _ in range(3)]
    acc = torch.zeros(4, dtype=torch.int64, device=dev)
    st = torch.cuda.current_stream().cuda_stream

    def call():
        _lib.check(L.btpost_surface_distance(B, S, C.c_void_p(pred.data_ptr()), C.c_void_p(gt.data_ptr()), _lib.MASK_U8,
                                             *(C.c_void_p(t.data_ptr()) for t in outs), C.c_void_p(acc.data_ptr()),
                                             C.c_void_p(scratch.data_ptr()), C.c_size_t(nb.value), C.c_void_p(st)), "surface")
    ms = [timed(call, N) for _ in range(args.reps)]
    print(json.dumps({"what": "btpost_surface_distance", "batch": B, "img": S, "scratch_bytes": nb.value, "ms_per_call": ms,
                      "pred_fg_fraction": float((pred != 0).float().mean()), "mean_hd": float(outs[0].nanmean()),
                      "mean_hd95": float(outs[1].nanmean()), "mean_assd": float(outs[2].nanmean())}), flush=True)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(10):
            call()
        torch.cuda.synchronize()
    split = {}
    for ev in prof.key_averages():
        if "surface" in ev.key:
            split[ev.key.split("surface_")[1].split("_kernel")[0]] = round(ev.device_time_total / ev.count / 1e3, 4)
    print(json.dumps({"what": "kernel split (profiler, ms per call)", "img": S, "split": split}), flush=True)
    del scratch, pred, gt, b
    torch.cuda.empty_cache()

S = 640
b = synthetic(S)
procs = {f: PostProcessor(PostConfig(batch=B, img_size=S, gt_mode=1, with_seg_mask=True, with_surface_dist=f), dev)
         for f in (False, True)}
pipes = {f: Pipeline(PostConfig(batch=B, img_size=S, gt_mode=1, with_seg_mask=True, with_surface_dist=f), dev, depth=4,
                     proj_weight=b["proj_weight"], proj_bias=float(b["proj_bias"])) for f in (False, True)}
for p in pipes.values():
    for inp in p.inputs:
        for k in ("head", "protos", "masks_gt"):
            inp[k].copy_(b[k].reshape(inp[k].shape))
        rows = b["det_boxes_gt"].shape[0]
        inp["det_boxes_gt"][:rows].copy_(b["det_boxes_gt"])
        inp["det_boxes_gt"][rows:, 0] = -1.0
torch.cuda.synchronize()


def serial(f):
    return lambda: procs[f].run(b["head"], b["protos"], b["det_boxes_gt"], b["masks_gt"], b["proj_weight"], float(b["proj_bias"]))


def piped(f):
    def go():
        p = pipes[f]
        p.fork()
        for _ in range(4 * 4):
            p.replay()
        p.join()
    return go


for rep in range(args.reps):
    for f in (False, True):
        print(json.dumps({"what": "serial step", "batch": B, "img": S, "with_surface_dist": f, "ms_per_step": timed(serial(f), N)}),
              flush=True)
    for f in (False, True):
        print(json.dumps({"what": "pipelined step (depth 4)", "batch": B, "img": S, "with_surface_dist": f,
                          "ms_per_step": timed(piped(f), 8) / 16}), flush=True)
