#!/usr/bin/env python
"""Cost of the binned PR / ROC curves of the projector probabilities (btpost_seg_curve, PostConfig.seg_curve) on the
synthetic workload.

    python scripts/seg_curve_timing.py [--reps 3]

1. Kernel time of btpost_seg_curve at 64 x 640^2 and 64 x 1024^2, T = 101 and 1024, on the projector logits and GT words
   the mask stage of the synthetic batch left in the workspace (they stay in the L2 between calls, as after a real mask
   stage): CUDA events around 50 back-to-back calls.
2. Step time at 64 x 640^2 with and without seg_curve=101, alternated: serial (PostProcessor.run back to back on one
   stream) and pipelined (Pipeline, 4 batches in flight, captured steps).
Prints the card's name and power limit first, then one JSON line per measurement."""
import argparse, ctypes as C, json, subprocess, sys
from pathlib import Path
ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "multitask-bonetumor-yolo_b200")]
import torch
from btpost import Pipeline, PostConfig, PostProcessor, _lib, segcurve, synth

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=3)
args = ap.parse_args()
dev = torch.device("cuda:0")
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip(), flush=True)
L = _lib.load()
B, N = 64, 50


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
    b = synth.make_batch_device(synth.SynthConfig(batch=B, img_size=S, seed=20262), dev)
    pp = PostProcessor(PostConfig(batch=B, img_size=S, gt_mode=1), dev)
    pp.run(b["head"], b["protos"], b["det_boxes_gt"], b["masks_gt"], b["proj_weight"], float(b["proj_bias"]))
    torch.cuda.synchronize()
    st = torch.cuda.current_stream().cuda_stream
    for T in (101, 1024):
        thr = segcurve.thresholds(T)
        arr = (C.c_float * T)(*thr.tolist())
        hist = torch.zeros(2, T + 1, dtype=torch.int64, device=dev)

        def call():
            _lib.check(L.btpost_seg_curve(C.byref(pp.params), C.c_void_p(pp._ws_ptr), C.c_size_t(pp._ws_bytes), arr, T,
                                          C.c_void_p(hist.data_ptr()), C.c_void_p(st)), "btpost_seg_curve")
        ms = [timed(call, N) for _ in range(args.reps)]
        hist.zero_()
        call()
        m = segcurve.curve_metrics(segcurve.confmat(hist), thr)
        print(json.dumps({"what": "btpost_seg_curve", "batch": B, "img": S, "T": T, "ms_per_call": ms,
                          "pixels_per_call": int(hist.sum()), "seg_ap": m["ap"], "seg_auroc": m["auroc"]}), flush=True)
    del pp, b
    torch.cuda.empty_cache()

S = 640
b = synth.make_batch_device(synth.SynthConfig(batch=B, img_size=S, seed=20262), dev)
curves = (None, 101)
procs = {c: PostProcessor(PostConfig(batch=B, img_size=S, gt_mode=1, seg_curve=c), dev) for c in curves}
pipes = {c: Pipeline(PostConfig(batch=B, img_size=S, gt_mode=1, seg_curve=c), dev, depth=4, proj_weight=b["proj_weight"],
                     proj_bias=float(b["proj_bias"])) for c in curves}
for p in pipes.values():
    for inp in p.inputs:
        for k in ("head", "protos", "masks_gt"):
            inp[k].copy_(b[k].reshape(inp[k].shape))
        rows = b["det_boxes_gt"].shape[0]
        inp["det_boxes_gt"][:rows].copy_(b["det_boxes_gt"])
        inp["det_boxes_gt"][rows:, 0] = -1.0
torch.cuda.synchronize()


def serial(c):
    return lambda: procs[c].run(b["head"], b["protos"], b["det_boxes_gt"], b["masks_gt"], b["proj_weight"], float(b["proj_bias"]))


def piped(c):
    def go():
        p = pipes[c]
        p.fork()
        for _ in range(4 * 4):
            p.replay()
        p.join()
    return go


for rep in range(args.reps):
    for c in curves:
        print(json.dumps({"what": "serial step", "batch": B, "img": S, "seg_curve": c, "ms_per_step": timed(serial(c), N)}),
              flush=True)
    for c in curves:
        print(json.dumps({"what": "pipelined step (depth 4)", "batch": B, "img": S, "seg_curve": c,
                          "ms_per_step": timed(piped(c), 8) / 16}), flush=True)
