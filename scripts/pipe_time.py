"""Developer tool: pipelined step time (btpost.Pipeline, distinct inputs per slot, CUDA events) of the library
(BTPOST_LIB names another build), plus the first image's detection count and Dice as a sanity check.
usage: python scripts/pipe_time.py [depth] [steps] [label]"""
import os, sys
from pathlib import Path
ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "multitask-bonetumor-yolo_b200")]
import torch
from btpost import DeviceSweep, Pipeline, PostConfig, synth
from btpost.api import map_iou_thresholds

depth = int(sys.argv[1]) if len(sys.argv) > 1 else 5
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 300
label = sys.argv[3] if len(sys.argv) > 3 else ""
B, S = 64, 640
dev = torch.device("cuda:0")
torch.zeros(1, device=dev)
first = synth.make_batch_device(synth.SynthConfig(batch=B, img_size=S, seed=20262), dev)
cfg = PostConfig(batch=B, img_size=S, nms_threads=int(os.environ.get("NMS_NT", "0")))
sweep = DeviceSweep(cfg.nc, map_iou_thresholds(), (1, 10, 100), capacity=1 << 23, max_det_per_image=300, device=dev) if os.environ.get("SWEEP") else None
FILL = bool(os.environ.get("FILL"))
pipe = Pipeline(cfg, dev, depth=depth, proj_weight=first["proj_weight"], proj_bias=first["proj_bias"], sweep=sweep)
for i in range(depth):
    d = first if i == 0 else synth.make_batch_device(synth.SynthConfig(batch=B, img_size=S, seed=20262, image_offset=i * B), dev)
    pipe.load(i, d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"])
torch.cuda.synchronize()


def run(n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); pipe.fork()
    for j in range(n): pipe.replay(image_offset=j * B if FILL else None)
    pipe.join(); e1.record(); torch.cuda.synchronize()
    pipe.reset_metrics()
    return e0.elapsed_time(e1) / n * 1e3


run(4 * depth)
t20 = min(run(20) for _ in range(5))
tn = min(run(steps) for _ in range(3))
o = pipe.procs[0].out
opts = " ".join(f"{k}={v}" for k, v in sorted(os.environ.items()) if k in ("NMS_NT", "SWEEP", "FILL"))
print(f"{label:24s} depth {depth}: {tn:7.2f} us/step over {steps} steps, {t20:7.2f} over 20 | dets {o['det_count'][:3].tolist()} "
      f"dice {o['seg_dice'][0].item():.6f} uni {o['uni_dice'][0].item():.6f} | {opts}", flush=True)
