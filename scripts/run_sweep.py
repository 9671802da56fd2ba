#!/usr/bin/env python
"""Sharded evaluation sweep (BASELINE config 5, scaled by --images): every rank post-processes its own batches
(synthetic head outputs generated on the device from the counter-based generator, so any sharding sees the same
images) with several batches in flight (btpost.Pipeline); the CUDA library appends the per-detection AP records and
all metric counters to a device-resident sweep state while it processes a batch (zero host work per batch), and the
only collectives are ONE all-reduce of the 4 KB sweep header and one all-gather of the records at the end, followed by
COCOeval.accumulate as CUDA kernels (btpost.DeviceSweep.finish).

    python scripts/run_sweep.py --images 16384                                  # 1 GPU
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 scripts/run_sweep.py --images 16384
Prints one JSON line with mAP / mAP50 / Dice / F1 and the device time of the sweep.  --seg-map adds the v3 segmentation
mAP (one record per image, appended by the mask stage to a second sweep state; seg_map / seg_map_50 in the line); the
default run leaves it out, so that its numbers stay comparable with earlier profiles.  --soft-dice adds v3's soft Dice
on the projector probabilities (seg_soft_dice in the line; one exp and one division per output pixel in the mask stage).
--micro adds the class-agnostic box mAP (torchmetrics average="micro": a third sweep state, one record per kept detection,
filled by a second matching pass of the COCO kernel; micro_map / micro_map_50 in the line).  --surface adds the projector
mask's Hausdorff distance, HD95 and ASSD against the GT mask (btpost_surface_distance after the mask stage of every batch;
the means seg_hd / seg_hd95 / seg_assd in the line).  --seg-curve T adds the binned PR / ROC state of the projector
probabilities at T thresholds (btpost_seg_curve after the mask stage of every batch; seg_ap / seg_auroc in the line)."""
import argparse, json, os, sys, time
from pathlib import Path
ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "multitask-bonetumor-yolo_b200")]
import numpy as np, torch, torch.distributed as dist
from btpost import DeviceSweep, Pipeline, PostConfig, synth
from btpost.api import map_iou_thresholds

ap = argparse.ArgumentParser()
ap.add_argument("--images", type=int, default=256)
ap.add_argument("--batch", type=int, default=64)
ap.add_argument("--img", type=int, default=640)
ap.add_argument("--max-det", dest="max_det", type=int, default=100)
ap.add_argument("--depth", type=int, default=4)
ap.add_argument("--seed", type=int, default=20265)
ap.add_argument("--seg-map", dest="seg_map", action="store_true", help="also the v3 segmentation mAP (seg_map, seg_map_50)")
ap.add_argument("--soft-dice", dest="soft_dice", action="store_true", help="also v3's soft Dice on the projector probabilities")
ap.add_argument("--micro", action="store_true", help="also the class-agnostic box mAP (micro_map, micro_map_50)")
ap.add_argument("--surface", action="store_true", help="also the projector mask's HD / HD95 / ASSD (seg_hd, seg_hd95, seg_assd)")
ap.add_argument("--seg-curve", dest="seg_curve", type=int, default=None,
                help="also pixel AP / AUROC of the projector probabilities at this many thresholds (seg_ap, seg_auroc)")
args = ap.parse_args()
rank, world, lrank = (int(os.environ.get(k, d)) for k, d in (("RANK", 0), ("WORLD_SIZE", 1), ("LOCAL_RANK", 0)))
torch.cuda.set_device(lrank)
dev = torch.device("cuda", lrank)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)
    dist.all_reduce(torch.zeros(1, device=dev))   # connect the peers now: communicator set-up is not part of the sweep
    dist.all_gather_into_tensor(torch.zeros(world, device=dev), torch.zeros(1, device=dev))
    _n = (args.images // args.batch // world + 1) * args.batch * args.max_det * 32   # a record all-gather of the real size
    dist.all_gather_into_tensor(torch.empty(world * _n, dtype=torch.uint8, device=dev), torch.empty(_n, dtype=torch.uint8, device=dev))
    dist.all_reduce(torch.zeros(512, dtype=torch.int64, device=dev))
B, K = args.batch, args.max_det
nbatches = args.images // B
mine = [i for i in range(nbatches) if i % world == rank]          # whole batches b = r (mod G)
cfg = PostConfig(batch=B, img_size=args.img, gt_mode=1, max_det=K, with_seg_map=args.seg_map, with_soft_dice=args.soft_dice,
                 with_surface_dist=args.surface, seg_curve=args.seg_curve)
sweep = DeviceSweep(cfg.nc, map_iou_thresholds(), (1, 10, 100), capacity=max(len(mine), 1) * B * K, max_det_per_image=K, device=dev,
                    seg_map_capacity=max(len(mine), 1) * B if args.seg_map else 0, soft_dice=args.soft_dice, micro=args.micro,
                    surface=args.surface, seg_curve=args.seg_curve)
probe = synth.make_batch_device(synth.SynthConfig(batch=B, img_size=args.img, seed=args.seed), dev)
pipe = Pipeline(cfg, dev, depth=args.depth, proj_weight=probe["proj_weight"], proj_bias=probe["proj_bias"], sweep=sweep)
del probe
sweep.reserve(nbatches * B * K, world)   # the end-of-sweep buffers come out of the allocator's cache
# host part of the generator for all of this rank's batches, done before the clock starts
preps = [synth.prepare_batch_device(synth.SynthConfig(batch=B, img_size=args.img, seed=args.seed, image_offset=i * B), dev) for i in mine]
torch.cuda.synchronize()
if world > 1:
    dist.barrier()              # the ranks start the sweep together: a rank that began early would wait in the collectives
    torch.cuda.synchronize()
ev0, ev1, ev2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
t_host = time.perf_counter()
ev0.record()
pipe.fork()
for n, (i, prep) in enumerate(zip(mine, preps)):
    slot = n % args.depth
    inp = pipe.inputs[slot]
    with torch.cuda.stream(pipe.streams[slot]):
        # this rank's images, generated on the device straight into the slot's input buffers (bit-identical to the numpy
        # generator: tests/test_gpu_synth.py); the generator kernel is inside the timed region, its host set-up is not
        synth.generate_into(prep, inp["head"], inp["protos"], inp["masks_gt"], stream=pipe.streams[slot])
        rows = prep["det_boxes_gt"].shape[0]
        inp["det_boxes_gt"][:rows].copy_(prep["det_boxes_gt"], non_blocking=True)
        inp["det_boxes_gt"][rows:, 0] = -1.0
    pipe.replay(slot, image_offset=i * B)
pipe.join()
ev1.record()
tim = {} if os.environ.get("SWEEP_TIMINGS") else None
res = sweep.finish(num_images_bound=nbatches * B, timings=tim)
ev2.record()
torch.cuda.synchronize()
tms = torch.tensor([ev0.elapsed_time(ev1), ev1.elapsed_time(ev2), ev0.elapsed_time(ev2)], dtype=torch.float64, device=dev)
if world > 1:
    dist.all_reduce(tms, op=dist.ReduceOp.MAX)   # device times are the maximum over the ranks
tms = tms.tolist()
if rank == 0:
    keys = ("n_images", "n_records", "map", "map_50", "map_75", "mar_100", "seg_f1", "seg_dice", "seg_iou", "uni_dice", "uni_iou")
    if args.seg_map:
        keys += ("seg_map", "seg_map_50")
    if args.soft_dice:
        keys += ("seg_soft_dice",)
    if args.micro:
        keys += ("micro_map", "micro_map_50")
    if args.surface:
        keys += ("seg_hd", "seg_hd95", "seg_assd", "n_surface_images")
    if args.seg_curve is not None:
        keys += ("seg_ap", "seg_auroc")
    line = {k: res[k] for k in keys}
    line.update(world=world, images=nbatches * B, batches_in_flight=args.depth, device_ms_batches_incl_generation=tms[0],
                device_ms_reduce_gather_accumulate=tms[1], device_ms_total=tms[2], host_s=time.perf_counter() - t_host)
    if tim is not None:
        line["finish_stage_ms_rank0"] = tim
    print(json.dumps(line))
if world > 1:
    dist.destroy_process_group()
