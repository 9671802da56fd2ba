#!/usr/bin/env python
"""bench.py -- images/sec of the post-processing + evaluation hot path (BASELINE.json metric).

A "step" is one pass of the whole hot path (decode+filter -> NMS+COCO matching+sweep records -> mask assembly +
Dice/IoU counters) over one batch of synthetic head outputs.  At N GPUs every rank owns its own batch of `--batch`
images per step (images are independent units: weak scaling, no data-path collective); the only NCCL traffic is one
all-reduce of the 4 KB sweep header (the metric counters) at the end of the timed region.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --workload c2                                  # BASELINE config 2: decode+NMS+mask assembly, masks out
    python bench.py --impl reference ...                           # the reference's ops on the host cores (torch port)
    python bench.py ... --dump-outputs DIR                         # also write the last timed step's outputs as DIR/*.npy

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the definition of every key.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
for _p in (ROOT, ROOT / "multitask-bonetumor-yolo_b200"):
    if str(_p) not in sys.path:
        sys.path.insert(0, str(_p))

import numpy as np  # noqa: E402

METRIC = "images/sec post-proc+eval"
UNIT = "images/s"
SEED = 20262
KERNELS = ["gt_pack_kernel", "decode_filter_l2_kernel", "nms_kernel", "plan_kernel", "coeff_gather_kernel", "match_kernel",
           "contract_kernel", "cells_kernel", "finalize_kernel"]
DUMP_BYTES = 64 * 10**6    # --dump-outputs: all files of one dump together


def dump_outputs(out, path, budget=DUMP_BYTES):
    """Writes one step's outputs (`out`: name -> tensor) as <path>/<name>.npy, so that two builds can be compared output
    for output.  Integer and float64 outputs are stored as float64, the others as float32: every value is kept exactly.
    When the whole set would exceed `budget` bytes, each output larger than a common element count is cut to that many
    of its flattened elements at most: distinct flat indices drawn from a generator seeded with SEED and the output's name,
    in ascending order, so that the same arguments select the same elements.  Returns the names of the cut outputs."""
    import zlib

    import torch
    path = Path(path)
    path.mkdir(parents=True, exist_ok=True)
    wide = {k: t.dtype == torch.float64 or (not t.is_floating_point() and t.element_size() >= 4) for k, t in out.items()}
    sizes = {k: t.numel() for k, t in out.items()}

    def nbytes(cap):                                    # 256 bytes per file for the .npy header
        return sum((8 if wide[k] else 4) * min(n, cap) + 256 for k, n in sizes.items())

    lo, hi = 0, max(sizes.values(), default=0)          # the largest common cap that fits the budget
    while lo < hi:
        mid = (lo + hi + 1) // 2
        lo, hi = (mid, hi) if nbytes(mid) <= budget else (lo, mid - 1)
    cut = []
    for k in sorted(out):
        t = out[k]
        if sizes[k] > lo:
            rng = np.random.default_rng([SEED, zlib.crc32(k.encode())])
            t = t.reshape(-1)[torch.from_numpy(np.unique(rng.integers(0, sizes[k], lo))).to(t.device)]
            cut.append(k)
        np.save(path / f"{k}.npy", t.to(torch.float64 if wide[k] else torch.float32).cpu().numpy())
    return cut


def algorithmic_bytes_per_image(S, nc=3, nm=32):
    """SURVEY.md §8(d): head + protos + u8 GT mask (full eval, masks fused away)."""
    N = sum((S // s) ** 2 for s in (8, 16, 32))
    head = 4 * (4 + nc + nm) * N
    protos = 4 * nm * (S // 4) ** 2
    gt_mask = S * S
    return dict(head=head, protos=protos, gt_mask=gt_mask, total=head + protos + gt_mask)


def workload_name(args):
    if args.workload == "c2":
        return (f"batch {args.batch} x {args.img}^2 synthetic head outputs (L2 [B,39,N] + 32ch protos), decode+NMS+mask assembly "
                f"with every instance mask written out ({args.masks_out}), conf {args.conf}, iou {args.iou}, max_det {args.max_det}")
    return (f"batch {args.batch} x {args.img}^2 synthetic head outputs (L2 [B,39,N] + 32ch protos), "
            f"decode+NMS+mask assembly+Dice/IoU+COCO matching, conf {args.conf}, iou {args.iou}, max_det {args.max_det}")


# --------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons DURING the timed region.  NVML is read in-process from the launching thread, but only
    after every step of the region has been enqueued and until the closing event completes: the GPU is still working
    through the region while the host has nothing left to launch (NVML calls made from a second thread serialise against
    CUDA launches and were measured to double the step time; a `nvidia-smi -lms` child process started next to the region
    spends the region's 2 ms loading NVML and competes for the driver with the launches).  Falls back to the recipe's
    `nvidia-smi --query-gpu=... -lms` line, started before the warm-up, when pynvml is missing."""

    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index, period_ms=100):
        self.nv = self.handle = self.proc = self.path = None
        self.mhz, self.max_mhz, self.reasons, self.t0 = [], None, set(), None
        if period_ms <= 0:
            return
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            pr = torch.cuda.get_device_properties(index)
            try:
                bus = f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
                self.handle = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
            return
        except Exception:
            self.nv = self.handle = None
        import shutil
        import subprocess
        import tempfile
        exe = shutil.which("nvidia-smi")
        if exe is None:
            return
        f = tempfile.NamedTemporaryFile(prefix="btpost_clocks_", suffix=".csv", delete=False)
        self.path = f.name
        self.proc = subprocess.Popen([exe, "-i", str(index), f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                      "-lms", str(period_ms)], stdout=f, stderr=subprocess.DEVNULL)

    def mark_start(self):
        """The timed region starts now (the nvidia-smi fallback keeps only the lines written from here on)."""
        if self.path is not None:
            self.t0 = os.path.getsize(self.path)

    def poll_until(self, event):
        """Called once the whole region is enqueued: sample until `event` (recorded at its end) has completed."""
        if self.nv is None:
            return
        while True:
            try:
                self.mhz.append(int(self.nv.nvmlDeviceGetClockInfo(self.handle, self.nv.NVML_CLOCK_SM)))
                mask = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                self.reasons.update(n for n, bit in self.REASONS.items() if mask & bit)
            except Exception:
                break
            if event.query():
                break

    def stop(self):
        if self.nv is not None:
            mhz = sorted(self.mhz)
            return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                    "samples": len(mhz), "source": "nvml, polled by the launching thread between the last launch and the end of the region"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "note": "neither pynvml nor nvidia-smi found"}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        mhz, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        text = open(self.path).read()
        for ln in text[self.t0 or 0:].splitlines() or text.splitlines()[-1:]:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 6 or not parts[0].isdigit():
                continue
            mhz.append(int(parts[0]))
            mx = int(parts[1]) if parts[1].isdigit() else mx
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        try:
            os.unlink(self.path)
        except OSError:
            pass
        mhz.sort()
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(mhz), "source": "nvidia-smi -lms child process"}


# --------------------------------------------------------------------------------------------
def reference_rate(args, n_images, steps, warmup):
    """The reference's ops (oracle/ref_torch.py: torch + torchvision + the C COCO matcher) on `n_images` images of the
    workload per step, all host threads.  Returns (images/s, seconds per step, threads)."""
    import torch

    from btpost import synth
    from oracle import ref_torch
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    batch = synth.make_batch(synth.SynthConfig(batch=n_images, img_size=args.img, seed=SEED))
    kw = dict(conf_thres=args.conf, iou_thres=args.iou, max_det=args.max_det, img_size=args.img, with_coco=args.workload != "c2")
    for _ in range(warmup):
        ref_torch.run_batch(batch, **kw)
    t0 = time.perf_counter()
    for _ in range(steps):
        ref_torch.run_batch(batch, **kw)
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return n_images / dt, dt, threads


def run_reference(args):
    """Reference arm.  The reference is pure Python/PyTorch and /root/reference is not on the GPU box, so this runs the
    torch port of its ops on all host threads.  Each step is a bounded sample of the B-image batch: the per-image cost is
    probed first (one image) and the sample is sized so that warm-up + steps stay within ~3 minutes."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    rate1, dt1, threads = reference_rate(args, 1, 1, 1)
    budget = 170.0 / max(args.steps + args.warmup, 1)          # seconds per step
    sample = int(max(1, min(args.batch, budget / dt1 * 1.5)))  # batching amortises the per-call overheads a little
    v, dt, threads = reference_rate(args, sample, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args), "sample_images_per_step": sample, "global_batch": args.batch},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{sample} of the {args.batch} images of a step, {args.steps} steps: torch port of the reference's ops "
                                   f"(torchvision nms, conv2d, interpolate, einsum; C COCO matcher), torch.set_num_threads({threads})"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="full", choices=["full", "c2"],
                    help="full = BASELINE headline (decode+NMS+masks+Dice/IoU+COCO); c2 = decode+NMS+mask assembly, masks written out")
    ap.add_argument("--masks-out", dest="masks_out", default="dense", choices=["dense", "bits"], help="c2: [B,K,S,S] bytes or bit-packed")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--img", type=int, default=640)
    ap.add_argument("--conf", type=float, default=0.05)
    ap.add_argument("--iou", type=float, default=0.6)
    ap.add_argument("--max-det", dest="max_det", type=int, default=300)
    ap.add_argument("--cpu-sample", type=int, default=64,
                    help="images the cpu_baseline leg times (0 = skip); default: one full batch, ~10-25 s of CPU work with warm-up")
    ap.add_argument("--pipeline", type=int, default=0,
                    help="batches in flight = slots with their own input set (0 = auto: 6, 5 or 4, whichever divides --steps; 2 for c2; 1 = strictly serial steps)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--clock-period-ms", type=int, default=100, help="nvidia-smi sampling period during the timed region (0 = off)")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="after the timed steps, write the outputs the last of them returned (rank 0's) as DIR/<name>.npy, "
                         f"float32 / float64, at most {DUMP_BYTES // 10**6} MB in all (larger outputs: a fixed, seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.pipeline <= 0:
        # a slot runs its steps one after the other, so a ragged last round (steps not a multiple of the depth) leaves
        # most slots idle at the end: take the deepest of 6, 5, 4 that divides the number of steps
        args.pipeline = 2 if args.workload == "c2" else next((d for d in (6, 5, 4) if args.steps % d == 0), 6)

    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist

    from btpost import DeviceSweep, Pipeline, PostConfig, PostProcessor, _lib, synth
    from btpost.api import map_iou_thresholds

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product path has no CPU fallback")
    _lib.load()  # fail loudly if libbtpost.so is missing
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B, S, depth = args.batch, args.img, args.pipeline
    c2 = args.workload == "c2"
    cfg = PostConfig(batch=B, img_size=S, conf_thres=args.conf, iou_thres=args.iou, max_det=args.max_det, with_coco=not c2,
                     with_inst_masks=args.masks_out if c2 else None)
    # ---------------- sweep state (metric counters + AP records live on the device) and the slots
    sweep = None
    if not c2:
        cap = min((args.steps + args.warmup + 8) * B * args.max_det, 1 << 23)
        sweep = DeviceSweep(cfg.nc, map_iou_thresholds(), (1, 10, 100), capacity=cap, max_det_per_image=args.max_det, device=dev)
    first = synth.make_batch_device(synth.SynthConfig(batch=B, img_size=S, seed=SEED, image_offset=(rank * depth) * B), dev)
    bias = float(first["proj_bias"])
    pipe = Pipeline(cfg, dev, depth=depth, proj_weight=first["proj_weight"], proj_bias=bias, sweep=sweep, auto_image_offset=True)
    # every slot gets its OWN, different batch (generated on the device, bit-identical to the numpy generator): a buffer
    # is read again only after the other depth-1 input sets (depth x 320 MB at 640^2) have streamed through
    gt_rows = []
    for i in range(depth):
        d = first if i == 0 else synth.make_batch_device(synth.SynthConfig(batch=B, img_size=S, seed=SEED, image_offset=(rank * depth + i) * B), dev)
        pipe.load(i, d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"])
        gt_rows.append(int(d["det_boxes_gt"].shape[0]))
        torch.cuda.synchronize()
    del d, first
    torch.cuda.empty_cache()
    # one batch in flight: strictly serial steps, per-stage timings (own workspace / outputs; reads slot 0's inputs)
    pp = PostProcessor(cfg, dev, sweep=None)
    i0 = pipe.inputs[0]

    def step(stage="run"):
        return pp.run(i0["head"], i0["protos"], i0["det_boxes_gt"], i0["masks_gt"], pipe.proj_weight, bias, stage=stage)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    graph = pp.capture(i0["head"], i0["protos"], i0["det_boxes_gt"], i0["masks_gt"], pipe.proj_weight, bias)
    sampler = ClockSampler(local_rank, args.clock_period_ms)   # NVML is initialised here, outside the timed region
    # the images are numbered on the device (every captured step bumps its slot's counter): no host work per step
    pipe.set_image_base(rank * (args.steps + args.warmup) * B)
    pipe.fork()
    for _ in range(args.warmup):
        pipe.replay()
    pipe.join()
    hdr = sweep.hdr if sweep is not None else torch.zeros(8, dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(hdr.clone())    # connects the NCCL peers: communicator set-up is not part of the timed region
    barrier()

    # ---------------- timed region: K steps over rotating input sets, inputs resident in HBM
    pipe.reset_metrics()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.mark_start()
    ev0.record()
    pipe.fork()
    for _ in range(args.steps):
        last = pipe.replay()      # step i on slot i % depth: consecutive batches overlap, every step does all of its work
    pipe.join()
    if world > 1:
        dist.all_reduce(hdr)  # the only collective: the sweep header = all metric counters (NCCL over NVLink)
    ev1.record()
    sampler.poll_until(ev1)   # everything is enqueued: read the clocks while the GPU works through the region
    barrier()
    ms = ev0.elapsed_time(ev1)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = B * world * args.steps / (ms / 1e3)
    det_mean = float(sum(p.out["det_count"].sum() for p in pipe.procs)) / (depth * B)
    if args.dump_outputs and rank == 0:
        # the slot's outputs as a caller of the last step receives them; cm / seg_cnt4 / uni_cnt4 are the counters all
        # slots share, summed over the timed steps
        cut = dump_outputs(last.out, args.dump_outputs)
        print(f"bench: wrote {len(last.out)} outputs of the last timed step to {args.dump_outputs}"
              + (f" (sampled: {', '.join(cut)})" if cut else ""), file=sys.stderr, flush=True)

    # ---------------- strictly serial steps (one stream, one batch in flight): the latency of a step
    torch.cuda.synchronize()
    es0, es1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    es0.record()
    for _ in range(args.steps):
        graph.replay()
    es1.record()
    torch.cuda.synchronize()
    serial_ms = es0.elapsed_time(es1) / args.steps

    # ---------------- per-stage device times (CUDA events on the launching stream)
    stage_ms = {}
    ORDER = ("decode_filter", "nms_match", "masks_pack", "masks_contract", "masks_cells")
    nrep = min(args.steps, 50)
    for stage in ORDER:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tot = 0.0
        for _ in range(nrep):
            for s2 in ORDER:   # keep the real order so caches look like a step
                if s2 == stage:
                    e0.record()
                step(stage=s2)
                if s2 == stage:
                    e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        stage_ms[stage] = tot / nrep

    # ---------------- end to end through the public API with HOST buffers (pinned), copies inside the timed region
    def e2e_run(bf16):
        """Pipeline.submit() from pinned host tensors (H2D of head + protos + GT masks + GT rows on the slot's stream),
        the captured step, D2H of the step's results; `edepth` batches in flight so that batch i+1's copies run under
        batch i's kernels.  Every step reads a different host batch."""
        edepth = 3
        ecfg = PostConfig(batch=B, img_size=S, conf_thres=args.conf, iou_thres=args.iou, max_det=args.max_det, with_coco=not c2,
                          head_bf16=bf16, proto_bf16=bf16)
        epipe = Pipeline(ecfg, dev, depth=edepth, proj_weight=pipe.proj_weight, proj_bias=bias)
        hosts = []
        for i in range(edepth):
            inp = pipe.inputs[i % depth]
            h = {k: inp[k] for k in ("head", "protos", "masks_gt")}
            if bf16:
                h["head"], h["protos"] = h["head"].bfloat16(), h["protos"].bfloat16()
            h = {k: v.cpu().pin_memory() for k, v in h.items()}
            h["det_boxes_gt"] = inp["det_boxes_gt"][:gt_rows[i % depth]].cpu().pin_memory()
            hosts.append(h)
        keys = ("det_count", "dets", "seg_dice", "seg_iou", "uni_dice", "uni_iou")
        res_host = [{k: torch.empty_like(epipe.procs[i].out[k], device="cpu").pin_memory() for k in keys} for i in range(edepth)]
        done = [torch.cuda.Event() for _ in range(edepth)]

        def run(n):
            for j in range(n):
                i = j % edepth
                if j >= edepth:
                    done[i].synchronize()               # the caller has read slot i's previous results
                h = hosts[i]
                epipe.submit(h["head"], h["protos"], h["det_boxes_gt"], h["masks_gt"])
                with torch.cuda.stream(epipe.streams[i]):
                    for k in keys:
                        res_host[i][k].copy_(epipe.procs[i].out[k], non_blocking=True)
                    done[i].record()
            for e in done:
                e.synchronize()

        run(edepth + 1)
        barrier()
        t0 = time.perf_counter()
        run(args.steps)
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        h2d = int(sum(v.numel() * v.element_size() for v in hosts[0].values()))
        d2h = int(sum(v.numel() * v.element_size() for v in res_host[0].values()))
        sec = float(dt.item())

        # the host-side ceiling: the same pinned buffers copied to the same device buffers with NO kernels in between, all
        # ranks at once (what PCIe / the host memory system give this rank while its neighbours copy too)
        def copy_only(n):
            for j in range(n):
                h = hosts[j % edepth]
                epipe.load(j % edepth, h["head"], h["protos"], h["det_boxes_gt"], h["masks_gt"])
            torch.cuda.synchronize()

        ncopy = max(3, min(args.steps, 20))
        copy_only(edepth)
        barrier()
        t0 = time.perf_counter()
        copy_only(ncopy)
        barrier()
        dc = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dc, op=dist.ReduceOp.MAX)
        out = {"value": B * world * args.steps / sec, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "h2d_gbs_per_rank": h2d * args.steps / sec / 1e9, "h2d_copy_only_gbs_per_rank": h2d * ncopy / float(dc.item()) / 1e9,
               "batches_in_flight": edepth, "inputs": "bf16 head + protos" if bf16 else "fp32"}
        del epipe, hosts, res_host
        torch.cuda.empty_cache()
        return out

    e2e = e2e_bf16 = None
    if not args.no_e2e and not c2:
        e2e = e2e_run(False)
        e2e_bf16 = e2e_run(True)
    clocks = sampler.stop()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    pk = ROOT / "MEASURED_PEAKS.json"
    if pk.exists():
        peaks = json.loads(pk.read_text())
    peak_gbs, peak_src = (peaks["hbm_gbs"], "measured") if "hbm_gbs" in peaks else (6650.0, "fallback")
    ab = algorithmic_bytes_per_image(S)
    step_bytes = ab["total"] * B
    if c2:
        mask_px = S * S if args.masks_out == "dense" else S * S // 8
        step_bytes = (ab["head"] + ab["protos"]) * B + int(det_mean * B) * mask_px + 24 * int(det_mean * B)
    mask_bytes = ab["protos"] * B       # algorithmic bytes of one contract_kernel launch: the prototypes, once
    achieved = mask_bytes / (stage_ms["masks_contract"] / 1e3) / 1e9
    traffic = None
    tf = ROOT / "profiles" / "roofline_traffic.json"
    if tf.exists():
        try:
            traffic = json.loads(tf.read_text()).get(f"contract_kernel_B{B}_S{S}")
        except Exception:
            traffic = None
    kernels = [k for k in KERNELS if not (c2 and k == "match_kernel")] + (["inst_dense_kernel"] if c2 and args.masks_out == "dense" else [])
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args), "global_batch": B * world, "sharding": f"images sharded, {B}/GPU",
                   "batches_in_flight": depth, "input_sets": depth,
                   "l2": "every slot owns a different input set (%.0f MB each): a buffer is re-read after %.2f GB of other inputs, "
                         "far beyond the 126 MB L2" % (ab["total"] * B / 1e6, ab["total"] * B * (depth - 1) / 1e9),
                   "detections_per_image": det_mean},
        "roofline": {"bound": "hbm", "kernel": "contract_kernel", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                     "frac": achieved / peak_gbs, "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": mask_bytes},
        "pipeline": {"algorithmic_bytes_per_step": step_bytes, "algorithmic_bytes_per_image": step_bytes / B,
                     "achieved_gbs": step_bytes / (ms / args.steps / 1e3) / 1e9,
                     "frac_of_peak": step_bytes / (ms / args.steps / 1e3) / 1e9 / peak_gbs,
                     "stage_ms": stage_ms, "ms_per_step_one_batch_in_flight": serial_ms},
        "clocks": clocks, "gpu_launches": len(kernels) * args.steps, "kernels_per_step": kernels,
    }
    if e2e:
        line["e2e"] = e2e
        line["e2e_bf16"] = e2e_bf16
    elif c2:
        line["e2e"] = None
    if world == 1 and args.cpu_sample > 0:
        v, dt, threads = reference_rate(args, args.cpu_sample, 1, 1)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": f"{args.cpu_sample} images of the same workload, torch port of the reference's ops "
                                          f"(oracle/ref_torch.py), {threads} threads, {dt:.1f} s"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
