"""Sweep-level metric state: what `on_validation_epoch_end` / `evaluate()` compute from the per-batch
outputs (`/root/reference/src/running_main_v2.py:959-1177`, `evaluate_model.py:240-355`).

Per batch the CUDA library leaves integer counters and per-detection COCO match bits on the device.
`SweepState.add` appends them to device-resident buffers (no host sync).  At the end of the sweep:

  * `all_reduce(group)` -- ONE `all_reduce(SUM)` of a packed int64 counter vector (confusion matrix,
    pixel tp/fp/fn/tn, GT counts, image count) and one of an fp64 vector (sums of per-image Dice/IoU):
    the only collective on the path (NCCL over NVLink on the GPU box, gloo in the CPU tests);
  * `gather(group)` -- COCO AP is not a sum of counters (it needs the globally score-sorted record
    list), so the compact per-detection records are all-gathered (padded to the largest shard);
  * `compute()` -- COCOeval.accumulate + summarize (SURVEY.md A.3) on the gathered records.  The stable
    global order pycocotools gets from concatenating images in order and a mergesort on -score is
    reproduced with the sort key (score desc, global image index, rank in image), so the result does
    not depend on how images were sharded.

`SweepState` runs as tensor ops on whatever device the state lives on; it is the host-logic restatement used by
the gloo tests on CPU and by the host path of the v3 segmentation mAP (one record per image, `btpost.segmap`).

`DeviceSweep` is the production path for the detection sweep (BASELINE config 5): the CUDA library itself appends the
per-detection records, GT counts, image count and Dice / IoU sums to a caller-owned device buffer while it processes a
batch (`BtIO.sweep`, zero host work per batch), shards are merged by ONE all-reduce of the 4 KB header and one
`all_gather_into_tensor` of the records, and COCOeval.accumulate runs as CUDA kernels (`btpost_sweep_accumulate`:
radix sort + scans + 101-point lookup).  With `seg_map_capacity` it also owns the v3 segmentation-mAP state, to which the
mask stage appends one record per image (`BtIO.seg_sweep`); with `micro=True` it owns the class-agnostic state
(`BtIOMicro.micro_sweep`, torchmetrics `average="micro"`), to which the COCO matching appends one record per kept
detection.  Every state rides in the same collectives (`merge_sweeps`).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from . import _lib, segcurve

AREA_NAMES = ("all", "small", "medium", "large")


class SweepState:
    def __init__(self, nc: int, num_thrs: int, iou_thrs, max_dets=(1, 10, 100), device="cpu"):
        self.nc, self.T, self.A = nc, num_thrs, 4
        self.iou_thrs = [float(t) for t in iou_thrs]
        self.max_dets = tuple(max_dets)
        self.device = torch.device(device)
        self.reset()

    def reset(self):
        d = self.device
        self.cm = torch.zeros(self.nc, self.nc, dtype=torch.int64, device=d)
        self.seg_cnt4 = torch.zeros(4, dtype=torch.int64, device=d)
        self.uni_cnt4 = torch.zeros(4, dtype=torch.int64, device=d)
        self.n_images = torch.zeros(1, dtype=torch.int64, device=d)
        self.npig = torch.zeros(self.A, self.nc, dtype=torch.int64, device=d)      # non-ignored GT per (area, class)
        self.fsum = torch.zeros(4, dtype=torch.float64, device=d)                   # sum seg dice, seg iou, uni dice, uni iou
        self._rec = []                                                              # per-batch record tensors

    # ------------------------------------------------------------------ per batch
    @torch.no_grad()
    def add(self, out: dict, image_offset: int, accumulate_counters: bool = False):
        """Append one batch.  `out` = PostProcessor.run(...) outputs (device tensors, padded).  The
        library accumulates cm / seg_cnt4 / uni_cnt4 itself across calls, so by default they are
        taken once at the end through `take_counters`; pass accumulate_counters=True when `out`
        holds per-batch values (the oracle's layout)."""
        dets, cnt = out["dets"], out["det_count"].long()
        B, K, _ = dets.shape
        valid = torch.arange(K, device=dets.device)[None, :] < cnt[:, None]                        # [B,K]
        labels = dets[..., 5].long()
        onehot = torch.nn.functional.one_hot(labels.clamp(0, self.nc - 1), self.nc) * valid[..., None]
        class_rank = (onehot.cumsum(1) - onehot).gather(2, labels.clamp(0, self.nc - 1)[..., None])[..., 0]   # earlier same-class dets
        img = (torch.arange(B, device=dets.device) + image_offset)[:, None].expand(B, K)
        rank = torch.arange(K, device=dets.device)[None, :].expand(B, K)
        matched = (out["dt_match"] > 0).permute(0, 3, 1, 2)                                         # [B,K,A,T]
        ignored = (out["dt_ignore"] > 0).permute(0, 3, 1, 2)
        # padded per-batch records + their validity mask: the ragged compaction (a host sync per batch) happens once,
        # in _records(); the library reuses its output buffers, so everything kept here is a copy
        self._rec.append({
            "score": dets[..., 4].reshape(-1).clone(), "label": labels.reshape(-1), "img": img.reshape(-1),
            "rank": rank.reshape(-1), "class_rank": class_rank.reshape(-1),
            "matched": matched.reshape(B * K, self.A, self.T), "ignored": ignored.reshape(B * K, self.A, self.T),
            "_valid": valid.reshape(-1),
        })
        if len(self._rec) >= 64:   # bound the padded backlog: one compaction (and host sync) per 64 batches
            self._rec = [self._records()]
        G = out["gt_labels"].shape[1]
        gvalid = torch.arange(G, device=dets.device)[None, :] < out["gt_count"].long()[:, None]     # [B,G]
        gl = out["gt_labels"].long()
        inrange = gvalid & (gl >= 0) & (gl < self.nc)
        keep = inrange[:, None, :] & ~(out["gt_ignore"] > 0)                                         # [B,A,G]
        goh = torch.nn.functional.one_hot(gl.clamp(0, self.nc - 1), self.nc)                        # [B,G,nc]
        # integer contraction written as a masked sum (CUDA has no int64 matmul)
        self.npig += (keep[:, :, :, None] & (goh[:, None, :, :] > 0)).sum(dim=(0, 2))
        self.n_images += B
        self.fsum += torch.stack([out["seg_dice"].double().sum(), out["seg_iou"].double().sum(),
                                  out["uni_dice"].double().sum(), out["uni_iou"].double().sum()])
        if accumulate_counters:
            self.cm += out["cm"].long(); self.seg_cnt4 += out["seg_cnt4"].long(); self.uni_cnt4 += out["uni_cnt4"].long()

    @torch.no_grad()
    def take_counters(self, out: dict):
        """Copy the counters the library accumulated over the whole sweep (cm, seg_cnt4, uni_cnt4)."""
        self.cm.copy_(out["cm"]); self.seg_cnt4.copy_(out["seg_cnt4"]); self.uni_cnt4.copy_(out["uni_cnt4"])

    # ------------------------------------------------------------------ collectives
    def _pack_i64(self):
        return torch.cat([self.cm.flatten(), self.seg_cnt4, self.uni_cnt4, self.n_images, self.npig.flatten()])

    def _unpack_i64(self, v):
        n = self.nc * self.nc
        self.cm = v[:n].view(self.nc, self.nc).clone(); self.seg_cnt4 = v[n:n + 4].clone()
        self.uni_cnt4 = v[n + 4:n + 8].clone(); self.n_images = v[n + 8:n + 9].clone()
        self.npig = v[n + 9:].view(self.A, self.nc).clone()

    @torch.no_grad()
    def all_reduce(self, group=None):
        """The metric-counter all-reduce (north star: the only NCCL traffic on the path)."""
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return
        v = self._pack_i64()
        dist.all_reduce(v, group=group)
        self._unpack_i64(v)
        dist.all_reduce(self.fsum, group=group)

    def _records(self):
        if not self._rec:
            z = lambda *s, dt: torch.zeros(*s, dtype=dt, device=self.device)
            return {"score": z(0, dt=torch.float32), "label": z(0, dt=torch.int64), "img": z(0, dt=torch.int64),
                    "rank": z(0, dt=torch.int64), "class_rank": z(0, dt=torch.int64),
                    "matched": z(0, self.A, self.T, dt=torch.bool), "ignored": z(0, self.A, self.T, dt=torch.bool)}
        parts = []
        for r in self._rec:
            if "_valid" in r:   # a padded batch as `add` left it
                v = r["_valid"]
                r = {k: t[v] for k, t in r.items() if k != "_valid"}
            parts.append(r)
        return {k: torch.cat([r[k] for r in parts]) for k in parts[0]}

    @torch.no_grad()
    def gather(self, group=None):
        """All-gather of the ragged record lists (padded to the largest shard, then trimmed)."""
        rec = self._records()
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            self._rec = [rec]
            return
        W = dist.get_world_size(group)
        n = torch.tensor([rec["score"].shape[0]], dtype=torch.int64, device=self.device)
        ns = [torch.zeros_like(n) for _ in range(W)]
        dist.all_gather(ns, n, group=group)
        ns = [int(x.item()) for x in ns]
        cap = max(max(ns), 1)
        out = {}
        for k, t in rec.items():
            pad = torch.zeros((cap,) + tuple(t.shape[1:]), dtype=torch.uint8 if t.dtype == torch.bool else t.dtype, device=self.device)
            pad[: t.shape[0]] = t.to(pad.dtype)
            parts = [torch.zeros_like(pad) for _ in range(W)]
            dist.all_gather(parts, pad, group=group)
            cat = torch.cat([p[:m] for p, m in zip(parts, ns)])
            out[k] = cat.bool() if t.dtype == torch.bool else cat
        self._rec = [out]

    # ------------------------------------------------------------------ epoch end
    @torch.no_grad()
    def compute(self) -> dict:
        rec = self._records()
        T, A, nc, M = self.T, self.A, self.nc, len(self.max_dets)
        dev = self.device
        # global stable order: score desc, then image index, then rank inside the image
        key2 = rec["img"] * 65536 + rec["rank"]
        order = torch.argsort(key2, stable=True)
        order = order[torch.argsort(-rec["score"][order].double(), stable=True)]
        rec = {k: v[order] for k, v in rec.items()}
        rec_thrs = torch.linspace(0.0, 1.0, 101, dtype=torch.float64, device=dev)
        precision = -torch.ones(T, 101, nc, A, M, dtype=torch.float64, device=dev)
        recall = -torch.ones(T, nc, A, M, dtype=torch.float64, device=dev)
        eps = torch.finfo(torch.float64).eps
        for c in range(nc):
            in_c = rec["label"] == c
            for mi, md in enumerate(self.max_dets):
                sel = in_c & (rec["class_rank"] < md)
                mt, ig = rec["matched"][sel], rec["ignored"][sel]                 # [R,A,T]
                tps = (mt & ~ig).permute(1, 2, 0).double().cumsum(-1)             # [A,T,R]
                fps = (~mt & ~ig).permute(1, 2, 0).double().cumsum(-1)
                R = tps.shape[-1]
                for a in range(A):
                    npig = int(self.npig[a, c].item())
                    if npig == 0:
                        continue
                    if R == 0:
                        recall[:, c, a, mi] = 0.0
                        precision[:, :, c, a, mi] = 0.0
                        continue
                    rc = tps[a] / npig                                            # [T,R]
                    pr = tps[a] / (fps[a] + tps[a] + eps)
                    pr = torch.flip(torch.cummax(torch.flip(pr, [-1]), -1).values, [-1])   # right-to-left running max
                    recall[:, c, a, mi] = rc[:, -1]
                    idx = torch.searchsorted(rc.contiguous(), rec_thrs[None, :].expand(T, 101).contiguous(), right=False)
                    q = torch.where(idx < R, pr.gather(1, idx.clamp(max=R - 1)), torch.zeros((), dtype=torch.float64, device=dev))
                    precision[:, :, c, a, mi] = q

        def mean(x):
            x = x[x > -1]
            return float(x.mean().item()) if x.numel() else -1.0

        def thr_idx(v):
            for i, t in enumerate(self.iou_thrs):
                if abs(t - v) < 1e-6:
                    return i
            return None
        res = {"map": mean(precision[:, :, :, 0, -1])}
        for name, v in (("map_50", 0.5), ("map_75", 0.75)):
            ti = thr_idx(v)
            res[name] = mean(precision[ti, :, :, 0, -1]) if ti is not None else -1.0
        for ai in (1, 2, 3):
            res[f"map_{AREA_NAMES[ai]}"] = mean(precision[:, :, :, ai, -1])
            res[f"mar_{AREA_NAMES[ai]}"] = mean(recall[:, :, ai, -1])
        for mi, md in enumerate(self.max_dets):
            res[f"mar_{md}"] = mean(recall[:, :, 0, mi])
        res["map_per_class"] = [mean(precision[:, :, c, 0, -1]) for c in range(nc)]
        res[f"mar_{self.max_dets[-1]}_per_class"] = [mean(recall[:, c, 0, -1]) for c in range(nc)]
        n = max(int(self.n_images.item()), 1)
        tp, fp, fn, tn = [int(v) for v in self.seg_cnt4.tolist()]
        res.update({
            "n_images": int(self.n_images.item()), "cm": self.cm.clone(),
            "seg_f1": 2 * tp / (2 * tp + fp + fn) if (2 * tp + fp + fn) else 0.0,
            "seg_precision": tp / (tp + fp) if (tp + fp) else 0.0, "seg_recall": tp / (tp + fn) if (tp + fn) else 0.0,
            "seg_accuracy": (tp + tn) / max(tp + tn + fp + fn, 1),
            "seg_dice": float(self.fsum[0].item()) / n, "seg_iou": float(self.fsum[1].item()) / n,
            "uni_dice": float(self.fsum[2].item()) / n, "uni_iou": float(self.fsum[3].item()) / n,
            "precision": precision, "recall": recall,
        })
        return res


# ======================================================================================================================
# device-resident sweep (include/btpost.h "Sweep state")
# ======================================================================================================================
HDR = _lib.SWEEP_HEADER_I64
REC_BYTES = 32
REC_DTYPE = np.dtype([("matched", "<u8"), ("ignored", "<u8"), ("score_key", "<u4"), ("image", "<u4"), ("rank", "<u2"),
                      ("class_rank", "<u2"), ("label", "u1"), ("pad", "u1", (3,))])
FSUM_SCALE = float(2 ** 40)
SURF_SCALE = float(2 ** 32)   # seg_surf_acc (btpost_surface_distance's acc)


def summarize(precision, recall, iou_thrs, max_dets):
    """COCOeval.summarize as torchmetrics reports it (SURVEY.md A.3) from the accumulate tables
    precision [T, R, nc, A, M] and recall [T, nc, A, M] (numpy float64, -1 = undefined)."""
    nc = precision.shape[2]

    def mean(x):
        x = x[x > -1]
        return float(x.mean()) if x.size else -1.0

    def thr_idx(v):
        for i, t in enumerate(iou_thrs):
            if abs(float(t) - v) < 1e-6:
                return i
        return None
    res = {"map": mean(precision[:, :, :, 0, -1])}
    for name, v in (("map_50", 0.5), ("map_75", 0.75)):
        ti = thr_idx(v)
        res[name] = mean(precision[ti, :, :, 0, -1]) if ti is not None else -1.0
    for ai in (1, 2, 3):
        res[f"map_{AREA_NAMES[ai]}"] = mean(precision[:, :, :, ai, -1])
        res[f"mar_{AREA_NAMES[ai]}"] = mean(recall[:, :, ai, -1])
    for mi, md in enumerate(max_dets):
        res[f"mar_{md}"] = mean(recall[:, :, 0, mi])
    res["map_per_class"] = [mean(precision[:, :, c, 0, -1]) for c in range(nc)]
    res[f"mar_{max_dets[-1]}_per_class"] = [mean(recall[:, c, 0, -1]) for c in range(nc)]
    return res


@torch.no_grad()
def merge_shards(hdr: torch.Tensor, records: torch.Tensor, group=None):
    """Merge the shards of a sweep over `torch.distributed`: `hdr` int64 [HDR] (summed in place by ONE all-reduce: the
    metric-counter all-reduce), `records` uint8 [capacity, 32] of which the first min(hdr[0], capacity) rows are valid
    (one `all_gather_into_tensor`, padded to the largest shard).  Returns (n_per_rank list, records of all ranks
    concatenated in rank order).  Device-agnostic (NCCL on the GPU box, gloo in the CPU tests)."""
    ns, merged = merge_sweeps([hdr], [records], group)
    return ns[0], merged[0]


@torch.no_grad()
def merge_sweeps(hdrs, rings, group=None, extra=()):
    """`merge_shards` for several sweep states at once (the detection sweep and the segmentation-mAP sweep) with the
    same three collectives: the record counts in one all-gather, the headers, concatenated, in ONE all-reduce (each
    `hdrs[s]` is summed in place), the valid records of every state in one `all_gather_into_tensor` (each state padded to
    its largest shard).  `extra`: further int64 counter tensors (the binned curve state), contiguous and on the headers'
    device, concatenated into the same all-reduce and summed in place.  Returns (ns, merged): per state, the n_per_rank
    list and the records of all ranks concatenated in rank order."""
    S = len(hdrs)
    n_local = [int(min(int(h[_lib.SWEEP_N_RECORDS]), r.shape[0])) for h, r in zip(hdrs, rings)]
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return [[n] for n in n_local], [r[:n] for r, n in zip(rings, n_local)]
    W, dev = dist.get_world_size(group), hdrs[0].device
    counts = torch.zeros(W * S, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(counts, torch.tensor(n_local, dtype=torch.int64, device=dev), group=group)
    summed = list(hdrs) + [e.view(-1) for e in extra]
    if len(summed) == 1:
        dist.all_reduce(hdrs[0], group=group)
    else:
        cat = torch.cat(summed)
        dist.all_reduce(cat, group=group)
        for h, v in zip(summed, cat.split([h.numel() for h in summed])):
            h.copy_(v)
    ns = [[int(v) for v in col] for col in zip(*counts.view(W, S).tolist())]   # ns[s][rank]
    caps = [max(max(n), 1) for n in ns]
    rows, rdev = sum(caps), rings[0].device
    if S == 1 and rings[0].shape[0] >= caps[0]:
        send = rings[0][:caps[0]]
    else:   # a ring smaller than the largest shard, or several states back to back: pad (rows beyond n_local are never read)
        send = torch.zeros(rows, REC_BYTES, dtype=torch.uint8, device=rdev)
        o = 0
        for r, n, c in zip(rings, n_local, caps):
            send[o: o + n] = r[:n]
            o += c
    allrec = torch.empty(W * rows, REC_BYTES, dtype=torch.uint8, device=rdev)
    dist.all_gather_into_tensor(allrec, send.contiguous(), group=group)
    if S == 1 and all(n == caps[0] for n in ns[0]):
        return ns, [allrec]                    # equal shards: the gathered buffer is the merged list
    # ragged shards: contiguous 8-byte copies (torch.cat on [n, 32] uint8 rows copies byte by byte: 13 ms for 52 MB on a B200)
    a64, out, base = allrec.view(torch.int64), [], 0
    for s in range(S):
        merged = torch.empty(sum(ns[s]), REC_BYTES, dtype=torch.uint8, device=rdev)
        m64, o = merged.view(torch.int64), 0
        for r in range(W):
            m64[o: o + ns[s][r]].copy_(a64[r * rows + base: r * rows + base + ns[s][r]])
            o += ns[s][r]
        out.append(merged)
        base += caps[s]
    return ns, out


def decode_records(records: torch.Tensor, T: int):
    """uint8 [n, 32] record rows -> dict of numpy arrays (tests / debugging): matched / ignored as bool [n, A, T]."""
    raw = records.detach().cpu().numpy().reshape(-1).view(REC_DTYPE)
    bits = np.arange(4 * T, dtype=np.uint64)
    unpack = lambda w: ((w[:, None] >> bits[None, :]) & np.uint64(1)).astype(bool).reshape(-1, 4, T)
    key = raw["score_key"].astype(np.uint32)
    asc = ~key                                                   # undo desc_key: smaller key = higher score
    u = np.where(asc & np.uint32(0x80000000), asc & np.uint32(0x7FFFFFFF), ~asc).astype(np.uint32)
    return {"score": u.view(np.float32), "label": raw["label"].astype(np.int64), "image": raw["image"].astype(np.int64),
            "rank": raw["rank"].astype(np.int64), "class_rank": raw["class_rank"].astype(np.int64),
            "matched": unpack(raw["matched"]), "ignored": unpack(raw["ignored"])}


class DeviceSweep:
    """Sweep state on one GPU, filled by the CUDA library (`PostProcessor.sweep = DeviceSweep(...)` or
    `Pipeline(..., sweep=...)`).  `capacity` = records the ring can hold (one per kept detection of this rank's
    shard; 32 bytes each).  `seg_map_capacity` > 0 adds a second sweep state for the v3 segmentation mAP
    (`BtIO.seg_sweep`: one record per image, so the number of images of this rank's shard; needs
    `PostConfig.with_seg_map`); `finish()` then also returns the `seg_`-prefixed mAP keys.  `soft_dice=True` (needs
    `PostConfig.with_soft_dice`): `finish()` also returns v3's soft Dice, `seg_soft_dice` (the mean over the images with
    a defined value, NaN when there is none) and `n_soft_dice_images`, from the `seg_soft_acc` header slots.
    `micro=True` adds the class-agnostic state (`BtIOMicro.micro_sweep`, torchmetrics `MeanAveragePrecision(
    average="micro")`: every label counts as one class, so a well-placed box with the wrong class is a hit): one record
    per kept detection, so the same capacity as the detection ring; `finish()` then also returns the `micro_`-prefixed
    mAP / mAR keys and the `micro_precision` / `micro_recall` tables (the per-class keys stay the class-aware ones, as in
    torchmetrics).  `surface=True` (needs `PostConfig.with_surface_dist`): `finish()` also returns the means over the images
    with defined values (NaN when there is none) of the projector mask's Hausdorff distance, HD95 and ASSD, `seg_hd`,
    `seg_hd95` and `seg_assd`, and `n_surface_images`, from the `seg_surf_acc` header slots.  `seg_curve` = T or a list of
    thresholds (needs `PostConfig.seg_curve` with the same thresholds): the sweep owns the binned curve state `seg_curve`
    [2, T+1] (`counters()`), merged in the header all-reduce; `finish()` also returns `seg_curve_thresholds`,
    `seg_curve_confmat` (torchmetrics' [T, 2, 2] state), `seg_pr_curve` (precision, recall, thresholds), `seg_roc` (fpr,
    tpr, thresholds), `seg_ap` and `seg_auroc` of the projector probabilities over every pixel (`btpost.segcurve`)."""

    def __init__(self, nc: int, iou_thrs, max_dets=(1, 10, 100), capacity: int = 1 << 20, max_det_per_image: int = 300,
                 device="cuda:0", seg_map_capacity: int = 0, soft_dice: bool = False, micro: bool = False,
                 surface: bool = False, seg_curve: int | list | None = None):
        self.lib = _lib.load()
        self.nc, self.iou_thrs, self.max_dets = nc, [float(t) for t in iou_thrs], tuple(int(m) for m in max_dets)
        self.T, self.capacity, self.K = len(self.iou_thrs), int(capacity), int(max_det_per_image)
        self.seg_map_capacity = int(seg_map_capacity)
        self.soft_dice = bool(soft_dice)
        self.surface = bool(surface)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("DeviceSweep lives on a CUDA device (the records are written by the CUDA library)")
        if not (0 < len(self.max_dets) <= 4) or nc > 16 or 4 * self.T > 64:
            raise ValueError("DeviceSweep: at most 4 maxDets, 16 classes, 16 IoU thresholds")
        if self.seg_map_capacity < 0:
            raise ValueError("DeviceSweep: seg_map_capacity must be >= 0")
        self.buf, self.hdr, self.records = self._state(self.capacity)
        self.ptr = self.buf.data_ptr()
        self.seg_buf = self.seg_hdr = self.seg_records = self.seg_ptr = None
        if self.seg_map_capacity:
            self.seg_buf, self.seg_hdr, self.seg_records = self._state(self.seg_map_capacity)
            self.seg_ptr = self.seg_buf.data_ptr()
        self.micro_buf = self.micro_hdr = self.micro_records = self.micro_ptr = None
        if micro:
            self.micro_buf, self.micro_hdr, self.micro_records = self._state(self.capacity)
            self.micro_ptr = self.micro_buf.data_ptr()
        u = _lib.SWEEP_USER
        self.cm = self.hdr[u: u + nc * nc].view(nc, nc)
        self.seg_cnt4 = self.hdr[u + 256: u + 260]
        self.uni_cnt4 = self.hdr[u + 260: u + 264]
        self.seg_soft_acc = self.hdr[u + 264: u + 266]   # sum of soft Dice (2^-40 units), images with a defined value
        self.seg_surf_acc = self.hdr[u + 266: u + 270]   # sums of HD, HD95, ASSD (2^-32 units), images with defined values
        self.seg_curve_thresholds = self.seg_curve = None
        if seg_curve is not None:
            self.seg_curve_thresholds = segcurve.thresholds(seg_curve)
            self.seg_curve = torch.zeros(2, len(self.seg_curve_thresholds) + 1, dtype=torch.int64, device=self.device)
        self.rec_thrs = torch.from_numpy(np.linspace(0.0, 1.0, 101)).to(self.device)
        self._md = (C.c_int32 * len(self.max_dets))(*self.max_dets)
        self.reset()

    def _state(self, capacity):
        """(buffer, header view, record-ring view) of one sweep state of `capacity` records."""
        nbytes = C.c_size_t()
        _lib.check(self.lib.btpost_sweep_bytes(C.c_int64(capacity), C.byref(nbytes)), "btpost_sweep_bytes")
        buf = torch.zeros((nbytes.value + 7) // 8, dtype=torch.int64, device=self.device)   # torch allocations are 512-byte aligned
        return buf, buf[:HDR], buf[HDR:].view(torch.uint8)[: capacity * REC_BYTES].view(capacity, REC_BYTES)

    def reserve(self, total_records: int, world: int = 1):
        """Optional: warm torch's caching allocator for `finish()` on a sweep of `total_records` records over `world`
        ranks (the gathered record buffer, the merged copy and the accumulate scratch, for the segmentation ring too), so
        that the end of the sweep does not pay cudaMalloc calls while the GPU waits."""
        def scratch(n):
            sb = C.c_size_t()
            _lib.check(self.lib.btpost_sweep_accumulate_bytes(C.c_int64(int(n)), C.byref(sb)), "btpost_sweep_accumulate_bytes")
            return torch.empty(sb.value, dtype=torch.uint8, device=self.device)

        def tables(nc):
            M = len(self.max_dets)
            return [torch.empty(self.T, 101, nc, 4, M, dtype=torch.float64, device=self.device),
                    torch.empty(self.T, nc, 4, M, dtype=torch.float64, device=self.device)]
        world = max(world, 1)
        per, seg = -(-int(total_records) // world), self.seg_map_capacity
        rows = lambda n: torch.empty(max(n, 1), REC_BYTES, dtype=torch.uint8, device=self.device)
        micro = per if self.micro_ptr is not None else 0
        keep = [scratch(total_records), rows(world * (per + seg + micro)), rows(int(total_records))] + tables(self.nc)
        if seg:
            keep += [scratch(world * seg), rows(per + seg), rows(world * seg)] + tables(1)
        if micro:
            keep += [scratch(total_records), rows(int(total_records))] + tables(1)
        del keep   # back to the allocator's cache

    def counters(self):
        """cm / seg_cnt4 / uni_cnt4 / seg_soft_acc / seg_surf_acc views INSIDE the header, and the seg_curve state when
        the sweep has one: hand them to PostProcessor / Pipeline as accumulators and they are merged by the same
        all-reduce."""
        c = {"cm": self.cm, "seg_cnt4": self.seg_cnt4, "uni_cnt4": self.uni_cnt4, "seg_soft_acc": self.seg_soft_acc,
             "seg_surf_acc": self.seg_surf_acc}
        if self.seg_curve is not None:
            c["seg_curve"] = self.seg_curve
        return c

    def reset(self, stream=None):
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        with torch.cuda.device(self.device):
            for ptr, cap in ((self.ptr, self.capacity), (self.seg_ptr, self.seg_map_capacity), (self.micro_ptr, self.capacity)):
                if ptr is not None:
                    _lib.check(self.lib.btpost_sweep_reset(C.c_void_p(ptr), C.c_int64(cap), C.c_void_p(st.cuda_stream)),
                               "btpost_sweep_reset")
        if self.seg_curve is not None:
            with torch.cuda.stream(st):
                self.seg_curve.zero_()

    def _accumulate(self, rec, n, hdr, nc, max_det_per_image, num_images_bound, scores=False):
        """btpost_sweep_accumulate_ext on `n` merged records (reordered in place) -> (precision, recall) device tables, and
        the score table when `scores`."""
        T, A, M = self.T, 4, len(self.max_dets)
        precision = torch.empty(T, 101, nc, A, M, dtype=torch.float64, device=self.device)
        recall = torch.empty(T, nc, A, M, dtype=torch.float64, device=self.device)
        sc = torch.empty_like(precision) if scores else None
        sb = C.c_size_t()
        _lib.check(self.lib.btpost_sweep_accumulate_bytes(C.c_int64(n), C.byref(sb)), "btpost_sweep_accumulate_bytes")
        scratch = torch.empty(sb.value, dtype=torch.uint8, device=self.device)
        npig = hdr[_lib.SWEEP_NPIG: _lib.SWEEP_NPIG + 64]
        bound = num_images_bound if num_images_bound is not None else (int(rec[:, 20:24].contiguous().view(torch.int32).max()) + 1 if n else 1)
        st = torch.cuda.current_stream(self.device)
        with torch.cuda.device(self.device):
            rc = self.lib.btpost_sweep_accumulate_ext(
                C.c_void_p(rec.data_ptr() if n else 0), C.c_int64(n), C.c_void_p(npig.data_ptr()), C.c_void_p(self.rec_thrs.data_ptr()),
                C.c_int32(101), C.c_int32(nc), C.c_int32(T), self._md, C.c_int32(M), C.c_int32(max_det_per_image), C.c_int64(bound),
                C.c_void_p(precision.data_ptr()), C.c_void_p(recall.data_ptr()), C.c_void_p(sc.data_ptr() if scores else 0),
                C.c_void_p(scratch.data_ptr()), C.c_size_t(sb.value), C.c_void_p(st.cuda_stream))
        _lib.check(rc, "btpost_sweep_accumulate_ext")
        return (precision, recall, sc) if scores else (precision, recall)

    @torch.no_grad()
    def finish(self, group=None, num_images_bound: int | None = None, timings: dict | None = None,
               extended_summary: bool = False) -> dict:
        """End of the sweep: merge the shards (header all-reduce + record all-gather), run COCOeval.accumulate on the
        device and summarize.  Every rank returns the same result.  `extended_summary=True` (torchmetrics'
        flag of that name) also returns COCOeval.accumulate's score table: `scores` next to `precision` / `recall`, and
        `seg_map_scores` / `micro_scores` for the other states (same layout as the precision tables: the confidence at
        which each recall threshold is reached).  `timings` (developer aid): filled with the host time of each stage in
        ms, with a device synchronisation after each."""
        import time as _time
        _t = [_time.perf_counter()]

        def _mark(name):
            if timings is not None:
                torch.cuda.synchronize(self.device)
                now = _time.perf_counter()
                timings[name] = (now - _t[0]) * 1e3
                _t[0] = now

        seg = self.seg_map_capacity > 0
        states = [("", self.hdr, self.records, self.capacity)]
        if seg:
            states.append(("segmentation ", self.seg_hdr, self.seg_records, self.seg_map_capacity))
        micro = self.micro_ptr is not None
        if micro:
            states.append(("class-agnostic ", self.micro_hdr, self.micro_records, self.capacity))
        n_here = [int(h[_lib.SWEEP_N_RECORDS]) for _, h, _, _ in states]
        _mark("read_count")
        for (what, _, _, cap), n in zip(states, n_here):
            if n > cap:
                raise RuntimeError(f"DeviceSweep {what}ring too small: {n} records offered, capacity {cap}")
        hdrs = [h.clone() for _, h, _, _ in states]
        curve = self.seg_curve.clone() if self.seg_curve is not None else None
        ns, recs = merge_sweeps(hdrs, [r for _, _, r, _ in states], group, extra=() if curve is None else (curve,))
        _mark("merge_shards")
        for i, ((_, _, ring, _), rec) in enumerate(zip(states, recs)):
            if sum(ns[i]) and rec.data_ptr() == ring.data_ptr():
                rec = rec.clone()                          # the sort reorders in place: keep the ring as it was
            recs[i] = rec.contiguous()
        hdr, n = hdrs[0], int(sum(ns[0]))
        n_images = int(hdr[_lib.SWEEP_N_IMAGES])
        nc = self.nc
        ext = bool(extended_summary)
        tables = self._accumulate(recs[0], n, hdr, nc, self.K, num_images_bound, ext)
        if seg:
            seg_tables = self._accumulate(recs[1], int(sum(ns[1])), hdrs[1], 1, 1, num_images_bound, ext)
        if micro:
            mi = len(states) - 1
            micro_tables = self._accumulate(recs[mi], int(sum(ns[mi])), hdrs[mi], 1, self.K, num_images_bound, ext)
        _mark("accumulate")
        tables = [t.cpu().numpy() for t in tables]
        pr, rcl = tables[0], tables[1]
        h = hdr.cpu().numpy()
        res = summarize(pr, rcl, self.iou_thrs, self.max_dets)
        if ext:
            res["scores"] = tables[2]
        if seg:
            st = [t.cpu().numpy() for t in seg_tables]
            res.update({f"seg_{k}": v for k, v in summarize(st[0], st[1], self.iou_thrs, self.max_dets).items()})
            # seg_precision is the pixel precision of the projector mask: the seg-mAP tables carry the seg_map_ prefix
            res.update(n_seg_records=int(sum(ns[1])), seg_map_precision=st[0], seg_map_recall=st[1])
            if ext:
                res["seg_map_scores"] = st[2]
        if micro:
            mt = [t.cpu().numpy() for t in micro_tables]
            # the per-class keys stay the class-aware ones (torchmetrics recomputes them in macro mode under "micro")
            res.update({f"micro_{k}": v for k, v in summarize(mt[0], mt[1], self.iou_thrs, self.max_dets).items()
                        if not k.endswith("per_class")})
            res.update(n_micro_records=int(sum(ns[mi])), micro_precision=mt[0], micro_recall=mt[1])
            if ext:
                res["micro_scores"] = mt[2]
        _mark("summarize")
        ni = max(n_images, 1)
        u = _lib.SWEEP_USER
        tp, fp, fn, tn = [int(v) for v in h[u + 256: u + 260]]
        fs = h[_lib.SWEEP_FSUM: _lib.SWEEP_FSUM + 4].astype(np.float64) / FSUM_SCALE
        res.update({
            "n_images": n_images, "n_records": n, "records_per_rank": ns[0], "cm": torch.from_numpy(h[u: u + nc * nc].reshape(nc, nc).copy()),
            "seg_f1": 2 * tp / (2 * tp + fp + fn) if (2 * tp + fp + fn) else 0.0,
            "seg_precision": tp / (tp + fp) if (tp + fp) else 0.0, "seg_recall": tp / (tp + fn) if (tp + fn) else 0.0,
            "seg_accuracy": (tp + tn) / max(tp + tn + fp + fn, 1),
            "seg_dice": float(fs[0]) / ni, "seg_iou": float(fs[1]) / ni, "uni_dice": float(fs[2]) / ni, "uni_iou": float(fs[3]) / ni,
            "npig": h[_lib.SWEEP_NPIG: _lib.SWEEP_NPIG + 64].reshape(4, 16)[:, :nc].copy(), "precision": pr, "recall": rcl,
        })
        if self.soft_dice:
            s, k = int(h[u + 264]), int(h[u + 265])
            res.update(seg_soft_dice=s / FSUM_SCALE / k if k else float("nan"), n_soft_dice_images=k)
        if self.surface:
            k = int(h[u + 269])
            res.update({key: int(h[u + 266 + i]) / SURF_SCALE / k if k else float("nan")
                        for i, key in enumerate(("seg_hd", "seg_hd95", "seg_assd"))}, n_surface_images=k)
        if curve is not None:
            cm = segcurve.confmat(curve)
            m = segcurve.curve_metrics(cm, self.seg_curve_thresholds)
            res.update(seg_curve_thresholds=self.seg_curve_thresholds.copy(), seg_curve_confmat=cm, seg_pr_curve=m["pr_curve"],
                       seg_roc=m["roc"], seg_ap=m["ap"], seg_auroc=m["auroc"])
        return res
