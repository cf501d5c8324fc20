"""Host-side mirror of /root/reference/gapro/gen_ps_utils.py for the GP pseudo-label path and the heuristic labelers.

Same call surface as the reference (names, argument meaning, return arity, dtypes,
shapes — including the per-superpoint `mu`/`var` of gen_ps_utils.py:482), backed by the
CUDA library through `gapro_b200.engine`.  Everything here is host orchestration; the
arithmetic runs in libgapro_b200.so.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from .engine import SceneInputs, get_engine

__all__ = ["gen_pseudo_label_gaussian_process", "gen_pseudo_labels_batch", "gen_pseudo_label_box2mask",
           "gen_pseudo_label", "gen_pseudo_labels_heuristic_batch", "getInstanceInfo", "getInstanceInfo_cuda", "batch_giou_cross", "is_box1_in_box2", "is_within_bb_torch",
           "SceneInputs"]


def gen_pseudo_label_gaussian_process(
    coords_float,
    mask_feats,
    spp,
    instance_cls,
    instance_box,
    instance_box_volume,
    wall_box,
    wall_box_volume,
    instance_classes=18,
    dataset_name="scannetv2",
    ground_h=0.1,
    training_iter=50,
    thresh_spp_occu=0.8,
    *,
    noise_seed=None,
    jitter_zz=1e-4,
    return_debug=False,
):
    """Drop-in for gen_pseudo_label_gaussian_process (/root/reference/gapro/gen_ps_utils.py:293-482).

    Returns (ps_semantic_label[N] int32, ps_instance_label[N] int32, ps_prob_label[N] float32,
    ps_mu_label[S] float32, ps_variance_label[S] float32) on the device of `coords_float`.
    `dataset_name` is accepted and unused, as in the reference.  Keyword-only extras:
    `noise_seed` makes the GP initialisation reproducible (the reference draws it from the
    unseeded global RNG inside gpytorch); `jitter_zz` is gpytorch's K_ZZ jitter (1e-4 since
    gpytorch 1.6, 1e-3 before)."""
    eng = get_engine(coords_float.device if coords_float.is_cuda else None)
    scene = SceneInputs(coords_float, mask_feats, spp, instance_cls, instance_box, instance_box_volume,
                        wall_box, wall_box_volume, noise_seed=noise_seed)
    res = eng.run([scene], instance_classes=instance_classes, ground_h=ground_h, training_iter=training_iter,
                  thresh_spp_occu=thresh_spp_occu, jitter_zz=jitter_zz, debug=return_debug, want_cnt_in=return_debug)
    if return_debug:
        return res[0][0], res[1]
    return res[0]


class BatchResults(list):
    """One 5-tuple per scene; with on_error="mark" a scene whose GP fit failed holds None and `.errors` maps its
    batch index to the message."""
    errors: dict = {}


def gen_pseudo_labels_batch(scenes, instance_classes=18, ground_h=0.1, training_iter=50, thresh_spp_occu=0.8,
                            jitter_zz=1e-4, device=None, return_debug=False, on_error="raise"):
    """Many scenes through ONE pass of the hot path (scenes are independent: gen_ps.py:36).
    `scenes` is a sequence of SceneInputs; returns one 5-tuple per scene.  A GP region that cannot be fitted
    (NotPSDError after the jitter retries / NanError — where the reference dies, gen_ps_utils.py:434-437) fails
    its own scene only: on_error="raise" raises GaproSceneError carrying the other scenes' results,
    on_error="mark" returns None at that position."""
    eng = get_engine(device)
    res = eng.run(list(scenes), instance_classes=instance_classes, ground_h=ground_h, training_iter=training_iter,
                  thresh_spp_occu=thresh_spp_occu, jitter_zz=jitter_zz, debug=return_debug, on_error=on_error)
    if return_debug:
        return res
    out = BatchResults(res)
    out.errors = dict(eng.last_errors)
    return out


def gen_pseudo_label_box2mask(coords_float, spp, instance_cls, instance_box, instance_box_volume,
                              instance_classes=18, dataset_name="scannetv2"):
    """Drop-in for gen_pseudo_label_box2mask (/root/reference/gapro/gen_ps_utils.py:242-290): points in
    several boxes take the smallest one; for scannetv2 the labels are then aligned to superpoints by
    majority vote (spp_align_label, :99-129).  Returns (ps_semantic_label[N] int32, ps_instance_label[N] int32)."""
    return _heuristic_one(coords_float, spp, instance_cls, instance_box, instance_box_volume, "box2mask",
                          instance_classes, dataset_name)


def gen_pseudo_label(coords_float, spp, instance_cls, instance_box, instance_box_volume, instance_classes=18,
                     dataset_name="scannetv2", heuristic_rule="volume"):
    """Drop-in for gen_pseudo_label (/root/reference/gapro/gen_ps_utils.py:485-569): rule "volume", "dist" or
    "none" for points in several boxes; for scannetv2 a majority vote per superpoint in which a box can only
    win if it holds at least 70 % of the superpoint (:538-550)."""
    if heuristic_rule not in ("volume", "dist", "none"):
        raise Exception
    return _heuristic_one(coords_float, spp, instance_cls, instance_box, instance_box_volume, heuristic_rule,
                          instance_classes, dataset_name)


# method -> (rule for points in several boxes, occupancy a box needs to win a superpoint's vote)
HEURISTIC_METHODS = {"box2mask": ("volume", None), "volume": ("volume", 0.7), "dist": ("dist", 0.7),
                     "none": ("none", 0.7)}


def _heuristic_one(coords_float, spp, instance_cls, instance_box, instance_box_volume, method, instance_classes,
                   dataset_name):
    scene = SceneInputs(coords_float, None, spp, instance_cls, instance_box, instance_box_volume)
    return gen_pseudo_labels_heuristic_batch([scene], method=method, instance_classes=instance_classes,
                                             dataset_name=dataset_name,
                                             device=coords_float.device if coords_float.is_cuda else None)[0]


def gen_pseudo_labels_heuristic_batch(scenes, method="box2mask", instance_classes=18, dataset_name="scannetv2",
                                      device=None):
    """Many scenes through ONE pass of the heuristic labelers.  `scenes` is a sequence of SceneInputs, of which only
    coords_float, spp and the instance boxes / classes / volumes are read (no wall boxes, no floor slab).
    method "box2mask" labels as gen_pseudo_label_box2mask, "volume" / "dist" / "none" as gen_pseudo_label with
    that heuristic_rule; for scannetv2 the labels are aligned to superpoints, otherwise (s3dis) they stay per point.
    Returns one (ps_semantic_label[N] int32, ps_instance_label[N] int32) pair per scene."""
    if method not in HEURISTIC_METHODS:
        raise ValueError(f"unknown heuristic method {method!r}; expected one of {sorted(HEURISTIC_METHODS)}")
    rule, occ_thresh = HEURISTIC_METHODS[method]
    eng = get_engine(device)
    return eng.run_heuristic(list(scenes), rule=rule, spp_align=(dataset_name == "scannetv2"), occ_thresh=occ_thresh,
                             instance_classes=instance_classes)


# --------------------------------------------------------------------------------------------
# host helpers of the reference's call surface
# --------------------------------------------------------------------------------------------
def getInstanceInfo(xyz, instance_label, semantic_label, dataset_name="scannetv2"):
    """Per-instance axis-aligned boxes from labelled points — same contract as
    getInstanceInfo (/root/reference/gapro/gen_ps_utils.py:195-239): instances are listed in
    increasing GT id with empty ids skipped, class = semantic label of the instance's first
    point (minus 2 for scannetv2 unless -100), volume = prod(clip(max-min, 0)); returns None
    when there is no instance.  Vectorised (one stable sort) instead of a per-instance scan."""
    xyz = np.asarray(xyz)
    inst = np.asarray(instance_label)
    sem = np.asarray(semantic_label)
    instance_num = int(inst.max()) + 1
    corners_label = np.full((xyz.shape[0], 6), -100.0, dtype=np.float32)
    idx = np.flatnonzero((inst >= 0) & (inst == np.floor(inst)))
    if idx.size == 0:
        return None
    ids = inst[idx].astype(np.int64)
    order = np.argsort(ids, kind="stable")
    idx, ids = idx[order], ids[order]
    starts = np.flatnonzero(np.r_[True, ids[1:] != ids[:-1]])
    pts = xyz[idx]
    lo = np.minimum.reduceat(pts, starts, axis=0)
    hi = np.maximum.reduceat(pts, starts, axis=0)
    seg = np.cumsum(np.r_[True, ids[1:] != ids[:-1]]) - 1
    corners_label[idx, :3] = lo[seg] - pts
    corners_label[idx, 3:] = hi[seg] - pts
    instance_cls = np.array(sem[idx[starts]])
    instance_box = np.concatenate([lo, hi], axis=1)
    ext = np.clip(hi - lo, 0.0, None)
    instance_box_volume = ext[:, 0] * ext[:, 1] * ext[:, 2]
    if dataset_name == "scannetv2":
        instance_cls[instance_cls != -100] -= 2
    return instance_num, instance_cls, instance_box, instance_box_volume, corners_label


def getInstanceInfo_cuda(xyz, instance_label, semantic_label, dataset_name="scannetv2"):
    """getInstanceInfo on the device (gapro_instance_info): same instance order, boxes, classes and volumes as
    the host version (bit for bit: min / max are exact and the volume is the same float64 product), from CUDA
    tensors xyz (N,3) float64, instance_label / semantic_label (N,) float64.  Returns
    (instance_num, instance_cls (K,) float64, instance_box (K,6) float64, instance_box_volume (K,) float64) as
    device tensors, or None when no instance is labelled (gen_ps_utils.py:229-230).  `corners_label` - never read by
    gen_ps.py - is not produced."""
    if not xyz.is_cuda:
        raise _lib.GaproError("getInstanceInfo_cuda needs CUDA tensors; use getInstanceInfo on the host")
    lib = _lib.load()
    dev = xyz.device
    xyz = xyz.to(torch.float64).contiguous()
    inst = instance_label.to(dev, torch.float64).contiguous()
    sem = semantic_label.to(dev, torch.float64).contiguous()
    n_ids = int(inst.max().item()) + 1
    if n_ids <= 0:
        return None
    boxes = torch.empty((n_ids, 6), dtype=torch.float64, device=dev)
    vol = torch.empty(n_ids, dtype=torch.float64, device=dev)
    cls = torch.empty(n_ids, dtype=torch.float64, device=dev)
    n_used = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = torch.empty(lib.gapro_instance_info_workspace_bytes(n_ids), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.gapro_instance_info(xyz.data_ptr(), inst.data_ptr(), sem.data_ptr(), xyz.shape[0], n_ids,
                                           1 if dataset_name == "scannetv2" else 0, boxes.data_ptr(), vol.data_ptr(),
                                           cls.data_ptr(), n_used.data_ptr(), ws.data_ptr(), ws.numel(),
                                           torch.cuda.current_stream(dev).cuda_stream), "gapro_instance_info")
    k = int(n_used.item())
    if k == 0:
        return None
    return n_ids, cls[:k], boxes[:k], vol[:k]


def batch_giou_cross(boxes1, boxes2):
    """IoU / GIoU of every box of `boxes1` (N,6) with every box of `boxes2` (M,6) — the
    formulas of /root/reference/gapro/gen_ps_utils.py:33-61 (1e-6 in both denominators)."""
    a, b = boxes1[:, None, :], boxes2[None, :, :]
    inter = (torch.minimum(a[..., 3:], b[..., 3:]) - torch.maximum(a[..., :3], b[..., :3])).clamp(min=0.0).prod(-1)
    va = (a[..., 3:] - a[..., :3]).clamp(min=0.0).prod(-1)
    vb = (b[..., 3:] - b[..., :3]).clamp(min=0.0).prod(-1)
    union = va + vb - inter
    iou = inter / (union + 1e-6)
    hull = (torch.maximum(a[..., 3:], b[..., 3:]) - torch.minimum(a[..., :3], b[..., :3])).clamp(min=0.0).prod(-1)
    return iou, iou - (hull - union) / (hull + 1e-6)


def is_box1_in_box2(box1, box2, offset=0.05):
    """/root/reference/gapro/gen_ps_utils.py:75-76."""
    return torch.all((box1[:3] + offset) >= box2[:3]) & torch.all((box1[3:] - offset) <= box2[3:])


def is_within_bb_torch(points, bb_min, bb_max):
    """/root/reference/gapro/gen_ps_utils.py:79-80 (kept for API parity; the hot path uses the
    fused CUDA containment kernel, not this)."""
    return torch.all(points >= bb_min, dim=-1) & torch.all(points <= bb_max, dim=-1)
