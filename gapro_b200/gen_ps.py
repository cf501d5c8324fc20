"""CLI and per-scene host steps of the pseudo-label generator — the counterpart of
/root/reference/gapro/gen_ps.py.

    python -m gapro_b200.gen_ps [--save_folder D] [--use_deepfeat] [--deepfeat_folder D] [--eval_pslabel]
                                [--label_method {gp,box2mask,volume,dist,none}]

keeps the reference flags (gen_ps.py:15-21), the relative dataset layout
(dataset/scannetv2/{train,superpoints,scans_transform}), the output naming
<save_folder>/<scan_name>.pth with scan_name = basename[:12] (gen_ps.py:37-39), the
skip-if-exists resume rule (:39-41) and the saved tuple of five numpy arrays (:126-132).
Additions: scenes are processed in batches on the GPU, and when launched under torchrun
the sorted scene list is sharded across ranks (one process per GPU, no per-step collective;
one final gather of per-scene metadata).  --label_method other than gp writes the box-only
heuristic labels instead (the alternative commented out at gen_ps.py:112-114:
gen_pseudo_label_box2mask, or gen_pseudo_label with rule volume / dist / none), superpoint-aligned,
in the same 5-tuple with prob = 1 and mu = var = -100; scenes are sharded round-robin, there is no
GP cost pass.
"""
from __future__ import annotations

import argparse
import os
import os.path as osp
import time
import zlib
from glob import glob

import numpy as np
import torch

from .engine import SceneInputs
from .gen_ps_utils import gen_pseudo_labels_batch, gen_pseudo_labels_heuristic_batch, getInstanceInfo
from .sharding import gather_records, shard_scenes

DATA_ROOT = "dataset/scannetv2"


def read_axis_align_matrix(meta_file: str) -> np.ndarray:
    """The 'axisAlignment = ...' line of a ScanNet scene meta file (gen_ps.py:58-64)."""
    with open(meta_file) as f:
        for line in f:
            if "axisAlignment" in line:
                vals = [float(x) for x in line.split("=", 1)[1].split()]
                return np.array(vals, dtype=np.float64).reshape(4, 4)
    raise ValueError(f"no axisAlignment line in {meta_file}")


def prepare_inputs(xyz, rgb, semantic_label, instance_label, spp, axis_align_matrix, wall_box=None,
                   wall_volume=None, deep_feats=None, dataset_name="scannetv2", device_boxes=False):
    """Host steps of gen_ps.py:48-77 on numpy arrays.  NOTE the reference builds the GP features
    from the UN-aligned xyz (concat at :55 happens before the alignment at :66-69); kept.
    device_boxes=True leaves getInstanceInfo (:72-74) to the GPU: the labels travel with the scene and
    `to_scene_inputs` derives the boxes there (gapro_instance_info)."""
    xyz = np.asarray(xyz)
    mask_feats = np.asarray(deep_feats) if deep_feats is not None else np.concatenate([xyz, np.asarray(rgb)], axis=-1)
    pts = np.ones((xyz.shape[0], 4))
    pts[:, 0:3] = xyz[:, 0:3]
    xyz_al = np.dot(pts, np.asarray(axis_align_matrix).transpose())[:, :3]
    if device_boxes:
        inst = np.asarray(instance_label, dtype=np.float64)
        if not np.any(inst >= 0):
            raise ValueError("scene has no labelled instance (getInstanceInfo returned None, gen_ps_utils.py:229-230)")
        return dict(xyz=xyz_al, mask_feats=mask_feats, spp=np.asarray(spp), instance_label=inst,
                    semantic_label=np.asarray(semantic_label, dtype=np.float64), dataset_name=dataset_name,
                    wall_box=wall_box if wall_box is not None else [],
                    wall_volume=wall_volume if wall_volume is not None else [])
    info = getInstanceInfo(xyz_al, instance_label=instance_label, semantic_label=semantic_label,
                           dataset_name=dataset_name)
    if info is None:
        raise ValueError("scene has no labelled instance (getInstanceInfo returned None, gen_ps_utils.py:229-230)")
    _, instance_cls, instance_box, instance_box_volume, _ = info
    return dict(xyz=xyz_al, mask_feats=mask_feats, spp=np.asarray(spp), instance_cls=instance_cls,
                instance_box=instance_box, instance_box_volume=instance_box_volume,
                wall_box=wall_box if wall_box is not None else [], wall_volume=wall_volume if wall_volume is not None else [])


def to_scene_inputs(inp: dict, device, noise_seed=None, pin=False) -> SceneInputs:
    """Host -> device boundary of gen_ps.py:79-89 (dtypes as there: xyz stays float64, boxes and
    features become float32, classes int64)."""
    def dev(a, dtype):
        t = torch.from_numpy(np.ascontiguousarray(a)).to(dtype)
        if pin:
            t = t.pin_memory()
        return t.to(device, non_blocking=pin)

    wall_box, wall_vol = inp["wall_box"], inp["wall_volume"]
    has_wall = len(wall_box) > 0
    coords = dev(inp["xyz"], torch.float64)
    if "instance_box" in inp:
        cls, box, vol = (dev(inp["instance_cls"], torch.int64), dev(inp["instance_box"], torch.float32),
                         dev(inp["instance_box_volume"], torch.float32))
    else:       # boxes from the labelled points on the device (getInstanceInfo, gen_ps.py:72-74), then the casts of :79-81
        from .gen_ps_utils import getInstanceInfo_cuda
        info = getInstanceInfo_cuda(coords, dev(inp["instance_label"], torch.float64), dev(inp["semantic_label"], torch.float64),
                                    dataset_name=inp.get("dataset_name", "scannetv2"))
        if info is None:
            raise ValueError("scene has no labelled instance (getInstanceInfo returned None, gen_ps_utils.py:229-230)")
        cls, box, vol = info[1].long(), info[2].float(), info[3].float()
    return SceneInputs(
        coords_float=coords,
        mask_feats=dev(inp["mask_feats"], torch.float32),
        spp=dev(inp["spp"], torch.int64),
        instance_cls=cls,
        instance_box=box,
        instance_box_volume=vol,
        wall_box=dev(wall_box, torch.float32) if has_wall else [],
        wall_box_volume=dev(wall_vol, torch.float32) if has_wall else [],
        noise_seed=noise_seed,
    )


def synthetic_inputs(scene, use_deepfeat=False) -> dict:
    """gapro_b200.synthetic.Scene -> the dict prepare_inputs returns."""
    return prepare_inputs(scene.xyz_raw, scene.rgb, scene.sem, scene.inst, scene.spp, scene.axis_align,
                          wall_box=scene.wall_box, wall_volume=scene.wall_volume,
                          deep_feats=scene.deep_feats if use_deepfeat else None)


def load_scene(filename, scan_name, use_deepfeat=False, deepfeat_folder=None, data_root=DATA_ROOT, device_boxes=False):
    """Disk -> host arrays for one scene (gen_ps.py:45-77): scene tuple, superpoints, optional deep
    features, axis alignment, instance boxes, optional wall boxes.  Returns (inputs, sem, inst)."""
    from .scannet_planes import get_wall_boxes
    xyz, rgb, sem, inst = torch.load(filename, weights_only=False)
    spp = torch.load(osp.join(data_root, "superpoints", scan_name + ".pth"), weights_only=False)
    deep = torch.load(osp.join(deepfeat_folder, scan_name + ".pth"), weights_only=False) if use_deepfeat else None
    A = read_axis_align_matrix(osp.join(data_root, "scans_transform", scan_name, scan_name + ".txt"))
    _, wall_box, wall_vol = get_wall_boxes(scan_name, planes_root=osp.join(data_root, "scannet_planes"),
                                           transform_root=osp.join(data_root, "scans_transform"))
    return prepare_inputs(xyz, rgb, sem, inst, spp, A, wall_box, wall_vol, deep, device_boxes=device_boxes), sem, inst


def save_pseudo_labels(path, result, per_point_uncertainty=False, spp_dense=None):
    """torch.save of the 5-tuple of numpy arrays (gen_ps.py:126-132).  The reference saves mu/var
    per SUPERPOINT although its consumers index them per point (SURVEY.md Q1);
    per_point_uncertainty=True saves mu[spp], var[spp] instead."""
    sem, inst, prob, mu, var = result
    if per_point_uncertainty:
        mu, var = mu[spp_dense], var[spp_dense]
    arrs = (sem.int().cpu().numpy(), inst.int().cpu().numpy(), prob.cpu().numpy(), mu.cpu().numpy(), var.cpu().numpy())
    tmp = path + ".tmp%d" % os.getpid()
    torch.save(arrs, tmp)
    os.replace(tmp, path)


def heuristic_result(sem, inst, spp):
    """Heuristic labels as the 5-tuple the GP path saves: prob = 1 per point, mu = var = -100 (the reference's
    "no GP value") per superpoint of the scene's raw superpoint ids `spp`."""
    n_spp = int(torch.unique(spp).numel())
    prob = torch.ones(sem.shape[0], dtype=torch.float32, device=sem.device)
    none = torch.full((n_spp,), -100.0, dtype=torch.float32, device=sem.device)
    return sem, inst, prob, none, none


def _dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def _load_batch(pool, chunk, args):
    """Disk -> host for a batch on worker threads; a scene that cannot be loaded (missing file, no labelled
    instance - SURVEY Q9, where the reference crashes) is reported and skipped, the rest of the batch goes on."""
    futs = [pool.submit(load_scene, fn, scan, args.use_deepfeat, args.deepfeat_folder, DATA_ROOT, args.device_boxes)
            for fn, scan in chunk]

    def collect():
        out = []
        for (fn, scan), f in zip(chunk, futs):
            try:
                out.append((fn, scan, f.result(), None))
            except Exception as e:      # noqa: BLE001 - reported per scene, never fatal for the other scenes
                out.append((fn, scan, None, f"{type(e).__name__}: {e}"))
        return out
    return collect


def estimate_costs(items, args, device, pool):
    """Cheap pass over `items` (stages U, F, A, A', P — no GP): seconds-of-GPU estimate per scene for the
    cost-balanced sharding (SURVEY 8e: per-scene cost ~ sum of M^3 over its GP regions, orders of magnitude
    apart between scenes)."""
    from .engine import get_engine
    from .sharding import scene_cost
    eng = get_engine(device)
    costs = {}
    chunks = [items[i:i + args.batch_scenes] for i in range(0, len(items), args.batch_scenes)]
    pending = _load_batch(pool, chunks[0], args) if chunks else None
    for ci, chunk in enumerate(chunks):
        loaded = pending()
        pending = _load_batch(pool, chunks[ci + 1], args) if ci + 1 < len(chunks) else None
        ok = [(scan, inp) for _, scan, inp, err in loaded if err is None]
        for _, scan, _, err in loaded:
            if err is not None:
                costs[scan] = 0.0
        if not ok:
            continue
        scenes = [to_scene_inputs(inp[0], device, pin=True) for _, inp in ok]
        st = eng.run(scenes, thresh_spp_occu=0.999, plan_only=True)
        for k, (scan, _) in enumerate(ok):
            costs[scan] = scene_cost(st["sum_m3"][k], st["n_points"][k], st["n_regions"][k], st["sum_m2"][k])
    return costs


LABEL_METHODS = ("gp", "box2mask", "volume", "dist", "none")


def parse_args(argv=None):
    parser = argparse.ArgumentParser("GaPro_GenPS")
    parser.add_argument("--save_folder", type=str, default=osp.join(DATA_ROOT, "gaussian_process_kl_pseudo_labels"))
    parser.add_argument("--use_deepfeat", action="store_true")
    parser.add_argument("--deepfeat_folder", type=str, default=osp.join(DATA_ROOT, "pretrain_maskfeats2"))
    parser.add_argument("--eval_pslabel", action="store_true")
    # additions
    parser.add_argument("--batch_scenes", type=int, default=16, help="scenes per GPU pass")
    parser.add_argument("--seed", type=int, default=None, help="seed of the GP initialisation noise")
    parser.add_argument("--load_workers", type=int, default=8, help="host threads reading / preparing the next batch")
    parser.add_argument("--per_point_uncertainty", action="store_true",
                        help="save mu/var broadcast to points (what the ISBNet/SPFormer loaders index)")
    parser.add_argument("--jitter_zz", type=float, default=1e-4,
                        help="K_ZZ jitter of the variational strategy: 1e-4 is gpytorch >= 1.6 (float32 "
                             "settings.variational_cholesky_jitter), 1e-3 the add_jitter() default of gpytorch <= 1.5; "
                             "the reference does not pin a gpytorch version")
    parser.add_argument("--device_boxes", action="store_true",
                        help="derive the instance boxes from the labelled points on the GPU (gapro_instance_info) "
                             "instead of in the host loader threads; identical boxes")
    parser.add_argument("--balance", choices=["cost", "static"], default="cost",
                        help="multi-GPU sharding: LPT by a cost estimated from the cheap stages, or round-robin")
    parser.add_argument("--label_method", choices=LABEL_METHODS, default="gp",
                        help="gp: the GP labels of gen_ps.py; box2mask: gen_pseudo_label_box2mask; volume / dist / "
                             "none: gen_pseudo_label with that heuristic rule (the alternative commented out at "
                             "gen_ps.py:112-114).  The heuristic methods save prob = 1 and mu = var = -100")
    args = parser.parse_args(argv)
    if args.label_method != "gp" and args.use_deepfeat:
        parser.error(f"--use_deepfeat has no effect with --label_method {args.label_method}: "
                     "the heuristic labelers read no features")
    return args


def main(argv=None):
    args = parse_args(argv)
    heuristic = args.label_method != "gp"

    rank, world, local = _dist_env()
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    os.makedirs(args.save_folder, exist_ok=True)

    # ONE view of the work list for every rank: rank 0 applies the resume rule (gen_ps.py:39-41) and broadcasts,
    # so ranks that list the save folder at different moments cannot disagree about who owns which scene
    todo = None
    if rank == 0:
        filenames = sorted(glob(osp.join(DATA_ROOT, "train", "*_inst_nostuff.pth")))
        todo = [(fn, osp.basename(fn)[:12]) for fn in filenames
                if not osp.exists(osp.join(args.save_folder, osp.basename(fn)[:12] + ".pth"))]
    if world > 1:
        box = [todo]
        dist.broadcast_object_list(box, src=0)
        todo = box[0]

    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(max_workers=max(1, min(args.load_workers, args.batch_scenes)))
    t0 = time.time()
    balance = None
    if world > 1 and args.balance == "cost" and todo and not heuristic:      # no GP work to balance otherwise
        from .sharding import balance_stats, lpt_assignment
        part = estimate_costs(todo[rank::world], args, device, pool)
        merged = {}
        for d in gather_records([part], world):
            merged.update(d)
        costs = [merged.get(scan, 0.0) for _, scan in todo]
        assign = lpt_assignment(costs, world)
        balance = balance_stats(costs, assign)
        todo = [todo[i] for i in assign[rank]]          # heavy scenes first
    else:
        todo = shard_scenes(todo, rank, world)

    from .eval_ps_labels import get_miou_scene
    ious, meta = [], []
    chunks = [todo[i:i + args.batch_scenes] for i in range(0, len(todo), args.batch_scenes)]
    # host side of the NEXT batch (disk reads, alignment, boxes) runs on worker threads while the GPU
    # works on the current one
    pending = _load_batch(pool, chunks[0], args) if chunks else None
    for ci, chunk in enumerate(chunks):
        loaded = pending()
        pending = _load_batch(pool, chunks[ci + 1], args) if ci + 1 < len(chunks) else None
        scenes, kept = [], []
        for fn, scan, res, err in loaded:
            if err is not None:
                print(f"[rank {rank}] {scan}: not labelled - {err}", flush=True)
                meta.append((scan, 0, 0, err))
                continue
            inp, sem, inst = res
            seed = None if args.seed is None else (zlib.crc32(scan.encode()) ^ args.seed) & 0x7fffffff
            scenes.append(to_scene_inputs(inp, device, noise_seed=seed, pin=True))
            kept.append((scan, sem, inst))
        if not scenes:
            continue
        if heuristic:
            labels = gen_pseudo_labels_heuristic_batch(scenes, method=args.label_method, instance_classes=18,
                                                       dataset_name="scannetv2", device=device)
            results, errors = [heuristic_result(s, i, sc.spp) for (s, i), sc in zip(labels, scenes)], {}
        else:
            results = gen_pseudo_labels_batch(scenes, instance_classes=18, ground_h=0.1, training_iter=50,
                                              thresh_spp_occu=0.999, jitter_zz=args.jitter_zz, device=device,
                                              on_error="mark")                          # gen_ps.py:106-110
            errors = results.errors
        for k, ((scan, sem, inst), res, sc) in enumerate(zip(kept, results, scenes)):
            if res is None:      # a GP region of this scene failed: the scene is reported, the others are saved
                print(f"[rank {rank}] {scan}: not labelled - {errors.get(k)}", flush=True)
                meta.append((scan, 0, 0, errors.get(k)))
                continue
            if args.eval_pslabel:      # gen_ps.py:116-124
                s = torch.from_numpy(np.asarray(sem)).to(device).int()
                g = torch.from_numpy(np.asarray(inst)).to(device).int()
                s[s != -100] -= 2
                s[(s == -1) | (s == -2)] = 18
                iou = get_miou_scene(s.long(), g.long(), res[0].long(), res[1].long())
                print("miou", iou)
                ious.append(iou)
            dense = torch.unique(sc.spp, return_inverse=True)[1] if args.per_point_uncertainty else None
            save_pseudo_labels(osp.join(args.save_folder, scan + ".pth"), res, args.per_point_uncertainty, dense)
            meta.append((scan, int(res[0].numel()), int(res[3].numel()), None))
    t_rank = time.time() - t0
    if args.eval_pslabel:
        local_iou = torch.cat(ious) if ious else torch.zeros(0, device=device)
        if world > 1:
            gathered = [None] * world
            dist.all_gather_object(gathered, local_iou.cpu())
            local_iou = torch.cat(gathered)
        if rank == 0 and local_iou.numel():
            print("Mean instance iou of pseudo labels", torch.mean(local_iou.float()).item())
    if world > 1:
        records = gather_records(meta, world)       # the one collective of the labelling pass: label metadata
        walls = gather_records([t_rank], world)
        if rank == 0:
            failed = [m for m in records if m[3] is not None]
            print(f"{len(records) - len(failed)} scenes / {sum(m[1] for m in records)} points labelled on {world} GPUs "
                  f"in {time.time() - t0:.1f}s; per-rank wall max/mean {max(walls) / (sum(walls) / world):.3f}"
                  + (f"; estimated load max/mean {balance['max_over_mean']:.3f}" if balance else "")
                  + (f"; {len(failed)} scenes FAILED: {[m[0] for m in failed]}" if failed else ""))
        dist.destroy_process_group()
    if rank == 0:
        print("Finish")


if __name__ == "__main__":
    main()
