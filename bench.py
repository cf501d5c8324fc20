#!/usr/bin/env python
"""Benchmark of the pseudo-label generator hot path (BASELINE.json metric: scenes/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step is one pass of the whole hot path over one batch of synthetic ScanNet-shaped scenes
per GPU (configs[2] of BASELINE.json: scenes of the 1201-scene ScanNetv2-train-shaped set,
N ~ U(50k, 250k) points); scenes shard across ranks with no data-path collective (weak
scaling), one final NCCL gather of label metadata.  Prints ONE JSON line on rank 0.

`--impl reference` times the CPU restatement of the reference (oracle/, gpytorch precision
policy: float32 everywhere, float64 Cholesky + solve) on the host cores — the reference itself
cannot be installed here (gpytorch and torch_scatter are absent, see DESIGN.md).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "scenes/sec pseudo-labelled"
WORKLOADS = {
    "c3": "c3: ScanNetv2-train-shaped synthetic scenes (scene i of the 1201-scene list: N~U(50k,250k) pts, 12-40 boxes + 4 walls + floor, D=6)",
    "c1": "c1: ScanNet-shaped synthetic scenes (150k pts, 30 boxes + 4 walls + floor, ~4.7k superpoints, D=6)",
    "c1_deep": "c1_deep: c1 with 32-d deep features (--use_deepfeat)",
    "c4": "c4: heavy-overlap stress (400k pts, 80 boxes incl. 20 nested and two structures whose pair is one region of ~8k superpoints, M > 5k)",
    "c5": "c5: S3DIS-area-shaped large rooms (1M pts, 120 boxes + 4 walls + floor, ~34k superpoints, regions up to M ~ 3.6k)",
    "small": "small: 20k-point test scenes", "tiny": "tiny: 6k-point test scenes",
}


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def scene_ids(args, world):
    """Scene indices of the job.  strong: the first --total-scenes scenes of the workload's list, whatever N is
    (BASELINE configs[2]: a fixed scene list sharded over 1/2/4/8 GPUs).  weak: --scenes per GPU (round-1 shape)."""
    n = args.total_scenes if args.mode == "strong" else args.scenes * world
    return list(range(n))


def make_input(idx, workload):
    from gapro_b200 import synthetic
    from gapro_b200.gen_ps import synthetic_inputs
    cfg = synthetic.c3_config(idx) if workload == "c3" else synthetic.CONFIGS[workload]
    return synthetic_inputs(synthetic.make_scene(1000 + idx, cfg), use_deepfeat=cfg.feat_dim == 32)


def static_config(args, world):
    """The part of `config` both arms share word for word (the driver compares the two lines' configs)."""
    ids = scene_ids(args, world)
    return {"workload": WORKLOADS[args.workload], "mode": args.mode, "total_scenes": len(ids),
            "scenes_per_pass": args.scenes, "gp_iters": 50, "thresh_spp_occu": 0.999,
            "sharding": "LPT by the cost the cheap stages A/A'/P estimate (sum M^3 per scene)" if world > 1 else "single GPU",
            "l2": "256 MiB buffer written between passes (flush)"}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle with the reference's precision policy, regions spread over all host cores
# ------------------------------------------------------------------------------------------------
def _warm_worker():
    """Pool initializer: absorb torch's one-off first-call cost (seconds) outside the timed region."""
    try:
        import torch as _t
        from oracle import gp_oracle
        _t.set_num_threads(1)
        r = np.random.default_rng(0)
        gp_oracle.fit_region_autograd(r.normal(size=(6, 3)).astype(np.float32), 3, r.normal(size=(2, 3)).astype(np.float32),
                                      r.normal(size=6).astype(np.float32), iters=2, policy="gpytorch")
    except Exception:      # never let a failing initializer make the pool respawn workers forever
        pass


def _noop(_):
    return 0


def _fit_one(job):
    import torch as _t
    from oracle import gp_oracle
    _t.set_num_threads(1)
    X, n1, Xt, nz = job
    t0 = time.perf_counter()
    gp_oracle.fit_region_autograd(X, n1, Xt, nz, policy="gpytorch")
    return time.perf_counter() - t0


def _cpu_cost_model(m):
    """Rough single-core seconds of one 50-step fit with M rows (launch-overhead, M^2 and M^3 terms; SURVEY section 6
    figures).  Only used as the size measure of the ratio estimator below - a constant factor cancels."""
    m = np.asarray(m, dtype=np.float64)
    return 0.15 + 2e-6 * m ** 2 + 2e-9 * m ** 3


def cpu_scene_sample(inp, budget_s, pool, n_workers, rng):
    """One bounded step of the CPU arm on one scene: the scene-level stages are timed in full; the GP regions are
    timed on a RANDOM subset (a prefix of a random permutation, so it is a uniform sample whatever its length)
    that fits the budget.  Returns (seconds spent, fraction of the scene's work that was done)."""
    from oracle import gen_ps_oracle as O
    jobs = []

    def record(X, n1, Xt, nz):
        jobs.append((np.array(X), n1, np.array(Xt), np.array(nz)))
        n = len(Xt)
        return dict(conf=np.full(n, 0.75, np.float32), label=np.ones(n, bool), mu=np.zeros(n, np.float32),
                    var=np.ones(n, np.float32))

    t0 = time.perf_counter()
    O.gen_pseudo_label_oracle(inp["xyz"], inp["mask_feats"].astype(np.float32), inp["spp"],
                              inp["instance_cls"].astype(np.int64), inp["instance_box"].astype(np.float32),
                              inp["instance_box_volume"].astype(np.float32), inp["wall_box"], inp["wall_volume"],
                              thresh_spp_occu=0.999, fit_fn=record)
    t_stage = time.perf_counter() - t0
    if not jobs:
        return t_stage, 1.0, 0, 0
    cost = _cpu_cost_model([len(j[0]) for j in jobs])
    order = rng.permutation(len(jobs))
    done, t_reg = 0, 0.0
    group = max(n_workers, 1)
    while done < len(jobs) and (done == 0 or t_reg < budget_s - t_stage):
        sel = order[done:done + group]
        t1 = time.perf_counter()
        list(pool.imap_unordered(_fit_one, [jobs[i] for i in sel]))
        t_reg += time.perf_counter() - t1
        done += len(sel)
    frac_gp = cost[order[:done]].sum() / cost.sum()
    spent = t_stage + t_reg
    est_full = t_stage + t_reg / frac_gp            # ratio estimator of the scene's full CPU time
    return spent, spent / est_full, done, len(jobs)


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    import multiprocessing as mp
    n_workers = len(os.sched_getaffinity(0))
    ids = scene_ids(args, world)
    budget = args.cpu_budget or max(4.0, min(30.0, 150.0 / max(args.steps + args.warmup, 1)))
    ctx = mp.get_context("fork")
    rng = np.random.default_rng(0)
    spent, fracs, log = [], [], []
    with ctx.Pool(n_workers, initializer=_warm_worker) as pool:
        pool.map(_noop, range(4 * n_workers))      # returns once every worker has finished its initializer
        for s in range(args.warmup + args.steps):
            idx = ids[(s * 5) % len(ids)]          # stride 5: the steps walk over the whole scene list
            t, f, done, total = cpu_scene_sample(make_input(idx, args.workload), budget, pool, n_workers, rng)
            if s >= args.warmup:
                spent.append(t)
                fracs.append(f)
                log.append(f"scene {idx}: {done}/{total} regions")
    val = float(np.sum(fracs) / np.sum(spent))     # scenes (fractions of scenes) labelled per second
    desc = (f"each step = one scene of the job's list (stride 5 through it): its scene-level stages in full plus a "
            f"uniform random subset of its GP regions on a {n_workers}-process pool, bounded to ~{budget:.0f} s; the "
            f"fraction of the scene a step covers is time spent / (stages + region time / cost-model share of the "
            f"subset); value = sum of fractions / sum of seconds; [{'; '.join(log[:6])}{' ...' if len(log) > 6 else ''}]")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "scenes/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(spent)) * 1e3, "higher_is_better": True,
        "scaling": args.mode, "vs_baseline": None, "dtype": "f32 (f64 Cholesky/solve), CPU", "data": "synthetic",
        "config": static_config(args, world),
        "scene_fraction_per_step": float(np.mean(fracs)),
        "note": "CPU restatement of the reference (oracle/, gpytorch precision policy); the reference itself needs "
                "gpytorch + torch_scatter, not installable here (DESIGN.md)",
        "cpu_baseline": {"value": val, "unit": "scenes/s", "cores": n_workers, "kind": "port", "sample": desc},
        "e2e": {"value": val, "unit": "scenes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), file=_RESULT_OUT, flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.FIELDS}",
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm)}
        return out


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def stage_rooflines(eng, lib, stream, flush):
    """HBM-bound stages timed alone with CUDA events on the batch left in eng.last."""
    from gapro_b200 import _lib
    L = eng.last
    peak, peak_src = hbm_peak()
    N, S, Bt, D, words = L["N"], L["St"], L["Bt"], L["D"], L["words"]

    def time_it(fn, reps=5):
        ts = []
        for _ in range(reps):
            flush()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts))

    occ_gather = lambda: _lib.check(lib.gapro_occupancy(
        L["xyz"].data_ptr(), L["perm"].data_ptr(), L["seg_off"].data_ptr(), L["spp_off_dev"].data_ptr(),
        L["box_off_dev"].data_ptr(), L["boxes"].data_ptr(), L["ns"], S, Bt, words, 0.005, L["thresh"],
        L["occ_bits"].data_ptr(), L["n_bbs"].data_ptr(), 0, L["excl_cnt"].data_ptr(), L["inter_cnt"].data_ptr(), stream), "occ")
    ows = torch.empty(max(lib.gapro_occupancy_points_workspace_bytes(L["ns"], words), 256), dtype=torch.uint8,
                      device=L["xyz"].device)
    cnt_tab = L["cnt_in"] if L.get("cnt_in") is not None else torch.empty((S, 32 * words), dtype=torch.int32,
                                                                          device=L["xyz"].device)
    occ = lambda: _lib.check(lib.gapro_occupancy_points(
        L["xyz"].data_ptr(), L["spp_gid"].data_ptr(), L["seg_off"].data_ptr(), L["pt_off_dev"].data_ptr(),
        L["spp_off_dev"].data_ptr(), L["box_off_dev"].data_ptr(), L["boxes"].data_ptr(), L["scratch"].data_ptr(), L["ns"], N,
        S, Bt, words, 0.005, L["thresh"], L["occ_bits"].data_ptr(), L["n_bbs"].data_ptr(), cnt_tab.data_ptr(),
        L["excl_cnt"].data_ptr(), L["inter_cnt"].data_ptr(), ows.data_ptr(), ows.numel(), stream), "occ points")
    pool = lambda: _lib.check(lib.gapro_pool_feats(L["feats"].data_ptr(), L["perm"].data_ptr(), L["seg_off"].data_ptr(),
                                                   S, D, L["feats_spp"].data_ptr(), stream), "pool")
    bc = lambda: _lib.check(lib.gapro_broadcast_labels(L["spp_gid"].data_ptr(), N, L["packed_spp"].data_ptr(),
                                                       L["sem"].data_ptr(), L["inst"].data_ptr(), L["prob"].data_ptr(),
                                                       stream), "bcast")
    # the gather wall: the same number of 24-byte records read at random addresses and nothing else
    gidx = torch.randperm(N, device=L["xyz"].device, dtype=torch.int32)
    sink = torch.zeros(1, dtype=torch.float64, device=L["xyz"].device)
    gather = lambda: _lib.check(lib.gapro_gather_peak(gidx.data_ptr(), L["xyz"].data_ptr(), N, sink.data_ptr(), stream),
                                "gather")
    g_ms = time_it(gather)
    g_gbs = N * 28 / (g_ms * 1e-3) / 1e9
    out = {}
    for name, fn, nbytes in (
        ("containment+occupancy (A+A')", occ_gather, N * (24 + 4) + 48 * Bt + 4 * S * words + 4 * S),
        ("containment+occupancy, point-order alternative (GAPRO_OCCUPANCY=points, not the default path)", occ,
         N * (24 + 4) + 48 * Bt + 4 * S * words + 4 * S),
        ("feature pooling (B)", pool, N * (4 * D + 4) + 4 * S * D),
        ("broadcast (E)", bc, N * 4 + 16 * S + N * 12),
    ):
        ms = time_it(fn)
        gbs = nbytes / (ms * 1e-3) / 1e9
        out[name] = {"ms": ms, "algorithmic_bytes": int(nbytes), "achieved": gbs, "peak": peak, "unit": "GB/s",
                     "frac": gbs / peak, "peak_source": peak_src}
    for name in ("containment+occupancy (A+A')", "feature pooling (B)"):
        # both read N random 24-byte records + a coalesced index (the points grouped by superpoint): the random-gather
        # microbenchmark is shown next to the copy peak, which stays the roofline (`frac`)
        out[name]["random_gather_peak"] = g_gbs
        out[name]["frac_of_random_gather_peak"] = out[name]["achieved"] / g_gbs
    out["random 24-byte gather microbenchmark (gapro_gather_peak)"] = {
        "ms": g_ms, "algorithmic_bytes": int(N * 28), "achieved": g_gbs, "peak": peak, "unit": "GB/s",
        "frac": g_gbs / peak, "peak_source": peak_src}
    return out


_RESULT_OUT = sys.stdout

PHASE_ID = {"A": 2, "B": 3, "GA": 5, "GT": 6, "GC": 8, "GL": 9, "Y": 11, "GK": 12}


def morton_order(scene):
    """The same scene with its points re-ordered along a Morton (Z-order) curve of xyz - the locality a real scan's
    mesh-vertex order has and the fully shuffled synthetic points lack.  Input plumbing only (torch index ops)."""
    from gapro_b200.engine import SceneInputs
    xyz = scene.coords_float
    lo, hi = xyz.min(0)[0], xyz.max(0)[0]
    q = ((xyz - lo) / (hi - lo).clamp_min(1e-9) * 1023.0).long().clamp_(0, 1023)
    code = torch.zeros(xyz.shape[0], dtype=torch.int64, device=xyz.device)
    for b in range(10):
        for d in range(3):
            code |= ((q[:, d] >> b) & 1) << (3 * b + d)
    order = torch.argsort(code)
    return SceneInputs(xyz[order].contiguous(), scene.mask_feats[order].contiguous(), scene.spp[order].contiguous(),
                       scene.instance_cls, scene.instance_box, scene.instance_box_volume, scene.wall_box,
                       scene.wall_box_volume, noise_seed=scene.noise_seed)


def ncu_traffic(kernel_regex, args):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
    `ncu --set full` capture (profiles/r02_traffic.json, written by profiles/summarize.py); null when there is no
    capture of this workload."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        path = os.path.join(ROOT, "profiles", name)
        try:
            with open(path) as f:
                t = json.load(f)
        except OSError:
            continue
        if not str(t.get("workload", "")).startswith(args.workload):
            continue
        for k, v in t["kernels"].items():
            if kernel_regex in k:
                return v["dram_read_bytes"] + v["dram_write_bytes"], f"profiles/{name}: {k} ({t.get('command', 'ncu --set full')})"
    return None, "no ncu capture of this workload committed"


OUTPUT_FIELDS = ("sem", "inst", "prob", "mu", "var")


def dump_outputs(outs, out_dir, max_bytes=64 << 20):
    """Write what one step of the timed path returned, so that two builds can be compared output for output: for
    each field of the per-scene (sem, inst, prob, mu, var) tuples, the scenes' arrays concatenated in job order as
    float32 <out_dir>/<field>.npy (the integer labels are small, so float32 holds them exactly).  A field longer than
    its share of max_bytes is cut to a uniform sample of positions drawn with a fixed seed, kept in position order:
    the same positions on every run with the same arguments, and the same for sem / inst / prob."""
    os.makedirs(out_dir, exist_ok=True)
    cap = (max_bytes // len(OUTPUT_FIELDS) - 128) // 4       # float32 elements per file (128: the .npy header)
    for i, name in enumerate(OUTPUT_FIELDS):
        a = torch.cat([o[i].reshape(-1) for o in outs]).float().cpu().numpy()
        if len(a) > cap:
            a = a[np.sort(np.random.default_rng(0).choice(len(a), cap, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_gpu(args):
    rank, world, local = dist_env()
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from gapro_b200 import _lib, sharding
    from gapro_b200.engine import SceneInputs, get_engine
    from gapro_b200.gen_ps import to_scene_inputs
    lib = _lib.load()
    eng = get_engine(dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    kw = dict(thresh_spp_occu=0.999, training_iter=50)      # gen_ps.py:106-110
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    flush = lambda: flush_buf.zero_()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def gather_floats(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            out = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(out, t)
            return [float(o.item()) for o in out]
        return [float(x)]

    # ---- the job: a fixed scene list, sharded by estimated cost (the CLI's path: gapro_b200/gen_ps.py) -------
    ids = scene_ids(args, world)
    if world > 1:
        # cost pass: every rank runs the cheap stages (U, F, A, A', P) on a round-robin share, one gather of the
        # estimates, LPT on every rank (deterministic)
        mine = ids[rank::world]
        est = {}
        for i0 in range(0, len(mine), args.scenes):
            part = mine[i0:i0 + args.scenes]
            st = eng.run([to_scene_inputs(make_input(i, args.workload), dev) for i in part], plan_only=True, **kw)
            for k, i in enumerate(part):
                est[i] = sharding.scene_cost(st["sum_m3"][k], st["n_points"][k], st["n_regions"][k], st["sum_m2"][k])
        merged = {}
        for d in sharding.gather_records([est], world):
            merged.update(d)
        costs = [merged[i] for i in ids]
        assign = sharding.lpt_assignment(costs, world)
        est_balance = sharding.balance_stats(costs, assign)["max_over_mean"]
        my_ids = [ids[k] for k in assign[rank]]
    else:
        my_ids, est_balance = ids, 1.0
    inps = [make_input(i, args.workload) for i in my_ids]
    scenes = [to_scene_inputs(inp, dev, noise_seed=1000 + i) for i, inp in zip(my_ids, inps)]
    passes = [scenes[i:i + args.scenes] for i in range(0, len(scenes), args.scenes)]

    def step():
        outs = []
        for p in passes:
            flush()
            outs.extend(eng.run(p, **kw))
        return outs

    launches_per_step = 0
    for _ in range(args.warmup):
        step()
    # launches of one step (counted by the library for the GP stage, by the host mirror for the rest)
    for p in passes:
        eng.run(p, **kw)
        launches_per_step += eng.last_stats["launches"]
    stats = [dict(eng.last_stats)]

    # ---- device-resident timing (value) ---------------------------------------------------------
    sampler = ClockSampler(local)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        outs = step()
    e_work = torch.cuda.Event(enable_timing=True)
    e_work.record()
    # the one collective of the job: gather of label metadata (per-rank semantic histogram)
    if outs:
        sem_all = torch.cat([o[0] for o in outs]).long()
        hist = torch.bincount(torch.where(sem_all < 0, 19, sem_all), minlength=20)
    else:
        hist = torch.zeros(20, dtype=torch.long, device=dev)
    if world > 1:
        gathered = [torch.empty_like(hist) for _ in range(world)]
        dist.all_gather(gathered, hist)
        hist = torch.stack(gathered).sum(0)
    e1.record()
    barrier()
    rank_ms = gather_floats(e0.elapsed_time(e_work) / args.steps)     # every rank's own work per step
    ms_total = max(gather_floats(e0.elapsed_time(e1)))
    clocks = sampler.stop()
    ms_step = ms_total / args.steps
    value = len(ids) / (ms_step * 1e-3)
    if args.dump_outputs:
        dump_outputs(outs, args.dump_outputs)

    # ---- end to end: pinned host inputs -> device -> hot path -> host ----------------------------
    pinned, h2d = [], 0
    for inp in inps:
        d = {}
        for k, dt in (("xyz", torch.float64), ("mask_feats", torch.float32), ("spp", torch.int64),
                      ("instance_cls", torch.int64), ("instance_box", torch.float32),
                      ("instance_box_volume", torch.float32), ("wall_box", torch.float32), ("wall_volume", torch.float32)):
            t = torch.from_numpy(np.ascontiguousarray(inp[k])).to(dt).pin_memory()
            d[k] = t
            h2d += t.numel() * t.element_size()
        pinned.append(d)

    def e2e_step():
        host = []
        for i0 in range(0, len(pinned), args.scenes):
            flush()
            sc = []
            for k, d in enumerate(pinned[i0:i0 + args.scenes]):
                g = {kk: v.to(dev, non_blocking=True) for kk, v in d.items()}
                sc.append(SceneInputs(g["xyz"], g["mask_feats"], g["spp"], g["instance_cls"], g["instance_box"],
                                      g["instance_box_volume"], g["wall_box"], g["wall_volume"],
                                      noise_seed=1000 + my_ids[i0 + k]))
            res = eng.run(sc, **kw)
            host.extend([t.to("cpu", non_blocking=True) for t in r] for r in res)
        return host

    host = e2e_step()
    torch.cuda.synchronize(dev)
    d2h = sum(t.numel() * t.element_size() for r in host for t in r)
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    barrier()
    e0.record()
    t_wall = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    e1.record()
    barrier()
    t_wall = time.perf_counter() - t_wall
    ms_e2e = max(gather_floats(max(e0.elapsed_time(e1), t_wall * 1e3))) / e2e_steps
    e2e_val = len(ids) / (ms_e2e * 1e-3)
    h2d_all = sum(gather_floats(float(h2d)))
    d2h_all = sum(gather_floats(float(d2h)))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (profiled pass, outside the timed regions) ---------------
    import ctypes
    lib.gapro_gp_set_profiling(1)
    flush()
    eng.run(passes[0], keep=True, **kw)
    st0 = dict(eng.last_stats)
    n_slots = 17
    ms = (ctypes.c_double * n_slots)()
    fa = (ctypes.c_double * n_slots)()
    fe = (ctypes.c_double * n_slots)()
    _lib.check(lib.gapro_gp_get_profile(ms, fa, fe, n_slots), "gapro_gp_get_profile")
    lib.gapro_gp_set_profiling(0)
    names = lib.gapro_gp_phase_names().decode().split(",")
    phases = {n: {"ms": ms[i], "alg_gflop": fa[i] / 1e9, "exe_gflop": fe[i] / 1e9} for i, n in enumerate(names)}
    gp_ms = sum(ms)
    gemm_names = ["A", "B", "GA", "GT", "GC", "GL", "SP", "Y", "GK"]
    top = max(gemm_names, key=lambda n: phases[n]["ms"])
    scratch = torch.zeros(8, dtype=torch.float64, device=dev)
    peak_dmma = ctypes.c_double()
    peak_dfma = ctypes.c_double()
    _lib.check(lib.gapro_fp64_peak(1, 20000, ctypes.byref(peak_dmma), scratch.data_ptr(), stream), "fp64 peak")
    _lib.check(lib.gapro_fp64_peak(0, 20000, ctypes.byref(peak_dfma), scratch.data_ptr(), stream), "fp64 peak")
    peak = max(peak_dmma.value, peak_dfma.value)
    iters = 50
    ach = phases[top]["alg_gflop"] / 1e3 / max(phases[top]["ms"] * 1e-3, 1e-9)
    fam_ms = sum(phases[n]["ms"] for n in gemm_names)
    fam_alg = sum(phases[n]["alg_gflop"] for n in gemm_names) / 1e3
    fam_exe = sum(phases[n]["exe_gflop"] for n in gemm_names) / 1e3
    roofline = {
        "bound": "tensor", "kernel": f"k_gemm<{top}> (FP64 DMMA tile kernel)", "achieved": ach, "peak": peak,
        "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
        "peak_source": "in-repo FP64 microbenchmark gapro_fp64_peak on this GPU (DMMA %.1f / DFMA %.1f TFLOP/s); "
                       "MEASURED_PEAKS.json has no FP64 figure; cross-check: B200 FP64 datasheet figure 37-40 TFLOP/s "
                       "(SURVEY.md section 7), i.e. measured / spec = %.2f-%.2f"
                       % (peak_dmma.value, peak_dfma.value, peak / 40.0, peak / 37.0),
        "avg_launch_ms": phases[top]["ms"] / iters,
        "profiled_pass": "first pass of rank 0 (%d scenes, sum M^3 = %.3g), phases timed on one stream"
                         % (len(passes[0]), st0["sum_m3"]),
        "gemm_family": {"ms": fam_ms, "share_of_gp_stage": fam_ms / max(gp_ms, 1e-9),
                        "achieved_alg": fam_alg / max(fam_ms * 1e-3, 1e-9), "achieved_issued": fam_exe / max(fam_ms * 1e-3, 1e-9),
                        "frac_alg": fam_alg / max(fam_ms * 1e-3, 1e-9) / peak,
                        "frac_issued": fam_exe / max(fam_ms * 1e-3, 1e-9) / peak},
        "gp_stage_ms": gp_ms, "phases_ms": {n: round(phases[n]["ms"], 3) for n in names},
    }
    roofline["traffic"], roofline["traffic_source"] = ncu_traffic(f"k_gemm<{PHASE_ID.get(top, -1)}>", args)
    stages = stage_rooflines(eng, lib, stream, flush)
    # the same kernels on a batch large enough to amortise launch latency (the pass's scenes, 8 times over)
    eng.run(passes[0] * 8, stages_only=True, **kw)
    stages_large = stage_rooflines(eng, lib, stream, flush)
    for v in stages_large.values():
        v["points"] = eng.last["N"]
    # ... and on the same points in a spatially coherent order (Morton curve), the order of a real scan's vertices
    eng.run([morton_order(sc) for sc in passes[0]] * 8, stages_only=True, **kw)
    stages_morton = stage_rooflines(eng, lib, stream, flush)
    for v in stages_morton.values():
        v["points"] = eng.last["N"]
    eng.last = None

    # ---- single-scene latency through the reference's per-scene call (BASELINE configs[1]) ---------
    latency = None
    if world == 1 and not args.no_latency:
        from gapro_b200.gen_ps_utils import gen_pseudo_label_gaussian_process
        sc = to_scene_inputs(make_input(0, "c1"), dev, noise_seed=1)
        ts = []
        for r in range(4):
            flush()
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            out = gen_pseudo_label_gaussian_process(sc.coords_float, sc.mask_feats, sc.spp, sc.instance_cls,
                                                    sc.instance_box, sc.instance_box_volume, sc.wall_box,
                                                    sc.wall_box_volume, instance_classes=18, dataset_name="scannetv2",
                                                    ground_h=0.1, training_iter=50, thresh_spp_occu=0.999, noise_seed=1)
            torch.cuda.synchronize(dev)
            ts.append((time.perf_counter() - t0) * 1e3)
        latency = {"workload": WORKLOADS["c1"] + ", ONE scene through gen_pseudo_label_gaussian_process "
                   "(gen_ps_utils.py:293), device-resident inputs, wall clock with a synchronize on both sides",
                   "ms": float(np.median(ts[1:])), "first_call_ms": ts[0], "gp_regions": eng.last_stats["n_regions"],
                   "launches": eng.last_stats["launches"]}

    # ---- CPU baseline (bounded sample) -------------------------------------------------------------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        # fresh interpreter with the GPUs hidden: this process holds a CUDA context and must not fork workers
        env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
        try:
            # two scenes of the list (a heavy and a typical one), ~15 s of CPU work each
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2",
                                "--cpu-budget", "15",
                                "--warmup", "0", "--workload", args.workload, "--scenes", str(args.scenes),
                                "--mode", args.mode, "--total-scenes", str(args.total_scenes)],
                               env=env, capture_output=True, text=True, timeout=300)
            cpu = json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
        except Exception as e:      # reported, never fatal for the GPU line
            cpu = {"value": None, "unit": "scenes/s", "cores": len(os.sched_getaffinity(0)), "kind": "port",
                   "sample": "CPU baseline run failed: %r" % (e,)}

    mean_ms = sum(rank_ms) / len(rank_ms)
    line = {
        "metric": METRIC, "value": value, "unit": "scenes/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.mode,
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": static_config(args, world),
        "workload_stats": {"scenes_this_rank": len(my_ids), "passes_per_step_this_rank": len(passes),
                           "label_histogram_points": int(hist.sum().item()),
                           "first_pass": {"points": st0["n_points"], "superpoints": st0["n_spp"],
                                          "gp_regions": st0["n_regions"], "sum_M": st0["sum_m"], "sum_M3": st0["sum_m3"]}},
        "balance": {"rank_ms_per_step": [round(x, 2) for x in rank_ms], "max_over_mean": max(rank_ms) / mean_ms,
                    "estimated_max_over_mean": est_balance},
        "e2e": {"value": e2e_val, "unit": "scenes/s", "h2d_bytes_per_step": int(h2d_all), "d2h_bytes_per_step": int(d2h_all),
                "ms_per_step": ms_e2e, "steps": e2e_steps},
        "gpu_launches": int(launches_per_step * args.steps),
        "clocks": clocks, "roofline": roofline, "stage_rooflines": stages, "stage_rooflines_large_batch": stages_large,
        "stage_rooflines_large_batch_morton_order": stages_morton,
        "latency": latency, "cpu_baseline": cpu,
    }
    print(json.dumps(line), file=_RESULT_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="strong", choices=["strong", "weak"],
                    help="strong: a fixed list of --total-scenes scenes sharded over the GPUs; weak: --scenes per GPU")
    ap.add_argument("--total-scenes", type=int, default=48,
                    help="scenes of the job (strong mode); 48 keeps the LPT assignment within 1 % of balance up to 8 GPUs "
                         "(32: the heaviest scene alone exceeds an eighth of the job)")
    ap.add_argument("--scenes", type=int, default=16,
                    help="scenes per GPU pass (and per GPU per step in weak mode); measured on the 48-scene job: 6.49 / 6.72 / "
                         "6.73 / 6.71 scenes/s with passes of 8 / 16 / 24 / 48 scenes")
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--e2e-steps", type=int, default=3, help="steps of the end-to-end timing (at most --steps)")
    ap.add_argument("--cpu-budget", type=float, default=None, help="seconds of CPU work per step of the CPU arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's outputs to DIR/<sem|inst|prob|mu|var>.npy (float32, "
                         "64 MB at most: longer fields are a fixed seeded sample); single-process GPU arm only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or dist_env()[1] > 1):
        ap.error("--dump-outputs needs the GPU arm in a single process")
    # stdout carries exactly ONE line (the JSON); whatever libraries print there (NCCL prints its version banner
    # to stdout at communicator creation) goes to stderr instead
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        os.environ["CUDA_VISIBLE_DEVICES"] = ""       # CPU arm: keep forked workers away from CUDA
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback "
                             "(use --impl reference for the CPU arm)")
        run_gpu(args)


if __name__ == "__main__":
    main()
