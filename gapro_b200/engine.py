"""Batch driver of the CUDA hot path: a concatenation of scenes goes through
densify -> floor slab -> containment/occupancy -> feature pooling -> (host) pair state
machine -> index compaction -> batched GP regions -> per-superpoint resolution ->
broadcast, all through the C ABI of include/gapro_b200.h.

torch is used for device memory, the current stream and host<->device copies only.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib, plan

MARGIN = 0.005      # /root/reference/gapro/gen_ps_utils.py:350


@dataclass
class SceneInputs:
    """Exactly what /root/reference/gapro/gen_ps.py:91-111 passes for one scene (device tensors)."""
    coords_float: torch.Tensor          # (N,3) float64
    mask_feats: torch.Tensor            # (N,D) float32
    spp: torch.Tensor                   # (N,) int64 raw superpoint ids
    instance_cls: torch.Tensor          # (K,) int64
    instance_box: torch.Tensor          # (K,6) float32
    instance_box_volume: torch.Tensor   # (K,) float32
    wall_box: object = None             # (W,6) float32 tensor or [] (gen_ps.py:87-89)
    wall_box_volume: object = None
    noise_seed: Optional[int] = None    # seeds this scene's GP init noise (None: torch device RNG)


@dataclass
class BatchDebug:
    spp_off: np.ndarray = None
    box_off: np.ndarray = None
    boxes: np.ndarray = None
    boxes_vol: np.ndarray = None
    occ_bits: torch.Tensor = None
    n_bbs: torch.Tensor = None
    cnt_in: torch.Tensor = None
    seg_off: torch.Tensor = None
    spp_gid: torch.Tensor = None
    feats_spp: torch.Tensor = None
    excl_cnt: np.ndarray = None
    inter_cnt: np.ndarray = None
    events: list = field(default_factory=list)       # per scene: list of (kind, b1, b2)
    regions: list = field(default_factory=list)      # per GP region: dict(scene, b1, b2, train_idx, n_b1, test_idx, ...)
    gp_launches: int = 0
    n_launches: int = 0
    stats: dict = field(default_factory=dict)


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _len(x):
    return 0 if x is None else len(x)


class GaproEngine:
    """Holds the library handle and reusable device workspaces for one GPU."""

    def __init__(self, device=None, gp_workspace_bytes: Optional[int] = None):
        if not torch.cuda.is_available():
            raise _lib.GaproError("gapro_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.gp_workspace_cap = gp_workspace_bytes
        self._ws = {}
        # "gather" (default): one warp per superpoint reads its points through the sort permutation; "points": A + A'
        # stream the points in input order and count with integer reductions (csrc/occupancy_points.cu) - bit-identical
        # results, measured slower on B200 (90 vs 45 us on the bench batch, 394 vs 251 us on 9.5M points), kept as an
        # alternative and covered by the parity suite
        import os
        self.occupancy_path = os.environ.get("GAPRO_OCCUPANCY", "gather")
        if self.occupancy_path not in ("points", "gather"):
            raise ValueError("GAPRO_OCCUPANCY must be 'points' or 'gather'")

    # ------------------------------------------------------------------ helpers
    def _workspace(self, key: str, nbytes: int) -> torch.Tensor:
        buf = self._ws.get(key)
        if buf is None or buf.numel() < nbytes:
            # drop EVERY reference to the old buffer before growing: old + new do not fit side by side
            # when the GP workspace is most of the HBM
            buf = None
            self._ws[key] = None
            try:
                buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=self.device)
            except torch.OutOfMemoryError:
                torch.cuda.empty_cache()
                buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=self.device)
            self._ws[key] = buf
        return buf

    def _to_host(self, tensors):
        """Device -> host for the few KB the host state machine needs: async copies into persistent pinned buffers,
        ONE synchronisation for all of them (a plain `.cpu()` per tensor is a blocking copy each)."""
        out = []
        for i, t in enumerate(tensors):
            key = ("host", i, t.dtype)
            buf = self._ws.get(key)
            if buf is None or buf.numel() < t.numel():
                buf = torch.empty(max(t.numel(), 1), dtype=t.dtype).pin_memory()
                self._ws[key] = buf
            view = buf[:t.numel()].view(t.shape)
            view.copy_(t, non_blocking=True)
            out.append(view)
        torch.cuda.current_stream(self.device).synchronize()
        return [v.numpy().copy() for v in out]

    def _dev(self, arr: np.ndarray) -> torch.Tensor:
        return torch.from_numpy(np.ascontiguousarray(arr)).to(self.device, non_blocking=False)

    # ------------------------------------------------------------------ main entry
    def run(self, scenes: Sequence[SceneInputs], instance_classes=18, ground_h=0.1, training_iter=50,
            thresh_spp_occu=0.8, jitter_zz=1e-4, jitter_xx=1e-4, lr=0.1, debug: bool = False,
            want_cnt_in: bool = False, keep: bool = False, stages_only: bool = False, on_error: str = "raise",
            plan_only: bool = False):
        """Returns a list of (sem[N] i32, inst[N] i32, prob[N] f32, mu[S] f32, var[S] f32) device
        tensors, one tuple per scene — the return of gen_pseudo_label_gaussian_process
        (/root/reference/gapro/gen_ps_utils.py:482) — plus a BatchDebug when debug=True."""
        lib, dev = self.lib, self.device
        stream = torch.cuda.current_stream(dev).cuda_stream
        ns = len(scenes)
        if ns == 0:
            return ([], BatchDebug()) if debug else []
        n_launch = 0

        # ---- concatenate scene inputs (device plumbing) -----------------------------------
        n_pts = [int(s.coords_float.shape[0]) for s in scenes]
        pt_off = np.zeros(ns + 1, dtype=np.int64)
        pt_off[1:] = np.cumsum(n_pts)
        N = int(pt_off[-1])
        D = int(scenes[0].mask_feats.shape[1])
        for s in scenes:
            if int(s.mask_feats.shape[1]) != D:
                raise ValueError("all scenes of a batch must share the feature dimension")
        cat = (lambda ts: ts[0].contiguous()) if ns == 1 else (lambda ts: torch.cat(ts, 0))
        xyz = cat([s.coords_float.to(dev, torch.float64) for s in scenes])
        feats = cat([s.mask_feats.to(dev).float() for s in scenes])
        spp_raw = cat([s.spp.to(dev, torch.int64).reshape(-1) for s in scenes])

        n_fg = np.array([_len(s.instance_box) for s in scenes], dtype=np.int32)
        n_wall = np.array([_len(s.wall_box) for s in scenes], dtype=np.int32)
        n_box = n_fg + n_wall + 1
        box_off = np.zeros(ns + 1, dtype=np.int32)
        box_off[1:] = np.cumsum(n_box)
        Bt = int(box_off[-1])
        words = 1
        while 32 * words < int(n_box.max()):
            words *= 2
        if words > 8:
            raise ValueError("more than 256 boxes in one scene")
        boxes = torch.zeros((Bt, 6), dtype=torch.float64, device=dev)
        boxes_vol = torch.zeros((Bt,), dtype=torch.float64, device=dev)
        boxes_cls = torch.full((Bt,), int(instance_classes), dtype=torch.int64, device=dev)
        for i, s in enumerate(scenes):
            b0, k = int(box_off[i]), int(n_fg[i])
            if k:
                # float32 boxes widened to float64 (cat promotion, gen_ps_utils.py:329,338)
                boxes[b0:b0 + k] = s.instance_box.to(dev).float().double()
                boxes_vol[b0:b0 + k] = s.instance_box_volume.to(dev).float().double()
                boxes_cls[b0:b0 + k] = s.instance_cls.to(dev, torch.int64)
            w = int(n_wall[i])
            if w:
                boxes[b0 + k:b0 + k + w] = s.wall_box.to(dev).float().double()
                boxes_vol[b0 + k:b0 + k + w] = s.wall_box_volume.to(dev).float().double()
        pt_off_dev = self._dev(pt_off)
        box_off_dev = self._dev(box_off)
        n_fg_dev = self._dev(n_fg)

        # ---- U: densify --------------------------------------------------------------------
        spp_gid = torch.empty(N, dtype=torch.int32, device=dev)
        perm = torch.empty(N, dtype=torch.int32, device=dev)
        seg_off = torch.empty(N + 1, dtype=torch.int32, device=dev)
        spp_off = np.zeros(ns + 1, dtype=np.int32)
        ws = self._workspace("densify", lib.gapro_densify_workspace_bytes(N, ns))
        _lib.check(lib.gapro_densify_spp(spp_raw.data_ptr(), pt_off.ctypes.data, ns, spp_gid.data_ptr(), perm.data_ptr(),
                                         seg_off.data_ptr(), spp_off.ctypes.data, ws.data_ptr(), ws.numel(), stream),
                   "gapro_densify_spp")
        n_launch += 9
        St = int(spp_off[-1])
        spp_off_dev = self._dev(spp_off)

        # ---- F: floor slab -----------------------------------------------------------------
        scratch = torch.empty(ns * 6, dtype=torch.int64, device=dev)
        _lib.check(lib.gapro_floor_boxes(xyz.data_ptr(), pt_off_dev.data_ptr(), box_off_dev.data_ptr(), ns, N,
                                         float(ground_h), boxes.data_ptr(), boxes_vol.data_ptr(), scratch.data_ptr(),
                                         stream), "gapro_floor_boxes")
        n_launch += 3

        # ---- A + A': containment / occupancy ----------------------------------------------
        occ_bits = torch.empty((St, words), dtype=torch.int32, device=dev)
        n_bbs = torch.empty(St, dtype=torch.int32, device=dev)
        excl_cnt = torch.empty(Bt, dtype=torch.int32, device=dev)
        stride = 32 * words
        inter_cnt = torch.empty((ns, stride, stride), dtype=torch.int32, device=dev)
        thresh32 = float(np.float32(thresh_spp_occu))
        if self.occupancy_path == "points":
            # point order: stream xyz + dense ids, per-scene grid of box masks, integer counts in L2 (opt-in)
            cnt_in = torch.empty((St, stride), dtype=torch.int32, device=dev)
            ows = self._workspace("occ", lib.gapro_occupancy_points_workspace_bytes(ns, words))
            _lib.check(lib.gapro_occupancy_points(xyz.data_ptr(), spp_gid.data_ptr(), seg_off.data_ptr(),
                                                  pt_off_dev.data_ptr(), spp_off_dev.data_ptr(), box_off_dev.data_ptr(),
                                                  boxes.data_ptr(), scratch.data_ptr(), ns, N, St, Bt, words, MARGIN,
                                                  thresh32, occ_bits.data_ptr(), n_bbs.data_ptr(), cnt_in.data_ptr(),
                                                  excl_cnt.data_ptr(), inter_cnt.data_ptr(), ows.data_ptr(), ows.numel(),
                                                  stream), "gapro_occupancy_points")
            n_launch += 3
        else:
            # by superpoint: gather through the sort permutation
            cnt_in = torch.empty((St, stride), dtype=torch.int32, device=dev) if want_cnt_in else None
            _lib.check(lib.gapro_occupancy(xyz.data_ptr(), perm.data_ptr(), seg_off.data_ptr(), spp_off_dev.data_ptr(),
                                           box_off_dev.data_ptr(), boxes.data_ptr(), ns, St, Bt, words, MARGIN,
                                           thresh32, occ_bits.data_ptr(), n_bbs.data_ptr(),
                                           _ptr(cnt_in), excl_cnt.data_ptr(), inter_cnt.data_ptr(), stream),
                       "gapro_occupancy")
            n_launch += 1

        # ---- B: feature pooling ------------------------------------------------------------
        feats_spp = torch.empty((St, D), dtype=torch.float32, device=dev)
        _lib.check(lib.gapro_pool_feats(feats.data_ptr(), perm.data_ptr(), seg_off.data_ptr(), St, D,
                                        feats_spp.data_ptr(), stream), "gapro_pool_feats")
        n_launch += 1

        if stages_only:      # benchmarking hook: stop after the memory-bound stages, keep their buffers
            self.last = dict(xyz=xyz, feats=feats, perm=perm, seg_off=seg_off, spp_gid=spp_gid, spp_off_dev=spp_off_dev,
                             box_off_dev=box_off_dev, boxes=boxes, occ_bits=occ_bits, n_bbs=n_bbs, excl_cnt=excl_cnt,
                             inter_cnt=inter_cnt, feats_spp=feats_spp, pt_off_dev=pt_off_dev, scratch=scratch,
                             cnt_in=cnt_in,
                             packed_spp=torch.zeros((St, 4), dtype=torch.int32, device=dev),
                             sem=torch.empty(N, dtype=torch.int32, device=dev),
                             inst=torch.empty(N, dtype=torch.int32, device=dev),
                             prob=torch.empty(N, dtype=torch.float32, device=dev), ns=ns, St=St, Bt=Bt, N=N, D=D,
                             words=words, thresh=float(np.float32(thresh_spp_occu)))
            return None

        # ---- P: pair state machine on the host --------------------------------------------
        boxes_h, excl_h, inter_h = self._to_host([boxes, excl_cnt, inter_cnt])
        ev = plan.enumerate_events(boxes_h, excl_h, inter_h, box_off, stride)
        pl = plan.plan_lists(ev, box_off, excl_h, inter_h)
        ev_off, ev_scene, ev_kind, ev_b1, ev_b2 = ev["ev_off"], ev["ev_scene"], ev["ev_kind"], ev["ev_b1"], ev["ev_b2"]
        n_ev, R, gp_ev, inter_len = pl["n_events"], pl["n_regions"], pl["gp_ev"], pl["inter_len"]
        ev_list_off, n_inter_total, n_test_total = pl["ev_list_off"], pl["n_inter_total"], pl["n_test_total"]
        n_train_total, test_off, train_off, m1, m2 = pl["n_train_total"], pl["test_off"], pl["train_off"], pl["m1"], pl["m2"]
        if plan_only:
            # cost estimate for load balancing (sharding.py): what the cheap stages A / A' / P say about the GP work
            # of every scene - sum of M^3 over its regions (the GP stage is ~385 * M^3 flops per region)
            m = (m1 + m2).astype(np.float64)
            rs = pl["region_scene"]
            return dict(sum_m3=np.bincount(rs, weights=m ** 3, minlength=ns)[:ns] if R else np.zeros(ns),
                        sum_m2=np.bincount(rs, weights=m ** 2, minlength=ns)[:ns] if R else np.zeros(ns),
                        n_regions=np.bincount(rs, minlength=ns)[:ns] if R else np.zeros(ns, np.int64),
                        max_m=np.array([m[rs == i].max() if np.any(rs == i) else 0 for i in range(ns)]),
                        n_points=np.array(n_pts), n_spp=np.diff(spp_off).astype(np.int64))
        L_scene, L_b1, L_b2, L_off = pl["list_scene"], pl["list_b1"], pl["list_b2"], pl["list_off"]
        n_lists = len(L_scene)
        lists_idx = torch.empty(max(n_inter_total + n_train_total, 1), dtype=torch.int32, device=dev)
        if n_lists:
            Ls, Lb1, Lb2, Lo = self._dev(L_scene), self._dev(L_b1), self._dev(L_b2), self._dev(L_off)
            _lib.check(lib.gapro_compact_lists(occ_bits.data_ptr(), n_bbs.data_ptr(), spp_off_dev.data_ptr(), words,
                                               Ls.data_ptr(), Lb1.data_ptr(), Lb2.data_ptr(), Lo.data_ptr(), n_lists,
                                               lists_idx.data_ptr(), stream), "gapro_compact_lists")
            n_launch += 1

        # ---- C: GP regions -----------------------------------------------------------------
        gp_prob = torch.empty(max(n_test_total, 1), dtype=torch.float32, device=dev)
        gp_conf = torch.empty_like(gp_prob)
        gp_mu = torch.empty_like(gp_prob)
        gp_var = torch.empty_like(gp_prob)
        gp_label = torch.empty(max(n_test_total, 1), dtype=torch.uint8, device=dev)
        gp_mu64 = torch.empty(max(n_test_total, 1), dtype=torch.float64, device=dev) if debug else None
        gp_var64 = torch.empty(max(n_test_total, 1), dtype=torch.float64, device=dev) if debug else None
        gp_launches = 0
        noise = None
        failed_scenes = {}
        gp_retries = np.zeros(0, np.int64)
        if R:
            noise = self._make_noise(scenes, ev_scene[gp_ev], m1 + m2, n_train_total)
            n_b1 = m1.astype(np.int32)
            status = torch.zeros(R, dtype=torch.int32, device=dev)
            full = lib.gapro_gp_workspace_bytes(R, train_off.ctypes.data, test_off.ctypes.data, D)
            need = lib.gapro_gp_min_workspace_bytes(R, train_off.ctypes.data, test_off.ctypes.data, D)
            cap = self.gp_workspace_cap
            if cap is None:
                free, _ = torch.cuda.mem_get_info(dev)
                held = self._ws.get("gp")
                held_bytes = held.numel() if held is not None else 0
                del held            # no alias may survive into _workspace(): growing frees the old buffer first
                cap = int(0.7 * (free + held_bytes))
            nbytes = max(min(full, cap), need)
            ws = self._workspace("gp", nbytes)
            train_idx_ptr = lists_idx.data_ptr() + 4 * n_inter_total
            _lib.check(lib.gapro_gp_fit_batch(feats_spp.data_ptr(), D, R, train_off.ctypes.data, n_b1.ctypes.data,
                                              test_off.ctypes.data, train_idx_ptr, lists_idx.data_ptr(),
                                              noise.data_ptr(), int(training_iter), float(lr), float(jitter_zz),
                                              float(jitter_xx), gp_prob.data_ptr(), gp_conf.data_ptr(),
                                              gp_label.data_ptr(), gp_mu.data_ptr(), gp_var.data_ptr(), _ptr(gp_mu64),
                                              _ptr(gp_var64), status.data_ptr(), ws.data_ptr(), ws.numel(), stream),
                       "gapro_gp_fit_batch")
            gp_launches = int(lib.gapro_gp_last_launch_count())
            n_launch += gp_launches
            st = status.cpu().numpy()
            gp_retries = (st >> _lib.GP_RETRY_SHIFT) & 0xffff
            # a failed region fails ITS scene only (the reference would have died on that scene, gen_ps_utils.py:434-437)
            for r in np.flatnonzero(st & (_lib.GP_NOT_PSD | _lib.GP_NAN)):
                sc = int(ev_scene[gp_ev[r]])
                what = ("NotPSDError: K_ZZ is not positive definite after the jitter retries of psd_safe_cholesky"
                        if st[r] & _lib.GP_NOT_PSD else "NanError: non-finite GP posterior")
                failed_scenes.setdefault(sc, f"GP region {int(r)} (boxes {int(ev_b1[gp_ev[r]])}, "
                                             f"{int(ev_b2[gp_ev[r]])}, M={int(m1[r] + m2[r])}): {what}")

        # ---- S0 + M + D + labels, then E ------------------------------------------------------
        ev_gp_off = pl["ev_gp_off"]
        sem_spp = torch.empty(St, dtype=torch.int32, device=dev)
        inst_spp = torch.empty(St, dtype=torch.int32, device=dev)
        prob_spp = torch.empty(St, dtype=torch.float32, device=dev)
        mu_spp = torch.empty(St, dtype=torch.float32, device=dev)
        var_spp = torch.empty(St, dtype=torch.float32, device=dev)
        packed_spp = torch.empty((St, 4), dtype=torch.int32, device=dev)
        d_ev = [self._dev(a) for a in (ev_off, ev_kind.astype(np.int32), ev_b1.astype(np.int32),
                                       ev_b2.astype(np.int32), ev_list_off.astype(np.int32),
                                       inter_len.astype(np.int32), ev_gp_off)]
        if n_ev == 0:
            d_ev = [d_ev[0]] + [torch.zeros(1, dtype=torch.int32, device=dev) for _ in range(6)]
        _lib.check(lib.gapro_resolve_spp(occ_bits.data_ptr(), n_bbs.data_ptr(), words, spp_off_dev.data_ptr(),
                                         box_off_dev.data_ptr(), boxes_vol.data_ptr(), boxes_cls.data_ptr(),
                                         n_fg_dev.data_ptr(), int(instance_classes), ns, *[t.data_ptr() for t in d_ev],
                                         lists_idx.data_ptr(), gp_conf.data_ptr(), gp_label.data_ptr(),
                                         gp_mu.data_ptr(), gp_var.data_ptr(), sem_spp.data_ptr(), inst_spp.data_ptr(),
                                         prob_spp.data_ptr(), mu_spp.data_ptr(), var_spp.data_ptr(),
                                         packed_spp.data_ptr(), stream), "gapro_resolve_spp")
        sem = torch.empty(N, dtype=torch.int32, device=dev)
        inst = torch.empty(N, dtype=torch.int32, device=dev)
        prob = torch.empty(N, dtype=torch.float32, device=dev)
        _lib.check(lib.gapro_broadcast_labels(spp_gid.data_ptr(), N, packed_spp.data_ptr(), sem.data_ptr(),
                                              inst.data_ptr(), prob.data_ptr(), stream), "gapro_broadcast_labels")
        n_launch += 2

        if keep:
            self.last = dict(xyz=xyz, feats=feats, perm=perm, seg_off=seg_off, spp_gid=spp_gid, spp_off_dev=spp_off_dev,
                             box_off_dev=box_off_dev, boxes=boxes, occ_bits=occ_bits, n_bbs=n_bbs, excl_cnt=excl_cnt,
                             inter_cnt=inter_cnt, feats_spp=feats_spp, pt_off_dev=pt_off_dev, scratch=scratch,
                             cnt_in=cnt_in, packed_spp=packed_spp, sem=sem, inst=inst, prob=prob, ns=ns, St=St, Bt=Bt, N=N, D=D,
                             words=words, thresh=float(np.float32(thresh_spp_occu)))
        out = []
        for i in range(ns):
            p0, p1, s0, s1 = int(pt_off[i]), int(pt_off[i + 1]), int(spp_off[i]), int(spp_off[i + 1])
            out.append(None if i in failed_scenes else
                       (sem[p0:p1], inst[p0:p1], prob[p0:p1], mu_spp[s0:s1], var_spp[s0:s1]))
        self.last_errors = failed_scenes
        self.last_stats = dict(gp_cholesky_retries=int(gp_retries.sum()),
                               n_points=N, n_spp=St, n_boxes=Bt, n_events=n_ev, n_regions=R,
                               sum_m=n_train_total, sum_m3=float(((m1 + m2).astype(np.float64) ** 3).sum()) if R else 0.0,
                               launches=n_launch, gp_launches=gp_launches, feat_dim=D,
                               m_list=(m1 + m2).astype(np.int64) if R else np.zeros(0, np.int64),
                               n_list=inter_len[gp_ev] if R else np.zeros(0, np.int64))
        if failed_scenes and on_error == "raise":
            raise _lib.GaproSceneError(failed_scenes, out)
        if not debug:
            return out
        dbg = BatchDebug(spp_off=spp_off, box_off=box_off, boxes=boxes_h, boxes_vol=boxes_vol.cpu().numpy(),
                         occ_bits=occ_bits, n_bbs=n_bbs, cnt_in=cnt_in, seg_off=seg_off, spp_gid=spp_gid,
                         feats_spp=feats_spp, excl_cnt=excl_h, inter_cnt=inter_h, gp_launches=gp_launches,
                         n_launches=n_launch, stats=self.last_stats)
        for i in range(ns):
            e0, e1 = int(ev_off[i]), int(ev_off[i + 1])
            dbg.events.append([(int(ev_kind[e]), int(ev_b1[e]), int(ev_b2[e])) for e in range(e0, e1)])
        li = lists_idx.cpu().numpy()
        if R:
            res = dict(prob=gp_prob.cpu().numpy(), conf=gp_conf.cpu().numpy(), label=gp_label.cpu().numpy(),
                       mu=gp_mu.cpu().numpy(), var=gp_var.cpu().numpy(), mu64=gp_mu64.cpu().numpy(),
                       var64=gp_var64.cpu().numpy())
            nz = noise.cpu().numpy()
            for r, e in enumerate(gp_ev):
                t0, t1, q0, q1 = int(train_off[r]), int(train_off[r + 1]), int(test_off[r]), int(test_off[r + 1])
                s0 = int(spp_off[ev_scene[e]])
                dbg.regions.append(dict(scene=int(ev_scene[e]), b1=int(ev_b1[e]), b2=int(ev_b2[e]), n_b1=int(m1[r]),
                                        train_idx=li[n_inter_total + t0:n_inter_total + t1] - s0,
                                        test_idx=li[q0:q1] - s0, noise=nz[t0:t1],
                                        **{k: v[q0:q1] for k, v in res.items()}))
        return out, dbg

    # ------------------------------------------------------------------ heuristic labelers (SURVEY 8f)
    def run_heuristic(self, scenes: Sequence[SceneInputs], rule="volume", spp_align=True, occ_thresh=None,
                      instance_classes=18):
        """Scenes through the heuristic labelers in one pass: per-point containment in the instance boxes, the rule
        for points in several boxes, optional majority vote per superpoint, final labels.  Only the coordinates, the
        superpoints and the instance boxes / classes / volumes of each scene are read (no wall boxes, no floor slab).
        Returns one (sem[N] i32, inst[N] i32) pair of device views per scene."""
        lib, dev = self.lib, self.device
        stream = torch.cuda.current_stream(dev).cuda_stream
        ns = len(scenes)
        if ns == 0:
            return []
        rule_id = {"volume": 0, "dist": 1, "none": 2}[rule]
        n_pts = [int(s.coords_float.shape[0]) for s in scenes]
        pt_off = np.zeros(ns + 1, dtype=np.int64)
        pt_off[1:] = np.cumsum(n_pts)
        N = int(pt_off[-1])
        n_box = np.array([int(s.instance_box.shape[0]) for s in scenes], dtype=np.int32)
        box_off = np.zeros(ns + 1, dtype=np.int32)
        box_off[1:] = np.cumsum(n_box)
        words = 1
        while 32 * words < int(n_box.max()):
            words *= 2
        if words > 8:
            raise ValueError("more than 256 boxes in one scene")
        cat = (lambda ts: ts[0].contiguous()) if ns == 1 else (lambda ts: torch.cat(ts, 0))
        xyz = cat([s.coords_float.to(dev, torch.float64) for s in scenes])
        spp_raw = cat([s.spp.to(dev, torch.int64).reshape(-1) for s in scenes])
        # the boxes stay float32 (gen_ps.py:80): margins and centres are float32 values in the kernels
        boxes = cat([s.instance_box.to(dev).float().reshape(-1, 6) for s in scenes])
        vol = cat([s.instance_box_volume.to(dev).float().reshape(-1) for s in scenes])
        cls = cat([s.instance_cls.to(dev, torch.int64).reshape(-1) for s in scenes])

        spp_gid = torch.empty(N, dtype=torch.int32, device=dev)
        perm = torch.empty(N, dtype=torch.int32, device=dev)
        seg_off = torch.empty(N + 1, dtype=torch.int32, device=dev)
        spp_off = np.zeros(ns + 1, dtype=np.int32)
        ws = self._workspace("densify", lib.gapro_densify_workspace_bytes(N, ns))
        _lib.check(lib.gapro_densify_spp(spp_raw.data_ptr(), pt_off.ctypes.data, ns, spp_gid.data_ptr(), perm.data_ptr(),
                                         seg_off.data_ptr(), spp_off.ctypes.data, ws.data_ptr(), ws.numel(), stream),
                   "gapro_densify_spp")
        St = int(spp_off[-1])
        offs = self._dev(np.concatenate([box_off, spp_off]))         # one upload for both int32 offset tables
        box_off_dev, spp_off_dev = offs[:ns + 1], offs[ns + 1:]
        pt_off_dev = self._dev(pt_off) if rule_id == 1 or not spp_align else None
        thr = -1.0 if occ_thresh is None else float(np.float32(occ_thresh))
        dist_src = None
        if rule_id == 1:
            # the reference measures the k-th multi-box point from the coordinates of point k (gen_ps_utils.py:516,526)
            dist_src = torch.empty(N, dtype=torch.int32, device=dev)
            mws = self._workspace("multibox", lib.gapro_multibox_workspace_bytes(N))
            _lib.check(lib.gapro_multibox_sources(xyz.data_ptr(), pt_off_dev.data_ptr(), box_off_dev.data_ptr(),
                                                  boxes.data_ptr(), ns, N, dist_src.data_ptr(), mws.data_ptr(),
                                                  mws.numel(), stream), "gapro_multibox_sources")
        inst_spp = torch.empty(St, dtype=torch.int32, device=dev) if spp_align else None
        inst_pt = None if spp_align else torch.empty(N, dtype=torch.int32, device=dev)
        _lib.check(lib.gapro_heuristic_labels(xyz.data_ptr(), perm.data_ptr(), seg_off.data_ptr(), spp_off_dev.data_ptr(),
                                              box_off_dev.data_ptr(), boxes.data_ptr(), vol.data_ptr(), _ptr(dist_src),
                                              ns, St, words, rule_id, 1 if spp_align else 0, thr, _ptr(inst_spp),
                                              _ptr(inst_pt), stream), "gapro_heuristic_labels")
        sem = torch.empty(N, dtype=torch.int32, device=dev)
        inst = torch.empty(N, dtype=torch.int32, device=dev)
        packed = torch.empty((St, 4), dtype=torch.int32, device=dev) if spp_align else None
        _lib.check(lib.gapro_heuristic_finalize(_ptr(inst_spp), _ptr(inst_pt), spp_off_dev.data_ptr(), _ptr(pt_off_dev),
                                                box_off_dev.data_ptr(), cls.data_ptr(), int(instance_classes), ns, St,
                                                N, 1 if spp_align else 0, _ptr(packed), _ptr(None if spp_align else sem),
                                                _ptr(None if spp_align else inst), stream), "gapro_heuristic_finalize")
        if spp_align:
            # per-superpoint records (sem, inst, 1.0, 0) -> points with the 128-bit broadcast of the GP path
            prob = torch.empty(N, dtype=torch.float32, device=dev)
            _lib.check(lib.gapro_broadcast_labels(spp_gid.data_ptr(), N, packed.data_ptr(), sem.data_ptr(),
                                                  inst.data_ptr(), prob.data_ptr(), stream), "gapro_broadcast_labels")
        return [(sem[int(pt_off[i]):int(pt_off[i + 1])], inst[int(pt_off[i]):int(pt_off[i + 1])]) for i in range(ns)]

    def _make_noise(self, scenes, region_scene, region_m, total):
        """Standard-normal draws for the variational-mean init (gpytorch draws them from the unseeded
        global RNG).  Seeded scenes: ONE numpy Generator per scene, regions consume it in event order."""
        if all(s.noise_seed is None for s in scenes):
            return torch.randn(total, dtype=torch.float32, device=self.device)
        parts = []
        per_scene = {}
        for sc, m in zip(region_scene, region_m):
            per_scene[int(sc)] = per_scene.get(int(sc), 0) + int(m)
        for sc in sorted(per_scene):     # regions are ordered by scene, then event order
            seed = scenes[sc].noise_seed
            if seed is None:
                parts.append(torch.randn(per_scene[sc], dtype=torch.float32).numpy())
            else:
                parts.append(np.random.default_rng(seed).standard_normal(per_scene[sc]).astype(np.float32))
        return self._dev(np.concatenate(parts))


_engines = {}


def get_engine(device=None) -> GaproEngine:
    if not torch.cuda.is_available():
        raise _lib.GaproError("gapro_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    dev = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
    key = (dev.type, dev.index)
    if key not in _engines:
        _engines[key] = GaproEngine(dev)
    return _engines[key]
