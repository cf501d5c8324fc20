"""Golden vectors at BASELINE.json sizes (oracle outputs, fp64 policy; minutes of CPU each, so they are
committed rather than recomputed by the GPU tests):

  gp_case_8k.npz       one GP region with M = 4200 training rows and N = 3800 test rows (M + N = 8000,
                       the "ambiguous regions up to 8k" of configs[3]; fit_gp_spp,
                       /root/reference/gapro/gaussian_process_utils.py:382-445)
  scene_c1_full.npz    one full configs[1] scene (150k points, seed 1000) through the whole pipeline
  scene_c3_full.npz    scene 0 of the configs[2] batch (the first scene of the bench batch, seed 1000)
  scene_c4_full.npz    one configs[3] scene (400k points, 85 boxes, 201 GP regions, the largest with M = 5122
                       training and 2746 test superpoints)

  scene_c5_full.npz    one configs[4] scene (1M points, 125 boxes, 349 GP regions up to M = 3587; ~3 CPU-hours)

The scene files hold the point labels once per superpoint (sem_spp / inst_spp / prob_spp); load_scene expands them.

    python tests/golden/make_golden_fullsize.py [gp8k] [c1] [c3] [c4] [c5]

Like make_golden.py these pin the CUDA path to the ORACLE at full size; the oracle's scene pipeline is
pinned to the reference's own code by make_ref_golden.py, the inside of the GP fit is a restatement
("parity unpinned", oracle/__init__.py).
"""
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from gapro_b200 import synthetic                       # noqa: E402
from gapro_b200.gen_ps import synthetic_inputs         # noqa: E402
from oracle import gen_ps_oracle as O                  # noqa: E402
from oracle import gp_oracle as G                      # noqa: E402
from tests.golden.make_golden import gp_case, input_digest   # noqa: E402

GP_8K = (300, 4200, 6, 3800)        # (case id, M, D, N)
SCENES = {"c1": ("c1", 1000, 11), "c3": ("c3:0", 1000, 12), "c4": ("c4", 1000, 13), "c5": ("c5", 1000, 14)}     # name -> (config, scene seed, noise seed)


def scene_cfg(name):
    return synthetic.c3_config(int(name.split(":")[1])) if name.startswith("c3:") else synthetic.CONFIGS[name]


def scene_args(cfg_name, seed):
    inp = synthetic_inputs(synthetic.make_scene(seed, scene_cfg(cfg_name)))
    return (inp["xyz"], inp["mask_feats"].astype(np.float32), inp["spp"], inp["instance_cls"].astype(np.int64),
            inp["instance_box"].astype(np.float32), inp["instance_box_volume"].astype(np.float32),
            inp["wall_box"], inp["wall_volume"])


def make_gp8k():
    i, M, D, N = GP_8K
    X, n1, Xt, noise = gp_case(i, M, D, N)
    t0 = time.time()
    r = G.fit_region_autograd(X, n1, Xt, noise)
    np.savez_compressed(os.path.join(HERE, "gp_case_8k.npz"), mu64=r["mu64"], var64=r["var64"], prob=r["prob"],
                        label=r["label"], conf=r["conf"], case=np.array(GP_8K),
                        min_margin=np.array(np.abs(r["prob64"] - 0.5).min()))
    print(f"gp 8k: M={M} N={N} mu[0]={r['mu64'][0]:.6f} min margin {np.abs(r['prob64'] - 0.5).min():.3g} "
          f"({time.time() - t0:.0f}s)")


def to_superpoints(spp, point_labels):
    """sem / inst / prob of a scene are broadcast from its superpoints: one value per superpoint, in the order of
    mu / var (np.unique of the raw superpoint ids).  Keeps the full-size fixtures small."""
    dense = np.unique(spp, return_inverse=True)[1]
    out = []
    for a in point_labels:
        s = np.zeros(dense.max() + 1, a.dtype)
        s[dense] = a
        assert (s[dense] == a).all(), "a label differs inside a superpoint"
        out.append(s)
    return out


def load_scene(tag, spp):
    """scene_<tag>_full.npz with sem / inst / prob expanded from superpoints back to the scene's points."""
    gold = dict(np.load(os.path.join(HERE, f"scene_{tag}_full.npz")))
    dense = np.unique(spp, return_inverse=True)[1]
    for k in ("sem", "inst", "prob"):
        gold[k] = gold.pop(k + "_spp")[dense]
    return gold


def make_scene(tag):
    cfg_name, seed, nseed = SCENES[tag]
    args = scene_args(cfg_name, seed)
    t0 = time.time()
    res, dbg = O.gen_pseudo_label_oracle(*args, thresh_spp_occu=0.999, noise_seed=nseed, return_debug=True)
    margins = [np.abs(r["res"]["prob64"] - 0.5).min() for r in dbg["regions"]]
    sem, inst, prob = to_superpoints(args[2], (res[0].astype(np.int8), res[1].astype(np.int16), res[2]))
    # competition margin: |new confidence - confidence being replaced| over all merges, from a replay
    np.savez_compressed(os.path.join(HERE, f"scene_{tag}_full.npz"), sem_spp=sem, inst_spp=inst,
                        prob_spp=prob, mu=res[3], var=res[4], digest=np.array(input_digest(args)),
                        n_regions=np.array(len(dbg["regions"])), min_margin=np.array(min(margins) if margins else 1.0),
                        max_m=np.array(max((len(r["b1_inds"]) + len(r["b2_inds"]) for r in dbg["regions"]), default=0)),
                        occ_spp=np.packbits(dbg["occ_spp"], axis=1))
    print(f"scene {tag}: {len(res[0])} pts, {len(res[3])} spp, {len(dbg['regions'])} GP regions, max M "
          f"{max((len(r['b1_inds']) + len(r['b2_inds']) for r in dbg['regions']), default=0)}, "
          f"min posterior margin {min(margins) if margins else 1:.3g} ({time.time() - t0:.0f}s)")


if __name__ == "__main__":
    what = sys.argv[1:] or ["c1", "c3", "gp8k"]
    for w in what:
        make_gp8k() if w == "gp8k" else make_scene(w)
