"""Development probe (GPU): the whole configs[3] scene against its offline oracle fixture, on the DMMA path and with
the large regions on tcgen05."""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gapro_b200.engine import SceneInputs, get_engine  # noqa: E402
from tests.conftest import rel_err  # noqa: E402
from tests.golden.make_golden_fullsize import SCENES, load_scene, scene_args  # noqa: E402

dev = torch.device("cuda:0")
TAG = sys.argv[1] if len(sys.argv) > 1 else "c4"
cfg_name, seed, nseed = SCENES[TAG]
args = scene_args(cfg_name, seed)
gold = load_scene(TAG, args[2])
T = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(dt).to(dev)
sc = SceneInputs(T(args[0], torch.float64), T(args[1], torch.float32), T(args[2], torch.int64), T(args[3], torch.int64),
                 T(args[4], torch.float32), T(args[5], torch.float32), T(args[6], torch.float32), T(args[7], torch.float32),
                 noise_seed=nseed)
eng = get_engine(dev)
for oz in ("0", "1"):
    os.environ["GAPRO_GP_OZAKI"] = oz
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = eng.run([sc], thresh_spp_occu=0.999)[0]
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    sem, inst, prob, mu, var = [t.cpu().numpy() for t in out]
    g = gold["mu"] != -100
    print(f"GAPRO_GP_OZAKI={oz}: {dt * 1e3:.0f} ms; labels differ at {int((sem != gold['sem']).sum())} sem / "
          f"{int((inst != gold['inst']).sum())} inst of {len(sem)} points; sentinel pattern equal {bool(((mu != -100) == g).all())}; "
          f"mu rel {rel_err(mu[g], gold['mu'][g]):.2e} var rel {rel_err(var[g], gold['var'][g]):.2e} "
          f"prob max abs {np.abs(prob - gold['prob']).max():.2e}; elementwise mu rtol max "
          f"{np.max(np.abs(mu[g] - gold['mu'][g]) / np.abs(gold['mu'][g])):.2e}", flush=True)
    bad = np.flatnonzero((sem != gold["sem"]) | (inst != gold["inst"]))
    if len(bad):
        print("   first differing points:", bad[:5], "prob there", prob[bad[:5]], "oracle prob", gold["prob"][bad[:5]],
              "n_regions", eng.last_stats["n_regions"], int(gold["n_regions"]))
    k = np.argsort(-np.abs(mu[g] - gold["mu"][g]))[:3]
    print("   worst mu:", mu[g][k], gold["mu"][g][k], "var:", var[g][k], gold["var"][g][k])
