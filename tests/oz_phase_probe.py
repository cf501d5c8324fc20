"""Development probe (GPU): one training step, phase by phase, DMMA path vs tcgen05 digit-plane path -
which buffer diverges first and by how much."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gapro_b200 import _debug  # noqa: E402
from tests.golden.make_golden import gp_case  # noqa: E402

PH = _debug.PHASES


def state(case, iters, stop, oz):
    os.environ["GAPRO_GP_OZAKI"] = "1" if oz else "0"
    os.environ["GAPRO_GP_OZAKI_MIN_M"] = "128"
    X, n1, Xt, noise = case
    dev = torch.device("cuda:0")
    feats = torch.from_numpy(np.concatenate([X, Xt])).to(dev)
    M, N = len(X), len(Xt)
    return _debug.gp_debug_state(feats, np.arange(M), n1, np.arange(M, M + N), noise, iters=iters, stop_phase=stop)


def main():
    for (cid, M, D, N) in [(100, 200, 6, 40), (102, 520, 32, 48), (103, 520, 6, 48), (104, 576, 6, 48), (105, 640, 6, 20),
                           (101, 1000, 6, 64)]:
        case = gp_case(cid, M, D, N)
        print(f"== M={M} D={D}")
        for iters in (0, 3):
            prev = None
            for stop in range(3, len(PH) + 1):
                a = state(case, iters, stop, False)
                b = state(case, iters, stop, True)
                worst = []
                for k in ("A", "Bm", "GA", "GC", "T", "Tm", "m", "Z", "gZ", "scal", "gmu", "gv", "gsrow", "glrow"):
                    da = np.abs(a[k] - b[k]).max()
                    sc = max(np.abs(a[k]).max(), 1e-300)
                    worst.append((da / sc, k))
                worst.sort(reverse=True)
                msg = ", ".join(f"{k}:{v:.1e}" for v, k in worst[:4])
                print(f"  iters={iters} after phase {PH[stop - 1]:9s}: {msg}", flush=True)


if __name__ == "__main__":
    main()
