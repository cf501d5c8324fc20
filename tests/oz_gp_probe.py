"""Development probe (GPU): accuracy and time of whole GP fits on the DMMA path and on the tcgen05 digit-plane path
(8 digits) against the golden fp64-oracle vectors.  Env knobs are read per call by the library."""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gapro_b200.gaussian_process_utils import fit_gp_regions  # noqa: E402
from tests.conftest import rel_err  # noqa: E402
from tests.golden.make_golden import GP_CASES_LARGE, gp_case  # noqa: E402
from tests.golden.make_golden_fullsize import GP_8K  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def run(case_id, M, D, N, mu_ref, var_ref, label):
    dev = torch.device("cuda:0")
    X, n1, Xt, noise = gp_case(case_id, M, D, N)
    feats = torch.from_numpy(np.concatenate([X, Xt])).to(dev)
    for env in ({"GAPRO_GP_OZAKI": "0"}, {"GAPRO_GP_OZAKI": "1"}):
        os.environ.update(env)
        os.environ["GAPRO_GP_OZAKI_MIN_M"] = "512"
        ts = []
        for rep in range(2):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = fit_gp_regions(feats, [np.arange(M)], [n1], [np.arange(M, M + N)], init_noise=[noise], return_float64=True)[0]
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        print(f"{label} M={M} D={D} {env}: mu rel {rel_err(r[5].cpu().numpy(), mu_ref):.2e} var rel "
              f"{rel_err(r[6].cpu().numpy(), var_ref):.2e}  {min(ts) * 1e3:.1f} ms", flush=True)


def main():
    gold = np.load(os.path.join(GOLD, "gp_cases_large.npz"))
    for i, (M, D, N) in enumerate(GP_CASES_LARGE):
        if M >= 512:
            run(100 + i, M, D, N, gold[f"c{i}_mu64"], gold[f"c{i}_var64"], "large")
    g8 = np.load(os.path.join(GOLD, "gp_case_8k.npz"))
    i, M, D, N = GP_8K
    run(i, M, D, N, g8["mu64"], g8["var64"], "8k")


if __name__ == "__main__":
    main()
