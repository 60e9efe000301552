"""Device time of k_weights (exact left folds) and k_resample_indices by population size (run on a GPU box).
--tau T: with the adaptive-resampling threshold T (> 0 adds the exact fold of the squares); --sizes n,n,...:
populations (default 1024, 8192, 65536, 262144); --out FILE: also write the rows there as JSON."""
import argparse, json, sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from slamrs_b200.slam import debug_resample
ap = argparse.ArgumentParser()
ap.add_argument("--tau", type=float, default=0.0)
ap.add_argument("--sizes", default="1024,8192,65536,262144")
ap.add_argument("--out", default=None)
args = ap.parse_args()
rng = np.random.default_rng(0)
rows = []
for n in (int(s) for s in args.sizes.split(",")):
    for name, w in (("uniform", rng.random(n)), ("lognormal10", np.exp(rng.normal(-200, 10, n))),
                    ("peaked", np.concatenate([[1.0], np.exp(rng.normal(-38, 2, n - 1))]))):
        r = debug_resample(w, 0.37, timing=True, tau=args.tau)
        rows.append(dict(n=n, weights=name, tau=args.tau, k_weights_us=r["us"][0], k_resample_indices_us=r["us"][1],
                         rounds=r["fold_rounds"], heads=r["fold_heads"], fallback=r["fold_fallback"]))
        print(rows[-1], flush=True)
if args.out:
    os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
    json.dump(rows, open(args.out, "w"), indent=1)
