#!/usr/bin/env python
"""Compare two directories written by `bench.py --dump-outputs`: per array, the largest |new - old| / max(|old|, 1),
whether the two are bitwise equal, and how many units (last axis) differ by more than 1e-10 / 1e-6.  Integer arrays
(status words) are compared for identity.

    python scripts/compare_dumps.py OLD_DIR NEW_DIR        # prints one JSON object, exits 1 if an array is missing
"""
import json
import os
import sys

import numpy as np


def compare(old_dir, new_dir):
    out = {}
    for name in sorted(f for f in os.listdir(old_dir) if f.endswith(".npy")):
        a = np.load(os.path.join(old_dir, name))
        path = os.path.join(new_dir, name)
        if not os.path.exists(path):
            out[name[:-4]] = {"missing": True}
            continue
        b = np.load(path)
        r = {"shape": list(a.shape), "bitwise_equal": bool(a.shape == b.shape and a.tobytes() == b.tobytes())}
        if a.shape == b.shape:
            if np.issubdtype(a.dtype, np.floating):
                with np.errstate(invalid="ignore"):
                    rel = np.abs(b - a) / np.maximum(np.abs(a), 1.0)
                both_nan = np.isnan(a) & np.isnan(b)
                rel = np.where(both_nan, 0.0, rel)
                r["max_rel_diff"] = float(np.nanmax(rel)) if rel.size else 0.0
                r["nan_mismatch"] = int(np.count_nonzero(np.isnan(a) != np.isnan(b)))
                # per unit (last axis: trajectories / parameter samples): how the difference is distributed
                per_unit = np.nanmax(rel.reshape(-1, rel.shape[-1]), axis=0) if rel.size else rel
                r["units"] = int(per_unit.size)
                r["units_above_1e-10"] = int(np.count_nonzero(per_unit > 1e-10))
                r["units_above_1e-6"] = int(np.count_nonzero(per_unit > 1e-6))
                if per_unit.size:
                    r["per_unit_quantiles_50_99_99.9"] = [float(q) for q in np.quantile(per_unit, [0.5, 0.99, 0.999])]
            else:
                r["entries_differing"] = int(np.count_nonzero(a != b))
        out[name[:-4]] = r
    return out


def main():
    res = compare(sys.argv[1], sys.argv[2])
    print(json.dumps(res, indent=1))
    sys.exit(1 if any(v.get("missing") for v in res.values()) else 0)


if __name__ == "__main__":
    main()
