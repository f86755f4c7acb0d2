"""Times the pixel GP (ski.GridGPRegression) with the Kronecker solver at grid_size 30, 64, 100 and 300, and the dense
solver where it runs, on n = 224^2 training pixels: a full lattice, a lattice with an uncovered 44-column strip, and a
lattice with an uncovered 44 x 44 square (not a lattice: the preconditioner is inexact there, and the iteration counts
show by how much).  Writes one JSON (default profiles/ski_kron_probe.json).

Per configuration: fit, mean-only predict at all 224^2 pixels, and mean + variance predict at all 224^2 pixels (8192
seeded pixels for the square hole), in seconds from a host clock around work that ends in a device synchronise, with
the PCG iteration counts of the mean solve and of each variance block.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ski_kron_probe.json"))
    ap.add_argument("--grids", default="30,64,100,300")
    args = ap.parse_args()
    from network_interpretation_imagenet_b200 import build
    build.build()
    from network_interpretation_imagenet_b200.ski import GridGPRegression

    full = np.stack(np.meshgrid(np.arange(224.0), np.arange(224.0), indexing="ij"), -1).reshape(-1, 2)
    strip = (full[:, 1] < 150) | (full[:, 1] >= 194)
    square = ~((full[:, 0] >= 90) & (full[:, 0] < 134) & (full[:, 1] >= 90) & (full[:, 1] < 134))
    y_all = 20.0 * np.exp(-((full[:, 0] - 100) ** 2 + (full[:, 1] - 120) ** 2) / (2 * 40.0 ** 2))
    sets = {"full": np.ones(full.shape[0], bool), "strip44": strip, "square44": square}
    q_all = torch.from_numpy(full).cuda()
    q_sub = q_all[torch.from_numpy(np.random.RandomState(0).choice(full.shape[0], 8192, replace=False)).cuda()]
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    rows = []
    for gs in (int(g) for g in args.grids.split(",")):
        for ell in (1.0, 10.0):
            for name, keep in sets.items():
                X, y = torch.from_numpy(full[keep]).cuda(), torch.from_numpy(y_all[keep]).cuda()
                q = q_sub if name == "square44" else q_all
                for solver in ("kron", "dense") if gs <= 100 else ("kron",):
                    gp = GridGPRegression(gs, ((0.0, 224.0), (0.0, 224.0)), ell, 1.0, 1.0, solver=solver)
                    gp.fit(X, y)                                                    # warm-up of every shape
                    gp.predict(q[:256])
                    t_fit, _ = timed(lambda: gp.fit(X, y))
                    t_mean, _ = timed(lambda: gp.predict(q_all, return_var=False))
                    t_var, _ = timed(lambda: gp.predict(q))
                    row = {"grid_size": gs, "length_scale": ell, "train": name, "n": int(keep.sum()), "solver": solver,
                           "fit_s": t_fit, "predict_mean_s": t_mean, "predict_mean_var_s": t_var,
                           "var_queries": int(q.shape[0])}
                    if solver == "kron":
                        row.update(mean_iters=gp.mean_iters, var_block_iters=gp.var_iters)
                    rows.append(row)
                    print(json.dumps(row), flush=True)
                    del gp
                    torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump({"device": card, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
