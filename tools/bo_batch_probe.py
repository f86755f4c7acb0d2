"""Batch acquisition rounds of BASELINE configs[3]: ResNet-101 bf16 (engine defaults, tie policy on), n = m = 8192,
S = 50, fixed length scale 3.0.  For each batch size q, one warm-up round, then rounds of select_batch(q) + one batched
score_masks + set_batch_values until 1024 masks are acquired.  One JSON line per q:

  round_ms          host clock per round, each round ends in a device synchronise
  acq_per_s         acquired evaluations per second
  pick_ms           device time of the selection kernels (CUDA events around nib_gp_kb_select) over q
  pick_bytes        bytes one pick moves: the (n+k) x m fp64 pass over V plus its O(m) vectors (mean of the batch)
  pick_hbm_share    pick_bytes / pick time against 7.7 TB/s
  score_ms          score_masks of the round's q masks (host clock, synchronised)

    python tools/bo_batch_probe.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import network_interpretation_imagenet_b200 as nib
from network_interpretation_imagenet_b200 import gp as _gp, synthetic
from network_interpretation_imagenet_b200.masks import KEEP_MUL

HBM_PEAK = 7.7e12   # B/s, HGX B200 data sheet, one GPU


def pick_bytes(n, k, m, words, sms):
    """What nib_gp_kb_select moves for pick k: V rows 0..n+k-1 once, the colreduce partials written and read back,
    the new V row, ssq read + written, mu, alive, the candidate bits (the slice count as kb_slices picks it)."""
    nk = n + k
    tiles = -(-m // 512)
    s = max(1, min(-(-nk // 64), -(-4 * sms // tiles)))
    rows = -(-nk // s)
    slices = -(-nk // rows)
    return nk * m * 8 + m * (2 * 8 * slices + 8 + 16 + 8 + 1 + 8 * words)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--acquire", type=int, default=1024)
    ap.add_argument("--qs", type=int, nargs="+", default=[1, 16, 64, 256])
    args = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]
    n = m = 8192
    S = 50
    model = synthetic.build_imagenet_model("resnet101")
    x = synthetic.synthetic_image("imagenet")
    seg = synthetic.voronoi_labels(224, 224, S)
    bits = nib.selection_bits(nib.draw_selections("subset_keep", S, n + m, seed=1), S)
    eng = nib.PerturbationEngine(model, x, seg, target=0, mode=KEEP_MUL, precision="bf16", max_batch=256, S=S)
    score = lambda b: eng.score_masks(b)["target_prob"].double().cpu().numpy()
    y = score(bits[:n])
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    lines = []
    for q in args.qs:
        rounds = args.acquire // q
        gp = _gp.ActiveMaskGP(bits[n:], alpha=1e-5, length_scale=3.0, normalize_y=True,
                              capacity=(rounds + 1) * q).fit(bits[:n], y)
        t_round, t_score, t_pick, nbytes = [], [], [], []
        for r in range(rounds + 1):
            torch.cuda.synchronize()
            n0 = gp.n
            t0 = time.perf_counter()
            picks, _ = gp.select_batch(q)
            t1 = time.perf_counter()
            s = score(bits[n:][picks])
            t2 = time.perf_counter()
            gp.set_batch_values(s)
            torch.cuda.synchronize()
            t3 = time.perf_counter()
            assert len(picks) == q
            if r == 0:
                continue   # warm-up round
            t_round.append(t3 - t0)
            t_score.append(t2 - t1)
            t_pick.append(gp.stats["select_ms"] / q)
            nbytes.append(np.mean([pick_bytes(n0, k, m, gp.words, sms) for k in range(q)]))
        round_ms = 1e3 * float(np.mean(t_round))
        pick_ms = float(np.mean(t_pick))
        pb = float(np.mean(nbytes))
        line = {"q": q, "n": n, "m": m, "S": S, "rounds": rounds, "acquired": rounds * q, "round_ms": round(round_ms, 3),
                "acq_per_s": round(q / (round_ms * 1e-3), 1), "pick_ms": round(pick_ms, 4), "pick_bytes": int(pb),
                "pick_TBps": round(pb / (pick_ms * 1e-3) / 1e12, 3),
                "pick_hbm_share": round(pb / (pick_ms * 1e-3) / HBM_PEAK, 3),
                "score_ms": round(1e3 * float(np.mean(t_score)), 3), "card": card}
        print(json.dumps(line), flush=True)
        lines.append(line)
        del gp
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
