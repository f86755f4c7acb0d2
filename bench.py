#!/usr/bin/env python
"""bench.py — masked forward evals/sec of the perturbation-interpretation hot path on N B200s.

Workload (BASELINE.json configs[2], generate_gp_training_data_imagenet.py): ResNet-101 224x224, one synthetic image,
S = 50 superpixels, random keep-masks (the k = int(0.4*S) subset variant of imagenet :231), each mask synthesised,
multiplied into the image, scored through the classifier and reduced to (top-1, target-class probability), with the
bf16 tie policy (near-tied masks re-scored in fp32, device side) inside the timed region.
One "step" = `--masks-per-step` masks per GPU through that whole path (weak scaling: per-GPU work is fixed); the
16384-mask job of configs[2] is 8 ranks x 2048 masks = one step at N = 8.  After every step the per-rank score
blocks are all-gathered (libnib's NCCL call) so each rank holds the global (prob, top1) table, as the GP rank needs.

  value   masks/s with selections already resident in HBM when the timed region starts (CUDA events)
  e2e     same path through the public API with HOST buffers: every step copies the image, label map and
          selection bit-vectors host->device from pinned memory and reads the score table back
  roofline  the dominant kernel (tcgen05 implicit-GEMM conv): algorithmic FLOPs / summed launch time measured
          with CUDA events on the launching stream, against MEASURED_PEAKS.json bf16_tflops_sustained
  roofline_mask_synth, gp.roofline   the HBM-bound mask kernel and the fp64 GP stage against their own peaks
  cpu_baseline  the oracle's restated reference loop (numpy mask + torch CPU fp32 forward, batch 1, all host threads),
          plus scikit-learn's fixed-theta GP fit + predict for the GP half of the metric
  library_bar   torch eager (cuDNN) bf16 channels-last forward of the same network on the same GPU: a measurement
          beside the product, never on its path

Other modes:  --strong (the literal configs[2] job: --total-masks 16384 split over the ranks, strong scaling);
--arch densenet121 --images 64 --masks-per-image 4096 (configs[4]: the flattened (image, mask) index space sharded over
the ranks).  `--impl reference` times the CPU loop alone (the reference has no GPU-independent implementation we could
install: its scripts do not parse on Python 3.12 — see DESIGN.md).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = "evals/s"
# SURVEY.md §8d: conv+fc 2*MAC per evaluation (torchvision 0.26), and App. B conv input + output elements per eval (bf16)
FLOPS_PER_EVAL = {"resnet101": 15.602810880e9, "densenet121": 5.668323328e9}
ACT_BYTES_PER_EVAL = {"resnet101": (15.78e6 + 16.23e6) * 2, "densenet121": 43.7e6}
MASK_BYTES_PER_EVAL = 3 * 224 * 224 * 2      # SURVEY.md §8d: bf16 224^2, unpadded C = 3 (output bytes only)


def metric_name(arch):
    return "masked forward evals/sec (ResNet-101 224^2)" if arch == "resnet101" else f"masked forward evals/sec ({arch} 224^2)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--masks-per-step", type=int, default=3072, help="masks per GPU per step (weak scaling)")
    ap.add_argument("--strong", action="store_true", help="fixed job of --total-masks per step split over the ranks")
    ap.add_argument("--total-masks", type=int, default=16384, help="--strong: BASELINE configs[2] is 16384 masks of one image")
    ap.add_argument("--images", type=int, default=1, help="> 1: sweep over that many synthetic images (configs[4]: 64)")
    ap.add_argument("--masks-per-image", type=int, default=4096, help="with --images > 1 (configs[4]: 4096)")
    ap.add_argument("--micro-batch", type=int, default=384,
                    help="masks per forward; 384 x 196 output pixels = 294 pair tiles = 3.97 waves on 74 CTA pairs in layer 3 "
                         "(256 gives 2.65 waves: same evals/s at the power cap, but 17 %% lower per-kernel rate)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--arch", default="resnet101")
    ap.add_argument("--streams", type=int, default=2,
                    help="copies of the lowered classifier fed round-robin with micro-batches from their own CUDA streams")
    ap.add_argument("--refine-ties", default="auto", help="'auto' (engine default band), a float band, or 0 to switch the tie policy off")
    ap.add_argument("--tie-capacity", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-bar", action="store_true")
    ap.add_argument("--no-gp", action="store_true")
    ap.add_argument("--gp-n", type=int, default=8192, help="GP training-set size (BASELINE configs[3]: n = 8192)")
    ap.add_argument("--graph", action="store_true", help="replay each micro-batch forward as a CUDA graph")
    ap.add_argument("--profile-json", default=None, help="write the per-op CUDA-event profile of one micro-batch here")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the score table of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl ours")
    return args


NCU_CAPTURES = ("r02_ncu_all_launches_one_forward.csv", "r01_ncu_all_launches_one_forward_v6_mb256.csv")


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum summed over the tcgen05 conv launches of ONE forward, from the newest
    committed ncu capture (profiles/, one pass with cache control on: cold-L2 per launch).  Returns (total bytes, number of
    conv launches, micro-batch of the capture, file name) or None."""
    import csv
    import re
    for name in NCU_CAPTURES:
        p = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(p):
            continue
        tot, n = 0.0, 0
        for r in csv.DictReader(open(p)):
            if r["kernel"].startswith("conv_tc") or r["kernel"].startswith("conv_fused"):
                tot += float(r["dram__bytes_read.sum"]) + float(r["dram__bytes_write.sum"])
                n += 1
        mb = 256
        meta = p.replace(".csv", ".meta.json")
        if os.path.exists(meta):
            mb = int(json.load(open(meta)).get("micro_batch", mb))
        else:
            m = re.search(r"_mb(\d+)", name)
            mb = int(m.group(1)) if m else mb
        if n:
            return tot, n, mb, name
    return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---- the CPU arm -----------------------------------------------------------------------------------------
def cpu_reference_loop(model, x, seg, sels, target, torch):
    """One iteration of generate_gp_training_data_imagenet.py:221-266 per mask, restated in oracle/ (batch 1)."""
    from oracle import masks as om
    correct = 0
    with torch.no_grad():
        for sel in sels:
            mask = om.pixel_mask_keep(seg, sel)
            masked = om.apply_keep(x, mask)
            out = model(torch.from_numpy(masked[None]))
            pred = out.max(1, keepdim=True)[1]
            correct += int(pred[0, 0] == target)
    return correct


def cpu_baseline(arch, seconds_budget=12.0):
    import torch
    from oracle import classifier as ocls, synthetic
    import network_interpretation_imagenet_b200.masks as pmasks
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model = ocls.build_imagenet_model(arch)
    x = synthetic.synthetic_image("imagenet")
    seg = synthetic.voronoi_labels(224, 224, 50)
    sels = pmasks.draw_selections("subset_keep", 50, 4096, seed=1)
    cpu_reference_loop(model, x, seg, sels[:2], 0, torch)            # warm-up
    t0 = time.perf_counter()
    cpu_reference_loop(model, x, seg, sels[2:6], 0, torch)
    per = (time.perf_counter() - t0) / 4
    n = int(max(8, min(1024, seconds_budget / max(per, 1e-4))))
    t0 = time.perf_counter()
    cpu_reference_loop(model, x, seg, sels[6:6 + n], 0, torch)
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n} masks of the same workload, batch 1 per forward like the reference (imagenet :246), "
                      f"numpy mask ops + torch {torch.__version__} CPU fp32, {cores} threads, {dt:.1f} s"}


def cpu_gp_baseline(np, S, sizes=(1024, 8192), budget_s=40.0):
    """scikit-learn's own GaussianProcessRegressor at fixed theta (optimizer=None), the estimator BayesianOptimization.py
    :154-166 builds: fit + predict(return_std) ms on the host cores, same inputs as gp_bench."""
    from oracle import gp as ogp
    import sklearn
    cores = os.cpu_count() or 1
    res = {}
    spent = 0.0
    for n in sizes:
        if n > 2048 and spent + 30.0 * (n / 8192.0) ** 3 > budget_s:
            res[str(n)] = {"skipped": "time budget"}
            continue
        rng = np.random.RandomState(0)
        sels = [list(rng.choice(S - 1, size=20, replace=False)) for _ in range(2 * n)]
        X = np.zeros((2 * n, S))
        for i, s in enumerate(sels):
            X[i, s] = 1.0
        y = rng.rand(n)
        est = ogp.sklearn_gp(alpha=1e-5, n_restarts_optimizer=0, optimizer=None, length_scale=3.0)
        t0 = time.perf_counter()
        est.fit(X[:n], y)
        t1 = time.perf_counter()
        est.predict(X[n:], return_std=True)
        t2 = time.perf_counter()
        spent += t2 - t0
        res[str(n)] = {"fit_ms": (t1 - t0) * 1e3, "predict_ms": (t2 - t1) * 1e3, "fit_plus_predict_ms": (t2 - t0) * 1e3}
    return {"kind": "reference dependency", "what": f"scikit-learn {sklearn.__version__} GaussianProcessRegressor(RBF(3.0), alpha=1e-5, "
            "normalize_y=True, optimizer=None).fit + .predict(return_std=True), n = m", "cores": cores, "unit": "ms", "by_n": res}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from oracle import classifier as ocls, synthetic
    import network_interpretation_imagenet_b200.masks as pmasks
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model = ocls.build_imagenet_model(args.arch)
    x = synthetic.synthetic_image("imagenet")
    seg = synthetic.voronoi_labels(224, 224, 50)
    per_step = 24   # bounded sample of the step: the CPU path is ~10^3 x slower
    total = (args.steps + args.warmup) * per_step
    sels = pmasks.draw_selections("subset_keep", 50, total, seed=1)
    k = 0
    for _ in range(args.warmup):
        cpu_reference_loop(model, x, seg, sels[k:k + per_step], 0, torch); k += per_step
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_reference_loop(model, x, seg, sels[k:k + per_step], 0, torch); k += per_step
    dt = time.perf_counter() - t0
    v = args.steps * per_step / dt
    sample = (f"{per_step} masks per step (bounded sample of the {args.masks_per_step}-mask step), batch 1 per forward, "
              f"oracle port of the reference loop on {cores} host threads")
    print(json.dumps({
        "impl": "reference", "metric": metric_name(args.arch), "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong" if (args.strong or args.images > 1) else "weak",
        "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": {"workload": f"generate_gp_training_data_imagenet.py: {args.arch} 224^2, S=50 superpixels, keep-masks",
                   "masks_per_step_per_gpu": per_step, "arch": args.arch},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


# ---- our arm ---------------------------------------------------------------------------------------------
DUMP_MAX_ROWS = 1 << 21      # 16 bytes per row with the row index: 32 MiB, under the 64 MB a dump may take


def dump_outputs(out_dir, table, np):
    """The [N, 2] score table of a step as PerturbationEngine.score_masks hands it out: target_prob.npy and top1.npy,
    float32, one entry per mask in job order.  Inputs are seeded, so two builds can be compared file for file.  A table
    of more than DUMP_MAX_ROWS masks is written as a fixed seeded sample of its rows, with their indices in row.npy
    (float64)."""
    t = table.float().cpu().numpy()
    arrays = {"target_prob": t[:, 0].copy(), "top1": t[:, 1].copy()}
    if t.shape[0] > DUMP_MAX_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(t.shape[0], DUMP_MAX_ROWS, replace=False))
        arrays = {k: v[rows] for k, v in arrays.items()}
        arrays["row"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import network_interpretation_imagenet_b200 as nib
    from network_interpretation_imagenet_b200 import synthetic
    from network_interpretation_imagenet_b200.masks import MaskSynth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    peaks = load_peaks()
    arch = args.arch
    S, mb = 50, args.micro_batch

    # ---- the job: a list of images, each with its own mask table; the flattened (image, mask) index space is sharded
    n_img = max(1, args.images)
    if n_img > 1:
        per_image = args.masks_per_image
        scaling = "strong"
    elif args.strong:
        per_image = args.total_masks
        scaling = "strong"
    else:
        per_image = args.masks_per_step * world
        scaling = "weak"
    total = n_img * per_image
    lo, hi, per = nib.shard_range(total, rank, world)

    model = synthetic.build_imagenet_model(arch)     # random-init torchvision model, seeded (no network for weights)
    x0 = synthetic.synthetic_image("imagenet")
    seg0 = synthetic.voronoi_labels(224, 224, S)
    refine = args.refine_ties
    refine = "auto" if refine == "auto" else (float(refine) or None)
    kw = {} if args.tie_capacity is None else {"tie_capacity": args.tie_capacity}
    eng = nib.PerturbationEngine(model, x0, seg0, target=0, mode=nib.KEEP_MUL, precision=args.precision, max_batch=mb,
                                 S=S, device=dev, use_graph=args.graph, streams=args.streams, refine_ties=refine, **kw)
    clf = eng.classifier
    # images / label maps / selections generated identically on every rank from seeds (zero input communication)
    synths, imgs_host, labs_host = [eng.synth], [torch.from_numpy(x0).pin_memory()], [torch.from_numpy(seg0.astype(np.uint8)).pin_memory()]
    for i in range(1, n_img):
        xi = synthetic.synthetic_image("imagenet", seed=1234 + i)
        si = synthetic.voronoi_labels(224, 224, S, seed=7 + i)
        synths.append(MaskSynth(xi, si, S=S, device=dev))
        imgs_host.append(torch.from_numpy(xi).pin_memory())
        labs_host.append(torch.from_numpy(si.astype(np.uint8)).pin_memory())
    # this rank's segments of the flattened index space: (image, first mask, last mask, offset in the local block)
    segments = []
    for i in range(n_img):
        a, b = max(lo, i * per_image), min(hi, (i + 1) * per_image)
        if a < b:
            segments.append((i, a - i * per_image, b - i * per_image, a - lo))
    bits_host, bits_dev = {}, {}
    for (i, a, b, off) in segments:
        sels = nib.draw_selections("subset_keep", S, per_image, seed=1 + i)
        bh = torch.from_numpy(nib.selection_bits(sels, S)[a:b].view(np.int64).copy()).pin_memory()
        bits_host[i], bits_dev[i] = bh, bh.to(dev)
    scores_host = torch.empty(world * per, 2, dtype=torch.float32).pin_memory()
    local_scores = torch.zeros(per, 2, dtype=torch.float32, device=dev)
    table = torch.zeros(world * per, 2, dtype=torch.float32, device=dev)

    def device_step(bits):
        """mask synthesis -> classifier (micro-batches of mb, round-robin over the stream copies) -> scores (+ tie policy)
        for this rank's part of the job, then the all-gather."""
        for (i, a, b, off) in segments:
            eng.score_local(bits[i], out=local_scores[off:off + (b - a)], synth=synths[i])
        return eng.gather(local_scores, total, out=table)

    def e2e_step():
        staged = {}
        for (i, a, b, off) in segments:
            synths[i].img.copy_(imgs_host[i], non_blocking=True)
            synths[i].labels.copy_(labs_host[i], non_blocking=True)
            staged[i] = bits_host[i].to(dev, non_blocking=True)
        t = device_step(staged)
        scores_host[: t.shape[0]].copy_(t, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def all_launches():
        a, b = clf.launch_counts()
        if eng._fp32 is not None:           # the tie policy's re-score lowering
            a2, b2 = eng._fp32.launch_counts()
            a, b = a + a2, b + b2
        return a, b

    for _ in range(args.warmup):
        device_step(bits_dev)
    torch.cuda.synchronize()
    l0, t0 = all_launches()
    ties0 = eng.tie_stats()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    last = [None]

    def timed_step():
        last[0] = device_step(bits_dev)

    ms = timed(timed_step, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last[0], np)     # before the e2e steps below overwrite the table
    l1, t1 = all_launches()
    ties1 = eng.tie_stats()
    # + per score_local call: score kernel (+ compact, fp32 score, scatter with the tie policy); + one all-gather per step
    per_pass = 1 + (3 if eng.refine_ties is not None else 0)
    win = eng.tie_window if eng.refine_ties is not None else 1 << 30
    passes = sum((b_ - a_ + win - 1) // win for (_, a_, b_, _) in segments)
    gpu_launches = (l1 - l0) + args.steps * per_pass * passes
    value = total * args.steps / (ms / 1e3)

    for _ in range(2):
        e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    e2e_value = total * args.steps / (ms_e2e / 1e3)
    h2d = sum(imgs_host[i].numel() * 4 + labs_host[i].numel() + bits_host[i].numel() * 8 for (i, _, _, _) in segments)
    d2h = world * per * 2 * 4

    allgather_us = None
    if world > 1:
        reps = 50
        ms_ag = timed(lambda: eng.gather(local_scores, total, out=table), reps)
        allgather_us = ms_ag / reps * 1e3

    # ---- rooflines (rank 0) ------------------------------------------------------------------------------
    roofline = roofline_mask = None
    n_prof = min(mb, per)
    if rank == 0:
        first = segments[0][0]
        clf.forward_masked(synths[first], bits_dev[first][:n_prof], nib.KEEP_MUL)
        profs = sorted((clf.profile(n_prof) for _ in range(5)), key=lambda pr: sum(p[0] for p in pr))
        prof = profs[len(profs) // 2]     # median of five passes by total time (the GPU sits at its power cap: +-5 %)
        KIND = ["simt_conv", "tc_conv", "pool", "fc", "tc_conv_fused_into_previous"]
        if args.profile_json:
            with open(args.profile_json, "w") as f:
                json.dump({"micro_batch": n_prof, "ops": [
                    {"ms": p[0], "kind": KIND[p[1]], "gflop": p[2] / 1e9,
                     "tflops": (p[2] / (p[0] / 1e3) / 1e12) if p[0] > 0 else None,
                     "Hout": p[3][0], "Wout": p[3][1], "Cin": p[3][2], "Cout": p[3][3], "k": p[3][4], "stride": p[3][5],
                     "residual": p[3][6], "block_n": p[3][7]} for p in prof]}, f, indent=0)
        tc_ms = sum(p[0] for p in prof if p[1] in (1, 4))
        tc_fl = sum(p[2] for p in prof if p[1] in (1, 4))
        all_ms = sum(p[0] for p in prof)
        n_tc = sum(1 for p in prof if p[1] == 1)          # launches that really happen (fused partners excluded)
        if n_tc and tc_ms > 0:
            ach = tc_fl / (tc_ms / 1e3) / 1e12
            cap = ncu_traffic()
            traffic = traffic_per_mask = None
            src = None
            if cap is not None:
                tot_b, n_cap, mb_cap, src = cap
                traffic_per_mask = tot_b / mb_cap
                traffic = traffic_per_mask * n_prof / n_tc      # per launch, over the launch count of THIS forward
            alg_per_mask = ACT_BYTES_PER_EVAL.get(arch)
            roofline = {"bound": "tensor", "kernel": "conv_tc3_kernel + conv_fused_ca_kernel (tcgen05 cta_group::2 implicit GEMM)",
                        "achieved": ach, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                        "frac": ach / peaks["bf16_tflops_sustained"], "traffic": traffic,
                        "traffic_per_mask": traffic_per_mask, "algorithmic_bytes_per_mask": alg_per_mask,
                        "traffic_over_algorithmic": (traffic_per_mask / alg_per_mask) if (traffic_per_mask and alg_per_mask) else None,
                        "traffic_source": (f"profiles/{src}: DRAM read+write bytes of every conv launch of one forward (ncu, cold L2 "
                                           "per launch), per mask, re-expressed per launch of this forward") if src else None,
                        "algorithmic_bytes_per_launch": (alg_per_mask * n_prof / n_tc) if alg_per_mask else None,
                        "flops_per_launch": tc_fl / n_tc,
                        "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peaks['source']})",
                        "launches_per_forward": n_tc, "convs_per_forward": sum(1 for p in prof if p[1] in (0, 1, 4)),
                        "share_of_forward": tc_ms / all_ms if all_ms else None,
                        # the same flops over (timed-region time x this share): what the conv kernels deliver inside the
                        # real step, where launches run back to back (PDL, two streams) instead of between event records
                        "achieved_in_step": (tc_fl * (per / n_prof) * args.steps / ((ms / 1e3) * (tc_ms / all_ms)) / 1e12)
                        if all_ms else None,
                        "per_kind_ms": {"simt_conv": sum(p[0] for p in prof if p[1] == 0), "tc_conv": tc_ms,
                                        "pool": sum(p[0] for p in prof if p[1] == 2), "fc": sum(p[0] for p in prof if p[1] == 3)}}
        else:
            simt_ms = sum(p[0] for p in prof if p[1] == 0)
            simt_fl = sum(p[2] for p in prof if p[1] == 0)
            ach = simt_fl / (simt_ms / 1e3) / 1e12 if simt_ms > 0 else 0.0
            roofline = {"bound": "tensor", "kernel": "conv_simt_kernel (CUDA cores; tcgen05 path disabled)", "achieved": ach,
                        "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": ach / peaks["bf16_tflops_sustained"],
                        "traffic": None}
        # mask synthesis alone, into a buffer of the network input's layout (NHWC, 4-channel pixels, 3-pixel halo)
        if args.precision == "bf16":
            cs, pad = clf.in_c_stride, clf.in_pad
            buf = torch.zeros(n_prof, 224 + 2 * pad, 224 + 2 * pad, cs, dtype=torch.bfloat16, device=dev)
            fn = lambda: synths[first].synth(bits_dev[first][:n_prof], nib.KEEP_MUL, dtype=torch.bfloat16, layout="nhwc",
                                             c_stride=cs, pad=pad, out=buf)
            fn(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 20
            e0.record()
            for _ in range(reps):
                fn()
            e1.record(); torch.cuda.synchronize()
            us = e0.elapsed_time(e1) / reps * 1e3
            gbs = MASK_BYTES_PER_EVAL * n_prof / (us * 1e-6) / 1e9
            roofline_mask = {"bound": "hbm", "kernel": "mask_synth_kernel (+ halo_zero_kernel on a caller-owned buffer)",
                             "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                             "us_per_launch": us, "masks_per_launch": n_prof,
                             "algorithmic_bytes_per_mask": MASK_BYTES_PER_EVAL,
                             "written_bytes_per_mask": (224 + 2 * pad) ** 2 * cs * 2,
                             "achieved_on_written_bytes": (224 + 2 * pad) ** 2 * cs * 2 * n_prof / (us * 1e-6) / 1e9,
                             "traffic": None}

    library_bar = None
    if rank == 0 and world == 1 and not args.no_library_bar:
        library_bar = library_forward_bar(torch, synthetic, arch, n_prof, dev)

    gp_info = None
    if rank == 0 and not args.no_gp:
        gp_info = gp_bench(nib, torch, np, args.gp_n, S)

    cpu = cpu_gp = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(arch)
        if not args.no_gp:
            cpu_gp = cpu_gp_baseline(np, S)

    if rank == 0:
        steps = args.steps
        near = (ties1.get("near_ties", 0) - ties0.get("near_ties", 0)) / steps
        over = (ties1.get("overflow", 0) - ties0.get("overflow", 0)) / steps
        if n_img > 1:
            workload = (f"{arch} 224^2 sweep: {n_img} synthetic images x {per_image} keep-masks each (S=50, k=20), flattened "
                        f"(image, mask) index space sharded over {world} ranks; mask synthesis + forward + scoring + tie policy + all-gather")
        else:
            workload = (f"generate_gp_training_data_imagenet.py: {arch} 224^2, S=50 superpixels, k=20 keep-masks, mask synthesis + "
                        "forward + top-1/softmax scoring + fp32 re-score of near-ties + score all-gather")
        line = {
            "metric": metric_name(arch), "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": args.warmup,
            "ms_per_step": ms / steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": args.precision, "data": "synthetic",
            "config": {"workload": workload, "arch": arch, "masks_per_step_per_gpu": per, "masks_per_step_total": total,
                       "images": n_img, "micro_batch": mb, "streams": args.streams,
                       "refine_ties": eng.refine_ties, "tie_capacity": eng.tie_capacity if eng.refine_ties is not None else None,
                       "tie_window": eng.tie_window if eng.refine_ties is not None else None,
                       "fused_expand_reduce": os.environ.get("NIB_TC_FUSE", "1") != "0", "sharding": f"masks over {world} ranks",
                       "allgather": "nib_allgather_scores (NCCL from the C ABI)" if world > 1 else None,
                       "weights": "random init, seeded (no network for pretrained weights)", "cuda_graph": bool(args.graph),
                       "l2": "no explicit flush: each step streams > 10 GB of activations through the 126 MB L2"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": ms_e2e / steps},
            "gpu_launches": int(gpu_launches), "tcgen05_launches": int(t1 - t0),
            "near_ties_per_step": near, "refined_per_step": near - over, "tie_overflow_per_step": over,
            "clocks": clocks, "roofline": roofline, "roofline_mask_synth": roofline_mask,
            "tflops_effective": value / world * FLOPS_PER_EVAL[arch] / 1e12 if arch in FLOPS_PER_EVAL else None,
        }
        if allgather_us is not None:
            line["allgather_us"] = allgather_us
        if library_bar is not None:
            line["library_bar"] = library_bar
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if gp_info is not None:
            if cpu_gp is not None:
                gp_info["cpu_baseline"] = cpu_gp
            line["gp"] = gp_info
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def library_forward_bar(torch, synthetic, arch, n, dev):
    """torch eager (cuDNN / cuBLAS) forward of the same torchvision network, bf16 channels-last, same micro-batch, same
    GPU: the 'library bar' SURVEY.md §8(d) asks for.  A measurement only; nothing of it is on the product path."""
    try:
        m = synthetic.build_imagenet_model(arch).to(dev).to(torch.bfloat16).to(memory_format=torch.channels_last).eval()
        xb = torch.randn(n, 3, 224, 224, device=dev, dtype=torch.bfloat16).contiguous(memory_format=torch.channels_last)
        with torch.no_grad():
            for _ in range(3):
                m(xb)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 10
            e0.record()
            for _ in range(reps):
                m(xb)
            e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        del m, xb
        torch.cuda.empty_cache()
        return {"what": f"torch {torch.__version__} eager forward, bf16 channels_last, batch {n}, forward only (no mask synthesis, "
                        "no scoring)", "value": n / (ms / 1e3), "unit": UNIT, "ms_per_forward": ms,
                "tflops": n / (ms / 1e3) * FLOPS_PER_EVAL.get(arch, 0) / 1e12}
    except Exception as e:   # the bar is optional evidence; never let it break the bench line
        return {"unavailable": repr(e)[:200]}


def gp_bench(nib, torch, np, n, S):
    """GP fit + predict ms at fixed theta on n masks / n candidates (the second half of BASELINE's metric)."""
    rng = np.random.RandomState(0)
    sels = [list(rng.choice(S - 1, size=20, replace=False)) for _ in range(2 * n)]
    Z = nib.selection_bits(sels, S)
    y = rng.rand(n)
    gp = nib.GaussianProcessRegressor(alpha=1e-5, length_scale=3.0, optimizer=None, query_chunk=8192)
    gp.fit(Z[:n], y)
    gp.predict_device(Z[n:])
    torch.cuda.synchronize()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    e[0].record()
    gp.fit(Z[:n], y)
    e[1].record()
    mu, var, sd = gp.predict_device(Z[n:])
    nib.expected_improvement_device(mu, sd, float(y.max()), True)
    e[2].record()
    torch.cuda.synchronize()
    fit_ms, pred_ms = e[0].elapsed_time(e[1]), e[1].elapsed_time(e[2])
    del gp
    chol_flops = n ** 3 / 3
    trsm_flops = float(n) * n * n
    # fp64 peak: the library DGEMM (cuBLAS through torch.matmul) on this GPU in this run, next to the DMMA microbenchmark
    lib_peak = None
    try:
        k = 8192
        A = torch.randn(k, k, dtype=torch.float64, device="cuda")
        B = torch.randn(k, k, dtype=torch.float64, device="cuda")
        torch.matmul(A, B); torch.cuda.synchronize()
        best = 1e9
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch.matmul(A, B); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        lib_peak = 2.0 * k ** 3 / (best / 1e3) / 1e12
        del A, B
        torch.cuda.empty_cache()
    except Exception:
        pass
    micro_peak = 37.1   # mma.sync.m8n8k4.f64 chains measured on this pool's B200 (tools/microbench/fp64_peak.cu)
    fp64_peak = max(micro_peak, lib_peak or 0.0)
    return {"n": n, "m": n, "fit_ms": fit_ms, "predict_ei_ms": pred_ms, "fit_plus_predict_ms": fit_ms + pred_ms,
            "fp64_tflops_fit": chol_flops / (fit_ms / 1e3) / 1e12, "fp64_tflops_predict": trsm_flops / (pred_ms / 1e3) / 1e12,
            "roofline": {"bound": "fp64 tensor pipe (DMMA)", "peak": fp64_peak, "unit": "TFLOP/s",
                         "frac_fit": chol_flops / (fit_ms / 1e3) / 1e12 / fp64_peak,
                         "frac_predict": trsm_flops / (pred_ms / 1e3) / 1e12 / fp64_peak,
                         "peak_library_dgemm_8192": lib_peak, "peak_dmma_microbench": micro_peak,
                         "peak_source": "max(torch.matmul fp64 8192^3 in this run, tools/microbench/fp64_peak.cu DMMA 37.1 TFLOP/s)"},
            "note": "fixed theta (optimizer=None); n^3/3 (Cholesky) and m*n^2 (variance TRSM) flops; includes host upload of masks and y"}


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
