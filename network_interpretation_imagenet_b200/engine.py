"""The whole hot path behind one object: masks -> classifier -> scores (-> GP), sharded over ranks.

Replaces the body of the reference's hot loops (generate_gp_training_data_imagenet.py:221-266,
generate_gp_training_data_mnist.py:203-269, generate_gp_training_data_cifar.py:307-342,
bayesian_active_learning_imagenet.py:178-198): instead of one mask, one H2D copy, one batch-1 forward and
one device sync per iteration, all N masks of an image are synthesised and scored in micro-batches on the
device, and each rank of a torch.distributed job scores a contiguous slice of the masks (masks are
independent work units, SURVEY.md §8e); one all-gather of (target_prob, top1) per call is the only
collective (libnib's nib_allgather_scores on NCCL; torch.distributed on CPU/gloo for the host-logic tests).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from .classifier import Classifier
from .masks import KEEP_MUL, REMOVE_MINMAX, MaskSynth
from .scoring import score

# Relative top-2 margin, (top1 - runner-up) / max|logit|, below which a bf16-scored mask is re-scored in fp32.
#
# A bf16 arg-max differs from the fp32 one only if the error of the DIFFERENCE between the fp32 top-1 and some other logit
# exceeds that difference, so the band has to cover the largest such error among classes close enough to overtake.
# Flip study on the bench workload (tools/r02_diag2.py, profiles/r02_flip_study_resnet101.json: ResNet-101, 16384 masks,
# bf16 micro-batch 384 x 2 streams against the fp32 lowering): row-wise logit error <= 5.7e-3 of max|logit|; error of
# (top1 - j) over all 1000 classes <= 6.5e-3, over the classes within 2e-2 of the top-1 <= 4.1e-3; 9 of 16384 arg-maxes
# differ, all at bf16 margins <= 2.35e-3.  DenseNet-121 (profiles/r02_flip_study_densenet121.json, 8192 masks): near-class
# difference error <= 3.2e-3, 118 flips, all at margins <= 2.17e-3.  The default band sits above the numbers that matter
# (4.1e-3 / 3.2e-3, 2.35e-3 / 2.17e-3); it re-scores 2.7 % of the ResNet-101 workload's masks, 13 % of DenseNet-121's.  This is a measured bound, not a proof: north_star's 1e-2 logit tolerance taken
# literally (band 2e-2) would send 99.6 % of the masks of this near-tied random-init network to fp32.  Trained networks
# have top-2 margins far outside any of these bands and the policy costs them one empty launch sequence (~0.6 ms).
DEFAULT_TIE_BAND = 4.5e-3
# Arch-keyed bands (Classifier.arch) where a network's flip study puts the numbers above DEFAULT_TIE_BAND.
# torchvision VGG / AlexNet ("tv_plain"): flip study on the bench workload (tools/r02_diag2.py 16384 <arch>, bf16 at micro-batch
# 384 x 2 streams against the fp32 lowering; profiles/vgg_flip_study_vgg16.json, profiles/vgg_flip_study_vgg16_bn.json): error
# of (top1 - j) over the classes within 2e-2 of the top-1 <= 1.38e-2 (vgg16) / 1.15e-2 (vgg16_bn); 318 / 217 of 16384 arg-maxes
# differ, at bf16 margins <= 7.4e-3 / 8.8e-3; row-wise logit error <= 1.35e-2 / 1.12e-2.  The band sits above the
# near-class error and every flip margin; 17.8 % of vgg16's masks have a bf16 margin below 1.25e-2, 27.5 % below 2e-2.
TIE_BANDS = {"tv_plain": 1.5e-2}
DEFAULT_TIE_CAPACITY = 1024     # rows of the re-score buffer per window of masks
DEFAULT_TIE_WINDOW = 4096       # masks scored per tie-policy pass (capacity = 25 % of a window: the seeded DenseNet-121,
                                # the most tied of the networks here, has 13 % of its masks inside the band on average and
                                # overflowed a 640-row buffer in 24 of 4096 masks per window, profiles/r02_bench_final_n8_
                                # densenet_config5.json; the pass costs what its live rows cost, not what the buffer holds)


def shard_range(N: int, rank: int, world: int) -> tuple[int, int, int]:
    """Contiguous slice [lo, hi) of N masks for `rank`, and the padded per-rank length (equal on all ranks so a
    single all-gather works).  Mask order is global, so results are identical to a 1-GPU run."""
    per = (N + world - 1) // world
    lo = min(N, rank * per)
    hi = min(N, lo + per)
    return lo, hi, per


def gather_scores(local: torch.Tensor, N: int, group=None) -> torch.Tensor:
    """All-gather a [per, F] per-rank score block into the global [N, F] table through torch.distributed (works on
    gloo/CPU and nccl/CUDA).  The CUDA engine uses ScoreComm (libnib, NCCL from the C ABI) instead."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local[:N]
    world = dist.get_world_size(group)
    out = torch.empty((world * local.shape[0],) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, local.contiguous(), group=group)
    return out[:N]


class ScoreComm:
    """NCCL communicator owned by libnib (nib_comm_init / nib_allgather_scores).  The 128-byte unique id is created
    by rank 0 inside the library and broadcast over the existing torch.distributed group (bootstrap only); the
    all-gather itself is the C-ABI call on the caller's stream."""

    def __init__(self, group=None, device=None):
        self.lib = _lib.load()
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        ident = torch.zeros(128, dtype=torch.uint8)
        if self.rank == 0:
            buf = (C.c_ubyte * 128)()
            _lib.check(self.lib.nib_comm_unique_id(buf), "nib_comm_unique_id")
            ident = torch.frombuffer(bytearray(buf), dtype=torch.uint8).clone()
        backend = dist.get_backend(group)
        t = ident.to(device) if backend == "nccl" else ident
        dist.broadcast(t, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        raw = bytes(t.cpu().numpy().tobytes())
        h = C.c_void_p()
        _lib.check(self.lib.nib_comm_init(raw, self.rank, self.world, C.byref(h)), "nib_comm_init")
        self.h = h

    def allgather(self, local: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
        """local [per, 2] fp32 cuda -> out [world*per, 2] on the current stream."""
        per = int(local.shape[0])
        _lib.check(self.lib.nib_allgather_scores(self.h, local.data_ptr(), per, out.data_ptr(), _lib.stream_handle()),
                   "nib_allgather_scores")
        return out

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.nib_comm_destroy(self.h)
                self.h = None
        except Exception:
            pass


class PerturbationEngine:
    """refine_ties: relative top-2 margin (top1 - runner-up) / max|logit| below which a bf16-scored mask is re-scored by
    an fp32-grade copy of the classifier (`tie_precision`: "split" = the tcgen05 pair kernel over split-bf16 tensors,
    torchvision ResNets, VGGs and AlexNet; "x3" = fp32 activations with split-bf16 mma.sync products; both within ~3e-5 of the fp32
    lowering; "fp32" = the CUDA-core lowering itself; "auto" picks "split" where it applies, else "x3"), so that top-1
    equals the reference's on every mask outside numerical noise.
    "auto" (default) = TIE_BANDS[arch] (else DEFAULT_TIE_BAND) for bf16 classifiers lowered from a torch module, off otherwise; None/0 = off.
    The policy runs entirely on the device (no host synchronisation): near-tie rows are compacted into a buffer of
    `tie_capacity` rows (per window of `tie_window` masks), the fp32 network runs on that buffer with the device-side
    count as its live batch size, and the refined scores are scattered back.  `tie_stats()` reads the counters (near-ties
    found, rows refined, rows that did not fit: overflow > 0 means some near-ties kept their bf16 score)."""

    def __init__(self, model, image, segments, target: int, mode: int = KEEP_MUL, precision: str = "bf16",
                 max_batch: int = 128, S: int | None = None, device="cuda", group=None, use_graph: bool = False,
                 refine_ties="auto", streams: int = 1, tie_capacity: int = DEFAULT_TIE_CAPACITY,
                 tie_window: int = DEFAULT_TIE_WINDOW, tie_precision: str = "auto"):
        self.lib = _lib.load()
        self.device = torch.device(device)
        self.target = int(target)
        self.mode = mode
        self.group = group
        self.synth = MaskSynth(image, segments, S=S, device=device)
        self.classifier = model if isinstance(model, Classifier) else Classifier.from_torch(
            model, (self.synth.H, self.synth.W), precision=precision, max_batch=max_batch, streams=streams)
        self._model_src = None if isinstance(model, Classifier) else model
        if isinstance(refine_ties, str):
            if refine_ties != "auto":
                raise ValueError("refine_ties must be 'auto', None or a float")
            band = TIE_BANDS.get(self.classifier.arch, DEFAULT_TIE_BAND)
            refine_ties = band if (self.classifier.precision == "bf16" and self._model_src is not None) else None
        self.refine_ties = float(refine_ties) if (refine_ties and self.classifier.precision == "bf16") else None
        if self.refine_ties is not None and self._model_src is None:
            raise ValueError("refine_ties needs the torch module (to lower an fp32 copy), not a lowered Classifier")
        self.tie_capacity = int(tie_capacity)
        self.tie_window = max(1, int(tie_window))
        if tie_precision == "auto":
            # torchvision ResNets, VGGs and AlexNet (every body conv a multiple of 64 channels wide) re-score on the tcgen05
            # pair kernel over split-bf16 tensors; everything else on the mma.sync split-bf16 kernel over fp32 tensors
            tie_precision = "split" if self.classifier.arch in ("tv_resnet", "tv_plain") else "x3"
        if tie_precision not in ("split", "x3", "fp32"):
            raise ValueError("tie_precision must be 'auto', 'split' (split-bf16 tensors, tcgen05), 'x3' (split-bf16 products on "
                             "fp32 tensors, mma.sync) or 'fp32' (CUDA cores)")
        self.tie_precision = tie_precision
        self._fp32 = None
        self._tie = None
        self._calls = 0
        if use_graph:
            self.classifier.set_graph(True)
        self.rank = dist.get_rank(group) if dist.is_available() and dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self._comm = None
        self._bufs: dict = {}

    # -- tie policy ------------------------------------------------------------------------------------
    def _tie_state(self, n: int):
        """Buffers and the re-score lowering for a window of `n` masks: at most `tie_capacity` rows, but no larger than the
        window itself (a 16-mask call does not need a 640-image network); grown, never shrunk."""
        cap = min(self.tie_capacity, max(8, int(n)))
        if self._tie is not None and self._tie["cap"] >= cap:
            return self._tie
        totals = self._tie["totals"] if self._tie is not None else torch.zeros(2, dtype=torch.int64, device=self.device)
        if self._tie is not None:
            torch.cuda.current_stream().synchronize()       # the smaller lowering may still be running
        self._tie = self._fp32 = None
        dev = self.device
        f32 = Classifier.from_torch(self._model_src, (self.synth.H, self.synth.W), precision=self.tie_precision, max_batch=cap)
        t = {"cap": cap, "net": f32,
             "idx": torch.full((cap,), -1, dtype=torch.int32, device=dev),
             "sel": torch.zeros(cap, self.synth.words, dtype=torch.int64, device=dev),
             "count": torch.zeros(1, dtype=torch.int32, device=dev),
             "logits": torch.zeros(cap, f32.num_classes, dtype=torch.float32, device=dev),
             "totals": totals}   # (near-ties, did not fit), read by tie_stats()
        t["score"] = {"top1": torch.empty(cap, dtype=torch.int32, device=dev),
                      "target_prob": torch.empty(cap, dtype=torch.float32, device=dev),
                      "max_prob": torch.empty(cap, dtype=torch.float32, device=dev),
                      "correct": torch.empty(cap, dtype=torch.uint8, device=dev),
                      "margin": torch.empty(cap, dtype=torch.float32, device=dev)}
        _lib.check(self.lib.nib_net_set_dynamic_batch(f32.h, t["count"].data_ptr()), "nib_net_set_dynamic_batch")
        self._tie, self._fp32 = t, f32
        return t

    def _refine(self, d_sel: torch.Tensor, s: dict, table: torch.Tensor | None, synth: MaskSynth):
        """Device-side tie policy on the scores `s` of the rows `d_sel` (no host sync)."""
        n = int(d_sel.shape[0])
        t = self._tie_state(n)
        cap, f32 = t["cap"], t["net"]
        st = _lib.stream_handle()
        _lib.check(self.lib.nib_tie_compact(s["margin"].data_ptr(), n, self.refine_ties, d_sel.data_ptr(), self.synth.words,
                                            cap, t["idx"].data_ptr(), t["sel"].data_ptr(), t["count"].data_ptr(),
                                            t["totals"].data_ptr(), st), "nib_tie_compact")
        f32.forward_masked(synth, t["sel"], self.mode, out=t["logits"])
        score(t["logits"], self.target, out=t["score"])
        r = t["score"]
        _lib.check(self.lib.nib_tie_scatter(t["idx"].data_ptr(), t["count"].data_ptr(), cap, r["top1"].data_ptr(),
                                            r["target_prob"].data_ptr(), r["max_prob"].data_ptr(), r["correct"].data_ptr(),
                                            s["top1"].data_ptr(), s["target_prob"].data_ptr(), s["max_prob"].data_ptr(),
                                            s["correct"].data_ptr(), table.data_ptr() if table is not None else None, st),
                   "nib_tie_scatter")

    def tie_stats(self) -> dict:
        """Counters of the tie policy since construction (one host read)."""
        if self._tie is None:
            return {"band": self.refine_ties, "capacity": self.tie_capacity, "calls": self._calls, "near_ties": 0, "overflow": 0}
        found, over = (int(v) for v in self._tie["totals"].tolist())
        return {"band": self.refine_ties, "capacity": self.tie_capacity, "calls": self._calls, "near_ties": found,
                "refined": found - over, "overflow": over}

    @property
    def refined(self) -> int:
        st = self.tie_stats()
        return st.get("refined", 0)

    # -- scoring ---------------------------------------------------------------------------------------
    def _scratch(self, n: int) -> dict:
        b = self._bufs.get(n)
        if b is None:
            dev = self.device
            b = {"logits": torch.empty(n, self.classifier.num_classes, dtype=torch.float32, device=dev),
                 "top1": torch.empty(n, dtype=torch.int32, device=dev),
                 "target_prob": torch.empty(n, dtype=torch.float32, device=dev),
                 "max_prob": torch.empty(n, dtype=torch.float32, device=dev),
                 "correct": torch.empty(n, dtype=torch.uint8, device=dev),
                 "margin": torch.empty(n, dtype=torch.float32, device=dev)}
            if len(self._bufs) > 8:
                self._bufs.clear()
            self._bufs[n] = b
        return b

    def score_local(self, sel_bits, out: torch.Tensor | None = None, synth: MaskSynth | None = None):
        """Scores for the given selections on this rank only.  Returns [n, 2] fp32: (target_prob, top1).  No host
        synchronisation: mask synthesis, forward, scoring (which writes the table directly) and the tie policy are all
        queued on the current stream.  `synth`: another image + label map of the same geometry (sweeps over many
        images share one lowered classifier, BASELINE configs[4])."""
        synth = self.synth if synth is None else synth
        d_sel = synth.device_bits(sel_bits)
        n = int(d_sel.shape[0])
        if out is None:
            out = torch.zeros(n, 2, dtype=torch.float32, device=self.device)
        if n == 0:
            return out
        self._calls += 1
        # windows bound the number of near-ties one pass of the tie policy can meet (its buffer holds tie_capacity rows)
        win = self.tie_window if self.refine_ties is not None else n
        for w0 in range(0, n, win):
            w1 = min(n, w0 + win)
            b = self._scratch(w1 - w0)
            self.classifier.forward_masked(synth, d_sel[w0:w1], self.mode, out=b["logits"])
            s = score(b["logits"], self.target, out=b, table=out[w0:w1])
            if self.refine_ties is not None:
                self._refine(d_sel[w0:w1], s, out[w0:w1], synth)
        return out

    def gather(self, local: torch.Tensor, N: int, out: torch.Tensor | None = None) -> torch.Tensor:
        """Global [N, 2] table from the per-rank [per, 2] blocks."""
        if self.world == 1:
            return local[:N]
        if local.is_cuda and dist.get_backend(self.group) == "nccl":
            if self._comm is None:
                self._comm = ScoreComm(self.group, self.device)
            if out is None:
                out = torch.empty(self.world * local.shape[0], 2, dtype=torch.float32, device=local.device)
            return self._comm.allgather(local, out)[:N]
        return gather_scores(local, N, self.group)

    def score_masks(self, sel_bits) -> dict:
        """All N masks, sharded over the ranks of `group`; every rank returns the full tables."""
        bits = np.ascontiguousarray(sel_bits, dtype=np.uint64)
        N = bits.shape[0]
        lo, hi, per = shard_range(N, self.rank, self.world)
        local = torch.zeros(per, 2, dtype=torch.float32, device=self.device)
        self.score_local(bits[lo:hi], out=local)
        table = self.gather(local, N)
        top1 = table[:, 1].to(torch.int32)
        return {"target_prob": table[:, 0], "top1": top1, "correct": (top1 == self.target)}
