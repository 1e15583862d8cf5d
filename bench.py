#!/usr/bin/env python
"""bench.py - SSD multibox head path on B200: images/sec and fraction of the HBM roofline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload train|detect|stress] [--batch B] [--collective peer|nccl] [--no-others]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic head outputs:
  train  (default)  match + hard-negative-mined CE + L1 loss, forward AND gradients, SSD300 (8732 priors, 1-10 gt/image)
                    (BASELINE.json configs[1]/[3]; default batch 256 per GPU = north_star's target size)
  detect            decode + conf 0.01 threshold + per-class NMS + global top-200 (configs[2]; default batch 64,
                    `--batch 256` = north_star's target size)
  stress            configs[4]: SSD512-style 24 564 priors, 100 gt boxes per image, batch 128 per GPU - the match + loss
                    step is the timed step, the detect step of the same shape is reported next to it
Under torchrun (N > 1) every rank owns `--batch` images (weak scaling); the batch-global positive count and the loss
sums cross GPUs exactly as a sharded ssd() call needs them (Losses.py:182,197), and after the timed loop one extra
sharded step in which every rank feeds rank 0's shard is compared bit for bit with the single-GPU step of that shard
(`sharded_check`; a mismatch ends the run with a non-zero exit code).
Rank 0 prints ONE JSON line.  `--impl reference` times the reference's own CPU implementation (the unmodified
`Losses.ssd` / `Losses.inference` from oracle/_ref when it travelled with the tree, else the oracle port) on all host
cores, on a bounded sample of the same workload.
`--dump-outputs DIR` writes what the last timed step returned (losses and gradients, or the detections) as .npy files;
the inputs depend only on the arguments, so the dumps of two builds can be compared file by file.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch

L2_BYTES = 126 * 1024 * 1024
C = 21


def algo_bytes(P: int, what: str) -> int:
    """SURVEY.md 8(d): algorithmic bytes per image, fp32."""
    if what == "train":          # loc + conf in, dense grad_loc + grad_conf out
        return 2 * P * 25 * 4
    if what == "train_fwd":
        return P * 25 * 4
    return P * 25 * 4 + 200 * 28   # detect: loc + conf in, <= 200 x 28 B out


def ce_stream_bytes(P: int) -> int:
    """Dominant kernel alone (DESIGN.md 3.2): conf in (84 B/prior), CE (4) + class byte (1) + dense gradient background
    (100) out."""
    return P * (84 + 4 + 1 + 100)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def source_hash() -> str:
    """Hash of the kernel sources the shipped libssdhead.so was built from (profiles/traffic.json records the same)."""
    from objectdetection_ssd_b200 import build
    return build.source_hash()


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


class ClockSampler:
    """SM clock + throttle reasons through NVML while the timed region runs (polled every millisecond)."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._timed = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake": 0x80}
        while not self._stop.is_set():
            try:
                timed = self._timed.is_set()
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                timed = timed or self._timed.is_set()       # a sample that straddles the start still saw the load
                self.samples.append((timed, mhz))
                if timed:
                    for k, bit in names.items():
                        if r & bit:
                            self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.001)

    def start(self):
        if self.nv:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def timed(self, on: bool):
        (self._timed.set if on else self._timed.clear)()

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=1.0)
        timed = [m for t, m in self.samples if t]
        return {"sm_mhz": float(np.median(timed)) if timed else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples_in_timed_region": len(timed)}


DUMP_BYTES = 64_000_000 - 4096      # --dump-outputs: 64 MB in all, .npy headers included


def dump_sample(whole, per_image, seed=0):
    """Host copies of one step's outputs for --dump-outputs: float32 / float64 arrays (integers widened to float64,
    exactly).  The `per_image` tensors share their leading batch axis; when the dump would exceed DUMP_BYTES they all
    keep the same fixed, seeded subset of images, in batch order."""
    def host(t):
        return t.detach().cpu().numpy() if t.dtype.is_floating_point else t.detach().cpu().to(torch.float64).numpy()

    out = {k: host(t) for k, t in whole.items()}
    per_img = sum(t[0].numel() * (t.element_size() if t.dtype.is_floating_point else 8) for t in per_image.values())
    B = next(iter(per_image.values())).shape[0]
    keep = min(B, (DUMP_BYTES - sum(a.nbytes for a in out.values())) // per_img)
    idx = None
    if keep < B:
        idx = np.sort(np.random.default_rng(seed).choice(B, keep, replace=False))
    for k, t in per_image.items():
        out[k] = host(t if idx is None else t[torch.from_numpy(idx).to(t.device)])
    return out


def dump_outputs(path, outputs):
    os.makedirs(path, exist_ok=True)
    for k, a in outputs.items():
        np.save(os.path.join(path, k + ".npy"), a)
    print(f"bench.py: wrote {', '.join(f'{k}.npy {list(a.shape)}' for k, a in outputs.items())} to {path}", file=sys.stderr)


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


WORKLOADS = {
    # name: (prior spec, default batch per GPU, gt per image lo..hi, seed)
    "train": ("ssd300", 256, 1, 10, 1),
    "detect": ("ssd300", 64, 0, 0, 3),
    "stress": ("ssd512", 128, 100, 100, 4),
}


def prior_table(kind: str):
    from objectdetection_ssd_b200 import priors as PR
    return PR.make_priors(PR.SSD300_SPEC if kind == "ssd300" else PR.SSD512_SPEC)


def workload_config(args, world):
    kind, _, glo, ghi, _ = WORKLOADS[args.workload]
    P = 8732 if kind == "ssd300" else 24564
    l2 = "inputs rotate through >= 2 x 126 MB of distinct device buffers (larger than L2)"
    if args.workload == "detect":
        return {"workload": "SSD300 inference post-processing: decode + conf 0.01 threshold + per-class NMS (iou 0.45) + "
                            "global top-200; background-logit bias +6 (~1.1k candidates/class)",
                "batch_per_gpu": args.batch, "global_batch": args.batch * world, "num_priors": P, "num_classes": C,
                "parallelism": f"image-sharded x{world}, no collective", "l2": l2}
    name = ("SSD300-VGG16 VOC head, 8732 priors, 21 classes: match + hard-negative-mined CE + L1 loss, forward and "
            "gradients (north_star target size: batch 256 per GPU)" if args.workload == "train" else
            "stress (BASELINE.json configs[4]): SSD512-style 24 564 priors, 100 gt boxes per image, 21 classes: match + "
            "hard-negative-mined CE + L1 loss, forward and gradients; decode + NMS of the same shape reported in `stress_detect`")
    coll = getattr(args, "collective", "peer")
    par = "single GPU" if world == 1 else (
        f"image-sharded x{world}; Npos and the loss sums cross GPUs " +
        ("through NVLink peer-memory stores inside the mining kernel (--collective peer)" if coll == "peer"
         else "through two NCCL all-reduces (--collective nccl)"))
    return {"workload": name, "batch_per_gpu": args.batch, "global_batch": args.batch * world, "num_priors": P,
            "num_classes": C, "gt_per_image": f"U{{{glo}..{ghi}}}" if glo != ghi else str(glo), "parallelism": par, "l2": l2}


def metric_name(workload):
    if workload == "detect":
        return "images/sec, SSD300 decode + NMS (conf 0.01, top-200)"
    if workload == "stress":
        return "images/sec, SSD512-style (24 564 priors, 100 gt/image) match + multibox loss fwd+bwd"
    return "images/sec, SSD300 match + multibox loss fwd+bwd"


# ----------------------------------------------------------------------------------------------- reference arm
def reference_inputs(workload, B):
    from objectdetection_ssd_b200 import synth
    kind, _, glo, ghi, seed = WORKLOADS[workload]
    P = 8732 if kind == "ssd300" else 24564
    if workload in ("train", "stress"):
        gb, gc = synth.make_gt(seed, B, glo, ghi)
        loc, conf = synth.make_head(seed, B, P)
        return (torch.from_numpy(loc), torch.from_numpy(conf), [torch.from_numpy(b) for b in gb],
                [torch.from_numpy(c) for c in gc])
    loc, conf = synth.make_head(seed, B, P, loc_scale=0.5, bg_bias=6.0)
    return torch.from_numpy(loc), torch.from_numpy(conf)


class ReferenceImpl:
    """The reference's CPU implementation of the path: the UNMODIFIED Losses.ssd / Losses.inference when the reference
    sources are importable (oracle/ref_import: $SSD_REFERENCE_DIR or oracle/_ref), else the oracle's port of them
    (torch-CPU ops, same algorithm)."""

    def __init__(self, workload):
        from oracle import ssd_oracle as O
        from oracle import ref_import
        self.O, self.workload = O, workload
        kind = WORKLOADS[workload][0]
        self.pri = O.make_priors() if kind == "ssd300" else O.make_priors(**O.SSD512)
        self.pxy = O.cxcywh_to_xyxy(self.pri)
        self.kind, self.R = "port", None
        if ref_import.available() and os.environ.get("SSD_BENCH_REFERENCE", "1") != "0":
            try:
                self.R = ref_import.load()
                self.ref_import = ref_import
                self.kind = "reference"
            except Exception as e:                              # noqa: BLE001 - fall back to the port, say so
                print(f"bench.py: unmodified reference not importable ({e}); timing the oracle port", file=sys.stderr)

    def step(self, data):
        if self.workload in ("train", "stress"):
            loc, conf, tb, tc = data
            l = loc.clone().requires_grad_(True)
            c = conf.clone().requires_grad_(True)
            if self.R is not None:
                _, RL = self.R
                with self.ref_import.quiet(), self._priors(RL):
                    a, b = RL.ssd((l, c), tc, tb)
                    (a + b).backward()
            else:
                a, b = self.O.ssd_reference_style((l, c), tc, tb, self.pri, self.pxy)
                (a + b).backward()
            return a.item() + b.item()
        loc, conf = data
        n = 0
        for i in range(loc.shape[0]):
            if self.R is not None:
                _, RL = self.R
                with self.ref_import.quiet(), self._priors(RL):
                    out = RL.inference(loc[i], conf[i], 0, top_k=200, toDraw=False, min_score=0.01, iou_threshold=0.45)
                n += len(out[0])
            else:
                n += self.O.detect_image(loc[i], conf[i], self.pri, 0.01, 0.45, 200)[0].shape[0]
        return n

    def _priors(self, RL):
        """The reference reads its module-global prior tables at call time: swap them only for the 24 564-prior shape."""
        import contextlib
        if WORKLOADS[self.workload][0] == "ssd300":
            return contextlib.nullcontext()
        return self.ref_import.priors(RL, self.pri)

    def describe(self, B):
        fn = {"train": "ssd() fwd+bwd", "stress": "ssd() fwd+bwd (24 564 priors, 100 gt/image)",
              "detect": "inference() looped over the images, bg bias +6, min_score 0.01"}[self.workload]
        who = "unmodified reference Losses." if self.kind == "reference" else "oracle port of Losses."
        return f"{who}{fn}, batch {B}"


def cpu_baseline(workload, budget_s=20.0):
    """Bounded CPU sample of the same workload (SURVEY.md 8(d) 'CPU baseline'), all host cores."""
    torch.set_num_threads(host_cores())
    impl = ReferenceImpl(workload)
    B = {"train": 32, "stress": 4, "detect": 1}[workload]
    data = reference_inputs(workload, B)
    t0 = time.perf_counter()
    impl.step(data)            # warm-up
    best = time.perf_counter() - t0
    reps = 0
    while reps < 3 and (time.perf_counter() - t0) + best < budget_s:
        t = time.perf_counter()
        impl.step(data)
        best = min(best, time.perf_counter() - t)
        reps += 1
    return {"value": B / best, "unit": "images/s", "cores": torch.get_num_threads(), "kind": impl.kind,
            "sample": f"{impl.describe(B)}; best of {reps + 1} runs, {best * 1e3:.1f} ms/pass"}


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    # rank 0 runs alone (the other ranks have exited): it may use every core this process is allowed on, whatever
    # OMP_NUM_THREADS torchrun exported
    torch.set_num_threads(host_cores())
    impl = ReferenceImpl(args.workload)
    # bounded sample: the full batch for the loss (the reference gets FASTER per image with the batch size), a few images
    # for its per-image detect loop and for the 24 564-prior / 100-gt stress shape
    B = {"train": args.batch, "stress": min(args.batch, 8), "detect": min(args.batch, 4)}[args.workload]
    data = reference_inputs(args.workload, B)
    warm = min(args.warmup, 1)
    for _ in range(warm):
        impl.step(data)
    steps = args.steps
    t0 = time.perf_counter()
    for _ in range(steps):
        impl.step(data)
    dt = (time.perf_counter() - t0) / steps
    val = B / dt
    sample = (f"{impl.describe(B)} per step (bounded sample of the {args.batch}-image workload), {steps} timed steps, "
              f"torch {torch.__version__} CPU ops, {torch.get_num_threads()} threads")
    line = {
        "impl": "reference", "metric": metric_name(args.workload),
        "value": val, "unit": "images/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": torch.get_num_threads(), "kind": impl.kind, "sample": sample},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- our arm
def max_over_ranks(ms, world, dev):
    if world == 1:
        return ms
    import torch.distributed as dist
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


class _DevPtrView:
    """Zero-copy torch view of device memory owned by the library (for the NCCL all-reduce)."""

    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


class LossRunner:
    """One rank's training-head step through the context's C entry points: single GPU, peer-memory sharded, or the
    NCCL route."""

    def __init__(self, pri, B, dev, world, rank, collective, max_total_gt):
        from objectdetection_ssd_b200.ctx import SSDHeadContext
        self.pri, self.B, self.dev, self.world, self.rank = pri, B, dev, world, rank
        self.P = int(pri.shape[0])
        self.max_total_gt = max_total_gt
        self.ctx = SSDHeadContext(pri.numpy(), max_batch=B, max_total_gt=max_total_gt, device=dev.index)
        self.collective = "none"
        self.npos_norm = torch.zeros(1, dtype=torch.int32, device=dev)
        if world > 1:
            import torch.distributed as dist
            self.collective = collective
            if collective == "peer" and B > 2 * torch.cuda.get_device_properties(dev).multi_processor_count:
                self.collective = "nccl"     # the in-kernel exchange needs one co-resident CTA per image (B <= 2 x SMs)
            if self.collective == "peer":
                # one-off: exchange the CUDA IPC handles of the ranks' exchange buffers; afterwards the step is the same
                # two kernels as on one GPU, the mining kernel trading Npos and the loss sums with its peers over NVLink
                handles = [None] * world
                dist.all_gather_object(handles, self.ctx.xchg_export())
                ok = torch.ones(1, dtype=torch.int32, device=dev)
                try:
                    self.ctx.xchg_import(handles, rank)
                except RuntimeError as e:                  # no peer access between these GPUs: every rank falls back
                    print(f"bench.py: rank {rank}: peer-memory import failed ({e}); using --collective nccl", file=sys.stderr)
                    ok.zero_()
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
                if int(ok.item()) == 0:
                    self.ctx.close()
                    self.ctx = SSDHeadContext(pri.numpy(), max_batch=B, max_total_gt=max_total_gt, device=dev.index)
                    self.collective = "nccl"
                dist.barrier()

    def step(self, l, c, tgx, tgc, toff, sumG, sums, losses, gl, gcf, st):
        ctx, B = self.ctx, self.B
        if self.world == 1 or self.collective == "peer":
            ctx.loss_dev(l.data_ptr(), c.data_ptr(), tgx.data_ptr(), tgc.data_ptr(), toff.data_ptr(), B, sumG,
                         sums.data_ptr(), losses.data_ptr(), gl.data_ptr(), gcf.data_ptr(), st)
        else:
            import torch.distributed as dist
            p = ctx.loss_begin(c.data_ptr(), tgx.data_ptr(), tgc.data_ptr(), toff.data_ptr(), B, sumG,
                               gl.data_ptr(), gcf.data_ptr(), st)
            self.npos_norm.copy_(torch.as_tensor(_DevPtrView(p, 1, "<i4"), device=self.dev))
            dist.all_reduce(self.npos_norm)
            ctx.loss_end(l.data_ptr(), c.data_ptr(), tgx.data_ptr(), tgc.data_ptr(), toff.data_ptr(), B,
                         self.npos_norm.data_ptr(), sums.data_ptr(), losses.data_ptr(), gl.data_ptr(), gcf.data_ptr(), st)
            dist.all_reduce(sums)
            ctx.finish_loss(sums.data_ptr(), self.npos_norm.data_ptr(), losses.data_ptr(), st)

    def sharded_check(self, workload, st):
        """Every rank feeds RANK 0's shard: the global positive count is world x Npos_0, the global sums world x sums_0,
        so the global losses must equal the single-GPU losses of that shard BIT FOR BIT (world is a power of two: the
        scaling is exact) and every gradient element must be exactly 1/world of the single-GPU one.  The single-GPU
        step runs on a second context without the exchange."""
        from objectdetection_ssd_b200 import synth
        from objectdetection_ssd_b200.ctx import SSDHeadContext
        _, _, glo, ghi, seed = WORKLOADS[workload]
        B, P, dev, world = self.B, self.P, self.dev, self.world
        gb, gc = synth.make_gt(seed, B, glo, ghi)
        gx, gcl, off = synth.pack_gt(gb, gc)
        loc, conf = synth.make_head(seed, B, P)
        d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        tl, tc, tgx, tgc, toff = d(loc), d(conf), d(gx), d(gcl), d(off)
        sumG = int(off[-1])
        out = {}
        for name in ("sharded", "single"):
            sums = torch.zeros(2, dtype=torch.float64, device=dev)
            losses = torch.zeros(2, device=dev)
            gl, gcf = torch.zeros_like(tl), torch.zeros_like(tc)
            if name == "sharded":
                for _ in range(2):                             # twice: both parities of the exchange slots
                    self.step(tl, tc, tgx, tgc, toff, sumG, sums, losses, gl, gcf, st)
            else:
                one = SSDHeadContext(self.pri.numpy(), max_batch=B, max_total_gt=self.max_total_gt, device=dev.index)
                one.loss_dev(tl.data_ptr(), tc.data_ptr(), tgx.data_ptr(), tgc.data_ptr(), toff.data_ptr(), B, sumG,
                             sums.data_ptr(), losses.data_ptr(), gl.data_ptr(), gcf.data_ptr(), st)
                torch.cuda.synchronize()
                one.close()
            torch.cuda.synchronize()
            out[name] = (sums, losses, gl, gcf)
        (ss, sl, sgl, sgc), (os_, ol, ogl, ogc) = out["sharded"], out["single"]
        pow2 = world & (world - 1) == 0
        ok_loss = bool(torch.equal(sl, ol)) if pow2 else bool(torch.allclose(sl, ol, rtol=1e-6))
        ok_sums = bool(torch.allclose(ss, os_ * world, rtol=1e-14, atol=0))
        ok_grad = bool(torch.equal(sgl * world, ogl) and torch.equal(sgc * world, ogc)) if pow2 else \
            bool(torch.allclose(sgl * world, ogl, rtol=1e-6) and torch.allclose(sgc * world, ogc, rtol=1e-6))
        ok = ok_loss and ok_sums and ok_grad and not (self.collective == "peer" and self.ctx.xchg_error())
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
        import torch.distributed as dist
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        return {"ok": bool(int(flag.item())), "this_rank_ok": ok, "loss": sl.tolist(), "expect": ol.tolist(),
                "grad_rows_checked": int((ogc != 0).any(-1).sum()), "collective": self.collective,
                "what": f"every rank fed rank 0's shard: global losses == single-GPU losses bit for bit, "
                        f"gradients x {world} == single-GPU gradients bit for bit, sums x {world} to 1e-14"}

    def close(self):
        self.ctx.close()


def time_loss(args, rank, world, dev, sampler, workload, B, steps, warmup, kernel_alone=True, e2e=True, capture=False):
    """The training-head step (match + loss fwd + gradients) of `workload` ('train' or 'stress') at batch B per GPU.
    capture: r["outputs"] holds what the last timed step returned (see dump_outputs)."""
    from objectdetection_ssd_b200 import _lib, synth, priors as PR
    from objectdetection_ssd_b200.ctx import SparseRows, pinned_empty
    lib = _lib.load()
    kind, _, glo, ghi, seed = WORKLOADS[workload]
    pri = prior_table(kind)
    P = pri.shape[0]
    run = LossRunner(pri, B, dev, world, rank, getattr(args, "collective", "peer"), max(128 * B, ghi * B))
    ctx = run.ctx
    gb, gc = synth.make_gt(seed + rank, B, glo, ghi)
    gx, gcl, off = synth.pack_gt(gb, gc)
    loc, conf = synth.make_head(seed + rank, B, P)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    tgx, tgc, toff = d(gx), d(gcl), d(off)
    per_set = B * P * 25 * 4
    nset = max(2, -(-2 * L2_BYTES // per_set))
    sets = [(d(loc) + 0.001 * i, d(conf) + 0.001 * i) for i in range(nset)]
    sums = torch.empty(2, dtype=torch.float64, device=dev)
    losses = torch.empty(2, device=dev)
    gl, gcf = torch.empty_like(sets[0][0]), torch.empty_like(sets[0][1])
    stream = torch.cuda.current_stream(dev)
    st = stream.cuda_stream
    sumG = int(off[-1])

    def step(i):
        l, c = sets[i % nset]
        run.step(l, c, tgx, tgc, toff, sumG, sums, losses, gl, gcf, st)

    for i in range(warmup):
        step(i)
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = _lib.launch_count()
    sampler.timed(True)
    e0.record(stream)
    for i in range(steps):
        step(i)
    e1.record(stream)
    barrier(world)
    sampler.timed(False)
    launches = _lib.launch_count() - n0
    ms = max_over_ranks(e0.elapsed_time(e1), world, dev)
    if run.collective == "peer" and ctx.xchg_error():
        raise SystemExit("bench.py: a wait for a peer rank expired inside the sharded step (results invalid)")
    r = dict(ms_total=ms, launches=launches, P=P, algo=algo_bytes(P, "train"), collective=run.collective, kern_ms=None)
    if capture:
        r["outputs"] = dump_sample({"losses": losses, "loss_sums": sums}, {"grad_loc": gl, "grad_conf": gcf})
    # losses of set 0 (the data the end-to-end leg uses), for the e2e cross-check
    step(0)
    torch.cuda.synchronize()
    r["losses"] = losses.tolist()

    if world > 1:
        r["sharded_check"] = run.sharded_check(workload, st)

    if kernel_alone:
        # ---- the dominant kernel alone, CUDA events on its launch stream: the streaming CE kernel with the fused
        # natural match (ssdhead_ce_match_stream with run_finalizer = 0, on a scratch match workspace) ----
        ws = torch.zeros(int(lib.ssdhead_workspace_bytes(_lib.WS_LOSS, B, P, C, 0)) + 256, dtype=torch.uint8, device=dev)
        wm = torch.zeros(int(lib.ssdhead_workspace_bytes(_lib.WS_MATCH, B, P, C, sumG)) + 256, dtype=torch.uint8, device=dev)
        pri_xyxy = PR.cxcywh_to_xyxy_host(pri).to(dev)
        cls_u8 = torch.empty(B, P, dtype=torch.uint8, device=dev)
        bestp = torch.empty(max(sumG, 1), dtype=torch.int32, device=dev)
        npos_k = torch.empty(B + 1, dtype=torch.int32, device=dev)

        def kern(i):
            return lib.ssdhead_ce_match_stream(sets[i % nset][1].data_ptr(), tgx.data_ptr(), tgc.data_ptr(), toff.data_ptr(),
                                               pri_xyxy.data_ptr(), B, P, C, sumG, 0.5, None, gl.data_ptr(), gcf.data_ptr(),
                                               cls_u8.data_ptr(), bestp.data_ptr(), npos_k.data_ptr(),
                                               ws.data_ptr(), ws.numel(), wm.data_ptr(), wm.numel(), 0, st)

        kn = max(10, min(steps, 200))
        for i in range(3):
            _lib.check(kern(i), "ssdhead_ce_match_stream")
        torch.cuda.synchronize()
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record(stream)
        for i in range(kn):
            kern(i)
        k1.record(stream)
        torch.cuda.synchronize()
        r.update(kern_ms=k0.elapsed_time(k1) / kn, kernel="ce_stream_kernel<21,true,true>", kernel_bytes=ce_stream_bytes(P) * B)

    if e2e:
        # ---- end to end through the host-buffer C ABI: pinned host tensors in, losses + gradient ROWS back in host
        # memory (ssdhead_ctx_multibox_loss_host_sparse).  With N > 1 and the peer exchange it is the SHARDED loss: the
        # ranks call in lock step and the global normalisation crosses GPUs inside the call. ----
        hl, hc = pinned_empty(loc.shape), pinned_empty(conf.shape)
        hl[:] = loc
        hc[:] = conf
        cap = 1024 if workload == "train" else 8192
        rows = SparseRows(B, cap=cap)
        en = max(3, min(steps, 20))
        for _ in range(2):
            e2e_loss = ctx.loss_host_sparse(hl, hc, gx, gcl, off, rows)
        barrier(world)
        t0 = time.perf_counter()
        for _ in range(en):
            e2e_loss = ctx.loss_host_sparse(hl, hc, gx, gcl, off, rows)
        torch.cuda.synchronize()
        e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / en, world, dev)
        if int(rows.cnt[:, 0].max()) > cap:
            raise SystemExit("bench.py: an image produced more gradient rows than the e2e row buffers hold")
        sharded_e2e = world > 1 and run.collective == "peer"
        # conf and gt are copied; loc is read in place from the page-locked host buffer, positive rows only (32-byte
        # sectors); the rows come back by direct stores into the page-locked row buffers
        h2d = conf.nbytes + gx.nbytes + gcl.nbytes + off.nbytes + int(rows.cnt[:, 1].sum()) * 32
        d2h = rows.nbytes_used() + 8
        want = r["losses"] if (world == 1 or sharded_e2e) else None
        chk = {"loss": list(e2e_loss), "device_step_loss": want, "copies_declared": True,
               "ok": None if want is None else bool(abs(e2e_loss[0] - want[0]) <= 1e-5 * abs(want[0]) and
                                                    abs(e2e_loss[1] - want[1]) <= 1e-5 * abs(want[1]))}
        # the dense variant (caller's [B,P,*] gradient tensors in host memory), for the record
        hgl, hgc = pinned_empty(loc.shape), pinned_empty(conf.shape)
        dn = max(2, min(steps, 5))
        ctx.loss_host(hl, hc, gx, gcl, off, hgl, hgc)
        barrier(world)
        t0 = time.perf_counter()
        for _ in range(dn):
            ctx.loss_host(hl, hc, gx, gcl, off, hgl, hgc)
        torch.cuda.synchronize()
        dense_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / dn, world, dev)
        r.update(e2e_ms=e2e_ms, h2d=h2d, d2h=d2h, e2e_steps=en, e2e_check=chk, e2e_dense_ms=dense_ms,
                 e2e_sharded=sharded_e2e)
        if chk["ok"] is False:
            raise SystemExit(f"bench.py: end-to-end losses {e2e_loss} differ from the device step's {want}")
    run.close()
    return r


def time_detect(args, rank, world, dev, sampler, B, steps, warmup, workload="detect", e2e=True, capture=False):
    from objectdetection_ssd_b200 import _lib, synth
    from objectdetection_ssd_b200.head import MultiboxHead
    from objectdetection_ssd_b200.ctx import SSDHeadContext, pinned_empty
    kind = WORKLOADS[workload][0]
    pri = prior_table(kind)
    P = pri.shape[0]
    head = MultiboxHead(pri, dev)
    loc, conf = synth.make_head(3 + rank, B, P, loc_scale=0.5, bg_bias=6.0)
    per_set = B * P * 25 * 4
    nset = max(2, -(-2 * L2_BYTES // per_set))
    sets = [(torch.from_numpy(loc).to(dev) + 1e-4 * i, torch.from_numpy(conf).to(dev)) for i in range(nset)]
    stream = torch.cuda.current_stream(dev)
    st = stream.cuda_stream
    lib = _lib.load()
    top_k = 200
    out = dict(boxes=torch.empty(B, top_k, 4, device=dev), prob=torch.empty(B, top_k, device=dev),
               cls=torch.empty(B, top_k, dtype=torch.int32, device=dev),
               prior=torch.empty(B, top_k, dtype=torch.int32, device=dev),
               cnt=torch.empty(B, dtype=torch.int32, device=dev))
    ws = torch.zeros(int(lib.ssdhead_workspace_bytes(_lib.WS_DETECT, B, P, C, 0)) + 256, dtype=torch.uint8, device=dev)
    pri_dev = head.pri_cxcywh

    def step(i):
        # the C ABI directly (what objectdetection_ssd_b200.head.detect calls after allocating its outputs)
        l, c = sets[i % nset]
        return lib.ssdhead_detect(l.data_ptr(), c.data_ptr(), pri_dev.data_ptr(), B, P, C, 0.01, 0.45, top_k, None, 0,
                                  out["boxes"].data_ptr(), out["prob"].data_ptr(), out["cls"].data_ptr(),
                                  out["prior"].data_ptr(), out["cnt"].data_ptr(), ws.data_ptr(), ws.numel(), st)

    for i in range(max(warmup, 1)):
        _lib.check(step(i), "ssdhead_detect")
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = _lib.launch_count()
    sampler.timed(True)
    e0.record(stream)
    for i in range(steps):
        step(i)
    e1.record(stream)
    barrier(world)
    sampler.timed(False)
    launches = _lib.launch_count() - n0
    ms = max_over_ranks(e0.elapsed_time(e1), world, dev)
    r = dict(ms_total=ms, launches=launches, kern_ms=None, B=B, steps=steps, P=P, algo=algo_bytes(P, "detect"),
             kernel="detect kernels (whole step)", detections=int(out["cnt"].clamp(min=0).sum()))
    if capture:
        # slots past an image's count hold whatever the buffers held before: zeroed, they are not part of the result
        valid = torch.arange(top_k, device=dev)[None, :] < out["cnt"][:, None]
        r["outputs"] = dump_sample({}, {"cnt": out["cnt"], "boxes": out["boxes"] * valid[..., None],
                                        **{k: out[k] * valid for k in ("prob", "cls", "prior")}})
    import ctypes
    nfb = ctypes.c_int32(-1)
    _lib.check(lib.ssdhead_detect_fallbacks(ws.data_ptr(), ws.numel(), B, P, C, 0, ctypes.addressof(nfb), st), "ssdhead_detect_fallbacks")
    env = os.environ.get("SSDHEAD_DETECT_SHORTLIST")
    shortlist = (int(env) != 0) if env else B * P >= 900000           # the library's own rule (csrc/detect.cu, shortlist_enabled)
    r["detect_route"] = {"route": "short list (sampled score floor; stream kernel + sweep kernel)" if shortlist
                         else "exhaustive (score kernel + sweep kernel)",
                         "images_listed_twice_in_last_step": int(nfb.value),
                         "note": "identical outputs on both routes; chosen by call size unless SSDHEAD_DETECT_SHORTLIST is set"}
    if e2e:
        # end to end: host buffers in, detections out
        ctx = SSDHeadContext(pri.numpy(), max_batch=B, device=dev.index)
        hl, hc = pinned_empty(loc.shape), pinned_empty(conf.shape)
        hl[:] = loc
        hc[:] = conf
        ob, op = pinned_empty((B, 200, 4)), pinned_empty((B, 200))
        oc, oi, on = pinned_empty((B, 200), np.int32), pinned_empty((B, 200), np.int32), pinned_empty((B,), np.int32)
        for _ in range(2):
            ctx.detect_host(hl, hc, ob, op, oc, oi, on, 0.01, 0.45)
        en = max(3, min(steps, 20))
        barrier(world)
        t0 = time.perf_counter()
        for _ in range(en):
            ctx.detect_host(hl, hc, ob, op, oc, oi, on, 0.01, 0.45)
        e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / en, world, dev)
        ctx.close()
        # conf is copied; of loc only the rows of the candidates the sweep visits cross PCIe (the kernel reads the
        # page-locked host buffer in place): counted as 512 rows of 32-byte sectors per image, an upper bound here
        r.update(e2e_ms=e2e_ms, h2d=conf.nbytes + B * 512 * 32,
                 d2h=ob.nbytes + op.nbytes + oc.nbytes + oi.nbytes + on.nbytes, e2e_steps=en,
                 e2e_check={"detections_per_image": float(np.clip(on, 0, None).mean()), "copies_declared": True,
                            "ok": bool((on >= 0).all() and (on <= 200).all())})
    return r


def time_train_levels(rank, dev, B=256, steps=200):
    """Training-head step on the six per-level tensors (NHWC conv outputs viewed as rows) instead of the concatenated
    [B,8732,*] pair - SURVEY.md 8(f) #3 - next to what building that pair costs (the torch.cat of Model.py:234-235)."""
    import ctypes
    from objectdetection_ssd_b200 import _lib, synth
    from objectdetection_ssd_b200.head import MultiboxHead, PackedGT
    lib = _lib.load()
    pri = prior_table("ssd300")
    P = pri.shape[0]
    head = MultiboxHead(pri, dev)
    gb, gc = synth.make_gt(1 + rank, B)
    gt = PackedGT([torch.from_numpy(b) for b in gb], [torch.from_numpy(c) for c in gc], head.dev)
    loc, conf = synth.make_head(1 + rank, B, P)
    counts = (5776, 2166, 600, 150, 36, 4)
    nset = max(2, -(-2 * L2_BYTES // (B * P * 25 * 4)))
    sets, structs = [], []
    for i in range(nset):
        l, c = torch.from_numpy(loc).to(dev) + 0.001 * i, torch.from_numpy(conf).to(dev) + 0.001 * i
        ls, cs, s0 = [], [], 0
        for n in counts:
            ls.append(l[:, s0:s0 + n].contiguous())
            cs.append(c[:, s0:s0 + n].contiguous())
            s0 += n
        sets.append((ls, cs))
    gls = [torch.empty_like(t) for t in sets[0][0]]
    gcs = [torch.empty_like(t) for t in sets[0][1]]
    for ls, cs in sets:
        st_ = _lib.Levels()
        st_.num_levels = len(counts)
        for i in range(len(counts)):
            st_.count[i] = counts[i]
            st_.conf[i], st_.loc[i] = cs[i].data_ptr(), ls[i].data_ptr()
            st_.grad_conf[i], st_.grad_loc[i] = gcs[i].data_ptr(), gls[i].data_ptr()
        structs.append(st_)
    sums = torch.empty(2, dtype=torch.float64, device=dev)
    losses = torch.empty(2, device=dev)
    m = head._match_outputs(gt, False)
    ws = head._workspace(_lib.WS_LOSS, B, 0)
    wm = head._workspace(_lib.WS_MATCH, B, gt.sumG)
    stream = torch.cuda.current_stream(dev)
    st = stream.cuda_stream

    def step(i):
        return lib.ssdhead_multibox_step_levels(
            ctypes.addressof(structs[i % nset]), gt.boxes.data_ptr(), gt.classes.data_ptr(), gt.off.data_ptr(),
            head.pri_xyxy.data_ptr(), head.pri_cxcywh.data_ptr(), B, P, C, gt.sumG, 3, 0.5, sums.data_ptr(), losses.data_ptr(),
            m["cls_u8"].data_ptr(), m["best_prior"].data_ptr(), m["npos"].data_ptr(),
            ws.data_ptr(), ws.numel(), wm.data_ptr(), wm.numel(), st)

    def cat(i):
        ls, cs = sets[i % nset]
        return torch.cat(ls, 1), torch.cat(cs, 1)

    def timeit(f):
        for i in range(5):
            f(i)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(steps):
            f(i)
        e1.record(stream)
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / steps

    _lib.check(step(0), "ssdhead_multibox_step_levels")
    return dict(ms_step=timeit(step), ms_cat=timeit(cat), losses=losses.tolist())


def time_dropin(dev, B, steps=100, host_lists=False):
    """The call a user of the reference makes (train_function.py:82-94): ``Losses.ssd((loc, conf), classes, bboxes)``
    with ragged gt LISTS and autograd-tracked outputs, then ``(loss1 + loss2).backward()`` - gt packing, output
    allocation, the autograd node and the gradient hand-over included.  Device-timed (CUDA events) and wall-clock
    (the Python surface can be launch-bound)."""
    from objectdetection_ssd_b200 import Losses, synth
    pri = prior_table("ssd300")
    P = pri.shape[0]
    gb, gc = synth.make_gt(1, B)
    loc, conf = synth.make_head(1, B, P)
    to = (lambda a: torch.from_numpy(a)) if host_lists else (lambda a: torch.from_numpy(a).to(dev))
    classes, bboxes = [to(c) for c in gc], [to(b) for b in gb]
    nset = max(2, -(-2 * L2_BYTES // (B * P * 25 * 4)))
    sets = [((torch.from_numpy(loc).to(dev) + 0.001 * i).requires_grad_(True),
             (torch.from_numpy(conf).to(dev) + 0.001 * i).requires_grad_(True)) for i in range(nset)]
    stream = torch.cuda.current_stream(dev)

    def it(i):
        l, c = sets[i % nset]
        l.grad = None
        c.grad = None
        l1, l2 = Losses.ssd((l, c), classes, bboxes)
        (l1 + l2).backward()
        return l1, l2

    for i in range(5):
        l1, l2 = it(i)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(stream)
    for i in range(steps):
        l1, l2 = it(i)
    e1.record(stream)
    torch.cuda.synchronize(dev)
    wall = (time.perf_counter() - t0) * 1e3 / steps
    return dict(ms_device=e0.elapsed_time(e1) / steps, ms_wall=wall, losses=[l1.item(), l2.item()])


def run_ours(args):
    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the SSD head path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    peak, peak_src = peaks()
    sampler = ClockSampler(local)
    sampler.start()
    B = args.batch
    capture = bool(args.dump_outputs) and rank == 0
    if args.workload == "detect":
        r = time_detect(args, rank, world, dev, sampler, B, args.steps, args.warmup, capture=capture)
    else:
        r = time_loss(args, rank, world, dev, sampler, args.workload, B, args.steps, args.warmup, capture=capture)
        args.collective = r["collective"] if world > 1 else args.collective       # what actually ran
    if capture:
        dump_outputs(args.dump_outputs, r.pop("outputs"))
    clocks = sampler.stop()
    ms_step = r["ms_total"] / args.steps
    value = B * world / (ms_step * 1e-3)
    e2e_val = B * world / (r["e2e_ms"] * 1e-3)
    step_gbs = r["algo"] * B / (ms_step * 1e-3) / 1e9
    is_loss = args.workload != "detect"
    line = {
        "metric": metric_name(args.workload),
        "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(args, world),
        "clocks": clocks,
        "e2e": {"value": e2e_val, "unit": "images/s", "h2d_bytes_per_step": int(r["h2d"]), "d2h_bytes_per_step": int(r["d2h"]),
                "ms_per_step": r["e2e_ms"], "steps": r["e2e_steps"],
                "api": "ssdhead_ctx_multibox_loss_host_sparse" if is_loss else "ssdhead_ctx_detect_host",
                "check": r.get("e2e_check"),
                "note": ("pinned host buffers in; losses + the gradient ROWS (positives and mined negatives: the only rows "
                         "of the dense gradient that are not zero) back in pinned host buffers: conf is copied, loc is read in "
                         "place (positive rows only), the mining kernel stores its ~4 Npos rows per image straight into the "
                         "host row buffers; "
                         + ("the ranks call in lock step and the loss is the SHARDED one (global normalisation through the "
                            "peer exchange)" if r.get("e2e_sharded") else
                            ("per-rank call" + (", local normalisation (NCCL route: no exchange inside the C call)" if world > 1 else "")))
                         if is_loss else
                         "pinned host buffers in, detections back to host: conf is copied, loc is read in place (visited "
                         "candidates only); per-rank call, no collective")},
        "gpu_launches": int(r["launches"]),
        "step_roofline": {"bound": "hbm", "achieved": step_gbs, "peak": peak, "unit": "GB/s", "frac": step_gbs / peak,
                          "algorithmic_bytes_per_image": r["algo"], "peak_source": peak_src,
                          "note": "whole step (all kernels of the step) against SURVEY.md 8(d) bytes/image"},
    }
    if is_loss and "e2e_dense_ms" in r:
        line["e2e"]["dense_gradient_tensors"] = {
            "api": "ssdhead_ctx_multibox_loss_host", "value": B * world / (r["e2e_dense_ms"] * 1e-3), "ms_per_step": r["e2e_dense_ms"],
            "note": "the caller's dense [B,P,*] gradient tensors in host memory: host threads zero them while the inputs "
                    "stream in, the mining kernel stores its rows into them"}
    if r["kern_ms"] is not None:
        ach = r["kernel_bytes"] / (r["kern_ms"] * 1e-3) / 1e9
        traffic, tnote = None, None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            with open(tp) as f:
                tj = json.load(f)
            ent = tj.get(f"ce_stream_b{B}" if args.workload == "train" else f"ce_stream_{args.workload}_b{B}")
            if ent:
                if tj.get("source_hash") == source_hash():
                    traffic = ent["dram_bytes_per_launch"]
                else:
                    tnote = ("profiles/traffic.json was captured from other kernel sources than this libssdhead.so "
                             "(source hash differs): not quoted")
        line["roofline"] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                            "traffic": traffic, "kernel": r["kernel"], "kernel_us": r["kern_ms"] * 1e3,
                            "algorithmic_bytes_per_launch": r["kernel_bytes"], "peak_source": peak_src}
        if tnote:
            line["roofline"]["traffic_note"] = tnote
    else:
        line["roofline"] = {"bound": "hbm", "achieved": step_gbs, "peak": peak, "unit": "GB/s", "frac": step_gbs / peak,
                            "traffic": None, "kernel": r["kernel"],
                            "note": "whole step: algorithmic bytes of the step / step time", "peak_source": peak_src}
    if "detect_route" in r:
        line["detect_route"] = r["detect_route"]
    if "losses" in r:
        line["loss"] = r["losses"]
    if "sharded_check" in r:
        line["sharded_check"] = r["sharded_check"]
    if args.workload == "stress":
        rd = time_detect(args, rank, world, dev, ClockSampler(local), B, max(5, min(args.steps, 50)), 3, workload="stress", e2e=False)
        md = rd["ms_total"] / rd["steps"]
        line["stress_detect"] = {"workload": "decode + conf 0.01 threshold + per-class NMS + top-200, 24 564 priors, bias +6",
                                 "images_per_s": B * world / (md * 1e-3), "ms_per_step": md,
                                 "step_roofline_frac": rd["algo"] * B / (md * 1e-3) / 1e9 / peak}
    if rank == 0 and world == 1:
        line["cpu_baseline"] = cpu_baseline(args.workload)
        if args.workload == "train" and not args.no_others:
            line["others"] = others(args, rank, dev, local, peak)
    elif rank == 0:
        line["cpu_baseline"] = None
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    if "sharded_check" in r and not r["sharded_check"]["ok"]:
        if rank == 0:
            print(json.dumps(line), flush=True)
        raise SystemExit("bench.py: sharded_check FAILED - the sharded step does not reproduce the single-GPU step")
    if rank == 0:
        print(json.dumps(line), flush=True)


def time_resident(dev, B=256, steps=200, warmup=10):
    """The training-head step with RESIDENT gradient tensors (ssdhead_ctx_multibox_loss_dev_resident): the same
    grad_loc / grad_conf from step to step, every step retracts the previous step's rows and writes its own, no dense
    zero background is written.  Inputs rotate through >= 2 x 126 MB of distinct device buffers."""
    from objectdetection_ssd_b200 import synth
    from objectdetection_ssd_b200.ctx import SSDHeadContext
    from objectdetection_ssd_b200.priors import make_priors
    pri = make_priors()
    P = int(pri.shape[0])
    ctx = SSDHeadContext(pri.numpy(), max_batch=B, device=dev.index)
    nset = max(2, int(2 * 126e6 // (B * P * 25 * 4)) + 1)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    sets = []
    for i in range(nset):
        gb, gc = synth.make_gt(500 + i, B)
        loc, conf = synth.make_head(500 + i, B, P)
        gx, gcl, off = synth.pack_gt(gb, gc)
        sets.append((d(loc), d(conf), d(gx), d(gcl), d(off), int(off[-1])))
    gl = torch.empty(B, P, 4, device=dev)
    gcf = torch.empty(B, P, 21, device=dev)
    sums = torch.empty(2, dtype=torch.float64, device=dev)
    losses = torch.empty(2, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream

    def step(i, fresh=False):
        l, c, gx, gcl, off, sg = sets[i % nset]
        ctx.loss_dev_resident(l.data_ptr(), c.data_ptr(), gx.data_ptr(), gcl.data_ptr(), off.data_ptr(), B, sg,
                              sums.data_ptr(), losses.data_ptr(), gl.data_ptr(), gcf.data_ptr(), st, fresh=fresh)
    step(0, fresh=True)
    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    # the tensors must hold exactly the dense step's gradient of the LAST batch
    l, c, gx, gcl, off, sg = sets[(steps - 1) % nset]
    gl2, gc2 = torch.empty_like(gl), torch.empty_like(gcf)
    ctx.loss_dev(l.data_ptr(), c.data_ptr(), gx.data_ptr(), gcl.data_ptr(), off.data_ptr(), B, sg,
                 sums.data_ptr(), losses.data_ptr(), gl2.data_ptr(), gc2.data_ptr(), st)
    torch.cuda.synchronize()
    same = bool(torch.equal(gl, gl2) and torch.equal(gcf, gc2))
    ctx.close()
    return {"ms_step": ms, "equals_dense_step": same}


def others(args, rank, dev, local, peak):
    """The other single-GPU configurations of BASELINE.json and the reference-facing Python surface, short runs."""
    out = []
    a2 = argparse.Namespace(**vars(args))
    r2 = time_loss(a2, rank, 1, dev, ClockSampler(local), "train", 32, 200, 10, kernel_alone=False)
    m2 = r2["ms_total"] / 200
    out.append({"workload": "train head, batch 32 (configs[1])", "images_per_s": 32 / (m2 * 1e-3),
                "ms_per_step": m2, "step_roofline_frac": r2["algo"] * 32 / (m2 * 1e-3) / 1e9 / peak,
                "e2e_images_per_s": 32 / (r2["e2e_ms"] * 1e-3)})
    for b3, n3 in ((64, 100), (256, 50)):
        r3 = time_detect(args, rank, 1, dev, ClockSampler(local), b3, n3, 5)
        m3 = r3["ms_total"] / n3
        out.append({"workload": f"detect, batch {b3}, bias +6 (configs[2]" + (")" if b3 == 64 else ", north_star size)"),
                    "images_per_s": b3 / (m3 * 1e-3), "ms_per_step": m3,
                    "step_roofline_frac": r3["algo"] * b3 / (m3 * 1e-3) / 1e9 / peak,
                    "e2e_images_per_s": b3 / (r3["e2e_ms"] * 1e-3), "gpu_launches_per_step": r3["launches"] / n3})
    r4 = time_train_levels(rank, dev)
    out.append({"workload": "train head, batch 256, from the 6 per-level tensors (ssdhead_multibox_step_levels, "
                            "SURVEY 8(f) #3; no concatenated tensor in either direction)",
                "images_per_s": 256 / (r4["ms_step"] * 1e-3), "ms_per_step": r4["ms_step"],
                "step_roofline_frac": algo_bytes(8732, "train") * 256 / (r4["ms_step"] * 1e-3) / 1e9 / peak,
                "torch_cat_of_the_levels_ms": r4["ms_cat"],
                "note": "the concatenated layout pays value's step PLUS torch_cat_of_the_levels_ms (Model.py:234-235) "
                        "and the same again in backward"})
    r8 = time_resident(dev)
    out.append({"workload": "train head, batch 256, RESIDENT gradient tensors (ssdhead_ctx_multibox_loss_dev_resident: the "
                            "caller keeps grad_loc / grad_conf from step to step; every step retracts the previous step's "
                            "~4 Npos rows per image and writes its own - no dense zero background)",
                "images_per_s": 256 / (r8["ms_step"] * 1e-3), "ms_per_step": r8["ms_step"],
                "tensors_equal_the_dense_step_bit_for_bit": r8["equals_dense_step"],
                "note": "234 MB fewer HBM writes per step, yet only a few us faster: without the zero-fill the streaming kernel "
                        "is bound by its fused match + softmax instruction stream (~72 us, IPC 2.3 at 18 warps per SM), "
                        "just under the 78 us the dense step needs for its HBM traffic"})
    if not r8["equals_dense_step"]:
        raise SystemExit("bench.py: the resident gradient tensors differ from the dense step's")
    for b5, host in ((256, False), (256, True), (32, False)):
        r5 = time_dropin(dev, b5, steps=100, host_lists=host)
        out.append({"workload": f"drop-in surface: Losses.ssd((loc, conf), classes, bboxes) + (l1 + l2).backward(), batch {b5}, "
                                f"{'host' if host else 'device'} gt lists (train_function.py:62-63,82-94)",
                    "images_per_s": b5 / (max(r5["ms_device"], r5["ms_wall"]) * 1e-3), "ms_per_step_device": r5["ms_device"],
                    "ms_per_step_wall": r5["ms_wall"],
                    "note": "includes gt packing + upload, output allocation, the autograd node and scale_grads"})
    a6 = argparse.Namespace(**vars(args))
    a6.workload = "stress"
    r6 = time_loss(a6, rank, 1, dev, ClockSampler(local), "stress", 128, 30, 3, kernel_alone=False, e2e=False)
    m6 = r6["ms_total"] / 30
    r7 = time_detect(a6, rank, 1, dev, ClockSampler(local), 128, 30, 3, workload="stress", e2e=False)
    m7 = r7["ms_total"] / 30
    out.append({"workload": "stress (configs[4]): 24 564 priors, 100 gt/image, batch 128: match + loss fwd+bwd",
                "images_per_s": 128 / (m6 * 1e-3), "ms_per_step": m6,
                "step_roofline_frac": r6["algo"] * 128 / (m6 * 1e-3) / 1e9 / peak})
    out.append({"workload": "stress (configs[4]): 24 564 priors, batch 128: decode + NMS",
                "images_per_s": 128 / (m7 * 1e-3), "ms_per_step": m7,
                "step_roofline_frac": r7["algo"] * 128 / (m7 * 1e-3) / 1e9 / peak})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default 2000 train / detect, 200 stress, 5 for --impl reference)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="train", choices=["train", "detect", "stress"])
    ap.add_argument("--batch", type=int, default=None, help="images per GPU (default 256 train, 64 detect, 128 stress)")
    ap.add_argument("--no-others", action="store_true", help="skip the short secondary-configuration runs")
    ap.add_argument("--collective", default="peer", choices=["peer", "nccl"],
                    help="N > 1: how Npos and the loss sums cross GPUs - 'peer' = stores into peer memory over NVLink "
                         "from inside the mining kernel (2 kernels/step, no NCCL call), 'nccl' = two NCCL all-reduces "
                         "around the mining kernel (3 kernels/step)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32 / "
                         "float64, at most 64 MB; rank 0 only) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.batch is None:
        args.batch = WORKLOADS[args.workload][1]
    if args.steps is None:
        args.steps = 5 if args.impl == "reference" else (200 if args.workload == "stress" else 2000)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
