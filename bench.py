#!/usr/bin/env python
"""bench.py -- headline benchmark of the warp / filter engine (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one ``warp_perspective`` call on a synthetic B x 3 x 1080 x 1920 fp32 batch
(BASELINE.json configs[1]: bilinear, zeros padding, align_corners=True), B per GPU fixed (weak
scaling: the batch dimension shards with no data-path collective, SURVEY.md section 8e).

One JSON line on stdout (rank 0):
  value     Mpix/s, whole job, inputs resident in HBM, through the public Python API
            (prelude + kernel), CUDA events around exactly K steps, max over ranks
  roofline  the fused warp kernel alone: CUDA events around each launch inside the timed region,
            algorithmic bytes = 24 B/pixel (read 3 fp32 + write 3 fp32; DESIGN.md)
  e2e       same metric with HOST buffers: pinned src -> H2D -> kernel -> D2H of the full output,
            chunked and pipelined over three streams, copies inside the timed region
  cpu_baseline  the oracle's torch-op port of the reference composition on the host cores,
            bounded sample (rank 0, N=1 only)
``--impl reference`` times that CPU port alone (the reference is pure Python and cannot travel to
the GPU box; the port issues the same ATen calls: oracle/kornia_restated.py).
``--dump-outputs DIR`` writes what the last timed step returned as DIR/<name>.npy (see dump_outputs); the inputs
are generated from fixed seeds, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

H_IMG, W_IMG, C_IMG = 1080, 1920, 3
BYTES_PER_PIX = 24.0  # algorithmic: 3 channels x 4 B read + 3 x 4 B written per output pixel
METRIC = "Mpix/s warp_perspective Bx3x1080x1920 fwd bilinear fp32"


def headline_config(B: int, world: int) -> dict:
    """The `config` both arms print for the headline (BASELINE.json configs[1]); the reference arm times a per-step SAMPLE of this
    configuration (stated in its `cpu_baseline.sample`), the metric is per pixel."""
    return {"workload": f"warp_perspective fwd B={B}x3x1080x1920 per GPU, bilinear, zeros, align_corners=True (BASELINE.json configs[1])",
            "global_batch": B * world, "parallelism": f"batch-sharded x{world}, no data-path collective",
            "l2": "inputs (6.37 GB/GPU) exceed the 126 MB L2; no explicit flush",
            "homographies": "corner quad jittered by 8*randn px (benchmarks/geometry/flagship.py recipe), seed 1000+rank"}


# ------------------------------------------------------------------------------------------ inputs
def perspective_from_quads(src_q: torch.Tensor, dst_q: torch.Tensor) -> torch.Tensor:
    """DLT: the (B,3,3) homography mapping 4 source corners to 4 destination corners (what
    kornia.geometry.get_perspective_transform returns; used by the reference's flagship benchmark,
    benchmarks/geometry/flagship.py:101-107).  Solved in float64 on the host."""
    s, d = src_q.double(), dst_q.double()
    B = s.shape[0]
    A = torch.zeros(B, 8, 8, dtype=torch.float64)
    b = torch.zeros(B, 8, dtype=torch.float64)
    for i in range(4):
        x, y, u, v = s[:, i, 0], s[:, i, 1], d[:, i, 0], d[:, i, 1]
        A[:, 2 * i, 0], A[:, 2 * i, 1], A[:, 2 * i, 2] = x, y, 1.0
        A[:, 2 * i, 6], A[:, 2 * i, 7] = -u * x, -u * y
        A[:, 2 * i + 1, 3], A[:, 2 * i + 1, 4], A[:, 2 * i + 1, 5] = x, y, 1.0
        A[:, 2 * i + 1, 6], A[:, 2 * i + 1, 7] = -v * x, -v * y
        b[:, 2 * i], b[:, 2 * i + 1] = u, v
    hvec = torch.linalg.solve(A, b)
    return torch.cat([hvec, torch.ones(B, 1, dtype=torch.float64)], 1).view(B, 3, 3).float()


def make_homographies_hw(B: int, seed: int, Hh: int, Ww: int) -> torch.Tensor:
    g = torch.Generator().manual_seed(seed)
    quad = torch.tensor([[0.0, 0.0], [Ww - 1.0, 0.0], [Ww - 1.0, Hh - 1.0], [0.0, Hh - 1.0]]).expand(B, 4, 2)
    return perspective_from_quads(quad, quad + 8.0 * torch.randn(B, 4, 2, generator=g))


def make_homographies(B: int, seed: int) -> torch.Tensor:
    return make_homographies_hw(B, seed, H_IMG, W_IMG)


# ------------------------------------------------------------------------------------------ outputs
DUMP_BYTES = 60 * 10**6  # array data written by --dump-outputs; with the .npy headers the files stay under 64 MB


def dump_outputs(directory: str, arrays: dict) -> None:
    """Write what the timed path returned as ``directory/<name>.npy`` (float64 tensors as float64, all others as float32),
    so that two builds run with the same arguments can be compared output for output.  Arrays are taken smallest first and
    each may use an equal share of what is left of DUMP_BYTES: one that fits is written whole, a larger one as the elements
    at a fixed set of flat indices (drawn with seed 0, sorted; the same for every run with the same shape), flattened."""
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    left, todo = DUMP_BYTES, sorted(arrays.items(), key=lambda kv: kv[1].numel())
    for i, (name, t) in enumerate(todo):
        t = t.detach()
        t = t.double() if t.dtype == torch.float64 else t.float()
        share = left // (len(todo) - i)
        if t.numel() * t.element_size() <= share:
            a, note = t.cpu().numpy(), "whole"
        else:
            k = share // t.element_size()
            idx = torch.randint(t.numel(), (k,), generator=torch.Generator().manual_seed(0)).unique()
            a, note = t.reshape(-1)[idx.to(t.device)].cpu().numpy(), f"{idx.numel()} of {t.numel()} elements at seeded indices"
        np.save(os.path.join(directory, name + ".npy"), a)
        left -= a.nbytes
        print(f"bench.py: wrote {name}.npy {tuple(t.shape)} {a.dtype} ({note})", file=sys.stderr)


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons for one GPU while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        return False

    def hold_load(self, fn, sync, min_samples: int = 2, max_seconds: float = 1.0) -> int:
        """A timed region of a few tens of milliseconds can end before nvidia-smi's first 100 ms report.  Keep the very
        same load running -- untimed, after the stop event -- until a few samples exist, so that the clocks line
        describes the GPU under this load.  Returns the number of extra (untimed) steps."""
        self.extra = 0
        if self.proc is None:
            return 0
        deadline = time.time() + max_seconds
        try:
            while len(self.rows) < min_samples and time.time() < deadline:
                for _ in range(4):
                    fn()
                sync()
                self.extra += 4
        except Exception:
            pass
        return self.extra

    def summary(self):
        out = self._summary()
        out["untimed_steps_for_sampling"] = getattr(self, "extra", 0)
        return out

    def _summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ CPU port
def cpu_reference_run(steps: int, warmup: int, sample_b: int):
    """Time the oracle's torch-op port of the reference on the host cores.  The thread count that serves
    the reference best is picked by a one-shot calibration (ATen's CPU sampler parallelises over the batch,
    the elementwise ops over elements; 128 threads on an 8-image batch oversubscribe badly)."""
    from oracle import kornia_restated as R

    cores = os.cpu_count() or 1
    g = torch.Generator().manual_seed(0)
    src = torch.rand(sample_b, C_IMG, H_IMG, W_IMG, generator=g)
    M = make_homographies(sample_b, 0)

    def once():
        t0 = time.perf_counter()
        R.warp_perspective(src, M, (H_IMG, W_IMG))
        return time.perf_counter() - t0

    best_t, best_n = None, cores
    for n in sorted({cores, max(1, cores // 2), max(1, cores // 4), min(cores, sample_b)}, reverse=True):
        torch.set_num_threads(n)
        once()
        t = once()
        if best_t is None or t < best_t:
            best_t, best_n = t, n
    torch.set_num_threads(best_n)
    for _ in range(warmup):
        once()
    dt = sum(once() for _ in range(steps)) / steps
    mpix = sample_b * H_IMG * W_IMG / dt / 1e6
    return mpix, dt * 1e3, best_n


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample_b = 32
    mpix, ms, cores = cpu_reference_run(args.steps, max(args.warmup, 1), sample_b)
    line = {
        "impl": "reference", "metric": METRIC, "value": mpix, "unit": "Mpix/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": headline_config(args.batch, args.gpus),
        "cpu_baseline": {"value": mpix, "unit": "Mpix/s", "cores": cores, "kind": "port",
                         "sample": f"each step = B={sample_b}x3x1080x1920 of the configuration's batch (CPU per-image throughput is batch independent), torch CPU ops "
                                   f"(oracle/kornia_restated.py: the reference's ATen call sequence), {cores} of {os.cpu_count()} threads (best of a calibration)"},
        "e2e": {"value": mpix, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ side legs (untimed context)
def bandlimited(shape, dev, seed: int) -> torch.Tensor:
    """SURVEY 8d band-limited set: per (b,c) a sum of 6 sinusoids of <= 8 cycles per image with random phases, scaled to [0,1]."""
    B, C, Hh, Ww = shape
    g = torch.Generator().manual_seed(seed)
    fx = torch.randint(0, 9, (B, C, 6, 1, 1), generator=g).float().to(dev)
    fy = torch.randint(0, 9, (B, C, 6, 1, 1), generator=g).float().to(dev)
    ph = (torch.rand(B, C, 6, 1, 1, generator=g) * 2 * math.pi).to(dev)
    ys = torch.linspace(0, 1, Hh, device=dev).view(1, 1, 1, Hh, 1)
    xs = torch.linspace(0, 1, Ww, device=dev).view(1, 1, 1, 1, Ww)
    img = torch.sin(2 * math.pi * (fx * xs + fy * ys) + ph).sum(2)
    lo, hi = img.amin((2, 3), keepdim=True), img.amax((2, 3), keepdim=True)
    return (img - lo) / (hi - lo).clamp_min(1e-6)


def _rel(a: torch.Tensor, b: torch.Tensor) -> float:
    a, b = a.double().flatten(), b.double().flatten()
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


def parity_table(K, dev) -> dict:
    """SURVEY 8d "parity reported alongside": rel-L2 of (ours vs the reference composition in fp32 on the SAME device, cuDNN
    off), (ours vs the fp64 composition) and (fp32 composition vs fp64) for out, d/dsrc, d/dM, on white-noise and band-limited
    images at native resolution (forward 1080p, gradients at the cfg4 720p shape; two samples each, the bench homographies).
    The composition is oracle/kornia_restated.py (the ATen calls the reference issues): checker only, nothing here is timed."""
    from oracle import kornia_restated as R

    table = {"tolerance": 1e-4, "ref": "oracle/kornia_restated.py on cuda, cudnn disabled", "sets": {}}
    with torch.backends.cudnn.flags(enabled=False):
        for name in ("white", "bandlimited"):
            rows = {}
            # forward, 1080p
            shape = (2, C_IMG, H_IMG, W_IMG)
            src = torch.rand(shape, device=dev) if name == "white" else bandlimited(shape, dev, 11)
            M = make_homographies(2, 77).to(dev)
            with torch.no_grad():
                ours = K.warp_perspective(src, M, (H_IMG, W_IMG))
                r32 = R.warp_perspective(src, M, (H_IMG, W_IMG))
                r64 = R.warp_perspective(src.double(), M.double(), (H_IMG, W_IMG))
            rows["out_1080p"] = {"ours_vs_ref32": _rel(ours, r32), "ours_vs_fp64": _rel(ours, r64), "ref32_vs_fp64": _rel(r32, r64),
                                 "max_abs_ours_vs_ref32": float((ours - r32).abs().max())}
            del ours, r32, r64, src
            # gradients, 720p (cfg4): mean squared error against a band-limited target (smooth set), fixed random cotangent (white)
            Hh, Ww = 720, 1280
            shape = (2, C_IMG, Hh, Ww)
            src = torch.rand(shape, device=dev) if name == "white" else bandlimited(shape, dev, 12)
            g = torch.Generator().manual_seed(7)
            quad = torch.tensor([[0.0, 0.0], [Ww - 1.0, 0.0], [Ww - 1.0, Hh - 1.0], [0.0, Hh - 1.0]]).expand(2, 4, 2)
            M = perspective_from_quads(quad, quad + 8.0 * torch.randn(2, 4, 2, generator=g)).to(dev)
            target = bandlimited(shape, dev, 13)
            cot = torch.randn(shape, device=dev)

            def grads(impl, dt):
                s = src.to(dt).detach().requires_grad_(True)
                m = M.to(dt).detach().requires_grad_(True)
                out = impl.warp_perspective(s, m, (Hh, Ww))
                if name == "white":
                    out.backward(cot.to(dt))
                else:
                    ((out - target.to(dt)) ** 2).mean().backward()
                return out.detach(), s.grad, m.grad

            o, r32, r64 = grads(K, torch.float32), grads(R, torch.float32), grads(R, torch.float64)
            for key, i in (("out_720p", 0), ("dsrc_720p", 1), ("dM_720p", 2)):
                rows[key] = {"ours_vs_ref32": _rel(o[i], r32[i]), "ours_vs_fp64": _rel(o[i], r64[i]), "ref32_vs_fp64": _rel(r32[i], r64[i])}
            table["sets"][name] = rows
            del o, r32, r64, src, target, cot
    torch.cuda.empty_cache()
    return table


def _time_gpu(fn, dev, warmup: int = 2, iters: int = 5) -> float:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize(dev)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    torch.cuda.synchronize(dev)
    return t0.elapsed_time(t1) / iters


def torch_gpu_legs(workload: str, dev, sample_b: int = 32, with_compile: bool = True) -> dict:
    """The reference's own torch composition ON THIS GPU (SURVEY 8d: "the real bar to beat"): oracle/kornia_restated.py in
    eager mode and under torch.compile, on a bounded sample of the workload (per-pixel metric; the composition's temporaries
    -- a (B,h,w,2) grid plus ~15 elementwise intermediates -- are why the sample is smaller than the batch).  Reported context,
    never part of value / e2e."""
    from oracle import kornia_restated as R

    out = {}
    torch.manual_seed(5)
    if workload == "warp":
        x = torch.rand(sample_b, C_IMG, H_IMG, W_IMG, device=dev)
        M = make_homographies(sample_b, 5).to(dev)
        fn, pix = (lambda f: (lambda: f(x, M, (H_IMG, W_IMG)))), sample_b * H_IMG * W_IMG
        target = R.warp_perspective
    elif workload == "blur":
        x = torch.rand(sample_b, C_IMG, H_IMG, W_IMG, device=dev)
        fn, pix = (lambda f: (lambda: f(x, (11, 11), (2.0, 2.0), "reflect", True))), sample_b * H_IMG * W_IMG
        target = R.gaussian_blur2d
    elif workload == "warp_bwd":
        Hh, Ww = 720, 1280
        x = torch.rand(sample_b, C_IMG, Hh, Ww, device=dev)
        M = make_homographies_hw(sample_b, 5, Hh, Ww).to(dev)
        cot = torch.rand(sample_b, C_IMG, Hh, Ww, device=dev) - 0.5

        def fn(f):
            def step():
                s, m = x.detach().requires_grad_(True), M.detach().requires_grad_(True)
                return torch.autograd.grad(f(s, m, (Hh, Ww)), [s, m], grad_outputs=cot)
            return step

        pix, target = sample_b * Hh * Ww, R.warp_perspective
    else:
        return out
    sample = f"B={sample_b} of the workload, CUDA events, 2 warm-ups + 5 iterations"
    try:
        ms = _time_gpu(fn(target), dev)
        out["torch_eager_gpu"] = {"value": pix / (ms * 1e-3) / 1e6, "unit": "Mpix/s", "ms": ms, "sample": sample, "what": "oracle/kornia_restated.py (the reference's ATen call sequence) in torch eager on this GPU"}
    except Exception as e:  # out of memory on a busy box, ...
        out["torch_eager_gpu"] = {"value": None, "error": f"{type(e).__name__}: {str(e)[:160]}"}
    if with_compile:
        try:
            torch._dynamo.reset()
            compiled = torch.compile(target)
            t_c0 = time.perf_counter()
            ms = _time_gpu(fn(compiled), dev)
            out["torch_compile_gpu"] = {"value": pix / (ms * 1e-3) / 1e6, "unit": "Mpix/s", "ms": ms, "sample": sample,
                                        "what": "torch.compile (inductor) of the same composition", "compile_and_measure_s": time.perf_counter() - t_c0}
        except Exception as e:  # inductor toolchain missing / failing on the box
            out["torch_compile_gpu"] = {"value": None, "error": f"{type(e).__name__}: {str(e)[:160]}"}
    del x
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------ ours
def host_ring_samples(B: int, chunk: int, available_bytes=None, local_ranks=None) -> int:
    """How many samples of the batch each rank keeps in pinned host memory (source and destination each); the arithmetic
    lives in the library (kornia_b200/streaming.py:host_ring_samples)."""
    from kornia_b200.streaming import host_ring_samples as ring

    return ring(B, chunk, 2 * C_IMG * H_IMG * W_IMG * 4, available_bytes, local_ranks)


def e2e_run(K, M_dev, B, steps, warmup, chunk, dev, uint8_frames=False):
    """Host-buffer throughput through the library's own host pipeline (kornia_b200.streaming.warp_perspective_host: pinned
    src -> device -> warp -> pinned dst, chunked over 3 streams, the process bound to the GPU's NUMA node).  ``uint8_frames``:
    the source is what a decoder delivers -- interleaved uint8 (B,H,W,3), 3 bytes per pixel over PCIe instead of 12 -- converted
    and warped in one kernel (warp_perspective_from_uint8); the fp32 result comes back as before."""
    from kornia_b200 import streaming

    n_el = B * C_IMG * H_IMG * W_IMG
    numa = streaming.bind_to_device_numa_node(dev.index)  # before the pinned allocations: their pages follow the policy
    # Host side of the step: the whole batch in pinned memory (2 x 6.37 GB per rank at B=256).  When the box cannot
    # spare that for every local rank (8 ranks would lock 102 GB), the batch is streamed through a shorter pinned ring
    # of whole chunks instead: the bytes crossing PCIe per step are the same, the note says which form ran.
    HB = host_ring_samples(B, chunk)
    try:
        if uint8_frames:
            src_h = streaming.pinned_empty((HB, H_IMG, W_IMG, C_IMG), torch.uint8, dev.index)
        else:
            src_h = streaming.pinned_empty((HB, C_IMG, H_IMG, W_IMG), torch.float32, dev.index)
        dst_h = streaming.pinned_empty((HB, C_IMG, H_IMG, W_IMG), torch.float32, dev.index)
    except RuntimeError as e:  # not enough lockable host memory
        return None, f"pinned allocation failed: {e}"
    # cheap deterministic fill (content does not affect timing); touching every page also places it
    if uint8_frames:
        src_h.view(-1)[: 1 << 20].random_(0, 256)
        src_h.view(-1)[1 << 20:] = 127
    else:
        src_h.view(-1)[: 1 << 20].uniform_()
        src_h.view(-1)[1 << 20:] = 0.5
    dst_h.zero_()

    def one_step():
        # join=False: consecutive steps overlap like any stream of batches would (the first copies of step n+1 run under the
        # tail of step n); streaming.join() below orders the stop event after everything, copies included
        streaming.warp_perspective_host(src_h, M_dev, (H_IMG, W_IMG), out=dst_h, device=dev, chunk=chunk, logical_batch=B, synchronize=False,
                                        join=False)

    for _ in range(warmup):
        one_step()
    streaming.join(dev, chunk)
    torch.cuda.synchronize(dev)
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        one_step()
    streaming.join(dev, chunk)
    t1.record()
    torch.cuda.synchronize(dev)
    ms = t0.elapsed_time(t1) / steps
    del src_h, dst_h
    host = "whole batch pinned" if HB == B else f"pinned ring of {HB} samples reused {B / HB:.1f}x per step (host memory per local rank)"
    h2d = n_el * (1 if uint8_frames else 4)
    return ms, (f"kornia_b200.streaming.warp_perspective_host: pinned host buffers ({host}), chunk={chunk} samples, 3 streams (H2D / kernel / D2H), "
                f"{h2d} B in / {n_el * 4} B out per step; NUMA binding {numa}")


def max_over_ranks_or_none(dist, ms, note, device):
    """Max over ranks of a per-rank time that some ranks may not have (None, e.g. a pinned allocation that failed): EVERY rank
    takes part in the one all_reduce -- a missing value travels as +inf -- and all ranks return the same (ms | None, note)."""
    t = torch.tensor([ms if ms is not None else float("inf")], device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    worst = float(t.item())
    if math.isfinite(worst):
        return worst, note
    return None, note if ms is None else "unavailable on another rank"


def run_ours(args) -> None:
    import kornia_b200 as K
    from kornia_b200 import _lib, _ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; kornia_b200 has no CPU path (use --impl reference for the CPU port)")
    _lib.load()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    B = args.batch
    # per-rank shard generated in place: no scatter needed (SURVEY.md 8e), seed = 1000 + rank
    torch.manual_seed(1000 + rank)
    src = torch.rand(B, C_IMG, H_IMG, W_IMG, device=dev)
    M = make_homographies(B, 1000 + rank).to(dev)
    dsize = (H_IMG, W_IMG)

    def barrier():
        if dist is not None:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        out = K.warp_perspective(src, M, dsize)
    variant = _lib.last_warp_variant()
    barrier()
    _ops.kernel_events = []
    launches0 = _ops.launch_count
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        barrier()
        t0.record()
        for _ in range(args.steps):
            out = K.warp_perspective(src, M, dsize)
        t1.record()
        barrier()
        timed_events, _ops.kernel_events = _ops.kernel_events, None
        launches = _ops.launch_count - launches0
        clk.hold_load(lambda: K.warp_perspective(src, M, dsize), lambda: torch.cuda.synchronize(dev))
    total_ms = t0.elapsed_time(t1)
    kern_ms = [s.elapsed_time(e) for (_, s, e) in timed_events]
    checksum = float(out[0, :, ::97, ::89].sum())  # touch the result
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"out": out})
    del out
    if dist is not None:
        t = torch.tensor([total_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    ms_step = total_ms / args.steps
    pix_step = world * B * H_IMG * W_IMG
    value = pix_step / (ms_step * 1e-3) / 1e6

    # ---------------------------------------------------------------- e2e (host buffers)
    e2e_ms, e2e_note = e2e_run(K, M, B, steps=max(3, min(args.steps, 5)), warmup=1, chunk=args.e2e_chunk, dev=dev)
    if dist is not None:
        e2e_ms, e2e_note = max_over_ranks_or_none(dist, e2e_ms, e2e_note, dev)
    barrier()
    # the same step fed with decoder bytes (SURVEY 8f row 4): context for the e2e number, not the headline (a different wire format)
    u8_ms, u8_note = e2e_run(K, M, B, steps=3, warmup=1, chunk=args.e2e_chunk, dev=dev, uint8_frames=True)
    if dist is not None:
        u8_ms, u8_note = max_over_ranks_or_none(dist, u8_ms, u8_note, dev)
    barrier()
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    peaks, peak_src = None, "fallback 6650 GB/s (B200_PROFILING.md)"
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peak = float(peaks["hbm_gbs"])
        peak_src = "measured MEASURED_PEAKS.json hbm_gbs (burst copy)"
    except Exception:
        peak = 6650.0
    k_ms = statistics.mean(kern_ms) if kern_ms else float("nan")
    achieved = BYTES_PER_PIX * B * H_IMG * W_IMG / (k_ms * 1e-3) / 1e9
    traffic = None
    try:  # per-launch DRAM bytes of the same kernel from the committed ncu capture, if any
        traffic = json.load(open(os.path.join(ROOT, "profiles", "warp_fwd_traffic.json"))).get("dram_bytes_per_launch")
    except Exception:
        pass

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        mpix, ms, cores = cpu_reference_run(steps=3, warmup=1, sample_b=32)
        cpu = {"value": mpix, "unit": "Mpix/s", "cores": cores, "kind": "port",
               "sample": f"3 steps of B=32x3x1080x1920 ({ms:.0f} ms each) with torch CPU ops, {cores} of {os.cpu_count()} threads "
                         "(best of a calibration): oracle/kornia_restated.py"}

    side = {}
    if world == 1 and not args.no_side_legs:
        del src
        torch.cuda.empty_cache()
        side["parity"] = parity_table(K, dev)
        side["same_gpu_reference"] = torch_gpu_legs("warp", dev, with_compile=not args.no_compile_leg)
    bytes_step = B * C_IMG * H_IMG * W_IMG * 4
    line = {
        "metric": METRIC, "value": value, "unit": "Mpix/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": headline_config(B, world), "kernel_variant": variant,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "kernel_ms": k_ms, "kernel_launches_timed": len(kern_ms), "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": BYTES_PER_PIX * B * H_IMG * W_IMG},
        "cpu_baseline": cpu,
        "e2e": ({"value": pix_step / (e2e_ms * 1e-3) / 1e6, "unit": "Mpix/s", "h2d_bytes_per_step": bytes_step,
                 "d2h_bytes_per_step": bytes_step, "ms_per_step": e2e_ms, "note": e2e_note}
                if e2e_ms is not None else {"value": None, "unit": "Mpix/s", "note": e2e_note}),
        "e2e_uint8_frames": ({"value": pix_step / (u8_ms * 1e-3) / 1e6, "unit": "Mpix/s", "h2d_bytes_per_step": bytes_step // 4,
                              "d2h_bytes_per_step": bytes_step, "ms_per_step": u8_ms, "note": u8_note}
                             if u8_ms is not None else {"value": None, "unit": "Mpix/s", "note": u8_note}),
        "gpu_launches": launches,
        "clocks": clk.summary(),
        "checksum": checksum,
    }
    line.update(side)
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def run_extra(args) -> None:
    """Secondary BASELINE.json configs (not the driver's headline line): ``--workload blur`` = configs[2]
    gaussian_blur2d k=11 B=256x3x1080x1920; ``--workload warp_bwd`` = configs[3] warp_perspective fwd+bwd
    (grad wrt image and H) B=128x3x720x1280; ``--workload ingest`` = warp_perspective_from_uint8 on B x 1080 x 1920 x 3 decoder
    bytes (SURVEY 8f row 4; 15 algorithmic bytes per pixel).  Single GPU, inputs resident, CUDA events, one JSON line."""
    import kornia_b200 as K
    from kornia_b200 import _lib, _ops

    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    _lib.load()
    peak = 6650.0
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    torch.manual_seed(1000)
    if args.workload == "blur":
        B = args.batch
        x = torch.rand(B, 3, H_IMG, W_IMG, device=dev)
        step = lambda: K.gaussian_blur2d(x, (11, 11), (2.0, 2.0), "reflect", True)  # noqa: E731
        pix, bytes_per_pix = B * H_IMG * W_IMG, 24.0
        name = f"gaussian_blur2d k=11 sigma=2 reflect separable B={B}x3x1080x1920"
        tag = "sepfilter_forward"
    elif args.workload == "ingest":
        B = args.batch
        frames = torch.randint(0, 256, (B, H_IMG, W_IMG, 3), device=dev, dtype=torch.uint8)
        M = make_homographies(B, 1000).to(dev)
        step = lambda: K.geometry.transform.warp_perspective_from_uint8(frames, M, (H_IMG, W_IMG))  # noqa: E731
        pix, bytes_per_pix = B * H_IMG * W_IMG, 15.0
        name = f"warp_perspective_from_uint8 (decoder bytes HWC -> warped fp32 NCHW) B={B}x1080x1920x3, bilinear, zeros"
        tag = "warp_u8hwc_forward"
    else:
        B, Hh, Ww = min(args.batch, 128), 720, 1280
        src = torch.rand(B, 3, Hh, Ww, device=dev, requires_grad=True)
        g = torch.Generator().manual_seed(7)
        quad = torch.tensor([[0.0, 0.0], [Ww - 1.0, 0.0], [Ww - 1.0, Hh - 1.0], [0.0, Hh - 1.0]]).expand(B, 4, 2)
        M = perspective_from_quads(quad, quad + 8.0 * torch.randn(B, 4, 2, generator=g)).to(dev).requires_grad_(True)
        cot = torch.rand(B, 3, Hh, Ww, device=dev) - 0.5  # fixed upstream gradient: no loss glue in the timed region

        def step():
            out = K.warp_perspective(src, M, (Hh, Ww))
            return torch.autograd.grad(out, [src, M], grad_outputs=cot)

        pix, bytes_per_pix = B * Hh * Ww, 60.0
        name = f"warp_perspective fwd+bwd (d/dsrc, d/dM), fixed cotangent, B={B}x3x720x1280"
        tag = "warp_backward"
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize(dev)
    _ops.kernel_events = [] if tag else None
    launches0 = _ops.launch_count
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(dev.index or 0) as clk:
        t0.record()
        for _ in range(args.steps):
            res = step()
        t1.record()
        torch.cuda.synchronize(dev)
        timed_events, _ops.kernel_events = (_ops.kernel_events or []), None
        launches = _ops.launch_count - launches0
        clk.hold_load(step, lambda: torch.cuda.synchronize(dev))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(("grad_src", "grad_M"), res)) if args.workload == "warp_bwd" else {"out": res})
    del res
    ms = t0.elapsed_time(t1) / args.steps
    kern = [s.elapsed_time(e) for (tg, s, e) in timed_events if tg == tag]
    k_ms = statistics.mean(kern) if kern else None
    line = {"metric": "Mpix/s " + name, "value": pix / (ms * 1e-3) / 1e6, "unit": "Mpix/s", "n_gpus": 1, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "dtype": "f32", "data": "synthetic",
            "config": {"workload": name, "note": "whole step through the public API (for warp_bwd: forward, zero-fill of d/dsrc, backward, d/dM reduction, torch prelude autograd)"},
            "roofline": {"bound": "hbm", "unit": "GB/s", "peak": peak, "algorithmic_bytes_per_pixel": bytes_per_pix,
                         "achieved_step": bytes_per_pix * pix / (ms * 1e-3) / 1e9, "frac_step": bytes_per_pix * pix / (ms * 1e-3) / 1e9 / peak,
                         "kernel_ms": k_ms, "achieved": (bytes_per_pix * pix / (k_ms * 1e-3) / 1e9) if k_ms else None,
                         "frac": (bytes_per_pix * pix / (k_ms * 1e-3) / 1e9 / peak) if k_ms else None},
            "gpu_launches": launches, "clocks": clk.summary()}
    if not args.no_side_legs and args.workload in ("blur", "warp_bwd"):
        line["same_gpu_reference"] = torch_gpu_legs(args.workload, dev, sample_b=32 if args.workload == "blur" else 16, with_compile=not args.no_compile_leg)
        if args.workload == "warp_bwd":
            line["parity"] = parity_table(K, dev)
    if args.workload == "warp_bwd":  # the timed kernel is the backward alone: 36 B/pixel (read gout + src, write gsrc)
        line["roofline"].update({"kernel": "warp_backward (+ d/dM reduction)", "kernel_bytes_per_pixel": 36.0,
                                 "achieved": (36.0 * pix / (k_ms * 1e-3) / 1e9) if k_ms else None,
                                 "frac": (36.0 * pix / (k_ms * 1e-3) / 1e9 / peak) if k_ms else None})
    print(json.dumps(line), flush=True)


def run_small(args) -> None:
    """The only operating point the reference PUBLISHES (benchmarks/README.md:154-157; benchmarks/geometry/flagship.py): 256x256,
    batch 32, fp32, throughput in images/s of back-to-back calls -- host launch cost included, the reference's own method
    (torch.utils.benchmark blocked_autorange: wall clock over many calls with one sync at the end).  Published on an RTX PRO 6000
    Blackwell: warp_perspective 96 022 eager / 232 170 compiled, warp_affine 120 089 / 217 083, rotate 58 357 / 159 196
    (torchvision 298 016), get_perspective_transform 78 071 / 431 034 solves/s.  One JSON line; `vs_published` = ours / published."""
    import kornia_b200 as K
    from kornia_b200 import _lib, _ops
    from oracle import kornia_restated as R

    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    _lib.load()
    b, h, w = 32, 256, 256
    torch.manual_seed(0)
    x = torch.rand(b, 3, h, w, device=dev)
    angle = torch.full((b,), 30.0, device=dev)
    center = torch.tensor([[w / 2, h / 2]], device=dev).expand(b, 2).contiguous()
    scale = torch.ones(b, 2, device=dev)
    quad = torch.tensor([[[0.0, 0.0], [w - 1.0, 0.0], [w - 1.0, h - 1.0], [0.0, h - 1.0]]]).expand(b, 4, 2).contiguous()
    dst = (quad + 8.0 * torch.randn(b, 4, 2, generator=torch.Generator().manual_seed(0))).to(dev)
    quad = quad.to(dev)
    m_aff = K.geometry.transform.get_rotation_matrix2d(center, angle, scale)
    h_mat = K.geometry.transform.get_perspective_transform(quad, dst)
    published = {"warp_perspective": (96022, 232170), "warp_affine": (120089, 217083), "rotate": (58357, 159196), "get_perspective_transform": (78071, 431034)}

    def cases(impl):
        return {"warp_perspective": lambda: impl.warp_perspective(x, h_mat, (h, w)),
                "warp_affine": lambda: impl.warp_affine(x, m_aff, (h, w)),
                "rotate": (lambda: impl.geometry.transform.rotate(x, angle)) if impl is K else (lambda: impl.rotate(x, angle)),
                "get_perspective_transform": (lambda: impl.geometry.transform.get_perspective_transform(quad, dst)) if impl is K else (lambda: impl.get_perspective_transform(quad, dst))}

    def throughput(fn, seconds=1.0):
        for _ in range(20):
            fn()
        torch.cuda.synchronize(dev)
        n, t0 = 0, time.perf_counter()
        while True:
            for _ in range(100):
                fn()
            n += 100
            torch.cuda.synchronize(dev)
            dt = time.perf_counter() - t0
            if dt >= seconds:
                return b * n / dt, dt / n * 1e6

    def device_us(fn, n=200):  # what the GPU needs per call once the host is out of the way (events around n queued calls)
        for _ in range(20):
            fn()
        torch.cuda.synchronize(dev)
        big = torch.empty(1 << 28, dtype=torch.uint8, device=dev)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        big.zero_()  # ~40 us of queued device work: the n calls are enqueued behind it, so the events bracket back-to-back kernels
        big.zero_()
        t0.record()
        for _ in range(n):
            fn()
        t1.record()
        torch.cuda.synchronize(dev)
        return t0.elapsed_time(t1) * 1e3 / n

    rows = {}
    with torch.no_grad():
        launches0 = _ops.launch_count
        for name, fn in cases(K).items():
            ips, us = throughput(fn)
            rows[name] = {"ours_img_s": ips, "ours_us_per_call": us, "events_us_per_call": device_us(fn), "published_eager": published[name][0], "published_compiled": published[name][1],
                          "vs_published_eager": ips / published[name][0], "vs_published_compiled": ips / published[name][1]}
        launches = _ops.launch_count - launches0
        # the same calls replayed from a CUDA graph (kornia_b200.graphs.GraphedCall: one cudaGraphLaunch per call, inputs already in
        # the graph's static buffers) -- the launch-bound regime's answer on this hardware
        graph_specs = {"warp_perspective": (lambda a, m: K.warp_perspective(a, m, (h, w)), (x, h_mat)),
                       "warp_affine": (lambda a, m: K.warp_affine(a, m, (h, w)), (x, m_aff)),
                       # the centre is passed in: building it from Python floats is a host->device copy, which a capture cannot hold
                       "rotate": (lambda a, ang, c: K.geometry.transform.rotate(a, ang, c), (x, angle, (center - 0.5).contiguous()))}
        for name, (fn, tensors) in graph_specs.items():
            try:
                gc = K.graphs.GraphedCall(fn, *tensors)
                ins = gc.inputs
                ips, us = throughput(lambda: gc(*ins))
                rows[name].update({"cuda_graph_img_s": ips, "cuda_graph_us_per_call": us, "cuda_graph_vs_published_compiled": ips / published[name][1]})
            except Exception as e:
                rows[name].update({"cuda_graph_img_s": None, "cuda_graph_error": f"{type(e).__name__}: {str(e)[:160]}"})
                torch.cuda.synchronize(dev)
        if not args.no_side_legs:
            for name, fn in cases(R).items():  # the reference composition in torch eager on THIS GPU
                ips, us = throughput(fn, 0.5)
                rows[name].update({"torch_eager_here_img_s": ips, "vs_torch_eager_here": rows[name]["ours_img_s"] / ips})
    # class API (SURVEY 8f row 1; benchmarks/README.md:195-199 publishes CPU / MPS numbers only): parameter sampling on the device
    # + application, p = 1.  "torch_composition_here" = the same classes with the image functions swapped for the oracle's
    # torch composition on this GPU (the reference's classes cannot travel to the GPU box).
    import importlib

    A = importlib.import_module("kornia_b200.augmentation")
    published_cpu = {"RandomPerspective": 843, "RandomAffine": 899, "RandomGaussianBlur": 1103}
    swaps = {"warp_perspective": R.warp_perspective, "warp_affine": R.warp_affine, "gaussian_blur2d": R.gaussian_blur2d,
             "get_perspective_transform": R.get_perspective_transform, "get_rotation_matrix2d": R.get_rotation_matrix2d}
    aug_rows = {}
    with torch.no_grad():
        for name, make in (("RandomPerspective", lambda: A.RandomPerspective(0.5, p=1.0)),
                           ("RandomAffine", lambda: A.RandomAffine(30.0, translate=(0.1, 0.1), scale=(0.8, 1.2), shear=10.0, p=1.0)),
                           ("RandomGaussianBlur", lambda: A.RandomGaussianBlur((5, 5), (0.1, 2.0), p=1.0))):
            aug = make().to(dev)
            ips, us = throughput(lambda: aug(x))
            aug_rows[name] = {"ours_img_s": ips, "ours_us_per_call": us, "published_cpu_eager_apple": published_cpu[name]}
            if not args.no_side_legs:
                saved = {k: getattr(A, k) for k in swaps}
                try:
                    for k, v in swaps.items():
                        setattr(A, k, v)
                    ips_t, _ = throughput(lambda: aug(x), 0.5)
                finally:
                    for k, v in saved.items():
                        setattr(A, k, v)
                aug_rows[name].update({"torch_composition_here_img_s": ips_t, "vs_torch_composition_here": ips / ips_t})
    head = rows["warp_perspective"]
    line = {"metric": "img/s warp_perspective 32x3x256x256 fwd bilinear fp32 (back-to-back calls, wall clock, host cost included)", "value": head["ours_img_s"],
            "unit": "img/s", "n_gpus": 1, "higher_is_better": True, "dtype": "f32", "data": "synthetic",
            "vs_baseline": head["vs_published_compiled"],
            "config": {"workload": "benchmarks/geometry/flagship.py operating point: batch 32, 256x256, fp32; rotate 30 deg about the centre, corner quad jittered by 8*randn px",
                       "baseline": "benchmarks/README.md:154-157, RTX PRO 6000 Blackwell, kornia + torch.compile (other hardware: published context, not a same-box comparison)",
                       "timing": ">= 1 s of back-to-back calls per op, one synchronize per 100 calls, wall clock"},
            "ops": rows, "augmentation_classes": aug_rows, "gpu_launches": launches}
    print(json.dumps(line), flush=True)


def run_scatter_gather(args) -> None:
    """cfg5 as BASELINE.json words it ("batch-sharded ... via NCCL"), the secondary numbers of SURVEY 8d: the batch starts and ends
    on rank 0.  (1) kornia_b200.sharding.sharded_apply: ONE NCCL scatter of the inputs, the warp on every rank, ONE NCCL gather of
    the outputs -- timed with CUDA events on every rank, max over ranks, reported with the NVLink GB/s the two collectives
    achieve; (2) strong scaling: the same global batch with shards already resident (what (1) costs without its collectives)."""
    import torch.distributed as dist

    import kornia_b200 as K
    from kornia_b200 import _lib
    from kornia_b200.sharding import shard_range, sharded_apply

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    _lib.load()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    else:
        dist.init_process_group("gloo", init_method="tcp://127.0.0.1:29512", rank=0, world_size=1)
    Bg = args.global_batch or 64 * world  # rank 0 holds the whole input and output: 2 x 24.9 MB per sample
    torch.manual_seed(1000)
    src = torch.rand(Bg, C_IMG, H_IMG, W_IMG, device=dev) if rank == 0 else None
    M = make_homographies(Bg, 1000).to(dev)
    dsize = (H_IMG, W_IMG)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize(dev)

    def max_ms(ms):
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(steps):
            fn()
        t1.record()
        barrier()
        return max_ms(t0.elapsed_time(t1) / steps)

    steps, warmup = max(2, min(args.steps, 5)), max(2, min(args.warmup, 3))

    def sg_step():
        return sharded_apply(lambda s, m: K.warp_perspective(s, m, dsize), (src, M if rank == 0 else None), batch=Bg,
                             shapes=[(C_IMG, H_IMG, W_IMG), (3, 3)], dtypes=[torch.float32, torch.float32], device=dev, root=0)

    out = sg_step()
    checksum = float(out[0, :, ::97, ::89].sum()) if rank == 0 else 0.0
    del out
    sg_ms = timed(sg_step, steps, warmup)
    # strong scaling: same global batch, shard already resident on its rank (generated from the same seed, then sliced)
    a, b = shard_range(Bg, world, rank)
    if rank == 0:
        shard = src[a:b].clone()
        del src
    else:
        shard = torch.rand(b - a, C_IMG, H_IMG, W_IMG, device=dev)
    src = None
    Ms = M[a:b].contiguous()
    res_ms = timed(lambda: K.warp_perspective(shard, Ms, dsize), max(args.steps, 5), max(args.warmup, 3))
    if rank == 0:
        pix = Bg * H_IMG * W_IMG
        moved = (Bg - (b - a)) * C_IMG * H_IMG * W_IMG * 4  # bytes leaving rank 0 in the scatter (= bytes arriving in the gather)
        coll_ms = max(sg_ms - res_ms, 1e-6)
        line = {"metric": "Mpix/s warp_perspective global batch on rank 0: NCCL scatter -> warp on every rank -> NCCL gather", "value": pix / (sg_ms * 1e-3) / 1e6,
                "unit": "Mpix/s", "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": sg_ms, "higher_is_better": True, "scaling": "strong",
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": f"warp_perspective fwd global B={Bg}x3x1080x1920 held by rank 0 (BASELINE.json configs[4] 'via NCCL', secondary number of SURVEY 8d)",
                           "global_batch": Bg, "parallelism": f"kornia_b200.sharding.sharded_apply over {world} ranks: 1 scatter + 1 gather, no other collective"},
                "collectives": {"bytes_out_of_rank0_per_direction": moved, "ms_scatter_plus_gather": coll_ms,
                                "nvlink_GBps_per_direction_rank0": moved / (coll_ms / 2 * 1e-3) / 1e9,
                                "note": "rank 0's NVLink ports serialise the scatter and the gather: 2 x bytes over its 900 GB/s per direction"},
                "strong_scaling_resident": {"value": pix / (res_ms * 1e-3) / 1e6, "unit": "Mpix/s", "ms_per_step": res_ms,
                                            "note": f"same global batch, shards of {b - a} samples already on their ranks, max over ranks"},
                "checksum": checksum}
        print(json.dumps(line), flush=True)
    dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--batch", type=int, default=256, help="samples per GPU")
    ap.add_argument("--e2e-chunk", type=int, default=16)
    ap.add_argument("--global-batch", type=int, default=0, help="scatter_gather workload: samples held by rank 0 (default 64 per rank)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side-legs", action="store_true", help="skip the untimed context legs (parity table, torch eager / torch.compile of the "
                    "reference composition on the same GPU)")
    ap.add_argument("--no-compile-leg", action="store_true", help="skip only the torch.compile leg (inductor needs a host compiler and ~1 min)")
    ap.add_argument("--workload", choices=["warp", "blur", "warp_bwd", "ingest", "small", "scatter_gather"], default="warp",
                    help="warp = the headline (BASELINE.json configs[1]); blur / warp_bwd = configs[2] / configs[3]; ingest = the uint8 wire-format warp "
                         "(SURVEY 8f row 4, not a BASELINE config); single GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last step returned as DIR/<name>.npy "
                    "(float32 / float64, under 64 MB in all: a larger output as a fixed, seeded sample); warp, blur, warp_bwd and ingest")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload in ("small", "scatter_gather")):
        ap.error("--dump-outputs covers the warp, blur, warp_bwd and ingest workloads of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "small":
        run_small(args)
    elif args.workload == "scatter_gather":
        run_scatter_gather(args)
    elif args.workload != "warp":
        run_extra(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
