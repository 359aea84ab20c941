#!/usr/bin/env python
"""Headline benchmark: fused SQ implicit-loss forward+backward throughput (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch: ``ImplicitLoss(64, dev, 1.5, 260)(images, pred)`` followed by
``.backward()`` on BASELINE config 2 (batch 256, 64^3 grid, fp32) -- 67 108 864 points per GPU.  Under torchrun
(N > 1) every rank runs its own batch (the path shards by sample, no data-path collective: weak scaling) and the
step time is the max over ranks.

Printed line (rank 0):
  ``value``        Gpoints/s with inputs resident in HBM (CUDA events over exactly K graph-replayed steps)
  ``dense``        the same call on a second workload, sizes a ~ U(0.5, 1): objects fill the grid, culling cannot help
  ``e2e``          host buffers in, host results out, copies inside the timed region: 8-bit depth maps and fp32 parameters in
                   pinned memory through sq_implicit_loss_host_submit / _wait, several batches in flight; H2D bytes counted and
                   measured (NVML PCIe receive counter); round 1's blocking fp32-image call next to it
  ``roofline``     the dominant kernel against the measured MUFU (SFU) peak of this GPU: issued MUFU-pipe ops from the counting
                   build of the same sources, ``walked_fraction``, ``evaluated_gpoints_per_s``; DRAM traffic from the ncu capture
  ``cpu_baseline`` the UNMODIFIED reference (staged under oracle/_ref) on the box's host cores on a bounded sample
``--impl reference`` times that CPU path alone (same ``config``; ``--steps`` / ``--warmup`` honoured).

``--steps K`` sets the timed window of ``value`` and of ``one_batch_at_a_time`` exactly.  The secondary windows time their
own counts, each reported next to its figure: ``dense`` max(4, min(K, 80)) steps, ``e2e`` max(4, K), its blocking fp32 call
and the kernel-alone times at most 20.

``--dump-outputs DIR`` writes what the last timed step returned to its caller -- the loss (float64) and the gradient with
respect to the parameters (float32, B x 12) of the headline workload and of ``dense`` -- as DIR/<name>.npy (``_rank<r>``
appended under torchrun).  The inputs are seeded, so two builds run with the same arguments can be compared file by file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "fused SQ implicit-loss fwd+bwd throughput"
UNIT = "Gpoints/s"
B, R, H, W = 256, 64, 256, 256           # BASELINE config 2; depth maps are 256x256 like the reference's dataset
TAU, SHARP = 1.5, 260.0                  # torch/train.py:64
MUFU_PER_POINT = 16                      # SURVEY 8d: 12 (five pows + sigmoid) + 1 (exp(-tau cs)) + 3 (backward rcp)
CPU_SAMPLE_B = 8                         # bounded CPU sample: a B=8 slice of the same workload


def workload_config(n_gpus):
    return {"workload": f"ImplicitLoss(render_size={R}, tau={TAU}, sigmoid_sharpness={SHARP:g}) fwd+bwd, batch {B} per GPU, "
                        f"{R}^3 grid, depth maps {H}x{W} (BASELINE config 2)",
            "points_per_step_per_gpu": B * R ** 3, "batch_per_gpu": B, "render_size": R,
            "l2": "inputs rotate over 4 independent batches (4 x 67 MB of depth maps > 126 MB L2)",
            "reference_arm_sample": REFERENCE_SAMPLE,
            "parallelism": f"{n_gpus} x independent batch shards, no data-path collective"}


# ----------------------------------------------------------------------------------------------- CPU reference arm
REFERENCE_SAMPLE = (f"the reference arm and cpu_baseline run a B={CPU_SAMPLE_B} slice of this workload per step on the host cores "
                    f"({CPU_SAMPLE_B * R ** 3} points), scaled per point")


def cpu_reference(steps, warmup):
    """The reference's own ImplicitLoss (UNMODIFIED torch/classes.py staged under oracle/_ref by oracle/build_ref.py;
    the oracle port's loop form when that is absent) on all host cores, fwd+bwd, on a B=8 slice of the workload.
    This is the one place bench.py executes anything under oracle/ (the checker timed as the CPU baseline)."""
    from oracle import ref_import
    from oracle import sq_oracle as O
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    cpu = torch.device("cpu")
    true = O.random_params(CPU_SAMPLE_B, 0)
    pred = O.perturbed_params(true, 5)
    if ref_import.available() or ref_import.staged():
        rc, _ = ref_import.load()
        crit, kind = rc.ImplicitLoss(R, cpu, TAU, SHARP), "reference"
        what = f"UNMODIFIED reference torch/classes.py ImplicitLoss({R}, cpu, {TAU}, {SHARP:g}) (oracle/_ref)"
    else:
        crit, kind = O.ImplicitLoss(R, "cpu", TAU, SHARP, form="loop"), "port"
        what = "oracle/sq_oracle.py loop form (the reference's per-sample op sequence; oracle/_ref not staged)"
    with torch.no_grad():   # depth maps: the reference's own render of the true parameters at R, blown up to H x W so that
        small = crit.depth_projection(true).float()          # the nearest resize inside the loss returns it unchanged
    img = small.repeat_interleave(H // R, dim=1).repeat_interleave(W // R, dim=2).unsqueeze(1).contiguous()
    times = []
    for i in range(warmup + steps):
        p = pred.clone().requires_grad_(True)
        t0 = time.perf_counter()
        loss = crit(img, p)
        loss.backward()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    pts = CPU_SAMPLE_B * R ** 3
    mean = float(np.mean(times))
    cpu_name = ""
    try:
        cpu_name = [l.split(":")[1].strip() for l in open("/proc/cpuinfo") if l.startswith("model name")][0]
    except Exception:
        pass
    return {"value": pts / mean / 1e9, "unit": UNIT, "cores": threads, "kind": kind,
            "sample": f"B={CPU_SAMPLE_B} slice of the workload ({pts} points per step), {steps} timed steps after {warmup} warm-up: "
                      f"mean {mean * 1e3:.1f} ms, best {np.min(times) * 1e3:.1f} ms per fwd+bwd; {what}; torch fp64, "
                      f"{threads} threads on {os.cpu_count()} host cores ({cpu_name})"}, mean


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = args.steps, max(0, args.warmup)
    cb, mean = cpu_reference(steps, warmup)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": mean * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(args.gpus),
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- helpers
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        busy = [v for v in sm if v > 0.5 * (max(mx) if mx else 1)] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_mufu_peak():
    """thread-MUFU-ops per clock per SM and the clock it was measured at, from the in-tree microbenchmark."""
    exe = os.path.join(ROOT, "sq_recovery_b200", "sq_peaks")
    try:
        out = subprocess.run([exe, "/dev/null", "--quick"], capture_output=True, text=True, timeout=120).stdout
        d = json.loads(out)
        return {"mufu_per_clk_sm": d["MUFU_MIX"]["mufu_per_clk_sm"], "sm_mhz": d["MUFU_MIX"]["sm_mhz"], "sms": d["sms"],
                "fp32_per_clk_sm": d["FFMA"]["fp32_per_clk_sm"], "source": "sq_peaks --quick, this run"}
    except Exception as e:   # fall back to the committed round-1 measurement
        try:
            d = json.load(open(os.path.join(ROOT, "profiles", "peaks_r01.json")))
            return {"mufu_per_clk_sm": d["MUFU_MIX"]["mufu_per_clk_sm"], "sm_mhz": d["MUFU_MIX"]["sm_mhz"], "sms": d["sms"],
                    "fp32_per_clk_sm": d["FFMA"]["fp32_per_clk_sm"], "source": f"profiles/peaks_r01.json ({type(e).__name__} running sq_peaks)"}
        except Exception:
            return {"mufu_per_clk_sm": 16.0, "sm_mhz": 1965.0, "sms": 148, "fp32_per_clk_sm": 128.0, "source": "nominal"}


def ncu_summary():
    """DRAM bytes per launch of the dominant kernel and the ncu count of its XU-pipe instructions, from the committed
    `ncu --set full` capture of this seeded workload (tools/profile_step.py + tools/ncu_summary.py), or None."""
    for name in ("implicit_kernel_ncu_summary_r02.json", "implicit_kernel_ncu_summary.json"):
        try:
            d = json.load(open(os.path.join(ROOT, "profiles", name)))
            d["file"] = "profiles/" + name
            return d
        except Exception:
            continue
    return None


class PcieSampler:
    """NVML PCIe receive counter (bytes the GPU pulled from the host) while a loop runs: the measured H2D traffic."""

    def __init__(self, index):
        self.rx, self.stop_flag, self.thread = [], False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self.nv = None

    def start(self):
        if self.nv is None:
            return
        def loop():
            while not self.stop_flag:
                try:      # KB/s over the driver's 20 ms window
                    self.rx.append(self.nv.nvmlDeviceGetPcieThroughput(self.h, self.nv.NVML_PCIE_UTIL_RX_BYTES))
                except Exception:
                    break
        self.thread = threading.Thread(target=loop, daemon=True)
        self.thread.start()

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=2)
        vals = [v for v in self.rx if v > 0]
        return (float(np.mean(vals)) * 1024.0) if vals else None          # bytes / s


# ----------------------------------------------------------------------------------------------- GPU arm
class Workload:
    """Four independent input batches of one parameter distribution, the step on them (public class call + backward), its
    CUDA-graph captures, and the timing / counting of it."""

    def __init__(self, name, size_range, S, O, dev, rank, side, side2):
        self.name, self.dev, self.S = name, dev, S
        self.crit = S.ImplicitLoss(R, dev, TAU, SHARP)
        render = S.ImplicitLoss(H, dev, TAU, SHARP)            # synthetic depth maps = soft renders of the true params
        self.sets = []
        for k in range(4):                                      # 4 independent batches, rotated -> inputs exceed L2
            true = O.random_params(B, 1000 * rank + k, size_range=size_range)
            pred = O.perturbed_params(true, 7 + k).to(dev)
            img = render.depth_projection(true.to(dev)).unsqueeze(1).contiguous()
            self.sets.append((img, pred))
        torch.cuda.synchronize()
        self.graphs, self.quad, self.quad_out, self.quad_seq = [], None, [], None
        self.side, self.side2 = side, side2

    def eager_step(self, i):
        img, pred = self.sets[i % 4]
        p = pred.detach().requires_grad_(True)
        loss = self.crit(img, p)
        loss.backward()
        return loss, p.grad

    def capture(self):
        """The same step captured once per input set (public API inside the capture: the class call and .backward());
        replaying it removes the ~100 us of Python/autograd launch overhead per step, which is longer than the kernels.
        And the four steps (one per input set) in ONE graph: a single launch then covers ~0.2 ms of GPU work, so the host's
        launch rate cannot leave the GPU idle between steps.  Same kernels, same work per step, same results (asserted).
        Two versions of that graph: `quad_seq` runs the four steps one after the other; `quad` (what `value` times) puts
        them alternately on two streams, i.e. TWO INDEPENDENT BATCHES IN FLIGHT: the plan / finalize kernels and the
        end-game of one batch's persistent kernel (its last warps finishing) run under the other batch's kernel -- the
        device-side counterpart of the two slots of the host-buffer API.  Warm-up and capture run on the side streams: the
        per-stream workspace must exist before a capture starts (INTEGRATION.md 5)."""
        dev, side, side2 = self.dev, self.side, self.side2
        for s_ in (side, side2):
            s_.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(s_):
                for k in range(4):
                    for _ in range(2):
                        self.eager_step(k)
            torch.cuda.current_stream(dev).wait_stream(s_)
        torch.cuda.synchronize()
        for k in range(4):
            gph = torch.cuda.CUDAGraph()
            img, pred = self.sets[k]
            p = pred.detach().requires_grad_(True)
            with torch.cuda.graph(gph, stream=side):
                loss_k = self.crit(img, p)
                loss_k.backward()
            self.graphs.append((gph, loss_k, p))
        self.quad_seq, seq_out = torch.cuda.CUDAGraph(), []
        with torch.cuda.graph(self.quad_seq, stream=side):
            for k in range(4):
                img, pred = self.sets[k]
                p = pred.detach().requires_grad_(True)
                loss_k = self.crit(img, p)
                loss_k.backward()
                seq_out.append((loss_k, p))
        self.quad = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.quad, stream=side):
            side2.wait_stream(side)
            for k in range(4):
                with torch.cuda.stream(side if k % 2 == 0 else side2):
                    img, pred = self.sets[k]
                    p = pred.detach().requires_grad_(True)
                    loss_k = self.crit(img, p)
                    loss_k.backward()
                    self.quad_out.append((loss_k, p))
            side.wait_stream(side2)
        self.quad_seq.replay(); self.quad.replay()
        torch.cuda.synchronize()
        for (l0, p0), (l1, p1) in zip(seq_out, self.quad_out):      # two in flight or one after the other: the same bits
            assert l0.item() == l1.item() and torch.equal(p0.grad, p1.grad)

    def step(self, i):
        if not self.graphs:
            return self.eager_step(i)
        gph, loss_k, p = self.graphs[i % 4]
        gph.replay()
        return loss_k, p.grad

    def run(self, steps, sequential=False):
        """`steps` steps enqueued back to back (four per graph launch when captured); returns the last (loss, grad)."""
        if self.graphs:
            for _ in range(steps // 4):
                (self.quad_seq if sequential else self.quad).replay()
            out = (self.quad_out[3][0], self.quad_out[3][1].grad)
            for i in range(steps - steps % 4, steps):
                out = self.step(i)
            return out
        for i in range(steps):
            out = self.eager_step(i)
        return out

    def kernel_ms(self, lib, n):
        """The column kernel alone: CUDA events recorded around its launch on its stream (sq_profile_events), eager."""
        ms = []
        for i in range(n):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); b.record()                              # materialise the cudaEvent_t handles
            torch.cuda.synchronize()
            lib.sq_profile_events(a.cuda_event, b.cuda_event)
            self.eager_step(i)
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
        return float(np.mean(ms))

    def counts(self):
        """What the column kernel did per launch on these inputs (counting build), averaged over the four batches."""
        from sq_recovery_b200 import counting
        per = [counting.implicit_counts(img, pred, R, TAU, SHARP, want_grad=True) for img, pred in self.sets]
        keys = per[0]["counters"].keys()
        return {"counters": {k: float(np.mean([p["counters"][k] for p in per])) for k in keys},
                "walked_fraction": float(np.mean([p["walked_fraction"] for p in per])),
                "point_evaluations": float(np.mean([p["point_evaluations"] for p in per])),
                "xu_warp_inst_model": float(np.mean([p["xu_warp_inst_model"] for p in per]))}


def roofline_block(kernel_ms, counts, peak, ncu, pts, clock):
    peak_gops = peak["mufu_per_clk_sm"] * peak["sms"] * peak["sm_mhz"] * 1e6 / 1e9       # thread-MUFU ops/s, measured
    issued = counts["xu_warp_inst_model"] * 32 if counts else None
    achieved = issued / (kernel_ms * 1e-3) / 1e9 if issued else None
    dense_equiv = pts * MUFU_PER_POINT / (kernel_ms * 1e-3) / 1e9
    out = {"bound": "sfu", "kernel": "implicit_kernel<true>", "achieved": achieved, "peak": peak_gops, "unit": "G MUFU-op/s",
           "frac": (achieved / peak_gops) if achieved else None, "kernel_ms": kernel_ms,
           "issued_xu_warp_inst_per_launch": counts["xu_warp_inst_model"] if counts else None,
           "walked_fraction": counts["walked_fraction"] if counts else None,
           "evaluated_gpoints_per_s": counts["point_evaluations"] / (kernel_ms * 1e-3) / 1e9 if counts else None,
           "counters_per_launch": counts["counters"] if counts else None,
           "reference_algorithm_equivalent": {"mufu_per_point": MUFU_PER_POINT, "achieved": dense_equiv, "frac": dense_equiv / peak_gops},
           "sm_mhz_during_run": clock}
    return out


def run_gpu(args):
    import torch.distributed as dist
    from sq_recovery_b200 import inputs as O                # seeded randsq / randquat workloads
    import sq_recovery_b200 as S
    from sq_recovery_b200 import _lib
    from sq_recovery_b200.functional import HostContext

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    steps, warmup = args.steps, max(args.warmup, 3)
    side, side2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    main = Workload("config2", O.SIZE_RANGE, S, O, dev, rank, side, side2)
    dense = Workload("dense", O.DENSE_SIZE_RANGE, S, O, dev, rank, side, side2)
    if not args.eager:
        main.capture()
        dense.capture()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(warmup):
        main.step(i)
    main.run(12)
    # The timed region may last only milliseconds, shorter than nvidia-smi's sampling period, so the same step is
    # also run untimed for ~0.7 s right before it with the sampler on: the clocks / throttle reasons reported are
    # those of this workload under sustained load, and the timed steps follow back to back.
    t_soak = time.perf_counter()
    while time.perf_counter() - t_soak < 0.7:
        main.run(48)
        torch.cuda.synchronize()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    loss, grad = main.run(steps)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    assert torch.isfinite(loss).item() and torch.isfinite(grad).all().item()
    # copied now: later replays of the same graphs overwrite their output buffers
    outputs = {"loss": loss.detach().cpu(), "grad": grad.cpu()}
    # the same K steps one batch at a time (no overlap between consecutive steps)
    main.run(8, sequential=True)
    barrier()
    ev0.record()
    main.run(steps, sequential=True)
    ev1.record()
    barrier()
    seq_ms = ev0.elapsed_time(ev1)
    # the second workload: objects that fill the grid (a ~ U(0.5, 1)), where culling cannot help
    dsteps = max(4, min(steps, 80))
    dense.run(8)
    barrier()
    ev0.record()
    dense_loss, dense_grad = dense.run(dsteps)
    ev1.record()
    barrier()
    dms = ev0.elapsed_time(ev1)
    outputs.update(dense_loss=dense_loss.detach().cpu(), dense_grad=dense_grad.cpu())
    kms = main.kernel_ms(_lib.lib(), min(steps, 20))
    dkms = dense.kernel_ms(_lib.lib(), min(steps, 12))
    eager_ms = None
    if main.graphs:                                         # eager (no graph) step time for comparison
        torch.cuda.synchronize()
        ev0.record()
        for i in range(min(steps, 20)):
            main.eager_step(i)
        ev1.record(); torch.cuda.synchronize()
        eager_ms = ev0.elapsed_time(ev1) / min(steps, 20)
    t = torch.tensor([ms, dms, seq_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, dms, seq_ms = t[0].item(), t[1].item(), t[2].item()

    # ---- e2e: host buffers -> C-ABI host calls -> host results, copies inside the timed region.  Headline: 8-bit depth
    # images (what the reference's data are, torch/test.py:29-30) in pinned memory, several calls in flight on the context's
    # slots (sq_implicit_loss_host_submit / _wait): while one batch is being computed the next ones cross PCIe.
    # Also reported: the blocking fp32-image call of round 1.
    ctx = HostContext(local)
    h_sets = []
    for img, pred in main.sets:
        hu = torch.empty(img.shape, dtype=torch.uint8).pin_memory(); hu.copy_((img * 255.0).round().clamp(0, 255).to(torch.uint8))
        hf = torch.empty(img.shape, dtype=torch.float32).pin_memory(); hf.copy_(img)
        hp = torch.empty(pred.shape, dtype=torch.float32).pin_memory(); hp.copy_(pred)
        # the same targets already at the render size (what F.interpolate would pick: every 4th pixel of every 4th row) -- a data
        # pipeline that resizes once when it builds the dataset ships 1/16 of the bytes
        small = img[:, :, ::H // R, ::W // R].contiguous()
        hs = torch.empty(small.shape, dtype=torch.uint8).pin_memory(); hs.copy_((small * 255.0).round().clamp(0, 255).to(torch.uint8))
        h_sets.append((hu.numpy(), hf.numpy(), hp.numpy(), hs.numpy()))

    # calls in flight (the context has SQ_HOST_SLOTS = 8 slots).  Measured on config 2 (profiles/e2e_depth_r02.txt): 2 -> 105 us per
    # step, 4..6 -> 83 us (the strided copy-engine transfer of the sampled rows alone is 80 us, tools/pcie_probe.cu: the bus is
    # busy all the time), 8 -> 91 us; with pre-resized images (1/16 of the bytes) 8 in flight reach the device-resident pace
    DEPTH = int(os.environ.get("SQ_E2E_DEPTH", 5))
    DEPTH_SMALL = int(os.environ.get("SQ_E2E_DEPTH_SMALL", 8))

    def pipelined(n, which=0, depth=DEPTH):
        """n steps, `depth` in flight; every step: pinned inputs in, loss + gradient out to host memory."""
        for j in range(min(depth - 1, n)):
            ctx.submit_implicit(j % depth, h_sets[j % 4][2], h_sets[j % 4][which], R, TAU, SHARP)
        out = None
        for i in range(n):
            j = i + depth - 1
            if j < n:
                ctx.submit_implicit(j % depth, h_sets[j % 4][2], h_sets[j % 4][which], R, TAU, SHARP)
            out = ctx.result(i % depth)
        return out

    pipelined(12)
    for i in range(3):
        ctx.implicit_loss(h_sets[i % 4][2], h_sets[i % 4][1], R, TAU, SHARP)
    barrier()
    e2e_steps = max(4, steps)
    t0 = time.perf_counter()
    l_h, g_h = pipelined(e2e_steps)
    e2e_s = time.perf_counter() - t0
    barrier()
    f32_steps = min(steps, 20)
    t0 = time.perf_counter()
    for i in range(f32_steps):
        l_f, g_f = ctx.implicit_loss(h_sets[i % 4][2], h_sets[i % 4][1], R, TAU, SHARP)
    f32_s = time.perf_counter() - t0
    pipelined(12, which=3, depth=DEPTH_SMALL)
    barrier()
    t0 = time.perf_counter()
    l_s, g_s = pipelined(e2e_steps, which=3, depth=DEPTH_SMALL)
    small_s = time.perf_counter() - t0
    assert abs(l_s - l_h) <= 1e-12 * abs(l_h) and np.array_equal(g_s, g_h)     # same pixels, same bits
    te = torch.tensor([e2e_s, f32_s, small_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s, f32_s, small_s = te[0].item(), te[1].item(), te[2].item()
    # measured H2D traffic of the same loop (NVML PCIe receive counter, ~1 s of it)
    pcie = None
    if rank == 0:
        ps = PcieSampler(local)
        ps.start()
        t0 = time.perf_counter(); n_soak = 0
        while time.perf_counter() - t0 < 1.0:
            pipelined(64); n_soak += 64
        soak_s = time.perf_counter() - t0
        rate = ps.stop()
        if rate:
            pcie = {"rx_bytes_per_s": rate, "bytes_per_step": rate * soak_s / n_soak, "steps": n_soak,
                    "how": "nvmlDeviceGetPcieThroughput(RX) averaged over ~1 s of the same pipelined loop"}
    with torch.no_grad():                                   # the host paths and the torch path agree
        k_last = (e2e_steps - 1) % 4
        img_u = torch.from_numpy(h_sets[k_last][0]).to(dev).float() * np.float32(1.0 / 255.0)
        l_t = main.crit(img_u, main.sets[k_last][1]).item()
        assert abs(l_h - l_t) <= 1e-6 * abs(l_t) and np.isfinite(g_h).all(), (l_h, l_t)
        l_t = main.crit(*main.sets[(f32_steps - 1) % 4]).item()
        assert abs(l_f - l_t) <= 1e-6 * abs(l_t) and np.isfinite(g_f).all(), (l_f, l_t)
    ctx.close()

    if rank == 0:
        pts = B * R ** 3
        value = world * pts * steps / (ms * 1e-3) / 1e9
        peak = measured_mufu_peak()
        clock = clocks["sm_mhz"] or peak["sm_mhz"]
        ncu = ncu_summary()
        try:
            c_main, c_dense = main.counts(), dense.counts()
        except Exception as e:      # the counting build is optional evidence, not part of the product path
            c_main = c_dense = None
            print(f"counting build unavailable: {e}", file=sys.stderr)
        roof = roofline_block(kms, c_main, peak, ncu, pts, clock)
        roof["traffic"] = ncu["dram_bytes_per_launch"] if ncu else None
        roof["ncu"] = {"file": ncu.get("file"), "xu_warp_inst_per_launch": ncu.get("xu_warp_inst_per_launch"),
                       "warp_inst_per_launch": ncu.get("warp_inst_per_launch")} if ncu else None
        roof["how"] = ("achieved = MUFU-pipe (XU) thread-ops the kernel ISSUES per launch / live CUDA-event kernel time (events "
                       "around the launch, eager: includes ~3 us of launch latency).  Issued ops = events counted by the "
                       "counting build of the same sources (libsqloss_count.so) on these inputs x the per-event MUFU cost read "
                       "off the kernel source (sq_recovery_b200/counting.py); the committed ncu capture holds the hardware count "
                       "for comparison.  The kernel skips grid points whose occupancy is below 2^-32, stops a column once its "
                       "transmittance is gone and evaluates F with 8 MUFU ops instead of 10, so issued ops are far fewer than "
                       "the reference algorithm's 16 per grid point (`reference_algorithm_equivalent`)")
        roof["peak_source"] = (f"{peak['source']}: {peak['mufu_per_clk_sm']:.2f} MUFU/clk/SM x {peak['sms']} SMs x "
                               f"{peak['sm_mhz']:.0f} MHz (measured)")
        droof = roofline_block(dkms, c_dense, peak, None, pts, clock)
        h2d_u8 = B * R * W + B * 12 * 4        # the sampled rows + parameters (the offset tables stay on the device)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(world),
            "launch": ("CUDA graph replay, four steps (one per input set) per graph launch, TWO independent batches in flight "
                       "(the steps alternate between two streams inside the graph)") if main.graphs else "eager",
            "one_batch_at_a_time": {"value": world * pts * steps / (seq_ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": seq_ms / steps,
                                    "note": "the same K steps with consecutive steps serialised on one stream (round 1's protocol)"},
            "eager_ms_per_step": eager_ms,
            "walked_fraction": roof["walked_fraction"], "evaluated_gpoints_per_s": roof["evaluated_gpoints_per_s"],
            "clocks": clocks,
            "e2e": {"value": world * pts * e2e_steps / e2e_s / 1e9, "unit": UNIT,
                    # of the pinned 8-bit depth maps only the sampled rows cross the bus (every 4th row of a 256 x 256 image, all of
                    # its 256 bytes), as one strided copy-engine transfer per call
                    "h2d_bytes_per_step": h2d_u8, "d2h_bytes_per_step": 8 + B * 12 * 4,
                    "h2d_bytes_per_step_measured": pcie["bytes_per_step"] if pcie else None, "pcie": pcie,
                    "host_image_bytes": B * H * W, "steps": e2e_steps, "ms_per_step": e2e_s / e2e_steps * 1e3,
                    "api": "sq_implicit_loss_host_submit / _wait (include/sqloss.h): uint8 depth images and fp32 parameters in "
                           f"pinned host memory, loss + gradient back to host memory every step, {DEPTH} calls in flight",
                    "calls_in_flight": DEPTH,
                    "pre_resized_u8_images": {"value": world * pts * e2e_steps / small_s / 1e9, "ms_per_step": small_s / e2e_steps * 1e3,
                                              "h2d_bytes_per_step": B * R * R + B * 12 * 4, "calls_in_flight": DEPTH_SMALL,
                                              "note": f"the same call on depth maps stored at the render size ({R}x{R} uint8: the pixels the "
                                                      "nearest resize would pick): 1/16 of the bytes, the step is then bound by the kernels"},
                    "blocking_f32_images": {"value": world * pts * f32_steps / f32_s / 1e9, "ms_per_step": f32_s / f32_steps * 1e3,
                                            "h2d_bytes_per_step": B * R * min(W * 4, R * 32) + B * 12 * 4 + 4 * R * 4,
                                            "api": "sq_implicit_loss_host, fp32 images, one call at a time (round 1's e2e)"}},
            "gpu_launches": 3 * steps,
            "roofline": roof,
            "dense": {"workload": f"same call, sizes a ~ U{O.DENSE_SIZE_RANGE} (objects fill the grid; BASELINE config 2 draws "
                                  f"a ~ U{O.SIZE_RANGE})", "value": world * pts * dsteps / (dms * 1e-3) / 1e9, "unit": UNIT,
                      "steps": dsteps, "ms_per_step": dms / dsteps, "roofline": droof},
        }
        if world == 1:
            line["cpu_baseline"] = cpu_reference(5, 1)[0]
        print(json.dumps(line), flush=True)
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        suffix = f"_rank{rank}" if world > 1 else ""
        for name, t in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + suffix + ".npy"), t.numpy())
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--eager", action="store_true", help="time eager launches instead of CUDA-graph replay")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's loss and gradient as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path only")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
