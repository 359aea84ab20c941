"""Build variants of libsqloss.so with different -D tunables on the GPU box and time the column kernels.

    python tools/tune.py "" "SQ_IMPB_MINB=4" "SQ_IMPB_MINB=4,SQ_BWD_DEPTH=16" ...

Each variant is compiled to /tmp and loaded with ctypes next to torch (no package import, so several variants can
coexist in one process).  Prints one line per variant: kernel-only ms (sq_profile_events) for the implicit fwd+bwd,
implicit fwd, explicit fwd+bwd and IoU kernels on BASELINE config 2 (B=256, R=64).
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from sq_recovery_b200 import inputs as O      # seeded randsq / randquat workloads
from sq_recovery_b200 import _lib as L0     # prototypes

B, R = int(os.environ.get("SQ_B", 256)), 64
dev = torch.device("cuda:0")


def build(defs):
    tag = defs.replace("=", "").replace(",", "_").replace("/", "_") or "default"
    out = f"/tmp/libsq_{tag}.so"
    # "SRC=<dir>" among the definitions: build <dir>/sqloss.cu instead (A/B of two source trees on the same box)
    src_dir = next((d[4:] for d in defs.split(",") if d.startswith("SRC=")), os.path.join("sq_recovery_b200", "csrc"))
    cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-ftz=true", "-std=c++17", "-shared",
           "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-I", os.path.join(ROOT, "include"), "-o", out, os.path.join(ROOT, src_dir, "sqloss.cu")]
    cmd += [f"-D{d}" for d in defs.split(",") if d and not d.startswith("SRC=")]
    log = subprocess.run(cmd, capture_output=True, text=True)
    if log.returncode:
        print(log.stderr[-2000:]); raise SystemExit(1)
    regs = {}
    lines = log.stderr.splitlines()
    for i, l in enumerate(lines):
        if "Compiling entry function" in l:
            name = "imp_bwd" if "implicit_kernelILb1" in l else "imp_fwd" if "implicit_kernelILb0" in l else \
                   "exp_bwd" if "explicit_kernelILb1" in l else "iou" if "iou_kernel" in l else None
            if name:
                txt = " ".join(lines[i + 1:i + 5])
                r = txt.split("Used ")[1].split(" registers")[0] if "Used " in txt else "?"
                sp = txt.split("bytes stack frame, ")[1].split(" bytes spill stores")[0] if "spill stores" in txt else "0"
                regs[name] = f"{r}r/{sp}sp"
    h = ctypes.CDLL(out)
    for name, (res, args) in L0._PROTOS.items():
        fn = getattr(h, name); fn.restype, fn.argtypes = res, args
    return h, regs


def timed(h, launch, iters=20):
    ms = []
    for i in range(iters + 3):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); b.record(); torch.cuda.synchronize()
        h.sq_profile_events(a.cuda_event, b.cuda_event)
        launch()
        torch.cuda.synchronize()
        if i >= 3:
            ms.append(a.elapsed_time(b))
    return float(np.median(ms)), float(np.min(ms))


def main():
    import sq_recovery_b200 as S
    from sq_recovery_b200.functional import nearest_offsets
    true = O.random_params(B, 0)
    pred = O.perturbed_params(true, 7)
    if os.environ.get("SQ_SORT"):            # experiment: heaviest samples (largest clamped volume) first / last
        vol = pred[:, 0].clamp(0.05, 1) * pred[:, 1].clamp(0.05, 1) * pred[:, 2].clamp(0.05, 1)
        order = torch.argsort(vol, descending=os.environ["SQ_SORT"] == "desc")
        true, pred = true[order].contiguous(), pred[order].contiguous()
    true, pred = true.to(dev), pred.to(dev)
    img = S.ImplicitLoss(256, dev, 1.5, 260).depth_projection(true).unsqueeze(1).contiguous()
    row_off, col_off = nearest_offsets(256, 256, R, dev)
    loss = torch.empty((), dtype=torch.float64, device=dev)
    grad = torch.empty_like(pred)
    cnt = torch.empty((2, B), dtype=torch.int64, device=dev)
    P = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
    st = torch.cuda.current_stream().cuda_stream
    ref = None
    for defs in (sys.argv[1:] or [""]):
        h, regs = build(defs)
        nb = h.sq_scratch_bytes(B, R + 1)
        scratch = torch.zeros(nb, dtype=torch.uint8, device=dev)
        def imp(g):
            rc = h.sq_implicit_loss(P(pred), 0, B, R, 1.0 / (R - 1), 1e-4, P(img), 256 * 256, P(row_off), P(col_off), 1.5, 260.0,
                                    P(loss), None, P(g), None, P(scratch), nb, st)
            assert rc == 0, rc
        def exp(g):
            rc = h.sq_explicit_loss(P(true), P(pred), 0, B, R + 1, 1.0 / R, 1e-4, 5.0, 100.0, P(loss), None, P(g), P(scratch), nb, st)
            assert rc == 0, rc
        def iou():
            rc = h.sq_iou_counts(P(true), P(pred), 0, B, R, 1.0 / (R - 1), 0.0, P(cnt[0]), P(cnt[1]), P(scratch), nb, st)
            assert rc == 0, rc
        # back-to-back calls (plan + column + finalize kernels) between one event pair: resolves 0.1 us differences,
        # which single CUDA-event readings (0.5-1 us granularity) do not
        for _ in range(20):
            imp(grad)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        for _ in range(400):
            imp(grad)
        e1.record(); torch.cuda.synchronize()
        call_us = e0.elapsed_time(e1) / 400 * 1e3
        # the same three kernels replayed from a CUDA graph (no launch gaps from the host)
        graph_us = float("nan")
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                st_side = side.cuda_stream
                def imp_side():
                    rc = h.sq_implicit_loss(P(pred), 0, B, R, 1.0 / (R - 1), 1e-4, P(img), 256 * 256, P(row_off), P(col_off), 1.5, 260.0,
                                            P(loss), None, P(grad), None, P(scratch), nb, st_side)
                    assert rc == 0, rc
                imp_side(); imp_side()
                side.synchronize()
                gph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gph, stream=side):
                    rc = h.sq_implicit_loss(P(pred), 0, B, R, 1.0 / (R - 1), 1e-4, P(img), 256 * 256, P(row_off), P(col_off), 1.5, 260.0,
                                            P(loss), None, P(grad), None, P(scratch), nb, torch.cuda.current_stream().cuda_stream)
                    assert rc == 0, rc
            torch.cuda.current_stream().wait_stream(side)
            for _ in range(20):
                gph.replay()
            torch.cuda.synchronize(); e0.record()
            for _ in range(400):
                gph.replay()
            e1.record(); torch.cuda.synchronize()
            graph_us = e0.elapsed_time(e1) / 400 * 1e3
        except Exception as exc:      # keep the tool usable if capture fails for a variant
            print("graph capture failed:", exc)
        t_ib = timed(h, lambda: imp(grad))
        chk = (loss.item(), grad.double().abs().sum().item())
        if ref is None:
            ref = chk
        t_if = timed(h, lambda: imp(None))
        t_eb = timed(h, lambda: exp(grad))
        t_io = timed(h, iou)
        pts = B * R ** 3
        print(f"{defs or 'default':40s} call {call_us:6.2f}us graph {graph_us:6.2f}us imp_bwd {t_ib[0]*1e3:7.1f}us ({pts/t_ib[0]/1e6:6.1f} Gpt/s) imp_fwd {t_if[0]*1e3:7.1f}us "
              f"exp_bwd {t_eb[0]*1e3:7.1f}us iou {t_io[0]*1e3:7.1f}us  regs {regs}  same={abs(chk[0]-ref[0])<1e-9 and abs(chk[1]-ref[1])<1e-6*ref[1]}",
              flush=True)


if __name__ == "__main__":
    main()
