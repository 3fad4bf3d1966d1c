"""The offset heads' 3x3 convolutions (ofsMap / ofs_residual, nn.Conv2d(256, 98, 3, padding=1)) on one GPU: forward
(fprop), input gradient (dgrad) and weight + bias gradient (wgrad), each timed separately.

  lib        ops.conv3x3 / ops.conv3x3_backward (tcgen05 kind::tf32, 3-term split, fp32 accuracy), packing included
  cudnn      F.conv2d and its autograd pieces in fp32 with TF32 off (what training runs today)
  cudnn_tf32 the same with TF32 on (~1e-3 relative: below this project's accuracy bars; for reference only)

All arms run alternately in one process on the same inputs, warmed up, with CUDA events around each call.  At E = 96 the
48x64 input alone is 302 MB, larger than the 126 MB L2.  TFLOP/s is on the algorithmic 2*E*H*W*C_out*C_in*9 FLOPs per
product; "share" counts three tf32 MMAs per product against the data sheet's 1,125 TFLOP/s dense TF32 (a share of that
figure, not of a measured peak).  Max errors against F.conv2d / autograd in float64 at E = 3.  The GPU's name, power limit
and max SM clock are printed first.

    python tools/bench_offset_conv.py [--edges 48,96] [--iters 20] [--warmup 3]

Prints one JSON line per (edges, grid).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

TF32_DENSE_TFLOPS = 1125.0
C_IN, C_OUT = 256, 98
GRIDS = [(48, 64), (24, 32)]


def flops(E, H, W):
    return 2.0 * E * H * W * C_OUT * C_IN * 9


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"nvidia-smi unavailable: {e}"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--edges", default="48,96")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()

    import torch
    import torch.nn.functional as F
    import lgu_slam_b200  # noqa: F401
    from importlib import import_module
    ops = import_module("lgu-slam_b200.ops")
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing measured")
    dev = torch.device("cuda:0")
    print(json.dumps({"gpu": gpu_info(), "torch": torch.__version__}), flush=True)

    def inputs(E, H, W, seed):
        g = torch.Generator(device=dev).manual_seed(seed)
        x = torch.randn(E, C_IN, H, W, generator=g, device=dev)
        w = (torch.rand(C_OUT, C_IN, 3, 3, generator=g, device=dev) * 2 - 1) / 48
        b = (torch.rand(C_OUT, generator=g, device=dev) * 2 - 1) / 48
        gy = torch.randn(E, C_OUT, H, W, generator=g, device=dev)
        return x, w, b, gy

    def cudnn_arms(tf32):
        def run(fn):
            def go(*args):
                prev = torch.backends.cudnn.allow_tf32
                torch.backends.cudnn.allow_tf32 = tf32
                try:
                    return fn(*args)
                finally:
                    torch.backends.cudnn.allow_tf32 = prev
            return go
        return {
            "fprop": run(lambda x, w, b, gy: F.conv2d(x, w, b, padding=1)),
            "dgrad": run(lambda x, w, b, gy: torch.nn.grad.conv2d_input(x.shape, w, gy, padding=1)),
            "wgrad": run(lambda x, w, b, gy: (torch.nn.grad.conv2d_weight(x, w.shape, gy, padding=1), gy.sum((0, 2, 3)))),
        }

    arms = {
        "lib": {
            "fprop": lambda x, w, b, gy: ops.conv3x3(x, w, b),
            "dgrad": lambda x, w, b, gy: ops.conv3x3_backward(x, w, gy, True, False, False)[0],
            "wgrad": lambda x, w, b, gy: ops.conv3x3_backward(x, w, gy, False, True, True)[1:],
        },
        "cudnn": cudnn_arms(False),
        "cudnn_tf32": cudnn_arms(True),
    }

    # accuracy at E = 3 against float64, per arm and product
    errors = {}
    for H, W in GRIDS:
        x, w, b, gy = inputs(3, H, W, 7)
        xd, wd, bd = (t.double().requires_grad_() for t in (x, w, b))
        y = F.conv2d(xd, wd, bd, padding=1)
        rgx, rgw, rgb = torch.autograd.grad(y, (xd, wd, bd), gy.double())
        ref = {"fprop": y.detach(), "dgrad": rgx, "wgrad": rgw}
        for arm, fns in arms.items():
            for prod, fn in fns.items():
                got = fn(x, w, b, gy)
                got = got[0] if isinstance(got, tuple) else got
                r = ref[prod]
                errors[(arm, prod, H)] = (got.double() - r).abs().max().item() / max(1.0, r.abs().max().item())
        del x, w, b, gy, xd, wd, bd, y, rgx, rgw, rgb, ref
    torch.cuda.empty_cache()

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)                                # ms

    for E in [int(v) for v in a.edges.split(",")]:
        for H, W in GRIDS:
            x, w, b, gy = inputs(E, H, W, 1000 + E)
            args = (x, w, b, gy)
            ts = {(arm, prod): [] for arm in arms for prod in arms[arm]}
            for _ in range(a.warmup):
                for arm, fns in arms.items():
                    for fn in fns.values():
                        fn(*args)
            torch.cuda.synchronize()
            for _ in range(a.iters):                              # alternate arms and products, one call each
                for arm, fns in arms.items():
                    for prod, fn in fns.items():
                        ts[(arm, prod)].append(timed(lambda: fn(*args)))
            fl = flops(E, H, W)
            res = {"edges": E, "grid": [H, W], "GFLOP_per_product": round(fl / 1e9, 1)}
            for (arm, prod), t in ts.items():
                ms = statistics.median(t)
                tfs = fl / (ms * 1e-3) / 1e12
                res[f"{arm}_{prod}_ms"] = round(ms, 3)
                res[f"{arm}_{prod}_ms_spread"] = [round(min(t), 3), round(max(t), 3)]
                res[f"{arm}_{prod}_TFLOPs"] = round(tfs, 1)
                if arm == "lib":
                    res[f"{arm}_{prod}_share_of_1125_tf32_x3"] = round(3 * tfs / TF32_DENSE_TFLOPS, 3)
                res[f"{arm}_{prod}_max_rel_err_E3"] = errors[(arm, prod, H)]
            for arm in arms:
                res[f"{arm}_total_ms"] = round(sum(res[f"{arm}_{p}_ms"] for p in ("fprop", "dgrad", "wgrad")), 3)
            print(json.dumps(res), flush=True)
            del x, w, b, gy, args
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
