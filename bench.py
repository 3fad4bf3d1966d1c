#!/usr/bin/env python
"""bench.py -- correlation edges/sec of the LGU-SLAM hot path on B200 (BASELINE.json metric).

N = 1 -- config.workload = "frontend_w20_e48": BASELINE.json configs[1], the frontend window of 20 keyframes with
E = 48 factor-graph edges on 48x64x128 feature maps (droid_frontend.py:13 max_factors=48), 4-level pyramid, r = 3
deformable lookup + Gaussian weighting, forward + backward.  One STEP is one pass of the hot path over that edge batch
(SURVEY.md section 8d's composite: build fwd + lookup fwd + lookup bwd + gaussian bwd):

    pack      fmaps [T,128,48,64] -> channels-last fp16 planes            (1 launch, ours)
    build     all-pairs volume + Gaussian residual + 4-level pyramid       (1 launch, tcgen05/TMA, ours)
    lookup    r=1 mask lookup on level 1 -> var -> sigmoid -> offset[1] *= mask -> 4 x deformable r=3 lookups -> cat
              (CorrBlock.__call__, corr.py:88-109)                         (1 launch, TMA-staged, ours)
    lookup^T  backward of the above: dense gradients of all 4 pyramid levels (mask path folded into level 1)
              + offset gradients of levels 0-1                             (1 launch, ours)
    gauss^T   Gaussian-head gradients (means, covs, den) straight from those four level gradients -- what autograd runs
              for gaussianMask_cuda.py:84-86 behind 3 x avg_pool2d (gaussianAttn.cu:72-131)   (1 launch, ours)
The feature-map gradients of the build (matmul backward) are not part of section 8d's composite; they are timed
beside the step (`extra_ops.build_bwd_fmaps`), as is the drop-in `gaussianMask_backward` operator.

`value` = E / step time with every input resident in HBM (CUDA events); `e2e` = the same step driven from pinned HOST
buffers: per-step inputs (coords, upstream gradient) go H2D and every result goes D2H inside the timed region; what a
caller keeps resident between steps (feature maps, offset / Gaussian head outputs, edge lists) stays on the device.

N > 1 (torchrun) -- config.workload = "backend_t256_e4096_sharded": BASELINE.json configs[3], global-BA correlation over
T = 256 keyframes and 4096 edges, STRONG scaling: the reference's chunks of 8 source frames (factor_graph.py:272-279) are
partitioned over the ranks; one STEP = one backend pass with everything that crosses GPUs inside the timed region:
all-gather of the fp16 keyframe maps (NCCL) -> per-rank pyramid (AltCorrBlock) -> per chunk: offset heads, four
tcgen05 volumes, fused per-corner-gated lookup -> per-edge outputs RETURNED TO RANK 0 through NVLink peer stores
(sharded.PeerOutput: the lookup kernels write their rows straight into rank 0's buffer).  `value` = edges / step time
(max over ranks) with outputs returned as fp16 (what update_op reads under autocast); outputs left sharded, returned
as fp32, and the same step on ONE GPU of the same job (for the strong-scaling ratio) are reported under "backend".

`--impl reference` times the CPU oracle port (oracle/lgu_oracle.c, OpenMP over all host threads) on the same workload
the chosen N selects; the reference ships no CPU implementation of this path (CUDA only), so the port is the CPU arm
("kind": "port").  The reference's own CUDA kernels recompiled for sm_100 (oracle/_ref) are timed beside ours when present
and reported under "ref_cuda" for information.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
sys.dont_write_bytecode = True          # the benchmark may run from a read-only tree: no __pycache__ beside the sources

H, W, C, R, LEVELS, GR = 48, 64, 128, 3, 4, 4
P = H * W
QS = [P >> (2 * l) for l in range(LEVELS)]
TAPS = (2 * R + 1) ** 2
METRIC = "correlation edges/sec (48x64, 4 lvl, r=3, deformable+Gaussian) fwd+bwd"
# The Gaussian head's backward reads the level gradients only inside its 9 x 9 window.  LGU_BENCH_GAUSS selects how:
#   fused  (default) the fused lookup backward forms that window from its shared-memory accumulators and finishes the
#          Gaussian head's gradients in the same launch (lgu_corr_lookup_fused_backward_gauss);
#   window the fused backward emits the window as a contiguous record, a second kernel consumes it
#          (lgu_corr_lookup_fused_backward_win + lgu_build_backward_gauss_window);
#   levels a second kernel gathers the window from the four dense level gradients (lgu_build_backward_gauss: the form a
#          multi-lookup training step uses).  All three give the same bits (tests/test_fused_lookup_gpu.py).
GAUSS_MODE = os.environ.get("LGU_BENCH_GAUSS", "fused")       # fused | window | levels
GAUSS_WINDOW = GAUSS_MODE == "window"
GAUSS_FUSED = GAUSS_MODE == "fused"


def algorithmic_bytes_per_edge():
    """SURVEY.md section 8(d): compulsory HBM bytes per edge of each op (fp32 tensors, fp16 packed fmaps)."""
    gather = [TAPS * 16, TAPS * 16, 64 * 4, 64 * 4]          # deformed levels 0-1: 4 corners/tap; zero-offset 2-3: 8x8 patch
    return {
        "pack": C * P * 2 + C * P * 2,                        # read fp16 NCHW + write fp16 NHWC (per frame, ~per edge)
        "build": 2 * P * C * 2 + 16 * P + 4 * P * sum(QS),
        # fused 4-level lookup, cumulative-mask form: coords, offsets of levels 0-1 (read only), the per-pixel running
        # mask (read + write), gathers (incl. the 16 corners of the r=1 mask lookup), 196-ch output
        "lookup_fwd": P * (8 + 2 * 8 * TAPS + 8 + sum(gather) + 64 + 4 * LEVELS * TAPS),
        # fused backward: coords, 2 offset records + mask, 196-ch upstream grad, level-0/1 gathers (+ mask taps),
        # dense gradient slices of all 4 levels written once, 2 offset-gradient records
        # ... plus the Gaussian head's part: folded in ("fused": the 81-tap window of lvl0 and 5 parameter floats in, 5
        # gradient floats out) or prepared for a second kernel ("window": the window centres in, an 81-float record out)
        "lookup_bwd": P * (8 + 2 * 8 * TAPS + 4 + 4 * LEVELS * TAPS + gather[0] + gather[1] + 64 + 4 * sum(QS)
                           + 2 * 8 * TAPS + (81 * 4 + 40 if GAUSS_FUSED else 8 + 81 * 4 if GAUSS_WINDOW else 0)),
        # Gaussian-head gradients as a kernel of their own: the 81-tap window of lvl0, 5 parameter floats in, 5 gradient
        # floats out, and EITHER the 81-float window record of the merged level-0 gradient that the fused backward emitted,
        # OR (from the level gradients) the 81-tap window of g0 and its 2x2 / 4x4 / 8x8 parents in g1..g3 (25 + 9 + 4 taps)
        "gauss_bwd": 0 if GAUSS_FUSED else P * (2 * 81 * 4 + 40) if GAUSS_WINDOW else P * (2 * 81 * 4 + (25 + 9 + 4) * 4 + 40),
    }


def pin_to_gpu_numa(index):
    """Pin this process to the CPU cores NVML reports as local to GPU `index` (its NUMA node), so that pinned host
    buffers and the launch thread of every rank sit next to their own GPU instead of all on node 0."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = (ncpu + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0)) or cpus
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"{len(cpus)} cores local to GPU {index}"
    except Exception as ex:
        return f"not pinned ({type(ex).__name__})"
    return "not pinned"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.max_mhz, self.stop_flag, self.ok = [], set(), None, False, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.005)

    def result(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


DUMP_BYTES = 64_000_000                 # --dump-outputs writes at most this much in all
DUMP_SEED = 0


def dump_outputs(out_dir, results):
    """Write each result as out_dir/<name>.npy in float32.  The arrays share DUMP_BYTES equally; one with more entries
    than its share is written as a 1-D sample: the entries of its flattened form at sorted positions drawn without
    replacement by numpy.random.default_rng(DUMP_SEED), the same positions on every run with the same arguments."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    cap = (DUMP_BYTES - 4096 * len(results)) // (4 * len(results))      # 4096: room for each .npy header
    for name, t in results.items():
        a = t.detach().float().cpu().numpy()
        if a.size > cap:
            a = a.reshape(-1)[np.sort(np.random.default_rng(DUMP_SEED).choice(a.size, cap, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def load_peak():
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    return peak, src


# ------------------------------------------------------------------------------------------------ frontend (N = 1)
def make_host_inputs(E, T, seed, pin):
    import torch
    import inputs
    c = inputs.frontend_case(E=E, T=T, H=H, W=W, C=C, seed=seed, half_fmaps=True)
    g = inputs.gen(seed + 7)
    host = dict(
        fmaps=c["fmaps"].half().contiguous(),                      # fp16 frame buffer (depth_video.py:36)
        ii=c["ii"], jj=c["jj"], means=c["means"], covs=c["covs"],
        den=(6.28 * torch.sqrt(c["covs"][..., 0] * c["covs"][..., 1])).contiguous(),
        coords=c["coords"], off0=c["offsets"][0], off1=c["offsets"][1],
        corr_grad=torch.randn(E, LEVELS * TAPS, H, W, generator=g),
    )
    if pin:
        host = {k: v.pin_memory() for k, v in host.items()}
    return host


class Workload:
    """The frontend-window step on one GPU, through the package's public operator API."""

    PER_STEP_INPUTS = ("coords", "corr_grad")                     # everything else stays resident between steps
    RESULT_KEYS = ("corr", "offset_grad0", "offset_grad1", "means_grad", "covs_grad", "den_grad")

    def __init__(self, E, T, seed, device):
        import torch
        import lgu_slam_b200
        self.torch, self.ops, self.lib, self.E, self.T, self.dev = torch, lgu_slam_b200.ops, lgu_slam_b200._lib, E, T, device
        self.host = make_host_inputs(E, T, seed, pin=True)
        self.d = {k: v.to(device) for k, v in self.host.items()}
        self.cum = torch.ones(E, H, W, device=device)
        self.launches_per_step = None

    def step(self, d=None, record=None):
        torch, ops = self.torch, self.ops
        d = d or self.d

        def mark(name):
            if record is not None:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                record.append((name, e))

        n0 = self.lib.LAUNCHES
        mark("start")
        hi, _ = ops.pack_fmaps(d["fmaps"])
        self.cum.fill_(1.0)                                        # state of a freshly built block: no mask applied yet
        mark("pack")
        pyr = ops.build_pyramid(hi, None, d["ii"], d["jj"], H, W, means=d["means"], covs=d["covs"], den=d["den"],
                                num_levels=LEVELS, gauss_radius=GR, precision=1)
        mark("build")
        # ---- CorrBlock.__call__ (corr.py:88-109): one fused TMA-staged launch (mask lookup + 4 deformable levels); the
        # block's cumulative offset[1] mask (Q7) lives in a per-pixel buffer, offset[1] itself stays pristine
        corr, mask = ops.corr_lookup_fused(pyr, d["coords"], d["off0"], d["off1"], R, return_mask=True, cum_mask=self.cum)
        mark("lookup_fwd")
        # ---- its backward (what autograd runs for corr.py:88-109): one launch, dense gradients of all 4 levels; the
        # post-mask offsets offset[1] * cum_mask are formed in registers, as in the forward
        # ---- ... and the Gaussian-head gradients of the build (gaussianMask_cuda.py:77-86 backward through corr.py:83-86)
        if GAUSS_FUSED:
            grads = ops.corr_lookup_fused_backward(pyr, d["coords"], d["off0"], d["off1"], mask, d["corr_grad"],
                                                   cum_mask=self.cum, gauss_head=(d["means"], d["covs"], d["den"]))
            gm, gc, gd = grads[6:9]
            mark("lookup_bwd")
        else:
            grads = ops.corr_lookup_fused_backward(pyr, d["coords"], d["off0"], d["off1"], mask, d["corr_grad"],
                                                   cum_mask=self.cum, gauss_window_means=d["means"] if GAUSS_WINDOW else None)
            mark("lookup_bwd")
            gm, gc, gd = ops.build_backward_gauss(d["means"], d["covs"], d["den"], pyr[0], list(grads[:4]), GR,
                                                  window=grads[6] if GAUSS_WINDOW else None)
            mark("gauss_bwd")
        if self.launches_per_step is None:
            self.launches_per_step = self.lib.LAUNCHES - n0
        return dict(corr=corr, offset_grad0=grads[4], offset_grad1=grads[5], means_grad=gm, covs_grad=gc, den_grad=gd,
                    _keep=(grads, pyr))

    # ---- ops timed beside the step
    def extra_ops(self, iters=5):
        """build_backward_fmaps (feature-map gradients of the build, tcgen05 kind::tf32) and the drop-in
        gaussianMask_backward operator on a dense raw volume, timed with CUDA events on the step's tensors."""
        torch, ops, d, E = self.torch, self.ops, self.d, self.E
        out = self.step()
        grads = list(out["_keep"][0][:4])
        f = d["fmaps"].float()
        f1, f2 = f[d["ii"].long()].contiguous(), f[d["jj"].long()].contiguous()
        hi, _ = ops.pack_fmaps(d["fmaps"])
        v_raw = ops.build_pyramid(hi, None, d["ii"], d["jj"], H, W, num_levels=1, gauss_radius=0)[0]
        res = {}
        for name, fn in (("build_bwd_fmaps", lambda: ops.build_backward_fmaps(grads, f1, f2)),
                         ("gaussianMask_backward_dropin",
                          lambda: ops.gaussianMask_backward(d["means"], d["covs"], v_raw, grads[0], GR))):
            fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                fn()
            e1.record()
            torch.cuda.synchronize()
            res[name] = {"ms": round(e0.elapsed_time(e1) / iters, 4)}
        res["build_bwd_fmaps"]["what"] = ("g_f1, g_f2 from the 4 level gradients (tf32 split operands + 2 tcgen05 launches); "
                                          "reads 2 x 50.1 MB/edge")
        res["gaussianMask_backward_dropin"]["alg_MB_per_edge"] = round(P * (2 * 81 * 4 + 32) / 1e6, 3)
        return res

    def e2e_setup(self):
        """Two device sets of the per-step inputs and two pinned result sets so that step i+1's H2D, step i's kernels and
        step i-1's D2H overlap on three streams (copies run on the two DMA engines, full duplex)."""
        torch = self.torch
        self.s_in, self.s_out = torch.cuda.Stream(self.dev), torch.cuda.Stream(self.dev)
        self.dsets = []
        for _ in range(2):
            ds = dict(self.d)                                       # resident tensors are shared, per-step ones are private
            for k in self.PER_STEP_INPUTS:
                ds[k] = torch.empty_like(self.d[k])
            self.dsets.append(ds)
        out = self.step()
        self.hres = [{k: torch.empty(out[k].shape, dtype=out[k].dtype).pin_memory() for k in self.RESULT_KEYS}
                     for _ in range(2)]
        self.ev_in = [torch.cuda.Event() for _ in range(2)]
        self.ev_comp = [torch.cuda.Event() for _ in range(2)]
        self.ev_out = [torch.cuda.Event() for _ in range(2)]
        self.live = [None, None]
        self.e2e_i = 0
        torch.cuda.synchronize()

    def step_e2e(self):
        """The same step driven from pinned HOST buffers: H2D of this step's inputs, the kernels, D2H of every result a
        caller consumes (corr, offset / mean / cov / den gradients) into pinned host memory.  Returns the host result set
        of the step that has just COMPLETED (two steps back), i.e. the call blocks on that step's D2H."""
        torch = self.torch
        i = self.e2e_i
        b = i & 1
        cur = torch.cuda.current_stream(self.dev)
        with torch.cuda.stream(self.s_in):
            self.s_in.wait_event(self.ev_comp[b])               # set b was last read by the kernels of step i-2
            for k in self.PER_STEP_INPUTS:
                self.dsets[b][k].copy_(self.host[k], non_blocking=True)
            self.ev_in[b].record(self.s_in)
        cur.wait_event(self.ev_in[b])
        out = self.step(self.dsets[b])
        self.ev_comp[b].record(cur)
        self.ev_out[b].synchronize()                            # host result set b (step i-2) has landed: "read" it
        done = self.hres[b] if i >= 2 else None
        with torch.cuda.stream(self.s_out):
            self.s_out.wait_event(self.ev_comp[b])
            for k in self.RESULT_KEYS:
                self.hres[b][k].copy_(out[k], non_blocking=True)
            self.ev_out[b].record(self.s_out)
        self.live[b] = out                                      # keep the device results alive until their D2H is done
        self.e2e_i += 1
        return done

    def e2e_drain(self):
        self.torch.cuda.synchronize()

    def e2e_bytes(self):
        h2d = sum(self.host[k].numel() * self.host[k].element_size() for k in self.PER_STEP_INPUTS)
        d2h = sum(v.numel() * v.element_size() for v in self.hres[0].values())
        return h2d, d2h


def time_ref_cuda(wl, iters=3):
    """The same step on the reference's OWN kernels recompiled unmodified for sm_100 (oracle/_ref, built in the dev
    container from /root/reference/offersample_LGS) + the torch glue the reference uses (corr.py:61-109).  Reported
    under "ref_cuda" beside our numbers; never part of the product path or of `value`."""
    import torch
    from oracle import build_ref
    ref = build_ref.load_ref("defCorrSample_ref")
    if ref is None:
        return None
    d, E = wl.d, wl.E
    f = d["fmaps"].float()
    zero_off = torch.zeros(E, H, W, 2 * TAPS, device=wl.dev)
    zero_off2 = torch.zeros(E, H, W, 2 * TAPS, device=wl.dev)
    g = torch.Generator(device=wl.dev)
    g.manual_seed(7)
    g_mask = torch.randn(E, 3, 3, H, W, device=wl.dev, generator=g)   # upstream grad of the r=1 mask lookup
    hi, _ = wl.ops.pack_fmaps(d["fmaps"])
    v_raw = wl.ops.build_pyramid(hi, None, d["ii"], d["jj"], H, W, num_levels=1, gauss_radius=0)[0]
    g_vol = torch.randn(E, H, W, H, W, device=wl.dev, generator=g)

    def step():
        f1 = f[d["ii"].long()].reshape(E, C, P) / 4
        f2 = f[d["jj"].long()].reshape(E, C, P) / 4
        v = torch.matmul(f1.transpose(1, 2), f2).view(E, H, W, H, W)
        v1, = ref.gaussianMask(d["means"], d["covs"], v, GR)
        cur = (v1 / d["den"].view(E, H, W, 1, 1) + v).reshape(E * P, 1, H, W)
        pyr = []
        for i in range(LEVELS):
            pyr.append(cur.view(E, H, W, H >> i, W >> i))
            cur = torch.nn.functional.avg_pool2d(cur, 2, stride=2)
        c = d["coords"].permute(0, 3, 1, 2).contiguous()
        cl = [(c / 2 ** l).contiguous() for l in range(LEVELS)]
        m, = ref.corr_index_forward(pyr[1], cl[1], 1)
        mask = torch.sigmoid(torch.var(m.permute(0, 3, 4, 1, 2), dim=[3, 4])).view(E, H, W, 1)
        offs = [d["off0"].clone(), d["off1"] * mask, zero_off, zero_off2]
        offs = [o.view(E, H, W, 2 * R + 1, 2 * R + 1, 2) for o in offs]
        outs = [ref.defCorr_index_forward(pyr[l], cl[l], offs[l], R)[0].view(E, TAPS, H, W) for l in range(LEVELS)]
        corr = torch.cat(outs, dim=1)
        gl = d["corr_grad"].view(E, LEVELS, 2 * R + 1, 2 * R + 1, H, W)
        grads = [ref.defCorr_index_backward(pyr[l], cl[l], offs[l], gl[:, l].contiguous(), R) for l in range(LEVELS)]
        gmask, = ref.corr_index_backward(pyr[1], cl[1], g_mask, 1)
        gm, gc = ref.gaussianMask_backward(d["means"], d["covs"], v_raw, g_vol, GR)
        return corr, grads, gmask, gm, gc

    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            step()
        e1.record()
        torch.cuda.synchronize()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    ms = e0.elapsed_time(e1) / iters
    return {"value": E / (ms * 1e-3), "unit": "edges/s", "ms_per_step": ms,
            "what": "reference offersample_LGS kernels recompiled unmodified for sm_100 + the reference's torch glue "
                    "(fp32 matmul, no TF32), same tensors, same GPU, 1 rank"}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_step(orc, host, E_cpu):
    """The frontend step on the CPU oracle for the first E_cpu edges."""
    import torch
    f = host["fmaps"].float()
    ii, jj = host["ii"][:E_cpu].long(), host["jj"][:E_cpu].long()
    means, covs = host["means"][:E_cpu].contiguous(), host["covs"][:E_cpu].contiguous()
    pyr = orc.build_pyramid(f[ii].contiguous(), f[jj].contiguous(), means, covs, LEVELS, GR, False)
    coords = host["coords"][:E_cpu].contiguous()
    offs = [host["off0"][:E_cpu].clone(), host["off1"][:E_cpu].clone(), torch.zeros(E_cpu, H, W, 2 * TAPS),
            torch.zeros(E_cpu, H, W, 2 * TAPS)]
    corr = orc.corr_block_lookup(pyr, coords, offs, R)
    c = coords.permute(0, 3, 1, 2).contiguous()
    gl = host["corr_grad"][:E_cpu].reshape(E_cpu, LEVELS, 2 * R + 1, 2 * R + 1, H, W)
    for l in range(LEVELS):
        orc.defCorr_index_backward(pyr[l], (c / 2 ** l).contiguous(),
                                   offs[l].view(E_cpu, H, W, 2 * R + 1, 2 * R + 1, 2).contiguous(),
                                   gl[:, l].contiguous(), R)
    m, = orc.corr_index_forward(pyr[1], (c / 2).contiguous(), 1)
    orc.corr_index_backward(pyr[1], (c / 2).contiguous(), m, 1)
    orc.gaussianMask_backward(means, covs, pyr[0], pyr[0], GR)
    return corr


def cpu_backend_step(orc, case, E_cpu):
    """The backend step (AltCorrBlock.corr_fn, corr.py:174-215: altcorr_forward r=1 on level 1 + 4 x lowMem_defSample)
    on the CPU oracle for the first E_cpu edges of the edge list (offset heads excluded: they are torch convs in both)."""
    import torch
    f = case["fmaps"].float() / 4
    pyr = [f]
    for _ in range(LEVELS - 1):
        pyr.append(torch.nn.functional.avg_pool2d(pyr[-1], 2, 2).half().float())
    ii, jj = case["ii"][:E_cpu].long(), case["jj"][:E_cpu].long()
    f1 = pyr[0][ii].permute(0, 2, 3, 1).contiguous()
    coords = case["coords"][:E_cpu]
    outs = []
    for l in range(LEVELS):
        f2 = pyr[l][jj].permute(0, 2, 3, 1).contiguous()
        c = (coords / 2 ** l).view(E_cpu, 1, H, W, 2).contiguous()
        if l == 1:
            orc.altcorr_forward(f1, f2, c, 1)
        o, = orc.lowMem_defSample(f1, f2, c, case["offsets"][l][:E_cpu].view(E_cpu, H, W, 7, 7, 2).contiguous(), R)
        outs.append(o)
    return outs


def time_cpu(workload, E_cpu, steps, warmup, seed, budget_s=150.0):
    """Median step time of the oracle port on all host threads; the number of timed steps is cut so that the whole run
    stays inside `budget_s` seconds."""
    import inputs
    from oracle import oracle as orc
    orc.build()
    orc.set_num_threads(os.cpu_count() or 1)
    if workload == "frontend":
        host = make_host_inputs(max(E_cpu, 2), 20 if E_cpu > 8 else 6, seed, pin=False)
        fn = lambda: cpu_step(orc, host, E_cpu)
    else:
        case = inputs.frontend_case(E=E_cpu, T=max(4, E_cpu // 2), seed=seed, half_fmaps=True)
        fn = lambda: cpu_backend_step(orc, case, E_cpu)
    t0 = time.perf_counter()
    fn()                                                           # first call: page-in + thread pool start
    first = time.perf_counter() - t0
    for _ in range(max(warmup - 1, 0)):
        fn()
    n = max(1, min(steps, int(budget_s / max(first, 1e-3))))
    ts = []
    for _ in range(n):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    med = statistics.median(ts)
    return E_cpu / med, med * 1e3, orc.num_threads(), n


# ------------------------------------------------------------------------------------------------ backend (N > 1)
def backend_edges(T, E, g):
    """Proximity-style edge set: every edge links a frame to a neighbour within +-8 (factor_graph.py:319-383 in spirit)."""
    import torch
    ii = torch.randint(0, T, (E,), generator=g)
    jj = (ii + torch.randint(-8, 9, (E,), generator=g)).clamp(0, T - 1)
    jj = torch.where(jj == ii, (ii + 1).clamp(max=T - 1), jj)
    jj = torch.where(jj == ii, ii - 1, jj)
    return ii, jj


class BackendWorkload:
    """BASELINE configs[3]: global-BA correlation, edge-sharded over the ranks of one box (lgu-slam_b200/sharded.py)."""

    def __init__(self, T, E, dev, rank, world):
        import torch
        import torch.nn as nn
        import inputs
        import lgu_slam_b200
        from importlib import import_module
        self.torch, self.lib = torch, lgu_slam_b200._lib
        self.corr = import_module("lgu-slam_b200.corr")
        self.sh = import_module("lgu-slam_b200.sharded")
        self.T, self.E, self.dev, self.rank, self.world = T, E, dev, rank, world
        g = inputs.gen(4242)
        self.ii, self.jj = backend_edges(T, E, g)
        self.ii_d, self.jj_d = self.ii.to(dev), self.jj.to(dev)
        torch.manual_seed(0)                                         # identical learned heads on every rank
        self.ofsMap = nn.Conv2d(256, 98, 3, padding=1).to(dev)
        self.ofs_res = nn.Conv2d(256, 98, 3, padding=1).to(dev)
        self.GA = self.corr.GaussianMask(H, W).to(dev)
        # this rank's block of keyframes (as if it had encoded them): fp16, seeded per frame
        per = (T + world - 1) // world
        lo, hi = rank * per, min(T, (rank + 1) * per)
        maps = torch.empty(hi - lo, C, H, W, dtype=torch.float16)
        for t in range(lo, hi):
            maps[t - lo] = torch.randn(C, H, W, generator=inputs.gen(7000 + t)).half()
        self.maps_host = maps.pin_memory()
        self.maps_dev = maps.to(dev)
        self.all_maps_dev = None                                     # filled by the 1-GPU arm only
        self.blk = None
        self.plans = {}

    def engine(self, single):
        key = "single" if single else "sharded"
        if key not in self.plans:
            def compute(c, i, j, out=None, out_index=None, pass_edges=None, pass_hook=None, key=None):
                return self.blk(c, i, j, out=out, out_index=out_index, pass_edges=pass_edges, pass_hook=pass_hook, key=key)
            eng = self.sh.ShardedBackendCorr(compute, single_process=single)
            plan = eng.set_edges(self.ii, self.jj, dst=None if single else 0)   # outputs go back to rank 0: it gets the lighter chunks
            mine = plan.rank_edges[eng.rank]
            import inputs
            coords = inputs.make_coords(int(mine.numel()), H, W, H, W, inputs.gen(9000 + 17 * eng.rank + (1 if single else 0)))
            coords = coords.permute(0, 2, 3, 1).contiguous().view(1, -1, H, W, 2)
            self.plans[key] = dict(eng=eng, plan=plan, coords_host=coords.pin_memory(), coords=coords.to(self.dev))
        return self.plans[key]

    def gather_maps(self, single, maps_dev):
        if single:
            if self.all_maps_dev is None:                             # the 1-GPU arm owns every keyframe
                import inputs
                torch = self.torch
                full = torch.empty(self.T, C, H, W, dtype=torch.float16)
                for t in range(self.T):
                    full[t] = torch.randn(C, H, W, generator=inputs.gen(7000 + t)).half()
                self.all_maps_dev = full.to(self.dev)
            return self.all_maps_dev
        per = (self.T + self.world - 1) // self.world                  # the block layout of __init__: known on every rank
        counts = [max(0, min(self.T, (r + 1) * per) - r * per) for r in range(self.world)]
        return self.sh.all_gather_frames(maps_dev, counts=counts)     # collective 1 (NCCL all_gather_into_tensor)

    def step(self, mode, peer=None, single=False, coords=None, maps_dev=None):
        """mode 'peer': outputs returned to rank 0 through `peer`; 'sharded': outputs stay in `peer` = a local buffer."""
        torch = self.torch
        st = self.engine(single)
        eng = st["eng"]
        with torch.no_grad():
            fmaps = self.gather_maps(single, self.maps_dev if maps_dev is None else maps_dev)
            # cold block per step: the pyramid and every per-chunk quantity are rebuilt (cache only de-duplicates the
            # offset-head work WITHIN the step: under strict_ref the sampler reads slab 0 only, quirk Q2)
            self.blk = self.corr.AltCorrBlock(self.ofsMap, self.ofs_res, self.GA, fmaps.view(1, self.T, C, H, W),
                                              strict_ref=True, materialize=True, cache=True, volume_cache_gb=0)
            c = st["coords"] if coords is None else coords
            if mode in ("peer", "peer_store"):
                return eng.lookup_into_peer(c, self.ii_d, self.jj_d, peer, coords_are_local=True,
                                            via="copy" if mode == "peer" else "store")
            # outputs left on the owning rank: same kernels, destination = a local buffer indexed by local position
            at = 0
            for ch in st["plan"].rank_chunks[eng.rank]:
                vd, _ = eng._chunk_index(ch, self.dev)
                n = vd.numel()
                idx = torch.arange(at, at + n, dtype=torch.int32, device=self.dev)
                self.blk(c[:, at:at + n], self.ii_d[vd], self.jj_d[vd], out=peer, out_index=idx, key=("chunk", ch))
                at += n
            torch.cuda.synchronize(self.dev)
            return peer


def run_backend(a, rank, world, local):
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pinned = pin_to_gpu_numa(local)
    dist.init_process_group("nccl", device_id=dev)
    T, E = a.backend_frames, a.backend_edges
    wl = BackendWorkload(T, E, dev, rank, world)
    sh = wl.sh

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, everyone=True):
        for _ in range(warmup):
            fn()
        if everyone:
            barrier()
        else:
            torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = wl.lib.LAUNCHES
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        if everyone:
            barrier()
        else:
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        launches = wl.lib.LAUNCHES - n0
        if everyone:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches

    st = wl.engine(False)
    plan = st["plan"]
    visited = plan.num_edges
    e_local = int(plan.rank_edges[rank].numel())
    # warm the NCCL communicator (connection set-up is a one-off of the process, not of a backend call)
    sh.all_gather_frames(wl.maps_dev)
    results = {}
    # (1) outputs returned to rank 0 as fp16 through NVLink peer stores -- the headline
    peer16 = sh.PeerOutput(E, (LEVELS * TAPS, H, W), torch.float16, dev, dst=0, plan=plan)
    sampler = ClockSampler(local)
    sampler.start()
    ms16, launches = timed(lambda: wl.step("peer", peer16), a.steps, a.warmup)
    sampler.stop_flag = True
    results["outputs_returned_fp16"] = {"ms_per_step": ms16, "edges_per_s": visited / ms16 * 1e3,
                                        "bytes_into_rank0": visited * LEVELS * TAPS * P * 2}
    # ---- end to end: this rank's keyframe maps and coords go H2D from pinned host memory every step; rank 0 reads a
    # per-edge checksum of the gathered result back
    maps_in = torch.empty_like(wl.maps_dev)
    coords_in = torch.empty_like(st["coords"])
    chk_host = torch.empty(E, dtype=torch.float32).pin_memory()

    def e2e_step():
        maps_in.copy_(wl.maps_host, non_blocking=True)
        coords_in.copy_(st["coords_host"], non_blocking=True)
        res = wl.step("peer", peer16, coords=coords_in, maps_dev=maps_in)
        if res is not None:
            chk_host.copy_(res[0].view(E, -1)[:, ::1009].float().mean(1), non_blocking=True)
        torch.cuda.synchronize()

    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    h2d = wl.maps_host.numel() * 2 + st["coords_host"].numel() * 4
    t = torch.tensor([float(h2d)], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    h2d_total = int(t.item())
    # (2) outputs returned as fp32
    peer32 = sh.PeerOutput(E, (LEVELS * TAPS, H, W), torch.float32, dev, dst=0, plan=plan)
    ms32, _ = timed(lambda: wl.step("peer", peer32), max(a.steps // 2, 2), 1)
    results["outputs_returned_fp32"] = {"ms_per_step": ms32, "edges_per_s": visited / ms32 * 1e3,
                                        "bytes_into_rank0": visited * LEVELS * TAPS * P * 4}
    # (2b) fp16 again, but with the lookup kernels storing straight into rank 0's memory (no staging, no copy engine)
    msd, _ = timed(lambda: wl.step("peer_store", peer16), max(a.steps // 2, 2), 1)
    results["outputs_returned_fp16_direct_stores"] = {"ms_per_step": msd, "edges_per_s": visited / msd * 1e3}
    peer32.close()
    del peer32
    # (3) outputs left sharded (fp32, the operator's own dtype)
    local_buf = torch.empty(max(e_local, 1), LEVELS * TAPS, H, W, dtype=torch.float32, device=dev)
    mss, _ = timed(lambda: wl.step("sharded", local_buf), max(a.steps // 2, 2), 1)
    results["outputs_sharded_fp32"] = {"ms_per_step": mss, "edges_per_s": visited / mss * 1e3}
    del local_buf
    torch.cuda.empty_cache()
    # (4) the same step on ONE GPU of this job (rank 0 alone, the others wait): the strong-scaling denominator
    ms1 = None
    if rank == 0:
        own = sh.PeerOutput(E, (LEVELS * TAPS, H, W), torch.float16, dev, single_process=True)
        ms1, _ = timed(lambda: wl.step("peer", own, single=True), 2, 1, everyone=False)
        own.close()
        del own
    barrier()
    # ---- roofline of the data path of one pass (128 edges), timed alone on rank 0: level 0 as compact per-pixel boxes,
    # levels 1-3 as volumes (tcgen05 builds), then the fused per-corner-gated lookup that consumes them
    roof = None
    if rank == 0:
        ops = wl.corr.ops
        planes = wl.blk._level_planes()
        n = min(128, visited)
        ii32, jj32 = wl.ii_d[:n].to(torch.int32).contiguous(), wl.jj_d[:n].to(torch.int32).contiguous()
        cpass = st["coords"][0, :n].contiguous()
        offs = [(4 * torch.tanh(torch.randn(1, H, W, 2 * TAPS, device=dev))).contiguous() for _ in range(2)]
        out_pass = torch.empty(n, LEVELS * TAPS, H, W, dtype=torch.float16, device=dev)

        def one_pass(parts):
            boxes = ops.build_boxes(planes[0][0], planes[0][0], ii32, jj32, cpass)
            vols = [None] + [ops.build_volume(planes[0][0], None, planes[l][0], None, ii32, jj32).view(n, H, W, H >> l, W >> l)
                             for l in range(1, LEVELS)]
            if parts == "all":
                ops.altcorr_lookup_fused(vols, cpass, offs[0], offs[1], R, shared_offsets=True, apply_mask=False,
                                         boxes0=boxes, out=out_pass)

        def clock(parts):
            one_pass(parts)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                one_pass(parts)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / 5

        bms_build, bms = clock("build"), clock("all")
        peak, peak_src = load_peak()
        gather = [TAPS * 16, TAPS * 16, 64 * 4, 64 * 4]
        # per edge: two map planes read, boxes + three volumes written; the lookup reads coords, its gathers (+ the 16 corners
        # of the r=1 mask lookup) and writes 196 fp16 channels (offset slab 0 is shared by the pass, quirk Q2)
        alg = (2 * P * C * 2 + P * 16 * 20 * 4 + 4 * P * sum(QS[1:])) + P * (8 + sum(gather) + 64 + 2 * LEVELS * TAPS)
        gbs = alg * n / (bms * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": "one backend pass: lgu_build_boxes (level 0) + 3 x lgu_build_volume (tcgen05) + "
                                          "lgu_altcorr_lookup_boxes_into",
                "achieved": round(gbs, 1), "peak": peak, "unit": "GB/s", "frac": round(gbs / peak, 4), "traffic": None,
                "peak_source": peak_src, "algorithmic_bytes_per_launch_group": alg * n,
                "what": f"{n} edges timed alone on rank 0 (CUDA events, 5 repeats): {bms:.3f} ms, of which the four builds "
                        f"{bms_build:.3f} ms; level 0 costs its MMAs and epilogue for the 62 % of the halves the boxes touch but "
                        f"writes 1.3 KB per pixel, so the pass is no longer bound by HBM writes alone"}
    peer16.close()
    if rank == 0:
        sp = ms1 / ms16
        limiting = ("NVLink ingress of rank 0 (peer stores of every rank's rows into one GPU)"
                    if results["outputs_sharded_fp32"]["ms_per_step"] < 0.8 * ms16 else
                    "none on the data path: per-rank compute (volume build + lookup); the fmap all-gather is < 2 ms")
        cpu = None
        if not a.no_cpu_baseline:
            try:
                v, ms, thr, n = time_cpu("backend", 8, 3, 1, 1235, budget_s=40)
                cpu = {"value": v, "unit": "edges/s", "cores": thr, "kind": "port",
                       "sample": f"8 edges per step (altcorr r=1 + 4 x lowMem_defSample, full 48x64x128 shapes), median of "
                                 f"{n} steps ({ms:.0f} ms each)"}
            except Exception as ex:
                cpu = {"value": None, "unit": "edges/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex}"}
        line = {"metric": METRIC, "value": visited / ms16 * 1e3, "unit": "edges/s", "n_gpus": world, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": ms16, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "backend_t256_e4096_sharded" if (T, E) == (256, 4096) else f"backend_t{T}_e{E}_sharded",
                           "keyframes": T, "edges": E, "edges_visited": visited, "chunks": len(plan.chunk_edges),
                           "edges_per_rank": plan.counts(), "fmap": [C, H, W], "levels": LEVELS, "radius": R,
                           "path": "forward only (the backend runs under no_grad): per chunk offset heads (torch convs) + "
                                   "4 tcgen05 volumes + fused per-corner-gated lookup; cold AltCorrBlock per step",
                           "collectives": "all_gather_into_tensor of the fp16 keyframe maps (NCCL) per step; outputs returned "
                                          "chunk by chunk into rank 0's buffer (CUDA IPC peer memory over NVLink: async "
                                          "peer-to-peer copies behind the next chunk's compute; direct kernel stores "
                                          "reported beside), one barrier per step",
                           "outputs": "fp16 [E,196,48,64] on rank 0, chunk-major rows (value); fp32 and sharded variants under 'backend'",
                           "l2_policy": "per-step working set (50 MB of volumes per edge) >> 126 MB L2; no explicit flush",
                           "parallelism": f"chunks of 8 source frames, LPT over {world} ranks", "host_pinning": pinned},
                "clocks": sampler.result(),
                "e2e": {"value": visited * a.steps / e2e_s, "unit": "edges/s", "h2d_bytes_per_step": h2d_total,
                        "d2h_bytes_per_step": E * 4,
                        "what": "per step every rank uploads its keyframe maps (fp16) and its edges' coords from pinned host "
                                "memory; rank 0 downloads a per-edge checksum of the gathered result"},
                "gpu_launches": launches, "roofline": roof, "cpu_baseline": cpu,
                "backend": dict(results, single_gpu_same_job={"ms_per_step": ms1, "edges_per_s": visited / ms1 * 1e3},
                                speedup_vs_single_gpu=sp, strong_scaling_efficiency=sp / world,
                                transport=peer16.transport, limiting=limiting)}
        print(json.dumps(line))
    dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--edges", type=int, default=48)
    ap.add_argument("--frames", type=int, default=20)
    ap.add_argument("--backend-edges", type=int, default=4096)
    ap.add_argument("--backend-frames", type=int, default=256)
    ap.add_argument("--cpu-edges", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the results of the last timed step (corr, offset / mean / cov / den "
                         "gradients) as DIR/<name>.npy; inputs are seeded, so runs with the same arguments are comparable")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    a.warmup = max(a.warmup, 3) if a.impl == "ours" else a.warmup

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if a.dump_outputs and (a.impl != "ours" or world > 1):
        ap.error("--dump-outputs is implemented for the single-GPU step of --impl ours")
    n_gpus = max(world, a.gpus)
    config = {"workload": "frontend_w20_e48" if (a.edges, a.frames) == (48, 20) else f"frontend_w{a.frames}_e{a.edges}",
              "edges_per_gpu": a.edges, "keyframes": a.frames, "fmap": [C, H, W], "levels": LEVELS, "radius": R,
              "gauss_radius": GR, "build_precision": "fp16 inputs (exact products), fp32 accumulate",
              "step": "pack + build (tcgen05) + fused lookup + fused lookup backward (dense level gradients"
                      + (" AND the Gaussian-head gradients, formed in the same launch from the shared-memory accumulators)"
                         if GAUSS_FUSED else
                         " + the Gaussian head's 9x9 window record of the merged level-0 gradient) + Gaussian-head gradients "
                         "from that record" if GAUSS_WINDOW else ") + Gaussian-head gradients from the level gradients")
                      + " (SURVEY 8d composite)",
              "gauss_backward": GAUSS_MODE,
              "l2_policy": "working set per step (2.4 GB pyramid + 2.4 GB grads at E=48) >> 126 MB L2; no explicit flush",
              "parallelism": "single GPU (the frontend window stays on one GPU)"}

    if a.impl == "reference":
        if rank != 0:
            return
        backend = n_gpus > 1
        e_cpu = a.cpu_edges or (8 if backend else a.edges)
        val, ms, thr, n = time_cpu("backend" if backend else "frontend", e_cpu, max(a.steps, 1), max(min(a.warmup, 1), 0), 1235)
        if backend:
            config = {"workload": "backend_t256_e4096_sharded", "keyframes": a.backend_frames, "edges": a.backend_edges,
                      "fmap": [C, H, W], "levels": LEVELS, "radius": R}
            sample = (f"{e_cpu} of {a.backend_edges} edges per step (altcorr r=1 + 4 x lowMem_defSample, full 48x64x128 shapes); "
                      f"median of {n} timed steps ({ms:.0f} ms each)")
        else:
            sample = (f"{e_cpu} of {a.edges} edges per step, full 48x64x128 shapes, same op sequence (build + lookup fwd/bwd + "
                      f"gaussian bwd); median of {n} timed steps ({ms:.0f} ms each)")
        line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "edges/s", "n_gpus": n_gpus,
                "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms / e_cpu * (a.backend_edges if backend else a.edges),
                "higher_is_better": True, "scaling": "strong" if backend else "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": val, "unit": "edges/s", "cores": thr, "kind": "port", "sample": sample},
                "e2e": {"value": val, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    if world > 1:
        return run_backend(a, rank, world, local)

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pinned = pin_to_gpu_numa(local)
    config["host_pinning"] = pinned
    wl = Workload(a.edges, a.frames, 1235 + rank, dev)

    # ---- device-resident timing
    for _ in range(a.warmup):
        wl.step()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    records = []
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start.record()
    for i in range(a.steps):
        rec = []
        out = wl.step(record=rec)
        records.append(rec)
        if i + 1 < a.steps:
            del out                       # only the last step's results outlive the step
    t_end.record()
    torch.cuda.synchronize()
    total_ms = t_start.elapsed_time(t_end)
    last = {k: out[k] for k in Workload.RESULT_KEYS} if a.dump_outputs else None
    del out
    # keep the GPU under the same load a little longer so that NVML has something to sample (20 steps are ~30 ms)
    t_load = time.perf_counter()
    while time.perf_counter() - t_load < 0.25:
        wl.step()
        torch.cuda.synchronize()
    sampler.stop_flag = True
    if last is not None:
        dump_outputs(a.dump_outputs, last)
        del last
    per_op = {}
    for rec in records:
        for (n0, e0), (n1, e1) in zip(rec[:-1], rec[1:]):
            per_op.setdefault(n1, []).append(e0.elapsed_time(e1))
    per_op_ms = {k: sum(v) / len(v) for k, v in per_op.items()}
    ms_per_step = total_ms / a.steps
    value = a.edges / (ms_per_step * 1e-3)

    # ---- end to end from pinned host buffers (3-stream pipeline: H2D | kernels | D2H)
    wl.e2e_setup()
    for _ in range(3):
        wl.step_e2e()
    wl.e2e_drain()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        wl.step_e2e()
    wl.e2e_drain()                        # every step's result is in pinned host memory
    e2e_s = time.perf_counter() - t0
    h2d, d2h = wl.e2e_bytes()
    e2e_val = a.edges * a.steps / e2e_s

    # ---- roofline of the dominant kernel group
    peak, peak_src = load_peak()
    alg = algorithmic_bytes_per_edge()
    table = {}
    for k, ms in per_op_ms.items():
        if k in alg and alg[k] > 0:
            gbs = alg[k] * a.edges / (ms * 1e-3) / 1e9
            table[k] = {"ms": round(ms, 4), "alg_MB_per_edge": round(alg[k] / 1e6, 3), "GBps": round(gbs, 1),
                        "frac": round(gbs / peak, 4)}
    dom = max((k for k in table if k != "pack"), key=lambda k: table[k]["ms"])
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if tr.get("edges") == a.edges:
            traffic = tr.get(dom)
    except Exception:
        pass
    comp_bytes = sum(alg[k] for k in ("build", "lookup_fwd", "lookup_bwd", "gauss_bwd"))
    roofline = {"bound": "hbm", "kernel": dom, "achieved": table[dom]["GBps"], "peak": peak, "unit": "GB/s",
                "frac": table[dom]["frac"], "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch_group": alg[dom] * a.edges, "per_op": table,
                "step_share": {k: round(v / sum(per_op_ms.values()), 3) for k, v in per_op_ms.items()},
                "composite": {"alg_MB_per_edge": round(comp_bytes / 1e6, 2),
                              "frac": round(comp_bytes * a.edges / (ms_per_step * 1e-3) / 1e9 / peak, 4)}}
    try:
        roofline["extra_ops"] = wl.extra_ops()
    except Exception as ex:
        roofline["extra_ops"] = {"failed": str(ex)}

    cpu = None
    if not a.no_cpu_baseline:
        try:
            v48, ms48, thr, n48 = time_cpu("frontend", a.edges, 3, 1, 1235, budget_s=30)
            v8, ms8, _, n8 = time_cpu("frontend", 8, 3, 1, 1235, budget_s=10)
            cpu = {"value": v48, "unit": "edges/s", "cores": thr, "kind": "port",
                   "sample": f"all {a.edges} edges per step (no extrapolation), full 48x64x128 shapes, same op sequence; median "
                             f"of {n48} steps ({ms48:.0f} ms each)",
                   "config0_e8": {"value": v8, "ms_per_step": ms8, "steps": n8,
                                  "what": "BASELINE configs[0]: the 8-edge batch in full"}}
        except Exception as ex:            # the oracle is test infrastructure; never let it break the product number
            cpu = {"value": None, "unit": "edges/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex}"}

    ref_cuda = None
    if not a.no_ref_cuda:
        try:
            ref_cuda = time_ref_cuda(wl)
        except Exception as ex:            # informational only
            ref_cuda = {"value": None, "what": f"failed: {ex}"}

    line = {"metric": METRIC, "value": value, "unit": "edges/s", "n_gpus": 1, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config, "clocks": sampler.result(),
            "e2e": {"value": e2e_val, "unit": "edges/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "what": "per step: coords + upstream gradient H2D from pinned memory, every result (corr, offset / mean / cov / "
                            "den gradients) D2H into pinned memory; feature maps, head outputs and edge lists stay resident"},
            "gpu_launches": (wl.launches_per_step or 0) * a.steps, "roofline": roofline, "cpu_baseline": cpu,
            "ref_cuda": ref_cuda}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
