#!/usr/bin/env python
"""Backend step with the consumer's first layer folded into the lookup (AltCorrBlock.lookup_encoded), against the step that
returns 196-channel rows.  One job, three arms, alternated and repeated (bench.py's backend workload: T = 256 keyframes,
4096 edges, chunks of 8 source frames partitioned over the ranks, rows returned to rank 0 through sharded.PeerOutput with
via="copy"):

  (a) rows196     today's step: 196-channel fp16 rows returned to rank 0;
  (b) rows196+enc (a) plus rank 0 running update_op's relu(conv1x1) under fp16 autocast on all returned rows -- the work
                  (c) moves to the ranks, so (b) is the fair baseline;
  (c) enc128      relu(conv1x1(corr)) computed by every rank inside its lookup kernel, 128-channel fp16 rows returned.

  torchrun --nproc-per-node N tools/bench_backend_enc.py [--steps 3 --warmup 1 --repeats 3]

Times are CUDA events over `steps` steps, max over ranks; printed as one JSON line (rank 0).  With --kernels (one
process) it instead times the single-GPU backend lookup kernel at 48 and 512 edges: no epilogue, the fp16 encoder
epilogue, and the frontend's TF32 encoder epilogue on the same volumes for scale."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
sys.dont_write_bytecode = True

import torch  # noqa: E402
import torch.nn as nn  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import bench  # noqa: E402
import inputs  # noqa: E402

H, W, C, P = bench.H, bench.W, bench.C, bench.H * bench.W


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def encoder(dev):
    torch.manual_seed(1)
    net = nn.Sequential(nn.Conv2d(196, 128, 1), nn.ReLU(inplace=True)).to(dev)     # UpdateModule.corr_encoder[0:2]
    return net


class EncWorkload(bench.BackendWorkload):
    """bench.BackendWorkload whose chunk compute calls lookup_encoded while `encoder` is set."""
    encoder = None

    def engine(self, single):
        st = super().engine(single)

        def compute(c, i, j, out=None, out_index=None, pass_edges=None, pass_hook=None, key=None):
            kw = dict(out=out, out_index=out_index, pass_edges=pass_edges, pass_hook=pass_hook, key=key)
            if self.encoder is None:
                return self.blk(c, i, j, **kw)
            return self.blk.lookup_encoded(c, i, j, self.encoder, **kw)
        st["eng"].compute = compute
        return st


def run_scaling(a):
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    wl = EncWorkload(a.frames, a.edges, dev, rank, world)
    sh = wl.sh
    net = encoder(dev)
    plan = wl.engine(False)["plan"]
    visited = plan.num_edges
    remote = sum(int(plan.rank_edges[r].numel()) for r in range(world) if r != 0)
    sh.all_gather_frames(wl.maps_dev)                              # NCCL connection set-up outside the timed steps
    peer196 = sh.PeerOutput(a.edges, (196, H, W), torch.float16, dev, dst=0, plan=plan)
    peer128 = sh.PeerOutput(a.edges, (128, H, W), torch.float16, dev, dst=0, plan=plan)

    def arm_a():
        wl.encoder = None
        wl.step("peer", peer196)

    def arm_b():
        wl.encoder = None
        res = wl.step("peer", peer196)
        if rank == 0:
            with torch.no_grad(), torch.autocast("cuda", torch.float16):
                torch.relu(F.conv2d(res[0], net[0].weight, net[0].bias))

    def arm_c():
        wl.encoder = net
        wl.step("peer", peer128)

    arms = {"rows196": (arm_a, 196), "rows196+enc": (arm_b, 196), "enc128": (arm_c, 128)}

    def timed(fn):
        for _ in range(a.warmup):
            fn()
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.steps):
            fn()
        e1.record()
        dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / a.steps], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    times = {k: [] for k in arms}
    for _ in range(a.repeats):
        for name, (fn, _) in arms.items():
            times[name].append(timed(fn))
    # what the arms return: (c) against (b)'s conv of (a)'s rows on rank 0, as a sanity line (same bar as the tests)
    check = None
    if rank == 0:
        with torch.no_grad(), torch.autocast("cuda", torch.float16):
            want = torch.relu(F.conv2d(peer196.buffer[:64], net[0].weight, net[0].bias))
        got = peer128.buffer[:64]
        d = (got.float() - want.float()).abs()
        check = {"rows_compared": 64, "max_abs_diff": float(torch.nan_to_num(d).max()),
                 "nan_patterns_equal": bool(torch.equal(torch.isnan(got), torch.isnan(want)))}
    peer196.close()
    peer128.close()
    if rank == 0:
        out = {"workload": "backend_enc", "n_gpus": world, "frames": a.frames, "edges": a.edges, "edges_visited": visited,
               "steps": a.steps, "repeats": a.repeats, "card": card(), "check": check, "arms": {}}
        for name, (_, ch) in arms.items():
            ms = statistics.median(times[name])
            out["arms"][name] = {"ms_per_step": ms, "ms_all": times[name], "spread_ms": max(times[name]) - min(times[name]),
                                 "edges_per_s": visited / ms * 1e3, "bytes_into_rank0": remote * ch * P * 2}
        print(json.dumps(out), flush=True)
    dist.destroy_process_group()


def run_kernels(a):
    from lgu_slam_b200 import ops
    dev = torch.device("cuda", 0)
    net = encoder(dev)
    packed = ops.pack_conv1x1_f16(net[0].weight.float(), net[0].bias.float())
    wfrag = ops.pack_conv1x1(net[0].weight.float())
    bias = net[0].bias.detach().float().contiguous()
    res = {"workload": "backend_lookup_kernels", "card": card(), "iters": a.iters, "cases": {}}
    for E in (48, 512):
        g = inputs.gen(300 + E)
        T = 64
        fm = (torch.randn(T, C, H, W, generator=g) / 4).half().to(dev)
        planes, cur = [], fm.float()
        for l in range(4):
            planes.append(cur.permute(0, 2, 3, 1).reshape(T, -1, C).half().contiguous())
            cur = F.avg_pool2d(cur, 2, stride=2)
        ii = torch.randint(0, T, (E,), generator=g).to(torch.int32).to(dev)
        jj = ((ii.cpu() + 1) % T).to(torch.int32).to(dev)
        coords = inputs.make_coords(E, H, W, H, W, g).permute(0, 2, 3, 1).contiguous().to(dev)
        vols = [ops.build_volume(planes[0], None, planes[l], None, ii, jj).view(E, H, W, H >> l, W >> l) for l in range(4)]
        off0 = (4.0 * torch.tanh(torch.randn(E, H, W, 98, generator=g))).to(dev).contiguous()
        off1 = (4.0 * torch.tanh(torch.randn(E, H, W, 98, generator=g))).to(dev).contiguous()
        cum = torch.ones(E, H, W, device=dev)
        out196 = torch.empty(E, 196, H, W, dtype=torch.float16, device=dev)
        out128 = torch.empty(E, 128, H, W, dtype=torch.float16, device=dev)
        kw = dict(shared_offsets=False, apply_mask=False)
        fns = {
            "backend_no_epilogue": lambda: ops.altcorr_lookup_fused(vols, coords, off0, off1, 3, out=out196, **kw),
            "backend_fp16_epilogue": lambda: ops.altcorr_lookup_encoded(vols, coords, off0, off1, 3, out=out128,
                                                                        packed=packed, **kw),
            "frontend_tf32_epilogue": lambda: ops.corr_lookup_fused_enc(vols, coords, off0, off1, cum, wfrag, bias,
                                                                        enc_half=True),
        }
        times = {k: [] for k in fns}
        for fn in fns.values():
            fn()
        torch.cuda.synchronize()
        for _ in range(a.repeats):
            for name, fn in fns.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.iters):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                times[name].append(e0.elapsed_time(e1) / a.iters * 1e3)
        res["cases"][E] = {k: {"us": statistics.median(v), "us_all": v} for k, v in times.items()}
        del vols
        torch.cuda.empty_cache()
    print(json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--edges", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--kernels", action="store_true", help="single-GPU lookup kernel timings at 48 and 512 edges")
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    if a.kernels:
        run_kernels(a)
    else:
        run_scaling(a)


if __name__ == "__main__":
    main()
