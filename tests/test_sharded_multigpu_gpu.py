"""The sharded backend on several GPUs of one box against the same lookup in ONE process on one GPU: every rank runs its
chunks of AltCorrBlock (196-channel rows) or AltCorrBlock.lookup_encoded (128-channel encoder rows) and returns them to
rank 0 through a chunk-major sharded.PeerOutput, by peer-to-peer copies of staged chunks (via="copy") or by the lookup
kernels' own stores into rank 0's memory (via="store").  Rank 0's buffer must equal the single-process result bit for
bit.  Uses 2 ranks, or every visible GPU when there are more; skipped with fewer than 2."""
import datetime
import os
import socket
import sys
import traceback

import pytest
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

pytestmark = pytest.mark.gpu

H, W, T, E = 48, 64, 24, 40
JOIN_S = 600


def _problem(dev):
    """Identical on every rank: heads, keyframe maps, edges, coords (seeded)."""
    from importlib import import_module
    import inputs
    import lgu_slam_b200  # noqa: F401
    corr = import_module("lgu-slam_b200.corr")
    torch.manual_seed(0)
    heads = [torch.nn.Conv2d(256, 98, 3, padding=1).to(dev), torch.nn.Conv2d(256, 98, 3, padding=1).to(dev),
             corr.GaussianMask(H, W).to(dev)]
    enc = torch.nn.Sequential(torch.nn.Conv2d(196, 128, 1), torch.nn.ReLU(inplace=True)).to(dev)
    g = inputs.gen(606)
    fmaps = torch.randn(1, T, 128, H, W, generator=g).half().to(dev)
    ii = torch.randint(0, T, (E,), generator=g)
    jj = (ii + torch.randint(1, 4, (E,), generator=g)).clamp(max=T - 1)
    jj = torch.where(jj == ii, (ii - 1).clamp(min=0), jj)
    coords = inputs.make_coords(E, H, W, H, W, g).permute(0, 2, 3, 1).contiguous().view(1, E, H, W, 2)
    return corr, heads, enc, fmaps, ii, jj, coords.to(dev)


def _compute(corr, heads, enc, fmaps, channels):
    blk = corr.AltCorrBlock(*heads, fmaps, strict_ref=False, materialize=True)

    def compute(c, i, j, out=None, out_index=None, pass_edges=None, pass_hook=None, key=None):
        kw = dict(out=out, out_index=out_index, pass_edges=pass_edges, pass_hook=pass_hook, key=key)
        return blk.lookup_encoded(c, i, j, enc, **kw) if channels == 128 else blk(c, i, j, **kw)
    return compute


def _run(rank, world, port, channels, via, path):
    import torch.distributed as dist
    try:
        dev = torch.device("cuda", rank)
        torch.cuda.set_device(dev)
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev,
                                timeout=datetime.timedelta(seconds=300))
        from importlib import import_module
        sharded = import_module("lgu-slam_b200.sharded")
        corr, heads, enc, fmaps, ii, jj, coords = _problem(dev)
        eng = sharded.ShardedBackendCorr(_compute(corr, heads, enc, fmaps, channels))
        plan = eng.set_edges(ii, jj, dst=0)
        peer = sharded.PeerOutput(E, (channels, H, W), torch.float16, dev, dst=0, plan=plan)
        try:
            with torch.no_grad():
                res = eng.lookup_into_peer(coords, ii.to(dev), jj.to(dev), peer, via=via)
                if rank == 0:
                    torch.save({"rows": res[0].cpu(), "row_of_edge": peer.row_of_edge}, path)
        finally:
            peer.close()
            dist.destroy_process_group()
    except BaseException:
        traceback.print_exc()
        raise


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("via", ["copy", "store"])
@pytest.mark.parametrize("channels", [128, 196])
def test_sharded_rows_equal_the_single_gpu_rows(channels, via, tmp_path):
    world = torch.cuda.device_count()
    if world < 2:
        pytest.skip("needs at least 2 GPUs")
    path = str(tmp_path / "rank0.pt")
    ctx = mp.get_context("spawn")
    port = _free_port()
    procs = [ctx.Process(target=_run, args=(r, world, port, channels, via, path)) for r in range(world)]
    try:
        for p in procs:
            p.start()
        for p in procs:
            p.join(JOIN_S)
        assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join(30)
            if p.is_alive():
                p.kill()
                p.join()
    got = torch.load(path)
    # the same chunks, computed in this process on one GPU
    from importlib import import_module
    sharded = import_module("lgu-slam_b200.sharded")
    dev = torch.device("cuda", 0)
    corr, heads, enc, fmaps, ii, jj, coords = _problem(dev)
    compute = _compute(corr, heads, enc, fmaps, channels)
    rows = got["row_of_edge"]
    want = torch.zeros(E, channels, H, W, dtype=torch.float16)
    with torch.no_grad():
        for v in sharded.reference_chunks(ii, jj):
            out = compute(coords[:, v.to(dev)], ii[v].to(dev), jj[v].to(dev))[0]
            want[rows[v]] = out.half().cpu()
    assert (rows >= 0).any()
    assert torch.equal(got["rows"].view(torch.int16), want.view(torch.int16))
