"""Edge-sharded backend correlation over the GPUs of one box (torch.distributed, NCCL over NVLink 5 / NVSwitch).

The reference is single-GPU (README.md:22).  Its global-BA path (`FactorGraph.update_lowmem`,
/root/reference/droid_slam/factor_graph.py:255-302) walks the edge set in CHUNKS -- all edges whose source frame
lies in [i, i+8) (`:272-279`) -- and calls `AltCorrBlock` once per chunk.  Factor-graph edges are independent
(SURVEY.md section 8e), so the chunks are the shardable unit.  Sharding at chunk granularity -- never splitting
a chunk -- keeps every per-chunk quantity of the reference identical on N GPUs, including the reference's
offset-slab quirk Q2 (every edge of a chunk reads the offsets of the chunk's first edge).

Collectives (only these; the lookups themselves exchange nothing):
  1. once per backend call: all-gather of the keyframe feature maps (fp16, 786 KB / frame) so that every rank
     holds the whole buffer and builds its own channels-last pyramid;
  2. per BA step (optional): return of the per-edge outputs [E_local,196,H,W] -- either left sharded
     (`gather=None`; the GRU update can run data-parallel on them), gathered on one rank (`gather="dst"`)
     or on every rank (`gather="all"`).  The fast form of `gather="dst"` is `PeerOutput` + `lookup_into_peer`: the
     destination rank's output buffer is mapped into every rank (CUDA IPC over NVLink / NVSwitch peer memory) and the
     lookup kernels STORE THEIR RESULT ROWS STRAIGHT INTO IT (each edge at its original position, optionally as
     fp16 -- what the consumer, `update_op` under autocast, reads anyway: factor_graph.py:284-286); the transfer is
     the kernel's own store stream, so it overlaps the compute tile by tile and no collective carries data.

Everything here is host logic on top of `torch.distributed`; the `compute` callable is the AltCorrBlock of
lgu-slam_b200/corr.py on a GPU box and may be any function with the same signature in CPU (gloo) tests.
"""
import ctypes
from dataclasses import dataclass, field
from typing import Callable, List, Optional

import torch
import torch.distributed as dist

FRAMES_PER_CHUNK = 8          # factor_graph.py:272 (`s = 8`)


@dataclass
class EdgePlan:
    """Assignment of reference chunks to ranks.  All index tensors are int64 on the CPU."""
    world_size: int
    chunk_edges: List[torch.Tensor]                 # per chunk: positions (into the edge list) of its edges, ascending
    chunk_owner: List[int]                          # per chunk: owning rank
    rank_chunks: List[List[int]] = field(default_factory=list)      # per rank: its chunk ids, in reference order
    rank_edges: List[torch.Tensor] = field(default_factory=list)    # per rank: edge positions, chunk by chunk
    total_edges: int = 0                            # length of the edge list (>= visited edges, see reference_chunks)

    @property
    def num_edges(self):
        return int(sum(e.numel() for e in self.chunk_edges))

    def counts(self):
        return [int(e.numel()) for e in self.rank_edges]


def reference_chunks(ii: torch.Tensor, jj: torch.Tensor, frames_per_chunk: int = FRAMES_PER_CHUNK):
    """The reference's chunking rule (factor_graph.py:272-279): for i in range(0, jj.max()+1, 8):
    v = (ii >= i) & (ii < i+8).  Returns the non-empty chunks as lists of edge positions, in loop order."""
    ii = ii.detach().to("cpu", torch.int64)
    jj = jj.detach().to("cpu", torch.int64)
    if ii.numel() == 0:
        return []
    chunks = []
    for i in range(0, int(jj.max()) + 1, frames_per_chunk):
        v = torch.nonzero((ii >= i) & (ii < i + frames_per_chunk)).flatten()
        if v.numel():
            chunks.append(v)
    return chunks


# What receiving one remote edge's output rows costs the destination rank, in units of one edge of its own compute: the
# rows (1.2 MB of fp16) are written into its HBM while its own bandwidth-bound kernels run (1.2 MB / 6.5 TB/s against
# 13.4 us per edge; measured at 8 GPUs: 9.3 ms with the outputs returned against 8.4 ms with them left sharded).
DST_INGRESS_COST = 0.0138
DST_HANDICAP_FROM = 8      # ranks from which the handicap is applied (measured there: 9.33 -> 9.11 ms; chunk granularity leaves
                           # nothing to gain with fewer, larger shares)


def partition_edges(ii: torch.Tensor, jj: torch.Tensor, world_size: int,
                    frames_per_chunk: int = FRAMES_PER_CHUNK, dst: Optional[int] = None,
                    dst_ingress_cost: float = DST_INGRESS_COST) -> EdgePlan:
    """Longest-processing-time assignment of reference chunks to ranks (cost = edge count; ties by chunk order, so
    the plan is deterministic and identical on every rank without communication).
    dst (world_size >= DST_HANDICAP_FROM): the rank every output is returned to starts with a handicap -- the ingress of the other
    ranks' rows competes with its own kernels for HBM bandwidth -- so it receives the lighter chunks."""
    if world_size < 1:
        raise ValueError("world_size must be >= 1")
    chunks = reference_chunks(ii, jj, frames_per_chunk)
    owner = [0] * len(chunks)
    load = [0.0] * world_size
    if dst is not None and world_size >= DST_HANDICAP_FROM:
        total = sum(int(c.numel()) for c in chunks)
        load[dst] = dst_ingress_cost * total * (world_size - 1) / world_size
    for c in sorted(range(len(chunks)), key=lambda c: (-chunks[c].numel(), c)):
        r = min(range(world_size), key=lambda r: (load[r], r))
        owner[c] = r
        load[r] += chunks[c].numel()
    plan = EdgePlan(world_size, chunks, owner, total_edges=int(ii.numel()))
    for r in range(world_size):
        mine = [c for c in range(len(chunks)) if owner[c] == r]
        plan.rank_chunks.append(mine)
        plan.rank_edges.append(torch.cat([chunks[c] for c in mine]) if mine else torch.zeros(0, dtype=torch.int64))
    return plan


def all_gather_frames(local: torch.Tensor, group=None, counts=None) -> torch.Tensor:
    """Collective 1: every rank contributes its contiguous block of keyframe feature maps [T_r, ...] (T_r may
    differ between ranks); returns the whole buffer [sum T_r, ...] on every rank.
    counts: the per-rank T_r if the caller knows them (saves a small collective and a host synchronisation per call)."""
    world = dist.get_world_size(group)
    if world == 1:
        return local
    if counts is None:
        n = torch.tensor([local.shape[0]], device=local.device, dtype=torch.int64)
        counts = [torch.zeros_like(n) for _ in range(world)]
        dist.all_gather(counts, n, group=group)
        counts = [int(c.item()) for c in counts]
    counts = [int(c) for c in counts]
    tmax = max(counts)
    padded = local
    if local.shape[0] != tmax:
        padded = torch.zeros((tmax,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
        padded[:local.shape[0]] = local
    out = torch.empty((world * tmax,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, padded.contiguous(), group=group)
    if all(c == tmax for c in counts):
        return out
    return torch.cat([out[r * tmax:r * tmax + counts[r]] for r in range(world)], dim=0)


class PeerOutput:
    """The gathered output buffer [E, *per_edge_shape] of one backend step, resident on rank `dst` and WRITABLE FROM EVERY
    RANK: on a GPU box `dst` allocates it and the other ranks map the same memory through CUDA IPC (NVLink / NVSwitch
    peer access), so a rank's lookup kernels store their result rows straight into the destination GPU's HBM at each
    edge's original position -- "return per-edge outputs" without a collective on the data path.  On CPU (gloo tests)
    the buffer is a file under /dev/shm mapped by every rank.  `transport` names what is in use.

    Lifetime: create once (collective), reuse every step, `close()` collectively before the process group goes away."""

    def __init__(self, num_edges, per_edge_shape, dtype, device, dst=0, group=None, single_process=False, plan=None):
        """plan (an EdgePlan): rows are laid out CHUNK-MAJOR -- chunk c of the reference loop occupies the contiguous rows
        chunk_rows[c] .. chunk_rows[c] + len(chunk c), which is how the consumer walks them (factor_graph.py:272-279
        runs update_op chunk by chunk) and lets a rank ship a whole chunk with one peer-to-peer copy; `row_of_edge`
        maps an edge position to its row (-1: never visited).  Without a plan, row = edge position."""
        self.group, self.dst = group, dst
        self.chunk_rows, self.row_of_edge = None, None
        if plan is not None:
            self.chunk_rows, at = [], 0
            self.row_of_edge = torch.full((int(num_edges),), -1, dtype=torch.int64)
            for v in plan.chunk_edges:
                self.chunk_rows.append(at)
                self.row_of_edge[v] = torch.arange(at, at + v.numel())
                at += int(v.numel())
        alone = single_process or not dist.is_initialized()
        self.rank = dst if alone else dist.get_rank(group)
        self.world = 1 if alone else dist.get_world_size(group)
        self.device = torch.device(device)
        shape = (int(num_edges),) + tuple(int(x) for x in per_edge_shape)
        self._path = None
        self._own = None
        if self.device.type == "cuda":
            self.transport = "cuda-ipc peer stores (NVLink)" if self.world > 1 else "local"
            self._ptr, self._opened = None, False
            nbytes = torch.empty(0, dtype=dtype).element_size()
            for x in shape:
                nbytes *= x
            box = [None]
            with torch.cuda.device(self.device):
                if self.rank == dst:
                    self._ptr, handle = self._native_alloc(nbytes)
                    box = [handle]
                if self.world > 1:
                    dist.broadcast_object_list(box, src=dist.get_global_rank(group, dst) if group is not None else dst,
                                               group=group)
                    if self.rank != dst:
                        self._ptr = self._native_open(box[0])     # mapped with THIS rank's device current
                        self._opened = True
                self.buffer = self._wrap(self._ptr, shape, dtype)
                if self.rank == dst:
                    self.buffer.zero_()
                    torch.cuda.synchronize(self.device)
        else:
            import os
            import tempfile
            self.transport = "shared file mapping (CPU test transport)" if self.world > 1 else "local"
            box = [None]
            if self.rank == dst:
                fd, self._path = tempfile.mkstemp(prefix="lgu_peer_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
                os.close(fd)
                box = [self._path]
            if self.world > 1:
                dist.broadcast_object_list(box, src=dst, group=group)
            n = 1
            for x in shape:
                n *= x
            if self.rank == dst:
                self.buffer = torch.from_file(box[0], shared=True, size=n, dtype=dtype).view(shape)
                self.buffer.zero_()
            if self.world > 1:
                dist.barrier(group=group)
            if self.rank != dst:
                self.buffer = torch.from_file(box[0], shared=True, size=n, dtype=dtype).view(shape)
        if self.world > 1:
            dist.barrier(group=group)                       # the zero-fill on `dst` precedes every remote store

    # ---- raw device memory through the C ABI (lgu_peer_*): a plain cudaMalloc allocation + its CUDA IPC handle.  The
    # package is imported here, not at the top: the CPU tests load this module on its own.
    @staticmethod
    def _native_alloc(nbytes):
        from . import _lib
        ptr, handle = ctypes.c_void_p(0), ctypes.create_string_buffer(64)
        _lib.call("lgu_peer_alloc", nbytes, ctypes.byref(ptr), handle)
        return ptr.value, handle.raw

    @staticmethod
    def _native_open(handle):
        from . import _lib
        ptr = ctypes.c_void_p(0)
        _lib.call("lgu_peer_open", ctypes.create_string_buffer(handle, 64), ctypes.byref(ptr))
        return ptr.value

    @staticmethod
    def _wrap(ptr, shape, dtype):
        """A torch tensor aliasing raw device memory (CUDA array interface, zero copy)."""
        typestr = {torch.float32: "<f4", torch.float16: "<f2"}[dtype]

        class _Mem:
            __cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2}
        return torch.as_tensor(_Mem(), device="cuda")

    def result(self):
        """[1, E, ...] on `dst` (call after `ShardedBackendCorr.lookup_into_peer` returned), None elsewhere."""
        return self.buffer[None] if self.rank == self.dst else None

    def close(self):
        """Collective.  A failed unmap or free raises LguError; a failed unmap raises only after the barrier that orders
        the unmaps before the free, so no other rank is left waiting in it."""
        if self.world > 1:
            dist.barrier(group=self.group)
        ptr = getattr(self, "_ptr", None)
        native = self.device.type == "cuda" and ptr is not None
        if native:
            from . import _lib
        self.buffer, self._ptr = None, None
        try:
            if native:
                with torch.cuda.device(self.device):
                    torch.cuda.synchronize(self.device)
                    if self._opened:
                        _lib.call("lgu_peer_close", ptr)   # drop the mapping before the owner frees the memory
        finally:
            if self.world > 1:
                dist.barrier(group=self.group)
        if native and not self._opened:
            with torch.cuda.device(self.device):
                _lib.call("lgu_peer_free", ptr)
        self._own = None
        if self._path is not None:
            import os
            try:
                os.unlink(self._path)
            except OSError:
                pass


class ShardedBackendCorr:
    """Runs `compute(coords[:, v], ii[v], jj[v])` (AltCorrBlock.__call__, corr.py:238-249) for the chunks this
    rank owns and returns the per-edge outputs sharded or gathered.

    compute: callable(coords [1,e,H,W,2], ii [e], jj [e]) -> [1,e,CH,H,W] on `coords.device`."""

    def __init__(self, compute: Callable, group=None, single_process=False):
        """single_process=True: behave as a one-rank job even inside an initialised process group (every chunk is
        local, no collective is ever called) -- the 1-GPU arm of a strong-scaling measurement."""
        self.compute = compute
        self.group = group
        alone = single_process or not dist.is_initialized()
        self.rank = 0 if alone else dist.get_rank(group)
        self.world = 1 if alone else dist.get_world_size(group)
        self.plan: Optional[EdgePlan] = None
        self._idx = {}
        try:
            import inspect
            params = inspect.signature(compute).parameters
            self._writes_in_place = "out" in params and "out_index" in params
            self._has_pass_hook = "pass_hook" in params and "pass_edges" in params
            self._takes_key = "key" in params
        except (TypeError, ValueError):
            self._writes_in_place = self._has_pass_hook = self._takes_key = False

    def set_edges(self, ii, jj, frames_per_chunk=FRAMES_PER_CHUNK, dst=None):
        """dst: the rank the outputs will be returned to (lookup_into_peer / gather="dst"), if any -- see partition_edges."""
        self.plan = partition_edges(ii, jj, self.world, frames_per_chunk, dst=dst)
        self._idx = {}
        return self.plan

    def _chunk_index(self, c, dev):
        """Edge positions of chunk c on `dev` (int64 for indexing, int32 for the kernels), uploaded once per plan."""
        key = (c, str(dev))
        if key not in self._idx:
            vd = self.plan.chunk_edges[c].to(dev)
            self._idx[key] = (vd, vd.to(torch.int32))
        return self._idx[key]

    def local_lookup(self, coords, ii, jj):
        """This rank's share: outputs [1,E_local,CH,H,W] in the order of plan.rank_edges[rank] (None if it owns none)."""
        assert self.plan is not None, "call set_edges(ii, jj) first"
        outs = []
        for c in self.plan.rank_chunks[self.rank]:
            v = self.plan.chunk_edges[c].to(coords.device)
            outs.append(self.compute(coords[:, v], ii[v], jj[v]))
        return torch.cat(outs, dim=1) if outs else None

    def lookup_streamed_to(self, coords, ii, jj, dst=0):
        """gather="dst" with the transfer hidden behind the compute: every chunk's outputs leave for rank `dst` as
        soon as the chunk is done (point-to-point isend over NVLink / NVSwitch, asynchronous to the next chunk's
        kernels); `dst` posts all receives up front, computes its own chunks into place and scatters the received
        chunks into the original edge order.  Returns [1,E,CH,H,W] on `dst` (E = full edge count; never-visited edges
        are zero), None elsewhere."""
        assert self.plan is not None, "call set_edges(ii, jj) first"
        plan, dev = self.plan, coords.device
        mine = plan.rank_chunks[self.rank]
        outs = {}
        first = None
        if mine:                                                   # the first chunk also tells the output shape
            v = plan.chunk_edges[mine[0]].to(dev)
            first = self.compute(coords[:, v], ii[v], jj[v])
            outs[mine[0]] = first
        shape = self._out_shape(first, coords)
        if self.rank != dst:
            reqs = []
            for k, c in enumerate(mine):
                if k > 0:
                    v = plan.chunk_edges[c].to(dev)
                    outs[c] = self.compute(coords[:, v], ii[v], jj[v])
                outs[c] = outs[c][0].contiguous()
                reqs.append(dist.isend(outs[c], dst=dst, group=self.group))
            for r in reqs:
                r.wait()
            return None
        full = torch.zeros((1, plan.total_edges) + shape, dtype=torch.float32, device=dev)
        recv = []
        for r in range(self.world):
            if r == dst:
                continue
            for c in plan.rank_chunks[r]:                          # same order as the sender's isend sequence
                buf = torch.empty((plan.chunk_edges[c].numel(),) + shape, dtype=torch.float32, device=dev)
                recv.append((c, buf, dist.irecv(buf, src=r, group=self.group)))
        for k, c in enumerate(mine):
            v = plan.chunk_edges[c]
            if k > 0:
                vd = v.to(dev)
                outs[c] = self.compute(coords[:, vd], ii[vd], jj[vd])
            full[:, v.to(dev)] = outs[c]
        for c, buf, req in recv:
            req.wait()
            full[:, plan.chunk_edges[c].to(dev)] = buf[None]
        return full

    # via="copy": whole chunks are shipped behind the NEXT chunk's compute; the rank's LAST chunk has nothing to hide behind,
    # so it runs in passes of SHIP_EDGES edges and only its last pass's rows are exposed (37 edges x 24 row tiles = 6 full
    # waves of the 148-CTA volume build)
    SHIP_EDGES = 37
    SHIP_TAIL = (18, 12, 6)            # 3 / 2 / 1 waves: the last, exposed shipment is 6 edges (7 MB of fp16 rows)
    SHIP_ALL_CHUNKS_FROM = 8           # from this many ranks on, EVERY chunk runs in passes (the destination's NVLink ingress is
                                       # then the scarce resource and must never idle: 9.33 -> 9.08 ms at 8 GPUs); with fewer
                                       # ranks only the last chunk does -- the extra passes cost more than they hide
                                       # (2 GPUs: 28.7 -> 30.8 ms, 4 GPUs: 15.4 -> 16.4 ms with all chunks in passes)

    @classmethod
    def _ship_schedule(cls, n, last=True):
        """Pass sizes of a chunk of n edges: passes of SHIP_EDGES; a rank's LAST chunk ends in the tapering tail.  The
        destination's NVLink ingress is the scarce resource of the step (4.3 GB into rank 0 at 8 GPUs in ~9 ms): measured,
        [104, 18, 6] for the last chunk is slower than [18, 37, 37, 18, 12, 6] (9.37 against 9.11 ms)."""
        tail = list(cls.SHIP_TAIL) if last else []
        if n <= sum(tail) or n <= cls.SHIP_EDGES:
            return [cls.SHIP_EDGES]                                # small chunk: plain passes
        body = n - sum(tail)
        k, r = divmod(body, cls.SHIP_EDGES)
        if 0 < r < 12:                                            # no tiny leading pass: fold it into its neighbour
            if k:
                return [cls.SHIP_EDGES + r] + [cls.SHIP_EDGES] * (k - 1) + tail
            if tail:
                tail[0] += r
                return tail
            return [r]
        return ([r] if r else []) + [cls.SHIP_EDGES] * k + tail

    def lookup_into_peer(self, coords, ii, jj, peer: PeerOutput, sync=True, coords_are_local=False, via="store"):
        """gather="dst" with NO collective on the data path.  via="store": every rank runs its chunks with the destination
        buffer as the kernels' output tensor (`compute(..., out=peer.buffer, out_index=rows)` -- AltCorrBlock's fused
        lookup stores its 196-channel rows through NVLink peer memory).  via="copy": the chunk is computed into a local
        staging buffer and shipped by an asynchronous peer-to-peer copy on a side stream (the copy engines move it while
        the SMs build the next chunk's volumes; measured at 8 GPUs the direct stores of all ranks' lookups collide on the
        destination's NVLink ingress, see profiles/r02_backend_scaling.md); with a chunk-major PeerOutput that is one
        copy per chunk.  A compute callable without out= support is served by copies of its result.  One barrier at the end
        publishes the step (`sync=False` leaves it to the caller).  Returns peer.result().
        coords_are_local: `coords` holds only this rank's edges, [1,E_local,...] in the order of plan.rank_edges[rank]
        (a rank then uploads 1/N of the coordinates per step)."""
        assert self.plan is not None, "call set_edges(ii, jj) first"
        plan, dev = self.plan, coords.device
        staged = via == "copy" and dev.type == "cuda" and self._writes_in_place and self.rank != peer.dst
        if staged:
            self._ensure_staging(peer, dev)
            cur = torch.cuda.current_stream(dev)
        at = 0
        for k, c in enumerate(plan.rank_chunks[self.rank]):
            v = plan.chunk_edges[c]
            nv = int(v.numel())
            vd, vd32 = self._chunk_index(c, dev)
            cc = coords[:, at:at + nv] if coords_are_local else coords[:, vd]
            at += nv
            if peer.chunk_rows is not None:                        # chunk-major destination: contiguous rows
                r0 = peer.chunk_rows[c]
                rows = None
            else:
                r0, rows = None, vd32
            if staged:
                b = k & 1
                cur.wait_event(self._stage_free[b])                # the previous shipment of this staging buffer has left
                stage = self._stage[b]

                def ship(first, last, b=b, stage=stage, r0=r0, v=v):
                    done = torch.cuda.Event()
                    done.record(cur)
                    with torch.cuda.stream(self._copy_stream):
                        self._copy_stream.wait_event(done)
                        if r0 is not None:
                            peer.buffer[r0 + first:r0 + last].copy_(stage[first:last], non_blocking=True)
                        else:
                            for a, n_run, src in self._runs(v[first:last]):
                                peer.buffer[a:a + n_run].copy_(stage[first + src:first + src + n_run], non_blocking=True)

                kw = {"key": ("chunk", c)} if self._takes_key else {}
                nck = len(plan.rank_chunks[self.rank])
                if self._has_pass_hook and (self.world >= self.SHIP_ALL_CHUNKS_FROM or k == nck - 1):      # ship pass by pass
                    self.compute(cc, ii[vd], jj[vd], out=stage, out_index=None,
                                 pass_edges=self._ship_schedule(nv, last=k == nck - 1), pass_hook=ship, **kw)
                else:
                    self.compute(cc, ii[vd], jj[vd], out=stage, out_index=None, **kw)
                    ship(0, nv)
                with torch.cuda.stream(self._copy_stream):
                    self._stage_free[b].record(self._copy_stream)
            elif self._writes_in_place:
                if rows is None:
                    rows = torch.arange(r0, r0 + nv, dtype=torch.int32, device=dev)
                self.compute(cc, ii[vd], jj[vd], out=peer.buffer, out_index=rows,
                             **({"key": ("chunk", c)} if self._takes_key else {}))
            else:                                                  # plain callable: copy its result over
                res = self.compute(cc, ii[vd], jj[vd])[0].to(peer.buffer.dtype)
                if r0 is not None:
                    peer.buffer[r0:r0 + nv].copy_(res)
                else:
                    for a, n_run, src in self._runs(v):
                        peer.buffer[a:a + n_run].copy_(res[src:src + n_run])
        if staged:
            self._copy_stream.synchronize()
        if sync:
            if dev.type == "cuda":
                torch.cuda.synchronize(dev)                        # this rank's peer stores have landed
            if self.world > 1:
                dist.barrier(group=self.group)
        return peer.result()

    @staticmethod
    def _runs(v):
        """Runs of consecutive edge positions: (first position, length, offset in the chunk)."""
        pos = v.tolist()
        k = 0
        while k < len(pos):
            e = k + 1
            while e < len(pos) and pos[e] == pos[e - 1] + 1:
                e += 1
            yield pos[k], e - k, k
            k = e

    def _ensure_staging(self, peer, dev):
        need = max((int(self.plan.chunk_edges[c].numel()) for c in self.plan.rank_chunks[self.rank]), default=0)
        shape = (max(need, 1),) + tuple(peer.buffer.shape[1:])
        st = getattr(self, "_stage", None)
        if st is None or st[0].shape != shape or st[0].dtype != peer.buffer.dtype or st[0].device != dev:
            self._stage = [torch.empty(shape, dtype=peer.buffer.dtype, device=dev) for _ in range(2)]
            self._copy_stream = torch.cuda.Stream(dev)
            self._stage_free = [torch.cuda.Event() for _ in range(2)]
            for e in self._stage_free:
                e.record(torch.cuda.current_stream(dev))

    def __call__(self, coords, ii, jj, gather="all", dst=0):
        """gather=None: (local outputs, their edge positions).  gather="all": full [1,E,CH,H,W] in the original edge
        order on every rank.  gather="dst": the same on rank `dst`, None elsewhere (see also lookup_streamed_to)."""
        local = self.local_lookup(coords, ii, jj)
        mine = self.plan.rank_edges[self.rank]
        if gather is None:
            return local, mine
        if self.world == 1:
            return self._reorder([local], coords.device)
        counts = self.plan.counts()
        emax = max(counts)
        shape = self._out_shape(local, coords)
        pad = torch.zeros((emax,) + shape, dtype=torch.float32, device=coords.device)
        if local is not None:
            pad[:local.shape[1]] = local[0]
        if gather == "all":
            buf = torch.empty((self.world * emax,) + shape, dtype=torch.float32, device=coords.device)
            dist.all_gather_into_tensor(buf, pad, group=self.group)
            parts = [buf[r * emax:r * emax + counts[r]][None] for r in range(self.world)]
            return self._reorder(parts, coords.device)
        if gather == "dst":
            bufs = [torch.empty_like(pad) for _ in range(self.world)] if self.rank == dst else None
            dist.gather(pad, bufs, dst=dst, group=self.group)
            if self.rank != dst:
                return None
            return self._reorder([bufs[r][:counts[r]][None] for r in range(self.world)], coords.device)
        raise ValueError("gather must be None, 'all' or 'dst'")

    def _out_shape(self, local, coords):
        # every rank must agree on the per-edge output shape even if it owns no edge: probe it collectively
        shp = torch.tensor(list(local.shape[2:]) if local is not None else [0, 0, 0], device=coords.device)
        if self.world > 1:
            dist.all_reduce(shp, op=dist.ReduceOp.MAX, group=self.group)
        return tuple(int(x) for x in shp.tolist())

    def _reorder(self, parts, device):
        """Per-rank outputs -> [1, E, ...] in the ORIGINAL edge order, E = the full edge count.  Edges the reference's
        chunk loop never visits (source frame beyond the last loop start, factor_graph.py:272-279) stay zero."""
        order = torch.cat(self.plan.rank_edges).to(device)
        parts = [p for p in parts if p is not None and p.shape[1] > 0]
        if not parts:
            return None
        full = torch.cat(parts, dim=1)
        out = torch.zeros((1, self.plan.total_edges) + tuple(full.shape[2:]), dtype=full.dtype, device=device)
        out[:, order] = full
        return out
