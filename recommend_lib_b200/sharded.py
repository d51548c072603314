"""Row-sharded BPR-MF for catalogues larger than one GPU (BASELINE.json configs[4]; SURVEY.md section 8e).

No counterpart in the reference (single process, single device, SURVEY 2b).  One process per GPU; tables are
block-sharded by row: rank r owns users [r*u_per, (r+1)*u_per) and items [r*i_per, (r+1)*i_per).  Triples are routed
to the owner of their user (the sampler draws each rank's users from its own block), so the user gather / update is
local and only item rows travel.  One step:

    plan      unique item ids of the batch (sorted => already grouped by owner), remap triples to cache indices
    exchange  ids -> owners                                   (all-to-all, int32)
    serve     owners gather the requested rows                (local gather)
    exchange  rows -> requesters  = the batch's row cache     (all-to-all, 4*D B per row)
    compute   daisy_bpr_shard_step: fused step on (P_local, cache); users updated in place, one descent sum per
              cache row written out
    exchange  descent sums -> owners                          (all-to-all, 4*D B per row)
    apply     daisy_owner_apply: per row, contributions summed in sender-rank order, Q_local updated once

Every accumulation order is fixed (stable sorts, rank order), so the sharded step is deterministic and equals the
single-GPU step up to fp32 summation order.  The collectives are NCCL all-to-all(v) over NVLink; on the gloo backend
(CPU tests of the routing logic) the same exchanges run as batched isend/irecv.
"""
from __future__ import annotations

import ctypes
import math
import os
import time

import numpy as np
import torch
import torch.distributed as dist


class ShardLayout:
    """Block sharding of both tables over `world` ranks."""

    def __init__(self, user_num, item_num, world):
        self.user_num, self.item_num, self.world = int(user_num), int(item_num), int(world)
        self.u_per = math.ceil(self.user_num / self.world)
        self.i_per = math.ceil(self.item_num / self.world)

    def user_range(self, rank):
        return min(rank * self.u_per, self.user_num), min((rank + 1) * self.u_per, self.user_num)

    def item_range(self, rank):
        return min(rank * self.i_per, self.item_num), min((rank + 1) * self.i_per, self.item_num)

    def item_bounds(self, device):
        b = [min(r * self.i_per, self.item_num) for r in range(self.world + 1)]
        return torch.tensor(b, dtype=torch.int64, device=device)


class DistComm:
    """Variable-size all-to-all over torch.distributed (NCCL: all_to_all_single; gloo: batched P2P)."""

    def __init__(self, group=None):
        self.group = group
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        self.nccl = dist.get_backend(group) == "nccl"

    def counts(self, send_counts, device):
        """send_counts[r] = how many rows this rank sends to r  ->  recv_counts[r] = how many it receives from r."""
        t = torch.tensor(send_counts, dtype=torch.int64, device=device)
        if self.nccl:
            out = torch.empty_like(t)
            dist.all_to_all_single(out, t, group=self.group)
            return out.tolist()
        allc = [torch.empty_like(t) for _ in range(self.world)]
        dist.all_gather(allc, t, group=self.group)
        return [int(allc[r][self.rank]) for r in range(self.world)]

    def exchange(self, x, send_counts, recv_counts):
        """x: rows grouped by destination rank (send_counts each); returns rows grouped by source rank."""
        out = x.new_empty((int(sum(recv_counts)),) + tuple(x.shape[1:]))
        if self.nccl:
            dist.all_to_all_single(out, x.contiguous(), list(recv_counts), list(send_counts), group=self.group)
            return out
        ops, so, ro = [], 0, 0
        keep = []
        for r in range(self.world):
            s, c = send_counts[r], recv_counts[r]
            if r == self.rank:
                out[ro:ro + c] = x[so:so + s]
            else:
                if s:
                    chunk = x[so:so + s].contiguous()
                    keep.append(chunk)
                    ops.append(dist.P2POp(dist.isend, chunk, r, group=self.group))
                if c:
                    ops.append(dist.P2POp(dist.irecv, out[ro:ro + c], r, group=self.group))
            so += s
            ro += c
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()
        return out


class CudaBackend:
    """The product backend: libdaisy_b200 kernels on this rank's GPU.  No CPU fallback."""

    def __init__(self, layout, rank, dim, max_batch, device):
        from . import _lib
        _lib.require_cuda()
        self._lib = _lib
        self.device = torch.device(device)
        u0, u1 = layout.user_range(rank)
        i0, i1 = layout.item_range(rank)
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.h = _lib.Handle(idx, max(u1 - u0, 1), max(i1 - i0, 1), dim, max_batch)
        self.dim = dim
        self.loss = torch.zeros(1, dtype=torch.float64, device=self.device)

    def _s(self):
        return self._lib.stream_ptr(torch, self.device)

    def gather_rows(self, Q_local, rows_local):
        return Q_local.index_select(0, rows_local.long())

    def shard_step(self, P_local, cache, tri_local, lr, wd):
        vp = self._lib.c_vp
        grads = torch.empty_like(cache)
        self._lib.check(self.h.L.daisy_bpr_shard_step(self.h.ptr, vp(P_local.data_ptr()), vp(cache.data_ptr()),
                                                      cache.shape[0], vp(tri_local.data_ptr()), tri_local.shape[0],
                                                      lr, wd, vp(grads.data_ptr()), vp(self.loss.data_ptr()), self._s()))
        return grads

    def owner_apply(self, Q_local, rows_local, grads, lr, wd):
        vp = self._lib.c_vp
        self._lib.check(self.h.L.daisy_owner_apply(self.h.ptr, vp(Q_local.data_ptr()), vp(rows_local.data_ptr()),
                                                   vp(grads.data_ptr()), rows_local.shape[0], lr, wd, self._s()))

    def materialize(self, P_local, Q_local):
        vp = self._lib.c_vp
        self._lib.check(self.h.L.daisy_materialize(self.h.ptr, vp(P_local.data_ptr()), vp(Q_local.data_ptr()), self._s()))

    def check(self):
        self._lib.check(self.h.L.daisy_check(self.h.ptr, self._s()))

    def loss_sum(self, reset=True):
        v = float(self.loss.item())
        if reset:
            self.loss.zero_()
        return v


class ShardedBPR:
    """One rank's share of a row-sharded BPR-MF model.

    ``step(triples)``: ``triples`` int32 [B, 3] on this rank's device with columns (LOCAL user index, GLOBAL positive
    item, GLOBAL negative item).  ``P_full`` / ``Q_full`` (optional, host tensors) initialise the shards from given
    tables (parity tests); otherwise shards are drawn N(0, 0.01^2) from a (seed, rank) generator
    (BPRMFRecommender.py:39-40).
    """

    def __init__(self, user_num, item_num, factor_num, lr=0.01, wd=0.001, max_batch=4096, rank=None, world=None,
                 device=None, comm=None, backend=None, P_full=None, Q_full=None, seed=2019):
        self.rank = dist.get_rank() if rank is None else rank
        self.world = dist.get_world_size() if world is None else world
        self.layout = ShardLayout(user_num, item_num, self.world)
        self.dim, self.lr, self.wd = int(factor_num), float(lr), float(wd)
        self.device = torch.device(device if device is not None else "cpu")
        u0, u1 = self.layout.user_range(self.rank)
        i0, i1 = self.layout.item_range(self.rank)
        self.u0, self.i0 = u0, i0
        if P_full is not None:
            self.P = torch.as_tensor(P_full)[u0:u1].to(self.device, torch.float32).contiguous()
            self.Q = torch.as_tensor(Q_full)[i0:i1].to(self.device, torch.float32).contiguous()
        else:
            g = torch.Generator(device=self.device).manual_seed(seed * 1000 + self.rank)
            self.P = torch.empty((u1 - u0, self.dim), device=self.device).normal_(0, 0.01, generator=g)
            self.Q = torch.empty((i1 - i0, self.dim), device=self.device).normal_(0, 0.01, generator=g)
        self.comm = comm
        self.backend = backend if backend is not None else CudaBackend(self.layout, self.rank, self.dim, max_batch,
                                                                       self.device)
        self._bounds = self.layout.item_bounds(self.device)
        self.profile = None
        self.wire_rows = 0         # rows received + sent over the interconnect (both exchanges), for reporting

    # ---- phases (also driven one by one by the in-process multi-rank emulation in the tests) --------------------
    def plan(self, triples):
        B = triples.shape[0]
        items = triples[:, 1:].t().reshape(-1)                       # [i_0..i_B-1, j_0..j_B-1]
        uniq, inv = torch.unique(items, sorted=True, return_inverse=True)
        pos = torch.searchsorted(uniq.long(), self._bounds)          # sorted ids are already grouped by owner block
        send_counts = (pos[1:] - pos[:-1]).tolist()                  # host sync: split sizes of the exchanges
        tri_local = torch.stack([triples[:, 0], inv[:B].to(torch.int32), inv[B:].to(torch.int32)], dim=1).contiguous()
        return uniq.to(torch.int32), send_counts, tri_local

    def serve(self, recv_ids):
        return self.backend.gather_rows(self.Q, recv_ids - self.i0)

    def compute(self, tri_local, cache):
        return self.backend.shard_step(self.P, cache, tri_local, self.lr, self.wd)

    def apply(self, recv_ids, grads_in):
        self.backend.owner_apply(self.Q, (recv_ids - self.i0).to(torch.int32).contiguous(), grads_in, self.lr, self.wd)

    # ---- one full step over torch.distributed -----------------------------------------------------------------------
    PHASES = ("plan", "counts", "ids", "serve", "rows", "compute", "grads", "apply")

    def _mark(self, name):
        if self.profile is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            self.profile.append((name, e, time.perf_counter()))

    def step(self, triples):
        c = self.comm
        self._mark("start")
        ids, send_counts, tri_local = self.plan(triples)
        self._mark("plan")
        recv_counts = c.counts(send_counts, self.device)
        self._mark("counts")
        recv_ids = c.exchange(ids, send_counts, recv_counts)
        self._mark("ids")
        rows = self.serve(recv_ids)
        self._mark("serve")
        cache = c.exchange(rows, recv_counts, send_counts)
        self._mark("rows")
        grads = self.compute(tri_local, cache)
        self._mark("compute")
        grads_in = c.exchange(grads, send_counts, recv_counts)
        self._mark("grads")
        self.apply(recv_ids, grads_in)
        self._mark("apply")
        remote = sum(send_counts) - send_counts[self.rank]
        self.wire_rows += 2 * remote

    def profile_summary(self):
        """Mean device ms and host ms per phase over the profiled steps (enable with ``self.profile = []``)."""
        torch.cuda.synchronize(self.device)
        dev, host, n = {}, {}, 0
        prev = None
        for name, ev, t in self.profile:
            if name == "start":
                n += 1
            else:
                dev[name] = dev.get(name, 0.0) + prev[1].elapsed_time(ev)
                host[name] = host.get(name, 0.0) + (t - prev[2]) * 1e3
            prev = (name, ev, t)
        return {k: (round(dev[k] / n, 3), round(host[k] / n, 3)) for k in dev}

    def materialize(self):
        self.backend.materialize(self.P, self.Q)

    def full_tables(self):
        """All-gather the (materialised) shards: (P [U, D], Q [I, D]) on every rank.  Test / small-model helper."""
        self.materialize()
        out = []
        for t in (self.P, self.Q):
            n = torch.tensor([t.shape[0]], device=self.device)
            ns = [torch.zeros_like(n) for _ in range(self.world)]
            dist.all_gather(ns, n)
            mx = int(max(int(x) for x in ns))
            pad = torch.zeros((mx, self.dim), device=self.device)
            pad[:t.shape[0]] = t
            parts = [torch.empty_like(pad) for _ in range(self.world)]
            dist.all_gather(parts, pad)
            out.append(torch.cat([p[:int(k)] for p, k in zip(parts, ns)]))
        return out[0], out[1]


class _DeviceView:
    """A [rows, dim] fp32 window on device memory owned by the library (the item shard inside the rank's arena),
    exposed to torch through __cuda_array_interface__."""

    def __init__(self, ptr, rows, dim):
        self.__cuda_array_interface__ = {"shape": (int(rows), int(dim)), "typestr": "<f4", "data": (int(ptr), False),
                                         "version": 3, "strides": None}


def exchange_ipc_handles(blob, group=None, device=None):
    """All-gather one 64-byte CUDA IPC handle per rank over torch.distributed (any backend) -> list of bytes."""
    world = dist.get_world_size(group)
    dev = device if (device is not None and dist.get_backend(group) == "nccl") else torch.device("cpu")
    mine = torch.tensor(list(blob), dtype=torch.uint8, device=dev)
    parts = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(parts, mine, group=group)
    return [bytes(p.cpu().tolist()) for p in parts]


class PeerShardedBPR:
    """One rank's share of a row-sharded BPR-MF model whose exchange runs over PEER MEMORY (NVLink) inside the step
    kernels -- the product path of BASELINE.json configs[4] (include/daisy_b200.h, daisy_shard_*).  No CPU fallback.

    ``P`` [local users, D] is an ordinary CUDA tensor; ``Q`` [local items, D] is a view of the item shard inside the
    rank's arena, which the peer GPUs map.  ``mapping``:
      "symm"  (default for world > 1) the arena is a torch symmetric-memory buffer (cuMem VMM, rendezvous over the
              process group) -- peer reads of random rows run at NVLink speed through this mapping;
      "ipc"   the library cudaMallocs the arena and the ranks exchange legacy CUDA IPC handles (measured 2x slower
              for random row reads; kept for platforms without symmetric memory);
      "local" all ranks live in this process on one device (tests): wire with ``connect_in_process``.
    ``step(triples)``: int32 [B, 3] with columns (LOCAL user index, GLOBAL positive item, GLOBAL negative item), on the
    device or in pinned host memory.  Every rank must call ``step`` the same number of times.
    """

    def __init__(self, user_num, item_num, factor_num, lr=0.01, wd=0.001, max_batch=4096, rank=None, world=None,
                 device=None, P_full=None, Q_full=None, seed=2019, mapping=None, group=None):
        from . import _lib
        _lib.require_cuda()
        self._lib = _lib
        self.rank = dist.get_rank() if rank is None else rank
        self.world = dist.get_world_size() if world is None else world
        self.group = group
        self.mapping = mapping or ("symm" if self.world > 1 else "local")
        assert self.mapping in ("symm", "ipc", "local")
        self.layout = ShardLayout(user_num, item_num, self.world)
        self.dim, self.lr, self.wd = int(factor_num), float(lr), float(wd)
        self.device = torch.device(device if device is not None else "cuda")
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", idx)
        u0, u1 = self.layout.user_range(self.rank)
        i0, i1 = self.layout.item_range(self.rank)
        self.u0, self.i0 = u0, i0
        self.h = _lib.Handle(idx, max(u1 - u0, 1), max(i1 - i0, 1), self.dim, max_batch)
        L, vp = self.h.L, _lib.c_vp
        self._symm_buf = self._symm_hdl = None
        arena_arg = None
        if self.mapping == "symm":
            import torch.distributed._symmetric_memory as symm
            need = _lib.c_i64()
            _lib.check(L.daisy_shard_arena_size(self.dim, int(max_batch), self.world, int(item_num), ctypes.byref(need)))
            with torch.cuda.device(self.device):
                self._symm_buf = symm.empty((need.value + 3) // 4, dtype=torch.float32, device=self.device)
            arena_arg = vp(self._symm_buf.data_ptr())
        _lib.check(L.daisy_shard_init(self.h.ptr, self.rank, self.world, int(item_num), arena_arg))
        arena, q, nbytes = vp(), vp(), _lib.c_i64()
        _lib.check(L.daisy_shard_arena(self.h.ptr, ctypes.byref(arena), ctypes.byref(q), ctypes.byref(nbytes)))
        self.arena_ptr, self.arena_bytes = arena.value, nbytes.value
        with torch.cuda.device(self.device):
            self.Q = torch.as_tensor(_DeviceView(q.value, max(i1 - i0, 1), self.dim), device=self.device)[:i1 - i0]
            if P_full is not None:
                self.P = torch.as_tensor(P_full)[u0:u1].to(self.device, torch.float32).contiguous()
                self.Q.copy_(torch.as_tensor(Q_full)[i0:i1].to(self.device, torch.float32))
            else:
                g = torch.Generator(device=self.device).manual_seed(seed * 1000 + self.rank)
                self.P = torch.empty((u1 - u0, self.dim), device=self.device).normal_(0, 0.01, generator=g)
                self.Q.normal_(0, 0.01, generator=g)
            self.loss = torch.zeros(1, dtype=torch.float64, device=self.device)
            self._P_keep = self.P if self.P.shape[0] else torch.zeros((1, self.dim), device=self.device)
        self._P_ptr = self._P_keep.data_ptr()
        self.attached = self.world == 1
        torch.cuda.synchronize(self.device)

    # ---- wiring ---------------------------------------------------------------------------------------------------
    def ipc_handle(self):
        buf = (ctypes.c_ubyte * 64)()
        self._lib.check(self.h.L.daisy_shard_ipc_handle(self.h.ptr, ctypes.cast(buf, ctypes.c_void_p)))
        return bytes(buf)

    def connect(self):
        """Map the peers' arenas (one process per GPU): symmetric-memory rendezvous, or legacy IPC handle exchange."""
        if self.world > 1:
            L = self.h.L
            if self.mapping == "symm":
                import torch.distributed._symmetric_memory as symm
                self._symm_hdl = symm.rendezvous(self._symm_buf, self.group if self.group is not None else dist.group.WORLD)
                ptrs = [int(p) for p in self._symm_hdl.buffer_ptrs]
                assert ptrs[self.rank] == self.arena_ptr, "symmetric-memory rendezvous returned a different local address"
                arr = (ctypes.c_void_p * self.world)(*ptrs)
                self._lib.check(L.daisy_shard_attach(self.h.ptr, None, arr, 0))
            elif self.mapping == "ipc":
                blobs = exchange_ipc_handles(self.ipc_handle(), self.group, self.device)
                raw = b"".join(blobs)
                buf = (ctypes.c_ubyte * len(raw)).from_buffer_copy(raw)
                self._lib.check(L.daisy_shard_attach(self.h.ptr, ctypes.cast(buf, ctypes.c_void_p), None, 0))
            else:
                raise ValueError('mapping "local" is wired with PeerShardedBPR.connect_in_process(shards)')
            self.attached = True
            torch.cuda.synchronize(self.device)
            dist.barrier(self.group)
        return self

    @staticmethod
    def connect_in_process(shards):
        """All ranks live in this process on one device (tests): hand every rank the others' arena pointers."""
        G = len(shards)
        arr = (ctypes.c_void_p * G)(*[s.arena_ptr for s in shards])
        for s in shards:
            if G > 1:
                s._lib.check(s.h.L.daisy_shard_attach(s.h.ptr, None, arr, 1))
            s.attached = True

    def _s(self):
        return self._lib.stream_ptr(torch, self.device)

    # ---- the step ---------------------------------------------------------------------------------------------------
    def step(self, triples):
        vp = self._lib.c_vp
        B = int(triples.shape[0])
        fn = self.h.L.daisy_shard_step if triples.is_cuda else self.h.L.daisy_shard_step_host
        self._lib.check(fn(self.h.ptr, vp(self._P_ptr), vp(triples.data_ptr() if B else 0), B, self.lr, self.wd,
                           vp(self.loss.data_ptr()), self._s()))

    def compute(self, triples):
        vp = self._lib.c_vp
        B = int(triples.shape[0])
        self._lib.check(self.h.L.daisy_shard_compute(self.h.ptr, vp(self._P_ptr), vp(triples.data_ptr() if B else 0), B,
                                                     self.lr, self.wd, vp(self.loss.data_ptr()), self._s()))

    def prepare(self, triples):
        """Lockstep protocol with the exclusive-row bypass: prepare (all ranks) -> classify (all) -> compute (all, the
        same triples) -> apply (all)."""
        vp = self._lib.c_vp
        B = int(triples.shape[0])
        self._lib.check(self.h.L.daisy_shard_prepare(self.h.ptr, vp(self._P_ptr), vp(triples.data_ptr() if B else 0), B,
                                                     self._s()))

    def classify(self):
        self._lib.check(self.h.L.daisy_shard_classify(self.h.ptr, self._s()))

    def apply(self):
        self._lib.check(self.h.L.daisy_shard_apply(self.h.ptr, self.lr, self.wd, self._s()))

    def materialize(self):
        self._lib.check(self.h.L.daisy_shard_materialize(self.h.ptr, self._lib.c_vp(self._P_ptr), self._s()))

    def check(self):
        self._lib.check(self.h.L.daisy_check(self.h.ptr, self._s()))

    def last_counts(self):
        """Distinct item rows the most recent step exchanged with every owner (list of `world` ints).  Synchronises."""
        buf = (ctypes.c_uint32 * (self.world + 1))()
        self._lib.check(self.h.L.daisy_shard_last_counts(self.h.ptr, ctypes.cast(buf, ctypes.c_void_p), self._s()))
        return [int(buf[o + 1]) - int(buf[o]) for o in range(self.world)]

    SHARD_PHASES = ("bookkeeping", "fetch", "compute_push", "barrier1", "apply", "barrier2")

    def phase_ms(self):
        arr = (ctypes.c_double * 6)()
        n = ctypes.c_int64()
        self._lib.check(self.h.L.daisy_shard_phase_ms(self.h.ptr, arr, ctypes.byref(n)))
        return dict(zip(self.SHARD_PHASES, [round(x, 4) for x in arr])), n.value

    def loss_sum(self, reset=True, group=None, reduce=False):
        t = self.loss.clone()
        if reduce and self.world > 1:
            dist.all_reduce(t, group=group)
        if reset:
            self.loss.zero_()
        return float(t.item())

    def full_tables(self):
        """All-gather the (materialised) shards: (P [U, D], Q [I, D]) on every rank.  Test / small-model helper."""
        self.materialize()
        out = []
        for t, per in ((self.P, self.layout.u_per), (self.Q, self.layout.i_per)):
            pad = torch.zeros((per, self.dim), device=self.device)
            pad[:t.shape[0]] = t
            parts = [torch.empty_like(pad) for _ in range(self.world)]
            dist.all_gather(parts, pad)
            out.append(torch.cat(parts))
        return out[0][:self.layout.user_num], out[1][:self.layout.item_num]

    # ---- owner routing ----------------------------------------------------------------------------------------------
    def route(self, triples, batch):
        """The rank's share of a GLOBAL epoch (``daisy_route_triples``): ``triples`` int32 [n, 3] on the device with global
        ids, identical on every rank and already shuffled.  Returns (local triples [m, 3] with the user column made local,
        offsets: a list of ceil(n / batch) + 1 ints) -- step k of this rank runs on ``local[off[k]:off[k + 1]]``, its part
        of global batch k, so the sharded step equals the single-device step on that batch."""
        vp = self._lib.c_vp
        t = triples
        if not (t.is_cuda and t.dtype == torch.int32 and t.dim() == 2 and t.shape[1] == 3 and t.is_contiguous()):
            raise ValueError("triples must be a contiguous int32 [n, 3] device tensor")
        n, batch = int(t.shape[0]), int(batch)
        nb = (n + batch - 1) // batch
        out = torch.empty((max(n, 1), 3), dtype=torch.int32, device=self.device)
        off = torch.zeros(nb + 1, dtype=torch.int64, device=self.device)
        u0, u1 = self.layout.user_range(self.rank)
        self._lib.check(self.h.L.daisy_route_triples(self.h.ptr, vp(t.data_ptr()), n, batch, u0, u1, vp(out.data_ptr()),
                                                     vp(off.data_ptr()), self._s()))
        off = off.cpu().tolist()                          # synchronises: the step loop slices on the host
        return out[:off[-1]], off

    # ---- evaluation over the sharded item table (users partitioned: every rank ranks its own users, no merge across
    #      ranks; SURVEY.md section 8e) --------------------------------------------------------------------------------
    def _peer_q(self, owner):
        """The item shard of ``owner`` as mapped into this process: a [rows, D] tensor view on peer memory."""
        q = self._lib.c_vp()
        self._lib.check(self.h.L.daisy_shard_peer_q(self.h.ptr, int(owner), ctypes.byref(q)))
        i0, i1 = self.layout.item_range(owner)
        with torch.cuda.device(self.device):
            return torch.as_tensor(_DeviceView(q.value, max(i1 - i0, 1), self.dim), device=self.device)[:i1 - i0], q.value

    def _eval_handle(self, rows):
        """A light handle (no step workspace) over (local users x `rows` item rows) for the evaluation kernels."""
        key = int(rows)
        hs = self.__dict__.setdefault("_eval_handles", {})
        if key not in hs:
            hs[key] = self._lib.Handle(self.device.index, max(self.P.shape[0], 1), max(key, 1), self.dim, 0)
        return hs[key]

    def gather_item_rows(self, items_global):
        """Rows of the GLOBAL item table for sorted, duplicate-free ids (int64 / int32 device tensor): every owner's part
        is read straight from that owner's memory (``daisy_gather_rows`` on the peer mapping).  Call after
        ``materialize()`` (true weights; the call ends with the barrier that makes the peers' shards final)."""
        vp = self._lib.c_vp
        ids = items_global.to(device=self.device, dtype=torch.int64)
        out = torch.empty((ids.shape[0], self.dim), dtype=torch.float32, device=self.device)
        bounds = torch.searchsorted(ids, self.layout.item_bounds(self.device)).tolist()
        for o in range(self.world):
            a, b = bounds[o], bounds[o + 1]
            if b > a:
                _, qptr = self._peer_q(o)
                idx = (ids[a:b] - self.layout.item_range(o)[0]).to(torch.int32).contiguous()
                self._lib.check(self.h.L.daisy_gather_rows(self.h.ptr, vp(qptr), vp(idx.data_ptr()), b - a,
                                                           vp(out[a:b].data_ptr()), self._s()))
        return out

    def topk_candidates(self, users_local, cands_global, top_k):
        """``metric_eval`` semantics (util/metrics.py:46-66) for THIS rank's users: users_local [N] (local indices),
        cands_global [N, C] (global item ids, ground truth first) -> candidate positions [N, K] in rank order.  The
        candidates' rows are fetched once from their owners; scores and the (score desc, position asc) order are those of
        ``daisy_topk_candidates`` on the unsharded tables."""
        users = torch.as_tensor(np.asarray(users_local)).to(self.device, torch.int32).contiguous()
        cands = torch.as_tensor(np.asarray(cands_global)).to(self.device, torch.int64)
        N, C = cands.shape
        if N == 0:
            return torch.empty((N, top_k), dtype=torch.int32, device=self.device)
        uniq, inv = torch.unique(cands.reshape(-1), return_inverse=True)
        cache = self.gather_item_rows(uniq)
        cidx = inv.reshape(N, C).to(torch.int32).contiguous()
        h = self._eval_handle(uniq.shape[0])
        pos, _, _ = self._lib.call_topk_candidates(h, self._P_ptr, cache.data_ptr(), users, cidx, top_k, self._s())
        self._lib.check(h.L.daisy_check(h.ptr, self._s()))
        return pos

    def metric_eval(self, eval_users, eval_cands, top_k, group=None):
        """(HR@K, NDCG@K) over ALL evaluated users (global ids; every rank passes the same arrays): each rank ranks the
        users it owns, the per-user hits / gains are summed over the ranks."""
        eu = np.asarray(eval_users).reshape(-1)
        u0, u1 = self.layout.user_range(self.rank)
        mine = np.nonzero((eu >= u0) & (eu < u1))[0]
        self.materialize()
        pos = self.topk_candidates(eu[mine] - u0, np.asarray(eval_cands)[mine], top_k).cpu().numpy()
        hit = pos == 0
        hr = hit.any(axis=1)
        ndcg = np.where(hr, 1.0 / np.log2(hit.argmax(axis=1) + 2.0), 0.0)
        t = torch.tensor([hr.sum(), ndcg.sum(), float(len(mine))], dtype=torch.float64, device=self.device)
        if self.world > 1 and self.mapping != "local":
            dist.all_reduce(t, group=group if group is not None else self.group)
        t = t.cpu().numpy()
        return float(t[0] / max(t[2], 1.0)), float(t[1] / max(t[2], 1.0))

    def topk_full(self, users_local, k, exclude=None):
        """Full-catalogue top-k for THIS rank's users over the sharded item table: the shards are streamed one owner at a
        time into a local buffer (one NVLink copy per shard), ``daisy_topk_full`` ranks the users against each, and the
        per-shard winners are merged -- scores are the exact fp32 scores and the order is (score desc, global item asc),
        so the result equals ``daisy_topk_full`` on the unsharded table.  Returns (items [N, k] int64 global ids,
        scores [N, k])."""
        users = torch.as_tensor(np.asarray(users_local)).to(self.device, torch.int32).contiguous()
        N = users.shape[0]
        self.materialize()
        all_items, all_scores = [], []
        buf = None
        for o in range(self.world):
            i0, i1 = self.layout.item_range(o)
            rows = i1 - i0
            if rows <= 0:
                continue
            kk = min(int(k), rows)
            view, qptr = self._peer_q(o)
            if o == self.rank:
                q_local_ptr = qptr
            else:
                if buf is None:
                    buf = torch.empty((self.layout.i_per, self.dim), dtype=torch.float32, device=self.device)
                buf[:rows].copy_(view)                     # the shard crosses NVLink once
                q_local_ptr = buf.data_ptr()
            h = self._eval_handle(rows)
            excl = self._lib.exclusion_csr(exclude, N, self.device, (i0, i1))
            items, scores = self._lib.call_topk_full(h, self._P_ptr, q_local_ptr, users, kk, excl, self._s())
            self._lib.check(h.L.daisy_check(h.ptr, self._s()))
            all_items.append(items.to(torch.int64) + i0)
            all_scores.append(scores)
        items, scores = torch.cat(all_items, 1), torch.cat(all_scores, 1)
        # (score desc, item asc): stable sort by item, then stable sort by score
        o1 = torch.argsort(items, dim=1, stable=True)
        items, scores = items.gather(1, o1), scores.gather(1, o1)
        o2 = torch.argsort(scores, dim=1, descending=True, stable=True)
        kk = min(int(k), items.shape[1])
        if self.world > 1 and self.mapping != "local":
            dist.barrier(self.group)                      # nobody steps (and rewrites its shard) while a peer still reads it
        return items.gather(1, o2)[:, :kk], scores.gather(1, o2)[:, :kk]

    # ---- the training loop --------------------------------------------------------------------------------------------
    def fit(self, train_pairs, epochs, batch_size, num_ng=4, seed=2019, eval_users=None, eval_cands=None, topk=10,
            verbose=False):
        """The epoch loop of BPRMFRecommender.py:157-181 over the row-sharded model: every rank draws the SAME epoch from
        the deterministic host sampler (``sampler.TripleSampler``: global ids, global shuffle), keeps the triples of the
        users it owns (``route``), and step k of every rank is its part of global batch k -- so losses and metrics are
        those of the single-device ``BPRMFRecommender.fit`` on the same triples, up to the fp32 summation order of row
        sums that arrive from several ranks.  ``batch_size`` is the GLOBAL batch; the handle must have been created
        with ``max_batch`` >= the largest local share (``max_batch=batch_size`` is always enough).
        Returns ``history`` = [{epoch, loss, hr, ndcg}]."""
        from .sampler import TripleSampler
        sampler = TripleSampler(train_pairs, self.layout.item_num, num_ng=num_ng, seed=seed)
        n = len(sampler)
        pinned = torch.empty((n, 3), dtype=torch.int32).pin_memory()
        history = []
        for ep in range(int(epochs)):
            pinned.numpy()[:] = sampler.sample_epoch(ep)
            local, off = self.route(pinned.to(self.device, non_blocking=True), batch_size)
            for k in range(len(off) - 1):
                self.step(local[off[k]:off[k + 1]])
            self.materialize()
            rec = dict(epoch=ep + 1, loss=self.loss_sum(reduce=True))
            self.check()
            if eval_users is not None:
                rec["hr"], rec["ndcg"] = self.metric_eval(eval_users, eval_cands, topk)
            history.append(rec)
            if verbose and self.rank == 0:
                print(rec, flush=True)
        return history

    def close(self):
        torch.cuda.synchronize(self.device)
        self.Q = None
        for h in self.__dict__.get("_eval_handles", {}).values():
            h.close()
        self.h.close()
        self._symm_hdl = self._symm_buf = None
