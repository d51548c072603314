"""bench.py --gpus N (N > 1): the row-sharded BPR-MF step of BASELINE.json configs[4] on N GPUs of one node, one rank per
GPU under torchrun.  Measurement code only -- the product is recommend_lib_b200.sharded.PeerShardedBPR."""
import json
import os

import numpy as np
import torch
import torch.distributed as dist

from recommend_lib_b200.sharded import DistComm, PeerShardedBPR, ShardedBPR


def sharded_parity_selfcheck(rank, world, dev, mapping):
    """Cross-GPU correctness inside the run that is timed: three steps of a scaled-down replica (same kernels, same
    peer mapping, barriers and owner merge; 40 000 x 30 001 x 128, 30 000 triples per global batch with hot rows) on all
    ranks, all-gathered and compared on rank 0 with (a) the float64 closed form of the reference step (oracle, the
    checker) and (b) the unsharded CUDA step.  Returns the dict that goes into config.parity_selfcheck; raises on a
    mismatch beyond the north star's 1e-5."""
    U, I, D, B, steps, lr, wd = 40_000, 30_001, 128, 30_000, 3, 0.05, 0.01
    rng = np.random.default_rng(5)
    P0 = (rng.standard_normal((U, D)) * 0.3).astype(np.float32)
    Q0 = (rng.standard_normal((I, D)) * 0.3).astype(np.float32)
    batches = []
    for _ in range(steps):
        b = np.stack([rng.integers(0, U, B), rng.integers(0, I, B), rng.integers(0, I, B)], 1).astype(np.int32)
        b[: B // 4, 1] = 3
        b[-B // 8:, 2] = 3
        batches.append(b)
    m = PeerShardedBPR(U, I, D, lr=lr, wd=wd, max_batch=B, rank=rank, world=world, device=dev, P_full=P0, Q_full=Q0,
                       mapping=mapping).connect()
    u0, u1 = m.layout.user_range(rank)
    for b in batches:
        t = b[(b[:, 0] >= u0) & (b[:, 0] < u1)].copy()
        t[:, 0] -= u0
        m.step(torch.from_numpy(t).to(dev))
    m.check()
    P, Q = m.full_tables()
    loss = m.loss_sum(reduce=True)
    out = None
    if rank == 0:
        from oracle import bpr_oracle                 # the checker, not the thing measured
        from recommend_lib_b200.bpr import BPR, BPRSGD
        Pr, Qr, losses = bpr_oracle.bpr_run_closed_form(P0, Q0, batches, lr, wd, np.float64)
        rel = lambda a, b: float(np.abs(a - b).max() / np.abs(b).max())
        one = BPR(U, I, D, max_batch=B)
        with torch.no_grad():
            one.embed_user.weight.copy_(torch.from_numpy(P0))
            one.embed_item.weight.copy_(torch.from_numpy(Q0))
        one = one.to(dev)
        opt = BPRSGD(one, lr=lr, weight_decay=wd)
        for b in batches:
            opt.step(torch.from_numpy(b).to(dev))
        one.materialize()
        P1, Q1 = (t.detach().cpu().numpy() for t in one._tables())
        Pg, Qg = P.cpu().numpy(), Q.cpu().numpy()
        out = {"ranks": world, "steps": steps, "vs_oracle_P": rel(Pg, Pr), "vs_oracle_Q": rel(Qg, Qr),
               "vs_oracle_loss": abs(loss - sum(losses)) / sum(losses), "vs_single_gpu_P": rel(Pg, P1),
               "vs_single_gpu_Q": rel(Qg, Q1), "tolerance": 1e-5}
        bad = [k for k, v in out.items() if k.startswith("vs_") and not v <= 1e-5]
        assert not bad, f"sharded parity self-check failed: {out}"
        del one
    dist.barrier()
    m.close()
    del m
    torch.cuda.empty_cache()
    return out


def bench_sharded(args, cfg, metric, unit):
    from recommend_lib_b200.sampler import _rng, zipf_items
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    U, I, D, B = cfg["user_num"], cfg["item_num"], cfg["dim"], cfg["batch"]
    if args.scale != 1.0:
        U, I = int(U * args.scale), int(I * args.scale)
    if args.batch:
        B = args.batch
    K, W = args.steps, max(args.warmup, 3)
    peer = args.exchange == "peer"
    parity = sharded_parity_selfcheck(rank, world, dev, args.mapping) if peer else None
    if peer:
        model = PeerShardedBPR(U, I, D, lr=cfg["lr"], wd=cfg["wd"], max_batch=B, rank=rank, world=world, device=dev,
                               seed=2019, mapping=args.mapping).connect()
        handle, loss_dev, check = model.h, model.loss, model.check
    else:
        model = ShardedBPR(U, I, D, lr=cfg["lr"], wd=cfg["wd"], max_batch=B, rank=rank, world=world, device=dev,
                           comm=DistComm(), seed=2019)
        handle, loss_dev, check = model.backend.h, model.backend.loss, model.backend.check
    u0, u1 = model.layout.user_range(rank)
    nb = K + W
    g = _rng(2019, 40, rank)
    host = np.empty((nb * B, 3), dtype=np.int32)
    host[:, 0] = g.integers(0, u1 - u0, size=nb * B)                       # local user index: routed by owner
    host[:, 1] = zipf_items(g, nb * B, I, cfg["zipf"], perm_seed=2019)     # global ids, Zipf over a permuted catalogue
    host[:, 2] = g.integers(0, I, size=nb * B)
    host = torch.from_numpy(host.reshape(nb, B, 3)).pin_memory()
    devtri = host.to(dev)
    if peer:
        handle.set_inputs_ready(True)      # device triples are uploaded and synchronised before they are used

    def run(first, count, src):
        for s in range(first, first + count):
            if peer:
                model.step(src[s])
            else:
                model.step(src[s] if src is devtri else src[s].to(dev, non_blocking=True))

    run(0, W, devtri)
    model.materialize()                             # warm the lazy-decay pass too (first launch loads its code)
    check()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if not peer:
        model.wire_rows = 0
    launches0 = handle.launches
    clocks = None
    try:                                            # every rank samples its own GPU (rank 0's goes into `clocks`)
        import bench as _bench
        clocks = _bench.ClockSampler(local)         # NVML initialisation takes tens of ms: before the barrier
    except Exception:
        clocks = None
    torch.cuda.synchronize()
    dist.barrier()                                  # all ranks enter the timed region together
    if clocks is not None:
        clocks.start()
    if os.environ.get("DAISY_TRACE_TIMED") and peer:
        handle.trace_start()
    ev0.record()
    run(W, K, devtri)
    ev1.record()                                    # (the lazy decay stays lazy: the library folds it in by itself when
    torch.cuda.synchronize()                        #  c < 1e-4, evaluation honours c^2, an epoch end materialises once)
    model.materialize()
    if clocks is not None:
        clocks.stop()
    if os.environ.get("DAISY_TRACE_TIMED") and peer:
        rows = [[round(x, 2) for x in row] for row in handle.trace_dump()]
        print(f"rank {rank} timed-region trace:", rows, flush=True)
    dist.barrier()
    ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    launches = handle.launches - launches0
    if peer:
        cnt = model.last_counts()
        remote = sum(cnt) - cnt[rank]
        wire_rows = 2 * remote * K         # fetched rows in + pushed sums out, per rank (last step's count, every step alike)
    else:
        wire_rows = model.wire_rows
    # e2e: the product's data path (PeerShardedBPR.fit): triples arrive in pinned HOST memory with GLOBAL ids, are copied
    # to the device and ROUTED there (daisy_route_triples: ownership test, local user index, compaction, per-step
    # offsets) in chunks of 10 steps on a side stream -- chunk c + 1 is copied and routed while the device runs the
    # steps of chunk c -- then stepped; every step's loss is read back.  All of it inside the timed region.
    loss_host = torch.zeros(nb, dtype=torch.float64).pin_memory()
    host_g = host.clone()
    host_g[:, :, 0] += u0                                # global user ids, as a host sampler produces them
    host_g = host_g.pin_memory()
    side = torch.cuda.Stream(device=dev)
    CH = 10

    def route_chunk(first, last):
        with torch.cuda.stream(side):
            d = host_g[first:last].reshape(-1, 3).to(dev, non_blocking=True)
            local, off = model.route(d, B)               # synchronises the SIDE stream only (offsets read on the host)
        return local, off

    def run_routed(first, last):
        nxt = route_chunk(first, min(first + CH, last))
        for c0 in range(first, last, CH):
            c1 = min(c0 + CH, last)
            local, off = nxt
            local.record_stream(torch.cuda.current_stream(dev))
            for k in range(c1 - c0):
                model.step(local[off[k]:off[k + 1]])
                loss_host[c0 + k:c0 + k + 1].copy_(loss_dev, non_blocking=True)
            if c1 < last:
                nxt = route_chunk(c1, min(c1 + CH, last))

    if peer:
        run_routed(0, W)
    else:
        run(0, W, host)
    torch.cuda.synchronize()
    dist.barrier()
    ev0.record()
    if peer:
        run_routed(W, W + K)
    else:
        for s in range(W, W + K):
            model.step(host[s].to(dev, non_blocking=True))
            loss_host[s:s + 1].copy_(loss_dev, non_blocking=True)
    ev1.record()
    torch.cuda.synchronize()
    dist.barrier()
    ms2 = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
    dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    check()
    phases = None
    # the fused peer path always adds its per-rank phase profile (10 serialised steps AFTER both timed regions): it is
    # what says which rank the others wait for at the barrier; --no-phases drops it
    want_phases = args.phases or (peer and not getattr(args, "no_phases", False))
    if args.phases and not peer:
        model.profile = []
        run(0, min(nb, 10), devtri)
        phases = model.profile_summary()
        model.profile = None
    elif want_phases:
        handle.set_timing(2)
        run(0, min(nb, 10), devtri)
        phases, _ = model.phase_ms()
        inner, _ = handle.phase_ms()
        phases["compute_push_detail"] = {k: round(v, 4) for k, v in inner.items()}
        handle.set_timing(0)
    if args.trace and peer:
        torch.cuda.synchronize()
        dist.barrier()
        handle.trace_start()
        run(0, min(nb, 12), devtri)
        rows = [[round(x, 3) for x in row] for row in handle.trace_dump()]
        for r in range(world):
            if r == rank:
                print(f"rank {rank} trace_ms(book_begin, book_end, kernels_begin, compute_end):", rows, flush=True)
            dist.barrier()
    by_rank = None
    if want_phases and peer:                        # which rank waits for which: the phases of every rank, side by side
        mine = {"rank": rank, "sm_mhz": (clocks.summary()["sm_mhz"] if clocks is not None else None)}
        mine.update({k: round(v, 4) for k, v in phases.items() if k != "compute_push_detail"})
        mine["main"] = phases["compute_push_detail"].get("main")
        by_rank = [None] * world
        dist.all_gather_object(by_rank, mine)
    if rank == 0:
        ms_total, ms_e2e = float(ms), float(ms2)
        value = B * world * K / (ms_total * 1e-3)
        # NVLink bytes per step and direction at one GPU: it RECEIVES the rows it fetches and SERVES the rows its peers
        # fetch from it (egress), and it PUSHES its row sums (egress) and receives its peers' (ingress); by symmetry
        # every direction carries (remote rows) x 4D bytes twice.  wire_rows = 2 x remote rows of this rank.
        each_way = wire_rows / K * 4 * D
        peak_nvl = 770.0
        step_s = ms_total / K * 1e-3
        line = {"metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": cfg["workload"], "user_num": U, "item_num": I, "dim": D,
                           "batch_per_gpu": B, "global_batch": B * world, "lr": cfg["lr"], "wd": cfg["wd"],
                           "sharding": ("block rows, triples routed to the user's owner; item rows read from / row "
                                        "sums stored to the owners' memory by the step kernels over NVLink (peer "
                                        "pointers), flag barriers, deterministic owner-side merge") if peer else
                                       ("block rows, triples routed to the user's owner, item rows + row gradients "
                                        "exchanged by NCCL all-to-all"),
                           "exchange": args.exchange, "peer_mapping": args.mapping if peer else None,
                           "main_schedule": f"chunks dealt round-robin over {world} owner ranges" if peer else None,
                           "l2": "inputs larger than L2", "lazy_decay_materialized_in_timed_region": False,
                           "parity_selfcheck": parity},
                "clocks": clocks.summary() if clocks is not None else None,
                "e2e": {"value": B * world * K / (ms_e2e * 1e-3), "unit": unit, "ms_per_step": ms_e2e / K,
                        "h2d_bytes_per_step": B * 12 * world, "d2h_bytes_per_step": 8 * world,
                        "path": ("pinned host triples with global ids -> device copy -> daisy_route_triples (owner "
                                 "routing on the device, chunks of 10 steps on a side stream) -> daisy_shard_step, "
                                 "loss read back per step") if peer else "host triples -> NCCL-exchange step"},
                "gpu_launches": int(launches),
                "roofline": {"bound": "nvlink", "achieved": each_way / step_s / 1e9, "peak": peak_nvl,
                             "unit": "GB/s per direction per GPU", "frac": each_way / step_s / 1e9 / peak_nvl,
                             "traffic": None, "peak_source": "measured peer copy (B200_PROFILING.md)",
                             "remote_rows_per_step_per_gpu": wire_rows / K / 2,
                             "nvlink_bytes_per_step_per_gpu_each_way": each_way,
                             "note": "whole step (compute + barriers + owner merge), not the fused kernel alone",
                             "hbm_whole_step_frac": (B * (24 * D + 12) / step_s / 1e9) / 6461.8}}
        if phases:
            line["phase_ms(device,host)"] = phases
        if by_rank:
            line["phase_ms_by_rank"] = by_rank
        print(json.dumps(line), flush=True)
    dist.destroy_process_group()
