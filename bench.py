#!/usr/bin/env python
"""bench.py -- BPR-MF training throughput (triples/s) and HBM roofline fraction on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]

N = 1 : BASELINE.json configs[3] -- BPR-MF synthetic 10M users x 2M items, dim 128, batch 1M triples (the largest
        single-GPU configuration the metric is quoted on): users uniform, positive items Zipf(1.0) over a permuted
        catalogue, negatives uniform; fp32; lr .01, wd .001 (SURVEY.md 8d).
N > 1 : BASELINE.json configs[4] -- 100M users x 20M items row-sharded over the N GPUs, 1M triples per GPU per
        step (weak scaling), launched by torchrun (one rank per GPU).

One step = one pass of the hot path (daisy_bpr_step) over one batch of synthetic triples.  The lazy L2 decay is exact
(c updated every step, scores use c^2); folding c into all rows is needed when weights leave the library or c < 1e-4, is
timed next to the steps and reported as materialize_ms (--materialize-every N puts one inside the timed region).
  value : whole-job triples/s with the triples already resident in HBM (CUDA events, max over ranks)
  e2e   : the same through the public API (BPRSGD.step on pinned HOST triples -> daisy_bpr_step_host), with
          the H2D copy of every step's triples and a D2H read of every step's loss inside the timed region
  roofline : dominant kernel (k_bpr_main_tma) -- algorithmic bytes (24*D+12 per triple) / its mean launch time,
          measured live with CUDA events on the launching stream, against MEASURED_PEAKS.json
  cpu_baseline : the reference's CPU path (oracle TorchPort: nn.Embedding-equivalent tables + autograd +
          optim.SGD, the calls of BPRMFRecommender.py:172-176) timed on this box's host cores, bounded sample
--impl reference : the reference arm -- the same CPU path timed alone, same metric / config.

Secondary lines (not the driver's metric; `profiles/` holds one of each):
  --workload config3 [--batch B] [--epoch-api]   ml-20m shape (L2-resident), B = 65 536 by default; --epoch-api runs the K
                     timed steps through ONE daisy_bpr_epoch call (what BPRMFRecommender.fit does)
  --workload bprfm_bn / sgns / neumf   the next-row paths (BPR-FM with batch norm + dropout, Item2Vec / SGNS,
                     NCF 'NeuMF-end')
  --workload svdpp     SVD++ (daisy_svdpp_fit) on the ml-1m shape at the script's defaults (n_factors 20)
  --workload config1   ml-100k, 20 epochs + HR@10 / NDCG@10 through BPRMFRecommender.fit, reference loop beside it
  --workload config2   funk-SVD (daisy_mf_fit) on the ml-1m shape
  --workload eval      full-catalogue top-100 for 16 384 users x 2 M items
  --workload sampler   device-side negative sampler on the ml-20m shape
  --workload gmf       NCF-GMF training step (daisy_gmf_step) on the ml-100k shape, batch 256
  --workload bprfm     BPR-FM training step (daisy_bprfm_adagrad_step) on the ml-100k shape, batch 4 096
  --phases / --trace   per-phase device times (serialised) / timeline of bookkeeping vs table kernels
  --dump-outputs DIR   config3 / config4: after the timed steps, the loss of the last timed call and a fixed sample of
                     the trained tables as DIR/<name>.npy (sample_outputs), so that two builds can be compared on the same
                     seeded inputs
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True                  # the benchmark writes nothing into the tree it runs from

import numpy as np  # noqa: E402

CFG4 = dict(workload="BPR-MF synthetic 10M users x 2M items, dim 128, batch 1M triples (BASELINE.json configs[3])",
            user_num=10_000_000, item_num=2_000_000, dim=128, batch=1_000_000, lr=0.01, wd=0.001, zipf=1.0)
CFG5 = dict(workload="BPR-MF synthetic 100M users x 20M items, dim 128, row-sharded, 1M triples per GPU per step "
                     "(BASELINE.json configs[4])",
            user_num=100_000_000, item_num=20_000_000, dim=128, batch=1_000_000, lr=0.01, wd=0.001, zipf=1.0)
CFG3 = dict(workload="BPR-MF on ml-20m-shaped synthetic implicit data (138k users x 27k items, dim 128), Zipf item "
                     "popularity, batch 65536 (BASELINE.json configs[2])",
            user_num=138_493, item_num=27_278, dim=128, batch=65_536, lr=0.01, wd=0.001, zipf=1.0)
CFG2 = dict(workload="Funk-SVD SGD (matrix_factorization.pyx) on ml-1m-shaped synthetic ratings, dim 128 "
                     "(BASELINE.json configs[1])",
            user_num=6040, item_num=3706, n=1_000_209, dim=128, lr=0.005, reg=0.02)
METRIC = "bpr_mf_train_triples_per_s"
UNIT = "triples/s"


def alg_bytes_per_triple(dim):
    """SURVEY.md 8d: gather 3 rows + scatter 3 rows (fp32) + 12 B of ids."""
    return 24 * dim + 12


DUMP_ROWS = 16_384


def sample_outputs(model, last_batch, loss, seed=2019):
    """What a caller of the timed step holds after its last call, as a fixed sample small enough to store (about 42 MB
    at D = 128): the loss the call returned, the rows of the last batch's first DUMP_ROWS triples (rows that step
    updated; hot items included) and DUMP_ROWS rows of each table at ids drawn with a fixed seed.  The tables must be
    materialized."""
    import torch
    P, Q = model.embed_user.weight.detach(), model.embed_item.weight.detach()
    rng = np.random.default_rng(seed)
    uid = torch.from_numpy(np.sort(rng.choice(P.shape[0], min(DUMP_ROWS, P.shape[0]), replace=False)))
    iid = torch.from_numpy(np.sort(rng.choice(Q.shape[0], min(DUMP_ROWS, Q.shape[0]), replace=False)))
    tri = last_batch[:DUMP_ROWS].long()

    def rows(table, ids):
        return table.index_select(0, ids.to(table.device)).cpu().numpy().astype(np.float32)

    return {"loss": loss.detach().reshape(1).cpu().numpy().astype(np.float64),
            "user_rows": rows(P, uid), "item_rows": rows(Q, iid),
            "last_batch_user_rows": rows(P, tri[:, 0]), "last_batch_pos_item_rows": rows(Q, tri[:, 1]),
            "last_batch_neg_item_rows": rows(Q, tri[:, 2])}


def write_outputs(dirname, outputs):
    os.makedirs(dirname, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", d
    return 6650.0, "fallback (B200_PROFILING.md)", {}


# ------------------------------------------------------------------------------------------------
# clocks: sampled with NVML during the timed regions
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index, period_s=None):
        self.period_s = float(os.environ.get("DAISY_CLOCK_PERIOD_S", "0.02")) if period_s is None else period_s
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        self._h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._h = None

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                    nv.nvmlDeviceGetCurrentClocksThrottleReasons
                r = int(get(self._h))
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period_s)

    def start(self):
        if self._h is not None:
            self._stop.clear()
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        if self._thread is not None:
            self._stop.set()
            self._thread.join()
            self._thread = None

    def summary(self):
        return {"sm_mhz": int(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the reference's own CPU path (oracle port), bounded sample
# ------------------------------------------------------------------------------------------------
def cpu_reference(cfg, steps, warmup, budget_s, seed=2019):
    """Times TorchPort.step (== BPRMFRecommender.py:172-176) on the host cores on `cfg`'s shapes.
    Each step is a full batch of cfg['batch'] triples; the number of timed steps is capped by `budget_s`."""
    import torch
    from oracle.bpr_oracle import TorchPort
    from recommend_lib_b200.sampler import synthetic_triples
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    U, I, D, B = cfg["user_num"], cfg["item_num"], cfg["dim"], cfg["batch"]
    note = ""
    try:
        g = torch.Generator().manual_seed(seed)
        P0 = torch.empty((U, D), dtype=torch.float32).normal_(0, 0.01, generator=g)
        Q0 = torch.empty((I, D), dtype=torch.float32).normal_(0, 0.01, generator=g)
        port = TorchPort(P0, Q0, cfg["lr"], cfg["wd"], threads=cores)
        del P0, Q0
    except (MemoryError, RuntimeError) as e:          # host too small for the dense tables + dense grads
        raise SystemExit(f"cpu reference cannot allocate config tables: {e}")
    n_batches = max(1, min(steps + warmup, 4))
    tri = synthetic_triples(n_batches * B, U, I, seed=seed, stream=99, zipf=cfg["zipf"]).reshape(n_batches, B, 3)
    t_w0 = time.time()
    for w in range(max(1, min(warmup, 1))):
        port.step(tri[w % n_batches])
    t_step = (time.time() - t_w0) / max(1, min(warmup, 1))
    k = int(max(1, min(steps, budget_s // max(t_step, 1e-3))))
    t0 = time.time()
    for s in range(k):
        port.step(tri[(s + 1) % n_batches])
    dt = time.time() - t0
    if k < steps:
        note = f"; timed {k} of the requested {steps} steps to stay inside {budget_s:.0f} s"
    return dict(value=B * k / dt, steps=k, ms_per_step=1e3 * dt / k, cores=cores, kind="port",
                sample=f"{k} full steps of {B} triples on the full {U}x{I}x{D} tables (dense grads + dense SGD/L2 "
                       f"over every row, as the reference does){note}")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CFG4 if args.gpus == 1 else CFG5
    if args.gpus > 1:
        # config 5's 61 GB of tables + dense gradients do not fit the reference's single-process CPU path;
        # the reference arm times the per-GPU shard shape (tables / N) -- one rank's share of the work.
        cfg = dict(CFG5, user_num=CFG5["user_num"] // args.gpus, item_num=CFG5["item_num"] // args.gpus,
                   workload=CFG5["workload"] + f" -- reference arm on one rank's 1/{args.gpus} shard")
    r = cpu_reference(cfg, args.steps, args.warmup, budget_s=150.0)
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": r["steps"], "warmup": min(args.warmup, 1), "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["workload"], "user_num": cfg["user_num"], "item_num": cfg["item_num"],
                       "dim": cfg["dim"], "batch": cfg["batch"], "lr": cfg["lr"], "wd": cfg["wd"]},
            "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                             "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if args.gpus > 1:
        # said in the line itself: this arm is NOT the b200 arm's configuration (one rank's 1/N shard of the tables, one
        # rank's batch), so a ratio of the two values is not a like-for-like speed-up
        line["same_config"] = False
        line["config"]["note"] = (f"config 5 does not fit the reference's single-process CPU path (61 GB of tables + dense "
                                  f"gradients): one rank's 1/{args.gpus} shard with one rank's batch, for scale only -- "
                                  f"not comparable with the {args.gpus}-GPU line")
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# single GPU: config 4
# ------------------------------------------------------------------------------------------------
def run_single(args):
    import torch
    from recommend_lib_b200.bpr import BPR, BPRSGD
    from recommend_lib_b200.sampler import synthetic_triples
    cfg = dict(CFG3 if args.workload == "config3" else CFG4)
    if args.scale != 1.0:                      # debugging aid only; the default (1.0) is the named configuration
        cfg["user_num"] = int(cfg["user_num"] * args.scale)
        cfg["item_num"] = int(cfg["item_num"] * args.scale)
        cfg["workload"] += f" SCALED x{args.scale}"
    if args.batch:
        cfg["batch"] = args.batch
    U, I, D, B = cfg["user_num"], cfg["item_num"], cfg["dim"], cfg["batch"]
    K, W = args.steps, args.warmup
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    torch.manual_seed(2019)
    model = BPR(1, 1, D, max_batch=B)                      # tiny CPU init, real tables allocated on the device
    model.user_num, model.item_num = U, I
    model.embed_user.weight = torch.nn.Parameter(torch.empty((U, D), device=dev).normal_(0, 0.01), requires_grad=False)
    model.embed_item.weight = torch.nn.Parameter(torch.empty((I, D), device=dev).normal_(0, 0.01), requires_grad=False)
    opt = BPRSGD(model, lr=cfg["lr"], weight_decay=cfg["wd"])
    h = model.handle(B)
    if args.l2_window:                          # north star: hot item rows pinned in L2 (access-policy window)
        model.pin_hot_items(args.l2_window_rows or None, 1.0)

    nb = K + W
    # --hot-prefix: item id = popularity rank (what a popularity-ordered catalogue, or a popularity remap, looks like):
    # the Zipf head is a contiguous prefix of the item table, which is what an access-policy window can cover
    host = torch.from_numpy(synthetic_triples(nb * B, U, I, seed=2019, zipf=cfg["zipf"],
                                              permute_items=not args.hot_prefix).reshape(nb, B, 3)).pin_memory()
    devtri = host.to(dev)
    loss_dev = torch.zeros(nb, dtype=torch.float64, device=dev)
    loss_host = torch.zeros(nb, dtype=torch.float64).pin_memory()
    clocks = ClockSampler(0)
    mat_every = args.materialize_every

    def device_resident_pass(first, count):
        if args.epoch_api:                      # one daisy_bpr_epoch call runs all `count` steps (BPRSGD.epoch)
            opt.epoch(devtri[first:first + count].reshape(-1, 3), B, loss_out=loss_dev[first:first + 1])
            return
        for s in range(first, first + count):
            opt.step(devtri[s], loss_out=loss_dev[s:s + 1], ready=True)   # uploaded + synchronised before timing
            if mat_every and (s + 1) % mat_every == 0:
                model.materialize()

    # ---- value: triples resident in HBM ----
    device_resident_pass(0, W)
    model.check()
    torch.cuda.synchronize()
    h.set_timing(1)
    launches0 = h.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    clocks.start()
    torch.cuda.synchronize()
    ev0.record()
    t_host0 = time.perf_counter()
    device_resident_pass(W, K)
    ev1.record()
    host_enqueue_ms = (time.perf_counter() - t_host0) * 1e3 / K
    torch.cuda.synchronize()
    clocks.stop()
    ms_total = ev0.elapsed_time(ev1)
    # The lazy L2 decay (DESIGN.md section 3) is exact, not deferred arithmetic: every step updates c, scores use c^2,
    # and the tables only need folding when weights leave the library or c < 1e-4 (every ~920 000 steps at this lr*wd).
    # It is therefore timed NEXT TO the steps, not inside them (same accounting as the N > 1 line); materialize_ms says
    # what one fold of the 12.3 GB costs, --materialize-every N puts one inside the timed region every N steps.
    evm0, evm1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    evm0.record()
    model.materialize()
    evm1.record()
    torch.cuda.synchronize()
    materialize_ms = evm0.elapsed_time(evm1)
    launches = h.launches - launches0
    main_ms, main_n = h.main_kernel_ms()
    h.set_timing(0)
    model.check()
    value = B * K / (ms_total * 1e-3)
    outputs = None
    if args.dump_outputs:                       # the e2e pass below trains on: sample the timed pass's result now
        outputs = sample_outputs(model, devtri[W + K - 1], loss_dev[W if args.epoch_api else W + K - 1])

    # ---- e2e: host triples through the public API, loss read back every step ----
    def e2e_pass(first, count):
        if args.epoch_api:                      # pinned host triples of `count` steps, loss read back once per call
            opt.epoch(host[first:first + count].reshape(-1, 3), B, loss_out=loss_dev[first:first + 1])
            loss_host[first:first + 1].copy_(loss_dev[first:first + 1], non_blocking=True)
            return
        for s in range(first, first + count):
            opt.step(host[s], loss_out=loss_dev[s:s + 1])
            loss_host[s:s + 1].copy_(loss_dev[s:s + 1], non_blocking=True)
            if mat_every and (s + 1) % mat_every == 0:
                model.materialize()

    loss_dev.zero_()
    e2e_pass(0, W)
    torch.cuda.synchronize()
    clocks.start()
    ev0.record()
    e2e_pass(W, K)
    ev1.record()
    torch.cuda.synchronize()
    clocks.stop()
    ms_e2e = ev0.elapsed_time(ev1)
    model.materialize()
    model.check()
    e2e_value = B * K / (ms_e2e * 1e-3)
    losses = loss_host[W:W + K].numpy()
    if args.epoch_api:
        losses = losses[:1] / K                 # the call accumulates the loss of its K steps
    assert np.isfinite(losses).all() and (losses > 0).all(), "e2e losses not finite"

    # ---- optional per-phase breakdown (not part of the timed numbers) ----
    trace = None
    if args.trace:
        torch.cuda.synchronize()
        h.trace_start()
        device_resident_pass(0, min(nb, 12))
        trace = [[round(x, 4) for x in row] for row in h.trace_dump()]
    phases = None
    if args.phases:
        h.set_timing(2)
        device_resident_pass(0, min(nb, 10))
        phases, _ = h.phase_ms()
        h.set_timing(0)

    peak, peak_src, _ = measured_peaks()
    abytes = alg_bytes_per_triple(D) * B
    achieved = abytes / (main_ms * 1e-3) / 1e9 if main_ms > 0 else 0.0
    traffic = None
    tp = os.path.join(ROOT, "profiles", "main_kernel_traffic.json")
    if os.path.exists(tp) and args.workload == "config4" and not args.batch and args.scale == 1.0:
        try:
            traffic = json.load(open(tp)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    cpu = None
    if not args.no_cpu_baseline:
        del devtri
        r = cpu_reference(cfg, steps=3, warmup=1, budget_s=args.cpu_budget)
        cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["workload"], "user_num": U, "item_num": I, "dim": D, "batch": B,
                       "lr": cfg["lr"], "wd": cfg["wd"], "item_popularity": "zipf(1.0), " + ("id = popularity rank" if args.hot_prefix else "permuted"),
                       "l2": ("inputs larger than L2 (6.1 GB of tables, ~3 GB touched per step vs 126 MB L2)"
                              if args.workload == "config4" else
                              "tables (85 MB) fit the 126 MB L2: L2-resident workload, the HBM roofline does not bound it"),
                       "l2_access_policy_window": bool(args.l2_window),
                       "l2_window_rows": (args.l2_window_rows or I) if args.l2_window else 0,
                       "hot_items_are_a_prefix": bool(args.hot_prefix),
                       "lazy_decay_materialized_in_timed_region": (False if not mat_every else f"every {mat_every} steps"),
                       "lazy_decay": ("exact: c updated every step, scores use c^2; one fold of all rows takes materialize_ms "
                                      "and is needed when weights leave the library or c < 1e-4 (every ~920 000 steps here)"),
                       "api": ("BPRSGD.epoch -> daisy_bpr_epoch: ONE library call runs the K timed steps"
                               if args.epoch_api else "BPRSGD.step -> daisy_bpr_step[_host]: one library call per step"),
                       "e2e_loss_readback": ("async D2H of the call's accumulated loss, once per daisy_bpr_epoch call"
                                             if args.epoch_api else
                                             "async D2H of every step's loss into pinned memory, synchronised at the end")},
            "clocks": clocks.summary(),
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / K, "h2d_bytes_per_step": B * 12,
                    "d2h_bytes_per_step": 8 / K if args.epoch_api else 8},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "k_bpr_main_tma<1, SgdOpt, false>", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak if peak else None, "traffic": traffic,
                         "traffic_source": "ncu --set full capture of this kernel on this workload (profiles/main_kernel_traffic.json)",
                         "frac_on_dram_traffic": (traffic / (main_ms * 1e-3) / 1e9 / peak) if (traffic and main_ms > 0 and peak) else None,
                         "algorithmic_bytes_per_launch": abytes, "kernel_ms": main_ms, "launches_timed": int(main_n),
                         "peak_source": peak_src,
                         "whole_step_frac": (abytes / (ms_total / K * 1e-3) / 1e9) / peak},
            "cpu_baseline": cpu,
            "final_loss_per_triple": float(losses[-1] / B)}
    line["host_enqueue_ms_per_step"] = round(host_enqueue_ms, 4)
    line["materialize_ms"] = round(materialize_ms, 4)
    if phases:
        line["phase_ms"] = {k: round(v, 4) for k, v in phases.items()}
    if trace:
        line["trace_ms(book_begin,book_end,kernels_begin,kernels_end)"] = trace
    if outputs:
        write_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# config 1: ml-100k, 20 epochs + HR@10 / NDCG@10 (secondary line: the reference's own CPU-runnable case)
# ------------------------------------------------------------------------------------------------
def run_config1(args):
    """BPRMFRecommender.fit on the real ml-100k split (tests/golden/ml100k_split.npz: loo-by-time, 99 057 train
    pairs x num_ng 4 = 396 228 triples per epoch, B 4 096, D 64, lr 0.01, wd 0.001), 20 epochs, HR@10 / NDCG@10 on
    1 + 999 candidates per user.  value = training triples/s over the epochs' step loops (daisy_bpr_epoch: H2D of
    the epoch's triples + 97 steps + loss read-back; sampling and evaluation are timed separately).  The CPU line
    beside it is the reference's loop restated (TorchPort == BPRMFRecommender.py:172-176) on the same triples."""
    import torch
    from recommend_lib_b200 import data
    from recommend_lib_b200.bpr import BPRMFRecommender
    from recommend_lib_b200.sampler import TripleSampler
    s = np.load(os.path.join(ROOT, "tests", "golden", "ml100k_split.npz"))
    tr, te = s["train_pairs"].astype(np.int64), s["test_pairs"].astype(np.int64)
    U, I = int(s["user_num"]), int(s["item_num"])
    allp = np.concatenate([tr, te])
    eu, ec = data.eval_candidates(allp[:, 0], allp[:, 1], te[:, 0], te[:, 1], I, 999, 2019)
    epochs = 20
    clocks = ClockSampler(0)
    rec = BPRMFRecommender(U, I, factor_num=64, lr=0.01, wd=0.001, batch_size=4096, epochs=2, num_ng=4, topk=10,
                           seed=2019, device="cuda:0")
    rec.fit(tr)                                            # warm-up: 2 epochs on a throw-away model
    rec = BPRMFRecommender(U, I, factor_num=64, lr=0.01, wd=0.001, batch_size=4096, epochs=epochs, num_ng=4, topk=10,
                           seed=2019, device="cuda:0")
    h0 = rec.model.handle(4096).launches
    clocks.start()
    t0 = time.time()
    rec.fit(tr, eu, ec)
    wall = time.time() - t0
    clocks.stop()
    launches = rec.model.handle(4096).launches - h0
    # the same fit with negatives drawn on the device (daisy_sample_triples): no host sampling, no H2D of triples
    rec_d = BPRMFRecommender(U, I, factor_num=64, lr=0.01, wd=0.001, batch_size=4096, epochs=epochs, num_ng=4, topk=10,
                             seed=2019, device="cuda:0", sampler="device")
    rec_d.fit(tr[:4096])                                   # warm-up (first launch of the sampler kernels)
    rec_d = BPRMFRecommender(U, I, factor_num=64, lr=0.01, wd=0.001, batch_size=4096, epochs=epochs, num_ng=4, topk=10,
                             seed=2019, device="cuda:0", sampler="device")
    t0 = time.time()
    rec_d.fit(tr, eu, ec)
    wall_d = time.time() - t0
    n = len(tr) * 4
    train_s = sum(e["train_s"] for e in rec.history)
    steps = epochs * ((n + 4095) // 4096)
    # CPU: one epoch of the reference's loop on the same triples
    from oracle.bpr_oracle import TorchPort
    torch.manual_seed(2019)
    cores = os.cpu_count() or 1
    P0 = torch.empty((U, 64)).normal_(0, 0.01)
    Q0 = torch.empty((I, 64)).normal_(0, 0.01)
    port = TorchPort(P0, Q0, 0.01, 0.001, threads=cores)
    tri = TripleSampler(tr, I, num_ng=4, seed=2019).sample_epoch(0)
    t0 = time.time()
    for b in range(0, len(tri), 4096):
        port.step(tri[b:b + 4096])
    cpu_dt = time.time() - t0
    last = rec.history[-1]
    line = {"metric": METRIC, "value": n * epochs / train_s, "unit": UNIT, "n_gpus": 1, "steps": steps, "warmup": 2 * 97,
            "ms_per_step": 1e3 * train_s / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "ml-100k (tests/golden/ml100k_split.npz)",
            "config": {"workload": "BPR-MF on ml-100k (943 users x 1682 items, dim 64, fp32), 20 epochs + HR@10/NDCG@10 "
                                   "(BASELINE.json configs[0])", "user_num": U, "item_num": I, "dim": 64, "batch": 4096,
                       "lr": 0.01, "wd": 0.001, "num_ng": 4, "epochs": epochs, "triples_per_epoch": n,
                       "timing": "host wall clock around each epoch's daisy_bpr_epoch call + loss read-back "
                                 "(synchronised); latency-bound (0.67 MB of tables), no roofline",
                       "l2": "tables are L2-resident"},
            "clocks": clocks.summary(),
            "e2e": {"value": n * epochs / wall, "unit": UNIT, "h2d_bytes_per_step": 4096 * 12, "d2h_bytes_per_step": 8 / 97,
                    "note": "whole fit(): host negative sampling + training + per-epoch metric_eval"},
            "gpu_launches": int(launches),
            "roofline": None,
            "cpu_baseline": {"value": n / cpu_dt, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "one epoch (97 steps of 4 096 triples) of the reference loop, same triples"},
            "final": {"loss": last["loss"], "hr@10": last["hr"], "ndcg@10": last["ndcg"]},
            "device_sampler": {"e2e_value": n * epochs / wall_d, "unit": UNIT, "fit_wall_s": wall_d,
                               "final": {"loss": rec_d.history[-1]["loss"], "hr@10": rec_d.history[-1]["hr"],
                                         "ndcg@10": rec_d.history[-1]["ndcg"]},
                               "note": "whole fit() with BPRMFRecommender(sampler='device'): other negatives than the "
                                       "host sampler's, so the trajectory is its own (same distribution)"},
            "fit_wall_s": wall,
            "sample_s_per_epoch": float(np.mean([e["sample_s"] for e in rec.history]))}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# NCF-GMF (SURVEY 8f N3; secondary line)
# ------------------------------------------------------------------------------------------------
def run_gmf(args):
    """samples/s of the fused GMF step (daisy_gmf_step: gather, BCE, deterministic row sums, dense Adam) at the
    reference script's defaults on the ml-100k shape (943 x 1 682, factor_num 32, batch 256, lr 0.001;
    NCFRecommender.py:140-160), 1 positive + 4 sampled negatives per interaction, next to the closed-form restatement
    of the reference loop (oracle/gmf_oracle.py, numpy) on the host."""
    import torch
    from recommend_lib_b200.ncf import NCF, GMFAdam
    U, I, D, B = 943, 1682, 32, args.batch or 256
    K, W = max(args.steps, 200), max(args.warmup, 20)
    rng = np.random.default_rng(2019)
    n = (K + W) * B
    users = rng.integers(0, U, n).astype(np.int64)
    items = rng.integers(0, I, n).astype(np.int64)
    labels = (np.arange(n) % 5 == 0).astype(np.float32)
    dev = torch.device("cuda:0")
    torch.manual_seed(2019)
    model = NCF(U, I, D, 3, 0.0, "GMF", max_batch=B).to(dev)
    opt = GMFAdam(model, lr=0.001)
    packed = torch.from_numpy(np.stack([users, items, labels.astype(np.int64)], 1).astype(np.int32)).reshape(K + W, B, 3)
    host = packed.pin_memory()
    devs = packed.to(dev)

    run = lambda first, count, src: opt.epoch(src[first:first + count].reshape(-1, 3), B)   # ONE daisy_gmf_epoch call
    run(0, W, devs)
    model.check()
    torch.cuda.synchronize()
    l0 = model.handle(B).launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    run(W, K, devs)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    launches = model.handle(B).launches - l0
    loss_host = torch.zeros(K + W, dtype=torch.float64).pin_memory()
    ev0.record()
    run(W, K, host)                                 # e2e: pinned host samples in, the call's summed loss read back
    loss_host[:1].copy_(opt._loss, non_blocking=True)
    ev1.record()
    torch.cuda.synchronize()
    ms2 = ev0.elapsed_time(ev1)
    loss = float(loss_host[0]) / K
    model.check()
    from oracle import gmf_oracle
    st = gmf_oracle.GMFAdam(np.random.default_rng(1).normal(0, 0.01, (U, D)), np.random.default_rng(2).normal(0, 0.01, (I, D)),
                            np.random.default_rng(3).normal(0, 0.3, D), np.zeros(1), lr=0.001, dtype=np.float32)
    nc = 200
    t0 = time.time()
    for s in range(nc):
        st.step(users[s * B:(s + 1) * B], items[s * B:(s + 1) * B], labels[s * B:(s + 1) * B])
    cpu_dt = time.time() - t0
    bytes_step = B * (2 * 4 * D * 3) + 8 * 4 * D * (U + I)      # gather + stage + grad rows, dense Adam pass
    line = {"metric": "gmf_train_samples_per_s", "value": B * K / (ms * 1e-3), "unit": "samples/s", "n_gpus": 1, "steps": K,
            "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "NCF-GMF training step on the ml-100k shape (943 x 1682, factor_num 32, batch 256, Adam lr 0.001)",
                       "user_num": U, "item_num": I, "dim": D, "batch": B,
                       "l2": "tables + Adam moments (1 MB) are L2-resident; the step is launch-latency-bound (5 launches)"},
            "e2e": {"value": B * K / (ms2 * 1e-3), "unit": "samples/s", "ms_per_step": ms2 / K,
                    "h2d_bytes_per_step": B * 12, "d2h_bytes_per_step": 8 / K,
                    "api": "GMFAdam.epoch -> daisy_gmf_epoch: one library call runs the K timed steps"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": bytes_step / (ms / K * 1e-3) / 1e9, "peak": measured_peaks()[0],
                         "unit": "GB/s", "frac": bytes_step / (ms / K * 1e-3) / 1e9 / measured_peaks()[0], "traffic": None,
                         "note": "latency-bound at this size; bytes = per-sample rows + the dense Adam pass over both tables"},
            "cpu_baseline": {"value": B * nc / cpu_dt, "unit": "samples/s", "cores": 1, "kind": "port",
                             "sample": f"{nc} steps of the closed-form restatement (numpy, float32) of the reference loop"},
            "final_loss": loss}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# BPR-FM (SURVEY 8f N3; secondary line)
# ------------------------------------------------------------------------------------------------
def run_bprfm(args):
    """triples/s of the fused BPR-FM step (daisy_bprfm_adagrad_step: the BPR kernels on augmented rows + Adagrad) at the
    reference script's defaults on the ml-100k shape (943 + 1 682 features, hidden_factor 64, batch 4 096, Adagrad lr
    0.05; BPRFMRecommender.py:122-150) with batch_norm off / dropout 0, next to the closed-form restatement of the
    reference loop (oracle/bprfm_oracle.py, numpy) on the host."""
    import torch
    from recommend_lib_b200.bprfm import BPRFM, FMAdagrad
    from recommend_lib_b200.sampler import synthetic_triples
    U, I, F, B = 943, 1682, 64, args.batch or 4096
    K, W = max(args.steps, 200), max(args.warmup, 20)
    tri = synthetic_triples((K + W) * B, U, I, seed=2019, zipf=1.0).reshape(K + W, B, 3)
    dev = torch.device("cuda:0")
    torch.manual_seed(2019)
    model = BPRFM(U + I, F, False, [0.0, 0.0], user_num=U, max_batch=B).to(dev)
    opt = FMAdagrad(model, lr=0.05)
    devt = torch.from_numpy(tri).to(dev)
    for s in range(W):
        opt.step(devt[s])
    model.check()
    torch.cuda.synchronize()
    l0 = model.handle(B).launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for s in range(W, W + K):
        opt.step(devt[s])
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    launches = model.handle(B).launches - l0
    host = torch.from_numpy(tri).pin_memory()
    loss_host = torch.zeros(K + W, dtype=torch.float64).pin_memory()
    opt.loss_sum()
    ev0.record()
    for s in range(W, W + K):                       # e2e: pinned host triples in, loss read back every step
        opt.step(host[s].to(dev, non_blocking=True))
        loss_host[s:s + 1].copy_(opt._loss, non_blocking=True)
    ev1.record()
    torch.cuda.synchronize()
    ms2 = ev0.elapsed_time(ev1)
    model.check()
    from oracle import bprfm_oracle
    rng = np.random.default_rng(1)
    E = rng.normal(0, 0.01, (U + I, F)).astype(np.float32)
    b = np.zeros(U + I, np.float32)
    aE, ab = np.full_like(E, 1e-8), np.full_like(b, 1e-8)
    nc = 20
    t0 = time.time()
    for s in range(nc):
        fi = np.stack([tri[s, :, 0], U + tri[s, :, 1]], 1)
        fj = np.stack([tri[s, :, 0], U + tri[s, :, 2]], 1)
        bprfm_oracle.bprfm_adagrad_step(E, b, 0.0, aE, ab, fi, fj, lr=0.05)
    cpu_dt = time.time() - t0
    line = {"metric": "bprfm_train_triples_per_s", "value": B * K / (ms * 1e-3), "unit": "triples/s", "n_gpus": 1, "steps": K,
            "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "BPR-FM training step on the ml-100k shape (943 + 1682 features, hidden_factor 64, batch "
                                   "4096, Adagrad lr 0.05, batch_norm off, dropout 0)", "user_num": U, "item_num": I,
                       "dim": F, "batch": B, "l2": "tables (0.7 MB) are L2-resident; launch-latency-bound (3 launches)"},
            "e2e": {"value": B * K / (ms2 * 1e-3), "unit": "triples/s", "ms_per_step": ms2 / K,
                    "h2d_bytes_per_step": B * 12, "d2h_bytes_per_step": 8},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": B * (24 * (F + 4) + 12) / (ms / K * 1e-3) / 1e9,
                         "peak": measured_peaks()[0], "unit": "GB/s",
                         "frac": B * (24 * (F + 4) + 12) / (ms / K * 1e-3) / 1e9 / measured_peaks()[0], "traffic": None,
                         "note": "latency-bound at this size"},
            "cpu_baseline": {"value": B * nc / cpu_dt, "unit": "triples/s", "cores": 1, "kind": "port",
                             "sample": f"{nc} steps of the closed-form restatement (numpy, float32) of the reference loop"},
            "mean_loss_per_triple": float(loss_host[W + K - 1]) / (B * K)}      # the loss accumulates over the K e2e steps
    print(json.dumps(line), flush=True)


def run_experimental(args):
    """Secondary lines of three next-row paths (SURVEY.md 8f rows N3 / N4; DESIGN.md section 9): `--workload bprfm_bn` = BPR-FM at the script's defaults (batch norm + dropout 0.5, ml-100k shape,
    hidden_factor 64, batch 4 096, Adagrad) through FMBNAdagrad.step; `--workload sgns` = Item2Vec / SGNS at the script's
    defaults (window 5 -> 10 context items, 20 negatives, e_dim 300, batch 4 096, Adam; ml-100k vocabulary) through
    SGNSAdam.step.  Device-timed steps with resident inputs, then the same steps from pinned host inputs with the loss
    read back; the closed-form oracle on one host core beside them."""
    import torch
    dev = torch.device("cuda:0")
    torch.manual_seed(2019)
    rng = np.random.default_rng(2019)
    K, W = max(args.steps, 50), max(args.warmup, 5)
    if args.workload == "bprfm_bn":
        from recommend_lib_b200.bprfm_bn import BPRFMBN, FMBNAdagrad
        from recommend_lib_b200.sampler import synthetic_triples
        from oracle import bprfm_oracle
        U, I, F, B = 943, 1682, 64, args.batch or 4096
        tri = synthetic_triples((K + W) * B, U, I, seed=2019, zipf=1.0).reshape(K + W, B, 3)
        model = BPRFMBN(U + I, F, True, [0.5, 0.2], user_num=U).to(dev)
        model.train()
        opt = FMBNAdagrad(model, lr=0.05)
        inputs = [(torch.from_numpy(tri[s]),) for s in range(K + W)]
        units, unit, metric = B, "triples/s", "bprfm_bn_train_triples_per_s"
        handle = model.handle
        ora = bprfm_oracle.BPRFMFull(rng.normal(0, 0.01, (U + I, F)), np.zeros(U + I), 0.0, True, lr=0.05)
        ones = np.ones((B, 2))

        def cpu_step(s):
            keep = lambda: (rng.random((B, F)) >= 0.5) * 2.0
            ora.step(np.stack([tri[s, :, 0], U + tri[s, :, 1]], 1), ones, np.stack([tri[s, :, 0], U + tri[s, :, 2]], 1), ones,
                     keep(), keep())
        workload = ("BPR-FM training step at the script's defaults on the ml-100k shape (943 + 1682 features, hidden_factor "
                    "64, batch 4096, batch norm, dropout 0.5 drawn on the device, Adagrad lr 0.05)")
        h2d = B * 12
        # per triple: 3 feature rows and their Adagrad accumulators read and written (embedding + bias) + the ids
        alg_bytes = B * (3 * 2 * 2 * 4 * (F + 1) + 12)
        alg_note = "3 rows x (value + Adagrad state) x (read + write) x 4 (F + 1) B + 12 B of ids per triple"
    elif args.workload == "neumf":
        from recommend_lib_b200.ncf_mlp import NeuMF, NeuMFAdam
        from oracle import neumf_oracle
        U, I, F, L, B = 943, 1682, 32, 3, args.batch or 256
        K, W = max(args.steps, 400), max(args.warmup, 20)
        model = NeuMF(U, I, F, L, 0.0, "NeuMF-end").to(dev)
        opt = NeuMFAdam(model, lr=0.001)
        us, its = rng.integers(0, U, (K + W, B)), (rng.zipf(1.2, (K + W, B)) - 1) % I
        ys = (rng.random((K + W, B)) < 0.2).astype(np.int32)
        inputs = [(torch.from_numpy(np.stack([us[s], its[s], ys[s]], 1).astype(np.int32)),) for s in range(K + W)]
        _step = opt.step
        opt.step = lambda smp: _step(smp[:, 0], smp[:, 1], smp[:, 2])      # one packed [B, 3] tensor per step crosses PCIe
        units, unit, metric = B, "samples/s", "neumf_train_samples_per_s"
        handle = model.handle
        c = lambda t: t.detach().cpu().numpy()
        ora = neumf_oracle.NeuMFAdam("NeuMF-end", c(model.embed_user_GMF.weight), c(model.embed_item_GMF.weight),
                                     c(model.embed_user_MLP.weight), c(model.embed_item_MLP.weight),
                                     [c(m.weight) for m in model.linears()], [c(m.bias) for m in model.linears()],
                                     c(model.predict_layer.weight), c(model.predict_layer.bias))

        def cpu_step(s):
            ora.step(us[s], its[s], ys[s])
        workload = ("NCF training step, model 'NeuMF-end' at the script's defaults on the ml-100k shape (943 x 1682, factor_num "
                    "32, 3 MLP layers, batch 256, dropout 0, Adam lr 0.001)")
        h2d = B * 12
        n_param = sum(p.numel() for p in model.parameters())
        alg_bytes = 8 * 4 * n_param + B * 12       # torch's dense Adam: param, grad, m, v read + written, whatever B is
        alg_note = "dense Adam over every parameter (8 x 4 B per element per step, independent of the batch) + ids"
    else:
        from recommend_lib_b200.item2vec import Item2Vec, SGNS, SGNSAdam
        from oracle import sgns_oracle
        V, D, B, C, N = 1683, 300, args.batch or 4096, 10, 20
        counts = 1.0 / np.arange(1, V + 1)
        model = Item2Vec(vocab_size=V, embedding_size=D)
        sgns = SGNS(embedding=model, vocab_size=V, n_negs=N, weights=counts).to(dev)
        opt = SGNSAdam(sgns)
        pw = counts / counts.sum()
        iw = rng.choice(V - 1, size=(K + W, B), p=pw[1:] / pw[1:].sum()) + 1
        ow = rng.choice(V, size=(K + W, B, C), p=pw)
        inputs = [(torch.from_numpy(iw[s]).int(), torch.from_numpy(ow[s]).int()) for s in range(K + W)]
        units, unit, metric = B, "examples/s", "sgns_train_examples_per_s"
        handle = opt.handle
        ora = sgns_oracle.SGNSAdam(model.ivectors.weight.detach().cpu().numpy(), model.ovectors.weight.detach().cpu().numpy())
        wneg = pw ** 0.75 / (pw ** 0.75).sum()

        def cpu_step(s):
            ora.step(iw[s], ow[s], rng.choice(V, size=(B, C * N), p=wneg))
        workload = ("Item2Vec / SGNS training step at the script's defaults (ml-100k vocabulary of 1683, e_dim 300, batch "
                    "4096, 10 context items, 20 negatives each drawn on the device from unigram^0.75, dense Adam)")
        h2d = B * 4 * (1 + C)
        # per example: the centre row + C (1 + n_negs) output rows gathered; per step: dense Adam over both tables
        alg_bytes = B * (1 + C * (1 + N)) * 4 * D + 2 * V * D * 8 * 4
        alg_note = ("(1 + C (1 + n_negs)) rows x 4 e_dim B gathered per example + dense Adam over both tables "
                    "(8 x 4 B per element per step)")
    devin = [tuple(t.to(dev) for t in x) for x in inputs]
    for s in range(W):
        opt.step(*devin[s])
    torch.cuda.synchronize()
    opt.loss_sum()
    l0 = handle().launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for s in range(W, W + K):
        opt.step(*devin[s])
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    launches = handle().launches - l0
    loss_dev = opt.loss_sum() / K
    host = [tuple(t.pin_memory() for t in x) for x in inputs]
    loss_host = torch.zeros(K + W, dtype=torch.float64).pin_memory()
    ev0.record()
    for s in range(W, W + K):                       # e2e: pinned host ids in, loss read back every step
        opt.step(*(t.to(dev, non_blocking=True) for t in host[s]))
        loss_host[s:s + 1].copy_(opt._loss, non_blocking=True)
    ev1.record()
    torch.cuda.synchronize()
    ms2 = ev0.elapsed_time(ev1)
    nc = 20 if args.workload == "neumf" else 3
    t0 = time.time()
    for s in range(nc):
        cpu_step(s)
    cpu_dt = time.time() - t0
    line = {"metric": metric, "value": units * K / (ms * 1e-3), "unit": unit, "n_gpus": 1, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": workload, "batch": B, "status": "first version (GPU-verified in round 2)",
                                            "l2": "tables are L2-resident at this size"},
            "e2e": {"value": units * K / (ms2 * 1e-3), "unit": unit, "ms_per_step": ms2 / K, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": 8},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": alg_bytes / (ms / K * 1e-3) / 1e9, "peak": measured_peaks()[0], "unit": "GB/s",
                         "frac": alg_bytes / (ms / K * 1e-3) / 1e9 / measured_peaks()[0], "traffic": None,
                         "algorithmic_bytes_per_step": alg_bytes, "kernel": "whole step (every launch of the step)",
                         "peak_source": measured_peaks()[1],
                         "note": alg_note + "; the tables are L2-resident at the script's sizes, so the step is bound by "
                                 "launch latency and dependent passes, not by HBM: the fraction says how far from a "
                                 "bandwidth-bound regime this shape is, not how good the kernels are"},
            "cpu_baseline": {"value": units * nc / cpu_dt, "unit": unit, "cores": 1, "kind": "port",
                             "sample": f"{nc} steps of the closed-form restatement (numpy, float64) of the reference loop"},
            "mean_loss_per_step": loss_dev}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# config 2: funk-SVD (secondary line, not the driver's metric)
# ------------------------------------------------------------------------------------------------
def run_mf(args):
    """ratings/s of SVD.fit (daisy_mf_fit, dataflow kernel, float64, strictly sequential semantics) on the ml-1m
    shape, next to the reference's own Cython extension (oracle/_ref, when it was built) or its C restatement on a
    bounded sample."""
    import torch
    from recommend_lib_b200 import _lib
    from recommend_lib_b200._lib import MFParams, c_vp
    from recommend_lib_b200.sampler import synthetic_ratings
    import ctypes
    cfg = CFG2
    U, I, D, N = cfg["user_num"], cfg["item_num"], cfg["dim"], cfg["n"]
    users, items, ratings = synthetic_ratings(N, U, I, seed=2019)
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(0)
    pu = rng.normal(0, 0.1, (U, D)); qi = rng.normal(0, 0.1, (I, D))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    dpu, dqi, dbu, dbi = t(pu), t(qi), t(np.zeros(U)), t(np.zeros(I))
    du, di, dr = t(users.astype(np.int32)), t(items.astype(np.int32)), t(ratings.astype(np.float64))
    prm = MFParams(0, 1, cfg["lr"], cfg["lr"], cfg["lr"], cfg["lr"], cfg["reg"], cfg["reg"], cfg["reg"], cfg["reg"], 0.0,
                   float(ratings.mean()))
    h = _lib.Handle(0, U, I, D, 0)
    s = _lib.stream_ptr(torch, dev)
    fit = lambda ep: _lib.check(h.L.daisy_mf_fit(h.ptr, c_vp(dpu.data_ptr()), c_vp(dqi.data_ptr()), c_vp(dbu.data_ptr()),
                                                 c_vp(dbi.data_ptr()), c_vp(du.data_ptr()), c_vp(di.data_ptr()),
                                                 c_vp(dr.data_ptr()), N, ep, ctypes.byref(prm), None, s))
    fit(max(1, min(args.warmup, 2)))
    torch.cuda.synchronize()
    K = max(1, min(args.steps, 20))                     # 20 = the reference's default n_epochs (matrix_factorization.pyx:82)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    fit(K)                                              # K epochs = K passes over the 1M ratings
    ev1.record()
    torch.cuda.synchronize()
    _lib.check(h.L.daisy_check(h.ptr, s))
    ms = ev0.elapsed_time(ev1)
    # CPU side: the reference's compiled Cython SVD when present, else the C restatement; bounded sample
    from oracle import mf_oracle
    n_cpu = 200_000
    pu_c, qi_c = pu.copy(), qi.copy()
    t0 = time.time()
    mf_oracle.svd_fit(users[:n_cpu], items[:n_cpu], ratings[:n_cpu], pu_c, qi_c, n_epochs=1, biased=True,
                      lr_all=cfg["lr"], reg_all=cfg["reg"])
    cpu_dt = time.time() - t0
    line = {"metric": "funk_svd_train_ratings_per_s", "value": N * K / (ms * 1e-3), "unit": "ratings/s", "n_gpus": 1,
            "steps": K, "warmup": max(1, min(args.warmup, 2)), "ms_per_step": ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": cfg["workload"], "user_num": U, "item_num": I, "ratings": N, "dim": D,
                       "step": "one epoch (a pass over all ratings in the given order, sequential semantics); the timed "
                               "region is ONE daisy_mf_fit call of `steps` epochs, its per-fit preprocessing included",
                       "l2": "tables (10 MB in f64) are L2-resident; the bound is the longest dependency chain"},
            "roofline": {"bound": "hbm", "achieved": N * K * (2 * (16 * D + 12) + 16) / (ms * 1e-3) / 1e9,
                         "peak": measured_peaks()[0], "unit": "GB/s",
                         "frac": N * K * (2 * (16 * D + 12) + 16) / (ms * 1e-3) / 1e9 / measured_peaks()[0],
                         "traffic": None, "note": "f64 rows: 2 x (16 D + 12) + 16 B per rating; dependency-bound"},
            "cpu_baseline": {"value": n_cpu / cpu_dt, "unit": "ratings/s", "cores": 1, "kind": "port",
                             "sample": f"C restatement of the Cython loop (bit-identical to it, tests/test_oracle_golden.py), "
                                       f"one epoch over the first {n_cpu} ratings, single thread (the loop is serial); "
                                       "the reference's own fit adds ~50 us/rating of DataFrame.iterrows overhead"},
            "gpu_launches": int(h.launches)}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# SVD++ (SURVEY 8f N4; secondary line)
# ------------------------------------------------------------------------------------------------
def run_svdpp(args):
    """ratings/s of SVDpp.fit (daisy_svdpp_fit: one thread block walking the ratings in order, float64) on the
    ml-1m-shaped synthetic ratings of config 2 at the script's defaults (n_factors 20, lr 0.007, reg 0.02, SVDppRecommender.py:30-44),
    next to the C restatement of the reference loop on a bounded sample.  EXPERIMENTAL path (csrc/svdpp.cu)."""
    import ctypes
    import torch
    from recommend_lib_b200 import _lib
    from recommend_lib_b200._lib import SVDppParams, c_vp
    from recommend_lib_b200.sampler import synthetic_ratings
    from recommend_lib_b200.svdpp import user_histories
    cfg = CFG2
    U, I, D, N = cfg["user_num"], cfg["item_num"], 20, cfg["n"]
    users, items, ratings = synthetic_ratings(N, U, I, seed=2019)
    ratings = ratings.astype(np.float64)
    ptr, idx, mult = user_histories(users, items, U)
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(0)
    pu, qi, yj = rng.normal(0, 0.1, (U, D)), rng.normal(0, 0.1, (I, D)), rng.normal(0, 0.1, (I, D))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    dpu, dqi, dyj, dbu, dbi = t(pu), t(qi), t(yj), t(np.zeros(U)), t(np.zeros(I))
    du, di, dr = t(users.astype(np.int32)), t(items.astype(np.int32)), t(ratings)
    dptr, didx = t(ptr), t(idx)
    dmult = t(mult) if mult is not None else None
    prm = SVDppParams(.007, .007, .007, .007, .007, .02, .02, .02, .02, .02, float(ratings.mean()))
    h = _lib.Handle(0, U, I, D, 0)
    s = _lib.stream_ptr(torch, dev)
    fit = lambda ep: _lib.check(h.L.daisy_svdpp_fit(
        h.ptr, c_vp(dpu.data_ptr()), c_vp(dqi.data_ptr()), c_vp(dyj.data_ptr()), c_vp(dbu.data_ptr()), c_vp(dbi.data_ptr()),
        c_vp(du.data_ptr()), c_vp(di.data_ptr()), c_vp(dr.data_ptr()), N, ep, c_vp(dptr.data_ptr()), c_vp(didx.data_ptr()),
        c_vp(dmult.data_ptr()) if dmult is not None else None, ctypes.byref(prm), None, s))
    fit(1)
    torch.cuda.synchronize()
    K = max(1, min(args.steps, 2))
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    fit(K)
    ev1.record()
    torch.cuda.synchronize()
    _lib.check(h.L.daisy_check(h.ptr, s))
    ms = ev0.elapsed_time(ev1)
    from oracle import mf_oracle
    n_cpu = 100_000
    t0 = time.time()
    mf_oracle.svdpp_fit(users[:n_cpu], items[:n_cpu], ratings[:n_cpu], pu, qi, yj, n_epochs=1, lists=(ptr, idx),
                        global_mean=float(ratings.mean()))
    cpu_dt = time.time() - t0
    rows = float(np.diff(ptr)[users].mean())                     # history rows gathered and rewritten per rating
    byts = N * K * (2 * rows * 8 * D + 4 * 8 * D + 12) / (ms * 1e-3) / 1e9
    line = {"metric": "svdpp_train_ratings_per_s", "value": N * K / (ms * 1e-3), "unit": "ratings/s", "n_gpus": 1, "steps": K,
            "warmup": 1, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"SVD++ (SVDpp.fit) on ml-1m-shaped synthetic ratings (config 2's set), n_factors {D}",
                       "status": "first version (one block walks the sequential loop)", "user_num": U, "item_num": I, "ratings": N, "dim": D,
                       "history_rows_per_rating": rows,
                       "step": "one epoch (a pass over the ratings in the given order, strictly sequential semantics)",
                       "l2": "tables are L2-resident; one thread block: the bound is one SM's L2 bandwidth and the barrier chain"},
            "roofline": {"bound": "hbm", "achieved": byts, "peak": measured_peaks()[0], "unit": "GB/s",
                         "frac": byts / measured_peaks()[0], "traffic": None,
                         "note": "2 x history rows x 8 D + 4 x 8 D + 12 B per rating; one SM, L2-resident: not an HBM-bound kernel"},
            "cpu_baseline": {"value": n_cpu / cpu_dt, "unit": "ratings/s", "cores": 1, "kind": "port",
                             "sample": f"C restatement of the Cython loop (bit-identical to the compiled reference class, "
                                       f"tests/test_oracle_golden.py), the first {n_cpu} ratings of the epoch with the full histories, single thread "
                                       "(the loop is serial); the reference's own fit adds DataFrame.iterrows and a Python "
                                       "list comprehension per rating"},
            "gpu_launches": int(h.launches)}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# device-side negative sampler (SURVEY 8f N1; secondary line)
# ------------------------------------------------------------------------------------------------
def run_sampler(args):
    """triples/s of daisy_sample_triples (rejection sampling + epoch shuffle, in device memory) on the ml-20m shape
    (config 3: 138 493 x 27 278, 20 M positives x num_ng 4 = 80 M triples per epoch), next to the reference's
    per-positive Python loop (ng_sample) on a bounded sample."""
    import torch
    from recommend_lib_b200.sampler import DeviceTripleSampler, zipf_items, _rng
    U, I, NP, NG = CFG3["user_num"], CFG3["item_num"], 20_000_263, 4
    g = _rng(2019, 77)
    pairs = np.stack([g.integers(0, U, NP), zipf_items(g, NP, I, 1.0, perm_seed=2019)], 1)
    pairs = np.unique(pairs, axis=0)
    smp = DeviceTripleSampler(pairs, I, U, num_ng=NG, seed=2019, device="cuda:0")
    n = len(smp)
    out = torch.empty((n, 3), dtype=torch.int32, device="cuda:0")
    K, W = max(1, min(args.steps, 10)), max(1, min(args.warmup, 3))
    for e in range(W):
        smp.sample_epoch(e, out=out)
    smp.check()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for e in range(W, W + K):
        smp.sample_epoch(e, out=out)
    ev1.record()
    torch.cuda.synchronize()
    smp.check()
    ms = ev0.elapsed_time(ev1) / K
    from oracle import sampler_oracle
    n_cpu = 50_000
    sub = pairs[:n_cpu]
    pos = set(map(tuple, pairs[pairs[:, 0] <= sub[:, 0].max()].tolist()))
    t0 = time.time()
    sampler_oracle.ng_sample_loop(sub, I, NG, positives=pos)
    cpu_dt = time.time() - t0
    line = {"metric": "bpr_negative_sampling_triples_per_s", "value": n / (ms * 1e-3), "unit": "triples/s", "n_gpus": 1,
            "steps": K, "warmup": W, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic",
            "config": {"workload": "negative sampling + epoch shuffle for config 3 (ml-20m shape)", "user_num": U,
                       "item_num": I, "positives": int(len(pairs)), "num_ng": NG, "triples_per_epoch": int(n),
                       "step": "one epoch of triples written to device memory, shuffled"},
            "roofline": {"bound": "hbm", "achieved": n * (12 * 3 + 16 * 4) / (ms * 1e-3) / 1e9, "peak": measured_peaks()[0],
                         "unit": "GB/s", "frac": n * (12 * 3 + 16 * 4) / (ms * 1e-3) / 1e9 / measured_peaks()[0],
                         "traffic": None,
                         "note": "per triple: write 12 + read 12 + write 12 B of triples, ~4 radix passes over 8 B "
                                 "(key, slot) pairs; the rejection test is a binary search in L2"},
            "cpu_baseline": {"value": n_cpu * NG / cpu_dt, "unit": "triples/s", "cores": 1, "kind": "port",
                             "sample": f"the reference's ng_sample loop (util/data_loader.py:680-690) restated, "
                                       f"{n_cpu} positives x {NG}, single thread as in the reference"},
            "gpu_launches": int(smp.h.launches)}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# full-catalogue top-K evaluation of config 4 (secondary line)
# ------------------------------------------------------------------------------------------------
def run_eval(args):
    """users/s of daisy_topk_full: top-100 of all 2 M items for a seeded sample of 16 384 users (SURVEY 8d, config 4's
    evaluation).  Default: candidates filtered on the tensor cores (k_filter_tc: tcgen05 BF16 MMA, TMEM accumulators, TMA
    operand tiles) with an error-bounded threshold, re-scored in exact fp32 and selected -- bit-identical to the fp32
    CUDA-core path (DAISY_TOPK_TC=0), which this line also times on a bounded sample of the users and compares."""
    import torch
    from recommend_lib_b200.bpr import BPR
    from recommend_lib_b200.metrics import topk_full
    U, I, D, N, K = 1_000_000, CFG4["item_num"], CFG4["dim"], args.eval_users, 100
    dev = torch.device("cuda:0")
    torch.manual_seed(2019)
    model = BPR(1, 1, D, max_batch=0)
    model.user_num, model.item_num = U, I
    model.embed_user.weight = torch.nn.Parameter(torch.empty((U, D), device=dev).normal_(0, 0.01), requires_grad=False)
    model.embed_item.weight = torch.nn.Parameter(torch.empty((I, D), device=dev).normal_(0, 0.01), requires_grad=False)
    users = torch.from_numpy(np.random.default_rng(2019).choice(U, N, replace=False).astype(np.int32)).to(dev)
    use_tc = os.environ.get("DAISY_TOPK_TC", "1") != "0"
    K_steps, W = max(1, min(args.steps, 5)), 3
    for _ in range(W):                                 # full size: the workspace pool grows to its final size here
        items, scores = topk_full(model, users, K)
    torch.cuda.synchronize()
    h = model.handle()
    h.set_timing(1)
    h.topk_tc_ms()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    watch = ClockSampler(0)
    watch.start()
    ev0.record()
    for _ in range(K_steps):
        items, scores = topk_full(model, users, K)
    ev1.record()
    torch.cuda.synchronize()
    model.check()
    watch.stop()
    clocks = watch.summary()
    ms = ev0.elapsed_time(ev1) / K_steps
    f_ms, r_ms, n_tc = h.topk_tc_ms()
    h.set_timing(0)
    flops = 2.0 * N * I * D
    # the CUDA-core filter on a bounded sample of the same users: same answer bit for bit, and its time beside it
    n_cmp = min(N, 2048)
    os.environ["DAISY_TOPK_TC"] = "0"
    topk_full(model, users[:256], K)
    torch.cuda.synchronize()
    ev0.record()
    it_s, sc_s = topk_full(model, users[:n_cmp], K)
    ev1.record()
    torch.cuda.synchronize()
    simt_ms = ev0.elapsed_time(ev1)
    os.environ["DAISY_TOPK_TC"] = "1" if use_tc else "0"
    same = bool(torch.equal(it_s, items[:n_cmp]) and torch.equal(sc_s, scores[:n_cmp]))
    assert same, "tensor-core filtered top-K differs from the CUDA-core path"
    # bounded CPU sample: exact fp32 scores + argpartition for a few users (what a vectorised CPU ranking costs)
    from oracle import bpr_oracle
    Pc = model._tables()[0][users[:8].long()].cpu().numpy()
    Qc = model._tables()[1].cpu().numpy()
    t0 = time.time()
    ref_items, _ = bpr_oracle.full_topk(Pc, Qc, np.arange(8), K)
    cpu_dt = time.time() - t0
    agree = float((items[:8].cpu().numpy() == ref_items).mean())
    peaks = measured_peaks()[2]
    if use_tc and n_tc:
        tc_peak = float(peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops") or 2250.0)
        ach = flops / (f_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": "k_filter_tc", "achieved": ach, "peak": tc_peak, "unit": "TFLOP/s",
                "frac": ach / tc_peak, "traffic": None, "kernel_ms": f_ms, "launches_timed": n_tc,
                "algorithmic_flops_per_launch": flops,
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (cuBLAS bf16, back to back)" if peaks else
                               "nominal dense bf16 2250 TFLOP/s (MEASURED_PEAKS.json absent)",
                "rescore_kernel_ms": r_ms, "whole_call_tflops": flops / (ms * 1e-3) / 1e12,
                "note": "BF16 tcgen05 filter with an error-bounded threshold (candidate superset), then exact fp32 "
                        "re-scoring + selection: results bit-identical to the fp32 CUDA-core path"}
    else:
        fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12
        roof = {"bound": "fp32-fma", "kernel": "k_score_tile", "achieved": flops / (ms * 1e-3) / 1e12, "peak": fp32_peak,
                "unit": "TFLOP/s", "frac": flops / (ms * 1e-3) / 1e12 / fp32_peak, "traffic": None,
                "note": "CUDA-core fp32 filter (DAISY_TOPK_TC=0); peak = 148 SMs x 128 FMA/clk x 1.965 GHz (nominal)"}
    line = {"metric": "bpr_full_catalogue_topk_users_per_s", "value": N / (ms * 1e-3), "unit": "users/s", "n_gpus": 1,
            "steps": K_steps, "warmup": W, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16 filter + f32 ranking" if use_tc else "f32", "data": "synthetic",
            "config": {"workload": "full-catalogue top-100 for 16 384 users of config 4 (2 M items, dim 128)", "users": N,
                       "item_num": I, "dim": D, "top_k": K, "step": "one evaluation of all sampled users",
                       "l2": "inputs larger than L2 (1 GB item table + 0.5 GB bf16 copy)"},
            "roofline": roof,
            "cuda_core_path": {"users": n_cmp, "ms": simt_ms, "users_per_s": n_cmp / (simt_ms * 1e-3),
                               "identical_items_and_scores": same},
            "cpu_baseline": {"value": 8 / cpu_dt, "unit": "users/s", "cores": os.cpu_count(), "kind": "port",
                             "sample": "numpy fp32 scores + exact top-100 for 8 users (oracle full_topk), agreement "
                                       f"with the device's items {agree:.3f}"},
            "gpu_launches": int(model.handle().launches)}
    if clocks:
        line["clocks"] = clocks
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scale", type=float, default=1.0, help="debug only: scale the table sizes")
    ap.add_argument("--batch", type=int, default=0, help="debug only: override the batch size")
    ap.add_argument("--materialize-every", type=int, default=0,
                    help="also fold the lazy L2 scale into the tables every N steps (0: only once, at the end of the "
                         "timed region -- what an epoch end does; the library itself only needs it when c < 1e-4)")
    ap.add_argument("--phases", action="store_true", help="also print the per-phase breakdown of the step")
    ap.add_argument("--no-phases", action="store_true", dest="no_phases",
                    help="N > 1: leave out the per-rank phase profile the fused peer path adds after the timed regions")
    ap.add_argument("--trace", action="store_true", help="also print a timeline of bookkeeping vs table kernels")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="config4", choices=["config4", "config3", "config2", "config1", "sampler", "eval", "gmf", "bprfm", "bprfm_bn", "sgns", "neumf", "svdpp"],
                    help="N = 1 only: config4 is the driver's metric; config3 (L2-resident ml-20m shape) and config2 "
                         "(funk-SVD) are secondary lines kept under profiles/")
    ap.add_argument("--eval-users", type=int, default=16384)
    ap.add_argument("--epoch-api", action="store_true",
                    help="config3/config4: run the K timed steps through ONE daisy_bpr_epoch call (BPRSGD.epoch)")
    ap.add_argument("--l2-window", action="store_true", help="pin the item table in L2 (access-policy window)")
    ap.add_argument("--l2-window-rows", type=int, default=0, help="rows of the item table the window covers (0 = all)")
    ap.add_argument("--hot-prefix", action="store_true",
                    help="experiment: item id = popularity rank (hot items are a prefix of the table)")
    ap.add_argument("--mapping", default="symm", choices=["symm", "ipc"],
                    help="N > 1, peer exchange: how the ranks map each other's arenas")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: peer = fused peer-memory step (product), nccl = all-to-all exchange (comparison)")
    ap.add_argument("--cpu-budget", type=float, default=25.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="config3/config4: after the timed steps, write the loss of the last timed call and a fixed "
                         "sample of the trained table rows as DIR/<name>.npy (float32 / float64, about 42 MB)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (args.impl != "b200" or args.gpus > 1 or world > 1
                              or args.workload not in ("config3", "config4")):
        ap.error("--dump-outputs: single-GPU config3 / config4 only")
    if args.impl == "reference":
        return run_reference(args)
    if args.gpus > 1 or world > 1:
        from bench_sharded import bench_sharded
        return bench_sharded(args, CFG5, METRIC, UNIT)
    if args.workload == "config1":
        return run_config1(args)
    if args.workload == "gmf":
        return run_gmf(args)
    if args.workload in ("bprfm_bn", "sgns", "neumf"):
        return run_experimental(args)
    if args.workload == "bprfm":
        return run_bprfm(args)
    if args.workload == "config2":
        return run_mf(args)
    if args.workload == "svdpp":
        return run_svdpp(args)
    if args.workload == "sampler":
        return run_sampler(args)
    if args.workload == "eval":
        return run_eval(args)
    return run_single(args)


if __name__ == "__main__":
    main()
