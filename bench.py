#!/usr/bin/env python
"""bench.py — SDF training points/sec (forward + backward) of the fused sm_100a step, with roofline,
CPU baseline and end-to-end (host buffers) numbers.  Contract: see the task statement / DESIGN.md §Measurement.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm (N>1: launched by torchrun)
    python bench.py --impl reference [--steps K] [--warmup W]      # the reference's CPU algorithm (oracle port)
    python bench.py ... --dump-outputs DIR                          # also save the last timed step's outputs (.npy)

Workload (BASELINE.json configs[1], "C2"): one synthetic MaiCity-like HDL-64 scan (64 x 2048 rays) of the
analytic street scene -> reference-style ray samples (3 surface + 3 free per hit) -> 4-level octree (leaf 0.2 m,
world level 12, F=8) + geo_decoder_8dim architecture (8->32->32->1, random init, trainable) + BCE loss.
One step = fwd+bwd over a whole-scan batch (N = number of samples of the scan, drawn with torch.randint like
LiDARDataset.get_batch).  N>1 GPUs: every rank owns its own spatial block (its own scan 100 m further along the
street, own table shard) and only the 1 377 decoder gradients are all-reduced (BASELINE configs[4] layout) — weak scaling.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the tree as build() left it (which may be read-only)

METRIC = "sdf_train_points_per_sec_fwd_bwd"
UNIT = "points/s"
L, F = 4, 8
BYTES_PER_POINT = 24 + L * 40 + 3 * L * 8 * F * 4   # SURVEY.md §8(d): 3 256 B at L=4, F=8
GATHER_BYTES_PER_POINT = L * 8 * F * 4               # SURVEY.md §8(d): the forward corner gather alone, 1 024 B
HBM_FALLBACK_GBS = 6650.0
C2_POINTS_PER_STEP = 776616   # samples of the C2 scan (64 x 2048 rays, seed 42): the per-GPU step size at every N
PROFILE_JSON = os.path.join(ROOT, "profiles", "r02_kernel_counters.json")   # ncu-derived per-point counters
DEC_KEYS = ["layers.0.weight", "layers.0.bias", "layers.1.weight", "layers.1.bias", "lout.weight", "lout.bias"]
DUMP_BYTES = 64_000_000


def workload_config(device):
    from shine_mapping_b200 import SHINEConfig
    return SHINEConfig(  # config/maicity/maicity_batch.yaml values, tree_level_feat 4 per BASELINE.json
        name="c2_maicity_like_single_scan", device=device, tree_level_world=12, tree_level_feat=L, leaf_vox_size=0.2,
        feature_dim=F, poly_int_on=True, surface_sample_range_m=0.15, surface_sample_n=3,
        free_sample_begin_ratio=0.3, free_sample_end_dist_m=0.8, free_sample_n=3, sigma_sigmoid_m=0.05,
        min_range=1.5, pc_radius=50.0, lr=0.01, weight_decay=1e-7, loss_weight_on=False, loss_reduction="mean",
        geo_mlp_level=2, geo_mlp_hidden_dim=32)


def build_workload(device, rank, world, n_azimuth):
    """N = 1: the C2 single-scan map."""
    from shine_mapping_b200 import Decoder, FeatureOctree, synth
    cfg = workload_config(device)
    torch.manual_seed(42)
    octree, decoder = FeatureOctree(cfg), Decoder(cfg)
    pool = synth.build_scene_map(cfg, octree, n_azimuth=n_azimuth, n_frames=1, seed=42, device=device)
    return cfg, octree, decoder, pool


SCAN_SPACING_M = 25.0    # multi-GPU map: one scan per GPU, 25 m apart along the street (pc_radius 50 m: they overlap)


def build_partitioned_workload(device, rank, world, n_azimuth, n_frames=None, exchange="auto"):
    """N > 1: ONE map of `world` overlapping scans, partitioned by Morton prefix at the coarsest featured level into
    `world` balanced ranges (partition.py).  Every rank generates the same global pool (seeded), keeps the samples of its
    range, grows its own octree from them; corner rows on the faces between ranges are duplicated and exchanged every
    step together with the decoder gradients.  -> cfg, octree, decoder, pool, boundary plan, NcclComm."""
    from shine_mapping_b200 import Decoder, FeatureOctree, dist as sdist, partition, synth
    import torch.distributed as dist
    cfg = workload_config(device)
    cfg.name = "c5_one_map_spatially_partitioned"
    torch.manual_seed(42)   # decoder init identical on every rank (it is replicated)
    octree, decoder = FeatureOctree(cfg), Decoder(cfg)
    n_frames = n_frames or world
    frames = synth.generate_scans(cfg, n_azimuth, n_frames, SCAN_SPACING_M, 42, device,
                                  origin_x0=-(n_frames - 1) * SCAN_SPACING_M / 2)
    coord = torch.cat([f[0] for f in frames]); label = torch.cat([f[1] for f in frames])
    weight = torch.cat([f[2] for f in frames])
    del frames
    level = cfg.tree_level_world - cfg.tree_level_feat + 1
    bounds = partition.balanced_key_bounds(partition.coarse_keys(coord, level).cpu(), world)
    box = [bounds]
    if world > 1:
        dist.broadcast_object_list(box, src=0)          # one agreed split even if RNG streams ever differed
    bounds, parts = partition.partition_pool(coord, label, weight, cfg, world, bounds=box[0])
    global_pool = int(coord.shape[0])
    del coord, label, weight
    pool = partition.build_rank_map(cfg, octree, parts[rank], device)
    del parts
    comm = sdist.NcclComm(rank, world, torch.device(device)) if world > 1 else None
    plan = partition.BoundaryPlan(rank, partition.gather_corner_keys(octree), cfg.feature_dim,
                                  partition.decoder_segment_floats(decoder)).to(device)
    if comm is not None:
        plan.unify_values(list(octree.hier_features), comm.all_reduce)
    p2p = None
    if world > 1 and exchange in ("p2p", "auto"):
        # peer-memory exchange when every rank can map every peer's buffer (CUDA IPC); all ranks take the same decision
        try:
            p2p = sdist.P2PExchange(rank, world, torch.device(device), plan.total_floats)
            ok = 1
        except Exception as exc:       # noqa: BLE001 — e.g. IPC not permitted in this container
            print(f"[bench] rank {rank}: peer-memory exchange unavailable ({exc}); using the NCCL path", file=sys.stderr)
            p2p, ok = None, 0
        if not ok and exchange == "p2p":       # P2PExchange agrees across ranks before raising: every rank lands here together
            raise SystemExit("--exchange p2p requested but CUDA IPC peer mapping failed")
    info = {"global_pool_samples": global_pool, "scans": n_frames, "scan_spacing_m": SCAN_SPACING_M,
            "boundary_rows": [int(c) for c in plan.counts], "exchange_floats": int(plan.total_floats),
            "exchange": "one NVLink peer-memory kernel (pack + publish + wait + reduce in place), IPC buffers" if p2p else
                        "shine_boundary_pack -> ncclAllReduce through the C ABI -> shine_boundary_unpack"}
    return cfg, octree, decoder, pool, plan, comm, p2p, info


BATCH_ORDER_NOTE = {
    "morton": "randint-drawn samples (with replacement, the reference's sampler) handed out in Morton order of their "
              "coordinates, free-space samples (no octree node on any level) behind the others (SamplePool.sort_morton + "
              "sorted indices); the loss of a batch does not depend on its order",
    "random": "randint-drawn samples in the order drawn (the reference's order)"}


def shared_config(cfg, n_azimuth, pool_len, n, world, rows, batch_order="morton", l2="rotate"):
    """The `config` object of the JSON line — identical for our arm and the reference arm (same workload, same N)."""
    return {"workload": cfg.name, "n_azimuth": n_azimuth, "pool_samples": pool_len, "points_per_step_per_gpu": n,
            "batch_order": batch_order, "batch_order_note": BATCH_ORDER_NOTE[batch_order],
            "l2_rule": "inputs larger than L2 (timed steps rotate over batches that together exceed it; GPU arm)" if l2 == "rotate"
                       else "L2 flushed before every timed step (GPU arm)",
            "global_points_per_step": n * world, "tree_level_feat": L, "feature_dim": F, "table_rows": rows,
            "decoder": "geo_decoder_8dim arch 8-32-32-1, trainable", "loss": "sdf_bce mean",
            "step": "grad zero + fwd + loss + bwd (table scatter-add + decoder grads); no optimizer"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (every 20 ms, timestamped; only the
    samples that fall inside [t0, t1] are reported)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def wait_first_sample(self, timeout=5.0):
        t0 = time.time()
        while self.p is not None and time.time() - t0 < timeout:
            if os.path.getsize(self.f.name) > 0:
                return
            time.sleep(0.02)

    def stop(self, t0, t1):
        import datetime
        if self.p is None:
            return None
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush(); self.f.seek(0)
        sm, mx, reasons, total = [], 0.0, set(), 0
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                clk, cmax = float(parts[1]), float(parts[2])
            except ValueError:
                continue
            total += 1
            if ts < t0 - 0.02 or ts > t1 + 0.02:
                continue
            sm.append(clk); mx = max(mx, cmax)
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "samples_total": total}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "window_s": round(t1 - t0, 3)}


def oracle_from_octree(octree, decoder):
    """CPU oracle (Python dict tables + torch CPU tensors) holding the same map as `octree`."""
    from oracle import shine_oracle as orc
    o = orc.OracleOctree(octree.max_level, octree.featured_level_num, octree.feature_dim, octree.feature_std,
                         octree.polynomial_interpolation)
    o.nodes_lookup_tables = octree.nodes_lookup_tables
    o.corners_lookup_tables = octree.corners_lookup_tables
    o.hier_features = [p.detach().cpu().clone().requires_grad_(True) for p in octree.hier_features]
    dec = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in decoder.state_dict().items()
           if not k.startswith("nclass_out")}
    return orc, o, dec


def pick_threads(orc, o, dec, batch, sigma):
    """The oracle's torch-CPU ops are small: too many threads hurt.  Try a few counts, keep the fastest."""
    best, best_t = None, None
    cands = sorted({min(c, os.cpu_count() or 1) for c in (8, 16, 32, os.cpu_count() or 1)})
    for c in cands:
        torch.set_num_threads(c)
        orc.train_step(o, dec, *batch, sigma, False, "mean")
        t0 = time.perf_counter()
        orc.train_step(o, dec, *batch, sigma, False, "mean")
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def time_oracle(orc, o, dec, batches, sigma, steps, warmup):
    ts = []
    for i in range(warmup + steps):
        c, l, w = batches[i % len(batches)]
        t0 = time.perf_counter()
        orc.train_step(o, dec, c, l, w, sigma, False, "mean")
        dt = time.perf_counter() - t0
        if i >= warmup:
            ts.append(dt)
    return ts


def run_reference(args):
    """The reference's own CPU algorithm for the path (oracle port: Python-dict Morton lookup + torch CPU
    gather/MLP/BCE/autograd, all host threads) on the SAME workload and the SAME points per step as our arm
    (one whole-scan batch per step; `--ref-sample` bounds it only if the run would not end within minutes)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    cfg, octree, decoder, pool = build_workload("cpu", 0, 1, args.n_azimuth)
    orc, o, dec = oracle_from_octree(octree, decoder)
    n = len(pool) if args.points <= 0 else args.points
    sample = n if args.ref_sample <= 0 else min(n, args.ref_sample)
    gen = torch.Generator().manual_seed(7)
    if args.batch_order == "morton":
        pool.sort_morton()
    batches = [pool.get_batch(sample, gen) for _ in range(2)]
    pick_threads(orc, o, dec, tuple(t[:20000] for t in batches[0]), cfg.sigma_sigmoid)
    ts = time_oracle(orc, o, dec, batches, cfg.sigma_sigmoid, args.steps, args.warmup)
    sec = statistics.mean(ts)
    value = sample / sec
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": shared_config(cfg, args.n_azimuth, len(pool), n, max(args.gpus, 1),
                                [int(p.shape[0]) for p in octree.hier_features], args.batch_order, args.l2),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                         "sample": f"{sample} randint-drawn samples of the {len(pool)}-sample C2 scan per step "
                                   f"(= the points_per_step_per_gpu of our arm)" if sample == n else
                                   f"{sample} of the {n} points of a step (bounded by --ref-sample)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def kernel_counters():
    """Per-point hardware counters of the step kernel taken from the committed ncu captures (profiles/): they turn the
    live kernel time into a physical roofline.  r01 values as fallback."""
    base = {"c2": {"lsu_wavefronts_per_point": 68.34, "dram_bytes_per_point": 36.87,
                   "source": "profiles/r01_step_full_v5_details.csv (raw page of gpurun r01_step_full_v5.ncu-rep)"},
            "hbm": {"dram_bytes_per_point": None, "source": None}}
    try:
        got = json.load(open(PROFILE_JSON))
        for k in base:
            base[k].update(got.get(k, {}))
    except Exception:
        pass
    return base


def e2e_record(n, n_global, pipe_sec, sync_sec, n_host, loss_last):
    """Both public host-step calls are timed on the same pinned host batches; the better one is the e2e figure (which
    one wins depends on the box: the copy engines' rate from host memory decides), the other is kept beside it."""
    modes = {"pipelined": {"value": n_global / pipe_sec, "ms_per_step": pipe_sec * 1e3,
                           "mode": "submit_host_step()/result(): step k+1's host->device copy under step k's kernels, depth 2"},
             "sync": {"value": n_global / sync_sec, "ms_per_step": sync_sec * 1e3,
                      "mode": "step_from_host(): chunked copy, step and loss read-back strictly inside one call"}}
    best = "pipelined" if pipe_sec <= sync_sec else "sync"
    other = "sync" if best == "pipelined" else "pipelined"
    rec = {"value": modes[best]["value"], "unit": UNIT, "h2d_bytes_per_step": n * 16, "d2h_bytes_per_step": 4,
           "ms_per_step": modes[best]["ms_per_step"], "mode": modes[best]["mode"], "host_batches": n_host,
           "h2d_gbps": n * 16 / (modes[best]["ms_per_step"] * 1e-3) / 1e9, "loss_last": loss_last}
    rec[other] = modes[other]
    return rec


L2_BYTES = 126 << 20


def batches_exceeding_l2(n_points, cap=64):
    """How many distinct device batches (16 B per point) it takes to exceed the L2 by 1.6x; None if more than `cap`."""
    need = -(-int(1.6 * L2_BYTES) // max(1, n_points * 16))
    return max(4, need) if need <= cap else None


def time_graph_steps(graphs, steps, flush_buf, dev):
    """K replays of the captured whole-step graphs (rotating), CUDA events around every replay -> mean ms per step."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for k in range(steps):
        if flush_buf is not None:
            flush_buf.fill_(k & 0xFF)
        ev[k][0].record()
        graphs[k % len(graphs)].replay()
        ev[k][1].record()
    torch.cuda.synchronize(dev)
    if flush_buf is None:          # back-to-back replays: first start -> last end, so that nothing between steps is left out
        return ev[0][0].elapsed_time(ev[-1][1]) / steps
    return statistics.mean(a.elapsed_time(b) for a, b in ev)


def time_steps(trainer, batches, steps, flush_buf, n_norm, dev, all_reduce=True):
    """K steps; flush_buf given: the L2 is flushed before each (untimed 256 MiB write), None: the batches rotate and are
    together larger than L2.  -> per-step (zero+kernel+reduce+allreduce), fused kernel alone, replica
    reduce alone, in ms (means).  CUDA events on the launching stream."""
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(steps)]
    for k in range(steps):
        if flush_buf is not None:
            flush_buf.fill_(k & 0xFF)                 # > L2 (126 MB): evicts tables, inputs and gradients
        b = batches[k % len(batches)]
        ev[k][0].record()
        trainer.zero_grad()
        ev[k][1].record()
        trainer.forward_backward(b[0], b[1], None, n_norm=n_norm, mid_event=ev[k][2])
        ev[k][3].record()
        if all_reduce:
            trainer.all_reduce_grads()
        ev[k][4].record()
    torch.cuda.synchronize(dev)
    mean = statistics.mean
    time_steps.last_exchange_ms = mean(e[3].elapsed_time(e[4]) for e in ev)      # exchange + waiting for the slowest rank
    return (mean(e[0].elapsed_time(e[4]) for e in ev), mean(e[1].elapsed_time(e[2]) for e in ev),
            mean(e[2].elapsed_time(e[3]) for e in ev))


def parity_block(orc, o, dec, trainer, octree, decoder, batch, sample, sigma):
    """CUDA step (the trainer of the timed steps: same kernel flavour) vs the oracle on `sample` points of a bench batch."""
    import numpy as np
    c, l = batch[0][:sample].contiguous(), batch[1][:sample].contiguous()
    res = orc.train_step(o, dec, c.cpu(), l.cpu(), None, sigma, False, "mean")
    trainer.zero_grad()
    pred = torch.empty(sample, device=c.device)
    loss = float(trainer.forward_backward(c, l, None, pred_out=pred))
    idx = octree.get_indices(c)
    idx_exact = all(bool(torch.equal(a.cpu(), b)) for a, b in zip(idx, o.hierarchical_indices))

    def rel(a, b):
        b = b.double()
        return float((a.detach().cpu().double() - b).abs().max() / b.abs().max().clamp_min(1e-30))
    got_dec = dict(zip(DEC_KEYS, trainer.dec_grads))    # views of THIS trainer's flat gradient buffer
    tg = max(rel(g[:-1], w[:-1]) for g, w in zip(trainer.table_grads, res["table_grads"]))
    dg = max(rel(got_dec[k], w) for k, w in res["dec_grads"].items())
    trainer.zero_grad()
    return {"n_points": sample, "idx_exact": idx_exact,
            "loss_rel": abs(loss - float(res["loss"])) / abs(float(res["loss"])),
            "pred_max_abs": float((pred.cpu() - res["pred"]).abs().max()),
            "table_grad_rel": tg, "dec_grad_rel": dg,
            "tolerance": {"idx": "exact", "loss_rel": 2e-5, "grad_rel": 2e-4},
            "ok": bool(idx_exact and tg <= 2e-4 and dg <= 2e-4)}


def hbm_leg(args, dev, peak):
    """The same step kernel on a map far larger than L2 (C3-like: many frames, leaf 0.05 m): the regime where the
    HBM roofline is physical.  Algorithmic bytes / measured kernel time against the measured copy bandwidth, plus the
    gather-only figure (1 024 B/pt over the forward kernel) for north_star's 60 % clause."""
    import ctypes as C
    from shine_mapping_b200 import Decoder, FeatureOctree, SdfTrainer, _abi, synth
    cfg = workload_config(str(dev))
    cfg.name = "c3_like_large_map"
    cfg.leaf_vox_size = 0.05
    cfg.calculate_world_scale()
    torch.manual_seed(42)
    octree, decoder = FeatureOctree(cfg), Decoder(cfg)
    t0 = time.time()
    # the world cube of a 0.05 m leaf at tree_level_world 12 is +-102.4 m: drive through all of it, centred
    step_m = 190.0 / max(1, args.hbm_frames - 1)
    pool = synth.build_scene_map(cfg, octree, n_azimuth=args.n_azimuth, n_frames=args.hbm_frames, frame_step_m=step_m,
                                 seed=42, device=str(dev), origin_x0=-95.0)
    torch.cuda.synchronize(dev)
    build_s = time.time() - t0
    rows = [int(p.shape[0]) for p in octree.hier_features]
    table_mb = sum(rows) * F * 4 / 1e6
    n = args.hbm_points
    trainer = SdfTrainer(cfg, octree, decoder)
    gen = torch.Generator(device=dev).manual_seed(3)
    batches = [pool.get_batch(n, gen) for _ in range(4)]
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for i in range(3):
        trainer.zero_grad(); trainer.forward_backward(batches[i][0], batches[i][1], None)
    torch.cuda.synchronize(dev)
    steps = args.steps
    step_ms, kern_ms, red_ms = time_steps(trainer, batches, steps, flush_buf, n, dev, all_reduce=False)
    # forward kernel (hash walk + gather + blend + MLP + loss): the gather figure
    od = octree._descriptor(None, None)
    dd = decoder.c_descriptor(None)
    pred = torch.empty(n, device=dev); loss = torch.zeros((), device=dev)
    lib, st = _abi.lib(), _abi.stream_ptr(dev)

    def fwd(b):
        _abi.check(lib.shine_sdf_bce_fwd(C.byref(od), C.byref(dd), _abi.ptr(b[0]), _abi.ptr(b[1]), None, n,
                                         float(cfg.sigma_sigmoid), 1.0 / n, _abi.ptr(pred), _abi.ptr(loss), 0, st),
                   "shine_sdf_bce_fwd")
    feat = torch.empty(n, F, device=dev)

    def gather(b):
        _abi.check(lib.shine_query_fwd(C.byref(od), _abi.ptr(b[0]), n, _abi.ptr(feat), st), "shine_query_fwd")
    out = {}
    for name, fn in (("fwd", fwd), ("gather", gather)):
        for i in range(3):
            fn(batches[i])
        ts = []
        for k in range(steps):
            flush_buf.fill_(k & 0xFF)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(batches[k % 4]); e1.record(); torch.cuda.synchronize(dev)
            ts.append(e0.elapsed_time(e1))
        out[name] = statistics.mean(ts)
    idx = octree.get_indices(batches[0][0][:200000])
    hit_frac = float(sum((t[:, 0] >= 0).float().mean() for t in idx) / len(idx))   # share of (point, level) pairs that hit
    octree.clear_temp()
    cnt = kernel_counters()["hbm"]
    achieved = n * BYTES_PER_POINT / (kern_ms * 1e-3) / 1e9
    g_fwd = n * GATHER_BYTES_PER_POINT / (out["fwd"] * 1e-3) / 1e9
    g_only = n * GATHER_BYTES_PER_POINT / (out["gather"] * 1e-3) / 1e9
    del flush_buf
    return {
        "bound": "hbm", "kernel": "sdf_fused_kernel<3,train,dec_grad,4>", "workload": cfg.name,
        "batch_order": "random (the order drawn: the access pattern that makes this leg HBM-bound)",
        "frames": args.hbm_frames, "table_rows": rows, "table_mb": table_mb, "grad_mb": table_mb,
        "points_per_step": n, "build_s": round(build_s, 1),
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "kernel_ms": kern_ms, "replica_reduce_ms": red_ms, "step_ms": step_ms,
        "points_per_s": n / (step_ms * 1e-3),
        "algorithmic_bytes_per_point": BYTES_PER_POINT, "hit_fraction": hit_frac,
        "note": "algorithmic bytes follow SURVEY 8(d) (every point charged 8 corners on all L levels); free-space samples "
                "that miss a level fetch nothing there (hit_fraction), so the fraction can touch 1",
        "traffic": (cnt["dram_bytes_per_point"] * n) if cnt.get("dram_bytes_per_point") else None,
        "traffic_source": cnt.get("source"),
        "gather": {"bytes_per_point": GATHER_BYTES_PER_POINT,
                   "forward_kernel_ms": out["fwd"], "forward_kernel_gbps": g_fwd, "forward_kernel_frac": g_fwd / peak,
                   "gather_only_kernel_ms": out["gather"], "gather_only_gbps": g_only, "gather_only_frac": g_only / peak,
                   "note": "north_star clause: >= 0.60 of the HBM roofline for the feature gather"},
        "l2": "flushed between timed launches (256 MiB write, not timed); tables + gradients are > 2x the 126 MB L2",
    }


def small_batch_records(cfg, octree, decoder, pool, dev, sizes=(4096, 8192), iters=200):
    """The reference's own batch sizes (config/*/*.yaml batch_size): one loop iteration {get_batch -> fused step ->
    Adam(+zero grads)} replayed as a CUDA graph (batch_loop._GraphedIteration)."""
    from shine_mapping_b200 import SdfTrainer
    from shine_mapping_b200.batch_loop import _GraphedIteration
    out = []
    state = [p.detach().clone() for p in list(octree.parameters()) + list(decoder.parameters())]
    for bs in sizes:
        tr = SdfTrainer(cfg, octree, decoder)
        tr.zero_grad()
        it = _GraphedIteration(tr, pool, bs)
        for _ in range(5):
            it.run()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            it.run()
        e1.record(); torch.cuda.synchronize(dev)
        us = e0.elapsed_time(e1) * 1e3 / iters
        out.append({"bs": bs, "us_per_iter": us, "iters_per_s": 1e6 / us, "points_per_s": bs * 1e6 / us,
                    "iteration": "get_batch (randint gather) + fused fwd/loss/bwd + dense Adam with grad re-zero, CUDA graph"})
    with torch.no_grad():      # the timing loop trained the model: put the weights back
        for p, q in zip(list(octree.parameters()) + list(decoder.parameters()), state):
            p.copy_(q)
    return out


def other_config_records(dev):
    """Short records for the BASELINE.json configs that are not the headline workload (their parity is covered by tests):
    C1 = 10 k ray-sampled points, 2-level octree (the reference's CPU-runnable case): GPU step next to the oracle's CPU step;
    C4 = incremental mapping with the regularisation terms (per-touched-row kernels): time per frame of the loop."""
    from shine_mapping_b200 import Decoder, FeatureOctree, SHINEConfig, SdfTrainer, synth
    from shine_mapping_b200.incre_loop import run_shine_mapping_incremental
    out = {}
    # ---- C1 ----
    cfg = workload_config(str(dev)); cfg.name = "c1_10k_points_2_levels"; cfg.tree_level_feat = 2
    torch.manual_seed(42)
    octree, decoder = FeatureOctree(cfg), Decoder(cfg)
    pool = synth.build_scene_map(cfg, octree, n_azimuth=256, n_frames=1, seed=42, device=str(dev))
    gen = torch.Generator(device=dev).manual_seed(1)
    coord, label, _ = pool.get_batch(10000, gen)
    tr = SdfTrainer(cfg, octree, decoder)
    for _ in range(5):
        tr.zero_grad(); tr.forward_backward(coord, label, None)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(50):
        tr.zero_grad(); tr.forward_backward(coord, label, None)
    e1.record(); torch.cuda.synchronize(dev)
    gpu_ms = e0.elapsed_time(e1) / 50
    orc, o, dec = oracle_from_octree(octree, decoder)
    torch.set_num_threads(os.cpu_count() or 1)
    cb = (coord.cpu(), label.cpu(), None)
    orc.train_step(o, dec, *cb, cfg.sigma_sigmoid, False, "mean")
    t0 = time.perf_counter(); res = orc.train_step(o, dec, *cb, cfg.sigma_sigmoid, False, "mean"); cpu_s = time.perf_counter() - t0
    out["c1"] = {"workload": cfg.name, "points": 10000, "table_rows": [int(p.shape[0]) for p in octree.hier_features],
                 "gpu_ms_per_step": gpu_ms, "gpu_points_per_s": 10000 / (gpu_ms * 1e-3),
                 "cpu_ms_per_step": cpu_s * 1e3, "cpu_points_per_s": 10000 / cpu_s,
                 "loss_rel_vs_oracle": abs(float(tr.loss) - float(res["loss"])) / abs(float(res["loss"]))}
    # ---- C4 ----
    cfg4 = workload_config(str(dev)); cfg4.name = "c4_incremental_with_regularisation"
    cfg4.bs, cfg4.iters, cfg4.continual_learning_reg, cfg4.lambda_forget, cfg4.loss_reduction = 4096, 50, True, 1e4, "sum"
    torch.manual_seed(42)
    octree4, decoder4 = FeatureOctree(cfg4), Decoder(cfg4)
    frames = [f[:3] for f in synth.generate_scans(cfg4, 1024, 6, 2.0, 42, str(dev))]
    run_shine_mapping_incremental(cfg4, octree4, decoder4, frames[:1])            # warm-up frame (kernel attributes, allocator)
    torch.cuda.synchronize(dev); t0 = time.perf_counter()
    hist = run_shine_mapping_incremental(cfg4, octree4, decoder4, frames[1:])
    torch.cuda.synchronize(dev); dt = time.perf_counter() - t0
    out["c4"] = {"workload": cfg4.name, "frames": len(frames) - 1, "iters_per_frame": cfg4.iters, "bs": cfg4.bs,
                 "samples_per_frame": int(frames[1][0].shape[0]),
                 "s_per_frame": dt / (len(frames) - 1), "frame_content": "octree.update (GPU build kernels) + 50 x {get_batch, fused "
                 "step, touched-row regulariser, Adam} + feature-importance sweep over the frame's pool",
                 "rows_last": hist[-1]["rows"], "bce_first_last": [hist[-1]["bce_first"], hist[-1]["bce_last"]]}
    return out


def step_outputs(trainer):
    """What a training step hands its caller, copied to the host: the loss and the gradient of every table level and
    decoder tensor (this rank's tables when the map is partitioned)."""
    out = {"loss": trainer.loss}
    out.update({f"table_grad_{k}": g for k, g in enumerate(trainer.table_grads)})
    out.update({"decoder_grad_" + k.replace(".", "_"): g for k, g in zip(DEC_KEYS, trainer.dec_grads) if g is not None})
    return {k: v.detach().float().cpu().numpy() for k, v in out.items()}


def dump_outputs(directory, arrays, budget=DUMP_BYTES):
    """DIR/<name>.npy for every array.  Beyond `budget` bytes in all, every array keeps the same fraction of its rows,
    a seeded sample that depends only on the shapes: runs with the same arguments stay comparable row for row."""
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    frac = min(1.0, (budget - 4096 * len(arrays)) / max(total, 1))     # room for the .npy headers
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        if frac < 1.0 and a.ndim > 0:
            k = max(1, int(a.shape[0] * frac))
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], k, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)


def run_ours(args):
    from shine_mapping_b200 import SdfTrainer, _abi, dist as sdist
    rank, world, local = sdist.init_from_env("nccl")
    if world != args.gpus:
        if rank == 0:
            print(f"[bench] note: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE", file=sys.stderr)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (our arm) needs a CUDA device: the hot path has no CPU fallback")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    numa = sdist.pin_to_gpu_numa_node(local) if world > 1 else {"numa_node": sdist.gpu_numa_node(local), "cpus": None}
    part_info, p2p = None, None
    ordered = args.batch_order == "morton"
    if world > 1:
        cfg, octree, decoder, pool, plan, comm, p2p, part_info = build_partitioned_workload(
            str(dev), rank, world, args.n_azimuth, exchange=args.exchange)
        # weak scaling: every GPU steps as many points as the single GPU does (one scan's worth), drawn from ITS range
        n = (args.points if args.points > 0 else C2_POINTS_PER_STEP) if args.global_points <= 0 else args.global_points // world
        trainer = SdfTrainer(cfg, octree, decoder, shard_mode="spatial", boundary=plan, comm=comm, p2p=p2p,
                             morton_ordered=ordered)
    else:
        cfg, octree, decoder, pool = build_workload(str(dev), rank, world, args.n_azimuth)
        n = len(pool) if args.points <= 0 else args.points
        trainer = SdfTrainer(cfg, octree, decoder, shard_mode="spatial", morton_ordered=ordered)
    if ordered:
        pool.sort_morton(octree=octree)      # once, with the map: Morton order, free-space samples (no node on any level) last
    n_global = n * world
    gen = torch.Generator(device=dev).manual_seed(1000 + rank)
    # L2 rule: inputs larger than L2 (default) -- the timed steps rotate over batches that together exceed the 126 MB L2 by
    # 1.6x, so every step streams its inputs from HBM while the persistent state (tables, gradients, exchange plan) stays
    # resident exactly as it does in a training run; `--l2 flush` evicts everything before every step instead.
    n_rot = batches_exceeding_l2(n) if args.l2 == "rotate" else None
    rotate = n_rot is not None
    batches = [pool.get_batch(n, gen) for _ in range(n_rot if rotate else 4)]
    nb = len(batches)
    flush_all = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    flush_buf = None if rotate else flush_all
    l2_note = (f"inputs larger than L2: the timed steps rotate over {nb} batches = {nb * n * 16 / 2**20:.0f} MiB (L2 126 MiB); "
               "tables and gradients stay resident as in training" if rotate else
               "flushed between timed steps (256 MiB write, not timed)")

    def step(b):
        trainer.zero_grad()
        trainer.forward_backward(b[0], b[1], None, n_norm=n_global)
        trainer.all_reduce_grads()

    warm = max(args.warmup, 3)
    for i in range(max(warm, nb if rotate else 0)):
        step(batches[i % nb])
    torch.cuda.synchronize(dev)
    graphs = None
    if not args.eager and (world == 1 or p2p is not None):     # the NCCL route of the exchange is launched eagerly
        graphs = [trainer.capture_step(b[0], b[1], None, n_norm=n_global, exchange=world > 1) for b in batches]
        for g_ in graphs[:2]:
            g_.replay()
        torch.cuda.synchronize(dev)

    # ---- `value`: inputs resident in HBM, CUDA events on the launching stream, L2 flushed between steps ----
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.wait_first_sample()
    sdist.barrier(dev); torch.cuda.synchronize(dev)     # after the sampler start-up so that no rank enters late
    launches0 = _abi.LAUNCHES["count"]
    t_clk0 = time.time()
    if args.cuda_profiler:
        torch.cuda.profiler.start()                   # ncu --profile-from-start off: only the timed steps
    # the timed steps: every rotating batch's whole step {grad memset, fused kernel, exchange} captured once as a CUDA graph
    # (SdfTrainer.capture_step) and replayed -- the host only enqueues graph launches; an eager pass with events between
    # the phases follows for the kernel / exchange breakdown
    host_t0 = time.perf_counter()
    outputs = None
    if graphs is not None:
        step_ms = time_graph_steps(graphs, args.steps, flush_buf, dev)
        launches = _abi.LAUNCHES["count"] - launches0
        if args.dump_outputs and rank == 0:
            outputs = step_outputs(trainer)
        sdist.barrier(dev)
        eager_ms, kern_ms, red_ms = time_steps(trainer, batches, args.steps, flush_buf, n_global, dev)
    else:
        step_ms, kern_ms, red_ms = time_steps(trainer, batches, args.steps, flush_buf, n_global, dev)
        eager_ms = step_ms
        launches = _abi.LAUNCHES["count"] - launches0
        if args.dump_outputs and rank == 0:
            outputs = step_outputs(trainer)
    sdist.barrier(dev)
    if args.cuda_profiler:
        torch.cuda.profiler.stop()
    step_ms = sdist.max_over_ranks(step_ms, dev)
    eager_ms = sdist.max_over_ranks(eager_ms, dev)
    kern_ms_max = sdist.max_over_ranks(kern_ms, dev)
    red_ms_max = sdist.max_over_ranks(red_ms, dev)
    exch_ms = getattr(time_steps, "last_exchange_ms", 0.0)
    other_order = None
    if world == 1 and ordered:      # the same step on batches in the order drawn (general kernel), for the record
        tr_r = SdfTrainer(cfg, octree, decoder, shard_mode="spatial", morton_ordered=False)
        br = [pool.get_batch(n, gen, ordered=False) for _ in range(nb if rotate else 2)]
        for i in range(3):
            tr_r.zero_grad(); tr_r.forward_backward(br[i % 2][0], br[i % 2][1], None, n_norm=n_global)
        r_step, r_kern, _ = time_steps(tr_r, br, args.steps, flush_buf, n_global, dev)
        other_order = {"batch_order": "random", "value": n_global / (r_step * 1e-3), "ms_per_step": r_step,
                       "kernel_ms": r_kern, "kernel": "sdf_fused_kernel<3,train,dec_grad,4> (per-point reds)",
                       "note": BATCH_ORDER_NOTE["random"]}
        del tr_r, br
    flushed = None
    if world == 1 and rotate:       # the conservative variant, for the record: everything evicted before every step
        _, f_kern, _ = time_steps(trainer, batches, args.steps, flush_all, n_global, dev)
        f_step = time_graph_steps(graphs, args.steps, flush_all, dev) if graphs is not None else _
        flushed = {"value": n_global / (f_step * 1e-3), "ms_per_step": f_step, "kernel_ms": f_kern,
                   "l2": "flushed between timed steps (256 MiB write, not timed): tables and gradients come from HBM too"}
    exch_ms_max = sdist.max_over_ranks(exch_ms, dev)
    exch_ms_min = -sdist.max_over_ranks(-exch_ms, dev)
    kern_ms_min = -sdist.max_over_ranks(-kern_ms, dev)
    # nvidia-smi cannot sample faster than ~20 ms: keep the SAME steps running (not counted) so that the sampled
    # window under load is ~0.5 s.  The count is derived from the rank-agreed step time: every rank issues the same
    # number of collectives.
    n_cont = max(0, min(20000, int(500.0 / max(step_ms, 0.02)) - args.steps))
    for k in range(n_cont):
        if graphs is not None:
            graphs[k % nb].replay()
        else:
            step(batches[k % nb])
        if k % 64 == 63:
            torch.cuda.synchronize(dev)
    torch.cuda.synchronize(dev)
    clocks = sampler.stop(t_clk0, time.time()) if sampler else None
    value = n_global / (step_ms * 1e-3)

    # ---- `e2e`: pinned HOST buffers through the public host-step API; every step copies its inputs host->device
    #      and reads its loss back.  Pipelined: step k+1's copy overlaps step k's kernels (submit/result); the inputs
    #      rotate over host batches that together exceed L2.  The synchronous call is reported next to it. ----
    n_host = max(4, min(16, (160 << 20) // max(1, n * 16) + 1))
    host = []
    for i in range(n_host):
        b = pool.get_batch(n, gen)
        host.append(tuple(t.cpu().pin_memory() for t in b[:2]))
    for i in range(max(4, warm)):
        trainer.submit_host_step(*host[i % n_host], n_norm=n_global, exchange=world > 1).result()
    sdist.barrier(dev); torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    pending, losses = None, []
    for k in range(args.steps):
        h = trainer.submit_host_step(*host[k % n_host], n_norm=n_global, exchange=world > 1)
        if pending is not None:
            losses.append(pending.result())
        pending = h
    losses.append(pending.result())
    torch.cuda.synchronize(dev)
    e2e_sec = sdist.max_over_ranks((time.perf_counter() - t0) / args.steps, dev)
    e2e_value = n_global / e2e_sec
    for i in range(n_host):       # synchronous variant: every pinned host batch once -> its CUDA graph is captured untimed
        trainer.step_from_host(*host[i])
    sync_ts = []
    sdist.barrier(dev); torch.cuda.synchronize(dev)
    for k in range(args.steps):
        if flush_buf is not None:
            flush_buf.fill_(k & 0xFF)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        trainer.step_from_host(*host[k % n_host])     # ends with loss.item(): device -> host read
        if world > 1:
            trainer.all_reduce_grads(); torch.cuda.synchronize(dev)
        sync_ts.append(time.perf_counter() - t0)
    e2e_sync_sec = sdist.max_over_ranks(statistics.mean(sync_ts), dev)

    if rank != 0:
        return
    del flush_buf, flush_all
    peak, peak_src = peaks()
    cnt = kernel_counters()
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    wf = cnt["c2"]["lsu_wavefronts_per_point"]
    wf_rate = wf * n / (kern_ms_max * 1e-3) / 1e9                       # G wavefronts / s
    wf_peak = n_sm * sm_mhz * 1e6 / 1e9                                  # 1 wavefront / clk / SM
    alg = n * BYTES_PER_POINT / (kern_ms_max * 1e-3) / 1e9
    rows = [int(p.shape[0]) for p in octree.hier_features]
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": shared_config(cfg, args.n_azimuth, len(pool), n, world, rows, args.batch_order,
                                args.l2 if rotate else "flush"),
        "impl_notes": {"decoder_math": "3xTF32 mma.sync (fp32-grade)",
                       "other_batch_order": other_order,
                       "parallelism": "single GPU" if world == 1 else
                       f"one map, Morton-prefix ranges x{world}; ONE exchange per step over [decoder grads | "
                       "gradients of corner rows shared between ranges] (see partition.exchange)",
                       "partition": part_info,
                       "exchange_ms": {"max_over_ranks": exch_ms_max, "min_over_ranks": exch_ms_min,
                                       "note": "events around the exchange: its latency + the wait for the slowest rank's kernel"},
                       "kernel_ms_min_over_ranks": kern_ms_min,
                       "l2": l2_note, "l2_flushed": flushed,
                       "timed_step": "grad memset + fused fwd+loss+bwd kernel (+ replica fold for unordered batches) (+ exchange when N>1)"
                                     + ("; captured per rotating batch as a CUDA graph (SdfTrainer.capture_step) and replayed" if graphs is not None else "; launched eagerly"),
                       "eager_ms_per_step": eager_ms},
        # the C2 map (2.75 MB of features) lives in L2: the kernel's physical bound there is the L1TEX LSU data pipe
        # (1 wavefront / clk / SM), not HBM.  wavefronts/point come from the committed ncu capture, time is live.
        "roofline": {"bound": "l1tex_lsu",
                     "kernel": "sdf_fused_kernel<3,train,dec_grad,4" + (",grouped>" if ordered else ">"),
                     "achieved": wf_rate, "peak": wf_peak, "unit": "Gwavefront/s", "frac": wf_rate / wf_peak,
                     "traffic": cnt["c2"]["dram_bytes_per_point"] * n, "kernel_ms": kern_ms_max,
                     "replica_reduce_ms": red_ms_max,
                     "lsu_wavefronts_per_point": wf, "counter_source": cnt["c2"]["source"],
                     "peak_source": f"{n_sm} SMs x {sm_mhz:.0f} MHz x 1 wavefront/clk",
                     "algorithmic_bytes_per_point": BYTES_PER_POINT, "algorithmic_gbps": alg,
                     "algorithmic_over_hbm_peak": alg / peak,
                     "note": "algorithmic bytes / time exceeds the HBM peak because >98 % of them are served by L2 "
                             "(measured DRAM traffic in `traffic`); the HBM roofline proper is `roofline_hbm`"},
        "e2e": e2e_record(n, n_global, e2e_sec, e2e_sync_sec, n_host, losses[-1]),
        "gpu_launches": launches,
        "clocks": clocks,
        "host": {"numa": numa, "cpu_count": os.cpu_count(), "affinity": len(os.sched_getaffinity(0))},
    }
    if world == 1 and not args.no_hbm_leg:
        free_state = (trainer, batches, host)
        del free_state
        line["roofline_hbm"] = hbm_leg(args, dev, peak)
        line["roofline_hbm"]["peak_source"] = peak_src
    if world == 1 and not args.no_cpu_baseline:
        was_ordered, pool.ordered = pool.ordered, False      # the reference's batch sizes in the reference's order
        line["small_batch"] = small_batch_records(cfg, octree, decoder, pool, dev)
        pool.ordered = was_ordered
        torch.set_num_threads(os.cpu_count() or 1)
        orc, o, dec = oracle_from_octree(octree, decoder)
        sample = min(n, args.ref_sample if args.ref_sample > 0 else 100000)
        stride = max(1, n // sample)      # every stride-th point: a subsequence of a Morton-ordered batch is Morton-ordered
        sub = [tuple(t[::stride][:sample].contiguous() for t in b) for b in batches[:2]]
        cb = [tuple(t.cpu() for t in b) for b in sub]
        pick_threads(orc, o, dec, tuple(t[:20000] for t in cb[0]), cfg.sigma_sigmoid)
        ts = time_oracle(orc, o, dec, cb, cfg.sigma_sigmoid, 3, 1)
        line["cpu_baseline"] = {"value": sample / statistics.mean(ts), "unit": UNIT, "cores": torch.get_num_threads(),
                                "kind": "port", "sample": f"every {stride}-th point ({sample}) of the step's batch, 1 warm-up + 3 "
                                                           "timed oracle steps (Python-dict lookup + torch CPU autograd)"}
        line["parity"] = parity_block(orc, o, dec, trainer, octree, decoder, sub[0], sample, cfg.sigma_sigmoid)
        line["configs"] = other_config_records(dev)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n-azimuth", type=int, default=2048, help="rays per ring of the synthetic scan (C2: 2048)")
    ap.add_argument("--points", type=int, default=0, help="points per step per GPU (default: the whole scan)")
    ap.add_argument("--global-points", type=int, default=0,
                    help="N>1 only: GLOBAL points per step, split over the ranks (BASELINE configs[4]: 1048576)")
    ap.add_argument("--ref-sample", type=int, default=0,
                    help="points per oracle step: reference arm default 0 = the whole step (same config as ours); "
                         "cpu_baseline / parity legs of our arm default to 100000")
    ap.add_argument("--hbm-frames", type=int, default=100, help="frames of the HBM-bound leg's map")
    ap.add_argument("--hbm-points", type=int, default=1 << 20, help="points per step of the HBM-bound leg")
    ap.add_argument("--exchange", default=os.environ.get("SHINE_EXCHANGE", "auto"), choices=["auto", "nccl", "p2p"],
                    help="N>1: the step's exchange — NCCL all-reduce through the C ABI, or the one-kernel NVLink peer-memory path")
    ap.add_argument("--batch-order", default="morton", choices=["morton", "random"],
                    help="order the sampler hands a batch out in (same random index multiset either way)")
    ap.add_argument("--l2", default="rotate", choices=["rotate", "flush"],
                    help="L2 rule of the timed steps: rotate over batches that together exceed L2 (default) or flush before every step")
    ap.add_argument("--eager", action="store_true", help="launch the timed steps eagerly instead of replaying captured graphs")
    ap.add_argument("--no-hbm-leg", action="store_true")
    ap.add_argument("--hbm-only", action="store_true", help="run only the HBM-bound leg and print its object (ncu target)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cuda-profiler", action="store_true", help="cudaProfilerStart/Stop around the timed steps")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last timed step's loss and gradients as DIR/<name>.npy "
                         "(float32; a seeded sample of rows beyond 64 MB in all)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        from shine_mapping_b200 import _abi
        _abi.lib()      # the kernels build() compiled: the benchmark compiles nothing and writes nothing into the tree
        if args.hbm_only:
            dev = torch.device("cuda", 0)
            torch.cuda.set_device(dev)
            print(json.dumps(hbm_leg(args, dev, peaks()[0])), flush=True)
            return
        run_ours(args)
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
