#!/usr/bin/env python
"""bench.py — q x g pairs/sec (distance + rank) of the PPS retrieval hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

A "step" is one pass of the ranking hot path over the workload: operand split -> tcgen05 distance
-> junk mask / positive thresholds -> counting sweep -> AP / first-match ranks (reference:
reid_dataset_evaluator.py:104-122, compute_dist -> mean_ap + cmc).  At N = 1 the workload is BASELINE.json
configs[1] (Market-1501-shaped, 3 368 x 19 732 x 2048 fp32).  At N > 1 every rank holds a gallery shard of
that size (weak scaling; global gallery = N x 19 732) and only the positives' distances and the integer
counters cross NVLink (NCCL all-reduce).

`value`  : whole-job pairs/s with the features resident in HBM (CUDA events, max over ranks).
`e2e`    : the same metric through the host-buffer entry point (N = 1: the C ABI's pps_evaluate_host;
           N > 1: pinned host -> device copies + the sharded path), H2D and D2H inside the timed region.
`roofline`: the distance GEMM (dominant kernel), timed with CUDA events inside the timed steps.
`cpu_baseline`: the reference's CPU path on this box's host cores (rank 0, N = 1): the UNMODIFIED
           reid_dataset_evaluator.py staged under baseline/_ref/ (kind "reference"), else the oracle port (kind "port").
`--impl reference`: only that CPU path, on a bounded query sample per step.
`large_gallery`: BASELINE configs[3] (Market + 500 k distractors, fp32) and configs[4] (10 M x 2048 fp16) - top-100 +
           exact positive ranks, the gallery sharded over the N GPUs of the run (STRONG scaling: total rows fixed), each
           with an oracle check on a query slice x the whole gallery (reference arithmetic on the host).
`dim8064`: the Market shape at the real concat width D = 8 064 = 63 x 128 (SURVEY 8d).
`checks`:  at N > 1 the headline result is checked against the oracle on a 64-query slice of the GLOBAL gallery.
`--dump-outputs DIR`: the per-query results of the last timed step as DIR/<name>.npy, to compare two builds.
The process exits non-zero (after printing the line) if any oracle check is outside north_star's tolerances.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import sys
import threading
import time

import numpy as np

if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
    os.environ["NCCL_DEBUG"] = "NONE"              # NCCL prints its version to stdout at these levels: keep stdout
                                                   # to the one JSON line (set NCCL_DEBUG=INFO to debug)

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "qxg_pairs_per_sec_distance_plus_rank"
UNIT = "pairs/s"
WORKLOAD = "market1501"          # BASELINE.json configs[1]


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def load_traffic(key):
    """Measured DRAM bytes per launch of a kernel at a given shape (ncu capture summarised under profiles/), or None."""
    path = os.path.join(ROOT, "profiles", "r02_traffic.json")
    try:
        with open(path) as f:
            return json.load(f).get(key)
    except (OSError, ValueError):
        return None


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm=float(p["hbm_gbs"]), tf_burst=float(p["bf16_tflops"]),
                    tf_sustained=float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), source="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback")


# ------------------------------------------------------------------------------------------------
# clocks sampler (NVML, in-process thread)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting"}

    def __init__(self, index, period=0.01):
        self.index, self.period = index, period
        self.samples, self.mask, self.max_mhz = [], 0, None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis:
                try:
                    phys = int(vis.split(",")[index])
                except (ValueError, IndexError):
                    phys = index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:                                 # noqa: BLE001 — no NVML: report nulls
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:                             # noqa: BLE001
                pass
            self._stop.wait(self.period)

    def start(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        if self._thr is not None:
            self._stop.set()
            self._thr.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": []}
        reasons = [name for bit, name in self.REASONS.items() if self.mask & bit]
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------
def make_workload(rank, world, gallery_per_gpu=None, dim=None):
    """Market-1501-shaped set; rank r gets gallery rows [r*ngl, (r+1)*ngl) of a world*ngl-row gallery.
    ids / cams are global (every rank builds the same arrays), features only for the local shard."""
    from pps_b200 import synthetic
    cfg = dict(synthetic.CONFIGS[WORKLOAD])
    if dim:
        cfg["dim"] = dim
    ngl = gallery_per_gpu or cfg["ng"]
    if world == 1 and ngl == cfg["ng"]:
        d = synthetic.make_reid_set(seed=0, **cfg)
        d["g_local"], d["row0"] = d["g"], 0
        return d, cfg
    nq, D, n_ids, n_cams = cfg["nq"], cfg["dim"], cfg["n_ids"], cfg["n_cams"]
    ng = ngl * world
    rs = np.random.RandomState(0)
    centers = rs.randn(n_ids, D)
    qid = rs.randint(1, n_ids + 1, size=nq).astype(np.int64)
    qcam = rs.randint(0, n_cams, size=nq).astype(np.int64)
    n_real = min(ng, cfg["ng"] - cfg["n_distractors"])            # Market's real ids + id-0 distractors
    gid = np.zeros(ng, dtype=np.int64)
    gid[rs.permutation(ng)[:n_real]] = rs.randint(1, n_ids + 1, size=n_real)
    gcam = rs.randint(0, n_cams, size=ng).astype(np.int64)

    def feats(ids, seed):
        r = np.random.RandomState(seed)
        out = np.empty((len(ids), D), dtype=np.float32)
        for r0 in range(0, len(ids), 8192):
            sl = ids[r0:r0 + 8192]
            x = np.where(sl[:, None] > 0, centers[np.maximum(sl, 1) - 1], 0.0) + 4.0 * r.standard_normal((len(sl), D))
            x /= np.linalg.norm(x, axis=1, keepdims=True)
            out[r0:r0 + 8192] = x
        return out

    row0 = rank * ngl
    shard = lambda r: feats(gid[r * ngl:(r + 1) * ngl], 100 + r)       # any rank's shard, regenerated for the oracle check
    d = dict(q=feats(qid, 1), g_local=shard(rank), qid=qid, gid=gid, qcam=qcam, gcam=gcam, row0=row0, shard=shard)
    cfg = dict(cfg, ng=ng)
    return d, cfg


# ------------------------------------------------------------------------------------------------
# CPU path (oracle port of the reference) — cpu_baseline and --impl reference
# ------------------------------------------------------------------------------------------------
_CPU_IMPL = None


def cpu_impl():
    """(kind, module): the unmodified reference evaluator if it is available (/root/reference in the authoring container,
    baseline/_ref/ on the GPU box), else the oracle port."""
    global _CPU_IMPL
    if _CPU_IMPL is None:
        from oracle import ref_loader
        if ref_loader.available():
            with contextlib.redirect_stdout(sys.stderr):
                _CPU_IMPL = ("reference", ref_loader.load(), ref_loader.EVALUATOR)
        else:
            from oracle import pps_oracle as O
            _CPU_IMPL = ("port", O, "oracle/pps_oracle.py")
    return _CPU_IMPL


def cpu_eval(d, nq_sample):
    """compute_dist -> mean_ap + cmc(topk=10, first_match_break) on the first nq_sample queries x full gallery, exactly as
    the reference's evaluate() closure calls them (reid_dataset_evaluator.py:70-93)."""
    kind, M, _ = cpu_impl()
    q = d["q"][:nq_sample]
    ids = dict(query_ids=d["qid"][:nq_sample], gallery_ids=d["gid"], query_cams=d["qcam"][:nq_sample],
               gallery_cams=d["gcam"])
    with contextlib.redirect_stdout(sys.stderr):      # the reference prints a scikit-learn version note to stdout
        t0 = time.perf_counter()
        dist = M.compute_dist(q, d["g"], type="euclidean")
        t1 = time.perf_counter()
        m = M.mean_ap(dist, **ids)
        t2 = time.perf_counter()
        c = M.cmc(dist, topk=10, separate_camera_set=False, single_gallery_shot=False, first_match_break=True, **ids) \
            if kind == "reference" else M.cmc(dist, topk=10, first_match_break=True, **ids)
        t3 = time.perf_counter()
    return dict(total=t3 - t0, dist=t1 - t0, mean_ap=t2 - t1, cmc=t3 - t2, mAP=m, cmc1=float(c[0]), kind=kind)


def cpu_sample_text(nq_s, nq, ng):
    kind, _, path = cpu_impl()
    what = ("the UNMODIFIED reference functions compute_dist / mean_ap / cmc of %s" % os.path.relpath(path, ROOT)
            if kind == "reference" else "oracle/pps_oracle.py (numpy sgemm + argsort + sklearn AP, as reid_dataset_evaluator.py:244-439)")
    return "first %d of %d queries x full %d-row gallery per pass; %s" % (nq_s, nq, ng, what)


def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    from pps_b200 import synthetic
    cfg = dict(synthetic.CONFIGS[WORKLOAD])
    d = synthetic.make_reid_set(seed=0, **cfg)
    cores = os.cpu_count() or 1
    probe = cpu_eval(d, 32)
    per_q = probe["total"] / 32.0
    budget = 150.0 / max(args.steps + args.warmup, 1)                 # whole run within a few minutes
    nq_s = int(max(16, min(cfg["nq"], budget / max(per_q, 1e-6))))
    for _ in range(args.warmup):
        cpu_eval(d, nq_s)
    t0 = time.perf_counter()
    last = None
    for _ in range(args.steps):
        last = cpu_eval(d, nq_s)
    dt = time.perf_counter() - t0
    pairs = float(nq_s) * cfg["ng"]
    value = pairs * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "market1501-shaped 3368x19732x2048 fp32 (BASELINE configs[1])", "nq": cfg["nq"],
                   "ng": cfg["ng"], "dim": cfg["dim"], "sample": "first %d queries x full gallery per step" % nq_s},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": last["kind"],
                         "sample": cpu_sample_text(nq_s, cfg["nq"], cfg["ng"]),
                         "split_s": {k: last[k] for k in ("dist", "mean_ap", "cmc")}},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
# sub-records: large galleries (BASELINE configs[3] / configs[4]) and the D = 8 064 shape
# ------------------------------------------------------------------------------------------------
def timed_passes(torch, engine, q, g, steps, warmup, world, dev):
    """ms per pass of engine.run(q, g): CUDA events on the launching stream, barrier + synchronize on both sides, max over
    ranks; also the distance-GEMM launch times (events the engine records around its distance calls)."""
    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()
    res = None
    for _ in range(warmup):
        res = engine.run(q, g)
    barrier()
    engine.set_phase_timing(True)          # the C pass sums the device time of its distance launches per pass
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    gemm, phases = [], {}
    e0.record()
    for _ in range(steps):
        res = engine.run(q, g)
        ph = engine.last_phase_ms()
        gemm.append(ph["dist_gemm"])
        for k_, v_ in ph.items():
            phases[k_] = phases.get(k_, 0.0) + v_ / steps
    e1.record()
    barrier()
    engine.set_phase_timing(False)
    engine.last_pass_phases = {"split": phases.get("split"), "dist_gemm": phases.get("dist_gemm"), "rank_count_and_merge": phases.get("rank_count"),
                               "finalize": phases.get("finalize"), "host_wait_pair_lists": phases.get("pairs_enqueue"),
                               "host_wait_final_sync": phases.get("d2h")}
    t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t[0]), res, (float(np.sum(gemm)) / steps if gemm else None)


def oracle_rows_device_gallery(torch, q_rows_host, ids_global, shard_iter):
    """Oracle distance rows [n_sel, ng] of a gallery that only exists on the device: every block is brought to the host,
    cast to float32 (BASELINE.md section 3) and goes through the CPU compute_dist (reference arithmetic)."""
    from oracle import pps_oracle as O
    ng = len(ids_global)
    out = np.empty((q_rows_host.shape[0], ng), dtype=np.float32)
    for col0, block in shard_iter:
        gh = block.float().cpu().numpy()
        out[:, col0:col0 + gh.shape[0]] = O.compute_dist(q_rows_host, gh)
    return out


def bench_large_gallery(torch, evaluator, synthetic, args, name, ng, dtype_name, world, rank, dev, group, peaks, steps, warmup,
                        n_check):
    """Top-100 retrieval + exact positive ranks over a gallery of `ng` rows sharded over the `world` GPUs of the run
    (strong scaling).  Returns the sub-record (rank 0) or None."""
    from oracle import parity as P
    nq, dim, topk, sigma = 3368, 2048, 100, 4.0
    tdt = torch.float16 if dtype_name == "fp16" else torch.float32
    qid, qcam, gid, gcam = synthetic.make_distractor_ids(nq, ng)
    row0, ngl = evaluator.gallery_shard(ng, rank, world)
    q = synthetic.make_features_device(qid, dim, 750, sigma, 7, dev, tdt)
    g = synthetic.make_features_device(gid[row0:row0 + ngl], dim, 750, sigma, 1000 + rank, dev, tdt)
    eng = evaluator.RankEngine(qid, gid, qcam, gcam, nq=nq, ng_local=ngl, dim=dim, gallery_offset=row0, precision=args.precision,
                               topk=topk, group=group, device=dev, in_dtype=tdt)
    n0 = evaluator._lib.launch_count()
    ms, res, gemm_ms = timed_passes(torch, eng, q, g, steps, warmup, world, dev)
    launches = (evaluator._lib.launch_count() - n0) / float(steps + warmup)
    rec = None
    if rank == 0:
        pairs = float(nq) * float(ng)
        tf = 2.0 * dim * pairs / (ms * 1e-3) / 1e12
        rec = {"workload": name, "nq": nq, "ng": ng, "dim": dim, "dtype": dtype_name, "topk": topk, "n_gpus": world,
               "scaling": "strong", "rows_per_gpu": ngl, "blocks_per_gpu": eng.pass_blocks or len(eng._chunk_list()),
               "counting_epilogue": bool(eng.used_fused_count),   # blocks after the first never written (fp16 rows)
               "steps": steps,
               "ms_per_pass": ms, "pairs_per_s": pairs / (ms * 1e-3), "algorithmic_tflops": tf,
               "frac_of_sustained_bf16_all_gpus": tf / (peaks["tf_sustained"] * world),
               "dist_gemm_ms_per_pass_rank0": gemm_ms, "gpu_launches_per_pass_rank0": launches,
               "phase_sums_ms_rank0": getattr(eng, "last_pass_phases", None),
               "mAP": res.mean_ap(), "cmc1": float(res.cmc(10, True)[0])}
        # oracle check: a query slice x the WHOLE gallery, regenerated shard by shard on this GPU and ranked on the host
        del g
        sel = np.arange(0, nq, nq // n_check)[:n_check]
        qh = q[torch.from_numpy(sel).to(dev)].float().cpu().numpy()

        def blocks():
            for r in range(world):
                r0, rows = evaluator.gallery_shard(ng, r, world)
                for b0, blk in synthetic.iter_features_device(gid[r0:r0 + rows], dim, 750, sigma, 1000 + r, dev, tdt):
                    yield r0 + b0, blk
        t0 = time.perf_counter()
        dist = oracle_rows_device_gallery(torch, qh, gid, blocks())
        chk = P.subset_check(res, sel, dist, qid, qcam, gid, gcam, topk=topk)
        chk["seconds"] = time.perf_counter() - t0
        chk["what"] = "oracle (CPU compute_dist on float32 casts + count-based AP / first match / top-%d) on %d queries x all %d rows" % (
            topk, len(sel), ng)
        rec["oracle_check"] = chk
    del eng
    torch.cuda.empty_cache()
    return rec


def bench_dim8064(torch, evaluator, synthetic, args, dev, peaks):
    """SURVEY 8d: the Market shape at D = 8 064 = 63 x 128 (reid_heads.py:95-101 concat width), one GPU."""
    from oracle import parity as P
    from oracle import pps_oracle as O
    cfg = dict(synthetic.CONFIGS[WORKLOAD])
    nq, ng, dim = cfg["nq"], cfg["ng"], 8064
    rs = np.random.RandomState(0)
    qid = rs.randint(1, cfg["n_ids"] + 1, size=nq).astype(np.int64)
    qcam = rs.randint(0, cfg["n_cams"], size=nq).astype(np.int64)
    gid = np.concatenate([rs.randint(1, cfg["n_ids"] + 1, size=ng - cfg["n_distractors"]),
                          np.zeros(cfg["n_distractors"], dtype=np.int64)])[rs.permutation(ng)].astype(np.int64)
    gcam = rs.randint(0, cfg["n_cams"], size=ng).astype(np.int64)
    sigma = 4.0 * 2.0                                   # 4x the dimensions of the D = 2048 set: same mid-range mAP
    q = synthetic.make_features_device(qid, dim, cfg["n_ids"], sigma, 7, dev, torch.float32)
    g = synthetic.make_features_device(gid, dim, cfg["n_ids"], sigma, 8, dev, torch.float32)
    eng = evaluator.RankEngine(qid, gid, qcam, gcam, nq=nq, ng_local=ng, dim=dim, precision=args.precision, device=dev)
    eng.use_c_path = False                              # the pass reports the device time of its distance launches
    ms, res, gemm_ms = timed_passes(torch, eng, q, g, 20, 3, 1, dev)
    flops = 2.0 * dim * nq * ng
    sel = np.arange(0, nq, nq // 64)[:64]
    dist = O.compute_dist(q[torch.from_numpy(sel).to(dev)].cpu().numpy(), g.cpu().numpy())
    chk = P.subset_check(res, sel, dist, qid, qcam, gid, gcam)
    terms = 1 if args.precision == "bf16x1" else (6 if args.precision == "bf16x6" else 3)
    return {"workload": "market1501-shaped %dx%dx%d fp32 (real reid_feature_concat width)" % (nq, ng, dim), "ms_per_pass": ms,
            "pairs_per_s": nq * float(ng) / (ms * 1e-3), "mAP": res.mean_ap(), "oracle_check": chk,
            "roofline": {"kernel": "dist_tc2_kernel", "bound": "tensor", "ms_per_launch": gemm_ms,
                         "achieved": flops / (gemm_ms * 1e-3) / 1e12, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                         "frac": flops / (gemm_ms * 1e-3) / 1e12 / peaks["tf_sustained"],
                         "tensor_pipe_frac": terms * flops / (gemm_ms * 1e-3) / 1e12 / peaks["tf_sustained"],
                         "algorithmic_flops_per_pair": 2 * dim}}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def synthetic_mod():
    from pps_b200 import synthetic
    return synthetic


def run_ours(args):
    import torch
    import pps_b200
    from pps_b200 import _lib, evaluator

    world = env_int("WORLD_SIZE", 1)
    rank = env_int("RANK", 0)
    local_rank = env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # one process per GPU: keep this rank (and, by first touch, its pinned staging buffers) on the GPU's NUMA node
    from pps_b200 import numa
    numa_info = numa.bind_to_gpu_node(local_rank) if (world > 1 and not args.no_numa_bind) else {"bound": False, "reason": "single GPU"}
    group = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
    peaks = load_peaks()

    d, cfg = make_workload(rank, world, args.gallery_per_gpu, args.dim)
    nq, ng, dim = cfg["nq"], cfg["ng"], cfg["dim"]
    ngl = d["g_local"].shape[0]
    pairs_step = float(nq) * float(ng)                            # all ranks together

    q_host = torch.from_numpy(d["q"]).pin_memory()
    g_host = torch.from_numpy(d["g_local"]).pin_memory()
    q_dev, g_dev = q_host.to(dev), g_host.to(dev)

    engine = evaluator.RankEngine(d["qid"], d["gid"], d["qcam"], d["gcam"], nq=nq, ng_local=ngl, dim=dim,
                                  gallery_offset=d["row0"], precision=args.precision, topk=args.topk, group=group,
                                  device=dev)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def step_device():
        return engine.run(q_dev, g_dev)

    def step_e2e():
        if world == 1 and args.topk == 0:
            return pps_b200.evaluate_host(q_host, g_host, d["qid"], d["gid"], d["qcam"], d["gcam"], cmc_topk=10,
                                          precision=args.precision, device=local_rank)
        return engine.run_host(q_host, g_host)

    # ---- correctness gate on the first warm-up result (rank 0 prints mAP with the line) ----
    res = step_device()
    mAP = res.mean_ap()
    cmc = res.cmc(10, True)

    # secondary number (SURVEY 8c): the same ranking under the scikit-learn 0.18.1 (trapezoid) AP the reference asks for
    mAP_trap = None
    if world == 1:
        dmat = pps_b200.compute_dist(q_dev, g_dev, precision=args.precision)
        mAP_trap = pps_b200.mean_ap(dmat, d["qid"], d["gid"], d["qcam"], d["gcam"], ap_definition="trapezoid")
        del dmat

    sampler = ClockSampler(local_rank)
    for _ in range(max(args.warmup - 1, 0)):
        step_device()
    barrier()
    sampler.start()
    n0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c_path = engine.n_chunks == 1 and args.topk == 0
    phase_sum = {}
    if c_path:
        engine.set_phase_timing(True)      # events between the phases of the one C call, on the same stream
    else:
        engine.kernel_events = []          # events around the distance GEMM launches
    ev0.record()
    for _ in range(args.steps):
        last = step_device()
        if c_path:
            for k, v in engine.last_phase_ms().items():
                phase_sum[k] = phase_sum.get(k, 0.0) + v
    ev1.record()
    barrier()
    launches = _lib.launch_count() - n0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)     # here: the e2e passes below reuse the engine's top-k arrays
    ms_total = ev0.elapsed_time(ev1)
    if c_path:
        engine.set_phase_timing(False)
        gemm_ms = [phase_sum["dist_gemm"] / args.steps]
        phases = {k: v / args.steps for k, v in phase_sum.items()}
        if not engine.use_c_path or world > 1:
            # the C pass reports SUMS per pass: split, dist_gemm, rank_count, finalize; two of the slots carry host stalls
            phases = {"split": phases["split"], "dist_gemm": phases["dist_gemm"], "rank_count": phases["rank_count"],
                      "finalize": phases["finalize"], "host_wait_pair_lists": phases["pairs_enqueue"],
                      "host_wait_final_sync": phases["d2h"]}
    else:
        gemm_ms = [a.elapsed_time(b) for a, b in engine.kernel_events]
        engine.kernel_events = None
        phases = None

    # ---- e2e: host buffers -> metrics, copies inside ----
    for _ in range(min(args.warmup, 3)):
        step_e2e()
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        out = step_e2e()
    barrier()
    e2e_s = time.perf_counter() - t0
    sampler.stop()

    # ---- part 1 of the path, reported beside the headline: fused pooling kernel (HBM-bound) ----
    pooling = None
    if world == 1 and not args.no_pooling:
        pooling = bench_pooling(torch, pps_b200, _lib, peaks, dev, args)

    t = torch.tensor([ms_total, e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    ms_total, e2e_s = float(t[0]), float(t[1])

    # ---- N > 1: the sharded result against the oracle on a 64-query slice of the GLOBAL gallery ----
    checks = {}
    if world > 1 and rank == 0 and not args.no_checks:
        from oracle import parity as P
        from oracle import pps_oracle as O
        sel = np.arange(0, nq, nq // 64)[:64]
        g_all = np.concatenate([d["shard"](r) for r in range(world)])
        chk = P.subset_check(res, sel, O.compute_dist(d["q"][sel], g_all), d["qid"], d["qcam"], d["gid"], d["gcam"], topk=args.topk)
        chk["what"] = "oracle (CPU compute_dist + count-based AP / first match) on 64 queries x all %d rows of the %d shards" % (ng, world)
        checks["sharded_vs_oracle"] = chk
        del g_all

    # ---- sub-records: the >= 1M-row galleries north_star's scaling target names, and D = 8 064 ----
    h2d = (q_host.numel() + g_host.numel()) * 4
    engine = q_dev = g_dev = g_host = None
    release_contexts = getattr(evaluator, "release_host_contexts", None)
    if release_contexts:
        release_contexts()
    torch.cuda.empty_cache()
    large = None
    if not args.no_large_gallery:
        large = {}
        for key, name, rows, dt, st, wu, nchk in (
                ("config3", "BASELINE configs[3]: Market-1501 + 500k distractors, fp32", args.c3_rows, "fp32", 5, 2, 64),
                ("config4", "BASELINE configs[4]: 10M-row gallery, 2048-d fp16", args.c4_rows, "fp16", 3, 1, 32)):
            if rows <= 0:
                continue
            rec = bench_large_gallery(torch, evaluator, synthetic_mod(), args, name, rows, dt, world, rank, dev, group, peaks,
                                      st, wu, nchk)
            if rank == 0:
                large[key] = rec
    dim8064 = None
    if world == 1 and not args.no_dim8064:
        dim8064 = bench_dim8064(torch, evaluator, synthetic_mod(), args, dev, peaks)

    if rank == 0:
        ms_step = ms_total / args.steps
        value = pairs_step / (ms_step * 1e-3)
        gemm_avg_ms = float(np.mean(gemm_ms)) if gemm_ms else None
        flops_alg = 2.0 * dim * float(nq) * float(ngl)               # per launch (this rank's block)
        terms = {"bf16x1": 1, "bf16x3": 3, "bf16x6": 6, "f16x3": 3}[args.precision]
        roofline = None
        if gemm_avg_ms:
            achieved = flops_alg / (gemm_avg_ms * 1e-3) / 1e12
            roofline = {"kernel": "dist_tc2_kernel", "bound": "tensor", "achieved": achieved,
                        "peak": peaks["tf_sustained"], "unit": "TFLOP/s", "frac": achieved / peaks["tf_sustained"],
                        "traffic": load_traffic("dist_tc2_kernel@%dx%dx%d/%s" % (nq, ngl, dim, args.precision)) or
                                   load_traffic("dist_tc2_kernel@%dx%dx%d/bf16x3" % (nq, ngl, dim)),
                        "traffic_unit": "DRAM bytes per launch (ncu --set full, profiles/r02_e_kernels.md); algorithmic = %d" %
                                        int((nq + ngl) * dim * 2 * (2 if args.precision in ("bf16x3", "f16x3") else 1) + nq * ngl * 4),
                        "peak_source": peaks["source"] + " (sustained bf16)",
                        "ms_per_launch": gemm_avg_ms, "share_of_step": gemm_avg_ms / ms_step,
                        "tensor_pipe_issued_tflops": achieved * terms,
                        "tensor_pipe_frac": achieved * terms / peaks["tf_sustained"],
                        "note": "achieved counts ALGORITHMIC flops (2*D per pair); the fp32-accurate %s split issues "
                                "%dx that on the tensor pipe" % (args.precision, terms)}
        # the HBM-bound kernels of the step, from the same phase events (algorithmic bytes / device time)
        kernels = None
        if phases:
            n_planes = {"bf16x1": 1, "bf16x3": 2, "bf16x6": 3, "f16x3": 2}[args.precision]
            split_b = (nq + ngl) * dim * 4.0 + (nq + ngl) * dim * 2.0 * n_planes
            count_b = 4.0 * nq * ngl
            kernels = {
                "split_rows_kernel": {"bound": "hbm", "ms": phases["split"], "achieved": split_b / phases["split"] / 1e6,
                                      "peak": peaks["hbm"], "unit": "GB/s", "frac": split_b / phases["split"] / 1e6 / peaks["hbm"],
                                      "note": "two launches (queries, gallery) + launch gap; overlaps the pair-list sweeps"},
                "rank_count_kernel": {"bound": "hbm (shared-atomic limited)", "ms": phases["rank_count"],
                                      "achieved": count_b / phases["rank_count"] / 1e6, "peak": peaks["hbm"], "unit": "GB/s",
                                      "frac": count_b / phases["rank_count"] / 1e6 / peaks["hbm"],
                                      "traffic": load_traffic("rank_count_kernel@%dx%d" % (nq, ngl))},
            }
        d2h = nq * (8 + 1 + 4)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": {"bf16x3": "bf16x3-split fp32 (fp32 accumulate)",
                                           "f16x3": "f16x3-split fp32 (two scaled fp16 planes, fp32 accumulate)"}.get(args.precision, args.precision),
            "data": "synthetic",
            "config": {"workload": "market1501-shaped %dx%dx%d fp32 (BASELINE configs[1]%s)" %
                                   (nq, ng, dim, "" if world == 1 else ", gallery sharded %d rows/GPU" % ngl),
                       "nq": nq, "ng": ng, "dim": dim, "gallery_rows_per_gpu": ngl, "precision": args.precision,
                       "topk": args.topk, "l2": "inputs larger than L2 (features %.0f MB + planes + %.0f MB distance block per step)" %
                                                ((nq + ngl) * dim * 4 / 1e6, nq * ngl * 4 / 1e6)},
            "e2e": {"value": pairs_step * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "steps": e2e_steps, "ms_per_step": 1e3 * e2e_s / e2e_steps,
                    "api": "pps_evaluate_host (C ABI, pinned host buffers)" if world == 1 and args.topk == 0
                           else "RankEngine.run_host (C pass with pps_pass_set_host_input: slab-pipelined upload of the shard from pinned, NUMA-local host rows)"},
            "gpu_launches": int(launches),
            "numa": numa_info,
            "clocks": sampler.summary(),
            "roofline": roofline,
            "phases_ms": phases,
            "kernels": kernels,
            "pooling": pooling,
            "large_gallery": large,
            "dim8064": dim8064,
            "checks": checks,
            "result": {"mAP": mAP, "cmc1": float(cmc[0]), "cmc5": float(cmc[4]), "cmc10": float(cmc[9]),
                       "mAP_trapezoid_sklearn_0_18_1": mAP_trap},
        }
        if world == 1 and not args.no_cpu_baseline:
            dd = dict(d, g=d["g_local"])
            nq_s = min(nq, args.cpu_sample)
            r = cpu_eval(dd, nq_s)
            line["cpu_baseline"] = {"value": nq_s * float(ng) / r["total"], "unit": UNIT, "cores": os.cpu_count() or 1,
                                    "kind": r["kind"], "sample": cpu_sample_text(nq_s, nq, ng),
                                    "split_s": {k: r[k] for k in ("dist", "mean_ap", "cmc")}, "mAP_on_sample": r["mAP"]}
            if nq_s == nq:
                line["result"]["mAP_cpu"] = r["mAP"]
                line["result"]["mAP_abs_diff"] = abs(r["mAP"] - mAP)
        else:
            line["cpu_baseline"] = None
        failed = []
        if line["result"].get("mAP_abs_diff") is not None and line["result"]["mAP_abs_diff"] > 1e-6:
            failed.append("headline mAP differs from the CPU reference by %.3g" % line["result"]["mAP_abs_diff"])
        for name_, c in list(checks.items()) + [(k, (v or {}).get("oracle_check")) for k, v in (large or {}).items()] + \
                [("dim8064", (dim8064 or {}).get("oracle_check"))]:
            if c is not None and not c.get("ok", True):
                failed.append("%s: %s" % (name_, "; ".join(c.get("errors", []))))
        line["parity_ok"] = not failed
        if failed:
            line["parity_failures"] = failed
        print(json.dumps(line))
        rc = 0 if not failed else 3
    else:
        rc = 0
    if world > 1:
        t = torch.tensor([rc], dtype=torch.int32, device=dev)
        torch.distributed.broadcast(t, src=0)
        rc = int(t[0])
        torch.distributed.destroy_process_group()
    return rc


def dump_outputs(out_dir, res):
    """What one step of the headline path returns to its caller (RankEngine.run's RankResult, plus the mAP / CMC the caller
    reads from it) as DIR/<name>.npy in float32 / float64: the workload is seeded, so two builds of the project can be
    compared output for output.  nq = 3 368 and topk <= 128 keep the files under 6 MB in all."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"ap": res.ap, "is_valid": res.is_valid, "first_rank": res.first_rank, "topk_index": res.topk_index,
              "topk_dist": res.topk_dist, "mAP": np.float64(res.mean_ap()), "cmc": res.cmc(10, True)}
    for name, a in arrays.items():
        if a is None:
            continue
        a = np.asarray(a)
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)                  # integer outputs (ranks, indices, flags) are exact in float64
        np.save(os.path.join(out_dir, name + ".npy"), a)


def bench_pooling(torch, pps_b200, _lib, peaks, dev, args):
    """pps_pool_fwd on Market-shaped conv5 maps: [1024, 2048, 24, 8] fp32 (1.6 GB in, 0.5 GB out per launch;
    far larger than L2), n = 6 parts, 63 combos, mode max_ave.  Algorithmic bytes = 4*C*H*W + 4*63*C per image."""
    n_img, C, H, W, n_parts = args.pool_images, 2048, 24, 8, 6
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn((n_img, C, H, W), device=dev, generator=g).clamp_min_(0)
    y = torch.empty((n_img, 63, C), device=dev)
    for _ in range(3):
        pps_b200.pps_pool(x, n_parts=n_parts, mode="max_ave", out=y)
    torch.cuda.synchronize()
    iters = 20
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        pps_b200.pps_pool(x, n_parts=n_parts, mode="max_ave", out=y)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    bytes_alg = n_img * (4.0 * C * H * W + 4.0 * 63 * C)
    gbs = bytes_alg / (ms * 1e-3) / 1e9
    return {"kernel": "pool_tma_kernel", "images_per_s": n_img / (ms * 1e-3), "ms_per_launch": ms,
            "shape": [n_img, C, H, W], "n_parts": n_parts, "combos": 63, "mode": "max_ave",
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s",
                         "frac": gbs / peaks["hbm"],
                         "traffic": load_traffic("pool_tma_kernel@%dx%dx%dx%d/n%d/max_ave" % (n_img, C, H, W, n_parts)),
                         "algorithmic_bytes": int(bytes_alg), "peak_source": peaks["source"]}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="f16x3", choices=["bf16x1", "bf16x3", "bf16x6", "f16x3"])
    ap.add_argument("--topk", type=int, default=0)
    ap.add_argument("--gallery-per-gpu", type=int, default=None)
    ap.add_argument("--dim", type=int, default=None)
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--cpu-sample", type=int, default=3368)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pooling", action="store_true")
    ap.add_argument("--pool-images", type=int, default=1024)
    ap.add_argument("--no-large-gallery", action="store_true")
    ap.add_argument("--c3-rows", type=int, default=519732, help="gallery rows of the configs[3] sub-record (0 = skip)")
    ap.add_argument("--c4-rows", type=int, default=10_000_000, help="gallery rows of the configs[4] sub-record (0 = skip)")
    ap.add_argument("--no-dim8064", action="store_true")
    ap.add_argument("--no-checks", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
