"""Top-k search of a resident gallery (pps_b200.GalleryIndex) against the same top-k through rank_eval, one JSON line per
(gallery, batch).

Galleries: fp16 at 1 M and 10 M rows x 2048 (configs[4]'s arithmetic) and fp32 split f16x3 at 519 732 rows (configs[3]);
batches of 1, 16, 64, 256 and 3 368 queries, k = 100.  Every gallery is far larger than the 126 MB L2, so each search
reads it from HBM.  A line records:
  search_ms          median device time of GalleryIndex.search (queries in, [nq, k] distances / indices out; the call
                     ends in its one 4-byte read-back), CUDA events, after warm-up
  rank_eval_ms       median time of the same top-k through rank_eval with ids that match no gallery row (the way a user
                     gets it without the index: the gallery is split again by every call)
  agree              the two outputs are identical (indices and distance bits)
  gallery_bytes      bytes of resident gallery operands read per search (planes + norms, once), and hbm_share: those bytes
                     over search_ms against the data sheet's 7.7 TB/s - what bounds small batches
  tflops             algorithmic rate 2 * nq * ng * dim * terms / search_ms (terms: 1 for fp16, 3 for f16x3) - what bounds
                     large batches
  gpu, power_limit_w the card and its enforced power limit, read in the same run

--tags MODES (comma-separated; default none: the lines above) measures searches that leave out rows by tag instead, one
line per (gallery, mode, batch).  The index holds the mode's tags; an unfiltered search of the same index (the untagged
answer and code path) alternates with the excluding search, so both see the same card state.  Modes:
  cam6   tag = camera: 6 cameras evenly (make_distractor_ids), exclude tag = the query's camera (cross-camera search)
  half   one tag on a random half of the rows (the others carry 5 more tags), every query excludes it
  junk   tag = id << 32 | camera on both sides (make_distractor_ids labels): the evaluation's junk rule
A line records untagged_ms / excluding_ms (medians of the alternated searches) and their ratio, excluded_share (the mean
share of rows a query leaves out) and, for junk, rank_eval_ms and agree against rank_eval(..., topk=k) with the same
labels.  The camera modes have no rank_eval equivalent at these sizes (every id equal: nq x ng pair lists).

usage: python tools/index_bench.py [--reps 10] [--warmup 2] [--out FILE] [--cases fp16_1M,fp16_10M,fp32_520k]
                                   [--tags none,cam6,half,junk] [--batches 1,16,64,256,3368]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DIM, K = 2048, 100
HBM_BYTES_PER_S = 7.7e12          # HGX B200 data sheet, one GPU
CASES = {"fp16_1M": (1_000_000, "fp16"), "fp16_10M": (10_000_000, "fp16"), "fp32_520k": (519_732, "fp32")}
BATCHES = [1, 16, 64, 256, 3368]
TAG_MODES = ["none", "cam6", "half", "junk"]


def card(index):
    import torch
    name = torch.cuda.get_device_name(index)
    watts = None
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[index]) if vis else index
        watts = pynvml.nvmlDeviceGetEnforcedPowerLimit(pynvml.nvmlDeviceGetHandleByIndex(phys)) / 1000.0
    except Exception:                                          # noqa: BLE001 — no NVML: ask nvidia-smi
        try:
            out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", str(index)],
                                 stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout
            watts = float(out.strip().splitlines()[0])
        except Exception:                                      # noqa: BLE001
            watts = None
    return name, watts


def timed(fn, reps, warmup):
    import torch
    for _ in range(warmup):
        out = fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms)), float(np.min(ms)), out


def timed_alternating(fa, fb, reps, warmup):
    """medians of fa's and fb's device times, the two timed in turn"""
    import torch
    for _ in range(warmup):
        fa()
        fb()
    torch.cuda.synchronize()
    ms = ([], [])
    outs = [None, None]
    for _ in range(reps):
        for j, fn in enumerate((fa, fb)):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            outs[j] = fn()
            b.record()
            b.synchronize()
            ms[j].append(a.elapsed_time(b))
    return float(np.median(ms[0])), float(np.median(ms[1])), outs[1]


def mode_tags(mode, ng, nq, labels):
    """(gallery tags [ng], query exclude tags [nq]) of a tag mode"""
    qid, qcam, gid, gcam = labels
    if mode == "cam6":
        return gcam, qcam[:nq]
    if mode == "half":
        rs = np.random.RandomState(3)
        return np.where(rs.rand(ng) < 0.5, 0, rs.randint(1, 6, ng)).astype(np.int64), np.zeros(nq, np.int64)
    return (gid << 32) | gcam, (qid[:nq] << 32) | qcam[:nq]


def run_tagged_case(name, modes, batches, reps, warmup, emit):
    import torch
    import pps_b200
    from pps_b200 import synthetic
    ng, dtype_name = CASES[name]
    dev = torch.device("cuda")
    tdt = torch.float16 if dtype_name == "fp16" else torch.float32
    labels = synthetic.make_distractor_ids(max(batches), ng)
    qid, qcam, gid, gcam = labels
    q_all = synthetic.make_features_device(qid, DIM, 750, 4.0, 7, dev, tdt)
    g = synthetic.make_features_device(gid, DIM, 750, 4.0, 1000, dev, tdt)
    gpu, watts = card(torch.cuda.current_device())
    for mode in modes:
        gtags, qtags_all = mode_tags(mode, ng, max(batches), labels)
        idx = pps_b200.GalleryIndex(DIM, dtype=tdt, precision="f16x3")
        idx.add(g, gtags)
        vals, counts = np.unique(gtags, return_counts=True)
        rows_of = dict(zip(vals.tolist(), counts.tolist()))
        for nq in batches:
            q = q_all[:nq].contiguous()
            qt = torch.from_numpy(np.ascontiguousarray(qtags_all[:nq])).to(dev)
            u_ms, x_ms, (xd, xi) = timed_alternating(lambda: idx.search(q, K), lambda: idx.search(q, K, exclude_tags=qt),
                                                     reps, warmup)
            share = float(np.mean([rows_of.get(int(t), 0) for t in qtags_all[:nq]])) / ng
            rec = {"case": name, "dtype": dtype_name, "precision": "f16x1" if dtype_name == "fp16" else "f16x3", "ng": ng,
                   "dim": DIM, "nq": nq, "k": K, "tags": mode, "untagged_ms": round(u_ms, 4), "excluding_ms": round(x_ms, 4),
                   "ratio": round(x_ms / u_ms, 3), "excluded_share": round(share, 4)}
            if mode == "junk":
                r_ms, _, res = timed(lambda: pps_b200.rank_eval(q, g, qid[:nq], gid, qcam[:nq], gcam, topk=K),
                                     max(2, reps // 3), 1)
                rec["rank_eval_ms"] = round(r_ms, 3)
                rec["agree"] = bool(np.array_equal(xi.cpu().numpy(), res.topk_index.astype(np.int64))
                                    and np.array_equal(xd.cpu().numpy().view(np.uint32), res.topk_dist.view(np.uint32)))
            else:
                rec["rank_eval"] = "no equivalent: camera-only exclusion needs every id equal (nq x ng pair lists)"
            rec.update({"reps": reps, "gpu": gpu, "power_limit_w": watts})
            emit(rec)
        del idx
        torch.cuda.empty_cache()
    del g, q_all
    torch.cuda.empty_cache()


def run_case(name, reps, warmup, emit, batches=BATCHES):
    import torch
    import pps_b200
    from pps_b200 import synthetic
    ng, dtype_name = CASES[name]
    dev = torch.device("cuda")
    tdt = torch.float16 if dtype_name == "fp16" else torch.float32
    qid, _, gid, _ = synthetic.make_distractor_ids(max(batches), ng)
    q_all = synthetic.make_features_device(qid, DIM, 750, 4.0, 7, dev, tdt)
    g = synthetic.make_features_device(gid, DIM, 750, 4.0, 1000, dev, tdt)
    idx = pps_b200.GalleryIndex(DIM, dtype=tdt, precision="f16x3")
    t0 = time.perf_counter()
    idx.add(g)
    torch.cuda.synchronize()
    add_s = time.perf_counter() - t0
    planes, terms = (1, 1) if dtype_name == "fp16" else (2, 3)
    gallery_bytes = ng * DIM * 2 * planes + ng * 4 * (1 if dtype_name == "fp16" else 2)
    gpu, watts = card(torch.cuda.current_device())
    zeros_g = np.zeros(ng, np.int64)
    for nq in batches:
        q = q_all[:nq].contiguous()
        fake = np.full(nq, -1)
        s_ms, s_min, (sd, si) = timed(lambda: idx.search(q, K), reps, warmup)
        r_ms, r_min, res = timed(lambda: pps_b200.rank_eval(q, g, fake, np.arange(ng), np.zeros(nq, np.int64), zeros_g, topk=K),
                                 max(2, reps // 3), 1)
        agree = bool(np.array_equal(si.cpu().numpy(), res.topk_index.astype(np.int64))
                     and np.array_equal(sd.cpu().numpy().view(np.uint32), res.topk_dist.view(np.uint32)))
        emit({"case": name, "dtype": dtype_name, "precision": "f16x1" if dtype_name == "fp16" else "f16x3", "ng": ng,
              "dim": DIM, "nq": nq, "k": K, "search_ms": round(s_ms, 4), "search_min_ms": round(s_min, 4),
              "rank_eval_ms": round(r_ms, 3), "rank_eval_min_ms": round(r_min, 3),
              "speedup": round(r_ms / s_ms, 2), "agree": agree,
              "gallery_bytes": gallery_bytes, "hbm_share": round(gallery_bytes / (s_ms * 1e-3) / HBM_BYTES_PER_S, 4),
              "tflops": round(2.0 * nq * ng * DIM * terms / (s_ms * 1e-3) / 1e12, 2),
              "add_s": round(add_s, 3), "reps": reps, "gpu": gpu, "power_limit_w": watts})
    del idx, g, q_all
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also append the lines to this file")
    ap.add_argument("--cases", default=",".join(CASES))
    ap.add_argument("--tags", default="none", help="comma-separated tag modes: " + ", ".join(TAG_MODES))
    ap.add_argument("--batches", default=",".join(str(b) for b in BATCHES))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("index_bench needs a CUDA device (B200)")
    names = [c for c in args.cases.split(",") if c]
    for c in names:
        if c not in CASES:
            raise SystemExit("unknown case %r (expected %s)" % (c, ", ".join(CASES)))
    modes = [m for m in args.tags.split(",") if m]
    for m in modes:
        if m not in TAG_MODES:
            raise SystemExit("unknown tag mode %r (expected %s)" % (m, ", ".join(TAG_MODES)))
    batches = [int(b) for b in args.batches.split(",") if b]

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")

    tagged = [m for m in modes if m != "none"]
    for c in names:
        if "none" in modes:
            run_case(c, args.reps, args.warmup, emit, batches)
        if tagged:
            run_tagged_case(c, tagged, batches, args.reps, args.warmup, emit)


if __name__ == "__main__":
    main()
