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

--remove measures GalleryIndex.remove instead, one line per (gallery, pattern): a fresh index of the whole gallery
loses one pattern of rows, then the same pattern again on what is left (the first call also allocates the removal's
scratch).  Patterns: row0 (everything after row 0 moves), last1000 (nothing moves), random1 / random10 (1 % / 10 % of the
rows at random, drawn again for the second call), front (the first tenth of the rows: 1 M of 10 M, then 900 000 of
the 9 M left).  A line records:
  remove_ms / remove_first_ms  host time of the second / first call, ending in a device synchronise
  moved_rows, moved_bytes      rows (and their planes, norms, scales) that the second call moved down
  copy_gbps, copy_share        4 x moved_bytes (a gather into the piece buffer, then a copy into place: each reads and
                               writes the bytes) over remove_ms, and that rate over the 6 525 GB/s copy rate of DESIGN §7
  search_ms / fresh_search_ms  medians of searches (per batch size) of the compacted index and of a fresh index of the
                               same rows, alternated; agree: their outputs are identical (indices and distance bits)

--range measures GalleryIndex.range_search instead, one line per (gallery, batch, target): every query gets the radius
that admits about `target` rows (its target-th distance, from a top-128 search of the same index for 10 and 100 hits,
from compute_dist's rows of the batch otherwise), targets 10, 1 000 and 100 000, plus inf (every row) at 1 and 16
queries.  Default galleries fp16_10M and fp32_520k, batches 1, 16, 64, 256.  A line records:
  range_ms / topk_ms     medians of range_search and of search(q, 100) on the same index, alternated
  hits_mean, hits_max    results per query
  total_keys             keys of the whole result (8 bytes each)
  split_ms               one more call with CUDA events around its parts: the first pass (search kernel), the second
                         pass (when a slice ran over) and the sort, from torch.profiler's kernel times
  ok                     the output against the top-k invariant: the first k results of each query equal search's row
                         (k = min(100, hits)), every result is within the radius, lims add up

--groups measures GalleryIndex.search_groups instead, one line per (gallery, layout, batch), k = 100.  The rows form
tracklets of 1, 16, 256 or 2 048 rows (group = row // length), stored contiguously or with the groups shuffled over the
rows.  Default galleries fp16_10M and fp32_520k, batches 1, 16, 64, 256.  A line records:
  groups_ms / search_ms  medians of search_groups(q, 100) and of search(q, 100) on the same index, alternated
  prefix_rows, chunks, fallback   the grouped schedule of the last call: rows swept as materialised blocks, chunks after
                         them, and whether the materialised fallback ran
  launches               kernels the library launched for one grouped call
  ok                     query 0's result against NumPy on compute_dist's own distances of the whole gallery (first row
                         of each group in key order), bit for bit

usage: python tools/index_bench.py [--reps 10] [--warmup 2] [--out FILE] [--cases fp16_1M,fp16_10M,fp32_520k]
                                   [--tags none,cam6,half,junk] [--batches 1,16,64,256,3368] [--remove] [--range]
                                   [--groups]
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
COPY_BYTES_PER_S = 6.525e12       # measured device-to-device copy rate (MEASURED_PEAKS.json, DESIGN §7)
REMOVE_PATTERNS = ["row0", "last1000", "random1", "random10", "front"]
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


def remove_rows(pattern, ng, rs):
    """local rows of a removal pattern on an index of ng rows"""
    if pattern == "row0":
        return np.array([0])
    if pattern == "last1000":
        return np.arange(ng - 1000, ng)
    if pattern == "random1":
        return rs.choice(ng, ng // 100, replace=False)
    if pattern == "random10":
        return rs.choice(ng, ng // 10, replace=False)
    return np.arange(ng // 10)


def run_remove_case(name, batches, reps, warmup, emit):
    import torch
    import pps_b200
    from pps_b200 import synthetic
    ng, dtype_name = CASES[name]
    dev = torch.device("cuda")
    tdt = torch.float16 if dtype_name == "fp16" else torch.float32
    qid, _, gid, _ = synthetic.make_distractor_ids(max(batches), ng)
    q_all = synthetic.make_features_device(qid, DIM, 750, 4.0, 7, dev, tdt)
    planes = 1 if dtype_name == "fp16" else 2
    row_bytes = DIM * 2 * planes + (4 if dtype_name == "fp16" else 8)      # planes (kpad = 2048) + norm (+ inverse scale)
    gpu, watts = card(torch.cuda.current_device())
    for pattern in REMOVE_PATTERNS:
        rs = np.random.RandomState(REMOVE_PATTERNS.index(pattern))
        # the seeded gallery again for every pattern: at most two indexes and one copy of the rows are held at a time
        # (about 123 GB at 10 M fp16 rows)
        g = synthetic.make_features_device(gid, DIM, 750, 4.0, 1000, dev, tdt)
        idx = pps_b200.GalleryIndex(DIM, dtype=tdt, precision="f16x3")
        idx.add(g)
        live = np.arange(ng)
        ms, moved = [], 0
        for _ in range(2):
            rows = remove_rows(pattern, len(live), rs)
            rows_t = torch.from_numpy(rows).to(dev)
            moved = len(live) - int(rows.min()) - len(rows)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n = idx.remove(rows_t)
            torch.cuda.synchronize()
            ms.append((time.perf_counter() - t0) * 1e3)
            assert n == len(rows)
            live = np.delete(live, rows)
        g = g.index_select(0, torch.from_numpy(live).to(dev))
        torch.cuda.empty_cache()
        fresh = pps_b200.GalleryIndex(DIM, dtype=tdt, precision="f16x3")
        fresh.add(g)                      # one add: the capacity is the row count, as the compacted index's
        del g
        torch.cuda.synchronize()
        rec = {"case": name, "dtype": dtype_name, "precision": "f16x1" if dtype_name == "fp16" else "f16x3", "ng": ng,
               "dim": DIM, "pattern": pattern, "removed_per_call": int(len(rows)), "size_after": len(idx),
               "remove_ms": round(ms[1], 3), "remove_first_ms": round(ms[0], 3), "moved_rows": moved,
               "moved_bytes": moved * row_bytes}
        rec["copy_gbps"] = round(4 * moved * row_bytes / (ms[1] * 1e-3) / 1e9, 1)
        rec["copy_share"] = round(rec["copy_gbps"] * 1e9 / COPY_BYTES_PER_S, 3)
        for nq in batches:
            q = q_all[:nq].contiguous()
            s_ms, f_ms, _ = timed_alternating(lambda: idx.search(q, K), lambda: fresh.search(q, K), reps, warmup)
            (ad, ai), (bd, bi) = idx.search(q, K), fresh.search(q, K)
            rec["search_ms_nq%d" % nq] = round(s_ms, 4)
            rec["fresh_search_ms_nq%d" % nq] = round(f_ms, 4)
            rec["agree_nq%d" % nq] = bool(torch.equal(ai, bi) and torch.equal(ad.view(torch.int32), bd.view(torch.int32)))
        rec.update({"k": K, "reps": reps, "gpu": gpu, "power_limit_w": watts})
        emit(rec)
        del idx, fresh
        torch.cuda.empty_cache()
    del q_all
    torch.cuda.empty_cache()


RANGE_TARGETS = [10, 1000, 100000, "inf"]


def range_radius(idx, q, own_rows, target):
    """[nq] float32 radii admitting about `target` rows per query"""
    import torch
    if target == "inf":
        return torch.full((q.shape[0],), float("inf"), dtype=torch.float32, device=q.device)
    if target <= 128:
        d, _ = idx.search(q, target)
        return d[:, target - 1].contiguous()
    return torch.kthvalue(own_rows(), target, dim=1).values.contiguous()


def check_range(idx, q, radius, out):
    """the top-k invariant (k = min(100, hits)) and the radius, on the GPU"""
    import torch
    lims, dist, index = out
    counts = (lims[1:] - lims[:-1]).cpu()
    if int(lims[0]) != 0 or int(lims[-1]) != dist.shape[0] or (counts < 0).any():
        return False
    if not bool((dist <= torch.repeat_interleave(radius, counts.to(radius.device))).all()):
        return False
    k = int(min(100, int(counts.min())))
    if k == 0:
        return True
    sd, si = idx.search(q, k)
    first = lims[:-1, None] + torch.arange(k, device=lims.device)[None, :]
    return bool(torch.equal(index[first], si) and torch.equal(dist[first].view(torch.int32), sd.view(torch.int32)))


def range_split_ms(fn):
    """device time of one call's kernels by part: first pass, second pass (search kernels after the first), sort"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    search, sort = [], 0.0
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        if "dist_tc2_kernel" in ev.name:
            search.append((ev.time_range.start, us))
        elif "seg_tile_sort" in ev.name or "seg_merge" in ev.name:
            sort += us
    search.sort()
    return {"first_pass_ms": round(search[0][1] / 1e3, 4) if search else None,
            "second_pass_ms": round(sum(u for _, u in search[1:]) / 1e3, 4),
            "sort_ms": round(sort / 1e3, 4)}


def run_range_case(name, batches, reps, warmup, emit):
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
    idx.add(g)
    gpu, watts = card(torch.cuda.current_device())
    for nq in batches:
        q = q_all[:nq].contiguous()
        rows = {}

        def own_rows():                    # compute_dist's rows of the batch, in pieces of the gallery (memory)
            if "d" not in rows:
                step = max(1, (1 << 30) // (4 * nq))
                rows["d"] = torch.cat([pps_b200.compute_dist(q, g[i:i + step]).float() for i in range(0, ng, step)], 1)
            return rows["d"]
        for target in RANGE_TARGETS:
            if target == "inf" and nq > 16:
                continue
            if target != "inf" and target >= ng:
                continue
            radius = range_radius(idx, q, own_rows, target)
            s_ms, r_ms, out = timed_alternating(lambda: idx.search(q, K), lambda: idx.range_search(q, radius), reps, warmup)
            lims = out[0]
            counts = (lims[1:] - lims[:-1]).float()
            rec = {"case": name, "dtype": dtype_name, "precision": "f16x1" if dtype_name == "fp16" else "f16x3", "ng": ng,
                   "dim": DIM, "nq": nq, "target_hits": target, "range_ms": round(r_ms, 4), "topk_ms": round(s_ms, 4),
                   "ratio": round(r_ms / s_ms, 3), "hits_mean": round(float(counts.mean()), 1),
                   "hits_max": int(counts.max()), "total_keys": int(lims[-1])}
            rec.update(range_split_ms(lambda: idx.range_search(q, radius)))
            rec["ok"] = check_range(idx, q, radius, out)
            rec.update({"k_topk": K, "reps": reps, "gpu": gpu, "power_limit_w": watts})
            emit(rec)
            del out
        rows.clear()
        torch.cuda.empty_cache()
    del idx, g, q_all
    torch.cuda.empty_cache()


GROUP_LENGTHS = [1, 16, 256, 2048]


def np_first_per_group(dist_row, groups, k):
    """(dist, index) of the first row of each group in (distance bits, row) order, the first k"""
    order = np.lexsort((np.arange(len(dist_row)), dist_row.view(np.uint32)))
    _, first = np.unique(groups[order], return_index=True)
    pick = order[np.sort(first)][:k]
    return dist_row[pick], pick


def run_groups_case(name, batches, reps, warmup, emit):
    import torch
    import pps_b200
    from pps_b200 import _lib, synthetic
    ng, dtype_name = CASES[name]
    dev = torch.device("cuda")
    tdt = torch.float16 if dtype_name == "fp16" else torch.float32
    qid, _, gid, _ = synthetic.make_distractor_ids(max(batches), ng)
    q_all = synthetic.make_features_device(qid, DIM, 750, 4.0, 7, dev, tdt)
    g = synthetic.make_features_device(gid, DIM, 750, 4.0, 1000, dev, tdt)
    own0 = pps_b200.compute_dist(q_all[:1], g)[0].cpu().numpy()          # query 0 against every row
    gpu, watts = card(torch.cuda.current_device())
    rs = np.random.RandomState(11)
    for length in GROUP_LENGTHS:
        for layout in ("contiguous", "shuffled"):
            groups = (np.arange(ng) // length).astype(np.int64)
            if layout == "shuffled":
                groups = groups[rs.permutation(ng)]
            want_d, want_i = np_first_per_group(own0, groups, K)
            idx = pps_b200.GalleryIndex(DIM, dtype=tdt, precision="f16x3")
            idx.add(g, None, torch.from_numpy(groups).to(dev))
            for nq in batches:
                q = q_all[:nq].contiguous()
                s_ms, g_ms, (gd, gi, _) = timed_alternating(lambda: idx.search(q, K), lambda: idx.search_groups(q, K),
                                                            reps, warmup)
                n0 = _lib.launch_count()
                idx.search_groups(q, K)
                launches = _lib.launch_count() - n0
                prefix, chunks, fallback = idx._group_stats()
                ok = bool(np.array_equal(gi[0].cpu().numpy(), want_i)
                          and np.array_equal(gd[0].cpu().numpy().view(np.uint32), want_d.view(np.uint32)))
                emit({"case": name, "dtype": dtype_name, "precision": "f16x1" if dtype_name == "fp16" else "f16x3",
                      "ng": ng, "dim": DIM, "nq": nq, "k": K, "group_rows": length, "layout": layout,
                      "groups_ms": round(g_ms, 4), "search_ms": round(s_ms, 4), "ratio": round(g_ms / s_ms, 3),
                      "prefix_rows": prefix, "chunks": chunks, "fallback": fallback, "launches": launches, "ok": ok,
                      "reps": reps, "gpu": gpu, "power_limit_w": watts})
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
    ap.add_argument("--remove", action="store_true", help="measure GalleryIndex.remove (default batches 1,64)")
    ap.add_argument("--range", action="store_true",
                    help="measure GalleryIndex.range_search (default galleries fp16_10M,fp32_520k, batches 1,16,64,256)")
    ap.add_argument("--groups", action="store_true",
                    help="measure GalleryIndex.search_groups (default galleries fp16_10M,fp32_520k, batches 1,16,64,256)")
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
    if args.remove and args.batches == ap.get_default("batches"):
        batches = [1, 64]
    if (args.range or args.groups) and args.batches == ap.get_default("batches"):
        batches = [1, 16, 64, 256]
    if (args.range or args.groups) and args.cases == ap.get_default("cases"):
        names = ["fp16_10M", "fp32_520k"]

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")

    if args.remove:
        for c in names:
            run_remove_case(c, batches, args.reps, args.warmup, emit)
        return
    if args.range:
        for c in names:
            run_range_case(c, batches, args.reps, args.warmup, emit)
        return
    if args.groups:
        for c in names:
            run_groups_case(c, batches, args.reps, args.warmup, emit)
        return
    tagged = [m for m in modes if m != "none"]
    for c in names:
        if "none" in modes:
            run_case(c, args.reps, args.warmup, emit, batches)
        if tagged:
            run_tagged_case(c, tagged, batches, args.reps, args.warmup, emit)


if __name__ == "__main__":
    main()
