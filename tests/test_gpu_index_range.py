"""GalleryIndex.range_search: every gallery row within a radius of each query (include/pps_b200.h part 2h,
pps_index_range_search / pps_search_range_tc / pps_sort_key_segments).

The oracle is NumPy over compute_dist's matrix of the same rows (the search's distances, bit for bit): keep d <= r, order
by (distance, index).  With r the k-th distance of search(q, k), the first k results are search's row."""
import os
import socket

import numpy as np
import pytest

from conftest import GOLDEN_CASES, GOLDEN_DIR

S = 4096                                  # keys per tile of the segment sort
PRECISIONS = ["fp16", "f16x3", "bf16x1", "bf16x3", "bf16x6"]     # fp16: float16 rows; the others split float32 rows


def _dtype_name(prec):
    return "fp16" if prec == "fp16" else "fp32"


def _as(a, dtype_name):
    return np.ascontiguousarray(a, dtype=np.float16 if dtype_name == "fp16" else np.float32)


def _index(g, prec, tags=None):
    import torch
    import pps_b200
    f16 = prec == "fp16"
    idx = pps_b200.GalleryIndex(g.shape[1], dtype=torch.float16 if f16 else torch.float32,
                                precision="f16x3" if f16 else prec)
    idx.add(g, tags)
    return idx


def _own_dist(q, g, prec):
    """compute_dist's matrix for the index's arithmetic"""
    import torch
    import pps_b200
    if prec == "fp16":
        return pps_b200.compute_dist(torch.from_numpy(q).cuda(), torch.from_numpy(g).cuda()).cpu().numpy()
    return np.asarray(pps_b200.compute_dist(q, g, precision=prec))


def _oracle(dist, radius, keep=None):
    """(lims, dist, index) of every kept entry with d <= radius[i], per row in (distance, index) order"""
    lims, ds, ix = [0], [], []
    for i in range(dist.shape[0]):
        ok = dist[i] <= np.float32(radius[i])
        if keep is not None:
            ok &= keep[i]
        cand = np.nonzero(ok)[0]
        order = cand[np.lexsort((cand, dist[i, cand]))]
        ix.append(order)
        ds.append(dist[i, order])
        lims.append(lims[-1] + len(order))
    return np.array(lims, np.int64), np.concatenate(ds).astype(np.float32), np.concatenate(ix).astype(np.int64)


def _assert_same(got, want, msg=""):
    np.testing.assert_array_equal(np.asarray(got[0]), want[0], err_msg="lims " + msg)
    np.testing.assert_array_equal(np.asarray(got[2]), want[2], err_msg="index " + msg)
    np.testing.assert_array_equal(np.asarray(got[1]).view(np.uint32), np.asarray(want[1]).view(np.uint32),
                                  err_msg="dist " + msg)


def _range(idx, q, radius, flags=0, exclude_tags=None):
    return idx._unpack_range(*idx._range_keys(q, radius, 0, flags, exclude_tags))


def _queries(d, nq):
    pool = np.concatenate([d["q"], d["g"]])
    return np.ascontiguousarray(pool[np.arange(nq) % len(pool)])


def _radii(dist, ks):
    """named per-query radii: 0, the k-th distance for each k (inf when the gallery is shorter), a mix, inf, -1, NaN"""
    nq, ng = dist.shape
    srt = np.sort(dist, axis=1)
    out = {"zero": np.zeros(nq, np.float32)}
    for k in ks:
        out["kth%d" % k] = srt[:, k - 1] if k <= ng else np.full(nq, np.inf, np.float32)
    mix = srt[np.arange(nq), np.arange(nq) * 7 % ng].copy()
    mix[::5] = -1.0
    mix[1::5] = np.inf
    mix[2::5] = np.nan
    out.update({"mix": mix, "inf": np.full(nq, np.inf, np.float32), "neg": np.full(nq, -1.0, np.float32),
                "nan": np.full(nq, np.nan, np.float32)})
    return out


def _check_topk_invariant(idx, q, got, radius, k):
    """the first k results of row i are search(q, k)'s row; every further one has distance exactly radius[i]"""
    sd, si = idx.search(q, k)
    lims, dist, index = got
    for i in range(q.shape[0]):
        a, b = lims[i], lims[i + 1]
        assert b - a >= k
        np.testing.assert_array_equal(index[a:a + k], si[i])
        np.testing.assert_array_equal(dist[a:a + k].view(np.uint32), sd[i].view(np.uint32))
        assert (dist[a + k:b] == np.float32(radius[i])).all()


@pytest.mark.gpu
@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_range_search_equals_oracle(golden, name, prec):
    """Every golden case and precision, query batches of every tile width: the NumPy oracle over compute_dist, bit for
    bit, and the top-k invariant at the k-th distances."""
    d = golden(name)
    dn = _dtype_name(prec)
    g = _as(d["g"], dn)
    idx = _index(g, prec)
    ng = g.shape[0]
    for nq in (1, 33, 257):
        q = _as(_queries(d, nq), dn)
        dist = _own_dist(q, g, prec)
        for rname, radius in _radii(dist, (1, 13, 100)).items():
            got = _range(idx, q, radius)
            _assert_same(got, _oracle(dist, radius), "%s %s nq=%d radius=%s" % (name, prec, nq, rname))
            if rname.startswith("kth") and int(rname[3:]) <= ng:
                _check_topk_invariant(idx, q, got, radius, int(rname[3:]))
    # the public call with a scalar radius: numpy in, numpy out
    q = _as(d["q"], dn)
    dist = _own_dist(q, g, prec)
    r = float(np.median(dist))
    lims, dd, ii = idx.range_search(q, r)
    assert lims.dtype == np.int64 and dd.dtype == np.float32 and ii.dtype == np.int64
    _assert_same((lims, dd, ii), _oracle(dist, np.full(q.shape[0], r, np.float32)))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f16x3", "bf16x1", "bf16x3", "bf16x6", "fp16"])
@pytest.mark.parametrize("nq", [20, 50, 100, 200, 300])
def test_range_kernel_counts_and_capacity(precision, nq):
    """pps_search_range_tc directly: per-query limits (every row, a median, none), slices at arbitrary offsets and
    capacities below the count.  cnt is exact, each slice holds cap of the hits with compute_dist's bits, and nothing
    past a capacity is written."""
    import torch
    import pps_b200
    from pps_b200 import _lib, evaluator
    lib = _lib.load()
    rs = np.random.RandomState(nq)
    ng, dim, col0 = 700, 200, 1000
    f16 = precision == "fp16"
    dt = np.float16 if f16 else np.float32
    q = rs.randn(nq, dim).astype(dt)
    g = rs.randn(ng, dim).astype(dt)
    g[5] = q[3]
    prec = _lib.PREC_F16X1 if f16 else _lib.PRECISIONS[precision]
    planes = _lib.PLANES_FOR[prec]
    scaled = prec == _lib.PREC_F16X3
    sq = evaluator.SplitOperand(torch.from_numpy(q).cuda(), planes, scaled)
    sg = evaluator.SplitOperand(torch.from_numpy(g).cuda(), planes, scaled)
    if f16:
        want = pps_b200.compute_dist(torch.from_numpy(q).cuda(), torch.from_numpy(g).cuda()).cpu().numpy()
    else:
        want = np.asarray(pps_b200.compute_dist(q, g, precision=precision))
    bits = np.ascontiguousarray(want).view(np.uint32)
    med = np.median(want, axis=1).astype(np.float32).view(np.uint32)
    lim = np.where(np.arange(nq) % 3 == 0, np.uint32(0x7f800001), med + np.uint32(1)).astype(np.uint32)
    lim[2::3] = 0
    want_cnt = (bits < lim[:, None]).sum(1)
    cap = np.where(np.arange(nq) % 2 == 0, ng, np.arange(nq) % 50).astype(np.uint32)
    gap = 5
    off = np.concatenate([[0], np.cumsum(cap.astype(np.int64) + gap)[:-1]]) + 3
    out_n = int(off[-1] + cap[-1] + gap)
    lim_t = torch.from_numpy(lim.view(np.int32)).cuda()
    cnt = torch.zeros(nq, dtype=torch.int32, device="cuda")
    off_t = torch.from_numpy(off).cuda()
    cap_t = torch.from_numpy(cap.view(np.int32)).cuda()
    out = torch.full((out_n,), -7, dtype=torch.int64, device="cuda")
    _lib.check(lib.pps_search_range_tc(_lib.ptr(sg.planes), _lib.ptr(sg.sqnorm), ng, planes, 0, _lib.ptr(sq.planes),
                                       _lib.ptr(sq.sqnorm), nq, planes, 0, dim, prec, 0, col0, _lib.ptr(lim_t),
                                       _lib.ptr(cnt), _lib.ptr(off_t), _lib.ptr(cap_t), _lib.ptr(out), None, None,
                                       _lib.stream_ptr()), "pps_search_range_tc")
    np.testing.assert_array_equal(cnt.cpu().numpy(), want_cnt)
    o = out.cpu().numpy()
    written = np.zeros(out_n, bool)
    for i in range(nq):
        n = min(int(cap[i]), int(want_cnt[i]))
        seg = o[off[i]:off[i] + n].view(np.uint64)
        written[off[i]:off[i] + n] = True
        rows = (seg & np.uint64(0xffffffff)).astype(np.int64) - col0
        assert len(np.unique(rows)) == n and (rows >= 0).all() and (rows < ng).all()
        np.testing.assert_array_equal((seg >> np.uint64(32)).astype(np.uint32), bits[i, rows])
        assert (bits[i, rows] < lim[i]).all()
        if n == want_cnt[i]:
            np.testing.assert_array_equal(np.sort(rows), np.nonzero(bits[i] < lim[i])[0])
    assert (o[~written] == -7).all()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_second_pass_forced_by_small_slices(dtype_name):
    """Slices of 1, 7 and 64 keys per query run over and the second pass writes the result layout: the same answer as
    the default slices, before and after (the index then remembers a slice large enough for the largest count)."""
    from pps_b200 import _lib
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    prec = "fp16" if dtype_name == "fp16" else "f16x3"
    g = _as(d["g"], dtype_name)
    q = _as(_queries(d, 40), dtype_name)
    dist = _own_dist(q, g, prec)
    idx = _index(g, prec)
    radius = np.sort(dist, axis=1)[:, 300]
    want = _oracle(dist, radius)
    assert np.diff(want[0]).max() > 64
    _assert_same(_range(idx, q, radius), want, "default")
    for n in (1, 7, 64):
        _assert_same(_range(idx, q, radius, _lib.index_tkcap(n)), want, "tkcap %d" % n)
    _assert_same(_range(idx, q, np.full(40, np.inf, np.float32)), _oracle(dist, np.full(40, np.inf)), "inf")
    _assert_same(_range(idx, q, radius), want, "default after")


def _sort_segments(keys, lims):
    import torch
    from pps_b200 import _lib
    lib = _lib.load()
    k = torch.from_numpy(keys.view(np.int64)).cuda()
    l = torch.from_numpy(lims).cuda()
    scratch = torch.empty_like(k)
    _lib.check(lib.pps_sort_key_segments(_lib.ptr(k), _lib.ptr(l), len(lims) - 1, _lib.ptr(scratch), _lib.stream_ptr()),
               "pps_sort_key_segments")
    return k.cpu().numpy().view(np.uint64)


@pytest.mark.gpu
def test_sort_key_segments_equals_numpy():
    """Segment lengths around every boundary of the tile and merge stages, in one call, on random unique keys; then with
    duplicate keys, and with a first segment that starts past position 0 (keys before it are left alone)."""
    rs = np.random.RandomState(5)
    lens = [0, 1, 31, 32, 33, S - 1, S, S + 1, 3 * S + 7, (1 << 20) + 3, 0, 5, 2 * S]
    rs.shuffle(lens)
    lims = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    n = int(lims[-1])
    keys = rs.randint(0, 1 << 62, size=n, dtype=np.int64).view(np.uint64)
    got = _sort_segments(keys.copy(), lims)
    for s in range(len(lens)):
        np.testing.assert_array_equal(got[lims[s]:lims[s + 1]], np.sort(keys[lims[s]:lims[s + 1]]), err_msg="segment %d" % s)
    dup = rs.randint(0, 50, size=n).astype(np.uint64)
    got = _sort_segments(dup.copy(), lims)
    for s in range(len(lens)):
        np.testing.assert_array_equal(got[lims[s]:lims[s + 1]], np.sort(dup[lims[s]:lims[s + 1]]))
    keys2 = rs.randint(0, 1 << 62, size=3 * S + 100, dtype=np.int64).view(np.uint64)
    lims2 = np.array([77, 77 + S + 5, 3 * S + 90], np.int64)
    got = _sort_segments(keys2.copy(), lims2)
    np.testing.assert_array_equal(got[:77], keys2[:77])
    np.testing.assert_array_equal(got[3 * S + 90:], keys2[3 * S + 90:])
    for s in range(2):
        np.testing.assert_array_equal(got[lims2[s]:lims2[s + 1]], np.sort(keys2[lims2[s]:lims2[s + 1]]))


def _junk_tags(ids, cams):
    return (np.asarray(ids, np.int64) << 32) | np.asarray(cams, np.int64)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_excluding_range_search(golden, name, dtype_name):
    """Camera tags and junk-rule tags: the plain range result with the excluded rows filtered out in NumPy."""
    d = golden(name)
    prec = "fp16" if dtype_name == "fp16" else "f16x3"
    g = _as(d["g"], dtype_name)
    q = _as(d["q"], dtype_name)
    dist = _own_dist(q, g, prec)
    for gt, qt in ((d["gcam"], d["qcam"]), (_junk_tags(d["gid"], d["gcam"]), _junk_tags(d["qid"], d["qcam"]))):
        gt, qt = np.asarray(gt, np.int64), np.asarray(qt, np.int64)
        idx = _index(g, prec, gt)
        keep = gt[None, :] != qt[:, None]
        for radius in (np.sort(dist, axis=1)[:, min(40, g.shape[0] - 1)], np.full(q.shape[0], np.inf, np.float32)):
            _assert_same(_range(idx, q, radius, exclude_tags=qt), _oracle(dist, radius, keep))
            _assert_same(_range(idx, q, radius), _oracle(dist, radius))       # without exclude tags: every row


@pytest.mark.gpu
def test_range_search_errors_and_edges():
    """Untagged index with exclude tags, wrong lengths, bad radius; empty index, nq = 0, no result, CUDA in / out."""
    import torch
    import pps_b200
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    g, q = d["g"], d["q"][:9]
    idx = _index(g, "f16x3")
    tagged = _index(g, "f16x3", np.arange(g.shape[0]) % 3)
    for bad in (lambda: idx.range_search(q, 1.0, exclude_tags=np.zeros(9, np.int64)),
                lambda: tagged.range_search(q, 1.0, exclude_tags=np.zeros(8, np.int64)),
                lambda: idx.range_search(q, np.ones(8, np.float32)),
                lambda: idx.range_search(q, np.ones((9, 1), np.float32)),
                lambda: idx.range_search(q, np.ones(9, np.complex64)),
                lambda: idx.range_search(q, np.ones(9, bool)),
                lambda: idx.range_search(q, True),
                lambda: idx.range_search(q, "1.0"),
                lambda: idx.range_search(q, torch.ones(9, dtype=torch.bool)),
                lambda: idx.range_search(q.astype(np.float16), 1.0),
                lambda: idx.range_search(q[0], 1.0)):
        with pytest.raises(RuntimeError):
            bad()
    dist = _own_dist(q, g, "f16x3")
    r = float(np.median(dist))
    # integer and float64 radii are converted to float32
    for radius, as_f32 in ((np.full(9, int(r), np.int32), np.full(9, int(r), np.float32)),
                           (torch.full((9,), r, dtype=torch.float64), np.full(9, r, np.float32)),
                           (int(r), np.full(9, int(r), np.float32)), (np.float64(r), np.full(9, r, np.float32))):
        _assert_same(idx.range_search(q, radius), _oracle(dist, as_f32))
    # no result at all, nq = 0
    lims, dd, ii = idx.range_search(q, -1.0)
    assert (lims == 0).all() and lims.shape == (10,) and dd.shape == (0,) and ii.shape == (0,)
    lims, dd, ii = idx.range_search(q[:0], np.zeros(0, np.float32))
    assert lims.shape == (1,) and lims[0] == 0 and dd.shape == (0,)
    # an empty index answers with empty lists, also with exclude tags
    empty = pps_b200.GalleryIndex(g.shape[1], dtype=torch.float32)
    for kw in ({}, {"exclude_tags": np.zeros(9, np.int64)}):
        lims, dd, ii = empty.range_search(q, np.inf, **kw)
        assert (lims == 0).all() and lims.shape == (10,) and ii.shape == (0,)
    # CUDA in -> CUDA tensors on the index's device
    r = np.sort(dist, axis=1)[:, 20]
    lims_t, dd_t, ii_t = idx.range_search(torch.from_numpy(q).cuda(), torch.from_numpy(r).cuda())
    assert lims_t.is_cuda and dd_t.is_cuda and ii_t.dtype == torch.int64
    _assert_same((lims_t.cpu().numpy(), dd_t.cpu().numpy(), ii_t.cpu().numpy()), _oracle(dist, r))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_range_after_remove_and_growth_equals_fresh_index(dtype_name):
    """Adds through two capacity doublings, then a removal: the same answer as a fresh index of the remaining rows."""
    import torch
    import pps_b200
    rs = np.random.RandomState(11)
    prec = "fp16" if dtype_name == "fp16" else "f16x3"
    g = _as(rs.randn(2600, 96), dtype_name)
    q = _as(rs.randn(40, 96), dtype_name)
    parts = pps_b200.GalleryIndex(96, dtype=torch.float16 if dtype_name == "fp16" else torch.float32)
    parts.add(g[:100])
    parts.add(g[100:1600])
    parts.add(g[1600:])
    dist = _own_dist(q, g, prec)
    radius = np.sort(dist, axis=1)[:, 150]
    _assert_same(parts.range_search(q, radius), _oracle(dist, radius))
    gone = rs.choice(2600, 700, replace=False)
    parts.remove(gone)
    live = np.delete(g, gone, axis=0)
    fresh = _index(live, prec)
    a, b = parts.range_search(q, radius), fresh.range_search(q, radius)
    _assert_same(a, b)
    _assert_same(a, _oracle(_own_dist(q, live, prec), radius))


def _shards(ng, sizes):
    b = np.cumsum([0] + list(sizes))
    assert b[-1] == ng
    return [(int(b[i]), int(b[i + 1])) for i in range(len(sizes))]


@pytest.mark.gpu
@pytest.mark.parametrize("sizes", [(350, 350), (0, 500, 200), (100, 0, 300, 300)])
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_sharded_range_equals_one_index(sizes, dtype_name):
    """2, 3 and 4 indexes (one empty) stand for ranks: each searches with its shard's offset and merge_range_lists joins
    the results - the single index's answer bit for bit."""
    import pps_b200
    from pps_b200 import index as index_mod
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    prec = "fp16" if dtype_name == "fp16" else "f16x3"
    g = _as(d["g"], dtype_name)
    q = _as(_queries(d, 33), dtype_name)
    one = _index(g, prec)
    dist = _own_dist(q, g, prec)
    for radius in (np.sort(dist, axis=1)[:, 100], np.full(33, np.inf, np.float32), np.full(33, -1.0, np.float32)):
        lims, keys = [], []
        for r0, r1 in _shards(g.shape[0], sizes):
            shard = pps_b200.GalleryIndex(g.shape[1], dtype=one.dtype)
            shard.add(g[r0:r1])
            lx, kx, _ = shard._range_keys(q, radius, r0)
            lims.append(lx)
            keys.append(kx)
        got = one._unpack_range(*index_mod.merge_range_lists(lims, keys), True)
        _assert_same(got, _range(one, q, radius))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _nccl_radius(d):
    """a radius that admits about half of small_mid's rows"""
    diff = d["q"].astype(np.float64)[:, None, :] - d["g"].astype(np.float64)[None, :, :]
    return float(np.median(np.sqrt((diff ** 2).sum(-1))))


def _nccl_worker(rank, world, port, out_dir):
    import torch
    import torch.distributed as dist
    import pps_b200
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    r0, r1 = [(0, 300), (300, 700)][rank]
    idx = pps_b200.GalleryIndex(d["g"].shape[1], dtype=torch.float32, group=dist.group.WORLD)
    idx.add(d["g"][r0:r1])
    lims, dist_, index = idx.range_search(d["q"], _nccl_radius(d))
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), lims=lims, dist=dist_, index=index)
    dist.destroy_process_group()


@pytest.mark.gpu
def test_sharded_range_search_over_nccl(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    world = 2
    mp.spawn(_nccl_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    want = _index(d["g"], "f16x3").range_search(d["q"], _nccl_radius(d))
    for r in range(world):
        o = dict(np.load(os.path.join(str(tmp_path), "rank%d.npz" % r)))
        _assert_same((o["lims"], o["dist"], o["index"]), want)


@pytest.mark.gpu
def test_config4_shaped_fp16_gallery_range():
    """A 600 000 x 2048 fp16 gallery: 64 queries at a radius of about 1 000 hits, and 2 queries at inf (600 000-key
    segments through the merge passes), against the oracle on the GPU's own compute_dist rows."""
    import torch
    import pps_b200
    from pps_b200 import synthetic
    dev = torch.device("cuda")
    ng, dim = 600000, 2048
    qid, _, gid, _ = synthetic.make_distractor_ids(3368, ng)
    q = synthetic.make_features_device(qid[:64], dim, 750, 4.0, 7, dev, torch.float16)
    g = synthetic.make_features_device(gid, dim, 750, 4.0, 1000, dev, torch.float16)
    idx = pps_b200.GalleryIndex(dim, dtype=torch.float16)
    idx.add(g)
    own = pps_b200.compute_dist(q, g).cpu().numpy()
    radius = np.partition(own, 999, axis=1)[:, 999]
    lims, dd, ii = idx.range_search(q, torch.from_numpy(radius).to(dev))
    _assert_same((lims.cpu().numpy(), dd.cpu().numpy(), ii.cpu().numpy()), _oracle(own, radius))
    lims, dd, ii = idx.range_search(q[:2].contiguous(), float("inf"))
    _assert_same((lims.cpu().numpy(), dd.cpu().numpy(), ii.cpu().numpy()), _oracle(own[:2], np.full(2, np.inf)))
