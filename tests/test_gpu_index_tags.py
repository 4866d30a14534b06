"""GalleryIndex with row tags: a search that leaves out, for every query, the gallery rows whose tag is the query's
exclude tag (include/pps_b200.h part 2h, pps_index_add_tagged / pps_index_search_excluding).

With tag = (id << 32) | camera the answer is rank_eval's top-k (the evaluation's junk rule) bit for bit; with tag = camera
it is the cross-camera top-k of compute_dist's own distances."""
import os
import socket

import numpy as np
import pytest

import parity_util as P
from conftest import GOLDEN_CASES, GOLDEN_DIR
from oracle import pps_oracle as O

NQS = [1, 7, 31, 32, 33, 200, 257, 600]        # every query tile width (32 / 64 / 128 / 256) and its edges
KS = [1, 13, 100, 128]


def _hooks(prefix_blocks=0, tk_cap=0):
    from pps_b200 import _lib
    return _lib.index_prefix(prefix_blocks) | _lib.index_tkcap(tk_cap)


def _junk_tags(ids, cams):
    return (np.asarray(ids, np.int64) << 32) | np.asarray(cams, np.int64)


def _queries(d, nq):
    """nq query rows and their labels: the fixture's queries, then its gallery rows (exact self matches at distance 0,
    which the junk rule excludes)."""
    sel = np.arange(nq) % (len(d["q"]) + len(d["g"]))
    pick = lambda a, b: np.ascontiguousarray(np.concatenate([a, b])[sel])   # noqa: E731
    return pick(d["q"], d["g"]), pick(d["qid"], d["gid"]), pick(d["qcam"], d["gcam"])


def _as(a, dtype_name):
    return np.ascontiguousarray(a, dtype=np.float16 if dtype_name == "fp16" else np.float32)


def _torch_dtype(dtype_name):
    import torch
    return torch.float16 if dtype_name == "fp16" else torch.float32


def _index(g, dtype_name, tags=None):
    import pps_b200
    idx = pps_b200.GalleryIndex(g.shape[1], dtype=_torch_dtype(dtype_name))
    idx.add(g, tags)
    return idx


def _search(idx, q, k, flags=0, exclude_tags=None):
    keys, is_np = idx._search_keys(q, k, 0, flags, exclude_tags)
    return idx._unpack(keys, is_np)


def _rank_eval_topk(q, g, qid, gid, qcam, gcam, k):
    import torch
    import pps_b200
    res = pps_b200.rank_eval(torch.from_numpy(q).cuda(), torch.from_numpy(g).cuda(), qid, gid, qcam, gcam, topk=k)
    return res.topk_dist, res.topk_index.astype(np.int64)


def _own_dist(q, g, dtype_name):
    """compute_dist's matrix (the search's distances, bit for bit)."""
    import torch
    import pps_b200
    if dtype_name == "fp16":
        return pps_b200.compute_dist(torch.from_numpy(q).cuda(), torch.from_numpy(g).cuda()).cpu().numpy()
    return np.asarray(pps_b200.compute_dist(q, g))


def _np_topk(dist, keep, k):
    """the k smallest kept entries of every row, ordered by (distance, index); -1 / inf padded."""
    nq = dist.shape[0]
    out_i = np.full((nq, k), -1, np.int64)
    out_d = np.full((nq, k), np.inf, np.float32)
    for i in range(nq):
        cand = np.nonzero(keep[i])[0]
        order = cand[np.lexsort((cand, dist[i, cand]))][:k]
        out_i[i, :len(order)] = order
        out_d[i, :len(order)] = dist[i, order]
    return out_d, out_i


def _assert_same(got, want, msg=""):
    np.testing.assert_array_equal(got[1], want[1], err_msg=msg)
    np.testing.assert_array_equal(np.asarray(got[0]).view(np.uint32), np.asarray(want[0]).view(np.uint32), err_msg=msg)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_junk_rule_equals_rank_eval_topk(golden, name, dtype_name):
    """tag = id << 32 | cam on both sides: every batch width and k, with the default schedule and with a 256-row prefix
    (the excluding swapped-operand kernel + candidate merges cover the rest), bit for bit rank_eval's top-k."""
    d = golden(name)
    g = _as(d["g"], dtype_name)
    idx = _index(g, dtype_name, _junk_tags(d["gid"], d["gcam"]))
    for nq in NQS:
        q, qid, qcam = _queries(d, nq)
        q = _as(q, dtype_name)
        qtags = _junk_tags(qid, qcam)
        for k in KS:
            want = _rank_eval_topk(q, g, qid, d["gid"], qcam, d["gcam"], k)
            for flags in (0, _hooks(prefix_blocks=1)):
                got = _search(idx, q, k, flags, qtags)
                assert got[0].dtype == np.float32 and got[1].dtype == np.int64 and got[1].shape == (nq, k)
                _assert_same(got, want, "%s nq=%d k=%d flags=%x" % (name, nq, k, flags))
    # the public call
    q = _as(d["q"], dtype_name)
    got = idx.search(q, 13, exclude_tags=_junk_tags(d["qid"], d["qcam"]))
    _assert_same(got, _rank_eval_topk(q, g, d["qid"], d["gid"], d["qcam"], d["gcam"], 13))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_cross_camera_equals_masked_oracle(golden, name, dtype_name):
    """tag = camera: the k nearest rows from other cameras of compute_dist's own matrix, ordered by (distance, index);
    and rank_eval with every id equal (the same rows are junk) agrees."""
    d = golden(name)
    g = _as(d["g"], dtype_name)
    gcam = d["gcam"]
    idx = _index(g, dtype_name, gcam)
    for nq in (1, 33, 257):
        q, _, qcam = _queries(d, nq)
        q = _as(q, dtype_name)
        own = _own_dist(q, g, dtype_name)
        keep = gcam[None, :] != qcam[:, None]
        for k in (13, 100):
            want = _np_topk(own, keep, k)
            for flags in (0, _hooks(prefix_blocks=1)):
                _assert_same(_search(idx, q, k, flags, qcam), want, "%s nq=%d k=%d flags=%x" % (name, nq, k, flags))
            same = _rank_eval_topk(q, g, np.zeros(nq, np.int64), np.zeros(len(g), np.int64), qcam, gcam, k)
            _assert_same(same, want, "rank_eval %s nq=%d k=%d" % (name, nq, k))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f16x3", "bf16x1", "bf16x3", "bf16x6", "fp16"])
@pytest.mark.parametrize("nq", [20, 50, 100, 200, 300])
def test_excluding_search_kernel_candidates(precision, nq):
    """pps_search_topk_excl_tc with an all-ones bound and room for every row: the candidates are exactly the (query, row)
    pairs with different tags, each with compute_dist's distance bits (BN 32 / 64 / 128 / 256 and two query tiles)."""
    import torch
    import pps_b200
    from pps_b200 import _lib, evaluator
    lib = _lib.load()
    rs = np.random.RandomState(nq + 7)
    ng, dim, col0 = 700, 200, 1000
    f16 = precision == "fp16"
    dt = np.float16 if f16 else np.float32
    q = rs.randn(nq, dim).astype(dt)
    g = rs.randn(ng, dim).astype(dt)
    g[5] = q[3]
    gtags = rs.randint(0, 5, ng).astype(np.int64)
    qtags = rs.randint(0, 6, nq).astype(np.int64)        # tag 5: a query that excludes nothing
    prec = _lib.PREC_F16X1 if f16 else _lib.PRECISIONS[precision]
    planes = _lib.PLANES_FOR[prec]
    scaled = prec == _lib.PREC_F16X3
    sq = evaluator.SplitOperand(torch.from_numpy(q).cuda(), planes, scaled)
    sg = evaluator.SplitOperand(torch.from_numpy(g).cuda(), planes, scaled)
    cap = ng + 3
    bound = torch.full((nq,), -1, dtype=torch.int32, device="cuda")
    cnt = torch.zeros(nq, dtype=torch.int32, device="cuda")
    cand = torch.zeros((nq, cap), dtype=torch.int64, device="cuda")
    gt, qt = torch.from_numpy(gtags).cuda(), torch.from_numpy(qtags).cuda()
    _lib.check(lib.pps_search_topk_excl_tc(_lib.ptr(sg.planes), _lib.ptr(sg.sqnorm), ng, planes, 0, _lib.ptr(sq.planes),
                                           _lib.ptr(sq.sqnorm), nq, planes, 0, dim, prec, 0, col0, _lib.ptr(bound),
                                           _lib.ptr(cnt), _lib.ptr(cand), cap, _lib.stream_ptr(), _lib.ptr(gt), _lib.ptr(qt)),
               "pps_search_topk_excl_tc")
    keep = gtags[None, :] != qtags[:, None]
    cnt = cnt.cpu().numpy()
    np.testing.assert_array_equal(cnt, keep.sum(1))
    if f16:
        want = pps_b200.compute_dist(torch.from_numpy(q).cuda(), torch.from_numpy(g).cuda()).cpu().numpy()
    else:
        want = pps_b200.compute_dist(q, g, precision=precision)
    want = np.ascontiguousarray(want).view(np.uint32)
    cand = cand.cpu().numpy().view(np.uint64)
    for i in range(nq):
        keys = cand[i, :cnt[i]]
        idx = np.sort((keys & np.uint64(0xffffffff)).astype(np.int64) - col0)
        np.testing.assert_array_equal(idx, np.nonzero(keep[i])[0], err_msg="query %d" % i)
        rows = (keys & np.uint64(0xffffffff)).astype(np.int64) - col0
        np.testing.assert_array_equal((keys >> np.uint64(32)).astype(np.uint32), want[i, rows], err_msg="query %d" % i)
    # both tag arrays are required
    assert lib.pps_search_topk_excl_tc(_lib.ptr(sg.planes), _lib.ptr(sg.sqnorm), ng, planes, 0, _lib.ptr(sq.planes),
                                       _lib.ptr(sq.sqnorm), nq, planes, 0, dim, prec, 0, col0, _lib.ptr(bound), _lib.ptr(bound),
                                       _lib.ptr(bound), 1, _lib.stream_ptr(), None, _lib.ptr(qt)) == _lib.PPS_ERR_INVALID_ARG


def _np_update(keys, dist, col0, gtags, qtags, k):
    """numpy pps_topk_update_excl: the k smallest of the state and the kept columns' keys."""
    nq, ncols = dist.shape
    bits = dist.view(np.uint32).astype(np.uint64) << np.uint64(32)
    new = bits | (np.arange(ncols, dtype=np.uint64) + np.uint64(col0))[None, :]
    keep = gtags[None, :] != qtags[:, None]
    out = np.empty_like(keys)
    for i in range(nq):
        out[i] = np.sort(np.concatenate([keys[i], new[i, keep[i]]]))[:k]
    return out, (~keep).sum(1)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 13, 100, 128])
def test_topk_update_excl_equals_numpy(k):
    """pps_topk_update_excl over two blocks (the second one merges into the first one's state), with and without the
    excluded counts: numpy's k smallest kept keys, and the counts of the block's excluded columns."""
    import torch
    from pps_b200 import _lib
    lib = _lib.load()
    rs = np.random.RandomState(k)
    nq, ldd = 37, 3100
    blocks = [(3000, 50), (2100, 3050)]                     # (ncols, col0)
    keys_t = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    plain_t = torch.empty_like(keys_t)
    _lib.check(lib.pps_topk_init(_lib.ptr(keys_t), nq, k, _lib.stream_ptr()), "pps_topk_init")
    _lib.check(lib.pps_topk_init(_lib.ptr(plain_t), nq, k, _lib.stream_ptr()), "pps_topk_init")
    want = np.full((nq, k), np.uint64(0xffffffffffffffff), np.uint64)
    qtags = rs.randint(0, 4, nq).astype(np.int64)
    qtags[0] = 99                                           # excludes nothing
    qt = torch.from_numpy(qtags).cuda()
    for ncols, col0 in blocks:
        dist = np.abs(rs.randn(nq, ldd)).astype(np.float32)
        dist[:, 7] = dist[:, 8]                             # ties by index
        gtags = rs.randint(0, 4, ncols).astype(np.int64)
        dt, gt = torch.from_numpy(dist).cuda(), torch.from_numpy(gtags).cuda()
        n_ex = torch.full((nq,), 12345, dtype=torch.int32, device="cuda")
        _lib.check(lib.pps_topk_update_excl(_lib.ptr(dt), ldd, nq, ncols, col0, _lib.ptr(gt), _lib.ptr(qt), _lib.ptr(keys_t), k,
                                            _lib.ptr(n_ex), _lib.stream_ptr()), "pps_topk_update_excl")
        _lib.check(lib.pps_topk_update_excl(_lib.ptr(dt), ldd, nq, ncols, col0, _lib.ptr(gt), _lib.ptr(qt), _lib.ptr(plain_t),
                                            k, None, _lib.stream_ptr()), "pps_topk_update_excl")
        want, counts = _np_update(want, np.ascontiguousarray(dist[:, :ncols]), col0, gtags, qtags, k)
        np.testing.assert_array_equal(keys_t.cpu().numpy().view(np.uint64), want)
        np.testing.assert_array_equal(plain_t.cpu().numpy().view(np.uint64), want)
        np.testing.assert_array_equal(n_ex.cpu().numpy(), counts)
    assert lib.pps_topk_update_excl(_lib.ptr(dt), ldd, nq, 10, 0, None, _lib.ptr(qt), _lib.ptr(keys_t), k, None,
                                    _lib.stream_ptr()) == _lib.PPS_ERR_INVALID_ARG


@pytest.mark.gpu
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_excluding_edge_cases(dtype_name):
    """A tag covering the whole gallery leaves nothing; fewer than k remaining rows are padded; an unfiltered search on a
    tagged index is the untagged index's answer; an empty index answers with padding."""
    import torch
    import pps_b200
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    g, q = _as(d["g"], dtype_name), _as(d["q"][:40], dtype_name)
    ng = len(g)
    for flags in (0, _hooks(prefix_blocks=1)):
        everything = _index(g, dtype_name, np.full(ng, 7))
        dist, index = _search(everything, q, 100, flags, np.full(40, 7))
        assert (index == -1).all() and np.isinf(dist).all()
        # most rows share tag 1; queries 0..19 exclude them (30 rows remain), the others exclude nothing
        tags = np.where(np.arange(ng) % 70 < 67, 1, 2)
        idx = _index(g, dtype_name, tags)
        qtags = np.where(np.arange(40) < 20, 1, 3)
        want = _np_topk(_own_dist(q, g, dtype_name), tags[None, :] != qtags[:, None], 100)
        got = _search(idx, q, 100, flags, qtags)
        _assert_same(got, want)
        assert (got[1][:20, :30] >= 0).all() and (got[1][:20, 30:] == -1).all() and (got[1][20:] >= 0).all()
        # the tags do not change an unfiltered search
        _assert_same(_search(idx, q, 100, flags), _search(_index(g, dtype_name), q, 100, flags))
    empty = pps_b200.GalleryIndex(g.shape[1], dtype=_torch_dtype(dtype_name))
    dist, index = empty.search(q, 5, exclude_tags=np.zeros(40, np.int64))
    assert (index == -1).all() and np.isinf(dist).all()
    # CUDA tensors in, int32 tags: CUDA out
    qt = torch.from_numpy(q).cuda()
    dist_t, index_t = idx.search(qt, 100, exclude_tags=torch.from_numpy(qtags.astype(np.int32)).cuda())
    assert dist_t.is_cuda and index_t.is_cuda
    np.testing.assert_array_equal(index_t.cpu().numpy(), want[1])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_tagged_adds_in_pieces_equal_one_add(dtype_name):
    """Three tagged appends through two capacity doublings (first capacity 1 024 rows): the tags move with the rows."""
    import torch
    import pps_b200
    rs = np.random.RandomState(12)
    g = _as(rs.randn(2600, 96), dtype_name)
    q = _as(rs.randn(40, 96), dtype_name)
    tags = rs.randint(0, 6, 2600).astype(np.int64)
    qtags = rs.randint(0, 6, 40).astype(np.int64)
    one = _index(g, dtype_name, tags)
    parts = pps_b200.GalleryIndex(96, dtype=_torch_dtype(dtype_name))
    assert parts.add(g[:100], tags[:100]) == (0, 100)
    assert parts.add(torch.from_numpy(g[100:1600]).cuda(), torch.from_numpy(tags[100:1600]).cuda()) == (100, 1500)
    assert parts.add(g[1600:], tags[1600:].astype(np.int16)) == (1600, 1000)
    assert len(parts) == 2600
    want = _np_topk(_own_dist(q, g, dtype_name), tags[None, :] != qtags[:, None], 100)
    for flags in (0, _hooks(prefix_blocks=1)):
        _assert_same(_search(one, q, 100, flags, qtags), want)
        _assert_same(_search(parts, q, 100, flags, qtags), want)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_heavy_exclusion_through_chunks_and_fallback(dtype_name):
    """One tag on half the rows, excluded by every query: through the prefix + chunk path (chunks shrunk by the excluded
    share), and with rows sorted nearest-last and a 4-entry candidate buffer (every chunk overflows, the search repeats
    with materialised blocks) - exact either way."""
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    rs = np.random.RandomState(3)
    q = _as(d["q"][:33], dtype_name)
    ng = len(d["g"])
    tags = np.where(rs.permutation(ng) < ng // 2, 5, rs.randint(0, 5, ng))
    qtags = np.full(33, 5)
    d0 = O.compute_dist(d["q"][:33].astype(np.float32), d["g"].astype(np.float32)).mean(0)
    order = np.argsort(-d0, kind="stable")
    for perm, tk_cap in ((np.arange(ng), 0), (order, 4)):
        g = _as(d["g"][perm], dtype_name)
        idx = _index(g, dtype_name, tags[perm])
        own = _own_dist(q, g, dtype_name)
        for k in (1, 13, 100):
            want = _np_topk(own, tags[perm][None, :] != qtags[:, None], k)
            _assert_same(_search(idx, q, k, _hooks(prefix_blocks=1, tk_cap=tk_cap), qtags), want, "k=%d cap=%d" % (k, tk_cap))


def _shards(ng, sizes):
    b = np.cumsum([0] + list(sizes))
    assert b[-1] == ng
    return [(int(b[i]), int(b[i + 1])) for i in range(len(sizes))]


@pytest.mark.gpu
@pytest.mark.parametrize("sizes", [(350, 350), (0, 500, 200), (100, 0, 300, 300)])
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_sharded_tagged_indexes_equal_one_index(sizes, dtype_name):
    """2, 3 and 4 tagged indexes (one empty) stand for ranks: the same exclude tags on every shard, the keys merged as
    merge_topk_keys merges them - the single index's answer bit for bit."""
    import pps_b200
    from pps_b200 import evaluator
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    g = _as(d["g"], dtype_name)
    gtags = _junk_tags(d["gid"], d["gcam"])
    q, qid, qcam = _queries(d, 33)
    q = _as(q, dtype_name)
    qtags = _junk_tags(qid, qcam)
    one = _index(g, dtype_name, gtags)
    for k in (13, 100):
        for flags in (0, _hooks(prefix_blocks=1)):
            keys = []
            for r0, r1 in _shards(g.shape[0], sizes):
                shard = pps_b200.GalleryIndex(g.shape[1], dtype=one.dtype)
                shard.add(g[r0:r1], gtags[r0:r1])
                keys.append(shard._search_keys(q, k, r0, flags, qtags)[0])
            got = one._unpack(evaluator.merge_key_lists(keys, k), True)
            _assert_same(got, _search(one, q, k, flags, qtags))
            _assert_same(got, _rank_eval_topk(q, g, qid, d["gid"], qcam, d["gcam"], k))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


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
    idx.add(d["g"][r0:r1], _junk_tags(d["gid"][r0:r1], d["gcam"][r0:r1]))
    dist_, index = idx.search(d["q"], 100, exclude_tags=_junk_tags(d["qid"], d["qcam"]))
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), dist=dist_, index=index)
    dist.destroy_process_group()


@pytest.mark.gpu
def test_sharded_excluding_search_over_nccl(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    world = 2
    mp.spawn(_nccl_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    want = _rank_eval_topk(d["q"], d["g"], d["qid"], d["gid"], d["qcam"], d["gcam"], 100)
    for r in range(world):
        o = dict(np.load(os.path.join(str(tmp_path), "rank%d.npz" % r)))
        _assert_same((o["dist"], o["index"]), want)


@pytest.mark.gpu
@pytest.mark.parametrize("nq", [1, 64])
def test_config4_shaped_fp16_gallery_with_tags(nq):
    """A 600 000 x 2048 fp16 gallery with make_distractor_ids labels: junk-rule tags against the oracle on the whole
    gallery (differences proven ties) and exactly on compute_dist's own distances; then camera tags where half the rows
    carry the queries' camera."""
    import torch
    import pps_b200
    from pps_b200 import synthetic
    dev = torch.device("cuda")
    ng, dim, k = 600000, 2048, 100
    qid, qcam, gid, gcam = synthetic.make_distractor_ids(3368, ng)
    qid, qcam = qid[:nq], qcam[:nq]
    q = synthetic.make_features_device(qid, dim, 750, 4.0, 7, dev, torch.float16)
    g = synthetic.make_features_device(gid, dim, 750, 4.0, 1000, dev, torch.float16)
    oracle = O.compute_dist(q.float().cpu().numpy(), g.float().cpu().numpy())
    own = pps_b200.compute_dist(q, g).cpu().numpy()
    idx = pps_b200.GalleryIndex(dim, dtype=torch.float16)
    idx.add(g, _junk_tags(gid, gcam))
    dist, index = idx.search(q, k, exclude_tags=_junk_tags(qid, qcam))
    dist, index = dist.cpu().numpy(), index.cpu().numpy()
    P.assert_topk_parity(index, dist, oracle, qid, qcam, gid, gcam, what="junk nq=%d" % nq)
    keep = ~((gid[None, :] == qid[:, None]) & (gcam[None, :] == qcam[:, None]))
    _assert_same((dist, index), _np_topk(own, keep, k))
    del idx
    # camera tags: every query has camera 0, and so has half the gallery
    rs = np.random.RandomState(5)
    cams = np.where(rs.rand(ng) < 0.5, 0, rs.randint(1, 6, ng)).astype(np.int64)
    qc = np.zeros(nq, np.int64)
    idx = pps_b200.GalleryIndex(dim, dtype=torch.float16)
    idx.add(g, torch.from_numpy(cams).cuda())
    dist, index = idx.search(q, k, exclude_tags=qc)
    dist, index = dist.cpu().numpy(), index.cpu().numpy()
    zq, zg = np.zeros(nq, np.int64), np.zeros(ng, np.int64)
    P.assert_topk_parity(index, dist, oracle, zq, qc, zg, cams, what="camera nq=%d" % nq)
    _assert_same((dist, index), _np_topk(own, cams[None, :] != qc[:, None], k))


@pytest.mark.gpu
def test_tag_errors():
    """Wrong tag length or dtype, mixed tagged and untagged adds, exclude tags on an untagged index, null tag pointers."""
    import torch
    import pps_b200
    from pps_b200 import _lib
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    g, q = d["g"], d["q"][:9]
    ng = len(g)
    idx = pps_b200.GalleryIndex(g.shape[1], dtype=torch.float32)
    for bad in (np.zeros(ng - 1, np.int64), np.zeros(ng, np.float32), np.zeros(ng, bool), np.zeros((ng, 1), np.int64),
                torch.zeros(ng, dtype=torch.float32), torch.zeros(ng, dtype=torch.bool), [0] * ng):
        with pytest.raises(RuntimeError):
            idx.add(g, bad)
    assert len(idx) == 0
    idx.add(g[:100], np.arange(100))
    with pytest.raises(RuntimeError):
        idx.add(g[100:])                                     # untagged rows into a tagged index
    idx.add(g[100:0])                                        # (an empty add is no add)
    for bad in (np.zeros(8, np.int64), np.zeros(9, np.float64), torch.zeros(9, dtype=torch.bool)):
        with pytest.raises(RuntimeError):
            idx.search(q, 5, exclude_tags=bad)
    plain = pps_b200.GalleryIndex(g.shape[1], dtype=torch.float32)
    plain.add(g[:100])
    with pytest.raises(RuntimeError):
        plain.add(g[100:], np.arange(ng - 100))              # tagged rows into an untagged index
    with pytest.raises(RuntimeError):
        plain.search(q, 5, exclude_tags=np.zeros(9, np.int64))
    assert len(idx) == len(plain) == 100
    # the C entry points: null tag pointers
    lib = _lib.load()
    qt = torch.from_numpy(q).cuda()
    gt = torch.from_numpy(g[:10]).cuda()
    keys = torch.empty((9, 5), dtype=torch.int64, device="cuda")
    assert lib.pps_index_search_excluding(idx._h, _lib.ptr(qt), 9, g.shape[1], None, 5, 0, 0, _lib.stream_ptr(),
                                          _lib.ptr(keys)) == _lib.PPS_ERR_INVALID_ARG
    assert lib.pps_index_add_tagged(idx._h, _lib.ptr(gt), 10, g.shape[1], None, _lib.stream_ptr()) == _lib.PPS_ERR_INVALID_ARG
    assert len(idx) == 100
