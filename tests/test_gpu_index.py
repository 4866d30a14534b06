"""GalleryIndex (resident gallery, top-k search for unlabelled queries; include/pps_b200.h part 2h).

Its answer is rank_eval's top-k when no gallery item shares a query's id: the same distances (pps_dist_tc's, bit for bit,
also from the swapped-operand search kernel) in the same order (distance, then gallery index)."""
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


def _queries(d, nq):
    """nq query rows: the fixture's queries, then its gallery rows (exact self matches: distances that clamp to 0)."""
    pool = np.concatenate([d["q"], d["g"]])
    return np.ascontiguousarray(pool[np.arange(nq) % len(pool)])


def _rank_eval_topk(q, g, k):
    """rank_eval's top-k with query ids that match no gallery id (so nothing is junk): the plain top-k."""
    import torch
    import pps_b200
    nq, ng = q.shape[0], g.shape[0]
    res = pps_b200.rank_eval(torch.from_numpy(q).cuda(), torch.from_numpy(g).cuda(), np.full(nq, -1), np.arange(ng),
                             np.zeros(nq, np.int64), np.zeros(ng, np.int64), topk=k)
    return res.topk_dist, res.topk_index.astype(np.int64)


def _search(idx, q, k, flags=0):
    keys, is_np = idx._search_keys(q, k, 0, flags)
    return idx._unpack(keys, is_np)


def _index(g, dtype_name, precision="f16x3"):
    import torch
    import pps_b200
    idx = pps_b200.GalleryIndex(g.shape[1], dtype=torch.float16 if dtype_name == "fp16" else torch.float32,
                                precision=precision)
    idx.add(g)
    return idx


def _as(a, dtype_name):
    return np.ascontiguousarray(a, dtype=np.float16 if dtype_name == "fp16" else np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_search_equals_rank_eval_topk(golden, name, dtype_name):
    """Every batch width and k, with the default schedule (galleries this small are one materialised block) and with a
    256-row prefix (the swapped-operand kernel + candidate merges cover the rest): bit for bit rank_eval's top-k."""
    d = golden(name)
    g = _as(d["g"], dtype_name)
    idx = _index(g, dtype_name)
    assert len(idx) == g.shape[0]
    for nq in NQS:
        q = _as(_queries(d, nq), dtype_name)
        for k in KS:
            want_d, want_i = _rank_eval_topk(q, g, k)
            for flags in (0, _hooks(prefix_blocks=1)):
                got_d, got_i = _search(idx, q, k, flags)
                assert got_d.dtype == np.float32 and got_i.dtype == np.int64 and got_i.shape == (nq, k)
                np.testing.assert_array_equal(got_i, want_i, err_msg="%s nq=%d k=%d flags=%x" % (name, nq, k, flags))
                np.testing.assert_array_equal(got_d, want_d, err_msg="%s nq=%d k=%d flags=%x" % (name, nq, k, flags))
    # the public call: numpy in, numpy out
    got_d, got_i = idx.search(_as(d["q"], dtype_name), 13)
    want_d, want_i = _rank_eval_topk(_as(d["q"], dtype_name), g, 13)
    np.testing.assert_array_equal(got_i, want_i)
    np.testing.assert_array_equal(got_d, want_d)


@pytest.mark.gpu
def test_short_gallery_pads_and_empty_index():
    import torch
    import pps_b200
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    g, q = d["g"][:50], d["q"][:9]
    idx = _index(g, "fp32")
    dist, index = idx.search(q, 100)
    want_d, want_i = _rank_eval_topk(q, g, 50)
    np.testing.assert_array_equal(index[:, :50], want_i)
    np.testing.assert_array_equal(dist[:, :50], want_d)
    assert (index[:, 50:] == -1).all() and np.isinf(dist[:, 50:]).all()
    # CUDA in -> CUDA out on the index's device
    dist_t, index_t = idx.search(torch.from_numpy(q).cuda(), 100)
    assert dist_t.is_cuda and index_t.dtype == torch.int64
    np.testing.assert_array_equal(index_t.cpu().numpy(), index)
    empty = pps_b200.GalleryIndex(g.shape[1], dtype=torch.float32)
    assert len(empty) == 0
    dist, index = empty.search(q, 5)
    assert (index == -1).all() and np.isinf(dist).all()
    for bad in (lambda: idx.search(q, 0), lambda: idx.search(q, 129), lambda: idx.search(q.astype(np.float16), 5),
                lambda: idx.search(q[:, :-1], 5), lambda: idx.add(g[:, :-1]), lambda: idx.search(q[0], 5)):
        with pytest.raises(RuntimeError):
            bad()
    with pytest.raises(RuntimeError):
        pps_b200.GalleryIndex(g.shape[1], dtype=torch.float32, precision="fp32")


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f16x3", "bf16x1", "bf16x3", "bf16x6", "fp16"])
@pytest.mark.parametrize("nq", [20, 50, 100, 200, 300])
def test_search_kernel_distances_equal_compute_dist(precision, nq):
    """pps_search_topk_tc with an all-ones bound and room for every row: each (query, row) is a candidate whose distance
    has the bits of compute_dist's value there (the operand swap keeps the products and their order)."""
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
    g[5] = q[3]                                                  # an exact match: distance 0 (or its rounding)
    prec = _lib.PREC_F16X1 if f16 else _lib.PRECISIONS[precision]
    planes = _lib.PLANES_FOR[prec]
    scaled = prec == _lib.PREC_F16X3
    sq = evaluator.SplitOperand(torch.from_numpy(q).cuda(), planes, scaled)
    sg = evaluator.SplitOperand(torch.from_numpy(g).cuda(), planes, scaled)
    cap = ng + 3
    bound = torch.full((nq,), -1, dtype=torch.int32, device="cuda")
    cnt = torch.zeros(nq, dtype=torch.int32, device="cuda")
    cand = torch.zeros((nq, cap), dtype=torch.int64, device="cuda")
    _lib.check(lib.pps_search_topk_tc(_lib.ptr(sg.planes), _lib.ptr(sg.sqnorm), ng, planes, 0, _lib.ptr(sq.planes),
                                      _lib.ptr(sq.sqnorm), nq, planes, 0, dim, prec, 0, col0, _lib.ptr(bound), _lib.ptr(cnt),
                                      _lib.ptr(cand), cap, _lib.stream_ptr()), "pps_search_topk_tc")
    np.testing.assert_array_equal(cnt.cpu().numpy(), np.full(nq, ng))
    keys = cand.cpu().numpy()[:, :ng].view(np.uint64)
    idx = (keys & np.uint64(0xffffffff)).astype(np.int64) - col0
    order = np.argsort(idx, axis=1)
    idx = np.take_along_axis(idx, order, axis=1)
    bits = np.take_along_axis((keys >> np.uint64(32)).astype(np.uint32), order, axis=1)
    np.testing.assert_array_equal(idx, np.broadcast_to(np.arange(ng), (nq, ng)))
    if f16:      # fp16 tensors take the single-plane fp16 product (numpy input would be cast to float32)
        want = pps_b200.compute_dist(torch.from_numpy(q).cuda(), torch.from_numpy(g).cuda()).cpu().numpy()
    else:
        want = pps_b200.compute_dist(q, g, precision=precision)
    np.testing.assert_array_equal(bits, np.ascontiguousarray(want).view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_adding_in_pieces_equals_one_add(dtype_name):
    """Three uneven appends through two capacity doublings (the first capacity is 1 024 rows) give the same search."""
    import torch
    import pps_b200
    rs = np.random.RandomState(11)
    g = _as(rs.randn(2600, 96), dtype_name)
    q = _as(rs.randn(40, 96), dtype_name)
    one = _index(g, dtype_name)
    parts = pps_b200.GalleryIndex(96, dtype=torch.float16 if dtype_name == "fp16" else torch.float32)
    assert parts.add(g[:100]) == (0, 100)
    assert parts.add(torch.from_numpy(g[100:1600]).cuda()) == (100, 1500)
    assert parts.add(g[1600:]) == (1600, 1000)
    assert len(parts) == len(one) == 2600
    for flags in (0, _hooks(prefix_blocks=1)):
        a, b = _search(one, q, 100, flags), _search(parts, q, 100, flags)
        np.testing.assert_array_equal(a[1], b[1])
        np.testing.assert_array_equal(a[0], b[0])
    want_d, want_i = _rank_eval_topk(q, g, 100)
    np.testing.assert_array_equal(a[1], want_i)
    np.testing.assert_array_equal(a[0], want_d)


@pytest.mark.gpu
@pytest.mark.parametrize("nq", [1, 64])
def test_config4_shaped_fp16_gallery(nq):
    """A 600 000 x 2048 fp16 gallery (configs[4]'s arithmetic, tests/test_gpu_large.py's features): the default schedule
    (32 768-row prefix, then swapped-operand chunks) against the oracle on the whole gallery, differences proven ties."""
    import torch
    import pps_b200
    from pps_b200 import synthetic
    dev = torch.device("cuda")
    ng, dim, k = 600000, 2048, 100
    qid, _, gid, gcam = synthetic.make_distractor_ids(3368, ng)
    q = synthetic.make_features_device(qid[:nq], dim, 750, 4.0, 7, dev, torch.float16)
    g = synthetic.make_features_device(gid, dim, 750, 4.0, 1000, dev, torch.float16)
    idx = pps_b200.GalleryIndex(dim, dtype=torch.float16)
    idx.add(g)
    dist, index = idx.search(q, k)
    dist, index = dist.cpu().numpy(), index.cpu().numpy()
    oracle = O.compute_dist(q.float().cpu().numpy(), g.float().cpu().numpy())
    none = np.full(nq, -1)
    P.assert_topk_parity(index, dist, oracle, none, np.zeros(nq, np.int64), gid, gcam, what="search nq=%d" % nq)
    # and the GPU's own distances, exactly
    own = pps_b200.compute_dist(q, g).cpu().numpy()
    np.testing.assert_array_equal(dist, np.take_along_axis(own, index, axis=1))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_candidate_overflow_falls_back(dtype_name):
    """Rows sorted so that the nearest come last, a 256-row prefix and a 4-entry candidate buffer: every chunk overflows
    its buffer and the search repeats with materialised blocks - still rank_eval's answer."""
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    q = _as(d["q"][:7], dtype_name)
    d0 = O.compute_dist(d["q"][:7].astype(np.float32), d["g"].astype(np.float32)).mean(0)
    g = _as(d["g"][np.argsort(-d0, kind="stable")], dtype_name)
    idx = _index(g, dtype_name)
    for k in (1, 13, 100):
        want_d, want_i = _rank_eval_topk(q, g, k)
        got_d, got_i = _search(idx, q, k, _hooks(prefix_blocks=1, tk_cap=4))
        np.testing.assert_array_equal(got_i, want_i)
        np.testing.assert_array_equal(got_d, want_d)


def _shards(ng, sizes):
    b = np.cumsum([0] + list(sizes))
    assert b[-1] == ng
    return [(int(b[i]), int(b[i + 1])) for i in range(len(sizes))]


@pytest.mark.gpu
@pytest.mark.parametrize("sizes", [(350, 350), (0, 500, 200), (100, 0, 300, 300)])
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_sharded_indexes_equal_one_index(sizes, dtype_name):
    """2, 3 and 4 indexes (one empty) stand for ranks: each searches with its shard's offset, the keys are exchanged by
    hand and merged as merge_topk_keys merges them - the single index's answer bit for bit."""
    import pps_b200
    from pps_b200 import evaluator
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    g = _as(d["g"], dtype_name)
    q = _as(_queries(d, 33), dtype_name)
    one = _index(g, dtype_name)
    for k in (13, 100):
        for flags in (0, _hooks(prefix_blocks=1)):
            keys = []
            for r0, r1 in _shards(g.shape[0], sizes):
                shard = pps_b200.GalleryIndex(g.shape[1], dtype=one.dtype)
                shard.add(g[r0:r1])
                keys.append(shard._search_keys(q, k, r0, flags)[0])
            got = one._unpack(evaluator.merge_key_lists(keys, k), True)
            want = _search(one, q, k, flags)
            np.testing.assert_array_equal(got[1], want[1])
            np.testing.assert_array_equal(got[0], want[0])


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
    idx.add(d["g"][r0:r1])
    dist_, index = idx.search(d["q"], 100)
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), dist=dist_, index=index)
    dist.destroy_process_group()


@pytest.mark.gpu
def test_sharded_search_over_nccl(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    world = 2
    mp.spawn(_nccl_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    want_d, want_i = _index(d["g"], "fp32").search(d["q"], 100)
    for r in range(world):
        o = dict(np.load(os.path.join(str(tmp_path), "rank%d.npz" % r)))
        np.testing.assert_array_equal(o["index"], want_i)
        np.testing.assert_array_equal(o["dist"], want_d)


def test_index_refuses_to_run_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    import pps_b200
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pps_b200.GalleryIndex(64)
