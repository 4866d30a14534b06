"""GalleryIndex.remove (include/pps_b200.h part 2h, pps_index_remove): rows deleted with np.delete's renumbering, the
resident gallery compacted on the device.

After a removal the index must answer every search, plain or excluding, exactly as a fresh index of the remaining rows
(in their order, with their tags) does: the same distance bits and the same indices."""
import os

import numpy as np
import pytest

from conftest import GOLDEN_CASES, GOLDEN_DIR


def _hooks(prefix_blocks=0):
    from pps_b200 import _lib
    return _lib.index_prefix(prefix_blocks)


def _piece(n):
    from pps_b200 import _lib
    return _lib.index_piece(n)


def _as(a, dtype_name):
    return np.ascontiguousarray(a, dtype=np.float16 if dtype_name == "fp16" else np.float32)


def _index(g, dtype_name, tags=None, precision="f16x3"):
    import torch
    import pps_b200
    idx = pps_b200.GalleryIndex(g.shape[1], dtype=torch.float16 if dtype_name == "fp16" else torch.float32,
                                precision=precision)
    idx.add(g, tags)
    return idx


def _search(idx, q, k, flags=0, exclude_tags=None):
    keys, is_np = idx._search_keys(q, k, 0, flags, exclude_tags)
    return idx._unpack(keys, is_np)


def _np(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def _assert_same(got, want, msg=""):
    np.testing.assert_array_equal(_np(got[1]), _np(want[1]), err_msg=msg)
    np.testing.assert_array_equal(_np(got[0]).view(np.uint32), _np(want[0]).view(np.uint32), err_msg=msg)


def _junk_tags(ids, cams):
    return (np.asarray(ids, np.int64) << 32) | np.asarray(cams, np.int64)


def _rank_eval_topk(q, g, k, qid=None, gid=None, qcam=None, gcam=None):
    """rank_eval's top-k; without labels, query ids that match no gallery row (the plain top-k)."""
    import torch
    import pps_b200
    nq, ng = q.shape[0], g.shape[0]
    if qid is None:
        qid, gid, qcam, gcam = np.full(nq, -1), np.arange(ng), np.zeros(nq, np.int64), np.zeros(ng, np.int64)
    res = pps_b200.rank_eval(torch.from_numpy(q).cuda(), torch.from_numpy(g).cuda(), qid, gid, qcam, gcam, topk=k)
    return res.topk_dist, res.topk_index.astype(np.int64)


def _patterns(ng, seed=0):
    rs = np.random.RandomState(seed)
    return {
        "first": np.array([0]),
        "last": np.array([ng - 1]),
        "run": np.arange(ng // 3, ng // 3 + ng // 4),
        "every_other": np.arange(0, ng, 2),
        "random10": rs.choice(ng, max(1, ng // 10), replace=False),
        "unsorted_dups": np.concatenate([rs.randint(0, ng, ng // 5), [ng - 1, 0, ng // 2, ng // 2]])[::-1].copy(),
        "all": rs.permutation(ng),
    }


def _queries(d, nq):
    pool = np.concatenate([d["q"], d["g"]])
    return np.ascontiguousarray(pool[np.arange(nq) % len(pool)])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_remove_patterns_equal_fresh_index(golden, name, dtype_name):
    """Every removal pattern, moved in one piece and in pieces of 7 rows: plain searches with the default schedule and
    with a 256-row prefix equal a fresh index of np.delete(g, R) and rank_eval's top-k on the kept rows."""
    d = golden(name)
    g = _as(d["g"], dtype_name)
    ng = g.shape[0]
    cases = [(nq, k, _as(_queries(d, nq), dtype_name)) for nq in (7, 257) for k in (13, 100)]
    for pat, rows in _patterns(ng).items():
        kept = np.delete(g, rows, axis=0)
        fresh = _index(kept, dtype_name)
        wants = [_search(fresh, q, k) for _, k, q in cases]
        for (nq, k, q), want in zip(cases, wants):
            if len(kept):
                _assert_same(want, _rank_eval_topk(q, kept, k), "%s %s nq=%d k=%d rank_eval" % (name, pat, nq, k))
            else:
                assert (want[1] == -1).all() and np.isinf(want[0]).all()
        for rm_flags in (0, _piece(7)):
            idx = _index(g, dtype_name)
            assert idx._remove(rows, rm_flags) == len(np.unique(rows))
            assert len(idx) == len(kept) == ng - len(np.unique(rows))
            for (nq, k, q), want in zip(cases, wants):
                for flags in (0, _hooks(1)):
                    _assert_same(_search(idx, q, k, flags), want, "%s %s nq=%d k=%d piece=%x flags=%x"
                                 % (name, pat, nq, k, rm_flags, flags))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f16x3", "bf16x1", "bf16x3", "bf16x6", "fp16"])
def test_remove_every_precision(precision):
    """One to three planes and the scaled norm layout (norms, then inverse scales): a random tenth and a block removed
    in pieces of 5 rows, then the search equals a fresh index's."""
    rs = np.random.RandomState(21)
    dtype_name = "fp16" if precision == "fp16" else "fp32"
    g = _as(rs.randn(3000, 200), dtype_name)
    q = _as(rs.randn(40, 200), dtype_name)
    prec = "f16x3" if precision == "fp16" else precision
    idx = _index(g, dtype_name, precision=prec)
    live = np.arange(3000)
    for rows in (rs.choice(3000, 300, replace=False), np.arange(100, 1100)):
        assert idx._remove(rows, _piece(5)) == len(rows)
        live = np.delete(live, rows)
        fresh = _index(g[live], dtype_name, precision=prec)
        for flags in (0, _hooks(1)):
            for k in (1, 100):
                _assert_same(_search(idx, q, k, flags), _search(fresh, q, k, flags), "%s k=%d flags=%x" % (precision, k, flags))


@pytest.mark.gpu
@pytest.mark.parametrize("tagged", [False, True])
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_add_remove_sequence_through_capacity_doublings(dtype_name, tagged):
    """add, remove, add, remove, add, remove (capacities 1 024 -> 2 048 -> 4 096), moves in pieces of 3 rows: the
    final index equals a fresh index of the final row list."""
    import torch
    rs = np.random.RandomState(5)
    g_all = _as(rs.randn(4000, 96), dtype_name)
    t_all = rs.randint(0, 4, 4000).astype(np.int64)
    q = _as(rs.randn(33, 96), dtype_name)
    qt = rs.randint(0, 5, 33).astype(np.int64)
    idx = _index(g_all[:0], dtype_name)
    live = np.zeros(0, np.int64)
    nxt = 0
    for n_add, n_rm in ((700, 90), (1500, 400), (1600, 1200)):
        rows = np.arange(nxt, nxt + n_add)
        idx.add(torch.from_numpy(g_all[rows]).cuda(), t_all[rows] if tagged else None)
        live = np.concatenate([live, rows])
        nxt += n_add
        rm = rs.choice(len(live), n_rm, replace=False)
        assert idx._remove(torch.from_numpy(rm).cuda(), _piece(3)) == n_rm
        live = np.delete(live, rm)
        assert len(idx) == len(live)
    fresh = _index(g_all[live], dtype_name, t_all[live] if tagged else None)
    for flags in (0, _hooks(1)):
        _assert_same(_search(idx, q, 100, flags), _search(fresh, q, 100, flags))
        if tagged:
            _assert_same(_search(idx, q, 100, flags, qt), _search(fresh, q, 100, flags, qt))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_tags_move_with_their_rows(golden, name, dtype_name):
    """Junk-rule tags: after removing a random tenth (pieces of 11 rows) and an unsorted list with duplicates, excluding
    searches equal the fresh tagged index and rank_eval's junk-filtered top-k on the kept rows; camera tags likewise
    equal the fresh index."""
    d = golden(name)
    g = _as(d["g"], dtype_name)
    ng = g.shape[0]
    pats = _patterns(ng, seed=3)
    live = np.arange(ng)
    idx = _index(g, dtype_name, _junk_tags(d["gid"], d["gcam"]))
    cam = _index(g, dtype_name, d["gcam"])
    for rows in (pats["random10"], pats["unsorted_dups"] % (ng - len(pats["random10"]))):
        assert idx._remove(rows, _piece(11)) == len(np.unique(rows))
        assert cam._remove(rows) == len(np.unique(rows))
        live = np.delete(live, rows)
        gk, gid, gcam = g[live], d["gid"][live], d["gcam"][live]
        fresh = _index(gk, dtype_name, _junk_tags(gid, gcam))
        fresh_cam = _index(gk, dtype_name, gcam)
        for nq in (7, 257):
            sel = np.arange(nq) % len(d["q"])
            q, qid, qcam = _as(d["q"][sel], dtype_name), d["qid"][sel], d["qcam"][sel]
            for k in (13, 100):
                want = _search(fresh, q, k, 0, _junk_tags(qid, qcam))
                _assert_same(want, _rank_eval_topk(q, gk, k, qid, gid, qcam, gcam), "%s nq=%d k=%d" % (name, nq, k))
                for flags in (0, _hooks(1)):
                    msg = "%s nq=%d k=%d flags=%x" % (name, nq, k, flags)
                    _assert_same(_search(idx, q, k, flags, _junk_tags(qid, qcam)), want, msg)
                    _assert_same(_search(cam, q, k, flags, qcam), _search(fresh_cam, q, k, flags, qcam), msg + " cam")
                    _assert_same(_search(idx, q, k, flags), _search(fresh, q, k, flags), msg + " plain")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_emptied_index_behaves_like_a_new_one(dtype_name):
    """Removing every row leaves an empty index (searches pad with -1 / inf) whose next non-empty add decides again
    whether it is tagged: a tagged index takes untagged rows and the other way round."""
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    g, q = _as(d["g"], dtype_name), _as(d["q"][:9], dtype_name)
    ng = len(g)
    tags = d["gcam"]
    for first_tags, second_tags in ((tags, None), (None, tags)):
        idx = _index(g, dtype_name, first_tags)
        assert idx.remove(np.arange(ng)[::-1].copy()) == ng and len(idx) == 0
        dist, index = idx.search(q, 5)
        assert (index == -1).all() and np.isinf(dist).all()
        idx.add(g[:300], None if second_tags is None else second_tags[:300])
        fresh = _index(g[:300], dtype_name, None if second_tags is None else second_tags[:300])
        _assert_same(idx.search(q, 50), fresh.search(q, 50))
        if second_tags is None:
            with pytest.raises(RuntimeError):
                idx.search(q, 5, exclude_tags=d["qcam"][:9])
        else:
            _assert_same(idx.search(q, 50, exclude_tags=d["qcam"][:9]), fresh.search(q, 50, exclude_tags=d["qcam"][:9]))


@pytest.mark.gpu
def test_remove_errors_leave_the_index_unchanged():
    """Rows -1 or size refuse the whole call (nothing moves, not even the valid rows listed with them); float, 2-D or
    list input raises; the C call refuses a null pointer with n > 0, unknown flags and rows of an empty index, and does
    nothing for n = 0."""
    import torch
    import pps_b200
    from pps_b200 import _lib
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    g, q = d["g"], d["q"][:9]
    ng = len(g)
    idx = _index(g, "fp32", d["gcam"])
    before = _search(idx, q, 100), _search(idx, q, 100, _hooks(1), d["qcam"][:9])
    for bad in (np.array([3, -1, 5]), np.array([0, ng]), torch.tensor([ng + 7], device="cuda"),
                np.zeros(3, np.float32), torch.zeros(3), np.zeros((2, 2), np.int64), torch.zeros(2, 2, dtype=torch.int64),
                np.zeros(2, bool), [0, 1]):
        with pytest.raises(RuntimeError):
            idx.remove(bad)
        assert len(idx) == ng
    _assert_same(_search(idx, q, 100), before[0])
    _assert_same(_search(idx, q, 100, _hooks(1), d["qcam"][:9]), before[1])
    lib = _lib.load()
    rows = torch.tensor([1, 2], dtype=torch.int64, device="cuda")
    n_removed = _lib.C.c_longlong(-5)
    assert lib.pps_index_remove(idx._h, None, 2, 0, _lib.stream_ptr(), _lib.C.byref(n_removed)) == _lib.PPS_ERR_INVALID_ARG
    assert lib.pps_index_remove(idx._h, _lib.ptr(rows), -1, 0, _lib.stream_ptr(), None) == _lib.PPS_ERR_INVALID_ARG
    assert lib.pps_index_remove(idx._h, _lib.ptr(rows), 2, 1, _lib.stream_ptr(), None) == _lib.PPS_ERR_INVALID_ARG
    assert lib.pps_index_remove(None, _lib.ptr(rows), 2, 0, _lib.stream_ptr(), None) == _lib.PPS_ERR_INVALID_ARG
    assert lib.pps_index_remove(idx._h, None, 0, 0, _lib.stream_ptr(), _lib.C.byref(n_removed)) == _lib.PPS_OK
    assert n_removed.value == 0
    assert idx.remove(np.zeros(0, np.int64)) == 0 and idx.remove(torch.zeros(0, dtype=torch.int32)) == 0
    assert len(idx) == ng
    _assert_same(_search(idx, q, 100), before[0])
    empty = pps_b200.GalleryIndex(g.shape[1], dtype=torch.float32)
    with pytest.raises(RuntimeError):
        empty.remove(np.array([0]))
    assert empty.remove(np.zeros(0, np.int64)) == 0
    # int32 / uint8 rows work, and the count is of distinct rows
    assert idx.remove(np.array([4, 4, 2], np.int32)) == 2 and idx.remove(torch.tensor([0, 0], dtype=torch.uint8)) == 1
    assert len(idx) == ng - 3
    _assert_same(_search(idx, q, 100), _search(_index(np.delete(g, [0, 2, 4], axis=0), "fp32"), q, 100))


@pytest.mark.gpu
@pytest.mark.parametrize("sizes", [(350, 350), (0, 500, 200), (100, 0, 300, 300)])
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_removal_on_one_shard_equals_one_index(sizes, dtype_name):
    """Indexes standing for ranks; the largest shard removes a random third of its local rows (pieces of 9 rows).  The
    shards' keys, with offsets from the new shard sizes, merge to one index of the concatenated kept rows."""
    from pps_b200 import evaluator
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    g = _as(d["g"], dtype_name)
    q = _as(_queries(d, 33), dtype_name)
    bounds = np.cumsum([0] + list(sizes))
    shards, kept = [], []
    victim = int(np.argmax(sizes))
    rs = np.random.RandomState(len(sizes))
    for i in range(len(sizes)):
        rows = g[bounds[i]:bounds[i + 1]]
        shard = _index(rows, dtype_name)
        if i == victim:
            rm = rs.choice(len(rows), len(rows) // 3, replace=False)
            assert shard._remove(rm, _piece(9)) == len(rm)
            rows = np.delete(rows, rm, axis=0)
        shards.append(shard)
        kept.append(rows)
    one = _index(np.concatenate(kept), dtype_name)
    for k in (13, 100):
        for flags in (0, _hooks(1)):
            keys, offset = [], 0
            for shard in shards:
                keys.append(shard._search_keys(q, k, offset, flags)[0])
                offset += len(shard)
            got = one._unpack(evaluator.merge_key_lists(keys, k), True)
            _assert_same(got, _search(one, q, k, flags), "k=%d flags=%x" % (k, flags))


@pytest.mark.gpu
@pytest.mark.parametrize("nq", [1, 64])
def test_config4_shaped_fp16_gallery_removal(nq):
    """600 000 x 2048 fp16 rows (the default piece size, several pieces; the default search schedule): a random 1 %
    removed, then a 100 000-row block - after each, the search equals a fresh index of the kept rows."""
    import torch
    import pps_b200
    from pps_b200 import synthetic
    dev = torch.device("cuda")
    ng, dim, k = 600000, 2048, 100
    qid, _, gid, _ = synthetic.make_distractor_ids(3368, ng)
    q = synthetic.make_features_device(qid[:nq], dim, 750, 4.0, 7, dev, torch.float16)
    g = synthetic.make_features_device(gid, dim, 750, 4.0, 1000, dev, torch.float16)
    idx = pps_b200.GalleryIndex(dim, dtype=torch.float16)
    idx.add(g)
    rs = np.random.RandomState(nq)
    live = np.arange(ng)
    for rows in (rs.choice(ng, ng // 100, replace=False), np.arange(200000, 300000)):
        assert idx.remove(torch.from_numpy(rows).to(dev)) == len(rows)
        live = np.delete(live, rows)
        fresh = pps_b200.GalleryIndex(dim, dtype=torch.float16)
        fresh.add(g[torch.from_numpy(live).to(dev)])
        _assert_same(idx.search(q, k), fresh.search(q, k))
        del fresh
