"""GalleryIndex grouped search: the nearest row of each of the k nearest groups (include/pps_b200.h part 2h,
pps_index_add_grouped / pps_index_search_groups and the kernel-level pps_topk_group_*).

The oracle is NumPy over compute_dist's own matrix (the search's distances, bit for bit): per query, the rows the search
may return ordered by the key (distance bits, row), the first row of each group, the first k."""
import os
import socket

import numpy as np
import pytest

from conftest import GOLDEN_CASES, GOLDEN_DIR

pytestmark = pytest.mark.gpu

KS = [1, 13, 100, 128]
ALL_ONES = np.uint64(0xffffffffffffffff)


def _hooks(prefix_blocks=0, tk_cap=0):
    from pps_b200 import _lib
    return _lib.index_prefix(prefix_blocks) | _lib.index_tkcap(tk_cap)


def _as(a, dtype_name):
    return np.ascontiguousarray(a, dtype=np.float16 if dtype_name == "fp16" else np.float32)


def _torch_dtype(dtype_name):
    import torch
    return torch.float16 if dtype_name == "fp16" else torch.float32


def _index(g, dtype_name, groups, tags=None, precision="f16x3"):
    import pps_b200
    idx = pps_b200.GalleryIndex(g.shape[1], dtype=_torch_dtype(dtype_name), precision=precision)
    idx.add(g, tags, groups)
    return idx


def _own_dist(q, g, dtype_name, precision="f16x3"):
    import torch
    import pps_b200
    if dtype_name == "fp16":
        return pps_b200.compute_dist(torch.from_numpy(q).cuda(), torch.from_numpy(g).cuda()).cpu().numpy()
    return np.asarray(pps_b200.compute_dist(q, g, precision=precision))


def _np_groups(dist, groups, k, keep=None):
    """per row of dist: the kept columns in (distance bits, column) order, the first of each group, the first k;
    (dist, index, group) padded with inf / -1 / -1"""
    nq = dist.shape[0]
    bits = np.ascontiguousarray(dist, np.float32).view(np.uint32)
    out_d = np.full((nq, k), np.inf, np.float32)
    out_i = np.full((nq, k), -1, np.int64)
    out_g = np.full((nq, k), -1, np.int64)
    for i in range(nq):
        cand = np.arange(dist.shape[1]) if keep is None else np.nonzero(keep[i])[0]
        order = cand[np.lexsort((cand, bits[i, cand]))]
        _, first = np.unique(groups[order], return_index=True)
        pick = order[np.sort(first)][:k]
        out_d[i, :len(pick)] = dist[i, pick]
        out_i[i, :len(pick)] = pick
        out_g[i, :len(pick)] = groups[pick]
    return out_d, out_i, out_g


def _search(idx, q, k, flags=0, exclude_tags=None):
    keys, groups, is_np = idx._search_group_keys(q, k, 0, flags, exclude_tags)
    d, i = idx._unpack(keys, is_np)
    return d, i, groups.cpu().numpy()


def _assert_same(got, want, msg=""):
    for a, b in zip(got[1:], want[1:]):
        np.testing.assert_array_equal(np.asarray(a), np.asarray(b), err_msg=msg)
    np.testing.assert_array_equal(np.asarray(got[0]).view(np.uint32), np.asarray(want[0]).view(np.uint32), err_msg=msg)


def _structures(ng, rs):
    """name -> [ng] int64 groups"""
    rows = np.arange(ng)
    return {
        "singletons": rows.astype(np.int64) * 3 - 1000,
        "one_group": np.full(ng, 42, np.int64),
        "tracklets16": (rows // 16).astype(np.int64),
        "tracklets256": (rows // 256).astype(np.int64),
        "shuffled": rs.randint(0, max(2, ng // 5), ng).astype(np.int64) - (1 << 40),
        "few_groups": rs.randint(0, 9, ng).astype(np.int64),
    }


def _queries(d, nq):
    sel = np.arange(nq) % (len(d["q"]) + len(d["g"]))
    return np.ascontiguousarray(np.concatenate([d["q"], d["g"]])[sel])


@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_group_structures_equal_numpy(golden, name, dtype_name):
    """Every group structure, k, batch width and schedule (default, and a 256-row prefix so that the chunks and the
    grouped merge cover the rest): NumPy's answer on the own distances bit for bit; singletons equal search."""
    d = golden(name)
    g = _as(d["g"], dtype_name)
    rs = np.random.RandomState(len(g))
    for sname, groups in _structures(len(g), rs).items():
        idx = _index(g, dtype_name, groups)
        for nq in (1, 33, 257):
            q = _as(_queries(d, nq), dtype_name)
            own = _own_dist(q, g, dtype_name)
            for k in KS:
                want = _np_groups(own, groups, k)
                for flags in (0, _hooks(prefix_blocks=1)):
                    got = _search(idx, q, k, flags)
                    assert got[0].dtype == np.float32 and got[1].dtype == np.int64 and got[1].shape == (nq, k)
                    _assert_same(got, want, "%s %s nq=%d k=%d flags=%x" % (name, sname, nq, k, flags))
                    if sname == "singletons":
                        plain = idx.search(q, k)
                        _assert_same((got[0], got[1]), plain)
                if sname == "one_group":
                    assert (want[1][:, 1:] == -1).all()
    # the public call, numpy in and CUDA in
    q = _as(d["q"], dtype_name)
    groups = (np.arange(len(g)) // 16).astype(np.int64)
    idx = _index(g, dtype_name, groups)
    want = _np_groups(_own_dist(q, g, dtype_name), groups, 13)
    _assert_same(idx.search_groups(q, 13), want)
    import torch
    got = idx.search_groups(torch.from_numpy(q).cuda(), 13)
    assert all(t.is_cuda for t in got)
    _assert_same(tuple(t.cpu().numpy() for t in got), want)


@pytest.mark.parametrize("precision", ["f16x3", "bf16x1", "bf16x3", "bf16x6", "fp16"])
def test_every_precision(precision):
    """Each tensor-core precision, tracklets of 8 rows, through the prefix and the chunks."""
    rs = np.random.RandomState(5)
    dtype_name = "fp16" if precision == "fp16" else "fp32"
    g = _as(rs.randn(3000, 160), dtype_name)
    q = _as(rs.randn(70, 160), dtype_name)
    groups = (np.arange(3000) // 8).astype(np.int64)
    prec = "f16x3" if precision == "fp16" else precision
    idx = _index(g, dtype_name, groups, precision=prec)
    own = _own_dist(q, g, dtype_name, prec)
    for k in (13, 100):
        want = _np_groups(own, groups, k)
        for flags in (0, _hooks(prefix_blocks=1), _hooks(prefix_blocks=2, tk_cap=600)):
            _assert_same(_search(idx, q, k, flags), want, "%s k=%d flags=%x" % (precision, k, flags))
        single = _index(g, dtype_name, np.arange(3000), precision=prec)
        _assert_same(_search(single, q, k, _hooks(prefix_blocks=1))[:2], single.search(q, k))


def _tracklet_gallery(n_tracks, length, dim, seed, contiguous=True):
    """near-duplicate tracklets: a centre per tracklet plus small noise per frame; (features, groups)"""
    rs = np.random.RandomState(seed)
    centres = rs.randn(n_tracks, dim).astype(np.float32)
    groups = np.repeat(np.arange(n_tracks, dtype=np.int64), length)
    if not contiguous:
        groups = groups[rs.permutation(len(groups))]
    g = centres[groups] + 0.05 * rs.randn(len(groups), dim).astype(np.float32)
    return g, groups, centres


@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_chunks_and_fallback_with_long_tracklets(dtype_name):
    """Near-duplicate tracklets of 64 frames: contiguous and shuffled, through the prefix + chunk schedule (which must
    not fall back), and with the rows ordered nearest-last and a 64-entry candidate buffer, where the fallback provably
    runs - exact either way."""
    for contiguous in (True, False):
        g, groups, centres = _tracklet_gallery(120, 64, 96, 4, contiguous)
        g = _as(g, dtype_name)
        rs = np.random.RandomState(9)
        q = _as(centres[rs.randint(0, 120, 20)] + 0.05 * rs.randn(20, 96), dtype_name)
        idx = _index(g, dtype_name, groups)
        own = _own_dist(q, g, dtype_name)
        for k in (1, 13, 100):
            want = _np_groups(own, groups, k)
            _assert_same(_search(idx, q, k, _hooks(prefix_blocks=2)), want, "contiguous=%s k=%d" % (contiguous, k))
            prefix, chunks, fallback = idx._group_stats()
            assert prefix >= 512 and not fallback
            if prefix < len(g):
                assert chunks > 0
    # nearest-last order: every chunk admits far more than 64 candidates per query
    g, groups, centres = _tracklet_gallery(60, 64, 96, 6)
    q = centres[:10] + 0.05 * np.random.RandomState(2).randn(10, 96).astype(np.float32)
    order = np.argsort(-_own_dist(q, g, "fp32").mean(0), kind="stable")
    g, groups = _as(g[order], dtype_name), groups[order]
    q = _as(q, dtype_name)
    idx = _index(g, dtype_name, groups)
    own = _own_dist(q, g, dtype_name)
    for k in (1, 13):
        _assert_same(_search(idx, q, k, _hooks(prefix_blocks=1, tk_cap=64)), _np_groups(own, groups, k))
        assert idx._group_stats()[2], "the fallback did not run"


@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_exclude_tags(dtype_name):
    """Camera tags with tracklet groups (a tracklet lies in one camera); and a group whose nearest row is excluded, so its
    next row represents it."""
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    g = _as(d["g"], dtype_name)
    ng = len(g)
    groups = (np.arange(ng) // 16).astype(np.int64)
    cams = (groups % 4).astype(np.int64)
    q = _as(_queries(d, 33), dtype_name)
    qcam = np.arange(33) % 5                                  # camera 4: excludes nothing
    own = _own_dist(q, g, dtype_name)
    idx = _index(g, dtype_name, groups, cams)
    keep = cams[None, :] != qcam[:, None]
    for k in KS:
        want = _np_groups(own, groups, k, keep)
        for flags in (0, _hooks(prefix_blocks=1)):
            _assert_same(_search(idx, q, k, flags, qcam), want, "k=%d flags=%x" % (k, flags))
    # per-row tags: each query excludes its nearest row only; that row's group is then represented by its next row
    nearest = np.argmin(own, axis=1)
    tags = np.arange(ng, dtype=np.int64)
    idx = _index(g, dtype_name, groups, tags)
    keep = tags[None, :] != nearest[:, None]
    for k in (1, 13):
        want = _np_groups(own, groups, k, keep)
        got = _search(idx, q, k, 0, nearest)
        _assert_same(got, want)
        assert (got[2][:, 0] == groups[nearest]).any() and not (got[1] == nearest[:, None]).any()


def test_non_finite_rows_order_last():
    """Gallery rows with inf / NaN elements (test_gpu_extreme_inputs' construction), each in a group of its own or
    sharing a group with finite rows: NaN and inf groups come after every finite one, NumPy's answer bit for bit."""
    from test_gpu_extreme_inputs import IG_SPECIAL, IQ_SPECIAL, NG, NQ, _features
    for dtype_name in ("fp32", "fp16"):
        g = _as(_features(NG, IG_SPECIAL, 21, integer=True), dtype_name)
        q = _as(_features(NQ, IQ_SPECIAL, 22, integer=True), dtype_name)
        groups = (np.arange(NG) // 4).astype(np.int64)
        own = _own_dist(q, g, dtype_name)
        idx = _index(g, dtype_name, groups)
        for k in (13, 100, 128):
            want = _np_groups(own, groups, k)
            for flags in (0, _hooks(prefix_blocks=1)):
                got = _search(idx, q, k, flags)
                _assert_same(got, want, "%s k=%d" % (dtype_name, k))
                fin = np.isfinite(got[0]) & (got[1] >= 0)
                assert (np.diff(fin.astype(np.int8), axis=1) <= 0).all()     # finite first, then non-finite, padding


@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_adds_in_pieces_and_remove(dtype_name):
    """Three grouped appends through two capacity doublings equal one add; remove then search_groups equals a fresh
    index of the remaining rows with their groups (and tags)."""
    import torch
    import pps_b200
    rs = np.random.RandomState(12)
    g = _as(rs.randn(2600, 96), dtype_name)
    q = _as(rs.randn(40, 96), dtype_name)
    groups = (np.arange(2600) // 10).astype(np.int64)
    tags = rs.randint(0, 4, 2600).astype(np.int64)
    qtags = rs.randint(0, 4, 40).astype(np.int64)
    parts = pps_b200.GalleryIndex(96, dtype=_torch_dtype(dtype_name))
    assert parts.add(g[:100], tags[:100], groups[:100]) == (0, 100)
    assert parts.add(torch.from_numpy(g[100:1600]).cuda(), torch.from_numpy(tags[100:1600]).cuda(),
                     torch.from_numpy(groups[100:1600]).cuda()) == (100, 1500)
    assert parts.add(g[1600:], tags[1600:], groups[1600:].astype(np.int32)) == (1600, 1000)
    own = _own_dist(q, g, dtype_name)
    for k in (13, 100):
        want = _np_groups(own, groups, k, tags[None, :] != qtags[:, None])
        for flags in (0, _hooks(prefix_blocks=1)):
            _assert_same(_search(parts, q, k, flags, qtags), want)
            _assert_same(_search(_index(g, dtype_name, groups, tags), q, k, flags, qtags), want)
    gone = np.concatenate([[0, 5, 999], np.arange(1200, 1650), rs.randint(0, 2600, 300)])
    assert parts._remove(gone, _lib_piece(97)) == len(np.unique(gone))
    left = np.setdiff1d(np.arange(2600), gone)
    fresh = _index(g[left], dtype_name, groups[left], tags[left])
    for k in (13, 100):
        for flags in (0, _hooks(prefix_blocks=1)):
            _assert_same(_search(parts, q, k, flags, qtags), _search(fresh, q, k, flags, qtags))
            _assert_same(_search(parts, q, k, flags), _search(fresh, q, k, flags))
        # search on the grouped index is unchanged by the groups
        np.testing.assert_array_equal(parts.search(q, k)[1], fresh.search(q, k)[1])
    # emptied, the index decides again
    assert parts.remove(np.arange(len(parts))) == len(left)
    parts.add(g[:50])
    with pytest.raises(RuntimeError):
        parts.search_groups(q, 5)


def _lib_piece(n):
    from pps_b200 import _lib
    return _lib.index_piece(n)


def _shards(ng, sizes):
    b = np.cumsum([0] + list(sizes))
    assert b[-1] == ng
    return [(int(b[i]), int(b[i + 1])) for i in range(len(sizes))]


@pytest.mark.parametrize("sizes", [(350, 350), (0, 500, 200), (100, 0, 300, 300)])
@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_sharded_indexes_equal_one_index(sizes, dtype_name):
    """2, 3 and 4 grouped indexes (one empty) stand for ranks, with tracklets that span shard boundaries and shuffled
    groups: the lists merged by merge_group_lists equal the single index bit for bit."""
    import pps_b200
    from pps_b200 import index as index_mod
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    g = _as(d["g"], dtype_name)
    ng = len(g)
    q = _as(_queries(d, 33), dtype_name)
    rs = np.random.RandomState(1)
    for groups in ((np.arange(ng) // 64).astype(np.int64), rs.randint(0, 40, ng).astype(np.int64)):
        one = _index(g, dtype_name, groups)
        for k in (13, 100):
            for flags in (0, _hooks(prefix_blocks=1)):
                keys, grps = [], []
                for r0, r1 in _shards(ng, sizes):
                    shard = pps_b200.GalleryIndex(g.shape[1], dtype=one.dtype)
                    shard.add(g[r0:r1], None, groups[r0:r1])
                    kk, gg, _ = shard._search_group_keys(q, k, r0, flags)
                    keys.append(kk)
                    grps.append(gg)
                mk, mg = index_mod.merge_group_lists(keys, grps, k)
                d_, i_ = one._unpack(mk, True)
                _assert_same((d_, i_, mg.cpu().numpy()), _search(one, q, k, flags))


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
    groups = (np.arange(len(d["g"])) // 64).astype(np.int64)
    idx = pps_b200.GalleryIndex(d["g"].shape[1], dtype=torch.float32, group=dist.group.WORLD)
    idx.add(d["g"][r0:r1], None, groups[r0:r1])
    dist_, index, grp = idx.search_groups(d["q"], 100)
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), dist=dist_, index=index, group=grp)
    dist.destroy_process_group()


def test_sharded_search_groups_over_nccl(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    world = 2
    mp.spawn(_nccl_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    d = dict(np.load(os.path.join(GOLDEN_DIR, "small_mid.npz")))
    groups = (np.arange(len(d["g"])) // 64).astype(np.int64)
    want = _np_groups(_own_dist(d["q"], d["g"], "fp32"), groups, 100)
    for r in range(world):
        o = dict(np.load(os.path.join(str(tmp_path), "rank%d.npz" % r)))
        _assert_same((o["dist"], o["index"], o["group"]), want)


def _np_state(keys, groups, k):
    """grouped state of (key, group) pairs: sorted by key, first per group, first k; ~0 / -1 padded"""
    keys = np.asarray(keys, np.uint64)
    ok = keys != ALL_ONES
    keys, groups = keys[ok], np.asarray(groups, np.int64)[ok]
    o = np.argsort(keys, kind="stable")
    _, first = np.unique(groups[o], return_index=True)
    pick = o[np.sort(first)][:k]
    out_k = np.full(k, ALL_ONES, np.uint64)
    out_g = np.full(k, -1, np.int64)
    out_k[:len(pick)] = keys[pick]
    out_g[:len(pick)] = groups[pick]
    return out_k, out_g


@pytest.mark.parametrize("k", [1, 13, 100, 128])
def test_group_update_kernel_equals_numpy(k):
    """pps_topk_group_update over two blocks (the second merges into the first's state), with and without tags: many
    duplicates of one group, and exact distance ties at the k-th place (resolved by the row)."""
    import torch
    from pps_b200 import _lib
    lib = _lib.load()
    rs = np.random.RandomState(k)
    nq, ldd = 37, 3100
    blocks = [(3000, 50), (2100, 3050)]
    state = {}
    for tagged in (False, True):
        keys_t = torch.empty((nq, k), dtype=torch.int64, device="cuda")
        grp_t = torch.full((nq, k), -1, dtype=torch.int64, device="cuda")
        _lib.check(lib.pps_topk_init(_lib.ptr(keys_t), nq, k, _lib.stream_ptr()), "pps_topk_init")
        state[tagged] = (keys_t, grp_t)
    want = {t: [(np.full(k, ALL_ONES, np.uint64), np.full(k, -1, np.int64)) for _ in range(nq)] for t in (False, True)}
    qtags = rs.randint(0, 4, nq).astype(np.int64)
    qt = torch.from_numpy(qtags).cuda()
    for ncols, col0 in blocks:
        dist = np.round(np.abs(rs.randn(nq, ldd)) * 8).astype(np.float32) / 8     # many exact ties
        groups = rs.randint(0, 3 * k + 5, ncols).astype(np.int64)
        groups[rs.rand(ncols) < 0.4] = 7                                          # one group with many rows
        gtags = rs.randint(0, 4, ncols).astype(np.int64)
        dt, gg, gt = (torch.from_numpy(x).cuda() for x in (dist, groups, gtags))
        for tagged in (False, True):
            keys_t, grp_t = state[tagged]
            _lib.check(lib.pps_topk_group_update(_lib.ptr(dt), ldd, nq, ncols, col0, _lib.ptr(gg),
                                                 _lib.ptr(gt if tagged else None), _lib.ptr(qt if tagged else None),
                                                 _lib.ptr(keys_t), _lib.ptr(grp_t), k, _lib.stream_ptr()),
                       "pps_topk_group_update")
            bits = dist[:, :ncols].view(np.uint32).astype(np.uint64)
            new = (bits << np.uint64(32)) | (np.arange(ncols, dtype=np.uint64) + np.uint64(col0))[None, :]
            for i in range(nq):
                keep = gtags != qtags[i] if tagged else np.ones(ncols, bool)
                sk, sg = want[tagged][i]
                want[tagged][i] = _np_state(np.concatenate([sk, new[i, keep]]), np.concatenate([sg, groups[keep]]), k)
            np.testing.assert_array_equal(keys_t.cpu().numpy().view(np.uint64), np.stack([w[0] for w in want[tagged]]))
            np.testing.assert_array_equal(grp_t.cpu().numpy(), np.stack([w[1] for w in want[tagged]]))


@pytest.mark.parametrize("k", [1, 13, 100, 128])
def test_group_merge_kernels_equal_numpy(k):
    """pps_topk_group_merge: state + candidates (more than the 2 048-entry buffer, candidates duplicating the state's
    groups, exact ties at the k-th place), the new bound, the reset count; a count above the capacity raises the flag.
    pps_topk_group_merge_lists: three lists whose groups overlap."""
    import torch
    from pps_b200 import _lib
    lib = _lib.load()
    rs = np.random.RandomState(100 + k)
    nq, cap, off, ng = 9, 5000, 1000, 60000
    g_groups = rs.randint(0, 2 * k + 3, ng).astype(np.int64)
    g_groups[::3] = 11
    st_k, st_g = [], []
    for i in range(nq):
        rows = rs.choice(ng, 3 * k, replace=False)
        d = rs.randint(100, 130, 3 * k).astype(np.uint64)
        sk, sg = _np_state((d << np.uint64(32)) | (rows + off).astype(np.uint64), g_groups[rows], k)
        st_k.append(sk)
        st_g.append(sg)
    st_k, st_g = np.stack(st_k), np.stack(st_g)
    cnt = np.array([0, 1, 17, 2047, 2048, 2049, 4999, 5000, 5003], np.uint32)
    cand = np.full((nq, cap), ALL_ONES, np.uint64)
    for i in range(nq):
        n = min(int(cnt[i]), cap)
        rows = rs.choice(ng, n, replace=False)
        d = rs.randint(90, 125, n).astype(np.uint64)
        cand[i, :n] = (d << np.uint64(32)) | (rows + off).astype(np.uint64)
    keys_t = torch.from_numpy(st_k.view(np.int64).copy()).cuda()
    grp_t = torch.from_numpy(st_g.copy()).cuda()
    cand_t = torch.from_numpy(cand.view(np.int64)).cuda()
    cnt_t = torch.from_numpy(cnt.view(np.int32).copy()).cuda()
    bound_t = torch.full((nq,), 12345, dtype=torch.int32, device="cuda")
    flag_t = torch.zeros(1, dtype=torch.int32, device="cuda")
    gg = torch.from_numpy(g_groups).cuda()
    _lib.check(lib.pps_topk_group_merge(_lib.ptr(keys_t), _lib.ptr(grp_t), nq, k, _lib.ptr(cand_t), cap, _lib.ptr(cnt_t),
                                        _lib.ptr(bound_t), _lib.ptr(gg), off, _lib.ptr(flag_t), _lib.stream_ptr()),
               "pps_topk_group_merge")
    got_k, got_g = keys_t.cpu().numpy().view(np.uint64), grp_t.cpu().numpy()
    bound = bound_t.cpu().numpy().view(np.uint32)
    for i in range(nq):
        if cnt[i] == 0:                                     # untouched
            np.testing.assert_array_equal(got_k[i], st_k[i])
            assert bound[i] == 12345
            continue
        n = min(int(cnt[i]), cap)
        rows = (cand[i, :n] & np.uint64(0xffffffff)).astype(np.int64) - off
        wk, wg = _np_state(np.concatenate([st_k[i], cand[i, :n]]), np.concatenate([st_g[i], g_groups[rows]]), k)
        np.testing.assert_array_equal(got_k[i], wk, err_msg="query %d" % i)
        np.testing.assert_array_equal(got_g[i], wg)
        assert bound[i] == (0xffffffff if wk[-1] == ALL_ONES else int(wk[-1] >> np.uint64(32)))
    assert (cnt_t.cpu().numpy() == 0).all() and int(flag_t.item()) == 1
    # no count above the capacity: no flag
    flag_t.zero_()
    cnt_t = torch.from_numpy(np.minimum(cnt, cap).view(np.int32).copy()).cuda()
    _lib.check(lib.pps_topk_group_merge(_lib.ptr(keys_t), _lib.ptr(grp_t), nq, k, _lib.ptr(cand_t), cap, _lib.ptr(cnt_t),
                                        _lib.ptr(bound_t), _lib.ptr(gg), off, _lib.ptr(flag_t), _lib.stream_ptr()),
               "pps_topk_group_merge")
    assert int(flag_t.item()) == 0
    # lists
    lists = 3
    lk = np.full((lists, nq, k), ALL_ONES, np.uint64)
    lg = np.full((lists, nq, k), -1, np.int64)
    for w in range(lists):
        for i in range(nq):
            n = rs.randint(0, 3 * k + 1)
            rows = rs.choice(ng, n, replace=False)
            d = rs.randint(100, 110, n).astype(np.uint64)
            lk[w, i], lg[w, i] = _np_state((d << np.uint64(32)) | rows.astype(np.uint64), g_groups[rows], k)
    ok_t = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    og_t = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    lk_t, lg_t = torch.from_numpy(lk.view(np.int64)).cuda(), torch.from_numpy(lg).cuda()
    _lib.check(lib.pps_topk_group_merge_lists(_lib.ptr(lk_t), _lib.ptr(lg_t), lists, nq, k, _lib.ptr(ok_t), _lib.ptr(og_t),
                                              _lib.stream_ptr()), "pps_topk_group_merge_lists")
    for i in range(nq):
        wk, wg = _np_state(lk[:, i].ravel(), lg[:, i].ravel(), k)
        np.testing.assert_array_equal(ok_t.cpu().numpy().view(np.uint64)[i], wk)
        np.testing.assert_array_equal(og_t.cpu().numpy()[i], wg)


@pytest.mark.parametrize("layout", ["contiguous", "shuffled"])
def test_config4_shaped_fp16_gallery_with_tracklets(layout):
    """A 600 000 x 2048 fp16 gallery in tracklets of 32 rows, stored contiguously or shuffled: search_groups on a query
    slice equals NumPy on compute_dist's own distances, without the fallback."""
    import torch
    import pps_b200
    from pps_b200 import synthetic
    dev = torch.device("cuda")
    ng, dim, k, nq = 600000, 2048, 100, 16
    qid, _, gid, _ = synthetic.make_distractor_ids(3368, ng)
    qid = qid[:nq]
    q = synthetic.make_features_device(qid, dim, 750, 4.0, 7, dev, torch.float16)
    g = synthetic.make_features_device(gid, dim, 750, 4.0, 1000, dev, torch.float16)
    groups = (np.arange(ng) // 32).astype(np.int64)
    if layout == "shuffled":
        groups = groups[np.random.RandomState(3).permutation(ng)]
    idx = pps_b200.GalleryIndex(dim, dtype=torch.float16)
    idx.add(g, None, torch.from_numpy(groups).cuda())
    own = pps_b200.compute_dist(q, g).cpu().numpy()
    got = idx.search_groups(q, k)
    got = tuple(t.cpu().numpy() for t in got)
    _assert_same(got, _np_groups(own, groups, k))
    assert not idx._group_stats()[2]


def test_group_errors():
    """Mixed grouped and ungrouped adds, search_groups on an ungrouped index, k out of range, groups of the wrong shape
    or dtype, null group pointers."""
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
            idx.add(g, None, bad)
    assert len(idx) == 0
    empty = idx.search_groups(q, 5)
    assert (empty[1] == -1).all() and (empty[2] == -1).all() and np.isinf(empty[0]).all()
    idx.add(g[:100], None, np.arange(100))
    with pytest.raises(RuntimeError):
        idx.add(g[100:])                                     # ungrouped rows into a grouped index
    with pytest.raises(RuntimeError):
        idx.add(g[100:], np.arange(ng - 100), np.arange(ng - 100))   # tagged rows into an untagged index
    for k in (0, 129, 1.5, -1):
        with pytest.raises(RuntimeError):
            idx.search_groups(q, k)
    with pytest.raises(RuntimeError):
        idx.search_groups(q, 5, exclude_tags=np.zeros(9, np.int64))  # not tagged
    plain = pps_b200.GalleryIndex(g.shape[1], dtype=torch.float32)
    plain.add(g[:100])
    with pytest.raises(RuntimeError):
        plain.add(g[100:], None, np.arange(ng - 100))        # grouped rows into an ungrouped index
    with pytest.raises(RuntimeError):
        plain.search_groups(q, 5)
    assert len(idx) == len(plain) == 100
    lib = _lib.load()
    qt = torch.from_numpy(q).cuda()
    gt = torch.from_numpy(g[:10]).cuda()
    keys = torch.empty((9, 5), dtype=torch.int64, device="cuda")
    assert lib.pps_index_add_grouped(idx._h, _lib.ptr(gt), 10, g.shape[1], None, None,
                                     _lib.stream_ptr()) == _lib.PPS_ERR_INVALID_ARG
    assert lib.pps_index_search_groups(idx._h, _lib.ptr(qt), 9, g.shape[1], None, 5, 0, 0, _lib.stream_ptr(),
                                       _lib.ptr(keys), None) == _lib.PPS_ERR_INVALID_ARG
    assert len(idx) == 100
