"""Resident gallery index: the k nearest gallery rows of unlabelled query features (person retrieval).

The gallery is split into tensor-core operand planes once, when rows are added (C ABI part 2h, ``pps_index_*``); a search
splits only the queries and streams the resident planes, the gallery as the 256-row side of every MMA
(``pps_search_topk_tc``).  Distances and order are those of ``compute_dist`` / ``rank_eval``'s top-k: Euclidean, smallest
first, ties by gallery index.

Rows may carry one int64 tag each (``add(feats, tags)``), and a search may leave out, for every query, the rows whose
tag equals the query's exclude tag (``search(q, k, exclude_tags)``); the test runs inside the search kernels.  Two
encodings cover person retrieval:

- cross-camera search: ``tags = gallery cameras``, ``exclude_tags = query cameras``;
- the evaluation protocol's junk rule (same id and same camera): ``tag = (id << 32) | camera`` for ids in int32 and
  cameras in [0, 2^32), on both sides.  The result then equals ``rank_eval(..., topk=k)`` bit for bit.

Rows may also carry one int64 group each (``add(feats, groups=...)``: a tracklet or an identity), and
``search_groups(q, k)`` returns the nearest row of each of the k nearest groups, so that the frames of one tracklet
take one place of the result instead of all of them.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .evaluator import _prec_code, merge_topk_keys


class GalleryIndex:
    """A gallery kept on one GPU (or sharded over the ranks of a ``torch.distributed`` group) for top-k search.

    ``idx = GalleryIndex(dim, dtype=torch.float16)``; ``row0, rows = idx.add(feats)`` appends rows (CUDA tensor or numpy
    [n, dim]) and returns their local row range; ``dist, index = idx.search(q, k)`` gives [nq, k] float32 distances and
    int64 gallery indices (-1 and inf past the end of a gallery with fewer than k rows).  numpy in gives numpy out, CUDA in
    gives CUDA tensors on the index's device.  float16 rows use the exact single-plane fp16 product; float32 rows the
    split ``precision`` (default ``f16x3``, as compute_dist).

    With ``group`` every rank adds its own rows and ``search`` is collective: one all-gather of the shard sizes (a shard's
    indices start after the rows of the ranks before it) and one of the keys; every rank gets the result of one index
    holding the concatenated shards.

    ``add(feats, tags)`` gives every row an integer tag (numpy or torch, [n], converted to int64 on the index's device);
    the first non-empty add decides whether the index is tagged, and a later add of the other kind raises.
    ``search(q, k, exclude_tags)`` ([nq] integers) leaves row r out of query i's result when
    ``tags[r] == exclude_tags[i]`` and pads with -1 / inf when fewer than k rows remain; it needs a tagged index (an
    empty one answers with padding).  Without ``exclude_tags`` the tags are ignored.  Sharded: every rank passes the
    same exclude tags and its own rows' tags.

    ``remove(rows)`` deletes local rows (integer numpy or torch, [n], any order, duplicates allowed) as ``np.delete``
    does: every later row moves down by the number of removed rows before it, ``len`` shrinks by the number of distinct
    rows removed (the return value), and every later search equals that of a fresh index given the remaining rows in
    their order (with their tags), bit for bit.  Apply the same deletion to the rows' metadata.  A row outside
    ``[0, len)`` raises and leaves the index unchanged.  The memory is kept for later adds; an index emptied by
    ``remove`` decides again at its next non-empty add whether it is tagged.  Sharded: ``remove`` is local, not
    collective; a rank removes its own rows, and the next ``search`` gathers the new shard sizes.

    ``lims, dist, index = range_search(q, radius, exclude_tags=None)`` returns every row within ``radius`` of each query
    (FAISS's ``range_search`` layout): row r is a result of query i when ``d(i, r) <= radius[i]``, d being ``search``'s
    distance bit for bit.  ``radius`` is a number or [nq] floats or integers (numpy or torch), converted to float32; the
    comparison is IEEE (a negative or NaN radius selects nothing, ``inf`` every row).  ``lims`` is [nq + 1] int64 and
    query i's results are ``dist[lims[i]:lims[i + 1]]`` (float32) and ``index[lims[i]:lims[i + 1]]`` (int64) in
    (distance, index) order, so with ``radius[i]`` the k-th distance of ``search(q, k)`` the first k equal ``search``'s
    row and the rest are ties at ``radius[i]``.  ``exclude_tags`` as in ``search``.  Sharded: collective, every rank gets
    the result of one index holding the concatenated shards.

    ``add(feats, tags=None, groups=None)`` with ``groups`` ([n] integers, e.g. tracklet or identity ids) makes the index
    grouped; as with tags, the first non-empty add decides, a later add of the other kind raises, and an index emptied by
    ``remove`` decides again.  ``dist, index, group = search_groups(q, k, exclude_tags=None)`` returns, per query, the
    rows ``search(q, k, exclude_tags)`` would order, by the same (distance, index) keys, with every row after the first
    of its group dropped, the first k of them: [nq, k] float32 distances, int64 rows (each group's nearest row) and int64
    groups, padded with inf / -1 / -1 past the last group (find padding by ``index == -1``).  When every row is its own
    group, ``dist`` and ``index`` equal ``search``'s bit for bit.  k is in [1, 128]; it needs a grouped index (an empty
    one answers with padding).  Groups move with their rows in ``remove``.  Sharded: collective, and a group may have rows
    on several ranks; every rank gets the result of one index holding the concatenated shards.
    """

    def __init__(self, dim, dtype=None, precision="f16x3", device=None, group=None):
        torch = _lib.require_cuda()
        lib = _lib.load()
        dtype = torch.float16 if dtype is None else dtype
        if dtype not in (torch.float16, torch.float32):
            raise RuntimeError("GalleryIndex: dtype must be torch.float16 or torch.float32, got %s" % (dtype,))
        if int(dim) <= 0:
            raise RuntimeError("GalleryIndex: dim must be positive")
        self.dim, self.dtype, self.group = int(dim), dtype, group
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("GalleryIndex: device must be a CUDA device")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._lib = lib
        self._h = C.c_void_p()
        code = _lib.DTYPE_F16 if dtype == torch.float16 else _lib.DTYPE_F32
        _lib.check(lib.pps_index_create(self.device.index, self.dim, code, _prec_code(precision), C.byref(self._h)),
                   "pps_index_create")

    def __len__(self):
        return int(self._lib.pps_index_size(self._h))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self._lib.pps_index_destroy(h)
            self._h = None

    def _rows(self, x, name):
        """(contiguous-row CUDA tensor on the index's device, whether the input was numpy)"""
        import torch
        is_np = isinstance(x, np.ndarray)
        if is_np:
            x = torch.from_numpy(np.ascontiguousarray(x))
        elif not isinstance(x, torch.Tensor):
            raise RuntimeError("%s: expected numpy.ndarray or torch.Tensor, got %s" % (name, type(x)))
        if x.dim() != 2 or int(x.shape[1]) != self.dim:
            raise RuntimeError("%s: expected shape [n, %d], got %s" % (name, self.dim, tuple(x.shape)))
        if x.dtype != self.dtype:
            raise RuntimeError("%s: expected %s rows (the index's dtype), got %s" % (name, self.dtype, x.dtype))
        x = x.to(self.device)
        if x.stride(1) != 1 or (x.shape[0] > 1 and x.stride(0) < self.dim):
            x = x.contiguous()
        return x, is_np

    def _tags(self, t, n, name):
        """[n] int64 CUDA tensor on the index's device from integer numpy or torch values (n None: any length)"""
        import torch
        if isinstance(t, np.ndarray):
            if not np.issubdtype(t.dtype, np.integer):
                raise RuntimeError("%s: expected integers, got %s" % (name, t.dtype))
            t = torch.from_numpy(np.ascontiguousarray(t, dtype=np.int64))
        elif isinstance(t, torch.Tensor):
            if t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
                raise RuntimeError("%s: expected integers, got %s" % (name, t.dtype))
        else:
            raise RuntimeError("%s: expected numpy.ndarray or torch.Tensor, got %s" % (name, type(t)))
        if t.dim() != 1 or (n is not None and int(t.shape[0]) != n):
            raise RuntimeError("%s: expected shape [%s], got %s" % (name, "n" if n is None else n, tuple(t.shape)))
        return t.to(device=self.device, dtype=torch.int64).contiguous()

    def add(self, feats, tags=None, groups=None):
        """Append rows (with their tags and groups); returns (row0, rows), their range among this index's (local) rows."""
        import torch
        x, _ = self._rows(feats, "feats")
        row0, n = len(self), int(x.shape[0])
        ld = int(x.stride(0)) if n else self.dim
        with torch.cuda.device(self.device):
            if groups is not None:
                gr = self._tags(groups, n, "groups")
                t = None if tags is None else self._tags(tags, n, "tags")
                _lib.check(self._lib.pps_index_add_grouped(self._h, _lib.ptr(x), n, ld, _lib.ptr(t), _lib.ptr(gr),
                                                           _lib.stream_ptr()), "pps_index_add_grouped")
            elif tags is None:
                _lib.check(self._lib.pps_index_add(self._h, _lib.ptr(x), n, ld, _lib.stream_ptr()), "pps_index_add")
            else:
                t = self._tags(tags, n, "tags")
                _lib.check(self._lib.pps_index_add_tagged(self._h, _lib.ptr(x), n, ld, _lib.ptr(t), _lib.stream_ptr()),
                           "pps_index_add_tagged")
        return row0, n

    def remove(self, rows):
        """Delete local rows (np.delete's renumbering); returns the number of distinct rows removed."""
        return self._remove(rows)

    def _remove(self, rows, flags=0):
        """remove() with flags: 0 or the PPS_INDEX_PIECE(n) test hook"""
        import torch
        t = self._tags(rows, None, "rows")
        n_removed = C.c_longlong(0)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.pps_index_remove(self._h, _lib.ptr(t), int(t.shape[0]), int(flags), _lib.stream_ptr(),
                                                  C.byref(n_removed)), "pps_index_remove")
        return int(n_removed.value)

    def _search_keys(self, q, k, index_offset=0, flags=0, exclude_tags=None):
        """[nq, k] top-k keys (distance bits << 32 | index_offset + row) of this index alone; flags: PPS_INDEX_* hooks."""
        import torch
        x, is_np = self._rows(q, "q")
        if not isinstance(k, (int, np.integer)) or not 1 <= int(k) <= _lib.TOPK_MAX:
            raise RuntimeError("k must be an integer in [1, %d], got %r" % (_lib.TOPK_MAX, k))
        nq, k = int(x.shape[0]), int(k)
        ldq = int(x.stride(0)) if nq else self.dim
        keys = torch.empty((nq, k), dtype=torch.int64, device=self.device)
        with torch.cuda.device(self.device):
            if exclude_tags is None:
                _lib.check(self._lib.pps_index_search(self._h, _lib.ptr(x), nq, ldq, k, int(index_offset), int(flags),
                                                      _lib.stream_ptr(), _lib.ptr(keys)), "pps_index_search")
            else:
                t = self._tags(exclude_tags, nq, "exclude_tags")
                _lib.check(self._lib.pps_index_search_excluding(self._h, _lib.ptr(x), nq, ldq, _lib.ptr(t), k,
                                                                int(index_offset), int(flags), _lib.stream_ptr(),
                                                                _lib.ptr(keys)), "pps_index_search_excluding")
        return keys, is_np

    def _unpack(self, keys, is_np):
        import torch
        nq, k = int(keys.shape[0]), int(keys.shape[1])
        dist = torch.empty((nq, k), dtype=torch.float32, device=self.device)
        index = torch.empty((nq, k), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.pps_topk_unpack(_lib.ptr(keys), nq, k, _lib.ptr(dist), _lib.ptr(index), _lib.stream_ptr()),
                       "pps_topk_unpack")
        index = index.long()
        if is_np:
            return dist.cpu().numpy(), index.cpu().numpy()
        return dist, index

    def _radius(self, radius, nq):
        """[nq] float32 CUDA tensor on the index's device from a number or [nq] floats / integers (numpy or torch)"""
        import torch
        if isinstance(radius, (bool, np.bool_)):
            raise RuntimeError("radius: expected a number or [nq] floats, got %r" % (radius,))
        if isinstance(radius, (int, float, np.integer, np.floating)):
            return torch.full((nq,), float(radius), dtype=torch.float32, device=self.device)
        if isinstance(radius, np.ndarray):
            if not (np.issubdtype(radius.dtype, np.integer) or np.issubdtype(radius.dtype, np.floating)):
                raise RuntimeError("radius: expected floats or integers, got %s" % radius.dtype)
            radius = torch.from_numpy(np.ascontiguousarray(radius))
        elif isinstance(radius, torch.Tensor):
            if radius.dtype.is_complex or radius.dtype == torch.bool:
                raise RuntimeError("radius: expected floats or integers, got %s" % radius.dtype)
        else:
            raise RuntimeError("radius: expected a number, numpy.ndarray or torch.Tensor, got %s" % type(radius))
        if radius.dim() != 1 or int(radius.shape[0]) != nq:
            raise RuntimeError("radius: expected a number or shape [%d], got %s" % (nq, tuple(radius.shape)))
        return radius.to(device=self.device, dtype=torch.float32).contiguous()

    def _range_keys(self, q, radius, index_offset=0, flags=0, exclude_tags=None):
        """(lims [nq + 1] int64, keys [total] of this index alone, sorted per query, whether q was numpy); flags: 0 or the
        PPS_INDEX_TKCAP(n) hook (keys per query in the first pass's slices)."""
        import torch
        x, is_np = self._rows(q, "q")
        nq = int(x.shape[0])
        ldq = int(x.stride(0)) if nq else self.dim
        r = self._radius(radius, nq)
        t = None if exclude_tags is None else self._tags(exclude_tags, nq, "exclude_tags")
        lims = torch.empty(nq + 1, dtype=torch.int64, device=self.device)
        total = C.c_longlong(0)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.pps_index_range_search(self._h, _lib.ptr(x), nq, ldq, _lib.ptr(r), _lib.ptr(t),
                                                        int(index_offset), int(flags), _lib.stream_ptr(), _lib.ptr(lims),
                                                        C.byref(total)), "pps_index_range_search")
            keys = torch.empty(int(total.value), dtype=torch.int64, device=self.device)
            _lib.check(self._lib.pps_index_range_keys(self._h, _lib.ptr(keys), _lib.stream_ptr()), "pps_index_range_keys")
        return lims, keys, is_np

    def _unpack_range(self, lims, keys, is_np):
        import torch
        n = int(keys.shape[0])
        dist = torch.empty(n, dtype=torch.float32, device=self.device)
        index = torch.empty(n, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.pps_topk_unpack(_lib.ptr(keys), n, 1, _lib.ptr(dist), _lib.ptr(index), _lib.stream_ptr()),
                       "pps_topk_unpack")
        index = index.long()
        if is_np:
            return lims.cpu().numpy(), dist.cpu().numpy(), index.cpu().numpy()
        return lims, dist, index

    def _offset(self):
        """index_offset of this rank's rows: one all-gather of the shard sizes (0 without a group)"""
        import torch
        if self.group is None:
            return 0
        import torch.distributed as dist_mod
        mine = torch.tensor([len(self)], dtype=torch.int64, device=self.device)
        sizes = [torch.empty_like(mine) for _ in range(dist_mod.get_world_size(self.group))]
        dist_mod.all_gather(sizes, mine, group=self.group)
        return int(sum(int(s.item()) for s in sizes[:dist_mod.get_rank(self.group)]))

    def range_search(self, q, radius, exclude_tags=None):
        """(lims [nq + 1] int64, dist [total] float32, index [total] int64): every gallery row within radius of each query
        row (with exclude_tags: of the rows whose tag is not the query's), per query in (distance, index) order."""
        lims, keys, is_np = self._range_keys(q, radius, self._offset(), exclude_tags=exclude_tags)
        if self.group is not None:
            lims, keys = gather_range_keys(lims, keys, self.group)
        return self._unpack_range(lims, keys, is_np)

    def _search_group_keys(self, q, k, index_offset=0, flags=0, exclude_tags=None):
        """([nq, k] keys, [nq, k] groups, whether q was numpy) of this index alone; flags: PPS_INDEX_* hooks."""
        import torch
        x, is_np = self._rows(q, "q")
        if not isinstance(k, (int, np.integer)) or not 1 <= int(k) <= _lib.TOPK_MAX:
            raise RuntimeError("k must be an integer in [1, %d], got %r" % (_lib.TOPK_MAX, k))
        nq, k = int(x.shape[0]), int(k)
        ldq = int(x.stride(0)) if nq else self.dim
        t = None if exclude_tags is None else self._tags(exclude_tags, nq, "exclude_tags")
        keys = torch.empty((nq, k), dtype=torch.int64, device=self.device)
        groups = torch.empty((nq, k), dtype=torch.int64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.pps_index_search_groups(self._h, _lib.ptr(x), nq, ldq, _lib.ptr(t), k, int(index_offset),
                                                         int(flags), _lib.stream_ptr(), _lib.ptr(keys), _lib.ptr(groups)),
                       "pps_index_search_groups")
        return keys, groups, is_np

    def _group_stats(self):
        """(rows swept as materialised blocks before the chunks, chunks, whether the fallback ran) of the last
        search_groups on this index"""
        prefix, chunks, fallback = C.c_longlong(0), C.c_longlong(0), C.c_int(0)
        _lib.check(self._lib.pps_index_group_stats(self._h, C.byref(prefix), C.byref(chunks), C.byref(fallback)),
                   "pps_index_group_stats")
        return int(prefix.value), int(chunks.value), bool(fallback.value)

    def search_groups(self, q, k, exclude_tags=None):
        """(dist [nq, k] float32, index [nq, k] int64, group [nq, k] int64): the nearest row of each of the k nearest
        groups of every query row (with exclude_tags: among the rows whose tag is not the query's)."""
        keys, groups, is_np = self._search_group_keys(q, k, self._offset(), exclude_tags=exclude_tags)
        if self.group is not None:
            keys, groups = merge_group_keys(keys, groups, int(k), self.group)
        dist, index = self._unpack(keys, False)
        if is_np:
            return dist.cpu().numpy(), index.cpu().numpy(), groups.cpu().numpy()
        return dist, index, groups

    def search(self, q, k, exclude_tags=None):
        """(dist [nq, k] float32, index [nq, k] int64) of the k nearest gallery rows of every query row (with
        exclude_tags: of the rows whose tag is not the query's)."""
        keys, is_np = self._search_keys(q, k, self._offset(), exclude_tags=exclude_tags)
        if self.group is not None:
            keys = merge_topk_keys(keys, int(k), self.group)
        return self._unpack(keys, is_np)


def merge_group_keys(keys, groups, k, group):
    """All-gather every rank's [nq, k] grouped keys and groups and merge them (merge_group_lists)."""
    import torch.distributed as dist_mod
    world = dist_mod.get_world_size(group)
    all_keys = [keys.new_empty(keys.shape) for _ in range(world)]
    all_groups = [groups.new_empty(groups.shape) for _ in range(world)]
    dist_mod.all_gather(all_keys, keys, group=group)
    dist_mod.all_gather(all_groups, groups, group=group)
    return merge_group_lists(all_keys, all_groups, k)


def merge_group_lists(keys_list, groups_list, k):
    """One grouped result from several ([nq, k] keys, [nq, k] groups) of disjoint row sets (shards; a group may span
    them): per query, every list's keys in key order, the first of each group, the first k (pps_topk_group_merge_lists)."""
    import torch
    keys = torch.stack(list(keys_list)).contiguous()
    groups = torch.stack(list(groups_list)).contiguous()
    lists, nq = int(keys.shape[0]), int(keys.shape[1])
    out_k = torch.empty((nq, k), dtype=torch.int64, device=keys.device)
    out_g = torch.empty((nq, k), dtype=torch.int64, device=keys.device)
    lib = _lib.load()
    with torch.cuda.device(keys.device):
        _lib.check(lib.pps_topk_group_merge_lists(_lib.ptr(keys), _lib.ptr(groups), lists, nq, k, _lib.ptr(out_k),
                                                  _lib.ptr(out_g), _lib.stream_ptr()), "pps_topk_group_merge_lists")
    return out_k, out_g


def gather_range_keys(lims, keys, group):
    """All-gather every rank's range-search result (lims [nq + 1], keys [total]) and merge them (merge_range_lists)."""
    import torch
    import torch.distributed as dist_mod
    world = dist_mod.get_world_size(group)
    all_lims = [torch.empty_like(lims) for _ in range(world)]
    dist_mod.all_gather(all_lims, lims, group=group)
    totals = [int(x[-1].item()) for x in all_lims]
    pad = torch.zeros(max(totals), dtype=torch.int64, device=keys.device)
    pad[:keys.shape[0]] = keys
    all_keys = [torch.empty_like(pad) for _ in range(world)]
    dist_mod.all_gather(all_keys, pad, group=group)
    return merge_range_lists(all_lims, [k[:n] for k, n in zip(all_keys, totals)])


def merge_range_lists(lims_list, keys_list):
    """One range-search result from several (lims [nq + 1] int64, keys [total]) of disjoint row sets (shards, in rank
    order): every query's keys of every list, query-major, then each query's keys sorted (pps_sort_key_segments)."""
    import torch
    nq = int(lims_list[0].shape[0]) - 1
    dev = lims_list[0].device
    counts = torch.stack([x[1:] - x[:-1] for x in lims_list])                        # [lists, nq]
    lims = torch.zeros(nq + 1, dtype=torch.int64, device=dev)
    lims[1:] = torch.cumsum(counts.sum(0), 0)
    before = torch.cumsum(counts, 0) - counts                                         # keys of earlier lists, per query
    total = int(lims[-1].item())
    keys = torch.empty(total, dtype=torch.int64, device=dev)
    for j, (lx, kx) in enumerate(zip(lims_list, keys_list)):
        n = int(kx.shape[0])
        if n == 0:
            continue
        q = torch.repeat_interleave(torch.arange(nq, device=dev), counts[j])        # query of every key of list j
        dest = lims[:-1][q] + before[j][q] + (torch.arange(n, device=dev) - lx[:-1][q])
        keys[dest] = kx
    if total:
        lib = _lib.load()
        scratch = torch.empty_like(keys)
        with torch.cuda.device(dev):
            _lib.check(lib.pps_sort_key_segments(_lib.ptr(keys), _lib.ptr(lims), nq, _lib.ptr(scratch), _lib.stream_ptr()),
                       "pps_sort_key_segments")
    return lims, keys
