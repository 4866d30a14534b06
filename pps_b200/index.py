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

    def add(self, feats, tags=None):
        """Append rows (with their tags); returns (row0, rows), their range among this index's (local) rows."""
        import torch
        x, _ = self._rows(feats, "feats")
        row0, n = len(self), int(x.shape[0])
        ld = int(x.stride(0)) if n else self.dim
        with torch.cuda.device(self.device):
            if tags is None:
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

    def search(self, q, k, exclude_tags=None):
        """(dist [nq, k] float32, index [nq, k] int64) of the k nearest gallery rows of every query row (with
        exclude_tags: of the rows whose tag is not the query's)."""
        import torch
        offset = 0
        if self.group is not None:
            import torch.distributed as dist_mod
            mine = torch.tensor([len(self)], dtype=torch.int64, device=self.device)
            sizes = [torch.empty_like(mine) for _ in range(dist_mod.get_world_size(self.group))]
            dist_mod.all_gather(sizes, mine, group=self.group)
            offset = int(sum(int(s.item()) for s in sizes[:dist_mod.get_rank(self.group)]))
        keys, is_np = self._search_keys(q, k, offset, exclude_tags=exclude_tags)
        if self.group is not None:
            keys = merge_topk_keys(keys, int(k), self.group)
        return self._unpack(keys, is_np)
