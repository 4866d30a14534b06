"""Test-time ranking: host-side mirror of detectron/datasets/reid_dataset_evaluator.py.

Same entry points, argument order and error behaviour as the reference:
  compute_dist(array1, array2, type='euclidean')                                  (:244-272)
  cmc(distmat, query_ids, gallery_ids, query_cams, gallery_cams, topk=100, ...)   (:283-363)
  mean_ap(distmat, query_ids, gallery_ids, query_cams, gallery_cams, average)     (:366-439)
  evaluate(json_dataset, all_feats, output_dir) -> (mAP, cmc, mq_mAP, mq_cmc)     (:29-209)
plus ``rank_eval`` — the fused path from features to AP / first-match ranks / top-k that never
needs more than one gallery chunk of the distance matrix — and ``evaluate_host`` (the C ABI's
pps_evaluate_host: host buffers in, metrics out).

All arithmetic runs in the CUDA library (tcgen05 distance GEMM, counting rank kernels); this
module only marshals arrays, builds the same-id pair lists through the library's host code and
does the final averaging over queries exactly as the reference does.  There is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import os
from collections import OrderedDict, defaultdict
from typing import Optional

import numpy as np

from . import _lib

DEFAULT_PRECISION = "f16x3"         # two scaled fp16 planes, three terms: see DESIGN.md 4.3
# extra PPS_DIST_* flags OR-ed into every tensor-core distance call (tests / profiling use
# _lib.DIST_KERNEL_1CTA to select the single-CTA kernel; 0 = the 2-CTA default)
DIST_KERNEL_FLAGS = _lib.DIST_KERNEL_1CTA if os.environ.get("PPS_DIST_KERNEL", "") == "1cta" else 0


# ------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------
def _torch():
    return _lib.require_cuda()


def _as_cuda_f32(a, name):
    torch = _torch()
    if isinstance(a, np.ndarray):
        if a.ndim != 2:
            raise RuntimeError("%s: expected a 2-D array, got ndim=%d" % (name, a.ndim))
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda(), True
    if isinstance(a, torch.Tensor):
        if a.dim() != 2:
            raise RuntimeError("%s: expected a 2-D tensor, got ndim=%d" % (name, a.dim()))
        t = a if a.is_cuda else a.cuda()
        if t.dtype not in (torch.float32, torch.float16):
            t = t.float()
        return t.contiguous(), False
    raise RuntimeError("%s: expected numpy.ndarray or torch.Tensor, got %s" % (name, type(a)))


def _ids64(a, name):
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    a = np.ascontiguousarray(np.asarray(a), dtype=np.int64)
    if a.ndim != 1:
        raise RuntimeError("%s: expected a 1-D array" % name)
    return a


PREFILTER_MIN_ROWS = 131072      # galleries at least this long get the candidate pre-filter before the pair sweeps


class PairLists:
    """Same-id (query, gallery) pairs in CSR form (C ABI part 2c); host arrays + device copies."""

    def __init__(self, query_ids, query_cams, gallery_ids, gallery_cams, device=None):
        lib = _lib.load()
        qi, qc = _ids64(query_ids, "query_ids"), _ids64(query_cams, "query_cams")
        gi, gc = _ids64(gallery_ids, "gallery_ids"), _ids64(gallery_cams, "gallery_cams")
        if qi.shape != qc.shape or gi.shape != gc.shape:
            raise RuntimeError("ids and cams must have the same length")
        self.nq, self.ng = int(qi.shape[0]), int(gi.shape[0])
        n = int(lib.pps_pairs_count(_lib.ptr(qi), self.nq, _lib.ptr(gi), self.ng))
        if n < 0:
            _lib.check(n, "pps_pairs_count")
        self.n_pairs = n
        self.off = np.zeros(self.nq + 1, dtype=np.int32)
        self.q = np.zeros(max(n, 1), dtype=np.int32)
        self.g = np.zeros(max(n, 1), dtype=np.int32)
        self.pos = np.zeros(max(n, 1), dtype=np.uint8)
        _lib.check(lib.pps_pairs_fill(_lib.ptr(qi), _lib.ptr(qc), self.nq, _lib.ptr(gi), _lib.ptr(gc), self.ng,
                                      _lib.ptr(self.off), _lib.ptr(self.q), _lib.ptr(self.g), _lib.ptr(self.pos)),
                   "pps_pairs_fill")
        per_q = np.diff(self.off)
        self.max_pairs = int(per_q.max()) if self.nq else 0
        # junk (same id, same camera) as its own CSR: the exclusion list of the valid-filtered top-k
        junk = self.pos[:n] == 0
        self.junk_g = np.ascontiguousarray(self.g[:n][junk])
        jcount = np.bincount(self.q[:n][junk], minlength=self.nq) if n else np.zeros(self.nq, dtype=np.int64)
        self.junk_off = np.zeros(self.nq + 1, dtype=np.int32)
        self.junk_off[1:] = np.cumsum(jcount)
        self.n_pos_per_q = (np.bincount(self.q[:n][~junk], minlength=self.nq) if n
                            else np.zeros(self.nq, dtype=np.int64))
        self._dev = None
        if device is not None:
            self.to(device)

    def to(self, device):
        torch = _torch()
        f = lambda a: torch.from_numpy(a).to(device)
        self._dev = dict(off=f(self.off), q=f(self.q), g=f(self.g), pos=f(self.pos), junk_off=f(self.junk_off),
                         junk_g=f(self.junk_g if self.junk_g.size else np.zeros(1, dtype=np.int32)))
        self.device = device
        return self

    def dev(self, name):
        return self._dev[name]


class DevicePairs:
    """Same-id pair lists built ON THE DEVICE (C ABI part 2c, pairs.cu) from resident id / camera arrays.

    ``begin()`` launches count + scan and an 8-byte read-back of {n_pairs, max_pairs}; ``finish()`` waits
    for that read-back (the caller enqueues the distance GEMM in between, so the device never idles),
    sizes the lists and launches the fill.  Host copies (``off``, ``q``, ``g``, ``pos`` ...) are
    downloaded lazily, only for the outputs that need them (cmc with first_match_break=False)."""

    def __init__(self, query_ids, query_cams, gallery_ids, gallery_cams, device):
        torch = _torch()
        self.lib = _lib.load()
        qi, qc = _ids64(query_ids, "query_ids"), _ids64(query_cams, "query_cams")
        gi, gc = _ids64(gallery_ids, "gallery_ids"), _ids64(gallery_cams, "gallery_cams")
        if qi.shape != qc.shape or gi.shape != gc.shape:
            raise RuntimeError("ids and cams must have the same length")
        self.nq, self.ng = int(qi.shape[0]), int(gi.shape[0])
        if self.ng > 0x7fffffff or self.nq > 0x7fffffff:
            raise RuntimeError("pair lists index the gallery with int32")
        self.device = torch.device(device)
        up = lambda a: torch.from_numpy(a if a.size else np.zeros(1, np.int64)).to(self.device)
        self.qid, self.qcam, self.gid, self.gcam = up(qi), up(qc), up(gi), up(gc)
        ws = int(self.lib.pps_pairs_workspace_bytes(self.nq, self.ng))
        self.ws = torch.empty(max(ws, 16), dtype=torch.uint8, device=self.device)
        self.off_d = torch.empty(self.nq + 1, dtype=torch.int32, device=self.device)
        self.totals_d = torch.empty(2, dtype=torch.int32, device=self.device)
        self.totals_h = torch.empty(2, dtype=torch.int32).pin_memory()
        self.event = torch.cuda.Event()
        self.cap = 0
        self.q_d = self.g_d = self.pos_d = None
        self.n_pairs = self.max_pairs = 0
        self._host = None
        # very large galleries: the sweeps run on the rows whose id is some query's id (pps_pairs_prefilter)
        self.prefilter = self.ng >= PREFILTER_MIN_ROWS and self.nq > 0
        self.n_cand = self.ng
        if self.prefilter:
            self.pf_ws = torch.empty(int(self.lib.pps_pairs_prefilter_workspace_bytes(self.nq, self.ng)), dtype=torch.uint8,
                                     device=self.device)
            self.cand_rows = torch.empty(self.ng, dtype=torch.int32, device=self.device)
            self.cand_gid = torch.empty(self.ng, dtype=torch.int64, device=self.device)
            self.cand_gcam = torch.empty(self.ng, dtype=torch.int64, device=self.device)
            self.n_cand_d = torch.zeros(1, dtype=torch.int32, device=self.device)
            self.n_cand_h = torch.zeros(1, dtype=torch.int32).pin_memory()

    def _sweep_arrays(self):
        """(gallery ids, gallery cameras, rows) the pair sweeps run on."""
        if self.prefilter:
            return self.cand_gid, self.cand_gcam, self.n_cand
        return self.gid, self.gcam, self.ng

    def begin(self):
        lib = self.lib
        if self.prefilter:
            torch = _torch()
            _lib.check(lib.pps_pairs_prefilter(_lib.ptr(self.qid), self.nq, _lib.ptr(self.gid), _lib.ptr(self.gcam), self.ng,
                                               _lib.ptr(self.pf_ws), _lib.ptr(self.cand_rows), _lib.ptr(self.cand_gid),
                                               _lib.ptr(self.cand_gcam), _lib.ptr(self.n_cand_d), _lib.stream_ptr()),
                       "pps_pairs_prefilter")
            self.n_cand_h.copy_(self.n_cand_d, non_blocking=True)
            torch.cuda.current_stream().synchronize()      # 4 bytes: the candidate count sizes the sweeps
            self.n_cand = int(self.n_cand_h[0])
        gid, _, rows = self._sweep_arrays()
        _lib.check(lib.pps_pairs_count_device(_lib.ptr(self.qid), self.nq, _lib.ptr(gid), rows, _lib.ptr(self.ws),
                                              _lib.ptr(self.off_d), _lib.ptr(self.totals_d), _lib.stream_ptr()),
                   "pps_pairs_count_device")
        self.totals_h.copy_(self.totals_d, non_blocking=True)
        self.event.record()
        self._host = None
        return self

    def finish(self, zero_f32=None, zero_u32=None, zero_per_query=None):
        """``zero_f32`` / ``zero_u32``: optional per-pair device arrays (capacity >= n_pairs) the fill kernel
        zero-fills (pair_d / cnt_le); pass callables to allocate them once n_pairs is known.
        ``zero_per_query``: optional int32 [nq] device tensor it zero-fills too (cnt_first)."""
        torch = _torch()
        self.event.synchronize()
        self.n_pairs, self.max_pairs = int(self.totals_h[0]), int(self.totals_h[1])
        if self.n_pairs > self.cap or self.q_d is None:
            self.cap = max(int(self.n_pairs * 1.25), 1024)
            self.q_d = torch.empty(self.cap, dtype=torch.int32, device=self.device)
            self.g_d = torch.empty(self.cap, dtype=torch.int32, device=self.device)
            self.pos_d = torch.empty(self.cap, dtype=torch.uint8, device=self.device)
        if callable(zero_f32):
            zero_f32 = zero_f32(self.n_pairs)
        if callable(zero_u32):
            zero_u32 = zero_u32(self.n_pairs)
        gid, gcam, rows = self._sweep_arrays()
        _lib.check(self.lib.pps_pairs_fill_device(_lib.ptr(self.qid), _lib.ptr(self.qcam), self.nq, _lib.ptr(gid),
                                                  _lib.ptr(gcam), rows, _lib.ptr(self.ws),
                                                  _lib.ptr(self.q_d), _lib.ptr(self.g_d), _lib.ptr(self.pos_d),
                                                  _lib.ptr(zero_f32), _lib.ptr(zero_u32), _lib.ptr(zero_per_query),
                                                  self.n_pairs, _lib.stream_ptr()), "pps_pairs_fill_device")
        if self.prefilter and self.n_pairs:
            _lib.check(self.lib.pps_pairs_remap(_lib.ptr(self.g_d), self.n_pairs, _lib.ptr(self.cand_rows), 0,
                                                _lib.stream_ptr()), "pps_pairs_remap")
        return self

    def dev(self, name):
        return {"off": self.off_d, "q": self.q_d, "g": self.g_d, "pos": self.pos_d}[name]

    # ---- lazy host mirrors (same fields as PairLists) ----
    def _download(self):
        if self._host is None:
            n = self.n_pairs
            self._host = dict(off=self.off_d.cpu().numpy(), q=self.q_d[:max(n, 1)].cpu().numpy(),
                              g=self.g_d[:max(n, 1)].cpu().numpy(), pos=self.pos_d[:max(n, 1)].cpu().numpy())
        return self._host

    off = property(lambda self: self._download()["off"])
    q = property(lambda self: self._download()["q"])
    g = property(lambda self: self._download()["g"])
    pos = property(lambda self: self._download()["pos"])

    @property
    def n_pos_per_q(self):
        n = self.n_pairs
        if not n:
            return np.zeros(self.nq, dtype=np.int64)
        return np.bincount(self.q[:n][self.pos[:n] == 1], minlength=self.nq)


class RankResult:
    """Per-query outputs of the rank kernels (host numpy) + the reference's averages."""

    def __init__(self, ap, is_valid, first_rank, neg_before=None, pairs: Optional[PairLists] = None,
                 topk_index=None, topk_dist=None):
        self.ap, self.is_valid, self.first_rank = ap, is_valid, first_rank
        self.neg_before, self.pairs = neg_before, pairs
        self.topk_index, self.topk_dist = topk_index, topk_dist

    def mean_ap(self):
        if len(self.ap) == 0:
            raise RuntimeError("No valid query")
        return float(np.sum(self.ap)) / np.sum(self.is_valid)   # :437-438 (nan if no query is valid)

    def cmc_matrix(self, topk, first_match_break):
        m = len(self.ap)
        ret = np.zeros([m, topk])
        if first_match_break:
            ok = (self.is_valid > 0) & (self.first_rank >= 0) & (self.first_rank < topk)
            ret[np.nonzero(ok)[0], self.first_rank[ok]] += 1
        else:
            p = self.pairs
            n = p.n_pairs
            sel = (p.pos[:n] == 1) & (self.neg_before[:n] < topk)
            delta = 1.0 / np.maximum(p.n_pos_per_q, 1)
            np.add.at(ret, (p.q[:n][sel], self.neg_before[:n][sel]), delta[p.q[:n][sel]])
        return ret.cumsum(axis=1)

    def cmc(self, topk=10, first_match_break=True, average=True):
        num_valid = int(np.sum(self.is_valid))
        if num_valid == 0:
            raise RuntimeError("No valid query")                 # :358-359
        ret = self.cmc_matrix(topk, first_match_break)
        if average:
            return np.sum(ret, axis=0) / num_valid
        return ret, self.is_valid.astype(np.float64)


def _rank_block(lib, dist, ldd, nq, ncols, col0, pairs: PairLists, pair_d, cnt_le, cnt_first, do_gather, do_count,
                topk_key=None, topk=0, topk_filtered=True):
    s = _lib.stream_ptr()
    if do_gather and pairs.n_pairs:
        _lib.check(lib.pps_rank_gather(_lib.ptr(dist), ldd, nq, ncols, col0, _lib.ptr(pairs.dev("q")),
                                       _lib.ptr(pairs.dev("g")), pairs.n_pairs, _lib.ptr(pair_d), s),
                   "pps_rank_gather")
    if do_count:
        if topk_key is not None:
            # counts + first-match counter + top-k in one read of the block
            use = pairs.n_pairs > 0
            _lib.check(lib.pps_rank_sweep(_lib.ptr(dist), ldd, nq, ncols, col0, _lib.ptr(pairs.dev("off")),
                                          _lib.ptr(pairs.dev("g")) if use else None,
                                          _lib.ptr(pairs.dev("pos")) if use else None, _lib.ptr(pair_d) if use else None,
                                          pairs.max_pairs if use else 0, _lib.ptr(cnt_le) if use else None,
                                          _lib.ptr(cnt_first), _lib.ptr(topk_key), topk, 1 if topk_filtered else 0, s),
                       "pps_rank_sweep")
        elif pairs.n_pairs:
            _lib.check(lib.pps_rank_count(_lib.ptr(dist), ldd, nq, ncols, col0, _lib.ptr(pairs.dev("off")),
                                          _lib.ptr(pairs.dev("g")), _lib.ptr(pairs.dev("pos")), _lib.ptr(pair_d),
                                          pairs.max_pairs, _lib.ptr(cnt_le), _lib.ptr(cnt_first), s),
                       "pps_rank_count")


def _finalize(lib, nq, pairs: PairLists, pair_d, cnt_le, cnt_first, want_neg_before):
    torch = _torch()
    dev = pair_d.device
    ap = torch.empty(nq, dtype=torch.float64, device=dev)
    valid = torch.empty(nq, dtype=torch.uint8, device=dev)
    first = torch.empty(nq, dtype=torch.int32, device=dev)
    negb = torch.zeros(max(pairs.n_pairs, 1), dtype=torch.int32, device=dev) if want_neg_before else None
    _lib.check(lib.pps_rank_finalize(nq, _lib.ptr(pairs.dev("off")), _lib.ptr(pairs.dev("g")),
                                     _lib.ptr(pairs.dev("pos")), _lib.ptr(pair_d), _lib.ptr(cnt_le),
                                     _lib.ptr(cnt_first), _lib.ptr(ap), _lib.ptr(valid), _lib.ptr(first),
                                     _lib.ptr(negb), _lib.stream_ptr()), "pps_rank_finalize")
    return ap, valid, first, negb


def rank_distmat(distmat, query_ids, gallery_ids, query_cams, gallery_cams, want_neg_before=False, topk=0,
                 topk_filtered=True, ap_definition="step") -> RankResult:
    """Ranking outputs for a materialised [m, n] distance matrix (numpy or CUDA tensor).

    ap_definition: 'step' = scikit-learn >= 0.19 ``average_precision_score`` (what an unpinned install runs today);
    'trapezoid' = scikit-learn 0.18.1 (the version reid_dataset_evaluator.py:398-407 asks for; needs one more pass
    over the matrix for the exact-tie counts)."""
    if ap_definition not in ("step", "trapezoid"):
        raise RuntimeError("ap_definition must be 'step' or 'trapezoid'")
    torch = _torch()
    lib = _lib.load()
    if getattr(distmat, "dtype", None) in (np.float64, torch.float64):
        # the reference ranks whatever dtype it is given; this path ranks float32, and distinct float64 distances can
        # collapse into float32 ties (tie-grouped AP / first-match rank would then differ)
        import warnings
        warnings.warn("rank_distmat: float64 distances are ranked as float32 (values closer than 2^-24 relative become ties)",
                      RuntimeWarning, stacklevel=3)
    dist, _ = _as_cuda_f32(distmat, "distmat")
    if dist.dtype != torch.float32:
        dist = dist.float()
    m, n = int(dist.shape[0]), int(dist.shape[1])
    if topk and dist.numel() and bool((dist < 0).any()):
        # top-k keys order by the bits of a NON-NEGATIVE float; the counting half handles any sign
        raise RuntimeError("rank_distmat: top-k needs non-negative distances (got negative entries, e.g. a negated similarity); "
                           "shift the matrix or call it with topk=0")
    with torch.cuda.device(dist.device):
        pairs = DevicePairs(query_ids, query_cams, gallery_ids, gallery_cams, dist.device)
        if pairs.nq != m or pairs.ng != n:
            raise RuntimeError("distmat shape %s does not match %d query / %d gallery ids" % ((m, n), pairs.nq, pairs.ng))
        cnt_first = torch.empty(max(m, 1), dtype=torch.int32, device=dist.device)
        pairs.begin().finish(zero_per_query=cnt_first)
        E = max(pairs.n_pairs, 1)
        pair_d = torch.zeros(E, dtype=torch.float32, device=dist.device)
        cnt_le = torch.zeros(E, dtype=torch.int32, device=dist.device)
        key = None
        if topk:
            key = torch.empty((m, topk), dtype=torch.int64, device=dist.device)
            _lib.check(lib.pps_topk_init(_lib.ptr(key), m, topk, _lib.stream_ptr()), "pps_topk_init")
        _rank_block(lib, dist, int(dist.stride(0)), m, n, 0, pairs, pair_d, cnt_le, cnt_first, True, True, key, topk,
                    topk_filtered)
        ap, valid, first, negb = _finalize(lib, m, pairs, pair_d, cnt_le, cnt_first, want_neg_before)
        if ap_definition == "trapezoid" and pairs.n_pairs:
            cnt_eq = torch.zeros(E, dtype=torch.int32, device=dist.device)
            _lib.check(lib.pps_rank_count_eq(_lib.ptr(dist), int(dist.stride(0)), m, n, _lib.ptr(pairs.dev("off")),
                                             _lib.ptr(pair_d), pairs.max_pairs, _lib.ptr(cnt_eq), _lib.stream_ptr()),
                       "pps_rank_count_eq")
            _lib.check(lib.pps_rank_finalize_trapezoid(m, _lib.ptr(pairs.dev("off")), _lib.ptr(pairs.dev("g")),
                                                       _lib.ptr(pairs.dev("pos")), _lib.ptr(pair_d), _lib.ptr(cnt_le),
                                                       _lib.ptr(cnt_eq), _lib.ptr(ap), _lib.stream_ptr()),
                       "pps_rank_finalize_trapezoid")
        ti = td = None
        if topk:
            td = torch.empty((m, topk), dtype=torch.float32, device=dist.device)
            ti = torch.empty((m, topk), dtype=torch.int32, device=dist.device)
            _lib.check(lib.pps_topk_unpack(_lib.ptr(key), m, topk, _lib.ptr(td), _lib.ptr(ti), _lib.stream_ptr()),
                       "pps_topk_unpack")
            ti, td = ti.cpu().numpy(), td.cpu().numpy()
        return RankResult(ap.cpu().numpy(), valid.cpu().numpy(), first.cpu().numpy(),
                          negb.cpu().numpy() if negb is not None else None, pairs, ti, td)


# ------------------------------------------------------------------------------------
# distance
# ------------------------------------------------------------------------------------
class SplitOperand:
    """Rows prepared for the tensor-core distance: bf16 residual planes (or fp16 rows) + |x|^2."""

    def __init__(self, feats, planes: int, f16_scaled: bool = False):
        """``f16_scaled``: two power-of-two-scaled fp16 planes (what the 'f16x3' precision consumes) instead of bf16
        planes; ``sqnorm`` then carries the inverse row scales after the norms."""
        torch = _torch()
        lib = _lib.load()
        if feats.dtype == torch.float16:
            dtype, planes, f16_scaled = _lib.DTYPE_F16, 1, False
        elif feats.dtype == torch.float32:
            dtype = _lib.DTYPE_F32
        else:
            raise RuntimeError("features must be float32 or float16")
        if feats.stride(1) != 1:
            feats = feats.contiguous()
        self.rows, self.dim = int(feats.shape[0]), int(feats.shape[1])
        self.planes_n, self.is_f16, self.f16_scaled = planes, dtype == _lib.DTYPE_F16, bool(f16_scaled)
        if f16_scaled and planes != 2:
            raise RuntimeError("scaled fp16 operands have two planes")
        nbytes = int(lib.pps_split_bytes(self.rows, self.dim, planes)) if self.rows else 0
        self.planes = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=feats.device)
        self.sqnorm = torch.empty(2 * max(self.rows, 1), dtype=torch.float32, device=feats.device)
        if self.rows:
            _lib.check(lib.pps_split_rows(_lib.ptr(feats), dtype, self.rows, self.dim, int(feats.stride(0)),
                                          planes | (_lib.SPLIT_F16_SCALED if f16_scaled else 0),
                                          _lib.ptr(self.planes), _lib.ptr(self.sqnorm), _lib.stream_ptr()),
                       "pps_split_rows")


def _prec_code(precision):
    if precision not in _lib.PRECISIONS:
        raise RuntimeError("unknown precision %r (expected one of %s)" % (precision, sorted(_lib.PRECISIONS)))
    return _lib.PRECISIONS[precision]


def dist_block(a: SplitOperand, b: SplitOperand, prec: int, out, flags=0, b_row0=0, b_rows=None):
    """out[:, :b_rows] = distance(a rows, b rows [b_row0, b_row0+b_rows)) on the tensor cores."""
    lib = _lib.load()
    b_rows = b.rows - b_row0 if b_rows is None else b_rows
    if a.is_f16 != b.is_f16:
        raise RuntimeError("query and gallery features must have the same dtype")
    if a.is_f16:
        prec = _lib.PREC_F16X1
    if (prec == _lib.PREC_F16X3) != (a.f16_scaled and b.f16_scaled):
        raise RuntimeError("precision 'f16x3' needs (and only it takes) scaled fp16 operands")
    if b_row0 != 0 or b_rows != b.rows:
        # a row window of every plane: planes are [planes][rows][kpad], the TMA map needs the full
        # plane stride, so windows are expressed by a shifted base and the full row count upstream.
        raise RuntimeError("dist_block: gallery windows are handled by GalleryChunks")
    _lib.check(lib.pps_dist_tc(_lib.ptr(a.planes), _lib.ptr(a.sqnorm), a.rows, a.planes_n, 0, _lib.ptr(b.planes),
                               _lib.ptr(b.sqnorm), b.rows, b.planes_n, 0, a.dim, prec, flags | DIST_KERNEL_FLAGS,
                               _lib.ptr(out),
                               int(out.stride(0)), _lib.stream_ptr()), "pps_dist_tc")


def compute_dist(array1, array2, type="euclidean", precision: str = DEFAULT_PRECISION):
    """Pairwise distance, reid_dataset_evaluator.py:244-272.

    'euclidean' -> sqrt(max(0, |a|^2 + |b|^2 - 2ab)).  'cosine' -> the reference calls an undefined
    ``normalize`` (NameError, :259-260); what it intends — rows L2-normalised as
    detectron/core/test_engine.py:52-55 does, then a.b^T (a similarity) — is what this returns.
    numpy in -> numpy out; CUDA tensor in -> CUDA tensor out (a [m1, m2] view whose row stride is m2 rounded up to a
    multiple of 4).
    """
    assert type in ["cosine", "euclidean"]
    torch = _torch()
    lib = _lib.load()
    a, a_np = _as_cuda_f32(array1, "array1")
    b, b_np = _as_cuda_f32(array2, "array2")
    if a.shape[1] != b.shape[1]:
        raise RuntimeError("shapes %s and %s not aligned" % (tuple(a.shape), tuple(b.shape)))
    prec = _prec_code(precision)
    m1, m2, dim = int(a.shape[0]), int(b.shape[0]), int(a.shape[1])
    with torch.cuda.device(a.device):
        if type == "cosine":
            def unit_rows(x):
                x = x.float().contiguous()
                out = torch.empty_like(x)
                if x.shape[0]:
                    _lib.check(lib.pps_l2_normalize_rows(_lib.ptr(x), int(x.shape[0]), int(x.shape[1]), int(x.stride(0)),
                                                         _lib.ptr(out), int(out.stride(0)), _lib.stream_ptr()),
                               "pps_l2_normalize_rows")
                return out
            a, b = unit_rows(a), unit_rows(b)
        flags = _lib.DIST_DOT if type == "cosine" else 0
        # row stride padded to a multiple of 4 floats (16 bytes): what the 2-CTA kernel's TMA store needs - an odd stride
        # would silently select the single-CTA kernel, whose accumulation order (and last bits) differ from the ranking path
        buf = torch.empty((m1, (m2 + 3) // 4 * 4), dtype=torch.float32, device=a.device)
        out = buf[:, :m2]
        if m1 and m2:
            if prec == _lib.PREC_FP32:
                a32, b32 = a.float().contiguous(), b.float().contiguous()
                an = torch.empty(m1, dtype=torch.float32, device=a.device)
                bn = torch.empty(m2, dtype=torch.float32, device=a.device)
                _lib.check(lib.pps_row_sqnorm(_lib.ptr(a32), _lib.DTYPE_F32, m1, dim, dim, _lib.ptr(an),
                                              _lib.stream_ptr()), "pps_row_sqnorm")
                _lib.check(lib.pps_row_sqnorm(_lib.ptr(b32), _lib.DTYPE_F32, m2, dim, dim, _lib.ptr(bn),
                                              _lib.stream_ptr()), "pps_row_sqnorm")
                _lib.check(lib.pps_dist_fp32(_lib.ptr(a32), dim, _lib.ptr(an), m1, _lib.ptr(b32), dim, _lib.ptr(bn),
                                             m2, dim, flags, _lib.ptr(out), int(out.stride(0)), _lib.stream_ptr()), "pps_dist_fp32")
            else:
                planes = _lib.PLANES_FOR[prec]
                scaled = prec == _lib.PREC_F16X3 and a.dtype == torch.float32 and b.dtype == torch.float32
                sa, sb = SplitOperand(a, planes, scaled), SplitOperand(b, planes, scaled)
                dist_block(sa, sb, prec, out, flags)
    if a_np and b_np:
        return out.cpu().numpy()
    return out


# ------------------------------------------------------------------------------------
# reference-shaped metric entry points on a materialised distance matrix
# ------------------------------------------------------------------------------------
def _ensure_arrays(distmat, query_ids, gallery_ids, query_cams, gallery_cams):
    torch = _torch()
    ok = lambda a: isinstance(a, np.ndarray) or isinstance(a, torch.Tensor)
    assert ok(distmat)
    assert ok(query_ids)
    assert ok(gallery_ids)
    assert ok(query_cams)
    assert ok(gallery_cams)


def cmc(distmat, query_ids=None, gallery_ids=None, query_cams=None, gallery_cams=None, topk=100,
        separate_camera_set=False, single_gallery_shot=False, first_match_break=False, average=True):
    """reid_dataset_evaluator.py:283-363.

    ``separate_camera_set=True`` (:329-331) removes EVERY gallery item taken by the query's camera, whatever its id: the
    queries are grouped by camera and each group is ranked against the columns of the other cameras (nothing is junk
    then).  ``single_gallery_shot=True`` is the one branch that is not provided: it averages 100 np.random.choice draws
    per query and calls the removed ``np.bool`` (:274-279, :334-347) - it does not run in the reference either under the
    installed numpy - and the evaluator never selects it (:35-37).
    """
    _ensure_arrays(distmat, query_ids, gallery_ids, query_cams, gallery_cams)
    if single_gallery_shot:
        raise NotImplementedError("cmc: single_gallery_shot is not on the PPS eval path (reid_dataset_evaluator.py:35-37 fixes "
                                  "it to False; the branch draws random samples and calls the removed np.bool)")
    if separate_camera_set:
        return _cmc_separate_camera_set(distmat, query_ids, gallery_ids, query_cams, gallery_cams, topk, first_match_break,
                                        average)
    res = rank_distmat(distmat, query_ids, gallery_ids, query_cams, gallery_cams,
                       want_neg_before=not first_match_break)
    return res.cmc(topk=topk, first_match_break=first_match_break, average=average)


def _cmc_separate_camera_set(distmat, query_ids, gallery_ids, query_cams, gallery_cams, topk, first_match_break, average):
    torch = _torch()
    dist, _ = _as_cuda_f32(distmat, "distmat")
    qi, qc = _ids64(query_ids, "query_ids"), _ids64(query_cams, "query_cams")
    gi, gc = _ids64(gallery_ids, "gallery_ids"), _ids64(gallery_cams, "gallery_cams")
    m = int(dist.shape[0])
    if len(qi) != m or len(gi) != int(dist.shape[1]):
        raise RuntimeError("distmat shape %s does not match %d query / %d gallery ids" % (tuple(dist.shape), len(qi), len(gi)))
    ret = np.zeros([m, topk])
    is_valid = np.zeros(m)
    for cam in np.unique(qc):
        rows = np.nonzero(qc == cam)[0]
        cols = np.nonzero(gc != cam)[0]
        if len(cols) == 0:
            continue
        sub = dist[torch.from_numpy(rows).to(dist.device)][:, torch.from_numpy(cols).to(dist.device)].contiguous()
        res = rank_distmat(sub, qi[rows], gi[cols], qc[rows], gc[cols], want_neg_before=not first_match_break)
        ret[rows] = res.cmc_matrix(topk, first_match_break)
        is_valid[rows] = res.is_valid
    num_valid = int(is_valid.sum())
    if num_valid == 0:
        raise RuntimeError("No valid query")                 # :358-359
    if average:
        return np.sum(ret, axis=0) / num_valid
    return ret, is_valid


def mean_ap(distmat, query_ids=None, gallery_ids=None, query_cams=None, gallery_cams=None, average=True,
            ap_definition="step"):
    """reid_dataset_evaluator.py:366-439.  ``ap_definition='step'``: the AP of scikit-learn >= 0.19 (what an unpinned
    install computes); ``'trapezoid'``: the scikit-learn 0.18.1 AP the reference asks for at :398-407."""
    _ensure_arrays(distmat, query_ids, gallery_ids, query_cams, gallery_cams)
    res = rank_distmat(distmat, query_ids, gallery_ids, query_cams, gallery_cams, ap_definition=ap_definition)
    if average:
        return res.mean_ap()
    return res.ap, res.is_valid.astype(np.float64)


# ------------------------------------------------------------------------------------
# fused path: features -> metrics
# ------------------------------------------------------------------------------------
class _DevArray:
    """A raw device pointer dressed as a __cuda_array_interface__ object (so torch can alias library-owned memory)."""

    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (int(ptr), False), "version": 2}


_WRAPPED = {}


def _wrap_device(torch, ptr, n, typestr, dtype, device):
    """torch tensor aliasing `n` elements of library-owned device memory (cached: the buffers of a ctx are grow-only, so the
    same (pointer, length) comes back pass after pass and the __cuda_array_interface__ round trip is paid once)."""
    key = (int(ptr), int(n), typestr, str(device))
    t = _WRAPPED.get(key)
    if t is None:
        if len(_WRAPPED) > 64:
            _WRAPPED.clear()
        t = torch.as_tensor(_DevArray(ptr, n, typestr), device=device)
        assert t.dtype == dtype and t.data_ptr() == ptr
        _WRAPPED[key] = t
    return t


class RankEngine:
    """Preallocated state for repeated distance + rank passes over one (query set, gallery shard) shape.

    ``run(q, g)`` takes CUDA feature tensors ([nq, D] and this rank's [ng_local, D] gallery shard starting at
    global row ``gallery_offset``) and returns a RankResult.  Every pass rebuilds the same-id pair lists from
    the id / camera arrays (the junk mask and the matches are part of the timed path), splits the operands,
    runs the tcgen05 distance per gallery chunk and the two rank sweeps:
      sweep 1  gather the positives' / junk distances (the thresholds)        [all-reduce SUM over shards]
      sweep 2  count <= thresholds, first-match counter, top-k                [all-reduce SUM, all-gather]
    With one chunk the distance block of sweep 1 is reused by sweep 2.
    """

    def __init__(self, query_ids, gallery_ids, query_cams, gallery_cams, nq, ng_local, dim, gallery_offset=0,
                 precision=DEFAULT_PRECISION, topk=0, topk_filtered=True, want_neg_before=False, group=None,
                 device=None, max_block_bytes=8 << 30, in_dtype=None):
        torch = _torch()
        self.lib = _lib.load()
        self.torch = torch
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.qi, self.qc = _ids64(query_ids, "query_ids"), _ids64(query_cams, "query_cams")
        self.gi, self.gc = _ids64(gallery_ids, "gallery_ids"), _ids64(gallery_cams, "gallery_cams")
        self.nq, self.ngl, self.dim = int(nq), int(ng_local), int(dim)
        if len(self.qi) != self.nq:
            raise RuntimeError("q_feats has %d rows but %d query ids" % (self.nq, len(self.qi)))
        if group is None and len(self.gi) != self.ngl:
            raise RuntimeError("g_feats has %d rows but %d gallery ids" % (self.ngl, len(self.gi)))
        self.offset, self.group = int(gallery_offset), group
        self.max_block_bytes = int(max_block_bytes)
        self.topk, self.topk_filtered, self.want_neg_before = int(topk), topk_filtered, want_neg_before
        self.is_f16 = in_dtype == torch.float16
        self.prec = _lib.PREC_F16X1 if self.is_f16 else _prec_code(precision)
        if self.prec == _lib.PREC_FP32:
            raise RuntimeError("rank_eval runs the distance on the tensor cores; use bf16x1/bf16x3/bf16x6 (or fp16 inputs)")
        self.planes = _lib.PLANES_FOR[self.prec]
        self.split_arg = _lib.split_planes_arg(self.prec)        # `planes` argument of the split calls
        self.in_code = _lib.DTYPE_F16 if self.is_f16 else _lib.DTYPE_F32
        nq_, ngl_ = max(self.nq, 1), self.ngl
        chunk = ngl_ if self.nq == 0 else max(256, min(ngl_, max_block_bytes // (4 * nq_)))
        chunk = max(256, (chunk // 256) * 256) if chunk < ngl_ else ngl_
        self.chunk = chunk
        self.n_chunks = (ngl_ + chunk - 1) // chunk if ngl_ else 0
        self.ldd = (max(min(chunk, max(ngl_, 1)), 1) + 3) // 4 * 4
        lib, dev = self.lib, self.dev
        with torch.cuda.device(dev):
            e8 = lambda n: torch.empty(max(int(n), 16), dtype=torch.uint8, device=dev)
            self.q_planes = e8(lib.pps_split_bytes(nq_, self.dim, self.planes))
            self.g_planes = e8(lib.pps_split_bytes(max(chunk, 1), self.dim, self.planes))
            self.q_sq = torch.empty(2 * nq_, dtype=torch.float32, device=dev)           # norms (+ 'f16x3' row scales)
            self.g_sq = torch.empty(2 * max(chunk, 1), dtype=torch.float32, device=dev)
            self.block = torch.empty((nq_, self.ldd), dtype=torch.float32, device=dev)
            self.cnt_first = torch.zeros(nq_, dtype=torch.int32, device=dev)
            self.key = torch.empty((nq_, self.topk), dtype=torch.int64, device=dev) if self.topk else None
            self.pairs = DevicePairs(self.qi, self.qc, self.gi, self.gc, dev)
        self._pair_cap = 0
        self.kernel_events = None        # bench.py: list collecting (start, stop) events around the distance GEMM
        self.use_c_path = False          # True: one device, one block, no top-k through the single C call pps_evaluate_device_ctx
                                         # (round 1's fast path; the speculative pass below measured faster: 0.864 vs 0.883 ms)
        self.use_c_pass = True           # everything else (several blocks, top-k, sharded): pps_pass_begin / _count / _end
        self.tk_cap = 0                  # test hook: top-k candidate entries per query of the C pass (0 = default 2048)
        self._gathered = None
        self._gathered_x1 = None
        self._res_ring, self._res_turn = None, 0
        self.trace = None                # list collecting (name, cuda event, host time) marks of _run_pass when set
        self._stage = None               # device staging of run_host
        self._cnt_all = None
        self._side = None
        self.h2d_bytes = 0
        self.compact_thresholds = True   # multi-chunk galleries: thresholds from the compacted same-id gallery
        self._g_ptr, self._g_keepalive = None, None
        self._c_fixed = {}
        self.fused_topk = True           # blocks after the first: top-k admission in the distance epilogue
        self.used_fused_topk = False
        self.fused_count = os.environ.get("PPS_NO_FUSED_COUNT", "0") != "1"   # C pass, single-plane operands (fp16 rows), several blocks: counters AND top-k admission
                                         # in the distance epilogue, so no block after the first is written (pps_dist_rank_topk_tc)
        self.used_fused_count = False
        self.pass_blocks = 0
        self._tk = None
        self.fused_rank = False          # counters in the epilogue of the distance kernel (no distance block written):
                                         # bit-identical, saves the block's memory, but measured slower than block +
                                         # count kernel on B200 (the MMA mainloop already saturates shared-memory bandwidth)
        self.used_fused_rank = False
        self._tab = None
        self._gp_cap, self._gp_rows, self._pair_col, self._gp_ws = 0, None, None, None
        self.threshold_rows = 0

    # -- helpers --
    def _pair_buffers(self, n_pairs):
        """(pair_d, cnt_le) with capacity >= n_pairs; the pair fill kernel zero-fills the used part."""
        torch = self.torch
        if n_pairs > self._pair_cap or self._pair_cap == 0:
            cap = max(int(n_pairs * 1.25), 1024)
            self.pair_d = torch.zeros(cap, dtype=torch.float32, device=self.dev)
            self.cnt_le = torch.zeros(cap, dtype=torch.int32, device=self.dev)
            self._pair_cap = cap
        return self.pair_d, self.cnt_le

    def _finish_pairs(self, pairs):
        pairs.finish(zero_f32=lambda n: self._pair_buffers(n)[0], zero_u32=lambda n: self._pair_buffers(n)[1],
                     zero_per_query=self.cnt_first)
        return self.pair_d, self.cnt_le

    def set_phase_timing(self, enabled: bool):
        """Device-time the phases of the C fast path (pps_ctx_set_timing); read them with last_phase_ms()."""
        _lib.check(self.lib.pps_ctx_set_timing(_host_ctx(self.dev.index or 0), 1 if enabled else 0), "pps_ctx_set_timing")

    def last_phase_ms(self):
        out = np.zeros(_lib.N_PHASES, dtype=np.float32)
        _lib.check(self.lib.pps_ctx_phase_ms(_host_ctx(self.dev.index or 0), _lib.ptr(out)), "pps_ctx_phase_ms")
        return dict(zip(_lib.PHASE_NAMES, out.tolist()))

    def _run_resident_c(self, q, g):
        """One gallery block per rank: the pass is four C calls (pps_rank_begin / _distance / _count_local / _end) with,
        for a sharded gallery, the three NCCL exchanges in between: all-gather of the per-query local pair counts,
        all-reduce of the thresholds (+ pair metadata), all-reduce of the integer counters."""
        torch = self.torch
        nq, topk = self.nq, self.topk
        p = self.pairs
        ctx = _host_ctx(self.dev.index or 0)
        s = _lib.stream_ptr()
        sharded = self.group is not None
        world = rank = None
        if sharded:
            import torch.distributed as dist_mod
            world, rank = dist_mod.get_world_size(self.group), dist_mod.get_rank(self.group)
        if not sharded:
            # one C call: begin -> thresholds -> count -> end (no exchange points needed)
            out_map = C.c_double(0.0)
            out_cmc = np.empty(10, dtype=np.float64)
            ap = np.empty(nq, dtype=np.float64)
            valid = np.empty(nq, dtype=np.uint8)
            first = np.empty(nq, dtype=np.int32)
            ti = np.empty((nq, topk), dtype=np.int32) if topk else None
            td = np.empty((nq, topk), dtype=np.float32) if topk else None
            key = (q.data_ptr(), g.data_ptr())
            fixed = self._c_fixed.get(key)
            if fixed is None:                    # the input-side arguments of the call, converted once per buffer pair
                self._c_fixed.clear()
                fixed = self._c_fixed[key] = (ctx, _lib.ptr(q), nq, _lib.ptr(g), self.ngl, self.dim, _lib.ptr(p.qid),
                                              _lib.ptr(p.qcam), _lib.ptr(p.gid), _lib.ptr(p.gcam), self.prec, 10, topk)
            rc = self.lib.pps_evaluate_device_ctx(*fixed, s, C.cast(C.byref(out_map), C.c_void_p), out_cmc.ctypes.data, ap.ctypes.data,
                                                  valid.ctypes.data, first.ctypes.data, ti.ctypes.data if topk else None,
                                                  td.ctypes.data if topk else None)
            if rc != _lib.PPS_ERR_NO_VALID_QUERY:
                _lib.check(rc, "pps_evaluate_device_ctx")
            return RankResult(ap, valid, first, None, None, ti, td)
        gid_l = p.gid[self.offset:self.offset + self.ngl] if sharded else p.gid
        gcam_l = p.gcam[self.offset:self.offset + self.ngl] if sharded else p.gcam
        d_lc = C.c_void_p(0)
        side = None
        if sharded:
            if self._side is None:
                self._side = torch.cuda.Stream(device=self.dev)
            side = self._side
        _lib.check(self.lib.pps_rank_begin(ctx, _lib.ptr(q), nq, _lib.ptr(g), self.ngl, self.dim, _lib.ptr(p.qid),
                                           _lib.ptr(p.qcam), _lib.ptr(gid_l), _lib.ptr(gcam_l), self.offset,
                                           world if sharded else 1, self.prec, topk, s,
                                           C.c_void_p(side.cuda_stream) if side is not None else None, C.byref(d_lc)),
                   "pps_rank_begin")
        cnt_all = None
        if sharded:
            # the local pair counts were launched on the side stream; gather them there too, so that the pair-list
            # work (count -> all-gather -> offsets -> fill) overlaps the split + GEMM on the main stream
            local_cnt = _wrap_device(torch, d_lc.value, nq, "<i4", torch.int32, self.dev)
            if self._cnt_all is None:
                self._cnt_all = torch.empty((world, nq), dtype=torch.int32, device=self.dev)
            cnt_all = self._cnt_all
            with torch.cuda.stream(side):
                dist_mod.all_gather_into_tensor(cnt_all.view(-1), local_cnt, group=self.group)
        n_pairs, n_words, n_cnt = C.c_longlong(0), C.c_longlong(0), C.c_longlong(0)
        d_x, d_cnt = C.c_void_p(0), C.c_void_p(0)
        _lib.check(self.lib.pps_rank_thresholds(ctx, _lib.ptr(cnt_all), rank if sharded else 0, s, C.byref(n_pairs),
                                              C.byref(d_x), C.byref(n_words)), "pps_rank_thresholds")
        if sharded and n_words.value:
            xbuf = _wrap_device(torch, d_x.value, n_words.value, "<i4", torch.int32, self.dev)
            dist_mod.all_reduce(xbuf, op=dist_mod.ReduceOp.SUM, group=self.group)
        _lib.check(self.lib.pps_rank_count_local(ctx, s, C.byref(d_cnt), C.byref(n_cnt)), "pps_rank_count_local")
        if sharded:
            counters = _wrap_device(torch, d_cnt.value, n_cnt.value, "<i4", torch.int32, self.dev)
            dist_mod.all_reduce(counters, op=dist_mod.ReduceOp.SUM, group=self.group)
        out_map = C.c_double(0.0)
        out_cmc = np.zeros(10, dtype=np.float64)
        ap = np.zeros(nq, dtype=np.float64)
        valid = np.zeros(nq, dtype=np.uint8)
        first = np.zeros(nq, dtype=np.int32)
        ti = np.zeros((nq, topk), dtype=np.int32) if topk else None
        td = np.zeros((nq, topk), dtype=np.float32) if topk else None
        rc = self.lib.pps_rank_end(ctx, 10, s, C.cast(C.byref(out_map), C.c_void_p), _lib.ptr(out_cmc), _lib.ptr(ap),
                                   _lib.ptr(valid), _lib.ptr(first), _lib.ptr(ti), _lib.ptr(td))
        if rc != _lib.PPS_ERR_NO_VALID_QUERY:
            _lib.check(rc, "pps_rank_end")
        return RankResult(ap, valid, first, None, None, ti, td)

    def _run_pass(self, q, g):
        """The pass driven from C (csrc/pass.cu): pair lists from the global id vectors, blocks, top-k admission, and - for
        a sharded gallery - exactly two collectives: all-reduce(SUM) of the thresholds, all-gather of
        [top-k keys | counters | flags] (reduced / merged by the library's own kernels in pps_pass_end)."""
        torch, lib = self.torch, self.lib
        nq, topk = self.nq, self.topk
        p = self.pairs
        ctx = _host_ctx(self.dev.index or 0)
        s = _lib.stream_ptr()
        sharded = self.group is not None
        world, rank = 1, 0
        if sharded:
            import torch.distributed as dist_mod
            world, rank = dist_mod.get_world_size(self.group), dist_mod.get_rank(self.group)
        flags = (0 if self.fused_topk else _lib.PASS_NO_EPILOGUE_TOPK) | ((int(self.tk_cap) & 0xffff) << 8)
        if not self.fused_count:
            flags |= _lib.PASS_NO_FUSED_COUNT
        tr = self.trace                  # optional: CUDA events + host clocks around the segments of the pass (tools/pass_trace.py)
        import time as _time

        def mark(name):
            if tr is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                tr.append((name, ev, _time.perf_counter()))
        for attempt in (0, 1, 2):
            mark("start")
            d_x1, n_x1 = C.c_void_p(0), C.c_longlong(0)
            _lib.check(lib.pps_pass_begin(ctx, _lib.ptr(q), nq, _lib.ptr(g) if self.ngl else None, self.ngl, self.dim, self.in_code,
                                          _lib.ptr(p.qid), _lib.ptr(p.qcam), _lib.ptr(p.gid), _lib.ptr(p.gcam), len(self.gi),
                                          self.offset, world, rank, self.prec, topk, self.max_block_bytes, flags, s,
                                          C.byref(d_x1), C.byref(n_x1)), "pps_pass_begin")
            mark("begin_done")
            g1 = None
            if sharded and n_x1.value:
                x1 = _wrap_device(torch, d_x1.value, n_x1.value, "<i4", torch.int32, self.dev)
                if self._gathered_x1 is None or self._gathered_x1.numel() != world * n_x1.value:
                    self._gathered_x1 = torch.empty(world * n_x1.value, dtype=torch.int32, device=self.dev)
                g1 = self._gathered_x1
                dist_mod.all_gather_into_tensor(g1, x1, group=self.group)
            mark("x1_done")
            d_x2, nb = C.c_void_p(0), C.c_longlong(0)
            _lib.check(lib.pps_pass_count(ctx, _lib.ptr(g1), s, C.byref(d_x2), C.byref(nb)), "pps_pass_count")
            mark("count_done")
            gathered = None
            if sharded:
                packed = _wrap_device(torch, d_x2.value, nb.value, "|u1", torch.uint8, self.dev)
                if self._gathered is None or self._gathered.numel() != world * nb.value:
                    self._gathered = torch.empty(world * nb.value, dtype=torch.uint8, device=self.dev)
                gathered = self._gathered
                dist_mod.all_gather_into_tensor(gathered, packed, group=self.group)
            mark("x2_done")
            out_map = C.c_double(0.0)
            out_cmc = np.zeros(10, dtype=np.float64)
            ap = np.zeros(nq, dtype=np.float64)
            valid = np.zeros(nq, dtype=np.uint8)
            first = np.zeros(nq, dtype=np.int32)
            ti = td = None
            if topk:
                # the top-k lists (MBs) come back into PINNED arrays: a device -> pageable copy runs at a fraction of the
                # PCIe rate.  Two sets, used alternately: a result stays valid until the second-next pass of this engine.
                if self._res_ring is None:
                    mk = lambda dt: torch.empty((max(nq, 1), topk), dtype=dt).pin_memory()
                    self._res_ring = [(mk(torch.int32), mk(torch.float32)) for _ in range(2)]
                self._res_turn ^= 1
                ti, td = (t.numpy()[:nq] for t in self._res_ring[self._res_turn])
            rc = lib.pps_pass_end(ctx, _lib.ptr(gathered), 10, s, C.cast(C.byref(out_map), C.c_void_p), _lib.ptr(out_cmc),
                                  _lib.ptr(ap), _lib.ptr(valid), _lib.ptr(first), _lib.ptr(ti), _lib.ptr(td))
            mark("end_done")
            self.used_fused_topk = bool(topk and not (flags & _lib.PASS_NO_EPILOGUE_TOPK))
            self.used_fused_count = bool(lib.pps_pass_stat(ctx, 1) == 1)
            self.pass_blocks = int(lib.pps_pass_stat(ctx, 0))      # (the C plan also splits a gallery that fits one block)
            if rc == _lib.PPS_ERR_PASS_RESIZE and not (flags & _lib.PASS_SIZING):
                # the speculative size bounds (taken from the last sizing pass of this shape) were too small - the ids
                # changed: every rank sees the same flag and repeats the pass as a sizing pass
                flags |= _lib.PASS_SIZING
                continue
            if rc == _lib.PPS_ERR_TOPK_OVERFLOW and not (flags & _lib.PASS_NO_EPILOGUE_TOPK):
                # a candidate buffer ran over (adversarial column order): every rank sees the same flag (it travels in the
                # gathered buffers), so every rank repeats the pass with the one-read sweep
                flags |= _lib.PASS_NO_EPILOGUE_TOPK
                continue
            if rc != _lib.PPS_ERR_NO_VALID_QUERY:
                _lib.check(rc, "pps_pass_end")
            return RankResult(ap, valid, first, None, None, ti, td)

    def _split(self, feats, rows, planes_buf, sq_buf):
        if planes_buf is self.g_planes:
            self._g_ptr = _lib.ptr(self.g_planes)
        if rows:
            if feats.stride(1) != 1:
                feats = feats.contiguous()
            if (planes_buf is self.g_planes and self.is_f16 and self.dim % 64 == 0 and int(feats.stride(0)) == self.dim
                    and feats.data_ptr() % 16 == 0):
                # fp16 rows that already are a K-major operand plane: no copy, only the row norms
                self._g_ptr = _lib.ptr(feats)
                self._g_keepalive = feats
                _lib.check(self.lib.pps_row_sqnorm(_lib.ptr(feats), self.in_code, rows, self.dim, self.dim, _lib.ptr(sq_buf),
                                                   _lib.stream_ptr()), "pps_row_sqnorm")
                return
            _lib.check(self.lib.pps_split_rows(_lib.ptr(feats), self.in_code, rows, self.dim, int(feats.stride(0)),
                                               self.split_arg, _lib.ptr(planes_buf), _lib.ptr(sq_buf), _lib.stream_ptr()),
                       "pps_split_rows")

    def _fused_count_sweep(self, g, chunks, pairs, pair_d, cnt_le, cnt_first):
        torch, lib = self.torch, self.lib
        nq = self.nq
        p_cap = max(8, (pairs.max_pairs + 7) // 8 * 8)
        elems = int(lib.pps_rank_tab_elems(nq, p_cap))
        if self._tab is None or self._tab[0] < elems:
            mk = lambda dt, n: torch.empty(n, dtype=dt, device=self.dev)
            self._tab = (elems, mk(torch.float32, elems), mk(torch.int32, elems), mk(torch.int32, elems),
                         mk(torch.float32, max(nq, 1)), mk(torch.int32, max(nq, 1)), mk(torch.int32, 1))
        _, thr, tpair, cnt, dstar, gstar, ovf = self._tab
        s = _lib.stream_ptr()
        _lib.check(lib.pps_rank_tab_prep(nq, _lib.ptr(pairs.dev("off")), _lib.ptr(pairs.dev("g")), _lib.ptr(pairs.dev("pos")),
                                         _lib.ptr(pair_d), p_cap, _lib.ptr(thr), _lib.ptr(tpair), _lib.ptr(cnt),
                                         _lib.ptr(dstar), _lib.ptr(gstar), _lib.ptr(ovf), s), "pps_rank_tab_prep")
        for r0, rows in chunks:
            self._split(g[r0:r0 + rows], rows, self.g_planes, self.g_sq)
            ev = None
            if self.kernel_events is not None:
                ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                ev[0].record()
            _lib.check(lib.pps_dist_rank_tc(_lib.ptr(self.q_planes), _lib.ptr(self.q_sq), nq, self.planes, 0,
                                            self._g_ptr, _lib.ptr(self.g_sq), rows, self.planes, 0, self.dim,
                                            self.prec, 0, self.offset + r0, p_cap, _lib.ptr(thr), _lib.ptr(cnt),
                                            _lib.ptr(dstar), _lib.ptr(gstar), _lib.ptr(cnt_first), s), "pps_dist_rank_tc")
            if ev is not None:
                ev[1].record()
                self.kernel_events.append(ev)
        _lib.check(lib.pps_rank_tab_finish(nq, p_cap, _lib.ptr(tpair), _lib.ptr(cnt), _lib.ptr(cnt_le), s),
                   "pps_rank_tab_finish")

    def _threshold_pass(self, g, pairs, pair_d):
        """pair_d[e] = d(query, gallery row) for every same-id pair whose row lives in this shard, from the product
        queries x (the distinct rows that appear in a pair) — pps_pairs_compact_rows + pps_split_rows_gather."""
        torch, lib = self.torch, self.lib
        n = pairs.n_pairs
        if self._gp_cap < n:
            self._gp_cap = max(int(n * 1.25), 1024)
            self._gp_rows = torch.empty(self._gp_cap, dtype=torch.int32, device=self.dev)
            self._pair_col = torch.empty(self._gp_cap, dtype=torch.int32, device=self.dev)
        if self._gp_ws is None:
            self._gp_ws = torch.empty(int(lib.pps_pairs_compact_workspace_bytes(self.nq)), dtype=torch.uint8, device=self.dev)
            self._gp_n_d = torch.zeros(1, dtype=torch.int32, device=self.dev)
            self._gp_n_h = torch.zeros(1, dtype=torch.int32).pin_memory()
        s = _lib.stream_ptr()
        _lib.check(lib.pps_pairs_compact_rows(_lib.ptr(pairs.qid), self.nq, _lib.ptr(pairs.dev("off")),
                                              _lib.ptr(pairs.dev("q")), _lib.ptr(pairs.dev("g")), n, self.offset,
                                              self.offset + self.ngl, _lib.ptr(self._gp_ws), _lib.ptr(self._gp_rows),
                                              _lib.ptr(self._pair_col), _lib.ptr(self._gp_n_d), s),
                   "pps_pairs_compact_rows")
        self._gp_n_h.copy_(self._gp_n_d, non_blocking=True)
        torch.cuda.current_stream().synchronize()          # 4 bytes: the row count sizes the product
        n_rows = int(self._gp_n_h[0])
        self.threshold_rows = n_rows
        if g.stride(1) != 1:
            g = g.contiguous()
        for c0 in range(0, n_rows, self.chunk):
            rows = min(self.chunk, n_rows - c0)
            self._g_ptr = _lib.ptr(self.g_planes)
            _lib.check(lib.pps_split_rows_gather(_lib.ptr(g), self.in_code, _lib.ptr(self._gp_rows[c0:]), self.offset, rows,
                                                 self.dim, int(g.stride(0)), self.split_arg, _lib.ptr(self.g_planes),
                                                 _lib.ptr(self.g_sq), s), "pps_split_rows_gather")
            self._distance(rows)
            _lib.check(lib.pps_rank_gather(_lib.ptr(self.block), self.ldd, self.nq, rows, c0, _lib.ptr(pairs.dev("q")),
                                           _lib.ptr(self._pair_col), n, _lib.ptr(pair_d), s), "pps_rank_gather")

    TOPK_CAND_CAP = 2048             # candidates per query and block the distance epilogue may append

    def _chunk_list(self):
        """(row0, rows) of the gallery blocks of one pass (see plan_blocks)."""
        short_first = bool(self.fused_topk and self.topk and DIST_KERNEL_FLAGS == 0)
        return plan_blocks(self.ngl, self.chunk, self.topk if short_first else 0, self.TOPK_CAND_CAP)

    def _topk_epilogue_begin(self, key):
        torch = self.torch
        if self._tk is None:
            nq_ = max(self.nq, 1)
            self._tk = (torch.empty(nq_, dtype=torch.int32, device=self.dev), torch.empty(nq_, dtype=torch.int32, device=self.dev),
                        torch.empty((nq_, self.TOPK_CAND_CAP), dtype=torch.int64, device=self.dev),
                        torch.zeros(1, dtype=torch.int32, device=self.dev))
        bound, cnt, _, ovf = self._tk
        ovf.zero_()
        _lib.check(self.lib.pps_topk_bound(_lib.ptr(key), self.nq, self.topk, _lib.ptr(bound), _lib.ptr(cnt), _lib.stream_ptr()),
                   "pps_topk_bound")

    def _topk_epilogue_merge(self, key, pairs):
        bound, cnt, cand, ovf = self._tk
        use = self.topk_filtered and pairs.n_pairs > 0
        _lib.check(self.lib.pps_topk_merge(_lib.ptr(key), self.nq, self.topk, _lib.ptr(cand), self.TOPK_CAND_CAP, _lib.ptr(cnt),
                                           _lib.ptr(bound), _lib.ptr(pairs.dev("off")), _lib.ptr(pairs.dev("g")) if use else None,
                                           _lib.ptr(pairs.dev("pos")) if use else None, pairs.max_pairs if use else 0,
                                           1 if use else 0, _lib.ptr(ovf), _lib.stream_ptr()), "pps_topk_merge")

    def _distance(self, rows, topk_col0=None):
        torch = self.torch
        ev = None
        if self.kernel_events is not None:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
        if topk_col0 is not None:
            bound, cnt, cand, _ = self._tk
            _lib.check(self.lib.pps_dist_topk_tc(_lib.ptr(self.q_planes), _lib.ptr(self.q_sq), self.nq, self.planes, 0,
                                                 self._g_ptr, _lib.ptr(self.g_sq), rows, self.planes, 0, self.dim,
                                                 self.prec, DIST_KERNEL_FLAGS, _lib.ptr(self.block), self.ldd, topk_col0,
                                                 _lib.ptr(bound), _lib.ptr(cnt), _lib.ptr(cand), self.TOPK_CAND_CAP,
                                                 _lib.stream_ptr()), "pps_dist_topk_tc")
        else:
            _lib.check(self.lib.pps_dist_tc(_lib.ptr(self.q_planes), _lib.ptr(self.q_sq), self.nq, self.planes, 0,
                                            self._g_ptr, _lib.ptr(self.g_sq), rows, self.planes, 0, self.dim,
                                            self.prec, DIST_KERNEL_FLAGS, _lib.ptr(self.block), self.ldd,
                                            _lib.stream_ptr()), "pps_dist_tc")
        if ev is not None:
            ev[1].record()
            self.kernel_events.append(ev)

    def run(self, q, g) -> RankResult:
        torch, lib = self.torch, self.lib
        want = torch.float16 if self.is_f16 else torch.float32
        if q.dtype != want or g.dtype != want or not q.is_cuda or not g.is_cuda:
            raise RuntimeError("RankEngine.run: expected CUDA %s features" % want)
        if tuple(q.shape) != (self.nq, self.dim) or tuple(g.shape) != (self.ngl, self.dim):
            raise RuntimeError("RankEngine.run: expected q %s and g %s, got %s and %s" % (
                (self.nq, self.dim), (self.ngl, self.dim), tuple(q.shape), tuple(g.shape)))
        dist_mod = None
        if self.group is not None:
            import torch.distributed as dist_mod
        nq = self.nq
        # Which path runs depends only on options that are the same on every rank of a sharded run (never on the shard).
        plain = (not self.want_neg_before and self.topk_filtered and nq > 0 and self.kernel_events is None
                 and not self.fused_rank and DIST_KERNEL_FLAGS == 0 and q.is_contiguous() and g.is_contiguous())
        if (plain and self.use_c_path and self.group is None and self.n_chunks == 1 and self.topk == 0 and not self.is_f16
                and self.ngl > 0):
            with torch.cuda.device(self.dev):
                return self._run_resident_c(q, g)
        if plain and self.use_c_pass:
            with torch.cuda.device(self.dev):
                return self._run_pass(q, g)
        with torch.cuda.device(self.dev):
            pairs = self.pairs.begin()          # junk mask / matches from the resident ids, on the device
            key = self.key
            if self.topk:
                _lib.check(lib.pps_topk_init(_lib.ptr(key), nq, self.topk, _lib.stream_ptr()), "pps_topk_init")
            self._split(q, nq, self.q_planes, self.q_sq)
            chunks = self._chunk_list()
            # sweep 1: thresholds
            first_chunk = True
            pair_d = cnt_le = None
            cnt_first = self.cnt_first
            if self.n_chunks > 1 and self.compact_thresholds:
                # The thresholds are the distances of the same-id pairs only: one dense product of the queries with
                # just the gallery rows that appear in a pair (a few 10^4 rows however large the gallery is), with
                # the same kernel and operands as sweep 2 (bit-identical values), instead of a sweep over every chunk.
                pair_d, cnt_le = self._finish_pairs(pairs)
                first_chunk = False
                if pairs.n_pairs:
                    self._threshold_pass(g, pairs, pair_d)
            else:
                for r0, rows in chunks:
                    self._split(g[r0:r0 + rows], rows, self.g_planes, self.g_sq)
                    self._distance(rows)
                    if first_chunk:                 # the pair count came back while the GEMM was queued / running
                        pair_d, cnt_le = self._finish_pairs(pairs)
                        first_chunk = False
                    _rank_block(lib, self.block, self.ldd, nq, rows, self.offset + r0, pairs, pair_d, cnt_le, cnt_first,
                                True, False)
            if first_chunk:                     # empty gallery shard
                pair_d, cnt_le = self._finish_pairs(pairs)
            if self.group is not None:
                dist_mod.all_reduce(pair_d, op=dist_mod.ReduceOp.SUM, group=self.group)
            # sweep 2: counts (+ top-k); a single chunk is still resident in the block
            fused = (self.fused_rank and self.n_chunks > 1 and not self.topk and pairs.n_pairs > 0
                     and pairs.max_pairs <= 64 and self.prec != _lib.PREC_F16X3)
            self.used_fused_rank = bool(fused)
            if fused:
                # thresholds are known: the counters are taken in the epilogue of the distance kernel and the
                # distance blocks are never written (pps_dist_rank_tc)
                self._fused_count_sweep(g, chunks, pairs, pair_d, cnt_le, cnt_first)
                chunks = []
            # Blocks after the first: the top-k candidates are admitted by the EPILOGUE of the distance kernel (one
            # compare per element against the bound the first block's sweep established) and the block is only
            # counted, instead of being swept for counts and top-k together.
            epi_topk = bool(self.fused_topk and self.topk and self.n_chunks > 1 and chunks and DIST_KERNEL_FLAGS == 0)
            self.used_fused_topk = epi_topk
            for ci, (r0, rows) in enumerate(chunks):
                if self.n_chunks > 1:
                    self._split(g[r0:r0 + rows], rows, self.g_planes, self.g_sq)
                    if epi_topk and ci >= 1:
                        if ci == 1:
                            self._topk_epilogue_begin(key)
                        self._distance(rows, topk_col0=self.offset + r0)
                        _rank_block(lib, self.block, self.ldd, nq, rows, self.offset + r0, pairs, pair_d, cnt_le, cnt_first,
                                    False, True)
                        self._topk_epilogue_merge(key, pairs)
                        continue
                    self._distance(rows)
                _rank_block(lib, self.block, self.ldd, nq, rows, self.offset + r0, pairs, pair_d, cnt_le, cnt_first,
                            False, True, key, self.topk, self.topk_filtered)
            overflow = False
            may_epi = bool(self.fused_topk and self.topk and DIST_KERNEL_FLAGS == 0)    # the same on every rank
            if may_epi and (epi_topk or self.group is not None):
                # the decision to repeat must be the same on every rank (shards differ, so the flags do too): the flag is
                # max-reduced, and whether this exchange happens depends on options only, never on the shard
                flag = self._tk[3] if (epi_topk and len(chunks) > 1) else torch.zeros(1, dtype=torch.int32, device=self.dev)
                if self.group is not None:
                    flag = flag.clone()
                    dist_mod.all_reduce(flag, op=dist_mod.ReduceOp.MAX, group=self.group)
                overflow = int(flag.item()) != 0
            if overflow:
                # a candidate buffer ran over (adversarial column order): repeat the pass with the one-read sweep
                self.fused_topk = False
                try:
                    return self.run(q, g)
                finally:
                    self.fused_topk = True
            if self.group is not None:
                dist_mod.all_reduce(cnt_le, op=dist_mod.ReduceOp.SUM, group=self.group)
                dist_mod.all_reduce(cnt_first, op=dist_mod.ReduceOp.SUM, group=self.group)
                if self.topk:
                    key = merge_topk_keys(key, self.topk, self.group)
            ap, valid, first, negb = _finalize(lib, nq, pairs, pair_d, cnt_le, cnt_first, self.want_neg_before)
            ti = td = None
            if self.topk:
                td = torch.empty((nq, self.topk), dtype=torch.float32, device=self.dev)
                ti = torch.empty((nq, self.topk), dtype=torch.int32, device=self.dev)
                _lib.check(lib.pps_topk_unpack(_lib.ptr(key), nq, self.topk, _lib.ptr(td), _lib.ptr(ti),
                                               _lib.stream_ptr()), "pps_topk_unpack")
                ti, td = ti.cpu().numpy(), td.cpu().numpy()
            return RankResult(ap.cpu().numpy(), valid.cpu().numpy(), first.cpu().numpy(),
                              negb.cpu().numpy() if negb is not None else None, pairs, ti, td)

    def run_host(self, q_host, g_host) -> RankResult:
        """Host (ideally pinned) feature tensors in: the H2D copies are part of the call.  Through the C pass the gallery
        goes up block by block (slab by slab when the shard is one block) on a copy stream, overlapping the split +
        distance of the rows that have already arrived (pps_pass_set_host_input)."""
        torch = self.torch
        want = torch.float16 if self.is_f16 else torch.float32
        for t, shape, name in ((q_host, (self.nq, self.dim), "q"), (g_host, (self.ngl, self.dim), "g")):
            if t.is_cuda or t.dtype != want or tuple(t.shape) != shape or not t.is_contiguous():
                raise RuntimeError("RankEngine.run_host: %s must be a contiguous host %s tensor of shape %s" % (name, want, shape))
        self.h2d_bytes = q_host.numel() * q_host.element_size() + g_host.numel() * g_host.element_size()
        with torch.cuda.device(self.dev):
            plain = (not self.want_neg_before and self.topk_filtered and self.nq > 0 and self.kernel_events is None
                     and not self.fused_rank and DIST_KERNEL_FLAGS == 0 and self.use_c_pass)
            if not plain:
                return self.run(q_host.to(self.dev, non_blocking=True), g_host.to(self.dev, non_blocking=True))
            if self._stage is None:
                self._stage = (torch.empty((self.nq, self.dim), dtype=want, device=self.dev),
                               torch.empty((max(self.ngl, 1), self.dim), dtype=want, device=self.dev))
            _lib.check(self.lib.pps_pass_set_host_input(_host_ctx(self.dev.index or 0), _lib.ptr(q_host),
                                                        _lib.ptr(g_host) if self.ngl else None), "pps_pass_set_host_input")
            return self._run_pass(self._stage[0], self._stage[1][:self.ngl])


def plan_blocks(ng_local, block_rows, topk=0, cand_cap=2048):
    """Gallery blocks [(row0, rows), ...] of one pass over ``ng_local`` rows in blocks of at most ``block_rows``.

    With top-k admission in the distance epilogue (``topk`` > 0) the FIRST block is kept short: it is the one that still
    takes the one-read sweep, and all it has to do is establish a bound tight enough that a full block admits well
    under ``cand_cap`` candidates per query (rows in random order: a block of R rows after F swept rows admits about
    k * R / F per query, so F >= 2.2 * k * R / cap, at least 32 768 rows)."""
    ng_local, block_rows = int(ng_local), int(block_rows)
    if ng_local <= 0:
        return []
    if ng_local <= block_rows:
        return [(0, ng_local)]
    first = block_rows
    if topk:
        want = int(2.2 * topk * block_rows / cand_cap)
        first = min(block_rows, max(32768, (want + 255) // 256 * 256))
    out, r0, rows = [], 0, min(first, ng_local)
    while r0 < ng_local:
        out.append((r0, rows))
        r0 += rows
        rows = min(block_rows, ng_local - r0)
    return out


def rank_eval(q_feats, g_feats, query_ids, gallery_ids, query_cams, gallery_cams, topk: int = 0,
              precision: str = DEFAULT_PRECISION, want_neg_before: bool = False, max_block_bytes: int = 8 << 30,
              gallery_offset: int = 0, group=None, topk_filtered: bool = True) -> RankResult:
    """distance + junk filter + exact positive ranks (+ top-k) without keeping the full matrix.

    q_feats [nq, D], g_feats [ng_local, D]: CUDA float32 / float16 tensors.  ``query_ids`` ... are
    the GLOBAL id / camera arrays.  With ``group`` (a torch.distributed group) every rank passes
    its contiguous gallery shard ``g_feats`` starting at global row ``gallery_offset``; the three
    exchanges are one sum-allreduce of the positives' distances, one of the integer counters and
    an all-gather of the top-k keys, so the merged result equals the unsharded one bit for bit.
    """
    torch = _torch()
    q, _ = _as_cuda_f32(q_feats, "q_feats")
    g, _ = _as_cuda_f32(g_feats, "g_feats")
    if q.shape[1] != g.shape[1]:
        raise RuntimeError("feature dims differ: %d vs %d" % (q.shape[1], g.shape[1]))
    if q.dtype != g.dtype:
        raise RuntimeError("query and gallery features must have the same dtype")
    with torch.cuda.device(q.device):
        eng = RankEngine(query_ids, gallery_ids, query_cams, gallery_cams, nq=int(q.shape[0]), ng_local=int(g.shape[0]),
                         dim=int(q.shape[1]), gallery_offset=gallery_offset, precision=precision, topk=topk,
                         topk_filtered=topk_filtered, want_neg_before=want_neg_before, group=group, device=q.device,
                         max_block_bytes=max_block_bytes, in_dtype=q.dtype)
        return eng.run(q, g)


def gallery_shard(ng, rank, world):
    """Contiguous row block of rank ``rank`` when ``ng`` gallery rows are split over ``world`` GPUs
    (the same np.array_split rule the reference uses to shard test images over GPUs:
    detectron/utils/subprocess.py:39-103).  Returns (row0, rows)."""
    base, extra = divmod(int(ng), int(world))
    rows = base + (1 if rank < extra else 0)
    row0 = rank * base + min(rank, extra)
    return row0, rows


def merge_topk_keys(key, topk, group):
    """All-gather every shard's [nq, k] candidate keys and keep the k smallest per query.

    Keys are (float bits << 32 | gallery index) of non-negative distances, so they are positive
    int64 values except the all-ones "empty" marker, which is mapped to INT64_MAX for the sort.
    """
    import torch
    import torch.distributed as dist_mod
    world = dist_mod.get_world_size(group)
    gathered = [torch.empty_like(key) for _ in range(world)]
    dist_mod.all_gather(gathered, key, group=group)
    return merge_key_lists(gathered, topk)


def merge_key_lists(keys, topk):
    """The k smallest of several [nq, k] top-k key lists per query (the merge step of merge_topk_keys)."""
    import torch
    allk = torch.cat(list(keys), dim=1)
    big = torch.iinfo(torch.int64).max
    allk = torch.where(allk == -1, torch.full_like(allk, big), allk)
    merged = torch.sort(allk, dim=1).values[:, :topk]
    return torch.where(merged == big, torch.full_like(merged, -1), merged).contiguous()


# ------------------------------------------------------------------------------------
# evaluate(): the reference's driver (single-query and multi-query branches)
# ------------------------------------------------------------------------------------
def parse_im_name(im_name, parse_type="id"):
    """reid_dataset_evaluator.py:224-231: '{pid:08d}_{cam:04d}_{k:08d}.jpg'."""
    assert parse_type in ("id", "cam")
    return int(im_name[:8]) if parse_type == "id" else int(im_name[9:13])


def get_info(entry):
    im_name = os.path.basename(entry["image"])
    return parse_im_name(im_name, "id"), parse_im_name(im_name, "cam"), im_name, entry["mark"], entry["image"]


def group_mean_rows(feats, groups):
    """np.stack([np.mean(feats[rows], axis=0) for rows in groups]) on the device (pps_group_mean_rows): float32 sums
    of the listed rows in order, one division by the count - the reference's multi-query pooling (:131-143)."""
    torch = _torch()
    lib = _lib.load()
    if not feats.is_cuda or feats.dtype != torch.float32 or feats.dim() != 2 or feats.stride(1) != 1:
        raise RuntimeError("group_mean_rows: expected a 2-D float32 CUDA tensor with unit column stride")
    off = np.zeros(len(groups) + 1, dtype=np.int32)
    off[1:] = np.cumsum([len(g) for g in groups])
    idx = np.asarray([r for g in groups for r in g], dtype=np.int32)
    out = torch.empty((len(groups), int(feats.shape[1])), dtype=torch.float32, device=feats.device)
    if len(groups):
        off_d = torch.from_numpy(off).to(feats.device)
        idx_d = torch.from_numpy(idx if idx.size else np.zeros(1, np.int32)).to(feats.device)
        with torch.cuda.device(feats.device):
            _lib.check(lib.pps_group_mean_rows(_lib.ptr(feats), int(feats.stride(0)), int(feats.shape[1]), _lib.ptr(off_d),
                                               _lib.ptr(idx_d), len(groups), _lib.ptr(out), int(out.stride(0)),
                                               _lib.stream_ptr()), "pps_group_mean_rows")
    return out


def evaluate_arrays(all_feats, ids, cams, marks, precision: str = DEFAULT_PRECISION, verbose: bool = False,
                    to_re_rank: bool = False):
    """The body of ``evaluate`` after the roidb has been flattened to arrays (:57-209).

    marks: 0 = query, 1 = gallery, 2 = multi-query (json_dataset.py:149,188-189).
    Returns (mAP, cmc_scores[10], mq_mAP, mq_cmc_scores) like the reference; with ``to_re_rank`` (the reference's
    ``cfg.REID.RERANK``, :30) these are the scores of the k-reciprocal re-ranked distances (:161-207), as there.
    """
    torch = _torch()
    ids, cams, marks = _ids64(ids, "ids"), _ids64(cams, "cams"), _ids64(marks, "marks")
    feat = all_feats
    if isinstance(feat, np.ndarray):
        feat = torch.from_numpy(np.ascontiguousarray(feat, dtype=np.float32))
    q_inds, g_inds, mq_inds = marks == 0, marks == 1, marks == 2
    qsel, gsel = torch.from_numpy(np.nonzero(q_inds)[0]), torch.from_numpy(np.nonzero(g_inds)[0])
    feat_dev = feat.cuda() if not feat.is_cuda else feat
    gf = feat_dev[gsel.to(feat_dev.device)]

    def compute_score(qf, query_ids, query_cams):
        res = rank_eval(qf, gf, query_ids, ids[g_inds], query_cams, cams[g_inds], precision=precision)
        return res.mean_ap(), res.cmc(topk=10, first_match_break=True)     # :70-93

    def print_scores(mAP, cmc_scores):
        print("[mAP: {:5.2%}], [cmc1: {:5.2%}], [cmc5: {:5.2%}], [cmc10: {:5.2%}]".format(mAP, *cmc_scores[[0, 4, 9]]))

    mAP, cmc_scores = compute_score(feat_dev[qsel.to(feat_dev.device)], ids[q_inds], cams[q_inds])
    if verbose:
        print("{:<30}".format("Single Query:"), end="")
        print_scores(mAP, cmc_scores)

    mq_mAP, mq_cmc_scores = None, None
    if np.any(mq_inds):
        # multi-query: average the mark==2 features of each (id, cam) group (:131-143)
        mq_ids, mq_cams = ids[mq_inds], cams[mq_inds]
        mq_rows = np.nonzero(mq_inds)[0]
        groups = OrderedDict()
        for row, (i, c) in zip(mq_rows.tolist(), zip(mq_ids.tolist(), mq_cams.tolist())):
            groups.setdefault((i, c), []).append(row)
        keys = list(groups.keys())
        src = feat_dev if feat_dev.dtype == torch.float32 and feat_dev.stride(1) == 1 else feat_dev.float().contiguous()
        pooled = group_mean_rows(src, [groups[k] for k in keys])         # rows of the full feature array, in place
        mq_mAP, mq_cmc_scores = compute_score(pooled, np.array([k[0] for k in keys]), np.array([k[1] for k in keys]))
        if verbose:
            print("{:<30}".format("Multi Query:"), end="")
            print_scores(mq_mAP, mq_cmc_scores)
    if to_re_rank:
        from . import rerank as _rerank

        def rerank_score(qf, query_ids, query_cams):
            d = _rerank.re_ranking_from_features(qf, gf, precision=precision)          # :165-171
            res = rank_distmat(d, query_ids, ids[g_inds], query_cams, cams[g_inds])
            return res.mean_ap(), res.cmc(topk=10, first_match_break=True)             # :174-175

        mAP, cmc_scores = rerank_score(feat_dev[qsel.to(feat_dev.device)], ids[q_inds], cams[q_inds])
        if verbose:
            print("{:<30}".format("Re-ranked Single Query:"), end="")
            print_scores(mAP, cmc_scores)
        if np.any(mq_inds):
            mq_mAP, mq_cmc_scores = rerank_score(pooled, np.array([k[0] for k in keys]), np.array([k[1] for k in keys]))
            if verbose:
                print("{:<30}".format("Re-ranked Multi Query:"), end="")
                print_scores(mq_mAP, mq_cmc_scores)
    return mAP, cmc_scores, mq_mAP, mq_cmc_scores


def evaluate(json_dataset, all_feats, output_dir=None, precision: str = DEFAULT_PRECISION, verbose: bool = True,
             to_re_rank: bool = False):
    """reid_dataset_evaluator.py:29-209.  ``to_re_rank`` is the reference's ``cfg.REID.RERANK`` (:30).

    NOTE - the one behavioural default that differs from an unconfigured reference: there ``cfg.REID.RERANK`` defaults
    to True (detectron/core/config.py:1022), so a bare ``evaluate(json_dataset, all_feats, output_dir)`` returns the
    RE-RANKED scores; here there is no global cfg, ``to_re_rank`` defaults to False and the caller passes the value of
    its ``cfg.REID.RERANK`` (``python -m pps_b200.dataset_io --rerank`` on the command line).

    ``json_dataset`` only needs ``get_roidb(gt=True)`` returning entries with 'image' and 'mark'.
    """
    roidb = json_dataset.get_roidb(gt=True)
    ids, cams, marks = [], [], []
    for entry in roidb:
        pid, cam, _, mark, _ = get_info(entry)
        ids.append(pid)
        cams.append(cam)
        marks.append(mark)
    return evaluate_arrays(all_feats, np.asarray(ids), np.asarray(cams), np.asarray(marks), precision, verbose, to_re_rank)


def reid_results(coco_eval, name="reid"):
    """detectron/datasets/task_evaluation.py:54-60,345-360: result tuple -> {'ReID': {...}} dict."""
    res = OrderedDict({"ReID": OrderedDict([("mAP", -1), ("CMC1", -1), ("CMC5", -1), ("CMC10", -1),
                                             ("mq_mAP", -1), ("mq_CMC1", -1), ("mq_CMC5", -1), ("mq_CMC10", -1)])})
    if coco_eval is not None:
        s = coco_eval
        res["ReID"]["mAP"], res["ReID"]["CMC1"], res["ReID"]["CMC5"], res["ReID"]["CMC10"] = s[0], s[1][0], s[1][4], s[1][9]
        if s[2] is not None:
            res["ReID"]["mq_mAP"] = s[2]
        if s[3] is not None:
            res["ReID"]["mq_CMC1"], res["ReID"]["mq_CMC5"], res["ReID"]["mq_CMC10"] = s[3][0], s[3][4], s[3][9]
    return OrderedDict([(name, res)])


# ------------------------------------------------------------------------------------
# host-buffer entry point (what bench.py times as e2e)
# ------------------------------------------------------------------------------------
_HOST_CTX = {}


def _host_ctx(device: int):
    """One pps_ctx (streams + grow-only device / pinned scratch) per device, created on first use."""
    ctx = _HOST_CTX.get(device)
    if ctx is None:
        lib = _lib.load()
        handle = C.c_void_p(0)
        _lib.check(lib.pps_ctx_create(int(device), C.byref(handle)), "pps_ctx_create")
        ctx = _HOST_CTX[device] = handle
    return ctx


def release_host_contexts():
    lib = _lib.load()
    for dev, handle in list(_HOST_CTX.items()):
        lib.pps_ctx_destroy(handle)
        del _HOST_CTX[dev]


def evaluate_host(q_feats, g_feats, query_ids, gallery_ids, query_cams, gallery_cams, cmc_topk: int = 10,
                  topk: int = 0, precision: str = DEFAULT_PRECISION, device: int = 0):
    """pps_evaluate_host_ctx: HOST float32 arrays (numpy, or pinned torch CPU tensors) in, metrics out.

    Every host<->device copy happens inside the call.  Returns a dict with mAP, cmc, ap, valid,
    first_rank and (if topk) topk_index / topk_dist.
    """
    lib = _lib.load()
    _lib.require_cuda()

    def host_f32(a, name):
        if hasattr(a, "is_cuda"):
            if a.is_cuda:
                raise RuntimeError("%s: evaluate_host takes host buffers" % name)
            import torch
            if a.dtype != torch.float32 or not a.is_contiguous() or a.dim() != 2:
                raise RuntimeError("%s: expected a contiguous 2-D float32 tensor" % name)
            return a, int(a.shape[0]), int(a.shape[1])
        a = np.ascontiguousarray(a, dtype=np.float32)
        if a.ndim != 2:
            raise RuntimeError("%s: expected a 2-D array" % name)
        return a, int(a.shape[0]), int(a.shape[1])

    q, nq, dq = host_f32(q_feats, "q_feats")
    g, ng, dg = host_f32(g_feats, "g_feats")
    if dq != dg:
        raise RuntimeError("feature dims differ: %d vs %d" % (dq, dg))
    qi, qc = _ids64(query_ids, "query_ids"), _ids64(query_cams, "query_cams")
    gi, gc = _ids64(gallery_ids, "gallery_ids"), _ids64(gallery_cams, "gallery_cams")
    if len(qi) != nq or len(gi) != ng or len(qc) != nq or len(gc) != ng:
        raise RuntimeError("ids / cams lengths do not match the feature rows")
    out_map = C.c_double(0.0)
    out_cmc = np.zeros(max(cmc_topk, 1), dtype=np.float64)
    ap = np.zeros(nq, dtype=np.float64)
    valid = np.zeros(nq, dtype=np.uint8)
    first = np.zeros(nq, dtype=np.int32)
    ti = np.zeros((nq, topk), dtype=np.int32) if topk else None
    td = np.zeros((nq, topk), dtype=np.float32) if topk else None
    rc = lib.pps_evaluate_host_ctx(_host_ctx(device), _lib.ptr(q), nq, _lib.ptr(g), ng, dq, _lib.ptr(qi), _lib.ptr(qc),
                                   _lib.ptr(gi), _lib.ptr(gc), _prec_code(precision), cmc_topk, topk,
                                   C.cast(C.byref(out_map), C.c_void_p), _lib.ptr(out_cmc), _lib.ptr(ap),
                                   _lib.ptr(valid), _lib.ptr(first), _lib.ptr(ti), _lib.ptr(td))
    _lib.check(rc, "pps_evaluate_host_ctx")
    return dict(mAP=float(out_map.value), cmc=out_cmc[:cmc_topk], ap=ap, valid=valid, first_rank=first,
                topk_index=ti, topk_dist=td)
