"""Non-finite and extreme-magnitude features on every distance path, against the reference's semantics.

The reference (oracle/pps_oracle.py compute_dist) forms -2 a b^T + |a|^2 + |b|^2, sets negatives to 0 with
d2[d2 < 0] = 0 (which keeps NaN) and takes the square root.  It is restated here in float64 from the values the kernel
receives.  A split into several planes turns an infinite element into inf + NaN (the residual plane holds inf - inf), so
for those precisions the restatement sees NaN there: kernel and reference may legitimately disagree on NaN versus inf
for a pair with a non-finite row, never on finite versus non-finite.

- compute_dist, pps_dist_topk_tc: np.isfinite(kernel) == np.isfinite(reference) element for element (no non-finite pair
  yields a finite number, 0 in particular); finite pairs keep tests/test_gpu_dist.py's tolerances.
- GalleryIndex.search: the order is NumPy's stable argsort of the reference (NaN last, inf before NaN: the order of the
  uint32 distance keys).  Integer-valued features make every finite distance exact up to the square root, so the order
  has no near-ties and indices are compared exactly.
- GalleryIndex.range_search: IEEE comparison, so no non-finite row is within a finite radius, and radius inf takes rows
  at distance inf and leaves NaN rows out.
- Evaluation: non-finite gallery rows carry ids that match no query; every output must equal the oracle on the
  reference matrix with each non-finite distance replaced by float32 max (argsort's "after every number").
  Non-finite query rows and non-finite positives are out of scope: there the reference itself raises in sklearn.
- f16x3 magnitudes: rows whose largest element runs over 2^-60 .. 2^60 keep the error of a float32 evaluation.
"""
import numpy as np
import pytest

from oracle import pps_oracle as O

pytestmark = pytest.mark.gpu

DIM = 64
NQ, NG = 40, 300
F16_MAX = 65504.0
F16_TINY = 2.0 ** -24                          # smallest fp16 subnormal
MULTI_PLANE = ("f16x3", "bf16x3", "bf16x6")
# non-finite rows at the tile edges: gallery rows 255, 256 and the last; query columns 31 and 32 of the search tiles
G_SPECIAL = {0: "inf", 3: "-inf", 7: "nan", 11: "all_nan", 20: "f16max", 21: "f16max_one", 22: "subnormal", 23: "tiny",
             255: "inf", 256: "nan", NG - 1: "-inf"}
Q_SPECIAL = {1: "nan", 5: "f16max", 6: "subnormal", 8: "tiny", 31: "inf", 32: "nan", NQ - 1: "-inf"}


def _features(n, special, seed, integer=False):
    """[n, DIM] float32 rows that fp16 holds exactly, with the rows of `special` replaced"""
    rs = np.random.RandomState(seed)
    x = (rs.randint(-8, 9, size=(n, DIM)) if integer else rs.randn(n, DIM)).astype(np.float16).astype(np.float32)
    for row, kind in special.items():
        col = (row * 7) % DIM
        if kind == "inf":
            x[row, col] = np.inf
        elif kind == "-inf":
            x[row, col] = -np.inf
        elif kind == "nan":
            x[row, col] = np.nan
        elif kind == "all_nan":
            x[row] = np.nan
        elif kind == "f16max":
            x[row] = np.where(rs.rand(DIM) < 0.5, -F16_MAX, F16_MAX)
        elif kind == "f16max_one":
            x[row, col] = F16_MAX
        elif kind == "subnormal":
            x[row] = rs.randint(-1023, 1024, size=DIM) * F16_TINY
        elif kind == "tiny":
            x[row] = F16_TINY
    return x


def _received(x, prec):
    """the values the kernel's product sees: a multi-plane split carries an infinite element as inf + NaN"""
    return np.where(np.isinf(x), np.nan, x) if prec in MULTI_PLANE else x


def _ref_dist(a, b):
    """the reference's compute_dist in float64 (element-wise sums: IEEE for inf and NaN)"""
    a, b = a.astype(np.float64), b.astype(np.float64)
    with np.errstate(all="ignore"):
        sq1 = np.einsum("ik,ik->i", a, a)[:, None]
        sq2 = np.einsum("ik,ik->i", b, b)[None, :]
        d2 = -2 * np.einsum("ik,jk->ij", a, b) + sq1 + sq2
        d2[d2 < 0] = 0
        return np.sqrt(d2)


def _ref_cos(a, b, unit=lambda n: n + 1e-12):
    """the cosine branch in float64: rows divided by unit(|x|) (the reference's |x| + 1e-12 by default)"""
    a, b = a.astype(np.float64), b.astype(np.float64)
    with np.errstate(all="ignore"):
        a = a / unit(np.sqrt(np.einsum("ik,ik->i", a, a)))[:, None]
        b = b / unit(np.sqrt(np.einsum("ik,ik->i", b, b)))[:, None]
        return np.einsum("ik,jk->ij", a, b)


def _norms(x):
    with np.errstate(all="ignore"):
        return np.sqrt(np.einsum("ik,ik->i", x.astype(np.float64), x.astype(np.float64)))


def _check(got, ref, a, b, rtol, stol, what, cosine=False):
    """same finiteness everywhere; finite pairs within rtol of the value plus stol of the larger norm (1: cosine)"""
    got = np.asarray(got, np.float64)
    fin = np.isfinite(ref)
    bad = np.argwhere(np.isfinite(got) != fin)
    assert len(bad) == 0, "%s: finiteness differs at %s: kernel %s, reference %s" % (
        what, bad[:5].tolist(), got[tuple(bad[:5].T)], ref[tuple(bad[:5].T)])
    scale = np.ones(ref.shape) if cosine else np.maximum(_norms(a)[:, None], _norms(b)[None, :])
    err = np.where(fin, np.abs(got - np.where(fin, ref, 0)), 0)
    lim = rtol * np.abs(np.where(fin, ref, 0)) + stol * np.where(fin, scale, 0)
    worst = np.unravel_index(np.argmax(err - lim), err.shape)
    assert np.all(err <= lim), "%s: error %g > %g at %s" % (what, err[worst], lim[worst], worst)


def _tol(prec, cosine=False):
    """tests/test_gpu_dist.py's tolerances; bf16x1 (8-bit planes) is the coarse product"""
    if prec == "bf16x1":
        return (0.0, 1e-2) if cosine else (0.0, 4e-3)
    return (1e-4, 2e-6) if cosine else (1e-4, 1e-6)


@pytest.fixture(scope="module")
def rows():
    return _features(NQ, Q_SPECIAL, 1), _features(NG, G_SPECIAL, 2)


# ------------------------------------------------------------------------------------------------------------------
# compute_dist
# ------------------------------------------------------------------------------------------------------------------
CASES = [(p, v) for p in ("f16x3", "bf16x1", "bf16x3", "bf16x6", "fp16") for v in ("2cta", "1cta", "sqrt_rn", "cosine")]
CASES += [("fp32", "2cta"), ("fp32", "cosine")]


@pytest.mark.parametrize("prec,variant", CASES)
def test_compute_dist_non_finite_rows(rows, monkeypatch, prec, variant):
    """Every precision (fp16: float16 tensors) through the default 2-CTA kernel, the 1-CTA kernel, the correctly rounded
    square root and the cosine branch."""
    import torch
    import pps_b200
    from pps_b200 import _lib, evaluator
    q, g = rows
    flags = {"2cta": 0, "1cta": _lib.DIST_KERNEL_1CTA, "sqrt_rn": _lib.DIST_SQRT_RN, "cosine": 0}[variant]
    monkeypatch.setattr(evaluator, "DIST_KERNEL_FLAGS", flags)
    kind = "cosine" if variant == "cosine" else "euclidean"
    if prec == "fp16":
        got = pps_b200.compute_dist(torch.from_numpy(q.astype(np.float16)).cuda(),
                                    torch.from_numpy(g.astype(np.float16)).cuda(), type=kind).cpu().numpy()
    else:
        got = pps_b200.compute_dist(q, g, type=kind, precision=prec)
    # the cosine branch normalises float32 rows and splits them with `precision`; fp16 tensors become float32 there
    seen = "f16x3" if (prec == "fp16" and kind == "cosine") else prec
    qr, gr = _received(q, seen), _received(g, seen)
    ref = _ref_cos(qr, gr) if kind == "cosine" else _ref_dist(qr, gr)
    rtol, stol = _tol(prec, kind == "cosine")
    _check(got, ref, q, g, rtol, stol, "%s %s" % (prec, variant), cosine=kind == "cosine")
    assert not np.isfinite(got[list(Q_SPECIAL)[0]]).any()
    assert not np.isfinite(got[:, 7]).any()               # a single NaN element: no pair is finite, none is 0


def _split(x, planes=1, scaled=False):
    import torch
    from pps_b200 import evaluator
    t = torch.from_numpy(x).cuda()
    return evaluator.SplitOperand(t, planes, scaled)


def test_cluster4_kernel_non_finite_rows(rows):
    """The cluster-of-4 multicast kernel (PPS_DIST_CLUSTER4, single-plane fp16, more than 256 rows of A): the same
    semantics as the reference and the bits of the 2-CTA kernel, with and without the top-k admission epilogue."""
    import torch
    from pps_b200 import _lib
    lib = _lib.load()
    q, g = rows
    a16, b16 = g.astype(np.float16), q.astype(np.float16)          # A = the gallery: 300 > 256 rows
    sa, sb = _split(a16), _split(b16)
    m1, m2 = NG, NQ
    ld = (m2 + 3) // 4 * 4
    out = {}
    for name, flags in (("cl4", _lib.DIST_CLUSTER4), ("cl2", 0)):
        d = torch.zeros((m1, ld), dtype=torch.float32, device="cuda")
        _lib.check(lib.pps_dist_tc(_lib.ptr(sa.planes), _lib.ptr(sa.sqnorm), m1, 1, 0, _lib.ptr(sb.planes), _lib.ptr(sb.sqnorm),
                                   m2, 1, 0, DIM, _lib.PREC_F16X1, flags, _lib.ptr(d), ld, _lib.stream_ptr()), "pps_dist_tc")
        out[name] = d[:, :m2].cpu().numpy()
        bound = torch.full((m1,), -1, dtype=torch.int32, device="cuda")
        cnt = torch.zeros(m1, dtype=torch.int32, device="cuda")
        cand = torch.zeros((m1, m2), dtype=torch.int64, device="cuda")
        d2 = torch.zeros((m1, ld), dtype=torch.float32, device="cuda")
        _lib.check(lib.pps_dist_topk_tc(_lib.ptr(sa.planes), _lib.ptr(sa.sqnorm), m1, 1, 0, _lib.ptr(sb.planes),
                                        _lib.ptr(sb.sqnorm), m2, 1, 0, DIM, _lib.PREC_F16X1, flags, _lib.ptr(d2), ld, 0,
                                        _lib.ptr(bound), _lib.ptr(cnt), _lib.ptr(cand), m2, _lib.stream_ptr()), "pps_dist_topk_tc")
        np.testing.assert_array_equal(d2[:, :m2].cpu().numpy().view(np.uint32), out[name].view(np.uint32))
        np.testing.assert_array_equal(cnt.cpu().numpy(), np.full(m1, m2))
    np.testing.assert_array_equal(out["cl4"].view(np.uint32), out["cl2"].view(np.uint32))
    _check(out["cl4"], _ref_dist(a16.astype(np.float32), b16.astype(np.float32)), g, q, *_tol("fp16"), what="cluster4")


@pytest.mark.parametrize("prec", ["fp16", "bf16x3"])
def test_dist_topk_epilogue_admits_non_finite_only_unbounded(rows, prec):
    """pps_dist_topk_tc (EPI_DIST_TOPK): its block follows the reference's semantics, and a non-finite element is a
    candidate only under the unbounded bound 0xffffffff; under the bound bits(float32 max) every finite element is."""
    import torch
    from pps_b200 import _lib
    lib = _lib.load()
    q, g = rows
    if prec == "fp16":
        a, b = q.astype(np.float16), g.astype(np.float16)
        sa, sb, code, planes = _split(a), _split(b), _lib.PREC_F16X1, 1
        qr, gr = a.astype(np.float32), b.astype(np.float32)
    else:
        sa, sb, code, planes = _split(q, 2), _split(g, 2), _lib.PREC_BF16X3, 2
        qr, gr = _received(q, prec), _received(g, prec)
    ld = (NG + 3) // 4 * 4
    col0 = 1000
    bound_np = np.where(np.arange(NQ) % 2 == 0, 0xffffffff, np.float32(np.finfo(np.float32).max).view(np.uint32))
    bound = torch.from_numpy(bound_np.astype(np.uint32).view(np.int32)).cuda()
    cnt = torch.zeros(NQ, dtype=torch.int32, device="cuda")
    cand = torch.zeros((NQ, NG), dtype=torch.int64, device="cuda")
    d = torch.zeros((NQ, ld), dtype=torch.float32, device="cuda")
    _lib.check(lib.pps_dist_topk_tc(_lib.ptr(sa.planes), _lib.ptr(sa.sqnorm), NQ, planes, 0, _lib.ptr(sb.planes),
                                    _lib.ptr(sb.sqnorm), NG, planes, 0, DIM, code, 0, _lib.ptr(d), ld, col0, _lib.ptr(bound),
                                    _lib.ptr(cnt), _lib.ptr(cand), NG, _lib.stream_ptr()), "pps_dist_topk_tc")
    block = d[:, :NG].cpu().numpy()
    _check(block, _ref_dist(qr, gr), q, g, *_tol(prec), what="topk block " + prec)
    cnt, cand = cnt.cpu().numpy(), cand.cpu().numpy().view(np.uint64)
    for i in range(NQ):
        keys = cand[i, :cnt[i]]
        cols = np.sort((keys & np.uint64(0xffffffff)).astype(np.int64) - col0)
        want = np.arange(NG) if bound_np[i] == 0xffffffff else np.nonzero(np.isfinite(block[i]))[0]
        np.testing.assert_array_equal(cols, want, err_msg="row %d" % i)
        got_bits = (keys >> np.uint64(32)).astype(np.uint32)
        np.testing.assert_array_equal(got_bits, block[i, (keys & np.uint64(0xffffffff)).astype(np.int64) - col0].view(np.uint32))


# ------------------------------------------------------------------------------------------------------------------
# GalleryIndex.search / range_search
# ------------------------------------------------------------------------------------------------------------------
# integer-valued rows: every finite distance is exact up to the square root, so the order has no near-ties
IG_SPECIAL = {0: "inf", 3: "-inf", 7: "nan", 11: "all_nan", 20: "f16max", 255: "inf", 256: "nan", NG - 1: "-inf"}
IQ_SPECIAL = {1: "nan", 31: "inf", 32: "nan", NQ - 1: "-inf"}
SMALL_NG = 40
SMALL_SPECIAL = {0: "inf", 3: "-inf", 7: "nan", 11: "all_nan", 31: "inf", 32: "nan", SMALL_NG - 1: "nan"}


def _index(g, dtype_name, tags=None):
    import torch
    import pps_b200
    f16 = dtype_name == "fp16"
    idx = pps_b200.GalleryIndex(DIM, dtype=torch.float16 if f16 else torch.float32, precision="f16x3")
    idx.add(g.astype(np.float16) if f16 else g, tags)
    return idx


def _index_ref(q, g, dtype_name):
    prec = "fp16" if dtype_name == "fp16" else "f16x3"
    return _ref_dist(_received(q, prec), _received(g, prec))


def _category(x):
    return np.where(np.isnan(x), 2, np.where(np.isinf(x), 1, 0))


def _check_search(got_d, got_i, ref, keep, k, what):
    for i in range(ref.shape[0]):
        cand = np.nonzero(keep[i])[0]
        order = cand[np.argsort(ref[i, cand], kind="stable")][:k]
        want_i = np.full(k, -1, np.int64)
        want_i[:len(order)] = order
        np.testing.assert_array_equal(got_i[i], want_i, err_msg="%s query %d" % (what, i))
        want_d = np.full(k, np.inf)
        want_d[:len(order)] = ref[i, order]
        fin = np.isfinite(want_d[:len(order)])
        np.testing.assert_array_equal(_category(got_d[i, :len(order)]), _category(want_d[:len(order)]),
                                      err_msg="%s query %d" % (what, i))
        np.testing.assert_allclose(got_d[i, :len(order)][fin], want_d[:len(order)][fin], rtol=1e-6,
                                   err_msg="%s query %d" % (what, i))
        # a non-finite row only after every finite row
        cat = _category(got_d[i, :len(order)])
        assert np.all(np.diff(cat) >= 0), "%s query %d: %s" % (what, i, cat)


@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
@pytest.mark.parametrize("ng", [NG, SMALL_NG])
def test_index_search_orders_non_finite_rows_last(dtype_name, ng):
    """Plain and excluding search, fp32 (f16x3) and fp16 indexes, the materialised prefix and the search kernel, k below,
    equal to and above the number of finite rows: the stable argsort of the reference, indices exactly."""
    from pps_b200 import _lib
    special = IG_SPECIAL if ng == NG else SMALL_SPECIAL
    q = _features(NQ, IQ_SPECIAL, 3, integer=True)
    g = _features(ng, special, 4, integer=True)
    rs = np.random.RandomState(ng)
    tags = rs.randint(0, 4, size=ng).astype(np.int64)
    ex = rs.randint(0, 4, size=NQ).astype(np.int64)
    idx = _index(g, dtype_name, tags)
    ref = _index_ref(q, g, dtype_name)
    n_finite = ng - len(special)
    ks = (1, 16, 128) if ng == NG else (10, n_finite - 1, n_finite, n_finite + 1, ng, 64)
    qx = q.astype(np.float16) if dtype_name == "fp16" else q
    for flags in (0, _lib.index_prefix(1)):
        for k in ks:
            for excl in (None, ex):
                keys, _ = idx._search_keys(qx, k, 0, flags, excl)
                got_d, got_i = idx._unpack(keys, True)
                keep = np.ones((NQ, ng), bool) if excl is None else tags[None, :] != excl[:, None]
                _check_search(got_d, got_i, ref, keep, k, "%s ng=%d flags=%x k=%d excl=%s" % (
                    dtype_name, ng, flags, k, excl is not None))


@pytest.mark.parametrize("dtype_name", ["fp32", "fp16"])
def test_index_range_search_ieee_radius(dtype_name):
    """No non-finite row is within a finite radius; radius inf takes the rows at distance inf and leaves NaN rows out."""
    q = _features(NQ, IQ_SPECIAL, 5, integer=True)
    g = _features(NG, IG_SPECIAL, 6, integer=True)
    rs = np.random.RandomState(7)
    tags = rs.randint(0, 4, size=NG).astype(np.int64)
    ex = rs.randint(0, 4, size=NQ).astype(np.int64)
    idx = _index(g, dtype_name, tags)
    ref = _index_ref(q, g, dtype_name)
    qx = q.astype(np.float16) if dtype_name == "fp16" else q
    # finite squared distances are integers (or far apart): a radius of sqrt(m + 1/2) has no distance near it
    med = np.ones(NQ, np.float32)
    for i in range(NQ):
        f = ref[i][np.isfinite(ref[i])]
        if len(f):
            med[i] = np.sqrt(np.floor(np.median(f * f)) + 0.5)
    radii = {"median": med, "f32max": np.float32(np.finfo(np.float32).max), "inf": np.float32(np.inf)}
    for rname, radius in radii.items():
        r = np.full(NQ, radius, np.float32)
        for excl in (None, ex):
            lims, dist, index = idx.range_search(qx, r, exclude_tags=excl)
            keep = np.ones((NQ, NG), bool) if excl is None else tags[None, :] != excl[:, None]
            what = "%s radius=%s excl=%s" % (dtype_name, rname, excl is not None)
            for i in range(NQ):
                with np.errstate(invalid="ignore"):
                    ok = keep[i] & (ref[i].astype(np.float32) <= r[i])          # IEEE: NaN is never <= r
                cand = np.nonzero(ok)[0]
                order = cand[np.argsort(ref[i, cand], kind="stable")]
                a, b = lims[i], lims[i + 1]
                np.testing.assert_array_equal(index[a:b], order, err_msg="%s query %d" % (what, i))
                assert not np.isnan(dist[a:b]).any(), what
                if not np.isinf(r[i]):
                    assert np.isfinite(dist[a:b]).all(), what
                f = np.isfinite(ref[i, order])
                np.testing.assert_array_equal(np.isfinite(dist[a:b]), f, err_msg=what)
                np.testing.assert_allclose(dist[a:b][f], ref[i, order][f], rtol=1e-6, err_msg=what)


# ------------------------------------------------------------------------------------------------------------------
# evaluation: rank_eval, RankEngine's passes, evaluate_arrays
# ------------------------------------------------------------------------------------------------------------------
EV_NQ, EV_NG = 50, 1200
EV_SPECIAL = {0: "inf", 255: "nan", 256: "-inf", 511: "all_nan", 512: "inf", 700: "nan", EV_NG - 1: "inf"}


@pytest.fixture(scope="module")
def eval_set():
    q = _features(EV_NQ, {}, 8, integer=True)
    g = _features(EV_NG, EV_SPECIAL, 9, integer=True)
    rs = np.random.RandomState(10)
    qid = rs.randint(0, 60, size=EV_NQ).astype(np.int64)
    gid = rs.randint(0, 60, size=EV_NG).astype(np.int64)           # ~20 pairs per query: within the counting epilogue's 64
    bad = np.array(sorted(EV_SPECIAL))
    gid[bad] = 10 ** 6 + bad                                    # non-finite rows match no query
    qcam = rs.randint(0, 3, size=EV_NQ).astype(np.int64)
    gcam = rs.randint(0, 3, size=EV_NG).astype(np.int64)
    ref = _ref_dist(q, g)
    assert not np.isfinite(ref[:, bad]).any() and np.isfinite(np.delete(ref, bad, axis=1)).all()
    refm = np.where(np.isfinite(ref), ref, np.finfo(np.float32).max).astype(np.float32)
    return dict(q=q, g=g, qid=qid, gid=gid, qcam=qcam, gcam=gcam, refm=refm)


def _check_eval(res, e, topk, what):
    ids = (e["qid"], e["gid"], e["qcam"], e["gcam"])
    ap, valid, first, neg_before = O.rank_counts(e["refm"], *ids)
    np.testing.assert_array_equal(res.is_valid, valid, err_msg=what)
    np.testing.assert_array_equal(res.first_rank, first, err_msg=what)
    np.testing.assert_allclose(res.ap, ap, rtol=0, atol=1e-12, err_msg=what)
    assert abs(res.mean_ap() - ap[valid == 1].mean()) < 1e-12, what
    want_cmc = O.cmc(e["refm"], *ids, topk=10, first_match_break=True, stable=True)
    np.testing.assert_allclose(res.cmc(10, True), want_cmc, atol=1e-12, err_msg=what)
    if res.neg_before is not None:
        p = res.pairs
        for i in range(p.nq):
            idx = np.arange(p.off[i], p.off[i + 1])
            np.testing.assert_array_equal(res.neg_before[idx[p.pos[idx] == 1]], neg_before[i], err_msg=what)
    if topk:
        ti, td = O.topk_filtered(e["refm"], *ids, topk)
        np.testing.assert_array_equal(res.topk_index, ti, err_msg=what)
        np.testing.assert_allclose(res.topk_dist, td, rtol=1e-6, err_msg=what)


@pytest.mark.parametrize("topk", [0, 10])
def test_evaluation_passes_count_non_finite_rows_last(eval_set, topk):
    """fp16 gallery over five 256-row blocks: rank_eval's C pass (counting epilogue EPI_RANK with top-k admission after
    the first block) and the launch-by-launch pass with the separate count, sweep and top-k kernels of rank.cu, and with
    the counting epilogue."""
    import torch
    import pps_b200
    from pps_b200 import evaluator
    e = eval_set
    q = torch.from_numpy(e["q"].astype(np.float16)).cuda()
    g = torch.from_numpy(e["g"].astype(np.float16)).cuda()
    ids = (e["qid"], e["gid"], e["qcam"], e["gcam"])
    block = EV_NQ * 256 * 4
    res = pps_b200.rank_eval(q, g, *ids, topk=topk, max_block_bytes=block)
    _check_eval(res, e, topk, "rank_eval")
    for c_pass, fused in ((True, False), (False, False), (False, True)):
        # (the C pass serves the plain evaluation: per-positive negatives-before counts take the launch-by-launch pass)
        eng = evaluator.RankEngine(*ids, nq=EV_NQ, ng_local=EV_NG, dim=DIM, topk=topk, want_neg_before=not c_pass,
                                   max_block_bytes=block, in_dtype=torch.float16)
        eng.use_c_pass = c_pass
        eng.fused_rank = fused
        assert eng.n_chunks > 1
        r = eng.run(q, g)
        if c_pass:
            assert eng.used_fused_count and eng.pass_blocks > 1
        else:
            assert eng.used_fused_rank == (fused and not topk)     # (the launch-by-launch counting epilogue has no top-k)
        _check_eval(r, e, topk, "RankEngine c_pass=%s fused_rank=%s" % (c_pass, fused))


def test_evaluate_arrays_non_finite_gallery_rows(eval_set):
    """evaluate_arrays on fp16 features: mAP and CMC of the oracle on the replaced reference matrix."""
    import torch
    import pps_b200
    e = eval_set
    feats = torch.from_numpy(np.concatenate([e["q"], e["g"]]).astype(np.float16)).cuda()
    ids = np.concatenate([e["qid"], e["gid"]])
    cams = np.concatenate([e["qcam"], e["gcam"]])
    marks = np.concatenate([np.zeros(EV_NQ, np.int64), np.ones(EV_NG, np.int64)])
    mAP, cmc_scores, _, _ = pps_b200.evaluate_arrays(feats, ids, cams, marks)
    args = (e["qid"], e["gid"], e["qcam"], e["gcam"])
    ap, valid, _, _ = O.rank_counts(e["refm"], *args)
    assert abs(mAP - ap[valid == 1].mean()) < 1e-12
    np.testing.assert_allclose(cmc_scores, O.cmc(e["refm"], *args, topk=10, first_match_break=True, stable=True), atol=1e-12)


# ------------------------------------------------------------------------------------------------------------------
# f16x3 row scales over the whole float32 range
# ------------------------------------------------------------------------------------------------------------------
def _sweep_rows():
    """rows whose largest element is 2^p, p = -66 .. 60, three per magnitude, kept where the float64 |x|^2 rounds to a
    normal float32 (down to p = -64 at this width); B holds eight other rows of every magnitude (more than one 256-row
    tile) and copies of A's (distance ~0)"""
    rs = np.random.RandomState(21)
    a, b = [], []
    for p in list(range(-66, -60, 2)) + list(range(-60, 61, 4)):
        for dst in [a] * 3 + [b] * 8:
            x = rs.randn(DIM)
            x = x / np.abs(x).max() * 2.0 ** p
            n2 = float(np.dot(x, x))
            if np.finfo(np.float32).tiny <= n2 <= np.finfo(np.float32).max:
                dst.append(x)
    a = np.array(a, np.float32)
    b = np.concatenate([np.array(b, np.float32), a[::3]])
    return a, b


def _f64(a, b):
    return _ref_dist(a, b)


def _assert_float32_grade(got, exact, scale, ref_err, what):
    err = np.max(np.abs(np.asarray(got, np.float64) - exact) / scale)
    assert err < 4 * max(ref_err, 1e-7), "%s: %g against %g" % (what, err, ref_err)


def test_f16x3_magnitude_sweep(monkeypatch):
    """Equal-scale pairs of small rows, small rows of different scales and small rows against large ones.  The epilogue
    multiplies by -2 / (s_a s_b), formed as one float: with two rows whose largest element is below about 2^-61 it must
    not underflow (split_prep.cu bounds the row scales for that).  compute_dist
    (both kernels, and the cosine branch), GalleryIndex.search and rank_eval stay within 4x the float32 reference's
    error relative to the larger norm (the criterion of test_f16x3_row_scaling_covers_the_dynamic_range)."""
    import torch
    import pps_b200
    from pps_b200 import _lib, evaluator
    a, b = _sweep_rows()
    assert a.shape[0] >= 90 and b.shape[0] > 256
    exact = _f64(a, b)
    scale = np.maximum(_norms(a)[:, None], _norms(b)[None, :])
    ref_err = float(np.max(np.abs(O.compute_dist(a, b).astype(np.float64) - exact) / scale))
    for kernel, flags in (("2cta", 0), ("1cta", _lib.DIST_KERNEL_1CTA)):
        monkeypatch.setattr(evaluator, "DIST_KERNEL_FLAGS", flags)
        got = pps_b200.compute_dist(a, b, precision="f16x3")
        _assert_float32_grade(got, exact, scale, ref_err, "compute_dist " + kernel)
        # the cosine branch divides by max(|x|, 1e-12) (Caffe2's Normalize, pps_l2_normalize_rows); the reference's
        # |x| + 1e-12 differs from that only for norms near 1e-12, which this sweep has, so the restatement uses max
        cos = pps_b200.compute_dist(a, b, type="cosine", precision="f16x3")
        want = _ref_cos(a, b, unit=lambda n: np.maximum(n, 1e-12))
        np.testing.assert_allclose(cos, want, rtol=1e-4, atol=2e-6, err_msg="cosine " + kernel)
    monkeypatch.setattr(evaluator, "DIST_KERNEL_FLAGS", 0)
    k = 128
    idx = pps_b200.GalleryIndex(DIM, dtype=torch.float32, precision="f16x3")
    idx.add(b)
    for flags in (0, _lib.index_prefix(1)):                  # (prefix of 256 rows: the rest through the search kernel)
        keys, _ = idx._search_keys(a, k, 0, flags)
        sd, si = idx._unpack(keys, True)
        _assert_float32_grade(sd, np.take_along_axis(exact, si, 1), np.take_along_axis(scale, si, 1), ref_err,
                              "search flags=%x" % flags)
    qid, gid = np.arange(a.shape[0]) % 5, np.arange(b.shape[0]) % 5
    res = pps_b200.rank_eval(torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda(), qid, gid, np.zeros_like(qid),
                             np.ones_like(gid), topk=k, precision="f16x3")
    ti = np.asarray(res.topk_index).astype(np.int64)
    _assert_float32_grade(res.topk_dist, np.take_along_axis(exact, ti, 1), np.take_along_axis(scale, ti, 1), ref_err,
                          "rank_eval")
