"""Every width of the HNSW search and build kernels against an exhaustive f64 reference, and NaN ordering.

The kernels are instantiated per `NV = ceil(ld / 128)` in {1, 2, 4, 6, 8, 16} (ld = dim rounded up to 4), per metric and
per form (hnsw.mode 0 = plain loads, 1 = TMA ring, 2 = cooperative).  These tests need no oracle: a single-layer graph
that is connected from the entry point, searched with ef >= n, is exhaustive.  Nothing is evicted from the beam and the
`candidate_dist > furthest_dist` break (hnsw.rs:562) never fires, so for every kernel form and launch geometry

  * the result is the exact k-NN in the f64 distances of hnsw.rs:66-109 (NaN ordered last, as OrderedFloat does),
  * dist_evals == nodes_expanded == B * n.

Distances are checked against an a-priori bound, not a tuned tolerance.  With u = 2^-24 and h = 4 * NV + 6 (each lane
runs an fma chain of at most 4 * NV terms, then a 5-level shuffle tree; 2h covers the inner sum and the norms):
  L2      |d - d64| <= 2 (h + 2) u d64                  (+2: the f32 difference q_i - x_i before squaring)
  IP      |d - d64| <= 2 h u sum|q_i x_i| + u |d|        (u |d|: the final rounding of 1 - a to f32)
  Cosine  |d - d64| <= 2 h u (sum|q_i x_i| / (|q| |x|) + |cos|) + u |d|
The F64 kernel uses u = 2^-53 and h = ceil(dim / 32) + 6 (one fma chain per lane over a 32-strided slice); its reference
is computed in long double.  f32 inputs give exact products in f64, so the f64 reference of the f32 kernels is exact up
to its own summation error, ~log2(dim) 2^-53, far below the bound.

Ids are compared with the exact top-k up to ties: an id may differ only if its f64 distance is within twice the bound
of the k-th distance (two ids can swap only when their reference distances are closer than the sum of their bounds).

COZO_EMU_LIB (the CPU-emulated build of the library, tests/conftest.py) runs every kernel about 100x slower; the sizes
shrink there.
"""
import math
import os

import numpy as np
import pytest

from oracle import oracle as O
from tests.util import recall, SEED_LEVEL

pytestmark = pytest.mark.gpu
EMU = bool(os.environ.get("COZO_EMU_LIB"))
NONE = 0xFFFFFFFF
L2, COSINE, IP = O.L2, O.COSINE, O.IP
METRICS = [L2, COSINE, IP]
MODES = [0, 1, 2]
SEARCH_OPTIONS = {"hnsw.mode": -1, "hnsw.stages": 4, "hnsw.warps_per_cta": 4, "hnsw.max_ctas_per_sm": 0}


def _nv(dim):
    need = -(-((dim + 3) // 4 * 4) // 128)
    return next(v for v in (1, 2, 4, 6, 8, 16) if v >= need)


# ---- inputs -------------------------------------------------------------------------------------------------------
def _data(n, dim, seed, dtype=np.float32):
    """centred, so that Cosine and IP see sign cancellation"""
    return (np.random.default_rng(seed).random((n, dim)) - 0.5).astype(dtype)


def _ring_csr(n, seed, chords=6, hubs=4, hub_degree=40):
    """connected single layer: ring i +- 1 plus seeded random chords; a few hub rows have more than 32 neighbours, so
    the 32-wide chunk loop over an adjacency row and the wrap-around of the row ring both run"""
    rng = np.random.default_rng(seed)
    rows = [{(i + 1) % n, (i - 1) % n} for i in range(n)]
    for i in range(n):
        rows[i].update(int(t) for t in rng.integers(0, n, chords))
    for h in rng.choice(n, min(hubs, n), replace=False):
        rows[h].update(int(t) for t in rng.choice(n, min(hub_degree, n), replace=False))
    for i in range(n):
        rows[i].discard(i)
    rp = np.zeros(n + 1, np.uint64)
    rp[1:] = np.cumsum([len(r) for r in rows])
    ci = np.concatenate([np.array(sorted(r), np.uint32) for r in rows])
    return rp, ci


def _stage(gpu, X, metric, seed=1):
    rp, ci = _ring_csr(X.shape[0], seed)
    return gpu.HnswIndex.stage(X, [None], [rp], [ci], 0, metric=metric)


# ---- reference ----------------------------------------------------------------------------------------------------
def _dist_bound(q, x, metric, f64_kernel=False):
    """reference distance and error bound for broadcastable row arrays q, x (last axis = dim), see the module docstring"""
    dim = q.shape[-1]
    if f64_kernel:
        u, h = 2.0 ** -53, math.ceil(dim / 32) + 6
        q, x = q.astype(np.longdouble), x.astype(np.longdouble)
    else:
        u, h = 2.0 ** -24, 4 * _nv(dim) + 6
        q, x = q.astype(np.float64), x.astype(np.float64)
    if metric == L2:
        d = ((q - x) ** 2).sum(-1)
        return d, 2 * (h + 2) * u * d
    p = q * x
    dot, s = p.sum(-1), np.abs(p).sum(-1)
    if metric == IP:
        d = 1 - dot
        return d, 2 * h * u * s + u * np.abs(d)
    den = np.sqrt((q * q).sum(-1) * (x * x).sum(-1))
    with np.errstate(invalid="ignore", divide="ignore"):
        cos = dot / den                      # 0 / 0 = NaN for a zero row or query, as in hnsw.rs:80-84
        d = 1 - cos
        return d, 2 * h * u * (s / den + np.abs(cos)) + u * np.abs(d)


def _reference(Q, X, metric, f64_kernel=False):
    """[B, n] distances and bounds"""
    step = max(1, (1 << 22) // (X.shape[0] * X.shape[1]))
    parts = [_dist_bound(Q[i:i + step, None, :], X[None, :, :], metric, f64_kernel) for i in range(0, len(Q), step)]
    return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])


def _check_topk(ids, dist, cnt, D, T, k):
    """device lists == exact top-k of D (NaN last) up to ties; distances within the bound, sorted, NaN only at the end"""
    B, n = D.shape
    kk = min(k, n)
    assert np.all(cnt == kk)
    got = ids[:, :kk].astype(np.int64)
    assert got.max() < n and all(len(set(r.tolist())) == kk for r in got), "ids out of range or repeated"
    if kk < k:
        assert np.all(ids[:, kk:] == NONE) and np.all(np.isinf(dist[:, kk:]))
    Dg, Tg, dg = np.take_along_axis(D, got, 1), np.take_along_axis(T, got, 1), dist[:, :kk]
    fin = ~np.isnan(Dg)
    assert np.array_equal(np.isnan(dg), ~fin), "NaN distances where the reference has none, or the reverse"
    assert np.all(np.diff(fin.astype(np.int8), axis=1) <= 0), "a NaN entry before a finite one"
    err = np.abs(dg[fin] - Dg[fin])
    assert np.all(err <= Tg[fin]), f"distance error {float(np.max(err - Tg[fin]))} beyond the bound"
    asc = np.where(fin, dg, np.inf)
    assert np.all(asc[:, 1:] >= asc[:, :-1]), "distances not ascending"
    order = np.argsort(D, axis=1, kind="stable")[:, :kk]
    for b in range(B):
        kth = order[b, -1]
        for i in set(order[b].tolist()) ^ set(got[b].tolist()):
            both_nan = np.isnan(D[b, i]) and np.isnan(D[b, kth])      # order among NaN keys is unspecified
            assert both_nan or abs(D[b, i] - D[b, kth]) <= 2 * max(T[b, i], T[b, kth]), \
                f"query {b}: id {i} at {D[b, i]} vs k-th distance {D[b, kth]}"


def _check_exhaustive(out, D, T, k, n):
    ids, dist, cnt, st = out
    _check_topk(ids, dist, cnt, D, T, k)
    B = D.shape[0]
    assert st.dist_evals == B * n and st.nodes_expanded == B * n, (st.dist_evals, st.nodes_expanded, B * n)


class _options:
    """set search options for a block; on the way out, even after a failure, every option is put back"""

    def __init__(self, gpu, **kv):
        self.gpu, self.kv = gpu, {k.replace("__", "."): v for k, v in kv.items()}

    def __enter__(self):
        for k, v in self.kv.items():
            self.gpu.set_option(k, v)

    def __exit__(self, *exc):
        for k, v in SEARCH_OPTIONS.items():
            self.gpu.set_option(k, v)
        self.gpu.set_option("hnsw.coop_below", 6 * _sm_count())   # the library's default: 6 CTAs per SM


def _torch_cuda():
    try:
        import torch
    except ImportError:
        return None
    return torch if torch.cuda.is_available() else None


def _sm_count():
    torch = _torch_cuda()
    if torch is not None:
        return torch.cuda.get_device_properties(0).multi_processor_count
    return int(os.environ.get("COZO_EMU_SM_COUNT") or 4)      # the emulated device (tests/emu/fake_cuda)


def _smem_optin():
    torch = _torch_cuda()
    if torch is not None:
        return torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    assert EMU, "no torch CUDA device to read the shared-memory limit from"
    return 232448                                              # what the emulated device reports (the B200 limit)


# ---- a. every width boundary --------------------------------------------------------------------------------------
WIDTH_DIMS = [1, 3, 4, 5, 127, 128, 129, 255, 256, 257, 384, 511, 512, 513, 767, 768, 769, 1023, 1024, 1025, 1536, 2047,
              2048]


@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("dim", WIDTH_DIMS)
def test_exhaustive_search_every_width(gpu, dim, metric):
    n, B = (120, 4) if EMU else (400, 32)
    X, Q = _data(n, dim, 10 + dim), _data(B, dim, 20 + dim)
    g = _stage(gpu, X, metric)
    D, T = _reference(Q, X, metric)
    for mode in MODES:
        with _options(gpu, hnsw__mode=mode):
            for k in (10, n):
                _check_exhaustive(g.search(Q, k, n), D, T, k, n)


# ---- b. launch geometry -------------------------------------------------------------------------------------------
GEOMETRY_DIMS = [(61, L2), (200, COSINE), (384, IP), (700, L2), (1000, COSINE), (1536, IP)]     # NV = 1, 2, 4, 6, 8, 16


@pytest.mark.parametrize("dim,metric", GEOMETRY_DIMS)
def test_exhaustive_search_launch_geometry(gpu, dim, metric):
    """ring stages, warps per CTA, persistent warps that serve several queries in turn (a stale visited bit would
    show up as a missing distance evaluation) and the cooperative form on a large batch"""
    n, B = (80, 3) if EMU else (256, 16)
    big = 4 * _sm_count() + 3                   # > 4 queries per warp slot with 1 CTA of 1 warp per SM
    X, Q = _data(n, dim, 30 + dim), _data(big, dim, 40 + dim)
    g = _stage(gpu, X, metric, seed=dim)
    D, T = _reference(Q, X, metric)
    k = 10
    for mode in (1, 2):
        for ns in (1, 2, 4):
            with _options(gpu, hnsw__mode=mode, hnsw__stages=ns):
                _check_exhaustive(g.search(Q[:B], k, n), D[:B], T[:B], k, n)
    for mode in (0, 1):
        for wpc in (1, 2, 4):
            with _options(gpu, hnsw__mode=mode, hnsw__warps_per_cta=wpc):
                _check_exhaustive(g.search(Q[:B], k, n), D[:B], T[:B], k, n)
        with _options(gpu, hnsw__mode=mode, hnsw__warps_per_cta=1, hnsw__max_ctas_per_sm=1):
            _check_exhaustive(g.search(Q, k, n), D, T, k, n)
    with _options(gpu, hnsw__coop_below=1 << 30):               # default mode picks the cooperative form for any batch
        _check_exhaustive(g.search(Q, k, n), D, T, k, n)


# ---- c. shared-memory fallback ------------------------------------------------------------------------------------
def _ru(x, m):
    return (x + m - 1) // m * m


def _warp_smem(ef, ns, ld):
    """per-warp shared memory of the warp-per-query kernel, as hnsw_launch_search lays it out"""
    efcap = _ru(ef, 32)
    return _ru(_ru(efcap * 8 + 128 + ns * 8, 128) + ns * ld * 4, 128)


def _coop_smem(ef, ns, ld):
    """shared memory per CTA of the cooperative kernel (at most 3 ring stages per warp, 4 warps)"""
    efcap, cns = _ru(ef, 32), min(ns, 3)
    return _ru(efcap * 8 + 288, 128) + 4 * _ru(_ru(cns * 8, 128) + cns * ld * 4, 128)


def _max_ef(fits):
    ef = 32
    while fits(ef + 32):
        ef += 32
    return ef


def test_shared_memory_fallback_dim_2048(gpu):
    """ef past what 4 (then 2) warps per CTA can hold drops to fewer warps per CTA; past one warp it is E_UNSUP, and
    the handle keeps working.  ef > n is still exhaustive."""
    dim, ns, limit = 2048, 4, _smem_optin()
    n, B = (40, 2) if EMU else (200, 8)
    X, Q = _data(n, dim, 50), _data(B, dim, 51)
    g = _stage(gpu, X, L2)
    D, T = _reference(Q, X, L2)
    ef4 = _max_ef(lambda ef: 4 * _warp_smem(ef, ns, dim) <= limit)
    ef2 = _max_ef(lambda ef: 2 * _warp_smem(ef, ns, dim) <= limit)
    ef1 = _max_ef(lambda ef: _warp_smem(ef, ns, dim) <= limit)
    assert n < ef4 < ef2 < ef1
    with _options(gpu, hnsw__mode=1, hnsw__stages=ns):
        for ef in (ef4, ef4 + 1, ef2, ef2 + 1, ef1):
            _check_exhaustive(g.search(Q, 10, ef), D, T, 10, n)
        with pytest.raises(gpu.CozoGpuError) as e:
            g.search(Q, 10, ef1 + 1)
        assert e.value.code == gpu.E_UNSUP
        _check_exhaustive(g.search(Q, 10, n), D, T, 10, n)
    efc = _max_ef(lambda ef: _coop_smem(ef, ns, dim) <= limit)
    with _options(gpu, hnsw__mode=2, hnsw__stages=ns):
        _check_exhaustive(g.search(Q, 10, efc), D, T, 10, n)
        with pytest.raises(gpu.CozoGpuError) as e:
            g.search(Q, 10, efc + 1)
        assert e.value.code == gpu.E_UNSUP
        _check_exhaustive(g.search(Q, 10, n), D, T, 10, n)


# ---- d. the width limit -------------------------------------------------------------------------------------------
def test_dim_2049_is_refused(gpu):
    n, dim = 50, 2049
    X = _data(n, dim, 60)
    g = _stage(gpu, X, L2)
    for mode in (-1, 0, 1, 2):
        with _options(gpu, hnsw__mode=mode):
            with pytest.raises(gpu.CozoGpuError) as e:
                g.search(X[:2], 5, 50)
            assert e.value.code == gpu.E_UNSUP
    with pytest.raises(gpu.CozoGpuError) as e:
        gpu.HnswIndex.build(X, m=8, ef_construction=20)
    assert e.value.code == gpu.E_UNSUP
    torch = _torch_cuda()
    if torch is not None:                        # nothing was launched: the device outputs keep their sentinel
        q = torch.from_numpy(X[:4]).cuda()
        ids = torch.full((4, 5), 7, dtype=torch.int32, device="cuda")
        dist = torch.full((4, 5), 7.0, dtype=torch.float32, device="cuda")
        stream = torch.cuda.current_stream().cuda_stream
        with pytest.raises(gpu.CozoGpuError) as e:
            g.search_dev(q.data_ptr(), 4, 5, 50, ids.data_ptr(), dist.data_ptr(), stream=stream)
        assert e.value.code == gpu.E_UNSUP
        torch.cuda.synchronize()
        assert bool((ids == 7).all()) and bool((dist == 7.0).all())


# ---- e. the builder at the widths no other test builds ------------------------------------------------------------
@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("dim", [129, 384, 769, 1536, 2048])
def test_builder_at_untested_widths(gpu, dim, metric):
    n, nq, m, efc, ef = (300, 20, 8, 40, 40) if EMU else (2500, 200, 12, 80, 80)
    X, Q = _data(n, dim, 70 + dim), _data(nq, dim, 80 + dim)
    g = gpu.HnswIndex.build(X, metric=metric, m=m, ef_construction=efc, level_seed=SEED_LEVEL)
    ni, rp, ci, ep = g.export_levels()
    deg0 = np.diff(rp[0].astype(np.int64))
    assert deg0.max() <= 2 * m and deg0.min() >= 1
    for L in range(1, len(rp)):
        assert np.diff(rp[L].astype(np.int64)).max() <= m
    # stored edge distances (build_edge_dist_kernel) against f64
    for L, dl in enumerate(g.export_dists()):
        nodes = np.arange(n) if L == 0 else ni[L].astype(np.int64)
        src = np.repeat(nodes, np.diff(rp[L].astype(np.int64)))
        dst = ci[L].astype(np.int64)
        for s in range(0, src.size, 4096):
            d64, t = _dist_bound(X[src[s:s + 4096]], X[dst[s:s + 4096]], metric)
            assert np.all(np.abs(dl[s:s + 4096] - d64) <= t), f"layer {L}: stored distance beyond the bound"
    # device search == oracle search on the exported graph
    ix = O.OracleHnsw.from_levels(X, O.HnswLevels(ni, rp, ci, ep), metric=metric)
    gi, gd, gc, st = g.search(Q, 10, ef)
    oi, od, oc, ost = ix.search(Q, 10, ef, n_threads=8)
    assert np.array_equal(gc, oc) and recall(gi, oi) >= 0.999
    assert abs(int(st.dist_evals) - int(ost[:, 0].sum())) <= 0.001 * ost[:, 0].sum()
    assert abs(int(st.nodes_expanded) - int(ost[:, 1].sum())) <= 0.001 * ost[:, 1].sum()
    D, T = _reference(Q, X, metric)
    Dg, Tg = np.take_along_axis(D, gi.astype(np.int64), 1), np.take_along_axis(T, gi.astype(np.int64), 1)
    assert np.all(np.abs(gd - Dg) <= Tg)
    # graph quality: as good as the reference's sequential build, against f64 brute force
    if dim in (384, 1536) and metric in (L2, COSINE) and not EMU:
        exact = np.argsort(D, axis=1, kind="stable")[:, :10]
        seq = O.OracleHnsw.new(n, dim, metric=metric, m=m, ef_construction=efc, level_seed=SEED_LEVEL)
        seq.insert_all(X)
        seq_ids = seq.search(Q, 10, ef, n_threads=8)[0]
        assert recall(gi, exact) >= recall(seq_ids, exact) - 0.02


# ---- f. the F64 kernel --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("dim", [1, 33, 384, 1536, 2048])
def test_f64_exhaustive_search(gpu, dim, metric):
    n, B = (100, 3) if EMU else (300, 16)
    X, Q = _data(n, dim, 90 + dim, np.float64), _data(B, dim, 91 + dim, np.float64)
    g = _stage(gpu, X, metric)
    D, T = _reference(Q, X, metric, f64_kernel=True)
    for k in (10, n):
        out = g.search_f64(Q, k, n)
        assert out[1].dtype == np.float64
        _check_exhaustive(out, D, T, k, n)


# ---- g. NaN: zero-norm rows and queries under Cosine --------------------------------------------------------------
def _nan_setup(f64):
    n, B, dim = (96, 4, 64) if EMU else (300, 40, 64)
    dtype = np.float64 if f64 else np.float32
    X, Q = _data(n, dim, 100, dtype), _data(B, dim, 101, dtype)
    zero = np.array([3, n // 3, n - 7])
    X[zero] = 0
    return X, Q, zero


@pytest.mark.parametrize("kernel", ["f32_mode0", "f32_mode1", "f32_mode2", "f64"])
def test_nan_cosine_exhaustive(gpu, kernel):
    """0/0 of a zero row gives NaN (hnsw.rs:80-84); the reference's OrderedFloat puts NaN after every number, so an
    exhaustive search lists the zero rows last, and a top-10 never holds one.  Every distance of a zero query is NaN:
    any min(k, n) distinct ids, in unspecified order (the reference's priority_queue tie order)."""
    f64 = kernel == "f64"
    X, Q, zero = _nan_setup(f64)
    n = X.shape[0]
    g = _stage(gpu, X, COSINE)
    D, T = _reference(Q, X, COSINE, f64_kernel=f64)
    Z = np.zeros((2, X.shape[1]), X.dtype)
    DZ, TZ = _reference(Z, X, COSINE, f64_kernel=f64)
    assert np.isnan(D[:, zero]).all() and np.isnan(DZ).all()
    mode = -1 if f64 else int(kernel[-1])
    with _options(gpu, hnsw__mode=mode):
        search = g.search_f64 if f64 else g.search
        for k in (10, n):
            out = search(Q, k, n)
            _check_exhaustive(out, D, T, k, n)
            if k == n:
                assert np.array_equal(np.sort(out[0][:, n - zero.size:], axis=1), np.tile(np.sort(zero), (len(Q), 1)))
            else:
                assert not np.isin(out[0], zero).any()
            zi, zd, zc, _ = search(Z, k, n)
            assert np.all(zc == k) and np.isnan(zd).all()
            assert all(len(set(r.tolist())) == k for r in zi) and zi.max() < n


@pytest.mark.parametrize("mode", MODES)
def test_nan_non_exhaustive_built_index(gpu, mode):
    """ef < n on a device-built Cosine index that holds zero rows: every list ascends over its finite entries and NaN
    entries come only after them (a full beam whose furthest entry is NaN admits nothing more, as in the reference)"""
    n, dim, nq = (300, 32, 20) if EMU else (2000, 32, 200)
    X, Q = _data(n, dim, 110), _data(nq, dim, 111)
    zero = np.random.default_rng(112).choice(n, n // 50, replace=False)
    X[zero] = 0
    Q[:2] = 0
    g = gpu.HnswIndex.build(X, metric=COSINE, m=8, ef_construction=40)       # finishes, degree bounds hold
    ni, rp, ci, ep = g.export_levels()
    assert np.diff(rp[0].astype(np.int64)).max() <= 16
    for L in range(1, len(rp)):
        assert np.diff(rp[L].astype(np.int64)).max() <= 8
    with _options(gpu, hnsw__mode=mode):
        ids, dist, cnt, _ = g.search(Q, 10, 40)
    for q in range(nq):
        d = dist[q, :cnt[q]]
        fin = ~np.isnan(d)
        assert np.all(np.diff(fin.astype(np.int8)) <= 0), f"query {q}: NaN before a finite distance"
        assert np.all(np.diff(d[fin]) >= 0), f"query {q}: finite distances not ascending"
        if q < 2:                                       # zero queries: every distance is NaN
            assert cnt[q] >= 1 and not fin.any()
        else:
            assert np.isin(ids[q, :cnt[q]][~fin], zero).all()


# ---- h. top-k merge of per-shard lists (merge.cu) -----------------------------------------------------------------
def _merge_inputs(S, B, k, seed):
    """per-shard lists, nearest first: finite distances on a coarse grid (exact ties across shards), then maybe +inf,
    then maybe NaN, then NONE / +inf padding for lists shorter than k"""
    rng = np.random.default_rng(seed)
    pos = np.arange(k)
    length = rng.integers(0, k + 1, (S, B, 1))
    nfin = (rng.random((S, B, 1)) * (length + 1)).astype(np.int64)
    ninf = np.where(rng.random((S, B, 1)) < 0.2, (rng.random((S, B, 1)) * (length - nfin + 1)).astype(np.int64), 0)
    grid = np.sort(rng.integers(0, 16, (S, B, k)) / 4.0, axis=2)
    dist = np.where(pos < nfin, grid, np.where(pos < nfin + ninf, np.inf, np.where(pos < length, np.nan, np.inf)))
    ids = np.where(pos < length, rng.integers(0, 1 << 31, (S, B, k)), NONE)
    offsets = np.arange(S, dtype=np.uint64) * np.uint64(3_000_000_000) + np.uint64(5)      # >= 2^32 from shard 2 on
    return dist.astype(np.float32), ids.astype(np.uint32), offsets


def _merge_expected(dist, ids, offsets, k):
    """stable sort of every shard's entries by (dist with NaN after every number, shard, position); NONE dropped"""
    S, B, _ = dist.shape
    d = dist.transpose(1, 0, 2).reshape(B, S * k)                  # per query: shard-major, then position
    gid = (ids.astype(np.uint64) + offsets[:, None, None]).transpose(1, 0, 2).reshape(B, S * k)
    pad = (ids == NONE).transpose(1, 0, 2).reshape(B, S * k)
    o1 = np.argsort(d, axis=1, kind="stable")                      # NaN last
    o = np.take_along_axis(o1, np.argsort(np.take_along_axis(pad, o1, 1), axis=1, kind="stable"), 1)[:, :k]
    ed, ei, ep = (np.take_along_axis(a, o, 1) for a in (d, gid, pad))
    ei[ep] = np.iinfo(np.uint64).max
    ed[ep] = np.inf
    return ei, ed


def test_topk_merge_against_numpy(gpu):
    torch = _torch_cuda()
    if torch is None:
        pytest.skip("needs torch CUDA buffers")
    stream = torch.cuda.current_stream().cuda_stream
    for S in (1, 31, 32, 33, 64, 256):
        for k in (1, 10, 64):
            for B in (1, 5, 1001):
                dist, ids, offsets = _merge_inputs(S, B, k, seed=S * 1000 + k * 10 + B)
                dd = torch.from_numpy(dist).cuda()
                di = torch.from_numpy(ids.view(np.int32)).cuda()
                do = torch.from_numpy(offsets.view(np.int64)).cuda()
                oi = torch.empty((B, k), dtype=torch.int64, device="cuda")
                od = torch.empty((B, k), dtype=torch.float32, device="cuda")
                gpu.topk_merge_dev(dd.data_ptr(), di.data_ptr(), S, B, k, do.data_ptr(), oi.data_ptr(), od.data_ptr(),
                                   stream=stream)
                torch.cuda.synchronize()
                ei, ed = _merge_expected(dist, ids, offsets, k)
                gi, gd = oi.cpu().numpy().view(np.uint64), od.cpu().numpy()
                assert np.array_equal(gi, ei), (S, k, B)
                assert np.array_equal(gd, ed, equal_nan=True), (S, k, B)
    dd = torch.zeros((257, 1, 10), dtype=torch.float32, device="cuda")
    di = torch.zeros((257, 1, 10), dtype=torch.int32, device="cuda")
    do = torch.zeros(257, dtype=torch.int64, device="cuda")
    for S, k in ((257, 10), (4, 0)):
        with pytest.raises(gpu.CozoGpuError) as e:
            gpu.topk_merge_dev(dd.data_ptr(), di.data_ptr(), S, 1, k, do.data_ptr(), oi.data_ptr(), od.data_ptr(),
                               stream=stream)
        assert e.value.code == gpu.E_INVAL
