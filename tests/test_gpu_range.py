"""GPU tests of the range search (EmbeddingStore.search_range, range_graph, the sharded form and the
C ABI `isx_knn_range` / `isx_knn_range_sort`).

Two bars:
- against `search(q, 16)` on the same store, with no tolerance: a range score is bit for bit the score
  `search` reports, so a query's hits are exactly the prefix of its top-16 whose scores are >= τ;
- against the plain numpy references of `range_oracle` (fp64 and the oracle's fp32 scores): every row
  at least 1e-3 above τ is a hit and no row 1e-3 below it is."""

from __future__ import annotations

import numpy as np
import pytest
import torch

import range_oracle as R
from oracle import oracle as O

pytestmark = pytest.mark.gpu

from imagescry_b200 import _lib  # noqa: E402
from imagescry_b200 import search as S  # noqa: E402

BAND = 1e-3

# the shape table of test_gpu_knn.test_knn_vs_oracle without k: single CTAs and pairs, the resident
# query tile, several N-splits, ragged tiles
SHAPES = [
    (300, 7, 64), (256, 128, 64), (1000, 130, 128), (5000, 200, 1280), (4096, 64, 256), (3000, 50, 1280),
    (700, 33, 72), (40000, 300, 128), (2000, 257, 128), (2500, 513, 64), (60000, 1000, 256), (20000, 19000, 64),
    (9000, 700, 200), (5000, 300, 8),
]


def make(n, q, d, seed, dup=False):
    rng = np.random.default_rng(seed)
    store = O.bf16_round(rng.standard_normal((n, d)).astype(np.float32))
    queries = O.bf16_round(rng.standard_normal((q, d)).astype(np.float32))
    if dup and n > 20:
        store[17] = store[3]
        store[n - 1] = store[3]
        queries[0] = store[3]
    return store, queries


def bits(x: torch.Tensor) -> torch.Tensor:
    return x.contiguous().view(torch.int32)


def check_csr(offsets, idx, scores, tau, nq, lo=0, hi=2**31):
    """Structure of one result: offsets consistent, scores >= τ, (score desc, row asc), no duplicates."""
    assert offsets.dtype == torch.int64 and idx.dtype == torch.int64 and scores.dtype == torch.float32
    assert offsets.shape == (nq + 1,) and int(offsets[0]) == 0 and int(offsets[-1]) == idx.numel() == scores.numel()
    assert bool((offsets[1:] >= offsets[:-1]).all())
    if idx.numel() == 0:
        return
    assert bool((scores >= tau).all())
    assert int(idx.min()) >= lo and int(idx.max()) < hi
    q_of = torch.repeat_interleave(torch.arange(nq, device=idx.device), offsets[1:] - offsets[:-1])
    same = q_of[1:] == q_of[:-1]
    ordered = (scores[1:] < scores[:-1]) | ((scores[1:] == scores[:-1]) & (idx[1:] > idx[:-1]))
    assert bool((ordered | ~same).all()), "hits not ordered by (score desc, row asc) or duplicated"


def first16(offsets, idx, scores):
    """Q×16 of each query's first min(count, 16) hits (mask where valid) and the hit counts."""
    cnt = offsets[1:] - offsets[:-1]
    j = torch.arange(16, device=idx.device)
    valid = j[None, :] < cnt[:, None]
    pos = (offsets[:-1, None] + j[None, :]).clamp(max=max(idx.numel() - 1, 0))
    if idx.numel() == 0:
        return torch.full((len(cnt), 16), -1, device=idx.device), torch.zeros((len(cnt), 16), device=idx.device), valid, cnt
    return torch.where(valid, idx[pos], -1), torch.where(valid, scores[pos], 0.0), valid, cnt


def check_vs_search(res, s16, i16, tau):
    """A query with c <= 15 hits has exactly search's first c rows and scores, bit for bit, and
    search's (c + 1)-th score is < τ; a query with more hits starts with search's 16 entries."""
    offsets, idx, scores = res
    ri, rs, valid, cnt = first16(offsets, idx, scores)
    assert bool(((ri == i16) | ~valid).all()), "rows differ from search's"
    assert bool(((bits(rs) == bits(s16)) | ~valid).all()), "scores differ from search's bit for bit"
    short = cnt < 16
    nxt = s16.gather(1, cnt.clamp(max=15)[:, None])[:, 0]
    assert bool(((nxt < tau) | ~short).all()), "a search hit at or above τ is missing"


def check_fp64(res, store, queries, tau, index_base=0, exclude_self=False):
    offsets, idx, scores = (t.cpu().numpy() for t in res)
    ex = R.exact_scores(store, queries)
    if exclude_self:
        np.fill_diagonal(ex, -np.inf)
    for r in range(queries.shape[0]):
        got = idx[offsets[r]:offsets[r + 1]] - index_base
        must = np.nonzero(ex[r] >= tau + BAND)[0]
        assert np.isin(must, got).all(), f"query {r}: rows {np.setdiff1d(must, got)[:8]} missing"
        assert (ex[r, got] >= tau - BAND).all(), f"query {r}: rows far below τ returned"
        assert np.abs(scores[offsets[r]:offsets[r + 1]] - ex[r, got]).max(initial=0) <= BAND


def thresholds(st, q, s16):
    """τ such that queries have about 0, 1, 10 and 200 hits (medians over the queries)."""
    taus = [float(s16[:, 0].max()) + 0.01, float(s16[:, 0].median()), float(s16[:, 9].median())]
    if len(st) >= 200:
        qn = torch.nn.functional.normalize(q.float(), dim=1)
        en = torch.nn.functional.normalize(st.embeddings.float(), dim=1)
        kth = torch.cat([(qn[i:i + 1024] @ en.T).topk(200, dim=1).values[:, 199] for i in range(0, q.shape[0], 1024)])
        taus.append(float(kth.median()))
    return taus


@pytest.mark.parametrize("n,q,d", SHAPES)
def test_range_matches_search_exactly(n, q, d):
    store, queries = make(n, q, d, seed=n + q + d, dup=True)
    st = S.EmbeddingStore(torch.from_numpy(store).cuda())
    qt = torch.from_numpy(queries).cuda()
    s16, i16 = st.search(qt, 16)
    for tau in thresholds(st, qt, s16):
        res = st.search_range(qt, tau)
        check_csr(*res, tau, q, 0, n)
        check_vs_search(res, s16, i16, tau)


@pytest.mark.parametrize("n,q,d", [(5000, 200, 1280), (40000, 300, 128), (2500, 513, 64), (9000, 100, 200)])
def test_range_vs_fp64(n, q, d):
    store, queries = make(n, q, d, seed=7 * n + d)
    st = S.EmbeddingStore(torch.from_numpy(store).cuda())
    ex = R.exact_scores(store, queries)
    for hits in (1, 10, 200):
        tau = float(np.median(np.sort(ex, axis=1)[:, -hits]))
        res = st.search_range(torch.from_numpy(queries).cuda(), tau)
        check_csr(*res, tau, q, 0, n)
        check_fp64(res, store, queries, tau)


def test_range_correlated_store_many_hits():
    """A per-image store (49 correlated cells per image): hundreds to thousands of hits per query."""
    n, q, d, c = 49 * 800, 96, 256, 49
    rng = np.random.default_rng(5)
    groups = np.arange(n) // c
    base = rng.standard_normal((n // c, d)).astype(np.float32)
    store = O.bf16_round(base[groups] + 0.1 * rng.standard_normal((n, d)).astype(np.float32))
    queries = O.bf16_round(base[rng.integers(0, len(base), q)] + 0.3 * rng.standard_normal((q, d)).astype(np.float32))
    st = S.EmbeddingStore(torch.from_numpy(store).cuda(), groups=c)
    ex = R.exact_scores(store, queries)
    tau = float(np.median(np.sort(ex, axis=1)[:, -1500]))
    qt = torch.from_numpy(queries).cuda()
    res = st.search_range(qt, tau)
    cnt = (res[0][1:] - res[0][:-1]).cpu()
    assert int(cnt.max()) >= 1000 and int(cnt.median()) >= 200, cnt
    check_csr(*res, tau, q, 0, n)
    check_fp64(res, store, queries, tau)
    s16, i16 = st.search(qt, 16)
    check_vs_search(res, s16, i16, tau)
    # the oracle's fp32 scores agree too
    o_off, o_idx, _ = R.cosine_range(store, queries, tau)
    got, off = res[1].cpu().numpy(), res[0].cpu().numpy()
    for r in range(q):
        sym = np.setxor1d(got[off[r]:off[r + 1]], o_idx[o_off[r]:o_off[r + 1]])
        assert (np.abs(ex[r, sym] - tau) <= BAND).all(), f"query {r}"


def test_range_graph_excludes_self_and_keeps_duplicates():
    n, d = 3000, 128
    store, _ = make(n, 1, d, seed=11, dup=True)
    st = S.EmbeddingStore(torch.from_numpy(store).cuda())
    ex = R.exact_scores(store, store)
    np.fill_diagonal(ex, -np.inf)
    tau = float(np.median(np.sort(ex, axis=1)[:, -20]))
    res = st.range_graph(tau)
    check_csr(*res, tau, n, 0, n)
    check_fp64(res, store, store, tau, exclude_self=True)
    offsets, idx = res[0].cpu(), res[1].cpu()
    for r in range(n):
        assert r not in idx[offsets[r]:offsets[r + 1]].tolist()
    for a, b in [(3, 17), (3, n - 1), (17, 3), (17, n - 1), (n - 1, 3), (n - 1, 17)]:
        assert b in idx[offsets[a]:offsets[a + 1]].tolist()[:2], (a, b)
    s16, i16 = st.knn_graph(16)
    check_vs_search(res, s16, i16, tau)


def test_range_index_base_and_narrow_rows():
    store, queries = make(2000, 40, 37, seed=3)
    base = 123_456
    st0 = S.EmbeddingStore(torch.from_numpy(store).cuda())
    st = S.EmbeddingStore(torch.from_numpy(store).cuda(), index_base=base)
    qt = torch.from_numpy(queries).cuda()
    tau = 0.3
    r0, r1 = st0.search_range(qt, tau), st.search_range(qt, tau)
    assert torch.equal(r1[0], r0[0]) and torch.equal(r1[1], r0[1] + base) and torch.equal(bits(r1[2]), bits(r0[2]))
    check_csr(*r1, tau, 40, base, base + 2000)
    check_fp64(r1, store, queries, tau, index_base=base)
    s16, i16 = st.search(qt, 16)
    check_vs_search(r1, s16, i16, tau)


def test_range_zero_vectors_and_extreme_thresholds():
    n, q, d = 500, 6, 64
    store, queries = make(n, q, d, seed=9)
    store[[5, 260, 499]] = 0
    queries[2] = 0
    st = S.EmbeddingStore(torch.from_numpy(store).cuda())
    qt = torch.from_numpy(queries).cuda()
    s16, i16 = st.search(qt, 16)
    for tau in (0.0, -0.25):
        off, idx, sc = st.search_range(qt, tau)
        check_csr(off, idx, sc, tau, q, 0, n)
        check_fp64((off, idx, sc), store, queries, tau)
        check_vs_search((off, idx, sc), s16, i16, tau)  # zero scores too, bit for bit
        for r in range(q):
            hit = set(idx[off[r]:off[r + 1]].tolist())
            assert {5, 260, 499} <= hit  # score exactly 0
        assert int(off[3] - off[2]) == n  # a zero query scores 0 against every row
    off, idx, sc = st.search_range(qt, 0.05)
    assert not ({5, 260, 499} & set(idx.tolist()))
    assert int(off[3] - off[2]) == 0
    off, idx, sc = st.search_range(qt, -1.0001)
    assert torch.equal(off, torch.arange(q + 1, device="cuda") * n)
    check_csr(off, idx, sc, -1.0001, q, 0, n)
    off, idx, sc = st.search_range(qt, 1.0001)
    assert idx.numel() == 0 and torch.equal(off, torch.zeros(q + 1, dtype=torch.int64, device="cuda"))
    with pytest.raises(ValueError):
        st.search_range(qt, float("nan"))
    with pytest.raises(ValueError):
        st.search_range(qt, float("inf"))
    # empty store, zero queries
    empty = S.EmbeddingStore(torch.zeros((0, d), device="cuda"))
    off, idx, sc = empty.search_range(qt, 0.0)
    assert torch.equal(off, torch.zeros(q + 1, dtype=torch.int64, device="cuda")) and idx.numel() == 0
    off, idx, sc = st.search_range(qt[:0], 0.0)
    assert off.tolist() == [0] and idx.numel() == 0 and sc.numel() == 0


def _range_call(lib, st, qt, qr, tau, records_ptr, cap, count_ptr, rows=None, base=None, flags=0):
    rows = st.embeddings if rows is None else rows
    rn = st.rnorm if base is None else S.row_rnorm(rows)
    ws = torch.empty(_lib.KNN_RANGE_WORKSPACE_BYTES, dtype=torch.uint8, device="cuda")
    rc = lib.isx_knn_range(rows.data_ptr(), rn.data_ptr(), rows.shape[0], qt.data_ptr(), qr.data_ptr(), qt.shape[0],
                           qt.shape[1], tau, 0 if base is None else base, 0, flags, records_ptr, cap, count_ptr,
                           ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "isx_knn_range")


def test_range_overflow_guard_bands_retry_and_continue():
    from test_gpu_guard_bands import Guarded

    lib = _lib.load()
    n, q, d = 7000, 300, 128
    store, queries = make(n, q, d, seed=21)
    st = S.EmbeddingStore(torch.from_numpy(store).cuda())
    qt = S._as_bf16_matrix(torch.from_numpy(queries).cuda(), "q")
    qr = S.row_rnorm(qt)
    tau = 0.12
    full = st.search_range(qt, tau)
    hits = int(full[0][-1])
    assert hits > 2000
    # capacity below the hit count: count is exact, nothing is written past the records
    cap = hits // 3
    rec = Guarded(cap * 12)
    cnt = Guarded(8)
    _range_call(lib, st, qt, qr, tau, rec.ptr, cap, cnt.ptr)
    rec.check("isx_knn_range records")
    cnt.check("isx_knn_range count")
    assert int(cnt.as_tensor(torch.int64, (1,))[0]) == hits
    part = rec.as_tensor(torch.int32, (cap, 3))
    assert int(part[:, 0].min()) >= 0 and int(part[:, 0].max()) < q and int(part[:, 1].max()) < n
    # the ordering pass stays in bounds, with padding records in the input
    padded = torch.cat([part, torch.full((17, 3), -1, dtype=torch.int32, device="cuda")])
    ws = torch.empty(int(lib.isx_knn_range_sort_workspace_bytes(padded.shape[0], q)), dtype=torch.uint8, device="cuda")
    off, rows, sc = Guarded((q + 1) * 8), Guarded(cap * 4), Guarded(cap * 4)
    rc = lib.isx_knn_range_sort(padded.data_ptr(), padded.shape[0], q, off.ptr, rows.ptr, sc.ptr, ws.data_ptr(), ws.numel(),
                                torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "isx_knn_range_sort")
    for g, what in ((off, "offsets"), (rows, "rows"), (sc, "scores")):
        g.check(f"isx_knn_range_sort {what}")
    assert int(off.as_tensor(torch.int64, (q + 1,))[-1]) == cap
    # the wrapper's retry equals a call with room for everything
    small, small_hits = st.range_records(qt, qr, tau, _capacity=10)
    assert small_hits == hits and small.shape[0] == hits
    got = S.range_sort(small, q, hits)
    assert torch.equal(got[0], full[0]) and torch.equal(got[1], full[1]) and torch.equal(bits(got[2]), bits(full[2]))
    # two ISX_KNN_CONTINUE blocks (the cut inside a tile) equal one call on the whole store
    buf = torch.empty((hits, 3), dtype=torch.int32, device="cuda")
    count = torch.zeros(1, dtype=torch.int64, device="cuda")
    cut = 3001
    _range_call(lib, st, qt, qr, tau, buf.data_ptr(), hits, count.data_ptr(), rows=st.embeddings[:cut], base=0)
    _range_call(lib, st, qt, qr, tau, buf.data_ptr(), hits, count.data_ptr(), rows=st.embeddings[cut:], base=cut,
                flags=_lib.KNN_CONTINUE)
    assert int(count.item()) == hits
    blocks = S.range_sort(buf, q, hits)
    assert torch.equal(blocks[0], full[0]) and torch.equal(blocks[1], full[1]) and torch.equal(bits(blocks[2]), bits(full[2]))
    # bad arguments
    for bad in (dict(tau=float("nan")), dict(tau=float("inf")), dict(flags=_lib.KNN_PACKED)):
        with pytest.raises(ValueError):
            _range_call(lib, st, qt, qr, bad.get("tau", tau), buf.data_ptr(), hits, count.data_ptr(), flags=bad.get("flags", 0))


def _sort(lib, records, q, hits):
    offsets = torch.empty(q + 1, dtype=torch.int64, device="cuda")
    rows = torch.empty(hits, dtype=torch.int32, device="cuda")
    scores = torch.empty(hits, dtype=torch.float32, device="cuda")
    ws = torch.empty(int(lib.isx_knn_range_sort_workspace_bytes(records.shape[0], q)), dtype=torch.uint8, device="cuda")
    rc = lib.isx_knn_range_sort(records.data_ptr(), records.shape[0], q, offsets.data_ptr(), rows.data_ptr(),
                                scores.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "isx_knn_range_sort")
    return offsets, rows, scores


def test_range_sort_keeps_negative_zero():
    """A score of -0.0 keeps its sign through the ordering pass, and sorts with +0.0 by row (the k-NN
    search compares scores as floats)."""
    lib = _lib.load()
    f = torch.tensor([0.0, -0.0, 0.5, 0.0, -0.0, -0.25, 0.0, 0.75], dtype=torch.float32)
    rec = torch.stack([torch.tensor([0, 0, 0, 0, 0, 0, 1, 1]), torch.tensor([9, 4, 5, 7, 1, 3, 2, -1]),
                       f.view(torch.int32).long()], dim=1).to(torch.int32).cuda()
    offsets, rows, scores = _sort(lib, rec, 2, 7)
    assert offsets.tolist() == [0, 6, 7]
    assert rows.tolist() == [5, 1, 4, 7, 9, 3, 2]
    want = torch.tensor([0.5, -0.0, -0.0, 0.0, 0.0, -0.25, 0.0])
    assert torch.equal(bits(scores.cpu()), bits(want))


def test_range_sort_past_int32_record_index():
    """More than 2^31 / 3 records (3 * index no longer fits in int32): every record is read and sorted.
    About 45 GB of device memory."""
    lib = _lib.load()
    q, total = 1000, 716_000_017
    i = torch.arange(total, dtype=torch.int64, device="cuda")
    row = i // q
    rec = torch.empty((total, 3), dtype=torch.int32, device="cuda")
    rec[:, 0] = (i % q).to(torch.int32)
    rec[:, 1] = row.to(torch.int32)
    rec[:, 2] = (-(row % 1000).float() / 1000).view(torch.int32)
    want_rows = int(row.sum())
    del i, row
    offsets, rows, scores = _sort(lib, rec, q, total)
    del rec
    per = torch.full((q,), total // q, dtype=torch.int64)
    per[: total % q] += 1
    assert torch.equal(offsets.cpu(), torch.cat([torch.zeros(1, dtype=torch.int64), per.cumsum(0)]))
    assert int(rows.long().sum()) == want_rows and int(rows.max()) == (total - 1) // q
    assert bool((scores == -(rows % 1000).float() / 1000).all())
    # (score desc, row asc) inside every query's segment
    boundary = torch.zeros(total, dtype=torch.bool, device="cuda")
    boundary[offsets[1:-1]] = True
    ordered = (scores[1:] < scores[:-1]) | ((scores[1:] == scores[:-1]) & (rows[1:] > rows[:-1]))
    assert bool((ordered | boundary[1:]).all())


def test_range_capacity_follows_the_last_call():
    """The record buffer is sized from the previous call of the same kind, so a loose threshold does
    not inflate later strict calls; search_range and range_graph keep separate hints."""
    store, queries = make(20000, 400, 128, seed=31)
    st = S.EmbeddingStore(torch.from_numpy(store).cuda())
    qt = torch.from_numpy(queries).cuda()
    loose = st.search_range(qt, 0.1)
    assert st._range_hints[0] == int(loose[0][-1]) / 400 > 100
    strict = st.search_range(qt, 0.35)
    assert st._range_hints[0] == int(strict[0][-1]) / 400 < 1
    graph = st.range_graph(0.3)
    assert st._range_hints[_lib.KNN_EXCLUDE_SELF] == int(graph[0][-1]) / 20000
    assert st._range_hints[0] == int(strict[0][-1]) / 400
    again = st.search_range(qt, 0.1)  # one rerun at the exact count, same result
    assert torch.equal(again[0], loose[0]) and torch.equal(again[1], loose[1]) and torch.equal(bits(again[2]), bits(loose[2]))


def test_range_deterministic():
    store, queries = make(60000, 1000, 256, seed=4)
    st = S.EmbeddingStore(torch.from_numpy(store).cuda())
    qt = torch.from_numpy(queries).cuda()
    a = st.search_range(qt, 0.2)
    b = st.search_range(qt, 0.2)
    assert int(a[0][-1]) > 1000
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(bits(a[2]), bits(b[2]))


def test_full_size_range_sampled_queries():
    """1 M × 1280 store, 10 k queries, τ at about 10 hits per query: every query against search(16),
    64 sampled queries against an fp32 brute force over the full store."""
    n, d, q = 1_000_000, 1280, 10_000
    g = torch.Generator(device="cuda").manual_seed(1234)
    store = torch.empty((n, d), dtype=torch.bfloat16, device="cuda")
    for s0 in range(0, n, 1 << 18):
        e = min(n, s0 + (1 << 18))
        store[s0:e] = torch.randn((e - s0, d), generator=g, device="cuda").to(torch.bfloat16)
    queries = torch.randn((q, d), generator=g, device="cuda").to(torch.bfloat16)
    st = S.EmbeddingStore(store)
    s16, i16 = st.search(queries, 16)
    tau = float(s16[:, 9].median())
    res = st.search_range(queries, tau)
    check_csr(*res, tau, q, 0, n)
    check_vs_search(res, s16, i16, tau)
    pick = torch.arange(0, q, q // 64, device="cuda")[:64]
    qn = torch.nn.functional.normalize(queries[pick].float(), dim=1)
    rn = S.row_rnorm(store)
    offsets, idx = res[0].cpu(), res[1].cpu()
    for j, r in enumerate(pick.tolist()):
        sc = torch.cat([(qn[j:j + 1] @ store[s0:s0 + (1 << 18)].float().T)[0] * rn[s0:s0 + (1 << 18)]
                        for s0 in range(0, n, 1 << 18)])
        got = idx[offsets[r]:offsets[r + 1]].cuda()
        must = torch.nonzero(sc >= tau + BAND)[:, 0]
        assert bool(torch.isin(must, got).all()), r
        assert bool((sc[got] >= tau - BAND).all()), r


_WORKER = r"""
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["ISX_REPO"])
from imagescry_b200 import search as S
from oracle import oracle as O
rank = int(os.environ["ISX_RANK"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{os.environ['ISX_PORT']}", rank=rank, world_size=2)
rng = np.random.default_rng(0)
n, d = 20001, 128
store = O.bf16_round(rng.standard_normal((n, d)).astype(np.float32))
# query 0 sits between rows 10000 and 10001 (the shard cut): its hits span both shards
queries = O.bf16_round(np.concatenate([store[[10000]] + store[[10001]], rng.standard_normal((40, d))]).astype(np.float32))
b, e = S.shard_range(n, 2, rank)
sh = S.ShardedEmbeddingStore(torch.from_numpy(store[b:e]).cuda(), total_rows=n)
one = S.EmbeddingStore(torch.from_numpy(store).cuda())
qt = torch.from_numpy(queries).cuda()
for tau in (0.2, 0.5):
    got = sh.search_range(qt, tau)
    want = one.search_range(qt, tau)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), rank
    assert torch.equal(got[2].view(torch.int32), want[2].view(torch.int32)), rank
hits0 = got[1][got[0][0]:got[0][1]].tolist()
assert 10000 in hits0 and 10001 in hits0, hits0
dist.barrier()
dist.destroy_process_group()
print("OK", rank)
"""


def test_two_gpu_sharded_search_range(tmp_path):
    import os
    import socket
    import subprocess
    import sys

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from conftest import REPO

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(os.environ, ISX_REPO=REPO, ISX_PORT=str(port), ISX_RANK=str(r)),
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=300)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"OK {r}" in o, o
