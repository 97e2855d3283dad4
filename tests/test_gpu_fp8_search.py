"""GPU checks of the fp8 search: the E4M3 quantizer, the fp8 scan, the exact re-score and
`EmbeddingStore.search_fp8`, against tests/fp8_oracle.py and against `search`."""

from __future__ import annotations

import numpy as np
import pytest
import torch

import fp8_oracle as F
from oracle import oracle as O

pytestmark = pytest.mark.gpu

from imagescry_b200 import _lib  # noqa: E402
from imagescry_b200 import search as S  # noqa: E402
from test_gpu_guard_bands import Guarded, stream  # noqa: E402
from test_gpu_knn import check  # noqa: E402


def make(n, q, d, seed):
    rng = np.random.default_rng(seed)
    return (O.bf16_round(rng.standard_normal((n, d)).astype(np.float32)),
            O.bf16_round(rng.standard_normal((q, d)).astype(np.float32)))


def gpu(x):
    return torch.from_numpy(x).cuda().to(torch.bfloat16)


def quantize_c(x: np.ndarray):
    """isx_quantize_rows_e4m3 on the rows of x exactly as given (any d)."""
    xd = gpu(x)
    n, d = x.shape
    out = torch.empty((n, F.fp8_width(d)), dtype=torch.uint8, device="cuda")
    rn = torch.empty(n, dtype=torch.float32, device="cuda")
    _lib.check(_lib.load().isx_quantize_rows_e4m3(xd.data_ptr(), n, d, F.fp8_width(d), out.data_ptr(), rn.data_ptr(), stream()),
               "quantize")
    return out.cpu().numpy(), rn.cpu().numpy()


@pytest.mark.parametrize("d", [8, 37, 72, 1280])
def test_quantizer_matches_reference(d):
    rng = np.random.default_rng(d)
    n = 600
    x = rng.standard_normal((n, d)) * 10.0 ** rng.uniform(-30, 30, (n, 1))  # row norms across bf16's range
    x[3] = 0.0
    x[4] = -0.0
    x[5, :] = 0.0
    x[5, 0] = 1e-40  # a lone bf16 subnormal
    x[6, : min(d, 6)] = [1.0, 2.0**-12, 2.0**-15, 3 * 2.0**-17, 2.0**-18, 1.5 * 2.0**-18][: min(d, 6)]  # subnormal / zero outputs
    x[8] = rng.standard_normal(d)
    x[7] = x[8] * 2.0**40  # power-of-two multiples
    x = O.bf16_round(x.astype(np.float32))
    got, rn = quantize_c(x)
    ref, rref = F.quantize(x)
    assert np.array_equal(got, ref), np.argwhere(got != ref)[:5]
    ulp = np.abs(rn.view(np.int32).astype(np.int64) - rref.view(np.int32).astype(np.int64))
    assert ulp.max() <= 1
    assert np.array_equal(got[7], got[8]) and rn[7] == rn[8]
    assert np.all((got[3] & 0x7F) == 0) and rn[3] == np.float32(1e12)


SCAN_SHAPES = [
    (300, 7, 64, 10),        # one CTA, one partial tile
    (1000, 130, 128, 10),    # CTA pairs, resident query tile, one k-block
    (5000, 200, 1280, 10),   # streamed query tiles, 10 k-blocks
    (9000, 700, 400, 16),    # resident, 4 k-blocks, ragged last (400 % 128 = 16)
    (9000, 300, 600, 10),    # streamed, d16 = 608 > 512, ragged last k-block
    (3000, 50, 1280, 100),   # one CTA, 256-entry buffers
    (2500, 513, 72, 100),    # pairs, 256-entry buffers, d16 = 80
    (40000, 300, 128, 10),   # several N-splits
    (20000, 19000, 64, 10),  # several items per unit
    (60000, 1000, 256, 32),  # pairs x splits, 256-entry buffers
    (5000, 300, 8, 5),       # d16 = 16
]


@pytest.mark.parametrize("n,q,d,k", SCAN_SHAPES)
def test_scan_vs_reference(n, q, d, k):
    store, queries = make(n, q, d, seed=n + q + d + k)
    st = S.EmbeddingStore(gpu(store), fp8=True)
    scores, idx = st.scan_fp8(gpu(queries), k)
    sq, qq = F.dequantize(F.quantize(store)[0]), F.dequantize(F.quantize(queries)[0])
    check(sq, qq, k, scores, idx.to(torch.int64))


@pytest.mark.parametrize("k", [1, 10, 16, 40])
def test_scan_ties_between_power_of_two_multiples(k):
    """Power-of-two multiples quantize to identical bytes, so their fp8 scores tie exactly; a dozen
    copies of every prototype are spread over tiles, splits and CTAs, and each tie goes to the lower row."""
    rng = np.random.default_rng(91 + k)
    n, q, d, base = 6000, 300, 256, 500
    proto = O.bf16_round(rng.standard_normal((base, d)).astype(np.float32))
    store = O.bf16_round(proto[rng.integers(0, base, n)] * np.exp2(rng.integers(-3, 4, (n, 1))).astype(np.float32))
    queries = O.bf16_round(proto[rng.integers(0, base, q)] + 0.25 * rng.standard_normal((q, d)).astype(np.float32))
    st = S.EmbeddingStore(gpu(store), fp8=True)
    scores, idx = st.scan_fp8(gpu(queries), k)
    ref_s, ref_i = F.scan(store, queries, k)
    assert np.array_equal(idx.cpu().numpy(), ref_i)
    assert np.abs(scores.cpu().numpy() - ref_s).max() <= 1e-3
    assert (ref_s[:, 0] == ref_s[:, min(k, 3) - 1]).mean() > 0.9


def test_rescore_hand_made_candidates():
    rng = np.random.default_rng(5)
    n, q, d, base = 3000, 40, 200, 7000
    store, queries = make(n, q, d, seed=5)
    store[100] = store[7]  # duplicated store rows: equal scores, the lower row first
    store[2999] = store[7]
    st = S.EmbeddingStore(gpu(store), index_base=base)
    for kc, k in [(16, 10), (5, 10), (40, 40), (128, 100), (100, 7)]:
        cand = rng.integers(base, base + n, (q, kc))
        cand[:, rng.random(kc) < 0.2] = -1  # padding anywhere
        cand[0, : min(kc, 3)] = [base + 7, base + 100, base + 2999][: min(kc, 3)]
        cand[1, :] = -1
        cand[2, -1] = cand[2, 0]  # a row listed twice
        ref_s, ref_i = F.rescore(store, queries, cand, k, index_base=base)
        outs = [st.rescore(gpu(queries), torch.from_numpy(cand).cuda(), k) for _ in range(3)]
        s, i = outs[0]
        for s2, i2 in outs[1:]:
            assert torch.equal(s2.view(torch.int32), s.view(torch.int32)) and torch.equal(i2, i)
        s, i = s.cpu().numpy(), i.cpu().numpy()
        assert np.array_equal(i, ref_i)
        valid = ref_i >= 0
        assert np.all(np.isneginf(s[~valid]))
        assert np.abs(s[valid] - ref_s[valid]).max() <= 1e-5


@pytest.mark.parametrize("n,q,d,k,c", [(5000, 200, 1280, 10, 16), (20000, 300, 256, 10, 32), (3000, 130, 72, 16, 16),
                                       (4000, 50, 128, 1, 100)])
def test_search_fp8_is_rescore_of_scan(n, q, d, k, c):
    store, queries = make(n, q, d, seed=n + k + c)
    st = S.EmbeddingStore(gpu(store), fp8=True)
    qd = gpu(queries)
    s, i = st.search_fp8(qd, k, candidates=c)
    _, cand = st.scan_fp8(qd, c)
    rs, ri = st.rescore(qd, cand, k)
    assert torch.equal(s.view(torch.int32), rs.view(torch.int32)) and torch.equal(i, ri.to(torch.int64))
    ref_s, ref_i = F.rescore(store, queries, cand.cpu().numpy(), k)
    assert np.array_equal(i.cpu().numpy(), ref_i)
    assert np.abs(s.cpu().numpy() - ref_s).max() <= 1e-5
    # within 1e-5 of search's score for the same pair
    es, ei = st.search(qd, min(128, max(k, 64)))
    es, ei, s, i = es.cpu().numpy(), ei.cpu().numpy(), s.cpu().numpy(), i.cpu().numpy()
    for r in range(q):
        pos = {int(j): t for t, j in enumerate(ei[r])}
        for t, j in enumerate(i[r]):
            if int(j) in pos:
                assert abs(s[r, t] - es[r, pos[int(j)]]) <= 1e-5


def _store_randn(n, d, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    store = torch.empty((n, d), dtype=torch.bfloat16, device="cuda")
    for s0 in range(0, n, 1 << 17):
        store[s0:s0 + (1 << 17)] = torch.randn((min(n, s0 + (1 << 17)) - s0, d), generator=g, device="cuda").to(torch.bfloat16)
    return store, torch.randn((10_000, d), generator=g, device="cuda").to(torch.bfloat16)


def test_recall_at_metric_shape():
    """1 M x 1280 N(0, 1) rows, 10 k queries: recall@10 of search_fp8 (16 candidates) against search."""
    store, queries = _store_randn(1_000_000, 1280, 2024)
    st = S.EmbeddingStore(store, fp8=True)
    es, ei = st.search(queries, 10)
    s, i = st.search_fp8(queries, 10)
    hit = (i[:, :, None] == ei[:, None, :]).any(dim=2)
    recall = float(hit.float().mean())
    assert recall >= 0.99, recall
    # a returned row that search also returned carries search's score to 1e-5
    same = i[:, :, None] == ei[:, None, :]
    diff = (s[:, :, None] - es[:, None, :]).abs()
    assert float(diff[same].max()) <= 1e-5


def test_correlated_store_finds_every_image():
    """Per-cell store (256 cells per image = base + 0.1 noise): every image of search's top 10 is among the
    images of search_fp8's top `candidates`."""
    n, d, cells = 1_000_000 - 1_000_000 % 256, 1280, 256
    g = torch.Generator(device="cuda").manual_seed(7)
    base = torch.randn((n // cells, d), generator=g, device="cuda")
    store = torch.empty((n, d), dtype=torch.bfloat16, device="cuda")
    for s0 in range(0, n, 1 << 17):
        e = min(n, s0 + (1 << 17))
        store[s0:e] = (base[torch.arange(s0, e, device="cuda") // cells] + 0.1 * torch.randn((e - s0, d), generator=g, device="cuda")).to(torch.bfloat16)
    pick = torch.randint(0, n // cells, (2000,), generator=g, device="cuda")
    queries = (base[pick] + 0.3 * torch.randn((2000, d), generator=g, device="cuda")).to(torch.bfloat16)
    st = S.EmbeddingStore(store, fp8=True)
    _, ei = st.search(queries, 10)
    _, i = st.search_fp8(queries, S.FP8_CANDIDATES, candidates=S.FP8_CANDIDATES)
    want, got = (ei // cells).cpu().numpy(), (i // cells).cpu().numpy()
    missing = [r for r in range(want.shape[0]) if not set(want[r].tolist()) <= set(got[r].tolist())]
    assert not missing, f"{len(missing)} queries miss an image, e.g. {missing[:5]}"


def test_arguments_and_store_without_fp8():
    store, queries = make(500, 9, 64, seed=11)
    plain = S.EmbeddingStore(gpu(store))
    with pytest.raises(ValueError):
        plain.search_fp8(gpu(queries), 10)
    st = S.EmbeddingStore(gpu(store), fp8=True)
    assert st.embeddings_e4m3.shape == (500, 64) and st.embeddings_e4m3.dtype == torch.uint8
    for k, c in [(0, 16), (17, 16), (10, 129), (10, 0), (True, 16)]:
        with pytest.raises(ValueError):
            st.search_fp8(gpu(queries), k, candidates=c)
    s0, i0 = st.search_fp8(torch.zeros((0, 64), device="cuda"), 10)
    assert s0.shape == (0, 10) and i0.shape == (0, 10) and i0.dtype == torch.int64
    empty = S.EmbeddingStore(torch.zeros((0, 64), device="cuda"), fp8=True)
    s, i = empty.search_fp8(gpu(queries), 10)
    ps, pi = empty.search(gpu(queries), 10)
    assert torch.equal(s, ps) and torch.equal(i, pi)
    # zero query: every score 0, ties to the lowest rows, like search
    zq = np.zeros((1, 64), np.float32)
    s, i = st.search_fp8(gpu(zq), 10)
    assert torch.all(s == 0) and i[0].tolist() == list(range(10))
    lib = _lib.load()
    q8, qr8 = S.quantize_e4m3(gpu(queries))
    ws = torch.empty(lib.isx_knn_workspace_bytes(500, 9, 64, 10), dtype=torch.uint8, device="cuda")
    out_s = torch.empty((9, 10), device="cuda")
    out_i = torch.empty((9, 10), dtype=torch.int32, device="cuda")
    for d16, k in [(72, 10), (64, 129), (0, 10)]:
        rc = lib.isx_knn_search_fp8(st.embeddings_e4m3.data_ptr(), st.rnorm_e4m3.data_ptr(), 500, q8.data_ptr(), qr8.data_ptr(), 9,
                                    d16, k, 0, out_s.data_ptr(), out_i.data_ptr(), ws.data_ptr(), ws.numel(), stream())
        assert rc == _lib.ERR_INVALID_ARG
    assert lib.isx_quantize_rows_e4m3(q8.data_ptr(), 9, 64, 40, q8.data_ptr(), qr8.data_ptr(), stream()) == _lib.ERR_INVALID_ARG
    cand = torch.zeros((9, 4), dtype=torch.int32, device="cuda")
    assert lib.isx_knn_rescore(st.embeddings.data_ptr(), st.rnorm.data_ptr(), 500, q8.data_ptr(), qr8.data_ptr(), 9, 64, cand.data_ptr(),
                               129, 0, 10, out_s.data_ptr(), out_i.data_ptr(), stream()) == _lib.ERR_INVALID_ARG


@pytest.mark.parametrize("n,q,d,k,kc", [(3000, 70, 64, 10, 16), (700, 33, 72, 100, 128), (5000, 257, 400, 16, 16),
                                        (2500, 513, 600, 100, 40), (300, 7, 8, 5, 3)])
def test_outputs_stay_in_bounds(n, q, d, k, kc):
    lib = _lib.load()
    store, queries = make(n, q, d, seed=n + q)
    sd, qd = gpu(store), gpu(queries)
    d16 = F.fp8_width(d)
    s8, srn = Guarded(n * d16), Guarded(n * 4)
    q8, qrn = Guarded(q * d16), Guarded(q * 4)
    _lib.check(lib.isx_quantize_rows_e4m3(sd.data_ptr(), n, d, d16, s8.ptr, srn.ptr, stream()), "quantize")
    _lib.check(lib.isx_quantize_rows_e4m3(qd.data_ptr(), q, d, d16, q8.ptr, qrn.ptr, stream()), "quantize")
    for g, what in [(s8, "store e4m3"), (srn, "store rnorm"), (q8, "query e4m3"), (qrn, "query rnorm")]:
        g.check(what)
    ws = Guarded(int(lib.isx_knn_workspace_bytes(n, q, d16, kc)))
    cs, ci = Guarded(q * kc * 4), Guarded(q * kc * 4)
    _lib.check(lib.isx_knn_search_fp8(s8.ptr, srn.ptr, n, q8.ptr, qrn.ptr, q, d16, kc, 0, cs.ptr, ci.ptr, ws.ptr, ws.nbytes,
                                      stream()), "scan")
    for g, what in [(cs, "scan scores"), (ci, "scan rows"), (ws, "scan workspace")]:
        g.check(what)
    st = S.EmbeddingStore(sd)
    qr = S.row_rnorm(qd)
    out_s, out_i = Guarded(q * k * 4), Guarded(q * k * 4)
    _lib.check(lib.isx_knn_rescore(sd.data_ptr(), st.rnorm.data_ptr(), n, qd.data_ptr(), qr.data_ptr(), q, d, ci.ptr, kc, 0, k,
                                   out_s.ptr, out_i.ptr, stream()), "rescore")
    out_s.check("rescore scores")
    out_i.check("rescore rows")
    idx = out_i.as_tensor(torch.int32, (q, k))
    assert int(idx.max()) < n and int(idx[:, : min(k, kc)].min()) >= 0


def test_sharded_merge_keeps_exact_scores():
    """Row shards (emulated on one device) each scan and re-score their own rows, and the packed records
    are merged as `ShardedEmbeddingStore.search_fp8` merges them.  Every merged score is bit for bit the
    unsharded store's exact score of that row, and the result is the exact top-k of the union of the
    shards' candidates, which holds the unsharded candidates."""
    store, queries = make(20000, 64, 256, seed=8)
    qd = gpu(queries)
    full = S.EmbeddingStore(gpu(store), fp8=True)
    k, c = 10, 16
    _, cand_full = full.scan_fp8(qd, c)
    recs, cands = [], []
    for r in range(4):
        b, e = S.shard_range(len(store), 4, r)
        part = S.EmbeddingStore(gpu(store[b:e]), index_base=b, fp8=True)
        s, i = part.search_fp8_raw(qd, k, candidates=c)
        recs.append(S.pack_records(s, i))
        cands.append(part.scan_fp8(qd, c)[1])
    ms, mi = S.merge_topk_packed(torch.stack(recs), k)
    union = torch.cat(cands, dim=1)
    us, ui = full.rescore(qd, union, k)
    assert torch.equal(ms.view(torch.int32), us.view(torch.int32)) and torch.equal(mi, ui)
    for r in range(qd.shape[0]):
        assert set(cand_full[r].tolist()) <= set(union[r].tolist())
