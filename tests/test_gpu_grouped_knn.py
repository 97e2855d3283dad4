"""GPU parity of the image-level (grouped) search against the CPU reference `grouped_oracle.cosine_knn_groups`.

Tolerance (the rule of test_gpu_knn.check): scores within 1e-3; representative rows and groups
identical except where every differing group's exact score lies within 1e-3 of the exact k-th
distinct-group score."""

from __future__ import annotations

import numpy as np
import pytest
import torch

import grouped_oracle as G
from oracle import oracle as O

pytestmark = pytest.mark.gpu

from imagescry_b200 import _lib  # noqa: E402
from imagescry_b200 import search as S  # noqa: E402

SCORE_TOL = 1e-3

# the shape table of test_gpu_knn.test_knn_vs_oracle: every kernel variant (CAP 32 / 256, single CTAs
# and pairs, the resident query tile, several N-splits, ragged tiles)
SHAPES = [
    (300, 7, 64, 10), (256, 128, 64, 1), (1000, 130, 128, 10), (5000, 200, 1280, 10), (4096, 64, 256, 16),
    (3000, 50, 1280, 100), (700, 33, 72, 100), (40000, 300, 128, 10), (2000, 257, 128, 10), (2500, 513, 64, 100),
    (60000, 1000, 256, 32), (20000, 19000, 64, 10), (9000, 700, 200, 16), (5000, 300, 8, 5),
]


def make(n, q, d, seed, correlated=False, groups=None):
    rng = np.random.default_rng(seed)
    if correlated:
        # every group's rows = one base vector + small noise: many cells of the best images pass
        base = rng.standard_normal((int(groups.max()) + 1, d)).astype(np.float32)
        store = O.bf16_round(base[groups] + 0.1 * rng.standard_normal((n, d)).astype(np.float32))
        queries = O.bf16_round(base[rng.integers(0, len(base), q)] + 0.3 * rng.standard_normal((q, d)).astype(np.float32))
    else:
        store = O.bf16_round(rng.standard_normal((n, d)).astype(np.float32))
        queries = O.bf16_round(rng.standard_normal((q, d)).astype(np.float32))
    return store, queries


def layout(kind, n, seed=0):
    """(groups argument of EmbeddingStore or None, per-row group ids)"""
    if kind == "ids":  # random, non-contiguous ids: only the C ABI takes these
        return None, np.random.default_rng(seed).integers(0, max(1, n // 50), n)
    if kind == "one":
        return n, np.zeros(n, np.int64)
    if kind == "offsets":
        sizes = np.random.default_rng(seed).integers(1, 300, n)
        off = np.concatenate([[0], np.cumsum(sizes)])
        off = off[off < n]
        off = np.append(off, n)
        return torch.from_numpy(off), np.searchsorted(off, np.arange(n), side="right") - 1
    c = int(kind)
    n_fit = n - n % c
    return c, np.arange(n_fit) // c


def grouped_raw(store_t, rnorm, row_group_t, queries_t, k, index_base=0):
    lib = _lib.load()
    q, d = queries_t.shape
    n = store_t.shape[0]
    qr = S.row_rnorm(queries_t)
    ws = torch.empty(max(int(lib.isx_knn_workspace_bytes(max(n, 1), q, d, k)), 256), dtype=torch.uint8, device="cuda")
    out_s = torch.empty((q, k), dtype=torch.float32, device="cuda")
    out_r = torch.empty((q, k), dtype=torch.int32, device="cuda")
    out_g = torch.empty((q, k), dtype=torch.int32, device="cuda")
    rc = lib.isx_knn_search_grouped(store_t.data_ptr(), rnorm.data_ptr(), row_group_t.data_ptr(), n, queries_t.data_ptr(),
                                    qr.data_ptr(), q, d, k, index_base, out_s.data_ptr(), out_r.data_ptr(),
                                    out_g.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "isx_knn_search_grouped")
    return out_s, out_r, out_g


def check(store, queries, k, groups, scores, rows, images, index_base=0):
    ref_s, ref_r, ref_g = G.cosine_knn_groups(store, queries, k, groups, index_base=index_base)
    scores, rows, images = (t.cpu().numpy() for t in (scores, rows, images))
    valid = ref_r >= 0
    assert np.array_equal(rows >= 0, valid) and np.array_equal(images >= 0, valid)
    assert np.all(np.isneginf(scores[~valid]))
    assert np.abs(scores[valid] - ref_s[valid]).max(initial=0.0) <= SCORE_TOL
    for r in range(scores.shape[0]):
        row_s, row_i = scores[r][valid[r]], rows[r][valid[r]]
        assert np.array_equal(np.lexsort((row_i, -row_s)), np.arange(len(row_s))), f"row {r} not ordered"
        assert len(set(images[r][valid[r]].tolist())) == valid[r].sum(), f"row {r}: an image twice"
    g_arr = np.asarray(groups)
    ok_rows = valid & (g_arr[np.clip(rows - index_base, 0, None)] == images)
    assert np.array_equal(ok_rows, valid), "a representative row outside its reported image"
    exact = np.array_equal(rows, ref_r)
    if not exact:
        sn = store * O.row_rnorm(store)[:, None]
        qn = queries * O.row_rnorm(queries)[:, None]
        for r in np.nonzero((rows != ref_r).any(axis=1))[0]:
            full = qn[r] @ sn.T
            gbest = {}
            for g, s in zip(g_arr.tolist(), full.tolist()):
                gbest[g] = max(gbest.get(g, -np.inf), s)
            kth = sorted(gbest.values())[-k] if len(gbest) >= k else -np.inf
            for g in set(images[r].tolist()) ^ set(ref_g[r].tolist()):
                assert g >= 0, f"row {r}: padding mismatch"
                assert abs(gbest[g] - kth) < SCORE_TOL, f"row {r}: image {g} differs beyond tolerance"
            # same image, other representative: only between cells whose scores tie within tolerance
            for j in np.nonzero((rows[r] != ref_r[r]) & (images[r] == ref_g[r]))[0]:
                assert abs(full[rows[r, j] - index_base] - full[ref_r[r, j] - index_base]) < SCORE_TOL
    return exact


@pytest.mark.parametrize("n,q,d,k", SHAPES)
@pytest.mark.parametrize("kind", ["256", "7", "one", "ids", "offsets"])
def test_grouped_vs_oracle(n, q, d, k, kind):
    arg, groups = layout(kind, n, seed=n + k)
    n = len(groups)
    store, queries = make(n, q, d, seed=n + q + d + k)
    st = torch.from_numpy(store).cuda().to(torch.bfloat16)
    qt = torch.from_numpy(queries).cuda().to(torch.bfloat16)
    if arg is None:
        s, r, g = grouped_raw(st, S.row_rnorm(st), torch.from_numpy(groups.astype(np.int32)).cuda(), qt, k)
    else:
        store_obj = S.EmbeddingStore(st, groups=arg)
        s, r, g = store_obj.search_images_raw(qt, k)
        s2, img, cells = store_obj.search_images(qt, k)
        assert torch.equal(s2, s) and torch.equal(img, g.to(torch.int64))
        first = store_obj.group_first_row.cpu()
        want = torch.where(g.cpu() >= 0, r.cpu().to(torch.int64) - first[g.cpu().clamp(min=0).long()], torch.tensor(-1))
        assert torch.equal(cells.cpu(), want)
    check(store, queries, k, groups, s, r, g)


@pytest.mark.parametrize("n,q,d,k,c", [(20480, 300, 256, 10, 256), (20006, 300, 1280, 10, 7), (9216, 140, 128, 100, 256),
                                       (40000, 600, 64, 16, 64)])
def test_grouped_correlated_cells(n, q, d, k, c):
    """Cells of one image = base + small noise: the best images' cells pass the distinct-image
    threshold in bulk."""
    groups = np.arange(n) // c
    store, queries = make(n, q, d, seed=n + c + k, correlated=True, groups=groups)
    st = S.EmbeddingStore(torch.from_numpy(store).cuda(), groups=c)
    s, r, g = st.search_images_raw(torch.from_numpy(queries).cuda(), k)
    check(store, queries, k, groups, s, r, g)


@pytest.mark.parametrize("k", [1, 10, 16, 17, 128])
@pytest.mark.parametrize("n,q,d", [(40000, 300, 128), (20000, 700, 256), (5000, 100, 1280)])
def test_grouped_c1_bit_identical_to_search(n, q, d, k):
    """One row per group: the grouped launch runs the same kernel variant as `search`, so scores and
    rows are bit-identical."""
    store, queries = make(n, q, d, seed=k + d)
    st = S.EmbeddingStore(torch.from_numpy(store).cuda(), groups=1)
    qt = torch.from_numpy(queries).cuda()
    ws, wi = st.search_raw(qt, k)
    s, r, g = st.search_images_raw(qt, k)
    assert torch.equal(s, ws) and torch.equal(r, wi) and torch.equal(g, wi)


@pytest.mark.parametrize("k", [10, 100])
def test_grouped_blocks_merge_equals_one_search(k):
    """Two store blocks (the second with index_base) searched separately and merged with
    isx_topk_merge_grouped equal one search, including the image cut by the block boundary."""
    n, q, d, c = 30000, 200, 128, 64
    groups = np.arange(n) // c
    store, queries = make(n, q, d, seed=k, correlated=True, groups=groups)
    cut = 15000 + 17  # inside image 234
    qt = torch.from_numpy(queries).cuda().to(torch.bfloat16)
    st = torch.from_numpy(store).cuda().to(torch.bfloat16)
    rg = torch.from_numpy(groups.astype(np.int32)).cuda()
    rn = S.row_rnorm(st)
    parts = [grouped_raw(st[:cut], rn[:cut], rg[:cut], qt, k, 0), grouped_raw(st[cut:], rn[cut:], rg[cut:], qt, k, cut)]
    rec = torch.stack([S.pack_group_records(*p) for p in parts])
    ms, mr, mg = S.merge_topk_groups(rec)
    ws, wr, wg = grouped_raw(st, rn, rg, qt, k)
    assert torch.equal(mr, wr) and torch.equal(mg, wg) and torch.equal(ms, ws)
    for r_ in range(q):
        assert len(set(mg[r_].tolist())) == k
    check(store, queries, k, groups, ms, mr, mg)
    # the oracle's merge of the same records agrees
    os_, or_, og = G.topk_merge_groups(*(torch.stack([p[i] for p in parts]).cpu().numpy() for i in range(3)), k)
    assert np.array_equal(or_, mr.cpu().numpy()) and np.array_equal(og, mg.cpu().numpy())


def test_grouped_mixed_blobs_store_and_validation():
    from imagescry_b200 import store_format as F

    rng = np.random.default_rng(13)
    shapes = [(3, 4), (5, 6), (3, 4), (2, 7), (5, 6), (3, 4), (16, 16), (1, 1)] * 5
    maps = [rng.standard_normal((72, h, w)).astype(np.float32) for h, w in shapes]
    records = [(O.blob_encode(m), 72, m.shape[1], m.shape[2]) for m in maps]
    store, offsets = F.store_from_mixed_blobs(records)
    groups = np.searchsorted(offsets.numpy(), np.arange(len(store)), side="right") - 1
    q = torch.from_numpy(np.stack([maps[3][:, 1, 5], maps[6][:, 9, 2]])).cuda()
    s, img, cells = store.search_images(q, 5)
    assert img[:, 0].tolist() == [3, 6] and cells[:, 0].tolist() == [1 * 7 + 5, 9 * 16 + 2]
    _, r, g = store.search_images_raw(q, 5)
    check(store.embeddings.float().cpu().numpy(), O.bf16_round(q.cpu().numpy()), 5, groups, s, r, g)
    per_cell = F.store_from_maps(torch.from_numpy(np.stack(maps[:3:2])))
    assert per_cell.row_group.tolist() == [0] * 12 + [1] * 12
    pooled = F.store_from_maps(torch.from_numpy(np.stack(maps[:3:2])), pool="mean")
    assert pooled.row_group.tolist() == [0, 1]
    plain = S.EmbeddingStore(torch.randn(10, 64).cuda())
    with pytest.raises(ValueError):
        plain.search_images(torch.randn(1, 64).cuda(), 3)
    with pytest.raises(ValueError):
        per_cell.search_images(q, 129)
    with pytest.raises(ValueError):
        S.EmbeddingStore(torch.randn(10, 64).cuda(), groups=3)


def _device_store(n, d, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    store = torch.empty((n, d), dtype=torch.bfloat16, device="cuda")
    for s0 in range(0, n, 1 << 18):
        e = min(n, s0 + (1 << 18))
        store[s0:e] = torch.randn((e - s0, d), generator=g, device="cuda").to(torch.bfloat16)
    return store, g


def test_full_size_grouped_sampled_queries():
    """1 M x 1280 with 256 cells per image, k = 10: 64 sampled queries against an fp32 brute force
    over the full store, reduced to the best cell per image."""
    n, d, q, c, k = 1_000_000, 1280, 10_000, 256, 10
    n = n - n % c
    store, g = _device_store(n, d, 1234)
    queries = torch.randn((q, d), generator=g, device="cuda").to(torch.bfloat16)
    st = S.EmbeddingStore(store, groups=c)
    scores, images, cells = st.search_images(queries, k)
    assert int(images.min()) >= 0 and int(images.max()) < n // c and int(cells.min()) >= 0 and int(cells.max()) < c
    assert torch.all(scores[:, 1:] <= scores[:, :-1])
    pick = torch.arange(0, q, q // 64, device="cuda")[:64]
    qn = torch.nn.functional.normalize(queries[pick].float(), dim=1)
    best = torch.full((64, n // c), -float("inf"), device="cuda")
    for s0 in range(0, n, 1 << 17):
        e = min(n, s0 + (1 << 17))
        sc = qn @ torch.nn.functional.normalize(store[s0:e].float(), dim=1).T
        best[:, s0 // c:e // c] = sc.view(64, -1, c).amax(dim=2)
    ex_s, ex_i = best.topk(k, dim=1)
    got_s, got_i = scores[pick], images[pick]
    assert (got_s - ex_s).abs().max().item() <= SCORE_TOL
    kth = ex_s[:, -1:]
    for r_ in range(64):
        for j in set(got_i[r_].tolist()) ^ set(ex_i[r_].tolist()):
            assert abs(best[r_, j].item() - kth[r_].item()) < SCORE_TOL
    # the representative cell is the image's best cell
    rows = images[pick] * c + cells[pick]
    rep = (qn.unsqueeze(1) * torch.nn.functional.normalize(store[rows.view(-1)].float(), dim=1).view(64, k, d)).sum(-1)
    assert (rep - got_s).abs().max().item() <= SCORE_TOL


class Guarded:
    """A device buffer of `nbytes` with a 64 KiB guard band on either side (test_gpu_guard_bands)."""

    GUARD, PATTERN = 1 << 16, 0xA5

    def __init__(self, nbytes: int) -> None:
        self.nbytes = nbytes
        pad = (256 - nbytes % 256) % 256
        self.raw = torch.full((2 * self.GUARD + nbytes + pad,), self.PATTERN, dtype=torch.uint8, device="cuda")
        self.view = self.raw[self.GUARD:self.GUARD + nbytes]
        self.ptr = self.view.data_ptr()

    def check(self, what: str) -> None:
        torch.cuda.synchronize()
        assert bool((self.raw[:self.GUARD] == self.PATTERN).all()), f"{what}: wrote before the buffer"
        assert bool((self.raw[self.GUARD + self.nbytes:] == self.PATTERN).all()), f"{what}: wrote past the buffer"


@pytest.mark.parametrize("n,q,d,k", [(300, 7, 64, 10), (2500, 513, 64, 100), (9000, 300, 200, 16), (700, 33, 72, 128)])
def test_grouped_entry_points_stay_in_bounds(n, q, d, k):
    lib = _lib.load()
    store, queries = make(n, q, d, seed=n)
    st = torch.from_numpy(store).cuda().to(torch.bfloat16)
    qt = torch.from_numpy(queries).cuda().to(torch.bfloat16)
    rg = (torch.arange(n, device="cuda", dtype=torch.int32) // 7).contiguous()
    rn, qr = S.row_rnorm(st), S.row_rnorm(qt)
    wsb = int(lib.isx_knn_workspace_bytes(n, q, d, k))
    ws, os_, or_, og = Guarded(wsb), Guarded(q * k * 4), Guarded(q * k * 4), Guarded(q * k * 4)
    _lib.check(lib.isx_knn_search_grouped(st.data_ptr(), rn.data_ptr(), rg.data_ptr(), n, qt.data_ptr(), qr.data_ptr(), q, d, k,
                                          0, os_.ptr, or_.ptr, og.ptr, ws.ptr, wsb, torch.cuda.current_stream().cuda_stream),
               "search_grouped")
    for b, w in ((ws, "workspace"), (os_, "scores"), (or_, "rows"), (og, "groups")):
        b.check(f"isx_knn_search_grouped {w}")
    s = os_.view.view(torch.float32).reshape(q, k)
    r = or_.view.view(torch.int32).reshape(q, k)
    g = og.view.view(torch.int32).reshape(q, k)
    check(store, queries, k, (np.arange(n) // 7), s, r, g)
    rec = torch.stack([S.pack_group_records(s, r, g)] * 3).contiguous()
    ms, mr, mg = Guarded(q * k * 4), Guarded(q * k * 4), Guarded(q * k * 4)
    _lib.check(lib.isx_topk_merge_grouped(rec.data_ptr(), 3, q, k, ms.ptr, mr.ptr, mg.ptr, torch.cuda.current_stream().cuda_stream),
               "merge_grouped")
    for b, w in ((ms, "scores"), (mr, "rows"), (mg, "groups")):
        b.check(f"isx_topk_merge_grouped {w}")
    assert torch.equal(mr.view.view(torch.int32).reshape(q, k), r)


_WORKER = r"""
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["ISX_REPO"])
sys.path.insert(0, os.path.join(os.environ["ISX_REPO"], "tests"))
import grouped_oracle as G
from imagescry_b200 import search as S
from oracle import oracle as O
rank = int(os.environ["ISX_RANK"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{os.environ['ISX_PORT']}", rank=rank, world_size=2)
rng = np.random.default_rng(0)
n, c, d, k = 20001, 7, 128, 10      # 2857 images; the shard cut (row 10001) falls inside image 1428
groups = np.arange(n) // c
base = rng.standard_normal((groups.max() + 1, d)).astype(np.float32)
store = O.bf16_round(base[groups] + 0.1 * rng.standard_normal((n, d)).astype(np.float32))
queries = O.bf16_round(store[[3, 10000, 10002, 19990]] + 0.05 * rng.standard_normal((4, d)).astype(np.float32))
b, e = S.shard_range(n, 2, rank)
offsets = torch.from_numpy(np.append(np.arange(0, n, c), n))
sh = S.ShardedEmbeddingStore(torch.from_numpy(store[b:e]).cuda(), total_rows=n, groups=offsets)
s, img, cells = sh.search_images(torch.from_numpy(queries).cuda(), k)
ws, wr, wg = G.cosine_knn_groups(store, queries, k, groups)
assert np.array_equal(img.cpu().numpy(), wg) and np.abs(s.cpu().numpy() - ws).max() <= 1e-3, rank
assert np.array_equal(cells.cpu().numpy(), wr - groups[wr] * c)
assert 1428 in img[1].tolist() and len(set(img[1].tolist())) == k
dist.barrier()
dist.destroy_process_group()
print("OK", rank)
"""


def test_two_gpu_sharded_search_images(tmp_path):
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
