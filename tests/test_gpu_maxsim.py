"""GPU checks of multi-vector (maxsim) image search against the CPU reference `maxsim_oracle` and against
`search_images`, whose per-image scores the search's per-cell terms are, bit for bit.

Tolerances: cell maxima within 1e-3 of the fp32 reference; set scores EXACTLY the ordered fp32 sum of
the per-cell terms divided by the set's size; images identical to the fp64 reference except where a
differing image's exact score lies within 1e-3 of the exact k-th (the rule of test_gpu_knn.check)."""

from __future__ import annotations

import numpy as np
import pytest
import torch

import maxsim_oracle as M
from oracle import oracle as O

pytestmark = pytest.mark.gpu

from imagescry_b200 import _lib  # noqa: E402
from imagescry_b200 import geometry as GEO  # noqa: E402
from imagescry_b200 import search as S  # noqa: E402
from imagescry_b200 import store_format as F  # noqa: E402
from test_gpu_grouped_knn import SHAPES, Guarded, grouped_raw, make  # noqa: E402

SCORE_TOL = 1e-3


def stream():
    return torch.cuda.current_stream().cuda_stream


def groups_of(kind, n, seed):
    """(groups argument of EmbeddingStore or None, per-row group ids)"""
    rng = np.random.default_rng(seed)
    if kind == "ids":  # random, non-contiguous ids (C ABI only): most chunks are mixed
        return None, rng.integers(0, max(2, n // 40), n)
    if kind == "offsets":
        off = np.concatenate([[0], np.cumsum(rng.integers(1, 300, n))])
        off = np.append(off[off < n], n)
        return torch.from_numpy(off), np.searchsorted(off, np.arange(n), side="right") - 1
    c = int(kind)
    return c, np.arange(n - n % c) // c


def maxsim_raw(st, rn, rg, qt, group_base, num_groups):
    lib = _lib.load()
    q, d = qt.shape
    cm = torch.empty((q, num_groups), dtype=torch.float32, device="cuda")
    ws = torch.empty(_lib.KNN_RANGE_WORKSPACE_BYTES, dtype=torch.uint8, device="cuda")
    qr = S.row_rnorm(qt)
    _lib.check(lib.isx_knn_maxsim(st.data_ptr(), rn.data_ptr(), rg.data_ptr(), st.shape[0], qt.data_ptr(), qr.data_ptr(), q, d,
                                  group_base, num_groups, cm.data_ptr(), ws.data_ptr(), ws.numel(), stream()), "isx_knn_maxsim")
    return cm, qr


def terms(cm, qr):
    """The per-cell terms fl(max · rnorm_q) the set reduce forms (fp32 products, as on the device)."""
    return (cm.cpu() * qr.cpu()[:, None]).numpy()


def search_images_matrix(scores, images, num_groups):
    """Q × groups matrix of `search_images` scores (k = every group); -inf where a group is absent."""
    s, g = scores.cpu().numpy(), images.cpu().numpy()
    out = np.full((s.shape[0], num_groups), -np.inf, np.float32)
    rows = np.repeat(np.arange(s.shape[0]), s.shape[1]).reshape(s.shape)
    ok = g >= 0
    out[rows[ok], g[ok]] = s[ok]
    return out


@pytest.mark.parametrize("n,q,d,k", SHAPES)
@pytest.mark.parametrize("kind", ["1", "7", "32", "256", "offsets", "ids"])
def test_cell_max_vs_oracle(n, q, d, k, kind):
    _, groups = groups_of(kind, n, seed=n + k)
    n = len(groups)
    store, queries = make(n, q, d, seed=n + q + d)
    st = torch.from_numpy(store).cuda().to(torch.bfloat16)
    qt = torch.from_numpy(queries).cuda().to(torch.bfloat16)
    total = int(groups.max()) + 1
    base = 2 if kind in ("7", "ids") and total > 4 else 0  # rows of groups below `base` write nothing
    ng = total - base
    rg = torch.from_numpy(groups.astype(np.int32)).cuda()
    cm, qr = maxsim_raw(st, S.row_rnorm(st), rg, qt, base, ng)
    got = terms(cm, qr)
    ref = M.cell_image_max(store, queries, groups, ng, group_base=base)
    assert np.array_equal(np.isneginf(got), np.isneginf(ref))
    fin = np.isfinite(ref)
    assert np.abs(got[fin] - ref[fin]).max(initial=0.0) <= SCORE_TOL
    if total <= 128:
        # each term is bit for bit the image-level search's score of that group for that row
        s, _, g = grouped_raw(st, S.row_rnorm(st), rg, qt, total)
        want = search_images_matrix(s, g, total)[:, base:]
        assert np.all((got == want) | (np.isneginf(got) & np.isneginf(want)))


def random_sets(q, seed, empty=True):
    rng = np.random.default_rng(seed)
    cuts = np.sort(rng.integers(0, q + 1, max(1, q // 6)))
    if empty:
        cuts = np.concatenate([cuts, cuts[:2]])  # repeated cuts: empty sets
    return torch.from_numpy(np.concatenate([[0], np.sort(cuts), [q]]))


def check_sets(scores, images, v32, f64, off, k):
    """scores / images of search_images_maxsim against the exact fp32 rule over the per-cell terms v32
    and the fp64 reference f64 (S × images)."""
    want32 = M.set_scores_fp32(v32, off)
    s, i = scores.cpu().numpy(), images.cpu().numpy()
    off = np.asarray(off)
    valid = i >= 0
    assert np.all(np.isneginf(s[~valid]))
    ref_s, ref_i = M.topk_images(f64, k)
    assert np.array_equal(valid, ref_i >= 0)
    for r in range(s.shape[0]):
        si, ii = s[r][valid[r]], i[r][valid[r]]
        assert np.all(si == want32[r, ii]), f"set {r}: a score is not the ordered fp32 sum"
        assert np.array_equal(np.lexsort((ii, -si)), np.arange(len(si))), f"set {r} not ordered"
        assert len(set(ii.tolist())) == len(ii)
        kth = ref_s[r][valid[r]][-1] if valid[r].any() else -np.inf
        for g in set(ii.tolist()) ^ set(ref_i[r][valid[r]].tolist()):
            assert abs(f64[r, g] - kth) < SCORE_TOL, f"set {r}: image {g} differs beyond tolerance"
    if off[-1]:
        assert np.abs(s[valid] - np.take_along_axis(f64, np.clip(i, 0, None), 1)[valid]).max(initial=0.0) <= SCORE_TOL


@pytest.mark.parametrize("n,q,d,kind,k", [(4999, 300, 128, "offsets", 10), (20480, 257, 256, "256", 16),
                                          (7000, 130, 1280, "7", 100), (3000, 40, 72, "32", 128), (9000, 700, 64, "256", 5)])
def test_set_scores_are_exact(n, q, d, kind, k):
    arg, groups = groups_of(kind, n, seed=k)
    n = len(groups)
    store, queries = make(n, q, d, seed=n + d, correlated=True, groups=groups)
    st = S.EmbeddingStore(torch.from_numpy(store).cuda(), groups=arg)
    qt = torch.from_numpy(queries).cuda()
    off = random_sets(q, seed=q)
    scores, images = st.search_images_maxsim(qt, off, k)
    total = int(groups.max()) + 1
    cm, qr = maxsim_raw(st.embeddings, st.rnorm, st.row_group, st._queries(qt), 0, total)
    v32 = terms(cm, qr)
    if total <= 128:
        s, g, _ = st.search_images(qt, total)
        assert np.array_equal(v32, search_images_matrix(s, g, total))
    f64 = M.set_scores_fp64(M.cell_image_max(store, queries, groups, total), off)
    check_sets(scores, images, v32, f64, off, k)


def test_invariants():
    n, q, d, c = 10_000 - 37, 333, 128, 50  # ragged store end (offsets), Q not a multiple of 128
    off_rows = torch.from_numpy(np.append(np.arange(0, n, c), n))
    groups = np.searchsorted(off_rows.numpy(), np.arange(n), side="right") - 1
    store, queries = make(n, q, d, seed=5, correlated=True, groups=groups)
    st = S.EmbeddingStore(torch.from_numpy(store).cuda(), groups=off_rows)
    qt = torch.from_numpy(queries).cuda()
    # sets of one cell: exactly search_images
    s1, i1 = st.search_images_maxsim(qt, 1, 10)
    ws, wi, _ = st.search_images(qt, 10)
    assert torch.all(s1 == ws) and torch.equal(i1, wi)
    # several blocks give the one-block result bit for bit
    sets = random_sets(q, seed=1)
    one = st.search_images_maxsim(qt, sets, 20)
    many = st.search_images_maxsim(qt, sets, 20, budget_bytes=q * 4 * 70)  # 70 images per block: 3 blocks
    assert len(S.maxsim_block_plan(off_rows, q, q * 4 * 70)) >= 3
    assert torch.equal(one[0], many[0]) and torch.equal(one[1], many[1])
    tiny, whole = (st.search_images_maxsim(qt[:50], 10, 20, budget_bytes=b) for b in (1, 1 << 30))  # one image per block
    assert torch.equal(tiny[0], whole[0]) and torch.equal(tiny[1], whole[1])
    # empty sets and k > #images
    sets2 = torch.tensor([0, 0, 5, 5, q])
    s2, i2 = st.search_images_maxsim(qt, sets2, 128)
    images = len(off_rows) - 1
    assert torch.all(i2[[0, 2]] == -1) and torch.all(torch.isneginf(s2[[0, 2]]))
    small = S.EmbeddingStore(torch.from_numpy(store[:3 * c]).cuda(), groups=c)
    s3, i3 = small.search_images_maxsim(qt, sets2, 5)
    assert torch.all(i3[[1, 3], :3] >= 0) and torch.all(i3[:, 3:] == -1) and torch.all(torch.isneginf(s3[:, 3:]))
    assert images > 128 and torch.all(i2[[1, 3]] >= 0)
    # a one-image store
    single = S.EmbeddingStore(torch.from_numpy(store[:c]).cuda(), groups=c)
    s4, i4 = single.search_images_maxsim(qt, sets2, 3)
    assert i4[:, 0].tolist() == [-1, 0, -1, 0] and torch.all(i4[:, 1:] == -1)
    v = terms(*maxsim_raw(single.embeddings, single.rnorm, single.row_group, single._queries(qt), 0, 1))
    assert s4[1, 0].item() == M.set_scores_fp32(v, [0, 5])[0, 0]
    # no queries, no store rows
    e_s, e_i = st.search_images_maxsim(qt[:0], torch.tensor([0, 0]), 4)
    assert e_s.shape == (1, 4) and torch.all(e_i == -1)
    with pytest.raises(ValueError):
        S.EmbeddingStore(torch.randn(10, 64).cuda()).search_images_maxsim(qt[:, :64], 1, 3)
    with pytest.raises(ValueError):
        st.search_images_maxsim(qt, 1, 129)
    with pytest.raises(ValueError):
        st.search_images_maxsim(qt, 2, 3)  # 333 rows are not sets of 2


@pytest.mark.parametrize("n,q,d", [(3000, 70, 64), (9000, 300, 200), (700, 33, 72), (5000, 257, 1280)])
def test_guard_bands(n, q, d):
    lib = _lib.load()
    store, queries = make(n, q, d, seed=n)
    st = torch.from_numpy(store).cuda().to(torch.bfloat16)
    qt = torch.from_numpy(queries).cuda().to(torch.bfloat16)
    groups = (np.arange(n) // 7).astype(np.int32)
    groups[::11] = -3  # ids outside every range
    rg = torch.from_numpy(groups).cuda()
    rn, qr = S.row_rnorm(st), S.row_rnorm(qt)
    base, ng = 5, int(groups.max()) - 20  # ids below 5 and above base + ng - 1 are outside
    cm = Guarded(q * ng * 4)
    ws = Guarded(_lib.KNN_RANGE_WORKSPACE_BYTES)
    _lib.check(lib.isx_knn_maxsim(st.data_ptr(), rn.data_ptr(), rg.data_ptr(), n, qt.data_ptr(), qr.data_ptr(), q, d, base, ng,
                                  cm.ptr, ws.ptr, ws.nbytes, stream()), "maxsim")
    cm.check("isx_knn_maxsim cell_max")
    ws.check("isx_knn_maxsim workspace")
    got = cm.view.view(torch.float32).reshape(q, ng)
    ref = M.cell_image_max(store, queries, groups, ng, group_base=base)
    v = terms(got, qr)
    assert np.array_equal(np.isneginf(v), np.isneginf(ref)) and np.abs(v[np.isfinite(ref)] - ref[np.isfinite(ref)]).max() <= SCORE_TOL
    sets = random_sets(q, seed=d).cuda()
    num_sets, k = len(sets) - 1, 17
    rec = Guarded(num_sets * k * 8)
    _lib.check(lib.isx_maxsim_sets_topk(got.data_ptr(), qr.data_ptr(), q, ng, 3, ng - 2, sets.data_ptr(), num_sets, k, base,
                                        rec.ptr, stream()), "sets_topk")
    rec.check("isx_maxsim_sets_topk records")
    s, i = S.unpack_records(rec.view.view(torch.int64).reshape(num_sets, k))
    i = i.cpu().numpy()
    assert np.all((i == -1) | ((i >= base + 3) & (i < base + ng - 2)))  # the column range only


def test_user_size_sampled_sets():
    """999 936 rows of 256 features, 256 cells per image, 10 000 query rows in sets of 40: 8 sampled
    sets against an fp32 brute force over the whole store."""
    n, d, c, q, m, k = 999_936, 256, 256, 10_000, 40, 10
    g = torch.Generator(device="cuda").manual_seed(77)
    store = torch.empty((n, d), dtype=torch.bfloat16, device="cuda")
    for s0 in range(0, n, 1 << 18):
        e = min(n, s0 + (1 << 18))
        store[s0:e] = torch.randn((e - s0, d), generator=g, device="cuda").to(torch.bfloat16)
    queries = torch.randn((q, d), generator=g, device="cuda").to(torch.bfloat16)
    st = S.EmbeddingStore(store, groups=c)
    scores, images = st.search_images_maxsim(queries, m, k)
    assert scores.shape == (q // m, k) and int(images.min()) >= 0 and int(images.max()) < n // c
    pick = [0, 1, 37, 100, 128, 199, 248, 249]
    rows = torch.cat([torch.arange(p * m, (p + 1) * m) for p in pick]).cuda()
    qn = torch.nn.functional.normalize(queries[rows].float(), dim=1)
    best = torch.empty((len(rows), n // c), device="cuda")
    for s0 in range(0, n, 1 << 17):
        e = min(n, s0 + (1 << 17))
        best[:, s0 // c:e // c] = (qn @ torch.nn.functional.normalize(store[s0:e].float(), dim=1).T).view(len(rows), -1, c).amax(2)
    f64 = best.double().view(len(pick), m, -1).mean(1)
    ex_s, ex_i = f64.topk(k, dim=1)
    got_s, got_i = scores[pick].double(), images[pick]
    assert (got_s - ex_s).abs().max().item() <= SCORE_TOL
    for r in range(len(pick)):
        for j in set(got_i[r].tolist()) ^ set(ex_i[r].tolist()):
            assert abs(f64[r, j].item() - ex_s[r, -1].item()) < SCORE_TOL


def test_roi_cells():
    rng = np.random.default_rng(3)
    maps = torch.from_numpy(rng.standard_normal((6, 64, 8, 10)).astype(np.float32)).cuda()
    mask = torch.zeros((6, 8, 10), dtype=torch.int64, device="cuda")
    mask[0, 2:5, 3:7] = 1
    mask[2, 0, 0] = 1
    mask[3, 6:, 1:9] = 2  # another class: not covered for class 1
    mask[5, 1:7, 2:4] = 1
    cells, sets = GEO.roi_cells(maps, mask)
    rows = F.maps_to_rows(maps)
    want = rows[(mask == 1).reshape(-1)]
    assert cells.dtype == torch.bfloat16 and torch.equal(cells, want)
    assert sets.tolist() == [0, 12, 12, 13, 13, 13, 25]
    # one ROI shared by every image
    c2, s2 = GEO.roi_cells(maps, mask[0])
    assert torch.equal(c2, rows.view(6, 80, 64)[:, (mask[0] == 1).reshape(-1)].reshape(-1, 64)) and s2.tolist() == [0, 12, 24, 36, 48, 60, 72]
    c3, s3 = GEO.roi_cells(maps[1], mask[3], class_index=2)
    assert s3.tolist() == [0, 16] and torch.equal(c3, F.maps_to_rows(maps[1:2])[(mask[3] == 2).reshape(-1)])
    # the store built from the same maps returns each ROI's own image first
    store = F.store_from_maps(maps)
    s, i = store.search_images_maxsim(cells, sets, 3)
    assert i[0, 0].item() == 0 and i[2, 0].item() == 2 and i[5, 0].item() == 5
    assert torch.all(i[[1, 3, 4]] == -1)
    with pytest.raises(ValueError):
        GEO.roi_cells(maps, mask[:, :4])


_WORKER = r"""
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["ISX_REPO"])
from imagescry_b200 import search as S
rank = int(os.environ["ISX_RANK"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{os.environ['ISX_PORT']}", rank=rank, world_size=2)
rng = np.random.default_rng(0)
n, d = 20001, 128
sizes = rng.integers(1, 120, n)
off = np.concatenate([[0], np.cumsum(sizes)])
off = np.append(off[off < n], n)
half = n // 2 + 1  # shard_range(20001, 2): rank 0 holds [0, 10001)
assert not np.isin(half, off), "the shard boundary must cut an image"
groups = np.searchsorted(off, np.arange(n), side="right") - 1
base = rng.standard_normal((len(off) - 1, d)).astype(np.float32)
store = torch.from_numpy(base[groups] + 0.1 * rng.standard_normal((n, d)).astype(np.float32)).to(torch.bfloat16)
cut = int(groups[half])
queries = (store[[3, 10000, 10002, half - 1, half, 19990]].float() + 0.05 * torch.from_numpy(rng.standard_normal((6, d)).astype(np.float32))).repeat(7, 1)
sets = torch.tensor([0, 4, 4, 12, 30, 31, 42])
b, e = S.shard_range(n, 2, rank)
sh = S.ShardedEmbeddingStore(store[b:e].cuda(), total_rows=n, groups=torch.from_numpy(off))
full = S.EmbeddingStore(store.cuda(), groups=torch.from_numpy(off))
for budget in (1 << 30, 42 * 4 * 50):
    s, i = sh.search_images_maxsim(queries.cuda(), sets, 20, budget_bytes=budget)
    ws, wi = full.search_images_maxsim(queries.cuda(), sets, 20, budget_bytes=budget)
    assert torch.equal(s, ws) and torch.equal(i, wi), (rank, budget)
assert cut in i[2].tolist() or cut in i[3].tolist(), (rank, cut)
dist.barrier()
dist.destroy_process_group()
print("OK", rank)
"""


def test_two_gpu_sharded_maxsim(tmp_path):
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
