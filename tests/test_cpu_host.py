"""CPU-side checks: the C-ABI library loads and exports every declared symbol, host logic of the
mirror modules, and the multi-process plumbing of the sharded search (gloo, world size 2).
No compute entry point is called here — there is no GPU in this environment."""

from __future__ import annotations

import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import REPO
from oracle import oracle as O


def test_library_exports_every_declared_symbol():
    from imagescry_b200 import _lib

    header = open(os.path.join(REPO, "include", "imagescry_b200.h")).read()
    declared = set(re.findall(r"\b(isx_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations found"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.isx_abi_version() == 1
    assert lib.isx_last_error() is not None
    # size queries are pure host arithmetic
    assert lib.isx_preprocess_stats_workspace_bytes(3) > 0
    assert lib.isx_project_packed_bytes(1280, 256) >= 2 * 256 * 1280 * 2 + 256 * 4
    assert lib.isx_project_packed_bytes(1280, 300) == 0  # more than 256 components: unsupported
    nm = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    for name in declared:
        assert re.search(rf"\bT {name}\b", nm), f"{name} is not an exported text symbol"


def test_no_cpu_fallback():
    from imagescry_b200 import search
    from imagescry_b200.image import transforms as T
    from imagescry_b200.models.decomposition import PCA

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        T.normalize_per_channel(torch.zeros(1, 3, 4, 4, dtype=torch.uint8))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        T.resize(torch.zeros(3, 8, 8, dtype=torch.uint8), 4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        search.EmbeddingStore(torch.zeros(4, 8))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        PCA().fit(torch.randn(50, 6))  # the moments come from the sm_100a kernels: CUDA tensors only
    from imagescry_b200.models.embedding import l2_normalize_cells
    from imagescry_b200.image.transforms import preprocess_patches

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        l2_normalize_cells(torch.zeros(1, 8, 2, 2))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        preprocess_patches(torch.zeros(1, 8, 8, 3, dtype=torch.uint8), 4)


def test_product_never_imports_oracle():
    pkg = os.path.join(REPO, "imagescry_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(root, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f
                assert "sift_oracle" not in src, f


def test_host_shape_logic_matches_oracle_and_reference_rules():
    from imagescry_b200.image.transforms import _calc_scale_factor, resized_shape, to_4d

    for h, w in [(30, 45), (45, 30), (512, 512), (61, 37)]:
        for size in (16, 31, 46, 256):
            for side_ref in ("height", "width", "long", "short"):
                assert resized_shape(h, w, size, side_ref) == O.resized_shape(h, w, size, side_ref)
                assert _calc_scale_factor(h, w, size, side_ref) == O.calc_scale_factor(h, w, size, side_ref)
    assert resized_shape(30, 45, (5, 7)) == (5, 7)
    assert resized_shape(512, 512, 256) == (256, 256)
    assert to_4d(torch.zeros(3, 4)).shape == (1, 1, 3, 4)
    assert to_4d(torch.zeros(3, 5, 7)).shape == (1, 3, 5, 7)
    assert to_4d(torch.zeros(16, 3, 5, 7)).shape == (16, 3, 5, 7)


def test_batch_dataclasses_and_typechecking():
    from jaxtyping import TypeCheckError

    from imagescry_b200.data import EmbeddingBatch, ImageBatch

    ib = ImageBatch(indices=torch.arange(2), images=torch.zeros(2, 3, 4, 5, dtype=torch.uint8))
    assert len(ib) == 2 and ib.device.type == "cpu" and ib.cpu().images.shape == (2, 3, 4, 5)
    eb = EmbeddingBatch(indices=torch.arange(3), embeddings=torch.randn(3, 128, 7, 10))
    assert eb.embedding_dim == 128 and eb.spatial_dims == (7, 10)
    flat = eb.get_flat_vectors()  # test_embedding.py:56-75
    assert flat.shape == (3 * 7 * 10, 128)
    assert torch.equal(flat, eb.embeddings.permute(0, 2, 3, 1).reshape(-1, 128))
    with pytest.raises(TypeCheckError):
        ImageBatch(indices=torch.arange(2), images=torch.zeros(2, 3, 4, 5))  # float images
    with pytest.raises(TypeCheckError):
        ImageBatch(indices=torch.arange(2), images=torch.zeros(2, 1, 4, 5, dtype=torch.uint8))  # 1 channel
    with pytest.raises((AttributeError, Exception)):
        ib.indices = torch.arange(3)  # frozen


def test_pca_component_selection_rule():
    """The selection rule of decomposition.py:128-137 on the explained-variance ratios of the
    reference's own fixtures (test_decomposition.py:42-81,84-124): expected component counts."""
    from imagescry_b200.models.decomposition import PCA, select_num_components

    g = np.load(os.path.join(REPO, "tests", "golden", "embed_pca.npz"))
    unc = torch.from_numpy(g["pca_unc_explained"])
    for mev, want in [(0.2, 1), (0.4, 2), (0.6, 3), (1.0, 4)]:
        assert select_num_components(unc, 1, None, mev) == want
    cor = torch.from_numpy(g["pca_cor_explained"])
    for mev, want in [(0.2, 1), (0.4, 2), (0.6, 2), (0.8, 3), (1.0, 4)]:
        k = select_num_components(cor, 1, None, mev)
        assert k == want and cor[:k].sum() >= mev - 1e-6
    assert select_num_components(cor, 3, None, 0.1) == 3   # min_num_components
    assert select_num_components(cor, 1, 2, 1.0) == 2      # max_num_components
    with pytest.raises(ValueError):
        PCA(min_num_components=0)
    with pytest.raises(ValueError):
        PCA(min_num_components=3, max_num_components=2)
    with pytest.raises(ValueError):
        PCA(min_explained_variance=1.5)
    with pytest.raises(RuntimeError, match="not fitted"):
        PCA().transform(torch.zeros(2, 3))
    assert {"feature_means", "component_vectors", "_fitted"} <= set(PCA().state_dict())
    # re-assigned weights drop the packed operand
    p = PCA(num_features=4, num_components=2)
    p.__dict__["_packed"] = torch.zeros(1)
    p.component_vectors = torch.nn.Parameter(torch.zeros(4, 2), requires_grad=False)
    assert p._packed is None
    p.__dict__["_packed"] = torch.zeros(1)
    p.load_state_dict(PCA(num_features=4, num_components=2).state_dict())
    assert p._packed is None


def test_patch_grid_and_graph_chunk_plan():
    from imagescry_b200.image.transforms import patch_grid
    from imagescry_b200.search import graph_chunk_plan, pack_records, unpack_records

    assert patch_grid(2048, 2048, 512) == (4, 4)
    assert patch_grid(100, 130, 32, 16) == (5, 7)
    assert patch_grid(32, 32, 32, 7) == (1, 1)
    with pytest.raises(ValueError):
        patch_grid(31, 64, 32)
    for img_h, img_w, p_, s_ in [(100, 130, 32, 16), (64, 64, 64, 64), (50, 77, 20, 9)]:
        x = np.zeros((1, img_h, img_w, 3), dtype=np.uint8)
        ny, nx = patch_grid(img_h, img_w, p_, s_)
        assert O.extract_patches(x, p_, s_).shape == (ny * nx, p_, p_, 3)
    assert graph_chunk_plan([125000] * 8, 256, 2 << 30) == (125000, 1)
    chunk, steps = graph_chunk_plan([2502, 2501], 64, 64 * 700 * 2 * 2)
    assert chunk == 700 and steps == 4
    s = torch.tensor([[1.5, float("-inf")]])
    i = torch.tensor([[7, -1]], dtype=torch.int32)
    us, ui = unpack_records(pack_records(s, i))
    assert torch.equal(us, s) and torch.equal(ui, i)


def test_similar_shape_batches_matches_reference_sampler_rule():
    """`SimilarShapeBatcher` (data.py:403-452) on the reference test's own shape list
    (tests/test_data.py:24-39): batches never exceed `max_batch_size`, hold one shape each, cover every
    index once, and equal sort -> group -> chunk computed independently."""
    import itertools

    from imagescry_b200.ingest import HwcTileIngest, similar_shape_batches

    shapes = [(7, 7), (7, 8), (8, 8), (8, 8), (7, 7), (5, 7), (8, 8), (8, 7), (8, 7), (7, 7), (7, 7), (2, 2), (3, 2), (2, 2)]
    for mbs in (1, 2, 3, 4, 100):
        got = similar_shape_batches(shapes, mbs)
        assert all(1 <= len(b) <= mbs for b in got)
        assert all(len({shapes[i] for i in b}) == 1 for b in got)
        assert sorted(i for b in got for i in b) == list(range(len(shapes)))
        want = []
        ordered = sorted(enumerate(shapes), key=lambda t: t[1])
        for _, grp in itertools.groupby(ordered, key=lambda t: t[1]):
            idx = [i for i, _ in grp]
            want += [idx[j:j + mbs] for j in range(0, len(idx), mbs)]
        assert got == want
    assert similar_shape_batches([], 4) == []
    with pytest.raises(ValueError):
        similar_shape_batches(shapes, 0)
    with pytest.raises(RuntimeError, match="no CPU path"):
        HwcTileIngest("cpu", 4)


def test_shard_range_partition():
    from imagescry_b200.search import shard_range

    for n in (0, 1, 7, 100, 100_000_000):
        for world in (1, 2, 3, 8):
            spans = [shard_range(n, world, r) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [e - b for b, e in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_range(10, 2, 2)


_WORKER = r"""
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["ISX_REPO"])
from imagescry_b200.search import gather_partials, gather_records, pack_records, unpack_records, shard_range
from oracle import oracle as O
dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{os.environ['ISX_PORT']}",
                        rank=int(os.environ["ISX_RANK"]), world_size=2)
rank = dist.get_rank()
rng = np.random.default_rng(0)
store = O.bf16_round(rng.standard_normal((1001, 32)).astype(np.float32))
queries = O.bf16_round(rng.standard_normal((9, 32)).astype(np.float32))
b, e = shard_range(len(store), 2, rank)
# the local search is the CUDA kernel's job on a GPU box; here the oracle stands in for it so that
# the partition + gather + merge plumbing can be checked on CPU
ls, li = O.cosine_knn(store[b:e], queries, 5, index_base=b)
all_s, all_i = gather_partials(torch.from_numpy(ls), torch.from_numpy(li.astype(np.int32)))
assert all_s.shape == (2, 9, 5) and all_i.shape == (2, 9, 5)
ms, mi = O.topk_merge(all_s.numpy(), all_i.numpy(), 5)
gs, gi = O.cosine_knn(store, queries, 5)
assert np.array_equal(mi, gi) and np.array_equal(ms, gs), rank
# the packed form: ONE all-gather of 8-byte (score, index) records
rec = gather_records(pack_records(torch.from_numpy(ls), torch.from_numpy(li.astype(np.int32))))
assert rec.shape == (2, 9, 5) and rec.dtype == torch.int64
us, ui = unpack_records(rec)
assert torch.equal(us, all_s) and torch.equal(ui, all_i)
dist.barrier()
dist.destroy_process_group()
print("OK", rank)
"""


def test_sharded_gather_plumbing_gloo_world2(tmp_path):
    import socket

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    procs = []
    for r in range(2):
        env = dict(os.environ, ISX_REPO=REPO, ISX_PORT=str(port), ISX_RANK=str(r), OMP_NUM_THREADS="1")
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=180)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"OK {r}" in o, o


def test_bench_dump_outputs_and_argument_checks(tmp_path):
    """bench.py --dump-outputs: scores as float32 and indices as float64, every index exact (2^24 + 1
    is not representable in float32); --steps below 1 and a dump of the calibrated reference arm are
    rejected before any device work."""
    from bench import dump_outputs

    s = torch.tensor([[0.75, -0.125], [float("-inf"), 1.0]])
    i = torch.tensor([[(1 << 24) + 1, 3], [-1, 999_999]], dtype=torch.int32)
    dump_outputs(str(tmp_path / "out"), s, i)
    got_s, got_i = np.load(tmp_path / "out" / "scores.npy"), np.load(tmp_path / "out" / "indices.npy")
    assert got_s.dtype == np.float32 and np.array_equal(got_s, s.numpy())
    assert got_i.dtype == np.float64 and np.array_equal(got_i, i.numpy().astype(np.int64))
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "ref")]):
        r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), *argv], capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and "error:" in r.stderr, (argv, r.stderr)
    assert not (tmp_path / "ref").exists()


def test_store_format_codec_matches_reference_wire_format():
    """storage/models.py:94-129: float32 C-order bytes; decode(encode(x)) == x and the byte string
    equals numpy's tobytes() of the C×H×W array (what `Embedding.create` writes)."""
    import numpy as np
    import torch

    from imagescry_b200 import store_format as F
    from oracle import oracle as O

    x = torch.arange(2 * 3 * 4, dtype=torch.float32).reshape(2, 3, 4) * 0.5
    data, c, h, w = F.encode_embedding_blob(x)
    assert (c, h, w) == (2, 3, 4) and data == x.numpy().tobytes() == O.blob_encode(x.numpy())
    assert torch.equal(F.decode_embedding_blob(data, c, h, w), x)
    stacked = F.stack_blobs([(data, c, h, w)] * 3)
    assert stacked.shape == (3, 2, 3, 4)
    import pytest

    with pytest.raises(ValueError):
        F.stack_blobs([])
    with pytest.raises(RuntimeError):
        F.maps_to_rows(stacked)  # CPU tensor: the conversion runs on the GPU only
    img, cell = F.rows_to_image_cell([0, 11, 12, 25], 12)
    assert img.tolist() == [0, 0, 1, 2] and cell.tolist() == [0, 11, 0, 1]


def test_polygon_edges_host_logic():
    """geometry.polygon_edges: the edge list handed to isx_roi_rasterize, for every accepted polygon
    form (vertex list, closed ring, dict with holes, shapely-like object, list of polygons)."""
    from imagescry_b200 import geometry as G

    sq = [(0, 0), (4, 0), (4, 3), (0, 3)]
    e, off = G.polygon_edges(sq)
    assert e.dtype == np.float32 and e.shape == (4, 4) and off.tolist() == [0, 4]
    assert e[0].tolist() == [0, 0, 4, 0] and e[3].tolist() == [0, 3, 0, 0]  # the ring is closed
    e2, off2 = G.polygon_edges(sq + [sq[0]])  # shapely repeats the first vertex
    assert np.array_equal(e, e2) and off2.tolist() == [0, 4]
    hole = [(1, 1), (2, 1), (2, 2)]
    e3, off3 = G.polygon_edges({"exterior": sq, "interiors": [hole]})
    assert e3.shape == (7, 4) and off3.tolist() == [0, 7]

    class Ring:
        def __init__(self, pts):
            self.coords = pts

    class Poly:  # duck-typed shapely.geometry.Polygon
        def __init__(self, ext, holes=()):
            self.exterior, self.interiors = Ring(ext), [Ring(h) for h in holes]

    e4, off4 = G.polygon_edges([Poly(sq, [hole]), Poly(hole)])
    assert off4.tolist() == [0, 7, 10] and np.array_equal(e4[:7], e3)
    e5, off5 = G.polygon_edges([sq, hole])  # list of plain vertex lists = two polygons
    assert off5.tolist() == [0, 4, 7]
    with pytest.raises(ValueError):
        G.polygon_edges([(0, 0), (1, 1)])
    with pytest.raises(RuntimeError):  # no CPU rasteriser: the product path needs the GPU
        G.create_roi_mask(sq, (6, 8), (3, 4), device="cpu")
    with pytest.raises(ValueError):
        G.create_roi_mask(sq, (6, 8), (0, 4), device="cpu")


def test_binding_matches_header_prototypes():
    """Every ctypes signature in imagescry_b200/_lib.py has the argument count, and pointer / integer /
    float kinds, of its prototype in include/imagescry_b200.h (a mismatch would corrupt a call silently)."""
    import ctypes

    from imagescry_b200 import _lib

    header = open(os.path.join(REPO, "include", "imagescry_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", " ", header, flags=re.S)
    protos = dict(re.findall(r"\b(isx_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", header, flags=re.S))
    assert set(protos) == set(_lib.SIGNATURES)

    def kind(decl: str) -> str:
        decl = decl.strip()
        if "*" in decl or decl.startswith("isx_stream_t"):
            return "ptr"
        if decl.startswith(("float", "double")):
            return "float"
        return "int"

    ckind = {ctypes.c_void_p: "ptr", ctypes.c_char_p: "ptr", ctypes.c_float: "float", ctypes.c_double: "float"}
    for name, args in protos.items():
        params = [] if args.strip() in ("", "void") else [a for a in args.split(",")]
        _, argtypes = _lib.SIGNATURES[name]
        assert len(params) == len(argtypes), f"{name}: header has {len(params)} parameters, binding {len(argtypes)}"
        for i, (decl, ct) in enumerate(zip(params, argtypes)):
            want = kind(decl)
            got = "ptr" if hasattr(ct, "contents") else ckind.get(ct, "int")
            assert want == got, f"{name} argument {i} ({decl.strip()}): header {want}, binding {got}"
