"""GPU parity: stage 2 (L2-normalise + pool + PCA projection) through the C ABI vs the CPU oracle
and the golden vectors.  Tolerance (BASELINE.json north_star): embeddings within 1e-3 relative —
written here as |out - ref| <= 1e-3 * |ref| + 1e-4 * rms(ref): relative, with an absolute floor of
1e-4 of the output's RMS for near-zero components (there every fp32 evaluation order, the
reference's own included, differs by more than 1e-3 of the value).  What the bf16 hi/lo split
actually delivers, 2^-16 per product, is asserted as well: max error <= 6e-5 * rms(ref)."""

from __future__ import annotations

import numpy as np
import pytest
import torch

from oracle import oracle as O

pytestmark = pytest.mark.gpu

from imagescry_b200.data import EmbeddingBatch, ImageBatch  # noqa: E402
from imagescry_b200.models.decomposition import PCA  # noqa: E402


def fitted_pca(means, comps):
    F, k = comps.shape
    pca = PCA(num_features=F, num_components=k)
    pca.feature_means.data = torch.from_numpy(np.ascontiguousarray(means)).reshape(1, F).float()
    # keep the reference's memory layout: a transposed view of a k×F row-major matrix
    pca.component_vectors = torch.nn.Parameter(torch.from_numpy(np.ascontiguousarray(comps.T)).float().T, requires_grad=False)
    pca._fitted.data = torch.tensor(True)
    pca._num_features.data = torch.tensor(F)
    pca._num_components.data = torch.tensor(k)
    return pca.cuda()


def assert_close(out, ref):
    out = out.detach().cpu().numpy()
    assert out.shape == ref.shape
    scale = np.sqrt((ref.astype(np.float64) ** 2).mean())
    assert np.all(np.abs(out - ref) <= 1e-3 * np.abs(ref) + 1e-4 * scale), np.abs(out - ref).max()
    assert np.abs(out - ref).max() <= 6e-5 * max(scale, 1e-30) + 1e-7  # what bf16x3 actually delivers


def test_golden_projection(golden):
    g = golden("embed_pca")
    for name in ("unc", "cor"):
        pca = fitted_pca(g[f"pca_{name}_means"], g[f"pca_{name}_comps"])
        out = pca.transform(torch.from_numpy(g[f"pca_{name}_x"]).cuda())
        assert_close(out, g[f"pca_{name}_out"])
    pca = fitted_pca(g["eb_means"], g["eb_comps"])
    assert_close(pca.transform(torch.from_numpy(g["eb_flat"]).cuda()), g["eb_proj"])
    out = pca.project_feature_map(torch.from_numpy(g["eb_fmap"]).cuda())
    assert tuple(out.stride()) == tuple(int(v) for v in g["eb_out_strides"])  # NHWC memory, as the reference returns
    assert_close(out, g["eb_out_nchw"])
    pca = fitted_pca(g["pipe_means"], g["pipe_comps"])
    assert_close(pca.project_feature_map(torch.from_numpy(g["pipe_fmap"]).cuda()), g["pipe_out"])


@pytest.mark.parametrize(
    "B,E,h,w,k",
    [
        (3, 128, 7, 10, 24),     # ragged cells (70 per image), k padded to 32
        (4, 1280, 8, 8, 256),    # 256² tiles
        (2, 1280, 16, 16, 256),  # 512² tiles
        (5, 200, 3, 5, 7),       # E not a multiple of 64, tiny k
        (1, 64, 1, 1, 16),
        (9, 1280, 4, 4, 100),
    ],
)
@pytest.mark.parametrize("pool", [None, "mean"])
def test_project_vs_oracle(B, E, h, w, k, pool):
    rng = np.random.default_rng(B * E + k)
    fmap = np.abs(rng.standard_normal((B, E, h, w))).astype(np.float32) * 2 + 0.05
    fmap[0, :, 0, 0] = 0.0  # an all-zero cell: x / max(||x||, 1e-12) = 0
    means = (rng.standard_normal(E) * 0.02).astype(np.float32)
    comps = np.linalg.qr(rng.standard_normal((E, k)))[0].astype(np.float32)
    pca = fitted_pca(means, comps)
    out = pca.project_feature_map(torch.from_numpy(fmap).cuda(), pool=pool)
    ref = O.pipeline_project(fmap, means, comps, pool=pool)
    assert_close(out, ref)


def test_transform_matches_reference_semantics():
    rng = np.random.default_rng(0)
    x = rng.standard_normal((1000, 96)).astype(np.float32)
    pca = PCA(min_num_components=5, max_num_components=5).fit(torch.from_numpy(x).cuda())
    out = pca.transform(torch.from_numpy(x).cuda())
    ref = O.pca_transform(x, pca.feature_means.cpu().numpy(), pca.component_vectors.cpu().numpy())
    assert_close(out, ref)
    c = np.corrcoef(out.cpu().numpy().T)
    assert np.abs(c - np.eye(5)).max() <= 1e-3  # decorrelated, as test_decomposition.py:84-124 checks
    with pytest.raises(RuntimeError):
        PCA().cuda().transform(torch.zeros(4, 3).cuda())
    assert pca.transform(torch.zeros((0, 96)).cuda()).shape == (0, 5)


def test_pipeline_predict_step_end_to_end(golden):
    """ImageBatch → preprocess (CUDA) → tiny conv backbone (torch, not owned) → fused L2+projection,
    against the reference pipeline's frozen output."""
    from imagescry_b200.image.transforms import normalize_per_channel
    from imagescry_b200.models.embedding import EmbeddingModule
    from imagescry_b200.models.pipelines import EmbeddingPCAPipeline

    g = golden("embed_pca")

    class Tiny(EmbeddingModule):
        def __init__(self):
            super().__init__()
            self.net = torch.nn.Sequential(torch.nn.Conv2d(3, 64, 8, stride=8), torch.nn.SiLU())

        def preprocess(self, images):
            return normalize_per_channel(images, min_value=-3, max_value=3)

        def forward(self, x):
            return self.net(x)

        @property
        def embedding_dim(self):
            return 64

    model = Tiny()
    model.net[0].weight.data = torch.from_numpy(g["pipe_conv_w"])
    model.net[0].bias.data = torch.from_numpy(g["pipe_conv_b"])
    model = model.cuda().eval()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    pca = fitted_pca(g["pipe_means"], g["pipe_comps"])
    pipe = EmbeddingPCAPipeline(embedding_model=model, pca=pca)
    batch = ImageBatch(indices=torch.arange(4).cuda(), images=torch.from_numpy(g["pipe_images"]).cuda())
    with torch.inference_mode():
        res = pipe.predict_step(batch)
        assert np.abs(model.preprocess(batch.images).cpu().numpy() - g["pipe_pre"]).max() <= 1e-6
    assert isinstance(res, EmbeddingBatch) and res.embeddings.shape == g["pipe_out"].shape
    ref = g["pipe_out"]
    out = res.embeddings.cpu().numpy()
    scale = np.sqrt((ref.astype(np.float64) ** 2).mean())
    # the backbone is cuDNN on the GPU vs MKL on the CPU: allow its fp32 reordering on top
    assert np.all(np.abs(out - ref) <= 1e-3 * np.abs(ref) + 1e-3 * scale)


def test_full_size_feature_map_properties():
    """BASELINE.json config 3b at full size (4096 x 1280 x 16 x 16 fp32 -> 256-d): one image from every
    round of pair tiles (an image is one 256-cell pair tile; pair p runs tiles p, p + P, ...) against
    an fp64 torch evaluation of the reference's formula (embedding.py:74, data.py:118,
    decomposition.py:91), layout of pipelines.py:82-84, pooled == mean of normalised cells, and two
    calls give bit-identical outputs."""
    import torch

    from imagescry_b200.models.decomposition import PCA

    B, E, h, w, k = 4096, 1280, 16, 16, 256
    g = torch.Generator(device="cuda").manual_seed(7)
    fmap = torch.empty((B, E, h, w), dtype=torch.float32, device="cuda")
    for s in range(0, B, 256):
        fmap[s:s + 256] = torch.randn((256, E, h, w), generator=g, device="cuda").abs_()
    comps = torch.linalg.qr(torch.randn((E, k), generator=g, device="cuda"))[0]
    pca = PCA(num_features=E, num_components=k).cuda()
    pca.feature_means.data = torch.randn((1, E), generator=g, device="cuda") * 0.01
    pca.component_vectors.data = comps.contiguous()
    pca._fitted.data = torch.tensor(True, device="cuda")
    pca._num_features.data = torch.tensor(E, device="cuda")
    pca._num_components.data = torch.tensor(k, device="cuda")
    out = pca.project_feature_map(fmap)
    assert out.shape == (B, k, h, w) and out.stride() == (h * w * k, 1, w * k, k)  # NHWC memory
    assert torch.equal(pca.project_feature_map(fmap), out)
    pooled = pca.project_feature_map(fmap, pool="mean")
    assert pooled.shape == (B, k)
    P = min(torch.cuda.get_device_properties(0).multi_processor_count // 2, B)  # CTA pairs launched
    rounds = -(-B // P)
    images = [min(r * P + (r * 29) % P, B - 1) for r in range(rounds)]  # a different pair in every round
    assert len(images) >= 3 and images[-1] >= B - P
    for b in images:
        x = fmap[b].double()
        e = x / x.norm(dim=0, keepdim=True).clamp_min(1e-12)
        flat = e.permute(1, 2, 0).reshape(-1, E)
        ref = (flat - pca.feature_means.double()) @ pca.component_vectors.double()
        got = out[b].permute(1, 2, 0).reshape(-1, k).double()
        scale = ref.norm(dim=1, keepdim=True)
        assert float(((got - ref).abs() / scale).max()) < 1e-4  # bar: 1e-3 relative
        refp = (e.mean(dim=(1, 2)).unsqueeze(0) - pca.feature_means.double()) @ pca.component_vectors.double()
        assert float((pooled[b].double() - refp[0]).abs().max() / refp.norm()) < 1e-4


def test_pca_fit_gpu_moments_and_components(golden):
    """PCA.fit on the GPU (isx_pca_moments + eigen-decomposition) vs the oracle's restatement of
    decomposition.py:94-148: reference fixtures, then a larger correlated matrix.  Directions are
    compared up to sign (the reference's SVD signs are arbitrary too); the projections then agree up
    to those signs."""
    import torch

    from imagescry_b200.models.decomposition import PCA

    g = golden("embed_pca")
    for name in ("unc", "cor"):
        x = g[f"pca_{name}_x"]
        k_ref = int(g[f"pca_{name}_k"])
        cum = np.cumsum(g[f"pca_{name}_explained"])
        thr = float((cum[k_ref - 2] + cum[k_ref - 1]) / 2) if k_ref > 1 else float(cum[0] / 2)
        pca = PCA(min_explained_variance=thr).cuda().fit(torch.from_numpy(x).cuda())
        assert pca.num_components == k_ref
        assert np.allclose(pca.feature_means.cpu().numpy(), g[f"pca_{name}_means"], atol=1e-6)
        assert np.allclose(pca.explained_variance.cpu().numpy(), g[f"pca_{name}_explained"], atol=1e-5)
        dots = np.abs(np.sum(pca.component_vectors.cpu().numpy() * g[f"pca_{name}_comps"], axis=0))
        assert np.all(dots > 1 - 1e-4)
        out = pca.transform(torch.from_numpy(x).cuda()).cpu().numpy()
        assert np.allclose(np.abs(out), np.abs(g[f"pca_{name}_out"]), atol=2e-4)

    rng = np.random.default_rng(42)
    n, F, r = 20000, 200, 12
    basis = rng.standard_normal((r, F)).astype(np.float32)
    x = (rng.standard_normal((n, r)).astype(np.float32) * np.linspace(10, 1, r, dtype=np.float32)) @ basis
    x += 0.05 * rng.standard_normal((n, F)).astype(np.float32) + 3.0
    means, comps, explained, k = O.pca_fit(x, min_explained_variance=0.99, max_num_components=64)
    pca = PCA(min_explained_variance=0.99, max_num_components=64).cuda().fit(torch.from_numpy(x).cuda())
    assert pca.num_components == k
    assert np.allclose(pca.feature_means.cpu().numpy(), means, atol=1e-5)
    assert np.allclose(pca.explained_variance.cpu().numpy(), explained, atol=1e-5)
    got = pca.component_vectors.cpu().numpy()
    assert np.all(np.abs(np.sum(got[:, :r] * comps[:, :r], axis=0)) > 1 - 1e-3)
    # the moments themselves against fp64 numpy
    mean_d, cov_d = pca._moments(torch.from_numpy(x).cuda())
    ref_cov = np.cov(x.astype(np.float64), rowvar=False)
    assert np.abs(cov_d.cpu().numpy() - ref_cov).max() <= 1e-5 * np.abs(ref_cov).max()
    assert np.array_equal(cov_d.cpu().numpy(), cov_d.cpu().numpy().T)
    with pytest.raises(ValueError):
        PCA().cuda().fit(torch.zeros((1, 4)).cuda())
    # fitted and used under inference mode (what Lightning's predict loop runs in): the fitted tensors
    # are inference tensors without a version counter
    with torch.inference_mode():
        p2 = PCA(min_num_components=8, max_num_components=8).cuda().fit(torch.from_numpy(x).cuda())
        out = p2.transform(torch.from_numpy(x[:64]).cuda())
    assert out.shape == (64, 8) and torch.isfinite(out).all()


@pytest.mark.parametrize(
    "E,h,w,k,aligned",
    [
        (320, 16, 16, 96, True),   # rule 2: staged kernel; hw = 256, a 128-cell tile is half an image
        (320, 8, 8, 96, True),     # rule 2: staged kernel; hw = 64, a tile spans two images
        (320, 16, 16, 96, False),  # rule 3: K3d
        (320, 8, 8, 96, False),    # rule 3: K3d
        (320, 16, 16, 95, False),  # rule 4: register path through k % 4 != 0
        (320, 8, 8, 95, False),    # rule 4: register path through k % 4 != 0
        (320, 7, 10, 96, True),    # rule 3: K3d; 70 cells per image fit no TMA box
        (320, 7, 10, 95, True),    # rule 4: register path through k % 4 != 0
        (200, 7, 10, 100, True),   # rule 4: register path through E % 16 != 0; float4 stores, scalar tail
        (200, 16, 16, 96, False),  # rule 4: register path through E % 16 != 0; float4 stores only
    ],
)
def test_per_cell_kernel_variants_agree(E, h, w, k, aligned):
    """Every per-cell kernel meets the oracle.  The launch picks the kernel from the input alone, by
    the first rule that fits (launch_project in project.cu):
      rule 2, l2norm_project_kernel<true> (staged): 16-byte aligned map, 4 | hw, hw = 128 n or 128 = hw n;
      rule 3, l2norm_project_direct_kernel (K3d): otherwise, if k % 4 == 0 and E % 16 == 0;
      rule 4, l2norm_project_kernel<false> (register path): otherwise.  With k % 4 == 0 its epilogue
      writes float4 pieces, else single floats.
    An unaligned map is a view 4 bytes into its allocation, so 16 x 16 and 8 x 8 maps reach all three.
    B = 9 leaves the last CTA pair ragged."""
    import torch

    from imagescry_b200.models.decomposition import PCA

    rng = np.random.default_rng(3)
    B = 9
    fmap = np.abs(rng.standard_normal((B, E, h, w))).astype(np.float32)
    comps = np.linalg.qr(rng.standard_normal((E, k)))[0].astype(np.float32)
    means = (rng.standard_normal(E) * 0.01).astype(np.float32)
    pca = PCA(num_features=E, num_components=k)
    pca.feature_means.data = torch.from_numpy(means).reshape(1, -1)
    pca.component_vectors.data = torch.from_numpy(comps)
    pca._fitted.data = torch.tensor(True)
    pca._num_features.data = torch.tensor(E)
    pca._num_components.data = torch.tensor(k)
    pca = pca.cuda()
    off = 0 if aligned else 1  # one float into the allocation: 4 bytes off a 16-byte boundary
    x = torch.empty(fmap.size + off, device="cuda")[off:].view(fmap.shape)
    x.copy_(torch.from_numpy(fmap))
    assert (x.data_ptr() % 16 == 0) == aligned
    out = pca.project_feature_map(x).cpu().numpy()
    ref = O.pipeline_project(fmap, means, comps)
    scale = np.linalg.norm(ref, axis=1, keepdims=True)
    assert (np.abs(out - ref) / scale).max() < 2e-5


@pytest.mark.parametrize("pool", [None, "mean"])
def test_fp16_single_pass_mode_within_tolerance(pool):
    """precision="fp16": one fp16 tensor pass instead of the three-pass bf16 split.  Bar: 1e-3
    relative (BASELINE.json north_star); measured against the oracle relative to each row's norm and
    elementwise on the elements that carry the row."""
    import torch

    from imagescry_b200.models.decomposition import PCA

    rng = np.random.default_rng(8)
    B, E, h, w, k = 6, 1280, 16, 16, 256
    fmap = (np.abs(rng.standard_normal((B, E, h, w))) * 3.0).astype(np.float32)
    fmap[0, 5, 0, 0] = 7.0e4  # beyond fp16's range: saturates instead of turning into inf
    comps = np.linalg.qr(rng.standard_normal((E, k)))[0].astype(np.float32)
    means = (rng.standard_normal(E) * 0.01).astype(np.float32)
    pca = PCA(num_features=E, num_components=k)
    pca.feature_means.data = torch.from_numpy(means).reshape(1, -1)
    pca.component_vectors.data = torch.from_numpy(comps)
    pca._fitted.data = torch.tensor(True)
    pca._num_features.data = torch.tensor(E)
    pca._num_components.data = torch.tensor(k)
    pca = pca.cuda()
    fm = torch.from_numpy(fmap).cuda()
    out = pca.project_feature_map(fm, pool=pool, precision="fp16").cpu().numpy()
    exact = pca.project_feature_map(fm, pool=pool).cpu().numpy()
    ref = O.pipeline_project(fmap, means, comps, pool=pool)
    assert np.isfinite(out).all()
    axis = 1
    norm = np.linalg.norm(ref, axis=axis, keepdims=True)
    err = np.abs(out - ref) / norm
    if pool is None:
        err[0, :, 0, 0] = 0  # the saturated cell is outside the mode's contract
    assert err.max() < 1e-4, err.max()  # 10x inside the bar, relative to the row
    big = np.abs(ref) > norm / np.sqrt(k)  # elements at least as large as the row's rms element
    if pool is None:
        big[0, :, 0, 0] = False
    # elementwise, on elements that carry the row's energy: the tail of the rounding noise reaches the
    # 1e-3 bar (max ~1.1e-3 over 1e5 elements) — which is why "exact" stays the default mode
    rel = np.abs(out - ref)[big] / np.abs(ref)[big]
    assert np.quantile(rel, 0.999) < 1e-3 and rel.max() < 3e-3
    assert (np.abs(exact - ref) / norm).max() < 2e-5
