"""Out-of-bounds write detection without compute-sanitizer (closed on this GPU pool): every output
the C ABI writes is placed between two 64 KiB guard bands filled with a pattern; after the call the
bands must be untouched.  Shapes are ragged on purpose (partial tiles, odd widths, clipped TMA boxes).
Calls go straight through ctypes, like a foreign binding would."""

from __future__ import annotations

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from imagescry_b200 import _lib  # noqa: E402

GUARD = 1 << 16
PATTERN = 0xA5


class Guarded:
    """A device buffer of `nbytes` (256-byte aligned start) with a guard band on either side."""

    def __init__(self, nbytes: int) -> None:
        self.nbytes = nbytes
        pad = (256 - nbytes % 256) % 256
        self.raw = torch.full((GUARD + nbytes + pad + GUARD,), PATTERN, dtype=torch.uint8, device="cuda")
        self.view = self.raw[GUARD:GUARD + nbytes]

    @property
    def ptr(self) -> int:
        return self.view.data_ptr()

    def check(self, what: str) -> None:
        torch.cuda.synchronize()
        lo = self.raw[:GUARD]
        hi = self.raw[GUARD + self.nbytes:]
        assert bool((lo == PATTERN).all()), f"{what}: wrote BEFORE the output buffer"
        assert bool((hi == PATTERN).all()), f"{what}: wrote PAST the output buffer (first bad byte +{int((hi != PATTERN).nonzero()[0])})"

    def as_tensor(self, dtype, shape):
        return self.view.view(dtype).reshape(shape)


def stream():
    return torch.cuda.current_stream().cuda_stream


@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("shape,out_hw", [((3, 61, 37), None), ((5, 64, 96), (32, 48)), ((2, 50, 70), (33, 41)), ((4, 32, 32), None)])
@pytest.mark.parametrize("out_dtype", [_lib.DTYPE_F32, _lib.DTYPE_BF16])
def test_preprocess_apply_stays_in_bounds(layout, shape, out_hw, out_dtype):
    lib = _lib.load()
    B, H, W = shape
    g = torch.Generator(device="cuda").manual_seed(B * H + W)
    x = torch.randint(0, 256, (B, 3, H, W) if layout == "nchw" else (B, H, W, 3), dtype=torch.uint8, device="cuda", generator=g)
    oh, ow = out_hw or (H, W)
    lay = _lib.LAYOUT_NCHW if layout == "nchw" else _lib.LAYOUT_NHWC
    mean = Guarded(12)
    std = Guarded(12)
    ws = torch.empty(lib.isx_preprocess_stats_workspace_bytes(3), dtype=torch.uint8, device="cuda")
    _lib.check(lib.isx_preprocess_stats(x.data_ptr(), _lib.DTYPE_U8, lay, B, 3, H, W, oh, ow, mean.ptr, std.ptr, ws.data_ptr(),
                                        ws.numel(), stream()), "stats")
    mean.check("stats mean")
    std.check("stats std")
    out = Guarded(B * 3 * oh * ow * (4 if out_dtype == _lib.DTYPE_F32 else 2))
    _lib.check(lib.isx_preprocess_apply(x.data_ptr(), _lib.DTYPE_U8, lay, B, 3, H, W, oh, ow, mean.ptr, std.ptr, 1, 1e-6, 1, -3.0,
                                        1, 3.0, out.ptr, out_dtype, stream()), "apply")
    out.check(f"preprocess_apply {layout} {shape} -> {out_hw}")
    vals = out.as_tensor(torch.float32 if out_dtype == _lib.DTYPE_F32 else torch.bfloat16, (B, 3, oh, ow)).float()
    assert bool(torch.isfinite(vals).all()) and float(vals.abs().max()) <= 3.0


@pytest.mark.parametrize("case", [(2, 128, 192, 64, 64, None), (1, 100, 130, 32, 16, None), (2, 70, 90, 24, 24, (12, 12)), (1, 96, 128, 32, 16, None)])
@pytest.mark.parametrize("layout", ["nhwc", "nchw"])
def test_patch_apply_stays_in_bounds(case, layout):
    lib = _lib.load()
    n, H, W, P, S, out_hw = case
    g = torch.Generator(device="cuda").manual_seed(H + W)
    x = torch.randint(0, 256, (n, H, W, 3) if layout == "nhwc" else (n, 3, H, W), dtype=torch.uint8, device="cuda", generator=g)
    lay = _lib.LAYOUT_NHWC if layout == "nhwc" else _lib.LAYOUT_NCHW
    oh, ow = out_hw or (P, P)
    ny, nx = (H - P) // S + 1, (W - P) // S + 1
    mean = torch.full((3,), 120.0, device="cuda")
    std = torch.full((3,), 60.0, device="cuda")
    out = Guarded(n * ny * nx * 3 * oh * ow * 4)
    _lib.check(lib.isx_preprocess_patches_apply(x.data_ptr(), lay, n, 3, H, W, P, S, oh, ow, mean.data_ptr(), std.data_ptr(), 1e-6,
                                                1, -3.0, 1, 3.0, out.ptr, _lib.DTYPE_F32, stream()), "patches apply")
    out.check(f"patches {case} {layout}")
    assert bool(torch.isfinite(out.as_tensor(torch.float32, (-1,))).all())


@pytest.mark.parametrize("B,E,h,w", [(3, 320, 8, 8), (2, 96, 7, 10), (3, 200, 5, 4), (1, 1280, 16, 16)])
def test_l2norm_cells_stays_in_bounds(B, E, h, w):
    lib = _lib.load()
    x = torch.randn((B, E, h, w), device="cuda")
    out = Guarded(x.numel() * 4)
    _lib.check(lib.isx_l2norm_cells(x.data_ptr(), B, E, h, w, 1e-12, out.ptr, stream()), "l2norm")
    out.check(f"l2norm_cells {(B, E, h, w)}")
    norms = out.as_tensor(torch.float32, (B, E, h, w)).norm(dim=1)
    assert torch.allclose(norms, torch.ones_like(norms), atol=1e-5)


@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("B,E,h,w,k", [(3, 320, 16, 16, 96), (3, 320, 16, 16, 95), (5, 128, 8, 8, 24), (5, 128, 8, 8, 23),
                                       (2, 192, 7, 10, 100), (2, 192, 7, 10, 99), (9, 64, 4, 4, 256), (9, 64, 4, 4, 255),
                                       (2, 200, 7, 10, 100)])
def test_project_stays_in_bounds(B, E, h, w, k, aligned):
    """Each per-cell kernel, reached by shape and alignment (launch_project in project.cu): an aligned
    16 x 16, 8 x 8 or 4 x 4 map takes the staged kernel (rule 2) for any k; otherwise k % 4 == 0 takes
    K3d (rule 3) and k % 4 != 0 the register path (rule 4), which writes rows of k floats without TMA
    stores.  E = 200 (E % 16 != 0) takes the register path with k % 4 == 0 (rule 4 through E % 16), so
    its float4 stores and their scalar tail are checked too.  An unaligned map starts 4 bytes into its
    allocation."""
    lib = _lib.load()
    rng = np.random.default_rng(k)
    comps = torch.from_numpy(np.linalg.qr(rng.standard_normal((E, k)))[0].astype(np.float32) if k <= E else
                             rng.standard_normal((E, k)).astype(np.float32)).cuda().contiguous()
    means = torch.zeros(E, device="cuda")
    packed = torch.empty(lib.isx_project_packed_bytes(E, k), dtype=torch.uint8, device="cuda")
    _lib.check(lib.isx_project_pack(means.data_ptr(), comps.data_ptr(), E, k, comps.stride(0), comps.stride(1), packed.data_ptr(),
                                    packed.numel(), stream()), "pack")
    off = 0 if aligned else 1
    fmap = torch.empty(B * E * h * w + off, device="cuda")[off:].view(B, E, h, w)
    fmap.copy_(torch.randn((B, E, h, w), device="cuda").abs_())
    assert (fmap.data_ptr() % 16 == 0) == aligned
    out = Guarded(B * h * w * k * 4)
    _lib.check(lib.isx_l2norm_project(fmap.data_ptr(), B, E, h, w, 0, 1, packed.data_ptr(), k, out.ptr, None, 0, stream()), "project")
    out.check(f"l2norm_project {(B, E, h, w, k)} aligned={aligned}")
    got = out.as_tensor(torch.float32, (B * h * w, k))
    ref = torch.nn.functional.normalize(fmap, dim=1).permute(0, 2, 3, 1).reshape(-1, E) @ comps
    assert (got - ref).abs().max() <= 1e-4 * max(1.0, float(ref.abs().max()))


@pytest.mark.parametrize("n,q,d,k", [(3000, 70, 64, 10), (700, 33, 72, 100), (5000, 257, 128, 16), (2500, 513, 64, 100), (300, 7, 8, 5)])
@pytest.mark.parametrize("packed", [False, True])
def test_knn_outputs_and_workspace_stay_in_bounds(n, q, d, k, packed):
    lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(n + q)
    store = torch.randn((n, d), generator=g, device="cuda").to(torch.bfloat16)
    queries = torch.randn((q, d), generator=g, device="cuda").to(torch.bfloat16)
    srn = Guarded(n * 4)
    qrn = Guarded(q * 4)
    _lib.check(lib.isx_row_rnorm_bf16(store.data_ptr(), n, d, 1e-12, srn.ptr, stream()), "rnorm")
    _lib.check(lib.isx_row_rnorm_bf16(queries.data_ptr(), q, d, 1e-12, qrn.ptr, stream()), "rnorm")
    srn.check("store rnorm")
    qrn.check("query rnorm")
    ws = Guarded(int(lib.isx_knn_workspace_bytes(n, q, d, k)))
    if packed:
        out = Guarded(q * k * 8)
        _lib.check(lib.isx_knn_search_ex(store.data_ptr(), srn.ptr, n, queries.data_ptr(), qrn.ptr, q, d, k, 0, 0, _lib.KNN_PACKED,
                                         out.ptr, None, ws.ptr, ws.nbytes, stream()), "search packed")
        out.check("packed records")
    else:
        out_s, out_i = Guarded(q * k * 4), Guarded(q * k * 4)
        _lib.check(lib.isx_knn_search(store.data_ptr(), srn.ptr, n, queries.data_ptr(), qrn.ptr, q, d, k, 0, out_s.ptr, out_i.ptr,
                                      ws.ptr, ws.nbytes, stream()), "search")
        out_s.check("scores")
        out_i.check("indices")
        idx = out_i.as_tensor(torch.int32, (q, k))
        assert int(idx.max()) < n and int(idx[:, : min(k, n)].min()) >= 0
    ws.check(f"knn workspace {(n, q, d, k)}")


@pytest.mark.parametrize("n,F", [(3000, 320), (100, 37), (5000, 1280)])
def test_pca_moments_stay_in_bounds(n, F):
    lib = _lib.load()
    x = torch.randn((n, F), device="cuda") + 0.5
    mean, cov = Guarded(F * 4), Guarded(F * F * 4)
    ws = Guarded(int(lib.isx_pca_moments_workspace_bytes(n, F)))
    _lib.check(lib.isx_pca_moments(x.data_ptr(), n, F, mean.ptr, cov.ptr, ws.ptr, ws.nbytes, stream()), "moments")
    mean.check("pca mean")
    cov.check("pca cov")
    ws.check(f"pca workspace {(n, F)}")
    ref = torch.cov(x.double().T)
    got = cov.as_tensor(torch.float32, (F, F)).double()
    assert (got - ref).abs().max() <= 2e-5 * float(ref.abs().max())
