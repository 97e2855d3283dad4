#!/usr/bin/env python
"""Small invocation of every kernel family, for `compute-sanitizer --tool memcheck` (one tool per
gpurun call, small shapes: the sanitizer slows kernels by 10-50x).

    compute-sanitizer --tool memcheck --error-exitcode 1 python tools/sanitize_case.py"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from imagescry_b200.image.transforms import preprocess_patches, preprocess_tiles, resize  # noqa: E402
from imagescry_b200.models.decomposition import PCA  # noqa: E402
from imagescry_b200.models.embedding import l2_normalize_cells  # noqa: E402
from imagescry_b200.search import EmbeddingStore  # noqa: E402

g = torch.Generator(device="cuda").manual_seed(0)
tiles = torch.randint(0, 256, (6, 64, 96, 3), dtype=torch.uint8, device="cuda", generator=g)
for kw in (dict(), dict(output_hw=(32, 48)), dict(output_hw=(37, 50)), dict(out_dtype=torch.bfloat16)):
    preprocess_tiles(tiles, layout="nhwc", min_value=-3, max_value=3, **kw)
planar = tiles.permute(0, 3, 1, 2).contiguous()
preprocess_tiles(planar, min_value=-3, max_value=3)
preprocess_tiles(planar, output_hw=(30, 45), min_value=-3, max_value=3)
resize(planar, 40)
big = torch.randint(0, 256, (2, 128, 192, 3), dtype=torch.uint8, device="cuda", generator=g)
preprocess_patches(big, 64, min_value=-3, max_value=3)                         # stream stats + LUT apply
preprocess_patches(big, 64, stride=48, min_value=-3, max_value=3)              # sampling stats + LUT apply
preprocess_patches(big, 50, stride=33, output_hw=(20, 20), min_value=-3, max_value=3)
print("stage 1 ok", flush=True)

fmap = torch.randn((3, 320, 8, 8), generator=g, device="cuda").abs_()
l2_normalize_cells(fmap)
l2_normalize_cells(torch.randn((2, 96, 7, 10), generator=g, device="cuda"))
x = torch.randn((3000, 320), generator=g, device="cuda") * torch.linspace(2, 0.1, 320, device="cuda") + 0.3
pca = PCA(min_num_components=32, max_num_components=32).cuda().fit(x)
pca.transform(x[:500])
pca31 = PCA(min_num_components=31, max_num_components=31).cuda().fit(x)
unaligned = torch.empty(fmap.numel() + 1, device="cuda")[1:].view(fmap.shape).copy_(fmap)  # 4 bytes off 16
odd = torch.randn((2, 320, 7, 10), generator=g, device="cuda")
pca.project_feature_map(fmap)          # staged kernel
pca.project_feature_map(unaligned)     # K3d: no TMA boxes for an unaligned map
pca31.project_feature_map(unaligned)   # register path: k % 4 != 0
pca.project_feature_map(odd)           # odd shape: K3d
pca31.project_feature_map(odd)         # odd shape, k % 4 != 0: register path
pca200 = PCA(min_num_components=32, max_num_components=32).cuda().fit(x[:, :200].contiguous())
pca200.project_feature_map(torch.randn((2, 200, 7, 10), generator=g, device="cuda"))  # E % 16 != 0: register path, float4 stores
pca.project_feature_map(fmap, pool="mean")
print("stage 2 ok", flush=True)

store = torch.randn((6000, 128), generator=g, device="cuda").to(torch.bfloat16)
q = torch.randn((300, 128), generator=g, device="cuda").to(torch.bfloat16)
st = EmbeddingStore(store)
for k in (10, 100):
    st.search(q, k)
st.search_packed(q, 10)
st.knn_graph(5)
EmbeddingStore(torch.randn((700, 37), generator=g, device="cuda")).search(torch.randn((9, 37), generator=g, device="cuda"), 3)
torch.cuda.synchronize()
print("stage 3 ok", flush=True)
