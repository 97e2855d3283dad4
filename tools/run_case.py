#!/usr/bin/env python
"""Run one kernel case in isolation (for ncu / quick timing on the GPU box).

    python tools/run_case.py knn --n 1000000 --q 10000 --k 100 [--iters 3]
    python tools/run_case.py preprocess --case resize256|nhwc_f32|nhwc_bf16|nchw_f32 [--batch 1024]
    python tools/run_case.py project --pool none|mean [--batch 1024] [--side 16]
Prints the CUDA-event time per iteration and the roofline fraction."""
from __future__ import annotations

import argparse
import json
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)


def timeit(fn, iters, warm=2):
    import torch

    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return ts


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("what", choices=["knn", "preprocess", "project", "l2norm", "graph", "pcafit"])
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--q", type=int, default=10_000)
    ap.add_argument("--d", type=int, default=1280)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--case", default="resize256")
    ap.add_argument("--pool", default="none")
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--precision", default="exact")
    ap.add_argument("--side", type=int, default=16, help="feature-map side for the l2norm and project cases")
    a = ap.parse_args()
    peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(REPO, "MEASURED_PEAKS.json")) else {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(1)
    if a.what == "knn":
        from imagescry_b200.search import EmbeddingStore

        store = torch.empty((a.n, a.d), dtype=torch.bfloat16, device=dev)
        for s in range(0, a.n, 1 << 20):
            e = min(a.n, s + (1 << 20))
            store[s:e] = torch.randn((e - s, a.d), generator=g, device=dev).to(torch.bfloat16)
        q = torch.randn((a.q, a.d), generator=g, device=dev).to(torch.bfloat16)
        st = EmbeddingStore(store)
        ts = timeit(lambda: st.search_raw(q, a.k), a.iters, a.warm)
        ms = min(ts)
        tf = 2.0 * a.q * a.n * a.d / (ms * 1e-3) / 1e12
        print(json.dumps({"case": f"knn n={a.n} q={a.q} d={a.d} k={a.k}", "ms": ts, "tflops": tf,
                          "frac_sustained": tf / peaks["bf16_tflops_sustained"], "frac_burst": tf / peaks["bf16_tflops"]}))
    elif a.what == "l2norm":
        from imagescry_b200.models.embedding import l2_normalize_cells

        B, E, h, w = a.batch, 1280, a.side, a.side
        fmap = torch.randn((B, E, h, w), generator=g, device=dev)
        ts = timeit(lambda: l2_normalize_cells(fmap), a.iters, a.warm)
        gbs = fmap.numel() * 8 / (min(ts) * 1e-3) / 1e9
        print(json.dumps({"case": f"l2norm B={B} {h}x{w}", "ms": ts, "GBps": gbs, "frac_hbm": gbs / peaks["hbm_gbs"]}))
    elif a.what == "graph":
        from imagescry_b200.search import EmbeddingStore

        store = torch.randn((a.n, a.d), generator=g, device=dev).to(torch.bfloat16)
        st = EmbeddingStore(store)
        ts = timeit(lambda: st.knn_graph(a.k), a.iters, a.warm)
        tf = 2.0 * a.n * a.n * a.d / (min(ts) * 1e-3) / 1e12
        print(json.dumps({"case": f"graph n={a.n} d={a.d} k={a.k}", "ms": ts, "tflops": tf, "frac_sustained": tf / peaks["bf16_tflops_sustained"]}))
    elif a.what == "pcafit":
        from imagescry_b200.models.decomposition import PCA

        x = torch.randn((a.n, a.d), generator=g, device=dev) + 0.5
        pca = PCA(min_num_components=64, max_num_components=64).cuda()
        ts = timeit(lambda: pca._moments(x), a.iters, a.warm)
        print(json.dumps({"case": f"pca moments n={a.n} F={a.d}", "ms": ts}))
    elif a.what == "preprocess":
        from imagescry_b200.image.transforms import preprocess_tiles

        B = a.batch
        tiles = torch.randint(0, 256, (B, 512, 512, 3), dtype=torch.uint8, device=dev, generator=g)
        n = tiles.numel()
        if a.case == "resize256":
            kw, algo = dict(layout="nhwc", output_hw=(256, 256)), 2 * n + 4 * (n // 4)
        elif a.case == "resize384":
            kw, algo = dict(layout="nhwc", output_hw=(384, 384)), 2 * n + 4 * (n * 9 // 16)
        elif a.case == "nhwc_f32":
            kw, algo = dict(layout="nhwc"), 2 * n + 4 * n
        elif a.case == "nhwc_bf16":
            kw, algo = dict(layout="nhwc", out_dtype=torch.bfloat16), 2 * n + 2 * n
        elif a.case == "nchw_f32":
            tiles = tiles.permute(0, 3, 1, 2).contiguous()
            kw, algo = dict(layout="nchw"), 2 * n + 4 * n
        elif a.case == "nchw_resize256":
            tiles = tiles.permute(0, 3, 1, 2).contiguous()
            kw, algo = dict(layout="nchw", output_hw=(256, 256)), 2 * n + 4 * (n // 4)
        else:
            raise SystemExit(f"unknown case {a.case}")
        ts = timeit(lambda: preprocess_tiles(tiles, min_value=-3, max_value=3, **kw), a.iters, a.warm)
        ms = min(ts)
        gbs = algo / (ms * 1e-3) / 1e9
        print(json.dumps({"case": f"preprocess {a.case} B={B}", "ms": ts, "GBps": gbs, "frac_hbm": gbs / peaks["hbm_gbs"], "tiles_per_s": B / (ms * 1e-3)}))
    else:
        from imagescry_b200.models.decomposition import PCA

        B, E, h, w, k = a.batch, 1280, a.side, a.side, 256
        fmap = torch.empty((B, E, h, w), dtype=torch.float32, device=dev)
        for s in range(0, B, 256):
            e = min(B, s + 256)
            fmap[s:e] = torch.randn((e - s, E, h, w), generator=g, device=dev).abs_()
        comps = torch.linalg.qr(torch.randn((E, k), generator=g, device=dev))[0]
        pca = PCA(num_features=E, num_components=k).cuda()
        pca.feature_means.data = torch.randn((1, E), generator=g, device=dev) * 0.01
        pca.component_vectors.data = comps.contiguous()
        pca._fitted.data = torch.tensor(True, device=dev)
        pca._num_features.data = torch.tensor(E, device=dev)
        pca._num_components.data = torch.tensor(k, device=dev)
        pca.packed_weights()
        pool = None if a.pool in ("none", "flat") else a.pool
        algo = fmap.numel() * 4 + (B * h * w * k * 4 if pool is None else B * k * 4)
        if a.pool == "flat":
            # the reference's literal seam: PCA.transform on the (B*h*w) x E flat-vector matrix
            flat = fmap.permute(0, 2, 3, 1).reshape(-1, E).contiguous()
            del fmap
            ts = timeit(lambda: pca.transform(flat), a.iters, a.warm)
        else:
            ts = timeit(lambda: pca.project_feature_map(fmap, pool=pool, precision=a.precision), a.iters, a.warm)
        ms = min(ts)
        gbs = algo / (ms * 1e-3) / 1e9
        print(json.dumps({"case": f"project pool={a.pool} B={B}", "ms": ts, "GBps": gbs, "frac_hbm": gbs / peaks["hbm_gbs"]}))


if __name__ == "__main__":
    main()
