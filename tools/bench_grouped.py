"""Image-level search against row-level search on the same store, in one process, alternating.

For every case (store 1 M rows with 256 cells per image, 10 k queries, k = 10 and 100, d = 1280 and
256, N(0, 1) rows or correlated rows = per-image base vector + small noise) the two calls are timed
with CUDA events, alternating `search` and `search_images`, and one JSON line is printed with both
times, their ratio, the fraction of the sustained bf16 rate (bench.load_peaks(), with its source)
each call reaches on the Q x N x d product, and the GPU's name and power limit read in the same run.

    python tools/bench_grouped.py [--reps 5] [--cases d1280_k10_randn,...]
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from bench import load_peaks  # noqa: E402
from imagescry_b200 import search as S  # noqa: E402


def gpu_info() -> dict:
    out = {"gpu": torch.cuda.get_device_name()}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        out["power_limit_clocks"] = r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as ex:
        out["power_limit_clocks"] = f"unavailable ({ex!r})"
    return out


def make_store(n, d, cells, kind, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    store = torch.empty((n, d), dtype=torch.bfloat16, device="cuda")
    images = n // cells
    base = torch.randn((images, d), generator=g, device="cuda") if kind == "correlated" else None
    for s0 in range(0, n, 1 << 17):
        e = min(n, s0 + (1 << 17))
        x = torch.randn((e - s0, d), generator=g, device="cuda")
        if base is not None:
            x = base[torch.arange(s0, e, device="cuda") // cells] + 0.1 * x
        store[s0:e] = x.to(torch.bfloat16)
    if base is not None:  # queries near random images (an ROI or cell query of a stored image)
        pick = torch.randint(0, images, (10_000,), generator=g, device="cuda")
        queries = (base[pick] + 0.3 * torch.randn((10_000, d), generator=g, device="cuda")).to(torch.bfloat16)
    else:
        queries = torch.randn((10_000, d), generator=g, device="cuda").to(torch.bfloat16)
    return store, queries


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cases", default="")
    args = ap.parse_args()
    peaks = load_peaks()
    info = gpu_info()
    n, cells = 1_000_000, 256
    n -= n % cells
    cases = [(d, k, kind) for d in (1280, 256) for kind in ("randn", "correlated") for k in (10, 100)]
    want = set(filter(None, args.cases.split(",")))
    for d, k, kind in cases:
        name = f"d{d}_k{k}_{kind}"
        if want and name not in want:
            continue
        store, queries = make_store(n, d, cells, kind, seed=d + k)
        st = S.EmbeddingStore(store, groups=cells)
        calls = {"search": lambda: st.search_raw(queries, k), "search_images": lambda: st.search_images_raw(queries, k)}
        for f in calls.values():  # warm-up: module load, workspace allocation, clocks
            f()
            f()
        times = {name_: [] for name_ in calls}
        for _ in range(args.reps):
            for cname, f in calls.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                f()
                e1.record()
                e1.synchronize()
                times[cname].append(e0.elapsed_time(e1))
        ms = {c: sorted(t)[len(t) // 2] for c, t in times.items()}
        flop = 2.0 * queries.shape[0] * n * d
        rate = peaks["bf16_tflops_sustained"] * 1e12
        print(json.dumps({
            "case": name, "n": n, "q": queries.shape[0], "d": d, "k": k, "cells_per_image": cells, "data": kind,
            "search_ms": round(ms["search"], 3), "search_images_ms": round(ms["search_images"], 3),
            "ratio": round(ms["search_images"] / ms["search"], 4),
            "search_frac_of_sustained_bf16": round(flop / (ms["search"] * 1e-3) / rate, 4),
            "search_images_frac_of_sustained_bf16": round(flop / (ms["search_images"] * 1e-3) / rate, 4),
            "peak_source": peaks["_source"], "all_ms": {c: [round(x, 3) for x in t] for c, t in times.items()}, **info,
        }), flush=True)
        del st, store, queries
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
