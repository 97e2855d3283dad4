"""fp8 search against `search(k=10)` on the same store, in one process, alternating.

For every case (1 M-row store, 10 k queries, d = 1280 and 256, N(0, 1) rows or correlated rows = a
per-image base vector (256 cells per image) + small noise, as in bench_grouped.make_store) four calls
are timed with CUDA events, alternating:
  search      `search_raw(queries, 10)` (query norms, bf16 search kernel, finalising merge);
  scan16      `scan_fp8(queries, 16)`: query quantization and the fp8 scan alone;
  fp8_c16     `search_fp8_raw(queries, 10, candidates=16)`: scan, query norms, exact re-score;
  fp8_c32     the same with 32 candidates (the CAP-256 epilogue).
One JSON line per case is printed with the median times, their ratios to `search`, recall@10 of both
fp8 calls against `search`, and the GPU's name and power limit read in the same run.

    python tools/bench_fp8.py [--reps 5] [--cases d1280_randn,...] [--out FILE]
"""

from __future__ import annotations

import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from bench_grouped import gpu_info, make_store  # noqa: E402
from imagescry_b200 import search as S  # noqa: E402


def recall(idx, ref):
    return float((idx[:, :, None] == ref[:, None, :]).any(dim=2).float().mean())


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cases", default="")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    info = gpu_info()
    n, cells = 1_000_000, 256
    n -= n % cells
    want = set(filter(None, args.cases.split(",")))
    out = open(args.out, "a") if args.out else None
    for d in (1280, 256):
        for kind in ("randn", "correlated"):
            name = f"d{d}_{kind}"
            if want and name not in want:
                continue
            store, queries = make_store(n, d, cells, kind, seed=d + 20)
            st = S.EmbeddingStore(store, fp8=True)
            calls = {
                "search": lambda: st.search_raw(queries, 10),
                "scan16": lambda: st.scan_fp8(queries, 16),
                "fp8_c16": lambda: st.search_fp8_raw(queries, 10, candidates=16),
                "fp8_c32": lambda: st.search_fp8_raw(queries, 10, candidates=32),
            }
            for f in calls.values():  # warm-up: module load, workspace allocation, clocks
                f()
                f()
            times = {c: [] for c in calls}
            for _ in range(args.reps):
                for c, f in calls.items():
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    f()
                    e1.record()
                    e1.synchronize()
                    times[c].append(e0.elapsed_time(e1))
            _, ref = st.search_raw(queries, 10)
            r16 = recall(calls["fp8_c16"]()[1], ref)
            r32 = recall(calls["fp8_c32"]()[1], ref)
            ms = {c: sorted(t)[len(t) // 2] for c, t in times.items()}
            line = json.dumps({
                "case": name, "n": n, "q": queries.shape[0], "d": d, "data": kind, "k": 10,
                **{f"{c}_ms": round(v, 3) for c, v in ms.items()},
                **{f"{c}_ratio": round(ms[c] / ms["search"], 4) for c in ("scan16", "fp8_c16", "fp8_c32")},
                "recall10_c16": round(r16, 5), "recall10_c32": round(r32, 5),
                "all_ms": {c: [round(x, 3) for x in t] for c, t in times.items()}, **info,
            })
            print(line, flush=True)
            if out:
                out.write(line + "\n")
                out.flush()
            del st, store, queries
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
