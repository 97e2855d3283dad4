"""Range search against `search(k=10)` on the same store, in one process, alternating.

For every case (1 M-row store, 10 k queries, d = 1280 and 256, N(0, 1) rows or correlated rows = a
per-image base vector (256 cells per image) + small noise, τ at about 10 and about 200 hits per query)
three calls are timed with CUDA events, alternating:
  search        `search_raw(queries, 10)` (query norms, search kernel, finalising merge);
  range_kernel  one `isx_knn_range` launch into a buffer large enough for every hit;
  range_total   `search_range(queries, τ)`: query norms, kernel, count read, ordering pass.
One JSON line per case is printed with the median times, the mean hits per query, and the GPU's name
and power limit read in the same run.  τ for about 10 hits is the median over the queries of the 10th
score of `search(k=10)`; for about 200 it is the median 200th score of 256 sampled queries (fp32 brute
force).

    python tools/bench_range.py [--reps 5] [--cases d1280_randn_h10,...] [--out FILE]
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
from imagescry_b200 import _lib  # noqa: E402
from imagescry_b200 import search as S  # noqa: E402


def tau_for(st, queries, s10, hits):
    if hits <= 10:
        return float(s10[:, hits - 1].median())
    pick = torch.arange(0, queries.shape[0], queries.shape[0] // 256, device="cuda")[:256]
    qn = torch.nn.functional.normalize(queries[pick].float(), dim=1)
    kth = []
    for s0 in range(0, len(st), 1 << 17):
        e = st.embeddings[s0:s0 + (1 << 17)].float()
        kth.append((qn @ e.T * st.rnorm[s0:s0 + (1 << 17)]).topk(hits, dim=1).values)
    return float(torch.cat(kth, dim=1).topk(hits, dim=1).values[:, hits - 1].median())


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cases", default="")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    info = gpu_info()
    lib = _lib.load()
    n, cells = 1_000_000, 256
    n -= n % cells
    want = set(filter(None, args.cases.split(",")))
    out = open(args.out, "a") if args.out else None
    for d in (1280, 256):
        for kind in ("randn", "correlated"):
            if want and not any(w.startswith(f"d{d}_{kind}_") for w in want):
                continue
            store, queries = make_store(n, d, cells, kind, seed=d + 10)
            st = S.EmbeddingStore(store)
            nq = queries.shape[0]
            qr = S.row_rnorm(queries)
            s10, _ = st.search_raw(queries, 10)
            for hits in (10, 200):
                name = f"d{d}_{kind}_h{hits}"
                if want and name not in want:
                    continue
                tau = tau_for(st, queries, s10, hits)
                _, total = st.range_records(queries, qr, tau)
                records = torch.empty((max(total, 1), 3), dtype=torch.int32, device="cuda")
                count = torch.zeros(1, dtype=torch.int64, device="cuda")
                ws = torch.empty(_lib.KNN_RANGE_WORKSPACE_BYTES, dtype=torch.uint8, device="cuda")

                def kernel():
                    rc = lib.isx_knn_range(store.data_ptr(), st.rnorm.data_ptr(), n, queries.data_ptr(), qr.data_ptr(), nq, d,
                                           tau, 0, 0, 0, records.data_ptr(), records.shape[0], count.data_ptr(), ws.data_ptr(),
                                           ws.numel(), torch.cuda.current_stream().cuda_stream)
                    _lib.check(rc, "isx_knn_range")

                calls = {"search": lambda: st.search_raw(queries, 10), "range_kernel": kernel,
                         "range_total": lambda: st.search_range(queries, tau)}
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
                assert int(count.item()) == total
                ms = {c: sorted(t)[len(t) // 2] for c, t in times.items()}
                line = json.dumps({
                    "case": name, "n": n, "q": nq, "d": d, "data": kind, "tau": tau, "hits": total,
                    "mean_hits_per_query": round(total / nq, 2), "search_k10_ms": round(ms["search"], 3),
                    "range_kernel_ms": round(ms["range_kernel"], 3), "range_total_ms": round(ms["range_total"], 3),
                    "kernel_ratio": round(ms["range_kernel"] / ms["search"], 4),
                    "total_ratio": round(ms["range_total"] / ms["search"], 4),
                    "all_ms": {c: [round(x, 3) for x in t] for c, t in times.items()}, **info,
                })
                print(line, flush=True)
                if out:
                    out.write(line + "\n")
                    out.flush()
                del records
            del st, store, queries
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
