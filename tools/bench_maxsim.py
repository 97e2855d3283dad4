"""Multi-vector (maxsim) image search against `search(k=10)` on the same query rows, in one process,
alternating.

For every case (999 936-row store, 256 cells per image, d = 1280 and 256, N(0, 1) rows or correlated
rows = a per-image base vector + 0.1 noise, as in bench_grouped.make_store) and 10 000 query rows in
250 sets of 40, four calls are timed with CUDA events, alternating:
  search      `search_raw(queries, 10)` on the 10 000 rows (query norms, search kernel, merge);
  maxsim      `search_images_maxsim(queries, 40, 10)`: the whole call (norms, cell-max kernel, set
              reduce, merge);
  cellmax     `isx_knn_maxsim` alone (Q × 3 906 fp32 maxima, 156 MB);
  reduce      `isx_maxsim_sets_topk` alone over that matrix.
One JSON line per case is printed with the median of `--reps` runs, the ratio of maxsim to search,
a check of 8 sampled sets against an fp32 brute force over the whole store, and the GPU's name and
power limit read in the same run.

    python tools/bench_maxsim.py [--reps 5] [--cases d1280_randn,...] [--out FILE]
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

SET = 40
PICK = [0, 1, 37, 100, 128, 199, 248, 249]


def verify(store, queries, cells, scores, images, k):
    """Sampled sets against an fp32 brute force: (max |score error|, every differing image within 1e-3
    of the exact k-th)."""
    n = store.shape[0]
    rows = torch.cat([torch.arange(p * SET, (p + 1) * SET) for p in PICK]).cuda()
    qn = torch.nn.functional.normalize(queries[rows].float(), dim=1)
    best = torch.empty((len(rows), n // cells), device="cuda")
    for s0 in range(0, n, 1 << 16):
        e = min(n, s0 + (1 << 16))
        sc = qn @ torch.nn.functional.normalize(store[s0:e].float(), dim=1).T
        best[:, s0 // cells:e // cells] = sc.view(len(rows), -1, cells).amax(2)
    f64 = best.double().view(len(PICK), SET, -1).mean(1)
    ex_s, ex_i = f64.topk(k, dim=1)
    err = (scores[PICK].double() - ex_s).abs().max().item()
    ok = err <= 1e-3
    for r in range(len(PICK)):
        for j in set(images[PICK[r]].tolist()) ^ set(ex_i[r].tolist()):
            ok &= abs(f64[r, j].item() - ex_s[r, -1].item()) < 1e-3
    return err, bool(ok)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cases", default="")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    info = gpu_info()
    cells, k = 256, 10
    n = 999_936
    want = set(filter(None, args.cases.split(",")))
    out = open(args.out, "a") if args.out else None
    lib = _lib.load()
    for d in (1280, 256):
        for kind in ("randn", "correlated"):
            name = f"d{d}_{kind}"
            if want and name not in want:
                continue
            store, queries = make_store(n, d, cells, kind, seed=d + 30)
            st = S.EmbeddingStore(store, groups=cells)
            nq, images = queries.shape[0], n // cells
            qr = S.row_rnorm(queries)
            cm = torch.empty((nq, images), dtype=torch.float32, device="cuda")
            ws = torch.empty(_lib.KNN_RANGE_WORKSPACE_BYTES, dtype=torch.uint8, device="cuda")
            sets = torch.arange(0, nq + 1, SET, dtype=torch.int64, device="cuda")
            rec = torch.empty((nq // SET, k), dtype=torch.int64, device="cuda")
            strm = torch.cuda.current_stream().cuda_stream

            def cellmax():
                _lib.check(lib.isx_knn_maxsim(store.data_ptr(), st.rnorm.data_ptr(), st.row_group.data_ptr(), n,
                                              queries.data_ptr(), qr.data_ptr(), nq, d, 0, images, cm.data_ptr(),
                                              ws.data_ptr(), ws.numel(), strm), "isx_knn_maxsim")

            def reduce():
                _lib.check(lib.isx_maxsim_sets_topk(cm.data_ptr(), qr.data_ptr(), nq, images, 0, images, sets.data_ptr(),
                                                    nq // SET, k, 0, rec.data_ptr(), strm), "isx_maxsim_sets_topk")

            calls = {
                "search": lambda: st.search_raw(queries, k),
                "maxsim": lambda: st.search_images_maxsim(queries, SET, k),
                "cellmax": cellmax,
                "reduce": reduce,
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
            scores, imgs = st.search_images_maxsim(queries, SET, k)
            err, ok = verify(store, queries, cells, scores, imgs, k)
            ms = {c: sorted(t)[len(t) // 2] for c, t in times.items()}
            line = json.dumps({
                "case": name, "n": n, "q": nq, "sets": nq // SET, "set_size": SET, "images": images, "d": d, "data": kind,
                "k": k, **{f"{c}_ms": round(v, 3) for c, v in ms.items()},
                "maxsim_ratio": round(ms["maxsim"] / ms["search"], 4), "verify_max_err": err, "verify_ok": ok,
                "all_ms": {c: [round(x, 3) for x in t] for c, t in times.items()}, **info,
            })
            print(line, flush=True)
            if out:
                out.write(line + "\n")
                out.flush()
            del st, store, queries, cm
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
