#!/usr/bin/env python
"""Benchmark of the sift path on B200 — the metric of BASELINE.json.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Primary line (one JSON object on stdout, rank 0):
  metric   knn_queries_per_sec — cosine k-NN, k=10, 1280-d, over a 1 M x 1280 bf16 embedding store
           with 10 k queries (BASELINE.json configs[1]).  A step = one pass of all queries over the
           store: query inverse norms + tcgen05 GEMM with fused top-k + merge (N > 1, store
           row-sharded: the finalising pass stores packed records into every rank's gather buffer
           over NVLink, barrier, merge; scaling = strong: the 1 M-row store is fixed and split N ways).
  value    device-timed (CUDA events, max over ranks), inputs resident in HBM, after a 2 s pre-heat.
  e2e      the same metric through the public API from pinned HOST query buffers, every step's H2D
           and D2H inside the timed region: `value` streams the steps through HostBatchSearch.run
           (copies on a copy stream beside the neighbouring step's search), `one_batch_at_a_time` is
           the strictly sequential form (upload, search, download, host sync).
  roofline bf16 tensor roofline of the search kernel, timed live with CUDA events on its stream.
  verify   (untimed) sampled queries through the product path against an exact fp32 brute force over
           every rank's shard; every differing index justified by its score gap.
  cpu_baseline  the torch-CPU port of the same workload (oracle/torch_port.py) on a bounded sample,
           plus stage 1 / stage 2 / PCA.fit and a config-1 sample on the host cores.
  extra    stage 1 (tiles/s, HBM roofline) and stage 2 (cells/s, HBM roofline) of config 3 on every
           rank, PCA.fit, other search shapes, the scaled sift run; at N > 1 config 4 at its full
           100 M-row size (k = 10 and 100, verified) and the config-5 all-pairs graph.

--impl reference times the reference-side CPU implementation only (rank 0), same metric/config.
--dump-outputs DIR writes what the last timed step returned (rank 0): DIR/scores.npy and
DIR/indices.npy.  The inputs are seeded, so two builds run with the same arguments can be compared
output for output.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

Q = 10_000
D = 1280
K = 10
N_STORE = 1_000_000
METRIC = "knn_queries_per_sec"
UNIT = "queries/s"


def load_peaks() -> dict:
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        p["_source"] = "measured"
        return p
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "_source": "fallback"}


def load_traffic():
    """DRAM bytes per launch of the search kernel (dram__bytes_read.sum + dram__bytes_write.sum) from
    the committed `ncu --set full` capture of this same workload, or None."""
    path = os.path.join(REPO, "profiles", "knn_search_traffic.json")
    try:
        with open(path) as fh:
            return json.load(fh)["dram_bytes_per_launch"]
    except Exception:
        return None


class ClockSampler:
    """Samples nvidia-smi clocks and throttle reasons while the timed region runs."""

    FIELDS = (
        "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
        "clocks_event_reasons.sw_power_cap"
    )

    def __init__(self, gpu_index: int) -> None:
        self.gpu_index = gpu_index
        self.samples: list[list[str]] = []
        self._stop = threading.Event()
        self._thread: threading.Thread | None = None

    def _run(self) -> None:
        # one long-lived nvidia-smi streaming a sample every 100 ms (spawning it per sample takes
        # longer than a whole timed region)
        try:
            self._proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )
        except Exception:
            self._proc = None
            return
        for line in self._proc.stdout:  # ends when __exit__ terminates the process
            line = line.strip()
            if line:
                self.samples.append([v.strip() for v in line.split(",")])

    def __enter__(self):
        self._proc = None
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()
        time.sleep(0.35)  # let the first samples arrive before the timed region starts
        self._n_before = len(self.samples)
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._proc is not None:
            try:
                self._proc.terminate()
            except Exception:
                pass
        if self._thread:
            self._thread.join(timeout=3)

    def summary(self) -> dict:
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples[getattr(self, "_n_before", 0):] or self.samples:
            try:
                sm.append(float(s[0]))
                mx.append(float(s[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(names, s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {
            "sm_mhz": statistics.median(sm) if sm else None,
            "sm_max_mhz": max(mx) if mx else None,
            "reasons": sorted(reasons),
            "samples": len(sm),
        }


# ------------------------------------------------------------------------------------------------
# reference arm: CPU port on the host cores
# ------------------------------------------------------------------------------------------------
def host_store(n: int, d: int, seed: int):
    import torch

    g = torch.Generator().manual_seed(seed)
    out = torch.empty((n, d), dtype=torch.bfloat16)
    for s in range(0, n, 131072):
        e = min(n, s + 131072)
        out[s:e] = torch.randn((e - s, d), generator=g).to(torch.bfloat16)
    return out


def cpu_knn_sample(store_bf16, queries_bf16, seconds_target: float = 12.0) -> dict:
    """Time oracle/torch_port.cosine_knn on all host threads for a bounded number of queries over
    the FULL store (no extrapolation in N)."""
    import torch

    from oracle import torch_port as TP

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    prepared = TP.prepare_store(store_bf16)  # store build: outside the timed region, like the GPU's rnorm
    t0 = time.perf_counter()
    TP.cosine_knn(prepared, queries_bf16[:16], K, prepared=True)
    t_cal = time.perf_counter() - t0
    t0 = time.perf_counter()
    TP.cosine_knn(prepared, queries_bf16[:64], K, prepared=True)
    t_64 = time.perf_counter() - t0
    per_q = max((t_64 - t_cal) / 48.0, 1e-6)
    qs = int(max(64, min(queries_bf16.shape[0], (seconds_target - t_cal) / per_q)))
    t0 = time.perf_counter()
    TP.cosine_knn(prepared, queries_bf16[:qs], K, prepared=True)
    dt = time.perf_counter() - t0
    return {
        "value": qs / dt, "unit": UNIT, "cores": cores, "kind": "port",
        "sample": f"{qs} of the {queries_bf16.shape[0]} queries over the full {store_bf16.shape[0]}x{store_bf16.shape[1]} store, "
                  f"pre-normalised fp32, torch-CPU matmul+topk ({dt:.2f} s)",
        "seconds": dt, "queries": qs,
    }


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    from oracle import torch_port as TP

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    store = host_store(N_STORE, D, seed=1234)
    queries = host_store(Q, D, seed=4321)
    store = TP.prepare_store(store)  # store build (fp32, normalised): outside the timed steps
    knn = lambda q: TP.cosine_knn(store, q, K, prepared=True)  # noqa: E731
    # size one step to ~4 s from a calibration on 32 queries
    knn(queries[:8])  # thread-pool / allocator warm-up
    t0 = time.perf_counter()
    knn(queries[:32])
    t32 = time.perf_counter() - t0
    t0 = time.perf_counter()
    knn(queries[:128])
    t128 = time.perf_counter() - t0
    per_q = max((t128 - t32) / 96.0, 1e-6)
    budget = 150.0 / max(1, args.steps + args.warmup)
    qs = int(max(32, min(Q, (min(budget, 6.0) - (t32 - 32 * per_q)) / per_q)))
    for _ in range(args.warmup):
        knn(queries[:qs])
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        knn(queries[:qs])
        times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    value = qs / dt
    sample = f"{qs} of {Q} queries per step over the full {N_STORE}x{D} store (pre-normalised fp32), torch-CPU matmul+topk port on {cores} threads"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir: str, scores, indices) -> None:
    """Write one timed step's result as `scores.npy` (float32, Q x k) and `indices.npy` (float64,
    Q x k: every int32 row index is exact in it), so that two builds can be compared output for
    output on the same seeded inputs.  10 k x 10 entries: 1.2 MB in all."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "scores.npy"), scores.cpu().numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "indices.npy"), indices.cpu().numpy().astype(np.float64))


def workload_config(n_gpus: int) -> dict:
    return {
        "workload": f"cosine k-NN k={K}: {N_STORE}x{D} bf16 embedding store"
                    + (f" row-sharded over {n_gpus} GPUs" if n_gpus > 1 else " on 1 GPU")
                    + f", {Q} bf16 queries (BASELINE.json configs[1])",
        "store_rows": N_STORE, "dim": D, "queries": Q, "k": K,
        "parallelism": f"row-sharded store x{n_gpus}, replicated queries, one gather of packed records + merge" if n_gpus > 1 else "single GPU",
        "l2": "inputs larger than L2 (store shard >= 320 MB vs 126 MB L2); no explicit flush",
    }


# ------------------------------------------------------------------------------------------------
# verification (untimed): sampled queries against an independent fp32 brute force (torch library ops —
# a checker, never the thing measured).  Also imported by tests/test_gpu_knn.py and test_gpu_multi.py.
# ------------------------------------------------------------------------------------------------
def exact_topk_local(store_bf16, index_base: int, qn_f32, kk: int, chunk: int = 1 << 18, exclude=None):
    """Exact fp32 cosine top-kk of the pre-normalised fp32 queries `qn_f32` over one bf16 store shard,
    chunk by chunk: (scores nq x kk, GLOBAL indices nq x kk int64), ordered (score desc, index asc).
    `exclude`: optional int64 nq vector of global rows that may not be returned (all-pairs graph)."""
    import torch

    nq = qn_f32.shape[0]
    dev = qn_f32.device
    best_v = torch.full((nq, kk), float("-inf"), device=dev)
    best_i = torch.full((nq, kk), -1, dtype=torch.int64, device=dev)
    n = store_bf16.shape[0]
    for s in range(0, n, chunk):
        e = min(n, s + chunk)
        rows = store_bf16[s:e, : qn_f32.shape[1]].float()
        sc = qn_f32 @ torch.nn.functional.normalize(rows, dim=1).T
        if exclude is not None:
            loc = exclude - (index_base + s)
            hit = (loc >= 0) & (loc < e - s)
            if bool(hit.any()):
                sc[hit.nonzero().squeeze(1), loc[hit]] = float("-inf")
        v, i = sc.topk(min(kk, e - s), dim=1)
        best_v, best_i = merge_exact([best_v, v], [best_i, i + (index_base + s)], kk)
    return best_v, best_i


def merge_exact(vals: list, idxs: list, kk: int):
    """Union of candidate lists -> best kk by (score desc, index asc); padding (-inf, -1) sorts last."""
    import torch

    cv, ci = torch.cat(vals, 1), torch.cat(idxs, 1)
    key_i = torch.where(ci < 0, torch.full_like(ci, 1 << 62), ci)
    o = key_i.argsort(dim=1, stable=True)
    cv, ci = cv.gather(1, o), ci.gather(1, o)
    o = cv.argsort(dim=1, descending=True, stable=True)[:, :kk]
    return cv.gather(1, o), ci.gather(1, o)


def judge_topk(prod_s, prod_i, ex_s, ex_i, k: int, tol: float = 1e-3) -> dict:
    """Compare a product result (nq x k) with the exact top-(k + margin) lists `ex_s`, `ex_i`.
    Scores: |product - exact| of every returned index that the exact list holds.  Indices: a returned
    index outside the exact top-k, or an exact top-k index not returned, is accepted only if its exact
    score lies within `tol` of the exact k-th score (BASELINE.json: "index sets identical except where
    score gaps fall below that tolerance"); everything else counts as a mismatch beyond tolerance."""
    import torch

    nq = prod_i.shape[0]
    prod_i = prod_i.to(torch.int64)
    bad = 0
    max_err = 0.0
    differing = 0
    for r in range(nq):
        exact = {int(i): float(v) for v, i in zip(ex_s[r].tolist(), ex_i[r].tolist()) if i >= 0}
        kk = min(k, len(exact))
        kth = sorted(exact.values(), reverse=True)[kk - 1] if kk else float("-inf")
        want = set(ex_i[r, :kk].tolist())
        got = [int(i) for i in prod_i[r].tolist() if i >= 0]
        if len(got) != kk:
            bad += 1
            continue
        for v, i in zip(prod_s[r].tolist(), prod_i[r].tolist()):
            if i < 0:
                continue
            if i in exact:
                max_err = max(max_err, abs(v - exact[i]))
        for i in set(got) ^ want:
            differing += 1
            if i not in exact or abs(exact[i] - kth) > tol:
                bad += 1
    return {"checked": nq, "k": k, "index_mismatch_beyond_tol": bad, "indices_differing_within_tol": differing - bad,
            "max_score_err": max_err, "score_tol": tol}


def verify_search(search_fn, local_store, local_base: int, queries, k: int, dist_on: bool, samples: int = 64,
                  margin: int = 32, exclude_self_base=None) -> dict:
    """Run the product path for `samples` evenly spaced query rows and judge it against the exact fp32
    brute force over EVERY rank's shard (each rank scores its shard; candidates are all-gathered and
    sorted exactly) — this proves the gather + merge + index_base plumbing, not just the local kernel."""
    import torch
    import torch.distributed as dist

    q = queries.shape[0]
    pick = torch.arange(0, q, max(1, q // samples), device=queries.device)[:samples]
    prod_s, prod_i = search_fn(pick)
    qn = torch.nn.functional.normalize(queries[pick].float(), dim=1)
    excl = None if exclude_self_base is None else (pick + exclude_self_base)
    ex_s, ex_i = exact_topk_local(local_store, local_base, qn, k + margin, exclude=excl)
    if dist_on:
        world = dist.get_world_size()
        all_s = [torch.empty_like(ex_s) for _ in range(world)]
        all_i = [torch.empty_like(ex_i) for _ in range(world)]
        dist.all_gather(all_s, ex_s)
        dist.all_gather(all_i, ex_i)
        ex_s, ex_i = merge_exact(all_s, all_i, k + margin)
    out = judge_topk(prod_s.cpu(), prod_i.cpu(), ex_s.cpu(), ex_i.cpu(), k)
    out["ok"] = out["index_mismatch_beyond_tol"] == 0 and out["max_score_err"] <= out["score_tol"]
    return out


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def device_randn_bf16(n: int, d: int, seed: int, device):
    import torch

    g = torch.Generator(device=device).manual_seed(seed)
    out = torch.empty((n, d), dtype=torch.bfloat16, device=device)
    for s in range(0, n, 1 << 20):
        e = min(n, s + (1 << 20))
        out[s:e] = torch.randn((e - s, d), generator=g, device=device).to(torch.bfloat16)
    return out


def timed_steps(fn, steps: int, warmup: int, dist_on: bool):
    """W untimed + K timed steps between barrier + synchronize; CUDA events; returns seconds/step
    (max over ranks) and the per-step event times of this rank."""
    import torch
    import torch.distributed as dist

    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist_on:
        dist.barrier()
        torch.cuda.synchronize()
    start = torch.cuda.Event(enable_timing=True)
    end = torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(steps):
        fn()
    end.record()
    torch.cuda.synchronize()
    if dist_on:
        dist.barrier()
        torch.cuda.synchronize()
    total = start.elapsed_time(end) / 1e3
    if dist_on:
        t = torch.tensor([total], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total = float(t.item())
    return total / steps


def _hbm(algo_bytes: float, sec: float, peaks: dict) -> dict:
    gbs = algo_bytes / sec / 1e9
    return {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"]}


def bench_preprocess(peaks: dict, steps: int, warmup: int, world: int = 1, rank: int = 0) -> dict:
    """Config 3a on EVERY rank (batch-sharded, no collective — each rank normalises its own batch with
    its own batch statistics, which is what the reference does per predict_step): 4096 uint8
    512x512x3 tiles per GPU -> normalised NCHW (no resize at the default max_side_length=640),
    -> 256x256 (max_side_length=256, exact 2x box path), -> 384x384 (max_side_length=384, the generic
    bilinear path) and 2048x2048 images cut into 512x512 patches.  `tiles_per_s` is the aggregate over
    all ranks (weak scaling), `roofline` is per GPU."""
    import torch

    from imagescry_b200.image.transforms import preprocess_patches, preprocess_tiles

    dist_on = world > 1
    out: dict = {}
    B, H, W = 4096, 512, 512
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    tiles = torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8, device="cuda", generator=g)
    nin = tiles.numel()
    cases = [
        ("nhwc_u8_to_nchw_f32", dict(layout="nhwc", out_dtype=torch.float32, output_hw=None), 2 * nin + 4 * nin),
        ("nhwc_u8_to_nchw_bf16", dict(layout="nhwc", out_dtype=torch.bfloat16, output_hw=None), 2 * nin + 2 * nin),
        ("nhwc_u8_resize256_f32", dict(layout="nhwc", out_dtype=torch.float32, output_hw=(256, 256)), 2 * nin + 4 * (nin // 4)),
        ("nhwc_u8_resize384_f32_generic_bilinear", dict(layout="nhwc", out_dtype=torch.float32, output_hw=(384, 384)),
         2 * nin + 4 * (B * 3 * 384 * 384)),
    ]
    for name, kw, algo_bytes in cases:
        fn = lambda: preprocess_tiles(tiles, min_value=-3, max_value=3, **kw)  # noqa: E731
        sec = timed_steps(fn, steps, warmup, dist_on)
        out[name] = {"tiles_per_s": world * B / sec, "ms": sec * 1e3, "algorithmic_bytes": algo_bytes,
                     "roofline": _hbm(algo_bytes, sec, peaks)}
    # patch tiling: the same bytes viewed as 256 images of 2048 x 2048, cut into 16 512 x 512 patches each
    big = tiles.view(B // 16, 2048, 2048, 3)
    sec = timed_steps(lambda: preprocess_patches(big, 512, min_value=-3, max_value=3), steps, warmup, dist_on)
    out["nhwc_u8_2048px_images_to_512px_patches_f32"] = {
        "tiles_per_s": world * B / sec, "ms": sec * 1e3, "algorithmic_bytes": 6 * nin, "roofline": _hbm(6 * nin, sec, peaks),
        "note": "256 images of 2048x2048x3 -> 4096 patches of 512x512 (stride 512), windows addressed inside the kernels' reads",
    }
    # planar (ImageBatch) input, the reference's own layout
    planar = tiles.permute(0, 3, 1, 2).contiguous()
    del tiles, big
    sec = timed_steps(lambda: preprocess_tiles(planar, min_value=-3, max_value=3), steps, warmup, dist_on)
    out["nchw_u8_to_nchw_f32"] = {"tiles_per_s": world * B / sec, "ms": sec * 1e3, "algorithmic_bytes": 6 * nin,
                                  "roofline": _hbm(6 * nin, sec, peaks)}
    out["batch"] = (f"{B} tiles uint8 {H}x{W}x3 per GPU x {world} GPU(s), batch statistics computed per rank "
                    "(stats pass + apply pass); tiles_per_s aggregate, roofline per GPU")
    out["scaling"] = "weak"
    del planar
    torch.cuda.empty_cache()
    return out


def synthetic_pca(E: int, k: int, gen):
    import torch

    from imagescry_b200.models.decomposition import PCA

    comps = torch.linalg.qr(torch.randn((E, k), generator=gen, device="cuda"))[0]
    pca = PCA(num_features=E, num_components=k).cuda()
    pca.feature_means.data = torch.randn((1, E), generator=gen, device="cuda") * 0.01
    pca.component_vectors.data = comps.contiguous()
    pca._fitted.data = torch.tensor(True, device="cuda")
    pca._num_features.data = torch.tensor(E, device="cuda")
    pca._num_components.data = torch.tensor(k, device="cuda")
    pca.packed_weights()
    return pca


def bench_project(peaks: dict, steps: int, warmup: int, world: int = 1, rank: int = 0) -> dict:
    """Config 3b on every rank (batch-sharded, PCA weights replicated, no collective):
    4096 x 1280 x 16 x 16 fp32 feature map per GPU -> L2-normalise -> project to 256-d."""
    import torch

    from imagescry_b200.models.embedding import l2_normalize_cells

    dist_on = world > 1
    B, E, h, w, k = 4096, 1280, 16, 16, 256
    g = torch.Generator(device="cuda").manual_seed(7 + rank)
    fmap = torch.empty((B, E, h, w), dtype=torch.float32, device="cuda")
    for s in range(0, B, 256):
        fmap[s:s + 256] = torch.randn((256, E, h, w), generator=g, device="cuda").abs_()
    pca = synthetic_pca(E, k, torch.Generator(device="cuda").manual_seed(7))
    out = {}
    for name, pool, algo in (
        ("per_cell", None, fmap.numel() * 4 + B * h * w * k * 4),
        ("mean_pooled", "mean", fmap.numel() * 4 + B * k * 4),
    ):
        sec = timed_steps(lambda: pca.project_feature_map(fmap, pool=pool), steps, warmup, dist_on)
        out[name] = {"cells_per_s": world * B * h * w / sec, "tiles_per_s": world * B / sec, "ms": sec * 1e3,
                     "algorithmic_bytes": algo, "roofline": _hbm(algo, sec, peaks)}
        if pool is None:
            # fp32-class accuracy costs three bf16 tensor passes (hi.hi + lo.hi + hi.lo): the tensor
            # roofline of the issued FLOPs sits above the HBM one for this kernel
            tf = 3 * 2.0 * B * h * w * E * k / sec / 1e12
            peak_sus = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
            out[name]["tensor_roofline"] = {
                "bound": "tensor", "achieved": tf, "peak": peak_sus, "unit": "TFLOP/s", "frac": tf / peak_sus,
                "note": "issued bf16 FLOPs (3 passes of 2*cells*1280*256) / sustained cuBLAS bf16 peak",
            }
    # opt-in single-pass mode (precision="fp16"): HBM-bound instead of tensor-bound
    sec = timed_steps(lambda: pca.project_feature_map(fmap, precision="fp16"), steps, warmup, dist_on)
    algo = fmap.numel() * 4 + B * h * w * k * 4
    out["per_cell_fp16_single_pass"] = {
        "cells_per_s": world * B * h * w / sec, "tiles_per_s": world * B / sec, "ms": sec * 1e3, "algorithmic_bytes": algo,
        "roofline": _hbm(algo, sec, peaks),
        "note": "one fp16 tensor pass; ~1e-5 of a row's norm vs ~1e-6 for the default three-pass bf16 split",
    }
    # the stand-alone F.normalize(x, dim=1) of EmbeddingModule.predict_step (embedding.py:74); the
    # output buffer is as large as the map, so this leg runs on the first 2048 images
    half = fmap[:2048]
    sec = timed_steps(lambda: l2_normalize_cells(half), steps, warmup, dist_on)
    algo = half.numel() * 8
    out["l2_normalize_cells"] = {"cells_per_s": world * 2048 * h * w / sec, "ms": sec * 1e3, "algorithmic_bytes": algo,
                                 "roofline": _hbm(algo, sec, peaks), "batch": f"2048x{E}x{h}x{w} fp32 in and out"}
    out["batch"] = f"feature map {B}x{E}x{h}x{w} fp32 per GPU x {world} GPU(s) -> {k}-d; rates aggregate, roofline per GPU"
    out["scaling"] = "weak"
    del fmap, half
    torch.cuda.empty_cache()
    return out


def bench_pca_fit(peaks: dict) -> dict:
    """SURVEY.md 8f.2: PCA.fit of a 65 536 x 1280 fp32 sample (decomposition.py:94-148): fp64 column
    means + tcgen05 SYRK covariance (isx_pca_moments), then the 1280 x 1280 eigh (torch library)."""
    import torch

    from imagescry_b200.models.decomposition import PCA

    n, F = 65536, 1280
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.randn((n, F), generator=g, device="cuda") * torch.linspace(3.0, 0.1, F, device="cuda") + 0.5
    pca = PCA(min_num_components=256, max_num_components=256).cuda()
    sec_m = timed_steps(lambda: pca._moments(x), 5, 2, False)
    sec_f = timed_steps(lambda: pca.fit(x), 2, 1, False)
    flops = 3 * 2.0 * n * F * F * (30.0 / 50.0)  # three passes over the 30 of 50 tiles that touch the upper triangle
    launches = (n + 5 * 1024 - 1) // (5 * 1024)
    out = {
        "sample": f"{n}x{F} fp32", "moments_ms": sec_m * 1e3, "fit_ms_incl_eigh": sec_f * 1e3,
        "moments_algorithmic_bytes": n * F * 4 * 2, "syrk_issued_tflops": flops / sec_m / 1e12,
        "bound": "latency",
        "note": (f"moments = fp64 column means (one read of x) + {launches} x (centre/split/transpose 5120 rows + tcgen05 SYRK "
                 "launch): one TMEM accumulation covers at most 1024 rows (the tensor core's fp32 accumulate truncates), so the "
                 "work is many short launches — latency-bound, not an HBM or tensor roofline; the fp64 eigh of the 1280x1280 "
                 "covariance (torch / cuSOLVER) is 94 % of the fit"),
    }
    del x
    torch.cuda.empty_cache()
    return out


def cpu_stage_baselines() -> dict:
    """BASELINE.md §4: the reference's torch-CPU path for stages 1 and 2 on the box's host cores, at the
    down-scaled sizes it names (B = 256 tiles; 65 536 rows), best of 3 after one warm-up."""
    import torch

    from oracle import torch_port as TP

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    out: dict = {"cores": cores, "kind": "port", "timing": "perf_counter, 1 warm-up, best of 3"}

    def best(fn):
        fn()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        return min(ts)

    g = torch.Generator().manual_seed(1234)
    tiles = torch.randint(0, 256, (256, 3, 512, 512), dtype=torch.uint8, generator=g)
    with torch.inference_mode():
        t = best(lambda: TP.preprocess(tiles, 640))
        out["preprocess_no_resize"] = {"tiles_per_s": 256 / t, "seconds": t, "sample": "256 tiles 3x512x512 u8 (of config 3's 4096), normalise + clip"}
        t = best(lambda: TP.preprocess(tiles, 256))
        out["preprocess_resize256"] = {"tiles_per_s": 256 / t, "seconds": t, "sample": "256 tiles, bilinear 512->256 + normalise + clip"}
        del tiles
        fmap = torch.randn((256, 1280, 16, 16), generator=g).abs_()
        comps = torch.linalg.qr(torch.randn((1280, 256), generator=g))[0]
        means = torch.randn((1, 1280), generator=g) * 0.01
        t = best(lambda: TP.l2_project(fmap, means, comps))
        out["l2_project_per_cell"] = {"cells_per_s": 65536 / t, "tiles_per_s": 256 / t, "seconds": t,
                                      "sample": "65 536 cells (256x1280x16x16 fp32 map) -> F.normalize + permute + (x - mean) @ W, 256-d"}
        t = best(lambda: TP.l2_project(fmap, means, comps, pool="mean"))
        out["l2_project_mean_pooled"] = {"tiles_per_s": 256 / t, "seconds": t, "sample": "same map, spatial mean then projection"}
        x = torch.randn((4096, 1280), generator=g)
        t0 = time.perf_counter()
        xc = x - x.mean(dim=0, keepdim=True)
        torch.linalg.svd(xc, full_matrices=False)
        out["pca_fit"] = {"seconds": time.perf_counter() - t0, "sample": "4096x1280 fp32, centre + reduced SVD (the reference takes the full SVD)"}
    out["extrapolation"] = "rates are per-item and linear in the batch: config 3's 4096 tiles take 16x the 256-tile time"
    return out


def bench_sift(world: int, rank: int, peaks: dict, tiles_per_gpu: int = 8192) -> dict:
    """BASELINE.json config 5 scaled to `tiles_per_gpu` tiles on every GPU (weak scaling; the full
    1 M tiles are backbone-bound minutes): HWC uint8 256x256 tiles -> stage 1 -> EfficientNetV2-S
    features (torchvision module, NOT owned: reported only) -> L2 + mean pool + PCA projection to
    256-d (PCA fitted on the GPU from rank 0's first batch, broadcast) -> row-sharded bf16 store ->
    all-pairs k=10 graph over ALL ranks' rows.  Per-stage device times (CUDA events, max over ranks)."""
    import torch
    import torch.distributed as dist

    from imagescry_b200.models.decomposition import PCA
    from imagescry_b200.models.embedding import EfficientNetEmbedder
    from imagescry_b200.search import EmbeddingStore, ShardedEmbeddingStore

    dist_on = world > 1
    n_tiles, bs, k_comp = tiles_per_gpu, 512, 256
    torch.manual_seed(1234)
    model = EfficientNetEmbedder(backbone_size="s").cuda().eval()
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    tiles = torch.randint(0, 256, (n_tiles, 256, 256, 3), dtype=torch.uint8, device="cuda", generator=g)

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    t_pre = t_bb = t_proj = 0.0
    pca = None
    rows = []
    with torch.inference_mode():
        for s0 in range(0, n_tiles, bs):
            batch = tiles[s0:s0 + bs]
            e0 = ev()
            x = model.preprocess_hwc(batch)
            e1 = ev()
            fmap = model(x)
            e2 = ev()
            if pca is None:
                # fit on the L2-normalised cells of the first batch (reference: PCA.fit on flat vectors)
                cells = model_cells(fmap)
                pca = PCA(min_num_components=k_comp, max_num_components=k_comp).cuda().fit(cells)
                if dist_on:  # one model for all ranks
                    for t in (pca.feature_means, pca.component_vectors):
                        buf = t.data.contiguous()
                        dist.broadcast(buf, src=0)
                        t.data = buf
                pca.packed_weights()
                e2 = ev()
            rows.append(pca.project_feature_map(fmap, pool="mean"))
            e3 = ev()
            torch.cuda.synchronize()
            if s0 > 0:  # first batch = warm-up (cuDNN autotune, PCA fit)
                t_pre += e0.elapsed_time(e1)
                t_bb += e1.elapsed_time(e2)
                t_proj += e2.elapsed_time(e3)
        emb = torch.cat(rows)
        total = n_tiles * world
        if dist_on:
            build = lambda: ShardedEmbeddingStore(emb, total_rows=total)  # noqa: E731
        else:
            build = lambda: EmbeddingStore(emb)  # noqa: E731
        build().knn_graph(10)  # warm-up
        torch.cuda.synchronize()
        if dist_on:
            dist.barrier()
        e0 = ev()
        store = build()
        scores, idx = store.knn_graph(10)  # k nearest OTHER rows of every row
        e1 = ev()
        torch.cuda.synchronize()
        t_search = e0.elapsed_time(e1)
    timed = n_tiles - bs
    times = torch.tensor([t_pre, t_bb, t_proj, t_search], dtype=torch.float64, device="cuda")
    if dist_on:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    t_pre, t_bb, t_proj, t_search = times.tolist()
    self_left = float((idx == torch.arange(idx.shape[0], device="cuda").reshape(-1, 1)).float().mean())
    out = {
        "workload": f"{total} uint8 256x256x3 HWC tiles ({n_tiles} per GPU x {world}), batch {bs}, EfficientNetV2-S weights=None "
                    "seed 1234 (fp32), pooled PCA-256, all-pairs k=10 over all ranks' rows",
        "preprocess_tiles_per_s": world * timed / (t_pre / 1e3), "backbone_img_per_s_not_owned": world * timed / (t_bb / 1e3),
        "pool_project_tiles_per_s": world * timed / (t_proj / 1e3), "graph_rows_per_s": total / (t_search / 1e3),
        "ms": {"preprocess": t_pre, "backbone": t_bb, "pool_project": t_proj, "store_build_and_all_pairs": t_search},
        "self_matches_left": self_left, "scaling": "weak",
    }
    del tiles, model, store
    torch.cuda.empty_cache()
    return out


def model_cells(fmap):
    from imagescry_b200.models.embedding import l2_normalize_cells

    return l2_normalize_cells(fmap).permute(0, 2, 3, 1).reshape(-1, fmap.shape[1])


def cpu_config1_sample(n_tiles: int = 96) -> dict:
    """BASELINE.json config 1 (the reference's own CPU-runnable case) on a bounded sample: `n_tiles`
    synthetic 256x256 tiles -> reference preprocess -> EfficientNetV2-S features (torchvision, CPU) ->
    L2 + mean pool -> k=10 cosine search over a 10 000 x 1280 store, per-stage wall time on all host
    threads, with the linear extrapolation to 10 000 tiles."""
    import torch
    from torchvision.models import efficientnet_v2_s

    from oracle import torch_port as TP

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(1234)
    net = efficientnet_v2_s(weights=None).features.eval()
    g = torch.Generator().manual_seed(1234)
    tiles = torch.randint(0, 256, (n_tiles, 3, 256, 256), dtype=torch.uint8, generator=g)
    with torch.inference_mode():
        t0 = time.perf_counter()
        x = TP.preprocess(tiles, 640)
        t1 = time.perf_counter()
        fm = torch.cat([net(x[i:i + 32]) for i in range(0, n_tiles, 32)])
        t2 = time.perf_counter()
        emb = torch.nn.functional.normalize(fm, p=2, dim=1).mean(dim=(2, 3))
        t3 = time.perf_counter()
        store = TP.prepare_store(torch.randn((10_000, 1280), generator=g))
        t4 = time.perf_counter()
        TP.cosine_knn(store, emb, 10, prepared=True)
        t5 = time.perf_counter()
    per = {"preprocess": (t1 - t0) / n_tiles, "backbone_not_owned": (t2 - t1) / n_tiles, "l2_pool": (t3 - t2) / n_tiles,
           "knn_k10_over_10k": (t5 - t4) / n_tiles}
    return {
        "cores": cores, "kind": "port", "sample": f"{n_tiles} of config 1's 10 000 tiles (256x256x3 u8), batch 32 through the backbone",
        "seconds_per_tile": per, "extrapolated_seconds_10k_tiles": {k2: v * 10_000 for k2, v in per.items()},
        "tiles_per_s_end_to_end": 1.0 / sum(per.values()),
    }


def run_b200(args) -> None:
    import torch
    import torch.distributed as dist

    from imagescry_b200 import _lib
    from imagescry_b200.search import EmbeddingStore, ShardedEmbeddingStore, row_rnorm, shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit(f"--gpus {args.gpus} needs torchrun with {args.gpus} processes (WORLD_SIZE=1 here)")
        args.gpus = world
    assert torch.cuda.is_available(), "bench.py needs CUDA devices; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist_on = world > 1
    real_stdout = None
    if dist_on:
        # stdout carries exactly one JSON line.  NCCL prints its version banner (and, at NCCL_DEBUG=INFO,
        # its whole log) with printf on fd 1; NCCL_DEBUG is left as the caller set it and fd 1 is pointed
        # at stderr for the run instead — the JSON line is written to the saved descriptor at the end
        sys.stdout.flush()
        real_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    peaks = load_peaks()

    # ---- workload: 1 M x 1280 store (row-sharded when world > 1), 10 k queries replicated
    b, e = shard_range(N_STORE, world, rank)
    if world == 1:
        store_rows = device_randn_bf16(N_STORE, D, 1234, dev)
    else:
        # every rank generates the same global stream chunk by chunk and keeps its rows
        g = torch.Generator(device=dev).manual_seed(1234)
        store_rows = torch.empty((e - b, D), dtype=torch.bfloat16, device=dev)
        for s in range(0, N_STORE, 1 << 20):
            ee = min(N_STORE, s + (1 << 20))
            chunk = torch.randn((ee - s, D), generator=g, device=dev).to(torch.bfloat16)
            lo, hi = max(s, b), min(ee, e)
            if lo < hi:
                store_rows[lo - b:hi - b] = chunk[lo - s:hi - s]
            del chunk
    queries = device_randn_bf16(Q, D, 4321, dev)
    sharded = None
    if dist_on:
        sharded = ShardedEmbeddingStore(store_rows, total_rows=N_STORE)
        store = sharded.local
    else:
        store = EmbeddingStore(store_rows, index_base=b)
    torch.cuda.synchronize()

    lib = _lib.load()
    ws_bytes = int(lib.isx_knn_workspace_bytes(len(store), Q, D, K))
    ws = torch.empty(max(ws_bytes, 256), dtype=torch.uint8, device=dev)
    scores = torch.empty((Q, K), dtype=torch.float32, device=dev)
    idx = torch.empty((Q, K), dtype=torch.int32, device=dev)
    ev_pairs: list = []

    def search_local(q_dev, record: bool):
        """N = 1: row norms of the queries + the fused search, straight through the C ABI"""
        qr = row_rnorm(q_dev)
        stream = torch.cuda.current_stream(dev)
        if record:
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record(stream)
        rc = lib.isx_knn_search_ex(
            store.embeddings.data_ptr(), store.rnorm.data_ptr(), len(store), q_dev.data_ptr(), qr.data_ptr(), Q, D, K,
            store.index_base, 0, 0, scores.data_ptr(), idx.data_ptr(), ws.data_ptr(), ws.numel(), stream.cuda_stream,
        )
        _lib.check(rc, "isx_knn_search_ex")
        if record:
            e1.record(stream)
            ev_pairs.append((e0, e1))

    last_out: list = [None]  # (scores, indices) of the latest step: what --dump-outputs writes

    def step(q_dev=queries, record=True):
        if dist_on:
            # row norms + fused search whose finalising pass stores the packed records into every rank's
            # gather buffer over NVLink (symmetric memory) + device barrier + merge; NCCL all-gather of
            # the packed records where peer mapping is unavailable
            sharded._event_sink = ev_pairs if record else None
            last_out[0] = sharded.search_raw(q_dev, K)
        else:
            search_local(q_dev, record)
            last_out[0] = (scores, idx)
        return last_out[0]

    # kernels of mine per step: row_rnorm + search + finalise(+scatter) (+ cross-rank merge); the two
    # memsets, the symmetric-memory barrier / NCCL all-gather are library work
    launches = 3 + (1 if dist_on else 0)

    # Pre-heat: the part is power-limited (sw_power_cap); its SM clock settles about two seconds into a
    # tensor-bound loop.  The timed steps start from that steady state, so `roofline.frac` against the
    # SUSTAINED cuBLAS peak (measured the same way) compares like with like.
    t_heat = time.perf_counter()
    heat_steps = 0
    while time.perf_counter() - t_heat < args.preheat:
        for _ in range(8):
            step(record=False)
        torch.cuda.synchronize()
        heat_steps += 8
    with ClockSampler(local_rank) as clocks:
        # warm-up happens inside timed_steps; events recorded during warm-up are dropped below
        sec = timed_steps(step, args.steps, args.warmup, dist_on)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last_out[0])
    kernel_ms = [e0.elapsed_time(e1) for e0, e1 in ev_pairs[args.warmup:]]
    clock_summary = clocks.summary()
    value = Q / sec
    k_ms = sum(kernel_ms) / max(1, len(kernel_ms))
    flops = 2.0 * Q * len(store) * D
    achieved = flops / (k_ms * 1e-3) / 1e12
    peak_sus = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
    roofline = {
        "bound": "tensor", "achieved": achieved, "peak": peak_sus, "unit": "TFLOP/s", "frac": achieved / peak_sus,
        # dram bytes of one launch from the committed `ncu --set full` capture of the N = 1 workload; a
        # 1/N shard is a different launch, so there is no figure at N > 1
        "traffic": load_traffic() if world == 1 else None,
        "kernel": "knn_search_kernel<32, 2> (CTA pairs; + 2 memsets and the finalising topk_merge pass, <1 % of the interval)",
        "kernel_ms": k_ms, "flops_per_launch": flops,
        "peak_source": f"{peaks['_source']} bf16_tflops_sustained (kernel timed inside a step loop that was pre-heated for {args.preheat:.1f} s)",
        "frac_of_burst_peak": achieved / peaks["bf16_tflops"],
    }

    if dist_on:
        # the ranks meet at a barrier every step, so a step lasts as long as its slowest rank's kernel:
        # report every rank's own average kernel time next to rank 0's
        t = torch.tensor([k_ms], dtype=torch.float64, device=dev)
        allk = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allk, t)
        roofline["kernel_ms_per_rank"] = [float(x.item()) for x in allk]
        roofline["note"] = ("ms_per_step - kernel_ms = query norms + barrier + merge + the wait for the slowest rank of every step "
                            "(per-rank kernel times differ with each GPU's clock)")

    # ---- e2e: pinned host queries -> H2D -> search -> D2H of the result, through the public API
    q_host = queries.cpu().pin_memory()
    out_s_host = torch.empty((Q, K), dtype=torch.float32).pin_memory()
    out_i_host = torch.empty((Q, K), dtype=torch.int32).pin_memory()
    q_stage = torch.empty_like(queries)

    def e2e_step():
        if dist_on:
            # every rank uploads 1/N of the query rows; one all-gather over NVLink replicates them
            sharded._event_sink = None
            s, i = sharded.search_raw(sharded.replicate_queries(q_host), K)
        else:
            q_stage.copy_(q_host, non_blocking=True)
            s, i = store.search_raw(q_stage, K)
        out_s_host.copy_(s, non_blocking=True)
        out_i_host.copy_(i, non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the caller holds the answer before the next step

    sec_e2e = timed_steps(e2e_step, args.steps, args.warmup, dist_on)

    # the serving form of the same thing: a stream of host batches through search_host_batches — the H2D
    # of step i + 1 and the D2H of step i ride a copy stream (DMA engines) beside the search of the
    # neighbouring step.  Every step still uploads its queries from pinned host memory and downloads
    # its result inside the timed region; every rank uploads the whole batch over its own PCIe link.
    from imagescry_b200.search import HostBatchSearch

    streamer = HostBatchSearch(sharded if dist_on else store, K)

    def e2e_stream(nsteps: int):
        if dist_on:
            sharded._event_sink = None
        got = 0
        for s_h, _ in streamer.run(q_host for _ in range(nsteps)):
            got += s_h.shape[0]
        assert got == nsteps * Q

    e2e_stream(args.warmup)
    torch.cuda.synchronize()
    if dist_on:
        dist.barrier()
        torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    e2e_stream(args.steps)  # returns once the last result is in host memory
    ev1.record()
    torch.cuda.synchronize()
    if dist_on:
        dist.barrier()
        torch.cuda.synchronize()
    sec_stream = ev0.elapsed_time(ev1) / 1e3 / args.steps
    if dist_on:
        t = torch.tensor([sec_stream], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec_stream = float(t.item())
    e2e = {
        "value": Q / sec_stream, "unit": UNIT, "h2d_bytes_per_step": q_host.numel() * 2,
        "d2h_bytes_per_step": out_s_host.numel() * 4 + out_i_host.numel() * 4, "ms_per_step": sec_stream * 1e3,
        "api": ("HostBatchSearch(store, k).run(host_batches): pinned host query batches streamed through "
                + ("ShardedEmbeddingStore.search_raw (every rank uploads the batch over its own PCIe link; gather of packed "
                   f"records: {sharded.gather_path})" if dist_on else "EmbeddingStore.search_raw")
                + "; H2D of step i+1 and D2H of step i on a copy stream beside the search; bytes are per rank"),
        "one_batch_at_a_time": {
            "value": Q / sec_e2e, "ms_per_step": sec_e2e * 1e3,
            "api": ("ShardedEmbeddingStore.search_raw: each rank uploads 1/N of the pinned host queries, all-gather over NVLink, "
                    "local search, gather + merge, D2H, host sync" if dist_on
                    else "EmbeddingStore.search_raw: H2D, search, D2H, host sync — strictly sequential, nothing overlapped"),
        },
    }

    # ---- verification (untimed): sampled queries against an exact fp32 brute force over every shard
    verify: dict = {}
    if not args.no_verify:
        for kk in (10, 100):
            if dist_on:
                fn = lambda pick, kk=kk: sharded.search_raw(queries[pick], kk)  # noqa: E731
            else:
                fn = lambda pick, kk=kk: store.search_raw(queries[pick], kk)  # noqa: E731
            verify[f"k{kk}"] = verify_search(fn, store.embeddings, b, queries, kk, dist_on)
        verify["what"] = ("64 evenly spaced queries through the product path (N > 1: local search + one all-gather + merge) against an exact "
                          "fp32 torch brute force over every rank's shard (candidates all-gathered, exact (score desc, index asc) sort)")
        verify["checked"] = sum(v["checked"] for v in verify.values() if isinstance(v, dict))
        verify["index_mismatch_beyond_tol"] = sum(v["index_mismatch_beyond_tol"] for v in verify.values() if isinstance(v, dict))
        verify["max_score_err"] = max(v["max_score_err"] for v in verify.values() if isinstance(v, dict))

    extra: dict = {}
    cpu_baseline = None
    if not args.no_extra:
        st = max(3, min(args.steps, 5))
        for name, fn in (("preprocess", lambda: bench_preprocess(peaks, st, 3, world, rank)),
                         ("project", lambda: bench_project(peaks, st, 3, world, rank))):
            try:
                extra[name] = fn()
            except Exception as ex:  # keep the primary line even if an extra stage fails
                if dist_on:
                    raise  # a rank that drops out of a collective-free leg would desynchronise the barriers
                extra[name] = {"error": repr(ex)}
        if world == 1:
            for name, fn in (("search_other_shapes", lambda: bench_search_shapes(store, queries, peaks)),
                             ("pca_fit", lambda: bench_pca_fit(peaks))):
                try:
                    extra[name] = fn()
                except Exception as ex:
                    extra[name] = {"error": repr(ex)}
        try:
            extra["sift"] = bench_sift(world, rank, peaks)
        except Exception as ex:
            if dist_on:
                raise
            extra["sift"] = {"error": repr(ex)}
        if world == 1 and rank == 0:
            try:
                cpu_baseline = cpu_knn_sample(store.embeddings.cpu(), q_host, seconds_target=12.0)
                cpu_baseline["stages"] = cpu_stage_baselines()
                cpu_baseline["config1_sample"] = cpu_config1_sample()
            except Exception as ex:
                cpu_baseline = cpu_baseline or {}
                cpu_baseline["error"] = repr(ex)
    if dist_on and not args.no_extra:
        del store_rows
        extra["sharded_graph"] = bench_sharded_graph(world, rank, dev, peaks, verify=not args.no_verify)
        extra["sharded_large"] = bench_sharded_large(args, world, rank, dev, peaks)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic", "config": dict(workload_config(world), preheat_s=args.preheat, preheat_steps=heat_steps),
            "clocks": clock_summary, "e2e": e2e, "gpu_launches": launches * args.steps, "roofline": roofline,
        }
        if dist_on:
            line["config"]["gather"] = sharded.gather_path
        if verify:
            line["verify"] = verify
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        if extra:
            line["extra"] = extra
        if real_stdout is not None:
            sys.stdout.flush()
            os.write(real_stdout, (json.dumps(line) + "\n").encode())
        else:
            print(json.dumps(line), flush=True)
    if dist_on:
        dist.barrier()
        dist.destroy_process_group()


def bench_search_shapes(store, queries, peaks: dict) -> dict:
    """The other search shapes BASELINE.json names, on one GPU: k = 100 over the metric's store
    (config 4's k) and k = 10 over a 1 M x 256 store (config 5's dimensionality)."""
    import torch

    from imagescry_b200.search import EmbeddingStore

    peak_sus = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])

    def run(st, q, k):
        sec = timed_steps(lambda: st.search_raw(q, k), 5, 3, False)
        tf = 2.0 * q.shape[0] * len(st) * st.dim / sec / 1e12
        return {"queries_per_s": q.shape[0] / sec, "ms": sec * 1e3, "tflops": tf,
                "frac_of_sustained_bf16_peak": tf / peak_sus, "frac_of_burst_bf16_peak": tf / peaks["bf16_tflops"]}

    out = {"k100_d1280": run(store, queries, 100)}
    dev = queries.device
    st256 = EmbeddingStore(device_randn_bf16(N_STORE, 256, 1234, dev))
    out["k10_d256"] = run(st256, device_randn_bf16(Q, 256, 4321, dev), 10)
    # the single-GPU all-pairs graph of a 131 072-row slice (queries = store rows, self skipped in the kernel)
    sub = EmbeddingStore(st256.embeddings[:131072])
    sec = timed_steps(lambda: sub.knn_graph(10), 3, 1, False)
    tf = 2.0 * 131072 * 131072 * 256 / sec / 1e12
    out["graph_k10_d256_131072_rows"] = {"rows_per_s": 131072 / sec, "ms": sec * 1e3, "tflops": tf, "frac_of_sustained_bf16_peak": tf / peak_sus}
    out["store"] = f"{N_STORE} rows, {Q} queries"
    del st256, sub
    torch.cuda.empty_cache()
    return out


def bench_sharded_graph(world: int, rank: int, dev, peaks: dict, rows: int = 1_000_000, dim: int = 256, k: int = 10,
                        verify: bool = True) -> dict:
    """The search step of BASELINE.json config 5: all-pairs k=10 similarity graph over a 1 M x 256
    bf16 store row-sharded over the ranks.  Queries are sharded too (a rank answers for its own rows);
    the store shards are all-gathered once over NVLink and searched by one fused kernel launch with
    the running lists in its workspace; no partial result is gathered or merged; the finished lists
    are all-gathered once so that every rank returns the whole graph."""
    import torch

    from imagescry_b200.search import ShardedEmbeddingStore, shard_range

    b, e = shard_range(rows, world, rank)
    g = torch.Generator(device=dev).manual_seed(77)
    full = torch.randn((rows, dim), generator=g, device=dev).to(torch.bfloat16)  # identical on every rank
    local = full[b:e].contiguous()
    del full
    store = ShardedEmbeddingStore(local, total_rows=rows)
    sec = timed_steps(lambda: store.knn_graph(k), 3, 1, True)
    # per GPU: its N / G query rows against all N store rows
    tf = 2.0 * (e - b) * rows * dim / sec / 1e12
    peak_sus = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
    out = {
        "workload": f"all-pairs k={k} graph, {rows}x{dim} bf16 store row-sharded over {world} GPUs; queries sharded, store all-gathered once, "
                    "one fused search per rank, finished lists all-gathered",
        "graph_rows_per_s": rows / sec, "ms": sec * 1e3, "per_gpu_tflops_incl_collectives": tf,
        "frac_of_sustained_bf16_peak": tf / peak_sus, "frac_of_burst_bf16_peak": tf / peaks["bf16_tflops"],
    }
    if verify:
        gs, gi = store.knn_graph(k)
        fn = lambda pick: (gs[pick], gi[pick])  # noqa: E731
        # queries = the store's own rows: every rank needs the sampled rows' vectors -> rebuild them
        gfull = torch.Generator(device=dev).manual_seed(77)
        allrows = torch.randn((rows, dim), generator=gfull, device=dev).to(torch.bfloat16)
        out["verify"] = verify_search(fn, local, b, allrows, k, True, exclude_self_base=0)
        del allrows, gs, gi
    del store, local
    torch.cuda.empty_cache()
    return out


def bench_sharded_large(args, world: int, rank: int, dev, peaks: dict) -> dict:
    """BASELINE.json config 4: a 100 M x 1280 bf16 store row-sharded over the GPUs (100 M / N rows each
    when that fits 70 % of the device memory — 32 GB per GPU at N = 8 —, else as many as fit; override
    with --large-rows-per-gpu), 10 k queries, k = 10 and k = 100, one all-gather of packed records +
    merge; 64 sampled queries verified against an exact fp32 brute force over all shards."""
    import torch
    import torch.distributed as dist

    from imagescry_b200.search import ShardedEmbeddingStore

    rows = args.large_rows_per_gpu
    if rows <= 0:
        free, total_mem = torch.cuda.mem_get_info(dev)
        fit = int(min(0.70 * total_mem, free - (12 << 30)) // (D * 2))
        rows = max(1 << 20, min(100_000_000 // world, fit))
    t = torch.tensor([rows], dtype=torch.int64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)  # every rank must hold the same number of rows
    rows = int(t.item())
    g = torch.Generator(device=dev).manual_seed(99 + rank)
    # allocate and fill; if ANY rank cannot (another tenant's memory, fragmentation) every rank halves the
    # shard and tries again — a rank that raised alone would leave the others hanging in a collective
    while True:
        ok = 1
        local = None
        try:
            local = torch.empty((rows, D), dtype=torch.bfloat16, device=dev)
            for s in range(0, rows, 1 << 20):
                ee = min(rows, s + (1 << 20))
                local[s:ee] = torch.randn((ee - s, D), generator=g, device=dev).to(torch.bfloat16)
        except torch.OutOfMemoryError:
            ok = 0
            local = None
            torch.cuda.empty_cache()
        t = torch.tensor([ok], dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        if int(t.item()) == 1:
            break
        local = None
        torch.cuda.empty_cache()
        rows //= 2
        if rows < (1 << 20):
            return {"error": "could not allocate a shard of even 1 Mi rows on every rank"}
    store = ShardedEmbeddingStore(local, index_base=rank * rows)
    queries = device_randn_bf16(Q, D, 4321, dev)
    out = {"workload": f"{rows * world}x{D} bf16 store row-sharded over {world} GPUs ({rows} rows = {rows * D * 2 / 2**30:.1f} GiB each), {Q} queries",
           "store_rows": rows * world, "full_config4_size": rows * world >= 100_000_000}
    peak_sus = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
    for kk in (10, 100):
        sec = timed_steps(lambda: store.search_raw(queries, kk), 2, 1, True)
        tf = 2.0 * Q * rows * D / sec / 1e12
        out[f"k{kk}"] = {
            "queries_per_s": Q / sec, "ms_per_step": sec * 1e3, "per_gpu_tflops_incl_collective": tf,
            "frac_of_sustained_bf16_peak": tf / peak_sus, "frac_of_burst_bf16_peak": tf / peaks["bf16_tflops"],
        }
        if not args.no_verify:
            out[f"k{kk}"]["verify"] = verify_search(lambda pick, kk=kk: store.search_raw(queries[pick], kk), local, rank * rows,
                                                    queries, kk, True)
    if not args.no_verify:
        out["verify"] = {"checked": sum(out[f"k{kk}"]["verify"]["checked"] for kk in (10, 100)),
                         "index_mismatch_beyond_tol": sum(out[f"k{kk}"]["verify"]["index_mismatch_beyond_tol"] for kk in (10, 100)),
                         "max_score_err": max(out[f"k{kk}"]["verify"]["max_score_err"] for kk in (10, 100))}
    del store, local
    torch.cuda.empty_cache()
    dist.barrier()
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--no-extra", action="store_true", help="skip the stage-1/2 and CPU-baseline legs")
    ap.add_argument("--no-verify", action="store_true", help="skip the untimed sampled brute-force verification")
    ap.add_argument("--preheat", type=float, default=2.0, help="seconds of untimed steps before the timed loop (clock steady state)")
    ap.add_argument("--large-rows-per-gpu", type=int, default=0, help="config-4 leg at N > 1: rows per GPU (0 = 100 M / N when it fits)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the metric's result of the last timed step (scores, indices) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        # the reference arm sizes its query sample from a timing calibration: not the same inputs every run
        ap.error("--dump-outputs needs --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
