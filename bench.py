#!/usr/bin/env python
"""Headline benchmark: user-item pairs scored / second (fused top-k) at rank 50.

    python bench.py --gpus N --steps K --warmup W            (our arm)
    python bench.py --impl reference --gpus N --steps K ...  (the reference's own CPU path, oracle/_ref)

Workload (BASELINE.json configs[1], "C2"): synthetic 1M users x 100K items, ~0.1% nnz (1e8 interactions, Zipf item
popularity, log-normal user degrees), SVDModel rank 50, filter_seen, top-10, every user scored against every item.
One *step* = one full pass of the hot path on device-resident inputs: SpMM E = P.V, fused score + mask + top-k, merge.

What the JSON line carries besides the contract keys:
  value                 default product path (norm-bound early termination of the sweep ON -- exact, see DESIGN.md 3.1)
  value_full_sweep      same step with the early termination OFF: every pair goes through the tensor-core filter
  value_flat_norms      same step on random orthonormal item factors (flat norms: nothing can be cut, many candidates)
  roofline              the kernel that dominates the default step (measured live, CUDA events)
  rooflines             {"spmm": HBM-bound, "fused_full_sweep": tensor-bound} -- hardware-utilisation numbers; the fused
                        kernel's fraction is taken on the FULL sweep so that skipped work never inflates it
  e2e                   B200SVDModel.get_recommendations() from the (user, item, feedback) triplets a Polara data model
                        hands over, in pinned host memory: H2D + device ingest + scoring + D2H inside the timed region
  e2e_csr_fastpath      same call fed with a ready-made pinned host CSR (3x fewer bytes over PCIe)
  build_e2e_s           build() from host triplets: H2D + ingest + transpose + panels + randomized SVD
  cpu_baseline          the reference (polara) itself on this box's host cores: default knobs and tuned knobs

--dump-outputs DIR writes what the last timed step returned to DIR/<name>.npy (see dump_outputs): the top-k lists for
c2, the factors and core of the CoFFee build for c4, the lists of every rank of the sweep for c5.  The inputs are seeded
and identical from run to run, so two builds can be compared output for output.  bench.py runs on the library build()
made, refuses one that is missing or older than its sources, and writes nothing into the tree (no compile, no bytecode).

Multi-GPU (weak scaling in items, SURVEY.md 8e): every rank owns a 100K-item shard of the item factors (total items =
N x 100K); user embeddings are computed row-sharded (each rank its block of users) and all-gathered; per-shard top-k
candidates are exchanged with ONE all-to-all by user range and merged on the owning rank.  value = all (user, item)
pairs of the job / max-over-ranks step time.  After the timed loop rank 0 re-scores its users unsharded and compares
("selfcheck").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
DUMP_BYTES = 64 << 20


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--users", type=int, default=1_000_000)
    ap.add_argument("--items", type=int, default=100_000, help="items PER GPU (weak scaling)")
    ap.add_argument("--nnz", type=int, default=100_000_000)
    ap.add_argument("--rank", type=int, default=50)
    ap.add_argument("--topk", type=int, default=10)
    ap.add_argument("--kernel", default=None, choices=[None, "simt", "tcgen05"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="strong: --items is the TOTAL item count, split over the GPUs")
    ap.add_argument("--cpu-seconds", type=float, default=24.0, help="budget of the CPU-baseline sample")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-variants", action="store_true", help="skip value_full_sweep / value_flat_norms")
    ap.add_argument("--skip-build", action="store_true", help="random orthonormal factors instead of build()")
    ap.add_argument("--config", default="c2", choices=["c2", "c4", "c5"],
                    help="c2 (default; with --users/--items/--nnz/--rank/--gpus also C3's shape), c4 = CoFFee HOOI on a "
                         "1M x 50K x 5 tensor, c5 = ScaledSVD rank sweep on 5M x 500K (one build at rank 500)")
    ap.add_argument("--scale", type=float, default=1.0, help="c4/c5: shrink users, items and nnz by this factor")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


def require_built_library():
    """The numbers must be those of the current sources: a library that is missing or older than them is an error
    (build() makes it; bench.py compiles nothing, so that it can run from a read-only tree)."""
    from polara_b200 import _build
    if _build.needs_build():
        raise SystemExit("%s is missing or older than its sources: run build() first" % _build.LIB_PATH)


def dump_outputs(out_dir, arrays):
    """Writes every ``name -> array`` to ``out_dir/<name>.npy``: floating arrays in float64 when they are float64, else
    float32; integer arrays (item ids) in float32 when below 2**24, else float64 -- exact either way.  At most DUMP_BYTES
    in all: the budget is shared out smallest array first, and an array larger than its share is replaced by a fixed,
    seeded sample of its rows, whose row numbers go to ``<name>_rows.npy`` (float64)."""
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BYTES - 2 * 128 * len(arrays)          # .npy headers: 128 bytes for each of at most two files an array
    names = sorted(arrays, key=lambda k: arrays[k].size)
    for n, name in enumerate(names):
        a = np.asarray(arrays[name])
        if a.dtype == np.float64 or (a.dtype.kind in "iu" and a.size and np.abs(a).max() >= 2 ** 24):
            a = a.astype(np.float64)
        else:
            a = a.astype(np.float32)
        share = left // (len(names) - n)
        if a.nbytes > share:
            row_bytes = a[0].nbytes + 8
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], share // row_bytes, replace=False))
            a = a[rows]
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
            left -= rows.size * 8
        np.save(os.path.join(out_dir, name + ".npy"), a)
        left -= a.nbytes


# ------------------------------------------------------------------ data ------------
def synth_csr_torch(n_users, n_items, nnz_target, seed, device):
    """Zipf-popular items, log-normal degrees, ratings 1..5; built with torch on `device`
    (data generation is not part of any timed region).  Returns device CSR tensors."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    deg = torch.exp(torch.randn(n_users, generator=g, device=device))
    deg = torch.clamp((deg * (nnz_target / n_users / deg.mean())).round(), 1, max(1, n_items // 2)).to(torch.int64)
    w = 1.0 / torch.arange(1, n_items + 1, device=device, dtype=torch.float64)
    cdf = torch.cumsum(w, 0)
    cdf /= cdf[-1].clone()
    perm = torch.randperm(n_items, generator=g, device=device)
    rows = torch.repeat_interleave(torch.arange(n_users, device=device), deg)
    u = torch.rand(rows.shape[0], generator=g, device=device, dtype=torch.float64)
    cols = perm[torch.searchsorted(cdf, u).clamp_(max=n_items - 1)]
    key = torch.unique(rows * n_items + cols)          # sorted by (row, col), duplicates dropped
    rows = key // n_items
    cols = (key - rows * n_items).to(torch.int32)
    counts = torch.bincount(rows, minlength=n_users)
    indptr = torch.zeros(n_users + 1, dtype=torch.int64, device=device)
    indptr[1:] = torch.cumsum(counts, 0)
    vals = torch.randint(1, 6, (cols.shape[0],), generator=g, device=device).to(torch.float32)
    return indptr, cols, vals


def synth_triplets_host(n_users, n_items, nnz_target, seed, sample_users=50_000):
    """host-only data of the same shape for the reference arm (no GPU there): a seeded sample of users is generated
    with the numpy generator of polara_b200.synth and tiled over the user range (rows are statistically identical)."""
    from polara_b200.synth import popularity_csr
    su = min(n_users, sample_users)
    indptr, indices, values = popularity_csr(su, n_items, int(nnz_target * su / n_users), seed=seed)
    reps = -(-n_users // su)
    deg = np.diff(indptr)
    user = np.repeat(np.arange(su, dtype=np.int64), deg)
    users = np.concatenate([user + r * su for r in range(reps)])
    keep = users < n_users
    items = np.tile(indices.astype(np.int64), reps)[keep]
    fdbk = np.tile(values.astype(np.float64), reps)[keep]
    return users[keep], items, fdbk


def sample_clocks(stop, out):
    q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    while not stop.is_set():
        try:
            txt = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader,nounits", "-i",
                                  os.environ.get("LOCAL_RANK", "0")], capture_output=True, text=True, timeout=5).stdout
            out.append(txt.strip().split("\n")[0])
        except Exception:
            pass
        stop.wait(0.2)


def summarize_clocks(samples):
    sm, mx, reasons = [], [], set()
    for line in samples:
        p = [x.strip() for x in line.split(",")]
        if len(p) < 7:
            continue
        try:
            sm.append(float(p[0])); mx.append(float(p[1]))
        except ValueError:
            continue
        for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
            if v.lower().startswith("active"):
                reasons.add(name)
    if not sm:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
    return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons)}


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


# ------------------------------------------------------------- CPU baseline ---------
def reference_baseline(triplets, shape, v64, topk, budget_s):
    """The reference itself (polara, from oracle/_ref) on this box's host cores: SVDModel.get_recommendations()'s own
    chunk driver over the first chunks of users with the FULL test arrays in place (so each chunk pays what it pays in
    the full job, models.py:260-270), (i) library defaults (memory_hard_limit 1 GiB, no thread pool,
    polara/recommender/defaults.py:50-51) and (ii) tuned (larger chunks + max_test_workers), as BASELINE.md 2 promises.
    Falls back to the oracle port when the reference cannot be imported (kind says which)."""
    n_users, n_items = shape
    try:
        from oracle import ref_driver as rd
        rd.import_reference()
    except Exception as exc:                                  # noqa: BLE001
        return port_baseline(triplets, shape, v64, topk, budget_s, why=str(exc))
    host = rd.host_description()
    cores = host.get("cores") or os.cpu_count() or 1
    data = rd.StubData(shape, test=triplets)
    model = rd.make_svd_model(data, v64, topk=topk)
    old = rd.set_knobs(1)
    out = {}
    try:
        model.max_test_workers = None
        r0 = rd.time_reference_scoring(model, max_chunks=1)                      # warm-up (numpy/BLAS threads, page faults)
        per_chunk = max(r0["seconds"], 1e-3)
        n_chunks = int(max(1, min(20, (0.45 * budget_s) // per_chunk)))
        r1 = rd.time_reference_scoring(model, max_chunks=n_chunks)
        out["default"] = dict(value=r1["users"] * n_items / r1["seconds"], users=r1["users"], chunk_users=r1["chunk_users"],
                              chunks=r1["chunks"], seconds=r1["seconds"], memory_hard_limit_gib=1, max_test_workers=None)
        # tuned: bigger chunks, one worker thread per chunk; bounded by the memory the box really has
        try:
            import psutil
            avail = psutil.virtual_memory().available / 2 ** 30
        except Exception:                                     # noqa: BLE001
            avail = 64.0
        limit = 2.0
        workers = int(max(2, min(cores, 32, (0.35 * avail) // (limit * 2.5))))
        rd.set_knobs(limit)
        model.max_test_workers = workers
        est = per_chunk * (limit / 1.0) * 1.3                                    # one tuned chunk ~ limit x the default one
        if est < 0.5 * budget_s:
            r2 = rd.time_reference_scoring(model, max_chunks=workers)
            out["tuned"] = dict(value=r2["users"] * n_items / r2["seconds"], users=r2["users"], chunk_users=r2["chunk_users"],
                                chunks=r2["chunks"], seconds=r2["seconds"], memory_hard_limit_gib=limit,
                                max_test_workers=workers)
    finally:
        rd.set_knobs(old)
    best = max(out.values(), key=lambda d: d["value"])
    which = [k for k, v in out.items() if v is best][0]
    return {"value": best["value"], "unit": "pairs/s", "cores": cores, "kind": "reference",
            "sample": "polara SVDModel chunk driver (models.py:359-405) from %s, %s knobs: first %d chunks of %d users "
                      "(%d of %d users) with the full %d-triplet test arrays in place, %.1f s"
                      % (os.path.relpath(rd.reference_root(), ROOT), which, best["chunks"], best["chunk_users"],
                         best["users"], n_users, len(triplets[0]), best["seconds"]),
            "settings": out, "host": host}


def port_baseline(triplets, shape, v64, topk, budget_s, why=""):
    """oracle port of the chunk driver (used only when the reference itself cannot be imported)."""
    from oracle import polara_oracle as po
    import scipy.sparse as sps
    user, item, fdbk = triplets
    n_users, n_items = shape
    chunk = po.get_chunk_size((n_users, n_items), topk, 1, 1.0)
    bounds = po.range_division(n_users, chunk)
    cuts = np.searchsorted(user, bounds)
    t0 = time.perf_counter()
    done = n_chunks = 0
    for c, (a, b) in enumerate(zip(bounds[:-1], bounds[1:])):
        lo, hi = cuts[c], cuts[c + 1]
        u, i, f = user[lo:hi] - a, item[lo:hi], fdbk[lo:hi]
        p = sps.csr_matrix((f, (u, i)), shape=(b - a, n_items))
        scores = po.svd_slice_scores(p, v64)
        po.downvote_seen_items(scores, u, i)
        po.get_topk_elements(scores, topk)
        done += b - a
        n_chunks += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return {"value": done * n_items / dt, "unit": "pairs/s", "cores": os.cpu_count(), "kind": "port",
            "sample": "oracle port of the chunk driver (reference not importable: %s): %d chunks of %d users in %.1f s"
                      % (why[:80], n_chunks, chunk, dt)}


def timed(fn, steps, sync, barrier=None):
    """CUDA-event time of `steps` calls of fn (ms per call), bracketed by barrier + synchronize on both sides."""
    import torch
    if barrier:
        barrier()
    sync()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        fn()
    ev1.record()
    sync()
    if barrier:
        barrier()
    return ev0.elapsed_time(ev1) / steps


def run_c4(args):
    """BASELINE config C4: CoffeeModel HOOI on a user x item x feedback(5) tensor, 1M x 50K, nnz 5e7, core (60, 60, 4)
    (the reference cannot run r2 = 5 on 5 levels: ARPACK needs k < min(shape), lib/tensor.py:78-79).  One step = one HOOI
    iteration (three TTMs + three thin SVDs).  Roofline: the mode-0 TTM against its algorithmic bytes (SURVEY.md 8d)."""
    import torch
    from polara_b200.engine import get_engine
    from polara_b200.host import ArrayData
    from polara_b200.models import B200CoffeeModel
    require_built_library()
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    eng = get_engine(0)
    n_users, n_items, nnz_t = int(1_000_000 * args.scale), int(50_000 * args.scale), int(50_000_000 * args.scale)
    indptr_d, indices_d, values_d = synth_csr_torch(n_users, n_items, int(nnz_t * 1.15), 20260924, dev)
    user = torch.repeat_interleave(torch.arange(n_users, device=dev), torch.diff(indptr_d))
    idx = torch.stack([user, indices_d.to(torch.int64), (values_d - 1).to(torch.int64)], dim=1).cpu().numpy()
    nnz = idx.shape[0]
    shape = (n_users, n_items, 5)
    data = ArrayData(idx, np.ones(nnz), shape, fields=("userid", "itemid", "rating"), n_feedback=5)
    model = B200CoffeeModel(data)
    model.verbose = False
    model.mlrank = (60, 60, 4)
    model.seed = 0
    model.growth_tol = 0.0                         # run exactly num_iters iterations
    iters_w, iters_t = max(1, min(args.warmup, 2)), args.steps
    model.num_iters = iters_w
    model.build(); torch.cuda.synchronize()
    model.num_iters = iters_w + iters_t
    t0 = time.perf_counter(); model.build(); torch.cuda.synchronize(); t_all = time.perf_counter() - t0
    if args.dump_outputs:          # the build whose last iteration is the last timed step
        dump_outputs(args.dump_outputs, {k: model.factors[k] for k in ("userid", "itemid", "rating", "core")})
    model.num_iters = iters_w
    t0 = time.perf_counter(); model.build(); torch.cuda.synchronize(); t_w = time.perf_counter() - t0
    s_per_iter = (t_all - t_w) / iters_t
    # mode-0 TTM alone
    i0 = eng.upload(idx[:, 0].astype(np.int32)); i1 = eng.upload(idx[:, 1].astype(np.int32)); i2 = eng.upload(idx[:, 2].astype(np.int32))
    vals = eng.upload(np.ones(nnz, dtype=np.float32))
    seg, a1, a2, vv = eng.coo_group(i0, n_users, i1, i2, vals)
    r0, r1, r2 = model.mlrank
    u1 = eng.upload(model.factors["itemid"].astype(np.float32)); u2 = eng.upload(model.factors["rating"].astype(np.float32))
    ttm_ms = timed(lambda: eng.ttm(n_users, seg, a2, a1, vv, u2, r2, u1, r1), 5, torch.cuda.synchronize)
    ttm_bytes = nnz * 16.0 + 4.0 * (n_items * r1 + 5 * r2) + 4.0 * n_users * r1 * r2
    peaks = load_peaks(); peak_hbm = float(peaks.get("hbm_gbs", 6500.0))
    out = {"metric": "HOOI iterations per second (CoFFee build), core (60,60,4)", "value": 1.0 / s_per_iter, "unit": "iterations/s",
           "n_gpus": 1, "steps": iters_t, "warmup": iters_w, "ms_per_step": s_per_iter * 1e3, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32 (f64 Gram / eigen)", "data": "synthetic",
           "config": {"workload": "C4: CoffeeModel HOOI, %d x %d x 5 tensor, nnz %d, mlrank (60,60,4)" % (n_users, n_items, nnz)},
           "core_norm_trace": model.core_norm_trace,
           "roofline": {"bound": "hbm", "kernel": "ttm_kernel (mode 0: unfolded tensor x Khatri-Rao panel formed on the fly)",
                        "achieved": ttm_bytes / ttm_ms / 1e6, "peak": peak_hbm, "unit": "GB/s",
                        "frac": ttm_bytes / ttm_ms / 1e6 / peak_hbm, "traffic": None, "kernel_ms": ttm_ms,
                        "algorithmic_bytes_per_launch": ttm_bytes}}
    print(json.dumps(out))


def run_c5(args):
    """BASELINE config C5: ScaledSVD (col_scaling 0.4, EIGENREC) on 5M x 500K, nnz 5e8: ONE build at rank 500, then
    scoring at rank in {10, 50, 100, 200, 500} by rank truncation without rebuilding (models.py:819-832,
    pipelines.py:81-116).  Every rank runs the tcgen05 kernel (K-slab pipeline above rank 61)."""
    import torch
    import warnings
    from polara_b200.engine import DeviceCSR, get_engine
    from polara_b200.host import ArrayData
    from polara_b200.models import B200ScaledSVD
    from polara_b200 import dist as pdist
    require_built_library()
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    eng = get_engine(0)
    n_users, n_items, nnz_t = int(5_000_000 * args.scale), int(500_000 * args.scale), int(500_000_000 * args.scale)
    indptr_d, indices_d, values_d = synth_csr_torch(n_users, n_items, int(nnz_t * 1.12), 20260924, dev)
    nnz = int(indices_d.shape[0])
    shape = (n_users, n_items)
    data = ArrayData(np.zeros((1, 2), dtype=np.int64), np.ones(1), shape)
    data.train_csr = (indptr_d, indices_d, values_d.clone(), shape)      # the scaling works in place: P keeps the raw values
    model = B200ScaledSVD(data)
    model.verbose = False
    model.col_scaling = 0.4
    model.rank = 500
    torch.cuda.synchronize(); t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        model.build()
    torch.cuda.synchronize(); build_s = time.perf_counter() - t0
    p_dev = DeviceCSR(indptr_d, indices_d, values_d, shape)
    peaks = load_peaks(); peak_tf = float(peaks.get("bf16_tflops", 1590.0))
    pairs = float(n_users) * float(n_items)
    sweep = []
    lists = {}
    for rank in (500, 200, 100, 50, 10):
        model.rank = rank
        v_dev = model._device_factor("itemid")
        step = pdist.make_step(eng, p_dev, v_dev, rank, args.topk, None)
        step(); torch.cuda.synchronize()
        s0 = eng.stats()
        last = [None]

        def run_step():
            last[0] = step()
        ms = timed(run_step, args.steps, torch.cuda.synchronize)
        s1 = eng.stats()
        if args.dump_outputs:       # copied now: the next steps may reuse the engine's result buffers
            lists["ids_rank%d" % rank] = last[0].cpu().numpy()
        del last
        eng.set_prune(False)
        ms_full = timed(step, 1, torch.cuda.synchronize)
        fused_full = eng.last_score_kernel_ms()
        eng.set_prune(True)
        sweep.append({"rank": rank, "value": pairs / (ms * 1e-3), "ms_per_step": ms, "ms_per_step_full_sweep": ms_full,
                      "fused_full_sweep_ms": fused_full, "fused_full_sweep_frac": 2.0 * pairs * rank / (fused_full * 1e-3) / 1e12 / peak_tf,
                      "executed_share": (s1[5] - s0[5]) / max(s1[6] - s0[6], 1),
                      "on_tensor_cores": (s1[6] - s0[6]) > 0})
        del step, v_dev
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, lists)
    best50 = [x for x in sweep if x["rank"] == 50][0]
    out = {"metric": "user-item pairs scored/sec (fused top-k) at rank 50", "value": best50["value"], "unit": "pairs/s", "n_gpus": 1,
           "steps": args.steps, "warmup": 1, "ms_per_step": best50["ms_per_step"], "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32 (bf16 tensor-core filter, exact fp32 rescoring)", "data": "synthetic",
           "config": {"workload": "C5: ScaledSVD (col_scaling 0.4) %d x %d, nnz %d: one build at rank 500, scoring at the "
                                  "truncated ranks" % (n_users, n_items, nnz)},
           "build_s": build_s, "build_detail": model.last_timings, "rank_sweep": sweep}
    print(json.dumps(out))


def main():
    args = parse_args()
    if args.impl == "b200" and args.config == "c4":
        return run_c4(args)
    if args.impl == "b200" and args.config == "c5":
        return run_c5(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n_gpus = args.gpus
    if world > 1 and world != n_gpus:
        raise SystemExit("--gpus must equal WORLD_SIZE under torchrun")
    n_items_total = args.items * n_gpus if args.scaling == "weak" else args.items
    workload = "C2: synthetic %dM users x %dK items%s, nnz %.0e, SVD rank %d, filter_seen, top-%d" % (
        args.users // 1_000_000, args.items // 1000, "/GPU" if args.scaling == "weak" else " in total", args.nnz,
        args.rank, args.topk)
    base = {"metric": "user-item pairs scored/sec (fused top-k) at rank %d" % args.rank, "unit": "pairs/s",
            "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "data": "synthetic",
            "config": {"workload": workload, "users": args.users, "items_total": n_items_total,
                       "items_per_gpu": n_items_total // n_gpus, "nnz": args.nnz, "rank": args.rank, "topk": args.topk,
                       "parallelism": "item-shard x%d" % n_gpus,
                       "l2_policy": "inputs (P, E, lists > 1 GB) larger than the 126 MB L2"}}

    if args.impl == "reference":
        if rank != 0:
            return
        run_reference(args, base, n_items_total)
        return

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    require_built_library()
    from polara_b200.engine import DeviceCSR, get_engine
    from polara_b200.host import ArrayData
    from polara_b200.models import B200SVDModel
    from polara_b200 import dist as pdist
    eng = get_engine(local_rank)
    if args.kernel:
        eng.set_score_kernel(args.kernel)
    sync = torch.cuda.synchronize
    barrier = dist.barrier if world > 1 else None

    # ---------------- synthetic inputs (same seed on every rank) ----------------------
    indptr_d, indices_d, values_d = synth_csr_torch(args.users, n_items_total, args.nnz, 20260924, dev)
    nnz = int(indices_d.shape[0])
    if nnz < 0.97 * args.nnz:      # duplicates of popular items were dropped: draw more to land on the target
        del indptr_d, indices_d, values_d
        indptr_d, indices_d, values_d = synth_csr_torch(args.users, n_items_total,
                                                        int(args.nnz * (args.nnz / nnz) ** 1.15), 20260924, dev)
        nnz = int(indices_d.shape[0])
    need_host = not (args.no_e2e and (args.no_cpu_baseline or n_gpus > 1))
    if need_host:
        indptr_h = indptr_d.cpu().pin_memory(); indices_h = indices_d.cpu().pin_memory(); values_h = values_d.cpu().pin_memory()
    shape = (args.users, n_items_total)
    want_coo = world == 1 and not args.no_e2e
    if want_coo:
        # what a Polara data model hands over (data.py:794-862): intp index arrays, float64 feedback -- in pinned memory
        user_h = torch.repeat_interleave(torch.arange(args.users, device=dev), torch.diff(indptr_d)).cpu().pin_memory()
        item_h = indices_d.to(torch.int64).cpu().pin_memory()
        fdbk_h = values_d.to(torch.float64).cpu().pin_memory()
        idx_h = torch.stack([user_h, item_h], dim=1).pin_memory()
        data = ArrayData(idx_h.numpy(), fdbk_h.numpy(), shape, user_h.numpy(), item_h.numpy(), fdbk_h.numpy(), shape)
    else:
        data = ArrayData(np.zeros((1, 2), dtype=np.int64), np.ones(1), shape)
        # build() from a ready CSR: pinned host arrays when an e2e leg needs them anyway, else the device arrays (big shapes)
        data.train_csr = (indptr_h, indices_h, values_h, shape) if need_host else (indptr_d, indices_d, values_d, shape)
    model = B200SVDModel(data)
    model.verbose = False
    model.rank = args.rank
    model.topk = args.topk
    model.score_kernel = args.kernel
    sharder = pdist.ItemShard(rank, world, n_items_total) if world > 1 else None
    model.shard = sharder          # world > 1: row-sharded build, item-sharded scoring

    # ---------------- build() (timed once; not part of the step) ----------------------
    import warnings
    sync()
    t0 = time.perf_counter()
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        if args.skip_build:
            q = np.linalg.qr(np.random.default_rng(0).standard_normal((n_items_total, args.rank)))[0]
            model.factors = {"userid": None, "itemid": q, "singular_values": np.ones(args.rank)}
            model._is_ready = True
        else:
            model.build()
    sync()
    build_s = time.perf_counter() - t0
    build_warnings = [str(w.message)[:160] for w in caught]

    # ---------------- device-resident step --------------------------------------------
    p_dev = DeviceCSR(indptr_d, indices_d, values_d, shape)
    v_dev = model._device_factor("itemid")
    step = pdist.make_step(eng, p_dev, v_dev, args.rank, args.topk, sharder)
    for _ in range(args.warmup):
        ids = step()
    sync()
    stats0 = eng.stats()
    clocks, stop = [], threading.Event()
    th = threading.Thread(target=sample_clocks, args=(stop, clocks), daemon=True)
    if barrier:
        barrier()
    sync()
    th.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        ids = step()
    ev1.record()
    sync()
    if barrier:
        barrier()
    stop.set(); th.join()
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs:
        # copied now: later variant steps may reuse the engine's result buffers
        last = ids.cpu().numpy() if world == 1 else pdist.gather_lists(ids.cpu().numpy(), sharder, args.users, dev)
        if rank == 0:
            dump_outputs(args.dump_outputs, {"ids": last})
    stats1 = eng.stats()
    launches = stats1[0] - stats0[0]
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / args.steps
    pairs = float(args.users) * float(n_items_total)
    value = pairs / (ms_per_step * 1e-3)
    swept, swept_full = stats1[5] - stats0[5], stats1[6] - stats0[6]

    # ---------------- per-phase table (one extra, untimed-loop step with event marks) --
    phases = []
    pstep = pdist.make_step(eng, p_dev, v_dev, args.rank, args.topk, sharder, phases=phases)
    pstep(); sync()
    phase_ms = {b[0]: a[1].elapsed_time(b[1]) for a, b in zip(phases[:-1], phases[1:])}
    fused_ms_default = eng.last_score_kernel_ms()

    # ---------------- rooflines --------------------------------------------------------
    peaks = load_peaks()
    peak_tf = float(peaks.get("bf16_tflops", 1590.0))
    peak_hbm = float(peaks.get("hbm_gbs", 6500.0))
    peak_src = "measured (MEASURED_PEAKS.json, burst)" if peaks else "fallback (B200_PROFILING.md)"
    items_local = n_items_total // world
    # (a) SpMM E = P V alone (this rank's rows when sharded): algorithmic bytes of SURVEY.md 8d
    p_sp = pdist.row_block(eng, p_dev, sharder) if sharder is not None else p_dev
    ld = v_dev.shape[1]
    p_sp = eng.block_columns(p_sp, eng.panel_cols_for(p_sp.shape[1], ld))      # as the step does (panel-major when V > L2)
    e_buf = eng.empty((p_sp.shape[0], ld))
    spmm_ms = timed(lambda: eng.spmm(p_sp, v_dev, ell=ld, out=e_buf), max(3, args.steps), sync)
    spmm_bytes = 8.0 * p_sp.nnz + 8.0 * (p_sp.shape[0] + 1) + 4.0 * ld * (n_items_total + p_sp.shape[0])
    roof_spmm = {"bound": "hbm", "kernel": "%s (E = P V, ell %d, %d column panel%s)" % (
                     # pb_spmm_panel: 128-bit gathers for <= 64 and 97..128 columns (per 128-column group), 32-bit for 65..96
                     "spmm_window4_kernel" if (ld % 128 == 0 or (ld % 128) <= 64 or (ld % 128) > 96) else "spmm_window_kernel",
                     ld, p_sp.n_panels, "" if p_sp.n_panels == 1 else "s"), "achieved": spmm_bytes / spmm_ms / 1e6,
                 "peak": peak_hbm, "unit": "GB/s", "frac": spmm_bytes / spmm_ms / 1e6 / peak_hbm, "traffic": None,
                 "kernel_ms": spmm_ms, "algorithmic_bytes_per_launch": spmm_bytes,
                 "l2_gather_tb_s": p_sp.nnz * ld * 4.0 / spmm_ms / 1e9, "peak_source": peak_src}
    # (b) fused kernel on the FULL sweep (early termination off): hardware utilisation of the tensor-core pipeline
    out = dict(base)
    roof_fused = None
    if not args.no_variants:
        eng.set_prune(False)
        full_step = pdist.make_step(eng, p_dev, v_dev, args.rank, args.topk, sharder)
        full_step(); sync()
        ms_full = timed(full_step, max(2, args.steps // 2), sync, barrier)
        score_ms = pdist.time_score_kernel(eng, p_dev, v_dev, args.rank, args.topk, sharder, reps=max(3, args.steps))
        eng.set_prune(True)
        if world > 1:
            t = torch.tensor([ms_full], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms_full = float(t.item())
        flops = 2.0 * args.users * items_local * args.rank
        achieved_tf = flops / (score_ms * 1e-3) / 1e12
        roof_fused = {"bound": "tensor", "kernel": "score_topk_tc_kernel, full sweep (pb200_set_prune(0))",
                      "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                      "traffic": None, "kernel_ms": score_ms, "peak_source": peak_src,
                      "algorithmic_flops_per_launch": flops}
        out["value_full_sweep"] = pairs / (ms_full * 1e-3)
        out["ms_per_step_full_sweep"] = ms_full
    # the default step's dominant kernel
    fused_share = fused_ms_default / max(ms_per_step, 1e-9)
    spmm_share = phase_ms.get("spmm", phase_ms.get("spmm_rows+allgather", 0.0)) / max(ms_per_step, 1e-9)
    flops = 2.0 * args.users * items_local * args.rank
    roof_default_fused = {"bound": "tensor", "kernel": "score_topk_tc_kernel (default: sweep cut by the norm bound; "
                          "%.1f%% of the tile products executed)" % (100.0 * swept / max(swept_full, 1)),
                          "achieved": flops * (swept / max(swept_full, 1)) / (fused_ms_default * 1e-3) / 1e12, "peak": peak_tf,
                          "unit": "TFLOP/s", "kernel_ms": fused_ms_default, "peak_source": peak_src, "traffic": None,
                          "note": "achieved counts only the EXECUTED tile products (algorithmic flops x executed share)"}
    roof_default_fused["frac"] = roof_default_fused["achieved"] / peak_tf
    # DRAM traffic per launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed `ncu --set full` captures of
    # exactly this command (profiles/spmm_step_r2_ncu.txt, score_topk_tc_r2_ncu.txt, score_topk_tc_pruned_r2_ncu.txt): only
    # for the configuration they were taken on (C2 defaults, one GPU, tcgen05 kernel); null for anything else.
    if (world == 1 and (args.users, args.items, args.nnz, args.rank, args.topk) == (1_000_000, 100_000, 100_000_000, 50, 10)
            and (args.kernel or "tcgen05") == "tcgen05"):
        src = "ncu --set full, C2, one B200 (profiles/*_r2_ncu.txt)"
        roof_spmm.update(traffic=840.361472e6 + 241.191680e6, traffic_source=src)
        if roof_fused is not None:
            roof_fused.update(traffic=284.461824e6 + 137.639424e6, traffic_source=src)
        roof_default_fused.update(traffic=282.235904e6 + 129.994752e6, traffic_source=src)
    roofline = roof_spmm if spmm_share >= fused_share else roof_default_fused
    roofline = dict(roofline, share_of_step=max(spmm_share, fused_share))
    out.update({"value": value, "ms_per_step": ms_per_step,
                "dtype": "f32 (bf16 tensor-core filter, exact fp32 rescoring)" if (args.kernel or "tcgen05") == "tcgen05" else "f32",
                "gpu_launches": int(launches), "roofline": roofline,
                "rooflines": {"spmm": roof_spmm, "fused_full_sweep": roof_fused, "fused_default": roof_default_fused},
                "phase_ms": phase_ms, "sweep": {"tile_products_executed": int(swept), "tile_products_full": int(swept_full),
                                                "executed_share": swept / max(swept_full, 1)},
                "clocks": summarize_clocks(clocks), "build_s": build_s, "build_detail": model.last_timings,
                "build_warnings": build_warnings, "nnz_actual": nnz,
                "build_route": "host triplets (to_coo) -> device ingest" if want_coo else
                               ("pinned host CSR" if need_host else "device CSR") + (" (row-sharded)" if world > 1 else "")})
    if want_coo:
        out["build_e2e_s"] = build_s

    # ---------------- flat item norms: the unfriendly input -----------------------------
    if not args.no_variants and world == 1:
        q = np.linalg.qr(np.random.default_rng(0).standard_normal((n_items_total, args.rank)))[0].astype(np.float32)
        vf = eng.zeros((n_items_total, ld)); vf[:, :args.rank].copy_(torch.from_numpy(q))
        flat_step = pdist.make_step(eng, p_dev, vf, args.rank, args.topk, None)
        flat_step(); sync()
        s0 = eng.stats()
        ms_flat = timed(flat_step, max(2, args.steps // 2), sync)
        s1 = eng.stats()
        out["value_flat_norms"] = pairs / (ms_flat * 1e-3)
        out["flat_norms"] = {"ms_per_step": ms_flat, "fused_kernel_ms": eng.last_score_kernel_ms(),
                             "rescored_per_user": (s1[1] - s0[1]) / max(2, args.steps // 2) / args.users,
                             "executed_share": (s1[5] - s0[5]) / max(s1[6] - s0[6], 1)}
        del vf, flat_step

    # ---------------- N > 1: the merged lists must equal an unsharded scoring ------------
    if world > 1:
        # same user embeddings as the step (bit-identical: the row-sharded SpMM + all-gather is deterministic), scored
        # UNSHARDED against the whole V on this rank: checks sharding, candidate exchange, merge and seen fill-up exactly.
        # (E itself is checked against scipy in the tests; re-deriving it from a differently sliced matrix would change the
        # summation order of rows that straddle nnz windows and flip near-ties.)
        lo, hi = sharder.user_range(args.users)
        n_chk = min(hi - lo, 20_000)
        p_blk = pdist.row_block(eng, p_dev, sharder)
        p_blk = eng.block_columns(p_blk, eng.panel_cols_for(p_blk.shape[1], ld))
        e_all = pdist.gather_embeddings(eng, p_blk, v_dev, sharder, args.users)
        a0 = int(indptr_d[lo])
        a1 = int(indptr_d[lo + n_chk])
        ip = indptr_d[lo:lo + n_chk + 1].clone()
        eng.shift_i64(ip, -a0)
        ref_ids = eng.score_topk(e_all[lo:lo + n_chk], v_dev, args.rank, args.topk, seen=(ip, indices_d[a0:a1]))
        n_bad = int((ref_ids != ids[:n_chk]).any(dim=1).sum().item())
        flag = torch.tensor([n_bad], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.SUM)
        out["selfcheck"] = "ok" if int(flag.item()) == 0 else "MISMATCH in %d user rows" % int(flag.item())
        out["selfcheck_detail"] = ("every rank: the first %d users it owns, scored unsharded against all %d items from the "
                                   "step's own embeddings == the exchanged + merged lists" % (n_chk, n_items_total))
        del e_all, p_blk

    # ---------------- end to end through the model API (host buffers) -----------------
    if not args.no_e2e:
        def run_e2e(fn, reps):
            recs = None
            for _ in range(3):
                recs = fn()          # holding the previous result, like the timed loop: both pinned result blocks get cached
            sync()
            if barrier:
                barrier()
            t0 = time.perf_counter()
            for _ in range(reps):
                recs = fn()
            sync()
            dt = (time.perf_counter() - t0) / reps
            if world > 1:
                t = torch.tensor([dt], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            return dt, recs
        reps = max(2, min(args.steps, 5))
        d2h = args.users * args.topk * 8
        if want_coo:
            data.test_csr = None
            dt, recs = run_e2e(model.get_recommendations, reps)
            h2d = user_h.numel() * 8 + item_h.numel() * 8 + fdbk_h.numel() * 8
            out["e2e"] = {"value": pairs / dt, "unit": "pairs/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                          "s_per_step": dt, "call": "B200SVDModel.get_recommendations() from the pinned host (user, item, "
                          "feedback) triplets of test_to_coo: H2D, device COO->CSR ingest, SpMM, fused scoring, D2H"}
            if os.environ.get("BENCH_DEBUG"):
                model.profile_phases = True
                model.get_recommendations()
                print("e2e (triplets) phases", model.last_score_timings, file=sys.stderr)
                model.profile_phases = False
        data.test_csr = ((indptr_h, indices_h, values_h), shape)
        dt, recs = run_e2e(model.get_recommendations, reps)
        # whole-job bytes: every rank copies the row pointers, the nnz arrays cross PCIe once (sliced by rank)
        h2d = indptr_h.numel() * 8 * world + indices_h.numel() * 4 + values_h.numel() * 4
        fast = {"value": pairs / dt, "unit": "pairs/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "s_per_step": dt, "call": "B200SVDModel.get_recommendations() on a ready-made pinned host CSR (data.test_csr)"}
        if want_coo:
            out["e2e_csr_fastpath"] = fast
        else:
            out["e2e"] = fast
        if os.environ.get("BENCH_DEBUG"):
            model.profile_phases = True
            model.get_recommendations()
            print("rank", rank, "e2e (csr) phases", model.last_score_timings, file=sys.stderr)

    # ---------------- CPU baseline on this box's host cores (rank 0, N=1) -------------
    if rank == 0 and n_gpus == 1 and not args.no_cpu_baseline:
        v64 = model.factors["itemid"].astype(np.float64)
        if want_coo:
            trip = (user_h.numpy(), item_h.numpy(), fdbk_h.numpy())
        else:
            from oracle.ref_driver import csr_to_test_triplets
            trip = csr_to_test_triplets(indptr_h.numpy(), indices_h.numpy(), values_h.numpy())
        out["cpu_baseline"] = reference_baseline(trip, shape, v64, args.topk, args.cpu_seconds)
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def run_reference(args, base, n_items_total):
    """Reference arm: the UNMODIFIED reference (polara, installed into oracle/_ref by build()) scores a bounded sample of the
    workload per step through its own chunk driver on the host cores; no GPU, none of our code on the path (the data
    generator is numpy; the data stub replays test_to_coo)."""
    from oracle import ref_driver as rd
    rng = np.random.default_rng(0)
    shape = (args.users, n_items_total)
    trip = synth_triplets_host(args.users, n_items_total, args.nnz, seed=20260924)
    v64 = np.linalg.qr(rng.standard_normal((n_items_total, args.rank)))[0]
    try:
        rd.import_reference()
    except Exception as exc:                                  # noqa: BLE001
        cb = port_baseline(trip, shape, v64, args.topk, 20.0, why=str(exc))
        out = dict(base)
        out.update({"impl": "reference", "value": cb["value"], "ms_per_step": None, "dtype": "f64", "cpu_baseline": cb,
                    "e2e": {"value": cb["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                    "gpu_launches": 0})
        print(json.dumps(out))
        return
    host = rd.host_description()
    cores = host.get("cores") or os.cpu_count() or 1
    data = rd.StubData(shape, test=trip)
    model = rd.make_svd_model(data, v64, topk=args.topk)
    # pick the better of the two settings once (warm-up), then time K steps with it
    settings = {}
    rd.set_knobs(1)
    model.max_test_workers = None
    r = rd.time_reference_scoring(model, max_chunks=2)
    settings["default"] = dict(value=r["users"] * n_items_total / r["seconds"], chunk_users=r["chunk_users"],
                               memory_hard_limit_gib=1, max_test_workers=None, chunks_per_step=4)
    try:
        import psutil
        avail = psutil.virtual_memory().available / 2 ** 30
    except Exception:                                         # noqa: BLE001
        avail = 64.0
    limit = 2.0
    workers = int(max(2, min(cores, 16, (0.35 * avail) // (limit * 2.5))))     # 16 chunks in flight keep a step near 15 s
    rd.set_knobs(limit)
    model.max_test_workers = workers
    r = rd.time_reference_scoring(model, max_chunks=workers)
    settings["tuned"] = dict(value=r["users"] * n_items_total / r["seconds"], chunk_users=r["chunk_users"],
                             memory_hard_limit_gib=limit, max_test_workers=workers, chunks_per_step=workers)
    which = max(settings, key=lambda k: settings[k]["value"])
    cfg = settings[which]
    rd.set_knobs(cfg["memory_hard_limit_gib"])
    model.max_test_workers = cfg["max_test_workers"]

    def one_step():
        return rd.time_reference_scoring(model, max_chunks=cfg["chunks_per_step"])
    for _ in range(max(0, min(args.warmup, 1))):
        one_step()
    t0 = time.perf_counter()
    users_done = 0
    for _ in range(args.steps):
        users_done += one_step()["users"]
    dt = (time.perf_counter() - t0) / args.steps
    per_step_users = users_done / args.steps
    value = per_step_users * n_items_total / dt
    out = dict(base)
    out.update({"impl": "reference", "value": value, "ms_per_step": dt * 1e3, "dtype": "f64",
                "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": "reference",
                                 "sample": "polara SVDModel chunk driver (oracle/_ref, unmodified), %s knobs: %d users "
                                           "(%d chunks of %d) x %d items per step, full-size test arrays in place"
                                           % (which, per_step_users, cfg["chunks_per_step"], cfg["chunk_users"], n_items_total),
                                 "settings": settings, "host": host},
                "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0})
    print(json.dumps(out))


if __name__ == "__main__":
    main()
