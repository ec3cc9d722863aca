"""ProbabilisticMF build and scoring at the C2 shape (1 M users x 100 K items, 1e8 interactions, bench.py's generator
and seed), rank 10.  Prints one JSON line.

    python bench_pmf.py [--steps K] [--warmup W] [--epochs E] [--strata B] [--sweep 256,512,...]
    python bench_pmf.py --impl reference        # one epoch of the reference's numba sweep on one CPU core

``--impl b200`` needs a CUDA device and fails without one.  ``epoch_ms`` is the median host time of the timed epochs
(each pb200_sgd_epoch call ends in a stream synchronise); ``build_e2e_s`` is ``B200ProbabilisticMF.build()`` from host
triplets for ``--epochs`` epochs (ingest, plan, initial factors, epochs, factors back to the host); ``pairs_per_s`` is
``get_recommendations()`` for every tenth user over all items.  The SGD epoch is latency-bound (each update is a chain
of dependent loads and a warp reduction), so its bytes/s over the HBM peak is small by nature; it is reported as a
fraction of the bandwidth bound, nothing more.  Writes nothing into the tree.
"""
import sys

sys.dont_write_bytecode = True

import argparse  # noqa: E402
import json  # noqa: E402
import os  # noqa: E402
import subprocess  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12           # HGX B200 data sheet, one GPU


def bytes_per_update(rank):
    """algorithmic bytes of one update: the (user, item, value) triplet plus a read and a write of both fp64 rows."""
    return 12 + 4 * 8 * rank


def device_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=20).stdout.strip().split("\n")[0]
        name, power, clock = (x.strip() for x in out.split(","))
        return dict(device=name, power_limit=power, max_sm_clock=clock)
    except Exception as exc:                       # reported, not hidden
        return dict(device=None, power_limit=None, nvidia_smi_error=repr(exc))


def load_balance(block_ptr, strata):
    """per sub-epoch: the largest block against the mean block; the sum of the largest blocks is the critical path of an
    epoch in updates."""
    sizes = np.diff(block_ptr).reshape(strata, strata)          # [s, b]
    mx, mean = sizes.max(axis=1), sizes.mean(axis=1)
    ratio = mx / np.maximum(mean, 1e-30)
    return dict(max_over_mean_median=float(np.median(ratio)), max_over_mean_worst=float(ratio.max()),
                critical_path_updates=int(mx.sum()), nnz=int(sizes.sum()))


def run_epochs(eng, plan, rank, n_epochs, seed=1):
    import torch
    rs = np.random.RandomState(seed)
    n_users, n_items = plan.shape
    ld = (rank + 31) // 32 * 32
    p = eng.zeros((n_users, ld), torch.float64)
    q = eng.zeros((n_items, ld), torch.float64)
    p[:, :rank].copy_(torch.from_numpy(rs.normal(scale=0.1, size=(n_users, rank))))
    q[:, :rank].copy_(torch.from_numpy(rs.normal(scale=0.1, size=(n_items, rank))))
    times, errs = [], []
    for _ in range(n_epochs):
        t = time.perf_counter()
        errs.append(eng.sgd_epoch(plan, p, q, rank, 0.005, 0.5))
        times.append(time.perf_counter() - t)
    return times, [float(np.sqrt(e / plan.nnz)) for e in errs]


def bench_b200(args):
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_pmf.py --impl b200 needs a CUDA device")
    from polara_b200 import _build
    if _build.needs_build():
        raise SystemExit("libpolara_b200.so is missing or older than its sources: run build() first")
    from bench import synth_csr_torch
    from polara_b200.engine import DeviceCSR, get_engine
    from polara_b200.host import ArrayData
    from polara_b200.models import DEFAULT_SGD_STRATA, B200ProbabilisticMF
    torch.cuda.set_device(0)
    eng = get_engine(0)
    info = device_info()
    strata = DEFAULT_SGD_STRATA if args.strata is None else args.strata
    indptr, indices, values = synth_csr_torch(args.users, args.items, args.nnz, 20260924, eng.device)
    a = DeviceCSR(indptr, indices, values, (args.users, args.items))
    nnz = a.nnz
    out = dict(config="pmf_c2", users=args.users, items=args.items, nnz=nnz, rank=args.rank, sgd_strata=strata, **info)
    sweep = []
    for b in ([int(x) for x in args.sweep.split(",")] if args.sweep else []):
        t = time.perf_counter()
        plan = eng.sgd_plan(a, b)
        plan_s = time.perf_counter() - t
        times, rmse = run_epochs(eng, plan, args.rank, args.sweep_epochs)
        sweep.append(dict(sgd_strata=b, plan_s=round(plan_s, 3), epoch_ms=[round(x * 1e3, 2) for x in times],
                          rmse=rmse, **load_balance(plan.block_ptr.cpu().numpy(), b)))
        del plan
        print(json.dumps(sweep[-1]), file=sys.stderr, flush=True)
    t = time.perf_counter()
    plan = eng.sgd_plan(a, strata)
    out["plan_s"] = time.perf_counter() - t
    out["load_balance"] = load_balance(plan.block_ptr.cpu().numpy(), strata)
    out["max_item_nnz"] = int(plan.col_cnt.max())
    times, rmse = run_epochs(eng, plan, args.rank, args.warmup + args.steps)
    timed = times[args.warmup:]
    epoch_s = float(np.median(timed))
    out.update(epoch_ms=epoch_s * 1e3, epoch_ms_all=[t_ * 1e3 for t_ in timed], updates_per_s=nnz / epoch_s,
               rmse_history=rmse, bytes_per_update=bytes_per_update(args.rank))
    achieved = bytes_per_update(args.rank) * nnz / epoch_s
    out["algorithmic_bytes_per_s"] = achieved
    out["fraction_of_hbm_bandwidth_bound"] = achieved / HBM_BYTES_PER_S
    del plan
    # end to end from host triplets (what a data model hands over)
    ip = indptr.cpu().numpy()
    user = np.repeat(np.arange(args.users, dtype=np.int64), np.diff(ip))
    item = indices.cpu().numpy().astype(np.int64)
    val = values.cpu().numpy().astype(np.float64)
    del a, indptr, indices, values
    test = user % 10 == 0
    data = ArrayData(np.stack([user, item], axis=1), val, (args.users, args.items), user[test], item[test], val[test],
                     (int(np.unique(user[test]).size), args.items), warm_start=False)
    model = B200ProbabilisticMF(data, seed=1)
    model.verbose = False
    model.num_epochs = args.epochs
    model.tolerance = 0.0
    model.sgd_strata = strata
    t = time.perf_counter()
    model.build()
    out["build_e2e_s"] = time.perf_counter() - t
    out["build_epochs"] = args.epochs
    out["build_rmse_history"] = [float(x) for x in model.rmse_history]
    model.get_recommendations()                                    # warm-up
    reps = []
    for _ in range(3):
        t = time.perf_counter()
        recs = model.get_recommendations()
        reps.append(time.perf_counter() - t)
    out["score_s"] = float(np.median(reps))
    out["score_users"] = int(recs.shape[0])
    out["pairs_per_s"] = recs.shape[0] * args.items / out["score_s"]
    if sweep:
        out["strata_sweep"] = sweep
    return out


def bench_reference(args):
    from bench import synth_triplets_host
    from oracle import ref_driver as rd
    rd.import_reference()
    from polara.lib.optimize import generalized_sgd_sweep, identity
    user, item, fdbk = synth_triplets_host(args.users, args.items, args.nnz, seed=20260924)
    rn = np.bincount(user, minlength=args.users)
    cn = np.bincount(item, minlength=args.items)
    rs = np.random.RandomState(1)
    P = rs.normal(scale=0.1, size=(args.users, args.rank))
    Q = rs.normal(scale=0.1, size=(args.items, args.rank))
    k = 1000                                                       # JIT warm-up on the same dtypes
    generalized_sgd_sweep(user[:k], item[:k], fdbk[:k], P.copy(), Q.copy(), 0.005, 0.5, rn, cn, identity, ((), ()),
                          identity, ((), ()))
    t = time.perf_counter()
    err = generalized_sgd_sweep(user, item, fdbk, P, Q, 0.005, 0.5, rn, cn, identity, ((), ()), identity, ((), ()))
    epoch_s = time.perf_counter() - t
    return dict(config="pmf_c2", impl="reference", users=args.users, items=args.items, nnz=int(len(fdbk)), rank=args.rank,
                epoch_ms=epoch_s * 1e3, updates_per_s=len(fdbk) / epoch_s, rmse=float(np.sqrt(err / len(fdbk))),
                cpu=os.uname().machine)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--users", type=int, default=1_000_000)
    ap.add_argument("--items", type=int, default=100_000)
    ap.add_argument("--nnz", type=int, default=100_000_000)
    ap.add_argument("--rank", type=int, default=10)
    ap.add_argument("--steps", type=int, default=5, help="timed epochs")
    ap.add_argument("--warmup", type=int, default=1, help="epochs before the timed ones")
    ap.add_argument("--epochs", type=int, default=3, help="epochs of the end-to-end build")
    ap.add_argument("--strata", type=int, default=None, help="sgd_strata (default: the model's default)")
    ap.add_argument("--sweep", default=None, help="comma-separated sgd_strata values to time before the main run")
    ap.add_argument("--sweep-epochs", type=int, default=3)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    out = bench_b200(args) if args.impl == "b200" else bench_reference(args)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
