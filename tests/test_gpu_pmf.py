"""ProbabilisticMF on the device (pb200_sgd_plan / pb200_sgd_epoch + the fused scoring kernel) against the reference's
recorded runs (tests/golden/ref_pmf.npz), the oracle's restatement of the SGD sweep, and the reference's own numba
sweep.  The stratified epoch is the reference's sweep over a permutation of the interactions, so with the oracle fed the
same permutation the only difference left is the summation order of one r-term dot product per update: factors agree to
rtol 1e-9 and the RMSE history to 1e-12 relative."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import pmf_oracle as pmf
from tests.helpers import check_topk_against_scores
from tests.pmf_helpers import planted, reference_interactions, replay_known_split

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

FACTOR_RTOL, FACTOR_ATOL, RMSE_RTOL = 1e-9, 1e-12, 1e-12


@pytest.fixture(scope="module")
def fx(golden):
    g = golden("ref_pmf")
    (tr_u, tr_i, tr_f), (ts_u, ts_i, ts_f) = replay_known_split(*planted(g), g)
    return g, (tr_u, tr_i, tr_f), (ts_u, ts_i, ts_f)


def _data(fx):
    import pandas as pd
    from polara_b200.host import ArrayData
    g, (tr_u, tr_i, tr_f), (ts_u, ts_i, ts_f) = fx
    u, i, r = planted(g)
    new_user = np.full(u.max() + 1, -1, dtype=np.int64); new_user[g["user_old"]] = np.arange(len(g["user_old"]))
    new_item = np.full(i.max() + 1, -1, dtype=np.int64); new_item[g["item_old"]] = np.arange(len(g["item_old"]))
    h = g["holdout_rows"]
    hold = pd.DataFrame({"userid": new_user[u[h]], "itemid": new_item[i[h]], "rating": r[h]})
    return ArrayData(np.stack([tr_u, tr_i], axis=1), tr_f, g["train_shape"], ts_u, ts_i, ts_f, g["test_shape"],
                     holdout=hold, warm_start=False)


def _model(fx, **attrs):
    from polara_b200.models import B200ProbabilisticMF
    m = B200ProbabilisticMF(_data(fx), seed=5)
    m.verbose = False
    for k, v in attrs.items():
        setattr(m, k, v)
    return m


def _assert_run(model, P, Q, rmse):
    f = model.data.fields
    assert len(model.rmse_history) == len(rmse)
    np.testing.assert_allclose(model.rmse_history, rmse, rtol=RMSE_RTOL, atol=0)
    np.testing.assert_allclose(model.factors[f.userid], P, rtol=FACTOR_RTOL, atol=FACTOR_ATOL)
    np.testing.assert_allclose(model.factors[f.itemid], Q, rtol=FACTOR_RTOL, atol=FACTOR_ATOL)


@pytest.mark.parametrize("run", ["default", "early"])
def test_device_strata1_reproduces_the_reference(fx, run):
    g = fx[0]
    m = _model(fx, sgd_strata=1, tolerance=float(g["%s_tolerance" % run]))
    m.build()
    _assert_run(m, g["%s_P" % run], g["%s_Q" % run], g["%s_rmse" % run])
    assert len(m.rmse_history) == (25 if run == "default" else len(g["early_rmse"]))
    recs = m.get_recommendations()
    ref = g["%s_recs" % run].astype(np.int64)
    (tu, ti, tf), shape, users = m._get_test_data()
    scores = m.factors["userid"][users] @ m.factors["itemid"].T
    check_topk_against_scores(recs, scores, tu, ti, m.topk, tol=1e-4)
    assert (recs == ref).mean() >= 0.995
    if run == "default":
        hits = m.evaluate("hits")
        assert abs(hits.true_positive - g["default_hits"][0]) <= 2


@pytest.mark.parametrize("strata", [2, 7, 16])
@pytest.mark.parametrize("rank", [10, 32, 40, 100])
def test_device_matches_oracle_on_its_permutation(fx, strata, rank):
    g, (tr_u, tr_i, tr_f), _ = fx
    rows, cols, vals, rn, cn = reference_interactions(tr_u, tr_i, tr_f, g["train_shape"])
    order = pmf.sgd_strata_permutation(rows, cols, rn, cn, strata)
    epochs = 3
    P, Q, rmse = pmf.pmf_sgd(rows, cols, vals, g["train_shape"], rn, cn, rank, num_epochs=epochs, tol=0.0, seed=5,
                             order=order)
    m = _model(fx, sgd_strata=strata, rank=rank, num_epochs=epochs, tolerance=0.0)
    m.build()
    u, i, _ = m._sgd_plan.permutation()
    np.testing.assert_array_equal(u, rows[order])
    np.testing.assert_array_equal(i, cols[order])
    _assert_run(m, P, Q, rmse)


def _mid_size():
    from polara_b200.synth import popularity_csr
    indptr, indices, values = popularity_csr(50_000, 10_000, 2_000_000, seed=3)
    user = np.repeat(np.arange(50_000, dtype=np.int64), np.diff(indptr))
    return user, indices.astype(np.int64), values.astype(np.float64), (50_000, 10_000)


def test_determinism_and_reference_numba_sweep_on_the_device_permutation():
    from polara_b200.host import ArrayData
    from polara_b200.models import B200ProbabilisticMF
    user, item, val, shape = _mid_size()
    data = ArrayData(np.stack([user, item], axis=1), val, shape)
    runs = []
    for _ in range(2):
        m = B200ProbabilisticMF(data, seed=11)
        m.verbose = False
        m.num_epochs = 2
        m.build()
        runs.append(m)
    for key in ("userid", "itemid"):
        assert np.array_equal(runs[0].factors[key], runs[1].factors[key])
    assert runs[0].rmse_history == runs[1].rmse_history
    from oracle import ref_driver as rd
    if rd.reference_root() is None:
        pytest.skip("reference not installed (oracle/_ref)")
    rd.import_reference()
    from polara.lib.optimize import generalized_sgd_sweep, identity
    m = runs[0]
    pu, pi, pv = m._sgd_plan.permutation()
    rn, cn = np.bincount(user, minlength=shape[0]), np.bincount(item, minlength=shape[1])
    rs = np.random.RandomState(11)
    P = rs.normal(scale=0.1, size=(shape[0], m.rank))
    Q = rs.normal(scale=0.1, size=(shape[1], m.rank))
    errs = [generalized_sgd_sweep(pu.astype(np.intp), pi.astype(np.intp), pv.astype(np.float64), P, Q, m.learn_rate,
                                  0.5 * m.sigma ** 2, rn, cn, identity, ((), ()), identity, ((), ()))
            for _ in range(2)]
    np.testing.assert_allclose(m.rmse_history, np.sqrt(np.array(errs) / len(pv)), rtol=RMSE_RTOL)
    np.testing.assert_allclose(m.factors["userid"], P, rtol=FACTOR_RTOL, atol=FACTOR_ATOL)
    np.testing.assert_allclose(m.factors["itemid"], Q, rtol=FACTOR_RTOL, atol=FACTOR_ATOL)


@pytest.mark.parametrize("kernel", ["simt", "tcgen05"])
@pytest.mark.parametrize("filter_seen", [True, False])
def test_scoring_is_a_valid_topk_of_the_f64_scores(fx, kernel, filter_seen):
    m = _model(fx, num_epochs=8, score_kernel=kernel)
    m.build()
    m.filter_seen = filter_seen
    recs = m.get_recommendations()
    (tu, ti, tf), shape, users = m._get_test_data()
    scores = m.factors["userid"][users] @ m.factors["itemid"].T
    seen = (tu, ti) if filter_seen else (np.zeros(0, np.int64), np.zeros(0, np.int64))
    check_topk_against_scores(recs, scores, seen[0], seen[1], m.topk, tol=1e-4)
    # the single-user helper path (dense rows of slice_recommendations)
    row, _ = m.slice_recommendations((tu, ti, tf), shape, 3, 4)
    np.testing.assert_allclose(row[0], scores[3], rtol=1e-5, atol=1e-5)


def test_dropin_pmf_against_the_real_reference():
    pd = pytest.importorskip("pandas")
    from oracle import ref_driver as rd
    if rd.reference_root() is None:
        pytest.skip("reference not installed (oracle/_ref)")
    rd.import_reference()
    from polara.recommender.data import RecommenderData
    from polara.recommender.models import ProbabilisticMF
    from polara_b200.models import dropin, dropin_pmf
    from polara_b200.synth import planted_ratings
    assert len(dropin()) == 3
    u, i, r = planted_ratings(1500, 700, 60, rank=8, seed=17)
    data = RecommenderData(pd.DataFrame({"userid": u, "itemid": i, "rating": r}), "userid", "itemid", "rating", seed=0)
    data.verbose = False
    data.warm_start = False
    data.prepare()
    ref = ProbabilisticMF(data, seed=3); ref.verbose = False
    ref.build()
    ref_recs = ref.get_recommendations()
    mine = dropin_pmf()(data, seed=3); mine.verbose = False
    mine.sgd_strata = 1
    mine.build()
    f = data.fields
    np.testing.assert_allclose(mine.factors[f.userid], ref.factors[f.userid], rtol=FACTOR_RTOL, atol=FACTOR_ATOL)
    np.testing.assert_allclose(mine.factors[f.itemid], ref.factors[f.itemid], rtol=FACTOR_RTOL, atol=FACTOR_ATOL)
    np.testing.assert_allclose(mine.rmse_history, ref.rmse_history, rtol=RMSE_RTOL)
    recs = mine.get_recommendations()
    assert (recs == ref_recs).mean() >= 0.995
    assert abs(mine.evaluate("hits").true_positive - ref.evaluate("hits").true_positive) <= 3
    with pytest.raises(NotImplementedError):
        mine.build(adjust_gradient=None)


@pytest.mark.skipif(os.environ.get("PB200_SKIP_FULLSIZE") == "1", reason="full-size tests disabled")
def test_fullsize_c2_two_epochs():
    """C2 shape (1 M users x 100 K items, 1e8 interactions, bench.py's generator and seed), rank 10, default strata."""
    from polara_b200.engine import DeviceCSR, get_engine
    from polara_b200.models import DEFAULT_SGD_STRATA
    sys.path.insert(0, ROOT)
    from bench import synth_csr_torch
    if torch.cuda.get_device_properties(0).total_memory < 60e9:
        pytest.skip("needs a large-memory GPU")
    eng = get_engine(0)
    n_users, n_items, rank = 1_000_000, 100_000, 10
    indptr, indices, values = synth_csr_torch(n_users, n_items, 100_000_000, 20260924, eng.device)
    a = DeviceCSR(indptr, indices, values, (n_users, n_items))
    plan = eng.sgd_plan(a, DEFAULT_SGD_STRATA)
    assert int(plan.block_ptr[-1]) == a.nnz and int(plan.block_ptr[0]) == 0
    assert bool((plan.block_ptr[1:] >= plan.block_ptr[:-1]).all())
    # every nnz exactly once: the permuted (user, item) keys sort back to the CSR's keys
    rows = torch.repeat_interleave(torch.arange(n_users, device=eng.device), indptr[1:] - indptr[:-1])
    want = rows * n_items + indices.to(torch.int64)
    got = torch.sort(plan.users.to(torch.int64) * n_items + plan.items.to(torch.int64)).values
    assert torch.equal(got, want)
    del rows, want, got

    def run():
        rs = np.random.RandomState(1)
        p = eng.zeros((n_users, 32), torch.float64); q = eng.zeros((n_items, 32), torch.float64)
        p[:, :rank].copy_(torch.from_numpy(rs.normal(scale=0.1, size=(n_users, rank))))
        q[:, :rank].copy_(torch.from_numpy(rs.normal(scale=0.1, size=(n_items, rank))))
        errs = [eng.sgd_epoch(plan, p, q, rank, 0.005, 0.5) for _ in range(2)]
        return p, q, errs
    p1, q1, e1 = run()
    assert e1[1] < e1[0]
    p2, q2, e2 = run()
    assert e1 == e2 and torch.equal(p1, p2) and torch.equal(q1, q2)
    del p2, q2
    m = 100_000
    e = p1[:m].to(torch.float32).contiguous()
    v = q1.to(torch.float32).contiguous()
    ids = eng.score_topk(e, v, rank, 10, seen=(indptr[:m + 1], indices)).cpu().numpy()
    assert ids.min() >= 0 and ids.max() < n_items
    srt = np.sort(ids, axis=1)
    assert (srt[:, 1:] != srt[:, :-1]).all()
    ip, ix = indptr[:m + 1].cpu().numpy(), indices[: int(indptr[m])].cpu().numpy()
    seen_key = np.repeat(np.arange(m, dtype=np.int64), np.diff(ip)) * n_items + ix
    rec_key = np.repeat(np.arange(m, dtype=np.int64), 10) * n_items + ids.ravel()
    assert not np.isin(rec_key, seen_key).any()
