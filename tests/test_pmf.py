"""ProbabilisticMF without a GPU: the oracle's restatement of the reference's SGD sweep against the recorded reference
runs (tests/golden/ref_pmf.npz), the stratified order of the device build, and the host-side model logic."""
import numpy as np
import pytest

from oracle import pmf_oracle as pmf
from oracle import polara_oracle as po
from polara_b200.engine import sgd_strata_bounds
from tests.helpers import ratings_digest
from tests.pmf_helpers import planted, reference_interactions, replay_known_split


@pytest.fixture(scope="module")
def fx(golden):
    g = golden("ref_pmf")
    u, i, r = planted(g)
    assert ratings_digest(u, i, r) == str(g["planted_sha256"]), "the ratings generator changed: fixture inputs differ"
    (tr_u, tr_i, tr_f), test = replay_known_split(u, i, r, g)
    return g, reference_interactions(tr_u, tr_i, tr_f, g["train_shape"]), test


@pytest.mark.parametrize("run", ["default", "early"])
def test_oracle_pmf_sgd_is_bit_exact_against_the_reference(fx, run):
    """The oracle runs the same f64 operations in the same order as the reference's numba sweep (the dot product is
    BLAS ddot on both sides), so equality is exact here."""
    g, (rows, cols, vals, rn, cn), _ = fx
    P, Q, rmse = pmf.pmf_sgd(rows, cols, vals, g["train_shape"], rn, cn, int(g["rank"]), float(g["learn_rate"]),
                            float(g["sigma"]), int(g["num_epochs"]), float(g["%s_tolerance" % run]), seed=int(g["seed"]))
    assert len(rmse) == len(g["%s_rmse" % run])
    assert len(rmse) == (25 if run == "default" else 2)
    np.testing.assert_array_equal(rmse, g["%s_rmse" % run])
    np.testing.assert_array_equal(P, g["%s_P" % run])
    np.testing.assert_array_equal(Q, g["%s_Q" % run])
    # the lists of the reference's scoring on these factors (models.py:779-787)
    tu, ti, _ = fx[2]
    users = np.unique(tu)
    scores = P[users] @ Q.T
    seen_r = np.searchsorted(users, tu)
    po.downvote_seen_items(scores, seen_r, ti)
    np.testing.assert_array_equal(po.get_topk_elements(scores, 10), g["%s_recs" % run])


def _zipf_counts(rng, n, total, a=1.3):
    c = np.floor(total / np.arange(1, n + 1) ** a).astype(np.int64)
    rng.shuffle(c)
    return c


@pytest.mark.parametrize("strata", [1, 2, 5, 16, 64])
def test_strata_bounds_match_the_product_cut(strata):
    rng = np.random.default_rng(strata)
    cases = [_zipf_counts(rng, 300, 5000), rng.integers(0, 4, 200),
             np.r_[np.zeros(10, np.int64), [10_000], rng.integers(0, 3, 50)],          # one row with most of the nnz
             np.r_[np.zeros(40, np.int64), [3, 0, 5, 0, 0, 2], np.zeros(30, np.int64)]]   # B > non-empty rows
    for counts in cases:
        b = pmf.sgd_strata_bounds(counts, strata)
        np.testing.assert_array_equal(sgd_strata_bounds(counts, strata), b)
        assert len(b) == strata + 1 and b[0] == 0 and b[-1] == len(counts) and (np.diff(b) >= 0).all()


@pytest.mark.parametrize("strata", [1, 3, 7, 16])
def test_strata_permutation(fx, strata):
    _, (rows, cols, _, rn, cn), _ = fx
    order = pmf.sgd_strata_permutation(rows, cols, rn, cn, strata)
    assert np.array_equal(np.sort(order), np.arange(len(rows)))
    if strata == 1:
        assert np.array_equal(order, np.arange(len(rows)))
    rb_of = np.searchsorted(pmf.sgd_strata_bounds(rn, strata), np.arange(len(rn)), side="right") - 1
    cb_of = np.searchsorted(pmf.sgd_strata_bounds(cn, strata), np.arange(len(cn)), side="right") - 1
    r, c = rows[order], cols[order]
    rb, cb = rb_of[r], cb_of[c]
    sub = (cb - rb) % strata
    assert (np.diff(sub) >= 0).all()
    for s in range(strata):
        sel = sub == s
        # blocks of one sub-epoch share no user and no item
        for blocks, idx in ((rb, r), (cb, c)):
            owner = {}
            for blk, x in zip(blocks[sel].tolist(), idx[sel].tolist()):
                assert owner.setdefault(x, blk) == blk
        # row-major inside each block, blocks in b order
        key = rb[sel].astype(np.int64) * (len(rn) * len(cn)) + r[sel].astype(np.int64) * len(cn) + c[sel]
        assert (np.diff(key) > 0).all()


def test_host_model_logic_without_a_gpu(fx):
    from polara_b200.host import ArrayData
    from polara_b200.models import DEFAULT_SGD_STRATA, B200ProbabilisticMF
    g, (rows, cols, vals, _, _), (tu, ti, tf) = fx
    data = ArrayData(np.stack([rows, cols], axis=1), vals, g["train_shape"], tu, ti, tf, g["test_shape"],
                     warm_start=False)
    m = B200ProbabilisticMF(data, seed=5)
    # ProbabilisticMF.__init__ (models.py:729-741)
    assert (m.seed, m.method, m.learn_rate, m.sigma, m.num_epochs, m.rank, m.tolerance) == (5, "PMF", 0.005, 1, 25, 10, 1e-4)
    assert m.factors == {} and m.rmse_history is None and m.iterations_time is None and m.show_rmse is False
    assert m.sgd_strata == DEFAULT_SGD_STRATA
    m.rank = 7                                    # a plain attribute: no truncation, no invalidation
    assert m.rank == 7
    with pytest.raises(NotImplementedError):
        m.build(adjust_gradient="adagrad")
    with pytest.raises(NotImplementedError):
        m.build(None)
    m.optimizer = lambda *a, **k: None
    with pytest.raises(NotImplementedError):
        m.build()
    m.optimizer = None

    class Shard:
        world = 2
    m.shard = Shard()
    with pytest.raises(NotImplementedError):
        m.build()
    del m.shard
    data.warm_start = True
    with pytest.raises(NotImplementedError):
        m.get_recommendations()
    data.warm_start = False
    # the build wrapper (MetaModel, models.py:59-67) drops cached lists before building
    m._recommendations = np.zeros((1, 10), dtype=np.int64)
    m._is_ready = True
    with pytest.raises(NotImplementedError):
        m.build(adjust_gradient="adam")
    assert m._recommendations is None and m._is_ready is False


def test_stratified_schedule_stays_close_to_the_reference(fx):
    """B = 16 on the fixture data with the reference's defaults.  Observed (this computation): final RMSE 0.69238 against
    the reference's 0.68160 (+1.6 %), true positives 222 against 236 of 480 holdout items.  Margins: RMSE within 2.5 %,
    true positives within 20 (about 4 % of the holdout)."""
    g, (rows, cols, vals, rn, cn), (tu, ti, _) = fx
    order = pmf.sgd_strata_permutation(rows, cols, rn, cn, 16)
    P, Q, rmse = pmf.pmf_sgd(rows, cols, vals, g["train_shape"], rn, cn, 10, seed=5, order=order)
    assert len(rmse) == 25
    assert abs(rmse[-1] - g["default_rmse"][-1]) <= 0.025 * g["default_rmse"][-1]
    users = np.unique(tu)
    scores = P[users] @ Q.T
    po.downvote_seen_items(scores, np.searchsorted(users, tu), ti)
    recs = po.get_topk_elements(scores, 10)
    u, i, _ = planted(g)
    h = g["holdout_rows"]
    new_user = np.full(u.max() + 1, -1); new_user[g["user_old"]] = np.arange(len(g["user_old"]))
    new_item = np.full(i.max() + 1, -1); new_item[g["item_old"]] = np.arange(len(g["item_old"]))
    hu, hi = new_user[u[h]], new_item[i[h]]
    row = np.searchsorted(users, hu)
    tp = sum(int(item in recs[rr]) for rr, item in zip(row, hi))
    assert abs(tp - int(g["default_hits"][0])) <= 20, tp
