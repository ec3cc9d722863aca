"""Generate ``tests/golden/*.npz`` by running the REAL reference (the polara
checkout ``oracle.ref_shim.REFERENCE_ROOT`` names: ``POLARA_REFERENCE_ROOT``, or its
default when the variable is unset).  TEST INFRASTRUCTURE.

    POLARA_REFERENCE_ROOT=<polara checkout> python oracle/make_golden.py [fixture ...]

Without arguments every fixture is regenerated.

Each fixture stores the hot path's *inputs* exactly as the reference's data
model hands them to the model (``to_coo``, ``_get_test_data``), plus the
reference's *outputs* (factors, recommendations, evaluate() hit counts), so the
fixtures can be replayed where the reference is not installed.  The ``ref_*``
fixtures hold what tests/test_oracle_vs_reference.py compares the oracle with;
the larger ones store the split of the seeded ratings instead of the ratings
(``_record_split``), which tests/helpers.py ``replay_split`` turns back into
the data model's arrays.
"""
import os
import sys

import numpy as np
import pandas as pd
import scipy.sparse as sps

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle.ref_shim import import_reference  # noqa: E402
from polara_b200.synth import planted_ratings  # noqa: E402
from tests.helpers import ratings_digest, replay_split  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def _frame(n_users, n_items, per_user, rank, seed):
    u, i, r = planted_ratings(n_users, n_items, per_user, rank=rank, seed=seed)
    return pd.DataFrame({"userid": u, "itemid": i, "rating": r})


def _holdout_arrays(model):
    h = model.data.test.holdout
    f = model.data.fields
    return (h[f.userid].values.astype(np.int64), h[f.itemid].values.astype(np.int64),
            h[f.feedback].values.astype(np.float64))


def _hits(model, **kw):
    hits = model.evaluate("hits", **kw)
    return np.array([-1 if x is None else x for x in hits], dtype=np.float64)


def _relevance(model, **kw):
    rel = model.evaluate("relevance", **kw)
    return np.array([np.nan if x is None else x for x in rel], dtype=np.float64)


def svd_fixture(name, warm_start, rank, scaled=False, feedback_threshold=None, seed=7,
                switch_positive=None):
    polara = import_reference()
    from polara.recommender.data import RecommenderData
    from polara.recommender.models import SVDModel, ScaledSVD
    df = _frame(420, 260, 36, rank=6, seed=seed)
    data = RecommenderData(df, "userid", "itemid", "rating", seed=0)
    data.warm_start = warm_start
    data.verbose = False
    data.prepare()
    model = (ScaledSVD if scaled else SVDModel)(data, feedback_threshold=feedback_threshold)
    model.verbose = False
    model.rank = rank
    model.switch_positive = switch_positive
    model.build()
    recs = model.get_recommendations()
    idx, val, shp = data.to_coo(tensor_mode=False, feedback_threshold=model.feedback_threshold)
    (tu, ti, tf), tshape, tusers = model._get_test_data()
    hu, hi, hf = _holdout_arrays(model)
    out = dict(
        train_idx=idx.astype(np.int64), train_val=val.astype(np.float64), train_shape=np.array(shp),
        test_user=tu.astype(np.int64), test_item=ti.astype(np.int64), test_fdbk=np.asarray(tf, dtype=np.float64),
        test_shape=np.array(tshape), test_users=np.asarray(tusers, dtype=np.int64),
        holdout_user=hu, holdout_item=hi, holdout_fdbk=hf,
        rank=np.array(rank), topk=np.array(model.topk),
        item_factors=model.factors["itemid"], singular_values=model.factors["singular_values"],
        recs=recs.astype(np.int64),
        hits=_hits(model), relevance=_relevance(model),
        warm_start=np.array(warm_start), scaled=np.array(scaled),
        col_scaling=np.array(getattr(model, "col_scaling", 1.0)),
        row_scaling=np.array(getattr(model, "row_scaling", 1.0)),
        feedback_threshold=np.array(np.nan if feedback_threshold is None else feedback_threshold),
        switch_positive=np.array(np.nan if switch_positive is None else switch_positive),
    )
    # reduced-rank replay (models.py:819-832): same factors truncated, no rebuild
    model.rank = rank - 3
    out["recs_reduced"] = model.get_recommendations().astype(np.int64)
    out["rank_reduced"] = np.array(rank - 3)
    # wider list
    model.topk = 25
    out["recs_top25"] = model.get_recommendations().astype(np.int64)
    # unfiltered
    model.filter_seen = False
    model.topk = 10
    out["recs_unfiltered"] = model.get_recommendations().astype(np.int64)
    np.savez_compressed(os.path.join(GOLDEN, name + ".npz"), **out)
    print(name, "train nnz", len(val), "test users", tshape[0], "hits", out["hits"])


def coffee_fixture(name, mlrank=(6, 5, 3), seed=11, flattener=None):
    polara = import_reference()
    from polara.recommender.data import RecommenderData
    from polara.recommender.models import CoffeeModel
    df = _frame(360, 220, 30, rank=5, seed=seed)
    data = RecommenderData(df, "userid", "itemid", "rating", seed=0)
    data.verbose = False
    data.prepare()
    model = CoffeeModel(data)
    model.verbose = False
    model.mlrank = mlrank
    model.seed = 3
    model.num_iters = 12
    if flattener is not None:
        model.flattener = flattener
    model.build()
    recs = model.get_recommendations()
    idx, val, shp = data.to_coo(tensor_mode=True)
    (tu, ti, tf), tshape, tusers = model._get_test_data()
    hu, hi, hf = _holdout_arrays(model)
    out = dict(
        train_idx=idx.astype(np.int64), train_val=val.astype(np.float64), train_shape=np.array(shp),
        test_user=tu.astype(np.int64), test_item=ti.astype(np.int64), test_fdbk=np.asarray(tf, dtype=np.int64),
        test_shape=np.array(tshape), test_users=np.asarray(tusers, dtype=np.int64),
        holdout_user=hu, holdout_item=hi, holdout_fdbk=hf,
        mlrank=np.array(mlrank), topk=np.array(model.topk), seed=np.array(model.seed),
        num_iters=np.array(model.num_iters), growth_tol=np.array(model.growth_tol),
        u0=model.factors["userid"], u1=model.factors["itemid"], u2=model.factors["rating"],
        core=model.factors["core"], recs=recs.astype(np.int64), hits=_hits(model),
        flattener=np.array(-1 if flattener is None else flattener),
    )
    np.savez_compressed(os.path.join(GOLDEN, name + ".npz"), **out)
    print(name, "nnz", len(val), "shape", shp, "hits", out["hits"])


def kernel_fixture(name="kernels_small", seed=5):
    """Direct calls of the reference's static kernels on random inputs."""
    polara = import_reference()
    from polara.recommender.models import RecommenderModel
    from polara.preprocessing.matrices import rescale_matrix
    from polara.lib.tensor import ttm3d_seq
    from polara.recommender.utils import get_chunk_size
    from polara.recommender import defaults
    import scipy.sparse as sps
    rng = np.random.default_rng(seed)
    scores = rng.standard_normal((37, 91))
    seen_r = np.repeat(np.arange(37), 6)
    seen_c = np.concatenate([rng.choice(91, 6, replace=False) for _ in range(37)])
    down = scores.copy()
    RecommenderModel.downvote_seen_items(down, (seen_r, seen_c))

    class _K:  # get_topk_elements only needs ``self.topk``
        topk = 7
        topsort = staticmethod(RecommenderModel.topsort)
    top = RecommenderModel.get_topk_elements(_K(), down)
    a = sps.random(60, 45, density=0.15, random_state=3, format="csr")
    a.data = np.rint(1 + 4 * a.data)
    sc_rows = rescale_matrix(a, 0.7, 1)
    sc_cols = rescale_matrix(a, 0.4, 0)
    nnz = 500
    shp = (30, 20, 4)
    idx = np.stack([rng.integers(0, s, nnz) for s in shp], axis=1).astype(np.intp)
    val = rng.random(nnz)
    u = rng.standard_normal((20, 3))
    v = rng.standard_normal((4, 2))
    ttm0 = ttm3d_seq(idx, val, shp, v, u, ((2, 0), (1, 0)))
    old = defaults.memory_hard_limit
    chunks = np.array([get_chunk_size((1_000_000, 100_000), 10, 1),
                       get_chunk_size((6040, 3706), 10, 1)])
    defaults.memory_hard_limit = old
    np.savez_compressed(
        os.path.join(GOLDEN, name + ".npz"), scores=scores, seen_r=seen_r, seen_c=seen_c, downvoted=down,
        topk7=top.astype(np.int64), a_indptr=a.indptr, a_indices=a.indices, a_data=a.data,
        a_shape=np.array(a.shape), sc_rows=sc_rows.toarray(), sc_cols=sc_cols.toarray(),
        ttm_idx=idx.astype(np.int64), ttm_val=val, ttm_shape=np.array(shp), ttm_u=u, ttm_v=v, ttm0=ttm0,
        chunks=chunks)
    print(name, "done")


def _save(name, **arrays):
    np.savez_compressed(os.path.join(GOLDEN, name + ".npz"), **arrays)
    print(name, "done")


def ref_downvote_topk_rescale(seed):
    """Static kernels on seeded inputs: downvote_seen_items, topsort and rescale_matrix."""
    import_reference()
    from polara.recommender.models import RecommenderModel
    from polara.preprocessing.matrices import rescale_matrix
    rng = np.random.default_rng(seed)
    s = rng.standard_normal((20, 50))
    rows = np.repeat(np.arange(20), 4)
    cols = np.concatenate([rng.choice(50, 4, replace=False) for _ in range(20)])
    down = s.copy()
    RecommenderModel.downvote_seen_items(down, (rows, cols))
    top = np.stack([RecommenderModel.topsort(down[row], 6) for row in range(20)])
    unseen = np.ones(s.shape, dtype=bool)
    unseen[rows, cols] = False
    np.testing.assert_array_equal(down[unseen], s[unseen])        # only the seen entries are stored
    a = sps.random(40, 30, density=0.2, random_state=seed, format="csr")
    cases = np.array([(0.4, 0), (0.8, 1), (1, 0)])
    rescaled = np.stack([rescale_matrix(a, scaling, int(axis)).toarray() for scaling, axis in cases])
    _save("ref_downvote_topk_rescale_s%d" % seed, scores=s, seen_rows=rows, seen_cols=cols, downvoted_seen=down[rows, cols],
          topsort6=top.astype(np.int64), a_indptr=a.indptr, a_indices=a.indices, a_data=a.data, a_shape=np.array(a.shape),
          rescale_cases=cases, rescaled=rescaled)


def ref_hooi():
    import_reference()
    from polara.lib.tensor import hooi
    rng = np.random.default_rng(3)
    shp = (40, 30, 5)
    idx = np.unique(np.stack([rng.integers(0, s, 900) for s in shp], axis=1), axis=0).astype(np.intp)
    val = np.ones(len(idx))
    u0, u1, u2, core = hooi(idx, val, shp, (4, 3, 2), num_iters=6, growth_tol=1e-4, seed=5)[:4]
    _save("ref_hooi", idx=idx.astype(np.int64), val=val, shape=np.array(shp), mlrank=np.array((4, 3, 2)),
          num_iters=np.array(6), growth_tol=np.array(1e-4), seed=np.array(5), u0=u0, u1=u1, u2=u2, core=core)


def ref_round_core():
    """CoffeeModel.round_core (models.py:949-980) on a seeded core, one output pair per (mode, rank) case."""
    import_reference()
    from polara.recommender.models import CoffeeModel
    core = np.random.default_rng(9).standard_normal((7, 6, 4))
    cases = np.array([(0, 3), (1, 6), (1, 2), (2, 1), (2, 3)])
    out = dict(core=core, cases=cases)
    for c, (mode, rank) in enumerate(cases):
        out["rot%d" % c], out["core%d" % c] = CoffeeModel.round_core(core, int(mode), int(rank))
    _save("ref_round_core", **out)


def ref_simple_rates():
    """evaluate(simple_rates=True) (models.py:451-458): hit rate, ARHR and MRR of random lists, without and with
    switch_positive=4."""
    import_reference()
    from polara.recommender.evaluation import assemble_scoring_matrices, get_hr_score, get_rr_scores
    rng = np.random.default_rng(12)
    m, n, k = 60, 90, 10
    recs = np.stack([rng.choice(n, k, replace=False) for _ in range(m)])
    hu = np.repeat(np.arange(m), 3)
    hi = np.concatenate([rng.choice(n, 3, replace=False) for _ in range(m)])
    hf = rng.integers(1, 6, size=len(hu)).astype(np.float64)
    holdout = pd.DataFrame({"userid": hu, "itemid": hi, "rating": hf})
    out = dict(recs=recs.astype(np.int64), holdout_user=hu, holdout_item=hi, holdout_fdbk=hf, n_items=np.array(n))
    for tag, switch_positive in (("none", None), ("4", 4)):
        is_positive = None if switch_positive is None else (hf >= switch_positive)
        scoring = assemble_scoring_matrices(recs, holdout, "userid", "itemid", is_positive, feedback="rating")
        out["hr_" + tag] = np.array(get_hr_score(scoring[1]).hr)
        rr = get_rr_scores(scoring[1])
        out["arhr_" + tag], out["mrr_" + tag] = np.array(rr.arhr), np.array(rr.mrr)
    _save("ref_simple_rates", **out)


def _record_split(data, planted):
    """The split ``RecommenderData.prepare()`` made of the ratings ``planted_ratings(*planted)``: which original users
    went to training and to test (ordered by their new index), the item index, and the original rows held out."""
    def old_by_new(frame):
        return _small_int(frame.sort_values("new")["old"].to_numpy())
    return dict(planted=np.array(planted), planted_sha256=np.array(ratings_digest(*_planted(planted))),
                train_user_old=old_by_new(data.index.userid.training),
                test_user_old=old_by_new(data.index.userid.test), item_old=old_by_new(data.index.itemid),
                holdout_rows=np.sort(data.test.holdout.index.to_numpy()).astype(np.int32))


def _small_int(a):
    """Index arrays in int16 when they fit (smaller fixtures)."""
    return a.astype(np.int16) if a.size and 0 <= a.min() and a.max() < 2 ** 15 else a.astype(np.int32)


def _stored_f32(factors, recs, recommend):
    """Factor matrices are stored in float32 to keep the fixtures small; the reference's lists must come out unchanged
    when its own scoring path is fed the rounded factors, so the tests can still demand exact equality."""
    f32 = {k: np.asarray(v, dtype=np.float32) for k, v in factors.items()}
    np.testing.assert_array_equal(recommend(**{k: v.astype(np.float64) for k, v in f32.items()}), recs)
    return f32


def _planted(planted):
    n_users, n_items, per_user, rank, seed = (int(x) for x in planted)
    return planted_ratings(n_users, n_items, per_user, rank=rank, seed=seed)


def ref_c1_svd():
    """BASELINE config C1 (ML-1M shape: 6040 x 3706, ~1.0e6 ratings, PureSVD rank 10, top-10) through the reference's
    RecommenderData.prepare + SVDModel.build + get_recommendations with its default chunking."""
    import_reference()
    from polara.recommender.data import RecommenderData
    from polara.recommender.models import SVDModel
    planted = (6040, 3706, 166, 12, 11)
    u, i, r = _planted(planted)
    data = RecommenderData(pd.DataFrame({"userid": u, "itemid": i, "rating": r}), "userid", "itemid", "rating", seed=0)
    data.verbose = False
    data.prepare()
    model = SVDModel(data)
    model.verbose = False
    model.rank = 10
    model.build()
    recs = model.get_recommendations()
    idx, val, shp = data.to_coo(tensor_mode=False)
    (tu, ti, tf), tshape, _ = model._get_test_data()
    g = _record_split(data, planted)
    train, test = replay_split(u, i, r, g)
    for got, want in zip(train + test, (idx[:, 0], idx[:, 1], val, tu, ti, tf)):
        np.testing.assert_array_equal(got, want)
    itemid = data.fields.itemid

    def recommend(item_factors):
        model.factors[itemid] = item_factors
        return model.get_recommendations()
    sigma = model.factors["singular_values"]
    stored = _stored_f32({"item_factors": model.factors[itemid]}, recs, recommend)
    _save("ref_c1_svd", train_shape=np.array(shp), test_shape=np.array(tshape), rank=np.array(10),
          singular_values=sigma, recs=_small_int(recs), **stored, **g)


def ref_coffee_default_mlrank():
    """CoffeeModel with the reference's default multilinear rank (13, 10, 2) on a 1500 x 600 x 5 tensor: HOOI from seed 3
    (8 iterations) and the recommendation lists."""
    import_reference()
    from polara.recommender.data import RecommenderData
    from polara.recommender.models import CoffeeModel
    planted = (1500, 600, 40, 6, 13)
    u, i, r = _planted(planted)
    data = RecommenderData(pd.DataFrame({"userid": u, "itemid": i, "rating": r}), "userid", "itemid", "rating", seed=0)
    data.verbose = False
    data.prepare()
    model = CoffeeModel(data)
    model.verbose = False
    model.seed = 3
    model.num_iters = 8
    model.build()
    recs = model.get_recommendations()
    idx, val, shp = data.to_coo(tensor_mode=True)
    (tu, ti, tf), tshape, _ = model._get_test_data()
    g = _record_split(data, planted)
    g["fdbk_old"] = data.index.feedback.sort_values("new")["old"].to_numpy().astype(np.float64)
    (tr_u, tr_i, tr_f), (ts_u, ts_i, ts_f) = replay_split(u, i, r, g)
    assert (val == 1).all()
    level = lambda f: np.searchsorted(g["fdbk_old"], f)       # noqa: E731  (tensor mode: feedback -> level index)
    for got, want in zip((tr_u, tr_i, level(tr_f), ts_u, ts_i, level(ts_f)),
                         (idx[:, 0], idx[:, 1], idx[:, 2], tu, ti, tf)):
        np.testing.assert_array_equal(got, want)
    f = data.fields

    def recommend(u0, u1, u2):
        model.factors.update({f.userid: u0, f.itemid: u1, f.feedback: u2})
        return model.get_recommendations()
    core = model.factors["core"]
    stored = _stored_f32({"u0": model.factors[f.userid], "u1": model.factors[f.itemid], "u2": model.factors[f.feedback]},
                         recs, recommend)
    _save("ref_coffee_default_mlrank", train_shape=np.array(shp), test_shape=np.array(tshape),
          mlrank=np.array(model.mlrank), num_iters=np.array(model.num_iters), growth_tol=np.array(model.growth_tol),
          seed=np.array(model.seed), core=core, recs=_small_int(recs), **stored, **g)


FIXTURES = {
    "kernels_small": kernel_fixture,
    "svd_warm_r10": lambda: svd_fixture("svd_warm_r10", warm_start=True, rank=10),
    "svd_known_r8": lambda: svd_fixture("svd_known_r8", warm_start=False, rank=8, switch_positive=4),
    "svd_scaled_r10": lambda: svd_fixture("svd_scaled_r10", warm_start=True, rank=10, scaled=True),
    # NOTE: a feedback_threshold fixture cannot be produced through the full
    # reference stack under pandas>=3 (data.py:790 writes into a read-only
    # ``.values`` view); that semantic (zeroed feedback stays in the seen list,
    # models.py:191-211) is covered through the oracle in tests/test_oracle_golden.py.
    "coffee_small": lambda: coffee_fixture("coffee_small"),
    "coffee_flat34": lambda: coffee_fixture("coffee_flat34", flattener=[2, 3], seed=12),
    "ref_downvote_topk_rescale_s1": lambda: ref_downvote_topk_rescale(1),
    "ref_downvote_topk_rescale_s2": lambda: ref_downvote_topk_rescale(2),
    "ref_hooi": ref_hooi,
    "ref_round_core": ref_round_core,
    "ref_simple_rates": ref_simple_rates,
    "ref_c1_svd": ref_c1_svd,
    "ref_coffee_default_mlrank": ref_coffee_default_mlrank,
}


if __name__ == "__main__":
    os.makedirs(GOLDEN, exist_ok=True)
    for fixture in sys.argv[1:] or FIXTURES:
        FIXTURES[fixture]()
