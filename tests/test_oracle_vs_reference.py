"""Oracle vs the reference, on what the reference computed from seeded inputs (``tests/golden/ref_*.npz``, recorded by
``oracle/make_golden.py``).  CPU only; the reference itself is not needed to run them."""
import numpy as np
import pytest
import scipy.sparse as sps

from oracle import polara_oracle as po
from polara_b200.synth import planted_ratings
from tests.helpers import ratings_digest, replay_split


def _planted_split(g):
    n_users, n_items, per_user, rank, seed = (int(x) for x in g["planted"])
    ratings = planted_ratings(n_users, n_items, per_user, rank=rank, seed=seed)
    assert ratings_digest(*ratings) == str(g["planted_sha256"]), \
        "fixture inputs changed: planted_ratings no longer reproduces the ratings the reference was run on"
    return replay_split(*ratings, g)


@pytest.mark.parametrize("seed", [1, 2])
def test_downvote_topk_rescale_live(golden, seed):
    g = golden("ref_downvote_topk_rescale_s%d" % seed)
    s = g["scores"]
    ref = s.copy()
    ref[g["seen_rows"], g["seen_cols"]] = g["downvoted_seen"]         # the rest of the block is left as it was
    mine = po.downvote_seen_items(s.copy(), g["seen_rows"], g["seen_cols"])
    np.testing.assert_array_equal(mine, ref)
    for row in range(20):
        np.testing.assert_array_equal(po.topsort(ref[row], 6), g["topsort6"][row])
    a = sps.csr_matrix((g["a_data"], g["a_indices"], g["a_indptr"]), shape=tuple(g["a_shape"]))
    for (scaling, axis), rescaled in zip(g["rescale_cases"], g["rescaled"]):
        np.testing.assert_allclose(po.rescale_matrix(a, scaling, int(axis)).toarray(), rescaled, rtol=1e-14)


def test_hooi_live(golden):
    g = golden("ref_hooi")
    mine = po.hooi(g["idx"].astype(np.intp), g["val"], tuple(g["shape"]), tuple(g["mlrank"]),
                   num_iters=int(g["num_iters"]), growth_tol=float(g["growth_tol"]), seed=int(g["seed"]))
    for a, b in zip(mine[:3], (g["u0"], g["u1"], g["u2"])):
        sv = np.linalg.svd(a.T @ b, compute_uv=False)
        assert sv.min() > 1 - 1e-9
    np.testing.assert_allclose(np.linalg.norm(mine[3]), np.linalg.norm(g["core"]), rtol=1e-10)


def test_c1_shaped_svd_model_live(golden):
    """BASELINE config C1 (ML-1M shape: 6040 x 3706, ~1.0e6 ratings, PureSVD rank 10, top-10) as the reference ran it
    (RecommenderData.prepare + SVDModel.build + get_recommendations with its default chunking) against the oracle on the
    arrays the reference's data model handed over: singular values, item-factor subspace, and every recommendation list
    (scored with the reference's own factors: exact; with the oracle's factors: up to near-ties)."""
    g = golden("ref_c1_svd")
    (u, i, r), (tu, ti, tf) = _planted_split(g)
    assert len(g["test_user_old"]) == 1208 and len(u) + len(tf) + len(g["holdout_rows"]) == 6040 * 166
    a = sps.csr_matrix((r, (u, i)), shape=tuple(g["train_shape"]), dtype=np.float64)
    v, s, _ = po.svd_build(a, int(g["rank"]))
    np.testing.assert_allclose(s, g["singular_values"], rtol=1e-9)
    vref = g["item_factors"].astype(np.float64)
    assert np.linalg.svd(v.T @ vref, compute_uv=False).min() > 1 - 1e-6
    recs = g["recs"]
    tshape = tuple(g["test_shape"])
    mine = po.recommend_svd(tu, ti, tf, tshape, vref, topk=10)
    assert mine.shape == recs.shape and recs.shape[1] == 10
    np.testing.assert_array_equal(mine, recs)
    own = po.recommend_svd(tu, ti, tf, tshape, v, topk=10)
    assert (own == recs).mean() > 0.99


def test_coffee_model_live_default_mlrank(golden):
    """CoffeeModel with the reference's default multilinear rank (13, 10, 2) on a 1500 x 600 x 5 tensor as the reference
    ran it, against the oracle: HOOI from the same seed (factor subspaces, core norm) and every recommendation list
    scored with the reference's factors."""
    g = golden("ref_coffee_default_mlrank")
    assert tuple(g["mlrank"]) == (13, 10, 2)
    (u, i, r), (tu, ti, tf) = _planted_split(g)
    level = lambda f: np.searchsorted(g["fdbk_old"], f)       # noqa: E731  (tensor mode: feedback -> level index)
    idx = np.stack([u, i, level(r)], axis=1).astype(np.intp)
    mine = po.hooi(idx, np.ones(len(idx)), tuple(g["train_shape"]), tuple(g["mlrank"]), num_iters=int(g["num_iters"]),
                   growth_tol=float(g["growth_tol"]), seed=int(g["seed"]))
    for got, key in zip(mine[:3], ("u0", "u1", "u2")):
        assert np.linalg.svd(got.T @ g[key].astype(np.float64), compute_uv=False).min() > 1 - 1e-6, key
    np.testing.assert_allclose(np.linalg.norm(mine[3]), np.linalg.norm(g["core"]), rtol=1e-8)
    lists = po.recommend_coffee(tu, ti, level(tf).astype(np.int64), tuple(g["test_shape"]),
                                g["u1"].astype(np.float64), g["u2"].astype(np.float64), topk=10)
    np.testing.assert_array_equal(lists, g["recs"])


def test_round_core_live(golden):
    """CoffeeModel.round_core / _check_reduced_rank (models.py:949-980) against the oracle restatement."""
    g = golden("ref_round_core")
    core = g["core"]
    for c, (mode, rank) in enumerate(g["cases"]):
        mode, rank = int(mode), int(rank)
        rot, new_core = po.round_core(core, mode, rank)
        np.testing.assert_allclose(rot, g["rot%d" % c], rtol=0, atol=1e-13)
        np.testing.assert_allclose(new_core, g["core%d" % c], rtol=0, atol=1e-13)
        assert new_core.shape[mode] == rank


@pytest.mark.parametrize("switch_positive", [None, 4])
def test_simple_rates_match_reference_live(golden, switch_positive):
    """evaluate(simple_rates=True) / holdout_size == 1 (models.py:451-458): hit rate, ARHR and MRR of the host mirror
    against the reference's own evaluation functions on random lists."""
    from polara_b200.host import evaluate_lists
    g = golden("ref_simple_rates")
    tag = "none" if switch_positive is None else str(switch_positive)
    rel, rank = evaluate_lists(g["recs"], g["holdout_user"], g["holdout_item"], g["holdout_fdbk"], int(g["n_items"]),
                               metric_type=["relevance", "ranking"], switch_positive=switch_positive, simple_rates=True)
    np.testing.assert_allclose(rel.hr, g["hr_" + tag], rtol=1e-12)
    np.testing.assert_allclose(rank.arhr, g["arhr_" + tag], rtol=1e-12)
    np.testing.assert_allclose(rank.mrr, g["mrr_" + tag], rtol=1e-12)
