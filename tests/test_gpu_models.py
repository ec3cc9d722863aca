"""End-to-end parity of the device models against fixtures recorded from the REAL
reference (tests/golden, made by oracle/make_golden.py).  B200 box only."""
import numpy as np
import pytest

from oracle import polara_oracle as po
from tests.helpers import subspace_gap

pytestmark = pytest.mark.gpu


def _svd_model(g, scaled=False):
    from polara_b200.host import ArrayData
    from polara_b200.models import B200ScaledSVD, B200SVDModel
    data = ArrayData.from_golden(g)
    model = (B200ScaledSVD if scaled else B200SVDModel)(data)
    model.verbose = False
    model.rank = int(g["rank"])
    if scaled:
        model.col_scaling = float(g["col_scaling"])
        model.row_scaling = float(g["row_scaling"])
    sp = float(g["switch_positive"])
    model.switch_positive = None if np.isnan(sp) else sp
    return model


@pytest.mark.parametrize("name", ["svd_warm_r10", "svd_known_r8", "svd_scaled_r10"])
def test_svd_model_reproduces_reference(golden, name):
    g = golden(name)
    model = _svd_model(g, scaled=bool(g["scaled"]))
    model.build()
    np.testing.assert_allclose(model.factors["singular_values"], g["singular_values"], rtol=2e-4)
    assert subspace_gap(model.factors["itemid"], g["item_factors"]) < 2e-2
    recs = model.get_recommendations()
    assert recs.dtype == np.int64 and recs.shape == g["recs"].shape
    assert (recs == g["recs"]).mean() > 0.97          # fp32 + subspace tolerance: a few near-tie swaps
    # evaluate(): hit counts within a couple of hits of the recorded reference numbers
    hits = model.evaluate("hits")
    ref = g["hits"]
    assert abs(hits.true_positive - ref[0]) <= 3
    assert abs(hits.false_negative - ref[3]) <= 3


@pytest.mark.parametrize("name", ["svd_warm_r10", "svd_known_r8"])
def test_scoring_with_reference_factors_is_exact(golden, name):
    """Feeding the reference's own factors isolates the scoring path: lists must match the
    reference's lists except where its f64 scores are tied to within fp32 resolution."""
    g = golden(name)
    model = _svd_model(g)
    f = model.data.fields
    model.factors = {f.userid: None, f.itemid: g["item_factors"].copy(), "singular_values": g["singular_values"]}
    model._is_ready = True
    for kernel in ("simt", "tcgen05"):
        model.score_kernel = kernel
        model._recommendations = None
        recs = model.get_recommendations()
        assert (recs == g["recs"]).mean() > 0.995, kernel
        model.topk = 25
        model.rank = int(g["rank_reduced"])          # rank truncation without rebuild (models.py:819-832)
        recs25 = model.get_recommendations()
        assert (recs25 == g["recs_top25"]).mean() > 0.995, kernel
        model.topk = 10
        assert (model.get_recommendations() == g["recs_reduced"]).mean() > 0.995
        model.filter_seen = False
        assert (model.get_recommendations() == g["recs_unfiltered"]).mean() > 0.995
        model.filter_seen = True
        model.factors = {f.userid: None, f.itemid: g["item_factors"].copy(), "singular_values": g["singular_values"]}
        model._rank = int(g["rank"])


@pytest.mark.parametrize("name,flat", [("coffee_small", None), ("coffee_flat34", [2, 3])])
def test_coffee_model_reproduces_reference(golden, name, flat):
    from polara_b200.host import ArrayData
    from polara_b200.models import B200CoffeeModel
    g = golden(name)
    model = B200CoffeeModel(ArrayData.from_golden(g))
    model.verbose = False
    model.mlrank = tuple(int(x) for x in g["mlrank"])
    model.seed = int(g["seed"])
    model.num_iters = int(g["num_iters"])
    model.growth_tol = float(g["growth_tol"])
    if flat is not None:
        model.flattener = flat
    model.build()
    for key, ref in (("userid", "u0"), ("itemid", "u1"), ("rating", "u2")):
        assert subspace_gap(model.factors[key], g[ref]) < 2e-2, key
    np.testing.assert_allclose(np.linalg.norm(model.factors["core"]), np.linalg.norm(g["core"]), rtol=1e-3)
    assert model.factors["core"].shape == g["core"].shape
    recs = model.get_recommendations()
    assert (recs == g["recs"]).mean() > 0.95
    # scoring alone, from the reference's factors: near-exact
    f = model.data.fields
    model.factors = {f.userid: g["u0"], f.itemid: g["u1"], f.feedback: g["u2"], "core": g["core"]}
    recs = model.get_recommendations()
    assert (recs == g["recs"]).mean() > 0.995


def test_threshold_zero_feedback_stays_seen():
    """models.py:191-211: zeroed (sub-threshold) feedback is dropped from P but still masked."""
    from polara_b200.host import ArrayData
    from polara_b200.models import B200SVDModel
    rng = np.random.default_rng(0)
    v = np.linalg.qr(rng.standard_normal((30, 4)))[0]
    user = np.array([0, 0, 0, 1, 1]); item = np.array([3, 7, 9, 1, 2])
    fdbk = np.array([5.0, 0.0, 4.0, 0.0, 3.0])
    data = ArrayData(np.zeros((1, 2), dtype=np.int64), np.ones(1), (2, 30), user, item, fdbk, (2, 30), warm_start=True)
    model = B200SVDModel(data)
    model.verbose = False
    model.rank = 4
    model.topk = 5
    model.factors = {"userid": None, "itemid": v, "singular_values": np.ones(4)}
    model._is_ready = True
    recs = model.get_recommendations()
    ref = po.recommend_svd(user, item, fdbk, (2, 30), v, topk=5)
    np.testing.assert_array_equal(recs, ref)
    assert 7 not in recs[0] and 1 not in recs[1]


def test_missing_inputs_raise():
    from polara_b200.host import ArrayData
    from polara_b200.models import B200SVDModel
    data = ArrayData(np.zeros((1, 2), dtype=np.int64), np.ones(1), (2, 30))
    model = B200SVDModel(data)
    with pytest.raises(NotImplementedError):
        model.build(operator=object())
    model.factors = {"userid": None, "itemid": np.zeros((30, 4)), "singular_values": np.ones(4)}
    with pytest.raises(ValueError):
        model.get_recommendations()        # no test data (data.py:840-841)


def test_streamed_fast_path_matches_plain():
    """The pinned-CSR fast path (user chunks, H2D overlapped with scoring) returns exactly what the plain path does."""
    import scipy.sparse as sps
    import torch
    from polara_b200.host import ArrayData
    from polara_b200.models import B200SVDModel
    from polara_b200.synth import popularity_csr
    m, n = 4 * 65536 + 777, 3000
    indptr, indices, values = popularity_csr(m, n, 12 * m, seed=9)
    v = np.linalg.qr(np.random.default_rng(1).standard_normal((n, 12)))[0] * (0.9 ** np.arange(12))
    data = ArrayData(np.zeros((1, 2), dtype=np.int64), np.ones(1), (m, n))
    data.test_csr = ((torch.from_numpy(indptr).pin_memory(), torch.from_numpy(indices).pin_memory(),
                      torch.from_numpy(values).pin_memory()), (m, n))
    model = B200SVDModel(data)
    model.verbose = False
    model.rank = 12
    model.factors = {"userid": None, "itemid": v, "singular_values": np.ones(12)}
    model._is_ready = True
    streamed = model.get_recommendations()
    model.stream_chunks = 1
    single = model.get_recommendations()
    np.testing.assert_array_equal(streamed, single)
    # and the COO route (what a polara data model feeds) gives the same lists
    rows = np.repeat(np.arange(m), np.diff(indptr))
    data2 = ArrayData(np.zeros((1, 2), dtype=np.int64), np.ones(1), (m, n), rows, indices.astype(np.int64),
                      values.astype(np.float64), (m, n), warm_start=True)
    model2 = B200SVDModel(data2)
    model2.verbose = False
    model2.rank = 12
    model2.factors = {"userid": None, "itemid": v, "singular_values": np.ones(12)}
    model2._is_ready = True
    np.testing.assert_array_equal(model2.get_recommendations(), single)
    # triplets that are not sorted by user: the reference asserts (models.py:246); here the ingest kernel (inside a chunk)
    # or the cut check (across chunks) refuses
    bad = rows.copy()
    mid = len(bad) // 2
    bad[mid] += 3
    data3 = ArrayData(np.zeros((1, 2), dtype=np.int64), np.ones(1), (m, n), bad, indices.astype(np.int64),
                      values.astype(np.float64), (m, n), warm_start=True)
    model3 = B200SVDModel(data3)
    model3.verbose = False
    model3.rank = 12
    model3.factors = dict(model2.factors)
    model3._is_ready = True
    with pytest.raises((ValueError, AssertionError)):
        model3.get_recommendations()


# ---------------------------------------------------------------------------------------------------------------------
#  round-2 parity additions
# ---------------------------------------------------------------------------------------------------------------------
def _c1_data(warm=True):
    """BASELINE config C1 at its real size (ML-1M shape: 6040 x 3706, 166 ratings per user ~ 1.0e6, PureSVD rank 10): the
    same seeded generator tests/test_oracle_vs_reference.py feeds to the REAL reference; test users = the last 1208 users'
    rows (known-user style: P = their training rows)."""
    from polara_b200.host import ArrayData
    from polara_b200.synth import planted_ratings
    u, i, r = planted_ratings(6040, 3706, 166, rank=12, seed=11)
    idx = np.stack([u, i], axis=1)
    sel = u >= 6040 - 1208
    return ArrayData(idx, r, (6040, 3706), u[sel] - (6040 - 1208), i[sel], r[sel], (1208, 3706)), (u, i, r), sel


def test_c1_size_model_against_oracle():
    """C1 through the device model at full size: sigma / item subspace vs ARPACK (oracle svd_build), and every list vs the
    oracle's chunk driver on the DEVICE factors (tie-aware check on f64 scores), plus plain agreement with the lists of
    the oracle's own factors."""
    import scipy.sparse as sps
    from polara_b200.models import B200SVDModel
    from tests.helpers import check_topk_against_scores
    data, (u, i, r), sel = _c1_data()
    model = B200SVDModel(data)
    model.verbose = False
    model.rank = 10
    model.build()
    a = sps.csr_matrix((r, (u, i)), shape=(6040, 3706), dtype=np.float64)
    v_ref, s_ref, _ = po.svd_build(a, 10)
    np.testing.assert_allclose(model.factors["singular_values"], s_ref, rtol=2e-4)
    assert subspace_gap(model.factors["itemid"], v_ref) < 1e-2
    recs = model.get_recommendations()
    assert recs.shape == (1208, 10) and recs.dtype == np.int64
    tu, ti, tf = u[sel] - (6040 - 1208), i[sel], r[sel]
    v_dev64 = model.factors["itemid"].astype(np.float64)
    p = sps.csr_matrix((tf, (tu, ti)), shape=(1208, 3706))
    s64 = np.asarray(p @ v_dev64 @ v_dev64.T)
    tol = 4e-6 * np.abs(p @ v_dev64).sum(1).max() * np.abs(v_dev64).max()
    assert check_topk_against_scores(recs, s64, tu, ti, 10, tol) > 0.995
    own = po.recommend_svd(tu, ti, tf, (1208, 3706), v_ref, topk=10)
    assert (own == recs).mean() > 0.97


@pytest.mark.parametrize("name", ["svd_warm_r10", "svd_known_r8", "svd_scaled_r10"])
def test_model_lists_are_valid_topk_of_their_own_factors(golden, name):
    """The loose '> 97 % of entries equal the recorded lists' above tolerates subspace error; a systematic error must not
    hide behind it: every list is also checked as a valid top-k (tie-aware, f64) of the scores of the model's OWN factors."""
    import scipy.sparse as sps
    from tests.helpers import check_topk_against_scores
    g = golden(name)
    model = _svd_model(g, scaled=bool(g["scaled"]))
    model.build()
    recs = model.get_recommendations()
    (tu, ti, tf), shape, _ = model._get_test_data()
    v64 = model.factors["itemid"].astype(np.float64)
    keep = tf != 0
    p = sps.csr_matrix((np.asarray(tf, dtype=np.float64)[keep], (tu[keep], ti[keep])), shape=shape[:2])
    s64 = np.asarray(p @ v64 @ v64.T)
    tol = 4e-6 * max(np.abs(p @ v64).sum(1).max(), 1e-30) * np.abs(v64).max()
    assert check_topk_against_scores(recs, s64, tu, ti, model.topk, tol) > 0.995


def test_scaled_svd_rank_sweep_at_scale():
    """ScaledSVD (col_scaling 0.4, the EIGENREC setting of config C5) on 20000 x 50000: one build at rank 64, then the
    rank sweep 64 -> 48 -> 24 -> 10 WITHOUT rebuilding (models.py:819-832; pipelines.py:81-116); each rank's lists are a
    valid top-k of the truncated factors and the device copy follows the truncation."""
    import scipy.sparse as sps
    from polara_b200.host import ArrayData
    from polara_b200.models import B200ScaledSVD
    from polara_b200.synth import popularity_csr
    from tests.helpers import check_topk_against_scores
    m, n = 20000, 50000
    indptr, indices, values = popularity_csr(m, n, 60 * m, seed=21)
    user = np.repeat(np.arange(m, dtype=np.int64), np.diff(indptr))
    idx = np.stack([user, indices.astype(np.int64)], axis=1)
    sel = user < 300
    data = ArrayData(idx, values.astype(np.float64), (m, n), user[sel], indices[sel].astype(np.int64),
                     values[sel].astype(np.float64), (300, n))
    model = B200ScaledSVD(data)
    model.verbose = False
    model.col_scaling = 0.4
    model.rank = 64
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)      # flat tail at rank 64: the non-convergence warning is expected
        model.build()
    v_full = model.factors["itemid"].copy()
    a_scaled = po.scaled_training_matrix(sps.csr_matrix((values.astype(np.float64), indices, indptr), shape=(m, n)), 1, 0.4)
    # Ritz check of the leading triplets against the scaled matrix (|A v_j| = sigma_j)
    av = a_scaled @ v_full[:, :10]
    np.testing.assert_allclose(np.linalg.norm(av, axis=0), model.factors["singular_values"][:10], rtol=5e-4)
    p = sps.csr_matrix((values[sel].astype(np.float64), (user[sel], indices[sel])), shape=(300, n))   # test matrix is NOT scaled
    for rank in (64, 48, 24, 10):
        model.rank = rank
        assert model.factors["itemid"].shape == (n, rank)
        recs = model.get_recommendations()
        v64 = v_full[:, :rank].astype(np.float64)
        s64 = np.asarray(p @ v64 @ v64.T)
        tol = 4e-6 * np.abs(p @ v64).sum(1).max() * np.abs(v64).max()
        assert check_topk_against_scores(recs, s64, user[sel], indices[sel], 10, tol) > 0.995, rank


def test_dropin_classes_against_the_real_reference():
    """polara_b200.models.dropin(): our device mixins grafted on the REAL polara classes, driven by a real RecommenderData
    (needs the reference: build() installs it into oracle/_ref, which travels with the tree).  Same data object for both: singular values, subspace,
    lists and evaluate() hit counts vs polara's own SVDModel."""
    pd = pytest.importorskip("pandas")
    from oracle import ref_driver as rd
    if rd.reference_root() is None:
        pytest.skip("reference not installed (oracle/_ref)")
    rd.import_reference()
    from polara.recommender.data import RecommenderData
    from polara.recommender.models import SVDModel
    from polara_b200.models import dropin
    from polara_b200.synth import planted_ratings
    u, i, r = planted_ratings(1500, 700, 60, rank=8, seed=17)
    data = RecommenderData(pd.DataFrame({"userid": u, "itemid": i, "rating": r}), "userid", "itemid", "rating", seed=0)
    data.verbose = False
    data.prepare()
    ref = SVDModel(data); ref.verbose = False; ref.rank = 8
    ref.build()
    ref_recs = ref.get_recommendations()
    PolaraB200SVD, _, _ = dropin()
    mine = PolaraB200SVD(data); mine.verbose = False; mine.rank = 8
    mine.build()
    np.testing.assert_allclose(mine.factors["singular_values"], ref.factors["singular_values"], rtol=2e-4)
    assert subspace_gap(mine.factors[data.fields.itemid], ref.factors[data.fields.itemid]) < 1e-2
    recs = mine.get_recommendations()
    assert recs.shape == ref_recs.shape and recs.dtype == ref_recs.dtype
    assert (recs == ref_recs).mean() > 0.97
    h_ref, h_mine = ref.evaluate("hits"), mine.evaluate("hits")          # polara's own evaluate() on our lists
    assert abs(h_ref.true_positive - h_mine.true_positive) <= 3
    # scoring alone (reference factors in our class): exact up to f32 near-ties
    mine.factors = dict(ref.factors); mine._recommendations = None
    assert (mine.get_recommendations() == ref_recs).mean() > 0.995


def test_sampled_scoring_matches_numpy():
    """SURVEY.md 8(f)-1: holdout items ranked against sampled unseen items (RandomSampleEvaluationSVDMixin,
    models.py:1095-1183): gather-dot scores vs numpy f64, and the returned top-k POSITIONS vs row-wise topsort."""
    from polara_b200.host import ArrayData
    from polara_b200.models import B200SVDModel
    from polara_b200.synth import planted_ratings
    rng = np.random.default_rng(5)
    m, n, r = 700, 1500, 16
    u, i, rt = planted_ratings(m, n, 30, rank=8, seed=3)
    data = ArrayData(np.zeros((1, 2), dtype=np.int64), np.ones(1), (m, n), u, i, rt, (m, n))
    model = B200SVDModel(data)
    model.verbose = False
    model.rank = r
    model.topk = 10
    v = np.linalg.qr(rng.standard_normal((n, r)))[0] * (0.9 ** np.arange(r))
    model.factors = {"userid": None, "itemid": v, "singular_values": np.ones(r)}
    model._is_ready = True
    draw = np.argsort(rng.random((m, n)), axis=1)[:, :203]        # distinct items per user: no exactly tied scores
    holdout, unseen = draw[:, :3], draw[:, 3:]
    pos = model.sampled_recommendations(holdout, unseen)
    import scipy.sparse as sps
    e64 = sps.csr_matrix((rt, (u, i)), shape=(m, n)) @ v
    items = np.concatenate([holdout, unseen], axis=1)
    s64 = np.einsum("ur,ujr->uj", e64, v[items])
    ref = po.get_topk_elements(s64, 10)
    assert pos.shape == (m, 10)
    # positions may swap only where f64 scores are within fp32 resolution
    got = np.take_along_axis(s64, pos, axis=1)
    want = np.take_along_axis(s64, ref, axis=1)
    np.testing.assert_allclose(got, want, atol=4e-6 * np.abs(e64).sum(1).max() * np.abs(v).max())
    assert (pos == ref).mean() > 0.97


def test_coldstart_scoring_matches_numpy():
    """SURVEY.md 8(f)-3: cold-item scoring (coldstart/models.py:216-222) -- the fused kernel with roles swapped -- against
    the f64 formula, top-k over users, nothing filtered."""
    import scipy.sparse as sps
    from polara_b200.host import ArrayData
    from polara_b200.models import B200SVDModel
    from tests.helpers import check_topk_against_scores
    rng = np.random.default_rng(8)
    n_users, n_items, n_feat, n_cold, r = 900, 400, 60, 37, 12
    data = ArrayData(np.zeros((1, 2), dtype=np.int64), np.ones(1), (n_users, n_items))
    model = B200SVDModel(data)
    model.verbose = False
    model.rank = r
    model.topk = 10
    u = np.linalg.qr(rng.standard_normal((n_users, r)))[0]
    v = np.linalg.qr(rng.standard_normal((n_items, r)))[0]
    sig = np.sort(rng.random(r) + 0.5)[::-1]
    model.factors = {"userid": u, "itemid": v, "singular_values": sig}
    model._is_ready = True
    feats = sps.random(n_items, n_feat, density=0.1, random_state=1, format="csr", dtype=np.float64)
    w = np.asarray(feats.T @ v)                                  # compute_item_features_mapping, :233-236
    helper = np.linalg.pinv(w.T @ w)                             # update_item_features_transform, :192-195
    cold = sps.random(n_cold, n_feat, density=0.15, random_state=2, format="csr", dtype=np.float64)
    recs = model.coldstart_recommendations(cold, w, helper)
    s64 = (np.asarray(cold @ w) @ helper) @ (u * sig[None, :]).T
    assert recs.shape == (n_cold, 10)
    tol = 1e-5 * np.abs(s64).max()
    assert check_topk_against_scores(recs, s64, [], [], 10, tol) > 0.97


def _hybrid_setup(seed=21, m=900, n=260, per_user=30, rank=10):
    """A planted rating matrix, an SPD item-similarity matrix and its (sparse) Cholesky factor L_S -- what HybridSVD's
    CholeskyFactorsMixin produces with CHOLMOD (hybrid/models.py:234-331); numpy's dense Cholesky stands in at this size."""
    import scipy.sparse as sps
    from polara_b200.synth import planted_ratings
    user, item, val = planted_ratings(m, n, per_user, rank=rank, seed=seed)
    a = sps.csr_matrix((val.astype(np.float64), (user, item)), shape=(m, n))
    a.sum_duplicates()
    rng = np.random.default_rng(seed)
    f = rng.standard_normal((n, 6)) * (rng.random((n, 6)) < 0.5)            # sparse item features
    sim = 0.4 * (f @ f.T) / 6.0
    np.fill_diagonal(sim, 0.0)
    spd = np.eye(n) + 0.9 * sim / max(1e-9, np.abs(sim).sum(1).max())       # diagonally dominant: SPD
    chol = np.linalg.cholesky(spd)                                           # S = L L^T
    return user, item, val, a, sps.csr_matrix(chol), chol


def test_build_accepts_an_explicit_sparse_operator():
    """SVDModel.build(operator=...) (models.py:835-837) as HybridSVD uses it with precompute_auxiliary_matrix: the explicit
    product A . L_S is factorised instead of the training matrix (hybrid/models.py:364-370).  Against svds(operator)."""
    from polara_b200.host import ArrayData
    from polara_b200.models import B200SVDModel
    user, item, val, a, l_s, _ = _hybrid_setup()
    operator = (l_s.T.dot(a.T)).T.tocsr()                                    # cholesky_items.T.dot(svd_matrix.T).T
    rank = 4                                                                 # sigma_4 / sigma_5 = 1.19: a clear cut
    data = ArrayData(np.stack([user, item], axis=1), val, a.shape)
    model = B200SVDModel(data)
    model.verbose = False
    model.rank = rank
    model.build(operator=operator)
    v_ref, s_ref, _ = po.svd_build(operator, rank)
    np.testing.assert_allclose(model.factors["singular_values"], s_ref, rtol=2e-4)
    assert subspace_gap(model.factors["itemid"], v_ref) < 2e-2
    # the factors belong to the operator: its Ritz values on the returned basis are the returned singular values
    ritz = np.linalg.norm(operator @ model.factors["itemid"], axis=0)
    np.testing.assert_allclose(ritz, model.factors["singular_values"], rtol=1e-3)
    with pytest.raises(NotImplementedError):
        from scipy.sparse.linalg import aslinearoperator
        model.build(operator=aslinearoperator(operator))


def test_item_projectors_score_like_hybrid_svd():
    """HybridSVD.slice_recommendations (hybrid/models.py:390-394): scores = P . vr . vl^T with vr = L_S v, vl = L_S^-T v
    (build_item_projector, 315-325).  A model that carries the two projectors is scored that way on the device; rank
    truncation cuts them with the other factors (round_item_projector, 341-350)."""
    import scipy.sparse as sps
    from polara_b200.host import ArrayData
    from polara_b200.models import B200SVDModel
    from tests.helpers import check_topk_against_scores
    user, item, val, a, l_s, chol = _hybrid_setup(seed=33)
    rank, k = 10, 10
    v, s, _ = po.svd_build((l_s.T.dot(a.T)).T.tocsr(), rank)
    vl, vr = po.hybrid_item_projectors(chol, v)
    order = np.lexsort((item, user))                                         # test triplets come sorted by user
    data = ArrayData(np.stack([user, item], axis=1), val, a.shape, test_user=user[order], test_item=item[order],
                     test_fdbk=val[order], test_shape=a.shape)
    model = B200SVDModel(data)
    model.verbose = False
    model.rank = rank
    model.factors = {"userid": None, "itemid": v, "singular_values": s,
                     "itemid_projector_left": vl, "itemid_projector_right": vr}
    model._is_ready = True
    model.topk = k
    recs = model.get_recommendations()
    p = sps.csr_matrix((val.astype(np.float64), (user, item)), shape=a.shape)
    scores = po.hybrid_slice_scores(p, vl, vr)
    tol = 4e-6 * np.abs(np.asarray(p.dot(vr))).sum(1).max() * np.abs(vl).max()
    assert check_topk_against_scores(recs, scores, user, item, k, tol) > 0.99
    # with the plain factors on both sides the lists differ: the projectors were really used
    plain = np.asarray(p.dot(v)).dot(v.T)
    plain[user, item] = -np.inf
    assert (np.sort(recs, 1) != np.sort(np.argsort(-plain, 1)[:, :k], 1)).any()
    # rank truncation (models.py:819-832 + hybrid/models.py:341-350)
    model.rank = 6
    assert model.factors["itemid_projector_left"].shape[1] == 6 and model.factors["itemid_projector_right"].shape[1] == 6
    recs6 = model.get_recommendations()
    scores6 = po.hybrid_slice_scores(p, vl[:, :6], vr[:, :6])
    assert check_topk_against_scores(recs6, scores6, user, item, k, tol) > 0.99
