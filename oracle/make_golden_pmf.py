"""Generate ``tests/golden/ref_pmf.npz`` by running the REAL reference's ProbabilisticMF (the polara checkout
``oracle.ref_shim.REFERENCE_ROOT`` names).  TEST INFRASTRUCTURE, a companion of oracle/make_golden.py.

    POLARA_REFERENCE_ROOT=<polara checkout> python oracle/make_golden_pmf.py
"""
import os
import sys

import numpy as np
import pandas as pd

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from oracle.make_golden import _hits, _planted, _save, _small_int  # noqa: E402
from oracle.ref_shim import import_reference  # noqa: E402
from tests.helpers import ratings_digest  # noqa: E402
from tests.pmf_helpers import replay_known_split  # noqa: E402


def _record_known_split(data, planted):
    """The split ``RecommenderData.prepare()`` made of the ratings ``planted_ratings(*planted)`` with
    ``warm_start = False`` (known users): the user and item indices, the original rows held out and the test users
    (new indices).  tests/pmf_helpers.py ``replay_known_split`` turns it back into the data model's arrays."""
    def old_by_new(frame):
        return _small_int(frame.sort_values("new")["old"].to_numpy())
    f = data.fields
    return dict(planted=np.array(planted), planted_sha256=np.array(ratings_digest(*_planted(planted))),
                user_old=old_by_new(data.index.userid.training), item_old=old_by_new(data.index.itemid),
                holdout_rows=np.sort(data.test.holdout.index.to_numpy()).astype(np.int32),
                test_users=np.unique(data.test.holdout[f.userid].to_numpy()).astype(np.int64))


def ref_pmf():
    """ProbabilisticMF (models.py:728-787) on an 800 x 400 planted split with known users: the defaults (all 25 epochs)
    and a raised tolerance (the early stop fires), both from seed 5.  Factors are stored in float64: the SGD sweep is
    reproduced exactly, so nothing is lost to rounding."""
    import_reference()
    from polara.recommender.data import RecommenderData
    from polara.recommender.models import ProbabilisticMF
    planted = (800, 400, 30, 6, 5)
    u, i, r = _planted(planted)
    data = RecommenderData(pd.DataFrame({"userid": u, "itemid": i, "rating": r}), "userid", "itemid", "rating", seed=0)
    data.verbose = False
    data.warm_start = False
    data.prepare()
    g = _record_known_split(data, planted)
    idx, val, shp = data.to_coo(tensor_mode=False)
    test = data.test_to_coo(tensor_mode=False)
    (tr_u, tr_i, tr_f), (ts_u, ts_i, ts_f) = replay_known_split(u, i, r, g)
    for got, want in zip((tr_u, tr_i, tr_f, ts_u, ts_i, ts_f), (idx[:, 0], idx[:, 1], val) + tuple(test)):
        np.testing.assert_array_equal(got, want)
    out = dict(train_shape=np.array(shp), test_shape=np.array(data.get_test_shape(tensor_mode=False)), **g)
    for tag, tolerance in (("default", None), ("early", 0.02)):
        model = ProbabilisticMF(data, seed=5)
        model.verbose = False
        if tolerance is not None:
            model.tolerance = tolerance
        model.build()
        f = data.fields
        out.update({"%s_P" % tag: model.factors[f.userid], "%s_Q" % tag: model.factors[f.itemid],
                    "%s_rmse" % tag: np.array(model.rmse_history), "%s_tolerance" % tag: np.array(model.tolerance),
                    "%s_recs" % tag: _small_int(model.get_recommendations())})
        if tolerance is None:
            out["default_hits"] = _hits(model)
    out.update(seed=np.array(5), rank=np.array(10), learn_rate=np.array(0.005), sigma=np.array(1.0),
               num_epochs=np.array(25))
    assert len(out["default_rmse"]) == 25 and len(out["early_rmse"]) < 25
    _save("ref_pmf", **out)


if __name__ == "__main__":
    ref_pmf()
