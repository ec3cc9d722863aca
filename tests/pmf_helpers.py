"""Helpers of the ProbabilisticMF tests (CPU side): the known-user split of the ``ref_pmf`` fixture and the
interactions in the reference's order."""
import numpy as np
import scipy.sparse as sps

from polara_b200.synth import planted_ratings


def planted(g):
    n_users, n_items, per_user, rank, seed = (int(x) for x in g["planted"])
    return planted_ratings(n_users, n_items, per_user, rank=rank, seed=seed)


def replay_known_split(user, item, fdbk, g):
    """What the reference's ``RecommenderData.prepare()`` with ``warm_start = False`` hands a model for the ratings
    ``(user, item, fdbk)``, rebuilt from the split recorded in ``g`` (oracle/make_golden_pmf.py ``_record_known_split``):
    ``(train, test)`` triplets in the data model's new indices.  Training keeps every row that is not held out;
    ``test_to_coo`` then returns the training rows of the test users (the users with held-out rows), in the same
    order."""
    def index_of(old, size):
        new = np.full(size, -1, dtype=np.int64)
        new[old] = np.arange(len(old))
        return new
    new_user = index_of(g["user_old"], user.max() + 1)[user]
    new_item = index_of(g["item_old"], item.max() + 1)[item]
    train = (new_user >= 0) & (new_item >= 0)
    train[g["holdout_rows"]] = False
    tr = (new_user[train], new_item[train], fdbk[train])
    test = np.isin(tr[0], g["test_users"])
    return tr, tuple(a[test] for a in tr)


def reference_interactions(user, item, fdbk, shape):
    """``get_training_matrix(sparse_format='coo', dtype='f8')`` followed by ``.nonzero()`` (models.py:743-746):
    ``(rows, cols, vals, row_nnz, col_nnz)`` in row-major order, duplicates summed.  Without zero values the indices
    and ``matrix.data`` stay aligned."""
    a = sps.coo_matrix((np.asarray(fdbk, dtype=np.float64), (user, item)), shape=tuple(int(s) for s in shape))
    a.sum_duplicates()
    rows, cols = a.nonzero()
    assert len(rows) == len(a.data), "zero-valued interactions: the reference misaligns indices and values"
    return rows, cols, a.data, a.getnnz(axis=1), a.getnnz(axis=0)
