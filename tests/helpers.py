"""Shared test helpers (CPU side)."""
import numpy as np
import scipy.sparse as sps

from oracle import polara_oracle as po


def subspace_gap(v_a, v_b):
    s = np.linalg.svd(np.asarray(v_a, dtype=np.float64).T @ np.asarray(v_b, dtype=np.float64), compute_uv=False)
    return float(np.sqrt(max(0.0, 1.0 - s.min() ** 2)))


def check_topk_against_scores(ids, scores64, seen_rows, seen_cols, k, tol):
    """``ids`` [m x k] must be, for every row, a valid top-k of the f64 oracle scores under
    the reference's order (unseen by score desc, then seen by score desc), allowing swaps
    only between items whose oracle scores differ by less than ``tol`` (fp32 near-ties).
    Returns the fraction of entries that agree exactly with the oracle order."""
    m, n = scores64.shape
    seen = sps.csr_matrix((np.ones(len(seen_rows), dtype=bool), (seen_rows, seen_cols)), shape=(m, n)).toarray() \
        if len(seen_rows) else np.zeros((m, n), dtype=bool)
    exact = 0
    for u in range(m):
        ref = po.rank_key_order(scores64[u], np.flatnonzero(seen[u]), k)
        mine = ids[u]
        assert len(set(mine.tolist())) == k, "duplicate items in row %d" % u
        n_unseen = n - seen[u].sum()
        # seen items may only appear after all unseen ones are exhausted
        assert not seen[u][mine[:min(k, n_unseen)]].any(), "seen item recommended in row %d" % u
        s_ref = scores64[u][ref]
        s_mine = scores64[u][mine]
        key_ref = np.where(seen[u][ref], -1e30, 0) + s_ref
        key_mine = np.where(seen[u][mine], -1e30, 0) + s_mine
        np.testing.assert_allclose(key_mine, key_ref, rtol=0, atol=tol,
                                   err_msg="row %d is not a top-%d within tolerance" % (u, k))
        exact += (mine == ref).sum()
    return exact / (m * k)


def ratings_digest(user, item, fdbk):
    """sha256 of seeded ratings (int64 user and item ids, float64 feedback): a fixture that stores a split instead of
    the ratings records it, so that a change of the generator shows as changed inputs, not as a disagreement."""
    import hashlib
    h = hashlib.sha256()
    for a, dtype in ((user, np.int64), (item, np.int64), (fdbk, np.float64)):
        h.update(np.ascontiguousarray(a, dtype=dtype).tobytes())
    return h.hexdigest()


def replay_split(user, item, fdbk, g):
    """What the reference's ``RecommenderData.prepare()`` hands a model for the ratings ``(user, item, fdbk)``, rebuilt
    from the split it recorded in the fixture ``g`` (oracle/make_golden.py ``_record_split``): ``(train, test)``, each a
    ``(user, item, fdbk)`` triplet in the data model's new indices and in the original row order.  Training keeps the
    rows of the training users, test keeps the test users' rows that are not held out and whose item is in training.
    Feedback values are passed through unchanged."""
    def index_of(old, size):
        new = np.full(size, -1, dtype=np.int64)
        new[old] = np.arange(len(old))
        return new
    tr_user = index_of(g["train_user_old"], user.max() + 1)[user]
    ts_user = index_of(g["test_user_old"], user.max() + 1)[user]
    new_item = index_of(g["item_old"], item.max() + 1)[item]
    train = tr_user >= 0
    test = (ts_user >= 0) & (new_item >= 0)
    test[g["holdout_rows"]] = False
    return ((tr_user[train], new_item[train], fdbk[train]),
            (ts_user[test], new_item[test], fdbk[test]))


def random_seen_csr(rng, m, n, per_row):
    rows, cols = [], []
    for u in range(m):
        c = np.sort(rng.choice(n, size=min(n, per_row[u]), replace=False))
        rows.append(np.full(len(c), u))
        cols.append(c)
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    indptr = np.zeros(m + 1, dtype=np.int64)
    np.cumsum(np.bincount(rows, minlength=m), out=indptr[1:])
    return rows, cols, indptr
