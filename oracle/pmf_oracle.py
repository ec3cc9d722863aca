"""CPU oracle for ProbabilisticMF  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A numpy restatement (written from the algorithm, not copied) of the reference's SGD sweep and of the stratified order in
which the device build applies it.  Like ``oracle/polara_oracle.py`` it is imported only by ``tests/``,
``__graft_entry__.smoke()`` and the benchmarks; the product path never imports it.  Pinned against recorded reference
runs (``oracle/make_golden_pmf.py`` -> ``tests/golden/ref_pmf.npz``, checked in tests/test_pmf.py).
"""
from __future__ import annotations

import numpy as np

__all__ = ["pmf_sgd", "sgd_strata_bounds", "sgd_strata_permutation"]


def pmf_sgd(rows, cols, vals, shape, row_nnz, col_nnz, rank, learn_rate=0.005, sigma=1, num_epochs=25, tol=1e-4,
            seed=None, order=None):
    """ProbabilisticMF.build (models.py:743-770) -> simple_pmf_sgd -> mf_sgd_boilerplate -> generalized_sgd_sweep
    (lib/optimize.py:123-250) with the identity transform and no gradient adjustment.  ``rows, cols, vals`` are the
    interactions in the reference's order (``coo.sum_duplicates()`` then ``.nonzero()``: row-major); ``order`` (optional)
    is a permutation of them, applied to every epoch's sweep.  ``row_nnz`` / ``col_nnz`` are ``getnnz(axis=1/0)``.
    Returns ``(P, Q, rmse_history)``; the loop stops early as the reference does."""
    rnds = np.random if seed is None else np.random.RandomState(seed)
    P = rnds.normal(scale=0.1, size=(int(shape[0]), rank))
    Q = rnds.normal(scale=0.1, size=(int(shape[1]), rank))
    lambd = 0.5 * sigma ** 2
    row_lambda = lambd / np.asarray(row_nnz)          # elementwise: the same IEEE division as per interaction
    col_lambda = lambd / np.asarray(col_nnz)
    rows, cols, vals = np.asarray(rows), np.asarray(cols), np.asarray(vals, dtype=np.float64)
    if order is not None:
        rows, cols, vals = rows[order], cols[order], vals[order]
    triplets = list(zip(rows.tolist(), cols.tolist(), vals.tolist()))
    nnz = len(triplets)
    last_err = np.finfo("f8").max
    history = []
    for _ in range(num_epochs):
        cum_error = 0
        for m, n, a in triplets:
            p, q = P[m], Q[n]
            err = a - p @ q
            gp = err * q - p * row_lambda[m]
            gq = err * p - q * col_lambda[n]        # both gradients from the rows before the update
            P[m] = p + learn_rate * gp
            Q[n] = q + learn_rate * gq
            cum_error += err * err
        refined = abs(last_err - cum_error) / last_err
        last_err = cum_error
        history.append(np.sqrt(cum_error / nnz))
        if refined < tol:
            break
    return P, Q, history


def sgd_strata_bounds(counts, strata):
    """Contiguous ranges of rows (or columns) with balanced nnz, by the rule DESIGN.md 3.6 states: range b < B-1 ends
    after the first row whose cumulative nnz reaches ceil((b+1) * nnz / B); the last range ends at the last row.
    Returns the B + 1 bounds.  Written as a scan, independently of the device path's vectorised cut."""
    total = int(np.sum(counts))
    bounds, cum, b = [0], 0, 0
    for i, c in enumerate(np.asarray(counts).tolist()):
        cum += c
        while b < strata - 1 and cum * strata >= (b + 1) * total:      # cum >= ceil((b+1) total / B), integers
            bounds.append(i + 1)
            b += 1
    while len(bounds) < strata:
        bounds.append(len(counts))
    bounds.append(len(counts))
    return np.array(bounds, dtype=np.int64)


def sgd_strata_permutation(rows, cols, row_nnz, col_nnz, strata):
    """The order in which the stratified device epoch applies the interactions ``(rows, cols)`` (given in reference
    order): sub-epoch s takes the blocks (b, (b + s) mod B), b = 0..B-1, in that order, each block in reference order.
    Returns the permutation (an index array into the interactions)."""
    def block_of(counts):
        bounds = sgd_strata_bounds(counts, strata)
        out = np.empty(len(counts), dtype=np.int64)
        for b in range(strata):
            out[bounds[b]:bounds[b + 1]] = b
        return out
    rb = block_of(row_nnz)[np.asarray(rows)]
    cb = block_of(col_nnz)[np.asarray(cols)]
    sub = (cb - rb) % strata
    return np.lexsort((np.arange(len(rb)), rb, sub))
