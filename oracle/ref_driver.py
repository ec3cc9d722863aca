"""Drive the UNMODIFIED reference (evfro/polara) on plain arrays  --  TEST INFRASTRUCTURE.

Used by ``bench.py --impl reference`` / the ``cpu_baseline`` leg (timing the reference's
own CPU path on the host cores) and by the drop-in tests.  The reference is imported
from ``oracle/_ref`` (the git-ignored install ``build()`` makes with oracle/install_ref.py,
so it goes wherever the tree is copied) or else from the checkout ``oracle.ref_shim``
names.
Nothing of ``polara_b200`` (models, kernels, engine) is on this path.

The reference's models read their inputs from a ``RecommenderData`` object
(polara/recommender/data.py); its splitting / re-indexing logic is out of scope
(SURVEY.md §2), so :class:`StubData` replays what that object hands to a model:
``to_coo`` (data.py:794-817), ``test_to_coo`` (data.py:835-862), ``get_test_shape``
(data.py:865-884), ``fields``, ``warm_start`` and the event hooks (data.py:35-76).
"""
from __future__ import annotations

import os
import sys
import time
from collections import namedtuple

import numpy as np

from oracle.install_ref import TARGET as _INSTALLED
from oracle.ref_shim import REFERENCE_ROOT as _CHECKOUT

_REF_CANDIDATES = (_INSTALLED, _CHECKOUT)

Fields = namedtuple("Fields", "userid itemid feedback")
_Index = namedtuple("Index", "userid itemid feedback")
_Test = namedtuple("TestData", "testset holdout")


def reference_root():
    for root in _REF_CANDIDATES:
        if root and os.path.isdir(os.path.join(root, "polara")):
            return root
    return None


def import_reference():
    """Returns the reference's ``polara`` package (pandas>=3 shim applied, reference untouched)."""
    root = reference_root()
    if root is None:
        raise ImportError("reference not found (looked in %s)" % ", ".join(str(r) for r in _REF_CANDIDATES))
    from oracle.ref_shim import _apply_pandas_shim
    _apply_pandas_shim()
    if root not in sys.path:
        sys.path.insert(0, root)
    import polara  # noqa: F401
    return polara


class StubData:
    """What a model reads from ``RecommenderData`` (see module docstring).  ``test`` is the user-sorted triplet
    ``(user_idx, item_idx, feedback)`` the reference's ``test_to_coo`` returns; ``train`` is ``(idx [nnz x 2], val)``."""

    on_change_event = "on_change"
    on_update_event = "on_update"

    def __init__(self, shape, test=None, train=None, warm_start=True, fields=("userid", "itemid", "rating"),
                 holdout=None):
        self.fields = Fields(*fields)
        self._shape = tuple(int(s) for s in shape)
        self._test, self._train = test, train
        self.warm_start = warm_start
        self.test_sample = None
        self.holdout_size = 3
        self.test = _Test(None, holdout)
        self.index = _Index(None, np.empty((self._shape[1], 2)), None)

    def subscribe(self, event, callback):          # data.py:35-76 -- a frozen replay never fires
        pass

    def to_coo(self, tensor_mode=False, feedback_threshold=None):
        idx, val = self._train
        return idx, val, self._shape

    def test_to_coo(self, tensor_mode=False, feedback_threshold=None):
        return self._test

    def get_test_shape(self, tensor_mode=False):
        return self._shape


def csr_to_test_triplets(indptr, indices, values):
    """host CSR -> the (user_idx intp, item_idx intp, feedback f64) arrays of test_to_coo (data.py:849-862)."""
    n = len(indptr) - 1
    user = np.repeat(np.arange(n, dtype=np.intp), np.diff(indptr))
    return user, np.asarray(indices).astype(np.intp), np.asarray(values).astype(np.float64)


def make_svd_model(data, item_factors, topk=10, filter_seen=True):
    """The reference's ``SVDModel`` with given factors (no build): ``get_recommendations()`` then runs the stock
    chunk driver (models.py:391-405) -> slice_recommendations (857-861) -> downvote_seen_items (494-519) ->
    get_topk_elements (522-564)."""
    import_reference()
    from polara.recommender.models import SVDModel
    model = SVDModel(data)
    model.verbose = False
    model.verify_integrity = False                 # the stub has no training frame to verify against
    model.topk = topk
    model.filter_seen = filter_seen
    model._rank = item_factors.shape[1]
    model.factors = {data.fields.userid: None, data.fields.itemid: item_factors,
                     "singular_values": np.ones(item_factors.shape[1])}
    model._is_ready = True
    return model


def set_knobs(memory_hard_limit=None):
    """the reference's chunking knob (polara/recommender/defaults.py:51, read at utils.py:34-36)."""
    import_reference()
    from polara.recommender import defaults
    old = defaults.memory_hard_limit
    if memory_hard_limit is not None:
        defaults.memory_hard_limit = memory_hard_limit
    return old


def time_reference_scoring(model, max_chunks=None, max_seconds=None):
    """Runs the reference's own per-chunk recommender (``_slice_recommender``, models.py:359-371, through
    ``run_sequential_recommender`` / ``run_parallel_recommender``, models.py:374-388) over the FIRST chunks of the
    user range with the FULL test arrays in place -- so every chunk pays what it pays in the full job, including the
    O(nnz_total) mask of ``_slice_test_data`` (models.py:260-270).  Returns users scored, seconds, chunk size."""
    test_data, test_shape, test_users = model._get_test_data()
    slices_idx = model._get_slices_idx(test_shape)
    slices = list(zip(slices_idx[:-1], slices_idx[1:]))
    chunk = int(slices_idx[1] - slices_idx[0])
    workers = model.max_test_workers
    if max_chunks is not None:
        slices = slices[:max_chunks]
    top_recs = np.empty((test_shape[0], model.topk), dtype=np.int64)
    t0 = time.perf_counter()
    done = 0
    if workers and len(slices) > 1:
        model.run_parallel_recommender(top_recs, slices, test_data, test_shape, test_users)
        done = int(slices[-1][1] - slices[0][0])
    else:
        for sl in slices:
            model.run_sequential_recommender(top_recs, [sl], test_data, test_shape, test_users)
            done += int(sl[1] - sl[0])
            if max_seconds is not None and time.perf_counter() - t0 > max_seconds:
                break
    dt = time.perf_counter() - t0
    return dict(users=done, seconds=dt, chunk_users=chunk, chunks=(done + chunk - 1) // chunk,
                recs=top_recs[:done])


def host_description():
    """what BASELINE.md §2 asks to print with every CPU result."""
    info = {"cores": os.cpu_count()}
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    info["cpu"] = line.split(":", 1)[1].strip()
                    break
    except OSError:
        pass
    try:
        import numba
        info["numba_threads"] = int(numba.config.NUMBA_NUM_THREADS)
        info["numba"] = numba.__version__
    except Exception:
        pass
    try:
        from threadpoolctl import threadpool_info
        info["blas_threads"] = max([p.get("num_threads", 0) for p in threadpool_info()] or [0])
    except Exception:
        pass
    import scipy
    info["numpy"], info["scipy"] = np.__version__, scipy.__version__
    return info
