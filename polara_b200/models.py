"""B200 drop-ins for the reference's SVDModel / ScaledSVD / CoffeeModel hot path.

``build()`` and ``get_recommendations()`` run entirely on the device through the C-ABI
(:mod:`polara_b200.engine`); host code only converts the data model's COO arrays to CSR
and moves buffers.  There is no CPU fallback: without the CUDA library or an sm_100
device every call raises.

Two families of classes share the device logic (mixins below):

* ``B200SVDModel`` / ``B200ScaledSVD`` / ``B200CoffeeModel`` -- stand-alone, built on the
  mirror base in :mod:`polara_b200.host` (works without the reference installed);
* :func:`dropin` -- the same mixins grafted onto the *real* ``polara`` classes when that
  package is importable, so that ``polara.evaluation`` pipelines keep working unchanged.
"""
from __future__ import annotations

import time

import numpy as np
import torch

from . import host
from .engine import DeviceCSR, get_engine, round_up

__all__ = ["B200SVDModel", "B200ScaledSVD", "B200CoffeeModel", "B200ProbabilisticMF", "dropin", "dropin_pmf",
           "default_ell", "DEFAULT_SGD_STRATA"]


def default_ell(rank, oversample=None):
    """Subspace width of the randomized range finder: rank + max(22, rank/2), rounded to 32."""
    p = max(22, rank // 2) if oversample is None else oversample
    return min(1024, round_up(rank + p, 32))


def _pinned(arr):
    t = torch.from_numpy(np.ascontiguousarray(arr))
    try:
        return t.pin_memory()
    except RuntimeError:
        return t


def _as_index_array(x):
    """index arrays cross PCIe as int64 (what ``to_coo`` / ``test_to_coo`` produce: np.intp, data.py:815,849)."""
    x = np.asarray(x)
    return x if x.dtype == np.int64 else x.astype(np.int64)


def _as_value_array(x):
    x = np.asarray(x)
    return x if x.dtype in (np.float32, np.float64) else x.astype(np.float64)


class _DeviceModelMixin:
    """State shared by the device models: engine handle and cached device buffers."""

    _engine = None
    score_kernel = None          # None = engine default; 'simt' | 'tcgen05'
    last_timings = None

    @property
    def engine(self):
        if self._engine is None:
            self._engine = get_engine()
        return self._engine

    @property
    def recommendations(self):
        """models.py:100-108, plus: on an item-sharded model ``get_recommendations()`` returns the lists of the users this
        rank owns; the cached ``recommendations`` (what ``evaluate()`` consumes, aligned with the holdout rows) are the
        lists of ALL users, all-gathered once."""
        if self._recommendations is None:
            if not self._is_ready:
                if self.verbose:
                    print("{} model is not ready. Rebuilding.".format(self.method))
                self.build()
            recs = self.get_recommendations()
            shard = getattr(self, "shard", None)
            if shard is not None and shard.world > 1:
                from .dist import gather_lists
                recs = gather_lists(recs, shard, None, self.engine.device)      # user count = sum of the ranks' shares
            self._recommendations = recs
        return self._recommendations

    def _device_factor(self, key, width_multiple=32):
        """Device copy [n x ld] (zero padded to a multiple of 32 columns) of the numpy factor
        ``self.factors[key]``; re-uploaded whenever the host array object changes (rank
        truncation, models.py:819-832, replaces the array by a view)."""
        host_arr = self.factors[key]
        cache = self.__dict__.setdefault("_dev_cache", {})
        hit = cache.get(key)
        if hit is not None and hit[0] is host_arr:
            return hit[1]
        r = host_arr.shape[1]
        ld = round_up(r, width_multiple)
        buf = np.zeros((host_arr.shape[0], ld), dtype=np.float32)
        buf[:, :r] = host_arr
        dev = self.engine.upload(buf)
        cache[key] = (host_arr, dev)
        return dev

    def _remember_device_factor(self, key, host_arr, dev):
        self.__dict__.setdefault("_dev_cache", {})[key] = (host_arr, dev)

    # ----- test data -> device CSR --------------------------------------------------
    def _test_csr_device(self, test_data, shape, values=None, stream_arrays=None, sorted_users=False):
        """Device CSR of the test matrix P (zero feedback dropped, models.py:197-201; duplicates summed, models.py:208-210)
        and the (indptr, indices) pair of the *seen* pattern (ALL triplets, models.py:191-196,211), built on the device
        from the triplets of ``_get_test_data`` (pb200_coo_to_csr).  ``values`` (CoFFee: per-triplet weights, the feedback
        there is an index, never "zero feedback") replaces the feedback as matrix values; nothing is dropped then."""
        eng = self.engine
        n_users, n_items = int(shape[0]), int(shape[1])
        if stream_arrays is None:
            user, item, fdbk = test_data
        if stream_arrays is not None:
            u_d, i_d, f_d, w_d = stream_arrays
        else:
            u_d, i_d = eng.upload(_as_index_array(user)), eng.upload(_as_index_array(item))
            f_d = None if values is not None else eng.upload(_as_value_array(fdbk))
            w_d = None if values is None else eng.upload(_as_value_array(values))
        if w_d is None:
            p = eng.coo_to_csr(u_d, i_d, f_d, (n_users, n_items), drop_zeros=True, require_sorted_rows=sorted_users)
        else:
            p = eng.coo_to_csr(u_d, i_d, w_d, (n_users, n_items), drop_zeros=False)
        if p.nnz == int(u_d.shape[0]):
            seen = (p.indptr, p.indices)          # nothing dropped, nothing merged: same pattern
        else:
            s = eng.coo_to_csr(u_d, i_d, None, (n_users, n_items), drop_zeros=False)
            seen = (s.indptr, s.indices)
        return p, seen

    def _item_projector_device(self, v_dev):
        """HybridSVD scores with two item-side matrices, ``scores = P . vr . vl^T`` (hybrid/models.py:390-394:
        ``<itemid>_projector_right`` folds the history in, ``<itemid>_projector_left`` scores); a model that carries them
        in ``factors`` is scored the same way, everything else with the item factors on both sides."""
        itemid = self.data.fields.itemid
        vl = self.factors.get("%s_projector_left" % itemid)
        vr = self.factors.get("%s_projector_right" % itemid)
        if vl is None or vr is None:
            return v_dev, v_dev
        if getattr(self, "shard", None) is not None:
            raise NotImplementedError("item projectors on an item-sharded model")
        return self._device_factor("%s_projector_right" % itemid), self._device_factor("%s_projector_left" % itemid)

    def _score(self, p_dev: DeviceCSR, seen_dev, v_dev, rank, topk):
        eng = self.engine
        if self.score_kernel is not None:
            eng.set_score_kernel(self.score_kernel)
        v_fold, v_dev = self._item_projector_device(v_dev)
        e = eng.spmm(p_dev, v_fold, ell=v_fold.shape[1])    # padded width: the unpredicated SpMM variant is the faster one
        seen = seen_dev if self.filter_seen else None
        shard = getattr(self, "shard", None)
        if shard is not None:
            # item-factor sharding: returns the lists of the user range this rank owns
            from .dist import sharded_topk
            ids = sharded_topk(eng, e, v_dev, rank, topk, seen, shard, p_dev.shape[0])
            lo, hi = shard.user_range(p_dev.shape[0])
            return ids[: hi - lo]
        return eng.score_topk(e, v_dev, rank, topk, seen=seen)


class _SVDDeviceMixin(_DeviceModelMixin):
    """Device implementation of SVDModel.build / get_recommendations
    (polara/recommender/models.py:835-861, 391-405)."""

    oversample = None        # subspace width = rank + oversample (None -> default_ell)
    power_iters = 12         # cap on subspace iterations
    tol = 1e-6               # stop when the leading Ritz values move less than this (relative) ...
    vec_tol = 1e-3           # ... and the leading-rank subspaces of two successive iterates are this close (sine bound)
    rsvd_seed = 1

    def _training_csr_device(self):
        data = self.data
        fast = getattr(data, "train_csr", None)
        if fast is not None:
            indptr, indices, values, shape = fast
        else:
            # the triplets of RecommenderData.to_coo go to the device as they are; the CSR is built there
            idx, val, shape = data.to_coo(tensor_mode=False, feedback_threshold=self.feedback_threshold)
            idx = _as_index_array(idx)
            val = _as_value_array(val)
            self._n_train_users = int(shape[0])
            rows = self._build_rows(shape[0])
            if rows is not None:
                # row-sharded build: this rank ingests only its block of user rows (re-based)
                keep = (idx[:, 0] >= rows[0]) & (idx[:, 0] < rows[1])
                idx = idx[keep] - np.array([rows[0], 0], dtype=np.int64)
                val = val[keep]
                shape = (rows[1] - rows[0], shape[1])
            eng = self.engine
            idx_d = eng.upload(np.ascontiguousarray(idx))
            a = eng.coo_to_csr(idx_d[:, 0], idx_d[:, 1], eng.upload(val), shape)
            return self._scaled(a)
        self._n_train_users = int(shape[0])
        rows = self._build_rows(shape[0])
        if rows is not None:
            # row-sharded build: this rank keeps (and copies to its GPU) only its block of user rows
            indptr, indices, values, shape = csr_row_block(indptr, indices, values, shape, rows[0], rows[1])
        a = self.engine.upload_csr(indptr, indices, values, shape)
        return self._scaled(a)

    def _scaled(self, a):
        row_s = getattr(self, "row_scaling", 1)
        col_s = getattr(self, "col_scaling", 1) if hasattr(self, "_col_scaling") else 1
        if hasattr(self, "_col_scaling"):
            self.engine.rescale(a, row_s, col_s)      # ScaledMatrixMixin, models.py:891-895
        return a

    def _build_rows(self, n_users):
        """user rows this rank factorises when the build is sharded (``self.shard`` set, world > 1), else None."""
        shard = getattr(self, "shard", None)
        if shard is None or shard.world <= 1 or not self.shard_build:
            return None
        return shard.user_range(n_users)

    def build(self, operator=None, return_factors="vh"):
        """models.py:835-855.  ``operator`` (``svd_matrix = operator``, models.py:836-837): an EXPLICIT sparse matrix of the
        training matrix's shape is factorised in its place -- what HybridSVD passes with ``precompute_auxiliary_matrix``
        (``L_K^T A L_S`` formed on the host, hybrid/models.py:364-370).  The matrix-free ``LinearOperator`` form wraps CHOLMOD
        solves on the host (hybrid/models.py:372-388) and has no device counterpart: NotImplementedError, as before."""
        op_csr = None
        if operator is not None:
            import scipy.sparse as sps
            if not sps.issparse(operator):
                raise NotImplementedError("only an explicit sparse matrix is accepted as `operator` on the device path "
                                          "(HybridSVD: set precompute_auxiliary_matrix = True); a LinearOperator is not")
            if self._build_rows(1) is not None:
                raise NotImplementedError("row-sharded build of an explicit operator")
            op_csr = sps.csr_matrix(operator)
            op_csr.sum_duplicates()
            op_csr.sort_indices()
        eng = self.engine
        sharded = self._build_rows(1) is not None
        if sharded:
            import torch.distributed as dist
            eng.set_reduce_hook(dist.all_reduce)       # sums Gram matrices / A^T W panels / column counts over ranks
        try:
            self._build_factors(eng, return_factors, sharded, op_csr)
        finally:
            if sharded:
                eng.set_reduce_hook(None)

    def _build_factors(self, eng, return_factors, sharded, op_csr=None):
        t0 = time.perf_counter()
        if op_csr is None:
            a = self._training_csr_device()
        else:
            a = eng.upload_csr(op_csr.indptr.astype(np.int64), op_csr.indices.astype(np.int32),
                               op_csr.data.astype(np.float32), op_csr.shape)
            self._n_train_users = op_csr.shape[0]
        at = eng.transpose(a)
        rank = self.rank
        ell = default_ell(rank, self.oversample)
        ell = min(ell, round_up(min(a.shape), 32)) if min(a.shape) >= 32 else 32
        # panel-major copies where the dense operand of a product would not stay L2-resident (A^T W gathers user rows:
        # 1e6 x 96 floats = 384 MB at C2); format conversion, part of the preparation like the transpose
        at = eng.block_columns(at, eng.panel_cols_for(at.shape[1], ell))
        a = eng.block_columns(a, eng.panel_cols_for(a.shape[1], ell))
        want_u = return_factors is True
        eng.sync()
        t1 = time.perf_counter()
        v, sigma, u, iters = eng.rsvd(a, at, rank, ell, max_iters=self.power_iters, tol=self.tol, vec_tol=self.vec_tol,
                                      seed=self.rsvd_seed, want_u=want_u)
        eng.sync()
        info = dict(eng.last_rsvd_info)
        if not info["converged"]:
            import warnings
            warnings.warn("%s: subspace iteration stopped at the cap of %d iterations -- leading Ritz values still move by "
                          "%.1e (tol %.1e), successive-subspace sine bound %.1e (tol %.1e).  The factors are the best "
                          "rank-%d subspace found, not a converged one (flat spectrum at the cut?); raise power_iters or "
                          "oversample." % (self.method, self.power_iters, info["value_change"], self.tol,
                                           info["angle_bound"], self.vec_tol, rank), RuntimeWarning, stacklevel=3)
        if sharded and u is not None:
            u = self._gather_user_rows(u)
        t2 = time.perf_counter()
        if self.training_time is not None:
            self.training_time.append(t2 - t1)       # what track_time covers, models.py:843
        if self.verbose:
            print("{} training time: {:.3f}s".format(self.method, t2 - t1))
        f = self.data.fields
        v_host = v[:, :rank].cpu().numpy().astype(np.float64)
        self.factors[f.userid] = None if u is None else u[:, :rank].cpu().numpy().astype(np.float64)
        self.factors[f.itemid] = v_host
        self.factors["singular_values"] = sigma.cpu().numpy()
        self._remember_device_factor(f.itemid, v_host, v)
        self.last_timings = dict(prepare_s=t1 - t0, rsvd_s=t2 - t1, subspace_iters=iters, ell=ell,
                                 panels=(a.n_panels, at.n_panels), converged=info["converged"],
                                 value_change=info["value_change"], angle_bound=info["angle_bound"])

    shard_build = True       # with ``self.shard`` set (world > 1) factorise row blocks in parallel (SURVEY.md 8e)

    def _gather_user_rows(self, u_local):
        """assemble the user factors from the row blocks of all ranks (one broadcast per rank)."""
        import torch.distributed as dist
        shard = self.shard
        n_users = self._n_train_users
        full = torch.empty((n_users, u_local.shape[1]), dtype=u_local.dtype, device=u_local.device)
        lo, hi = shard.user_range(n_users)
        full[lo:hi].copy_(u_local)
        c = shard.user_chunk(n_users)
        for src in range(shard.world):
            a, b = min(n_users, src * c), min(n_users, (src + 1) * c)
            if b > a:
                dist.broadcast(full[a:b], src=src)
        return full

    stream_chunks = None     # user chunks of the pinned-CSR fast path (H2D of chunk i+1 overlaps scoring of chunk i);
                             # None = stream_schedule(), an int = that many equal chunks

    def get_recommendations(self):
        if self.verify_integrity and hasattr(self, "verify_data_integrity"):
            self.verify_data_integrity()
        eng = self.engine
        fast = getattr(self.data, "test_csr", None)
        if fast is not None:
            (indptr, indices, values), shape = fast
            if self.topk > shape[1]:
                raise ValueError("topk exceeds the number of items")
            if getattr(self, "shard", None) is None and isinstance(indptr, torch.Tensor) and shape[0] >= 4 * 65536:
                return self._streamed_recommendations(indptr, indices, values, shape)
            if getattr(self, "shard", None) is not None and isinstance(indptr, torch.Tensor):
                return self._sharded_recommendations(indptr, indices, values, shape)
            t0 = time.perf_counter()
            p_dev = eng.upload_csr(indptr, indices, values, shape[:2])
            seen_dev = (p_dev.indptr, p_dev.indices)
        else:
            # the route a Polara user takes: triplets of test_to_coo (sorted by user) -> device ingest -> scoring
            big = self._big_test_triplets()
            if big is not None:
                test_data, shape = big
                if self.topk > shape[1]:
                    raise ValueError("topk exceeds the number of items")
                return self._streamed_recommendations(None, None, None, shape, triplets=test_data)
            test_data, shape, _ = self._get_test_data()
            if self.topk > shape[1]:
                raise ValueError("topk exceeds the number of items")   # np.argpartition would raise, models.py:490
            t0 = time.perf_counter()
            p_dev, seen_dev = self._test_csr_device(test_data, shape)
        v_dev = self._device_factor(self.data.fields.itemid)
        if getattr(self, "profile_phases", False):
            torch.cuda.synchronize()
        t1 = time.perf_counter()
        ids = self._score(p_dev, seen_dev, v_dev, self.factors[self.data.fields.itemid].shape[1], self.topk)
        if getattr(self, "profile_phases", False):
            torch.cuda.synchronize()
        t2 = time.perf_counter()
        out = ids.cpu().numpy()
        self.last_score_timings = dict(h2d_s=t1 - t0, score_s=t2 - t1, d2h_s=time.perf_counter() - t2)
        return out

    def _big_test_triplets(self):
        """Large test sets skip the host-side passes of ``_get_test_data`` (models.py:227-257: np.diff over all triplets
        for the sortedness assert and the gap test -- four passes over 1e8 int64 cost more than the whole device path).
        The same facts are established differently: the ingest kernel checks the order of every chunk on the device (and
        sorts if it has to), and users that start at 0 and end at n_test_users - 1 leave no room for a gap because
        ``get_test_shape`` counts the distinct test users (data.py:865-884).  Anything else returns None and takes the
        reference's path."""
        if getattr(self, "shard", None) is not None:
            return None
        data = self.data
        shape = data.get_test_shape(tensor_mode=False)
        if shape[0] < 4 * 65536:
            return None
        threshold = None if data.warm_start else self.feedback_threshold
        user, item, fdbk = data.test_to_coo(tensor_mode=False, feedback_threshold=threshold)
        if len(user) == 0 or int(user[0]) != 0 or int(user[-1]) != shape[0] - 1:
            return None
        return (user, item, fdbk), shape

    def _sharded_recommendations(self, indptr, indices, values, shape):
        """Item-sharded scoring from a pinned host CSR that every rank holds: each rank copies only ITS slice of the rows
        over PCIe, the slices are exchanged GPU-to-GPU (one broadcast per rank over NVLink) so that every GPU ends up with
        the whole test matrix (needed for the user embeddings and the seen lists), then SpMM + fused scoring on the own
        item shard + all-to-all + merge.  Returns the lists of the user range this rank owns."""
        import torch.distributed as dist
        eng, shard = self.engine, self.shard
        m, n_items = shape[0], shape[1]
        rank_r = self.factors[self.data.fields.itemid].shape[1]
        v_dev = self._device_factor(self.data.fields.itemid)
        self._item_projector_device(v_dev)                    # raises for a model that carries item projectors
        if self.score_kernel is not None:
            eng.set_score_kernel(self.score_kernel)
        indptr64 = indptr if indptr.dtype == torch.int64 else indptr.to(torch.int64)
        world = shard.world
        chunk_u = shard.user_chunk(m)
        row_bounds = [min(m, c * chunk_u) for c in range(world + 1)]       # the user ranges the ranks own (ItemShard)
        nnz_bounds = [int(indptr64[b]) for b in row_bounds]
        nnz = nnz_bounds[-1]
        prof = getattr(self, "profile_phases", False)
        tp = [time.perf_counter()]

        def mark():
            if prof:
                torch.cuda.synchronize()
                tp.append(time.perf_counter())
        ip_dev = indptr64.to(eng.device, non_blocking=True)
        ix_dev = torch.empty(nnz, dtype=torch.int32, device=eng.device)
        lo, hi = nnz_bounds[shard.rank], nnz_bounds[shard.rank + 1]
        ix_dev[lo:hi].copy_(indices[lo:hi], non_blocking=True)
        vl_blk = values[lo:hi].to(eng.device, non_blocking=True)        # values are needed for the own row block only
        mark()
        for src in range(world):
            a, b = nnz_bounds[src], nnz_bounds[src + 1]
            if b > a:
                dist.broadcast(ix_dev[a:b], src=src)                     # the seen lists of ALL users are needed everywhere
        from .dist import gather_embeddings, sharded_topk
        mark()
        # user embeddings: every rank multiplies its block of rows, the blocks are all-gathered (SURVEY.md 8e)
        r_lo, r_hi = row_bounds[shard.rank], row_bounds[shard.rank + 1]
        ip_blk = ip_dev[r_lo:r_hi + 1].clone()
        eng.shift_i64(ip_blk, -lo)
        p_block = DeviceCSR(ip_blk, ix_dev[lo:hi], vl_blk if vl_blk.dtype == torch.float32 else vl_blk.to(torch.float32),
                            (r_hi - r_lo, n_items))
        e = gather_embeddings(eng, p_block, v_dev, shard, m)
        seen = (ip_dev, ix_dev) if self.filter_seen else None
        ids = sharded_topk(eng, e, v_dev, rank_r, self.topk, seen, shard, m)
        mark()
        u_lo, u_hi = shard.user_range(m)
        out_t = torch.empty((u_hi - u_lo, self.topk), dtype=torch.int64, pin_memory=True)
        out_t.copy_(ids[: u_hi - u_lo], non_blocking=True)
        torch.cuda.current_stream(eng.device).synchronize()
        out = out_t.numpy()
        mark()
        if prof:
            self.last_score_timings = dict(zip(("h2d_s", "assemble_s", "score_s", "d2h_s"), np.diff(tp).round(4)))
        return out

    def _streamed_recommendations(self, indptr, indices, values, shape, triplets=None):
        """Host test data -> recommendations in user chunks: the H2D copy of chunk i+1 (side stream) overlaps ingest +
        SpMM + fused scoring of chunk i (context stream); results go back into one pinned buffer on a third stream.
        Two sources: a pinned host CSR (``data.test_csr``) or, with ``triplets``, the user-sorted
        ``(user, item, feedback)`` arrays of ``test_to_coo`` -- what a Polara data model hands over -- which are
        converted to CSR on the device chunk by chunk (pb200_coo_to_csr)."""
        t_entry = time.perf_counter()
        eng = self.engine
        m, n_items = shape[0], shape[1]
        rank = self.factors[self.data.fields.itemid].shape[1]
        v_dev = self._device_factor(self.data.fields.itemid)
        v_fold, v_score = self._item_projector_device(v_dev)
        if self.score_kernel is not None:
            eng.set_score_kernel(self.score_kernel)
        if self.stream_chunks is None:
            sms = torch.cuda.get_device_properties(eng.device).multi_processor_count
            bounds = stream_schedule(m, sms * 128)
        else:
            n_chunks = max(1, int(self.stream_chunks))
            bounds = [m * c // n_chunks for c in range(n_chunks + 1)]
        n_chunks = len(bounds) - 1
        # fresh pinned result buffer: torch's caching host allocator re-uses the block once the previous result is
        # garbage-collected, so steady-state calls pay neither cudaHostAlloc nor page faults, and results never alias
        out = torch.empty((m, self.topk), dtype=torch.int64, pin_memory=True)
        main = torch.cuda.current_stream(eng.device)
        side = self.__dict__.setdefault("_copy_stream", torch.cuda.Stream(device=eng.device))
        back = self.__dict__.setdefault("_result_stream", torch.cuda.Stream(device=eng.device))
        prof = [] if getattr(self, "profile_phases", False) else None
        if triplets is None:
            indptr64 = indptr if indptr.dtype == torch.int64 else indptr.to(torch.int64)
            cuts = [int(indptr64[b]) for b in bounds]
            host = (indices, values)
        else:
            user, item, fdbk = (np.asarray(x) for x in triplets)
            cuts = [int(c) for c in np.searchsorted(user, np.asarray(bounds))]
            # the chunks are cut on the assumption that the triplets are sorted by user (the reference asserts it,
            # models.py:246): inside a chunk the ingest kernel verifies it, across the cuts it is verified here
            for bnd, cut in zip(bounds[1:-1], cuts[1:-1]):
                if (cut > 0 and user[cut - 1] >= bnd) or (cut < len(user) and user[cut] < bnd):
                    raise AssertionError("calculations assume testset is sorted by users!")
            host = tuple(torch.from_numpy(x) for x in (_as_index_array(user), _as_index_array(item), _as_value_array(fdbk)))

        def upload(c):
            a, b = bounds[c], bounds[c + 1]
            lo, hi = cuts[c], cuts[c + 1]
            with torch.cuda.stream(side):
                if triplets is None:
                    dev = (indptr64[a:b + 1].to(eng.device, non_blocking=True),) + \
                        tuple(t[lo:hi].to(eng.device, non_blocking=True) for t in host)
                else:
                    dev = tuple(t[lo:hi].to(eng.device, non_blocking=True) for t in host)
                ev = torch.cuda.Event(enable_timing=prof is not None)
                ev.record(side)
            return (dev, ev, a, b, lo)

        t_host0 = time.perf_counter()

        def mark(stream):
            ev_ = torch.cuda.Event(enable_timing=True)
            ev_.record(stream)
            return ev_

        side.wait_stream(main)
        if prof is not None:
            ev_start = mark(main)
        nxt = upload(0)
        keep = []
        for c in range(n_chunks):
            dev, ev, a, b, lo = nxt
            if c + 1 < n_chunks:
                nxt = upload(c + 1)
            main.wait_event(ev)
            if prof is not None:
                prof.append(["chunk%d" % c, ev, mark(main), None, None, time.perf_counter() - t_host0])
            for t in dev:
                t.record_stream(main)                      # allocated on the side stream, consumed on the main one
            if triplets is None:
                ip, ix, vl = dev
                eng.shift_i64(ip, -lo)                     # re-base the row pointers of the chunk
                p_dev = DeviceCSR(ip, ix if ix.dtype == torch.int32 else ix.to(torch.int32),
                                  vl if vl.dtype == torch.float32 else vl.to(torch.float32), (b - a, n_items))
                seen = (p_dev.indptr, p_dev.indices)
            else:
                u_d, i_d, f_d = dev
                eng.shift_i64(u_d, -a)                     # users of the chunk count from 0
                p_dev, seen = self._test_csr_device(None, (b - a, n_items), stream_arrays=(u_d, i_d, f_d, None),
                                                    sorted_users=True)
            e = eng.spmm(p_dev, v_fold, ell=v_fold.shape[1])
            ids = eng.score_topk(e, v_score, rank, self.topk, seen=seen if self.filter_seen else None)
            if prof is not None:
                prof[-1][3] = mark(main)
            scored = torch.cuda.Event()
            scored.record(main)
            with torch.cuda.stream(back):                  # results leave on their own stream / copy engine
                back.wait_event(scored)
                out[a:b].copy_(ids, non_blocking=True)
                done = torch.cuda.Event(enable_timing=prof is not None)
                done.record(back)
            if prof is not None:
                prof[-1][4] = done
            keep.append((p_dev, seen, e, ids))
        main.synchronize()
        back.synchronize()
        if prof is not None:
            # per chunk, ms after the start of the call: upload done, compute start, compute end, D2H done, host enqueue time
            self.last_score_timings = {
                "host_total_ms": (time.perf_counter() - t_host0) * 1e3, "setup_ms": (t_host0 - t_entry) * 1e3,
                "chunks": [[name, ev_start.elapsed_time(up), ev_start.elapsed_time(c0), ev_start.elapsed_time(c1),
                            ev_start.elapsed_time(d1), host_t * 1e3] for name, up, c0, c1, d1, host_t in prof]}
        return out.numpy()

    # ---- sampled evaluation (RandomSampleEvaluationSVDMixin, models.py:1095-1183) ---------------------------------------
    def sampled_recommendations(self, holdout_items, unseen_items, test_data=None, shape=None):
        """Rank every test user's holdout items against a sample of unseen items (the EIGENREC protocol): scores of the
        ``[n_users x holdout_size]`` holdout items and of the ``[n_users x n_unseen]`` sampled items come from one
        gather-dot over the resident factors (pb200_gather_dot = inner_product_at, lib/sparse.py:58-72), then the top-k
        POSITIONS in the concatenated ``[holdout | unseen]`` row are returned (``np.apply_along_axis(topsort, ...)``,
        models.py:1182): position < holdout_size means a holdout item was ranked there."""
        eng = self.engine
        if test_data is None:
            test_data, shape, _ = self._get_test_data()
        f = self.data.fields
        p_dev, _ = self._test_csr_device(test_data, shape)
        v_dev = self._device_factor(f.itemid)
        r_live = self.factors[f.itemid].shape[1]
        e = eng.spmm(p_dev, v_dev, ell=r_live)                       # user_factors = test_matrix.dot(item_factors), :1158
        items = np.concatenate([np.asarray(holdout_items, dtype=np.int64).reshape(shape[0], -1),
                                np.asarray(unseen_items, dtype=np.int64).reshape(shape[0], -1)], axis=1)
        if self.topk > items.shape[1]:
            raise ValueError("topk exceeds the number of sampled items")
        users = np.broadcast_to(np.arange(shape[0], dtype=np.int64)[:, None], items.shape)
        scores = eng.gather_dot(e, v_dev, r_live, eng.upload(np.ascontiguousarray(users)), eng.upload(items))
        return eng.topk_dense(scores, self.topk).cpu().numpy()

    # ---- item cold start (ItemColdStartSVDModelMixin.slice_recommendations, coldstart/models.py:216-222) ---------------
    def coldstart_recommendations(self, cold_item_features, feature_embeddings, transform_helper):
        """Top-k USERS for cold items: ``scores = (F_cold W) (W^T W)^+ (U diag(sigma))^T`` followed by
        ``get_topk_elements`` over users, ``filter_seen = False`` (coldstart/models.py:13-18, 216-222) -- the fused kernel
        with the roles swapped: the cold items' factors are the left operand, ``U diag(sigma)`` the right one.
        ``cold_item_features``: scipy sparse / dense [n_cold x n_features]; ``feature_embeddings`` W [n_features x r];
        ``transform_helper`` (W^T W)^+ [r x r] (``_item_features_transform_helper``).  Needs the user factors
        (``build(return_factors=True)``)."""
        import scipy.sparse as sps_
        eng = self.engine
        f = self.data.fields
        u = self.factors.get(f.userid, None)
        if u is None:
            raise ValueError("cold start needs the user factors: build(return_factors=True)")
        s = np.asarray(self.factors["singular_values"])
        r = u.shape[1]
        w = np.asarray(feature_embeddings)[:, :r] @ np.asarray(transform_helper)[:r, :r]      # fold the r x r map into W
        fc = sps_.csr_matrix(cold_item_features)
        fc.sort_indices()
        ld = round_up(r, 32)
        w_pad = np.zeros((w.shape[0], ld), dtype=np.float32); w_pad[:, :r] = w
        us = np.zeros((u.shape[0], ld), dtype=np.float32); us[:, :r] = u * s[None, :r]
        f_dev = eng.upload_csr(fc.indptr.astype(np.int64), fc.indices.astype(np.int32), fc.data.astype(np.float32), fc.shape)
        e = eng.spmm(f_dev, eng.upload(w_pad), ell=ld)                      # cold item factors [n_cold x r]
        if self.topk > u.shape[0]:
            raise ValueError("topk exceeds the number of users")
        return eng.score_topk(e, eng.upload(us), r, self.topk, seen=None).cpu().numpy()

    def slice_recommendations(self, test_data, shape, start, stop, test_users=None):
        """Dense score rows for a (small) user slice -- kept for the single-user helpers
        (models.py:277-293,324-356).  Returns ``(scores float64 [m x n_items], slice_data)``."""
        user, item, fdbk = test_data
        sel = (user >= start) & (user < stop)
        sl = (user[sel] - start, item[sel], fdbk[sel])
        eng = self.engine
        p_dev, _ = self._test_csr_device(sl, (stop - start, shape[1]))
        v_dev = self._device_factor(self.data.fields.itemid)
        r_live = self.factors[self.data.fields.itemid].shape[1]
        e = eng.spmm(p_dev, v_dev, ell=r_live)
        s = eng.score_dense(e, v_dev, r_live)
        return s.cpu().numpy().astype(np.float64), sl


def round_tucker_core(core, mode, rank):
    """Rank reduction of one mode of a Tucker core (CoffeeModel.round_core, models.py:966-980): thin SVD of the mode
    unfolding, keep the leading ``rank`` directions.  Returns ``(rotation [r_mode x rank], new_core)``.  Host numpy on
    purpose: the core is a few thousand numbers (<= 60 x 60 x 5) and the reference does this on the host as well."""
    moved = np.moveaxis(np.asarray(core), mode, 0)                  # [r_mode, remaining modes in their order]
    flat = moved.reshape((moved.shape[0], -1), order="F")
    u, s, vt = np.linalg.svd(flat, full_matrices=False)
    small = (s[:rank, None] * vt[:rank]).reshape((rank,) + moved.shape[1:], order="F")
    return u[:, :rank], np.moveaxis(small, 0, mode)


def csr_row_block(indptr, indices, values, shape, lo, hi):
    """rows [lo, hi) of a host CSR (numpy arrays or torch tensors) as a CSR of its own (views, re-based pointers)."""
    a, b = int(indptr[lo]), int(indptr[hi])
    return indptr[lo:hi + 1] - a, indices[a:b], values[a:b], (hi - lo, shape[1])


def stream_schedule(m, unit, first=0.06, growth=1.6):
    """Chunk bounds for the streamed path.  Chunks are whole waves of the scoring grid (``unit`` users = one 128-user
    tile per SM); the first is small so that little of the upload is exposed, each next one grows by at most ``growth``
    (< compute time / upload time per user, so the copy of chunk i+1 always hides behind the scoring of chunk i)."""
    waves = m / float(unit)
    if waves <= 2.0:
        return [0, m]
    size = max(1.0, round(waves * first))
    bounds, done = [0], 0.0
    while True:
        rest = waves - done
        if rest <= size * (1.0 + growth):              # the remainder fits one last chunk without starving the pipeline
            bounds.append(m)
            return bounds
        done += size
        bounds.append(int(done) * unit)
        size = float(int(size * growth + 0.999))


class _SVDState:
    """rank handling of SVDModel (models.py:802-832)."""

    def _init_svd_state(self):
        self._rank = host.DEFAULTS["svd_rank"]
        self.method = "PureSVD"
        self.factors = {}

    @property
    def rank(self):
        return self._rank

    @rank.setter
    def rank(self, new_value):
        if new_value != self._rank:
            self._rank = new_value
            self._check_reduced_rank(new_value)
            self._recommendations = None

    def _check_reduced_rank(self, rank):
        for entity, factor in self.factors.items():
            if factor is None:
                continue
            if factor.shape[-1] < rank:
                self._is_ready = False
                self.factors = dict.fromkeys(self.factors.keys())
                break
            else:
                self.factors = dict(**self.factors)
                self.factors[entity] = factor[..., :rank]


class B200SVDModel(_SVDDeviceMixin, _SVDState, host.RecommenderModel):
    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self._init_svd_state()

    def build(self, operator=None, return_factors="vh"):
        return _SVDDeviceMixin.build(self, operator=operator, return_factors=return_factors)


class B200ScaledSVD(B200SVDModel):
    """ScaledMatrixMixin + SVDModel (models.py:864-898)."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self._col_scaling = 0.4
        self._row_scaling = 1
        self.method = f"{self.method}-s"

    @property
    def col_scaling(self):
        return self._col_scaling

    @col_scaling.setter
    def col_scaling(self, new_value):
        if new_value != self._col_scaling:
            self._col_scaling = new_value
            self._recommendations = None

    @property
    def row_scaling(self):
        return self._row_scaling

    @row_scaling.setter
    def row_scaling(self, new_value):
        if new_value != self._row_scaling:
            self._row_scaling = new_value
            self._recommendations = None


# ------------------------------------------------------------------ CoFFee ----------
def flatten_weights(w, flattener):
    """``flatten_scores(w.T, flattener)`` (models.py:983-1006,1052) for the flatteners that are
    linear in the scores; returns the vector ``wt_flat`` [r2]."""
    wt = np.asarray(w).T
    if flattener is None:
        flattener = slice(None)
    if isinstance(flattener, str):
        if flattener not in ("sum", "mean"):
            raise NotImplementedError("only linear flatteners run on the device path")
        return getattr(np, flattener)(wt, axis=-1)
    if isinstance(flattener, int):
        return wt[..., flattener]
    if isinstance(flattener, (list, slice)):
        return np.sum(wt[..., flattener], axis=-1)
    if isinstance(flattener, tuple):
        sl, how = flattener
        if how not in ("sum", "mean"):
            raise NotImplementedError("only linear flatteners run on the device path")
        return getattr(np, how)(wt[..., sl or slice(None)], axis=-1)
    raise NotImplementedError("callable flatteners need dense tensor scores; not available on the device path")


class _CoffeeDeviceMixin(_DeviceModelMixin):
    """Device implementation of CoffeeModel.build (-> hooi, polara/lib/tensor.py:37-96) and
    CoffeeModel scoring (models.py:1042-1054)."""

    def _hooi_device(self, idx, val, shape, mlrank, init=None):
        """HOOI (polara/lib/tensor.py:37-96) on the device.  With ``self.shard`` set (world > 1) the nnz are sharded by
        user (SURVEY.md 8e): the mode-0 unfolding and ``u0`` hold this rank's users only (its Gram matrix is summed over
        the ranks inside pb200_tall_svd), the mode-1 / mode-2 TTM outputs are all-reduced and factored redundantly."""
        eng = self.engine
        r0, r1, r2 = mlrank
        n0, n1, n2 = (int(s) for s in shape)
        shard = getattr(self, "shard", None)
        sharded = shard is not None and shard.world > 1
        n0_all = n0
        if sharded:
            import torch.distributed as dist
            lo, hi = shard.user_range(n0)
            keep = (idx[:, 0] >= lo) & (idx[:, 0] < hi)
            idx = idx[keep].copy()
            idx[:, 0] -= lo
            val = np.asarray(val)[keep]
            n0 = hi - lo
        i0 = eng.upload(idx[:, 0].astype(np.int32))
        i1 = eng.upload(idx[:, 1].astype(np.int32))
        i2 = eng.upload(idx[:, 2].astype(np.int32))
        vals = eng.upload(np.asarray(val, dtype=np.float32))
        g0 = eng.coo_group(i0, n0, i1, i2, vals)        # seg, i1, i2, val grouped by user
        g1 = eng.coo_group(i1, n1, i0, i2, vals)        # grouped by item
        g2 = eng.coo_group(i2, n2, i0, i1, vals)        # grouped by feedback level
        if init is None:
            # same start as the reference (lib/tensor.py:57-63): RandomState(seed).rand + QR, on the host
            rs = np.random if self.seed is None else np.random.RandomState(self.seed)
            u1 = np.linalg.qr(rs.rand(n1, r1), mode="reduced")[0]
            u2 = np.linalg.qr(rs.rand(n2, r2), mode="reduced")[0]
        else:
            u1, u2 = init
        u1_d = eng.upload(np.ascontiguousarray(u1, dtype=np.float32))
        u2_d = eng.upload(np.ascontiguousarray(u2, dtype=np.float32))
        norm_old = 0.0
        trace = []
        for it in range(self.num_iters):
            # mode 0: res[i0, a(u2), b(u1)]  (ttm(..., u2, u1, ((2,0),(1,0))), tensor.py:70)
            unf = eng.ttm(n0, g0[0], g0[2], g0[1], g0[3], u2_d, r2, u1_d, r1)
            if sharded:
                eng.set_reduce_hook(dist.all_reduce)                 # rows of the unfolding are sharded: global Gram matrix
            try:
                u0_d, _, _ = self._tall_svd(unf, r2 * r1, r0)
            finally:
                if sharded:
                    eng.set_reduce_hook(None)
            # mode 1: res[i1, a(u2), b(u0)]  (tensor.py:74)
            unf = eng.ttm(n1, g1[0], g1[2], g1[1], g1[3], u2_d, r2, u0_d, r0)
            if sharded:
                dist.all_reduce(unf)                                  # every rank holds part of every item's nnz
            u1_d, _, _ = self._tall_svd(unf, r2 * r0, r1)
            # mode 2: res[i2, a(u1), b(u0)] (tensor.py:78) -- few huge segments; work on the transpose
            small = eng.ttm_reduce(n2, g2[0], g2[2], g2[1], g2[3], u1_d, r1, u0_d, r0)     # [n2 x r1*r0]
            if sharded:
                dist.all_reduce(small)
            small_t = small.t().contiguous()                                                 # [r1*r0 x n2]
            vv_d, ss, uut = self._tall_svd(small_t, n2, r2, want_vt=True)                    # left vecs of M^T = vv
            u2_d = uut.t().contiguous()                                                      # [n2 x r2]
            ss_h = ss.cpu().numpy()
            norm_new = float(np.linalg.norm(ss_h))
            trace.append(norm_new)
            growth = (norm_new - norm_old) / norm_new
            norm_old = norm_new
            if growth < self.growth_tol:
                break
        # core (tensor.py:90-92): rows of (ss * vv^T) are already descending here
        vv = vv_d[:, :r2].cpu().numpy().astype(np.float64)            # [r1*r0 x r2]
        core = (ss_h[:, None] * vv.T).reshape(r2, r1, r0).transpose(2, 1, 0)
        to_host = lambda t, r: t[:, :r].cpu().numpy().astype(np.float64)   # noqa: E731
        if sharded:
            full = torch.zeros((n0_all, u0_d.shape[1]), dtype=u0_d.dtype, device=u0_d.device)
            full[lo:hi].copy_(u0_d)
            dist.all_reduce(full)                                     # assemble the user factors (disjoint row blocks)
            u0_d = full
        return to_host(u0_d, r0), to_host(u1_d, r1), to_host(u2_d, r2), np.ascontiguousarray(core), trace

    def _tall_svd(self, m, width, rank, want_vt=False):
        eng = self.engine
        u, s, vt = eng.tall_svd(m if m.shape[1] == width else m[:, :width], rank, want_vt=want_vt)
        return u, s, vt

    def build(self):
        idx, val, shp = self.data.to_coo(tensor_mode=True)
        t0 = time.perf_counter()
        u0, u1, u2, core, trace = self._hooi_device(idx, val, shp, self.mlrank)
        self.engine.sync()
        t1 = time.perf_counter()
        if self.training_time is not None:
            self.training_time.append(t1 - t0)
        if self.verbose:
            print("{} training time: {:.3f}s".format(self.method, t1 - t0))
        f = self.data.fields
        self.factors[f.userid] = u0
        self.factors[f.itemid] = u1
        self.factors[f.feedback] = u2
        self.factors["core"] = core
        self.core_norm_trace = trace

    def get_recommendations(self):
        if self.verify_integrity and hasattr(self, "verify_data_integrity"):
            self.verify_data_integrity()
        eng = self.engine
        f = self.data.fields
        test_data, shape, _ = self._get_test_data()
        user, item, fdbk_idx = test_data
        w = self.factors[f.feedback]
        # E[u,:] = sum_{(i,f) in u} (w[f,:] . wt_flat) v[i,:]   (SURVEY.md §8a row A9)
        c = np.asarray(w) @ flatten_weights(w, self.flattener)
        weights = c[np.asarray(fdbk_idx, dtype=np.int64)].astype(np.float32)
        if self.topk > shape[1]:
            raise ValueError("topk exceeds the number of items")
        p_dev, seen_dev = self._test_csr_device((user, item, None), shape, values=weights)
        v_dev = self._device_factor(f.itemid)
        ids = self._score(p_dev, seen_dev, v_dev, self.factors[f.itemid].shape[1], self.topk)
        return ids.cpu().numpy()


class B200CoffeeModel(_CoffeeDeviceMixin, host.RecommenderModel):
    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self._mlrank = host.DEFAULTS["mlrank"]
        self.factors = {}
        self.method = "CoFFee"
        self._flattener = host.DEFAULTS["flattener"]
        self.growth_tol = host.DEFAULTS["growth_tol"]
        self.num_iters = host.DEFAULTS["num_iters"]
        self.show_output = False
        self.seed = None
        self.parallel_ttm = True

    @property
    def mlrank(self):
        return self._mlrank

    @mlrank.setter
    def mlrank(self, new_value):
        if new_value != self._mlrank:
            self._mlrank = new_value
            self._check_reduced_rank(new_value)
            self._recommendations = None

    def _check_reduced_rank(self, mlrank):
        """models.py:949-963: lowering a mode's rank rotates its factor and shrinks the core (no rebuild); raising it
        invalidates the model."""
        for mode, entity in enumerate(self.data.fields):
            factor = self.factors.get(entity, None)
            if factor is None:
                continue
            rank = mlrank[mode]
            if factor.shape[1] < rank:
                self._is_ready = False
                self.factors = {}
                break
            if factor.shape[1] > rank:
                self.factors = dict(self.factors)             # a backup of the old dict stays untouched
                rotation, self.factors["core"] = round_tucker_core(self.factors["core"], mode, rank)
                self.factors[entity] = factor.dot(rotation)

    round_core = staticmethod(round_tucker_core)

    @property
    def flattener(self):
        return self._flattener

    @flattener.setter
    def flattener(self, new_value):
        if new_value != self._flattener:
            self._flattener = new_value
            self._recommendations = None

    def build(self):
        return _CoffeeDeviceMixin.build(self)


# ------------------------------------------------------------- ProbabilisticMF ------
DEFAULT_SGD_STRATA = 1024     # user / item ranges of the stratified SGD epoch (DESIGN.md 3.6: chosen at C2 on a B200)


def _padded_f32(arr, width_multiple=32):
    r = arr.shape[1]
    buf = np.zeros((arr.shape[0], round_up(r, width_multiple)), dtype=np.float32)
    buf[:, :r] = arr
    return buf


class _PMFDeviceMixin(_DeviceModelMixin):
    """Device implementation of ProbabilisticMF.build / get_recommendations (polara/recommender/models.py:728-787).
    ``build()`` runs the reference's SGD sweep (lib/optimize.py:123-250) in fp64 on the device, in a stratified order
    whose ``sgd_strata`` user and item ranges let disjoint blocks run concurrently (pb200_sgd_epoch, DESIGN.md 3.6);
    ``sgd_strata = 1`` is the reference's own order.  Scoring is the fused kernel on ``P[test_users]`` and ``Q``."""

    sgd_strata = DEFAULT_SGD_STRATA   # changes the result like ``seed`` does: part of the algorithm, not a speed switch

    def _check_device_pmf(self, args, kwargs):
        if args or kwargs:
            raise NotImplementedError("ProbabilisticMF.build arguments %s (gradient adjusters such as adjust_gradient) "
                                      "are not on the device path" % (list(args) + sorted(kwargs),))
        opt = getattr(self, "optimizer", None)
        if opt is not None and (getattr(opt, "__name__", None), getattr(opt, "__module__", None)) != \
                ("simple_pmf_sgd", "polara.lib.optimize"):
            raise NotImplementedError("optimizer %r is not on the device path: only simple_pmf_sgd is" % (opt,))
        shard = getattr(self, "shard", None)
        if shard is not None and shard.world > 1:
            raise NotImplementedError("ProbabilisticMF on an item-sharded model")

    def _pmf_training_csr(self):
        """training triplets of ``to_coo`` -> device CSR (duplicates summed, zero values dropped: the reference's
        ``.nonzero()`` drops them from the indices only, INTEGRATION.md)."""
        idx, val, shape = self.data.to_coo(tensor_mode=False, feedback_threshold=self.feedback_threshold)
        eng = self.engine
        idx_d = eng.upload(np.ascontiguousarray(_as_index_array(idx)))
        return eng.coo_to_csr(idx_d[:, 0], idx_d[:, 1], eng.upload(_as_value_array(val)), shape, drop_zeros=True)

    def build(self, *args, **kwargs):
        self._check_device_pmf(args, kwargs)
        eng = self.engine
        t0 = time.perf_counter()
        a = self._pmf_training_csr()
        n_users, n_items = a.shape
        rank = int(self.rank)
        plan = eng.sgd_plan(a, max(1, min(int(self.sgd_strata), n_users, n_items)))
        del a
        # initial factors: the reference's calls on the host (lib/optimize.py:173-175)
        rnds = np.random if self.seed is None else np.random.RandomState(self.seed)
        p_host = rnds.normal(scale=0.1, size=(n_users, rank))
        q_host = rnds.normal(scale=0.1, size=(n_items, rank))
        ld = round_up(rank, 32)
        p = eng.zeros((n_users, ld), torch.float64)
        q = eng.zeros((n_items, ld), torch.float64)
        p[:, :rank].copy_(torch.from_numpy(p_host))
        q[:, :rank].copy_(torch.from_numpy(q_host))
        lam = 0.5 * self.sigma ** 2
        self.rmse_history = []
        self.iterations_time = []
        last_err = np.finfo("f8").max
        t1 = time.perf_counter()
        for epoch in range(self.num_epochs):
            te = time.perf_counter()
            new_err = eng.sgd_epoch(plan, p, q, rank, self.learn_rate, lam)       # synchronises
            self.iterations_time.append(time.perf_counter() - te)
            refined = abs(last_err - new_err) / last_err
            last_err = new_err
            rmse = np.sqrt(new_err / plan.nnz)
            self.rmse_history.append(rmse)
            if self.show_rmse:
                print("Epoch: {}. RMSE: {}".format(epoch, rmse))
            if refined < self.tolerance:
                break
        t2 = time.perf_counter()
        if self.training_time is not None:
            self.training_time.append(t2 - t0)
        if self.verbose:
            print("{} training time: {:.3f}s".format(self.method, t2 - t0))
        f = self.data.fields
        self.factors[f.userid] = p[:, :rank].cpu().numpy()
        self.factors[f.itemid] = q[:, :rank].cpu().numpy()
        self.last_timings = dict(prepare_s=t1 - t0, sgd_s=t2 - t1, epochs=len(self.rmse_history), sgd_strata=plan.strata)
        self._sgd_plan = plan              # kept for inspection (the permutation a build applied)

    def _user_rows_device(self, test_users):
        """fp32 copy of ``P[test_users]`` padded to 32 columns (the fused kernel's operand layout)."""
        return self.engine.upload(_padded_f32(self.factors[self.data.fields.userid][np.asarray(test_users)]))

    def get_recommendations(self):
        if self.data.warm_start:
            raise NotImplementedError                               # models.py:772-776
        if self.verify_integrity and hasattr(self, "verify_data_integrity"):
            self.verify_data_integrity()
        eng = self.engine
        f = self.data.fields
        test_data, shape, test_users = self._get_test_data()
        if self.topk > shape[1]:
            raise ValueError("topk exceeds the number of items")
        _, seen = self._test_csr_device(test_data, shape)
        e = self._user_rows_device(test_users)
        v_dev = self._device_factor(f.itemid)
        if self.score_kernel is not None:
            eng.set_score_kernel(self.score_kernel)
        ids = eng.score_topk(e, v_dev, self.factors[f.itemid].shape[1], self.topk,
                             seen=seen if self.filter_seen else None)
        return ids.cpu().numpy()

    def slice_recommendations(self, test_data, shape, start, stop, test_users=None):
        """Dense score rows ``P[test_users[start:stop]] Q^T`` for a (small) user slice (models.py:779-787).  Returns
        ``(scores float64 [m x n_items], slice_data)``; without ``test_users`` (what ``_user_scores`` passes) they are
        taken from the test data."""
        if test_users is None:
            test_users = self._get_test_data()[2]
        user, item, fdbk = (np.asarray(x) for x in test_data)
        sel = (user >= start) & (user < stop)
        sl = (user[sel] - start, item[sel], fdbk[sel])
        f = self.data.fields
        e = self._user_rows_device(np.asarray(test_users)[start:stop])
        v_dev = self._device_factor(f.itemid)
        s = self.engine.score_dense(e, v_dev, self.factors[f.itemid].shape[1])
        return s.cpu().numpy().astype(np.float64), sl


class B200ProbabilisticMF(_PMFDeviceMixin, host.RecommenderModel):
    """ProbabilisticMF (models.py:728-787) on the device, standalone.  ``optimizer = None`` stands for the reference's
    ``simple_pmf_sgd``, the only one on the device path."""

    def __init__(self, *args, **kwargs):
        self.seed = kwargs.pop("seed", None)
        super().__init__(*args, **kwargs)
        self.method = "PMF"
        self.optimizer = None
        self.learn_rate = 0.005
        self.sigma = 1
        self.num_epochs = 25
        self.rank = 10
        self.tolerance = 1e-4
        self.factors = {}
        self.rmse_history = None
        self.show_rmse = False
        self.iterations_time = None

    def build(self, *args, **kwargs):
        return _PMFDeviceMixin.build(self, *args, **kwargs)


def dropin_pmf():
    """``PolaraB200PMF``: the device path under the REAL ``polara`` ``ProbabilisticMF`` (requires the reference package
    to be importable)."""
    from polara.recommender.models import ProbabilisticMF

    class PolaraB200PMF(_PMFDeviceMixin, ProbabilisticMF):
        def build(self, *args, **kwargs):
            return _PMFDeviceMixin.build(self, *args, **kwargs)

    return PolaraB200PMF


def dropin():
    """Returns ``(B200SVDModel, B200ScaledSVD, B200CoffeeModel)`` derived from the REAL
    ``polara`` classes (requires the reference package to be importable)."""
    from polara.recommender.models import CoffeeModel, ScaledSVD, SVDModel

    class PolaraB200SVD(_SVDDeviceMixin, SVDModel):
        def build(self, operator=None, return_factors="vh"):
            return _SVDDeviceMixin.build(self, operator=operator, return_factors=return_factors)

    class PolaraB200ScaledSVD(_SVDDeviceMixin, ScaledSVD):
        def build(self, operator=None, return_factors="vh"):
            return _SVDDeviceMixin.build(self, operator=operator, return_factors=return_factors)

    class PolaraB200Coffee(_CoffeeDeviceMixin, CoffeeModel):
        def build(self):
            return _CoffeeDeviceMixin.build(self)

    return PolaraB200SVD, PolaraB200ScaledSVD, PolaraB200Coffee


def dropin_sampled():
    """``PolaraB200SampledSVD``: the device path under the reference's ``RandomSampleEvaluationSVDMixin`` (models.py:1095-
    1183) for data models built with ``RandomSampleEvaluationMixin`` (data.py:938-993) whose unseen interactions were set
    with ``set_unseen_interactions``.  Sampling on the fly (``unseen_interactions is None``: numba's per-thread Mersenne
    twister, lib/sampler.py) is not reproduced on the device and raises."""
    import pandas as pd
    from polara.recommender.models import RandomSampleEvaluationSVDMixin, SVDModel

    class PolaraB200SampledSVD(_SVDDeviceMixin, RandomSampleEvaluationSVDMixin, SVDModel):
        def build(self, operator=None, return_factors="vh"):
            return _SVDDeviceMixin.build(self, operator=operator, return_factors=return_factors)

        def get_recommendations(self):
            data = self.data
            userid, itemid = data.fields.userid, data.fields.itemid
            if self._prediction_target == itemid:
                return _SVDDeviceMixin.get_recommendations(self)
            if data.unseen_interactions is None:
                raise NotImplementedError("on-the-fly sampling of unseen items (numba RNG) is not on the device path; "
                                          "call data.set_unseen_interactions(...) first")
            holdout = data.test.holdout
            assert data.holdout_size >= 1                               # models.py:1106
            holdout_items = holdout[itemid].values.reshape(-1, data.holdout_size)
            test_users = holdout[userid].drop_duplicates().values      # preserve sorted (models.py:1123)
            unseen = np.concatenate(data.unseen_interactions.loc[test_users].values).reshape(len(test_users), data.unseen_items_num)
            return self.sampled_recommendations(holdout_items, unseen)

    return PolaraB200SampledSVD
