"""Thin typed wrapper over the C-ABI: torch tensors are only device-memory holders
(``tensor.data_ptr()``), no torch op computes anything on the hot path."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _abi


def _p(t, dtype=None):
    """device pointer of a tensor (None -> NULL); the dtype is asserted because the C-ABI
    takes raw pointers and would silently misread anything else."""
    if t is None:
        return C.c_void_p(0)
    if dtype is not None and t.dtype != dtype:
        raise TypeError("expected a %s tensor, got %s" % (dtype, t.dtype))
    if not t.is_cuda:
        raise TypeError("expected a CUDA tensor")
    if t.dim() > 1 and t.stride(-1) != 1:
        raise TypeError("innermost dimension must be contiguous")
    return C.c_void_p(t.data_ptr())


_F32, _I32, _I64, _F64 = torch.float32, torch.int32, torch.int64, torch.float64


def round_up(x, m):
    return (x + m - 1) // m * m


class DeviceCSR:
    """CSR matrix resident in HBM: indptr int64, indices int32, values float32.  ``n_panels > 1``: panel-major storage
    (``pb200_csr_block_columns``): indptr has n_panels * n_rows + 1 entries, ``panel_ptr`` is the host array of panel
    offsets."""

    __slots__ = ("indptr", "indices", "values", "shape", "n_panels", "panel_cols", "panel_ptr")

    def __init__(self, indptr, indices, values, shape, n_panels=1, panel_cols=None, panel_ptr=None):
        self.indptr, self.indices, self.values, self.shape = indptr, indices, values, tuple(int(s) for s in shape)
        self.n_panels = int(n_panels)
        self.panel_cols = int(self.shape[1] if panel_cols is None else panel_cols)
        self.panel_ptr = panel_ptr          # ctypes int64 array (host) or None

    @property
    def nnz(self):
        return int(self.indices.shape[0])

    def view(self):
        """the ``pb200_csr_view`` struct for the C-ABI (holds raw pointers: keep ``self`` alive while it is used)."""
        return _abi.CsrView(self.shape[0], self.shape[1], self.nnz, self.indptr.data_ptr(), self.indices.data_ptr(),
                            self.values.data_ptr(), self.n_panels, self.panel_cols,
                            C.cast(self.panel_ptr, C.c_void_p) if self.panel_ptr is not None else None)

    def nbytes(self):
        return self.indptr.numel() * 8 + self.indices.numel() * 4 + self.values.numel() * 4


def sgd_strata_bounds(counts, strata):
    """Cut rows (or columns) with nnz ``counts`` into ``strata`` contiguous ranges with balanced nnz: range b < B-1
    ends after the first row whose cumulative nnz reaches ceil((b+1) * nnz / B), the last range ends at the last row
    (DESIGN.md 3.6).  Ranges may be empty (one row holding more than nnz / B).  Returns the B + 1 bounds (int64)."""
    counts = np.asarray(counts, dtype=np.int64)
    total = int(counts.sum())
    if total <= 0:
        raise ValueError("sgd_strata_bounds: no interactions")
    targets = -(-np.arange(1, strata, dtype=np.int64) * total // strata)          # ceil((b+1) nnz / B), b < B-1
    ends = np.searchsorted(np.cumsum(counts), targets, side="left") + 1
    return np.concatenate(([0], ends, [len(counts)])).astype(np.int64)


class SgdPlan:
    """Device buffers of a stratified SGD schedule (pb200_sgd_plan): the training interactions permuted into processing
    order (``users`` / ``items`` int32, ``vals`` float32), ``block_ptr`` [B*B + 1] (block s*B + b of sub-epoch s),
    the row / column nnz counts, and the host-side range bounds of the cut."""

    __slots__ = ("strata", "shape", "nnz", "row_bounds", "col_bounds", "block_ptr", "users", "items", "vals",
                 "row_cnt", "col_cnt")

    def __init__(self, **kw):
        for k, v in kw.items():
            setattr(self, k, v)

    def permutation(self):
        """the processing order as (user, item, value) host arrays."""
        return self.users.cpu().numpy(), self.items.cpu().numpy(), self.vals.cpu().numpy()


class _StreamFollowingLib:
    """Every C-ABI call runs on torch's CURRENT stream of the engine's device: tensors are allocated, uploaded and waited
    for relative to that stream (``torch.cuda.current_stream``), so the library context must enqueue on the same one.  When
    the current stream changed since the last call (``with torch.cuda.stream(s):``), the context is re-pointed first."""

    def __init__(self, lib, engine):
        self._lib, self._engine = lib, engine

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        if name in ("pb200_ctx_create", "pb200_ctx_destroy", "pb200_ctx_set_stream", "pb200_last_error", "pb200_version"):
            return fn
        eng = self._engine

        def call(*args):
            cur = torch.cuda.current_stream(eng.device).cuda_stream
            if cur != eng._stream:
                self._lib.pb200_ctx_set_stream(eng.h, C.c_void_p(cur))
                eng._stream = cur
            return fn(*args)
        return call


class Engine:
    """One context = one device; work is enqueued on torch's current stream of that device (followed per call)."""

    def __init__(self, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("polara_b200 needs a CUDA device (sm_100); there is no CPU fallback")
        self.lib = _StreamFollowingLib(_abi.load(), self)
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
        self._stream = stream
        handle = C.c_void_p()
        st = self.lib.pb200_ctx_create(self.device.index, C.c_void_p(stream), C.byref(handle))
        if st != _abi.OK:
            raise RuntimeError("pb200_ctx_create failed with status %d (an sm_100 GPU is required)" % st)
        self.h = handle

    def close(self):
        if getattr(self, "h", None):
            self.lib.pb200_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---------------------------------------------------------------- helpers --
    def _check(self, st, where):
        try:
            _abi.check(self.h, st, where)
        except Exception as err:
            # a Python exception inside a reduce / bound hook cannot unwind through the C frames: it was parked and the
            # C call returned "hook failed"; surface the real cause
            cause = getattr(self, "_reduce_error", None)
            if cause is not None:
                self._reduce_error = None
                raise err from cause
            raise

    def empty(self, shape, dtype=torch.float32):
        return torch.empty(shape, dtype=dtype, device=self.device)

    def zeros(self, shape, dtype=torch.float32):
        return torch.zeros(shape, dtype=dtype, device=self.device)

    def upload(self, array, dtype=None):
        """numpy / host tensor -> device tensor (async on the context stream when pinned)."""
        if isinstance(array, torch.Tensor):
            t = array
        else:
            t = torch.from_numpy(np.ascontiguousarray(array))
        if dtype is not None and t.dtype != dtype:
            t = t.to(dtype)
        return t.to(self.device, non_blocking=True)

    def upload_csr(self, indptr, indices, values, shape):
        return DeviceCSR(self.upload(indptr, torch.int64), self.upload(indices, torch.int32),
                         self.upload(values, torch.float32), shape)

    def sync(self):
        self._check(self.lib.pb200_ctx_sync(self.h), "sync")

    def set_score_kernel(self, kind):
        kind = {"simt": 0, "tcgen05": 1}.get(kind, kind)
        self._check(self.lib.pb200_set_score_kernel(self.h, int(kind)), "set_score_kernel")

    def set_spmm_kernel(self, kind):
        kind = {"ldg": 0, "bulk": 1, "cpasync": 2, "window": 3, "window32": 4}.get(kind, kind)
        self._check(self.lib.pb200_set_spmm_kernel(self.h, int(kind)), "set_spmm_kernel")

    def set_prune(self, on):
        """norm-bound early termination of the fused scoring sweep (exact; on by default)."""
        self._check(self.lib.pb200_set_prune(self.h, int(bool(on))), "set_prune")

    def set_reduce_hook(self, reduce=None):
        """Install (or with None remove) the global-sum hook of the row-sharded build.  ``reduce(tensor)`` must sum the
        CUDA tensor in place over all ranks, ordered on the current stream (``torch.distributed.all_reduce``)."""
        if reduce is None:
            self._check(self.lib.pb200_set_reduce_hook(self.h, None, None), "set_reduce_hook")
            self._reduce_cb = None
            return
        dev = self.device
        dtypes = {0: (torch.float32, "<f4"), 1: (torch.float64, "<f8"), 2: (torch.int32, "<i4")}

        class _Span:                                   # raw device pointer -> torch tensor (zero copy)
            def __init__(self, p, count, typestr):
                self.__cuda_array_interface__ = {"shape": (int(count),), "typestr": typestr, "data": (int(p), False),
                                                 "version": 2}

        def hook(_user, p, count, dtype):
            try:
                tdtype, typestr = dtypes[int(dtype)]
                t = torch.as_tensor(_Span(p, count, typestr), device=dev)
                assert t.dtype == tdtype and t.data_ptr() == int(p)
                reduce(t)
                return 0
            except Exception as exc:                   # never unwind through the C frames
                self._reduce_error = exc
                return 1
        self._reduce_cb = _abi.REDUCE_FN(hook)         # keep the trampoline alive
        self._reduce_error = None
        self._check(self.lib.pb200_set_reduce_hook(self.h, C.cast(self._reduce_cb, C.c_void_p), None), "set_reduce_hook")

    def set_bound_hook(self, bound_max=None):
        """Install (or with None remove) the hook of item-sharded scoring (pb200_set_bound_hook): ``bound_max(tensor)`` must
        replace the float32 CUDA tensor of per-user lower bounds by its elementwise maximum over all ranks, ordered on the
        current stream (``torch.distributed.all_reduce(t, op=ReduceOp.MAX)``)."""
        if bound_max is None:
            self._check(self.lib.pb200_set_bound_hook(self.h, None, None), "set_bound_hook")
            self._bound_cb = None
            return
        dev = self.device

        class _Span:
            def __init__(self, p, count):
                self.__cuda_array_interface__ = {"shape": (int(count),), "typestr": "<f4", "data": (int(p), False), "version": 2}

        def hook(_user, p, count, dtype):
            try:
                assert int(dtype) == 0
                t = torch.as_tensor(_Span(p, count), device=dev)
                assert t.dtype == torch.float32 and t.data_ptr() == int(p)
                bound_max(t)
                return 0
            except Exception as exc:                   # never unwind through the C frames
                self._reduce_error = exc
                return 1
        self._bound_cb = _abi.REDUCE_FN(hook)          # keep the trampoline alive
        self._reduce_error = None
        self._check(self.lib.pb200_set_bound_hook(self.h, C.cast(self._bound_cb, C.c_void_p), None), "set_bound_hook")

    def stats(self):
        out = (C.c_uint64 * 8)()
        self._check(self.lib.pb200_get_stats(self.h, out), "get_stats")
        return [int(x) for x in out]

    # ------------------------------------------------------------------- ops ---
    def spmm(self, a: DeviceCSR, x, ell=None, out=None):
        """Y = A @ X ; X [n_cols x ldx] float32, uses the leading ``ell`` columns.  Y is [n_rows x round_up(ell, 32)],
        zero beyond column ``ell`` (padding columns are neither gathered nor accumulated)."""
        ell = x.shape[1] if ell is None else ell
        if out is None:
            out = self.empty((a.shape[0], round_up(ell, 32)))
        if a.n_panels > 1:
            view = a.view()
            st = self.lib.pb200_spmm_csr(self.h, C.byref(view), _p(x, _F32), x.stride(0), _p(out, _F32), out.stride(0), ell)
        else:
            st = self.lib.pb200_spmm(self.h, a.shape[0], a.shape[1], a.nnz, _p(a.indptr, _I64), _p(a.indices, _I32),
                                     _p(a.values, _F32), _p(x, _F32), x.stride(0), _p(out, _F32), out.stride(0), ell)
        self._check(st, "spmm")
        return out

    # L2 budget for the dense panel one column panel of a matrix gathers from (B200: 126 MB L2 in two halves; data
    # read from both dies may be held twice, so well under half of it is planned for)
    PANEL_BYTES = 40 << 20

    def panel_cols_for(self, n_cols, ell):
        """columns per panel so that the gathered slice of X (panel_cols rows of min(ell,128) floats) stays in L2;
        returns n_cols when the whole operand fits (no blocking needed)."""
        row_bytes = 4 * min(round_up(max(int(ell), 1), 32), 128)
        if n_cols * row_bytes <= self.PANEL_BYTES * 5 // 4:
            return int(n_cols)
        cols = max(1024, self.PANEL_BYTES // row_bytes)
        n_panels = -(-n_cols // cols)
        return int(-(-n_cols // n_panels))           # equal panels

    def block_columns(self, a: DeviceCSR, panel_cols):
        """panel-major copy of ``a`` (pb200_csr_block_columns); returns ``a`` itself when one panel suffices."""
        panel_cols = int(panel_cols)
        n_panels = max(1, -(-a.shape[1] // panel_cols))
        if n_panels == 1 or a.n_panels > 1:
            return a
        b_indptr = self.empty((n_panels * a.shape[0] + 1,), torch.int64)
        b_indices = self.empty((a.nnz,), torch.int32)
        b_values = self.empty((a.nnz,), torch.float32)
        panel_ptr = (C.c_int64 * (n_panels + 1))()
        st = self.lib.pb200_csr_block_columns(self.h, a.shape[0], a.shape[1], a.nnz, _p(a.indptr, _I64), _p(a.indices, _I32),
                                              _p(a.values, _F32), panel_cols, n_panels, _p(b_indptr), _p(b_indices),
                                              _p(b_values), C.cast(panel_ptr, C.c_void_p))
        self._check(st, "csr_block_columns")
        return DeviceCSR(b_indptr, b_indices, b_values, a.shape, n_panels, panel_cols, panel_ptr)

    def coo_to_csr(self, rows, cols, vals, shape, drop_zeros=False, require_sorted_rows=False):
        """device ingest (pb200_coo_to_csr): ``rows`` / ``cols`` int64 CUDA tensors (1-d, any element stride -- e.g. the
        two columns of the [nnz x 2] index array of ``to_coo``), ``vals`` float32/float64 CUDA tensor or None (= ones).
        Returns a DeviceCSR with duplicates summed and sorted columns."""
        nnz = int(rows.shape[0])
        n_rows, n_cols = int(shape[0]), int(shape[1])
        if rows.dtype != _I64 or cols.dtype != _I64 or not rows.is_cuda or not cols.is_cuda:
            raise TypeError("coo_to_csr: rows / cols must be int64 CUDA tensors")
        if vals is not None and vals.dtype not in (_F32, _F64):
            raise TypeError("coo_to_csr: values must be float32 or float64")
        if vals is not None and vals.stride(0) != 1:
            vals = vals.contiguous()
        indptr = self.empty((n_rows + 1,), torch.int64)
        indices = self.empty((max(nnz, 1),), torch.int32)
        values = self.empty((max(nnz, 1),), torch.float32)
        out_nnz = C.c_int64(0)
        st = self.lib.pb200_coo_to_csr(self.h, n_rows, n_cols, nnz, C.c_void_p(rows.data_ptr()), rows.stride(0) if nnz else 1,
                                       C.c_void_p(cols.data_ptr()), cols.stride(0) if nnz else 1,
                                       C.c_void_p(vals.data_ptr()) if vals is not None else None,
                                       1 if (vals is not None and vals.dtype == _F64) else 0, int(bool(drop_zeros)),
                                       int(bool(require_sorted_rows)), _p(indptr), _p(indices), _p(values), C.byref(out_nnz))
        self._check(st, "coo_to_csr")
        n = int(out_nnz.value)
        return DeviceCSR(indptr, indices[:n], values[:n], (n_rows, n_cols))

    def shift_i64(self, t, delta):
        """t += delta in place (int64 CUDA tensor): re-basing row pointers / user ids of a chunk."""
        st = self.lib.pb200_shift_i64(self.h, _p(t, _I64), t.numel(), int(delta))
        self._check(st, "shift_i64")
        return t

    def transpose(self, a: DeviceCSR):
        t = DeviceCSR(self.empty((a.shape[1] + 1,), torch.int64), self.empty((a.nnz,), torch.int32),
                      self.empty((a.nnz,), torch.float32), (a.shape[1], a.shape[0]))
        st = self.lib.pb200_csr_transpose(self.h, a.shape[0], a.shape[1], a.nnz, _p(a.indptr), _p(a.indices),
                                          _p(a.values), _p(t.indptr), _p(t.indices), _p(t.values))
        self._check(st, "csr_transpose")
        return t

    def rescale(self, a: DeviceCSR, row_scaling, col_scaling):
        st = self.lib.pb200_rescale(self.h, a.shape[0], a.shape[1], a.nnz, _p(a.indptr), _p(a.indices),
                                    _p(a.values), float(row_scaling), float(col_scaling))
        self._check(st, "rescale")

    def rsvd(self, a: DeviceCSR, at: DeviceCSR, rank, ell, max_iters=8, tol=1e-6, seed=1, want_u=False, vec_tol=0.0):
        """returns (V, sigma, U | None, iters); convergence details of the call are left in ``self.last_rsvd_info``:
        ``dict(iters, value_change, angle_bound, converged)`` (see pb200_rsvd_csr)."""
        ldv = round_up(rank, 32)
        v = self.zeros((a.shape[1], ldv))
        sigma = self.empty((rank,), torch.float64)
        u = self.zeros((a.shape[0], ldv)) if want_u else None
        info = (C.c_double * 8)()
        va, vt = a.view(), at.view()
        st = self.lib.pb200_rsvd_csr(self.h, C.byref(va), C.byref(vt), rank, ell, max_iters, float(tol), float(vec_tol),
                                     int(seed), _p(v), ldv, _p(sigma), _p(u), ldv, info)
        self._check(st, "rsvd")
        self.last_rsvd_info = dict(iters=int(info[0]), value_change=float(info[1]), angle_bound=float(info[2]),
                                   converged=bool(info[3]))
        return v, sigma, u, int(info[0])

    def tall_svd(self, m, rank, want_vt=False):
        n, c = m.shape
        ldu = round_up(rank, 32)
        u = self.zeros((n, ldu))
        sigma = self.empty((rank,), torch.float64)
        vt = self.empty((rank, c)) if want_vt else None
        st = self.lib.pb200_tall_svd(self.h, _p(m, _F32), n, c, m.stride(0), rank, _p(sigma), _p(u), ldu, _p(vt))
        self._check(st, "tall_svd")
        return u, sigma, vt

    def score_topk(self, e, v, r, k, seen=None, item_offset=0, want_scores=False, m=None):
        m = e.shape[0] if m is None else m
        ids = self.empty((m, k), torch.int64)
        scores = self.empty((m, k), torch.float32) if want_scores else None
        sp, si = (seen if seen is not None else (None, None))
        st = self.lib.pb200_score_topk(self.h, _p(e, _F32), e.stride(0), _p(v, _F32), v.stride(0), m, v.shape[0], r,
                                       _p(sp, _I64), _p(si, _I32), k, item_offset, _p(ids), _p(scores))
        self._check(st, "score_topk")
        return (ids, scores) if want_scores else ids

    def last_score_kernel_ms(self):
        """duration of the last fused scoring kernel (CUDA events inside the library)."""
        return self.stats()[4] / 1000.0

    def score_topk_cands(self, e, v, r, k, seen=None, item_offset=0, m=None, m_alloc=None, bound_max=None):
        """candidate lists of ALL users against one item shard.  ``bound_max`` (see ``set_bound_hook``) shares the seed bounds
        between the shards for the duration of this call."""
        m = e.shape[0] if m is None else m
        m_alloc = m if m_alloc is None else m_alloc
        # {f32 score, i32 id} pairs; rows >= m (padding for the exchange) are empty lists
        cands = torch.empty((m_alloc, k, 2), dtype=torch.int32, device=self.device)
        if m_alloc > m:
            self._check(self.lib.pb200_fill_empty_cands(self.h, C.c_void_p(cands[m:].data_ptr()), (m_alloc - m) * k),
                        "fill_empty_cands")
        sp, si = (seen if seen is not None else (None, None))
        if bound_max is not None:
            self.set_bound_hook(bound_max)
        try:
            st = self.lib.pb200_score_topk_cands(self.h, _p(e, _F32), e.stride(0), _p(v, _F32), v.stride(0), m, v.shape[0], r,
                                                 _p(sp, _I64), _p(si, _I32), k, item_offset, _p(cands))
        finally:
            if bound_max is not None:
                self.set_bound_hook(None)
        self._check(st, "score_topk_cands")
        return cands

    def merge_cands(self, cands, parts, m, k, want_scores=False):
        ids = self.empty((m, k), torch.int64)
        scores = self.empty((m, k), torch.float32) if want_scores else None
        st = self.lib.pb200_merge_cands(self.h, _p(cands), parts, m, k, _p(ids), _p(scores))
        self._check(st, "merge_cands")
        return (ids, scores) if want_scores else ids

    def merge_cands_fill(self, cands, parts, part_rows, m, k, e, v, r, seen):
        """merge + seen-item fill-up for the rows this rank owns (pb200_merge_cands_fill).  ``cands`` [parts, part_rows, k, 2];
        ``e`` [>= m rows] embeddings of those rows, ``v`` the whole item factor matrix, ``seen`` = (indptr view starting at
        the first owned row, global indices)."""
        ids = self.empty((part_rows, k), torch.int64)
        st = self.lib.pb200_merge_cands_fill(self.h, _p(cands), parts, part_rows * k, m, k, _p(e, _F32), e.stride(0),
                                             _p(v, _F32), v.stride(0), r, v.shape[0], _p(seen[0], _I64), _p(seen[1], _I32),
                                             _p(ids), None)
        self._check(st, "merge_cands_fill")
        return ids

    def gather_dot(self, e, v, r, user_idx, item_idx):
        """scores of explicit (user, item) pairs: ``user_idx`` / ``item_idx`` int64 CUDA tensors of one shape; returns
        float32 scores of that shape (pb200_gather_dot)."""
        out = self.empty(tuple(user_idx.shape), torch.float32)
        st = self.lib.pb200_gather_dot(self.h, _p(e, _F32), e.stride(0), e.shape[0], _p(v, _F32), v.stride(0), v.shape[0], r,
                                       _p(user_idx.contiguous(), _I64), _p(item_idx.contiguous(), _I64), user_idx.numel(), _p(out))
        self._check(st, "gather_dot")
        return out

    def score_dense(self, e, v, r):
        m, n = e.shape[0], v.shape[0]
        s = self.empty((m, n))
        st = self.lib.pb200_score_dense(self.h, _p(e, _F32), e.stride(0), _p(v, _F32), v.stride(0), m, n, r, _p(s), n)
        self._check(st, "score_dense")
        return s

    def topk_dense(self, scores, k, seen=None, want_scores=False):
        """top-k of a dense CUDA score block [m x n] (float32 / float64), optional fused seen handling (pb200_topk_dense)."""
        if scores.dtype not in (_F32, _F64):
            raise TypeError("topk_dense: scores must be float32 or float64")
        m, n = scores.shape
        ids = self.empty((m, k), torch.int64)
        out = self.empty((m, k), scores.dtype) if want_scores else None
        sp, si = (seen if seen is not None else (None, None))
        st = self.lib.pb200_topk_dense(self.h, _p(scores), 1 if scores.dtype == _F64 else 0, scores.stride(0), m, n,
                                       _p(sp, _I64), _p(si, _I32), int(k), _p(ids), _p(out))
        self._check(st, "topk_dense")
        return (ids, out) if want_scores else ids

    def downvote_dense(self, scores, rows, cols):
        """in place: push the scores at (rows, cols) below the block minimum, order preserved (pb200_downvote_dense)."""
        m, n = scores.shape
        st = self.lib.pb200_downvote_dense(self.h, _p(scores), 1 if scores.dtype == _F64 else 0, scores.stride(0), m, n,
                                           _p(rows, _I64), _p(cols, _I64), int(rows.shape[0]))
        self._check(st, "downvote_dense")
        return scores

    def coo_group(self, key, n_keys, a, b, val):
        nnz = key.shape[0]
        seg = self.empty((n_keys + 1,), torch.int64)
        ao, bo = self.empty((nnz,), torch.int32), self.empty((nnz,), torch.int32)
        vo = self.empty((nnz,), torch.float32)
        st = self.lib.pb200_coo_group(self.h, nnz, n_keys, _p(key, _I32), _p(a, _I32), _p(b, _I32), _p(val, _F32), _p(seg), _p(ao), _p(bo), _p(vo))
        self._check(st, "coo_group")
        return seg, ao, bo, vo

    def ttm(self, n0, seg, i1, i2, val, u, ru, w, rw):
        """out[i0, x*rw + y] = sum_{nnz in row i0} val * u[i1, x] * w[i2, y]."""
        ldo = round_up(ru * rw, 4)
        out = self.empty((n0, ldo))
        st = self.lib.pb200_ttm(self.h, n0, i1.shape[0], _p(seg, _I64), _p(i1, _I32), _p(i2, _I32), _p(val, _F32), _p(u, _F32), ru, u.stride(0),
                                _p(w, _F32), rw, w.stride(0), _p(out), ldo)
        self._check(st, "ttm")
        return out

    def ttm_reduce(self, n_seg, seg, ia, ib, val, a, ra, b, rb):
        out = self.empty((n_seg, ra * rb))
        st = self.lib.pb200_ttm_reduce(self.h, n_seg, ia.shape[0], _p(seg, _I64), _p(ia, _I32), _p(ib, _I32), _p(val, _F32), _p(a, _F32), ra,
                                       a.stride(0), _p(b, _F32), rb, b.stride(0), _p(out), ra * rb)
        self._check(st, "ttm_reduce")
        return out

    def sgd_plan(self, a: DeviceCSR, strata):
        """stratified schedule of the training CSR ``a`` (sorted, duplicates summed, no zero values) with ``strata``
        user and item ranges (pb200_sgd_plan); the cut is made on the host from the row / column counts."""
        if a.n_panels != 1:
            raise ValueError("sgd_plan: needs a plain CSR")
        n_rows, n_cols = a.shape
        strata = int(strata)
        at = self.transpose(a)
        row_bounds = sgd_strata_bounds(np.diff(a.indptr.cpu().numpy()), strata)
        col_bounds = sgd_strata_bounds(np.diff(at.indptr.cpu().numpy()), strata)
        plan = SgdPlan(strata=strata, shape=(n_rows, n_cols), nnz=a.nnz, row_bounds=row_bounds, col_bounds=col_bounds,
                       block_ptr=self.empty((strata * strata + 1,), _I64), users=self.empty((a.nnz,), _I32),
                       items=self.empty((a.nnz,), _I32), vals=self.empty((a.nnz,), _F32),
                       row_cnt=self.empty((n_rows,), _I32), col_cnt=self.empty((n_cols,), _I32))
        rb, cb = self.upload(row_bounds), self.upload(col_bounds)
        st = self.lib.pb200_sgd_plan(self.h, n_rows, n_cols, a.nnz, _p(a.indptr, _I64), _p(a.indices, _I32),
                                     _p(a.values, _F32), _p(at.indptr, _I64), strata, _p(rb, _I64), _p(cb, _I64),
                                     _p(plan.block_ptr), _p(plan.users), _p(plan.items), _p(plan.vals), _p(plan.row_cnt),
                                     _p(plan.col_cnt))
        self._check(st, "sgd_plan")
        self.sync()                               # the bound arrays and the transpose are released on return
        return plan

    def sgd_epoch(self, plan: SgdPlan, p, q, rank, learn_rate, lam):
        """one stratified SGD epoch in place on the float64 factors ``p`` [n_users x ld] / ``q`` [n_items x ld];
        returns the epoch's sum of squared errors (pb200_sgd_epoch)."""
        if p.shape[0] != plan.shape[0] or q.shape[0] != plan.shape[1]:
            raise ValueError("sgd_epoch: factor shapes do not match the plan")
        cum = C.c_double(0.0)
        st = self.lib.pb200_sgd_epoch(self.h, plan.strata, _p(plan.block_ptr, _I64), _p(plan.users, _I32),
                                      _p(plan.items, _I32), _p(plan.vals, _F32), _p(plan.row_cnt, _I32),
                                      _p(plan.col_cnt, _I32), _p(p, _F64), p.stride(0), _p(q, _F64), q.stride(0),
                                      int(rank), float(learn_rate), float(lam), C.byref(cum))
        self._check(st, "sgd_epoch")
        return float(cum.value)


_ENGINES = {}


def get_engine(device=None):
    """Process-wide engine per device (created on first use)."""
    if not torch.cuda.is_available():
        raise RuntimeError("polara_b200 needs a CUDA device (sm_100); there is no CPU fallback")
    idx = torch.cuda.current_device() if device is None else int(device)
    eng = _ENGINES.get(idx)
    if eng is None:
        eng = _ENGINES[idx] = Engine(idx)
    return eng
