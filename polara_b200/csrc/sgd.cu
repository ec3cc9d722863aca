// ProbabilisticMF build: the SGD sweep of generalized_sgd_sweep (polara/lib/optimize.py:123-156, identity transform, no
// gradient adjustment) as called by mf_sgd_boilerplate / simple_pmf_sgd (optimize.py:160-250), in a stratified order.
//
// Users and items are cut into B contiguous ranges each (host side, DESIGN.md 3.6); block (b, c) holds the interactions
// of user range b and item range c in the reference's row-major order.  Sub-epoch s processes the blocks
// (b, (b + s) mod B), b = 0..B-1: they share no user and no item, so running them concurrently equals running them one
// after another, and an epoch is exactly the reference's sweep over a permutation of the interactions.
//
// pb200_sgd_plan sorts the nnz by processing key s * B + b (stable: reference order inside a block) and writes the
// permuted (user, item, value) triplets and block_ptr.  pb200_sgd_epoch runs one launch per sub-epoch; one warp walks
// one block in order.  Factors are fp64 and every update is __dmul_rn / __dadd_rn / __dsub_rn in the reference's
// operation order (no FMA contraction), so the only difference from the reference is the summation order of the
// r-term dot product.  No atomics: results are bit-identical from run to run.
#include <algorithm>

#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"

namespace {

constexpr int kWarpsPerCta = 4;

// which range each row falls in: bounds [B + 1] ascending (empty ranges allowed), out [n]
__global__ void range_of_kernel(const int64_t* __restrict__ bounds, int strata, int64_t n, int32_t* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        int lo = 0, hi = strata;                       // last b with bounds[b] <= i
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (bounds[mid] <= i) lo = mid; else hi = mid;
        }
        out[i] = lo;
    }
}

__global__ void counts_kernel(const int64_t* __restrict__ indptr, int64_t n, int32_t* __restrict__ cnt) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) cnt[i] = (int32_t)(indptr[i + 1] - indptr[i]);
}

// one warp per CSR row: processing key and row id of every nnz
__global__ void plan_keys_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices, int64_t n_rows,
                                 const int32_t* __restrict__ row_range, const int32_t* __restrict__ col_range, int strata,
                                 uint32_t* __restrict__ keys, uint32_t* __restrict__ pos, int32_t* __restrict__ row_of) {
    const int lane = threadIdx.x & 31;
    int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (; w < n_rows; w += n_warps) {
        const int b = row_range[w];
        for (int64_t e = indptr[w] + lane; e < indptr[w + 1]; e += 32) {
            int s = col_range[indices[e]] - b;
            if (s < 0) s += strata;
            keys[e] = (uint32_t)s * (uint32_t)strata + (uint32_t)b;
            pos[e] = (uint32_t)e;
            row_of[e] = (int32_t)w;
        }
    }
}

__global__ void plan_gather_kernel(const uint32_t* __restrict__ perm, const int32_t* __restrict__ row_of,
                                   const int32_t* __restrict__ indices, const float* __restrict__ values, int64_t nnz,
                                   int32_t* __restrict__ users, int32_t* __restrict__ items, float* __restrict__ vals) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < nnz; i += stride) {
        const uint32_t p = perm[i];
        users[i] = row_of[p];
        items[i] = indices[p];
        vals[i] = values[p];
    }
}

// block_ptr[k] = first sorted position whose key >= k, k = 0..B*B
__global__ void block_ptr_kernel(const uint32_t* __restrict__ keys, int64_t nnz, int64_t n_blocks, int64_t* __restrict__ ptr) {
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; k <= n_blocks; k += stride) {
        int64_t lo = 0, hi = nnz;
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if ((int64_t)keys[mid] < k) lo = mid + 1; else hi = mid;
        }
        ptr[k] = lo;
    }
}

__device__ __forceinline__ double warp_dot(double x) {
    // fixed butterfly: addition is commutative, so every lane ends with the same bits
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) x = __dadd_rn(x, __shfl_xor_sync(0xffffffffu, x, m));
    return x;
}

// One warp per block of sub-epoch s.  Lane j holds dimensions j, j + 32, ... (DPL per lane).  The user row stays in
// registers while consecutive entries share the user; the next entry's rows are loaded one step ahead (an item row equal
// to the current one is forwarded from registers instead, since its store is still in flight).  Plain loads, not the
// read-only path: rows written earlier in this kernel by the same thread must be read back.
template <int DPL>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
sgd_subepoch_kernel(int strata, int s, const int64_t* __restrict__ block_ptr, const int32_t* __restrict__ users,
                    const int32_t* __restrict__ items, const float* __restrict__ vals, const int32_t* __restrict__ row_cnt,
                    const int32_t* __restrict__ col_cnt, double* P, int64_t ldp, double* Q, int64_t ldq, int rank,
                    double eta, double lambd, double* __restrict__ partials) {
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
    if (b >= strata) return;
    const int64_t blk = (int64_t)s * strata + b;
    const int64_t begin = block_ptr[blk], end = block_ptr[blk + 1];
    double cum = 0.0;
    if (begin < end) {
        bool live[DPL];
#pragma unroll
        for (int t = 0; t < DPL; ++t) live[t] = lane + 32 * t < rank;
        double p[DPL], q[DPL], pn[DPL], qn[DPL];
        int m = users[begin], n = items[begin];
        float a = vals[begin];
#pragma unroll
        for (int t = 0; t < DPL; ++t) {
            p[t] = live[t] ? P[(int64_t)m * ldp + lane + 32 * t] : 0.0;
            q[t] = live[t] ? Q[(int64_t)n * ldq + lane + 32 * t] : 0.0;
        }
        double row_lambda = __ddiv_rn(lambd, (double)row_cnt[m]);
        int m_next = 0, n_next = 0;
        float a_next = 0.f;
        if (begin + 1 < end) { m_next = users[begin + 1]; n_next = items[begin + 1]; a_next = vals[begin + 1]; }
        for (int64_t e = begin; e < end; ++e) {
            const bool more = e + 1 < end;
            // loads for entry e + 1 (independent of this update unless the rows coincide, handled below)
            if (more) {
#pragma unroll
                for (int t = 0; t < DPL; ++t) {
                    qn[t] = (live[t] && n_next != n) ? Q[(int64_t)n_next * ldq + lane + 32 * t] : 0.0;
                    pn[t] = (live[t] && m_next != m) ? P[(int64_t)m_next * ldp + lane + 32 * t] : 0.0;
                }
            }
            const double col_lambda = __ddiv_rn(lambd, (double)col_cnt[n]);
            double part = 0.0;
#pragma unroll
            for (int t = 0; t < DPL; ++t) part = __dadd_rn(part, __dmul_rn(p[t], q[t]));
            const double err = __dsub_rn((double)a, warp_dot(part));
#pragma unroll
            for (int t = 0; t < DPL; ++t) {
                // gp = err*q - p*row_lambda ; gq = err*p - q*col_lambda ; both from the old rows
                const double gp = __dsub_rn(__dmul_rn(err, q[t]), __dmul_rn(p[t], row_lambda));
                const double gq = __dsub_rn(__dmul_rn(err, p[t]), __dmul_rn(q[t], col_lambda));
                p[t] = __dadd_rn(p[t], __dmul_rn(eta, gp));
                q[t] = __dadd_rn(q[t], __dmul_rn(eta, gq));
                if (live[t]) Q[(int64_t)n * ldq + lane + 32 * t] = q[t];
            }
            cum = __dadd_rn(cum, __dmul_rn(err, err));
            if (!more) break;
            if (m_next != m) {
#pragma unroll
                for (int t = 0; t < DPL; ++t) {
                    if (live[t]) P[(int64_t)m * ldp + lane + 32 * t] = p[t];
                    p[t] = pn[t];
                }
                row_lambda = __ddiv_rn(lambd, (double)row_cnt[m_next]);
            }
            if (n_next != n) {
#pragma unroll
                for (int t = 0; t < DPL; ++t) q[t] = qn[t];
            }
            m = m_next; n = n_next; a = a_next;
            if (e + 2 < end) { m_next = users[e + 2]; n_next = items[e + 2]; a_next = vals[e + 2]; }
        }
#pragma unroll
        for (int t = 0; t < DPL; ++t)
            if (live[t]) P[(int64_t)m * ldp + lane + 32 * t] = p[t];
    }
    if (lane == 0) partials[blk] = cum;
}

// sum of the block partials in (s, b) order: each thread adds a contiguous run in order, thread 0 adds the runs in order
__global__ void sum_partials_kernel(const double* __restrict__ partials, int64_t count, double* __restrict__ out) {
    __shared__ double run[1024];
    const int64_t per = (count + blockDim.x - 1) / blockDim.x;
    const int64_t lo = threadIdx.x * per, hi = min(count, lo + per);
    double acc = 0.0;
    for (int64_t i = lo; i < hi; ++i) acc = __dadd_rn(acc, partials[i]);
    run[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double total = 0.0;
        for (int t = 0; t < (int)blockDim.x; ++t) total = __dadd_rn(total, run[t]);
        *out = total;
    }
}

template <int DPL>
int launch_epoch(pb200_ctx* ctx, int strata, const int64_t* block_ptr, const int32_t* users, const int32_t* items,
                 const float* vals, const int32_t* row_cnt, const int32_t* col_cnt, double* P, int64_t ldp, double* Q,
                 int64_t ldq, int rank, double eta, double lambd, double* partials) {
    const unsigned grid = (unsigned)((strata + kWarpsPerCta - 1) / kWarpsPerCta);
    for (int s = 0; s < strata; ++s)
        sgd_subepoch_kernel<DPL><<<grid, kWarpsPerCta * 32, 0, ctx->stream>>>(strata, s, block_ptr, users, items, vals,
                                                                             row_cnt, col_cnt, P, ldp, Q, ldq, rank, eta,
                                                                             lambd, partials);
    PB_CUDA(ctx, cudaGetLastError());
    return PB200_OK;
}

}  // namespace

extern "C" int pb200_sgd_plan(pb200_ctx* ctx, int64_t n_rows, int64_t n_cols, int64_t nnz, const int64_t* indptr,
                              const int32_t* indices, const float* values, const int64_t* t_indptr, int strata,
                              const int64_t* row_bounds, const int64_t* col_bounds, int64_t* block_ptr,
                              int32_t* users_out, int32_t* items_out, float* vals_out, int32_t* row_cnt_out,
                              int32_t* col_cnt_out) {
    PB_ENTER(ctx);
    PB_REQUIRE(ctx, n_rows > 0 && n_cols > 0 && nnz > 0, "sgd_plan: empty matrix");
    PB_REQUIRE(ctx, nnz < (int64_t)4294967295ll, "sgd_plan: nnz must be < 2^32");
    PB_REQUIRE(ctx, n_rows < (int64_t)2147483647 && n_cols < (int64_t)2147483647, "sgd_plan: dimensions must fit int32");
    PB_REQUIRE(ctx, strata >= 1 && (int64_t)strata <= std::min<int64_t>(std::min(n_rows, n_cols), 65535),
               "sgd_plan: strata must be in [1, min(n_rows, n_cols, 65535)]");
    Scratch sc(ctx);
    const int blocks = 8 * ctx->num_sms;
    int32_t *row_range = nullptr, *col_range = nullptr, *row_of = nullptr;
    uint32_t *keys = nullptr, *keys_sorted = nullptr, *pos = nullptr, *perm = nullptr;
    PB_TRY(sc.alloc(&row_range, (size_t)n_rows));
    PB_TRY(sc.alloc(&col_range, (size_t)n_cols));
    PB_TRY(sc.alloc(&row_of, (size_t)nnz));
    PB_TRY(sc.alloc(&keys, (size_t)nnz));
    PB_TRY(sc.alloc(&keys_sorted, (size_t)nnz));
    PB_TRY(sc.alloc(&pos, (size_t)nnz));
    PB_TRY(sc.alloc(&perm, (size_t)nnz));
    range_of_kernel<<<blocks, 256, 0, ctx->stream>>>(row_bounds, strata, n_rows, row_range);
    range_of_kernel<<<blocks, 256, 0, ctx->stream>>>(col_bounds, strata, n_cols, col_range);
    counts_kernel<<<blocks, 256, 0, ctx->stream>>>(indptr, n_rows, row_cnt_out);
    counts_kernel<<<blocks, 256, 0, ctx->stream>>>(t_indptr, n_cols, col_cnt_out);
    plan_keys_kernel<<<blocks, 256, 0, ctx->stream>>>(indptr, indices, n_rows, row_range, col_range, strata, keys, pos, row_of);
    const uint64_t n_blocks = (uint64_t)strata * (uint64_t)strata;
    int bits = 1;
    while (bits < 32 && (1ull << bits) < n_blocks) ++bits;
    size_t temp_bytes = 0;
    PB_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, keys, keys_sorted, pos, perm, nnz, 0, bits, ctx->stream));
    uint8_t* temp = nullptr;
    PB_TRY(sc.alloc(&temp, temp_bytes));
    PB_CUDA(ctx, cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys, keys_sorted, pos, perm, nnz, 0, bits, ctx->stream));
    plan_gather_kernel<<<blocks, 256, 0, ctx->stream>>>(perm, row_of, indices, values, nnz, users_out, items_out, vals_out);
    block_ptr_kernel<<<(unsigned)std::min<int64_t>(ceil_div64((int64_t)n_blocks + 1, 256), blocks), 256, 0, ctx->stream>>>(
        keys_sorted, nnz, (int64_t)n_blocks, block_ptr);
    ctx->stats[0] += 8;
    PB_CUDA(ctx, cudaGetLastError());
    return PB200_OK;
}

extern "C" int pb200_sgd_epoch(pb200_ctx* ctx, int strata, const int64_t* block_ptr, const int32_t* users,
                               const int32_t* items, const float* vals, const int32_t* row_cnt, const int32_t* col_cnt,
                               double* P, int64_t ldp, double* Q, int64_t ldq, int rank, double learn_rate,
                               double lambd, double* cum_error_host) {
    PB_ENTER(ctx);
    PB_REQUIRE(ctx, strata >= 1 && strata <= 65535, "sgd_epoch: strata must be in [1, 65535]");
    PB_REQUIRE(ctx, rank >= 1 && rank <= 512, "sgd_epoch: rank must be in [1, 512]");
    PB_REQUIRE(ctx, ldp >= rank && ldq >= rank, "sgd_epoch: leading dimensions must be >= rank");
    PB_REQUIRE(ctx, cum_error_host != nullptr, "sgd_epoch: cum_error_host is required");
    Scratch sc(ctx);
    const int64_t n_blocks = (int64_t)strata * strata;
    double *partials = nullptr, *total = nullptr;
    PB_TRY(sc.alloc(&partials, (size_t)n_blocks));
    PB_TRY(sc.alloc(&total, 1));
    const int dpl = (rank + 31) / 32;
    int st;
    switch (dpl) {
#define PB_SGD_CASE(D)                                                                                                 \
    case D:                                                                                                            \
        st = launch_epoch<D>(ctx, strata, block_ptr, users, items, vals, row_cnt, col_cnt, P, ldp, Q, ldq, rank,        \
                             learn_rate, lambd, partials);                                                             \
        break;
        PB_SGD_CASE(1) PB_SGD_CASE(2) PB_SGD_CASE(3) PB_SGD_CASE(4)
        PB_SGD_CASE(5) PB_SGD_CASE(6) PB_SGD_CASE(7) PB_SGD_CASE(8)
#undef PB_SGD_CASE
    default:
        st = launch_epoch<16>(ctx, strata, block_ptr, users, items, vals, row_cnt, col_cnt, P, ldp, Q, ldq, rank,
                              learn_rate, lambd, partials);
    }
    PB_TRY(st);
    sum_partials_kernel<<<1, 1024, 0, ctx->stream>>>(partials, n_blocks, total);
    PB_CUDA(ctx, cudaGetLastError());
    PB_CUDA(ctx, cudaMemcpyAsync(cum_error_host, total, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    PB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->stats[0] += (uint64_t)strata + 1;
    return PB200_OK;
}
