// compact.cuh -- per-row staging segments -> (row, col)-sorted sparse output (CSR).
//
// Tail of the emit loops `for i, smp in enumerate(conf.samples): if nu > 0: "%d\t%d\t%d"`
// (xcltk/rdr/fc/core.py:109-124, xcltk/baf/fc/core.py:84-113): the finalize kernels write every
// row's non-zeros in column order to a staging area; here rows are put in input order.
#pragma once
#include <cstring>

#include "common.cuh"
#include "owner.hpp"

// Exclusive scan of n int32 -> int64 (n+1 outputs); one CTA, carries across chunks.
static __global__ void __launch_bounds__(1024) k_exclusive_scan(const int32_t *in, int64_t *out, int32_t n) {
    __shared__ int64_t warp_sum[32], warp_excl[32];
    __shared__ int64_t carry_s, chunk_total;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int base = 0; base < n; base += blockDim.x) {
        int i = base + threadIdx.x;
        int64_t x = (i < n) ? in[i] : 0, s = x;
        for (int d = 1; d < 32; d <<= 1) {
            int64_t y = __shfl_up_sync(0xffffffffu, s, d);
            if (lane >= d) s += y;
        }
        if (lane == 31) warp_sum[w] = s;
        __syncthreads();
        if (w == 0) {
            int64_t t = warp_sum[lane], ts = t;
            for (int d = 1; d < 32; d <<= 1) {
                int64_t y = __shfl_up_sync(0xffffffffu, ts, d);
                if (lane >= d) ts += y;
            }
            warp_excl[lane] = ts - t;
            if (lane == 31) chunk_total = ts;
        }
        __syncthreads();
        int64_t carry = carry_s;
        if (i < n) out[i] = carry + warp_excl[w] + (s - x);
        __syncthreads();
        if (threadIdx.x == 0) carry_s = carry + chunk_total;
        __syncthreads();
    }
    if (threadIdx.x == 0) out[n] = carry_s;
}

// Rows were written to a staging area in completion order (seg_base / seg_nnz per row);
// copy them to their place in row order.
static __global__ void __launch_bounds__(256) k_gather_rows(int32_t n_rows, const int64_t *seg_base,
                                                            const int32_t *seg_nnz, const int64_t *row_ptr,
                                                            const int32_t *st_col, const int32_t *st_val,
                                                            int32_t *o_col, int32_t *o_val) {
    for (int row = blockIdx.x; row < n_rows; row += gridDim.x) {
        const int n = seg_nnz[row];
        const int64_t src = seg_base[row], dst = row_ptr[row];
        for (int k = threadIdx.x; k < n; k += blockDim.x) {
            o_col[dst + k] = st_col[src + k];
            o_val[dst + k] = st_val[src + k];
        }
    }
}

// seg_nnz -> row_ptr (scan), staging -> (row, col)-sorted device CSR (gather), -> pinned host.
// One host synchronisation for nnz.  `tag` names the scratch buffers.
static int xg_staging_to_coo(xg_ctx *ctx, const char *tag, int32_t n_rows, int32_t n_cols,
                             const int64_t *seg_base, const int32_t *seg_nnz, const int32_t *st_col,
                             const int32_t *st_val, xg_coo **out, int *n_launches) {
    std::string t(tag);
    XG_GET(row_ptr, int64_t, (t + "_row_ptr").c_str(), n_rows + 2);
    k_exclusive_scan<<<1, 1024, 0, ctx->stream>>>(seg_nnz, row_ptr, n_rows);
    int64_t nnz = 0;
    XG_CUDA(cudaMemcpyAsync(&nnz, row_ptr + n_rows, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    XG_CUDA(cudaStreamSynchronize(ctx->stream));
    XG_GET(d_col, int32_t, (t + "_coo_col").c_str(), nnz + 1);
    XG_GET(d_val, int32_t, (t + "_coo_val").c_str(), nnz + 1);
    *n_launches += 1;
    if (nnz > 0) {
        k_gather_rows<<<n_rows < 148 * 32 ? n_rows : 148 * 32, 256, 0, ctx->stream>>>(
            n_rows, seg_base, seg_nnz, row_ptr, st_col, st_val, d_col, d_val);
        *n_launches += 1;
    }
    cudaEventRecord(ctx->ev[3], ctx->stream);
    XG_CUDA(cudaGetLastError());
    xg_coo_owner *o = new xg_coo_owner();
    memset(&o->m, 0, sizeof(o->m));
    void *hp[3] = {nullptr, nullptr, nullptr};
    size_t hs[3] = {(size_t)(nnz + 1) * 4, (size_t)(nnz + 1) * 4, (size_t)(n_rows + 1) * 8};
    for (int k = 0; k < 3; k++)
        if (!(hp[k] = ctx->pinned_get(hs[k]))) {
            for (int q = 0; q < k; q++) ctx->pinned_put(hp[q]);
            delete o;
            return ctx->fail(XG_E_NOMEM, "out of pinned host memory for the result");
        }
    o->bufs = {hp[0], hp[1], hp[2]};
    o->ctx = ctx;
    cudaEventRecord(ctx->ev[4], ctx->stream);
    if (nnz > 0) {
        cudaMemcpyAsync(hp[0], d_col, (size_t)nnz * 4, cudaMemcpyDeviceToHost, ctx->stream);
        cudaMemcpyAsync(hp[1], d_val, (size_t)nnz * 4, cudaMemcpyDeviceToHost, ctx->stream);
    }
    cudaMemcpyAsync(hp[2], row_ptr, (size_t)(n_rows + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream);
    cudaEventRecord(ctx->ev[5], ctx->stream);
    cudaError_t ce = cudaStreamSynchronize(ctx->stream);
    if (ce != cudaSuccess) {
        for (void *q : o->bufs) ctx->pinned_put(q);
        delete o;
        return ctx->fail(XG_E_CUDA, std::string("result D2H: ") + cudaGetErrorString(ce));
    }
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]);
    ctx->timing[4] += ms;
    o->m.nnz = nnz;
    o->m.n_rows = n_rows;
    o->m.n_cols = n_cols;
    o->m.col = (const int32_t *)hp[0];
    o->m.val = (const int32_t *)hp[1];
    o->m.row_ptr = (const int64_t *)hp[2];
    *out = &o->m;
    return XG_OK;
}

// The three matrices of the baf count at once: seg_base / seg_nnz hold 3 x n_rows rows (matrix k's rows at
// [k * n_rows, (k + 1) * n_rows), its staging area at st_col + k * st_stride).  One scan over all the rows, one
// host synchronisation for the three sizes, one gather, one round of copies: the call is short enough for
// every synchronisation to show (xg_staging_to_coo three times: 0.8 ms; this: 0.3 ms).
static __global__ void __launch_bounds__(256) k_gather_rows3(int32_t n_rows, int64_t st_stride, const int64_t *seg_base,
                                                             const int32_t *seg_nnz, const int64_t *row_ptr,
                                                             const int32_t *st_col, const int32_t *st_val,
                                                             int32_t *o_col, int32_t *o_val, int64_t *o_ptr) {
    for (int g = blockIdx.x; g < 3 * n_rows; g += gridDim.x) {
        const int wh = g / n_rows, row = g - wh * n_rows;
        const int n = seg_nnz[g];
        const int64_t src = seg_base[g] + (int64_t)wh * st_stride, dst = row_ptr[g];
        const int64_t first = row_ptr[(int64_t)wh * n_rows];
        if (threadIdx.x == 0) {
            o_ptr[(int64_t)wh * (n_rows + 1) + row] = dst - first;
            if (row == n_rows - 1) o_ptr[(int64_t)wh * (n_rows + 1) + n_rows] = dst + n - first;
        }
        for (int k = threadIdx.x; k < n; k += blockDim.x) {
            o_col[dst + k] = st_col[src + k];
            o_val[dst + k] = st_val[src + k];
        }
    }
}

static int xg_staging_to_coo3(xg_ctx *ctx, const char *tag, int32_t n_rows, int32_t n_cols, const int64_t *seg_base,
                              const int32_t *seg_nnz, const int32_t *st_col, const int32_t *st_val, int64_t st_stride,
                              xg_coo **out[3], int *n_launches) {
    std::string t(tag);
    XG_GET(row_ptr, int64_t, (t + "_row_ptr").c_str(), 3 * (size_t)n_rows + 2);
    XG_GET(o_ptr, int64_t, (t + "_o_ptr").c_str(), 3 * ((size_t)n_rows + 1) + 1);
    k_exclusive_scan<<<1, 1024, 0, ctx->stream>>>(seg_nnz, row_ptr, 3 * n_rows);
    *n_launches += 1;
    int64_t edge[4] = {0, 0, 0, 0};             // row_ptr at the three matrix boundaries and the end
    for (int k = 1; k <= 3; k++)
        XG_CUDA(cudaMemcpyAsync(&edge[k], row_ptr + (size_t)k * n_rows, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    XG_CUDA(cudaStreamSynchronize(ctx->stream));
    const int64_t total = edge[3];
    XG_GET(d_col, int32_t, (t + "_coo_col").c_str(), total + 1);
    XG_GET(d_val, int32_t, (t + "_coo_val").c_str(), total + 1);
    if (n_rows > 0) {
        k_gather_rows3<<<3 * n_rows < 148 * 32 ? 3 * n_rows : 148 * 32, 256, 0, ctx->stream>>>(
            n_rows, st_stride, seg_base, seg_nnz, row_ptr, st_col, st_val, d_col, d_val, o_ptr);
        *n_launches += 1;
    } else {
        XG_CUDA(cudaMemsetAsync(o_ptr, 0, sizeof(int64_t) * 4, ctx->stream));
    }
    cudaEventRecord(ctx->ev[3], ctx->stream);
    XG_CUDA(cudaGetLastError());
    xg_coo_owner *own[3] = {nullptr, nullptr, nullptr};
    auto drop = [&]() {
        for (int k = 0; k < 3; k++)
            if (own[k]) {
                for (void *q : own[k]->bufs) ctx->pinned_put(q);
                delete own[k];
            }
    };
    cudaEventRecord(ctx->ev[4], ctx->stream);
    for (int k = 0; k < 3; k++) {
        const int64_t nnz = edge[k + 1] - edge[k];
        xg_coo_owner *o = own[k] = new xg_coo_owner();
        memset(&o->m, 0, sizeof(o->m));
        o->ctx = ctx;
        size_t hs[3] = {(size_t)(nnz + 1) * 4, (size_t)(nnz + 1) * 4, (size_t)(n_rows + 1) * 8};
        void *hp[3];
        for (int q = 0; q < 3; q++) {
            if (!(hp[q] = ctx->pinned_get(hs[q]))) {
                drop();
                return ctx->fail(XG_E_NOMEM, "out of pinned host memory for the result");
            }
            o->bufs.push_back(hp[q]);
        }
        if (nnz > 0) {
            cudaMemcpyAsync(hp[0], d_col + edge[k], (size_t)nnz * 4, cudaMemcpyDeviceToHost, ctx->stream);
            cudaMemcpyAsync(hp[1], d_val + edge[k], (size_t)nnz * 4, cudaMemcpyDeviceToHost, ctx->stream);
        }
        cudaMemcpyAsync(hp[2], o_ptr + (size_t)k * ((size_t)n_rows + 1), (size_t)(n_rows + 1) * 8, cudaMemcpyDeviceToHost,
                        ctx->stream);
        o->m.nnz = nnz;
        o->m.n_rows = n_rows;
        o->m.n_cols = n_cols;
        o->m.col = (const int32_t *)hp[0];
        o->m.val = (const int32_t *)hp[1];
        o->m.row_ptr = (const int64_t *)hp[2];
    }
    cudaEventRecord(ctx->ev[5], ctx->stream);
    const cudaError_t ce = cudaStreamSynchronize(ctx->stream);
    if (ce != cudaSuccess) {
        drop();
        return ctx->fail(XG_E_CUDA, std::string("result D2H: ") + cudaGetErrorString(ce));
    }
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]);
    ctx->timing[4] += ms;
    for (int k = 0; k < 3; k++) *out[k] = &own[k]->m;
    return XG_OK;
}
