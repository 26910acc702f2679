// phase.cu -- local phasing of long regions (the pre-step of `xcltk baf`), the EM of every region on the device.
//
// What xcltk_b200/baf/fc/phasing.py:reg_local_phasing and baf/localphase.py:snp_local_phasing / phasing_em compute
// for one region (xcltk/baf/fc/phasing.py:13-78, xcltk/baf/localphase.py:14-243), sparse over the region's DP
// support.  One CTA runs one region to the end: the outer rounds (BAF cell filter, EM, flips, re-orientation) and
// the inner EM iterations, with no host round trip.  Regions that share a SNP are ordered by waves (one launch per
// wave, in order on one stream): a region reads the orientation (ref_idx) the earlier waves left and writes its own
// flips before the next wave starts.
//
// Per region the host hands over its entries (cell with DP > 0 at a SNP of the region) twice: SNP-major (per slot,
// by cell) and cell-major (per local cell, by SNP).  Per-cell sums (theta) walk the cell-major list, per-SNP sums
// (log-likelihood, the starting Z) the SNP-major one, each in a fixed order: no floating-point atomics, the results
// are the same from run to run.
//
// NaN rule: once the BAF filter has removed every cell that expresses a SNP, that SNP's starting Z is 0/0, and the
// reference's dense products spread the NaN to every theta, Z and log-likelihood; its flips are then all False.
// Here such a round is detected from the integer depth sums and given no flips, without running the EM.
//
// Ties: a flip whose Z1 - Z0, or a convergence test whose ll_new - ll_old - 1e-3, is that close to 0 goes the
// way the reference's rounding sends it, which another FP64 order cannot reproduce.  Such a region is reported
// with status 2 (its flips are still applied here); the caller decides it with the reference and runs the later
// waves again.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>
#include <vector>

#include "common.cuh"

#define LP_THREADS 256
#define LP_WARPS (LP_THREADS / 32)
#define LP_MIN_ROUNDS 5           // snp_local_phasing: min_iter
#define LP_MAX_ROUNDS 50          // snp_local_phasing: max_iter
#define LP_MIN_ITER 10            // phasing_em: min_iter
#define LP_MAX_ITER 1000          // phasing_em: max_iter
#define LP_EPS_CONV 1e-3          // phasing_em: epsilon_conv
#define LP_CLIP 1e-6              // _loglik: eps
#define LP_LOW_BAF 0.45
#define LP_UP_BAF 0.55
#define LP_B2 (20000.0 * 20000.0) // smoothing_kernel: b ** 2
#define LP_CUT 746.0              // exp(-q) is exactly 0 in double for q >= 746: |dx| <= b * sqrt(746) only
// A decision this close to its threshold is decided by the last bits of the reference's own arithmetic (BLAS
// summation order, libm): |Z1 - Z0| of a flip (near a symmetric point the EM can grow a last-bit difference by orders
// of magnitude before the end), or |dll - 1e-3| of the convergence test, relative to |ll|.
#define LP_TIE 1e-6
#define LP_TIE_LL 1e-9

namespace {

struct LpDev {
    const int32_t *snp_pos;
    uint8_t *ref_idx;
    const int64_t *reg_snp_ptr, *reg_cell_ptr, *slot_ent_ptr, *cell_ent_ptr;
    const int32_t *reg_snp;
    const int32_t *sm_cell, *sm_ad, *sm_dp;     // SNP-major entries
    const int32_t *cm_snp, *cm_ad, *cm_dp;      // cell-major entries
    uint8_t *keep_out, *flip_out;
    int8_t *status_out;
    int32_t *iters_out;
    unsigned long long *ns_out;
    // scratch, per slot
    int32_t *kidx, *wlo, *whi;
    uint8_t *ori, *ffin, *fround;
    double *z0, *zr, *ll0, *ll1, *lse, *wsum;
    // scratch, per local cell
    uint8_t *alive;
    int64_t *dpc;
    double *lt0, *lt1, *lm0, *lm1;
};

__device__ __forceinline__ unsigned long long lp_now() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// smoothing_kernel's weight, the host's expression: exp(0.0 - (x_j - x_i)**2 / b**2) with integer positions
__device__ __forceinline__ double lp_q(int32_t xi, int32_t xj) {
    const long long d = (long long)xj - (long long)xi;
    return (double)(d * d) / LP_B2;
}

__device__ __forceinline__ double lp_clip(double t) {
    if (t <= 0.0) t = LP_CLIP;
    if (t >= 1.0) t = 1.0 - LP_CLIP;
    return t;
}

// scipy.special.logsumexp of two finite values: log1p(sum of the others' exp(a - max)) + log(#max) + max
__device__ __forceinline__ double lp_lse2(double a, double b) {
    const double mx = fmax(a, b), mn = fmin(a, b);
    if (mx == mn) return (log1p(0.0) + log(2.0)) + mx;
    return (log1p(exp(mn - mx)) + 0.0) + mx;
}

__device__ __forceinline__ double lp_warp_sum(double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block sum of one value per thread in a fixed tree (deterministic).
__device__ double lp_block_sum(double v, double *red) {
    v = lp_warp_sum(v);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) red[w] = v;
    __syncthreads();
    double s = 0.0;
    for (int k = 0; k < LP_WARPS; k++) s += red[k];
    return s;
}

// M step (thetas over the live cells, cell-major) then the log-likelihood matrix (per kept SNP, SNP-major) and
// ll = sum_j logsumexp(ll_mat[j, :]).  z0 holds Z[:, 0]; Z[:, 1] = 1 - Z[:, 0].
__device__ double lp_mstep_ll(const LpDev &P, int64_t s0, int64_t c0, int nk, int nc, double *red) {
    for (int c = threadIdx.x; c < nc; c += LP_THREADS) {
        if (!P.alive[c0 + c]) continue;
        double a0 = 0.0, b0 = 0.0, a1 = 0.0, b1 = 0.0;
        for (int64_t e = P.cell_ent_ptr[c0 + c]; e < P.cell_ent_ptr[c0 + c + 1]; e++) {
            const int j = P.cm_snp[e];
            const int32_t dp = P.cm_dp[e], ad0 = P.cm_ad[e];
            const int32_t ad = P.ori[s0 + j] ? dp - ad0 : ad0, bd = dp - ad;
            const double z = P.z0[s0 + j], z1 = 1.0 - z;
            a0 += (double)ad * z;
            b0 += (double)bd * (1.0 - z);
            a1 += (double)ad * z1;
            b1 += (double)bd * (1.0 - z1);
        }
        const double den = (double)P.dpc[c0 + c];
        const double t0 = lp_clip((a0 + b0) / den), t1 = lp_clip((a1 + b1) / den);
        P.lt0[c0 + c] = log(t0);
        P.lt1[c0 + c] = log(t1);
        P.lm0[c0 + c] = log(1.0 - t0);
        P.lm1[c0 + c] = log(1.0 - t1);
    }
    __syncthreads();
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    const int64_t sc = c0;                    // the entries' local cell ids count from the region's first cell
    for (int k = w; k < nk; k += LP_WARPS) {
        const int j = P.kidx[s0 + k];
        const bool o = P.ori[s0 + j];
        double a0 = 0.0, b0 = 0.0, a1 = 0.0, b1 = 0.0;
        for (int64_t e = P.slot_ent_ptr[s0 + j] + l; e < P.slot_ent_ptr[s0 + j + 1]; e += 32) {
            const int c = P.sm_cell[e];
            if (!P.alive[sc + c]) continue;
            const int32_t dp = P.sm_dp[e], ad = o ? dp - P.sm_ad[e] : P.sm_ad[e], bd = dp - ad;
            a0 += (double)ad * P.lt0[sc + c];
            b0 += (double)bd * P.lm0[sc + c];
            a1 += (double)ad * P.lt1[sc + c];
            b1 += (double)bd * P.lm1[sc + c];
        }
        a0 = lp_warp_sum(a0);
        b0 = lp_warp_sum(b0);
        a1 = lp_warp_sum(a1);
        b1 = lp_warp_sum(b1);
        if (l == 0) {
            const double l0 = a0 + b0, l1 = a1 + b1;
            P.ll0[s0 + k] = l0;
            P.ll1[s0 + k] = l1;
            P.lse[s0 + k] = lp_lse2(l0, l1);
        }
    }
    __syncthreads();
    double part = 0.0;
    for (int k = threadIdx.x; k < nk; k += LP_THREADS) part += P.lse[s0 + k];
    return lp_block_sum(part, red);
}

// One region per CTA: regions [r_beg, r_beg + gridDim.x) of the wave.
__global__ void __launch_bounds__(LP_THREADS) k_local_phase(LpDev P, int32_t r_beg) {
    const int r = r_beg + blockIdx.x;
    const int64_t s0 = P.reg_snp_ptr[r], c0 = P.reg_cell_ptr[r];
    const int m = (int)(P.reg_snp_ptr[r + 1] - s0), nc = (int)(P.reg_cell_ptr[r + 1] - c0);
    __shared__ int sh_nk, sh_cnt, sh_flag, sh_tie;
    __shared__ double red[LP_WARPS];
    const unsigned long long t_beg = lp_now();

    for (int j = threadIdx.x; j < m; j += LP_THREADS) {
        P.keep_out[s0 + j] = P.slot_ent_ptr[s0 + j + 1] > P.slot_ent_ptr[s0 + j];
        P.flip_out[s0 + j] = 0;
        P.ori[s0 + j] = P.ref_idx[P.reg_snp[s0 + j]] == 1;
        P.ffin[s0 + j] = 0;
    }
    for (int c = threadIdx.x; c < nc; c += LP_THREADS) {
        int64_t d = 0;
        for (int64_t e = P.cell_ent_ptr[c0 + c]; e < P.cell_ent_ptr[c0 + c + 1]; e++) d += P.cm_dp[e];
        P.dpc[c0 + c] = d;
        P.alive[c0 + c] = 1;
    }
    __syncthreads();
    if (threadIdx.x == 0) {                 // pruned list: the SNPs with depth, in the region's order
        sh_tie = 0;
        int nk = 0;
        for (int j = 0; j < m; j++)
            if (P.keep_out[s0 + j]) P.kidx[s0 + nk++] = j;
        sh_nk = nk;
    }
    __syncthreads();
    const int nk = sh_nk;
    int8_t status = 0;
    int32_t iters = 0;
    if (nk > 0 && nc > 0) {
        // smoothing windows over the pruned list (positions sorted) and the row sums of the kernel
        for (int k = threadIdx.x; k < nk; k += LP_THREADS) {
            const int32_t x = P.snp_pos[P.reg_snp[s0 + P.kidx[s0 + k]]];
            int lo = k, hi = k;
            while (lo > 0 && lp_q(x, P.snp_pos[P.reg_snp[s0 + P.kidx[s0 + lo - 1]]]) < LP_CUT) lo--;
            while (hi + 1 < nk && lp_q(x, P.snp_pos[P.reg_snp[s0 + P.kidx[s0 + hi + 1]]]) < LP_CUT) hi++;
            double s = 0.0;
            for (int q = lo; q <= hi; q++) s += exp(0.0 - lp_q(x, P.snp_pos[P.reg_snp[s0 + P.kidx[s0 + q]]]));
            P.wlo[s0 + k] = lo;
            P.whi[s0 + k] = hi;
            P.wsum[s0 + k] = s;
        }
        status = 1;
        for (int round = 0; round < LP_MAX_ROUNDS; round++) {
            // cells whose aggregated BAF lies in [0.45, 0.55] leave for good
            if (threadIdx.x == 0) sh_cnt = 0;
            __syncthreads();
            int live = 0;
            for (int c = threadIdx.x; c < nc; c += LP_THREADS) {
                if (!P.alive[c0 + c]) continue;
                int64_t a = 0;
                for (int64_t e = P.cell_ent_ptr[c0 + c]; e < P.cell_ent_ptr[c0 + c + 1]; e++) {
                    const int32_t dp = P.cm_dp[e], ad = P.cm_ad[e];
                    a += P.ori[s0 + P.cm_snp[e]] ? dp - ad : ad;
                }
                const double baf = (double)a / (double)P.dpc[c0 + c];
                const bool keep = baf < LP_LOW_BAF || baf > LP_UP_BAF;
                P.alive[c0 + c] = keep;
                live += keep;
            }
            atomicAdd(&sh_cnt, live);
            if (threadIdx.x == 0) sh_flag = 0;
            __syncthreads();
            if (sh_cnt == 0) {
                status = 0;
                break;
            }
            // starting Z[:, 0] = AD.sum(1) / DP.sum(1) over the live cells; a SNP without depth poisons the round
            const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
            for (int k = w; k < nk; k += LP_WARPS) {
                const int j = P.kidx[s0 + k];
                const bool o = P.ori[s0 + j];
                long long a = 0, d = 0;
                for (int64_t e = P.slot_ent_ptr[s0 + j] + l; e < P.slot_ent_ptr[s0 + j + 1]; e += 32) {
                    if (!P.alive[c0 + P.sm_cell[e]]) continue;
                    const int32_t dp = P.sm_dp[e];
                    a += o ? dp - P.sm_ad[e] : P.sm_ad[e];
                    d += dp;
                }
                for (int s = 16; s > 0; s >>= 1) {
                    a += __shfl_xor_sync(0xffffffffu, a, s);
                    d += __shfl_xor_sync(0xffffffffu, d, s);
                }
                if (l == 0) {
                    if (d == 0) atomicOr(&sh_flag, 1);
                    P.z0[s0 + j] = (double)a / (double)d;
                }
            }
            __syncthreads();
            const bool poisoned = sh_flag != 0;
            if (!poisoned) {
                double ll = lp_mstep_ll(P, s0, c0, nk, nc, red);
                for (int it = 0; it < LP_MAX_ITER; it++) {
                    const double ll_old = ll;
                    for (int k = threadIdx.x; k < nk; k += LP_THREADS) {       // E step
                        const double a = P.ll0[s0 + k], b = P.ll1[s0 + k], mx = fmax(a, b);
                        const double e0 = exp(a - mx), e1 = exp(b - mx);
                        P.zr[s0 + k] = e0 / (e0 + e1);
                    }
                    __syncthreads();
                    for (int k = threadIdx.x; k < nk; k += LP_THREADS) {       // Z[:, 0] smoothed along the genome
                        const int32_t x = P.snp_pos[P.reg_snp[s0 + P.kidx[s0 + k]]];
                        const double rs = P.wsum[s0 + k];
                        double u = 0.0;
                        for (int q = P.wlo[s0 + k]; q <= P.whi[s0 + k]; q++) {
                            const double wq = exp(0.0 - lp_q(x, P.snp_pos[P.reg_snp[s0 + P.kidx[s0 + q]]])) / rs;
                            u += P.zr[s0 + q] * wq;
                        }
                        P.z0[s0 + P.kidx[s0 + k]] = u;
                    }
                    __syncthreads();
                    ll = lp_mstep_ll(P, s0, c0, nk, nc, red);
                    iters++;
                    if (it >= LP_MIN_ITER && threadIdx.x == 0 &&
                        fabs((ll - ll_old) - LP_EPS_CONV) < LP_TIE_LL * fmax(1.0, fabs(ll)))
                        sh_tie = 1;
                    if (it >= LP_MIN_ITER && ll - ll_old < LP_EPS_CONV) break;
                }
            }
            // flip = Z[:, 1] >= Z[:, 0]; flip_final ^= flip; stop when a later round flips all or none
            if (threadIdx.x == 0) sh_cnt = 0;
            __syncthreads();
            int nf = 0;
            for (int k = threadIdx.x; k < nk; k += LP_THREADS) {
                const int j = P.kidx[s0 + k];
                const double z = P.z0[s0 + j];
                const uint8_t f = poisoned ? 0 : (1.0 - z) >= z;
                if (!poisoned && fabs((1.0 - z) - z) < LP_TIE) sh_tie = 1;
                P.fround[s0 + j] = f;
                P.ffin[s0 + j] ^= f;
                nf += f;
            }
            atomicAdd(&sh_cnt, nf);
            __syncthreads();
            if (round >= LP_MIN_ROUNDS && (sh_cnt == 0 || sh_cnt == nk)) break;
            for (int k = threadIdx.x; k < nk; k += LP_THREADS) {
                const int j = P.kidx[s0 + k];
                P.ori[s0 + j] ^= P.fround[s0 + j];
            }
            __syncthreads();
        }
    }
    if (status) {
        // as few changes as possible: the flips are inverted when more than half of the SNPs flip
        if (threadIdx.x == 0) sh_cnt = 0;
        __syncthreads();
        int nf = 0;
        for (int k = threadIdx.x; k < nk; k += LP_THREADS) nf += P.ffin[s0 + P.kidx[s0 + k]];
        atomicAdd(&sh_cnt, nf);
        __syncthreads();
        const uint8_t inv = 2 * (int64_t)sh_cnt > nk;
        for (int k = threadIdx.x; k < nk; k += LP_THREADS) {
            const int j = P.kidx[s0 + k];
            const uint8_t f = P.ffin[s0 + j] ^ inv;
            P.flip_out[s0 + j] = f;
            if (f) P.ref_idx[P.reg_snp[s0 + j]] ^= 1;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        P.status_out[r] = status && sh_tie ? 2 : status;
        P.iters_out[r] = iters;
        P.ns_out[r] = lp_now() - t_beg;
    }
}

struct LpEvents {
    cudaEvent_t e[3] = {};
    ~LpEvents() {
        for (auto x : e)
            if (x) cudaEventDestroy(x);
    }
};

template <typename T>
int lp_put(xg_ctx *ctx, const char *name, const T *src, int64_t n, T **dst) {
    *dst = (T *)ctx->get(name, sizeof(T) * (size_t)std::max<int64_t>(n, 1));
    if (!*dst) return XG_E_CUDA;
    if (n > 0 && src) XG_CUDA(cudaMemcpyAsync(*dst, src, sizeof(T) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    return XG_OK;
}

}  // namespace

extern "C" int xg_local_phase(xg_ctx *ctx, int32_t n_snps, const int32_t *snp_pos, uint8_t *ref_idx,
                              const xg_phase_regions *R, uint8_t *keep_out, uint8_t *flip_out, int8_t *status_out) {
    if (!ctx || !ctx->stream) return ctx ? ctx->fail(XG_E_CUDA, "context has no device") : XG_E_ARG;
    if (!R || n_snps < 0 || (n_snps > 0 && (!snp_pos || !ref_idx)))
        return ctx->fail(XG_E_ARG, "xg_local_phase: null argument");
    const int32_t nr = R->n_regions, nw = R->n_waves;
    if (nr < 0 || nw < 0 || (nr > 0 && (!R->wave_ptr || !R->reg_snp_ptr || !R->reg_cell_ptr || !R->slot_ent_ptr ||
                                        !R->cell_ent_ptr || !keep_out || !flip_out || !status_out)))
        return ctx->fail(XG_E_ARG, "xg_local_phase: null region arrays");
    for (double &t : ctx->timing) t = 0;
    if (nr == 0) return XG_OK;
    if (R->wave_ptr[0] != 0 || R->wave_ptr[nw] != nr || R->reg_snp_ptr[0] != 0 || R->reg_cell_ptr[0] != 0)
        return ctx->fail(XG_E_ARG, "xg_local_phase: bad wave / region offsets");
    for (int32_t w = 0; w < nw; w++)
        if (R->wave_ptr[w + 1] < R->wave_ptr[w]) return ctx->fail(XG_E_ARG, "xg_local_phase: bad wave offsets");
    const int64_t n_slot = R->reg_snp_ptr[nr], n_cell = R->reg_cell_ptr[nr];
    const int64_t n_ent = R->slot_ent_ptr[n_slot];
    if (R->cell_ent_ptr[n_cell] != n_ent || R->slot_ent_ptr[0] != 0 || R->cell_ent_ptr[0] != 0)
        return ctx->fail(XG_E_ARG, "xg_local_phase: SNP-major and cell-major entries differ");
    for (int32_t r = 0; r < nr; r++) {
        const int64_t a = R->reg_snp_ptr[r], b = R->reg_snp_ptr[r + 1], c = R->reg_cell_ptr[r], d = R->reg_cell_ptr[r + 1];
        if (b < a || d < c || b - a >= INT32_MAX || d - c >= INT32_MAX ||
            R->slot_ent_ptr[a] != R->cell_ent_ptr[c] || R->slot_ent_ptr[b] != R->cell_ent_ptr[d])
            return ctx->fail(XG_E_ARG, "xg_local_phase: region " + std::to_string(r) + " has bad offsets");
    }
    for (int64_t s = 0; s < n_slot; s++)
        if (R->reg_snp[s] < 0 || R->reg_snp[s] >= n_snps)
            return ctx->fail(XG_E_ARG, "xg_local_phase: SNP index out of range");
    XG_CUDA(cudaSetDevice(ctx->device));
    const auto t_call = std::chrono::steady_clock::now();
    LpEvents ev;
    for (auto &e : ev.e) XG_CUDA(cudaEventCreate(&e));
    cudaEventRecord(ev.e[0], ctx->stream);

    LpDev P;
    memset(&P, 0, sizeof(P));
    int rc;
    int32_t *d_pos, *d_reg_snp, *d_smc, *d_sma, *d_smd, *d_cms, *d_cma, *d_cmd;
    uint8_t *d_ref;
    int64_t *d_rsp, *d_rcp, *d_sep, *d_cep;
    if ((rc = lp_put(ctx, "lp_pos", snp_pos, n_snps, &d_pos)) || (rc = lp_put(ctx, "lp_ref", ref_idx, n_snps, &d_ref)) ||
        (rc = lp_put(ctx, "lp_rsp", R->reg_snp_ptr, (int64_t)nr + 1, &d_rsp)) ||
        (rc = lp_put(ctx, "lp_rcp", R->reg_cell_ptr, (int64_t)nr + 1, &d_rcp)) ||
        (rc = lp_put(ctx, "lp_sep", R->slot_ent_ptr, n_slot + 1, &d_sep)) ||
        (rc = lp_put(ctx, "lp_cep", R->cell_ent_ptr, n_cell + 1, &d_cep)) ||
        (rc = lp_put(ctx, "lp_rs", R->reg_snp, n_slot, &d_reg_snp)) ||
        (rc = lp_put(ctx, "lp_smc", R->sm_cell, n_ent, &d_smc)) || (rc = lp_put(ctx, "lp_sma", R->sm_ad, n_ent, &d_sma)) ||
        (rc = lp_put(ctx, "lp_smd", R->sm_dp, n_ent, &d_smd)) || (rc = lp_put(ctx, "lp_cms", R->cm_snp, n_ent, &d_cms)) ||
        (rc = lp_put(ctx, "lp_cma", R->cm_ad, n_ent, &d_cma)) || (rc = lp_put(ctx, "lp_cmd", R->cm_dp, n_ent, &d_cmd)))
        return rc;
    P.snp_pos = d_pos;
    P.ref_idx = d_ref;
    P.reg_snp_ptr = d_rsp;
    P.reg_cell_ptr = d_rcp;
    P.slot_ent_ptr = d_sep;
    P.cell_ent_ptr = d_cep;
    P.reg_snp = d_reg_snp;
    P.sm_cell = d_smc;
    P.sm_ad = d_sma;
    P.sm_dp = d_smd;
    P.cm_snp = d_cms;
    P.cm_ad = d_cma;
    P.cm_dp = d_cmd;
    const int64_t ns = std::max<int64_t>(n_slot, 1), nc = std::max<int64_t>(n_cell, 1);
    {
        XG_GET(keep, uint8_t, "lp_keep", ns);
        XG_GET(flip, uint8_t, "lp_flip", ns);
        XG_GET(st, int8_t, "lp_status", nr);
        XG_GET(it, int32_t, "lp_iters", nr);
        XG_GET(tns, unsigned long long, "lp_ns", nr);
        XG_GET(kidx, int32_t, "lp_kidx", ns);
        XG_GET(wlo, int32_t, "lp_wlo", ns);
        XG_GET(whi, int32_t, "lp_whi", ns);
        XG_GET(flags, uint8_t, "lp_sflags", 3 * ns);
        XG_GET(sd, double, "lp_sd", 6 * ns);
        XG_GET(alive, uint8_t, "lp_alive", nc);
        XG_GET(dpc, int64_t, "lp_dpc", nc);
        XG_GET(cd, double, "lp_cd", 4 * nc);
        P.keep_out = keep;
        P.flip_out = flip;
        P.status_out = st;
        P.iters_out = it;
        P.ns_out = tns;
        P.kidx = kidx;
        P.wlo = wlo;
        P.whi = whi;
        P.ori = flags;
        P.ffin = flags + ns;
        P.fround = flags + 2 * ns;
        P.z0 = sd;
        P.zr = sd + ns;
        P.ll0 = sd + 2 * ns;
        P.ll1 = sd + 3 * ns;
        P.lse = sd + 4 * ns;
        P.wsum = sd + 5 * ns;
        P.alive = alive;
        P.dpc = dpc;
        P.lt0 = cd;
        P.lt1 = cd + nc;
        P.lm0 = cd + 2 * nc;
        P.lm1 = cd + 3 * nc;
    }
    cudaEventRecord(ev.e[1], ctx->stream);
    for (int32_t w = 0; w < nw; w++) {          // waves in order on one stream: no host synchronisation between them
        const int32_t b = R->wave_ptr[w], n = R->wave_ptr[w + 1] - b;
        if (n == 0) continue;
        k_local_phase<<<n, LP_THREADS, 0, ctx->stream>>>(P, b);
        XG_CUDA(cudaGetLastError());
    }
    cudaEventRecord(ev.e[2], ctx->stream);
    std::vector<int32_t> iters((size_t)nr);
    std::vector<unsigned long long> tns((size_t)nr);
    XG_CUDA(cudaMemcpyAsync(keep_out, P.keep_out, (size_t)n_slot, cudaMemcpyDeviceToHost, ctx->stream));
    XG_CUDA(cudaMemcpyAsync(flip_out, P.flip_out, (size_t)n_slot, cudaMemcpyDeviceToHost, ctx->stream));
    XG_CUDA(cudaMemcpyAsync(status_out, P.status_out, (size_t)nr, cudaMemcpyDeviceToHost, ctx->stream));
    XG_CUDA(cudaMemcpyAsync(iters.data(), P.iters_out, 4 * (size_t)nr, cudaMemcpyDeviceToHost, ctx->stream));
    XG_CUDA(cudaMemcpyAsync(tns.data(), P.ns_out, 8 * (size_t)nr, cudaMemcpyDeviceToHost, ctx->stream));
    if (n_snps > 0) XG_CUDA(cudaMemcpyAsync(ref_idx, d_ref, (size_t)n_snps, cudaMemcpyDeviceToHost, ctx->stream));
    const cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) return ctx->fail(XG_E_CUDA, std::string("local phase: ") + cudaGetErrorString(e));
    float t_all = 0, t_em = 0;
    cudaEventElapsedTime(&t_all, ev.e[0], ev.e[2]);
    cudaEventElapsedTime(&t_em, ev.e[1], ev.e[2]);
    double it_sum = 0, t_max = 0, n_tie = 0;
    for (int32_t r = 0; r < nr; r++) {
        it_sum += iters[(size_t)r];
        n_tie += status_out[r] == 2;
        t_max = std::max(t_max, tns[(size_t)r] * 1e-6);
    }
    ctx->timing[0] = t_all;
    ctx->timing[1] = t_em;
    ctx->timing[2] = nw;
    ctx->timing[3] = nr;
    ctx->timing[4] = it_sum;
    ctx->timing[5] = t_max;
    ctx->timing[6] = t_em > 0 ? t_max / t_em : 0.0;
    ctx->timing[7] = (double)n_ent;
    ctx->timing[8] = n_tie;
    ctx->timing[12] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_call).count();
    return XG_OK;
}
