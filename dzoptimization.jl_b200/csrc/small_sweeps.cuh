// small_sweeps.cuh -- the n^2 sweeps of step! for BATCHES of small matrices (32 < n <= 64): one WARP per problem.
//
// gemv_kernel / update_gemv_kernel (large_bfgs.cuh) give every problem of a batch its own CTA (blockIdx.z); at n = 64 that
// CTA has 32 working threads and a shared-memory prologue per 32 KB of matrix (0.58 of the HBM peak for 16384 problems).
// Here a lane owns RPL = 2 adjacent rows of its problem's matrix (n = 34: 0.203 -> 0.177 ms for 16384 problems, n = 64:
// 0.338 -> 0.307), a warp reads 512 contiguous bytes of every column, the vector operands are broadcast loads, and four
// problems share a CTA with nothing in common.  Per row the accumulation is the same strictly sequential walk over the
// columns (n <= 1024: a single chunk of the canonical GEMV order), so the results are those of the tiled kernels bit for bit.
// The templates take any even RPL (n <= 32 RPL), but only RPL = 2 is dispatched and tested: RPL = 4 for n <= 128 was
// measured no faster than the tiled kernels (0.549 vs 0.542 ms per step! call for 8192 problems of n = 128).
//
// legacy/DZOptimization.jl:875 (t = H * dg), :878-886 (rank-2 update, exact operation order of :882-884) fused with
// :958-960 (d = H' * g), :981 (identity_matrix! after a gradient-descent step).
#pragma once
#include "large_bfgs.cuh"

namespace dzo {

constexpr int kSmallSweepWarps = 4;      // problems per CTA
constexpr int kSmallSweepMaxN = 64;       // dispatched up to here (see above)

struct SmallSweepArgs {
    double* H;              // batch matrices of n x n, column-major, problem q at H + q*n*n
    const double* v;        // GEMV operand (delta_gradient for t, gradient for d), problem q at v + q*n
    const double* s;        // step_direction / overlap
    const double* t;        // H * delta_gradient
    double* out;            // result vector
    const LargeCtrl* ctrl;  // one control block per problem
    long long n, batch;
};

// t = H * dg for the problems whose step is BFGS-type
template <int RPL, int U>
static __global__ void __launch_bounds__(32 * kSmallSweepWarps) warp_gemv_kernel(SmallSweepArgs a) {
    const long long q = (long long)blockIdx.x * kSmallSweepWarps + (threadIdx.x >> 5);
    if (q >= a.batch) return;
    if (a.ctrl[q].kind != DZO_STEP_BFGS) return;
    const int lane = threadIdx.x & 31;
    const long long n = a.n;
    const double* H = a.H + q * n * n;
    const double* v = a.v + q * n;
    const long long i0 = (long long)RPL * lane;
    double acc[RPL];
#pragma unroll
    for (int r = 0; r < RPL; ++r) acc[r] = 0.0;
    long long j = 0;
    for (; j + U <= n; j += U) {
        double2 h[U][RPL / 2];
        double vj[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            vj[u] = v[j + u];
#pragma unroll
            for (int p = 0; p < RPL / 2; ++p)
                h[u][p] = (i0 + 2 * p < n) ? __ldcs(reinterpret_cast<const double2*>(H + (j + u) * n + i0 + 2 * p)) : make_double2(0.0, 0.0);
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int p = 0; p < RPL / 2; ++p) {
                acc[2 * p] += h[u][p].x * vj[u];
                acc[2 * p + 1] += h[u][p].y * vj[u];
            }
    }
    for (; j < n; ++j) {
        const double vj = v[j];
#pragma unroll
        for (int p = 0; p < RPL / 2; ++p)
            if (i0 + 2 * p < n) {
                const double2 h = __ldcs(reinterpret_cast<const double2*>(H + j * n + i0 + 2 * p));
                acc[2 * p] += h.x * vj;
                acc[2 * p + 1] += h.y * vj;
            }
    }
#pragma unroll
    for (int p = 0; p < RPL / 2; ++p)
        if (i0 + 2 * p < n) reinterpret_cast<double2*>(a.out + q * n + i0)[p] = make_double2(acc[2 * p], acc[2 * p + 1]);
}

// rank-2 update fused with d = H' * g (BFGS-type step), or H = I (gradient-descent step)
template <int RPL, int U>
static __global__ void __launch_bounds__(32 * kSmallSweepWarps) warp_update_gemv_kernel(SmallSweepArgs a) {
    const long long q = (long long)blockIdx.x * kSmallSweepWarps + (threadIdx.x >> 5);
    if (q >= a.batch) return;
    const int kind = a.ctrl[q].kind;
    if (kind != DZO_STEP_BFGS && kind != DZO_STEP_GRADIENT_DESCENT) return;
    const int lane = threadIdx.x & 31;
    const long long n = a.n;
    double* H = a.H + q * n * n;
    const long long i0 = (long long)RPL * lane;
    if (kind == DZO_STEP_GRADIENT_DESCENT) {                                   // :981 identity_matrix!
        for (long long j = 0; j < n; ++j)
#pragma unroll
            for (int p = 0; p < RPL / 2; ++p)
                if (i0 + 2 * p < n)
                    __stcs(reinterpret_cast<double2*>(H + j * n + i0 + 2 * p),
                           make_double2(j == i0 + 2 * p ? 1.0 : 0.0, j == i0 + 2 * p + 1 ? 1.0 : 0.0));
        return;
    }
    const double* s = a.s + q * n;
    const double* t = a.t + q * n;
    const double* g = a.v + q * n;
    const double delta = a.ctrl[q].delta_norm;
    double si[RPL], ti[RPL], acc[RPL];
#pragma unroll
    for (int r = 0; r < RPL; ++r) {
        const bool in = i0 + r < n;
        si[r] = in ? s[i0 + r] : 0.0;
        ti[r] = in ? t[i0 + r] : 0.0;
        acc[r] = 0.0;
    }
    long long j = 0;
    for (; j + U <= n; j += U) {
        double2 h[U][RPL / 2];
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int p = 0; p < RPL / 2; ++p)
                h[u][p] = (i0 + 2 * p < n) ? __ldcg(reinterpret_cast<const double2*>(H + (j + u) * n + i0 + 2 * p)) : make_double2(0.0, 0.0);
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const double sj = s[j + u], tj = t[j + u], gj = g[j + u];
#pragma unroll
            for (int p = 0; p < RPL / 2; ++p) {
                h[u][p].x = h[u][p].x + (delta * (si[2 * p] * sj) - (ti[2 * p] * sj + si[2 * p] * tj));              // :882-884
                h[u][p].y = h[u][p].y + (delta * (si[2 * p + 1] * sj) - (ti[2 * p + 1] * sj + si[2 * p + 1] * tj));
                if (i0 + 2 * p < n) __stcs(reinterpret_cast<double2*>(H + (j + u) * n + i0 + 2 * p), h[u][p]);
                acc[2 * p] += h[u][p].x * gj;                                                                         // :958-960
                acc[2 * p + 1] += h[u][p].y * gj;
            }
        }
    }
    for (; j < n; ++j) {
        const double sj = s[j], tj = t[j], gj = g[j];
#pragma unroll
        for (int p = 0; p < RPL / 2; ++p)
            if (i0 + 2 * p < n) {
                double2 h = __ldcg(reinterpret_cast<const double2*>(H + j * n + i0 + 2 * p));
                h.x = h.x + (delta * (si[2 * p] * sj) - (ti[2 * p] * sj + si[2 * p] * tj));
                h.y = h.y + (delta * (si[2 * p + 1] * sj) - (ti[2 * p + 1] * sj + si[2 * p + 1] * tj));
                __stcs(reinterpret_cast<double2*>(H + j * n + i0 + 2 * p), h);
                acc[2 * p] += h.x * gj;
                acc[2 * p + 1] += h.y * gj;
            }
    }
#pragma unroll
    for (int p = 0; p < RPL / 2; ++p)
        if (i0 + 2 * p < n) reinterpret_cast<double2*>(a.out + q * n + i0)[p] = make_double2(acc[2 * p], acc[2 * p + 1]);
}

}  // namespace dzo
