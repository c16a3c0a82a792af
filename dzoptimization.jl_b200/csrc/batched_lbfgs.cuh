// batched_lbfgs.cuh -- batches of independent live LBFGSOptimizer problems (src/DZOptimization.jl:321-509) on extended
// Rosenbrock, even n <= DZO_SMALL_N_MAX: ONE THREAD PER PROBLEM.
//
// In DZO_ORDER_SEQUENTIAL every dot product of the two-loop recursion (:430-451) is one dependent chain of n adds, so a
// team of lanes per problem would buy only shuffles and divergence; the parallelism comes from the batch.  Thread p owns
// problem p for the constructor (mode 1, :347-427) and for k consecutive step! calls (mode 0, :454-509).  x, g and d
// live in registers (the kernel is a template on n), every sum runs strictly left to right, and every operation is the
// one of lbfgs_step_one / lbfgs_direction in oracle/dzo_oracle.c, in the same order: the bits are those of `batch`
// separate oracle handles in DZO_ORDER_SEQUENTIAL.
//
// Device layout: the batch is innermost in every array -- element e of problem p at e*batch + p, element e of history
// slot s at (s*n + e)*batch + p, rho of slot s at s*batch + p -- so a warp's load of one element is 256 contiguous bytes.
// The history is a ring with a per-problem head (logical slot i = physical slot (head + i) mod m, as LbfgsCtrl.head):
// nothing is shifted.  The live problems of a batch all advance one iteration per step!, so their heads agree and the
// history loads stay coalesced; correctness does not depend on it.
//
// take_backtracking_step! (:107-154) halves forever when no trial point is ever isequal to the current point (a NaN in
// the direction; a -0.0 coordinate whose direction is +0.0).  One such problem would hang a whole launch, so the loop
// here runs at most DZO_LINESEARCH_CAP trials and then takes the reference's not-accepted branch (delta_point = the copy
// of the point, :118; is_stuck).  [GLUE] This changes no input on which the reference terminates: from step 1.0 the
// step reaches exactly 0 after 1075 halvings, after which the trial point is the point itself.
#pragma once
#include "common.cuh"
#include "large_bfgs.cuh"      // RosenbrockVec
#include "lbfgs_kernels.cuh"   // julia_isequal

namespace dzo {

constexpr int kBatchedLbfgsMaxThreads = 256;

struct BatchedLbfgsArgs {
    double *x, *dx, *g, *dg, *d;     // n x batch, batch innermost
    double *S, *Y;                   // m slots of n x batch
    double* rho;                     // m x batch, PHYSICAL slots
    double *f, *df;                  // batch
    long long* iter;                 // batch
    int *count, *head;               // batch: valid history entries, physical slot of the newest one
    unsigned char* stuck;            // batch
    long long batch;
    int m, ksteps;
    int mode;                        // 0 = ksteps step! calls, 1 = constructor (x already holds the initial points)
    double initial_step_length;
};

// dynamic shared memory: alpha of the first loop, m x blockDim.x doubles
template <int N>
__global__ void __launch_bounds__(kBatchedLbfgsMaxThreads) batched_lbfgs_kernel(BatchedLbfgsArgs a) {
    extern __shared__ double alpha_sm[];
    const long long B = a.batch;
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= B) return;
    double* alpha = alpha_sm + threadIdx.x;
    const int T = blockDim.x;
    double d[N];

    if (a.mode == 1) {                                                                      // :347-427
        double x[N], g[N];
#pragma unroll
        for (int e = 0; e < N; ++e) x[e] = a.x[e * B + p];
        double f = 0.0;
#pragma unroll
        for (int k = 0; k < N / 2; ++k) f += RosenbrockVec::term(x[2 * k], x[2 * k + 1]);  // :417
#pragma unroll
        for (int k = 0; k < N / 2; ++k) {                                                   // :419-422
            const double2 gg = RosenbrockVec::grad(x[2 * k], x[2 * k + 1]);
            g[2 * k] = gg.x; g[2 * k + 1] = gg.y;
        }
        double nn = 0.0;
#pragma unroll
        for (int e = 0; e < N; ++e) nn += g[e] * g[e];
        const double gnorm = sqrt(nn);                                                      // :376
        const bool stuck = (gnorm == 0.0);                                                  // :377
        const double c = -a.initial_step_length / gnorm;
#pragma unroll
        for (int e = 0; e < N; ++e) {
            a.g[e * B + p] = g[e];
            a.d[e * B + p] = stuck ? 0.0 : g[e] * c;                                        // :378-383
            a.dx[e * B + p] = 0.0;                                                          // :367
            a.dg[e * B + p] = 0.0;                                                          // :372
        }
        a.f[p] = f; a.df[p] = 0.0; a.iter[p] = 0; a.count[p] = 0; a.head[p] = 0; a.stuck[p] = stuck;
        return;
    }

    if (a.stuck[p]) return;                                                                 // :456-458
    const int m = a.m;
    double f = a.f[p], df = a.df[p];
    long long iter = a.iter[p];
    int cnt = a.count[p], head = a.head[p];
    bool stuck = false;
    if (iter == 0) {
#pragma unroll
        for (int e = 0; e < N; ++e) d[e] = a.d[e * B + p];                                  // the constructor's direction
    }
    const long long slot_stride = (long long)N * B;

    #pragma unroll 1
    for (int step_i = 0; step_i < a.ksteps; ++step_i) {
        if (iter > 0) {
            // compute_lbfgs_step_direction!  :430-451 (logical slot i -> physical (head + i) mod m)
#pragma unroll
            for (int e = 0; e < N; ++e) d[e] = a.g[e * B + p];
            double yy = 0.0;                                                                // dot(y_0, y_0), :443
            #pragma unroll 1
            for (int i = 0; i < cnt; ++i) {
                int s = head + i;
                if (s >= m) s -= m;
                const double* Sp = a.S + s * slot_stride + p;
                const double* Yp = a.Y + s * slot_stride + p;
                double dot = 0.0;
#pragma unroll
                for (int e = 0; e < N; ++e) dot += Sp[e * B] * d[e];
                const double al = dot / a.rho[s * B + p];                                   // :439
                alpha[i * T] = al;
                const double na = -al;
                if (i == 0) {
#pragma unroll
                    for (int e = 0; e < N; ++e) {
                        const double y = Yp[e * B];
                        d[e] += na * y;                                                     // :440
                        yy += y * y;
                    }
                } else {
#pragma unroll
                    for (int e = 0; e < N; ++e) d[e] += na * Yp[e * B];                     // :440
                }
            }
            if (cnt > 0) {
                const double c = -a.rho[head * B + p] / yy;                                 // :443
#pragma unroll
                for (int e = 0; e < N; ++e) d[e] *= c;
            }
            #pragma unroll 1
            for (int i = cnt - 1; i >= 0; --i) {
                int s = head + i;
                if (s >= m) s -= m;
                const double* Sp = a.S + s * slot_stride + p;
                const double* Yp = a.Y + s * slot_stride + p;
                double dot = 0.0;
#pragma unroll
                for (int e = 0; e < N; ++e) dot += Yp[e * B] * d[e];
                const double beta = dot / a.rho[s * B + p];                                 // :446
                const double na = -(alpha[i * T] + beta);
#pragma unroll
                for (int e = 0; e < N; ++e) d[e] += na * Sp[e * B];                         // :447
            }
#pragma unroll
            for (int e = 0; e < N; ++e) a.d[e * B + p] = d[e];
        }
        // take_backtracking_step!(opt, 1, step_direction)  :107-154, at most DZO_LINESEARCH_CAP trials (header comment)
        double x[N];
#pragma unroll
        for (int e = 0; e < N; ++e) x[e] = a.x[e * B + p];
        double step = 1.0, next = 0.0;
        bool accepted = false;
        #pragma unroll 1
        for (int trial = 0; trial < DZO_LINESEARCH_CAP; ++trial) {
            bool same = true;
            double acc = 0.0;
#pragma unroll
            for (int k = 0; k < N / 2; ++k) {
                const double w0 = x[2 * k] + step * d[2 * k], w1 = x[2 * k + 1] + step * d[2 * k + 1];   // :124 axpy!
                same &= julia_isequal(w0, x[2 * k]) & julia_isequal(w1, x[2 * k + 1]);                    // :128
                acc += RosenbrockVec::term(w0, w1);                                                       // :138
            }
            if (same) break;                                                                // :128-131
            if (acc < f) { next = acc; accepted = true; break; }                            // :139
            step *= 0.5;                                                                    // :152
        }
        if (!accepted) {
            // delta_point keeps the COPY of the point (:118); x, g, dg, f, df, iteration_count and the history stay
#pragma unroll
            for (int e = 0; e < N; ++e) a.dx[e * B + p] = x[e];
            stuck = true;
            break;
        }
        // accept: x, delta_point (:145), gradient and delta_gradient (:478-480), history push (:482-505)
        int slot = head - 1;
        if (slot < 0) slot += m;
        double* Sn = a.S + slot * slot_stride + p;
        double* Yn = a.Y + slot * slot_stride + p;
        double go[N];                                   // loaded before the stores below, which the compiler must assume alias
#pragma unroll
        for (int e = 0; e < N; ++e) go[e] = a.g[e * B + p];
        double r = 0.0;
#pragma unroll
        for (int k = 0; k < N / 2; ++k) {
            const double xn0 = x[2 * k] + step * d[2 * k], xn1 = x[2 * k + 1] + step * d[2 * k + 1];
            const double dx0 = 1.0 * xn0 + (-1.0) * x[2 * k], dx1 = 1.0 * xn1 + (-1.0) * x[2 * k + 1];   // axpby!
            const long long e0 = (long long)(2 * k) * B, e1 = (long long)(2 * k + 1) * B;
            const double2 gn = RosenbrockVec::grad(xn0, xn1);
            const double dg0 = 1.0 * gn.x + (-1.0) * go[2 * k], dg1 = 1.0 * gn.y + (-1.0) * go[2 * k + 1];
            r += dx0 * dg0;                                                                 // :505
            r += dx1 * dg1;
            a.x[e0 + p] = xn0; a.x[e1 + p] = xn1;
            a.dx[e0 + p] = dx0; a.dx[e1 + p] = dx1;
            a.g[e0 + p] = gn.x; a.g[e1 + p] = gn.y;
            a.dg[e0 + p] = dg0; a.dg[e1 + p] = dg1;
            Sn[e0] = dx0; Sn[e1] = dx1;
            Yn[e0] = dg0; Yn[e1] = dg1;
        }
        df = next - f;                                                                      // :142
        f = next;                                                                           // :143
        a.rho[slot * B + p] = r;
        head = slot;
        cnt = (cnt < m) ? cnt + 1 : m;
        iter += 1;                                                                          // :507
    }
    a.f[p] = f; a.df[p] = df; a.iter[p] = iter; a.count[p] = cnt; a.head[p] = head;
    if (stuck) a.stuck[p] = 1;
}

}  // namespace dzo
