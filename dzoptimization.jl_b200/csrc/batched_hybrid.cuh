// batched_hybrid.cuh -- batched small-n BFGS step! (every even n <= 32): the kernel behind BASELINE configs[1].
//
// Same arithmetic and the same SEQUENTIAL summation order (legacy/Kernels.jl:12-20) as the sequential oracle, hence the
// same bits.  A warp owns a TILE of 32 problems and works in two phases per step!:
//
//   phase 1  ONE THREAD PER PROBLEM (32 problems per instruction): norms, both bracketing line searches as ONE
//            per-thread state machine whose loop body is exactly one probe evaluation (so lanes in different stages of
//            different searches share the expensive code), the BFGS / GD / terminate decision, overlap.
//            The vectors live in a per-warp shared-memory tile [32 problems][n + 2] (16-byte aligned rows).
//   phase 2  NP LANES PER PROBLEM (NP = n rounded up to a power of two), uniform control flow: lane r recomputes element r
//            of x, g, dx, dg (bit-identical elementwise formulas) and stores them coalesced (the derived layout stores
//            only x, into the other point buffer), streams ROW r of the
//            inverse Hessian from HBM into registers with coalesced loads (for a fixed column the lanes of a problem
//            read n consecutive doubles; two register tiles ping-pong so the next round's rows are in flight while the
//            current round computes; tiles further ahead are pulled into L2 with prefetch.global.L2), t = H*dg,
//            delta, the rank-2 update fused with d = H'*g, rows streamed back.
//
// What round 2 changed (each step A/B'd inside one gpurun call, profiles/README.md; 0.89 -> 0.74 ms per 1M-problem launch):
//   * LAZY identity: identity_matrix! (:981) after a gradient-descent step is not written to HBM; a per-problem byte
//     `flags` bit BF_IDENT says "H is the identity, the copy in HBM is stale".  The next BFGS-type step builds its rows of I in registers
//     instead of loading them (the same arithmetic on the same values), the constructor writes no H at all, and
//     dzo_bfgs_get_inverse_hessian materialises I for the caller.  A GD-type step moves 1.1 KB instead of 3.1 KB and a
//     BFGS-type step after it 3.1 KB instead of 5.2 KB (n = 16).
//   * phase 1 hands its per-problem results to phase 2 through the two spare doubles of each tile row instead of
//     registers + shuffles; the per-problem scalars are stored right after phase 1.  ncu had shown 17 % of all stall
//     samples on two local-memory reloads (the 28 KB of L1 left beside the tile do not hold the spills of 16 warps).
//   * a tile starts cold, so everything it needs first is requested at once: the vectors as 16-byte cp.async copies
//     straight into the tile, flags and scalars as loads in flight beside them; iteration_count is bumped with a
//     fire-and-forget reduction.
//   * the (w == reference point) test of the expansion loop (:150) is evaluated only while some lane is expanding.
//   * per-launch step-kind counters (warp ballots -> one atomicAdd per warp and kind) feed bench.py's roofline.
//   Measured and rejected: both line searches side by side in one thread (0.95 ms: register spills in the probe loop, and
//   max(probes) per iteration of two searches costs more issue slots than the shared state machine); persistent CTAs with
//   tiles handed to warps through a counter (0.80 ms: 2.0 instead of 0.3 no-instruction stall cycles per issue).
// What round 3 changed: the DERIVED layout (Tuning::batched_derived).  g is always rosenbrock_gradient!(x) and dx, dg are
//   differences of two points, so a move writes its new x into the second point buffer (the old x stays in the first)
//   and stores no g, dx or dg; the tile's G rows are recomputed from X after staging, and the getters recompute the
//   fields bit for bit from the two points (flags bits BF_PARITY / BF_EXPLICIT, batched_bfgs.cuh).  512 B less per
//   moving problem-step at n = 16 (DESIGN.md section 3).
//
// legacy/DZOptimization.jl:891-994 (step!), :864-889 (update_inverse_hessian!), :49-216 (line search).
#pragma once
#include <cstdlib>

#include "batched_bfgs.cuh"

namespace dzo {

#ifndef DZO_HYBRID_WARPS
#define DZO_HYBRID_WARPS 4              // warps per CTA (A/B knob of tools/build_variant.sh; 16 / 8 warps per SM in total either way)
#endif
constexpr int kHybridWarps = DZO_HYBRID_WARPS;
constexpr int kHybridThreads = 32 * kHybridWarps;

template <int N>
struct HybridCfg {
    static_assert(N >= 2 && N <= 32 && N % 2 == 0, "hybrid mapping: even n <= 32");
    static constexpr int NP = N <= 2 ? 2 : N <= 4 ? 4 : N <= 8 ? 8 : N <= 16 ? 16 : 32;   // lanes per problem in phase 2
    static constexpr int PPR = 32 / NP;                     // problems per phase-2 round
    static constexpr int ROUNDS = NP;                       // 32 / PPR
    static constexpr int STRIDE = (N <= 16) ? 18 : N + 2;   // doubles per tile row: the elements + two hand-off slots,
                                                            // 16-byte aligned rows (phase 2 reads pairs with one 128-bit load)
    static constexpr int SLOT = STRIDE - 2;
    static constexpr bool PINGPONG = (N <= 16);             // two register tiles of n doubles each
    static constexpr int CTAS_PER_SM = ((N <= 16) ? 16 : 8) / kHybridWarps;   // 16 / 8 warps per SM: what the shared tile
                                                                              // (14 KB ... 26 KB per warp) allows
};

template <int N>
struct HybridSmem {
    using C = HybridCfg<N>;
    alignas(16) double X[32][C::STRIDE];       // current_point          -> in phase 2: delta_gradient
    alignas(16) double G[32][C::STRIDE];       // current_gradient (staged, or recomputed from X by the derived layout)
                                               //                        -> in phase 2: new gradient
    alignas(16) double D[32][C::STRIDE];       // next_step_direction    -> after phase 1: step_direction / overlap
    alignas(16) double T[C::PPR][C::NP];       // scratch = H * delta_gradient of the problems of the current round
    alignas(16) double P[C::PPR][C::NP];       // products for the sequential dot of :876
};
// The two spare doubles of the three rows of problem q carry what phase 1 hands to phase 2:
//   X[q][SLOT]    lane q < HK_COUNT: running step-kind counter q of this warp     X[q][SLOT+1]  alpha = -step length (:945/:973)
//   G[q][SLOT]    alpha * overlap  (first operand of :876)                         G[q][SLOT+1]  1 / overlap          (:874)
//   D[q][SLOT]    low word: step kind | where H comes from << 8 | x goes to g << 16  D[q][SLOT+1]  (free)

enum : int { HS_INIT = 0, HS_EXPAND = 1, HS_SHRINK = 2, HS_QUAD = 3, HS_DONE = 4 };

DZO_DEVINL void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

struct HybridSearch {
    int st;
    int cap;
    double step, fa, xb, fb, trial, tref;
};

// QuadraticLineSearch  :196-214 on a finished bracket (0, f0), (x1, f1), (x2, f2): best of the three, then either the
// parabola-vertex probe (HS_QUAD) or done.  The bracket itself never outlives this call.
DZO_DEVINL void hs_bracket(HybridSearch& s, double f0, double x1, double f1, double x2, double f2) {
    s.xb = 0.0; s.fb = f0;
    if (f1 < s.fb) { s.xb = x1; s.fb = f1; }
    if (f2 < s.fb) { s.xb = x2; s.fb = f2; }
    const double delta_1 = f0 - f1;
    const double delta_2 = f2 - f1;
    const double sum_deltas = delta_1 + delta_2;
    if (delta_1 >= 0.0 && delta_2 >= 0.0 && sum_deltas > 0.0) {
        const double twice_delta_1 = delta_1 + delta_1;
        const double delta_ratio = (twice_delta_1 + sum_deltas) / (sum_deltas + sum_deltas);
        s.trial = delta_ratio * x1;
        s.st = HS_QUAD;
    } else {
        s.st = HS_DONE;
    }
}
// find_three_point_bracket prologue  :64-85 (+ [GLUE] guards), first trial step t1 = L / norm.  The degenerate
// bracket (0,f0,0,f0) of the early returns resolves to (t*, f*) = (0, f0) without a probe (:196-206 with all deltas 0).
template <int N>
DZO_DEVINL void hs_setup(HybridSearch& s, const double* dir, double f0, double t1, bool active) {
    s.xb = 0.0; s.fb = f0; s.fa = 0.0;
    s.step = t1; s.trial = t1; s.tref = 0.0; s.cap = DZO_LINESEARCH_CAP;
    s.st = active ? HS_INIT : HS_DONE;
    if (active) {
        bool zero = true;
#pragma unroll
        for (int i = 0; i < N; ++i) zero &= (dir[i] == 0.0);
        if (!isfinite(f0) || !isfinite(t1) || t1 == 0.0 || zero) s.st = HS_DONE;
    }
}
// one probe result -> next state  (:91-101, :126-170, :210-213)
DZO_DEVINL void hs_advance(HybridSearch& s, double f0, double fv, bool changed, bool same) {
    if (s.st == HS_INIT) {
        if (!changed) {                                                       // :91-101
            s.step += s.step; s.trial = s.step;
            if (--s.cap == 0) s.st = HS_DONE;                                 // [GLUE] bracket (0,f0,0,f0)
        } else {                                                              // :126
            s.fa = fv;
            s.cap = DZO_LINESEARCH_CAP;
            if (s.fa <= f0) { s.st = HS_EXPAND; s.tref = s.step; s.trial = s.step + s.step; }   // :130-136
            else { s.st = HS_SHRINK; s.trial = 0.5 * s.step; }                                  // :157
        }
    } else if (s.st == HS_EXPAND) {                                           // :143-156
        --s.cap;
        if (!isfinite(fv) || fv > s.fa || same || s.cap == 0) {
            hs_bracket(s, f0, s.step, s.fa, s.trial, fv);
        } else {
            s.step = s.trial; s.fa = fv; s.tref = s.step; s.trial = s.step + s.step;
        }
    } else if (s.st == HS_SHRINK) {                                           // :162-170
        --s.cap;
        if (fv <= f0 || s.cap == 0) {
            hs_bracket(s, f0, s.trial, fv, s.step, s.fa);
        } else {
            s.step = s.trial; s.fa = fv; s.trial = 0.5 * s.step;
        }
    } else if (s.st == HS_QUAD) {                                             // :210-213
        if (fv < s.fb) { s.xb = s.trial; s.fb = fv; }
        s.st = HS_DONE;
    }
}

// lse(t): w = x + (-t)*dir ; f(w)   (sign fixed by :945,:973).  SAME: also compare w with the reference point x + (-tref)*dir (:150)
template <int N, bool SAME>
DZO_DEVINL void hs_probe(const double* X, const double* Dir, double a, double ar, double& fv, bool& ch, bool& sm) {
    const double2* X2 = reinterpret_cast<const double2*>(X);
    const double2* D2 = reinterpret_cast<const double2*>(Dir);
    fv = 0.0; ch = false; sm = true;
#pragma unroll
    for (int k = 0; k < N / 2; ++k) {
        const double2 x = X2[k], d = D2[k];
        const double w0 = x.x + a * d.x, w1 = x.y + a * d.y;
        ch |= (x.x != w0) | (x.y != w1);
        if (SAME) {
            const double r0 = x.x + ar * d.x, r1 = x.y + ar * d.y;
            sm &= (w0 == r0) & (w1 == r1);
        }
        const double t1_ = 1 - w0;
        const double t2_ = w1 - w0 * w0;
        fv += t1_ * t1_ + 100 * (t2_ * t2_);                                  // legacy/ExampleFunctions.jl:10-15
    }
}

// step kinds as counted for the roofline (include/dzopt.h, dzo_bfgs_get_step_kind_counts)
enum : int { HK_BFGS_READ = 0, HK_BFGS_IDENT = 1, HK_GD = 2, HK_TERMINATE = 3, HK_IDLE = 4, HK_IDLE_WARP = 5, HK_COUNT = 6 };

// VTILE: problems per warp taken from A.tile (small batches) instead of the compile-time 32 -- a second instantiation
// because the run-time tile costs the n = 16 kernel two more spilled registers (0.699 -> 0.706 ms per 1 M-problem launch).
// DERIVED: the layout of BatchedArgs::derived, a template parameter for the same reason (run-time branches on it cost
// the n = 16 full-tile kernel 8 more bytes of spill stores).
template <int N, bool VTILE, bool DERIVED>
__global__ void __launch_bounds__(kHybridThreads, HybridCfg<N>::CTAS_PER_SM) bfgs_batched_hybrid_kernel(BatchedArgs A) {
    using C = HybridCfg<N>;
    static_assert(HK_COUNT <= 32, "one counter per lane");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr unsigned FULL = 0xffffffffu;
    constexpr int NN = N * N;
    constexpr int NP = C::NP, PPR = C::PPR, SLOT = C::SLOT;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    HybridSmem<N>& S = reinterpret_cast<HybridSmem<N>*>(smem_raw)[warp];
    // A tile is A.tile <= 32 consecutive problems (32 for a large batch; the host shrinks it when the batch would fill the
    // GPU's warp slots only a few times over, so that the last wave of warps is as full as the first)
    const int tile = VTILE ? A.tile : 32;
    const long long p0 = ((long long)blockIdx.x * kHybridWarps + warp) * tile;  // first problem of this warp's tile
    if (p0 >= A.batch) return;
    const long long p = p0 + lane;
    const bool valid = VTILE ? (lane < tile && p < A.batch) : (p < A.batch);
    const int nprob = (int)((A.batch - p0 < tile) ? (A.batch - p0) : tile);
    const bool lazy = A.lazy != 0;
    constexpr bool derived = DERIVED;

    // A tile starts cold: everything it needs first is requested at once -- the vectors as 16-byte asynchronous copies
    // straight into the shared tile (no registers held), flags and scalars as ordinary loads in flight beside them.
    // The derived layout copies no g (filled from X below) and takes x of problem q from g when bit q of `odd` is set;
    // `odd` is a ballot of the flags bytes, so its first copies wait for the flags load (one dependent round trip per
    // tile; not measured on its own -- the layout A/B in profiles/ includes it).
    auto stage_vectors = [&](unsigned odd) {
        for (int e2 = lane; e2 < nprob * (N / 2); e2 += 32) {
            const int q = (2 * e2) / N, i = 2 * e2 - q * N;
            cp_async16(&S.X[q][i], (((odd >> q) & 1u) ? A.g : A.x) + p0 * N + 2 * e2);
            if (!derived) cp_async16(&S.G[q][i], A.g + p0 * N + 2 * e2);
            cp_async16(&S.D[q][i], A.d + p0 * N + 2 * e2);
        }
        cp_async_commit();
    };
    unsigned fl = (valid && (lazy || derived)) ? A.flags[p] : 0u;   // BF_* (batched_bfgs.cuh)
    stage_vectors(derived ? __ballot_sync(FULL, (fl & BF_PARITY) != 0u) : 0u);
    bool term = valid ? (A.term[p] != 0) : true;
    bool moved_any = false;
    double& cnt_slot = S.X[lane][SLOT];                        // lane k < HK_COUNT: running counter k (exact below 2^53)
    cnt_slot = 0.0;
    auto count = [&](int k, unsigned ballot) { if (lane == k) cnt_slot += (double)__popc(ballot); };

    for (int s = 0; s < A.ksteps; ++s) {
        if (!__any_sync(FULL, !term)) {
            if (lane == HK_IDLE_WARP) cnt_slot += (double)nprob * (double)(A.ksteps - s);
            cp_async_wait_all();
            break;
        }
        if (s > 0) {
            // a later step of the same launch: the vectors were stored by other lanes of this warp in phase 2
            __threadfence_block();
            __syncwarp();
            stage_vectors(derived ? __ballot_sync(FULL, (fl & BF_PARITY) != 0u) : 0u);
        }
        const bool ident = lazy && (fl & BF_IDENT);    // H == I and the copy in HBM is stale
        double f0 = valid ? A.f[p] : 0.0;              // (a later step of the same launch reads back its own stores)
        double L = valid ? A.L[p] : 0.0;
        const double* X = S.X[lane];
        const double* G = S.G[lane];
        const double* D = S.D[lane];
        // Pull the inverse Hessians of the first phase-2 rounds into L2 now: they arrive while phase 1 computes.  One
        // 128-byte line per lane and request; tiles of terminated problems and of problems whose H is the
        // (unmaterialised) identity are skipped.
        const bool term_in = term;
        unsigned live = __ballot_sync(FULL, !term && !ident);  // before phase 1: every problem that MAY read its H; after
                                                               // phase 1: exactly those that do (a gradient-descent step and a
                                                               // termination do not -- ncu: the blind prefetch read 0.4 GB per
                                                               // launch that nobody used)
        auto prefetch_round = [&](int round) {
            if (round >= C::ROUNDS) return;
            const char* base = reinterpret_cast<const char*>(A.H + (p0 + round * PPR) * NN);
            if constexpr ((NN * 8) % 128 == 0) {               // a problem's H is a whole number of lines (n = 4, 8, 12, 16, ...)
                constexpr int LINES = PPR * NN * 8 / 128;
                for (int l = lane; l < LINES; l += 32) {
                    const int q = round * PPR + (l * 128) / (NN * 8);
                    if ((live >> q) & 1u) prefetch_l2(base + l * 128);
                }
            } else {                                           // lines straddle problems: all lines of a round with live problems
                constexpr int LINES = (PPR * NN * 8 + 127) / 128 + 1;
                const unsigned in_round = (PPR == 32) ? live : ((live >> (round * PPR)) & ((1u << PPR) - 1u));
                const char* first = reinterpret_cast<const char*>(reinterpret_cast<uintptr_t>(base) & ~uintptr_t(127));
                if (in_round)
                    for (int l = lane; l < LINES; l += 32) prefetch_l2(first + l * 128);
            }
        };
        for (int rr = 0; rr < A.prefetch_rounds; ++rr) prefetch_round(rr);
        cp_async_wait_all();
        __syncwarp();
        if (derived) {
            // g = rosenbrock_gradient!(x): the bits the old layout stored and staged
            for (int e2 = lane; e2 < nprob * (N / 2); e2 += 32) {
                const int q = (2 * e2) / N, i = 2 * e2 - q * N;
                const double2 x2 = *reinterpret_cast<const double2*>(&S.X[q][i]);
                *reinterpret_cast<double2*>(&S.G[q][i]) = rosen_pair_grad(x2.x, x2.y);
            }
            __syncwarp();
        }

        // ---------------------------------------------------------------- phase 1: one thread per problem
        {
            int kind = DZO_STEP_NULL;
            double alpha = 0.0, overlap = 0.0;
            double grad_norm = 0.0, bfgs_norm = 0.0;
            if (!term) {
                double sg = 0.0, sd = 0.0;
#pragma unroll
                for (int i = 0; i < N; ++i) { sg += G[i] * G[i]; sd += D[i] * D[i]; }   // :921, :928
                grad_norm = sqrt(sg);
                bfgs_norm = sqrt(sd);
            }
            // one search after the other, but as ONE per-thread state machine whose loop body is exactly one probe
            // evaluation: lanes in different stages of different searches share the expensive code
            HybridSearch sc;
            int which = 0;
            double grad_step_length = 0.0, grad_obj = f0;
            hs_setup<N>(sc, G, f0, L / grad_norm, !term);                                 // :922
            for (;;) {
                if (sc.st == HS_DONE && which == 0 && !term) {
                    grad_step_length = sc.xb; grad_obj = sc.fb;
                    which = 1;
                    hs_setup<N>(sc, D, f0, L / bfgs_norm, true);                          // :929
                }
                if (!__any_sync(FULL, sc.st != HS_DONE)) break;
                const double* dir = which ? D : G;
                double fv;
                bool ch, sm;
                if (__any_sync(FULL, sc.st == HS_EXPAND)) hs_probe<N, true>(X, dir, -sc.trial, -sc.tref, fv, ch, sm);
                else hs_probe<N, false>(X, dir, -sc.trial, -sc.tref, fv, ch, sm);
                hs_advance(sc, f0, fv, ch, sm);
            }
            const double bfgs_step_length = sc.xb, bfgs_obj = sc.fb;
            // ---- decision and bookkeeping  :934-990
            if (!term) {
                if (bfgs_obj < f0 && !(bfgs_obj > grad_obj)) {                            // :934
                    kind = DZO_STEP_BFGS; alpha = -bfgs_step_length;
                    L = bfgs_step_length * bfgs_norm; f0 = bfgs_obj;                      // :937-938
                } else if (grad_obj < f0) {                                               // :962
                    kind = DZO_STEP_GRADIENT_DESCENT; alpha = -grad_step_length;
                    L = grad_step_length * grad_norm; f0 = grad_obj;                      // :965-966
                } else {
                    term = true;                                                          // :989
                }
            }
            if (kind == DZO_STEP_BFGS) {
                // overlap = dot(step_direction, delta_gradient)  :873 -- thread-local and strictly sequential.
                // The elementwise results (x, g, dx, dg, d/overlap) are recomputed bit-identically by the
                // phase-2 lanes, which store the ones the layout keeps coalesced.
#pragma unroll
                for (int k = 0; k < N / 2; ++k) {
                    const double xa = X[2 * k], xc = X[2 * k + 1];
                    const double ga = G[2 * k], gc = G[2 * k + 1];
                    const double da = D[2 * k], dc = D[2 * k + 1];
                    const double na = xa + alpha * da, nc = xc + alpha * dc;              // :945
                    const double t1_ = 1 - na;
                    const double t2_ = nc - na * na;
                    const double gna = -2 * t1_ - 400 * na * t2_;                         // :948 rosenbrock_gradient!
                    const double gnc = 200 * t2_;
                    const double dga = (-ga) + gna, dgc = (-gc) + gnc;                    // :944, :950
                    overlap += da * dga;
                    overlap += dc * dgc;
                }
            }
            // what this step does to each problem, for the roofline (uniform across the warp)
            count(HK_BFGS_READ, __ballot_sync(FULL, kind == DZO_STEP_BFGS && !ident));
            count(HK_BFGS_IDENT, __ballot_sync(FULL, kind == DZO_STEP_BFGS && ident));
            count(HK_GD, __ballot_sync(FULL, kind == DZO_STEP_GRADIENT_DESCENT));
            count(HK_TERMINATE, __ballot_sync(FULL, valid && term && !term_in));
            count(HK_IDLE, __ballot_sync(FULL, valid && term_in));
            // ---- the per-problem scalars are final for this step: store them now, hand the rest to phase 2 through the tile
            const int hsrc = (kind == DZO_STEP_BFGS) ? (ident ? 2 : 1) : 0;   // rows from HBM (1) or the implicit identity (2)
            live = __ballot_sync(FULL, hsrc == 1);
            if (valid) {
                if (kind != DZO_STEP_NULL) {
                    A.f[p] = f0;
                    A.L[p] = L;
                    atomicAdd(reinterpret_cast<unsigned long long*>(A.iter + p), 1ull);  // :940 / :968 (no load to wait for)
                    A.type[p] = kind;                                                     // :939 / :967
                    moved_any = true;
                }
                if (term && !term_in) {
                    A.term[p] = 1;
                    if (A.term_host) A.term_host[p] = 1;
                }
                const bool ident_next = (kind == DZO_STEP_BFGS) ? false : ((kind == DZO_STEP_GRADIENT_DESCENT) ? lazy : ident);
                unsigned fl_next = ident_next ? (fl | BF_IDENT) : (fl & ~BF_IDENT);
                if (derived && kind != DZO_STEP_NULL) fl_next = (fl_next ^ BF_PARITY) & ~BF_EXPLICIT;   // x moves to the other buffer
                if (fl_next != fl) A.flags[p] = (unsigned char)fl_next;
                fl = fl_next;
            }
            S.X[lane][SLOT + 1] = alpha;
            S.G[lane][SLOT] = alpha * overlap;                                            // first operand of :876
            S.G[lane][SLOT + 1] = 1.0 / overlap;                                          // :874 inv(overlap)
            reinterpret_cast<int*>(&S.D[lane][SLOT])[0] = kind | (hsrc << 8) | ((derived && (fl & BF_PARITY)) ? (1 << 16) : 0);
        }
        __syncwarp();

        // ---------------------------------------------------------------- phase 2: NP lanes per problem
        // Lane r < n of problem q owns element r of every vector and row r of H.  Every global access below
        // is coalesced: for a fixed instruction the lanes of a problem touch n consecutive doubles.
        const int r = lane % NP, sub = lane / NP;
        const bool act = r < N;
        const unsigned gmask = ((N == 32) ? FULL : ((1u << N) - 1u)) << (sub * NP);      // the n lanes of my problem
        auto load_rows = [&](int round, double (&row)[N], int& meta) {
            const int q = round * PPR + sub;
            meta = reinterpret_cast<const int*>(&S.D[q][SLOT])[0];
            if (act && ((meta >> 8) & 0xff) == 1) {
                const double* Hp = A.H + (p0 + q) * NN + r;          // H[r, j] at Hp[j*N] (column-major)
#pragma unroll
                for (int j = 0; j < N; ++j) row[j] = __ldcs(Hp + j * N);
            }
        };
        auto process = [&](int round, double (&cur)[N], int meta) {
            const int kcur = meta & 0xff;
            if (!act || kcur == DZO_STEP_NULL) return;
            const int q = round * PPR + sub;
            const long long e = (p0 + q) * N + r;
            const double xo = S.X[q][r], go = S.G[q][r], dol = S.D[q][r];
            const double alpha_q = S.X[q][SLOT + 1];
            const double dirv = (kcur == DZO_STEP_BFGS) ? dol : go;
            const double xn = xo + alpha_q * dirv;                                    // :945 / :973
            const double xp = __shfl_xor_sync(gmask, xn, 1);                          // the other element of my pair
            const double xe = (r & 1) ? xp : xn, xod = (r & 1) ? xn : xp;
            const double t1_ = 1 - xe;
            const double t2_ = xod - xe * xe;
            const double gn = (r & 1) ? (200 * t2_) : (-2 * t1_ - 400 * xe * t2_);    // :948 rosenbrock_gradient!
            const double dgv = (-go) + gn;                                            // :944, :950
            ((derived && (meta >> 16)) ? A.g : A.x)[e] = xn;                          // derived: the buffer the flags now name
            if (!derived) {
                A.g[e] = gn;
                A.dx[e] = (-xo) + xn;                                                 // :943, :949
                A.dg[e] = dgv;
            }
            double* Hp = A.H + (p0 + q) * NN + r;
            if (kcur == DZO_STEP_BFGS) {
                // update_inverse_hessian!  :874-886 fused with mul!(d, H, g)  :958-960
                const double ao_q = S.G[q][SLOT], inv_overlap_q = S.G[q][SLOT + 1];
                if (((meta >> 8) & 0xff) == 2) {
#pragma unroll
                    for (int j = 0; j < N; ++j) cur[j] = (j == r) ? 1.0 : 0.0;        // the rows identity_matrix! would have left
                }
                const double sd = dol * inv_overlap_q;                                // :874
                __syncwarp(gmask);              // every lane has read the old tile values
                S.X[q][r] = dgv;
                S.G[q][r] = gn;
                S.D[q][r] = sd;
                __syncwarp(gmask);
                const double2* dg2 = reinterpret_cast<const double2*>(S.X[q]);
                const double2* g2 = reinterpret_cast<const double2*>(S.G[q]);
                const double2* sd2 = reinterpret_cast<const double2*>(S.D[q]);
                const double2* t2 = reinterpret_cast<const double2*>(S.T[sub]);
                const double2* p2 = reinterpret_cast<const double2*>(S.P[sub]);
                double t = 0.0;
#pragma unroll
                for (int j = 0; j < N; j += 2) {                                      // :875
                    const double2 v = dg2[j >> 1];
                    t += cur[j] * v.x;
                    t += cur[j + 1] * v.y;
                }
                S.T[sub][r] = t;
                S.P[sub][r] = dgv * t;
                __syncwarp(gmask);
                double dot = 0.0;
#pragma unroll
                for (int j = 0; j < N; j += 2) {                                      // Kernels.dot order
                    const double2 v = p2[j >> 1];
                    dot += v.x;
                    dot += v.y;
                }
                const double delta_norm = ao_q + dot;                                 // :876
                double dnew = 0.0;
#pragma unroll
                for (int j = 0; j < N; j += 2) {
                    const double2 sj = sd2[j >> 1], tj = t2[j >> 1], gj = g2[j >> 1];
                    cur[j] += (delta_norm * (sd * sj.x) - (t * sj.x + sd * tj.x));    // :882-884
                    cur[j + 1] += (delta_norm * (sd * sj.y) - (t * sj.y + sd * tj.y));
                    dnew += cur[j] * gj.x;                                            // :958-960
                    dnew += cur[j + 1] * gj.y;
                }
#pragma unroll
                for (int j = 0; j < N; ++j) __stcs(Hp + j * N, cur[j]);
                A.d[e] = dnew;
                __syncwarp(gmask);
            } else {
                if (!lazy) {
#pragma unroll
                    for (int j = 0; j < N; ++j) __stcs(Hp + j * N, (j == r) ? 1.0 : 0.0);  // :981 identity_matrix!
                }
                A.d[e] = gn;                                                          // :984-986
            }
        };
        if constexpr (C::PINGPONG) {
            // two rounds per trip, ping-pong between two register tiles: the loads of round i+1 are in flight while
            // round i computes, and no tile is ever copied
            double rowsA[N], rowsB[N];
            int metaA, metaB = 0;
            load_rows(0, rowsA, metaA);
#pragma unroll 1
            for (int round = 0; round < C::ROUNDS; round += 2) {
                load_rows(round + 1, rowsB, metaB);
                prefetch_round(round + A.prefetch_rounds);
                process(round, rowsA, metaA);
                if (round + 2 < C::ROUNDS) load_rows(round + 2, rowsA, metaA);
                prefetch_round(round + 1 + A.prefetch_rounds);
                process(round + 1, rowsB, metaB);
            }
        } else {
            // n > 16: one register tile of n doubles (two would not fit); the L2 prefetch alone runs ahead
            double rows[N];
            int meta;
#pragma unroll 1
            for (int round = 0; round < C::ROUNDS; ++round) {
                load_rows(round, rows, meta);
                prefetch_round(round + A.prefetch_rounds);
                process(round, rows, meta);
            }
        }
        __syncwarp();
    }

    if (valid && moved_any && A.f_host) A.f_host[p] = A.f[p];     // 32 lanes = 256 contiguous bytes of posted PCIe writes
    if (A.stats && lane < HK_COUNT && cnt_slot != 0.0) atomicAdd(A.stats + lane, (unsigned long long)cnt_slot);
}

template <int N>
inline size_t hybrid_smem() { return sizeof(HybridSmem<N>) * kHybridWarps; }
inline int hybrid_warps_per_sm(int n) { return n <= 16 ? 16 : 8; }      // CTAS_PER_SM * kHybridWarps

// host side of the launch, instantiated in two translation units (batched_hybrid_tu_{a,b}.cu) so that ptxas works on the
// sixteen kernels in parallel
template <int N>
inline cudaError_t hybrid_launch(const BatchedArgs& args, cudaStream_t stream, int device) {
    static bool attr_set[64] = {};
    static const size_t pad = getenv("DZO_HYBRID_SMEM_PAD") ? (size_t)atoi(getenv("DZO_HYBRID_SMEM_PAD")) : 0;   // occupancy experiments
    const size_t smem = hybrid_smem<N>() + pad;
    if (!attr_set[device & 63]) {
        for (auto* k : {bfgs_batched_hybrid_kernel<N, false, false>, bfgs_batched_hybrid_kernel<N, true, false>,
                        bfgs_batched_hybrid_kernel<N, false, true>, bfgs_batched_hybrid_kernel<N, true, true>}) {
            const cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        attr_set[device & 63] = true;
    }
    const bool vtile = (args.tile > 0 && args.tile < 32);
    const int tile = vtile ? args.tile : 32;
    const unsigned grid = (unsigned)((args.batch + (long long)tile * kHybridWarps - 1) / ((long long)tile * kHybridWarps));
    if (args.derived) {
        if (vtile) bfgs_batched_hybrid_kernel<N, true, true><<<grid, kHybridThreads, smem, stream>>>(args);
        else bfgs_batched_hybrid_kernel<N, false, true><<<grid, kHybridThreads, smem, stream>>>(args);
    } else {
        if (vtile) bfgs_batched_hybrid_kernel<N, true, false><<<grid, kHybridThreads, smem, stream>>>(args);
        else bfgs_batched_hybrid_kernel<N, false, false><<<grid, kHybridThreads, smem, stream>>>(args);
    }
    return cudaGetLastError();
}
cudaError_t hybrid_launch_n2_16(int n, const BatchedArgs& args, cudaStream_t stream, int device);    // batched_hybrid_tu_a.cu
cudaError_t hybrid_launch_n18_32(int n, const BatchedArgs& args, cudaStream_t stream, int device);   // batched_hybrid_tu_b.cu

}  // namespace dzo
