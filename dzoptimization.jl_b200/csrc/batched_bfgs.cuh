// batched_bfgs.cuh -- batched small-n BFGS: the constructor and resume kernels, the lanes-per-problem building blocks
// (Group, RosenbrockSmall, group_line_search) the kernel-level entry points of small_ops.cuh are made of, and the
// argument block of the step kernel (batched_hybrid.cuh).
//
// Everything here implements, per problem, SURVEY.md 8.0 / legacy/DZOptimization.jl:762-810 (ctor), :819-862 (resume)
// with SEQUENTIAL summation order (legacy/Kernels.jl:12-20): bitwise equal to the sequential oracle.
// Mapping: LPP lanes per problem (n <= LPP, LPP in {2,..,32}); lane r owns element r of every vector; a CTA of 256
// threads holds 256/LPP problems; cross-lane traffic is warp shuffles or group-private shared-memory broadcast buffers.
// (The first-generation step! kernel that lived here -- LPP lanes per problem for the whole step, H staged through
// shared memory by cp.async.bulk -- was retired in round 2: 1.63 ms per 1M-problem launch against 0.74 ms.)
#pragma once
#include "common.cuh"

namespace dzo {

struct BatchedArgs {
    double *x, *g, *d, *dx, *dg, *H, *f, *L;
    long long* iter;
    int* type;
    unsigned char* term;
    double* f_host;              // optional zero-copy mirrors in page-locked HOST memory (may be null): the step kernel
    unsigned char* term_host;    //   stores f / has_terminated there too, so the fields cross PCIe while it runs
    int n;
    long long batch;
    int ksteps;
    int prefetch_rounds;  // hybrid kernel: phase-2 rounds whose H tiles are pulled into L2 ahead of use
    int tile;             // hybrid kernel: problems per warp (0 or 32: a full warp; smaller for batches of a few waves)
    unsigned char* flags;        // Rosenbrock handles: per-problem state byte, BF_* bits below
    int lazy;                    // keep H = I implicit (BF_IDENT)
    int derived;                 // derived layout: a move stores x into the other point buffer (x / g, BF_PARITY) and no
                                 //   g, dx or dg; g = rosenbrock_gradient!(x), dx, dg are recomputed from the two points
    unsigned long long* stats;   // optional (may be null): HK_COUNT running step-kind counters
};
// flags[p]: BF_IDENT     H of problem p is the identity and its copy in HBM is stale (identity_matrix! :981 / :781-783
//                        not materialised)
//           BF_PARITY    derived layout: the current point is in g (set) or x (clear); the other buffer holds the previous one
//           BF_EXPLICIT  derived layout: delta_point / delta_gradient are the dx / dg arrays (constructor, set_state), not
//                        the differences of the two points
enum : unsigned { BF_IDENT = 1u, BF_PARITY = 2u, BF_EXPLICIT = 4u };

// rosenbrock_gradient! of one consecutive pair (legacy/ExampleFunctions.jl): the expression, hence the bits, of
// RosenbrockSmall::grad and of the step kernel, so the derived layout can recompute g wherever it needs it
DZO_DEVINL double2 rosen_pair_grad(double xe, double xo) {
    const double t1 = 1 - xe;
    const double t2 = xo - xe * xe;
    return make_double2(-2 * t1 - 400 * xe * t2, 200 * t2);
}

constexpr int kBatchedThreads = 256;
constexpr int kBcBufs = 5;  // 2 rotating reduction buffers + 3 vector broadcast buffers

template <int LPP>
struct Group {
    int r;          // element / row owned by this lane
    int n;
    unsigned mask;  // lanes of this problem
    bool act;       // r < n
    double* bc;     // kBcBufs * LPP doubles, private to the group
    int flip;       // rotating reduction buffer
    unsigned long long probes;

    DZO_DEVINL void sync() const { __syncwarp(mask); }
    DZO_DEVINL bool all(bool p) const { return __all_sync(mask, p || !act) != 0; }
    DZO_DEVINL bool any(bool p) const { return __any_sync(mask, p && act) != 0; }
    DZO_DEVINL double* vbuf(int k) const { return bc + (2 + k) * LPP; }

    // Kernels.dot / norm2 order: result = 0; result += v[i], i ascending (legacy/Kernels.jl:12-20)
    DZO_DEVINL double seq_sum(double v) {
        double* b = bc + flip * LPP;
        flip ^= 1;
        if (act) b[r] = v;
        sync();
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j < LPP; ++j)
            if (j < n) acc += b[j];
        return acc;
    }
};

// ----------------------------------------------------------------------------- objectives
// Extended Rosenbrock, legacy/ExampleFunctions.jl:10-24 per consecutive pair.
struct RosenbrockSmall {
    template <int LPP>
    static DZO_DEVINL double eval(Group<LPP>& G, double w) {
        const double y = __shfl_down_sync(G.mask, w, 1, LPP);
        const double t1 = 1 - w;
        const double t2 = y - w * w;
        const double term = t1 * t1 + 100 * (t2 * t2);
        double* b = G.bc + G.flip * LPP;
        G.flip ^= 1;
        if (G.act && !(G.r & 1)) b[G.r >> 1] = term;
        G.sync();
        G.probes++;
        double acc = 0.0;
        const int m = G.n >> 1;
#pragma unroll
        for (int k = 0; k < LPP / 2; ++k)
            if (k < m) acc += b[k];
        return acc;
    }
    template <int LPP>
    static DZO_DEVINL double grad(const Group<LPP>& G, double w) {
        const double up = __shfl_down_sync(G.mask, w, 1, LPP);  // element r+1
        const double dn = __shfl_up_sync(G.mask, w, 1, LPP);    // element r-1
        if (!(G.r & 1)) {
            const double t1 = 1 - w;
            const double t2 = up - w * w;
            return -2 * t1 - 400 * w * t2;
        }
        const double t2 = w - dn * dn;
        return 200 * t2;
    }
};

// ----------------------------------------------------------------------------- line search
// quadratic_line_search(functor, f0, t1): find_three_point_bracket (legacy/DZOptimization.jl
// :49-172, first trial step t1) + QuadraticLineSearch (:191-216), along w = x + (-t)*dir
// (sign from :945,:973).  Control flow is uniform across the lanes of a group.
template <int LPP, class Obj>
DZO_DEVINL void group_line_search(Group<LPP>& G, double x, double dir, double f0, double t1, double& t_best,
                                  double& f_best) {
    double x1 = 0.0, f1 = f0, x2 = 0.0, f2 = f0;
    do {
        if (!isfinite(f0)) break;                                  // :64-66
        if (!isfinite(t1) || t1 == 0.0) break;                     // [GLUE]
        if (G.all(dir == 0.0)) break;                              // :71-85
        double step = t1;
        double w = x + (-step) * dir;                              // :73-80
        bool changed = G.any(x != w);
        bool small = false;
        int cap = DZO_LINESEARCH_CAP;
        bool capped = false;
        while (!changed) {                                         // :91-101
            step += step;
            small = true;
            w = x + (-step) * dir;
            changed = G.any(x != w);
            if (--cap == 0) { capped = true; break; }
        }
        if (capped) break;
        if (small && G.all(x == w)) break;                         // :107-123 (constraint is the identity)
        double fa = Obj::eval(G, w);                               // :126
        if (fa <= f0) {                                            // :130
            double ref = w;                                        // :136
            cap = DZO_LINESEARCH_CAP;
            for (;;) {                                             // :143-156
                const double ds = step + step;
                w = x + (-ds) * dir;
                const double fb = Obj::eval(G, w);
                const bool same = G.all(w == ref);
                --cap;
                if (!isfinite(fb) || fb > fa || same || cap == 0) {
                    x1 = step; f1 = fa; x2 = ds; f2 = fb;
                    break;
                }
                step = ds; fa = fb; ref = w;
            }
        } else {                                                   // :157-171
            cap = DZO_LINESEARCH_CAP;
            for (;;) {
                const double hs = 0.5 * step;
                w = x + (-hs) * dir;
                const double fb = Obj::eval(G, w);
                --cap;
                if (fb <= f0 || cap == 0) {
                    x1 = hs; f1 = fb; x2 = step; f2 = fa;
                    break;
                }
                step = hs; fa = fb;
            }
        }
    } while (0);
    double xb = 0.0, fb = f0;                                      // :196-202
    if (f1 < fb) { xb = x1; fb = f1; }
    if (f2 < fb) { xb = x2; fb = f2; }
    const double delta_1 = f0 - f1;                                // :203-205
    const double delta_2 = f2 - f1;
    const double sum_deltas = delta_1 + delta_2;
    if (delta_1 >= 0.0 && delta_2 >= 0.0 && sum_deltas > 0.0) {    // :206-214
        const double twice_delta_1 = delta_1 + delta_1;
        const double delta_ratio = (twice_delta_1 + sum_deltas) / (sum_deltas + sum_deltas);
        const double xq = delta_ratio * x1;
        const double w = x + (-xq) * dir;
        const double fq = Obj::eval(G, w);
        if (fq < fb) { xb = xq; fb = fq; }
    }
    t_best = xb;
    f_best = fb;
}

// ----------------------------------------------------------------------------- constructor kernel
// BFGSOptimizer(f, g!, x0, L0)  legacy/DZOptimization.jl:762-810.  x already holds copy(x0).
template <int LPP, class Obj>
static __global__ void __launch_bounds__(kBatchedThreads) bfgs_batched_init_kernel(BatchedArgs A, double initial_step_length) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int PPC = kBatchedThreads / LPP;
    double* bc_all = reinterpret_cast<double*>(smem_raw);
    const int lane = threadIdx.x & 31;
    const int gi = threadIdx.x / LPP;
    Group<LPP> G;
    G.r = threadIdx.x % LPP;
    G.n = A.n;
    G.act = G.r < A.n;
    G.mask = (LPP == 32) ? 0xffffffffu : (((1u << LPP) - 1u) << (lane - (lane % LPP)));
    G.bc = bc_all + gi * (kBcBufs * LPP);
    G.flip = 0;
    G.probes = 0;
    const long long p = (long long)blockIdx.x * PPC + gi;
    if (p >= A.batch) return;
    const int n = A.n;
    const double x = G.act ? A.x[p * n + G.r] : 0.0;
    const double f0 = Obj::eval(G, x);                              // :772
    const double g = Obj::grad(G, x);                               // :775-776
    if (G.act) {
        if (!A.derived) A.g[p * n + G.r] = g;
        A.d[p * n + G.r] = g;                                       // :784 next_step_direction = copy(gradient)
        A.dx[p * n + G.r] = 0.0;                                    // :777
        A.dg[p * n + G.r] = 0.0;                                    // :778
        if (!A.lazy) {
            double* Hp = A.H + p * n * n;                           // :781-783 identity_matrix!
            for (int j = 0; j < n; ++j) Hp[G.r + j * n] = (j == G.r) ? 1.0 : 0.0;
        }
    }
    if (G.r == 0) {
        A.f[p] = f0;
        A.L[p] = initial_step_length;                               // :779
        A.iter[p] = 0;                                              // :767
        A.type[p] = DZO_STEP_NULL;                                  // :780
        A.term[p] = 0;                                              // :768
        A.flags[p] = (A.lazy ? BF_IDENT : 0u) | BF_EXPLICIT;        // H = I kept implicit (batched_hybrid.cuh); x in x
    }
}

// ----------------------------------------------------------------------------- resume kernel
// State-rebuilding constructor legacy/DZOptimization.jl:819-862: x, H, dx, dg, L, type, iter were
// copied in by the host; recompute f (:828), g (:830-831), d = H*g (:833-836), clear the flag (:849).
template <int LPP, class Obj>
static __global__ void __launch_bounds__(kBatchedThreads) bfgs_batched_restore_kernel(BatchedArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int PPC = kBatchedThreads / LPP;
    double* bc_all = reinterpret_cast<double*>(smem_raw);
    const int lane = threadIdx.x & 31;
    const int gi = threadIdx.x / LPP;
    Group<LPP> G;
    G.r = threadIdx.x % LPP;
    G.n = A.n;
    G.act = G.r < A.n;
    G.mask = (LPP == 32) ? 0xffffffffu : (((1u << LPP) - 1u) << (lane - (lane % LPP)));
    G.bc = bc_all + gi * (kBcBufs * LPP);
    G.flip = 0;
    G.probes = 0;
    const long long p = (long long)blockIdx.x * PPC + gi;
    if (p >= A.batch) return;
    const int n = A.n;
    const double x = G.act ? A.x[p * n + G.r] : 0.0;
    const double f0 = Obj::eval(G, x);
    const double g = Obj::grad(G, x);
    double* v0 = G.vbuf(0);
    if (G.act) v0[G.r] = g;
    G.sync();
    double d = 0.0;
    const double* Hp = A.H + p * n * n;
    if (G.act)
        for (int j = 0; j < n; ++j) d += Hp[G.r + j * n] * v0[j];   // mul!(d, H, g), row sum j ascending
    if (G.act) {
        if (!A.derived) A.g[p * n + G.r] = g;
        A.d[p * n + G.r] = d;
    }
    if (G.r == 0) {
        A.f[p] = f0;
        A.term[p] = 0;
        A.flags[p] = BF_EXPLICIT;                                   // the caller's H, x, dx and dg are in HBM
    }
}

// number of problems with has_terminated == false
static __global__ void count_active_kernel(const unsigned char* term, long long batch, unsigned long long* out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int v = (i < batch) ? (term[i] == 0) : 0;
    v = __reduce_add_sync(0xffffffffu, v);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(out, (unsigned long long)v);
}

template <int LPP>
inline size_t batched_init_smem() {
    constexpr int PPC = kBatchedThreads / LPP;
    return sizeof(double) * ((size_t)PPC * kBcBufs * LPP);
}

}  // namespace dzo
