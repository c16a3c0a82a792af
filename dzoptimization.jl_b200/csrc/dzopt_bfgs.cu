// dzopt_bfgs.cu -- C ABI (include/dzopt.h) of the BFGSOptimizer path: handles, step!, field
// reads, resume, kernel-level entry points, measurement hooks.  sm_100a only; -fmad=false.
#include <dlfcn.h>

#include <new>

#include "batched_bfgs.cuh"
#include "batched_hybrid.cuh"
#include "cluster_search.cuh"
#include "gd_batched.cuh"
#include "host_common.h"
#include "large_bfgs.cuh"
#include "small_ops.cuh"
#include "small_sweeps.cuh"
#include "warp_search.cuh"

namespace dzo {
thread_local char g_err[512] = "";
Tuning g_tuning;

int check_problem(int objective, int constraint, int64_t obj_param, int64_t n, int64_t batch) {
    if (n <= 0 || batch <= 0) return fail(DZO_ERR_INVALID_ARGUMENT, "n and batch must be positive");
    if (objective == DZO_OBJ_ROSENBROCK) {
        if (n % 2) return fail(DZO_ERR_INVALID_ARGUMENT, "extended Rosenbrock needs even n");
        if (constraint != DZO_CONSTRAINT_NONE) return fail(DZO_ERR_INVALID_ARGUMENT, "Rosenbrock takes DZO_CONSTRAINT_NONE");
    } else if (objective == DZO_OBJ_RIESZ) {
        if (obj_param <= 0 || obj_param > 16 || n % obj_param)
            return fail(DZO_ERR_INVALID_ARGUMENT, "Riesz needs n = dim * N, 1 <= dim <= 16");
        if (constraint != DZO_CONSTRAINT_NONE && constraint != DZO_CONSTRAINT_SPHERE)
            return fail(DZO_ERR_INVALID_ARGUMENT, "unknown constraint id");
    } else
        return fail(DZO_ERR_INVALID_ARGUMENT, "unknown objective id");
    return DZO_OK;
}

// ----------------------------------------------------------------------------- NCCL (dlopen'ed: only the
// row-sharded mode needs it, and the process may already hold torch's copy of libnccl.so.2)
struct NcclId128 { char b[128]; };  // ncclUniqueId (passed by value)
struct NcclApi {
    void* so = nullptr;
    int (*GetUniqueId)(void*) = nullptr;
    int (*CommInitRank)(void**, int, NcclId128, int) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;
static int load_nccl() {
    if (g_nccl.so) return DZO_OK;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    void* so = nullptr;
    for (const char* nm : names) {
        so = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (so) break;
    }
    if (!so) return fail(DZO_ERR_NCCL, "cannot dlopen libnccl.so.2: %s", dlerror());
    g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))dlsym(so, "ncclGetUniqueId");
    g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))dlsym(so, "ncclCommInitRank");
    g_nccl.AllGather = (decltype(g_nccl.AllGather))dlsym(so, "ncclAllGather");
    g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))dlsym(so, "ncclCommDestroy");
    g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))dlsym(so, "ncclGetErrorString");
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllGather || !g_nccl.CommDestroy)
        return fail(DZO_ERR_NCCL, "libnccl lacks a required symbol");
    g_nccl.so = so;
    return DZO_OK;
}
#define DZO_NCCL(call)                                                                               \
    do {                                                                                             \
        int r__ = (call);                                                                            \
        if (r__ != 0)                                                                                \
            return ::dzo::fail(DZO_ERR_NCCL, "%s:%d %s -> %s", __FILE__, __LINE__, #call,            \
                               g_nccl.GetErrorString ? g_nccl.GetErrorString(r__) : "nccl error");   \
    } while (0)
constexpr int kNcclFloat64 = 8;  // ncclDouble

}  // namespace dzo

namespace dzo {   // BFGS x Riesz hook, dzopt_gd.cu
int riesz_bfgs_attach(int64_t n, int64_t dim, int constraint, int device, void** out);
void riesz_bfgs_detach(void* p);
int riesz_bfgs_launch(void* p, int mode, cudaStream_t stream, double* x, double* g, double* d, double* dx, double* dg,
                      double* sd, LargeCtrl* ctrl, double initial_step_length);
}

using namespace dzo;

// ============================================================================= handle
struct dzo_bfgs {
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    int objective = 0, constraint = 0;
    int64_t dim = 0, n = 0, batch = 0;
    bool small = false;  // batched warp-resident path (n <= DZO_SMALL_N_MAX), SEQUENTIAL order
    int lpp = 0;
    int tile = 32;                          // batched hybrid kernel: problems per warp (see create_common)
    // optimizer fields (device)
    double *x = nullptr, *g = nullptr, *d = nullptr, *dx = nullptr, *dg = nullptr, *H = nullptr;
    double *f = nullptr, *L = nullptr;
    long long* iter = nullptr;
    int* type = nullptr;
    unsigned char* term = nullptr;
    double* f_host = nullptr;            // dzo_bfgs_mirror_fields: page-locked host mirrors written by the step kernels
    unsigned char* term_host = nullptr;
    unsigned long long* counter = nullptr;
    unsigned char* flags = nullptr;      // batched hybrid kernel: per-problem state byte (BF_* in batched_bfgs.cuh)
    bool lazy = false;                   // batched hybrid kernel: H = I kept implicit (BF_IDENT)
    bool derived = false;                // batched hybrid kernel: x double-buffered in x / g; g, dx, dg recomputed (BF_PARITY)
    unsigned long long* stats = nullptr; // batched hybrid kernel: running step-kind counters (HK_COUNT words)
    // large path
    double *sd = nullptr, *t = nullptr, *partial = nullptr;
    unsigned* tile_counters = nullptr;
    LargeCtrl* ctrl = nullptr;
    // row sharding
    int rank = 0, nranks = 1;
    int64_t row0 = 0, rows = 0;
    void* comm = nullptr;
    // fused gathers over peer memory (CUDA IPC): every rank's t, d and flag words mapped here
    bool pooled = true;                 // device memory from the stream-ordered pool (false: cudaMalloc, IPC-able)
    bool fused = false;
    bool constructed = false;           // create_common finished: destroy takes part in the ranks' rendezvous
    unsigned long long *flags_t = nullptr, *flags_d = nullptr;   // local, kMaxPeers words each
    unsigned* done = nullptr;
    cudaGraphExec_t step_graph = nullptr;   // one large-n step! (4 launches) captured once, replayed per step
    cudaStream_t graph_stream = nullptr;
    int graph_tuning_epoch = -1;
    void* riesz = nullptr;              // Riesz objective: the cooperative search-stage kernel's workspace
    char* arena = nullptr;              // sharded: ONE cudaMalloc block [t | d | flags_t | flags_d] exported through IPC
    char* peer_arena[kMaxPeers] = {};   // mapped base pointers of the peers' blocks
    double *peer_t[kMaxPeers] = {}, *peer_d[kMaxPeers] = {};
    unsigned long long *peer_flags_t[kMaxPeers] = {}, *peer_flags_d[kMaxPeers] = {};
};

// Device memory of a handle comes from the device's stream-ordered pool (cudaMallocAsync) with an
// unbounded release threshold: constructing optimizer after optimizer in one process reuses the
// pages instead of paying cudaMalloc / cudaFree of gigabytes each time.
// Destroying a row-sharded handle is COLLECTIVE (include/dzopt.h): every rank drains its stream (behind
// peer_arrival_kernel that means all stores INTO this rank's arena have landed and all of this rank's stores into
// its peers' arenas are complete), closes the peers' mappings, and only after a rendezvous of all ranks -- nobody
// holds a mapping of anybody's arena any more -- frees the exported arena (the CUDA IPC contract).
static void free_handle(dzo_bfgs* o) {
    if (!o) return;
    cudaSetDevice(o->device);
    if (o->own_stream) cudaStreamSynchronize(o->stream);
    if (o->nranks > 1) {
        for (int p = 0; p < kMaxPeers; ++p)
            if (p != o->rank && o->peer_arena[p]) { cudaIpcCloseMemHandle(o->peer_arena[p]); o->peer_arena[p] = nullptr; }
        if (o->constructed && o->comm && o->partial && g_nccl.AllGather && o->own_stream) {
            // rendezvous: one byte per rank through the scratch that is no longer in use
            char* scratch = reinterpret_cast<char*>(o->partial);
            if (g_nccl.AllGather(scratch + o->rank, scratch, 1, /*ncclInt8*/ 0, o->comm, o->own_stream) == 0)
                cudaStreamSynchronize(o->own_stream);
        }
    }
    if (o->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(o->comm);
    if (o->riesz) riesz_bfgs_detach(o->riesz);
    if (o->step_graph) cudaGraphExecDestroy(o->step_graph);
    if (o->arena) { o->t = nullptr; o->d = nullptr; o->flags_t = nullptr; o->flags_d = nullptr; }   // live inside the arena
    void* ptrs[] = {o->x, o->g, o->d, o->dx, o->dg, o->H, o->f, o->L, o->iter, o->type, o->term, o->counter,
                    o->sd, o->t, o->partial, o->tile_counters, o->ctrl, o->flags_t, o->flags_d, o->done, o->arena,
                    o->flags, o->stats};
    if (o->own_stream) {
        for (void* p : ptrs) {
            if (!p) continue;
            if (o->pooled) cudaFreeAsync(p, o->own_stream); else cudaFree(p);
        }
        cudaStreamSynchronize(o->own_stream);
        cudaStreamDestroy(o->own_stream);
    }
    cudaGetLastError();
    delete o;
}

static void init_pool(int device) {
    static bool done[64] = {};
    if (done[device & 63]) return;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        unsigned long long keep = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    cudaGetLastError();
    done[device & 63] = true;
}

template <class T>
static int dmalloc_on(cudaStream_t stream, T** p, size_t count, bool pooled = true) {
    cudaError_t e = pooled ? cudaMallocAsync((void**)p, (count ? count : 1) * sizeof(T), stream)
                           : cudaMalloc((void**)p, (count ? count : 1) * sizeof(T));
    if (e != cudaSuccess) {
        *p = nullptr;
        cudaGetLastError();
        return fail(DZO_ERR_ALLOC, "cudaMallocAsync of %zu bytes failed: %s", count * sizeof(T), cudaGetErrorString(e));
    }
    return DZO_OK;
}
#define dmalloc(p, count) dmalloc_on(o->own_stream, p, count, o->pooled)

// problem-major matrices [p][e] -> batch-innermost [e][p] (set_state of the generic batched kernel)
static __global__ void h_to_batch_inner_kernel(const double* in, double* out, long long nn, long long batch) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;      // t = e * batch + p: coalesced stores
    if (t >= nn * batch) return;
    const long long e = t / batch, p = t - e * batch;
    out[t] = in[p * nn + e];
}

// any(isnan(f)) on the device: 4 bytes come back instead of the whole objective vector
static __global__ void any_nan_kernel(const double* f, long long count, int* flag) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool bad = (i < count) && (f[i] != f[i]);
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(flag, 1);
}
static int any_nan(dzo_bfgs* o, const double* f, long long count, bool* out) {
    int* flag = reinterpret_cast<int*>(o->counter);
    DZO_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), o->stream));
    any_nan_kernel<<<(unsigned)((count + 255) / 256), 256, 0, o->stream>>>(f, count, flag);
    DZO_CUDA(cudaGetLastError());
    int h = 0;
    DZO_CUDA(cudaMemcpyAsync(&h, flag, sizeof(int), cudaMemcpyDeviceToHost, o->stream));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    *out = (h != 0);
    return DZO_OK;
}

static BatchedArgs batched_args(const dzo_bfgs* o, int ksteps) {
    BatchedArgs A;
    A.x = o->x; A.g = o->g; A.d = o->d; A.dx = o->dx; A.dg = o->dg; A.H = o->H; A.f = o->f; A.L = o->L;
    A.iter = o->iter; A.type = o->type; A.term = o->term;
    A.f_host = o->f_host; A.term_host = o->term_host;
    A.n = (int)o->n; A.batch = o->batch; A.ksteps = ksteps; A.prefetch_rounds = g_tuning.batched_prefetch;
    A.flags = o->flags; A.lazy = o->lazy; A.derived = o->derived; A.stats = o->stats;
    A.tile = o->tile;
    return A;
}

static int pick_lpp(int64_t n) {
    int l = 2;
    while (l < n) l <<= 1;
    return l;
}

// ---- batched launches, dispatched on lanes-per-problem
template <int LPP>
static int launch_batched_init(dzo_bfgs* o, double L0) {
    constexpr int PPC = kBatchedThreads / LPP;
    const unsigned grid = (unsigned)((o->batch + PPC - 1) / PPC);
    bfgs_batched_init_kernel<LPP, RosenbrockSmall><<<grid, kBatchedThreads, batched_init_smem<LPP>(), o->stream>>>(batched_args(o, 0), L0);
    DZO_CUDA(cudaGetLastError());
    return DZO_OK;
}
template <int LPP>
static int launch_batched_restore(dzo_bfgs* o) {
    constexpr int PPC = kBatchedThreads / LPP;
    const unsigned grid = (unsigned)((o->batch + PPC - 1) / PPC);
    bfgs_batched_restore_kernel<LPP, RosenbrockSmall><<<grid, kBatchedThreads, batched_init_smem<LPP>(), o->stream>>>(batched_args(o, 0));
    DZO_CUDA(cudaGetLastError());
    return DZO_OK;
}
#define DZO_LPP_DISPATCH(o, fn, ...)                                   \
    switch ((o)->lpp) {                                                \
        case 2: return fn<2>(__VA_ARGS__);                             \
        case 4: return fn<4>(__VA_ARGS__);                             \
        case 8: return fn<8>(__VA_ARGS__);                             \
        case 16: return fn<16>(__VA_ARGS__);                           \
        default: return fn<32>(__VA_ARGS__);                           \
    }
// objectives the warp-resident kernels do not cover (Riesz): generic one-thread-per-problem kernel
static int generic_launch(dzo_bfgs* o, int mode, int k, double L0) {
    BfgsGenericArgs a;
    a.x = o->x; a.g = o->g; a.d = o->d; a.dx = o->dx; a.dg = o->dg; a.H = o->H; a.f = o->f; a.L = o->L;
    a.iter = o->iter; a.type = o->type; a.term = o->term; a.n = (int)o->n; a.dim = (int)o->dim;
    a.objective = o->objective; a.sphere = (o->constraint == DZO_CONSTRAINT_SPHERE); a.ksteps = k; a.batch = o->batch;
    a.initial_step_length = L0; a.mode = mode;
    a.hs = o->batch;                          // batch-innermost inverse Hessians (gd_batched.cuh)
    bfgs_generic_kernel<<<(unsigned)((o->batch + 63) / 64), 64, 0, o->stream>>>(a);
    DZO_CUDA(cudaGetLastError());
    return DZO_OK;
}
static int batched_init(dzo_bfgs* o, double L0) {
    if (o->objective != DZO_OBJ_ROSENBROCK) return generic_launch(o, 1, 0, L0);
    DZO_LPP_DISPATCH(o, launch_batched_init, o, L0)
}
static int batched_restore(dzo_bfgs* o) {
    if (o->objective != DZO_OBJ_ROSENBROCK) return generic_launch(o, 2, 0, 0.0);
    DZO_LPP_DISPATCH(o, launch_batched_restore, o)
}
static bool hybrid_n(int64_t n) { return n >= 2 && n <= 32 && n % 2 == 0; }
// step! of a batched handle: ONE launch of bfgs_batched_hybrid_kernel<n> (Rosenbrock; every even n <= 32), or the generic
// one-thread-per-problem kernel (Riesz)
static int batched_step(dzo_bfgs* o, int k) {
    if (o->objective != DZO_OBJ_ROSENBROCK) return generic_launch(o, 0, k, 0.0);
    const BatchedArgs args = batched_args(o, k);
    const cudaError_t e = (o->n <= 16) ? hybrid_launch_n2_16((int)o->n, args, o->stream, o->device)
                                       : hybrid_launch_n18_32((int)o->n, args, o->stream, o->device);
    if (e != cudaSuccess) return fail(DZO_ERR_CUDA, "batched step! launch failed: %s", cudaGetErrorString(e));
    return DZO_OK;
}

// ---- large-path launches
static LargeVecs large_vecs(const dzo_bfgs* o) {
    LargeVecs v;
    v.x = o->x; v.g = o->g; v.d = o->d; v.dx = o->dx; v.dg = o->dg; v.sd = o->sd; v.t = o->t;
    v.ctrl = o->ctrl; v.n = o->n;
    v.flags_t = o->flags_t; v.flags_d = o->flags_d; v.nranks = o->fused ? o->nranks : 1;
    return v;
}
static PeerSet peer_set(const dzo_bfgs* o, bool for_t) {
    PeerSet ps;
    memset(&ps, 0, sizeof ps);
    ps.nranks = o->fused ? o->nranks : 1;
    ps.rank = o->rank;
    ps.done = o->done;
    for (int p = 0; p < kMaxPeers; ++p) {
        ps.out[p] = for_t ? o->peer_t[p] : o->peer_d[p];
        ps.flags[p] = for_t ? o->peer_flags_t[p] : o->peer_flags_d[p];
    }
    return ps;
}
static SweepArgs sweep_args(const dzo_bfgs* o) {
    SweepArgs a;
    a.H = o->H; a.ld = o->rows; a.rows = o->rows; a.n = o->n; a.row0 = o->row0;
    a.v = nullptr; a.s = o->sd; a.t = o->t; a.partial = o->partial; a.out = nullptr;
    a.counters = o->tile_counters; a.ctrl = o->ctrl; a.need_kind = DZO_STEP_BFGS;
    a.nchunks = (int)((o->n + DZO_GEMV_CHUNK - 1) / DZO_GEMV_CHUNK);
    memset(&a.peers, 0, sizeof a.peers);
    a.peers.nranks = 1;
    return a;
}
// threads per sweep CTA (each thread owns 2 rows): the largest size that still gives >= 4 tiles per SM -- counting the
// problems of a batch (blockIdx.z), whose tiles fill the GPU by themselves -- but never a CTA more than twice as tall as
// the slab (batches of n = 256 problems: 128 threads 0.495 ms per step! call, 64 threads 0.558; n = 64: 64 threads)
static int sweep_threads(int64_t rows, int64_t n, int64_t batch = 1) {
    if (g_tuning.sweep_threads > 0) return g_tuning.sweep_threads;
    const int64_t nchunks = (n + DZO_GEMV_CHUNK - 1) / DZO_GEMV_CHUNK;
    int t = kSweepThreads;
    while (t > 64 && ((rows + 2 * t - 1) / (2 * t)) * nchunks * batch < 4 * 148) t >>= 1;   // (8 GPUs, n=16384: 64 and 128 measured equal)
    while (t > 64 && t > rows) t >>= 1;
    return t;
}
static dim3 sweep_grid(int64_t rows, int64_t n, int64_t batch = 1) {
    const int64_t r = 2 * sweep_threads(rows, n, batch);
    return dim3((unsigned)((rows + r - 1) / r), (unsigned)((n + DZO_GEMV_CHUNK - 1) / DZO_GEMV_CHUNK), (unsigned)batch);
}
static void launch_gemv(dim3 grid, int threads, cudaStream_t st, const SweepArgs& a) {
    switch (g_tuning.sweep_unroll) {
        case 4: gemv_kernel<4><<<grid, threads, 0, st>>>(a); break;
        case 16: gemv_kernel<16><<<grid, threads, 0, st>>>(a); break;
        case 24: gemv_kernel<24><<<grid, threads, 0, st>>>(a); break;
        case 32: gemv_kernel<32><<<grid, threads, 0, st>>>(a); break;
        default: gemv_kernel<8><<<grid, threads, 0, st>>>(a); break;
    }
}
static void launch_update(dim3 grid, int threads, cudaStream_t st, const SweepArgs& a) {
    switch (g_tuning.sweep_unroll) {
        case 4: update_gemv_kernel<4><<<grid, threads, 0, st>>>(a); break;
        case 16: update_gemv_kernel<16><<<grid, threads, 0, st>>>(a); break;
        case 24: update_gemv_kernel<24><<<grid, threads, 0, st>>>(a); break;
        case 32: update_gemv_kernel<32><<<grid, threads, 0, st>>>(a); break;
        default: update_gemv_kernel<8><<<grid, threads, 0, st>>>(a); break;
    }
}

static int allgather_rows(dzo_bfgs* o, double* vec) {
    if (o->nranks == 1) return DZO_OK;
    DZO_NCCL(g_nccl.AllGather(vec + o->row0, vec, (size_t)o->rows, kNcclFloat64, o->comm, o->stream));
    return DZO_OK;
}

// out = H * v on the local slab (+ allgather when sharded); predicate on ctrl->kind if need_kind >= 0
static int large_gemv(dzo_bfgs* o, const double* v, double* out, int need_kind, bool fused_t = false) {
    SweepArgs a = sweep_args(o);
    a.v = v; a.out = out;
    if (need_kind < 0) a.ctrl = nullptr; else a.need_kind = need_kind;
    if (fused_t) a.peers = peer_set(o, true);      // rows go straight into every peer's t; no collective call
    launch_gemv(sweep_grid(o->rows, o->n, o->batch), sweep_threads(o->rows, o->n, o->batch), o->stream, a);
    DZO_CUDA(cudaGetLastError());
    return fused_t ? DZO_OK : allgather_rows(o, out);
}

// medium n (32 < n <= 512), one GPU, Rosenbrock: the O(n) stage of every problem on one warp (warp_search.cuh)
static int warp_vw(const dzo_bfgs* o) {
    if (o->riesz || o->nranks != 1 || o->n > kWarpSearchMaxN || !g_tuning.warp_search) return 0;
    int vw = 1;
    while (64 * vw < o->n) vw <<= 1;
    return vw;
}
static void launch_warp_search(const dzo_bfgs* o, int vw, const LargeVecs& v, bool delta) {
    const unsigned grid = (unsigned)((o->batch + kWarpSearchWarps - 1) / kWarpSearchWarps);
    const int threads = 32 * kWarpSearchWarps;
#define DZO_WS(VW)                                                                                  \
    if (delta) warp_delta_kernel<VW><<<grid, threads, 0, o->stream>>>(v, o->batch);                  \
    else warp_bfgs_search_kernel<VW><<<grid, threads, 0, o->stream>>>(v, o->batch)
    switch (vw) {
        case 1: DZO_WS(1); break;
        case 2: DZO_WS(2); break;
        case 4: DZO_WS(4); break;
        default: DZO_WS(8); break;
    }
#undef DZO_WS
}

static int large_step_once(dzo_bfgs* o) {
    const LargeVecs v = large_vecs(o);
    const int vw = warp_vw(o);
    if (vw && o->batch > 1 && o->n <= kSmallSweepMaxN && g_tuning.small_sweeps) {
        // a batch of small matrices: the n^2 sweeps on one warp per problem too (small_sweeps.cuh)
        const unsigned grid = (unsigned)((o->batch + kSmallSweepWarps - 1) / kSmallSweepWarps);
        const int threads = 32 * kSmallSweepWarps;
        SmallSweepArgs sa;
        sa.H = o->H; sa.s = o->sd; sa.t = o->t; sa.ctrl = o->ctrl; sa.n = o->n; sa.batch = o->batch;
        launch_warp_search(o, vw, v, false);                                            // :891-950, :873-874
        DZO_CUDA(cudaGetLastError());
        sa.v = o->dg; sa.out = o->t;                                                    // :875
        warp_gemv_kernel<2, 16><<<grid, threads, 0, o->stream>>>(sa);
        DZO_CUDA(cudaGetLastError());
        launch_warp_search(o, vw, v, true);                                             // :876
        DZO_CUDA(cudaGetLastError());
        sa.v = o->g; sa.out = o->d;                                                     // :878-886 + :958-960, :981
        warp_update_gemv_kernel<2, 16><<<grid, threads, 0, o->stream>>>(sa);
        DZO_CUDA(cudaGetLastError());
        return DZO_OK;
    }
    if (vw) {
        launch_warp_search(o, vw, v, false);                                            // :891-950, :873-874
        DZO_CUDA(cudaGetLastError());
        DZO_TRY(large_gemv(o, o->dg, o->t, DZO_STEP_BFGS, false));                      // :875
        launch_warp_search(o, vw, v, true);                                             // :876
        DZO_CUDA(cudaGetLastError());
        SweepArgs a = sweep_args(o);
        a.v = o->g; a.out = o->d;
        a.need_kind = DZO_STEP_GRADIENT_DESCENT + 100;   // this launch also serves identity_matrix! (:981) after a GD step
        launch_update(sweep_grid(o->rows, o->n, o->batch), sweep_threads(o->rows, o->n, o->batch), o->stream, a);   // :878-886 + :958-960
        DZO_CUDA(cudaGetLastError());
        return DZO_OK;
    }
    if (o->riesz) {
        DZO_TRY(riesz_bfgs_launch(o->riesz, 5, o->stream, o->x, o->g, o->d, o->dx, o->dg, o->sd, o->ctrl, 0.0));
    }
    // 8-CTA cluster with DSMEM reductions (a single problem: lowest latency) vs one 1024-thread CTA per problem (a batch:
    // only ~18 clusters are co-resident on a B200, but 148+ CTAs -- n = 1024 x 256 problems spent a quarter of the step!
    // call queueing for clusters); the peer-flag waits of the row-sharded mode live in the cluster kernels
    const bool cluster = o->fused || (g_tuning.search_variant == 0 && o->batch < 4) || g_tuning.search_variant == 2;
    if (o->riesz) { /* search stage already enqueued above (cooperative Riesz kernel) */ }
    else if (cluster) cluster_bfgs_search_kernel<<<kClusterCtas * (unsigned)o->batch, kClusterThreads, 0, o->stream>>>(v);   // :891-950, :873-874
    else vec_bfgs_search_kernel<<<(unsigned)o->batch, 1024, 0, o->stream>>>(v);
    DZO_CUDA(cudaGetLastError());
    DZO_TRY(large_gemv(o, o->dg, o->t, DZO_STEP_BFGS, o->fused));               // :875
    if (cluster) cluster_delta_kernel<<<kClusterCtas * (unsigned)o->batch, kClusterThreads, 0, o->stream>>>(v);         // :876
    else vec_delta_kernel<<<(unsigned)o->batch, 1024, 0, o->stream>>>(v);
    DZO_CUDA(cudaGetLastError());
    SweepArgs a = sweep_args(o);
    a.v = o->g; a.out = o->d;
    a.need_kind = DZO_STEP_GRADIENT_DESCENT + 100;   // this launch also serves identity_matrix! (:981) after a GD step
    if (o->fused) a.peers = peer_set(o, false);
    launch_update(sweep_grid(o->rows, o->n, o->batch), sweep_threads(o->rows, o->n, o->batch), o->stream, a);   // :878-886 + :958-960
    DZO_CUDA(cudaGetLastError());
    if (!o->fused) DZO_TRY(allgather_rows(o, o->d));
    else {
        peer_arrival_kernel<<<1, 32, 0, o->stream>>>(v);     // drained stream => every peer's rows of d have landed
        DZO_CUDA(cudaGetLastError());
    }
    return DZO_OK;
}

// Map every peer's t, d and flag words into this process (CUDA IPC; NVLink peer access).  The 4 x 64-byte
// handles of all ranks travel over the NCCL communicator that was just created -- the only collective the
// fused mode ever issues.  Falls back to NCCL all-gathers (o->fused = false) if any rank cannot map.
struct IpcBundle { cudaIpcMemHandle_t arena; unsigned long long offset; int ok; int pad; };
// cudaIpcGetMemHandle exports the whole underlying allocation: find its base so peers can add the offset
static bool allocation_base(const void* p, unsigned long long* offset) {
    typedef int (*GetRange)(unsigned long long*, size_t*, unsigned long long);
    static GetRange fn = nullptr;
    if (!fn) {
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &sym, cudaEnableDefault, &q) != cudaSuccess || !sym) {
            cudaGetLastError();
            return false;
        }
        fn = (GetRange)sym;
    }
    unsigned long long base = 0;
    size_t size = 0;
    if (fn(&base, &size, (unsigned long long)(uintptr_t)p) != 0) return false;
    *offset = (unsigned long long)(uintptr_t)p - base;
    return true;
}
// Every rank issues BOTH collectives whatever happens locally: a local CUDA error only turns this rank's vote into
// "cannot map", so the peers never block in a gather this rank skipped, and all ranks end in the same mode (fused, or the
// NCCL all-gather fallback) or fail together.  The scratch buffers are released on every path.
static int exchange_peer_memory(dzo_bfgs* o) {
    o->fused = false;
    IpcBundle mine;
    memset(&mine, 0, sizeof mine);
    mine.ok = (g_tuning.sharded_variant == 0) && o->arena && allocation_base(o->arena, &mine.offset) &&
              cudaIpcGetMemHandle(&mine.arena, o->arena) == cudaSuccess;
    cudaGetLastError();
    // one scratch allocation: [nranks bundles][nranks votes]
    const size_t bundles = sizeof(IpcBundle) * o->nranks;
    char* dev = nullptr;
    if (cudaMalloc((void**)&dev, bundles + sizeof(int) * o->nranks) != cudaSuccess) {
        cudaGetLastError();
        return fail(DZO_ERR_ALLOC, "row-sharded constructor: scratch allocation failed (no collective was issued on any stream yet)");
    }
    IpcBundle* dev_b = reinterpret_cast<IpcBundle*>(dev);
    int* dev_v = reinterpret_cast<int*>(dev + bundles);
    IpcBundle all[kMaxPeers];
    memset(all, 0, sizeof all);
    bool local_ok = cudaMemcpyAsync(dev_b + o->rank, &mine, sizeof mine, cudaMemcpyHostToDevice, o->stream) == cudaSuccess;
    const int r1 = g_nccl.AllGather(dev_b + o->rank, dev_b, sizeof(IpcBundle), /*ncclInt8*/ 0, o->comm, o->stream);
    local_ok = local_ok && r1 == 0 &&
               cudaMemcpyAsync(all, dev_b, bundles, cudaMemcpyDeviceToHost, o->stream) == cudaSuccess &&
               cudaStreamSynchronize(o->stream) == cudaSuccess;
    bool ok = local_ok;
    for (int p = 0; p < o->nranks; ++p) ok = ok && all[p].ok;
    const size_t nb = (size_t)o->n;
    for (int p = 0; p < o->nranks && ok; ++p) {
        char* base = nullptr;
        if (p == o->rank) {
            base = o->arena;
        } else {
            void* mapped = nullptr;
            ok = cudaIpcOpenMemHandle(&mapped, all[p].arena, cudaIpcMemLazyEnablePeerAccess) == cudaSuccess;
            if (!ok) break;
            o->peer_arena[p] = static_cast<char*>(mapped);
            base = o->peer_arena[p] + all[p].offset;
        }
        o->peer_t[p] = reinterpret_cast<double*>(base);
        o->peer_d[p] = o->peer_t[p] + nb;
        o->peer_flags_t[p] = reinterpret_cast<unsigned long long*>(o->peer_d[p] + nb);
        o->peer_flags_d[p] = o->peer_flags_t[p] + kMaxPeers;
    }
    cudaGetLastError();
    // every rank must agree on the mode: one more tiny gather of the outcome (issued even after a local failure)
    int okint = ok ? 1 : 0;
    int res[kMaxPeers];
    memset(res, 0, sizeof res);
    bool vote_ok = cudaMemcpyAsync(dev_v + o->rank, &okint, sizeof(int), cudaMemcpyHostToDevice, o->stream) == cudaSuccess;
    const int r2 = (r1 == 0) ? g_nccl.AllGather(dev_v + o->rank, dev_v, sizeof(int), /*ncclInt8*/ 0, o->comm, o->stream) : r1;
    vote_ok = vote_ok && r2 == 0 &&
              cudaMemcpyAsync(res, dev_v, sizeof(int) * o->nranks, cudaMemcpyDeviceToHost, o->stream) == cudaSuccess;
    const bool drained = cudaStreamSynchronize(o->stream) == cudaSuccess;
    cudaFree(dev);
    cudaGetLastError();
    if (r1 != 0 || r2 != 0) return fail(DZO_ERR_NCCL, "row-sharded constructor: ncclAllGather of the peer-memory handles failed");
    if (!vote_ok || !drained) return fail(DZO_ERR_CUDA, "row-sharded constructor: exchanging the peer-memory handles failed");
    bool all_ok = true;
    for (int p = 0; p < o->nranks; ++p) all_ok = all_ok && res[p];
    o->fused = all_ok;
    return DZO_OK;
}

// ============================================================================= create / destroy
static int create_common(dzo_bfgs** out, int objective, int constraint, int64_t obj_param, int64_t n, int64_t batch,
                         const double* x0, double L0, int device, int rank, int nranks, const void* nccl_id) {
    if (!out || !x0) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    *out = nullptr;
    DZO_TRY(check_problem(objective, constraint, obj_param, n, batch));
    if (objective == DZO_OBJ_RIESZ && (obj_param > 4 || nranks != 1))
        return fail(DZO_ERR_UNSUPPORTED, "BFGSOptimizer with the Riesz objective: dim <= 4, one GPU");
    if (batch > 1 && n > DZO_SMALL_N_MAX && (objective != DZO_OBJ_ROSENBROCK || nranks != 1))
        return fail(DZO_ERR_UNSUPPORTED, "a batch of n > %d problems: DZO_OBJ_ROSENBROCK on one GPU (one thread-block cluster per problem)", DZO_SMALL_N_MAX);
    if (batch > 1 && n > DZO_SMALL_N_MAX && (double)n * (double)n * (double)batch * 8.0 > 160e9)
        return fail(DZO_ERR_ALLOC, "batch of %lld inverse Hessians of n = %lld does not fit one GPU", (long long)batch, (long long)n);
    if (nranks < 1 || rank < 0 || rank >= nranks) return fail(DZO_ERR_INVALID_ARGUMENT, "bad rank/nranks");
    if (nranks > 1 && (n <= DZO_SMALL_N_MAX || n % (2 * nranks)))
        return fail(DZO_ERR_INVALID_ARGUMENT, "row sharding needs n > %d and n divisible by 2*nranks", DZO_SMALL_N_MAX);
    DZO_TRY(use_device(device));
    dzo_bfgs* o = new (std::nothrow) dzo_bfgs();
    if (!o) return fail(DZO_ERR_ALLOC, "out of memory");
    o->device = device; o->objective = objective; o->constraint = constraint; o->dim = obj_param;
    o->n = n; o->batch = batch; o->small = (n <= DZO_SMALL_N_MAX); o->lpp = pick_lpp(n);
    o->tile = 32;
    if (o->small && objective == DZO_OBJ_ROSENBROCK && hybrid_n(n) && g_tuning.batched_tile != 32) {
        // problems per warp of the batched kernel: a batch that fills the resident warps of the GPU at most three times over
        // is spread evenly over that many full waves (125 k problems: 2 waves of 27 instead of 1.65 waves of 32)
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
        const long long slots = (long long)sms * hybrid_warps_per_sm((int)n);
        const long long tiles32 = (batch + 31) / 32;
        const long long waves = (tiles32 + slots - 1) / slots;
        if (g_tuning.batched_tile > 0) o->tile = g_tuning.batched_tile < 32 ? g_tuning.batched_tile : 32;
        else if (waves <= 3) {
            const long long t = (batch + waves * slots - 1) / (waves * slots);
            o->tile = (int)(t < 1 ? 1 : (t > 32 ? 32 : t));
        }
    }
    o->rank = rank; o->nranks = nranks; o->rows = n / nranks; o->row0 = o->rows * rank;
    o->pooled = (nranks == 1);        // sharded handles use cudaMalloc: CUDA IPC cannot export pool memory
    if (nranks > kMaxPeers) { delete o; return fail(DZO_ERR_INVALID_ARGUMENT, "at most %d ranks", kMaxPeers); }
    int rc = DZO_OK;
    auto bail = [&](int code) { free_handle(o); return code; };
    if (cudaStreamCreateWithFlags(&o->own_stream, cudaStreamNonBlocking) != cudaSuccess)
        return bail(fail(DZO_ERR_CUDA, "cudaStreamCreate failed"));
    o->stream = o->own_stream;
    init_pool(device);
    const size_t nb = (size_t)n * (size_t)batch;
    const bool use_arena = (nranks > 1);
    if (use_arena) {
        const size_t bytes = 2 * nb * sizeof(double) + 2 * kMaxPeers * sizeof(unsigned long long);
        if ((rc = dmalloc(&o->arena, bytes))) return bail(rc);
        o->t = reinterpret_cast<double*>(o->arena);
        o->d = o->t + nb;
        o->flags_t = reinterpret_cast<unsigned long long*>(o->d + nb);
        o->flags_d = o->flags_t + kMaxPeers;
    }
    if ((rc = dmalloc(&o->x, nb)) || (rc = dmalloc(&o->g, nb)) || (!use_arena && (rc = dmalloc(&o->d, nb))) ||
        (rc = dmalloc(&o->dx, nb)) || (rc = dmalloc(&o->dg, nb)) || (rc = dmalloc(&o->counter, 1)))
        return bail(rc);
    if (o->small) {
        if ((rc = dmalloc(&o->H, nb * (size_t)n)) || (rc = dmalloc(&o->f, (size_t)batch)) || (rc = dmalloc(&o->L, (size_t)batch)) ||
            (rc = dmalloc(&o->iter, (size_t)batch)) || (rc = dmalloc(&o->type, (size_t)batch)) || (rc = dmalloc(&o->term, (size_t)batch)) ||
            (rc = dmalloc(&o->stats, (size_t)HK_COUNT)))
            return bail(rc);
        if (cudaMemsetAsync(o->stats, 0, HK_COUNT * sizeof(unsigned long long), o->stream) != cudaSuccess)
            return bail(fail(DZO_ERR_CUDA, "memset failed"));
        if (objective == DZO_OBJ_ROSENBROCK && hybrid_n(n)) {
            o->lazy = g_tuning.batched_lazy != 0;       // implicit identities: no H written by the constructor or after a GD step
            // derived layout where the kernel is bound by HBM bytes; n <= 8 is bound by FP64 issue, where the recomputed
            // gradients cost more than the bytes they save (1 M problems, n = 8: 0.320 vs 0.318 ms per launch)
            o->derived = (g_tuning.batched_derived < 0) ? (n > 8) : (g_tuning.batched_derived != 0);
            if ((rc = dmalloc(&o->flags, (size_t)batch))) return bail(rc);
        }
    } else {
        const size_t nchunks = (size_t)((n + DZO_GEMV_CHUNK - 1) / DZO_GEMV_CHUNK);
        const size_t rblocks = (size_t)((o->rows + kSweepMinRows - 1) / kSweepMinRows);
        const size_t B = (size_t)batch;     // > 1: a batch of medium-n problems, every array holds B consecutive copies
        if ((rc = dmalloc(&o->H, (size_t)o->rows * (size_t)n * B)) || (rc = dmalloc(&o->sd, (size_t)n * B)) ||
            (!use_arena && (rc = dmalloc(&o->t, (size_t)n * B))) ||
            (rc = dmalloc(&o->partial, nchunks * (size_t)o->rows * B)) || (rc = dmalloc(&o->tile_counters, rblocks * B)) ||
            (rc = dmalloc(&o->ctrl, B)) || (!use_arena && (rc = dmalloc(&o->flags_t, (size_t)kMaxPeers))) ||
            (!use_arena && (rc = dmalloc(&o->flags_d, (size_t)kMaxPeers))) || (rc = dmalloc(&o->done, 1)))
            return bail(rc);
        if (cudaMemsetAsync(o->tile_counters, 0, rblocks * B * sizeof(unsigned), o->stream) != cudaSuccess ||
            cudaMemsetAsync(o->flags_t, 0, kMaxPeers * 8, o->stream) != cudaSuccess ||
            cudaMemsetAsync(o->flags_d, 0, kMaxPeers * 8, o->stream) != cudaSuccess ||
            cudaMemsetAsync(o->done, 0, sizeof(unsigned), o->stream) != cudaSuccess)
            return bail(fail(DZO_ERR_CUDA, "memset failed"));
    }
    if (nranks > 1) {
        if ((rc = load_nccl())) return bail(rc);
        NcclId128 id;
        memcpy(id.b, nccl_id, 128);
        int r = g_nccl.CommInitRank(&o->comm, nranks, id, rank);
        if (r != 0) return bail(fail(DZO_ERR_NCCL, "ncclCommInitRank failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?"));
        if ((rc = exchange_peer_memory(o))) return bail(rc);
    }
    // copy(initial_point)  legacy/DZOptimization.jl:769
    if (cudaMemcpyAsync(o->x, x0, nb * sizeof(double), cudaMemcpyHostToDevice, o->stream) != cudaSuccess)
        return bail(fail(DZO_ERR_CUDA, "H2D copy of x0 failed: %s", cudaGetErrorString(cudaGetLastError())));
    if (o->small) {
        if ((rc = batched_init(o, L0))) return bail(rc);
    } else {
        if (objective == DZO_OBJ_RIESZ) {
            if ((rc = riesz_bfgs_attach(n, obj_param, constraint, device, &o->riesz))) return bail(rc);
            if ((rc = riesz_bfgs_launch(o->riesz, 6, o->stream, o->x, o->g, o->d, o->dx, o->dg, o->sd, o->ctrl, L0))) return bail(rc);
        } else
            vec_bfgs_init_kernel<<<(unsigned)batch, 1024, 0, o->stream>>>(large_vecs(o), L0);
        SweepArgs a = sweep_args(o);
        a.ctrl = nullptr;
        identity_kernel<<<sweep_grid(o->rows, o->n, o->batch), sweep_threads(o->rows, o->n, o->batch), 0, o->stream>>>(a);   // :781-783
    }
    if (cudaStreamSynchronize(o->stream) != cudaSuccess || cudaGetLastError() != cudaSuccess)
        return bail(fail(DZO_ERR_CUDA, "constructor kernels failed: %s", cudaGetErrorString(cudaGetLastError())));
    // @assert !isnan(initial_objective_value)   :773
    {
        bool bad = false;
        if (o->small) {
            if ((rc = any_nan(o, o->f, batch, &bad))) return bail(rc);
        } else {
            for (int64_t q = 0; q < batch && !bad; ++q) {
                LargeCtrl c;
                cudaMemcpy(&c, o->ctrl + q, sizeof c, cudaMemcpyDeviceToHost);
                bad = (c.f != c.f);
            }
        }
        if (bad) return bail(fail(DZO_ERR_NAN_OBJECTIVE, "objective is NaN at the initial point"));
    }
    o->constructed = true;
    *out = o;
    return DZO_OK;
}

extern "C" {

const char* dzo_last_error(void) { return g_err; }

int dzo_bfgs_create(dzo_bfgs** out, int objective, int constraint, int64_t obj_param, int64_t n, int64_t batch,
                    const double* x0, double initial_step_length, int device) {
    return create_common(out, objective, constraint, obj_param, n, batch, x0, initial_step_length, device, 0, 1, nullptr);
}

int dzo_nccl_get_unique_id(void* out128) {
    if (!out128) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    DZO_TRY(load_nccl());
    DZO_NCCL(g_nccl.GetUniqueId(out128));
    return DZO_OK;
}

int dzo_bfgs_create_sharded(dzo_bfgs** out, int objective, int constraint, int64_t obj_param, int64_t n,
                            const double* x0, double initial_step_length, int device, int rank, int nranks,
                            const void* nccl_unique_id) {
    if (nranks > 1 && !nccl_unique_id) return fail(DZO_ERR_INVALID_ARGUMENT, "nccl_unique_id is null");
    return create_common(out, objective, constraint, obj_param, n, 1, x0, initial_step_length, device, rank, nranks,
                         nccl_unique_id);
}

void dzo_bfgs_destroy(dzo_bfgs* o) { free_handle(o); }

int dzo_bfgs_set_stream(dzo_bfgs* o, void* cuda_stream) {
    if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");
    DZO_TRY(use_device(o->device));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    o->stream = cuda_stream ? (cudaStream_t)cuda_stream : o->own_stream;
    return DZO_OK;
}

// ============================================================================= step!
// One large-n step! is a fixed sequence of four launches whose behaviour is decided on the device, so it is
// captured into a CUDA graph once and replayed: the launches reach the GPU front end as one unit.
static int large_step_graph(dzo_bfgs* o) {
    const bool eligible = g_tuning.use_graph && !o->riesz && (o->nranks == 1 || o->fused);
    if (!eligible) return large_step_once(o);
    if (!o->step_graph || o->graph_stream != o->stream || o->graph_tuning_epoch != g_tuning.epoch) {
        if (o->step_graph) { cudaGraphExecDestroy(o->step_graph); o->step_graph = nullptr; }
        cudaGraph_t graph = nullptr;
        DZO_CUDA(cudaStreamBeginCapture(o->stream, cudaStreamCaptureModeThreadLocal));
        const int rc = large_step_once(o);
        const cudaError_t e = cudaStreamEndCapture(o->stream, &graph);
        if (rc != DZO_OK || e != cudaSuccess || !graph) {
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            g_tuning.use_graph = 0;                       // capture unavailable: plain launches from now on
            return large_step_once(o);
        }
        const cudaError_t ei = cudaGraphInstantiate(&o->step_graph, graph, 0);
        cudaGraphDestroy(graph);
        if (ei != cudaSuccess) {
            o->step_graph = nullptr;
            cudaGetLastError();
            g_tuning.use_graph = 0;
            return large_step_once(o);
        }
        o->graph_stream = o->stream;
        o->graph_tuning_epoch = g_tuning.epoch;
    }
    DZO_CUDA(cudaGraphLaunch(o->step_graph, o->stream));
    return DZO_OK;
}

int dzo_bfgs_step_async(dzo_bfgs* o, int k) {
    if (!o || k < 0) return fail(DZO_ERR_INVALID_ARGUMENT, "bad arguments");
    DZO_TRY(use_device(o->device));
    if (k == 0) return DZO_OK;
    if (o->small) return batched_step(o, k);
    for (int s = 0; s < k; ++s) DZO_TRY(large_step_graph(o));
    return DZO_OK;
}
int dzo_bfgs_sync(dzo_bfgs* o) {
    if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");
    DZO_TRY(use_device(o->device));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    if (o->fused) {                       // did a wait for a peer's slab give up?
        LargeCtrl c;
        DZO_CUDA(cudaMemcpy(&c, o->ctrl, sizeof c, cudaMemcpyDeviceToHost));
        if (c.pad) return fail(DZO_ERR_NCCL, "row-sharded step!: timed out waiting for a peer GPU's rows (is every rank stepping?)");
    }
    return DZO_OK;
}
int dzo_bfgs_step(dzo_bfgs* o, int k) {
    DZO_TRY(dzo_bfgs_step_async(o, k));
    return dzo_bfgs_sync(o);
}

// ============================================================================= field reads
static int read_back(dzo_bfgs* o, void* dst, const void* src, size_t bytes) {
    if (!o || !dst) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    DZO_TRY(use_device(o->device));
    DZO_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, o->stream));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    return DZO_OK;
}
static int read_ctrl(dzo_bfgs* o, LargeCtrl* c) { return read_back(o, c, o->ctrl, sizeof *c); }
}  // extern "C" (templates need C++ linkage)
// scalar field of a (batch of) large-n handle(s): one control block per problem
template <class T, class F>
static int ctrl_field(dzo_bfgs* o, T* out, F pick) {
    for (int64_t q = 0; q < o->batch; ++q) {
        LargeCtrl c;
        DZO_TRY(read_back(o, &c, o->ctrl + q, sizeof c));
        out[q] = (T)pick(c);
    }
    return DZO_OK;
}
// derived layout: the four fields the step kernel does not store, recomputed per pair of elements from the two point
// buffers with the operations (hence the bits) the old layout stored
enum : int { DF_POINT = 0, DF_GRADIENT = 1, DF_DELTA_POINT = 2, DF_DELTA_GRADIENT = 3 };
static __global__ void derived_field_kernel(BatchedArgs A, int field, double* out) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // pair t of the batch
    const int half = A.n / 2;
    if (t >= (long long)half * A.batch) return;
    const long long p = t / half, e = 2 * t;
    const unsigned fl = A.flags[p];
    const double* cur = (fl & BF_PARITY) ? A.g : A.x;
    const double* prev = (fl & BF_PARITY) ? A.x : A.g;
    const double2 xc = *reinterpret_cast<const double2*>(cur + e);
    double2 v = xc;
    if (field == DF_GRADIENT) {
        v = rosen_pair_grad(xc.x, xc.y);
    } else if (field == DF_DELTA_POINT || field == DF_DELTA_GRADIENT) {
        const bool dp = (field == DF_DELTA_POINT);
        if (fl & BF_EXPLICIT) {
            v = *reinterpret_cast<const double2*>((dp ? A.dx : A.dg) + e);
        } else {
            const double2 xp = *reinterpret_cast<const double2*>(prev + e);
            const double2 a = dp ? xp : rosen_pair_grad(xp.x, xp.y), b = dp ? xc : rosen_pair_grad(xc.x, xc.y);
            v = make_double2((-a.x) + b.x, (-a.y) + b.y);                  // :943-944, :949-950
        }
    }
    *reinterpret_cast<double2*>(out + e) = v;
}
static int read_vec(dzo_bfgs* o, double* out, const double* field_ptr, int derived_field) {
    if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");
    const size_t count = (size_t)o->n * (size_t)o->batch;
    if (derived_field < 0 || !o->derived) return read_back(o, out, field_ptr, count * 8);
    if (!out) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    DZO_TRY(use_device(o->device));
    double* tmp = nullptr;
    DZO_TRY(dmalloc_on(o->stream, &tmp, count, o->pooled));
    const long long pairs = (long long)(count / 2);
    derived_field_kernel<<<(unsigned)((pairs + 255) / 256), 256, 0, o->stream>>>(batched_args(o, 0), derived_field, tmp);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, tmp, count * 8, cudaMemcpyDeviceToHost, o->stream);
    cudaFreeAsync(tmp, o->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(o->stream);
    if (e != cudaSuccess) return fail(DZO_ERR_CUDA, "reading a derived field failed: %s", cudaGetErrorString(e));
    return DZO_OK;
}
extern "C" {
int dzo_bfgs_get_point(dzo_bfgs* o, double* out) { return read_vec(o, out, o ? o->x : nullptr, DF_POINT); }
int dzo_bfgs_get_gradient(dzo_bfgs* o, double* out) { return read_vec(o, out, o ? o->g : nullptr, DF_GRADIENT); }
int dzo_bfgs_get_delta_point(dzo_bfgs* o, double* out) { return read_vec(o, out, o ? o->dx : nullptr, DF_DELTA_POINT); }
int dzo_bfgs_get_delta_gradient(dzo_bfgs* o, double* out) { return read_vec(o, out, o ? o->dg : nullptr, DF_DELTA_GRADIENT); }
int dzo_bfgs_get_direction(dzo_bfgs* o, double* out) { return read_vec(o, out, o ? o->d : nullptr, -1); }

int dzo_bfgs_get_inverse_hessian(dzo_bfgs* o, int64_t problem, double* out) {
    if (!o || problem < 0 || problem >= o->batch) return fail(DZO_ERR_INVALID_ARGUMENT, "bad arguments");
    if (o->small && o->lazy) {           // an implicit identity is materialised for the caller, not in HBM
        unsigned char flag = 0;
        DZO_TRY(read_back(o, &flag, o->flags + problem, 1));
        if (flag & BF_IDENT) {
            for (int64_t j = 0; j < o->n; ++j)
                for (int64_t i = 0; i < o->n; ++i) out[j * o->n + i] = (i == j) ? 1.0 : 0.0;
            return DZO_OK;
        }
    }
    if (o->small && o->objective != DZO_OBJ_ROSENBROCK) {
        // generic batched kernel: element e of problem p lives at H[e * batch + p]
        DZO_TRY(use_device(o->device));
        DZO_CUDA(cudaMemcpy2DAsync(out, 8, o->H + problem, (size_t)o->batch * 8, 8, (size_t)o->n * o->n, cudaMemcpyDeviceToHost, o->stream));
        DZO_CUDA(cudaStreamSynchronize(o->stream));
        return DZO_OK;
    }
    if (o->small) return read_back(o, out, o->H + (size_t)problem * o->n * o->n, (size_t)o->n * o->n * 8);
    return read_back(o, out, o->H + (size_t)problem * (size_t)o->rows * (size_t)o->n, (size_t)o->rows * (size_t)o->n * 8);
}
// the mirrored fields are already in the caller's buffer once the stream has drained
static int mirror_sync(dzo_bfgs* o) {
    DZO_TRY(use_device(o->device));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    return DZO_OK;
}
int dzo_bfgs_mirror_fields(dzo_bfgs* o, double* objective_host, uint8_t* terminated_host) {
    if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");
    if (!o->small) return fail(DZO_ERR_UNSUPPORTED, "field mirrors: batched (n <= 32) optimizers only");
    if (o->objective != DZO_OBJ_ROSENBROCK && (objective_host || terminated_host))
        return fail(DZO_ERR_UNSUPPORTED, "field mirrors: the warp-resident batched kernels (DZO_OBJ_ROSENBROCK) only");
    DZO_TRY(use_device(o->device));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    o->f_host = nullptr; o->term_host = nullptr;
    if (!objective_host && !terminated_host) return DZO_OK;
    void* ptrs[2] = {objective_host, terminated_host};
    for (void* p : ptrs) {
        if (!p) continue;
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, p) != cudaSuccess || at.type != cudaMemoryTypeHost || at.devicePointer != p) {
            cudaGetLastError();
            return fail(DZO_ERR_INVALID_ARGUMENT, "field mirrors must be page-locked host memory the device can address "
                                                  "(dzo_host_alloc, or cudaHostRegister with the mapped flag)");
        }
    }
    // bring the mirrors up to date, then let the step kernels maintain them
    if (objective_host) DZO_CUDA(cudaMemcpyAsync(objective_host, o->f, (size_t)o->batch * 8, cudaMemcpyDeviceToHost, o->stream));
    if (terminated_host) DZO_CUDA(cudaMemcpyAsync(terminated_host, o->term, (size_t)o->batch, cudaMemcpyDeviceToHost, o->stream));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    o->f_host = objective_host; o->term_host = terminated_host;
    return DZO_OK;
}
int dzo_bfgs_get_objective(dzo_bfgs* o, double* out) {
    if (!o || !out) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    if (o->small && out == o->f_host) return mirror_sync(o);
    if (o->small) return read_back(o, out, o->f, (size_t)o->batch * 8);
    return ctrl_field(o, out, [](const LargeCtrl& c) { return c.f; });
}
int dzo_bfgs_get_step_length(dzo_bfgs* o, double* out) {
    if (!o || !out) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    if (o->small) return read_back(o, out, o->L, (size_t)o->batch * 8);
    return ctrl_field(o, out, [](const LargeCtrl& c) { return c.L; });
}
int dzo_bfgs_get_step_type(dzo_bfgs* o, int32_t* out) {
    if (!o || !out) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    if (o->small) return read_back(o, out, o->type, (size_t)o->batch * 4);
    return ctrl_field(o, out, [](const LargeCtrl& c) { return c.type; });
}
int dzo_bfgs_get_iteration_count(dzo_bfgs* o, int64_t* out) {
    if (!o || !out) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    if (o->small) return read_back(o, out, o->iter, (size_t)o->batch * 8);
    return ctrl_field(o, out, [](const LargeCtrl& c) { return c.iter; });
}
int dzo_bfgs_get_terminated(dzo_bfgs* o, uint8_t* out) {
    if (!o || !out) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    if (o->small && out == o->term_host) return mirror_sync(o);
    if (o->small) return read_back(o, out, o->term, (size_t)o->batch);
    return ctrl_field(o, out, [](const LargeCtrl& c) { return c.term != 0; });
}
int dzo_bfgs_count_active(dzo_bfgs* o, int64_t* out) {
    if (!o || !out) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    if (!o->small) {
        int64_t active = 0;
        for (int64_t q = 0; q < o->batch; ++q) {
            LargeCtrl c;
            DZO_TRY(read_back(o, &c, o->ctrl + q, sizeof c));
            active += c.term ? 0 : 1;
        }
        *out = active;
        return DZO_OK;
    }
    DZO_TRY(use_device(o->device));
    DZO_CUDA(cudaMemsetAsync(o->counter, 0, 8, o->stream));
    count_active_kernel<<<(unsigned)((o->batch + 255) / 256), 256, 0, o->stream>>>(o->term, o->batch, o->counter);
    DZO_CUDA(cudaGetLastError());
    unsigned long long c = 0;
    DZO_TRY(read_back(o, &c, o->counter, 8));
    *out = (int64_t)c;
    return DZO_OK;
}
int dzo_bfgs_get_step_log(dzo_bfgs* o, int64_t* calls, uint8_t* kinds64) {
    if (!o || !calls || !kinds64) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    if (o->small) return fail(DZO_ERR_UNSUPPORTED, "step log exists for large-n handles only");
    LargeCtrl c; DZO_TRY(read_ctrl(o, &c));
    *calls = c.calls;
    memcpy(kinds64, c.kind_log, 64);
    return DZO_OK;
}
int dzo_bfgs_get_step_kind_counts(dzo_bfgs* o, int64_t* counts8, int reset) {
    if (!o || !counts8) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    if (!o->small || !o->stats) return fail(DZO_ERR_UNSUPPORTED, "step-kind counters exist for batched handles only (large n: dzo_bfgs_get_step_log)");
    unsigned long long c[HK_COUNT];
    DZO_TRY(read_back(o, c, o->stats, sizeof c));
    for (int k = 0; k < 8; ++k) counts8[k] = (k < HK_COUNT) ? (int64_t)c[k] : 0;
    if (reset) {
        DZO_CUDA(cudaMemsetAsync(o->stats, 0, sizeof c, o->stream));
        DZO_CUDA(cudaStreamSynchronize(o->stream));
    }
    return DZO_OK;
}
int dzo_bfgs_batched_layout(dzo_bfgs* o, int* lazy, int* derived) {
    if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");
    if (!o->flags) return fail(DZO_ERR_UNSUPPORTED, "layout knobs exist for batched handles with the small-n step kernel only");
    if (lazy) *lazy = o->lazy ? 1 : 0;
    if (derived) *derived = o->derived ? 1 : 0;
    return DZO_OK;
}
int dzo_bfgs_gather_mode(dzo_bfgs* o, int* mode) {
    if (!o || !mode) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    *mode = (o->nranks <= 1) ? 0 : (o->fused ? 1 : 2);
    return DZO_OK;
}
int dzo_bfgs_info(dzo_bfgs* o, int64_t* n, int64_t* batch, int* order, int64_t* row_begin, int64_t* row_end) {
    if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");
    if (n) *n = o->n;
    if (batch) *batch = o->batch;
    if (order) *order = o->small ? DZO_ORDER_SEQUENTIAL : DZO_ORDER_TREE;
    if (row_begin) *row_begin = o->small ? 0 : o->row0;
    if (row_end) *row_end = o->small ? o->n : o->row0 + o->rows;
    return DZO_OK;
}

// ============================================================================= resume
int dzo_bfgs_set_state(dzo_bfgs* o, const double* point, const double* inverse_hessian, const double* delta_point,
                       const double* delta_gradient, const double* last_step_length, const int32_t* last_step_type,
                       const int64_t* iteration_count) {
    if (!o || !point || !inverse_hessian || !delta_point || !delta_gradient || !last_step_length || !last_step_type ||
        !iteration_count)
        return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    DZO_TRY(use_device(o->device));
    if (o->riesz) return fail(DZO_ERR_UNSUPPORTED, "set_state is not available for the large-n Riesz objective yet");
    const size_t nb = (size_t)o->n * (size_t)o->batch * 8;
    DZO_CUDA(cudaMemcpyAsync(o->x, point, nb, cudaMemcpyHostToDevice, o->stream));              // :825
    DZO_CUDA(cudaMemcpyAsync(o->dx, delta_point, nb, cudaMemcpyHostToDevice, o->stream));       // :853
    DZO_CUDA(cudaMemcpyAsync(o->dg, delta_gradient, nb, cudaMemcpyHostToDevice, o->stream));    // :854
    if (o->small) {
        if (o->objective != DZO_OBJ_ROSENBROCK) {
            // generic batched kernel: scatter the caller's problem-major matrices into the batch-innermost layout
            double* tmp = nullptr;
            DZO_TRY(dmalloc_on(o->stream, &tmp, (size_t)o->n * o->n * (size_t)o->batch, o->pooled));
            DZO_CUDA(cudaMemcpyAsync(tmp, inverse_hessian, nb * (size_t)o->n, cudaMemcpyHostToDevice, o->stream));
            const long long total = (long long)o->n * o->n * o->batch;
            h_to_batch_inner_kernel<<<(unsigned)((total + 255) / 256), 256, 0, o->stream>>>(tmp, o->H, (long long)o->n * o->n, o->batch);
            DZO_CUDA(cudaGetLastError());
            if (o->pooled) cudaFreeAsync(tmp, o->stream); else { cudaStreamSynchronize(o->stream); cudaFree(tmp); }
        } else
        DZO_CUDA(cudaMemcpyAsync(o->H, inverse_hessian, nb * (size_t)o->n, cudaMemcpyHostToDevice, o->stream));  // :832
        DZO_CUDA(cudaMemcpyAsync(o->L, last_step_length, (size_t)o->batch * 8, cudaMemcpyHostToDevice, o->stream));
        DZO_CUDA(cudaMemcpyAsync(o->type, last_step_type, (size_t)o->batch * 4, cudaMemcpyHostToDevice, o->stream));
        DZO_CUDA(cudaMemcpyAsync(o->iter, iteration_count, (size_t)o->batch * 8, cudaMemcpyHostToDevice, o->stream));
        DZO_TRY(batched_restore(o));
        bool bad = false;
        DZO_TRY(any_nan(o, o->f, o->batch, &bad));
        if (bad) return fail(DZO_ERR_NAN_OBJECTIVE, "objective is NaN at the restored point");   // :829
        if (o->f_host) DZO_CUDA(cudaMemcpyAsync(o->f_host, o->f, (size_t)o->batch * 8, cudaMemcpyDeviceToHost, o->stream));
        if (o->term_host) DZO_CUDA(cudaMemcpyAsync(o->term_host, o->term, (size_t)o->batch, cudaMemcpyDeviceToHost, o->stream));
        if (o->f_host || o->term_host) DZO_CUDA(cudaStreamSynchronize(o->stream));
        return DZO_OK;
    }
    // large: the caller passes the full n x n matrix (per problem); keep rows [row0, row0+rows) of every column
    DZO_CUDA(cudaMemcpy2DAsync(o->H, (size_t)o->rows * 8, inverse_hessian + o->row0, (size_t)o->n * 8, (size_t)o->rows * 8,
                               (size_t)o->n * (size_t)o->batch, cudaMemcpyHostToDevice, o->stream));   // (batch > 1: rows == n)
    for (int64_t q = 0; q < o->batch; ++q) {
        LargeCtrl c;
        DZO_CUDA(cudaMemcpyAsync(&c, o->ctrl + q, sizeof c, cudaMemcpyDeviceToHost, o->stream));
        DZO_CUDA(cudaStreamSynchronize(o->stream));
        c.L = last_step_length[q]; c.type = last_step_type[q]; c.iter = iteration_count[q];          // :848, :855-856
        DZO_CUDA(cudaMemcpyAsync(o->ctrl + q, &c, sizeof c, cudaMemcpyHostToDevice, o->stream));
        DZO_CUDA(cudaStreamSynchronize(o->stream));
    }
    vec_bfgs_restore_kernel<<<(unsigned)o->batch, 1024, 0, o->stream>>>(large_vecs(o));
    DZO_CUDA(cudaGetLastError());
    DZO_TRY(large_gemv(o, o->g, o->d, -1));                                                          // :833-836
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    for (int64_t q = 0; q < o->batch; ++q) {
        LargeCtrl c;
        DZO_TRY(read_back(o, &c, o->ctrl + q, sizeof c));
        if (c.f != c.f) return fail(DZO_ERR_NAN_OBJECTIVE, "objective is NaN at the restored point");
    }
    return DZO_OK;
}

// ============================================================================= kernel-level entry points
static int h2d(DevBuf& b, const double* src, size_t count) {
    DZO_TRY(b.alloc(count * 8));
    if (src) DZO_CUDA(cudaMemcpy(b.p, src, count * 8, cudaMemcpyHostToDevice));
    return DZO_OK;
}
static int d2h(double* dst, const DevBuf& b, size_t count) {
    DZO_CUDA(cudaMemcpy(dst, b.p, count * 8, cudaMemcpyDeviceToHost));
    return DZO_OK;
}
static int order_ok(int order, int64_t n) {
    if (order == DZO_ORDER_SEQUENTIAL) {
        if (n > DZO_SMALL_N_MAX) return fail(DZO_ERR_UNSUPPORTED, "SEQUENTIAL order on the device needs n <= %d", DZO_SMALL_N_MAX);
        return DZO_OK;
    }
    if (order != DZO_ORDER_TREE) return fail(DZO_ERR_INVALID_ARGUMENT, "unknown summation order");
    return DZO_OK;
}

int dzo_dev_dot(int order, int64_t n, const double* v, const double* w, double* out, int device) {
    if (!v || !w || !out || n <= 0) return fail(DZO_ERR_INVALID_ARGUMENT, "bad arguments");
    DZO_TRY(order_ok(order, n));
    DZO_TRY(use_device(device));
    DevBuf dv, dw, dout;
    DZO_TRY(h2d(dv, v, (size_t)n)); DZO_TRY(h2d(dw, w, (size_t)n)); DZO_TRY(h2d(dout, nullptr, 1));
    if (order == DZO_ORDER_SEQUENTIAL) small_dot_kernel<<<1, 32>>>(dv.as<double>(), dw.as<double>(), (int)n, dout.as<double>());
    else vec_dot_kernel<<<1, 1024>>>(dv.as<double>(), dw.as<double>(), n, dout.as<double>());
    DZO_CUDA(cudaGetLastError());
    DZO_CUDA(cudaDeviceSynchronize());
    return d2h(out, dout, 1);
}

// scratch for a stand-alone TREE sweep on an n x n matrix
struct SweepScratch {
    DevBuf partial, counters, ctrl;
    int init(int64_t n) {
        const size_t nchunks = (size_t)((n + DZO_GEMV_CHUNK - 1) / DZO_GEMV_CHUNK);
        const size_t rblocks = (size_t)((n + kSweepMinRows - 1) / kSweepMinRows);
        DZO_TRY(partial.alloc(nchunks * (size_t)n * 8));
        DZO_TRY(counters.alloc(rblocks * 4));
        DZO_TRY(ctrl.alloc(sizeof(LargeCtrl)));
        DZO_CUDA(cudaMemset(counters.p, 0, rblocks * 4));
        DZO_CUDA(cudaMemset(ctrl.p, 0, sizeof(LargeCtrl)));
        return DZO_OK;
    }
    SweepArgs args(double* H, int64_t n) const {
        SweepArgs a;
        a.H = H; a.ld = n; a.rows = n; a.n = n; a.row0 = 0; a.v = nullptr; a.s = nullptr; a.t = nullptr;
        a.partial = partial.as<double>(); a.out = nullptr; a.counters = counters.as<unsigned>();
        a.ctrl = nullptr; a.need_kind = DZO_STEP_BFGS;
        a.nchunks = (int)((n + DZO_GEMV_CHUNK - 1) / DZO_GEMV_CHUNK);
        memset(&a.peers, 0, sizeof a.peers);
        a.peers.nranks = 1;
        return a;
    }
};

int dzo_dev_gemv(int order, int64_t n, const double* H, const double* v, double* out, int device) {
    if (!H || !v || !out || n <= 0) return fail(DZO_ERR_INVALID_ARGUMENT, "bad arguments");
    DZO_TRY(order_ok(order, n));
    DZO_TRY(use_device(device));
    DevBuf dH, dv, dout;
    DZO_TRY(h2d(dH, H, (size_t)n * n)); DZO_TRY(h2d(dv, v, (size_t)n)); DZO_TRY(h2d(dout, nullptr, (size_t)n));
    if (order == DZO_ORDER_SEQUENTIAL) {
        small_gemv_kernel<<<1, 32>>>(dH.as<double>(), dv.as<double>(), (int)n, dout.as<double>());
    } else {
        SweepScratch sc;
        DZO_TRY(sc.init(n));
        SweepArgs a = sc.args(dH.as<double>(), n);
        a.v = dv.as<double>(); a.out = dout.as<double>();
        launch_gemv(sweep_grid(n, n), sweep_threads(n, n), nullptr, a);
        DZO_CUDA(cudaGetLastError());
        DZO_CUDA(cudaDeviceSynchronize());
    }
    DZO_CUDA(cudaGetLastError());
    DZO_CUDA(cudaDeviceSynchronize());
    return d2h(out, dout, (size_t)n);
}

int dzo_dev_update_inverse_hessian(int order, int64_t n, double* H, double step_length, double* step_direction,
                                   const double* delta_gradient, double* scratch, const double* next_gradient,
                                   double* next_direction, int device) {
    if (!H || !step_direction || !delta_gradient || !scratch || n <= 0) return fail(DZO_ERR_INVALID_ARGUMENT, "bad arguments");
    DZO_TRY(order_ok(order, n));
    DZO_TRY(use_device(device));
    const bool fused = next_gradient && next_direction;
    DevBuf dH, dd, ddg, dt, dg, dnd, dsd;
    DZO_TRY(h2d(dH, H, (size_t)n * n)); DZO_TRY(h2d(dd, step_direction, (size_t)n)); DZO_TRY(h2d(ddg, delta_gradient, (size_t)n));
    DZO_TRY(h2d(dt, nullptr, (size_t)n)); DZO_TRY(h2d(dg, fused ? next_gradient : nullptr, (size_t)n));
    DZO_TRY(h2d(dnd, nullptr, (size_t)n)); DZO_TRY(h2d(dsd, nullptr, (size_t)n));
    if (order == DZO_ORDER_SEQUENTIAL) {
        small_update_kernel<<<1, 32>>>(dH.as<double>(), step_length, dd.as<double>(), ddg.as<double>(), dt.as<double>(),
                                       fused ? dg.as<double>() : nullptr, fused ? dnd.as<double>() : nullptr, (int)n);
        DZO_CUDA(cudaGetLastError());
        DZO_CUDA(cudaDeviceSynchronize());
        DZO_TRY(d2h(step_direction, dd, (size_t)n));
    } else {
        SweepScratch sc;
        DZO_TRY(sc.init(n));
        LargeVecs v;
        v.x = nullptr; v.g = dg.as<double>(); v.d = dd.as<double>(); v.dx = nullptr; v.dg = ddg.as<double>();
        v.sd = dsd.as<double>(); v.t = dt.as<double>(); v.ctrl = sc.ctrl.as<LargeCtrl>(); v.n = n;
        vec_overlap_scale_kernel<<<1, 1024>>>(v, step_length);                        // :873-874
        SweepArgs a = sc.args(dH.as<double>(), n);
        a.ctrl = sc.ctrl.as<LargeCtrl>();
        a.v = ddg.as<double>(); a.out = dt.as<double>();
        launch_gemv(sweep_grid(n, n), sweep_threads(n, n), nullptr, a);                // :875
        vec_delta_kernel<<<1, 1024>>>(v);                                              // :876
        a.v = fused ? dg.as<double>() : nullptr; a.out = fused ? dnd.as<double>() : nullptr;
        a.s = dsd.as<double>(); a.t = dt.as<double>();
        launch_update(sweep_grid(n, n), sweep_threads(n, n), nullptr, a);             // :878-886 (+ :958-960)
        DZO_CUDA(cudaGetLastError());
        DZO_CUDA(cudaDeviceSynchronize());
        DZO_TRY(d2h(step_direction, dsd, (size_t)n));
    }
    DZO_TRY(d2h(H, dH, (size_t)n * n));
    DZO_TRY(d2h(scratch, dt, (size_t)n));
    if (fused) DZO_TRY(d2h(next_direction, dnd, (size_t)n));
    return DZO_OK;
}

int dzo_dev_identity(int64_t n, double* H, int device) {
    if (!H || n <= 0) return fail(DZO_ERR_INVALID_ARGUMENT, "bad arguments");
    DZO_TRY(use_device(device));
    DevBuf dH;
    DZO_TRY(h2d(dH, nullptr, (size_t)n * n));
    SweepScratch sc;
    DZO_TRY(sc.init(n));
    SweepArgs a = sc.args(dH.as<double>(), n);
    identity_kernel<<<sweep_grid(n, n), sweep_threads(n, n)>>>(a);
    DZO_CUDA(cudaGetLastError());
    DZO_CUDA(cudaDeviceSynchronize());
    return d2h(H, dH, (size_t)n * n);
}

int dzo_dev_line_search(int objective, int constraint, int64_t obj_param, int order, int64_t n, const double* x,
                        const double* dir, double f0, double t1, double* t_best, double* f_best, int device);
int dzo_dev_objective(int objective, int constraint, int64_t obj_param, int order, int64_t n, int64_t batch,
                      const double* x, double* f, int device);
int dzo_dev_gradient(int objective, int constraint, int64_t obj_param, int order, int64_t n, int64_t batch,
                     const double* x, double* g, int device);

}  // extern "C"

// line search / objective / gradient: Rosenbrock handled here, Riesz in dzopt_gd.cu
namespace dzo {
int riesz_dev_objective(int constraint, int64_t dim, int order, int64_t n, int64_t batch, const double* x, double* f);
int riesz_dev_gradient(int constraint, int64_t dim, int order, int64_t n, int64_t batch, const double* x, double* g);
int riesz_dev_line_search(int constraint, int64_t dim, int order, int64_t n, const double* x, const double* dir, double f0,
                          double t1, double* t_best, double* f_best);

__global__ void __launch_bounds__(1024, 1) vec_line_search_kernel(const double* x, const double* dir, long long n, double f0,
                                                                  double t1, double* out2) {
    __shared__ double sm[132];
    double tb, fb;
    long long evals = 0;
    cta_line_search_rosenbrock(x, dir, n, f0, t1, -1.0, 0, sm, tb, fb, evals);
    if (threadIdx.x == 0) { out2[0] = tb; out2[1] = fb; }
}
}  // namespace dzo

extern "C" {

int dzo_dev_line_search(int objective, int constraint, int64_t obj_param, int order, int64_t n, const double* x,
                        const double* dir, double f0, double t1, double* t_best, double* f_best, int device) {
    if (!x || !dir || !t_best || !f_best) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    DZO_TRY(check_problem(objective, constraint, obj_param, n, 1));
    DZO_TRY(order_ok(order, n));
    DZO_TRY(use_device(device));
    if (objective == DZO_OBJ_RIESZ) return riesz_dev_line_search(constraint, obj_param, order, n, x, dir, f0, t1, t_best, f_best);
    DevBuf dx, dd, dout;
    DZO_TRY(h2d(dx, x, (size_t)n)); DZO_TRY(h2d(dd, dir, (size_t)n)); DZO_TRY(h2d(dout, nullptr, 2));
    if (order == DZO_ORDER_SEQUENTIAL)
        small_line_search_kernel<RosenbrockSmall><<<1, 32>>>(dx.as<double>(), dd.as<double>(), (int)n, f0, t1, dout.as<double>());
    else
        vec_line_search_kernel<<<1, 1024>>>(dx.as<double>(), dd.as<double>(), n, f0, t1, dout.as<double>());
    DZO_CUDA(cudaGetLastError());
    DZO_CUDA(cudaDeviceSynchronize());
    double r[2];
    DZO_TRY(d2h(r, dout, 2));
    *t_best = r[0]; *f_best = r[1];
    return DZO_OK;
}

int dzo_dev_objective(int objective, int constraint, int64_t obj_param, int order, int64_t n, int64_t batch,
                      const double* x, double* f, int device) {
    if (!x || !f) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    DZO_TRY(check_problem(objective, constraint, obj_param, n, batch));
    DZO_TRY(order_ok(order, n));
    DZO_TRY(use_device(device));
    if (objective == DZO_OBJ_RIESZ) return riesz_dev_objective(constraint, obj_param, order, n, batch, x, f);
    DevBuf dx, df;
    DZO_TRY(h2d(dx, x, (size_t)n * batch)); DZO_TRY(h2d(df, nullptr, (size_t)batch));
    if (order == DZO_ORDER_SEQUENTIAL) small_objective_kernel<RosenbrockSmall><<<(unsigned)batch, 32>>>(dx.as<double>(), (int)n, df.as<double>());
    else vec_rosenbrock_objective_kernel<<<(unsigned)batch, 1024>>>(dx.as<double>(), n, df.as<double>());
    DZO_CUDA(cudaGetLastError());
    DZO_CUDA(cudaDeviceSynchronize());
    return d2h(f, df, (size_t)batch);
}

int dzo_dev_gradient(int objective, int constraint, int64_t obj_param, int order, int64_t n, int64_t batch,
                     const double* x, double* g, int device) {
    if (!x || !g) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    DZO_TRY(check_problem(objective, constraint, obj_param, n, batch));
    DZO_TRY(order_ok(order, n));
    DZO_TRY(use_device(device));
    if (objective == DZO_OBJ_RIESZ) return riesz_dev_gradient(constraint, obj_param, order, n, batch, x, g);
    DevBuf dx, dg;
    DZO_TRY(h2d(dx, x, (size_t)n * batch)); DZO_TRY(h2d(dg, nullptr, (size_t)n * batch));
    if (order == DZO_ORDER_SEQUENTIAL) {
        small_gradient_kernel<RosenbrockSmall><<<(unsigned)batch, 32>>>(dx.as<double>(), (int)n, dg.as<double>());
    } else {
        const long long pairs = (long long)n * batch / 2;
        vec_rosenbrock_gradient_kernel<<<(unsigned)((pairs + 255) / 256), 256>>>(dx.as<double>(), pairs, dg.as<double>());
    }
    DZO_CUDA(cudaGetLastError());
    DZO_CUDA(cudaDeviceSynchronize());
    return d2h(g, dg, (size_t)n * batch);
}

// ============================================================================= measurement hooks
int dzo_bench_kernel(int which, int64_t n, int reps, int variant, float* ms_per_launch, int device) {
    if (!ms_per_launch || n <= 0 || reps <= 0) return fail(DZO_ERR_INVALID_ARGUMENT, "bad arguments");
    (void)variant;
    DZO_TRY(use_device(device));
    DevBuf dH, vs, vt, vg, vo;
    DZO_TRY(h2d(dH, nullptr, (size_t)n * n));
    DZO_TRY(h2d(vs, nullptr, (size_t)n)); DZO_TRY(h2d(vt, nullptr, (size_t)n)); DZO_TRY(h2d(vg, nullptr, (size_t)n));
    DZO_TRY(h2d(vo, nullptr, (size_t)n));
    SweepScratch sc;
    DZO_TRY(sc.init(n));
    SweepArgs a = sc.args(dH.as<double>(), n);
    // H = I and tiny vectors: the sweeps are data-independent, values only need to stay finite
    identity_kernel<<<sweep_grid(n, n), sweep_threads(n, n)>>>(a);
    DZO_CUDA(cudaMemset(vs.p, 0, (size_t)n * 8)); DZO_CUDA(cudaMemset(vt.p, 0, (size_t)n * 8));
    DZO_CUDA(cudaMemset(vg.p, 0, (size_t)n * 8));
    LargeCtrl c;
    memset(&c, 0, sizeof c);
    c.kind = DZO_STEP_BFGS; c.delta_norm = 1.0;
    DZO_CUDA(cudaMemcpy(sc.ctrl.p, &c, sizeof c, cudaMemcpyHostToDevice));
    a.ctrl = sc.ctrl.as<LargeCtrl>();
    a.v = vg.as<double>(); a.s = vs.as<double>(); a.t = vt.as<double>(); a.out = vo.as<double>();
    cudaEvent_t e0, e1;
    DZO_CUDA(cudaEventCreate(&e0)); DZO_CUDA(cudaEventCreate(&e1));
    auto launch = [&]() {
        if (which == DZO_BENCH_GEMV) launch_gemv(sweep_grid(n, n), sweep_threads(n, n), nullptr, a);
        else if (which == DZO_BENCH_UPDATE_GEMV) launch_update(sweep_grid(n, n), sweep_threads(n, n), nullptr, a);
        else identity_kernel<<<sweep_grid(n, n), sweep_threads(n, n)>>>(a);
    };
    for (int i = 0; i < 3; ++i) launch();
    DZO_CUDA(cudaDeviceSynchronize());
    DZO_CUDA(cudaEventRecord(e0));
    for (int i = 0; i < reps; ++i) launch();
    DZO_CUDA(cudaEventRecord(e1));
    DZO_CUDA(cudaEventSynchronize(e1));
    DZO_CUDA(cudaGetLastError());
    float ms = 0;
    DZO_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *ms_per_launch = ms / reps;
    return DZO_OK;
}

int dzo_host_register(void* ptr, uint64_t bytes) {
    if (!ptr || bytes == 0) return fail(DZO_ERR_INVALID_ARGUMENT, "bad arguments");
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(DZO_ERR_NO_DEVICE, "no CUDA device available");
    }
    DZO_CUDA(cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterPortable));
    return DZO_OK;
}
int dzo_host_unregister(void* ptr) {
    if (!ptr) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    DZO_CUDA(cudaHostUnregister(ptr));
    return DZO_OK;
}

int dzo_host_alloc(void** out, uint64_t bytes) {
    if (!out || bytes == 0) return fail(DZO_ERR_INVALID_ARGUMENT, "bad arguments");
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(DZO_ERR_NO_DEVICE, "no CUDA device available");
    }
    if (cudaHostAlloc(out, (size_t)bytes, cudaHostAllocPortable | cudaHostAllocMapped) != cudaSuccess) {
        cudaGetLastError();
        return fail(DZO_ERR_ALLOC, "cudaHostAlloc of %llu bytes failed", (unsigned long long)bytes);
    }
    return DZO_OK;
}
int dzo_host_free(void* ptr) {
    if (!ptr) return DZO_OK;
    DZO_CUDA(cudaFreeHost(ptr));
    return DZO_OK;
}

int dzo_set_tuning(const char* key, int value) {
    if (!key) return fail(DZO_ERR_INVALID_ARGUMENT, "null key");
    g_tuning.epoch += 1;                                  // captured step graphs are rebuilt
    if (!strcmp(key, "use_graph")) { g_tuning.use_graph = value; return DZO_OK; }
    if (!strcmp(key, "search_variant")) { g_tuning.search_variant = value; return DZO_OK; }
    if (!strcmp(key, "riesz_profile")) { g_tuning.riesz_profile = value; return DZO_OK; }
    if (!strcmp(key, "riesz_esplit")) { g_tuning.riesz_esplit = value; return DZO_OK; }
    if (!strcmp(key, "riesz_pair")) { g_tuning.riesz_pair = value; return DZO_OK; }
    if (!strcmp(key, "riesz_threads")) { g_tuning.riesz_threads = value; return DZO_OK; }
    if (!strcmp(key, "riesz_bar")) { g_tuning.riesz_bar = value; return DZO_OK; }
    if (!strcmp(key, "batched_tile")) { g_tuning.batched_tile = value; return DZO_OK; }
    if (!strcmp(key, "small_sweeps")) { g_tuning.small_sweeps = value; return DZO_OK; }
    if (!strcmp(key, "warp_search")) { g_tuning.warp_search = value; return DZO_OK; }
    if (!strcmp(key, "grid_ll")) { g_tuning.grid_ll = value; return DZO_OK; }
    if (!strcmp(key, "grid_stage")) { g_tuning.grid_stage = value; return DZO_OK; }
    if (!strcmp(key, "grid_profile")) { g_tuning.grid_profile = value; return DZO_OK; }
    if (!strcmp(key, "grid_ll_backoff")) { g_tuning.grid_ll_backoff = value; return DZO_OK; }
    if (!strcmp(key, "grid_ll_first_seq")) { g_tuning.grid_ll_first_seq = value; return DZO_OK; }
    if (!strcmp(key, "riesz_gvariant")) { g_tuning.riesz_gvariant = value; return DZO_OK; }
    if (!strcmp(key, "sharded_variant")) { g_tuning.sharded_variant = value; return DZO_OK; }
    if (!strcmp(key, "sweep_unroll")) { g_tuning.sweep_unroll = value; return DZO_OK; }
    if (!strcmp(key, "sweep_threads")) {
        if (value != 0 && value != 32 && value != 64 && value != 128 && value != 256) return fail(DZO_ERR_INVALID_ARGUMENT, "sweep_threads: 0, 32, 64, 128 or 256");
        g_tuning.sweep_threads = value; return DZO_OK;
    }
    if (!strcmp(key, "lbfgs_batched_threads")) {
        if (value != 64 && value != 128 && value != 256) return fail(DZO_ERR_INVALID_ARGUMENT, "lbfgs_batched_threads: 64, 128 or 256");
        g_tuning.lbfgs_batched_threads = value; return DZO_OK;
    }
    if (!strcmp(key, "batched_prefetch")) { g_tuning.batched_prefetch = value; return DZO_OK; }
    if (!strcmp(key, "batched_lazy")) { g_tuning.batched_lazy = value; return DZO_OK; }
    if (!strcmp(key, "batched_derived")) { g_tuning.batched_derived = value; return DZO_OK; }
    return fail(DZO_ERR_INVALID_ARGUMENT, "unknown tuning key '%s'", key);
}

}  // extern "C"
