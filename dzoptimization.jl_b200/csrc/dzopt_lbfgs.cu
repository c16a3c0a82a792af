// dzopt_lbfgs.cu -- C ABI of the live package's LBFGSOptimizer (src/DZOptimization.jl:321-509).
#include <new>

#include "host_common.h"
#include "grid_lbfgs.cuh"
#include "legacy_lbfgs.cuh"
#include "grid_legacy_lbfgs.cuh"
#include "batched_lbfgs.cuh"

using namespace dzo;

// the grid-wide kernels live in grid_lbfgs_tu.cu / grid_legacy_tu.cu
namespace dzo {
void* grid_lbfgs_kernel_ptr(int own);
void* grid_adgd_kernel_ptr();
void* grid_legacy_kernel_ptr(int own);
// the batched kernel lives in batched_lbfgs_tu.cu
const void* batched_lbfgs_kernel_ptr(int n);
cudaError_t batched_lbfgs_transpose(const double* src, double* dst, int n, long long batch, int to_public, cudaStream_t stream);
}

struct dzo_lbfgs {
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    int64_t n = 0;
    int m = 0;
    double *x = nullptr, *dx = nullptr, *g = nullptr, *dg = nullptr, *d = nullptr, *S = nullptr, *Y = nullptr;
    LbfgsCtrl* ctrl = nullptr;
    // n > DZO_TREE_BLOCK: cooperative grid of clusters, one cluster per block (grid_lbfgs.cuh)
    bool use_grid = false;
    int nblocks = 0, nclusters = 0;          // nclusters: CTAs of the cooperative grid
    double* part = nullptr;
    unsigned* fpart = nullptr;
    // batch > 0: dzo_lbfgs_create_batched, one thread per problem (batched_lbfgs.cuh); every array has the batch innermost
    // and the per-problem scalars replace ctrl
    int64_t batch = 0;
    int threads = 0, ctas = 0;
    size_t smem = 0;
    double *rho = nullptr, *f = nullptr, *df = nullptr;
    long long* iter = nullptr;
    int *count = nullptr, *head = nullptr;
    unsigned char* stuck = nullptr;
    double* scratch = nullptr;               // n x batch: the public column-major layout on its way in and out
};

static void free_lbfgs(dzo_lbfgs* o) {
    if (!o) return;
    cudaSetDevice(o->device);
    void* ptrs[] = {o->x, o->dx, o->g, o->dg, o->d, o->S, o->Y, o->ctrl, o->part, o->fpart,
                    o->rho, o->f, o->df, o->iter, o->count, o->head, o->stuck, o->scratch};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (o->own_stream) cudaStreamDestroy(o->own_stream);
    delete o;
}

static int lbfgs_launch(dzo_lbfgs* o, int mode, int k, double L0) {
    if (o->batch) {
        BatchedLbfgsArgs a;
        a.x = o->x; a.dx = o->dx; a.g = o->g; a.dg = o->dg; a.d = o->d; a.S = o->S; a.Y = o->Y; a.rho = o->rho;
        a.f = o->f; a.df = o->df; a.iter = o->iter; a.count = o->count; a.head = o->head; a.stuck = o->stuck;
        a.batch = o->batch; a.m = o->m; a.ksteps = k; a.mode = mode; a.initial_step_length = L0;
        void* params[] = {&a};
        DZO_CUDA(cudaLaunchKernel(batched_lbfgs_kernel_ptr((int)o->n), dim3((unsigned)o->ctas), dim3((unsigned)o->threads),
                                  params, o->smem, o->stream));
        return DZO_OK;
    }
    if (o->use_grid) {
        GridLbfgsArgs g;
        g.x = o->x; g.dx = o->dx; g.g = o->g; g.dg = o->dg; g.d = o->d; g.S = o->S; g.Y = o->Y; g.ctrl = o->ctrl;
        g.part = o->part; g.fpart = o->fpart; g.n = o->n; g.m = o->m; g.ksteps = k; g.nblocks = o->nblocks;
        g.mode = mode; g.initial_step_length = L0;
        const bool own1 = (8 * o->nblocks <= o->nclusters);       // one eighth per CTA: direction in registers, staged passes
        g.stage = (own1 && g_tuning.grid_stage) ? 1 : 0;
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof cfg);
        cfg.gridDim = dim3((unsigned)o->nclusters);
        cfg.blockDim = dim3(kClusterThreads);
        cfg.dynamicSmemBytes = g.stage ? kGridStageBytes : 0;
        if (g_tuning.grid_profile && mode == 0) g.stage |= 2;
        cfg.stream = o->stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeCooperative;
        attr[0].val.cooperative = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        void* params[] = {&g};
        DZO_CUDA(cudaLaunchKernelExC(&cfg, grid_lbfgs_kernel_ptr(own1 ? 1 : kGridOwnMax), params));
        return DZO_OK;
    }
    LbfgsArgs a;
    a.x = o->x; a.dx = o->dx; a.g = o->g; a.dg = o->dg; a.d = o->d; a.S = o->S; a.Y = o->Y; a.ctrl = o->ctrl;
    a.n = o->n; a.m = o->m; a.ksteps = k; a.initial_step_length = L0; a.mode = mode;
    cluster_lbfgs_kernel<<<kClusterCtas, kClusterThreads, 0, o->stream>>>(a);
    DZO_CUDA(cudaGetLastError());
    return DZO_OK;
}

extern "C" {

int dzo_lbfgs_create(dzo_lbfgs** out, int objective, int constraint, int64_t obj_param, int64_t n, const double* x0,
                     double initial_step_length, int history_length, int device) {
    if (!out || !x0) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    *out = nullptr;
    DZO_TRY(check_problem(objective, constraint, obj_param, n, 1));
    if (objective != DZO_OBJ_ROSENBROCK) return fail(DZO_ERR_UNSUPPORTED, "LBFGSOptimizer device objective: DZO_OBJ_ROSENBROCK");
    if (history_length < 1 || history_length > DZO_LBFGS_MAX_HISTORY)
        return fail(DZO_ERR_INVALID_ARGUMENT, "history_length must be in [1, %d]", DZO_LBFGS_MAX_HISTORY);
    if (!(initial_step_length > 0.0)) return fail(DZO_ERR_INVALID_ARGUMENT, "initial_step_length must be positive");   // :375
    DZO_TRY(use_device(device));
    dzo_lbfgs* o = new (std::nothrow) dzo_lbfgs();
    if (!o) return fail(DZO_ERR_ALLOC, "out of memory");
    o->device = device; o->n = n; o->m = history_length;
    auto bail = [&](int code) { free_lbfgs(o); return code; };
    if (cudaStreamCreateWithFlags(&o->own_stream, cudaStreamNonBlocking) != cudaSuccess)
        return bail(fail(DZO_ERR_CUDA, "cudaStreamCreate failed"));
    o->stream = o->own_stream;
    const size_t vb = (size_t)n * 8;
    double** vecs[] = {&o->x, &o->dx, &o->g, &o->dg, &o->d};
    for (double** v : vecs)
        if (cudaMalloc((void**)v, vb) != cudaSuccess) return bail(fail(DZO_ERR_ALLOC, "cudaMalloc failed"));
    if (cudaMalloc((void**)&o->S, vb * history_length) != cudaSuccess || cudaMalloc((void**)&o->Y, vb * history_length) != cudaSuccess ||
        cudaMalloc((void**)&o->ctrl, sizeof(LbfgsCtrl)) != cudaSuccess)
        return bail(fail(DZO_ERR_ALLOC, "cudaMalloc failed"));
    if (cudaMemcpyAsync(o->x, x0, vb, cudaMemcpyHostToDevice, o->stream) != cudaSuccess ||
        cudaMemsetAsync(o->S, 0, vb * history_length, o->stream) != cudaSuccess ||
        cudaMemsetAsync(o->Y, 0, vb * history_length, o->stream) != cudaSuccess)
        return bail(fail(DZO_ERR_CUDA, "initial copies failed"));
    if (n > DZO_TREE_BLOCK) {
        // eight 512-thread CTAs per block of DZO_TREE_BLOCK elements, as many CTAs as are co-resident (cooperative launch)
        o->nblocks = (int)((n + DZO_TREE_BLOCK - 1) / DZO_TREE_BLOCK);
        int per_sm = 0, sms = 0;
        int per_sm_one = 0;               // the launch picks OWN = 1 or kGridOwnMax: size the grid for the tighter of the two
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)grid_lbfgs_kernel_ptr(kGridOwnMax), kClusterThreads, 0) != cudaSuccess ||
            cudaFuncSetAttribute((const void*)grid_lbfgs_kernel_ptr(1), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGridStageBytes) != cudaSuccess ||
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_one, (const void*)grid_lbfgs_kernel_ptr(1), kClusterThreads, kGridStageBytes) != cudaSuccess ||
            (per_sm = per_sm < per_sm_one ? per_sm : per_sm_one) < 0 ||
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || per_sm < 1 || sms < 1) {
            cudaGetLastError();
            return bail(fail(DZO_ERR_CUDA, "the grid-wide L-BFGS kernel does not fit on this device"));
        }
        const int resident = per_sm * sms;
        o->nclusters = 8 * o->nblocks < resident ? 8 * o->nblocks : resident;      // CTAs of the grid
        if (o->nblocks > kGridMaxBlocks || 8 * o->nblocks > kGridOwnMax * o->nclusters)
            return bail(fail(DZO_ERR_UNSUPPORTED, "n = %lld needs %d CTA shares; the grid-wide L-BFGS kernel holds at most %d",
                             (long long)n, 8 * o->nblocks, kGridOwnMax * o->nclusters));
        if (cudaMalloc((void**)&o->part, grid_part_bytes()) != cudaSuccess || grid_part_init(o->part, g_tuning.grid_ll, g_tuning.grid_ll_backoff, (unsigned)g_tuning.grid_ll_first_seq) != cudaSuccess ||
            cudaMalloc((void**)&o->fpart, sizeof(unsigned) * 2 * kGridMaxParts) != cudaSuccess)
            return bail(fail(DZO_ERR_ALLOC, "cudaMalloc failed"));
        o->use_grid = true;
    }
    int rc = lbfgs_launch(o, 1, 0, initial_step_length);
    if (rc) return bail(rc);
    if (cudaStreamSynchronize(o->stream) != cudaSuccess)
        return bail(fail(DZO_ERR_CUDA, "constructor kernel failed: %s", cudaGetErrorString(cudaGetLastError())));
    *out = o;
    return DZO_OK;
}

int dzo_lbfgs_create_batched(dzo_lbfgs** out, int objective, int constraint, int64_t obj_param, int64_t n, int64_t batch,
                             const double* x0, double initial_step_length, int history_length, int device) {
    if (!out || !x0) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    *out = nullptr;
    DZO_TRY(check_problem(objective, constraint, obj_param, n, batch));
    if (objective != DZO_OBJ_ROSENBROCK)
        return fail(DZO_ERR_UNSUPPORTED, "batched LBFGSOptimizer device objective: DZO_OBJ_ROSENBROCK");
    if (n > DZO_SMALL_N_MAX) return fail(DZO_ERR_UNSUPPORTED, "batched LBFGSOptimizer needs n <= %d, got %lld", DZO_SMALL_N_MAX, (long long)n);
    if (history_length < 1 || history_length > DZO_LBFGS_MAX_HISTORY)
        return fail(DZO_ERR_INVALID_ARGUMENT, "history_length must be in [1, %d]", DZO_LBFGS_MAX_HISTORY);
    if (!(initial_step_length > 0.0)) return fail(DZO_ERR_INVALID_ARGUMENT, "initial_step_length must be positive");   // :375
    DZO_TRY(use_device(device));
    dzo_lbfgs* o = new (std::nothrow) dzo_lbfgs();
    if (!o) return fail(DZO_ERR_ALLOC, "out of memory");
    o->device = device; o->n = n; o->m = history_length; o->batch = batch;
    o->threads = g_tuning.lbfgs_batched_threads;
    o->ctas = (int)((batch + o->threads - 1) / o->threads);
    o->smem = (size_t)history_length * o->threads * sizeof(double);
    auto bail = [&](int code) { free_lbfgs(o); return code; };
    if (cudaStreamCreateWithFlags(&o->own_stream, cudaStreamNonBlocking) != cudaSuccess)
        return bail(fail(DZO_ERR_CUDA, "cudaStreamCreate failed"));
    o->stream = o->own_stream;
    const size_t vb = (size_t)n * (size_t)batch * 8, hb = vb * (size_t)history_length, sb = (size_t)batch;
    struct { void** p; size_t bytes; } allocs[] = {
        {(void**)&o->x, vb}, {(void**)&o->dx, vb}, {(void**)&o->g, vb}, {(void**)&o->dg, vb}, {(void**)&o->d, vb},
        {(void**)&o->scratch, vb}, {(void**)&o->S, hb}, {(void**)&o->Y, hb}, {(void**)&o->rho, sb * 8 * history_length},
        {(void**)&o->f, sb * 8}, {(void**)&o->df, sb * 8}, {(void**)&o->iter, sb * 8}, {(void**)&o->count, sb * 4},
        {(void**)&o->head, sb * 4}, {(void**)&o->stuck, sb}};
    for (auto& a : allocs)
        if (cudaMalloc(a.p, a.bytes) != cudaSuccess) {
            cudaGetLastError();
            return bail(fail(DZO_ERR_ALLOC, "cudaMalloc(%zu) failed", a.bytes));
        }
    const void* kernel = batched_lbfgs_kernel_ptr((int)n);
    if (o->smem > 48 * 1024 &&
        cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)o->smem) != cudaSuccess)
        return bail(fail(DZO_ERR_CUDA, "the batched L-BFGS kernel cannot get %zu bytes of shared memory", o->smem));
    if (cudaMemcpyAsync(o->scratch, x0, vb, cudaMemcpyHostToDevice, o->stream) != cudaSuccess ||
        batched_lbfgs_transpose(o->scratch, o->x, (int)n, batch, 0, o->stream) != cudaSuccess)
        return bail(fail(DZO_ERR_CUDA, "initial copies failed"));
    int rc = lbfgs_launch(o, 1, 0, initial_step_length);
    if (rc) return bail(rc);
    if (cudaStreamSynchronize(o->stream) != cudaSuccess)
        return bail(fail(DZO_ERR_CUDA, "constructor kernel failed: %s", cudaGetErrorString(cudaGetLastError())));
    *out = o;
    return DZO_OK;
}

void dzo_lbfgs_destroy(dzo_lbfgs* o) { free_lbfgs(o); }

int dzo_lbfgs_set_stream(dzo_lbfgs* o, void* cuda_stream) {
    if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");
    DZO_TRY(use_device(o->device));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    o->stream = cuda_stream ? (cudaStream_t)cuda_stream : o->own_stream;
    return DZO_OK;
}
int dzo_lbfgs_step_async(dzo_lbfgs* o, int k) {
    if (!o || k < 0) return fail(DZO_ERR_INVALID_ARGUMENT, "bad arguments");
    DZO_TRY(use_device(o->device));
    if (k == 0) return DZO_OK;
    return lbfgs_launch(o, 0, k, 0.0);
}
int dzo_lbfgs_sync(dzo_lbfgs* o) {
    if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");
    DZO_TRY(use_device(o->device));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    return DZO_OK;
}
int dzo_lbfgs_step(dzo_lbfgs* o, int k) {
    DZO_TRY(dzo_lbfgs_step_async(o, k));
    return dzo_lbfgs_sync(o);
}

static int lb_read(dzo_lbfgs* o, void* dst, const void* src, size_t bytes) {
    if (!o || !dst) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    DZO_TRY(use_device(o->device));
    DZO_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, o->stream));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    return DZO_OK;
}
// a batched handle transposes its n x batch vectors into the public column-major layout on the way out
static int lb_read_vec(dzo_lbfgs* o, double* out, const double* field) {
    if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");
    if (!o->batch) return lb_read(o, out, field, (size_t)o->n * 8);
    if (!out) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    DZO_TRY(use_device(o->device));
    DZO_CUDA(batched_lbfgs_transpose(field, o->scratch, (int)o->n, o->batch, 1, o->stream));
    return lb_read(o, out, o->scratch, (size_t)o->n * (size_t)o->batch * 8);
}
#define DZO_LB_VEC(name, field)                                                   \
    int name(dzo_lbfgs* o, double* out) {                                         \
        return lb_read_vec(o, out, o ? o->field : nullptr);                       \
    }
DZO_LB_VEC(dzo_lbfgs_get_point, x)
DZO_LB_VEC(dzo_lbfgs_get_delta_point, dx)
DZO_LB_VEC(dzo_lbfgs_get_gradient, g)
DZO_LB_VEC(dzo_lbfgs_get_delta_gradient, dg)
DZO_LB_VEC(dzo_lbfgs_get_direction, d)
#undef DZO_LB_VEC
// batched handles: `batch` values straight from the per-problem array
#define DZO_LB_SCALAR(name, type, expr, array)                                    \
    int name(dzo_lbfgs* o, type* out) {                                           \
        if (!o || !out) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");    \
        if (o->batch) return lb_read(o, out, o->array, (size_t)o->batch * sizeof(type)); \
        LbfgsCtrl c;                                                              \
        DZO_TRY(lb_read(o, &c, o->ctrl, sizeof c));                               \
        *out = (type)(expr);                                                      \
        return DZO_OK;                                                            \
    }
DZO_LB_SCALAR(dzo_lbfgs_get_objective, double, c.f, f)
DZO_LB_SCALAR(dzo_lbfgs_get_delta_objective, double, c.df, df)
DZO_LB_SCALAR(dzo_lbfgs_get_iteration_count, int64_t, c.iter, iter)
DZO_LB_SCALAR(dzo_lbfgs_get_stuck, uint8_t, c.stuck != 0, stuck)
#undef DZO_LB_SCALAR

int dzo_lbfgs_info(dzo_lbfgs* o, int64_t* n, int* order, int* clusters) {
    if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");
    if (n) *n = o->n;
    if (o->batch) {
        if (order) *order = DZO_ORDER_SEQUENTIAL;
        if (clusters) *clusters = o->ctas;
        return DZO_OK;
    }
    if (order) *order = DZO_ORDER_TREE_BLOCKED;          // == DZO_ORDER_TREE for n <= DZO_TREE_BLOCK
    if (clusters) *clusters = o->use_grid ? o->nclusters : kClusterCtas;
    return DZO_OK;
}
int dzo_lbfgs_get_rho_history(dzo_lbfgs* o, int64_t* count, double* rho) {
    if (!o || !count || !rho) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    if (o->batch) {
        // column p: the count[p] entries of problem p newest first, zero-padded to DZO_LBFGS_MAX_HISTORY
        const size_t B = (size_t)o->batch;
        double* r = new (std::nothrow) double[B * o->m];
        int* ch = new (std::nothrow) int[2 * B];
        if (!r || !ch) { delete[] r; delete[] ch; return fail(DZO_ERR_ALLOC, "out of memory"); }
        int rc = lb_read(o, r, o->rho, B * o->m * 8);
        if (!rc) rc = lb_read(o, ch, o->count, B * 4);
        if (!rc) rc = lb_read(o, ch + B, o->head, B * 4);
        if (!rc)
            for (size_t p = 0; p < B; ++p) {
                count[p] = ch[p];
                for (int i = 0; i < DZO_LBFGS_MAX_HISTORY; ++i)
                    rho[p * DZO_LBFGS_MAX_HISTORY + i] = (i < ch[p]) ? r[((ch[B + p] + i) % o->m) * B + p] : 0.0;
            }
        delete[] r; delete[] ch;
        return rc;
    }
    LbfgsCtrl c;
    DZO_TRY(lb_read(o, &c, o->ctrl, sizeof c));
    *count = c.count;
    for (int i = 0; i < DZO_LBFGS_MAX_HISTORY; ++i) rho[i] = (i < c.count) ? c.rho[(c.head + i) % o->m] : 0.0;   // newest first
    return DZO_OK;
}

}  // extern "C"

// ============================================================================= AdGDOptimizer (src/DZOptimization.jl:179-312)
struct dzo_adgd {
    int device = 0;
    cudaStream_t stream = nullptr;
    int64_t n = 0;
    double *x = nullptr, *dx = nullptr, *g = nullptr, *dg = nullptr;
    AdgdCtrl* ctrl = nullptr;
    // n > DZO_TREE_BLOCK: cooperative grid (grid_adgd_kernel)
    int nblocks = 0, nctas = 0;
    double* part = nullptr;
    unsigned* fpart = nullptr;
};
static void free_adgd(dzo_adgd* o) {
    if (!o) return;
    cudaSetDevice(o->device);
    void* ptrs[] = {o->x, o->dx, o->g, o->dg, o->ctrl, o->part, o->fpart};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (o->stream) cudaStreamDestroy(o->stream);
    delete o;
}
static int adgd_launch(dzo_adgd* o, int mode, int k, double L0) {
    AdgdArgs a;
    a.x = o->x; a.dx = o->dx; a.g = o->g; a.dg = o->dg; a.ctrl = o->ctrl; a.n = o->n; a.ksteps = k; a.mode = mode;
    a.initial_step_length = L0;
    if (o->nblocks > 1) {
        GridAdgdArgs ga;
        ga.a = a; ga.part = o->part; ga.fpart = o->fpart; ga.nblocks = o->nblocks;
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof cfg);
        cfg.gridDim = dim3((unsigned)o->nctas);
        cfg.blockDim = dim3(kClusterThreads);
        cfg.stream = o->stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeCooperative;
        attr[0].val.cooperative = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        void* params[] = {&ga};
        DZO_CUDA(cudaLaunchKernelExC(&cfg, grid_adgd_kernel_ptr(), params));
        return DZO_OK;
    }
    cluster_adgd_kernel<<<kClusterCtas, kClusterThreads, 0, o->stream>>>(a);
    DZO_CUDA(cudaGetLastError());
    return DZO_OK;
}
extern "C" {
int dzo_adgd_create(dzo_adgd** out, int objective, int constraint, int64_t obj_param, int64_t n, const double* x0,
                    double initial_step_length, int device) {
    if (!out || !x0) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    *out = nullptr;
    DZO_TRY(check_problem(objective, constraint, obj_param, n, 1));
    if (objective != DZO_OBJ_ROSENBROCK) return fail(DZO_ERR_UNSUPPORTED, "AdGDOptimizer device objective: DZO_OBJ_ROSENBROCK");
    if (!(initial_step_length > 0.0)) return fail(DZO_ERR_INVALID_ARGUMENT, "initial_step_length must be positive");   // :232
    DZO_TRY(use_device(device));
    dzo_adgd* o = new (std::nothrow) dzo_adgd();
    if (!o) return fail(DZO_ERR_ALLOC, "out of memory");
    o->device = device; o->n = n;
    auto bail = [&](int code) { free_adgd(o); return code; };
    if (cudaStreamCreateWithFlags(&o->stream, cudaStreamNonBlocking) != cudaSuccess) return bail(fail(DZO_ERR_CUDA, "cudaStreamCreate failed"));
    double** vecs[] = {&o->x, &o->dx, &o->g, &o->dg};
    for (double** v : vecs)
        if (cudaMalloc((void**)v, (size_t)n * 8) != cudaSuccess) return bail(fail(DZO_ERR_ALLOC, "cudaMalloc failed"));
    if (cudaMalloc((void**)&o->ctrl, sizeof(AdgdCtrl)) != cudaSuccess) return bail(fail(DZO_ERR_ALLOC, "cudaMalloc failed"));
    if (cudaMemcpyAsync(o->x, x0, (size_t)n * 8, cudaMemcpyHostToDevice, o->stream) != cudaSuccess)
        return bail(fail(DZO_ERR_CUDA, "H2D copy failed"));
    o->nblocks = (int)((n + DZO_TREE_BLOCK - 1) / DZO_TREE_BLOCK);
    if (o->nblocks > 1) {
        int per_sm = 0, sms = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)grid_adgd_kernel_ptr(), kClusterThreads, 0) != cudaSuccess ||
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || per_sm < 1 || sms < 1) {
            cudaGetLastError();
            return bail(fail(DZO_ERR_CUDA, "the grid-wide AdGD kernel does not fit on this device"));
        }
        const int resident = per_sm * sms;
        o->nctas = 8 * o->nblocks < resident ? 8 * o->nblocks : resident;
        if (o->nblocks > kGridMaxBlocks || 8 * o->nblocks > kGridOwnMax * o->nctas)
            return bail(fail(DZO_ERR_UNSUPPORTED, "n = %lld is too large for the grid-wide AdGD kernel", (long long)n));
        if (cudaMalloc((void**)&o->part, grid_part_bytes()) != cudaSuccess || grid_part_init(o->part, g_tuning.grid_ll, g_tuning.grid_ll_backoff, (unsigned)g_tuning.grid_ll_first_seq) != cudaSuccess ||
            cudaMalloc((void**)&o->fpart, sizeof(unsigned) * 2 * kGridMaxParts) != cudaSuccess)
            return bail(fail(DZO_ERR_ALLOC, "cudaMalloc failed"));
    }
    int rc = adgd_launch(o, 1, 0, initial_step_length);
    if (rc) return bail(rc);
    if (cudaStreamSynchronize(o->stream) != cudaSuccess) return bail(fail(DZO_ERR_CUDA, "constructor kernel failed"));
    *out = o;
    return DZO_OK;
}
void dzo_adgd_destroy(dzo_adgd* o) { free_adgd(o); }
int dzo_adgd_step(dzo_adgd* o, int k) {
    if (!o || k < 0) return fail(DZO_ERR_INVALID_ARGUMENT, "bad arguments");
    DZO_TRY(use_device(o->device));
    if (k > 0) DZO_TRY(adgd_launch(o, 0, k, 0.0));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    return DZO_OK;
}
static int ad_read(dzo_adgd* o, void* dst, const void* src, size_t bytes) {
    if (!o || !dst) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    DZO_TRY(use_device(o->device));
    DZO_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, o->stream));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    return DZO_OK;
}
int dzo_adgd_get_point(dzo_adgd* o, double* out) { return o ? ad_read(o, out, o->x, (size_t)o->n * 8) : fail(DZO_ERR_INVALID_ARGUMENT, "null handle"); }
int dzo_adgd_get_delta_point(dzo_adgd* o, double* out) { return o ? ad_read(o, out, o->dx, (size_t)o->n * 8) : fail(DZO_ERR_INVALID_ARGUMENT, "null handle"); }
int dzo_adgd_get_gradient(dzo_adgd* o, double* out) { return o ? ad_read(o, out, o->g, (size_t)o->n * 8) : fail(DZO_ERR_INVALID_ARGUMENT, "null handle"); }
int dzo_adgd_get_delta_gradient(dzo_adgd* o, double* out) { return o ? ad_read(o, out, o->dg, (size_t)o->n * 8) : fail(DZO_ERR_INVALID_ARGUMENT, "null handle"); }
int dzo_adgd_get_scalars(dzo_adgd* o, double* s) {
    if (!o || !s) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    AdgdCtrl c;
    DZO_TRY(ad_read(o, &c, o->ctrl, sizeof c));
    s[0] = c.f; s[1] = c.df; s[2] = c.cur; s[3] = c.prev; s[4] = (double)c.iter; s[5] = (double)c.stuck;
    return DZO_OK;
}
}  // extern "C"

// ============================================================================= legacy LBFGSOptimizer (legacy/DZOptimization.jl:458-695)
struct dzo_legacy_lbfgs {
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    int64_t n = 0;
    int m = 0, max_increases = 0, decor = 0;
    double l2 = 0.0, lo = 0.0, hi = 0.0;
    double *x = nullptr, *dx = nullptr, *g = nullptr, *dg = nullptr, *d = nullptr, *S = nullptr, *Y = nullptr;
    LegacyCtrl* ctrl = nullptr;
    // n > DZO_TREE_BLOCK: cooperative grid, eight CTAs per block (grid_legacy_lbfgs.cuh)
    bool use_grid = false;
    int nblocks = 0, nctas = 0;
    double* part = nullptr;
    unsigned* fpart = nullptr;
};
static void free_legacy(dzo_legacy_lbfgs* o) {
    if (!o) return;
    cudaSetDevice(o->device);
    void* ptrs[] = {o->x, o->dx, o->g, o->dg, o->d, o->S, o->Y, o->ctrl, o->part, o->fpart};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (o->own_stream) cudaStreamDestroy(o->own_stream);
    delete o;
}
static int legacy_launch(dzo_legacy_lbfgs* o, int mode, int k, double L0) {
    LegacyArgs a;
    a.x = o->x; a.dx = o->dx; a.g = o->g; a.dg = o->dg; a.d = o->d; a.S = o->S; a.Y = o->Y; a.ctrl = o->ctrl;
    a.n = o->n; a.m = o->m; a.ksteps = k; a.max_increases = o->max_increases; a.mode = mode; a.decor = o->decor;
    a.initial_step_length = L0; a.l2 = o->l2; a.lo = o->lo; a.hi = o->hi; a.algo = 0;
    if (o->use_grid) {
        GridLegacyArgs ga;
        ga.a = a; ga.part = o->part; ga.fpart = o->fpart; ga.nblocks = o->nblocks;
        const bool own1 = (8 * o->nblocks <= o->nctas);
        ga.stage = (own1 && g_tuning.grid_stage) ? 1 : 0;
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof cfg);
        cfg.gridDim = dim3((unsigned)o->nctas);
        cfg.blockDim = dim3(kClusterThreads);
        cfg.dynamicSmemBytes = ga.stage ? kGridStageBytes : 0;
        cfg.stream = o->stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeCooperative;
        attr[0].val.cooperative = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        void* params[] = {&ga};
        DZO_CUDA(cudaLaunchKernelExC(&cfg, grid_legacy_kernel_ptr(8 * o->nblocks <= o->nctas ? 1 : kGridOwnMax), params));
        return DZO_OK;
    }
    cluster_legacy_lbfgs_kernel<<<kClusterCtas, kClusterThreads, 0, o->stream>>>(a);
    DZO_CUDA(cudaGetLastError());
    return DZO_OK;
}
extern "C" {
int dzo_legacy_lbfgs_create(dzo_legacy_lbfgs** out, int objective, int constraint, int64_t obj_param, int64_t n,
                            const double* x0, double initial_step_length, int history_length, int max_increases,
                            int decor, double l2_lambda, double box_lower, double box_upper, int device) {
    if (!out || !x0) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    *out = nullptr;
    DZO_TRY(check_problem(objective, constraint, obj_param, n, 1));
    if (objective != DZO_OBJ_ROSENBROCK) return fail(DZO_ERR_UNSUPPORTED, "legacy LBFGSOptimizer device objective: DZO_OBJ_ROSENBROCK");
    if (decor & ~(DZO_DECOR_L2 | DZO_DECOR_BOX)) return fail(DZO_ERR_INVALID_ARGUMENT, "unknown decorator bits");
    if ((decor & DZO_DECOR_L2) && l2_lambda != l2_lambda) return fail(DZO_ERR_INVALID_ARGUMENT, "lambda is NaN");
    if ((decor & DZO_DECOR_BOX) && !(box_lower <= box_upper)) return fail(DZO_ERR_INVALID_ARGUMENT, "box needs lower_bound <= upper_bound");
    if (history_length < 1 || history_length > DZO_LBFGS_MAX_HISTORY)                            // :528
        return fail(DZO_ERR_INVALID_ARGUMENT, "history_length must be in [1, %d]", DZO_LBFGS_MAX_HISTORY);
    DZO_TRY(use_device(device));
    dzo_legacy_lbfgs* o = new (std::nothrow) dzo_legacy_lbfgs();
    if (!o) return fail(DZO_ERR_ALLOC, "out of memory");
    o->device = device; o->n = n; o->m = history_length; o->max_increases = max_increases; o->decor = decor;
    o->l2 = l2_lambda; o->lo = box_lower; o->hi = box_upper;
    auto bail = [&](int code) { free_legacy(o); return code; };
    if (cudaStreamCreateWithFlags(&o->own_stream, cudaStreamNonBlocking) != cudaSuccess)
        return bail(fail(DZO_ERR_CUDA, "cudaStreamCreate failed"));
    o->stream = o->own_stream;
    const size_t vb = (size_t)n * 8;
    double** vecs[] = {&o->x, &o->dx, &o->g, &o->dg, &o->d};
    for (double** v : vecs)
        if (cudaMalloc((void**)v, vb) != cudaSuccess) return bail(fail(DZO_ERR_ALLOC, "cudaMalloc failed"));
    if (cudaMalloc((void**)&o->S, vb * history_length) != cudaSuccess || cudaMalloc((void**)&o->Y, vb * history_length) != cudaSuccess ||
        cudaMalloc((void**)&o->ctrl, sizeof(LegacyCtrl)) != cudaSuccess)
        return bail(fail(DZO_ERR_ALLOC, "cudaMalloc failed"));
    if (cudaMemcpyAsync(o->x, x0, vb, cudaMemcpyHostToDevice, o->stream) != cudaSuccess ||
        cudaMemsetAsync(o->S, 0, vb * history_length, o->stream) != cudaSuccess ||
        cudaMemsetAsync(o->Y, 0, vb * history_length, o->stream) != cudaSuccess)
        return bail(fail(DZO_ERR_CUDA, "initial copies failed"));
    if (n > DZO_TREE_BLOCK) {
        o->nblocks = (int)((n + DZO_TREE_BLOCK - 1) / DZO_TREE_BLOCK);
        int per_sm = 0, sms = 0;
        int per_sm_one = 0;               // OWN = 1 or kGridOwnMax is picked at launch: size the grid for the tighter of the two
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)grid_legacy_kernel_ptr(kGridOwnMax), kClusterThreads, 0) != cudaSuccess ||
            cudaFuncSetAttribute((const void*)grid_legacy_kernel_ptr(1), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGridStageBytes) != cudaSuccess ||
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_one, (const void*)grid_legacy_kernel_ptr(1), kClusterThreads, kGridStageBytes) != cudaSuccess ||
            (per_sm = per_sm < per_sm_one ? per_sm : per_sm_one) < 0 ||
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || per_sm < 1 || sms < 1) {
            cudaGetLastError();
            return bail(fail(DZO_ERR_CUDA, "the grid-wide legacy L-BFGS kernel does not fit on this device"));
        }
        const int resident = per_sm * sms;
        o->nctas = 8 * o->nblocks < resident ? 8 * o->nblocks : resident;
        if (o->nblocks > kGridMaxBlocks || 8 * o->nblocks > kGridOwnMax * o->nctas)
            return bail(fail(DZO_ERR_UNSUPPORTED, "n = %lld needs %d CTA shares; the grid-wide legacy L-BFGS kernel holds at most %d",
                             (long long)n, 8 * o->nblocks, kGridOwnMax * o->nctas));
        if (cudaMalloc((void**)&o->part, grid_part_bytes()) != cudaSuccess || grid_part_init(o->part, g_tuning.grid_ll, g_tuning.grid_ll_backoff, (unsigned)g_tuning.grid_ll_first_seq) != cudaSuccess ||
            cudaMalloc((void**)&o->fpart, sizeof(unsigned) * 2 * kGridMaxParts) != cudaSuccess)
            return bail(fail(DZO_ERR_ALLOC, "cudaMalloc failed"));
        o->use_grid = true;
    }
    int rc = legacy_launch(o, 1, 0, initial_step_length);
    if (rc) return bail(rc);
    if (cudaStreamSynchronize(o->stream) != cudaSuccess)
        return bail(fail(DZO_ERR_CUDA, "constructor kernel failed: %s", cudaGetErrorString(cudaGetLastError())));
    *out = o;
    return DZO_OK;
}
void dzo_legacy_lbfgs_destroy(dzo_legacy_lbfgs* o) { free_legacy(o); }
int dzo_legacy_lbfgs_set_stream(dzo_legacy_lbfgs* o, void* cuda_stream) {
    if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");
    DZO_TRY(use_device(o->device));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    o->stream = cuda_stream ? (cudaStream_t)cuda_stream : o->own_stream;
    return DZO_OK;
}
int dzo_legacy_lbfgs_step_async(dzo_legacy_lbfgs* o, int k) {
    if (!o || k < 0) return fail(DZO_ERR_INVALID_ARGUMENT, "bad arguments");
    DZO_TRY(use_device(o->device));
    if (k == 0) return DZO_OK;
    return legacy_launch(o, 0, k, 0.0);
}
int dzo_legacy_lbfgs_sync(dzo_legacy_lbfgs* o) {
    if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");
    DZO_TRY(use_device(o->device));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    return DZO_OK;
}
int dzo_legacy_lbfgs_step(dzo_legacy_lbfgs* o, int k) {
    DZO_TRY(dzo_legacy_lbfgs_step_async(o, k));
    return dzo_legacy_lbfgs_sync(o);
}
static int lg_read(dzo_legacy_lbfgs* o, void* dst, const void* src, size_t bytes) {
    if (!o || !dst) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    DZO_TRY(use_device(o->device));
    DZO_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, o->stream));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    return DZO_OK;
}
#define DZO_LG_VEC(name, field)                                                   \
    int name(dzo_legacy_lbfgs* o, double* out) {                                  \
        if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");             \
        return lg_read(o, out, o->field, (size_t)o->n * 8);                       \
    }
DZO_LG_VEC(dzo_legacy_lbfgs_get_point, x)
DZO_LG_VEC(dzo_legacy_lbfgs_get_delta_point, dx)
DZO_LG_VEC(dzo_legacy_lbfgs_get_gradient, g)
DZO_LG_VEC(dzo_legacy_lbfgs_get_delta_gradient, dg)
DZO_LG_VEC(dzo_legacy_lbfgs_get_direction, d)
#undef DZO_LG_VEC
int dzo_legacy_lbfgs_get_scalars(dzo_legacy_lbfgs* o, double* s) {
    if (!o || !s) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    LegacyCtrl c;
    DZO_TRY(lg_read(o, &c, o->ctrl, sizeof c));
    s[0] = c.f; s[1] = c.df; s[2] = c.L; s[3] = (double)c.iter; s[4] = (double)(c.term != 0); s[5] = (double)c.hist_count;
    return DZO_OK;
}
int dzo_legacy_lbfgs_get_history(dzo_legacy_lbfgs* o, double* rho, double* alpha) {
    if (!o || !rho || !alpha) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    LegacyCtrl c;
    DZO_TRY(lg_read(o, &c, o->ctrl, sizeof c));
    for (int i = 0; i < o->m; ++i) { rho[i] = c.rho[i]; alpha[i] = c.alpha[i]; }
    return DZO_OK;
}
}  // extern "C"

// ============================================================================= live LineSearchEvaluator (src/DZOptimization.jl:12-92)
extern "C" int dzo_dev_line_search_evaluate(int objective, int constraint, int64_t obj_param, int order, int64_t n,
                                            const double* x, double f_old, const double* dir, double overlap,
                                            double step_size, int compute_gradient, double* trial_point,
                                            double* trial_gradient, double* results3, int device) {
    if (!x || !dir || !trial_point || !results3 || (compute_gradient && !trial_gradient))
        return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    DZO_TRY(check_problem(objective, constraint, obj_param, n, 1));
    if (objective != DZO_OBJ_ROSENBROCK) return fail(DZO_ERR_UNSUPPORTED, "LineSearchEvaluator device objective: DZO_OBJ_ROSENBROCK");
    if (order != DZO_ORDER_TREE) return fail(DZO_ERR_UNSUPPORTED, "device LineSearchEvaluator computes in DZO_ORDER_TREE");
    DZO_TRY(use_device(device));
    DevBuf dx, dd, dt, dg, dout;
    const size_t vb = (size_t)n * 8;
    DZO_TRY(dx.alloc(vb)); DZO_TRY(dd.alloc(vb)); DZO_TRY(dt.alloc(vb)); DZO_TRY(dg.alloc(vb)); DZO_TRY(dout.alloc(24));
    DZO_CUDA(cudaMemcpy(dx.p, x, vb, cudaMemcpyHostToDevice));
    DZO_CUDA(cudaMemcpy(dd.p, dir, vb, cudaMemcpyHostToDevice));
    LseArgs a;
    a.x = dx.as<double>(); a.dir = dd.as<double>(); a.trial = dt.as<double>(); a.trial_g = dg.as<double>();
    a.out3 = dout.as<double>(); a.n = n; a.f_old = f_old; a.overlap = overlap; a.step = step_size;
    a.compute_gradient = compute_gradient ? 1 : 0;
    cluster_lse_kernel<<<kClusterCtas, kClusterThreads>>>(a);
    DZO_CUDA(cudaGetLastError());
    DZO_CUDA(cudaDeviceSynchronize());
    DZO_CUDA(cudaMemcpy(trial_point, dt.p, vb, cudaMemcpyDeviceToHost));
    if (compute_gradient) DZO_CUDA(cudaMemcpy(trial_gradient, dg.p, vb, cudaMemcpyDeviceToHost));
    DZO_CUDA(cudaMemcpy(results3, dout.p, 24, cudaMemcpyDeviceToHost));
    return DZO_OK;
}


// ============================================================================= GradientDescentOptimizer, Rosenbrock, n > DZO_TREE_BLOCK
// (hook used by dzopt_gd.cu: the grid-wide legacy kernel with algo = 1)
namespace dzo {
struct GridGd {
    int nblocks = 0, nctas = 0;
    double* part = nullptr;
    unsigned* fpart = nullptr;
    LegacyCtrl* lctrl = nullptr;
    double* scal = nullptr;      // { f, df, L, iteration_count, has_terminated, evals } for the getters of dzopt_gd.cu
};
static __global__ void grid_gd_publish_kernel(const LegacyCtrl* c, double* s) {
    s[0] = c->f; s[1] = c->df; s[2] = c->L; s[3] = (double)c->iter; s[4] = (double)(c->term != 0); s[5] = (double)c->evals;
}
void grid_gd_detach(void* p) {
    GridGd* h = static_cast<GridGd*>(p);
    if (!h) return;
    void* ptrs[] = {h->part, h->fpart, h->lctrl, h->scal};
    for (void* q : ptrs)
        if (q) cudaFree(q);
    delete h;
}
int grid_gd_attach(int64_t n, int device, void** out, double** scal) {
    *out = nullptr;
    GridGd* h = new (std::nothrow) GridGd();
    if (!h) return fail(DZO_ERR_ALLOC, "out of memory");
    h->nblocks = (int)((n + DZO_TREE_BLOCK - 1) / DZO_TREE_BLOCK);
    if (h->nblocks == 1) {       // one block: the 8-CTA cluster kernel (DSMEM reductions), no grid-wide scratch
        if (cudaMalloc((void**)&h->lctrl, sizeof(LegacyCtrl)) != cudaSuccess || cudaMalloc((void**)&h->scal, 6 * sizeof(double)) != cudaSuccess) {
            grid_gd_detach(h);
            return fail(DZO_ERR_ALLOC, "cudaMalloc failed");
        }
        *out = h;
        *scal = h->scal;
        return DZO_OK;
    }
    int per_sm = 0, sms = 0;
    int per_sm_one = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)grid_legacy_kernel_ptr(kGridOwnMax), kClusterThreads, 0) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_one, (const void*)grid_legacy_kernel_ptr(1), kClusterThreads, 0) != cudaSuccess ||
        (per_sm = per_sm < per_sm_one ? per_sm : per_sm_one) < 0 ||
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || per_sm < 1 || sms < 1) {
        cudaGetLastError();
        delete h;
        return fail(DZO_ERR_CUDA, "the grid-wide GD kernel does not fit on this device");
    }
    const int resident = per_sm * sms;
    h->nctas = 8 * h->nblocks < resident ? 8 * h->nblocks : resident;
    if (h->nblocks > kGridMaxBlocks || 8 * h->nblocks > kGridOwnMax * h->nctas) {
        delete h;
        return fail(DZO_ERR_UNSUPPORTED, "n = %lld is too large for the grid-wide GD kernel", (long long)n);
    }
    if (cudaMalloc((void**)&h->part, grid_part_bytes()) != cudaSuccess || grid_part_init(h->part, g_tuning.grid_ll, g_tuning.grid_ll_backoff, (unsigned)g_tuning.grid_ll_first_seq) != cudaSuccess ||
        cudaMalloc((void**)&h->fpart, sizeof(unsigned) * 2 * kGridMaxParts) != cudaSuccess ||
        cudaMalloc((void**)&h->lctrl, sizeof(LegacyCtrl)) != cudaSuccess || cudaMalloc((void**)&h->scal, 6 * sizeof(double)) != cudaSuccess) {
        grid_gd_detach(h);
        return fail(DZO_ERR_ALLOC, "cudaMalloc failed");
    }
    *out = h;
    *scal = h->scal;
    return DZO_OK;
}
int grid_gd_launch(void* p, int mode, int k, cudaStream_t stream, double* x, double* dx, double* g, double* dg, double* d,
                   int64_t n, int max_increases, double L0) {
    GridGd* h = static_cast<GridGd*>(p);
    GridLegacyArgs ga;
    memset(&ga, 0, sizeof ga);
    ga.a.x = x; ga.a.dx = dx; ga.a.g = g; ga.a.dg = dg; ga.a.d = d; ga.a.S = nullptr; ga.a.Y = nullptr;   // no history in GD mode
    ga.a.ctrl = h->lctrl; ga.a.n = n; ga.a.m = 1; ga.a.ksteps = k; ga.a.max_increases = max_increases; ga.a.mode = mode;
    ga.a.decor = 0; ga.a.algo = 1; ga.a.initial_step_length = L0;
    ga.part = h->part; ga.fpart = h->fpart; ga.nblocks = h->nblocks;
    if (h->nblocks == 1) {
        cluster_legacy_lbfgs_kernel<<<kClusterCtas, kClusterThreads, 0, stream>>>(ga.a);
        DZO_CUDA(cudaGetLastError());
        grid_gd_publish_kernel<<<1, 1, 0, stream>>>(h->lctrl, h->scal);
        DZO_CUDA(cudaGetLastError());
        return DZO_OK;
    }
    ga.stage = 0;                              // (GD has no history passes to stage)
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3((unsigned)h->nctas);
    cfg.blockDim = dim3(kClusterThreads);
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    void* params[] = {&ga};
    DZO_CUDA(cudaLaunchKernelExC(&cfg, grid_legacy_kernel_ptr(8 * h->nblocks <= h->nctas ? 1 : kGridOwnMax), params));
    grid_gd_publish_kernel<<<1, 1, 0, stream>>>(h->lctrl, h->scal);
    DZO_CUDA(cudaGetLastError());
    return DZO_OK;
}
}  // namespace dzo
