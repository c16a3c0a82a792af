// dzopt_gd.cu -- C ABI of the GradientDescentOptimizer path (legacy/DZOptimization.jl:305-449) and the
// Riesz-energy device objectives (legacy/ExampleFunctions.jl:30-83).  sm_100a only; -fmad=false.
#include <new>
#include <vector>

#include "gd_batched.cuh"
#include "gd_kernels.cuh"
#include "host_common.h"

using namespace dzo;

// GradientDescentOptimizer for extended Rosenbrock, n > 32, on the legacy L-BFGS kernels with algo = 1 (dzopt_lbfgs.cu)
namespace dzo {
int grid_gd_attach(int64_t n, int device, void** out, double** scal);
void grid_gd_detach(void* p);
int grid_gd_launch(void* p, int mode, int k, cudaStream_t stream, double* x, double* dx, double* g, double* dg, double* d,
                   int64_t n, int max_increases, double L0);
}

// ============================================================================= handle
struct dzo_gd {
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    int objective = 0, constraint = 0, max_increases = 0;
    int64_t dim = 0, n = 0, batch = 0;
    double *x = nullptr, *g = nullptr, *d = nullptr, *dx = nullptr, *dg = nullptr;
    GdCtrl* ctrl = nullptr;
    // batched small-n path (n <= DZO_SMALL_N_MAX): one thread per problem, SEQUENTIAL order
    bool small = false;
    double *f = nullptr, *df = nullptr, *L = nullptr;
    long long* iter = nullptr;
    unsigned char* term = nullptr;
    // Riesz cooperative kernel
    double *segE = nullptr, *rowE = nullptr, *segG = nullptr, *fbox = nullptr;
    int2* e_items = nullptr;
    int n_e_items = 0;
    unsigned* counter = nullptr;
    unsigned* rbcnt = nullptr;
    unsigned long long* bar = nullptr;
    int esplit = 2, gcnt_off = 0, ecnt_stride = 0, espec = 0;
    int2* g_jobs = nullptr;
    int n_g_jobs = 0, gvariant = 0;
    unsigned long long* prof = nullptr;   // phase log (tuning knob "riesz_profile")
    int grid = 0, nt = 512;
    // Rosenbrock, n > 32: cluster kernel up to n = DZO_TREE_BLOCK, cooperative grid above (DZO_ORDER_TREE_BLOCKED)
    void* gridgd = nullptr;
    double* gscal = nullptr;              // { f, df, L, iteration_count, has_terminated, evals } (owned by gridgd)
};

static void free_gd(dzo_gd* o) {
    if (!o) return;
    cudaSetDevice(o->device);
    void* ptrs[] = {o->x, o->g, o->d, o->dx, o->dg, o->ctrl, o->segE, o->rowE, o->segG, o->fbox, o->e_items, o->counter, o->rbcnt, o->prof, o->g_jobs, o->bar,
                    o->f, o->df, o->L, o->iter, o->term};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (o->gridgd) grid_gd_detach(o->gridgd);
    if (o->own_stream) cudaStreamDestroy(o->own_stream);
    delete o;
}

template <class T>
static int dmalloc(T** p, size_t count) {
    cudaError_t e = cudaMalloc((void**)p, (count ? count : 1) * sizeof(T));
    if (e != cudaSuccess) {
        *p = nullptr;
        return fail(DZO_ERR_ALLOC, "cudaMalloc of %zu bytes failed: %s", count * sizeof(T), cudaGetErrorString(e));
    }
    return DZO_OK;
}

// (row block of `rows` rows, segment of 128 sources) items that contain at least one pair i < j,
// heaviest first so the round-robin over warps stays balanced
// gradient tile jobs (a, b), a <= b over the segments of 128 points: off-diagonal (two families of partials) first
static std::vector<int2> gradient_jobs(int N) {
    const int nseg = (N + DZO_RIESZ_SEG - 1) / DZO_RIESZ_SEG;
    std::vector<int2> jobs;
    for (int a = 0; a < nseg; ++a)
        for (int b = a + 1; b < nseg; ++b) jobs.push_back(make_int2(a, b));
    for (int a = 0; a < nseg; ++a) jobs.push_back(make_int2(a, a));
    return jobs;
}

static std::vector<int2> energy_items(int N, int rows) {
    std::vector<int2> full, diag;
    const int nrb = (N + rows - 1) / rows;
    for (int rb = 0; rb < nrb; ++rb) {
        const int jmax = std::min(N, rb * rows + rows) - 1;
        for (int s = 0; s * DZO_RIESZ_SEG < jmax; ++s) {
            const bool whole = (s + 1) * DZO_RIESZ_SEG <= rb * rows;
            (whole ? full : diag).push_back(make_int2(rb, s));
        }
    }
    full.insert(full.end(), diag.begin(), diag.end());
    return full;
}

// one translation unit per instance (riesz_dim<N>.cu)
namespace dzo {
void* riesz_kernel_dim1(int nt);
void* riesz_kernel_dim2(int nt);
void* riesz_kernel_dim3(int nt);
void* riesz_kernel_dim4(int nt);
}
static void* riesz_kernel_for(int dim, int nt) {
    switch (dim) {
        case 1: return riesz_kernel_dim1(nt);
        case 2: return riesz_kernel_dim2(nt);
        case 3: return riesz_kernel_dim3(nt);
        case 4: return riesz_kernel_dim4(nt);
        default: return nullptr;
    }
}

// Everything the cooperative Riesz kernel needs besides the vectors
struct RieszWork {
    double *segE = nullptr, *rowE = nullptr, *segG = nullptr, *fbox = nullptr;
    int2* e_items = nullptr;
    int n_e_items = 0;
    unsigned* counter = nullptr;
    unsigned* rbcnt = nullptr;
    unsigned long long* bar = nullptr;
    int esplit = 2, gcnt_off = 0, ecnt_stride = 0, espec = 0;
    int2* g_jobs = nullptr;
    int n_g_jobs = 0, gvariant = 0;
    int grid = 0, nt = 512;
    void* kernel = nullptr;
    size_t smem = 0;
    int init(int N, int dim, int device) {
        // threads per CTA: 512 (128 registers: twice the pair terms in flight per lane) unless the symmetric-tile gradient
        // variant, which is written for 32 warps, or the tuning knob asks for the 1024-thread kernel
        nt = (g_tuning.riesz_threads == 1024 || g_tuning.riesz_gvariant) ? 1024 : 512;
        kernel = riesz_kernel_for(dim, nt);
        if (!kernel) return fail(DZO_ERR_UNSUPPORTED, "device Riesz kernels support 1 <= dim <= 4");
        const int nseg = (N + DZO_RIESZ_SEG - 1) / DZO_RIESZ_SEG;
        DZO_TRY(dmalloc(&segE, (size_t)2 * nseg * N));       // two probes of a paired evaluation
        DZO_TRY(dmalloc(&rowE, (size_t)4 * N));              // [phase parity][probe]
        DZO_CUDA(cudaMemset(rowE, 0, (size_t)4 * N * sizeof(double)));
        esplit = (g_tuning.riesz_esplit == 2) ? 2 : 1;   // measured: 2 lanes per row is 11 % slower (the loops are issue-bound, not latency-bound)
        espec = g_tuning.riesz_pair ? 1 : 0;
        ecnt_stride = (N + 15) / 16;
        gcnt_off = 2 * ecnt_stride;
        DZO_TRY(dmalloc(&rbcnt, (size_t)3 * ecnt_stride));   // items finished per row block: energy probe 0 | probe 1 | gradient
        DZO_CUDA(cudaMemset(rbcnt, 0, (size_t)3 * ecnt_stride * sizeof(unsigned)));
        if (g_tuning.riesz_bar) {
            DZO_TRY(dmalloc(&bar, riesz_bar_bytes() / sizeof(unsigned long long)));
            DZO_CUDA(cudaMemset(bar, 0, riesz_bar_bytes()));
        }
        DZO_TRY(dmalloc(&segG, (size_t)nseg * N * dim));
        DZO_TRY(dmalloc(&fbox, 4));
        DZO_TRY(dmalloc(&counter, 1));
        DZO_CUDA(cudaMemset(counter, 0, sizeof(unsigned)));
        std::vector<int2> items = energy_items(N, esplit == 2 ? 16 : 32);
        n_e_items = (int)items.size();
        DZO_TRY(dmalloc(&e_items, items.size()));
        if (!items.empty())
            DZO_CUDA(cudaMemcpy(e_items, items.data(), items.size() * sizeof(int2), cudaMemcpyHostToDevice));
        gvariant = g_tuning.riesz_gvariant ? 1 : 0;
        std::vector<int2> jobs = gradient_jobs(N);
        n_g_jobs = (int)jobs.size();
        DZO_TRY(dmalloc(&g_jobs, jobs.size()));
        if (!jobs.empty())
            DZO_CUDA(cudaMemcpy(g_jobs, jobs.data(), jobs.size() * sizeof(int2), cudaMemcpyHostToDevice));
        smem = riesz_gd_smem(dim, nt);
        DZO_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cudaDeviceProp prop;
        DZO_CUDA(cudaGetDeviceProperties(&prop, device));
        int per_sm = 0;
        DZO_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, nt, smem));
        if (per_sm < 1) return fail(DZO_ERR_CUDA, "riesz_gd_kernel does not fit on an SM");
        if (!prop.cooperativeLaunch) return fail(DZO_ERR_UNSUPPORTED, "device lacks cooperative launch");
        grid = prop.multiProcessorCount;   // one persistent CTA per SM
        return DZO_OK;
    }
    void release() {
        void* ptrs[] = {segE, rowE, segG, fbox, e_items, counter, rbcnt, g_jobs, bar};
        for (void* p : ptrs)
            if (p) cudaFree(p);
        segE = rowE = segG = fbox = nullptr; e_items = nullptr; counter = nullptr; rbcnt = nullptr; g_jobs = nullptr; bar = nullptr;
    }
    void fill(RieszGdArgs& a) const {
        a.segE = segE; a.rowE = rowE; a.segG = segG; a.e_items = e_items; a.n_e_items = n_e_items;
        a.counter = counter; a.fbox = fbox; a.rbcnt = rbcnt; a.dscale = 1.0; a.esplit = esplit; a.gcnt_off = gcnt_off;
        a.ecnt_stride = ecnt_stride; a.espec = espec; a.bar = bar;
        a.g_jobs = g_jobs; a.n_g_jobs = n_g_jobs; a.gvariant = gvariant;
    }
    int launch(RieszGdArgs& a, cudaStream_t stream) const {
        void* params[] = {&a};
        DZO_CUDA(cudaLaunchCooperativeKernel(kernel, dim3(grid), dim3(nt), params, smem, stream));
        return DZO_OK;
    }
};

static RieszGdArgs riesz_args(const dzo_gd* o, int mode, int k) {
    RieszGdArgs a;
    memset(&a, 0, sizeof a);
    a.x = o->x; a.g = o->g; a.d = o->d; a.dx = o->dx; a.dg = o->dg;
    a.segE = o->segE; a.rowE = o->rowE; a.segG = o->segG; a.e_items = o->e_items; a.n_e_items = o->n_e_items;
    a.ctrl = o->ctrl; a.counter = o->counter; a.fbox = o->fbox; a.rbcnt = o->rbcnt; a.dscale = 1.0; a.esplit = o->esplit; a.gcnt_off = o->gcnt_off;
    a.ecnt_stride = o->ecnt_stride; a.espec = o->espec; a.bar = o->bar;
    a.g_jobs = o->g_jobs; a.n_g_jobs = o->n_g_jobs; a.gvariant = o->gvariant;
    a.N = (int)(o->n / o->dim); a.sphere = (o->constraint == DZO_CONSTRAINT_SPHERE); a.max_increases = o->max_increases;
    a.ksteps = k; a.mode = mode;
    return a;
}

static int gd_launch(dzo_gd* o, int mode, int k, double L0) {
    if (o->small) {
        GdBatchedArgs a;
        a.x = o->x; a.dx = o->dx; a.g = o->g; a.dg = o->dg; a.d = o->d; a.f = o->f; a.df = o->df; a.L = o->L;
        a.iter = o->iter; a.term = o->term; a.n = (int)o->n; a.dim = (int)o->dim; a.objective = o->objective;
        a.sphere = (o->constraint == DZO_CONSTRAINT_SPHERE); a.max_increases = o->max_increases; a.ksteps = k;
        a.batch = o->batch; a.initial_step_length = L0; a.mode = mode;
        gd_batched_kernel<<<(unsigned)((o->batch + 127) / 128), 128, 0, o->stream>>>(a);
        DZO_CUDA(cudaGetLastError());
        return DZO_OK;
    }
    if (o->objective == DZO_OBJ_RIESZ) {
        RieszGdArgs a = riesz_args(o, mode, k);
        a.initial_step_length = L0;
        if (g_tuning.riesz_profile && mode == 0) {
            if (!o->prof) DZO_TRY(dmalloc(&o->prof, (size_t)1 + 2 * kRieszProfCap));
            DZO_CUDA(cudaMemsetAsync(o->prof, 0, 8, o->stream));
            a.prof = o->prof;
        }
        void* params[] = {&a};
        DZO_CUDA(cudaLaunchCooperativeKernel(riesz_kernel_for((int)o->dim, o->nt), dim3(o->grid), dim3(o->nt), params,
                                             riesz_gd_smem((int)o->dim, o->nt), o->stream));
        return DZO_OK;
    }
    if (o->gridgd)
        return grid_gd_launch(o->gridgd, mode, k, o->stream, o->x, o->dx, o->g, o->dg, o->d, o->n, o->max_increases, L0);
    return fail(DZO_ERR_UNSUPPORTED, "no device kernel for this objective / size");
}

extern "C" {

int dzo_gd_create(dzo_gd** out, int objective, int constraint, int64_t obj_param, int64_t n, int64_t batch,
                  const double* x0, double initial_step_length, int max_increases, int device) {
    if (!out || !x0) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    *out = nullptr;
    DZO_TRY(check_problem(objective, constraint, obj_param, n, batch));
    if (batch != 1 && n > DZO_SMALL_N_MAX)
        return fail(DZO_ERR_UNSUPPORTED, "batched GradientDescentOptimizer needs n <= %d; larger n runs one problem per handle", DZO_SMALL_N_MAX);
    if (objective == DZO_OBJ_RIESZ && (obj_param < 1 || obj_param > 4))
        return fail(DZO_ERR_UNSUPPORTED, "device Riesz kernels support 1 <= dim <= 4");
    if (n / (objective == DZO_OBJ_RIESZ ? obj_param : 1) > (1 << 30)) return fail(DZO_ERR_INVALID_ARGUMENT, "n too large");
    DZO_TRY(use_device(device));
    dzo_gd* o = new (std::nothrow) dzo_gd();
    if (!o) return fail(DZO_ERR_ALLOC, "out of memory");
    o->device = device; o->objective = objective; o->constraint = constraint; o->max_increases = max_increases;
    o->dim = obj_param; o->n = n; o->batch = batch;
    o->small = (n <= DZO_SMALL_N_MAX);
    int rc = DZO_OK;
    auto bail = [&](int code) { free_gd(o); return code; };
    if (cudaStreamCreateWithFlags(&o->own_stream, cudaStreamNonBlocking) != cudaSuccess)
        return bail(fail(DZO_ERR_CUDA, "cudaStreamCreate failed"));
    o->stream = o->own_stream;
    const size_t nb = (size_t)n * (size_t)batch;
    if ((rc = dmalloc(&o->x, nb)) || (rc = dmalloc(&o->g, nb)) || (rc = dmalloc(&o->d, nb)) ||
        (rc = dmalloc(&o->dx, nb)) || (rc = dmalloc(&o->dg, nb)) || (rc = dmalloc(&o->ctrl, 1)))
        return bail(rc);
    if (o->small) {
        if ((rc = dmalloc(&o->f, (size_t)batch)) || (rc = dmalloc(&o->df, (size_t)batch)) || (rc = dmalloc(&o->L, (size_t)batch)) ||
            (rc = dmalloc(&o->iter, (size_t)batch)) || (rc = dmalloc(&o->term, (size_t)batch)))
            return bail(rc);
    } else if (objective == DZO_OBJ_RIESZ) {
        RieszWork w;
        if ((rc = w.init((int)(n / obj_param), (int)obj_param, device))) { w.release(); return bail(rc); }
        o->segE = w.segE; o->rowE = w.rowE; o->segG = w.segG; o->fbox = w.fbox; o->e_items = w.e_items;
        o->n_e_items = w.n_e_items; o->counter = w.counter; o->rbcnt = w.rbcnt; o->esplit = w.esplit; o->gcnt_off = w.gcnt_off; o->grid = w.grid;
        o->ecnt_stride = w.ecnt_stride; o->espec = w.espec; o->nt = w.nt; o->bar = w.bar;
        o->g_jobs = w.g_jobs; o->n_g_jobs = w.n_g_jobs; o->gvariant = w.gvariant;
    }
    if (!o->small && objective == DZO_OBJ_ROSENBROCK) {       // one 8-CTA cluster up to n = DZO_TREE_BLOCK, the whole grid above
        if ((rc = grid_gd_attach(n, device, &o->gridgd, &o->gscal))) return bail(rc);
    }
    if (cudaMemcpyAsync(o->x, x0, nb * 8, cudaMemcpyHostToDevice, o->stream) != cudaSuccess)   // :339 collect
        return bail(fail(DZO_ERR_CUDA, "H2D copy of x0 failed"));
    if ((rc = gd_launch(o, 1, 0, initial_step_length))) return bail(rc);
    if (cudaStreamSynchronize(o->stream) != cudaSuccess)
        return bail(fail(DZO_ERR_CUDA, "constructor kernel failed: %s", cudaGetErrorString(cudaGetLastError())));
    *out = o;
    return DZO_OK;
}

void dzo_gd_destroy(dzo_gd* o) { free_gd(o); }

int dzo_gd_set_stream(dzo_gd* o, void* cuda_stream) {
    if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");
    DZO_TRY(use_device(o->device));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    o->stream = cuda_stream ? (cudaStream_t)cuda_stream : o->own_stream;
    return DZO_OK;
}

int dzo_gd_step_async(dzo_gd* o, int k) {
    if (!o || k < 0) return fail(DZO_ERR_INVALID_ARGUMENT, "bad arguments");
    DZO_TRY(use_device(o->device));
    if (k == 0) return DZO_OK;
    return gd_launch(o, 0, k, 0.0);
}
int dzo_gd_sync(dzo_gd* o) {
    if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");
    DZO_TRY(use_device(o->device));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    return DZO_OK;
}
int dzo_gd_step(dzo_gd* o, int k) {
    DZO_TRY(dzo_gd_step_async(o, k));
    return dzo_gd_sync(o);
}

static int gd_read(dzo_gd* o, void* dst, const void* src, size_t bytes) {
    if (!o || !dst) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    DZO_TRY(use_device(o->device));
    DZO_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, o->stream));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    return DZO_OK;
}
#define DZO_GD_VEC(name, field)                                                   \
    int name(dzo_gd* o, double* out) {                                            \
        if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");             \
        return gd_read(o, out, o->field, (size_t)o->n * (size_t)o->batch * 8);    \
    }
DZO_GD_VEC(dzo_gd_get_point, x)
DZO_GD_VEC(dzo_gd_get_delta_point, dx)
DZO_GD_VEC(dzo_gd_get_gradient, g)
DZO_GD_VEC(dzo_gd_get_delta_gradient, dg)
DZO_GD_VEC(dzo_gd_get_direction, d)
#undef DZO_GD_VEC
#define DZO_GD_SCALAR(name, type, expr, field)                                    \
    int name(dzo_gd* o, type* out) {                                              \
        if (!o || !out) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");    \
        if (o->small) return gd_read(o, out, o->field, (size_t)o->batch * sizeof(type));   \
        GdCtrl c;                                                                 \
        if (o->gridgd) {                                                          \
            double s6[6];                                                         \
            DZO_TRY(gd_read(o, s6, o->gscal, sizeof s6));                         \
            c.f = s6[0]; c.df = s6[1]; c.L = s6[2]; c.iter = (long long)s6[3]; c.term = (int)s6[4]; \
        } else {                                                                  \
            DZO_TRY(gd_read(o, &c, o->ctrl, sizeof c));                           \
        }                                                                         \
        *out = (type)(expr);                                                      \
        return DZO_OK;                                                            \
    }
DZO_GD_SCALAR(dzo_gd_get_objective, double, c.f, f)
DZO_GD_SCALAR(dzo_gd_get_delta_objective, double, c.df, df)
DZO_GD_SCALAR(dzo_gd_get_step_length, double, c.L, L)
DZO_GD_SCALAR(dzo_gd_get_iteration_count, int64_t, c.iter, iter)
DZO_GD_SCALAR(dzo_gd_get_terminated, uint8_t, c.term != 0, term)
#undef DZO_GD_SCALAR

int dzo_gd_get_evaluation_count(dzo_gd* o, int64_t* out) {
    if (!o || !out) return fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    if (o->small) return fail(DZO_ERR_UNSUPPORTED, "evaluation count: one-problem (n > 32) handles only");
    if (o->gridgd) {
        double s6[6];
        DZO_TRY(gd_read(o, s6, o->gscal, sizeof s6));
        *out = (int64_t)s6[5];
        return DZO_OK;
    }
    GdCtrl c;
    DZO_TRY(gd_read(o, &c, o->ctrl, sizeof c));
    *out = (int64_t)c.evals;
    return DZO_OK;
}
int dzo_gd_get_phase_log(dzo_gd* o, uint64_t* events, int64_t cap_events, int64_t* count) {
    if (!o || !events || !count || cap_events < 0) return fail(DZO_ERR_INVALID_ARGUMENT, "bad arguments");
    *count = 0;
    if (!o->prof) return DZO_OK;
    DZO_TRY(use_device(o->device));
    DZO_CUDA(cudaStreamSynchronize(o->stream));
    unsigned long long k = 0;
    DZO_CUDA(cudaMemcpy(&k, o->prof, 8, cudaMemcpyDeviceToHost));
    if (k > (unsigned long long)cap_events) k = (unsigned long long)cap_events;
    if (k) DZO_CUDA(cudaMemcpy(events, o->prof + 1, (size_t)k * 16, cudaMemcpyDeviceToHost));
    *count = (int64_t)k;
    return DZO_OK;
}
int dzo_gd_info(dzo_gd* o, int64_t* n, int64_t* batch, int* order) {
    if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");
    if (n) *n = o->n;
    if (batch) *batch = o->batch;
    if (order) *order = o->small ? DZO_ORDER_SEQUENTIAL : (o->gridgd ? DZO_ORDER_TREE_BLOCKED : DZO_ORDER_TREE);
    return DZO_OK;
}
int dzo_gd_riesz_info(dzo_gd* o, int* threads_per_cta, int* ctas, int* energy_lanes_per_row, int* paired_probes,
                      int* gradient_tiles, int* flag_barrier) {
    if (!o) return fail(DZO_ERR_INVALID_ARGUMENT, "null handle");
    if (o->small || o->objective != DZO_OBJ_RIESZ)
        return fail(DZO_ERR_UNSUPPORTED, "riesz info: one-problem Riesz handles (n > %d) only", DZO_SMALL_N_MAX);
    if (threads_per_cta) *threads_per_cta = o->nt;
    if (ctas) *ctas = o->grid;
    if (energy_lanes_per_row) *energy_lanes_per_row = o->esplit;
    if (paired_probes) *paired_probes = (o->espec != 0 && o->esplit != 2) ? 1 : 0;   // what line_search uses
    if (gradient_tiles) *gradient_tiles = o->gvariant;
    if (flag_barrier) *flag_barrier = (o->bar != nullptr) ? 1 : 0;
    return DZO_OK;
}

}  // extern "C"

// ============================================================================= BFGS x Riesz hook (used by dzopt_bfgs.cu)
namespace dzo {

struct RieszBfgs {
    RieszWork w;
    int N = 0, dim = 0, sphere = 0;
};

int riesz_bfgs_attach(int64_t n, int64_t dim, int constraint, int device, void** out) {
    *out = nullptr;
    if (dim < 1 || dim > 4) return fail(DZO_ERR_UNSUPPORTED, "device Riesz kernels support 1 <= dim <= 4");
    RieszBfgs* r = new (std::nothrow) RieszBfgs();
    if (!r) return fail(DZO_ERR_ALLOC, "out of memory");
    r->N = (int)(n / dim); r->dim = (int)dim; r->sphere = (constraint == DZO_CONSTRAINT_SPHERE);
    int rc = r->w.init(r->N, r->dim, device);
    if (rc) { r->w.release(); delete r; return rc; }
    *out = r;
    return DZO_OK;
}
void riesz_bfgs_detach(void* p) {
    RieszBfgs* r = static_cast<RieszBfgs*>(p);
    if (!r) return;
    r->w.release();
    delete r;
}
// mode 6 = constructor, 5 = search stage of one step!
int riesz_bfgs_launch(void* p, int mode, cudaStream_t stream, double* x, double* g, double* d, double* dx, double* dg,
                      double* sd, LargeCtrl* ctrl, double initial_step_length) {
    RieszBfgs* r = static_cast<RieszBfgs*>(p);
    RieszGdArgs a;
    memset(&a, 0, sizeof a);
    a.x = x; a.g = g; a.d = d; a.dx = dx; a.dg = dg; a.sd = sd; a.bctrl = ctrl;
    r->w.fill(a);
    a.N = r->N; a.sphere = r->sphere; a.max_increases = 0; a.mode = mode; a.initial_step_length = initial_step_length;
    return r->w.launch(a, stream);
}

}  // namespace dzo

// ============================================================================= Riesz kernel-level entries
namespace dzo {

struct RieszScratch {
    DevBuf x, g, d;
    RieszWork w;
    RieszGdArgs a;
    ~RieszScratch() { w.release(); }
    int init(int constraint, int64_t dim, int64_t n, const double* xh, const double* dh) {
        int device = 0;
        DZO_CUDA(cudaGetDevice(&device));
        DZO_TRY(x.alloc((size_t)n * 8)); DZO_TRY(g.alloc((size_t)n * 8)); DZO_TRY(d.alloc((size_t)n * 8));
        DZO_CUDA(cudaMemcpy(x.p, xh, (size_t)n * 8, cudaMemcpyHostToDevice));
        if (dh) DZO_CUDA(cudaMemcpy(d.p, dh, (size_t)n * 8, cudaMemcpyHostToDevice));
        DZO_TRY(w.init((int)(n / dim), (int)dim, device));
        memset(&a, 0, sizeof a);
        a.x = x.as<double>(); a.g = g.as<double>(); a.d = d.as<double>(); a.dx = nullptr; a.dg = nullptr;
        w.fill(a);
        a.N = (int)(n / dim); a.sphere = (constraint == DZO_CONSTRAINT_SPHERE);
        return DZO_OK;
    }
};

static int riesz_order_ok(int order, int64_t dim) {
    if (order != DZO_ORDER_TREE) return fail(DZO_ERR_UNSUPPORTED, "device Riesz kernels compute in DZO_ORDER_TREE");
    if (dim < 1 || dim > 4) return fail(DZO_ERR_UNSUPPORTED, "device Riesz kernels support 1 <= dim <= 4");
    return DZO_OK;
}

int riesz_dev_objective(int constraint, int64_t dim, int order, int64_t n, int64_t batch, const double* x, double* f) {
    DZO_TRY(riesz_order_ok(order, dim));
    for (int64_t p = 0; p < batch; ++p) {
        RieszScratch s;
        DZO_TRY(s.init(constraint, dim, n, x + p * n, nullptr));
        s.a.mode = 2;
        DZO_TRY(s.w.launch(s.a, 0));
        DZO_CUDA(cudaDeviceSynchronize());
        double box[4];
        DZO_CUDA(cudaMemcpy(box, s.w.fbox, sizeof box, cudaMemcpyDeviceToHost));
        f[p] = box[1];
    }
    return DZO_OK;
}

int riesz_dev_gradient(int constraint, int64_t dim, int order, int64_t n, int64_t batch, const double* x, double* g) {
    DZO_TRY(riesz_order_ok(order, dim));
    for (int64_t p = 0; p < batch; ++p) {
        RieszScratch s;
        DZO_TRY(s.init(constraint, dim, n, x + p * n, nullptr));
        s.a.mode = 3;
        DZO_TRY(s.w.launch(s.a, 0));
        DZO_CUDA(cudaDeviceSynchronize());
        DZO_CUDA(cudaMemcpy(g + p * n, s.g.p, (size_t)n * 8, cudaMemcpyDeviceToHost));
    }
    return DZO_OK;
}

// along x - t*dir (the BFGS functor sign), like dzo_cpu_line_search
int riesz_dev_line_search(int constraint, int64_t dim, int order, int64_t n, const double* x, const double* dir, double f0,
                          double t1, double* t_best, double* f_best) {
    DZO_TRY(riesz_order_ok(order, dim));
    RieszScratch s;
    DZO_TRY(s.init(constraint, dim, n, x, dir));
    s.a.mode = 4; s.a.ls_f0 = f0; s.a.ls_t1 = t1; s.a.ls_sign = -1.0; s.a.max_increases = 0;
    DZO_TRY(s.w.launch(s.a, 0));
    DZO_CUDA(cudaDeviceSynchronize());
    double box[4];
    DZO_CUDA(cudaMemcpy(box, s.w.fbox, sizeof box, cudaMemcpyDeviceToHost));
    *t_best = box[1]; *f_best = box[2];
    return DZO_OK;
}

}  // namespace dzo

// ============================================================================= ieee_fast.cuh self-test
extern "C" int dzo_dev_selftest_ieee_fast(uint64_t count, uint64_t seed, uint64_t* mismatches, int device) {
    if (!mismatches) return dzo::fail(DZO_ERR_INVALID_ARGUMENT, "null pointer");
    DZO_TRY(dzo::use_device(device));
    dzo::DevBuf b;
    DZO_TRY(b.alloc(8));
    DZO_CUDA(cudaMemset(b.p, 0, 8));
    dzo::ieee_fast_selftest_kernel<<<148 * 8, 256>>>(count, seed, b.as<unsigned long long>());
    DZO_CUDA(cudaGetLastError());
    DZO_CUDA(cudaDeviceSynchronize());
    DZO_CUDA(cudaMemcpy(mismatches, b.p, 8, cudaMemcpyDeviceToHost));
    return DZO_OK;
}
