// host_common.h -- host-side plumbing shared by the C-ABI translation units of libdzopt_b200.
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/dzopt.h"

namespace dzo {

extern thread_local char g_err[512];

inline int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

#define DZO_CUDA(call)                                                                              \
    do {                                                                                            \
        cudaError_t e__ = (call);                                                                   \
        if (e__ != cudaSuccess)                                                                     \
            return ::dzo::fail(DZO_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #call,           \
                               cudaGetErrorString(e__));                                            \
    } while (0)

#define DZO_TRY(call)                                                                               \
    do {                                                                                            \
        int rc__ = (call);                                                                          \
        if (rc__ != DZO_OK) return rc__;                                                            \
    } while (0)

// There is no CPU fallback: every entry point that computes goes through this.
inline int use_device(int device) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(DZO_ERR_NO_DEVICE, "no CUDA device available (libdzopt_b200 has no CPU fallback): %s",
                    cudaGetErrorString(e));
    }
    if (device < 0 || device >= count) return fail(DZO_ERR_INVALID_ARGUMENT, "device %d out of range [0,%d)", device, count);
    DZO_CUDA(cudaSetDevice(device));
    return DZO_OK;
}

int check_problem(int objective, int constraint, int64_t obj_param, int64_t n, int64_t batch);

// process-wide tuning knobs (A/B measurements only; never change results)
struct Tuning {
    int batched_prefetch = 3;  // hybrid kernel: L2 prefetch distance in phase-2 rounds (round 2, ms per 1M-problem launch: 1: 1.06,
                               // 2: 0.740, 3: 0.736, 4: 0.740, 6: 0.766)
    int use_graph = 1;        // large-n step!: replay a captured CUDA graph of its four launches
    int epoch = 0;            // bumped by every dzo_set_tuning call
    int sweep_unroll = 16;    // columns in flight per thread in the n^2 sweeps; measured on one box at n=16384:
                              // update kernel 0.79 (U=8), 0.96 (U=16), 0.84 (U=24), 0.87 (U=32) of HBM peak
    int sweep_threads = 0;    // threads per sweep CTA (0 = pick from the slab shape)
    int sharded_variant = 0;  // row-sharded gathers: 0 = fused into the producing kernels over peer memory, 1 = ncclAllGather
    int search_variant = 0;   // large-n O(n) stage: 0 = 8-CTA cluster + DSMEM reductions for one problem, one 1024-thread CTA per
                              // problem for a batch of >= 4; 1 = always single CTA; 2 = always cluster
    int riesz_esplit = 1;     // lanes per row in the Riesz energy items (1 or 2), read when an optimizer is created
    int riesz_gvariant = 0;   // Riesz gradient: 0 = (32 rows x 128 sources) warp items, 1 = symmetric 128 x 128 CTA tiles (each pair
                              // weight computed once; measured 0.183 vs 0.177 ms per GD step at N = 4096, so not the default)
    int grid_ll = 1;          // grid-wide kernels (L-BFGS / AdGD / GD above n = 65536): 1 = reductions through flagged 16-byte lines
                              // (no grid barrier), 0 = one grid.sync per reduction; read when an optimizer is created
    int grid_ll_first_seq = 1; // first sequence number of a new handle's flagged lines (tests start near the recycling threshold 2^27)
    int grid_ll_backoff = 0;  // ns a consumer sleeps after a poll that found a line missing (0 = poll back to back)
    int grid_profile = 0;     // 1: the grid-wide live L-BFGS kernel prints the cycle split of its leader CTA (measurement only)
    int grid_stage = 1;       // live L-BFGS grid kernel with one eighth per CTA: fetch the next pass's history vectors into shared
                              // memory (cp.async) while the current reduction is in flight
    int warp_search = 1;      // O(n) stage of step! for 32 < n <= 512: 1 = one warp per problem (warp_search.cuh), 0 = 8-CTA cluster
    int riesz_threads = 512;  // threads per CTA of the cooperative Riesz kernel (512: 128 registers, 8 / 4 pair terms in flight per
                              // lane; 1024: 64 registers, 4 / 2); read when an optimizer is created
    int riesz_bar = 0;        // cooperative Riesz kernel, k-step mode: 1 = flag-word barrier (per-CTA inboxes) instead of grid.sync().
                              // Measured SLOWER (0.152-0.157 vs 0.146-0.151 ms per GD step!; a pure barrier of 148 CTAs is
                              // cheaper through one atomic counter than through 148 x 148 words), so off; read at create time
    int riesz_pair = 1;       // Riesz line search: evaluate the probe it needs and the one it will most likely need next in one
                              // phase (the second rides in warps the first leaves idle); read when an optimizer is created
    int riesz_profile = 0;    // 1: the cooperative Riesz kernel logs (phase id, %globaltimer) events of its leader thread
    int small_sweeps = 1;     // batches of 32 < n <= 64 problems: n^2 sweeps on one warp per problem (small_sweeps.cuh); 0 = tiled kernels
    int batched_tile = 0;     // batched kernel, problems per warp: 0 = automatic (32, fewer for batches of at most three waves of
                              // warps), 32 = always a full warp, 1..31 = forced; read when an optimizer is created
    int batched_lazy = 1;     // batched kernel: keep H = I implicit (no HBM traffic for identity_matrix!); read at create time
                              // (1M x n=16: 0.74 ms per launch with, 0.86 ms without)
    int batched_derived = -1; // batched kernel: derived layout (batched_bfgs.cuh, BatchedArgs::derived) -- a move stores x into the
                              // other of two point buffers and no g, dx, dg, which the getters recompute; 1 = always, 0 = every
                              // field stored, -1 = derived for n > 8 only; read at create time.  1 M problems per launch on a
                              // B200 (1000 W), stored -> derived ms: n = 16: 0.696 -> 0.635, n = 32: 2.39 -> 2.21, n = 8: 0.318
                              // -> 0.320 (profiles/r03_batched_derived_ab.jsonl, DESIGN.md section 3)
    int lbfgs_batched_threads = 128; // batched live L-BFGS (batched_lbfgs.cuh): threads per CTA, 64 / 128 / 256; read at create
                                     // time
};
extern Tuning g_tuning;

// scoped device buffer for the kernel-level entry points
struct DevBuf {
    void* p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    int alloc(size_t bytes) {
        if (bytes == 0) bytes = 8;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) { p = nullptr; return fail(DZO_ERR_ALLOC, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e)); }
        return DZO_OK;
    }
    template <class T> T* as() const { return static_cast<T*>(p); }
};

}  // namespace dzo
