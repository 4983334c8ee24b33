// common.cuh -- shared helpers for the d3d_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include "../../include/d3d_b200.h"

namespace d3d {

extern std::atomic<int64_t> g_launches;
// tuning knobs (core.cu): environment read once at first use, d3d_tuning_set() overrides
enum { D3D_TUNE_NMS_PATH = 0, D3D_TUNE_CROP_PATH, D3D_TUNE_VOX_ROUTE, D3D_TUNE_NMS_STOP, D3D_TUNE_SCATTER_PATH, D3D_TUNE_NMS_FIX, D3D_TUNE_NMS_BATCH_PATH,
       D3D_TUNE_SORT_COOP, D3D_TUNE_COUNT };
int tuning(int knob, int dflt);
void set_cuda_error(cudaError_t e);

#define D3D_CUDA_TRY(expr)                                  \
    do {                                                    \
        cudaError_t _e = (expr);                            \
        if (_e != cudaSuccess) { ::d3d::set_cuda_error(_e); return D3D_ERR_CUDA; } \
    } while (0)

// count + check a kernel launch (launch errors only; execution stays asynchronous)
#define D3D_LAUNCHED()                                      \
    do {                                                    \
        ::d3d::g_launches.fetch_add(1, std::memory_order_relaxed); \
        cudaError_t _e = cudaGetLastError();                \
        if (_e != cudaSuccess) { ::d3d::set_cuda_error(_e); return D3D_ERR_CUDA; } \
    } while (0)

static inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }
static inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// bump allocator over the caller's workspace
struct Arena {
    char *base; size_t cap, off;
    Arena(void *p, size_t n) : base((char *)p), cap(n), off(0) {}
    template <typename T> T *take(size_t count) {
        size_t bytes = align_up(count * sizeof(T));
        T *r = (T *)(base + off); off += bytes; return r;
    }
    bool ok() const { return off <= cap; }
};

// explicitly rounded arithmetic, never contracted into an FMA: results that must equal code compiled without contraction (the
// reference's CPU code, torch's elementwise operators) bit for bit
template <typename T> __device__ __forceinline__ T rn_mul(T a, T b);
template <> __device__ __forceinline__ float rn_mul<float>(float a, float b) { return __fmul_rn(a, b); }
template <> __device__ __forceinline__ double rn_mul<double>(double a, double b) { return __dmul_rn(a, b); }
template <typename T> __device__ __forceinline__ T rn_sub(T a, T b);
template <> __device__ __forceinline__ float rn_sub<float>(float a, float b) { return __fsub_rn(a, b); }
template <> __device__ __forceinline__ double rn_sub<double>(double a, double b) { return __dsub_rn(a, b); }
template <typename T> __device__ __forceinline__ T rn_add(T a, T b);
template <> __device__ __forceinline__ float rn_add<float>(float a, float b) { return __fadd_rn(a, b); }
template <> __device__ __forceinline__ double rn_add<double>(double a, double b) { return __dadd_rn(a, b); }
template <typename T> __device__ __forceinline__ T rn_div2(T a);
template <> __device__ __forceinline__ float rn_div2<float>(float a) { return __fmul_rn(a, 0.5f); }     // x / 2 is exact
template <> __device__ __forceinline__ double rn_div2<double>(double a) { return __dmul_rn(a, 0.5); }
template <typename T> __device__ __forceinline__ T rn_sqrt(T a);
template <> __device__ __forceinline__ float rn_sqrt<float>(float a) { return __fsqrt_rn(a); }
template <> __device__ __forceinline__ double rn_sqrt<double>(double a) { return __dsqrt_rn(a); }

// projection of 3-D rows to an axis (box3dp_crop, box3dr_pdist): the plane of the two other axes is point columns (a, b) of [n, 3] and
// box columns (a, b, 3 + a, 3 + b, 6) of [m, 7] (x, y, z, lx, ly, lz, r)
__device__ __forceinline__ void proj_plane(int axis, int *a, int *b) { *a = axis == 0 ? 1 : 0; *b = axis == 2 ? 1 : 2; }

__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31u; }
__device__ __forceinline__ unsigned lanemask_lt() { unsigned m; asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m)); return m; }

}  // namespace d3d
