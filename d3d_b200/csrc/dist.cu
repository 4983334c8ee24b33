// dist.cu -- signed distance from points to rotated boxes (SURVEY.md 8(f) row f4, second half).
//
// Replaces pdist2dr_forward / pdist2dr_backward[_cuda] (reference d3d/box/dist.h:7-23, dist.cpp:11-110, dist_cuda.cu:9-81) behind
// box2dr_pdist / box3dr_pdist (d3d/box/__init__.py:149-166, 330-381).  The value is the signed Euclidean distance to the box's boundary,
// positive inside, computed in the box's own frame (dist.cuh) -- not dgal's line-by-line distance(Poly2, Point2), whose sign at points on
// the line through an edge and whose projection at headings of pi / 2 are wrong (DESIGN.md section 2, deviation P1).  The backward is the
// analytic gradient of that value; box gradients are reduced per box inside the CTA and leave with one atomic per field.
#include "common.cuh"
#include "dist.cuh"

namespace d3d {

constexpr int PD_THREADS = 256;
constexpr int PD_BOXES = 8;          // boxes per tile (their frames live in shared memory)
constexpr int64_t PD_MAX_GY = 65535; // grid.y limit: larger box counts stride over their tiles

template <typename T>
__global__ void __launch_bounds__(PD_THREADS) pdist_fwd_kernel(const T *__restrict__ pts, int64_t n, const T *__restrict__ boxes, int64_t m, T *__restrict__ dist,
                                                               uint8_t *__restrict__ iedge)
{
    __shared__ PBox<T> sb[PD_BOXES];
    const int64_t j = (int64_t)blockIdx.x * PD_THREADS + threadIdx.x;
    const bool in = j < n;
    const T px = in ? pts[2 * j] : T(0), py = in ? pts[2 * j + 1] : T(0);
    for (int64_t b0 = (int64_t)blockIdx.y * PD_BOXES; b0 < m; b0 += (int64_t)gridDim.y * PD_BOXES) {
        if (threadIdx.x < PD_BOXES && b0 + threadIdx.x < m) sb[threadIdx.x] = pd_box<T>(boxes + 5 * (b0 + threadIdx.x));
        __syncthreads();
        if (in) {
            for (int k = 0; k < PD_BOXES && b0 + k < m; k++) {
                int e;
                const T d = pd_pair<T, false>(sb[k], px, py, &e, T(0), nullptr, nullptr);
                dist[(b0 + k) * n + j] = d;
                if (iedge) iedge[(b0 + k) * n + j] = (uint8_t)e;
            }
        }
        __syncthreads();
    }
}

__device__ __forceinline__ void pd_atomic_add(float *p, float v) { atomicAdd(p, v); }
__device__ __forceinline__ void pd_atomic_add(double *p, double v) { atomicAdd(p, v); }

template <typename T>
__global__ void __launch_bounds__(PD_THREADS) pdist_bwd_kernel(const T *__restrict__ pts, int64_t n, const T *__restrict__ boxes, int64_t m, const T *__restrict__ grad,
                                                               T *__restrict__ grad_boxes, T *__restrict__ grad_pts)
{
    __shared__ PBox<T> sb[PD_BOXES];
    __shared__ T sacc[PD_BOXES][5];
    const int64_t j = (int64_t)blockIdx.x * PD_THREADS + threadIdx.x;
    const bool in = j < n;
    const T px = in ? pts[2 * j] : T(0), py = in ? pts[2 * j + 1] : T(0);
    T gp[2] = {0, 0};
    const unsigned lane = threadIdx.x & 31u;
    for (int64_t b0 = (int64_t)blockIdx.y * PD_BOXES; b0 < m; b0 += (int64_t)gridDim.y * PD_BOXES) {
        if (threadIdx.x < PD_BOXES && b0 + threadIdx.x < m) {
            sb[threadIdx.x] = pd_box<T>(boxes + 5 * (b0 + threadIdx.x));
            for (int f = 0; f < 5; f++) sacc[threadIdx.x][f] = T(0);
        }
        __syncthreads();
        for (int k = 0; k < PD_BOXES && b0 + k < m; k++) {
            T gb[5] = {0, 0, 0, 0, 0};
            if (in) {
                int e;
                pd_pair<T, true>(sb[k], px, py, &e, grad[(b0 + k) * n + j], gp, gb);
            }
#pragma unroll
            for (int f = 0; f < 5; f++) {
                T v = gb[f];
#pragma unroll
                for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
                if (lane == 0 && v != T(0)) pd_atomic_add(&sacc[k][f], v);
            }
        }
        __syncthreads();
        if (threadIdx.x < PD_BOXES * 5) {
            const int k = threadIdx.x / 5, f = threadIdx.x % 5;
            if (b0 + k < m && sacc[k][f] != T(0)) pd_atomic_add(grad_boxes + 5 * (b0 + k) + f, sacc[k][f]);
        }
        __syncthreads();
    }
    if (in) { pd_atomic_add(grad_pts + 2 * j, gp[0]); pd_atomic_add(grad_pts + 2 * j + 1, gp[1]); }
}

template <typename T>
static int pdist_fwd(const T *pts, int64_t n, const T *boxes, int64_t m, T *dist, uint8_t *iedge, cudaStream_t st)
{
    if (n < 0 || m < 0) return D3D_ERR_INVALID_ARGUMENT;
    if (n == 0 || m == 0) return D3D_OK;
    if (!pts || !boxes || !dist) return D3D_ERR_INVALID_ARGUMENT;
    const int64_t tiles = cdiv(m, PD_BOXES), gy = tiles < PD_MAX_GY ? tiles : PD_MAX_GY;
    pdist_fwd_kernel<T><<<dim3((unsigned)cdiv(n, PD_THREADS), (unsigned)gy), PD_THREADS, 0, st>>>(pts, n, boxes, m, dist, iedge);
    D3D_LAUNCHED();
    return D3D_OK;
}

template <typename T>
static int pdist_bwd(const T *pts, int64_t n, const T *boxes, int64_t m, const T *grad, T *grad_boxes, T *grad_pts, cudaStream_t st)
{
    if (n < 0 || m < 0) return D3D_ERR_INVALID_ARGUMENT;
    if (n == 0 || m == 0) return D3D_OK;
    if (!pts || !boxes || !grad || !grad_boxes || !grad_pts) return D3D_ERR_INVALID_ARGUMENT;
    const int64_t tiles = cdiv(m, PD_BOXES), gy = tiles < PD_MAX_GY ? tiles : PD_MAX_GY;
    pdist_bwd_kernel<T><<<dim3((unsigned)cdiv(n, PD_THREADS), (unsigned)gy), PD_THREADS, 0, st>>>(pts, n, boxes, m, grad, grad_boxes, grad_pts);
    D3D_LAUNCHED();
    return D3D_OK;
}

}  // namespace d3d

using namespace d3d;
extern "C" int d3d_pdist2dr_f32(const float *points, int64_t n, const float *boxes, int64_t m, float *dist, uint8_t *iedge, void *stream)
{ return pdist_fwd<float>(points, n, boxes, m, dist, iedge, (cudaStream_t)stream); }
extern "C" int d3d_pdist2dr_f64(const double *points, int64_t n, const double *boxes, int64_t m, double *dist, uint8_t *iedge, void *stream)
{ return pdist_fwd<double>(points, n, boxes, m, dist, iedge, (cudaStream_t)stream); }
extern "C" int d3d_pdist2dr_backward_f32(const float *points, int64_t n, const float *boxes, int64_t m, const float *grad, float *grad_boxes, float *grad_points, void *stream)
{ return pdist_bwd<float>(points, n, boxes, m, grad, grad_boxes, grad_points, (cudaStream_t)stream); }
extern "C" int d3d_pdist2dr_backward_f64(const double *points, int64_t n, const double *boxes, int64_t m, const double *grad, double *grad_boxes, double *grad_points, void *stream)
{ return pdist_bwd<double>(points, n, boxes, m, grad, grad_boxes, grad_points, (cudaStream_t)stream); }
