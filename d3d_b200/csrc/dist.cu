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

// ------------------------------------------------------------------ frame-batched distance
// Frame f owns points [poff[f], poff[f+1]) and boxes [boff[f], boff[f+1]) of the packed inputs and writes its row-major [m_f, n_f] block
// at dist + doff[f].  Frames on grid.x, 256-point blocks on grid.y and 8-box tiles on grid.z, each striding over the frame's own tiles
// (tiles beyond the frame's size exit at once).  The pairs run pd_pair on boxes staged as above, so project_axis -1 gives the values of
// d3d_pdist2dr_* bit for bit.  project_axis 0, 1 or 2: 3-D rows (points [n,3], boxes [m,7]); pd_pair runs in the plane of the two other
// axes, and the value is box3dr_pdist's combination of that distance with seg1d_pdist's along the axis, rounded like torch's operators.
template <typename T> struct PdZ { T c, hd; };   // box centre and half extent along the axis

template <typename T>
__device__ __forceinline__ void pd_stage(const T *b, int axis, int pa, int pb, PBox<T> *q, PdZ<T> *z)
{
    if (axis < 0) { *q = pd_box<T>(b); return; }
    const T r[5] = {b[pa], b[pb], b[3 + pa], b[3 + pb], b[6]};
    *q = pd_box<T>(r);
    z->c = b[axis]; z->hd = rn_div2(b[3 + axis]);
}

// seg1d_pdist: (c + d/2) - p above the centre, p - (c - d/2) below it; positive inside
template <typename T> __device__ __forceinline__ T pd_seg(T p, const PdZ<T> &z) { return p > z.c ? rn_sub(rn_add(z.c, z.hd), p) : rn_sub(p, rn_sub(z.c, z.hd)); }

// box3dr_pdist's where-tree over the in-plane distance d2 and the axial distance dp
template <typename T>
__device__ __forceinline__ T pd3_value(T d2, T dp)
{
    const T sq = rn_add(rn_mul(d2, d2), rn_mul(dp, dp));
    const T corner = sq > T(0) ? -rn_sqrt(sq) : T(0);
    return dp > T(0) ? (d2 > T(0) ? (dp < d2 ? dp : d2) : d2) : (d2 > T(0) ? dp : corner);
}

// its derivatives in (d2, dp): torch.minimum's rule on the prism's inside (equal values get half each); -(d2, dp) / sqrt(d2^2 + dp^2)
// on the corner branch, and 0 where both are 0 (an edge of the prism)
template <typename T>
__device__ __forceinline__ void pd3_grad(T d2, T dp, T *g2, T *gp)
{
    *g2 = T(0); *gp = T(0);
    if (dp > T(0)) {
        if (d2 > T(0)) { *g2 = d2 < dp ? T(1) : d2 == dp ? T(0.5) : T(0); *gp = dp < d2 ? T(1) : d2 == dp ? T(0.5) : T(0); }
        else *g2 = T(1);
    } else if (d2 > T(0)) {
        *gp = T(1);
    } else {
        const T sq = rn_add(rn_mul(d2, d2), rn_mul(dp, dp));
        if (sq > T(0)) { const T r = rn_sqrt(sq); *g2 = -d2 / r; *gp = -dp / r; }
    }
}

template <typename T, bool P3>
__global__ void __launch_bounds__(PD_THREADS) pdist_fwd_batch_kernel(const T *__restrict__ pts, const int64_t *__restrict__ poff, const T *__restrict__ boxes,
                                                                     const int64_t *__restrict__ boff, int axis, const int64_t *__restrict__ doff, T *__restrict__ dist)
{
    __shared__ PBox<T> sb[PD_BOXES];
    __shared__ PdZ<T> sz[PD_BOXES];
    const int64_t f = blockIdx.x, j0 = poff[f], n = poff[f + 1] - j0, i0 = boff[f], m = boff[f + 1] - i0;
    if ((int64_t)blockIdx.y * PD_THREADS >= n || (int64_t)blockIdx.z * PD_BOXES >= m) return;
    int pa = 0, pb = 1;
    if (P3) proj_plane(axis, &pa, &pb);
    constexpr int PS = P3 ? 3 : 2, BS = P3 ? 7 : 5;   // row lengths
    T *blk = dist + doff[f];
    for (int64_t t0 = (int64_t)blockIdx.y * PD_THREADS; t0 < n; t0 += (int64_t)gridDim.y * PD_THREADS) {
        const int64_t j = t0 + threadIdx.x;
        const bool in = j < n;
        const T px = in ? pts[PS * (j0 + j) + pa] : T(0), py = in ? pts[PS * (j0 + j) + pb] : T(0), pz = in && P3 ? pts[PS * (j0 + j) + axis] : T(0);
        for (int64_t b0 = (int64_t)blockIdx.z * PD_BOXES; b0 < m; b0 += (int64_t)gridDim.z * PD_BOXES) {
            if (threadIdx.x < PD_BOXES && b0 + threadIdx.x < m) pd_stage<T>(boxes + BS * (i0 + b0 + threadIdx.x), P3 ? axis : -1, pa, pb, sb + threadIdx.x, sz + threadIdx.x);
            __syncthreads();
            if (in) {
                for (int k = 0; k < PD_BOXES && b0 + k < m; k++) {
                    int e;
                    const T d2 = pd_pair<T, false>(sb[k], px, py, &e, T(0), nullptr, nullptr);
                    blk[(b0 + k) * n + j] = P3 ? pd3_value(d2, pd_seg(pz, sz[k])) : d2;
                }
            }
            __syncthreads();
        }
    }
}

// grad_pts [n, PS] and grad_boxes [m, BS] accumulate like pdist_bwd_kernel's: per-CTA box sums, one atomic per field
// column of box gradient slot c (pd_pair's x, y, w, h, r, then the axis' centre and extent) in a box row
__device__ __forceinline__ int pd_box_col(int c, int axis, int pa, int pb)
{
    if (axis < 0) return c;
    return c == 0 ? pa : c == 1 ? pb : c == 2 ? 3 + pa : c == 3 ? 3 + pb : c == 4 ? 6 : c == 5 ? axis : 3 + axis;
}

// (the minimum of 2 CTAs per SM lifts ptxas' register target: at its default the registers live across the slow-path sin / cos call of the
// box staging spill)
template <typename T, bool P3>
__global__ void __launch_bounds__(PD_THREADS, 2) pdist_bwd_batch_kernel(const T *__restrict__ pts, const int64_t *__restrict__ poff, const T *__restrict__ boxes,
                                                                     const int64_t *__restrict__ boff, int axis, const int64_t *__restrict__ doff,
                                                                     const T *__restrict__ grad, T *__restrict__ grad_boxes, T *__restrict__ grad_pts)
{
    constexpr int PS = P3 ? 3 : 2, BS = P3 ? 7 : 5;
    __shared__ PBox<T> sb[PD_BOXES];
    __shared__ PdZ<T> sz[PD_BOXES];
    __shared__ T sacc[PD_BOXES][BS];
    const int64_t f = blockIdx.x, j0 = poff[f], n = poff[f + 1] - j0, i0 = boff[f], m = boff[f + 1] - i0;
    if ((int64_t)blockIdx.y * PD_THREADS >= n || (int64_t)blockIdx.z * PD_BOXES >= m) return;
    int pa = 0, pb = 1;
    if (P3) proj_plane(axis, &pa, &pb);
    const T *g = grad + doff[f];
    const unsigned lane = threadIdx.x & 31u;
    for (int64_t t0 = (int64_t)blockIdx.y * PD_THREADS; t0 < n; t0 += (int64_t)gridDim.y * PD_THREADS) {
        const int64_t j = t0 + threadIdx.x;
        const bool in = j < n;
        const T px = in ? pts[PS * (j0 + j) + pa] : T(0), py = in ? pts[PS * (j0 + j) + pb] : T(0), pz = in && P3 ? pts[PS * (j0 + j) + axis] : T(0);
        T gp[PS] = {};
        for (int64_t b0 = (int64_t)blockIdx.z * PD_BOXES; b0 < m; b0 += (int64_t)gridDim.z * PD_BOXES) {
            if (threadIdx.x < PD_BOXES && b0 + threadIdx.x < m) {
                pd_stage<T>(boxes + BS * (i0 + b0 + threadIdx.x), P3 ? axis : -1, pa, pb, sb + threadIdx.x, sz + threadIdx.x);
                for (int c = 0; c < BS; c++) sacc[threadIdx.x][c] = T(0);
            }
            __syncthreads();
            for (int k = 0; k < PD_BOXES && b0 + k < m; k++) {
                T gb[BS];
#pragma unroll
                for (int c = 0; c < BS; c++) gb[c] = T(0);
                if (in) {
                    int e;
                    const T up = g[(b0 + k) * n + j];
                    if (!P3) {
                        pd_pair<T, true>(sb[k], px, py, &e, up, gp, gb);
                    } else {
                        T tp[2] = {0, 0}, tb[5] = {0, 0, 0, 0, 0};
                        const T d2 = pd_pair<T, true>(sb[k], px, py, &e, T(1), tp, tb);
                        const T dp = pd_seg(pz, sz[k]);
                        T g2, gz;
                        pd3_grad(d2, dp, &g2, &gz);
                        g2 *= up; gz *= up;
                        gp[0] += g2 * tp[0]; gp[1] += g2 * tp[1];
#pragma unroll
                        for (int c = 0; c < 5; c++) gb[c] = g2 * tb[c];
                        const T s = pz > sz[k].c ? T(-1) : T(1);   // d dp / d p; d dp / d c = -s, d dp / d extent = 1 / 2
                        gp[2] += s * gz;
                        gb[5] = -s * gz; gb[6] = T(0.5) * gz;
                    }
                }
#pragma unroll
                for (int c = 0; c < BS; c++) {
                    T v = gb[c];
#pragma unroll
                    for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
                    if (lane == 0 && v != T(0)) pd_atomic_add(&sacc[k][c], v);
                }
            }
            __syncthreads();
            if (threadIdx.x < PD_BOXES * BS) {
                const int k = threadIdx.x / BS, c = threadIdx.x % BS;
                if (b0 + k < m && sacc[k][c] != T(0)) pd_atomic_add(grad_boxes + BS * (i0 + b0 + k) + pd_box_col(c, P3 ? axis : -1, pa, pb), sacc[k][c]);
            }
            __syncthreads();
        }
        if (in) {
#pragma unroll
            for (int c = 0; c < PS; c++) pd_atomic_add(grad_pts + PS * (j0 + j) + (c == 0 ? pa : c == 1 ? pb : axis), gp[c]);
        }
    }
}

// the checks shared by the forward and the backward; *run = false: nothing to do
static int pd_batch_args(int64_t total_pts, const int64_t *poff, int64_t total_boxes, const int64_t *boff, int64_t nframes, int64_t *max_pts,
                         int64_t *max_boxes, int axis, const int64_t *doff, dim3 *grid, bool *run)
{
    *run = false;
    if (total_pts < 0 || total_boxes < 0 || nframes < 0 || *max_pts < 0 || *max_boxes < 0 || axis < -1 || axis > 2) return D3D_ERR_INVALID_ARGUMENT;
    if (nframes == 0 || total_pts == 0 || total_boxes == 0) return D3D_OK;   // every block is empty
    if (!poff || !boff || !doff) return D3D_ERR_INVALID_ARGUMENT;
    if (nframes > 0x7fffffffll) return D3D_ERR_UNSUPPORTED;
    if (*max_pts == 0) *max_pts = total_pts;   // 0: bound unknown
    if (*max_boxes == 0) *max_boxes = total_boxes;
    const int64_t gy = cdiv(*max_pts, PD_THREADS), gz = cdiv(*max_boxes, PD_BOXES);
    *grid = dim3((unsigned)nframes, (unsigned)(gy < PD_MAX_GY ? gy : PD_MAX_GY), (unsigned)(gz < PD_MAX_GY ? gz : PD_MAX_GY));
    *run = true;
    return D3D_OK;
}

template <typename T>
static int pdist_fwd_batch(const T *pts, int64_t total_pts, const int64_t *poff, const T *boxes, int64_t total_boxes, const int64_t *boff, int64_t nframes,
                           int64_t max_pts, int64_t max_boxes, int axis, const int64_t *doff, T *dist, cudaStream_t st)
{
    dim3 grid;
    bool run;
    const int rc = pd_batch_args(total_pts, poff, total_boxes, boff, nframes, &max_pts, &max_boxes, axis, doff, &grid, &run);
    if (rc || !run) return rc;
    if (!pts || !boxes || !dist) return D3D_ERR_INVALID_ARGUMENT;
    if (axis < 0) pdist_fwd_batch_kernel<T, false><<<grid, PD_THREADS, 0, st>>>(pts, poff, boxes, boff, axis, doff, dist);
    else pdist_fwd_batch_kernel<T, true><<<grid, PD_THREADS, 0, st>>>(pts, poff, boxes, boff, axis, doff, dist);
    D3D_LAUNCHED();
    return D3D_OK;
}

template <typename T>
static int pdist_bwd_batch(const T *pts, int64_t total_pts, const int64_t *poff, const T *boxes, int64_t total_boxes, const int64_t *boff, int64_t nframes,
                           int64_t max_pts, int64_t max_boxes, int axis, const int64_t *doff, const T *grad, T *grad_boxes, T *grad_pts, cudaStream_t st)
{
    dim3 grid;
    bool run;
    const int rc = pd_batch_args(total_pts, poff, total_boxes, boff, nframes, &max_pts, &max_boxes, axis, doff, &grid, &run);
    if (rc || !run) return rc;
    if (!pts || !boxes || !grad || !grad_boxes || !grad_pts) return D3D_ERR_INVALID_ARGUMENT;
    if (axis < 0) pdist_bwd_batch_kernel<T, false><<<grid, PD_THREADS, 0, st>>>(pts, poff, boxes, boff, axis, doff, grad, grad_boxes, grad_pts);
    else pdist_bwd_batch_kernel<T, true><<<grid, PD_THREADS, 0, st>>>(pts, poff, boxes, boff, axis, doff, grad, grad_boxes, grad_pts);
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
#define D3D_PD_BATCH(SUF, T)                                                                                                                          \
    extern "C" int d3d_pdist2dr_batch_##SUF(const T *points, int64_t total_points, const int64_t *point_offsets, const T *boxes, int64_t total_boxes, \
                                            const int64_t *box_offsets, int64_t nframes, int64_t max_frame_points, int64_t max_frame_boxes,         \
                                            int project_axis, const int64_t *dist_offsets, T *dist, void *stream)                                   \
    {                                                                                                                                                 \
        return pdist_fwd_batch<T>(points, total_points, point_offsets, boxes, total_boxes, box_offsets, nframes, max_frame_points, max_frame_boxes,  \
                                  project_axis, dist_offsets, dist, (cudaStream_t)stream);                                                            \
    }                                                                                                                                                 \
    extern "C" int d3d_pdist2dr_batch_backward_##SUF(const T *points, int64_t total_points, const int64_t *point_offsets, const T *boxes,            \
                                                     int64_t total_boxes, const int64_t *box_offsets, int64_t nframes, int64_t max_frame_points,      \
                                                     int64_t max_frame_boxes, int project_axis, const int64_t *dist_offsets, const T *grad,          \
                                                     T *grad_boxes, T *grad_points, void *stream)                                                    \
    {                                                                                                                                                 \
        return pdist_bwd_batch<T>(points, total_points, point_offsets, boxes, total_boxes, box_offsets, nframes, max_frame_points, max_frame_boxes,  \
                                  project_axis, dist_offsets, grad, grad_boxes, grad_points, (cudaStream_t)stream);                                  \
    }
D3D_PD_BATCH(f32, float)
D3D_PD_BATCH(f64, double)
