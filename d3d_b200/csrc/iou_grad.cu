// iou_grad.cu -- differentiable IoU family: backward of the AABB / rotated IoU and forward + backward of the rotated GIoU / DIoU
// (SURVEY.md 8(a) row A2, 8(f) row f2).
//
// Replaces iou2d_backward, iou2dr_backward, giou2dr_forward/backward, diou2dr_forward/backward [_cuda] (reference d3d/box/iou.h,
// iou.cpp:48-92, 143-419, iou_cuda.cu:50-97, 153-444; dgal::iou_grad / giou_grad / diou_grad, thirdparty/dgal/geometry_grad.hpp:327-606,
// over merge / dimension, geometry.hpp:934-1192, 1232-1291) behind the autograd functions of d3d/box/__init__.py:38-147.
//
// Not a translation of dgal's gradient code, which differentiates through the vertex list of the clipped polygon and therefore has to
// save the list's topology (nx, xflags: 9 B per pair) in the forward pass.  Here the gradient of the intersection area is the boundary
// integral of the normal velocity (Reynolds transport): the boundary of A n B is made of the pieces of A's edges that lie inside B and
// the pieces of B's edges that lie inside A, and moving an end point of an edge moves every point of the edge linearly.  With the piece
// of edge p0 -> p1 inside the other box being t in [t0, t1] (a Liang-Barsky clip against four half planes),
//     dI/dp0 = perp(e) ((t1 - t0) - (t1^2 - t0^2)/2),   dI/dp1 = perp(e) (t1^2 - t0^2)/2,   perp(e) = (e.y, -e.x),
// while the value I / U is geom.cuh's rotated IoU -- nothing is saved between forward and backward.  The hull area of GIoU is the
// shoelace sum over the monotone-chain hull of the eight vertices, the DIoU diameter the largest vertex distance; their gradients sit on
// the vertices involved, and vertices chain to (x, y, w, h, r) in closed form.  Every pair is evaluated in the frame of the row box's
// (forward) or the owned box's (backward) centre; the pair code is in iou_grad.cuh.
// Accumulation is race free and deterministic: one warp owns one box of the side it differentiates, walks the other side and writes
// the five sums once (the reference adds pair gradients into the box rows from all threads, iou_cuda.cu:184-185).
#include "iou_grad.cuh"

namespace d3d {

constexpr int GI_THREADS = 256;

template <typename T, int TYPE>
__global__ void __launch_bounds__(GI_THREADS) iou_ex_fwd_kernel(const T *__restrict__ b1, int64_t n, const T *__restrict__ b2, int64_t m, T *__restrict__ out, int64_t ld)
{
    const int64_t j = (int64_t)blockIdx.x * GI_THREADS + threadIdx.x, i = blockIdx.y;
    if (j >= m) return;
    const T *a = b1 + 5 * i;   // in the frame of the row box's centre
    const GBox<T> A = g_make<T>(a, a[0], a[1]), B = g_make<T>(b2 + 5 * j, a[0], a[1]);
    out[i * ld + j] = g_pair<T, TYPE, false>(A, B, T(0), nullptr, nullptr);
}

// SIDE 0: one warp per box of boxes1 (sums over the columns of its row), SIDE 1: one warp per box of boxes2 (sums over its column)
template <typename T, int TYPE, int SIDE>
__global__ void __launch_bounds__(GI_THREADS) iou_bwd_kernel(const T *__restrict__ b1, int64_t n, const T *__restrict__ b2, int64_t m, const T *__restrict__ grad, int64_t ld,
                                                             T *__restrict__ gout)
{
    const unsigned lane = threadIdx.x & 31u;
    const int64_t own = (int64_t)blockIdx.x * (GI_THREADS / 32) + (threadIdx.x >> 5);
    const int64_t nown = SIDE ? m : n, nother = SIDE ? n : m;
    if (own >= nown) return;
    const T *ob = (SIDE ? b2 : b1) + 5 * own, ox = ob[0], oy = ob[1];   // every pair in the frame of the owned box's centre
    const GBox<T> O = g_make<T>(ob, ox, oy);
    T acc[5] = {0, 0, 0, 0, 0};
    for (int64_t o = lane; o < nother; o += 32) {
        const T up = SIDE ? grad[o * ld + own] : grad[own * ld + o];
        if (up == T(0)) continue;
        const GBox<T> P = g_make<T>((SIDE ? b1 : b2) + 5 * o, ox, oy);
        T dump[5] = {0, 0, 0, 0, 0};
        if (SIDE) g_pair<T, TYPE, true>(P, O, up, dump, acc);
        else g_pair<T, TYPE, true>(O, P, up, acc, dump);
    }
#pragma unroll
    for (int k = 0; k < 5; k++) {
        T v = acc[k];
#pragma unroll
        for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
        if (lane == 0) gout[5 * own + k] = v;
    }
}

template <typename T, int TYPE>
static int iou_ex_fwd(const T *b1, int64_t n, const T *b2, int64_t m, T *out, int64_t ld, cudaStream_t st)
{
    if (n < 0 || m < 0 || ld < m) return D3D_ERR_INVALID_ARGUMENT;
    if (n == 0 || m == 0) return D3D_OK;
    if (!b1 || !b2 || !out || n > 0x7fffffffll) return D3D_ERR_INVALID_ARGUMENT;
    for (int64_t r0 = 0; r0 < n; r0 += 65535) {
        const int64_t rows = n - r0 < 65535 ? n - r0 : 65535;
        iou_ex_fwd_kernel<T, TYPE><<<dim3((unsigned)cdiv(m, GI_THREADS), (unsigned)rows), GI_THREADS, 0, st>>>(b1 + 5 * r0, rows, b2, m, out + r0 * ld, ld);
        D3D_LAUNCHED();
    }
    return D3D_OK;
}

template <typename T, int TYPE>
static int iou_bwd(const T *b1, int64_t n, const T *b2, int64_t m, const T *grad, int64_t ld, T *g1, T *g2, cudaStream_t st)
{
    if (n < 0 || m < 0 || ld < m) return D3D_ERR_INVALID_ARGUMENT;
    if ((n > 0 && !g1) || (m > 0 && !g2)) return D3D_ERR_INVALID_ARGUMENT;
    if (n == 0 || m == 0) {   // no pairs: zero gradients
        if (n > 0) D3D_CUDA_TRY(cudaMemsetAsync(g1, 0, (size_t)n * 5 * sizeof(T), st));
        if (m > 0) D3D_CUDA_TRY(cudaMemsetAsync(g2, 0, (size_t)m * 5 * sizeof(T), st));
        return D3D_OK;
    }
    if (!b1 || !b2 || !grad) return D3D_ERR_INVALID_ARGUMENT;
    iou_bwd_kernel<T, TYPE, 0><<<(unsigned)cdiv(n, GI_THREADS / 32), GI_THREADS, 0, st>>>(b1, n, b2, m, grad, ld, g1);
    D3D_LAUNCHED();
    iou_bwd_kernel<T, TYPE, 1><<<(unsigned)cdiv(m, GI_THREADS / 32), GI_THREADS, 0, st>>>(b1, n, b2, m, grad, ld, g2);
    D3D_LAUNCHED();
    return D3D_OK;
}

}  // namespace d3d

using namespace d3d;
#define D3D_FWD_ENTRY(NAME, T, TYPE)                                                                                                  \
    extern "C" int NAME(const T *boxes1, int64_t n, const T *boxes2, int64_t m, T *out, int64_t ld, void *stream)                     \
    { return iou_ex_fwd<T, TYPE>(boxes1, n, boxes2, m, out, ld, (cudaStream_t)stream); }
#define D3D_BWD_ENTRY(NAME, T, TYPE)                                                                                                  \
    extern "C" int NAME(const T *boxes1, int64_t n, const T *boxes2, int64_t m, const T *grad, int64_t ld, T *grad_boxes1,            \
                        T *grad_boxes2, void *stream)                                                                                 \
    { return iou_bwd<T, TYPE>(boxes1, n, boxes2, m, grad, ld, grad_boxes1, grad_boxes2, (cudaStream_t)stream); }
D3D_FWD_ENTRY(d3d_giou2dr_f32, float, GT_GIOU)
D3D_FWD_ENTRY(d3d_giou2dr_f64, double, GT_GIOU)
D3D_FWD_ENTRY(d3d_diou2dr_f32, float, GT_DIOU)
D3D_FWD_ENTRY(d3d_diou2dr_f64, double, GT_DIOU)
D3D_BWD_ENTRY(d3d_iou2d_backward_f32, float, GT_BOX)
D3D_BWD_ENTRY(d3d_iou2d_backward_f64, double, GT_BOX)
D3D_BWD_ENTRY(d3d_iou2dr_backward_f32, float, GT_RBOX)
D3D_BWD_ENTRY(d3d_iou2dr_backward_f64, double, GT_RBOX)
D3D_BWD_ENTRY(d3d_giou2dr_backward_f32, float, GT_GIOU)
D3D_BWD_ENTRY(d3d_giou2dr_backward_f64, double, GT_GIOU)
D3D_BWD_ENTRY(d3d_diou2dr_backward_f32, float, GT_DIOU)
D3D_BWD_ENTRY(d3d_diou2dr_backward_f64, double, GT_DIOU)
