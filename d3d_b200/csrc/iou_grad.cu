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

// SIDE 0: one warp per box of boxes1 (sums over the columns of its row), SIDE 1: one warp per box of boxes2 (sums over its column).
// The warp of box `own` (< n or < m) walks the other side with its lanes in a fixed order, so a box's five sums do not depend on the
// kernel that runs this body: the single-matrix kernel and the frame-batched kernel give the same bits.
template <typename T, int TYPE, int SIDE>
__device__ __forceinline__ void iou_bwd_own(const T *__restrict__ b1, int64_t n, const T *__restrict__ b2, int64_t m, const T *__restrict__ grad,
                                            int64_t ld, T *__restrict__ gout, const int64_t own, const unsigned lane)
{
    const int64_t nother = SIDE ? n : m;
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

template <typename T, int TYPE, int SIDE>
__global__ void __launch_bounds__(GI_THREADS) iou_bwd_kernel(const T *__restrict__ b1, int64_t n, const T *__restrict__ b2, int64_t m, const T *__restrict__ grad, int64_t ld,
                                                             T *__restrict__ gout)
{
    const int64_t own = (int64_t)blockIdx.x * (GI_THREADS / 32) + (threadIdx.x >> 5);
    if (own >= (SIDE ? m : n)) return;
    iou_bwd_own<T, TYPE, SIDE>(b1, n, b2, m, grad, ld, gout, own, threadIdx.x & 31u);
}

// ------------------------------------------------------------------ frame-batched (box2d_iou_batch)
// Frame f owns boxes [off1[f], off1[f+1]) and [off2[f], off2[f+1]) of the packed inputs; its n_f x m_f block (leading dimension m_f) is at
// out + out_off[f].  Frames on grid.x; the threads of grid.y stride over the frame's n_f * m_f pairs, row-major, so that a frame with a
// few dozen columns still fills its CTAs and the stores stay contiguous.
template <typename T, int TYPE>
__global__ void __launch_bounds__(GI_THREADS) iou_ex_fwd_batch_kernel(const T *__restrict__ b1, const int64_t *__restrict__ off1, const T *__restrict__ b2,
                                                                      const int64_t *__restrict__ off2, const int64_t *__restrict__ out_off, T *__restrict__ out)
{
    const int64_t f = blockIdx.x, a0 = off1[f], c0 = off2[f], n = off1[f + 1] - a0, m = off2[f + 1] - c0, np = n * m;
    const T *fb1 = b1 + 5 * a0, *fb2 = b2 + 5 * c0;
    T *o = out + out_off[f];
    for (int64_t p = (int64_t)blockIdx.y * GI_THREADS + threadIdx.x; p < np; p += (int64_t)gridDim.y * GI_THREADS) {
        const int64_t i = p / m, j = p - i * m;
        const T *a = fb1 + 5 * i;   // iou_ex_fwd_kernel's pair code: in the frame of the row box's centre
        const GBox<T> A = g_make<T>(a, a[0], a[1]), B = g_make<T>(fb2 + 5 * j, a[0], a[1]);
        o[p] = g_pair<T, TYPE, false>(A, B, T(0), nullptr, nullptr);
    }
}

// iou_bwd_own behind a call: its arguments are opaque to the compiler, as iou_bwd_kernel's parameters are, so the body compiles to the
// same arithmetic (the same contractions into FMA) as in iou_bwd_kernel, where it is inlined
template <typename T, int TYPE, int SIDE>
__device__ __noinline__ void iou_bwd_own_call(const T *__restrict__ b1, int64_t n, const T *__restrict__ b2, int64_t m, const T *__restrict__ grad,
                                              int64_t ld, T *__restrict__ gout, const int64_t own)
{
    if (own >= (SIDE ? m : n)) return;
    iou_bwd_own<T, TYPE, SIDE>(b1, n, b2, m, grad, ld, gout, own, threadIdx.x & 31u);
}

// one warp per owned box of a frame: frames on grid.x, the frame's owned boxes in blocks of 8 on grid.y + 65535 * grid.z; a box of a frame
// whose other side is empty gets exact zeros
template <typename T, int TYPE, int SIDE>
__global__ void __launch_bounds__(GI_THREADS, sizeof(T) == 8 ? 1 : 2) iou_bwd_batch_kernel(const T *__restrict__ b1, const int64_t *__restrict__ off1, const T *__restrict__ b2,
                                                                   const int64_t *__restrict__ off2, const int64_t *__restrict__ out_off,
                                                                   const T *__restrict__ grad, T *__restrict__ gout)
{
    const int64_t f = blockIdx.x, a0 = off1[f], c0 = off2[f], n = off1[f + 1] - a0, m = off2[f + 1] - c0;
    const int64_t own = ((int64_t)blockIdx.y + (int64_t)blockIdx.z * 65535) * (GI_THREADS / 32) + (threadIdx.x >> 5);
    if (own < (SIDE ? m : n)) iou_bwd_own_call<T, TYPE, SIDE>(b1 + 5 * a0, n, b2 + 5 * c0, m, grad + out_off[f], m, gout + 5 * (SIDE ? c0 : a0), own);
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

template <typename T>
int iou_ex_batch_fwd(const T *b1, const int64_t *off1, const T *b2, const int64_t *off2, int64_t nframes, int64_t max_pairs, int iou_type,
                     const int64_t *out_off, T *out, cudaStream_t st)
{
    const dim3 grid((unsigned)nframes, stride_blocks(max_pairs, GI_THREADS));
    if (iou_type == D3D_IOU_GRBOX) iou_ex_fwd_batch_kernel<T, GT_GIOU><<<grid, GI_THREADS, 0, st>>>(b1, off1, b2, off2, out_off, out);
    else iou_ex_fwd_batch_kernel<T, GT_DIOU><<<grid, GI_THREADS, 0, st>>>(b1, off1, b2, off2, out_off, out);
    D3D_LAUNCHED();
    return D3D_OK;
}
template int iou_ex_batch_fwd<float>(const float *, const int64_t *, const float *, const int64_t *, int64_t, int64_t, int, const int64_t *, float *,
                                     cudaStream_t);
template int iou_ex_batch_fwd<double>(const double *, const int64_t *, const double *, const int64_t *, int64_t, int64_t, int, const int64_t *,
                                      double *, cudaStream_t);

template <typename T, int TYPE>
static int iou_bwd_batch_launch(const T *b1, const int64_t *off1, const T *b2, const int64_t *off2, unsigned nf, int64_t max1, int64_t max2,
                                const int64_t *out_off, const T *grad, T *g1, T *g2, cudaStream_t st)
{
    const int64_t blocks1 = cdiv(max1, GI_THREADS / 32), blocks2 = cdiv(max2, GI_THREADS / 32);   // <= 2^60: grid.z <= 65535 for any real frame
    iou_bwd_batch_kernel<T, TYPE, 0><<<dim3(nf, stride_blocks(blocks1, 1), (unsigned)cdiv(blocks1, 65535)), GI_THREADS, 0, st>>>(b1, off1, b2, off2, out_off,
                                                                                                                              grad, g1);
    D3D_LAUNCHED();
    iou_bwd_batch_kernel<T, TYPE, 1><<<dim3(nf, stride_blocks(blocks2, 1), (unsigned)cdiv(blocks2, 65535)), GI_THREADS, 0, st>>>(b1, off1, b2, off2, out_off,
                                                                                                                              grad, g2);
    D3D_LAUNCHED();
    return D3D_OK;
}

// both gradients of every frame of a packed batch: two launches whatever the number of frames
template <typename T>
static int iou_bwd_batch(const T *b1, int64_t total1, const int64_t *off1, const T *b2, int64_t total2, const int64_t *off2, int64_t nframes,
                         int64_t max1, int64_t max2, int iou_type, const int64_t *out_off, const T *grad, T *g1, T *g2, cudaStream_t st)
{
    if (iou_type != D3D_IOU_BOX && iou_type != D3D_IOU_RBOX && iou_type != D3D_IOU_GRBOX && iou_type != D3D_IOU_DRBOX) return D3D_ERR_INVALID_ARGUMENT;
    if (total1 < 0 || total2 < 0 || nframes < 0 || max1 < 0 || max2 < 0) return D3D_ERR_INVALID_ARGUMENT;
    if (nframes == 0) return D3D_OK;
    if ((total1 > 0 && !g1) || (total2 > 0 && !g2)) return D3D_ERR_INVALID_ARGUMENT;
    if (total1 == 0 || total2 == 0) {   // no pairs: zero gradients
        if (total1 > 0) D3D_CUDA_TRY(cudaMemsetAsync(g1, 0, (size_t)total1 * 5 * sizeof(T), st));
        if (total2 > 0) D3D_CUDA_TRY(cudaMemsetAsync(g2, 0, (size_t)total2 * 5 * sizeof(T), st));
        return D3D_OK;
    }
    if (!b1 || !b2 || !off1 || !off2 || !out_off || !grad) return D3D_ERR_INVALID_ARGUMENT;
    if (nframes > 0x7fffffffll) return D3D_ERR_UNSUPPORTED;
    if (max1 == 0) max1 = total1;   // 0: bound unknown
    if (max2 == 0) max2 = total2;
    const unsigned nf = (unsigned)nframes;
    switch (iou_type) {
    case D3D_IOU_BOX: return iou_bwd_batch_launch<T, GT_BOX>(b1, off1, b2, off2, nf, max1, max2, out_off, grad, g1, g2, st);
    case D3D_IOU_RBOX: return iou_bwd_batch_launch<T, GT_RBOX>(b1, off1, b2, off2, nf, max1, max2, out_off, grad, g1, g2, st);
    case D3D_IOU_GRBOX: return iou_bwd_batch_launch<T, GT_GIOU>(b1, off1, b2, off2, nf, max1, max2, out_off, grad, g1, g2, st);
    default: return iou_bwd_batch_launch<T, GT_DIOU>(b1, off1, b2, off2, nf, max1, max2, out_off, grad, g1, g2, st);
    }
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
#define D3D_BATCH_BWD_ENTRY(NAME, T)                                                                                                  \
    extern "C" int NAME(const T *boxes1, int64_t total1, const int64_t *offsets1, const T *boxes2, int64_t total2, const int64_t *offsets2, \
                        int64_t nframes, int64_t max_frame1, int64_t max_frame2, int iou_type, const int64_t *out_offsets, const T *grad,  \
                        T *grad_boxes1, T *grad_boxes2, void *stream)                                                                 \
    {                                                                                                                                 \
        return iou_bwd_batch<T>(boxes1, total1, offsets1, boxes2, total2, offsets2, nframes, max_frame1, max_frame2, iou_type,        \
                                out_offsets, grad, grad_boxes1, grad_boxes2, (cudaStream_t)stream);                                   \
    }
D3D_BATCH_BWD_ENTRY(d3d_box2d_iou_batch_backward_f32, float)
D3D_BATCH_BWD_ENTRY(d3d_box2d_iou_batch_backward_f64, double)
