// twin.cu -- TEST INFRASTRUCTURE: compiles the product's clip math (d3d_b200/csrc/geom.cuh), the pair math of the
// differentiable IoU family (d3d_b200/csrc/iou_grad.cuh) and of the point-to-box distance (d3d_b200/csrc/dist.cuh) as HOST
// code so the algorithm can be checked against the CPU oracle on a machine without a GPU.  Nothing in the product loads this library.
#include "../../d3d_b200/csrc/geom.cuh"
#include "../../d3d_b200/csrc/dist.cuh"
#include "../../d3d_b200/csrc/iou_grad.cuh"
using namespace d3d;
template <typename T> static void run(const T *b1, long n, const T *b2, long m, T *out, int aabb)
{
    for (long i = 0; i < n; i++)
        for (long j = 0; j < m; j++) {
            const T *p = b1 + 5 * i, *q = b2 + 5 * j;
            if (aabb) out[i * m + j] = aabb_iou(make_aabb_rec<T>(p[0], p[1], p[2], p[3], p[4]), make_aabb_rec<T>(q[0], q[1], q[2], q[3], q[4]));
            else {
                BoxRec<T> A = make_box_rec<T>(p[0], p[1], p[2], p[3], p[4]), B = make_box_rec<T>(q[0], q[1], q[2], q[3], q[4]);
                T ddx = A.cx - B.cx, ddy = A.cy - B.cy, rs = A.rho + B.rho;
                out[i * m + j] = (ddx * ddx + ddy * ddy <= rs * rs) ? rbox_iou<T>(A, B) : T(0);
            }
        }
}
extern "C" void twin_iou_f32(const float *b1, long n, const float *b2, long m, float *out, int aabb) { run<float>(b1, n, b2, m, out, aabb); }
extern "C" void twin_iou_f64(const double *b1, long n, const double *b2, long m, double *out, int aabb) { run<double>(b1, n, b2, m, out, aabb); }

// the differentiable family as iou_grad.cu runs it: values [n, m] as iou_ex_fwd_kernel computes them and, for the upstream gradient
// `up` [n, m], the gradient sums g1 [n, 5] and g2 [m, 5] as iou_bwd_kernel computes them (one owned box against the other side)
template <typename T, int TYPE> static void run_ex(const T *b1, long n, const T *b2, long m, const T *up, T *out, T *g1, T *g2)
{
    for (long i = 0; i < n; i++)
        for (long j = 0; j < m; j++)
            out[i * m + j] = g_pair<T, TYPE, false>(g_make<T>(b1 + 5 * i, b1[5 * i], b1[5 * i + 1]), g_make<T>(b2 + 5 * j, b1[5 * i], b1[5 * i + 1]),
                                                    T(0), nullptr, nullptr);
    for (long s = 0; s < 2; s++)
        for (long o = 0; o < (s ? m : n); o++) {
            const T *own = (s ? b2 : b1) + 5 * o;
            const GBox<T> O = g_make<T>(own, own[0], own[1]);
            T acc[5] = {0, 0, 0, 0, 0};
            for (long p = 0; p < (s ? n : m); p++) {
                const T u = s ? up[p * m + o] : up[o * m + p];
                if (u == T(0)) continue;
                const GBox<T> P = g_make<T>((s ? b1 : b2) + 5 * p, own[0], own[1]);
                T dump[5] = {0, 0, 0, 0, 0};
                if (s) g_pair<T, TYPE, true>(P, O, u, dump, acc);
                else g_pair<T, TYPE, true>(O, P, u, acc, dump);
            }
            for (int k = 0; k < 5; k++) (s ? g2 : g1)[5 * o + k] = acc[k];
        }
}
template <typename T> static void run_ex_type(const T *b1, long n, const T *b2, long m, int type, const T *up, T *out, T *g1, T *g2)
{
    if (type == GT_BOX) run_ex<T, GT_BOX>(b1, n, b2, m, up, out, g1, g2);
    else if (type == GT_RBOX) run_ex<T, GT_RBOX>(b1, n, b2, m, up, out, g1, g2);
    else if (type == GT_GIOU) run_ex<T, GT_GIOU>(b1, n, b2, m, up, out, g1, g2);
    else run_ex<T, GT_DIOU>(b1, n, b2, m, up, out, g1, g2);
}
extern "C" void twin_iou_ex_f32(const float *b1, long n, const float *b2, long m, int type, const float *up, float *out, float *g1, float *g2)
{ run_ex_type<float>(b1, n, b2, m, type, up, out, g1, g2); }
extern "C" void twin_iou_ex_f64(const double *b1, long n, const double *b2, long m, int type, const double *up, double *out, double *g1, double *g2)
{ run_ex_type<double>(b1, n, b2, m, type, up, out, g1, g2); }

// the point-to-box distance as dist.cu runs it: values and edge indices [m boxes, n points] as pdist_fwd_kernel computes them and, for
// the upstream gradient `up` [m, n], the gradient sums gp [n, 2] and gb [m, 5] of pdist_bwd_kernel
template <typename T> static void run_pd(const T *pts, long n, const T *boxes, long m, const T *up, T *out, unsigned char *edge, T *gp, T *gb)
{
    for (long j = 0; j < 2 * n; j++) gp[j] = T(0);
    for (long i = 0; i < m; i++) {
        const PBox<T> b = pd_box<T>(boxes + 5 * i);
        T acc[5] = {0, 0, 0, 0, 0};
        for (long j = 0; j < n; j++) {
            int e;
            out[i * n + j] = pd_pair<T, false>(b, pts[2 * j], pts[2 * j + 1], &e, T(0), nullptr, nullptr);
            edge[i * n + j] = (unsigned char)e;
            pd_pair<T, true>(b, pts[2 * j], pts[2 * j + 1], &e, up[i * n + j], gp + 2 * j, acc);
        }
        for (int k = 0; k < 5; k++) gb[5 * i + k] = acc[k];
    }
}
extern "C" void twin_pdist_f32(const float *pts, long n, const float *boxes, long m, const float *up, float *out, unsigned char *edge, float *gp, float *gb)
{ run_pd<float>(pts, n, boxes, m, up, out, edge, gp, gb); }
extern "C" void twin_pdist_f64(const double *pts, long n, const double *boxes, long m, const double *up, double *out, unsigned char *edge, double *gp, double *gb)
{ run_pd<double>(pts, n, boxes, m, up, out, edge, gp, gb); }
