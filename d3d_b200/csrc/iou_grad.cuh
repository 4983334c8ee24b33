// iou_grad.cuh -- pair math of the differentiable IoU family (iou_grad.cu): corners of a box, the clip of one box against the other
// with the boundary-motion gradient, the convex hull of GIoU, the diameter of DIoU, and the chain from corner gradients to (x, y, w, h, r).
// D3D_HD like geom.cuh, so that the CPU test-suite can compile the same code as host code.
#pragma once
#include "geom.cuh"

namespace d3d {

enum { GT_BOX = 0, GT_RBOX = 1, GT_GIOU = 2, GT_DIOU = 3 };

template <typename T> struct GBox { T x, y, w, h, cr, sr, vx[4], vy[4]; };
template <typename T> struct GTol;
template <> struct GTol<float> { static constexpr float v = 1e-6f; };
template <> struct GTol<double> { static constexpr double v = 1e-13; };

// the box b in the frame whose origin is (ox, oy).  The pair code takes every box relative to one of the pair's centres: its shoelace
// sums and products of corner coordinates then stay at the scale of the boxes however far they are from the origin (75 m at sensor
// scale, 1e5 m in a map frame), where absolute coordinates cancel to the point of noise.  Values are translation invariant, so the
// gradients taken in that frame are the gradients in the caller's.
template <typename T>
D3D_HD GBox<T> g_make(const T *b, T ox, T oy)
{
    GBox<T> q;
    q.x = b[0] - ox; q.y = b[1] - oy; q.w = b[2]; q.h = b[3];
    q.sr = sin(b[4]); q.cr = cos(b[4]);
    const T dxsin = q.w * q.sr / 2, dxcos = q.w * q.cr / 2, dysin = q.h * q.sr / 2, dycos = q.h * q.cr / 2;   // geometry.hpp:417-429
    q.vx[0] = q.x - dxcos + dysin; q.vy[0] = q.y - dxsin - dycos;
    q.vx[1] = q.x + dxcos + dysin; q.vy[1] = q.y + dxsin - dycos;
    q.vx[2] = q.x + dxcos - dysin; q.vy[2] = q.y + dxsin + dycos;
    q.vx[3] = q.x - dxcos - dysin; q.vy[3] = q.y - dxsin + dycos;
    return q;
}

// vertex gradients -> (x, y, w, h, r): v_k = c + s_k (w/2) u + t_k (h/2) v with u = (cos r, sin r), v = (-sin r, cos r)
template <typename T>
D3D_HD void g_chain(const GBox<T> &b, const T gx[4], const T gy[4], T scale, T g[5])
{
    const T sk[4] = {-1, 1, 1, -1}, tk[4] = {-1, -1, 1, 1};
#pragma unroll
    for (int v = 0; v < 4; v++) {
        const T ax = scale * gx[v], ay = scale * gy[v];
        g[0] += ax; g[1] += ay;
        g[2] += sk[v] * T(0.5) * (ax * b.cr + ay * b.sr);
        g[3] += tk[v] * T(0.5) * (-ax * b.sr + ay * b.cr);
        g[4] += ax * (-sk[v] * T(0.5) * b.w * b.sr - tk[v] * T(0.5) * b.h * b.cr) + ay * (sk[v] * T(0.5) * b.w * b.cr - tk[v] * T(0.5) * b.h * b.sr);
    }
}

// record of geom.cuh's rotated IoU for a box of this frame
template <typename T>
D3D_HD BoxRec<T> g_rec(const GBox<T> &b)
{
    BoxRec<T> r;
    r.cx = b.x; r.cy = b.y; r.c = b.cr; r.s = b.sr;
    r.hw = T(0.5) * Num<T>::abs_(b.w); r.hh = T(0.5) * Num<T>::abs_(b.h);
    r.rho = 0; r.area = Num<T>::abs_(b.w) * Num<T>::abs_(b.h);
    return r;
}

// pieces of P's edges inside Q: the boundary-motion gradient on P's vertices (added).  Only the gradient: where two edges are nearly
// parallel the crossing parameter c0 / (c0 - c1) carries a rounding error of order ulp / angle, the pieces of the two passes then do not
// meet, and their shoelace sum would not be the area of one polygon (the value comes from rbox_iou instead, see g_pair)
// `closed`: points ON Q's boundary count as inside (the pass over A's edges) or as outside (the pass over B's), so that edges the two
// boxes share -- identical boxes above all -- are counted once.  An edge on the line of one of Q's edges but running against it has P
// and Q on opposite sides of that line: the boxes touch there and share no area, so it is outside in both passes and both gradients are
// zero there (in one pass only, one box alone would get the gradient of a segment)
template <typename T>
D3D_HD void g_clip(const GBox<T> &P, const GBox<T> &Q, bool closed, T gx[4], T gy[4])
{
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int k1 = (k + 1) & 3;
        const T p0x = P.vx[k], p0y = P.vy[k], ex = P.vx[k1] - p0x, ey = P.vy[k1] - p0y;
        T t0 = 0, t1 = 1;
#pragma unroll
        for (int m = 0; m < 4; m++) {
            const int m1 = (m + 1) & 3;
            const T nx = Q.vx[m1] - Q.vx[m], ny = Q.vy[m1] - Q.vy[m];
            const T c0 = nx * (p0y - Q.vy[m]) - ny * (p0x - Q.vx[m]);   // > 0: left of Q's edge = inside
            const T c1 = c0 + nx * ey - ny * ex;
            const T band = GTol<T>::v * (nx * nx + ny * ny + ex * ex + ey * ey), lim = closed ? -band : band;
            if ((c0 < lim && c1 < lim) || (fabs(c0) <= band && fabs(c1) <= band && nx * ex + ny * ey < 0)) { t0 = 1; t1 = 0; }
            else if (c0 < lim) t0 = fmax(t0, c0 / (c0 - c1));
            else if (c1 < lim) t1 = fmin(t1, c0 / (c0 - c1));
        }
        if (t1 > t0) {
            const T sq = T(0.5) * (t1 * t1 - t0 * t0), w0 = (t1 - t0) - sq;
            gx[k] += ey * w0; gy[k] -= ex * w0;
            gx[k1] += ey * sq; gy[k1] -= ex * sq;
        }
    }
}

// area of the convex hull of the eight vertices (GIoU's merge, geometry.hpp:1021-1122) and its gradient on the vertices: Andrew's
// monotone chain over the vertices sorted by (x, y).  Every decision is the sign of one orientation, and a vertex that is not strictly
// left of the chain (coincident or collinear corners included) is dropped, so the edges always form one polygon.  Deciding each directed
// pair on its own, with a tolerance per pair, could take two overlapping edges across three nearly collinear corners.
template <typename T, bool GRAD>
D3D_HD T g_hull(const T px[8], const T py[8], T gx[8], T gy[8])
{
    int o[8] = {0, 1, 2, 3, 4, 5, 6, 7};
    // Batcher's odd-even merge sort of 8 keys: 19 compare-exchanges
    const int net[19][2] = {{0, 1}, {2, 3}, {4, 5}, {6, 7}, {0, 2}, {1, 3}, {4, 6}, {5, 7}, {1, 2}, {5, 6},
                            {0, 4}, {1, 5}, {2, 6}, {3, 7}, {2, 4}, {3, 5}, {1, 2}, {3, 4}, {5, 6}};
#pragma unroll
    for (int c = 0; c < 19; c++) {
        const int i = o[net[c][0]], j = o[net[c][1]];
        if (px[j] < px[i] || (px[j] == px[i] && py[j] < py[i])) { o[net[c][0]] = j; o[net[c][1]] = i; }
    }
    auto left = [&](int a, int b, int q) { return (px[b] - px[a]) * (py[q] - py[a]) - (py[b] - py[a]) * (px[q] - px[a]) > 0; };
    // lower chain left to right, then upper chain right to left; h[k - 1] == h[0] closes the polygon
    int h[16], k = 0;
    for (int s = 0; s < 8; s++) {
        while (k >= 2 && !left(h[k - 2], h[k - 1], o[s])) k--;
        h[k++] = o[s];
    }
    for (int s = 6, lo = k + 1; s >= 0; s--) {
        while (k >= lo && !left(h[k - 2], h[k - 1], o[s])) k--;
        h[k++] = o[s];
    }
    T area2 = 0;
    for (int e = 0; e + 1 < k; e++) {
        const int i = h[e], j = h[e + 1];
        area2 += px[i] * py[j] - py[i] * px[j];
        if (GRAD) { gx[i] += T(0.5) * py[j]; gy[i] -= T(0.5) * px[j]; gx[j] -= T(0.5) * py[i]; gy[j] += T(0.5) * px[i]; }
    }
    return T(0.5) * area2;
}

// value of one pair and, when GRAD, its gradient with respect to both boxes (ga, gb are ADDED to, scaled by `up`)
template <typename T, int TYPE, bool GRAD>
D3D_HD T g_pair(const GBox<T> &A, const GBox<T> &B, T up, T ga[5], T gb[5])
{
    if (TYPE == GT_BOX) {   // IoU of the axis-aligned bounding boxes (geometry.hpp:398-414, 513-529, 1206-1212)
        T lo[2][2], hi[2][2];
        int ilo[2][2], ihi[2][2];
#pragma unroll
        for (int s = 0; s < 2; s++) {
            const GBox<T> &P = s ? B : A;
#pragma unroll
            for (int d = 0; d < 2; d++) {
                const T *v = d ? P.vy : P.vx;
                lo[s][d] = v[0]; hi[s][d] = v[0]; ilo[s][d] = 0; ihi[s][d] = 0;
#pragma unroll
                for (int k = 1; k < 4; k++) {
                    if (v[k] < lo[s][d]) { lo[s][d] = v[k]; ilo[s][d] = k; }
                    if (v[k] > hi[s][d]) { hi[s][d] = v[k]; ihi[s][d] = k; }
                }
            }
        }
        const T ix0 = fmax(lo[0][0], lo[1][0]), ix1 = fmin(hi[0][0], hi[1][0]), iy0 = fmax(lo[0][1], lo[1][1]), iy1 = fmin(hi[0][1], hi[1][1]);
        const bool ov = ix1 > ix0 && iy1 > iy0;
        const T I = ov ? (ix1 - ix0) * (iy1 - iy0) : T(0);
        const T a0 = (hi[0][0] - lo[0][0]) * (hi[0][1] - lo[0][1]), a1 = (hi[1][0] - lo[1][0]) * (hi[1][1] - lo[1][1]);
        const T U = a0 + a1 - I;
        if (!(U > 0)) return T(0);
        const T f = I / U;
        if (GRAD) {
            // f = I/U: df = ((a0 + a1) dI - I (da0 + da1)) / U^2; every extent is one coordinate of one vertex
            const T cI = up * (a0 + a1) / (U * U), cA = -up * I / (U * U);
#pragma unroll
            for (int s = 0; s < 2; s++) {
                const GBox<T> &P = s ? B : A;
                T gx[4] = {0, 0, 0, 0}, gy[4] = {0, 0, 0, 0};
                const T wx = hi[s][0] - lo[s][0], wy = hi[s][1] - lo[s][1];
                gx[ihi[s][0]] += cA * wy; gx[ilo[s][0]] -= cA * wy; gy[ihi[s][1]] += cA * wx; gy[ilo[s][1]] -= cA * wx;
                if (ov) {
                    const int o = 1 - s;
                    if (hi[s][0] < hi[o][0] || (hi[s][0] == hi[o][0] && s == 0)) gx[ihi[s][0]] += cI * (iy1 - iy0);
                    if (lo[s][0] > lo[o][0] || (lo[s][0] == lo[o][0] && s == 0)) gx[ilo[s][0]] -= cI * (iy1 - iy0);
                    if (hi[s][1] < hi[o][1] || (hi[s][1] == hi[o][1] && s == 0)) gy[ihi[s][1]] += cI * (ix1 - ix0);
                    if (lo[s][1] > lo[o][1] || (lo[s][1] == lo[o][1] && s == 0)) gy[ilo[s][1]] -= cI * (ix1 - ix0);
                }
                g_chain<T>(P, gx, gy, T(1), s ? gb : ga);
            }
        }
        return f;
    }
    // I / U is geom.cuh's rotated IoU (a continuous integral over the clamped boundary, exact to rounding also for touching, flush and
    // nearly parallel edges); I and U follow from it and the two areas
    const T aA = A.w * A.h, aB = B.w * B.h, iou = rbox_iou<T>(g_rec(A), g_rec(B));
    const T U = (aA + aB) / (1 + iou), I = iou * U;
    if (!(U > 0)) return T(0);
    T f = iou;
    T gax[4] = {0, 0, 0, 0}, gay[4] = {0, 0, 0, 0}, gbx[4] = {0, 0, 0, 0}, gby[4] = {0, 0, 0, 0};
    if (GRAD) { g_clip<T>(A, B, true, gax, gay); g_clip<T>(B, A, false, gbx, gby); }
    // d(I/U) = ((aA + aB) dI - I (daA + daB)) / U^2
    const T cI = (aA + aB) / (U * U), cArea = -I / (U * U);
    T cM = 0, cU2 = 0, M = 0;       // GIoU: + U/M - 1
    T hx[8], hy[8];
    if (TYPE == GT_GIOU) {
        T px[8], py[8];
#pragma unroll
        for (int k = 0; k < 4; k++) { px[k] = A.vx[k]; py[k] = A.vy[k]; px[4 + k] = B.vx[k]; py[4 + k] = B.vy[k]; hx[k] = hy[k] = hx[4 + k] = hy[4 + k] = 0; }
        M = g_hull<T, GRAD>(px, py, hx, hy);
        if (M > 0) { f += U / M - 1; cU2 = 1 / M; cM = -U / (M * M); }
    }
    T cd2 = 0, md2 = 0;
    int ia = 0, ib = 0;
    if (TYPE == GT_DIOU) {
        T px[8], py[8];
#pragma unroll
        for (int k = 0; k < 4; k++) { px[k] = A.vx[k]; py[k] = A.vy[k]; px[4 + k] = B.vx[k]; py[4 + k] = B.vy[k]; }
        for (int i = 0; i < 8; i++)
            for (int j = i + 1; j < 8; j++) {
                const T dx = px[i] - px[j], dy = py[i] - py[j], d2 = dx * dx + dy * dy;
                if (d2 > md2) { md2 = d2; ia = i; ib = j; }
            }
        cd2 = (A.x - B.x) * (A.x - B.x) + (A.y - B.y) * (A.y - B.y);
        if (md2 > 0) f -= cd2 / md2;
    }
    if (GRAD) {
        // I/U part (+ the U part of GIoU: dU = daA + daB - dI)
        const T kI = up * (cI - cU2), kA = up * (cArea + cU2);
        g_chain<T>(A, gax, gay, kI, ga);
        g_chain<T>(B, gbx, gby, kI, gb);
        ga[2] += kA * A.h; ga[3] += kA * A.w; gb[2] += kA * B.h; gb[3] += kA * B.w;
        if (TYPE == GT_GIOU && M > 0) {
            g_chain<T>(A, hx, hy, up * cM, ga);
            g_chain<T>(B, hx + 4, hy + 4, up * cM, gb);
        }
        if (TYPE == GT_DIOU && md2 > 0) {
            // - cd2/md2: d = -(dcd2 md2 - cd2 dmd2) / md2^2
            const T k1 = -up / md2, k2 = up * cd2 / (md2 * md2);
            ga[0] += k1 * 2 * (A.x - B.x); ga[1] += k1 * 2 * (A.y - B.y); gb[0] -= k1 * 2 * (A.x - B.x); gb[1] -= k1 * 2 * (A.y - B.y);
            T vx[8] = {0, 0, 0, 0, 0, 0, 0, 0}, vy[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            const T pax = ia < 4 ? A.vx[ia] : B.vx[ia - 4], pay = ia < 4 ? A.vy[ia] : B.vy[ia - 4];
            const T pbx = ib < 4 ? A.vx[ib] : B.vx[ib - 4], pby = ib < 4 ? A.vy[ib] : B.vy[ib - 4];
            vx[ia] += 2 * (pax - pbx); vy[ia] += 2 * (pay - pby); vx[ib] -= 2 * (pax - pbx); vy[ib] -= 2 * (pay - pby);
            g_chain<T>(A, vx, vy, k2, ga);
            g_chain<T>(B, vx + 4, vy + 4, k2, gb);
        }
    }
    return f;
}

}  // namespace d3d
