// dist.cuh -- pair math of the signed point-to-box distance (dist.cu): the value, the edge that realises it and its analytic gradient in
// the point and in (x, y, w, h, r).  D3D_HD like geom.cuh, so that the CPU test-suite can compile the same code as host code.
//
// The box is the closed rectangle with half extents |w|/2, |h|/2 turned by r; the value is the signed Euclidean distance to its boundary,
// positive inside.  Every pair is evaluated in the box's own frame, q = R(-r) (p - c): there the box is axis-aligned and centred, so the
// value needs no line through two corners (whose coefficients cancel far from the origin and vanish at headings of pi / 2) and no
// decision between equal candidates on the sign.
#pragma once
#include "geom.cuh"

namespace d3d {

// centre, cos r, sin r, signed half extents w / 2 and h / 2 (the signs fix which edge of the quad lies on which side)
template <typename T> struct PBox { T x, y, c, s, hx, hy; };

template <typename T>
D3D_HD PBox<T> pd_box(const T *b)
{
    PBox<T> q;
    q.x = b[0]; q.y = b[1]; q.c = cos(b[4]); q.s = sin(b[4]);
    q.hx = b[2] / 2; q.hy = b[3] / 2;
    return q;
}

// Signed distance from (px, py) to box b; *edge = k of the edge v_k -> v_k+1 of pd_quad's vertex order (v_k = c + s_k w/2 u + t_k h/2 v,
// s = (-1, 1, 1, -1), t = (-1, -1, 1, 1)) that realises it: edges 1 and 3 lie at local x = +w/2 and -w/2, edges 0 and 2 at y = -h/2 and
// +h/2.  Equal distances go to the first edge of the loop order 3, 0, 1, 2; outside, a corner belongs to both of its edges.
// With GRAD, up * dD/d(point) is added to gp[2] and up * dD/d(x, y, w, h, r) to gb[5]: the gradient of the distance to the reported edge.
template <typename T, bool GRAD>
D3D_HD T pd_pair(const PBox<T> &b, T px, T py, int *edge, T up, T gp[2], T gb[5])
{
    const T dx = px - b.x, dy = py - b.y;
    const T qx = b.c * dx + b.s * dy, qy = b.c * dy - b.s * dx;
    const T hw = fabs(b.hx), hh = fabs(b.hy);
    const T ex = fabs(qx) - hw, ey = fabs(qy) - hh;
    // the nearer edge of each pair of parallel edges; on the centre line (or for a zero extent) both are as near and 3 (0) comes first
    const int ix = ((qx > 0 && b.hx > 0) || (qx < 0 && b.hx < 0)) ? 1 : 3;
    const int iy = ((qy > 0 && b.hy > 0) || (qy < 0 && b.hy < 0)) ? 2 : 0;
    const bool inside = ex <= 0 && ey <= 0;
    const bool tie = inside ? ex == ey : (ex >= 0 && ey >= 0);
    const bool onx = tie ? (ix == 3 || iy == 2) : ex > ey;
    *edge = onx ? ix : iy;
    T d, gqx = 0, gqy = 0, ghw = 0, ghh = 0;
    if (inside) {
        d = -(onx ? ex : ey);
        if (GRAD) {
            // D = hw - sx qx with sx the side of the reported edge (+1 for edge 1 when w >= 0)
            const T sx = (ix == 1) == (b.hx >= 0) ? T(1) : T(-1), sy = (iy == 2) == (b.hy >= 0) ? T(1) : T(-1);
            if (onx) { gqx = -sx; ghw = 1; }
            else { gqy = -sy; ghh = 1; }
        }
    } else {
        const T ux = ex > 0 ? ex : T(0), uy = ey > 0 ? ey : T(0);
        const T n = hypot(ux, uy);
        d = -n;
        if (GRAD && n > 0) {
            const T nx = ux / n, ny = uy / n;
            gqx = qx < 0 ? nx : -nx; gqy = qy < 0 ? ny : -ny;
            ghw = nx; ghh = ny;
        }
    }
    if (GRAD) {
        const T gx = b.c * gqx - b.s * gqy, gy = b.s * gqx + b.c * gqy;   // R(r) dD/dq
        gp[0] += up * gx; gp[1] += up * gy;
        gb[0] -= up * gx; gb[1] -= up * gy;
        gb[2] += up * (b.hx < 0 ? T(-0.5) : T(0.5)) * ghw;
        gb[3] += up * (b.hy < 0 ? T(-0.5) : T(0.5)) * ghh;
        gb[4] += up * (gqx * qy - gqy * qx);                             // dq/dr = (qy, -qx)
    }
    return d;
}

}  // namespace d3d
