// crop.cu -- point-in-rotated-box mask (SURVEY.md 8(f) row f4).
//
// Replaces reference crop_2dr (d3d/box/utils.h:45, utils.cpp:10-47; the reference has no CUDA version of it): for M boxes
// and N points, mask[i][j] = the AABB of box i strictly contains point j AND no edge of the quad has the point on its
// right (dgal Poly2::contains, thirdparty/dgal/geometry.hpp:218-229 over _cross :160-163; vertices as
// poly2_from_xywhr :417-429, bounding box as aabox2_from_poly2 :398-414 with the open test of :185-188).
//
// Layout / roofline: the output is bool[M, N] row-major = 1 byte per pair; a thread owns 16 consecutive points and
// writes their 16 mask bytes of one box as a single 16-byte store, a warp writes 512 contiguous bytes of a mask row.
// The box tile's 12 numbers per box (4 vertices + AABB) sit in shared memory.  ~35 flops per pair against 1 stored
// byte: FP32 issue bound for float (59 TFLOP/s -> ~1.7 T pairs/s), nearer the HBM store stream for small M.
// The per-pair arithmetic uses the explicit round-to-nearest intrinsics: the reference is compiled without FMA
// contraction and the mask is compared bit for bit.
#include "common.cuh"
#include "prims.cuh"
#include <stdlib.h>
#include <mutex>

namespace d3d {

template <typename T> struct CropBox { T vx[4], vy[4], minx, maxx, miny, maxy; };

template <typename T>
__device__ __forceinline__ CropBox<T> crop_prep_one(T x, T y, T w, T h, T r)
{
    T sn, cs;
    if (sizeof(T) == 4) { sn = (T)sinf((float)r); cs = (T)cosf((float)r); } else { sn = (T)sin((double)r); cs = (T)cos((double)r); }
    const T dxsin = rn_div2(rn_mul(w, sn)), dxcos = rn_div2(rn_mul(w, cs)), dysin = rn_div2(rn_mul(h, sn)), dycos = rn_div2(rn_mul(h, cs));
    CropBox<T> b;
    b.vx[0] = rn_add(rn_sub(x, dxcos), dysin); b.vy[0] = rn_sub(rn_sub(y, dxsin), dycos);
    b.vx[1] = rn_add(rn_add(x, dxcos), dysin); b.vy[1] = rn_sub(rn_add(y, dxsin), dycos);
    b.vx[2] = rn_sub(rn_add(x, dxcos), dysin); b.vy[2] = rn_add(rn_add(y, dxsin), dycos);
    b.vx[3] = rn_sub(rn_sub(x, dxcos), dysin); b.vy[3] = rn_add(rn_sub(y, dxsin), dycos);
    b.minx = b.maxx = b.vx[0]; b.miny = b.maxy = b.vy[0];
#pragma unroll
    for (int k = 1; k < 4; k++) {
        b.minx = b.vx[k] < b.minx ? b.vx[k] : b.minx; b.maxx = b.vx[k] > b.maxx ? b.vx[k] : b.maxx;
        b.miny = b.vy[k] < b.miny ? b.vy[k] : b.miny; b.maxy = b.vy[k] > b.maxy ? b.vy[k] : b.maxy;
    }
    return b;
}

template <typename T>
__global__ void __launch_bounds__(256) crop_prep_kernel(const T *__restrict__ boxes, int64_t m, CropBox<T> *__restrict__ recs)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    recs[i] = crop_prep_one<T>(boxes[5 * i], boxes[5 * i + 1], boxes[5 * i + 2], boxes[5 * i + 3], boxes[5 * i + 4]);
}

constexpr int CROP_THREADS = 256, CROP_PPT = 16, CROP_BT = 16;   // points per thread, boxes per CTA

struct CropGrid;
__device__ __forceinline__ bool crop_grid_ok(const CropGrid *g);

template <typename T>
__global__ void __launch_bounds__(CROP_THREADS) crop2dr_kernel(const T *__restrict__ pts, int64_t n, const CropBox<T> *__restrict__ recs, int64_t m,
                                                               uint8_t *__restrict__ mask, const CropGrid *__restrict__ skip_if_grid, int64_t tiles_x, int64_t tiles)
{
    if (skip_if_grid && crop_grid_ok(skip_if_grid)) return;   // the grid path produced the mask
    __shared__ CropBox<T> sb[CROP_BT];
    // tiles of 4096 points x 16 boxes, point tiles fastest; the grid strides over them (the fallback launch behind the grid path is small)
    for (int64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
        const int64_t box0 = (t / tiles_x) * CROP_BT;
        const int nb = (int)(m - box0 < CROP_BT ? m - box0 : CROP_BT);
        __syncthreads();
        for (int i = threadIdx.x; i < nb * (int)(sizeof(CropBox<T>) / sizeof(T)); i += CROP_THREADS)
            reinterpret_cast<T *>(sb)[i] = reinterpret_cast<const T *>(recs + box0)[i];
        __syncthreads();
        const int64_t p0 = ((t % tiles_x) * CROP_THREADS + threadIdx.x) * CROP_PPT;
        if (p0 >= n) continue;
        T px[CROP_PPT], py[CROP_PPT];
        const bool full = p0 + CROP_PPT <= n;
#pragma unroll
        for (int k = 0; k < CROP_PPT; k++) {
            const int64_t j = p0 + k < n ? p0 + k : n - 1;
            px[k] = pts[2 * j]; py[k] = pts[2 * j + 1];
        }
        const bool vec = full && (n % 16 == 0) && ((reinterpret_cast<uintptr_t>(mask) & 15) == 0);
        for (int b = 0; b < nb; b++) {
            const CropBox<T> B = sb[b];
            uint32_t wds[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (int k = 0; k < CROP_PPT; k++) {
                bool in = px[k] > B.minx && px[k] < B.maxx && py[k] > B.miny && py[k] < B.maxy;
                if (in) {
#pragma unroll
                    for (int e = 0; e < 4; e++) {   // edge a -> e in the reference's order 3->0, 0->1, 1->2, 2->3
                        const int a = (e + 3) & 3;
                        const T c = rn_sub(rn_mul(rn_sub(B.vx[e], B.vx[a]), rn_sub(py[k], B.vy[e])), rn_mul(rn_sub(B.vy[e], B.vy[a]), rn_sub(px[k], B.vx[e])));
                        in = in && !(c < T(0));
                    }
                }
                wds[k >> 2] |= (in ? 1u : 0u) << ((k & 3) * 8);
            }
            uint8_t *row = mask + (box0 + b) * n + p0;
            if (vec) {
                __stcs(reinterpret_cast<uint4 *>(row), make_uint4(wds[0], wds[1], wds[2], wds[3]));
            } else {
                for (int k = 0; k < CROP_PPT && p0 + k < n; k++) row[k] = (uint8_t)((wds[k >> 2] >> ((k & 3) * 8)) & 1u);
            }
        }
    }
}

// ------------------------------------------------------------------ grid path
// The brute-force kernel above spends ~10 ALU instructions on every (box, point) pair although a box contains a tiny
// fraction of the cloud.  For large problems the points are binned once into a 256 x 256 grid over their extent
// (cell-sorted records x, y, index); the mask is zero-filled at memset speed and one warp per box visits only the
// cells its AABB touches -- a contiguous run of the sorted list per grid row -- and stores a 1 for the points inside.
// The decision per point is the same code as above, so the mask is identical; the cell of a coordinate is a monotone
// function of it (subtract, multiply by a positive constant, floor, clamp), so every point strictly inside the AABB
// lies in a cell between the cells of the AABB's bounds.
constexpr int CG = 256, CG_CELLS = CG * CG;
struct CropGrid { float minx, miny, invx, invy; uint32_t ok, pad[3]; };
__device__ __forceinline__ bool crop_grid_ok(const CropGrid *g) { return g->ok != 0u; }
template <typename T> struct __align__(16) CropPt { T x, y; uint32_t idx, pad; };

__device__ __forceinline__ uint32_t f2ord(float f) { const uint32_t u = __float_as_uint(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }
__device__ __forceinline__ float ord2f(uint32_t o) { return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o); }

// acc[0..3] = ordered-int min x, max x, min y, max y; acc[4] = a non-finite coordinate was seen
template <typename T>
__global__ void __launch_bounds__(256) crop_bounds_kernel(const T *__restrict__ pts, int64_t n, uint32_t *__restrict__ acc)
{
    float mnx = 3e38f, mxx = -3e38f, mny = 3e38f, mxy = -3e38f;
    int bad = 0;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        const float x = (float)pts[2 * j], y = (float)pts[2 * j + 1];   // the grid only needs float bounds (rounded outwards below)
        if (!(fabsf(x) < 1e30f) || !(fabsf(y) < 1e30f)) bad = 1;
        mnx = fminf(mnx, x); mxx = fmaxf(mxx, x); mny = fminf(mny, y); mxy = fmaxf(mxy, y);
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        mnx = fminf(mnx, __shfl_xor_sync(0xffffffffu, mnx, d)); mxx = fmaxf(mxx, __shfl_xor_sync(0xffffffffu, mxx, d));
        mny = fminf(mny, __shfl_xor_sync(0xffffffffu, mny, d)); mxy = fmaxf(mxy, __shfl_xor_sync(0xffffffffu, mxy, d));
        bad |= __shfl_xor_sync(0xffffffffu, bad, d);
    }
    __shared__ uint32_t red[5];
    if (threadIdx.x < 5) red[threadIdx.x] = (threadIdx.x == 0 || threadIdx.x == 2) ? 0xffffffffu : 0u;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) {
        atomicMin(red + 0, f2ord(mnx)); atomicMax(red + 1, f2ord(mxx)); atomicMin(red + 2, f2ord(mny)); atomicMax(red + 3, f2ord(mxy));
        if (bad) red[4] = 1u;
    }
    __syncthreads();
    if (threadIdx.x == 0) {   // one set of global atomics per CTA
        atomicMin(acc + 0, red[0]); atomicMax(acc + 1, red[1]); atomicMin(acc + 2, red[2]); atomicMax(acc + 3, red[3]);
        if (red[4]) acc[4] = 1u;
    }
}

__global__ void crop_grid_kernel(const uint32_t *__restrict__ acc, CropGrid *__restrict__ g)
{
    CropGrid o;
    const float mnx = ord2f(acc[0]), mxx = ord2f(acc[1]), mny = ord2f(acc[2]), mxy = ord2f(acc[3]);
    o.minx = mnx; o.miny = mny; o.ok = 0; o.pad[0] = o.pad[1] = o.pad[2] = 0;
    const float ex = mxx - mnx, ey = mxy - mny;
    o.invx = ex > 0 ? (float)CG / ex : 0.f; o.invy = ey > 0 ? (float)CG / ey : 0.f;
    if (!acc[4] && ex >= 0 && ey >= 0 && ex < 1e30f && ey < 1e30f && (ex > 0 || ey > 0)) o.ok = 1;
    *g = o;
}

// cell coordinate of a value: monotone in v (the double -> float conversion of the fp64 instantiation is monotone too)
__device__ __forceinline__ int crop_cell(float v, float lo, float inv) { return min(CG - 1, max(0, (int)floorf((v - lo) * inv))); }

// pass 0 counts the points of every cell and keeps each point's cell and arrival rank; pass 1 (after the scan of the counts) places the records
template <typename T, int PASS>
__global__ void __launch_bounds__(256) crop_bin_kernel(const T *__restrict__ pts, int64_t n, const CropGrid *__restrict__ g, uint32_t *__restrict__ cellcnt,
                                                       const uint32_t *__restrict__ cellptr, uint2 *__restrict__ cellrank, CropPt<T> *__restrict__ sorted)
{
    if (!g->ok) return;
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const T x = pts[2 * j], y = pts[2 * j + 1];
    if (PASS == 0) {
        const uint32_t c = (uint32_t)(crop_cell((float)y, g->miny, g->invy) * CG + crop_cell((float)x, g->minx, g->invx));
        cellrank[j] = make_uint2(c, atomicAdd(cellcnt + c, 1u));
    } else {
        const uint2 cr = cellrank[j];
        CropPt<T> e; e.x = x; e.y = y; e.idx = (uint32_t)j; e.pad = 0;
        sorted[cellptr[cr.x] + cr.y] = e;
    }
}

template <typename T>
__device__ __forceinline__ bool crop_inside(const CropBox<T> &B, T px, T py)
{
    bool in = px > B.minx && px < B.maxx && py > B.miny && py < B.maxy;
    if (in) {
#pragma unroll
        for (int e = 0; e < 4; e++) {
            const int a = (e + 3) & 3;
            const T c = rn_sub(rn_mul(rn_sub(B.vx[e], B.vx[a]), rn_sub(py, B.vy[e])), rn_mul(rn_sub(B.vy[e], B.vy[a]), rn_sub(px, B.vx[e])));
            in = in && !(c < T(0));
        }
    }
    return in;
}

// The mask (1 byte per pair, the only large object) is written once by a pure store stream that depends on nothing -- it runs on an
// internal stream next to the binning kernels, at the speed HBM takes writes (tools/write_bw_probe.cu: 7.0 TB/s for this shape) -- and
// the hit kernel then stores a 1 for the few candidates that lie inside their box (a read-modify-write of one sector per hit: ~3 % of
// the mask bytes on the bench case).
constexpr int CROP_ZPIECE = 16384;   // bytes per CTA of the zero stream
__global__ void __launch_bounds__(256) crop_zero_kernel(uint8_t *__restrict__ mask, size_t bytes)
{
    const size_t head = (16 - (reinterpret_cast<uintptr_t>(mask) & 15)) & 15;   // bytes in front of the first aligned line
    const size_t h = head < bytes ? head : bytes;
    uint4 *p4 = reinterpret_cast<uint4 *>(mask + h);
    const size_t n4 = (bytes - h) >> 4, tail = (bytes - h) & 15;
    const size_t k0 = (size_t)blockIdx.x * (CROP_ZPIECE / 16);
    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
    for (int u = 0; u < CROP_ZPIECE / 16 / 256; u++) {
        const size_t k = k0 + (size_t)u * 256 + threadIdx.x;
        if (k < n4) p4[k] = z;
    }
    if (blockIdx.x == 0) {
        if (threadIdx.x < h) mask[threadIdx.x] = 0;
        if (threadIdx.x < tail) mask[h + n4 * 16 + threadIdx.x] = 0;
    }
}

// The candidates of a box are the points of the grid cells its AABB touches: per grid row one contiguous run of the cell-sorted list.
// Lane l of a warp fetches the run of grid row l, a warp scan turns the run lengths into a flat candidate index, and the threads walk
// that index four candidates deep (four independent loads per thread in flight; the run of a candidate is found with five shuffles),
// so a box costs one or two load round trips instead of one per grid row.
// crop_hits_kernel: one warp per box, for boxes of at most CROP_LIGHT candidates (median 28 on the bench case).  Larger boxes -- the
// ones on the dense first metres of a lidar cloud have 35 000 -- are cut into up to CROP_HSLICES items of ~1024 candidates on a list that
// crop_heavy_kernel serves with one CTA per item.
constexpr int CROP_LIGHT = 128, CROP_HSLICES = 16, CROP_HT = 256, CROP_ITEM = 4 * CROP_HT;

template <typename T>
__device__ __forceinline__ void crop_cells(const CropBox<T> &B, const CropGrid &G, int *x0, int *x1, int *y0, int *y1)
{
    // float bounds rounded outwards, so that the cell range covers the exact AABB of the fp64 instantiation as well
    const float lx = sizeof(T) == 8 ? __double2float_rd((double)B.minx) : (float)B.minx, hx = sizeof(T) == 8 ? __double2float_ru((double)B.maxx) : (float)B.maxx;
    const float ly = sizeof(T) == 8 ? __double2float_rd((double)B.miny) : (float)B.miny, hy = sizeof(T) == 8 ? __double2float_ru((double)B.maxy) : (float)B.maxy;
    *x0 = crop_cell(lx, G.minx, G.invx); *x1 = crop_cell(hx, G.minx, G.invx);
    *y0 = crop_cell(ly, G.miny, G.invy); *y1 = crop_cell(hy, G.miny, G.invy);
}

// the mask's hit action: a 1 in the box's row
template <typename T> struct CropMaskHit {
    uint8_t *__restrict__ row;
    __device__ __forceinline__ void operator()(const CropPt<T> &p) const { row[p.idx] = 1; }
};

// all 32 lanes of a warp call this with the same box; thread-private: first (its first candidate) -- candidates first, first + stride, ... are its own.
// hit(p) runs for every candidate p inside the box.
template <typename T, typename Hit>
__device__ __forceinline__ void crop_walk(const CropBox<T> &B, int x0, int x1, int y0, int y1, const CropPt<T> *__restrict__ sorted,
                                          const uint32_t *__restrict__ cellptr, Hit &hit, uint32_t first, uint32_t stride)
{
    const unsigned lane = threadIdx.x & 31;
    for (int yb = y0; yb <= y1; yb += 32) {
        uint32_t beg = 0, cnt = 0;
        if (yb + (int)lane <= y1) { beg = cellptr[(yb + (int)lane) * CG + x0]; cnt = cellptr[(yb + (int)lane) * CG + x1 + 1] - beg; }   // the cells of one grid row are contiguous in the sorted list
        uint32_t incl = cnt;   // inclusive prefix of the run lengths
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d); if ((int)lane >= d) incl += v; }
        const uint32_t tb = __shfl_sync(0xffffffffu, incl, 31), excl = incl - cnt;
        for (uint32_t c0 = 0; c0 < tb; c0 += 4 * stride) {   // c0 and tb are the same in every lane: the shuffles below are converged
            uint32_t k[4];
            bool ok[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const uint32_t c = c0 + u * stride + first;
                ok[u] = c < tb;
                const uint32_t cc = ok[u] ? c : tb - 1;
                uint32_t r = 0;   // number of runs that end at or before candidate cc = the run it belongs to
#pragma unroll
                for (int step = 16; step; step >>= 1) { const uint32_t v = __shfl_sync(0xffffffffu, incl, (int)(r + step - 1)); if (v <= cc) r += step; }
                k[u] = __shfl_sync(0xffffffffu, beg, (int)r) + (cc - __shfl_sync(0xffffffffu, excl, (int)r));
            }
            CropPt<T> p[4];
#pragma unroll
            for (int u = 0; u < 4; u++) if (ok[u]) p[u] = sorted[k[u]];
#pragma unroll
            for (int u = 0; u < 4; u++) if (ok[u] && crop_inside<T>(B, p[u].x, p[u].y)) hit(p[u]);
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(256) crop_hits_kernel(const CropPt<T> *__restrict__ sorted, int64_t n, const CropBox<T> *__restrict__ recs, int64_t m,
                                                        const CropGrid *__restrict__ g, const uint32_t *__restrict__ cellptr, uint8_t *__restrict__ mask,
                                                        uint32_t *__restrict__ heavy_count, uint2 *__restrict__ heavy_item)
{
    const unsigned lane = threadIdx.x & 31;
    const int64_t i = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (i >= m) return;
    const CropGrid G = *g;
    const CropBox<T> B = recs[i];
    if (!G.ok) return;                                      // no grid: the brute-force kernel that follows writes the whole mask
    if (!(B.minx < B.maxx) || !(B.miny < B.maxy)) return;   // empty or NaN box: no point passes the open AABB test
    int x0, x1, y0, y1;
    crop_cells<T>(B, G, &x0, &x1, &y0, &y1);
    uint32_t total = 0;
    for (int yb = y0; yb <= y1; yb += 32) {
        uint32_t c = 0;
        if (yb + (int)lane <= y1) c = cellptr[(yb + (int)lane) * CG + x1 + 1] - cellptr[(yb + (int)lane) * CG + x0];
        total += __reduce_add_sync(0xffffffffu, c);
    }
    if (total > (uint32_t)CROP_LIGHT) {   // at most CROP_HSLICES items per box
        const uint32_t ns = min((uint32_t)CROP_HSLICES, (total + CROP_ITEM - 1) / CROP_ITEM);
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(heavy_count, ns);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (lane < ns) heavy_item[base + lane] = make_uint2((uint32_t)i, lane | (ns << 16));
        return;
    }
    CropMaskHit<T> hit{mask + i * n};
    crop_walk<T>(B, x0, x1, y0, y1, sorted, cellptr, hit, lane, 32u);
}

template <typename T>
__global__ void __launch_bounds__(CROP_HT) crop_heavy_kernel(const CropPt<T> *__restrict__ sorted, int64_t n, const CropBox<T> *__restrict__ recs,
                                                             const CropGrid *__restrict__ g, const uint32_t *__restrict__ cellptr, uint8_t *__restrict__ mask,
                                                             const uint32_t *__restrict__ heavy_count, const uint2 *__restrict__ heavy_item)
{
    const CropGrid G = *g;
    if (!G.ok) return;
    const uint32_t items = *heavy_count;
    for (uint32_t w = blockIdx.x; w < items; w += gridDim.x) {
        const uint2 it = heavy_item[w];
        const int64_t i = it.x;
        const uint32_t j = it.y & 0xffffu, ns = it.y >> 16;
        const CropBox<T> B = recs[i];
        int x0, x1, y0, y1;
        crop_cells<T>(B, G, &x0, &x1, &y0, &y1);
        CropMaskHit<T> hit{mask + i * n};
        crop_walk<T>(B, x0, x1, y0, y1, sorted, cellptr, hit, j * CROP_HT + threadIdx.x, ns * CROP_HT);
    }
}

// one internal stream + fork / join events per device (created once): the binning kernels run on it next to the zero stream of the mask
struct CropLane { cudaStream_t s; cudaEvent_t fork, join; std::mutex mu; bool ok; };
static CropLane *crop_lane()
{
    static CropLane pool[64];
    static std::mutex init_mu;
    static bool made[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); return nullptr; }
    std::lock_guard<std::mutex> gd(init_mu);
    CropLane &L = pool[dev];
    if (!made[dev]) {
        made[dev] = true;
        // highest priority: its small binning kernels get SM slots as the CTAs of the zero stream (caller's stream) retire, instead of queueing behind that grid
        int lo = 0, hi = 0;
        L.ok = cudaDeviceGetStreamPriorityRange(&lo, &hi) == cudaSuccess && cudaStreamCreateWithPriority(&L.s, cudaStreamNonBlocking, hi) == cudaSuccess;
        L.ok = L.ok && cudaEventCreateWithFlags(&L.fork, cudaEventDisableTiming) == cudaSuccess;
        L.ok = L.ok && cudaEventCreateWithFlags(&L.join, cudaEventDisableTiming) == cudaSuccess;
        if (!L.ok) cudaGetLastError();
    }
    return L.ok ? &L : nullptr;
}

template <typename T> static size_t crop_grid_ws_bytes(int64_t m, int64_t n)
{
    const size_t n1 = (size_t)(n > 0 ? n : 1), m1 = (size_t)(m > 0 ? m : 1);
    return align_up(64) + align_up(sizeof(CropGrid)) + 2 * align_up((size_t)(CG_CELLS + 1) * 4) + align_up(n1 * sizeof(CropPt<T>)) + align_up(n1 * sizeof(uint2)) +
           align_up(m1 * CROP_HSLICES * sizeof(uint2)) + align_up(scan_workspace_bytes(CG_CELLS + 1));
}
template <typename T> static size_t crop_ws_bytes(int64_t m, int64_t n) { return align_up((size_t)(m > 0 ? m : 1) * sizeof(CropBox<T>)) + 256 + crop_grid_ws_bytes<T>(m, n); }

constexpr int64_t CROP_GRID_MIN_PAIRS = 64ll << 20;   // below this the binning costs more than the brute-force pass

template <typename T>
static int crop_impl(const T *pts, int64_t n, const T *boxes, int64_t m, uint8_t *mask, void *ws, size_t ws_bytes, cudaStream_t st)
{
    if (n < 0 || m < 0) return D3D_ERR_INVALID_ARGUMENT;
    if (n == 0 || m == 0) return D3D_OK;
    if (!pts || !boxes || !mask) return D3D_ERR_INVALID_ARGUMENT;
    if (!ws || ws_bytes < crop_ws_bytes<T>(m, n)) return D3D_ERR_WORKSPACE;
    const int64_t gy = cdiv(m, CROP_BT), gx = cdiv(n, (int64_t)CROP_THREADS * CROP_PPT);
    if (gx * gy > 0x7fffffffll || n >= (1ll << 32) || m > 0x7fffffffll) return D3D_ERR_INVALID_ARGUMENT;
    Arena a(ws, ws_bytes);
    CropBox<T> *recs = a.take<CropBox<T>>(m);
    int mode = 0;   // tuning / test override: D3D_B200_CROP_PATH=brute | grid
    if (const int t = tuning(D3D_TUNE_CROP_PATH, 0)) mode = t;   // 1 brute force, 2 grid
    const bool grid = mode == 2 || (mode == 0 && m * n >= CROP_GRID_MIN_PAIRS);
    if (!grid) {
        crop_prep_kernel<T><<<(unsigned)cdiv(m, 256), 256, 0, st>>>(boxes, m, recs); D3D_LAUNCHED();
        crop2dr_kernel<T><<<(unsigned)(gx * gy), CROP_THREADS, 0, st>>>(pts, n, recs, m, mask, nullptr, gx, gx * gy); D3D_LAUNCHED();
        return D3D_OK;
    }
    uint32_t *acc = a.take<uint32_t>(16);
    CropGrid *g = a.take<CropGrid>(1);
    uint32_t *cellcnt = a.take<uint32_t>((size_t)(CG_CELLS + 1));
    uint32_t *cellptr = a.take<uint32_t>((size_t)(CG_CELLS + 1));
    CropPt<T> *sorted = a.take<CropPt<T>>(n);
    uint2 *cellrank = a.take<uint2>(n);
    uint2 *heavy_item = a.take<uint2>((size_t)m * CROP_HSLICES);
    void *scan_ws = a.take<char>(scan_workspace_bytes(CG_CELLS + 1));
    if (!a.ok()) return D3D_ERR_WORKSPACE;
    uint32_t *heavy_count = acc + 5;
    const uint32_t init[6] = {0xffffffffu, 0u, 0xffffffffu, 0u, 0u, 0u};
    const size_t mbytes = (size_t)m * n;
    const unsigned gz = (unsigned)cdiv((int64_t)mbytes, (int64_t)CROP_ZPIECE);
    const unsigned gb = (unsigned)cdiv(n, 256);
    // fork: the binning chain runs on the internal high-priority stream next to the zero stream of the mask, which has no input
    CropLane *lane = crop_lane();
    std::unique_lock<std::mutex> lk;
    cudaStream_t sb = st;
    if (lane) {
        lk = std::unique_lock<std::mutex>(lane->mu);   // the events are shared by the callers of one device
        D3D_CUDA_TRY(cudaEventRecord(lane->fork, st));
        D3D_CUDA_TRY(cudaStreamWaitEvent(lane->s, lane->fork, 0));
        sb = lane->s;
    }
    crop_zero_kernel<<<gz, 256, 0, st>>>(mask, mbytes); D3D_LAUNCHED();
    crop_prep_kernel<T><<<(unsigned)cdiv(m, 256), 256, 0, sb>>>(boxes, m, recs); D3D_LAUNCHED();
    D3D_CUDA_TRY(cudaMemcpyAsync(acc, init, sizeof(init), cudaMemcpyHostToDevice, sb));
    D3D_CUDA_TRY(cudaMemsetAsync(cellcnt, 0, (size_t)(CG_CELLS + 1) * 4, sb));
    crop_bounds_kernel<T><<<gb < 592 ? gb : 592, 256, 0, sb>>>(pts, n, acc); D3D_LAUNCHED();
    crop_grid_kernel<<<1, 1, 0, sb>>>(acc, g); D3D_LAUNCHED();
    crop_bin_kernel<T, 0><<<gb, 256, 0, sb>>>(pts, n, g, cellcnt, nullptr, cellrank, nullptr); D3D_LAUNCHED();
    int rc = exclusive_scan_u32(cellcnt, cellptr, CG_CELLS + 1, nullptr, scan_ws, sb);
    if (rc) return rc;
    crop_bin_kernel<T, 1><<<gb, 256, 0, sb>>>(pts, n, g, nullptr, cellptr, cellrank, sorted); D3D_LAUNCHED();
    if (lane) {   // join
        D3D_CUDA_TRY(cudaEventRecord(lane->join, lane->s));
        D3D_CUDA_TRY(cudaStreamWaitEvent(st, lane->join, 0));
        lk.unlock();
    }
    crop_hits_kernel<T><<<(unsigned)cdiv(m, 8), 256, 0, st>>>(sorted, n, recs, m, g, cellptr, mask, heavy_count, heavy_item); D3D_LAUNCHED();
    crop_heavy_kernel<T><<<1184, CROP_HT, 0, st>>>(sorted, n, recs, g, cellptr, mask, heavy_count, heavy_item); D3D_LAUNCHED();
    // geometry that admits no grid (non-finite points, all points identical): the brute-force pass runs instead (it leaves at once otherwise)
    const int64_t gf = gx * gy < 1184 ? gx * gy : 1184;
    crop2dr_kernel<T><<<(unsigned)gf, CROP_THREADS, 0, st>>>(pts, n, recs, m, mask, g, gx, gx * gy); D3D_LAUNCHED();
    return D3D_OK;
}

// ------------------------------------------------------------------ frame-batched mask
// Frame f owns points [poff[f], poff[f+1]) and boxes [boff[f], boff[f+1]) of the packed inputs and writes its row-major [m_f, n_f] block
// at mask + moff[f].  The box records of the whole batch are prepared by one launch; the tile kernel runs crop2dr_kernel's tiles with
// frames on grid.x, so a frame costs no launch of its own, and decides a pair with crop_inside, the grid path's copy of crop2dr_kernel's
// test (crop2dr_kernel keeps its own inline copy: calling crop_inside there changes its register allocation).  A frame of
// CROP_GRID_MIN_PAIRS pairs or more is not written: the caller runs the single-frame entry point (its grid path) on it.
// project_axis >= 0 (3-D rows): the records come from the plane of the two other axes, and a pair also needs box3dp_crop's test along
// the axis, p - d / 2 < c < p + d / 2 with the box's centre c and extent d, rounded like torch's elementwise operators.
template <typename T> struct CropZ { T c, hd; };

template <typename T>
__global__ void __launch_bounds__(256) crop_prep_batch_kernel(const T *__restrict__ boxes, int64_t m, int axis, CropBox<T> *__restrict__ recs,
                                                              CropZ<T> *__restrict__ z)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    if (axis < 0) {
        const T *b = boxes + 5 * i;
        recs[i] = crop_prep_one<T>(b[0], b[1], b[2], b[3], b[4]);
        return;
    }
    const T *b = boxes + 7 * i;
    int pa, pb;
    proj_plane(axis, &pa, &pb);
    recs[i] = crop_prep_one<T>(b[pa], b[pb], b[3 + pa], b[3 + pb], b[6]);
    CropZ<T> q;
    q.c = b[axis]; q.hd = rn_div2(b[3 + axis]);
    z[i] = q;
}

// frames on grid.x; 4096-point tiles on grid.y and 16-box tiles on grid.z, each striding over the frame's own tiles (tiles beyond the
// frame's size exit at once)
template <typename T, bool P3>
__global__ void __launch_bounds__(CROP_THREADS) crop2dr_batch_kernel(const T *__restrict__ pts, const int64_t *__restrict__ poff, const CropBox<T> *__restrict__ recs,
                                                                     const CropZ<T> *__restrict__ zr, const int64_t *__restrict__ boff, int axis,
                                                                     const int64_t *__restrict__ moff, uint8_t *__restrict__ mask)
{
    __shared__ CropBox<T> sb[CROP_BT];
    __shared__ CropZ<T> sz[P3 ? CROP_BT : 1];
    const int64_t f = blockIdx.x, j0 = poff[f], n = poff[f + 1] - j0, i0 = boff[f], m = boff[f + 1] - i0;
    if (n * m >= CROP_GRID_MIN_PAIRS) return;
    const int64_t tiles_p = (n + CROP_THREADS * CROP_PPT - 1) / (CROP_THREADS * CROP_PPT), tiles_b = (m + CROP_BT - 1) / CROP_BT;
    if ((int64_t)blockIdx.y >= tiles_p || (int64_t)blockIdx.z >= tiles_b) return;
    int pa = 0, pb = 1;
    if (P3) proj_plane(axis, &pa, &pb);
    constexpr int PS = P3 ? 3 : 2;   // point row length
    uint8_t *blk = mask + moff[f];
    for (int64_t tb = blockIdx.z; tb < tiles_b; tb += gridDim.z) {
        const int64_t box0 = tb * CROP_BT;
        const int nb = (int)(m - box0 < CROP_BT ? m - box0 : CROP_BT);
        __syncthreads();
        for (int i = threadIdx.x; i < nb * (int)(sizeof(CropBox<T>) / sizeof(T)); i += CROP_THREADS)
            reinterpret_cast<T *>(sb)[i] = reinterpret_cast<const T *>(recs + i0 + box0)[i];
        if (P3 && threadIdx.x < nb) sz[threadIdx.x] = zr[i0 + box0 + threadIdx.x];
        __syncthreads();
        for (int64_t tp = blockIdx.y; tp < tiles_p; tp += gridDim.y) {
            const int64_t p0 = (tp * CROP_THREADS + threadIdx.x) * CROP_PPT;
            if (p0 >= n) continue;
            T px[CROP_PPT], py[CROP_PPT], pz[P3 ? CROP_PPT : 1];
            const bool full = p0 + CROP_PPT <= n;
#pragma unroll
            for (int k = 0; k < CROP_PPT; k++) {
                const int64_t j = j0 + (p0 + k < n ? p0 + k : n - 1);
                px[k] = pts[PS * j + pa]; py[k] = pts[PS * j + pb];
                if (P3) pz[k] = pts[PS * j + axis];
            }
            for (int b = 0; b < nb; b++) {
                const CropBox<T> B = sb[b];
                uint32_t wds[4] = {0u, 0u, 0u, 0u};
#pragma unroll
                for (int k = 0; k < CROP_PPT; k++) {
                    bool in = crop_inside<T>(B, px[k], py[k]);
                    if (P3) in = in && rn_sub(pz[k], sz[b].hd) < sz[b].c && sz[b].c < rn_add(pz[k], sz[b].hd);
                    wds[k >> 2] |= (in ? 1u : 0u) << ((k & 3) * 8);
                }
                uint8_t *row = blk + (box0 + b) * n + p0;
                if (full && (reinterpret_cast<uintptr_t>(row) & 15) == 0) {   // frame blocks and rows start anywhere: decide per row
                    __stcs(reinterpret_cast<uint4 *>(row), make_uint4(wds[0], wds[1], wds[2], wds[3]));
                } else {
                    for (int k = 0; k < CROP_PPT && p0 + k < n; k++) row[k] = (uint8_t)((wds[k >> 2] >> ((k & 3) * 8)) & 1u);
                }
            }
        }
    }
}

template <typename T> static size_t crop_batch_ws_bytes(int64_t total_boxes)
{
    const size_t m1 = (size_t)(total_boxes > 0 ? total_boxes : 1);
    return 256 + align_up(m1 * sizeof(CropBox<T>)) + align_up(m1 * sizeof(CropZ<T>));
}

template <typename T>
static int crop_batch_impl(const T *pts, int64_t total_pts, const int64_t *poff, const T *boxes, int64_t total_boxes, const int64_t *boff, int64_t nframes,
                           int64_t max_pts, int64_t max_boxes, int axis, const int64_t *moff, uint8_t *mask, void *ws, size_t ws_bytes, cudaStream_t st)
{
    if (total_pts < 0 || total_boxes < 0 || nframes < 0 || max_pts < 0 || max_boxes < 0 || axis < -1 || axis > 2) return D3D_ERR_INVALID_ARGUMENT;
    if (nframes == 0 || total_pts == 0 || total_boxes == 0) return D3D_OK;   // every block is empty
    if (!pts || !poff || !boxes || !boff || !moff || !mask) return D3D_ERR_INVALID_ARGUMENT;
    if (nframes > 0x7fffffffll) return D3D_ERR_UNSUPPORTED;
    if (!ws || ws_bytes < crop_batch_ws_bytes<T>(total_boxes)) return D3D_ERR_WORKSPACE;
    if (max_pts == 0) max_pts = total_pts;   // 0: bound unknown
    if (max_boxes == 0) max_boxes = total_boxes;
    Arena a(ws, ws_bytes);
    a.take<char>(256);
    CropBox<T> *recs = a.take<CropBox<T>>(total_boxes);
    CropZ<T> *z = a.take<CropZ<T>>(total_boxes);
    if (!a.ok()) return D3D_ERR_WORKSPACE;
    crop_prep_batch_kernel<T><<<(unsigned)cdiv(total_boxes, 256), 256, 0, st>>>(boxes, total_boxes, axis, recs, z); D3D_LAUNCHED();
    const int64_t gy = cdiv(max_pts, (int64_t)CROP_THREADS * CROP_PPT), gz = cdiv(max_boxes, CROP_BT);
    const dim3 grid((unsigned)nframes, (unsigned)(gy < 65535 ? gy : 65535), (unsigned)(gz < 65535 ? gz : 65535));
    if (axis < 0) crop2dr_batch_kernel<T, false><<<grid, CROP_THREADS, 0, st>>>(pts, poff, recs, z, boff, axis, moff, mask);
    else crop2dr_batch_kernel<T, true><<<grid, CROP_THREADS, 0, st>>>(pts, poff, recs, z, boff, axis, moff, mask);
    D3D_LAUNCHED();
    return D3D_OK;
}

// ------------------------------------------------------------------ fused reductions of the mask
// point_box[j] = the lowest frame-local index of a box whose mask entry for point j is 1, or -1; box_npoints[i] = the number of points
// in box i.  Nothing of the mask is stored.  The outputs are handled as unsigned 64-bit words: -1 is the all-ones word, so the per-point
// result is an unsigned atomicMin into an output filled with 0xff bytes (no finalise pass), and the counts are atomicAdds into a zeroed
// output.  The decision per pair is the mask's: crop_inside, and for 3-D rows the same rounded test along the axis.
typedef unsigned long long u64;

// crop2dr_batch_kernel's tiles and frame mapping (frames on grid.x; poff == nullptr: one frame of n1 points and m1 boxes).  A thread
// decides its 16 points against each box of the tile as a 16-bit word; hits are rare, so a warp votes first and only a warp with a hit
// reduces: its count goes to a shared counter per box (one global atomic per box and CTA at the end of the box tile), and each point
// not already claimed by a lower box of the tile takes an atomicMin.  Frames of skip_pairs pairs or more are left to the grid path.
template <typename T, bool P3>
__global__ void __launch_bounds__(CROP_THREADS) crop_assign_tile_kernel(const T *__restrict__ pts, const int64_t *__restrict__ poff, int64_t n1,
                                                                        const CropBox<T> *__restrict__ recs, const CropZ<T> *__restrict__ zr,
                                                                        const int64_t *__restrict__ boff, int64_t m1, int axis, int64_t skip_pairs,
                                                                        const CropGrid *__restrict__ skip_if_grid, u64 *__restrict__ point_box,
                                                                        u64 *__restrict__ box_npoints)
{
    if (skip_if_grid && crop_grid_ok(skip_if_grid)) return;   // the grid path produced the outputs
    __shared__ CropBox<T> sb[CROP_BT];
    __shared__ CropZ<T> sz[P3 ? CROP_BT : 1];
    __shared__ uint32_t scnt[CROP_BT];
    const int64_t f = blockIdx.x;
    const int64_t j0 = poff ? poff[f] : 0, n = poff ? poff[f + 1] - j0 : n1, i0 = boff ? boff[f] : 0, m = boff ? boff[f + 1] - i0 : m1;
    if (n * m >= skip_pairs) return;
    const int64_t tiles_p = (n + CROP_THREADS * CROP_PPT - 1) / (CROP_THREADS * CROP_PPT), tiles_b = (m + CROP_BT - 1) / CROP_BT;
    if ((int64_t)blockIdx.y >= tiles_p || (int64_t)blockIdx.z >= tiles_b) return;
    int pa = 0, pb = 1;
    if (P3) proj_plane(axis, &pa, &pb);
    constexpr int PS = P3 ? 3 : 2;   // point row length
    const unsigned lane = threadIdx.x & 31;
    for (int64_t tb = blockIdx.z; tb < tiles_b; tb += gridDim.z) {
        const int64_t box0 = tb * CROP_BT;
        const int nb = (int)(m - box0 < CROP_BT ? m - box0 : CROP_BT);
        __syncthreads();
        for (int i = threadIdx.x; i < nb * (int)(sizeof(CropBox<T>) / sizeof(T)); i += CROP_THREADS)
            reinterpret_cast<T *>(sb)[i] = reinterpret_cast<const T *>(recs + i0 + box0)[i];
        if (P3 && threadIdx.x < nb) sz[threadIdx.x] = zr[i0 + box0 + threadIdx.x];
        if (threadIdx.x < CROP_BT) scnt[threadIdx.x] = 0u;
        __syncthreads();
        for (int64_t tp = blockIdx.y; tp < tiles_p; tp += gridDim.y) {
            const int64_t p0 = (tp * CROP_THREADS + threadIdx.x) * CROP_PPT;
            // threads past the frame's end stay for the warp votes, with no valid point
            const int np = p0 >= n ? 0 : (n - p0 < CROP_PPT ? (int)(n - p0) : CROP_PPT);
            const uint32_t valid = (1u << np) - 1u;
            T px[CROP_PPT], py[CROP_PPT], pz[P3 ? CROP_PPT : 1];
#pragma unroll
            for (int k = 0; k < CROP_PPT; k++) {
                const int64_t j = j0 + (p0 + k < n ? p0 + k : n - 1);
                px[k] = pts[PS * j + pa]; py[k] = pts[PS * j + pb];
                if (P3) pz[k] = pts[PS * j + axis];
            }
            uint32_t seen = 0u;   // points already claimed by a lower box of this tile
            for (int b = 0; b < nb; b++) {
                const CropBox<T> B = sb[b];
                uint32_t hb = 0u;
#pragma unroll
                for (int k = 0; k < CROP_PPT; k++) {
                    bool in = crop_inside<T>(B, px[k], py[k]);
                    if (P3) in = in && rn_sub(pz[k], sz[b].hd) < sz[b].c && sz[b].c < rn_add(pz[k], sz[b].hd);
                    hb |= (in ? 1u : 0u) << k;
                }
                hb &= valid;
                if (__any_sync(0xffffffffu, hb != 0u)) {
                    const uint32_t c = __reduce_add_sync(0xffffffffu, (uint32_t)__popc(hb));
                    if (lane == 0) atomicAdd(scnt + b, c);
                    for (uint32_t fresh = hb & ~seen; fresh; fresh &= fresh - 1u)
                        atomicMin(point_box + j0 + p0 + (__ffs(fresh) - 1), (u64)(box0 + b));
                    seen |= hb;
                }
            }
        }
        __syncthreads();
        if (threadIdx.x < nb && scnt[threadIdx.x]) atomicAdd(box_npoints + i0 + box0 + threadIdx.x, (u64)scnt[threadIdx.x]);
    }
}

// the grid path's hit action: the point's atomicMin and the walker's count; for 3-D rows the test along the axis comes first (the
// sorted records hold the plane coordinates, the axis coordinate is read through the point's index)
template <typename T, bool P3> struct CropAssignHit {
    const T *__restrict__ pts;
    int axis;
    CropZ<T> z;
    int64_t box;
    u64 *__restrict__ point_box;
    uint32_t count;
    __device__ __forceinline__ void operator()(const CropPt<T> &p)
    {
        if (P3) {
            const T c = pts[3 * (int64_t)p.idx + axis];
            if (!(rn_sub(c, z.hd) < z.c && z.c < rn_add(c, z.hd))) return;
        }
        atomicMin(point_box + p.idx, (u64)box);
        count++;
    }
};

// crop_hits_kernel / crop_heavy_kernel with the reducing hit action: a warp's count is one atomicAdd
template <typename T, bool P3>
__global__ void __launch_bounds__(256) crop_assign_hits_kernel(const CropPt<T> *__restrict__ sorted, const T *__restrict__ pts, int axis,
                                                               const CropBox<T> *__restrict__ recs, const CropZ<T> *__restrict__ zr, int64_t m,
                                                               const CropGrid *__restrict__ g, const uint32_t *__restrict__ cellptr,
                                                               u64 *__restrict__ point_box, u64 *__restrict__ box_npoints,
                                                               uint32_t *__restrict__ heavy_count, uint2 *__restrict__ heavy_item)
{
    const unsigned lane = threadIdx.x & 31;
    const int64_t i = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (i >= m) return;
    const CropGrid G = *g;
    const CropBox<T> B = recs[i];
    if (!G.ok) return;                                      // no grid: the tile kernel that follows computes the outputs
    if (!(B.minx < B.maxx) || !(B.miny < B.maxy)) return;   // empty or NaN box: no point passes the open AABB test
    int x0, x1, y0, y1;
    crop_cells<T>(B, G, &x0, &x1, &y0, &y1);
    uint32_t total = 0;
    for (int yb = y0; yb <= y1; yb += 32) {
        uint32_t c = 0;
        if (yb + (int)lane <= y1) c = cellptr[(yb + (int)lane) * CG + x1 + 1] - cellptr[(yb + (int)lane) * CG + x0];
        total += __reduce_add_sync(0xffffffffu, c);
    }
    if (total > (uint32_t)CROP_LIGHT) {   // at most CROP_HSLICES items per box
        const uint32_t ns = min((uint32_t)CROP_HSLICES, (total + CROP_ITEM - 1) / CROP_ITEM);
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(heavy_count, ns);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (lane < ns) heavy_item[base + lane] = make_uint2((uint32_t)i, lane | (ns << 16));
        return;
    }
    CropAssignHit<T, P3> hit{pts, axis, P3 ? zr[i] : CropZ<T>{}, i, point_box, 0u};
    crop_walk<T>(B, x0, x1, y0, y1, sorted, cellptr, hit, lane, 32u);
    const uint32_t c = __reduce_add_sync(0xffffffffu, hit.count);
    if (lane == 0 && c) atomicAdd(box_npoints + i, (u64)c);
}

template <typename T, bool P3>
__global__ void __launch_bounds__(CROP_HT) crop_assign_heavy_kernel(const CropPt<T> *__restrict__ sorted, const T *__restrict__ pts, int axis,
                                                                    const CropBox<T> *__restrict__ recs, const CropZ<T> *__restrict__ zr,
                                                                    const CropGrid *__restrict__ g, const uint32_t *__restrict__ cellptr,
                                                                    u64 *__restrict__ point_box, u64 *__restrict__ box_npoints,
                                                                    const uint32_t *__restrict__ heavy_count, const uint2 *__restrict__ heavy_item)
{
    const CropGrid G = *g;
    if (!G.ok) return;
    const uint32_t items = *heavy_count;
    for (uint32_t w = blockIdx.x; w < items; w += gridDim.x) {
        const uint2 it = heavy_item[w];
        const int64_t i = it.x;
        const uint32_t j = it.y & 0xffffu, ns = it.y >> 16;
        const CropBox<T> B = recs[i];
        int x0, x1, y0, y1;
        crop_cells<T>(B, G, &x0, &x1, &y0, &y1);
        CropAssignHit<T, P3> hit{pts, axis, P3 ? zr[i] : CropZ<T>{}, i, point_box, 0u};
        crop_walk<T>(B, x0, x1, y0, y1, sorted, cellptr, hit, j * CROP_HT + threadIdx.x, ns * CROP_HT);
        const uint32_t c = __reduce_add_sync(0xffffffffu, hit.count);
        if ((threadIdx.x & 31) == 0 && c) atomicAdd(box_npoints + i, (u64)c);
    }
}

// 3-D rows on the grid path: the two plane columns, packed as the 2-D rows the binning kernels read
template <typename T>
__global__ void __launch_bounds__(256) crop_plane_kernel(const T *__restrict__ pts, int64_t n, int axis, T *__restrict__ plane)
{
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    int pa, pb;
    proj_plane(axis, &pa, &pb);
    plane[2 * j] = pts[3 * j + pa]; plane[2 * j + 1] = pts[3 * j + pb];
}

template <typename T> static size_t crop_assign_ws_bytes(int64_t m, int64_t n)
{
    const size_t n1 = (size_t)(n > 0 ? n : 1), m1 = (size_t)(m > 0 ? m : 1);
    return align_up(m1 * sizeof(CropBox<T>)) + align_up(m1 * sizeof(CropZ<T>)) + align_up(n1 * 2 * sizeof(T)) + crop_grid_ws_bytes<T>(m, n);
}

template <typename T>
static int crop_assign_impl(const T *pts, int64_t n, const T *boxes, int64_t m, int axis, int64_t *point_box, int64_t *box_npoints, void *ws,
                            size_t ws_bytes, cudaStream_t st)
{
    if (n < 0 || m < 0 || axis < -1 || axis > 2) return D3D_ERR_INVALID_ARGUMENT;
    if (n == 0 && m == 0) return D3D_OK;
    if ((n && (!pts || !point_box)) || (m && (!boxes || !box_npoints))) return D3D_ERR_INVALID_ARGUMENT;
    if (n >= (1ll << 32) || m > 0x7fffffffll) return D3D_ERR_INVALID_ARGUMENT;
    if (n && m && (!ws || ws_bytes < crop_assign_ws_bytes<T>(m, n))) return D3D_ERR_WORKSPACE;
    if (n) D3D_CUDA_TRY(cudaMemsetAsync(point_box, 0xff, (size_t)n * sizeof(int64_t), st));
    if (m) D3D_CUDA_TRY(cudaMemsetAsync(box_npoints, 0, (size_t)m * sizeof(int64_t), st));
    if (!n || !m) return D3D_OK;
    Arena a(ws, ws_bytes);
    CropBox<T> *recs = a.take<CropBox<T>>(m);
    CropZ<T> *z = a.take<CropZ<T>>(m);
    T *plane = a.take<T>((size_t)n * 2);
    u64 *pbox = reinterpret_cast<u64 *>(point_box), *bcnt = reinterpret_cast<u64 *>(box_npoints);
    int mode = 0;   // D3D_B200_CROP_PATH=brute | grid, as for the mask
    if (const int t = tuning(D3D_TUNE_CROP_PATH, 0)) mode = t;
    const bool grid = mode == 2 || (mode == 0 && m * n >= CROP_GRID_MIN_PAIRS);
    crop_prep_batch_kernel<T><<<(unsigned)cdiv(m, 256), 256, 0, st>>>(boxes, m, axis, recs, z); D3D_LAUNCHED();
    const int64_t gy = cdiv(n, (int64_t)CROP_THREADS * CROP_PPT), gz = cdiv(m, CROP_BT);
    if (!grid) {
        const dim3 tg(1u, (unsigned)(gy < 65535 ? gy : 65535), (unsigned)(gz < 65535 ? gz : 65535));
        if (axis < 0) crop_assign_tile_kernel<T, false><<<tg, CROP_THREADS, 0, st>>>(pts, nullptr, n, recs, z, nullptr, m, axis, INT64_MAX, nullptr, pbox, bcnt);
        else crop_assign_tile_kernel<T, true><<<tg, CROP_THREADS, 0, st>>>(pts, nullptr, n, recs, z, nullptr, m, axis, INT64_MAX, nullptr, pbox, bcnt);
        D3D_LAUNCHED();
        return D3D_OK;
    }
    uint32_t *acc = a.take<uint32_t>(16);
    CropGrid *g = a.take<CropGrid>(1);
    uint32_t *cellcnt = a.take<uint32_t>((size_t)(CG_CELLS + 1));
    uint32_t *cellptr = a.take<uint32_t>((size_t)(CG_CELLS + 1));
    CropPt<T> *sorted = a.take<CropPt<T>>(n);
    uint2 *cellrank = a.take<uint2>(n);
    uint2 *heavy_item = a.take<uint2>((size_t)m * CROP_HSLICES);
    void *scan_ws = a.take<char>(scan_workspace_bytes(CG_CELLS + 1));
    if (!a.ok()) return D3D_ERR_WORKSPACE;
    uint32_t *heavy_count = acc + 5;
    const uint32_t init[6] = {0xffffffffu, 0u, 0xffffffffu, 0u, 0u, 0u};
    const unsigned gb = (unsigned)cdiv(n, 256);
    const T *p2 = pts;   // the 2-D rows the grid is built from
    if (axis >= 0) { crop_plane_kernel<T><<<gb, 256, 0, st>>>(pts, n, axis, plane); D3D_LAUNCHED(); p2 = plane; }
    D3D_CUDA_TRY(cudaMemcpyAsync(acc, init, sizeof(init), cudaMemcpyHostToDevice, st));
    D3D_CUDA_TRY(cudaMemsetAsync(cellcnt, 0, (size_t)(CG_CELLS + 1) * 4, st));
    crop_bounds_kernel<T><<<gb < 592 ? gb : 592, 256, 0, st>>>(p2, n, acc); D3D_LAUNCHED();
    crop_grid_kernel<<<1, 1, 0, st>>>(acc, g); D3D_LAUNCHED();
    crop_bin_kernel<T, 0><<<gb, 256, 0, st>>>(p2, n, g, cellcnt, nullptr, cellrank, nullptr); D3D_LAUNCHED();
    const int rc = exclusive_scan_u32(cellcnt, cellptr, CG_CELLS + 1, nullptr, scan_ws, st);
    if (rc) return rc;
    crop_bin_kernel<T, 1><<<gb, 256, 0, st>>>(p2, n, g, nullptr, cellptr, cellrank, sorted); D3D_LAUNCHED();
    // geometry that admits no grid (non-finite points, all points identical): the tile kernel runs instead (it leaves at once otherwise)
    const dim3 fg(1u, (unsigned)(gy < 74 ? gy : 74), (unsigned)(gz < 16 ? gz : 16));
    if (axis < 0) {
        crop_assign_hits_kernel<T, false><<<(unsigned)cdiv(m, 8), 256, 0, st>>>(sorted, pts, axis, recs, z, m, g, cellptr, pbox, bcnt, heavy_count, heavy_item); D3D_LAUNCHED();
        crop_assign_heavy_kernel<T, false><<<1184, CROP_HT, 0, st>>>(sorted, pts, axis, recs, z, g, cellptr, pbox, bcnt, heavy_count, heavy_item); D3D_LAUNCHED();
        crop_assign_tile_kernel<T, false><<<fg, CROP_THREADS, 0, st>>>(pts, nullptr, n, recs, z, nullptr, m, axis, INT64_MAX, g, pbox, bcnt); D3D_LAUNCHED();
    } else {
        crop_assign_hits_kernel<T, true><<<(unsigned)cdiv(m, 8), 256, 0, st>>>(sorted, pts, axis, recs, z, m, g, cellptr, pbox, bcnt, heavy_count, heavy_item); D3D_LAUNCHED();
        crop_assign_heavy_kernel<T, true><<<1184, CROP_HT, 0, st>>>(sorted, pts, axis, recs, z, g, cellptr, pbox, bcnt, heavy_count, heavy_item); D3D_LAUNCHED();
        crop_assign_tile_kernel<T, true><<<fg, CROP_THREADS, 0, st>>>(pts, nullptr, n, recs, z, nullptr, m, axis, INT64_MAX, g, pbox, bcnt); D3D_LAUNCHED();
    }
    return D3D_OK;
}

template <typename T>
static int crop_assign_batch_impl(const T *pts, int64_t total_pts, const int64_t *poff, const T *boxes, int64_t total_boxes, const int64_t *boff,
                                  int64_t nframes, int64_t max_pts, int64_t max_boxes, int axis, int64_t *point_box, int64_t *box_npoints, void *ws,
                                  size_t ws_bytes, cudaStream_t st)
{
    if (total_pts < 0 || total_boxes < 0 || nframes < 0 || max_pts < 0 || max_boxes < 0 || axis < -1 || axis > 2) return D3D_ERR_INVALID_ARGUMENT;
    if (nframes == 0 || (total_pts == 0 && total_boxes == 0)) return D3D_OK;
    if (!poff || !boff || (total_pts && (!pts || !point_box)) || (total_boxes && (!boxes || !box_npoints))) return D3D_ERR_INVALID_ARGUMENT;
    if (nframes > 0x7fffffffll) return D3D_ERR_UNSUPPORTED;
    if (total_pts && total_boxes && (!ws || ws_bytes < crop_batch_ws_bytes<T>(total_boxes))) return D3D_ERR_WORKSPACE;
    if (total_pts) D3D_CUDA_TRY(cudaMemsetAsync(point_box, 0xff, (size_t)total_pts * sizeof(int64_t), st));
    if (total_boxes) D3D_CUDA_TRY(cudaMemsetAsync(box_npoints, 0, (size_t)total_boxes * sizeof(int64_t), st));
    if (!total_pts || !total_boxes) return D3D_OK;
    if (max_pts == 0) max_pts = total_pts;   // 0: bound unknown
    if (max_boxes == 0) max_boxes = total_boxes;
    Arena a(ws, ws_bytes);
    a.take<char>(256);
    CropBox<T> *recs = a.take<CropBox<T>>(total_boxes);
    CropZ<T> *z = a.take<CropZ<T>>(total_boxes);
    if (!a.ok()) return D3D_ERR_WORKSPACE;
    u64 *pbox = reinterpret_cast<u64 *>(point_box), *bcnt = reinterpret_cast<u64 *>(box_npoints);
    crop_prep_batch_kernel<T><<<(unsigned)cdiv(total_boxes, 256), 256, 0, st>>>(boxes, total_boxes, axis, recs, z); D3D_LAUNCHED();
    const int64_t gy = cdiv(max_pts, (int64_t)CROP_THREADS * CROP_PPT), gz = cdiv(max_boxes, CROP_BT);
    const dim3 grid((unsigned)nframes, (unsigned)(gy < 65535 ? gy : 65535), (unsigned)(gz < 65535 ? gz : 65535));
    if (axis < 0) crop_assign_tile_kernel<T, false><<<grid, CROP_THREADS, 0, st>>>(pts, poff, 0, recs, z, boff, 0, axis, CROP_GRID_MIN_PAIRS, nullptr, pbox, bcnt);
    else crop_assign_tile_kernel<T, true><<<grid, CROP_THREADS, 0, st>>>(pts, poff, 0, recs, z, boff, 0, axis, CROP_GRID_MIN_PAIRS, nullptr, pbox, bcnt);
    D3D_LAUNCHED();
    return D3D_OK;
}

}  // namespace d3d

using namespace d3d;
extern "C" size_t d3d_crop2dr_workspace_bytes(int64_t n, int64_t m, int dtype) { return dtype == D3D_F64 ? crop_ws_bytes<double>(m, n) : crop_ws_bytes<float>(m, n); }
extern "C" int d3d_crop2dr_f32(const float *points, int64_t n, const float *boxes, int64_t m, uint8_t *mask, void *ws, size_t wsb, void *stream)
{ return crop_impl<float>(points, n, boxes, m, mask, ws, wsb, (cudaStream_t)stream); }
extern "C" int d3d_crop2dr_f64(const double *points, int64_t n, const double *boxes, int64_t m, uint8_t *mask, void *ws, size_t wsb, void *stream)
{ return crop_impl<double>(points, n, boxes, m, mask, ws, wsb, (cudaStream_t)stream); }
extern "C" int64_t d3d_crop2dr_grid_min_pairs(void) { return CROP_GRID_MIN_PAIRS; }
extern "C" size_t d3d_crop2dr_batch_workspace_bytes(int64_t total_boxes, int dtype)
{
    if (total_boxes < 0) return 0;
    return dtype == D3D_F64 ? crop_batch_ws_bytes<double>(total_boxes) : crop_batch_ws_bytes<float>(total_boxes);
}
extern "C" int d3d_crop2dr_batch_f32(const float *points, int64_t total_points, const int64_t *point_offsets, const float *boxes, int64_t total_boxes,
                                     const int64_t *box_offsets, int64_t nframes, int64_t max_frame_points, int64_t max_frame_boxes, int project_axis,
                                     const int64_t *mask_offsets, uint8_t *mask, void *ws, size_t wsb, void *stream)
{
    return crop_batch_impl<float>(points, total_points, point_offsets, boxes, total_boxes, box_offsets, nframes, max_frame_points, max_frame_boxes,
                                  project_axis, mask_offsets, mask, ws, wsb, (cudaStream_t)stream);
}
extern "C" int d3d_crop2dr_batch_f64(const double *points, int64_t total_points, const int64_t *point_offsets, const double *boxes, int64_t total_boxes,
                                     const int64_t *box_offsets, int64_t nframes, int64_t max_frame_points, int64_t max_frame_boxes, int project_axis,
                                     const int64_t *mask_offsets, uint8_t *mask, void *ws, size_t wsb, void *stream)
{
    return crop_batch_impl<double>(points, total_points, point_offsets, boxes, total_boxes, box_offsets, nframes, max_frame_points, max_frame_boxes,
                                   project_axis, mask_offsets, mask, ws, wsb, (cudaStream_t)stream);
}
extern "C" size_t d3d_crop2dr_assign_workspace_bytes(int64_t n, int64_t m, int dtype)
{
    if (n < 0 || m < 0) return 0;
    return dtype == D3D_F64 ? crop_assign_ws_bytes<double>(m, n) : crop_assign_ws_bytes<float>(m, n);
}
extern "C" int d3d_crop2dr_assign_f32(const float *points, int64_t n, const float *boxes, int64_t m, int project_axis, int64_t *point_box,
                                      int64_t *box_npoints, void *ws, size_t wsb, void *stream)
{ return crop_assign_impl<float>(points, n, boxes, m, project_axis, point_box, box_npoints, ws, wsb, (cudaStream_t)stream); }
extern "C" int d3d_crop2dr_assign_f64(const double *points, int64_t n, const double *boxes, int64_t m, int project_axis, int64_t *point_box,
                                      int64_t *box_npoints, void *ws, size_t wsb, void *stream)
{ return crop_assign_impl<double>(points, n, boxes, m, project_axis, point_box, box_npoints, ws, wsb, (cudaStream_t)stream); }
extern "C" size_t d3d_crop2dr_assign_batch_workspace_bytes(int64_t total_boxes, int dtype)
{
    if (total_boxes < 0) return 0;
    return dtype == D3D_F64 ? crop_batch_ws_bytes<double>(total_boxes) : crop_batch_ws_bytes<float>(total_boxes);
}
extern "C" int d3d_crop2dr_assign_batch_f32(const float *points, int64_t total_points, const int64_t *point_offsets, const float *boxes,
                                            int64_t total_boxes, const int64_t *box_offsets, int64_t nframes, int64_t max_frame_points,
                                            int64_t max_frame_boxes, int project_axis, int64_t *point_box, int64_t *box_npoints, void *ws, size_t wsb,
                                            void *stream)
{
    return crop_assign_batch_impl<float>(points, total_points, point_offsets, boxes, total_boxes, box_offsets, nframes, max_frame_points,
                                         max_frame_boxes, project_axis, point_box, box_npoints, ws, wsb, (cudaStream_t)stream);
}
extern "C" int d3d_crop2dr_assign_batch_f64(const double *points, int64_t total_points, const int64_t *point_offsets, const double *boxes,
                                            int64_t total_boxes, const int64_t *box_offsets, int64_t nframes, int64_t max_frame_points,
                                            int64_t max_frame_boxes, int project_axis, int64_t *point_box, int64_t *box_npoints, void *ws, size_t wsb,
                                            void *stream)
{
    return crop_assign_batch_impl<double>(points, total_points, point_offsets, boxes, total_boxes, box_offsets, nframes, max_frame_points,
                                          max_frame_boxes, project_axis, point_box, box_npoints, ws, wsb, (cudaStream_t)stream);
}
