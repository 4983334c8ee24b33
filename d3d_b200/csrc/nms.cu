// nms.cu -- greedy hard NMS on rotated boxes (or their AABBs) with 64-bit suppression words.
//
// Replaces reference nms2d / nms2d_cuda (d3d/box/nms.cpp:9-119, d3d/box/nms_cuda.cu:16-244).
// Pipeline, all asynchronous on the caller's stream (the reference syncs the device three times):
//   1. keys: score -> order-preserving integer key (descending), our stable radix sort (prims.cu)
//      => order[]; ties keep the lower original index first (the reference's torch.argsort leaves
//      ties unspecified, nms.cpp:103).
//   2. gather + prep: sorted box records (geom.cuh) and the score-threshold flag (score > thr, the
//      reference CUDA rule nms_cuda.cu:223).
//   3. mask: one CTA per 64x64 tile of the upper triangle of the sorted IoU matrix.  Same warp-queue
//      compaction as the IoU kernel: cheap bounding-circle reject, survivors clipped by full warps,
//      `iou > thr` sets bit (col) of the row's 64-bit word with a shared-memory atomicOr.
//   4. resolve: one CTA walks the 64-box blocks in score order.  The 64x64 diagonal word block is
//      resolved by a single thread with register bit-ops; the rows of the survivors are then OR-ed
//      into the removal bitmap by all threads in parallel (coalesced, independent loads).  The
//      reference does this whole phase in a <<<1,1>>> kernel (nms_cuda.cu:79-106,201).
//      The suppression matrix is sparse (a proposal overlaps a few dozen others): the mask kernels also
//      append every non-zero word to a list per 64-row block, and the resolve walks those lists, streamed
//      through shared memory four blocks ahead with cp.async, so that a block costs a few hundred cycles of
//      shared-memory work instead of two dependent L2 round trips.  The dense matrix remains the fallback
//      (a list overflow, or more than 8192 blocks).
#include "geom.cuh"
#include "prims.cuh"
#include <cuda_pipeline.h>
#include <stdlib.h>

namespace d3d {

template <typename T> struct KeyBits;
template <> struct KeyBits<float>  { static constexpr int bits = 32; };
template <> struct KeyBits<double> { static constexpr int bits = 64; };

// descending-order key: larger score -> smaller key.  -0.0 and +0.0 compare equal in the reference
// (float comparison), so both map to the key of +0.0.
__device__ __forceinline__ uint64_t desc_key(float s)
{
    if (s == 0.0f) s = 0.0f;
    uint32_t u = __float_as_uint(s);
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);   // ascending order-preserving
    return (uint64_t)(~u);
}
__device__ __forceinline__ uint64_t desc_key(double s)
{
    if (s == 0.0) s = 0.0;
    uint64_t u = (uint64_t)__double_as_longlong(s);
    u = (u >> 63) ? ~u : (u | 0x8000000000000000ull);
    return ~u;
}

template <typename T>
__global__ void __launch_bounds__(256) nms_keys_kernel(const T *__restrict__ scores, int64_t n, uint64_t *__restrict__ keys, uint32_t *__restrict__ vals)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    keys[i] = desc_key(scores[i]);
    vals[i] = (uint32_t)i;
}

constexpr int NMS_TILE = 64;

// extent of the box centres and the largest bounding radius, reduced by the gather kernel for the candidate grid: five minima of
// order-preserving encodings of x, y, -x, -y, -rho (one memset to 0xff initialises all of them) and a word that is cleared when a box
// is not finite
struct NmsExt { unsigned long long v[5]; uint32_t good, pad; };
__device__ __forceinline__ unsigned long long ext_enc(double x)
{
    const unsigned long long u = (unsigned long long)__double_as_longlong(x);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double ext_dec(unsigned long long e)
{
    return __longlong_as_double((long long)((e >> 63) ? (e & 0x7fffffffffffffffull) : ~e));
}

// sorted position p -> record of box order[p]; padded to a multiple of 64 with NaN-rho records
template <typename T, bool AABB>
__global__ void __launch_bounds__(256) nms_gather_kernel(const T *__restrict__ boxes, const T *__restrict__ scores, const uint32_t *__restrict__ order,
                                                         int64_t n, int64_t npad, float score_thr, BoxRec<T> *__restrict__ recs,
                                                         AABBRec<T> *__restrict__ arecs, T *__restrict__ raw, uint8_t *__restrict__ valid, NmsExt *__restrict__ ext)
{
    int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double e[5] = {1e300, 1e300, 1e300, 1e300, 0.0};   // x, y, -x, -y, -rho
    int bad = 0;
    if (p < n) {
        const uint32_t i = order[p];
        const T *b = boxes + 5 * (int64_t)i;
        if (AABB) arecs[p] = make_aabb_rec<T>(b[0], b[1], b[2], b[3], b[4]);
        else {
            const BoxRec<T> r = make_box_rec<T>(b[0], b[1], b[2], b[3], b[4]);
            recs[p] = r;
            if (raw) { for (int k = 0; k < 5; k++) raw[5 * p + k] = b[k]; }
            const double x = (double)r.cx, y = (double)r.cy, rho = (double)r.rho;
            if (!(fabs(x) < 1e150) || !(fabs(y) < 1e150) || !(rho < 1e150) || !(rho >= 0)) bad = 1;
            else { e[0] = x; e[1] = y; e[2] = -x; e[3] = -y; e[4] = -rho; }
        }
        valid[p] = scores[i] > score_thr ? 1 : 0;   // T vs float, promoted to T (nms.cpp:26, nms_cuda.cu:223)
    } else if (p < npad) {
        if (AABB) { AABBRec<T> a; a.minx = a.maxx = a.miny = a.maxy = T(NAN); arecs[p] = a; }
        else { BoxRec<T> r; r.cx = r.cy = r.c = r.s = r.hw = r.hh = r.area = T(0); r.rho = T(NAN); recs[p] = r; }
        valid[p] = 0;
    }
    if (AABB || !ext) return;   // (uniform)
    __shared__ double sred[5][8];
    __shared__ int sbad;
    if (threadIdx.x == 0) sbad = 0;
#pragma unroll
    for (int k = 0; k < 5; k++)
#pragma unroll
        for (int d = 16; d; d >>= 1) e[k] = fmin(e[k], __shfl_xor_sync(0xffffffffu, e[k], d));
    bad = __any_sync(0xffffffffu, bad);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int k = 0; k < 5; k++) sred[k][threadIdx.x >> 5] = e[k];
        if (bad) sbad = 1;
    }
    __syncthreads();
    if (threadIdx.x < 5) {
        double m = sred[threadIdx.x][0];
        for (int w = 1; w < 8; w++) m = fmin(m, sred[threadIdx.x][w]);
        atomicMin(&ext->v[threadIdx.x], ext_enc(m));
    }
    if (threadIdx.x == 5 && sbad) atomicAnd(&ext->good, 0u);
}

constexpr int NMS_THREADS = 128;
constexpr int NMS_WARPS = NMS_THREADS / 32;

// fp32 decisions within this distance of the threshold are re-evaluated in fp64 from the raw boxes,
// so that the float path reproduces the decisions of the double path (SURVEY.md 8(c), T1)
#define NMS_F32_RECHECK 1e-3f

template <typename T>
__device__ __forceinline__ bool over_threshold(T v, T thr, const T *raw, unsigned gi, unsigned gj)
{
    (void)raw; (void)gi; (void)gj;
    return v > thr;
}
template <>
__device__ __forceinline__ bool over_threshold<float>(float v, float thr, const float *raw, unsigned gi, unsigned gj)
{
    if (raw && v != 0.0f && fabsf(v - thr) < NMS_F32_RECHECK) {   // an exact 0 is a pair the clip found disjoint: nothing to re-evaluate
        const float *a = raw + 5 * (int64_t)gi, *b = raw + 5 * (int64_t)gj;
        BoxRec<double> A = make_box_rec<double>(a[0], a[1], a[2], a[3], a[4]);
        BoxRec<double> B = make_box_rec<double>(b[0], b[1], b[2], b[3], b[4]);
        return rbox_iou<double>(A, B) > (double)thr;
    }
    return v > thr;
}

// ---- sparse side product of the mask kernels: the non-zero words of row block rb, in any order
constexpr uint32_t NMS_LIST_CAP = 4096;      // entries per 64-row block (64 rows x 64 words); more -> dense resolve
struct NmsLists {
    uint32_t *blkcnt;      // [nwords] entries appended per row block; blkcnt[nwords] = overflow flag
    uint32_t *ent_w;       // [nwords * NMS_LIST_CAP] column word index | row inside the block << 16
    uint64_t *ent_bits;    // [nwords * NMS_LIST_CAP]
};

// called by every thread of the CTA after the tile's words are final in smask[] (one per row, threads < NMS_TILE own them)
__device__ __forceinline__ void nms_append_tile(const NmsLists &L, const unsigned long long *smask, int64_t rb, int64_t cb, int64_t n, int64_t nwords,
                                                uint32_t *s_cnt, uint32_t *s_base)
{
    if (!L.blkcnt) return;
    const unsigned tid = threadIdx.x;
    if (tid == 0) *s_cnt = 0;
    __syncthreads();
    unsigned long long bits = 0;
    uint32_t rank = 0;
    if (tid < NMS_TILE && rb * NMS_TILE + tid < n) bits = smask[tid];
    if (bits) rank = atomicAdd(s_cnt, 1u);
    __syncthreads();
    const uint32_t cnt = *s_cnt;
    if (cnt == 0) return;   // CTA-uniform
    if (tid == 0) {
        const uint32_t base = atomicAdd(L.blkcnt + rb, cnt);
        if (base + cnt > NMS_LIST_CAP) L.blkcnt[nwords] = 1u;
        *s_base = base;
    }
    __syncthreads();
    const uint32_t at = *s_base + rank;
    if (bits && at < NMS_LIST_CAP) {
        L.ent_w[rb * NMS_LIST_CAP + at] = (uint32_t)cb | (tid << 16);
        L.ent_bits[rb * NMS_LIST_CAP + at] = bits;
    }
}

// ---- spatial candidate search (rbox).  Boxes whose bounding circles overlap lie in adjacent cells of a grid whose cell
// is wider than 2 * max rho, so a box meets all its candidates in 3x3 cells instead of the whole upper triangle of
// the sorted matrix (C3: ~500 candidates per box instead of 25 000).  Everything is decided on the device: when the
// geometry does not allow a grid (non-finite boxes, no extent, too few cells) or a list overflows, the dense tile
// kernel below runs instead -- otherwise its CTAs exit on their first instruction.
constexpr int NMS_GRID_MAX = 256;                                   // cells per axis
constexpr int NMS_GRID_CELLS = NMS_GRID_MAX * NMS_GRID_MAX;
struct NmsGrid { double minx, miny, inv_cell; int nx, ny; uint32_t ok; uint32_t pad; };
// what the candidate scan needs of a box, stored in cell order so that a warp reads consecutive records
// (single precision whatever the box type: 16 bytes per entry.  The circle test on these numbers is widened by the conversion error of
// the centres, so it passes a superset of the pairs whose circles meet -- the clip decides, the keep mask does not depend on it)
// The entry also carries the numbers of the area bound (axes, half extents grown by 1e-6, area): a tile of the cell kernel stages its
// columns with one coalesced pass over the list, no gather of records.
struct __align__(16) NmsCandF { float cx, cy, rho; uint32_t idx; float c, s, hw, hh; float area, pad0, pad1, pad2; };
template <typename T> using NmsCand = NmsCandF;

// grid geometry from the extents the gather kernel reduced (one thread)
__global__ void nms_grid_kernel(const NmsExt *__restrict__ ext, int64_t n, NmsGrid *__restrict__ g)
{
    if (threadIdx.x != 0) return;
    const double mnx = ext_dec(ext->v[0]), mny = ext_dec(ext->v[1]), mxx = -ext_dec(ext->v[2]), mxy = -ext_dec(ext->v[3]), mr = -ext_dec(ext->v[4]);
    const bool bad = ext->good == 0u || !(mnx <= mxx) || !(mny <= mxy);
    NmsGrid o;
    o.minx = mnx; o.miny = mny; o.inv_cell = 0; o.nx = o.ny = 1; o.ok = 0; o.pad = 0;
    const double ex = mxx - mnx, ey = mxy - mny;
    double cell = 2.0 * mr * (1.0 + 1e-6);     // the margin absorbs the rounding of the cell index
    cell = fmax(cell, fmax(ex, ey) / NMS_GRID_MAX * (1.0 + 1e-6));
    if (!bad && n > 0 && cell > 0 && cell < 1e150) {
        const int nx = (int)fmin((double)NMS_GRID_MAX, floor(ex / cell) + 1), ny = (int)fmin((double)NMS_GRID_MAX, floor(ey / cell) + 1);
        if ((int64_t)nx * ny >= 16) { o.inv_cell = 1.0 / cell; o.nx = nx; o.ny = ny; o.ok = 1; }
    }
    *g = o;
}

template <typename T>
__device__ __forceinline__ void nms_cell_of(const NmsGrid &g, const BoxRec<T> &r, int *ix, int *iy)
{
    // clamping merges cells at the border: a superset of candidates, never a miss
    *ix = min(g.nx - 1, max(0, (int)floor(((double)r.cx - g.minx) * g.inv_cell)));
    *iy = min(g.ny - 1, max(0, (int)floor(((double)r.cy - g.miny) * g.inv_cell)));
}

// pass 0: count boxes per cell; pass 1: fill the cell lists (order inside a cell is arbitrary: results are ORs)
template <typename T, int PASS>
__global__ void __launch_bounds__(256) nms_bin_kernel(const BoxRec<T> *__restrict__ recs, int64_t n, const NmsGrid *__restrict__ g,
                                                      uint32_t *__restrict__ cellcnt, const uint32_t *__restrict__ cellptr, NmsCand<T> *__restrict__ celllist)
{
    if (!g->ok) return;
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    int ix, iy;
    const BoxRec<T> r = recs[p];
    nms_cell_of<T>(*g, r, &ix, &iy);
    const uint32_t c = (uint32_t)(iy * g->nx + ix);
    const uint32_t at = atomicAdd(cellcnt + c, 1u);
    if (PASS == 1) {
        NmsCand<T> e;
        e.cx = (float)r.cx; e.cy = (float)r.cy; e.rho = __double2float_ru((double)r.rho); e.idx = (uint32_t)p;
        e.c = (float)r.c; e.s = (float)r.s; e.hw = (float)r.hw * 1.000001f; e.hh = (float)r.hh * 1.000001f;
        e.area = (float)r.area; e.pad0 = e.pad1 = e.pad2 = 0.f;
        celllist[cellptr[c] + at] = e;
    }
}

// A pair can only pass an IoU threshold t if its intersection exceeds t / (1 + t) of the two areas together (IoU = I / (S - I)), and the
// intersection lies inside box B and inside the bounding rectangle of box A in B's frame, so I <= ox * oy, the overlaps of those two
// rectangles along B's axes.  For the near-parallel proposals around one object this bound is almost the intersection itself, and most
// pairs whose circles meet but whose IoU stays below the threshold never reach the clip.  Single precision: the overlaps are grown by
// what the converted centres may be off by (err) and the comparison keeps a 1e-3 margin, so the test only drops pairs whose true IoU is
// below the threshold -- the keep mask cannot change.  (px, py): A's centre in B's frame needs B's axes (bc, bs).
struct NmsShape { float c, s, hw, hh; };
__device__ __forceinline__ bool nms_area_bound(const float dx, const float dy, const NmsShape A, const float areaA, const NmsShape B, const float areaB,
                                               const float err, const float tau)
{
    const float px = B.c * dx + B.s * dy, py = B.c * dy - B.s * dx;
    const float cr = fabsf(A.c * B.c + A.s * B.s), sr = fabsf(A.s * B.c - A.c * B.s);
    const float ex = cr * A.hw + sr * A.hh + err, ey = sr * A.hw + cr * A.hh + err;
    const float ox = fminf(B.hw, px + ex) - fmaxf(-B.hw, px - ex), oy = fminf(B.hh, py + ey) - fmaxf(-B.hh, py - ey);
    return fmaxf(ox, 0.f) * fmaxf(oy, 0.f) * 1.001f >= tau * (areaA + areaB);
}

// ---- the candidate search, a CTA per grid cell.  The boxes of one cell are the rows of a tile and the boxes of its 3x3 neighbourhood the columns, both staged in shared
// memory; every thread tests its column against the rows (single precision, widened as above), the survivors of a 64 x 128 tile go to
// one queue of the CTA, and the warps clip them 32 at a time -- full warps except for the tile's last step.  The hits of a row chunk wait in
// shared memory and are appended to their rows' block lists together (the atomics' round trips overlap).  NC_SPLIT work items share a cell,
// each taking every NC_SPLIT-th column chunk.
#ifndef D3D_NC_SPLIT
#define D3D_NC_SPLIT 4
#endif
#ifndef D3D_NC_CTAS
#define D3D_NC_CTAS 4
#endif
constexpr int NC_ROWS = 64, NC_COLS = 128, NC_THREADS = 256, NC_SPLIT = D3D_NC_SPLIT, NC_HB = 1024;

template <typename T>
__global__ void __launch_bounds__(NC_THREADS, D3D_NC_CTAS) nms_cells_kernel(const BoxRec<T> *__restrict__ recs, const T *__restrict__ raw, int64_t n, int64_t nwords, T thr,
                                                                  const NmsGrid *__restrict__ g, const uint32_t *__restrict__ cellptr,
                                                                  const NmsCand<T> *__restrict__ celllist, const NmsLists lists, uint32_t *__restrict__ ticket)
{
    if (!g->ok) return;
    const NmsGrid G = *g;
    __shared__ BoxRec<T> sR[NC_ROWS];
    __shared__ float4 fR[NC_ROWS];                    // centre, widened radius, index (bits) of the rows
    __shared__ NmsShape gR[NC_ROWS];                  // axes and half extents of the rows (area bound)
    __shared__ float aR[NC_ROWS], eR[NC_ROWS];        // area, coordinate error of the rows
    __shared__ uint32_t cidx[NC_COLS];
    extern __shared__ __align__(16) uint16_t queue0[];   // [NC_ROWS * NC_COLS] row << 8 | column of the pairs that passed the circle test (dynamic: 56 KB in all)
    __shared__ uint16_t queue[NC_ROWS * NC_COLS];     // ... and the area bound: the clip queue
    __shared__ NmsShape gC[NC_COLS];                  // axes and half extents of the columns
    __shared__ float4 cC[NC_COLS];                    // centre, area, coordinate error of the columns
    __shared__ uint2 hbuf[NC_HB];                     // hits (row box, column box) of the row chunk
    __shared__ uint32_t seg_beg[3], seg_off[4], qn, qn0, hn, s_item;
    const unsigned tid = threadIdx.x, lane = tid & 31u, w = tid >> 5;
    auto append = [&](const uint32_t i, const uint32_t j) {   // one entry of row i's 64-row block
        const uint32_t rb = i >> 6, at = atomicAdd(lists.blkcnt + rb, 1u);
        if (at < NMS_LIST_CAP) {
            lists.ent_w[(size_t)rb * NMS_LIST_CAP + at] = (j >> 6) | ((i & 63u) << 16);
            lists.ent_bits[(size_t)rb * NMS_LIST_CAP + at] = 1ull << (j & 63u);
        } else lists.blkcnt[nwords] = 1u;
    };
    // work items (cell, share of the column chunks) are handed out by a ticket counter (the grid does not know how many cells the frame has;
    // the counter starts at 0xffffffff: it shares the memset of the extents)
    const uint32_t items = (uint32_t)(G.nx * G.ny) * NC_SPLIT;
    const float tau = (float)thr / (1.f + (float)thr) * 0.999999f;
  for (;;) {
    __syncthreads();   // the previous item is done with the shared words
    if (tid == 0) s_item = atomicAdd(ticket, 1u) + 1u;
    __syncthreads();
    const uint32_t item = s_item;
    if (item >= items) break;
    const int cell = (int)(item / NC_SPLIT);
    const uint32_t split = item % NC_SPLIT;
    const uint32_t r_beg = cellptr[cell], r_end = cellptr[cell + 1];
    if (r_beg == r_end) continue;   // (CTA-uniform)
    if (tid == 0) {   // the three cells of a grid row are contiguous in the cell-sorted list
        const int ix = cell % G.nx, iy = cell / G.nx;
        uint32_t off = 0;
        for (int k = 0; k < 3; k++) {
            const int cy = iy + k - 1;
            uint32_t beg = 0, len = 0;
            if (cy >= 0 && cy < G.ny) {
                const int x0 = max(ix - 1, 0), x1 = min(ix + 1, G.nx - 1);
                beg = cellptr[cy * G.nx + x0];
                len = cellptr[cy * G.nx + x1 + 1] - beg;
            }
            seg_beg[k] = beg; seg_off[k] = off; off += len;
        }
        seg_off[3] = off;
        hn = 0;
    }
    __syncthreads();
    const uint32_t ncols = seg_off[3];
    for (uint32_t rc = r_beg; rc < r_end; rc += NC_ROWS) {
        const uint32_t nr = min((uint32_t)NC_ROWS, r_end - rc);
        __syncthreads();   // the previous row chunk is done with the row arrays
        if (tid < nr) {
            const NmsCand<T> e = celllist[rc + tid];
            const BoxRec<T> rr = recs[e.idx];
            sR[tid] = rr;
            const float er = (fabsf(e.cx) + fabsf(e.cy)) * 2.4e-7f;   // 2^-22 of the coordinates: what the float centres may be off by
            fR[tid] = make_float4(e.cx, e.cy, e.rho + er, __uint_as_float(e.idx));
            NmsShape sh; sh.c = e.c; sh.s = e.s; sh.hw = e.hw; sh.hh = e.hh;
            gR[tid] = sh; aR[tid] = e.area; eR[tid] = er;
        }
        for (uint32_t cc = split * NC_COLS; cc < ncols; cc += NC_SPLIT * NC_COLS) {
            __syncthreads();   // rows staged; the previous tile is done with the columns and the queue
            if (tid == 0) { qn = 0; qn0 = 0; }
            const uint32_t c = tid & (NC_COLS - 1), v = cc + c;
            const bool have = v < ncols;
            NmsCand<T> ce;
            ce.cx = ce.cy = ce.rho = 0.f; ce.idx = 0;
            if (have) {
                const int sg = v >= seg_off[2] ? 2 : (v >= seg_off[1] ? 1 : 0);
                ce = celllist[seg_beg[sg] + (v - seg_off[sg])];
                if (tid < NC_COLS) {
                    cidx[c] = ce.idx;
                    NmsShape sh; sh.c = ce.c; sh.s = ce.s; sh.hw = ce.hw; sh.hh = ce.hh;
                    gC[c] = sh; cC[c] = make_float4(ce.cx, ce.cy, ce.area, (fabsf(ce.cx) + fabsf(ce.cy)) * 2.4e-7f);
                }
            }
            __syncthreads();
            const float cerr = (fabsf(ce.cx) + fabsf(ce.cy)) * 2.4e-7f, cr = ce.rho + cerr;
            for (uint32_t r = tid / NC_COLS; r < nr; r += NC_THREADS / NC_COLS) {   // (warp-uniform r)
                const float4 f = fR[r];
                const float dx = f.x - ce.cx, dy = f.y - ce.cy, rs = f.z + cr;
                const bool cand = have && ce.idx > __float_as_uint(f.w) && dx * dx + dy * dy <= rs * rs * 1.00001f;   // every unordered pair once: from its higher-scored box
                const unsigned bal = __ballot_sync(0xffffffffu, cand);
                if (bal) {
                    uint32_t at = 0;
                    if (lane == 0) at = atomicAdd(&qn0, (uint32_t)__popc(bal));
                    at = __shfl_sync(0xffffffffu, at, 0);
                    if (cand) queue0[at + __popc(bal & lanemask_lt())] = (uint16_t)((r << 8) | c);
                }
            }
            __syncthreads();
            // the area bound on the survivors of the circle test, all lanes busy; what passes goes to the clip queue
            const uint32_t n0 = qn0;
            for (uint32_t e0 = w * 32u; e0 < n0; e0 += (NC_THREADS / 32) * 32u) {
                const bool live = e0 + lane < n0;
                const uint32_t ent = queue0[live ? e0 + lane : n0 - 1], r = ent >> 8, cq = ent & 255u;
                const float4 f = fR[r];
                const bool cand = live && nms_area_bound(f.x - cC[cq].x, f.y - cC[cq].y, gR[r], aR[r], gC[cq], cC[cq].z, 2.f * (eR[r] + cC[cq].w), tau);
                const unsigned bal = __ballot_sync(0xffffffffu, cand);
                if (bal) {
                    uint32_t at = 0;
                    if (lane == 0) at = atomicAdd(&qn, (uint32_t)__popc(bal));
                    at = __shfl_sync(0xffffffffu, at, 0);
                    if (cand) queue[at + __popc(bal & lanemask_lt())] = (uint16_t)ent;
                }
            }
            __syncthreads();
            const uint32_t nq = qn;
            for (uint32_t e0 = w * 32u; e0 < nq; e0 += (NC_THREADS / 32) * 32u) {
                const bool live = e0 + lane < nq;
                const uint32_t ent = queue[live ? e0 + lane : nq - 1];
                const uint32_t r = ent >> 8, cq = ent & 255u;
                const uint32_t i = __float_as_uint(fR[r].w), j = cidx[cq];
                const T iou = rbox_iou<T>(sR[r], recs[j]);   // iou(higher score box, lower score box), nms.cpp:50; few pairs get here: the column's record comes from L2
                if (live && over_threshold<T>(iou, thr, raw, i, j)) {
                    const uint32_t h = atomicAdd(&hn, 1u);
                    if (h < (uint32_t)NC_HB) hbuf[h] = make_uint2(i, j);
                    else append(i, j);
                }
            }
        }
        __syncthreads();
        const uint32_t nh = min(hn, (uint32_t)NC_HB);
        for (uint32_t h = tid; h < nh; h += NC_THREADS) append(hbuf[h].x, hbuf[h].y);
        __syncthreads();
        if (tid == 0) hn = 0;
    }
  }
}

template <typename T>
__device__ __forceinline__ void nms_mask_rbox_body(const BoxRec<T> *__restrict__ recs, const T *__restrict__ raw, int64_t n, int64_t nwords, T thr, uint64_t *__restrict__ mask,
                                                   const NmsLists lists, const int64_t cb, const int64_t rb_first, const int64_t rb_stride)
{
    // one CTA per column tile cb and per residue of the row tile: rb = rb_first, rb_first + rb_stride, ... <= cb
    if (cb < rb_first) return;
    constexpr int RW = NMS_TILE / NMS_WARPS;  // 16 rows per warp
    constexpr int KC = NMS_TILE / 32;         // 2 column chunks
    __shared__ BoxRec<T> sA[NMS_TILE];
    __shared__ BoxRec<T> sB[NMS_TILE];
    __shared__ unsigned long long smask[NMS_TILE];
    __shared__ uint16_t queue[NMS_WARPS][128];
    __shared__ uint32_t s_cnt, s_base;
    const unsigned lane = lane_id(), w = threadIdx.x >> 5;
    constexpr int NV = NMS_TILE * sizeof(BoxRec<T>) / 16;
    {
        const float4 *gb = reinterpret_cast<const float4 *>(recs + cb * NMS_TILE);
        float4 *db = reinterpret_cast<float4 *>(sB);
        for (int i = threadIdx.x; i < NV; i += NMS_THREADS) db[i] = __ldg(gb + i);
    }
    __syncthreads();
    T bx[KC], by[KC], br[KC];
#pragma unroll
    for (int k = 0; k < KC; k++) { bx[k] = sB[k * 32 + lane].cx; by[k] = sB[k * 32 + lane].cy; br[k] = sB[k * 32 + lane].rho; }
    uint16_t *q = queue[w];
  for (int64_t rb = rb_first; rb <= cb; rb += rb_stride) {
    {
        const float4 *ga = reinterpret_cast<const float4 *>(recs + rb * NMS_TILE);
        float4 *da = reinterpret_cast<float4 *>(sA);
        for (int i = threadIdx.x; i < NV; i += NMS_THREADS) da[i] = __ldg(ga + i);
        if (threadIdx.x < NMS_TILE) smask[threadIdx.x] = 0ull;
    }
    __syncthreads();
    unsigned head = 0, tail = 0;
    const bool diag = (rb == cb);
#pragma unroll 1
    for (int r = 0; r <= RW; r++) {
        if (r < RW) {
            const unsigned rl = w * RW + r;
            const BoxRec<T> &a = sA[rl];
            const T ax = a.cx, ay = a.cy, ar = a.rho;
#pragma unroll
            for (int k = 0; k < KC; k++) {
                T dx = ax - bx[k], dy = ay - by[k], rs = ar + br[k];
                bool cand = ((dx * dx + dy * dy <= rs * rs) || thr < T(0)) && (!diag || (unsigned)(k * 32 + lane) > rl);   // thr < 0: disjoint pairs (IoU 0) suppress too, like the reference
                unsigned bal = __ballot_sync(0xffffffffu, cand);
                if (cand) q[(tail + __popc(bal & lanemask_lt())) & 127] = (uint16_t)((rl << 8) | (k * 32 + lane));
                tail += __popc(bal);
            }
        }
        while (tail - head >= 32u || (r == RW && tail != head)) {
            __syncwarp();
            unsigned cnt = min(tail - head, 32u);
            unsigned e = q[(head + min(lane, cnt - 1)) & 127];
            const unsigned row = e >> 8, col = e & 255u;
            BoxRec<T> A = sA[row], B = sB[col];
            T v = rbox_iou<T>(A, B);   // iou(higher score box, lower score box), nms.cpp:50
            if (lane < cnt && over_threshold<T>(v, thr, raw, (unsigned)(rb * NMS_TILE + row), (unsigned)(cb * NMS_TILE + col)))
                atomicOr(&smask[row], 1ull << col);
            head += cnt;
            __syncwarp();
        }
    }
    __syncthreads();
    if (threadIdx.x < NMS_TILE) {
        int64_t row = rb * NMS_TILE + threadIdx.x;
        if (row < n) mask[row * nwords + cb] = smask[threadIdx.x];
    }
    nms_append_tile(lists, smask, rb, cb, n, nwords, &s_cnt, &s_base);
    __syncthreads();   // sA, smask and the counters are reused by the next row tile
  }
}

template <typename T>
__global__ void __launch_bounds__(NMS_THREADS)
nms_mask_rbox_kernel(const BoxRec<T> *__restrict__ recs, const T *__restrict__ raw, int64_t n, int64_t nwords, T thr, uint64_t *__restrict__ mask, const NmsLists lists,
                     const NmsGrid *__restrict__ grid)
{
    // The short grid (gridDim.y row residues) keeps the launch cheap when the spatial path has already produced the lists and every
    // CTA leaves at once.
    if (grid && grid->ok && lists.blkcnt[nwords] == 0u) return;   // the spatial path produced the lists: nothing to do
    nms_mask_rbox_body<T>(recs, raw, n, nwords, thr, mask, lists, blockIdx.x, blockIdx.y, gridDim.y);
}

// AABB variant: every pair is a handful of instructions, no queue needed.  One CTA of NMS_TILE threads per tile (rb, cb), a thread per row.
template <typename T>
__device__ __forceinline__ void nms_mask_aabb_body(const AABBRec<T> *__restrict__ recs, int64_t n, int64_t nwords, T thr, uint64_t *__restrict__ mask,
                                                   const NmsLists lists, const int64_t rb, const int64_t cb)
{
    if (cb < rb || cb * NMS_TILE >= n) return;   // below the diagonal, or past the end of a batch frame shorter than the grid
    __shared__ AABBRec<T> sB[NMS_TILE];
    __shared__ unsigned long long smask[NMS_TILE];
    __shared__ uint32_t s_cnt, s_base;
    sB[threadIdx.x] = recs[cb * NMS_TILE + threadIdx.x];
    __syncthreads();
    const int64_t row = rb * NMS_TILE + threadIdx.x;
    unsigned long long bits = 0;
    if (row < n) {
        const AABBRec<T> a = recs[row];
        const int start = (rb == cb) ? threadIdx.x + 1 : 0;
        for (int c = start; c < NMS_TILE; c++) {
            if (cb * NMS_TILE + c >= n) break;
            if (aabb_iou<T>(a, sB[c]) > thr) bits |= 1ull << c;
        }
        mask[row * nwords + cb] = bits;
    }
    if (!lists.blkcnt) return;   // (CTA-uniform)
    smask[threadIdx.x] = bits;
    __syncthreads();
    nms_append_tile(lists, smask, rb, cb, n, nwords, &s_cnt, &s_base);
}

template <typename T>
__global__ void __launch_bounds__(NMS_TILE)
nms_mask_aabb_kernel(const AABBRec<T> *__restrict__ recs, int64_t n, int64_t nwords, T thr, uint64_t *__restrict__ mask, const NmsLists lists)
{
    nms_mask_aabb_body<T>(recs, n, nwords, thr, mask, lists, blockIdx.y, blockIdx.x);
}

constexpr int RESOLVE_THREADS = 1024;

constexpr int RS_STAGES = 6;          // blocks of list entries in flight

// shared-memory OR of a 64-bit word through its 32-bit halves (native ATOMS.OR; the 64-bit form is a CAS loop)
__device__ __forceinline__ void smem_or64(unsigned long long *word, unsigned long long bits)
{
    uint32_t *h = reinterpret_cast<uint32_t *>(word);
    const uint32_t lo = (uint32_t)bits, hi = (uint32_t)(bits >> 32);
    if (lo) atomicOr(h, lo);
    if (hi) atomicOr(h + 1, hi);
}

// greedy pass over one 64-box block: cur = boxes already removed, diag[t] = boxes of the block that box t removes.
// This chain is the critical path of the whole resolve (one thread, every step depends on the previous one), so it
// jumps from survivor to survivor (a handful per block) and works on 32-bit halves: find-first-set, one shared-memory
// load, two ORs and one mask per survivor.
__device__ __forceinline__ unsigned long long nms_resolve_diag(unsigned long long cur, const unsigned long long *diag)
{
    uint32_t clo = (uint32_t)cur, chi = (uint32_t)(cur >> 32), klo = 0, khi = 0;
    const uint2 *d2 = reinterpret_cast<const uint2 *>(diag);
    uint32_t cand = ~clo;
#pragma unroll 1
    while (cand) {          // boxes 0..31: a survivor removes boxes of both halves
        const int t = __ffs((int)cand) - 1;
        klo |= 1u << t;
        const uint2 row = d2[t];
        clo |= row.x; chi |= row.y;
        cand = ~clo & (0xfffffffeu << t);
    }
    cand = ~chi;
#pragma unroll 1
    while (cand) {          // boxes 32..63
        const int t = __ffs((int)cand) - 1;
        khi |= 1u << t;
        chi |= d2[32 + t].y;
        cand = ~chi & (0xfffffffeu << t);
    }
    return (unsigned long long)klo | ((unsigned long long)khi << 32);
}

// boxes at or below the score threshold (and the padding past n) start out removed
__device__ __forceinline__ void nms_removed_init(unsigned long long *remv, int64_t n, int64_t nwords, const uint8_t *__restrict__ valid)
{
    for (int64_t w = threadIdx.x; w < nwords; w += blockDim.x) {
        unsigned long long b = 0;
        for (int t = 0; t < 64; t++) {
            const int64_t p = w * 64 + t;
            if (p >= n || !valid[p]) b |= 1ull << t;
        }
        remv[w] = b;
    }
}

// the walk over a dense suppression matrix (rows of `stride` words, the first nwords of them used) by the whole CTA, after
// nms_removed_init: per 64-box block, thread 0 resolves the diagonal word block, then the survivors' rows are ORed into the bitmap
__device__ __forceinline__ void nms_dense_walk(const uint64_t *__restrict__ mask, int64_t stride, int64_t n, int64_t nwords, const uint32_t *__restrict__ order,
                                               uint8_t *__restrict__ suppressed, unsigned long long *remv, unsigned long long *diag0, unsigned long long *keptbits)
{
    const int tid = threadIdx.x;
    const uint32_t NT = blockDim.x;
    __syncthreads();
    for (int64_t blk = 0; blk < nwords; blk++) {
        if (tid < 64) {
            const int64_t row = blk * 64 + tid;
            diag0[tid] = row < n ? mask[row * stride + blk] : 0ull;
        }
        __syncthreads();
        if (tid == 0) *keptbits = nms_resolve_diag(remv[blk], diag0);
        __syncthreads();
        const unsigned long long kept = *keptbits;
        if (tid < 64) {
            const int64_t row = blk * 64 + tid;
            if (row < n) suppressed[order[row]] = ((kept >> tid) & 1ull) ? 0 : 1;
        }
        if (kept) {
            for (int64_t w = blk + 1 + tid; w < nwords; w += NT) {
                unsigned long long acc = remv[w], k = kept;
                const uint64_t *col = mask + (blk * 64) * stride + w;
                while (k) {   // up to 4 independent row loads in flight
                    const int t0 = __ffsll((long long)k) - 1; k &= k - 1;
                    unsigned long long v0 = col[(int64_t)t0 * stride], v1 = 0, v2 = 0, v3 = 0;
                    if (k) { const int t1 = __ffsll((long long)k) - 1; k &= k - 1; v1 = col[(int64_t)t1 * stride]; }
                    if (k) { const int t2 = __ffsll((long long)k) - 1; k &= k - 1; v2 = col[(int64_t)t2 * stride]; }
                    if (k) { const int t3 = __ffsll((long long)k) - 1; k &= k - 1; v3 = col[(int64_t)t3 * stride]; }
                    acc |= v0 | v1 | v2 | v3;
                }
                remv[w] = acc;
            }
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(RESOLVE_THREADS)
nms_resolve_kernel(const uint64_t *__restrict__ mask, int64_t n, int64_t nwords, const uint8_t *__restrict__ valid,
                   const uint32_t *__restrict__ order, uint8_t *__restrict__ suppressed, const NmsLists lists, const uint32_t stage_cap,
                   const uint32_t *__restrict__ skip_if)
{
    extern __shared__ unsigned long long remv[];   // [nwords] removal bitmap in sorted order (+ the sparse path's arrays behind it)
    __shared__ unsigned long long diag[2][64];
    __shared__ unsigned long long keptbits;
    if (skip_if && *skip_if) return;   // the parallel resolve produced the keep mask (CTA-uniform)
    const int tid = threadIdx.x;
    const uint32_t NT = blockDim.x;   // >= 128
    nms_removed_init(remv, n, nwords, valid);
    const bool sparse = lists.blkcnt != nullptr && lists.blkcnt[nwords] == 0u;   // CTA-uniform: no list overflowed
    if (sparse) {
        // ---- sparse walk.  Per block: thread 0 resolves the diagonal tile while the other warps pick the diagonal words of the
        // NEXT block out of its staged list; barrier; everybody ORs the survivors' words into the bitmap; barrier.  The lists
        // arrive through cp.async RS_STAGES-1 blocks ahead, the keep bits leave in one pass at the end.
        const uint32_t SC = stage_cap;
        unsigned long long *keptw = remv + nwords;                                   // [nwords]
        unsigned long long *sbits = keptw + nwords;                                  // [RS_STAGES][SC]
        uint32_t *sw = reinterpret_cast<uint32_t *>(sbits + (size_t)RS_STAGES * SC); // [RS_STAGES][SC]
        uint32_t *cnts = sw + (size_t)RS_STAGES * SC;                                // [nwords]
        for (int64_t w = tid; w < nwords; w += NT) cnts[w] = min(lists.blkcnt[w], NMS_LIST_CAP);
        if (tid < 128) diag[tid >> 6][tid & 63] = 0ull;
        __syncthreads();
        auto issue = [&](int64_t b) {
            if (b < nwords) {
                const uint32_t c = min(cnts[b], SC);
                const int st = (int)(b % RS_STAGES);
                for (uint32_t e = tid; e < c; e += NT) {
                    __pipeline_memcpy_async(sw + st * SC + e, lists.ent_w + b * NMS_LIST_CAP + e, 4);
                    __pipeline_memcpy_async(sbits + st * SC + e, lists.ent_bits + b * NMS_LIST_CAP + e, 8);
                }
            }
            __pipeline_commit();
        };
        auto extract = [&](int64_t b, uint32_t first, uint32_t stride) {   // diagonal words of block b -> diag[b & 1] (zeroed beforehand)
            if (b >= nwords) return;
            const int st = (int)(b % RS_STAGES);
            const uint32_t c = cnts[b];
            const uint32_t *gw = lists.ent_w + b * NMS_LIST_CAP;
            const uint64_t *gb = lists.ent_bits + b * NMS_LIST_CAP;
            for (uint32_t e = first; e < c; e += stride) {
                const uint32_t we = e < SC ? sw[st * SC + e] : gw[e];
                if ((we & 0xffffu) == (uint32_t)b) smem_or64(&diag[b & 1][we >> 16], e < SC ? sbits[st * SC + e] : gb[e]);   // several entries may share a word
            }
        };
        for (int b = 0; b < RS_STAGES - 1; b++) issue(b);
        __pipeline_wait_prior(RS_STAGES - 3);   // blocks 0 and 1 have landed (this thread's copies)
        __syncthreads();
        extract(0, tid, NT);
        __syncthreads();
        for (int64_t blk = 0; blk < nwords; blk++) {
            // phase A: resolve blk (thread 0) | diagonal words of blk + 1 (everybody else)
            if (tid == 0) { const unsigned long long k = nms_resolve_diag(remv[blk], diag[blk & 1]); keptbits = k; keptw[blk] = k; }
            else if (tid >= 32) extract(blk + 1, tid - 32, NT - 32);
            __syncthreads();
            // phase B: the survivors' words of blk into the bitmap; recycle buffers; keep the pipeline full
            const unsigned long long kept = keptbits;
            if (tid < 64) diag[blk & 1][tid] = 0ull;   // next used by block blk + 2
            if (kept) {
                const int st = (int)(blk % RS_STAGES);
                const uint32_t c = cnts[blk];
                const uint32_t *gw = lists.ent_w + blk * NMS_LIST_CAP;
                const uint64_t *gb = lists.ent_bits + blk * NMS_LIST_CAP;
                for (uint32_t e = tid; e < c; e += NT) {
                    const uint32_t we = e < SC ? sw[st * SC + e] : gw[e];
                    if ((kept >> (we >> 16)) & 1ull) smem_or64(&remv[we & 0xffffu], e < SC ? sbits[st * SC + e] : gb[e]);
                }
            }
            issue(blk + RS_STAGES - 1);             // into stage (blk - 1) % RS_STAGES, last read before the previous iteration's final barrier
            __pipeline_wait_prior(RS_STAGES - 3);   // this thread's copies of block blk + 2 have landed ...
            __syncthreads();                        // ... and everybody's are visible; remv[blk + 1] is final
        }
        __syncthreads();
        for (int64_t row = tid; row < n; row += NT) suppressed[order[row]] = ((keptw[row >> 6] >> (row & 63)) & 1ull) ? 0 : 1;
        return;
    }
    nms_dense_walk(mask, nwords, n, nwords, order, suppressed, remv, diag[0], &keptbits);
}

// ------------------------------------------------------------------------------------------------ parallel resolve
// Greedy NMS keeps a box iff no KEPT box of higher score overlaps it.  The list walk above follows the score order block by block on
// one SM (782 dependent steps of ~1.2 us for 50 000 boxes).  The same keep mask is the fixpoint of two rules: a box is suppressed as soon
// as one of its higher-scored overlapping boxes is kept, and kept as soon as all of them are suppressed.  The highest-scored undecided
// box can always be decided, so the fixpoint is reached, and the number of dependent decisions is the longest chain of alternating
// decisions -- the depth of a cluster of proposals around one object, not the number of boxes.  The edges are the per-block hit lists
// the candidate kernels wrote (row -> column bits, row < column in score order).
// Here the fixpoint is PULLED: decisions are final and only depend on decided boxes of higher score, so every thread may simply re-read
// the states of its box's predecessors until it can decide -- no barrier, no round counter; the time is the depth of the longest chain
// times one L2 round trip.  The predecessors of a box are the transposed hit lists (nms_inlist_kernel: one list of at most NMS_IN_CAP
// entries per box; boxes at or below the score threshold never suppress anything and are left out).  An overflow of a hit list or of an
// in-list leaves `done` at 0 and the list walk runs; the result is the same keep mask either way.
constexpr int NMS_FIX_THREADS = 1024;
constexpr uint8_t NMS_UNDECIDED = 0, NMS_KEPT = 1, NMS_SUPPRESSED = 2;
constexpr uint32_t NMS_IN_CAP = 128;

__global__ void __launch_bounds__(256)
nms_inlist_kernel(int64_t n, int64_t nwords, const uint8_t *__restrict__ valid, const NmsLists lists, uint8_t *__restrict__ state, uint32_t *__restrict__ incnt,
                  uint32_t *__restrict__ inlist, uint32_t *__restrict__ ctl /* [4]: an in-list overflowed */)
{
    if (lists.blkcnt[nwords] != 0u) return;   // a hit list overflowed (grid-uniform): the dense walk decides
    const int64_t b = blockIdx.x;
    const unsigned tid = threadIdx.x;
    if (tid < 64u) { const int64_t j = b * 64 + tid; state[j] = (j < n && valid[j]) ? NMS_UNDECIDED : NMS_SUPPRESSED; }
    const uint32_t c = min(lists.blkcnt[b], NMS_LIST_CAP);
    const uint32_t *gw = lists.ent_w + b * NMS_LIST_CAP;
    const uint64_t *gb = lists.ent_bits + b * NMS_LIST_CAP;
    for (uint32_t e = tid; e < c; e += 256u) {
        const uint32_t we = gw[e];
        const int64_t i = b * 64 + (we >> 16);
        if (!valid[i]) continue;
        unsigned long long bits = gb[e];
        const int64_t col0 = (int64_t)(we & 0xffffu) * 64;
        while (bits) {
            const int t = __ffsll((long long)bits) - 1;
            bits &= bits - 1;
            const int64_t j = col0 + t;
            const uint32_t slot = atomicAdd(incnt + j, 1u);
            if (slot < NMS_IN_CAP) inlist[j * NMS_IN_CAP + slot] = (uint32_t)i;
            else ctl[4] = 1u;
        }
    }
}

__global__ void __launch_bounds__(NMS_FIX_THREADS, 1)
nms_pull_kernel(int64_t n, int64_t nwords, const uint32_t *__restrict__ order, uint8_t *__restrict__ suppressed, const NmsLists lists, uint8_t *state,
                const uint32_t *__restrict__ incnt, const uint32_t *__restrict__ inlist, uint32_t *ctl /* [2] done, [4] in-list overflow */)
{
    if (lists.blkcnt[nwords] != 0u || ctl[4] != 0u) return;   // (both written by earlier kernels: grid-uniform)
    const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, gsize = (int64_t)gridDim.x * blockDim.x;
    // a thread takes its boxes in ascending order, so whatever a box waits for is held by a thread that is running or done
    for (int64_t j = gtid; j < n; j += gsize) {
        uint32_t s = __ldcg(state + j);
        if (s == NMS_UNDECIDED) {
            const uint32_t c = incnt[j];
            const uint32_t *L = inlist + j * NMS_IN_CAP;
            bool done = false;
            while (!done) {
                bool kept = false, open = false;
                for (uint32_t k = 0; k < c; k++) {
                    const uint32_t si = __ldcg(state + __ldg(L + k));
                    kept |= si == NMS_KEPT;
                    open |= si == NMS_UNDECIDED;
                }
                if (kept || !open) {
                    s = kept ? NMS_SUPPRESSED : NMS_KEPT;
                    // published INSIDE the loop: lanes of this warp may be waiting for this box, and a lane parked behind the loop would
                    // never let them see it
                    asm volatile("st.global.cg.u8 [%0], %1;" ::"l"(state + j), "r"(s) : "memory");
                    done = true;
                }
            }
        }
        suppressed[order[j]] = s == NMS_KEPT ? 0 : 1;
    }
    if (gtid == 0) ctl[2] = 1u;
}

// ------------------------------------------------------------------------------------------------ soft-NMS
// LINEAR / GAUSSIAN suppression (reference d3d/box/nms.cpp:33-94; its CUDA version, nms_cuda.cu:108-153, needs a dense N x N
// coefficient matrix and indexes it with tile-local positions).  The rule is sequential in the boxes AND in the scores: after
// box i has decayed the scores of everything behind it, the reference re-sorts the positions between i and the last suppressed
// box with a stable insertion sort, so the next box is not known before the previous one is done.  One CTA walks that sequence:
//   * the decay of the boxes behind position _i runs over all threads (one IoU each per round);
//   * the re-sort is incremental: boxes whose score did not change since they were last sorted are still in order, so only the
//     changed ones (a handful) are merged back -- rank among the unchanged ones by binary search, rank among the changed ones by
//     counting -- which is the same permutation the insertion sort produces (both are THE stable sort by "not suppressed first,
//     then score descending"); suppressed boxes keep their relative order, which the mask does not depend on.
// Arrays are indexed by the box's position in the initial stable score order.
constexpr int SOFT_THREADS = 1024;
constexpr int SOFT_BCAP = 1024;   // changed boxes merged per step without falling back to counting all pairs

template <typename T> struct SoftState {
    T *sc;             // current scores
    uint32_t *ord;     // ord[q] = box at position q of the emulated order
    uint32_t *tmp;     // [n] unchanged boxes of the range, compacted
    uint8_t *sup;      // suppressed
    uint8_t *mk;       // score changed since the box was last sorted
};

// a before b in the order the reference's insertion sort produces
template <typename T>
__device__ __forceinline__ bool soft_before(const SoftState<T> &S, const uint32_t *pos, uint32_t a, uint32_t b)
{
    const bool sa = S.sup[a] != 0, sb = S.sup[b] != 0;
    if (sa != sb) return sb;
    if (!sa) { const T xa = S.sc[a], xb = S.sc[b]; if (xa != xb) return xa > xb; }
    return pos[a] < pos[b];
}

// re-sort of the range [_i + 1, Sp) after the decay of step _i (the reference's insertion sort, nms.cpp:74-94), by all NT threads of
// the CTA.  *s_cnt must be 0 on entry.  Boxes whose score changed are marked in S.mk; positions >= E count as changed.
template <typename T, uint32_t NT>
__device__ __forceinline__ void soft_resort(const SoftState<T> &S, uint32_t *pos, uint32_t _i, uint32_t Sp, uint32_t &E, uint32_t *s_red,
                                            uint32_t *s_cnt, uint32_t *s_dirty, uint32_t *Bp)
{
    const uint32_t tid = threadIdx.x;
    if (Sp <= _i + 2) return;   // zero or one box in the range: nothing to sort (uniform); marks stay for a later sort
    const uint32_t r0 = _i + 1, m = Sp - r0;   // range [r0, Sp)
    // split the range into unchanged boxes (still mutually sorted) and the rest
    const uint32_t per = (m + NT - 1) / NT, q0 = r0 + tid * per, q1 = min(q0 + per, Sp);
    uint32_t na = 0;
    for (uint32_t q = q0; q < q1; q++) { const uint32_t j = S.ord[q]; if (!(S.mk[j] || q >= E)) na++; }
    // exclusive prefix of na over the threads
    uint32_t inc = na;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, inc, d); if ((tid & 31u) >= (unsigned)d) inc += x; }
    if ((tid & 31u) == 31u) s_red[tid >> 5] = inc;
    __syncthreads();
    if (tid < 32) {
        uint32_t v = tid < NT / 32 ? s_red[tid] : 0u, iv = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, iv, d); if (tid >= (unsigned)d) iv += x; }
        if (tid < NT / 32) s_red[tid] = iv - v;
        if (tid == 31) *s_dirty = iv;   // unchanged boxes in the range
    }
    __syncthreads();
    uint32_t abase = s_red[tid >> 5] + inc - na;
    const uint32_t nA = *s_dirty, nB = m - nA;
    if (nB == 0) return;        // nothing changed inside the range: it is still sorted
    const bool brute = nB > (uint32_t)SOFT_BCAP;
    for (uint32_t q = q0; q < q1; q++) {
        const uint32_t j = S.ord[q];
        if (!(S.mk[j] || q >= E)) S.tmp[abase++] = j;
        else if (!brute) Bp[atomicAdd(s_cnt, 1u)] = j;
    }
    __syncthreads();
    if (!brute) {
        // unchanged box a at compact index ia: new position = r0 + ia + (changed boxes before it)
        for (uint32_t ia = tid; ia < nA; ia += NT) {
            const uint32_t a = S.tmp[ia];
            uint32_t c = 0;
            for (uint32_t k = 0; k < nB; k++) c += soft_before<T>(S, pos, Bp[k], a) ? 1u : 0u;
            S.ord[r0 + ia + c] = a;
        }
        // changed box b: unchanged boxes before it (binary search: they are sorted) + changed boxes before it
        for (uint32_t kb = tid; kb < nB; kb += NT) {
            const uint32_t b = Bp[kb];
            uint32_t lo = 0, hi = nA;
            while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (soft_before<T>(S, pos, S.tmp[mid], b)) lo = mid + 1; else hi = mid; }
            uint32_t c = lo;
            for (uint32_t k = 0; k < nB; k++) c += (k != kb && soft_before<T>(S, pos, Bp[k], b)) ? 1u : 0u;
            S.ord[r0 + c] = b;
        }
    } else {
        // many changed boxes: count all pairs (tmp receives a copy of the range first)
        __syncthreads();
        for (uint32_t q = r0 + tid; q < Sp; q += NT) S.tmp[q - r0] = S.ord[q];
        __syncthreads();
        for (uint32_t x = tid; x < m; x += NT) {
            const uint32_t a = S.tmp[x];
            uint32_t c = 0;
            for (uint32_t y = 0; y < m; y++) c += (y != x && soft_before<T>(S, pos, S.tmp[y], a)) ? 1u : 0u;
            S.ord[r0 + c] = a;
        }
    }
    __syncthreads();
    for (uint32_t q = r0 + tid; q < Sp; q += NT) { const uint32_t j = S.ord[q]; pos[j] = q; S.mk[j] = 0; }
    E = Sp;
    __syncthreads();
}

template <typename T, bool AABB>
__global__ void __launch_bounds__(SOFT_THREADS) nms_soft_kernel(const BoxRec<T> *__restrict__ recs, const AABBRec<T> *__restrict__ arecs, const T *__restrict__ scores,
                                                                const uint32_t *__restrict__ order, int64_t n64, T thr, T sthr, T param, int sup_type,
                                                                SoftState<T> S, uint32_t *__restrict__ pos, uint8_t *__restrict__ suppressed)
{
    const uint32_t n = (uint32_t)n64, tid = threadIdx.x, NT = SOFT_THREADS;
    __shared__ uint32_t s_red[32], s_cnt, s_S, s_dirty;
    __shared__ uint32_t Bp[SOFT_BCAP];
    for (uint32_t p = tid; p < n; p += NT) {
        const T v = scores[order[p]];
        S.sc[p] = v; S.ord[p] = p; pos[p] = p; S.mk[p] = 0;
        S.sup[p] = v > sthr ? 0 : 1;   // reference CUDA rule (nms_cuda.cu:223), as for hard NMS
    }
    __syncthreads();
    uint32_t E = n;   // positions (_i, E) that are not marked are mutually sorted
    for (uint32_t _i = 0; _i < n; _i++) {
        __syncthreads();       // the previous step's reads of the shared words are done
        const uint32_t i = S.ord[_i];
        if (S.sup[i]) break;   // nms.cpp:37-42: everything behind a suppressed box is suppressed
        if (tid == 0) { s_S = _i; s_cnt = 0; s_dirty = 0; }
        __syncthreads();
        // decay
        {
            BoxRec<T> A; AABBRec<T> AA;
            if (AABB) AA = arecs[i]; else A = recs[i];
            uint32_t smax = _i;
            for (uint32_t q = _i + 1 + tid; q < n; q += NT) {
                const uint32_t j = S.ord[q];
                const T iou = AABB ? aabb_iou<T>(AA, arecs[j]) : rbox_iou<T>(A, recs[j]);
                if (iou > thr) {
                    const T coef = sup_type == D3D_SUP_LINEAR ? T(1) - pow(iou, param) : exp(-iou * iou / param);
                    const T v = S.sc[j] * coef;
                    S.sc[j] = v; S.sup[j] = v < sthr ? 1 : 0; S.mk[j] = 1;
                }
                if (S.sup[j]) smax = q;
            }
            // S = last position behind _i that holds a suppressed box (nms.cpp:77-78)
#pragma unroll
            for (int d = 16; d; d >>= 1) smax = max(smax, __shfl_xor_sync(0xffffffffu, smax, d));
            if ((tid & 31u) == 0) atomicMax(&s_S, smax);
        }
        __syncthreads();
        soft_resort<T, SOFT_THREADS>(S, pos, _i, s_S, E, s_red, &s_cnt, &s_dirty, Bp);
    }
    __syncthreads();
    for (uint32_t p = tid; p < n; p += NT) suppressed[order[p]] = S.sup[p];
}

// ------------------------------------------------------------------------------------------------ batched hard NMS
// Frame-batched NMS (BASELINE.json config 5, SURVEY.md 8(e)): boxes of all frames packed back to back + device offsets, like the voxel
// ABI.  The single-frame pipeline above spends ~50 launches on one frame and resolves it on ONE SM; here three launches cover the
// batch and every stage has a frame dimension: (1) one CTA per frame sorts the frame's scores in shared memory (bitonic network on
// (key, index) pairs: the same stable order as the radix sort) and writes the sorted records, (2) dense 64x64 tiles of every frame's
// upper triangle (blockIdx.z = frame), (3) one resolve CTA per frame, so 64 frames occupy 64 SMs instead of 1.
constexpr int NMSB_MAX = 8192;        // boxes per frame the shared-memory sort takes
constexpr int NMSB_SORT_THREADS = 1024;

template <typename T, bool AABB>
__global__ void __launch_bounds__(NMSB_SORT_THREADS) nmsb_sort_kernel(const T *__restrict__ boxes, const T *__restrict__ scores, const int64_t *__restrict__ offs,
                                                                    int64_t stride, float score_thr, uint32_t *__restrict__ order, BoxRec<T> *__restrict__ recs,
                                                                    AABBRec<T> *__restrict__ arecs, T *__restrict__ raw, uint8_t *__restrict__ valid,
                                                                    uint32_t *__restrict__ fail, const uint32_t *__restrict__ run_if)
{
    extern __shared__ unsigned long long sk[];   // [npow] keys, then [npow] u32 indices
    if (run_if && !*run_if) return;   // the edge-list path produced the keep masks
    const int64_t f = blockIdx.x, b = offs[f];
    int64_t n64 = offs[f + 1] - b;
    if (n64 > stride) { if (threadIdx.x == 0) *fail = 1u; n64 = stride; }   // longer than max_frame_boxes: cut (documented hard bound)
    const uint32_t n = (uint32_t)n64;
    uint32_t npow = 64;
    while (npow < n) npow <<= 1;
    uint32_t *si = reinterpret_cast<uint32_t *>(sk + npow);
    for (uint32_t p = threadIdx.x; p < npow; p += NMSB_SORT_THREADS) {
        sk[p] = p < n ? desc_key(scores[b + p]) : ~0ull;
        si[p] = p < n ? p : 0xffffffffu;
    }
    __syncthreads();
    for (uint32_t k = 2; k <= npow; k <<= 1)
        for (uint32_t j = k >> 1; j > 0; j >>= 1) {
            for (uint32_t t = threadIdx.x; t < npow / 2; t += NMSB_SORT_THREADS) {
                const uint32_t lo = ((t & ~(j - 1)) << 1) | (t & (j - 1)), hi = lo + j;   // j is a power of two
                const bool up = (lo & k) == 0;
                const unsigned long long ka = sk[lo], kb = sk[hi];
                const uint32_t ia = si[lo], ib = si[hi];
                const bool gt = ka > kb || (ka == kb && ia > ib);
                if (gt == up) { sk[lo] = kb; sk[hi] = ka; si[lo] = ib; si[hi] = ia; }
            }
            __syncthreads();
        }
    const int64_t base = f * stride;
    for (int64_t p = threadIdx.x; p < stride; p += NMSB_SORT_THREADS) {
        if (p < n) {
            const uint32_t i = si[p];
            order[base + p] = i;
            const T *bx = boxes + 5 * (b + i);
            if (AABB) arecs[base + p] = make_aabb_rec<T>(bx[0], bx[1], bx[2], bx[3], bx[4]);
            else {
                recs[base + p] = make_box_rec<T>(bx[0], bx[1], bx[2], bx[3], bx[4]);
                if (raw) { for (int q = 0; q < 5; q++) raw[5 * (base + p) + q] = bx[q]; }
            }
            valid[base + p] = scores[b + i] > score_thr ? 1 : 0;
        } else {
            if (AABB) { AABBRec<T> a; a.minx = a.maxx = a.miny = a.maxy = T(NAN); arecs[base + p] = a; }
            else { BoxRec<T> r; r.cx = r.cy = r.c = r.s = r.hw = r.hh = r.area = T(0); r.rho = T(NAN); recs[base + p] = r; }
            valid[base + p] = 0;
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(NMS_THREADS)
nmsb_mask_rbox_kernel(const BoxRec<T> *__restrict__ recs, const T *__restrict__ raw, const int64_t *__restrict__ offs, int64_t stride, int64_t nwords, T thr,
                      uint64_t *__restrict__ mask, const uint32_t *__restrict__ run_if)
{
    if (run_if && !*run_if) return;   // the edge-list path produced the keep masks
    const int64_t f = blockIdx.z;
    const int64_t n = min(offs[f + 1] - offs[f], stride);
    if ((int64_t)blockIdx.x * NMS_TILE >= n) return;
    const NmsLists none = {nullptr, nullptr, nullptr};
    nms_mask_rbox_body<T>(recs + f * stride, raw ? raw + 5 * f * stride : nullptr, n, nwords, thr, mask + f * stride * nwords, none, blockIdx.x, blockIdx.y, gridDim.y);
}

template <typename T>
__global__ void __launch_bounds__(NMS_TILE)
nmsb_mask_aabb_kernel(const AABBRec<T> *__restrict__ recs, const int64_t *__restrict__ offs, int64_t stride, int64_t nwords, T thr, uint64_t *__restrict__ mask)
{
    const int64_t f = blockIdx.z;
    const int64_t n = min(offs[f + 1] - offs[f], stride);
    const NmsLists none = {nullptr, nullptr, nullptr};
    nms_mask_aabb_body<T>(recs + f * stride, n, nwords, thr, mask + f * stride * nwords, none, blockIdx.y, blockIdx.x);
}

// one CTA per frame: the dense walk over the frame's suppression matrix
__global__ void __launch_bounds__(RESOLVE_THREADS)
nmsb_resolve_kernel(const uint64_t *__restrict__ mask, const int64_t *__restrict__ offs, int64_t stride, int64_t nwords_max, const uint8_t *__restrict__ valid,
                    const uint32_t *__restrict__ order, uint8_t *__restrict__ suppressed, const uint32_t *__restrict__ run_if)
{
    extern __shared__ unsigned long long remv[];   // [nwords]
    __shared__ unsigned long long diag0[64];
    __shared__ unsigned long long keptbits;
    if (run_if && !*run_if) return;   // the edge-list path produced the keep masks
    const int64_t f = blockIdx.x, b = offs[f];
    const int64_t n = min(offs[f + 1] - b, stride);
    if (n == 0) return;
    const int64_t nwords = (n + 63) / 64;
    nms_removed_init(remv, n, nwords, valid + f * stride);
    nms_dense_walk(mask + f * stride * nwords_max, nwords_max, n, nwords, order + f * stride, suppressed + b, remv, diag0, &keptbits);
}

// ------------------------------------------------------------------ batched rotated NMS over an edge list (threshold >= 0)
// The dense path above tests every pair of a frame (64 frames x 4096 proposals: 545 M circle tests, 1.08 ms) because boxes that are
// neighbours in score order are anywhere in the scene.  Greedy NMS does not need the score order as a memory order, only as a relation:
// box a suppresses box b iff a is kept, overlaps b and comes first in (score descending, index ascending).  So a frame is sorted along
// a Morton curve through the box centres instead, 64 consecutive boxes cover a small patch of the scene, a tile of two blocks whose
// bounding rectangles do not meet is skipped without looking at its pairs, every surviving pair above the threshold becomes one
// directed edge (first box -> later box; circle test per tile, clips over the flat candidate list), and the keep mask is the fixpoint of
// the parallel resolve over that edge list (nmsb_fix_kernel) -- one CTA per frame, box states in shared memory.  An edge list that
// overflows its capacity (frames of near-identical boxes) raises a device flag and the dense kernels, launched behind it, redo the batch.
constexpr int NMSB_ECAP_PER_BOX = 32;   // edge capacity per frame = 32 x max_frame_boxes
constexpr int NMSB_HQ = 256;            // hits a warp of the clip kernel collects before it reserves room in the frame's edge list
constexpr int NMSB_CQ = 512;            // candidates a warp of the candidate kernel collects before it reserves room in the frame's list

__device__ __forceinline__ uint32_t morton_part(uint32_t x) { x &= 0x3ffu; x = (x | (x << 8)) & 0x00ff00ffu; x = (x | (x << 4)) & 0x0f0f0f0fu; x = (x | (x << 2)) & 0x33333333u; return (x | (x << 1)) & 0x55555555u; }

template <typename T>
__global__ void __launch_bounds__(NMSB_SORT_THREADS) nmsb_morton_kernel(const T *__restrict__ boxes, const T *__restrict__ scores, const int64_t *__restrict__ offs,
                                                                      int64_t stride, float score_thr, uint32_t *__restrict__ order, BoxRec<T> *__restrict__ recs,
                                                                      T *__restrict__ raw, uint8_t *__restrict__ valid, uint64_t *__restrict__ skey,
                                                                      float4 *__restrict__ bounds, uint32_t *__restrict__ fail)
{
    extern __shared__ unsigned long long sk[];   // [npow] keys, then [npow] u32 indices
    __shared__ float red[4][32];
    const int64_t f = blockIdx.x, b = offs[f];
    int64_t n64 = offs[f + 1] - b;
    if (n64 > stride) { if (threadIdx.x == 0) fail[0] = 1u; n64 = stride; }   // longer than max_frame_boxes: cut (documented hard bound)
    const uint32_t n = (uint32_t)n64;
    uint32_t npow = 64;
    while (npow < n) npow <<= 1;
    uint32_t *si = reinterpret_cast<uint32_t *>(sk + npow);
    // extent of the finite box centres
    float mnx = 3e38f, mxx = -3e38f, mny = 3e38f, mxy = -3e38f;
    for (uint32_t p = threadIdx.x; p < n; p += NMSB_SORT_THREADS) {
        const float x = (float)boxes[5 * (b + p)], y = (float)boxes[5 * (b + p) + 1];
        if (fabsf(x) < 1e30f && fabsf(y) < 1e30f) { mnx = fminf(mnx, x); mxx = fmaxf(mxx, x); mny = fminf(mny, y); mxy = fmaxf(mxy, y); }
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        mnx = fminf(mnx, __shfl_xor_sync(0xffffffffu, mnx, d)); mxx = fmaxf(mxx, __shfl_xor_sync(0xffffffffu, mxx, d));
        mny = fminf(mny, __shfl_xor_sync(0xffffffffu, mny, d)); mxy = fmaxf(mxy, __shfl_xor_sync(0xffffffffu, mxy, d));
    }
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = mnx; red[1][threadIdx.x >> 5] = mxx; red[2][threadIdx.x >> 5] = mny; red[3][threadIdx.x >> 5] = mxy; }
    __syncthreads();
    for (int w = 0; w < NMSB_SORT_THREADS / 32; w++) { mnx = fminf(mnx, red[0][w]); mxx = fmaxf(mxx, red[1][w]); mny = fminf(mny, red[2][w]); mxy = fmaxf(mxy, red[3][w]); }
    const float ivx = mxx > mnx ? 1023.f / (mxx - mnx) : 0.f, ivy = mxy > mny ? 1023.f / (mxy - mny) : 0.f;
    for (uint32_t p = threadIdx.x; p < npow; p += NMSB_SORT_THREADS) {
        unsigned long long key = ~0ull;
        if (p < n) {   // the order only decides which tiles can be skipped, never a result: any value is a valid key (NaN -> cell 0)
            const float x = (float)boxes[5 * (b + p)], y = (float)boxes[5 * (b + p) + 1];
            const uint32_t qx = (uint32_t)fminf(fmaxf((x - mnx) * ivx, 0.f), 1023.f), qy = (uint32_t)fminf(fmaxf((y - mny) * ivy, 0.f), 1023.f);
            key = morton_part(qx) | (morton_part(qy) << 1);
        }
        sk[p] = key;
        si[p] = p < n ? p : 0xffffffffu;
    }
    __syncthreads();
    if (npow >= 1024u && npow <= 4096u) {
        // 1024 < n <= 4096 (the C5 shape): 32-bit keys (cell << 12 | index: unique, so the network needs no tie rule), npow / 1024 per
        // thread, element e = r * 1024 + tid.  Steps between the elements of one thread run in registers, steps inside a warp as
        // shuffles, the others through shared memory (two buffers in turn: one barrier per step) -- 25 of the 78 steps of a
        // 4096-key network touch shared memory
        const uint32_t R = npow >> 10, tid = threadIdx.x;
        uint32_t *const buf0 = reinterpret_cast<uint32_t *>(sk), *const buf1 = buf0 + npow;
        uint32_t v[4];
#pragma unroll
        for (uint32_t r = 0; r < 4; r++) {
            const uint32_t e = r * 1024u + tid;
            v[r] = e < n ? (((uint32_t)sk[e] << 12) | e) : 0xffffffffu;
        }
        __syncthreads();   // the 64-bit keys have been read: their memory becomes the exchange buffers
        auto cx = [](uint32_t &a, uint32_t &c, const bool up) {
            const uint32_t lo = min(a, c), hi = max(a, c);
            a = up ? lo : hi; c = up ? hi : lo;
        };
        int pb = 0;
        for (uint32_t k = 2; k <= npow; k <<= 1)
            for (uint32_t j = k >> 1; j > 0; j >>= 1) {
                if (j >= 1024u) {   // partner in the same thread (k > j >= 1024: the direction bit of e is a bit of r or above)
                    if (j == 1024u) { cx(v[0], v[1], true); if (R > 2) cx(v[2], v[3], k != 2048u); }   // elements 2, 3 have bit 11 set: descending while k = 2048
                    else { cx(v[0], v[2], true); cx(v[1], v[3], true); }                               // j = 2048, k = 4096
                } else if (j < 32u) {
#pragma unroll
                    for (uint32_t r = 0; r < 4; r++)
                        if (r < R) {
                            const uint32_t e = r * 1024u + tid, o = __shfl_xor_sync(0xffffffffu, v[r], j);
                            const bool takemin = ((e & j) == 0) == ((e & k) == 0);
                            v[r] = takemin ? min(v[r], o) : max(v[r], o);
                        }
                } else {
                    uint32_t *bf = pb ? buf1 : buf0; pb ^= 1;
#pragma unroll
                    for (uint32_t r = 0; r < 4; r++) if (r < R) bf[r * 1024u + tid] = v[r];
                    __syncthreads();
#pragma unroll
                    for (uint32_t r = 0; r < 4; r++)
                        if (r < R) {
                            const uint32_t e = r * 1024u + tid, o = bf[e ^ j];
                            const bool takemin = ((e & j) == 0) == ((e & k) == 0);
                            v[r] = takemin ? min(v[r], o) : max(v[r], o);
                        }
                }
            }
#pragma unroll
        for (uint32_t r = 0; r < 4; r++) if (r < R) si[r * 1024u + tid] = v[r] & 0xfffu;   // (entries past n are never read)
        __syncthreads();
    } else {
        for (uint32_t k = 2; k <= npow; k <<= 1)
            for (uint32_t j = k >> 1; j > 0; j >>= 1) {
                for (uint32_t t = threadIdx.x; t < npow / 2; t += NMSB_SORT_THREADS) {
                    const uint32_t lo = ((t & ~(j - 1)) << 1) | (t & (j - 1)), hi = lo + j;   // j is a power of two
                    const bool up = (lo & k) == 0;
                    const unsigned long long ka = sk[lo], kb = sk[hi];
                    const uint32_t ia = si[lo], ib = si[hi];
                    const bool gt = ka > kb || (ka == kb && ia > ib);
                    if (gt == up) { sk[lo] = kb; sk[hi] = ka; si[lo] = ib; si[hi] = ia; }
                }
                __syncthreads();
            }
    }
    const int64_t base = f * stride;
    for (int64_t p = threadIdx.x; p < stride; p += NMSB_SORT_THREADS) {
        if (p < n) {
            const uint32_t i = si[p];
            order[base + p] = i;
            const T *bx = boxes + 5 * (b + i);
            recs[base + p] = make_box_rec<T>(bx[0], bx[1], bx[2], bx[3], bx[4]);
            if (raw) { for (int q = 0; q < 5; q++) raw[5 * (base + p) + q] = bx[q]; }
            valid[base + p] = scores[b + i] > score_thr ? 1 : 0;
            skey[base + p] = desc_key(scores[b + i]);
        } else {
            BoxRec<T> r; r.cx = r.cy = r.c = r.s = r.hw = r.hh = r.area = T(0); r.rho = T(NAN); recs[base + p] = r;
            valid[base + p] = 0;
            skey[base + p] = ~0ull;
        }
    }
    __syncthreads();   // this CTA's records are visible to its own threads
    // bounding rectangle of every 64-box block's circles, rounded outwards (a block without a finite box gets an empty rectangle)
    const int64_t nwords = stride / 64;
    for (int64_t blk = threadIdx.x >> 5; blk < nwords; blk += NMSB_SORT_THREADS / 32) {
        float lox = 3e38f, hix = -3e38f, loy = 3e38f, hiy = -3e38f;
        for (int t = threadIdx.x & 31; t < 64; t += 32) {
            const BoxRec<T> r = recs[base + blk * 64 + t];
            const double cx = (double)r.cx, cy = (double)r.cy, rho = (double)r.rho;
            if (fabs(cx) < 1e30 && fabs(cy) < 1e30 && rho < 1e30) {   // false for the NaN padding
                lox = fminf(lox, __double2float_rd(cx - rho)); hix = fmaxf(hix, __double2float_ru(cx + rho));
                loy = fminf(loy, __double2float_rd(cy - rho)); hiy = fmaxf(hiy, __double2float_ru(cy + rho));
            }
        }
#pragma unroll
        for (int d = 16; d; d >>= 1) {
            lox = fminf(lox, __shfl_xor_sync(0xffffffffu, lox, d)); hix = fmaxf(hix, __shfl_xor_sync(0xffffffffu, hix, d));
            loy = fminf(loy, __shfl_xor_sync(0xffffffffu, loy, d)); hiy = fmaxf(hiy, __shfl_xor_sync(0xffffffffu, hiy, d));
        }
        if ((threadIdx.x & 31) == 0) bounds[f * nwords + blk] = make_float4(lox, hix, loy, hiy);
    }
}

// one CTA per (row block, frame): the column blocks cb >= rb whose rectangle meets the row block's are tested pair by pair with the
// bounding-circle test; every surviving pair goes to the frame's candidate list as (first box | later box << 16), first = the one that
// comes first in (score descending, index ascending).  The clips run in a second kernel over the flat list: the candidates of a frame
// sit in a few diagonal tiles (the proposals around one object), and a kernel that clipped its own tiles would wait for those CTAs.
template <typename T>
__global__ void __launch_bounds__(NMS_THREADS)
nmsb_cand_kernel(const BoxRec<T> *__restrict__ recs_all, const uint64_t *__restrict__ skey_all, const uint32_t *__restrict__ order_all,
                 const float4 *__restrict__ bounds_all, const int64_t *__restrict__ offs, int64_t stride, int64_t nwords, uint32_t *__restrict__ cands_all,
                 uint32_t *__restrict__ ccount, uint32_t ccap, size_t cand_stride, uint32_t *__restrict__ fail, float tau /* thr / (1 + thr): area bound */)
{
    constexpr int RW = NMS_TILE / NMS_WARPS;  // 16 rows per warp
    constexpr int KC = NMS_TILE / 32;         // 2 column chunks
    const int64_t f = blockIdx.y, rb = blockIdx.x;
    const int64_t n = min(offs[f + 1] - offs[f], stride);
    if (rb * NMS_TILE >= n) return;
    const int64_t nb = (n + NMS_TILE - 1) / NMS_TILE;
    const BoxRec<T> *recs = recs_all + f * stride;
    const uint64_t *skey = skey_all + f * stride;
    const uint32_t *order = order_all + f * stride;
    const float4 *bounds = bounds_all + f * nwords;
    uint32_t *cands = cands_all + (size_t)f * cand_stride;
    // the circle test runs in single precision, widened by what the converted centres may be off by: it passes a superset of the pairs
    // whose circles meet, the clip decides
    __shared__ float ax_[NMS_TILE], ay_[NMS_TILE], ar_[NMS_TILE], aa_[NMS_TILE], ae_[NMS_TILE];   // + area, coordinate error
    __shared__ NmsShape as_[NMS_TILE];                                                              // axes and half extents (area bound)
    __shared__ unsigned long long kA[NMS_TILE], kB[NMS_TILE];
    __shared__ uint32_t oA[NMS_TILE], oB[NMS_TILE];
    __shared__ uint32_t queue[NMS_WARPS][NMSB_CQ];
    __shared__ uint16_t stage[NMS_WARPS][(NMS_TILE / NMS_WARPS) * NMS_TILE];   // a warp's circle-test survivors of the current tile
    __shared__ float bx_[NMS_TILE], by_[NMS_TILE], ba_[NMS_TILE], be_[NMS_TILE];
    __shared__ NmsShape bs_[NMS_TILE];
    const unsigned lane = lane_id(), w = threadIdx.x >> 5;
    uint16_t *sq = stage[w];
    if (threadIdx.x < NMS_TILE) {
        const BoxRec<T> a = recs[rb * NMS_TILE + threadIdx.x];
        const float fx = (float)a.cx, fy = (float)a.cy, fe = (fabsf(fx) + fabsf(fy)) * 2.4e-7f;   // 2^-22 of the coordinates
        ax_[threadIdx.x] = fx; ay_[threadIdx.x] = fy; ar_[threadIdx.x] = __double2float_ru((double)a.rho) + fe;
        NmsShape sh; sh.c = (float)a.c; sh.s = (float)a.s; sh.hw = (float)a.hw * 1.000001f; sh.hh = (float)a.hh * 1.000001f;
        as_[threadIdx.x] = sh; aa_[threadIdx.x] = (float)a.area; ae_[threadIdx.x] = fe;
        kA[threadIdx.x] = skey[rb * NMS_TILE + threadIdx.x]; oA[threadIdx.x] = order[rb * NMS_TILE + threadIdx.x];
    }
    // the column blocks whose rectangle meets this row block's, compacted in ascending order (one global round trip for all of them).
    // The order matters: the gridDim.z CTAs of a row block each build this list for themselves and take every gridDim.z-th entry of
    // it, so all of them must arrive at the SAME list (positions handed out by an atomic counter differ from CTA to CTA: tiles were
    // then clipped twice or never)
    __shared__ uint16_t cbs[NMSB_MAX / NMS_TILE];
    __shared__ uint32_t wbal[NMS_WARPS];
    uint32_t ncbs = 0;
    {
        const float4 mine = bounds[rb];
        for (int64_t cb0 = rb; cb0 < nb; cb0 += NMS_THREADS) {
            const int64_t cb = cb0 + threadIdx.x;
            bool meet = false;
            if (cb < nb) { const float4 other = bounds[cb]; meet = mine.x <= other.y && other.x <= mine.y && mine.z <= other.w && other.z <= mine.w; }
            const unsigned bal = __ballot_sync(0xffffffffu, meet);
            __syncthreads();   // the previous pass is done with wbal
            if (lane == 0) wbal[w] = bal;
            __syncthreads();
            uint32_t at = ncbs;
#pragma unroll
            for (int ww = 0; ww < NMS_WARPS; ww++) { const uint32_t c = (uint32_t)__popc(wbal[ww]); if (ww < (int)w) at += c; ncbs += c; }
            if (meet) cbs[at + __popc(bal & lanemask_lt())] = (uint16_t)cb;
        }
    }
    __syncthreads();
    const uint32_t ntiles = ncbs;
    uint32_t *q = queue[w];
    unsigned tail = 0;
    auto flush = [&](bool all) {   // a nearly full queue (at the end: the rest) leaves for the frame's list with ONE reservation: the warp waits for the atomic's round trip
        if (tail > (unsigned)NMSB_CQ - 32u || (all && tail != 0u)) {
            __syncwarp();
            uint32_t at = 0;
            if (lane == 0) at = atomicAdd(ccount + f, tail);
            at = __shfl_sync(0xffffffffu, at, 0);
            for (unsigned h = lane; h < tail; h += 32) {
                if (at + h < ccap) cands[at + h] = q[h];
                else fail[1] = 1u;
            }
            tail = 0;
            __syncwarp();
        }
    };
    for (uint32_t ti = blockIdx.z; ti < ntiles; ti += gridDim.z) {   // the row block's tiles are dealt to gridDim.z CTAs
        const int64_t cb = cbs[ti];
        __syncthreads();   // the previous tile's readers are done with the column arrays
        float bx[KC], by[KC], br[KC];
#pragma unroll
        for (int k = 0; k < KC; k++) {
            const BoxRec<T> bb = recs[cb * NMS_TILE + k * 32 + lane];
            bx[k] = (float)bb.cx; by[k] = (float)bb.cy;
            const float fe = (fabsf(bx[k]) + fabsf(by[k])) * 2.4e-7f;
            br[k] = __double2float_ru((double)bb.rho) + fe;
            if (w == 0) {   // the first warp also leaves the columns' numbers for the area bound in shared memory
                const unsigned cl = k * 32 + lane;
                NmsShape sh; sh.c = (float)bb.c; sh.s = (float)bb.s; sh.hw = (float)bb.hw * 1.000001f; sh.hh = (float)bb.hh * 1.000001f;
                bs_[cl] = sh; bx_[cl] = bx[k]; by_[cl] = by[k]; ba_[cl] = (float)bb.area; be_[cl] = fe;
            }
        }
        if (threadIdx.x < NMS_TILE) { kB[threadIdx.x] = skey[cb * NMS_TILE + threadIdx.x]; oB[threadIdx.x] = order[cb * NMS_TILE + threadIdx.x]; }
        __syncthreads();
        const bool diag = (rb == cb);
        // first the circle test of the warp's 16 x 64 pairs (the survivors wait as row << 8 | column), then the area bound and the
        // orientation of the survivors with all lanes busy
        unsigned ns = 0;
#pragma unroll 1
        for (int r = 0; r < RW; r++) {
            const unsigned rl = w * RW + r;
            const float ax = ax_[rl], ay = ay_[rl], ar = ar_[rl];
#pragma unroll
            for (int k = 0; k < KC; k++) {
                const unsigned cl = k * 32 + lane;
                const float dx = ax - bx[k], dy = ay - by[k], rs = ar + br[k];
                const bool cand = (dx * dx + dy * dy <= rs * rs * 1.00001f) && (!diag || cl > rl);   // every unordered pair once (NaN padding fails)
                const unsigned bal = __ballot_sync(0xffffffffu, cand);
                if (cand) sq[ns + __popc(bal & lanemask_lt())] = (uint16_t)((rl << 8) | cl);
                ns += __popc(bal);
            }
        }
        __syncwarp();
        for (unsigned e0 = 0; e0 < ns; e0 += 32) {
            const bool live = e0 + lane < ns;
            const unsigned ent = sq[live ? e0 + lane : ns - 1], rl = ent >> 8, cl = ent & 255u;
            const bool cand = live && nms_area_bound(ax_[rl] - bx_[cl], ay_[rl] - by_[cl], as_[rl], aa_[rl], bs_[cl], ba_[cl], 2.f * (ae_[rl] + be_[cl]), tau);
            const unsigned bal = __ballot_sync(0xffffffffu, cand);
            if (cand) {
                const bool a_first = kA[rl] < kB[cl] || (kA[rl] == kB[cl] && oA[rl] < oB[cl]);
                const uint32_t pa = (uint32_t)(rb * NMS_TILE + rl), pb = (uint32_t)(cb * NMS_TILE + cl);
                q[tail + __popc(bal & lanemask_lt())] = a_first ? (pa | (pb << 16)) : (pb | (pa << 16));
            }
            tail += __popc(bal);
            flush(false);
        }
    }
    flush(true);
}

// the clips of a frame's candidate list, 32 per warp step: candidate (first | later << 16) -> edge first -> later when iou(first, later) > threshold (nms.cpp:50)
template <typename T>
__global__ void __launch_bounds__(NMS_THREADS)
nmsb_clip_kernel(const BoxRec<T> *__restrict__ recs_all, const T *__restrict__ raw_all, int64_t stride, T thr, const uint32_t *__restrict__ cands_all,
                 const uint32_t *__restrict__ ccount, uint32_t ccap, size_t cand_stride, uint32_t *__restrict__ edges_all, uint32_t *__restrict__ ecount, uint32_t ecap,
                 uint32_t *__restrict__ fail)
{
    const int64_t f = blockIdx.y;
    const uint32_t nc = min(ccount[f], ccap);
    const BoxRec<T> *recs = recs_all + f * stride;
    const T *raw = raw_all ? raw_all + 5 * f * stride : nullptr;
    const uint32_t *cands = cands_all + (size_t)f * cand_stride;
    uint32_t *edges = edges_all + (size_t)f * ecap;
    const unsigned lane = lane_id(), w = threadIdx.x >> 5;
    __shared__ uint32_t hits[NMS_WARPS][NMSB_HQ];
    uint32_t *hb = hits[w];
    unsigned nh = 0;
    auto flush = [&]() {   // the warp's hits leave with one reservation in the frame's edge list
        __syncwarp();
        uint32_t at = 0;
        if (lane == 0) at = atomicAdd(ecount + f, nh);
        at = __shfl_sync(0xffffffffu, at, 0);
        for (unsigned h = lane; h < nh; h += 32) {
            if (at + h < ecap) edges[at + h] = hb[h];   // source | destination << 16
            else fail[1] = 1u;
        }
        nh = 0;
        __syncwarp();
    };
    for (uint32_t base = (blockIdx.x * NMS_WARPS + w) * 32u; base < nc; base += gridDim.x * NMS_WARPS * 32u) {
        const bool live = base + lane < nc;
        const uint32_t c = cands[live ? base + lane : nc - 1];
        const uint32_t pa = c & 0xffffu, pb = c >> 16;
        const BoxRec<T> A = recs[pa], B = recs[pb];
        const T v = rbox_iou<T>(A, B);
        const bool hit = live && over_threshold<T>(v, thr, raw, pa, pb);
        const unsigned bal = __ballot_sync(0xffffffffu, hit);
        if (bal) {
            if (nh + 32u > (unsigned)NMSB_HQ) flush();
            if (hit) hb[nh + __popc(bal & lanemask_lt())] = c;
            nh += __popc(bal);
        }
    }
    if (nh) flush();
}

// one CTA per frame: the keep mask as the fixpoint over the frame's edge list, everything in shared memory.
// Pushed form: the edges are gathered into one list of successors per box (count, prefix sum, fill: two passes over the edge list)
// and every box counts its predecessors.  A thread owns the boxes tid, tid + 1024, ...: a box whose predecessors have all reported
// "suppressed" is kept; a decided box reports to its successors once -- a kept box marks them suppressed, a suppressed box takes itself
// off their counts -- so the work is one visit per edge and the time is the depth of the longest chain of alternating decisions times a
// shared-memory round trip.  (Polling the predecessors instead, as nms_pull_kernel does with a thread per box, costs depth x in-degree
// here: 38 us per frame against 8.)  The boxes of a frame are in Morton order, not score order, so a thread never WAITS for one box
// (two threads could wait for each other's second box): it sweeps over its boxes and takes what can be decided.  Boxes at or below the
// score threshold never suppress anything and are left out of lists and counts.
// Frames whose edges do not fit the shared-memory lists reach the fixpoint in rounds over the edge list in global memory: in a round every
// undecided box whose earlier overlapping boxes are all suppressed becomes kept, and every box overlapped by a kept box becomes
// suppressed; two barriers per round, as many rounds as the longest chain of alternating decisions (D3D_B200_NMS_FIX=2 forces this form).
__global__ void __launch_bounds__(1024)
nmsb_fix_kernel(const uint32_t *__restrict__ edges_all, const uint32_t *__restrict__ ecount, uint32_t ecap, const int64_t *__restrict__ offs, int64_t stride,
                const uint8_t *__restrict__ valid_all, const uint32_t *__restrict__ order_all, uint8_t *__restrict__ suppressed, const uint32_t *__restrict__ fail,
                uint32_t lcap /* predecessor entries that fit the dynamic shared memory */)
{
    extern __shared__ __align__(16) unsigned char fx_dyn[];
    if (fail[1]) return;   // an edge list overflowed: the dense kernels behind this one redo the batch (CTA-uniform)
    const int64_t f = blockIdx.x, b = offs[f];
    const uint32_t n = (uint32_t)min(offs[f + 1] - b, stride);
    if (n == 0) return;
    const uint32_t npad = ((uint32_t)stride + 3u) & ~3u;
    // layout: off[npad + 4] u32 | cnt[npad] u32 (the rounds form keeps its u16 stamps there) | pend[npad] u32 | state[npad] u8 | lst[lcap] u16
    uint32_t *off = reinterpret_cast<uint32_t *>(fx_dyn), *cnt = off + npad + 4, *pend = cnt + npad;
    uint8_t *state = reinterpret_cast<uint8_t *>(pend + npad);
    uint16_t *lst = reinterpret_cast<uint16_t *>(state + npad);
    __shared__ uint32_t s_warp[32], s_total;
    const uint32_t ne = min(ecount[f], ecap);
    const uint32_t *edges = edges_all + (size_t)f * ecap;
    const uint8_t *valid = valid_all + f * stride;
    const uint32_t *order = order_all + f * stride;
    const unsigned tid = threadIdx.x, lane = tid & 31u, w = tid >> 5;
    for (uint32_t j = tid; j < n; j += 1024u) { state[j] = valid[j] ? NMS_UNDECIDED : NMS_SUPPRESSED; cnt[j] = 0; pend[j] = 0; }
    __syncthreads();
    // successors per box and predecessors still open per box
    const uint4 *edges4 = reinterpret_cast<const uint4 *>(edges);   // four edges per load: a frame's list starts on a 16-byte boundary
    const uint32_t ne4 = (ne + 3u) / 4u;
    for (uint32_t e = tid; e < ne4; e += 1024u) {
        const uint4 q = edges4[e];
        const uint32_t ed[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const uint32_t src = ed[u] & 0xffffu, dst = ed[u] >> 16;
            if (e * 4u + u < ne && state[src] != NMS_SUPPRESSED) { atomicAdd(&cnt[src], 1u); atomicAdd(&pend[dst], 1u); }
        }
    }
    __syncthreads();
    // exclusive prefix of cnt over the frame's boxes: a thread owns the boxes [tid * per, tid * per + per)
    const uint32_t per = (n + 1023u) / 1024u;
    uint32_t mine = 0;
    for (uint32_t k = 0; k < per; k++) { const uint32_t j = tid * per + k; if (j < n) mine += cnt[j]; }
    uint32_t inc = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= (unsigned)d) inc += x; }
    if (lane == 31u) s_warp[w] = inc;
    __syncthreads();
    if (w == 0) {
        uint32_t x = s_warp[lane], y = x;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t z = __shfl_up_sync(0xffffffffu, y, d); if (lane >= (unsigned)d) y += z; }
        s_warp[lane] = y - x;
        if (lane == 31u) s_total = y;
    }
    __syncthreads();
    uint32_t run = s_warp[w] + inc - mine;
    for (uint32_t k = 0; k < per; k++) { const uint32_t j = tid * per + k; if (j < n) { off[j] = run; run += cnt[j]; } }
    if (tid == 0) off[n] = s_total;
    __syncthreads();
    if (s_total <= lcap) {
        for (uint32_t e = tid; e < ne4; e += 1024u) {
            const uint4 q = edges4[e];
            const uint32_t ed[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const uint32_t src = ed[u] & 0xffffu, dst = ed[u] >> 16;
                if (e * 4u + u < ne && state[src] != NMS_SUPPRESSED) lst[off[src] + atomicSub(&cnt[src], 1u) - 1u] = (uint16_t)dst;
            }
        }
        __syncthreads();
        volatile uint8_t *vstate = state;
        volatile uint32_t *vpend = pend;
        uint32_t todo = 0;   // bit u: box tid + 1024 u has not reported to its successors yet
        for (uint32_t j = tid, u = 0; j < n; j += 1024u, u++) if (state[j] == NMS_UNDECIDED) todo |= 1u << u;
        while (todo) {
            for (uint32_t m = todo; m; m &= m - 1u) {
                const uint32_t u = (uint32_t)__ffs((int)m) - 1u, j = tid + 1024u * u;
                uint8_t st = vstate[j];
                if (st == NMS_UNDECIDED && vpend[j] == 0u) { st = NMS_KEPT; vstate[j] = NMS_KEPT; }
                if (st != NMS_UNDECIDED) {   // (all of this inside the loop: lanes of this warp may be waiting for these reports)
                    for (uint32_t k = off[j], k1 = off[j + 1]; k < k1; k++) {
                        const uint32_t d = lst[k];
                        if (st == NMS_KEPT) vstate[d] = NMS_SUPPRESSED;   // d still counts this box: it cannot have been kept
                        else atomicSub(&pend[d], 1u);
                    }
                    todo &= ~(1u << u);
                }
            }
        }
        __syncthreads();
    } else {
        uint16_t *blocked = reinterpret_cast<uint16_t *>(cnt);
        __syncthreads();
        for (uint32_t j = tid; j < n; j += 1024u) blocked[j] = 0;
        __syncthreads();
        for (uint32_t round = 1;; round++) {
            const uint16_t stamp = (uint16_t)(1u + (round - 1u) % 65535u);   // never 0; a stamp is only compared within its own round
            if (stamp == 1u && round > 1u) { for (uint32_t j = tid; j < n; j += 1024u) blocked[j] = 0; __syncthreads(); }
            for (uint32_t e = tid; e < ne; e += 1024u) {
                const uint32_t ed = edges[e], src = ed & 0xffffu, dst = ed >> 16;
                const uint8_t ss = state[src];
                if (ss == NMS_KEPT) state[dst] = NMS_SUPPRESSED;
                else if (ss == NMS_UNDECIDED) blocked[dst] = stamp;   // a box that comes first and overlaps is still undecided
            }
            __syncthreads();
            int left = 0;
            for (uint32_t j = tid; j < n; j += 1024u) {
                if (state[j] == NMS_UNDECIDED) {
                    if (blocked[j] != stamp) state[j] = NMS_KEPT;
                    else left = 1;
                }
            }
            if (!__syncthreads_or(left)) break;
        }
    }
    for (uint32_t j = tid; j < n; j += 1024u) suppressed[b + order[j]] = state[j] == NMS_KEPT ? 0 : 1;
}

// ------------------------------------------------------------------------------------------------ batched soft-NMS
// LINEAR / GAUSSIAN suppression of a batch of frames: the walk of nms_soft_kernel, one CTA per frame, its whole state in shared memory.
// A kept box only decays boxes whose IoU with it exceeds the threshold; for a threshold >= 0 those are a few spatial neighbours, so the
// frame's candidate pairs are found once, before the walk (nmsbs_cand_kernel), and every step clips the kept box against its own
// candidates instead of against every box behind it.  The lists hold candidates, not IoU values: the re-sorts decide which box of a pair
// is visited first, and the clip iou(visited, later) is the one the reference evaluates.
constexpr int NMSBS_PAIRS_PER_BOX = 32;   // candidate pairs per frame = 32 x max_frame_boxes; more -> that frame decays over all boxes
constexpr int NMSBS_THREADS = 512;    // 1024 threads leave 64 registers: the fp64 clip spills

// one CTA per (64-box row block, frame): every pair p < q of sorted positions that may have IoU > threshold (threshold >= 0) goes to the
// frame's pair list as p | q << 16.  The tests only drop pairs whose IoU cannot exceed the threshold, whichever box comes first:
// rbox: bounding circles meet (single precision, widened by what the converted centres may be off by; a record that is not finite is a
// candidate of every box); box: the closed AABBs overlap (a NaN coordinate fails every comparison and keeps the pair).
// pcount[f] counts every pair found, also those past the capacity: pcount[f] > pcap flags the frame's list as incomplete.
template <typename T, bool AABB>
__global__ void __launch_bounds__(256) nmsbs_cand_kernel(const BoxRec<T> *__restrict__ recs_all, const AABBRec<T> *__restrict__ arecs_all,
                                                         const int64_t *__restrict__ offs, int64_t stride, uint32_t *__restrict__ pairs_all,
                                                         uint32_t *__restrict__ pcount, uint32_t pcap)
{
    const int64_t f = blockIdx.y, rb = blockIdx.x;
    const int64_t n = min(offs[f + 1] - offs[f], stride);
    if (rb * NMS_TILE >= n) return;
    const int64_t nb = (n + NMS_TILE - 1) / NMS_TILE;
    __shared__ float4 rowc[NMS_TILE], colc[NMS_TILE];         // rbox: centre, widened radius
    __shared__ AABBRec<T> rowa[NMS_TILE], cola[NMS_TILE];     // box
    __shared__ uint32_t hits[NMS_TILE * NMS_TILE];
    __shared__ uint32_t s_n, s_base;
    uint32_t *pairs = pairs_all + (size_t)f * pcap;
    const unsigned tid = threadIdx.x;
    auto stage = [&](int64_t blk, float4 *c, AABBRec<T> *a) {
        const int64_t p = blk * NMS_TILE + tid;
        if (AABB) a[tid] = arecs_all[f * stride + p];
        else {
            const BoxRec<T> r = recs_all[f * stride + p];
            const float fx = (float)r.cx, fy = (float)r.cy, fr = __double2float_ru((double)r.rho) + (fabsf(fx) + fabsf(fy)) * 2.4e-7f;
            c[tid] = isfinite(fx) && isfinite(fy) && isfinite(fr) ? make_float4(fx, fy, fr, 0.f) : make_float4(0.f, 0.f, INFINITY, 0.f);
        }
    };
    if (tid < NMS_TILE) stage(rb, rowc, rowa);
    for (int64_t cb = rb + blockIdx.z; cb < nb; cb += gridDim.z) {
        __syncthreads();   // the previous tile's readers are done with the columns and the hits
        if (tid < NMS_TILE) stage(cb, colc, cola);
        if (tid == 0) s_n = 0;
        __syncthreads();
        for (unsigned k = tid; k < NMS_TILE * NMS_TILE; k += 256) {
            const unsigned rl = k >> 6, cl = k & 63u;
            const int64_t p = rb * NMS_TILE + rl, q = cb * NMS_TILE + cl;
            if (p >= q || q >= n) continue;
            bool cand;
            if (AABB) {
                const AABBRec<T> &a = rowa[rl], &b = cola[cl];
                cand = !(a.maxx < b.minx || b.maxx < a.minx || a.maxy < b.miny || b.maxy < a.miny);
            } else {
                const float4 a = rowc[rl], b = colc[cl];
                const float dx = a.x - b.x, dy = a.y - b.y, rs = a.z + b.z;
                cand = !(dx * dx + dy * dy > rs * rs * 1.00001f);
            }
            if (cand) hits[atomicAdd(&s_n, 1u)] = (uint32_t)p | ((uint32_t)q << 16);
        }
        __syncthreads();
        const uint32_t nh = s_n;
        if (nh == 0) continue;   // (uniform)
        if (tid == 0) s_base = atomicAdd(pcount + f, nh);
        __syncthreads();
        const uint32_t base = s_base;
        for (uint32_t h = tid; h < nh; h += 256) if (base + h < pcap) pairs[base + h] = hits[h];
    }
}

// one CTA per frame: the walk of nms_soft_kernel over the frame's score order (nmsb_sort_kernel), state in dynamic shared memory.
// Prologue: the frame's pair list becomes a symmetric adjacency (CSR: nboff / nblst, sorted positions) when it is complete.
// Step _i (kept box i): the decay runs over i's candidates whose position is behind _i -- the pairs left out have IoU <= threshold and
// the reference's decay does not touch them.  The end S of the re-sort range (last position holding a suppressed box) is then a running
// value: suppressed boxes stay behind S (the re-sort of [_i + 1, S) keeps them in the range, positions >= S are not moved), so S only
// grows, by the positions of the boxes suppressed at this step.  A decay can lift a score back over the threshold (negative scores):
// then S is found again by a scan of all positions behind _i.  Frames without a complete list (negative threshold: every pair decays;
// an overflowed list) take the decay of nms_soft_kernel over every position behind _i.  The re-sort is nms_soft_kernel's.
template <typename T, bool AABB>
__global__ void __launch_bounds__(NMSBS_THREADS, 1)
nmsbs_walk_kernel(const BoxRec<T> *__restrict__ recs_all, const AABBRec<T> *__restrict__ arecs_all, const T *__restrict__ scores,
                  const int64_t *__restrict__ offs, int64_t stride, const uint32_t *__restrict__ order_all, const uint32_t *__restrict__ pairs_all,
                  const uint32_t *__restrict__ pcount, uint32_t pcap, uint32_t *__restrict__ nboff_all, uint16_t *__restrict__ nblst_all,
                  T thr, T sthr, T param, int sup_type, uint8_t *__restrict__ suppressed)
{
    extern __shared__ __align__(16) unsigned char sw_dyn[];   // sc T[stride] | ord, tmp, pos u32[stride] | sup, mk u8[stride]
    __shared__ uint32_t s_red[32], s_cnt, s_S, s_dirty, s_rev;
    __shared__ uint32_t Bp[SOFT_BCAP];
    constexpr uint32_t NT = NMSBS_THREADS;
    const int64_t f = blockIdx.x, b = offs[f];
    const uint32_t n = (uint32_t)min(offs[f + 1] - b, stride), tid = threadIdx.x, lane = tid & 31u;
    if (n == 0) return;
    SoftState<T> S;
    S.sc = reinterpret_cast<T *>(sw_dyn);
    S.ord = reinterpret_cast<uint32_t *>(S.sc + stride); S.tmp = S.ord + stride;
    uint32_t *pos = S.tmp + stride;
    S.sup = reinterpret_cast<uint8_t *>(pos + stride); S.mk = S.sup + stride;
    const uint32_t *order = order_all + f * stride;
    const BoxRec<T> *recs = recs_all ? recs_all + f * stride : nullptr;
    const AABBRec<T> *arecs = arecs_all ? arecs_all + f * stride : nullptr;
    const uint32_t np = pairs_all ? pcount[f] : 0u;
    const bool nbr = pairs_all && np <= pcap;   // (uniform)
    uint32_t *nboff = nboff_all + f * (stride + 1);
    uint16_t *nbl = nblst_all + (size_t)f * 2 * pcap;
    if (nbr) {
        const uint32_t *pairs = pairs_all + (size_t)f * pcap;
        uint32_t *cnt = reinterpret_cast<uint32_t *>(S.sc);   // degrees, then fill cursors (the scores take this memory afterwards)
        for (uint32_t p = tid; p < n; p += NT) cnt[p] = 0;
        __syncthreads();
        for (uint32_t e = tid; e < np; e += NT) { const uint32_t pq = pairs[e]; atomicAdd(&cnt[pq & 0xffffu], 1u); atomicAdd(&cnt[pq >> 16], 1u); }
        __syncthreads();
        // exclusive prefix of the degrees: a thread owns the boxes [tid * per, tid * per + per)
        const uint32_t per = (n + NT - 1) / NT;
        uint32_t mine = 0;
        for (uint32_t k = 0; k < per; k++) { const uint32_t j = tid * per + k; if (j < n) mine += cnt[j]; }
        uint32_t inc = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t x = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= (unsigned)d) inc += x; }
        if (lane == 31u) s_red[tid >> 5] = inc;
        __syncthreads();
        if (tid < 32) {
            const uint32_t x = tid < NT / 32 ? s_red[tid] : 0u;
            uint32_t y = x;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const uint32_t z = __shfl_up_sync(0xffffffffu, y, d); if (tid >= (unsigned)d) y += z; }
            if (tid < NT / 32) s_red[tid] = y - x;
        }
        __syncthreads();
        uint32_t run = s_red[tid >> 5] + inc - mine;
        for (uint32_t k = 0; k < per; k++) { const uint32_t j = tid * per + k; if (j < n) { nboff[j] = run; run += cnt[j]; } }
        if (tid == NT - 1) nboff[n] = run;   // the last thread's range ends at n (or it owns no box: run = the total)
        __syncthreads();
        for (uint32_t e = tid; e < np; e += NT) {
            const uint32_t pq = pairs[e], p = pq & 0xffffu, q = pq >> 16;
            nbl[nboff[p] + atomicSub(&cnt[p], 1u) - 1u] = (uint16_t)q;
            nbl[nboff[q] + atomicSub(&cnt[q], 1u) - 1u] = (uint16_t)p;
        }
        __syncthreads();
    }
    if (tid == 0) s_S = 0;
    __syncthreads();
    uint32_t smax = 0;
    for (uint32_t p = tid; p < n; p += NT) {
        const T v = scores[b + order[p]];
        S.sc[p] = v; S.ord[p] = p; pos[p] = p; S.mk[p] = 0;
        S.sup[p] = v > sthr ? 0 : 1;   // reference CUDA rule (nms_cuda.cu:223), as for hard NMS
        if (S.sup[p]) smax = p;
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) smax = max(smax, __shfl_xor_sync(0xffffffffu, smax, d));
    if (lane == 0) atomicMax(&s_S, smax);
    __syncthreads();
    uint32_t Srun = s_S;   // last position holding a suppressed box (0: none)
    uint32_t E = n;        // positions (_i, E) that are not marked are mutually sorted
    for (uint32_t _i = 0; _i < n; _i++) {
        __syncthreads();       // the previous step's reads of the shared words are done
        const uint32_t i = S.ord[_i];
        if (S.sup[i]) break;   // nms.cpp:37-42: everything behind a suppressed box is suppressed
        if (tid == 0) { s_S = _i; s_cnt = 0; s_dirty = 0; s_rev = 0; }
        __syncthreads();
        // decay: i's candidates behind _i, or every position behind _i
        {
            BoxRec<T> A; AABBRec<T> AA;
            if (AABB) AA = arecs[i]; else A = recs[i];
            const uint32_t k0 = nbr ? nboff[i] : _i + 1, k1 = nbr ? nboff[i + 1] : n;
            uint32_t sm = _i, rev = 0;
            for (uint32_t k = k0 + tid; k < k1; k += NT) {
                uint32_t j, q;
                if (nbr) { j = nbl[k]; q = pos[j]; if (q <= _i) continue; }
                else { q = k; j = S.ord[q]; }
                const T iou = AABB ? aabb_iou<T>(AA, arecs[j]) : rbox_iou<T>(A, recs[j]);
                if (iou > thr) {
                    const T coef = sup_type == D3D_SUP_LINEAR ? T(1) - pow(iou, param) : exp(-iou * iou / param);
                    const T v = S.sc[j] * coef;
                    const uint8_t was = S.sup[j];
                    S.sc[j] = v; S.sup[j] = v < sthr ? 1 : 0; S.mk[j] = 1;
                    if (was && !S.sup[j]) rev = 1;
                }
                if (S.sup[j]) sm = max(sm, q);
            }
#pragma unroll
            for (int d = 16; d; d >>= 1) { sm = max(sm, __shfl_xor_sync(0xffffffffu, sm, d)); rev |= __shfl_xor_sync(0xffffffffu, rev, d); }
            if (lane == 0) { atomicMax(&s_S, sm); if (rev) s_rev = 1; }
        }
        __syncthreads();
        uint32_t Sp = s_S;
        if (nbr) {
            if (s_rev) {   // a suppressed box came back: the last suppressed position is found again (uniform)
                uint32_t sm = _i;
                for (uint32_t q = _i + 1 + tid; q < n; q += NT) if (S.sup[S.ord[q]]) sm = q;
#pragma unroll
                for (int d = 16; d; d >>= 1) sm = max(sm, __shfl_xor_sync(0xffffffffu, sm, d));
                __syncthreads();   // every thread has read s_S
                if (tid == 0) s_S = _i;
                __syncthreads();
                if (lane == 0) atomicMax(&s_S, sm);
                __syncthreads();
                Sp = s_S;
            } else Sp = max(Sp, Srun);
            Srun = Sp;
        }
        soft_resort<T, NT>(S, pos, _i, Sp, E, s_red, &s_cnt, &s_dirty, Bp);
    }
    __syncthreads();
    for (uint32_t p = tid; p < n; p += NT) suppressed[b + order[p]] = S.sup[p];
}

template <typename T> static size_t nmsbs_ws_bytes(int64_t nframes, int64_t max_frame_boxes)
{
    if (nframes < 1) nframes = 1;
    if (max_frame_boxes < 1) max_frame_boxes = 1;
    const int64_t stride = cdiv(max_frame_boxes, NMS_TILE) * NMS_TILE;
    const size_t rec = sizeof(BoxRec<T>) > sizeof(AABBRec<T>) ? sizeof(BoxRec<T>) : sizeof(AABBRec<T>), pcap = (size_t)stride * NMSBS_PAIRS_PER_BOX;
    const size_t per = align_up((size_t)stride * 4) + align_up((size_t)stride * rec) + align_up((size_t)stride) +   // order, records, valid
                       align_up(pcap * 4) + align_up((size_t)(stride + 1) * 4) + align_up(pcap * 2 * 2);            // pairs, CSR offsets and lists
    return per * (size_t)nframes + align_up((size_t)nframes * 4) + align_up(64 * 4) + 4096;
}

template <typename T>
static int nmsbs_impl(const T *boxes, const T *scores, int64_t total, const int64_t *offs, int64_t nframes, int64_t max_frame_boxes, int iou_type, int sup_type,
                      float iou_thr, float score_thr, float sup_param, uint8_t *suppressed, void *ws, size_t ws_bytes, cudaStream_t st)
{
    if (total < 0 || nframes < 0) return D3D_ERR_INVALID_ARGUMENT;
    if (iou_type != D3D_IOU_BOX && iou_type != D3D_IOU_RBOX) return D3D_ERR_INVALID_ARGUMENT;
    if (sup_type != D3D_SUP_LINEAR && sup_type != D3D_SUP_GAUSSIAN) return D3D_ERR_INVALID_ARGUMENT;   // hard NMS: d3d_nms2d_batch_*
    if (nframes == 0 || total == 0) return D3D_OK;
    if (!boxes || !scores || !offs || !suppressed) return D3D_ERR_INVALID_ARGUMENT;
    if (max_frame_boxes <= 0 || max_frame_boxes > total) max_frame_boxes = total;
    if (max_frame_boxes > NMSB_MAX) return D3D_ERR_UNSUPPORTED;   // the walk state lives in shared memory: use d3d_nms2d_* per frame
    if (nframes > 65535) return D3D_ERR_INVALID_ARGUMENT;
    if (!ws || ws_bytes < nmsbs_ws_bytes<T>(nframes, max_frame_boxes)) return D3D_ERR_WORKSPACE;
    const int64_t stride = cdiv(max_frame_boxes, NMS_TILE) * NMS_TILE, nwords = stride / 64;
    const bool aabb = iou_type == D3D_IOU_BOX;
    const uint32_t pcap = (uint32_t)(stride * NMSBS_PAIRS_PER_BOX);
    Arena a(ws, ws_bytes);
    uint32_t *order = a.take<uint32_t>((size_t)nframes * stride);
    void *recs = a.take<char>((size_t)nframes * stride * (sizeof(BoxRec<T>) > sizeof(AABBRec<T>) ? sizeof(BoxRec<T>) : sizeof(AABBRec<T>)));
    uint8_t *valid = a.take<uint8_t>((size_t)nframes * stride);
    uint32_t *pairs = a.take<uint32_t>((size_t)nframes * pcap);
    uint32_t *nboff = a.take<uint32_t>((size_t)nframes * (stride + 1));
    uint16_t *nblst = a.take<uint16_t>((size_t)nframes * 2 * pcap);
    uint32_t *pcount = a.take<uint32_t>(nframes);
    uint32_t *fail = a.take<uint32_t>(64);   // [0] a frame was longer than max_frame_boxes (cut)
    if (!a.ok()) return D3D_ERR_WORKSPACE;
    uint32_t npow = 64;
    while (npow < (uint32_t)stride) npow <<= 1;
    const size_t sort_smem = (size_t)npow * 12;
    const T thr = (T)iou_thr;   // (T)(float), as d3d_nms2d_*
    BoxRec<T> *br = aabb ? nullptr : (BoxRec<T> *)recs;
    AABBRec<T> *ar = aabb ? (AABBRec<T> *)recs : nullptr;
    D3D_CUDA_TRY(cudaMemsetAsync(fail, 0, 256, st));
    if (aabb) {
        if (sort_smem > 40 * 1024) D3D_CUDA_TRY(cudaFuncSetAttribute(nmsb_sort_kernel<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sort_smem));
        nmsb_sort_kernel<T, true><<<(unsigned)nframes, NMSB_SORT_THREADS, sort_smem, st>>>(boxes, scores, offs, stride, score_thr, order, nullptr, ar, nullptr, valid, fail, nullptr);
    } else {
        if (sort_smem > 40 * 1024) D3D_CUDA_TRY(cudaFuncSetAttribute(nmsb_sort_kernel<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sort_smem));
        nmsb_sort_kernel<T, false><<<(unsigned)nframes, NMSB_SORT_THREADS, sort_smem, st>>>(boxes, scores, offs, stride, score_thr, order, br, nullptr, nullptr, valid, fail, nullptr);
    }
    D3D_LAUNCHED();
    // candidate pairs exist for a threshold >= 0 only (a negative one lets every pair decay: every frame walks over all positions)
    const bool lists = thr >= T(0);
    if (lists) {
        D3D_CUDA_TRY(cudaMemsetAsync(pcount, 0, (size_t)nframes * 4, st));
        if (aabb) nmsbs_cand_kernel<T, true><<<dim3((unsigned)nwords, (unsigned)nframes, 4), 256, 0, st>>>(nullptr, ar, offs, stride, pairs, pcount, pcap);
        else nmsbs_cand_kernel<T, false><<<dim3((unsigned)nwords, (unsigned)nframes, 4), 256, 0, st>>>(br, nullptr, offs, stride, pairs, pcount, pcap);
        D3D_LAUNCHED();
    }
    const size_t walk_smem = (size_t)stride * (sizeof(T) + 3 * 4 + 2);
    if (aabb) {
        D3D_CUDA_TRY(cudaFuncSetAttribute(nmsbs_walk_kernel<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)walk_smem));
        nmsbs_walk_kernel<T, true><<<(unsigned)nframes, NMSBS_THREADS, walk_smem, st>>>(nullptr, ar, scores, offs, stride, order, lists ? pairs : nullptr, pcount, pcap,
                                                                                       nboff, nblst, thr, (T)score_thr, (T)sup_param, sup_type, suppressed);
    } else {
        D3D_CUDA_TRY(cudaFuncSetAttribute(nmsbs_walk_kernel<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)walk_smem));
        nmsbs_walk_kernel<T, false><<<(unsigned)nframes, NMSBS_THREADS, walk_smem, st>>>(br, nullptr, scores, offs, stride, order, lists ? pairs : nullptr, pcount, pcap,
                                                                                        nboff, nblst, thr, (T)score_thr, (T)sup_param, sup_type, suppressed);
    }
    D3D_LAUNCHED();
    return D3D_OK;
}

template <typename T> static size_t nmsb_ws_bytes(int64_t nframes, int64_t max_frame_boxes)
{
    if (nframes < 1) nframes = 1;
    if (max_frame_boxes < 1) max_frame_boxes = 1;
    const int64_t stride = cdiv(max_frame_boxes, NMS_TILE) * NMS_TILE, nwords = stride / 64;
    const size_t rec = sizeof(BoxRec<T>) > sizeof(AABBRec<T>) ? sizeof(BoxRec<T>) : sizeof(AABBRec<T>);
    const size_t per = align_up((size_t)stride * 4) + align_up((size_t)stride * rec) + align_up((size_t)stride * 5 * sizeof(T)) + align_up((size_t)stride) +
                       align_up((size_t)stride * nwords * 8) +
                       align_up((size_t)stride * 8) + align_up((size_t)nwords * 16) + align_up((size_t)stride * NMSB_ECAP_PER_BOX * 4);   // edge-list path: score keys, block rectangles, edges
    return per * (size_t)nframes + align_up((size_t)nframes * 8) + 4096;
}

template <typename T>
static int nmsb_impl(const T *boxes, const T *scores, int64_t total, const int64_t *offs, int64_t nframes, int64_t max_frame_boxes, int iou_type, int sup_type,
                     float iou_thr, float score_thr, uint8_t *suppressed, void *ws, size_t ws_bytes, cudaStream_t st)
{
    if (total < 0 || nframes < 0) return D3D_ERR_INVALID_ARGUMENT;
    if (iou_type != D3D_IOU_BOX && iou_type != D3D_IOU_RBOX) return D3D_ERR_INVALID_ARGUMENT;
    if (sup_type < D3D_SUP_HARD || sup_type > D3D_SUP_GAUSSIAN) return D3D_ERR_INVALID_ARGUMENT;
    if (sup_type != D3D_SUP_HARD) return D3D_ERR_UNSUPPORTED;   // soft-NMS is sequential in the scores: one frame per call
    if (nframes == 0 || total == 0) return D3D_OK;
    if (!boxes || !scores || !offs || !suppressed) return D3D_ERR_INVALID_ARGUMENT;
    if (max_frame_boxes <= 0 || max_frame_boxes > total) max_frame_boxes = total;
    if (max_frame_boxes > NMSB_MAX) return D3D_ERR_UNSUPPORTED;   // the per-frame sort lives in shared memory: use d3d_nms2d_* per frame
    if (nframes > 65535) return D3D_ERR_INVALID_ARGUMENT;
    if (!ws || ws_bytes < nmsb_ws_bytes<T>(nframes, max_frame_boxes)) return D3D_ERR_WORKSPACE;
    const int64_t stride = cdiv(max_frame_boxes, NMS_TILE) * NMS_TILE, nwords = stride / 64;
    const bool aabb = iou_type == D3D_IOU_BOX, recheck = sizeof(T) == 4 && !aabb;
    Arena a(ws, ws_bytes);
    uint32_t *order = a.take<uint32_t>((size_t)nframes * stride);
    void *recs = a.take<char>((size_t)nframes * stride * (sizeof(BoxRec<T>) > sizeof(AABBRec<T>) ? sizeof(BoxRec<T>) : sizeof(AABBRec<T>)));
    T *raw = a.take<T>((size_t)nframes * stride * 5);
    uint8_t *valid = a.take<uint8_t>((size_t)nframes * stride);
    uint64_t *mask = a.take<uint64_t>((size_t)nframes * stride * nwords);
    uint32_t *fail = a.take<uint32_t>(64);   // [0] a frame was longer than max_frame_boxes (cut), [1] an edge list overflowed
    uint64_t *skey = a.take<uint64_t>((size_t)nframes * stride);
    float4 *bounds = a.take<float4>((size_t)nframes * nwords);
    const uint32_t ecap = (uint32_t)(stride * NMSB_ECAP_PER_BOX);
    uint32_t *edges = a.take<uint32_t>((size_t)nframes * ecap);
    uint32_t *ecount = a.take<uint32_t>(2 * nframes), *ccount = ecount + nframes;
    if (!a.ok()) return D3D_ERR_WORKSPACE;
    uint32_t npow = 64;
    while (npow < (uint32_t)stride) npow <<= 1;
    const size_t sort_smem = (size_t)npow * 12;
    const T thr = (T)iou_thr;
    D3D_CUDA_TRY(cudaMemsetAsync(fail, 0, 256, st));
    // rotated boxes, threshold >= 0 (pairs with disjoint bounding circles have IoU 0 and never exceed it): Morton order + edge list + fixpoint;
    // D3D_B200_NMS_BATCH_PATH=dense forces the score-ordered dense path
    const bool edge_path = !aabb && thr >= T(0) && tuning(D3D_TUNE_NMS_BATCH_PATH, 0) != 1;
    const uint32_t *run_if = nullptr;
    if (edge_path) {
        D3D_CUDA_TRY(cudaMemsetAsync(ecount, 0, (size_t)nframes * 8, st));
        if (sort_smem > 40 * 1024) D3D_CUDA_TRY(cudaFuncSetAttribute(nmsb_morton_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sort_smem));
        nmsb_morton_kernel<T><<<(unsigned)nframes, NMSB_SORT_THREADS, sort_smem, st>>>(boxes, scores, offs, stride, score_thr, order, (BoxRec<T> *)recs, recheck ? raw : nullptr, valid,
                                                                                     skey, bounds, fail);
        D3D_LAUNCHED();
        // the candidate lists live in the frames' dense-matrix slabs (only the fallback behind the flag uses them as matrices)
        const size_t cand_stride = (size_t)stride * nwords * 2;
        const uint32_t ccap = (uint32_t)(cand_stride < 0xffffffffull ? cand_stride : 0xffffffffull);
        nmsb_cand_kernel<T><<<dim3((unsigned)nwords, (unsigned)nframes, 4), NMS_THREADS, 0, st>>>((const BoxRec<T> *)recs, skey, order, bounds, offs, stride, nwords,
                                                                                           reinterpret_cast<uint32_t *>(mask), ccount, ccap, cand_stride, fail,
                                                                                           (float)thr / (1.f + (float)thr) * 0.999999f);
        D3D_LAUNCHED();
        nmsb_clip_kernel<T><<<dim3(32, (unsigned)nframes), NMS_THREADS, 0, st>>>((const BoxRec<T> *)recs, recheck ? raw : nullptr, stride, thr, reinterpret_cast<const uint32_t *>(mask),
                                                                              ccount, ccap, cand_stride, edges, ecount, ecap, fail);
        D3D_LAUNCHED();
        {
            // shared memory of the per-frame resolve: offsets, counters, states + as many predecessor entries as fit (D3D_B200_NMS_FIX=2: none, rounds only)
            const size_t spad = ((size_t)stride + 3) & ~(size_t)3, fixed = (spad + 4) * 4 + spad * 8 + spad;
            const size_t room = 200 * 1024 > fixed ? 200 * 1024 - fixed : 0;
            const uint32_t lcap = tuning(D3D_TUNE_NMS_FIX, -1) == 2 ? 0u : (uint32_t)(room / 2);
            const size_t fx_smem = fixed + (size_t)lcap * 2;
            if (fx_smem > 40 * 1024) D3D_CUDA_TRY(cudaFuncSetAttribute(nmsb_fix_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fx_smem));
            nmsb_fix_kernel<<<(unsigned)nframes, 1024, fx_smem, st>>>(edges, ecount, ecap, offs, stride, valid, order, suppressed, fail, lcap); D3D_LAUNCHED();
        }
        run_if = fail + 1;   // the dense kernels below leave at once unless an edge list overflowed
    }
    if (aabb) {
        if (sort_smem > 40 * 1024) D3D_CUDA_TRY(cudaFuncSetAttribute(nmsb_sort_kernel<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sort_smem));
        nmsb_sort_kernel<T, true><<<(unsigned)nframes, NMSB_SORT_THREADS, sort_smem, st>>>(boxes, scores, offs, stride, score_thr, order, nullptr, (AABBRec<T> *)recs, nullptr, valid, fail, run_if);
    } else {
        if (sort_smem > 40 * 1024) D3D_CUDA_TRY(cudaFuncSetAttribute(nmsb_sort_kernel<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sort_smem));
        nmsb_sort_kernel<T, false><<<(unsigned)nframes, NMSB_SORT_THREADS, sort_smem, st>>>(boxes, scores, offs, stride, score_thr, order, (BoxRec<T> *)recs, nullptr, recheck ? raw : nullptr, valid, fail, run_if);
    }
    D3D_LAUNCHED();
    if (aabb) nmsb_mask_aabb_kernel<T><<<dim3((unsigned)nwords, (unsigned)nwords, (unsigned)nframes), NMS_TILE, 0, st>>>((const AABBRec<T> *)recs, offs, stride, nwords, thr, mask);
    else nmsb_mask_rbox_kernel<T><<<dim3((unsigned)nwords, (unsigned)(edge_path ? 1 : (nwords < 8 ? nwords : 8)), (unsigned)nframes), NMS_THREADS, 0, st>>>((const BoxRec<T> *)recs, recheck ? raw : nullptr, offs, stride, nwords, thr, mask, run_if);
    D3D_LAUNCHED();
    nmsb_resolve_kernel<<<(unsigned)nframes, 256, (size_t)nwords * 8, st>>>(mask, offs, stride, nwords, valid, order, suppressed, run_if);
    D3D_LAUNCHED();
    return D3D_OK;
}

constexpr int64_t NMS_SPARSE_MAX_WORDS = 8192;   // block counters + staging must fit shared memory next to the bitmap

template <typename T> static size_t nms_ws_bytes(int64_t n)
{
    if (n <= 0) n = 1;
    int64_t npad = cdiv(n, NMS_TILE) * NMS_TILE, nwords = npad / 64;
    size_t recs = sizeof(BoxRec<T>) > sizeof(AABBRec<T>) ? sizeof(BoxRec<T>) : sizeof(AABBRec<T>);
    return align_up((size_t)n * 8) + align_up((size_t)n * 4) + radix_sort_workspace_bytes(n) + align_up((size_t)npad * recs) +
           align_up((size_t)npad * 5 * sizeof(T)) + align_up((size_t)npad) + align_up((size_t)npad * nwords * 8) +
           align_up((size_t)(nwords + 1) * 4) + align_up((size_t)nwords * NMS_LIST_CAP * 4) + align_up((size_t)nwords * NMS_LIST_CAP * 8) +
           align_up(sizeof(NmsGrid)) + align_up(sizeof(NmsExt)) + 2 * align_up((size_t)2 * (NMS_GRID_CELLS + 1) * 4) + align_up((size_t)npad * sizeof(NmsCand<T>)) + scan_workspace_bytes(NMS_GRID_CELLS + 1) + 4096 +
           align_up((size_t)npad * sizeof(T)) + 3 * align_up((size_t)npad * 4) + 2 * align_up((size_t)npad) +   // soft-NMS state
           align_up((size_t)npad) + align_up(64) +   // parallel resolve: state, control words
           align_up((size_t)npad * 4) + align_up((size_t)npad * NMS_IN_CAP * 4);    // parallel resolve: in-list counts and in-lists
}

template <typename T>
static int nms_impl(const T *boxes, const T *scores, int64_t n, int iou_type, int sup_type, float iou_thr, float score_thr, float sup_param, uint8_t *suppressed,
                    void *ws, size_t ws_bytes, cudaStream_t st)
{
    if (n < 0) return D3D_ERR_INVALID_ARGUMENT;
    if (iou_type != D3D_IOU_BOX && iou_type != D3D_IOU_RBOX) return D3D_ERR_INVALID_ARGUMENT;  // reference: "Unsupported iou type!"
    if (sup_type < D3D_SUP_HARD || sup_type > D3D_SUP_GAUSSIAN) return D3D_ERR_INVALID_ARGUMENT;
    if (n == 0) return D3D_OK;
    if (!boxes || !scores || !suppressed) return D3D_ERR_INVALID_ARGUMENT;
    if (n >= (1ll << 31)) return D3D_ERR_INVALID_ARGUMENT;
    if (!ws || ws_bytes < nms_ws_bytes<T>(n)) return D3D_ERR_WORKSPACE;
    const int64_t npad = cdiv(n, NMS_TILE) * NMS_TILE, nwords = npad / 64;
    if ((size_t)nwords * 8 > 200 * 1024) return D3D_ERR_INVALID_ARGUMENT;  // removal bitmap must fit shared memory (n <= 1.6M)
    Arena a(ws, ws_bytes);
    uint64_t *keys = a.take<uint64_t>(n);
    uint32_t *order = a.take<uint32_t>(n);
    size_t sort_bytes = radix_sort_workspace_bytes(n);
    void *sort_ws = a.take<char>(sort_bytes);
    const bool aabb = iou_type == D3D_IOU_BOX;
    void *recs = a.take<char>((size_t)npad * (sizeof(BoxRec<T>) > sizeof(AABBRec<T>) ? sizeof(BoxRec<T>) : sizeof(AABBRec<T>)));
    T *raw = a.take<T>((size_t)npad * 5);
    uint8_t *valid = a.take<uint8_t>(npad);
    uint64_t *mask = a.take<uint64_t>((size_t)npad * nwords);
    NmsLists lists = {nullptr, nullptr, nullptr};
    uint32_t *blkcnt = a.take<uint32_t>((size_t)nwords + 1);
    uint32_t *ent_w = a.take<uint32_t>((size_t)nwords * NMS_LIST_CAP);
    uint64_t *ent_bits = a.take<uint64_t>((size_t)nwords * NMS_LIST_CAP);
    NmsGrid *grid = a.take<NmsGrid>(1);
    NmsExt *ext = a.take<NmsExt>(1);
    uint32_t *cellcnt = a.take<uint32_t>((size_t)2 * (NMS_GRID_CELLS + 1));   // [0] counts (pass 0), [1] fill cursors (pass 1)
    uint32_t *cellptr = a.take<uint32_t>((size_t)2 * (NMS_GRID_CELLS + 1));
    NmsCand<T> *celllist = a.take<NmsCand<T>>((size_t)npad);
    void *cell_scan_ws = a.take<char>(scan_workspace_bytes(NMS_GRID_CELLS + 1));
    SoftState<T> soft;
    soft.sc = a.take<T>(npad); soft.ord = a.take<uint32_t>(npad); soft.tmp = a.take<uint32_t>(npad);
    uint32_t *soft_pos = a.take<uint32_t>(npad);
    soft.sup = a.take<uint8_t>(npad); soft.mk = a.take<uint8_t>(npad);
    uint8_t *fix_state = a.take<uint8_t>(npad);
    uint32_t *fix_ctl = a.take<uint32_t>(16);
    uint32_t *fix_incnt = a.take<uint32_t>(npad), *fix_inlist = a.take<uint32_t>((size_t)npad * NMS_IN_CAP);
    if (!a.ok()) return D3D_ERR_WORKSPACE;
    // tuning / test override: D3D_B200_NMS_PATH=dense (dense matrix, dense resolve) | tiles (dense tiles + list resolve); default: spatial
    const int path_knob = tuning(D3D_TUNE_NMS_PATH, 0);
    const bool force_dense = path_knob == 2, force_tiles = path_knob == 1;
    if (nwords <= NMS_SPARSE_MAX_WORDS && !force_dense) {
        lists.blkcnt = blkcnt; lists.ent_w = ent_w; lists.ent_bits = ent_bits;
        D3D_CUDA_TRY(cudaMemsetAsync(blkcnt, 0, (size_t)(nwords + 1) * 4, st));
    }

    nms_keys_kernel<T><<<(unsigned)cdiv(n, 256), 256, 0, st>>>(scores, n, keys, order); D3D_LAUNCHED();
    int rc = KeyBits<T>::bits == 64 ? radix_sort_pairs_u64_hi32(keys, order, n, sort_ws, sort_bytes, fix_ctl + 8, st)
                                    : radix_sort_pairs_u64(keys, order, n, KeyBits<T>::bits, sort_ws, sort_bytes, st);
    if (rc) return rc;
    const bool recheck = sizeof(T) == 4 && !aabb;
    if (aabb)
        nms_gather_kernel<T, true><<<(unsigned)cdiv(npad, 256), 256, 0, st>>>(boxes, scores, order, n, npad, score_thr, nullptr, (AABBRec<T> *)recs, nullptr, valid, nullptr);
    else {
        D3D_CUDA_TRY(cudaMemsetAsync(ext, 0xff, sizeof(NmsExt), st));
        nms_gather_kernel<T, false><<<(unsigned)cdiv(npad, 256), 256, 0, st>>>(boxes, scores, order, n, npad, score_thr, (BoxRec<T> *)recs, nullptr, recheck ? raw : nullptr, valid, ext);
    }
    D3D_LAUNCHED();
    const T thr = (T)iou_thr;   // (T)(float): SURVEY.md 8(c) T2
    const int stop = tuning(D3D_TUNE_NMS_STOP, 0);   // measurement only (bench.py phase times): 1 = stop after sort + gather, 2 = after the candidate phase
    if (stop == 1) return D3D_OK;
    if (sup_type != D3D_SUP_HARD) {   // sequential in boxes and scores: one CTA emulates the reference's order
        if (aabb) nms_soft_kernel<T, true><<<1, SOFT_THREADS, 0, st>>>(nullptr, (const AABBRec<T> *)recs, scores, order, n, thr, (T)score_thr, (T)sup_param, sup_type, soft, soft_pos, suppressed);
        else nms_soft_kernel<T, false><<<1, SOFT_THREADS, 0, st>>>((const BoxRec<T> *)recs, nullptr, scores, order, n, thr, (T)score_thr, (T)sup_param, sup_type, soft, soft_pos, suppressed);
        D3D_LAUNCHED();
        return D3D_OK;
    }
    if (nwords > 65535) return D3D_ERR_INVALID_ARGUMENT;
    // spatial candidate search: pairs with disjoint bounding circles have IoU 0, which never exceeds a threshold >= 0
    const bool spatial = !aabb && lists.blkcnt && thr >= T(0) && !force_tiles;
    if (spatial) {
        const BoxRec<T> *br = (const BoxRec<T> *)recs;
        const unsigned gb = (unsigned)cdiv(n, 256);
        int dev_c = 0, nsm_cells = 0;
        D3D_CUDA_TRY(cudaGetDevice(&dev_c));
        D3D_CUDA_TRY(cudaDeviceGetAttribute(&nsm_cells, cudaDevAttrMultiProcessorCount, dev_c));
        if (nsm_cells < 1) nsm_cells = 1;
        D3D_CUDA_TRY(cudaMemsetAsync(cellcnt, 0, (size_t)2 * (NMS_GRID_CELLS + 1) * 4, st));
        nms_grid_kernel<<<1, 32, 0, st>>>(ext, n, grid); D3D_LAUNCHED();
        nms_bin_kernel<T, 0><<<gb, 256, 0, st>>>(br, n, grid, cellcnt, nullptr, nullptr); D3D_LAUNCHED();
        if ((rc = exclusive_scan_u32(cellcnt, cellptr, NMS_GRID_CELLS + 1, nullptr, cell_scan_ws, st))) return rc;
        nms_bin_kernel<T, 1><<<gb, 256, 0, st>>>(br, n, grid, cellcnt + NMS_GRID_CELLS + 1, cellptr, celllist); D3D_LAUNCHED();
        D3D_CUDA_TRY(cudaFuncSetAttribute(nms_cells_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, NC_ROWS * NC_COLS * 2));   // static + dynamic > 48 KB
        // a CTA per grid cell (cells that do not exist or hold no box leave at once)
        nms_cells_kernel<T><<<(unsigned)(nsm_cells * D3D_NC_CTAS), NC_THREADS, NC_ROWS * NC_COLS * 2, st>>>(br, recheck ? raw : nullptr, n, nwords, thr, grid, cellptr, celllist, lists, &ext->pad);
        D3D_LAUNCHED();
    }
    dim3 tiles((unsigned)nwords, (unsigned)nwords);
    if (aabb) nms_mask_aabb_kernel<T><<<tiles, NMS_TILE, 0, st>>>((const AABBRec<T> *)recs, n, nwords, thr, mask, lists);
    // (behind the spatial path of a large frame its CTAs only read the grid's flag and leave: fewer of them, each striding over more row tiles)
    else nms_mask_rbox_kernel<T><<<dim3((unsigned)nwords, (unsigned)(spatial && nwords >= 128 ? 4 : (nwords < 24 ? nwords : 24))), NMS_THREADS, 0, st>>>((const BoxRec<T> *)recs, recheck ? raw : nullptr, n, nwords, thr, mask, lists, spatial ? grid : nullptr);
    D3D_LAUNCHED();
    if (stop == 2) return D3D_OK;
    size_t smem = (size_t)nwords * 8;
    uint32_t stage_cap = 0;
    if (lists.blkcnt) {   // bitmap + keep words + block counts, the rest of ~200 KB goes to the list stages
        const size_t fixed = (size_t)nwords * 20;
        size_t sc = (200 * 1024 - fixed) / ((size_t)RS_STAGES * 12);
        if (sc > NMS_LIST_CAP) sc = NMS_LIST_CAP;
        stage_cap = (uint32_t)(sc & ~(size_t)1);   // even: the 64-bit stage arrays stay 8-byte aligned
        smem = fixed + (size_t)RS_STAGES * stage_cap * 12;
    }
    if (smem > 40 * 1024) D3D_CUDA_TRY(cudaFuncSetAttribute(nms_resolve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int resolve_nt = lists.blkcnt ? 512 : RESOLVE_THREADS;   // list walk: 64 threads 1.9x slower, 256 +10 %, 512 = 1024
    // parallel resolve for frames where the block-by-block walk is long; it leaves fix_ctl[2] = 1 when it produced the mask
    const uint32_t *skip_if = nullptr;
    const int fix_knob = tuning(D3D_TUNE_NMS_FIX, -1);   // 0: never, >= 1: always (where lists exist); default: from 128 blocks (8192 boxes) on
    if (lists.blkcnt && (fix_knob >= 1 || (fix_knob < 0 && nwords >= 128))) {
        int dev = 0, nsm = 0, per_sm = 0;
        D3D_CUDA_TRY(cudaGetDevice(&dev));
        D3D_CUDA_TRY(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev));
        D3D_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, nms_pull_kernel, NMS_FIX_THREADS, 0));
        if (nsm > 0 && per_sm > 0) {
            D3D_CUDA_TRY(cudaMemsetAsync(fix_ctl, 0, 64, st));
            D3D_CUDA_TRY(cudaMemsetAsync(fix_incnt, 0, (size_t)npad * 4, st));
            nms_inlist_kernel<<<(unsigned)nwords, 256, 0, st>>>(n, nwords, valid, lists, fix_state, fix_incnt, fix_inlist, fix_ctl); D3D_LAUNCHED();
            // every CTA of the pull kernel must be running while others wait for its boxes: a cooperative launch (one CTA per SM) guarantees it
            int64_t n_ = n, nwords_ = nwords;
            const uint32_t *order_ = order, *incnt_ = fix_incnt, *inlist_ = fix_inlist; uint8_t *sup_ = suppressed;
            void *args[] = {&n_, &nwords_, &order_, &sup_, &lists, &fix_state, &incnt_, &inlist_, &fix_ctl};
            D3D_CUDA_TRY(cudaLaunchCooperativeKernel((const void *)nms_pull_kernel, dim3((unsigned)nsm), dim3(NMS_FIX_THREADS), args, 0, st)); D3D_LAUNCHED();
            skip_if = fix_ctl + 2;
        }
    }
    nms_resolve_kernel<<<1, resolve_nt, smem, st>>>(mask, n, nwords, valid, order, suppressed, lists, stage_cap, skip_if); D3D_LAUNCHED();
    return D3D_OK;
}

}  // namespace d3d

using namespace d3d;
extern "C" size_t d3d_nms2d_workspace_bytes(int64_t n, int dtype) { return dtype == D3D_F64 ? nms_ws_bytes<double>(n) : nms_ws_bytes<float>(n); }
extern "C" int d3d_nms2d_f32(const float *boxes, const float *scores, int64_t n, int iou_type, int sup_type, float iou_thr, float score_thr, float sup_param,
                             uint8_t *suppressed, void *ws, size_t wsb, void *stream)
{ return nms_impl<float>(boxes, scores, n, iou_type, sup_type, iou_thr, score_thr, sup_param, suppressed, ws, wsb, (cudaStream_t)stream); }
extern "C" int d3d_nms2d_f64(const double *boxes, const double *scores, int64_t n, int iou_type, int sup_type, float iou_thr, float score_thr, float sup_param,
                             uint8_t *suppressed, void *ws, size_t wsb, void *stream)
{ return nms_impl<double>(boxes, scores, n, iou_type, sup_type, iou_thr, score_thr, sup_param, suppressed, ws, wsb, (cudaStream_t)stream); }
extern "C" size_t d3d_nms2d_batch_soft_workspace_bytes(int64_t total, int64_t nframes, int64_t max_frame_boxes, int dtype)
{
    if (max_frame_boxes <= 0 || max_frame_boxes > total) max_frame_boxes = total;
    return dtype == D3D_F64 ? nmsbs_ws_bytes<double>(nframes, max_frame_boxes) : nmsbs_ws_bytes<float>(nframes, max_frame_boxes);
}
extern "C" int d3d_nms2d_batch_soft_f32(const float *boxes, const float *scores, int64_t total, const int64_t *frame_offsets, int64_t nframes,
                                        int64_t max_frame_boxes, int iou_type, int sup_type, float iou_thr, float score_thr, float sup_param,
                                        uint8_t *suppressed, void *ws, size_t wsb, void *stream)
{ return nmsbs_impl<float>(boxes, scores, total, frame_offsets, nframes, max_frame_boxes, iou_type, sup_type, iou_thr, score_thr, sup_param, suppressed, ws, wsb, (cudaStream_t)stream); }
extern "C" int d3d_nms2d_batch_soft_f64(const double *boxes, const double *scores, int64_t total, const int64_t *frame_offsets, int64_t nframes,
                                        int64_t max_frame_boxes, int iou_type, int sup_type, float iou_thr, float score_thr, float sup_param,
                                        uint8_t *suppressed, void *ws, size_t wsb, void *stream)
{ return nmsbs_impl<double>(boxes, scores, total, frame_offsets, nframes, max_frame_boxes, iou_type, sup_type, iou_thr, score_thr, sup_param, suppressed, ws, wsb, (cudaStream_t)stream); }
extern "C" size_t d3d_nms2d_batch_workspace_bytes(int64_t total, int64_t nframes, int64_t max_frame_boxes, int dtype)
{
    if (max_frame_boxes <= 0 || max_frame_boxes > total) max_frame_boxes = total;
    return dtype == D3D_F64 ? nmsb_ws_bytes<double>(nframes, max_frame_boxes) : nmsb_ws_bytes<float>(nframes, max_frame_boxes);
}
extern "C" int d3d_nms2d_batch_f32(const float *boxes, const float *scores, int64_t total, const int64_t *frame_offsets, int64_t nframes, int64_t max_frame_boxes,
                                   int iou_type, int sup_type, float iou_thr, float score_thr, uint8_t *suppressed, void *ws, size_t wsb, void *stream)
{ return nmsb_impl<float>(boxes, scores, total, frame_offsets, nframes, max_frame_boxes, iou_type, sup_type, iou_thr, score_thr, suppressed, ws, wsb, (cudaStream_t)stream); }
extern "C" int d3d_nms2d_batch_f64(const double *boxes, const double *scores, int64_t total, const int64_t *frame_offsets, int64_t nframes, int64_t max_frame_boxes,
                                   int iou_type, int sup_type, float iou_thr, float score_thr, uint8_t *suppressed, void *ws, size_t wsb, void *stream)
{ return nmsb_impl<double>(boxes, scores, total, frame_offsets, nframes, max_frame_boxes, iou_type, sup_type, iou_thr, score_thr, suppressed, ws, wsb, (cudaStream_t)stream); }
