// iou.cu -- pairwise N x M IoU of rotated boxes (method "rbox") and of their AABBs (method "box").
//
// Replaces reference iou2dr_forward[_cuda] / iou2d_forward[_cuda] (d3d/box/iou.cpp:11-141,
// d3d/box/iou_cuda.cu:9-151).  Design (B200, sm_100a):
//   * a prep kernel turns every box into a 32-byte record once (1 sincos per box instead of 4 per pair);
//   * one CTA owns a TR x TC tile of the output.  The records of its TR rows and TC columns are staged
//     in shared memory; the output tile itself lives in shared memory and is streamed to HBM with
//     full-line 16-byte stores (the reference stores 4-byte values column-major, iou_cuda.cu:110-111);
//   * candidate compaction: each warp scans its 8 rows x TC columns with a 7-instruction
//     bounding-circle test, pushes the survivors into a per-warp shared-memory queue
//     (ballot + popc), and whenever 32 survivors are queued runs the ~150-instruction branch-free clip
//     (geom.cuh) on a FULL warp.  Divergence is gone: with 1/3 of the pairs being candidates a naive
//     thread-per-pair kernel would run the clip at ~1/3 lane utilisation;
//   * 64-bit indexing throughout: 100k x 100k (1e10 pairs) does not fit the reference's int pair index
//     (iou_cuda.cu:16,137).
// Roofline: FP32/FP64 CUDA-core issue rate (not a contraction -> no tensor cores); HBM store-bound
// when fewer than ~1 pair in 6 is a candidate.
#include "geom.cuh"

namespace d3d {

// ------------------------------------------------------------------ prep
// TILE == 0: one 8-field record per box (rows of the IoU kernel, NMS, the candidate counter).
// TILE > 0: field-major inside blocks of TILE boxes -- block t holds cx[TILE], cy[TILE], c, s, hw, hh, rho, area -- so that
// a column tile is staged with one contiguous copy and a warp's shared-memory reads of one field of 32 different
// columns of a 32-column chunk hit 32 different banks.
// Box i of n; i >= n writes padding.
template <typename T, int TILE>
__device__ __forceinline__ void box_prep_one(const T *__restrict__ boxes, int64_t n, int64_t i, BoxRec<T> *__restrict__ recs)
{
    BoxRec<T> r;
    if (i < n) {
        const T *b = boxes + 5 * i;
        r = make_box_rec<T>(b[0], b[1], b[2], b[3], b[4]);
    } else {
        r.cx = r.cy = r.c = r.s = r.hw = r.hh = r.area = T(0);
        r.rho = T(NAN);  // padding: fails every candidate test
    }
    if (TILE == 0) {
        recs[i] = r;
    } else {
        T *f = reinterpret_cast<T *>(recs + (i / TILE) * TILE) + (i % TILE);
        f[0 * TILE] = r.cx; f[1 * TILE] = r.cy; f[2 * TILE] = r.c; f[3 * TILE] = r.s;
        f[4 * TILE] = r.hw; f[5 * TILE] = r.hh; f[6 * TILE] = r.rho; f[7 * TILE] = r.area;
    }
}

template <typename T, int TILE>
__global__ void __launch_bounds__(256) box_prep_kernel(const T *__restrict__ boxes, int64_t n, int64_t npad, BoxRec<T> *__restrict__ recs)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npad) return;
    box_prep_one<T, TILE>(boxes, n, i, recs);
}

template <typename T>
__global__ void __launch_bounds__(256) aabb_prep_kernel(const T *__restrict__ boxes, int64_t n, AABBRec<T> *__restrict__ recs)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const T *b = boxes + 5 * i;
    recs[i] = make_aabb_rec<T>(b[0], b[1], b[2], b[3], b[4]);
}

// ------------------------------------------------------------------ rotated IoU tile kernel
// box2d_iou_batch (d3d_b200/box/__init__.py, _IOU_TILE) repeats these shapes: it sends "rbox" frames of more than 65535 tiles on an axis
// to the single-matrix kernel instead of the batch, so a change here must be made there too
template <typename T> struct IouTile;
template <> struct IouTile<float>  { static constexpr int TR = 64, TC = 128; };
template <> struct IouTile<double> { static constexpr int TR = 64, TC = 64; };

constexpr int IOU_THREADS = 256;
constexpr int IOU_WARPS = IOU_THREADS / 32;

// shared-memory image of one CTA (dynamic: more than the 48 KB static limit for fp32)
template <typename T> struct IouSmem {
    static constexpr int TR = IouTile<T>::TR, TC = IouTile<T>::TC;
    static constexpr int RW = TR / IOU_WARPS;          // rows per warp
    static constexpr int KC = TC / 32;                 // columns per lane
    static constexpr int DEPTH = RW * KC;              // pairs one lane tests per tile (<= 32: one bit each)
    BoxRec<T> sA[TR];                                   // row records
    T sB[8][TC];                                        // column records, field-major: cx, cy, c, s, hw, hh, rho, area
    T tile[TR][TC];
    uint16_t queue[IOU_WARPS][DEPTH * 32 + 32];        // the warp's candidates packed back to back (row_local * TC + col)
};

// z extent of a 3-D box (zmin, zmax), for the detection-evaluation distance matrix
struct ZRange { float lo, hi; };

// z overlap ratio of two boxes with the reference's float arithmetic (d3d/dgal_wrap.h:55-66): i / max(u, 1e-6)
__device__ __forceinline__ float z_iou(const ZRange &a, const ZRange &b)
{
    const float i = fmaxf(__fsub_rn(fminf(a.hi, b.hi), fmaxf(a.lo, b.lo)), 0.f);
    const float u = fmaxf(__fsub_rn(fmaxf(a.hi, b.hi), fminf(a.lo, b.lo)), 1e-6f);
    return __fdiv_rn(i, u);
}

// ZD: the stored value is the matcher's distance 1 - iou2d * ziou (d3d/tracking/matcher.pyx:55-76) instead of iou2d.
// The z factor is applied to the clipped candidates only (the tile is pre-filled with 1 = the distance of a rejected
// pair), so the detection-evaluation matrix costs little more than the IoU matrix.
// One CTA computes the TR x TC tile at (row0, col0) of the n x m matrix `out` (leading dimension ld); row0 < n and col0 < m.
// recA / zA hold n rows padded to a multiple of TR, recB / zB m columns padded to a multiple of TC (field-major in blocks of TC).
// The single-matrix kernel, the frame-batched kernel and the max-IoU reduction all run iou2dr_tile_fill, so a pair gets the same reject
// test and clip in all of them.  It leaves the tile's values in sm.tile: a warp's own rows are complete after __syncwarp (fp32) or
// __syncthreads (fp64); the whole tile after a __syncthreads.  Every value is +0 (rejected pairs, padding rows and columns), positive
// or NaN (rbox_iou: ai >= +0 and au > 0, so never negative and never -0).
template <typename T, bool ZD>
__device__ __forceinline__ void iou2dr_tile_fill(const BoxRec<T> *__restrict__ recA, const BoxRec<T> *__restrict__ recB, const ZRange *__restrict__ zA,
                                                 const ZRange *__restrict__ zB, const int64_t row0, const int64_t col0)
{
    using S = IouSmem<T>;
    constexpr int TR = S::TR, TC = S::TC, RW = S::RW, KC = S::KC;
    constexpr int V = 16 / sizeof(T);    // elements per 16-byte vector
    extern __shared__ __align__(16) unsigned char iou_smem_raw[];
    S &sm = *reinterpret_cast<S *>(iou_smem_raw);
    const unsigned lane = lane_id(), w = threadIdx.x >> 5;

    {   // stage records (arrays are padded to tile multiples, so no bounds checks)
        const float4 *ga = reinterpret_cast<const float4 *>(recA + row0);
        const float4 *gb = reinterpret_cast<const float4 *>(recB + col0);
        float4 *da = reinterpret_cast<float4 *>(sm.sA), *db = reinterpret_cast<float4 *>(&sm.sB[0][0]);
        constexpr int NA = TR * sizeof(BoxRec<T>) / 16, NB = TC * sizeof(BoxRec<T>) / 16;
        for (int i = threadIdx.x; i < NA; i += IOU_THREADS) da[i] = __ldg(ga + i);
        for (int i = threadIdx.x; i < NB; i += IOU_THREADS) db[i] = __ldg(gb + i);
    }
    // zero this warp's rows of the output tile (rejected pairs are exactly +0; distance matrix: 1 - 0 * ziou = 1)
    {
        float4 *z = reinterpret_cast<float4 *>(&sm.tile[w * RW][0]);
        const float fill = ZD ? 1.f : 0.f;
#pragma unroll
        for (int i = 0; i < RW * TC / (32 * V); i++) z[i * 32 + lane] = make_float4(fill, fill, fill, fill);
    }
    __shared__ ZRange szA[ZD ? TR : 1], szB[ZD ? TC : 1];   // z extents of the tile's rows / columns (distance matrix only)
    if (ZD) {
        for (int i = threadIdx.x; i < TR + TC; i += IOU_THREADS) {
            if (i < TR) szA[i] = zA[row0 + i]; else szB[i - TR] = zB[col0 + i - TR];
        }
    }
    __syncthreads();

    // ---- scan: reject test of this warp's RW x TC pairs: 8 flops, two compares, a ballot and a select per pair (no popc, no
    // shared-memory traffic on the per-pair path).  A pair survives when the centre of box B, seen in box A's frame, lies inside A's
    // rectangle grown by B's bounding radius (the separating-axis test on A's two axes with B replaced by its bounding circle):
    // 28.6 % of the pairs of the C1 distribution against 32.8 % for the bounding-circle test it replaces (21 % truly overlap), and
    // what it rejects has an empty intersection, stored as exactly +0.  The thresholds carry a relative slack of 2^-16 so that
    // rounding in the frame change never rejects a pair whose IoU would exceed the tolerance.
    // The flops run on pairs of column chunks (FADD2 / FMUL2 / FFMA2 on sm_100a: two pairs per issue slot).
    using PV = typename Vec2<T>::type;
    static_assert(KC % 2 == 0, "column chunks are tested two at a time");
    PV bx2[KC / 2], by2[KC / 2], br2[KC / 2];
    const T slack = T(1) + T(1.52587890625e-5);
#pragma unroll
    for (int k = 0; k < KC / 2; k++) {
        bx2[k] = P2<T>::mk(sm.sB[0][(2 * k) * 32 + lane], sm.sB[0][(2 * k + 1) * 32 + lane]);
        by2[k] = P2<T>::mk(sm.sB[1][(2 * k) * 32 + lane], sm.sB[1][(2 * k + 1) * 32 + lane]);
        br2[k] = P2<T>::mk(sm.sB[6][(2 * k) * 32 + lane] * slack, sm.sB[6][(2 * k + 1) * 32 + lane] * slack);   // NaN for padding
    }
    static_assert(RW * KC <= 32, "one lane per tested (row, column chunk)");
    unsigned mybal = 0;     // lane r*KC+k keeps the ballot of (row r, columns k*32 .. k*32+31)
#pragma unroll
    for (int r = 0; r < RW; r++) {
        const BoxRec<T> &a = sm.sA[w * RW + r];
        const T grow = (a.hw + a.hh) * T(1.52587890625e-5) + (a.rho - a.rho);   // NaN for a padding row: every test fails
        const PV ax2 = P2<T>::mk(a.cx, a.cx), ay2 = P2<T>::mk(a.cy, a.cy);
        const PV ac2 = P2<T>::mk(a.c, a.c), as2 = P2<T>::mk(a.s, a.s), nas2 = P2<T>::mk(-a.s, -a.s);
        const PV aw2 = P2<T>::mk(a.hw + grow, a.hw + grow), ah2 = P2<T>::mk(a.hh + grow, a.hh + grow);
#pragma unroll
        for (int k = 0; k < KC / 2; k++) {
            const PV dx = P2<T>::sub(bx2[k], ax2), dy = P2<T>::sub(by2[k], ay2);
            const PV xl = P2<T>::fma(dy, as2, P2<T>::mul(dx, ac2)), yl = P2<T>::fma(dx, nas2, P2<T>::mul(dy, ac2));
            const PV tx = P2<T>::add(aw2, br2[k]), ty = P2<T>::add(ah2, br2[k]);
            const unsigned bal0 = __ballot_sync(0xffffffffu, Num<T>::abs_(xl.x) <= tx.x && Num<T>::abs_(yl.x) <= ty.x);   // false for NaN padding
            const unsigned bal1 = __ballot_sync(0xffffffffu, Num<T>::abs_(xl.y) <= tx.y && Num<T>::abs_(yl.y) <= ty.y);
            if (lane == (unsigned)(r * KC + 2 * k)) mybal = bal0;
            if (lane == (unsigned)(r * KC + 2 * k + 1)) mybal = bal1;
        }
    }
    // ---- pack: exclusive prefix of the per-(row, chunk) counts; lane r*KC+k expands its ballot into the warp queue, so
    // the queue is ordered by row, then column: the 32 pairs of one clip step share (mostly) one row -> the row record is a
    // broadcast read, and their columns are distinct modulo 32 -> the field-major column reads and the tile store are
    // bank-conflict free.  Entry = row_local * TC + column.
    const unsigned cnt = __popc(mybal);
    unsigned incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { unsigned t = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= (unsigned)d) incl += t; }
    // fp64: one queue for the CTA -- the warps' candidates back to back (still ordered by row, then column), the clip steps dealt round
    // robin to the warps: a queue per warp pads the last step of every warp (half a step of ~11), one queue pads once per tile
    // (7.20 -> 7.04 ms on 30k x 30k).  fp32 keeps a queue per warp: the two CTA barriers cost more than the padding (25.3 against 22.6 ms).
    constexpr bool CTAQ = sizeof(T) == 8;
    __shared__ unsigned s_wtot[IOU_WARPS];
    unsigned wbase = 0, total = __shfl_sync(0xffffffffu, incl, 31);
    uint16_t *q = sm.queue[w];
    if constexpr (CTAQ) {
        if (lane == 31) s_wtot[w] = incl;
        __syncthreads();
        total = 0;
#pragma unroll
        for (int i = 0; i < IOU_WARPS; i++) { const unsigned t = s_wtot[i]; if (i < (int)w) wbase += t; total += t; }
        q = &sm.queue[0][0];
    }
    const unsigned rowbase = CTAQ ? w * RW * TC : 0u;   // queue entry = row of the CTA's tile (shared queue) / of the warp's rows
    for (unsigned pos = wbase + incl - cnt; mybal; mybal &= mybal - 1, pos++)
        q[pos] = (uint16_t)(rowbase + ((lane << 5) | (__ffs(mybal) - 1)));
    if constexpr (CTAQ) __syncthreads(); else __syncwarp();

    // ---- clip: full warps of 32 queued candidates (the last step padded with a repeat of the final entry)
#pragma unroll 1
    for (unsigned h = CTAQ ? w * 32 : 0u; h < total; h += CTAQ ? IOU_WARPS * 32 : 32) {
        const unsigned e = q[min(h + lane, total - 1)];
        const unsigned row = (CTAQ ? 0u : w * RW) + e / TC, col = e % TC;
        BoxRec<T> A = sm.sA[row], B;
        B.cx = sm.sB[0][col]; B.cy = sm.sB[1][col]; B.c = sm.sB[2][col]; B.s = sm.sB[3][col];
        B.hw = sm.sB[4][col]; B.hh = sm.sB[5][col]; B.area = sm.sB[7][col]; B.rho = T(0);
        T v = rbox_iou<T>(A, B);
        if (ZD) v = (T)__fsub_rn(1.f, __fmul_rn((float)v, z_iou(szA[row], szB[col])));   // only candidates pay for the z factor
        if (h + lane < total) sm.tile[row][col] = v;
    }
    if constexpr (CTAQ) __syncthreads();   // other warps clipped candidates of this warp's rows
    else __syncwarp();
}

template <typename T, bool ZD>
__device__ __forceinline__ void iou2dr_tile(const BoxRec<T> *__restrict__ recA, int64_t n, const BoxRec<T> *__restrict__ recB, int64_t m,
                                            T *__restrict__ out, int64_t ld, const ZRange *__restrict__ zA, const ZRange *__restrict__ zB,
                                            const int64_t row0, const int64_t col0)
{
    using S = IouSmem<T>;
    constexpr int TC = S::TC, RW = S::RW;
    constexpr int V = 16 / sizeof(T);    // elements per 16-byte vector
    extern __shared__ __align__(16) unsigned char iou_smem_raw[];
    S &sm = *reinterpret_cast<S *>(iou_smem_raw);
    const unsigned lane = lane_id(), w = threadIdx.x >> 5;
    iou2dr_tile_fill<T, ZD>(recA, recB, zA, zB, row0, col0);

    // stream this warp's rows to HBM: full-line 16-byte stores when the row pointers are 16-byte aligned
    const int64_t wrow0 = row0 + w * RW;
    const int nrows = (int)(n - wrow0 < RW ? (n - wrow0 > 0 ? n - wrow0 : 0) : RW);
    const bool vec_ok = (ld % V == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0) && col0 + TC <= m;
    T *orow = out + wrow0 * ld + col0;
    if (vec_ok && nrows == RW) {
        orow += lane * V;
#pragma unroll
        for (int r = 0; r < RW; r++) {
#pragma unroll
            for (int c = 0; c < TC; c += 32 * V)
                __stcs(reinterpret_cast<float4 *>(orow + c), *reinterpret_cast<const float4 *>(&sm.tile[w * RW + r][lane * V + c]));
            orow += ld;
        }
    } else {
        for (int r = 0; r < nrows; r++, orow += ld) {
            const T *trow = sm.tile[w * RW + r];
            for (int c = lane; c < TC; c += 32)
                if (col0 + c < m) orow[c] = trow[c];
        }
    }
}

template <typename T, bool ZD = false>
__global__ void __launch_bounds__(IOU_THREADS, 3)
iou2dr_tile_kernel(const BoxRec<T> *__restrict__ recA, int64_t n, const BoxRec<T> *__restrict__ recB, int64_t m,
                   T *__restrict__ out, int64_t ld, const ZRange *__restrict__ zA = nullptr, const ZRange *__restrict__ zB = nullptr)
{
    // column tiles on grid.x (fastest): A rows reused, B streams through L2
    const int64_t row0 = ((int64_t)blockIdx.y + (int64_t)blockIdx.z * 65535) * IouTile<T>::TR, col0 = (int64_t)blockIdx.x * IouTile<T>::TC;
    if (row0 >= n) return;
    iou2dr_tile<T, ZD>(recA, n, recB, m, out, ld, zA, zB, row0, col0);
}

// ------------------------------------------------------------------ AABB IoU (method "box"): cheap, one thread per 4 columns
// columns c0 .. c0+3 of the row at out + rowoff
template <typename T>
__device__ __forceinline__ void iou2d_cols(const AABBRec<T> a, const AABBRec<T> *__restrict__ recB, int64_t m, int64_t c0, T *__restrict__ out, int64_t rowoff)
{
#pragma unroll
    for (int k = 0; k < 4; k++)
        if (c0 + k < m) out[rowoff + c0 + k] = aabb_iou<T>(a, recB[c0 + k]);
}

template <typename T>
__global__ void __launch_bounds__(256) iou2d_kernel(const AABBRec<T> *__restrict__ recA, int64_t n, const AABBRec<T> *__restrict__ recB, int64_t m,
                                                    T *__restrict__ out, int64_t ld)
{
    const int64_t row = blockIdx.y;
    const int64_t c0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (row >= n || c0 >= m) return;
    iou2d_cols<T>(recA[row], recB, m, c0, out, row * ld);
}

// AABB variant of the matcher distance (DistanceTypes.IoU, d3d/dgal_wrap.h:70-91): 1 - iou(AABBs) * ziou.  Columns c0 .. c0+3 of the row at out + rowoff.
__device__ __forceinline__ void dist3d_aabb_cols(const AABBRec<float> a, const ZRange za, const AABBRec<float> *__restrict__ recB,
                                                 const ZRange *__restrict__ zB, int64_t m, int64_t c0, float *__restrict__ out, int64_t rowoff)
{
#pragma unroll
    for (int k = 0; k < 4; k++)
        if (c0 + k < m) out[rowoff + c0 + k] = __fsub_rn(1.f, __fmul_rn(aabb_iou<float>(a, recB[c0 + k]), z_iou(za, zB[c0 + k])));
}

__global__ void __launch_bounds__(256) dist3d_aabb_kernel(const AABBRec<float> *__restrict__ recA, const ZRange *__restrict__ zA, int64_t n,
                                                          const AABBRec<float> *__restrict__ recB, const ZRange *__restrict__ zB, int64_t m,
                                                          float *__restrict__ out, int64_t ld)
{
    const int64_t row = blockIdx.y;
    const int64_t c0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (row >= n || c0 >= m) return;
    const AABBRec<float> a = recA[row];
    const ZRange za = zA[row];
    dist3d_aabb_cols(a, za, recB, zB, m, c0, out, row * ld);
}

// 3-D boxes (x, y, z, lx, ly, lz, rz) -> BEV records + z extents.  MODE 0: row records, 1: field-major column records, 2: AABB records
// Box i of n; i >= n writes padding.
template <int MODE, int TILE>
__device__ __forceinline__ void box3d_prep_one(const float *__restrict__ boxes, int64_t n, int64_t i, BoxRec<float> *__restrict__ recs,
                                               AABBRec<float> *__restrict__ arecs, ZRange *__restrict__ z)
{
    BoxRec<float> r;
    ZRange zr = {0.f, 0.f};
    if (i < n) {
        const float *b = boxes + 7 * i;
        if (MODE == 2) arecs[i] = make_aabb_rec<float>(b[0], b[1], b[3], b[4], b[6]);
        else r = make_box_rec<float>(b[0], b[1], b[3], b[4], b[6]);
        const float h = __fdiv_rn(b[5], 2.f);
        zr.lo = __fsub_rn(b[2], h); zr.hi = __fadd_rn(b[2], h);   // z -+ lz / 2 in float (dgal_wrap.h:50-53)
    } else {
        r.cx = r.cy = r.c = r.s = r.hw = r.hh = r.area = 0.f;
        r.rho = NAN;
    }
    z[i] = zr;
    if (MODE == 0) recs[i] = r;
    else if (MODE == 1) {
        float *f = reinterpret_cast<float *>(recs + (i / TILE) * TILE) + (i % TILE);
        f[0 * TILE] = r.cx; f[1 * TILE] = r.cy; f[2 * TILE] = r.c; f[3 * TILE] = r.s;
        f[4 * TILE] = r.hw; f[5 * TILE] = r.hh; f[6 * TILE] = r.rho; f[7 * TILE] = r.area;
    }
}

template <int MODE, int TILE>
__global__ void __launch_bounds__(256) box3d_prep_kernel(const float *__restrict__ boxes, int64_t n, int64_t npad, BoxRec<float> *__restrict__ recs,
                                                         AABBRec<float> *__restrict__ arecs, ZRange *__restrict__ z)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npad) return;
    box3d_prep_one<MODE, TILE>(boxes, n, i, recs, arecs, z);
}

// ------------------------------------------------------------------ frame-batched distance matrix
// Frame f owns boxes [off1[f], off1[f+1]) and [off2[f], off2[f+1]) of the packed inputs and writes its n_f x m_f block (leading
// dimension m_f) at dist + dist_off[f].  Its records and z extents start at off[f] + f * pad: one tile of slack per frame holds the
// frame's own padding, so the layout needs no scan over the frame sizes and the tile body stages full tiles without bounds checks,
// exactly as for one matrix.
__device__ __forceinline__ int64_t frame_rec_base(const int64_t *off, int64_t f, int pad) { return off[f] + f * pad; }

// one CTA per frame: box3d_prep_one over the frame's boxes, padded to a multiple of pad (pad 1: AABB records, no padding)
template <int MODE, int TILE>
__global__ void __launch_bounds__(256) box3d_prep_batch_kernel(const float *__restrict__ boxes, const int64_t *__restrict__ off, int pad,
                                                               BoxRec<float> *__restrict__ recs, AABBRec<float> *__restrict__ arecs, ZRange *__restrict__ z)
{
    const int64_t f = blockIdx.x, b0 = off[f], n = off[f + 1] - b0, base = frame_rec_base(off, f, pad), npad = (n + pad - 1) / pad * pad;
    for (int64_t i = threadIdx.x; i < npad; i += blockDim.x)
        box3d_prep_one<MODE, TILE>(boxes + 7 * b0, n, i, MODE == 2 ? nullptr : recs + base, MODE == 2 ? arecs + base : nullptr, z + base);
}

// rotated: frames on grid.x, column tiles on grid.y, row tiles on grid.z; tiles beyond the frame's own size exit at once
__global__ void __launch_bounds__(IOU_THREADS, 3)
dist3d_batch_tile_kernel(const BoxRec<float> *__restrict__ recA, const int64_t *__restrict__ off1, const BoxRec<float> *__restrict__ recB,
                         const int64_t *__restrict__ off2, const ZRange *__restrict__ zA, const ZRange *__restrict__ zB,
                         const int64_t *__restrict__ dist_off, float *__restrict__ dist)
{
    constexpr int TR = IouTile<float>::TR, TC = IouTile<float>::TC;
    const int64_t f = blockIdx.x, n = off1[f + 1] - off1[f], m = off2[f + 1] - off2[f];
    const int64_t row0 = (int64_t)blockIdx.z * TR, col0 = (int64_t)blockIdx.y * TC;
    if (row0 >= n || col0 >= m) return;
    const int64_t a0 = frame_rec_base(off1, f, TR), b0 = frame_rec_base(off2, f, TC);
    iou2dr_tile<float, true>(recA + a0, n, recB + b0, m, dist + dist_off[f], m, zA + a0, zB + b0, row0, col0);
}

// axis-aligned: frames on grid.x, rows r0 + grid.y, 1024-column chunks on grid.z
__global__ void __launch_bounds__(256) dist3d_aabb_batch_kernel(const AABBRec<float> *__restrict__ recA, const int64_t *__restrict__ off1,
                                                                const AABBRec<float> *__restrict__ recB, const int64_t *__restrict__ off2,
                                                                const ZRange *__restrict__ zA, const ZRange *__restrict__ zB,
                                                                const int64_t *__restrict__ dist_off, float *__restrict__ dist, int64_t r0)
{
    const int64_t f = blockIdx.x, n = off1[f + 1] - off1[f], m = off2[f + 1] - off2[f];
    const int64_t row = r0 + blockIdx.y, c0 = ((int64_t)blockIdx.z * blockDim.x + threadIdx.x) * 4;
    if (row >= n || c0 >= m) return;
    const int64_t a = frame_rec_base(off1, f, 1) + row, b0 = frame_rec_base(off2, f, 1);
    dist3d_aabb_cols(recA[a], zA[a], recB + b0, zB + b0, m, c0, dist + dist_off[f], row * m);
}

// ------------------------------------------------------------------ frame-batched IoU matrix (box2d_iou_batch, methods "rbox" / "box")
// Same layout as the distance matrix: frame f's n_f x m_f block (leading dimension m_f) at out + out_off[f], its records at
// off[f] + f * pad.  Frames on grid.x, the frame's boxes strided over grid.y: box_prep_one over the frame, padded to a multiple of pad.
// A frame of more than max_n boxes is skipped: the tile kernel skips it too (the caller runs the single-matrix kernel on it).
template <typename T, int TILE>
__global__ void __launch_bounds__(256) box_prep_batch_kernel(const T *__restrict__ boxes, const int64_t *__restrict__ off, int pad, int64_t max_n,
                                                             BoxRec<T> *__restrict__ recs)
{
    const int64_t f = blockIdx.x, b0 = off[f], n = off[f + 1] - b0, npad = (n + pad - 1) / pad * pad;
    if (n > max_n) return;
    BoxRec<T> *r = recs + frame_rec_base(off, f, pad);
    for (int64_t i = (int64_t)blockIdx.y * blockDim.x + threadIdx.x; i < npad; i += (int64_t)gridDim.y * blockDim.x)
        box_prep_one<T, TILE>(boxes + 5 * b0, n, i, r);
}

// rotated: frames on grid.x, column tiles on grid.y, row tiles on grid.z; tiles beyond the frame's own size exit at once, and so does
// every tile of a frame beyond the bounds max1 x max2 that size the grid
template <typename T>
__global__ void __launch_bounds__(IOU_THREADS, 3)
iou2dr_batch_tile_kernel(const BoxRec<T> *__restrict__ recA, const int64_t *__restrict__ off1, const BoxRec<T> *__restrict__ recB,
                         const int64_t *__restrict__ off2, int64_t max1, int64_t max2, const int64_t *__restrict__ out_off, T *__restrict__ out)
{
    constexpr int TR = IouTile<T>::TR, TC = IouTile<T>::TC;
    const int64_t f = blockIdx.x, n = off1[f + 1] - off1[f], m = off2[f + 1] - off2[f];
    const int64_t row0 = (int64_t)blockIdx.z * TR, col0 = (int64_t)blockIdx.y * TC;
    if (row0 >= n || col0 >= m || n > max1 || m > max2) return;
    iou2dr_tile<T, false>(recA + frame_rec_base(off1, f, TR), n, recB + frame_rec_base(off2, f, TC), m, out + out_off[f], m, nullptr, nullptr,
                          row0, col0);
}

// axis-aligned: frames on grid.x; the threads of grid.y stride over the frame's (row, 4-column chunk) pairs, each running iou2d_kernel's
// 4 columns of one row, so that a frame of a few dozen columns still fills its CTAs.  Records are the packed AABBs.
template <typename T>
__global__ void __launch_bounds__(256) iou2d_batch_kernel(const AABBRec<T> *__restrict__ recA, const int64_t *__restrict__ off1,
                                                          const AABBRec<T> *__restrict__ recB, const int64_t *__restrict__ off2,
                                                          const int64_t *__restrict__ out_off, T *__restrict__ out)
{
    const int64_t f = blockIdx.x, a0 = off1[f], b0 = off2[f], n = off1[f + 1] - a0, m = off2[f + 1] - b0, cm = (m + 3) / 4, nq = n * cm;
    T *o = out + out_off[f];
    for (int64_t q = (int64_t)blockIdx.y * blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.y * blockDim.x) {
        const int64_t i = q / cm;
        iou2d_cols<T>(recA[a0 + i], recB + b0, m, (q - i * cm) * 4, o, i * m);
    }
}

// ------------------------------------------------------------------ fused max-IoU reduction (box2d_iou_max_batch, methods "rbox" / "box")
// Per box of either set, the largest IoU over the other set of its frame and the frame-local index that attains it, with torch.max's
// rules on the output dtype O: ties (+0 against -0 included) go to the lower index, NaN is the maximum at the first NaN's index.
// Tiles reduce their rows and columns to (value, index) keys and combine them across tiles with atomics on an order-preserving key:
//   hi: the value's bits mapped so that unsigned order is value order (sign flip for >= 0, complement for < 0; -0 maps like +0,
//       every NaN to the top), lo: the complement of the index, so that a larger key is a larger value or, on a tie, a lower index.
// fp32 keys pack (hi << 32 | lo) into one 64-bit atomicMax; fp64 keys are 16 bytes, combined by a 16-byte atomicCAS loop (sm_90+).
// A CAS loop costs retries under contention, but no value is below +0 and keys start at (+0, index 0), so a row or column whose tile
// maximum is +0 commits nothing: on sparse frames almost every tile, and the loop runs rarely.  The initial key is also the answer
// of a row whose every value is +0.  EMPTY (key 0, unreachable from a value) marks a box whose frame's other side is empty: (0, -1).
template <typename O> struct MaxKey;
template <> struct MaxKey<float> {
    using K = unsigned long long;
    static __device__ __forceinline__ K make(float v, int64_t i)
    {
        const unsigned b = __float_as_uint(v);
        const unsigned o = v != v ? 0xffffffffu : v == 0.f ? 0x80000000u : (b >> 31) ? ~b : b | 0x80000000u;
        return (K)o << 32 | (0xffffffffu - (unsigned)i);
    }
    static __device__ __forceinline__ K init() { return 0x80000000ull << 32 | 0xffffffffull; }
    static __device__ __forceinline__ K empty() { return 0; }
    static __device__ __forceinline__ bool above(K a, K b) { return a > b; }
    static __device__ __forceinline__ void commit(K *p, K k) { atomicMax(p, k); }
    static __device__ __forceinline__ void decode(K k, float *v, int64_t *i)
    {
        const unsigned o = (unsigned)(k >> 32);
        if (o == 0) { *v = 0.f; *i = -1; return; }
        *v = o == 0xffffffffu ? __uint_as_float(0x7fffffffu) : __uint_as_float((o >> 31) ? o & 0x7fffffffu : ~o);
        *i = (int64_t)(0xffffffffu - (unsigned)k);
    }
};
struct __align__(16) Key128 { unsigned long long lo, hi; };
template <> struct MaxKey<double> {
    using K = Key128;
    static __device__ __forceinline__ K make(double v, int64_t i)
    {
        const unsigned long long b = (unsigned long long)__double_as_longlong(v), sign = 1ull << 63;
        K k;
        k.hi = v != v ? ~0ull : v == 0.0 ? sign : (b >> 63) ? ~b : b | sign;
        k.lo = ~(unsigned long long)i;
        return k;
    }
    static __device__ __forceinline__ K init() { K k; k.hi = 1ull << 63; k.lo = ~0ull; return k; }
    static __device__ __forceinline__ K empty() { K k; k.hi = 0; k.lo = 0; return k; }
    static __device__ __forceinline__ bool above(K a, K b) { return a.hi > b.hi || (a.hi == b.hi && a.lo > b.lo); }
    static __device__ __forceinline__ void commit(K *p, K k)
    {
        K old = *p;   // possibly stale: keys only grow, so a stale key is below the current one and the CAS corrects it
        while (above(k, old)) {
            const K prev = atomicCAS(p, old, k);
            if (prev.hi == old.hi && prev.lo == old.lo) break;
            old = prev;
        }
    }
    static __device__ __forceinline__ void decode(K k, double *v, int64_t *i)
    {
        if (k.hi == 0) { *v = 0.0; *i = -1; return; }
        const unsigned long long sign = 1ull << 63;
        *v = k.hi == ~0ull ? __longlong_as_double(0x7ff8000000000000ll) : __longlong_as_double((long long)((k.hi & sign) ? k.hi & ~sign : ~k.hi));
        *i = (int64_t)~k.lo;
    }
};
template <typename O> __device__ __forceinline__ typename MaxKey<O>::K key_max(typename MaxKey<O>::K a, typename MaxKey<O>::K b)
{
    return MaxKey<O>::above(b, a) ? b : a;
}

// every box's key: init(), or empty() when its frame's other side is empty.  Frames on grid.x, the frame's boxes of both sets strided over grid.y.
template <typename O>
__global__ void __launch_bounds__(256) iou_max_init_kernel(const int64_t *__restrict__ off1, const int64_t *__restrict__ off2, typename MaxKey<O>::K *__restrict__ key1,
                                                           typename MaxKey<O>::K *__restrict__ key2)
{
    const int64_t f = blockIdx.x, a0 = off1[f], b0 = off2[f], n = off1[f + 1] - a0, m = off2[f + 1] - b0;
    for (int64_t i = (int64_t)blockIdx.y * blockDim.x + threadIdx.x; i < n + m; i += (int64_t)gridDim.y * blockDim.x) {
        if (i < n) key1[a0 + i] = m ? MaxKey<O>::init() : MaxKey<O>::empty();
        else key2[b0 + i - n] = n ? MaxKey<O>::init() : MaxKey<O>::empty();
    }
}

// keys -> values and int64 indices, both sets in one flat pass
template <typename O>
__global__ void __launch_bounds__(256) iou_max_finalise_kernel(const typename MaxKey<O>::K *__restrict__ key1, int64_t total1, const typename MaxKey<O>::K *__restrict__ key2,
                                                               int64_t total2, O *__restrict__ max1, int64_t *__restrict__ idx1, O *__restrict__ max2,
                                                               int64_t *__restrict__ idx2)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total1 + total2; i += (int64_t)gridDim.x * blockDim.x) {
        if (i < total1) MaxKey<O>::decode(key1[i], max1 + i, idx1 + i);
        else MaxKey<O>::decode(key2[i - total1], max2 + i - total1, idx2 + i - total1);
    }
}

// Inside a tile the values are compared as their bits in O: every value is +0, positive or NaN (iou2dr_tile_fill, aabb_iou), so with
// NaN canonicalised the unsigned order of the bits is the value order, +0 is 0 and ties are equal bits.  Keys are built only for commits.
template <typename O> struct OBits;
template <> struct OBits<float> {
    using U = unsigned;
    static __device__ __forceinline__ U canon(float v) { const U u = __float_as_uint(v); return u > 0x7f800000u ? 0x7fffffffu : u; }
    static __device__ __forceinline__ float value(U u) { return __uint_as_float(u); }
};
template <> struct OBits<double> {
    using U = unsigned long long;
    static __device__ __forceinline__ U canon(double v)
    {
        const U u = (U)__double_as_longlong(v);
        return u > 0x7ff0000000000000ull ? 0x7fffffffffffffffull : u;
    }
    static __device__ __forceinline__ double value(U u) { return __longlong_as_double((long long)u); }
};

// rotated: iou2dr_tile_fill's tile, then its row and column maxima instead of the stores.  Frames on grid.x, column tiles ct0 + grid.y,
// row tiles rt0 + grid.z (slabs of 65535 tiles for larger frames: the keys combine across slabs as across tiles).  Records as for the matrix.
template <typename T, typename O>
__global__ void __launch_bounds__(IOU_THREADS, 3)
iou2dr_max_batch_tile_kernel(const BoxRec<T> *__restrict__ recA, const int64_t *__restrict__ off1, const BoxRec<T> *__restrict__ recB,
                             const int64_t *__restrict__ off2, int64_t rt0, int64_t ct0, typename MaxKey<O>::K *__restrict__ key1,
                             typename MaxKey<O>::K *__restrict__ key2)
{
    using S = IouSmem<T>;
    using KT = MaxKey<O>;
    using K = typename KT::K;
    using B = OBits<O>;
    using U = typename B::U;
    constexpr int TR = S::TR, TC = S::TC, RW = S::RW, KC = S::KC;
    const int64_t f = blockIdx.x, n = off1[f + 1] - off1[f], m = off2[f + 1] - off2[f];
    const int64_t row0 = (rt0 + blockIdx.z) * TR, col0 = (ct0 + blockIdx.y) * TC;
    if (row0 >= n || col0 >= m) return;
    iou2dr_tile_fill<T, false>(recA + frame_rec_base(off1, f, TR), recB + frame_rec_base(off2, f, TC), nullptr, nullptr, row0, col0);
    __syncthreads();   // the column maxima read every warp's rows
    extern __shared__ __align__(16) unsigned char iou_smem_raw[];
    S &sm = *reinterpret_cast<S *>(iou_smem_raw);
    const unsigned lane = lane_id(), w = threadIdx.x >> 5;
    K *krow = key1 + off1[f], *kcol = key2 + off2[f];
    // rows: warp w owns rows w*RW .. w*RW+RW-1, lane the KC adjacent columns lane*KC ..; the warp's maximum, then the lowest column
    // holding it.  A row whose maximum is +0 commits nothing (the initial key).  Padding columns hold +0.
    static_assert(KC * sizeof(T) == 16, "one 16-byte load per lane and row");
#pragma unroll
    for (int r = 0; r < RW; r++) {
        const int row = w * RW + r;
        T v[KC];
        *reinterpret_cast<float4 *>(v) = *reinterpret_cast<const float4 *>(&sm.tile[row][lane * KC]);
        U bu = B::canon((O)v[0]);
        int bc = 0;
#pragma unroll
        for (int c = 1; c < KC; c++) { const U u = B::canon((O)v[c]); if (u > bu) { bu = u; bc = c; } }
        U mx = bu;
#pragma unroll
        for (int d = 16; d; d >>= 1) { const U t = __shfl_xor_sync(0xffffffffu, mx, d); mx = t > mx ? t : mx; }
        if (mx == 0) continue;
        int col = bu == mx ? (int)lane * KC + bc : TC;
#pragma unroll
        for (int d = 16; d; d >>= 1) col = min(col, __shfl_xor_sync(0xffffffffu, col, d));
        if (lane == 0 && row0 + row < n) KT::commit(krow + row0 + row, KT::make(B::value(mx), col0 + col));
    }
    // columns: PARTS threads per column, RP rows each, combined through the candidate queue's shared memory (free after the clip)
    constexpr int PARTS = IOU_THREADS / TC, RP = TR / PARTS;
    static_assert(sizeof(sm.queue) >= IOU_THREADS * sizeof(K), "column partials fit the queue");
    K *part = reinterpret_cast<K *>(&sm.queue[0][0]);
    const int c = threadIdx.x % TC, p = threadIdx.x / TC;
    U bu = B::canon((O)sm.tile[p * RP][c]);
    int br = 0;
#pragma unroll 8
    for (int r = 1; r < RP; r++) { const U u = B::canon((O)sm.tile[p * RP + r][c]); if (u > bu) { bu = u; br = r; } }
    part[threadIdx.x] = KT::make(B::value(bu), row0 + p * RP + br);
    __syncthreads();
    if (threadIdx.x < TC) {
        K k = part[threadIdx.x];
#pragma unroll
        for (int q = 1; q < PARTS; q++) k = key_max<O>(k, part[q * TC + threadIdx.x]);
        if (col0 + c < m && KT::above(k, KT::init())) KT::commit(kcol + col0 + c, k);
    }
}

// axis-aligned: a CTA owns a BR x BC tile of a frame.  Its threads fill the tile in shared memory with iou2d_cols, called as
// iou2d_batch_kernel calls it (the row record by value, 4 columns from the records): FMA contraction of aabb_iou<T> depends on how the
// code around it reuses the row's extents, and this shape rounds as the matrix does.  Then rows reduce across the warp and columns
// across the threads of a column, as in the rotated tile.  Frames on grid.x, row tiles rt0 + grid.y, column tiles ct0 + grid.z.
// Records are the packed AABBs.
constexpr int IOU_MAX_BOX_BR = 32, IOU_MAX_BOX_BC = 128;
template <typename T, typename O>
__global__ void __launch_bounds__(256) iou2d_max_batch_kernel(const AABBRec<T> *__restrict__ recA, const int64_t *__restrict__ off1,
                                                              const AABBRec<T> *__restrict__ recB, const int64_t *__restrict__ off2, int64_t rt0,
                                                              int64_t ct0, typename MaxKey<O>::K *__restrict__ key1, typename MaxKey<O>::K *__restrict__ key2)
{
    using KT = MaxKey<O>;
    using K = typename KT::K;
    using B = OBits<O>;
    using U = typename B::U;
    constexpr int BR = IOU_MAX_BOX_BR, BC = IOU_MAX_BOX_BC, RW = BR / 8, PARTS = 256 / BC, RP = BR / PARTS;
    __shared__ __align__(16) T tile[BR][BC];
    __shared__ K part[256];
    const int64_t f = blockIdx.x, a0 = off1[f], b0 = off2[f], n = off1[f + 1] - a0, m = off2[f + 1] - b0;
    const int64_t row0 = (rt0 + blockIdx.y) * BR, col0 = (ct0 + blockIdx.z) * BC;
    if (row0 >= n || col0 >= m) return;
    const int nr = (int)(n - row0 < BR ? n - row0 : BR), nc = (int)(m - col0 < BC ? m - col0 : BC);
    for (int q = threadIdx.x; q < BR * (BC / 4); q += 256) {
        const int r = q / (BC / 4), c4 = q % (BC / 4);
        if (r < nr) iou2d_cols<T>(recA[a0 + row0 + r], recB + b0 + col0, nc, c4 * 4, &tile[0][0], r * BC);
    }
    __syncthreads();
    const unsigned lane = lane_id(), w = threadIdx.x >> 5;
    // rows: warp w owns rows w*RW ..; lane the 4 adjacent columns lane*4 ..
#pragma unroll
    for (int rr = 0; rr < RW; rr++) {
        const int r = w * RW + rr;
        U bu = 0;
        int bc = 0;
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const int col = (int)lane * 4 + c;
            const U u = r < nr && col < nc ? B::canon((O)tile[r][col]) : U(0);
            if (u > bu) { bu = u; bc = col; }
        }
        U mx = bu;
#pragma unroll
        for (int d = 16; d; d >>= 1) { const U t = __shfl_xor_sync(0xffffffffu, mx, d); mx = t > mx ? t : mx; }
        if (mx == 0) continue;
        int col = bu == mx ? bc : BC;
#pragma unroll
        for (int d = 16; d; d >>= 1) col = min(col, __shfl_xor_sync(0xffffffffu, col, d));
        if (lane == 0) KT::commit(key1 + a0 + row0 + r, KT::make(B::value(mx), col0 + col));
    }
    // columns: PARTS threads per column, RP rows each
    const int c = threadIdx.x % BC, p = threadIdx.x / BC;
    U bu = 0;
    int br = 0;
#pragma unroll 4
    for (int r = 0; r < RP; r++) {
        const U u = p * RP + r < nr && c < nc ? B::canon((O)tile[p * RP + r][c]) : U(0);
        if (u > bu) { bu = u; br = r; }
    }
    part[threadIdx.x] = bu ? KT::make(B::value(bu), row0 + p * RP + br) : KT::init();
    __syncthreads();
    if ((int)threadIdx.x < nc) {
        K k = part[threadIdx.x];
#pragma unroll
        for (int q = 1; q < PARTS; q++) k = key_max<O>(k, part[q * BC + threadIdx.x]);
        if (KT::above(k, KT::init())) KT::commit(key2 + b0 + col0 + threadIdx.x, k);
    }
}

// ------------------------------------------------------------------ candidate counter (measurement only; SURVEY.md 8(d) accounting)
template <typename T>
__global__ void __launch_bounds__(256) count_candidates_kernel(const BoxRec<T> *__restrict__ recA, int64_t n, const BoxRec<T> *__restrict__ recB, int64_t m,
                                                               unsigned long long *__restrict__ counter)
{
    __shared__ unsigned long long bsum;
    if (threadIdx.x == 0) bsum = 0;
    __syncthreads();
    const int64_t row = blockIdx.y;
    unsigned long long c = 0;
    if (row < n) {
        const T ax = recA[row].cx, ay = recA[row].cy, ar = recA[row].rho;
        for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < m; j += (int64_t)gridDim.x * blockDim.x) {
            T dx = ax - recB[j].cx, dy = ay - recB[j].cy, rs = ar + recB[j].rho;
            c += (dx * dx + dy * dy <= rs * rs) ? 1 : 0;
        }
    }
    for (int d = 16; d; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
    if (lane_id() == 0 && c) atomicAdd(&bsum, c);
    __syncthreads();
    if (threadIdx.x == 0 && bsum) atomicAdd(counter + (blockIdx.y & 63), bsum);
}

// ------------------------------------------------------------------ host side
template <typename T> static size_t iou_ws_bytes(int64_t n, int64_t m)
{
    constexpr int TR = IouTile<T>::TR, TC = IouTile<T>::TC;
    return 256 + align_up((size_t)cdiv(n > 0 ? n : 1, TR) * TR * sizeof(BoxRec<T>)) + align_up((size_t)cdiv(m > 0 ? m : 1, TC) * TC * sizeof(BoxRec<T>));
}

template <typename T, int FIELD_MAJOR_TILE = 0>
static int prep_boxes(const T *boxes, int64_t n, int tile, BoxRec<T> *recs, cudaStream_t st)
{
    int64_t npad = cdiv(n, tile) * tile;
    box_prep_kernel<T, FIELD_MAJOR_TILE><<<(unsigned)cdiv(npad, 256), 256, 0, st>>>(boxes, n, npad, recs); D3D_LAUNCHED();
    return D3D_OK;
}

template <typename T>
static int iou2dr_impl(const T *b1, int64_t n, const T *b2, int64_t m, T *out, int64_t ld, void *ws, size_t ws_bytes, cudaStream_t st)
{
    if (n < 0 || m < 0 || ld < m) return D3D_ERR_INVALID_ARGUMENT;
    if (n == 0 || m == 0) return D3D_OK;
    if (!b1 || !b2 || !out) return D3D_ERR_INVALID_ARGUMENT;
    if (ws_bytes < iou_ws_bytes<T>(n, m) || !ws) return D3D_ERR_WORKSPACE;
    constexpr int TR = IouTile<T>::TR, TC = IouTile<T>::TC;
    Arena a(ws, ws_bytes);
    a.take<char>(256);
    int64_t tiles_r = cdiv(n, TR), tiles_c = cdiv(m, TC);
    BoxRec<T> *ra = a.take<BoxRec<T>>(tiles_r * TR), *rb = a.take<BoxRec<T>>(tiles_c * TC);
    int rc;
    if ((rc = prep_boxes<T>(b1, n, TR, ra, st))) return rc;
    if ((rc = prep_boxes<T, TC>(b2, m, TC, rb, st))) return rc;
    if (tiles_c > 0x7fffffffll || tiles_r > 65535ll * 65535ll) return D3D_ERR_INVALID_ARGUMENT;
    const dim3 grid((unsigned)tiles_c, (unsigned)(tiles_r < 65535 ? tiles_r : 65535), (unsigned)cdiv(tiles_r, 65535));
    static bool smem_opt_in[64] = {};   // per instantiation and per device: the attribute is per function and context, and sticky
    int dev = 0;
    D3D_CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !smem_opt_in[dev]) {
        D3D_CUDA_TRY(cudaFuncSetAttribute(iou2dr_tile_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(IouSmem<T>)));
        if (dev >= 0 && dev < 64) smem_opt_in[dev] = true;
    }
    iou2dr_tile_kernel<T><<<grid, IOU_THREADS, sizeof(IouSmem<T>), st>>>(ra, n, rb, m, out, ld); D3D_LAUNCHED();
    return D3D_OK;
}

template <typename T>
static int iou2d_impl(const T *b1, int64_t n, const T *b2, int64_t m, T *out, int64_t ld, void *ws, size_t ws_bytes, cudaStream_t st)
{
    if (n < 0 || m < 0 || ld < m) return D3D_ERR_INVALID_ARGUMENT;
    if (n == 0 || m == 0) return D3D_OK;
    if (!b1 || !b2 || !out) return D3D_ERR_INVALID_ARGUMENT;
    if (ws_bytes < iou_ws_bytes<T>(n, m) || !ws) return D3D_ERR_WORKSPACE;
    if (n > 65535ll * 65535ll) return D3D_ERR_INVALID_ARGUMENT;
    Arena a(ws, ws_bytes);
    a.take<char>(256);
    AABBRec<T> *ra = a.take<AABBRec<T>>(n), *rb = a.take<AABBRec<T>>(m);
    aabb_prep_kernel<T><<<(unsigned)cdiv(n, 256), 256, 0, st>>>(b1, n, ra); D3D_LAUNCHED();
    aabb_prep_kernel<T><<<(unsigned)cdiv(m, 256), 256, 0, st>>>(b2, m, rb); D3D_LAUNCHED();
    // rows on grid.y in slabs of 65535
    for (int64_t r0 = 0; r0 < n; r0 += 65535) {
        int64_t nr = n - r0 < 65535 ? n - r0 : 65535;
        dim3 grid((unsigned)cdiv(m, 1024), (unsigned)nr);
        iou2d_kernel<T><<<grid, 256, 0, st>>>(ra + r0, nr, rb, m, out + r0 * ld, ld); D3D_LAUNCHED();
    }
    return D3D_OK;
}

static size_t dist3d_ws_bytes(int64_t n, int64_t m)
{
    constexpr int TR = IouTile<float>::TR, TC = IouTile<float>::TC;
    const size_t np = (size_t)cdiv(n > 0 ? n : 1, TR) * TR, mp = (size_t)cdiv(m > 0 ? m : 1, TC) * TC;
    return iou_ws_bytes<float>(n, m) + align_up(np * sizeof(ZRange)) + align_up(mp * sizeof(ZRange));
}

// replaces the pair loops of ScoreMatcher.prepare_boxes (d3d/tracking/matcher.pyx:55-76) over box3dr_iou / box3d_iou (d3d/dgal_wrap.h:45-91)
static int dist3d_impl(const float *b1, int64_t n, const float *b2, int64_t m, int rotated, float *out, int64_t ld, void *ws, size_t ws_bytes, cudaStream_t st)
{
    if (n < 0 || m < 0 || ld < m) return D3D_ERR_INVALID_ARGUMENT;
    if (n == 0 || m == 0) return D3D_OK;
    if (!b1 || !b2 || !out) return D3D_ERR_INVALID_ARGUMENT;
    if (ws_bytes < dist3d_ws_bytes(n, m) || !ws) return D3D_ERR_WORKSPACE;
    constexpr int TR = IouTile<float>::TR, TC = IouTile<float>::TC;
    Arena a(ws, ws_bytes);
    a.take<char>(256);
    const int64_t tiles_r = cdiv(n, TR), tiles_c = cdiv(m, TC), np = tiles_r * TR, mp = tiles_c * TC;
    BoxRec<float> *ra = a.take<BoxRec<float>>(np), *rb = a.take<BoxRec<float>>(mp);
    ZRange *za = a.take<ZRange>(np), *zb = a.take<ZRange>(mp);
    if (!a.ok()) return D3D_ERR_WORKSPACE;
    if (!rotated) {
        if (n > 65535ll * 65535ll) return D3D_ERR_INVALID_ARGUMENT;
        AABBRec<float> *aa = reinterpret_cast<AABBRec<float> *>(ra), *ab = reinterpret_cast<AABBRec<float> *>(rb);   // 16-byte records fit the 32-byte slots
        box3d_prep_kernel<2, 1><<<(unsigned)cdiv(n, 256), 256, 0, st>>>(b1, n, n, nullptr, aa, za); D3D_LAUNCHED();
        box3d_prep_kernel<2, 1><<<(unsigned)cdiv(m, 256), 256, 0, st>>>(b2, m, m, nullptr, ab, zb); D3D_LAUNCHED();
        for (int64_t r0 = 0; r0 < n; r0 += 65535) {
            const int64_t nr = n - r0 < 65535 ? n - r0 : 65535;
            dist3d_aabb_kernel<<<dim3((unsigned)cdiv(m, 1024), (unsigned)nr), 256, 0, st>>>(aa + r0, za + r0, nr, ab, zb, m, out + r0 * ld, ld); D3D_LAUNCHED();
        }
        return D3D_OK;
    }
    box3d_prep_kernel<0, 1><<<(unsigned)cdiv(np, 256), 256, 0, st>>>(b1, n, np, ra, nullptr, za); D3D_LAUNCHED();
    box3d_prep_kernel<1, TC><<<(unsigned)cdiv(mp, 256), 256, 0, st>>>(b2, m, mp, rb, nullptr, zb); D3D_LAUNCHED();
    if (tiles_c > 0x7fffffffll || tiles_r > 65535ll * 65535ll) return D3D_ERR_INVALID_ARGUMENT;
    const dim3 grid((unsigned)tiles_c, (unsigned)(tiles_r < 65535 ? tiles_r : 65535), (unsigned)cdiv(tiles_r, 65535));
    static bool smem_opt_in[64] = {};
    int dev = 0;
    D3D_CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !smem_opt_in[dev]) {
        D3D_CUDA_TRY(cudaFuncSetAttribute(iou2dr_tile_kernel<float, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(IouSmem<float>)));
        if (dev >= 0 && dev < 64) smem_opt_in[dev] = true;
    }
    iou2dr_tile_kernel<float, true><<<grid, IOU_THREADS, sizeof(IouSmem<float>), st>>>(ra, n, rb, m, out, ld, za, zb); D3D_LAUNCHED();
    return D3D_OK;
}

static size_t dist3d_batch_ws_bytes(int64_t total1, int64_t total2, int64_t nframes)
{
    constexpr int TR = IouTile<float>::TR, TC = IouTile<float>::TC;
    if (total1 < 0 || total2 < 0 || nframes < 0) return 0;
    const size_t np = (size_t)(total1 + nframes * TR), mp = (size_t)(total2 + nframes * TC);
    return 256 + align_up(np * sizeof(BoxRec<float>)) + align_up(mp * sizeof(BoxRec<float>)) + align_up(np * sizeof(ZRange)) + align_up(mp * sizeof(ZRange));
}

// every frame of a packed batch through dist3d_impl's kernels: one prep launch per box set and one distance launch (AABB: one per
// 65535 rows of the largest frame), whatever the number of frames
static int dist3d_batch_impl(const float *b1, int64_t total1, const int64_t *off1, const float *b2, int64_t total2, const int64_t *off2, int64_t nframes,
                             int64_t max1, int64_t max2, int rotated, const int64_t *dist_off, float *dist, void *ws, size_t ws_bytes, cudaStream_t st)
{
    if (total1 < 0 || total2 < 0 || nframes < 0 || max1 < 0 || max2 < 0) return D3D_ERR_INVALID_ARGUMENT;
    if (nframes == 0 || total1 == 0 || total2 == 0) return D3D_OK;   // every block is empty
    if (!b1 || !b2 || !off1 || !off2 || !dist_off || !dist) return D3D_ERR_INVALID_ARGUMENT;
    if (nframes > 0x7fffffffll) return D3D_ERR_UNSUPPORTED;
    if (ws_bytes < dist3d_batch_ws_bytes(total1, total2, nframes) || !ws) return D3D_ERR_WORKSPACE;
    constexpr int TR = IouTile<float>::TR, TC = IouTile<float>::TC;
    if (max1 == 0) max1 = total1;   // 0: bound unknown
    if (max2 == 0) max2 = total2;
    const int64_t tiles_r = cdiv(max1, TR), tiles_c = cdiv(max2, TC), np = total1 + nframes * TR, mp = total2 + nframes * TC;
    if (rotated ? (tiles_r > 65535 || tiles_c > 65535) : cdiv(max2, 1024) > 65535) return D3D_ERR_UNSUPPORTED;
    Arena a(ws, ws_bytes);
    a.take<char>(256);
    BoxRec<float> *ra = a.take<BoxRec<float>>(np), *rb = a.take<BoxRec<float>>(mp);
    ZRange *za = a.take<ZRange>(np), *zb = a.take<ZRange>(mp);
    if (!a.ok()) return D3D_ERR_WORKSPACE;
    const unsigned nf = (unsigned)nframes;
    if (!rotated) {
        AABBRec<float> *aa = reinterpret_cast<AABBRec<float> *>(ra), *ab = reinterpret_cast<AABBRec<float> *>(rb);   // 16-byte records in 32-byte slots
        box3d_prep_batch_kernel<2, 1><<<nf, 256, 0, st>>>(b1, off1, 1, nullptr, aa, za); D3D_LAUNCHED();
        box3d_prep_batch_kernel<2, 1><<<nf, 256, 0, st>>>(b2, off2, 1, nullptr, ab, zb); D3D_LAUNCHED();
        for (int64_t r0 = 0; r0 < max1; r0 += 65535) {
            const int64_t nr = max1 - r0 < 65535 ? max1 - r0 : 65535;
            dist3d_aabb_batch_kernel<<<dim3(nf, (unsigned)nr, (unsigned)cdiv(max2, 1024)), 256, 0, st>>>(aa, off1, ab, off2, za, zb, dist_off, dist, r0);
            D3D_LAUNCHED();
        }
        return D3D_OK;
    }
    box3d_prep_batch_kernel<0, 1><<<nf, 256, 0, st>>>(b1, off1, TR, ra, nullptr, za); D3D_LAUNCHED();
    box3d_prep_batch_kernel<1, TC><<<nf, 256, 0, st>>>(b2, off2, TC, rb, nullptr, zb); D3D_LAUNCHED();
    static bool smem_opt_in[64] = {};
    int dev = 0;
    D3D_CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !smem_opt_in[dev]) {
        D3D_CUDA_TRY(cudaFuncSetAttribute(dist3d_batch_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(IouSmem<float>)));
        if (dev >= 0 && dev < 64) smem_opt_in[dev] = true;
    }
    dist3d_batch_tile_kernel<<<dim3(nf, (unsigned)tiles_c, (unsigned)tiles_r), IOU_THREADS, sizeof(IouSmem<float>), st>>>(ra, off1, rb, off2, za, zb, dist_off, dist);
    D3D_LAUNCHED();
    return D3D_OK;
}

template <typename T> static size_t iou_batch_ws_bytes(int64_t total1, int64_t total2, int64_t nframes)
{
    constexpr int TR = IouTile<T>::TR, TC = IouTile<T>::TC;
    if (total1 < 0 || total2 < 0 || nframes < 0) return 0;
    const size_t np = (size_t)(total1 + nframes * TR), mp = (size_t)(total2 + nframes * TC);
    return 256 + align_up(np * sizeof(BoxRec<T>)) + align_up(mp * sizeof(BoxRec<T>));
}

// GIoU / DIoU forward of a packed batch (iou_grad.cu)
template <typename T>
int iou_ex_batch_fwd(const T *b1, const int64_t *off1, const T *b2, const int64_t *off2, int64_t nframes, int64_t max_pairs, int iou_type,
                     const int64_t *out_off, T *out, cudaStream_t st);

// every frame of a packed batch through the single-matrix per-pair code: "rbox" and "box" two prep launches and one IoU launch, "grbox" /
// "drbox" one launch, whatever the number of frames
template <typename T>
static int iou_batch_impl(const T *b1, int64_t total1, const int64_t *off1, const T *b2, int64_t total2, const int64_t *off2, int64_t nframes,
                          int64_t max1, int64_t max2, int iou_type, const int64_t *out_off, T *out, void *ws, size_t ws_bytes, cudaStream_t st)
{
    if (iou_type != D3D_IOU_BOX && iou_type != D3D_IOU_RBOX && iou_type != D3D_IOU_GRBOX && iou_type != D3D_IOU_DRBOX) return D3D_ERR_INVALID_ARGUMENT;
    if (total1 < 0 || total2 < 0 || nframes < 0 || max1 < 0 || max2 < 0) return D3D_ERR_INVALID_ARGUMENT;
    if (nframes == 0 || total1 == 0 || total2 == 0) return D3D_OK;   // every block is empty
    if (!b1 || !b2 || !off1 || !off2 || !out_off || !out) return D3D_ERR_INVALID_ARGUMENT;
    if (nframes > 0x7fffffffll) return D3D_ERR_UNSUPPORTED;
    if (max1 == 0) max1 = total1;   // 0: bound unknown
    if (max2 == 0) max2 = total2;
    if (iou_type == D3D_IOU_GRBOX || iou_type == D3D_IOU_DRBOX)   // no records: the pair code reads the boxes
        return iou_ex_batch_fwd<T>(b1, off1, b2, off2, nframes, pair_bound(max1, max2), iou_type, out_off, out, st);
    constexpr int TR = IouTile<T>::TR, TC = IouTile<T>::TC;
    const int64_t tiles_r = cdiv(max1, TR), tiles_c = cdiv(max2, TC);
    if (iou_type == D3D_IOU_RBOX && (tiles_r > 65535 || tiles_c > 65535)) return D3D_ERR_UNSUPPORTED;
    if (ws_bytes < iou_batch_ws_bytes<T>(total1, total2, nframes) || !ws) return D3D_ERR_WORKSPACE;
    Arena a(ws, ws_bytes);
    a.take<char>(256);
    BoxRec<T> *ra = a.take<BoxRec<T>>(total1 + nframes * TR), *rb = a.take<BoxRec<T>>(total2 + nframes * TC);
    if (!a.ok()) return D3D_ERR_WORKSPACE;
    const unsigned nf = (unsigned)nframes;
    if (iou_type == D3D_IOU_BOX) {   // the AABB records need no frame padding: box i's record is record i
        AABBRec<T> *aa = reinterpret_cast<AABBRec<T> *>(ra), *ab = reinterpret_cast<AABBRec<T> *>(rb);
        aabb_prep_kernel<T><<<(unsigned)cdiv(total1, 256), 256, 0, st>>>(b1, total1, aa); D3D_LAUNCHED();
        aabb_prep_kernel<T><<<(unsigned)cdiv(total2, 256), 256, 0, st>>>(b2, total2, ab); D3D_LAUNCHED();
        iou2d_batch_kernel<T><<<dim3(nf, stride_blocks(pair_bound(max1, cdiv(max2, 4)), 256)), 256, 0, st>>>(aa, off1, ab, off2, out_off, out); D3D_LAUNCHED();
        return D3D_OK;
    }
    box_prep_batch_kernel<T, 0><<<dim3(nf, stride_blocks(tiles_r * TR, 256)), 256, 0, st>>>(b1, off1, TR, max1, ra); D3D_LAUNCHED();
    box_prep_batch_kernel<T, TC><<<dim3(nf, stride_blocks(tiles_c * TC, 256)), 256, 0, st>>>(b2, off2, TC, max2, rb); D3D_LAUNCHED();
    static bool smem_opt_in[64] = {};   // per instantiation and per device
    int dev = 0;
    D3D_CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64 || !smem_opt_in[dev]) {
        D3D_CUDA_TRY(cudaFuncSetAttribute(iou2dr_batch_tile_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(IouSmem<T>)));
        if (dev >= 0 && dev < 64) smem_opt_in[dev] = true;
    }
    iou2dr_batch_tile_kernel<T><<<dim3(nf, (unsigned)tiles_c, (unsigned)tiles_r), IOU_THREADS, sizeof(IouSmem<T>), st>>>(ra, off1, rb, off2, max1, max2, out_off, out);
    D3D_LAUNCHED();
    return D3D_OK;
}

// the records of iou_batch_ws_bytes, then one key per box of each set (sized for the larger fp64 key when the inputs are fp64)
template <typename T> static size_t iou_max_batch_ws_bytes(int64_t total1, int64_t total2, int64_t nframes)
{
    if (total1 < 0 || total2 < 0 || nframes < 0) return 0;
    return iou_batch_ws_bytes<T>(total1, total2, nframes) + align_up((size_t)total1 * sizeof(typename MaxKey<T>::K)) +
           align_up((size_t)total2 * sizeof(typename MaxKey<T>::K));
}

template <typename T, typename O>
static int iou_max_batch_run(const T *b1, int64_t total1, const int64_t *off1, const T *b2, int64_t total2, const int64_t *off2, int64_t nframes,
                             int64_t max1, int64_t max2, int iou_type, O *max1o, int64_t *idx1, O *max2o, int64_t *idx2, void *ws, size_t ws_bytes,
                             cudaStream_t st)
{
    using K = typename MaxKey<O>::K;
    constexpr int TR = IouTile<T>::TR, TC = IouTile<T>::TC;
    if (sizeof(O) == 4 && (max1 > 0xffffffffll || max2 > 0xffffffffll)) return D3D_ERR_UNSUPPORTED;   // the fp32 key holds a 32-bit index
    Arena a(ws, ws_bytes);
    a.take<char>(256);
    BoxRec<T> *ra = a.take<BoxRec<T>>(total1 + nframes * TR), *rb = a.take<BoxRec<T>>(total2 + nframes * TC);
    K *k1 = reinterpret_cast<K *>(a.take<typename MaxKey<T>::K>(total1)), *k2 = reinterpret_cast<K *>(a.take<typename MaxKey<T>::K>(total2));
    if (!a.ok()) return D3D_ERR_WORKSPACE;
    const unsigned nf = (unsigned)nframes;
    iou_max_init_kernel<O><<<dim3(nf, stride_blocks(max1 + max2, 256)), 256, 0, st>>>(off1, off2, k1, k2); D3D_LAUNCHED();
    if (total1 > 0 && total2 > 0) {
        if (iou_type == D3D_IOU_BOX) {
            AABBRec<T> *aa = reinterpret_cast<AABBRec<T> *>(ra), *ab = reinterpret_cast<AABBRec<T> *>(rb);
            aabb_prep_kernel<T><<<(unsigned)cdiv(total1, 256), 256, 0, st>>>(b1, total1, aa); D3D_LAUNCHED();
            aabb_prep_kernel<T><<<(unsigned)cdiv(total2, 256), 256, 0, st>>>(b2, total2, ab); D3D_LAUNCHED();
            const int64_t tr = cdiv(max1, IOU_MAX_BOX_BR), tc = cdiv(max2, IOU_MAX_BOX_BC);
            for (int64_t r0 = 0; r0 < tr; r0 += 65535)
                for (int64_t c0 = 0; c0 < tc; c0 += 65535) {
                    const dim3 grid(nf, (unsigned)(tr - r0 < 65535 ? tr - r0 : 65535), (unsigned)(tc - c0 < 65535 ? tc - c0 : 65535));
                    iou2d_max_batch_kernel<T, O><<<grid, 256, 0, st>>>(aa, off1, ab, off2, r0, c0, k1, k2); D3D_LAUNCHED();
                }
        } else {
            const int64_t tr = cdiv(max1, TR), tc = cdiv(max2, TC);
            box_prep_batch_kernel<T, 0><<<dim3(nf, stride_blocks(tr * TR, 256)), 256, 0, st>>>(b1, off1, TR, max1, ra); D3D_LAUNCHED();
            box_prep_batch_kernel<T, TC><<<dim3(nf, stride_blocks(tc * TC, 256)), 256, 0, st>>>(b2, off2, TC, max2, rb); D3D_LAUNCHED();
            static bool smem_opt_in[64] = {};   // per instantiation and per device
            int dev = 0;
            D3D_CUDA_TRY(cudaGetDevice(&dev));
            if (dev < 0 || dev >= 64 || !smem_opt_in[dev]) {
                D3D_CUDA_TRY(cudaFuncSetAttribute(iou2dr_max_batch_tile_kernel<T, O>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(IouSmem<T>)));
                if (dev >= 0 && dev < 64) smem_opt_in[dev] = true;
            }
            for (int64_t r0 = 0; r0 < tr; r0 += 65535)
                for (int64_t c0 = 0; c0 < tc; c0 += 65535) {
                    const dim3 grid(nf, (unsigned)(tc - c0 < 65535 ? tc - c0 : 65535), (unsigned)(tr - r0 < 65535 ? tr - r0 : 65535));
                    iou2dr_max_batch_tile_kernel<T, O><<<grid, IOU_THREADS, sizeof(IouSmem<T>), st>>>(ra, off1, rb, off2, r0, c0, k1, k2); D3D_LAUNCHED();
                }
        }
    }
    iou_max_finalise_kernel<O><<<stride_blocks(total1 + total2, 256), 256, 0, st>>>(k1, total1, k2, total2, max1o, idx1, max2o, idx2); D3D_LAUNCHED();
    return D3D_OK;
}

// per box of a packed batch, the maximum IoU over the other set of its frame and its index: an init, two preparations, the tile
// launches (one per slab of 65535 x 65535 tiles) and a finalise, whatever the number of frames
template <typename T>
static int iou_max_batch_impl(const T *b1, int64_t total1, const int64_t *off1, const T *b2, int64_t total2, const int64_t *off2, int64_t nframes,
                              int64_t max1, int64_t max2, int iou_type, int out_dtype, void *max1o, int64_t *idx1, void *max2o, int64_t *idx2,
                              void *ws, size_t ws_bytes, cudaStream_t st)
{
    if (iou_type != D3D_IOU_BOX && iou_type != D3D_IOU_RBOX) return D3D_ERR_INVALID_ARGUMENT;
    if (out_dtype != D3D_F32 && !(sizeof(T) == 8 && out_dtype == D3D_F64)) return D3D_ERR_INVALID_ARGUMENT;
    if (total1 < 0 || total2 < 0 || nframes < 0 || max1 < 0 || max2 < 0) return D3D_ERR_INVALID_ARGUMENT;
    if (nframes == 0 || total1 + total2 == 0) return D3D_OK;   // no box
    if (!off1 || !off2 || (total1 && (!b1 || !max1o || !idx1)) || (total2 && (!b2 || !max2o || !idx2))) return D3D_ERR_INVALID_ARGUMENT;
    if (nframes > 0x7fffffffll) return D3D_ERR_UNSUPPORTED;
    if (ws_bytes < iou_max_batch_ws_bytes<T>(total1, total2, nframes) || !ws) return D3D_ERR_WORKSPACE;
    if (max1 == 0) max1 = total1;   // 0: bound unknown
    if (max2 == 0) max2 = total2;
    if constexpr (sizeof(T) == 8) {
        if (out_dtype == D3D_F64)
            return iou_max_batch_run<T, double>(b1, total1, off1, b2, total2, off2, nframes, max1, max2, iou_type, (double *)max1o, idx1, (double *)max2o,
                                                idx2, ws, ws_bytes, st);
    }
    return iou_max_batch_run<T, float>(b1, total1, off1, b2, total2, off2, nframes, max1, max2, iou_type, (float *)max1o, idx1, (float *)max2o, idx2,
                                       ws, ws_bytes, st);
}

template <typename T>
static int count_cand_impl(const T *b1, int64_t n, const T *b2, int64_t m, unsigned long long *counters64, void *ws, size_t ws_bytes, cudaStream_t st)
{
    if (n <= 0 || m <= 0) return D3D_ERR_INVALID_ARGUMENT;
    if (ws_bytes < iou_ws_bytes<T>(n, m) || !ws) return D3D_ERR_WORKSPACE;
    constexpr int TR = IouTile<T>::TR, TC = IouTile<T>::TC;
    Arena a(ws, ws_bytes);
    a.take<char>(256);
    BoxRec<T> *ra = a.take<BoxRec<T>>(cdiv(n, TR) * TR), *rb = a.take<BoxRec<T>>(cdiv(m, TC) * TC);
    int rc;
    if ((rc = prep_boxes<T>(b1, n, TR, ra, st))) return rc;
    if ((rc = prep_boxes<T>(b2, m, TC, rb, st))) return rc;
    D3D_CUDA_TRY(cudaMemsetAsync(counters64, 0, 64 * sizeof(unsigned long long), st));
    for (int64_t r0 = 0; r0 < n; r0 += 65535) {
        int64_t nr = n - r0 < 65535 ? n - r0 : 65535;
        dim3 grid((unsigned)(cdiv(m, 256) < 64 ? cdiv(m, 256) : 64), (unsigned)nr);
        count_candidates_kernel<T><<<grid, 256, 0, st>>>(ra + r0, nr, rb, m, counters64); D3D_LAUNCHED();
    }
    return D3D_OK;
}

}  // namespace d3d

using namespace d3d;

extern "C" size_t d3d_iou_workspace_bytes(int64_t n, int64_t m, int dtype)
{
    return dtype == D3D_F64 ? iou_ws_bytes<double>(n, m) : iou_ws_bytes<float>(n, m);
}
extern "C" int d3d_iou2dr_f32(const float *b1, int64_t n, const float *b2, int64_t m, float *ious, int64_t ld, void *ws, size_t wsb, void *stream)
{ return iou2dr_impl<float>(b1, n, b2, m, ious, ld, ws, wsb, (cudaStream_t)stream); }
extern "C" int d3d_iou2dr_f64(const double *b1, int64_t n, const double *b2, int64_t m, double *ious, int64_t ld, void *ws, size_t wsb, void *stream)
{ return iou2dr_impl<double>(b1, n, b2, m, ious, ld, ws, wsb, (cudaStream_t)stream); }
extern "C" int d3d_iou2d_f32(const float *b1, int64_t n, const float *b2, int64_t m, float *ious, int64_t ld, void *ws, size_t wsb, void *stream)
{ return iou2d_impl<float>(b1, n, b2, m, ious, ld, ws, wsb, (cudaStream_t)stream); }
extern "C" int d3d_iou2d_f64(const double *b1, int64_t n, const double *b2, int64_t m, double *ious, int64_t ld, void *ws, size_t wsb, void *stream)
{ return iou2d_impl<double>(b1, n, b2, m, ious, ld, ws, wsb, (cudaStream_t)stream); }
extern "C" size_t d3d_iou3d_distance_workspace_bytes(int64_t n, int64_t m) { return dist3d_ws_bytes(n, m); }
extern "C" int d3d_iou3d_distance_f32(const float *boxes1, int64_t n, const float *boxes2, int64_t m, int rotated, float *dist, int64_t ld, void *ws, size_t wsb,
                                      void *stream)
{ return dist3d_impl(boxes1, n, boxes2, m, rotated, dist, ld, ws, wsb, (cudaStream_t)stream); }
extern "C" size_t d3d_iou3d_distance_batch_workspace_bytes(int64_t total1, int64_t total2, int64_t nframes) { return dist3d_batch_ws_bytes(total1, total2, nframes); }
extern "C" int d3d_iou3d_distance_batch_f32(const float *boxes1, int64_t total1, const int64_t *offsets1, const float *boxes2, int64_t total2,
                                            const int64_t *offsets2, int64_t nframes, int64_t max_frame1, int64_t max_frame2, int rotated,
                                            const int64_t *dist_offsets, float *dist, void *ws, size_t wsb, void *stream)
{
    return dist3d_batch_impl(boxes1, total1, offsets1, boxes2, total2, offsets2, nframes, max_frame1, max_frame2, rotated, dist_offsets, dist, ws, wsb,
                             (cudaStream_t)stream);
}
extern "C" size_t d3d_box2d_iou_batch_workspace_bytes(int64_t total1, int64_t total2, int64_t nframes, int dtype)
{
    return dtype == D3D_F64 ? iou_batch_ws_bytes<double>(total1, total2, nframes) : iou_batch_ws_bytes<float>(total1, total2, nframes);
}
#define D3D_IOU_BATCH_ENTRY(NAME, T)                                                                                                  \
    extern "C" int NAME(const T *boxes1, int64_t total1, const int64_t *offsets1, const T *boxes2, int64_t total2, const int64_t *offsets2, \
                        int64_t nframes, int64_t max_frame1, int64_t max_frame2, int iou_type, const int64_t *out_offsets, T *out,     \
                        void *ws, size_t wsb, void *stream)                                                                           \
    {                                                                                                                                 \
        return iou_batch_impl<T>(boxes1, total1, offsets1, boxes2, total2, offsets2, nframes, max_frame1, max_frame2, iou_type,       \
                                 out_offsets, out, ws, wsb, (cudaStream_t)stream);                                                    \
    }
D3D_IOU_BATCH_ENTRY(d3d_box2d_iou_batch_f32, float)
D3D_IOU_BATCH_ENTRY(d3d_box2d_iou_batch_f64, double)
extern "C" size_t d3d_box2d_iou_max_batch_workspace_bytes(int64_t total1, int64_t total2, int64_t nframes, int dtype)
{
    return dtype == D3D_F64 ? iou_max_batch_ws_bytes<double>(total1, total2, nframes) : iou_max_batch_ws_bytes<float>(total1, total2, nframes);
}
#define D3D_IOU_MAX_BATCH_ENTRY(NAME, T)                                                                                                   \
    extern "C" int NAME(const T *boxes1, int64_t total1, const int64_t *offsets1, const T *boxes2, int64_t total2, const int64_t *offsets2,  \
                        int64_t nframes, int64_t max_frame1, int64_t max_frame2, int iou_type, int out_dtype, void *max1, int64_t *idx1,      \
                        void *max2, int64_t *idx2, void *ws, size_t wsb, void *stream)                                                     \
    {                                                                                                                                  \
        return iou_max_batch_impl<T>(boxes1, total1, offsets1, boxes2, total2, offsets2, nframes, max_frame1, max_frame2, iou_type,    \
                                     out_dtype, max1, idx1, max2, idx2, ws, wsb, (cudaStream_t)stream);                                \
    }
D3D_IOU_MAX_BATCH_ENTRY(d3d_box2d_iou_max_batch_f32, float)
D3D_IOU_MAX_BATCH_ENTRY(d3d_box2d_iou_max_batch_f64, double)
extern "C" int d3d_iou_count_candidates(const void *b1, int64_t n, const void *b2, int64_t m, int dtype, uint64_t *counters64, void *ws, size_t wsb, void *stream)
{
    return dtype == D3D_F64 ? count_cand_impl<double>((const double *)b1, n, (const double *)b2, m, (unsigned long long *)counters64, ws, wsb, (cudaStream_t)stream)
                            : count_cand_impl<float>((const float *)b1, n, (const float *)b2, m, (unsigned long long *)counters64, ws, wsb, (cudaStream_t)stream);
}
