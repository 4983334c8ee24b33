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
template <typename T, int TILE>
__global__ void __launch_bounds__(256) box_prep_kernel(const T *__restrict__ boxes, int64_t n, int64_t npad, BoxRec<T> *__restrict__ recs)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npad) return;
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

template <typename T>
__global__ void __launch_bounds__(256) aabb_prep_kernel(const T *__restrict__ boxes, int64_t n, AABBRec<T> *__restrict__ recs)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const T *b = boxes + 5 * i;
    recs[i] = make_aabb_rec<T>(b[0], b[1], b[2], b[3], b[4]);
}

// ------------------------------------------------------------------ rotated IoU tile kernel
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
// The single-matrix kernel and the frame-batched kernel both run this body, so a pair gets the same reject test and clip in both.
template <typename T, bool ZD>
__device__ __forceinline__ void iou2dr_tile(const BoxRec<T> *__restrict__ recA, int64_t n, const BoxRec<T> *__restrict__ recB, int64_t m,
                                            T *__restrict__ out, int64_t ld, const ZRange *__restrict__ zA, const ZRange *__restrict__ zB,
                                            const int64_t row0, const int64_t col0)
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
template <typename T>
__global__ void __launch_bounds__(256) iou2d_kernel(const AABBRec<T> *__restrict__ recA, int64_t n, const AABBRec<T> *__restrict__ recB, int64_t m,
                                                    T *__restrict__ out, int64_t ld)
{
    const int64_t row = blockIdx.y;
    const int64_t c0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (row >= n || c0 >= m) return;
    const AABBRec<T> a = recA[row];
#pragma unroll
    for (int k = 0; k < 4; k++)
        if (c0 + k < m) out[row * ld + c0 + k] = aabb_iou<T>(a, recB[c0 + k]);
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
extern "C" int d3d_iou_count_candidates(const void *b1, int64_t n, const void *b2, int64_t m, int dtype, uint64_t *counters64, void *ws, size_t wsb, void *stream)
{
    return dtype == D3D_F64 ? count_cand_impl<double>((const double *)b1, n, (const double *)b2, m, (unsigned long long *)counters64, ws, wsb, (cudaStream_t)stream)
                            : count_cand_impl<float>((const float *)b1, n, (const float *)b2, m, (unsigned long long *)counters64, ws, wsb, (cudaStream_t)stream);
}
