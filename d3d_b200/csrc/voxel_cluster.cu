// voxel_cluster.cu -- voxelization fast path: one thread-block CLUSTER per frame, one persistent launch.
//
// Replaces the same reference functions as voxel.cu (voxelize_sparse + voxelize_filter and
// voxelize_3d_dense, d3d/voxel/voxelize.cpp:288-484 and :45-199) for the common configurations; voxel.cu's
// sort-based pipeline stays as the general fallback (DESCENDING filter, dense reductions, > 2^32 cells).
//
// Why a cluster per frame: frames are independent, a frame's working set (120k-200k points) is a few MB,
// and the reference's sequential semantics (voxel ids in order of first appearance, first max_points points
// of a voxel in input order) need frame-wide prefix sums.  A cluster of 8 CTAs x 1024 threads owns a frame
// from the first point load to the last output store: the phases are separated by cluster barriers
// (barrier.cluster, ~1 us) instead of kernel launches, prefix sums cross CTAs through distributed shared
// memory, and the whole scratch state of the frames in flight (hash table, per-point words) stays in L2, so
// HBM sees the algorithmic traffic only: 16 B/point in, 32 B/kept point + 28 B/voxel out.
//
// Determinism without a sort.  Everything that decides an output is an order-independent function of the
// point set, although the hash-table slots themselves are handed out in race order:
//   * a voxel's slot holds (cell key << 32 | smallest point index) maintained by atomicMin, and its point
//     count by atomicAdd -- commutative, so first[] and count[] are unique;
//   * voxel ids = exclusive prefix sum, in point order, of "this point is the first of a voxel that passes
//     the voxel filter" -- exactly the reference's first-appearance numbering;
//   * "first max_points points of a voxel" only needs order inside voxels that hold MORE than max_points
//     points (a few per cent): their point indices are appended to a per-voxel list (position = the value
//     atomicAdd returned, any order) and a point's rank is the number of smaller indices in that list, found
//     by a direct scan (<= 32 entries) or, for big voxels, by a warp that extracts the max_points smallest
//     indices one minimum at a time -- both independent of the list order;
//   * kept points are compacted with a second prefix sum in point order.
#include "voxel.cuh"
#include <cooperative_groups.h>
#include <stdio.h>
#include <stdlib.h>

namespace cg = cooperative_groups;

namespace d3d {

constexpr int VC_THREADS = 1024;
constexpr int VC_WARPS = VC_THREADS / 32;
constexpr int VC_MAX_CSIZE = 8;               // portable cluster sizes only
constexpr int VC_MAX_CLUSTERS = 74;            // frames in flight the workspace is sized for
constexpr uint32_t VC_NONE = 0xffffffffu;
constexpr unsigned long long VC_EMPTY = ~0ull;
// per-point word after P3: VC_NONE (dropped) | VC_SINGLE + provisional voxel id (the only point of its voxel: no
// further table access needed) | table slot
constexpr uint32_t VC_SINGLE = 1u << 31;
// list record of a crowded voxel: [0] provisional voxel id, [1] big voxels: keep indices below this, [2] fill cursor, [3..] point indices
constexpr int VC_LIST_HDR = 3;
constexpr int VC_LOCAL_BITS = 20;              // provisional voxel id = (warp << 20) | rank inside the warp's chunk

struct __align__(16) VcEntry {
    unsigned long long kf;   // (cell key << 32) | smallest frame-local index of a point in the cell
    uint32_t count;          // points in the cell beyond the one that claimed the slot (total - 1)
    uint32_t aux;            // crowded voxel: start of its list record; otherwise the provisional voxel id
};

struct VcLayout {            // byte offsets inside one cluster's workspace slice
    size_t tab, pw, pkey, cw, lists, prank, tq, ctr, total;
    uint32_t cap_slots;
};

static VcLayout vc_layout(int64_t lmax)
{
    VcLayout l;
    if (lmax < 1) lmax = 1;
    const size_t lp = (size_t)lmax + 64;
    l.cap_slots = (uint32_t)(lmax + lmax / 2 + 64);
    size_t o = 0;
    l.tab = o;   o += align_up((size_t)l.cap_slots * sizeof(VcEntry));
    l.pw = o;    o += align_up(lp * 4);
    l.pkey = o;  o += align_up(lp * 4);
    l.cw = o;    o += align_up(lp * 4);
    l.lists = o; o += align_up((3 * lp) * 4);   // sum over crowded voxels (>= 2 points) of count + 3 header words
    l.prank = o; o += align_up(lp * 4);
    l.tq = o;    o += align_up((lp / 2 + 64) * 4);   // crowded voxels hold >= 2 points
    l.ctr = o;   o += 256;
    l.total = o;
    return l;
}

struct VcArgs {
    const float *pts; int nfeat; const int64_t *offs; int64_t nframes;
    VoxCfg cfg;
    float *out_points; int64_t *out_mask; int64_t *out_mapping; int32_t *out_npoints; int64_t *out_coords; int64_t *counts;
    float *voxels; uint8_t *pmask;
    char *ws; VcLayout lay;
    unsigned long long *vstate, *kstate;   // sparse: cross-frame look-back words, one per frame (zeroed before the launch)
    uint32_t dyn_bytes;                    // dynamic shared memory of the launch
    uint32_t *ticket;                      // frames are handed out in index order to the clusters that are running (zeroed before the launch)
    uint32_t lmax;                         // hard upper bound of a frame's length: the scratch is sized for it, longer frames are cut
    const uint32_t *run_if;                // optional device flag: the launch does nothing when it is zero (fallback of the tile pipeline)
    int route;                             // sparse: try the shared-memory routed path first (vc_frame_route)
};

// per-CTA shared memory handed to the per-frame functions
struct VcSh {
    uint32_t *mytot, *mytot2, *wt1, *wt2, *vbase, *pbase;
    unsigned long long *frow;      // first voxel row / first kept-point row of this frame in the packed outputs
    uint2 *hbp;                    // routed path: first-of-voxel bits of every 32-point round (.x) and their exclusive prefix inside the warp's chunk (.y)
    uint32_t *list, *lcount;       // routed path: work list
    uint32_t *pool_min, *pool_acc0, *pool_acc1;   // routed path: records of the crowded voxels this CTA owns
    uint32_t *qcount, *npool, *bail;
    unsigned char *dyn;            // dynamic region: L2 path = per-warp probe rings; routed path = queue, slot table, reply words
};

__device__ __forceinline__ VcEntry vc_load_entry(const VcEntry *p)
{
    uint4 v = __ldcg(reinterpret_cast<const uint4 *>(p));   // L2 only: other CTAs of the cluster write these
    VcEntry e;
    e.kf = ((unsigned long long)v.y << 32) | v.x;
    e.count = v.z; e.aux = v.w;
    return e;
}

__device__ __forceinline__ float4 vc_load_point(const float *pts, int nfeat, int64_t i)
{
    if (nfeat == 4) return __ldg(reinterpret_cast<const float4 *>(pts) + i);
    const float *q = pts + i * nfeat;
    return make_float4(q[0], q[1], q[2], 0.f);
}

// Cross-frame decoupled look-back (sparse path): the outputs of all frames are packed back to back, so frame f
// starts at the sum of the row counts of frames < f.  Frames are processed in index order by co-resident
// clusters, every frame publishes its own count as soon as it knows it (flag 1) and its inclusive prefix once
// it has looked back (flag 2); a frame only ever waits for lower-numbered frames, which are running or done.
// The clusters run in step, so the nearest inclusive prefix is usually a whole wave of frames away: one warp
// reads 32 predecessors per round trip instead of walking them one acquire-load at a time.
__device__ __forceinline__ unsigned long long vc_lookback(unsigned long long *state, int64_t f, unsigned long long mine, bool publish)
{
    constexpr unsigned long long VAL = (1ull << 62) - 1;
    const unsigned lane = threadIdx.x & 31u;
    if (publish && f > 0 && lane == 0) asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(state + f), "l"((1ull << 62) | mine) : "memory");
    unsigned long long excl = 0;
    for (int64_t j = f - 1; j >= 0; j -= 32) {
        const int64_t idx = j - (int64_t)lane;
        unsigned long long v = 2ull << 62;   // before the first frame: an inclusive prefix of zero
        unsigned first2, need;
        for (;;) {
            if (idx >= 0) asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(state + idx) : "memory");
            const unsigned flag = (unsigned)(v >> 62);
            const unsigned b2 = __ballot_sync(0xffffffffu, flag == 2), b0 = __ballot_sync(0xffffffffu, flag == 0);
            first2 = b2 ? (unsigned)__ffs((int)b2) - 1u : 32u;                       // nearest predecessor that already knows its prefix
            need = first2 >= 31u ? 0xffffffffu : ((2u << first2) - 1u);          // it and every frame after it must have published
            if (!(b0 & need)) break;
            __nanosleep(64);
        }
        unsigned long long x = ((need >> lane) & 1u) ? (v & VAL) : 0ull;
#pragma unroll
        for (int d = 16; d; d >>= 1) x += __shfl_xor_sync(0xffffffffu, x, d);
        excl += x;
        if (first2 < 32u) break;
    }
    if (publish && lane == 0) asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(state + f), "l"((2ull << 62) | (excl + mine)) : "memory");
    return excl;
}

// exchange the per-warp totals of every CTA of the cluster through distributed shared memory and turn them
// into exclusive bases: base[v] = sum of totals of warps < v, base[W] = grand total
__device__ __forceinline__ void vc_exchange(cg::cluster_group &cluster, uint32_t *mytot, uint32_t *wt, uint32_t *base, unsigned csize, unsigned crank)
{
    const unsigned tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    __syncthreads();   // mytot[] complete
    for (unsigned t = tid; t < csize * VC_WARPS; t += VC_THREADS) {
        uint32_t *remote = cluster.map_shared_rank(wt, t / VC_WARPS);
        remote[crank * VC_WARPS + (t % VC_WARPS)] = mytot[t % VC_WARPS];
    }
    cluster.sync();
    if (w == 0) {      // lane l owns totals [l*csize, (l+1)*csize): W = 32*csize values in warp order
        uint32_t s = 0;
        for (unsigned j = 0; j < csize; j++) s += wt[lane * csize + j];
        uint32_t inc = s;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= (unsigned)d) inc += t; }
        uint32_t run = inc - s;
        for (unsigned j = 0; j < csize; j++) { base[lane * csize + j] = run; run += wt[lane * csize + j]; }
        if (lane == 31) base[csize * VC_WARPS] = run;
    }
    __syncthreads();
}

// both prefix sums of a frame (voxel rows, kept-point rows) behind ONE cluster barrier, for configurations whose keep
// decision does not depend on the voxel id; warp 0 / warp 1 scan and look back concurrently
__device__ __forceinline__ void vc_exchange2(cg::cluster_group &cluster, const uint32_t *mytot1, const uint32_t *mytot2, uint32_t *wt1, uint32_t *wt2,
                                             uint32_t *base1, uint32_t *base2, unsigned csize, unsigned crank)
{
    const unsigned tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const unsigned nw = csize * VC_WARPS;
    __syncthreads();   // mytot1[], mytot2[] complete
    for (unsigned t = tid; t < 2 * nw; t += VC_THREADS) {
        const bool second = t >= nw;
        const unsigned tt = second ? t - nw : t;
        uint32_t *remote = cluster.map_shared_rank(second ? wt2 : wt1, tt / VC_WARPS);
        remote[crank * VC_WARPS + (tt % VC_WARPS)] = (second ? mytot2 : mytot1)[tt % VC_WARPS];
    }
    cluster.sync();
    if (w < 2) {
        const uint32_t *wt = w ? wt2 : wt1;
        uint32_t *base = w ? base2 : base1;
        uint32_t s = 0;
        for (unsigned j = 0; j < csize; j++) s += wt[lane * csize + j];
        uint32_t inc = s;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= (unsigned)d) inc += t; }
        uint32_t run = inc - s;
        for (unsigned j = 0; j < csize; j++) { base[lane * csize + j] = run; run += wt[lane * csize + j]; }
        if (lane == 31) base[nw] = run;
        __syncwarp();
    }
}

#ifndef D3D_VC_U
#define D3D_VC_U 2
#endif
constexpr int VC_U = D3D_VC_U;     // points per thread in flight in the streaming phases: independent loads are issued back to back
constexpr int VC_QCAP = 128;       // per-warp ring of points waiting for their next hash probe

#ifdef D3D_VC_TIMING   // tuning build only: per-phase time of a few frames, printed once per frame
#define VC_TICK(slot) do { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); tk_[slot] = (float)(t_ - t0_) * 1e-3f; t0_ = t_; } while (0)
#define VC_TICK_INIT float tk_[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}; unsigned long long t0_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0_));
#define VC_TICK_PRINT do { if (crank == 0 && tid == 0 && (cid == 0 || cid == ncl - 1) && f < 2 * (int64_t)ncl) \
    printf("frame %3d cl %2u  clear %6.1f insert %6.1f flags %6.1f join %6.1f big %6.1f ids %6.1f compact %6.1f us\n", (int)f, cid, tk_[0], tk_[1], tk_[2], tk_[3], tk_[4], tk_[5], tk_[6]); } while (0)
#else
#define VC_TICK(slot)
#define VC_TICK_INIT
#define VC_TICK_PRINT
#endif

// ---------------------------------------------------------------------------------------------------------
// L2 path: the frame's hash table and per-point words live in the cluster's workspace slice (L2-resident),
// inserts are 64-bit CAS / atomicMin / RED on global memory.  Handles every supported configuration and
// frame size; the routed path below falls back to it.
template <bool DENSE>
__device__ __forceinline__ void vc_frame_l2(const VcArgs &a, const VcDev &dv, const VcSh &sh, cg::cluster_group &cluster, const int64_t f,
                                            const unsigned cid, const unsigned ncl)
{
    const unsigned csize = cluster.num_blocks(), crank = cluster.block_rank();
    const unsigned tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const unsigned W = csize * VC_WARPS, g = crank * VC_WARPS + w;     // warps per cluster, index of this warp
    const unsigned CT = csize * VC_THREADS, ct = crank * VC_THREADS + tid;
    const unsigned ltmask = lanemask_lt();
    (void)ncl;

    uint32_t *mytot = sh.mytot, *wt1 = sh.wt1, *wt2 = sh.wt2, *vbase = sh.vbase, *pbase = sh.pbase;
    unsigned long long *frow = sh.frow;
    uint32_t *q_key = reinterpret_cast<uint32_t *>(sh.dyn), *q_pt = q_key + VC_WARPS * VC_QCAP;   // insert queue: cell key, (point index << 5 | probe number)

    char *slice = a.ws + (size_t)cid * a.lay.total;
    VcEntry *tab = reinterpret_cast<VcEntry *>(slice + a.lay.tab);
    uint32_t *pw = reinterpret_cast<uint32_t *>(slice + a.lay.pw);
    uint32_t *pkey = reinterpret_cast<uint32_t *>(slice + a.lay.pkey);
    uint32_t *cw = reinterpret_cast<uint32_t *>(slice + a.lay.cw);
    uint32_t *lists = reinterpret_cast<uint32_t *>(slice + a.lay.lists);
    uint32_t *prank = reinterpret_cast<uint32_t *>(slice + a.lay.prank);
    uint32_t *tq = reinterpret_cast<uint32_t *>(slice + a.lay.tq);
    uint32_t *ctr = reinterpret_cast<uint32_t *>(slice + a.lay.ctr);   // [1] list cursor, [2] crowded voxels queued for ranking

    const VoxCfg &cfg = a.cfg;
    const uint32_t K = cfg.max_points > 0 ? (uint32_t)cfg.max_points : 0u;
    const bool trim = DENSE || cfg.pfilter == D3D_PF_TRIM;
    const bool dropall = !DENSE && trim && K == 0;                       // sparse TRIM with max_points 0 keeps no point
    const uint32_t cthr = DENSE ? 1u : ((trim && K > 0) ? K : VC_NONE);  // voxels with more points than this need ranks
    const uint32_t vcap = (DENSE || cfg.vfilter != D3D_VF_NONE) ? (cfg.max_voxels > 0 ? (uint32_t)cfg.max_voxels : 0u) : VC_NONE;
    const int nfeat = a.nfeat;

    {
        const int64_t b = a.offs[f];
        const uint32_t L = (uint32_t)min((long long)(a.offs[f + 1] - b), (long long)a.lmax);
        const uint32_t nslots = L + (L >> 1) + 64;
        const uint32_t nit = (L + W * 32 - 1) / (W * 32);   // 32-point rounds per warp
        const uint32_t wbeg = g * nit * 32;                 // this warp owns points [wbeg, wbeg + nit*32)

        VC_TICK_INIT
        // ---- P0: clear the table; cell key of every point (the reference's fp32 arithmetic), streamed with VC_U loads in flight
        for (uint32_t s = ct; s < nslots; s += CT)
            *reinterpret_cast<uint4 *>(tab + s) = make_uint4(0xffffffffu, 0xffffffffu, 0u, VC_NONE);
        if (ct < 16) ctr[ct] = 0;
        for (uint32_t k0 = 0; k0 < nit; k0 += VC_U) {
            float4 p[VC_U];
            uint32_t idx[VC_U];
            bool in[VC_U];
#pragma unroll
            for (int u = 0; u < VC_U; u++) {
                idx[u] = wbeg + (k0 + u) * 32 + lane;
                in[u] = k0 + u < nit && idx[u] < L;
                p[u] = in[u] ? vc_load_point(a.pts, nfeat, b + idx[u]) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < VC_U; u++) {
                uint32_t key;
                const bool ok = vc_cell<DENSE>(dv, p[u], &key);
                if (in[u]) pkey[idx[u]] = ok ? key : VC_NOKEY;
            }
        }
        cluster.sync();
        VC_TICK(0);

        // ---- P1: hash insert (smallest point index wins), points that join an existing voxel count themselves.
        // One probe = one atomic round trip to L2, and a lane may need several.  Instead of letting 31 lanes wait for
        // the unluckiest one, points wait in a per-warp shared-memory ring between probes and every CAS instruction
        // is issued for 32 queued points (the same compaction the IoU kernel uses for its candidate pairs).
        {
            uint32_t *qk = q_key + w * VC_QCAP, *qp = q_pt + w * VC_QCAP;
            uint32_t head = 0, tail = 0;   // warp-uniform
            for (uint32_t k = 0; k <= nit; k++) {
                if (k < nit) {
                    const uint32_t i = wbeg + k * 32 + lane;
                    const uint32_t key = i < L ? pkey[i] : VC_NOKEY;
                    const bool ok = key != VC_NOKEY;
                    const unsigned bal = __ballot_sync(0xffffffffu, ok);
                    if (ok) { const uint32_t t = (tail + __popc(bal & ltmask)) & (VC_QCAP - 1); qk[t] = key; qp[t] = i << 5; }
                    else if (i < L) pw[i] = VC_NONE;
                    tail += __popc(bal);
                }
                while (tail - head >= 32u || (k == nit && tail != head)) {
                    __syncwarp();
                    const uint32_t cnt = min(tail - head, 32u);
                    const bool act = lane < cnt;
                    const uint32_t t = (head + lane) & (VC_QCAP - 1);
                    const uint32_t key = act ? qk[t] : 0u, pt = act ? qp[t] : 0u;
                    head += cnt;
                    const uint32_t i = pt >> 5, probe = pt & 31u;
                    uint32_t s = __umulhi(key * 0x9E3779B1u, nslots) + probe;
                    if (s >= nslots) s -= nslots;
                    bool again = false;
                    if (act) {
                        const unsigned long long mine = ((unsigned long long)key << 32) | i;
                        unsigned long long c = atomicCAS(&tab[s].kf, VC_EMPTY, mine);
                        if (probe == 31u) {   // out of probe-counter bits (never seen in practice): finish this point in place
                            while (c != VC_EMPTY && (uint32_t)(c >> 32) != key) {
                                if (++s == nslots) s = 0;
                                c = atomicCAS(&tab[s].kf, VC_EMPTY, mine);
                            }
                        }
                        if (c == VC_EMPTY) {
                            pw[i] = s;                                              // claimed an empty slot
                        } else if ((uint32_t)(c >> 32) == key) {
                            if (i < (uint32_t)c) atomicMin(&tab[s].kf, mine);       // results unused: REDs
                            atomicAdd(&tab[s].count, 1u);
                            pw[i] = s;
                        } else {
                            again = true;                                           // another voxel's slot: probe the next one later
                        }
                    }
                    __syncwarp();
                    const unsigned bal = __ballot_sync(0xffffffffu, again);
                    if (again) { const uint32_t t2 = (tail + __popc(bal & ltmask)) & (VC_QCAP - 1); qk[t2] = key; qp[t2] = pt + 1; }
                    tail += __popc(bal);
                }
            }
        }
        cluster.sync();
        VC_TICK(1);

        // ---- P3: first-of-voxel flags -> provisional voxel ids (rank inside the warp's chunk).  The first point of a
        // crowded voxel reserves the voxel's list record and queues the voxel for ranking; the points of crowded
        // voxels are compacted into cw[] so that the next phase touches only them.
        uint32_t ncw = 0;   // crowded points of this warp's chunk (warp-uniform, lives across the barriers)
        {
            uint32_t carry = 0;
            for (uint32_t k0 = 0; k0 < nit; k0 += VC_U) {
                uint32_t idx[VC_U], s[VC_U];
                VcEntry e[VC_U];
#pragma unroll
                for (int u = 0; u < VC_U; u++) {
                    idx[u] = wbeg + (k0 + u) * 32 + lane;
                    s[u] = (k0 + u < nit && idx[u] < L) ? pw[idx[u]] : VC_NONE;
                }
#pragma unroll
                for (int u = 0; u < VC_U; u++)
                    if (s[u] != VC_NONE) e[u] = vc_load_entry(tab + s[u]);
#pragma unroll
                for (int u = 0; u < VC_U; u++) {
                    bool f1 = false, first = false, crowded = false, single = false;
                    uint32_t total = 0;
                    if (s[u] != VC_NONE) {
                        total = e[u].count + 1;
                        single = e[u].count == 0;
                        crowded = total > cthr;
                        first = (uint32_t)e[u].kf == idx[u];
                        f1 = first && (DENSE || (long long)total >= (long long)cfg.min_points);
                    }
                    const unsigned bal = __ballot_sync(0xffffffffu, f1), balc = __ballot_sync(0xffffffffu, crowded);
                    const uint32_t prov = f1 ? ((g << VC_LOCAL_BITS) | (carry + __popc(bal & ltmask))) : VC_NONE;
                    if (s[u] != VC_NONE) {
                        if (crowded) {
                            cw[wbeg + ncw + __popc(balc & ltmask)] = idx[u];
                            if (first) {
                                const uint32_t base = atomicAdd(&ctr[1], total + VC_LIST_HDR);
                                lists[base] = prov; lists[base + 1] = 0; lists[base + 2] = 0;
                                tab[s[u]].aux = base;
                                tq[atomicAdd(&ctr[2], 1u)] = s[u];
                            }
                        } else if (single) {
                            pw[idx[u]] = f1 ? (VC_SINGLE | prov) : VC_NONE;     // everything later phases need is in this word
                        } else if (f1) {
                            tab[s[u]].aux = prov;
                        }
                    }
                    carry += __popc(bal);
                    ncw += __popc(balc);
                }
            }
            if (lane == 0) mytot[w] = carry;
            vc_exchange(cluster, mytot, wt1, vbase, csize, crank);
            if (!DENSE) {
                if (w == 0) { const unsigned long long x = vc_lookback(a.vstate, f, min(vbase[W], vcap), crank == 0); if (lane == 0) frow[0] = x; }
                __syncthreads();
            }
        }
        VC_TICK(2);

        const uint32_t ntask = __ldcg(&ctr[2]);   // cluster-uniform
        if (ntask) {
            // ---- P3b: points of crowded voxels join their voxel's list (any order)
            for (uint32_t j0 = 0; j0 < ncw; j0 += 32) {
                const uint32_t j = j0 + lane;
                if (j < ncw) {
                    const uint32_t i = cw[wbeg + j];
                    const uint32_t base = __ldcg(&tab[pw[i]].aux);
                    lists[base + VC_LIST_HDR + atomicAdd(&lists[base + 2], 1u)] = i;
                }
            }
            cluster.sync();
            VC_TICK(3);

            // ---- P4: one warp per crowded voxel ranks its points by index (the list order is arbitrary, the ranks are not)
            for (uint32_t q = g; q < ntask; q += W) {
                const uint32_t s = __ldcg(&tq[q]);
                const VcEntry e = vc_load_entry(tab + s);
                const uint32_t *lst = lists + e.aux + VC_LIST_HDR;
                const uint32_t total = e.count + 1;
                if (total <= 32u) {   // one index per lane: rank = number of smaller indices
                    const uint32_t x = lane < total ? __ldcg(lst + lane) : VC_NONE;
                    uint32_t r = 0;
                    for (uint32_t l = 0; l < total; l++) r += __shfl_sync(0xffffffffu, x, l) < x ? 1u : 0u;
                    if (lane < total) prank[x] = r;
                } else {              // extract the K smallest indices, one minimum per sweep; the rest is dropped by the bound
                    uint32_t lb = 0;
                    for (uint32_t r = 0; r < K; r++) {
                        uint32_t m = VC_NONE;
                        for (uint32_t j = lane; j < total; j += 32) {
                            const uint32_t x = __ldcg(lst + j);
                            if (x >= lb && x < m) m = x;
                        }
#pragma unroll
                        for (int d = 16; d; d >>= 1) m = min(m, __shfl_xor_sync(0xffffffffu, m, d));
                        if (m == VC_NONE) break;
                        if (lane == 0) prank[m] = r;
                        lb = m + 1;
                    }
                    if (lane == 0) lists[e.aux + 1] = lb;
                }
            }
            cluster.sync();
            VC_TICK(4);
        }

        // ---- P5: final voxel ids, per-voxel outputs, point keep decisions
        {
            uint32_t carry = 0;
            const uint32_t mask_y = (1u << (dv.sh_x - dv.sh_y)) - 1, mask_z = (1u << dv.sh_y) - 1;
            for (uint32_t k0 = 0; k0 < nit; k0 += VC_U) {
                uint32_t idx[VC_U], s[VC_U], prov[VC_U], ckey[VC_U];
                VcEntry e[VC_U];
                bool single[VC_U];
#pragma unroll
                for (int u = 0; u < VC_U; u++) {
                    idx[u] = wbeg + (k0 + u) * 32 + lane;
                    s[u] = (k0 + u < nit && idx[u] < L) ? pw[idx[u]] : VC_NONE;
                    single[u] = s[u] != VC_NONE && (s[u] & VC_SINGLE);
                }
#pragma unroll
                for (int u = 0; u < VC_U; u++) {
                    if (single[u]) ckey[u] = pkey[idx[u]];                      // coalesced: the voxel's row is written from here
                    else if (s[u] != VC_NONE) e[u] = vc_load_entry(tab + s[u]);
                }
#pragma unroll
                for (int u = 0; u < VC_U; u++) {
                    if (single[u]) prov[u] = s[u] & ~VC_SINGLE;
                    else if (s[u] != VC_NONE) prov[u] = e[u].count + 1 > cthr ? __ldcg(&lists[e[u].aux]) : e[u].aux;
                }
#pragma unroll
                for (int u = 0; u < VC_U; u++) {
                    const uint32_t i = idx[u];
                    bool keep = false;
                    uint32_t nid = VC_NONE, rank = 0;
                    if (s[u] != VC_NONE) {
                        const uint32_t c = single[u] ? 1u : e[u].count + 1;
                        const bool crowded = !single[u] && c > cthr;
                        const bool first = single[u] || (uint32_t)e[u].kf == i;
                        if (prov[u] != VC_NONE) {
                            nid = vbase[prov[u] >> VC_LOCAL_BITS] + (prov[u] & ((1u << VC_LOCAL_BITS) - 1));
                            if (nid >= vcap) nid = VC_NONE;
                        }
                        keep = nid != VC_NONE;
                        if (keep && crowded) {
                            if (c > 32u) keep = i < __ldcg(&lists[e[u].aux + 1]);   // big voxel: only the K smallest indices have a rank
                            if (keep) { rank = __ldcg(&prank[i]); keep = rank < K; }
                        }
                        if (DENSE) keep = keep && rank < K;
                        if (dropall) keep = false;
                        if (nid != VC_NONE && first) {   // first point of a kept voxel writes the voxel's row
                            const uint32_t key = single[u] ? ckey[u] : (uint32_t)(e[u].kf >> 32);
                            const int64_t o = DENSE ? f * (int64_t)cfg.max_voxels + nid : (int64_t)frow[0] + nid;
                            long long *co = reinterpret_cast<long long *>(a.out_coords) + o * 3;
                            __stcs(co + 0, (long long)(key >> dv.sh_x) + dv.cadd[0]);
                            __stcs(co + 1, (long long)((key >> dv.sh_y) & mask_y) + dv.cadd[1]);
                            __stcs(co + 2, (long long)(key & mask_z) + dv.cadd[2]);
                            __stcs(a.out_npoints + o, (!DENSE && cfg.pfilter == D3D_PF_TRIM && c > K) ? (int32_t)K : (int32_t)c);
                        }
                        if (DENSE && keep) {
                            const int64_t slot = (f * (int64_t)cfg.max_voxels + nid) * (int64_t)K + rank;
                            if (nfeat == 4) __stcs(reinterpret_cast<float4 *>(a.voxels) + slot, vc_load_point(a.pts, 4, b + i));
                            else for (int q = 0; q < nfeat; q++) a.voxels[slot * nfeat + q] = a.pts[(b + i) * nfeat + q];
                            a.pmask[slot] = 1;
                        }
                    }
                    if (!DENSE) {
                        if (k0 + u < nit && i < L) pw[i] = keep ? nid : VC_NONE;
                        carry += __popc(__ballot_sync(0xffffffffu, keep));
                    }
                }
            }
            if (DENSE) {
                if (ct == 0) { a.counts[2 * f] = 0; a.counts[2 * f + 1] = (long long)min(vbase[W], vcap); }
                cluster.sync();   // the next frame clears the table other CTAs may still be reading
                return;
            }
            if (lane == 0) mytot[w] = carry;
            vc_exchange(cluster, mytot, wt2, pbase, csize, crank);
            if (w == 0) { const unsigned long long x = vc_lookback(a.kstate, f, pbase[W], crank == 0); if (lane == 0) frow[1] = x; }
            __syncthreads();
        }
        VC_TICK(5);

        // ---- P6: compaction of the kept points, in input order
        {
            int64_t run = (int64_t)frow[1] + pbase[g];
            for (uint32_t k0 = 0; k0 < nit; k0 += VC_U) {
                uint32_t idx[VC_U], nid[VC_U];
                float4 p[VC_U];
#pragma unroll
                for (int u = 0; u < VC_U; u++) {
                    idx[u] = wbeg + (k0 + u) * 32 + lane;
                    nid[u] = (k0 + u < nit && idx[u] < L) ? pw[idx[u]] : VC_NONE;
                }
                if (nfeat == 4) {
#pragma unroll
                    for (int u = 0; u < VC_U; u++)
                        if (nid[u] != VC_NONE) p[u] = vc_load_point(a.pts, 4, b + idx[u]);
                }
#pragma unroll
                for (int u = 0; u < VC_U; u++) {
                    const bool keep = nid[u] != VC_NONE;
                    const unsigned bal = __ballot_sync(0xffffffffu, keep);
                    if (keep) {
                        const int64_t o = run + __popc(bal & ltmask);
                        if (nfeat == 4) __stcs(reinterpret_cast<float4 *>(a.out_points) + o, p[u]);
                        else for (int q = 0; q < nfeat; q++) a.out_points[o * nfeat + q] = a.pts[(b + idx[u]) * nfeat + q];
                        __stcs(reinterpret_cast<long long *>(a.out_mask) + o, (long long)idx[u]);
                        __stcs(reinterpret_cast<long long *>(a.out_mapping) + o, (long long)nid[u]);
                    }
                    run += __popc(bal);
                }
            }
            if (ct == 0) {   // frame_rows[f] = {first kept-point row, first voxel row}; the last frame also writes the totals
                a.counts[2 * f] = (long long)frow[1]; a.counts[2 * f + 1] = (long long)frow[0];
                if (f == a.nframes - 1) { a.counts[2 * f + 2] = (long long)(frow[1] + pbase[W]); a.counts[2 * f + 3] = (long long)(frow[0] + min(vbase[W], vcap)); }
            }
        }
        VC_TICK(6); VC_TICK_PRINT;
    }
}

// ---------------------------------------------------------------------------------------------------------
// Routed path (sparse): the frame never leaves the cluster's shared memory between the point load and the
// output stores, and no global atomic is issued.
//
// Every CTA plays two roles.  As POINT OWNER it holds a contiguous range of the frame's points (the same
// warp-chunk layout as the L2 path); as HASH OWNER it holds every point of the frame whose cell key hashes to
// it, so all points of one voxel meet in one CTA.
//   R1 push     point owners compute the cell keys (kept in registers) and append (key, index) to the hash
//               owner's queue through distributed shared memory; a warp reserves its exact share of every
//               queue with one remote atomicAdd per destination (8 per warp and frame).
//   R2 resolve  hash owners find one slot per distinct key in a shared-memory table WITHOUT atomics: in
//               round r every unresolved entry sits at probe position r of its key's double-hash sequence,
//               writes its queue position into the slot if it is empty (plain store, any writer wins),
//               and after a CTA barrier adopts the slot if the winner carries its key.  Entries of one key
//               move in lock step, so they agree on the slot and on the winner; a slot never changes once
//               it is filled.  Plain shared-memory loads/stores run at ~10 lanes/clk against 0.5 lanes/clk
//               for shared-memory atomics, which only the ~8 % of points that join an existing voxel issue
//               (atomicMin of the index, atomicAdd of the count on the winner's queue words).
//   R3 ranks    voxels with more than max_points points extract their max_points smallest indices, one
//               minimum per round (atomicMin on a per-voxel accumulator; the round number sits in the high
//               bits so a later round always wins and nothing is reset).
//   R4 reply    hash owners send every point one word back to its point owner: dropped | first point of its
//               voxel + the voxel's point count | index of the voxel's first point, plus the keep decision.
//   R5 ids      point owners turn the first-of-voxel bits into voxel ids (ballot/popc, DSMEM exchange of the
//               warp totals, cross-frame look-back); a point that is not the first of its voxel reads the id
//               at its first point's position (DSMEM when that lives in another CTA).
//   R6 write    second prefix sum over the keep flags, then coalesced stores of the voxel rows (coordinates
//               recomputed from the reloaded point, L2 hit) and of the packed point rows.
// Results are identical to the L2 path and to the reference: every decision is a function of the point set
// (smallest index, count, K smallest indices), never of the race order.
// The frame falls back to the L2 path (cluster-uniform decision, nothing published yet) when it does not fit:
// more than VR_NIT 32-point rounds per warp, a queue overflow (skewed hash or > ~85 % of a 120k-point frame in
// bounds), or more crowded voxels per CTA than the pool holds.
constexpr int VR_NIT = 16;                       // 32-point rounds per warp (cell keys live in registers during R1)
constexpr int VR_E = 13;                         // queue entries per hash-owner thread
constexpr int VR_POOL = 512;                     // crowded-voxel records per CTA
constexpr uint32_t VR_HEAD = 1u << 31, VR_KEEP = 1u << 30, VR_VAL = (1u << 30) - 1;   // reply word
constexpr uint32_t VR_IDX_BITS = 18, VR_IDX_MASK = (1u << VR_IDX_BITS) - 1;          // frame-local point index in packed words
constexpr uint32_t VR_SLOT_EMPTY = 0xffffu;
constexpr int VR_LIST = 2048;                    // work list: entries still probing (R2) / competing for a rank (R3)
constexpr uint32_t VR_LOSER = 1u << 31;          // key word of a resolved entry that is not its voxel's winner (cell keys use <= 31 bits)
constexpr uint32_t VR_KEPT = 1u << 31;           // index word: this entry of a crowded voxel is one of the K smallest

constexpr uint32_t VR_STAGE = VC_WARPS * 96 * 8;   // bytes: 32 voxel rows x 3 coordinates x 8 B per warp
struct VrPlan { uint32_t nit, Lc, lg, nslots, cap; };

// shared-memory budget of one frame: reply words 4*Lc, slot table 2*nslots (power of two), queue 8*cap
__host__ __device__ inline bool vr_plan(uint32_t L, uint32_t csize, uint32_t dyn, VrPlan *pl)
{
    if (csize < 1 || csize > (uint32_t)VC_MAX_CSIZE || L == 0) return false;
    const uint32_t W = csize * VC_WARPS;
    const uint32_t nit = (L + W * 32 - 1) / (W * 32);
    if (nit > (uint32_t)VR_NIT || (uint64_t)nit * W * 32 > (1u << VR_IDX_BITS)) return false;
    const uint32_t Lc = nit * VC_THREADS;
    if (dyn < 4 * Lc + 4096) return false;
    const uint32_t R = dyn - 4 * Lc;
    uint32_t best = 0, blg = 0;
    for (uint32_t lg = 10; lg <= 16; lg++) {
        const uint32_t ns = 1u << lg;
        const uint32_t sb = 2 * ns > VR_STAGE ? 2 * ns : VR_STAGE;   // the idle slot table doubles as R6's coordinate staging
        if (sb + 1024 > R) break;
        uint32_t c = (R - sb) / 8;
        if (c > ns - ns / 4) c = ns - ns / 4;                 // load factor <= 0.75
        if (c > (uint32_t)VR_E * VC_THREADS) c = VR_E * VC_THREADS;
        if (c > 0xfff0u) c = 0xfff0u;                         // 16-bit queue positions in the slot table
        c &= ~3u;
        if (c > best) { best = c; blg = lg; }
    }
    if ((uint64_t)best * 10 < (uint64_t)Lc * 6) return false;   // would overflow on ordinary frames: not worth the attempt
    pl->nit = nit; pl->Lc = Lc; pl->lg = blg; pl->nslots = 1u << blg; pl->cap = best;
    return true;
}

// One multiply serves both levels: the hash owner comes from the top of key * phi (umulhi with the cluster size),
// the first slot from the bits below; the probe step (odd, so it visits every slot of the power-of-two table)
// comes from a second multiply that only entries needing a second probe pay for.
__device__ __forceinline__ uint32_t vr_h1(uint32_t key) { return key * 0x9E3779B1u; }
__device__ __forceinline__ uint32_t vr_step(uint32_t key, uint32_t smask) { return (((key * 0x85EBCA6Bu) >> 15) | 1u) & smask; }

// every lane asks for cnt consecutive list positions: one shared-memory atomic per warp instead of one per thread
// (same-address atomics with a result serialise)
__device__ __forceinline__ uint32_t vr_reserve(uint32_t *counter, uint32_t cnt, unsigned lane)
{
    uint32_t inc = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= (unsigned)d) inc += t; }
    const uint32_t tot = __shfl_sync(0xffffffffu, inc, 31);
    uint32_t base = 0;
    if (lane == 31 && tot) base = atomicAdd(counter, tot);
    return __shfl_sync(0xffffffffu, base, 31) + inc - cnt;
}

#ifdef D3D_VC_TIMING
#define VR_SUB(slot) do { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); tk_[slot] = (float)(t_ - t0_) * 1e-3f; } while (0)
#else
#define VR_SUB(slot)
#endif
#ifdef D3D_VC_TIMING
#define VR_TICK_PRINT do { if (crank == 0 && tid == 0 && (cid == 0 || cid == ncl - 1) && f < 2 * (int64_t)ncl) \
    printf("frame %3d cl %2u  push %6.1f resolve %6.1f (r0 %.1f r1 %.1f rounds %.1f [handoff %.1f] fix %.1f) ranks %6.1f reply %6.1f heads %6.1f ids %6.1f write %6.1f us  (n %u)\n", (int)f, cid, tk_[0], tk_[1], tk_[8], tk_[9], tk_[10], tk_[12], tk_[11], tk_[2], tk_[3], tk_[4], tk_[5], tk_[6], n); } while (0)
#else
#define VR_TICK_PRINT
#endif

// returns false (cluster-uniform) when the frame has to be redone by the L2 path
__device__ __forceinline__ bool vc_frame_route(const VcArgs &a, const VcDev &dv, const VcSh &sh, cg::cluster_group &cluster, const int64_t f,
                                               const VrPlan &pl, const unsigned cid, const unsigned ncl)
{
    const unsigned csize = cluster.num_blocks(), crank = cluster.block_rank();
    const unsigned tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const unsigned W = csize * VC_WARPS, g = crank * VC_WARPS + w;
    const unsigned ltmask = lanemask_lt();
    (void)cid; (void)ncl;

    const VoxCfg &cfg = a.cfg;
    const uint32_t K = cfg.max_points > 0 ? (uint32_t)cfg.max_points : 0u;
    const bool trim = cfg.pfilter == D3D_PF_TRIM;
    const bool dropall = trim && K == 0;
    const uint32_t cthr = (trim && K > 0) ? K : VC_NONE;
    const uint32_t vcap = cfg.vfilter != D3D_VF_NONE ? (cfg.max_voxels > 0 ? (uint32_t)cfg.max_voxels : 0u) : VC_NONE;
    const float4 *pts4 = reinterpret_cast<const float4 *>(a.pts) + a.offs[f];   // the routed path serves xyz+1 clouds (nfeat == 4)

    const uint32_t L = (uint32_t)min((long long)(a.offs[f + 1] - a.offs[f]), (long long)a.lmax);
    const uint32_t nit = pl.nit, Lc = pl.Lc, cap = pl.cap, nslots = pl.nslots, smask = pl.nslots - 1, hshift = 32 - pl.lg;
    const uint32_t wbeg = g * nit * 32;        // frame-local index of this warp's first point
    const uint32_t lbeg = w * nit * 32;        // the same inside the CTA's range
    const uint32_t magic = 65536u / nit + 1;   // x / nit == (x * magic) >> 16 for x < 4096

    uint2 *q = reinterpret_cast<uint2 *>(sh.dyn);               // queue entry: .x cell key, .y point index.  After R2: winner .x = own index | joiners << 18,
                                                                // winner .y = smallest index of the voxel (crowded voxel: its pool record), loser .x = VR_LOSER | winner
    uint32_t *reply = reinterpret_cast<uint32_t *>(q + cap);    // one word per point of this CTA's range
    uint16_t *slot = reinterpret_cast<uint16_t *>(reply + Lc);  // queue position of the entry that claimed the slot
    uint2 *hbp = sh.hbp;
    uint32_t *list = sh.list;
    volatile uint32_t *vqcount = sh.qcount, *vbail = sh.bail, *vlcount = sh.lcount;

    VC_TICK_INIT
    // ---- R1: clear the slot table; keys; push to the hash owners
    for (uint32_t s4 = tid; s4 < nslots / 8; s4 += VC_THREADS) reinterpret_cast<uint4 *>(slot)[s4] = make_uint4(~0u, ~0u, ~0u, ~0u);
    {
        // a point that hears nothing back is the only point of its voxel
        const uint32_t dflt = cfg.min_points <= 1 ? (VR_HEAD | VR_KEEP | 1u) : VC_NONE;
        uint32_t keys[VR_NIT];
        unsigned long long c0 = 0, c1 = 0;   // 16-bit fields: this thread's points per destination CTA (0-3 | 4-7)
#pragma unroll
        for (int k0 = 0; k0 < VR_NIT; k0 += 4) {
            float4 p[4];
            bool in[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const uint32_t i = wbeg + (k0 + u) * 32 + lane;
                in[u] = (uint32_t)(k0 + u) < nit && i < L;
                p[u] = in[u] ? __ldg(pts4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                uint32_t key;
                const bool ok = vc_cell<false>(dv, p[u], &key) && in[u];
                keys[k0 + u] = ok ? key : VC_NOKEY;
                if (in[u]) reply[lbeg + (k0 + u) * 32 + lane] = ok ? dflt : VC_NONE;
                if (ok) {
                    const uint32_t own = __umulhi(vr_h1(key), csize);
                    const unsigned long long inc = 1ull << ((own & 3u) * 16u);
                    if (own & 4u) c1 += inc; else c0 += inc;
                }
            }
        }
        unsigned long long i0 = c0, i1 = c1;   // inclusive prefix over the lanes
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long t0 = __shfl_up_sync(0xffffffffu, i0, d), t1 = __shfl_up_sync(0xffffffffu, i1, d);
            if (lane >= (unsigned)d) { i0 += t0; i1 += t1; }
        }
        const unsigned long long tot0 = __shfl_sync(0xffffffffu, i0, 31), tot1 = __shfl_sync(0xffffffffu, i1, 31);
        uint32_t base = 0;
        if (lane < csize) {   // lane d reserves the warp's share of CTA d's queue
            const uint32_t mycnt = (uint32_t)(((lane & 4u) ? tot1 : tot0) >> ((lane & 3u) * 16u)) & 0xffffu;
            if (mycnt) {
                base = atomicAdd(cluster.map_shared_rank(sh.qcount, lane), mycnt);
                if (base + mycnt > cap)   // the destination queue is full: every CTA of the cluster learns it before the barrier
                    for (unsigned d = 0; d < csize; d++) *cluster.map_shared_rank(sh.bail, d) = 1u;
            }
        }
        unsigned long long s0 = i0 - c0, s1 = i1 - c1;   // next queue position per destination (garbage, but bounded, after an overflow)
#pragma unroll
        for (int d = 0; d < 4; d++) {
            s0 += (unsigned long long)(__shfl_sync(0xffffffffu, base, d) & 0xffffu) << (16 * d);
            s1 += (unsigned long long)(__shfl_sync(0xffffffffu, base, 4 + d) & 0xffffu) << (16 * d);
        }
#pragma unroll
        for (int k = 0; k < VR_NIT; k++) {
            const uint32_t key = keys[k];
            if (key != VC_NOKEY) {
                const uint32_t own = __umulhi(vr_h1(key), csize), shf = (own & 3u) * 16u;
                const uint32_t pos = (uint32_t)(((own & 4u) ? s1 : s0) >> shf) & 0xffffu;
                if (own & 4u) s1 += 1ull << shf; else s0 += 1ull << shf;
                if (pos < cap) cluster.map_shared_rank(q, own)[pos] = make_uint2(key, wbeg + k * 32 + lane);
            }
        }
    }
    cluster.sync();   // #1: every queue is complete
    const uint32_t n = *vqcount;
    {
        const uint32_t ov = *vbail;
        __syncthreads();
        if (tid == 0) { *sh.qcount = 0; *sh.npool = 0; sh.lcount[0] = 0; sh.lcount[1] = 0; if (ov) *sh.bail = 0; }
#ifdef D3D_VC_TIMING
        if (ov && tid == 0) printf("frame %d cl %u cta %u: queue overflow (n %u cap %u)\n", (int)f, cid, crank, n, cap);
#endif
        if (ov) return false;
        __syncthreads();
    }
    VC_TICK(0);

    // ---- R2: one slot per distinct key.  Two rounds of plain stores settle ~88 % of the entries; the stragglers
    // move to a work list and finish with compare-and-swap probes, which need no barrier and no lock step.
    uint32_t s[VR_E];
    {
        uint32_t unres = 0, moved = 0;
#pragma unroll
        for (int e = 0; e < VR_E; e++) {
            const uint32_t p = tid + e * VC_THREADS;
            s[e] = 0;
            if (p < n) { s[e] = (vr_h1(q[p].x) << 3) >> hshift; unres |= 1u << e; }
        }
#ifndef D3D_VR_ROUNDS
#define D3D_VR_ROUNDS 2
#endif
#pragma unroll 1
        for (int round = 0; round < D3D_VR_ROUNDS; round++) {
#pragma unroll
            for (int e = 0; e < VR_E; e++)
                if ((unres >> e) & 1u) { if (slot[s[e]] == VR_SLOT_EMPTY) slot[s[e]] = (uint16_t)(tid + e * VC_THREADS); }   // racy on purpose: any writer wins
            __syncthreads();
#pragma unroll
            for (int e = 0; e < VR_E; e++)
                if ((unres >> e) & 1u) {
                    const uint32_t kq = q[tid + e * VC_THREADS].x;
                    const uint32_t wv = slot[s[e]];
                    if (q[wv].x == kq) { unres &= ~(1u << e); s[e] = wv; }
                    else s[e] = (s[e] + vr_step(kq, smask)) & smask;
                }
            if (round + 1 < D3D_VR_ROUNDS) { __syncthreads(); VR_SUB(8); }   // the next round's stores must not overtake this round's lookups
        }
        VR_SUB(9);
        {   // hand the stragglers to the list (what does not fit stays with its thread); one reservation per warp
            const uint32_t cnt = __popc(unres);
            const uint32_t at = vr_reserve(sh.lcount, cnt, lane);
            if (cnt == 0) {
            } else if (at + cnt <= (uint32_t)VR_LIST) {
                uint32_t o = at;
#pragma unroll
                for (int e = 0; e < VR_E; e++)
                    if ((unres >> e) & 1u) list[o++] = (tid + e * VC_THREADS) | (s[e] << 16);
                moved = unres; unres = 0;
            } else {
                for (uint32_t o = at; o < (uint32_t)VR_LIST; o++) list[o] = VC_NONE;   // partial reservation: dead entries
            }
        }
        __syncthreads();
        VR_SUB(12);
        // claim-or-join with a 32-bit CAS on the slot pair; slots only ever fill, so an entry that walks its probe
        // sequence meets the slot its key settled in (or settles it) whatever the interleaving
        auto settle = [&](uint32_t p, uint32_t sl) -> uint32_t {
            const uint32_t kq = q[p].x;
            const uint32_t step = vr_step(kq, smask);
            for (;;) {
                uint32_t *wp = reinterpret_cast<uint32_t *>(slot) + (sl >> 1);
                const uint32_t sh16 = (sl & 1u) * 16u;
                uint32_t cur = *reinterpret_cast<volatile uint32_t *>(wp), h;
                for (;;) {
                    h = (cur >> sh16) & 0xffffu;
                    if (h != VR_SLOT_EMPTY) break;
                    const uint32_t old = atomicCAS(wp, cur, (cur & ~(0xffffu << sh16)) | (p << sh16));
                    if (old == cur) { h = p; break; }
                    cur = old;
                }
                if (h == p || q[h].x == kq) return h;
                sl = (sl + step) & smask;
            }
        };
        {
            const uint32_t nl = min(*vlcount, (uint32_t)VR_LIST);
            for (uint32_t j = tid; j < nl; j += VC_THREADS) {
                const uint32_t ent = list[j];
                if (ent != VC_NONE) {
                    const uint32_t p = ent & 0xffffu;
                    const uint32_t wv = settle(p, ent >> 16);
                    if (wv != p) q[p].x = VR_LOSER | wv;   // a loser's key word is dead (only winners' keys are looked up): it carries the winner to the entry's own thread
                }
            }
            if (unres) {
#pragma unroll
                for (int e = 0; e < VR_E; e++)
                    if ((unres >> e) & 1u) s[e] = settle(tid + e * VC_THREADS, s[e]);
            }
            __syncthreads();
        }
        VR_SUB(10);
        // entries resolved on the list left their winner in their key word (or kept the key: they are winners)
#pragma unroll
        for (int e = 0; e < VR_E; e++)
            if ((moved >> e) & 1u) { const uint32_t p = tid + e * VC_THREADS, x = q[p].x; s[e] = (x & VR_LOSER) ? (x & 0xffffu) : p; }
        // from here on s[e] is the queue position of the voxel's winner.  Winners: key word <- own index, 0 joiners
        // (the index word becomes the voxel's minimum); every lookup of a winner's key is behind the barrier above.
#pragma unroll
        for (int e = 0; e < VR_E; e++) {
            const uint32_t p = tid + e * VC_THREADS;
            if (p < n && s[e] == p) q[p].x = q[p].y;
        }
        __syncthreads();
#pragma unroll
        for (int e = 0; e < VR_E; e++) {
            const uint32_t p = tid + e * VC_THREADS;
            if (p < n && s[e] != p) { atomicMin(&q[s[e]].y, q[p].y); atomicAdd(&q[s[e]].x, 1u << VR_IDX_BITS); }
        }
        if (tid == 0) { sh.lcount[0] = 0; sh.lcount[1] = 0; }
        __syncthreads();
        VR_SUB(11);
    }
    VC_TICK(1);

    // frame-local index of queue entry p whose voxel's winner is win: a winner's index word was taken over by its voxel
    auto own_index = [&](uint32_t p, uint32_t win) -> uint32_t { return win == p ? (q[p].x & VR_IDX_MASK) : (q[p].y & VR_IDX_MASK); };

    // ---- R3: the K smallest indices of every voxel that holds more than K points.  The first point opens a
    // record for the voxel (the winner's index word now names the record), the other points go to the work
    // list as (entry | winner << 16) and compete in K-1 rounds; a kept entry gets VR_KEPT in its index word.
    if (cthr != VC_NONE) {
        uint32_t cm = 0, hd = 0;
#pragma unroll
        for (int e = 0; e < VR_E; e++) {
            const uint32_t p = tid + e * VC_THREADS;
            if (p < n && (q[s[e]].x >> VR_IDX_BITS) + 1 > cthr) {
                if (own_index(p, s[e]) == q[s[e]].y) hd |= 1u << e; else cm |= 1u << e;
            }
        }
        if (__syncthreads_or((int)(cm | hd))) {
            bool over = false;
            if (hd) {
#pragma unroll
                for (int e = 0; e < VR_E; e++)
                    if ((hd >> e) & 1u) {
                        uint32_t r = atomicAdd(sh.npool, 1u);
                        if (r >= (uint32_t)VR_POOL) { over = true; r = 0; }
                        else { sh.pool_min[r] = q[s[e]].y; sh.pool_acc0[r] = 0xffffffffu; sh.pool_acc1[r] = 0xffffffffu; }
                        q[s[e]].y = r;
                    }
            }
            {
                const uint32_t cnt = __popc(cm);
                uint32_t o = vr_reserve(sh.lcount, cnt, lane);
                if (cnt == 0) {
                } else if (o + cnt > (uint32_t)VR_LIST) {
                    over = true;
                    for (; o < (uint32_t)VR_LIST; o++) list[o] = VC_NONE;
                } else {
#pragma unroll
                    for (int e = 0; e < VR_E; e++)
                        if ((cm >> e) & 1u) list[o++] = (tid + e * VC_THREADS) | (s[e] << 16);
                }
            }
            if (over) for (unsigned d = 0; d < csize; d++) *cluster.map_shared_rank(sh.bail, d) = 1u;   // too crowded for this path
            __syncthreads();
            const uint32_t nc = min(*vlcount, (uint32_t)VR_LIST);
            for (uint32_t r = 1; r < K; r++) {
                uint32_t *acc = (r & 1u) ? sh.pool_acc1 : sh.pool_acc0;
                const uint32_t pre = (0x3fffu - (r & 0x3fffu)) << VR_IDX_BITS;   // a later round always wins the minimum: nothing to reset
                uint32_t open = 0;
                for (uint32_t j = tid; j < nc; j += VC_THREADS) {
                    const uint32_t ent = list[j];
                    if (ent != VC_NONE) { atomicMin(&acc[q[ent >> 16].y & 0xffffu], pre | own_index(ent & 0xffffu, ent >> 16)); open = 1; }
                }
                if (!__syncthreads_or((int)open)) break;
                for (uint32_t j = tid; j < nc; j += VC_THREADS) {
                    const uint32_t ent = list[j];
                    if (ent != VC_NONE) {
                        const uint32_t p = ent & 0xffffu, wv = ent >> 16;
                        // (racecheck flags this store against the next round's read of q[wv].y by faster threads when p == wv: only bit 31
                        // changes and every reader masks it off, so both values name the same record)
                        if (acc[q[wv].y & 0xffffu] == (pre | own_index(p, wv))) { list[j] = VC_NONE; q[p].y |= VR_KEPT; }
                    }
                }
            }
            __syncthreads();   // VR_KEPT was set by whoever processed the list entry, R4 reads it from the entry's own thread
        }
    }
    VC_TICK(2);

    // ---- R4: one word back to every point that shares its voxel (or whose voxel fails min_points)
#pragma unroll
    for (int e = 0; e < VR_E; e++) {
        const uint32_t p = tid + e * VC_THREADS;
        if (p < n) {
            const uint32_t total = (q[s[e]].x >> VR_IDX_BITS) + 1;
            if (total > 1) {
                const uint32_t my = own_index(p, s[e]);
                const bool crowded = total > cthr;
                const uint32_t wy = q[s[e]].y;
                const uint32_t mn = crowded ? sh.pool_min[wy & 0xffffu] : wy;
                uint32_t r;
                if ((long long)total < (long long)cfg.min_points) r = VC_NONE;
                else if (my == mn) r = VR_HEAD | VR_KEEP | total;                       // rank 0 is always kept (K >= 1 when crowded)
                else r = ((!crowded || (q[p].y & VR_KEPT)) ? VR_KEEP : 0u) | mn;
                const uint32_t c = ((my >> 10) * magic) >> 16;
                cluster.map_shared_rank(reply, c)[my - c * Lc] = r;
            }
        }
    }
    cluster.sync();   // #2: every reply has arrived
    {
        const uint32_t cb = *vbail;
        __syncthreads();
        if (tid == 0) *sh.bail = 0;
#ifdef D3D_VC_TIMING
        if (cb && tid == 0 && crank == 0) printf("frame %d cl %u: too many crowded voxels\n", (int)f, cid);
#endif
        if (cb) return false;
    }
    VC_TICK(3);

    // ---- R5: first-of-voxel bits -> voxel ids.  Without a voxel cap the keep decision is already in the reply word, so both
    // prefix sums share one exchange and the ids of the points that are not first of their voxel are looked up in R6.
    const bool twopass = vcap != VC_NONE;
    {
        uint32_t carry = 0, kcarry = 0;
        for (uint32_t k = 0; k < nit; k++) {
            const uint32_t i = wbeg + k * 32 + lane;
            const uint32_t r = i < L ? reply[lbeg + k * 32 + lane] : VC_NONE;
            const unsigned bal = __ballot_sync(0xffffffffu, r != VC_NONE && (r & VR_HEAD));
            if (lane == 0) hbp[w * nit + k] = make_uint2(bal, carry);
            carry += __popc(bal);
            if (!twopass) kcarry += __popc(__ballot_sync(0xffffffffu, r != VC_NONE && (r & VR_KEEP) && !dropall));
        }
        if (lane == 0) { sh.mytot[w] = carry; sh.mytot2[w] = kcarry; }
        if (twopass) {
            vc_exchange(cluster, sh.mytot, sh.wt1, sh.vbase, csize, crank);   // cluster barrier #3 inside
            if (w == 0) { const unsigned long long x = vc_lookback(a.vstate, f, min(sh.vbase[W], vcap), crank == 0); if (lane == 0) sh.frow[0] = x; }
        } else {
            vc_exchange2(cluster, sh.mytot, sh.mytot2, sh.wt1, sh.wt2, sh.vbase, sh.pbase, csize, crank);   // cluster barrier #3 inside
            if (w == 0) { const unsigned long long x = vc_lookback(a.vstate, f, sh.vbase[W], crank == 0); if (lane == 0) sh.frow[0] = x; }
            if (w == 1) { const unsigned long long x = vc_lookback(a.kstate, f, sh.pbase[W], crank == 0); if (lane == 0) sh.frow[1] = x; }
        }
        __syncthreads();
    }
    VC_TICK(4);
    if (twopass) {   // the voxel cap decides which points stay: ids first, then the second prefix sum
        uint32_t carry = 0;
        const uint32_t vb = sh.vbase[g];
        for (uint32_t k = 0; k < nit; k++) {
            const uint32_t i = wbeg + k * 32 + lane, li = lbeg + k * 32 + lane;
            const uint32_t r = i < L ? reply[li] : VC_NONE;
            uint32_t out = VC_NONE;
            bool keep = false;
            if (r != VC_NONE) {
                uint32_t vid;
                if (r & VR_HEAD) {
                    const uint2 h = hbp[li >> 5];
                    vid = vb + h.y + __popc(h.x & ltmask);
                } else {   // the id lives where the voxel's first point lives
                    const uint32_t m = r & VR_VAL;
                    const uint32_t c = ((m >> 10) * magic) >> 16;
                    const uint32_t lj = (m - c * Lc) >> 5;
                    const uint32_t wv = (lj * magic) >> 16;
                    const uint2 h = cluster.map_shared_rank(hbp, c)[lj];   // one remote load (2.7 clk per lane)
                    vid = sh.vbase[c * VC_WARPS + wv] + h.y + __popc(h.x & ((1u << (m & 31u)) - 1u));
                }
                if (vid < vcap) {
                    keep = (r & VR_KEEP) && !dropall;
                    out = (r & VR_HEAD) ? ((r & ~VR_KEEP) | (keep ? VR_KEEP : 0u)) : ((keep ? VR_KEEP : 0u) | vid);
                }
            }
            if (i < L) reply[li] = out;
            carry += __popc(__ballot_sync(0xffffffffu, keep));
        }
        if (lane == 0) sh.mytot[w] = carry;
        vc_exchange(cluster, sh.mytot, sh.wt2, sh.pbase, csize, crank);   // cluster barrier #4 inside
        if (w == 0) { const unsigned long long x = vc_lookback(a.kstate, f, sh.pbase[W], crank == 0); if (lane == 0) sh.frow[1] = x; }
        __syncthreads();
    }
    VC_TICK(5);

    // ---- R6: voxel rows (written by the voxel's first point) and packed point rows, in input order
    {
        int64_t run = (int64_t)sh.frow[1] + sh.pbase[g];
        const int64_t vrow = (int64_t)sh.frow[0];
        const uint32_t vb = sh.vbase[g];
        long long *stg = reinterpret_cast<long long *>(slot) + w * 96;   // the slot table is idle until the next frame
        for (uint32_t k0 = 0; k0 < nit; k0 += VC_U) {
            uint32_t r[VC_U];
            float4 p[VC_U];
            uint2 hrem[VC_U];
            uint32_t hoff[VC_U];
#pragma unroll
            for (int u = 0; u < VC_U; u++) {
                const uint32_t i = wbeg + (k0 + u) * 32 + lane;
                r[u] = (k0 + u < nit && i < L) ? reply[lbeg + (k0 + u) * 32 + lane] : VC_NONE;
                if (r[u] != VC_NONE && dropall) r[u] &= ~VR_KEEP;
                if (r[u] != VC_NONE && !(r[u] & (VR_HEAD | VR_KEEP))) r[u] = VC_NONE;
                hrem[u] = make_uint2(0u, 0u); hoff[u] = 0;
                if (!twopass && r[u] != VC_NONE && !(r[u] & VR_HEAD)) {   // id of a voxel whose first point lives elsewhere: loads of all rounds in flight together
                    const uint32_t m = r[u] & VR_VAL;
                    const uint32_t c = ((m >> 10) * magic) >> 16;
                    const uint32_t lj = (m - c * Lc) >> 5;
                    hrem[u] = cluster.map_shared_rank(hbp, c)[lj];
                    hoff[u] = sh.vbase[c * VC_WARPS + ((lj * magic) >> 16)];
                }
            }
#pragma unroll
            for (int u = 0; u < VC_U; u++)
                if (r[u] != VC_NONE) p[u] = __ldg(pts4 + wbeg + (k0 + u) * 32 + lane);
#pragma unroll
            for (int u = 0; u < VC_U; u++) {
                const uint32_t i = wbeg + (k0 + u) * 32 + lane, lj = (lbeg >> 5) + k0 + u;
                const bool valid = r[u] != VC_NONE;
                const bool head = valid && (r[u] & VR_HEAD), keep = valid && (r[u] & VR_KEEP);
                uint32_t nid = r[u] & VR_VAL;
                if (!twopass && valid && !head) nid = hoff[u] + hrem[u].y + __popc(hrem[u].x & ((1u << (nid & 31u)) - 1u));
                // voxel rows of this round are consecutive: the coordinates go through a per-warp staging row so that
                // the global stores are three dense 256-byte lines instead of three 24-byte-strided ones
                const unsigned hbal = __ballot_sync(0xffffffffu, head);
                if (hbal) {
                    const uint32_t rank = __popc(hbal & ltmask), nh3 = 3u * __popc(hbal);
                    const uint32_t first = vb + hbp[lj].y;
                    if (head) {
                        const uint32_t c = nid;   // points in the voxel
                        nid = first + rank;
                        const int c0 = (int)floorf(__fdiv_rn(p[u].x, dv.size[0])), c1 = (int)floorf(__fdiv_rn(p[u].y, dv.size[1])),
                                  c2 = (int)floorf(__fdiv_rn(p[u].z, dv.size[2]));
                        stg[rank * 3 + 0] = (long long)(uint32_t)(c0 - dv.vlo[0]) + dv.cadd[0];
                        stg[rank * 3 + 1] = (long long)(uint32_t)(c1 - dv.vlo[1]) + dv.cadd[1];
                        stg[rank * 3 + 2] = (long long)(uint32_t)(c2 - dv.vlo[2]) + dv.cadd[2];
                        __stcs(a.out_npoints + vrow + nid, (trim && c > K) ? (int32_t)K : (int32_t)c);
                    }
                    __syncwarp();
                    long long *co = reinterpret_cast<long long *>(a.out_coords) + (vrow + first) * 3;
#pragma unroll
                    for (int t = 0; t < 3; t++)
                        if (t * 32 + lane < nh3) __stcs(co + t * 32 + lane, stg[t * 32 + lane]);
                    __syncwarp();
                }
                const unsigned bal = __ballot_sync(0xffffffffu, keep);
                if (keep) {
                    const int64_t o = run + __popc(bal & ltmask);
                    __stcs(reinterpret_cast<float4 *>(a.out_points) + o, p[u]);
                    __stcs(reinterpret_cast<long long *>(a.out_mask) + o, (long long)i);
                    __stcs(reinterpret_cast<long long *>(a.out_mapping) + o, (long long)nid);
                }
                run += __popc(bal);
            }
        }
        if (crank == 0 && tid == 0) {
            a.counts[2 * f] = (long long)sh.frow[1]; a.counts[2 * f + 1] = (long long)sh.frow[0];
            if (f == a.nframes - 1) { a.counts[2 * f + 2] = (long long)(sh.frow[1] + sh.pbase[W]); a.counts[2 * f + 3] = (long long)(sh.frow[0] + min(sh.vbase[W], vcap)); }
        }
    }
    __syncthreads();   // the next frame may map points to threads differently: its defaults must not overtake this frame's reads of the reply words
    VC_TICK(6); VR_TICK_PRINT;
    return true;
}

template <bool DENSE>
__global__ void __launch_bounds__(VC_THREADS, 1) vox_cluster_kernel(const VcArgs a, const VcDev dv)
{
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned csize = cluster.num_blocks();
    const unsigned ncl = gridDim.x / csize, cid = blockIdx.x / csize;

    __shared__ uint32_t mytot[VC_WARPS], mytot2[VC_WARPS];
    __shared__ uint32_t wt1[VC_MAX_CSIZE * VC_WARPS], wt2[VC_MAX_CSIZE * VC_WARPS];
    __shared__ uint32_t vbase[VC_MAX_CSIZE * VC_WARPS + 1], pbase[VC_MAX_CSIZE * VC_WARPS + 1];
    __shared__ unsigned long long frow[2];
    __shared__ uint2 hbp[DENSE ? 1 : VC_WARPS * VR_NIT];
    __shared__ uint32_t list[DENSE ? 1 : VR_LIST];
    __shared__ uint32_t pool[DENSE ? 3 : 3 * VR_POOL];
    __shared__ uint32_t flags[8];
    extern __shared__ __align__(16) unsigned char vc_dyn[];

    VcSh sh;
    sh.mytot = mytot; sh.mytot2 = mytot2; sh.wt1 = wt1; sh.wt2 = wt2; sh.vbase = vbase; sh.pbase = pbase; sh.frow = frow;
    sh.hbp = hbp; sh.list = list; sh.lcount = flags + 4;
    sh.pool_min = pool; sh.pool_acc0 = pool + (DENSE ? 1 : VR_POOL); sh.pool_acc1 = pool + (DENSE ? 2 : 2 * VR_POOL);
    sh.qcount = flags; sh.npool = flags + 1; sh.bail = flags + 2;
    sh.dyn = vc_dyn;

    if (a.run_if && *a.run_if == 0) return;   // grid-uniform
    const bool route = !DENSE && a.route && a.nfeat == 4;
    __shared__ uint32_t s_frame;
    if (threadIdx.x < 8) flags[threadIdx.x] = 0;
    // Frames are taken from a ticket counter, not from the cluster index: a frame is only ever started by a cluster that
    // is running, so the look-back (which waits for lower-numbered frames) cannot wait for a cluster that the hardware
    // has not scheduled yet (other kernels on the GPU, MPS limits, out-of-order dispatch).
    for (;;) {
        if (cluster.block_rank() == 0 && threadIdx.x == 0) {
            const uint32_t t = atomicAdd(a.ticket, 1u);
            for (unsigned d = 0; d < csize; d++) *cluster.map_shared_rank(&s_frame, d) = t;
        }
        cluster.sync();   // also: nobody pushes into a queue whose counter is not initialised yet
        const int64_t f = (int64_t)s_frame;
        if (f >= a.nframes) break;
        if (route) {
            VrPlan pl;
            const uint32_t L = (uint32_t)min((long long)(a.offs[f + 1] - a.offs[f]), (long long)a.lmax);
            if (vr_plan(L, csize, a.dyn_bytes, &pl) && vc_frame_route(a, dv, sh, cluster, f, pl, cid, ncl)) continue;
        }
        vc_frame_l2<DENSE>(a, dv, sh, cluster, f, cid, ncl);
    }   // the barrier at the top of the loop also separates this frame's remote shared-memory reads from the next frame's writes
}

// ------------------------------------------------------------------ host side
bool vox_cluster_supported(const VoxCfg &cfg, int64_t total, int64_t nframes, int64_t max_frame_points)
{
    (void)total; (void)nframes;
    VcDev d;
    if (!vc_make_dev(cfg, &d)) return false;                           // bit-field cell keys, 32-bit cell arithmetic
    if (max_frame_points >= (1ll << 27)) return false;                 // provisional ids: 9 + 20 bits
    if (cfg.ext[0] <= 0 || cfg.ext[1] <= 0 || cfg.ext[2] <= 0) return false;
    if (!cfg.dense && cfg.vfilter == D3D_VF_DESCENDING) return false;  // needs a sort of the voxels
    if (cfg.dense && cfg.reduction != D3D_RED_NONE) return false;      // sequential float sums need sorted segments
    return true;
}

size_t vox_cluster_ws_bytes(int64_t total, int64_t nframes, int64_t max_frame_points)
{
    if (max_frame_points <= 0 || max_frame_points > total) max_frame_points = total;
    int64_t ncl = nframes < VC_MAX_CLUSTERS ? nframes : VC_MAX_CLUSTERS;
    if (ncl < 1) ncl = 1;
    return vc_layout(max_frame_points).total * (size_t)ncl + 512 + align_up((size_t)(nframes > 0 ? nframes : 1) * 16);
}

// Cluster shape: CTAs of one cluster must sit in one GPC, and a B200's GPCs do not all expose a multiple of 8
// SMs, so 8-CTA clusters leave SMs idle (15 clusters = 120 of 148 SMs on the boxes measured).  The L2 path
// takes the size (<= 8, portable) that occupies the most SMs; the routed path needs the frame to fit the
// cluster's shared memory, so among the sizes whose plan holds the largest frame it takes the one that
// occupies the most SMs, and the kernel falls back to the L2 path frame by frame.
struct VcShape { int csize, max_clusters; uint32_t dyn; int route; };

constexpr uint32_t VC_L2_DYN = 2u * VC_WARPS * VC_QCAP * sizeof(uint32_t);   // per-warp probe rings of the L2 path

template <bool DENSE>
static int vc_shape(VcShape *out, int64_t max_frame_points)
{
    auto kern = vox_cluster_kernel<DENSE>;
    // cached per device: function attributes and occupancy belong to the device's context (one process may drive several GPUs)
    static int occ_dev[64][VC_MAX_CSIZE + 1];   // co-resident clusters per cluster size (0 = not queried yet, -1 = unavailable)
    static uint32_t dyn_dev[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); return D3D_ERR_CUDA; }
    int *occ = occ_dev[dev];
    uint32_t &dyn = dyn_dev[dev];
    if (dyn == 0) {
        dyn = VC_L2_DYN;
        if (!DENSE) {
            int optin = 0;
            cudaFuncAttributes fa;
            if (cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess ||
                cudaFuncGetAttributes(&fa, kern) != cudaSuccess) { cudaGetLastError(); return D3D_ERR_CUDA; }
            const long long d = ((long long)optin - (long long)fa.sharedSizeBytes) & ~1023ll;
            if (d > (long long)dyn) dyn = (uint32_t)d;
        }
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn) != cudaSuccess) { cudaGetLastError(); dyn = 0; return D3D_ERR_CUDA; }
    }
    auto query = [&](int cs) -> int {
        if (occ[cs] == 0) {
            cudaLaunchConfig_t lc = {};
            lc.blockDim = dim3(VC_THREADS, 1, 1);
            lc.gridDim = dim3(cs, 1, 1);
            lc.dynamicSmemBytes = dyn;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = cs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            lc.attrs = at; lc.numAttrs = 1;
            int n = 0;
            if (cudaOccupancyMaxActiveClusters(&n, kern, &lc) != cudaSuccess || n < 1) { cudaGetLastError(); n = -1; }
            occ[cs] = n;
        }
        return occ[cs];
    };
    const int route = DENSE ? 0 : tuning(D3D_TUNE_VOX_ROUTE, 1);   // tuning override
    VcShape best = {0, 0, dyn, 0};
    if (route) {
        VrPlan pl;
        for (int cs = 8; cs >= 4; cs -= 2) {
            if (!vr_plan((uint32_t)(max_frame_points > 0 ? max_frame_points : 1), cs, dyn, &pl)) continue;
            const int n = query(cs);
            if (n > 0 && n * cs > best.csize * best.max_clusters) best = {cs, n, dyn, 1};
        }
    }
    if (best.csize == 0) {
        for (int cs = 8; cs >= 4; cs -= 2) {   // 8, 6, 4: smaller clusters put more frames in flight than L2 holds
            const int n = query(cs);
            if (n > 0 && n * cs > best.csize * best.max_clusters) best = {cs, n, dyn, route};
        }
    }
    if (best.csize == 0) return D3D_ERR_CUDA;
    *out = best;
    return D3D_OK;
}

template <bool DENSE>
static int vc_launch(VcArgs &args, int64_t nframes, int64_t max_frame_points, size_t ws_bytes, cudaStream_t st)
{
    VcDev dv;
    if (!vc_make_dev(args.cfg, &dv)) return D3D_ERR_UNSUPPORTED;
    VcShape shape;
    int rc = vc_shape<DENSE>(&shape, max_frame_points);
    if (rc) return rc;
    const int csize = shape.csize;
    args.dyn_bytes = shape.dyn; args.route = shape.route;
    auto kern = vox_cluster_kernel<DENSE>;
    cudaLaunchConfig_t lc = {};
    lc.blockDim = dim3(VC_THREADS, 1, 1);
    lc.dynamicSmemBytes = shape.dyn;
    lc.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = csize; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    lc.attrs = at; lc.numAttrs = 1;
    int64_t ncl = shape.max_clusters;
    if (ncl > nframes) ncl = nframes;
    if (ncl > VC_MAX_CLUSTERS) ncl = VC_MAX_CLUSTERS;
    const size_t state_bytes = 256 + align_up((size_t)nframes * 16);
    while (ncl > 1 && args.lay.total * (size_t)ncl + 256 + state_bytes > ws_bytes) ncl--;
    if (args.lay.total * (size_t)ncl + 256 + state_bytes > ws_bytes) return D3D_ERR_WORKSPACE;
    {   // ticket counter and (sparse) look-back words live behind the cluster slices
        char *state = args.ws + align_up(args.lay.total * (size_t)ncl);
        args.ticket = reinterpret_cast<uint32_t *>(state);
        args.vstate = reinterpret_cast<unsigned long long *>(state + 256);
        args.kstate = args.vstate + nframes;
        D3D_CUDA_TRY(cudaMemsetAsync(state, 0, DENSE ? 256 : 256 + (size_t)nframes * 16, st));
    }
    args.lmax = (uint32_t)(max_frame_points > 0 ? max_frame_points : 1);
    lc.gridDim = dim3((unsigned)(ncl * csize), 1, 1);
    D3D_CUDA_TRY(cudaLaunchKernelEx(&lc, kern, args, dv));
    D3D_LAUNCHED();
    return D3D_OK;
}

int vox_cluster_sparse(const float *points, int64_t total, int nfeat, const int64_t *offs, int64_t nframes, int64_t max_frame_points, const VoxCfg &cfg,
                       float *out_points, int64_t *out_mask, int64_t *out_mapping, int32_t *out_npoints, int64_t *out_coords, int64_t *counts,
                       void *ws, size_t ws_bytes, cudaStream_t st, const uint32_t *run_if)
{
    if (max_frame_points <= 0 || max_frame_points > total) max_frame_points = total;
    VcArgs a = {};
    a.run_if = run_if;
    a.pts = points; a.nfeat = nfeat; a.offs = offs; a.nframes = nframes; a.cfg = cfg;
    a.out_points = out_points; a.out_mask = out_mask; a.out_mapping = out_mapping; a.out_npoints = out_npoints; a.out_coords = out_coords;
    a.counts = counts; a.ws = (char *)ws; a.lay = vc_layout(max_frame_points);
    return vc_launch<false>(a, nframes, max_frame_points, ws_bytes, st);
}

int vox_cluster_dense(const float *points, int64_t total, int nfeat, const int64_t *offs, int64_t nframes, int64_t max_frame_points, const VoxCfg &cfg,
                      float *voxels, int64_t *coords, uint8_t *pmask, int32_t *npoints, int64_t *counts, void *ws, size_t ws_bytes, cudaStream_t st)
{
    if (max_frame_points <= 0 || max_frame_points > total) max_frame_points = total;
    VcArgs a = {};
    a.pts = points; a.nfeat = nfeat; a.offs = offs; a.nframes = nframes; a.cfg = cfg;
    a.out_npoints = npoints; a.out_coords = coords; a.counts = counts; a.voxels = voxels; a.pmask = pmask;
    a.ws = (char *)ws; a.lay = vc_layout(max_frame_points);
    return vc_launch<true>(a, nframes, max_frame_points, ws_bytes, st);
}

}  // namespace d3d
