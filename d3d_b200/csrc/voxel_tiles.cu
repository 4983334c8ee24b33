// voxel_tiles.cu -- sparse voxelization as a pipeline of streaming tile kernels (the default fast path).
//
// Replaces voxelize_sparse + voxelize_filter (reference d3d/voxel/voxelize.cpp:288-484) for the common
// configurations (no voxel cap, max_points filter NONE or TRIM with max_points <= 8, cell keys of <= 30 bits);
// everything else goes to the cluster path (voxel_cluster.cu) or the sort path (voxel.cu).  Same packed outputs,
// bit for bit.
//
// Why not one cluster per frame (voxel_cluster.cu): that kernel keeps a whole frame in the shared memory of 8 SMs,
// which pins one 1024-thread CTA per SM, all warps of an SM in the same phase, on the 120 SMs that 8-CTA clusters
// reach -- it is bound by exposed latency, not by HBM (ncu: issue slots 52 % busy, DRAM 15 %).  Here a chunk of
// frames runs through four ordinary kernels, each with the block size, register budget and occupancy its stage
// wants, on all 148 SMs:
//
//   split   (1024 points / CTA)  cell keys with the reference's fp32 arithmetic; a point's (key, index) goes to
//                                the queue of the BUCKET its key hashes to (256 buckets for a 120k-point frame);
//                                the tile counts per bucket in shared memory and reserves its share of every queue
//                                with one global atomic per bucket.  The point's word is its key: a point that
//                                hears nothing back is the only point of its voxel.
//   bucket  (one CTA / bucket)   all points of a voxel meet in one bucket: hash table in shared memory (CAS claim,
//                                atomicMin of the point index, count -- B200 issues a shared-memory atomic in
//                                ~1.3 clk per warp, tools/warp_prims_probe.cu), the K smallest indices of voxels with
//                                more than K points by a min-cascade (level j keeps the j-th smallest of everything
//                                it is offered and passes the larger value on: the result does not depend on the
//                                arrival order); the points that share a voxel get a new word.
//   scan    (8192 points / CTA)  first-of-voxel and keep bits -> ballots -> one chained scan over all tiles of all
//                                frames (decoupled look-back): voxel ids in order of first appearance, packed rows.
//   write   (1024 points / CTA)  voxel rows and kept point rows streamed out; no barrier, no waiting.
//
// A batch is cut into chunks of 64 frames (vt_geom).  Small chunks keep the scratch
// (queues, words, row tables: ~1.3 MB per frame, plus the frame itself) in L2 between the kernels, large chunks give fewer
// and fuller launches; on B200 the large chunks win (C2 x 128 frames: 0.59 ms against 0.74 ms with chunks of 16) although
// the scratch then travels through HBM (DRAM traffic ~1.9x the algorithmic 16 B/point in, 32 B/kept point + 28 B/voxel out).
//
// Determinism: every output is a function of the point set (smallest index, count, K smallest indices, prefix
// sums in point order), never of the race order of the queues and tables.
//
// Anything that does not fit (a bucket queue or table overflow: e.g. thousands of points in one voxel) raises a
// device flag; the cluster kernel is launched behind the pipeline on that flag and redoes the batch.
#include "voxel.cuh"
#include <stdlib.h>
#include <mutex>

namespace d3d {

constexpr int VT_THREADS = 256;
constexpr int VT_WARPS = VT_THREADS / 32;
constexpr int VT_PPT = 4;                         // points per thread (split, write)
constexpr int VT_TILE = VT_THREADS * VT_PPT;      // 1024 points per tile
constexpr int VT_SPT = 32;                        // points per thread (scan): lane u of a warp keeps the warp's row u
constexpr int VT_STILE = VT_THREADS * VT_SPT;     // 8192 points per scan tile
#ifndef D3D_VT_BT
#define D3D_VT_BT 128
#endif
#ifndef D3D_VT_EPT
#define D3D_VT_EPT 4
#endif
#ifndef D3D_VT_BPTS
#define D3D_VT_BPTS 512      // points per bucket the geometry aims at (if every point is kept)
#endif
#ifndef D3D_VT_BCTAS
#define D3D_VT_BCTAS 12
#endif
#ifndef D3D_VT_WCTAS
#define D3D_VT_WCTAS 4
#endif
#ifndef D3D_VT_SCTAS
#define D3D_VT_SCTAS 6
#endif
constexpr int VT_BT = D3D_VT_BT;                  // threads of a bucket CTA
constexpr int VT_EPT = D3D_VT_EPT;                // queue entries per bucket thread kept in registers (longer queues: the rest is re-read)
#ifndef D3D_VT_QCAP
#define D3D_VT_QCAP 1024
#endif
constexpr int VT_QCAP = D3D_VT_QCAP;              // largest queue a bucket CTA takes
constexpr int VT_SMAX = VT_QCAP <= 512 ? 512 : (VT_QCAP <= 1024 ? 1024 : 2048);   // table slots per bucket (maximum)
constexpr int VT_MAXK = 8;                        // deepest min-cascade (max_points of the TRIM filter)
constexpr int VT_POOL = 64;                       // crowded-voxel records per bucket
constexpr uint32_t VT_NONE = 0xffffffffu;         // empty table slot / queue entry
// point word, category in bits 31:30 -- 0: cell key (<= 30 bits) of a point that is alone in its voxel | 1: nothing to write |
// 2: kept point of a shared voxel + index of the voxel's first point | 3: first point of a shared voxel + point count
constexpr uint32_t VT_W_NONE = 1u << 30, VT_W_JOIN = 2u << 30, VT_W_HEAD = 3u << 30, VT_VAL = (1u << 30) - 1;
constexpr unsigned long long VT_PVAL = (1ull << 62) - 1;   // status word: flag << 62 | kept rows << 31 | voxel rows
constexpr uint32_t VT_F31 = 0x7fffffffu;

struct VtGeom {
    uint32_t lmax, lpad, tpf, spf; // longest frame, padded to whole scan tiles, tiles / scan tiles per frame
    uint32_t lgP, P, qcap;         // buckets per frame, queue entries per bucket
    uint32_t CF, nchunks;          // frames per chunk, chunks
};

struct VtArgs {
    const float *pts; int nfeat; const int64_t *offs; int64_t nframes;
    float *out_points; int64_t *out_mask; int64_t *out_mapping; int32_t *out_npoints; int64_t *out_coords; int64_t *counts;
    uint2 *queue; uint32_t *word, *hkey; uint4 *rowinfo; uint32_t *qcount;
    unsigned long long *status; uint32_t *tickets, *bail;
    VtGeom g;
    uint32_t K, cthr; int min_points; int trim, dropall, single_ok;
};

__device__ __forceinline__ unsigned long long vt_ld_acquire(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void vt_st_release(unsigned long long *p, unsigned long long v)
{
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// L2 residency hints.  The scratch of a chunk (queues, point words, row tables) and the chunk's points are used again by the next
// kernels: evict_last keeps them in L2 while the output rows, which nobody reads back, stream through with evict_first.
__device__ __forceinline__ uint64_t vt_policy_keep() { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p)); return p; }
__device__ __forceinline__ uint64_t vt_policy_stream() { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p)); return p; }
__device__ __forceinline__ uint32_t vt_ld32(const void *p, uint64_t pol)
{
    uint32_t v;
    asm volatile("ld.global.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ uint2 vt_ld64(const void *p, uint64_t pol)
{
    uint2 v;
    asm volatile("ld.global.L2::cache_hint.v2.u32 {%0,%1}, [%2], %3;" : "=r"(v.x), "=r"(v.y) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ uint4 vt_ld128(const void *p, uint64_t pol)
{
    uint4 v;
    asm volatile("ld.global.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ float4 vt_ldpt(const void *p, uint64_t pol)   // read-only input
{
    float4 v;
    asm volatile("ld.global.nc.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ void vt_st32(void *p, uint32_t v, uint64_t pol) { asm volatile("st.global.L2::cache_hint.u32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory"); }
__device__ __forceinline__ void vt_st64(void *p, uint32_t x, uint32_t y, uint64_t pol)
{
    asm volatile("st.global.L2::cache_hint.v2.u32 [%0], {%1,%2}, %3;" ::"l"(p), "r"(x), "r"(y), "l"(pol) : "memory");
}
__device__ __forceinline__ void vt_st64ll(void *p, long long v, uint64_t pol) { asm volatile("st.global.L2::cache_hint.u64 [%0], %1, %2;" ::"l"(p), "l"(v), "l"(pol) : "memory"); }
__device__ __forceinline__ void vt_st128(void *p, uint4 v, uint64_t pol)
{
    asm volatile("st.global.L2::cache_hint.v4.u32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "l"(pol) : "memory");
}
// programmatic dependent launch: the kernels of a call are chained in one stream; each lets the next one launch while it drains
// and waits for its predecessor's results before it touches global memory
__device__ __forceinline__ void vt_pdl_enter()
{
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;");
}

// Prefix of a scan tile over the tiles of all frames.  Every tile of a chunk publishes its own sums (flag 1) and then adds up the
// sums of the chunk's earlier tiles, one per thread -- a single round trip instead of a chain of look-back rounds; the chunk
// starts from the inclusive prefix its predecessor's last tile left behind (flag 2, written by an earlier kernel).  Tiles take
// their numbers from a ticket counter, so a tile only waits for tiles that are running or done.
__device__ __forceinline__ unsigned long long vt_tile_prefix(unsigned long long *state, int64_t g0, int64_t gt, int64_t glast, unsigned long long mine,
                                                             unsigned long long *red)
{
    const unsigned tid = threadIdx.x, lane = tid & 31u, w = tid >> 5;
    if (tid == 0 && gt != glast) vt_st_release(state + gt, (1ull << 62) | mine);   // the chunk's last tile has no successor inside the chunk
    unsigned long long x = 0;
    for (int64_t j = g0 + tid; j < gt; j += VT_THREADS) {
        unsigned long long v;
        while (((v = vt_ld_acquire(state + j)) >> 62) == 0ull) __nanosleep(40);
        x += v & VT_PVAL;
    }
    if (tid == 0 && g0 > 0) x += vt_ld_acquire(state + g0 - 1) & VT_PVAL;
#pragma unroll
    for (int d = 16; d; d >>= 1) x += __shfl_xor_sync(0xffffffffu, x, d);
    if (lane == 0) red[w] = x;
    __syncthreads();
    unsigned long long excl = 0;
#pragma unroll
    for (int k = 0; k < VT_WARPS; k++) excl += red[k];
    if (tid == 0 && gt == glast) vt_st_release(state + gt, (2ull << 62) | (excl + mine));
    return excl;
}

__device__ __forceinline__ uint32_t vt_bucket(uint32_t key, uint32_t lgP) { return lgP ? (key * 0x9E3779B1u) >> (32u - lgP) : 0u; }
__device__ __forceinline__ uint32_t vt_home(uint32_t key, uint32_t hshift) { return (key * 0x85EBCA6Bu) >> hshift; }

// what a point's word says (shared by scan and write)
__device__ __forceinline__ void vt_decode(const VtArgs &a, uint32_t w, bool *head, bool *keep)
{
    const uint32_t cat = w >> 30;
    *head = ((cat + 1u) & 3u) < 2u;      // categories 0 and 3
    *keep = cat != 1u && !a.dropall;
}

// ------------------------------------------------------------------------------------------------ split
template <bool NF4>
__global__ void __launch_bounds__(VT_THREADS, D3D_VT_SCTAS) vt_split_kernel(const VtArgs a, const VcDev dv, uint32_t chunk)
{
    extern __shared__ __align__(16) unsigned char vt_dyn[];
    vt_pdl_enter();
    const VtGeom &g = a.g;
    const unsigned tid = threadIdx.x;
    const uint32_t fl = blockIdx.y, t = blockIdx.x;
    const int64_t f = (int64_t)chunk * g.CF + fl;
    const int64_t b = a.offs[f];
    const uint32_t L = (uint32_t)min((long long)(a.offs[f + 1] - b), (long long)g.lmax);
    const uint32_t t0 = t * VT_TILE;
    if (t0 >= L) return;
    const uint64_t keep = vt_policy_keep();

    uint32_t *hist = reinterpret_cast<uint32_t *>(vt_dyn), *base = hist + g.P;
    uint32_t *word = a.word + (size_t)fl * g.lpad;
    uint32_t *qcount = a.qcount + (size_t)fl * g.P;
    uint2 *queue = a.queue + (size_t)fl * g.P * g.qcap;

    for (uint32_t p = tid; p < g.P; p += VT_THREADS) hist[p] = 0;
    __syncthreads();

    float4 p4[VT_PPT];
    bool in[VT_PPT];
#pragma unroll
    for (int u = 0; u < VT_PPT; u++) {
        const uint32_t i = t0 + u * VT_THREADS + tid;
        in[u] = i < L;
        p4[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (in[u]) {
            if (NF4) p4[u] = vt_ldpt(reinterpret_cast<const float4 *>(a.pts) + b + i, keep);   // read again by the write kernel
            else { const float *q = a.pts + (b + i) * a.nfeat; p4[u] = make_float4(q[0], q[1], q[2], 0.f); }
        }
    }
    uint32_t keys[VT_PPT], rank[VT_PPT];
#pragma unroll
    for (int u = 0; u < VT_PPT; u++) {
        uint32_t key;
        const bool ok = vc_cell<false>(dv, p4[u], &key) && in[u];
        keys[u] = ok ? key : VC_NOKEY;
        rank[u] = 0;
        if (in[u]) vt_st32(word + t0 + u * VT_THREADS + tid, (ok && a.single_ok) ? key : VT_W_NONE, keep);   // min_points > 1: a lone point is dropped
        if (ok) rank[u] = atomicAdd(&hist[vt_bucket(key, g.lgP)], 1u);
    }
    __syncthreads();
    for (uint32_t p = tid; p < g.P; p += VT_THREADS) {
        const uint32_t c = hist[p];
        base[p] = c ? atomicAdd(&qcount[p], c) : 0u;
    }
    __syncthreads();
    bool over = false;
#pragma unroll
    for (int u = 0; u < VT_PPT; u++) {
        if (keys[u] != VC_NOKEY) {
            const uint32_t bk = vt_bucket(keys[u], g.lgP);
            const uint32_t pos = base[bk] + rank[u];
            if (pos < g.qcap) vt_st64(queue + bk * g.qcap + pos, keys[u], t0 + u * VT_THREADS + tid, keep);
            else over = true;
        }
    }
    if (over) *a.bail = 1u;
}

// ------------------------------------------------------------------------------------------------ bucket
// table slot s: tkey cell key, tmc {smallest point index, points}, trec record of a crowded voxel
__global__ void __launch_bounds__(VT_BT, D3D_VT_BCTAS) vt_bucket_kernel(const VtArgs a)
{
    // keys apart from the {smallest index, count} pairs: the 32 lanes of a key claim spread over all 32 banks, those of the other two atomics over
    // 16 (16-byte slots put every field on 8 of them), and a lookup reads its pair with one load
    __shared__ __align__(16) uint32_t tkey[VT_SMAX], trec[VT_SMAX];
    __shared__ __align__(16) uint2 tmc[VT_SMAX];   // the pair every lookup reads comes with one 64-bit load
    __shared__ uint32_t pool[VT_POOL * VT_MAXK];   // records of VT_MAXK indices
    __shared__ uint32_t misc[4];                   // [1] records in use, [2] failure
    const VtGeom &g = a.g;
    const unsigned tid = threadIdx.x;
    const uint32_t fl = blockIdx.y, bk = blockIdx.x;
    const uint32_t K = a.K, cthr = a.cthr;
    uint32_t *qcount = a.qcount + (size_t)fl * g.P;
    const uint2 *q = a.queue + ((size_t)fl * g.P + bk) * g.qcap;
    uint32_t *word = a.word + (size_t)fl * g.lpad, *hkey = a.hkey + (size_t)fl * g.lpad;

    vt_pdl_enter();
    const uint64_t keep = vt_policy_keep();
    const uint32_t n = min(qcount[bk], g.qcap);
    if (n == 0) return;
    // the thread's entries e = tid, tid + 128, ... < n stay in registers; every loop over them stops at the bucket's count (CTA-uniform):
    // an ordinary bucket holds ~2.6 per thread
    uint2 en[VT_EPT];
#pragma unroll
    for (int k = 0; k < VT_EPT; k++) {
        en[k] = make_uint2(VT_NONE, 0u);
        if (k * VT_BT >= n) break;
        if (tid + k * VT_BT < n) en[k] = vt_ld64(q + tid + k * VT_BT, keep);
    }
    // table size for this bucket: load factor <= 2/3 when the maximum allows it
    uint32_t lgS = 32u - (uint32_t)__clz((int)(n + (n >> 1)));
    lgS = lgS < 6u ? 6u : lgS;
    if ((1u << lgS) > (uint32_t)VT_SMAX) lgS = 31u - (uint32_t)__clz(VT_SMAX);
    const uint32_t S = 1u << lgS, smask = S - 1, hshift = 32u - lgS;
    for (uint32_t s = tid; s < S / 4; s += VT_BT) {
        reinterpret_cast<uint4 *>(tkey)[s] = make_uint4(VT_NONE, VT_NONE, VT_NONE, VT_NONE);
        reinterpret_cast<uint4 *>(tmc)[2 * s] = make_uint4(VT_NONE, 0u, VT_NONE, 0u);
        reinterpret_cast<uint4 *>(tmc)[2 * s + 1] = make_uint4(VT_NONE, 0u, VT_NONE, 0u);
    }
    if (tid == 0) { misc[1] = 0; misc[2] = 0; }
    __syncthreads();
    if (tid == 0) qcount[bk] = 0;   // everybody has read it: the counter is ready for the next chunk
    if (n > S) { if (tid == 0) *a.bail = 1u; return; }   // (n is CTA-uniform)

    // per-entry steps; the first VT_EPT entries of a thread live in registers with their slot, the rest of a long queue (rare) is read
    // again from the queue and finds its slot by probing
    bool anyc = false;
    // counts the point; the (K+1)-th arrival of a voxel opens the record of its K smallest indices (exactly one thread sees the count step
    // from K to K+1, and the records are only read after the next barrier)
    auto count_and_open = [&](const uint32_t s) {
        const uint32_t c = atomicAdd(&tmc[s].y, 1u);
        if (c >= cthr) {
            anyc = true;
            if (c == cthr) {
                const uint32_t r = atomicAdd(&misc[1], 1u);
                if (r >= (uint32_t)VT_POOL) misc[2] = 1u;
                else {
                    trec[s] = r;
                    for (uint32_t j = 0; j < K; j++) pool[r * VT_MAXK + j] = VT_NONE;
                }
            }
        }
    };
    auto insert = [&](const uint2 x) -> uint32_t {
        uint32_t s = vt_home(x.x, hshift);
        for (uint32_t it = 0; it <= S; it++) {
            const uint32_t old = atomicCAS(&tkey[s], VT_NONE, x.x);
            if (old == VT_NONE || old == x.x) break;
            s = (s + 1) & smask;
        }
        atomicMin(&tmc[s].x, x.y);
        count_and_open(s);
        return s;
    };
    auto find = [&](const uint32_t key) -> uint32_t {
        uint32_t s = vt_home(key, hshift);
        while (tkey[s] != key) s = (s + 1) & smask;
        return s;
    };
    auto cascade = [&](const uint2 x, const uint32_t s) {
        const uint2 mc = tmc[s];
        const uint4 t = make_uint4(0u, mc.x, mc.y, 0u);
        if (t.z > cthr && x.y != t.y) {   // the smallest index is already known: the record keeps the next K - 1
            uint32_t *rec = pool + trec[s] * VT_MAXK;
            uint32_t v = x.y;
            for (uint32_t j = 0; j + 1 < K; j++) {
                const uint32_t old = atomicMin(&rec[j], v);
                v = max(old, v);              // the larger value moves on to the next level
                if (v == VT_NONE) break;
            }
        }
    };
    auto reply = [&](const uint2 x, const uint32_t s) {
        const uint2 mc = tmc[s];
        const uint4 t = make_uint4(0u, mc.x, mc.y, 0u);
        if (t.z != 1u) {
            uint32_t r;
            if ((long long)t.z < (long long)a.min_points) r = VT_W_NONE;
            else if (x.y == t.y) { r = VT_W_HEAD | min(t.z, VT_VAL); vt_st32(hkey + x.y, x.x, keep); }
            else {
                const bool kept = !(t.z > cthr) || (K >= 2u && x.y <= pool[trec[s] * VT_MAXK + K - 2]);
                r = kept ? (VT_W_JOIN | t.y) : VT_W_NONE;
            }
            vt_st32(word + x.y, r, keep);
        }
    };
    const uint32_t rest = tid + VT_EPT * VT_BT;   // this thread's first entry beyond the registers

    // the home-slot claims of the thread's register entries are issued back to back (independent atomics in flight), then the few that
    // met another voxel's key walk on
    uint32_t sl[VT_EPT], first[VT_EPT];
#pragma unroll
    for (int k = 0; k < VT_EPT; k++) {
        sl[k] = 0; first[k] = VT_NONE;
        if (k * VT_BT >= n) break;
        if (tid + k * VT_BT < n) { sl[k] = vt_home(en[k].x, hshift); first[k] = atomicCAS(&tkey[sl[k]], VT_NONE, en[k].x); }
    }
#pragma unroll
    for (int k = 0; k < VT_EPT; k++) {
        if (k * VT_BT >= n) break;
        if (tid + k * VT_BT < n) {
            uint32_t s = sl[k], old = first[k];
            for (uint32_t it = 0; it <= S && !(old == VT_NONE || old == en[k].x); it++) {
                s = (s + 1) & smask;
                old = atomicCAS(&tkey[s], VT_NONE, en[k].x);
            }
            atomicMin(&tmc[s].x, en[k].y);
            count_and_open(s);
            sl[k] = s;
        }
    }
    for (uint32_t e = rest; e < n; e += VT_BT) insert(vt_ld64(q + e, keep));
    // voxels with more than K points: their K smallest indices
    if (__syncthreads_or((int)anyc)) {
        if (misc[2]) { if (tid == 0) *a.bail = 1u; return; }
#pragma unroll
        for (int k = 0; k < VT_EPT; k++) {
            if (k * VT_BT >= n) break;
            if (tid + k * VT_BT < n) cascade(en[k], sl[k]);
        }
        for (uint32_t e = rest; e < n; e += VT_BT) { const uint2 x = vt_ld64(q + e, keep); cascade(x, find(x.x)); }
        __syncthreads();
    }

    // a new word for every point that shares its voxel (a point that hears nothing is the only point of its voxel)
#pragma unroll
    for (int k = 0; k < VT_EPT; k++) {
        if (k * VT_BT >= n) break;
        if (tid + k * VT_BT < n) reply(en[k], sl[k]);
    }
    for (uint32_t e = rest; e < n; e += VT_BT) { const uint2 x = vt_ld64(q + e, keep); reply(x, find(x.x)); }
}

// ------------------------------------------------------------------------------------------------ scan
// row table entry: .x first-of-voxel bits of the 32-point row, .y voxel rows before the row, .z keep bits, .w kept rows before the row
__global__ void __launch_bounds__(VT_THREADS) vt_scan_kernel(const VtArgs a, uint32_t chunk)
{
    const VtGeom &g = a.g;
    const unsigned tid = threadIdx.x, lane = tid & 31u, w = tid >> 5;
    __shared__ unsigned long long wsum[VT_WARPS], red[VT_WARPS];
    __shared__ uint32_t s_misc[2];
    vt_pdl_enter();
    const uint64_t keepp = vt_policy_keep();

    if (tid == 0) s_misc[0] = atomicAdd(&a.tickets[chunk], 1u);
    __syncthreads();
    const uint32_t lt = s_misc[0];
    const uint32_t fl = lt / g.spf, t = lt - fl * g.spf;
    const int64_t f = (int64_t)chunk * g.CF + fl;
    const int64_t gt = f * (int64_t)g.spf + t;
    const uint32_t L = (uint32_t)min((long long)(a.offs[f + 1] - a.offs[f]), (long long)g.lmax);
    const uint32_t t0 = t * VT_STILE;
    const uint32_t *word = a.word + (size_t)fl * g.lpad;
    uint4 *ri_f = a.rowinfo + (size_t)fl * (g.lpad / 32);

    // lane u of a warp keeps the bits of the warp's row u
    uint32_t myh = 0, myk = 0;
#pragma unroll
    for (int u = 0; u < VT_SPT; u++) {
        const uint32_t i = t0 + (w * VT_SPT + u) * 32 + lane;
        const uint32_t x = i < L ? vt_ld32(word + i, keepp) : VT_W_NONE;
        bool head, keep;
        vt_decode(a, x, &head, &keep);
        const uint32_t hb = __ballot_sync(0xffffffffu, head), kb = __ballot_sync(0xffffffffu, keep);
        if (lane == (unsigned)u) { myh = hb; myk = kb; }
    }
    // inclusive prefix over the rows of the warp
    uint32_t ih = __popc(myh), ik = __popc(myk);
#pragma unroll
    for (int d = 1; d < VT_SPT; d <<= 1) {
        const uint32_t xh = __shfl_up_sync(0xffffffffu, ih, d), xk = __shfl_up_sync(0xffffffffu, ik, d);
        if (lane >= (unsigned)d) { ih += xh; ik += xk; }
    }
    if (lane == 31) wsum[w] = ((unsigned long long)ik << 31) | ih;
    __syncthreads();
    unsigned long long total = 0, wex = 0;
#pragma unroll
    for (int k = 0; k < VT_WARPS; k++) { if ((unsigned)k == w) wex = total; total += wsum[k]; }
    const int64_t g0 = (int64_t)chunk * g.CF * g.spf;
    const int64_t nfc = min((int64_t)g.CF, a.nframes - (int64_t)chunk * g.CF);
    const unsigned long long ex = vt_tile_prefix(a.status, g0, gt, g0 + nfc * g.spf - 1, total, red);
    if (tid == 0) {
        if (t == 0) { a.counts[2 * f] = (long long)((ex >> 31) & VT_F31); a.counts[2 * f + 1] = (long long)(ex & VT_F31); }
        if (gt == a.nframes * (int64_t)g.spf - 1) {
            const unsigned long long e2 = ex + total;
            a.counts[2 * a.nframes] = (long long)((e2 >> 31) & VT_F31); a.counts[2 * a.nframes + 1] = (long long)(e2 & VT_F31);
        }
    }
    const unsigned long long run0 = ex + wex;
    const uint32_t Gh = ((uint32_t)run0 & VT_F31) + ih - __popc(myh), Gk = ((uint32_t)(run0 >> 31) & VT_F31) + ik - __popc(myk);
    vt_st128(ri_f + t * (VT_STILE / 32) + w * VT_SPT + lane, make_uint4(myh, Gh, myk, Gk), keepp);   // rows past the frame hold zero bits: harmless
}

// ------------------------------------------------------------------------------------------------ write
template <bool NF4>
__global__ void __launch_bounds__(VT_THREADS, D3D_VT_WCTAS) vt_write_kernel(const VtArgs a, const VcDev dv, uint32_t chunk)
{
    vt_pdl_enter();
    const VtGeom &g = a.g;
    const unsigned tid = threadIdx.x, lane = tid & 31u, w = tid >> 5;
    const unsigned ltmask = lanemask_lt();
    const uint32_t fl = blockIdx.y, t = blockIdx.x;
    const int64_t f = (int64_t)chunk * g.CF + fl;
    const int64_t b = a.offs[f];
    const uint32_t L = (uint32_t)min((long long)(a.offs[f + 1] - b), (long long)g.lmax);
    const uint32_t t0 = t * VT_TILE;
    if (t0 >= L) return;
    const uint64_t keepp = vt_policy_keep(), strm = vt_policy_stream();
    const uint32_t vb = (uint32_t)a.counts[2 * f + 1];   // the frame's first voxel row
    const uint32_t *word = a.word + (size_t)fl * g.lpad, *hkey = a.hkey + (size_t)fl * g.lpad;
    const uint4 *ri_f = a.rowinfo + (size_t)fl * (g.lpad / 32);
    const uint32_t row0 = (t0 >> 5) + w * VT_PPT;
    if (row0 * 32 >= L) return;
    const uint32_t mask_y = (1u << (dv.sh_x - dv.sh_y)) - 1u, mask_z = (1u << dv.sh_y) - 1u;

    // first round trip: words, row table entries (lane u holds row u's) and the points of the warp's four rows, unconditionally
    uint32_t wd[VT_PPT];
    float4 p4[VT_PPT];
    const uint4 rme = vt_ld128(ri_f + row0 + (lane & (VT_PPT - 1)), keepp);
#pragma unroll
    for (int u = 0; u < VT_PPT; u++) {
        const uint32_t i = (row0 + u) * 32 + lane;
        wd[u] = i < L ? vt_ld32(word + i, keepp) : VT_W_NONE;
        p4[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (NF4 && i < L) p4[u] = vt_ldpt(reinterpret_cast<const float4 *>(a.pts) + b + i, strm);   // last use
    }
    // second round trip, few lanes: keys of first points of shared voxels, row table entries of the joiners' first points
    uint32_t ckey[VT_PPT];
    uint2 rj[VT_PPT];
#pragma unroll
    for (int u = 0; u < VT_PPT; u++) {
        const uint32_t i = (row0 + u) * 32 + lane;
        const uint32_t cat = wd[u] >> 30;
        ckey[u] = wd[u]; rj[u] = make_uint2(0u, 0u);
        if (cat == 3u) ckey[u] = vt_ld32(hkey + i, keepp);
        if (cat == 2u) rj[u] = vt_ld64(ri_f + ((wd[u] & VT_VAL) >> 5), keepp);   // the id lives where the voxel's first point lives
    }
#pragma unroll
    for (int u = 0; u < VT_PPT; u++) {
        const uint32_t i = (row0 + u) * 32 + lane;
        const uint32_t x = wd[u];
        bool head, keep;
        vt_decode(a, x, &head, &keep);
        const uint32_t hb = __shfl_sync(0xffffffffu, rme.x, u), gh = __shfl_sync(0xffffffffu, rme.y, u);
        const uint32_t kb = __shfl_sync(0xffffffffu, rme.z, u), gk = __shfl_sync(0xffffffffu, rme.w, u);
        uint32_t vrow = 0;
        if (head) {
            vrow = gh + __popc(hb & ltmask);
            const uint32_t c = (x >> 30) ? (x & VT_VAL) : 1u, key = ckey[u];
            long long *co = reinterpret_cast<long long *>(a.out_coords) + (size_t)vrow * 3;
            vt_st64ll(co + 0, (long long)(key >> dv.sh_x) + dv.cadd[0], strm);
            vt_st64ll(co + 1, (long long)((key >> dv.sh_y) & mask_y) + dv.cadd[1], strm);
            vt_st64ll(co + 2, (long long)(key & mask_z) + dv.cadd[2], strm);
            vt_st32(a.out_npoints + vrow, (a.trim && c > a.K) ? a.K : c, strm);
        } else if (keep) {
            const uint32_t m = x & VT_VAL;
            vrow = rj[u].y + __popc(rj[u].x & ((1u << (m & 31u)) - 1u));
        }
        if (keep) {
            const size_t o = (size_t)gk + __popc(kb & ltmask);
            if (NF4) vt_st128(reinterpret_cast<float4 *>(a.out_points) + o, make_uint4(__float_as_uint(p4[u].x), __float_as_uint(p4[u].y), __float_as_uint(p4[u].z), __float_as_uint(p4[u].w)), strm);
            else for (int q = 0; q < a.nfeat; q++) a.out_points[o * a.nfeat + q] = a.pts[(b + i) * a.nfeat + q];
            vt_st64ll(reinterpret_cast<long long *>(a.out_mask) + o, (long long)i, strm);
            vt_st64ll(reinterpret_cast<long long *>(a.out_mapping) + o, (long long)(vrow - vb), strm);
        }
    }
}

// ------------------------------------------------------------------------------------------------ host side
static uint32_t vt_lg2_ceil(uint64_t x) { uint32_t l = 0; while ((1ull << l) < x) l++; return l; }

static bool vt_geom(int64_t max_frame_points, int64_t nframes, VtGeom *g)
{
    if (max_frame_points < 1) max_frame_points = 1;
    if (max_frame_points > (1ll << 21)) return false;            // 4096 buckets of 512 points
    g->lmax = (uint32_t)max_frame_points;
    g->tpf = (g->lmax + VT_TILE - 1) / VT_TILE;
    g->spf = (g->lmax + VT_STILE - 1) / VT_STILE;
    g->lpad = g->spf * VT_STILE;
    g->lgP = vt_lg2_ceil(((uint64_t)g->lmax + D3D_VT_BPTS - 1) / D3D_VT_BPTS);
    g->P = 1u << g->lgP;
    const uint32_t per = (g->lmax + g->P - 1) / g->P;            // points per bucket if every point is kept and the hash is even (<= 512)
    g->qcap = (per + per / 2 + 128 + 15) & ~15u;                 // multiple of 16 entries: every bucket's queue starts on a 128-byte line
    if (g->qcap > (uint32_t)VT_QCAP) g->qcap = VT_QCAP;
    int cf = 64;    // measured on C2 x 128 frames (one stream): 0.74 ms with chunks of 16 (scratch mostly L2-resident), 0.59 ms with one chunk of 128 (fewer, fuller launches)
    if ((int64_t)cf > nframes) cf = (int)(nframes > 0 ? nframes : 1);
    g->CF = (uint32_t)cf;
    g->nchunks = (uint32_t)((nframes + cf - 1) / cf);
    if ((int64_t)nframes * g->tpf >= (1ll << 31)) return false;
    return true;
}

struct VtLayout { size_t queue, word, hkey, rowinfo, zero, qcount, status, tickets, bail, zero_end, total; };

static VtLayout vt_layout(const VtGeom &g, int64_t nframes)
{
    VtLayout l;
    const size_t slots = (size_t)g.CF * (g.nchunks > 1 ? 2 : 1);   // two chunks in flight on two internal streams
    size_t o = 0;
    l.queue = o;   o += align_up(slots * g.P * g.qcap * sizeof(uint2));
    l.word = o;    o += align_up(slots * g.lpad * 4);
    l.hkey = o;    o += align_up(slots * g.lpad * 4);
    l.rowinfo = o; o += align_up(slots * (g.lpad / 32) * sizeof(uint4));
    l.zero = o;
    l.qcount = o;  o += align_up(slots * g.P * 4);
    l.status = o;  o += align_up((size_t)(nframes > 0 ? nframes : 1) * g.spf * 8);
    l.tickets = o; o += align_up((size_t)g.nchunks * 4);
    l.bail = o;    o += 256;
    l.zero_end = o;
    l.total = o;
    return l;
}

// two internal streams + events per device (created once; the library's only long-lived CUDA objects)
struct VtLanes { cudaStream_t s[2]; cudaEvent_t fork, scan_done[2], join[2]; std::mutex mu; bool ok; };
static VtLanes *vt_lanes()
{
    static VtLanes pool[64];
    static std::mutex init_mu;
    static bool made[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); return nullptr; }
    std::lock_guard<std::mutex> gd(init_mu);
    VtLanes &L = pool[dev];
    if (!made[dev]) {
        made[dev] = true;
        L.ok = true;
        for (int i = 0; i < 2; i++) {
            L.ok = L.ok && cudaStreamCreateWithFlags(&L.s[i], cudaStreamNonBlocking) == cudaSuccess;
            L.ok = L.ok && cudaEventCreateWithFlags(&L.scan_done[i], cudaEventDisableTiming) == cudaSuccess;
            L.ok = L.ok && cudaEventCreateWithFlags(&L.join[i], cudaEventDisableTiming) == cudaSuccess;
        }
        L.ok = L.ok && cudaEventCreateWithFlags(&L.fork, cudaEventDisableTiming) == cudaSuccess;
        if (!L.ok) cudaGetLastError();
    }
    return L.ok ? &L : nullptr;
}

bool vox_tiles_supported(const VoxCfg &cfg, int64_t total, int64_t nframes, int64_t max_frame_points)
{
    VcDev d;
    VtGeom g;
    if (cfg.dense || !vc_make_dev(cfg, &d)) return false;
    if (d.sh_x + (uint32_t)vox_bits_for(cfg.ext[0]) > 30u) return false;                // the point words keep two bits for the category
    if (cfg.vfilter != D3D_VF_NONE) return false;                                  // a voxel cap makes the keep decision depend on the ids
    if (cfg.pfilter == D3D_PF_TRIM && cfg.max_points > VT_MAXK) return false;
    if (cfg.pfilter != D3D_PF_TRIM && cfg.pfilter != D3D_PF_NONE) return false;
    if (!vox_cluster_supported(cfg, total, nframes, max_frame_points)) return false;   // the fallback behind the device flag
    return vt_geom(max_frame_points, nframes, &g);
}

size_t vox_tiles_ws_bytes(int64_t total, int64_t nframes, int64_t max_frame_points)
{
    if (max_frame_points <= 0 || max_frame_points > total) max_frame_points = total;
    VtGeom g;
    if (!vt_geom(max_frame_points, nframes, &g)) return 0;
    return align_up(vt_layout(g, nframes).total) + 256 + vox_cluster_ws_bytes(total, nframes, max_frame_points);
}

int vox_tiles_sparse(const float *points, int64_t total, int nfeat, const int64_t *offs, int64_t nframes, int64_t max_frame_points, const VoxCfg &cfg,
                     float *out_points, int64_t *out_mask, int64_t *out_mapping, int32_t *out_npoints, int64_t *out_coords, int64_t *counts,
                     void *ws, size_t ws_bytes, cudaStream_t st)
{
    if (max_frame_points <= 0 || max_frame_points > total) max_frame_points = total;
    VtGeom g;
    VcDev dv;
    if (!vt_geom(max_frame_points, nframes, &g) || !vc_make_dev(cfg, &dv)) return D3D_ERR_UNSUPPORTED;
    const VtLayout lay = vt_layout(g, nframes);
    const size_t mine = align_up(lay.total);
    if (ws_bytes < mine + vox_cluster_ws_bytes(total > 0 ? total : 1, nframes, max_frame_points)) return D3D_ERR_WORKSPACE;
    char *w = (char *)ws;
    VtArgs a = {};
    a.pts = points; a.nfeat = nfeat; a.offs = offs; a.nframes = nframes;
    a.out_points = out_points; a.out_mask = out_mask; a.out_mapping = out_mapping; a.out_npoints = out_npoints; a.out_coords = out_coords; a.counts = counts;
    a.queue = (uint2 *)(w + lay.queue); a.word = (uint32_t *)(w + lay.word); a.hkey = (uint32_t *)(w + lay.hkey);
    a.rowinfo = (uint4 *)(w + lay.rowinfo); a.qcount = (uint32_t *)(w + lay.qcount);
    a.status = (unsigned long long *)(w + lay.status); a.tickets = (uint32_t *)(w + lay.tickets); a.bail = (uint32_t *)(w + lay.bail);
    a.g = g;
    const bool trim = cfg.pfilter == D3D_PF_TRIM;
    a.K = cfg.max_points > 0 ? (uint32_t)cfg.max_points : 0u;
    a.trim = trim ? 1 : 0;
    a.dropall = (trim && a.K == 0) ? 1 : 0;
    a.cthr = (trim && a.K > 0) ? a.K : VT_NONE;
    a.min_points = cfg.min_points;
    a.single_ok = cfg.min_points <= 1 ? 1 : 0;

    D3D_CUDA_TRY(cudaMemsetAsync(w + lay.zero, 0, lay.zero_end - lay.zero, st));
    // Two chunks are in flight at a time, each on its own internal stream with its own scratch: the four kernels of a chunk have
    // different bottlenecks (issue slots, shared-memory latency, a short dependent chain, DRAM stores) and fill each other's tails.
    // Inside a stream the kernels are chained with programmatic dependent launch (each may be scheduled while its predecessor
    // drains and waits, griddepcontrol.wait, for the predecessor's results); the scan of chunk c waits for the scan of chunk c-1
    // (packed output rows) through an event.  The caller's stream forks into the two lanes and joins them again: the call stays
    // asynchronous and ordered on the caller's stream.
    VtLanes *lanes = g.nchunks > 1 ? vt_lanes() : nullptr;
    std::unique_lock<std::mutex> lock;
    cudaStream_t lane_stream[2] = {st, st};
    if (lanes) {
        lock = std::unique_lock<std::mutex>(lanes->mu);
        D3D_CUDA_TRY(cudaEventRecord(lanes->fork, st));
        for (int i = 0; i < 2; i++) { lane_stream[i] = lanes->s[i]; D3D_CUDA_TRY(cudaStreamWaitEvent(lanes->s[i], lanes->fork, 0)); }
    }
    cudaLaunchAttribute pdl[1];
    pdl[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pdl[0].val.programmaticStreamSerializationAllowed = 1;
    const uint32_t dyn_split = 8u * g.P;
    for (uint32_t c = 0; c < g.nchunks; c++) {
        const int64_t rem = nframes - (int64_t)c * g.CF;
        const uint32_t nf = (uint32_t)(rem < (int64_t)g.CF ? rem : g.CF);
        const int ln = lanes ? (int)(c & 1u) : 0;
        cudaStream_t cs = lane_stream[ln];
        VtArgs al = a;   // this lane's scratch
        al.queue += (size_t)ln * g.CF * g.P * g.qcap; al.word += (size_t)ln * g.CF * g.lpad; al.hkey += (size_t)ln * g.CF * g.lpad;
        al.rowinfo += (size_t)ln * g.CF * (g.lpad / 32); al.qcount += (size_t)ln * g.CF * g.P;
        auto cfg_of = [&](dim3 grid, unsigned threads, size_t smem) {
            cudaLaunchConfig_t lc = {};
            lc.gridDim = grid; lc.blockDim = dim3(threads, 1, 1); lc.dynamicSmemBytes = smem; lc.stream = cs;
            lc.attrs = pdl; lc.numAttrs = 1;
            return lc;
        };
        {
            cudaLaunchConfig_t lc = cfg_of(dim3(g.tpf, nf), VT_THREADS, dyn_split);
            if (nfeat == 4) D3D_CUDA_TRY(cudaLaunchKernelEx(&lc, vt_split_kernel<true>, al, dv, c));
            else D3D_CUDA_TRY(cudaLaunchKernelEx(&lc, vt_split_kernel<false>, al, dv, c));
            D3D_LAUNCHED();
        }
        { cudaLaunchConfig_t lc = cfg_of(dim3(g.P, nf), VT_BT, 0); D3D_CUDA_TRY(cudaLaunchKernelEx(&lc, vt_bucket_kernel, al)); D3D_LAUNCHED(); }
        if (lanes && c > 0) D3D_CUDA_TRY(cudaStreamWaitEvent(cs, lanes->scan_done[(c - 1) & 1u], 0));
        {
            cudaLaunchConfig_t lc = cfg_of(dim3(nf * g.spf), VT_THREADS, 0);
            if (lanes && c > 0) lc.numAttrs = 0;   // its predecessor in the other lane is a full dependency (event), not a programmatic one
            D3D_CUDA_TRY(cudaLaunchKernelEx(&lc, vt_scan_kernel, al, c)); D3D_LAUNCHED();
        }
        if (lanes) D3D_CUDA_TRY(cudaEventRecord(lanes->scan_done[c & 1u], cs));
        {
            cudaLaunchConfig_t lc = cfg_of(dim3(g.tpf, nf), VT_THREADS, 0);
            if (lanes) lc.numAttrs = 0;            // an event record sits between the scan and this launch
            if (nfeat == 4) D3D_CUDA_TRY(cudaLaunchKernelEx(&lc, vt_write_kernel<true>, al, dv, c));
            else D3D_CUDA_TRY(cudaLaunchKernelEx(&lc, vt_write_kernel<false>, al, dv, c));
            D3D_LAUNCHED();
        }
    }
    if (lanes) {
        for (int i = 0; i < 2; i++) { D3D_CUDA_TRY(cudaEventRecord(lanes->join[i], lanes->s[i])); D3D_CUDA_TRY(cudaStreamWaitEvent(st, lanes->join[i], 0)); }
        lock.unlock();
    }
    // the batch is redone by the cluster kernel when a queue, a table or a record pool overflowed (device flag)
    return vox_cluster_sparse(points, total, nfeat, offs, nframes, max_frame_points, cfg, out_points, out_mask, out_mapping, out_npoints, out_coords, counts,
                              w + mine, ws_bytes - mine, st, a.bail);
}

}  // namespace d3d
