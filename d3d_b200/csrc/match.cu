// match.cu -- greedy score-ordered matching over a distance matrix (SURVEY.md 8(f) row f1, second half).
//
// Replaces the pair walk of ScoreMatcher.match + BaseMatcher.match_by_order (reference d3d/tracking/matcher.pyx:93-122, 138-162), which
// the detection evaluator runs once per score threshold on the distance cache of prepare_boxes (d3d/benchmarks.pyx:220-238): source
// boxes are visited from the best score down, each takes the closest destination box of its own category that is still free and not
// farther than the category's threshold.  The walk is sequential in the sources, so one CTA owns one threshold set (the evaluator's
// 40 thresholds are 40 CTAs of one launch) and spends two barriers per source: all threads scan the row for the nearest free
// candidate, one thread commits it.  Ties in the distance go to the lower destination index (the reference's np.argsort leaves them
// unspecified).
#include "common.cuh"

namespace d3d {

constexpr int MT_THREADS = 256;

__device__ __forceinline__ unsigned long long mt_key(float d, uint32_t j)
{
    uint32_t u = __float_as_uint(d);
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);   // ascending order-preserving
    return ((unsigned long long)u << 32) | j;
}

__global__ void __launch_bounds__(MT_THREADS) match_greedy_kernel(const float *__restrict__ dist, int64_t n, int64_t m, int64_t ld, const int32_t *__restrict__ src_order,
                                                                  const int32_t *__restrict__ src_tag, const int32_t *__restrict__ dst_tag,
                                                                  const float *__restrict__ thresholds, int32_t ncat, int32_t *__restrict__ src_assign,
                                                                  int32_t *__restrict__ dst_assign)
{
    extern __shared__ unsigned char taken[];   // [m] destination already assigned
    __shared__ unsigned long long s_best[MT_THREADS / 32];
    const int t = blockIdx.x, tid = threadIdx.x;
    int32_t *sa = src_assign + (int64_t)t * n, *da = dst_assign + (int64_t)t * m;
    for (int64_t j = tid; j < m; j += MT_THREADS) { taken[j] = 0; da[j] = -1; }
    for (int64_t i = tid; i < n; i += MT_THREADS) sa[i] = -1;
    __syncthreads();
    for (int64_t p = 0; p < n; p++) {
        const int32_t i = src_order[p];
        const int32_t tag = src_tag[i];
        unsigned long long best = ~0ull;
        if (tag >= 0 && tag < ncat) {
            const float thr = thresholds[(int64_t)t * ncat + tag];
            const float *row = dist + (int64_t)i * ld;
            for (int64_t j = tid; j < m; j += MT_THREADS) {
                if (!taken[j] && dst_tag[j] == tag) {
                    const float d = row[j];
                    if (d <= thr) { const unsigned long long k = mt_key(d, (uint32_t)j); best = k < best ? k : best; }   // NaN never matches, like the reference's <=
                }
            }
        }
#pragma unroll
        for (int s = 16; s; s >>= 1) { const unsigned long long o = __shfl_xor_sync(0xffffffffu, best, s); best = o < best ? o : best; }
        if ((tid & 31) == 0) s_best[tid >> 5] = best;
        __syncthreads();
        if (tid == 0) {
            unsigned long long b = s_best[0];
#pragma unroll
            for (int w = 1; w < MT_THREADS / 32; w++) b = s_best[w] < b ? s_best[w] : b;
            if (b != ~0ull) { const uint32_t j = (uint32_t)b; taken[j] = 1; sa[i] = (int32_t)j; da[j] = i; }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------ frame-batched matching
// One warp walks one (frame, threshold set): the same rule as match_greedy_kernel (key mt_key, d <= thr, sources with a tag outside
// [0, ncat) take nothing) on the frame's block of the packed distance matrix.  An evaluator frame has tens of destinations, so a CTA per
// walk would idle most of its threads behind two barriers per source; a warp keeps its taken flags as a bitmask in shared memory and
// needs no barrier.  Warps of a CTA take consecutive threshold sets of one frame, so they share the frame's block in L1.
constexpr int MTB_WARPS = 4;
constexpr int MTB_MAX_DST = 4096;   // taken bits per warp: 512 bytes

__global__ void __launch_bounds__(MTB_WARPS * 32) match_greedy_batch_kernel(const float *__restrict__ dist, const int64_t *__restrict__ dist_off,
                                                                            const int64_t *__restrict__ src_off, const int64_t *__restrict__ dst_off,
                                                                            int64_t nframes, const int32_t *__restrict__ src_order,
                                                                            const int32_t *__restrict__ src_tag, const int32_t *__restrict__ dst_tag,
                                                                            const float *__restrict__ thresholds, int32_t nsets, int32_t ncat,
                                                                            int32_t *__restrict__ src_assign, int32_t *__restrict__ dst_assign)
{
    __shared__ uint32_t s_taken[MTB_WARPS][MTB_MAX_DST / 32];
    const unsigned lane = lane_id(), w = threadIdx.x >> 5;
    const int64_t g = (int64_t)blockIdx.x * MTB_WARPS + w;
    if (g >= nframes * nsets) return;   // the whole warp
    const int64_t f = g / nsets, t = g % nsets, total_src = src_off[nframes], total_dst = dst_off[nframes];
    const int64_t s0 = src_off[f], n = src_off[f + 1] - s0, d0 = dst_off[f], m = dst_off[f + 1] - d0;
    const float *blk = dist + dist_off[f];
    const int32_t *order = src_order + s0, *stag = src_tag + s0, *dtag = dst_tag + d0;
    const float *thr = thresholds + t * ncat;
    int32_t *sa = src_assign + t * total_src + s0, *da = dst_assign + t * total_dst + d0;
    uint32_t *taken = s_taken[w];
    for (int64_t j = lane; j < (m + 31) / 32 && j < MTB_MAX_DST / 32; j += 32) taken[j] = 0;
    for (int64_t j = lane; j < m; j += 32) da[j] = -1;
    for (int64_t i = lane; i < n; i += 32) sa[i] = -1;
    if (m > MTB_MAX_DST) return;   // a frame over the caller's bound max_frame_dst stays unmatched instead of overrunning the bitmask
    __syncwarp();
    int32_t my_i = 0, my_tag = -1;
    float my_thr = 0.f;
    for (int64_t p = 0; p < n; p++) {
        if ((p & 31) == 0) {   // the next 32 sources of the order, their tags and thresholds: one load each per lane, off the walk's path
            my_tag = -1;
            if (p + lane < n) {
                my_i = order[p + lane];
                my_tag = stag[my_i];
                if (my_tag >= 0 && my_tag < ncat) my_thr = thr[my_tag];
            }
        }
        const int32_t i = __shfl_sync(0xffffffffu, my_i, (int)(p & 31)), tag = __shfl_sync(0xffffffffu, my_tag, (int)(p & 31));
        const float th = __shfl_sync(0xffffffffu, my_thr, (int)(p & 31));
        if (tag < 0 || tag >= ncat) continue;   // uniform over the warp
        const float *row = blk + (int64_t)i * m;
        unsigned long long best = ~0ull;
        for (int64_t j = lane; j < m; j += 32) {
            if (!((taken[j >> 5] >> (j & 31)) & 1u) && dtag[j] == tag) {
                const float d = row[j];
                if (d <= th) { const unsigned long long k = mt_key(d, (uint32_t)j); best = k < best ? k : best; }   // NaN never matches
            }
        }
#pragma unroll
        for (int s = 16; s; s >>= 1) { const unsigned long long o = __shfl_xor_sync(0xffffffffu, best, s); best = o < best ? o : best; }
        if (best != ~0ull) {
            const uint32_t j = (uint32_t)best;
            if (lane == 0) { taken[j >> 5] |= 1u << (j & 31); sa[i] = (int32_t)j; da[j] = i; }
            __syncwarp();
        }
    }
}

}  // namespace d3d

using namespace d3d;
extern "C" int d3d_match_greedy_f32(const float *dist, int64_t n, int64_t m, int64_t ld, const int32_t *src_order, const int32_t *src_tag, const int32_t *dst_tag,
                                    const float *thresholds, int32_t nsets, int32_t ncat, int32_t *src_assign, int32_t *dst_assign, void *stream)
{
    if (n < 0 || m < 0 || nsets < 0 || ncat < 1 || ld < m) return D3D_ERR_INVALID_ARGUMENT;
    if (nsets == 0) return D3D_OK;
    if (!thresholds || (n > 0 && (!src_order || !src_tag || !src_assign)) || (m > 0 && (!dst_tag || !dst_assign)) || (n > 0 && m > 0 && !dist)) return D3D_ERR_INVALID_ARGUMENT;
    if (m > 200 * 1024) return D3D_ERR_UNSUPPORTED;   // one flag byte per destination box in shared memory
    const size_t smem = (size_t)(m > 0 ? m : 1);
    if (smem > 40 * 1024) D3D_CUDA_TRY(cudaFuncSetAttribute(match_greedy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    match_greedy_kernel<<<(unsigned)nsets, MT_THREADS, smem, (cudaStream_t)stream>>>(dist, n, m, ld, src_order, src_tag, dst_tag, thresholds, ncat, src_assign, dst_assign);
    D3D_LAUNCHED();
    return D3D_OK;
}

extern "C" int d3d_match_greedy_batch_f32(const float *dist, const int64_t *dist_offsets, const int64_t *src_offsets, const int64_t *dst_offsets,
                                          int64_t nframes, int64_t max_frame_dst, const int32_t *src_order, const int32_t *src_tag,
                                          const int32_t *dst_tag, const float *thresholds, int32_t nsets, int32_t ncat, int32_t *src_assign,
                                          int32_t *dst_assign, void *stream)
{
    if (nframes < 0 || max_frame_dst < 0 || nsets < 0 || ncat < 1) return D3D_ERR_INVALID_ARGUMENT;
    if (max_frame_dst > MTB_MAX_DST) return D3D_ERR_UNSUPPORTED;   // one taken bit per destination in 512 bytes of shared memory
    if (nframes == 0 || nsets == 0) return D3D_OK;
    if (!dist || !dist_offsets || !src_offsets || !dst_offsets || !src_order || !src_tag || !dst_tag || !thresholds || !src_assign || !dst_assign)
        return D3D_ERR_INVALID_ARGUMENT;
    const int64_t nwalks = nframes * nsets, blocks = (nwalks + MTB_WARPS - 1) / MTB_WARPS;
    if (blocks > 0x7fffffffll) return D3D_ERR_UNSUPPORTED;
    match_greedy_batch_kernel<<<(unsigned)blocks, MTB_WARPS * 32, 0, (cudaStream_t)stream>>>(dist, dist_offsets, src_offsets, dst_offsets, nframes, src_order,
                                                                                               src_tag, dst_tag, thresholds, nsets, ncat, src_assign,
                                                                                               dst_assign);
    D3D_LAUNCHED();
    return D3D_OK;
}
