// core.cu -- library-wide state of libd3d_b200.so: error reporting, launch counter, ALU-peak probe.
#include "common.cuh"
#include <string.h>
#include <stdlib.h>

namespace d3d {
std::atomic<int64_t> g_launches{0};
static thread_local char g_cuda_err[256] = "";
void set_cuda_error(cudaError_t e)
{
    strncpy(g_cuda_err, cudaGetErrorString(e), sizeof(g_cuda_err) - 1);
    g_cuda_err[sizeof(g_cuda_err) - 1] = 0;
}

// Tuning knobs.  The environment is read ONCE, at the first use of a knob (results of a call never depend on the environment at call
// time); tests and tuning tools change a knob through d3d_tuning_set().  Knobs select between back ends that produce identical results;
// the one exception is NMS_STOP, which is for measurement only: it ends d3d_nms2d_* after a phase and leaves the keep mask unwritten.
static const char *const g_tune_names[D3D_TUNE_COUNT] = {"D3D_B200_NMS_PATH", "D3D_B200_CROP_PATH", "D3D_B200_VOX_ROUTE", "D3D_B200_NMS_STOP",
                                                         "D3D_B200_SCATTER_PATH", "D3D_B200_NMS_FIX", "D3D_B200_NMS_BATCH_PATH", "D3D_B200_SORT_COOP"};
static std::atomic<int> g_tune_val[D3D_TUNE_COUNT];
static std::atomic<int> g_tune_state[D3D_TUNE_COUNT];   // 0 unread, 1 unset, 2 set
static int tune_parse(int knob, const char *e)
{
    if (knob == D3D_TUNE_NMS_PATH) return e[0] == 'd' ? 2 : (e[0] == 't' ? 1 : atoi(e));     // dense | tiles | (spatial)
    if (knob == D3D_TUNE_CROP_PATH) return e[0] == 'b' ? 1 : (e[0] == 'g' ? 2 : atoi(e));    // brute | grid | (auto)
    if (knob == D3D_TUNE_NMS_BATCH_PATH) return e[0] == 'd' ? 1 : atoi(e);                  // dense | (edges)
    if (knob == D3D_TUNE_SCATTER_PATH) return e[0] == 'g' ? 1 : (e[0] == 't' ? 2 : atoi(e)); // gather | tiles | (auto)
    return atoi(e);
}
int tuning(int knob, int dflt)
{
    if (knob < 0 || knob >= D3D_TUNE_COUNT) return dflt;
    int st = g_tune_state[knob].load(std::memory_order_acquire);
    if (st == 0) {
        const char *e = getenv(g_tune_names[knob]);
        if (e && e[0]) { g_tune_val[knob].store(tune_parse(knob, e)); st = 2; } else st = 1;
        g_tune_state[knob].store(st, std::memory_order_release);
    }
    return st == 2 ? g_tune_val[knob].load() : dflt;
}

// FMA-chain microbenchmark: 16 independent chains per thread -> measured CUDA-core peak.  fp32 uses the packed FFMA2 (two fp32 FMAs
// per lane and instruction), the instruction the IoU clip is written on; scalar FFMA chains reach 55-79 % of nominal on sm_100a
// because the issue slots are shared with the loop's uniform-datapath instructions, FFMA2 reaches 91 % at the maximum clock.
template <typename T> struct ProbeOp;
template <> struct ProbeOp<float> {
    using V = float2;
    static __device__ __forceinline__ V init(float s) { return make_float2(s, s + 0.5f); }
    static __device__ __forceinline__ V fma(V a, V m, V c) { return __ffma2_rn(a, m, c); }
    static __device__ __forceinline__ float sum(V a) { return a.x + a.y; }
    static constexpr double flops = 4.0;
};
template <> struct ProbeOp<double> {
    using V = double;
    static __device__ __forceinline__ V init(double s) { return s; }
    static __device__ __forceinline__ V fma(V a, V m, V c) { return ::fma(a, m, c); }
    static __device__ __forceinline__ float sum(V a) { return (float)a; }
    static constexpr double flops = 2.0;
};
constexpr int PROBE_CHAINS = 16;
template <typename T>
__global__ void __launch_bounds__(256) fma_probe_kernel(int64_t iters, T seed, float *sink)
{
    using Op = ProbeOp<T>;
    typename Op::V a[PROBE_CHAINS];
#pragma unroll
    for (int k = 0; k < PROBE_CHAINS; k++) a[k] = Op::init(seed + (T)(threadIdx.x + k));
    const typename Op::V m = Op::init(T(0.999)), c = Op::init(T(0.001));
#pragma unroll 8   // the loop's own instructions (counter, compare, branch) must not compete with the FMAs for issue slots
    for (int64_t i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < PROBE_CHAINS; k++) a[k] = Op::fma(a[k], m, c);
    }
    float s = 0;
#pragma unroll
    for (int k = 0; k < PROBE_CHAINS; k++) s += Op::sum(a[k]);
    if (s == -1.0f) sink[0] = s;  // never true; keeps the chains alive
}
}  // namespace d3d

using namespace d3d;

extern "C" int d3d_tuning_set(const char *name, int value, int set)
{
    if (!name) return D3D_ERR_INVALID_ARGUMENT;
    for (int k = 0; k < D3D_TUNE_COUNT; k++)
        if (!strcmp(name, g_tune_names[k])) {
            g_tune_val[k].store(value);
            g_tune_state[k].store(set ? 2 : 1, std::memory_order_release);
            return D3D_OK;
        }
    return D3D_ERR_INVALID_ARGUMENT;
}
extern "C" int d3d_abi_version(void) { return D3D_B200_ABI_VERSION; }
extern "C" int64_t d3d_launch_count(void) { return g_launches.load(); }
extern "C" const char *d3d_last_cuda_error(void) { return g_cuda_err; }
extern "C" const char *d3d_error_string(int s)
{
    switch (s) {
    case D3D_OK: return "ok";
    case D3D_ERR_INVALID_ARGUMENT: return "invalid argument";
    case D3D_ERR_CUDA: return "CUDA error";
    case D3D_ERR_WORKSPACE: return "workspace too small";
    case D3D_ERR_UNSUPPORTED: return "unsupported option";
    case D3D_ERR_RANGE: return "voxel grid exceeds the 63-bit key range";
    default: return "unknown status";
    }
}
extern "C" int d3d_fma_peak_probe(int dtype, int64_t iters, float *sink, double *flops_host, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    int dev = 0, sms = 0;
    D3D_CUDA_TRY(cudaGetDevice(&dev));
    D3D_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int blocks = sms * 8, threads = 256;   // 2048 threads per SM: every scheduler saturated
    if (dtype == D3D_F64) fma_probe_kernel<double><<<blocks, threads, 0, st>>>(iters, 1.0, sink);
    else fma_probe_kernel<float><<<blocks, threads, 0, st>>>(iters, 1.0f, sink);
    D3D_LAUNCHED();
    if (flops_host) *flops_host = (dtype == D3D_F64 ? ProbeOp<double>::flops : ProbeOp<float>::flops) * PROBE_CHAINS * (double)iters * (double)blocks * threads;
    return D3D_OK;
}
