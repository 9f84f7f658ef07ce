// Shared device helpers for the PointVS B200 kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdlib>

#include "pvs_b200.h"

namespace pvs {

extern thread_local int g_last_cuda_error;
// process-wide: the backward runs on autograd's worker thread
extern std::atomic<int64_t> g_launches;

// call after a group of `n` kernel launches
inline int check_launch(int n = 1) {
    g_launches += n;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        g_last_cuda_error = (int)e;
        return PVS_ERR_CUDA;
    }
    return PVS_OK;
}

inline int cuda_call(cudaError_t e) {
    if (e != cudaSuccess) {
        g_last_cuda_error = (int)e;
        return PVS_ERR_CUDA;
    }
    return PVS_OK;
}

// Programmatic dependent launch (sm_90+).  A kernel of the scoring chain calls
// pdl_launch_dependents() first thing and pdl_wait() after its prologue (weight
// tiles, TMEM, barriers: nothing a predecessor writes) and before it touches
// anything a predecessor produces or still reads.  Launched with
// launch_chained(..., chained = true) the next kernel's CTAs then start on the
// SMs the previous kernel has already left and run their prologue under its
// tail; launched the ordinary way both calls are no-ops.
__device__ __forceinline__ void pdl_launch_dependents() {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
__device__ __forceinline__ void pdl_wait() {
    asm volatile("griddepcontrol.wait;" ::: "memory");
}
// true while pvs_egnn_model_fwd / pvs_egnn_stack_fwd / pvs_egnn_layer_bwd issue
// their launch chain
extern thread_local bool g_pdl_chain;

// Chains the launches of its lifetime (unless PVS_NO_PDL is set, the A/B
// switch) and restores the previous setting on exit.
struct ChainScope {
    bool prev;
    ChainScope() : prev(g_pdl_chain) {
        static const bool off = getenv("PVS_NO_PDL") != nullptr;
        g_pdl_chain = !off;
    }
    ~ChainScope() { g_pdl_chain = prev; }
};

template <typename... KArgs, typename... Args>
inline cudaError_t launch_chained(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                  cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = g_pdl_chain ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

int num_sms();
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (kernel, device,
// size): it is a driver call and was being issued before every launch.
int ensure_dynamic_smem(const void *func, size_t bytes);
template <typename K>
inline int ensure_smem(K kernel, size_t bytes) {
    return ensure_dynamic_smem(reinterpret_cast<const void *>(kernel), bytes);
}
int max_optin_smem();

inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

// Raw MUFU ops.  __expf / __fdividef wrap these in range-fixup code (~12 SASS
// instructions per SiLU, 36 % of the edge kernel's issue slots in the first
// ncu capture); .ftz forms need none: ex2(+big) = inf -> rcp(inf) = 0.
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float tanh_approx(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// Packed fp32x2 arithmetic (Blackwell FFMA2/FADD2/FMUL2): one issue slot for
// two lanes.  The edge kernels are issue-bound, not FMA-pipe-bound.
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    unsigned long long ra = *reinterpret_cast<unsigned long long *>(&a);
    unsigned long long rb = *reinterpret_cast<unsigned long long *>(&b);
    unsigned long long rc = *reinterpret_cast<unsigned long long *>(&c), rd;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    return *reinterpret_cast<float2 *>(&rd);
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
    unsigned long long ra = *reinterpret_cast<unsigned long long *>(&a);
    unsigned long long rb = *reinterpret_cast<unsigned long long *>(&b), rd;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2 *>(&rd);
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
    unsigned long long ra = *reinterpret_cast<unsigned long long *>(&a);
    unsigned long long rb = *reinterpret_cast<unsigned long long *>(&b), rd;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
    return *reinterpret_cast<float2 *>(&rd);
}
// two SiLUs: 3 packed FMA-pipe ops + 4 MUFU (fp32-class) or 2 packed + 2 MUFU
__device__ __forceinline__ float2 silu2_(float2 v) {
    const float2 t = fmul2(v, make_float2(-1.4426950408889634f, -1.4426950408889634f));
    float2 e = make_float2(ex2_approx(t.x), ex2_approx(t.y));
    e = fadd2(e, make_float2(1.0f, 1.0f));
    return fmul2(v, make_float2(rcp_approx(e.x), rcp_approx(e.y)));
}
// Four SiLUs with 6 MUFU instead of 8: the two denominators a = 1 + e^-u and
// b = 1 + e^-v of a lane share one reciprocal, 1/a = b * rcp(a b).  Inputs are
// clamped at -43 (silu(-43) = -9e-18) so that a b stays finite.  Error ~3 ulp.
__device__ __forceinline__ void silu4_(float2 &u, float2 &v) {
    const float2 nl2e = make_float2(-1.4426950408889634f, -1.4426950408889634f);
    const float2 one = make_float2(1.0f, 1.0f);
    u = make_float2(fmaxf(u.x, -43.0f), fmaxf(u.y, -43.0f));
    v = make_float2(fmaxf(v.x, -43.0f), fmaxf(v.y, -43.0f));
    const float2 tu = fmul2(u, nl2e), tv = fmul2(v, nl2e);
    const float2 a = fadd2(make_float2(ex2_approx(tu.x), ex2_approx(tu.y)), one);
    const float2 b = fadd2(make_float2(ex2_approx(tv.x), ex2_approx(tv.y)), one);
    const float2 p = fmul2(a, b);
    const float2 r = make_float2(rcp_approx(p.x), rcp_approx(p.y));
    u = fmul2(fmul2(u, b), r);
    v = fmul2(fmul2(v, a), r);
}
__device__ __forceinline__ float2 silu2_fast_(float2 v) {
    const float2 h = fmul2(v, make_float2(0.5f, 0.5f));
    return ffma2(h, make_float2(tanh_approx(h.x), tanh_approx(h.y)), h);
}

__device__ __forceinline__ float sigmoidf_(float v) {
    return rcp_approx(1.0f + ex2_approx(-1.4426950408889634f * v));
}
// SiLU, fp32-class: 2 MUFU (ex2, rcp) + 3 FMA-pipe ops, error ~2 ulp.
__device__ __forceinline__ float siluf_(float v) {
    return v * rcp_approx(1.0f + ex2_approx(-1.4426950408889634f * v));
}
// SiLU for the single-pass bf16 mode: x*sigmoid(x) = h + h*tanh(h), h = x/2.
// 1 MUFU; tanh.approx error 2^-11 is below the bf16 operand rounding.
__device__ __forceinline__ float siluf_fast_(float v) {
    const float h = 0.5f * v;
    return fmaf(h, tanh_approx(h), h);
}
// d silu / dv given v
__device__ __forceinline__ float silu_gradf_(float v) {
    float s = sigmoidf_(v);
    return s * (1.0f + v * (1.0f - s));
}

__device__ __forceinline__ float apply_act(float v, int act) {
    switch (act) {
        case PVS_ACT_SIGMOID: return sigmoidf_(v);
        case PVS_ACT_TANH: return tanhf(v);
        case PVS_ACT_RELU: return fmaxf(v, 0.0f);
        case PVS_ACT_SILU: return siluf_(v);
        case PVS_ACT_SOFTPLUS:
            // torch.nn.Softplus(beta=1, threshold=20)
            return v > 20.0f ? v : log1pf(expf(v));
        default: return v;
    }
}
// derivative of act w.r.t. its input, from input v and output y
__device__ __forceinline__ float act_grad(float v, float y, int act) {
    switch (act) {
        case PVS_ACT_SIGMOID: return y * (1.0f - y);
        case PVS_ACT_TANH: return 1.0f - y * y;
        case PVS_ACT_RELU: return v > 0.0f ? 1.0f : 0.0f;
        case PVS_ACT_SILU: return silu_gradf_(v);
        case PVS_ACT_SOFTPLUS: return v > 20.0f ? 1.0f : sigmoidf_(v);
        default: return 1.0f;
    }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum_int(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// inclusive scan across the warp
__device__ __forceinline__ int warp_scan_incl(int v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
    }
    return v;
}

}  // namespace pvs
