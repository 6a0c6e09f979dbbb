// Shared device helpers for the TANTE B200 kernels.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "dropout.cuh"

namespace tante {

constexpr int kWarp = 32;

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) applies to the CURRENT device only: every *_set_attrs() keeps one
// "done" bit per device ordinal (a process may drive several GPUs through one engine each).
static inline bool attrs_needed(unsigned long long& mask) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { (void)cudaGetLastError(); dev = 0; }
    const unsigned long long bit = 1ull << (dev & 63);
    if (mask & bit) return false;
    mask |= bit;
    return true;
}

// ---- element conversion -------------------------------------------------------
template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// 4-wide vector load/store of either element type (16 B for f32, 8 B for bf16).
template <typename T> struct Vec4;
template <> struct Vec4<float> {
    static __device__ __forceinline__ void load(const float* p, float (&v)[4]) {
        float4 t = *reinterpret_cast<const float4*>(p);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
    static __device__ __forceinline__ void store(float* p, const float (&v)[4]) {
        *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    }
};
template <> struct Vec4<__nv_bfloat16> {
    static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&v)[4]) {
        uint2 t = *reinterpret_cast<const uint2*>(p);
        __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&t.x);
        __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&t.y);
        float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
        v[0] = fa.x; v[1] = fa.y; v[2] = fb.x; v[3] = fb.y;
    }
    static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&v)[4]) {
        __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]);
        __nv_bfloat162 b = __floats2bfloat162_rn(v[2], v[3]);
        uint2 t;
        t.x = *reinterpret_cast<uint32_t*>(&a);
        t.y = *reinterpret_cast<uint32_t*>(&b);
        *reinterpret_cast<uint2*>(p) = t;
    }
};

// Programmatic dependent launch (PDL).  The tcgen05 GEMM / weight-gradient kernels are launched with
// cudaLaunchAttributeProgrammaticStreamSerialization: their prologue (barrier init, TMEM allocation, the resident weight
// slice -- parameters only, never data of a kernel in flight) may run while the PREVIOUS kernel of the stream drains, and they
// execute griddepcontrol.wait before touching anything that kernel produced.  Every kernel that commonly precedes them calls
// pdl_trigger() first thing, which allows that early start once all of ITS blocks have been scheduled.  Both instructions are
// no-ops when the neighbouring launch is an ordinary one.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// fp32 runs of 2 or 4 elements (64- / 128-bit accesses)
template <int N> struct VecN;
template <> struct VecN<4> {
    static __device__ __forceinline__ void load(const float* p, float (&v)[4]) { Vec4<float>::load(p, v); }
    static __device__ __forceinline__ void store(float* p, const float (&v)[4]) { Vec4<float>::store(p, v); }
};
template <> struct VecN<2> {
    static __device__ __forceinline__ void load(const float* p, float (&v)[2]) {
        float2 t = *reinterpret_cast<const float2*>(p);
        v[0] = t.x; v[1] = t.y;
    }
    static __device__ __forceinline__ void store(float* p, const float (&v)[2]) {
        *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]);
    }
};

// ---- activations (accurate versions: the fp32 parity mode is compiled without fast-math) --
__device__ __forceinline__ float gelu_erf(float x) {
    return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}
__device__ __forceinline__ float gelu_tanh(float x) {
    const float k = 0.79788456080286535588f;  // sqrt(2/pi)
    return 0.5f * x * (1.0f + tanhf(k * (x + 0.044715f * x * x * x)));
}
// bf16-mode erf-GELU: erf(z) ~= tanh(z (a + b z^2 + c z^4)) (minimax fit on [0, 5], |err| <= 3.7e-5 -- below the 2^-11 of
// tanh.approx and two orders below bf16 resolution), folded into x (z = x / sqrt 2): 8 instructions + one MUFU per element
// instead of ~20 + two MUFU for the A&S erf + exp form, which made the propagator / patch-embed / activation kernels issue-bound.
// The odd polynomial is not monotone beyond |x| ~ 8.7 (c < 0), where tanh has long saturated: the argument is clamped.
__device__ __forceinline__ float tanh_approx_f(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
constexpr float kGeA = 0.7977190645145112f, kGeB = 0.036797175748107515f, kGeC = -0.00031560473741394456f;
__device__ __forceinline__ float gelu_erf_fast(float x) {
    const float xc = fminf(fmaxf(x, -8.0f), 8.0f);
    const float x2 = xc * xc;
    const float t = tanh_approx_f(xc * fmaf(x2, fmaf(x2, kGeC, kGeB), kGeA));
    const float hx = 0.5f * x;
    return fmaf(hx, t, hx);
}
template <typename T> __device__ __forceinline__ float gelu_erf_for(float x);
template <> __device__ __forceinline__ float gelu_erf_for<float>(float x) { return gelu_erf(x); }
template <> __device__ __forceinline__ float gelu_erf_for<__nv_bfloat16>(float x) { return gelu_erf_fast(x); }

// derivatives (training path)
__device__ __forceinline__ float gelu_erf_grad(float x) {
    const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752440f));
    const float pdf = 0.39894228040143267794f * expf(-0.5f * x * x);
    return cdf + x * pdf;
}
__device__ __forceinline__ float gelu_tanh_grad(float x) {
    const float k = 0.79788456080286535588f;
    const float u = k * (x + 0.044715f * x * x * x);
    const float t = tanhf(u);
    const float du = k * (1.0f + 3.0f * 0.044715f * x * x);
    return 0.5f * (1.0f + t) + 0.5f * x * (1.0f - t * t) * du;
}

// bf16-mode variants of the activations and their derivatives (approximate transcendental units; the errors are far
// below bf16 resolution).  Selected by the activation element type: float keeps the accurate versions.
__device__ __forceinline__ float gelu_tanh_fast_f(float x) {
    const float k = 0.79788456080286535588f;
    return 0.5f * x * (1.0f + tanh_approx_f(k * fmaf(0.044715f * x, x * x, x)));
}
// derivative of gelu_erf_fast (of the same approximant, so value and gradient stay consistent)
__device__ __forceinline__ float gelu_erf_grad_fast(float x) {
    const float xc = fminf(fmaxf(x, -8.0f), 8.0f);
    const float x2 = xc * xc;
    const float t = tanh_approx_f(xc * fmaf(x2, fmaf(x2, kGeC, kGeB), kGeA));
    const float du = fmaf(x2, fmaf(x2, 5.0f * kGeC, 3.0f * kGeB), kGeA);
    return fmaf(0.5f * xc * du, fmaf(-t, t, 1.0f), fmaf(0.5f, t, 0.5f));
}
__device__ __forceinline__ float gelu_tanh_grad_fast(float x) {
    const float k = 0.79788456080286535588f;
    const float x2 = x * x;
    const float t = tanh_approx_f(k * fmaf(0.044715f * x, x2, x));
    const float du = k * fmaf(3.0f * 0.044715f, x2, 1.0f);
    return fmaf(0.5f * x * du, fmaf(-t, t, 1.0f), fmaf(0.5f, t, 0.5f));
}
template <typename T> struct ActMath {     // accurate (exact fp32 mode)
    static __device__ __forceinline__ float gelu_erf_f(float x) { return gelu_erf(x); }
    static __device__ __forceinline__ float gelu_tanh_f(float x) { return gelu_tanh(x); }
    static __device__ __forceinline__ float gelu_erf_g(float x) { return gelu_erf_grad(x); }
    static __device__ __forceinline__ float gelu_tanh_g(float x) { return gelu_tanh_grad(x); }
};
template <> struct ActMath<__nv_bfloat16> {
    static __device__ __forceinline__ float gelu_erf_f(float x) { return gelu_erf_fast(x); }
    static __device__ __forceinline__ float gelu_tanh_f(float x) { return gelu_tanh_fast_f(x); }
    static __device__ __forceinline__ float gelu_erf_g(float x) { return gelu_erf_grad_fast(x); }
    static __device__ __forceinline__ float gelu_tanh_g(float x) { return gelu_tanh_grad_fast(x); }
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Epilogue selector shared by the SIMT and tcgen05 GEMMs.
enum Epilogue : int {
    EPI_BIAS = 0,        // C = acc + bias
    EPI_BIAS_RELU = 1,
    EPI_BIAS_GELU_ERF = 2,
    EPI_BIAS_GELU_TANH = 3,
    EPI_BIAS_RESID = 4,  // C = resid + acc + bias   (fp32 residual stream, may alias C)
    EPI_EMBED = 5,       // encoder tail: v=acc+bias; v += v*scale[t]+shift[t]; v += s_emb[hw]; v += t_emb[t]
    EPI_BIAS_RESID_LN = 6,  // EPI_BIAS_RESID + LayerNorm of the updated row written to a second (bf16) output
};

struct EpiParams {
    const float* bias = nullptr;    // [N]
    const float* resid = nullptr;   // [M, ldr] fp32
    int ldr = 0;                    // row stride of resid (EPI_BIAS_RESID) / of film,s_emb,t_emb (EPI_EMBED)
    // EPI_EMBED
    const float* film = nullptr;    // [T][2][N] scale,shift of t_encode
    const float* s_emb = nullptr;   // [L][N]
    const float* t_emb = nullptr;   // [T][N]
    int T = 0, L = 0;
    // EPI_BIAS_RESID_LN (tensor GEMM only, N == 256): next LayerNorm's affine + its bf16 output
    const float* ln_gamma = nullptr;
    const float* ln_beta = nullptr;
    void* ln_out = nullptr;         // bf16 [M, N]
    // optional device-side row count (rollout encoder cache): effective M = min(M, *m_dev * m_rows)
    const int* m_dev = nullptr;
    int m_rows = 0;
    // Keeps the layout (and the 136-byte size) that the FP32 FFMA GEMM was tuned with: it takes EpiParams by value, and at
    // 120 bytes nvcc keeps the fields in registers instead of re-reading the parameter space, which costs
    // gemm_simt_kernel<128, *> its second CTA per SM (142 registers; residual epilogue at M = 65536 on a B200 at 1000 W:
    // 245 -> 310 us).
    uint32_t reserved[4] = {0u, 0u, 0u, 0u};
    // EPI_BIAS_RESID in training with dropout (SIMT GEMM): C = resid + drop(acc + bias), element index m * ldr + n
    DropCfg drop;
    uint32_t drop_site = 0;
};

// encoder tail (t_encode FiLM + s_emb + t_emb, tante.py:132-141) with explicit roundings: the GEMM epilogues
// (EPI_EMBED, both GEMM kernels) and the rollout's embed_cached_kernel must agree bit for bit
__device__ __forceinline__ float embed_value(float v, float sc, float sh, float se, float te) {
    return __fadd_rn(__fadd_rn(__fadd_rn(v, __fmaf_rn(v, sc, sh)), se), te);
}

template <int EPI>
__device__ __forceinline__ float apply_epilogue(float acc, int m, int n, const EpiParams& p) {
    float v = acc + p.bias[n];
    if (EPI == EPI_BIAS_RELU) v = fmaxf(v, 0.0f);
    if (EPI == EPI_BIAS_GELU_ERF) v = gelu_erf(v);
    if (EPI == EPI_BIAS_GELU_TANH) v = gelu_tanh(v);
    if (EPI == EPI_BIAS_RESID) {
        if (p.drop.p > 0.f) v *= drop_elem(p.drop, p.drop_site, (unsigned long long)m * p.ldr + n);
        v = p.resid[(size_t)m * p.ldr + n] + v;
    }
    if (EPI == EPI_EMBED) {
        const int hw = m % p.L;
        const int t = (m / p.L) % p.T;
        v = embed_value(v, p.film[(size_t)(t * 2 + 0) * p.ldr + n], p.film[(size_t)(t * 2 + 1) * p.ldr + n],
                        p.s_emb[(size_t)hw * p.ldr + n], p.t_emb[(size_t)t * p.ldr + n]);
    }
    return v;
}

}  // namespace tante
