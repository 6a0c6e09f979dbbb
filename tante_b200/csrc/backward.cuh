// Backward (training) kernels of the TANTE hot path that are not GEMMs: activation derivatives, LayerNorm
// backward, axial attention backward, propagator backward, the Taylor-head backward, FiLM / interprator
// backward, embedding backward, the first patch conv's backward, a generic split-M weight-gradient kernel for
// the exact fp32 mode (and for shapes the tcgen05 wgrad kernel does not cover) and the gradient un-packer.
// Templated on the activation element type TA (float: exact mode, bf16: tensor mode) like the forward kernels.
//
// What they differentiate (reference, all through torch autograd there):
//   TransformerBlock.forward attn_backbone.py:59-83, Attn_Backbone.forward :134-191, enc_CNN/dec_CNN.forward
//   enc_dec_cnn.py:217-229,263-277, film/interprator tante.py:178-230, Taylor sum tante.py:156-171.
#pragma once
#include "common.cuh"
#include "kernels_simt.cuh"
#include "pack.cuh"

namespace tante {

enum ActKind : int { ACT_GELU_ERF = 2, ACT_GELU_TANH = 3, ACT_RELU = 1 };

// ---- elementwise: act = f(pre) -------------------------------------------------------------------
template <typename TA, int ACT>
__global__ void __launch_bounds__(256) act_fwd_kernel(const TA* __restrict__ pre, TA* __restrict__ out, long long n4) {
    pdl_trigger();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    float v[4], o[4];
    Vec4<TA>::load(pre + i * 4, v);
#pragma unroll
    for (int j = 0; j < 4; ++j)
        o[j] = ACT == ACT_GELU_ERF ? ActMath<TA>::gelu_erf_f(v[j]) : (ACT == ACT_GELU_TANH ? ActMath<TA>::gelu_tanh_f(v[j]) : fmaxf(v[j], 0.f));
    Vec4<TA>::store(out + i * 4, o);
}

// ---- elementwise: g <- g * f'(pre)   (ACT_RELU: `pre` may be the post-ReLU activation) --------------
template <typename TA, int ACT>
__global__ void __launch_bounds__(256) act_bwd_kernel(TA* __restrict__ g, const TA* __restrict__ pre, long long n4) {
    pdl_trigger();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    float v[4], d[4];
    Vec4<TA>::load(pre + i * 4, v);
    Vec4<TA>::load(g + i * 4, d);
#pragma unroll
    for (int j = 0; j < 4; ++j)
        d[j] *= ACT == ACT_GELU_ERF ? ActMath<TA>::gelu_erf_g(v[j]) : (ACT == ACT_GELU_TANH ? ActMath<TA>::gelu_tanh_g(v[j]) : (v[j] > 0.f ? 1.f : 0.f));
    Vec4<TA>::store(g + i * 4, d);
}

// ---- training loss of the rollout drivers (trainer/metrics.py:53-80: MSE.eval(...).mean()) -------------------------
// sum over (b, j < n_use, d, pixel) of (y - ref)^2 between channels-FIRST predictions y (B, nf, D, HW) -- the module's
// output layout -- and the channels-LAST targets ref (B, n_ref, HW, D), frames f0 .. f0+n_use-1; and/or its gradient
// grad_y = scale * gout * (y - ref) (frames >= n_use get zero).  One pass; replaces the formatter permute, the cat over
// model calls, sub, pow, the two means and their five autograd kernels.  thread = pixel, loop over the fields:
// y accesses coalesce across the warp, a warp's ref accesses cover 32*D consecutive floats.
__global__ void __launch_bounds__(256) mse_cf_cl_kernel(const float* __restrict__ y, const float* __restrict__ ref, int B, int nf,
                                                        int n_use, int D, long long HW, int n_ref, int f0, float scale,
                                                        const float* __restrict__ gout, float* __restrict__ loss_sum,
                                                        float* __restrict__ grad_y) {
    const long long total = (long long)B * nf * HW;
    const float gs = grad_y ? scale * (gout ? *gout : 1.f) : 0.f;
    float acc = 0.f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long p = i % HW;
        const long long bj = i / HW;
        const int j = (int)(bj % nf);
        const long long b = bj / nf;
        const float* yp = y + (size_t)bj * D * HW + p;
        float* gp = grad_y ? grad_y + (size_t)bj * D * HW + p : nullptr;
        if (j >= n_use) {
            if (gp) for (int d = 0; d < D; ++d) gp[(size_t)d * HW] = 0.f;
            continue;
        }
        const float* rp = ref + (((size_t)b * n_ref + f0 + j) * HW + p) * D;
        for (int d = 0; d < D; ++d) {
            const float df = yp[(size_t)d * HW] - rp[d];
            acc = fmaf(df, df, acc);
            if (gp) gp[(size_t)d * HW] = gs * df;
        }
    }
    if (loss_sum) {
        __shared__ float red[8];
        acc = warp_sum(acc);
        if (threadIdx.x % 32 == 0) red[threadIdx.x / 32] = acc;
        __syncthreads();
        if (threadIdx.x < 8) {
            float v = red[threadIdx.x];
#pragma unroll
            for (int o = 4; o > 0; o >>= 1) v += __shfl_xor_sync(0xffu, v, o);
            if (threadIdx.x == 0) atomicAdd(loss_sum, v);
        }
    }
}

// out = resid + mask / (1 - p) * y: residual add of a dropped-out branch output (tensor mode outside the fused block tail);
// element index = position in the [tokens][C] stream, as in the fused epilogues
template <typename TA>
__global__ void __launch_bounds__(256) resid_drop_kernel(const TA* __restrict__ y, const float* __restrict__ resid, float* __restrict__ out,
                                                         long long n4, DropCfg drop, uint32_t site) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    float v[4], r[4];
    Vec4<TA>::load(y + i * 4, v);
    Vec4<float>::load(resid + i * 4, r);
    const uint4 w = drop_words(drop, site, (unsigned long long)(i >> 1));
#pragma unroll
    for (int j = 0; j < 4; ++j) r[j] = fmaf(v[j], drop_mul(drop, w, (int)((i & 1) * 4 + j)), r[j]);
    Vec4<float>::store(out + i * 4, r);
}

// fp32 -> TA copy (gradient stream -> GEMM operand)
template <typename TA>
__global__ void __launch_bounds__(256) convert_kernel(const float* __restrict__ src, TA* __restrict__ dst, long long n4,
                                                      DropCfg drop = DropCfg(), uint32_t site = 0) {
    pdl_trigger();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    float v[4];
    Vec4<float>::load(src + i * 4, v);
    if (drop.p > 0.f) {
        // the copy is the dY operand of a residual BRANCH whose output went through dropout: dY = dx o mask / (1 - p)
        const uint4 w = drop_words(drop, site, (unsigned long long)(i >> 1));
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] *= drop_mul(drop, w, (int)((i & 1) * 4 + j));
    }
    Vec4<TA>::store(dst + i * 4, v);
}

// ---- column sums: out[n] += sum_m x[m][n]  (bias gradients) ----------------------------------------
// block (32, 8): 32 column groups of 4 columns, 8 row lanes; grid (ceil(N/128), row chunks).
template <typename TA>
__global__ void __launch_bounds__(256) colsum_kernel(const TA* __restrict__ x, int ld, long long M, int N,
                                                     float* __restrict__ out) {
    __shared__ float red[8][128];
    const int cx = threadIdx.x % 32, ry = threadIdx.x / 32;
    const int c0 = blockIdx.x * 128 + cx * 4;
    float s[4] = {0.f, 0.f, 0.f, 0.f};
    if (c0 < N) {
        for (long long m = (long long)blockIdx.y * 8 + ry; m < M; m += (long long)gridDim.y * 8) {
            float v[4];
            Vec4<TA>::load(x + (size_t)m * ld + c0, v);
#pragma unroll
            for (int j = 0; j < 4; ++j) s[j] += v[j];
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) red[ry][cx * 4 + j] = s[j];
    __syncthreads();
    if (threadIdx.x < 128) {
        float t = 0.f;
#pragma unroll
        for (int r = 0; r < 8; ++r) t += red[r][threadIdx.x];
        const int c = blockIdx.x * 128 + threadIdx.x;
        if (c < N) atomicAdd(out + c, t);
    }
}

// ---- embed forward (training mode: the encoder tail's FiLM + embeddings as its own pass so that the conv
//      output v stays available for the backward): x0 = v + (v*scale_t + shift_t) + s_emb + t_emb ------
__global__ void __launch_bounds__(256) embed_fwd_kernel(const float* __restrict__ v, const float* __restrict__ film,
                                                        const float* __restrict__ s_emb, const float* __restrict__ t_emb,
                                                        float* __restrict__ x0, long long tokens, int T, int L, int C) {
    const long long i4 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i4 >= tokens * C) return;
    const long long m = i4 / C;
    const int c = (int)(i4 % C);
    const int hw = (int)(m % L), t = (int)((m / L) % T);
    float a[4], sc[4], sh[4], se[4], te[4], o[4];
    Vec4<float>::load(v + i4, a);
    Vec4<float>::load(film + (size_t)(t * 2 + 0) * C + c, sc);
    Vec4<float>::load(film + (size_t)(t * 2 + 1) * C + c, sh);
    Vec4<float>::load(s_emb + (size_t)hw * C + c, se);
    Vec4<float>::load(t_emb + (size_t)t * C + c, te);
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = a[j] + (a[j] * sc[j] + sh[j]) + se[j] + te[j];
    Vec4<float>::store(x0 + i4, o);
}

// ---- embed backward: dv = g*(1+scale_t); dscale[t] += g*v; dshift[t] += g; ds_emb[hw] += g; dt_emb[t] += g ----
// Thread = (latent position hw, 4 channels): 128-bit loads of g and v, the batch loop unrolled for loads in flight; the block's
// positions are summed in shared memory before the atomics.  grid = ceil(L / (256 / (C / 4))), C % 4 == 0, C <= 1024.
template <typename TA>
__global__ void __launch_bounds__(256) embed_bwd_kernel(const float* __restrict__ g, const float* __restrict__ v,
                                                        const float* __restrict__ film, TA* __restrict__ dv,
                                                        float* __restrict__ dfilm /* [T][2][C] */,
                                                        float* __restrict__ ds_emb, float* __restrict__ dt_emb, int B,
                                                        int T, int L, int C) {
    __shared__ float red[256 * 4];
    const int c4n = C / 4;                       // threads per position
    const int ppb = blockDim.x / c4n;            // positions per block
    const int pl = threadIdx.x / c4n;            // local position
    const int c = (threadIdx.x % c4n) * 4;
    const int hw = blockIdx.x * ppb + pl;
    const bool live = pl < ppb && hw < L;
    float semb[4] = {0.f, 0.f, 0.f, 0.f};
    for (int t = 0; t < T; ++t) {
        float sc[4], dsc[4] = {0.f, 0.f, 0.f, 0.f}, dsh[4] = {0.f, 0.f, 0.f, 0.f};
        if (live) {
            Vec4<float>::load(film + (size_t)(t * 2) * C + c, sc);
#pragma unroll 4
            for (int b = 0; b < B; ++b) {
                const size_t m = ((size_t)(b * T + t) * L + hw) * C + c;
                float gg[4], vv[4], o[4];
                Vec4<float>::load(g + m, gg);
                Vec4<float>::load(v + m, vv);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    o[j] = gg[j] * (1.0f + sc[j]);
                    dsc[j] = fmaf(gg[j], vv[j], dsc[j]);
                    dsh[j] += gg[j];
                }
                Vec4<TA>::store(dv + m, o);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) semb[j] += dsh[j];
        }
        // sum the block's positions, then one atomic per (t, channel) and quantity
        for (int k = 0; k < 2; ++k) {
            __syncthreads();
#pragma unroll
            for (int j = 0; j < 4; ++j) red[threadIdx.x * 4 + j] = live ? (k == 0 ? dsc[j] : dsh[j]) : 0.f;
            __syncthreads();
            if (threadIdx.x < c4n) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float tot = 0.f;
                    for (int q = 0; q < ppb; ++q) tot += red[(q * c4n + threadIdx.x) * 4 + j];
                    if (k == 0) atomicAdd(dfilm + (size_t)(t * 2) * C + c + j, tot);
                    else {
                        atomicAdd(dfilm + (size_t)(t * 2 + 1) * C + c + j, tot);
                        atomicAdd(dt_emb + (size_t)t * C + c + j, tot);
                    }
                }
            }
        }
    }
    if (live) {
        float cur[4];
        Vec4<float>::load(ds_emb + (size_t)hw * C + c, cur);
#pragma unroll
        for (int j = 0; j < 4; ++j) cur[j] += semb[j];
        Vec4<float>::store(ds_emb + (size_t)hw * C + c, cur);
    }
}

// ---- FiLM generator backward (tante.py:206-220): for each condition n, given dscale/dshift [n][2][C] -----
// grads of the two 2-layer MLPs (atomics into the packed-gradient arena) and d cond[n].
__global__ void __launch_bounds__(256) film_bwd_kernel(const float* __restrict__ cond, const float* __restrict__ dfilm,
                                                       const float* __restrict__ w0s, const float* __restrict__ b0s,
                                                       const float* __restrict__ w2s, const float* __restrict__ w0h,
                                                       const float* __restrict__ b0h, const float* __restrict__ w2h,
                                                       float* __restrict__ gw0s, float* __restrict__ gb0s,
                                                       float* __restrict__ gw2s, float* __restrict__ gb2s,
                                                       float* __restrict__ gw0h, float* __restrict__ gb0h,
                                                       float* __restrict__ gw2h, float* __restrict__ gb2h, int C,
                                                       float* __restrict__ dcond /* nullable [n] */) {
    extern __shared__ float smem[];
    const int Ch = C / 2;
    float* hs = smem;            // [Ch] hidden of the scale branch
    float* hh = hs + Ch;         // [Ch]
    float* ds = hh + Ch;         // [C] dscale
    float* dh = ds + C;          // [C] dshift
    __shared__ float red[8];
    // grid (n conditions, Y slices): a slice takes 1/Y of the outer-product atomics and 8 hidden units per pass (one warp
    // each, lanes over the C outputs); dcond must be zeroed by the caller (slices add their partial sums)
    const int n = blockIdx.x, y = blockIdx.y, Y = gridDim.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float t = cond[n];
    for (int i = threadIdx.x; i < Ch; i += blockDim.x) {
        hs[i] = fmaxf(fmaf(w0s[i], t, b0s[i]), 0.f);
        hh[i] = fmaxf(fmaf(w0h[i], t, b0h[i]), 0.f);
    }
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        ds[c] = dfilm[((size_t)n * 2 + 0) * C + c];
        dh[c] = dfilm[((size_t)n * 2 + 1) * C + c];
    }
    __syncthreads();
    if (y == 0) {
        for (int c = threadIdx.x; c < C; c += blockDim.x) {
            atomicAdd(gb2s + c, ds[c]);
            atomicAdd(gb2h + c, dh[c]);
        }
    }
    for (int i = y * blockDim.x + threadIdx.x; i < C * Ch; i += Y * blockDim.x) {
        const int c = i / Ch, j = i % Ch;
        if (hs[j] != 0.f) atomicAdd(gw2s + i, ds[c] * hs[j]);
        if (hh[j] != 0.f) atomicAdd(gw2h + i, dh[c] * hh[j]);
    }
    float dt = 0.f;
    for (int j = y * 8 + warp; j < Ch; j += Y * 8) {
        float a = 0.f, b = 0.f;
        for (int c = lane; c < C; c += 32) {
            a = fmaf(ds[c], w2s[(size_t)c * Ch + j], a);
            b = fmaf(dh[c], w2h[(size_t)c * Ch + j], b);
        }
        a = warp_sum(a); b = warp_sum(b);
        if (hs[j] <= 0.f) a = 0.f;
        if (hh[j] <= 0.f) b = 0.f;
        if (lane == 0) {
            atomicAdd(gw0s + j, a * t);
            atomicAdd(gb0s + j, a);
            atomicAdd(gw0h + j, b * t);
            atomicAdd(gb0h + j, b);
            dt += a * w0s[j] + b * w0h[j];
        }
    }
    if (lane == 0) red[warp] = dt;
    __syncthreads();
    if (threadIdx.x == 0 && dcond) {
        float tot = 0.f;
        for (int w = 0; w < 8; ++w) tot += red[w];
        atomicAdd(dcond + n, tot);
    }
}

// ---- FiLM application backward on the (B, L, C) derivative latent (tante.py:222-230) --------------------
// dmod = d + d*s_b + h_b:  dx_last[b,l,c] += g*(1+s_b[c]);  dfilm[b][0][c] += sum_l g*d;  dfilm[b][1][c] += sum_l g.
// grid (B, chunks of L), block = C threads (C <= 1024).  dx_last is the gradient stream's last-frame slice.
template <typename TA>
__global__ void film_apply_bwd_kernel(const TA* __restrict__ g, const float* __restrict__ d32,
                                      const float* __restrict__ film, float* __restrict__ dxs, float* __restrict__ dfilm,
                                      int T, int L, int C) {
    const int b = blockIdx.x;
    const int c = threadIdx.x;
    const int per = (L + gridDim.y - 1) / gridDim.y;
    const int l0 = blockIdx.y * per, l1 = min(L, l0 + per);
    const float sc = film[((size_t)b * 2 + 0) * C + c];
    float dsc = 0.f, dsh = 0.f;
    for (int l = l0; l < l1; ++l) {
        const size_t i = ((size_t)b * L + l) * C + c;
        const float gg = to_f32<TA>(g[i]);
        dsc = fmaf(gg, d32[i], dsc);
        dsh += gg;
        dxs[((size_t)(b * T + T - 1) * L + l) * C + c] += gg * (1.0f + sc);
    }
    atomicAdd(dfilm + ((size_t)b * 2 + 0) * C + c, dsc);
    atomicAdd(dfilm + ((size_t)b * 2 + 1) * C + c, dsh);
}

// dxs[:, T-1] += src   (src: [B*L, C] TA)
template <typename TA>
__global__ void __launch_bounds__(256) add_last_frame_kernel(const TA* __restrict__ src, float* __restrict__ dxs, int B,
                                                             int T, long long LC) {
    const long long i4 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i4 >= (long long)B * LC) return;
    const long long b = i4 / LC, r = i4 % LC;
    float v[4], a[4];
    Vec4<TA>::load(src + i4, v);
    float* dst = dxs + ((size_t)(b * T + T - 1)) * LC + r;
    Vec4<float>::load(dst, a);
#pragma unroll
    for (int j = 0; j < 4; ++j) a[j] += v[j];
    Vec4<float>::store(dst, a);
}

// ---- interprator tail backward (tante.py:191-201).  rt_b = mean_l clampST(w3.h2 + b3) + 1.001; the straight-
// through clamp has unit gradient everywhere, so d t_l = drt_b / L for every token.
//   drt_b = gRt[b]/K (R_t = mean_k rt_k, tante.py:159-160) + dcond[b] (FiLM modifier path)
//   dh2[b,l,j] = drt_b/L * w3[j] * (h2 > 0);  gw3[j] += sum drt_b/L * h2;  gb3 += sum_b drt_b.     grid = B.
template <typename TA>
__global__ void __launch_bounds__(256) interp_tail_bwd_kernel(const TA* __restrict__ h2, const float* __restrict__ w3,
                                                              const float* __restrict__ gRt, float inv_K,
                                                              const float* __restrict__ dcond, int L, int C4,
                                                              TA* __restrict__ dh2, float* __restrict__ gw3,
                                                              float* __restrict__ gb3) {
    extern __shared__ float sacc[];     // [C4] per-block accumulators of gw3
    const int b = blockIdx.x;
    const float drt = (gRt ? gRt[b] * inv_K : 0.f) + (dcond ? dcond[b] : 0.f);
    const float dt = drt / (float)L;
    for (int j = threadIdx.x; j < C4; j += blockDim.x) sacc[j] = 0.f;
    __syncthreads();
    const long long n = (long long)L * C4;
    for (long long i = threadIdx.x; i < n; i += blockDim.x) {
        const int j = (int)(i % C4);
        const size_t idx = (size_t)b * n + i;
        const float hv = to_f32<TA>(h2[idx]);
        dh2[idx] = from_f32<TA>(hv > 0.f ? dt * w3[j] : 0.f);
        if (hv != 0.f) atomicAdd(&sacc[j], dt * hv);
    }
    __syncthreads();
    for (int j = threadIdx.x; j < C4; j += blockDim.x) atomicAdd(gw3 + j, sacc[j]);
    if (threadIdx.x == 0) atomicAdd(gb3, drt);
}

// ---- LayerNorm backward (one warp per row, C == 128*MAXV... C <= 128*MAXV) ------------------------------
//   xhat = (x-mean)*rstd; gy = dy*gamma; dx_ln = rstd*(gy - mean(gy) - xhat*mean(gy*xhat))
//   dxs (fp32 gradient stream, in place) += dx_ln; optional TA copy of the updated row (next GEMM operand);
//   dgamma += dy*xhat, dbeta += dy (per-warp registers -> shared -> atomics).
// (occupancy: 3 blocks of 256 threads per SM -- at the natural 87 registers only 2 fit, and the kernel is latency-bound)
template <typename TA, int MAXV, bool DROP = false>
__global__ void __launch_bounds__(256, MAXV <= 2 ? 3 : 1) ln_bwd_kernel(const TA* __restrict__ dy, const float* __restrict__ x,
                                                     const float* __restrict__ gamma, float* __restrict__ dxs,
                                                     TA* __restrict__ dxb, float* __restrict__ dgamma,
                                                     float* __restrict__ dbeta, long long rows, int C, float eps,
                                                     DropCfg drop = DropCfg(), uint32_t site = 0) {
    pdl_trigger();
    __shared__ float sg[128 * MAXV * 4], sb[128 * MAXV * 4];
    const int lane = threadIdx.x % kWarp;
    for (int i = threadIdx.x; i < C; i += blockDim.x) { sg[i] = 0.f; sb[i] = 0.f; }
    __syncthreads();
    float ag[MAXV][4], ab[MAXV][4], gm[MAXV][4];
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
        const int c = (i * kWarp + lane) * 4;
#pragma unroll
        for (int j = 0; j < 4; ++j) { ag[i][j] = 0.f; ab[i][j] = 0.f; gm[i][j] = 0.f; }
        if (c < C) Vec4<float>::load(gamma + c, gm[i]);
    }
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / kWarp;
    const long long nwarps = (long long)gridDim.x * blockDim.x / kWarp;
    constexpr int RPI = 1;       // rows in flight per warp iteration (2 measured slower on B200: register pressure)
    for (long long rb = warp0; rb < rows; rb += nwarps * RPI) {
        float xv[RPI][MAXV][4], dv[RPI][MAXV][4], ov[RPI][MAXV][4];
        long long rr[RPI];
#pragma unroll
        for (int u = 0; u < RPI; ++u) {
            rr[u] = rb + u * nwarps;
#pragma unroll
            for (int i = 0; i < MAXV; ++i) {
                const int c = (i * kWarp + lane) * 4;
                if (c < C && rr[u] < rows) {
                    Vec4<float>::load(x + (size_t)rr[u] * C + c, xv[u][i]);
                    Vec4<TA>::load(dy + (size_t)rr[u] * C + c, dv[u][i]);
                    Vec4<float>::load(dxs + (size_t)rr[u] * C + c, ov[u][i]);
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) { xv[u][i][j] = 0.f; dv[u][i][j] = 0.f; ov[u][i][j] = 0.f; }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < RPI; ++u) {
            if (rr[u] >= rows) continue;        // warp-uniform
            float s = 0.f;
#pragma unroll
            for (int i = 0; i < MAXV; ++i) s += (xv[u][i][0] + xv[u][i][1]) + (xv[u][i][2] + xv[u][i][3]);
            const float mean = warp_sum(s) / (float)C;
            float q = 0.f;
#pragma unroll
            for (int i = 0; i < MAXV; ++i) {
                const int c = (i * kWarp + lane) * 4;
                if (c < C) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) { const float d = xv[u][i][j] - mean; q = fmaf(d, d, q); }
                }
            }
            const float rstd = 1.0f / sqrtf(warp_sum(q) / (float)C + eps);
            float s1 = 0.f, s2 = 0.f;
#pragma unroll
            for (int i = 0; i < MAXV; ++i) {
                const int c = (i * kWarp + lane) * 4;
                if (c < C) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float xh = (xv[u][i][j] - mean) * rstd;
                        const float gy = dv[u][i][j] * gm[i][j];
                        s1 += gy;
                        s2 = fmaf(gy, xh, s2);
                        ag[i][j] = fmaf(dv[u][i][j], xh, ag[i][j]);
                        ab[i][j] += dv[u][i][j];
                        xv[u][i][j] = xh;          // keep xhat
                        dv[u][i][j] = gy;          // keep gy
                    }
                }
            }
            s1 = warp_sum(s1) / (float)C;
            s2 = warp_sum(s2) / (float)C;
#pragma unroll
            for (int i = 0; i < MAXV; ++i) {
                const int c = (i * kWarp + lane) * 4;
                if (c < C) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) ov[u][i][j] += rstd * (dv[u][i][j] - s1 - xv[u][i][j] * s2);
                    Vec4<float>::store(dxs + (size_t)rr[u] * C + c, ov[u][i]);
                    if (dxb) {
                        if (DROP) {
                            // the copy feeds the gradients of the residual branch below (its output went through dropout)
                            const unsigned long long e = (unsigned long long)rr[u] * C + c;
                            const uint4 w = drop_words(drop, site, e >> 3);
#pragma unroll
                            for (int j = 0; j < 4; ++j) ov[u][i][j] *= drop_mul(drop, w, (int)(e & 7) + j);
                        }
                        Vec4<TA>::store(dxb + (size_t)rr[u] * C + c, ov[u][i]);
                    }
                }
            }
        }
    }
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
        const int c = (i * kWarp + lane) * 4;
        if (c < C) {
#pragma unroll
            for (int j = 0; j < 4; ++j) { atomicAdd(&sg[c + j], ag[i][j]); atomicAdd(&sb[c + j], ab[i][j]); }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < C; i += blockDim.x) { atomicAdd(dgamma + i, sg[i]); atomicAdd(dbeta + i, sb[i]); }
}

// ---- axial attention backward (exact SIMT version) ---------------------------------------------------
// One CTA = one head x G packed sequences (R = G*S <= 64 rows, block-diagonal).  Recomputes P = softmax(QK^T*scale
// [+causal]) from the saved qkv, then dV = P^T dO, dP = dO V^T, dS = P o (dP - rowsum(dP o P)), dQ = scale dS K,
// dK = scale dS^T Q.  Token addressing as in the forward (attn_backbone.py:149-162, no rearrange copies).
template <typename TA, int HD>
__global__ void __launch_bounds__(128) attention_bwd_kernel(const TA* __restrict__ qkv, const TA* __restrict__ dout,
                                                            TA* __restrict__ dqkv, long long n_seq, int S, int inner_sz,
                                                            int n_head, int C, int causal, float scale, int G,
                                                            DropCfg drop = DropCfg(), uint32_t site = 0) {
    extern __shared__ float smem[];
    constexpr int P = HD + 1;
    const int R = G * S;
    float* sQ = smem;             // [R][P]
    float* sK = sQ + R * P;
    float* sV = sK + R * P;
    float* sO = sV + R * P;       // dO
    float* sP = sO + R * P;       // [R][S+1]
    float* sD = sP + R * (S + 1); // [R][S+1]  dP -> dS
    const int head = blockIdx.y;
    const long long seq0 = (long long)blockIdx.x * G;
    const int ld = 3 * C;
    const int SP = S + 1;
    // ---- load
    for (int i = threadIdx.x; i < R * (HD / 4); i += blockDim.x) {
        const int r = i / (HD / 4), d4 = (i % (HD / 4)) * 4;
        const long long seq = seq0 + r / S;
        float q4[4] = {0, 0, 0, 0}, k4[4] = {0, 0, 0, 0}, v4[4] = {0, 0, 0, 0}, o4[4] = {0, 0, 0, 0};
        if (seq < n_seq) {
            const long long outer = seq / inner_sz, inner = seq % inner_sz;
            const size_t tok = (size_t)outer * S * inner_sz + (size_t)(r % S) * inner_sz + inner;
            const TA* base = qkv + tok * ld + head * HD + d4;
            Vec4<TA>::load(base, q4);
            Vec4<TA>::load(base + C, k4);
            Vec4<TA>::load(base + 2 * C, v4);
            Vec4<TA>::load(dout + tok * C + head * HD + d4, o4);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            sQ[r * P + d4 + j] = q4[j]; sK[r * P + d4 + j] = k4[j]; sV[r * P + d4 + j] = v4[j]; sO[r * P + d4 + j] = o4[j];
        }
    }
    __syncthreads();
    // ---- scores and dP
    for (int i = threadIdx.x; i < R * S; i += blockDim.x) {
        const int r = i / S, j = i % S;
        const int kr = (r / S) * S + j;
        float s = 0.f, dp = 0.f;
#pragma unroll
        for (int d = 0; d < HD; ++d) {
            s = fmaf(sQ[r * P + d], sK[kr * P + d], s);
            dp = fmaf(sO[r * P + d], sV[kr * P + d], dp);
        }
        s *= scale;
        if (causal && j > (r % S)) s = -INFINITY;
        if (drop.p > 0.f) {
            // dP = (dO V^T) o Z with Z = mask / (1 - p) of (query token, head, key position), as the forward drew it
            const long long seq = seq0 + r / S;
            if (seq < n_seq) {
                const long long outer = seq / inner_sz, inner = seq % inner_sz;
                const long long tokq = outer * S * inner_sz + (long long)(r % S) * inner_sz + inner;
                const uint4 w = drop_words(drop, site, drop_attn_grp(tokq, n_head, head, j));
                dp *= drop_mul(drop, w, j & 7);
            }
        }
        sP[r * SP + j] = s;
        sD[r * SP + j] = dp;
    }
    __syncthreads();
    // ---- softmax rows + dS
    for (int r = threadIdx.x; r < R; r += blockDim.x) {
        float m = -INFINITY;
        for (int j = 0; j < S; ++j) m = fmaxf(m, sP[r * SP + j]);
        float l = 0.f;
        for (int j = 0; j < S; ++j) { const float p = expf(sP[r * SP + j] - m); sP[r * SP + j] = p; l += p; }
        const float inv = 1.0f / l;
        float dot = 0.f;
        for (int j = 0; j < S; ++j) { const float p = sP[r * SP + j] * inv; sP[r * SP + j] = p; dot = fmaf(p, sD[r * SP + j], dot); }
        for (int j = 0; j < S; ++j) sD[r * SP + j] = sP[r * SP + j] * (sD[r * SP + j] - dot) * scale;
    }
    __syncthreads();
    // ---- dQ, dK, dV  (thread per (row, 4 channels))
    for (int i = threadIdx.x; i < R * (HD / 4); i += blockDim.x) {
        const int r = i / (HD / 4), d4 = (i % (HD / 4)) * 4;
        const int g0 = (r / S) * S, p = r % S;
        float dq[4] = {0, 0, 0, 0}, dk[4] = {0, 0, 0, 0}, dv[4] = {0, 0, 0, 0};
        for (int j = 0; j < S; ++j) {
            const float ds_rj = sD[r * SP + j];             // dS[r][j]
            const float ds_jr = sD[(g0 + j) * SP + p];      // dS[j][r]
            float p_jr = sP[(g0 + j) * SP + p];             // P[j][r] (o Z[j][r] with dropout: dV = (P o Z)^T dO)
            if (drop.p > 0.f) {
                const long long seqj = seq0 + r / S;
                if (seqj < n_seq) {
                    const long long outer = seqj / inner_sz, inner = seqj % inner_sz;
                    const long long tokq = outer * S * inner_sz + (long long)j * inner_sz + inner;
                    const uint4 w = drop_words(drop, site, drop_attn_grp(tokq, n_head, head, p));
                    p_jr *= drop_mul(drop, w, p & 7);
                }
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                dq[e] = fmaf(ds_rj, sK[(g0 + j) * P + d4 + e], dq[e]);
                dk[e] = fmaf(ds_jr, sQ[(g0 + j) * P + d4 + e], dk[e]);
                dv[e] = fmaf(p_jr, sO[(g0 + j) * P + d4 + e], dv[e]);
            }
        }
        const long long seq = seq0 + r / S;
        if (seq < n_seq) {
            const long long outer = seq / inner_sz, inner = seq % inner_sz;
            const size_t tok = (size_t)outer * S * inner_sz + (size_t)p * inner_sz + inner;
            TA* base = dqkv + tok * ld + head * HD + d4;
            Vec4<TA>::store(base, dq);
            Vec4<TA>::store(base + C, dk);
            Vec4<TA>::store(base + 2 * C, dv);
        }
    }
}

// ---- propagator backward (attn_backbone.py:111-119,140-146):  y = x + W2 gelu(W1 x + b1) + b2 along an axis ----
// In place on the gradient stream: dx = dy + W1^T (gelu'(pre) o (W2^T dy)); weight gradients accumulated in
// registers across the slabs of a persistent CTA, reduced in shared memory and flushed with one atomic per entry.
// Slab = one `outer` x CW columns with S4*CW = 4096 (short axes get wide slabs, so all 256 threads work for
// the T axis, S = 4, as well as for S = 64): threads = (CW/4 column groups) x (S4/4 row groups) of 4 x 4 tiles.
constexpr int kPropBwdSlab = 4096;      // floats per slab array
template <typename TM /* float: accurate erf/exp; bf16: the approximate versions the tensor-mode forward uses */>
__global__ void __launch_bounds__(256) propagator_bwd_kernel(const float* __restrict__ xin, float* __restrict__ dy,
                                                             int S, long long IC, long long n_outer,
                                                             const float* __restrict__ W1, const float* __restrict__ b1,
                                                             const float* __restrict__ W2, float* __restrict__ gW1,
                                                             float* __restrict__ gb1, float* __restrict__ gW2,
                                                             float* __restrict__ gb2) {
    extern __shared__ __align__(16) float smem[];
    int S4 = (S + 3) & ~3;
    if (S4 > 4 && (S4 & (S4 - 1))) { int p2 = 8; while (p2 < S4) p2 <<= 1; S4 = p2; }   // power of two: 4, 8, 16, 32, 64
    const int CW = kPropBwdSlab / S4;   // 1024 .. 64 columns
    const int CWP = CW + 4;             // padded row pitch (bank spread for the row-strided weight-gradient reads)
    const int ncg = CW / 4;             // column groups of 4
    const int nrg = 256 / ncg;          // row groups working in parallel (== S4/4)
    float* sx = smem;                 // [S4][CW]  x
    float* sp = sx + S4 * CWP;        // [S4][CW]  pre -> dpre
    float* sh = sp + S4 * CWP;        // [S4][CW]  h
    float* sd = sh + S4 * CWP;        // [S4][CW]  dy
    float* w1 = sd + S4 * CWP;        // [S4][S4]  W1[j][i]
    float* w1t = w1 + S4 * S4;        // [S4][S4]  W1^T: w1t[i][j] = W1[j][i]
    float* w2 = w1t + S4 * S4;        // [S4][S4]  W2[j][i]
    float* sb1 = w2 + S4 * S4;        // [S4]
    for (int i = threadIdx.x; i < S4 * S4; i += blockDim.x) {
        const int a = i / S4, b = i % S4;
        const bool ok = a < S && b < S;
        w1[i] = ok ? W1[a * S + b] : 0.f;
        w1t[i] = ok ? W1[b * S + a] : 0.f;
        w2[i] = ok ? W2[a * S + b] : 0.f;
    }
    for (int i = threadIdx.x; i < S4; i += blockDim.x) sb1[i] = i < S ? b1[i] : 0.f;
    const int cg = threadIdx.x % ncg, rg = threadIdx.x / ncg;
    // weight-gradient work split: (S4/4)^2 tiles of 4x4 entries x ncp column partitions
    const int nt1 = S4 / 4, ntile = nt1 * nt1, ncp = 256 / ntile;
    const int tile = threadIdx.x % ntile, cpart = threadIdx.x / ntile;
    const int rj = tile / nt1, ci = tile % nt1;
    float aw1[4][4], aw2[4][4], ab1[4], ab2[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        ab1[a] = ab2[a] = 0.f;
#pragma unroll
        for (int b = 0; b < 4; ++b) aw1[a][b] = aw2[a][b] = 0.f;
    }
    const long long ncb = (IC + CW - 1) / CW;
    const long long nslab = n_outer * ncb;
    // out[o][c] = sum_k wt[k][o] * src[k][c]   (4x4 register tile)
    auto mm = [&](const float* wt, const float* src, int jt, float (&acc)[4][4]) {
#pragma unroll 4
        for (int k = 0; k < S4; ++k) {
            const float4 w4 = *reinterpret_cast<const float4*>(wt + k * S4 + jt * 4);
            const float4 v4 = *reinterpret_cast<const float4*>(src + k * CWP + cg * 4);
            const float w[4] = {w4.x, w4.y, w4.z, w4.w};
            const float v[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[a][c] = fmaf(w[a], v[c], acc[a][c]);
        }
    };
    for (long long slab = blockIdx.x; slab < nslab; slab += gridDim.x) {
        const long long outer = slab / ncb;
        const long long col0 = (slab % ncb) * CW;
        const int ncol = (int)min((long long)CW, IC - col0);
        const float* xb = xin + (size_t)outer * S * IC + col0;
        float* db = dy + (size_t)outer * S * IC + col0;
        __syncthreads();
        for (int i = threadIdx.x; i < S4 * ncg; i += blockDim.x) {
            const int p = i / ncg, c4 = (i % ncg) * 4;
            float4 xv = make_float4(0.f, 0.f, 0.f, 0.f), dv = xv;
            if (p < S && c4 < ncol) {
                xv = *reinterpret_cast<const float4*>(xb + (size_t)p * IC + c4);
                dv = *reinterpret_cast<const float4*>(db + (size_t)p * IC + c4);
            }
            *reinterpret_cast<float4*>(sx + p * CWP + c4) = xv;
            *reinterpret_cast<float4*>(sd + p * CWP + c4) = dv;
        }
        __syncthreads();
        // pass A: pre = W1 x + b1, h = gelu(pre)
        for (int jt = rg; jt < nt1; jt += nrg) {
            float acc[4][4];
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[a][c] = sb1[jt * 4 + a];
            mm(w1t, sx, jt, acc);
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                *reinterpret_cast<float4*>(sp + (jt * 4 + a) * CWP + cg * 4) = make_float4(acc[a][0], acc[a][1], acc[a][2], acc[a][3]);
                *reinterpret_cast<float4*>(sh + (jt * 4 + a) * CWP + cg * 4) =
                    make_float4(ActMath<TM>::gelu_erf_f(acc[a][0]), ActMath<TM>::gelu_erf_f(acc[a][1]), ActMath<TM>::gelu_erf_f(acc[a][2]),
                                ActMath<TM>::gelu_erf_f(acc[a][3]));
            }
        }
        __syncthreads();
        // pass B: dh[i] = sum_j W2[j][i] dy[j];  dpre = dh * gelu'(pre)   (overwrites sp)
        for (int it = rg; it < nt1; it += nrg) {
            float acc[4][4];
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[a][c] = 0.f;
            mm(w2, sd, it, acc);
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                float4* pp = reinterpret_cast<float4*>(sp + (it * 4 + a) * CWP + cg * 4);
                const float4 pr = *pp;
                *pp = make_float4(acc[a][0] * ActMath<TM>::gelu_erf_g(pr.x), acc[a][1] * ActMath<TM>::gelu_erf_g(pr.y),
                                  acc[a][2] * ActMath<TM>::gelu_erf_g(pr.z), acc[a][3] * ActMath<TM>::gelu_erf_g(pr.w));
            }
        }
        __syncthreads();
        // pass C: dx[i] = dy[i] + sum_j W1[j][i] dpre[j]
        for (int it = rg; it < nt1; it += nrg) {
            float acc[4][4];
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[a][c] = 0.f;
            mm(w1, sp, it, acc);
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                const int p = it * 4 + a;
                if (p < S && cg * 4 < ncol) {
                    const float4 d4 = *reinterpret_cast<const float4*>(sd + p * CWP + cg * 4);
                    *reinterpret_cast<float4*>(db + (size_t)p * IC + cg * 4) =
                        make_float4(d4.x + acc[a][0], d4.y + acc[a][1], d4.z + acc[a][2], d4.w + acc[a][3]);
                }
            }
        }
        // weight gradients: gW2[j][i] += sum_c dy[j][c] h[i][c];  gW1[j][i] += sum_c dpre[j][c] x[i][c]
        for (int c = cpart; c < CW; c += ncp) {
            float dyv[4], dpv[4], hv[4], xv[4];
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                dyv[a] = sd[(rj * 4 + a) * CWP + c];
                dpv[a] = sp[(rj * 4 + a) * CWP + c];
                hv[a] = sh[(ci * 4 + a) * CWP + c];
                xv[a] = sx[(ci * 4 + a) * CWP + c];
            }
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    aw2[a][b] = fmaf(dyv[a], hv[b], aw2[a][b]);
                    aw1[a][b] = fmaf(dpv[a], xv[b], aw1[a][b]);
                }
            if (ci == 0) {
#pragma unroll
                for (int a = 0; a < 4; ++a) { ab2[a] += dyv[a]; ab1[a] += dpv[a]; }
            }
        }
    }
    // reduce the column partitions in shared memory, then one global atomic per entry and CTA
    __syncthreads();
    float* r1 = sx;                    // [S4][S4]
    float* r2 = r1 + S4 * S4;          // [S4][S4]
    float* rb = r2 + S4 * S4;          // [2][S4]
    for (int i = threadIdx.x; i < 2 * S4 * S4 + 2 * S4; i += blockDim.x) r1[i] = 0.f;
    __syncthreads();
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int j = rj * 4 + a;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int i = ci * 4 + b;
            atomicAdd(&r1[j * S4 + i], aw1[a][b]);
            atomicAdd(&r2[j * S4 + i], aw2[a][b]);
        }
        if (ci == 0) { atomicAdd(&rb[j], ab1[a]); atomicAdd(&rb[S4 + j], ab2[a]); }
    }
    __syncthreads();
    for (int e = threadIdx.x; e < S * S; e += blockDim.x) {
        const int j = e / S, i = e % S;
        atomicAdd(gW1 + e, r1[j * S4 + i]);
        atomicAdd(gW2 + e, r2[j * S4 + i]);
    }
    for (int j = threadIdx.x; j < S; j += blockDim.x) { atomicAdd(gb1 + j, rb[j]); atomicAdd(gb2 + j, rb[S4 + j]); }
}

// ---- propagator backward for axes of 65 .. 96 tokens ---------------------------------------------------------------
// The tiled kernel above needs a power-of-two axis of at most 64 rows; this one keeps both S x S matrices and a slab of 32
// columns in shared memory and lets one lane own one column (warp w: rows w, w + 8, ...).  Weight gradients: thread t owns the
// entries t, t + 256, ... of the two S x S matrices, accumulated in registers over the slabs of a persistent CTA and flushed with
// one atomic per entry.  Same math as propagator_bwd_kernel.
constexpr int kPropWideMaxS = 96;
constexpr int kPropWideCols = 32;
constexpr int kPropWidePitch = kPropWideCols + 1;
constexpr int kPropWidePairs = (kPropWideMaxS * kPropWideMaxS + 255) / 256;
static inline size_t prop_bwd_wide_smem(int S) { return ((size_t)4 * S * kPropWidePitch + (size_t)2 * S * S + S) * sizeof(float); }
template <typename TM>
__global__ void __launch_bounds__(256) propagator_bwd_wide_kernel(const float* __restrict__ xin, float* __restrict__ dy, int S,
                                                                  long long IC, long long n_outer, const float* __restrict__ W1,
                                                                  const float* __restrict__ b1, const float* __restrict__ W2,
                                                                  float* __restrict__ gW1, float* __restrict__ gb1,
                                                                  float* __restrict__ gW2, float* __restrict__ gb2) {
    extern __shared__ __align__(16) float smem[];
    constexpr int CP = kPropWidePitch;
    float* sx = smem;               // [S][33] x
    float* sd = sx + S * CP;        // dy
    float* sp = sd + S * CP;        // pre -> dpre
    float* sh = sp + S * CP;        // h
    float* w1 = sh + S * CP;        // [S][S] W1[j][i]
    float* w2 = w1 + S * S;         // [S][S] W2[j][i]
    float* sb1 = w2 + S * S;        // [S]
    for (int i = threadIdx.x; i < S * S; i += blockDim.x) { w1[i] = W1[i]; w2[i] = W2[i]; }
    for (int i = threadIdx.x; i < S; i += blockDim.x) sb1[i] = b1[i];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float aw1[kPropWidePairs], aw2[kPropWidePairs];
#pragma unroll
    for (int k = 0; k < kPropWidePairs; ++k) aw1[k] = aw2[k] = 0.f;
    float ab1 = 0.f, ab2 = 0.f;
    const long long ncb = (IC + kPropWideCols - 1) / kPropWideCols;
    const long long nslab = n_outer * ncb;
    for (long long slab = blockIdx.x; slab < nslab; slab += gridDim.x) {
        const long long outer = slab / ncb;
        const long long col0 = (slab % ncb) * kPropWideCols;
        const int ncol = (int)min((long long)kPropWideCols, IC - col0);
        const float* xb = xin + (size_t)outer * S * IC + col0;
        float* db = dy + (size_t)outer * S * IC + col0;
        __syncthreads();
        for (int i = threadIdx.x; i < S * kPropWideCols; i += blockDim.x) {
            const int p = i / kPropWideCols, c = i % kPropWideCols;
            const bool ok = c < ncol;
            sx[p * CP + c] = ok ? xb[(size_t)p * IC + c] : 0.f;
            sd[p * CP + c] = ok ? db[(size_t)p * IC + c] : 0.f;
        }
        __syncthreads();
        // pre = W1 x + b1, h = gelu(pre);  dh[i] = sum_j W2[j][i] dy[j], dpre = dh * gelu'(pre)  (row i: the same warp, same lane)
        for (int j = warp; j < S; j += 8) {
            float acc = sb1[j], dh = 0.f;
            for (int i = 0; i < S; ++i) {
                acc = fmaf(w1[j * S + i], sx[i * CP + lane], acc);
                dh = fmaf(w2[i * S + j], sd[i * CP + lane], dh);
            }
            sh[j * CP + lane] = ActMath<TM>::gelu_erf_f(acc);
            sp[j * CP + lane] = dh * ActMath<TM>::gelu_erf_g(acc);
        }
        __syncthreads();
        // dx[i] = dy[i] + sum_j W1[j][i] dpre[j]
        for (int i = warp; i < S; i += 8) {
            float acc = sd[i * CP + lane];
            for (int j = 0; j < S; ++j) acc = fmaf(w1[j * S + i], sp[j * CP + lane], acc);
            if (lane < ncol) db[(size_t)i * IC + lane] = acc;
        }
        // weight gradients: gW2[j][i] += sum_c dy[j][c] h[i][c];  gW1[j][i] += sum_c dpre[j][c] x[i][c]  (padding columns hold zeros)
#pragma unroll
        for (int k = 0; k < kPropWidePairs; ++k) {
            const int q = threadIdx.x + 256 * k;
            if (q < S * S) {
                const int j = q / S, i = q % S;
                float a1 = 0.f, a2 = 0.f;
#pragma unroll 8
                for (int c = 0; c < kPropWideCols; ++c) {
                    a2 = fmaf(sd[j * CP + c], sh[i * CP + c], a2);
                    a1 = fmaf(sp[j * CP + c], sx[i * CP + c], a1);
                }
                aw1[k] += a1;
                aw2[k] += a2;
            }
        }
        if (threadIdx.x < S) {
            float a1 = 0.f, a2 = 0.f;
            for (int c = 0; c < kPropWideCols; ++c) { a2 += sd[threadIdx.x * CP + c]; a1 += sp[threadIdx.x * CP + c]; }
            ab1 += a1;
            ab2 += a2;
        }
    }
#pragma unroll
    for (int k = 0; k < kPropWidePairs; ++k) {
        const int q = threadIdx.x + 256 * k;
        if (q < S * S) { atomicAdd(gW1 + q, aw1[k]); atomicAdd(gW2 + q, aw2[k]); }
    }
    if (threadIdx.x < S) { atomicAdd(gb1 + threadIdx.x, ab1); atomicAdd(gb2 + threadIdx.x, ab2); }
}

// ---- Taylor head backward (tante.py:156-171 + dec_conv_3, enc_dec_cnn.py:273) ---------------------------
// frames_i = u0 + sum_k d_k c_ik, c_ik = (i*fi)^k/k!.  One thread per stage-1 row (k0 x k0 x D outputs) gathers
//   Gk[o]  = sum_{i<=n_b} gframes_i[o] * c_ik   -> G[k][row][kHeadPad]  (TA, zero-padded to 64 columns)
//   du0[o] = sum_{i<=n_b} gframes_i[o]          -> grad_input[b, T-1] (nullable)
// The two contractions that follow -- dz_k = G_k W3_k^T and dW3_k = z_k^T G_k -- are thin GEMMs on the padded
// matrices (tensor cores in bf16 mode), the bias gradient is a column sum of G_k.
constexpr int kHeadPad = 64;        // k0*k0*D <= 64 (D <= 16)
struct HeadBwdParams {
    void* G[kMaxOrder];             // [rows][kHeadPad]
    int K;
    float fi;
    const float* gframes;           // frame i of sample b at gframes + b * gf_bs + i * D * H * W
    long long gf_bs;                // (contiguous (B, n_cap, D, H, W): n_cap * D * H * W)
    int n_cap;
    const int* n_arr;               // [B]
    float* gi_last;                 // gradient of the LAST window frame (u0 path) of sample 0, += ; null: not needed
    long long gi_bs;                // its batch stride in elements
    // per-sample cursor mode (tante_backward_hist; null: off): gframes is the gradient of the whole prediction buffer, sample b's
    // frame i at (cur[b] + i - 1); once cur[b] > 0 the u0 of the call is prediction cur[b] - 1, whose gradient goes to gpred
    const int* cur;
    float* gpred;
};

// Window of a training call given as T separate frames (the chained BPTT rollout of the training drivers slides its window over
// ONE history instead of torch.cat-ing a new tensor per call, trainer/trainer.py:151-157): frame t of sample b lives at
// base + off[t] + b * bs[t] (elements, relative to the base pointer the kernel is given).  off[t] = kFrameSkip: no gradient wanted.
// Per-sample cursor mode (cur != null; tante_train_forward_hist / tante_backward_hist): every sample slides over its own history at
// its own pace -- window frame t of sample b is history frame i = cur[b] + t, the caller's input frame (off[i], bs[i]) below T, else
// prediction i - T at hoff + (i - T) * D * H * W + b * hbs.
constexpr long long kFrameSkip = (long long)(-0x7fffffffffffffffLL - 1);
struct FrameTab { long long off[16]; long long bs[16]; int on; const int* cur; long long hoff, hbs; };

// thread = (stage-1 row, group of 4 consecutive outputs): 16 threads per row, coalesced 128-byte row writes
__device__ __forceinline__ void patch_pixel(const PatchGeom& g, int h1, int w1, int oo, int& d, size_t& pix) {
    d = oo % g.D;
    const int cp = (oo / g.D) % g.k0;
    const int c = oo / (g.D * g.k0);
    pix = (size_t)(h1 * g.k0 + c) * g.W + (w1 * g.k0 + cp);
}
__device__ __forceinline__ void row_coords(const PatchGeom& g, long long row, long long& bt, int& h1, int& w1) {
    long long tkn = row / g.R1;
    const int r = (int)(row % g.R1);
    const int wp = (int)(tkn % g.Wp); tkn /= g.Wp;
    const int hpp = (int)(tkn % g.Hp);
    bt = tkn / g.Hp;
    stage1_row_to_hw(g, hpp, wp, r, h1, w1);
}

// ---- pixel planes <-> padded stage-1 row matrices, one 64-row tile per CTA -------------------------------------
// The row matrices are [rows][kHeadPad] with rows in the nested (image, hp, wp, a, a', b, b') order and columns
// (c, c', d); the pixel side is channels-first (image, d, H, W).  Both sides are touched with full-width accesses:
// pixel side = thread per VEC-pixel run along W of one (token, field, pixel row), consecutive threads walk along W;
// row side = thread per 16-byte chunk of a row.  A shared-memory tile S[row][kPatchPitch] sits in between.
__device__ __forceinline__ uint32_t bf16x2_bits(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}
constexpr int kPatchRows = 64;
constexpr int kPatchPitch = kHeadPad + 4;     // floats; rows 16 B aligned, row stride = 4 banks
struct PatchTile {
    int P, NT, lP, lNT;
    int stab[32];                             // RH[8], RW[8], OH[8], OW[8]   (see taylor_head_mma_kernel)
    long long pix0[kPatchRows];               // per token: pixel offset of its top-left corner in a plane
    long long img[kPatchRows];                // per token: image index (-1 = past the end)
    long long base[kPatchRows];               // per token: element offset of its image (frame tables only)
};
// image index b * T + t -> address through a frame table (call after patch_tile_init, before a __syncthreads)
__device__ __forceinline__ void patch_tile_frames(PatchTile& pt, const PatchGeom& g, const FrameTab& ft) {
    if (threadIdx.x < kPatchRows / g.R1) {
        const long long e = pt.img[threadIdx.x];
        if (e >= 0) {
            const long long b = e / g.T;
            const int t = (int)(e - b * g.T) + (ft.cur ? ft.cur[b] : 0);
            if (t >= g.T) pt.base[threadIdx.x] = ft.hoff + (long long)(t - g.T) * g.D * g.H * g.W + b * ft.hbs;
            else if (ft.off[t] == kFrameSkip) pt.img[threadIdx.x] = -1;
            else pt.base[threadIdx.x] = ft.off[t] + b * ft.bs[t];
        }
    }
}
__device__ __forceinline__ void patch_tile_init(PatchTile& pt, const PatchGeom& g, long long row0, long long rows_total) {
    const int tid = threadIdx.x;
    if (tid == 0) {
        pt.P = g.k0 * g.k1 * g.k2;
        pt.NT = kPatchRows / g.R1;
        pt.lP = 31 - __clz(pt.P);
        pt.lNT = 31 - __clz(pt.NT);
    }
    const int P = g.k0 * g.k1 * g.k2;
    if (tid < P) {
        const int c = tid % g.k0, b = (tid / g.k0) % g.k1, a = tid / (g.k0 * g.k1);
        pt.stab[tid] = a * g.k2 * g.k1 * g.k1 + b * g.k1;
        pt.stab[8 + tid] = a * g.k1 * g.k1 + b;
        pt.stab[16 + tid] = c * g.k0 * g.D;
        pt.stab[24 + tid] = c * g.D;
    }
    if (tid < kPatchRows / g.R1) {
        long long tkn = row0 / g.R1 + tid;
        if (tkn < rows_total / g.R1) {
            const int wp = (int)(tkn % g.Wp); tkn /= g.Wp;
            const int hpp = (int)(tkn % g.Hp);
            pt.img[tid] = tkn / g.Hp;
            pt.pix0[tid] = (long long)hpp * P * g.W + (long long)wp * P;
        } else {
            pt.img[tid] = -1; pt.pix0[tid] = 0;
        }
    }
}
// pixel-side work item -> (token, field, pixel row, run) ; returns false past the end
template <int VEC>
__device__ __forceinline__ bool patch_item(const PatchTile& pt, const PatchGeom& g, int item, int& tok, int& d, size_t& pix,
                                           int (&soff)[VEC]) {
    const int lPQ = pt.lP - (VEC == 4 ? 2 : 1);
    const int wq = item & ((1 << lPQ) - 1);
    tok = (item >> lPQ) & (pt.NT - 1);
    const int rest = item >> (lPQ + pt.lNT);
    const int hr = rest & (pt.P - 1);
    d = rest >> pt.lP;
    if (pt.img[tok] < 0) return false;
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
        const int wl = wq * VEC + e;
        soff[e] = (tok * g.R1 + pt.stab[hr] + pt.stab[8 + wl]) * kPatchPitch + pt.stab[16 + hr] + pt.stab[24 + wl] + d;
    }
    pix = (size_t)pt.pix0[tok] + (size_t)hr * g.W + wq * VEC;
    return true;
}
// row side: S tile -> [rows][kHeadPad] TA (columns >= ncols_valid come out as the zeros the tile was cleared to)
template <typename TA>
__device__ __forceinline__ void patch_rows_store(const float* S, TA* __restrict__ dst, long long row0, long long rows_total) {
    constexpr int CH = (int)(16 / sizeof(TA));       // elements per 16-byte chunk
    constexpr int NCH = kHeadPad / CH;
    for (int i = threadIdx.x; i < kPatchRows * NCH; i += blockDim.x) {
        const int r = i / NCH, ch = i % NCH;
        if (row0 + r >= rows_total) continue;
        const float* sp = S + r * kPatchPitch + ch * CH;
        TA* dp = dst + (size_t)(row0 + r) * kHeadPad + ch * CH;
        const float4 lo = *reinterpret_cast<const float4*>(sp);
        if constexpr (CH == 4) {
            *reinterpret_cast<float4*>(dp) = lo;
        } else {
            const float4 hi = *reinterpret_cast<const float4*>(sp + 4);
            uint4 u;
            u.x = bf16x2_bits(lo.x, lo.y); u.y = bf16x2_bits(lo.z, lo.w);
            u.z = bf16x2_bits(hi.x, hi.y); u.w = bf16x2_bits(hi.z, hi.w);
            *reinterpret_cast<uint4*>(dp) = u;
        }
    }
}
template <typename TA>
__device__ __forceinline__ void patch_rows_load(float* S, const TA* __restrict__ src, long long row0, long long rows_total) {
    constexpr int CH = (int)(16 / sizeof(TA));
    constexpr int NCH = kHeadPad / CH;
    for (int i = threadIdx.x; i < kPatchRows * NCH; i += blockDim.x) {
        const int r = i / NCH, ch = i % NCH;
        if (row0 + r >= rows_total) continue;
        const TA* gp = src + (size_t)(row0 + r) * kHeadPad + ch * CH;
        float* sp = S + r * kPatchPitch + ch * CH;
        float v[4];
        Vec4<TA>::load(gp, v);
        sp[0] = v[0]; sp[1] = v[1]; sp[2] = v[2]; sp[3] = v[3];
        if (CH == 8) {
            Vec4<TA>::load(gp + 4, v);
            sp[4] = v[0]; sp[5] = v[1]; sp[6] = v[2]; sp[7] = v[3];
        }
    }
}

template <typename TA, int VEC>
__global__ void __launch_bounds__(128) head_gather_kernel(HeadBwdParams hp, PatchGeom g, long long rows_total) {
    extern __shared__ __align__(16) float hg_smem[];          // [K][64][kPatchPitch]
    __shared__ PatchTile pt;
    const long long row0 = (long long)blockIdx.x * kPatchRows;
    patch_tile_init(pt, g, row0, rows_total);                 // rows are (b, hp, wp, r): the "image" is the sample
    for (int i = threadIdx.x; i < hp.K * kPatchRows * kPatchPitch; i += blockDim.x) hg_smem[i] = 0.f;
    __syncthreads();
    const size_t HW = (size_t)g.H * g.W;
    const int nitems = (g.D * pt.P * pt.NT) << (pt.lP - (VEC == 4 ? 2 : 1));
    for (int item = threadIdx.x; item < nitems; item += blockDim.x) {
        int tok, d, soff[VEC];
        size_t pix;
        if (!patch_item<VEC>(pt, g, item, tok, d, pix, soff)) continue;
        const long long b = pt.img[tok];
        const int n = min(hp.n_arr[b], hp.n_cap);
        const int c = hp.cur ? hp.cur[b] : 0;
        float Gk[4][VEC], du[VEC];
#pragma unroll
        for (int e = 0; e < VEC; ++e) { du[e] = 0.f; Gk[0][e] = Gk[1][e] = Gk[2][e] = Gk[3][e] = 0.f; }
        for (int i = 1; i <= n; ++i) {
            float gv[VEC];
            VecN<VEC>::load(hp.gframes + (size_t)b * hp.gf_bs + ((size_t)(c + i - 1) * g.D + d) * HW + pix, gv);
            const float dt = (float)i * hp.fi;
            float coef = 1.f;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                coef *= dt / (float)(k + 1);
#pragma unroll
                for (int e = 0; e < VEC; ++e) Gk[k][e] = fmaf(gv[e], coef, Gk[k][e]);
            }
#pragma unroll
            for (int e = 0; e < VEC; ++e) du[e] += gv[e];
        }
        float* gu0 = c > 0 ? hp.gpred + (size_t)b * hp.gf_bs + (size_t)(c - 1) * g.D * HW
                           : (hp.gi_last ? hp.gi_last + (size_t)b * hp.gi_bs : nullptr);
        if (gu0 && n > 0) {
            float* gp = gu0 + (size_t)d * HW + pix;
            float cur[VEC];
            VecN<VEC>::load(gp, cur);
#pragma unroll
            for (int e = 0; e < VEC; ++e) cur[e] += du[e];
            VecN<VEC>::store(gp, cur);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (k < hp.K) {
#pragma unroll
                for (int e = 0; e < VEC; ++e) hg_smem[k * kPatchRows * kPatchPitch + soff[e]] = Gk[k][e];
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (k < hp.K) patch_rows_store<TA>(hg_smem + k * kPatchRows * kPatchPitch, reinterpret_cast<TA*>(hp.G[k]), row0, rows_total);
}

// ---- first patch conv (enc_conv_1, enc_dec_cnn.py:220-221) as im2col + GEMM in training ----------------------
// im2col of the input patches, TA [rows][kHeadPad] zero-padded (K1 = k0*k0*D columns in the packed conv-weight
// order (c, c', d)): the A operand of the forward conv GEMM and the B operand of its weight-gradient GEMM.
template <typename TA, int VEC>
__global__ void __launch_bounds__(128) conv1_im2col_kernel(const float* __restrict__ x, PatchGeom g,
                                                           TA* __restrict__ cols, long long rows_total,
                                                           const int* __restrict__ enc_list = nullptr,
                                                           const int* __restrict__ enc_count = nullptr,
                                                           const int* __restrict__ fcount = nullptr, FrameTab ft = FrameTab()) {
    __shared__ __align__(16) float S[kPatchRows * kPatchPitch];
    __shared__ PatchTile pt;
    const long long row0 = (long long)blockIdx.x * kPatchRows;
    if (enc_list) {
        // blocks are numbered by compact image: everything past the list leaves before touching shared memory
        const long long first_img = row0 / ((long long)g.R1 * g.Hp * g.Wp);
        if (first_img >= *enc_count) return;
    }
    patch_tile_init(pt, g, row0, rows_total);
    for (int i = threadIdx.x; i < kPatchRows * kPatchPitch; i += blockDim.x) S[i] = 0.f;
    __syncthreads();
    // Rollout: the image a row block reads is not the one it is numbered after.  `enc_list` (encoder cache): block image e is
    // the frame in ring slot enc_list[e], images >= *enc_count are not encoded at all; `fcount` (ring window without the
    // cache): logical frame t of sample b lives in slot (fcount[b] + t) % T.
    if ((enc_list || fcount) && threadIdx.x < kPatchRows / g.R1) {
        long long e = pt.img[threadIdx.x];
        if (e >= 0) {
            if (enc_list) e = e < *enc_count ? enc_list[e] : -1;
            else { const long long b = e / g.T; e = b * g.T + (fcount[b] + (int)(e - b * g.T)) % g.T; }
            pt.img[threadIdx.x] = e;
        }
    }
    if (enc_list || fcount) __syncthreads();
    if (ft.on) { patch_tile_frames(pt, g, ft); __syncthreads(); }
    const size_t HW = (size_t)g.H * g.W;
    const int nitems = (g.D * pt.P * pt.NT) << (pt.lP - (VEC == 4 ? 2 : 1));
    bool any = false;
    for (int item = threadIdx.x; item < nitems; item += blockDim.x) {
        int tok, d, soff[VEC];
        size_t pix;
        if (!patch_item<VEC>(pt, g, item, tok, d, pix, soff)) continue;
        float v[VEC];
        const long long ib = ft.on ? pt.base[tok] : pt.img[tok] * (long long)(g.D * HW);
        VecN<VEC>::load(x + ib + (size_t)d * HW + pix, v);
#pragma unroll
        for (int e = 0; e < VEC; ++e) S[soff[e]] = v[e];
        any = true;
    }
    if (!__syncthreads_or(any)) return;          // nothing of this block is encoded (frames past the list)
    // rows of skipped tokens are written as zeros (harmless: past the GEMM's device-side row count or masked out)
    patch_rows_store<TA>(S, cols, row0, rows_total);
}

// grad_input[patch] += dpatch[row][kk]   (dpatch = da1 * W1, a thin GEMM; patches do not overlap)
template <typename TA, int VEC>
__global__ void __launch_bounds__(128) conv1_col2im_kernel(const TA* __restrict__ dpatch, PatchGeom g,
                                                           float* __restrict__ grad_input, long long rows_total,
                                                           FrameTab ft = FrameTab()) {
    __shared__ __align__(16) float S[kPatchRows * kPatchPitch];
    __shared__ PatchTile pt;
    const long long row0 = (long long)blockIdx.x * kPatchRows;
    patch_tile_init(pt, g, row0, rows_total);
    if (ft.on) { __syncthreads(); patch_tile_frames(pt, g, ft); }
    patch_rows_load<TA>(S, dpatch, row0, rows_total);
    __syncthreads();
    const size_t HW = (size_t)g.H * g.W;
    const int nitems = (g.D * pt.P * pt.NT) << (pt.lP - (VEC == 4 ? 2 : 1));
    for (int item = threadIdx.x; item < nitems; item += blockDim.x) {
        int tok, d, soff[VEC];
        size_t pix;
        if (!patch_item<VEC>(pt, g, item, tok, d, pix, soff)) continue;
        const long long ib = ft.on ? pt.base[tok] : pt.img[tok] * (long long)(g.D * HW);
        float* gp = grad_input + ib + (size_t)d * HW + pix;
        float cur[VEC];
        VecN<VEC>::load(gp, cur);
#pragma unroll
        for (int e = 0; e < VEC; ++e) cur[e] += S[soff[e]];
        VecN<VEC>::store(gp, cur);
    }
}

// ---- generic weight gradient: C[N][K] += A[M][N]^T * B[M][K]  (split over M, fp32 atomics) -------------------
// 64 x 64 output tile per CTA, 256 threads x (4 x 4); rows of A and B are contiguous -> coalesced staging.
template <typename TAa, typename TBb>
__global__ void __launch_bounds__(256) wgrad_simt_kernel(const TAa* __restrict__ A, int lda, const TBb* __restrict__ Bm,
                                                         int ldb, float* __restrict__ Cout, int ldc, long long M, int N,
                                                         int K, long long m_per_cta) {
    __shared__ __align__(16) float As[16][64 + 4];
    __shared__ __align__(16) float Bs[16][64 + 4];
    const int n0 = blockIdx.x * 64, k0 = blockIdx.y * 64;
    const long long m_begin = (long long)blockIdx.z * m_per_cta;
    const long long m_end = min(M, m_begin + m_per_cta);
    const int ty = threadIdx.x / 16, tx = threadIdx.x % 16;
    const int lr = threadIdx.x / 16, lc = (threadIdx.x % 16) * 4;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (long long m0 = m_begin; m0 < m_end; m0 += 16) {
        const long long m = m0 + lr;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int n = n0 + lc + e, k = k0 + lc + e;
            As[lr][lc + e] = (m < m_end && n < N) ? to_f32<TAa>(A[(size_t)m * lda + n]) : 0.f;
            Bs[lr][lc + e] = (m < m_end && k < K) ? to_f32<TBb>(Bm[(size_t)m * ldb + k]) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int mm = 0; mm < 16; ++mm) {
            const float4 a4 = *reinterpret_cast<const float4*>(&As[mm][ty * 4]);
            const float4 b4 = *reinterpret_cast<const float4*>(&Bs[mm][tx * 4]);
            const float a[4] = {a4.x, a4.y, a4.z, a4.w};
            const float b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int n = n0 + ty * 4 + i;
        if (n >= N) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0 + tx * 4 + j;
            if (k < K) atomicAdd(Cout + (size_t)n * ldc + k, acc[i][j]);
        }
    }
}

template <typename TAa, typename TBb>
static cudaError_t launch_wgrad_simt(const TAa* A, int lda, const TBb* Bm, int ldb, float* Cout, int ldc, long long M,
                                     int N, int K, int num_sms, cudaStream_t st) {
    if (M <= 0) return cudaSuccess;
    const int gx = (N + 63) / 64, gy = (K + 63) / 64;
    long long splits = std::max<long long>(1, (2LL * num_sms) / (gx * gy));
    long long per = (M + splits - 1) / splits;
    per = std::max<long long>(256, (per + 15) / 16 * 16);
    splits = (M + per - 1) / per;
    dim3 grid(gx, gy, (unsigned)splits);
    wgrad_simt_kernel<TAa, TBb><<<grid, 256, 0, st>>>(A, lda, Bm, ldb, Cout, ldc, M, N, K, per);
    return cudaGetLastError();
}

// ---- gradient un-packer: packed-layout gradient arena -> flat caller buffer in state_dict layout ------------
struct UnpackDesc {
    long long src_off;   // into the gradient arena
    long long dst_off;   // into the flat gradient buffer
    long long numel;     // parameter elements
    int mode;            // PackMode of the gradient entry
    int d0, d1, k;
};

__global__ void __launch_bounds__(256) unpack_grads_kernel(const UnpackDesc* __restrict__ descs,
                                                           const float* __restrict__ garena, float* __restrict__ flat) {
    const UnpackDesc d = descs[blockIdx.y];
    const int kk = d.k * d.k;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < d.numel;
         i += (long long)gridDim.x * blockDim.x) {
        // i indexes the PACKED layout for the permutation modes (a bijection), the parameter for BIAS_REP
        if (d.mode == PACK_BIAS_REP) {
            float s = 0.f;
            for (int r = 0; r < kk; ++r) s += garena[d.src_off + (long long)r * d.d0 + i];
            flat[d.dst_off + i] = s;
            continue;
        }
        long long s = i;
        if (d.mode == PACK_CONV) {
            const int Ci = d.d1;
            const int ci = (int)(i % Ci);
            const int dd = (int)((i / Ci) % kk);
            const int co = (int)(i / ((long long)Ci * kk));
            s = ((long long)co * Ci + ci) * kk + dd;
        } else if (d.mode == PACK_DECONV_NK) {
            const int Ci = d.d0, Co = d.d1;
            const int ci = (int)(i % Ci);
            const int n = (int)(i / Ci);
            const int co = n % Co, dd = n / Co;
            s = ((long long)ci * Co + co) * kk + dd;
        } else if (d.mode == PACK_DECONV_KN) {
            const int Co = d.d1;
            const int n = (int)(i % ((long long)kk * Co));
            const int ci = (int)(i / ((long long)kk * Co));
            const int co = n % Co, dd = n / Co;
            s = ((long long)ci * Co + co) * kk + dd;
        }
        flat[d.dst_off + s] = garena[d.src_off + i];
    }
}

// derived copies of the packed GEMM weights for the backward GEMMs, zero-padded to [dst_rows][dst_ld]:
//   transpose = 1:  dst[k][r] = src[r][k]   (input-gradient GEMMs: dX = dY W)
//   transpose = 0:  dst[r][k] = src[r][k]   (padding only)
struct TransDesc { long long src_off, dst_off; int rows, cols, dst_rows, dst_ld, transpose; };
__global__ void __launch_bounds__(256) transpose_packed_kernel(const TransDesc* __restrict__ descs, float* __restrict__ arena,
                                                               __nv_bfloat16* __restrict__ arena_bf16) {
    const TransDesc d = descs[blockIdx.y];
    const long long n = (long long)d.dst_rows * d.dst_ld;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int a = (int)(i / d.dst_ld), b = (int)(i % d.dst_ld);      // dst[a][b]
        const int r = d.transpose ? b : a, k = d.transpose ? a : b;      // src[r][k]
        const float v = (r < d.rows && k < d.cols) ? arena[d.src_off + (long long)r * d.cols + k] : 0.f;
        arena[d.dst_off + i] = v;
        if (arena_bf16) arena_bf16[d.dst_off + i] = __float2bfloat16_rn(v);
    }
}

}  // namespace tante
