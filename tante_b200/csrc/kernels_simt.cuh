// Bandwidth-/latency-bound kernels of the TANTE forward: patch gather + first conv, LayerNorm,
// axial attention on short sequences, axis propagators, the step-size head, FiLM, and the fused
// last-deconv + Taylor/Horner emit.  Templated on the activation element type so the fp32 parity
// mode and the bf16 tensor mode share them.
#pragma once
#include "common.cuh"

namespace tante {

// ------------------------------------------------------------------------------------------------
// Patch geometry.  Patch_map[patch_scale] = (k0,k1,k2) (reference enc_dec_cnn.py:39-46), all strides
// equal to the kernel (overlap_ratio 0).  Pixels are addressed in a *nested* order
//   h = ((hp*k2 + a)*k1 + b)*k0 + c ,  w = ((wp*k2 + a')*k1 + b')*k0 + c'
// and every conv stage stores its rows as (bt, hp, wp, a, a', b, b'), so that each strided patch conv
// (and each transposed conv of the decoder) is a plain row-major GEMM on a reshaped matrix.
// ------------------------------------------------------------------------------------------------
struct PatchGeom {
    int k0, k1, k2;  // conv1/deconv3, conv2/deconv2, conv3/deconv1 kernel = stride
    int D, H, W, Hp, Wp, T;
    int R1;          // rows of stage-1 activations per latent token = (k1*k2)^2
    int R2;          // rows of stage-2 activations per latent token = k2^2
};

__device__ __forceinline__ void stage1_row_to_hw(const PatchGeom& g, int hp, int wp, int r, int& h1, int& w1) {
    // r = ((a*k2 + a')*k1 + b)*k1 + b'
    const int bp = r % g.k1; r /= g.k1;
    const int b = r % g.k1; r /= g.k1;
    const int ap = r % g.k2;
    const int a = r / g.k2;
    h1 = (hp * g.k2 + a) * g.k1 + b;
    w1 = (wp * g.k2 + ap) * g.k1 + bp;
}

// ------------------------------------------------------------------------------------------------
// K1: patch gather + conv1 (k0 x k0, D -> C1) + erf-GELU.
// Replaces enc_conv_1 + act of enc_CNN.forward (reference enc_dec_cnn.py:220-222) and the
// `b t d h w -> (b t) d h w` rearrange.  One CTA per (bt, hp, chunk of WC latent columns): the
// D x P x (P*WC) input slab is staged in shared memory with 128-bit loads (rows are contiguous in w),
// then each thread produces 16 output channels of one stage-1 pixel.
// `fcount` (nullable) makes the input a ring buffer of T slots per sample: logical frame t of sample b
// lives in slot (fcount[b] + t) % T (rollout window, see rollout.cuh).
// ------------------------------------------------------------------------------------------------
template <typename TOut, bool ACT = true /* false: write the pre-activation (training tape) */>
__global__ void __launch_bounds__(128) patch_embed_conv1_kernel(const float* __restrict__ x,
                                                                const int* __restrict__ fcount, PatchGeom g,
                                                                const float* __restrict__ w1p,  // [C1][k0*k0*D]
                                                                const float* __restrict__ b1, int WC,
                                                                TOut* __restrict__ out,
                                                                const int* __restrict__ enc_list = nullptr,
                                                                const int* __restrict__ enc_count = nullptr) {
    constexpr int C1 = 64;
    extern __shared__ __align__(16) float smem[];
    const int P = g.k0 * g.k1 * g.k2;
    const int K1 = g.k0 * g.k0 * g.D;
    const int slabW = P * WC + 1;               // +1: rows of the slab start in different banks
    float* s_in = smem;                         // [D][P][slabW]
    float* s_w = s_in + ((g.D * P * slabW + 3) & ~3);   // [K1][C1]  (transposed: one 256-B row per input tap)
    float* s_b = s_w + K1 * C1;                 // [C1]
    TOut* s_out = reinterpret_cast<TOut*>(s_b + C1);    // [rows][C1] staged for a coalesced write-back

    const int bt = blockIdx.x / g.Hp, hp = blockIdx.x % g.Hp;
    const int wp0 = blockIdx.y * WC;
    const int nwp = min(WC, g.Wp - wp0);
    // `enc_list` (rollout with the encoder cache): CTA row bt encodes the frame in ring slot enc_list[bt] and writes
    // compact rows; frames past *enc_count are not encoded at all.
    int b = bt / g.T, t = bt % g.T;
    int slot = fcount ? (fcount[b] + t) % g.T : t;
    if (enc_list) {
        if (bt >= *enc_count) return;
        b = enc_list[bt] / g.T;
        slot = enc_list[bt] % g.T;
    }
    const float* xin = x + ((size_t)(b * g.T + slot) * g.D) * g.H * g.W;

    for (int i = threadIdx.x; i < C1 * K1; i += blockDim.x) s_w[(i % K1) * C1 + (i / K1)] = w1p[i];
    for (int i = threadIdx.x; i < C1; i += blockDim.x) s_b[i] = b1[i];
    const int validW = P * nwp;
    if ((validW & 3) == 0 && (g.W & 3) == 0 && ((P * wp0) & 3) == 0) {
        const int vec = validW / 4;
        for (int i = threadIdx.x; i < g.D * P * vec; i += blockDim.x) {
            const int v = i % vec, row = (i / vec) % P, d = i / (vec * P);
            const float4 val = *reinterpret_cast<const float4*>(
                xin + ((size_t)d * g.H + hp * P + row) * g.W + wp0 * P + v * 4);
            float* dst = s_in + (d * P + row) * slabW + v * 4;
            dst[0] = val.x; dst[1] = val.y; dst[2] = val.z; dst[3] = val.w;
        }
    } else {
        for (int i = threadIdx.x; i < g.D * P * validW; i += blockDim.x) {
            const int c = i % validW, row = (i / validW) % P, d = i / (validW * P);
            s_in[(d * P + row) * slabW + c] = xin[((size_t)d * g.H + hp * P + row) * g.W + wp0 * P + c];
        }
    }
    __syncthreads();

    const int rows = nwp * g.R1;          // stage-1 pixels in this CTA (consecutive rows of `out`)
    for (int rr = threadIdx.x; rr < rows; rr += blockDim.x) {
        const int wpl = rr / g.R1, r = rr % g.R1;
        int h1, w1;
        stage1_row_to_hw(g, 0, wpl, r, h1, w1);   // local coordinates inside the slab (hp -> 0)
        float acc[C1];
#pragma unroll
        for (int j = 0; j < C1; ++j) acc[j] = s_b[j];
        int kk = 0;
        for (int c = 0; c < g.k0; ++c)
            for (int cp = 0; cp < g.k0; ++cp)
                for (int d = 0; d < g.D; ++d, ++kk) {
                    const float v = s_in[(d * P + h1 * g.k0 + c) * slabW + w1 * g.k0 + cp];
                    const float4* wr = reinterpret_cast<const float4*>(s_w + kk * C1);   // warp-broadcast reads
#pragma unroll
                    for (int j4 = 0; j4 < C1 / 4; ++j4) {
                        const float4 w4 = wr[j4];
                        acc[j4 * 4 + 0] = fmaf(v, w4.x, acc[j4 * 4 + 0]);
                        acc[j4 * 4 + 1] = fmaf(v, w4.y, acc[j4 * 4 + 1]);
                        acc[j4 * 4 + 2] = fmaf(v, w4.z, acc[j4 * 4 + 2]);
                        acc[j4 * 4 + 3] = fmaf(v, w4.w, acc[j4 * 4 + 3]);
                    }
                }
        // stage with a 16-byte-chunk rotation per row so that neither this store nor the copy below conflicts
        constexpr int CH = (int)(16 / sizeof(TOut));       // elements per 16-byte chunk
        constexpr int NCH = C1 / CH;
#pragma unroll
        for (int c4 = 0; c4 < C1 / 4; ++c4) {
            float v4[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) v4[j] = ACT ? gelu_erf_for<TOut>(acc[c4 * 4 + j]) : acc[c4 * 4 + j];
            const int chunk = (c4 * 4) / CH, within = (c4 * 4) % CH;
            Vec4<TOut>::store(s_out + (size_t)rr * C1 + ((chunk + rr) % NCH) * CH + within, v4);
        }
    }
    __syncthreads();
    {
        constexpr int CH = (int)(16 / sizeof(TOut));
        constexpr int NCH = C1 / CH;
        const size_t row_g0 = ((size_t)(bt * g.Hp + hp) * g.Wp + wp0) * g.R1;
        uint4* dst = reinterpret_cast<uint4*>(out + row_g0 * C1);
        for (int i = threadIdx.x; i < rows * NCH; i += blockDim.x) {
            const int rr = i / NCH, chunk = i % NCH;
            dst[i] = *reinterpret_cast<const uint4*>(s_out + (size_t)rr * C1 + ((chunk + rr) % NCH) * CH);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K3: LayerNorm over the channel dim (eps 1e-5), one warp per token; fp32 in, TOut out.
// Replaces ln1/ln2 of TransformerBlock (reference attn_backbone.py:47,51,66,82).
// ------------------------------------------------------------------------------------------------
template <typename TOut, int MAXV /* float4 per lane, C <= 128*MAXV */>
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, TOut* __restrict__ y,
                                                        int rows, int C, float eps) {
    pdl_trigger();
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) / kWarp;
    const int lane = threadIdx.x % kWarp;
    if (warp >= rows) return;
    const float* xr = x + (size_t)warp * C;
    float v[MAXV][4];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
        const int c = (i * kWarp + lane) * 4;
        if (c < C) {
            Vec4<float>::load(xr + c, v[i]);
            s += (v[i][0] + v[i][1]) + (v[i][2] + v[i][3]);
        } else {
            v[i][0] = v[i][1] = v[i][2] = v[i][3] = 0.f;
        }
    }
    const float mean = warp_sum(s) / (float)C;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
        const int c = (i * kWarp + lane) * 4;
        if (c < C) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float d = v[i][j] - mean;
                q = fmaf(d, d, q);
            }
        }
    }
    const float rstd = 1.0f / sqrtf(warp_sum(q) / (float)C + eps);
    TOut* yr = y + (size_t)warp * C;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
        const int c = (i * kWarp + lane) * 4;
        if (c < C) {
            float g4[4], b4[4], o[4];
            Vec4<float>::load(gamma + c, g4);
            Vec4<float>::load(beta + c, b4);
#pragma unroll
            for (int j = 0; j < 4; ++j) o[j] = (v[i][j] - mean) * rstd * g4[j] + b4[j];
            Vec4<TOut>::store(yr + c, o);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K4: axial multi-head attention on short sequences, addressed *in place* in the (B,T,Hp,Wp) token
// order (no rearrange copies).  Sequence `seq` = (outer, inner): token(pos) = (outer*S + pos)*inner_sz
// + inner.  Axis T: S=T, inner_sz=L (causal); H: S=Hp, inner_sz=Wp; W: S=Wp, inner_sz=1.
// Replaces nn.MultiheadAttention's core (reference attn_backbone.py:74-80; q scaled by 1/sqrt(hd),
// softmax over keys, causal = keys <= query).  One thread per (seq, head, query); keys/values are
// warp-broadcast reads (all lanes of a warp share seq and head when S >= 32).
// ------------------------------------------------------------------------------------------------
template <typename TIn, typename TOut, int HD>
__global__ void __launch_bounds__(128) axial_attention_kernel(const TIn* __restrict__ qkv, TOut* __restrict__ out,
                                                              int n_seq, int S, int inner_sz, int n_head, int C,
                                                              int causal, float scale, DropCfg drop = DropCfg(),
                                                              uint32_t site = 0) {
    const long long item = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)n_seq * n_head * S;
    if (item >= total) return;
    const int qpos = (int)(item % S);
    const int head = (int)((item / S) % n_head);
    const int seq = (int)(item / ((long long)S * n_head));
    const int outer = seq / inner_sz, inner = seq % inner_sz;
    const size_t tok0 = (size_t)outer * S * inner_sz + inner;
    const int ld = 3 * C;

    float q[HD], acc[HD];
    {
        const TIn* qp = qkv + (tok0 + (size_t)qpos * inner_sz) * ld + head * HD;
#pragma unroll
        for (int d = 0; d < HD; d += 4) {
            float t4[4];
            Vec4<TIn>::load(qp + d, t4);
#pragma unroll
            for (int j = 0; j < 4; ++j) q[d + j] = t4[j] * scale;
        }
    }
#pragma unroll
    for (int d = 0; d < HD; ++d) acc[d] = 0.f;
    float m = -INFINITY, l = 0.f;
    const int jend = causal ? qpos + 1 : S;
    for (int j = 0; j < jend; ++j) {
        const TIn* kp = qkv + (tok0 + (size_t)j * inner_sz) * ld + C + head * HD;
        float s = 0.f;
#pragma unroll
        for (int d = 0; d < HD; d += 4) {
            float t4[4];
            Vec4<TIn>::load(kp + d, t4);
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) s = fmaf(q[d + jj], t4[jj], s);
        }
        const float mn = fmaxf(m, s);
        const float corr = expf(m - mn);   // exp(-inf) = 0 on the first key
        const float p = expf(s - mn);
        l = l * corr + p;                  // the softmax normaliser sees every key; dropout acts on the probabilities
        float pz = p;
        if (drop.p > 0.f) {
            const long long tokq = (long long)tok0 + (long long)qpos * inner_sz;
            const uint4 w = drop_words(drop, site, drop_attn_grp(tokq, n_head, head, j));
            pz *= drop_mul(drop, w, j & 7);
        }
        const TIn* vp = kp + C;
#pragma unroll
        for (int d = 0; d < HD; d += 4) {
            float t4[4];
            Vec4<TIn>::load(vp + d, t4);
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) acc[d + jj] = fmaf(acc[d + jj], corr, pz * t4[jj]);
        }
        m = mn;
    }
    const float inv = 1.0f / l;
    TOut* op = out + (tok0 + (size_t)qpos * inner_sz) * C + head * HD;
#pragma unroll
    for (int d = 0; d < HD; d += 4) {
        float o4[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) o4[j] = acc[d + j] * inv;
        Vec4<TOut>::store(op + d, o4);
    }
}

// ------------------------------------------------------------------------------------------------
// K5: residual axis MLP ("propagator"): x += W2 * gelu_erf(W1 * x_axis + b1) + b2 along one axis of
// length S (reference attn_backbone.py:111-119,140-146), in place on the fp32 latent.  Element
// (outer, pos, col) lives at (outer*S + pos)*IC + col, IC = inner_sz*C contiguous floats.
// One CTA = one `outer` x 64 columns; the S x 64 slab and both S x S matrices sit in shared memory.
// ------------------------------------------------------------------------------------------------
template <typename TM /* float: accurate erf; bf16: erf_fast, as every other tensor-mode kernel */>
__global__ void __launch_bounds__(256) propagator_kernel(const float* xin, float* x, int S, long long IC,
                                                         const float* __restrict__ W1, const float* __restrict__ b1,
                                                         const float* __restrict__ W2, const float* __restrict__ b2) {
    // Register-tiled: each thread owns a 4 (axis positions) x 4 (columns) output tile; per reduction step it
    // reads one float4 of transposed weights (warp-broadcast) and one float4 of the slab -> 16 FMAs / 2 LDS.128.
    extern __shared__ __align__(16) float smem[];
    const int S4 = (S + 3) & ~3;
    float* sv = smem;                // [S4][128]
    float* sh = sv + S4 * 128;       // [S4][128]
    float* sw1 = sh + S4 * 128;      // [S4][S4]  transposed: sw1[i][j] = W1[j][i]
    float* sw2 = sw1 + S4 * S4;      // [S4][S4]  transposed
    float* sb1 = sw2 + S4 * S4;      // [S4]
    float* sb2 = sb1 + S4;
    const long long col0 = (long long)blockIdx.y * 128;
    const long long outer = blockIdx.x;
    float* base = x + (size_t)outer * S * IC + col0;
    const float* ibase = xin + (size_t)outer * S * IC + col0;     // xin == x: in place (inference); else out of place
    for (int i = threadIdx.x; i < S4 * S4; i += blockDim.x) {
        const int ii = i / S4, jj = i % S4;            // sw[ii][jj] = W[jj][ii]
        const bool ok = ii < S && jj < S;
        sw1[i] = ok ? W1[jj * S + ii] : 0.f;
        sw2[i] = ok ? W2[jj * S + ii] : 0.f;
    }
    for (int i = threadIdx.x; i < S4; i += blockDim.x) { sb1[i] = i < S ? b1[i] : 0.f; sb2[i] = i < S ? b2[i] : 0.f; }
    const int ncol = (int)min((long long)128, IC - col0);      // IC is a multiple of 4
    for (int i = threadIdx.x; i < S4 * 32; i += blockDim.x) {
        const int p = i / 32, c4 = (i % 32) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p < S && c4 < ncol) v = *reinterpret_cast<const float4*>(ibase + (size_t)p * IC + c4);
        *reinterpret_cast<float4*>(sv + p * 128 + c4) = v;
    }
    __syncthreads();
    const int cg = threadIdx.x % 32, rg = threadIdx.x / 32, nrg = blockDim.x / 32;
    for (int pass = 0; pass < 2; ++pass) {
        const float* src = pass == 0 ? sv : sh;
        const float* wt = pass == 0 ? sw1 : sw2;
        const float* bb = pass == 0 ? sb1 : sb2;
        for (int jt = rg; jt < S4 / 4; jt += nrg) {
            float acc[4][4];
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[a][c] = bb[jt * 4 + a];
#pragma unroll 4
            for (int i = 0; i < S4; ++i) {
                const float4 w4 = *reinterpret_cast<const float4*>(wt + i * S4 + jt * 4);
                const float4 v4 = *reinterpret_cast<const float4*>(src + i * 128 + cg * 4);
                const float w[4] = {w4.x, w4.y, w4.z, w4.w};
                const float v[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int c = 0; c < 4; ++c) acc[a][c] = fmaf(w[a], v[c], acc[a][c]);
            }
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                const int p = jt * 4 + a;
                if (pass == 0) {
                    *reinterpret_cast<float4*>(sh + p * 128 + cg * 4) =
                        make_float4(ActMath<TM>::gelu_erf_f(acc[a][0]), ActMath<TM>::gelu_erf_f(acc[a][1]),
                                    ActMath<TM>::gelu_erf_f(acc[a][2]), ActMath<TM>::gelu_erf_f(acc[a][3]));
                } else if (p < S && cg * 4 < ncol) {
                    const float4 x4 = *reinterpret_cast<const float4*>(sv + p * 128 + cg * 4);
                    *reinterpret_cast<float4*>(base + (size_t)p * IC + cg * 4) =
                        make_float4(x4.x + acc[a][0], x4.y + acc[a][1], x4.z + acc[a][2], x4.w + acc[a][3]);
                }
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// Head: snapshot of the last-frame latent (reference tante.py:147 `x[:, -1:]`), fp32 -> TOut.
// ------------------------------------------------------------------------------------------------
template <typename TOut>
__global__ void __launch_bounds__(256) last_frame_kernel(const float* __restrict__ x, TOut* __restrict__ d,
                                                         float* __restrict__ d32, int B, int T, long long LC) {
    const long long i4 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i4 >= (long long)B * LC) return;
    const long long b = i4 / LC, r = i4 % LC;
    float v[4];
    Vec4<float>::load(x + ((size_t)(b * T + T - 1)) * LC + r, v);
    Vec4<TOut>::store(d + i4, v);
    if (d32) Vec4<float>::store(d32 + i4, v);
}

// ------------------------------------------------------------------------------------------------
// Head: interprator tail (reference tante.py:191-201).  h2 = relu(L2(relu(L1(d)))) comes from two
// GEMMs; this kernel does the last Linear(C/4 -> 1), the clamp to [0, out_T-1] (forward value of the
// straight-through trick), the mean over the L tokens in a *fixed* order (deterministic, so that
// floor(R_t) is reproducible run to run) and + 1.001.  One CTA per sample.
// ------------------------------------------------------------------------------------------------
template <typename TIn>
__global__ void __launch_bounds__(256) rt_reduce_kernel(const TIn* __restrict__ h2, const float* __restrict__ w3,
                                                        const float* __restrict__ b3, int L, int C4, float out_T,
                                                        float* __restrict__ rt /* [B] */) {
    __shared__ float red[256];
    const int b = blockIdx.x;
    float s = 0.f;
    for (int l = threadIdx.x; l < L; l += 256) {
        const TIn* r = h2 + ((size_t)b * L + l) * C4;
        float a = b3[0];
        for (int c = 0; c < C4; c += 4) {
            float t4[4];
            Vec4<TIn>::load(r + c, t4);
#pragma unroll
            for (int j = 0; j < 4; ++j) a = fmaf(t4[j], w3[c + j], a);
        }
        a = fminf(fmaxf(a, 0.0f), out_T - 1.0f);
        s += a;
    }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) rt[b] = red[0] / (float)L + 1.001f;
}

// FiLM generator: scale,shift = Lin(C/2->C)(relu(Lin(1->C/2)(t))) (reference tante.py:206-220) for a
// vector of N conditions (t_seq for t_encode, rt_k[b] for the modifiers).  out: [N][2][C].  Grid = N.
__global__ void __launch_bounds__(256) film_params_kernel(const float* __restrict__ cond, float cond_scale,
                                                          const float* __restrict__ w0s, const float* __restrict__ b0s,
                                                          const float* __restrict__ w2s, const float* __restrict__ b2s,
                                                          const float* __restrict__ w0h, const float* __restrict__ b0h,
                                                          const float* __restrict__ w2h, const float* __restrict__ b2h,
                                                          int C, float* __restrict__ out) {
    extern __shared__ float smem[];
    const int Ch = C / 2;
    float* hs = smem;        // [Ch]
    float* hh = smem + Ch;   // [Ch]
    const float t = cond[blockIdx.x] * cond_scale;
    for (int i = threadIdx.x; i < Ch; i += blockDim.x) {
        hs[i] = fmaxf(fmaf(w0s[i], t, b0s[i]), 0.f);
        hh[i] = fmaxf(fmaf(w0h[i], t, b0h[i]), 0.f);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float a = b2s[c], h = b2h[c];
        for (int i = 0; i < Ch; ++i) {
            a = fmaf(w2s[(size_t)c * Ch + i], hs[i], a);
            h = fmaf(w2h[(size_t)c * Ch + i], hh[i], h);
        }
        out[((size_t)blockIdx.x * 2 + 0) * C + c] = a;
        out[((size_t)blockIdx.x * 2 + 1) * C + c] = h;
    }
}

// FiLM application on the (B, L, C) derivative latent: d <- d + d*scale[b] + shift[b] (tante.py:222-230).
template <typename TOut>
__global__ void __launch_bounds__(256) film_apply_kernel(const float* __restrict__ d32, const float* __restrict__ film,
                                                         TOut* __restrict__ out, long long LC, int C, long long total) {
    const long long i4 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i4 >= total) return;
    const long long b = i4 / LC;
    const int c = (int)(i4 % C);
    float v[4], s[4], h[4], o[4];
    Vec4<float>::load(d32 + i4, v);
    Vec4<float>::load(film + ((size_t)b * 2 + 0) * C + c, s);
    Vec4<float>::load(film + ((size_t)b * 2 + 1) * C + c, h);
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = v[j] + (v[j] * s[j] + h[j]);
    Vec4<TOut>::store(out + i4, o);
}

// ------------------------------------------------------------------------------------------------
// Encoder tail on cached encoder outputs (rollout): x[b, t] = embed(enc[b, slot(t)], t) with
// embed = t_encode FiLM + s_emb + t_emb (tante.py:132-141).  The encoder output of a frame does not depend on its
// position in the window, so a rollout step only encodes the frames that entered the window (`cnew`, compact, in
// enc_list order) and takes the others from `cache` (per ring slot); new outputs are copied into the cache here.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) embed_cached_kernel(const float* __restrict__ cnew, float* __restrict__ cache,
                                                           const int* __restrict__ enc_map, const int* __restrict__ fcount,
                                                           const float* __restrict__ film, const float* __restrict__ s_emb,
                                                           const float* __restrict__ t_emb, float* __restrict__ x, int B, int T,
                                                           int L, int C, const int* __restrict__ act = nullptr) {
    // 32-bit index arithmetic (B*T*L*C/4 < 2^31 is checked by the launcher): the 64-bit div/mod chain cost more than the copy
    const unsigned c4n = (unsigned)C / 4;
    const unsigned total = (unsigned)B * T * L * c4n;
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int c = (int)(i % c4n) * 4;
        unsigned tok = i / c4n;
        const int l = (int)(tok % (unsigned)L); tok /= (unsigned)L;
        const int t = (int)(tok % (unsigned)T);
        const int bc = (int)(tok / (unsigned)T);            // compact index of the latent
        const int b = act ? act[bc] : bc;                   // trajectory (ring slot, cache)
        const int slot = (fcount[b] + t) % T;
        const int e = enc_map[b * T + slot];
        float* cp = cache + ((size_t)(b * T + slot) * L + l) * C + c;
        float4 v;
        if (e >= 0) {
            v = *reinterpret_cast<const float4*>(cnew + ((size_t)e * L + l) * C + c);
            *reinterpret_cast<float4*>(cp) = v;
        } else {
            v = *reinterpret_cast<const float4*>(cp);
        }
        const float4 sc = *reinterpret_cast<const float4*>(film + (size_t)(t * 2 + 0) * C + c);
        const float4 sh = *reinterpret_cast<const float4*>(film + (size_t)(t * 2 + 1) * C + c);
        const float4 se = *reinterpret_cast<const float4*>(s_emb + (size_t)l * C + c);
        const float4 te = *reinterpret_cast<const float4*>(t_emb + (size_t)t * C + c);
        float4 o;
        o.x = embed_value(v.x, sc.x, sh.x, se.x, te.x); o.y = embed_value(v.y, sc.y, sh.y, se.y, te.y);
        o.z = embed_value(v.z, sc.z, sh.z, se.z, te.z); o.w = embed_value(v.w, sc.w, sh.w, se.w, te.w);
        *reinterpret_cast<float4*>(x + ((size_t)(bc * T + t) * L + l) * C + c) = o;
    }
}

// ------------------------------------------------------------------------------------------------
// Step-size selection (reference tante.py:156-163): R_t = mean_k rt_k, n = floor(R_t[gov]) with
// gov = b (per-sample) or 0 (reference batch semantics).  Also the rollout bookkeeping.
// ------------------------------------------------------------------------------------------------
struct RolloutPtrs {   // caller-owned output buffers, kept in device memory so that captured graphs are reusable
    float* y_out;      // (B, n_roll, H, W, D) channels-last history
    float* rts_out;    // [max_steps][B]
    int* ns_out;       // [max_steps][B]
};

struct RolloutState {
    int* cum;       // [B] frames emitted so far
    int* fcount;    // [B] frames ever in the ring (starts at T)
    int* steps;     // [B] model calls so far
    int* n_cur;     // [B] frames to emit this step (0 = sample finished)
    int* remaining; // [1] samples still running (written at the end of each step)
    int* iter;      // [1] model calls issued in this rollout
    // encoder cache: frames whose ring slot changed since the previous model call (all B*T before the first one)
    int* enc_count; // [1] number of entries of enc_list (null: no cache, every frame is encoded every call)
    int* enc_list;  // [B*T] b*T + slot, compact
    int* enc_map;   // [B*T] ring slot -> index into enc_list, or -1 (encoder output is in the cache)
    int T;
    const RolloutPtrs* ptrs;
    int n_roll;
    int max_steps;
    // Compaction (per-sample rollouts): act[0 .. n_active) = trajectories still running, in a stable order, followed by the
    // finished ones.  A model call works on the FIRST `B` entries of act (its "bucket": the smallest captured batch size
    // that holds every running trajectory): compact index i of the latent = trajectory act[i] of the ring / caches / outputs.
    // act == nullptr: identity (no compaction).
    int* act;       // [B_full]
    int* n_active;  // [1]
    int B_full;     // trajectories of the rollout (= stride of rts_out / ns_out)
    int n_buckets;  // captured batch sizes, descending (bucket_sz[0] = B_full); 0 = no SWITCH node
    int bucket_sz[4];
    cudaGraphConditionalHandle sw;
};

__global__ void set_rollout_ptrs_kernel(RolloutPtrs* dst, float* y, float* rts, int* ns) {
    dst->y_out = y; dst->rts_out = rts; dst->ns_out = ns;
}

__global__ void select_step_kernel(const float* __restrict__ rt /* [K][Bstride] */, int K, int Bstride, int B,
                                   int deg, int output_length, int per_sample, int n_cap,
                                   float* __restrict__ R_t, int* __restrict__ n_out, RolloutState rs, int rollout,
                                   const int* __restrict__ cur = nullptr, int n_lim = 0) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;      // compact index (rt / R_t / n_out are compact)
    if (b >= B) return;
    const int bt = (rollout && rs.act) ? rs.act[b] : b;       // trajectory
    const int Bs = (rollout && rs.B_full > 0) ? rs.B_full : B;
    // per-sample cursor mode of the training rollout (cur != null): a sample that already holds its n_lim frames emits nothing
    // and its R_t is unused (0)
    const bool done = cur && cur[b] >= n_lim;
    int n;
    float Rb = 0.f;
    if (deg) {
        n = output_length;
    } else {
        const int gov = per_sample ? b : 0;
        float sg = 0.f;
        for (int k = 0; k < K; ++k) {
            Rb += rt[(size_t)k * Bstride + b];
            sg += rt[(size_t)k * Bstride + gov];
        }
        Rb /= (float)K;
        sg /= (float)K;
        n = (int)floorf(sg);
        if (R_t) R_t[b] = done ? 0.f : Rb;
    }
    n = done ? 0 : max(1, min(n, n_cap));
    if (rollout) {
        const bool active = rs.cum[bt] < rs.n_roll;
        if (!active) n = 0;
        else {
            const int s = rs.steps[bt];
            if (s < rs.max_steps) {
                rs.ptrs->ns_out[(size_t)s * Bs + bt] = n;
                if (!deg) rs.ptrs->rts_out[(size_t)s * Bs + bt] = Rb;
            }
        }
        rs.n_cur[bt] = n;
    }
    if (n_out) n_out[b] = n;
}

// Per-sample cursor mode of the training rollout (tante_train_forward_hist), after the head: sample b emitted n_arr[b] frames
// (0 once it holds n_lim).  Records them in ns, advances its cursor and call count, and counts the samples still short of n_lim
// into *n_active (nullable).  One CTA.
__global__ void hist_advance_kernel(const int* __restrict__ n_arr, int* __restrict__ cur, int* __restrict__ ns,
                                    int* __restrict__ steps, int* __restrict__ n_active, int B, int n_lim) {
    __shared__ int cnt;
    if (threadIdx.x == 0) cnt = 0;
    __syncthreads();
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        const int n = n_arr[b];
        ns[b] = n;
        const int c = cur[b] + n;
        if (n > 0) { cur[b] = c; steps[b] += 1; }
        if (c < n_lim) atomicAdd(&cnt, 1);
    }
    __syncthreads();
    if (threadIdx.x == 0 && n_active) *n_active = cnt;
}

__global__ void advance_state_kernel(RolloutState rs, int B, cudaGraphConditionalHandle cond, int use_cond) {
    // single CTA; after the head kernel of a step over the bucket act[0 .. B).  When the step runs as the body of a
    // CUDA-graph WHILE node, the loop condition (any trajectory still short of n_roll frames) is set here, on the device,
    // and so is the bucket (SWITCH node) of the next model call.
    __shared__ int rem, cnt;
    if (threadIdx.x == 0) { rem = 0; cnt = 0; }
    const int Bf = rs.B_full > 0 ? rs.B_full : B;
    if (rs.enc_count)
        for (int i = threadIdx.x; i < Bf * rs.T; i += blockDim.x) rs.enc_map[i] = -1;
    __syncthreads();
    for (int i = threadIdx.x; i < B; i += blockDim.x) {
        const int b = rs.act ? rs.act[i] : i;
        const int n = rs.n_cur[b];
        if (n > 0) {
            rs.cum[b] += n;
            const int fc = rs.fcount[b] + n;
            rs.fcount[b] = fc;
            rs.steps[b] += 1;
            // (a trajectory that just finished is never encoded again: its frames stay off the list, which therefore
            //  never outgrows the next call's bucket)
            if (rs.enc_count && rs.cum[b] < rs.n_roll) {      // the min(n, T) newest frames of the window sit in slots (fc - 1 - j) % T
                const int m = min(n, rs.T);
                const int e0 = atomicAdd(&cnt, m);
                for (int j = 0; j < m; ++j) {
                    const int slot = (fc - 1 - j) % rs.T;
                    rs.enc_list[e0 + j] = b * rs.T + slot;
                    rs.enc_map[b * rs.T + slot] = e0 + j;
                }
            }
        }
        if (rs.cum[b] < rs.n_roll) atomicAdd(&rem, 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (rs.enc_count) *rs.enc_count = cnt;
        *rs.remaining = rem;
        const int it = *rs.iter + 1;
        *rs.iter = it;
        if (use_cond) cudaGraphSetConditional(cond, (rem > 0 && it < rs.max_steps) ? 1u : 0u);
        if (rs.act) {
            // stable partition of the bucket: running trajectories first (B is small: one thread, in place through a
            // bounded scratch walk -- finished ones are appended behind in their old order)
            int w = 0;
            for (int i = 0; i < B; ++i) {
                const int b = rs.act[i];
                if (rs.cum[b] < rs.n_roll) {
                    // rotate b down to position w, shifting the finished ones in [w, i) up by one
                    for (int j = i; j > w; --j) rs.act[j] = rs.act[j - 1];
                    rs.act[w++] = b;
                }
            }
            *rs.n_active = w;
            if (rs.n_buckets > 1 && use_cond) {
                int k = 0;
                while (k + 1 < rs.n_buckets && rs.bucket_sz[k + 1] >= w) ++k;
                cudaGraphSetConditional(rs.sw, (unsigned)k);
            }
        }
    }
}

__global__ void init_state_kernel(RolloutState rs, int B, int T) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) {
        rs.cum[b] = 0; rs.fcount[b] = T; rs.steps[b] = 0; rs.n_cur[b] = 0;
        if (rs.act) rs.act[b] = b;
        if (rs.enc_count)
            for (int t = 0; t < T; ++t) { rs.enc_list[b * T + t] = b * T + t; rs.enc_map[b * T + t] = b * T + t; }
    }
    if (b == 0) { *rs.remaining = B; *rs.iter = 0; if (rs.enc_count) *rs.enc_count = B * T; if (rs.act) *rs.n_active = B; }
}

// ------------------------------------------------------------------------------------------------
// K9: fused last transposed conv (C1 -> D, k0 x k0, all K orders) + Taylor/Horner sum + residual u0 +
// multi-frame emit.  Replaces dec_conv_3 (reference enc_dec_cnn.py:273), the Python loop
// `output += derivatives[k]*(i*fi)**k/k!` + `input[:, -1:]` + torch.cat (tante.py:165-171), the
// formatter's channels-last transpose (data/datamodule.py:191-192) and the sliding-window
// torch.cat (trainer/r_evaler.py:98) in one pass:  reads K stage-1 rows (C1 values each) + u0,
// writes n frames.  One thread per stage-1 pixel (k0 x k0 x D outputs); a CTA stages its 128 rows
// per order in shared memory with coalesced loads.
//   out_i = u0 + sum_k deriv_k * (i*fi)^k / k!   evaluated in Horner form in registers.
// ------------------------------------------------------------------------------------------------
constexpr int kMaxOrder = 8;
struct HeadParams {
    const void* z[kMaxOrder];       // stage-1 activations per order: [B*L*R1][C1]
    const float* w3[kMaxOrder];     // packed [C1][k0*k0*D]  (col = (c*k0+c')*D + d)
    const float* b3[kMaxOrder];     // [D]
    int K;
    float fi;
    const float* u_ring;            // (B,T,D,H,W) window / input
    const int* fcount;              // nullable: ring position (rollout)
    const int* n_arr;               // [B] frames to emit
    // plain forward: frames (B, n_cap, D, H, W)
    float* frames; int n_cap;
    // rollout: channels-last history (B, n_roll, H, W, D) (pointer read from `ptrs`) + ring write-back
    const RolloutPtrs* ptrs; float* ring_out; const int* cum; int n_roll;
    // optional: decoded derivative fields for debugging/tests [K][B][D][H][W]
    float* deriv_dbg;
    // rollout compaction: sample index of the stage-1 rows (compact) -> trajectory of ring / counters / history (null: identity)
    const int* act;
    // training over a frame table: u0 = last window frame of sample b at u0_base + b * u0_bs (null: u_ring); frame i of sample b is
    // written to frames + b * frames_bs + i * D * H * W (0: contiguous (B, n_cap, D, H, W))
    const float* u0_base; long long u0_bs; long long frames_bs;
    // per-sample cursor mode (tante_train_forward_hist; null: off): frames is the prediction buffer and sample b has emitted cur[b]
    // frames into it so far -- its window ends with prediction cur[b] - 1 once cur[b] > 0, and frame i goes to cur[b] + i - 1
    const int* cur;
};

// u0 (the last window frame) of sample bt
__device__ __forceinline__ const float* head_u0(const HeadParams& hp, const PatchGeom& g, int bt, int fc, size_t HW) {
    const int c = hp.cur ? hp.cur[bt] : 0;
    if (c > 0) return hp.frames + (size_t)bt * hp.frames_bs + (size_t)(c - 1) * g.D * HW;
    return hp.u0_base ? hp.u0_base + (size_t)bt * hp.u0_bs : hp.u_ring + (size_t)(bt * g.T + (fc + g.T - 1) % g.T) * g.D * HW;
}

// Exact-mode (FFMA) variant: one thread per stage-1 row; the thread streams its own C1-long row(s)
// from global/L1 (each row is one or two full 128 B lines), weights of all K orders sit in shared
// memory and are warp-broadcast.  Outputs are produced MAXO at a time to bound registers.
template <typename TIn, int MAXO, int KORD>
__global__ void __launch_bounds__(128) taylor_head_kernel(HeadParams hp, PatchGeom g, int C1, long long rows_total,
                                                          int B) {
    extern __shared__ __align__(16) float smem[];
    const int NO = g.k0 * g.k0 * g.D;
    float* sw = smem;                        // [K][C1][NO]
    float* sb = sw + KORD * C1 * NO;         // [K][D]
#pragma unroll
    for (int k = 0; k < KORD; ++k) {
        for (int i = threadIdx.x; i < C1 * NO; i += blockDim.x) sw[k * C1 * NO + i] = hp.w3[k][i];
        for (int i = threadIdx.x; i < g.D; i += blockDim.x) sb[k * g.D + i] = hp.b3[k][i];
    }
    __syncthreads();
    const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rows_total) return;

    long long tkn = row / g.R1;
    const int r = (int)(row % g.R1);
    const int wp = (int)(tkn % g.Wp); tkn /= g.Wp;
    const int hpp = (int)(tkn % g.Hp);
    const int b = (int)(tkn / g.Hp);
    int h1, w1;
    stage1_row_to_hw(g, hpp, wp, r, h1, w1);

    const int bt = hp.act ? hp.act[b] : b;
    const int n = hp.n_arr[bt];
    if (n <= 0 && !hp.deriv_dbg) return;
    const size_t HW = (size_t)g.H * g.W;
    const int fc = hp.fcount ? hp.fcount[bt] : g.T;
    const float* u0p = head_u0(hp, g, bt, fc, HW);
    const int f0 = hp.cur ? hp.cur[bt] : 0;
    const int cum = hp.cum ? hp.cum[bt] : 0;
    float* y_out = hp.ptrs ? hp.ptrs->y_out : nullptr;

    for (int o0 = 0; o0 < NO; o0 += MAXO) {
        float acc[KORD][MAXO];
#pragma unroll
        for (int k = 0; k < KORD; ++k) {
#pragma unroll
            for (int o = 0; o < MAXO; ++o) acc[k][o] = (o0 + o < NO) ? sb[k * g.D + (o0 + o) % g.D] : 0.f;
            const TIn* zr = reinterpret_cast<const TIn*>(hp.z[k]) + (size_t)row * C1;
            const float* wk = sw + k * C1 * NO + o0;
            for (int c = 0; c < C1; c += 4) {
                float z4[4];
                Vec4<TIn>::load(zr + c, z4);
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int o = 0; o < MAXO; ++o)
                        if (o0 + o < NO) acc[k][o] = fmaf(z4[j], wk[(c + j) * NO + o], acc[k][o]);
            }
        }
#pragma unroll
        for (int o = 0; o < MAXO; ++o) {
            const int oo = o0 + o;
            if (oo >= NO) break;
            const int d = oo % g.D;
            const int cp = (oo / g.D) % g.k0;
            const int c = oo / (g.D * g.k0);
            const int h = h1 * g.k0 + c, w = w1 * g.k0 + cp;
            const size_t pix = (size_t)h * g.W + w;
            if (hp.deriv_dbg)
#pragma unroll
                for (int k = 0; k < KORD; ++k) hp.deriv_dbg[(((size_t)k * B + b) * g.D + d) * HW + pix] = acc[k][o];
            if (n <= 0) continue;
            const float u0 = u0p[(size_t)d * HW + pix];
            for (int i = 1; i <= n; ++i) {
                // Horner form of sum_k d_k (i*fi)^k / k!:  dt*(d1 + dt/2*(d2 + dt/3*(d3 + ...)))
                const float dt = (float)i * hp.fi;
                float v = 0.f;
#pragma unroll
                for (int k = KORD; k >= 1; --k) v = (acc[k - 1][o] + v) * (dt / (float)k);
                const float val = v + u0;
                if (hp.frames)
                    hp.frames[(size_t)b * (hp.frames_bs ? (size_t)hp.frames_bs : (size_t)hp.n_cap * g.D * HW) + ((size_t)(f0 + i - 1) * g.D + d) * HW + pix] = val;
                if (y_out) {
                    const int fidx = cum + i - 1;
                    if (fidx < hp.n_roll) y_out[(((size_t)bt * hp.n_roll + fidx) * HW + pix) * g.D + d] = val;
                    if (i > n - g.T) {
                        const int slot = (fc + i - 1) % g.T;
                        hp.ring_out[((size_t)(bt * g.T + slot) * g.D + d) * HW + pix] = val;
                    }
                }
            }
        }
    }
}

}  // namespace tante
