// Tensor-core (mma.sync, bf16) version of the long-sequence attention backward of attention_long_bwd.cuh: same three passes
// (statistics, dQ, dK / dV), same 64 x 64 recompute tiles, same addressing -- the five 64 x 64 x 32 products of a tile pair run on
// m16n8k16 MMAs with fp32 accumulation instead of FFMA loops.  Fragment plumbing as in attention_flash.cuh: one CTA = 64 rows of one
// (sequence, head), 4 warps x 16 rows; row tiles are [64][32 bf16] with the 16-byte chunks XOR-swizzled (att_off); the streamed
// tiles are double-buffered with cp.async; probabilities / dS go from the accumulator layout straight into A fragments.
//   stats:  per query row, online over key tiles:  lse2 = log2 sum_j 2^(s_ij),  delta = sum_j P_ij dP_ij      (s in the log2 domain)
//   dQ   :  per query tile over key tiles:          dS = P o (dP - delta) * scale,   dQ += dS K
//   dK/dV:  per key tile over query tiles, on the TRANSPOSED tiles (rows = keys):  dV += P^T dO,  dK += dS^T Q
// head_dim 32, no dropout, non-causal (the composite axes L / Y / A and 65 .. 96-token axes in the tensor mode).
#pragma once
#include "attention_mma.cuh"

namespace tante {

struct AlmGeom {
    int S, inner_sz, n_head, C;
    float sl2;        // scale * log2(e)
    float scale;
};

// 64 rows x 4 chunks of 16 B from row-strided global memory (two chunks per thread); rows past the sequence are zero-filled
__device__ __forceinline__ void alm_load_tile(uint32_t dst, const __nv_bfloat16* base, size_t row_stride, int pos0, int S, int tid) {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const int i = tid + j * 128;
        const int r = i >> 2, c = i & 3;
        const int pos = pos0 + r;
        const int nbytes = pos < S ? 16 : 0;
        const __nv_bfloat16* src = base + (size_t)(nbytes ? pos : 0) * row_stride + c * 8;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst + att_off(r, c)), "l"(src), "r"(nbytes) : "memory");
    }
}

// acc[nb] (16 rows of this warp x keys nb*8 .. +7) = A (two k-steps of fragments) x tile^T, tile = [64 rows][32] read non-transposed
__device__ __forceinline__ void alm_scores(const uint32_t (&a)[2][4], uint32_t tile, int lane, float (&acc)[8][4]) {
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
        acc[nb][0] = acc[nb][1] = acc[nb][2] = acc[nb][3] = 0.f;
        uint32_t b0, b1, b2, b3;
        ldsm_x4(tile + att_off(nb * 8 + (lane & 7), lane >> 3), b0, b1, b2, b3);
        mma_bf16_16816(acc[nb], a[0], b0, b1);
        mma_bf16_16816(acc[nb], a[1], b2, b3);
    }
}

// out (16 x 32) += P (16 x 64, accumulator layout, converted to A fragments) x tile (64 rows x 32, read transposed)
__device__ __forceinline__ void alm_accum(const float (&p)[8][4], uint32_t tile, int lrow, int lchk, float (&out)[4][4]) {
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
        uint32_t pa[4];
        pa[0] = pack_bf16x2(p[2 * kk][0], p[2 * kk][1]);
        pa[1] = pack_bf16x2(p[2 * kk][2], p[2 * kk][3]);
        pa[2] = pack_bf16x2(p[2 * kk + 1][0], p[2 * kk + 1][1]);
        pa[3] = pack_bf16x2(p[2 * kk + 1][2], p[2 * kk + 1][3]);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            uint32_t v0, v1, v2, v3;
            ldsm_x4_t(tile + att_off(kk * 16 + lrow, 2 * j + lchk), v0, v1, v2, v3);
            mma_bf16_16816(out[2 * j], pa, v0, v1);
            mma_bf16_16816(out[2 * j + 1], pa, v2, v3);
        }
    }
}

__device__ __forceinline__ void alm_locate(const AlmGeom& g, int& head, size_t& tok0) {
    head = blockIdx.x % g.n_head;
    const long long seq = blockIdx.x / g.n_head;
    const long long outer = seq / g.inner_sz, inner = seq % g.inner_sz;
    tok0 = (size_t)outer * g.S * g.inner_sz + (size_t)inner;
}

// MODE 0: statistics (lse2, delta);  MODE 1: dQ.  CTA = 64 queries, K / V tiles streamed.
template <int MODE>
__global__ void __launch_bounds__(128) attn_long_q_mma_kernel(const __nv_bfloat16* __restrict__ qkv, const __nv_bfloat16* __restrict__ dout,
                                                              __nv_bfloat16* __restrict__ dqkv, float* __restrict__ lse2,
                                                              float* __restrict__ delta, AlmGeom g) {
    __shared__ __align__(128) uint8_t sQ[64 * 64];
    __shared__ __align__(128) uint8_t sO[64 * 64];
    __shared__ __align__(128) uint8_t sKV[2][2][64 * 64];      // [buffer][K | V]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int head; size_t tok0;
    alm_locate(g, head, tok0);
    const int S = g.S, C = g.C, ld = 3 * C;
    const int q0 = blockIdx.y * 64;
    const __nv_bfloat16* qb = qkv + tok0 * ld + head * 32;
    const __nv_bfloat16* ob = dout + tok0 * C + head * 32;
    const size_t rs = (size_t)g.inner_sz * ld, rso = (size_t)g.inner_sz * C;
    const uint32_t aQ = (uint32_t)__cvta_generic_to_shared(sQ), aO = (uint32_t)__cvta_generic_to_shared(sO);
    const uint32_t aKV = (uint32_t)__cvta_generic_to_shared(&sKV[0][0][0]);
    const int nkb = (S + 63) / 64;
    alm_load_tile(aQ, qb, rs, q0, S, tid);
    alm_load_tile(aO, ob, rso, q0, S, tid);
    alm_load_tile(aKV, qb + C, rs, 0, S, tid);
    alm_load_tile(aKV + 4096, qb + 2 * C, rs, 0, S, tid);
    asm volatile("cp.async.commit_group;" ::: "memory");
    const int gq = lane >> 2, t = lane & 3;
    const int lrow = (lane & 7) + 8 * ((lane >> 3) & 1), lchk = lane >> 4;
    const int r0 = q0 + warp * 16 + gq, r1 = r0 + 8;       // this thread's two query rows
    uint32_t qa[2][4], oa[2][4];
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f, a0 = 0.f, a1 = 0.f;      // MODE 0
    float ls0 = 0.f, ls1 = 0.f, de0 = 0.f, de1 = 0.f;                                    // MODE 1
    float dq[4][4];
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) dq[nb][0] = dq[nb][1] = dq[nb][2] = dq[nb][3] = 0.f;
    if (MODE == 1) {
        const size_t base = (size_t)blockIdx.x * S;
        ls0 = lse2[base + (r0 < S ? r0 : 0)]; ls1 = lse2[base + (r1 < S ? r1 : 0)];
        de0 = delta[base + (r0 < S ? r0 : 0)]; de1 = delta[base + (r1 < S ? r1 : 0)];
    }
    for (int kb = 0; kb < nkb; ++kb) {
        const uint32_t aK = aKV + (uint32_t)((kb & 1) * 8192), aV = aK + 4096;
        if (kb + 1 < nkb) {
            const uint32_t nK = aKV + (uint32_t)(((kb + 1) & 1) * 8192);
            alm_load_tile(nK, qb + C, rs, (kb + 1) * 64, S, tid);
            alm_load_tile(nK + 4096, qb + 2 * C, rs, (kb + 1) * 64, S, tid);
            asm volatile("cp.async.commit_group;" ::: "memory");
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        if (kb == 0) {
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
                ldsm_x4(aQ + att_off(warp * 16 + lrow, ks * 2 + lchk), qa[ks][0], qa[ks][1], qa[ks][2], qa[ks][3]);
                ldsm_x4(aO + att_off(warp * 16 + lrow, ks * 2 + lchk), oa[ks][0], oa[ks][1], oa[ks][2], oa[ks][3]);
            }
        }
        float s[8][4], dp[8][4];
        alm_scores(qa, aK, lane, s);
        alm_scores(oa, aV, lane, dp);
        const int kend = S - kb * 64;
        if (MODE == 0) {
            float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
            for (int nb = 0; nb < 8; ++nb)
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const bool ok = nb * 8 + 2 * t + j < kend;
                    s[nb][j] = ok ? s[nb][j] * g.sl2 : -INFINITY;
                    s[nb][2 + j] = ok ? s[nb][2 + j] * g.sl2 : -INFINITY;
                    mx0 = fmaxf(mx0, s[nb][j]);
                    mx1 = fmaxf(mx1, s[nb][2 + j]);
                }
            mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
            mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
            const float n0 = fmaxf(m0, mx0), n1 = fmaxf(m1, mx1);      // finite: every block holds at least one existing key
            const float c0 = exp2f(m0 - n0), c1 = exp2f(m1 - n1);
            m0 = n0; m1 = n1;
            float p0 = 0.f, p1 = 0.f, d0 = 0.f, d1 = 0.f;
#pragma unroll
            for (int nb = 0; nb < 8; ++nb)
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const float e0 = exp2f(s[nb][j] - n0), e1 = exp2f(s[nb][2 + j] - n1);
                    p0 += e0; p1 += e1;
                    d0 = fmaf(e0, dp[nb][j], d0);
                    d1 = fmaf(e1, dp[nb][2 + j], d1);
                }
            l0 = l0 * c0 + p0; l1 = l1 * c1 + p1;       // per-thread partial sums (the quad shares c0 / c1): reduced at the end
            a0 = a0 * c0 + d0; a1 = a1 * c1 + d1;
        } else {
#pragma unroll
            for (int nb = 0; nb < 8; ++nb)
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const bool ok = nb * 8 + 2 * t + j < kend;
                    const float p0 = ok ? exp2f(s[nb][j] * g.sl2 - ls0) : 0.f;
                    const float p1 = ok ? exp2f(s[nb][2 + j] * g.sl2 - ls1) : 0.f;
                    s[nb][j] = p0 * (dp[nb][j] - de0) * g.scale;
                    s[nb][2 + j] = p1 * (dp[nb][2 + j] - de1) * g.scale;
                }
            alm_accum(s, aK, lrow, lchk, dq);
        }
        __syncthreads();      // this buffer is refilled by the loads of the next iteration
    }
    if (MODE == 0) {
        l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
        l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
        a0 += __shfl_xor_sync(0xffffffffu, a0, 1); a0 += __shfl_xor_sync(0xffffffffu, a0, 2);
        a1 += __shfl_xor_sync(0xffffffffu, a1, 1); a1 += __shfl_xor_sync(0xffffffffu, a1, 2);
        if (t == 0) {
            const size_t base = (size_t)blockIdx.x * S;
            if (r0 < S) { lse2[base + r0] = m0 + log2f(l0); delta[base + r0] = a0 / l0; }
            if (r1 < S) { lse2[base + r1] = m1 + log2f(l1); delta[base + r1] = a1 / l1; }
        }
    } else {
#pragma unroll
        for (int nb = 0; nb < 4; ++nb) {
            const int col = head * 32 + nb * 8 + 2 * t;
            if (r0 < S) *reinterpret_cast<uint32_t*>(dqkv + (tok0 + (size_t)r0 * g.inner_sz) * ld + col) = pack_bf16x2(dq[nb][0], dq[nb][1]);
            if (r1 < S) *reinterpret_cast<uint32_t*>(dqkv + (tok0 + (size_t)r1 * g.inner_sz) * ld + col) = pack_bf16x2(dq[nb][2], dq[nb][3]);
        }
    }
}

// dK / dV: CTA = 64 keys (warp = 16 keys), Q / dO tiles and the per-query statistics streamed; everything on the transposed tiles
__global__ void __launch_bounds__(128) attn_long_kv_mma_kernel(const __nv_bfloat16* __restrict__ qkv, const __nv_bfloat16* __restrict__ dout,
                                                               __nv_bfloat16* __restrict__ dqkv, const float* __restrict__ lse2,
                                                               const float* __restrict__ delta, AlmGeom g) {
    __shared__ __align__(128) uint8_t sK[64 * 64];
    __shared__ __align__(128) uint8_t sV[64 * 64];
    __shared__ __align__(128) uint8_t sQO[2][2][64 * 64];      // [buffer][Q | dO]
    __shared__ float sSt[2][2][64];                            // [buffer][lse2 | delta][query]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int head; size_t tok0;
    alm_locate(g, head, tok0);
    const int S = g.S, C = g.C, ld = 3 * C;
    const int k0 = blockIdx.y * 64;
    const __nv_bfloat16* qb = qkv + tok0 * ld + head * 32;
    const __nv_bfloat16* ob = dout + tok0 * C + head * 32;
    const size_t rs = (size_t)g.inner_sz * ld, rso = (size_t)g.inner_sz * C;
    const uint32_t aK = (uint32_t)__cvta_generic_to_shared(sK), aV = (uint32_t)__cvta_generic_to_shared(sV);
    const uint32_t aQO = (uint32_t)__cvta_generic_to_shared(&sQO[0][0][0]);
    const size_t sbase = (size_t)blockIdx.x * S;
    const int nqb = (S + 63) / 64;
    auto stage_stats = [&](int buf, int q0) {
        const int q = q0 + (tid & 63);
        const float v = q < S ? (tid < 64 ? lse2[sbase + q] : delta[sbase + q]) : 0.f;
        sSt[buf][tid >> 6][tid & 63] = v;
    };
    alm_load_tile(aK, qb + C, rs, k0, S, tid);
    alm_load_tile(aV, qb + 2 * C, rs, k0, S, tid);
    alm_load_tile(aQO, qb, rs, 0, S, tid);
    alm_load_tile(aQO + 4096, ob, rso, 0, S, tid);
    asm volatile("cp.async.commit_group;" ::: "memory");
    stage_stats(0, 0);
    const int gq = lane >> 2, t = lane & 3;
    const int lrow = (lane & 7) + 8 * ((lane >> 3) & 1), lchk = lane >> 4;
    uint32_t ka[2][4], va[2][4];
    float dk[4][4], dv[4][4];
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) {
        dk[nb][0] = dk[nb][1] = dk[nb][2] = dk[nb][3] = 0.f;
        dv[nb][0] = dv[nb][1] = dv[nb][2] = dv[nb][3] = 0.f;
    }
    for (int qt = 0; qt < nqb; ++qt) {
        const int buf = qt & 1;
        const uint32_t aQ = aQO + (uint32_t)(buf * 8192), aO = aQ + 4096;
        if (qt + 1 < nqb) {
            const uint32_t nQ = aQO + (uint32_t)((buf ^ 1) * 8192);
            alm_load_tile(nQ, qb, rs, (qt + 1) * 64, S, tid);
            alm_load_tile(nQ + 4096, ob, rso, (qt + 1) * 64, S, tid);
            asm volatile("cp.async.commit_group;" ::: "memory");
            stage_stats(buf ^ 1, (qt + 1) * 64);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        if (qt == 0) {
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
                ldsm_x4(aK + att_off(warp * 16 + lrow, ks * 2 + lchk), ka[ks][0], ka[ks][1], ka[ks][2], ka[ks][3]);
                ldsm_x4(aV + att_off(warp * 16 + lrow, ks * 2 + lchk), va[ks][0], va[ks][1], va[ks][2], va[ks][3]);
            }
        }
        float st[8][4], dpt[8][4];      // rows = this warp's keys (gq, gq + 8), columns = the 64 queries of the tile
        alm_scores(ka, aQ, lane, st);
        alm_scores(va, aO, lane, dpt);
        const int qend = S - qt * 64;
#pragma unroll
        for (int nb = 0; nb < 8; ++nb)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int qc = nb * 8 + 2 * t + j;
                const bool ok = qc < qend;
                const float ls = sSt[buf][0][qc], de = sSt[buf][1][qc];
                const float p0 = ok ? exp2f(st[nb][j] * g.sl2 - ls) : 0.f;
                const float p1 = ok ? exp2f(st[nb][2 + j] * g.sl2 - ls) : 0.f;
                st[nb][j] = p0; st[nb][2 + j] = p1;
                dpt[nb][j] = p0 * (dpt[nb][j] - de) * g.scale;
                dpt[nb][2 + j] = p1 * (dpt[nb][2 + j] - de) * g.scale;
            }
        alm_accum(st, aO, lrow, lchk, dv);       // dV += P^T dO
        alm_accum(dpt, aQ, lrow, lchk, dk);      // dK += dS^T Q
        __syncthreads();
    }
    const int r0 = k0 + warp * 16 + gq, r1 = r0 + 8;
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) {
        const int col = head * 32 + nb * 8 + 2 * t;
        if (r0 < S) {
            __nv_bfloat16* dst = dqkv + (tok0 + (size_t)r0 * g.inner_sz) * ld + C + col;
            *reinterpret_cast<uint32_t*>(dst) = pack_bf16x2(dk[nb][0], dk[nb][1]);
            *reinterpret_cast<uint32_t*>(dst + C) = pack_bf16x2(dv[nb][0], dv[nb][1]);
        }
        if (r1 < S) {
            __nv_bfloat16* dst = dqkv + (tok0 + (size_t)r1 * g.inner_sz) * ld + C + col;
            *reinterpret_cast<uint32_t*>(dst) = pack_bf16x2(dk[nb][2], dk[nb][3]);
            *reinterpret_cast<uint32_t*>(dst + C) = pack_bf16x2(dv[nb][2], dv[nb][3]);
        }
    }
}

// Host launcher: bf16, head_dim 32, no dropout, non-causal.  stats: 2 * n_seq * n_head * S floats.  Returns false otherwise.
static bool launch_attention_long_bwd_mma(const __nv_bfloat16* qkv, const __nv_bfloat16* dout, __nv_bfloat16* dqkv, float* stats,
                                          long long n_seq, int S, int inner_sz, int n_head, int C, int head_dim, int causal,
                                          cudaStream_t st, cudaError_t* err) {
    const long long gx = n_seq * n_head;
    const int tiles = (S + 63) / 64;
    if (head_dim != 32 || causal || gx > 0x7fffffffLL || tiles > 65535) return false;
    AlmGeom g{S, inner_sz, n_head, C, (1.0f / sqrtf((float)head_dim)) * 1.4426950408889634f, 1.0f / sqrtf((float)head_dim)};
    float* lse2 = stats;
    float* delta = stats + (size_t)gx * S;
    const dim3 grid((unsigned)gx, (unsigned)tiles);
    attn_long_q_mma_kernel<0><<<grid, 128, 0, st>>>(qkv, dout, dqkv, lse2, delta, g);
    attn_long_q_mma_kernel<1><<<grid, 128, 0, st>>>(qkv, dout, dqkv, lse2, delta, g);
    attn_long_kv_mma_kernel<<<grid, 128, 0, st>>>(qkv, dout, dqkv, lse2, delta, g);
    *err = cudaGetLastError();
    return true;
}

}  // namespace tante
