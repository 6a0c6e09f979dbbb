// Tiled ("flash") attention on mma.sync for sequences LONGER than 64 tokens: the composite axes L = (h w), Y = (t h),
// A = (t h w) of Attn_Backbone (reference models/attn_backbone.py:164-182) and plain axes of 65 .. 96 tokens.  Same
// addressing as the short-sequence kernel -- token(pos) = (outer * S + pos) * inner_sz + inner, packed qkv rows of 3C --
// but the keys stream through shared memory in blocks of 64 with an online softmax, so the work per query is O(S) loads of
// K / V tiles shared by 64 queries instead of the O(S) uncoalesced global rows PER QUERY of the general one-thread-per-query
// kernel (which stays the exact-mode / odd-head-dim path).  One CTA = 64 queries of one (sequence, head); 4 warps x 16 rows.
// K / V blocks are double-buffered with cp.async.  head_dim = 32, non-causal (no composite axis is causal), bf16, no dropout
// (these axes are inference-only).
#pragma once
#include "attention_mma.cuh"

namespace tante {

__global__ void __launch_bounds__(128) attention_flash_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ out,
                                                              int S, int inner_sz, int n_head, int C, float scale_log2e) {
    __shared__ __align__(128) uint8_t sQ[64 * 64];
    __shared__ __align__(128) uint8_t sKV[2][2][64 * 64];      // [buffer][K | V][64 keys x 64 B]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int qb = blockIdx.y;
    const int head = blockIdx.x % n_head;
    const long long seq = blockIdx.x / n_head;
    const long long outer = seq / inner_sz, inner = seq % inner_sz;
    const size_t tok0 = (size_t)outer * S * inner_sz + (size_t)inner;
    const int ld = 3 * C;
    const uint32_t aQ = (uint32_t)__cvta_generic_to_shared(sQ);
    const uint32_t aKV = (uint32_t)__cvta_generic_to_shared(&sKV[0][0][0]);

    // 64 rows x 4 chunks of 16 B per tile: two chunks per thread; rows past the sequence are zero-filled
    auto load_tile = [&](uint32_t dst, int pos0, int col) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int i = tid + j * 128;
            const int r = i >> 2, c = i & 3;
            const int pos = pos0 + r;
            const int nbytes = pos < S ? 16 : 0;
            const __nv_bfloat16* src = qkv + (tok0 + (size_t)(nbytes ? pos : 0) * inner_sz) * ld + col + head * 32 + c * 8;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst + att_off(r, c)), "l"(src), "r"(nbytes) : "memory");
        }
    };
    const int nkb = (S + 63) / 64;
    load_tile(aQ, qb * 64, 0);
    load_tile(aKV, 0, C);
    load_tile(aKV + 4096, 0, 2 * C);
    asm volatile("cp.async.commit_group;" ::: "memory");

    const int g = lane >> 2, t = lane & 3;
    const int lrow = (lane & 7) + 8 * ((lane >> 3) & 1), lchk = lane >> 4;
    uint32_t qa[2][4];
    float o[4][4];
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) o[nb][0] = o[nb][1] = o[nb][2] = o[nb][3] = 0.f;
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;

    for (int kb = 0; kb < nkb; ++kb) {
        const uint32_t aK = aKV + (uint32_t)((kb & 1) * 8192), aV = aK + 4096;
        if (kb + 1 < nkb) {      // next K / V block into the other buffer (consumed two iterations ago)
            const uint32_t nK = aKV + (uint32_t)(((kb + 1) & 1) * 8192);
            load_tile(nK, (kb + 1) * 64, C);
            load_tile(nK + 4096, (kb + 1) * 64, 2 * C);
            asm volatile("cp.async.commit_group;" ::: "memory");
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        if (kb == 0) {
#pragma unroll
            for (int ks = 0; ks < 2; ++ks)
                ldsm_x4(aQ + att_off(warp * 16 + lrow, ks * 2 + lchk), qa[ks][0], qa[ks][1], qa[ks][2], qa[ks][3]);
        }
        // ---- scores of this warp's 16 queries against the block's 64 keys ----
        float s[8][4];
#pragma unroll
        for (int nb = 0; nb < 8; ++nb) {
            s[nb][0] = s[nb][1] = s[nb][2] = s[nb][3] = 0.f;
            uint32_t k0, k1, k2, k3;
            ldsm_x4(aK + att_off(nb * 8 + (lane & 7), lane >> 3), k0, k1, k2, k3);
            mma_bf16_16816(s[nb], qa[0], k0, k1);
            mma_bf16_16816(s[nb], qa[1], k2, k3);
        }
        const int kend = S - kb * 64;      // keys of this block that exist
        float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
        for (int nb = 0; nb < 8; ++nb) {
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const bool ok = nb * 8 + 2 * t + j < kend;
                s[nb][j] = ok ? s[nb][j] * scale_log2e : -INFINITY;
                s[nb][2 + j] = ok ? s[nb][2 + j] * scale_log2e : -INFINITY;
                mx0 = fmaxf(mx0, s[nb][j]);
                mx1 = fmaxf(mx1, s[nb][2 + j]);
            }
        }
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
        const float n0 = fmaxf(m0, mx0), n1 = fmaxf(m1, mx1);       // finite: every block holds at least one existing key
        const float c0 = exp2f(m0 - n0), c1 = exp2f(m1 - n1);       // exp2(-inf) = 0 on the first block
        m0 = n0; m1 = n1;
        float r0 = 0.f, r1 = 0.f;
#pragma unroll
        for (int nb = 0; nb < 8; ++nb) {
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                s[nb][j] = exp2f(s[nb][j] - n0); r0 += s[nb][j];
                s[nb][2 + j] = exp2f(s[nb][2 + j] - n1); r1 += s[nb][2 + j];
            }
        }
        l0 = l0 * c0 + r0; l1 = l1 * c1 + r1;       // per-thread partial row sums (reduced across the quad at the end)
#pragma unroll
        for (int nb = 0; nb < 4; ++nb) { o[nb][0] *= c0; o[nb][1] *= c0; o[nb][2] *= c1; o[nb][3] *= c1; }
        // ---- O += P V: the probabilities are already in A-fragment layout ----
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            uint32_t pa[4];
            pa[0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
            pa[1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
            pa[2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
            pa[3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                uint32_t v0, v1, v2, v3;
                ldsm_x4_t(aV + att_off(kk * 16 + lrow, 2 * j + lchk), v0, v1, v2, v3);
                mma_bf16_16816(o[2 * j], pa, v0, v1);
                mma_bf16_16816(o[2 * j + 1], pa, v2, v3);
            }
        }
        __syncthreads();      // this buffer is refilled by the loads of the next iteration
    }
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float i0 = l0 > 0.f ? 1.0f / l0 : 0.f, i1 = l1 > 0.f ? 1.0f / l1 : 0.f;
    const int p0 = qb * 64 + warp * 16 + g, p1 = p0 + 8;
#pragma unroll
    for (int nb = 0; nb < 4; ++nb) {
        const int col = head * 32 + nb * 8 + 2 * t;
        if (p0 < S) *reinterpret_cast<uint32_t*>(out + (tok0 + (size_t)p0 * inner_sz) * C + col) = pack_bf16x2(o[nb][0] * i0, o[nb][1] * i0);
        if (p1 < S) *reinterpret_cast<uint32_t*>(out + (tok0 + (size_t)p1 * inner_sz) * C + col) = pack_bf16x2(o[nb][2] * i1, o[nb][3] * i1);
    }
}

// Host launcher: sequences longer than 64 tokens, head_dim 32, no dropout.  Returns false otherwise (caller falls back).
static bool launch_attention_flash(const __nv_bfloat16* qkv, __nv_bfloat16* out, long long n_seq, int S, int inner_sz, int n_head,
                                   int C, int head_dim, int causal, cudaStream_t st, cudaError_t* err) {
    if (head_dim != 32 || S <= 64 || causal || n_seq * n_head > 0x7fffffffLL || (S + 63) / 64 > 65535) return false;
    dim3 grid((unsigned)(n_seq * n_head), (unsigned)((S + 63) / 64));
    const float sl2 = (1.0f / sqrtf((float)head_dim)) * 1.4426950408889634f;
    attention_flash_kernel<<<grid, 128, 0, st>>>(qkv, out, S, inner_sz, n_head, C, sl2);
    *err = cudaGetLastError();
    return true;
}

}  // namespace tante
