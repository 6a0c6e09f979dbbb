// Residual axis MLP ("propagator") on tensor cores for the bf16 mode:
//   x += W2 * gelu_erf(W1 * x_axis + b1) + b2   along one axis of length S <= 64, in place on the fp32 latent
// (reference attn_backbone.py:111-119,140-146; under autocast the reference also runs these Linears in bf16).
// Element (outer, p, col) lives at (outer*S + p)*IC + col.  One tile = one `outer` x 128 columns, 4 warps x 32
// columns; CTAs are persistent over tiles (column blocks fastest) so that the S x S weight matrices are fetched and
// converted once per CTA, not once per 128-column slab (at S = 64 that prologue cost as much as the slab itself).
// Both weight matrices (bf16, padded to 16) are the A operands, the S x 128 slab is the B
// operand via ldmatrix.trans; the hidden tile never leaves shared memory.  HBM traffic: read x + write x.
#pragma once
#include "attention_mma.cuh"

namespace tante {

// slab tile: row pitch 256 B (128 bf16), 16-byte chunk index XOR-swizzled with the row inside groups of 8
__device__ __forceinline__ uint32_t slab_off(int r, int chunk) { return (uint32_t)(r * 256 + (((chunk & 8) | ((chunk ^ r) & 7)) << 4)); }

template <int MB /* S_pad / 16 */>
__global__ void __launch_bounds__(128, 3) propagator_mma_kernel(const float* xin, float* x, int S, long long IC, long long n_outer,
                                                             const float* __restrict__ W1, const float* __restrict__ b1,
                                                             const float* __restrict__ W2, const float* __restrict__ b2) {
    constexpr int SP = MB * 16;
    constexpr int THREADS = 128;
    constexpr int WPITCH = SP * 2 + 16;                       // bytes; odd number of 16-B chunks -> conflict-free ldmatrix
    extern __shared__ __align__(128) uint8_t pm_smem[];
    uint8_t* sV = pm_smem;
    uint8_t* sH = sV + SP * 256;
    uint8_t* sW1 = sH + SP * 256;
    uint8_t* sW2 = sW1 + SP * WPITCH;
    float* sb1 = reinterpret_cast<float*>(sW2 + SP * WPITCH);
    float* sb2 = sb1 + SP;

    const int tid = threadIdx.x, lane = tid % 32;
    const int warp = tid / 32;                                // column group: 32 of the tile's 128 columns
    const long long ncb = (IC + 127) / 128;

    for (int i = tid; i < SP * SP; i += THREADS) {
        const int j = i / SP, k = i % SP;
        const bool ok = j < S && k < S;
        *reinterpret_cast<__nv_bfloat16*>(sW1 + j * WPITCH + k * 2) = __float2bfloat16_rn(ok ? W1[j * S + k] : 0.f);
        *reinterpret_cast<__nv_bfloat16*>(sW2 + j * WPITCH + k * 2) = __float2bfloat16_rn(ok ? W2[j * S + k] : 0.f);
    }
    for (int i = tid; i < SP; i += THREADS) { sb1[i] = i < S ? b1[i] : 0.f; sb2[i] = i < S ? b2[i] : 0.f; }

    const uint32_t aV = (uint32_t)__cvta_generic_to_shared(sV), aH = (uint32_t)__cvta_generic_to_shared(sH);
    const uint32_t aW1 = (uint32_t)__cvta_generic_to_shared(sW1), aW2 = (uint32_t)__cvta_generic_to_shared(sW2);
    const int g = lane >> 2, t = lane & 3;
    const int lrow = (lane & 7) + 8 * ((lane >> 3) & 1);
    const int lchk = lane >> 4;

  for (long long tile = blockIdx.x; tile < n_outer * ncb; tile += gridDim.x) {
    // persistent (S <= 32): column blocks fastest; one tile per CTA (S > 32, see the launcher): `outer` fastest, as measured best
    const bool one_each = (long long)gridDim.x >= n_outer * ncb;
    const long long outer = one_each ? tile % n_outer : tile / ncb;
    const long long col0 = (one_each ? tile / n_outer : tile % ncb) * 128;
    float* base = x + (size_t)outer * S * IC + col0;
    const float* ibase = xin + (size_t)outer * S * IC + col0;    // xin == x: in place; else out of place (training)
    const int ncol = (int)min((long long)128, IC - col0);     // multiple of 4
    __syncthreads();      // the previous tile's slab has been consumed (and, first pass, the weights are in place)
#pragma unroll 4
    for (int i = tid; i < SP * 32; i += THREADS) {
        const int p = i / 32, c4 = (i % 32) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p < S && c4 < ncol) v = *reinterpret_cast<const float4*>(ibase + (size_t)p * IC + c4);
        uint2 pk;
        pk.x = pack_bf16x2(v.x, v.y);
        pk.y = pack_bf16x2(v.z, v.w);
        *reinterpret_cast<uint2*>(sV + slab_off(p, c4 / 8) + (c4 % 8) * 2) = pk;
    }
    __syncthreads();

    for (int pass = 0; pass < 2; ++pass) {
        const uint32_t aW = pass == 0 ? aW1 : aW2;
        const uint32_t aB = pass == 0 ? aV : aH;
        float acc[MB][4][4];
#pragma unroll
        for (int mb = 0; mb < MB; ++mb)
#pragma unroll
            for (int nb = 0; nb < 4; ++nb) acc[mb][nb][0] = acc[mb][nb][1] = acc[mb][nb][2] = acc[mb][nb][3] = 0.f;
#pragma unroll
        for (int kk = 0; kk < MB; ++kk) {
            uint32_t bf[4][2];
#pragma unroll
            for (int j = 0; j < 2; ++j)      // B fragments of this warp's 4 n-blocks (32 columns) for k-rows kk*16..+15
                ldsm_x4_t(aB + slab_off(kk * 16 + lrow, warp * 4 + 2 * j + lchk), bf[2 * j][0], bf[2 * j][1], bf[2 * j + 1][0],
                          bf[2 * j + 1][1]);
#pragma unroll
            for (int mb = 0; mb < MB; ++mb) {
                uint32_t af[4];
                ldsm_x4(aW + (uint32_t)((mb * 16 + lrow) * WPITCH + (kk * 2 + lchk) * 16), af[0], af[1], af[2], af[3]);
#pragma unroll
                for (int nb = 0; nb < 4; ++nb) mma_bf16_16816(acc[mb][nb], af, bf[nb][0], bf[nb][1]);
            }
        }
        if (pass == 0) {
#pragma unroll
            for (int mb = 0; mb < MB; ++mb) {
                const int j0 = mb * 16 + g, j1 = j0 + 8;
                const float bb0 = sb1[j0], bb1 = sb1[j1];
#pragma unroll
                for (int nb = 0; nb < 4; ++nb) {
                    const int chunk = warp * 4 + nb;
                    *reinterpret_cast<uint32_t*>(sH + slab_off(j0, chunk) + t * 4) =
                        pack_bf16x2(gelu_erf_fast(acc[mb][nb][0] + bb0), gelu_erf_fast(acc[mb][nb][1] + bb0));
                    *reinterpret_cast<uint32_t*>(sH + slab_off(j1, chunk) + t * 4) =
                        pack_bf16x2(gelu_erf_fast(acc[mb][nb][2] + bb1), gelu_erf_fast(acc[mb][nb][3] + bb1));
                }
            }
            __syncwarp();     // the hidden columns of a warp are consumed only by the same warp
        } else {
            // residual add in two sweeps: all loads first (x may alias the output, so a load cannot be hoisted over
            // an earlier store and an interleaved loop would serialise 8*MB L2 round trips per thread)
#pragma unroll
            for (int mb = 0; mb < MB; ++mb) {
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    const int p = mb * 16 + g + 8 * hh;
                    const float bb = p < S ? sb2[p] : 0.f;
#pragma unroll
                    for (int nb = 0; nb < 4; ++nb) {
                        const int c = warp * 32 + nb * 8 + 2 * t;
                        if (p < S && c < ncol) {
                            const float2 xv = *reinterpret_cast<const float2*>(ibase + (size_t)p * IC + c);
                            acc[mb][nb][2 * hh + 0] += xv.x + bb;
                            acc[mb][nb][2 * hh + 1] += xv.y + bb;
                        }
                    }
                }
            }
#pragma unroll
            for (int mb = 0; mb < MB; ++mb) {
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    const int p = mb * 16 + g + 8 * hh;
#pragma unroll
                    for (int nb = 0; nb < 4; ++nb) {
                        const int c = warp * 32 + nb * 8 + 2 * t;
                        if (p < S && c < ncol)
                            *reinterpret_cast<float2*>(base + (size_t)p * IC + c) = make_float2(acc[mb][nb][2 * hh], acc[mb][nb][2 * hh + 1]);
                    }
                }
            }
        }
    }
  }
}

static void prop_set_attrs() {
    static unsigned long long done = 0;
    if (!attrs_needed(done)) return;
    cudaFuncSetAttribute(propagator_mma_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
}

static bool launch_propagator_mma(const float* xin, float* x, int S, long long IC, long long outer, const float* W1, const float* b1,
                                  const float* W2, const float* b2, cudaStream_t st, cudaError_t* err, int num_sms = 148) {
    if (S < 1 || S > 64 || outer > 0x7fffffffLL) return false;
    const int MB = (S + 15) / 16;
    const int SP = MB * 16;
    const size_t smem = (size_t)2 * SP * 256 + (size_t)2 * SP * (SP * 2 + 16) + 2 * SP * sizeof(float);
    // persistent CTAs: as many as are resident (shared memory / 16 CTAs per SM), each walks over its share of the tiles
    const long long tiles = outer * ((IC + 127) / 128);
    prop_set_attrs();
    int per_sm = 1;      // registers, not shared memory, limit the S = 64 variant (189 registers: two CTAs per SM)
    {
        cudaError_t oe = cudaSuccess;
        switch (MB) {
            case 1: oe = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, propagator_mma_kernel<1>, 128, smem); break;
            case 2: oe = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, propagator_mma_kernel<2>, 128, smem); break;
            case 3: oe = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, propagator_mma_kernel<3>, 128, smem); break;
            default: oe = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, propagator_mma_kernel<4>, 128, smem); break;
        }
        if (oe != cudaSuccess || per_sm < 1) { (void)cudaGetLastError(); per_sm = 1; }
    }
    // S > 32 (189 registers, two CTAs of four warps per SM): a persistent CTA serialises load / pass 1 / pass 2 with nothing to
    // overlap them -- measured 282 us vs 243 us for one tile per CTA at S = 64 -- so only the short-axis variants are persistent
    if (MB >= 3 && tiles > 0x7fffffffLL) return false;
    dim3 grid((unsigned)(MB >= 3 ? tiles : std::min<long long>(tiles, (long long)num_sms * per_sm)));
    switch (MB) {
        case 1: propagator_mma_kernel<1><<<grid, 128, smem, st>>>(xin, x, S, IC, outer, W1, b1, W2, b2); break;
        case 2: propagator_mma_kernel<2><<<grid, 128, smem, st>>>(xin, x, S, IC, outer, W1, b1, W2, b2); break;
        case 3: propagator_mma_kernel<3><<<grid, 128, smem, st>>>(xin, x, S, IC, outer, W1, b1, W2, b2); break;
        default: propagator_mma_kernel<4><<<grid, 128, smem, st>>>(xin, x, S, IC, outer, W1, b1, W2, b2); break;
    }
    *err = cudaGetLastError();
    return true;
}

}  // namespace tante
