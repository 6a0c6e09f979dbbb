// Input-gradient chain of a transformer block's MLP on tcgen05, one kernel (backward of reference models/attn_backbone.py:83,
// `x + dropout(mlp(ln2(x)))`, mlp = Linear -> GELU(tanh) -> Linear):
//
//     dpre = (dy * W2) o gelu_tanh'(hpre)          (input gradient of the second Linear, times the activation derivative)
//     dln  = dpre * W1                             (input gradient of the first Linear = dY of the LayerNorm backward)
//
// The un-fused path is a GEMM, an elementwise pass and a GEMM (3.5 KB per token through HBM: dy 0.5 | dh 0.5 out, 0.5 + hpre 0.5
// in, dpre 0.5 out | dpre 0.5 in, dln 0.5 out); here dh never exists and dpre is stored once, for the weight gradient of the
// first Linear: dy 0.5 + hpre 0.5 in, dpre 0.5 + dln 0.5 out = 2 KB.  Same skeleton as block_tail_tc.cuh: persistent CTAs
// (pairs: cta_group::2, each CTA streams its half of every weight stage), one 64 KB A tile rewritten in place between the two
// GEMM phases, the [K][N] weight copies streamed from L2 through a ring, 16 epilogue warps (thread = token row, one 64-column
// k-block each).  No fp32 traffic, no row statistics.
// Warp roles: 0 = TMA producer, 1 = MMA issuer + TMEM owner (pair peer: forwards its epilogue's arrivals), 2..17 = epilogue.
#pragma once
#include "block_tail_tc.cuh"

namespace tante {

constexpr size_t kMbSmem = 1024 + 4 * kBtKBlk + kBtWStages * kBtWStage + kBtEpiWarps * kBtEbuf + 512;

template <int NCTA>
__global__ void __launch_bounds__(kBtThreads, 1)
mlp_bwd_kernel(const __grid_constant__ CUtensorMap tmDy, const __grid_constant__ CUtensorMap tmW2T,
               const __grid_constant__ CUtensorMap tmW1T, const __grid_constant__ CUtensorMap tmHpre,
               const __grid_constant__ CUtensorMap tmDpre, const __grid_constant__ CUtensorMap tmDln, int M) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* sA = smem;                                        // [4 k-blocks][128 rows][128 B]
    uint8_t* sW = sA + 4 * kBtKBlk;                            // [kBtWStages][128 rows][128 B]
    uint8_t* sE = sW + kBtWStages * kBtWStage;                 // [16 warps][4 KB]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sE + kBtEpiWarps * kBtEbuf);
    uint64_t* w_full = bars;                       // [kBtWStages]
    uint64_t* w_empty = bars + kBtWStages;         // [kBtWStages]
    uint64_t* a_full = bars + 2 * kBtWStages;      // dy tile landed
    uint64_t* a_empty = a_full + 1;                // the second GEMM has read the A tile and the dpre stores have left it
    uint64_t* a_ready = a_full + 2;                // the epilogue warps rewrote the A tile (dpre)
    uint64_t* acc_full = a_full + 3;               // one MMA phase finished
    uint64_t* acc_free = a_full + 4;               // the second epilogue has read the accumulator
    uint64_t* hbar = a_full + 5;                   // [16 warps] hpre tile landed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(hbar + kBtEpiWarps);

    pdl_trigger();
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const int crank = NCTA == 2 ? (int)ptx::cluster_ctarank() : 0;
    const int cid = blockIdx.x / NCTA;
    const int ncl = gridDim.x / NCTA;
    const int tiles = (M + 128 * NCTA - 1) / (128 * NCTA);

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmDy); ptx::prefetch_tmap(&tmW2T); ptx::prefetch_tmap(&tmW1T);
        ptx::prefetch_tmap(&tmHpre); ptx::prefetch_tmap(&tmDpre); ptx::prefetch_tmap(&tmDln);
        for (int s = 0; s < kBtWStages; ++s) { ptx::mbar_init(&w_full[s], 1); ptx::mbar_init(&w_empty[s], 1); }
        ptx::mbar_init(a_full, 1);
        ptx::mbar_init(a_empty, 1 + kBtEpiWarps);
        ptx::mbar_init(a_ready, kBtEpiWarps + ((NCTA == 2 && crank == 0) ? 1 : 0));
        ptx::mbar_init(acc_full, 1);
        ptx::mbar_init(acc_free, kBtEpiWarps + ((NCTA == 2 && crank == 0) ? 1 : 0));
        for (int i = 0; i < kBtEpiWarps; ++i) ptx::mbar_init(&hbar[i], 1);
        ptx::fence_barrier_init();
    }
    if (warp == 1) {
        if (NCTA == 2) { ptx::tmem_alloc_pair(tmem_slot, 256); ptx::tmem_relinquish_pair(); }
        else { ptx::tmem_alloc(tmem_slot, 256); ptx::tmem_relinquish(); }
    }
    ptx::tc_fence_before();
    if (NCTA == 2) ptx::cluster_sync_all();
    else __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();

    if (warp == 0) {
        // ===== TMA producer: the tile's dy rows, then its 2 x 4 (pairs) / 2 x 8 weight stages =====
        if (lane == 0) {
            int ws = 0;
            uint32_t wph = 0;
            int it = 0;
            for (int tile = cid; tile < tiles; tile += ncl, ++it) {
                ptx::mbar_wait(a_empty, (uint32_t)(it & 1) ^ 1u);
                if (NCTA == 2) {
                    if (crank == 0) ptx::mbar_arrive_expect_tx(a_full, 2 * 4 * kBtKBlk);
                    for (int kb = 0; kb < 4; ++kb)
                        ptx::tma_load_2d_pair(sA + kb * kBtKBlk, &tmDy, a_full, kb * 64, (tile * 2 + crank) * 128);
                } else {
                    ptx::mbar_arrive_expect_tx(a_full, 4 * kBtKBlk);
                    for (int kb = 0; kb < 4; ++kb) ptx::tma_load_2d(sA + kb * kBtKBlk, &tmDy, a_full, kb * 64, tile * 128);
                }
                for (int ph = 0; ph < 2; ++ph) {
                    const CUtensorMap* wm = ph == 0 ? &tmW2T : &tmW1T;
                    for (int kb = 0; kb < 4; ++kb) {
                        for (int nh = 0; nh < 2 / NCTA; ++nh) {
                            ptx::mbar_wait(&w_empty[ws], wph ^ 1u);
                            if (NCTA == 2) {
                                if (crank == 0) ptx::mbar_arrive_expect_tx(&w_full[ws], 2 * kBtWStage);
                                ptx::tma_load_2d_pair(sW + ws * kBtWStage, wm, &w_full[ws], kb * 64, crank * 128);
                            } else {
                                ptx::mbar_arrive_expect_tx(&w_full[ws], kBtWStage);
                                ptx::tma_load_2d(sW + ws * kBtWStage, wm, &w_full[ws], kb * 64, nh * 128);
                            }
                            if (++ws == kBtWStages) { ws = 0; wph ^= 1u; }
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc = NCTA == 2 ? ptx::umma_idesc_bf16(256, 256) : ptx::umma_idesc_bf16(128, 128);
        int ws = 0;
        uint32_t wph = 0;
        int it = 0;
        if (NCTA == 2 && crank == 1) {
            // the peer's otherwise idle warp forwards "A tile rewritten" and "accumulator free" to the leader
            for (int tile = cid; tile < tiles; tile += ncl, ++it) {
                ptx::mbar_wait(a_ready, (uint32_t)(it & 1));
                if (lane == 0) ptx::mbar_arrive_leader(a_ready);
                __syncwarp();
                ptx::mbar_wait(acc_free, (uint32_t)(it & 1));
                if (lane == 0) ptx::mbar_arrive_leader(acc_free);
                __syncwarp();
            }
        }
        for (int tile = cid; tile < tiles && crank == 0; tile += ncl, ++it) {
            for (int ph = 0; ph < 2; ++ph) {
                if (ph == 0) {
                    ptx::mbar_wait(acc_free, (uint32_t)(it & 1) ^ 1u);
                    ptx::mbar_wait(a_full, (uint32_t)(it & 1));
                } else {
                    ptx::mbar_wait(a_ready, (uint32_t)(it & 1));
                }
                ptx::tc_fence_after();
                for (int kb = 0; kb < 4; ++kb) {
                    for (int nh = 0; nh < 2 / NCTA; ++nh) {
                        ptx::mbar_wait(&w_full[ws], wph);
                        ptx::tc_fence_after();
                        if (lane == 0) {
                            const uint64_t da = ptx::umma_desc_k_sw128(ptx::smem_u32(sA + kb * kBtKBlk));
                            const uint64_t db = ptx::umma_desc_k_sw128(ptx::smem_u32(sW + ws * kBtWStage));
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                if (NCTA == 2) ptx::umma_bf16_pair(tmem_base, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) != 0);
                                else ptx::umma_bf16(tmem_base + (uint32_t)(nh * 128), da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc,
                                                    (kb | k) != 0);
                            }
                            if (NCTA == 2) ptx::umma_commit_pair(&w_empty[ws]); else ptx::umma_commit(&w_empty[ws]);
                        }
                        __syncwarp();
                        if (++ws == kBtWStages) { ws = 0; wph ^= 1u; }
                    }
                }
                if (lane == 0) {
                    if (NCTA == 2) {
                        ptx::umma_commit_pair(acc_full);
                        if (ph == 1) ptx::umma_commit_pair(a_empty);
                    } else {
                        ptx::umma_commit(acc_full);
                        if (ph == 1) ptx::umma_commit(a_empty);
                    }
                }
                __syncwarp();
            }
        }
    } else {
        // ===== 16 epilogue warps: TMEM lane quarter q (thread = token row), k-block cs (64 columns) =====
        const int ew = warp - 2;
        const int q = warp & 3;
        const int cs = ew >> 2;
        uint8_t* ebuf = sE + (size_t)ew * kBtEbuf;
        uint8_t* aown = sA + (size_t)cs * kBtKBlk + (size_t)q * 32 * 128;    // this warp's 32 rows of k-block cs inside the A tile
        uint64_t* hb = hbar + ew;
        const uint32_t tm = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(cs * 64);
        uint32_t af = 0, hph = 0;
        for (int tile = cid; tile < tiles; tile += ncl) {
            const int row0 = (tile * NCTA + crank) * 128 + q * 32;
            // the saved pre-activation tile of this warp: in flight while the first GEMM runs (the previous tile's dln store
            // has left the staging buffer: waited for below)
            if (lane == 0) {
                ptx::mbar_arrive_expect_tx(hb, kBtEbuf);
                ptx::tma_load_2d(ebuf, &tmHpre, hb, cs * 64, row0);
            }
            // ---------------- phase A: dpre = acc o gelu_tanh'(hpre) -> A tile (+ stored for the weight gradient) ----------------
            ptx::mbar_wait(acc_full, af & 1u); ++af;
            ptx::tc_fence_after();
            ptx::mbar_wait(hb, hph & 1u); ++hph;
#pragma unroll 1
            for (int hh = 0; hh < 2; ++hh) {
                uint32_t r0[32];
                ptx::tmem_ld_32x32(tm + (uint32_t)(hh * 32), r0);
                ptx::tc_wait_ld();
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const uint4 pre4 = *reinterpret_cast<const uint4*>(ebuf + sw128_off(lane, hh * 4 + c));
                    const uint32_t pw[4] = {pre4.x, pre4.y, pre4.z, pre4.w};
                    uint32_t pk[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int col = c * 8 + j * 2;
                        const float2 pv = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&pw[j]));
                        const float a = __uint_as_float(r0[col]) * gelu_tanh_grad_fast(pv.x);
                        const float b = __uint_as_float(r0[col + 1]) * gelu_tanh_grad_fast(pv.y);
                        __nv_bfloat162 h2 = __floats2bfloat162_rn(a, b);
                        pk[j] = *reinterpret_cast<uint32_t*>(&h2);
                    }
                    *reinterpret_cast<uint4*>(aown + sw128_off(lane, hh * 4 + c)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                }
            }
            ptx::fence_proxy_async();
            __syncwarp();
            if (lane == 0) { ptx::tma_store_2d(&tmDpre, aown, cs * 64, row0); ptx::bulk_commit(); }
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(a_ready);

            // ---------------- phase B: dln = acc -> bf16 ----------------
            ptx::mbar_wait(acc_full, af & 1u); ++af;
            ptx::tc_fence_after();
            if (lane == 0) {      // the dpre store left the A tile long ago: the producer may fetch the next tile's dy rows now
                ptx::bulk_wait_read<0>();
                ptx::mbar_arrive(a_empty);
            }
            __syncwarp();
#pragma unroll 1
            for (int hh = 0; hh < 2; ++hh) {
                uint32_t r0[32];
                ptx::tmem_ld_32x32(tm + (uint32_t)(hh * 32), r0);
                ptx::tc_wait_ld();
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    uint32_t pk[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int col = c * 8 + j * 2;
                        __nv_bfloat162 h2 = __floats2bfloat162_rn(__uint_as_float(r0[col]), __uint_as_float(r0[col + 1]));
                        pk[j] = *reinterpret_cast<uint32_t*>(&h2);
                    }
                    *reinterpret_cast<uint4*>(ebuf + sw128_off(lane, hh * 4 + c)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                }
            }
            ptx::tc_fence_before();
            ptx::fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                ptx::mbar_arrive(acc_free);                       // the next tile's first GEMM may overwrite the accumulator
                ptx::tma_store_2d(&tmDln, ebuf, cs * 64, row0);
                ptx::bulk_commit();
                ptx::bulk_wait_read<0>();                         // dln has left the staging buffer (the next hpre tile lands there)
            }
            __syncwarp();
        }
        if (lane == 0) ptx::bulk_wait_all<0>();
    }
    ptx::tc_fence_before();
    if (NCTA == 2) ptx::cluster_sync_all();
    else __syncthreads();
    if (warp == 1) { if (NCTA == 2) ptx::tmem_dealloc_pair(tmem_base, 256); else ptx::tmem_dealloc(tmem_base, 256); }
}

static cudaError_t mb_set_attrs() {
    static unsigned long long done = 0;
    if (!get_encode_tiled()) return cudaErrorNotSupported;
    if (!attrs_needed(done)) return cudaSuccess;
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(mlp_bwd_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMbSmem)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(mlp_bwd_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMbSmem)) != cudaSuccess) return e;
    return cudaSuccess;
}

// dy, hpre, dpre, dln: bf16 [M][256]; W2T, W1T: bf16 [256][256] = the [K][N] copies of the two Linear weights (what gemm_dx uses)
static cudaError_t launch_mlp_bwd(const __nv_bfloat16* dy, const __nv_bfloat16* W2T, const __nv_bfloat16* W1T,
                                  const __nv_bfloat16* hpre, __nv_bfloat16* dpre, __nv_bfloat16* dln, int M, int num_sms,
                                  cudaStream_t st) {
    if (M <= 0) return cudaSuccess;
    { cudaError_t e = mb_set_attrs(); if (e != cudaSuccess) return e; }
    CUtensorMap tmDy, tmW2T, tmW1T, tmHpre, tmDpre, tmDln;
    const CUtensorMapDataType BF = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    const bool ok = make_tmap_2d(&tmDy, BF, 2, dy, M, kBtC, kBtC, 64, 128) &&
                    make_tmap_2d(&tmW2T, BF, 2, W2T, kBtC, kBtC, kBtC, 64, 128) &&
                    make_tmap_2d(&tmW1T, BF, 2, W1T, kBtC, kBtC, kBtC, 64, 128) &&
                    make_tmap_2d(&tmHpre, BF, 2, hpre, M, kBtC, kBtC, 64, 32) &&
                    make_tmap_2d(&tmDpre, BF, 2, dpre, M, kBtC, kBtC, 64, 32) &&
                    make_tmap_2d(&tmDln, BF, 2, dln, M, kBtC, kBtC, 64, 32);
    if (!ok) return cudaErrorInvalidValue;
    const int ncta = M >= 256 * (num_sms / 2) ? 2 : 1;      // CTA pairs once 256-row units fill the machine
    const int tiles = (M + 128 * ncta - 1) / (128 * ncta);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(ncta * std::min(tiles, num_sms / ncta))); cfg.blockDim = dim3(kBtThreads);
    cfg.dynamicSmemBytes = kMbSmem; cfg.stream = st;
    cudaLaunchAttribute at[2];
    int na = 0;
    if (ncta == 2) {
        at[na].id = cudaLaunchAttributeClusterDimension;
        at[na].val.clusterDim.x = 2; at[na].val.clusterDim.y = 1; at[na].val.clusterDim.z = 1;
        ++na;
    }
    if (pdl_enabled(st)) {
        at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[na].val.programmaticStreamSerializationAllowed = 1;
        ++na;
    }
    cfg.attrs = at; cfg.numAttrs = (unsigned)na;
    if (ncta == 2) return cudaLaunchKernelEx(&cfg, mlp_bwd_kernel<2>, tmDy, tmW2T, tmW1T, tmHpre, tmDpre, tmDln, M);
    return cudaLaunchKernelEx(&cfg, mlp_bwd_kernel<1>, tmDy, tmW2T, tmW1T, tmHpre, tmDpre, tmDln, M);
}

}  // namespace tante
