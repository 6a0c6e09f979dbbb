// bf16 tensor-core GEMM for sm_100a:  C[M,N] = epi(A[M,K] * W[N,K]^T), fp32 accumulation in TMEM.
//
// Design (weight-stationary, persistent, warp-specialised):
//   * every GEMM of the TANTE block has a short reduction (K = 64..512) and a huge M (tokens), so the
//     K-major weight slice W[n0:n0+BN, :] (<= 128 KB) is TMA-loaded into shared memory ONCE per CTA and
//     stays resident while the CTA walks over its M tiles; only activations stream (16 KB k-blocks
//     through an mbarrier ring) -> ~256 FLOP per byte of L2/HBM traffic at BN = 256;
//   * one elected thread issues tcgen05.mma (M=128, N=BN, K=16) with both operands in SWIZZLE_128B
//     shared memory; the fp32 accumulator is double-buffered in TMEM (2 x BN columns) so the epilogue of
//     tile i overlaps the MMAs of tile i+1;
//   * 4 epilogue warps (one per TMEM lane quarter): tcgen05.ld -> registers (thread = row) -> bias /
//     activation -> swizzled shared-memory staging -> TMA bulk STORE (cp.async.bulk.tensor, OOB rows
//     clipped by the tensor map).  The fp32 residual-stream variants (x += ...) TMA-LOAD the residual
//     chunk into the same staging buffer one chunk ahead, add in place and TMA-store it back, so the
//     epilogue issues no per-element global memory instructions at all.
// Warp roles: 0 = TMA producer, 1 = MMA issuer + TMEM owner, 2..5 = epilogue.
#pragma once
#include "common.cuh"
#include "sm100_ptx.cuh"

namespace tante {

constexpr int kTcBlockM = 128;
constexpr int kTcBlockK = 64;                       // 64 bf16 = one 128-byte swizzle row
constexpr int kTcStageBytes = kTcBlockM * 128;      // 16 KB
constexpr int kTcMaxStages = 8;
constexpr int kTcEpiBuf = 32 * 128;                 // one staging buffer: 32 rows x 128 B (SWIZZLE_128B)
constexpr int kTcEpiWarps = 8;                      // 2 warps per TMEM lane quarter, interleaved column chunks
constexpr int kTcThreads = 64 + 32 * kTcEpiWarps;

__device__ __forceinline__ float gelu_tanh_fast(float x) {
    const float k = 0.79788456080286535588f;
    const float u = k * fmaf(0.044715f * x, x * x, x);
    return 0.5f * x * (1.0f + ptx::tanh_approx(u));
}

__device__ __forceinline__ float act_rt(int epi, float v) {
    switch (epi) {
        case EPI_BIAS_RELU: return fmaxf(v, 0.0f);
        case EPI_BIAS_GELU_ERF: return gelu_erf_fast(v);
        case EPI_BIAS_GELU_TANH: return gelu_tanh_fast(v);
        default: return v;
    }
}

// byte offset of 16-byte chunk `c` of row `r` inside a SWIZZLE_128B staging buffer (1024-B aligned)
__device__ __forceinline__ uint32_t sw128_off(int r, int c) { return (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4)); }

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// NCTA = 2: the CTA pair of a 2-cluster (one TPC) runs ONE tcgen05.mma.cta_group::2 of M = 256 per k-step -- each CTA
// streams its own 128 activation rows and keeps only HALF of the weight slice (BN/2 rows) resident, which frees 64 KB of
// shared memory per CTA for activation stages / epilogue staging at N = K = 256 and makes 128-wide tiles fit at K = 768.
// The leader (cluster rank 0) issues every MMA; its `full` barriers collect the TMA bytes of both CTAs, its commits are
// multicast to the `empty` / `tmem_full` barriers of both, and both epilogues release the accumulator on the leader.
template <int BN, int NCTA>
__global__ void __launch_bounds__(kTcThreads, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
               const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmR,
               const __grid_constant__ CUtensorMap tmL, int M, int N, int nkb, int nstage, int nebuf, int epi,
               int out_bf16, EpiParams ep) {
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment (SWIZZLE_128B) as an OFFSET into the shared array: a pointer -> integer -> pointer round trip would
    // lose the address space and turn every shared-memory access of the epilogue into a generic LD / ST
    uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* sW = smem;                                   // [nkb][BN rows][128 B]
    constexpr int BNC = BN / NCTA;                        // weight rows resident in THIS CTA
    uint8_t* sA = sW + (size_t)nkb * BNC * 128;           // [nstage][128 rows][128 B]
    uint8_t* sEpi = sA + (size_t)nstage * kTcStageBytes;  // [8 warps][nebuf][4 KB]
    float* sBias = reinterpret_cast<float*>(sEpi + (size_t)kTcEpiWarps * nebuf * kTcEpiBuf);   // bias, LN gamma, LN beta
    float* sStat = sBias + 3 * BN;                        // [4 quarters][2 halves][32 rows][2] partial sum / sumsq
    uint64_t* bars = reinterpret_cast<uint64_t*>(sStat + 4 * 2 * 32 * 2);
    uint64_t* full = bars;                    // [kTcMaxStages]
    uint64_t* empty = bars + kTcMaxStages;    // [kTcMaxStages]
    uint64_t* w_full = bars + 2 * kTcMaxStages;
    uint64_t* tmem_full = w_full + 1;         // [2]
    uint64_t* tmem_empty = tmem_full + 2;     // [2]
    uint64_t* rbar = tmem_empty + 2;          // [8 warps][3] residual-chunk barriers (one per staging buffer)
    uint64_t* w_pair = rbar + 3 * kTcEpiWarps;   // leader: the peer's weight half is resident
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w_pair + 1);

    pdl_trigger();
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const int crank = NCTA == 2 ? (int)ptx::cluster_ctarank() : 0;     // rank inside the CTA pair
    const int cid = blockIdx.x / NCTA;                                // cluster (= work unit) index
    const int n_slices = N / BN;
    const int slice = cid % n_slices;
    const int rank = cid / n_slices;
    const int per_slice = (gridDim.x / NCTA) / n_slices;
    const int n0 = slice * BN;
    const bool has_ln = epi == EPI_BIAS_RESID_LN;          // requires BN == N (whole row in this CTA)
    const bool has_res = epi == EPI_BIAS_RESID || has_ln;

    for (int i = threadIdx.x; i < BN; i += kTcThreads) {
        sBias[i] = ep.bias[n0 + i];
        if (has_ln) { sBias[BN + i] = ep.ln_gamma[n0 + i]; sBias[2 * BN + i] = ep.ln_beta[n0 + i]; }
    }
    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmA);
        ptx::prefetch_tmap(&tmW);
        ptx::prefetch_tmap(&tmC);
        if (has_res) ptx::prefetch_tmap(&tmR);
        if (has_ln) ptx::prefetch_tmap(&tmL);
        for (int s = 0; s < nstage; ++s) { ptx::mbar_init(&full[s], 1); ptx::mbar_init(&empty[s], 1); }
        ptx::mbar_init(w_full, 1);
        // accumulator release: the 8 local epilogue warps (+ in a pair, on the leader, one forwarded arrival of the peer)
        for (int i = 0; i < 2; ++i) {
            ptx::mbar_init(&tmem_full[i], 1);
            ptx::mbar_init(&tmem_empty[i], kTcEpiWarps + ((NCTA == 2 && ptx::cluster_ctarank() == 0) ? 1 : 0));
        }
        for (int i = 0; i < 3 * kTcEpiWarps; ++i) ptx::mbar_init(&rbar[i], 1);
        ptx::mbar_init(w_pair, 1);
        ptx::fence_barrier_init();
    }
    if (warp == 1) {
        if (NCTA == 2) { ptx::tmem_alloc_pair(tmem_slot, 2 * BN); ptx::tmem_relinquish_pair(); }
        else { ptx::tmem_alloc(tmem_slot, 2 * BN); ptx::tmem_relinquish(); }
    }
    ptx::tc_fence_before();
    if (NCTA == 2) ptx::cluster_sync_all();     // the peer's barriers are initialised before anything signals them
    else __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // Everything above touched parameters only, and so does the resident weight slice the producer requests now.  After that
    // every thread waits for the previous kernel of the stream (PDL; a no-op for an ordinary launch).
    if (warp == 0 && lane == 0) {
        ptx::mbar_arrive_expect_tx(w_full, (uint32_t)nkb * BNC * 128);
        for (int kb = 0; kb < nkb; ++kb)
            ptx::tma_load_2d(sW + (size_t)kb * BNC * 128, &tmW, w_full, kb * kTcBlockK, n0 + crank * BNC);
    }
    pdl_wait();
    if (ep.m_dev) M = min(M, *ep.m_dev * ep.m_rows);      // device-side row count (rollout encoder cache)
    const int m_tiles = (M + kTcBlockM * NCTA - 1) / (kTcBlockM * NCTA);   // tiles of 128 rows per CTA of the unit

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int mt = rank; mt < m_tiles; mt += per_slice) {
                for (int kb = 0; kb < nkb; ++kb) {
                    ptx::mbar_wait(&empty[stage], phase ^ 1);
                    if (NCTA == 2) {
                        // the leader's barrier counts the bytes of both CTAs' tiles (one arrival: the leader's)
                        if (crank == 0) ptx::mbar_arrive_expect_tx(&full[stage], 2 * kTcStageBytes);
                        ptx::tma_load_2d_pair(sA + (size_t)stage * kTcStageBytes, &tmA, &full[stage], kb * kTcBlockK,
                                              (mt * 2 + crank) * kTcBlockM);
                    } else {
                        ptx::mbar_arrive_expect_tx(&full[stage], kTcStageBytes);
                        ptx::tma_load_2d(sA + (size_t)stage * kTcStageBytes, &tmA, &full[stage], kb * kTcBlockK, mt * kTcBlockM);
                    }
                    if (++stage == nstage) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (CTA pair: the leader only; the peer just reports its weight half) =====
        constexpr uint32_t idesc = ptx::umma_idesc_bf16(kTcBlockM * NCTA, BN);
        ptx::mbar_wait(w_full, 0);
        if (NCTA == 2) {
            if (crank == 1) {
                if (lane == 0) ptx::mbar_arrive_leader(w_pair);
                // The peer's otherwise idle warp forwards "all 8 local epilogue warps released the accumulator" to the
                // leader: the cluster-scope release (MEMBAR + ERRBAR) stays off the epilogue warps' critical path.
                int tt = 0;
                for (int mt = rank; mt < m_tiles; mt += per_slice, ++tt) {
                    ptx::mbar_wait(&tmem_empty[tt & 1], (tt >> 1) & 1);
                    if (lane == 0) ptx::mbar_arrive_leader(&tmem_empty[tt & 1]);
                    __syncwarp();
                }
            } else {
                ptx::mbar_wait(w_pair, 0);
            }
        }
        int stage = 0;
        uint32_t phase = 0;
        int t = 0;
        for (int mt = rank; mt < m_tiles && crank == 0; mt += per_slice, ++t) {
            const int acc = t & 1;
            ptx::mbar_wait(&tmem_empty[acc], ((t >> 1) & 1) ^ 1);
            ptx::tc_fence_after();
            const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
            for (int kb = 0; kb < nkb; ++kb) {
                ptx::mbar_wait(&full[stage], phase);
                ptx::tc_fence_after();
                if (lane == 0) {
                    const uint64_t da = ptx::umma_desc_k_sw128(ptx::smem_u32(sA + (size_t)stage * kTcStageBytes));
                    const uint64_t db = ptx::umma_desc_k_sw128(ptx::smem_u32(sW + (size_t)kb * BNC * 128));
#pragma unroll
                    for (int k = 0; k < kTcBlockK / 16; ++k) {
                        if (NCTA == 2) ptx::umma_bf16_pair(tmem_d, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) != 0);
                        else ptx::umma_bf16(tmem_d, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) != 0);
                    }
                    // frees the smem stage (in both CTAs of a pair) when the MMAs retire
                    if (NCTA == 2) ptx::umma_commit_pair(&empty[stage]); else ptx::umma_commit(&empty[stage]);
                    if (kb == nkb - 1) { if (NCTA == 2) ptx::umma_commit_pair(&tmem_full[acc]); else ptx::umma_commit(&tmem_full[acc]); }
                }
                __syncwarp();
                if (++stage == nstage) { stage = 0; phase ^= 1; }
            }
        }
    } else {
        // ===== epilogue warps (2..9): TMEM lane quarter q = warp % 4, column chunks interleaved between the two
        //       warps of a quarter (half = 0/1); thread = one output row =====
        const int ew = warp - 2;
        const int q = warp & 3;
        const int half = ew >> 2;
        uint8_t* ebuf = sEpi + (size_t)ew * nebuf * kTcEpiBuf;
        uint64_t* rb = rbar + ew * 3;
        uint32_t rph = 0;           // fp32 path: bit b = phase of rb[b]
        int nbuf = 0;        // staging buffer the next chunk uses (bf16 path with nebuf == 2 only)
        int t = 0;
        for (int mt = rank; mt < m_tiles; mt += per_slice, ++t) {
            const int acc = t & 1;
            const int row0 = (mt * NCTA + crank) * kTcBlockM + q * 32;
            const uint32_t tm = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN);
            if (out_bf16) {
                ptx::mbar_wait(&tmem_full[acc], (t >> 1) & 1);
                ptx::tc_fence_after();
#pragma unroll 1
                for (int ch = half; ch < BN / 64; ch += 2) {
                    uint32_t r0[32], r1[32];
                    ptx::tmem_ld_32x32(tm + (uint32_t)(ch * 64), r0);
                    ptx::tmem_ld_32x32(tm + (uint32_t)(ch * 64 + 32), r1);
                    const bool alt = nebuf > 1;      // alternate the two staging buffers
                    uint8_t* buf = ebuf + (alt ? nbuf : 0) * kTcEpiBuf;
                    if (lane == 0) {
                        if (alt) ptx::bulk_wait_read<1>(); else ptx::bulk_wait_read<0>();
                    }
                    __syncwarp();
                    ptx::tc_wait_ld();
                    const float* bsm = sBias + ch * 64;
#pragma unroll
                    for (int c = 0; c < 8; ++c) {                 // 8 x 16 B chunks = 64 bf16 columns
                        uint32_t pk[4];
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const int col = c * 8 + j * 2;
                            const float a = act_rt(epi, __uint_as_float(col < 32 ? r0[col] : r1[col - 32]) + bsm[col]);
                            const float b = act_rt(epi, __uint_as_float(col + 1 < 32 ? r0[col + 1] : r1[col + 1 - 32]) + bsm[col + 1]);
                            __nv_bfloat162 h2 = __floats2bfloat162_rn(a, b);
                            pk[j] = *reinterpret_cast<uint32_t*>(&h2);
                        }
                        *reinterpret_cast<uint4*>(buf + sw128_off(lane, c)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                    }
                    ptx::fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) {
                        ptx::tma_store_2d(&tmC, buf, n0 + ch * 64, row0);
                        ptx::bulk_commit();
                    }
                    if (alt) nbuf ^= 1;
                }
            } else {
                // fp32 output in 32-column chunks, one staging buffer per warp.  The residual variants TMA-load the
                // residual chunk into the buffer (8 warps x 4 KB of loads in flight per SM), add in place and TMA-store it back.  The
                // first chunk's load is issued before the accumulator is ready, so it overlaps the MMAs.
                const int m = row0 + lane;
                // nebuf >= 2 (CTA pairs: the halved weight slice pays for up to three staging buffers per warp): the first
                // `nebuf` residual chunks of the tile are requested before the accumulator is even ready, and a buffer is
                // refilled with chunk j + nebuf as soon as the store of chunk j has drained it -- up to 3 x 4 KB of residual
                // loads in flight per warp (96 KB per SM) instead of 4 KB.
                const bool dbl = nebuf > 1;
                if (lane == 0 && (has_res || dbl)) {
                    ptx::bulk_wait_read<0>();
                    if (has_res) {
                        for (int b = 0; b < nebuf && half + 2 * b < BN / 32; ++b) {
                            ptx::mbar_arrive_expect_tx(&rb[b], kTcEpiBuf);
                            ptx::tma_load_2d(ebuf + b * kTcEpiBuf, &tmR, &rb[b], n0 + (half + 2 * b) * 32, row0);
                        }
                    }
                }
                ptx::mbar_wait(&tmem_full[acc], (t >> 1) & 1);
                ptx::tc_fence_after();
                float rsum = 0.f, rsq = 0.f;
                int jc = 0;
#pragma unroll 1
                for (int ch = half; ch < BN / 32; ch += 2, ++jc) {
                    uint32_t r0[32];
                    const int bsel = dbl ? (jc >= nebuf ? jc - nebuf : jc) : 0;      // jc % nebuf for jc < 2 * nebuf
                    uint8_t* buf = ebuf + bsel * kTcEpiBuf;
                    if (!dbl) {
                        if (lane == 0 && (ch != half || !has_res)) {
                            ptx::bulk_wait_read<0>();       // the previous store has finished reading the buffer
                            if (has_res) {
                                ptx::mbar_arrive_expect_tx(&rb[0], kTcEpiBuf);
                                ptx::tma_load_2d(buf, &tmR, &rb[0], n0 + ch * 32, row0);
                            }
                        }
                    } else if (!has_res && lane == 0 && jc >= nebuf) {
                        // this buffer's store of `nebuf` chunks ago has drained (the nebuf - 1 newer ones may be pending)
                        if (nebuf == 2) ptx::bulk_wait_read<1>(); else ptx::bulk_wait_read<2>();
                    }
                    ptx::tmem_ld_32x32(tm + (uint32_t)(ch * 32), r0);
                    __syncwarp();
                    if (has_res) { ptx::mbar_wait(&rb[bsel], (rph >> bsel) & 1u); rph ^= 1u << bsel; }
                    ptx::tc_wait_ld();
                    const float* bsm = sBias + ch * 32;
                    const int ncol = n0 + ch * 32;
#pragma unroll
                    for (int c = 0; c < 8; ++c) {                 // 8 x 16 B chunks = 32 fp32 columns
                        float4* p = reinterpret_cast<float4*>(buf + sw128_off(lane, c));
                        float4 o;
                        o.x = __uint_as_float(r0[c * 4 + 0]) + bsm[c * 4 + 0];
                        o.y = __uint_as_float(r0[c * 4 + 1]) + bsm[c * 4 + 1];
                        o.z = __uint_as_float(r0[c * 4 + 2]) + bsm[c * 4 + 2];
                        o.w = __uint_as_float(r0[c * 4 + 3]) + bsm[c * 4 + 3];
                        if (has_res) {
                            const float4 x = *p;
                            o.x += x.x; o.y += x.y; o.z += x.z; o.w += x.w;
                            if (has_ln) {       // keep the updated row in TMEM (over the accumulator) for the LN pass
                                r0[c * 4 + 0] = __float_as_uint(o.x); r0[c * 4 + 1] = __float_as_uint(o.y);
                                r0[c * 4 + 2] = __float_as_uint(o.z); r0[c * 4 + 3] = __float_as_uint(o.w);
                                rsum += (o.x + o.y) + (o.z + o.w);
                                rsq = fmaf(o.x, o.x, rsq); rsq = fmaf(o.y, o.y, rsq);
                                rsq = fmaf(o.z, o.z, rsq); rsq = fmaf(o.w, o.w, rsq);
                            }
                        } else if (epi == EPI_EMBED) {
                            if (m < M) {
                                const int hw = m % ep.L, tt = (m / ep.L) % ep.T;
                                const int n = ncol + c * 4;
                                const float4 sc = *reinterpret_cast<const float4*>(ep.film + (size_t)(tt * 2 + 0) * ep.ldr + n);
                                const float4 sh = *reinterpret_cast<const float4*>(ep.film + (size_t)(tt * 2 + 1) * ep.ldr + n);
                                const float4 se = *reinterpret_cast<const float4*>(ep.s_emb + (size_t)hw * ep.ldr + n);
                                const float4 te = *reinterpret_cast<const float4*>(ep.t_emb + (size_t)tt * ep.ldr + n);
                                o.x = embed_value(o.x, sc.x, sh.x, se.x, te.x);
                                o.y = embed_value(o.y, sc.y, sh.y, se.y, te.y);
                                o.z = embed_value(o.z, sc.z, sh.z, se.z, te.z);
                                o.w = embed_value(o.w, sc.w, sh.w, se.w, te.w);
                            }
                        } else {
                            o.x = act_rt(epi, o.x); o.y = act_rt(epi, o.y); o.z = act_rt(epi, o.z); o.w = act_rt(epi, o.w);
                        }
                        *p = o;
                    }
                    if (has_ln) ptx::tmem_st_32x32(tm + (uint32_t)(ch * 32), r0);
                    ptx::fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) {
                        ptx::tma_store_2d(&tmC, buf, ncol, row0);
                        ptx::bulk_commit();
                        if (dbl && has_res && ch + 2 * nebuf < BN / 32) {
                            ptx::bulk_wait_read<0>();       // the store just issued has drained this buffer: refill it
                            ptx::mbar_arrive_expect_tx(&rb[bsel], kTcEpiBuf);
                            ptx::tma_load_2d(buf, &tmR, &rb[bsel], n0 + (ch + 2 * nebuf) * 32, row0);
                        }
                    }
                }
                if (has_ln) {
                    // LayerNorm of the updated row: the two warps of this lane quarter exchange their partial row
                    // statistics through shared memory, then each normalises its share of the row straight out of
                    // TMEM (-> affine -> bf16 -> staging -> TMA store into the next GEMM's A operand).
                    float* st = sStat + ((q * 2 + half) * 32 + lane) * 2;
                    st[0] = rsum; st[1] = rsq;
                    ptx::tc_wait_st();
                    ptx::tc_fence_before();
                    named_bar_sync(1 + q, 64);
                    ptx::tc_fence_after();
                    const float* so = sStat + ((q * 2 + (half ^ 1)) * 32 + lane) * 2;
                    const float mean = (rsum + so[0]) * (1.0f / BN);
                    const float var = fmaxf((rsq + so[1]) * (1.0f / BN) - mean * mean, 0.f);
                    const float rstd = rsqrtf(var + 1e-5f);
#pragma unroll 1
                    for (int ch = half; ch < BN / 64; ch += 2) {
                        uint32_t r0[32], r1[32];
                        ptx::tmem_ld_32x32(tm + (uint32_t)(ch * 64), r0);
                        ptx::tmem_ld_32x32(tm + (uint32_t)(ch * 64 + 32), r1);
                        if (lane == 0) ptx::bulk_wait_read<0>();
                        __syncwarp();
                        ptx::tc_wait_ld();
                        uint8_t* buf = ebuf;
                        const float* gsm = sBias + BN + ch * 64;
                        const float* bsm2 = sBias + 2 * BN + ch * 64;
#pragma unroll
                        for (int c = 0; c < 8; ++c) {
                            uint32_t pk[4];
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const int col = c * 8 + j * 2;
                                const float a = (__uint_as_float(col < 32 ? r0[col] : r1[col - 32]) - mean) * rstd * gsm[col] + bsm2[col];
                                const float b = (__uint_as_float(col + 1 < 32 ? r0[col + 1] : r1[col + 1 - 32]) - mean) * rstd * gsm[col + 1] + bsm2[col + 1];
                                __nv_bfloat162 h2 = __floats2bfloat162_rn(a, b);
                                pk[j] = *reinterpret_cast<uint32_t*>(&h2);
                            }
                            *reinterpret_cast<uint4*>(buf + sw128_off(lane, c)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                        }
                        ptx::fence_proxy_async();
                        __syncwarp();
                        if (lane == 0) {
                            ptx::tma_store_2d(&tmL, buf, n0 + ch * 64, row0);
                            ptx::bulk_commit();
                        }
                    }
                    // sStat is reused by the next tile: make sure the partner has read it
                    named_bar_sync(1 + q, 64);
                }
            }
            ptx::tc_fence_before();
            if (lane == 0) ptx::mbar_arrive(&tmem_empty[acc]);
        }
        if (lane == 0) ptx::bulk_wait_all<0>();
    }
    ptx::tc_fence_before();
    if (NCTA == 2) ptx::cluster_sync_all();     // neither CTA leaves (or frees TMEM) while the pair's MMAs may still touch it
    else __syncthreads();
    if (warp == 1) { if (NCTA == 2) ptx::tmem_dealloc_pair(tmem_base, 2 * BN); else ptx::tmem_dealloc(tmem_base, 2 * BN); }
}

// ---- host side ----------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_tiled() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            return nullptr;
        fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}

// 2-D row-major tensor map, dims {cols, rows}; the box is one swizzle span wide (128 B for SWIZZLE_128B, 64 B for SWIZZLE_64B).
static bool make_tmap_2d(CUtensorMap* m, CUtensorMapDataType dt, int esize, const void* base, int rows, int cols,
                         int ld_elems, int box_cols, int box_rows, CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
    PFN_encodeTiled enc = get_encode_tiled();
    if (!enc) return false;
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld_elems * esize};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    return enc(m, dt, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

struct TcPlan { int BN, ncta, nkb, nstage, nebuf, grid; size_t smem; };

// CTA pairs (cta_group::2) where they pay off.  Measured on B200 (tools/gemm_probe.py, M = 262144 / 65536, N = K = 256): the fp32 residual (+LayerNorm) epilogues gain
// 16-19 % / 11-14 % from the second staging buffer the halved weight slice pays for (156.6 -> 126.9 us, 188.7 -> 158.2 us);
// plain bf16 epilogues lose 4-19 % to the lock-step of the pair, so they stay on single CTAs unless the reduction is so
// long (K = 768) that a single CTA could only keep a 64-wide weight slice resident.

static bool tc_plan(int M, int N, int K, int num_sms, int out_bf16, TcPlan* p) {
    if (K % kTcBlockK != 0 || K > 1024 || N % 64 != 0) return false;
    if ((size_t)(K / kTcBlockK) * 64 * 128 > 128 * 1024) return false;
    const int nkb = K / kTcBlockK;
    int BN = (N % 256 == 0) ? 256 : (N % 128 == 0 ? 128 : 64);
    // pairs need >= 128 columns (64 per CTA) and enough 256-row tiles to fill the machine
    const bool narrow_single = (size_t)nkb * 128 * 128 > 128 * 1024;        // a single CTA would be down to 64-wide slices
    const bool pays = !out_bf16 || (narrow_single && N >= 128);
    const int ncta = (pays && N % 128 == 0 && M >= 256 * (num_sms / 2)) ? 2 : 1;
    while ((size_t)nkb * (BN / ncta) * 128 > 128 * 1024 && BN > 64 * ncta) BN /= 2;   // keep the resident slice <= 128 KB
    if ((size_t)nkb * (BN / ncta) * 128 > 128 * 1024) return false;
    // pairs: the halved weight slice pays for a second staging buffer per epilogue warp (if >= 3 activation stages remain)
    int nebuf = ncta == 2 ? (out_bf16 ? 2 : 3) : 1;
    const size_t budget = 227 * 1024;
    size_t fixed = 0;
    int nstage = 0;
    for (;; --nebuf) {
        fixed = (size_t)nkb * (BN / ncta) * 128 + (size_t)kTcEpiWarps * nebuf * kTcEpiBuf + 3 * BN * 4 + 4 * 2 * 32 * 2 * 4 + 512 + 1024;
        nstage = fixed < budget ? (int)((budget - fixed) / kTcStageBytes) : 0;
        if (nstage >= 3 || nebuf == 1) break;
    }
    nstage = nstage > kTcMaxStages ? kTcMaxStages : nstage;
    if (ncta == 1 && nstage > 6) nstage = 6;
    if (nstage < 2) return false;
    const int n_slices = N / BN;
    const int m_tiles = (M + kTcBlockM * ncta - 1) / (kTcBlockM * ncta);
    int per_slice = (num_sms / ncta) / n_slices;
    if (per_slice < 1) per_slice = 1;
    if (per_slice > m_tiles) per_slice = m_tiles;
    p->BN = BN; p->ncta = ncta; p->nkb = nkb; p->nstage = nstage; p->nebuf = nebuf; p->grid = per_slice * n_slices * ncta;
    p->smem = fixed + (size_t)nstage * kTcStageBytes;
    return true;
}

static cudaError_t tc_set_attrs() {
    static unsigned long long attr_done = 0;
    if (!get_encode_tiled()) return cudaErrorNotSupported;
    if (!attrs_needed(attr_done)) return cudaSuccess;
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(gemm_tc_kernel<256, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(gemm_tc_kernel<128, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(gemm_tc_kernel<64, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(gemm_tc_kernel<256, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(gemm_tc_kernel<128, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)) != cudaSuccess) return e;
    return cudaSuccess;
}

// Programmatic dependent launch for the tensor-core kernels (common.cuh): not inside stream capture (the rollout graphs keep
// plain kernel nodes).
static bool pdl_enabled(cudaStream_t st) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    return cs == cudaStreamCaptureStatusNone;
}

static cudaError_t launch_gemm_tc(int epi, const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, int ldw, void* C,
                                  int ldc, int out_bf16, int M, int N, int K, const EpiParams& ep, int num_sms,
                                  cudaStream_t st) {
    if (M <= 0) return cudaSuccess;
    TcPlan p;
    if (!tc_plan(M, N, K, num_sms, out_bf16, &p)) return cudaErrorInvalidValue;
    if (!out_bf16 && N % 32 != 0) return cudaErrorInvalidValue;
    CUtensorMap tmA, tmW, tmC, tmR, tmL;
    const bool is_ln = epi == EPI_BIAS_RESID_LN;
    if (is_ln && (out_bf16 || p.BN != N || !ep.ln_out || !ep.ln_gamma || !ep.ln_beta)) return cudaErrorInvalidValue;
    if (!make_tmap_2d(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, A, M, K, lda, kTcBlockK, kTcBlockM)) return cudaErrorInvalidValue;
    if (!make_tmap_2d(&tmW, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, W, N, K, ldw, kTcBlockK, p.BN / p.ncta)) return cudaErrorInvalidValue;
    if (out_bf16) {
        if (!make_tmap_2d(&tmC, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, C, M, N, ldc, 64, 32)) return cudaErrorInvalidValue;
    } else {
        if (!make_tmap_2d(&tmC, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, C, M, N, ldc, 32, 32)) return cudaErrorInvalidValue;
    }
    tmR = tmC;
    tmL = tmC;
    if (is_ln && !make_tmap_2d(&tmL, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, ep.ln_out, M, N, N, 64, 32)) return cudaErrorInvalidValue;
    if (epi == EPI_BIAS_RESID || is_ln) {
        if (out_bf16) return cudaErrorInvalidValue;
        if (!make_tmap_2d(&tmR, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, ep.resid, M, N, ep.ldr, 32, 32)) return cudaErrorInvalidValue;
    }
    { cudaError_t e = tc_set_attrs(); if (e != cudaSuccess) return e; }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)p.grid); cfg.blockDim = dim3(kTcThreads); cfg.dynamicSmemBytes = p.smem; cfg.stream = st;
    cudaLaunchAttribute at[2];
    int na = 0;
    if (p.ncta == 2) {
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
#define TANTE_TC_LAUNCH(BNv, NC) \
    return cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BNv, NC>, tmA, tmW, tmC, tmR, tmL, M, N, p.nkb, p.nstage, p.nebuf, epi, out_bf16, ep)
    if (p.ncta == 2) { if (p.BN == 256) TANTE_TC_LAUNCH(256, 2); TANTE_TC_LAUNCH(128, 2); }
    if (p.BN == 256) TANTE_TC_LAUNCH(256, 1);
    if (p.BN == 128) TANTE_TC_LAUNCH(128, 1);
    TANTE_TC_LAUNCH(64, 1);
#undef TANTE_TC_LAUNCH
}

}  // namespace tante
