// Fused "tail" of a TANTE transformer block on tcgen05 (reference models/attn_backbone.py:81-83 + the LayerNorm of the
// next layer, :68): everything after the attention core of a TransformerBlock in ONE kernel --
//
//     x_mid = x + att * Wo^T + bo                          (attention out-projection + residual)
//     h     = gelu_tanh( LN2(x_mid) * W1^T + b1 )          (MLP in)
//     x_out = x_mid + h * W2^T + b2                        (MLP out + residual)
//     ln    = LN1'(x_out)                                  (pre-LN of the NEXT layer, the A operand of its QKV GEMM)
//
// The un-fused path runs three GEMM launches for this (gemm_tc_kernel: out-proj + residual + LN2, MLP-in + GELU, MLP-out +
// residual + LN1') and moves per token 512 + 1024 + 1024 + 512 | 512 + 512 | 512 + 1024 + 1024 + 512 = 7 KB through HBM; here the
// LN2 output, the hidden activations and x_mid never leave the SM: 512 (att) + 1024 (x) in, 1024 (x) + 512 (ln) out = 3 KB.
//
// One CTA per SM, persistent over 128-token tiles.  Per tile three chained MMAs share one TMEM accumulator (256 columns) and
// one 64 KB shared-memory A tile that is rewritten in place by the epilogue warps between the phases (att -> LN2 -> hidden, all
// K-major SWIZZLE_128B, exactly the layout TMA would have produced); x_mid lives in the other 256 TMEM columns from the first
// epilogue to the last.  The three 128 KB weight matrices do not fit next to that, so they STREAM from L2 through a ring of
// 16 KB stages ([128 rows of N][64 of K]; 24 stages per tile = 384 KB per 128 tokens, L2-resident: 0.4 MB of weights in total).
// The residual chunks arrive by TMA: the first of a warp's two into its staging buffer (requested before the accumulator
// is ready), the second into a 4 KB slot of the A tile, which is idle between the first GEMM and the LayerNorm pass;
// results leave by TMA stores from the staging buffers (training: LN2 / hidden straight from the A tile).
// TRAIN = true additionally stores what the backward needs (x_mid, LN2 output, MLP pre-activation, hidden).
// Warp roles: 0 = TMA producer, 1 = MMA issuer + TMEM owner, 2..17 = epilogue (four per TMEM lane quarter).
#pragma once
#include "common.cuh"
#include "gemm_tc.cuh"
#include "sm100_ptx.cuh"

namespace tante {

constexpr int kBtEpiWarps = 16;
// CTA pairs: true = the peer's 16 epilogue warps arrive on the leader's barriers themselves; false = the peer's idle warp 1 forwards
// ONE arrival.  Measured (B200, M = 262144): direct 230 us vs forwarded 220 us -- the cluster-scope release on every epilogue
// warp's critical path costs more than the extra hop.
constexpr bool kBtDirect = false;
constexpr int kBtThreads = 64 + 32 * kBtEpiWarps;
constexpr int kBtC = 256;                   // embed_dim the kernel is specialised for
constexpr int kBtKBlk = 128 * 128;          // one k-block of the A tile: [128 rows][64 bf16] = 16 KB
constexpr int kBtWStage = 128 * 128;        // one weight stage: [128 rows of N][64 of K] bf16 = 16 KB
constexpr int kBtWStages = 5;
constexpr int kBtEbuf = 32 * 128;           // staging buffer: 32 rows x 128 B
constexpr size_t kBtSmem = 1024 + 4 * kBtKBlk + kBtWStages * kBtWStage + kBtEpiWarps * kBtEbuf + 7 * kBtC * 4 + 2 * 4 * 4 * 32 * 2 * 4 + 512;

struct BtParams {
    const float* bo; const float* g2; const float* be2; const float* b1; const float* b2; const float* gn; const float* ben;
    int M;
    int has_ln_out;      // 0 for the last layer of a backbone (no next LayerNorm)
    DropCfg drop;        // training with dropout (attn_backbone.py:81-83): both residual branches are masked
    uint32_t site1, site2;
};

// NCTA = 2: the CTA pair of a 2-cluster runs every MMA as ONE tcgen05.mma.cta_group::2 of M = 256 (gemm_tc.cuh): each CTA owns
// 128 token rows (its own A tile, accumulator, x_mid, epilogue) and streams only ITS HALF of every weight stage (128 of the
// 256 output rows), so the weight traffic per token -- the L2 -> SM stream that bounds this kernel -- is halved and a ring
// stage covers a whole k-block.  The leader (cluster rank 0) issues the MMAs; its barriers collect the TMA bytes of both
// CTAs, its commits are multicast to both, and the peer's idle warp 1 forwards "A tile rewritten" / "accumulator free".
template <int MODE /* 0: inference, 1: training (stores the tape), 2: training with dropout */, int NCTA>
__global__ void __launch_bounds__(kBtThreads, 1)
block_tail_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmWo,
                  const __grid_constant__ CUtensorMap tmW1, const __grid_constant__ CUtensorMap tmW2,
                  const __grid_constant__ CUtensorMap tmXin, const __grid_constant__ CUtensorMap tmXmid,
                  const __grid_constant__ CUtensorMap tmXout, const __grid_constant__ CUtensorMap tmLn2,
                  const __grid_constant__ CUtensorMap tmHpre, const __grid_constant__ CUtensorMap tmHact,
                  const __grid_constant__ CUtensorMap tmLnOut, BtParams p) {
    constexpr bool TRAIN = MODE != 0;
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment (SWIZZLE_128B) as an OFFSET into the shared array: a pointer -> integer -> pointer round trip would
    // lose the address space and turn every shared-memory access of the epilogue into a generic LD / ST
    uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* sA = smem;                                        // [4 k-blocks][128 rows][128 B]
    uint8_t* sW = sA + 4 * kBtKBlk;                            // [kBtWStages][128 rows][128 B]
    uint8_t* sE = sW + kBtWStages * kBtWStage;                 // [16 warps][4 KB]
    float* sP = reinterpret_cast<float*>(sE + kBtEpiWarps * kBtEbuf);    // bo, g2, be2, b1, b2, gn, ben
    float* sStat = sP + 7 * kBtC;                              // [2 sets][4 quarters][4 slices][32 rows][2]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sStat + 2 * 4 * 4 * 32 * 2);
    uint64_t* w_full = bars;                       // [kBtWStages]
    uint64_t* w_empty = bars + kBtWStages;         // [kBtWStages]
    uint64_t* a_full = bars + 2 * kBtWStages;      // att tile landed
    uint64_t* a_empty = a_full + 1;                // the tile's last MMA has read the A tile
    uint64_t* a_ready = a_full + 2;                // the epilogue warps rewrote the A tile (16 arrivals)
    uint64_t* acc_full = a_full + 3;               // one MMA phase finished
    uint64_t* acc_free = a_full + 4;               // the last epilogue has read the accumulator (16 arrivals)
    uint64_t* rbar = a_full + 5;                   // [16 warps][2] residual-chunk barriers
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(rbar + 2 * kBtEpiWarps);

    pdl_trigger();
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const int crank = NCTA == 2 ? (int)ptx::cluster_ctarank() : 0;     // rank inside the CTA pair
    const int cid = blockIdx.x / NCTA;                                // work-unit sequence of this CTA (pair)
    const int ncl = gridDim.x / NCTA;
    const int tiles = (p.M + 128 * NCTA - 1) / (128 * NCTA);          // units of 128 rows per CTA

    for (int i = threadIdx.x; i < kBtC; i += kBtThreads) {
        sP[i] = p.bo[i]; sP[kBtC + i] = p.g2[i]; sP[2 * kBtC + i] = p.be2[i]; sP[3 * kBtC + i] = p.b1[i];
        sP[4 * kBtC + i] = p.b2[i];
        sP[5 * kBtC + i] = p.has_ln_out ? p.gn[i] : 1.f; sP[6 * kBtC + i] = p.has_ln_out ? p.ben[i] : 0.f;
    }
    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmA); ptx::prefetch_tmap(&tmWo); ptx::prefetch_tmap(&tmW1); ptx::prefetch_tmap(&tmW2);
        ptx::prefetch_tmap(&tmXin); ptx::prefetch_tmap(&tmXout);
        if (p.has_ln_out) ptx::prefetch_tmap(&tmLnOut);
        for (int s = 0; s < kBtWStages; ++s) { ptx::mbar_init(&w_full[s], 1); ptx::mbar_init(&w_empty[s], 1); }
        ptx::mbar_init(a_full, 1);
        ptx::mbar_init(a_empty, TRAIN ? 1 + kBtEpiWarps : 1);     // the last GEMM's commit (+ training: the stores that read the A tile)
        // pair: the leader's copies also take one forwarded arrival of the peer
        ptx::mbar_init(a_ready, kBtEpiWarps + ((NCTA == 2 && crank == 0) ? (kBtDirect ? kBtEpiWarps : 1) : 0));
        ptx::mbar_init(acc_full, 1);
        ptx::mbar_init(acc_free, kBtEpiWarps + ((NCTA == 2 && crank == 0) ? (kBtDirect ? kBtEpiWarps : 1) : 0));
        for (int i = 0; i < 2 * kBtEpiWarps; ++i) ptx::mbar_init(&rbar[i], 1);
        ptx::fence_barrier_init();
    }
    if (warp == 1) {
        if (NCTA == 2) { ptx::tmem_alloc_pair(tmem_slot, 512); ptx::tmem_relinquish_pair(); }
        else { ptx::tmem_alloc(tmem_slot, 512); ptx::tmem_relinquish(); }
    }
    ptx::tc_fence_before();
    if (NCTA == 2) ptx::cluster_sync_all();     // the peer's barriers are initialised before anything signals them
    else __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();

    if (warp == 0) {
        // ===== TMA producer: the tile's att rows, then its 24 weight stages =====
        if (lane == 0) {
            int ws = 0;
            uint32_t wph = 0;
            int it = 0;
            for (int tile = cid; tile < tiles; tile += ncl, ++it) {
                ptx::mbar_wait(a_empty, (uint32_t)(it & 1) ^ 1u);
                if (NCTA == 2) {
                    // the leader's barrier counts the bytes of both CTAs' tiles (one arrival: the leader's)
                    if (crank == 0) ptx::mbar_arrive_expect_tx(a_full, 2 * 4 * kBtKBlk);
                    for (int kb = 0; kb < 4; ++kb)
                        ptx::tma_load_2d_pair(sA + kb * kBtKBlk, &tmA, a_full, kb * 64, (tile * 2 + crank) * 128);
                } else {
                    ptx::mbar_arrive_expect_tx(a_full, 4 * kBtKBlk);
                    for (int kb = 0; kb < 4; ++kb) ptx::tma_load_2d(sA + kb * kBtKBlk, &tmA, a_full, kb * 64, tile * 128);
                }
                for (int ph = 0; ph < 3; ++ph) {
                    const CUtensorMap* wm = ph == 0 ? &tmWo : (ph == 1 ? &tmW1 : &tmW2);
                    for (int kb = 0; kb < 4; ++kb) {
                        for (int nh = 0; nh < 2 / NCTA; ++nh) {
                            ptx::mbar_wait(&w_empty[ws], wph ^ 1u);
                            if (NCTA == 2) {      // this CTA's half of the output rows of k-block kb
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
        // ===== MMA issuer: three chained GEMM phases per tile into the one accumulator =====
        constexpr uint32_t idesc = NCTA == 2 ? ptx::umma_idesc_bf16(256, 256) : ptx::umma_idesc_bf16(128, 128);
        int ws = 0;
        uint32_t wph = 0, ar = 0;
        int it = 0;
        if (NCTA == 2 && crank == 1 && !kBtDirect) {
            // the peer's otherwise idle warp forwards its epilogue's "A tile rewritten" (twice per tile) and "accumulator
            // free" to the leader's barriers
            for (int tile = cid; tile < tiles; tile += ncl, ++it) {
                for (int ph = 1; ph < 3; ++ph) {
                    ptx::mbar_wait(a_ready, ar & 1u);
                    ++ar;
                    if (lane == 0) ptx::mbar_arrive_leader(a_ready);
                    __syncwarp();
                }
                ptx::mbar_wait(acc_free, (uint32_t)(it & 1));
                if (lane == 0) ptx::mbar_arrive_leader(acc_free);
                __syncwarp();
            }
        }
        for (int tile = cid; tile < tiles && crank == 0; tile += ncl, ++it) {
            for (int ph = 0; ph < 3; ++ph) {
                if (ph == 0) {
                    ptx::mbar_wait(acc_free, (uint32_t)(it & 1) ^ 1u);     // the previous tile's accumulator has been read
                    ptx::mbar_wait(a_full, (uint32_t)(it & 1));
                } else {
                    ptx::mbar_wait(a_ready, ar & 1u);                       // the A tile was rewritten (and acc read) by the epilogue
                    ++ar;
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
                        if (ph == 2) ptx::umma_commit_pair(a_empty);
                    } else {
                        ptx::umma_commit(acc_full);
                        if (ph == 2) ptx::umma_commit(a_empty);
                    }
                }
                __syncwarp();
            }
        }
    } else {
        // ===== 16 epilogue warps: TMEM lane quarter q = warp % 4 (thread = one token row), column slice cs = 0..3 =====
        // fp32 passes: the warp owns the 32-column chunks cs and cs + 4 of its rows; bf16 passes: the 64-column k-block cs.
        // (Four warps per scheduler: the epilogue is a chain of TMEM / shared-memory round trips per row, and with two
        //  warps per scheduler -- the first version, 8 epilogue warps -- the issue slots were 30 % busy.)
        const int ew = warp - 2;
        const int q = warp & 3;
        const int cs = ew >> 2;
        uint8_t* ebuf = sE + (size_t)ew * kBtEbuf;             // own staging buffer (4 KB)
        uint8_t* aown = sA + (size_t)cs * kBtKBlk + (size_t)q * 32 * 128;    // this warp's 32 rows of k-block cs inside the A tile
        uint8_t* aslot = aown;     // phase 1: landing zone of the second residual chunk (the A tile is idle; no other warp touches this region)
        uint64_t* rb = rbar + ew * 2;
        uint32_t rph = 0;             // bit b = phase of rb[b]
        uint32_t af = 0;              // completed acc_full waits
        bool st_pending = false;      // a TMA store of this warp may still be reading ebuf
        auto ebuf_free = [&]() {
            if (st_pending && lane == 0) ptx::bulk_wait_read<0>();
            st_pending = false;
            __syncwarp();
        };
        const float* bo = sP; const float* g2 = sP + kBtC; const float* be2 = sP + 2 * kBtC; const float* b1 = sP + 3 * kBtC;
        const float* b2 = sP + 4 * kBtC; const float* gn = sP + 5 * kBtC; const float* ben = sP + 6 * kBtC;
        constexpr bool dropping = MODE == 2;

        // row statistics of the four column slices of a quarter -> mean, 1 / std
        auto row_stats = [&](int set, float rsum, float rsq, float& mean, float& rstd) {
            float* st = sStat + (size_t)set * 4 * 4 * 32 * 2;
            st[((q * 4 + cs) * 32 + lane) * 2 + 0] = rsum;
            st[((q * 4 + cs) * 32 + lane) * 2 + 1] = rsq;
            ptx::tc_wait_st();
            ptx::tc_fence_before();
            named_bar_sync(5 + q, 4 * 32);          // the four warps of the quarter (same token rows): statistics + TMEM rows written
            ptx::tc_fence_after();
            float s = 0.f, sq = 0.f;
#pragma unroll
            for (int c = 0; c < 4; ++c) { s += st[((q * 4 + c) * 32 + lane) * 2]; sq += st[((q * 4 + c) * 32 + lane) * 2 + 1]; }
            mean = s * (1.0f / kBtC);
            const float var = fmaxf(sq * (1.0f / kBtC) - mean * mean, 0.f);
            rstd = rsqrtf(var + 1e-5f);
        };
        // LayerNorm of this warp's k-block (64 columns out of the TMEM x region) -> bf16 -> 32 rows x 128 B at `dst` (SWIZZLE_128B)
        auto ln_kblock = [&](uint32_t tm_x, float mean, float rstd, const float* gam, const float* bet, uint8_t* dst, int drow) {
            const float mr = mean * rstd;
#pragma unroll 1
            for (int hh = 0; hh < 2; ++hh) {
                uint32_t r0[32];
                ptx::tmem_ld_32x32(tm_x + (uint32_t)(cs * 64 + hh * 32), r0);
                ptx::tc_wait_ld();
                const float* gs = gam + cs * 64 + hh * 32;
                const float* bs = bet + cs * 64 + hh * 32;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    uint32_t pk[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int col = c * 8 + j * 2;
                        const float a = fmaf(fmaf(__uint_as_float(r0[col]), rstd, -mr), gs[col], bs[col]);
                        const float bb = fmaf(fmaf(__uint_as_float(r0[col + 1]), rstd, -mr), gs[col + 1], bs[col + 1]);
                        __nv_bfloat162 h2 = __floats2bfloat162_rn(a, bb);
                        pk[j] = *reinterpret_cast<uint32_t*>(&h2);
                    }
                    *reinterpret_cast<uint4*>(dst + sw128_off(drow, hh * 4 + c)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                }
            }
        };

        for (int tile = cid; tile < tiles; tile += ncl) {
            const int row0 = (tile * NCTA + crank) * 128 + q * 32;
            const uint32_t tm_acc = tmem_base + ((uint32_t)(q * 32) << 16);
            const uint32_t tm_x = tm_acc + 256u;

            // ---------------- phase 1: x_mid = x + drop(acc + bo) ; LN2 -> A tile ----------------
            ebuf_free();
            if (lane == 0) {
                ptx::mbar_arrive_expect_tx(&rb[0], kBtEbuf);
                ptx::tma_load_2d(ebuf, &tmXin, &rb[0], cs * 32, row0);
            }
            ptx::mbar_wait(acc_full, af & 1u); ++af;
            ptx::tc_fence_after();
            if (lane == 0) {      // the A tile has been consumed by the first GEMM: its 4 KB slot takes the second chunk
                ptx::mbar_arrive_expect_tx(&rb[1], kBtEbuf);
                ptx::tma_load_2d(aslot, &tmXin, &rb[1], (cs + 4) * 32, row0);
            }
            float rsum = 0.f, rsq = 0.f;
#pragma unroll 1
            for (int jc = 0; jc < 2; ++jc) {
                const int ch = cs + 4 * jc;
                uint8_t* buf = jc == 0 ? ebuf : aslot;
                uint32_t r0[32];
                ptx::tmem_ld_32x32(tm_acc + (uint32_t)(ch * 32), r0);
                ptx::mbar_wait(&rb[jc], (rph >> jc) & 1u); rph ^= 1u << jc;
                ptx::tc_wait_ld();
                const float* bs = bo + ch * 32;
                uint4 dw = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    float4* pp = reinterpret_cast<float4*>(buf + sw128_off(lane, c));
                    const float4 x = *pp;
                    float4 o;
                    o.x = __uint_as_float(r0[c * 4 + 0]) + bs[c * 4 + 0];
                    o.y = __uint_as_float(r0[c * 4 + 1]) + bs[c * 4 + 1];
                    o.z = __uint_as_float(r0[c * 4 + 2]) + bs[c * 4 + 2];
                    o.w = __uint_as_float(r0[c * 4 + 3]) + bs[c * 4 + 3];
                    if (dropping) {       // x + drop(attention branch): 8 consecutive columns share one Philox group
                        if ((c & 1) == 0) dw = drop_words(p.drop, p.site1, (unsigned long long)(row0 + lane) * (kBtC / 8) + ch * 4 + (c >> 1));
                        const int l0 = (c & 1) * 4;
                        o.x *= drop_mul(p.drop, dw, l0); o.y *= drop_mul(p.drop, dw, l0 + 1);
                        o.z *= drop_mul(p.drop, dw, l0 + 2); o.w *= drop_mul(p.drop, dw, l0 + 3);
                    }
                    o.x += x.x; o.y += x.y; o.z += x.z; o.w += x.w;
                    r0[c * 4 + 0] = __float_as_uint(o.x); r0[c * 4 + 1] = __float_as_uint(o.y);
                    r0[c * 4 + 2] = __float_as_uint(o.z); r0[c * 4 + 3] = __float_as_uint(o.w);
                    rsum += (o.x + o.y) + (o.z + o.w);
                    rsq += fmaf(o.x, o.x, fmaf(o.y, o.y, fmaf(o.z, o.z, o.w * o.w)));
                    if (TRAIN) *pp = o;
                }
                ptx::tmem_st_32x32(tm_x + (uint32_t)(ch * 32), r0);
                if (TRAIN) {
                    ptx::fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) { ptx::tma_store_2d(&tmXmid, buf, ch * 32, row0); ptx::bulk_commit(); }
                }
            }
            if (TRAIN) {      // both x_mid stores have drained: the slot is about to be overwritten by the LayerNorm output
                if (lane == 0) ptx::bulk_wait_read<0>();
                __syncwarp();
            }
            {
                float mean, rstd;
                row_stats(0, rsum, rsq, mean, rstd);
                ln_kblock(tm_x, mean, rstd, g2, be2, aown, lane);
                if (TRAIN) {      // the saved LN2 output leaves straight from the A tile (same 32-row x 128-B swizzled box)
                    ptx::fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) { ptx::tma_store_2d(&tmLn2, aown, cs * 64, row0); ptx::bulk_commit(); }
                }
            }
            ptx::fence_proxy_async();
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) { if (NCTA == 2 && crank == 1 && kBtDirect) ptx::mbar_arrive_leader(a_ready); else ptx::mbar_arrive(a_ready); }

            // ---------------- phase 2: hidden = gelu_tanh(acc + b1) -> A tile ----------------
            ptx::mbar_wait(acc_full, af & 1u); ++af;
            ptx::tc_fence_after();
            if (lane == 0 && tile + ncl < tiles) {      // pull the next tile's residual rows into L2 (the loads themselves are issued late)
                const int nrow0 = ((tile + ncl) * NCTA + crank) * 128 + q * 32;
                ptx::tma_prefetch_l2_2d(&tmXin, cs * 32, nrow0);
                ptx::tma_prefetch_l2_2d(&tmXin, (cs + 4) * 32, nrow0);
            }
            if (TRAIN) {      // the LN2 store has finished reading this warp's rows of the A tile
                if (lane == 0) ptx::bulk_wait_read<0>();
                __syncwarp();
            }
#pragma unroll 1
            for (int hh = 0; hh < 2; ++hh) {
                uint32_t r0[32];
                ptx::tmem_ld_32x32(tm_acc + (uint32_t)(cs * 64 + hh * 32), r0);
                ptx::tc_wait_ld();
                const float* bs = b1 + cs * 64 + hh * 32;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    uint32_t pk[4], pp[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int col = c * 8 + j * 2;
                        float a = __uint_as_float(r0[col]) + bs[col];
                        float bb = __uint_as_float(r0[col + 1]) + bs[col + 1];
                        if (TRAIN) {
                            // the backward differentiates the activation at the SAVED (bf16) pre-activation: use it here too
                            __nv_bfloat162 pr = __floats2bfloat162_rn(a, bb);
                            pp[j] = *reinterpret_cast<uint32_t*>(&pr);
                            const float2 f = __bfloat1622float2(pr);
                            a = f.x; bb = f.y;
                        }
                        __nv_bfloat162 h2 = __floats2bfloat162_rn(gelu_tanh_fast(a), gelu_tanh_fast(bb));
                        pk[j] = *reinterpret_cast<uint32_t*>(&h2);
                    }
                    *reinterpret_cast<uint4*>(aown + sw128_off(lane, hh * 4 + c)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                    if (TRAIN) *reinterpret_cast<uint4*>(ebuf + sw128_off(lane, hh * 4 + c)) = make_uint4(pp[0], pp[1], pp[2], pp[3]);
                }
            }
            if (TRAIN) {
                ptx::fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
                    ptx::tma_store_2d(&tmHpre, ebuf, cs * 64, row0);
                    ptx::tma_store_2d(&tmHact, aown, cs * 64, row0);
                    ptx::bulk_commit();
                }
                st_pending = true;
            }
            ptx::fence_proxy_async();
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) { if (NCTA == 2 && crank == 1 && kBtDirect) ptx::mbar_arrive_leader(a_ready); else ptx::mbar_arrive(a_ready); }

            // ---------------- phase 3: x_out = x_mid + drop(acc + b2) ; LN1' ----------------
            ptx::mbar_wait(acc_full, af & 1u); ++af;
            ptx::tc_fence_after();
            if (TRAIN) {      // hidden / pre-activation stores drained: the producer may refill the A tile
                ebuf_free();
                if (lane == 0) ptx::mbar_arrive(a_empty);
            }
            rsum = 0.f; rsq = 0.f;
#pragma unroll 1
            for (int jc = 0; jc < 2; ++jc) {
                const int ch = cs + 4 * jc;
                uint32_t r0[32], r1[32];
                ptx::tmem_ld_32x32(tm_acc + (uint32_t)(ch * 32), r0);
                ptx::tmem_ld_32x32(tm_x + (uint32_t)(ch * 32), r1);
                ebuf_free();
                ptx::tc_wait_ld();
                const float* bs = b2 + ch * 32;
                uint4 dw = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    float4 o;
                    o.x = __uint_as_float(r0[c * 4 + 0]) + bs[c * 4 + 0];
                    o.y = __uint_as_float(r0[c * 4 + 1]) + bs[c * 4 + 1];
                    o.z = __uint_as_float(r0[c * 4 + 2]) + bs[c * 4 + 2];
                    o.w = __uint_as_float(r0[c * 4 + 3]) + bs[c * 4 + 3];
                    if (dropping) {       // x_mid + drop(MLP branch)
                        if ((c & 1) == 0) dw = drop_words(p.drop, p.site2, (unsigned long long)(row0 + lane) * (kBtC / 8) + ch * 4 + (c >> 1));
                        const int l0 = (c & 1) * 4;
                        o.x *= drop_mul(p.drop, dw, l0); o.y *= drop_mul(p.drop, dw, l0 + 1);
                        o.z *= drop_mul(p.drop, dw, l0 + 2); o.w *= drop_mul(p.drop, dw, l0 + 3);
                    }
                    o.x += __uint_as_float(r1[c * 4 + 0]); o.y += __uint_as_float(r1[c * 4 + 1]);
                    o.z += __uint_as_float(r1[c * 4 + 2]); o.w += __uint_as_float(r1[c * 4 + 3]);
                    *reinterpret_cast<float4*>(ebuf + sw128_off(lane, c)) = o;
                    r0[c * 4 + 0] = __float_as_uint(o.x); r0[c * 4 + 1] = __float_as_uint(o.y);
                    r0[c * 4 + 2] = __float_as_uint(o.z); r0[c * 4 + 3] = __float_as_uint(o.w);
                    rsum += (o.x + o.y) + (o.z + o.w);
                    rsq += fmaf(o.x, o.x, fmaf(o.y, o.y, fmaf(o.z, o.z, o.w * o.w)));
                }
                if (p.has_ln_out) ptx::tmem_st_32x32(tm_x + (uint32_t)(ch * 32), r0);
                ptx::fence_proxy_async();
                __syncwarp();
                if (lane == 0) { ptx::tma_store_2d(&tmXout, ebuf, ch * 32, row0); ptx::bulk_commit(); }
                st_pending = true;
            }
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) {                                    // the next tile's first GEMM may overwrite the accumulator
                if (NCTA == 2 && crank == 1 && kBtDirect) ptx::mbar_arrive_leader(acc_free); else ptx::mbar_arrive(acc_free);
            }
            if (p.has_ln_out) {
                float mean, rstd;
                row_stats(1, rsum, rsq, mean, rstd);
                ebuf_free();
                ln_kblock(tm_x, mean, rstd, gn, ben, ebuf, lane);
                ptx::fence_proxy_async();
                __syncwarp();
                if (lane == 0) { ptx::tma_store_2d(&tmLnOut, ebuf, cs * 64, row0); ptx::bulk_commit(); }
                st_pending = true;
                // the other warps of the quarter have read this warp's x_out columns out of TMEM: the next tile may overwrite them
                ptx::tc_fence_before();
                named_bar_sync(1 + q, 4 * 32);
                ptx::tc_fence_after();
            }
        }
        if (lane == 0) ptx::bulk_wait_all<0>();
    }
    ptx::tc_fence_before();
    if (NCTA == 2) ptx::cluster_sync_all();     // neither CTA leaves (or frees TMEM) while the pair's MMAs may still touch it
    else __syncthreads();
    if (warp == 1) { if (NCTA == 2) ptx::tmem_dealloc_pair(tmem_base, 512); else ptx::tmem_dealloc(tmem_base, 512); }
}

static cudaError_t bt_set_attrs() {
    static unsigned long long done = 0;
    if (!get_encode_tiled()) return cudaErrorNotSupported;
    if (!attrs_needed(done)) return cudaSuccess;
    cudaError_t e;
#define TANTE_BT_ATTR(MODE, NC) \
    if ((e = cudaFuncSetAttribute(block_tail_kernel<MODE, NC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBtSmem)) != cudaSuccess) return e
    TANTE_BT_ATTR(0, 1); TANTE_BT_ATTR(1, 1); TANTE_BT_ATTR(2, 1); TANTE_BT_ATTR(0, 2); TANTE_BT_ATTR(1, 2); TANTE_BT_ATTR(2, 2);
#undef TANTE_BT_ATTR
    return cudaSuccess;
}

struct BlockTailArgs {
    const __nv_bfloat16* att;                 // [M][256]
    const __nv_bfloat16 *Wo, *W1, *W2;        // [256][256] K-major (nn.Linear layout), bf16
    const float *bo, *g2, *be2, *b1, *b2, *gn, *ben;
    const float* x_in;                        // fp32 residual stream [M][256]
    float* x_out;                             // may alias x_in (inference)
    __nv_bfloat16* ln_out;                    // next layer's LN1 output, null for the last layer
    // training only
    float* x_mid = nullptr;
    __nv_bfloat16 *ln2 = nullptr, *hpre = nullptr, *hact = nullptr;
    DropCfg drop;
    uint32_t site1 = 0, site2 = 0;
};

static cudaError_t launch_block_tail(const BlockTailArgs& a, int M, bool train, int num_sms, cudaStream_t st) {
    if (M <= 0) return cudaSuccess;
    { cudaError_t e = bt_set_attrs(); if (e != cudaSuccess) return e; }
    if (train && (!a.x_mid || !a.ln2 || !a.hpre || !a.hact)) return cudaErrorInvalidValue;
    CUtensorMap tmA, tmWo, tmW1, tmW2, tmXin, tmXmid, tmXout, tmLn2, tmHpre, tmHact, tmLnOut;
    const CUtensorMapDataType BF = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, F32 = CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
    bool ok = make_tmap_2d(&tmA, BF, 2, a.att, M, kBtC, kBtC, 64, 128) &&
              make_tmap_2d(&tmWo, BF, 2, a.Wo, kBtC, kBtC, kBtC, 64, 128) &&
              make_tmap_2d(&tmW1, BF, 2, a.W1, kBtC, kBtC, kBtC, 64, 128) &&
              make_tmap_2d(&tmW2, BF, 2, a.W2, kBtC, kBtC, kBtC, 64, 128) &&
              make_tmap_2d(&tmXin, F32, 4, a.x_in, M, kBtC, kBtC, 32, 32) &&
              make_tmap_2d(&tmXout, F32, 4, a.x_out, M, kBtC, kBtC, 32, 32);
    if (!ok) return cudaErrorInvalidValue;
    tmXmid = tmXout; tmLn2 = tmA; tmHpre = tmA; tmHact = tmA; tmLnOut = tmA;
    if (a.ln_out && !make_tmap_2d(&tmLnOut, BF, 2, a.ln_out, M, kBtC, kBtC, 64, 32)) return cudaErrorInvalidValue;
    if (train) {
        ok = make_tmap_2d(&tmXmid, F32, 4, a.x_mid, M, kBtC, kBtC, 32, 32) &&
             make_tmap_2d(&tmLn2, BF, 2, a.ln2, M, kBtC, kBtC, 64, 32) &&
             make_tmap_2d(&tmHpre, BF, 2, a.hpre, M, kBtC, kBtC, 64, 32) &&
             make_tmap_2d(&tmHact, BF, 2, a.hact, M, kBtC, kBtC, 64, 32);
        if (!ok) return cudaErrorInvalidValue;
    }
    BtParams p;
    p.bo = a.bo; p.g2 = a.g2; p.be2 = a.be2; p.b1 = a.b1; p.b2 = a.b2; p.gn = a.gn; p.ben = a.ben;
    p.M = M; p.has_ln_out = a.ln_out != nullptr;
    p.drop = train ? a.drop : DropCfg(); p.site1 = a.site1; p.site2 = a.site2;
    // CTA pairs once there are enough 256-row units to fill the machine
    const int ncta = M >= 256 * (num_sms / 2) ? 2 : 1;
    const int tiles = (M + 128 * ncta - 1) / (128 * ncta);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(ncta * std::min(tiles, num_sms / ncta))); cfg.blockDim = dim3(kBtThreads); cfg.dynamicSmemBytes = kBtSmem; cfg.stream = st;
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
#define TANTE_BT_LAUNCH(MODE, NC) \
    return cudaLaunchKernelEx(&cfg, block_tail_kernel<MODE, NC>, tmA, tmWo, tmW1, tmW2, tmXin, tmXmid, tmXout, tmLn2, tmHpre, tmHact, tmLnOut, p)
    const int mode = (train && p.drop.p > 0.f) ? 2 : (train ? 1 : 0);
    if (ncta == 2) { if (mode == 2) TANTE_BT_LAUNCH(2, 2); if (mode == 1) TANTE_BT_LAUNCH(1, 2); TANTE_BT_LAUNCH(0, 2); }
    if (mode == 2) TANTE_BT_LAUNCH(2, 1);
    if (mode == 1) TANTE_BT_LAUNCH(1, 1);
    TANTE_BT_LAUNCH(0, 1);
#undef TANTE_BT_LAUNCH
}

}  // namespace tante
