// Fused Taylor head for the bf16 tensor mode (boundary B of SURVEY.md 8(d)):
//   last transposed conv (C1=64 -> D, k0 x k0) of all K orders on mma.sync tensor cores
//   + Horner evaluation of  u(t + i*fi) = u0 + sum_k d_k (i*fi)^k / k!   for i = 1..n_b (per-sample n)
//   + residual u0 + multi-frame emit into (a) the caller's frames (B,n_cap,D,H,W), or (b) the rollout's
//     channels-last history AND the channels-first ring window -- one pass, replacing dec_conv_3
//     (enc_dec_cnn.py:273), the Python Taylor loop + cat (tante.py:165-171), the formatter transpose
//     (datamodule.py:191-192) and the sliding-window cat (r_evaler.py:98).
// Per stage-1 row (one k0 x k0 pixel block): reads K*64 bf16 + 4D fp32 (u0), writes n*4D fp32 (+ ring copy).
// With the 2*64*4D*K FLOP/row on FFMA the kernel would be compute-bound (~8-12 FLOP/B); on mma.sync it is
// bandwidth-bound, which is the point of this variant.
#pragma once
#include "attention_mma.cuh"
#include "kernels_simt.cuh"

namespace tante {

constexpr int kHeadWPitch = 144;       // bytes per weight row (64 bf16 + 16 B pad): conflict-free 32-bit B-fragment loads

// Persistent CTA; tile = ROWS stage-1 rows = NT consecutive latent tokens of ONE latent row (b, hp), i.e. a pixel
// rectangle of P rows x XW = NT*P columns per field.  Per tile:
//   loads    z tile (K x ROWS x 128 B, contiguous in HBM) by cp.async, requested while the previous tile is emitted;
//            the u0 pixels of the tile as 128-bit register loads issued BEFORE phase 1, so they land under the MMAs
//   phase 1  z tile x resident bf16 weights on mma.sync; derivative values (+ bias) scattered into shared memory in
//            PIXEL-MAJOR planes S[k][d][pixel row][pixel column] (the MMA row/column -> pixel map is tile-invariant and
//            lives in registers)
//   phase 2  channels-first emit: thread = 4 consecutive pixels of one (field, pixel row): one 128-bit shared-memory
//            read per order, Horner, one 128-bit store per emitted frame; consecutive threads walk along W, so every
//            store instruction of a warp fills whole lines (frames / ring window / debug derivatives)
//   phase 3  (rollout only) channels-last history, thread = one (pixel, field) with the field fastest, u0 from the
//            copy phase 2 parked in shared memory (the ring slot may be overwritten by then)
// All per-tile quantities (sample, frames to emit, ring position) are CTA-uniform.
// THREADS = 128: one warp per 16-row MMA block (NB <= 2: the 4-field shapes).  THREADS = 256 (wide outputs, e.g. the 11 fields
// of Active Matter): two warps per MMA block, each owning half of the output columns, and half as many emit items per
// thread -- the per-thread accumulators / item registers halve (200 -> < 128 registers), so the same two CTAs per SM the
// shared memory allows for K >= 3 hold 16 warps instead of 8.
template <int KORD, int NB, int ROWS, int THREADS>
__global__ void __launch_bounds__(THREADS, THREADS == 256 ? 2 : 1)
taylor_head_mma_kernel(HeadParams hp, PatchGeom g, long long rows_total, int B) {
    constexpr int MW = ROWS / 16;                 // warps covering the tile's rows
    constexpr int CS = (THREADS / 32) / MW;       // column splits of the MMA phase (1 or 2)
    constexpr int NBH = (NB + CS - 1) / CS;       // 8-column blocks per warp
    constexpr int NJ = (NB * 128 + THREADS - 1) / THREADS;    // emit items per thread (nitems = 64 D <= 128 NB)
    static_assert(THREADS == 32 * MW * CS, "THREADS must be a whole number of column splits");
    extern __shared__ __align__(1024) uint8_t hsm[];
    const int NO = g.k0 * g.k0 * g.D;
    const int P = g.k0 * g.k1 * g.k2;
    const int NT = ROWS / g.R1;                                      // tokens per tile (power of two)
    const int XW = NT * P;                                           // pixel columns per tile (power of two, >= 16)
    const int PS = P * XW + 4;                                       // floats per field plane (+4: bank spread for phase 3)
    const int lXQ = 31 - __clz(XW / 4), lP = 31 - __clz(P), lXW = 31 - __clz(XW);
    uint8_t* sZ = hsm;                                              // [KORD][ROWS][128 B] swizzled
    uint8_t* sW = sZ + KORD * ROWS * 128;                           // [KORD][NB*8][144 B]
    int* sOoff = reinterpret_cast<int*>(sW + KORD * NB * 8 * kHeadWPitch);    // [NB*8] MMA column -> plane offset (-1: padding)
    float* sOb = reinterpret_cast<float*>(sOoff + NB * 8);                      // [KORD][NB*8] bias of the column's field
    float* sS = sOb + KORD * NB * 8;                                            // [KORD (+1: u0, rollout)][D][PS]
    const int tid = threadIdx.x, warp = tid / 32, lane = tid % 32;
    const size_t HW = (size_t)g.H * g.W;
    const int tpr = (g.Wp + NT - 1) / NT;                            // tiles per latent row
    const long long ntiles = (long long)B * g.Hp * tpr;
    const uint32_t zb = (uint32_t)__cvta_generic_to_shared(sZ);
    float* y_out = hp.ptrs ? hp.ptrs->y_out : nullptr;
    float* sU = sS + KORD * g.D * PS;                                // u0 planes (rollout only)

    // the z tile is one contiguous run of 16-byte chunks: chunk i of the tile -> row i/8, swizzled column chunk
    auto load_z = [&](long long tile) {
        const long long bh = tile / tpr;
        const int wpc = (int)(tile % tpr);
        const long long row0 = (bh * g.Wp + (long long)wpc * NT) * g.R1;
        const long long row_end = min(rows_total, (bh + 1) * g.Wp * g.R1);   // rows of the next latent row are not ours
#pragma unroll
        for (int k = 0; k < KORD; ++k) {
            const uint4* zk = reinterpret_cast<const uint4*>(hp.z[k]) + row0 * 8;
#pragma unroll
            for (int j = 0; j < ROWS * 8 / THREADS; ++j) {
                const int i = tid + j * THREADS;
                const int r = i >> 3, c = i & 7;
                const int nbytes = row0 + r < row_end ? 16 : 0;
                const uint32_t dst = zb + (uint32_t)(k * ROWS * 128 + r * 128 + ((c ^ (r & 7)) << 4));
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(zk + (nbytes ? i : 0)), "r"(nbytes) : "memory");
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };

    // ---- once per CTA: first z tile in flight, weights -> bf16 [o][c] ----
    if ((long long)blockIdx.x < ntiles) load_z(blockIdx.x);
#pragma unroll
    for (int k = 0; k < KORD; ++k) {
        for (int i = tid; i < NB * 8 * 64; i += THREADS) {
            const int c = i / (NB * 8), o = i % (NB * 8);            // consecutive threads read consecutive o: coalesced
            const float w = o < NO ? hp.w3[k][(size_t)c * NO + o] : 0.f;
            *reinterpret_cast<__nv_bfloat16*>(sW + (k * NB * 8 + o) * kHeadWPitch + c * 2) = __float2bfloat16_rn(w);
        }
    }

    // ---- tile-invariant maps (registers) ----
    const int gq = lane >> 2, t = lane & 3;
    const int lrow = (lane & 7) + 8 * ((lane >> 3) & 1), lchk = lane >> 4;
    // MMA fragment rows (gq, gq+8 of this warp's m-block) -> pixel (row, column) of the stage-1 pixel block:
    // stage-1 row r1 = ((a*k2 + a')*k1 + b)*k1 + b'  ->  pixel row (a*k1 + b)*k0, pixel column tok*P + (a'*k1 + b')*k0
    int rowbase[2];
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
        const int r = (warp % MW) * 16 + gq + 8 * hh;
        const int tok = r / g.R1;
        int r1 = r % g.R1;
        const int bp = r1 % g.k1; r1 /= g.k1;
        const int bq = r1 % g.k1; r1 /= g.k1;
        const int ap = r1 % g.k2;
        const int a = r1 / g.k2;
        rowbase[hh] = ((a * g.k1 + bq) * g.k0) * XW + tok * P + (ap * g.k1 + bp) * g.k0;
    }
    // MMA fragment columns o = (c*k0 + c')*D + d  ->  plane d, pixel (+c, +c'); bias of field d  (shared-memory tables)
    for (int o = tid; o < NB * 8; o += THREADS) {
        const int d = o % g.D, cp = (o / g.D) % g.k0, c = o / (g.D * g.k0);
        sOoff[o] = o < NO ? d * PS + c * XW + cp : -1;
#pragma unroll
        for (int k = 0; k < KORD; ++k) sOb[k * NB * 8 + o] = o < NO ? hp.b3[k][d] : 0.f;
    }
    // emit items of this thread: item = tid + THREADS*j -> (field, pixel row, 4-pixel run), all tile-invariant:
    // shared-memory float offset inside the planes / global float offset inside a frame
    const int nitems = g.D * P * (XW / 4);
    auto item_soff = [&](int item) {
        return (item >> (lXQ + lP)) * PS + ((item >> lXQ) & (P - 1)) * XW + ((item & ((1 << lXQ) - 1)) << 2);
    };
    auto item_goff = [&](int item) {
        return (size_t)(item >> (lXQ + lP)) * HW + (size_t)(((item >> lXQ) & (P - 1)) * g.W + ((item & ((1 << lXQ) - 1)) << 2));
    };
    // few fields (NB <= 2, e.g. the 4-field shapes): the per-item offsets of this thread stay in registers for all tiles
    constexpr bool kItemRegs = NB <= 2;
    int soffR[kItemRegs ? NJ : 1], goffR[kItemRegs ? NJ : 1], xcolR[kItemRegs ? NJ : 1];
    if (kItemRegs) {
#pragma unroll
        for (int j = 0; j < (kItemRegs ? NJ : 1); ++j) {
            const int item = tid + THREADS * j;
            soffR[j] = item < nitems ? item_soff(item) : -1;
            goffR[j] = (int)item_goff(item);
            xcolR[j] = (item & ((1 << lXQ) - 1)) << 2;
        }
    }

    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long bh = tile / tpr;
        const int wpc = (int)(tile % tpr);
        const int b = (int)(bh / g.Hp), hpp = (int)(bh % g.Hp);
        const int xvalid = min(NT, g.Wp - wpc * NT) * P;             // pixel columns of this tile that exist
        const int bt = hp.act ? hp.act[b] : b;                       // trajectory of ring / counters / history (compaction)
        const int n = hp.n_arr[bt];
        const int fc = hp.fcount ? hp.fcount[bt] : g.T;
        const int f0 = hp.cur ? hp.cur[bt] : 0;
        const size_t pix0 = (size_t)hpp * P * g.W + (size_t)wpc * XW;
        // u0 of this thread's items: in flight during phase 1  (requesting them one tile ahead was measured SLOWER on B200:
        // K = 1, n = 1 on the TRL shape 45.7 -> 63 us -- the extra per-tile index chain costs more than the latency it hides)
        float4 u0r[NJ];
        {
            const float* u0p = head_u0(hp, g, bt, fc, HW) + pix0;
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                u0r[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                const int item = tid + THREADS * j;
                if (kItemRegs) {
                    if (n > 0 && soffR[j] >= 0 && xcolR[j] < xvalid) u0r[j] = *reinterpret_cast<const float4*>(u0p + goffR[j]);
                } else if (n > 0 && item < nitems && ((item & ((1 << lXQ) - 1)) << 2) < xvalid) {
                    u0r[j] = *reinterpret_cast<const float4*>(u0p + item_goff(item));
                }
            }
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();                                             // z tile visible; previous emit is done with S

        // ---- phase 1: last deconv as [16 x 64] x [64 x NB*8] per order, + bias, scattered into the pixel planes ----
        {
            const int mw = warp % MW, nb0 = (warp / MW) * NBH;       // this warp's 16 rows and its first 8-column block
#pragma unroll
            for (int k = 0; k < KORD; ++k) {
                float acc[NBH][4];
#pragma unroll
                for (int nb = 0; nb < NBH; ++nb) acc[nb][0] = acc[nb][1] = acc[nb][2] = acc[nb][3] = 0.f;
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                    uint32_t a[4];
                    const int r = mw * 16 + lrow, c = ks * 2 + lchk;
                    ldsm_x4(zb + (uint32_t)(k * ROWS * 128 + r * 128 + ((c ^ (r & 7)) << 4)), a[0], a[1], a[2], a[3]);
#pragma unroll
                    for (int nb = 0; nb < NBH; ++nb) {
                        if (CS > 1 && nb0 + nb >= NB) continue;
                        const uint8_t* wr = sW + (k * NB * 8 + (nb0 + nb) * 8 + gq) * kHeadWPitch + (ks * 16 + 2 * t) * 2;
                        const uint32_t b0 = *reinterpret_cast<const uint32_t*>(wr);
                        const uint32_t b1 = *reinterpret_cast<const uint32_t*>(wr + 16);
                        mma_bf16_16816(acc[nb], a, b0, b1);
                    }
                }
                float* Sk = sS + k * g.D * PS;
#pragma unroll
                for (int nb = 0; nb < NBH; ++nb) {
                    if (CS > 1 && nb0 + nb >= NB) continue;
                    const int2 oo = *reinterpret_cast<const int2*>(sOoff + (nb0 + nb) * 8 + 2 * t);
                    const float2 ob = *reinterpret_cast<const float2*>(sOb + k * NB * 8 + (nb0 + nb) * 8 + 2 * t);
                    if (oo.x >= 0) {
                        Sk[rowbase[0] + oo.x] = acc[nb][0] + ob.x;
                        Sk[rowbase[1] + oo.x] = acc[nb][2] + ob.x;
                    }
                    if (oo.y >= 0) {
                        Sk[rowbase[0] + oo.y] = acc[nb][1] + ob.y;
                        Sk[rowbase[1] + oo.y] = acc[nb][3] + ob.y;
                    }
                }
            }
        }
        __syncthreads();                                             // S complete, z tile consumed
        if (tile + gridDim.x < ntiles) load_z(tile + gridDim.x);     // overlaps the emit below
        if (n <= 0 && !hp.deriv_dbg) continue;

        // ---- phase 2: channels-first emit ----
        const int cum = hp.cum ? hp.cum[bt] : 0;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const int item = tid + THREADS * j;
            if (kItemRegs) { if (soffR[j] < 0 || xcolR[j] >= xvalid) continue; }
            else if (item >= nitems || ((item & ((1 << lXQ) - 1)) << 2) >= xvalid) continue;
            const int soff = kItemRegs ? soffR[j] : item_soff(item);
            float4 dk[KORD];
#pragma unroll
            for (int k = 0; k < KORD; ++k) dk[k] = *reinterpret_cast<const float4*>(sS + k * g.D * PS + soff);
            const size_t goff = pix0 + (kItemRegs ? (size_t)goffR[j] : item_goff(item));
            if (hp.deriv_dbg) {
#pragma unroll
                for (int k = 0; k < KORD; ++k)
                    *reinterpret_cast<float4*>(hp.deriv_dbg + ((size_t)k * B + b) * g.D * HW + goff) = dk[k];
            }
            if (n <= 0) continue;
            const float4 u0 = u0r[j];
            if (y_out) *reinterpret_cast<float4*>(sU + soff) = u0;
            for (int i = 1; i <= n; ++i) {
                const float dt = (float)i * hp.fi;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int k = KORD; k >= 1; --k) {
                    const float sc = dt / (float)k;
                    v.x = (dk[k - 1].x + v.x) * sc; v.y = (dk[k - 1].y + v.y) * sc;
                    v.z = (dk[k - 1].z + v.z) * sc; v.w = (dk[k - 1].w + v.w) * sc;
                }
                v.x += u0.x; v.y += u0.y; v.z += u0.z; v.w += u0.w;
                if (hp.frames)
                    *reinterpret_cast<float4*>(hp.frames + (size_t)b * (hp.frames_bs ? (size_t)hp.frames_bs : (size_t)hp.n_cap * g.D * HW) +
                                               (size_t)(f0 + i - 1) * g.D * HW + goff) = v;
                if (y_out && i > n - g.T) {
                    const int slot = (fc + i - 1) % g.T;
                    *reinterpret_cast<float4*>(hp.ring_out + (size_t)(bt * g.T + slot) * g.D * HW + goff) = v;
                }
            }
        }
        if (!y_out || n <= 0) continue;
        __syncthreads();                                             // u0 planes visible

        // ---- phase 3: channels-last history, thread = one pixel: its D fields are D consecutive floats of the output
        //      (one 128-bit store when D == 4), adjacent threads = adjacent pixels ----
        const int npix = P * xvalid;
        const bool vec4 = g.D == 4 && (reinterpret_cast<uintptr_t>(y_out) & 15) == 0;
        for (int pi = tid; pi < npix; pi += THREADS) {
            const int hr = pi / xvalid;
            const int x = pi - hr * xvalid;
            const int so = hr * XW + x;
            const size_t pix = pix0 + (size_t)hr * g.W + x;
            for (int i = 1; i <= n; ++i) {
                const int fidx = cum + i - 1;
                if (fidx >= hp.n_roll) break;
                const float dt = (float)i * hp.fi;
                float* yp = y_out + (((size_t)bt * hp.n_roll + fidx) * HW + pix) * g.D;
                if (vec4) {
                    float o[4];
#pragma unroll
                    for (int d = 0; d < 4; ++d) {
                        float v = 0.f;
#pragma unroll
                        for (int k = KORD; k >= 1; --k) v = (sS[(k - 1) * g.D * PS + d * PS + so] + v) * (dt / (float)k);
                        o[d] = v + sU[d * PS + so];
                    }
                    *reinterpret_cast<float4*>(yp) = make_float4(o[0], o[1], o[2], o[3]);
                } else {
                    for (int d = 0; d < g.D; ++d) {
                        float v = 0.f;
#pragma unroll
                        for (int k = KORD; k >= 1; --k) v = (sS[(k - 1) * g.D * PS + d * PS + so] + v) * (dt / (float)k);
                        yp[d] = v + sU[d * PS + so];
                    }
                }
            }
        }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

template <int KORD, int NB>
static cudaError_t launch_head_mma_inst(const HeadParams& hp, const PatchGeom& g, long long rows, int B, int num_sms,
                                        cudaStream_t st) {
    constexpr int ROWS = 64;     // (32-row tiles for the high orders were measured slower: two idle MMA warps, 64-B runs)
    constexpr int THREADS = NB >= 4 ? 256 : 128;
    const int P = g.k0 * g.k1 * g.k2;
    const int NT = ROWS / g.R1;
    const int PS = P * NT * P + 4;
    const size_t smem = (size_t)KORD * ROWS * 128 + (size_t)KORD * NB * 8 * kHeadWPitch + (size_t)(KORD + 1) * NB * 8 * 4 +
                        (size_t)(KORD + (hp.ptrs ? 1 : 0)) * g.D * PS * 4;
    const long long tiles = (long long)B * g.Hp * ((g.Wp + NT - 1) / NT);
    static size_t attr_smem = 0, occ_smem = ~(size_t)0;      // per instantiation
    static int occ_cache = 1, attr_dev = -1;
    int cur_dev = 0;
    if (cudaGetDevice(&cur_dev) != cudaSuccess) { (void)cudaGetLastError(); cur_dev = 0; }
    if (smem > attr_smem || cur_dev != attr_dev) {      // the attribute is per device
        const size_t want = std::max(smem, attr_smem);
        cudaError_t e = cudaFuncSetAttribute(taylor_head_mma_kernel<KORD, NB, ROWS, THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)want);
        if (e != cudaSuccess) return e;
        attr_smem = want;
        attr_dev = cur_dev;
    }
    if (smem != occ_smem) {
        int occ = 1;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, taylor_head_mma_kernel<KORD, NB, ROWS, THREADS>, THREADS, smem) != cudaSuccess) occ = 1;
        occ_cache = std::max(1, occ);
        occ_smem = smem;
    }
    const unsigned blocks = (unsigned)std::min<long long>(tiles, (long long)num_sms * occ_cache);
    taylor_head_mma_kernel<KORD, NB, ROWS, THREADS><<<blocks, THREADS, smem, st>>>(hp, g, rows, B);
    return cudaGetLastError();
}

// Returns false when (K, D) is outside the instantiated set (caller falls back to the FFMA kernel).
static bool launch_head_mma(const HeadParams& hp, const PatchGeom& g, int C1, long long rows, int B, int num_sms,
                            cudaStream_t st, cudaError_t* err) {
    if (C1 != 64 || 32 % g.R1 != 0 || rows % g.R1 != 0 || (g.W & 3)) return false;
    const int NO = g.k0 * g.k0 * g.D;
    const int nb = (NO + 7) / 8;
    const int K = hp.K;
#define TANTE_HEAD(KO, NBv) \
    if (K == KO && nb <= NBv) { *err = launch_head_mma_inst<KO, NBv>(hp, g, rows, B, num_sms, st); return true; }
    TANTE_HEAD(1, 2) TANTE_HEAD(2, 2) TANTE_HEAD(3, 2) TANTE_HEAD(4, 2)
    TANTE_HEAD(1, 4) TANTE_HEAD(2, 4) TANTE_HEAD(3, 4)
    TANTE_HEAD(1, 6) TANTE_HEAD(2, 6) TANTE_HEAD(3, 6) TANTE_HEAD(4, 6)
    TANTE_HEAD(1, 8) TANTE_HEAD(2, 8) TANTE_HEAD(3, 8) TANTE_HEAD(4, 8)
#undef TANTE_HEAD
    return false;
}

}  // namespace tante
