// libtante_b200.so -- C ABI (include/tante_b200.h) over the sm_100a kernels.
// Host-side plan: parameter table (reference state_dict names), packed-weight arena, workspace,
// the per-step launch sequence and the device-resident rollout loop.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/tante_b200.h"
#include "common.cuh"
#include "gemm_simt.cuh"
#include "gemm_tc.cuh"
#include "attention_mma.cuh"
#include "attention_flash.cuh"
#include "propagator_mma.cuh"
#include "propagator_bwd_mma.cuh"
#include "propagator_small.cuh"
#include "head_mma.cuh"
#include "kernels_simt.cuh"
#include "pack.cuh"
#include "backward.cuh"
#include "attention_bwd_mma.cuh"
#include "attention_long_bwd.cuh"
#include "attention_long_bwd_mma.cuh"
#include "wgrad_tc.cuh"
#include "metrics.cuh"
#include "block_tail_tc.cuh"
#include "block_tail2_tc.cuh"
#include "mlp_bwd_tc.cuh"
#include "wide_patch.cuh"
#include "fno.cuh"
#include "channel_axis.cuh"
#include "optimizer.cuh"

using namespace tante;

namespace {

thread_local std::string g_err;

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

#define CK(expr)                                                                                       \
    do {                                                                                               \
        cudaError_t _e = (expr);                                                                       \
        if (_e != cudaSuccess)                                                                         \
            throw Error(TANTE_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e) + " at " + \
                                            __FILE__ + ":" + std::to_string(__LINE__));                \
    } while (0)

#define REQUIRE(cond, msg)                                   \
    do {                                                     \
        if (!(cond)) throw Error(TANTE_ERR_INVALID, (msg));  \
    } while (0)

struct Param {
    std::string name;
    int64_t numel = 0;
    const float* data = nullptr;
    float* grad = nullptr;
    // packing
    int mode = PACK_COPY;
    int d0 = 0, d1 = 0, k = 1;
    int64_t packed_numel = 0;
    int64_t off = -1;  // arena offset (elements)
    // gradient arena entry (packed layout, see unpack_grads_kernel) and position in the flat gradient buffer
    int64_t goff = -1, gnumel = 0, flat_off = 0;
    int gmode = PACK_COPY, gd0 = 0, gd1 = 0, gk = 1;
    bool cplx = false;      // complex64 parameter bound as (re, im) float pairs (SpectralLayer.weight)
};

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    void free() {
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
    }
};

struct LayerPlan {
    char axis;
    int64_t ln1w, ln1b, inw, inb, outw, outb, ln2w, ln2b, m0w, m0b, m2w, m2b;
    int64_t inwT, outwT, m0wT, m2wT;      // [K][N] copies for the input-gradient GEMMs
    // axis 'C' (channel attention, attn_backbone.py:124-130,184-189): the block works on E = expanded_channel features, its MLP
    // on Hc hidden units; cw0 .. cb2 = channel_blocks[j] = Linear(1, E/4), GELU, Linear(E/4, E).  Other axes: E = C, Hc = Hm.
    int E = 0, Hc = 0;
    int64_t cw0 = 0, cb0 = 0, cw2 = 0, cb2 = 0;
};
struct SpecPlan {            // one SpectralLayer (enc_dec_fno.py:184-222)
    int64_t w = 0, w0 = 0, b0 = 0;      // complex weight [Cin][Cout][wm1][wm2] (as float pairs), 1x1 conv [Cout][Cin], bias [Cout]
    int Cin = 0, Cout = 0, wm1 = 0, wm2 = 0;
};
struct OrderPlan {
    std::vector<LayerPlan> layers;
    SpecPlan fs1, fs2;                  // fno decoder: dec_spectral_1 / dec_spectral_2
    int64_t prop[3][4];   // [H,W,T][w0,b0,w2,b2]
    int64_t decw[3], decb[3];   // packed deconv 1,2 (GEMM NK + replicated bias), deconv 3 (KN + raw bias)
    int64_t intw[3], intb[3];
    int64_t mod[8];       // scale{0.w,0.b,2.w,2.b}, shift{...}
    int64_t decwT[2], intwT[2];
    int64_t w3pad = 0;
    int64_t w3nk = 0;        // wide patches: last deconv as a GEMM weight [round_up(k0*k0*D, 64)][C1]
};

}  // namespace

// Saved activations of one training forward (one autograd node): everything the backward reads.
struct OrderTape {
    DevBuf P[3];                        // fp32 inputs of the H / W / T propagators (P[0] only for order 0)
    std::vector<DevBuf> X;              // fp32 residual stream: X[0] after the propagators, X[2i+1] mid, X[2i+2] out of layer i
    std::vector<DevBuf> ln1, qkv, att, ln2, hpre, hact;
    DevBuf dl, d32, dmod, i1, i2, rt, film, z1pre, z1act, z2pre, z2act;
    DevBuf f0pre, f0act;                // fno decoder: [B][H][W][C/8] grid behind dec_conv_2 (the stages above reuse z1* = [B][H1][W1][C/2], z2* = [B][H1][W1][C/4])
};
struct Tape {
    DevBuf cols, a1pre, a1act, a2pre, a2act, v, n_arr;
    DevBuf cur;                         // per-sample cursor mode: the cursor this call saw (its backward addresses the same frames)
    DevBuf f0pre, f0act;                // fno encoder: [B*T][H][W][C/8] grid behind enc_spectral_1 (a1* = [..][H1][W1][C/4], a2* = [..][H1][W1][C/2])
    std::vector<OrderTape> ord;
    int B = 0;          // allocated batch
    int B_used = 0;     // batch of the taped forward
    float out_T = 1.f;
    int n_cap = 0;      // frames per sample the taped call could emit
    bool hist = false;  // taped by tante_train_forward_hist
    bool valid = false;
    DropCfg drop;       // dropout of this taped call (p = 0: none); the backward regenerates the forward's masks from it
};

struct tante_handle_s {
    tante_config_t cfg{};
    int device = 0;
    int C = 0, C1 = 0, C2 = 0, Hp = 0, Wp = 0, L = 0, T = 0, D = 0, K = 0, HD = 0;
    int Hm = 0;                          // hidden width of the block MLP = int(embed_dim * mlp_ratio) (attn_backbone.py:52)
    PatchGeom geom{};
    std::vector<Param> params;
    std::map<std::string, int> pindex;
    std::vector<OrderPlan> orders;
    int64_t enc_w[3], enc_b[3];
    int64_t tenc[8];
    int64_t t_emb = 0, s_emb = 0;
    int64_t film_t_off = 0;    // derived: t_encode scale/shift table [T][2][C]
    int64_t tseq_off = 0;      // derived: t_seq [T]
    int64_t arena_elems = 0;
    DevBuf arena, arena_bf16, descs;
    bool packed = false;
    DevBuf icols;                       // tensor mode: im2col'ed input patches of the first conv, [B*T*L*R1][64] bf16
    DevBuf enc_cache;                   // rollout: encoder output per ring slot, fp32 [B*T*L][C]
    DevBuf enc_state;                   // rollout: [8] count, [B*T] list, [B*T] map
    bool use_enc_cache = true;          // TANTE_ENC_CACHE=0 re-encodes the whole window every call
    bool axes_ok = true;                // Hp, Wp, T <= 64 (what the axial kernels cover)
    bool long_axes = false;             // an L / Y / A layer or an axis longer than 64 tokens: inference / rollout only
    bool chan = false;                  // an axis-'C' layer (channel_axis.cuh): inference / rollout only
    int chanE = 0, chanHc = 0, chan_tokens = 0;   // widest E / hidden of the 'C' layers; latent tokens per chunk of the channel pass
    DevBuf cx, cln, cqkv, catt, chid;   // channel pass scratch: fp32 stream [rows][E], LN / QKV / attention / hidden, rows = chan_tokens * C
    bool fno = false;                   // enc_dec_type = 'fno' (fno.cuh): spectral layers between two patch stages; inference / rollout
    int fp0 = 0, fp1 = 0;               // fno patch kernels (enc_dec_fno.py:39-46)
    SpecPlan fes1, fes2;                // fno encoder: enc_spectral_1 / enc_spectral_2
    DevBuf ftw, fA, fB, fg0, fg1, fg2;  // fno: twiddle tables, complex scratch x2, channels-last stage grids
    DevBuf fC, fD, fgr0, fgr1, fgr2;    // fno training: two more complex scratch buffers, gradient grids of the three stages
    size_t f_ca = 0;                    // complex elements per scratch buffer (tante_reserve)
    bool wide = false;                  // patch_scale >= 16 or overlap_ratio != 0: natural-order stages (wide_patch.cuh)
    bool overlap = false;               // overlap_ratio != 0: some stage's stride < its kernel (strided windows + pooling, overlap-add deconvs)
    int st[3] = {0, 0, 0};              // stride of the three patch stages (== kernel size without overlap)
    DevBuf cgrid;                       // overlap: conv grid of a stage before the adaptive average pooling
    int K1pad = 0, NOpad = 0;           // wide: first-conv reduction / last-deconv output width rounded up to 64
    int64_t enc_w1wide = 0;             // wide: first conv weight [C1][K1pad]
    DevBuf wbuf, dfield;                // wide: patch / sub-pixel matrix scratch; decoded derivative fields [K][B][D][H][W]
    float drop_p = 0.f;                 // tante_set_dropout: applies to the NEXT tante_train_forward calls
    unsigned long long drop_seed = 0;
    bool fuse_mlp_bwd = true;           // tensor mode: MLP input-gradient chain as ONE kernel (TANTE_FUSE_MLP_BWD=0: GEMM + elementwise + GEMM)
    bool no_switch = false;             // SWITCH conditional nodes unavailable on this driver: rollouts run without compaction
    bool fuse_tail = true;              // tensor mode: out-proj + LN2 + MLP + LN1' of a block as ONE kernel (TANTE_FUSE_TAIL=0: three GEMMs)

    // workspace
    int max_batch = 0, max_roll = 0;
    DevBuf x, ln, qkv, att, hid, a1, a2, d32, dmod, i1, i2, z1, rt, Rt, nbuf, filmbuf, ring, state, dbg_in;
    std::vector<DevBuf> z2;
    int64_t ws_bytes = 0;
    int* h_flag = nullptr;      // pinned: remaining-samples flag (ring of 2)
    cudaEvent_t ev[2] = {nullptr, nullptr};
    int64_t launches = 0;
    bool debug = false;
    int last_B = 0;
    int num_sms = 148;
    // rollout graphs: key -> instantiated graph (WHILE node whose body is one model step)
    struct RollGraph { cudaGraph_t graph = nullptr; cudaGraphExec_t exec = nullptr; bool while_node = false; int64_t launches_per_step = 0; };
    std::map<std::string, RollGraph> graphs;
    cudaStream_t cap_stream = nullptr;
    int rollout_mode = 2;       // 0 = eager launches, 1 = one graph per step + host loop, 2 = device WHILE graph
    cudaGraphConditionalHandle cond_handle = 0;
    int use_cond = 0;
    cudaGraphConditionalHandle sw_handle = 0;   // SWITCH node of the compaction buckets
    int last_graph_steps = 0;
    // live GEMM timing (tante_profile)
    bool prof_on = false;
    std::vector<cudaEvent_t> prof_ev;
    size_t prof_used = 0;
    double prof_flops = 0;
    struct ProfRec { int cls; double flops, bytes; };
    std::vector<ProfRec> prof_rec;      // one per bracketed launch (same order as the event pairs)
    // ---- training ----
    int64_t enc_wT[3] = {0, 0, 0};
    int64_t enc_w1pad = 0;                     // [C1][64]: first conv weight zero-padded along K (im2col GEMM)
    int64_t zero_off = 0;                      // 4096 zeros (bias of the input-gradient GEMMs)
    int64_t garena_elems = 0, flat_elems = 0;
    std::vector<TransDesc> tdescs;
    std::vector<char> desc_cache;
    std::map<int64_t, int64_t> goff_of;        // arena offset of a parameter -> gradient arena offset
    DevBuf garena, tdesc_dev, udesc_dev;
    std::vector<std::unique_ptr<Tape>> tapes;
    int bw_batch = 0;
    DevBuf dxs, dxb, g1, g2, gq, ga1, cols, hz, hG, hz1, hd, hi1, hi2, dfilm, dcond, att_stats;
    int chanb_tokens = 0;               // latent tokens per chunk of the channel-axis backward
    DevBuf cb_x0, cb_xm, cb_gx, cb_ln1, cb_qkv, cb_att, cb_ln2, cb_hpre, cb_hact, cb_gxb, cb_g1, cb_g2, cb_gq, cb_hh, cb_stats;
    DevBuf kscratch;                    // fp32 accumulator of the split-K input-gradient GEMMs (K > 1024 in the tensor mode)
    // ---- optimizer tail (optimizer.cuh) ----
    DevBuf opt_segs, opt_norm;                 // parameter segments of the flat gradient; f64 sum of squares
    std::vector<char> opt_seg_cache;
    void* nccl_comm = nullptr;                 // tante_comm_init
    int nccl_nranks = 1;
};

namespace {

int64_t add_param(tante_handle_s* h, const std::string& name, std::vector<int64_t> shape, int mode = PACK_COPY,
                  int d0 = 0, int d1 = 0, int k = 1) {
    Param p;
    p.name = name;
    p.numel = 1;
    for (auto s : shape) p.numel *= s;
    p.mode = mode;
    p.d0 = d0;
    p.d1 = d1;
    p.k = k;
    p.packed_numel = (mode == PACK_BIAS_REP) ? (int64_t)d0 * k * k : p.numel;
    p.off = h->arena_elems;
    h->arena_elems += (p.packed_numel + 63) / 64 * 64;   // 256-byte aligned tensors
    p.goff = h->garena_elems;
    p.gnumel = p.packed_numel; p.gmode = mode; p.gd0 = d0; p.gd1 = d1; p.gk = k;
    h->garena_elems += (p.gnumel + 63) / 64 * 64;
    p.flat_off = h->flat_elems;
    h->flat_elems += p.numel;
    h->goff_of[p.off] = p.goff;
    h->pindex[name] = (int)h->params.size();
    h->params.push_back(p);
    return p.off;
}

// derived copy of the packed [rows][cols] GEMM weight at `src` (filled by transpose_packed_kernel at pack time):
// transposed [cols][rows] by default; dst_rows / dst_ld > 0 zero-pad the destination.
int64_t add_trans(tante_handle_s* h, int64_t src, int rows, int cols, int transpose = 1, int dst_rows = 0, int dst_ld = 0) {
    TransDesc d;
    d.src_off = src; d.dst_off = h->arena_elems; d.rows = rows; d.cols = cols; d.transpose = transpose;
    d.dst_rows = dst_rows > 0 ? dst_rows : (transpose ? cols : rows);
    d.dst_ld = dst_ld > 0 ? dst_ld : (transpose ? rows : cols);
    h->arena_elems += ((int64_t)d.dst_rows * d.dst_ld + 63) / 64 * 64;
    h->tdescs.push_back(d);
    return d.dst_off;
}

void patch_kernels(int P, int k[3]) {
    switch (P) {   // reference enc_dec_cnn.py:39-46
        case 8: k[0] = 2; k[1] = 2; k[2] = 2; break;
        case 4: k[0] = 2; k[1] = 2; k[2] = 1; break;
        case 2: k[0] = 2; k[1] = 1; k[2] = 1; break;
        case 16: k[0] = 4; k[1] = 2; k[2] = 2; break;      // 4x4 / pad-1 stages: wide_patch.cuh (inference / rollout)
        case 32: k[0] = 4; k[1] = 4; k[2] = 2; break;
        case 64: k[0] = 4; k[1] = 4; k[2] = 4; break;
        default: throw Error(TANTE_ERR_INVALID, "KeyError: patch_scale not in Patch_map");
    }
}

void build_plan(tante_handle_s* h) {
    const tante_config_t& c = h->cfg;
    REQUIRE(c.in_T >= 1 && c.in_T <= 64, "in_T out of range");
    REQUIRE(c.taylor_order >= 1 && c.taylor_order <= 4, "taylor_order must be in 1..4");
    REQUIRE(c.embed_dim == 256 || c.embed_dim == 512, "embed_dim must be 256 or 512 (C/4 and the interprator widths must stay multiples of 64)");
    REQUIRE(c.n_head > 0 && c.embed_dim % c.n_head == 0, "embed_dim must be divisible by n_head");
    const int hd = c.embed_dim / c.n_head;
    REQUIRE(hd == 16 || hd == 32 || hd == 64, "head_dim must be 16, 32 or 64");
    REQUIRE(c.n_fields >= 1 && c.n_fields <= 16, "n_fields must be in 1..16");
    REQUIRE(c.precision == TANTE_PREC_FP32 || c.precision == TANTE_PREC_BF16, "unknown precision");
    int k[3];
    h->fno = c.enc_dec_fno != 0;
    if (h->fno) {
        // enc_dec_fno.py:39-46: two patch stages (p0 at full resolution, p1 after the second spectral layer)
        switch (c.patch_scale) {
            case 2: h->fp0 = 2; h->fp1 = 1; break;
            case 4: h->fp0 = 2; h->fp1 = 2; break;
            case 8: h->fp0 = 4; h->fp1 = 2; break;
            case 16: h->fp0 = 4; h->fp1 = 4; break;
            case 32: h->fp0 = 8; h->fp1 = 4; break;      // 8x8 stages: windows shifted by 3, transposed convs resized from 8h - 6
            case 64: h->fp0 = 8; h->fp1 = 8; break;
            default: throw Error(TANTE_ERR_INVALID, "KeyError: patch_scale not in Patch_map");
        }
        k[0] = h->fp0; k[1] = h->fp1; k[2] = 1;      // geometry bookkeeping only (rows per token of the two stage grids)
        const int H1 = c.H / h->fp0, W1 = c.W / h->fp0;
        REQUIRE(c.modes1 >= h->fp0 && c.modes2 >= h->fp0, "fno: modes1 / modes2 must be >= the first patch kernel");
        REQUIRE(2 * c.modes1 <= c.H && c.modes2 <= c.W / 2 && 2 * (c.modes1 / h->fp0) <= H1 && (c.modes2 / h->fp0) <= W1 / 2,
                "fno: the kept modes must fit the grid (2 * modes1 <= H, modes2 <= W / 2 at both resolutions)");
    } else {
        patch_kernels(c.patch_scale, k);
    }
    REQUIRE(c.H % c.patch_scale == 0 && c.W % c.patch_scale == 0, "H and W must be divisible by patch_scale");
    for (int i = 0; i < 3; ++i) {
        h->st[i] = c.stride[i] > 0 ? c.stride[i] : k[i];
        REQUIRE(h->st[i] >= 1 && h->st[i] <= k[i], "stride of a patch stage must be in 1..kernel size");
        if (h->st[i] != k[i]) h->overlap = true;
    }
    h->wide = c.patch_scale >= 16 || h->fno || h->overlap;
    h->K1pad = (k[0] * k[0] * c.n_fields + 63) / 64 * 64;
    h->NOpad = h->K1pad;
    if (h->wide) h->use_enc_cache = false;
    h->C = c.embed_dim; h->C1 = h->C / 4; h->C2 = h->C / 2;
    h->Hm = c.mlp_hidden > 0 ? c.mlp_hidden : h->C;
    REQUIRE(h->Hm % 64 == 0 && h->Hm >= 64 && h->Hm <= 1024, "MLP hidden width (embed_dim * mlp_ratio) must be a multiple of 64 in 64..1024");
    h->Hp = c.H / c.patch_scale; h->Wp = c.W / c.patch_scale; h->L = h->Hp * h->Wp;
    h->T = c.in_T; h->D = c.n_fields; h->K = c.taylor_order; h->HD = hd;
    // checked by the model entry points, not here: the head microbenchmark (tante_bench_head) needs no backbone
    h->axes_ok = h->Hp <= 96 && h->Wp <= 96 && h->T <= 64;      // propagator kernels: the S x S matrices + slab fit in shared memory
    if (h->Hp > 64 || h->Wp > 64) h->long_axes = true;
    PatchGeom& g = h->geom;
    g.k0 = k[0]; g.k1 = k[1]; g.k2 = k[2];
    g.D = h->D; g.H = c.H; g.W = c.W; g.Hp = h->Hp; g.Wp = h->Wp; g.T = h->T;
    g.R1 = (k[1] * k[2]) * (k[1] * k[2]);
    g.R2 = k[2] * k[2];
    const int C = h->C, C1 = h->C1, C2 = h->C2, D = h->D, T = h->T;

    h->t_emb = add_param(h, "t_emb", {1, T, C});
    h->s_emb = add_param(h, "s_emb", {1, h->Hp, h->Wp, C});
    auto add_spec = [&](const std::string& pre, int Cin, int Cout, int wm1, int wm2) {
        SpecPlan sp;
        sp.Cin = Cin; sp.Cout = Cout; sp.wm1 = wm1; sp.wm2 = wm2;
        sp.w = add_param(h, pre + "weight", {Cin, Cout, wm1, wm2, 2});        // cfloat viewed as (..., 2) floats
        h->params.back().cplx = true;
        sp.w0 = add_param(h, pre + "w0.weight", {Cout, Cin, 1, 1});
        sp.b0 = add_param(h, pre + "w0.bias", {Cout});
        return sp;
    };
    const int ech[4] = {D, C1, C2, C};
    if (h->fno) {
        const int p0 = h->fp0, p1 = h->fp1, C8 = C / 8;
        h->fes1 = add_spec("encoder.enc_spectral_1.", D, C8, c.modes1, c.modes2);
        h->enc_w[0] = add_param(h, "encoder.enc_conv_1.conv.weight", {C1, C8, p0, p0}, PACK_CONV, C1, C8, p0);
        h->enc_b[0] = add_param(h, "encoder.enc_conv_1.conv.bias", {C1});
        h->fes2 = add_spec("encoder.enc_spectral_2.", C1, C2, c.modes1 / p0, c.modes2 / p0);
        h->enc_w[1] = add_param(h, "encoder.enc_conv_2.conv.weight", {C, C2, p1, p1}, PACK_CONV, C, C2, p1);
        h->enc_b[1] = add_param(h, "encoder.enc_conv_2.conv.bias", {C});
        h->enc_wT[0] = add_trans(h, h->enc_w[0], C1, C8 * p0 * p0);      // [K][N] copies for the input-gradient GEMMs (training)
        h->enc_wT[1] = add_trans(h, h->enc_w[1], C, C2 * p1 * p1);
    }
    for (int i = 0; i < 3 && !h->fno; ++i) {
        const std::string p = "encoder.enc_conv_" + std::to_string(i + 1) + ".conv.";
        h->enc_w[i] = add_param(h, p + "weight", {ech[i + 1], ech[i], k[i], k[i]}, PACK_CONV, ech[i + 1], ech[i], k[i]);
        h->enc_b[i] = add_param(h, p + "bias", {ech[i + 1]});
        if (i > 0) h->enc_wT[i] = add_trans(h, h->enc_w[i], ech[i + 1], ech[i] * k[i] * k[i]);
        else if (h->wide) {
            h->enc_w1wide = add_trans(h, h->enc_w[0], ech[1], k[0] * k[0] * D, 0, ech[1], h->K1pad);   // [C1][K1pad]
            h->enc_wT[0] = add_trans(h, h->enc_w[0], ech[1], k[0] * k[0] * D, 1, h->K1pad, ech[1]);    // [K1pad][C1] (input gradient)
        } else {
            REQUIRE(k[0] * k[0] * D <= kHeadPad, "n_fields too large for the padded first-conv backward (k0*k0*D <= 64)");
            h->enc_wT[0] = add_trans(h, h->enc_w[0], ech[1], k[0] * k[0] * D, 1, kHeadPad, ech[1]);   // [64 (K1 pad)][C1]
            h->enc_w1pad = add_trans(h, h->enc_w[0], ech[1], k[0] * k[0] * D, 0, ech[1], kHeadPad);  // [C1][64]
        }
    }
    const char* fn[2] = {"condition_to_scale", "condition_to_shift"};
    auto add_film = [&](const std::string& pre, int64_t* out) {
        for (int s = 0; s < 2; ++s) {
            const std::string p = pre + fn[s];
            out[s * 4 + 0] = add_param(h, p + ".0.weight", {C / 2, 1});
            out[s * 4 + 1] = add_param(h, p + ".0.bias", {C / 2});
            out[s * 4 + 2] = add_param(h, p + ".2.weight", {C, C / 2});
            out[s * 4 + 3] = add_param(h, p + ".2.bias", {C});
        }
    };
    add_film("t_encode.", h->tenc);
    h->orders.resize(h->K);
    for (int o = 0; o < h->K; ++o) {
        OrderPlan& op = h->orders[o];
        const int nl = c.n_layers[o];
        REQUIRE(nl >= 1 && nl <= TANTE_MAX_LAYERS, "ValueError: Invalid block: empty segment.");
        const std::string bp = "blocks." + std::to_string(o) + ".";
        int n_chan = 0;
        for (int i = 0; i < nl; ++i) {
            LayerPlan lp;
            lp.axis = c.axes[o][i];
            // T / H / W: the axial layers of configs/tante.yaml; L / Y / A (attn_backbone.py:164-182): composite sequences;
            // C (:184-189): channel attention behind a 1 -> expanded_channel lift.  L / Y / A / C: forward / rollout only.
            // 'X' cannot be reached through TANTE's own validation (tante.py:76).
            REQUIRE(lp.axis == 'T' || lp.axis == 'H' || lp.axis == 'W' || lp.axis == 'L' || lp.axis == 'Y' || lp.axis == 'A' ||
                        lp.axis == 'C',
                    std::string("attention axis '") + lp.axis + "' is not implemented (supported: T, H, W, L, Y, A, C)");
            if (lp.axis == 'L' || lp.axis == 'Y' || lp.axis == 'A' || lp.axis == 'C') h->long_axes = true;
            const std::string p = bp + "blocks." + std::to_string(i) + ".";
            int Cb = C, Hb = h->Hm;
            if (lp.axis == 'C') {
                Cb = c.expanded_channel > 0 ? c.expanded_channel : 128;
                Hb = c.mlp_hidden_c > 0 ? c.mlp_hidden_c : Cb;
                REQUIRE(Cb % 64 == 0 && Cb >= 64 && Cb <= 256, "expanded_channel must be a multiple of 64 in 64..256");
                REQUIRE(Cb % c.n_head == 0 && (Cb / c.n_head == 16 || Cb / c.n_head == 32 || Cb / c.n_head == 64),
                        "expanded_channel / n_head must be 16, 32 or 64");
                REQUIRE(Hb % 64 == 0 && Hb >= 64 && Hb <= 1024, "int(expanded_channel * mlp_ratio) must be a multiple of 64 in 64..1024");
                const std::string q = bp + "channel_blocks." + std::to_string(n_chan++) + ".";
                lp.cw0 = add_param(h, q + "0.weight", {Cb / 4, 1});
                lp.cb0 = add_param(h, q + "0.bias", {Cb / 4});
                lp.cw2 = add_param(h, q + "2.weight", {Cb, Cb / 4});
                lp.cb2 = add_param(h, q + "2.bias", {Cb});
                h->chan = true;
                h->chanE = std::max(h->chanE, Cb);
                h->chanHc = std::max(h->chanHc, Hb);
            }
            lp.E = Cb; lp.Hc = Hb;
            lp.ln1w = add_param(h, p + "ln1.weight", {Cb});
            lp.ln1b = add_param(h, p + "ln1.bias", {Cb});
            lp.inw = add_param(h, p + "attn.in_proj_weight", {3 * Cb, Cb});
            lp.inb = add_param(h, p + "attn.in_proj_bias", {3 * Cb});
            lp.outw = add_param(h, p + "attn.out_proj.weight", {Cb, Cb});
            lp.outb = add_param(h, p + "attn.out_proj.bias", {Cb});
            lp.ln2w = add_param(h, p + "ln2.weight", {Cb});
            lp.ln2b = add_param(h, p + "ln2.bias", {Cb});
            lp.m0w = add_param(h, p + "mlp.0.weight", {Hb, Cb});      // hidden = int(C * mlp_ratio) (attn_backbone.py:52-56)
            lp.m0b = add_param(h, p + "mlp.0.bias", {Hb});
            lp.m2w = add_param(h, p + "mlp.2.weight", {Cb, Hb});
            lp.m2b = add_param(h, p + "mlp.2.bias", {Cb});
            lp.inwT = add_trans(h, lp.inw, 3 * Cb, Cb);
            lp.outwT = add_trans(h, lp.outw, Cb, Cb);
            lp.m0wT = add_trans(h, lp.m0w, Hb, Cb);
            lp.m2wT = add_trans(h, lp.m2w, Cb, Hb);
            op.layers.push_back(lp);
        }
        const char* pn[3] = {"vertical", "horizontal", "temporal"};
        const int plen[3] = {h->Hp, h->Wp, T};
        for (int a = 0; a < 3; ++a) {
            const std::string p = bp + pn[a] + "_propagator.";
            op.prop[a][0] = add_param(h, p + "0.weight", {plen[a], plen[a]});
            op.prop[a][1] = add_param(h, p + "0.bias", {plen[a]});
            op.prop[a][2] = add_param(h, p + "2.weight", {plen[a], plen[a]});
            op.prop[a][3] = add_param(h, p + "2.bias", {plen[a]});
        }
        const int dch[4] = {C, C2, C1, D};
        if (h->fno) {
            const int p0 = h->fp0, p1 = h->fp1, C8 = C / 8;
            const std::string p = "decoders." + std::to_string(o) + ".";
            op.decw[0] = add_param(h, p + "dec_conv_1.deconv.weight", {C, C2, p1, p1}, PACK_DECONV_NK, C, C2, p1);
            op.decb[0] = add_param(h, p + "dec_conv_1.deconv.bias", {C2}, PACK_BIAS_REP, C2, 0, p1);
            op.fs1 = add_spec(p + "dec_spectral_1.", C2, C1, c.modes1 / p0, c.modes2 / p0);
            op.decw[1] = add_param(h, p + "dec_conv_2.deconv.weight", {C1, C8, p0, p0}, PACK_DECONV_NK, C1, C8, p0);
            op.decb[1] = add_param(h, p + "dec_conv_2.deconv.bias", {C8}, PACK_BIAS_REP, C8, 0, p0);
            op.fs2 = add_spec(p + "dec_spectral_2.", C8, D, c.modes1, c.modes2);
            op.decwT[0] = add_trans(h, op.decw[0], p1 * p1 * C2, C);
            op.decwT[1] = add_trans(h, op.decw[1], p0 * p0 * C8, C1);
        }
        for (int i = 0; i < 3 && !h->fno; ++i) {
            const int kk = k[2 - i];
            const std::string p = "decoders." + std::to_string(o) + ".dec_conv_" + std::to_string(i + 1) + ".deconv.";
            op.decw[i] = add_param(h, p + "weight", {dch[i], dch[i + 1], kk, kk},
                                   i < 2 ? PACK_DECONV_NK : PACK_DECONV_KN, dch[i], dch[i + 1], kk);
            if (i < 2) {
                op.decb[i] = add_param(h, p + "bias", {dch[i + 1]}, PACK_BIAS_REP, dch[i + 1], 0, kk);
                op.decwT[i] = add_trans(h, op.decw[i], kk * kk * dch[i + 1], dch[i]);
            } else {
                op.decb[i] = add_param(h, p + "bias", {dch[i + 1]});
                // its gradient arrives as column sums over the k0*k0*D outputs of the fused head: folded at unpack
                Param& bp3 = h->params.back();
                h->garena_elems -= (bp3.gnumel + 63) / 64 * 64;
                bp3.gnumel = (int64_t)kk * kk * dch[i + 1]; bp3.gmode = PACK_BIAS_REP; bp3.gd0 = dch[i + 1]; bp3.gk = kk;
                h->garena_elems += (bp3.gnumel + 63) / 64 * 64;
                if (h->wide) {
                    op.w3nk = add_trans(h, op.decw[i], dch[i], kk * kk * dch[i + 1], 1, h->NOpad, dch[i]);   // [NOpad][C1]
                    op.w3pad = add_trans(h, op.decw[i], dch[i], kk * kk * dch[i + 1], 0, dch[i], h->NOpad);  // [C1][NOpad] (dz = G * W3^T)
                } else {
                    // [C1][64]: the packed [C1][k0*k0*D] weight zero-padded along its columns (dz = G * W3^T as a GEMM)
                    op.w3pad = add_trans(h, op.decw[i], dch[i], kk * kk * dch[i + 1], 0, dch[i], kHeadPad);
                }
            }
        }
        if (!c.deg) {
            const std::string p = "interprators." + std::to_string(o) + ".interprete.";
            const int ich[4] = {C, C / 2, C / 4, 1};
            for (int i = 0; i < 3; ++i) {
                op.intw[i] = add_param(h, p + std::to_string(2 * i) + ".weight", {ich[i + 1], ich[i]});
                op.intb[i] = add_param(h, p + std::to_string(2 * i) + ".bias", {ich[i + 1]});
                if (i < 2) op.intwT[i] = add_trans(h, op.intw[i], ich[i + 1], ich[i]);
            }
            add_film("modifiers." + std::to_string(o) + ".", op.mod);
        }
    }
    // flat gradient layout: the complex parameters first, so that each starts at an EVEN element offset and the host can view
    // its slice of the flat fp32 buffer as complex64 (torch.view_as_complex); the rest in tante_param order
    {
        int64_t off = 0;
        for (Param& p : h->params) if (p.cplx) { p.flat_off = off; off += p.numel; }
        for (Param& p : h->params) if (!p.cplx) { p.flat_off = off; off += p.numel; }
    }
    // derived tensors
    h->film_t_off = h->arena_elems; h->arena_elems += (int64_t)T * 2 * C;
    h->tseq_off = h->arena_elems;   h->arena_elems += 64;
    h->zero_off = h->arena_elems;   h->arena_elems += 8192;
}

void destroy_graphs(tante_handle_s* h);
inline float* AF(tante_handle_s* h, int64_t off) { return reinterpret_cast<float*>(h->arena.p) + off; }
// gradient-arena pointer of the parameter whose ARENA offset is `off` (plans store arena offsets)
inline float* GA(tante_handle_s* h, int64_t off) {
    auto it = h->goff_of.find(off);
    if (it == h->goff_of.end()) throw Error(TANTE_ERR_STATE, "no gradient entry for arena offset " + std::to_string(off));
    return reinterpret_cast<float*>(h->garena.p) + it->second;
}

void dev_alloc(tante_handle_s* h, DevBuf& b, size_t bytes) {
    bytes = (bytes + 255) / 256 * 256;
    if (b.bytes >= bytes) return;
    if (b.p) { h->ws_bytes -= b.bytes; b.free(); }
    cudaError_t e = cudaMalloc(&b.p, bytes);
    if (e != cudaSuccess) throw Error(TANTE_ERR_NOMEM, std::string("cudaMalloc failed: ") + cudaGetErrorString(e));
    b.bytes = bytes;
    h->ws_bytes += bytes;
}

struct StepIO {
    const float* input = nullptr;   // window / ring (B,T,D,H,W)
    const int* fcount = nullptr;
    float* frames = nullptr; int n_cap = 1;
    float* R_t = nullptr; int* n_dev = nullptr;
    float* ring_out = nullptr; int n_roll = 0;
    bool rollout = false;
    int per_sample = 0;
    float out_T = 1.f;
};

RolloutState make_state(tante_handle_s* h, int B, int n_roll) {
    RolloutState rs;
    int* s = reinterpret_cast<int*>(h->state.p);
    const int mb = h->max_batch;
    rs.cum = s; rs.fcount = s + mb; rs.steps = s + 2 * mb; rs.n_cur = s + 3 * mb; rs.remaining = s + 4 * mb;
    rs.iter = s + 4 * mb + 1;
    rs.ptrs = reinterpret_cast<const RolloutPtrs*>(s + 4 * mb + 8);   // 32-byte aligned slot after the counters
    rs.n_roll = n_roll; rs.max_steps = n_roll;
    rs.T = h->T;
    rs.act = nullptr; rs.n_active = s + 4 * mb + 2; rs.B_full = B; rs.n_buckets = 0; rs.sw = 0;
    for (int& v : rs.bucket_sz) v = 0;
    rs.enc_count = nullptr; rs.enc_list = nullptr; rs.enc_map = nullptr;
    if (h->enc_cache.p && h->use_enc_cache) {
        int* e = reinterpret_cast<int*>(h->enc_state.p);
        rs.enc_count = e; rs.enc_list = e + 8; rs.enc_map = e + 8 + (size_t)mb * h->T;
    }
    return rs;
}

inline __nv_bfloat16* AH(tante_handle_s* h, int64_t off) { return reinterpret_cast<__nv_bfloat16*>(h->arena_bf16.p) + off; }

// C = epi(A * W^T): fp32 mode -> FFMA GEMM; bf16 mode -> tcgen05 GEMM (C is fp32 when out_f32, else bf16).
template <typename TA>
void gemm(tante_handle_s* h, int epi, const TA* A, int lda, int64_t w_off, void* Cout, int ldc, bool out_f32, int M, int N,
          int K, const EpiParams& ep, cudaStream_t st, int ldw = 0);

struct ProfScope {
    tante_handle_s* h; cudaStream_t st; bool on;
    // cls: 0 = GEMM with a plain (bf16 / activation) epilogue: tensor-bound; 1 = GEMM with an fp32 residual / LayerNorm /
    // embedding epilogue: HBM-bound; 2 = weight-gradient GEMM: HBM-bound.  bytes = algorithmic HBM bytes of the launch.
    ProfScope(tante_handle_s* h_, cudaStream_t st_, double flops, int cls = 0, double bytes = 0) : h(h_), st(st_), on(h_->prof_on) {
        if (!on) return;
        h->prof_rec.push_back({cls, flops, bytes});
        if (h->prof_used + 2 > h->prof_ev.size()) {
            for (int i = 0; i < 2; ++i) { cudaEvent_t e; CK(cudaEventCreate(&e)); h->prof_ev.push_back(e); }
        }
        CK(cudaEventRecord(h->prof_ev[h->prof_used], st));
        h->prof_flops += flops;
    }
    ~ProfScope() {
        if (!on) return;
        cudaEventRecord(h->prof_ev[h->prof_used + 1], st);
        h->prof_used += 2;
    }
};

template <>
void gemm<float>(tante_handle_s* h, int epi, const float* A, int lda, int64_t w_off, void* Cout, int ldc, bool, int M,
                 int N, int K, const EpiParams& ep, cudaStream_t st, int ldw) {
    const bool res = epi == EPI_BIAS_RESID || epi == EPI_EMBED;
    ProfScope ps(h, st, 2.0 * M * N * K, res ? 1 : 0, (double)M * (4.0 * K + 4.0 * N * (epi == EPI_BIAS_RESID ? 2 : 1)));
    CK(launch_gemm_simt(epi, A, lda, AF(h, w_off), ldw > 0 ? ldw : K, reinterpret_cast<float*>(Cout), ldc, M, N, K, ep, st));
    h->launches++;
}

template <>
void gemm<__nv_bfloat16>(tante_handle_s* h, int epi, const __nv_bfloat16* A, int lda, int64_t w_off, void* Cout, int ldc,
                         bool out_f32, int M, int N, int K, const EpiParams& ep, cudaStream_t st, int ldw) {
    const bool res = epi == EPI_BIAS_RESID || epi == EPI_BIAS_RESID_LN;
    const double out_b = out_f32 ? 4.0 * N * (res ? 2 : 1) + (epi == EPI_BIAS_RESID_LN ? 2.0 * N : 0.0) : 2.0 * N;
    ProfScope ps(h, st, 2.0 * M * N * K, out_f32 ? 1 : 0, (double)M * (2.0 * K + out_b));
    CK(launch_gemm_tc(epi, A, lda, AH(h, w_off), ldw > 0 ? ldw : K, Cout, ldc, out_f32 ? 0 : 1, M, N, K, ep, h->num_sms, st));
    h->launches++;
}

template <typename TOut>
void launch_layernorm(tante_handle_s* h, const float* x, int64_t w, int64_t b, TOut* y, int rows, cudaStream_t st, int width = 0) {
    const int C = width > 0 ? width : h->C;
    const int blocks = (rows + 7) / 8;
    if (C <= 256) layernorm_kernel<TOut, 2><<<blocks, 256, 0, st>>>(x, AF(h, w), AF(h, b), y, rows, C, 1e-5f);
    else layernorm_kernel<TOut, 4><<<blocks, 256, 0, st>>>(x, AF(h, w), AF(h, b), y, rows, C, 1e-5f);
    CK(cudaGetLastError());
    h->launches++;
}

// Fused tail of a transformer block (block_tail_tc.cuh): out-projection + residual + LN2 + MLP + residual + the next layer's
// LN1 in one tcgen05 kernel.  `nx` = the next layer of the backbone (null for the last one: no LayerNorm output).
// Training (x_mid != null) also stores x_mid, the LN2 output, the MLP pre-activation and the hidden activation.
void launch_tail(tante_handle_s* h, const LayerPlan& lp, const LayerPlan* nx, const __nv_bfloat16* att, const float* x_in,
                 float* x_out, __nv_bfloat16* ln_out, int tokens, cudaStream_t st, float* x_mid = nullptr,
                 __nv_bfloat16* ln2 = nullptr, __nv_bfloat16* hpre = nullptr, __nv_bfloat16* hact = nullptr,
                 const DropCfg& drop = DropCfg(), uint32_t site1 = 0, uint32_t site2 = 0) {
    const bool train = x_mid != nullptr;
    const double C = h->C;
    // class 3: HBM-bound by construction -- att (2C) + x in (4C) + x out (4C) [+ ln out (2C)] per token; training adds
    // x_mid (4C) and the three saved bf16 activations (6C)
    ProfScope ps(h, st, 3.0 * 2.0 * tokens * C * C, 3,
                 (double)tokens * (2 * C + 4 * C + 4 * C + (nx ? 2 * C : 0) + (train ? 4 * C + 6 * C : 0)));
    BlockTailArgs a;
    a.att = att;
    a.Wo = AH(h, lp.outw); a.W1 = AH(h, lp.m0w); a.W2 = AH(h, lp.m2w);
    a.bo = AF(h, lp.outb); a.g2 = AF(h, lp.ln2w); a.be2 = AF(h, lp.ln2b); a.b1 = AF(h, lp.m0b); a.b2 = AF(h, lp.m2b);
    a.gn = nx ? AF(h, nx->ln1w) : nullptr; a.ben = nx ? AF(h, nx->ln1b) : nullptr;
    a.x_in = x_in; a.x_out = x_out; a.ln_out = nx ? ln_out : nullptr;
    a.x_mid = x_mid; a.ln2 = ln2; a.hpre = hpre; a.hact = hact;
    a.drop = drop; a.site1 = site1; a.site2 = site2;
    CK(launch_block_tail_any(a, tokens, train, h->num_sms, st));
    h->launches++;
}

// Attention core over n_seq sequences of S tokens addressed in place: token(pos) = (outer * S + pos) * inner + inner_idx, packed
// qkv rows of 3 * Cw, n_head heads of HD = Cw / n_head features.
template <typename TA>
void launch_attention_seq(tante_handle_s* h, const TA* qkv, TA* out, int nseq, int S, int inner, int n_head, int Cw, int HD,
                          bool causal_b, cudaStream_t st, const DropCfg& drop = DropCfg(), uint32_t site = 0) {
    if (sizeof(TA) == 2 && drop.p <= 0.f) {
        // long sequences (composite axes, 65 .. 96-token axes, channel tokens): tiled online-softmax kernel
        cudaError_t e = cudaSuccess;
        if (launch_attention_flash(reinterpret_cast<const __nv_bfloat16*>(qkv), reinterpret_cast<__nv_bfloat16*>(out), nseq, S,
                                   inner, n_head, Cw, HD, causal_b, st, &e)) {
            CK(e);
            h->launches++;
            return;
        }
    }
    if (sizeof(TA) == 2) {
        cudaError_t e = cudaSuccess;
        if (launch_attention_mma(reinterpret_cast<const __nv_bfloat16*>(qkv), reinterpret_cast<__nv_bfloat16*>(out), nseq, S,
                                 inner, n_head, Cw, HD, causal_b, st, &e, drop, site)) {
            CK(e);
            h->launches++;
            return;
        }
    }
    const long long total = (long long)nseq * n_head * S;
    REQUIRE((total + 127) / 128 < (1LL << 31), "attention grid too large");
    const int blocks = (int)((total + 127) / 128);
    const float scale = 1.0f / sqrtf((float)HD);
    const int causal = causal_b;
#define ATT(HDv) axial_attention_kernel<TA, TA, HDv><<<blocks, 128, 0, st>>>(qkv, out, nseq, S, inner, n_head, Cw, causal, scale, drop, site)
    if (HD == 32) ATT(32); else if (HD == 64) ATT(64); else ATT(16);
#undef ATT
    CK(cudaGetLastError());
    h->launches++;
}

template <typename TA>
void launch_attention(tante_handle_s* h, const TA* qkv, TA* out, int B, char axis, cudaStream_t st,
                      const DropCfg& drop = DropCfg(), uint32_t site = 0) {
    int S, inner, nseq;
    const int T = h->T, L = h->L, Hp = h->Hp, Wp = h->Wp;
    // sequence gid = (outer, inner): token(pos) = (outer * S + pos) * inner_sz + inner   (attn_backbone.py:149-182)
    if (axis == 'T') { S = T; inner = L; nseq = B * L; }
    else if (axis == 'H') { S = Hp; inner = Wp; nseq = B * T * Wp; }
    else if (axis == 'W') { S = Wp; inner = 1; nseq = B * T * Hp; }
    else if (axis == 'L') { S = L; inner = 1; nseq = B * T; }               // (b t) (h w)
    else if (axis == 'Y') { S = T * Hp; inner = Wp; nseq = B * Wp; }        // (b w) (t h)
    else { S = T * L; inner = 1; nseq = B; }                                // 'A': b (t h w)
    launch_attention_seq<TA>(h, qkv, out, nseq, S, inner, h->cfg.n_head, h->C, h->HD, axis == 'T', st, drop, site);
}

// One axis-'C' layer (attn_backbone.py:184-189; channel_axis.cuh) in place on the fp32 latent x [tokens][C]: lift every scalar to
// E features, TransformerBlock(E) over the C channel tokens of each latent token, keep the last feature.  Runs in chunks of
// h->chan_tokens latent tokens (rows = chunk * C) through the scratch buffers of tante_reserve.
template <typename TA>
void run_channel_layer(tante_handle_s* h, const LayerPlan& lp, const float* x, float* x_dst, int tokens, cudaStream_t st) {
    const int C = h->C, E = lp.E, Hc = lp.Hc, nh = h->cfg.n_head;
    float* xc = reinterpret_cast<float*>(h->cx.p);
    TA* ln = reinterpret_cast<TA*>(h->cln.p);
    TA* qkv = reinterpret_cast<TA*>(h->cqkv.p);
    TA* att = reinterpret_cast<TA*>(h->catt.p);
    TA* hid = reinterpret_cast<TA*>(h->chid.p);
    REQUIRE(h->chan_tokens > 0 && xc, "channel-axis workspace not reserved");
    const size_t lift_smem = ((size_t)(E / 4) * E + E + 10 * (size_t)(E / 4)) * sizeof(float);
    for (int t0 = 0; t0 < tokens; t0 += h->chan_tokens) {
        const int tc = std::min(h->chan_tokens, tokens - t0);
        const int rows = tc * C;
        const float* xs = x + (size_t)t0 * C;
        channel_lift_kernel<<<std::min((rows + 7) / 8, 16 * h->num_sms), 256, lift_smem, st>>>(
            xs, AF(h, lp.cw0), AF(h, lp.cb0), AF(h, lp.cw2), AF(h, lp.cb2), xc, rows, E);
        CK(cudaGetLastError());
        h->launches++;
        launch_layernorm<TA>(h, xc, lp.ln1w, lp.ln1b, ln, rows, st, E);
        EpiParams eq; eq.bias = AF(h, lp.inb);
        gemm<TA>(h, EPI_BIAS, ln, E, lp.inw, qkv, 3 * E, false, rows, 3 * E, E, eq, st);
        launch_attention_seq<TA>(h, qkv, att, tc, C, 1, nh, E, E / nh, false, st);
        EpiParams eo; eo.bias = AF(h, lp.outb); eo.resid = xc; eo.ldr = E;
        gemm<TA>(h, EPI_BIAS_RESID, att, E, lp.outw, xc, E, true, rows, E, E, eo, st);
        launch_layernorm<TA>(h, xc, lp.ln2w, lp.ln2b, ln, rows, st, E);
        EpiParams e0; e0.bias = AF(h, lp.m0b);
        gemm<TA>(h, EPI_BIAS_GELU_TANH, ln, E, lp.m0w, hid, Hc, false, rows, Hc, E, e0, st);
        EpiParams e2; e2.bias = AF(h, lp.m2b); e2.resid = xc; e2.ldr = E;
        gemm<TA>(h, EPI_BIAS_RESID, hid, Hc, lp.m2w, xc, E, true, rows, E, Hc, e2, st);
        channel_extract_kernel<<<(rows + 255) / 256, 256, 0, st>>>(xc, x_dst + (size_t)t0 * C, rows, E);
        CK(cudaGetLastError());
        h->launches++;
    }
}

void launch_propagator(tante_handle_s* h, const float* xin, float* x, int B, int axis /*0=H,1=W,2=T*/,
                       const OrderPlan& op, cudaStream_t st) {
    int S; long long IC, outer;
    const int T = h->T, L = h->L, Hp = h->Hp, Wp = h->Wp, C = h->C;
    if (axis == 0) { S = Hp; IC = (long long)Wp * C; outer = (long long)B * T; }
    else if (axis == 1) { S = Wp; IC = C; outer = (long long)B * T * Hp; }
    else { S = T; IC = (long long)L * C; outer = B; }
    if (S <= 4 && (IC & 3) == 0) {      // short axes (T = 4): per-column register mat-vecs, one pass over the latent
        const long long total = outer * (IC / 4);
        const unsigned grid = (unsigned)std::min<long long>((total + 255) / 256, 16LL * h->num_sms);
        const bool fast = h->cfg.precision == TANTE_PREC_BF16;
#define PSMALL(TM, SM) propagator_small_kernel<TM, SM><<<grid, 256, 0, st>>>(xin, x, S, IC, outer, AF(h, op.prop[axis][0]), \
            AF(h, op.prop[axis][1]), AF(h, op.prop[axis][2]), AF(h, op.prop[axis][3]))
        if (fast) PSMALL(__nv_bfloat16, 4); else PSMALL(float, 4);
#undef PSMALL
        CK(cudaGetLastError());
        h->launches++;
        return;
    }
    if (h->cfg.precision == TANTE_PREC_BF16 && S > 8) {
        cudaError_t e = cudaSuccess;
        if (launch_propagator_mma(xin, x, S, IC, outer, AF(h, op.prop[axis][0]), AF(h, op.prop[axis][1]), AF(h, op.prop[axis][2]),
                                  AF(h, op.prop[axis][3]), st, &e, h->num_sms)) {
            CK(e);
            h->launches++;
            return;
        }
    }
    const int S4 = (S + 3) & ~3;
    const size_t smem = (size_t)(2 * S4 * 128 + 2 * S4 * S4 + 2 * S4) * sizeof(float);
    dim3 grid((unsigned)outer, (unsigned)((IC + 127) / 128));
    REQUIRE((IC + 127) / 128 <= 65535, "latent too large for the propagator grid");
    const int threads = 32 * std::min(8, S4 / 4);
    if (h->cfg.precision == TANTE_PREC_BF16) propagator_kernel<__nv_bfloat16><<<grid, threads, smem, st>>>(xin, x, S, IC, AF(h, op.prop[axis][0]), AF(h, op.prop[axis][1]),
                                               AF(h, op.prop[axis][2]), AF(h, op.prop[axis][3]));
    else propagator_kernel<float><<<grid, threads, smem, st>>>(xin, x, S, IC, AF(h, op.prop[axis][0]), AF(h, op.prop[axis][1]),
                                               AF(h, op.prop[axis][2]), AF(h, op.prop[axis][3]));
    CK(cudaGetLastError());
    h->launches++;
}

inline unsigned blocks_for(long long n, int per) { return (unsigned)((n + per - 1) / per); }

template <typename TA>
void launch_head(tante_handle_s* h, const StepIO& io, int B, const RolloutState& rs, float* deriv_dbg, cudaStream_t st) {
    HeadParams hp{};
    for (int k = 0; k < h->K; ++k) {
        hp.z[k] = h->z2[k].p;
        hp.w3[k] = AF(h, h->orders[k].decw[2]);
        hp.b3[k] = AF(h, h->orders[k].decb[2]);
    }
    hp.K = h->K;
    hp.fi = h->cfg.frame_interval;
    hp.u_ring = io.input;
    hp.fcount = io.fcount;
    hp.n_arr = io.rollout ? rs.n_cur : reinterpret_cast<int*>(h->nbuf.p);
    hp.frames = io.frames; hp.n_cap = io.n_cap;
    hp.ptrs = io.rollout ? rs.ptrs : nullptr; hp.ring_out = io.ring_out; hp.cum = io.rollout ? rs.cum : nullptr; hp.n_roll = io.n_roll;
    hp.deriv_dbg = deriv_dbg;
    hp.act = io.rollout ? rs.act : nullptr;
    const long long rows = (long long)B * h->L * h->geom.R1;
    if (sizeof(TA) == 2) {
        cudaError_t e = cudaSuccess;
        if (launch_head_mma(hp, h->geom, h->C1, rows, B, h->num_sms, st, &e)) {
            CK(e);
            h->launches++;
            return;
        }
    }
    const int NO = h->geom.k0 * h->geom.k0 * h->D;
    const size_t smem = (size_t)(h->K * h->C1 * NO + h->K * h->D) * sizeof(float);
    const int blocks = (int)((rows + 127) / 128);
#define HEAD(KO) taylor_head_kernel<TA, 8, KO><<<blocks, 128, smem, st>>>(hp, h->geom, h->C1, rows, B)
    switch (h->K) {
        case 1: HEAD(1); break;
        case 2: HEAD(2); break;
        case 3: HEAD(3); break;
        default: HEAD(4); break;
    }
#undef HEAD
    CK(cudaGetLastError());
    h->launches++;
}

// ---- patch_scale >= 16 (wide_patch.cuh): encoder, decoder of one order, emit ----
// Grids of the natural-order encoder stages for a batch of B windows: patch grids (H1 x W1, H2 x W2, Hp x Wp) and the conv grids in
// front of them (kernel k, stride s, pad (k - 1) / 2); the two differ -- and an adaptive average pooling sits between -- only with
// overlap_ratio != 0.
struct WideDims {
    int H1, W1, H2, W2, Hc1, Wc1, Hc2, Wc2, Hc3, Wc3;
    bool pool1, pool2, pool3;
    long long rows1, rows2, rows3;
};
inline WideDims wide_dims(const tante_handle_s* h, int B) {
    const PatchGeom& g = h->geom;
    auto cdim = [](int n, int k, int s) { return (n + 2 * ((k - 1) / 2) - k) / s + 1; };
    WideDims d;
    d.H1 = h->cfg.H / g.k0; d.W1 = h->cfg.W / g.k0; d.H2 = d.H1 / g.k1; d.W2 = d.W1 / g.k1;
    d.Hc1 = cdim(h->cfg.H, g.k0, h->st[0]); d.Wc1 = cdim(h->cfg.W, g.k0, h->st[0]);
    d.Hc2 = cdim(d.H1, g.k1, h->st[1]); d.Wc2 = cdim(d.W1, g.k1, h->st[1]);
    d.Hc3 = cdim(d.H2, g.k2, h->st[2]); d.Wc3 = cdim(d.W2, g.k2, h->st[2]);
    d.pool1 = d.Hc1 != d.H1 || d.Wc1 != d.W1;
    d.pool2 = d.Hc2 != d.H2 || d.Wc2 != d.W2;
    d.pool3 = d.Hc3 != h->Hp || d.Wc3 != h->Wp;
    const long long NI = (long long)B * h->T;
    d.rows1 = NI * d.Hc1 * d.Wc1; d.rows2 = NI * d.Hc2 * d.Wc2; d.rows3 = NI * d.Hc3 * d.Wc3;
    return d;
}

// Tensor mode, K beyond the tcgen05 GEMM's resident weight slice (1024): out[M][N] (fp32) = A[M][K] W[N][K]^T + bias as K / parts
// column blocks accumulated through the fp32 output (first block EPI_BIAS, the rest EPI_BIAS_RESID in place).
inline void gemm_bigk_f32(tante_handle_s* h, const __nv_bfloat16* A, int lda, int64_t w_off, float* out, int M, int N, int K,
                          const float* bias, cudaStream_t st) {
    int parts = (K + 1023) / 1024;
    while (K % (parts * 64) != 0) ++parts;
    const int Kp = K / parts;
    REQUIRE(Kp >= 64 && Kp <= 1024, "split-K GEMM: K not covered");
    EpiParams e0; e0.bias = bias;
    gemm<__nv_bfloat16>(h, EPI_BIAS, A, lda, w_off, out, N, true, M, N, Kp, e0, st, K);
    for (int p = 1; p < parts; ++p) {
        EpiParams e; e.bias = AF(h, h->zero_off); e.resid = out; e.ldr = N;
        gemm<__nv_bfloat16>(h, EPI_BIAS_RESID, A + (size_t)p * Kp, lda, w_off + (int64_t)p * Kp, out, N, true, M, N, Kp, e, st, K);
    }
}

template <typename TA>
void run_encoder_wide(tante_handle_s* h, const StepIO& io, int B, cudaStream_t st) {
    const int C = h->C, C1 = h->C1, C2 = h->C2, T = h->T, L = h->L;
    const PatchGeom& g = h->geom;
    const int tokens = B * T * L;
    const int H = h->cfg.H, W = h->cfg.W, D = h->D;
    TA* wb = reinterpret_cast<TA*>(h->wbuf.p);
    TA* a1 = reinterpret_cast<TA*>(h->a1.p);
    TA* a2 = reinterpret_cast<TA*>(h->a2.p);
    float* x = reinterpret_cast<float*>(h->x.p);
    const int H1 = H / g.k0, W1 = W / g.k0, H2 = H1 / g.k1, W2 = W1 / g.k1;
    const long long NI = (long long)B * T;
    // conv grid of a stage (kernel k, stride s, pad (k - 1) / 2 over an Hin x Win grid); == the patch grid without overlap
    auto cdim = [](int n, int k, int s) { return (n + 2 * ((k - 1) / 2) - k) / s + 1; };
    const int Hc1 = cdim(H, g.k0, h->st[0]), Wc1 = cdim(W, g.k0, h->st[0]);
    const int Hc2 = cdim(H1, g.k1, h->st[1]), Wc2 = cdim(W1, g.k1, h->st[1]);
    const int Hc3 = cdim(H2, g.k2, h->st[2]), Wc3 = cdim(W2, g.k2, h->st[2]);
    const bool pool1 = Hc1 != H1 || Wc1 != W1, pool2 = Hc2 != H2 || Wc2 != W2, pool3 = Hc3 != h->Hp || Wc3 != h->Wp;
    const long long rows1 = NI * Hc1 * Wc1, rows2 = NI * Hc2 * Wc2, rows3 = NI * Hc3 * Wc3;
    REQUIRE(rows1 * h->K1pad < (1LL << 40) && rows1 < (1LL << 31) && rows2 < (1LL << 31) && rows3 < (1LL << 31),
            "input too large for the wide conv GEMMs");
    TA* cg = reinterpret_cast<TA*>(h->cgrid.p);
    auto pool = [&](const TA* in, int Hc, int Wc, int Cc, int Ho, int Wo, TA* out, float* out32, bool act) {
        const long long total4 = NI * Ho * Wo * Cc / 4;
        const unsigned nb = blocks_for(total4, 256);
        if (out32) wide_pool_kernel<TA, false, true><<<nb, 256, 0, st>>>(in, Hc, Wc, Cc, Ho, Wo, nullptr, out32, total4);
        else if (act) wide_pool_kernel<TA, true, false><<<nb, 256, 0, st>>>(in, Hc, Wc, Cc, Ho, Wo, out, nullptr, total4);
        else wide_pool_kernel<TA, false, false><<<nb, 256, 0, st>>>(in, Hc, Wc, Cc, Ho, Wo, out, nullptr, total4);
        CK(cudaGetLastError());
        h->launches++;
    };
    // conv1: (shifted / strided) windows of the ring frames -> [rows1][K1pad] -> GEMM (+ pooling) + GELU -> grid [BT][H1][W1][C1]
    {
        const long long total = rows1 * h->K1pad;
        wide_im2col_cf_kernel<TA><<<blocks_for(total, 256), 256, 0, st>>>(io.input, io.fcount, T, D, H, W, g.k0, (g.k0 - 1) / 2,
                                                                         h->K1pad, wb, total, h->st[0], Hc1, Wc1);
        CK(cudaGetLastError());
        h->launches++;
        EpiParams e1; e1.bias = AF(h, h->enc_b[0]);
        if (pool1) {
            gemm<TA>(h, EPI_BIAS, wb, h->K1pad, h->enc_w1wide, cg, C1, false, (int)rows1, C1, h->K1pad, e1, st);
            pool(cg, Hc1, Wc1, C1, H1, W1, a1, nullptr, true);
        } else {
            gemm<TA>(h, EPI_BIAS_GELU_ERF, wb, h->K1pad, h->enc_w1wide, a1, C1, false, (int)rows1, C1, h->K1pad, e1, st);
        }
    }
    // conv2
    {
        const int K2 = g.k1 * g.k1 * C1;
        const long long total4 = rows2 * K2 / 4;
        wide_im2col_cl_kernel<TA><<<blocks_for(total4, 256), 256, 0, st>>>(a1, H1, W1, C1, g.k1, (g.k1 - 1) / 2, wb, total4, h->st[1], Hc2, Wc2);
        CK(cudaGetLastError());
        h->launches++;
        EpiParams e2; e2.bias = AF(h, h->enc_b[1]);
        if (pool2) {
            gemm<TA>(h, EPI_BIAS, wb, K2, h->enc_w[1], cg, C2, false, (int)rows2, C2, K2, e2, st);
            pool(cg, Hc2, Wc2, C2, H2, W2, a2, nullptr, true);
        } else {
            gemm<TA>(h, EPI_BIAS_GELU_ERF, wb, K2, h->enc_w[1], a2, C2, false, (int)rows2, C2, K2, e2, st);
        }
    }
    // conv3 + t_encode FiLM + embeddings -> residual stream
    {
        const int K3 = g.k2 * g.k2 * C2;
        const long long total4 = rows3 * K3 / 4;
        wide_im2col_cl_kernel<TA><<<blocks_for(total4, 256), 256, 0, st>>>(a2, H2, W2, C2, g.k2, (g.k2 - 1) / 2, wb, total4, h->st[2], Hc3, Wc3);
        CK(cudaGetLastError());
        h->launches++;
        EpiParams e3; e3.bias = AF(h, h->enc_b[2]);
        if (pool3) {
            // overlap: conv grid -> adaptive average pooling -> fp32 pre-embedding -> embed pass
            float* v = reinterpret_cast<float*>(h->qkv.p);
            if (sizeof(TA) == 2 && K3 > 1024) {
                REQUIRE((size_t)rows3 * C * 4 <= h->kscratch.bytes, "split-K conv: scratch not reserved");
                float* acc = reinterpret_cast<float*>(h->kscratch.p);
                gemm_bigk_f32(h, reinterpret_cast<const __nv_bfloat16*>(wb), K3, h->enc_w[2], acc, (int)rows3, C, K3, e3.bias, st);
                f32_to_ta_kernel<TA, false><<<blocks_for(rows3 * C / 4, 256), 256, 0, st>>>(acc, cg, rows3 * C / 4);
                CK(cudaGetLastError());
                h->launches++;
            } else {
                gemm<TA>(h, EPI_BIAS, wb, K3, h->enc_w[2], cg, C, false, (int)rows3, C, K3, e3, st);
            }
            pool(cg, Hc3, Wc3, C, h->Hp, h->Wp, nullptr, v, false);
            embed_fwd_kernel<<<blocks_for((long long)tokens * C / 4, 256), 256, 0, st>>>(v, AF(h, h->film_t_off), AF(h, h->s_emb),
                                                                                      AF(h, h->t_emb), x, tokens, T, L, C);
            CK(cudaGetLastError());
            h->launches++;
        } else if (sizeof(TA) == 2 && K3 > 1024) {
            // K = 2048 (patch_scale 64) exceeds the resident weight slice of the tcgen05 GEMM: K blocks through an fp32
            // scratch, then the embed pass
            float* v = reinterpret_cast<float*>(h->qkv.p);
            gemm_bigk_f32(h, reinterpret_cast<const __nv_bfloat16*>(wb), K3, h->enc_w[2], v, tokens, C, K3, e3.bias, st);
            embed_fwd_kernel<<<blocks_for((long long)tokens * C / 4, 256), 256, 0, st>>>(v, AF(h, h->film_t_off), AF(h, h->s_emb),
                                                                                      AF(h, h->t_emb), x, tokens, T, L, C);
            CK(cudaGetLastError());
            h->launches++;
        } else {
            e3.film = AF(h, h->film_t_off); e3.s_emb = AF(h, h->s_emb); e3.t_emb = AF(h, h->t_emb);
            e3.T = T; e3.L = L; e3.ldr = C;
            gemm<TA>(h, EPI_EMBED, wb, K3, h->enc_w[2], x, C, true, tokens, C, K3, e3, st);
        }
    }
}

// decoder of order o on the (modified) last-frame latent dmod [B*L][C] -> derivative field dfield[o] (B, D, H, W)
template <typename TA>
void run_decoder_wide(tante_handle_s* h, int o, const TA* dmod, int B, cudaStream_t st) {
    const OrderPlan& op = h->orders[o];
    const int C = h->C, C1 = h->C1, C2 = h->C2, L = h->L, D = h->D, Hp = h->Hp, Wp = h->Wp;
    const PatchGeom& g = h->geom;
    const int H = h->cfg.H, W = h->cfg.W;
    TA* wb = reinterpret_cast<TA*>(h->wbuf.p);
    TA* z1 = reinterpret_cast<TA*>(h->z1.p);
    TA* z2 = reinterpret_cast<TA*>(h->z2[o].p);
    float* field = reinterpret_cast<float*>(h->dfield.p) + (size_t)o * B * D * H * W;
    const int H2 = Hp * g.k2, W2 = Wp * g.k2, H1 = H2 * g.k1, W1 = W2 * g.k1;
    auto post = [&](const TA* S, int ldS, int hi, int wi, int Cout, int k, int sd, const float* bias, TA* out, float* fld, bool act) {
        const long long total = (long long)B * (hi * k) * (wi * k) * Cout;
        const unsigned blocks = blocks_for(total, 256);
        if (fld) wide_deconv_post_kernel<TA, false, true><<<blocks, 256, 0, st>>>(S, ldS, hi, wi, Cout, k, bias, nullptr, fld, total, sd);
        else if (act) wide_deconv_post_kernel<TA, true, false><<<blocks, 256, 0, st>>>(S, ldS, hi, wi, Cout, k, bias, out, nullptr, total, sd);
        else wide_deconv_post_kernel<TA, false, false><<<blocks, 256, 0, st>>>(S, ldS, hi, wi, Cout, k, bias, out, nullptr, total, sd);
        CK(cudaGetLastError());
        h->launches++;
    };
    // With stride == kernel every output sample has ONE tap, so the (replicated) bias rides in the GEMM epilogue; with overlap
    // (stride < kernel) several taps are summed per sample: the GEMM runs bias-free and the pass after it adds bias[co] once (the
    // first Cout entries of the replicated vector are the raw bias).
    const bool ov1 = h->st[2] != g.k2, ov2 = h->st[1] != g.k1;
    // dec_conv_1 (k2): [B*L][C] -> sub-pixel [B*L][k2*k2*C2] (+ replicated bias) -> resample + GELU -> grid [B][H2][W2][C2]
    const int N1 = g.k2 * g.k2 * C2, N2 = g.k1 * g.k1 * C1;
    EpiParams ed; ed.bias = ov1 ? AF(h, h->zero_off) : AF(h, op.decb[0]);
    gemm<TA>(h, EPI_BIAS, dmod, C, op.decw[0], wb, N1, false, B * L, N1, C, ed, st);
    post(wb, N1, Hp, Wp, C2, g.k2, h->st[2], ov1 ? AF(h, op.decb[0]) : nullptr, z1, nullptr, true);
    // dec_conv_2 (k1)
    ed.bias = ov2 ? AF(h, h->zero_off) : AF(h, op.decb[1]);
    gemm<TA>(h, EPI_BIAS, z1, C2, op.decw[1], wb, N2, false, B * H2 * W2, N2, C2, ed, st);
    post(wb, N2, H2, W2, C1, g.k1, h->st[1], ov2 ? AF(h, op.decb[1]) : nullptr, z2, nullptr, true);
    // dec_conv_3 (k0): output width k0*k0*D padded to NOpad, bias added after the resample (its weights sum to one)
    EpiParams e3; e3.bias = AF(h, h->zero_off);
    gemm<TA>(h, EPI_BIAS, z2, C1, op.w3nk, wb, h->NOpad, false, B * H1 * W1, h->NOpad, C1, e3, st);
    post(wb, h->NOpad, H1, W1, D, g.k0, h->st[0], AF(h, op.decb[2]), nullptr, field, false);
}

// ---- enc_dec_type = 'fno' (fno.cuh) ----
// twiddle tables of the four axis lengths, (cos, sin)(2 pi j / N) in double precision: [W | H | W1 | H1]
void fno_twiddles(tante_handle_s* h) {
    if (h->ftw.p) return;
    const int W = h->cfg.W, H = h->cfg.H, W1 = W / h->fp0, H1 = H / h->fp0;
    std::vector<float> tw((size_t)2 * (W + H + W1 + H1));
    size_t o = 0;
    for (int N : {W, H, W1, H1})
        for (int j = 0; j < N; ++j) {
            const double a = 2.0 * 3.14159265358979323846 * (double)j / (double)N;
            tw[o++] = (float)cos(a); tw[o++] = (float)sin(a);
        }
    dev_alloc(h, h->ftw, tw.size() * sizeof(float));
    CK(cudaMemcpy(h->ftw.p, tw.data(), tw.size() * sizeof(float), cudaMemcpyHostToDevice));
}

// one SpectralLayer: in (view) -> TA channels-last grid `out` (+ GELU) or the fp32 channels-first `field`
template <typename TA>
void run_spectral(tante_handle_s* h, const SpecPlan& sp, const SpecView& in, long long N, int H, int W, int level, bool act,
                  TA* out, float* field, cudaStream_t st) {
    const int W0 = h->cfg.W, H0 = h->cfg.H, W1 = W0 / h->fp0;
    const float2* tw = reinterpret_cast<const float2*>(h->ftw.p);
    const float2* twW = level == 0 ? tw : tw + W0 + H0;
    const float2* twH = level == 0 ? tw + W0 : tw + W0 + H0 + W1;
    const int m1 = sp.wm1, m2 = sp.wm2;
    float2* A = reinterpret_cast<float2*>(h->fA.p);
    float2* Bc = reinterpret_cast<float2*>(h->fB.p);
    const long long rows = N * sp.Cin * H;
    spec_dft_w_kernel<TA><<<blocks_for(rows, 4), 128, 0, st>>>(in, sp.Cin, H, W, m2, twW, A, rows);
    CK(cudaGetLastError());
    const long long tx = N * sp.Cin * 2 * m1 * m2;
    spec_dft_h_kernel<<<blocks_for(tx, 256), 256, 0, st>>>(A, H, m1, m2, twH, Bc, tx);                 // X -> Bc
    CK(cudaGetLastError());
    const long long ty = N * sp.Cout * 2 * m1 * m2;
    spec_mix_kernel<<<blocks_for(ty, 256), 256, 0, st>>>(Bc, reinterpret_cast<const float2*>(AF(h, sp.w)), sp.Cin, sp.Cout, m1, m2,
                                                         sp.wm2, sp.wm1, A, ty);                        // Y -> A
    CK(cudaGetLastError());
    const long long tb = N * sp.Cout * H * m2;
    spec_idft_h_kernel<<<blocks_for(tb, 256), 256, 0, st>>>(A, H, m1, m2, twH, Bc, tb);                // Bh -> Bc
    CK(cudaGetLastError());
    const long long to = N * sp.Cout * H * W;
    const unsigned nb = blocks_for(to, 256);
    // the 1x1 convolution of the wide layers (channels-last grids, >= 64 channels each side) is a GEMM over the pixels: it writes
    // conv + bias into `out`, the last pass adds the spectral part in place (measured: the per-thread channel loop was 1.5 ms of a
    // 4.9 ms forward at the TRL shape)
    int conv_done = 0;
    if (!field && in.mode == 1 && sp.Cin % 64 == 0 && sp.Cout % 64 == 0 && N * H * W < (1LL << 31)) {
        EpiParams ec; ec.bias = AF(h, sp.b0);
        gemm<TA>(h, EPI_BIAS, reinterpret_cast<const TA*>(in.p), sp.Cin, sp.w0, out, sp.Cout, sizeof(TA) == 4, (int)(N * H * W), sp.Cout, sp.Cin,
                 ec, st);
        conv_done = 1;
    }
    if (field) spec_out_kernel<TA, false, true><<<nb, 256, 0, st>>>(Bc, in, AF(h, sp.w0), AF(h, sp.b0), sp.Cin, sp.Cout, H, W, m2, twW, nullptr, field, to);
    else if (act) spec_out_kernel<TA, true, false><<<nb, 256, 0, st>>>(Bc, in, AF(h, sp.w0), AF(h, sp.b0), sp.Cin, sp.Cout, H, W, m2, twW, out, nullptr, to, conv_done);
    else spec_out_kernel<TA, false, false><<<nb, 256, 0, st>>>(Bc, in, AF(h, sp.w0), AF(h, sp.b0), sp.Cin, sp.Cout, H, W, m2, twW, out, nullptr, to, conv_done);
    CK(cudaGetLastError());
    h->launches += 5;
}

// conv over a channels-last grid as gather + GEMM; K beyond the tcgen05 GEMM's resident slice (1024) runs in K blocks
template <typename TA>
void conv_cl_gemm(tante_handle_s* h, int epi, const TA* grid, int Hs, int Ws, int Cin, int k, int64_t w_off, void* out, int Cout,
                  bool out_f32, long long n_img, EpiParams ep, cudaStream_t st, int sd = 0) {
    TA* wb = reinterpret_cast<TA*>(h->wbuf.p);
    const int K = k * k * Cin;
    const int se = sd > 0 ? sd : k, pad = (k - 1) / 2;
    const int Hc = (Hs + 2 * pad - k) / se + 1, Wc = (Ws + 2 * pad - k) / se + 1;      // conv grid; == the patch grid without overlap
    const int Ho = Hs / k, Wo = Ws / k;
    const bool pooled = Hc != Ho || Wc != Wo;
    const long long rows = n_img * Hc * Wc;
    REQUIRE(rows < (1LL << 31), "input too large for the gather GEMM");
    const long long total4 = rows * K / 4;
    wide_im2col_cl_kernel<TA><<<blocks_for(total4, 256), 256, 0, st>>>(grid, Hs, Ws, Cin, k, pad, wb, total4, se, Hc, Wc);
    CK(cudaGetLastError());
    h->launches++;
    const bool bigk = sizeof(TA) == 2 && K > 1024;
    if (pooled) {
        // overlap_ratio != 0: GEMM (+ bias) onto the conv grid, adaptive average pooling (+ GELU) to the patch grid
        REQUIRE(epi == EPI_BIAS || epi == EPI_BIAS_GELU_ERF, "pooled conv: epilogue not covered");
        REQUIRE((size_t)rows * Cout * sizeof(TA) <= h->cgrid.bytes, "pooled conv: conv-grid scratch not reserved");
        TA* cg = reinterpret_cast<TA*>(h->cgrid.p);
        if (bigk) {
            REQUIRE((size_t)rows * Cout * 4 <= h->kscratch.bytes, "split-K conv: scratch not reserved");
            float* v = reinterpret_cast<float*>(h->kscratch.p);
            gemm_bigk_f32(h, reinterpret_cast<const __nv_bfloat16*>(wb), K, w_off, v, (int)rows, Cout, K, ep.bias, st);
            f32_to_ta_kernel<TA, false><<<blocks_for(rows * Cout / 4, 256), 256, 0, st>>>(v, cg, rows * Cout / 4);
            CK(cudaGetLastError());
            h->launches++;
        } else {
            EpiParams eb; eb.bias = ep.bias;
            gemm<TA>(h, EPI_BIAS, wb, K, w_off, cg, Cout, false, (int)rows, Cout, K, eb, st);
        }
        const long long p4 = n_img * Ho * Wo * Cout / 4;
        const unsigned nb = blocks_for(p4, 256);
        if (out_f32) wide_pool_kernel<TA, false, true><<<nb, 256, 0, st>>>(cg, Hc, Wc, Cout, Ho, Wo, nullptr, reinterpret_cast<float*>(out), p4);
        else if (epi == EPI_BIAS_GELU_ERF) wide_pool_kernel<TA, true, false><<<nb, 256, 0, st>>>(cg, Hc, Wc, Cout, Ho, Wo, reinterpret_cast<TA*>(out), nullptr, p4);
        else wide_pool_kernel<TA, false, false><<<nb, 256, 0, st>>>(cg, Hc, Wc, Cout, Ho, Wo, reinterpret_cast<TA*>(out), nullptr, p4);
        CK(cudaGetLastError());
        h->launches++;
        return;
    }
    if (bigk) {
        const __nv_bfloat16* wbh = reinterpret_cast<const __nv_bfloat16*>(wb);
        if (out_f32) {
            REQUIRE(epi == EPI_BIAS, "the split-K path writes plain fp32 outputs");
            gemm_bigk_f32(h, wbh, K, w_off, reinterpret_cast<float*>(out), (int)rows, Cout, K, ep.bias, st);
        } else {
            // 8x8 stages (K = 2048): accumulate in the fp32 scratch of tante_reserve, then bias-free activation + conversion
            REQUIRE(epi == EPI_BIAS || epi == EPI_BIAS_GELU_ERF, "split-K conv: epilogue not covered");
            REQUIRE((size_t)rows * Cout * 4 <= h->kscratch.bytes, "split-K conv: scratch not reserved");
            float* v = reinterpret_cast<float*>(h->kscratch.p);
            gemm_bigk_f32(h, wbh, K, w_off, v, (int)rows, Cout, K, ep.bias, st);
            const long long n4 = rows * Cout / 4;
            if (epi == EPI_BIAS_GELU_ERF) f32_to_ta_kernel<TA, true><<<blocks_for(n4, 256), 256, 0, st>>>(v, reinterpret_cast<TA*>(out), n4);
            else f32_to_ta_kernel<TA, false><<<blocks_for(n4, 256), 256, 0, st>>>(v, reinterpret_cast<TA*>(out), n4);
            CK(cudaGetLastError());
            h->launches++;
        }
    } else {
        gemm<TA>(h, epi, wb, K, w_off, out, Cout, out_f32, (int)rows, Cout, K, ep, st);
    }
}

template <typename TA>
void run_encoder_fno(tante_handle_s* h, const StepIO& io, int B, cudaStream_t st) {
    const int C = h->C, C1 = h->C1, C2 = h->C2, C8 = h->C / 8, T = h->T, L = h->L, D = h->D;
    const int H = h->cfg.H, W = h->cfg.W, p0 = h->fp0, p1 = h->fp1, H1 = H / p0, W1 = W / p0;
    const int tokens = B * T * L;
    const long long NI = (long long)B * T;
    float* x = reinterpret_cast<float*>(h->x.p);
    TA* g0 = reinterpret_cast<TA*>(h->fg0.p);      // [NI][H][W][C8]
    TA* g1 = reinterpret_cast<TA*>(h->fg1.p);      // [NI][H1][W1][C1]
    TA* g2 = reinterpret_cast<TA*>(h->fg2.p);      // [NI][H1][W1][C2]
    fno_twiddles(h);
    // enc_spectral_1 + GELU on the (ring) frames  (enc_dec_fno.py:258-259)
    SpecView v0{io.input, 0, io.fcount, T};
    run_spectral<TA>(h, h->fes1, v0, NI, H, W, 0, true, g0, nullptr, st);
    // enc_conv_1 + GELU (:260-261)
    EpiParams e1; e1.bias = AF(h, h->enc_b[0]);
    conv_cl_gemm<TA>(h, EPI_BIAS_GELU_ERF, g0, H, W, C8, p0, h->enc_w[0], g1, C1, false, NI, e1, st, h->st[0]);
    // enc_spectral_2 + GELU (:263-264)
    SpecView v1{g1, 1, nullptr, 1};
    run_spectral<TA>(h, h->fes2, v1, NI, H1, W1, 1, true, g2, nullptr, st);
    // enc_conv_2 (:265) + t_encode FiLM + embeddings -> residual stream
    EpiParams e2; e2.bias = AF(h, h->enc_b[1]);
    if ((sizeof(TA) == 2 && p1 * p1 * C2 > 1024) || h->st[1] != p1) {      // (split-K or pooled: fp32 pre-embedding, then the embed pass)
        float* v = reinterpret_cast<float*>(h->qkv.p);
        conv_cl_gemm<TA>(h, EPI_BIAS, g2, H1, W1, C2, p1, h->enc_w[1], v, C, true, NI, e2, st, h->st[1]);
        embed_fwd_kernel<<<blocks_for((long long)tokens * C / 4, 256), 256, 0, st>>>(v, AF(h, h->film_t_off), AF(h, h->s_emb),
                                                                                  AF(h, h->t_emb), x, tokens, T, L, C);
        CK(cudaGetLastError());
        h->launches++;
    } else {
        e2.film = AF(h, h->film_t_off); e2.s_emb = AF(h, h->s_emb); e2.t_emb = AF(h, h->t_emb);
        e2.T = T; e2.L = L; e2.ldr = C;
        conv_cl_gemm<TA>(h, EPI_EMBED, g2, H1, W1, C2, p1, h->enc_w[1], x, C, true, NI, e2, st);
    }
}

// dec_FNO.forward (enc_dec_fno.py:303-323) of order o on the last-frame latent dmod [B*L][C] -> dfield[o] (B, D, H, W)
template <typename TA>
void run_decoder_fno(tante_handle_s* h, int o, const TA* dmod, int B, cudaStream_t st) {
    const OrderPlan& op = h->orders[o];
    const int C = h->C, C1 = h->C1, C2 = h->C2, C8 = h->C / 8, L = h->L, D = h->D, Hp = h->Hp, Wp = h->Wp;
    const int H = h->cfg.H, W = h->cfg.W, p0 = h->fp0, p1 = h->fp1, H1 = H / p0, W1 = W / p0;
    TA* wb = reinterpret_cast<TA*>(h->wbuf.p);
    TA* g0 = reinterpret_cast<TA*>(h->fg0.p);      // [B][H][W][C8]
    TA* g1 = reinterpret_cast<TA*>(h->fg1.p);      // [B][H1][W1][C1]
    TA* g2 = reinterpret_cast<TA*>(h->fg2.p);      // [B][H1][W1][C2]
    float* field = reinterpret_cast<float*>(h->dfield.p) + (size_t)o * B * D * H * W;
    auto post = [&](const TA* S, int ldS, int hi, int wi, int Cout, int k, int sd, const float* bias, TA* out) {
        const long long total = (long long)B * (hi * k) * (wi * k) * Cout;
        wide_deconv_post_kernel<TA, true, false><<<blocks_for(total, 256), 256, 0, st>>>(S, ldS, hi, wi, Cout, k, bias, out, nullptr, total, sd);
        CK(cudaGetLastError());
        h->launches++;
    };
    // (overlapped stages: bias-free GEMM, bias once per output sample in the resample pass -- see run_decoder_wide)
    const bool ov1 = h->st[1] != p1, ov0 = h->st[0] != p0;
    // dec_conv_1 (p1) + GELU
    const int N1 = p1 * p1 * C2, N2 = p0 * p0 * C8;
    EpiParams ed; ed.bias = ov1 ? AF(h, h->zero_off) : AF(h, op.decb[0]);
    gemm<TA>(h, EPI_BIAS, dmod, C, op.decw[0], wb, N1, false, B * L, N1, C, ed, st);
    post(wb, N1, Hp, Wp, C2, p1, h->st[1], ov1 ? AF(h, op.decb[0]) : nullptr, g2);
    // dec_spectral_1 + GELU
    SpecView v2{g2, 1, nullptr, 1};
    run_spectral<TA>(h, op.fs1, v2, B, H1, W1, 1, true, g1, nullptr, st);
    // dec_conv_2 (p0) + GELU
    ed.bias = ov0 ? AF(h, h->zero_off) : AF(h, op.decb[1]);
    gemm<TA>(h, EPI_BIAS, g1, C1, op.decw[1], wb, N2, false, B * H1 * W1, N2, C1, ed, st);
    post(wb, N2, H1, W1, C8, p0, h->st[0], ov0 ? AF(h, op.decb[1]) : nullptr, g0);
    // dec_spectral_2 -> derivative field
    SpecView v0{g0, 1, nullptr, 1};
    run_spectral<TA>(h, op.fs2, v0, B, H, W, 0, false, nullptr, field, st);
}

void launch_emit_wide(tante_handle_s* h, const StepIO& io, int B, const RolloutState& rs, cudaStream_t st) {
    EmitParams ep{};
    ep.dfield = reinterpret_cast<const float*>(h->dfield.p);
    ep.K = h->K; ep.fi = h->cfg.frame_interval;
    ep.u_ring = io.input; ep.fcount = io.fcount;
    ep.n_arr = io.rollout ? rs.n_cur : reinterpret_cast<int*>(h->nbuf.p);
    ep.frames = io.frames; ep.n_cap = io.n_cap;
    ep.ptrs = io.rollout ? rs.ptrs : nullptr; ep.ring_out = io.ring_out; ep.cum = io.rollout ? rs.cum : nullptr; ep.n_roll = io.n_roll;
    ep.B = B; ep.D = h->D; ep.T = h->T; ep.HW = (long long)h->cfg.H * h->cfg.W;
    REQUIRE(ep.HW % 4 == 0, "H * W must be a multiple of 4");
    taylor_emit_kernel<<<dim3(blocks_for(ep.HW / 4, 256), (unsigned)h->D, (unsigned)B), 256, 0, st>>>(ep);
    CK(cudaGetLastError());
    h->launches++;
}

// One TANTE step (reference models/tante.py:125-176) as a launch sequence on `st`.
template <typename TA>
void run_step(tante_handle_s* h, const StepIO& io, int B, const RolloutState& rs, cudaStream_t st) {
    const int C = h->C, C1 = h->C1, C2 = h->C2, T = h->T, L = h->L, K = h->K, Hm = h->Hm;
    const PatchGeom& g = h->geom;
    const int tokens = B * T * L;
    float* x = reinterpret_cast<float*>(h->x.p);
    TA* ln = reinterpret_cast<TA*>(h->ln.p);
    TA* qkv = reinterpret_cast<TA*>(h->qkv.p);
    TA* att = reinterpret_cast<TA*>(h->att.p);
    TA* hid = reinterpret_cast<TA*>(h->hid.p);
    TA* a1 = reinterpret_cast<TA*>(h->a1.p);
    TA* a2 = reinterpret_cast<TA*>(h->a2.p);

    // --- encoder (enc_dec_cnn.py:217-229) + t_encode FiLM + s_emb + t_emb (tante.py:132-141) ---
    if (h->fno) {
        run_encoder_fno<TA>(h, io, B, st);
    } else if (h->wide) {
        run_encoder_wide<TA>(h, io, B, st);
    } else {
        const int P = g.k0 * g.k1 * g.k2;
        int WC = std::max(1, 128 / g.R1);
        WC = std::min(WC, g.Wp);
        const int K1 = g.k0 * g.k0 * g.D;
        const size_t smem = (size_t)(((g.D * P * (P * WC + 1) + 3) & ~3) + C1 * K1 + C1) * sizeof(float) +
                            (size_t)WC * g.R1 * C1 * sizeof(TA);
        dim3 grid(B * T * g.Hp, (g.Wp + WC - 1) / WC);
        const bool cached = io.rollout && rs.enc_count != nullptr;
        if (sizeof(TA) == 2 || C1 != 64) {      // (the FFMA patch kernel below is specialised for C/4 = 64)
            // tensor mode: enc_conv_1 as im2col (coalesced tiles, bf16 -- what the reference's autocast feeds its conv) + a
            // thin tcgen05 GEMM with the GELU in its epilogue; the FFMA kernel below is 64 erf-GELUs + 1024 FMAs per row
            const long long rows_in = (long long)tokens * g.R1;
            REQUIRE(rows_in < (1LL << 31), "input too large for the first-conv GEMM");
            TA* icols = reinterpret_cast<TA*>(h->icols.p);
            const int* el = cached ? rs.enc_list : nullptr;
            const int* ec = cached ? rs.enc_count : nullptr;
            const int* fc = cached ? nullptr : io.fcount;
            if (P >= 4) conv1_im2col_kernel<TA, 4><<<blocks_for(rows_in, kPatchRows), 128, 0, st>>>(io.input, g, icols, rows_in, el, ec, fc);
            else conv1_im2col_kernel<TA, 2><<<blocks_for(rows_in, kPatchRows), 128, 0, st>>>(io.input, g, icols, rows_in, el, ec, fc);
            CK(cudaGetLastError());
            h->launches++;
            EpiParams e1; e1.bias = AF(h, h->enc_b[0]);
            const bool prof = h->prof_on;
            if (cached) { e1.m_dev = rs.enc_count; e1.m_rows = L * g.R1; h->prof_on = false; }
            gemm<TA>(h, EPI_BIAS_GELU_ERF, icols, kHeadPad, h->enc_w1pad, a1, C1, false, (int)rows_in, C1, kHeadPad, e1, st);
            h->prof_on = prof;
        } else {
            patch_embed_conv1_kernel<TA><<<grid, 128, smem, st>>>(io.input, io.fcount, g, AF(h, h->enc_w[0]),
                                                                  AF(h, h->enc_b[0]), WC, a1, cached ? rs.enc_list : nullptr,
                                                                  cached ? rs.enc_count : nullptr);
            CK(cudaGetLastError());
            h->launches++;
        }
        EpiParams e2; e2.bias = AF(h, h->enc_b[1]);
        EpiParams e3; e3.bias = AF(h, h->enc_b[2]);
        if (cached) {
            // Rollout: only the frames that entered the window are encoded (their count lives on the device: the
            // GEMMs clip M to it); everything else comes out of the per-slot cache.  The encoder output of a frame
            // does not depend on its window position -- FiLM(t) and the embeddings are applied afterwards.
            e2.m_dev = rs.enc_count; e2.m_rows = L * g.R2;
            e3.m_dev = rs.enc_count; e3.m_rows = L;
            float* cnew = reinterpret_cast<float*>(h->qkv.p);       // scratch: free until the first QKV GEMM
            const bool prof = h->prof_on;
            h->prof_on = false;      // the row count of these two GEMMs lives on the device: keep them out of the FLOP tally
            gemm<TA>(h, EPI_BIAS_GELU_ERF, a1, g.k1 * g.k1 * C1, h->enc_w[1], a2, C2, false, tokens * g.R2, C2, g.k1 * g.k1 * C1, e2, st);
            gemm<TA>(h, EPI_BIAS, a2, g.k2 * g.k2 * C2, h->enc_w[2], cnew, C, true, tokens, C, g.k2 * g.k2 * C2, e3, st);
            h->prof_on = prof;
            const long long tot4 = (long long)tokens * (C / 4);
            REQUIRE(tot4 < (1LL << 31), "latent too large for the 32-bit indexing of the cached embed pass");
            embed_cached_kernel<<<(unsigned)std::min<long long>((tot4 + 255) / 256, 32LL * h->num_sms), 256, 0, st>>>(
                cnew, reinterpret_cast<float*>(h->enc_cache.p), rs.enc_map, io.fcount, AF(h, h->film_t_off), AF(h, h->s_emb),
                AF(h, h->t_emb), x, B, T, L, C, rs.act);
            CK(cudaGetLastError());
            h->launches++;
        } else {
            gemm<TA>(h, EPI_BIAS_GELU_ERF, a1, g.k1 * g.k1 * C1, h->enc_w[1], a2, C2, false, tokens * g.R2, C2, g.k1 * g.k1 * C1, e2, st);
            e3.film = AF(h, h->film_t_off); e3.s_emb = AF(h, h->s_emb); e3.t_emb = AF(h, h->t_emb);
            e3.T = T; e3.L = L; e3.ldr = C;
            // the embed epilogue writes the fp32 residual stream directly
            gemm<TA>(h, EPI_EMBED, a2, g.k2 * g.k2 * C2, h->enc_w[2], x, C, true, tokens, C, g.k2 * g.k2 * C2, e3, st);
        }
    }
    if (h->debug) CK(cudaMemcpyAsync(h->dbg_in.p, x, (size_t)tokens * C * sizeof(float), cudaMemcpyDeviceToDevice, st));

    float* rt = reinterpret_cast<float*>(h->rt.p);
    for (int o = 0; o < K; ++o) {
        const OrderPlan& op = h->orders[o];
        // --- Attn_Backbone.forward (attn_backbone.py:134-191) ---
        launch_propagator(h, x, x, B, 0, op, st);
        launch_propagator(h, x, x, B, 1, op, st);
        launch_propagator(h, x, x, B, 2, op, st);
        // In tensor mode every LayerNorm except the first one of an order is folded into the epilogue of the
        // residual GEMM that produces its input (EPI_BIAS_RESID_LN): the row is still on chip there.
        const bool kFuseLN = sizeof(TA) == 2 && C <= 256;      // (one CTA tile must hold the whole row)
        bool ln_ready = false;
        for (size_t li = 0; li < op.layers.size(); ++li) {
            const LayerPlan& lp = op.layers[li];
            if (lp.axis == 'C') {      // channel attention: its own width, its own LayerNorms (channel_axis.cuh)
                run_channel_layer<TA>(h, lp, x, x, tokens, st);
                ln_ready = false;
                continue;
            }
            // the next layer's LN1 rides in this layer's last epilogue -- unless that layer is a channel layer (other width)
            const bool nx_ok = li + 1 < op.layers.size() && op.layers[li + 1].axis != 'C';
            if (!ln_ready) launch_layernorm<TA>(h, x, lp.ln1w, lp.ln1b, ln, tokens, st);
            EpiParams eq; eq.bias = AF(h, lp.inb);
            gemm<TA>(h, EPI_BIAS, ln, C, lp.inw, qkv, 3 * C, false, tokens, 3 * C, C, eq, st);
            launch_attention<TA>(h, qkv, att, B, lp.axis, st);
            if constexpr (sizeof(TA) == 2) {
                if (h->fuse_tail && C == kBtC && h->Hm == C) {
                    const LayerPlan* nx = nx_ok ? &op.layers[li + 1] : nullptr;
                    launch_tail(h, lp, nx, att, x, x, ln, tokens, st);
                    ln_ready = nx != nullptr;
                    continue;
                }
            }
            EpiParams eo; eo.bias = AF(h, lp.outb); eo.resid = x; eo.ldr = C;
            if (kFuseLN) {
                eo.ln_gamma = AF(h, lp.ln2w); eo.ln_beta = AF(h, lp.ln2b); eo.ln_out = ln;
                gemm<TA>(h, EPI_BIAS_RESID_LN, att, C, lp.outw, x, C, true, tokens, C, C, eo, st);
            } else {
                gemm<TA>(h, EPI_BIAS_RESID, att, C, lp.outw, x, C, true, tokens, C, C, eo, st);
                launch_layernorm<TA>(h, x, lp.ln2w, lp.ln2b, ln, tokens, st);
            }
            EpiParams e0; e0.bias = AF(h, lp.m0b);
            gemm<TA>(h, EPI_BIAS_GELU_TANH, ln, C, lp.m0w, hid, Hm, false, tokens, Hm, C, e0, st);
            EpiParams e2; e2.bias = AF(h, lp.m2b); e2.resid = x; e2.ldr = C;
            if (kFuseLN && nx_ok && Hm == C) {      // (the LN-fused epilogue needs the K = C weight slice resident)
                const LayerPlan& nx = op.layers[li + 1];
                e2.ln_gamma = AF(h, nx.ln1w); e2.ln_beta = AF(h, nx.ln1b); e2.ln_out = ln;
                gemm<TA>(h, EPI_BIAS_RESID_LN, hid, Hm, lp.m2w, x, C, true, tokens, C, Hm, e2, st);
                ln_ready = true;
            } else {
                gemm<TA>(h, EPI_BIAS_RESID, hid, Hm, lp.m2w, x, C, true, tokens, C, Hm, e2, st);
                ln_ready = false;
            }
        }
        // --- head of order o (tante.py:147-154) ---
        float* d32 = reinterpret_cast<float*>(h->d32.p);
        TA* dmod = reinterpret_cast<TA*>(h->dmod.p);
        const long long LC = (long long)L * C;
        const long long tot = (long long)B * LC;
        const int eb = (int)((tot / 4 + 255) / 256);
        last_frame_kernel<TA><<<eb, 256, 0, st>>>(x, dmod, d32, B, T, LC);
        CK(cudaGetLastError());
        h->launches++;
        if (!h->cfg.deg) {
            TA* i1 = reinterpret_cast<TA*>(h->i1.p);
            TA* i2 = reinterpret_cast<TA*>(h->i2.p);
            EpiParams ei; ei.bias = AF(h, op.intb[0]);
            gemm<TA>(h, EPI_BIAS_RELU, dmod, C, op.intw[0], i1, C / 2, false, B * L, C / 2, C, ei, st);
            ei.bias = AF(h, op.intb[1]);
            gemm<TA>(h, EPI_BIAS_RELU, i1, C / 2, op.intw[1], i2, C / 4, false, B * L, C / 4, C / 2, ei, st);
            rt_reduce_kernel<TA><<<B, 256, 0, st>>>(i2, AF(h, op.intw[2]), AF(h, op.intb[2]), L, C / 4, io.out_T,
                                                    rt + (size_t)o * h->max_batch);
            CK(cudaGetLastError());
            h->launches++;
            float* fb = reinterpret_cast<float*>(h->filmbuf.p);
            film_params_kernel<<<B, 256, C * sizeof(float), st>>>(
                rt + (size_t)o * h->max_batch, 1.0f, AF(h, op.mod[0]), AF(h, op.mod[1]), AF(h, op.mod[2]),
                AF(h, op.mod[3]), AF(h, op.mod[4]), AF(h, op.mod[5]), AF(h, op.mod[6]), AF(h, op.mod[7]), C, fb);
            CK(cudaGetLastError());
            h->launches++;
            film_apply_kernel<TA><<<eb, 256, 0, st>>>(d32, fb, dmod, LC, C, tot);
            CK(cudaGetLastError());
            h->launches++;
        }
        if (h->fno) { run_decoder_fno<TA>(h, o, dmod, B, st); continue; }
        if (h->wide) { run_decoder_wide<TA>(h, o, dmod, B, st); continue; }
        TA* z1 = reinterpret_cast<TA*>(h->z1.p);
        TA* z2 = reinterpret_cast<TA*>(h->z2[o].p);
        EpiParams ed; ed.bias = AF(h, op.decb[0]);
        gemm<TA>(h, EPI_BIAS_GELU_ERF, dmod, C, op.decw[0], z1, g.k2 * g.k2 * C2, false, B * L, g.k2 * g.k2 * C2, C, ed, st);
        ed.bias = AF(h, op.decb[1]);
        gemm<TA>(h, EPI_BIAS_GELU_ERF, z1, C2, op.decw[1], z2, g.k1 * g.k1 * C1, false, B * L * g.R2, g.k1 * g.k1 * C1, C2, ed, st);
    }
    // --- step-size selection + fused Taylor head (tante.py:156-171) ---
    select_step_kernel<<<(B + 127) / 128, 128, 0, st>>>(rt, K, h->max_batch, B, h->cfg.deg, h->cfg.output_length,
                                                        io.per_sample, io.rollout ? (1 << 30) : io.n_cap,
                                                        io.rollout ? nullptr : io.R_t,
                                                        io.rollout ? nullptr : reinterpret_cast<int*>(h->nbuf.p), rs,
                                                        io.rollout ? 1 : 0);
    CK(cudaGetLastError());
    h->launches++;
    if (h->wide) launch_emit_wide(h, io, B, rs, st);
    else launch_head<TA>(h, io, B, rs, nullptr, st);
    if (io.rollout) {
        advance_state_kernel<<<1, 256, 0, st>>>(rs, B, h->cond_handle, h->use_cond);
        CK(cudaGetLastError());
        h->launches++;
    }
}

// ================================================================================================
// Training: forward with an activation tape + full backward (what torch autograd does for the reference:
// trainer/r_trainer.py:145-155, trainer/trainer.py:178-193).
// ================================================================================================
template <typename TA> inline TA* TP(DevBuf& b) { return reinterpret_cast<TA*>(b.p); }
inline float* FP(DevBuf& b) { return reinterpret_cast<float*>(b.p); }


template <typename TA, int ACT>
void launch_act_fwd(tante_handle_s* h, const TA* pre, TA* out, long long n, cudaStream_t st) {
    act_fwd_kernel<TA, ACT><<<blocks_for(n / 4, 256), 256, 0, st>>>(pre, out, n / 4);
    CK(cudaGetLastError());
    h->launches++;
}
template <typename TA, int ACT>
void launch_act_bwd(tante_handle_s* h, TA* g, const TA* pre, long long n, cudaStream_t st) {
    act_bwd_kernel<TA, ACT><<<blocks_for(n / 4, 256), 256, 0, st>>>(g, pre, n / 4);
    CK(cudaGetLastError());
    h->launches++;
}
template <typename TA>
void launch_colsum(tante_handle_s* h, const TA* x, int ld, long long M, int N, float* out, cudaStream_t st) {
    const unsigned gx = (unsigned)((N + 127) / 128);
    unsigned gy = (unsigned)std::max<long long>(1, std::min<long long>((M + 255) / 256, (4LL * h->num_sms + gx - 1) / gx));
    colsum_kernel<TA><<<dim3(gx, gy), 256, 0, st>>>(x, ld, M, N, out);
    CK(cudaGetLastError());
    h->launches++;
}
// dW[N][K] (+)= A[M][N]^T B[M][K] into the gradient arena
// `bias_out` (nullable): also db[N] += column sums of A (fused into the tensor-core kernel, else a colsum launch)
template <typename TA>
void wgrad(tante_handle_s* h, const TA* A, int lda, const TA* Bm, int ldb, float* out, long long M, int N, int K,
           cudaStream_t st, float* bias_out = nullptr) {
    {
        ProfScope ps(h, st, 2.0 * (double)M * N * K, 2, (double)M * (N + K) * sizeof(TA));
        if constexpr (sizeof(TA) == 2) {
            if (wgrad_tc_supported(M, N, K, K, lda, ldb, K)) {
                CK(launch_wgrad_tc(A, lda, Bm, ldb, out, K, M, N, K, K, h->num_sms, st, bias_out));
                h->launches++;
                return;
            }
        }
        CK((launch_wgrad_simt<TA, TA>(A, lda, Bm, ldb, out, K, M, N, K, h->num_sms, st)));
        h->launches++;
    }
    if (bias_out) launch_colsum<TA>(h, A, lda, M, N, bias_out, st);
}
// same with a zero-padded B operand: B is stored [M][Kb] (Kb % 64 == 0), only the first Kc columns of dW are kept
template <typename TA>
void wgrad_pad(tante_handle_s* h, const TA* A, int lda, int N, const TA* Bm, int ldb, int Kb, float* out, int ldc, int Kc,
               long long M, cudaStream_t st, float* bias_out = nullptr) {
    {
        ProfScope ps(h, st, 2.0 * (double)M * N * Kc, 2, (double)M * (N + Kb) * sizeof(TA));
        if constexpr (sizeof(TA) == 2) {
            if (wgrad_tc_supported(M, N, Kb, Kc, lda, ldb, ldc)) {
                CK(launch_wgrad_tc(A, lda, Bm, ldb, out, ldc, M, N, Kb, Kc, h->num_sms, st, bias_out));
                h->launches++;
                return;
            }
        }
        CK((launch_wgrad_simt<TA, TA>(A, lda, Bm, ldb, out, ldc, M, N, Kc, h->num_sms, st)));
        h->launches++;
    }
    if (bias_out) launch_colsum<TA>(h, A, lda, M, N, bias_out, st);
}
// dX = dY * W via the transposed packed weight (no bias)
template <typename TA>
void gemm_dx(tante_handle_s* h, const TA* A, int lda, int64_t wT_off, TA* out, int ldc, int M, int N, int K, cudaStream_t st) {
    EpiParams ep; ep.bias = AF(h, h->zero_off);
    REQUIRE(N <= 8192, "input-gradient GEMM wider than the zero-bias vector");
    if (sizeof(TA) == 2 && K > 1024) {
        // the tcgen05 GEMM keeps a K <= 1024 weight slice resident (K = 2048: first deconv of patch_scale 64): two K halves
        // accumulated through an fp32 scratch, then one conversion pass
        REQUIRE(ldc == N, "input-gradient GEMM: K not covered");
        if (h->kscratch.bytes < (size_t)M * N * 4) destroy_graphs(h);      // (a captured rollout may hold the old pointer)
        dev_alloc(h, h->kscratch, (size_t)M * N * 4);      // (training only: never inside a stream capture)
        float* v = FP(h->kscratch);
        gemm_bigk_f32(h, reinterpret_cast<const __nv_bfloat16*>(A), lda, wT_off, v, M, N, K, AF(h, h->zero_off), st);
        convert_kernel<TA><<<blocks_for((long long)M * N / 4, 256), 256, 0, st>>>(v, out, (long long)M * N / 4);
        CK(cudaGetLastError());
        h->launches++;
        return;
    }
    gemm<TA>(h, EPI_BIAS, A, lda, wT_off, out, ldc, sizeof(TA) == 4, M, N, K, ep, st);
}

// dX = (dY * W) o f'(pre): in tensor mode the activation derivative is applied in the GEMM epilogue (the saved
// pre-activation tile is TMA-loaded next to the accumulator); in the exact mode it is a separate elementwise pass.
// `out` and `pre` are both [M][N] contiguous.
template <typename TA, int ACT>
void gemm_dx_act(tante_handle_s* h, const TA* A, int lda, int64_t wT_off, TA* out, const TA* pre, int M, int N, int K,
                 cudaStream_t st) {
    // measured on B200 (Active Matter, M = 65536): fused epilogue 60 us vs 17 us GEMM + 26 us elementwise pass -- the
    // single 4 KB staging buffer per epilogue warp keeps too few bytes in flight, so the fusion is opt-in for now
    static const bool fuse = getenv("TANTE_FUSE_ACTGRAD") && atoi(getenv("TANTE_FUSE_ACTGRAD")) != 0;
    if (sizeof(TA) == 2 && fuse) {
        EpiParams ep; ep.bias = AF(h, h->zero_off);
        REQUIRE(N <= 8192, "input-gradient GEMM wider than the zero-bias vector");
        ep.mul_pre = pre; ep.ld_pre = N;
        const int epi = ACT == ACT_RELU ? EPI_MULGRAD_RELU : (ACT == ACT_GELU_ERF ? EPI_MULGRAD_GELU_ERF : EPI_MULGRAD_GELU_TANH);
        gemm<TA>(h, epi, A, lda, wT_off, out, N, false, M, N, K, ep, st);
    } else {
        gemm_dx<TA>(h, A, lda, wT_off, out, N, M, N, K, st);
        launch_act_bwd<TA, ACT>(h, out, pre, (long long)M * N, st);
    }
}

// Backward of one SpectralLayer (fno.cuh, "training"): x = the layer's saved input, g = the gradient of its output (after the
// GELU backward).  Accumulates the gradients of weight / w0 / bias, and writes the input gradient to the channels-last grid
// `dx` or accumulates it into the channels-first fp32 `gin` (first encoder layer); both null: parameters only.
template <typename TA>
void run_spectral_bwd(tante_handle_s* h, const SpecPlan& sp, const SpecView& x, const SpecView& g, long long N, int H, int W,
                      int level, TA* dx, float* gin, cudaStream_t st) {
    const int W0 = h->cfg.W, H0 = h->cfg.H, W1 = W0 / h->fp0;
    const float2* tw = reinterpret_cast<const float2*>(h->ftw.p);
    const float2* twW = level == 0 ? tw : tw + W0 + H0;
    const float2* twH = level == 0 ? tw + W0 : tw + W0 + H0 + W1;
    const int m1 = sp.wm1, m2 = sp.wm2, Cin = sp.Cin, Cout = sp.Cout;
    float2* A = reinterpret_cast<float2*>(h->fA.p);
    float2* Bc = reinterpret_cast<float2*>(h->fB.p);
    float2* Cc = reinterpret_cast<float2*>(h->fC.p);
    float2* Dd = reinterpret_cast<float2*>(h->fD.p);
    // gY = dft_h(dft_w(g))  -> Bc
    const long long rows_o = N * Cout * H, rows_i = N * Cin * H;
    spec_dft_w_kernel<TA><<<blocks_for(rows_o, 4), 128, 0, st>>>(g, Cout, H, W, m2, twW, A, rows_o);
    CK(cudaGetLastError());
    const long long ty = N * Cout * 2 * m1 * m2, tx = N * Cin * 2 * m1 * m2;
    spec_dft_h_kernel<<<blocks_for(ty, 256), 256, 0, st>>>(A, H, m1, m2, twH, Bc, ty);
    CK(cudaGetLastError());
    // X = dft_h(dft_w(x))  -> Cc (recomputed: two passes over the saved input)
    spec_dft_w_kernel<TA><<<blocks_for(rows_i, 4), 128, 0, st>>>(x, Cin, H, W, m2, twW, A, rows_i);
    CK(cudaGetLastError());
    spec_dft_h_kernel<<<blocks_for(tx, 256), 256, 0, st>>>(A, H, m1, m2, twH, Cc, tx);
    CK(cudaGetLastError());
    const long long tw_ = (long long)Cin * Cout * m1 * m2;
    spec_wt_grad_kernel<<<blocks_for(tw_, 256), 256, 0, st>>>(Cc, Bc, Cin, Cout, m1, m2, sp.wm2, sp.wm1, H, W, N,
                                                             reinterpret_cast<float2*>(GA(h, sp.w)), tw_);
    CK(cudaGetLastError());
    h->launches += 5;
    if (dx || gin) {
        spec_mix_adj_kernel<<<blocks_for(tx, 256), 256, 0, st>>>(Bc, reinterpret_cast<const float2*>(AF(h, sp.w)), Cin, Cout, m1, m2,
                                                                 sp.wm2, sp.wm1, H, W, A, tx);
        CK(cudaGetLastError());
        const long long ta = N * Cin * H * m2;
        spec_idft_h_kernel<<<blocks_for(ta, 256), 256, 0, st>>>(A, H, m1, m2, twH, Dd, ta);
        CK(cudaGetLastError());
        const long long to = N * Cin * H * W;
        if (gin) spec_in_bwd_kernel<TA, true><<<blocks_for(to, 256), 256, 0, st>>>(Dd, g, AF(h, sp.w0), Cin, Cout, H, W, m2, twW, nullptr, gin, to);
        else spec_in_bwd_kernel<TA, false><<<blocks_for(to, 256), 256, 0, st>>>(Dd, g, AF(h, sp.w0), Cin, Cout, H, W, m2, twW, dx, nullptr, to);
        CK(cudaGetLastError());
        h->launches += 3;
    }
    // 1x1 conv: dw0 = g^T x, db = colsum(g)
    if (x.mode == 1 && g.mode == 1 && Cin % 64 == 0 && Cout % 64 == 0) {
        wgrad<TA>(h, reinterpret_cast<const TA*>(g.p), Cout, reinterpret_cast<const TA*>(x.p), Cin, GA(h, sp.w0), N * H * W, Cout, Cin, st,
                  GA(h, sp.b0));
    } else {
        spec_w0_grad_kernel<TA><<<Cout * (Cin + 1), 256, 0, st>>>(g, x, Cin, Cout, H, W, N, GA(h, sp.w0), GA(h, sp.b0));
        CK(cudaGetLastError());
        h->launches++;
    }
}

template <typename TA>
void launch_ln_bwd(tante_handle_s* h, const TA* dy, const float* x, int64_t gamma, float* dxs, TA* dxb, float* dg, float* db,
                   long long rows, cudaStream_t st, const DropCfg& drop = DropCfg(), uint32_t site = 0, int width = 0) {
    const int C = width > 0 ? width : h->C;
    // persistent grid = exactly the resident blocks (3 per SM for C <= 256): no partial last wave
    const unsigned blocks = (unsigned)std::min<long long>((rows + 7) / 8, (C <= 256 ? 3LL : 2LL) * h->num_sms);
    if (drop.p > 0.f) {
        if (C <= 256) ln_bwd_kernel<TA, 2, true><<<blocks, 256, 0, st>>>(dy, x, AF(h, gamma), dxs, dxb, dg, db, rows, C, 1e-5f, drop, site);
        else ln_bwd_kernel<TA, 4, true><<<blocks, 256, 0, st>>>(dy, x, AF(h, gamma), dxs, dxb, dg, db, rows, C, 1e-5f, drop, site);
    } else {
        if (C <= 256) ln_bwd_kernel<TA, 2, false><<<blocks, 256, 0, st>>>(dy, x, AF(h, gamma), dxs, dxb, dg, db, rows, C, 1e-5f, drop, site);
        else ln_bwd_kernel<TA, 4, false><<<blocks, 256, 0, st>>>(dy, x, AF(h, gamma), dxs, dxb, dg, db, rows, C, 1e-5f, drop, site);
    }
    CK(cudaGetLastError());
    h->launches++;
}

template <typename TA>
void launch_attention_bwd(tante_handle_s* h, const TA* qkv, const TA* dout, TA* dqkv, int B, char axis, cudaStream_t st,
                          const DropCfg& drop = DropCfg(), uint32_t site = 0) {
    int S, inner; long long nseq;
    const int T = h->T, L = h->L, Hp = h->Hp, Wp = h->Wp;
    if (axis == 'T') { S = T; inner = L; nseq = (long long)B * L; }
    else if (axis == 'H') { S = Hp; inner = Wp; nseq = (long long)B * T * Wp; }
    else if (axis == 'W') { S = Wp; inner = 1; nseq = (long long)B * T * Hp; }
    else if (axis == 'L') { S = L; inner = 1; nseq = (long long)B * T; }               // (b t) (h w)
    else if (axis == 'Y') { S = T * Hp; inner = Wp; nseq = (long long)B * Wp; }        // (b w) (t h)
    else { S = T * L; inner = 1; nseq = B; }                                           // 'A': b (t h w)
    if (S > 64) {
        // composite axes and 65 .. 96-token axes: tiled recompute backward -- on mma.sync in the tensor mode without dropout
        // (attention_long_bwd_mma.cuh), on FFMA tiles otherwise (attention_long_bwd.cuh)
        cudaError_t e = cudaSuccess;
        if constexpr (sizeof(TA) == 2) {
            if (drop.p <= 0.f && launch_attention_long_bwd_mma(qkv, dout, dqkv, FP(h->att_stats), nseq, S, inner, h->cfg.n_head, h->C,
                                                               h->HD, axis == 'T', st, &e)) {
                CK(e);
                h->launches += 3;
                return;
            }
        }
        REQUIRE(launch_attention_long_bwd<TA>(qkv, dout, dqkv, FP(h->att_stats), nseq, S, inner, h->cfg.n_head, h->C, h->HD,
                                              axis == 'T', st, &e, drop, site),
                "attention backward: sequence shape not covered");
        CK(e);
        h->launches += 3;
        return;
    }
    if constexpr (sizeof(TA) == 2) {
        cudaError_t e = cudaSuccess;
        if (launch_attention_bwd_mma(qkv, dout, dqkv, nseq, S, inner, h->cfg.n_head, h->C, h->HD, axis == 'T', st, &e, drop, site)) {
            CK(e);
            h->launches++;
            return;
        }
    }
    const int G = std::max(1, 64 / S);
    const int R = G * S;
    const float scale = 1.0f / sqrtf((float)h->HD);
    dim3 grid((unsigned)((nseq + G - 1) / G), (unsigned)h->cfg.n_head);
#define ATTB(HDv)                                                                                              \
    do {                                                                                                       \
        const size_t smem = (size_t)(4 * R * (HDv + 1) + 2 * R * (S + 1)) * sizeof(float);                     \
        attention_bwd_kernel<TA, HDv><<<grid, 128, smem, st>>>(qkv, dout, dqkv, nseq, S, inner, h->cfg.n_head, \
                                                               h->C, axis == 'T', scale, G, drop, site);       \
    } while (0)
    if (h->HD == 32) ATTB(32); else if (h->HD == 64) ATTB(64); else ATTB(16);
#undef ATTB
    CK(cudaGetLastError());
    h->launches++;
}

void launch_propagator_bwd(tante_handle_s* h, const float* xin, float* dy, int B, int axis, const OrderPlan& op, cudaStream_t st) {
    int S; long long IC, outer;
    const int T = h->T, L = h->L, Hp = h->Hp, Wp = h->Wp, C = h->C;
    if (axis == 0) { S = Hp; IC = (long long)Wp * C; outer = (long long)B * T; }
    else if (axis == 1) { S = Wp; IC = C; outer = (long long)B * T * Hp; }
    else { S = T; IC = (long long)L * C; outer = B; }
    if (S <= 4 && (IC & 3) == 0) {
        const long long total = outer * (IC / 4);
        const unsigned grid = (unsigned)std::min<long long>((total + 255) / 256, 2LL * h->num_sms);
        const bool fast = h->cfg.precision == TANTE_PREC_BF16;
#define PSMALLB(TM, SM) propagator_small_bwd_kernel<TM, SM><<<grid, 256, 0, st>>>(xin, dy, S, IC, outer, AF(h, op.prop[axis][0]), \
            AF(h, op.prop[axis][1]), AF(h, op.prop[axis][2]), GA(h, op.prop[axis][0]), GA(h, op.prop[axis][1]),                \
            GA(h, op.prop[axis][2]), GA(h, op.prop[axis][3]))
        if (fast) PSMALLB(__nv_bfloat16, 4); else PSMALLB(float, 4);
#undef PSMALLB
        CK(cudaGetLastError());
        h->launches++;
        return;
    }
    if (h->cfg.precision == TANTE_PREC_BF16) {
        cudaError_t e = cudaSuccess;
        if (launch_propagator_bwd_mma(xin, dy, S, IC, outer, AF(h, op.prop[axis][0]), AF(h, op.prop[axis][1]),
                                      AF(h, op.prop[axis][2]), GA(h, op.prop[axis][0]), GA(h, op.prop[axis][1]),
                                      GA(h, op.prop[axis][2]), GA(h, op.prop[axis][3]), h->num_sms, st, &e)) {
            CK(e);
            h->launches++;
            return;
        }
    }
    if (S > 64) {      // 65 .. 96-token axes: the one-lane-per-column kernel (both S x S matrices in shared memory)
        REQUIRE(S <= kPropWideMaxS, "propagator backward: axis longer than 96 tokens");
        const long long nslabw = outer * ((IC + kPropWideCols - 1) / kPropWideCols);
        const unsigned gridw = (unsigned)std::min<long long>(nslabw, 2LL * h->num_sms);
        const size_t smw = prop_bwd_wide_smem(S);
        if (h->cfg.precision == TANTE_PREC_BF16) {
            CK(cudaFuncSetAttribute(propagator_bwd_wide_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smw));
            propagator_bwd_wide_kernel<__nv_bfloat16><<<gridw, 256, smw, st>>>(xin, dy, S, IC, outer, AF(h, op.prop[axis][0]), AF(h, op.prop[axis][1]),
                                                                              AF(h, op.prop[axis][2]), GA(h, op.prop[axis][0]), GA(h, op.prop[axis][1]),
                                                                              GA(h, op.prop[axis][2]), GA(h, op.prop[axis][3]));
        } else {
            CK(cudaFuncSetAttribute(propagator_bwd_wide_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smw));
            propagator_bwd_wide_kernel<float><<<gridw, 256, smw, st>>>(xin, dy, S, IC, outer, AF(h, op.prop[axis][0]), AF(h, op.prop[axis][1]),
                                                                      AF(h, op.prop[axis][2]), GA(h, op.prop[axis][0]), GA(h, op.prop[axis][1]),
                                                                      GA(h, op.prop[axis][2]), GA(h, op.prop[axis][3]));
        }
        CK(cudaGetLastError());
        h->launches++;
        return;
    }
    int S4 = (S + 3) & ~3;
    if (S4 > 4 && (S4 & (S4 - 1))) { int p2 = 8; while (p2 < S4) p2 <<= 1; S4 = p2; }
    const int CW = kPropBwdSlab / S4;
    const size_t smem = (size_t)(4 * (kPropBwdSlab + 4 * S4) + 3 * S4 * S4 + S4) * sizeof(float);
    const long long nslab = outer * ((IC + CW - 1) / CW);
    const unsigned grid = (unsigned)std::min<long long>(nslab, 2LL * h->num_sms);
    if (h->cfg.precision == TANTE_PREC_BF16)
        propagator_bwd_kernel<__nv_bfloat16><<<grid, 256, smem, st>>>(xin, dy, S, IC, outer, AF(h, op.prop[axis][0]), AF(h, op.prop[axis][1]),
                                                                     AF(h, op.prop[axis][2]), GA(h, op.prop[axis][0]), GA(h, op.prop[axis][1]),
                                                                     GA(h, op.prop[axis][2]), GA(h, op.prop[axis][3]));
    else
        propagator_bwd_kernel<float><<<grid, 256, smem, st>>>(xin, dy, S, IC, outer, AF(h, op.prop[axis][0]), AF(h, op.prop[axis][1]),
                                                             AF(h, op.prop[axis][2]), GA(h, op.prop[axis][0]), GA(h, op.prop[axis][1]),
                                                             GA(h, op.prop[axis][2]), GA(h, op.prop[axis][3]));
    CK(cudaGetLastError());
    h->launches++;
}

void free_tape(Tape& tp) {
    DevBuf* bufs[] = {&tp.cols, &tp.a1pre, &tp.a1act, &tp.a2pre, &tp.a2act, &tp.v, &tp.n_arr, &tp.cur, &tp.f0pre, &tp.f0act};
    for (DevBuf* b : bufs) b->free();
    for (OrderTape& ot : tp.ord) {
        DevBuf* ob[] = {&ot.P[0], &ot.P[1], &ot.P[2], &ot.dl, &ot.d32, &ot.dmod, &ot.i1, &ot.i2, &ot.rt, &ot.film, &ot.z1pre,
                        &ot.z1act, &ot.z2pre, &ot.z2act, &ot.f0pre, &ot.f0act};
        for (DevBuf* b : ob) b->free();
        for (auto* v : {&ot.X, &ot.ln1, &ot.qkv, &ot.att, &ot.ln2, &ot.hpre, &ot.hact})
            for (auto& b : *v) b.free();
    }
    tp.ord.clear();
    tp.B = 0;
    tp.valid = false;
}

void tape_alloc(tante_handle_s* h, Tape& tp, int B) {
    if (tp.B >= B && !tp.ord.empty()) return;
    const size_t es = h->cfg.precision == TANTE_PREC_BF16 ? 2 : 4;
    const size_t tokens = (size_t)B * h->T * h->L;
    const size_t BL = (size_t)B * h->L;
    const int C = h->C, C1 = h->C1, C2 = h->C2;
    const PatchGeom& g = h->geom;
    dev_alloc(h, tp.cols, (h->overlap ? (size_t)wide_dims(h, B).rows1 : tokens * g.R1) * (size_t)std::max(kHeadPad, h->wide ? h->K1pad : 0) * es);
    dev_alloc(h, tp.a1pre, tokens * g.R1 * C1 * es);
    dev_alloc(h, tp.a1act, tokens * g.R1 * C1 * es);
    // fno: the C/2 grid sits at the H1 x W1 resolution (R1 rows per token), and there is a C/8 grid at full resolution
    const size_t r2 = h->fno ? g.R1 : g.R2;
    dev_alloc(h, tp.a2pre, tokens * r2 * C2 * es);
    dev_alloc(h, tp.a2act, tokens * r2 * C2 * es);
    if (h->fno) {
        const size_t f0 = (size_t)B * h->T * h->cfg.H * h->cfg.W * (C / 8) * es;
        dev_alloc(h, tp.f0pre, f0);
        dev_alloc(h, tp.f0act, f0);
    }
    dev_alloc(h, tp.v, tokens * C * 4);
    dev_alloc(h, tp.n_arr, (size_t)B * 4);
    dev_alloc(h, tp.cur, (size_t)B * 4);
    tp.ord.resize(h->K);
    for (int o = 0; o < h->K; ++o) {
        OrderTape& ot = tp.ord[o];
        const size_t nl = h->orders[o].layers.size();
        for (int a = (o == 0 ? 0 : 1); a < 3; ++a) dev_alloc(h, ot.P[a], tokens * C * 4);
        ot.X.resize(2 * nl + 1);
        for (auto& b : ot.X) dev_alloc(h, b, tokens * C * 4);
        ot.ln1.resize(nl); ot.qkv.resize(nl); ot.att.resize(nl); ot.ln2.resize(nl); ot.hpre.resize(nl); ot.hact.resize(nl);
        for (size_t i = 0; i < nl; ++i) {
            dev_alloc(h, ot.ln1[i], tokens * C * es);
            dev_alloc(h, ot.qkv[i], tokens * 3 * C * es);
            dev_alloc(h, ot.att[i], tokens * C * es);
            dev_alloc(h, ot.ln2[i], tokens * C * es);
            dev_alloc(h, ot.hpre[i], tokens * h->Hm * es);
            dev_alloc(h, ot.hact[i], tokens * h->Hm * es);
        }
        dev_alloc(h, ot.dl, BL * C * es);
        dev_alloc(h, ot.d32, BL * C * 4);
        if (!h->cfg.deg) {
            dev_alloc(h, ot.dmod, BL * C * es);
            dev_alloc(h, ot.i1, BL * (C / 2) * es);
            dev_alloc(h, ot.i2, BL * (C / 4) * es);
            dev_alloc(h, ot.rt, (size_t)B * 4);
            dev_alloc(h, ot.film, (size_t)B * 2 * C * 4);
        }
        dev_alloc(h, ot.z1pre, BL * r2 * C2 * es);
        dev_alloc(h, ot.z1act, BL * r2 * C2 * es);
        if (h->fno) {
            const size_t f0 = (size_t)B * h->cfg.H * h->cfg.W * (C / 8) * es;
            dev_alloc(h, ot.f0pre, f0);
            dev_alloc(h, ot.f0act, f0);
        }
        dev_alloc(h, ot.z2pre, BL * g.R1 * C1 * es);
        dev_alloc(h, ot.z2act, BL * g.R1 * C1 * es);
    }
    tp.B = B;
}

void backward_alloc(tante_handle_s* h, int B) {
    if (h->fno) {      // sized by tante_reserve's max_batch, which may have grown since the last call
        dev_alloc(h, h->fC, h->f_ca * 8);
        dev_alloc(h, h->fD, h->f_ca * 8);
    }
    if (h->bw_batch >= B) return;
    const size_t es = h->cfg.precision == TANTE_PREC_BF16 ? 2 : 4;
    const size_t tokens = (size_t)B * h->T * h->L;
    const size_t BL = (size_t)B * h->L;
    const int C = h->C, C1 = h->C1, C2 = h->C2;
    const PatchGeom& g = h->geom;
    const int NO = g.k0 * g.k0 * h->D;
    dev_alloc(h, h->garena, (size_t)h->garena_elems * 4);
    dev_alloc(h, h->dxs, tokens * C * 4);
    dev_alloc(h, h->dxb, tokens * C * es);      // bf16 mirror of the gradient stream; in the exact mode: its dropout-masked copy
    dev_alloc(h, h->g1, tokens * std::max(C, h->Hm) * es);
    dev_alloc(h, h->g2, tokens * C * es);
    dev_alloc(h, h->gq, tokens * std::max(3 * C, g.R2 * C2) * es);
    dev_alloc(h, h->ga1, tokens * g.R1 * C1 * es);
    (void)NO;
    dev_alloc(h, h->cols, tokens * g.R1 * kHeadPad * es);
    dev_alloc(h, h->hz, (size_t)h->K * BL * g.R1 * C1 * es);
    dev_alloc(h, h->hG, (size_t)h->K * BL * g.R1 * (size_t)std::max(kHeadPad, h->wide ? h->NOpad : 0) * es);
    dev_alloc(h, h->hz1, BL * g.R2 * C2 * es);
    dev_alloc(h, h->hd, BL * C * es);
    dev_alloc(h, h->hi1, BL * (C / 2) * es);
    dev_alloc(h, h->hi2, BL * (C / 4) * es);
    dev_alloc(h, h->dfilm, (size_t)std::max(B, h->T) * 2 * C * 4);
    dev_alloc(h, h->dcond, (size_t)B * 4);
    if (h->fno) {
        const size_t NI = (size_t)B * h->T, HW = (size_t)h->cfg.H * h->cfg.W, HW1 = HW / (h->fp0 * h->fp0);
        dev_alloc(h, h->fgr0, NI * HW * (C / 8) * es);
        dev_alloc(h, h->fgr1, NI * HW1 * C1 * es);
        dev_alloc(h, h->fgr2, NI * HW1 * C2 * es);
    }
    if (h->chan) {
        // channel-axis backward: chunks of 512 latent tokens (131072 rows of width E; ~10 KB of scratch per row in the exact mode)
        h->chanb_tokens = (int)std::min<size_t>(tokens, 512);
        if (const char* e = getenv("TANTE_CHAN_CHUNK")) h->chanb_tokens = std::max(1, std::min(h->chanb_tokens, atoi(e)));
        const size_t rows = (size_t)h->chanb_tokens * C, E = h->chanE, Hc = h->chanHc;
        dev_alloc(h, h->cb_x0, rows * E * 4);
        dev_alloc(h, h->cb_xm, rows * E * 4);
        dev_alloc(h, h->cb_gx, rows * E * 4);
        dev_alloc(h, h->cb_ln1, rows * E * es);
        dev_alloc(h, h->cb_qkv, rows * 3 * E * es);
        dev_alloc(h, h->cb_att, rows * E * es);
        dev_alloc(h, h->cb_ln2, rows * E * es);
        dev_alloc(h, h->cb_hpre, rows * Hc * es);
        dev_alloc(h, h->cb_hact, rows * Hc * es);
        dev_alloc(h, h->cb_gxb, rows * E * es);
        dev_alloc(h, h->cb_g1, rows * std::max(E, Hc) * es);
        dev_alloc(h, h->cb_g2, rows * E * es);
        dev_alloc(h, h->cb_gq, rows * 3 * E * es);
        dev_alloc(h, h->cb_hh, rows * (E / 4) * es);
        dev_alloc(h, h->cb_stats, rows * h->cfg.n_head * 2 * 4);
    }
    if (h->long_axes) dev_alloc(h, h->att_stats, tokens * h->cfg.n_head * 2 * 4);      // LSE + delta per (token, head)
    if (!h->udesc_dev.p) {
        std::vector<UnpackDesc> ud;
        for (const Param& p : h->params) {
            UnpackDesc d;
            d.src_off = p.goff; d.dst_off = p.flat_off; d.numel = p.numel; d.mode = p.gmode; d.d0 = p.gd0; d.d1 = p.gd1; d.k = p.gk;
            ud.push_back(d);
        }
        dev_alloc(h, h->udesc_dev, ud.size() * sizeof(UnpackDesc));
        CK(cudaMemcpy(h->udesc_dev.p, ud.data(), ud.size() * sizeof(UnpackDesc), cudaMemcpyHostToDevice));
    }
    h->bw_batch = B;
}

// One TANTE step in training mode: same arithmetic as run_step, every activation the backward needs is kept.
// Window of a training call as a frame table (tante_train_forward_win / tante_backward_win)
struct TrainWin {
    FrameTab in;                  // forward: the T window frames, offsets relative to `input`
    long long frames_bs = 0;      // batch stride of the emitted frames (0: contiguous)
    int n_lim = 0;                // per-sample cursor mode (in.cur != null): frames a sample needs; it emits nothing once it has them
};

template <typename TA>
void run_step_train(tante_handle_s* h, Tape& tp, const float* input, int B, float out_T, int n_cap, float* frames,
                    float* R_t, cudaStream_t st, const TrainWin* win = nullptr) {
    const int C = h->C, C1 = h->C1, C2 = h->C2, T = h->T, L = h->L, K = h->K, Hm = h->Hm;
    const PatchGeom& g = h->geom;
    const int tokens = B * T * L;
    constexpr bool kTensor = sizeof(TA) == 2;
    tp.drop = make_drop_cfg(h->drop_p, h->drop_seed);
    const DropCfg& drop = tp.drop;
    // --- encoder ---
    if (h->fno) {
        // enc_FNO.forward (enc_dec_fno.py:254-272): spectral layer -> GELU -> patch conv -> GELU -> spectral layer -> GELU -> patch conv;
        // every pre-activation / activation grid is kept
        REQUIRE(!win, "windowed BPTT is not available with enc_dec_type='fno'");
        const int H = h->cfg.H, W = h->cfg.W, p0 = h->fp0, p1 = h->fp1, H1 = H / p0, W1 = W / p0, C8 = C / 8;
        const long long NI = (long long)B * T;
        SpecView v0{input, 0, nullptr, T};
        run_spectral<TA>(h, h->fes1, v0, NI, H, W, 0, false, TP<TA>(tp.f0pre), nullptr, st);
        launch_act_fwd<TA, ACT_GELU_ERF>(h, TP<TA>(tp.f0pre), TP<TA>(tp.f0act), NI * H * W * C8, st);
        EpiParams e1; e1.bias = AF(h, h->enc_b[0]);
        conv_cl_gemm<TA>(h, EPI_BIAS, TP<TA>(tp.f0act), H, W, C8, p0, h->enc_w[0], tp.a1pre.p, C1, false, NI, e1, st, h->st[0]);
        launch_act_fwd<TA, ACT_GELU_ERF>(h, TP<TA>(tp.a1pre), TP<TA>(tp.a1act), NI * H1 * W1 * C1, st);
        SpecView v1{tp.a1act.p, 1, nullptr, 1};
        run_spectral<TA>(h, h->fes2, v1, NI, H1, W1, 1, false, TP<TA>(tp.a2pre), nullptr, st);
        launch_act_fwd<TA, ACT_GELU_ERF>(h, TP<TA>(tp.a2pre), TP<TA>(tp.a2act), NI * H1 * W1 * C2, st);
        EpiParams e2; e2.bias = AF(h, h->enc_b[1]);
        conv_cl_gemm<TA>(h, EPI_BIAS, TP<TA>(tp.a2act), H1, W1, C2, p1, h->enc_w[1], tp.v.p, C, true, NI, e2, st, h->st[1]);
        embed_fwd_kernel<<<blocks_for((long long)tokens * C / 4, 256), 256, 0, st>>>(
            FP(tp.v), AF(h, h->film_t_off), AF(h, h->s_emb), AF(h, h->t_emb), FP(tp.ord[0].P[0]), tokens, T, L, C);
        CK(cudaGetLastError());
        h->launches++;
    } else if (h->wide) {
        // patch_scale 16 / 32 / 64 (wide_patch.cuh): natural-order stages, window gathers + GEMMs; the first patch matrix and every
        // pre-activation / activation grid are kept for the backward
        REQUIRE(!win, "windowed BPTT is not available at patch_scale >= 16 / with overlap");
        const int H = h->cfg.H, W = h->cfg.W, D = h->D;
        TA* wb = TP<TA>(h->wbuf);
        TA* cg = TP<TA>(h->cgrid);
        const WideDims wd = wide_dims(h, B);
        const int H1 = wd.H1, W1 = wd.W1, H2 = wd.H2, W2 = wd.W2;
        const long long NI = (long long)B * T;
        REQUIRE(wd.rows1 < (1LL << 31) && wd.rows2 < (1LL << 31) && wd.rows3 < (1LL << 31), "input too large for the wide conv GEMMs");
        auto pool = [&](const TA* in, int Hc, int Wc, int Cc, int Ho, int Wo, TA* out, float* out32) {
            const long long total4 = NI * Ho * Wo * Cc / 4;
            if (out32) wide_pool_kernel<TA, false, true><<<blocks_for(total4, 256), 256, 0, st>>>(in, Hc, Wc, Cc, Ho, Wo, nullptr, out32, total4);
            else wide_pool_kernel<TA, false, false><<<blocks_for(total4, 256), 256, 0, st>>>(in, Hc, Wc, Cc, Ho, Wo, out, nullptr, total4);
            CK(cudaGetLastError());
            h->launches++;
        };
        const long long total = wd.rows1 * h->K1pad;
        wide_im2col_cf_kernel<TA><<<blocks_for(total, 256), 256, 0, st>>>(input, nullptr, T, D, H, W, g.k0, (g.k0 - 1) / 2, h->K1pad,
                                                                         TP<TA>(tp.cols), total, h->st[0], wd.Hc1, wd.Wc1);
        CK(cudaGetLastError());
        h->launches++;
        EpiParams e1; e1.bias = AF(h, h->enc_b[0]);
        gemm<TA>(h, EPI_BIAS, TP<TA>(tp.cols), h->K1pad, h->enc_w1wide, wd.pool1 ? (void*)cg : tp.a1pre.p, C1, false, (int)wd.rows1, C1,
                 h->K1pad, e1, st);
        if (wd.pool1) pool(cg, wd.Hc1, wd.Wc1, C1, H1, W1, TP<TA>(tp.a1pre), nullptr);
        launch_act_fwd<TA, ACT_GELU_ERF>(h, TP<TA>(tp.a1pre), TP<TA>(tp.a1act), NI * H1 * W1 * C1, st);
        const int K2 = g.k1 * g.k1 * C1, K3 = g.k2 * g.k2 * C2;
        wide_im2col_cl_kernel<TA><<<blocks_for(wd.rows2 * K2 / 4, 256), 256, 0, st>>>(TP<TA>(tp.a1act), H1, W1, C1, g.k1, (g.k1 - 1) / 2, wb,
                                                                                     wd.rows2 * K2 / 4, h->st[1], wd.Hc2, wd.Wc2);
        CK(cudaGetLastError());
        h->launches++;
        EpiParams e2; e2.bias = AF(h, h->enc_b[1]);
        gemm<TA>(h, EPI_BIAS, wb, K2, h->enc_w[1], wd.pool2 ? (void*)cg : tp.a2pre.p, C2, false, (int)wd.rows2, C2, K2, e2, st);
        if (wd.pool2) pool(cg, wd.Hc2, wd.Wc2, C2, H2, W2, TP<TA>(tp.a2pre), nullptr);
        launch_act_fwd<TA, ACT_GELU_ERF>(h, TP<TA>(tp.a2pre), TP<TA>(tp.a2act), NI * H2 * W2 * C2, st);
        wide_im2col_cl_kernel<TA><<<blocks_for(wd.rows3 * K3 / 4, 256), 256, 0, st>>>(TP<TA>(tp.a2act), H2, W2, C2, g.k2, (g.k2 - 1) / 2, wb,
                                                                                     wd.rows3 * K3 / 4, h->st[2], wd.Hc3, wd.Wc3);
        CK(cudaGetLastError());
        h->launches++;
        EpiParams e3; e3.bias = AF(h, h->enc_b[2]);
        if (wd.pool3) {
            if (kTensor && K3 > 1024) {      // (patch_scale 64: K blocks through the fp32 scratch of tante_reserve, as in run_encoder_wide)
                REQUIRE((size_t)wd.rows3 * C * 4 <= h->kscratch.bytes, "split-K conv: scratch not reserved");
                float* acc = FP(h->kscratch);
                gemm_bigk_f32(h, reinterpret_cast<const __nv_bfloat16*>(wb), K3, h->enc_w[2], acc, (int)wd.rows3, C, K3, e3.bias, st);
                f32_to_ta_kernel<TA, false><<<blocks_for(wd.rows3 * C / 4, 256), 256, 0, st>>>(acc, cg, wd.rows3 * C / 4);
                CK(cudaGetLastError());
                h->launches++;
            } else {
                gemm<TA>(h, EPI_BIAS, wb, K3, h->enc_w[2], cg, C, false, (int)wd.rows3, C, K3, e3, st);
            }
            pool(cg, wd.Hc3, wd.Wc3, C, h->Hp, h->Wp, nullptr, FP(tp.v));
        } else if (kTensor && K3 > 1024) {      // (K = 2048 at patch_scale 64: K blocks, as in run_encoder_wide)
            gemm_bigk_f32(h, reinterpret_cast<const __nv_bfloat16*>(wb), K3, h->enc_w[2], FP(tp.v), tokens, C, K3, e3.bias, st);
        } else {
            gemm<TA>(h, EPI_BIAS, wb, K3, h->enc_w[2], tp.v.p, C, true, tokens, C, K3, e3, st);
        }
        embed_fwd_kernel<<<blocks_for((long long)tokens * C / 4, 256), 256, 0, st>>>(
            FP(tp.v), AF(h, h->film_t_off), AF(h, h->s_emb), AF(h, h->t_emb), FP(tp.ord[0].P[0]), tokens, T, L, C);
        CK(cudaGetLastError());
        h->launches++;
    } else {
        // enc_conv_1 as im2col (kept for the weight gradient) + GEMM over the zero-padded patch matrix
        const long long rows_in = (long long)tokens * g.R1;
        REQUIRE(rows_in < (1LL << 31), "input too large for the first-conv GEMM");
        const FrameTab ft = win ? win->in : FrameTab();
        if (g.k0 * g.k1 * g.k2 >= 4) conv1_im2col_kernel<TA, 4><<<blocks_for(rows_in, kPatchRows), 128, 0, st>>>(input, g, TP<TA>(tp.cols), rows_in, nullptr, nullptr, nullptr, ft);
        else conv1_im2col_kernel<TA, 2><<<blocks_for(rows_in, kPatchRows), 128, 0, st>>>(input, g, TP<TA>(tp.cols), rows_in, nullptr, nullptr, nullptr, ft);
        CK(cudaGetLastError());
        h->launches++;
        EpiParams e1; e1.bias = AF(h, h->enc_b[0]);
        gemm<TA>(h, EPI_BIAS, TP<TA>(tp.cols), kHeadPad, h->enc_w1pad, tp.a1pre.p, C1, false, (int)rows_in, C1, kHeadPad, e1, st);
        launch_act_fwd<TA, ACT_GELU_ERF>(h, TP<TA>(tp.a1pre), TP<TA>(tp.a1act), (long long)tokens * g.R1 * C1, st);
        EpiParams e2; e2.bias = AF(h, h->enc_b[1]);
        gemm<TA>(h, EPI_BIAS, TP<TA>(tp.a1act), g.k1 * g.k1 * C1, h->enc_w[1], tp.a2pre.p, C2, false, tokens * g.R2, C2,
                 g.k1 * g.k1 * C1, e2, st);
        launch_act_fwd<TA, ACT_GELU_ERF>(h, TP<TA>(tp.a2pre), TP<TA>(tp.a2act), (long long)tokens * g.R2 * C2, st);
        EpiParams e3; e3.bias = AF(h, h->enc_b[2]);
        gemm<TA>(h, EPI_BIAS, TP<TA>(tp.a2act), g.k2 * g.k2 * C2, h->enc_w[2], tp.v.p, C, true, tokens, C, g.k2 * g.k2 * C2, e3, st);
        embed_fwd_kernel<<<blocks_for((long long)tokens * C / 4, 256), 256, 0, st>>>(
            FP(tp.v), AF(h, h->film_t_off), AF(h, h->s_emb), AF(h, h->t_emb), FP(tp.ord[0].P[0]), tokens, T, L, C);
        CK(cudaGetLastError());
        h->launches++;
    }
    float* rt = reinterpret_cast<float*>(h->rt.p);
    for (int o = 0; o < K; ++o) {
        const OrderPlan& op = h->orders[o];
        OrderTape& ot = tp.ord[o];
        const float* pin = o == 0 ? FP(ot.P[0]) : FP(tp.ord[o - 1].X.back());
        launch_propagator(h, pin, FP(ot.P[1]), B, 0, op, st);
        launch_propagator(h, FP(ot.P[1]), FP(ot.P[2]), B, 1, op, st);
        launch_propagator(h, FP(ot.P[2]), FP(ot.X[0]), B, 2, op, st);
        bool ln_ready = false;
        const size_t nl = op.layers.size();
        for (size_t li = 0; li < nl; ++li) {
            const LayerPlan& lp = op.layers[li];
            float* x_in = FP(ot.X[2 * li]);
            float* x_mid = FP(ot.X[2 * li + 1]);
            float* x_out = FP(ot.X[2 * li + 2]);
            if (lp.axis == 'C') {
                // channel attention: only the layer's fp32 input is kept -- the backward recomputes the block chunk by chunk
                REQUIRE(drop.p <= 0.f, "dropout with an attention axis C layer is not implemented");
                run_channel_layer<TA>(h, lp, x_in, x_out, tokens, st);
                ln_ready = false;
                continue;
            }
            const bool nx_ok = li + 1 < nl && op.layers[li + 1].axis != 'C';
            if (!ln_ready) launch_layernorm<TA>(h, x_in, lp.ln1w, lp.ln1b, TP<TA>(ot.ln1[li]), tokens, st);
            EpiParams eq; eq.bias = AF(h, lp.inb);
            gemm<TA>(h, EPI_BIAS, TP<TA>(ot.ln1[li]), C, lp.inw, ot.qkv[li].p, 3 * C, false, tokens, 3 * C, C, eq, st);
            launch_attention<TA>(h, TP<TA>(ot.qkv[li]), TP<TA>(ot.att[li]), B, lp.axis, st, drop, drop_site(o, (int)li, 0));
            if constexpr (kTensor) {
                if (h->fuse_tail && C == kBtC && h->Hm == C) {
                    const LayerPlan* nx = nx_ok ? &op.layers[li + 1] : nullptr;
                    launch_tail(h, lp, nx, TP<TA>(ot.att[li]), x_in, x_out, nx ? TP<TA>(ot.ln1[li + 1]) : nullptr, tokens, st,
                                x_mid, TP<TA>(ot.ln2[li]), TP<TA>(ot.hpre[li]), TP<TA>(ot.hact[li]), drop,
                                drop_site(o, (int)li, 1), drop_site(o, (int)li, 2));
                    ln_ready = nx != nullptr;
                    continue;
                }
            }
            if (kTensor && drop.p > 0.f) {
                // Tensor mode with dropout outside the fused tail (mlp_ratio != 1, embed_dim 512, TANTE_FUSE_TAIL=0): the tcgen05 GEMM
                // epilogues carry no mask generator, so each residual branch is a plain GEMM into a bf16 scratch followed by one
                // pass  x <- x + mask * branch  (what autocast + nn.Dropout do in the reference); LayerNorms as their own passes.
                TA* br = TP<TA>(h->hid);
                const long long n4 = (long long)tokens * C / 4;
                EpiParams eb; eb.bias = AF(h, lp.outb);
                gemm<TA>(h, EPI_BIAS, TP<TA>(ot.att[li]), C, lp.outw, br, C, false, tokens, C, C, eb, st);
                resid_drop_kernel<TA><<<blocks_for(n4, 256), 256, 0, st>>>(br, x_in, x_mid, n4, drop, drop_site(o, (int)li, 1));
                CK(cudaGetLastError());
                h->launches++;
                launch_layernorm<TA>(h, x_mid, lp.ln2w, lp.ln2b, TP<TA>(ot.ln2[li]), tokens, st);
                EpiParams eh; eh.bias = AF(h, lp.m0b);
                gemm<TA>(h, EPI_BIAS, TP<TA>(ot.ln2[li]), C, lp.m0w, ot.hpre[li].p, Hm, false, tokens, Hm, C, eh, st);
                launch_act_fwd<TA, ACT_GELU_TANH>(h, TP<TA>(ot.hpre[li]), TP<TA>(ot.hact[li]), (long long)tokens * Hm, st);
                eb.bias = AF(h, lp.m2b);
                gemm<TA>(h, EPI_BIAS, TP<TA>(ot.hact[li]), Hm, lp.m2w, br, C, false, tokens, C, Hm, eb, st);
                resid_drop_kernel<TA><<<blocks_for(n4, 256), 256, 0, st>>>(br, x_mid, x_out, n4, drop, drop_site(o, (int)li, 2));
                CK(cudaGetLastError());
                h->launches++;
                ln_ready = false;
                continue;
            }
            EpiParams eo; eo.bias = AF(h, lp.outb); eo.resid = x_in; eo.ldr = C;
            eo.drop = drop; eo.drop_site = drop_site(o, (int)li, 1);
            if (kTensor && C <= 256) {
                eo.ln_gamma = AF(h, lp.ln2w); eo.ln_beta = AF(h, lp.ln2b); eo.ln_out = ot.ln2[li].p;
                gemm<TA>(h, EPI_BIAS_RESID_LN, TP<TA>(ot.att[li]), C, lp.outw, x_mid, C, true, tokens, C, C, eo, st);
            } else {
                gemm<TA>(h, EPI_BIAS_RESID, TP<TA>(ot.att[li]), C, lp.outw, x_mid, C, true, tokens, C, C, eo, st);
                launch_layernorm<TA>(h, x_mid, lp.ln2w, lp.ln2b, TP<TA>(ot.ln2[li]), tokens, st);
            }
            EpiParams e0; e0.bias = AF(h, lp.m0b);
            gemm<TA>(h, EPI_BIAS, TP<TA>(ot.ln2[li]), C, lp.m0w, ot.hpre[li].p, Hm, false, tokens, Hm, C, e0, st);
            launch_act_fwd<TA, ACT_GELU_TANH>(h, TP<TA>(ot.hpre[li]), TP<TA>(ot.hact[li]), (long long)tokens * Hm, st);
            EpiParams e2; e2.bias = AF(h, lp.m2b); e2.resid = x_mid; e2.ldr = C;
            e2.drop = drop; e2.drop_site = drop_site(o, (int)li, 2);
            if (kTensor && C <= 256 && nx_ok && Hm == C) {      // (the LN-fused epilogue needs the K = C weight slice resident)
                const LayerPlan& nx = op.layers[li + 1];
                e2.ln_gamma = AF(h, nx.ln1w); e2.ln_beta = AF(h, nx.ln1b); e2.ln_out = ot.ln1[li + 1].p;
                gemm<TA>(h, EPI_BIAS_RESID_LN, TP<TA>(ot.hact[li]), Hm, lp.m2w, x_out, C, true, tokens, C, Hm, e2, st);
                ln_ready = true;
            } else {
                gemm<TA>(h, EPI_BIAS_RESID, TP<TA>(ot.hact[li]), Hm, lp.m2w, x_out, C, true, tokens, C, Hm, e2, st);
                ln_ready = false;
            }
        }
        // --- head of order o ---
        const long long LC = (long long)L * C;
        const long long tot = (long long)B * LC;
        const int eb = (int)((tot / 4 + 255) / 256);
        last_frame_kernel<TA><<<eb, 256, 0, st>>>(FP(ot.X.back()), TP<TA>(ot.dl), FP(ot.d32), B, T, LC);
        CK(cudaGetLastError());
        h->launches++;
        TA* dmod = TP<TA>(ot.dl);
        if (!h->cfg.deg) {
            EpiParams ei; ei.bias = AF(h, op.intb[0]);
            gemm<TA>(h, EPI_BIAS_RELU, TP<TA>(ot.dl), C, op.intw[0], ot.i1.p, C / 2, false, B * L, C / 2, C, ei, st);
            ei.bias = AF(h, op.intb[1]);
            gemm<TA>(h, EPI_BIAS_RELU, TP<TA>(ot.i1), C / 2, op.intw[1], ot.i2.p, C / 4, false, B * L, C / 4, C / 2, ei, st);
            rt_reduce_kernel<TA><<<B, 256, 0, st>>>(TP<TA>(ot.i2), AF(h, op.intw[2]), AF(h, op.intb[2]), L, C / 4, out_T,
                                                    rt + (size_t)o * h->max_batch);
            CK(cudaGetLastError());
            h->launches++;
            CK(cudaMemcpyAsync(ot.rt.p, rt + (size_t)o * h->max_batch, (size_t)B * 4, cudaMemcpyDeviceToDevice, st));
            film_params_kernel<<<B, 256, C * sizeof(float), st>>>(
                FP(ot.rt), 1.0f, AF(h, op.mod[0]), AF(h, op.mod[1]), AF(h, op.mod[2]), AF(h, op.mod[3]), AF(h, op.mod[4]),
                AF(h, op.mod[5]), AF(h, op.mod[6]), AF(h, op.mod[7]), C, FP(ot.film));
            CK(cudaGetLastError());
            h->launches++;
            film_apply_kernel<TA><<<eb, 256, 0, st>>>(FP(ot.d32), FP(ot.film), TP<TA>(ot.dmod), LC, C, tot);
            CK(cudaGetLastError());
            h->launches++;
            dmod = TP<TA>(ot.dmod);
        }
        if (h->fno) {
            // dec_FNO.forward (enc_dec_fno.py:303-323): deconv -> GELU -> spectral -> GELU -> deconv -> GELU -> spectral
            TA* wb = TP<TA>(h->wbuf);
            const int H = h->cfg.H, W = h->cfg.W, p0 = h->fp0, p1 = h->fp1, H1 = H / p0, W1 = W / p0, C8 = C / 8, D = h->D;
            const int N1 = p1 * p1 * C2, N2 = p0 * p0 * C8;
            float* field = FP(h->dfield) + (size_t)o * B * D * H * W;
            const bool ovf1 = h->st[1] != p1, ovf0 = h->st[0] != p0;
            EpiParams ew; ew.bias = ovf1 ? AF(h, h->zero_off) : AF(h, op.decb[0]);
            gemm<TA>(h, EPI_BIAS, dmod, C, op.decw[0], wb, N1, false, B * L, N1, C, ew, st);
            long long tot = (long long)B * H1 * W1 * C2;
            wide_deconv_post_kernel<TA, false, false><<<blocks_for(tot, 256), 256, 0, st>>>(wb, N1, h->Hp, h->Wp, C2, p1, ovf1 ? AF(h, op.decb[0]) : nullptr,
                                                                                          TP<TA>(ot.z1pre), nullptr, tot, h->st[1]);
            CK(cudaGetLastError());
            h->launches++;
            launch_act_fwd<TA, ACT_GELU_ERF>(h, TP<TA>(ot.z1pre), TP<TA>(ot.z1act), tot, st);
            SpecView v2{ot.z1act.p, 1, nullptr, 1};
            run_spectral<TA>(h, op.fs1, v2, B, H1, W1, 1, false, TP<TA>(ot.z2pre), nullptr, st);
            launch_act_fwd<TA, ACT_GELU_ERF>(h, TP<TA>(ot.z2pre), TP<TA>(ot.z2act), (long long)B * H1 * W1 * C1, st);
            ew.bias = ovf0 ? AF(h, h->zero_off) : AF(h, op.decb[1]);
            gemm<TA>(h, EPI_BIAS, TP<TA>(ot.z2act), C1, op.decw[1], wb, N2, false, B * H1 * W1, N2, C1, ew, st);
            tot = (long long)B * H * W * C8;
            wide_deconv_post_kernel<TA, false, false><<<blocks_for(tot, 256), 256, 0, st>>>(wb, N2, H1, W1, C8, p0, ovf0 ? AF(h, op.decb[1]) : nullptr,
                                                                                          TP<TA>(ot.f0pre), nullptr, tot, h->st[0]);
            CK(cudaGetLastError());
            h->launches++;
            launch_act_fwd<TA, ACT_GELU_ERF>(h, TP<TA>(ot.f0pre), TP<TA>(ot.f0act), tot, st);
            SpecView v0{ot.f0act.p, 1, nullptr, 1};
            run_spectral<TA>(h, op.fs2, v0, B, H, W, 0, false, nullptr, field, st);
            continue;
        }
        if (h->wide) {
            // decoder stage = GEMM to the sub-pixel matrix -> crop + bilinear resample to the grid (pre-activation kept) -> GELU
            TA* wb = TP<TA>(h->wbuf);
            const int Hp = h->Hp, Wp = h->Wp, D = h->D;
            const int H2 = Hp * g.k2, W2 = Wp * g.k2, H1 = H2 * g.k1, W1 = W2 * g.k1;
            const int N1 = g.k2 * g.k2 * C2, N2 = g.k1 * g.k1 * C1;
            float* field = FP(h->dfield) + (size_t)o * B * D * h->cfg.H * h->cfg.W;
            // (overlapped stages: bias-free GEMM, the bias once per output sample in the pass after it -- see run_decoder_wide)
            const bool ov1 = h->st[2] != g.k2, ov2 = h->st[1] != g.k1;
            EpiParams ew; ew.bias = ov1 ? AF(h, h->zero_off) : AF(h, op.decb[0]);
            gemm<TA>(h, EPI_BIAS, dmod, C, op.decw[0], wb, N1, false, B * L, N1, C, ew, st);
            long long tot = (long long)B * H2 * W2 * C2;
            wide_deconv_post_kernel<TA, false, false><<<blocks_for(tot, 256), 256, 0, st>>>(wb, N1, Hp, Wp, C2, g.k2, ov1 ? AF(h, op.decb[0]) : nullptr,
                                                                                          TP<TA>(ot.z1pre), nullptr, tot, h->st[2]);
            CK(cudaGetLastError());
            h->launches++;
            launch_act_fwd<TA, ACT_GELU_ERF>(h, TP<TA>(ot.z1pre), TP<TA>(ot.z1act), tot, st);
            ew.bias = ov2 ? AF(h, h->zero_off) : AF(h, op.decb[1]);
            gemm<TA>(h, EPI_BIAS, TP<TA>(ot.z1act), C2, op.decw[1], wb, N2, false, B * H2 * W2, N2, C2, ew, st);
            tot = (long long)B * H1 * W1 * C1;
            wide_deconv_post_kernel<TA, false, false><<<blocks_for(tot, 256), 256, 0, st>>>(wb, N2, H2, W2, C1, g.k1, ov2 ? AF(h, op.decb[1]) : nullptr,
                                                                                          TP<TA>(ot.z2pre), nullptr, tot, h->st[1]);
            CK(cudaGetLastError());
            h->launches++;
            launch_act_fwd<TA, ACT_GELU_ERF>(h, TP<TA>(ot.z2pre), TP<TA>(ot.z2act), tot, st);
            EpiParams e3; e3.bias = AF(h, h->zero_off);
            gemm<TA>(h, EPI_BIAS, TP<TA>(ot.z2act), C1, op.w3nk, wb, h->NOpad, false, B * H1 * W1, h->NOpad, C1, e3, st);
            tot = (long long)B * D * h->cfg.H * h->cfg.W;
            wide_deconv_post_kernel<TA, false, true><<<blocks_for(tot, 256), 256, 0, st>>>(wb, h->NOpad, H1, W1, D, g.k0, AF(h, op.decb[2]), nullptr, field, tot, h->st[0]);
            CK(cudaGetLastError());
            h->launches++;
            continue;
        }
        EpiParams ed; ed.bias = AF(h, op.decb[0]);
        gemm<TA>(h, EPI_BIAS, dmod, C, op.decw[0], ot.z1pre.p, g.k2 * g.k2 * C2, false, B * L, g.k2 * g.k2 * C2, C, ed, st);
        launch_act_fwd<TA, ACT_GELU_ERF>(h, TP<TA>(ot.z1pre), TP<TA>(ot.z1act), (long long)B * L * g.R2 * C2, st);
        ed.bias = AF(h, op.decb[1]);
        gemm<TA>(h, EPI_BIAS, TP<TA>(ot.z1act), C2, op.decw[1], ot.z2pre.p, g.k1 * g.k1 * C1, false, B * L * g.R2,
                 g.k1 * g.k1 * C1, C2, ed, st);
        launch_act_fwd<TA, ACT_GELU_ERF>(h, TP<TA>(ot.z2pre), TP<TA>(ot.z2act), (long long)B * L * g.R1 * C1, st);
    }
    RolloutState rs{};
    const int* cur = win ? win->in.cur : nullptr;
    select_step_kernel<<<(B + 127) / 128, 128, 0, st>>>(rt, K, h->max_batch, B, h->cfg.deg, h->cfg.output_length, cur ? 1 : 0, n_cap,
                                                        R_t, reinterpret_cast<int*>(h->nbuf.p), rs, 0, cur, win ? win->n_lim : 0);
    CK(cudaGetLastError());
    h->launches++;
    CK(cudaMemcpyAsync(tp.n_arr.p, h->nbuf.p, (size_t)B * 4, cudaMemcpyDeviceToDevice, st));
    if (h->wide) {      // Horner sum + residual over the decoded derivative fields (boundary C)
        EmitParams ep{};
        ep.dfield = FP(h->dfield);
        ep.K = K; ep.fi = h->cfg.frame_interval;
        ep.u_ring = input; ep.fcount = nullptr;
        ep.n_arr = reinterpret_cast<int*>(h->nbuf.p);
        ep.frames = frames; ep.n_cap = n_cap;
        ep.B = B; ep.D = h->D; ep.T = T; ep.HW = (long long)h->cfg.H * h->cfg.W;
        REQUIRE(ep.HW % 4 == 0, "H * W must be a multiple of 4");
        taylor_emit_kernel<<<dim3(blocks_for(ep.HW / 4, 256), (unsigned)h->D, (unsigned)B), 256, 0, st>>>(ep);
        CK(cudaGetLastError());
        h->launches++;
    } else
    // fused Taylor head on the kept stage-1 activations
    {
        HeadParams hp{};
        for (int k = 0; k < K; ++k) {
            hp.z[k] = tp.ord[k].z2act.p;
            hp.w3[k] = AF(h, h->orders[k].decw[2]);
            hp.b3[k] = AF(h, h->orders[k].decb[2]);
        }
        hp.K = K; hp.fi = h->cfg.frame_interval; hp.u_ring = input; hp.fcount = nullptr;
        hp.n_arr = reinterpret_cast<int*>(h->nbuf.p); hp.frames = frames; hp.n_cap = n_cap;
        if (win) { hp.u0_base = input + win->in.off[T - 1]; hp.u0_bs = win->in.bs[T - 1]; hp.frames_bs = win->frames_bs; hp.cur = cur; }
        const long long rows = (long long)B * L * g.R1;
        bool done = false;
        if (kTensor) {
            cudaError_t e = cudaSuccess;
            if (launch_head_mma(hp, g, C1, rows, B, h->num_sms, st, &e)) { CK(e); done = true; }
        }
        if (!done) {
            const int NO = g.k0 * g.k0 * h->D;
            const size_t smem = (size_t)(K * C1 * NO + K * h->D) * sizeof(float);
            const int blocks = (int)((rows + 127) / 128);
#define HEAD(KO) taylor_head_kernel<TA, 8, KO><<<blocks, 128, smem, st>>>(hp, g, C1, rows, B)
            switch (K) { case 1: HEAD(1); break; case 2: HEAD(2); break; case 3: HEAD(3); break; default: HEAD(4); break; }
#undef HEAD
            CK(cudaGetLastError());
        }
        h->launches++;
    }
    tp.out_T = out_T;
    tp.n_cap = n_cap;
    tp.hist = cur != nullptr;
    tp.B_used = B;
    tp.valid = true;
}

// Backward of one taped step.  gframes: f32 (B, n_g, D, H, W) gradient of the emitted frames; gRt: f32 [B] or null;
// grad_input: f32 (B, T, D, H, W) or null (written, not accumulated; but see `win`); flat: f32 [sum numel] parameter gradients in
// tante_param order (written, not accumulated).
// win (frame-table mode): gframes has batch stride win->gf_bs; the input gradient is ACCUMULATED into the frames of win->gin
// (offsets relative to grad_input; kFrameSkip entries are not computed) instead of written to a contiguous (B, T, D, H, W).
// Backward of one axis-'C' layer (channel_axis.cuh): dxs [tokens][C] holds the gradient of the layer output on entry and of its
// input on return (the layer REPLACES the latent: no residual around it).  Per chunk of h->chanb_tokens latent tokens the block is
// recomputed from the saved fp32 input (lift, LN1, QKV, attention, out-proj, LN2, MLP -- everything the backward reads stays in
// the chunk scratch), then the usual backward kernels run at width E over rows = chunk * C.
template <typename TA>
void run_channel_layer_bwd(tante_handle_s* h, const LayerPlan& lp, const float* x_in, float* dxs, int tokens, cudaStream_t st) {
    const int C = h->C, E = lp.E, Hc = lp.Hc, nh = h->cfg.n_head, E4 = E / 4;
    constexpr bool kTensor = sizeof(TA) == 2;
    REQUIRE(h->chanb_tokens > 0 && h->cb_x0.p, "channel-axis backward workspace not allocated");
    float* x0 = FP(h->cb_x0);
    float* xm = FP(h->cb_xm);
    float* gx = FP(h->cb_gx);
    TA* ln1 = TP<TA>(h->cb_ln1);
    TA* qkv = TP<TA>(h->cb_qkv);
    TA* att = TP<TA>(h->cb_att);
    TA* ln2 = TP<TA>(h->cb_ln2);
    TA* hpre = TP<TA>(h->cb_hpre);
    TA* hact = TP<TA>(h->cb_hact);
    TA* gxb = kTensor ? TP<TA>(h->cb_gxb) : reinterpret_cast<TA*>(gx);
    TA* gxb_out = kTensor ? gxb : nullptr;
    TA* g1 = TP<TA>(h->cb_g1);
    TA* g2 = TP<TA>(h->cb_g2);
    TA* gq = TP<TA>(h->cb_gq);
    TA* hh = TP<TA>(h->cb_hh);
    const size_t lift_smem = ((size_t)E4 * E + E + 10 * (size_t)E4) * sizeof(float);
    const size_t lbw_smem = ((size_t)E * E4 + 2 * (size_t)E4 + 8 * (size_t)E) * sizeof(float);
    CK(cudaFuncSetAttribute(channel_lift_bwd_kernel<TA>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    for (int t0 = 0; t0 < tokens; t0 += h->chanb_tokens) {
        const int tc = std::min(h->chanb_tokens, tokens - t0);
        const int rows = tc * C;
        const float* xs = x_in + (size_t)t0 * C;
        float* gs = dxs + (size_t)t0 * C;
        // ---- recompute the forward of the chunk ----
        channel_lift_kernel<<<std::min((rows + 7) / 8, 16 * h->num_sms), 256, lift_smem, st>>>(
            xs, AF(h, lp.cw0), AF(h, lp.cb0), AF(h, lp.cw2), AF(h, lp.cb2), x0, rows, E);
        CK(cudaGetLastError());
        h->launches++;
        launch_layernorm<TA>(h, x0, lp.ln1w, lp.ln1b, ln1, rows, st, E);
        EpiParams eq; eq.bias = AF(h, lp.inb);
        gemm<TA>(h, EPI_BIAS, ln1, E, lp.inw, qkv, 3 * E, false, rows, 3 * E, E, eq, st);
        launch_attention_seq<TA>(h, qkv, att, tc, C, 1, nh, E, E / nh, false, st);
        EpiParams eo; eo.bias = AF(h, lp.outb); eo.resid = x0; eo.ldr = E;
        gemm<TA>(h, EPI_BIAS_RESID, att, E, lp.outw, xm, E, true, rows, E, E, eo, st);
        launch_layernorm<TA>(h, xm, lp.ln2w, lp.ln2b, ln2, rows, st, E);
        EpiParams e0; e0.bias = AF(h, lp.m0b);
        gemm<TA>(h, EPI_BIAS, ln2, E, lp.m0w, hpre, Hc, false, rows, Hc, E, e0, st);
        launch_act_fwd<TA, ACT_GELU_TANH>(h, hpre, hact, (long long)rows * Hc, st);
        // (the block output itself is not needed: x_out = x_mid + W2 hact + b2 only feeds the extract)
        // ---- backward ----
        channel_extract_bwd_kernel<TA><<<blocks_for((long long)rows * E, 256), 256, 0, st>>>(gs, gx, gxb_out, rows, E);
        CK(cudaGetLastError());
        h->launches++;
        wgrad<TA>(h, gxb, E, hact, Hc, GA(h, lp.m2w), rows, E, Hc, st, GA(h, lp.m2b));
        gemm_dx_act<TA, ACT_GELU_TANH>(h, gxb, E, lp.m2wT, g1, hpre, rows, Hc, E, st);
        wgrad<TA>(h, g1, Hc, ln2, E, GA(h, lp.m0w), rows, Hc, E, st, GA(h, lp.m0b));
        gemm_dx<TA>(h, g1, Hc, lp.m0wT, g2, E, rows, E, Hc, st);
        launch_ln_bwd<TA>(h, g2, xm, lp.ln2w, gx, gxb_out, GA(h, lp.ln2w), GA(h, lp.ln2b), rows, st, DropCfg(), 0, E);
        wgrad<TA>(h, gxb, E, att, E, GA(h, lp.outw), rows, E, E, st, GA(h, lp.outb));
        gemm_dx<TA>(h, gxb, E, lp.outwT, g2, E, rows, E, E, st);
        {
            cudaError_t e = cudaSuccess;
            bool done = false;
            if constexpr (kTensor) done = launch_attention_long_bwd_mma(qkv, g2, gq, FP(h->cb_stats), tc, C, 1, nh, E, E / nh, 0, st, &e);
            if (!done)
                REQUIRE(launch_attention_long_bwd<TA>(qkv, g2, gq, FP(h->cb_stats), tc, C, 1, nh, E, E / nh, 0, st, &e),
                        "channel attention backward: shape not covered");
            CK(e);
            h->launches += 3;
        }
        wgrad<TA>(h, gq, 3 * E, ln1, E, GA(h, lp.inw), rows, 3 * E, E, st, GA(h, lp.inb));
        gemm_dx<TA>(h, gq, 3 * E, lp.inwT, g2, E, rows, E, 3 * E, st);
        launch_ln_bwd<TA>(h, g2, x0, lp.ln1w, gx, gxb_out, GA(h, lp.ln1w), GA(h, lp.ln1b), rows, st, DropCfg(), 0, E);
        // ---- the lift: dx per (token, channel), gradients of Linear(1, E/4) in the kernel, of Linear(E/4, E) as a weight-gradient GEMM ----
        channel_lift_bwd_kernel<TA><<<std::min((rows + 7) / 8, 8 * h->num_sms), 256, lbw_smem, st>>>(
            xs, gx, AF(h, lp.cw0), AF(h, lp.cb0), AF(h, lp.cw2), gs, hh, E4, GA(h, lp.cw0), GA(h, lp.cb0), rows, E);
        CK(cudaGetLastError());
        h->launches++;
        wgrad<TA>(h, gxb, E, hh, E4, GA(h, lp.cw2), rows, E, E4, st, GA(h, lp.cb2));
    }
}

struct BackwardWin { long long gf_bs; FrameTab gin; };
template <typename TA>
void run_backward(tante_handle_s* h, Tape& tp, const float* input, const float* gframes, int n_g, const float* gRt,
                  float* grad_input, float* flat, cudaStream_t st, const BackwardWin* win = nullptr) {
    const int B = tp.B_used;
    const int C = h->C, C1 = h->C1, C2 = h->C2, T = h->T, L = h->L, K = h->K, D = h->D, Hm = h->Hm;
    const PatchGeom& g = h->geom;
    const int tokens = B * T * L;
    const int BL = B * L;
    const int NO = g.k0 * g.k0 * D;
    constexpr bool kTensor = sizeof(TA) == 2;
    const long long rows1 = (long long)BL * g.R1;       // stage-1 rows of the last frame (head)
    float* dxs = FP(h->dxs);
    const DropCfg& drop = tp.drop;
    // dY operand of the residual-branch GEMMs: the bf16 copy of the gradient stream (tensor mode) and / or its
    // dropout-masked copy; the exact mode without dropout reads the fp32 stream itself
    const bool mirror = kTensor || drop.p > 0.f;
    TA* dxb = mirror ? TP<TA>(h->dxb) : reinterpret_cast<TA*>(dxs);
    TA* g1 = TP<TA>(h->g1);
    TA* g2 = TP<TA>(h->g2);
    TA* gq = TP<TA>(h->gq);
    CK(cudaMemsetAsync(h->garena.p, 0, (size_t)h->garena_elems * 4, st));
    CK(cudaMemsetAsync(dxs, 0, (size_t)tokens * C * 4, st));
    const size_t in_elems = (size_t)B * T * D * h->cfg.H * h->cfg.W;
    if (grad_input && !win) CK(cudaMemsetAsync(grad_input, 0, in_elems * 4, st));

    // ---- Taylor head: all orders in one pass over the frame gradients ----
    if (h->wide) {
        // field-level emit (boundary C): gradient of every order's derivative field + of u0, from the frame gradients
        REQUIRE(!win, "windowed BPTT is not available at patch_scale >= 16");
        EmitBwdParams ep{};
        ep.gframes = gframes; ep.gf_bs = (long long)n_g * D * h->cfg.H * h->cfg.W;
        ep.n_arr = reinterpret_cast<const int*>(tp.n_arr.p); ep.n_g = n_g;
        ep.gfield = FP(h->dfield);
        ep.gu0 = grad_input ? grad_input + (size_t)(T - 1) * D * h->cfg.H * h->cfg.W : nullptr;
        ep.gu0_bs = (long long)T * D * h->cfg.H * h->cfg.W;
        ep.K = K; ep.fi = h->cfg.frame_interval; ep.B = B; ep.D = D; ep.HW = (long long)h->cfg.H * h->cfg.W;
        taylor_emit_bwd_kernel<<<dim3(blocks_for(ep.HW / 4, 256), (unsigned)D, (unsigned)B), 256, 0, st>>>(ep);
        CK(cudaGetLastError());
        h->launches++;
    } else {
        HeadBwdParams hp{};
        for (int k = 0; k < K; ++k) hp.G[k] = TP<TA>(h->hG) + (size_t)k * rows1 * kHeadPad;
        hp.K = K; hp.fi = h->cfg.frame_interval; hp.gframes = gframes; hp.n_cap = n_g;
        hp.gf_bs = win ? win->gf_bs : (long long)n_g * D * h->cfg.H * h->cfg.W;
        hp.n_arr = reinterpret_cast<const int*>(tp.n_arr.p);
        if (win) {
            const bool want = grad_input && win->gin.off[T - 1] != kFrameSkip;
            hp.gi_last = want ? grad_input + win->gin.off[T - 1] : nullptr;
            hp.gi_bs = win->gin.bs[T - 1];
            hp.cur = win->gin.cur;
            if (hp.cur) hp.gpred = grad_input + win->gin.hoff;
        } else {
            hp.gi_last = grad_input ? grad_input + (size_t)(T - 1) * D * h->cfg.H * h->cfg.W : nullptr;
            hp.gi_bs = (long long)T * D * h->cfg.H * h->cfg.W;
        }
        const size_t hsmem = (size_t)K * kPatchRows * kPatchPitch * sizeof(float);
        if (g.k0 * g.k1 * g.k2 >= 4) head_gather_kernel<TA, 4><<<blocks_for(rows1, kPatchRows), 128, hsmem, st>>>(hp, g, rows1);
        else head_gather_kernel<TA, 2><<<blocks_for(rows1, kPatchRows), 128, hsmem, st>>>(hp, g, rows1);
        CK(cudaGetLastError());
        h->launches++;
    }
    for (int o = K - 1; o >= 0; --o) {
        const OrderPlan& op = h->orders[o];
        OrderTape& ot = tp.ord[o];
        TA* dz = TP<TA>(h->hz) + (size_t)o * rows1 * C1;
        const int M2 = BL * g.R2, N2 = g.k1 * g.k1 * C1;
        const int N1 = g.k2 * g.k2 * C2;
        TA* dz1 = TP<TA>(h->hz1);
        TA* dmod = h->cfg.deg ? TP<TA>(ot.dl) : TP<TA>(ot.dmod);
        TA* hd = TP<TA>(h->hd);
        if (h->fno) {
            TA* wb = TP<TA>(h->wbuf);
            const int H = h->cfg.H, W = h->cfg.W, p0 = h->fp0, p1 = h->fp1, H1 = H / p0, W1 = W / p0, C8 = C / 8;
            const int NF1 = p1 * p1 * C2, NF2 = p0 * p0 * C8;
            TA* gr0 = TP<TA>(h->fgr0);
            TA* gr1 = TP<TA>(h->fgr1);
            TA* gr2 = TP<TA>(h->fgr2);
            const float* gf = FP(h->dfield) + (size_t)o * B * D * H * W;
            // dec_spectral_2 (field output, no activation)
            SpecView xg0{ot.f0act.p, 1, nullptr, 1}, gv0{gf, 0, nullptr, 1};
            run_spectral_bwd<TA>(h, op.fs2, xg0, gv0, B, H, W, 0, gr0, nullptr, st);
            launch_act_bwd<TA, ACT_GELU_ERF>(h, gr0, TP<TA>(ot.f0pre), (long long)B * H * W * C8, st);
            // dec_conv_2 (p0)
            const long long MF2 = (long long)B * H1 * W1;
            const bool ovf1 = h->st[1] != p1, ovf0 = h->st[0] != p0;      // overlapped stage: bias gradient = sum of the stage-output gradient
            if (ovf0) launch_colsum<TA>(h, gr0, C8, (long long)B * H * W, C8, GA(h, op.decb[1]), st);
            long long tot = MF2 * NF2;
            wide_deconv_post_bwd_kernel<TA, false><<<blocks_for(tot, 256), 256, 0, st>>>(gr0, nullptr, NF2, H1, W1, C8, p0, wb, tot, h->st[0]);
            CK(cudaGetLastError());
            h->launches++;
            wgrad<TA>(h, wb, NF2, TP<TA>(ot.z2act), C1, GA(h, op.decw[1]), MF2, NF2, C1, st, ovf0 ? nullptr : GA(h, op.decb[1]));
            gemm_dx_act<TA, ACT_GELU_ERF>(h, wb, NF2, op.decwT[1], gr1, TP<TA>(ot.z2pre), (int)MF2, C1, NF2, st);
            // dec_spectral_1
            SpecView xg1{ot.z1act.p, 1, nullptr, 1}, gv1{gr1, 1, nullptr, 1};
            run_spectral_bwd<TA>(h, op.fs1, xg1, gv1, B, H1, W1, 1, gr2, nullptr, st);
            launch_act_bwd<TA, ACT_GELU_ERF>(h, gr2, TP<TA>(ot.z1pre), MF2 * C2, st);
            // dec_conv_1 (p1)
            if (ovf1) launch_colsum<TA>(h, gr2, C2, MF2, C2, GA(h, op.decb[0]), st);
            tot = (long long)BL * NF1;
            wide_deconv_post_bwd_kernel<TA, false><<<blocks_for(tot, 256), 256, 0, st>>>(gr2, nullptr, NF1, h->Hp, h->Wp, C2, p1, wb, tot, h->st[1]);
            CK(cudaGetLastError());
            h->launches++;
            wgrad<TA>(h, wb, NF1, dmod, C, GA(h, op.decw[0]), BL, NF1, C, st, ovf1 ? nullptr : GA(h, op.decb[0]));
            gemm_dx<TA>(h, wb, NF1, op.decwT[0], hd, C, BL, C, NF1, st);
        } else if (h->wide) {
            // natural-order stages (wide_patch.cuh): transpose of (crop + bilinear resample) back to the sub-pixel matrix, then the
            // same weight / input gradient GEMMs as below, stage by stage
            TA* wb = TP<TA>(h->wbuf);
            TA* G = TP<TA>(h->hG);                                   // dS3 [rows1][NOpad]
            const int NP = h->NOpad;
            const int Hp = h->Hp, Wp = h->Wp;
            const int H2 = Hp * g.k2, W2 = Wp * g.k2, H1 = H2 * g.k1, W1 = W2 * g.k1;
            const float* gf = FP(h->dfield) + (size_t)o * B * D * h->cfg.H * h->cfg.W;
            // bias gradients: without overlap the replicated bias rode in the GEMM (column sums of dS, folded at unpack); an overlapped
            // stage added bias[co] once per output sample, so its gradient is the sum of the OUTPUT gradient (into the first Cout entries)
            const bool ov0 = h->st[0] != g.k0, ov1 = h->st[2] != g.k2, ov2 = h->st[1] != g.k1;
            long long tot = rows1 * NP;
            wide_deconv_post_bwd_kernel<TA, true><<<blocks_for(tot, 256), 256, 0, st>>>(nullptr, gf, NP, H1, W1, D, g.k0, G, tot, h->st[0]);
            CK(cudaGetLastError());
            h->launches++;
            wgrad_pad<TA>(h, TP<TA>(ot.z2act), C1, C1, G, NP, NP, GA(h, op.decw[2]), NO, NO, rows1, st);
            if (ov0) {
                const long long HWp = (long long)h->cfg.H * h->cfg.W;
                field_bias_grad_kernel<<<dim3((unsigned)D, 32), 256, 0, st>>>(gf, D, HWp, B, GA(h, op.decb[2]));
                CK(cudaGetLastError());
                h->launches++;
            } else {
                launch_colsum<TA>(h, G, NP, rows1, NO, GA(h, op.decb[2]), st);
            }
            gemm_dx_act<TA, ACT_GELU_ERF>(h, G, NP, op.w3pad, dz, TP<TA>(ot.z2pre), (int)rows1, C1, NP, st);
            if (ov2) launch_colsum<TA>(h, dz, C1, rows1, C1, GA(h, op.decb[1]), st);
            tot = (long long)M2 * N2;
            wide_deconv_post_bwd_kernel<TA, false><<<blocks_for(tot, 256), 256, 0, st>>>(dz, nullptr, N2, H2, W2, C1, g.k1, wb, tot, h->st[1]);
            CK(cudaGetLastError());
            h->launches++;
            wgrad<TA>(h, wb, N2, TP<TA>(ot.z1act), C2, GA(h, op.decw[1]), M2, N2, C2, st, ov2 ? nullptr : GA(h, op.decb[1]));
            gemm_dx_act<TA, ACT_GELU_ERF>(h, wb, N2, op.decwT[1], dz1, TP<TA>(ot.z1pre), M2, C2, N2, st);
            if (ov1) launch_colsum<TA>(h, dz1, C2, M2, C2, GA(h, op.decb[0]), st);
            tot = (long long)BL * N1;
            wide_deconv_post_bwd_kernel<TA, false><<<blocks_for(tot, 256), 256, 0, st>>>(dz1, nullptr, N1, Hp, Wp, C2, g.k2, wb, tot, h->st[2]);
            CK(cudaGetLastError());
            h->launches++;
            wgrad<TA>(h, wb, N1, dmod, C, GA(h, op.decw[0]), BL, N1, C, st, ov1 ? nullptr : GA(h, op.decb[0]));
            gemm_dx<TA>(h, wb, N1, op.decwT[0], hd, C, BL, C, N1, st);
        } else {
        TA* G = TP<TA>(h->hG) + (size_t)o * rows1 * kHeadPad;
        // dec_conv_3: d_k = z2act * W3 + b3  ->  dW3 = z2act^T G, db3 = colsum(G), dz2 = (G W3^T) o gelu'(z2pre)
        wgrad_pad<TA>(h, TP<TA>(ot.z2act), C1, C1, G, kHeadPad, kHeadPad, GA(h, op.decw[2]), NO, NO, rows1, st);
        launch_colsum<TA>(h, G, kHeadPad, rows1, NO, GA(h, op.decb[2]), st);
        gemm_dx_act<TA, ACT_GELU_ERF>(h, G, kHeadPad, op.w3pad, dz, TP<TA>(ot.z2pre), (int)rows1, C1, kHeadPad, st);
        // dec_conv_2: z2pre[M2, N2] = z1act[M2, C2] * Wd2^T + b
        wgrad<TA>(h, dz, N2, TP<TA>(ot.z1act), C2, GA(h, op.decw[1]), M2, N2, C2, st, GA(h, op.decb[1]));
        gemm_dx_act<TA, ACT_GELU_ERF>(h, dz, N2, op.decwT[1], dz1, TP<TA>(ot.z1pre), M2, C2, N2, st);
        // dec_conv_1: z1pre[BL, N1] = dmod[BL, C] * Wd1^T + b
        wgrad<TA>(h, dz1, N1, dmod, C, GA(h, op.decw[0]), BL, N1, C, st, GA(h, op.decb[0]));
        gemm_dx<TA>(h, dz1, N1, op.decwT[0], hd, C, BL, C, N1, st);
        }
        if (!h->cfg.deg) {
            // FiLM modifier (tante.py:151) and interprator (tante.py:149)
            CK(cudaMemsetAsync(h->dfilm.p, 0, (size_t)B * 2 * C * 4, st));
            {
                const int chunks = std::max(1, std::min(L, (2 * h->num_sms + B - 1) / B));
                film_apply_bwd_kernel<TA><<<dim3(B, chunks), C, 0, st>>>(hd, FP(ot.d32), FP(ot.film), dxs, FP(h->dfilm), T, L, C);
                CK(cudaGetLastError());
                h->launches++;
            }
            CK(cudaMemsetAsync(h->dcond.p, 0, (size_t)B * 4, st));
            film_bwd_kernel<<<dim3(B, 16), 256, 3 * C * sizeof(float), st>>>(
                FP(ot.rt), FP(h->dfilm), AF(h, op.mod[0]), AF(h, op.mod[1]), AF(h, op.mod[2]), AF(h, op.mod[4]),
                AF(h, op.mod[5]), AF(h, op.mod[6]), GA(h, op.mod[0]), GA(h, op.mod[1]), GA(h, op.mod[2]), GA(h, op.mod[3]),
                GA(h, op.mod[4]), GA(h, op.mod[5]), GA(h, op.mod[6]), GA(h, op.mod[7]), C, FP(h->dcond));
            CK(cudaGetLastError());
            h->launches++;
            TA* hi2 = TP<TA>(h->hi2);
            TA* hi1 = TP<TA>(h->hi1);
            interp_tail_bwd_kernel<TA><<<B, 256, (C / 4) * sizeof(float), st>>>(
                TP<TA>(ot.i2), AF(h, op.intw[2]), gRt, 1.0f / (float)K, FP(h->dcond), L, C / 4, hi2, GA(h, op.intw[2]),
                GA(h, op.intb[2]));
            CK(cudaGetLastError());
            h->launches++;
            wgrad<TA>(h, hi2, C / 4, TP<TA>(ot.i1), C / 2, GA(h, op.intw[1]), BL, C / 4, C / 2, st, GA(h, op.intb[1]));
            gemm_dx_act<TA, ACT_RELU>(h, hi2, C / 4, op.intwT[1], hi1, TP<TA>(ot.i1), BL, C / 2, C / 4, st);
            wgrad<TA>(h, hi1, C / 2, TP<TA>(ot.dl), C, GA(h, op.intw[0]), BL, C / 2, C, st, GA(h, op.intb[0]));
            gemm_dx<TA>(h, hi1, C / 2, op.intwT[0], hd, C, BL, C, C / 2, st);
        }
        add_last_frame_kernel<TA><<<blocks_for((long long)BL * C / 4, 256), 256, 0, st>>>(hd, dxs, B, T, (long long)L * C);
        CK(cudaGetLastError());
        h->launches++;
        // ---- backbone of order o ----
        if (mirror) {
            convert_kernel<TA><<<blocks_for((long long)tokens * C / 4, 256), 256, 0, st>>>(
                dxs, dxb, (long long)tokens * C / 4, drop, drop_site(o, (int)op.layers.size() - 1, 2));
            CK(cudaGetLastError());
            h->launches++;
        }
        TA* dxb_out = mirror ? dxb : nullptr;
        for (int li = (int)op.layers.size() - 1; li >= 0; --li) {
            const LayerPlan& lp = op.layers[li];
            const float* x_in = FP(ot.X[2 * li]);
            const float* x_mid = FP(ot.X[2 * li + 1]);
            if (lp.axis == 'C') {
                run_channel_layer_bwd<TA>(h, lp, x_in, dxs, tokens, st);
                if (mirror) {      // the layer below reads the TA mirror of the gradient stream as its dY
                    convert_kernel<TA><<<blocks_for((long long)tokens * C / 4, 256), 256, 0, st>>>(dxs, dxb, (long long)tokens * C / 4);
                    CK(cudaGetLastError());
                    h->launches++;
                }
                continue;
            }
            // MLP half: x_out = x_mid + W2 gelu_tanh(W0 ln2(x_mid) + b0) + b2
            wgrad<TA>(h, dxb, C, TP<TA>(ot.hact[li]), Hm, GA(h, lp.m2w), tokens, C, Hm, st, GA(h, lp.m2b));
            if (kTensor && h->fuse_mlp_bwd && C == kBtC && h->Hm == C) {
                // dpre = (dY W2) o gelu'(hpre) and dln2 = dpre W1 in one kernel (mlp_bwd_tc.cuh): dh never touches HBM
                {
                    ProfScope ps(h, st, 2.0 * 2.0 * tokens * C * C, 4, (double)tokens * 4 * 2 * C);
                    CK(launch_mlp_bwd(reinterpret_cast<const __nv_bfloat16*>(dxb), AH(h, lp.m2wT), AH(h, lp.m0wT),
                                      reinterpret_cast<const __nv_bfloat16*>(ot.hpre[li].p), reinterpret_cast<__nv_bfloat16*>(g1),
                                      reinterpret_cast<__nv_bfloat16*>(g2), tokens, h->num_sms, st));
                }
                h->launches++;
                wgrad<TA>(h, g1, C, TP<TA>(ot.ln2[li]), C, GA(h, lp.m0w), tokens, C, C, st, GA(h, lp.m0b));
            } else {
                gemm_dx_act<TA, ACT_GELU_TANH>(h, dxb, C, lp.m2wT, g1, TP<TA>(ot.hpre[li]), tokens, Hm, C, st);
                wgrad<TA>(h, g1, Hm, TP<TA>(ot.ln2[li]), C, GA(h, lp.m0w), tokens, Hm, C, st, GA(h, lp.m0b));
                gemm_dx<TA>(h, g1, Hm, lp.m0wT, g2, C, tokens, C, Hm, st);
            }
            launch_ln_bwd<TA>(h, g2, x_mid, lp.ln2w, dxs, dxb_out, GA(h, lp.ln2w), GA(h, lp.ln2b), tokens, st, drop,
                              drop_site(o, li, 1));
            // attention half: x_mid = x_in + Wo att(ln1(x_in)) + bo
            wgrad<TA>(h, dxb, C, TP<TA>(ot.att[li]), C, GA(h, lp.outw), tokens, C, C, st, GA(h, lp.outb));
            gemm_dx<TA>(h, dxb, C, lp.outwT, g2, C, tokens, C, C, st);
            launch_attention_bwd<TA>(h, TP<TA>(ot.qkv[li]), g2, gq, B, lp.axis, st, drop, drop_site(o, li, 0));
            wgrad<TA>(h, gq, 3 * C, TP<TA>(ot.ln1[li]), C, GA(h, lp.inw), tokens, 3 * C, C, st, GA(h, lp.inb));
            gemm_dx<TA>(h, gq, 3 * C, lp.inwT, g2, C, tokens, C, 3 * C, st);
            // the copy written here is the dY of the layer below's MLP branch
            launch_ln_bwd<TA>(h, g2, x_in, lp.ln1w, dxs, dxb_out, GA(h, lp.ln1w), GA(h, lp.ln1b), tokens, st, drop,
                              drop_site(o, std::max(li - 1, 0), 2));
        }
        const float* pin = o == 0 ? FP(ot.P[0]) : FP(tp.ord[o - 1].X.back());
        launch_propagator_bwd(h, FP(ot.P[2]), dxs, B, 2, op, st);
        launch_propagator_bwd(h, FP(ot.P[1]), dxs, B, 1, op, st);
        launch_propagator_bwd(h, pin, dxs, B, 0, op, st);
    }
    // ---- embeddings + t_encode FiLM (tante.py:136-141) ----
    CK(cudaMemsetAsync(h->dfilm.p, 0, (size_t)T * 2 * C * 4, st));
    embed_bwd_kernel<TA><<<(L + (256 / (C / 4)) - 1) / (256 / (C / 4)), 256, 0, st>>>(dxs, FP(tp.v), AF(h, h->film_t_off), g2, FP(h->dfilm), GA(h, h->s_emb),
                                          GA(h, h->t_emb), B, T, L, C);
    CK(cudaGetLastError());
    h->launches++;
    film_bwd_kernel<<<dim3(T, 16), 256, 3 * C * sizeof(float), st>>>(
        AF(h, h->tseq_off), FP(h->dfilm), AF(h, h->tenc[0]), AF(h, h->tenc[1]), AF(h, h->tenc[2]), AF(h, h->tenc[4]),
        AF(h, h->tenc[5]), AF(h, h->tenc[6]), GA(h, h->tenc[0]), GA(h, h->tenc[1]), GA(h, h->tenc[2]), GA(h, h->tenc[3]),
        GA(h, h->tenc[4]), GA(h, h->tenc[5]), GA(h, h->tenc[6]), GA(h, h->tenc[7]), C, nullptr);
    CK(cudaGetLastError());
    h->launches++;
    // ---- encoder (enc_dec_cnn.py:217-229) ----
    const int K3 = g.k2 * g.k2 * C2, K2 = g.k1 * g.k1 * C1;
    const int M2 = tokens * g.R2;
    const long long rows_in = (long long)tokens * g.R1;
    if (h->fno) {
        TA* wb = TP<TA>(h->wbuf);
        const int H = h->cfg.H, W = h->cfg.W, p0 = h->fp0, p1 = h->fp1, H1 = H / p0, W1 = W / p0, C8 = C / 8;
        const long long NI = (long long)B * T, MF1 = NI * H1 * W1;
        const int KF2 = p1 * p1 * C2, KF1 = p0 * p0 * C8;
        TA* gr0 = TP<TA>(h->fgr0);
        TA* gr1 = TP<TA>(h->fgr1);
        TA* gr2 = TP<TA>(h->fgr2);
        // conv grids (== the patch grids without overlap); with overlap the gradient of a pooled output first goes back to its conv grid
        auto cdimf = [](int n, int k, int sdv) { return (n + 2 * ((k - 1) / 2) - k) / sdv + 1; };
        const int Hc2 = cdimf(H1, p1, h->st[1]), Wc2 = cdimf(W1, p1, h->st[1]), Hc1 = cdimf(H, p0, h->st[0]), Wc1 = cdimf(W, p0, h->st[0]);
        const bool pool2 = Hc2 != h->Hp || Wc2 != h->Wp, pool1 = Hc1 != H1 || Wc1 != W1;
        const long long rows2 = NI * Hc2 * Wc2, rows1 = NI * Hc1 * Wc1;
        REQUIRE(rows1 < (1LL << 31) && rows2 < (1LL << 31), "input too large for the conv backward GEMMs");
        TA* cg = TP<TA>(h->cgrid);
        // enc_conv_2 (p1): windows of the kept C/2 grid
        const TA* dY2 = g2;
        if (pool2) {
            const long long t4 = rows2 * C / 4;
            wide_pool_bwd_kernel<TA, false><<<blocks_for(t4, 256), 256, 0, st>>>(g2, nullptr, Hc2, Wc2, C, h->Hp, h->Wp, cg, t4);
            CK(cudaGetLastError());
            h->launches++;
            dY2 = cg;
        }
        wide_im2col_cl_kernel<TA><<<blocks_for(rows2 * KF2 / 4, 256), 256, 0, st>>>(TP<TA>(tp.a2act), H1, W1, C2, p1, (p1 - 1) / 2, wb,
                                                                                   rows2 * KF2 / 4, h->st[1], Hc2, Wc2);
        CK(cudaGetLastError());
        h->launches++;
        wgrad<TA>(h, dY2, C, wb, KF2, GA(h, h->enc_w[1]), rows2, C, KF2, st, GA(h, h->enc_b[1]));
        gemm_dx<TA>(h, dY2, C, h->enc_wT[1], wb, KF2, (int)rows2, KF2, C, st);
        wide_col2im_cl_kernel<TA><<<blocks_for(MF1 * C2 / 4, 256), 256, 0, st>>>(wb, H1, W1, C2, p1, (p1 - 1) / 2, gr2, MF1 * C2 / 4, h->st[1], Hc2, Wc2);
        CK(cudaGetLastError());
        h->launches++;
        launch_act_bwd<TA, ACT_GELU_ERF>(h, gr2, TP<TA>(tp.a2pre), MF1 * C2, st);
        // enc_spectral_2
        SpecView xs1{tp.a1act.p, 1, nullptr, 1}, gs1{gr2, 1, nullptr, 1};
        run_spectral_bwd<TA>(h, h->fes2, xs1, gs1, NI, H1, W1, 1, gr1, nullptr, st);
        launch_act_bwd<TA, ACT_GELU_ERF>(h, gr1, TP<TA>(tp.a1pre), MF1 * C1, st);
        // enc_conv_1 (p0): windows of the kept C/8 grid
        const TA* dY1 = gr1;
        if (pool1) {
            const long long t4 = rows1 * C1 / 4;
            wide_pool_bwd_kernel<TA, false><<<blocks_for(t4, 256), 256, 0, st>>>(gr1, nullptr, Hc1, Wc1, C1, H1, W1, cg, t4);
            CK(cudaGetLastError());
            h->launches++;
            dY1 = cg;
        }
        wide_im2col_cl_kernel<TA><<<blocks_for(rows1 * KF1 / 4, 256), 256, 0, st>>>(TP<TA>(tp.f0act), H, W, C8, p0, (p0 - 1) / 2, wb, rows1 * KF1 / 4,
                                                                                   h->st[0], Hc1, Wc1);
        CK(cudaGetLastError());
        h->launches++;
        wgrad<TA>(h, dY1, C1, wb, KF1, GA(h, h->enc_w[0]), rows1, C1, KF1, st, GA(h, h->enc_b[0]));
        gemm_dx<TA>(h, dY1, C1, h->enc_wT[0], wb, KF1, (int)rows1, KF1, C1, st);
        wide_col2im_cl_kernel<TA><<<blocks_for(NI * H * W * C8 / 4, 256), 256, 0, st>>>(wb, H, W, C8, p0, (p0 - 1) / 2, gr0, NI * H * W * C8 / 4,
                                                                                       h->st[0], Hc1, Wc1);
        CK(cudaGetLastError());
        h->launches++;
        launch_act_bwd<TA, ACT_GELU_ERF>(h, gr0, TP<TA>(tp.f0pre), NI * H * W * C8, st);
        // enc_spectral_1 on the input frames (input gradient accumulated on top of the u0 path)
        SpecView xs0{input, 0, nullptr, T}, gs0{gr0, 1, nullptr, 1};
        run_spectral_bwd<TA>(h, h->fes1, xs0, gs0, NI, H, W, 0, nullptr, grad_input, st);
    } else if (h->wide) {
        // natural-order stages: the patch matrices of conv3 / conv2 are re-gathered from the kept activation grids (cheap, one
        // pass), their gradients go back to the grids through the transposed gather; with overlap_ratio != 0 the gradient of a
        // stage's (pooled) output first goes back to its conv grid (wide_pool_bwd_kernel)
        TA* wb = TP<TA>(h->wbuf);
        TA* cg = TP<TA>(h->cgrid);
        const int H = h->cfg.H, W = h->cfg.W;
        const WideDims wd = wide_dims(h, B);
        const int H1 = wd.H1, W1 = wd.W1, H2 = wd.H2, W2 = wd.W2;
        const long long NI = (long long)B * T;
        auto pool_bwd = [&](const TA* gp, int Hc, int Wc, int Cc, int Ho, int Wo) {
            const long long total4 = NI * Hc * Wc * Cc / 4;
            wide_pool_bwd_kernel<TA, false><<<blocks_for(total4, 256), 256, 0, st>>>(gp, nullptr, Hc, Wc, Cc, Ho, Wo, cg, total4);
            CK(cudaGetLastError());
            h->launches++;
        };
        // stage 3
        const TA* dY3 = g2;
        if (wd.pool3) { pool_bwd(g2, wd.Hc3, wd.Wc3, C, h->Hp, h->Wp); dY3 = cg; }
        wide_im2col_cl_kernel<TA><<<blocks_for(wd.rows3 * K3 / 4, 256), 256, 0, st>>>(TP<TA>(tp.a2act), H2, W2, C2, g.k2, (g.k2 - 1) / 2, wb,
                                                                                     wd.rows3 * K3 / 4, h->st[2], wd.Hc3, wd.Wc3);
        CK(cudaGetLastError());
        h->launches++;
        wgrad<TA>(h, dY3, C, wb, K3, GA(h, h->enc_w[2]), wd.rows3, C, K3, st, GA(h, h->enc_b[2]));
        gemm_dx<TA>(h, dY3, C, h->enc_wT[2], wb, K3, (int)wd.rows3, K3, C, st);
        wide_col2im_cl_kernel<TA><<<blocks_for(NI * H2 * W2 * C2 / 4, 256), 256, 0, st>>>(wb, H2, W2, C2, g.k2, (g.k2 - 1) / 2, gq,
                                                                                         NI * H2 * W2 * C2 / 4, h->st[2], wd.Hc3, wd.Wc3);
        CK(cudaGetLastError());
        h->launches++;
        launch_act_bwd<TA, ACT_GELU_ERF>(h, gq, TP<TA>(tp.a2pre), NI * H2 * W2 * C2, st);
        // stage 2
        const TA* dY2 = gq;
        if (wd.pool2) { pool_bwd(gq, wd.Hc2, wd.Wc2, C2, H2, W2); dY2 = cg; }
        wide_im2col_cl_kernel<TA><<<blocks_for(wd.rows2 * K2 / 4, 256), 256, 0, st>>>(TP<TA>(tp.a1act), H1, W1, C1, g.k1, (g.k1 - 1) / 2, wb,
                                                                                     wd.rows2 * K2 / 4, h->st[1], wd.Hc2, wd.Wc2);
        CK(cudaGetLastError());
        h->launches++;
        wgrad<TA>(h, dY2, C2, wb, K2, GA(h, h->enc_w[1]), wd.rows2, C2, K2, st, GA(h, h->enc_b[1]));
        gemm_dx<TA>(h, dY2, C2, h->enc_wT[1], wb, K2, (int)wd.rows2, K2, C2, st);
        TA* ga1 = TP<TA>(h->ga1);
        wide_col2im_cl_kernel<TA><<<blocks_for(NI * H1 * W1 * C1 / 4, 256), 256, 0, st>>>(wb, H1, W1, C1, g.k1, (g.k1 - 1) / 2, ga1,
                                                                                         NI * H1 * W1 * C1 / 4, h->st[1], wd.Hc2, wd.Wc2);
        CK(cudaGetLastError());
        h->launches++;
        launch_act_bwd<TA, ACT_GELU_ERF>(h, ga1, TP<TA>(tp.a1pre), NI * H1 * W1 * C1, st);
        // stage 1
        const TA* dY1 = ga1;
        if (wd.pool1) { pool_bwd(ga1, wd.Hc1, wd.Wc1, C1, H1, W1); dY1 = cg; }
        wgrad_pad<TA>(h, dY1, C1, C1, TP<TA>(tp.cols), h->K1pad, h->K1pad, GA(h, h->enc_w[0]), NO, NO, wd.rows1, st, GA(h, h->enc_b[0]));
        if (grad_input) {
            REQUIRE(wd.rows1 < (1LL << 31), "input too large for the first-conv backward GEMM");
            gemm_dx<TA>(h, dY1, C1, h->enc_wT[0], wb, h->K1pad, (int)wd.rows1, h->K1pad, C1, st);
            const long long tot = (long long)in_elems;
            wide_col2im_cf_kernel<TA><<<blocks_for(tot, 256), 256, 0, st>>>(wb, D, H, W, g.k0, (g.k0 - 1) / 2, h->K1pad, grad_input, tot,
                                                                           h->st[0], wd.Hc1, wd.Wc1);
            CK(cudaGetLastError());
            h->launches++;
        }
    } else {
    wgrad<TA>(h, g2, C, TP<TA>(tp.a2act), K3, GA(h, h->enc_w[2]), tokens, C, K3, st, GA(h, h->enc_b[2]));
    gemm_dx_act<TA, ACT_GELU_ERF>(h, g2, C, h->enc_wT[2], gq, TP<TA>(tp.a2pre), tokens, K3, C, st);
    wgrad<TA>(h, gq, C2, TP<TA>(tp.a1act), K2, GA(h, h->enc_w[1]), M2, C2, K2, st, GA(h, h->enc_b[1]));
    TA* ga1 = TP<TA>(h->ga1);
    gemm_dx_act<TA, ACT_GELU_ERF>(h, gq, C2, h->enc_wT[1], ga1, TP<TA>(tp.a1pre), M2, K2, C2, st);
    (void)input;      // the patches were kept by the forward (tape im2col)
    TA* cols = TP<TA>(h->cols);
    wgrad_pad<TA>(h, ga1, C1, C1, TP<TA>(tp.cols), kHeadPad, kHeadPad, GA(h, h->enc_w[0]), NO, NO, rows_in, st, GA(h, h->enc_b[0]));
    if (grad_input) {
        // dpatch[rows, 64 (K1 padded)] = da1[rows, C1] * W1[C1][K1]  (thin GEMM), then scatter-add into the pixels
        REQUIRE(rows_in < (1LL << 31), "input too large for the first-conv backward GEMM");
        gemm_dx<TA>(h, ga1, C1, h->enc_wT[0], cols, kHeadPad, (int)rows_in, kHeadPad, C1, st);
        const FrameTab gt = win ? win->gin : FrameTab();
        if (g.k0 * g.k1 * g.k2 >= 4) conv1_col2im_kernel<TA, 4><<<blocks_for(rows_in, kPatchRows), 128, 0, st>>>(cols, g, grad_input, rows_in, gt);
        else conv1_col2im_kernel<TA, 2><<<blocks_for(rows_in, kPatchRows), 128, 0, st>>>(cols, g, grad_input, rows_in, gt);
        CK(cudaGetLastError());
        h->launches++;
    }
    }
    // ---- packed gradient arena -> flat state_dict-layout buffer ----
    {
        int64_t max_numel = 0;
        for (const Param& p : h->params) max_numel = std::max(max_numel, p.numel);
        dim3 grid((unsigned)std::min<int64_t>((max_numel + 255) / 256, 64), (unsigned)h->params.size());
        unpack_grads_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const UnpackDesc*>(h->udesc_dev.p), FP(h->garena), flat);
        CK(cudaGetLastError());
        h->launches++;
    }
}

void ensure_ready(tante_handle_s* h, int B, bool need_backbone = true) {
    if (need_backbone && !h->axes_ok)
        throw Error(TANTE_ERR_INVALID, "axis length > 96 (H_p, W_p) or in_T > 64 is not supported by the propagator kernels");
    if (!h->packed) throw Error(TANTE_ERR_STATE, "parameters not packed: call tante_bind_param for every parameter, then tante_pack_params");
    if (B < 1 || B > h->max_batch) throw Error(TANTE_ERR_STATE, "batch exceeds tante_reserve(max_batch)");
}

void set_smem_attrs() {
    static unsigned long long done = 0;
    if (!attrs_needed(done)) return;
    const int big = 160 * 1024;
    CK(cudaFuncSetAttribute(channel_lift_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024));
    CK(cudaFuncSetAttribute(propagator_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    CK(cudaFuncSetAttribute(propagator_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    CK(cudaFuncSetAttribute(patch_embed_conv1_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
    CK(cudaFuncSetAttribute(patch_embed_conv1_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, big));
#define HEADATTR(TA, KO) CK(cudaFuncSetAttribute(taylor_head_kernel<TA, 8, KO>, cudaFuncAttributeMaxDynamicSharedMemorySize, big))
    HEADATTR(float, 1); HEADATTR(float, 2); HEADATTR(float, 3); HEADATTR(float, 4);
    HEADATTR(__nv_bfloat16, 1); HEADATTR(__nv_bfloat16, 2); HEADATTR(__nv_bfloat16, 3); HEADATTR(__nv_bfloat16, 4);
#undef HEADATTR
    CK(cudaFuncSetAttribute(propagator_bwd_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 120 * 1024));
    CK(cudaFuncSetAttribute(propagator_bwd_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 120 * 1024));
    CK((cudaFuncSetAttribute(head_gather_kernel<float, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024)));
    CK((cudaFuncSetAttribute(head_gather_kernel<float, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024)));
    CK((cudaFuncSetAttribute(head_gather_kernel<__nv_bfloat16, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024)));
    CK((cudaFuncSetAttribute(head_gather_kernel<__nv_bfloat16, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024)));
#define ATTBATTR(TA, HDv) CK(cudaFuncSetAttribute(attention_bwd_kernel<TA, HDv>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024))
    ATTBATTR(float, 16); ATTBATTR(float, 32); ATTBATTR(float, 64);
    ATTBATTR(__nv_bfloat16, 16); ATTBATTR(__nv_bfloat16, 32); ATTBATTR(__nv_bfloat16, 64);
#undef ATTBATTR
    CK(tc_set_attrs());
    CK(bt_set_attrs());
    CK(wg_set_attrs());
    att_set_attrs();
    prop_set_attrs();
}

void destroy_graphs(tante_handle_s* h);

template <typename F>
int guarded(F&& f) {
    try {
        f();
        return TANTE_OK;
    } catch (const Error& e) {
        g_err = e.what();
        return e.code;
    } catch (const std::exception& e) {
        g_err = e.what();
        return TANTE_ERR_INVALID;
    }
}

}  // namespace

namespace {
void destroy_graphs(tante_handle_s* h) {
    for (auto& kv : h->graphs) {
        if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
        if (kv.second.graph) cudaGraphDestroy(kv.second.graph);
    }
    h->graphs.clear();
}

// Compaction buckets of a per-sample rollout (TANTE_ROLLOUT_COMPACT=0 disables): the step body is captured once per batch
// size B, 3B/4, B/2, B/4 and a SWITCH node inside the WHILE body runs the smallest one that holds every running trajectory.
// Needs the encoder cache (its frame lists already speak trajectory ids) and the patch-GEMM encoder.
static bool compaction_wanted(const tante_handle_s* h, const StepIO& io, int B, const RolloutState& rs) {
    static const bool on = !(getenv("TANTE_ROLLOUT_COMPACT") && atoi(getenv("TANTE_ROLLOUT_COMPACT")) == 0);
    return on && io.per_sample && B >= 8 && rs.enc_count && !h->wide && !h->fno && !h->cfg.deg;
}

template <typename TA>
void build_roll_graph(tante_handle_s* h, tante_handle_s::RollGraph& rg, const StepIO& io, int B,
                             const RolloutState& rs_in, bool while_node) {
    if (!h->cap_stream) CK(cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking));
    const int64_t launches0 = h->launches;
    RolloutState rs = rs_in;
    if (while_node && rs.act && rs.n_buckets > 1) {
        // WHILE { SWITCH(bucket) { step(B_0) | step(B_1) | ... } }
        CK(cudaGraphCreate(&rg.graph, 0));
        CK(cudaGraphConditionalHandleCreate(&h->cond_handle, rg.graph, 1, cudaGraphCondAssignDefault));
        CK(cudaGraphConditionalHandleCreate(&h->sw_handle, rg.graph, 0, cudaGraphCondAssignDefault));
        rs.sw = h->sw_handle;
        cudaGraphNodeParams np = {cudaGraphNodeTypeConditional};
        np.conditional.handle = h->cond_handle;
        np.conditional.type = cudaGraphCondTypeWhile;
        np.conditional.size = 1;
        cudaGraphNode_t node;
        CK(cudaGraphAddNode(&node, rg.graph, nullptr, 0, &np));
        cudaGraph_t body = np.conditional.phGraph_out[0];
        cudaGraphNodeParams sp = {cudaGraphNodeTypeConditional};
        sp.conditional.handle = h->sw_handle;
        sp.conditional.type = cudaGraphCondTypeSwitch;
        sp.conditional.size = (unsigned)rs.n_buckets;
        cudaGraphNode_t snode;
        CK(cudaGraphAddNode(&snode, body, nullptr, 0, &sp));
        h->use_cond = 1;
        for (int k = 0; k < rs.n_buckets; ++k) {
            CK(cudaStreamBeginCaptureToGraph(h->cap_stream, sp.conditional.phGraph_out[k], nullptr, nullptr, 0,
                                             cudaStreamCaptureModeThreadLocal));
            const int64_t l0 = h->launches;
            try {
                run_step<TA>(h, io, rs.bucket_sz[k], rs, h->cap_stream);
            } catch (...) {
                cudaGraph_t dummy = nullptr;
                cudaStreamEndCapture(h->cap_stream, &dummy);
                h->use_cond = 0;
                throw;
            }
            CK(cudaStreamEndCapture(h->cap_stream, nullptr));
            if (k > 0) h->launches = l0;      // the per-step launch count is that of the full bucket
        }
        h->use_cond = 0;
    } else if (while_node) {
        CK(cudaGraphCreate(&rg.graph, 0));
        CK(cudaGraphConditionalHandleCreate(&h->cond_handle, rg.graph, 1, cudaGraphCondAssignDefault));
        cudaGraphNodeParams np = {cudaGraphNodeTypeConditional};
        np.conditional.handle = h->cond_handle;
        np.conditional.type = cudaGraphCondTypeWhile;
        np.conditional.size = 1;
        cudaGraphNode_t node;
        CK(cudaGraphAddNode(&node, rg.graph, nullptr, 0, &np));
        cudaGraph_t body = np.conditional.phGraph_out[0];
        h->use_cond = 1;
        CK(cudaStreamBeginCaptureToGraph(h->cap_stream, body, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal));
        try {
            run_step<TA>(h, io, B, rs, h->cap_stream);
        } catch (...) {
            cudaGraph_t dummy = nullptr;
            cudaStreamEndCapture(h->cap_stream, &dummy);
            h->use_cond = 0;
            throw;
        }
        CK(cudaStreamEndCapture(h->cap_stream, nullptr));
        h->use_cond = 0;
    } else {
        CK(cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeThreadLocal));
        try {
            run_step<TA>(h, io, B, rs, h->cap_stream);
        } catch (...) {
            cudaGraph_t dummy = nullptr;
            cudaStreamEndCapture(h->cap_stream, &dummy);
            throw;
        }
        CK(cudaStreamEndCapture(h->cap_stream, &rg.graph));
    }
    CK(cudaGraphInstantiate(&rg.exec, rg.graph, 0));
    rg.while_node = while_node;
    rg.launches_per_step = h->launches - launches0;
    h->launches = launches0;      // capture enqueued nothing
}
}  // namespace

// ================================================================================================
extern "C" {

const char* tante_last_error(void) { return g_err.c_str(); }
int tante_version(void) { return 1; }

int tante_create(const tante_config_t* cfg, int device, tante_handle_t* out) {
    return guarded([&] {
        REQUIRE(cfg && out, "null argument");
        std::unique_ptr<tante_handle_s> h(new tante_handle_s());
        h->cfg = *cfg;
        h->device = device;
        build_plan(h.get());
        if (const char* m = getenv("TANTE_ROLLOUT_MODE")) h->rollout_mode = std::max(0, std::min(2, atoi(m)));
        if (const char* m = getenv("TANTE_ENC_CACHE")) h->use_enc_cache = atoi(m) != 0;
        if (const char* m = getenv("TANTE_FUSE_TAIL")) h->fuse_tail = atoi(m) != 0;
        if (const char* m = getenv("TANTE_FUSE_MLP_BWD")) h->fuse_mlp_bwd = atoi(m) != 0;
        int sms = 0;   // stays at the B200 default when no device is visible (CPU-side plan checks)
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) h->num_sms = sms;
        else (void)cudaGetLastError();
        *out = h.release();
    });
}

int tante_destroy(tante_handle_t h) {
    return guarded([&] {
        if (!h) return;
        cudaSetDevice(h->device);
        DevBuf* bufs[] = {&h->arena, &h->arena_bf16, &h->descs, &h->x, &h->ln, &h->qkv, &h->att, &h->hid, &h->a1, &h->a2,
                          &h->d32, &h->dmod, &h->i1, &h->i2, &h->z1, &h->rt, &h->Rt, &h->nbuf, &h->filmbuf, &h->ring,
                          &h->state, &h->dbg_in, &h->enc_cache, &h->enc_state, &h->icols, &h->wbuf, &h->dfield, &h->ftw,
                          &h->fA, &h->fB, &h->fg0, &h->fg1, &h->fg2, &h->cgrid, &h->cx, &h->cln, &h->cqkv, &h->catt, &h->chid};
        for (DevBuf* b : bufs) b->free();
        for (auto& b : h->z2) b.free();
        DevBuf* tb[] = {&h->garena, &h->tdesc_dev, &h->udesc_dev, &h->dxs, &h->dxb, &h->g1, &h->g2, &h->gq, &h->ga1, &h->cols,
                        &h->hz, &h->hG, &h->hz1, &h->hd, &h->hi1, &h->hi2, &h->dfilm, &h->dcond, &h->att_stats, &h->kscratch, &h->cb_x0, &h->cb_xm, &h->cb_gx, &h->cb_ln1, &h->cb_qkv, &h->cb_att, &h->cb_ln2, &h->cb_hpre, &h->cb_hact, &h->cb_gxb, &h->cb_g1, &h->cb_g2, &h->cb_gq, &h->cb_hh, &h->cb_stats, &h->fC, &h->fD, &h->fgr0, &h->fgr1, &h->fgr2, &h->opt_segs, &h->opt_norm};
        for (DevBuf* b : tb) b->free();
        if (h->nccl_comm && nccl_api().ok()) nccl_api().CommDestroy(h->nccl_comm);
        for (auto& tp : h->tapes) free_tape(*tp);
        if (h->h_flag) cudaFreeHost(h->h_flag);
        for (auto& e : h->ev) if (e) cudaEventDestroy(e);
        for (auto& e : h->prof_ev) cudaEventDestroy(e);
        destroy_graphs(h);
        if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
        delete h;
    });
}

int32_t tante_param_count(tante_handle_t h) { return h ? (int32_t)h->params.size() : 0; }
const char* tante_param_name(tante_handle_t h, int32_t i) {
    if (!h || i < 0 || i >= (int32_t)h->params.size()) return nullptr;
    return h->params[i].name.c_str();
}
int64_t tante_param_numel(tante_handle_t h, int32_t i) {
    if (!h || i < 0 || i >= (int32_t)h->params.size()) return -1;
    return h->params[i].numel;
}

int tante_bind_param(tante_handle_t h, const char* name, const float* data, float* grad, int64_t numel) {
    return guarded([&] {
        REQUIRE(h && name && data, "null argument");
        auto it = h->pindex.find(name);
        REQUIRE(it != h->pindex.end(), std::string("unknown parameter: ") + name);
        Param& p = h->params[it->second];
        REQUIRE(p.numel == numel, std::string("size mismatch for ") + name + ": expected " + std::to_string(p.numel) +
                                      ", got " + std::to_string(numel));
        p.data = data;
        p.grad = grad;
        h->packed = false;
    });
}

int tante_pack_params(tante_handle_t h, void* stream) {
    return guarded([&] {
        REQUIRE(h, "null handle");
        CK(cudaSetDevice(h->device));
        set_smem_attrs();
        cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
        for (const Param& p : h->params)
            if (!p.data) throw Error(TANTE_ERR_STATE, "parameter not bound: " + p.name);
        dev_alloc(h, h->arena, (size_t)h->arena_elems * sizeof(float));
        if (h->cfg.precision == TANTE_PREC_BF16) dev_alloc(h, h->arena_bf16, (size_t)h->arena_elems * sizeof(__nv_bfloat16));
        std::vector<PackDesc> descs;
        int64_t max_numel = 0;
        for (const Param& p : h->params) {
            PackDesc d;
            d.src = p.data; d.dst_off = p.off; d.numel = p.packed_numel; d.mode = p.mode;
            d.d0 = p.d0; d.d1 = p.d1; d.k = p.k;
            descs.push_back(d);
            max_numel = std::max(max_numel, p.packed_numel);
        }
        dev_alloc(h, h->descs, descs.size() * sizeof(PackDesc));
        // the descriptor tables only change when a parameter is re-bound: upload them once (pageable H2D copy of a
        // small table: synchronous w.r.t. the host buffer, ordered on `st`), so that the per-optimizer-step repack
        // of a training loop is two kernel launches and no host sync
        const bool first = h->desc_cache.size() != descs.size() * sizeof(PackDesc) ||
                           memcmp(h->desc_cache.data(), descs.data(), h->desc_cache.size()) != 0;
        if (first) {
            CK(cudaMemcpyAsync(h->descs.p, descs.data(), descs.size() * sizeof(PackDesc), cudaMemcpyHostToDevice, st));
            CK(cudaStreamSynchronize(st));
            h->desc_cache.assign(reinterpret_cast<const char*>(descs.data()),
                                 reinterpret_cast<const char*>(descs.data()) + descs.size() * sizeof(PackDesc));
            if (!h->tdescs.empty()) {
                dev_alloc(h, h->tdesc_dev, h->tdescs.size() * sizeof(TransDesc));
                CK(cudaMemcpyAsync(h->tdesc_dev.p, h->tdescs.data(), h->tdescs.size() * sizeof(TransDesc),
                                   cudaMemcpyHostToDevice, st));
                CK(cudaStreamSynchronize(st));
            }
            CK(cudaMemsetAsync(AF(h, h->zero_off), 0, 4096 * sizeof(float), st));
        }
        dim3 grid((unsigned)std::min<int64_t>((max_numel + 255) / 256, 64), (unsigned)descs.size());
        pack_params_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const PackDesc*>(h->descs.p), AF(h, 0),
                                                 reinterpret_cast<__nv_bfloat16*>(h->arena_bf16.p));
        CK(cudaGetLastError());
        h->launches++;
        if (!h->tdescs.empty()) {
            dim3 tgrid(64, (unsigned)h->tdescs.size());
            transpose_packed_kernel<<<tgrid, 256, 0, st>>>(reinterpret_cast<const TransDesc*>(h->tdesc_dev.p), AF(h, 0),
                                                           reinterpret_cast<__nv_bfloat16*>(h->arena_bf16.p));
            CK(cudaGetLastError());
            h->launches++;
        }
        // derived: t_seq (tante.py:279-285: [-(T-2)..-1,-0,0]*fi) and the t_encode FiLM table
        std::vector<float> tseq(64, 0.f);
        {
            std::vector<float> s;
            s.push_back(0.0f);
            for (int i = 0; i < h->T - 1; ++i) s.push_back(-(float)i * h->cfg.frame_interval);
            std::reverse(s.begin(), s.end());
            for (int i = 0; i < h->T; ++i) tseq[i] = s[i];
        }
        if (first) {
            CK(cudaMemcpyAsync(AF(h, h->tseq_off), tseq.data(), 64 * sizeof(float), cudaMemcpyHostToDevice, st));
            CK(cudaStreamSynchronize(st));
        }
        film_params_kernel<<<h->T, 256, h->C * sizeof(float), st>>>(
            AF(h, h->tseq_off), 1.0f, AF(h, h->tenc[0]), AF(h, h->tenc[1]), AF(h, h->tenc[2]), AF(h, h->tenc[3]),
            AF(h, h->tenc[4]), AF(h, h->tenc[5]), AF(h, h->tenc[6]), AF(h, h->tenc[7]), h->C, AF(h, h->film_t_off));
        CK(cudaGetLastError());
        h->launches++;
        h->packed = true;
    });
}

int tante_reserve(tante_handle_t h, int32_t max_batch, int32_t max_roll, int32_t training) {
    return guarded([&] {
        REQUIRE(h && max_batch >= 1, "bad argument");
        REQUIRE(training >= 0 && training <= 65536, "training (tape slots) must be in 0..65536");
        CK(cudaSetDevice(h->device));
        while ((int)h->tapes.size() < training) h->tapes.emplace_back(new Tape());
        if (max_batch <= h->max_batch && max_roll <= h->max_roll) return;
        destroy_graphs(h);        // workspace pointers are baked into captured kernel arguments
        max_batch = std::max(max_batch, h->max_batch);
        max_roll = std::max(max_roll, h->max_roll);
        const size_t es = h->cfg.precision == TANTE_PREC_BF16 ? 2 : 4;
        const size_t tokens = (size_t)max_batch * h->T * h->L;
        const size_t BL = (size_t)max_batch * h->L;
        const int C = h->C, C1 = h->C1, C2 = h->C2;
        const PatchGeom& g = h->geom;
        dev_alloc(h, h->x, tokens * C * 4);
        dev_alloc(h, h->ln, tokens * C * es);
        dev_alloc(h, h->qkv, tokens * 3 * C * es);
        dev_alloc(h, h->att, tokens * C * es);
        dev_alloc(h, h->hid, tokens * std::max(C, h->Hm) * es);
        dev_alloc(h, h->a1, tokens * g.R1 * C1 * es);
        if (es == 2 || C1 != 64) dev_alloc(h, h->icols, tokens * g.R1 * kHeadPad * es);
        dev_alloc(h, h->a2, tokens * g.R2 * C2 * es);
        dev_alloc(h, h->d32, BL * C * 4);
        dev_alloc(h, h->dmod, BL * C * es);
        dev_alloc(h, h->i1, BL * (C / 2) * es);
        dev_alloc(h, h->i2, BL * (C / 4) * es);
        dev_alloc(h, h->z1, BL * g.R2 * C2 * es);
        h->z2.resize(h->K);
        for (auto& b : h->z2) dev_alloc(h, b, BL * g.R1 * C1 * es);
        dev_alloc(h, h->rt, (size_t)h->K * max_batch * 4);
        dev_alloc(h, h->Rt, (size_t)max_batch * 4);
        dev_alloc(h, h->nbuf, (size_t)max_batch * 4);
        dev_alloc(h, h->filmbuf, (size_t)max_batch * 2 * C * 4);
        dev_alloc(h, h->ring, (size_t)max_batch * h->T * h->D * h->cfg.H * h->cfg.W * 4);
        dev_alloc(h, h->state, ((size_t)5 * max_batch + 64) * 4);      // counters (4 per trajectory), scalars, pointer table, act list
        if (max_roll > 0 && h->use_enc_cache) {
            dev_alloc(h, h->enc_cache, tokens * C * 4);
            dev_alloc(h, h->enc_state, ((size_t)2 * max_batch * h->T + 8) * 4);
        }
        if (h->debug) dev_alloc(h, h->dbg_in, tokens * C * 4);
        if (h->chan) {
            // channel pass: chunks of latent tokens, rows = chunk * C channel tokens of width E (about 3.5 KB per row in fp32)
            h->chan_tokens = (int)std::min<size_t>(tokens, 2048);
            if (const char* e = getenv("TANTE_CHAN_CHUNK")) h->chan_tokens = std::max(1, std::min(h->chan_tokens, atoi(e)));      // (tests: ragged chunks)
            const size_t rows = (size_t)h->chan_tokens * C;
            dev_alloc(h, h->cx, rows * h->chanE * 4);
            dev_alloc(h, h->cln, rows * h->chanE * es);
            dev_alloc(h, h->cqkv, rows * 3 * h->chanE * es);
            dev_alloc(h, h->catt, rows * h->chanE * es);
            dev_alloc(h, h->chid, rows * h->chanHc * es);
        }
        if (h->fno) {
            const size_t NI = (size_t)max_batch * h->T, HW = (size_t)h->cfg.H * h->cfg.W, HW1 = HW / (h->fp0 * h->fp0);
            const int C8 = C / 8;
            dev_alloc(h, h->fg0, NI * HW * C8 * es);
            dev_alloc(h, h->fg1, NI * HW1 * C1 * es);
            dev_alloc(h, h->fg2, NI * HW1 * C2 * es);
            // complex scratch: A holds dft_w output [N][Cin][H][m2] or the mixed modes; B holds X / Bh [N][Cout][H][m2]
            const size_t m2a = h->cfg.modes2, m2b = h->cfg.modes2 / h->fp0, H0 = h->cfg.H, H1 = h->cfg.H / h->fp0;
            size_t ca = NI * std::max<size_t>((size_t)h->D, C8) * H0 * m2a;          // level 0 (D or C/8 channels)
            ca = std::max(ca, NI * (size_t)C2 * H1 * m2b);                            // level 1 (up to C/2 channels)
            dev_alloc(h, h->fA, ca * 8);
            dev_alloc(h, h->fB, ca * 8);
            h->f_ca = ca;
            if (es == 2 && h->fp0 * h->fp0 * C8 > 1024) dev_alloc(h, h->kscratch, NI * HW1 * C1 * 4);      // split-K enc_conv_1 (8x8 windows)
            auto cdimf = [](int n, int k, int sdv) { return (size_t)((n + 2 * ((k - 1) / 2) - k) / sdv + 1); };
            const int H1f = h->cfg.H / h->fp0, W1f = h->cfg.W / h->fp0;
            const size_t rc1 = NI * cdimf(h->cfg.H, h->fp0, h->st[0]) * cdimf(h->cfg.W, h->fp0, h->st[0]);      // conv grids (== patch grids
            const size_t rc2 = NI * cdimf(H1f, h->fp1, h->st[1]) * cdimf(W1f, h->fp1, h->st[1]);                // without overlap)
            size_t m = rc1 * (size_t)(h->fp0 * h->fp0 * C8);                          // conv_1 windows
            m = std::max(m, rc2 * (size_t)(h->fp1 * h->fp1 * C2));                    // conv_2 windows
            if (h->overlap) {
                dev_alloc(h, h->cgrid, std::max(rc1 * C1, rc2 * C) * es);
                if (es == 2) dev_alloc(h, h->kscratch, std::max(rc1 * C1, rc2 * C) * 4);
            }
            m = std::max(m, (size_t)max_batch * h->L * (size_t)(h->fp1 * h->fp1 * C2));            // deconv_1 sub-pixel matrix
            m = std::max(m, (size_t)max_batch * HW1 * (size_t)(h->fp0 * h->fp0 * C8));             // deconv_2 sub-pixel matrix
            dev_alloc(h, h->wbuf, m * es);
            dev_alloc(h, h->dfield, (size_t)h->K * max_batch * h->D * h->cfg.H * h->cfg.W * 4);
            fno_twiddles(h);      // (a synchronous upload: here, never inside a stream capture)
        } else if (h->wide) {
            const size_t BLs = BL;
            // conv grids of the three encoder stages (== the patch grids without overlap)
            auto cdim = [](int n, int k, int s) { return (size_t)((n + 2 * ((k - 1) / 2) - k) / s + 1); };
            const size_t NIw = (size_t)max_batch * h->T;
            const int Hh1 = h->cfg.H / g.k0, Ww1 = h->cfg.W / g.k0, Hh2 = Hh1 / g.k1, Ww2 = Ww1 / g.k1;
            const size_t r1 = NIw * cdim(h->cfg.H, g.k0, h->st[0]) * cdim(h->cfg.W, g.k0, h->st[0]);
            const size_t r2 = NIw * cdim(Hh1, g.k1, h->st[1]) * cdim(Ww1, g.k1, h->st[1]);
            const size_t r3 = NIw * cdim(Hh2, g.k2, h->st[2]) * cdim(Ww2, g.k2, h->st[2]);
            size_t m = r1 * (size_t)h->K1pad;                                              // conv1 windows
            m = std::max(m, r2 * (size_t)(g.k1 * g.k1 * C1));                               // conv2 windows
            m = std::max(m, r3 * (size_t)(g.k2 * g.k2 * C2));                               // conv3 windows
            if (h->overlap) {
                dev_alloc(h, h->cgrid, std::max(std::max(r1 * C1, r2 * C2), r3 * C) * es);
                if (es == 2 && g.k2 * g.k2 * C2 > 1024) dev_alloc(h, h->kscratch, r3 * C * 4);
            }
            m = std::max(m, BLs * (size_t)(g.k2 * g.k2 * C2));                             // sub-pixel matrices of the decoder
            m = std::max(m, BLs * g.R2 * (size_t)(g.k1 * g.k1 * C1));
            m = std::max(m, BLs * g.R1 * (size_t)h->NOpad);
            dev_alloc(h, h->wbuf, m * es);
            dev_alloc(h, h->dfield, (size_t)h->K * max_batch * h->D * h->cfg.H * h->cfg.W * 4);
        }
        if (!h->h_flag) {
            CK(cudaMallocHost(reinterpret_cast<void**>(&h->h_flag), 64));
            for (auto& e : h->ev) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        }
        // the state layout depends on max_batch -> re-derived in make_state
        h->max_batch = max_batch;
        h->max_roll = max_roll;
    });
}

int64_t tante_workspace_bytes(tante_handle_t h) { return h ? h->ws_bytes : -1; }

int tante_forward(tante_handle_t h, const float* input, int32_t B, float out_T, int32_t n_cap, int32_t per_sample,
                  float* frames, float* R_t, int32_t* n_dev, int32_t* n_host, void* stream) {
    return guarded([&] {
        REQUIRE(h && input && frames, "null argument");
        REQUIRE(n_cap >= 1, "n_cap must be >= 1");
        CK(cudaSetDevice(h->device));
        ensure_ready(h, B);
        cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
        StepIO io;
        io.input = input; io.frames = frames; io.n_cap = n_cap; io.R_t = R_t; io.n_dev = n_dev;
        io.per_sample = per_sample; io.out_T = out_T;
        RolloutState rs{};
        if (h->cfg.precision == TANTE_PREC_FP32) run_step<float>(h, io, B, rs, st);
        else run_step<__nv_bfloat16>(h, io, B, rs, st);
        h->last_B = B;
        if (n_dev) CK(cudaMemcpyAsync(n_dev, h->nbuf.p, (size_t)B * 4, cudaMemcpyDeviceToDevice, st));
        if (n_host) {
            CK(cudaMemcpyAsync(h->h_flag + 8, h->nbuf.p, 4, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            *n_host = h->h_flag[8];
        }
    });
}

int tante_rollout(tante_handle_t h, const float* window, int32_t B, int32_t n_roll, float out_T, int32_t per_sample,
                  float* y_out, float* rts_out, int32_t* ns_out, int32_t* steps_out, int32_t sync, void* stream) {
    return guarded([&] {
        REQUIRE(h && window && y_out, "null argument");
        REQUIRE(n_roll >= 1, "n_roll must be >= 1");
        REQUIRE(rts_out && ns_out, "rts_out/ns_out are required");
        CK(cudaSetDevice(h->device));
        ensure_ready(h, B);
        cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
        const bool f32 = h->cfg.precision == TANTE_PREC_FP32;
        const size_t wbytes = (size_t)B * h->T * h->D * h->cfg.H * h->cfg.W * 4;
        CK(cudaMemcpyAsync(h->ring.p, window, wbytes, cudaMemcpyDeviceToDevice, st));
        RolloutState rs = make_state(h, B, n_roll);
        {
            StepIO probe; probe.per_sample = per_sample;
            const int mode0 = h->prof_on || h->debug ? 0 : h->rollout_mode;
            if (mode0 == 2 && !h->no_switch && compaction_wanted(h, probe, B, rs)) {
                rs.act = reinterpret_cast<int*>(h->state.p) + 4 * h->max_batch + 32;
                const int cand[4] = {B, (3 * B + 3) / 4, (B + 1) / 2, (B + 3) / 4};
                static const bool one_bucket = getenv("TANTE_ROLLOUT_COMPACT") && atoi(getenv("TANTE_ROLLOUT_COMPACT")) == 2;   // debug: reorder only
                for (int c : cand)
                    if (rs.n_buckets == 0 || (!one_bucket && c < rs.bucket_sz[rs.n_buckets - 1])) rs.bucket_sz[rs.n_buckets++] = c;
            }
        }
        init_state_kernel<<<(B + 127) / 128, 128, 0, st>>>(rs, B, h->T);
        CK(cudaGetLastError());
        set_rollout_ptrs_kernel<<<1, 1, 0, st>>>(const_cast<RolloutPtrs*>(rs.ptrs), y_out, rts_out, ns_out);
        CK(cudaGetLastError());
        h->launches += 2;
        StepIO io;
        io.input = reinterpret_cast<const float*>(h->ring.p);
        io.fcount = rs.fcount;
        io.ring_out = reinterpret_cast<float*>(h->ring.p); io.n_roll = n_roll;
        io.rollout = true; io.per_sample = per_sample; io.out_T = out_T;

        int mode = h->prof_on || h->debug ? 0 : h->rollout_mode;
        tante_handle_s::RollGraph* rg = nullptr;
        if (mode > 0) {
            char key[96];
            snprintf(key, sizeof(key), "%d/%d/%d/%.9g/%d", B, n_roll, per_sample, (double)out_T, mode);
            auto it = h->graphs.find(key);
            if (it == h->graphs.end()) {
                tante_handle_s::RollGraph g;
                try {
                    try {
                        if (f32) build_roll_graph<float>(h, g, io, B, rs, mode == 2);
                        else build_roll_graph<__nv_bfloat16>(h, g, io, B, rs, mode == 2);
                    } catch (const Error&) {
                        if (!(mode == 2 && rs.act)) throw;
                        // SWITCH conditional nodes unavailable: same WHILE graph without the compaction buckets
                        (void)cudaGetLastError();
                        if (g.graph) { cudaGraphDestroy(g.graph); g.graph = nullptr; }
                        h->no_switch = true;
                        rs.act = nullptr; rs.n_buckets = 0;
                        if (f32) build_roll_graph<float>(h, g, io, B, rs, true);
                        else build_roll_graph<__nv_bfloat16>(h, g, io, B, rs, true);
                    }
                } catch (const Error& e) {
                    if (mode != 2) throw;
                    // conditional nodes unavailable: fall back to per-step graphs for this handle
                    (void)cudaGetLastError();
                    h->rollout_mode = mode = 1;
                    snprintf(key, sizeof(key), "%d/%d/%d/%.9g/%d", B, n_roll, per_sample, (double)out_T, mode);
                    if (f32) build_roll_graph<float>(h, g, io, B, rs, false);
                    else build_roll_graph<__nv_bfloat16>(h, g, io, B, rs, false);
                }
                it = h->graphs.emplace(key, g).first;
            }
            rg = &it->second;
        }
        if (mode == 2) {
            // the whole `while cumulative_length < n_steps_rollout` loop (r_evaler.py:94) is ONE graph launch:
            // a WHILE node re-runs the step body until the device-side counter of unfinished trajectories is 0
            CK(cudaGraphLaunch(rg->exec, st));
            h->launches += rg->launches_per_step;      // lower bound: the body runs >= 1 time (device decides)
            h->last_graph_steps = -1;
        } else {
            // host loop with a one-step-lagged look at the device's `remaining` counter (never stalls the stream)
            int pending[2] = {0, 0};
            for (int s = 0; s < n_roll; ++s) {
                const int slot = s & 1;
                if (pending[slot]) {
                    CK(cudaEventSynchronize(h->ev[slot]));
                    pending[slot] = 0;
                    if (h->h_flag[slot] == 0) break;
                }
                if (mode == 1) { CK(cudaGraphLaunch(rg->exec, st)); h->launches += rg->launches_per_step; }
                else if (f32) run_step<float>(h, io, B, rs, st);
                else run_step<__nv_bfloat16>(h, io, B, rs, st);
                CK(cudaMemcpyAsync(h->h_flag + slot, rs.remaining, 4, cudaMemcpyDeviceToHost, st));
                CK(cudaEventRecord(h->ev[slot], st));
                pending[slot] = 1;
            }
        }
        if (steps_out) CK(cudaMemcpyAsync(steps_out, rs.steps, (size_t)B * 4, cudaMemcpyDeviceToDevice, st));
        h->last_B = B;
        if (sync) CK(cudaStreamSynchronize(st));
    });
}

int tante_set_dropout(tante_handle_t h, float p, uint64_t seed) {
    return guarded([&] {
        REQUIRE(h, "null handle");
        REQUIRE(p >= 0.f && p < 1.f, "dropout probability must be in [0, 1)");
        h->drop_p = p;
        h->drop_seed = seed;
    });
}

int64_t tante_grad_numel(tante_handle_t h) { return h ? h->flat_elems : -1; }
int64_t tante_param_grad_offset(tante_handle_t h, int32_t i) {
    if (!h || i < 0 || i >= (int32_t)h->params.size()) return -1;
    return h->params[i].flat_off;
}

int tante_train_forward(tante_handle_t h, int32_t slot, const float* input, int32_t B, float out_T, int32_t n_cap,
                        float* frames, float* R_t, int32_t* n_host, void* stream) {
    return guarded([&] {
        REQUIRE(h && input && frames, "null argument");
        REQUIRE(n_cap >= 1, "n_cap must be >= 1");
        REQUIRE(slot >= 0 && slot < (int)h->tapes.size(), "tape slot out of range: call tante_reserve(.., training = slots)");
        REQUIRE(h->T <= 16, "training supports in_T <= 16");
        CK(cudaSetDevice(h->device));
        ensure_ready(h, B);
        cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
        Tape& tp = *h->tapes[slot];
        tape_alloc(h, tp, B);
        if (h->cfg.precision == TANTE_PREC_FP32) run_step_train<float>(h, tp, input, B, out_T, n_cap, frames, R_t, st);
        else run_step_train<__nv_bfloat16>(h, tp, input, B, out_T, n_cap, frames, R_t, st);
        h->last_B = B;
        if (n_host) {
            CK(cudaMemcpyAsync(h->h_flag + 8, h->nbuf.p, 4, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            *n_host = h->h_flag[8];
        }
    });
}

int tante_backward(tante_handle_t h, int32_t slot, const float* input, const float* grad_frames, int32_t n_frames,
                   const float* grad_Rt, float* grad_input, float* grad_params, void* stream) {
    return guarded([&] {
        REQUIRE(h && input && grad_frames && grad_params, "null argument");
        REQUIRE(slot >= 0 && slot < (int)h->tapes.size(), "tape slot out of range");
        REQUIRE(n_frames >= 1, "n_frames must be >= 1");
        Tape& tp = *h->tapes[slot];
        if (!tp.valid) throw Error(TANTE_ERR_STATE, "tape slot holds no forward (or was already consumed)");
        CK(cudaSetDevice(h->device));
        cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
        backward_alloc(h, tp.B_used);
        if (h->cfg.precision == TANTE_PREC_FP32)
            run_backward<float>(h, tp, input, grad_frames, n_frames, grad_Rt, grad_input, grad_params, st);
        else
            run_backward<__nv_bfloat16>(h, tp, input, grad_frames, n_frames, grad_Rt, grad_input, grad_params, st);
        tp.valid = false;
    });
}

// Frame-table variants: the window of a call is T separate frames (device pointer of sample 0 + batch stride each).
static FrameTab make_frame_tab(const float* base, const float* const* ptrs, const int64_t* bs, int T) {
    FrameTab ft{};
    ft.on = 1;
    for (int t = 0; t < T; ++t) {
        if (!ptrs[t]) { ft.off[t] = kFrameSkip; ft.bs[t] = 0; continue; }
        const intptr_t d = reinterpret_cast<intptr_t>(ptrs[t]) - reinterpret_cast<intptr_t>(base);
        REQUIRE(d % 4 == 0 && reinterpret_cast<uintptr_t>(ptrs[t]) % 16 == 0 && bs[t] % 4 == 0,
                "frame pointers must be 16-byte aligned and batch strides multiples of 4 elements");
        ft.off[t] = (long long)(d / 4);
        ft.bs[t] = (long long)bs[t];
    }
    return ft;
}

int tante_train_forward_win(tante_handle_t h, int32_t slot, const float* const* frame_ptrs, const int64_t* frame_bstride,
                            int32_t B, float out_T, int32_t n_cap, float* frames, int64_t frames_bstride, float* R_t,
                            int32_t* n_host, void* stream) {
    return guarded([&] {
        REQUIRE(h && frame_ptrs && frame_bstride && frames, "null argument");
        REQUIRE(n_cap >= 1, "n_cap must be >= 1");
        REQUIRE(slot >= 0 && slot < (int)h->tapes.size(), "tape slot out of range: call tante_reserve(.., training = slots)");
        REQUIRE(h->T <= 16, "training supports in_T <= 16");
        REQUIRE(!h->wide && !h->fno && !h->chan, "the windowed BPTT entry points cover patch_scale <= 8 with the CNN encoder and the axes T H W L Y A");
        for (int t = 0; t < h->T; ++t) REQUIRE(frame_ptrs[t], "null frame pointer");
        REQUIRE(frames_bstride % 4 == 0, "frames_bstride must be a multiple of 4 elements");
        CK(cudaSetDevice(h->device));
        ensure_ready(h, B);
        cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
        Tape& tp = *h->tapes[slot];
        tape_alloc(h, tp, B);
        const float* base = frame_ptrs[0];
        TrainWin win;
        win.in = make_frame_tab(base, frame_ptrs, frame_bstride, h->T);
        win.frames_bs = frames_bstride;
        if (h->cfg.precision == TANTE_PREC_FP32) run_step_train<float>(h, tp, base, B, out_T, n_cap, frames, R_t, st, &win);
        else run_step_train<__nv_bfloat16>(h, tp, base, B, out_T, n_cap, frames, R_t, st, &win);
        h->last_B = B;
        if (n_host) {
            CK(cudaMemcpyAsync(h->h_flag + 8, h->nbuf.p, 4, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            *n_host = h->h_flag[8];
        }
    });
}

int tante_backward_win(tante_handle_t h, int32_t slot, const float* grad_frames, int64_t gf_bstride, int32_t n_frames,
                       const float* grad_Rt, float* const* grad_frame_ptrs, const int64_t* grad_bstride, float* grad_params,
                       void* stream) {
    return guarded([&] {
        REQUIRE(h && grad_frames && grad_params, "null argument");
        REQUIRE(slot >= 0 && slot < (int)h->tapes.size(), "tape slot out of range");
        REQUIRE(n_frames >= 1 && gf_bstride % 4 == 0, "bad gradient frame layout");
        Tape& tp = *h->tapes[slot];
        if (!tp.valid) throw Error(TANTE_ERR_STATE, "tape slot holds no forward (or was already consumed)");
        CK(cudaSetDevice(h->device));
        cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
        backward_alloc(h, tp.B_used);
        BackwardWin win;
        win.gf_bs = gf_bstride;
        float* gbase = nullptr;
        if (grad_frame_ptrs)
            for (int t = 0; t < h->T && !gbase; ++t) gbase = grad_frame_ptrs[t];
        if (gbase) win.gin = make_frame_tab(gbase, grad_frame_ptrs, grad_bstride, h->T);
        else { win.gin = FrameTab{}; win.gin.on = 1; for (int t = 0; t < 16; ++t) win.gin.off[t] = kFrameSkip; }
        if (h->cfg.precision == TANTE_PREC_FP32)
            run_backward<float>(h, tp, nullptr, grad_frames, n_frames, grad_Rt, gbase, grad_params, st, &win);
        else
            run_backward<__nv_bfloat16>(h, tp, nullptr, grad_frames, n_frames, grad_Rt, gbase, grad_params, st, &win);
        tp.valid = false;
    });
}

// Per-sample cursor variants: every sample slides over its own history (input window, then its predictions) at its own pace.
static long long elem_offset(const float* p, const float* base) {
    const intptr_t d = reinterpret_cast<intptr_t>(p) - reinterpret_cast<intptr_t>(base);
    REQUIRE(d % 16 == 0, "buffers must be 16-byte aligned");
    return (long long)(d / 4);
}

int tante_train_forward_hist(tante_handle_t h, int32_t slot, const float* input, float* pred, int64_t pred_bstride, int32_t* cursor,
                             int32_t B, float out_T, int32_t n_cap, int32_t n_steps, float* R_t, int32_t* ns, int32_t* steps,
                             int32_t* n_active, void* stream) {
    return guarded([&] {
        REQUIRE(h && input && pred && cursor && R_t && ns && steps, "null argument");
        REQUIRE(n_cap >= 1 && n_steps >= 1, "n_cap and n_steps must be >= 1");
        REQUIRE(slot >= 0 && slot < (int)h->tapes.size(), "tape slot out of range: call tante_reserve(.., training = slots)");
        REQUIRE(h->T <= 16, "training supports in_T <= 16");
        REQUIRE(!h->wide && !h->fno && !h->chan, "the windowed BPTT entry points cover patch_scale <= 8 with the CNN encoder and the axes T H W L Y A");
        const long long DHW = (long long)h->D * h->cfg.H * h->cfg.W;
        REQUIRE(pred_bstride % 4 == 0 && pred_bstride >= (long long)(n_steps + n_cap - 1) * DHW,
                "pred_bstride must be a multiple of 4 elements and hold n_steps + n_cap - 1 frames");
        REQUIRE(reinterpret_cast<uintptr_t>(input) % 16 == 0, "input must be 16-byte aligned");
        CK(cudaSetDevice(h->device));
        ensure_ready(h, B);
        cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
        Tape& tp = *h->tapes[slot];
        tape_alloc(h, tp, B);
        CK(cudaMemcpyAsync(tp.cur.p, cursor, (size_t)B * 4, cudaMemcpyDeviceToDevice, st));
        TrainWin win;
        win.in = FrameTab{};
        win.in.on = 1;
        for (int t = 0; t < h->T; ++t) { win.in.off[t] = t * DHW; win.in.bs[t] = h->T * DHW; }
        win.in.cur = reinterpret_cast<const int*>(tp.cur.p);
        win.in.hoff = elem_offset(pred, input);
        win.in.hbs = pred_bstride;
        win.frames_bs = pred_bstride;
        win.n_lim = n_steps;
        if (h->cfg.precision == TANTE_PREC_FP32) run_step_train<float>(h, tp, input, B, out_T, n_cap, pred, R_t, st, &win);
        else run_step_train<__nv_bfloat16>(h, tp, input, B, out_T, n_cap, pred, R_t, st, &win);
        hist_advance_kernel<<<1, 256, 0, st>>>(reinterpret_cast<const int*>(tp.n_arr.p), cursor, ns, steps, n_active, B, n_steps);
        CK(cudaGetLastError());
        h->launches++;
        h->last_B = B;
    });
}

int tante_backward_hist(tante_handle_t h, int32_t slot, float* grad_pred, int64_t gp_bstride, const float* grad_Rt,
                        float* grad_input, float* grad_params, void* stream) {
    return guarded([&] {
        REQUIRE(h && grad_pred && grad_params, "null argument");
        REQUIRE(slot >= 0 && slot < (int)h->tapes.size(), "tape slot out of range");
        REQUIRE(gp_bstride % 4 == 0, "gp_bstride must be a multiple of 4 elements");
        Tape& tp = *h->tapes[slot];
        if (!tp.valid) throw Error(TANTE_ERR_STATE, "tape slot holds no forward (or was already consumed)");
        REQUIRE(tp.hist, "tape slot was not written by tante_train_forward_hist");
        CK(cudaSetDevice(h->device));
        cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
        backward_alloc(h, tp.B_used);
        const long long DHW = (long long)h->D * h->cfg.H * h->cfg.W;
        BackwardWin win;
        win.gf_bs = gp_bstride;
        win.gin = FrameTab{};
        win.gin.on = 1;
        const long long gi = grad_input ? elem_offset(grad_input, grad_pred) : 0;
        for (int t = 0; t < h->T; ++t) {
            win.gin.off[t] = grad_input ? gi + t * DHW : kFrameSkip;
            win.gin.bs[t] = h->T * DHW;
        }
        win.gin.cur = reinterpret_cast<const int*>(tp.cur.p);
        win.gin.hoff = 0;
        win.gin.hbs = gp_bstride;
        if (h->cfg.precision == TANTE_PREC_FP32)
            run_backward<float>(h, tp, nullptr, grad_pred, tp.n_cap, grad_Rt, grad_pred, grad_params, st, &win);
        else
            run_backward<__nv_bfloat16>(h, tp, nullptr, grad_pred, tp.n_cap, grad_Rt, grad_pred, grad_params, st, &win);
        tp.valid = false;
    });
}

int tante_test_wgrad(int32_t use_tc, const void* A, const void* Bm, float* C, float* bias, int64_t M, int32_t N, int32_t K,
                     int32_t iters, void* stream) {
    return guarded([&] {
        REQUIRE(A && Bm && C, "null argument");
        cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
        int dev = 0, sms = 148;
        CK(cudaGetDevice(&dev));
        CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        for (int i = 0; i < std::max(1, iters); ++i) {
            if (use_tc == 1) {
                // B is stored zero-padded to a multiple of 64 columns by the caller when K % 64 != 0
                const int Kb = (K + 63) / 64 * 64;
                REQUIRE(wgrad_tc_supported(M, N, Kb, K, N, Kb, K), "shape not covered by the tcgen05 wgrad kernel");
                CK(launch_wgrad_tc(reinterpret_cast<const __nv_bfloat16*>(A), N, reinterpret_cast<const __nv_bfloat16*>(Bm), Kb,
                                   C, K, M, N, Kb, K, sms, st, bias));
            } else if (use_tc == 2) {
                CK((launch_wgrad_simt<__nv_bfloat16, __nv_bfloat16>(reinterpret_cast<const __nv_bfloat16*>(A), N,
                                                                    reinterpret_cast<const __nv_bfloat16*>(Bm), K, C, K, M, N,
                                                                    K, sms, st)));
            } else {
                CK((launch_wgrad_simt<float, float>(reinterpret_cast<const float*>(A), N, reinterpret_cast<const float*>(Bm), K,
                                                    C, K, M, N, K, sms, st)));
            }
        }
    });
}

int tante_debug_stage(tante_handle_t h, const char* stage, float* dst, int64_t cap, int64_t* numel, void* stream) {
    return guarded([&] {
        REQUIRE(h && stage && dst && numel, "null argument");
        CK(cudaSetDevice(h->device));
        cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
        const std::string s(stage);
        if (s == "enable") { h->debug = true; *numel = 0; return; }
        const int B = h->last_B;
        REQUIRE(B > 0, "no forward has run yet");
        const int64_t lat = (int64_t)B * h->T * h->L * h->C;
        const void* src = nullptr;
        int64_t n = 0;
        if (s == "latent") { src = h->x.p; n = lat; }
        else if (s == "latent_in") { REQUIRE(h->debug && h->dbg_in.p, "debug capture not enabled before reserve"); src = h->dbg_in.p; n = lat; }
        else if (s == "rt") { src = h->rt.p; n = (int64_t)h->K * h->max_batch; }
        else if (s == "deriv") {
            // decoded derivative fields [K][B][D][H][W]: re-run the fused head on the kept stage-1
            // activations with every write but the debug one disabled
            n = (int64_t)h->K * B * h->D * h->cfg.H * h->cfg.W;
            REQUIRE(cap >= n, "destination too small");
            if (h->wide) {       // the decoder already wrote the fields
                CK(cudaMemcpyAsync(dst, h->dfield.p, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
                *numel = n;
                return;
            }
            CK(cudaMemsetAsync(h->nbuf.p, 0, (size_t)B * 4, st));
            StepIO io;
            io.input = reinterpret_cast<const float*>(h->ring.p);
            RolloutState rs{};
            if (h->cfg.precision == TANTE_PREC_FP32) launch_head<float>(h, io, B, rs, dst, st);
            else launch_head<__nv_bfloat16>(h, io, B, rs, dst, st);
            *numel = n;
            return;
        }
        else throw Error(TANTE_ERR_INVALID, "unknown stage " + s);
        REQUIRE(cap >= n, "destination too small");
        CK(cudaMemcpyAsync(dst, src, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
        *numel = n;
    });
}

int64_t tante_launch_count(tante_handle_t h) { return h ? h->launches : -1; }

int tante_bench_head(tante_handle_t h, const float* u, float* frames, int32_t B, int32_t n_frames, int32_t iters,
                     float* ms_out, void* stream) {
    return guarded([&] {
        REQUIRE(h && u && frames && ms_out && n_frames >= 1 && iters >= 1, "bad argument");
        CK(cudaSetDevice(h->device));
        ensure_ready(h, B, false);
        cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
        std::vector<int> n(B, n_frames);
        CK(cudaMemcpyAsync(h->nbuf.p, n.data(), (size_t)B * 4, cudaMemcpyHostToDevice, st));
        CK(cudaStreamSynchronize(st));
        StepIO io;
        io.input = u; io.frames = frames; io.n_cap = n_frames;
        RolloutState rs{};
        auto run = [&] {
            if (h->wide) launch_emit_wide(h, io, B, rs, st);       // boundary C: Horner emit over the decoded fields
            else if (h->cfg.precision == TANTE_PREC_FP32) launch_head<float>(h, io, B, rs, nullptr, st);
            else launch_head<__nv_bfloat16>(h, io, B, rs, nullptr, st);
        };
        for (int i = 0; i < 3; ++i) run();
        cudaEvent_t e0, e1;
        CK(cudaEventCreate(&e0));
        CK(cudaEventCreate(&e1));
        CK(cudaEventRecord(e0, st));
        for (int i = 0; i < iters; ++i) run();
        CK(cudaEventRecord(e1, st));
        CK(cudaEventSynchronize(e1));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        *ms_out = ms / iters;
        h->last_B = B;
    });
}

int tante_profile(tante_handle_t h, int32_t enable) {
    return guarded([&] {
        REQUIRE(h, "null handle");
        h->prof_on = enable != 0;
        h->prof_used = 0;
        h->prof_flops = 0;
        h->prof_rec.clear();
    });
}

int tante_profile_read_class(tante_handle_t h, int32_t cls, double* ms_out, double* flops, double* bytes, int64_t* launches) {
    return guarded([&] {
        REQUIRE(h && ms_out && flops && bytes && launches, "null argument");
        CK(cudaSetDevice(h->device));
        double ms = 0, fl = 0, by = 0;
        int64_t n = 0;
        for (size_t i = 0; i + 1 < h->prof_used && i / 2 < h->prof_rec.size(); i += 2) {
            if (h->prof_rec[i / 2].cls != cls) continue;
            CK(cudaEventSynchronize(h->prof_ev[i + 1]));
            float t = 0;
            CK(cudaEventElapsedTime(&t, h->prof_ev[i], h->prof_ev[i + 1]));
            ms += t; fl += h->prof_rec[i / 2].flops; by += h->prof_rec[i / 2].bytes; ++n;
        }
        *ms_out = ms; *flops = fl; *bytes = by; *launches = n;
    });
}

int tante_profile_read(tante_handle_t h, double* gemm_ms, double* gemm_flops, int64_t* gemm_launches) {
    return guarded([&] {
        REQUIRE(h && gemm_ms && gemm_flops && gemm_launches, "null argument");
        CK(cudaSetDevice(h->device));
        double ms = 0;
        for (size_t i = 0; i + 1 < h->prof_used; i += 2) {
            CK(cudaEventSynchronize(h->prof_ev[i + 1]));
            float t = 0;
            CK(cudaEventElapsedTime(&t, h->prof_ev[i], h->prof_ev[i + 1]));
            ms += t;
        }
        *gemm_ms = ms;
        *gemm_flops = h->prof_flops;
        *gemm_launches = (int64_t)(h->prof_used / 2);
        h->prof_used = 0;
        h->prof_flops = 0;
        h->prof_rec.clear();
    });
}

int tante_mse_cl(const float* y, const float* ref, int32_t B, int32_t nf, int32_t n_use, int32_t D, int64_t HW, int32_t n_ref,
                 int32_t f0, float scale, const float* gout, float* loss_sum, float* grad_y, void* stream) {
    return guarded([&] {
        REQUIRE(y && ref && B >= 1 && nf >= 1 && n_use >= 0 && n_use <= nf && D >= 1 && HW >= 1, "bad argument");
        REQUIRE(f0 >= 0 && f0 + n_use <= n_ref, "target frames out of range");
        REQUIRE(loss_sum || grad_y, "nothing to compute");
        const long long total = (long long)B * nf * HW;
        int dev = 0, sms = 148;
        {   // launch on the device that owns the prediction tensor, whatever the caller's current device is
            cudaPointerAttributes pa{};
            if (cudaPointerGetAttributes(&pa, y) == cudaSuccess && pa.type == cudaMemoryTypeDevice) CK(cudaSetDevice(pa.device));
            else (void)cudaGetLastError();
        }
        CK(cudaGetDevice(&dev));
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms = 148;
        const unsigned grid = (unsigned)std::min<long long>((total + 255) / 256, 16LL * sms);
        mse_cf_cl_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(y, ref, B, nf, n_use, D, HW, n_ref, f0, scale,
                                                                                 gout, loss_sum, grad_y);
        CK(cudaGetLastError());
    });
}

int tante_test_block_tail(const void* att, const void* Wo, const void* W1, const void* W2, const float* vec7, const float* x_in,
                          float* x_out, void* ln_out, float* x_mid, void* ln2, void* hpre, void* hact, int32_t M, int32_t iters,
                          void* stream) {
    return guarded([&] {
        REQUIRE(att && Wo && W1 && W2 && vec7 && x_in && x_out, "null argument");
        cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
        int dev = 0, sms = 148;
        CK(cudaGetDevice(&dev));
        CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        BlockTailArgs a;
        a.att = reinterpret_cast<const __nv_bfloat16*>(att);
        a.Wo = reinterpret_cast<const __nv_bfloat16*>(Wo); a.W1 = reinterpret_cast<const __nv_bfloat16*>(W1);
        a.W2 = reinterpret_cast<const __nv_bfloat16*>(W2);
        a.bo = vec7; a.g2 = vec7 + 256; a.be2 = vec7 + 512; a.b1 = vec7 + 768; a.b2 = vec7 + 1024; a.gn = vec7 + 1280;
        a.ben = vec7 + 1536;
        a.x_in = x_in; a.x_out = x_out; a.ln_out = reinterpret_cast<__nv_bfloat16*>(ln_out);
        a.x_mid = x_mid; a.ln2 = reinterpret_cast<__nv_bfloat16*>(ln2); a.hpre = reinterpret_cast<__nv_bfloat16*>(hpre);
        a.hact = reinterpret_cast<__nv_bfloat16*>(hact);
        for (int i = 0; i < std::max(1, iters); ++i) CK(launch_block_tail_any(a, M, x_mid != nullptr, sms, st));
    });
}

int tante_comm_unique_id(void* id128) {
    return guarded([&] {
        REQUIRE(id128, "null argument");
        NcclApi& n = nccl_api();
        if (!n.ok()) throw Error(TANTE_ERR_STATE, "NCCL (libnccl.so.2) is not loadable in this process");
        NcclId id;
        const int r = n.GetUniqueId(&id);
        if (r != 0) throw Error(TANTE_ERR_CUDA, std::string("ncclGetUniqueId: ") + (n.GetErrorString ? n.GetErrorString(r) : "error"));
        memcpy(id128, id.b, sizeof(id.b));
    });
}

int tante_comm_init(tante_handle_t h, const void* id128, int32_t nranks, int32_t rank) {
    return guarded([&] {
        REQUIRE(h && id128, "null argument");
        REQUIRE(nranks >= 1 && rank >= 0 && rank < nranks, "bad rank / world size");
        NcclApi& n = nccl_api();
        if (!n.ok()) throw Error(TANTE_ERR_STATE, "NCCL (libnccl.so.2) is not loadable in this process");
        CK(cudaSetDevice(h->device));
        if (h->nccl_comm) { n.CommDestroy(h->nccl_comm); h->nccl_comm = nullptr; }
        NcclId id;
        memcpy(id.b, id128, sizeof(id.b));
        const int r = n.CommInitRank(&h->nccl_comm, nranks, id, rank);
        if (r != 0) throw Error(TANTE_ERR_CUDA, std::string("ncclCommInitRank: ") + (n.GetErrorString ? n.GetErrorString(r) : "error"));
        h->nccl_nranks = nranks;
    });
}

int tante_allreduce_grads(tante_handle_t h, float* grad, void* comm, void* stream) {
    return guarded([&] {
        REQUIRE(h && grad, "null argument");
        void* c = comm ? comm : h->nccl_comm;
        if (!c) throw Error(TANTE_ERR_STATE, "no communicator: call tante_comm_init first (or pass an ncclComm_t)");
        NcclApi& n = nccl_api();
        if (!n.ok()) throw Error(TANTE_ERR_STATE, "NCCL (libnccl.so.2) is not loadable in this process");
        CK(cudaSetDevice(h->device));
        const int r = n.AllReduce(grad, grad, (size_t)h->flat_elems, /* ncclFloat32 */ 7, /* ncclSum */ 0, c,
                                  reinterpret_cast<cudaStream_t>(stream));
        if (r != 0) throw Error(TANTE_ERR_CUDA, std::string("ncclAllReduce: ") + (n.GetErrorString ? n.GetErrorString(r) : "error"));
    });
}

int tante_optimizer_step(tante_handle_t h, float* grad, float* exp_avg, float* exp_avg_sq, float lr, float beta1, float beta2,
                         float eps, float weight_decay, int64_t step, int32_t clip_mode, float clip, float grad_scale,
                         double* grad_sumsq, void* stream) {
    return guarded([&] {
        REQUIRE(h && grad && exp_avg && exp_avg_sq, "null argument");
        REQUIRE(step >= 1, "step counts from 1");
        REQUIRE(clip_mode >= 0 && clip_mode <= 2, "clip_mode: 0 none, 1 norm, 2 value");
        REQUIRE(h->params.size() <= (size_t)kOptMaxSegs, "too many parameters");
        CK(cudaSetDevice(h->device));
        cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
        std::vector<OptSeg> segs;
        for (const Param& p : h->params) {
            if (!p.data) throw Error(TANTE_ERR_STATE, "parameter not bound: " + p.name);
            segs.push_back(OptSeg{(long long)p.flat_off, (long long)p.numel, const_cast<float*>(p.data)});
        }
        std::sort(segs.begin(), segs.end(), [](const OptSeg& a, const OptSeg& b) { return a.off < b.off; });
        dev_alloc(h, h->opt_segs, segs.size() * sizeof(OptSeg));
        dev_alloc(h, h->opt_norm, sizeof(double));
        const size_t nb = segs.size() * sizeof(OptSeg);
        if (h->opt_seg_cache.size() != nb || memcmp(h->opt_seg_cache.data(), segs.data(), nb) != 0) {
            CK(cudaMemcpyAsync(h->opt_segs.p, segs.data(), nb, cudaMemcpyHostToDevice, st));
            CK(cudaStreamSynchronize(st));
            h->opt_seg_cache.assign(reinterpret_cast<const char*>(segs.data()), reinterpret_cast<const char*>(segs.data()) + nb);
        }
        double* norm = grad_sumsq ? grad_sumsq : reinterpret_cast<double*>(h->opt_norm.p);
        const long long n = h->flat_elems;
        const unsigned grid = (unsigned)std::min<long long>((n + 255) / 256, 8LL * h->num_sms);
        if (clip_mode == 1 || grad_sumsq) {
            CK(cudaMemsetAsync(norm, 0, sizeof(double), st));
            grad_sumsq_kernel<<<grid, 256, 0, st>>>(grad, n, grad_scale, norm);
            CK(cudaGetLastError());
            h->launches++;
        }
        AdamWArgs a;
        a.gscale = grad_scale; a.clip_mode = clip_mode; a.clip = clip;
        a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.weight_decay = weight_decay;
        a.bc1 = (float)(1.0 - std::pow((double)beta1, (double)step));
        a.bc2_sqrt = (float)std::sqrt(1.0 - std::pow((double)beta2, (double)step));
        adamw_flat_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const OptSeg*>(h->opt_segs.p), (int)segs.size(), grad, exp_avg,
                                                exp_avg_sq, n, norm, a);
        CK(cudaGetLastError());
        h->launches++;
    });
    // the packed weights follow the masters: the caller runs tante_pack_params next (the host mirror does)
}

int tante_metric_moments(const float* x, const float* y, int64_t BT, int64_t HW, int32_t C, double* out, void* stream) {
    return guarded([&] {
        REQUIRE(x && y && out, "null argument");
        REQUIRE(C >= 1 && C <= kMetricMaxC, "metric kernels support 1..16 fields");
        REQUIRE(BT >= 1 && BT <= 65535 && HW >= 1, "bad shape");
        int dev = 0, sms = 148;
        {
            cudaPointerAttributes pa{};
            if (cudaPointerGetAttributes(&pa, x) == cudaSuccess && pa.type == cudaMemoryTypeDevice) CK(cudaSetDevice(pa.device));
            else (void)cudaGetLastError();
        }
        CK(cudaGetDevice(&dev));
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms = 148;
        CK(launch_metric_moments(x, y, BT, HW, C, out, sms, reinterpret_cast<cudaStream_t>(stream)));
    });
}

int tante_test_gemm(int32_t use_tc, int32_t epi, const void* A, const void* W, const float* bias, const float* resid,
                    void* C, int32_t out_bf16, int32_t M, int32_t N, int32_t K, int32_t iters, const float* ln_gamma,
                    const float* ln_beta, void* ln_out, void* stream) {
    return guarded([&] {
        REQUIRE(A && W && bias && C, "null argument");
        REQUIRE((epi >= EPI_BIAS && epi <= EPI_BIAS_RESID) || epi == EPI_BIAS_RESID_LN, "unsupported epilogue for the test hook");
        cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
        EpiParams ep;
        ep.bias = bias; ep.resid = resid; ep.ldr = N;
        ep.ln_gamma = ln_gamma; ep.ln_beta = ln_beta; ep.ln_out = ln_out;
        int dev = 0, sms = 148;
        CK(cudaGetDevice(&dev));
        CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        for (int i = 0; i < std::max(1, iters); ++i) {
            if (use_tc)
                CK(launch_gemm_tc(epi, reinterpret_cast<const __nv_bfloat16*>(A), K, reinterpret_cast<const __nv_bfloat16*>(W),
                                  K, C, N, out_bf16, M, N, K, ep, sms, st));
            else
                CK(launch_gemm_simt(epi, reinterpret_cast<const float*>(A), K, reinterpret_cast<const float*>(W), K,
                                    reinterpret_cast<float*>(C), N, M, N, K, ep, st));
        }
    });
}

}  // extern "C"
