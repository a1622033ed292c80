// tcgen05 engine: the GEMM-shaped part of the forward graph on 5th-gen tensor cores.
//
// Specialised for the shipped widths (conv channels C = 32, GRU units H = 64; any number of residual
// blocks and GRU layers; network types ResNetRNN, RNN and ResNet).  Narrower networks (C < 32, H < 64)
// run on the same kernels: tc_create pads them once with zero channels and units, which stay exactly
// zero through every layer (pad_model).  Single bf16/fp16 operands do not
// meet the 1e-3 probability contract (DESIGN.md, precision table), so every product is evaluated
// with split operands and fp32 accumulation in TMEM, in one of two formats:
//   bf16x3  a_hi w_hi + a_lo w_hi + a_hi w_lo, three kind::f16 MMAs per K = 16 chunk
//   f16e5   fp16 product + one e5m2 MMA over [a_l S | a_h / S] [w_h / S ; w_l S]: two
//           pass-equivalents (default for the 128-wide fused GRU layers of ResNetRNN; tc_ptx.cuh)
//
// Default path of a pass (at most kTcChunkTiles tiles):
//   TK2   tc_conv4_kernel        residual conv stack, two chains, operands in tensor memory
//   TK4G  tc_gru_fused2_kernel   one GRU layer (input projection + recurrence), two tiles per CTA
//   TK5   tc_head_kernel         dense 128 -> 1 + sigmoid from the partial dots of the last layer, then
//                                probabilities and / or label bits (head_output, window_io.cuh)
// (the conv stack and the GRU layer it feeds use bf16x3, the 128-wide GRU layers f16e5).
// Other shapes: tc_conv2_kernel (networks with ONE residual block), tc_conv_block_kernel (every block
// after the second of deeper stacks, once per block, from and to the K = 32 operand form),
// tc_head_conv_kernel (ResNet-only networks other than two blocks).  Layer 0 of
// RNN-only networks, whose input is 1 wide, is the KX = 1 form of TK4G: no x MMAs, the rank-1 update
// x_t * w_row is added in the epilogue; k1_fill_windows gathers that input into the conv stack's buffer.
// The conv kernels gather their input by the same rule (window_input).
//
// Data layout: a tile is 128 windows (= 128 TMEM lanes = UMMA M); a block is (tile, t), one of
// the 35 positions of those windows.  Activations that feed an MMA live in global memory as
// ready-made UMMA operands: per block plane 0 then plane 1, each [K/8][128][16 bytes], so a
// block is one contiguous cp.async.bulk (TMA) copy.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "model.cuh"
#include "tc_ptx.cuh"
#include "window_io.cuh"

namespace cf {

using namespace ptx;

constexpr int kH = 64;            // GRU units
constexpr int kC = 32;            // conv channels
constexpr int kNX = 3 * kH;       // 192 projection columns per direction (r | u | c)
constexpr int kTcChunkTiles = 2368;  // tiles per internal pass (16 tiles per CTA of the GRU kernel; 1184: -1.4 %, 4736: -1.5 %)
constexpr float kGateScale = -1.4426950408889634f;    // -log2(e)
constexpr float kCandScale = 2.8853900817779268f;     // 2 log2(e)

constexpr int kFmtBf16x3 = 0, kFmtF16E5 = 1;   // operand formats, see "operand formats" below

struct ConvParams {                    // byte offsets inside the parameter block
    static constexpr int kFloats = 10 * 32;              // a_sc b_sc a1 b1 | b2 b3 b4 b5 b6 b7
    static constexpr int kW2 = kFloats * 4;              // 3 taps x {hi, lo} x [4][32][8]
    static constexpr int kW3 = kW2 + 3 * 4096;
    static constexpr int kW45 = kW3 + 4096;              // {hi, lo} x [4][64][8]
    static constexpr int kW6 = kW45 + 8192;
    static constexpr int kW7 = kW6 + 3 * 4096;
    static constexpr int kBytes = kW7 + 4096;            // 42240
};

// ====================================================================== weight packing (host)
// B operand of D = A * W for W [K][N] row-major: stored [plane][K/8][N][8] with plane 0 = hi.
static void pack_b_operand(const float* w, int K, int N, int ldw, int col0, std::vector<__nv_bfloat16>* out,
                           float scale = 1.f, int n_split = 1 << 30, float scale_hi = 1.f) {
    const size_t plane = (size_t)K * N;
    const size_t base = out->size();
    out->resize(base + 2 * plane);
    __nv_bfloat16* hi = out->data() + base;
    __nv_bfloat16* lo = hi + plane;
    for (int k = 0; k < K; ++k)
        for (int n = 0; n < N; ++n) {
            const float v = w[(size_t)k * ldw + col0 + n] * (n < n_split ? scale : scale_hi);
            const __nv_bfloat16 h = __float2bfloat16_rn(v);
            const __nv_bfloat16 l = __float2bfloat16_rn(v - __bfloat162float(h));
            const size_t idx = ((size_t)(k / 8) * N + n) * 8 + (k % 8);
            hi[idx] = h;
            lo[idx] = l;
        }
}

// B operand in the "f16e5" format (tc_ptx.cuh): plane 0 = fp16(S w_h) [K/8][N][8] (the A side stores
// a_h / S); plane 1 = e5m2 [2K/16][N][16]: per chunk of 16 K-rows first the 16 fp16 parts / S, then the
// 16 remainders * S - the K' order the A-side producers use.  Same byte count and the same per-chunk
// descriptor offsets as the split-bf16 layout.  Needs |w| < 65504 / S (tc_create checks).
static void pack_b_operand_f16e5(const float* w, int K, int N, int ldw, int col0, std::vector<__nv_bfloat16>* out,
                                 float scale = 1.f, int n_split = 1 << 30, float scale_hi = 1.f) {
    const size_t plane = (size_t)K * N;
    const size_t base = out->size();
    out->resize(base + 2 * plane);
    uint16_t* main = reinterpret_cast<uint16_t*>(out->data() + base);
    uint8_t* corr = reinterpret_cast<uint8_t*>(out->data() + base + plane);
    for (int k = 0; k < K; ++k)
        for (int n = 0; n < N; ++n) {
            const float v = w[(size_t)k * ldw + col0 + n] * (n < n_split ? scale : scale_hi);
            const __half h = __float2half_rn(v);
            const float hf = __half2float(h);
            const __half hs = __float2half_rn(hf * kCorrScale);          // exact: a power-of-two scale
            main[((size_t)(k / 8) * N + n) * 8 + (k % 8)] = *reinterpret_cast<const uint16_t*>(&hs);
            const int c = k / 16, kc = k % 16;
            corr[((size_t)(2 * c) * N + n) * 16 + kc] = (uint8_t)__nv_cvt_float_to_fp8(hf / kCorrScale, __NV_SATFINITE, __NV_E5M2);
            corr[((size_t)(2 * c + 1) * N + n) * 16 + kc] = (uint8_t)__nv_cvt_float_to_fp8((v - hf) * kCorrScale, __NV_SATFINITE, __NV_E5M2);
        }
}

struct TcLayer {
    int in = 0;                       // input features of this GRU layer (1, 32 or 128)
    DevBuf wfused;                    // [dir]{Wgx, Wcx, Wgh, Wch} as in GruF2Cfg (no Wgx, Wcx for in = 1), exponent domain
    int fmt = 0;                      // operand format of wfused / of this layer's x and state operands
    DevBuf bz;                        // float [384] biases in the exponent domain
    DevBuf wxz;                       // float [384] the single x row of gates / candidate kernels, exponent domain (in == 1)
};

struct TcEngine {
    DevBuf conv_params;               // TK2 parameter block (see ConvParams), then [conv_nres - 2] parameter blocks of
                                      // tc_conv_block_kernel (block-1 slots); empty = no residual blocks
    int conv_nres = 0;
    std::vector<TcLayer> layers;
    DevBuf head_w;                    // float [128]
    float head_b = 0.f;
    int n_sms = 148;
#ifdef CF_TRACE_PROBES
    bool trace_done = false;
    const char* trace_path = nullptr; // CF_TC_TRACE=<file>: in-kernel timeline of one TK4G launch (debug; results unaffected)
#endif
    int fmt = kFmtBf16x3;             // operand format of the 128-wide GRU layers (kFmtF16E5 unless the network is not
                                      // covered by f16e5 kernels or its weights are out of fp16 range); the conv stack
                                      // and the first GRU layer (input = conv output) always run bf16x3
};

bool tc_supported(const HostModel& hm) {
    if (hm.n_res() > 0 && hm.conv_channels() > kC) return false;     // any number of residual blocks
    if (hm.n_rnn() > 0 && hm.desc.layer_size > kH) return false;      // any number of GRU layers
    return true;
}

// The network padded to C = 32 channels and H = 64 units with zero weights and biases.  A zero channel stays
// relu(0) = 0; a zero unit keeps h = 0 through every GRU step (candidate tanh(0) = 0, h' = u 0 + (1 - u) 0);
// zero rows add nothing to the real outputs.  So the padded network computes exactly what the narrow one does.
// Layout: channel c stays at c; unit j of each gate group (r, u, candidate) stays at j of its 64-wide group;
// a 2H-wide input [fw | bw] (GRU layers after the first, the dense head) puts fw unit j at j and bw unit j at 64 + j.
static HostModel pad_model(const HostModel& hm) {
    HostModel p = hm;
    if (hm.n_res() > 0) {
        const int C = hm.conv_channels();
        p.desc.layer_size_res = kC;
        for (size_t i = 0; i < hm.convs.size(); ++i) {
            const ConvLayer& s = hm.convs[i];
            ConvLayer& d = p.convs[i];
            const bool scalar_in = i < 2;                 // the two Cin = 1 convolutions of block 0
            d.cin = scalar_in ? 1 : kC;
            d.cout = kC;
            d.w.assign((size_t)d.k * d.cin * kC, 0.f);
            d.b.assign(kC, 0.f);
            for (int co = 0; co < C; ++co) d.b[co] = s.b[co];
            for (int k = 0; k < s.k; ++k)
                for (int ci = 0; ci < s.cin; ++ci)
                    for (int co = 0; co < C; ++co) d.w[((size_t)k * d.cin + ci) * kC + co] = s.w[((size_t)k * s.cin + ci) * C + co];
        }
    }
    auto unit2 = [](int r, int H) { return r < H ? r : kH + (r - H); };       // row of a [fw | bw] input
    if (hm.n_rnn() > 0) {
        const int H = hm.desc.layer_size;
        p.desc.layer_size = kH;
        auto col = [&](int j) { return (j / H) * kH + j % H; };                // column of an r | u | c group
        for (size_t i = 0; i < hm.gru.size(); ++i) {
            const GruDir& s = hm.gru[i];
            GruDir& d = p.gru[i];
            const bool first = i < 2;
            d.in = first ? (hm.n_res() > 0 ? kC : 1) : 2 * kH;
            d.h = kH;
            d.wx.assign((size_t)d.in * kNX, 0.f);
            d.bx.assign(kNX, 0.f);
            d.wgh.assign((size_t)kH * 2 * kH, 0.f);
            d.wch.assign((size_t)kH * kH, 0.f);
            for (int r = 0; r < s.in; ++r)
                for (int j = 0; j < 3 * H; ++j) d.wx[(size_t)(first ? r : unit2(r, H)) * kNX + col(j)] = s.wx[(size_t)r * 3 * H + j];
            for (int j = 0; j < 3 * H; ++j) d.bx[col(j)] = s.bx[j];
            for (int r = 0; r < H; ++r) {
                for (int j = 0; j < 2 * H; ++j) d.wgh[(size_t)r * 2 * kH + col(j)] = s.wgh[(size_t)r * 2 * H + j];
                for (int j = 0; j < H; ++j) d.wch[(size_t)r * kH + j] = s.wch[(size_t)r * H + j];
            }
        }
        p.head_w.assign(2 * kH, 0.f);
        for (int r = 0; r < 2 * H; ++r) p.head_w[unit2(r, H)] = hm.head_w[r];
    } else {
        p.head_w.assign(kC, 0.f);
        std::copy(hm.head_w.begin(), hm.head_w.end(), p.head_w.begin());
    }
    return p;
}

void EngineDelete::operator()(TcEngine* e) const { delete e; }

static int tc_set_attributes();

int tc_create(const HostModel& narrow, TcEnginePtr* out) {
    CF_TRY(tc_set_attributes());
    TcEnginePtr e(new TcEngine());
    int dev = 0;
    CF_CUDA(cudaGetDevice(&dev));
    CF_CUDA(cudaDeviceGetAttribute(&e->n_sms, cudaDevAttrMultiProcessorCount, dev));
    const HostModel hm = pad_model(narrow);          // everything below, the operand format included, sees C = 32 / H = 64
#ifdef CF_TRACE_PROBES
    e->trace_path = getenv("CF_TC_TRACE");
#endif
    {
        // fp16 + e5m2 operands need every tensor-core kernel of the pass to speak the format: the default
        // conv stack (two residual blocks) followed by fused GRU layers only
        const bool covered = (hm.desc.network_type == CF_NET_RESNET_RNN && hm.n_res() == 2 && hm.conv_channels() == kC) ||
                             hm.desc.network_type == CF_NET_RNN;
        float wmax = 0.f;                             // the fp16 weight plane is stored times S = 64
        for (const GruDir& g : hm.gru) {
            for (float v : g.wx) wmax = std::max(wmax, std::fabs(v));
            for (float v : g.wgh) wmax = std::max(wmax, std::fabs(v));
            for (float v : g.wch) wmax = std::max(wmax, std::fabs(v));
        }
        const bool in_range = wmax * kCandScale * kCorrScale < 60000.f;
        e->fmt = covered && in_range ? kFmtF16E5 : kFmtBf16x3;
    }
    if (hm.n_res() >= 1) {
        // TK2 parameter block: fp32 vectors, then the B operands, split bf16 (see ConvParams).  Blocks 0 and 1 go
        // to TK2; every further block b gets a block of its own with only the block-1 slots filled, from convs[4 b..].
        const int n_extra = std::max(hm.n_res() - 2, 0);
        std::vector<uint8_t> all((size_t)(1 + n_extra) * ConvParams::kBytes, 0);
        uint8_t* blk = all.data();
        float* fp = reinterpret_cast<float*>(blk);
        auto put = [&](int slot, const std::vector<float>& v) { memcpy(fp + 32 * slot, v.data(), 32 * sizeof(float)); };
        auto put_w = [&](int off, const float* w, int n, int ldw, int col0, int dst_col0, int n_total) {
            // pack a [32][n] matrix into columns [dst_col0, dst_col0 + n) of a {hi, lo} x [4][n_total][8] operand
            __nv_bfloat16* hi = reinterpret_cast<__nv_bfloat16*>(blk + off);
            __nv_bfloat16* lo = hi + 32 * n_total;
            for (int k = 0; k < 32; ++k)
                for (int j = 0; j < n; ++j) {
                    const float v = w[(size_t)k * ldw + col0 + j];
                    const __nv_bfloat16 h = __float2bfloat16_rn(v);
                    const size_t idx = ((size_t)(k / 8) * n_total + dst_col0 + j) * 8 + (k % 8);
                    hi[idx] = h;
                    lo[idx] = __float2bfloat16_rn(v - __bfloat162float(h));
                }
        };
        auto put_block1 = [&](int i) {                    // a residual block with a 32-wide input, convs[i .. i + 3]
            put(6, hm.convs[i].b); put(7, hm.convs[i + 1].b); put(8, hm.convs[i + 2].b); put(9, hm.convs[i + 3].b);
            put_w(ConvParams::kW45, hm.convs[i].w.data(), 32, 32, 0, 0, 64);           // shortcut columns 0..31
            put_w(ConvParams::kW45, hm.convs[i + 1].w.data(), 32, 32, 0, 32, 64);      // p1 columns 32..63
            for (int tap = 0; tap < 3; ++tap) put_w(ConvParams::kW6 + tap * 4096, hm.convs[i + 2].w.data() + tap * 32 * 32, 32, 32, 0, 0, 32);
            put_w(ConvParams::kW7, hm.convs[i + 3].w.data(), 32, 32, 0, 0, 32);
        };
        put(0, hm.convs[0].w); put(1, hm.convs[0].b);          // shortcut of block 0: [1][1][32]
        put(2, hm.convs[1].w); put(3, hm.convs[1].b);
        put(4, hm.convs[2].b); put(5, hm.convs[3].b);
        for (int tap = 0; tap < 3; ++tap) put_w(ConvParams::kW2 + tap * 4096, hm.convs[2].w.data() + tap * 32 * 32, 32, 32, 0, 0, 32);
        put_w(ConvParams::kW3, hm.convs[3].w.data(), 32, 32, 0, 0, 32);
        if (hm.n_res() >= 2) put_block1(4);
        for (int b = 2; b < hm.n_res(); ++b) {
            blk = all.data() + (size_t)(b - 1) * ConvParams::kBytes;
            fp = reinterpret_cast<float*>(blk);
            put_block1(4 * b);
        }
        CF_TRY(e->conv_params.upload(all));
        e->conv_nres = hm.n_res();
    }
    e->layers.resize(hm.n_rnn());
    for (int l = 0; l < hm.n_rnn(); ++l) {
        TcLayer& L = e->layers[l];
        L.in = hm.gru[2 * l].in;
        // The layer fed by the conv stack stays bf16x3: it contributes nearly all of f16e5's extra error
        // (emulation: 5.8e-5 of 6.1e-5; conv activations span 2^-10 .. 60 and would need an fp16 range
        // guard) and its K = 32 input part is too small to gain from the cheaper passes.
        L.fmt = L.in == kC ? kFmtBf16x3 : e->fmt;
        std::vector<__nv_bfloat16> wf;
        for (int d = 0; d < 2; ++d) {
            const GruDir& g = hm.gru[2 * l + d];
            // exponent domain: gates scaled by -log2(e), candidate by 2 log2(e) (see sigmoid4_z / tanh4_z)
            // x rows of gates/kernel and candidate/kernel side by side: one N = 192 operand
            auto pack = L.fmt == kFmtF16E5 ? pack_b_operand_f16e5 : pack_b_operand;
            if (L.in > 1) pack(g.wx.data(), L.in, kNX, kNX, 0, &wf, kGateScale, 2 * kH, kCandScale);
            pack(g.wgh.data(), kH, 2 * kH, 2 * kH, 0, &wf, kGateScale, 1 << 30, 1.f);
            pack(g.wch.data(), kH, kH, kH, 0, &wf, kCandScale, 1 << 30, 1.f);
        }
        CF_TRY(L.wfused.upload(wf));
        std::vector<float> bz(2 * kNX);
        for (int d = 0; d < 2; ++d)
            for (int j = 0; j < kNX; ++j)
                bz[d * kNX + j] = hm.gru[2 * l + d].bx[j] * (j < 2 * kH ? kGateScale : kCandScale);
        CF_TRY(L.bz.upload(bz));
        if (L.in == 1) {
            // RNN-only layer 0 (neural_network.py:17-18): the x part of concat([x, h]) W is a rank-1 update
            // x_t * w_row, added to the bias in the epilogue of the fused kernel - no MMA
            std::vector<float> wxz(2 * kNX);
            for (int d = 0; d < 2; ++d)
                for (int j = 0; j < kNX; ++j)
                    wxz[d * kNX + j] = hm.gru[2 * l + d].wx[j] * (j < 2 * kH ? kGateScale : kCandScale);
            CF_TRY(L.wxz.upload(wxz));
        }
    }
    CF_TRY(e->head_w.upload(hm.head_w));
    e->head_b = hm.head_b;
    *out = std::move(e);
    return CF_OK;
}

int tc_operand_format(const TcEngine* e) { return e ? e->fmt : 0; }

// ====================================================================== TK2: residual conv stack
// Fuses, per tile of 128 windows: median/MAD normalisation of the raw signal, the 35-sample
// window gather with zero padding, and the residual blocks of resnet_class.py:44-82 with their
// batch-norms folded in.  The two Cin = 1 convolutions of block 0 are evaluated in fp32 on CUDA
// cores from the normalised sample (it is never rounded to bf16); every 32 -> 32 convolution is
// an implicit GEMM on tcgen05 with split-bf16 operands: rows = the 128 windows of one position
// t, so the k = 3 taps are whole 128-row operand slices of t-1, t, t+1 and the "same" padding at
// the window edges is simply a skipped MMA.
//
constexpr uint32_t kSliceBytes = 2u * 128 * kC * 2;       // one position of a tile as A operand: 16 KB
constexpr uint32_t kConvSmem = ConvParams::kBytes + 10 * kSliceBytes + 35 * 128 * 4 + 256;   // tc_conv2: O1 ring of 4

// ====================================================================== TK2, one residual block
// Every operand slice in shared memory; the two MMA stages of the block are skewed over time so that
// both are issued in one batch per iteration u = 0..36:
//   o2[u-1] = relu(conv3(o1) + b2)                  TMEM 0
//   o3[u-2] -> y0 = relu(relu(o3 + b3) + sc0)       TMEM 32; y0 is the kernel's output
// followed by ONE epilogue pass that consumes both accumulators (all TMEM loads in flight at once),
// writes the next operand, and computes o1[u+2] = relu(x a1 + b1) on CUDA cores (ring of 4 slices).
// One commit + one "operands ready" barrier per iteration.
//   warps 0-7 : epilogue; thread = (window, 16 of the 32 channels)
//   warp 8    : MMA issuer (warp-converged issue, elected lane)
__device__ __forceinline__ void store_a_row16(uint8_t* slice, int row, int c0, const float* v) {
#pragma unroll
    for (int g = 0; g < 2; ++g) {
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) split_bf16x2(v[g * 8 + 2 * i], v[g * 8 + 2 * i + 1], hi[i], lo[i]);
        uint8_t* dst = slice + (c0 / 8 + g) * 2048 + row * 16;
        *reinterpret_cast<uint4*>(dst) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(dst + 8192) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
}

template <int N>
__device__ __forceinline__ void conv_mma_pred(uint32_t tmem_d, uint32_t a_slice, uint32_t w_mat, bool first, uint32_t elected) {
    constexpr uint32_t idesc = make_idesc_bf16(128, N);
#pragma unroll
    for (int pass = 0; pass < 3; ++pass) {
        const uint32_t ap = a_slice + (pass == 1 ? 8192u : 0u);
        const uint32_t wp = w_mat + (pass == 2 ? (uint32_t)(kC * N * 2) : 0u);
#pragma unroll
        for (int kk = 0; kk < 2; ++kk)
            umma_bf16_pred(tmem_d, make_smem_desc(ap + kk * 4096, 2048, 128), make_smem_desc(wp + kk * 2 * (N * 16), N * 16, 128),
                           idesc, !(first && pass == 0 && kk == 0), elected);
    }
}

__global__ void __launch_bounds__(288, 1)
tc_conv2_kernel(const uint8_t* __restrict__ params, const int16_t* __restrict__ raw, const double* __restrict__ stats,
                const float* __restrict__ xwin, const int64_t* __restrict__ src, const int32_t* __restrict__ valid,
                const int32_t* __restrict__ read, int64_t tile0, int n_tiles, __nv_bfloat16* __restrict__ y_out) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* prm = smem;
    uint8_t* o1 = smem + ConvParams::kBytes;          // ring of 4 slices (o1 is produced two positions ahead)
    uint8_t* o2 = o1 + 4 * kSliceBytes;
    uint8_t* y0 = o2 + kSliceBytes;
    uint8_t* p1 = y0 + kSliceBytes;                   // ring of 3 slices
    uint8_t* p2 = p1 + 3 * kSliceBytes;
    float* xs = reinterpret_cast<float*>(p2 + kSliceBytes);      // [35][128]
    uint64_t* bars = reinterpret_cast<uint64_t*>(xs + 35 * 128); // bar_ready, bar_mma, bar_prm
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);
    const float* fp = reinterpret_cast<const float*>(prm);
    uint64_t* bar_ready = &bars[0];
    uint64_t* bar_mma = &bars[1];
    uint64_t* bar_prm = &bars[2];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        mbar_init(bar_ready, 8);
        mbar_init(bar_mma, 1);
        mbar_init(bar_prm, 1);
        fence_mbar_init();
        mbar_expect_tx(bar_prm, ConvParams::kBytes);
        bulk_g2s(prm, params, ConvParams::kBytes, bar_prm);
    }
    if (warp == 8) tmem_alloc<512>(tmem_slot);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    constexpr int kLastU = kWindow + 1;               // o3[34] at u = 36
    mbar_wait(bar_prm, 0);

    if (warp == 8) {
        // ------------------------------------------------------------ issuer (all lanes converged)
        const uint32_t elected = elect_one();
        const uint32_t prm_u = smem_u32(prm);
        const uint32_t o1_u = smem_u32(o1), o2_u = smem_u32(o2);
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            for (int u = 0; u <= kLastU; ++u, ++it) {
                mbar_wait(bar_ready, it & 1);
                tc_fence_after_sync();
                const int t1 = u - 1, t2 = u - 2;
                if (t1 >= 0 && t1 < kWindow) {
                    bool first = true;
#pragma unroll
                    for (int tap = 0; tap < 3; ++tap) {
                        const int tt = t1 + tap - 1;
                        if (tt < 0 || tt >= kWindow) continue;
                        conv_mma_pred<32>(tmem + 0, o1_u + (tt & 3) * kSliceBytes, prm_u + ConvParams::kW2 + tap * 4096, first, elected);
                        first = false;
                    }
                }
                if (t2 >= 0 && t2 < kWindow) conv_mma_pred<32>(tmem + 32, o2_u, prm_u + ConvParams::kW3, true, elected);
                umma_commit_pred(bar_mma, elected);
            }
        }
    } else {
        // ------------------------------------------------------------ epilogue
        const int q = warp & 3, ch = warp >> 2;
        const int row = q * 32 + lane;
        const int c0 = ch * 16;
        const uint32_t t_lane = tmem + ((uint32_t)(q * 32) << 16) + c0;
        auto relu_bias = [&](uint32_t* r, int slot, float* v) {
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
                const float4 b4 = *reinterpret_cast<const float4*>(fp + 32 * slot + c0 + i);
                v[i] = fmaxf(__uint_as_float(r[i]) + b4.x, 0.f);
                v[i + 1] = fmaxf(__uint_as_float(r[i + 1]) + b4.y, 0.f);
                v[i + 2] = fmaxf(__uint_as_float(r[i + 2]) + b4.z, 0.f);
                v[i + 3] = fmaxf(__uint_as_float(r[i + 3]) + b4.w, 0.f);
            }
        };
        auto make_o1 = [&](int t) {               // o1[t] = relu(x a1 + b1) on CUDA cores
            const float x = xs[t * 128 + row];
            float v[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = fmaxf(fmaf(x, fp[64 + c0 + i], fp[96 + c0 + i]), 0.f);
            store_a_row16(o1 + (t & 3) * kSliceBytes, row, c0, v);
        };
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            // ---- gather + normalise (infer.py:101-105, 32-38): the two threads of a window split its 35 samples
            asm volatile("bar.sync 1, 256;" ::: "memory");        // previous tile's readers of xs are done
            {
                const WindowInput x = window_input(raw, stats, xwin, src, valid, read, (tile0 + tile) * kTileWindows + row);
                const int tb = ch ? 18 : 0, te = ch ? kWindow : 18;
                for (int t = tb; t < te; ++t) xs[t * 128 + row] = x(t);
            }
            asm volatile("bar.sync 1, 256;" ::: "memory");
            make_o1(0);
            make_o1(1);
            fence_proxy_async_smem();
            tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_ready);
            for (int u = 0; u <= kLastU; ++u, ++it) {
                const int t1 = u - 1, t2 = u - 2;
                const bool h1 = t1 >= 0 && t1 < kWindow, h2 = t2 >= 0 && t2 < kWindow;
                mbar_wait(bar_mma, it & 1);
                tc_fence_after_sync();
                uint32_t r1[16], r2[16];
                if (h1) tmem_ld16_nowait(t_lane + 0, r1);
                if (h2) tmem_ld16_nowait(t_lane + 32, r2);
                tmem_ld_wait();
                tc_fence_before_sync();
                float v[16];
                if (h1) { relu_bias(r1, 4, v); store_a_row16(o2, row, c0, v); }                  // b2
                if (h2) {
                    relu_bias(r2, 5, v);                                                         // b3
                    const float x = xs[t2 * 128 + row];
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i] + fmaf(x, fp[c0 + i], fp[32 + c0 + i]), 0.f);   // + shortcut
                    store_a_row16(reinterpret_cast<uint8_t*>(y_out) + ((size_t)tile * kWindow + t2) * kSliceBytes, row, c0, v);
                }
                // operands of the next MMA batch are complete: hand over, then make o1 two positions ahead,
                // which that batch does not read
                if (u < kLastU) {
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_ready);
                }
                if (u + 2 < kWindow) make_o1(u + 2);
            }
        }
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 8) tmem_dealloc<512>(tmem);
}

// ====================================================================== operand formats
// FMT 0 = split bf16, three MMAs per K = 16 chunk (bf16x3).  FMT 1 = fp16 + e5m2 corrections, two
// MMAs per chunk ("f16e5", tc_ptx.cuh).  Both use the same byte positions everywhere: plane 0 holds
// the 16-bit main operand, plane 1 (same size) the bf16 remainders or, per chunk of 16 K values,
// 16 remainder bytes followed by 16 down-scaled main bytes.

// Four consecutive values i..i+3 (i = 0, 4, 8, 12 inside a 16-value chunk) into the chunk's 8 main
// words and 8 second-plane words.
template <int FMT>
__device__ __forceinline__ void split4(float v0, float v1, float v2, float v3, int i, uint32_t* m8, uint32_t* s8) {
    if (FMT == kFmtBf16x3) {
        split_bf16x2(v0, v1, m8[i >> 1], s8[i >> 1]);
        split_bf16x2(v2, v3, m8[(i >> 1) + 1], s8[(i >> 1) + 1]);
    } else {
        uint32_t la, lb;
        split_f16e5x2(v0, v1, m8[i >> 1], la);
        split_f16e5x2(v2, v3, m8[(i >> 1) + 1], lb);
        s8[i >> 2] = la | (lb << 16);
        s8[4 + (i >> 2)] = f16e5_hi4(m8[i >> 1], m8[(i >> 1) + 1]);
    }
}

// 16 channels of one window into an operand slice {plane 0, plane 1} x [4][128][8 x 16 bit] in shared
// or global memory / into a K = 16 chunk of a TMEM operand slot (plane 1 sixteen columns further).
template <int FMT>
__device__ __forceinline__ void store_a_row16_f(uint8_t* slice, int row, int c0, const float* v) {
    uint32_t m8[8], s8[8];
#pragma unroll
    for (int i = 0; i < 16; i += 4) split4<FMT>(v[i], v[i + 1], v[i + 2], v[i + 3], i, m8, s8);
    uint8_t* dst = slice + (c0 / 8) * 2048 + row * 16;
    *reinterpret_cast<uint4*>(dst) = make_uint4(m8[0], m8[1], m8[2], m8[3]);
    *reinterpret_cast<uint4*>(dst + 2048) = make_uint4(m8[4], m8[5], m8[6], m8[7]);
    *reinterpret_cast<uint4*>(dst + 8192) = make_uint4(s8[0], s8[1], s8[2], s8[3]);
    *reinterpret_cast<uint4*>(dst + 8192 + 2048) = make_uint4(s8[4], s8[5], s8[6], s8[7]);
}
template <int FMT>
__device__ __forceinline__ void store_a_tmem16_f(uint32_t t_slot, const float* v) {
    uint32_t m8[8], s8[8];
#pragma unroll
    for (int i = 0; i < 16; i += 4) split4<FMT>(v[i], v[i + 1], v[i + 2], v[i + 3], i, m8, s8);
    tmem_st8_u32(t_slot, m8);
    tmem_st8_u32(t_slot + 16, s8);
}

// ====================================================================== TK2 v4: two chains, k = 3 operands in tensor memory
// The two residual blocks as two independently clocked chains, with the A operands of both k = 3 convolutions (the o1 and p1 rings) and y0 held in
// TENSOR MEMORY: an N = 32 MMA that reads its 4 KB A operand from shared memory is bound by that
// read (~38 cycles for 17 cycles of math); the ".ts" form only fetches the 1 KB weight slice.
// To make room the [sc1|p1] accumulator is single-buffered: the epilogue thread that reads p1 also
// takes its 16 channels of sc1 (+ b4) and parks them for three positions in a thread-private
// shared-memory ring.  o2 and p2 (k = 1 operands, 6 MMAs each) stay in shared memory.
// TMEM: o2 0, o3 32, p2 64, p3 96, [sc1|p1] 128 | y0 ring of 3 at 192 + 32 k | o1 ring of 4 at
// 288 + 32 k | p1 ring of 3 at 416 + 32 k.  Operand slot: hi K 0-15 | hi K 16-31 | lo K 0-15 | lo K 16-31.
constexpr uint32_t kConv4Smem = ConvParams::kBytes + 2 * kSliceBytes + 4 * (32 * 128 * 4) + 35 * 128 * 4 + 256;

// conv_mma_pred with the A operand in tensor memory (".ts" form)
template <int N>
__device__ __forceinline__ void conv_mma_ts_pred(uint32_t tmem_d, uint32_t tmem_a, uint32_t w_mat, bool first, uint32_t elected) {
    constexpr uint32_t idesc = make_idesc_bf16(128, N);
#pragma unroll
    for (int pass = 0; pass < 3; ++pass) {
        const uint32_t ap = tmem_a + (pass == 1 ? 16u : 0u);
        const uint32_t wp = w_mat + (pass == 2 ? (uint32_t)(kC * N * 2) : 0u);
#pragma unroll
        for (int kk = 0; kk < 2; ++kk)
            umma_bf16_ts_pred(tmem_d, ap + kk * 8, make_smem_desc(wp + kk * 2 * (N * 16), N * 16, 128), idesc,
                              !(first && pass == 0 && kk == 0), elected);
    }
}

__global__ void __launch_bounds__(576, 1)
tc_conv4_kernel(const uint8_t* __restrict__ params, const int16_t* __restrict__ raw, const double* __restrict__ stats,
                const float* __restrict__ xwin, const int64_t* __restrict__ src, const int32_t* __restrict__ valid,
                const int32_t* __restrict__ read, int64_t tile0, int n_tiles, __nv_bfloat16* __restrict__ y_out,
                const float* __restrict__ head_w, float* __restrict__ head_part) {
    // head_w != nullptr (ResNet-only network, resnet_class.py:23): the dense 32 -> 1 layer is taken in this epilogue -
    // every thread writes the partial dot of its 16 channels to head_part[(block * 2 + half) * 128 + window] and the
    // 128 B/sample operand block is never stored; tc_head_kernel adds the two halves.
    // Every operand, the output (the first GRU layer's x operand) included, is split bf16: the epilogue, not the
    // tensor pipe, bounds this kernel and the bf16 split is the cheaper one.
    constexpr int kFmt = kFmtBf16x3;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* prm = smem;
    uint8_t* o2 = smem + ConvParams::kBytes;
    uint8_t* p2 = o2 + kSliceBytes;
    float* sc_ring = reinterpret_cast<float*>(p2 + kSliceBytes);   // [4][32][128]
    float* xs = sc_ring + 4 * 32 * 128;                             // [35][128]
    uint64_t* bars = reinterpret_cast<uint64_t*>(xs + 35 * 128);
    uint64_t* bar_ready_x = &bars[0];
    uint64_t* bar_mma_x = &bars[1];
    uint64_t* bar_ready_y = &bars[2];
    uint64_t* bar_mma_y = &bars[3];
    uint64_t* bar_prm = &bars[4];
    uint64_t* bar_y0_full = &bars[5];                 // [3]
    uint64_t* bar_y0_empty = &bars[8];                // [3]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 11);
    const float* fp = reinterpret_cast<const float*>(prm);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        mbar_init(bar_ready_x, 8);
        mbar_init(bar_mma_x, 1);
        mbar_init(bar_ready_y, 8);
        mbar_init(bar_mma_y, 1);
        mbar_init(bar_prm, 1);
        for (int i = 0; i < 3; ++i) { mbar_init(&bar_y0_full[i], 8); mbar_init(&bar_y0_empty[i], 1); }
        fence_mbar_init();
        mbar_expect_tx(bar_prm, ConvParams::kBytes);
        bulk_g2s(prm, params, ConvParams::kBytes, bar_prm);
    }
    if (warp == 16) tmem_alloc<512>(tmem_slot);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    constexpr int kLastX = kWindow + 1;               // o3[34] at u = 36
    constexpr int kFirstY = 3, kLastY = kWindow + 5;  // [sc1|p1][0] at u = 3, p3[34] at u = 40
    constexpr uint32_t kTmScp1 = 128, kTmY0 = 192, kTmO1 = 288, kTmP1 = 416;
    mbar_wait(bar_prm, 0);

    if (warp == 16) {
        // ------------------------------------------------------------ issuer of chain X
        const uint32_t elected = elect_one();
        const uint32_t prm_u = smem_u32(prm), o2_u = smem_u32(o2);
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            for (int u = 0; u <= kLastX; ++u, ++it) {
                mbar_wait(bar_ready_x, it & 1);
                tc_fence_after_sync();
                const int t1 = u - 1, t2 = u - 2;
                if (t1 >= 0 && t1 < kWindow) {
                    bool first = true;
#pragma unroll
                    for (int tap = 0; tap < 3; ++tap) {
                        const int tt = t1 + tap - 1;
                        if (tt < 0 || tt >= kWindow) continue;
                        conv_mma_ts_pred<32>(tmem + 0, tmem + kTmO1 + (tt & 3) * 32, prm_u + ConvParams::kW2 + tap * 4096, first, elected);
                        first = false;
                    }
                }
                if (t2 >= 0 && t2 < kWindow) conv_mma_pred<32>(tmem + 32, o2_u, prm_u + ConvParams::kW3, true, elected);
                umma_commit_pred(bar_mma_x, elected);
            }
        }
    } else if (warp == 17) {
        // ------------------------------------------------------------ issuer of chain Y
        const uint32_t elected = elect_one();
        const uint32_t prm_u = smem_u32(prm), p2_u = smem_u32(p2);
        uint32_t it = 0, ny = 0, ny_slot = 0, ny_par = 0;          // y0 positions consumed so far: slot = ny % 3
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            for (int u = kFirstY; u <= kLastY; ++u, ++it) {
                mbar_wait(bar_ready_y, it & 1);
                tc_fence_after_sync();
                const int t3 = u - 3, t4 = u - 5, t5 = u - 6;
                if (t3 < kWindow) {
                    mbar_wait(&bar_y0_full[ny_slot], ny_par);
                    tc_fence_after_sync();
                    conv_mma_ts_pred<64>(tmem + kTmScp1, tmem + kTmY0 + ny_slot * 32, prm_u + ConvParams::kW45, true, elected);
                    umma_commit_pred(&bar_y0_empty[ny_slot], elected);
                    ++ny;
                    if (++ny_slot == 3) { ny_slot = 0; ny_par ^= 1; }
                }
                if (t4 >= 0 && t4 < kWindow) {
                    bool first = true;
#pragma unroll
                    for (int tap = 0; tap < 3; ++tap) {
                        const int tt = t4 + tap - 1;
                        if (tt < 0 || tt >= kWindow) continue;
                        conv_mma_ts_pred<32>(tmem + 64, tmem + kTmP1 + (tt % 3) * 32, prm_u + ConvParams::kW6 + tap * 4096, first, elected);
                        first = false;
                    }
                }
                if (t5 >= 0 && t5 < kWindow) conv_mma_pred<32>(tmem + 96, p2_u, prm_u + ConvParams::kW7, true, elected);
                umma_commit_pred(bar_mma_y, elected);
            }
        }
    } else {
        const int ew = warp & 7;                      // warp within its epilogue group
        const int q = ew & 3, ch = ew >> 2;
        const int row = q * 32 + lane;
        const int c0 = ch * 16;
        const uint32_t t_row = tmem + ((uint32_t)(q * 32) << 16);
        const uint32_t t_lane = t_row + c0;           // this thread's 16 accumulator columns
        const uint32_t t_opnd = t_row + ch * 8;       // this thread's K = 16 chunk of an operand slot
        auto relu_bias = [&](uint32_t* r, int slot, float* v) {
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
                const float4 b4 = *reinterpret_cast<const float4*>(fp + 32 * slot + c0 + i);
                const float2 s0 = fadd2(make_float2(__uint_as_float(r[i]), __uint_as_float(r[i + 1])), make_float2(b4.x, b4.y));
                const float2 s1 = fadd2(make_float2(__uint_as_float(r[i + 2]), __uint_as_float(r[i + 3])), make_float2(b4.z, b4.w));
                v[i] = fmaxf(s0.x, 0.f);
                v[i + 1] = fmaxf(s0.y, 0.f);
                v[i + 2] = fmaxf(s1.x, 0.f);
                v[i + 3] = fmaxf(s1.y, 0.f);
            }
        };
        if (warp < 8) {
            // -------------------------------------------------------- epilogue of chain X
            auto make_o1 = [&](int t) {               // o1[t] = relu(x a1 + b1) on CUDA cores
                const float2 x = splat2(xs[t * 128 + row]);
                float v[16];
#pragma unroll
                for (int i = 0; i < 16; i += 2) {
                    const float2 o = ffma2(x, *reinterpret_cast<const float2*>(fp + 64 + c0 + i), *reinterpret_cast<const float2*>(fp + 96 + c0 + i));
                    v[i] = fmaxf(o.x, 0.f);
                    v[i + 1] = fmaxf(o.y, 0.f);
                }
                store_a_tmem16_f<kFmt>(t_opnd + kTmO1 + (t & 3) * 32, v);
            };
            uint32_t it = 0, ny = 0, ny_slot = 0, ny_par = 1;      // empty-barrier parity of the previous use
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                // gather + normalise (infer.py:101-105, 32-38): the two threads of a window split its 35 samples
                asm volatile("bar.sync 1, 256;" ::: "memory");        // previous tile's readers of xs are done
                {
                    const WindowInput x = window_input(raw, stats, xwin, src, valid, read, (tile0 + tile) * kTileWindows + row);
                    const int tb = ch ? 18 : 0, te = ch ? kWindow : 18;
                    for (int t = tb; t < te; ++t) xs[t * 128 + row] = x(t);
                }
                asm volatile("bar.sync 1, 256;" ::: "memory");
                // the previous tile's last X batch (which read o1 slots) completed before its last epilogue
                make_o1(0);
                make_o1(1);
                tmem_st_wait();
                tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_ready_x);
                for (int u = 0; u <= kLastX; ++u, ++it) {
                    const int t1 = u - 1, t2 = u - 2;
                    const bool h1 = t1 >= 0 && t1 < kWindow, h2 = t2 >= 0 && t2 < kWindow;
                    mbar_wait(bar_mma_x, it & 1);
                    tc_fence_after_sync();
                    uint32_t r1[16], r2[16];
                    if (h1) tmem_ld16_nowait(t_lane + 0, r1);
                    if (h2) tmem_ld16_nowait(t_lane + 32, r2);
                    tmem_ld_wait();
                    float v[16];
                    if (h1) { relu_bias(r1, 4, v); store_a_row16_f<kFmt>(o2, row, c0, v); }              // b2
                    // o2 and o1[u+1] (made one iteration ago, in TMEM) are all the next X batch reads
                    if (u < kLastX) {
                        fence_proxy_async_smem();
                        tmem_st_wait();
                        tc_fence_before_sync();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(bar_ready_x);
                    }
                    if (h2) {
                        relu_bias(r2, 5, v);                                                     // b3
                        const float2 x = splat2(xs[t2 * 128 + row]);
#pragma unroll
                        for (int i = 0; i < 16; i += 2) {                                         // + shortcut
                            const float2 sc = ffma2(x, *reinterpret_cast<const float2*>(fp + c0 + i), *reinterpret_cast<const float2*>(fp + 32 + c0 + i));
                            const float2 o = fadd2(make_float2(v[i], v[i + 1]), sc);
                            v[i] = fmaxf(o.x, 0.f);
                            v[i + 1] = fmaxf(o.y, 0.f);
                        }
                        if (ny >= 3) mbar_wait(&bar_y0_empty[ny_slot], ny_par);
                        tc_fence_after_sync();
                        store_a_tmem16_f<kFmt>(t_opnd + kTmY0 + ny_slot * 32, v);
                        tmem_st_wait();
                        tc_fence_before_sync();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&bar_y0_full[ny_slot]);
                        ++ny;
                        if (++ny_slot == 3) { ny_slot = 0; ny_par ^= 1; }
                    }
                    if (u + 2 < kWindow) make_o1(u + 2);
                }
            }
        } else {
            // -------------------------------------------------------- epilogue of chain Y
            float* sc_mine = sc_ring + c0 * 128 + row;            // + slot * 4096 + i * 128
            uint32_t it = 0;
            if (lane == 0) mbar_arrive(bar_ready_y);          // nothing to prepare for the first batch
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                for (int u = kFirstY; u <= kLastY; ++u, ++it) {
                    const int t3 = u - 3, t4 = u - 5, t5 = u - 6;
                    const bool h3 = t3 < kWindow, h4 = t4 >= 0 && t4 < kWindow, h5 = t5 >= 0 && t5 < kWindow;
                    mbar_wait(bar_mma_y, it & 1);
                    tc_fence_after_sync();
                    uint32_t r3[16], r4[16], r5[16], rs[16];
                    if (h3) {
                        tmem_ld16_nowait(t_lane + kTmScp1 + 32, r3);
                        tmem_ld16_nowait(t_lane + kTmScp1, rs);
                    }
                    if (h4) tmem_ld16_nowait(t_lane + 64, r4);
                    if (h5) tmem_ld16_nowait(t_lane + 96, r5);
                    tmem_ld_wait();
                    float v[16];
                    if (h3) { relu_bias(r3, 7, v); store_a_tmem16_f<kFmt>(t_opnd + kTmP1 + (t3 % 3) * 32, v); }   // b5
                    if (h4) { relu_bias(r4, 8, v); store_a_row16_f<kFmt>(p2, row, c0, v); }              // b6
                    fence_proxy_async_smem();
                    tmem_st_wait();
                    tc_fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_ready_y);
                    if (h3) {                                                                    // park sc1 + b4
                        float* dst = sc_mine + (t3 & 3) * 4096;
#pragma unroll
                        for (int i = 0; i < 16; ++i) dst[i * 128] = __uint_as_float(rs[i]) + fp[192 + c0 + i];
                    }
                    if (h5) {
                        relu_bias(r5, 9, v);                                                     // b7
                        const float* sc = sc_mine + (t5 & 3) * 4096;
#pragma unroll
                        for (int i = 0; i < 16; i += 2) {                                         // + (sc1 + b4)
                            const float2 o = fadd2(make_float2(v[i], v[i + 1]), make_float2(sc[i * 128], sc[(i + 1) * 128]));
                            v[i] = fmaxf(o.x, 0.f);
                            v[i + 1] = fmaxf(o.y, 0.f);
                        }
                        if (head_w) {
                            float2 acc2 = make_float2(0.f, 0.f);
#pragma unroll
                            for (int i = 0; i < 16; i += 2)
                                acc2 = ffma2(make_float2(v[i], v[i + 1]), __ldg(reinterpret_cast<const float2*>(head_w + c0 + i)), acc2);
                            head_part[(((size_t)tile * kWindow + t5) * 2 + ch) * 128 + row] = acc2.x + acc2.y;
                        } else {
                            store_a_row16_f<kFmt>(reinterpret_cast<uint8_t*>(y_out) + ((size_t)tile * kWindow + t5) * kSliceBytes, row, c0, v);
                        }
                    }
                }
            }
        }
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 16) tmem_dealloc<512>(tmem);
}

// ====================================================================== TK2, one further residual block
// Blocks after the second of a deeper conv stack, one launch per block.  Input and output are the K = 32 operand form
// TK2 writes (one 16 KB slice per (tile, t)), so the first GRU layer and tc_head_conv_kernel read the last block's
// output unchanged.  Per position t it is chain Y of tc_conv4_kernel with its input streamed from HBM:
//   [sc | p1] = y[t] [W_sc | W_1]                        N = 64, TMEM ring of 4 at 64 k (sc waits three positions)
//   p2[t] = relu(conv3(relu(p1 + b5)) + b6)              taps over p1 operands t-1, t, t+1; SAME padding = skipped MMA
//   y_out[t] = relu(relu(p2 W_3 + b7) + sc + b4)
// The stages are skewed so that one batch per iteration u = 0..37 issues [sc|p1][u], p2[u-2] and p3[u-3]; one
// epilogue pass then writes the p1 operand of u, the p2 operand of u-2 and the output of u-3.
//   warps 0-7 : epilogue; thread = (window, 16 of the 32 channels)
//   warp 8    : MMA issuer (warp-converged issue, elected lane)
//   warp 9    : producer, input slices by cp.async.bulk into a ring of 4
constexpr int kBlockRing = 4;
constexpr uint32_t kBlockSmem = ConvParams::kBytes + (kBlockRing + 3 + 1) * kSliceBytes + 256;

__global__ void __launch_bounds__(320, 1)
tc_conv_block_kernel(const uint8_t* __restrict__ params, const __nv_bfloat16* __restrict__ y_in, int n_tiles,
                     __nv_bfloat16* __restrict__ y_out) {
    constexpr int kFmt = kFmtBf16x3;
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* prm = smem;
    uint8_t* yin = smem + ConvParams::kBytes;         // ring of kBlockRing input slices
    uint8_t* p1 = yin + kBlockRing * kSliceBytes;     // ring of 3 p1 operand slices (slot t % 3)
    uint8_t* p2 = p1 + 3 * kSliceBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(p2 + kSliceBytes);
    uint64_t* bar_ready = &bars[0];
    uint64_t* bar_mma = &bars[1];
    uint64_t* bar_prm = &bars[2];
    uint64_t* bar_full = &bars[3];                    // [kBlockRing] input slice landed
    uint64_t* bar_empty = &bars[3 + kBlockRing];      // [kBlockRing] its MMA completed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 + 2 * kBlockRing);
    const float* fp = reinterpret_cast<const float*>(prm);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        mbar_init(bar_ready, 8);
        mbar_init(bar_mma, 1);
        mbar_init(bar_prm, 1);
        for (int i = 0; i < kBlockRing; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], 1); }
        fence_mbar_init();
        mbar_expect_tx(bar_prm, ConvParams::kBytes);
        bulk_g2s(prm, params, ConvParams::kBytes, bar_prm);
    }
    if (warp == 8) tmem_alloc<512>(tmem_slot);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    constexpr int kLastU = kWindow + 2;               // p3[34] at u = 37
    constexpr uint32_t kTmP2 = 256, kTmP3 = 288;      // [sc|p1] ring at 0, 64, 128, 192
    mbar_wait(bar_prm, 0);

    if (warp == 8) {
        // ------------------------------------------------------------ issuer (all lanes converged)
        const uint32_t elected = elect_one();
        const uint32_t prm_u = smem_u32(prm), yin_u = smem_u32(yin), p1_u = smem_u32(p1), p2_u = smem_u32(p2);
        uint32_t it = 0, n = 0;                       // n = input slices consumed so far
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            for (int u = 0; u <= kLastU; ++u, ++it) {
                mbar_wait(bar_ready, it & 1);
                tc_fence_after_sync();
                const int t2 = u - 2, t3 = u - 3;
                if (u < kWindow) {
                    const uint32_t slot = n % kBlockRing;
                    mbar_wait(&bar_full[slot], (n / kBlockRing) & 1);
                    conv_mma_pred<64>(tmem + (u & 3) * 64, yin_u + slot * kSliceBytes, prm_u + ConvParams::kW45, true, elected);
                    umma_commit_pred(&bar_empty[slot], elected);
                    ++n;
                }
                if (t2 >= 0 && t2 < kWindow) {
                    bool first = true;
#pragma unroll
                    for (int tap = 0; tap < 3; ++tap) {
                        const int tt = t2 + tap - 1;
                        if (tt < 0 || tt >= kWindow) continue;
                        conv_mma_pred<32>(tmem + kTmP2, p1_u + (tt % 3) * kSliceBytes, prm_u + ConvParams::kW6 + tap * 4096, first, elected);
                        first = false;
                    }
                }
                if (t3 >= 0 && t3 < kWindow) conv_mma_pred<32>(tmem + kTmP3, p2_u, prm_u + ConvParams::kW7, true, elected);
                umma_commit_pred(bar_mma, elected);
            }
        }
    } else if (warp == 9) {
        // ------------------------------------------------------------ producer
        if (lane == 0) {
            const uint8_t* src = reinterpret_cast<const uint8_t*>(y_in);
            uint32_t n = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
                for (int t = 0; t < kWindow; ++t, ++n) {
                    const uint32_t slot = n % kBlockRing;
                    if (n >= kBlockRing) mbar_wait(&bar_empty[slot], (n / kBlockRing - 1) & 1);
                    mbar_expect_tx(&bar_full[slot], kSliceBytes);
                    bulk_g2s(yin + slot * kSliceBytes, src + ((size_t)tile * kWindow + t) * kSliceBytes, kSliceBytes, &bar_full[slot]);
                }
        }
    } else {
        // ------------------------------------------------------------ epilogue
        const int q = warp & 3, ch = warp >> 2;
        const int row = q * 32 + lane;
        const int c0 = ch * 16;
        const uint32_t t_lane = tmem + ((uint32_t)(q * 32) << 16) + c0;
        auto relu_bias = [&](uint32_t* r, int slot, float* v) {
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
                const float4 b4 = *reinterpret_cast<const float4*>(fp + 32 * slot + c0 + i);
                const float2 s0 = fadd2(make_float2(__uint_as_float(r[i]), __uint_as_float(r[i + 1])), make_float2(b4.x, b4.y));
                const float2 s1 = fadd2(make_float2(__uint_as_float(r[i + 2]), __uint_as_float(r[i + 3])), make_float2(b4.z, b4.w));
                v[i] = fmaxf(s0.x, 0.f);
                v[i + 1] = fmaxf(s0.y, 0.f);
                v[i + 2] = fmaxf(s1.x, 0.f);
                v[i + 3] = fmaxf(s1.y, 0.f);
            }
        };
        uint32_t it = 0;
        if (lane == 0) mbar_arrive(bar_ready);        // nothing to prepare for the first batch
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            for (int u = 0; u <= kLastU; ++u, ++it) {
                const int t2 = u - 2, t3 = u - 3;
                const bool h1 = u < kWindow, h2 = t2 >= 0 && t2 < kWindow, h3 = t3 >= 0 && t3 < kWindow;
                mbar_wait(bar_mma, it & 1);
                tc_fence_after_sync();
                uint32_t r1[16], r2[16], r3[16], rs[16];
                if (h1) tmem_ld16_nowait(t_lane + (u & 3) * 64 + 32, r1);
                if (h2) tmem_ld16_nowait(t_lane + kTmP2, r2);
                if (h3) {
                    tmem_ld16_nowait(t_lane + kTmP3, r3);
                    tmem_ld16_nowait(t_lane + (t3 & 3) * 64, rs);
                }
                tmem_ld_wait();
                float v[16];
                if (h1) { relu_bias(r1, 7, v); store_a_row16_f<kFmt>(p1 + (u % 3) * kSliceBytes, row, c0, v); }   // b5
                if (h2) { relu_bias(r2, 8, v); store_a_row16_f<kFmt>(p2, row, c0, v); }                        // b6
                // the next batch's operands are written and every accumulator it overwrites has been read
                fence_proxy_async_smem();
                tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_ready);
                if (h3) {
                    relu_bias(r3, 9, v);                                                         // b7
#pragma unroll
                    for (int i = 0; i < 16; i += 2) {                                             // + (sc + b4)
                        const float2 sc = fadd2(make_float2(__uint_as_float(rs[i]), __uint_as_float(rs[i + 1])),
                                                *reinterpret_cast<const float2*>(fp + 192 + c0 + i));
                        const float2 o = fadd2(make_float2(v[i], v[i + 1]), sc);
                        v[i] = fmaxf(o.x, 0.f);
                        v[i + 1] = fmaxf(o.y, 0.f);
                    }
                    store_a_row16_f<kFmt>(reinterpret_cast<uint8_t*>(y_out) + ((size_t)tile * kWindow + t3) * kSliceBytes, row, c0, v);
                }
            }
        }
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 8) tmem_dealloc<512>(tmem);
}

// ====================================================================== TK4G: fused GRU layer, two tiles per CTA
// One GRU layer, input projection and recurrence in one kernel (TF GRUCell, reset gate applied before the
// candidate matmul; rnn_class.py:142-175).  Per step and chain: the x part x W_x (N = 192: r | u | c) and the
// state part h W_gh accumulate the gates, (r*h) W_ch adds to the candidate columns; the epilogue applies the
// activations and h = u h + (1 - u) c.  So that the tensor pipe never idles behind one chain's serial
// MMA -> epilogue -> MMA dependency, a CTA runs TWO independent chains (two tiles of the same direction,
// sharing the resident weights).  To make room for the second chain the state operand h / r*h lives in
// tensor memory: the epilogue writes it (packed, in the operand format FMT) with tcgen05.st and the
// state-part MMAs read A from TMEM (".ts" form).
// TMEM per chain (256 columns): gates accumulator 0..127, candidate 128..191, A plane 0 192..223,
// A plane 1 224..255.  Shared memory: weights (147 KB) + ONE x ring (8 stages of 8 KB for a 128-wide input = one
// entry per turn, 10 stages for a 32-wide one) that both chains
// consume in the fixed order (step 0, chain 0), (step 0, chain 1), (step 1, chain 0), ...: with a private
// 5-stage ring per chain only 5 of a step's 8 chunks could be requested before the step's x part began,
// so the last three arrived a full HBM latency later (x part 4 400-4 900 cycles for 1 536 of MMA time);
// in the shared ring a step's chunks are all requested while the OTHER chain's x part runs.
//   warps 0-15       : epilogue of BOTH chains; thread = (window, 16 of the hidden units)
//   warp 16 / 17     : MMA issuer of chain 0 / 1 (x part, then state part of gates, then of candidate)
//   warp 18          : lane 0 = producer (weights once, then the x ring)
//   warp 19 / 20     : f16e5 input only - rebuild each landed chunk's hi-byte slab from its main plane (the
//                      compact HBM form carries 3 of the 4 operand bytes; tc_ptx.cuh) and hand the stage on;
//                      even / odd ring stages
//   warps 21-23      : idle (they exist so that the warpgroup 20-23 can hand its registers back)
// Registers: launched with 80 per thread; the service warpgroups (16-23) shrink to 48 and the epilogue
// warpgroups (0-15) grow to 96 with setmaxnreg, the role code sits inside the branch that executed it.
template <int KX> struct GruF2Cfg {
    static constexpr bool kNoX = KX == 1;                                 // scalar layer input: x part added in the epilogue
    static constexpr int kChunks = KX / 16;
    // ONE ring shared by both chains (see the producer).  128-wide input: 8 stages = one entry per turn, which makes
    // every stage index in the issue loop a compile-time constant (see the issuer)
    static constexpr int kStages = KX == 128 ? 8 : 10;
    static constexpr uint32_t kWx = 0;                                   // {hi, lo} x [KX/8][192][8]  (r | u | c)
    static constexpr uint32_t kWgh = kWx + (kNoX ? 0u : 2u * KX * kNX * 2);
    static constexpr uint32_t kWch = kWgh + 2u * kH * 128 * 2;
    static constexpr uint32_t kWBytes = kWch + 2u * kH * 64 * 2;
    static constexpr uint32_t kRing = kWBytes;                            // [stage] x 8 KB
    static constexpr uint32_t kBias = kRing + (uint32_t)kStages * 8192;
    static constexpr uint32_t kBars = kBias + 2 * 192 * 4;               // bias, then the scalar-input weight row
    static constexpr uint32_t kSmem = kBars + 512;
    // barriers: a chain's group of 8, then the ring's full / empty pairs, then the weight barrier
    static constexpr int kBarG = 0, kBarC = 1, kBarRh = 2, kBarH = 3, kBarCfree = 4, kBarXdone = 5;
    static constexpr int kBarFull = 16, kBarEmpty = 16 + kStages, kBarTma = 16 + 2 * kStages, kBarW = 16 + 3 * kStages;
};
// Bytes of one (tile, t) block of a 128-wide layer output in HBM: split bf16 = two 16-bit planes; f16e5 =
// fp16 main plane [16][128][8 x 2 B] + remainder bytes [8 chunks][128][16 B] (the hi bytes are rebuilt by the reader).
__host__ __device__ constexpr uint32_t gru_out_block_bytes(int fmt) { return fmt == kFmtF16E5 ? 49152u : 65536u; }
// 24 warps = six per sub-partition.  Launched with 80 registers per thread; the two service warpgroups (16-23) give
// theirs back (setmaxnreg) and the four epilogue warpgroups grow to 96: 4 x 96 + 2 x 48 = 480 = 6 x 80 per lane.
constexpr int kGruF2Threads = 768;
constexpr int kGruF2Converters = 2;               // warps 19.. rebuilding hi-byte slabs; must divide the ring's stages
constexpr int kGruF2EpiRegs = 96, kGruF2ServiceRegs = 48;

template <int KX, int FMT, int FMT_OUT>
__global__ void __launch_bounds__(kGruF2Threads, 1)
tc_gru_fused2_kernel(const uint8_t* __restrict__ wpk, const float* __restrict__ bias,
                     const __nv_bfloat16* __restrict__ x_blocks, __nv_bfloat16* __restrict__ y_out,
                     const float* __restrict__ head_w, float* __restrict__ head_part, int n_tiles,
                     long long* __restrict__ trace, const float* __restrict__ x_scalar, const float* __restrict__ wx_scalar) {
    using Cfg = GruF2Cfg<KX>;
    constexpr bool kNoX = Cfg::kNoX;
    // debug timeline (build with -DCF_TRACE_PROBES, run with CF_TC_TRACE=<file>): block 0 records (tag, SM clock)
    // pairs for steps 36..39 of each role.  Compiled out of the shipped library: fourteen probes per step are
    // ~8 % of the epilogue's instruction stream even when they record nothing.
#ifdef CF_TRACE_PROBES
    int tr_n = 0;
#define CF_TR(region, step, tag)                                                                   \
    do {                                                                                           \
        if (trace && blockIdx.x == 0 && (step) >= 36 && (step) < 40 && tr_n < 200) {               \
            trace[((region) * 200 + tr_n) * 2] = (tag) + 1000 * (long long)(step);                      \
            trace[((region) * 200 + tr_n) * 2 + 1] = clock64();                                    \
            ++tr_n;                                                                                \
        }                                                                                          \
    } while (0)
#else
#define CF_TR(region, step, tag) do { } while (0)
#endif
#ifdef CF_TRACE_CHUNKS        // per-chunk probes of the x ring (issuer, converter, producer): they slow the ring itself
#define CF_TRC(region, step, tag) CF_TR(region, step, tag)
#else
#define CF_TRC(region, step, tag) do { } while (0)
#endif
    extern __shared__ __align__(128) uint8_t smem[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kBars);     // [2][8] per chain, ring full / empty, w_bar
    uint64_t* w_bar = &bars[Cfg::kBarW];
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(&bars[Cfg::kBarW + 1]);
    float* bias_s = reinterpret_cast<float*>(smem + Cfg::kBias);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int dir = blockIdx.x & 1;
    const int slot = blockIdx.x >> 1, n_slots = gridDim.x >> 1;
    const int stride = 2 * n_slots;                        // tiles between consecutive tiles of one chain
    auto tiles_of = [&](int chain) -> int {
        const int first = slot * 2 + chain;
        return first < n_tiles ? (n_tiles - first + stride - 1) / stride : 0;
    };
    auto blk_of = [&](int chain, int gs) -> size_t {
        const int ti = gs / kWindow, s = gs - ti * kWindow;
        return (size_t)(slot * 2 + chain + ti * stride) * kWindow + (dir ? kWindow - 1 - s : s);
    };

    if (threadIdx.x == 0) {
        for (int c = 0; c < 2; ++c) {
            uint64_t* b = &bars[8 * c];
            mbar_init(&b[Cfg::kBarG], 1);
            mbar_init(&b[Cfg::kBarC], 1);
            mbar_init(&b[Cfg::kBarRh], 16);
            mbar_init(&b[Cfg::kBarH], 16);
            mbar_init(&b[Cfg::kBarCfree], 16);
            mbar_init(&b[Cfg::kBarXdone], 1);
        }
        for (int i = 0; i < Cfg::kStages; ++i) {
            mbar_init(&bars[Cfg::kBarFull + i], 1);
            mbar_init(&bars[Cfg::kBarEmpty + i], 1);
            mbar_init(&bars[Cfg::kBarTma + i], 1);
        }
        mbar_init(w_bar, 1);
        fence_mbar_init();
    }
#ifndef CF_PRECISE_ACT
    // bias pre-multiplied by the activation's argument scale, so that bias add + scaling is one FFMA
    if (threadIdx.x < 192) bias_s[threadIdx.x] = bias[dir * kNX + threadIdx.x] * (threadIdx.x < 2 * kH ? kSigArgScale : kTanhArgScale);
    if (kNoX && threadIdx.x < 192) bias_s[192 + threadIdx.x] = wx_scalar[dir * kNX + threadIdx.x] * (threadIdx.x < 2 * kH ? kSigArgScale : kTanhArgScale);
#else
    if (threadIdx.x < 192) bias_s[threadIdx.x] = bias[dir * kNX + threadIdx.x];
    if (kNoX && threadIdx.x < 192) bias_s[192 + threadIdx.x] = wx_scalar[dir * kNX + threadIdx.x];
#endif
    if (warp == 16) tmem_alloc<512>(tmem_slot);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem = *tmem_slot;

    if (warp >= 16) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kGruF2ServiceRegs));
    if (warp == 18) {
        // ------------------------------------------------------------ producer: weights once, then the shared x ring
        if (lane == 0) {
            mbar_expect_tx(w_bar, Cfg::kWBytes);
            const uint8_t* wsrc = wpk + (size_t)dir * Cfg::kWBytes;
            for (uint32_t off = 0; off < Cfg::kWBytes; off += 32768) {
                const uint32_t n = Cfg::kWBytes - off < 32768 ? Cfg::kWBytes - off : 32768;
                bulk_g2s(smem + off, wsrc + off, n, w_bar);
            }
            // input block in HBM: split bf16 = two planes of 128 * KX * 2 bytes; compact f16e5 = main plane + KX / 16
            // remainder slabs of 2 KB (the chunk's hi slab, the last 2 KB of the stage, is filled by warps 19 / 20)
            constexpr bool kCompact = FMT == kFmtF16E5;
            constexpr size_t plane = (size_t)128 * KX * 2;
            constexpr size_t blk_bytes = kCompact ? plane + (size_t)(KX / 16) * 2048 : 2 * plane;
            const uint8_t* xbase = reinterpret_cast<const uint8_t*>(x_blocks);
            const int total0 = tiles_of(0) * kWindow, total1 = tiles_of(1) * kWindow;     // total1 <= total0
            uint32_t st = 0, par = 1;                     // ring position; parity of the empty barrier's previous phase
            for (int gs = 0; gs < (kNoX ? 0 : total0); ++gs) {
                for (int c = 0; c < 2; ++c) {
                    if (c == 1 && gs >= total1) break;
                    const uint8_t* xb = xbase + blk_of(c, gs) * blk_bytes;
                    if (kCompact) {
                        // The ring holds about one entry, so an entry's chunks are requested only while the entry
                        // before it is being consumed, and when two x parts run back to back the second one waited
                        // an HBM latency (~1 500 cycles) per chunk.  Ask L2 for the NEXT entry one entry ahead.
                        const int nc = (c == 0 && gs < total1) ? 1 : 0, ngs = nc ? gs : gs + 1;
                        if (ngs < total0 && (nc == 0 || ngs < total1)) {
                            const uint8_t* nb = xbase + blk_of(nc, ngs) * blk_bytes;
                            bulk_prefetch_l2(nb, (uint32_t)plane);
                            bulk_prefetch_l2(nb + plane, (uint32_t)(KX / 16) * 2048);
                        }
                    }
                    for (int kk = 0; kk < Cfg::kChunks; ++kk) {
                        mbar_wait(&bars[Cfg::kBarEmpty + st], par);
                        CF_TRC(5, gs, 80 + kk);
                        uint8_t* dst = smem + Cfg::kRing + st * 8192;
                        uint64_t* landed = &bars[(kCompact ? Cfg::kBarTma : Cfg::kBarFull) + st];
                        if (kCompact) {
                            mbar_expect_tx(landed, 6144);
                            bulk_g2s(dst, xb + kk * 4096, 4096, landed);
                            bulk_g2s(dst + 4096, xb + plane + kk * 2048, 2048, landed);
                        } else {
                            mbar_expect_tx(landed, 8192);
                            bulk_g2s(dst, xb + kk * 4096, 4096, landed);
                            bulk_g2s(dst + 4096, xb + plane + kk * 4096, 4096, landed);
                        }
                        if (++st == Cfg::kStages) { st = 0; par ^= 1; }
                    }
                }
            }
        }
    } else if (warp >= 19) {
        // ------------------------------------------------------------ hi-byte slab of every landed chunk (f16e5 input)
        // kGruF2Converters warps, warp 19 + i taking the ring stages == i (mod kGruF2Converters): a chunk's
        // conversion is a serial ~30-instruction chain on a sub-partition it shares with four epilogue warps, and
        // with one warp that chain paced the whole x part.
        if (FMT == kFmtF16E5 && warp < 19 + kGruF2Converters) {
            static_assert(Cfg::kStages % kGruF2Converters == 0, "converter warps split the ring by stage");
            const int total0 = tiles_of(0) * kWindow, total1 = tiles_of(1) * kWindow;
            const int n_chunks = (total0 + total1) * Cfg::kChunks;
            uint32_t st = warp - 19, par = 0;
            for (int cn = warp - 19; cn < n_chunks; cn += kGruF2Converters) {
                mbar_wait(&bars[Cfg::kBarTma + st], par);
                if (lane == 0 && warp == 19) CF_TRC(4, cn / (2 * Cfg::kChunks), 70);
                uint8_t* stage = smem + Cfg::kRing + st * 8192;
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const int row = r * 32 + lane;
                    const uint4 a = *reinterpret_cast<const uint4*>(stage + row * 16);            // K 0..7 of the chunk
                    const uint4 b = *reinterpret_cast<const uint4*>(stage + 2048 + row * 16);     // K 8..15
                    *reinterpret_cast<uint4*>(stage + 6144 + row * 16) =
                        make_uint4(f16e5_hi4(a.x, a.y), f16e5_hi4(a.z, a.w), f16e5_hi4(b.x, b.y), f16e5_hi4(b.z, b.w));
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars[Cfg::kBarFull + st]);
                if (lane == 0 && warp == 19) CF_TRC(4, cn / (2 * Cfg::kChunks), 71);
                if ((st += kGruF2Converters) >= Cfg::kStages) { st -= Cfg::kStages; par ^= 1; }
            }
        }
    } else if (warp >= 16 && warp < 18) {
        // ------------------------------------------------------------ MMA issuer of chain (warp - 16)
        // Warp-converged: all lanes run the control flow and the waits, one elected lane issues
        // (descriptor arithmetic stays on the uniform datapath: ~10 instead of ~80 cycles per MMA).
        {
            constexpr bool kE5 = FMT == kFmtF16E5;        // plane 1 = e5m2 corrections (one kind::f8f6f4 MMA per chunk)
            constexpr uint32_t idesc_g = kE5 ? make_idesc_f16(128, 2 * kH) : make_idesc_bf16(128, 2 * kH);
            constexpr uint32_t idesc_c = kE5 ? make_idesc_f16(128, kH) : make_idesc_bf16(128, kH);
            constexpr uint32_t idesc_x = kE5 ? make_idesc_f16(128, kNX) : make_idesc_bf16(128, kNX);
            constexpr uint32_t idesc_g8 = make_idesc_e5m2(128, 2 * kH), idesc_c8 = make_idesc_e5m2(128, kH);
            constexpr uint32_t idesc_x8 = make_idesc_e5m2(128, kNX);
            const uint32_t elected = elect_one();
            const int c = warp - 16;
            const uint32_t s0 = smem_u32(smem);
            uint64_t* b = &bars[8 * c];
            const uint32_t dg = tmem + c * 256, dc = dg + 2 * kH, ta = dg + 3 * kH;
            const int total = tiles_of(c) * kWindow;
            const int total1 = tiles_of(1) * kWindow;
            mbar_wait(w_bar, 0);
            for (int gs = 0; gs < total; ++gs) {
                const uint32_t par = gs & 1;
                // this step's chunks in the shared ring: entries are ordered (step, chain), chain 1 stops at total1
                uint32_t cn = (uint32_t)(c == 0 ? gs + (gs < total1 ? gs : total1) : 2 * gs + 1) * Cfg::kChunks;
                // An mbarrier wait only tells phases apart by parity, so a consumer must never look at a stage two
                // uses ahead of it: the issuers take their ring entries strictly in turn - this one starts after the
                // other chain's issuer has passed the full-waits of the entry before.
                if (kNoX) {
                } else if (c == 1) mbar_wait(&bars[Cfg::kBarXdone], gs & 1);
                else if (gs > 0 && gs - 1 < total1) mbar_wait(&bars[8 + Cfg::kBarXdone], (gs - 1) & 1);
                // x part: needs the previous step's accumulators drained
                if (gs > 0) mbar_wait(&b[Cfg::kBarCfree], (gs - 1) & 1);
                if (lane == 0) CF_TR(c, gs, 10);
                // The ring stage of a chunk is a compile-time constant in the issue loop, so that the operand
                // descriptors are `base + immediate` on the uniform datapath.  With a runtime stage they took a /10,
                // five dependent ALU ops and predicated R2URs per MMA (~165 cycles per MMA, the x part was issue-bound:
                // 2 650 cycles for 1 536 of tensor time).  128-wide input: an entry is one turn of the 8-stage ring
                // (chunk kk in stage kk); 32-wide input: an entry's two chunks start at an even stage of the 10.
                auto issue_x = [&](auto st0c) {
                    constexpr int kSt0 = decltype(st0c)::value;
                    static_assert(kSt0 + Cfg::kChunks <= Cfg::kStages || kNoX, "an entry does not wrap around the ring");
                    uint32_t ring_lo = (uint32_t)make_smem_desc(s0 + Cfg::kRing, 2048, 128);
                    uint32_t wx_lo = (uint32_t)make_smem_desc(s0 + Cfg::kWx, kNX * 16, 128);
                    asm volatile("" : "+r"(ring_lo), "+r"(wx_lo));       // per step, not hoisted: dozens of live descriptors spill
                    constexpr uint64_t ahi = make_smem_desc(0, 2048, 128) & 0xffffffff00000000ull;
                    constexpr uint64_t bhi = make_smem_desc(0, kNX * 16, 128) & 0xffffffff00000000ull;
                    const uint32_t xpar = (cn / Cfg::kStages) & 1;
#pragma unroll
                    for (int kk = 0; kk < Cfg::kChunks; ++kk) {
                        const int st = kSt0 + kk;
                        mbar_wait(&bars[Cfg::kBarFull + st], xpar);
                        if (lane == 0) CF_TRC(c, gs, 60 + kk);
                        tc_fence_after_sync();
                        const uint32_t a_lo = ring_lo + st * (8192 >> 4), w_lo = wx_lo + kk * (2 * kNX * 16 >> 4);
                        if (kE5) {
                            umma_bf16_pred(dg, ahi | a_lo, bhi | w_lo, idesc_x, kk != 0, elected);
                            umma_f8_pred(dg, ahi | (a_lo + (4096 >> 4)), bhi | (w_lo + (KX * kNX * 2 >> 4)), idesc_x8, 1, elected);
                        } else {
#pragma unroll
                            for (int pass = 0; pass < 3; ++pass)
                                umma_bf16_pred(dg, ahi | (a_lo + (pass == 1 ? 4096 >> 4 : 0)),
                                               bhi | (w_lo + (pass == 2 ? KX * kNX * 2 >> 4 : 0)), idesc_x, (kk | pass) != 0, elected);
                        }
                        umma_commit_pred(&bars[Cfg::kBarEmpty + st], elected);
                        if (lane == 0) CF_TRC(c, gs, 20 + kk);
                        if (kk == Cfg::kChunks - 1 && lane == 0) CF_TR(c, gs, 27);
                    }
                };
                if constexpr (kNoX) {
                } else if constexpr (Cfg::kChunks == Cfg::kStages) {
                    issue_x(std::integral_constant<int, 0>{});
                } else {
                    static_assert(Cfg::kStages == 10 && Cfg::kChunks == 2, "entries start at the even stages 0..8");
                    switch (cn % Cfg::kStages) {
                        case 0: issue_x(std::integral_constant<int, 0>{}); break;
                        case 2: issue_x(std::integral_constant<int, 2>{}); break;
                        case 4: issue_x(std::integral_constant<int, 4>{}); break;
                        case 6: issue_x(std::integral_constant<int, 6>{}); break;
                        default: issue_x(std::integral_constant<int, 8>{}); break;
                    }
                }
                if (!kNoX && lane == 0) mbar_arrive(&b[Cfg::kBarXdone]);
                // state part of the gates (weight descriptors = per-step base + immediate, as in the x part: kept
                // loop-invariant, the 36 descriptors of the split-bf16 form do not fit the service warps' registers)
                uint32_t wgh_lo = (uint32_t)make_smem_desc(s0 + Cfg::kWgh, 128 * 16, 128);
                uint32_t wch_lo = (uint32_t)make_smem_desc(s0 + Cfg::kWch, 64 * 16, 128);
                asm volatile("" : "+r"(wgh_lo), "+r"(wch_lo));
                constexpr uint64_t ghi = make_smem_desc(0, 128 * 16, 128) & 0xffffffff00000000ull;
                constexpr uint64_t chi = make_smem_desc(0, 64 * 16, 128) & 0xffffffff00000000ull;
                mbar_wait(&b[Cfg::kBarH], par);
                if (lane == 0) CF_TR(c, gs, 30);
                tc_fence_after_sync();
                if (kE5) {
#pragma unroll
                    for (int kk = 0; kk < kH / 16; ++kk) {
                        const uint32_t w_lo = wgh_lo + kk * (2 * 128 * 16 >> 4);
                        umma_bf16_ts_pred(dg, ta + kk * 8, ghi | w_lo, idesc_g, !kNoX || kk != 0, elected);
                        umma_f8_ts_pred(dg, ta + 32 + kk * 8, ghi | (w_lo + (kH * 128 * 2 >> 4)), idesc_g8, 1, elected);
                    }
                } else {
#pragma unroll
                    for (int pass = 0; pass < 3; ++pass) {
                        const uint32_t ap = ta + (pass == 1 ? 32u : 0u);
#pragma unroll
                        for (int kk = 0; kk < kH / 16; ++kk)
                            umma_bf16_ts_pred(dg, ap + kk * 8, ghi | (wgh_lo + (pass == 2 ? kH * 128 * 2 >> 4 : 0) + kk * (2 * 128 * 16 >> 4)),
                                              idesc_g, !kNoX || (pass | kk) != 0, elected);
                    }
                }
                umma_commit_pred(&b[Cfg::kBarG], elected);
                if (lane == 0) CF_TR(c, gs, 31);
                // state part of the candidate
                mbar_wait(&b[Cfg::kBarRh], par);
                if (lane == 0) CF_TR(c, gs, 40);
                tc_fence_after_sync();
                if (kE5) {
#pragma unroll
                    for (int kk = 0; kk < kH / 16; ++kk) {
                        const uint32_t w_lo = wch_lo + kk * (2 * 64 * 16 >> 4);
                        umma_bf16_ts_pred(dc, ta + kk * 8, chi | w_lo, idesc_c, !kNoX || kk != 0, elected);
                        umma_f8_ts_pred(dc, ta + 32 + kk * 8, chi | (w_lo + (kH * 64 * 2 >> 4)), idesc_c8, 1, elected);
                    }
                } else {
#pragma unroll
                    for (int pass = 0; pass < 3; ++pass) {
                        const uint32_t ap = ta + (pass == 1 ? 32u : 0u);
#pragma unroll
                        for (int kk = 0; kk < kH / 16; ++kk)
                            umma_bf16_ts_pred(dc, ap + kk * 8, chi | (wch_lo + (pass == 2 ? kH * 64 * 2 >> 4 : 0) + kk * (2 * 64 * 16 >> 4)),
                                              idesc_c, !kNoX || (pass | kk) != 0, elected);
                    }
                }
                umma_commit_pred(&b[Cfg::kBarC], elected);
                if (lane == 0) CF_TR(c, gs, 41);
            }
        }
    }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kGruF2EpiRegs));
        // ------------------------------------------------------------ epilogue: 16 warps serve BOTH chains
        // Thread = (window row, 16 of the 64 hidden units) of both chains.  A chain's step has two epilogue phases,
        // R (reset gate -> r*h operand) after its gate MMAs and C (update gate, candidate, new state) after its
        // candidate MMAs, and between them the warps would only wait for the tensor pipe.  With eight warps per
        // chain that wait was idle time (per-step latency ~6 500 cycles whatever the x part cost); here all sixteen
        // warps work through the phases of both chains in the fixed order
        //     R(A, g)  C(B, g-1)  C(A, g)  R(B, g)
        // so that every MMA group runs while the other chain's phase is being computed, each phase has half the
        // values per thread, and the register budget holds the state of 2 x 16 units without spilling.
        const int q = warp & 3, us = warp >> 2;
        const int row = q * 32 + lane;
        const int j0 = us * 16;
        const uint32_t t_row = tmem + ((uint32_t)(q * 32) << 16);
        const int tot[2] = {tiles_of(0) * kWindow, tiles_of(1) * kWindow};
        float2 h2[2][8];                       // state of this thread's 16 units, per chain, as packed pairs
        // position of each chain inside its tile and the block (tile * 35 + time step) it is at, advanced step by
        // step: no division, no 64-bit index arithmetic; the thread-constant parts of every address are folded
        // into base pointers once
        int spos[2] = {0, 0};
        const uint32_t blk_step = dir ? 0xffffffffu : 1u;                                  // +-1 per step
        const uint32_t blk_jump = (uint32_t)stride * kWindow - blk_step * (kWindow - 1);    // last block -> next tile's first
        uint32_t cblk[2] = {(uint32_t)(slot * 2) * kWindow + (dir ? kWindow - 1 : 0),
                            (uint32_t)(slot * 2 + 1) * kWindow + (dir ? kWindow - 1 : 0)};
        uint8_t* const y_main = reinterpret_cast<uint8_t*>(y_out) + ((size_t)(dir * kH + j0) / 8 * 128 + row) * 16;
        const int32_t y_lo_delta = FMT_OUT == kFmtF16E5
            ? 128 * 2 * kH * 2 + ((dir * kH + j0) / 16 * 128 + row) * 16 - ((dir * kH + j0) / 8 * 128 + row) * 16
            : 128 * 2 * kH * 2;
        float* const head_base = head_part + (dir * 4 + us) * 128 + row;
        const float* const xs_base = x_scalar + row;
#pragma unroll
        for (int c = 0; c < 2; ++c)
#pragma unroll
            for (int j = 0; j < 8; ++j) h2[c][j] = make_float2(0.f, 0.f);

        // activation argument bias (+ x_t * w for the scalar-input layer), 4 consecutive columns
        auto bias4 = [&](int idx, float xv) -> float4 {
            float4 b4 = *reinterpret_cast<const float4*>(bias_s + idx);
            if (kNoX) {
                const float4 w4 = *reinterpret_cast<const float4*>(bias_s + 192 + idx);
                b4.x = fmaf(xv, w4.x, b4.x); b4.y = fmaf(xv, w4.y, b4.y); b4.z = fmaf(xv, w4.z, b4.z); b4.w = fmaf(xv, w4.w, b4.w);
            }
            return b4;
        };
        auto sig4 = [&](const uint32_t* a, float4 b4, float2& o0, float2& o1) {
#ifndef CF_PRECISE_ACT
            o0 = sigmoid_zb2(make_float2(__uint_as_float(a[0]), __uint_as_float(a[1])), make_float2(b4.x, b4.y));
            o1 = sigmoid_zb2(make_float2(__uint_as_float(a[2]), __uint_as_float(a[3])), make_float2(b4.z, b4.w));
#else
            float z[4] = {__uint_as_float(a[0]) + b4.x, __uint_as_float(a[1]) + b4.y, __uint_as_float(a[2]) + b4.z, __uint_as_float(a[3]) + b4.w};
            float y[4];
            sigmoid4_z(z, y);
            o0 = make_float2(y[0], y[1]);
            o1 = make_float2(y[2], y[3]);
#endif
        };
        auto tanh4v = [&](const uint32_t* a, float4 b4, float2& o0, float2& o1) {
#ifndef CF_PRECISE_ACT
            o0 = tanh_zb2(make_float2(__uint_as_float(a[0]), __uint_as_float(a[1])), make_float2(b4.x, b4.y));
            o1 = tanh_zb2(make_float2(__uint_as_float(a[2]), __uint_as_float(a[3])), make_float2(b4.z, b4.w));
#else
            float z[4] = {__uint_as_float(a[0]) + b4.x, __uint_as_float(a[1]) + b4.y, __uint_as_float(a[2]) + b4.z, __uint_as_float(a[3]) + b4.w};
            float y[4];
            tanh4_z(z, y);
            o0 = make_float2(y[0], y[1]);
            o1 = make_float2(y[2], y[3]);
#endif
        };
        // zero state operand of a chain's next tile
        auto begin_tile = [&](int c) {
            const uint32_t t_ahi = t_row + c * 256 + 3 * kH + j0 / 2, t_alo = t_ahi + 32;
            const uint32_t z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
            for (int j = 0; j < 8; ++j) h2[c][j] = make_float2(0.f, 0.f);
            tmem_st8_u32(t_ahi, z);
            tmem_st8_u32(t_alo, z);
            tmem_st_wait();
            tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars[8 * c + Cfg::kBarH]);
        };
        // ---- phase R of chain c, step gs: reset gate -> r*h operand
        auto phase_r = [&](int c, int gs) {
            uint64_t* b = &bars[8 * c];
            const uint32_t t_acc = t_row + c * 256 + j0;
            const uint32_t t_ahi = t_row + c * 256 + 3 * kH + j0 / 2, t_alo = t_ahi + 32;
            const float xv = kNoX ? __ldg(xs_base + (size_t)cblk[c] * 128) : 0.f;
            if (warp == 0 && lane == 0) CF_TR(2 + c, gs, 49);
            mbar_wait(&b[Cfg::kBarG], gs & 1);
            if (warp == 0 && lane == 0) CF_TR(2 + c, gs, 50);
            tc_fence_after_sync();
            uint32_t ar[16];
            tmem_ld16_nowait(t_acc, ar);
            tmem_ld_wait();
            uint32_t hi[8], lo[8];
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
                float2 r0, r1;
                sig4(ar + i, bias4(j0 + i, xv), r0, r1);
                const float2 p0 = fmul2(r0, h2[c][i >> 1]), p1 = fmul2(r1, h2[c][(i >> 1) + 1]);
                split4<FMT>(p0.x, p0.y, p1.x, p1.y, i, hi, lo);
            }
            tmem_st8_u32(t_ahi, hi);
            tmem_st8_u32(t_alo, lo);
            tmem_st_wait();
            tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&b[Cfg::kBarRh]);
            if (warp == 0 && lane == 0) CF_TR(2 + c, gs, 51);
        };
        // ---- phase C of chain c, step gs: update gate (while the candidate MMAs finish), candidate, h = c + u (h - c)
        auto phase_c = [&](int c, int gs) {
            uint64_t* b = &bars[8 * c];
            const uint32_t t_acc = t_row + c * 256 + j0;
            const uint32_t t_ahi = t_row + c * 256 + 3 * kH + j0 / 2, t_alo = t_ahi + 32;
            const uint32_t blk = cblk[c];
            const int s = spos[c];
            const float xv = kNoX ? __ldg(xs_base + (size_t)blk * 128) : 0.f;
            float2 u2[8];
            {
                uint32_t au[16];
                tmem_ld16_nowait(t_acc + kH, au);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 16; i += 4) sig4(au + i, bias4(kH + j0 + i, xv), u2[i >> 1], u2[(i >> 1) + 1]);
            }
            if (warp == 0 && lane == 0) CF_TR(2 + c, gs, 52);
            mbar_wait(&b[Cfg::kBarC], gs & 1);
            if (warp == 0 && lane == 0) CF_TR(2 + c, gs, 53);
            tc_fence_after_sync();
            uint32_t ac[16];
            tmem_ld16_nowait(t_acc + 2 * kH, ac);
            tmem_ld_wait();
            tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&b[Cfg::kBarCfree]);      // accumulators drained: next x part may start
            uint32_t hi[8], lo[8];
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
                float2 c0v, c1v;
                tanh4v(ac + i, bias4(2 * kH + j0 + i, xv), c0v, c1v);
                float2& ha = h2[c][i >> 1];
                float2& hb = h2[c][(i >> 1) + 1];
                ha = ffma2(u2[i >> 1], ffma2(c0v, splat2(-1.f), ha), c0v);
                hb = ffma2(u2[(i >> 1) + 1], ffma2(c1v, splat2(-1.f), hb), c1v);
                split4<FMT>(ha.x, ha.y, hb.x, hb.y, i, hi, lo);
            }
            const bool more = gs + 1 < tot[c];
            if (s + 1 < kWindow) {                       // hand h to the next step before the global stores
                tmem_st8_u32(t_ahi, hi);
                tmem_st8_u32(t_alo, lo);
                tmem_st_wait();
                tc_fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&b[Cfg::kBarH]);
            }
            if (warp == 0 && lane == 0) CF_TR(2 + c, gs, 55);
            if (y_out) {
                // next layer's A operand, in the NEXT layer's operand format (a second split when it differs)
                if (FMT_OUT != FMT) {
#pragma unroll
                    for (int i = 0; i < 16; i += 4)
                        split4<FMT_OUT>(h2[c][i >> 1].x, h2[c][i >> 1].y, h2[c][(i >> 1) + 1].x, h2[c][(i >> 1) + 1].y, i, hi, lo);
                }
                // hi[] = main words of the 16 values; lo[] = 4 words of remainder bytes then 4 of hi bytes (f16e5) /
                // 8 words of bf16 remainders (split bf16)
                uint8_t* ym = y_main + (size_t)blk * gru_out_block_bytes(FMT_OUT);
                *reinterpret_cast<uint4*>(ym) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                *reinterpret_cast<uint4*>(ym + 2048) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
                // compact form: only the remainder bytes travel (one 2 KB slab per K = 16 chunk of the block)
                *reinterpret_cast<uint4*>(ym + y_lo_delta) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                if (FMT_OUT != kFmtF16E5)
                    *reinterpret_cast<uint4*>(ym + y_lo_delta + 2048) = make_uint4(lo[4], lo[5], lo[6], lo[7]);
            }
            if (head_part) {
                const float* hw = head_w + dir * kH + j0;
                float2 acc2 = make_float2(0.f, 0.f);
#pragma unroll
                for (int i = 0; i < 8; ++i) acc2 = ffma2(h2[c][i], __ldg(reinterpret_cast<const float2*>(hw) + i), acc2);
                head_base[(size_t)blk * 1024] = acc2.x + acc2.y;
            }
            if (s + 1 == kWindow) {
                spos[c] = 0;
                cblk[c] = blk + blk_jump;
                if (more) begin_tile(c);                 // the chain's next tile starts from a zero state
            } else {
                spos[c] = s + 1;
                cblk[c] = blk + blk_step;
            }
            if (warp == 0 && lane == 0) CF_TR(2 + c, gs, 56);
        };

        if (tot[0] > 0) begin_tile(0);
        if (tot[1] > 0) begin_tile(1);
        const int g_end = tot[0] > tot[1] ? tot[0] : tot[1];
        for (int g = 0; g <= g_end; ++g) {
            if (g < tot[0]) phase_r(0, g);
            if (g >= 1 && g - 1 < tot[1]) phase_c(1, g - 1);
            if (g < tot[0]) phase_c(0, g);
            if (g < tot[1]) phase_r(1, g);
        }
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 16) tmem_dealloc<512>(tmem);
}

#undef CF_TR
#undef CF_TRC

// ====================================================================== TK5: head
// p = sigmoid(sum of the partial dots + b), scattered to sample order with the padding cut
// (head_output).  One CTA per tile: the partials are read window-fastest (coalesced), transposed
// through shared memory, and the probabilities are written position-fastest, which is contiguous in
// the read because consecutive windows of a read are consecutive in the signal.
__global__ void __launch_bounds__(256)
tc_head_kernel(const float* __restrict__ head_part, int n_parts, float b, int64_t tile0, int64_t n_rows, HeadOut out) {
    __shared__ float logit[kWindow][kTileWindows + 1];
    const int64_t tile = blockIdx.x;
    if (tile * kTileWindows * kWindow >= n_rows) return;
    for (int i = threadIdx.x; i < kWindow * kTileWindows; i += blockDim.x) {
        const int t = i / kTileWindows, w = i % kTileWindows;
        const size_t blk = (size_t)tile * kWindow + t;
        float acc = b;
        for (int k = 0; k < n_parts; ++k) acc += head_part[(blk * n_parts + k) * 128 + w];
        logit[t][w] = acc;
    }
    __syncthreads();
    // 4480 = 35 * 128 = 17.5 * 256: the tail iteration runs whole warps, so head_output's lanes are converged
    for (int i = threadIdx.x; i < kWindow * kTileWindows; i += blockDim.x) {
        const int w = i / kWindow, t = i % kWindow;
        const int64_t g = (tile0 + tile) * kTileWindows + w;
        head_output(out, g, t, t < out.valid[g], logit[t][w]);
    }
}

// ResNet-only head (resnet_class.py:23 commented out): dense 32 -> 1 + sigmoid straight from the
// conv stack's output blocks ({hi, lo} x [4][128][8] bf16 per block), scattered to sample order.
// One CTA per tile, like tc_head_kernel: the operand blocks are read window-fastest (each warp reads 512
// contiguous bytes per plane and K group), the logits are transposed through shared memory and the
// probabilities written position-fastest (contiguous in the read).
__global__ void __launch_bounds__(256)
tc_head_conv_kernel(const __nv_bfloat16* __restrict__ y, const float* __restrict__ w, float b, int64_t tile0, int64_t n_rows,
                    HeadOut out) {
    __shared__ float logit[kWindow][kTileWindows + 1];
    __shared__ float ws[kC];
    const int64_t tile = blockIdx.x;
    if (tile * kTileWindows * kWindow >= n_rows) return;
    if (threadIdx.x < kC) ws[threadIdx.x] = w[threadIdx.x];
    __syncthreads();
    for (int i = threadIdx.x; i < kWindow * kTileWindows; i += blockDim.x) {
        const int t = i / kTileWindows, wr = i % kTileWindows;
        const __nv_bfloat16* blk = y + ((size_t)tile * kWindow + t) * (2 * 128 * kC);
        float acc = b;
#pragma unroll
        for (int kg = 0; kg < kC / 8; ++kg) {
            const uint4 hi = *reinterpret_cast<const uint4*>(blk + ((size_t)kg * 128 + wr) * 8);
            const uint4 lo = *reinterpret_cast<const uint4*>(blk + 128 * kC + ((size_t)kg * 128 + wr) * 8);
            const uint32_t hw[4] = {hi.x, hi.y, hi.z, hi.w}, lw[4] = {lo.x, lo.y, lo.z, lo.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float v0 = __uint_as_float(hw[k] << 16) + __uint_as_float(lw[k] << 16);
                const float v1 = __uint_as_float(hw[k] & 0xffff0000u) + __uint_as_float(lw[k] & 0xffff0000u);
                acc = fmaf(v0, ws[kg * 8 + 2 * k], acc);
                acc = fmaf(v1, ws[kg * 8 + 2 * k + 1], acc);
            }
        }
        logit[t][wr] = acc;
    }
    __syncthreads();
    // whole warps in the tail iteration, as in tc_head_kernel
    for (int i = threadIdx.x; i < kWindow * kTileWindows; i += blockDim.x) {
        const int wr = i / kWindow, t = i % kWindow;
        const int64_t g = (tile0 + tile) * kTileWindows + wr;
        head_output(out, g, t, t < out.valid[g], logit[t][wr]);
    }
}

// ====================================================================== forward
static size_t tc_workspace_bytes(int64_t tiles) {
    const size_t blocks = (size_t)tiles * kWindow;
    size_t b = 0;
    b += blocks * 128 * kC * 2 * 2;          // conv output as A operand (K = 32)
    b += 2 * blocks * 128 * 2 * kH * 2 * 2;  // y ping-pong (K = 128 operands)
    b += blocks * 8 * 128 * 4;               // head partials
    return b + 4096;
}

int tc_reserve(DevBuf* ws, int64_t n_tiles) {
    if (n_tiles <= 0) return CF_OK;
    return ws->ensure(tc_workspace_bytes(n_tiles < kTcChunkTiles ? n_tiles : kTcChunkTiles));
}

// Every tensor-core kernel allocates all 512 TMEM columns of its SM.  Calls on different execution contexts may
// run kernels at the same time, so a second TMEM CTA must never be placed on an SM that already holds one (its
// allocation would wait for the first CTA to finish): each such kernel's dynamic shared memory is more than half
// of an SM's 228 KiB.
constexpr uint32_t kSmemPerSm = 228 * 1024;
static_assert(GruF2Cfg<128>::kSmem > kSmemPerSm / 2, "two tc_gru_fused2_kernel<128> CTAs could share an SM's TMEM");
static_assert(GruF2Cfg<32>::kSmem > kSmemPerSm / 2, "two tc_gru_fused2_kernel<32> CTAs could share an SM's TMEM");
static_assert(GruF2Cfg<1>::kSmem > kSmemPerSm / 2, "two tc_gru_fused2_kernel<1> CTAs could share an SM's TMEM");
static_assert(kConv4Smem > kSmemPerSm / 2, "two tc_conv4_kernel CTAs could share an SM's TMEM");
static_assert(kBlockSmem > kSmemPerSm / 2, "two tc_conv_block_kernel CTAs could share an SM's TMEM");
static_assert(kConvSmem > kSmemPerSm / 2, "two tc_conv2_kernel CTAs could share an SM's TMEM");

// The opt-in to more than 48 KB of dynamic shared memory, once per engine (called from tc_create).
static int tc_set_attributes() {
    CF_CUDA(cudaFuncSetAttribute(tc_gru_fused2_kernel<1, 0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, GruF2Cfg<1>::kSmem));
    CF_CUDA(cudaFuncSetAttribute(tc_gru_fused2_kernel<1, 1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, GruF2Cfg<1>::kSmem));
    CF_CUDA(cudaFuncSetAttribute(tc_gru_fused2_kernel<32, 0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, GruF2Cfg<32>::kSmem));
    CF_CUDA(cudaFuncSetAttribute(tc_gru_fused2_kernel<32, 0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, GruF2Cfg<32>::kSmem));
    CF_CUDA(cudaFuncSetAttribute(tc_gru_fused2_kernel<128, 0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, GruF2Cfg<128>::kSmem));
    CF_CUDA(cudaFuncSetAttribute(tc_gru_fused2_kernel<128, 1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, GruF2Cfg<128>::kSmem));
    CF_CUDA(cudaFuncSetAttribute(tc_conv2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kConvSmem));
    CF_CUDA(cudaFuncSetAttribute(tc_conv4_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kConv4Smem));
    CF_CUDA(cudaFuncSetAttribute(tc_conv_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kBlockSmem));
    return CF_OK;
}

int tc_forward(TcEngine* e, DevBuf* ws, const int16_t* raw, const double* stats, const float* xwin, WindowTable tab,
               int64_t n_tiles, float* probs, cudaStream_t stream, Profiler* prof, bool want_logits, const LabelBits* bits) {
    if (n_tiles <= 0) return CF_OK;
    const HeadOut head{tab.src, tab.valid, tab.read, raw ? stats : nullptr, probs, bits ? bits->lwords : nullptr,
                      bits ? bits->threshold : 0.0, want_logits ? 1 : 0};
    const int64_t chunk = n_tiles < kTcChunkTiles ? n_tiles : kTcChunkTiles;
    CF_TRY(ws->ensure(tc_workspace_bytes(chunk)));
    const size_t blocks_max = (size_t)chunk * kWindow;
    uint8_t* p = static_cast<uint8_t*>(ws->ptr);
    __nv_bfloat16* a0 = reinterpret_cast<__nv_bfloat16*>(p);
    p += blocks_max * 128 * kC * 2 * 2;
    __nv_bfloat16* ybuf[2];
    ybuf[0] = reinterpret_cast<__nv_bfloat16*>(p);
    p += blocks_max * 128 * 2 * kH * 2 * 2;
    ybuf[1] = reinterpret_cast<__nv_bfloat16*>(p);
    p += blocks_max * 128 * 2 * kH * 2 * 2;
    float* head_part = reinterpret_cast<float*>(p);

    const int n_layers = (int)e->layers.size();
    for (int64_t tile0 = 0; tile0 < n_tiles; tile0 += kTcChunkTiles) {
        const int64_t tiles = std::min<int64_t>(kTcChunkTiles, n_tiles - tile0);
        const int64_t blocks = tiles * kWindow;
        const int64_t rows = blocks * 128;
        float* feat = nullptr;                   // RNN-only networks: the normalised scalar input x [rows]
        const __nv_bfloat16* a_in = nullptr;
        if (e->conv_params.ptr) {
            ProfScope ps(prof, KC_K2_CONV, stream);
            const int grid = (int)std::min<int64_t>(tiles, e->n_sms);
            const bool fused_head = n_layers == 0 && e->conv_nres == 2;
            if (e->conv_nres >= 2)
                tc_conv4_kernel<<<grid, 576, kConv4Smem, stream>>>(e->conv_params.as<uint8_t>(), raw, stats, xwin, tab.src,
                                                                  tab.valid, tab.read, tile0, (int)tiles, a0,
                                                                  fused_head ? e->head_w.as<float>() : nullptr,
                                                                  fused_head ? head_part : nullptr);
            else
                tc_conv2_kernel<<<grid, 288, kConvSmem, stream>>>(e->conv_params.as<uint8_t>(), raw, stats, xwin, tab.src, tab.valid,
                                                                  tab.read, tile0, (int)tiles, a0);
            CF_LAUNCHED();
            a_in = a0;
            // further blocks alternate between a0 and ybuf[1], which the GRU layers do not touch before layer 1
            // writes it; the last block's output is never in ybuf[0], which GRU layer 0 writes while reading it
            for (int b = 2; b < e->conv_nres; ++b) {
                __nv_bfloat16* out = a_in == a0 ? ybuf[1] : a0;
                tc_conv_block_kernel<<<grid, 320, kBlockSmem, stream>>>(
                    e->conv_params.as<uint8_t>() + (size_t)(b - 1) * ConvParams::kBytes, a_in, (int)tiles, out);
                CF_LAUNCHED();
                a_in = out;
            }
        } else {
            // no residual blocks: a0, which only the conv stack writes, holds the scalar input (rows * 4 bytes)
            ProfScope ps(prof, KC_K2_CONV, stream);
            feat = reinterpret_cast<float*>(a0);
            CF_TRY(k1_fill_windows(raw, stats, xwin, tab, tile0, tiles, feat, stream));
        }
        for (int l = 0; l < n_layers; ++l) {
            const TcLayer& L = e->layers[l];
            const bool last = l + 1 == n_layers;
            __nv_bfloat16* yo = last ? nullptr : ybuf[l & 1];
            // input projection + recurrence in one kernel; a_in is the A-operand form of the layer input
            ProfScope ps(prof, KC_K4_GRU, stream);
            long long* trace_dev = nullptr;
#ifdef CF_TRACE_PROBES
            if (e->trace_path && !e->trace_done && L.in != kC) {
                CF_CUDA(cudaMalloc(&trace_dev, 6 * 200 * 2 * sizeof(long long)));
                CF_CUDA(cudaMemsetAsync(trace_dev, 0, 6 * 200 * 2 * sizeof(long long), stream));
            }
#endif
            const int grid2 = 2 * (int)std::min<int64_t>((tiles + 1) / 2, e->n_sms / 2);
            const float* hw_l = last ? e->head_w.as<float>() : nullptr;
            float* hp_l = last ? head_part : nullptr;
            // operand format of this layer and of the layer that reads its output
            const int fmt_out = last ? L.fmt : e->layers[l + 1].fmt;
            if (L.in == 1) {
                // scalar input (RNN-only layer 0): x part in the epilogue from the fp32 signal rows
                if (L.fmt == kFmtF16E5)
                    tc_gru_fused2_kernel<1, 1, 1><<<grid2, kGruF2Threads, GruF2Cfg<1>::kSmem, stream>>>(
                        L.wfused.as<uint8_t>(), L.bz.as<float>(), nullptr, yo, hw_l, hp_l, (int)tiles, nullptr, feat, L.wxz.as<float>());
                else
                    tc_gru_fused2_kernel<1, 0, 0><<<grid2, kGruF2Threads, GruF2Cfg<1>::kSmem, stream>>>(
                        L.wfused.as<uint8_t>(), L.bz.as<float>(), nullptr, yo, hw_l, hp_l, (int)tiles, nullptr, feat, L.wxz.as<float>());
            } else if (L.in == kC) {
                if (fmt_out == kFmtF16E5)
                    tc_gru_fused2_kernel<32, 0, 1><<<grid2, kGruF2Threads, GruF2Cfg<32>::kSmem, stream>>>(
                        L.wfused.as<uint8_t>(), L.bz.as<float>(), a_in, yo, hw_l, hp_l, (int)tiles, nullptr, nullptr, nullptr);
                else
                    tc_gru_fused2_kernel<32, 0, 0><<<grid2, kGruF2Threads, GruF2Cfg<32>::kSmem, stream>>>(
                        L.wfused.as<uint8_t>(), L.bz.as<float>(), a_in, yo, hw_l, hp_l, (int)tiles, nullptr, nullptr, nullptr);
            } else if (L.fmt == kFmtF16E5) {
                tc_gru_fused2_kernel<128, 1, 1><<<grid2, kGruF2Threads, GruF2Cfg<128>::kSmem, stream>>>(
                    L.wfused.as<uint8_t>(), L.bz.as<float>(), a_in, yo, hw_l, hp_l, (int)tiles, trace_dev, nullptr, nullptr);
            } else {
                tc_gru_fused2_kernel<128, 0, 0><<<grid2, kGruF2Threads, GruF2Cfg<128>::kSmem, stream>>>(
                    L.wfused.as<uint8_t>(), L.bz.as<float>(), a_in, yo, hw_l, hp_l, (int)tiles, trace_dev, nullptr, nullptr);
            }
            CF_LAUNCHED();
#ifdef CF_TRACE_PROBES
            if (trace_dev) {
                // debug (CF_TC_TRACE=<file>): dump the timeline of block 0 once; results are unaffected
                CF_CUDA(cudaStreamSynchronize(stream));
                std::vector<long long> host(6 * 200 * 2);
                CF_CUDA(cudaMemcpy(host.data(), trace_dev, host.size() * sizeof(long long), cudaMemcpyDeviceToHost));
                if (FILE* f = fopen(e->trace_path, "w")) {
                    for (int rg = 0; rg < 6; ++rg)
                        for (int k = 0; k < 200; ++k)
                            if (host[(rg * 200 + k) * 2 + 1])
                                fprintf(f, "%d %lld %lld\n", rg, host[(rg * 200 + k) * 2], host[(rg * 200 + k) * 2 + 1]);
                    fclose(f);
                }
                cudaFree(trace_dev);
                e->trace_done = true;
            }
#endif
            a_in = yo;
        }
        if (n_layers == 0 && e->conv_nres == 2) {
            // ResNet-only, two residual blocks: the conv kernel's epilogue already took the dense layer (two partial dots)
            ProfScope ps(prof, KC_K5_HEAD, stream);
            tc_head_kernel<<<(unsigned)tiles, 256, 0, stream>>>(head_part, 2, e->head_b, tile0, rows, head);
            CF_LAUNCHED();
        } else if (n_layers == 0) {
            // ResNet-only: dense on the conv output
            ProfScope ps(prof, KC_K5_HEAD, stream);
            tc_head_conv_kernel<<<(unsigned)tiles, 256, 0, stream>>>(a_in, e->head_w.as<float>(), e->head_b, tile0, rows, head);
            CF_LAUNCHED();
        } else {
            // GRU head: the last layer's epilogue wrote eight partial dots per position (2 directions x 4 unit groups)
            ProfScope ps(prof, KC_K5_HEAD, stream);
            tc_head_kernel<<<(unsigned)tiles, 256, 0, stream>>>(head_part, 8, e->head_b, tile0, rows, head);
            CF_LAUNCHED();
        }
    }
    return CF_OK;
}

// ====================================================================== self-test of the f16e5 MMA pair
// out[w][n] = sum_k a[w][k] wm[k][n] for one 128-row tile through the fp16 + e5m2-correction scheme:
// A produced on the device by split_f16e5_chunk into shared memory (mode 0, ".ss") or tensor memory
// (mode 1, ".ts"), B packed on the host by pack_b_operand_f16e5.  Pins the operand byte orders, the
// kind::f8f6f4 descriptors and the mixing of MMA kinds on one fp32 accumulator.
__global__ void __launch_bounds__(128, 1)
tc_selftest_f16e5_kernel(const float* __restrict__ a, const uint8_t* __restrict__ wpk, int K, int N, int mode,
                         float* __restrict__ out) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* a_s = smem;                               // {fp16 [K/8][128][8] | e5m2 [2K/16][128][16]}
    uint8_t* w_s = smem + 128 * K * 4;                 // {fp16 [K/8][N][8] | e5m2 [2K/16][N][16]}
    uint64_t* bar = reinterpret_cast<uint64_t*>(w_s + (size_t)N * K * 4);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);
    const int row = threadIdx.x, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) { mbar_init(bar, 1); fence_mbar_init(); }
    if (warp == 0) tmem_alloc<256>(tmem_slot);
    for (int i = threadIdx.x; i < N * K * 4 / 16; i += 128)
        reinterpret_cast<uint4*>(w_s)[i] = reinterpret_cast<const uint4*>(wpk)[i];
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    const uint32_t t_row = tmem + ((uint32_t)(warp * 32) << 16);
    constexpr uint32_t kTmA = 128;                      // operand columns: chunk c -> fp16 at 16 c, e5m2 at 16 c + 8
    for (int c = 0; c < K / 16; ++c) {
        float v[16];
        for (int i = 0; i < 16; ++i) v[i] = a[(size_t)row * K + 16 * c + i];
        uint32_t m8[8], lo4[4], hi4[4];
        split_f16e5_chunk(v, m8, lo4, hi4);
        if (mode == 0) {
            *reinterpret_cast<uint4*>(a_s + (2 * c) * 2048 + row * 16) = make_uint4(m8[0], m8[1], m8[2], m8[3]);
            *reinterpret_cast<uint4*>(a_s + (2 * c + 1) * 2048 + row * 16) = make_uint4(m8[4], m8[5], m8[6], m8[7]);
            uint8_t* corr = a_s + 128 * K * 2;
            *reinterpret_cast<uint4*>(corr + (2 * c) * 2048 + row * 16) = make_uint4(lo4[0], lo4[1], lo4[2], lo4[3]);
            *reinterpret_cast<uint4*>(corr + (2 * c + 1) * 2048 + row * 16) = make_uint4(hi4[0], hi4[1], hi4[2], hi4[3]);
        } else {
            uint32_t c8[8] = {lo4[0], lo4[1], lo4[2], lo4[3], hi4[0], hi4[1], hi4[2], hi4[3]};
            tmem_st8_u32(t_row + kTmA + 16 * c, m8);
            tmem_st8_u32(t_row + kTmA + 16 * c + 8, c8);
        }
    }
    fence_proxy_async_smem();
    tmem_st_wait();
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after_sync();
        const uint32_t elected = elect_one();
        const uint32_t a_u = smem_u32(a_s), w_u = smem_u32(w_s);
        const uint32_t id16 = make_idesc_f16(128, N), id8 = make_idesc_e5m2(128, N);
        for (int c = 0; c < K / 16; ++c) {
            const uint64_t bm = make_smem_desc(w_u + c * 2 * (N * 16), N * 16, 128);
            const uint64_t bc = make_smem_desc(w_u + K * N * 2 + c * 2 * (N * 16), N * 16, 128);
            if (mode == 0) {
                umma_bf16_pred(tmem, make_smem_desc(a_u + c * 4096, 2048, 128), bm, id16, c > 0, elected);
                umma_f8_pred(tmem, make_smem_desc(a_u + 128 * K * 2 + c * 4096, 2048, 128), bc, id8, 1, elected);
            } else {
                umma_bf16_ts_pred(tmem, tmem + kTmA + 16 * c, bm, id16, c > 0, elected);
                umma_f8_ts_pred(tmem, tmem + kTmA + 16 * c + 8, bc, id8, 1, elected);
            }
        }
        umma_commit_pred(bar, elected);
    }
    mbar_wait(bar, 0);
    tc_fence_after_sync();
    for (int n0 = 0; n0 < N; n0 += 16) {
        float v[16];
        tmem_ld16(t_row + n0, v);
        for (int i = 0; i < 16; ++i) out[(size_t)row * N + n0 + i] = v[i];
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc<256>(tmem);
}

int tc_selftest_f16e5(const float* a_dev, int K, int N, const float* w_host, int mode, float* out_dev, cudaStream_t stream) {
    if (K % 16 || K < 16 || K > 64 || N % 16 || N < 16 || N > 128 || (mode != 0 && mode != 1)) {
        set_error("selftest_f16e5: K in {16..64} and N in {16..128}, multiples of 16; mode 0 or 1");
        return CF_ERR_BAD_ARG;
    }
    std::vector<__nv_bfloat16> wpk;
    pack_b_operand_f16e5(w_host, K, N, N, 0, &wpk);
    DevBuf w;
    CF_TRY(w.ensure(wpk.size() * 2));
    CF_CUDA(cudaMemcpyAsync(w.ptr, wpk.data(), wpk.size() * 2, cudaMemcpyHostToDevice, stream));
    const size_t smem = (size_t)128 * K * 4 + (size_t)N * K * 4 + 64;
    CF_CUDA(cudaFuncSetAttribute(tc_selftest_f16e5_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    tc_selftest_f16e5_kernel<<<1, 128, smem, stream>>>(a_dev, w.as<uint8_t>(), K, N, mode, out_dev);
    CF_LAUNCHED();
    CF_CUDA(cudaStreamSynchronize(stream));
    return CF_OK;
}

}  // namespace cf
