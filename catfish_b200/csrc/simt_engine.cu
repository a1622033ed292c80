// SIMT engine: the forward graph in fp32 on CUDA cores, for any hyper-parameters.
//
// Role: (1) on-device cross-check of the tcgen05 engine at sizes the CPU oracle cannot reach,
// (2) the path for shapes the tcgen05 kernels are not specialised for (e.g. H = 256).
// Restates resnet_class.py:44-82 (residual blocks), rnn_class.py:142-175 (bidirectional
// GRUCell stack, reset gate applied before the candidate matmul, zero initial state per
// window) and rnn_class.py:178-183,84 (dense + sigmoid).
//
// Activation layout ("tile-time-major"): row index ((tile * 35 + t) * 128 + w), channels last.
// A conv tap at t +- 1 is therefore a shift by a whole 128-row block inside the tile, and a GRU
// step reads one contiguous 128-row block.
#include <cmath>

#include "model.cuh"

namespace cf {

constexpr int kSimtChunkTiles = 256;

struct SimtEngine {
    // weights
    std::vector<DevBuf> conv_w, conv_b;
    std::vector<DevBuf> gru_wx, gru_bx;      // per layer: [in][6H], [6H] (fw r|u|c, bw r|u|c)
    std::vector<DevBuf> gru_wgh, gru_wch;    // per layer*2+dir
    DevBuf head_w;
    float head_b = 0.f;
};

void EngineDelete::operator()(SimtEngine* e) const { delete e; }

// Appends a device copy of v to list.
static int upload(std::vector<DevBuf>* list, const std::vector<float>& v) {
    list->emplace_back();
    return list->back().upload(v);
}

int simt_create(const HostModel& hm, SimtEnginePtr* out) {
    SimtEnginePtr e(new SimtEngine());
    for (const ConvLayer& c : hm.convs) {
        CF_TRY(upload(&e->conv_w, c.w));
        CF_TRY(upload(&e->conv_b, c.b));
    }
    const int n_rnn = hm.n_rnn();
    for (int l = 0; l < n_rnn; ++l) {
        const GruDir& f = hm.gru[2 * l];
        const GruDir& b = hm.gru[2 * l + 1];
        const int h3 = 3 * f.h;
        std::vector<float> wx((size_t)f.in * 2 * h3), bx(2 * h3);
        for (int k = 0; k < f.in; ++k)
            for (int j = 0; j < h3; ++j) {
                wx[(size_t)k * 2 * h3 + j] = f.wx[(size_t)k * h3 + j];
                wx[(size_t)k * 2 * h3 + h3 + j] = b.wx[(size_t)k * h3 + j];
            }
        for (int j = 0; j < h3; ++j) { bx[j] = f.bx[j]; bx[h3 + j] = b.bx[j]; }
        CF_TRY(upload(&e->gru_wx, wx));
        CF_TRY(upload(&e->gru_bx, bx));
        for (int d = 0; d < 2; ++d) {
            CF_TRY(upload(&e->gru_wgh, hm.gru[2 * l + d].wgh));
            CF_TRY(upload(&e->gru_wch, hm.gru[2 * l + d].wch));
        }
    }
    CF_TRY(e->head_w.upload(hm.head_w));
    e->head_b = hm.head_b;
    *out = std::move(e);
    return CF_OK;
}

// ---------------------------------------------------------------- input
// x[(tile*35+t)*128+w] = t < valid ? float((raw - shift) / scale) : 0   (infer.py:32-38,105; the
// f64 -> f32 cast is the placeholder feed of rnn_class.py:159)
__global__ void simt_fill_x_kernel(const int16_t* __restrict__ raw, const double* __restrict__ stats,
                                   const float* __restrict__ xwin, const int64_t* __restrict__ src,
                                   const int32_t* __restrict__ valid, const int32_t* __restrict__ read,
                                   int64_t tile0, int64_t n_rows, float* __restrict__ x) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // local row
    if (i >= n_rows) return;
    const int w = (int)(i % kTileWindows);
    const int64_t tt = i / kTileWindows;
    const int t = (int)(tt % kWindow);
    const int64_t tile = tt / kWindow;
    const int64_t g = (tile0 + tile) * kTileWindows + w;
    float v = 0.f;
    if (t < valid[g]) {
        if (raw) {
            const int r = read[g];
            v = (float)(((double)raw[src[g] + t] - stats[2 * r]) / stats[2 * r + 1]);
        } else {
            v = xwin[src[g] + t];
        }
    }
    x[i] = v;
}

// ---------------------------------------------------------------- conv1d (+ folded BN, relu, residual)
// out[row][co] = act( sum_tap sum_ci in[row + (tap-pad)*128][ci] * w[tap][ci][co] + b[co] )
// with zero contribution when t + tap - pad falls outside [0, 35) ("same" padding per window).
// If res != nullptr: out = relu(act(...) + res[row][co])   (resnet_class.py:79-80)
__global__ void simt_conv_kernel(const float* __restrict__ in, const float* __restrict__ w,
                                 const float* __restrict__ b, const float* __restrict__ res,
                                 float* __restrict__ out, int64_t n_rows, int k, int cin, int cout,
                                 int relu) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t row = idx / cout;
    const int co = (int)(idx % cout);
    if (row >= n_rows) return;
    const int t = (int)((row / kTileWindows) % kWindow);
    const int pad = (k - 1) / 2;
    float acc = b[co];
    for (int tap = 0; tap < k; ++tap) {
        const int tt = t + tap - pad;
        if (tt < 0 || tt >= kWindow) continue;
        const float* ip = in + (row + (int64_t)(tap - pad) * kTileWindows) * cin;
        const float* wp = w + (size_t)tap * cin * cout + co;
        for (int ci = 0; ci < cin; ++ci) acc = fmaf(ip[ci], wp[(size_t)ci * cout], acc);
    }
    if (relu) acc = fmaxf(acc, 0.f);
    if (res) acc = fmaxf(acc + res[row * cout + co], 0.f);
    out[row * cout + co] = acc;
}

// ---------------------------------------------------------------- C = A B + bias (fp32, smem tiled)
// A [M][K] row-major, B [K][N] row-major, C [M][N].  64x64 tile, 16-wide k slabs, 4x4 per thread.
__global__ void __launch_bounds__(256)
simt_gemm_bias_kernel(const float* __restrict__ A, const float* __restrict__ B, const float* __restrict__ bias,
                      float* __restrict__ C, int64_t M, int N, int K) {
    __shared__ float As[16][64 + 4];
    __shared__ float Bs[16][64 + 4];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int64_t m0 = (int64_t)blockIdx.x * 64;
    const int n0 = blockIdx.y * 64;
    float acc[4][4] = {};
    for (int k0 = 0; k0 < K; k0 += 16) {
        for (int i = threadIdx.x; i < 64 * 16; i += 256) {
            const int m = i >> 4, kk = i & 15;
            As[kk][m] = (m0 + m < M && k0 + kk < K) ? A[(m0 + m) * K + k0 + kk] : 0.f;
        }
        for (int i = threadIdx.x; i < 16 * 64; i += 256) {
            const int kk = i >> 6, n = i & 63;
            Bs[kk][n] = (k0 + kk < K && n0 + n < N) ? B[(size_t)(k0 + kk) * N + n0 + n] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            float a[4], bb[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) bb[j] = Bs[kk][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t m = m0 + ty * 4 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n < N) C[m * N + n] = acc[i][j] + bias[n];
        }
    }
}

// ---------------------------------------------------------------- GRU recurrence
// One CTA = 32 windows of one tile, one direction.  Thread (wl = tid % 32, ug = tid / 32) owns
// window wl and hidden units j = ug, ug + 8, ... ; xp holds x W_x + b for every (t, window).
//   g = sigmoid(xp[r|u] + h Wgh);  c = tanh(xp[c] + (r*h) Wch);  h' = u h + (1-u) c
__device__ __forceinline__ float sigmoid_f(float x) { return 1.f / (1.f + expf(-x)); }
__device__ __forceinline__ float tanh_f(float x) {
    const float e = expf(-2.f * fabsf(x));
    const float t = (1.f - e) / (1.f + e);
    return copysignf(t, x);
}

__global__ void __launch_bounds__(256)
simt_gru_kernel(const float* __restrict__ xp, const float* __restrict__ wgh_fw,
                const float* __restrict__ wch_fw, const float* __restrict__ wgh_bw,
                const float* __restrict__ wch_bw, float* __restrict__ y, int H) {
    extern __shared__ float sm[];
    const int hs = H + 1;                         // padded row stride
    float* hbuf = sm;                             // [32][hs]
    float* rhbuf = sm + 32 * hs;                  // [32][hs]
    const int64_t tile = blockIdx.x;
    const int wg = blockIdx.y;                    // window group 0..3
    const int dir = blockIdx.z;
    const float* wgh = dir ? wgh_bw : wgh_fw;
    const float* wch = dir ? wch_bw : wch_fw;
    const int wl = threadIdx.x & 31, ug = threadIdx.x >> 5;
    const int w = wg * 32 + wl;
    constexpr int kMaxUnits = 32;                 // H <= 256
    float u_keep[kMaxUnits], h_old[kMaxUnits];
    for (int j = ug; j < H; j += 8) hbuf[wl * hs + j] = 0.f;
    __syncthreads();
    for (int s = 0; s < kWindow; ++s) {
        const int t = dir ? kWindow - 1 - s : s;
        const int64_t row = (tile * kWindow + t) * kTileWindows + w;
        const float* xrow = xp + row * (6 * (int64_t)H) + dir * 3 * H;
        int n = 0;
        for (int j = ug; j < H; j += 8, ++n) {
            float ar = xrow[j], au = xrow[H + j];
            for (int k = 0; k < H; ++k) {
                const float hk = hbuf[wl * hs + k];
                ar = fmaf(hk, wgh[(size_t)k * 2 * H + j], ar);
                au = fmaf(hk, wgh[(size_t)k * 2 * H + H + j], au);
            }
            const float r = sigmoid_f(ar);
            const float hj = hbuf[wl * hs + j];
            u_keep[n] = sigmoid_f(au);
            h_old[n] = hj;
            rhbuf[wl * hs + j] = r * hj;
        }
        __syncthreads();
        n = 0;
        float hn[kMaxUnits];
        for (int j = ug; j < H; j += 8, ++n) {
            float ac = xrow[2 * H + j];
            for (int k = 0; k < H; ++k) ac = fmaf(rhbuf[wl * hs + k], wch[(size_t)k * H + j], ac);
            const float c = tanh_f(ac);
            hn[n] = u_keep[n] * h_old[n] + (1.f - u_keep[n]) * c;
        }
        __syncthreads();
        n = 0;
        for (int j = ug; j < H; j += 8, ++n) {
            hbuf[wl * hs + j] = hn[n];
            y[row * (2 * (int64_t)H) + dir * H + j] = hn[n];
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------- dense + sigmoid + un-window
// p = sigmoid(y[row] . w + b), written to probs[src[g] + t] for the real (unpadded) positions
// (rnn_class.py:178-183,84; the cut of the padding is infer.py:47).
__global__ void simt_head_kernel(const float* __restrict__ y, const float* __restrict__ w, float b, int F,
                                 const int64_t* __restrict__ src, const int32_t* __restrict__ valid,
                                 const int32_t* __restrict__ read, const double* __restrict__ stats,
                                 int64_t tile0, int64_t n_rows, float* __restrict__ probs, int want_logits) {
    // thread i handles (window, t) with t fastest so that the scatter is coalesced
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const int t = (int)(i % kWindow);
    const int64_t wi = i / kWindow;                      // tile * 128 + w (local)
    const int w_in = (int)(wi % kTileWindows);
    const int64_t tile = wi / kTileWindows;
    const int64_t g = (tile0 + tile) * kTileWindows + w_in;
    if (t >= valid[g]) return;
    const float* yr = y + ((tile * kWindow + t) * kTileWindows + w_in) * (int64_t)F;
    float acc = b;
    for (int k = 0; k < F; ++k) acc = fmaf(yr[k], w[k], acc);
    float p = want_logits ? acc : 1.f / (1.f + expf(-acc));
    if (stats) {                                         // scale == 0 or NaN: the reference divides by it
        const double sc = stats[2 * read[g] + 1];
        if (!(sc > 0.0)) p = nanf("");
    }
    probs[src[g] + t] = p;
}

// ---------------------------------------------------------------- forward
// Carve the workspace for passes of at most `chunk_tiles` tiles.
struct SimtBufs { float *x, *ca, *cb, *csc, *cout, *xproj, *y0, *y1; };

static int simt_prepare(DevBuf* ws, const HostModel& hm, int64_t chunk_tiles, bool with_rnn, SimtBufs* b) {
    const int64_t rows = chunk_tiles * kWindow * kTileWindows;
    const int C = hm.conv_channels(), H = hm.desc.layer_size;
    const bool res = hm.n_res() > 0, rnn = with_rnn && hm.n_rnn() > 0;
    size_t fl = (size_t)rows;
    if (res) fl += (size_t)rows * C * 4;
    if (rnn) fl += (size_t)rows * (6 * H + 2 * 2 * H);
    CF_TRY(ws->ensure(fl * sizeof(float) + 1024));
    b->x = ws->as<float>();
    b->ca = b->x + rows;
    b->cb = b->ca + (res ? rows * C : 0);
    b->csc = b->cb + (res ? rows * C : 0);
    b->cout = b->csc + (res ? rows * C : 0);
    b->xproj = b->cout + (res ? rows * C : 0);
    b->y0 = b->xproj + (rnn ? rows * 6 * H : 0);
    b->y1 = b->y0 + (rnn ? rows * 2 * H : 0);
    return CF_OK;
}

// Normalise + window gather + residual blocks for tiles [tile0, tile0 + tiles): *feat points at
// fp32 rows [(tile*35+t)*128+w][C] (or [..][1] when the network has no residual blocks).
static int conv_stack(SimtEngine* e, const HostModel& hm, const SimtBufs& b, const int16_t* raw, const double* stats,
                      const float* xwin, WindowTable tab, int64_t tile0, int64_t tiles, const float** feat,
                      cudaStream_t stream, Profiler* prof) {
    const int64_t rows = tiles * kWindow * kTileWindows;
    {
        ProfScope ps(prof, KC_K2_CONV, stream);
        simt_fill_x_kernel<<<(unsigned)ceil_div(rows, 256), 256, 0, stream>>>(
            raw, stats, xwin, tab.src, tab.valid, tab.read, tile0, rows, b.x);
        CF_LAUNCHED();
    }
    *feat = b.x;
    for (int blk = 0; blk < hm.n_res(); ++blk) {
        auto conv = [&](int i, const float* in, const float* res, float* out, int relu) -> int {
            const ConvLayer& c = hm.convs[i];
            const int64_t total = rows * c.cout;
            ProfScope ps(prof, KC_K2_CONV, stream);
            simt_conv_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, stream>>>(
                in, e->conv_w[i].as<float>(), e->conv_b[i].as<float>(), res, out, rows, c.k, c.cin, c.cout, relu);
            CF_LAUNCHED();
            return CF_OK;
        };
        const int i = 4 * blk;
        CF_TRY(conv(i, *feat, nullptr, b.csc, 0));          // shortcut: BN(conv k1)
        CF_TRY(conv(i + 1, *feat, nullptr, b.ca, 1));
        CF_TRY(conv(i + 2, b.ca, nullptr, b.cb, 1));
        CF_TRY(conv(i + 3, b.cb, b.csc, b.cout, 1));        // relu(relu(BN(conv)) + shortcut)
        *feat = b.cout;                                     // conv i+3 no longer reads the block input
    }
    return CF_OK;
}

int simt_conv_stack(SimtEngine* e, DevBuf* ws, const HostModel& hm, const int16_t* raw, const double* stats,
                    const float* xwin, WindowTable tab, int64_t tile0, int64_t tiles, int64_t chunk_tiles,
                    const float** feat, cudaStream_t stream, Profiler* prof) {
    SimtBufs b;
    CF_TRY(simt_prepare(ws, hm, chunk_tiles, false, &b));
    return conv_stack(e, hm, b, raw, stats, xwin, tab, tile0, tiles, feat, stream, prof);
}

int simt_reserve(DevBuf* ws, const HostModel& hm, int64_t n_tiles) {
    if (n_tiles <= 0) return CF_OK;
    SimtBufs b;
    return simt_prepare(ws, hm, n_tiles < kSimtChunkTiles ? n_tiles : kSimtChunkTiles, true, &b);
}

int simt_conv_stack_reserve(DevBuf* ws, const HostModel& hm, int64_t chunk_tiles) {
    if (chunk_tiles <= 0) return CF_OK;
    SimtBufs b;
    return simt_prepare(ws, hm, chunk_tiles, false, &b);
}

int simt_forward(SimtEngine* e, DevBuf* ws, const HostModel& hm, const int16_t* raw, const double* stats,
                 const float* xwin, WindowTable tab, int64_t n_tiles, float* probs,
                 cudaStream_t stream, Profiler* prof, bool want_logits) {
    if (n_tiles <= 0) return CF_OK;
    const int64_t chunk = n_tiles < kSimtChunkTiles ? n_tiles : kSimtChunkTiles;
    SimtBufs b;
    CF_TRY(simt_prepare(ws, hm, chunk, true, &b));
    const int H = hm.desc.layer_size;
    for (int64_t tile0 = 0; tile0 < n_tiles; tile0 += kSimtChunkTiles) {
        const int64_t tiles = (n_tiles - tile0) < kSimtChunkTiles ? (n_tiles - tile0) : kSimtChunkTiles;
        const int64_t rows = tiles * kWindow * kTileWindows;
        const float* feat = nullptr;
        CF_TRY(conv_stack(e, hm, b, raw, stats, xwin, tab, tile0, tiles, &feat, stream, prof));
        const int feat_dim = hm.n_res() ? hm.conv_channels() : 1;
        float* yin = nullptr;
        for (int l = 0; l < hm.n_rnn(); ++l) {
            const int in_dim = l == 0 ? feat_dim : 2 * H;
            const float* a = l == 0 ? feat : yin;
            dim3 grid((unsigned)ceil_div(rows, 64), (unsigned)ceil_div(6 * H, 64));
            {
                ProfScope ps(prof, KC_K3_XPROJ, stream);
                simt_gemm_bias_kernel<<<grid, 256, 0, stream>>>(a, e->gru_wx[l].as<float>(), e->gru_bx[l].as<float>(), b.xproj,
                                                                rows, 6 * H, in_dim);
                CF_LAUNCHED();
            }
            float* yout = (l & 1) ? b.y1 : b.y0;
            const size_t smem = sizeof(float) * 2 * 32 * (H + 1);
            if (smem > 48 * 1024)      // H > ~190: opt in to the larger dynamic shared memory carve-out
                CF_CUDA(cudaFuncSetAttribute(simt_gru_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            {
                ProfScope ps(prof, KC_K4_GRU, stream);
                simt_gru_kernel<<<dim3((unsigned)tiles, 4, 2), 256, smem, stream>>>(
                    b.xproj, e->gru_wgh[2 * l].as<float>(), e->gru_wch[2 * l].as<float>(), e->gru_wgh[2 * l + 1].as<float>(),
                    e->gru_wch[2 * l + 1].as<float>(), yout, H);
                CF_LAUNCHED();
            }
            yin = yout;
        }
        const float* hin = hm.n_rnn() ? yin : feat;
        ProfScope ps(prof, KC_K5_HEAD, stream);
        simt_head_kernel<<<(unsigned)ceil_div(rows, 256), 256, 0, stream>>>(
            hin, e->head_w.as<float>(), e->head_b, hm.head_features(), tab.src, tab.valid, tab.read, raw ? stats : nullptr,
            tile0, rows, probs, want_logits ? 1 : 0);
        CF_LAUNCHED();
    }
    return CF_OK;
}

}  // namespace cf
