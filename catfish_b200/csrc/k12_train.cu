// K12: one RMSProp training step of the catfish graph in fp32 on CUDA cores, and the cf_trainer C ABI.
//
// The step is the reference's training graph (rnn_class.py / resnet_class.py with tf.train.RMSPropOptimizer):
//   forward   the inference graph with output dropout on every GRU cell (DropoutWrapper(output_keep_prob), the
//             while/dropout nodes of the shipped graph); BN with its moving statistics (training is never set)
//   loss      mean sigmoid cross-entropy over all n*35 positions (compute_loss, the formula of K9)
//   backward  dL/dz = (sigmoid(z) - y) / (n*35) back through head, GRU stack and residual blocks
//   update    TF 1.x ApplyRMSProp (decay 0.9, momentum 0, epsilon 1e-10) on every trainable variable
// Activations use the SIMT engine's tile-time-major layout: row ((tile * 35 + t) * 128 + w), channels last.  The
// forward reuses the SIMT engine's conv and GEMM kernels on the un-folded weights (the backward needs the pre-BN
// conv outputs, which the folded inference conv never forms).  Windows past n_windows only pad the last tile: their
// dL/dz is 0, so they add nothing to the loss or to any gradient.
//
// Dropout mask: Philox4x32-10 with key = seed, counter = (step, 2 * layer + direction, window, t * H + unit); the
// unit is kept when the top 24 bits of output word 0 are < round(keep_prob * 2^24).  The backward recomputes the
// mask instead of storing it.  keep_prob = 1 draws nothing.
//
// Every reduction over rows (weight gradients, loss) runs in a fixed order with no float atomics: two runs of the
// same step give bit-identical variables.
#include <cmath>
#include <cstring>
#include <mutex>

#include "model.cuh"
#include "window_io.cuh"

namespace cf {

// the SIMT engine's kernels (simt_engine.cu)
__global__ void simt_conv_kernel(const float* __restrict__ in, const float* __restrict__ w, const float* __restrict__ b,
                                 const float* __restrict__ res, float* __restrict__ out, int64_t n_rows, int k, int cin,
                                 int cout, int relu);
__global__ void __launch_bounds__(256)
simt_gemm_bias_kernel(const float* __restrict__ A, const float* __restrict__ B, const float* __restrict__ bias,
                      float* __restrict__ C, int64_t M, int N, int K);

constexpr int kTileRows = kWindow * kTileWindows;
constexpr float kRmsDecay = 0.9f, kRmsMomentum = 0.f, kRmsEpsilon = 1e-10f;
constexpr int64_t kAtbPartialFloats = (int64_t)8 << 20;   // split-row partial sums of one Aᵀ·B (32 MiB)
constexpr int kZeros = 2048;                               // >= every GEMM / conv output width (6 * 256, 1024)

// ---------------------------------------------------------------- dropout mask
__host__ __device__ __forceinline__ uint32_t philox4x32_10_word0(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                                  uint32_t k0, uint32_t k1) {
    for (int i = 0; i < 10; ++i) {
        if (i) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        c1 = (uint32_t)p1;
        c3 = (uint32_t)p0;
        c0 = n0;
        c2 = n2;
    }
    return c0;
}

struct Dropout {
    float keep;              // 1: no mask
    uint32_t threshold;      // round(keep * 2^24)
    uint32_t k0, k1, step;
    __device__ __forceinline__ bool on() const { return keep < 1.f; }
    __device__ __forceinline__ bool kept(int stream, uint32_t window, uint32_t pos) const {
        return (philox4x32_10_word0(step, (uint32_t)stream, window, pos, k0, k1) >> 8) < threshold;
    }
};

__device__ __forceinline__ float k12_sigmoid(float x) { return 1.f / (1.f + expf(-x)); }

// ---------------------------------------------------------------- weight packing (once per step)
// wx [fin][6H] (fw r|u|c, bw r|u|c) and bx [6H] for the input projection, wxT [6H][fin] for the gradient of the layer
// input, from the TF variables gates/kernel [fin+H][2H], candidate/kernel [fin+H][H] and their biases.
struct GruVars { const float *gk[2], *gb[2], *ck[2], *cb[2]; };

__global__ void k12_pack_gru_kernel(GruVars v, int fin, int H, float* __restrict__ wx, float* __restrict__ bx,
                                    float* __restrict__ wxT) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int h6 = 6 * H, h3 = 3 * H;
    if (i < h6) {
        const int d = (int)i / h3, j = (int)i % h3;
        bx[i] = j < 2 * H ? v.gb[d][j] : v.cb[d][j - 2 * H];
    }
    if (i >= (int64_t)fin * h6) return;
    const int k = (int)(i / h6), col = (int)(i % h6), d = col / h3, j = col % h3;
    const float w = j < 2 * H ? v.gk[d][(size_t)k * 2 * H + j] : v.ck[d][(size_t)k * H + j - 2 * H];
    wx[i] = w;
    wxT[(size_t)col * fin + k] = w;
}

// wt[tap'][co][ci] = w[k - 1 - tap'][ci][co]: simt_conv_kernel with wt maps a conv output gradient to its input gradient
__global__ void k12_conv_flip_kernel(const float* __restrict__ w, int k, int cin, int cout, float* __restrict__ wt) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)k * cin * cout) return;
    const int tap = (int)(i / ((int64_t)cin * cout)), ci = (int)(i / cout % cin), co = (int)(i % cout);
    wt[((size_t)(k - 1 - tap) * cout + co) * cin + ci] = w[i];
}

// ---------------------------------------------------------------- batch norm (moving statistics) + relu + residual
struct BnVars { const float *gamma, *beta, *mean, *var; };

// out = act(a * s + (beta - mean * s)), s = gamma / sqrt(var + eps), act = relu or identity; with res also
// out2 = relu(out + res) (the end of a residual block, resnet_class.py:79-80).
__global__ void k12_bn_fwd_kernel(const float* __restrict__ a, BnVars v, float eps, int C, int64_t total, int relu,
                                  float* __restrict__ out, const float* __restrict__ res, float* __restrict__ out2) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c = (int)(i % C);
    const float s = v.gamma[c] / sqrtf(v.var[c] + eps);
    float y = a[i] * s + (v.beta[c] - v.mean[c] * s);
    if (relu) y = fmaxf(y, 0.f);
    out[i] = y;
    if (res) out2[i] = fmaxf(y + res[i], 0.f);
}

// g = dy masked by act > 0 (act == nullptr: no relu); da = g * s, gx = g * (a - mean) / sqrt(var + eps).
// Column sums of g / gx / da are dbeta / dgamma / dbias.
__global__ void k12_bn_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ act, const float* __restrict__ a,
                                  BnVars v, float eps, int C, int64_t total, float* __restrict__ da, float* __restrict__ g,
                                  float* __restrict__ gx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c = (int)(i % C);
    const float gg = (!act || act[i] > 0.f) ? dy[i] : 0.f;
    const float rs = 1.f / sqrtf(v.var[c] + eps);
    g[i] = gg;
    gx[i] = gg * ((a[i] - v.mean[c]) * rs);
    da[i] = gg * (v.gamma[c] * rs);
}

// out = dy where act > 0, else 0
__global__ void k12_relu_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ act, int64_t total,
                                    float* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < total) out[i] = act[i] > 0.f ? dy[i] : 0.f;
}

__global__ void k12_add_kernel(const float* __restrict__ a, const float* __restrict__ b, int64_t total, float* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < total) out[i] = a[i] + b[i];
}

// ---------------------------------------------------------------- GRU forward with saved gates
// simt_gru_kernel's recurrence (one CTA = 32 windows of one tile, one direction; thread (wl, ug) owns window wl and
// units ug, ug + 8, ...) that also stores per (row, direction) the gates r, u, c, the state h, r * h_prev and the
// dropped output y = h / keep * mask, the next layer's (or the head's) input.
__global__ void __launch_bounds__(256)
k12_gru_fwd_kernel(const float* __restrict__ xp, const float* __restrict__ wgh_fw, const float* __restrict__ wch_fw,
                   const float* __restrict__ wgh_bw, const float* __restrict__ wch_bw, int H, int layer, Dropout drop,
                   float* __restrict__ gates, float* __restrict__ hraw, float* __restrict__ rh, float* __restrict__ y) {
    extern __shared__ float sm[];
    const int hs = H + 1;
    float* hbuf = sm;                      // [32][hs] state
    float* rhbuf = sm + 32 * hs;           // [32][hs] r * h
    const int64_t tile = blockIdx.x;
    const int dir = blockIdx.z;
    const float* wgh = dir ? wgh_bw : wgh_fw;
    const float* wch = dir ? wch_bw : wch_fw;
    const int wl = threadIdx.x & 31, ug = threadIdx.x >> 5;
    const int w = blockIdx.y * 32 + wl;
    const uint32_t window = (uint32_t)(tile * kTileWindows + w);
    const int64_t h2 = 2 * (int64_t)H, h6 = 6 * (int64_t)H;
    for (int j = ug; j < H; j += 8) hbuf[wl * hs + j] = 0.f;
    __syncthreads();
    for (int s = 0; s < kWindow; ++s) {
        const int t = dir ? kWindow - 1 - s : s;
        const int64_t row = (tile * kWindow + t) * kTileWindows + w;
        const float* xrow = xp + row * h6 + dir * 3 * H;
        float* g = gates + row * h6 + dir * 3 * H;
        for (int j = ug; j < H; j += 8) {
            float ar = xrow[j], au = xrow[H + j];
            for (int k = 0; k < H; ++k) {
                const float hk = hbuf[wl * hs + k];
                ar = fmaf(hk, wgh[(size_t)k * 2 * H + j], ar);
                au = fmaf(hk, wgh[(size_t)k * 2 * H + H + j], au);
            }
            const float r = k12_sigmoid(ar), u = k12_sigmoid(au);
            const float v = r * hbuf[wl * hs + j];
            g[j] = r;
            g[H + j] = u;
            rhbuf[wl * hs + j] = v;
            rh[row * h2 + dir * H + j] = v;
        }
        __syncthreads();
        // only this thread reads hbuf[wl][j] of its own units from here on: the new state overwrites it in place
        for (int j = ug; j < H; j += 8) {
            float ac = xrow[2 * H + j];
            for (int k = 0; k < H; ++k) ac = fmaf(rhbuf[wl * hs + k], wch[(size_t)k * H + j], ac);
            const float c = tanhf(ac), u = g[H + j];
            const float hn = u * hbuf[wl * hs + j] + (1.f - u) * c;
            g[2 * H + j] = c;
            hbuf[wl * hs + j] = hn;
            hraw[row * h2 + dir * H + j] = hn;
            float out = hn;
            if (drop.on()) out = drop.kept(2 * layer + dir, window, (uint32_t)(t * H + j)) ? hn / drop.keep : 0.f;
            y[row * h2 + dir * H + j] = out;
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------- head + loss
// z = y[row] . w + b per row; for real windows (< n_windows) the loss term (fp32, summed in double as K9), the
// round-half-even hit and dL/dz = (sigmoid(z) - label) / (n * 35); padding rows get dL/dz = 0.
// partial[block] = (loss sum, hits) reduced in a fixed order.
__global__ void __launch_bounds__(256)
k12_head_loss_kernel(const float* __restrict__ yin, int F, const float* __restrict__ w, const float* __restrict__ b,
                     const uint8_t* __restrict__ labels, int64_t n_windows, int64_t n_rows, float inv_count,
                     float* __restrict__ dz, double* __restrict__ partial) {
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double l = 0.0, hit = 0.0;
    if (row < n_rows) {
        const int64_t tile = row / kTileRows;
        const int t = (int)(row / kTileWindows % kWindow);
        const int64_t g = tile * kTileWindows + row % kTileWindows;
        float d = 0.f;
        if (g < n_windows) {
            float z = b[0];
            const float* yr = yin + row * F;
            for (int k = 0; k < F; ++k) z = fmaf(yr[k], w[k], z);
            const float y = (float)labels[g * kWindow + t];
            const float p = head_sigmoid(z);
            l = (double)(fmaxf(z, 0.f) - z * y + log1pf(expf(-fabsf(z))));
            hit = rintf(p) == y ? 1.0 : 0.0;
            d = (p - y) * inv_count;
        }
        dz[row] = d;
    }
    __shared__ double sl[8], sh[8];
    for (int o = 16; o > 0; o >>= 1) {
        l += __shfl_down_sync(0xffffffffu, l, o);
        hit += __shfl_down_sync(0xffffffffu, hit, o);
    }
    if ((threadIdx.x & 31) == 0) { sl[threadIdx.x >> 5] = l; sh[threadIdx.x >> 5] = hit; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, c = 0.0;
        for (int i = 0; i < 8; ++i) { a += sl[i]; c += sh[i]; }
        partial[2 * blockIdx.x] = a;
        partial[2 * blockIdx.x + 1] = c;
    }
}

__global__ void k12_loss_reduce_kernel(const double* __restrict__ partial, int n_blocks, double* __restrict__ result) {
    double a = 0.0, c = 0.0;
    for (int i = 0; i < n_blocks; ++i) { a += partial[2 * i]; c += partial[2 * i + 1]; }
    result[0] = a;
    result[1] = c;
}

// dy[row][k] = dz[row] * w[k]: the gradient at the head's input
__global__ void k12_head_bwd_kernel(const float* __restrict__ dz, const float* __restrict__ w, int F, int64_t total,
                                    float* __restrict__ dy) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < total) dy[i] = dz[i / F] * w[i % F];
}

// ---------------------------------------------------------------- GRU backward through time
// Same CTA shape as the forward, walking the 35 steps in reverse order of the forward's.  dh (shared) carries the
// gradient of the state after the current step; the output's gradient dy enters through the dropout mask.
//   h = u h_prev + (1 - u) c,   c = tanh(xc + (r h_prev) Wch),   [r|u] = sigmoid(x[r|u] + h_prev Wgh)
//   dc_pre = dh (1 - u)(1 - c^2)          du_pre = dh (h_prev - c) u (1 - u)
//   d(rh)  = dc_pre Wchᵀ                  dr_pre = d(rh) h_prev r (1 - r)
//   dh_prev = dh u + d(rh) r + [dr_pre | du_pre] Wghᵀ
// Writes the pre-activation gradients dpre[row][dir*3H + (r|u|c)] and h_prev[row][dir*H + j] for the weight
// gradients.
__global__ void __launch_bounds__(256)
k12_gru_bwd_kernel(const float* __restrict__ dyin, const float* __restrict__ gates, const float* __restrict__ hraw,
                   const float* __restrict__ wgh_fw, const float* __restrict__ wch_fw, const float* __restrict__ wgh_bw,
                   const float* __restrict__ wch_bw, int H, int layer, Dropout drop, float* __restrict__ dpre,
                   float* __restrict__ hprev) {
    extern __shared__ float sm[];
    const int hs = H + 1, gs = 2 * H + 1;
    float* dh = sm;                        // [32][hs]
    float* acc = dh + 32 * hs;             // [32][hs] dh u + d(rh) r
    float* dcp = acc + 32 * hs;            // [32][hs] dc_pre
    float* dgp = dcp + 32 * hs;            // [32][gs] dr_pre | du_pre
    const int64_t tile = blockIdx.x;
    const int dir = blockIdx.z;
    const float* wgh = dir ? wgh_bw : wgh_fw;
    const float* wch = dir ? wch_bw : wch_fw;
    const int wl = threadIdx.x & 31, ug = threadIdx.x >> 5;
    const int w = blockIdx.y * 32 + wl;
    const uint32_t window = (uint32_t)(tile * kTileWindows + w);
    const int64_t h2 = 2 * (int64_t)H, h6 = 6 * (int64_t)H;
    for (int j = ug; j < H; j += 8) dh[wl * hs + j] = 0.f;
    __syncthreads();
    for (int s = 0; s < kWindow; ++s) {
        const int t = dir ? s : kWindow - 1 - s;
        const int tp = dir ? t + 1 : t - 1;
        const bool has_prev = tp >= 0 && tp < kWindow;
        const int64_t row = (tile * kWindow + t) * kTileWindows + w;
        const int64_t rowp = (tile * kWindow + tp) * kTileWindows + w;
        const float* g = gates + row * h6 + dir * 3 * H;
        float* dp = dpre + row * h6 + dir * 3 * H;
        float* hp_out = hprev + row * h2 + dir * H;
        for (int j = ug; j < H; j += 8) {
            float dy = dyin[row * h2 + dir * H + j];
            if (drop.on()) dy = drop.kept(2 * layer + dir, window, (uint32_t)(t * H + j)) ? dy / drop.keep : 0.f;
            const float ht = dh[wl * hs + j] + dy;
            const float u = g[H + j], c = g[2 * H + j];
            const float hp = has_prev ? hraw[rowp * h2 + dir * H + j] : 0.f;
            hp_out[j] = hp;
            const float dc = ht * (1.f - u) * (1.f - c * c);
            const float du = ht * (hp - c) * u * (1.f - u);
            dcp[wl * hs + j] = dc;
            dgp[wl * gs + H + j] = du;
            dp[H + j] = du;
            dp[2 * H + j] = dc;
            acc[wl * hs + j] = ht * u;
        }
        __syncthreads();
        for (int k = ug; k < H; k += 8) {
            float drh = 0.f;
            for (int j = 0; j < H; ++j) drh = fmaf(dcp[wl * hs + j], wch[(size_t)k * H + j], drh);
            const float r = g[k], hp = hp_out[k];
            const float dr = drh * hp * r * (1.f - r);
            dgp[wl * gs + k] = dr;
            dp[k] = dr;
            acc[wl * hs + k] += drh * r;
        }
        __syncthreads();
        for (int k = ug; k < H; k += 8) {
            float a = acc[wl * hs + k];
            for (int j = 0; j < 2 * H; ++j) a = fmaf(dgp[wl * gs + j], wgh[(size_t)k * 2 * H + j], a);
            dh[wl * hs + k] = a;
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------- weight gradients: Aᵀ·B over rows
// partial[z][k][n] = sum over rows m of chunk z of A(m, k) B(m, n), with A(m, k) = A[(m + shift * 128) * lda + k]
// when window step t(m) + shift lies in [0, 35), else 0 (the taps of a "same" conv; shift = 0 otherwise).  lda = 0
// with A = {1.f} gives column sums.  32 x 32 outputs per CTA, rows in 32-row slabs in ascending order.
__global__ void __launch_bounds__(256)
k12_atb_kernel(const float* __restrict__ A, int64_t lda, int shift, const float* __restrict__ B, int64_t ldb, int64_t M,
               int K, int N, int64_t chunk, float* __restrict__ partial) {
    __shared__ float As[32][33], Bs[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int k0 = blockIdx.y * 32, n0 = blockIdx.x * 32;
    const int64_t m_beg = (int64_t)blockIdx.z * chunk;
    const int64_t m_end = m_beg + chunk < M ? m_beg + chunk : M;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int64_t mb = m_beg; mb < m_end; mb += 32) {
        for (int i = threadIdx.x; i < 32 * 32; i += 256) {
            const int r = i >> 5, c = i & 31;
            const int64_t m = mb + r;
            float a = 0.f, b = 0.f;
            if (m < m_end) {
                if (k0 + c < K) {
                    const int tt = (int)(m / kTileWindows % kWindow) + shift;
                    if (tt >= 0 && tt < kWindow) a = A[(m + (int64_t)shift * kTileWindows) * lda + k0 + c];
                }
                if (n0 + c < N) b = B[m * ldb + n0 + c];
            }
            As[r][c] = a;
            Bs[r][c] = b;
        }
        __syncthreads();
#pragma unroll 8
        for (int r = 0; r < 32; ++r) {
            const float b = Bs[r][tx];
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[i] = fmaf(As[r][ty + 8 * i], b, acc[i]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int k = k0 + ty + 8 * i, n = n0 + tx;
        if (k < K && n < N) partial[((int64_t)blockIdx.z * K + k) * N + n] = acc[i];
    }
}

// C[k * ldc + n] = sum over z in ascending order of partial[z][k][n]
__global__ void k12_atb_reduce_kernel(const float* __restrict__ partial, int S, int K, int N, float* __restrict__ C,
                                      int64_t ldc) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)K * N) return;
    float s = 0.f;
    for (int z = 0; z < S; ++z) s += partial[(int64_t)z * K * N + i];
    C[(i / N) * ldc + i % N] = s;
}

// ---------------------------------------------------------------- RMSProp (TF 1.x ApplyRMSProp, centered = False)
__global__ void k12_rmsprop_kernel(float* __restrict__ var, float* __restrict__ ms, float* __restrict__ mom,
                                   const float* __restrict__ grad, const uint8_t* __restrict__ trainable, int64_t n,
                                   float lr) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !trainable[i]) return;
    const float g = grad[i];
    const float m = ms[i] + (g * g - ms[i]) * (1.f - kRmsDecay);
    const float v = mom[i] * kRmsMomentum + lr * g / sqrtf(m + kRmsEpsilon);
    ms[i] = m;
    mom[i] = v;
    var[i] -= v;
}

}  // namespace cf

// ================================================================== trainer handle
struct cf_trainer {
    cf_model_desc desc{};
    int device = 0;
    int n_res = 0, n_rnn = 0, C = 0, H = 0;
    std::vector<int64_t> off, size;          // per tensor: offset into the flat buffers, element count
    int64_t total = 0;
    cf::DevBuf var, ms, mom, grad, trainable;
    cf::DevBuf consts;                       // {1.f} then kZeros zeros
    std::vector<cf::DevBuf> wx, bx, wxT;     // per GRU layer, packed each step
    std::vector<cf::DevBuf> convT;           // per conv, flipped each step
    cf::DevBuf ws, partial, loss_partial, result, tab_src, tab_valid, tab_read;
    std::mutex mu;
    cf::Event last_done;
};

namespace cf {
namespace {

constexpr unsigned kThreads = 256;
inline unsigned blocks_for(int64_t n) { return (unsigned)ceil_div(n, kThreads); }

// Index of the tensors of conv i (kernel, bias, gamma, beta, mean, var) and GRU layer l direction d (gates/kernel,
// gates/bias, candidate/kernel, candidate/bias), in the order of expected_tensor_shapes.
inline int conv_tensor(int i, int v) { return 6 * i + v; }
inline int gru_tensor(const cf_trainer* tr, int l, int d, int v) { return 24 * tr->n_res + 8 * l + 4 * d + v; }

struct Scope {
    std::lock_guard<std::mutex> lock;
    int prev = -1;
    explicit Scope(cf_trainer* tr) : lock(tr->mu) {}
    ~Scope() { if (prev >= 0) cudaSetDevice(prev); }
    int enter(int device) {
        int n = 0;
        if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
            cudaGetLastError();
            set_error("no CUDA device available; catfish_b200 has no CPU fallback");
            return CF_ERR_NO_DEVICE;
        }
        int cur = -1;
        if (cudaGetDevice(&cur) != cudaSuccess) { cudaGetLastError(); cur = -1; }
        CF_CUDA(cudaSetDevice(device));
        if (cur >= 0 && cur != device) prev = cur;
        return CF_OK;
    }
};

struct Trainer {
    cf_trainer* tr;
    cudaStream_t st;
    float* V(int i) const { return tr->var.as<float>() + tr->off[i]; }
    float* G(int i) const { return tr->grad.as<float>() + tr->off[i]; }
    const float* ones() const { return tr->consts.as<float>(); }
    const float* zeros() const { return tr->consts.as<float>() + 1; }

    // C[k * ldc + n] = sum_m A(m, k) B(m, n) (k12_atb_kernel) in a fixed order
    int atb(const float* A, int64_t lda, int shift, const float* B, int64_t ldb, int64_t M, int K, int N, float* C,
            int64_t ldc) {
        const int64_t kn = (int64_t)K * N;
        int64_t S = std::min<int64_t>(ceil_div(M, 256), std::max<int64_t>(1, kAtbPartialFloats / kn));
        const int64_t chunk = round_up(ceil_div(M, S), 32);
        S = ceil_div(M, chunk);
        k12_atb_kernel<<<dim3((unsigned)ceil_div(N, 32), (unsigned)ceil_div(K, 32), (unsigned)S), kThreads, 0, st>>>(
            A, lda, shift, B, ldb, M, K, N, chunk, tr->partial.as<float>());
        CF_LAUNCHED();
        k12_atb_reduce_kernel<<<blocks_for(kn), kThreads, 0, st>>>(tr->partial.as<float>(), (int)S, K, N, C, ldc);
        CF_LAUNCHED();
        return CF_OK;
    }
    BnVars bn(int i) const {
        return {V(conv_tensor(i, 2)), V(conv_tensor(i, 3)), V(conv_tensor(i, 4)), V(conv_tensor(i, 5))};
    }
    // a = conv(in) + bias with the un-folded kernel (simt_conv_kernel)
    int conv(int i, const float* in, int k, int cin, int64_t R, float* a) {
        simt_conv_kernel<<<blocks_for(R * tr->C), kThreads, 0, st>>>(in, V(conv_tensor(i, 0)), V(conv_tensor(i, 1)),
                                                                     nullptr, a, R, k, cin, tr->C, 0);
        CF_LAUNCHED();
        return CF_OK;
    }
    // din = da * Wᵀ over the taps (simt_conv_kernel on the flipped kernel)
    int conv_input_grad(int i, const float* da, int k, int cin, int64_t R, float* din) {
        simt_conv_kernel<<<blocks_for(R * cin), kThreads, 0, st>>>(da, tr->convT[i].as<float>(), zeros(), nullptr, din, R,
                                                                   k, tr->C, cin, 0);
        CF_LAUNCHED();
        return CF_OK;
    }
    // gradients of conv i's kernel, bias, gamma and beta from dy at its BN output (act: the relu output, or nullptr)
    int conv_grads(int i, const float* dy, const float* act, const float* a, const float* in, int k, int cin, int64_t R,
                   float* da, float* g, float* gx) {
        const int C = tr->C;
        k12_bn_bwd_kernel<<<blocks_for(R * C), kThreads, 0, st>>>(dy, act, a, bn(i), tr->desc.bn_epsilon, C, R * C, da, g, gx);
        CF_LAUNCHED();
        CF_TRY(atb(ones(), 0, 0, g, C, R, 1, C, G(conv_tensor(i, 3)), C));
        CF_TRY(atb(ones(), 0, 0, gx, C, R, 1, C, G(conv_tensor(i, 2)), C));
        CF_TRY(atb(ones(), 0, 0, da, C, R, 1, C, G(conv_tensor(i, 1)), C));
        const int pad = (k - 1) / 2;
        for (int tap = 0; tap < k; ++tap)
            CF_TRY(atb(in, cin, tap - pad, da, C, R, cin, C, G(conv_tensor(i, 0)) + (int64_t)tap * cin * C, C));
        return CF_OK;
    }
};

// One forward + backward over n_windows windows: tr->grad holds dL/dvar (0 for the BN moving statistics) and
// tr->result (device) the loss sum and the number of hits.
int run_step(cf_trainer* tr, const float* x_dev, const uint8_t* labels, int64_t n_windows, float keep, uint64_t seed,
             int64_t step, cudaStream_t st) {
    Trainer T{tr, st};
    const int64_t tiles = ceil_div(n_windows, kTileWindows), R = tiles * kTileRows;
    const int C = tr->C, H = tr->H, nres = tr->n_res, nrnn = tr->n_rnn;
    const int64_t fmax = std::max<int64_t>(std::max(2 * H, C), 1);
    // workspace, in floats
    int64_t need = R;                                     // x
    need += (int64_t)nres * 9 * R * C;                    // per block: a0..a3, sc, ca, cb, o3, out
    need += (int64_t)nrnn * 12 * R * H;                   // per layer: gates, h, r*h, y
    if (nrnn) need += 6 * R * H * 2 + 2 * R * H;          // xproj, dpre, h_prev
    if (nres) need += 7 * R * C;                          // conv backward temporaries
    need += 2 * R * fmax + R;                             // gradient ping-pong, dL/dz
    CF_TRY(tr->ws.ensure(sizeof(float) * (size_t)need));
    CF_TRY(tr->partial.ensure(sizeof(float) * (size_t)kAtbPartialFloats));
    const unsigned head_blocks = blocks_for(R);
    CF_TRY(tr->loss_partial.ensure(sizeof(double) * 2 * head_blocks));
    CF_TRY(tr->result.ensure(sizeof(double) * 2));
    float* p = tr->ws.as<float>();
    auto take = [&](int64_t n) { float* q = p; p += n; return q; };
    float* xb = take(R);
    std::vector<float*> act(9 * (size_t)nres), gates(nrnn), hraw(nrnn), rh(nrnn), y(nrnn);
    for (auto& q : act) q = take(R * C);
    for (int l = 0; l < nrnn; ++l) { gates[l] = take(6 * R * H); hraw[l] = take(2 * R * H); rh[l] = take(2 * R * H); y[l] = take(2 * R * H); }
    float *xproj = nullptr, *dpre = nullptr, *hprev = nullptr;
    if (nrnn) { xproj = take(6 * R * H); dpre = take(6 * R * H); hprev = take(2 * R * H); }
    float* tmp[7] = {};
    if (nres) for (auto& q : tmp) q = take(R * C);
    float* dyA = take(R * fmax);
    float* dyB = take(R * fmax);
    float* dz = take(R);

    // input windows (the engines' own table and gather)
    const size_t slots = (size_t)tiles * kTileWindows;
    CF_TRY(tr->tab_src.ensure(slots * sizeof(int64_t)));
    CF_TRY(tr->tab_valid.ensure(slots * sizeof(int32_t)));
    CF_TRY(tr->tab_read.ensure(slots * sizeof(int32_t)));
    WindowTable tab{tr->tab_src.as<int64_t>(), tr->tab_valid.as<int32_t>(), tr->tab_read.as<int32_t>()};
    CF_TRY(k1_dense_window_table(n_windows, tiles, tab, st));
    CF_TRY(k1_fill_windows(nullptr, nullptr, x_dev, tab, 0, tiles, xb, st));

    Dropout drop{keep, (uint32_t)std::lround((double)keep * 16777216.0), (uint32_t)seed, (uint32_t)(seed >> 32),
                 (uint32_t)step};
    const float eps = tr->desc.bn_epsilon;

    // ---- forward: residual blocks
    const float* feat = xb;
    for (int b = 0; b < nres; ++b) {
        float** A = &act[9 * (size_t)b];      // a0 a1 a2 a3 sc ca cb o3 out
        const int cin = b ? C : 1, i = 4 * b;
        const int64_t tot = R * C;
        CF_TRY(T.conv(i, feat, 1, cin, R, A[0]));
        k12_bn_fwd_kernel<<<blocks_for(tot), kThreads, 0, st>>>(A[0], T.bn(i), eps, C, tot, 0, A[4], nullptr, nullptr);
        CF_LAUNCHED();
        CF_TRY(T.conv(i + 1, feat, 1, cin, R, A[1]));
        k12_bn_fwd_kernel<<<blocks_for(tot), kThreads, 0, st>>>(A[1], T.bn(i + 1), eps, C, tot, 1, A[5], nullptr, nullptr);
        CF_LAUNCHED();
        CF_TRY(T.conv(i + 2, A[5], 3, C, R, A[2]));
        k12_bn_fwd_kernel<<<blocks_for(tot), kThreads, 0, st>>>(A[2], T.bn(i + 2), eps, C, tot, 1, A[6], nullptr, nullptr);
        CF_LAUNCHED();
        CF_TRY(T.conv(i + 3, A[6], 1, C, R, A[3]));
        k12_bn_fwd_kernel<<<blocks_for(tot), kThreads, 0, st>>>(A[3], T.bn(i + 3), eps, C, tot, 1, A[7], A[4], A[8]);
        CF_LAUNCHED();
        feat = A[8];
    }
    // ---- forward: GRU stack
    const int feat_dim = nres ? C : 1;
    const size_t gru_smem_f = sizeof(float) * 2 * 32 * (H + 1);
    const size_t gru_smem_b = sizeof(float) * 32 * (3 * (H + 1) + 2 * H + 1);
    if (nrnn) {
        CF_CUDA(cudaFuncSetAttribute(k12_gru_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gru_smem_f));
        CF_CUDA(cudaFuncSetAttribute(k12_gru_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gru_smem_b));
    }
    auto gru_vars = [&](int l) {
        GruVars v;
        for (int d = 0; d < 2; ++d) {
            v.gk[d] = T.V(gru_tensor(tr, l, d, 0));
            v.gb[d] = T.V(gru_tensor(tr, l, d, 1));
            v.ck[d] = T.V(gru_tensor(tr, l, d, 2));
            v.cb[d] = T.V(gru_tensor(tr, l, d, 3));
        }
        return v;
    };
    for (int l = 0; l < nrnn; ++l) {
        const int fin = l ? 2 * H : feat_dim;
        const float* in = l ? y[l - 1] : feat;
        k12_pack_gru_kernel<<<blocks_for((int64_t)fin * 6 * H), kThreads, 0, st>>>(
            gru_vars(l), fin, H, tr->wx[l].as<float>(), tr->bx[l].as<float>(), tr->wxT[l].as<float>());
        CF_LAUNCHED();
        simt_gemm_bias_kernel<<<dim3((unsigned)ceil_div(R, 64), (unsigned)ceil_div(6 * H, 64)), 256, 0, st>>>(
            in, tr->wx[l].as<float>(), tr->bx[l].as<float>(), xproj, R, 6 * H, fin);
        CF_LAUNCHED();
        const GruVars v = gru_vars(l);
        k12_gru_fwd_kernel<<<dim3((unsigned)tiles, 4, 2), 256, gru_smem_f, st>>>(
            xproj, v.gk[0] + (int64_t)fin * 2 * H, v.ck[0] + (int64_t)fin * H, v.gk[1] + (int64_t)fin * 2 * H,
            v.ck[1] + (int64_t)fin * H, H, l, drop, gates[l], hraw[l], rh[l], y[l]);
        CF_LAUNCHED();
    }
    // ---- head + loss
    const int n_t = (int)tr->off.size();
    const int F = nrnn ? 2 * H : C;
    const float* yin = nrnn ? y[nrnn - 1] : feat;
    k12_head_loss_kernel<<<head_blocks, kThreads, 0, st>>>(yin, F, T.V(n_t - 2), T.V(n_t - 1), labels, n_windows, R,
                                                           1.f / (float)(n_windows * kWindow), dz,
                                                           tr->loss_partial.as<double>());
    CF_LAUNCHED();
    k12_loss_reduce_kernel<<<1, 1, 0, st>>>(tr->loss_partial.as<double>(), (int)head_blocks, tr->result.as<double>());
    CF_LAUNCHED();

    // ---- backward: head
    CF_CUDA(cudaMemsetAsync(tr->grad.ptr, 0, sizeof(float) * (size_t)tr->total, st));   // BN moving statistics stay 0
    CF_TRY(T.atb(yin, F, 0, dz, 1, R, F, 1, T.G(n_t - 2), 1));
    CF_TRY(T.atb(T.ones(), 0, 0, dz, 1, R, 1, 1, T.G(n_t - 1), 1));
    k12_head_bwd_kernel<<<blocks_for(R * F), kThreads, 0, st>>>(dz, T.V(n_t - 2), F, R * F, dyA);
    CF_LAUNCHED();
    float* dcur = dyA;     // gradient at the input of the head / of the layer above
    float* dnext = dyB;
    // ---- backward: GRU stack
    for (int l = nrnn - 1; l >= 0; --l) {
        const int fin = l ? 2 * H : feat_dim;
        const float* in = l ? y[l - 1] : feat;
        const GruVars v = gru_vars(l);
        k12_gru_bwd_kernel<<<dim3((unsigned)tiles, 4, 2), 256, gru_smem_b, st>>>(
            dcur, gates[l], hraw[l], v.gk[0] + (int64_t)fin * 2 * H, v.ck[0] + (int64_t)fin * H,
            v.gk[1] + (int64_t)fin * 2 * H, v.ck[1] + (int64_t)fin * H, H, l, drop, dpre, hprev);
        CF_LAUNCHED();
        for (int d = 0; d < 2; ++d) {
            const float* dg = dpre + d * 3 * H;         // dr_pre | du_pre, row stride 6H
            const float* dc = dg + 2 * H;               // dc_pre
            float* gk = T.G(gru_tensor(tr, l, d, 0));
            float* ck = T.G(gru_tensor(tr, l, d, 2));
            CF_TRY(T.atb(in, fin, 0, dg, 6 * H, R, fin, 2 * H, gk, 2 * H));
            CF_TRY(T.atb(hprev + d * H, 2 * H, 0, dg, 6 * H, R, H, 2 * H, gk + (int64_t)fin * 2 * H, 2 * H));
            CF_TRY(T.atb(in, fin, 0, dc, 6 * H, R, fin, H, ck, H));
            CF_TRY(T.atb(rh[l] + d * H, 2 * H, 0, dc, 6 * H, R, H, H, ck + (int64_t)fin * H, H));
            CF_TRY(T.atb(T.ones(), 0, 0, dg, 6 * H, R, 1, 2 * H, T.G(gru_tensor(tr, l, d, 1)), 2 * H));
            CF_TRY(T.atb(T.ones(), 0, 0, dc, 6 * H, R, 1, H, T.G(gru_tensor(tr, l, d, 3)), H));
        }
        if (l > 0 || nres > 0) {     // gradient of the layer input: dpre · Wxᵀ
            simt_gemm_bias_kernel<<<dim3((unsigned)ceil_div(R, 64), (unsigned)ceil_div(fin, 64)), 256, 0, st>>>(
                dpre, tr->wxT[l].as<float>(), T.zeros(), dnext, R, fin, 6 * H);
            CF_LAUNCHED();
            std::swap(dcur, dnext);
        }
    }
    // ---- backward: residual blocks
    for (int b = nres - 1; b >= 0; --b) {
        float** A = &act[9 * (size_t)b];
        const int cin = b ? C : 1, i = 4 * b;
        const float* in = b ? act[9 * (size_t)(b - 1) + 8] : xb;
        const int64_t tot = R * C;
        for (int j = 0; j < 4; ++j) {
            const int k = j == 2 ? 3 : 1, ci = j < 2 ? cin : C;
            k12_conv_flip_kernel<<<blocks_for((int64_t)k * ci * C), kThreads, 0, st>>>(T.V(conv_tensor(i + j, 0)), k, ci, C,
                                                                                     tr->convT[i + j].as<float>());
            CF_LAUNCHED();
        }
        float* ds = tmp[0];
        k12_relu_bwd_kernel<<<blocks_for(tot), kThreads, 0, st>>>(dcur, A[8], tot, ds);   // out = relu(o3 + sc)
        CF_LAUNCHED();
        // conv i+3 (o3 = relu(BN(a3)))
        CF_TRY(T.conv_grads(i + 3, ds, A[7], A[3], A[6], 1, C, R, tmp[1], tmp[2], tmp[3]));
        CF_TRY(T.conv_input_grad(i + 3, tmp[1], 1, C, R, tmp[4]));                        // d cb
        // shortcut conv i (sc = BN(a0))
        CF_TRY(T.conv_grads(i, ds, nullptr, A[0], in, 1, cin, R, tmp[5], tmp[2], tmp[3])); // tmp[5] = da0
        // conv i+2 (cb = relu(BN(a2)), k = 3)
        CF_TRY(T.conv_grads(i + 2, tmp[4], A[6], A[2], A[5], 3, C, R, tmp[1], tmp[2], tmp[3]));
        CF_TRY(T.conv_input_grad(i + 2, tmp[1], 3, C, R, tmp[6]));                        // d ca
        // conv i+1 (ca = relu(BN(a1)))
        CF_TRY(T.conv_grads(i + 1, tmp[6], A[5], A[1], in, 1, cin, R, tmp[1], tmp[2], tmp[3]));
        if (b > 0) {      // gradient of the block input: both branches
            CF_TRY(T.conv_input_grad(i + 1, tmp[1], 1, cin, R, tmp[2]));
            CF_TRY(T.conv_input_grad(i, tmp[5], 1, cin, R, tmp[3]));
            k12_add_kernel<<<blocks_for(R * cin), kThreads, 0, st>>>(tmp[2], tmp[3], R * cin, dnext);
            CF_LAUNCHED();
            std::swap(dcur, dnext);
        }
    }
    return CF_OK;
}

int check_run_args(cf_trainer* tr, const float* x, const uint8_t* labels, int64_t n, float keep, int64_t step,
                   const char* who) {
    if (!tr || !x || !labels || n < 1) { set_error("%s: bad argument", who); return CF_ERR_BAD_ARG; }
    if (!(keep > 0.f && keep <= 1.f)) { set_error("%s: keep_prob must be in (0, 1], got %g", who, keep); return CF_ERR_BAD_ARG; }
    if (step < 0 || step > (int64_t)0xffffffffLL) {
        set_error("%s: step must be in [0, 2^32), got %lld", who, (long long)step);
        return CF_ERR_BAD_ARG;
    }
    if (n > ((int64_t)1 << 31) / kWindow) { set_error("%s: too many windows (%lld)", who, (long long)n); return CF_ERR_BAD_ARG; }
    return CF_OK;
}

// Orders the call's work after the previous call on this trainer, and records the end of it on every path.
struct Ordered {
    cf_trainer* tr;
    cudaStream_t st;
    bool on = false;
    int enter() {
        CF_TRY(tr->last_done.create());
        CF_CUDA(cudaStreamWaitEvent(st, tr->last_done.ev, 0));
        on = true;
        return CF_OK;
    }
    ~Ordered() { if (on && cudaEventRecord(tr->last_done.ev, st) != cudaSuccess) cudaGetLastError(); }
};

int copy_out(cf_trainer* tr, const cf::DevBuf& buf, float* const* host, bool trainable_only) {
    for (size_t i = 0; i < tr->off.size(); ++i) {
        if (!host[i]) continue;
        const bool bn_stat = (int)i < 24 * tr->n_res && (i % 6 == 4 || i % 6 == 5);
        if (trainable_only && bn_stat) continue;
        CF_CUDA(cudaMemcpy(host[i], buf.as<float>() + tr->off[i], sizeof(float) * (size_t)tr->size[i], cudaMemcpyDeviceToHost));
    }
    return CF_OK;
}

}  // namespace
}  // namespace cf

// ================================================================== extern "C"
extern "C" {

int cf_trainer_create(const cf_model_desc* desc, const float* const* tensors, const int64_t* sizes, int32_t n_tensors,
                      const float* const* rms, const float* const* mom, int32_t device, cf_trainer** out) {
    if (!desc || !tensors || !sizes || !out) { cf::set_error("cf_trainer_create: NULL argument"); return CF_ERR_BAD_ARG; }
    *out = nullptr;
    std::vector<std::vector<int64_t>> shapes;
    CF_TRY(cf::expected_tensor_shapes(*desc, &shapes));
    if ((size_t)n_tensors != shapes.size()) {
        cf::set_error("cf_trainer_create: expected %zu tensors, got %d", shapes.size(), n_tensors);
        return CF_ERR_BAD_ARG;
    }
    std::unique_ptr<cf_trainer> tr(new cf_trainer());
    tr->desc = *desc;
    tr->device = device;
    tr->n_res = desc->network_type == CF_NET_RNN ? 0 : desc->n_layers_res;
    tr->n_rnn = desc->network_type == CF_NET_RESNET ? 0 : desc->n_layers;
    tr->C = tr->n_res ? desc->layer_size_res : 0;
    tr->H = tr->n_rnn ? desc->layer_size : 0;
    for (size_t i = 0; i < shapes.size(); ++i) {
        int64_t n = 1;
        for (int64_t v : shapes[i]) n *= v;
        const bool bn_stat = (int)i < 24 * tr->n_res && (i % 6 == 4 || i % 6 == 5);
        if (sizes[i] != n || !tensors[i] || (!bn_stat && ((rms && !rms[i]) || (mom && !mom[i])))) {
            cf::set_error("cf_trainer_create: tensor %zu has %lld elements (expected %lld) or a NULL entry", i,
                          (long long)sizes[i], (long long)n);
            return CF_ERR_BAD_ARG;
        }
        tr->off.push_back(tr->total);
        tr->size.push_back(n);
        tr->total += n;
    }
    std::vector<float> v((size_t)tr->total), m((size_t)tr->total, 1.f), p((size_t)tr->total, 0.f);
    std::vector<uint8_t> trainable((size_t)tr->total);
    for (size_t i = 0; i < shapes.size(); ++i) {
        const bool bn_stat = (int)i < 24 * tr->n_res && (i % 6 == 4 || i % 6 == 5);
        const size_t o = (size_t)tr->off[i], n = (size_t)tr->size[i];
        std::memcpy(&v[o], tensors[i], n * sizeof(float));
        std::fill(trainable.begin() + o, trainable.begin() + o + n, bn_stat ? 0 : 1);
        if (bn_stat) continue;
        if (rms) std::memcpy(&m[o], rms[i], n * sizeof(float));
        if (mom) std::memcpy(&p[o], mom[i], n * sizeof(float));
    }
    cf::Scope scope(tr.get());
    CF_TRY(scope.enter(device));
    CF_TRY(tr->var.upload(v));
    CF_TRY(tr->ms.upload(m));
    CF_TRY(tr->mom.upload(p));
    CF_TRY(tr->trainable.upload(trainable));
    CF_TRY(tr->grad.ensure(sizeof(float) * (size_t)tr->total));
    std::vector<float> consts(1 + cf::kZeros, 0.f);
    consts[0] = 1.f;
    CF_TRY(tr->consts.upload(consts));
    const int H = tr->H;
    for (int l = 0; l < tr->n_rnn; ++l) {
        const int fin = l ? 2 * H : (tr->n_res ? tr->C : 1);
        tr->wx.emplace_back();
        tr->bx.emplace_back();
        tr->wxT.emplace_back();
        CF_TRY(tr->wx.back().ensure(sizeof(float) * (size_t)fin * 6 * H));
        CF_TRY(tr->bx.back().ensure(sizeof(float) * 6 * (size_t)H));
        CF_TRY(tr->wxT.back().ensure(sizeof(float) * (size_t)fin * 6 * H));
    }
    for (int i = 0; i < 4 * tr->n_res; ++i) {
        tr->convT.emplace_back();
        CF_TRY(tr->convT.back().ensure(sizeof(float) * (size_t)tr->size[cf::conv_tensor(i, 0)]));
    }
    *out = tr.release();
    return CF_OK;
}

void cf_trainer_destroy(cf_trainer* tr) {
    if (!tr) return;
    {
        cf::Scope scope(tr);
        if (scope.enter(tr->device) != CF_OK) cudaSetDevice(tr->device);
        tr->last_done.sync();
    }
    delete tr;     // unlocked: a locked mutex must not be destroyed
}

int cf_trainer_step(cf_trainer* tr, const float* x_dev, const uint8_t* labels_dev, int64_t n_windows,
                    float learning_rate, float keep_prob, uint64_t seed, int64_t step, double* loss_out,
                    double* accuracy_out, void* stream) {
    CF_TRY(cf::check_run_args(tr, x_dev, labels_dev, n_windows, keep_prob, step, "cf_trainer_step"));
    if (!std::isfinite(learning_rate) || !(learning_rate > 0.f)) {
        cf::set_error("cf_trainer_step: learning_rate must be finite and > 0, got %g", learning_rate);
        return CF_ERR_BAD_ARG;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cf::Scope scope(tr);
    CF_TRY(scope.enter(tr->device));
    double host[2];
    {
        cf::Ordered ord{tr, st};
        CF_TRY(ord.enter());
        CF_TRY(cf::run_step(tr, x_dev, labels_dev, n_windows, keep_prob, seed, step, st));
        cf::k12_rmsprop_kernel<<<cf::blocks_for(tr->total), cf::kThreads, 0, st>>>(
            tr->var.as<float>(), tr->ms.as<float>(), tr->mom.as<float>(), tr->grad.as<float>(),
            tr->trainable.as<uint8_t>(), tr->total, learning_rate);
        CF_LAUNCHED();
        if (loss_out || accuracy_out) CF_CUDA(cudaMemcpyAsync(host, tr->result.ptr, sizeof(host), cudaMemcpyDeviceToHost, st));
    }
    if (loss_out || accuracy_out) {
        CF_CUDA(cudaStreamSynchronize(st));
        const double n = (double)(n_windows * cf::kWindow);
        if (loss_out) *loss_out = host[0] / n;
        if (accuracy_out) *accuracy_out = host[1] / n;
    }
    return CF_OK;
}

int cf_trainer_gradients(cf_trainer* tr, const float* x_dev, const uint8_t* labels_dev, int64_t n_windows,
                         float keep_prob, uint64_t seed, int64_t step, float* const* grads_host, double* loss_out,
                         void* stream) {
    CF_TRY(cf::check_run_args(tr, x_dev, labels_dev, n_windows, keep_prob, step, "cf_trainer_gradients"));
    if (!grads_host) { cf::set_error("cf_trainer_gradients: grads_host is NULL"); return CF_ERR_BAD_ARG; }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cf::Scope scope(tr);
    CF_TRY(scope.enter(tr->device));
    double host[2];
    {
        cf::Ordered ord{tr, st};
        CF_TRY(ord.enter());
        CF_TRY(cf::run_step(tr, x_dev, labels_dev, n_windows, keep_prob, seed, step, st));
        CF_CUDA(cudaMemcpyAsync(host, tr->result.ptr, sizeof(host), cudaMemcpyDeviceToHost, st));
    }
    CF_CUDA(cudaStreamSynchronize(st));
    CF_TRY(cf::copy_out(tr, tr->grad, grads_host, true));
    if (loss_out) *loss_out = host[0] / (double)(n_windows * cf::kWindow);
    return CF_OK;
}

int cf_trainer_read(cf_trainer* tr, float* const* tensors_host, float* const* rms_host, float* const* mom_host) {
    if (!tr || (!tensors_host && !rms_host && !mom_host)) { cf::set_error("cf_trainer_read: bad argument"); return CF_ERR_BAD_ARG; }
    cf::Scope scope(tr);
    CF_TRY(scope.enter(tr->device));
    CF_TRY(tr->last_done.sync());
    if (tensors_host) CF_TRY(cf::copy_out(tr, tr->var, tensors_host, false));
    if (rms_host) CF_TRY(cf::copy_out(tr, tr->ms, rms_host, true));
    if (mom_host) CF_TRY(cf::copy_out(tr, tr->mom, mom_host, true));
    return CF_OK;
}

}  // extern "C"
