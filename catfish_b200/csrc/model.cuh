// Model handle: folded / re-packed weights.  The engines own only what is read-only after creation; the
// workspace a forward pass writes belongs to the caller's execution context and is passed in.
#pragma once

#include <memory>
#include <vector>

#include "common.cuh"

namespace cf {

// One conv layer with the inference batch-norm folded in (resnet_class.py:60-76):
//   y = conv(x) * s + (beta - mean * s),  s = gamma / sqrt(var + eps)
struct ConvLayer {
    int k = 1, cin = 1, cout = 1;
    std::vector<float> w;   // [k][cin][cout]
    std::vector<float> b;   // [cout]
};

// One GRU direction (tf.contrib.rnn.GRUCell, rnn_class.py:146) split into the part that
// multiplies the layer input x and the part that multiplies the state h.
struct GruDir {
    int in = 0, h = 0;
    std::vector<float> wx;  // [in][3h]   columns: r | u | c
    std::vector<float> bx;  // [3h]       gates bias (r|u) then candidate bias
    std::vector<float> wgh; // [h][2h]    state rows of gates/kernel
    std::vector<float> wch; // [h][h]     state rows of candidate/kernel
};

struct HostModel {
    cf_model_desc desc{};
    std::vector<ConvLayer> convs;          // 4 per residual block: shortcut, k1, k3, k1
    std::vector<GruDir> gru;               // [layer][dir] flattened: 2*layer + dir
    std::vector<float> head_w;             // [F]
    float head_b = 0.f;
    int conv_channels() const { return desc.layer_size_res; }
    int feat_after_conv() const {
        return desc.network_type == CF_NET_RNN ? 1 : desc.layer_size_res;
    }
    int head_features() const {
        return desc.network_type == CF_NET_RESNET ? desc.layer_size_res : 2 * desc.layer_size;
    }
    int n_res() const { return desc.network_type == CF_NET_RNN ? 0 : desc.n_layers_res; }
    int n_rnn() const { return desc.network_type == CF_NET_RESNET ? 0 : desc.n_layers; }
};

int expected_tensor_shapes(const cf_model_desc& d, std::vector<std::vector<int64_t>>* shapes);
int build_host_model(const cf_model_desc& d, const float* const* tensors, HostModel* out);

// An engine owns its weights; each engine's source defines how one is deleted.
struct SimtEngine;
struct TcEngine;
struct EngineDelete {
    void operator()(SimtEngine* e) const;
    void operator()(TcEngine* e) const;
};
using SimtEnginePtr = std::unique_ptr<SimtEngine, EngineDelete>;
using TcEnginePtr = std::unique_ptr<TcEngine, EngineDelete>;

// ---------------------------------------------------------------- SIMT (fp32) engine
// Uploads the weights; CF_ERR_ALLOC / CF_ERR_CUDA when an allocation / a copy fails.
int simt_create(const HostModel& hm, SimtEnginePtr* out);
// Forward pass over n_tiles tiles of 128 windows.  Input is either the raw int16 signal with
// per-read (shift, scale) or already-normalised float windows; output probabilities are
// scattered to probs[tab.src[g] + t] for t < tab.valid[g].  With want_logits the dense layer's output
// (rnn_class.py:178-183) is written instead of its sigmoid - the validation row needs it for the loss.
// ws: the calling context's workspace, grown to the pass's needs.
int simt_forward(SimtEngine* e, DevBuf* ws, const HostModel& hm, const int16_t* raw, const double* stats,
                 const float* xwin, WindowTable tab, int64_t n_tiles, float* probs,
                 cudaStream_t stream, Profiler* prof, bool want_logits = false);

// Grow ws to what simt_forward needs for a pass over n_tiles tiles.
int simt_reserve(DevBuf* ws, const HostModel& hm, int64_t n_tiles);
// Grow ws to what simt_conv_stack needs for passes of chunk_tiles tiles (the tensor-core engine's RNN-only input).
int simt_conv_stack_reserve(DevBuf* ws, const HostModel& hm, int64_t chunk_tiles);

// ---------------------------------------------------------------- tcgen05 engine
bool tc_supported(const HostModel& hm);
// Sets the kernels' attributes and uploads the weights; CF_ERR_ALLOC / CF_ERR_CUDA when an allocation / a CUDA call
// fails.
int tc_create(const HostModel& hm, TcEnginePtr* out);
int tc_operand_format(const TcEngine* e);    // 0 = split bf16 (3 MMA passes), 1 = fp16 + e5m2 corrections (2 pass-equivalents)
// bits != nullptr (networks with a GRU head): the head thresholds its own scores and ORs label bits into
// bits->lwords (k6_bits_prepare) instead of writing probabilities - probs may then be nullptr.
bool tc_can_emit_bits(const TcEngine* e);
// ws: the calling context's tensor-core workspace; simt_ws: its CUDA-core workspace (RNN-only networks normalise
// their scalar input with simt_conv_stack).  Both grow to the pass's needs.
int tc_forward(TcEngine* e, DevBuf* ws, DevBuf* simt_ws, const HostModel& hm, const int16_t* raw, const double* stats,
               const float* xwin, WindowTable tab, int64_t n_tiles, float* probs,
               cudaStream_t stream, Profiler* prof, bool want_logits = false, const LabelBits* bits = nullptr);

// Grow ws / simt_ws to what tc_forward needs for a pass over n_tiles tiles.
int tc_reserve(const TcEngine* e, DevBuf* ws, DevBuf* simt_ws, const HostModel& hm, int64_t n_tiles);

int tc_selftest_f16e5(const float* a_dev, int K, int N, const float* w_host, int mode, float* out_dev, cudaStream_t stream);

}  // namespace cf
