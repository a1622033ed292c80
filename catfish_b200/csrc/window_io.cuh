// The per-sample rules every forward pass shares: what a window's input sample is, and what a head makes of one
// output logit.  Both engines' kernels read and write samples only through these, so that their inputs agree bit for
// bit and the validation kernels (K9, K11) recompute exactly the probabilities the heads write.
#pragma once

#include "common.cuh"

namespace cf {

// ---------------------------------------------------------------- input: one window's samples
// Sample t of the window = t < valid ? float((raw[src + t] - shift) / scale) : 0 with the read's (shift, scale) in
// fp64 (infer.py:32-38,105; the f64 -> f32 cast is the placeholder feed of rnn_class.py:159), or xwin[src + t] for
// already-normalised windows (raw == nullptr).
struct WindowInput {
    const int16_t* raw;
    const float* xwin;
    int valid;
    int64_t src;
    double shift, scale;
    __device__ __forceinline__ float operator()(int t) const {
        float v = 0.f;
        if (t < valid) v = raw ? (float)(((double)raw[src + t] - shift) / scale) : xwin[src + t];
        return v;
    }
};

__device__ __forceinline__ WindowInput window_input(const int16_t* raw, const double* stats, const float* xwin,
                                                    const int64_t* src, const int32_t* valid, const int32_t* read,
                                                    int64_t g) {
    WindowInput w{raw, xwin, valid[g], src[g], 0.0, 1.0};
    if (raw && w.valid > 0) { const int r = read[g]; w.shift = stats[2 * r]; w.scale = stats[2 * r + 1]; }
    return w;
}

// ---------------------------------------------------------------- output: one head sample
// The dense layer's sigmoid (rnn_class.py:84).
__device__ __forceinline__ float head_sigmoid(float z) { return 1.f / (1.f + expf(-z)); }

// Where a head writes its samples.
struct HeadOut {
    const int64_t* src;
    const int32_t* valid;
    const int32_t* read;
    const double* stats;      // per-read (shift, scale) of raw input; nullptr for normalised windows
    float* probs;             // nullptr: no probabilities
    unsigned* lwords;         // nullptr: no label bits (LabelBits::lwords, zeroed by k6_bits_prepare)
    double threshold;
    int want_logits;          // probs receives the logit (the validation row's loss needs it)
};

// Sample t of window g with logit z: p = sigmoid(z) (or z with want_logits), NaN when the read's scale is not > 0
// (the reference divides by it), written to probs[src[g] + t]; its label bit is (double)p >= threshold, the f32
// score widened to double as class_from_threshold does (infer.py:128-138), NaN giving 0.  `real`: t is one of the
// window's valid samples (the padding is cut, infer.py:47); other lanes write nothing.
// All 32 lanes of the warp must call it.  Consecutive lanes hold consecutive samples, so a warp touches at most a
// few label words: lanes of one word OR their bits together and one of them issues the atomic.
__device__ __forceinline__ void head_output(const HeadOut& o, int64_t g, int t, bool real, float z) {
    float p = o.want_logits ? z : head_sigmoid(z);
    int64_t s = 0;
    if (real) {
        s = o.src[g] + t;
        if (o.stats && !(o.stats[2 * o.read[g] + 1] > 0.0)) p = nanf("");
        if (o.probs) o.probs[s] = p;
    }
    if (!o.lwords) return;
    const bool hit = real && (double)p >= o.threshold;
    const unsigned hits = __ballot_sync(0xffffffffu, hit);
    if (hit) {
        const unsigned peers = __match_any_sync(hits, (unsigned long long)(s >> 5));
        const unsigned bits = __reduce_or_sync(peers, 1u << (s & 31));
        if ((threadIdx.x & 31) == __ffs(peers) - 1) atomicOr(&o.lwords[s >> 5], bits);
    }
}

}  // namespace cf
