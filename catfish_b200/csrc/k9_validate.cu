// K9 ("next" row N4 of SURVEY section 8f): the counting half of the validation path.
//
// Replaces, for one call of RNN.test_network (networks/rnn_class.py:222-261):
//   pred_vals = [1 if c >= threshold else 0 for c in confidences]            (:235)
//   accuracy  = mean(round(sigmoid(logits)) == y)                            (:80-86, tf.round = half to even)
//   loss      = mean(sigmoid_cross_entropy(y, logits))                       (:72-77)
//   confusion_matrix(test_labels, pred_vals)                                 (networks/trainingDB/metrics.py:10-37)
// over ALL n = n_windows * 35 positions, padding included (the reference subtracts padding_size
// from the true negatives afterwards, rnn_class.py:247 - the caller of this kernel does the same).
//
// Input is the dense layer's output (logits) that the forward pass leaves in HBM when asked to
// skip the sigmoid; the probability is recomputed here with the heads' own function (head_sigmoid) so that
// predictions are bit-identical to cf_infer_windows.  HBM-bound: 4 B logit + 1 B label per position.
// Deterministic: every block reduces in a fixed order into its own slot, one block adds the slots.
#include "window_io.cuh"

namespace cf {

constexpr int kValThreads = 256;
constexpr int kValFields = 6;        // tp, fp, tn, fn, correct, (loss as double bits)

struct ValAcc {
    long long tp = 0, fp = 0, tn = 0, fn = 0, correct = 0;
    double loss = 0.0;
};

__device__ __forceinline__ void val_accumulate(ValAcc& a, float z, unsigned label, double threshold) {
    const float p = head_sigmoid(z);
    const bool pred = (double)p >= threshold;
    // metrics.confusion_matrix: a predicted 1 is a TP only for label 1, a predicted 0 is a TN only
    // for label 0; any other label value lands in fp / fn
    if (pred) { if (label == 1u) ++a.tp; else ++a.fp; }
    else      { if (label == 0u) ++a.tn; else ++a.fn; }
    const float y = (float)label;
    if (rintf(p) == y) ++a.correct;
    // tf.nn.sigmoid_cross_entropy_with_logits: max(z, 0) - z*y + log(1 + exp(-|z|)), fp32 per element
    const float l = fmaxf(z, 0.f) - z * y + log1pf(expf(-fabsf(z)));
    a.loss += (double)l;
}

__device__ __forceinline__ void val_block_reduce(ValAcc& a, long long* out_i, double* out_d) {
    __shared__ long long si[kValThreads / 32][5];
    __shared__ double sd[kValThreads / 32];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        a.tp += __shfl_down_sync(0xffffffffu, a.tp, d);
        a.fp += __shfl_down_sync(0xffffffffu, a.fp, d);
        a.tn += __shfl_down_sync(0xffffffffu, a.tn, d);
        a.fn += __shfl_down_sync(0xffffffffu, a.fn, d);
        a.correct += __shfl_down_sync(0xffffffffu, a.correct, d);
        a.loss += __shfl_down_sync(0xffffffffu, a.loss, d);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
        si[warp][0] = a.tp; si[warp][1] = a.fp; si[warp][2] = a.tn; si[warp][3] = a.fn; si[warp][4] = a.correct;
        sd[warp] = a.loss;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        long long t[5] = {0, 0, 0, 0, 0};
        double l = 0.0;
        for (int w = 0; w < kValThreads / 32; ++w) {
            for (int k = 0; k < 5; ++k) t[k] += si[w][k];
            l += sd[w];
        }
        for (int k = 0; k < 5; ++k) out_i[k] = t[k];
        *out_d = l;
    }
}

// partial: [gridDim.x][kValFields] as 8-byte slots (5 x int64 + 1 x double)
__global__ void __launch_bounds__(kValThreads)
k9_count_kernel(const float* __restrict__ logits, const uint8_t* __restrict__ labels, int64_t n, double threshold,
                long long* __restrict__ partial) {
    ValAcc a;
    const int64_t stride = (int64_t)gridDim.x * kValThreads * 4;
    for (int64_t base = ((int64_t)blockIdx.x * kValThreads + threadIdx.x) * 4; base < n; base += stride) {
        if (base + 4 <= n) {
            const float4 z = *reinterpret_cast<const float4*>(logits + base);
            const uchar4 y = *reinterpret_cast<const uchar4*>(labels + base);
            val_accumulate(a, z.x, y.x, threshold);
            val_accumulate(a, z.y, y.y, threshold);
            val_accumulate(a, z.z, y.z, threshold);
            val_accumulate(a, z.w, y.w, threshold);
        } else {
            for (int64_t i = base; i < n; ++i) val_accumulate(a, logits[i], labels[i], threshold);
        }
    }
    long long* slot = partial + (size_t)blockIdx.x * kValFields;
    val_block_reduce(a, slot, reinterpret_cast<double*>(slot + 5));
}

// result: tp, fp, tn, fn, correct (int64) | loss sum (double)
__global__ void k9_final_kernel(const long long* __restrict__ partial, int n_blocks, long long* __restrict__ result) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    long long t[5] = {0, 0, 0, 0, 0};
    double l = 0.0;
    for (int b = 0; b < n_blocks; ++b) {
        const long long* slot = partial + (size_t)b * kValFields;
        for (int k = 0; k < 5; ++k) t[k] += slot[k];
        l += *reinterpret_cast<const double*>(slot + 5);
    }
    for (int k = 0; k < 5; ++k) result[k] = t[k];
    *reinterpret_cast<double*>(result + 5) = l;
}

int k9_validation_blocks(int64_t n) {
    const int64_t want = ceil_div(n, (int64_t)kValThreads * 4);
    return (int)(want < 1 ? 1 : (want > 592 ? 592 : want));      // 4 CTAs per SM on 148 SMs
}

int k9_validate(const float* logits, const uint8_t* labels, int64_t n, double threshold, long long* partial,
                long long* result, cudaStream_t stream) {
    const int blocks = k9_validation_blocks(n);
    k9_count_kernel<<<blocks, kValThreads, 0, stream>>>(logits, labels, n, threshold, partial);
    CF_LAUNCHED();
    k9_final_kernel<<<1, 32, 0, stream>>>(partial, blocks, result);
    CF_LAUNCHED();
    return CF_OK;
}

// ====================================================================== K10: event voting (row N3)
// Replaces the arithmetic of correct_events (networks/correct_output.py:38-61): the mean score of
// the measurements that belong to an event, rounded half-to-even, for the events the reference's
// loop visits.  The event range is derived by the caller from the scanned lengths; one thread per
// event adds its scores in order with the compensated (Neumaier) summation CPython's sum() uses
// for floats, so the averages - and therefore ties at 0.5 - are those of the reference.
__global__ void k10_vote_kernel(const double* __restrict__ scores, int64_t n_scores,
                                const int64_t* __restrict__ ev_begin, int64_t first_event, int64_t n_voted,
                                int32_t* __restrict__ classes, int32_t* __restrict__ empty_flag) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_voted) return;
    int64_t b = ev_begin[first_event + i], e = ev_begin[first_event + i + 1];
    // python slice clamping of scores[b:e]
    b = b < n_scores ? b : n_scores;
    e = e < n_scores ? e : n_scores;
    if (e <= b) { atomicExch(empty_flag, 1); classes[i] = 0; return; }
    double s = scores[b], c = 0.0;
    for (int64_t k = b + 1; k < e; ++k) {
        const double x = scores[k];
        const double t = s + x;
        if (fabs(s) >= fabs(x)) c += (s - t) + x; else c += (x - t) + s;
        s = t;
    }
    if (c != 0.0 && isfinite(c)) s += c;
    const double avg = s / (double)(e - b);
    classes[i] = (int32_t)rint(avg);
}

int k10_vote_events(const double* scores, int64_t n_scores, const int64_t* ev_begin, int64_t first_event,
                    int64_t n_voted, int32_t* classes, int32_t* empty_flag, cudaStream_t stream) {
    CF_CUDA(cudaMemsetAsync(empty_flag, 0, sizeof(int32_t), stream));
    if (n_voted > 0) {
        k10_vote_kernel<<<(unsigned)ceil_div(n_voted, (int64_t)256), 256, 0, stream>>>(
            scores, n_scores, ev_begin, first_event, n_voted, classes, empty_flag);
        CF_LAUNCHED();
    }
    return CF_OK;
}

}  // namespace cf
