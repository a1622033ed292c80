// K11: confusion counts at many thresholds from one pass over the scores (no reference counterpart; the
// reference's networks/precision_recall_ROC.py thresholds the same scores once per point of its curves).
//
// Per position, k = the number of thresholds t with (double)p >= t - the comparison of class_from_threshold
// (infer.py:128) and K9 - and the label class c (0, 1 or "any other value").  The count kernel adds one to
// hist[c][k] in a per-block shared-memory histogram and adds that histogram to a global int64 histogram with
// integer atomics (order-independent, hence deterministic).  A prediction at sorted threshold j is positive iff
// k > j, so one single-block scan turns the histogram into tp / fp / tn / fn at every threshold, with
// metrics.confusion_matrix's rule for labels other than 0 / 1 (as K9: a positive is a TP only for label 1, a
// negative a TN only for label 0).  NaN scores (reads with MAD = 0) satisfy no threshold: k = 0, predicted 0.
//
// The thresholds are held as floats: for a float p and a double t, (double)p >= t  <=>  p >= t', where t' is the
// smallest float >= t (k11_prepare_thresholds).  That halves the shared memory of the search and keeps every
// comparison exact.  HBM-bound for small T: 4 B score + 1 B label per position.
#include <algorithm>
#include <cmath>

#include "window_io.cuh"

namespace cf {

constexpr int kSweepThreads = 256;
constexpr int kSweepCountThreads = 1024;

__device__ __forceinline__ int sweep_key(float v, unsigned label, bool logits, const float* th, int T, int top) {
    const float p = logits ? head_sigmoid(v) : v;
    int k = 0;                                                // thresholds th[0..k) are <= p; NaN: none
    for (int step = top; step > 0; step >>= 1)
        if (k + step <= T && th[k + step - 1] <= p) k += step;
    const int c = label < 2u ? (int)label : 2;
    return c * (T + 1) + k;
}

// Lanes with equal keys add once (the scores of a read are mostly near 0: without aggregation a warp would
// serialise on one counter).  key < 0: no position.
__device__ __forceinline__ void sweep_add(unsigned* hist, int key) {
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    if (key >= 0 && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[key], (unsigned)__popc(peers));
}

// Dynamic shared memory: hist uint32 [3][T + 1] | thresholds float [T].  The loop runs a warp-uniform number of
// times (every lane reaches the __match_any_sync calls).  VEC: values 16-byte and labels 4-byte aligned.
template <bool VEC>
__global__ void __launch_bounds__(kSweepThreads)
k11_count_kernel(const float* __restrict__ values, const uint8_t* __restrict__ labels, int64_t n, int logits,
                 const float* __restrict__ thresholds, int T, unsigned long long* __restrict__ hist_out) {
    extern __shared__ unsigned sweep_smem[];
    const int nbins = 3 * (T + 1);
    unsigned* hist = sweep_smem;
    float* th = reinterpret_cast<float*>(sweep_smem + nbins);
    for (int i = threadIdx.x; i < nbins; i += kSweepThreads) hist[i] = 0;
    for (int i = threadIdx.x; i < T; i += kSweepThreads) th[i] = thresholds[i];
    __syncthreads();
    int top = 1;
    while (top * 2 <= T) top *= 2;
    const bool lg = logits != 0;
    const int lane = threadIdx.x & 31;
    const int64_t stride = (int64_t)gridDim.x * kSweepThreads * 4;
    for (int64_t wbase = ((int64_t)blockIdx.x * kSweepThreads + (threadIdx.x & ~31)) * 4; wbase < n; wbase += stride) {
        const int64_t base = wbase + lane * 4;
        float v[4];
        unsigned y[4];
        int m = 0;                                            // positions of this lane in this step
        if (VEC && base + 4 <= n) {
            const float4 z = *reinterpret_cast<const float4*>(values + base);
            const uchar4 l = *reinterpret_cast<const uchar4*>(labels + base);
            v[0] = z.x; v[1] = z.y; v[2] = z.z; v[3] = z.w;
            y[0] = l.x; y[1] = l.y; y[2] = l.z; y[3] = l.w;
            m = 4;
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                if (base + e < n) { v[e] = values[base + e]; y[e] = labels[base + e]; m = e + 1; }
            }
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) sweep_add(hist, e < m ? sweep_key(v[e], y[e], lg, th, T, top) : -1);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nbins; i += kSweepThreads)
        if (hist[i]) atomicAdd(&hist_out[i], (unsigned long long)hist[i]);
}

// One block: prefix sums P_c[k] = sum_{k' <= k} H_c[k'] of the three rows, then for sorted threshold j
//   tn = P_0[j], fn = P_1[j] + P_2[j], tp = N_1 - P_1[j], fp = N_0 + N_2 - P_0[j] - P_2[j].
// counts: int64 [T][4] = tp, fp, tn, fn in sorted-threshold order.
__global__ void __launch_bounds__(kSweepCountThreads)
k11_counts_kernel(const unsigned long long* __restrict__ hist, int T, long long* __restrict__ counts) {
    __shared__ long long warp_sum[kSweepCountThreads / 32][3];
    __shared__ long long total[3];
    const int nb = T + 1;
    const int per = (nb + kSweepCountThreads - 1) / kSweepCountThreads;
    const int b0 = threadIdx.x * per;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long s[3] = {0, 0, 0};
    for (int i = 0; i < per; ++i)
        if (b0 + i < nb)
            for (int c = 0; c < 3; ++c) s[c] += (long long)hist[c * nb + b0 + i];
    long long incl[3] = {s[0], s[1], s[2]};                   // inclusive scan over the warp
#pragma unroll
    for (int d = 1; d < 32; d <<= 1)
        for (int c = 0; c < 3; ++c) {
            const long long o = __shfl_up_sync(0xffffffffu, incl[c], d);
            if (lane >= d) incl[c] += o;
        }
    if (lane == 31)
        for (int c = 0; c < 3; ++c) warp_sum[warp][c] = incl[c];
    __syncthreads();
    if (threadIdx.x == 0) {                                   // exclusive scan of the 32 warp sums, in order
        long long run[3] = {0, 0, 0};
        for (int w = 0; w < kSweepCountThreads / 32; ++w)
            for (int c = 0; c < 3; ++c) { const long long t = warp_sum[w][c]; warp_sum[w][c] = run[c]; run[c] += t; }
        for (int c = 0; c < 3; ++c) total[c] = run[c];
    }
    __syncthreads();
    long long p[3];
    for (int c = 0; c < 3; ++c) p[c] = warp_sum[warp][c] + incl[c] - s[c];     // bins before this thread's
    for (int i = 0; i < per; ++i) {
        const int k = b0 + i;
        if (k >= T) break;                                    // bin T closes no threshold
        for (int c = 0; c < 3; ++c) p[c] += (long long)hist[c * nb + k];
        long long* out = counts + (size_t)k * 4;
        out[0] = total[1] - p[1];
        out[1] = total[0] + total[2] - p[0] - p[2];
        out[2] = p[0];
        out[3] = p[1] + p[2];
    }
}

int k11_prepare_thresholds(const double* thresholds, int n_thresholds, std::vector<float>* sorted,
                           std::vector<int>* index) {
    if (!thresholds || n_thresholds < 1 || n_thresholds > kSweepMaxThresholds) {
        set_error("threshold sweep: between 1 and %d thresholds, got %d", kSweepMaxThresholds, n_thresholds);
        return CF_ERR_BAD_ARG;
    }
    std::vector<int> order((size_t)n_thresholds);
    for (int i = 0; i < n_thresholds; ++i) {
        if (std::isnan(thresholds[i])) { set_error("threshold sweep: threshold %d is NaN", i); return CF_ERR_BAD_ARG; }
        order[i] = i;
    }
    std::sort(order.begin(), order.end(), [&](int a, int b) { return thresholds[a] < thresholds[b]; });
    sorted->clear();
    index->assign((size_t)n_thresholds, 0);
    for (int i : order) {
        const double t = thresholds[i];
        float f = (float)t;                                   // smallest float >= t (+-inf beyond the float range)
        if ((double)f < t) f = std::nextafter(f, INFINITY);
        if (sorted->empty() || sorted->back() != f) sorted->push_back(f);
        (*index)[i] = (int)sorted->size() - 1;
    }
    return CF_OK;
}

size_t k11_scratch_bytes(int n_thresholds) {
    return sizeof(unsigned long long) * 3 * ((size_t)n_thresholds + 1) + sizeof(long long) * 4 * (size_t)n_thresholds
           + sizeof(float) * (size_t)n_thresholds;
}

int k11_sweep(const float* values, bool values_are_logits, const uint8_t* labels, int64_t n,
              const std::vector<float>& thresholds, void* scratch, long long* counts_host, cudaStream_t stream) {
    const int T = (int)thresholds.size();
    unsigned long long* hist = static_cast<unsigned long long*>(scratch);
    long long* counts = reinterpret_cast<long long*>(hist + 3 * ((size_t)T + 1));
    float* th = reinterpret_cast<float*>(counts + 4 * (size_t)T);
    CF_CUDA(cudaMemcpyAsync(th, thresholds.data(), sizeof(float) * T, cudaMemcpyHostToDevice, stream));
    CF_CUDA(cudaMemsetAsync(hist, 0, sizeof(unsigned long long) * 3 * ((size_t)T + 1), stream));
    if (n > 0) {
        const bool vec = reinterpret_cast<uintptr_t>(values) % 16 == 0 && reinterpret_cast<uintptr_t>(labels) % 4 == 0;
        auto kernel = vec ? k11_count_kernel<true> : k11_count_kernel<false>;
        const size_t smem = sizeof(unsigned) * 3 * ((size_t)T + 1) + sizeof(float) * T;
        CF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int dev = 0, sms = 0, per_sm = 0;
        CF_CUDA(cudaGetDevice(&dev));
        CF_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        CF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kSweepThreads, smem));
        // K9's grid, cut to the blocks that fit at once; a block counts at most 2^30 positions (uint32 counters)
        int64_t blocks = std::min<int64_t>(k9_validation_blocks(n), (int64_t)std::max(per_sm, 1) * sms);
        blocks = std::max<int64_t>(blocks, ceil_div(n, (int64_t)1 << 30));
        kernel<<<(unsigned)blocks, kSweepThreads, smem, stream>>>(values, labels, n, values_are_logits ? 1 : 0, th, T,
                                                                  hist);
        CF_LAUNCHED();
    }
    k11_counts_kernel<<<1, kSweepCountThreads, 0, stream>>>(hist, T, counts);
    CF_LAUNCHED();
    CF_CUDA(cudaMemcpyAsync(counts_host, counts, sizeof(long long) * 4 * (size_t)T, cudaMemcpyDeviceToHost, stream));
    return CF_OK;
}

}  // namespace cf
