// K6: threshold -> short-run removal -> extended intervals, for a ragged batch of reads.
//
// Replaces the three Python loops after the network call in infer_class_from_signal
// (catfish/infer.py:47-49):
//     labels = correct_short(class_from_threshold(scores))     infer.py:128-138, 174-198
//     predicted_hps = hp_in_pred(labels)                       infer.py:141-162
// Net effect: every maximal run of positions with score >= threshold whose length is
// >= min_run (15) yields [start - ext_left (11), start + len + ext_right (16)], in read-local
// coordinates, unclamped, unmerged, ordered by start.  Runs never span two reads.
//
// Bit-parallel formulation over the concatenated sample index space:
//   L word  : label bits, ORed in by the network's head kernel (tc_engine.cu) or written by
//             k6_pack_bits from values in memory (warp ballot / nibble merge of 128-bit loads)
//   B word  : read-start bits (k1_window_table, or k6_read_starts from the offsets)
//   S word  : run-start bits  S = L & (~(L << 1 | carry) | B), evaluated where needed, not stored
//   run ends: E = L & (~(L >> 1 | next) | B >> 1); the start of the run ending at e is the
//             nearest S bit at or below e (scan S words backwards).
// Output order is the global rank of the run (count -> exclusive scan -> emit), so the
// result is deterministic and bit-exact against the reference's integer output.
#include "common.cuh"

namespace cf {

__device__ __forceinline__ int find_read(const int64_t* __restrict__ off, int n, int64_t i) {
    int lo = 0, hi = n;
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (off[mid] <= i) lo = mid; else hi = mid;
    }
    return lo;
}

// ---------------------------------------------------------------- read-start bits
__global__ void k6_bounds_kernel(const int64_t* __restrict__ offsets, int n_reads, int64_t total,
                                 unsigned* __restrict__ bwords) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_reads) return;
    const int64_t o = offsets[r];
    if (o < total && offsets[r + 1] > o) atomicOr(&bwords[o >> 5], 1u << (o & 31));
}

int k6_read_starts(const int64_t* offsets_dev, int32_t n_reads, int64_t total_samples, const LabelBits& bits,
                   cudaStream_t stream) {
    if (n_reads <= 0) return CF_OK;
    k6_bounds_kernel<<<(unsigned)ceil_div(n_reads, 256), 256, 0, stream>>>(offsets_dev, n_reads, total_samples, bits.bwords);
    CF_LAUNCHED();
    return CF_OK;
}

// ---------------------------------------------------------------- label bits from values in memory
template <int SRC> struct Src;
template <> struct Src<BITS_FROM_F32> {
    typedef float T;
    static __device__ __forceinline__ bool hit(float v, double thr, int64_t) { return (double)v >= thr; }
};
template <> struct Src<BITS_FROM_F64> {
    typedef double T;
    static __device__ __forceinline__ bool hit(double v, double thr, int64_t) { return v >= thr; }
};
template <> struct Src<BITS_FROM_I64_EQ> {
    typedef int64_t T;
    static __device__ __forceinline__ bool hit(int64_t v, double, int64_t label) { return v == label; }
};

// Generic path: one warp per 32-sample word per iteration, ballot.
template <int SRC>
__global__ void k6_pack_kernel(const typename Src<SRC>::T* __restrict__ vals, int64_t n, double thr,
                               int64_t label, int64_t n_words, unsigned* __restrict__ lwords) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t w = warp; w < n_words; w += n_warps) {
        const int64_t i = (w << 5) + lane;
        const bool h = i < n && Src<SRC>::hit(vals[i], thr, label);
        const unsigned L = __ballot_sync(0xffffffffu, h);
        if (lane == 0) lwords[w] = L;
    }
}

// f32 fast path: each lane loads 4 consecutive probabilities (128-bit), 8 lanes form a word; four
// independent 128-sample groups per warp iteration keep 4 loads per thread in flight (HBM-bound).
__global__ void __launch_bounds__(256)
k6_pack_f32x4_kernel(const float* __restrict__ vals, int64_t n, double thr,
                     int64_t n_words, unsigned* __restrict__ lwords) {
    constexpr int kUnroll = 4;
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t n_groups = (n_words + 3) >> 2;           // 128 samples per group
    const float thr_f = (float)thr;
    const bool thr_exact = (double)thr_f == thr;           // then the fp32 compare equals the fp64 one
    for (int64_t g0 = warp * kUnroll; g0 < n_groups; g0 += n_warps * kUnroll) {
        float4 v[kUnroll];
#pragma unroll
        for (int k = 0; k < kUnroll; ++k) {
            const int64_t i = ((g0 + k) << 7) + (lane << 2);
            v[k] = make_float4(-1.f, -1.f, -1.f, -1.f);
            if (i + 3 < n) {
                v[k] = __ldcs(reinterpret_cast<const float4*>(vals + i));
            } else if (i < n) {
                float t[4] = {-1.f, -1.f, -1.f, -1.f};
                for (int j = 0; j < 4; ++j)
                    if (i + j < n) t[j] = vals[i + j];
                v[k] = make_float4(t[0], t[1], t[2], t[3]);
            }
        }
#pragma unroll
        for (int k = 0; k < kUnroll; ++k) {
            const int64_t g = g0 + k;
            if (g >= n_groups) break;
            const int64_t i = (g << 7) + (lane << 2);
            unsigned nib;
            if (thr_exact) {
                nib = (v[k].x >= thr_f ? 1u : 0u) | (v[k].y >= thr_f ? 2u : 0u) | (v[k].z >= thr_f ? 4u : 0u) | (v[k].w >= thr_f ? 8u : 0u);
            } else {
                nib = ((double)v[k].x >= thr ? 1u : 0u) | ((double)v[k].y >= thr ? 2u : 0u) |
                      ((double)v[k].z >= thr ? 4u : 0u) | ((double)v[k].w >= thr ? 8u : 0u);
            }
            // positions past the end were filled with -1: mask them for thresholds <= -1
            if (i + 3 >= n) {
                unsigned m = 0;
                for (int j = 0; j < 4; ++j)
                    if (i + j < n) m |= 1u << j;
                nib &= m;
            }
            unsigned L = nib << ((lane & 7) << 2);
            L |= __shfl_xor_sync(0xffffffffu, L, 1);
            L |= __shfl_xor_sync(0xffffffffu, L, 2);
            L |= __shfl_xor_sync(0xffffffffu, L, 4);
            const int64_t w = (g << 2) + (lane >> 3);
            if ((lane & 7) == 0 && w < n_words) lwords[w] = L;
        }
    }
}

int k6_pack_bits(const void* values, int source, double threshold, int64_t label, int64_t n, const LabelBits& bits,
                 cudaStream_t stream) {
    const int64_t n_words = ceil_div(n, 32);
    int64_t pack_blocks = ceil_div(n_words, 8 * 16);  // 8 warps per block, 16 words per warp iteration
    if (pack_blocks < 1) pack_blocks = 1;
    if (pack_blocks > 148 * 8) pack_blocks = 148 * 8;
    if (source == BITS_FROM_F32) {
        if ((reinterpret_cast<uintptr_t>(values) & 15) == 0) {
            k6_pack_f32x4_kernel<<<(unsigned)pack_blocks, 256, 0, stream>>>(
                static_cast<const float*>(values), n, threshold, n_words, bits.lwords);
        } else {
            k6_pack_kernel<BITS_FROM_F32><<<(unsigned)pack_blocks, 256, 0, stream>>>(
                static_cast<const float*>(values), n, threshold, label, n_words, bits.lwords);
        }
    } else if (source == BITS_FROM_F64) {
        k6_pack_kernel<BITS_FROM_F64><<<(unsigned)pack_blocks, 256, 0, stream>>>(
            static_cast<const double*>(values), n, threshold, label, n_words, bits.lwords);
    } else {
        k6_pack_kernel<BITS_FROM_I64_EQ><<<(unsigned)pack_blocks, 256, 0, stream>>>(
            static_cast<const int64_t*>(values), n, threshold, label, n_words, bits.lwords);
    }
    CF_LAUNCHED();
    return CF_OK;
}

// ---------------------------------------------------------------- runs: count / emit
// S words are not stored: S[w] = L[w] & (~(L[w] << 1 | L[w-1] >> 31) | B[w]).
__device__ __forceinline__ unsigned start_word(const unsigned* __restrict__ lwords, const unsigned* __restrict__ bwords, int64_t w) {
    const unsigned L = lwords[w];
    const unsigned carry = w > 0 ? lwords[w - 1] >> 31 : 0u;
    return L & (~((L << 1) | carry) | bwords[w]);
}
__device__ __forceinline__ int64_t run_start_lb(const unsigned* __restrict__ lwords, const unsigned* __restrict__ bwords, int64_t w, int eb) {
    unsigned s = start_word(lwords, bwords, w) & (eb == 31 ? 0xffffffffu : ((2u << eb) - 1u));
    while (s == 0) {
        --w;
        s = start_word(lwords, bwords, w);
    }
    return (w << 5) + (31 - __clz(s));
}

// Count (EMIT = false): qualifying run ends per block; the LAST block to finish scans the block counts into
// block_base (so no separate scan launch).  Emit (EMIT = true): intervals in global rank order.
// A thread owns kBitsWordsPerThread consecutive words (one 128-bit load each of the label and boundary words):
// with one word per thread the 2e6 words of a 512-read batch were 7 waves of 256-thread blocks, each a
// load -> look-back -> block scan latency chain (39 us per launch for 8 MB of bits).
constexpr int kBitsThreads = 256, kBitsWordsPerThread = 4, kBitsWordsPerBlock = kBitsThreads * kBitsWordsPerThread;
template <bool EMIT>
__global__ void __launch_bounds__(kBitsThreads)
k6_runs_bits_kernel(const unsigned* __restrict__ lwords, const unsigned* __restrict__ bwords, int64_t n_words,
                    const int64_t* __restrict__ offsets, int n_reads, int min_run, int ext_left, int ext_right,
                    unsigned* __restrict__ block_cnt, int64_t* __restrict__ block_base, unsigned* __restrict__ done_counter,
                    int64_t* __restrict__ run_start_global, int64_t* __restrict__ intervals, int64_t capacity) {
    __shared__ unsigned warp_sums[kBitsThreads / 32];
    __shared__ long long scan_sums[kBitsThreads / 32];
    __shared__ long long scan_carry;
    __shared__ int is_last;
    constexpr int W = kBitsWordsPerThread;
    const int64_t w0 = ((int64_t)blockIdx.x * kBitsThreads + threadIdx.x) * W;
    unsigned L[W + 1], B[W + 1];                // this thread's words and the one after them (for the carry bits)
    if (w0 + W < n_words) {                      // both arrays are 16-byte aligned and hold n_words + 1 words
        const uint4 l4 = *reinterpret_cast<const uint4*>(lwords + w0), b4 = *reinterpret_cast<const uint4*>(bwords + w0);
        L[0] = l4.x; L[1] = l4.y; L[2] = l4.z; L[3] = l4.w; L[W] = lwords[w0 + W];
        B[0] = b4.x; B[1] = b4.y; B[2] = b4.z; B[3] = b4.w; B[W] = bwords[w0 + W];
    } else {
#pragma unroll
        for (int j = 0; j <= W; ++j) {
            const bool in = w0 + j < n_words;
            L[j] = in ? lwords[w0 + j] : 0u;
            B[j] = in ? bwords[w0 + j] : 0u;
        }
    }
    unsigned qual[W];
    int64_t starts[4];
    int nq = 0;
#pragma unroll
    for (int j = 0; j < W; ++j) {
        // run ends: a set label bit whose successor is clear or starts another read
        const unsigned E = L[j] & (~((L[j] >> 1) | ((L[j + 1] & 1u) << 31)) | (B[j] >> 1) | ((B[j + 1] & 1u) << 31));
        qual[j] = 0;
        for (unsigned e = E; e; e &= e - 1) {
            const int eb = __ffs(e) - 1;
            const int64_t s = run_start_lb(lwords, bwords, w0 + j, eb);
            const int64_t len = ((w0 + j) << 5) + eb - s + 1;
            if (len >= min_run) {
                qual[j] |= 1u << eb;
                if (nq < 4) starts[nq] = s;
                ++nq;
            }
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned inc = (unsigned)nq;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        unsigned o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
    }
    if (lane == 31) warp_sums[warp] = inc;
    __syncthreads();
    unsigned base = 0, total = 0;
    for (int i = 0; i < kBitsThreads / 32; ++i) {
        unsigned v = warp_sums[i];
        if (i < warp) base += v;
        total += v;
    }
    if (!EMIT) {
        if (threadIdx.x == 0) {
            block_cnt[blockIdx.x] = total;
            __threadfence();
            is_last = atomicAdd(done_counter, 1u) == gridDim.x - 1;
            scan_carry = 0;
        }
        __syncthreads();
        if (!is_last) return;
        __threadfence();
        const int64_t n = gridDim.x;
        for (int64_t b0 = 0; b0 < n; b0 += kBitsThreads) {
            const int64_t i = b0 + threadIdx.x;
            const long long v = i < n ? (long long)__ldcg(block_cnt + i) : 0;
            long long sc = v;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                long long o = __shfl_up_sync(0xffffffffu, sc, d);
                if (lane >= d) sc += o;
            }
            if (lane == 31) scan_sums[warp] = sc;
            __syncthreads();
            long long wbase = 0, tot = 0;
            for (int k = 0; k < kBitsThreads / 32; ++k) {
                const long long t = scan_sums[k];
                if (k < warp) wbase += t;
                tot += t;
            }
            const long long c = scan_carry;
            if (i < n) block_base[i] = c + wbase + sc - v;
            __syncthreads();
            if (threadIdx.x == 0) scan_carry = c + tot;
            __syncthreads();
        }
        if (threadIdx.x == 0) { block_base[n] = scan_carry; *done_counter = 0; }      // counter reset for the next call
    } else {
        int64_t rank = block_base[blockIdx.x] + base + inc - (unsigned)nq;
        int k = 0;
#pragma unroll
        for (int j = 0; j < W; ++j) {
            for (unsigned q = qual[j]; q; q &= q - 1, ++k, ++rank) {
                const int eb = __ffs(q) - 1;
                const int64_t s = k < 4 ? starts[k] : run_start_lb(lwords, bwords, w0 + j, eb);
                const int64_t len = ((w0 + j) << 5) + eb - s + 1;
                run_start_global[rank] = s;
                if (rank < capacity) {
                    const int64_t local = s - offsets[find_read(offsets, n_reads, s)];
                    intervals[2 * rank] = local - ext_left;
                    intervals[2 * rank + 1] = local + len + ext_right;
                }
            }
        }
    }
}

// interval_offsets[r] = number of emitted runs that start before read r = lower bound of
// offsets[r] in the (ascending) global run starts.  No atomics, any number of reads.
__global__ void k6_read_offsets_kernel(const int64_t* __restrict__ run_start_global, const int64_t* __restrict__ total_runs,
                                       const int64_t* __restrict__ offsets, int n_reads,
                                       int64_t* __restrict__ interval_offsets, int64_t* __restrict__ total_out) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > n_reads) return;
    const int64_t n = *total_runs;
    const int64_t key = offsets[r];
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (run_start_global[mid] < key) lo = mid + 1; else hi = mid;
    }
    interval_offsets[r] = lo;
    if (r == n_reads && total_out) *total_out = n;
}

int k6_bits_prepare(IntervalScratch& s, int64_t total_samples, LabelBits* out, cudaStream_t stream) {
    const int64_t n_words = ceil_div(total_samples > 0 ? total_samples : 1, 32);
    const int64_t stride = (n_words + 1 + 3) / 4 * 4;             // both word arrays 16-byte aligned (128-bit loads)
    CF_TRY(s.bits.ensure(sizeof(unsigned) * (size_t)(2 * stride)));
    CF_TRY(s.misc.ensure(256));
    static_assert(sizeof(unsigned) == 4, "");
    out->lwords = s.bits.as<unsigned>();
    out->bwords = out->lwords + stride;
    CF_CUDA(cudaMemsetAsync(out->lwords, 0, sizeof(unsigned) * (size_t)(2 * stride), stream));
    return CF_OK;
}

int k6_intervals_from_bits(IntervalScratch& s, const LabelBits& bits, const int64_t* offsets_dev, int32_t n_reads,
                           int64_t total_samples, int64_t* intervals, int64_t* interval_offsets, int64_t* total_out,
                           int64_t capacity, int32_t min_run, int32_t ext_left, int32_t ext_right, cudaStream_t stream) {
    const int64_t n = total_samples;
    const int64_t n_words = ceil_div(n, 32);
    const int64_t n_blocks = ceil_div(n_words, kBitsWordsPerBlock);
    if (n_reads <= 0 || n <= 0) {
        CF_CUDA(cudaMemsetAsync(interval_offsets, 0, sizeof(int64_t) * (size_t)((n_reads > 0 ? n_reads : 0) + 1), stream));
        if (total_out) CF_CUDA(cudaMemsetAsync(total_out, 0, sizeof(int64_t), stream));
        return CF_OK;
    }
    CF_TRY(s.block_cnt.ensure(sizeof(unsigned) * (size_t)n_blocks + sizeof(int64_t) * (size_t)(n_blocks + 1) + 16));
    int64_t* block_base = s.block_cnt.as<int64_t>();
    unsigned* block_cnt = reinterpret_cast<unsigned*>(block_base + n_blocks + 1);
    // global start of every emitted run (ascending): at most one run per min_run + 1 samples
    const int64_t max_runs = n / ((min_run < 1 ? 1 : min_run) + 1) + n_reads + 1;
    CF_TRY(s.read_cnt.ensure(sizeof(int64_t) * (size_t)max_runs));
    int64_t* run_start_global = s.read_cnt.as<int64_t>();
    if (!s.misc_zeroed) {                       // the done counter resets itself after every use
        CF_CUDA(cudaMemsetAsync(s.misc.ptr, 0, 256, stream));
        s.misc_zeroed = true;
    }
    unsigned* done = s.misc.as<unsigned>();
    k6_runs_bits_kernel<false><<<(unsigned)n_blocks, kBitsThreads, 0, stream>>>(
        bits.lwords, bits.bwords, n_words, offsets_dev, n_reads, min_run, ext_left, ext_right, block_cnt, block_base, done,
        nullptr, nullptr, 0);
    CF_LAUNCHED();
    k6_runs_bits_kernel<true><<<(unsigned)n_blocks, kBitsThreads, 0, stream>>>(
        bits.lwords, bits.bwords, n_words, offsets_dev, n_reads, min_run, ext_left, ext_right, nullptr, block_base, nullptr,
        run_start_global, intervals, capacity);
    CF_LAUNCHED();
    k6_read_offsets_kernel<<<(unsigned)ceil_div(n_reads + 1, 256), 256, 0, stream>>>(
        run_start_global, block_base + n_blocks, offsets_dev, n_reads, interval_offsets, total_out);
    CF_LAUNCHED();
    return CF_OK;
}

// ---------------------------------------------------------------- element-wise helpers
__global__ void k6_threshold_kernel(const double* __restrict__ scores, int64_t n, double thr,
                                    int64_t* __restrict__ labels) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x)
        labels[i] = scores[i] >= thr ? 1 : 0;
}

int k6_class_from_threshold(const double* scores, int64_t n, double threshold, int64_t* labels,
                            cudaStream_t stream) {
    if (n <= 0) return CF_OK;
    int64_t blocks = ceil_div(n, 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    k6_threshold_kernel<<<(unsigned)blocks, 256, 0, stream>>>(scores, n, threshold, labels);
    CF_LAUNCHED();
    return CF_OK;
}

// correct_short on arbitrary integer labels: a position keeps its value unless it is non-zero
// and its run of equal values is shorter than `threshold`.  Each thread measures its own run,
// looking at most threshold-1 positions to each side.
__global__ void k6_correct_short_kernel(const int64_t* __restrict__ in, int64_t n, int threshold,
                                        int64_t* __restrict__ out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t v = in[i];
        int64_t keep = v;
        if (v != 0) {
            int len = 1;
            for (int64_t j = i - 1; j >= 0 && len < threshold && in[j] == v; --j) ++len;
            for (int64_t j = i + 1; j < n && len < threshold && in[j] == v; ++j) ++len;
            if (len < threshold) keep = 0;
        }
        out[i] = keep;
    }
}

int k6_correct_short(const int64_t* labels, int64_t n, int32_t threshold, int64_t* out,
                     cudaStream_t stream) {
    if (n <= 0) return CF_OK;
    int64_t blocks = ceil_div(n, 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    k6_correct_short_kernel<<<(unsigned)blocks, 256, 0, stream>>>(labels, n, threshold, out);
    CF_LAUNCHED();
    return CF_OK;
}

}  // namespace cf
