// K1: per-read exact median / MAD of the raw int16 signal, the window tables, and the gathered scalar input of
// networks without residual blocks.
//
// Replaces infer.normalize_raw_signal (catfish/infer.py:96-105):
//     shift = np.median(raw); scale = np.median(np.abs(raw - shift)); (raw - shift) / scale
// np.median of an even-length array is the mean of the two middle order statistics, so
// shift is a multiple of 0.5 and scale a multiple of 0.25; both are reproduced exactly from a
// per-read histogram of the int16 values:
//   * the order statistics k_lo = (n-1)/2 and k_hi = n/2 of the value histogram give shift;
//   * |raw - shift| doubled is the integer |2v - s2| (s2 = v_lo + v_hi); its histogram is a
//     fold of the value histogram around s2/2 and is evaluated on the fly, giving scale.
// One CTA per read; the signal is read twice (min/max, then histogram) with 128-bit loads, the
// second pass out of L2.  Reads whose value range exceeds the shared-memory histogram take the
// same algorithm on a 65536-bin histogram in global scratch (k1_stats_wide_kernel).
#include "window_io.cuh"

namespace cf {

constexpr int kStatsThreads = 256;
constexpr int kSmemBins = 8192;   // covers the 13-bit MinION ADC range without the wide path

// ---------------------------------------------------------------- helpers
__device__ __forceinline__ int4 ld_nc_int4(const int4* p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

// Apply f(int value) to every element of p[0..n) using 128-bit loads on the aligned body.
template <typename F>
__device__ __forceinline__ void for_each_i16(const int16_t* __restrict__ p, int64_t n, F f) {
    const int tid = threadIdx.x, nt = blockDim.x;
    int64_t head = ((16 - (reinterpret_cast<uintptr_t>(p) & 15)) & 15) >> 1;
    if (head > n) head = n;
    for (int64_t i = tid; i < head; i += nt) f((int)p[i]);
    const int64_t nvec = (n - head) >> 3;
    const int4* pv = reinterpret_cast<const int4*>(p + head);
    for (int64_t i = tid; i < nvec; i += nt) {
        int4 v = ld_nc_int4(pv + i);
        int w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            f((int)(int16_t)(w[j] & 0xffff));
            f((int)(int16_t)((unsigned)w[j] >> 16));
        }
    }
    for (int64_t i = head + (nvec << 3) + tid; i < n; i += nt) f((int)p[i]);
}

// Exclusive block scan over kStatsThreads threads; every thread receives the grand total too.
__device__ __forceinline__ unsigned block_scan_excl(unsigned v, unsigned* total, unsigned* warp_sums) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        unsigned o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
    }
    __syncthreads();                       // protect warp_sums from a previous use
    if (lane == 31) warp_sums[warp] = inc;
    __syncthreads();
    unsigned base = 0, tot = 0;
    const int nw = blockDim.x >> 5;
    for (int w = 0; w < nw; ++w) {
        unsigned s = warp_sums[w];
        if (w < warp) base += s;
        tot += s;
    }
    *total = tot;
    return base + inc - v;
}

// Smallest i in [0, nb) with (sum_{j<=i} f(j)) > k, for k = k0 and k = k1.
template <typename F>
__device__ __forceinline__ void select2(F f, int nb, unsigned k0, unsigned k1, int* out,
                                        unsigned* warp_sums) {
    const int chunk = (nb + blockDim.x - 1) / blockDim.x;
    const int lo = threadIdx.x * chunk;
    const int hi = min(nb, lo + chunk);
    unsigned sum = 0;
    for (int i = lo; i < hi; ++i) sum += f(i);
    unsigned total;
    unsigned excl = block_scan_excl(sum, &total, warp_sums);
    if (sum) {
        const bool in0 = k0 >= excl && k0 < excl + sum;
        const bool in1 = k1 >= excl && k1 < excl + sum;
        if (in0 || in1) {
            unsigned cum = excl;
            for (int i = lo; i < hi; ++i) {
                unsigned c = f(i);
                if (in0 && k0 >= cum && k0 < cum + c) out[0] = i;
                if (in1 && k1 >= cum && k1 < cum + c) out[1] = i;
                cum += c;
            }
        }
    }
    __syncthreads();
}

// Median and MAD from a histogram `hist` of nb bins whose bin 0 holds value `base`; WRAP: the histogram is addressed
// by `value mod kSmemBins` instead (bin of value v = v & (kSmemBins - 1)).
template <bool WRAP = false>
__device__ __forceinline__ void stats_from_hist(const unsigned* hist, int base, int nb, unsigned n,
                                                double* stats_out, int* sel, unsigned* warp_sums) {
    auto H = [&](int i) -> unsigned { return WRAP ? hist[(base + i) & (kSmemBins - 1)] : hist[i]; };
    const unsigned k0 = (n - 1) >> 1, k1 = n >> 1;
    select2(H, nb, k0, k1, sel, warp_sums);
    const int s2 = (sel[0] + base) + (sel[1] + base);          // 2 * shift
    __syncthreads();
    // folded histogram: d2 = |2v - s2| in [0, 2*nb]
    auto folded = [&](int d2) -> unsigned {
        if ((d2 ^ s2) & 1) return 0u;                          // 2v = s2 +- d2 must be even
        const int a = ((s2 - d2) >> 1) - base;                 // arithmetic shift: value is even
        const int b = ((s2 + d2) >> 1) - base;
        unsigned c = 0;
        if (a >= 0 && a < nb) c += H(a);
        if (d2 != 0 && b >= 0 && b < nb) c += H(b);
        return c;
    };
    select2(folded, 2 * nb + 1, k0, k1, sel + 2, warp_sums);
    if (threadIdx.x == 0) {
        stats_out[0] = (double)s2 * 0.5;                       // mean of the two middle values
        stats_out[1] = ((double)sel[2] + (double)sel[3]) * 0.25;   // (d_lo/2 + d_hi/2) / 2
    }
}

// ---------------------------------------------------------------- fast path: smem histogram
__global__ void __launch_bounds__(kStatsThreads)
k1_stats_kernel(const int16_t* __restrict__ raw, const int64_t* __restrict__ offsets,
                double* __restrict__ stats, int32_t* __restrict__ wide_flags) {
    __shared__ unsigned hist[kSmemBins];
    __shared__ unsigned warp_sums[kStatsThreads / 32];
    __shared__ int red_min[kStatsThreads / 32], red_max[kStatsThreads / 32];
    __shared__ int sel[4];
    const int r = blockIdx.x;
    const int64_t beg = offsets[r];
    const int64_t n = offsets[r + 1] - beg;
    if (threadIdx.x == 0) wide_flags[r] = 0;
    if (n <= 0) {
        if (threadIdx.x == 0) { stats[2 * r] = nan(""); stats[2 * r + 1] = nan(""); }
        return;
    }
    const int16_t* p = raw + beg;
    // ONE pass: value range and a histogram addressed by value mod kSmemBins (no two values of a read that spans at
    // most kSmemBins values share a bin, so the range is not needed before the pass)
    for (int i = threadIdx.x; i < kSmemBins; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    int vmin = 32767, vmax = -32768;
    for_each_i16(p, n, [&](int v) {
        vmin = min(vmin, v);
        vmax = max(vmax, v);
        atomicAdd(&hist[v & (kSmemBins - 1)], 1u);
    });
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        vmin = min(vmin, __shfl_xor_sync(0xffffffffu, vmin, d));
        vmax = max(vmax, __shfl_xor_sync(0xffffffffu, vmax, d));
    }
    if ((threadIdx.x & 31) == 0) { red_min[threadIdx.x >> 5] = vmin; red_max[threadIdx.x >> 5] = vmax; }
    __syncthreads();
    for (int w = 0; w < kStatsThreads / 32; ++w) { vmin = min(vmin, red_min[w]); vmax = max(vmax, red_max[w]); }
    const int nb = vmax - vmin + 1;
    if (nb > kSmemBins) {                 // rare: defer to the global-histogram kernel
        if (threadIdx.x == 0) wide_flags[r] = 1;
        return;
    }
    stats_from_hist<true>(hist, vmin, nb, (unsigned)n, stats + 2 * r, sel, warp_sums);
}

// ---------------------------------------------------------------- wide path: global histogram
__global__ void __launch_bounds__(kStatsThreads)
k1_stats_wide_kernel(const int16_t* __restrict__ raw, const int64_t* __restrict__ offsets, int n_reads,
                     double* __restrict__ stats, const int32_t* __restrict__ wide_flags,
                     unsigned* __restrict__ scratch) {
    __shared__ unsigned warp_sums[kStatsThreads / 32];
    __shared__ int sel[4];
    unsigned* hist = scratch + (size_t)blockIdx.x * 65536;
    for (int r = blockIdx.x; r < n_reads; r += gridDim.x) {
        if (!wide_flags[r]) continue;     // block-uniform
        const int64_t beg = offsets[r];
        const int64_t n = offsets[r + 1] - beg;
        for (int i = threadIdx.x; i < 65536; i += blockDim.x) hist[i] = 0;
        __syncthreads();
        for_each_i16(raw + beg, n, [&](int v) { atomicAdd(&hist[v + 32768], 1u); });
        __syncthreads();
        stats_from_hist(hist, -32768, 65536, (unsigned)n, stats + 2 * r, sel, warp_sums);
        __syncthreads();
    }
}

size_t k1_wide_scratch_bytes(int n_slots) { return (size_t)n_slots * 65536 * sizeof(unsigned); }

int k1_read_stats(const int16_t* raw, const int64_t* offsets_dev, int32_t n_reads, double* stats,
                  int32_t* wide_flags, uint32_t* wide_scratch, int n_wide_slots,
                  cudaStream_t stream) {
    if (n_reads <= 0) return CF_OK;
    k1_stats_kernel<<<n_reads, kStatsThreads, 0, stream>>>(raw, offsets_dev, stats, wide_flags);
    CF_LAUNCHED();
    const int slots = n_reads < n_wide_slots ? n_reads : n_wide_slots;
    k1_stats_wide_kernel<<<slots, kStatsThreads, 0, stream>>>(raw, offsets_dev, n_reads, stats,
                                                              wide_flags, wide_scratch);
    CF_LAUNCHED();
    return CF_OK;
}

// ---------------------------------------------------------------- long reads: several CTAs per read
// A read is cut into chunks of kChunkSamples; every chunk is one CTA.  ONE pass over the signal: the chunk's value
// range (atomicMin/Max into the read's) and a shared-memory histogram addressed by `value mod kSmemBins` - as long
// as a read spans at most kSmemBins values no two of its values share a bin, so no origin has to be known before the
// pass (the earlier version read the signal twice: range first, then bins relative to the read's minimum).  The
// non-empty bins are added to the read's global histogram under the same addressing; pass 2 (one CTA per read)
// unwraps it from the read's minimum and evaluates the order statistics exactly as the one-CTA kernel does.  A read
// spanning more values is flagged there and redone by k1_stats_wide_kernel; what its chunks added is never read.
// Used when reads are long or few, so that one 1M-sample read does not sit on a single SM.
__global__ void __launch_bounds__(kStatsThreads)
k1_hist_chunks_kernel(const int16_t* __restrict__ raw, const int32_t* __restrict__ chunk_read,
                      const int64_t* __restrict__ chunk_beg, const int32_t* __restrict__ chunk_len,
                      int* __restrict__ gmin, int* __restrict__ gmax, unsigned* __restrict__ ghist) {
    __shared__ unsigned hist[kSmemBins];
    __shared__ int red_min[kStatsThreads / 32], red_max[kStatsThreads / 32];
    static_assert((kSmemBins & (kSmemBins - 1)) == 0, "bins are addressed by value & (kSmemBins - 1)");
    const int c = blockIdx.x;
    for (int i = threadIdx.x; i < kSmemBins; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    int vmin = 32767, vmax = -32768;
    for_each_i16(raw + chunk_beg[c], chunk_len[c], [&](int v) {
        vmin = min(vmin, v);
        vmax = max(vmax, v);
        atomicAdd(&hist[v & (kSmemBins - 1)], 1u);
    });
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        vmin = min(vmin, __shfl_xor_sync(0xffffffffu, vmin, d));
        vmax = max(vmax, __shfl_xor_sync(0xffffffffu, vmax, d));
    }
    if ((threadIdx.x & 31) == 0) { red_min[threadIdx.x >> 5] = vmin; red_max[threadIdx.x >> 5] = vmax; }
    __syncthreads();                            // also: every bin update of the chunk is in place
    for (int w = 0; w < kStatsThreads / 32; ++w) { vmin = min(vmin, red_min[w]); vmax = max(vmax, red_max[w]); }
    const int r = chunk_read[c];
    if (threadIdx.x == 0) {
        atomicMin(&gmin[r], vmin);
        atomicMax(&gmax[r], vmax);
    }
    const int nb = vmax - vmin + 1;
    if (nb > kSmemBins) return;                 // the read is wide: k1_stats_wide_kernel redoes it
    unsigned* gh = ghist + (size_t)r * kSmemBins;
    for (int i = threadIdx.x; i < nb; i += blockDim.x) {
        const int bin = (vmin + i) & (kSmemBins - 1);
        const unsigned v = hist[bin];
        if (v) atomicAdd(&gh[bin], v);
    }
}

__global__ void __launch_bounds__(kStatsThreads)
k1_stats_from_ghist_kernel(const int64_t* __restrict__ offsets, const int* __restrict__ gmin,
                           const int* __restrict__ gmax, const unsigned* __restrict__ ghist,
                           double* __restrict__ stats, int32_t* __restrict__ wide_flags) {
    __shared__ unsigned hist[kSmemBins];
    __shared__ unsigned warp_sums[kStatsThreads / 32];
    __shared__ int sel[4];
    const int r = blockIdx.x;
    const int64_t n = offsets[r + 1] - offsets[r];
    if (threadIdx.x == 0) wide_flags[r] = 0;
    if (n <= 0) {
        if (threadIdx.x == 0) { stats[2 * r] = nan(""); stats[2 * r + 1] = nan(""); }
        return;
    }
    const int base = gmin[r];
    const int nb = gmax[r] - base + 1;
    if (nb > kSmemBins) {
        if (threadIdx.x == 0) wide_flags[r] = 1;
        return;
    }
    const unsigned* gh = ghist + (size_t)r * kSmemBins;
    for (int i = threadIdx.x; i < nb; i += blockDim.x) hist[i] = gh[(base + i) & (kSmemBins - 1)];      // unwrap
    __syncthreads();
    stats_from_hist(hist, base, nb, (unsigned)n, stats + 2 * r, sel, warp_sums);
}

__global__ void k1_init_minmax_kernel(int* __restrict__ gmin, int* __restrict__ gmax, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { gmin[i] = 32767; gmax[i] = -32768; }
}

size_t k1_chunked_scratch_bytes(int n_reads) {
    return (size_t)n_reads * (kSmemBins * sizeof(unsigned) + 2 * sizeof(int)) + 256;
}

int k1_read_stats_chunked(const int16_t* raw, const int64_t* offsets_dev, int32_t n_reads, const int32_t* chunk_read,
                          const int64_t* chunk_beg, const int32_t* chunk_len, int64_t n_chunks, void* scratch,
                          double* stats, int32_t* wide_flags, uint32_t* wide_scratch, int n_wide_slots,
                          cudaStream_t stream) {
    if (n_reads <= 0) return CF_OK;
    unsigned* ghist = static_cast<unsigned*>(scratch);
    int* gmin = reinterpret_cast<int*>(ghist + (size_t)n_reads * kSmemBins);
    int* gmax = gmin + n_reads;
    CF_CUDA(cudaMemsetAsync(ghist, 0, (size_t)n_reads * kSmemBins * sizeof(unsigned), stream));
    k1_init_minmax_kernel<<<(unsigned)ceil_div(n_reads, 256), 256, 0, stream>>>(gmin, gmax, n_reads);
    CF_LAUNCHED();
    if (n_chunks > 0) {
        k1_hist_chunks_kernel<<<(unsigned)n_chunks, kStatsThreads, 0, stream>>>(raw, chunk_read, chunk_beg, chunk_len, gmin, gmax, ghist);
        CF_LAUNCHED();
    }
    k1_stats_from_ghist_kernel<<<n_reads, kStatsThreads, 0, stream>>>(offsets_dev, gmin, gmax, ghist, stats, wide_flags);
    CF_LAUNCHED();
    const int slots = n_reads < n_wide_slots ? n_reads : n_wide_slots;
    k1_stats_wide_kernel<<<slots, kStatsThreads, 0, stream>>>(raw, offsets_dev, n_reads, stats, wide_flags, wide_scratch);
    CF_LAUNCHED();
    return CF_OK;
}

// ---------------------------------------------------------------- (raw - shift) / scale in fp64
__device__ __forceinline__ int find_segment(const int64_t* __restrict__ off, int n, int64_t i) {
    int lo = 0, hi = n;                   // largest s with off[s] <= i, off has n+1 entries
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (off[mid] <= i) lo = mid; else hi = mid;
    }
    return lo;
}

__global__ void k1_normalize_f64_kernel(const int16_t* __restrict__ raw, const int64_t* __restrict__ offsets,
                                        int n_reads, int64_t total, const double* __restrict__ stats,
                                        double* __restrict__ norm) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int r = find_segment(offsets, n_reads, i);
        norm[i] = ((double)raw[i] - stats[2 * r]) / stats[2 * r + 1];
    }
}

int k1_normalize_f64(const int16_t* raw, const int64_t* offsets_dev, int32_t n_reads,
                     int64_t total_samples, const double* stats, double* norm, cudaStream_t stream) {
    if (total_samples <= 0) return CF_OK;
    const int threads = 256;
    int64_t blocks = ceil_div(total_samples, threads);
    if (blocks > 148 * 16) blocks = 148 * 16;
    k1_normalize_f64_kernel<<<(unsigned)blocks, threads, 0, stream>>>(raw, offsets_dev, n_reads,
                                                                       total_samples, stats, norm);
    CF_LAUNCHED();
    return CF_OK;
}

// ---------------------------------------------------------------- window table
// Window g of the batch: read r = segment of g in win_off, local window j = g - win_off[r];
// it covers raw[offsets[r] + 35 j ...] with min(35, L - 35 j) real samples, the rest of the
// window is the zero padding of infer.py:32-38 (a whole window of it when 35 divides L).
__global__ void k1_window_table_kernel(const int64_t* __restrict__ offsets, const int64_t* __restrict__ win_off,
                                       int n_reads, int64_t total_windows, int64_t n_slots,
                                       int64_t* __restrict__ src, int32_t* __restrict__ valid,
                                       int32_t* __restrict__ read, unsigned* __restrict__ bwords, int64_t total_samples) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g < n_reads) {                       // read-start bits for the interval caller (k6): one per non-empty read
        const int64_t o = offsets[g];
        if (o < total_samples && offsets[g + 1] > o) atomicOr(&bwords[o >> 5], 1u << (o & 31));
    }
    if (g >= n_slots) return;
    if (g >= total_windows) { src[g] = -1; valid[g] = 0; read[g] = -1; return; }
    const int r = find_segment(win_off, n_reads, g);
    const int64_t j = g - win_off[r];
    const int64_t len = offsets[r + 1] - offsets[r];
    const int64_t left = len - j * kWindow;
    src[g] = offsets[r] + j * kWindow;
    valid[g] = (int32_t)(left < kWindow ? (left < 0 ? 0 : left) : kWindow);
    read[g] = r;
}

int k1_window_table(const int64_t* offsets_dev, const int64_t* win_off_dev, int32_t n_reads,
                    int64_t total_windows, int64_t n_tiles, WindowTable tab, cudaStream_t stream,
                    unsigned* bwords, int64_t total_samples) {
    const int64_t slots = n_tiles * kTileWindows;
    if (slots <= 0) return CF_OK;
    // every read has at least one window, so slots >= n_reads and thread g < n_reads exists for every read
    k1_window_table_kernel<<<(unsigned)ceil_div(slots, 256), 256, 0, stream>>>(
        offsets_dev, win_off_dev, n_reads, total_windows, slots, tab.src, tab.valid, tab.read, bwords, total_samples);
    CF_LAUNCHED();
    return CF_OK;
}

// dense windows of cf_infer_windows and the validation row: window g covers x[35 g .. 35 g + 35)
__global__ void k1_dense_window_table_kernel(int64_t n_windows, int64_t n_slots, int64_t* __restrict__ src,
                                             int32_t* __restrict__ valid, int32_t* __restrict__ read) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_slots) return;
    const bool real = g < n_windows;
    src[g] = real ? g * kWindow : -1;
    valid[g] = real ? kWindow : 0;
    read[g] = -1;
}

int k1_dense_window_table(int64_t n_windows, int64_t n_tiles, WindowTable tab, cudaStream_t stream) {
    const int64_t slots = n_tiles * kTileWindows;
    k1_dense_window_table_kernel<<<(unsigned)ceil_div(slots, 256), 256, 0, stream>>>(n_windows, slots, tab.src, tab.valid, tab.read);
    CF_LAUNCHED();
    return CF_OK;
}

// ---------------------------------------------------------------- scalar network input
// x[(tile*35+t)*128+w] = sample t of window (tile0 + tile) * 128 + w (window_input)
__global__ void k1_fill_windows_kernel(const int16_t* __restrict__ raw, const double* __restrict__ stats,
                                       const float* __restrict__ xwin, const int64_t* __restrict__ src,
                                       const int32_t* __restrict__ valid, const int32_t* __restrict__ read,
                                       int64_t tile0, int64_t n_rows, float* __restrict__ x) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // local row
    if (i >= n_rows) return;
    const int w = (int)(i % kTileWindows);
    const int64_t tt = i / kTileWindows;
    const int t = (int)(tt % kWindow);
    const int64_t tile = tt / kWindow;
    x[i] = window_input(raw, stats, xwin, src, valid, read, (tile0 + tile) * kTileWindows + w)(t);
}

int k1_fill_windows(const int16_t* raw, const double* stats, const float* xwin, WindowTable tab, int64_t tile0,
                    int64_t tiles, float* x, cudaStream_t stream) {
    const int64_t rows = tiles * kWindow * kTileWindows;
    k1_fill_windows_kernel<<<(unsigned)ceil_div(rows, 256), 256, 0, stream>>>(raw, stats, xwin, tab.src, tab.valid, tab.read,
                                                                               tile0, rows, x);
    CF_LAUNCHED();
    return CF_OK;
}

}  // namespace cf
