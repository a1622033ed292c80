// K13: the exact ROC / precision-recall curve at every distinct score (no reference counterpart kernel: the
// reference's networks/metrics.py sorts on the host with sklearn's roc_curve / precision_recall_curve).
//
// Every position becomes one 32-bit key, sorted ascending by an LSD radix sort, then runs of equal score are counted:
//   key = (~bits(p) & 0x3FFFFFFF) << 1 | label   for p in [0, 1]: the bits of such a float fit in 30, so the
//                                                complement sorts descending; the mask gives -0.0 and +0.0 one key
//   key = 0x80000000 | label                     for NaN: after every score, p = 0 included
// Equal keys mean equal score and label, so the order of equal keys does not matter: the result is unique whatever
// the schedule.  A row is the end of a run of equal score (key >> 1); tp at that row is the number of label bits up
// to and including its position, and tp + fp is the position + 1, because every earlier key has a higher score.
//
//   k13_pack_kernel<VEC>      one read of scores and labels: validation (first bad index by atomicMin), the keys,
//                             and the digit histograms of all four 8-bit passes (shared memory, then integer atomics)
//   k13_scatter_kernel x 4    one digit pass each (onesweep): a tile claims its index from a counter, ranks its keys
//                             per warp with __match_any_sync (stable: input order), publishes its digit counts and
//                             looks back over its predecessors' (decoupled look-back, so no tile waits on one that has
//                             not been scheduled), then scatters
//   k13_runs_kernel<count>    per tile of sorted keys: run ends and label bits; the last tile to finish scans the tile
//                             counts (K6's count -> scan -> emit scheme)
//   k13_runs_kernel<emit>     threshold, tp and fp at every run end, in row order
//   k13_area_kernel / _sum    the AUROC sum (int64, exact) and the average-precision sum (float64) over the rows and the
//                             closing point (N0, N1), per-block partials summed in a fixed order: deterministic
#include <algorithm>
#include <cmath>

#include "common.cuh"
#include "window_io.cuh"

namespace cf {

constexpr int kCurveThreads = 256, kCurveItems = 16, kCurveTile = kCurveThreads * kCurveItems;
constexpr int kCurveWarps = kCurveThreads / 32, kCurveBins = 256, kCurvePasses = 4;
constexpr int kAreaBlocks = 1184, kAreaThreads = 256;
constexpr unsigned kNanKey = 0x80000000u;

__device__ __forceinline__ unsigned curve_key(float p, unsigned label) {
    return isnan(p) ? (kNanKey | label) : (((~__float_as_uint(p)) & 0x3FFFFFFFu) << 1) | label;
}

// The score of a (non-NaN) key: the complement of its 30 score bits.
__device__ __forceinline__ float curve_key_score(unsigned key) { return __uint_as_float(~(key >> 1) & 0x3FFFFFFFu); }

// Lanes with equal bins add once (the scores pile up near 0 and 1, so most lanes of a warp share their high digits).
__device__ __forceinline__ void curve_hist_add(unsigned* hist, int bin) {
    const unsigned peers = __match_any_sync(0xffffffffu, bin);
    if (bin >= 0 && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[bin], (unsigned)__popc(peers));
}

// ---------------------------------------------------------------- pack + histograms
// hist: uint32 [4][256], digit d of pass b at hist[b * 256 + d].  bad: the smallest index whose label is not 0 / 1 or
// whose score (after the logit mapping) is neither NaN nor in [0, 1]; all ones when there is none.  VEC: values
// 16-byte and labels 4-byte aligned (the keys are the library's own allocation).
template <bool VEC>
__global__ void __launch_bounds__(kCurveThreads)
k13_pack_kernel(const float* __restrict__ values, const uint8_t* __restrict__ labels, int64_t n, int logits,
                unsigned* __restrict__ keys, unsigned* __restrict__ hist_out, unsigned long long* __restrict__ bad) {
    __shared__ unsigned hist[kCurvePasses * kCurveBins];
    for (int i = threadIdx.x; i < kCurvePasses * kCurveBins; i += kCurveThreads) hist[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t stride = (int64_t)gridDim.x * kCurveThreads * 4;
    for (int64_t wbase = ((int64_t)blockIdx.x * kCurveThreads + (threadIdx.x & ~31)) * 4; wbase < n; wbase += stride) {
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
        unsigned k[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float p = logits ? head_sigmoid(v[e]) : v[e];
            if (e < m && (y[e] > 1u || !(isnan(p) || (p >= 0.f && p <= 1.f)))) atomicMin(bad, (unsigned long long)(base + e));
            k[e] = curve_key(p, y[e] & 1u);
        }
        if (VEC && m == 4) {
            *reinterpret_cast<uint4*>(keys + base) = make_uint4(k[0], k[1], k[2], k[3]);
        } else {
            for (int e = 0; e < m; ++e) keys[base + e] = k[e];
        }
#pragma unroll
        for (int e = 0; e < 4; ++e)
#pragma unroll
            for (int b = 0; b < kCurvePasses; ++b)
                curve_hist_add(hist, e < m ? b * kCurveBins + (int)((k[e] >> (8 * b)) & 0xFFu) : -1);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kCurvePasses * kCurveBins; i += kCurveThreads)
        if (hist[i]) atomicAdd(&hist_out[i], hist[i]);
}

// ---------------------------------------------------------------- one digit pass
// status: uint64 [tiles][256], shared by the four passes: high word = pass * 4 + kind (1 = the tile's own count,
// 2 = inclusive prefix over tiles 0..tile), low word = the count.  A word of an earlier pass reads as "not yet", so
// the array is zeroed once per sort.  tile_counter: this pass's counter (zeroed with the status).
constexpr unsigned kStatusLocal = 1, kStatusInclusive = 2;

__device__ __forceinline__ void status_store(unsigned long long* p, unsigned tag, unsigned value) {
    *reinterpret_cast<volatile unsigned long long*>(p) = ((unsigned long long)tag << 32) | value;
}

__global__ void __launch_bounds__(kCurveThreads)
k13_scatter_kernel(const unsigned* __restrict__ in, unsigned* __restrict__ out, int64_t n, int pass,
                   const unsigned* __restrict__ hist, unsigned* __restrict__ tile_counter,
                   unsigned long long* __restrict__ status) {
    __shared__ unsigned warp_cnt[kCurveWarps][kCurveBins];   // per warp and digit: count, then the warp's offset
    __shared__ unsigned digit_base[kCurveBins];               // output position of the tile's first key of each digit
    __shared__ unsigned scan_warp[kCurveWarps];
    __shared__ unsigned tile_s;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int shift = 8 * pass;
    if (threadIdx.x == 0) tile_s = atomicAdd(tile_counter, 1u);
    for (int i = threadIdx.x; i < kCurveWarps * kCurveBins; i += kCurveThreads) (&warp_cnt[0][0])[i] = 0;
    __syncthreads();
    const unsigned tile = tile_s;

    // rank: keys are taken in input order (item j of lane l is position warp_base + 32 j + l), so equal digits keep
    // their order - the stability an LSD sort needs
    const int64_t warp_base = (int64_t)tile * kCurveTile + warp * (32 * kCurveItems);
    const unsigned lt = (1u << lane) - 1u;
    unsigned key[kCurveItems], rank[kCurveItems];
#pragma unroll
    for (int j = 0; j < kCurveItems; ++j) {
        const int64_t i = warp_base + 32 * j + lane;
        const bool valid = i < n;
        key[j] = valid ? in[i] : 0u;
        const int d = valid ? (int)((key[j] >> shift) & 0xFFu) : kCurveBins;
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        rank[j] = valid ? warp_cnt[warp][d] + __popc(peers & lt) : 0u;
        __syncwarp();
        if (valid && (peers & lt) == 0) warp_cnt[warp][d] += __popc(peers);
        __syncwarp();
    }
    __syncthreads();

    // thread = digit: the warps' offsets within the tile, the tile's count, and the start of the digit in the output
    const int d = threadIdx.x;
    unsigned local = 0;
#pragma unroll
    for (int w = 0; w < kCurveWarps; ++w) { const unsigned c = warp_cnt[w][d]; warp_cnt[w][d] = local; local += c; }
    const unsigned h = hist[pass * kCurveBins + d];
    unsigned incl = h;                                        // exclusive scan of the pass's histogram over digits
#pragma unroll
    for (int s = 1; s < 32; s <<= 1) {
        const unsigned o = __shfl_up_sync(0xffffffffu, incl, s);
        if (lane >= s) incl += o;
    }
    if (lane == 31) scan_warp[warp] = incl;

    // decoupled look-back over the tiles before this one
    const unsigned tag = (unsigned)pass * 4u;
    unsigned long long* mine = status + (size_t)tile * kCurveBins + d;
    unsigned excl = 0;
    if (tile == 0) {
        status_store(mine, tag + kStatusInclusive, local);
    } else {
        status_store(mine, tag + kStatusLocal, local);
        for (int64_t p = (int64_t)tile - 1;; --p) {
            const volatile unsigned long long* q = status + (size_t)p * kCurveBins + d;
            unsigned long long v;
            do { v = *q; } while ((unsigned)(v >> 32) != tag + kStatusLocal && (unsigned)(v >> 32) != tag + kStatusInclusive);
            excl += (unsigned)v;
            if ((unsigned)(v >> 32) == tag + kStatusInclusive) break;
        }
        status_store(mine, tag + kStatusInclusive, excl + local);
    }
    __syncthreads();
    unsigned before = 0;
    for (int w = 0; w < warp; ++w) before += scan_warp[w];
    digit_base[d] = before + incl - h + excl;
    __syncthreads();

#pragma unroll
    for (int j = 0; j < kCurveItems; ++j) {
        const int64_t i = warp_base + 32 * j + lane;
        if (i < n) {
            const int dj = (int)((key[j] >> shift) & 0xFFu);
            out[digit_base[dj] + warp_cnt[warp][dj] + rank[j]] = key[j];
        }
    }
}

// ---------------------------------------------------------------- runs of equal score
// A thread owns kCurveItems consecutive sorted keys.  Position j ends a run when its key is a score (not NaN) and the
// next key has another score (or there is none).  Per tile: (run ends, label bits).
// Count: tile_cnt[tile] = (ends, positives); the last tile to finish writes the exclusive scan to tile_base[tile] and
// the totals to tile_base[tiles].  Emit: the rows, each (threshold, tp, fp) at its run end.
__device__ __forceinline__ bool curve_run_end(unsigned k, unsigned next, bool last) {
    return !(k & kNanKey) && (last || (k >> 1) != (next >> 1));
}

template <bool EMIT>
__global__ void __launch_bounds__(kCurveThreads)
k13_runs_kernel(const unsigned* __restrict__ keys, int64_t n, uint2* __restrict__ tile_cnt,
                unsigned long long* __restrict__ tile_base, unsigned* __restrict__ done_counter,
                float* __restrict__ thr, unsigned* __restrict__ tp, unsigned* __restrict__ fp) {
    __shared__ unsigned warp_e[kCurveWarps], warp_p[kCurveWarps];
    __shared__ unsigned long long carry_e, carry_p;
    __shared__ int is_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t j0 = (int64_t)blockIdx.x * kCurveTile + (int64_t)threadIdx.x * kCurveItems;
    unsigned k[kCurveItems + 1];
    if (j0 + kCurveItems < n) {                                // the keys are 16-byte aligned
#pragma unroll
        for (int q = 0; q < kCurveItems / 4; ++q) {
            const uint4 v = *reinterpret_cast<const uint4*>(keys + j0 + 4 * q);
            k[4 * q] = v.x; k[4 * q + 1] = v.y; k[4 * q + 2] = v.z; k[4 * q + 3] = v.w;
        }
        k[kCurveItems] = keys[j0 + kCurveItems];
    } else {
#pragma unroll
        for (int q = 0; q <= kCurveItems; ++q) k[q] = j0 + q < n ? keys[j0 + q] : kNanKey;
    }
    unsigned ends = 0, pos = 0;
#pragma unroll
    for (int q = 0; q < kCurveItems; ++q) {
        if (j0 + q < n) {
            ends += curve_run_end(k[q], k[q + 1], j0 + q + 1 == n);
            pos += k[q] & 1u;
        }
    }
    unsigned ie = ends, ip = pos;                             // inclusive scans over the warp
#pragma unroll
    for (int s = 1; s < 32; s <<= 1) {
        const unsigned oe = __shfl_up_sync(0xffffffffu, ie, s), op = __shfl_up_sync(0xffffffffu, ip, s);
        if (lane >= s) { ie += oe; ip += op; }
    }
    if (lane == 31) { warp_e[warp] = ie; warp_p[warp] = ip; }
    __syncthreads();
    unsigned be = 0, bp = 0, te = 0, tpos = 0;
    for (int w = 0; w < kCurveWarps; ++w) {
        if (w < warp) { be += warp_e[w]; bp += warp_p[w]; }
        te += warp_e[w];
        tpos += warp_p[w];
    }
    if (!EMIT) {
        if (threadIdx.x == 0) {
            tile_cnt[blockIdx.x] = make_uint2(te, tpos);
            __threadfence();
            is_last = atomicAdd(done_counter, 1u) == gridDim.x - 1;
            carry_e = carry_p = 0;
        }
        __syncthreads();
        if (!is_last) return;
        __threadfence();
        const int64_t tiles = gridDim.x;
        for (int64_t b0 = 0; b0 < tiles; b0 += kCurveThreads) {
            const int64_t i = b0 + threadIdx.x;
            const uint2 c = i < tiles ? __ldcg(tile_cnt + i) : make_uint2(0u, 0u);
            unsigned se = c.x, sp = c.y;
#pragma unroll
            for (int s = 1; s < 32; s <<= 1) {
                const unsigned oe = __shfl_up_sync(0xffffffffu, se, s), op = __shfl_up_sync(0xffffffffu, sp, s);
                if (lane >= s) { se += oe; sp += op; }
            }
            __syncthreads();                                   // the previous round has read warp_e / warp_p
            if (lane == 31) { warp_e[warp] = se; warp_p[warp] = sp; }
            __syncthreads();
            unsigned long long we = 0, wp = 0, sum_e = 0, sum_p = 0;
            for (int w = 0; w < kCurveWarps; ++w) {
                if (w < warp) { we += warp_e[w]; wp += warp_p[w]; }
                sum_e += warp_e[w];
                sum_p += warp_p[w];
            }
            const unsigned long long ce = carry_e, cp = carry_p;
            if (i < tiles) {
                tile_base[2 * i] = ce + we + se - c.x;
                tile_base[2 * i + 1] = cp + wp + sp - c.y;
            }
            __syncthreads();
            if (threadIdx.x == 0) { carry_e = ce + sum_e; carry_p = cp + sum_p; }
            __syncthreads();
        }
        if (threadIdx.x == 0) { tile_base[2 * tiles] = carry_e; tile_base[2 * tiles + 1] = carry_p; }
    } else {
        unsigned row = (unsigned)tile_base[2 * blockIdx.x] + be + ie - ends;
        unsigned cum = (unsigned)tile_base[2 * blockIdx.x + 1] + bp + ip - pos;
#pragma unroll
        for (int q = 0; q < kCurveItems; ++q) {
            const int64_t j = j0 + q;
            if (j < n) {
                cum += k[q] & 1u;
                if (curve_run_end(k[q], k[q + 1], j + 1 == n)) {
                    thr[row] = curve_key_score(k[q]);
                    tp[row] = cum;
                    fp[row] = (unsigned)(j + 1) - cum;
                    ++row;
                }
            }
        }
    }
}

// ---------------------------------------------------------------- areas
// Over the rows r = 0..R (row R: the closing point (fp, tp) = (N0, N1), NaN scores a tie below every number), with
// (tp, fp) = (0, 0) before row 0:
//   S  = sum (fp_r - fp_{r-1}) (tp_r + tp_{r-1})            int64, exact
//   AP = sum (tp_r - tp_{r-1}) tp_r / (tp_r + fp_r)          float64; divided by N1 on the host
// Fixed grid, fixed per-thread order and a fixed tree per block, then one block over the block partials: the sums do
// not depend on the schedule.
__device__ __forceinline__ void block_sum(long long& s, double& a, long long* ss, double* sa) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_down_sync(0xffffffffu, s, o);
        a += __shfl_down_sync(0xffffffffu, a, o);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { ss[warp] = s; sa[warp] = a; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < kAreaThreads / 32; ++w) { s += ss[w]; a += sa[w]; }
    }
}

__global__ void __launch_bounds__(kAreaThreads)
k13_area_kernel(const unsigned* __restrict__ tp, const unsigned* __restrict__ fp, int64_t rows, long long n0,
                long long n1, long long* __restrict__ part_s, double* __restrict__ part_a) {
    __shared__ long long ss[kAreaThreads / 32];
    __shared__ double sa[kAreaThreads / 32];
    long long s = 0;
    double a = 0.0;
    for (int64_t r = (int64_t)blockIdx.x * kAreaThreads + threadIdx.x; r <= rows; r += (int64_t)gridDim.x * kAreaThreads) {
        const long long t = r < rows ? tp[r] : n1, f = r < rows ? fp[r] : n0;
        const long long t0 = r > 0 ? tp[r - 1] : 0, f0 = r > 0 ? fp[r - 1] : 0;
        s += (f - f0) * (t + t0);
        if (t > t0) a += (double)(t - t0) * ((double)t / (double)(t + f));
    }
    block_sum(s, a, ss, sa);
    if (threadIdx.x == 0) { part_s[blockIdx.x] = s; part_a[blockIdx.x] = a; }
}

__global__ void __launch_bounds__(kAreaThreads)
k13_area_sum_kernel(const long long* __restrict__ part_s, const double* __restrict__ part_a, int parts,
                    long long* __restrict__ out_s, double* __restrict__ out_a) {
    __shared__ long long ss[kAreaThreads / 32];
    __shared__ double sa[kAreaThreads / 32];
    long long s = 0;
    double a = 0.0;
    for (int i = threadIdx.x; i < parts; i += kAreaThreads) { s += part_s[i]; a += part_a[i]; }
    block_sum(s, a, ss, sa);
    if (threadIdx.x == 0) { *out_s = s; *out_a = a; }
}

// ---------------------------------------------------------------- host
namespace {
struct CurveScratch {
    unsigned* keys[2];
    unsigned* hist;                    // [4][256]
    unsigned* counters;                // 4 pass counters + the runs kernel's done counter
    unsigned long long* bad;
    unsigned long long* status;        // [tiles][256]
    uint2* tile_cnt;                   // [tiles]
    unsigned long long* tile_base;     // [tiles + 1][2]
    long long* part_s;                 // [kAreaBlocks + 1]: the partials, then the total
    double* part_a;                    // [kAreaBlocks + 1]
};

size_t align256(size_t b) { return (b + 255) / 256 * 256; }

// Carves the scratch of n positions out of one allocation (nullptr base: only the size).
size_t carve(char* base, int64_t n, CurveScratch* s) {
    const int64_t tiles = ceil_div(n, kCurveTile);
    size_t off = 0;
    auto take = [&](size_t bytes) { char* p = base ? base + off : nullptr; off += align256(bytes); return p; };
    s->keys[0] = reinterpret_cast<unsigned*>(take(sizeof(unsigned) * (size_t)n));
    s->keys[1] = reinterpret_cast<unsigned*>(take(sizeof(unsigned) * (size_t)n));
    s->hist = reinterpret_cast<unsigned*>(take(sizeof(unsigned) * kCurvePasses * kCurveBins));
    s->counters = reinterpret_cast<unsigned*>(take(sizeof(unsigned) * (kCurvePasses + 1)));
    s->bad = reinterpret_cast<unsigned long long*>(take(sizeof(unsigned long long)));
    s->status = reinterpret_cast<unsigned long long*>(take(sizeof(unsigned long long) * kCurveBins * (size_t)tiles));
    s->tile_cnt = reinterpret_cast<uint2*>(take(sizeof(uint2) * (size_t)tiles));
    s->tile_base = reinterpret_cast<unsigned long long*>(take(sizeof(unsigned long long) * 2 * (size_t)(tiles + 1)));
    s->part_s = reinterpret_cast<long long*>(take(sizeof(long long) * (kAreaBlocks + 1)));
    s->part_a = reinterpret_cast<double*>(take(sizeof(double) * (kAreaBlocks + 1)));
    return off;
}
}  // namespace

int k13_curve(const float* values, bool values_are_logits, const uint8_t* labels, int64_t n, CurveRows* rows,
              CurveSummary* sum, cudaStream_t stream) {
    DevBuf scratch;
    CurveScratch s;
    CF_TRY(scratch.ensure(carve(nullptr, n, &s)));
    carve(static_cast<char*>(scratch.ptr), n, &s);
    const int64_t tiles = ceil_div(n, kCurveTile);
    // hist, counters and bad are adjacent: one memset each for the zeros and the "no bad index" ones
    CF_CUDA(cudaMemsetAsync(s.hist, 0, reinterpret_cast<char*>(s.bad) - reinterpret_cast<char*>(s.hist), stream));
    CF_CUDA(cudaMemsetAsync(s.bad, 0xFF, sizeof(unsigned long long), stream));
    CF_CUDA(cudaMemsetAsync(s.status, 0, sizeof(unsigned long long) * kCurveBins * (size_t)tiles, stream));

    const bool vec = reinterpret_cast<uintptr_t>(values) % 16 == 0 && reinterpret_cast<uintptr_t>(labels) % 4 == 0;
    auto pack = vec ? k13_pack_kernel<true> : k13_pack_kernel<false>;
    int dev = 0, sms = 0, per_sm = 0;
    CF_CUDA(cudaGetDevice(&dev));
    CF_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    CF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pack, kCurveThreads, 0));
    const int64_t pack_blocks = std::min<int64_t>(ceil_div(n, kCurveThreads * 4), (int64_t)std::max(per_sm, 1) * sms);
    pack<<<(unsigned)pack_blocks, kCurveThreads, 0, stream>>>(values, labels, n, values_are_logits ? 1 : 0, s.keys[0],
                                                               s.hist, s.bad);
    CF_LAUNCHED();
    for (int pass = 0; pass < kCurvePasses; ++pass) {
        k13_scatter_kernel<<<(unsigned)tiles, kCurveThreads, 0, stream>>>(s.keys[pass & 1], s.keys[(pass + 1) & 1], n, pass,
                                                                          s.hist, s.counters + pass, s.status);
        CF_LAUNCHED();
    }
    const unsigned* sorted = s.keys[kCurvePasses & 1];
    unsigned* done = s.counters + kCurvePasses;
    k13_runs_kernel<false><<<(unsigned)tiles, kCurveThreads, 0, stream>>>(sorted, n, s.tile_cnt, s.tile_base, done,
                                                                         nullptr, nullptr, nullptr);
    CF_LAUNCHED();

    // the histograms give N1 (odd keys of pass 0) and the NaN count (digit 0x80 of pass 3); the scan gives the rows
    std::vector<unsigned> hist(kCurvePasses * kCurveBins);
    unsigned long long bad = 0, totals[2] = {0, 0};
    CF_CUDA(cudaMemcpyAsync(hist.data(), s.hist, sizeof(unsigned) * hist.size(), cudaMemcpyDeviceToHost, stream));
    CF_CUDA(cudaMemcpyAsync(&bad, s.bad, sizeof(bad), cudaMemcpyDeviceToHost, stream));
    CF_CUDA(cudaMemcpyAsync(totals, s.tile_base + 2 * tiles, sizeof(totals), cudaMemcpyDeviceToHost, stream));
    CF_CUDA(cudaStreamSynchronize(stream));
    if (bad != ~0ull) {
        set_error("score curve: position %llu has a label other than 0 / 1 or a score that is neither NaN nor in [0, 1]",
                  bad);
        return CF_ERR_BAD_ARG;
    }
    long long n1 = 0;
    for (int d = 1; d < kCurveBins; d += 2) n1 += hist[d];
    sum->n_pos = n1;
    sum->n_neg = n - n1;
    sum->n_nan = hist[3 * kCurveBins + (kNanKey >> 24)];
    sum->n_rows = (int64_t)totals[0];

    CF_TRY(rows->thr.ensure(sizeof(float) * (size_t)std::max<int64_t>(sum->n_rows, 1)));
    CF_TRY(rows->tp.ensure(sizeof(unsigned) * (size_t)std::max<int64_t>(sum->n_rows, 1)));
    CF_TRY(rows->fp.ensure(sizeof(unsigned) * (size_t)std::max<int64_t>(sum->n_rows, 1)));
    k13_runs_kernel<true><<<(unsigned)tiles, kCurveThreads, 0, stream>>>(sorted, n, nullptr, s.tile_base, nullptr,
                                                                        rows->thr.as<float>(), rows->tp.as<unsigned>(),
                                                                        rows->fp.as<unsigned>());
    CF_LAUNCHED();
    const int area_blocks = (int)std::min<int64_t>(ceil_div(sum->n_rows + 1, kAreaThreads), kAreaBlocks);
    k13_area_kernel<<<area_blocks, kAreaThreads, 0, stream>>>(rows->tp.as<unsigned>(), rows->fp.as<unsigned>(),
                                                              sum->n_rows, sum->n_neg, sum->n_pos, s.part_s, s.part_a);
    CF_LAUNCHED();
    k13_area_sum_kernel<<<1, kAreaThreads, 0, stream>>>(s.part_s, s.part_a, area_blocks, s.part_s + kAreaBlocks,
                                                        s.part_a + kAreaBlocks);
    CF_LAUNCHED();
    long long area_s = 0;
    double area_a = 0.0;
    CF_CUDA(cudaMemcpyAsync(&area_s, s.part_s + kAreaBlocks, sizeof(area_s), cudaMemcpyDeviceToHost, stream));
    CF_CUDA(cudaMemcpyAsync(&area_a, s.part_a + kAreaBlocks, sizeof(area_a), cudaMemcpyDeviceToHost, stream));
    CF_CUDA(cudaStreamSynchronize(stream));
    sum->roc_auc = sum->n_neg > 0 && sum->n_pos > 0 ? (double)area_s / (2.0 * (double)sum->n_neg * (double)sum->n_pos) : NAN;
    sum->average_precision = sum->n_pos > 0 ? area_a / (double)sum->n_pos : NAN;
    return CF_OK;
}

}  // namespace cf
