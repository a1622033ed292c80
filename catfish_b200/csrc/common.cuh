// Shared declarations of the catfish_b200 CUDA library (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <vector>

#include "../../include/catfish_b200.h"

namespace cf {

constexpr int kWindow = 35;        // rnn_class.py:27
constexpr int kTileWindows = 128;  // windows per tile = TMEM lanes = UMMA M

// ---------------------------------------------------------------- errors
void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;

#define CF_CUDA(expr)                                                                   \
    do {                                                                                \
        cudaError_t _e = (expr);                                                        \
        if (_e != cudaSuccess) {                                                        \
            cf::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),       \
                          __FILE__, __LINE__);                                          \
            return CF_ERR_CUDA;                                                         \
        }                                                                               \
    } while (0)

#define CF_TRY(expr)                 \
    do {                             \
        int _s = (expr);             \
        if (_s != CF_OK) return _s;  \
    } while (0)

// Counts the launch and checks the launch error.
#define CF_LAUNCHED()                                                                   \
    do {                                                                                \
        cf::g_launches.fetch_add(1, std::memory_order_relaxed);                         \
        cudaError_t _e = cudaGetLastError();                                            \
        if (_e != cudaSuccess) {                                                        \
            cf::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e),   \
                          __FILE__, __LINE__);                                          \
            return CF_ERR_CUDA;                                                         \
        }                                                                               \
    } while (0)

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline int64_t round_up(int64_t a, int64_t b) { return ceil_div(a, b) * b; }

// ---------------------------------------------------------------- per-kernel-class timing
// Optional CUDA-event brackets around every launch, grouped by kernel class, so that bench.py can
// report the dominant kernel's duration measured on the launching stream.
enum KernelClass {
    KC_K1_STATS = 0,   // median / MAD
    KC_K1_TABLE,       // window table
    KC_K2_CONV,        // residual conv stack (incl. normalise + window gather)
    KC_K3_XPROJ,       // GRU input projection GEMM
    KC_K4_GRU,         // GRU recurrence
    KC_K5_HEAD,        // dense + sigmoid + un-window
    KC_K6_INTERVALS,   // threshold / run-length / interval emission
    KC_COUNT
};
const char* kernel_class_name(int cls);

struct Profiler {
    bool on = false;
    struct Rec { int cls; cudaEvent_t a, b; };
    std::vector<Rec> recs;
    std::vector<cudaEvent_t> pool;
    double ms[KC_COUNT] = {};
    long long launches[KC_COUNT] = {};
    Profiler() = default;
    Profiler(const Profiler&) = delete;
    Profiler& operator=(const Profiler&) = delete;
    ~Profiler();             // waits for the recorded events, then destroys every event
    cudaEvent_t get();
    void collect();          // synchronises on the recorded events and folds them into ms[]
    void reset();
};

// RAII bracket: records an event pair around the launches issued in its scope.
struct ProfScope {
    Profiler* p; cudaStream_t s; cudaEvent_t b = nullptr;
    ProfScope(Profiler* prof, int cls, cudaStream_t stream, int n_launches = 1) : p(prof), s(stream) {
        if (!p || !p->on) { p = nullptr; return; }
        cudaEvent_t a = p->get();
        b = p->get();
        cudaEventRecord(a, s);
        p->recs.push_back({cls, a, b});
        p->launches[cls] += n_launches;
    }
    ~ProfScope() { if (p) cudaEventRecord(b, s); }
};

// ---------------------------------------------------------------- device buffers
// A growable device allocation, freed by its destructor; grows only when asked for more.  Move-only: a moved-from
// buffer is empty.
struct DevBuf {
    void* ptr = nullptr;
    size_t bytes = 0;
    DevBuf() = default;
    DevBuf(DevBuf&& o) noexcept : ptr(o.ptr), bytes(o.bytes) { o.ptr = nullptr; o.bytes = 0; }
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { if (ptr) cudaFree(ptr); }
    int ensure(size_t want);
    // ensure + a synchronous copy of v from the host: the engines' weights
    template <typename T> int upload(const std::vector<T>& v) {
        CF_TRY(ensure(sizeof(T) * v.size()));
        CF_CUDA(cudaMemcpy(ptr, v.data(), sizeof(T) * v.size(), cudaMemcpyHostToDevice));
        return CF_OK;
    }
    template <typename T> T* as() const { return reinterpret_cast<T*>(ptr); }
};

// Pinned host staging buffer, freed by its destructor.
struct HostBuf {
    void* ptr = nullptr;
    size_t bytes = 0;
    HostBuf() = default;
    HostBuf(HostBuf&& o) noexcept : ptr(o.ptr), bytes(o.bytes) { o.ptr = nullptr; o.bytes = 0; }
    HostBuf(const HostBuf&) = delete;
    HostBuf& operator=(const HostBuf&) = delete;
    ~HostBuf() { if (ptr) cudaFreeHost(ptr); }
    int ensure(size_t want);
    template <typename T> T* as() const { return reinterpret_cast<T*>(ptr); }
};

// A CUDA event without timing, created on first use and destroyed by its destructor.
struct Event {
    cudaEvent_t ev = nullptr;
    Event() = default;
    Event(const Event&) = delete;
    Event& operator=(const Event&) = delete;
    ~Event() { if (ev) cudaEventDestroy(ev); }
    int create() {
        if (!ev) CF_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        return CF_OK;
    }
    int record(cudaStream_t stream) {
        CF_TRY(create());
        CF_CUDA(cudaEventRecord(ev, stream));
        return CF_OK;
    }
    // Waits for the last record; an event never recorded has nothing to wait for.
    int sync() {
        if (ev) CF_CUDA(cudaEventSynchronize(ev));
        return CF_OK;
    }
};

// ---------------------------------------------------------------- ragged batch plan
// Host-side description of one ragged batch of reads, and its device mirrors.
struct BatchPlan {
    int32_t n_reads = 0;
    int64_t total_samples = 0;
    int64_t total_windows = 0;     // sum over reads of L/35 + 1   (infer.py:32-38)
    int64_t n_tiles = 0;           // ceil(total_windows / 128)
    std::vector<int64_t> win_off;  // [R+1] first global window of each read
};

// Device arrays describing the windows of a batch (built by k1).
struct WindowTable {
    int64_t* src = nullptr;    // [n_tiles*128] first raw sample of the window, -1 = filler window
    int32_t* valid = nullptr;  // [n_tiles*128] real samples in the window (0..35)
    int32_t* read = nullptr;   // [n_tiles*128] read index, -1 = filler window
};

// ---------------------------------------------------------------- k1: normalisation
int k1_read_stats(const int16_t* raw, const int64_t* offsets_dev, int32_t n_reads, double* stats,
                  int32_t* wide_flags, uint32_t* wide_scratch, int n_wide_slots,
                  cudaStream_t stream);
int k1_normalize_f64(const int16_t* raw, const int64_t* offsets_dev, int32_t n_reads,
                     int64_t total_samples, const double* stats, double* norm,
                     cudaStream_t stream);
// Also sets the read-start bits of the interval caller (LabelBits::bwords, zeroed by k6_bits_prepare), so that k6
// needs no pass of its own.
int k1_window_table(const int64_t* offsets_dev, const int64_t* win_off_dev, int32_t n_reads,
                    int64_t total_windows, int64_t n_tiles, WindowTable tab, cudaStream_t stream,
                    unsigned* bwords, int64_t total_samples);
// One launch: the table of n_windows dense windows (window g covers xwin[35 g .. 35 g + 35)) over n_tiles tiles.
int k1_dense_window_table(int64_t n_windows, int64_t n_tiles, WindowTable tab, cudaStream_t stream);
// One launch: the normalised samples of the windows of tiles [tile0, tile0 + tiles) (window_input), as fp32 rows
// x[(tile * 35 + t) * 128 + w] - the input of the first layer of either engine when there are no residual blocks.
int k1_fill_windows(const int16_t* raw, const double* stats, const float* xwin, WindowTable tab, int64_t tile0,
                    int64_t tiles, float* x, cudaStream_t stream);
size_t k1_wide_scratch_bytes(int n_slots);
constexpr int kK1ChunkSamples = 32768;
size_t k1_chunked_scratch_bytes(int n_reads);
int k1_read_stats_chunked(const int16_t* raw, const int64_t* offsets_dev, int32_t n_reads, const int32_t* chunk_read,
                          const int64_t* chunk_beg, const int32_t* chunk_len, int64_t n_chunks, void* scratch,
                          double* stats, int32_t* wide_flags, uint32_t* wide_scratch, int n_wide_slots,
                          cudaStream_t stream);

// ---------------------------------------------------------------- k6: interval calling
struct IntervalScratch {
    DevBuf bits;        // label bit words
    DevBuf block_cnt;   // per-block counts + scanned bases
    DevBuf read_cnt;    // per-read counts
    DevBuf misc;        // "blocks done" counter of the count kernel (self-resetting)
    bool misc_zeroed = false;
};
enum BitSource { BITS_FROM_F32 = 0, BITS_FROM_F64 = 1, BITS_FROM_I64_EQ = 2 };
// Label bits and read-start bits over the concatenated sample index space.  k6_bits_prepare sizes and zeroes them; the
// producers set them; k6_intervals_from_bits turns them into intervals in three launches (count + scan by the last
// block, emit, per-read offsets).
//   label bits: on the inference path the head kernels of both engines threshold their own probabilities and OR
//               them in (head_output); the model-free entry points have the values in memory and call k6_pack_bits.
//   read-start bits: k1_window_table on the inference path, k6_read_starts for the model-free entry points.
struct LabelBits {
    unsigned* lwords = nullptr;     // [n_words + 1] label bits over the concatenated sample index space
    unsigned* bwords = nullptr;     // [n_words + 1] read-start bits
    double threshold = 0.5;
};
int k6_bits_prepare(IntervalScratch& s, int64_t total_samples, LabelBits* out, cudaStream_t stream);
// One launch: writes the label bits of n values, (double)value >= threshold for BITS_FROM_F32 / _F64 (NaN gives 0),
// value == label for BITS_FROM_I64_EQ.
int k6_pack_bits(const void* values, int source, double threshold, int64_t label, int64_t n, const LabelBits& bits,
                 cudaStream_t stream);
// One launch (none without reads): sets the read-start bit of every non-empty read.
int k6_read_starts(const int64_t* offsets_dev, int32_t n_reads, int64_t total_samples, const LabelBits& bits,
                   cudaStream_t stream);
// With no reads or no samples it zeroes interval_offsets[0..n_reads] and *total_out (if given) and launches nothing.
int k6_intervals_from_bits(IntervalScratch& s, const LabelBits& bits, const int64_t* offsets_dev, int32_t n_reads,
                           int64_t total_samples, int64_t* intervals, int64_t* interval_offsets, int64_t* total_out,
                           int64_t capacity, int32_t min_run, int32_t ext_left, int32_t ext_right, cudaStream_t stream);
int k6_class_from_threshold(const double* scores, int64_t n, double threshold, int64_t* labels,
                            cudaStream_t stream);
int k6_correct_short(const int64_t* labels, int64_t n, int32_t threshold, int64_t* out,
                     cudaStream_t stream);

// ---------------------------------------------------------------- k7: chunk merging (next row N1)
int k7_merge_chunks(int64_t* work, const int64_t* ioff, const int64_t* read_len, int n_reads, int64_t chunk,
                    int32_t* idx, int64_t* merged, int64_t* merged_cnt, int64_t* nonhp, int64_t* nonhp_cnt,
                    cudaStream_t stream);

// ---------------------------------------------------------------- k8: signal slicing (next row N2)
int k8_split_raw(const int16_t* raw, const int64_t* offsets_dev, const int64_t* ranges, const int32_t* range_read,
                 int64_t n_ranges, int64_t* lengths_scratch, int64_t* piece_off, int64_t capacity, int16_t* out,
                 cudaStream_t stream);

// ---------------------------------------------------------------- k9: validation counts (next row N4)
int k9_validation_blocks(int64_t n);
// partial: int64 [k9_validation_blocks(n)][6]; result: tp, fp, tn, fn, correct (int64) | loss sum (double)
int k9_validate(const float* logits, const uint8_t* labels, int64_t n, double threshold, long long* partial,
                long long* result, cudaStream_t stream);

// ---------------------------------------------------------------- k11: threshold sweep
constexpr int kSweepMaxThresholds = 4096;   // 3 x 4097 uint32 counters = 48 KiB of shared memory per block
// Checks the caller's thresholds (1..kSweepMaxThresholds, none NaN) and turns them into the sorted, deduplicated
// float thresholds K11 compares with; index[i] is the position of caller threshold i in `sorted`.
int k11_prepare_thresholds(const double* thresholds, int n_thresholds, std::vector<float>* sorted,
                           std::vector<int>* index);
// Device scratch of k11_sweep for n_thresholds thresholds.
size_t k11_scratch_bytes(int n_thresholds);
// Enqueues the sweep over n values (probabilities, or logits with values_are_logits) and the copy of the counts,
// int64 [sorted.size()][4] = tp, fp, tn, fn in sorted order, to counts_host; the caller synchronises the stream.
int k11_sweep(const float* values, bool values_are_logits, const uint8_t* labels, int64_t n,
              const std::vector<float>& sorted, void* scratch, long long* counts_host, cudaStream_t stream);

// ---------------------------------------------------------------- k10: event voting (next row N3)
int k10_vote_events(const double* scores, int64_t n_scores, const int64_t* ev_begin, int64_t first_event,
                    int64_t n_voted, int32_t* classes, int32_t* empty_flag, cudaStream_t stream);

}  // namespace cf
