// C-ABI entry points (include/catfish_b200.h): model construction, ragged-batch planning and
// the kernel sequence of one inference call.  No CPU fallback: every entry that computes
// requires a CUDA device and fails with CF_ERR_NO_DEVICE / CF_ERR_CUDA otherwise.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>

#include "model.cuh"

namespace cf {

static int use_device(int device);

// ---------------------------------------------------------------- errors / counters
static thread_local std::string t_error;
std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    t_error = buf;
}

int DevBuf::ensure(size_t want) {
    if (want <= bytes) return CF_OK;
    { DevBuf old(std::move(*this)); }      // free the smaller allocation before making the larger one
    const size_t grow = want + want / 8 + 256;
    cudaError_t e = cudaMalloc(&ptr, grow);
    if (e != cudaSuccess) {
        ptr = nullptr;
        set_error("cudaMalloc of %zu bytes failed: %s", grow, cudaGetErrorString(e));
        cudaGetLastError();
        return CF_ERR_ALLOC;
    }
    bytes = grow;
    return CF_OK;
}
const char* kernel_class_name(int cls) {
    static const char* names[KC_COUNT] = {"k1_stats", "k1_window_table", "k2_conv_stack", "k3_gru_input_proj",
                                          "k4_gru_recurrence", "k5_head", "k6_intervals"};
    return cls >= 0 && cls < KC_COUNT ? names[cls] : "?";
}

cudaEvent_t Profiler::get() {
    if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}
void Profiler::collect() {
    for (Rec& r : recs) {
        float t = 0.f;
        if (cudaEventSynchronize(r.b) == cudaSuccess && cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) ms[r.cls] += t;
        pool.push_back(r.a);
        pool.push_back(r.b);
    }
    recs.clear();
    cudaGetLastError();
}
void Profiler::reset() {
    collect();
    for (int i = 0; i < KC_COUNT; ++i) { ms[i] = 0; launches[i] = 0; }
}
Profiler::~Profiler() {
    collect();
    for (cudaEvent_t e : pool) cudaEventDestroy(e);
}

int HostBuf::ensure(size_t want) {
    if (want <= bytes) return CF_OK;
    { HostBuf old(std::move(*this)); }     // free the smaller allocation before making the larger one
    const size_t grow = want + want / 8 + 256;
    cudaError_t e = cudaMallocHost(&ptr, grow);
    if (e != cudaSuccess) {
        ptr = nullptr;
        set_error("cudaMallocHost of %zu bytes failed: %s", grow, cudaGetErrorString(e));
        cudaGetLastError();
        return CF_ERR_ALLOC;
    }
    bytes = grow;
    return CF_OK;
}

// ---------------------------------------------------------------- weights
static int check_desc(const cf_model_desc& d) {
    if (d.network_type < CF_NET_RESNET_RNN || d.network_type > CF_NET_RESNET) {
        set_error("unknown network_type %d", d.network_type);
        return CF_ERR_BAD_ARG;
    }
    if (d.window != kWindow) {
        set_error("window must be 35 (rnn_class.py:27), got %d", d.window);
        return CF_ERR_BAD_ARG;
    }
    const bool res = d.network_type != CF_NET_RNN, rnn = d.network_type != CF_NET_RESNET;
    if (res && (d.layer_size_res < 1 || d.layer_size_res > 1024 || d.n_layers_res < 1 || d.n_layers_res > 64)) {
        set_error("bad residual hyper-parameters (layer_size_res %d, n_layers_res %d)", d.layer_size_res, d.n_layers_res);
        return CF_ERR_BAD_ARG;
    }
    if (rnn && (d.layer_size < 1 || d.layer_size > 256 || d.n_layers < 1 || d.n_layers > 64)) {
        set_error("bad GRU hyper-parameters (layer_size %d in 1..256, n_layers %d)", d.layer_size, d.n_layers);
        return CF_ERR_BAD_ARG;
    }
    if (d.engine < CF_ENGINE_AUTO || d.engine > CF_ENGINE_SIMT) {
        set_error("unknown engine %d", d.engine);
        return CF_ERR_BAD_ARG;
    }
    return CF_OK;
}

int expected_tensor_shapes(const cf_model_desc& d, std::vector<std::vector<int64_t>>* shapes) {
    CF_TRY(check_desc(d));
    shapes->clear();
    int64_t feat = 1;
    if (d.network_type != CF_NET_RNN) {
        const int64_t c = d.layer_size_res;
        for (int b = 0; b < d.n_layers_res; ++b) {
            const int64_t cin = b == 0 ? 1 : c;
            const int64_t ks[4] = {1, 1, 3, 1};
            const int64_t ci[4] = {cin, cin, c, c};
            for (int j = 0; j < 4; ++j) {
                shapes->push_back({ks[j], ci[j], c});
                for (int v = 0; v < 5; ++v) shapes->push_back({c});   // bias, gamma, beta, mean, var
            }
        }
        feat = c;
    }
    if (d.network_type != CF_NET_RESNET) {
        const int64_t h = d.layer_size;
        for (int l = 0; l < d.n_layers; ++l) {
            const int64_t fin = l == 0 ? feat : 2 * h;
            for (int dir = 0; dir < 2; ++dir) {
                shapes->push_back({fin + h, 2 * h});
                shapes->push_back({2 * h});
                shapes->push_back({fin + h, h});
                shapes->push_back({h});
            }
        }
        feat = 2 * h;
    }
    shapes->push_back({feat, 1});
    shapes->push_back({1});
    return CF_OK;
}

int build_host_model(const cf_model_desc& d, const float* const* t, HostModel* out) {
    out->desc = d;
    int idx = 0;
    int feat = 1;
    if (d.network_type != CF_NET_RNN) {
        const int c = d.layer_size_res;
        for (int b = 0; b < d.n_layers_res; ++b) {
            const int cin = b == 0 ? 1 : c;
            const int ks[4] = {1, 1, 3, 1};
            const int ci[4] = {cin, cin, c, c};
            for (int j = 0; j < 4; ++j) {
                const float* kern = t[idx++];
                const float* bias = t[idx++];
                const float* gamma = t[idx++];
                const float* beta = t[idx++];
                const float* mean = t[idx++];
                const float* var = t[idx++];
                ConvLayer cl;
                cl.k = ks[j]; cl.cin = ci[j]; cl.cout = c;
                cl.w.resize((size_t)cl.k * cl.cin * c);
                cl.b.resize(c);
                for (int co = 0; co < c; ++co) {
                    // fold in double, store float (batch_normalization with moving statistics)
                    const double s = (double)gamma[co] / std::sqrt((double)var[co] + (double)d.bn_epsilon);
                    cl.b[co] = (float)((double)bias[co] * s + ((double)beta[co] - (double)mean[co] * s));
                    for (int q = 0; q < cl.k * cl.cin; ++q)
                        cl.w[(size_t)q * c + co] = (float)((double)kern[(size_t)q * c + co] * s);
                }
                out->convs.push_back(std::move(cl));
            }
        }
        feat = c;
    }
    if (d.network_type != CF_NET_RESNET) {
        const int h = d.layer_size;
        for (int l = 0; l < d.n_layers; ++l) {
            const int fin = l == 0 ? feat : 2 * h;
            for (int dir = 0; dir < 2; ++dir) {
                const float* wg = t[idx++];   // [fin+h][2h]
                const float* bg = t[idx++];   // [2h]
                const float* wc = t[idx++];   // [fin+h][h]
                const float* bc = t[idx++];   // [h]
                GruDir g;
                g.in = fin; g.h = h;
                g.wx.resize((size_t)fin * 3 * h);
                g.bx.resize(3 * h);
                g.wgh.resize((size_t)h * 2 * h);
                g.wch.resize((size_t)h * h);
                for (int k = 0; k < fin; ++k) {
                    for (int j = 0; j < 2 * h; ++j) g.wx[(size_t)k * 3 * h + j] = wg[(size_t)k * 2 * h + j];
                    for (int j = 0; j < h; ++j) g.wx[(size_t)k * 3 * h + 2 * h + j] = wc[(size_t)k * h + j];
                }
                for (int j = 0; j < 2 * h; ++j) g.bx[j] = bg[j];
                for (int j = 0; j < h; ++j) g.bx[2 * h + j] = bc[j];
                for (int k = 0; k < h; ++k) {
                    for (int j = 0; j < 2 * h; ++j) g.wgh[(size_t)k * 2 * h + j] = wg[(size_t)(fin + k) * 2 * h + j];
                    for (int j = 0; j < h; ++j) g.wch[(size_t)k * h + j] = wc[(size_t)(fin + k) * h + j];
                }
                out->gru.push_back(std::move(g));
            }
        }
        feat = 2 * h;
    }
    const float* hw = t[idx++];
    const float* hb = t[idx++];
    out->head_w.assign(hw, hw + feat);
    out->head_b = hb[0];
    return CF_OK;
}

// dense window table for cf_infer_windows: window g covers x[35 g .. 35 g + 35)
__global__ void dense_window_table_kernel(int64_t n_windows, int64_t n_slots, int64_t* __restrict__ src,
                                          int32_t* __restrict__ valid, int32_t* __restrict__ read) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_slots) return;
    const bool real = g < n_windows;
    src[g] = real ? g * kWindow : -1;
    valid[g] = real ? kWindow : 0;
    read[g] = -1;
}

}  // namespace cf

// ---------------------------------------------------------------- execution context
namespace cf {

// Everything an inference call writes.  The model (weights, engine, operand format) is read-only after
// cf_model_create; calls on different contexts of one model share nothing else and may overlap on the device.
// Its members free themselves; destroy it with the model's device current.
struct Exec {
    HostBuf pin_plan;                // offsets + win_off staging
    Event plan_copied;
    HostBuf pin_chunks;              // K1 chunk-table staging
    Event chunks_copied;
    DevBuf plan_dev;                 // offsets[R+1] | win_off[R+1]
    DevBuf stats, wide_flags, wide_scratch, k1_chunked, k1_chunk_tab;
    DevBuf tab_src, tab_valid, tab_read;
    DevBuf probs_internal;
    DevBuf val_logits, val_partial;  // validation row (N4)
    DevBuf val_sweep;                // its threshold sweep (K11 scratch)
    IntervalScratch k6;
    // host-buffer entry point
    DevBuf h_raw, h_intervals, h_ioff, h_probs;
    // engine workspaces: the tensor-core pass, and the CUDA-core pass (the tensor-core engine uses it for the
    // scalar input of RNN-only networks)
    DevBuf tc_ws, simt_ws;
    Profiler prof;                   // cf_profile_*: switched on for the model's default context only
    Event last_done;                 // end of the previous asynchronous call on this context (CallScope)
    std::mutex mu;
};

}  // namespace cf

// ---------------------------------------------------------------- handles
struct cf_model {
    cf::HostModel hm;
    int device = 0;
    int engine = CF_ENGINE_SIMT;
    cf::SimtEnginePtr simt;
    cf::TcEnginePtr tc;
    // the default context of every cf_model_* / cf_infer_* / cf_validate_* call; cf_model_destroy frees it
    std::unique_ptr<cf::Exec> def = std::make_unique<cf::Exec>();
    std::atomic<int> refs{1};        // the handle itself + one per live cf_exec
};

struct cf_exec {
    cf_model* model = nullptr;
    cf::Exec x;
};

namespace cf {

constexpr int kWideSlots = 64;

// Select `device` for the duration of a C-ABI call and restore the caller's current device on return
// (a multi-GPU process must not find its current device changed by creating, using or destroying a model).
struct DeviceGuard {
    int prev = -1;
    int set(int device);
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

static int use_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        cudaGetLastError();
        set_error("no CUDA device available (%s); catfish_b200 has no CPU fallback",
                  e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
        return CF_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= n) {
        set_error("device %d out of range (0..%d)", device, n - 1);
        return CF_ERR_BAD_ARG;
    }
    CF_CUDA(cudaSetDevice(device));
    return CF_OK;
}

int DeviceGuard::set(int device) {
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess) { cudaGetLastError(); cur = -1; }
    CF_TRY(use_device(device));
    if (cur >= 0 && cur != device) prev = cur;
    return CF_OK;
}

// The scope of one call on a context.  It holds the context's mutex and makes the model's device current.  A call
// that enqueues work also orders it on the device: one context = one set of scratch buffers, so a call on stream B
// must not start while the previous call's kernels (possibly on stream A) still use them.  Such a call waits on
// the event of the previous call on its context (a no-op on the same stream) and records it again when the scope
// ends - on every path, so that a call that fails after enqueueing work still orders the next call after that work.
// The destructor records the event while the model's device is current; the members then restore the caller's
// device and only after that release the mutex.
struct CallScope {
    std::lock_guard<std::mutex> lock;
    DeviceGuard device;
    Exec* x;
    cudaStream_t st = nullptr;
    bool ordered = false;
    explicit CallScope(Exec* ex) : lock(ex->mu), x(ex) {}
    ~CallScope() {
        if (ordered && cudaEventRecord(x->last_done.ev, st) != cudaSuccess) cudaGetLastError();
    }
    // Selects the model's device (reserve, profiling).
    int enter(int dev) { return device.set(dev); }
    // Also orders the call's work on `stream` after the previous call on this context.
    int enter(int dev, cudaStream_t stream) {
        CF_TRY(device.set(dev));
        CF_TRY(x->last_done.create());
        st = stream;
        ordered = true;
        CF_CUDA(cudaStreamWaitEvent(st, x->last_done.ev, 0));
        return CF_OK;
    }
};

static int engine_forward(cf_model* m, Exec* x, const int16_t* raw, const double* stats, const float* xwin,
                          WindowTable tab, int64_t n_tiles, float* probs, cudaStream_t stream,
                          bool want_logits = false, const LabelBits* bits = nullptr) {
    if (m->engine == CF_ENGINE_TCGEN05)
        return tc_forward(m->tc.get(), &x->tc_ws, &x->simt_ws, m->hm, raw, stats, xwin, tab, n_tiles, probs, stream,
                          &x->prof, want_logits, bits);
    return simt_forward(m->simt.get(), &x->simt_ws, m->hm, raw, stats, xwin, tab, n_tiles, probs, stream, &x->prof,
                        want_logits);
}

// Validate offsets and lay out the windows of every read (infer.py:32-43).
static int make_plan(const int64_t* offsets, int32_t n_reads, BatchPlan* p) {
    p->n_reads = n_reads;
    p->win_off.assign((size_t)n_reads + 1, 0);
    int64_t w = 0;
    for (int32_t r = 0; r < n_reads; ++r) {
        const int64_t len = offsets[r + 1] - offsets[r];
        if (len < 0 || offsets[r] < 0) {
            set_error("offsets must be non-negative and non-decreasing (read %d)", r);
            return CF_ERR_BAD_ARG;
        }
        if (len == 0) {
            set_error("read %d is empty: the reference raises IndexError (infer.py:151,184)", r);
            return CF_ERR_EMPTY_READ;
        }
        if (len >= (int64_t)1 << 31) {
            set_error("read %d has %lld samples; reads must be shorter than 2^31", r, (long long)len);
            return CF_ERR_BAD_ARG;
        }
        p->win_off[r] = w;
        w += len / kWindow + 1;          // padding 35 - L % 35, a whole window when 35 | L
    }
    p->win_off[n_reads] = w;
    p->total_windows = w;
    p->total_samples = n_reads > 0 ? offsets[n_reads] - offsets[0] : 0;
    p->n_tiles = ceil_div(w, kTileWindows);
    return CF_OK;
}

// Copy offsets (rebased to 0) and win_off to the device through the pinned staging buffer.
static int upload_plan(Exec* x, const int64_t* offsets, const BatchPlan& p, cudaStream_t stream,
                       const int64_t** offsets_dev, const int64_t** win_off_dev) {
    const size_t n = (size_t)p.n_reads + 1;
    CF_TRY(x->plan_copied.sync());                  // staging still in flight?
    CF_TRY(x->pin_plan.ensure(2 * n * sizeof(int64_t)));
    CF_TRY(x->plan_dev.ensure(2 * n * sizeof(int64_t)));
    int64_t* st = x->pin_plan.as<int64_t>();
    for (size_t i = 0; i < n; ++i) st[i] = offsets[i] - offsets[0];
    memcpy(st + n, p.win_off.data(), n * sizeof(int64_t));
    CF_CUDA(cudaMemcpyAsync(x->plan_dev.ptr, st, 2 * n * sizeof(int64_t), cudaMemcpyHostToDevice, stream));
    CF_TRY(x->plan_copied.record(stream));
    *offsets_dev = x->plan_dev.as<int64_t>();
    *win_off_dev = x->plan_dev.as<int64_t>() + n;
    return CF_OK;
}

// Median / MAD of every read: one CTA per read, or several CTAs per read when reads are long or few.
struct StatsScratch {
    DevBuf* flags; DevBuf* wide; DevBuf* chunked; DevBuf* chunk_tab;
    HostBuf* pinned = nullptr;        // optional pinned staging for the chunk table (keeps the call asynchronous)
    Event* staged = nullptr;          // recorded after the staging copy; waited on before the buffer is reused
};
// Whether a call of n_reads reads may take the chunked path, which needs k1_chunked_scratch_bytes(n_reads);
// stats_use_chunks decides from the read lengths.
static bool stats_may_use_chunks(int32_t n_reads) { return n_reads > 0 && n_reads <= 8192; }
static bool stats_use_chunks(const int64_t* offsets, int32_t n_reads) {
    if (!stats_may_use_chunks(n_reads)) return false;
    const int64_t total = offsets[n_reads] - offsets[0];
    return total / n_reads >= 2 * kK1ChunkSamples || n_reads < 2 * 148;
}
static int compute_read_stats(const int16_t* raw0, const int64_t* offsets_host, const int64_t* offsets_dev,
                              int32_t n_reads, double* stats, StatsScratch sc, cudaStream_t stream,
                              Profiler* prof = nullptr) {
    const bool chunks = stats_use_chunks(offsets_host, n_reads);
    CF_TRY(sc.flags->ensure(sizeof(int32_t) * (size_t)n_reads));
    CF_TRY(sc.wide->ensure(k1_wide_scratch_bytes(kWideSlots)));
    if (chunks) CF_TRY(sc.chunked->ensure(k1_chunked_scratch_bytes(n_reads)));   // allocate before the timed bracket
    ProfScope ps(prof, KC_K1_STATS, stream, chunks ? 4 : 2);
    if (!chunks)
        return k1_read_stats(raw0, offsets_dev, n_reads, stats, sc.flags->as<int32_t>(), sc.wide->as<uint32_t>(), kWideSlots, stream);
    // chunk table: [beg int64 | read int32 | len int32] per chunk, built on the host
    size_t nc = 0;
    for (int32_t r = 0; r < n_reads; ++r) nc += (size_t)ceil_div(offsets_host[r + 1] - offsets_host[r], kK1ChunkSamples);
    std::vector<uint8_t> pageable;
    uint8_t* host = nullptr;
    if (sc.pinned) {
        CF_TRY(sc.staged->sync());
        CF_TRY(sc.pinned->ensure(nc * 16 + 64));
        host = sc.pinned->as<uint8_t>();
    } else {
        pageable.resize(nc * 16 + 64);
        host = pageable.data();
    }
    int64_t* beg = reinterpret_cast<int64_t*>(host);
    int32_t* rd = reinterpret_cast<int32_t*>(host + nc * 8);
    int32_t* ln = reinterpret_cast<int32_t*>(host + nc * 12);
    size_t k = 0;
    for (int32_t r = 0; r < n_reads; ++r) {
        const int64_t b0 = offsets_host[r] - offsets_host[0], len = offsets_host[r + 1] - offsets_host[r];
        for (int64_t o = 0; o < len; o += kK1ChunkSamples, ++k) {
            beg[k] = b0 + o;
            rd[k] = r;
            ln[k] = (int32_t)std::min<int64_t>(kK1ChunkSamples, len - o);
        }
    }
    CF_TRY(sc.chunk_tab->ensure(nc * 16 + 64));
    uint8_t* tab = static_cast<uint8_t*>(sc.chunk_tab->ptr);
    if (nc) {
        CF_CUDA(cudaMemcpyAsync(tab, host, nc * 16, cudaMemcpyHostToDevice, stream));
        if (sc.pinned) {
            CF_TRY(sc.staged->record(stream));
        } else {
            CF_CUDA(cudaStreamSynchronize(stream));        // pageable, local staging
        }
    }
    return k1_read_stats_chunked(raw0, offsets_dev, n_reads, reinterpret_cast<int32_t*>(tab + nc * 8),
                                 reinterpret_cast<int64_t*>(tab), reinterpret_cast<int32_t*>(tab + nc * 12), (int64_t)nc,
                                 sc.chunked->ptr, stats, sc.flags->as<int32_t>(), sc.wide->as<uint32_t>(), kWideSlots, stream);
}

static int ensure_table(Exec* x, int64_t n_tiles, WindowTable* tab) {
    const size_t slots = (size_t)n_tiles * kTileWindows;
    CF_TRY(x->tab_src.ensure(slots * sizeof(int64_t)));
    CF_TRY(x->tab_valid.ensure(slots * sizeof(int32_t)));
    CF_TRY(x->tab_read.ensure(slots * sizeof(int32_t)));
    tab->src = x->tab_src.as<int64_t>();
    tab->valid = x->tab_valid.as<int32_t>();
    tab->read = x->tab_read.as<int32_t>();
    return CF_OK;
}

static int infer_reads_device(cf_model* m, Exec* x, const int16_t* raw_dev,
                              const int64_t* offsets_host, int32_t n_reads, float* probs_dev, int64_t* intervals_dev,
                              int64_t* interval_offsets_dev, int64_t capacity, double threshold,
                              int32_t min_run, int32_t ext_left, int32_t ext_right,
                              cudaStream_t stream) {
    BatchPlan plan;
    CF_TRY(make_plan(offsets_host, n_reads, &plan));
    if (n_reads == 0) {
        CF_CUDA(cudaMemsetAsync(interval_offsets_dev, 0, sizeof(int64_t), stream));
        return CF_OK;
    }
    const int16_t* raw0 = raw_dev + offsets_host[0];
    const int64_t *offsets_dev, *win_off_dev;
    CF_TRY(upload_plan(x, offsets_host, plan, stream, &offsets_dev, &win_off_dev));
    CF_TRY(x->stats.ensure(sizeof(double) * 2 * (size_t)n_reads));
    WindowTable tab;
    CF_TRY(ensure_table(x, plan.n_tiles, &tab));
    // When the caller does not want the probabilities, the head kernel thresholds them itself and emits label bits
    // (no 4 B/sample write + 4 B/sample read between the network and the interval caller).
    const bool fused_bits = !probs_dev && m->engine == CF_ENGINE_TCGEN05 && tc_can_emit_bits(m->tc.get());
    LabelBits bits;
    bits.threshold = threshold;
    CF_TRY(k6_bits_prepare(x->k6, plan.total_samples, &bits, stream));
    float* probs = probs_dev;
    if (!fused_bits && !probs) {
        CF_TRY(x->probs_internal.ensure(sizeof(float) * (size_t)plan.total_samples));
        probs = x->probs_internal.as<float>();
    }
    StatsScratch sc{&x->wide_flags, &x->wide_scratch, &x->k1_chunked, &x->k1_chunk_tab, &x->pin_chunks, &x->chunks_copied};
    CF_TRY(compute_read_stats(raw0, offsets_host, offsets_dev, n_reads, x->stats.as<double>(), sc, stream, &x->prof));
    {
        ProfScope ps(&x->prof, KC_K1_TABLE, stream);
        CF_TRY(k1_window_table(offsets_dev, win_off_dev, n_reads, plan.total_windows, plan.n_tiles, tab, stream,
                               bits.bwords, plan.total_samples));
    }
    CF_TRY(engine_forward(m, x, raw0, x->stats.as<double>(), nullptr, tab, plan.n_tiles, probs, stream, false,
                          fused_bits ? &bits : nullptr));
    ProfScope ps(&x->prof, KC_K6_INTERVALS, stream, fused_bits ? 3 : 4);
    if (!fused_bits) CF_TRY(k6_pack_bits(probs, BITS_FROM_F32, threshold, 1, plan.total_samples, bits, stream));
    CF_TRY(k6_intervals_from_bits(x->k6, bits, offsets_dev, n_reads, plan.total_samples, intervals_dev,
                                  interval_offsets_dev, nullptr, capacity, min_run, ext_left, ext_right, stream));
    return CF_OK;
}

}  // namespace cf

// ================================================================== extern "C"
// ---------------------------------------------------------------- model-free helpers
namespace {
int upload_offsets(const int64_t* offsets_host, int32_t n_reads, cf::DevBuf* buf, cudaStream_t st) {
    CF_TRY(buf->ensure(sizeof(int64_t) * ((size_t)n_reads + 1)));
    std::vector<int64_t> off((size_t)n_reads + 1);
    for (int32_t i = 0; i <= n_reads; ++i) off[i] = offsets_host[i] - offsets_host[0];
    CF_CUDA(cudaMemcpyAsync(buf->ptr, off.data(), sizeof(int64_t) * off.size(), cudaMemcpyHostToDevice, st));
    CF_CUDA(cudaStreamSynchronize(st));     // `off` is pageable and about to go out of scope
    return CF_OK;
}

// cf_call_intervals and cf_hp_in_pred: read-start bits from the offsets, label bits from `values` (k6_pack_bits), then
// the intervals.  Synchronises the stream on every path: the scratch is freed on return.
int model_free_intervals(const void* values, int source, double threshold, int64_t label, const int64_t* offsets_host,
                         int32_t n_reads, int64_t* intervals, int64_t* interval_offsets, int64_t* total_out,
                         int64_t capacity, int32_t min_run, int32_t ext_left, int32_t ext_right, cudaStream_t st) {
    const int64_t total = offsets_host[n_reads] - offsets_host[0];
    cf::DevBuf off;
    CF_TRY(upload_offsets(offsets_host, n_reads, &off, st));
    cf::IntervalScratch scratch;
    cf::LabelBits bits;
    int s = cf::k6_bits_prepare(scratch, total, &bits, st);
    if (s == CF_OK) s = cf::k6_read_starts(off.as<int64_t>(), n_reads, total, bits, st);
    if (s == CF_OK) s = cf::k6_pack_bits(values, source, threshold, label, total, bits, st);
    if (s == CF_OK) s = cf::k6_intervals_from_bits(scratch, bits, off.as<int64_t>(), n_reads, total, intervals,
                                                   interval_offsets, total_out, capacity, min_run, ext_left, ext_right, st);
    cudaStreamSynchronize(st);
    return s;
}
}  // namespace

extern "C" {

int cf_abi_version(void) { return CF_ABI_VERSION; }
const char* cf_last_error(void) { return cf::t_error.c_str(); }

int cf_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int cf_merge_chunks(int32_t device, const int64_t* intervals_dev, const int64_t* interval_offsets_host,
                    const int64_t* read_lengths_host, int32_t n_reads, int64_t chunk_size, int64_t* merged_dev,
                    int64_t* merged_count_dev, int64_t* nonhp_dev, int64_t* nonhp_count_dev, void* stream) {
    if (n_reads < 0 || !interval_offsets_host || !read_lengths_host || !merged_dev || !merged_count_dev || !nonhp_dev ||
        !nonhp_count_dev) {
        cf::set_error("cf_merge_chunks: bad argument");
        return CF_ERR_BAD_ARG;
    }
    if (n_reads == 0) return CF_OK;
    cf::DeviceGuard guard;
    CF_TRY(guard.set(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int64_t n_int = interval_offsets_host[n_reads] - interval_offsets_host[0];
    if (n_int < 0 || (n_int > 0 && !intervals_dev)) { cf::set_error("cf_merge_chunks: bad offsets"); return CF_ERR_BAD_ARG; }
    cf::DevBuf work, idx, meta;
    CF_TRY(work.ensure(sizeof(int64_t) * 2 * (size_t)(n_int + 1)));
    CF_TRY(idx.ensure(sizeof(int32_t) * (size_t)(n_int + n_reads + 1)));
    CF_TRY(meta.ensure(sizeof(int64_t) * (2 * (size_t)n_reads + 1)));
    std::vector<int64_t> host((size_t)2 * n_reads + 1);
    for (int32_t r = 0; r <= n_reads; ++r) host[r] = interval_offsets_host[r] - interval_offsets_host[0];
    for (int32_t r = 0; r < n_reads; ++r) host[n_reads + 1 + r] = read_lengths_host[r];
    CF_CUDA(cudaMemcpyAsync(meta.ptr, host.data(), sizeof(int64_t) * host.size(), cudaMemcpyHostToDevice, st));
    if (n_int > 0)
        CF_CUDA(cudaMemcpyAsync(work.ptr, intervals_dev + 2 * interval_offsets_host[0], sizeof(int64_t) * 2 * (size_t)n_int,
                                cudaMemcpyDeviceToDevice, st));
    int s = cf::k7_merge_chunks(work.as<int64_t>(), meta.as<int64_t>(), meta.as<int64_t>() + n_reads + 1, n_reads,
                                chunk_size, idx.as<int32_t>(), merged_dev, merged_count_dev, nonhp_dev, nonhp_count_dev, st);
    cudaStreamSynchronize(st);
    return s;
}

int cf_split_raw(int32_t device, const int16_t* raw_dev, const int64_t* offsets_host, int32_t n_reads,
                 const int64_t* ranges_dev, const int32_t* range_read_dev, int64_t n_ranges, int16_t* out_dev,
                 int64_t capacity, int64_t* piece_offsets_dev, void* stream) {
    if (n_reads < 0 || n_ranges < 0 || !offsets_host || !piece_offsets_dev || capacity < 0 ||
        (n_ranges > 0 && (!raw_dev || !ranges_dev || !range_read_dev)) || (capacity > 0 && !out_dev)) {
        cf::set_error("cf_split_raw: bad argument");
        return CF_ERR_BAD_ARG;
    }
    cf::DeviceGuard guard;
    CF_TRY(guard.set(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cf::DevBuf off, len;
    if (n_reads > 0) CF_TRY(upload_offsets(offsets_host, n_reads, &off, st));
    CF_TRY(len.ensure(sizeof(int64_t) * (size_t)(n_ranges + 1)));
    const int16_t* raw0 = n_reads > 0 ? raw_dev + offsets_host[0] : raw_dev;
    int s = cf::k8_split_raw(raw0, off.as<int64_t>(), ranges_dev, range_read_dev, n_ranges, len.as<int64_t>(),
                             piece_offsets_dev, capacity, out_dev, st);
    cudaStreamSynchronize(st);
    return s;
}

int cf_selftest_f16e5(int32_t device, const float* a_dev, int32_t k, int32_t n, const float* w_host, int32_t mode,
                      float* out_dev, void* stream) {
    if (!a_dev || !w_host || !out_dev) { cf::set_error("cf_selftest_f16e5: bad argument"); return CF_ERR_BAD_ARG; }
    cf::DeviceGuard guard;
    CF_TRY(guard.set(device));
    return cf::tc_selftest_f16e5(a_dev, k, n, w_host, mode, out_dev, static_cast<cudaStream_t>(stream));
}

int64_t cf_launch_count(void) { return (int64_t)cf::g_launches.load(); }

int cf_model_num_tensors(const cf_model_desc* desc) {
    if (!desc) { cf::set_error("desc is NULL"); return CF_ERR_BAD_ARG; }
    std::vector<std::vector<int64_t>> shapes;
    int s = cf::expected_tensor_shapes(*desc, &shapes);
    if (s != CF_OK) return s;
    return (int)shapes.size();
}

int cf_model_create(const cf_model_desc* desc, const float* const* tensors, const int64_t* tensor_sizes,
                    int32_t n_tensors, int32_t device, cf_model** out_model) {
    if (!desc || !tensors || !tensor_sizes || !out_model) {
        cf::set_error("cf_model_create: NULL argument");
        return CF_ERR_BAD_ARG;
    }
    *out_model = nullptr;
    std::vector<std::vector<int64_t>> shapes;
    CF_TRY(cf::expected_tensor_shapes(*desc, &shapes));
    if ((size_t)n_tensors != shapes.size()) {
        cf::set_error("cf_model_create: expected %zu tensors, got %d", shapes.size(), n_tensors);
        return CF_ERR_BAD_ARG;
    }
    for (size_t i = 0; i < shapes.size(); ++i) {
        int64_t n = 1;
        for (int64_t v : shapes[i]) n *= v;
        if (tensor_sizes[i] != n || !tensors[i]) {
            cf::set_error("cf_model_create: tensor %zu has %lld elements, expected %lld", i,
                          (long long)tensor_sizes[i], (long long)n);
            return CF_ERR_BAD_ARG;
        }
    }
    cf::DeviceGuard guard;
    CF_TRY(guard.set(device));
    cf::HostModel hm;
    cf::build_host_model(*desc, tensors, &hm);
    int engine = desc->engine;
    if (engine == CF_ENGINE_AUTO) engine = cf::tc_supported(hm) ? CF_ENGINE_TCGEN05 : CF_ENGINE_SIMT;
    if (engine == CF_ENGINE_TCGEN05 && !cf::tc_supported(hm)) {
        cf::set_error("the tcgen05 engine supports layer_size_res <= 32 and layer_size <= 64 only");
        return CF_ERR_BAD_ARG;
    }
    // a failed creation frees what it made (the engine pointers' destructors) and returns its status
    cf::TcEnginePtr tc;
    cf::SimtEnginePtr simt;
    CF_TRY(engine == CF_ENGINE_TCGEN05 ? cf::tc_create(hm, &tc) : cf::simt_create(hm, &simt));
    const cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        cf::set_error("cf_model_create: uploading weights failed: %s", cudaGetErrorString(e));
        return CF_ERR_CUDA;
    }
    cf_model* m = new cf_model();
    m->hm = std::move(hm);
    m->device = device;
    m->engine = engine;
    m->tc = std::move(tc);
    m->simt = std::move(simt);
    *out_model = m;
    return CF_OK;
}

// Drop one reference (the handle's or a context's); the last one frees the weights.  The caller has selected
// the model's device.
static void model_unref(cf_model* m) {
    if (m->refs.fetch_sub(1) != 1) return;
    cudaDeviceSynchronize();
    delete m;
}

void cf_model_destroy(cf_model* m) {
    if (!m) return;
    cf::DeviceGuard guard;
    if (guard.set(m->device) != CF_OK) cudaSetDevice(m->device);
    cudaDeviceSynchronize();
    m->def.reset();
    model_unref(m);
}

int cf_exec_create(cf_model* m, cf_exec** out) {
    if (!m || !out) { cf::set_error("cf_exec_create: NULL argument"); return CF_ERR_BAD_ARG; }
    *out = nullptr;
    cf::DeviceGuard guard;
    CF_TRY(guard.set(m->device));
    cf_exec* ex = new cf_exec();
    ex->model = m;
    m->refs.fetch_add(1);
    *out = ex;
    return CF_OK;
}

void cf_exec_destroy(cf_exec* ex) {
    if (!ex) return;
    cf::DeviceGuard guard;
    if (guard.set(ex->model->device) != CF_OK) cudaSetDevice(ex->model->device);
    {
        std::lock_guard<std::mutex> lock(ex->x.mu);      // a call on another thread finishes enqueueing first
        ex->x.last_done.sync();
    }
    cf_model* m = ex->model;
    delete ex;                                          // unlocked: a locked mutex must not be destroyed
    model_unref(m);
}

int cf_model_engine(const cf_model* m) { return m ? m->engine : CF_ERR_BAD_ARG; }
int cf_model_operand_format(const cf_model* m) {
    if (!m) return CF_ERR_BAD_ARG;
    return m->engine == CF_ENGINE_TCGEN05 ? cf::tc_operand_format(m->tc.get()) : -1;
}

int cf_profile_enable(cf_model* m, int32_t on) {
    if (!m) { cf::set_error("cf_profile_enable: NULL model"); return CF_ERR_BAD_ARG; }
    cf::CallScope call(m->def.get());
    CF_TRY(call.enter(m->device));
    m->def->prof.reset();
    m->def->prof.on = on != 0;
    return CF_OK;
}

int cf_profile_num_classes(void) { return cf::KC_COUNT; }
const char* cf_profile_class_name(int32_t cls) { return cf::kernel_class_name(cls); }

int cf_profile_read(cf_model* m, double* ms_out, int64_t* launches_out, int32_t n) {
    if (!m || !ms_out || !launches_out || n < cf::KC_COUNT) { cf::set_error("cf_profile_read: bad argument"); return CF_ERR_BAD_ARG; }
    cf::CallScope call(m->def.get());
    CF_TRY(call.enter(m->device));
    cf::Profiler& prof = m->def->prof;
    prof.collect();
    for (int i = 0; i < cf::KC_COUNT; ++i) { ms_out[i] = prof.ms[i]; launches_out[i] = prof.launches[i]; }
    return CF_OK;
}

// Grow every buffer of context x, the engine workspaces included, to what a call of at most max_samples samples
// and max_reads reads needs.
static int reserve(cf_model* m, cf::Exec* x, int64_t max_samples, int32_t max_reads) {
    cf::CallScope call(x);
    CF_TRY(call.enter(m->device));
    const int64_t tiles = cf::ceil_div(max_samples / cf::kWindow + max_reads, cf::kTileWindows);
    cf::WindowTable tab;
    CF_TRY(cf::ensure_table(x, tiles, &tab));
    CF_TRY(x->stats.ensure(sizeof(double) * 2 * (size_t)max_reads));
    CF_TRY(x->wide_flags.ensure(sizeof(int32_t) * (size_t)max_reads));
    CF_TRY(x->wide_scratch.ensure(cf::k1_wide_scratch_bytes(cf::kWideSlots)));
    if (cf::stats_may_use_chunks(max_reads)) CF_TRY(x->k1_chunked.ensure(cf::k1_chunked_scratch_bytes(max_reads)));
    CF_TRY(x->probs_internal.ensure(sizeof(float) * (size_t)max_samples));
    CF_TRY(x->val_sweep.ensure(cf::k11_scratch_bytes(cf::kSweepMaxThresholds)));
    if (m->engine == CF_ENGINE_TCGEN05) return cf::tc_reserve(m->tc.get(), &x->tc_ws, &x->simt_ws, m->hm, tiles);
    return cf::simt_reserve(&x->simt_ws, m->hm, tiles);
}

int cf_model_reserve(cf_model* m, int64_t max_samples, int32_t max_reads) {
    if (!m || max_samples < 0 || max_reads < 0) { cf::set_error("cf_model_reserve: bad argument"); return CF_ERR_BAD_ARG; }
    return reserve(m, m->def.get(), max_samples, max_reads);
}

int cf_exec_reserve(cf_exec* ex, int64_t max_samples, int32_t max_reads) {
    if (!ex || max_samples < 0 || max_reads < 0) { cf::set_error("cf_exec_reserve: bad argument"); return CF_ERR_BAD_ARG; }
    return reserve(ex->model, &ex->x, max_samples, max_reads);
}

int cf_infer_windows(cf_model* m, const float* x_dev, int64_t n_windows, float* probs_dev, void* stream) {
    if (!m || n_windows < 0 || (n_windows > 0 && (!x_dev || !probs_dev))) {
        cf::set_error("cf_infer_windows: bad argument");
        return CF_ERR_BAD_ARG;
    }
    if (n_windows == 0) return CF_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cf::Exec* x = m->def.get();
    cf::CallScope call(x);
    CF_TRY(call.enter(m->device, st));
    const int64_t tiles = cf::ceil_div(n_windows, cf::kTileWindows);
    cf::WindowTable tab;
    CF_TRY(cf::ensure_table(x, tiles, &tab));
    const int64_t slots = tiles * cf::kTileWindows;
    cf::dense_window_table_kernel<<<(unsigned)cf::ceil_div(slots, 256), 256, 0, st>>>(n_windows, slots, tab.src, tab.valid, tab.read);
    CF_LAUNCHED();
    return cf::engine_forward(m, x, nullptr, nullptr, x_dev, tab, tiles, probs_dev, st);
}

// The forward pass of the validation row: the logits of n_windows dense windows into x->val_logits, then K9 over
// all n_windows * 35 positions at `threshold`.  *result (device): tp, fp, tn, fn, correct (int64) | loss sum (double).
static int validate_forward(cf_model* m, cf::Exec* x, const float* x_dev, const uint8_t* labels_dev, int64_t n_windows,
                            double threshold, cudaStream_t st, const long long** result) {
    const int64_t n = n_windows * cf::kWindow;
    const int64_t tiles = cf::ceil_div(n_windows, cf::kTileWindows);
    const int blocks = cf::k9_validation_blocks(n);
    CF_TRY(x->val_logits.ensure(sizeof(float) * (size_t)n));
    CF_TRY(x->val_partial.ensure(sizeof(long long) * 6 * ((size_t)blocks + 1)));
    cf::WindowTable tab;
    CF_TRY(cf::ensure_table(x, tiles, &tab));
    const int64_t slots = tiles * cf::kTileWindows;
    cf::dense_window_table_kernel<<<(unsigned)cf::ceil_div(slots, 256), 256, 0, st>>>(n_windows, slots, tab.src, tab.valid, tab.read);
    CF_LAUNCHED();
    CF_TRY(cf::engine_forward(m, x, nullptr, nullptr, x_dev, tab, tiles, x->val_logits.as<float>(), st,
                              /*want_logits=*/true));
    long long* partial = x->val_partial.as<long long>();
    long long* res = partial + (size_t)blocks * 6;
    CF_TRY(cf::k9_validate(x->val_logits.as<float>(), labels_dev, n, threshold, partial, res, st));
    *result = res;
    return CF_OK;
}

// K9's accuracy and mean loss from its result (host copy) over n positions.
static void validate_means(const long long* host, int64_t n, double* accuracy_out, double* loss_out) {
    double loss_sum;
    std::memcpy(&loss_sum, &host[5], sizeof(double));
    if (accuracy_out) *accuracy_out = (double)host[4] / (double)n;
    if (loss_out) *loss_out = loss_sum / (double)n;
}

// K11's counts (sorted-threshold order) to the caller's threshold order, tn minus tn_shift.
static void sweep_scatter(const std::vector<long long>& sorted_counts, const std::vector<int>& index, int64_t tn_shift,
                          int64_t* out) {
    for (size_t i = 0; i < index.size(); ++i) {
        const long long* c = sorted_counts.data() + 4 * (size_t)index[i];
        out[4 * i + 0] = c[0];
        out[4 * i + 1] = c[1];
        out[4 * i + 2] = c[2] - tn_shift;
        out[4 * i + 3] = c[3];
    }
}

int cf_validate_windows(cf_model* m, const float* x_dev, const uint8_t* labels_dev, int64_t n_windows,
                        int64_t padding_size, double threshold, int64_t* counts_out, double* accuracy_out,
                        double* loss_out, void* stream) {
    if (!m || n_windows <= 0 || !x_dev || !labels_dev || padding_size < 0 || !counts_out) {
        cf::set_error("cf_validate_windows: bad argument");
        return CF_ERR_BAD_ARG;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cf::Exec* x = m->def.get();
    cf::CallScope call(x);
    CF_TRY(call.enter(m->device, st));
    const long long* result;
    CF_TRY(validate_forward(m, x, x_dev, labels_dev, n_windows, threshold, st, &result));
    long long host[6];
    CF_CUDA(cudaMemcpyAsync(host, result, sizeof(host), cudaMemcpyDeviceToHost, st));
    CF_CUDA(cudaStreamSynchronize(st));
    counts_out[0] = host[0];
    counts_out[1] = host[1];
    counts_out[2] = host[2] - padding_size;      // rnn_class.py:247
    counts_out[3] = host[3];
    validate_means(host, n_windows * cf::kWindow, accuracy_out, loss_out);
    return CF_OK;
}

int cf_validate_windows_sweep(cf_model* m, const float* x_dev, const uint8_t* labels_dev, int64_t n_windows,
                              int64_t padding_size, const double* thresholds_host, int32_t n_thresholds,
                              int64_t* counts_out_host, double* accuracy_out, double* loss_out, void* stream) {
    if (!m || n_windows <= 0 || !x_dev || !labels_dev || padding_size < 0 || !counts_out_host) {
        cf::set_error("cf_validate_windows_sweep: bad argument");
        return CF_ERR_BAD_ARG;
    }
    std::vector<float> sorted;
    std::vector<int> index;
    CF_TRY(cf::k11_prepare_thresholds(thresholds_host, n_thresholds, &sorted, &index));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cf::Exec* x = m->def.get();
    cf::CallScope call(x);
    CF_TRY(call.enter(m->device, st));
    CF_TRY(x->val_sweep.ensure(cf::k11_scratch_bytes((int)sorted.size())));
    const long long* result;
    // K9's counts at 0.5 are not used: it runs for the accuracy and the loss, which no threshold changes
    CF_TRY(validate_forward(m, x, x_dev, labels_dev, n_windows, 0.5, st, &result));
    const int64_t n = n_windows * cf::kWindow;
    std::vector<long long> counts(4 * sorted.size());
    CF_TRY(cf::k11_sweep(x->val_logits.as<float>(), true, labels_dev, n, sorted, x->val_sweep.ptr, counts.data(), st));
    long long host[6];
    CF_CUDA(cudaMemcpyAsync(host, result, sizeof(host), cudaMemcpyDeviceToHost, st));
    CF_CUDA(cudaStreamSynchronize(st));
    sweep_scatter(counts, index, padding_size, counts_out_host);      // rnn_class.py:247 at every threshold
    validate_means(host, n, accuracy_out, loss_out);
    return CF_OK;
}

int cf_sweep_thresholds(int32_t device, const float* values_dev, int32_t values_are_logits, const uint8_t* labels_dev,
                        int64_t n, const double* thresholds_host, int32_t n_thresholds, int64_t* counts_out_host,
                        void* stream) {
    if (n < 0 || !counts_out_host || (n > 0 && (!values_dev || !labels_dev))) {
        cf::set_error("cf_sweep_thresholds: bad argument");
        return CF_ERR_BAD_ARG;
    }
    std::vector<float> sorted;
    std::vector<int> index;
    CF_TRY(cf::k11_prepare_thresholds(thresholds_host, n_thresholds, &sorted, &index));
    if (n == 0) {
        std::fill(counts_out_host, counts_out_host + 4 * (size_t)n_thresholds, 0);
        return CF_OK;
    }
    cf::DeviceGuard guard;
    CF_TRY(guard.set(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cf::DevBuf scratch;
    CF_TRY(scratch.ensure(cf::k11_scratch_bytes((int)sorted.size())));
    std::vector<long long> counts(4 * sorted.size());
    const int s = cf::k11_sweep(values_dev, values_are_logits != 0, labels_dev, n, sorted, scratch.ptr, counts.data(), st);
    const cudaError_t e = cudaStreamSynchronize(st);    // scratch is freed on return, also after a failed launch
    CF_TRY(s);
    if (e != cudaSuccess) {
        cf::set_error("cf_sweep_thresholds: %s", cudaGetErrorString(e));
        return CF_ERR_CUDA;
    }
    sweep_scatter(counts, index, 0, counts_out_host);
    return CF_OK;
}

int cf_vote_events(int32_t device, const double* scores_dev, int64_t n_scores, const int64_t* event_lengths_host,
                   int64_t n_events, int64_t start, int64_t length, int32_t* classes_dev, int64_t* n_voted_out,
                   int64_t* start_event_out, int64_t* final_event_out, int32_t* empty_event_out, void* stream) {
    if (n_scores < 0 || n_events < 0 || (n_events > 0 && !event_lengths_host) || (n_scores > 0 && !scores_dev) ||
        !n_voted_out || !start_event_out || !final_event_out) {
        cf::set_error("cf_vote_events: bad argument");
        return CF_ERR_BAD_ARG;
    }
    // the control flow of the reference's loop (networks/correct_output.py:43-61) on the scanned lengths
    std::vector<int64_t> begin((size_t)n_events + 1, 0);
    int64_t start_event = -1, final_event = -2, n_voted = 0, summed = 0;
    for (int64_t n = 0; n < n_events; ++n) {
        begin[n] = summed;
        if (start_event < 0 && summed >= start) start_event = n;
        summed += event_lengths_host[n];
        begin[n + 1] = summed;
        if (summed > length) { final_event = n - 1; break; }
        if (start_event >= 0) {
            ++n_voted;
            if (summed == start + length) { final_event = n; break; }
        }
    }
    *n_voted_out = n_voted;
    *start_event_out = start_event;
    *final_event_out = final_event;
    if (empty_event_out) *empty_event_out = 0;
    if (n_voted == 0) return CF_OK;
    if (!classes_dev) { cf::set_error("cf_vote_events: classes_dev is NULL"); return CF_ERR_BAD_ARG; }
    cf::DeviceGuard guard;
    CF_TRY(guard.set(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cf::DevBuf ev, flag;
    CF_TRY(ev.ensure(sizeof(int64_t) * (size_t)(n_voted + 1)));
    CF_TRY(flag.ensure(sizeof(int32_t)));
    CF_CUDA(cudaMemcpyAsync(ev.ptr, begin.data() + start_event, sizeof(int64_t) * (size_t)(n_voted + 1),
                            cudaMemcpyHostToDevice, st));
    CF_TRY(cf::k10_vote_events(scores_dev, n_scores, ev.as<int64_t>(), 0, n_voted, classes_dev, flag.as<int32_t>(), st));
    int32_t empty = 0;
    CF_CUDA(cudaMemcpyAsync(&empty, flag.ptr, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CF_CUDA(cudaStreamSynchronize(st));
    if (empty_event_out) *empty_event_out = empty;
    return CF_OK;
}

static int infer_reads_call(const char* name, cf_model* m, cf::Exec* x, const int16_t* raw_dev,
                            const int64_t* offsets_host, int32_t n_reads, float* probs_dev, int64_t* intervals_dev,
                            int64_t* interval_offsets_dev, int64_t capacity, double threshold, int32_t min_run,
                            int32_t ext_left, int32_t ext_right, void* stream) {
    if (!m || n_reads < 0 || !offsets_host || !interval_offsets_dev || capacity < 0 ||
        (n_reads > 0 && !raw_dev) || (capacity > 0 && !intervals_dev)) {
        cf::set_error("%s: bad argument", name);
        return CF_ERR_BAD_ARG;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cf::CallScope call(x);
    CF_TRY(call.enter(m->device, st));
    return cf::infer_reads_device(m, x, raw_dev, offsets_host, n_reads, probs_dev, intervals_dev,
                                  interval_offsets_dev, capacity, threshold, min_run, ext_left, ext_right, st);
}

int cf_infer_reads(cf_model* m, const int16_t* raw_dev, const int64_t* offsets_host, int32_t n_reads,
                   float* probs_dev, int64_t* intervals_dev, int64_t* interval_offsets_dev,
                   int64_t capacity, double threshold, int32_t min_run, int32_t ext_left,
                   int32_t ext_right, void* stream) {
    return infer_reads_call("cf_infer_reads", m, m ? m->def.get() : nullptr, raw_dev, offsets_host, n_reads, probs_dev,
                            intervals_dev, interval_offsets_dev, capacity, threshold, min_run, ext_left, ext_right,
                            stream);
}

int cf_exec_infer_reads(cf_exec* ex, const int16_t* raw_dev, const int64_t* offsets_host, int32_t n_reads,
                        float* probs_dev, int64_t* intervals_dev, int64_t* interval_offsets_dev,
                        int64_t capacity, double threshold, int32_t min_run, int32_t ext_left,
                        int32_t ext_right, void* stream) {
    return infer_reads_call("cf_exec_infer_reads", ex ? ex->model : nullptr, ex ? &ex->x : nullptr, raw_dev,
                            offsets_host, n_reads, probs_dev, intervals_dev, interval_offsets_dev, capacity, threshold,
                            min_run, ext_left, ext_right, stream);
}

int64_t cf_max_intervals(int64_t total_samples, int32_t n_reads, int32_t min_run) {
    if (total_samples < 0 || n_reads < 0) return 0;
    const int64_t mr = min_run < 1 ? 1 : min_run;
    // a run of >= mr ones needs a zero (or a read boundary) before the next one
    return total_samples / (mr + 1) + n_reads + 1;
}

int cf_infer_reads_host(cf_model* m, const int16_t* raw_host, const int64_t* offsets_host, int32_t n_reads,
                        float* probs_host, int64_t* intervals_host, int64_t* interval_offsets_host,
                        int64_t capacity, double threshold, int32_t min_run, int32_t ext_left,
                        int32_t ext_right, int64_t* n_intervals_out, void* stream) {
    if (!m || n_reads < 0 || !offsets_host || !interval_offsets_host || capacity < 0 ||
        (n_reads > 0 && !raw_host) || (capacity > 0 && !intervals_host)) {
        cf::set_error("cf_infer_reads_host: bad argument");
        return CF_ERR_BAD_ARG;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cf::Exec* x = m->def.get();
    cf::CallScope call(x);
    CF_TRY(call.enter(m->device, st));
    const int64_t base = n_reads > 0 ? offsets_host[0] : 0;
    const int64_t total = n_reads > 0 ? offsets_host[n_reads] - base : 0;
    if (total < 0) { cf::set_error("cf_infer_reads_host: offsets decrease"); return CF_ERR_BAD_ARG; }
    CF_TRY(x->h_raw.ensure(sizeof(int16_t) * (size_t)(total > 0 ? total : 1)));
    CF_TRY(x->h_intervals.ensure(sizeof(int64_t) * 2 * (size_t)(capacity > 0 ? capacity : 1)));
    CF_TRY(x->h_ioff.ensure(sizeof(int64_t) * ((size_t)n_reads + 1)));
    float* probs_dev = nullptr;
    if (probs_host) {
        CF_TRY(x->h_probs.ensure(sizeof(float) * (size_t)(total > 0 ? total : 1)));
        probs_dev = x->h_probs.as<float>();
    }
    // offsets rebased so that raw_dev + offsets[0] is the staged copy
    std::vector<int64_t> off((size_t)n_reads + 1);
    for (int32_t i = 0; i <= n_reads; ++i) off[i] = offsets_host[i] - base;
    {
        cf::BatchPlan whole;                       // reject bad / empty reads before any asynchronous copy reads the caller's buffer
        CF_TRY(cf::make_plan(off.data(), n_reads, &whole));
    }
    // (Cutting the batch into groups of whole passes whose copies overlap the previous group's kernels was
    // measured: no gain - the copy is 1.2-1.5 ms of a 75 ms step and the extra K1 / K6 sequences cost as much.)
    if (total > 0)
        CF_CUDA(cudaMemcpyAsync(x->h_raw.ptr, raw_host + base, sizeof(int16_t) * (size_t)total, cudaMemcpyHostToDevice, st));
    CF_TRY(cf::infer_reads_device(m, x, x->h_raw.as<int16_t>(), off.data(), n_reads, probs_dev,
                                  x->h_intervals.as<int64_t>(), x->h_ioff.as<int64_t>(), capacity, threshold,
                                  min_run, ext_left, ext_right, st));
    CF_CUDA(cudaMemcpyAsync(interval_offsets_host, x->h_ioff.ptr, sizeof(int64_t) * ((size_t)n_reads + 1),
                            cudaMemcpyDeviceToHost, st));
    CF_CUDA(cudaStreamSynchronize(st));
    const int64_t found = interval_offsets_host[n_reads];
    if (n_intervals_out) *n_intervals_out = found;
    const int64_t ncopy = found < capacity ? found : capacity;
    if (ncopy > 0)
        CF_CUDA(cudaMemcpyAsync(intervals_host, x->h_intervals.ptr, sizeof(int64_t) * 2 * (size_t)ncopy,
                                cudaMemcpyDeviceToHost, st));
    if (probs_host && total > 0)
        CF_CUDA(cudaMemcpyAsync(probs_host, probs_dev, sizeof(float) * (size_t)total, cudaMemcpyDeviceToHost, st));
    CF_CUDA(cudaStreamSynchronize(st));
    if (found > capacity) {
        cf::set_error("cf_infer_reads_host: %lld intervals found, capacity %lld", (long long)found, (long long)capacity);
        return CF_ERR_CAPACITY;
    }
    return CF_OK;
}


int cf_normalize_reads(int32_t device, const int16_t* raw_dev, const int64_t* offsets_host, int32_t n_reads,
                       double* stats_dev, double* norm_dev, void* stream) {
    if (n_reads < 0 || !offsets_host || (n_reads > 0 && !raw_dev)) {
        cf::set_error("cf_normalize_reads: bad argument");
        return CF_ERR_BAD_ARG;
    }
    if (n_reads == 0) return CF_OK;
    cf::DeviceGuard guard;
    CF_TRY(guard.set(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    for (int32_t r = 0; r < n_reads; ++r)
        if (offsets_host[r + 1] < offsets_host[r]) { cf::set_error("cf_normalize_reads: offsets decrease"); return CF_ERR_BAD_ARG; }
    cf::DevBuf off, flags, wide, chunked, chunk_tab, stats_tmp;
    CF_TRY(upload_offsets(offsets_host, n_reads, &off, st));
    double* stats = stats_dev;
    if (!stats) {
        CF_TRY(stats_tmp.ensure(sizeof(double) * 2 * (size_t)n_reads));
        stats = stats_tmp.as<double>();
    }
    const int16_t* raw0 = raw_dev + offsets_host[0];
    cf::StatsScratch sc{&flags, &wide, &chunked, &chunk_tab};
    CF_TRY(cf::compute_read_stats(raw0, offsets_host, off.as<int64_t>(), n_reads, stats, sc, st));
    if (norm_dev)
        CF_TRY(cf::k1_normalize_f64(raw0, off.as<int64_t>(), n_reads, offsets_host[n_reads] - offsets_host[0],
                                    stats, norm_dev, st));
    CF_CUDA(cudaStreamSynchronize(st));      // scratch is freed on return
    return CF_OK;
}

int cf_call_intervals(int32_t device, const void* probs_dev, int32_t probs_is_f64, const int64_t* offsets_host,
                      int32_t n_reads, int64_t* intervals_dev, int64_t* interval_offsets_dev, int64_t capacity,
                      double threshold, int32_t min_run, int32_t ext_left, int32_t ext_right, void* stream) {
    if (n_reads < 0 || !offsets_host || !interval_offsets_dev || capacity < 0 || (capacity > 0 && !intervals_dev)) {
        cf::set_error("cf_call_intervals: bad argument");
        return CF_ERR_BAD_ARG;
    }
    cf::DeviceGuard guard;
    CF_TRY(guard.set(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    for (int32_t r = 0; r < n_reads; ++r)
        if (offsets_host[r + 1] < offsets_host[r]) { cf::set_error("cf_call_intervals: offsets decrease"); return CF_ERR_BAD_ARG; }
    const int64_t total = offsets_host[n_reads] - offsets_host[0];
    if (total > 0 && !probs_dev) { cf::set_error("cf_call_intervals: probs is NULL"); return CF_ERR_BAD_ARG; }
    const char* base = static_cast<const char*>(probs_dev) + (size_t)offsets_host[0] * (probs_is_f64 ? 8 : 4);
    return model_free_intervals(base, probs_is_f64 ? cf::BITS_FROM_F64 : cf::BITS_FROM_F32, threshold, 1, offsets_host,
                                n_reads, intervals_dev, interval_offsets_dev, nullptr, capacity, min_run, ext_left,
                                ext_right, st);
}

int cf_class_from_threshold(int32_t device, const double* scores_dev, int64_t n, double threshold,
                            int64_t* labels_dev, void* stream) {
    if (n < 0 || (n > 0 && (!scores_dev || !labels_dev))) { cf::set_error("cf_class_from_threshold: bad argument"); return CF_ERR_BAD_ARG; }
    cf::DeviceGuard guard;
    CF_TRY(guard.set(device));
    return cf::k6_class_from_threshold(scores_dev, n, threshold, labels_dev, static_cast<cudaStream_t>(stream));
}

int cf_correct_short(int32_t device, const int64_t* labels_dev, int64_t n, int32_t threshold, int64_t* out_dev,
                     void* stream) {
    if (n < 0 || (n > 0 && (!labels_dev || !out_dev)) || labels_dev == out_dev && n > 0) {
        cf::set_error("cf_correct_short: bad argument");
        return CF_ERR_BAD_ARG;
    }
    cf::DeviceGuard guard;
    CF_TRY(guard.set(device));
    return cf::k6_correct_short(labels_dev, n, threshold, out_dev, static_cast<cudaStream_t>(stream));
}

int cf_hp_in_pred(int32_t device, const int64_t* labels_dev, int64_t n, int32_t ext_left, int32_t ext_right,
                  int64_t label, int64_t* intervals_dev, int64_t capacity, int64_t* n_out_dev, void* stream) {
    if (n < 0 || capacity < 0 || !n_out_dev || (n > 0 && !labels_dev) || (capacity > 0 && !intervals_dev)) {
        cf::set_error("cf_hp_in_pred: bad argument");
        return CF_ERR_BAD_ARG;
    }
    if (n == 0) { cf::set_error("cf_hp_in_pred: empty input (the reference raises IndexError, infer.py:151)"); return CF_ERR_EMPTY_READ; }
    cf::DeviceGuard guard;
    CF_TRY(guard.set(device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cf::DevBuf ioff;
    const int64_t offsets[2] = {0, n};
    CF_TRY(ioff.ensure(sizeof(int64_t) * 2));
    return model_free_intervals(labels_dev, cf::BITS_FROM_I64_EQ, 0.0, label, offsets, 1, intervals_dev,
                                ioff.as<int64_t>(), n_out_dev, capacity, 1, ext_left, ext_right, st);
}

}  // extern "C"
