/*
 * catfish_b200.h - C ABI of the B200-native catfish inference hot path.
 *
 * Every entry point is plain C: pointers, sizes, scalars.  No torch types, no
 * exceptions across the boundary.  Functions return 0 on success or a negative
 * cf_status; cf_last_error() gives the message of the last failure on the
 * calling thread.  Unless stated otherwise "dev" pointers are CUDA device
 * pointers on the model's device, "host" pointers are ordinary host memory, and
 * work is enqueued on `stream` (a cudaStream_t passed as void*, NULL = default
 * stream) without synchronising.
 *
 * Each function names the reference interface it replaces (paths relative to
 * the catfish repository root).
 */
#ifndef CATFISH_B200_H
#define CATFISH_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CF_ABI_VERSION 1

typedef enum cf_status {
    CF_OK = 0,
    CF_ERR_BAD_ARG = -1,      /* NULL pointer, negative size, unsupported hyper-parameter */
    CF_ERR_CUDA = -2,         /* a CUDA runtime call failed */
    CF_ERR_NO_DEVICE = -3,    /* no usable sm_100 device: there is no CPU fallback */
    CF_ERR_EMPTY_READ = -4,   /* a read of length 0: the reference raises IndexError (infer.py:151,184) */
    CF_ERR_CAPACITY = -5,     /* an output buffer is too small */
    CF_ERR_ALLOC = -6         /* workspace allocation failed */
} cf_status;

typedef enum cf_network_type {
    CF_NET_RESNET_RNN = 0,    /* models/resnet_class.py:7-25  */
    CF_NET_RNN = 1,           /* models/rnn_class.py:9-54 used directly (neural_network.py:17-18) */
    CF_NET_RESNET = 2         /* resnet_class.py:23 commented out: conv stack -> dense */
} cf_network_type;

typedef enum cf_engine {
    CF_ENGINE_AUTO = 0,       /* tcgen05 kernels when the shape is supported, else SIMT */
    CF_ENGINE_TCGEN05 = 1,    /* split operands on tcgen05/TMEM (C <= 32, H <= 64, any depth) */
    CF_ENGINE_SIMT = 2        /* fp32 CUDA-core kernels, any shape (on-device cross-check) */
} cf_engine;

/* Hyper-parameters: the constructor kwargs of RNN / ResNetRNN
 * (models/rnn_class.py:10-31, models/resnet_class.py:9-14, neural_network.py:37-67). */
typedef struct cf_model_desc {
    int32_t network_type;     /* cf_network_type */
    int32_t window;           /* 35, rnn_class.py:27 */
    int32_t layer_size;       /* GRU units H */
    int32_t n_layers;         /* stacked bidirectional GRU layers */
    int32_t layer_size_res;   /* conv channels C */
    int32_t n_layers_res;     /* residual blocks */
    float bn_epsilon;         /* 1e-3 */
    int32_t engine;           /* cf_engine */
} cf_model_desc;

typedef struct cf_model cf_model;

/* Library / device probes. */
int cf_abi_version(void);
const char* cf_last_error(void);
int cf_device_count(void);

/*
 * cf_model_create - replaces RNN.__init__ + restore_network
 * (models/rnn_class.py:10-54, 191-198; neural_network.py:8-34).
 * `tensors` are host float32 arrays in TensorFlow layout, in this order:
 *   per residual block b, per conv j = 0..3 (shortcut k1, conv k1, conv k3, conv k1):
 *       conv1d_{4b+j}/kernel [K,Cin,Cout], /bias [Cout],
 *       batch_normalization_{4b+j}/gamma, /beta, /moving_mean, /moving_variance [Cout]
 *   per GRU layer l, per direction fw then bw:
 *       gates/kernel [in+H,2H], gates/bias [2H], candidate/kernel [in+H,H], candidate/bias [H]
 *   final_fully_connected/kernel [F,1], /bias [1]
 * `tensor_sizes[i]` is the element count of tensors[i] and is checked against the
 * shape the descriptor implies.  Weights are folded/re-packed once, here.
 */
int cf_model_create(const cf_model_desc* desc, const float* const* tensors,
                    const int64_t* tensor_sizes, int32_t n_tensors, int32_t device,
                    cf_model** out_model);
void cf_model_destroy(cf_model* model);

/* Number of weight tensors cf_model_create expects for `desc` (negative on bad desc). */
int cf_model_num_tensors(const cf_model_desc* desc);

/* Which engine the handle resolved to (cf_engine value). */
int cf_model_engine(const cf_model* model);
/* Tensor-core operand format of the handle: 0 = split bf16, three MMA passes ("bf16x3"); 1 = fp16 main
 * product + e5m2 correction product, two pass-equivalents ("f16e5"; chosen when every tensor-core kernel
 * of the pass supports it and the GRU weights fit fp16's range); -1 = fp32 CUDA-core engine. */
int cf_model_operand_format(const cf_model* model);

/* Pre-size the handle's buffers and engine workspaces (tensor-core engine: up to ~12.6 GB at a full pass
 * of 2368 tiles) for calls of at most max_samples samples / max_reads reads, so that such calls do not
 * allocate.  Optional: otherwise the first call that needs more allocates it. */
int cf_model_reserve(cf_model* model, int64_t max_samples, int32_t max_reads);

/*
 * cf_infer_windows - replaces RNN.infer / ResNetRNN.infer
 * (models/rnn_class.py:213-219, called from infer.py:44).
 * x_dev:     float32 [n_windows, 35] (the [B,35,1] placeholder feed), device
 * probs_dev: float32 [n_windows * 35], window-major then position, device
 */
int cf_infer_windows(cf_model* model, const float* x_dev, int64_t n_windows,
                     float* probs_dev, void* stream);

/*
 * cf_infer_reads - replaces infer.infer_class_from_signal (infer.py:12-51) for a
 * ragged batch of reads whose raw signal is already on the device (the FAST5
 * decode of process_signal, infer.py:77-90, stays on the host).
 *   raw_dev          int16, reads concatenated, device
 *   offsets_host     int64 [n_reads+1], host; read r = raw[offsets[r] : offsets[r+1]]
 *   probs_dev        float32 [total samples] or NULL: per-position probabilities with the
 *                    padding already cut (infer.py:47), in read order
 *   intervals_dev    int64 [capacity][2]: [start - ext_left, start + len + ext_right) of every
 *                    positive run of length >= min_run, read-local coordinates, unclamped,
 *                    unmerged, increasing start (infer.py:48-49, 141-162, 174-198)
 *   interval_offsets_dev int64 [n_reads+1]: CSR offsets of each read's intervals;
 *                    element n_reads is the total (compare with capacity)
 *   threshold        class_from_threshold's threshold (infer.py:128), compared in double
 * Defaults of the reference: threshold 0.5, min_run 15, ext_left 11, ext_right 16.
 */
int cf_infer_reads(cf_model* model, const int16_t* raw_dev, const int64_t* offsets_host,
                   int32_t n_reads, float* probs_dev, int64_t* intervals_dev,
                   int64_t* interval_offsets_dev, int64_t capacity, double threshold,
                   int32_t min_run, int32_t ext_left, int32_t ext_right, void* stream);

/*
 * cf_infer_reads_host - the same call with HOST buffers: copies the signal to the
 * device, runs cf_infer_reads, copies results back and synchronises.  This is the
 * end-to-end path the Python per-read entry points use.  probs_host may be NULL.
 * *n_intervals_out receives the total number of intervals found; if it exceeds
 * `capacity` the call returns CF_ERR_CAPACITY after filling the first `capacity`.
 */
int cf_infer_reads_host(cf_model* model, const int16_t* raw_host, const int64_t* offsets_host,
                        int32_t n_reads, float* probs_host, int64_t* intervals_host,
                        int64_t* interval_offsets_host, int64_t capacity, double threshold,
                        int32_t min_run, int32_t ext_left, int32_t ext_right,
                        int64_t* n_intervals_out, void* stream);

/*
 * Execution contexts (no reference counterpart): concurrent inference on one model.
 *
 * A model handle holds the weights, which no call changes, and one default context: the scratch
 * buffers, workspaces and completion event that every cf_model_* / cf_infer_* / cf_validate_* call
 * above uses.  Calls on the default context are serialised on the device, whatever their streams.
 * A cf_exec is one more such context of the same model, with buffers of its own:
 *   - calls on one context are serialised on the device as calls on the handle are (each waits for
 *     the previous call's work on that context, on any stream); they may come from any thread, one
 *     at a time (a context holds a mutex for the duration of a call);
 *   - calls on different contexts of one model, and calls on the default context, may overlap on
 *     the device when they are enqueued on different streams;
 *   - a context's buffers and engine workspaces grow to the largest batch it has run
 *     (cf_exec_reserve pre-sizes all of them) and are freed by cf_exec_destroy;
 *   - a context holds a reference on its model: cf_model_destroy while contexts are alive releases
 *     the handle's own buffers, and the weights are freed when the last context is destroyed;
 *   - context calls are not timed by cf_profile_* (which covers the default context only).
 * The caller's current device is restored by every call.
 */
typedef struct cf_exec cf_exec;
/* A new context on the model's device (allocates nothing until its first call). */
int cf_exec_create(cf_model* model, cf_exec** out);
/* Waits for the context's last work, then frees its buffers (and the model, if it was the last reference). */
void cf_exec_destroy(cf_exec* ex);
/* cf_model_reserve on a context: pre-sizes its buffers and engine workspaces. */
int cf_exec_reserve(cf_exec* ex, int64_t max_samples, int32_t max_reads);
/* cf_infer_reads on a context: same arguments after the model, same semantics and outputs; asynchronous. */
int cf_exec_infer_reads(cf_exec* ex, const int16_t* raw_dev, const int64_t* offsets_host,
                        int32_t n_reads, float* probs_dev, int64_t* intervals_dev,
                        int64_t* interval_offsets_dev, int64_t capacity, double threshold,
                        int32_t min_run, int32_t ext_left, int32_t ext_right, void* stream);

/* Upper bound on the number of intervals cf_infer_reads can emit. */
int64_t cf_max_intervals(int64_t total_samples, int32_t n_reads, int32_t min_run);

/*
 * cf_normalize_reads - replaces infer.normalize_raw_signal(raw, "median")
 * (infer.py:96-105; duplicate networks/trainingDB/helper_functions.py:87-98).
 *   stats_dev  double [n_reads][2] = (shift, scale) = (median, median |raw - median|), or NULL
 *   norm_dev   double [total samples] = (raw - shift) / scale, or NULL
 * Needs no model: pass device explicitly.  Scratch is allocated and freed inside.
 */
int cf_normalize_reads(int32_t device, const int16_t* raw_dev, const int64_t* offsets_host,
                       int32_t n_reads, double* stats_dev, double* norm_dev, void* stream);

/*
 * cf_call_intervals - threshold + short-run removal + interval emission on given
 * probabilities: class_from_threshold -> correct_short -> hp_in_pred
 * (infer.py:128-138, 174-198, 141-162) for a ragged batch.  Arguments as cf_infer_reads;
 * probs_dev is float32 (probs_is_f64 = 0) or float64 (1).
 */
int cf_call_intervals(int32_t device, const void* probs_dev, int32_t probs_is_f64,
                      const int64_t* offsets_host, int32_t n_reads, int64_t* intervals_dev,
                      int64_t* interval_offsets_dev, int64_t capacity, double threshold,
                      int32_t min_run, int32_t ext_left, int32_t ext_right, void* stream);

/* class_from_threshold (infer.py:128-138): labels[i] = scores[i] >= threshold ? 1 : 0. */
int cf_class_from_threshold(int32_t device, const double* scores_dev, int64_t n, double threshold,
                            int64_t* labels_dev, void* stream);

/* correct_short (infer.py:174-198): every run of equal non-zero labels shorter than
 * `threshold` becomes 0.  in/out may not alias. */
int cf_correct_short(int32_t device, const int64_t* labels_dev, int64_t n, int32_t threshold,
                     int64_t* out_dev, void* stream);

/* hp_in_pred (infer.py:141-162): [start - ext_left, start + len + ext_right] for every run
 * of `label`.  *n_out_dev (device int64) receives the count; at most `capacity` are written. */
int cf_hp_in_pred(int32_t device, const int64_t* labels_dev, int64_t n, int32_t ext_left,
                  int32_t ext_right, int64_t label, int64_t* intervals_dev, int64_t capacity,
                  int64_t* n_out_dev, void* stream);

/*
 * Per-kernel-class device timing (no reference counterpart; used by bench.py for the roofline).
 * When enabled, every launch group is bracketed by CUDA events on the launching stream;
 * cf_profile_read waits for them and returns accumulated milliseconds and launch counts per
 * class (arrays of at least cf_profile_num_classes() elements).  Enabling resets the counters.
 */
int cf_profile_enable(cf_model* model, int32_t on);
int cf_profile_num_classes(void);
const char* cf_profile_class_name(int32_t cls);
int cf_profile_read(cf_model* model, double* ms_out, int64_t* launches_out, int32_t n);

/*
 * cf_merge_chunks - "next" row N1: replaces the chunk merging of the reference's CLI loop
 * (catfish/catfish:58-81) and center_hp (catfish/catfish:121-135) for a batch of reads.
 *   intervals_dev / interval_offsets_host : the CSR output of cf_infer_reads (offsets on the host)
 *   read_lengths_host [n_reads]           : len_read of every read
 *   merged_dev  int64 [(n_intervals + n_reads)][2] : read r's merged chunks start at row offsets[r] + r
 *   nonhp_dev   int64 [(n_intervals + 2 n_reads)][2]: read r's non-HP ranges start at row offsets[r] + 2 r
 *   merged_count_dev / nonhp_count_dev int64 [n_reads]; nonhp_count -1 marks a read without any
 *   interval (the reference then stores the single odd entry [((0, len_read), len_read)], :81).
 * Reproduces the reference's list aliasing and the `i - 1` wrap-around at i == 0.  Synchronises.
 */
int cf_merge_chunks(int32_t device, const int64_t* intervals_dev, const int64_t* interval_offsets_host,
                    const int64_t* read_lengths_host, int32_t n_reads, int64_t chunk_size, int64_t* merged_dev,
                    int64_t* merged_count_dev, int64_t* nonhp_dev, int64_t* nonhp_count_dev, void* stream);

/*
 * cf_split_raw - "next" row N2: the computation inside split_f5.split_signal
 * (catfish/split_f5.py:36,64: `new_signal = signal_dset[s[0] : s[1]]`) for a batch of ranges.
 *   raw_dev / offsets_host [n_reads+1] : the reads, concatenated int16 on the device
 *   ranges_dev int64 [n_ranges][2], range_read_dev int32 [n_ranges] : (start, end) in read-local
 *                 coordinates and the read each range cuts; numpy slice semantics (negative bounds count
 *                 from the end, bounds clamp to the read, inverted ranges are empty)
 *   out_dev int16 [capacity] : the pieces, concatenated in range order
 *   piece_offsets_dev int64 [n_ranges+1] : start of every piece in out_dev; last element = total
 * Pieces that would exceed `capacity` are truncated (compare the total with capacity).  Synchronises.
 * HDF5 / gzip writing of the pieces stays on the host.
 */
int cf_split_raw(int32_t device, const int16_t* raw_dev, const int64_t* offsets_host, int32_t n_reads,
                 const int64_t* ranges_dev, const int32_t* range_read_dev, int64_t n_ranges, int16_t* out_dev,
                 int64_t capacity, int64_t* piece_offsets_dev, void* stream);

/*
 * cf_validate_windows - "next" row N4: one call of RNN.test_network (networks/rnn_class.py:222-261)
 * without its file writing: forward pass over n_windows dense windows (padding included, as
 * train_validate.padding :51-64 produced them), then on ALL n_windows*35 positions
 *   pred = 1 if sigmoid(logit) >= threshold else 0                      (rnn_class.py:235)
 *   counts_out[4] = tp, fp, tn - padding_size, fn                       (metrics.confusion_matrix,
 *                   networks/trainingDB/metrics.py:10-37; the tn correction is rnn_class.py:247)
 *   *accuracy_out = mean(round_half_even(sigmoid(logit)) == label)      (compute_accuracy :80-86)
 *   *loss_out     = mean(max(z,0) - z*label + log1p(exp(-|z|)))         (compute_loss :72-77)
 * x_dev float32 [n_windows][35] and labels_dev uint8 [n_windows*35] live on the device; the three
 * outputs are host pointers (accuracy_out / loss_out may be NULL).  Synchronises.  The caller
 * accumulates the counts over reads as the reference does in self.tp/fp/tn/fn (:244-248).
 */
int cf_validate_windows(cf_model* model, const float* x_dev, const uint8_t* labels_dev, int64_t n_windows,
                        int64_t padding_size, double threshold, int64_t* counts_out, double* accuracy_out,
                        double* loss_out, void* stream);

/*
 * Threshold sweeps (K11; the reference's networks/precision_recall_ROC.py thresholds the scores once per point):
 * confusion counts at up to 4096 thresholds from one pass over the scores.  A position is predicted 1 at
 * threshold t when (double)p >= t (class_from_threshold, infer.py:128); NaN scores are predicted 0 at every
 * threshold; labels other than 0 / 1 count as metrics.confusion_matrix counts them (a positive is a TP only for
 * label 1, a negative a TN only for label 0).  thresholds_host may be unsorted and may repeat; 1 <= n_thresholds
 * <= 4096 and no threshold NaN, else CF_ERR_BAD_ARG.  counts_out_host int64 [n_thresholds][4] = tp, fp, tn, fn,
 * in the caller's threshold order.  Integer counts: the result is exact and deterministic.
 */
/* Confusion counts at T thresholds over n positions.  values_dev holds probabilities (values_are_logits = 0) or
 * logits (1; p = 1 / (1 + exp(-z)) in fp32, as K9 and the head kernels).  labels_dev uint8 [n].  Needs no model:
 * scratch is allocated and freed inside.  Synchronises. */
int cf_sweep_thresholds(int32_t device, const float* values_dev, int32_t values_are_logits, const uint8_t* labels_dev,
                        int64_t n, const double* thresholds_host, int32_t n_thresholds, int64_t* counts_out_host,
                        void* stream);

/* cf_validate_windows at T thresholds, one forward pass: per threshold tn has padding_size subtracted
 * (rnn_class.py:247); accuracy / loss do not depend on the threshold and are returned once (either may be NULL).
 * Runs on the model's default context.  Synchronises. */
int cf_validate_windows_sweep(cf_model* model, const float* x_dev, const uint8_t* labels_dev, int64_t n_windows,
                              int64_t padding_size, const double* thresholds_host, int32_t n_thresholds,
                              int64_t* counts_out_host, double* accuracy_out, double* loss_out, void* stream);

/*
 * cf_vote_events - "next" row N3: the arithmetic of correct_events (networks/correct_output.py:38-61,
 * unfinished in the reference): walk the events as the reference's loop does (start found at the
 * first event whose first measurement is >= start; stop before the event that would pass `length`,
 * or after the one that ends at start + length) and give every visited event the class
 * round_half_even(mean(scores[event begin : event end])).
 *   scores_dev float64 [n_scores] (device); event_lengths_host int64 [n_events] (host)
 *   classes_dev int32 [>= *n_voted_out] (device; n_events is always enough)
 *   *start_event_out / *final_event_out : as the reference's variables; where the reference would
 *                 leave them unbound, start_event is -1 and final_event is -2 (-1 is a legitimate
 *                 final_event when the very first event already passes `length`); *empty_event_out != 0 when an event had no score (the
 *                 reference divides by zero there).  Synchronises.
 */
int cf_vote_events(int32_t device, const double* scores_dev, int64_t n_scores, const int64_t* event_lengths_host,
                   int64_t n_events, int64_t start, int64_t length, int32_t* classes_dev, int64_t* n_voted_out,
                   int64_t* start_event_out, int64_t* final_event_out, int32_t* empty_event_out, void* stream);

/*
 * cf_selftest_f16e5 - unit self-test of the fp16 + e5m2-correction MMA pair (no reference counterpart):
 * out[w][n] = sum_k a[w][k] * w[k][n] for one tile of 128 rows, A split on the device into an fp16
 * operand and an e5m2 operand of scaled remainders, placed in shared memory (mode 0) or tensor memory
 * (mode 1); B packed on the host.  a_dev float32 [128][k], w_host [k][n], out_dev float32 [128][n];
 * k in {16, 32, 48, 64}, n a multiple of 16 up to 128.  Synchronises.
 */
int cf_selftest_f16e5(int32_t device, const float* a_dev, int32_t k, int32_t n, const float* w_host, int32_t mode,
                      float* out_dev, void* stream);

/*
 * cf_trainer - RMSProp training of the network (rnn_class.py train_network with tf.train.RMSPropOptimizer), fp32 on
 * CUDA cores.  A trainer owns fp32 variables in TF layout (the tensors of cf_model_create, same order), the optimizer
 * slots <var>/RMSProp (ms) and <var>/RMSProp_1 (mom), and a workspace that only grows.  One step: the inference
 * graph with output dropout on every GRU cell, mean sigmoid cross-entropy over all n_windows * 35 positions, and
 * TF 1.x ApplyRMSProp (decay 0.9, momentum 0, epsilon 1e-10) on every variable but the BN moving statistics.
 * The dropout mask is Philox4x32-10 with key = seed and counter = (step, 2 * layer + direction, window, t * H + unit):
 * a unit is kept when the top 24 bits of output word 0 are < round(keep_prob * 2^24); keep_prob = 1 draws nothing.
 * Calls on one trainer are ordered on the device as calls on one execution context are.  Deterministic: the same
 * inputs give bit-identical variables and slots.
 */
typedef struct cf_trainer cf_trainer;
/* tensors / sizes as cf_model_create; rms / mom parallel to tensors (NULL = fresh slots: ones / zeros; entries of the
 * BN moving statistics are ignored).  desc->engine is ignored. */
int cf_trainer_create(const cf_model_desc* desc, const float* const* tensors, const int64_t* sizes, int32_t n_tensors,
                      const float* const* rms, const float* const* mom, int32_t device, cf_trainer** out);
void cf_trainer_destroy(cf_trainer* trainer);
/* One RMSProp step on x_dev float32 [n_windows][35], labels_dev uint8 [n_windows * 35] in {0, 1}; step in [0, 2^32).
 * loss / accuracy of the step's forward (either may be NULL; non-NULL synchronises).  CF_ERR_BAD_ARG for NULL
 * pointers, n_windows < 1, keep_prob outside (0, 1], a learning_rate that is not finite or <= 0. */
int cf_trainer_step(cf_trainer* trainer, const float* x_dev, const uint8_t* labels_dev, int64_t n_windows,
                    float learning_rate, float keep_prob, uint64_t seed, int64_t step, double* loss_out,
                    double* accuracy_out, void* stream);
/* Gradients of the same step without the update: grads_host parallel to tensors (entries may be NULL; the BN moving
 * statistics are never written).  Synchronises. */
int cf_trainer_gradients(cf_trainer* trainer, const float* x_dev, const uint8_t* labels_dev, int64_t n_windows,
                         float keep_prob, uint64_t seed, int64_t step, float* const* grads_host, double* loss_out,
                         void* stream);
/* Copy variables and slots out (any of the three arrays may be NULL, and any entry of them).  Synchronises. */
int cf_trainer_read(cf_trainer* trainer, float* const* tensors_host, float* const* rms_host, float* const* mom_host);

/* Kernel launches issued by this library since process start (bench.py's gpu_launches). */
int64_t cf_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* CATFISH_B200_H */
