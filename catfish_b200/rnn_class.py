"""Mirror of the reference's ``RNN`` model class, inference only.

Reference: /root/reference/catfish/models/rnn_class.py (``RNN.__init__`` :10-54,
``restore_network`` :191-198, ``initialize_network`` :186-188, ``infer`` :213-219).
Same constructor kwargs, attributes and return types; the TensorFlow graph and
session are replaced by a handle of the C-ABI CUDA library.  ``test_network``
follows the validation twin networks/rnn_class.py:222-261.  Training
(``train_network``, optimizer, TensorBoard) is out of scope and raises.
"""

import ctypes
import os
import threading

import numpy as np

from . import _cabi, weights as _weights


class RNN(object):
    network_type_name = "RNN"           # key for weights.expected_shapes

    def __init__(self, save=False, device=None, engine="auto", **kwargs):
        # adjustable parameters (rnn_class.py:13-19)
        self.batch_size = kwargs["batch_size"]
        self.optimizer_choice = kwargs["optimizer_choice"]
        self.learning_rate = kwargs["learning_rate"]
        self.layer_size = kwargs["layer_size"]
        self.n_layers = kwargs["n_layers"]
        self.keep_prob = kwargs["keep_prob"]
        self.keep_prob_test = 1.0
        # set parameters (rnn_class.py:25-31)
        self.n_inputs = 1
        self.n_outputs = 1
        self.window = 35
        self.layer_sizes = [self.layer_size, ] * self.n_layers
        self.saving_step = 10000
        self.cell_type = "GRU"
        if not hasattr(self, "network_type"):
            self.network_type = self.cell_type
        self.model_type = self.network_type
        if save:
            raise NotImplementedError("training / model saving is out of scope of catfish_b200")
        from . import get_device
        self.device = get_device() if device is None else int(device)
        self.engine = {"auto": _cabi.ENGINE_AUTO, "tcgen05": _cabi.ENGINE_TCGEN05,
                       "simt": _cabi.ENGINE_SIMT}[engine]
        self._handle = None
        self._weights = None
        self.tp = self.fp = self.tn = self.fn = 0
        self.sweep_counts = None        # test_network_sweep's [T, 4] accumulator (reset_sweep)
        # idle slots (infer._Slot: stream, buffers) of infer_reads / evaluate_reads on the default context; a call
        # takes what it needs and puts it back, so concurrent calls never share a buffer
        self._slots = []
        self._slot_lock = threading.Lock()

    # ------------------------------------------------------------------ hyper-parameters
    def _hpm(self):
        return dict(layer_size=self.layer_size, n_layers=self.n_layers,
                    layer_size_res=getattr(self, "layer_size_res", 32),
                    n_layers_res=getattr(self, "n_layers_res", 2))

    def _desc(self):
        nt = {"RNN": _cabi.NET_RNN, "ResNetRNN": _cabi.NET_RESNET_RNN, "ResNet": _cabi.NET_RESNET}
        h = self._hpm()
        return _cabi.ModelDesc(nt[self.network_type_name], self.window, h["layer_size"], h["n_layers"],
                               h["layer_size_res"], h["n_layers_res"], _weights.BN_EPSILON, self.engine)

    # ------------------------------------------------------------------ weights
    def set_weights(self, weights):
        """Install a ``{tf_variable_name: array}`` weight set and (re)build the device handle."""
        w = _weights.check_weights(weights, self.network_type_name, **self._hpm())
        lib = _cabi.load_library()
        self._release()
        names = list(_weights.expected_shapes(self.network_type_name, **self._hpm()).keys())
        arrays = [np.ascontiguousarray(w[n], np.float32) for n in names]
        ptrs = (ctypes.c_void_p * len(arrays))(*[a.ctypes.data for a in arrays])
        sizes = (ctypes.c_int64 * len(arrays))(*[a.size for a in arrays])
        handle = ctypes.c_void_p()
        desc = self._desc()
        _cabi.check(lib.cf_model_create(ctypes.byref(desc), ptrs, sizes, len(arrays), self.device,
                                        ctypes.byref(handle)))
        self._handle = handle
        self._weights = w
        return self

    def get_weights(self):
        return dict(self._weights) if self._weights is not None else None

    def initialize_network(self, seed=0):
        """rnn_class.py:186-188: fresh variables (one seeded draw of the reference's initializers)."""
        return self.set_weights(_weights.random_init(self.network_type_name, seed=seed, **self._hpm()))

    def restore_network(self, path, ckpnt="latest", meta=None):
        """rnn_class.py:191-198: ``path`` is the checkpoint directory, ``ckpnt`` e.g. "ckpnt-30000".

        Reads the TF-V2 bundle ``<path>/<ckpnt>.{index,data-00000-of-00001}`` directly, or a
        ``<path>/<ckpnt>.npz`` of the same tensors."""
        if ckpnt == "latest":
            ckpnt = _latest_checkpoint(path)
        prefix = os.path.join(path, ckpnt)
        if os.path.exists(prefix + ".index"):
            w = _weights.load_tf_checkpoint(prefix)
        elif os.path.exists(prefix + ".npz"):
            w = _weights.load_npz(prefix + ".npz")
        else:
            raise ValueError("checkpoint %s not found" % prefix)
        self.set_weights(w)
        print("Model {} restored\n".format(os.path.normpath(path).split(os.sep)[-2]
                                           if os.sep in os.path.normpath(path) else path))
        return self

    # ------------------------------------------------------------------ inference
    @property
    def handle(self):
        if self._handle is None:
            raise RuntimeError("network has no weights: call restore_network() or initialize_network() first")
        return self._handle

    @property
    def resolved_engine(self):
        return _cabi.ENGINE_NAMES[_cabi.load_library().cf_model_engine(self.handle)]

    @property
    def operand_format(self):
        """"f16e5" (fp16 + e5m2 correction MMAs), "bf16x3" (split bf16) or "f32" (CUDA-core engine)."""
        return {1: "f16e5", 0: "bf16x3"}.get(_cabi.load_library().cf_model_operand_format(self.handle), "f32")

    def infer(self, input_x):
        """rnn_class.py:213-219: ``input_x`` [n_windows, 35, 1] -> float64 [n_windows * 35]."""
        import torch
        x = np.ascontiguousarray(np.asarray(input_x, dtype=np.float32))
        if x.ndim != 3 or x.shape[1] != self.window or x.shape[2] != self.n_inputs:
            raise ValueError("Cannot feed value of shape %s for Tensor 'data/Placeholder:0', "
                             "which has shape '(?, %d, %d)'" % (x.shape, self.window, self.n_inputs))
        n_windows = x.shape[0]
        dev = torch.device("cuda", self.device)
        with torch.cuda.device(dev):
            xd = torch.from_numpy(x.reshape(n_windows, self.window)).to(dev)
            pd = torch.empty(n_windows * self.window, dtype=torch.float32, device=dev)
            stream = torch.cuda.current_stream(dev)
            _cabi.check(_cabi.load_library().cf_infer_windows(
                self.handle, xd.data_ptr(), n_windows, pd.data_ptr(), stream.cuda_stream))
            confidences = pd.cpu().numpy()
        return np.reshape(confidences, (-1)).astype(float)

    # ------------------------------------------------------------------ out of scope
    def train_network(self, *args, **kwargs):
        raise NotImplementedError("training is out of scope of catfish_b200 (inference hot path only)")

    def test_network(self, test_x, test_y, read_name=None, file_path=None, padding_size=0, threshold=0.5):
        """networks/rnn_class.py:222-261 ("next" row N4): forward pass + confusion counts.

        ``test_x`` / ``test_y`` are the padded ``[n_windows, 35, 1]`` arrays of
        ``train_validate.padding``; adds to ``self.tp/fp/tn/fn`` (true negatives minus
        ``padding_size``, :247) and returns ``(test_acc, test_loss)`` over all positions,
        padding included, like the reference's ``sess.run([self.accuracy, self.loss])``."""
        import torch
        x, y8 = self._validation_arrays(test_x, test_y)
        n_windows = x.shape[0]
        dev = torch.device("cuda", self.device)
        counts = np.zeros(4, np.int64)
        acc, loss = ctypes.c_double(), ctypes.c_double()
        with torch.cuda.device(dev):
            xd = torch.from_numpy(x.reshape(n_windows, self.window)).to(dev)
            yd = torch.from_numpy(np.ascontiguousarray(y8)).to(dev)
            stream = torch.cuda.current_stream(dev)
            _cabi.check(_cabi.load_library().cf_validate_windows(
                self.handle, xd.data_ptr(), yd.data_ptr(), n_windows, int(padding_size), float(threshold),
                counts.ctypes.data_as(_cabi.c_i64_p), ctypes.byref(acc), ctypes.byref(loss), stream.cuda_stream))
        self.tp += int(counts[0])
        self.fp += int(counts[1])
        self.tn += int(counts[2])
        self.fn += int(counts[3])
        return np.float32(acc.value), np.float32(loss.value)

    def test_network_sweep(self, test_x, test_y, thresholds, padding_size=0):
        """``test_network`` at every threshold of ``thresholds`` (unsorted / repeated allowed, 1..4096 of them) from
        ONE forward pass.  Adds the int64 ``[T, 4]`` rows (tp, fp, tn - padding_size, fn), in the order given, to
        ``self.sweep_counts`` (cleared by ``reset_sweep``; a sweep over another number of thresholds needs a reset
        first) and returns ``(test_acc, test_loss)`` exactly as ``test_network`` does: neither depends on the
        threshold.  Row i equals what ``test_network(..., threshold=thresholds[i])`` adds to tp / fp / tn / fn."""
        import torch
        x, y8 = self._validation_arrays(test_x, test_y)
        th = np.ascontiguousarray(np.asarray(thresholds, dtype=np.float64).reshape(-1))
        if self.sweep_counts is not None and self.sweep_counts.shape[0] != th.size:
            raise ValueError("sweep_counts holds %d thresholds, this sweep has %d: call reset_sweep() first"
                             % (self.sweep_counts.shape[0], th.size))
        n_windows = x.shape[0]
        dev = torch.device("cuda", self.device)
        counts = np.zeros((th.size, 4), np.int64)
        acc, loss = ctypes.c_double(), ctypes.c_double()
        with torch.cuda.device(dev):
            xd = torch.from_numpy(x.reshape(n_windows, self.window)).to(dev)
            yd = torch.from_numpy(np.ascontiguousarray(y8)).to(dev)
            stream = torch.cuda.current_stream(dev)
            _cabi.check(_cabi.load_library().cf_validate_windows_sweep(
                self.handle, xd.data_ptr(), yd.data_ptr(), n_windows, int(padding_size), th.ctypes.data,
                min(th.size, 2 ** 31 - 1), counts.ctypes.data_as(_cabi.c_i64_p), ctypes.byref(acc), ctypes.byref(loss),
                stream.cuda_stream))
        self.sweep_counts = counts if self.sweep_counts is None else self.sweep_counts + counts
        return np.float32(acc.value), np.float32(loss.value)

    def reset_sweep(self):
        """Clear ``self.sweep_counts``."""
        self.sweep_counts = None

    def _validation_arrays(self, test_x, test_y):
        """The padded ``[n_windows, 35, 1]`` input as float32 and its labels as uint8, checked."""
        x = np.ascontiguousarray(np.asarray(test_x, dtype=np.float32))
        if x.ndim != 3 or x.shape[1] != self.window or x.shape[2] != self.n_inputs:
            raise ValueError("Cannot feed value of shape %s for Tensor 'data/Placeholder:0', "
                             "which has shape '(?, %d, %d)'" % (x.shape, self.window, self.n_inputs))
        y = np.asarray(test_y).reshape(-1)
        if y.size != x.shape[0] * self.window:
            raise ValueError("Length of labels to compare is not equal.")
        y8 = y.astype(np.uint8)
        if not np.array_equal(y8, y):
            raise ValueError("labels must be small non-negative integers")
        return x, y8

    def _release(self):
        if getattr(self, "_slots", None):
            with self._slot_lock:
                slots, self._slots = self._slots, []
            for s in slots:
                try:
                    s.close()
                except Exception:
                    pass
        if getattr(self, "_handle", None) is not None:
            try:
                _cabi.load_library().cf_model_destroy(self._handle)
            except Exception:
                pass
            self._handle = None

    def close(self):
        self._release()

    def __del__(self):
        self._release()


def _latest_checkpoint(path):
    """tf.train.latest_checkpoint: the ``checkpoint`` state file, else the highest step present."""
    state = os.path.join(path, "checkpoint")
    if os.path.exists(state):
        with open(state) as f:
            for line in f:
                if line.startswith("model_checkpoint_path:"):
                    return os.path.basename(line.split(":", 1)[1].strip().strip('"'))
    best = None
    for fn in os.listdir(path):
        for ext in (".index", ".npz"):
            if fn.endswith(ext):
                stem = fn[:-len(ext)]
                try:
                    step = int(stem.rsplit("-", 1)[1])
                except (IndexError, ValueError):
                    continue
                if best is None or step > best[0]:
                    best = (step, stem)
    if best is None:
        raise ValueError("no checkpoint found in %s" % path)
    return best[1]
