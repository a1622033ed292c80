"""Weight sets for the catfish networks, keyed by the reference's TF variable names.

Variable names and shapes are the ones the reference graph creates
(/root/reference/catfish/models/resnet_class.py:44-82 for ``conv1d*`` /
``batch_normalization*``; /root/reference/catfish/models/rnn_class.py:142-183
for ``stack_bidirectional_rnn/cell_k/bidirectional_rnn/{fw,bw}/gru_cell/*`` and
``final_fully_connected/*``).  A weight set is a plain ``{name: float32 ndarray}``.

Three network types are supported (SURVEY.md section 8 row A14):

* ``"ResNetRNN"`` - residual blocks, then the bidirectional GRU stack, dense 2H->1
* ``"RNN"``       - GRU stack on the raw window (layer-0 input width 1)
* ``"ResNet"``    - residual blocks, dense C->1 (resnet_class.py:23 commented out)
"""

import os

import numpy as np

from . import tf_checkpoint

WINDOW = 35                # rnn_class.py:27
BN_EPSILON = 1e-3          # tf.layers.batch_normalization default, in the shipped meta-graph

NETWORK_TYPES = ("ResNetRNN", "RNN", "ResNet")

_DATA_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data")
SHIPPED_NPZ = os.path.join(_DATA_DIR, "ResNetRNN", "checkpoints", "ckpnt-30000.npz")
SHIPPED_HPARAMS = dict(batch_size=256, optimizer_choice="RMSProp", learning_rate=0.001,
                       layer_size=64, n_layers=3, keep_prob=0.8,
                       layer_size_res=32, n_layers_res=2)   # ResNetRNN/ResNetRNN.txt:3-10


def _suffix(i):
    return "" if i == 0 else "_%d" % i


def conv_name(i):
    return "conv1d" + _suffix(i)


def bn_name(i):
    return "batch_normalization" + _suffix(i)


def gru_prefix(layer, direction):
    return "stack_bidirectional_rnn/cell_%d/bidirectional_rnn/%s/gru_cell" % (layer, direction)


def expected_shapes(network_type, layer_size=64, n_layers=3, layer_size_res=32, n_layers_res=2):
    """``{name: shape}`` of every inference variable of the given network."""
    if network_type not in NETWORK_TYPES:
        raise ValueError("unknown network_type %r" % (network_type,))
    shapes = {}
    feat = 1
    if network_type in ("ResNetRNN", "ResNet"):
        c = layer_size_res
        for b in range(n_layers_res):
            cin = 1 if b == 0 else c
            # order inside residual_block: shortcut k1, conv k1, conv k3, conv k1
            for j, (k, ci) in enumerate(((1, cin), (1, cin), (3, c), (1, c))):
                i = 4 * b + j
                shapes[conv_name(i) + "/kernel"] = (k, ci, c)
                shapes[conv_name(i) + "/bias"] = (c,)
                for v in ("gamma", "beta", "moving_mean", "moving_variance"):
                    shapes[bn_name(i) + "/" + v] = (c,)
        feat = c
    if network_type in ("ResNetRNN", "RNN"):
        h = layer_size
        for l in range(n_layers):
            fin = feat if l == 0 else 2 * h
            for d in ("fw", "bw"):
                p = gru_prefix(l, d)
                shapes[p + "/gates/kernel"] = (fin + h, 2 * h)
                shapes[p + "/gates/bias"] = (2 * h,)
                shapes[p + "/candidate/kernel"] = (fin + h, h)
                shapes[p + "/candidate/bias"] = (h,)
        feat = 2 * h
    shapes["final_fully_connected/kernel"] = (feat, 1)
    shapes["final_fully_connected/bias"] = (1,)
    return shapes


def random_init(network_type, seed=0, **hpm):
    """One seeded draw from the reference's initializers.

    Kernels are Glorot-uniform, conv/dense/candidate biases 0, GRU gate biases
    1.0, BN gamma 1 / beta 0 / mean 0 / variance 1 (the Initializer nodes of the
    shipped meta-graph; SURVEY.md section 8c).  TensorFlow's own RNG stream is
    not reproducible, so parity runs hand this same draw to both sides.
    """
    rng = np.random.default_rng(seed)
    out = {}
    for name, shape in expected_shapes(network_type, **hpm).items():
        leaf = name.rsplit("/", 1)[1]
        if leaf == "kernel":
            if len(shape) == 3:
                fan_in, fan_out = shape[0] * shape[1], shape[0] * shape[2]
            else:
                fan_in, fan_out = shape
            lim = np.sqrt(6.0 / (fan_in + fan_out))
            out[name] = rng.uniform(-lim, lim, size=shape).astype(np.float32)
        elif leaf in ("gamma", "moving_variance"):
            out[name] = np.ones(shape, np.float32)
        elif leaf == "bias" and name.endswith("gates/bias"):
            out[name] = np.ones(shape, np.float32)
        else:
            out[name] = np.zeros(shape, np.float32)
    return out


def check_weights(weights, network_type, **hpm):
    want = expected_shapes(network_type, **hpm)
    for name, shape in want.items():
        if name not in weights:
            raise KeyError("missing variable %s" % name)
        if tuple(weights[name].shape) != tuple(shape):
            raise ValueError("variable %s has shape %s, expected %s"
                             % (name, tuple(weights[name].shape), tuple(shape)))
    return {k: np.ascontiguousarray(weights[k], dtype=np.float32) for k in want}


def load_npz(path):
    with np.load(path) as z:
        return {k: z[k].astype(np.float32) for k in z.files}


def save_npz(path, weights):
    np.savez(path, **{k: np.asarray(v, np.float32) for k, v in weights.items()})


def is_trainable(name):
    """Whether the optimizer updates ``name``: every inference variable but the BN moving statistics."""
    return not (name.endswith("/moving_mean") or name.endswith("/moving_variance"))


# the two slots tf.train.RMSPropOptimizer keeps per trainable variable, under the TF bundle's names
RMS_SLOT, MOM_SLOT = "/RMSProp", "/RMSProp_1"


def split_slots(tensors):
    """``{name: array}`` of a checkpoint -> (inference tensors, RMSProp slots)."""
    slots = {k: v for k, v in tensors.items() if k.endswith(RMS_SLOT) or k.endswith(MOM_SLOT)}
    return {k: v for k, v in tensors.items() if tf_checkpoint.is_inference_tensor(k)}, slots


def fresh_slots(weights):
    """Slots of a fresh optimizer: ``<var>/RMSProp`` ones, ``<var>/RMSProp_1`` zeros."""
    out = {}
    for k, v in weights.items():
        if is_trainable(k):
            out[k + RMS_SLOT] = np.ones(v.shape, np.float32)
            out[k + MOM_SLOT] = np.zeros(v.shape, np.float32)
    return out


def save_checkpoint(path, step, weights, slots):
    """Write ``<path>/ckpnt-<step>.npz`` (inference tensors + slots) and point ``<path>/checkpoint`` at it, as
    tf.train.Saver does for the reference's ``ckpnt-<step>`` bundles.  Returns the .npz path."""
    os.makedirs(path, exist_ok=True)
    name = "ckpnt-%d" % int(step)
    out = os.path.join(path, name + ".npz")
    tensors = dict(weights)
    tensors.update(slots)
    save_npz(out, tensors)
    with open(os.path.join(path, "checkpoint"), "w") as f:
        f.write('model_checkpoint_path: "%s"\nall_model_checkpoint_paths: "%s"\n' % (name, name))
    return out


def checkpoint_step(ckpnt):
    """The global step in a checkpoint name ``ckpnt-<step>``, or None."""
    try:
        return int(str(ckpnt).rsplit("-", 1)[1])
    except (IndexError, ValueError):
        return None


def load_tf_checkpoint(prefix):
    """Inference variables of a TF-V2 bundle (optimizer slots dropped)."""
    return tf_checkpoint.load_checkpoint(prefix, names=tf_checkpoint.is_inference_tensor)


def load_shipped():
    """The 74 inference tensors of catfish/ResNetRNN/checkpoints/ckpnt-30000."""
    return load_npz(SHIPPED_NPZ)
