import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden(name):
    with np.load(os.path.join(GOLDEN, name), allow_pickle=False) as z:
        return {k: z[k] for k in z.files}


def hpm_from_golden(g):
    return {k[4:]: int(v) for k, v in g.items() if k.startswith("hpm_")}


# tc_create runs f16e5 only while max |w| * kCandScale * kCorrScale < 60000 (the fp16 weight plane holds S w)
F16E5_WMAX = 60000.0 / (2.8853900817779268 * 64.0)


def hparams(kind, c=32, h=64, n_res=2, n_layers=3):
    """Hyper-parameters of a `kind` network: conv channels c and blocks n_res, GRU units h and layers n_layers."""
    hpm = {}
    if kind != "RNN":
        hpm.update(layer_size_res=c, n_layers_res=n_res)
    if kind != "ResNet":
        hpm.update(layer_size=h, n_layers=n_layers)
    return hpm


def build_model(kind, engine, w, **hpm):
    """A `kind` model on `engine` with weights w; hyper-parameters not in hpm are the shipped ones."""
    from catfish_b200 import neural_network, weights
    full = dict(weights.SHIPPED_HPARAMS)
    full.update(hpm)
    m = neural_network.build_model(kind, engine=engine, **full)
    m.set_weights(w)
    return m


def bn_weights(kind, seed, **hpm):
    """Seeded weights of any shape with non-trivial BN gamma / beta / moving statistics."""
    from catfish_b200 import weights
    w = weights.random_init(kind, seed=seed, **hpm)
    rng = np.random.default_rng(seed + 1000)
    for k in sorted(w):
        if k.endswith("moving_mean"):
            w[k] = rng.normal(0, 0.3, size=w[k].shape).astype(np.float32)
        elif k.endswith("moving_variance"):
            w[k] = rng.uniform(0.3, 2.0, size=w[k].shape).astype(np.float32)
        elif k.endswith("beta"):
            w[k] = rng.normal(0, 0.2, size=w[k].shape).astype(np.float32)
        elif k.endswith("gamma"):
            w[k] = rng.uniform(0.5, 1.5, size=w[k].shape).astype(np.float32)
    return w


def random_bn_weights(seed):
    """Seeded ResNetRNN weights (shipped hyper-parameters) with non-trivial BN gamma/beta/moving stats."""
    return bn_weights("ResNetRNN", seed, layer_size=64, n_layers=3, layer_size_res=32, n_layers_res=2)


def random_labels(rng, n, p_switch=0.08):
    """Binary label sequence with geometric run lengths (mean 1 / p_switch)."""
    out = np.empty(n, np.int64)
    i, cur = 0, int(rng.integers(0, 2))
    while i < n:
        run = int(rng.geometric(p_switch))
        out[i:i + run] = cur
        i += run
        cur ^= 1
    return out


def allowed_label_flips(p_ref, threshold=0.5, band=1e-3):
    """Positions where the contract allows a different label: reference p within `band` of the threshold."""
    return np.abs(np.asarray(p_ref, np.float64) - threshold) <= band


class FakeFast5(object):
    """In-memory stand-in for an open ``h5py.File`` with the three things infer.py:87-90 touches: the
    ``first_sample_template`` attribute of the segmentation summary, ``Raw/Reads/`` with ``visit`` (h5py calls
    the function on every member name and returns its first non-None result) and the ``Signal`` dataset."""

    class _Node(object):
        def __init__(self, attrs=None, members=None, data=None):
            self.attrs = attrs or {}
            self._members = members or []
            self._data = data

        def visit(self, func):
            for name in self._members:
                out = func(name)
                if out is not None:
                    return out
            return None

        def __getitem__(self, key):
            assert key == ()
            return self._data

    def __init__(self, signal, first_sample, read_names=("Read_117",)):
        self.signal = np.asarray(signal, np.int16)
        self.nodes = {
            "Analyses/Segmentation_000/Summary/segmentation": self._Node(attrs={"first_sample_template": first_sample}),
            "Raw/Reads/": self._Node(members=list(read_names)),
            "Raw/Reads/%s/Signal" % read_names[0]: self._Node(data=self.signal),
        }

    def __getitem__(self, path):
        return self.nodes[path]

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


def fake_h5py_module(files):
    """A module object to put into ``sys.modules['h5py']``: ``File(path, mode)`` returns ``files[path]``."""
    import types
    mod = types.ModuleType("h5py")
    mod.File = lambda path, mode="r": files[path]
    return mod
