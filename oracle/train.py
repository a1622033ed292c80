"""ORACLE (test infrastructure, never imported by the product): one training step in float64.

The step ``RNN.train_network`` runs on the device (catfish_b200/csrc/k12_train.cu), restated on the
CPU with torch autograd in float64:

* forward   ``tf_graph.TorchGraph``'s op sequence (the pinned inference graph) with output dropout on
            every GRU cell: each direction's per-step output becomes ``h / keep_prob * mask`` before it
            is concatenated (DropoutWrapper(output_keep_prob), the while/dropout nodes of the shipped
            graph); the recurrent state is never dropped; BN uses its moving statistics
* loss      mean sigmoid cross-entropy over all positions (``oracle.validation``'s formula)
* gradients autograd of that loss
* update    TF 1.x ApplyRMSProp: ms += (g^2 - ms)(1 - decay); mom = momentum mom + lr g / sqrt(ms + eps);
            var -= mom (decay 0.9, momentum 0, epsilon 1e-10)
* mask      Philox4x32-10 in numpy: key = seed, counter = (step, 2 layer + direction, window, t H + unit),
            kept when the top 24 bits of word 0 are < round(keep_prob 2^24)
"""

import numpy as np

from .tf_graph import TorchGraph, WINDOW, _gru_prefix, describe

RMS_DECAY, RMS_MOMENTUM, RMS_EPSILON = 0.9, 0.0, 1e-10

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)
_LO = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Random123's philox4x32-10 over arrays: ctr 4 uint32 arrays (broadcastable), key 2 uint32 -> 4 uint32 arrays."""
    c = [np.asarray(v, np.uint32).astype(np.uint64) for v in ctr]
    c = list(np.broadcast_arrays(*c))
    k0, k1 = np.uint32(key[0]), np.uint32(key[1])
    with np.errstate(over="ignore"):
        for i in range(10):
            if i:
                k0, k1 = np.uint32(k0 + _W0), np.uint32(k1 + _W1)
            p0 = _M0 * c[0]
            p1 = _M1 * c[2]
            c = [(p1 >> np.uint64(32)) ^ c[1] ^ np.uint64(k0), p1 & _LO,
                 (p0 >> np.uint64(32)) ^ c[3] ^ np.uint64(k1), p0 & _LO]
    return [v.astype(np.uint32) for v in c]


def dropout_mask(seed, step, layer, direction, n_windows, hidden, keep_prob, window0=0):
    """bool [n_windows, 35, hidden]: the device's mask of one GRU direction."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    w = np.arange(window0, window0 + n_windows, dtype=np.uint64)[:, None, None]
    t = np.arange(WINDOW, dtype=np.uint64)[None, :, None]
    u = np.arange(hidden, dtype=np.uint64)[None, None, :]
    word0 = philox4x32_10([np.uint32(step), np.uint32(2 * layer + direction), w, t * np.uint64(hidden) + u],
                          [seed & 0xFFFFFFFF, seed >> 32])[0]
    return (word0 >> np.uint32(8)) < np.uint32(int(round(keep_prob * 2 ** 24)))


def dropout_masks(weights, seed, step, n_windows, keep_prob):
    """{(layer, direction): mask} for every GRU cell of the network, or None at keep_prob = 1."""
    if keep_prob >= 1.0:
        return None
    n_rnn = describe(weights)[2]
    hidden = weights[_gru_prefix(0, "fw") + "/candidate/kernel"].shape[1] if n_rnn else 0
    return {(l, d): dropout_mask(seed, step, l, d, n_windows, hidden, keep_prob)
            for l in range(n_rnn) for d in range(2)}


def _is_trainable(name):
    return not (name.endswith("/moving_mean") or name.endswith("/moving_variance"))


class TrainGraph(TorchGraph):
    """TorchGraph with leaf tensors that carry gradients (float64 unless told otherwise), and dropout on the GRU
    outputs."""

    def __init__(self, weights, dtype=np.float64):
        import torch
        self.torch = torch
        TorchGraph.__init__(self, weights)
        self.dtype = dtype
        self.w = {k: torch.tensor(np.asarray(v, dtype), requires_grad=_is_trainable(k))
                  for k, v in weights.items()}

    def logits(self, x, keep_prob=1.0, masks=None):
        """x [B, 35, 1] -> float64 logits [B * 35] (a torch tensor in the autograd graph)."""
        t = self.torch
        y = t.from_numpy(np.asarray(x, np.float32).reshape(-1, WINDOW, 1).astype(self.dtype))
        for b in range(self.n_res):
            y = self._block(y, b)
        for l in range(self.n_rnn):
            outs = []
            for d, name in enumerate(("fw", "bw")):
                o = self._gru(y, _gru_prefix(l, name), d == 1)
                if masks is not None:
                    o = o / keep_prob * t.from_numpy(masks[(l, d)].astype(self.dtype))
                outs.append(o)
            y = t.cat(outs, dim=2)
        z = y.reshape(-1, y.shape[2]) @ self.w["final_fully_connected/kernel"] + self.w["final_fully_connected/bias"]
        return z.reshape(-1)


def loss_of_logits(z, labels):
    """compute_loss: mean(max(z, 0) - z y + log1p(exp(-|z|)))."""
    import torch
    y = torch.from_numpy(np.asarray(labels).reshape(-1)).to(z.dtype)
    return (torch.clamp(z, min=0) - z * y + torch.log1p(torch.exp(-torch.abs(z)))).mean()


def step_gradients(weights, x, labels, keep_prob=1.0, masks=None):
    """-> (loss, {trainable name: float64 dL/dvar}, float64 logits) of one step's forward."""
    g = TrainGraph(weights)
    z = g.logits(x, keep_prob, masks)
    loss = loss_of_logits(z, labels)
    loss.backward()
    grads = {k: v.grad.numpy().copy() for k, v in g.w.items() if v.requires_grad}
    return float(loss.item()), grads, z.detach().numpy()


def rmsprop(var, ms, mom, grad, lr):
    """ApplyRMSProp in float64 -> (var, ms, mom)."""
    ms = ms + (grad * grad - ms) * (1.0 - RMS_DECAY)
    mom = RMS_MOMENTUM * mom + lr * grad / np.sqrt(ms + RMS_EPSILON)
    return var - mom, ms, mom


def train_steps(weights, batches, lr, keep_prob=1.0, seed=0, step0=0, slots=None):
    """Run len(batches) steps of (x, labels) from ``weights`` (float64 master copies) -> (weights, slots, losses).
    ``slots`` {"<var>/RMSProp": ms, "<var>/RMSProp_1": mom}, fresh (ones / zeros) when None."""
    w = {k: np.asarray(v, np.float64) for k, v in weights.items()}
    if slots is None:
        slots = {}
        for k, v in w.items():
            if _is_trainable(k):
                slots[k + "/RMSProp"] = np.ones_like(v)
                slots[k + "/RMSProp_1"] = np.zeros_like(v)
    slots = {k: np.asarray(v, np.float64) for k, v in slots.items()}
    losses = []
    for i, (x, y) in enumerate(batches):
        masks = dropout_masks(w, seed, step0 + i, np.asarray(x).reshape(-1, WINDOW).shape[0], keep_prob)
        loss, grads, _ = step_gradients(w, x, y, keep_prob, masks)
        losses.append(loss)
        for k, g in grads.items():
            w[k], slots[k + "/RMSProp"], slots[k + "/RMSProp_1"] = rmsprop(
                w[k], slots[k + "/RMSProp"], slots[k + "/RMSProp_1"], g, lr)
    return w, slots, losses
