"""Validation driver of the reference over in-memory reads ("next" row N4).  The training half of
``train_and_validate`` is ``RNN.train_network`` / ``save_network`` (INTEGRATION.md, "Training loop").

Reference: /root/reference/networks/train_validate.py (``padding`` :51-64, ``reshape_input`` :15-31,
``validate`` :188-295).  ``validate`` here takes ``(data, labels)`` arrays instead of ``.npz``
paths (the file reader is host I/O), runs ``network.test_network`` per read - forward pass and
confusion counting on the GPU - and returns the same triple.  Note the padding rule differs from
``infer.py``: nothing is appended when the length is a multiple of the window.
"""

import random

import numpy as np

from . import metrics
from .infer import reshape_input  # noqa: F401  (same function, train_validate.py:15-31)


def padding(data, window=35, n_input=1):
    """train_validate.py:51-64: zero-pad to a multiple of ``window`` -> ([n, window, n_input], pad)."""
    data = np.asarray(data)
    padding_size = (-len(data)) % window
    if padding_size:
        data = np.hstack((data, np.zeros(padding_size, dtype=int)))
    return reshape_input(data, window, n_input), padding_size


def validate(network, squiggles, max_seq_length, file_path=None, validation_start="random", max_number=856,
             thresholds=None):
    """train_validate.py:188-295 over ``squiggles = [(data, labels), ...]``.

    Returns ``(whole_accuracy, whole_precision, whole_recall)`` and resets the network's counters;
    the per-read mean accuracy / loss and the summary line go to ``file_path + ".txt"`` when given.

    With ``thresholds`` (a sequence of up to 4096), every read goes through ``network.test_network_sweep`` instead -
    one forward pass for all thresholds - and the three results are float64 arrays with one entry per threshold, in
    the order given; the summary then has one line per threshold.  ``network.sweep_counts`` is cleared before and
    after, as the reference clears its counters.
    """
    if thresholds is not None:
        thresholds = np.asarray(thresholds, dtype=np.float64).reshape(-1)
        network.reset_sweep()
    total_length, accuracy, loss, valid_reads = 0, 0.0, 0.0, 0
    for data_sq, labels_sq in squiggles:
        data_sq, labels_sq = np.asarray(data_sq), np.asarray(labels_sq)
        if validation_start == "complete":
            total_length += len(data_sq)
        else:
            max_seq_length = max_seq_length // network.window * network.window
            if type(validation_start) == int:
                if len(data_sq) < validation_start + max_seq_length:
                    continue
                start_val = validation_start
            elif validation_start == "random":
                if len(data_sq) < max_seq_length:
                    continue
                start_val = random.randint(0, len(data_sq) - max_seq_length)
            labels_sq = labels_sq[start_val: start_val + max_seq_length]
            data_sq = data_sq[start_val: start_val + max_seq_length]
            total_length += max_seq_length
        valid_reads += 1
        set_x, padding_size = padding(data_sq, network.window, network.n_inputs)
        set_y, _ = padding(labels_sq, network.window, network.n_inputs)
        if thresholds is None:
            sgl_acc, sgl_loss = network.test_network(set_x, set_y, None, file_path, padding_size)
        else:
            sgl_acc, sgl_loss = network.test_network_sweep(set_x, set_y, thresholds, padding_size)
        if valid_reads >= max_number:       # the reference leaves before adding this read's accuracy (:254)
            break
        accuracy += sgl_acc
        loss += sgl_loss

    if thresholds is not None:
        return _sweep_summary(network, thresholds, file_path, accuracy, loss, valid_reads)
    whole_accuracy = metrics.calculate_accuracy(network.tp, network.fp, network.tn, network.fn)
    whole_precision, whole_recall = metrics.precision_recall(network.tp, network.fp, network.fn)
    whole_f1 = metrics.f1(whole_precision, whole_recall)
    if file_path:
        with open(file_path + ".txt", "a+") as dest:
            dest.write("\n---NEXT ROUND OF VALIDATION---")
            dest.write("\nAverage performance of validation set:\n")
            dest.write("\tAccuracy: {:.2%}\n".format(accuracy / valid_reads))
            dest.write("\tLoss: {0:.4f}".format(loss / valid_reads))
            dest.write("\nPerformance over whole set: \n")
            dest.write("\tDetected {} true positives, {} false positives, {} true negatives, {} false negatives in total.\n"
                       .format(network.tp, network.fp, network.tn, network.fn))
            dest.write("\tAccuracy: {:.2%}".format(whole_accuracy))
            dest.write("\n\tPrecision: {:.2%}\n\tRecall: {:.2%}".format(whole_precision, whole_recall))
            dest.write("\t\nF1 score: {0:.4f}".format(whole_f1))
    network.tp = network.fn = network.tn = network.fp = 0
    return whole_accuracy, whole_precision, whole_recall


def _sweep_summary(network, thresholds, file_path, accuracy, loss, valid_reads):
    """The end of ``validate`` with thresholds: per-threshold accuracy / precision / recall from
    ``network.sweep_counts`` (0 where a denominator is 0), the summary file, and the counters cleared."""
    counts = network.sweep_counts if network.sweep_counts is not None else np.zeros((thresholds.size, 4), np.int64)
    tp, fp, tn, fn = (counts[:, i].astype(np.float64) for i in range(4))
    whole_accuracy = metrics._rates(tp + tn, tp + fp + tn + fn)
    whole_precision = metrics._rates(tp, tp + fp)
    whole_recall = metrics._rates(tp, tp + fn)
    if file_path:
        with open(file_path + ".txt", "a+") as dest:
            dest.write("\n---NEXT ROUND OF VALIDATION---")
            dest.write("\nAverage performance of validation set:\n")
            dest.write("\tAccuracy: {:.2%}\n".format(accuracy / valid_reads))
            dest.write("\tLoss: {0:.4f}".format(loss / valid_reads))
            dest.write("\nPerformance over whole set, per threshold (threshold, TP, FP, TN, FN, accuracy, precision, "
                       "recall):\n")
            for i in range(thresholds.size):
                dest.write("\t{:.6g}\t{}\t{}\t{}\t{}\t{:.2%}\t{:.2%}\t{:.2%}\n".format(
                    thresholds[i], *counts[i].tolist(), whole_accuracy[i], whole_precision[i], whole_recall[i]))
    network.reset_sweep()
    return whole_accuracy, whole_precision, whole_recall
