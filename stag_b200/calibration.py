"""Calibration metrics of Categorical / Bernoulli predictions from the integer table of ``stag_calibration``.

The kernel (:func:`stag_b200.ops.calibration_table`) bins ``[N,C]`` probabilities into counts and fixed-point sums
(units of ``ONE = 2^32``; layout in include/stag_b200.h).  Integer tables add exactly, so the table of several
minibatches, or of several ranks after :meth:`Calibration.all_reduce`, is bit for bit the table of one call over all
their rows, and every metric below is a function of the table alone, computed in float64:

* ``accuracy`` (Categorical): rows whose argmax is the label / n.  ``micro_f1`` (Bernoulli): ``2tp / (2tp + fp + fn)``
  over all labels, a label predicted positive when p > 0.5.
* ``brier``: mean over rows of ``sum_c (q_c - [c == y])^2`` (Categorical), mean over the n C labels of ``(p - y)^2``
  (Bernoulli).
* ``ece``: ``sum_b |observed_b - confidence_b| / n_terms`` over the bins of the top-label confidence (Categorical, n
  terms) or of all labels pooled (Bernoulli, n C terms); ``mce``: the largest ``|observed - confidence|`` of a bin mean
  over the non-empty bins.
* ``classwise_ece``: ``(1/C) sum_c sum_b |label_sum_cb - prob_sum_cb| / n``.
* ``reliability()``: the bin edges, counts, mean confidence and observed frequency of the bins ``ece`` uses (NaN for
  empty bins): the points of sklearn's ``calibration_curve(strategy="uniform")``.

Every metric is NaN when the table holds no row, or when it counted an invalid row (``n_invalid``: a NaN, negative or
out-of-range probability, a Categorical row summing to zero, an out-of-range label), as the Monte-Carlo statistics of
``StagModel.predictive`` are NaN for such rows.
"""
import math
from typing import NamedTuple

import torch
import torch.distributed as dist

ONE = 2 ** 32
HEAD = 6
KINDS = ("categorical", "bernoulli")


class Reliability(NamedTuple):
    """Reliability diagram: ``edges [B+1]``, ``counts [B]``, ``confidence [B]`` (mean predicted probability) and
    ``frequency [B]`` (observed frequency of the positive outcome), float64 with NaN for empty bins."""
    edges: torch.Tensor
    counts: torch.Tensor
    confidence: torch.Tensor
    frequency: torch.Tensor


class Calibration:
    """Calibration table of ``n_classes`` classes in ``n_bins`` equal-width bins, ``table`` int64
    ``[6 + 3 n_bins + 3 n_classes n_bins]``, with the metrics it determines (module docstring)."""

    def __init__(self, kind, n_classes, n_bins, table):
        if kind not in KINDS:
            raise ValueError("Calibration: kind must be one of %s, got %r" % (KINDS, kind))
        n = HEAD + 3 * n_bins + 3 * n_classes * n_bins
        if table.dtype != torch.int64 or tuple(table.shape) != (n,):
            raise ValueError("Calibration: table must be int64 [%d], got %s %s" % (n, table.dtype, tuple(table.shape)))
        self.kind, self.n_classes, self.n_bins, self.table = kind, int(n_classes), int(n_bins), table

    def __repr__(self):
        return "Calibration(%s, n_classes=%d, n_bins=%d, n=%d, n_invalid=%d)" % (
            self.kind, self.n_classes, self.n_bins, self.n, self.n_invalid)

    def __add__(self, other):
        if not isinstance(other, Calibration):
            return NotImplemented
        if (self.kind, self.n_classes, self.n_bins) != (other.kind, other.n_classes, other.n_bins):
            raise ValueError("Calibration: cannot add a %s table of %d classes, %d bins to a %s table of %d classes, "
                             "%d bins" % (other.kind, other.n_classes, other.n_bins, self.kind, self.n_classes,
                                          self.n_bins))
        return Calibration(self.kind, self.n_classes, self.n_bins, self.table + other.table.to(self.table.device))

    def all_reduce(self, group=None):
        """Sum the tables of the ranks of ``group`` in place (one int64 all-reduce); returns self."""
        dist.all_reduce(self.table, op=dist.ReduceOp.SUM, group=group)
        return self

    # --- table views (on the host, as Python ints / int64 tensors) -------------------------------------------------
    def _host(self):
        t = self.table.detach().cpu()
        B, C = self.n_bins, self.n_classes
        return t[:HEAD].tolist(), t[HEAD:HEAD + 3 * B].view(3, B), t[HEAD + 3 * B:].view(3, C, B)

    @property
    def n(self):
        """Valid rows counted."""
        return int(self.table[0])

    @property
    def n_invalid(self):
        """Rows refused: they enter no other entry, and they make every metric NaN."""
        return int(self.table[1])

    def _undefined(self, head):
        return head[0] == 0 or head[1] > 0

    def _bins(self):
        """(count [B], probability sum [B], label sum [B]) of the bins ``ece`` uses, int64, sums in units of ONE."""
        _, top, cls = self._host()
        if self.kind == "categorical":
            return top[0], top[1], top[2] * ONE       # the correct count in fixed point
        return cls[0].sum(0), cls[1].sum(0), cls[2].sum(0)

    def _terms(self, head):
        return head[0] * (1 if self.kind == "categorical" else self.n_classes)

    @property
    def accuracy(self):
        """Fraction of rows whose argmax is the label (Categorical)."""
        if self.kind != "categorical":
            raise ValueError("Calibration.accuracy: Categorical tables only; a Bernoulli table has micro_f1")
        head = self._host()[0]
        return math.nan if self._undefined(head) else head[2] / head[0]

    @property
    def micro_f1(self):
        """``2tp / (2tp + fp + fn)`` over all labels (Bernoulli); NaN when no label is positive or predicted so."""
        if self.kind != "bernoulli":
            raise ValueError("Calibration.micro_f1: Bernoulli tables only; a Categorical table has accuracy")
        head = self._host()[0]
        tp, fp, fn = head[2:5]
        return math.nan if self._undefined(head) or 2 * tp + fp + fn == 0 else 2 * tp / (2 * tp + fp + fn)

    @property
    def brier(self):
        """Mean squared error of the probabilities against the one-hot label (per row, summed over the classes:
        Categorical) or the label values (per label: Bernoulli)."""
        head = self._host()[0]
        return math.nan if self._undefined(head) else head[5] / ONE / self._terms(head)

    def _gaps(self):
        count, prob, label = self._bins()
        return count, (label - prob).abs()            # exact int64 differences in units of ONE

    @property
    def ece(self):
        """Expected calibration error: ``sum_b |label_sum_b - prob_sum_b| / n_terms``."""
        head = self._host()[0]
        if self._undefined(head):
            return math.nan
        return float(self._gaps()[1].to(torch.float64).sum()) / ONE / self._terms(head)

    @property
    def mce(self):
        """Maximum calibration error: the largest gap between a bin's mean label and mean probability."""
        head = self._host()[0]
        if self._undefined(head):
            return math.nan
        count, gap = self._gaps()
        full = count > 0
        return float((gap[full].to(torch.float64) / ONE / count[full].to(torch.float64)).max())

    @property
    def classwise_ece(self):
        """``(1/C) sum_c sum_b |label_sum_cb - prob_sum_cb| / n``: the ECE of each class's one-vs-rest probability."""
        head, _, cls = self._host()
        if self._undefined(head):
            return math.nan
        label = cls[2] * ONE if self.kind == "categorical" else cls[2]
        gap = (label - cls[1]).abs().to(torch.float64).sum()
        return float(gap) / ONE / head[0] / self.n_classes

    def reliability(self):
        """:class:`Reliability` of the bins ``ece`` uses: top-label confidence (Categorical), all labels pooled
        (Bernoulli)."""
        head = self._host()[0]
        count, prob, label = self._bins()
        c = count.to(torch.float64)
        conf = prob.to(torch.float64) / ONE / c
        freq = label.to(torch.float64) / ONE / c
        if self._undefined(head):
            conf.fill_(math.nan)
            freq.fill_(math.nan)
        conf[count == 0] = math.nan
        freq[count == 0] = math.nan
        edges = torch.arange(self.n_bins + 1, dtype=torch.float64) * (1.0 / self.n_bins)   # np.linspace's values
        edges[-1] = 1.0
        return Reliability(edges, count, conf, freq)


def calibration(probs, y, kind, n_bins=15, mask=None, table_fn=None):
    """:class:`Calibration` of ``probs [N,C]`` against labels ``y`` (int [N]: Categorical; [N,C]: Bernoulli), rows
    where ``mask`` is set.  ``table_fn`` (default :func:`stag_b200.ops.calibration_table`, the kernel) computes the
    table."""
    if table_fn is None:
        from . import ops
        table_fn = ops.calibration_table
    return Calibration(kind, probs.shape[-1], n_bins, table_fn(probs, y, kind, n_bins, mask))
