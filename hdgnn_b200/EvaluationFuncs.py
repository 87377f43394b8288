"""Evaluation metrics with the semantics of the reference's EvaluationFuncs.py, vectorised.

Inputs are (N, 2, Ncr) arrays: `label` one-hot over the two channels (channel 0 = "no relation",
utils2.py:105), `real` the softmax output.  The reference's quirks are kept by default because
they define its printed numbers (SURVEY Q6, Q7):

  * prec / recall / f1 apply np.ceil to both arrays and score CHANNEL 0 (EvaluationFuncs.py:92-117),
    so every prediction is 1 unless a probability underflowed to exactly 0;
  * AUC re-zeroes its accumulator and counter inside the per-commit loop (EvaluationFuncs.py:119-153),
    so it returns the last commit's value (ZeroDivisionError when that commit has one class), and it
    scores each pair with the probability of the class the label does NOT have.

`quirks=False` gives the conventional definitions (relation class = channel 1, mean over commits).
"""
from __future__ import annotations

import numpy as np


def process_edge(Ra):                       # EvaluationFuncs.py:11-16: identity
    return Ra


def top_ACC(Ra, Ra_t):
    """Share of pairs whose arg-max channel matches the label (EvaluationFuncs.py:27-37)."""
    Ra = np.asarray(Ra); Ra_t = np.asarray(Ra_t)
    return float(np.mean(np.argmax(Ra_t, axis=1) == np.argmax(Ra, axis=1)))


def _binary_scores(y_true, y_pred):
    """Per-row precision / recall / F1 of the positive class, sklearn conventions (0 on empty denominators)."""
    tp = np.sum((y_true == 1) & (y_pred == 1), axis=1).astype(np.float64)
    fp = np.sum((y_true != 1) & (y_pred == 1), axis=1).astype(np.float64)
    fn = np.sum((y_true == 1) & (y_pred != 1), axis=1).astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        p = np.where(tp + fp > 0, tp / (tp + fp), 0.0)
        r = np.where(tp + fn > 0, tp / (tp + fn), 0.0)
        f = np.where(2 * tp + fp + fn > 0, 2 * tp / (2 * tp + fp + fn), 0.0)
    return p, r, f


def _prf(label, real, quirks):
    label = np.asarray(label); real = np.asarray(real)
    if quirks:
        return _binary_scores(np.ceil(label[:, 0, :]), np.ceil(real[:, 0, :]))
    return _binary_scores(label[:, 1, :] > 0.5, real[:, 1, :] > real[:, 0, :])


def prec(label, real, quirks=True):
    return float(_prf(label, real, quirks)[0].mean())


def recall(label, real, quirks=True):
    return float(_prf(label, real, quirks)[1].mean())


def f1(label, real, quirks=True):
    return float(_prf(label, real, quirks)[2].mean())


def _roc_auc(y_true, score):
    """Mann-Whitney AUC with average ranks for ties (== sklearn.metrics.roc_auc_score); None if one class."""
    y_true = np.asarray(y_true).astype(bool)
    npos = int(y_true.sum()); nneg = y_true.size - npos
    if npos == 0 or nneg == 0:
        return None
    order = np.argsort(score, kind="mergesort")
    s = np.asarray(score)[order]
    ranks = np.empty(s.size, dtype=np.float64)
    i = 0
    while i < s.size:
        j = i
        while j + 1 < s.size and s[j + 1] == s[i]:
            j += 1
        ranks[i:j + 1] = 0.5 * (i + j) + 1.0
        i = j + 1
    r = np.empty_like(ranks)
    r[order] = ranks
    return float((r[y_true].sum() - npos * (npos + 1) / 2.0) / (npos * nneg))


def AUC(label, real, quirks=True):
    label = np.asarray(label); real = np.asarray(real)
    vals = []
    for i in range(label.shape[0]):
        if quirks:
            y = np.argmax(label[i], axis=0)                  # 1 where the pair is a relation
            pick = np.argmin(label[i], axis=0)               # the channel the label does NOT have
            score = np.take_along_axis(real[i], pick[None, :], axis=0)[0]
        else:
            y = label[i, 1] > 0.5
            score = real[i, 1]
        a = _roc_auc(y, score)
        if a is None:
            print('ValueError: Only one class present in y_true. ROC AUC score is not defined in that case.')
        vals.append(a)
    if quirks:                                               # accumulator and counter reset every commit
        last = vals[-1]
        if last is None:
            raise ZeroDivisionError("float division by zero")
        return last
    good = [v for v in vals if v is not None]
    return float(np.mean(good)) if good else float("nan")


def metrics_from_counts(counts, quirks=True):
    """The printed metrics of model_2.py:535-540 from the integer counters of hdgnn_eval_counts (include/hdgnn.h):
    counts (N,8) = {arg-max hits, quirk tp fp fn, conventional tp fp fn, related pairs}.  Same conventions as the array
    functions above (sklearn: 0 on an empty denominator); top_ACC = hits / (N Ncr)."""
    c = np.asarray(counts, dtype=np.int64)
    o = 1 if quirks else 4
    tp, fp, fn = (c[:, o + k].astype(np.float64) for k in range(3))
    with np.errstate(divide="ignore", invalid="ignore"):
        p = np.where(tp + fp > 0, tp / (tp + fp), 0.0)
        r = np.where(tp + fn > 0, tp / (tp + fn), 0.0)
        f = np.where(2 * tp + fp + fn > 0, 2 * tp / (2 * tp + fp + fn), 0.0)
    out = dict(hits=int(c[:, 0].sum()), prec=float(p.mean()), recall=float(r.mean()), f1=float(f.mean()))
    return out


def _auc_from_counts(num, npos, ncr):
    npos = npos.astype(np.float64)
    den = 2.0 * npos * (ncr - npos)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(den > 0, num / den, np.nan)


def auc_from_counts(counts, auc, ncr, quirks=True, first=0):
    """AUC of EvaluationFuncs.py:119-153 from device counters: quirk form = the last commit's value
    (ZeroDivisionError when it has one class), conventional = mean over the commits with both classes."""
    c = np.asarray(counts, dtype=np.int64)
    a = np.asarray(auc, dtype=np.int64)
    vals = _auc_from_counts(a[:, 0 if quirks else 1], c[:, 7], ncr)
    if quirks:
        if np.isnan(vals[-1]):
            raise ZeroDivisionError("float division by zero")
        return float(vals[-1])
    good = vals[first:][~np.isnan(vals[first:])]
    return float(good.mean()) if good.size else float("nan")


def partition_metrics_from_counts(counts):
    """Group-level scores of an untangling from the partition-agreement counters of hdgnn_partition_counts (include/hdgnn.h):
    counts (N,8) = {real hunks m, pairs joined in both, by pred, by truth, groups of pred, of truth, sum of largest overlaps
    of the pred groups, of the truth groups}.
      exact            commits whose two partitions of the real hunks are equal (the three pair counts agree);
      pair_precision   sum both / sum pred, pair_recall = sum both / sum truth, pair_f1 = 2 sum both / (sum pred + sum truth):
                       pooled over commits, 0.0 on an empty denominator;
      rand, ari        mean over the commits with m >= 2 of sklearn's rand_score and adjusted_rand_score (1.0 when no pair
                       is joined by one partition and split by the other); nan if there is no such commit;
      purity           sum of largest overlaps of the pred groups / sum m (inverse_purity: of the truth groups), 0.0 if no hunk;
      groups_pred_mean, groups_truth_mean: groups per commit (nan if there is no commit).
    Raises ValueError on a row of -1 (a commit the kernel could not score)."""
    c = np.asarray(counts, dtype=np.int64).reshape(-1, 8)
    if (c < 0).any():
        raise ValueError("partition counters hold a row of -1: a commit with nh outside [0, n] or a label outside [0, n)")
    m, both, jp, jt = (c[:, k] for k in range(4))
    S = c.sum(0)

    def ratio(a, b):
        return float(a / b) if b > 0 else 0.0

    M = m * (m - 1) // 2                                     # pairs of real hunks
    fp, fn = jp - both, jt - both                            # joined by pred only, by truth only
    tn = M - both - fp - fn
    sel = m >= 2
    with np.errstate(divide="ignore", invalid="ignore"):
        rand = (both + tn) / M
        den = (both + fn) * (fn + tn) + (both + fp) * (fp + tn)
        ari = np.where((fp == 0) & (fn == 0), 1.0, 2.0 * (both * tn - fn * fp) / den)
    return dict(commits=int(c.shape[0]), exact=int(((both == jp) & (both == jt)).sum()),
                pair_precision=ratio(S[1], S[2]), pair_recall=ratio(S[1], S[3]), pair_f1=ratio(2 * S[1], S[2] + S[3]),
                rand=float(rand[sel].mean()) if sel.any() else float("nan"),
                ari=float(ari[sel].mean()) if sel.any() else float("nan"),
                purity=ratio(S[6], S[0]), inverse_purity=ratio(S[7], S[0]),
                groups_pred_mean=float(c[:, 4].mean()) if c.shape[0] else float("nan"),
                groups_truth_mean=float(c[:, 5].mean()) if c.shape[0] else float("nan"))
