"""Snapshot metrics on the scorer's outputs (host numpy / scipy, as the reference computes them; not the hot path):
Inception Score (trainer.py:88-99), Frechet Inception Distance (trainer.py:102-145) and the negative log posterior
probability (trainer.py:149-159). `pred` is the (N, 1000) softmax, `pool3` the (N, 2048) features of INCEPTION_V3."""
import numpy as np
from scipy import linalg


def _splits(x, splits):
    n = x.shape[0]
    return [x[i * n // splits:(i + 1) * n // splits] for i in range(splits)]


def inception_score(pred, splits=1):
    """(mean, std) over `splits` equal parts of exp(E_x KL(p(y|x) || p(y)))."""
    scores = []
    for part in _splits(np.asarray(pred, dtype=np.float64), splits):
        kl = part * (np.log(part) - np.log(np.mean(part, 0, keepdims=True)))
        scores.append(np.exp(np.mean(np.sum(kl, 1))))
    return float(np.mean(scores)), float(np.std(scores))


def negative_log_posterior_probability(pred, splits=1):
    """(mean, std) over `splits` equal parts of the mean of -log max_y p(y|x)."""
    scores = [np.mean(-np.log(np.max(part, 1))) for part in _splits(np.asarray(pred, dtype=np.float64), splits)]
    return float(np.mean(scores)), float(np.std(scores))


def frechet_distance(pool3_a, pool3_b, eps=1e-6):
    """||mu_a - mu_b||^2 + Tr(S_a + S_b - 2 (S_a S_b)^(1/2)) of the Gaussians fitted to two feature sets."""
    a, b = np.asarray(pool3_a, dtype=np.float64), np.asarray(pool3_b, dtype=np.float64)
    mu1, mu2 = a.mean(0), b.mean(0)
    s1, s2 = np.atleast_2d(np.cov(a, rowvar=False)), np.atleast_2d(np.cov(b, rowvar=False))
    diff = mu1 - mu2
    covmean = linalg.sqrtm(s1.dot(s2))
    if not np.isfinite(covmean).all():       # singular product: offset the diagonals
        off = np.eye(s1.shape[0]) * eps
        covmean = linalg.sqrtm((s1 + off).dot(s2 + off))
    if np.iscomplexobj(covmean):
        covmean = covmean.real
    return float(diff.dot(diff) + np.trace(s1) + np.trace(s2) - 2 * np.trace(covmean))
