"""Skill scores of simulated series against observations: NSE, KGE, RMSE and bias, from running sums.

The melt kernel scores every cell against an observed series while it runs (``tfg_bind_objective``,
``MeltEngine.set_objective``): per cell it adds ``S_s = sum s``, ``S_ss = sum s*s``, ``S_so = sum s*o`` and
``S_ee = sum (s - o)**2`` over the steps whose observation is finite.  The observations' own moments
``n, S_o = sum o, S_oo = sum o*o`` are known without the model.  This module turns the seven sums into scores, and
states the same metrics for series a caller already holds (``series_scores``, e.g. basin runoff against a gauge), so
that both paths share one definition:

    mean_s = S_s / n,   var_s = max(S_ss / n - mean_s**2, 0),   likewise mean_o, var_o,   cov = S_so / n - mean_s * mean_o
    NSE   = 1 - S_ee / (n * var_o)                         (Nash & Sutcliffe 1970)
    RMSE  = sqrt(S_ee / n),   bias = (S_s - S_o) / n
    r     = cov / sqrt(var_s * var_o),   alpha = sqrt(var_s / var_o),   beta = mean_s / mean_o
    KGE   = 1 - sqrt((r - 1)**2 + (alpha - 1)**2 + (beta - 1)**2)   (Gupta et al. 2009)

``S_ee`` is summed directly rather than derived as ``S_ss - 2 S_so + S_oo``: near NSE = 1, the candidates a calibration
cares about, that difference cancels to nothing.  Where ``n = 0``, ``var_o = 0`` or ``mean_o = 0`` (and, for ``r``,
``var_s = 0``) the affected scores are NaN, never +-inf.
"""

from __future__ import annotations

from typing import Tuple

import torch

__all__ = ["SCORE_NAMES", "skill_scores", "series_sums", "series_scores", "accumulate_step"]

SCORE_NAMES = ("n", "nse", "kge", "r", "alpha", "beta", "rmse", "bias")


def _t(x) -> torch.Tensor:
    return x.to(torch.float64) if torch.is_tensor(x) else torch.as_tensor(x, dtype=torch.float64)


def _ratio(num: torch.Tensor, den: torch.Tensor) -> torch.Tensor:
    """num / den where den > 0, else NaN (no +-inf from a zero denominator)."""
    nan = torch.full_like(num, float("nan"))
    return torch.where(den > 0, num / torch.where(den > 0, den, torch.ones_like(den)), nan)


def skill_scores(sums, obs_moments) -> dict:
    """Scores from the four simulation sums ``(S_s, S_ss, S_so, S_ee)`` (a ``[4, N]`` tensor or four ``[N]`` arrays) and
    the observations' moments ``(n, S_o, S_oo)``.  Returns ``{name: [N] float64 tensor}`` for ``SCORE_NAMES``."""
    S_s, S_ss, S_so, S_ee = (_t(v) for v in sums)
    n, S_o, S_oo = (_t(v).to(S_s.device) for v in obs_moments)
    mean_s, mean_o = _ratio(S_s, n), _ratio(S_o, n)
    var_s = torch.clamp_min(_ratio(S_ss, n) - mean_s * mean_s, 0.0)
    var_o = torch.clamp_min(_ratio(S_oo, n) - mean_o * mean_o, 0.0)
    cov = _ratio(S_so, n) - mean_s * mean_o
    nse = 1.0 - _ratio(S_ee, n * var_o)
    rmse = torch.sqrt(_ratio(S_ee, n))
    bias = _ratio(S_s - S_o, n)
    r = _ratio(cov, torch.sqrt(var_s * var_o))
    alpha = torch.sqrt(_ratio(var_s, var_o))
    nonzero = torch.where(mean_o != 0, mean_o, torch.ones_like(mean_o))
    beta = torch.where(mean_o != 0, mean_s / nonzero, torch.full_like(mean_s, float("nan")))
    kge = 1.0 - torch.sqrt((r - 1.0) ** 2 + (alpha - 1.0) ** 2 + (beta - 1.0) ** 2)
    return {"n": n.clone(), "nse": nse, "kge": kge, "r": r, "alpha": alpha, "beta": beta, "rmse": rmse, "bias": bias}


def series_sums(sim, obs) -> Tuple[torch.Tensor, Tuple[torch.Tensor, torch.Tensor, torch.Tensor]]:
    """The sums the kernel forms, from series ``sim[T, M]`` and ``obs[T, M]``: ``([4, M] sums, (n, S_o, S_oo))``.

    Steps are added in time order with one rounding per operation, exactly as the kernel adds them, so a series the
    engine recorded gives the device's sums bit for bit.  Steps with a non-finite observation are skipped."""
    s, o = _t(sim), _t(obs)
    if s.shape != o.shape or s.dim() != 2:
        raise ValueError(f"sim and obs must both be [T, M]; got {tuple(s.shape)} and {tuple(o.shape)}")
    M = s.shape[1]
    acc = torch.zeros(4, M, dtype=torch.float64, device=s.device)
    mom = torch.zeros(3, M, dtype=torch.float64, device=s.device)
    o = o.to(s.device)
    for t in range(s.shape[0]):
        accumulate_step(acc, mom, s[t], o[t])
    return acc, (mom[0], mom[1], mom[2])


def accumulate_step(acc: torch.Tensor, mom, s: torch.Tensor, o: torch.Tensor) -> None:
    """One scored step, in place: the kernel's ``d = s - o; S_s += s; S_ss += s*s; S_so += s*o; S_ee += d*d`` where
    ``o`` is finite, and the observation moments ``n += 1, S_o += o, S_oo += o*o`` (``mom`` may be None)."""
    f = torch.isfinite(o)
    zero = torch.zeros_like(o)
    if acc is not None:
        d = s - o
        for row, v in enumerate((s, s * s, s * o, d * d)):
            acc[row] = torch.where(f, acc[row] + v, acc[row])
    if mom is not None:
        oo = torch.where(f, o, zero)
        mom[0] += f.to(torch.float64)
        mom[1] = torch.where(f, mom[1] + oo, mom[1])
        mom[2] = torch.where(f, mom[2] + oo * oo, mom[2])


def series_scores(sim, obs) -> dict:
    """``skill_scores`` of series ``sim[T, M]`` against ``obs[T, M]`` (non-finite observations are not scored)."""
    acc, mom = series_sums(sim, obs)
    return skill_scores(acc, mom)
