"""The sampler between fits: what decides WHICH parameter sets the GPU evaluates next.

Mirrors /root/reference/R/adaptive_sampling.R: the Latin-hypercube design of initial_parameter_optimization
(:419-425), weighted_kde (:1901-1935), calculate_weighted_marginals (:2457-2519), generate_kde_samples (:1804-1885),
the draw / evaluate / append loop of adaptive_MC_sampling (:1593-1790), and clean_data / detect_outliers_mad
(R/data_preprocessing.R:864-879, :956-996) which they call.  Same names, arguments, column names and messages.

What changes is the shape of the work.  The reference runs one chain per process; every iteration of a chain reads
the CSV, builds four 512-point KDEs with an R-level loop over the evaluation points (forked again with mclapply),
draws ONE parameter set and spends `folds` fits on it.  `adaptive_mc_batch` keeps all chains in one process: the
marginals are computed once per round (a 512 x samples broadcast), every chain draws from them, and the draws of all
chains x folds go to the device as one topolow_fit_batch call (cv.likelihood_batch) - the batch the GPU needs to stay
full.  A sample table is a dict of equal-length numpy arrays keyed by the reference's column names.

R's RNG cannot be reproduced: every random step takes a numpy Generator (the tests inject the same uniforms into
this module and into the loop restatement in oracle/r_glue.py).  lhs::maximinLHS is an unpinned CRAN dependency
(DESCRIPTION:32); the design here is scipy's Latin hypercube with a maximin pick among candidates - same marginal
stratification, not the same points.
"""
from __future__ import annotations

import math
import warnings

import numpy as np

PAR_NAMES = ("log_N", "log_k0", "log_cooling_rate", "log_c_repulsion")
TEMPERATURE = 0.1          # R/adaptive_sampling.R:1834, :2499


def detect_outliers_mad(data, k=3):
    """R/data_preprocessing.R:956-996: |x - median| > k * 1.4826 * median(|x - median|); NA stays NA (False in the mask)."""
    if not isinstance(k, (int, float)) or k <= 0:
        raise ValueError("k must be a positive number")
    x = np.asarray(data, dtype=np.float64)
    med = np.nanmedian(x) if np.any(~np.isnan(x)) else np.nan
    mad = 1.4826 * np.nanmedian(np.abs(x - med)) if np.any(~np.isnan(x)) else np.nan
    with np.errstate(invalid="ignore"):
        mask = np.abs(x - med) > k * mad
    return dict(outlier_mask=mask, stats=dict(median=med, mad=mad, n_outliers=int(np.sum(mask))))


def clean_data(x, k=3):
    """R/data_preprocessing.R:864-879: outliers become NA."""
    x = np.array(x, dtype=np.float64, copy=True)
    x[detect_outliers_mad(x, k)["outlier_mask"]] = np.nan
    return x


def weighted_kde(x, weights, n=512, from_=None, to=None):
    """R/adaptive_sampling.R:1901-1935: Gaussian KDE with Silverman's bandwidth 1.06 sd(x) n^(-1/5) on n equally spaced
    points from min - bw to max + bw.  One broadcast instead of an R-level loop (forked with mclapply) over the points."""
    x = np.asarray(x, dtype=np.float64)
    w = np.asarray(weights, dtype=np.float64)
    w = w / w.sum()
    bw = 1.06 * np.std(x, ddof=1) * len(x) ** (-1 / 5)
    lo = x.min() - bw if from_ is None else from_
    hi = x.max() + bw if to is None else to
    pts = lo + np.arange(n) * ((hi - lo) / (n - 1))            # seq(from, to, length.out = n)
    with np.errstate(invalid="ignore", divide="ignore"):
        z = (pts[:, None] - x[None, :]) / bw
        dens = (w[None, :] * np.exp(-0.5 * z * z)).sum(axis=1) / (bw * math.sqrt(2 * math.pi))
    return dict(x=pts, y=dens, bw=bw)


def _as_table(samples):
    if hasattr(samples, "to_dict") and hasattr(samples, "columns"):          # pandas
        return {c: np.asarray(samples[c]) for c in samples.columns}
    return {k: np.asarray(v) for k, v in samples.items()}


def _rows(table, keep):
    return {k: v[keep] for k, v in table.items()}


def _softmax_weights(score):
    """exp(-(score - min) / (range + 1e-10) / temperature), normalised (R/adaptive_sampling.R:1830-1836, :2496-2501)."""
    norm = (score - score.min()) / (score.max() - score.min() + 1e-10)
    w = np.exp(-norm / TEMPERATURE)
    return w / w.sum()


def calculate_weighted_marginals(samples):
    """R/adaptive_sampling.R:2457-2519: four weighted KDEs, weights = temperature softmax of log(Holdout_MAE)
    (low MAE = high weight) after MAD cleaning of the MAE column."""
    t = _as_table(samples)
    required = list(PAR_NAMES) + ["Holdout_MAE"]
    missing = [c for c in required if c not in t]
    if missing:
        raise ValueError("Missing required columns: " + ", ".join(missing))
    if not all(np.asarray(t[c]).dtype.kind in "fiu" for c in required):
        raise ValueError("All required parameter and Holdout_MAE columns must be numeric.")
    t = {k: (v.astype(np.float64) if k in required else v) for k, v in t.items()}
    mae = t["Holdout_MAE"]
    if np.all(np.isinf(mae)):
        raise ValueError("All Holdout_MAE values are infinite")
    if np.any(np.isnan(mae)):
        warnings.warn("NA values in the Holdout_MAE column will be removed.")
        t = _rows(t, ~np.isnan(t["Holdout_MAE"]))
    if np.any(t["Holdout_MAE"] <= 0):
        warnings.warn("Non-positive MAE values found and will be removed.")
        t = _rows(t, t["Holdout_MAE"] > 0)
    if len(t["Holdout_MAE"]) < 2:
        raise ValueError("At least two valid samples are required after filtering.")
    t["Holdout_MAE"] = clean_data(t["Holdout_MAE"], k=3)
    with np.errstate(invalid="ignore"):
        t = _rows(t, ~np.isnan(t["Holdout_MAE"]) & (t["Holdout_MAE"] > 0))
    weights = _softmax_weights(np.log(t["Holdout_MAE"]))
    return {v: weighted_kde(t[v], weights) for v in PAR_NAMES}


def _approx(x, y, xout):
    """stats::approx(x, y, xout, rule = 2): linear interpolation, ties in x collapsed to the mean of their y,
    constant beyond the ends."""
    order = np.argsort(x, kind="stable")
    xs, ys = np.asarray(x)[order], np.asarray(y)[order]
    ux, inv = np.unique(xs, return_inverse=True)
    uy = np.bincount(inv, weights=ys) / np.bincount(inv)
    return np.interp(xout, ux, uy)


def generate_kde_samples(samples, n, epsilon=0, *, rng=None):
    """R/adaptive_sampling.R:1804-1885: n new parameter sets, every parameter drawn independently from its weighted
    KDE by inverse-transform sampling.  Kept as the reference has it, including two things that look unintended there:
    the weights are the softmax of -log(MAE) normalised the same way, which favours HIGH MAE (:1830-1835 - the sign is
    flipped relative to calculate_weighted_marginals), and the epsilon branch computes a wider bandwidth that
    weighted_kde is never given (:1850-1857) - only its runif(1) is consumed."""
    rng = rng or np.random.default_rng()
    t = _as_table(samples)
    if "Holdout_MAE" not in t:
        raise ValueError("Samples data frame must contain a 'Holdout_MAE' column.")
    t = {k: (v.astype(np.float64) if k in PAR_NAMES or k == "Holdout_MAE" else v) for k, v in t.items()}
    t["Holdout_MAE"] = clean_data(t["Holdout_MAE"], k=3)
    with np.errstate(invalid="ignore"):
        t = _rows(t, ~np.isnan(t["Holdout_MAE"]) & (t["Holdout_MAE"] > 0))
    if len(t["Holdout_MAE"]) < 2:
        raise ValueError("Insufficient samples remaining after removing NA & outliers (need at least 2)")
    weights = _softmax_weights(-np.log(t["Holdout_MAE"]))
    if np.any(np.isnan(weights)):
        warnings.warn("NA values in weights, replacing with uniform weights")
        weights = np.full(len(weights), 1.0 / len(weights))
    out = {}
    for param in PAR_NAMES:
        rng.random()                                    # runif(1) < epsilon: the draw happens, its outcome changes nothing
        kde = weighted_kde(t[param], weights)
        if np.any(np.isnan(kde["y"])) or np.any(kde["y"] < 0):
            warnings.warn("Invalid KDE values for parameter %s - using uniform sampling" % param)
            out[param] = rng.uniform(t[param].min(), t[param].max(), size=n)
            continue
        u = rng.random(n)
        cdf = np.cumsum(kde["y"]) / np.sum(kde["y"])
        if np.any(np.isnan(cdf)):
            warnings.warn("NA values in CDF for parameter %s - using uniform sampling" % param)
            out[param] = rng.uniform(t[param].min(), t[param].max(), size=n)
            continue
        out[param] = _approx(cdf, kde["x"], u)
    return out


def lhs_design(num_samples, N_range, k0_range, c_repulsion_range, cooling_rate_range, *, rng=None, candidates=8):
    """R/adaptive_sampling.R:419-425: a 4-column Latin hypercube mapped through qunif; N = floor(qunif(u, N_min, N_max + 1)).
    The hypercube is scipy's, the maximin criterion a best-of-`candidates` pick (lhs::maximinLHS is unpinned)."""
    from scipy.stats import qmc
    rng = rng or np.random.default_rng()
    best, best_d = None, -1.0
    for _ in range(max(1, candidates)):
        u = qmc.LatinHypercube(d=4, seed=rng).random(num_samples)
        if num_samples > 1:
            d = np.linalg.norm(u[:, None, :] - u[None, :, :], axis=2)
            d = d[np.triu_indices(num_samples, 1)].min()
        else:
            d = 0.0
        if d > best_d:
            best, best_d = u, d
    q = lambda col, lo, hi: lo + best[:, col] * (hi - lo)            # qunif
    return dict(N=np.floor(q(0, N_range[0], N_range[1] + 1)).astype(np.int64), k0=q(1, *k0_range),
                c_repulsion=q(2, *c_repulsion_range), cooling_rate=q(3, *cooling_rate_range))


def draw_from_marginals(marginals, rng, size=1):
    """sample(m$x, size, prob = m$y) per parameter (R/adaptive_sampling.R:1636-1643) -> dict of arrays."""
    out = {}
    for v in PAR_NAMES:
        y = np.asarray(marginals[v]["y"], dtype=np.float64)
        out[v] = rng.choice(marginals[v]["x"], size=size, p=y / y.sum())
    return out


def adaptive_mc_batch(samples, dissimilarity_matrix, iterations, chains, mapping_max_iter, relative_epsilon, folds=20,
                      preserve_order=True, *, rng=None, evaluate=None, device=0, verbose=False, interrupt=None,
                      mode="coloured"):
    """`chains` chains of adaptive_MC_sampling (R/adaptive_sampling.R:1593-1790) advanced together: per round the
    weighted marginals of the shared table are computed once, every chain draws one parameter set, all chains x folds
    fits run as one device batch, valid rows are appended (invalid evaluations are skipped, :1683-1686).  Returns the
    grown table.  `evaluate(matrix, param_sets)` stands in for cv.likelihood_batch in CPU tests.
    The reference's chains are separate processes that append to one CSV whenever they finish; here a round's draws
    all see the table as it was when the round began.
    `interrupt` is polled while a round's batch runs (cv.likelihood_batch); when it returns True the batch stops and
    TopolowError(ERR_INTERRUPTED) is raised.  `device` may be a sequence of ordinals (cv.likelihood_batch).  `mode`
    ("coloured" or "rowblock", as in cv.likelihood_batch) is the mode of every fit: "rowblock" for large maps and for
    N above 16."""
    rng = rng or np.random.default_rng()
    table = {k: np.array(v, copy=True) for k, v in _as_table(samples).items()}
    required = list(PAR_NAMES) + ["NLL", "Holdout_MAE"]
    missing = [c for c in required if c not in table]
    if missing:
        raise ValueError("Samples file missing required columns: " + ", ".join(missing))
    if evaluate is None:
        from . import cv

        def evaluate(matrix, sets):
            return cv.likelihood_batch(matrix, sets, mapping_max_iter, relative_epsilon, folds, preserve_order,
                                       rng=rng, device=device, interrupt=interrupt, mode=mode)
    for it in range(int(iterations)):
        try:
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                marginals = calculate_weighted_marginals(table)
        except ValueError as e:
            if verbose:
                print("  Warning: Failed to calculate marginals: %s" % e)
            continue
        draws = draw_from_marginals(marginals, rng, size=int(chains))
        sets = [dict(N=int(round(math.exp(draws["log_N"][c]))), k0=math.exp(draws["log_k0"][c]),
                     cooling_rate=math.exp(draws["log_cooling_rate"][c]), c_repulsion=math.exp(draws["log_c_repulsion"][c]))
                for c in range(int(chains))]
        results = evaluate(dissimilarity_matrix, sets)
        for c, res in enumerate(results):
            if res is None or math.isnan(res["Holdout_MAE"]) or math.isnan(res["NLL"]):
                continue
            row = {v: draws[v][c] for v in PAR_NAMES}
            row.update(Holdout_MAE=res["Holdout_MAE"], NLL=res["NLL"], mean_iter=res.get("mean_iter", np.nan),
                       pct_converged=res.get("pct_converged", np.nan))
            for k in table:
                table[k] = np.append(table[k], row.get(k, np.nan))
        if verbose:
            print("  round %d/%d: %d rows" % (it + 1, iterations, len(table["Holdout_MAE"])))
    return table
