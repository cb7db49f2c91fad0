"""The batched cross-validation evaluator: mirror of likelihood_function()
(/root/reference/R/adaptive_sampling.R:2552-2726) and of the residual part of
error_calculator_comparison() (/root/reference/R/error_metrics.R:89-143) that it consumes.

The reference runs the `folds` fits of one parameter sample one after another (or forks them with
mclapply); here all folds of all samples handed to `likelihood_batch` go to the GPU in ONE
topolow_fit_batch call - the fork boundary that would break CUDA (SURVEY.md section 3.3) is gone.
"""
from __future__ import annotations

import math
import warnings

import numpy as np

from . import _lib
from .core import build_problem, build_problem_coo, parse_dissimilarity, random_initial_positions

# the modes a fit batch runs (core.euclidean_embedding's names); replay fits are single fits only
_BATCH_MODES = {"coloured": _lib.MODE_COLOURED, "rowblock": _lib.MODE_ROWBLOCK}


def error_calculator_comparison(predicted_dissimilarities, true_dissimilarities, input_dissimilarities=None):
    """R/error_metrics.R:55-144.  Returns report_df columns (flattened column-major, NaN = NA)
    and Completeness."""
    if not isinstance(predicted_dissimilarities, np.ndarray) or not isinstance(true_dissimilarities, np.ndarray) \
            or predicted_dissimilarities.ndim != 2 or true_dissimilarities.ndim != 2:
        raise ValueError("predicted_dissimilarities and true_dissimilarities must be matrices")
    if input_dissimilarities is None:
        input_dissimilarities = true_dissimilarities
    if not isinstance(input_dissimilarities, np.ndarray) or input_dissimilarities.ndim != 2:
        raise ValueError("input_dissimilarities must be a matrix")
    if predicted_dissimilarities.shape != true_dissimilarities.shape or \
            predicted_dissimilarities.shape != input_dissimilarities.shape:
        raise ValueError("All matrices must have the same dimensions")

    def as_numeric(m):  # threshold strings and NA both become NA
        v, c, na = parse_dissimilarity(m)
        return np.where(na | (c != 0), np.nan, v).ravel(order="F")

    input_vec = as_numeric(input_dissimilarities)
    truth_vec = as_numeric(true_dissimilarities)
    pred_vec = np.asarray(predicted_dissimilarities, dtype=np.float64).ravel(order="F")
    missing = np.isnan(input_vec)
    in_err = truth_vec - np.where(missing, np.nan, pred_vec)
    out_err = truth_vec - np.where(missing, pred_vec, np.nan)
    nz = ~np.isnan(truth_vec) & (np.nan_to_num(truth_vec, nan=0.0) > 0)
    in_pct = np.full_like(in_err, np.nan)
    out_pct = np.full_like(out_err, np.nan)
    with np.errstate(invalid="ignore", divide="ignore"):
        in_pct[nz] = in_err[nz] / truth_vec[nz] * 100
        out_pct[nz] = out_err[nz] / truth_vec[nz] * 100
    validation_count = int(np.sum(~np.isnan(truth_vec[missing])))
    if validation_count > 0:
        completeness = int(np.sum(~np.isnan(out_err))) / validation_count
    else:
        total_possible = int(np.sum(~np.isnan(truth_vec)))
        completeness = int(np.sum(~np.isnan(pred_vec))) / total_possible if total_possible > 0 else 0
    return dict(report_df=dict(InSampleError=in_err, OutSampleError=out_err, InSamplePercentageError=in_pct,
                               OutSamplePercentageError=out_pct),
                Completeness=completeness)


def make_folds(dissimilarity_matrix, folds, rng):
    """R/adaptive_sampling.R:2568-2598.  Returns a list of column-major linear index arrays."""
    _, _, is_na = parse_dissimilarity(dissimilarity_matrix)
    n = is_na.shape[0]
    pool = ~is_na
    holdout_size = int(pool.sum()) // (folds * 2)
    out = []
    for _ in range(folds):
        if int(pool.sum()) < holdout_size:
            warnings.warn("Could not create all folds due to data sparsity. Using fewer folds.")
            break
        lin = np.flatnonzero(pool.ravel(order="F"))
        pick = rng.choice(lin, size=holdout_size, replace=False)
        out.append(pick)
        r, c = pick % n, pick // n
        pool[r, c] = False
        pool[c, r] = False
    return out


def create_cv_folds(dissimilarity_matrix, ground_truth_matrix=None, n_folds=10, random_seed=None, *, rng=None):
    """R/utils.R:69-150: a list of {truth, train} matrices; every fold masks floor(#non-NA / (2 n_folds)) cells drawn
    from the cells no earlier fold took, symmetrically.  `rng` (numpy Generator) stands in for R's sample();
    `random_seed` seeds a fresh one.  Matrices are float arrays with NaN = NA or object arrays, as everywhere."""
    if random_seed is not None:
        if not isinstance(random_seed, (int, float, np.integer, np.floating)) or random_seed != round(random_seed):
            raise ValueError("`random_seed` must be an integer.")
        rng = np.random.default_rng(int(random_seed))
    rng = rng or np.random.default_rng()
    if not isinstance(dissimilarity_matrix, np.ndarray) or dissimilarity_matrix.ndim != 2:
        raise ValueError("`dissimilarity_matrix` must be a matrix.")
    if ground_truth_matrix is not None:
        if not isinstance(ground_truth_matrix, np.ndarray) or ground_truth_matrix.ndim != 2:
            raise ValueError("`ground_truth_matrix` must be NULL or a matrix.")
        if ground_truth_matrix.shape != dissimilarity_matrix.shape:
            raise ValueError("`dissimilarity_matrix` and `ground_truth_matrix` must have the same dimensions.")
    if not isinstance(n_folds, (int, float, np.integer, np.floating)) or n_folds < 2 or n_folds != round(n_folds):
        raise ValueError("`n_folds` must be an integer greater than or equal to 2.")
    n_folds = int(n_folds)
    nrow, ncol = dissimilarity_matrix.shape
    if n_folds > nrow:
        raise ValueError("`n_folds` cannot be larger than the number of rows in the matrix.")
    truth = ground_truth_matrix if ground_truth_matrix is not None else dissimilarity_matrix
    pool = ~parse_dissimilarity(dissimilarity_matrix)[2]
    holdout_size = int(pool.sum()) // (n_folds * 2)
    na_cell = None if dissimilarity_matrix.dtype.kind == "O" else np.nan
    out = []
    for _ in range(n_folds):
        if int(pool.sum()) < holdout_size:
            warnings.warn("Could not create all requested folds due to data sparsity. Returning fewer folds.")
            break
        lin = np.flatnonzero(pool.ravel(order="F"))                 # which(!is.na(sampling_pool)), column-major
        pick = rng.choice(lin, size=holdout_size, replace=False)
        # the reference turns the linear index into (row, col) with `%/% nrow` for the row and `%% ncol` for the
        # column (R/utils.R:129-130) - transposed for a column-major index, harmless because the mask is symmetric
        r, c = pick // nrow, pick % ncol
        train = dissimilarity_matrix.copy()
        train[r, c] = na_cell
        train[c, r] = na_cell
        pool[r, c] = False
        pool[c, r] = False
        out.append(dict(truth=truth, train=train))
    return out


# ---------------------------------------------------------------------------------------------
# The same folds on an edge list: nothing n x n
# ---------------------------------------------------------------------------------------------
def make_folds_cells(n, cell_i, cell_j, folds, rng, diagonal=True):
    """R/adaptive_sampling.R:2568-2598 on the non-NA cells of a symmetric matrix given as its upper-triangle pairs
    (cell_i < cell_j) + optionally the n diagonal cells.  The pool holds every non-NA cell: the diagonal ones and BOTH
    orientations of every pair; a drawn cell takes its mirror out of the pool with it.  Returns one array of cell ids
    per fold: id < n = diagonal cell (id, id); n + 2p = pair p as (i, j), n + 2p + 1 = pair p as (j, i).
    Walking the pool in id order instead of column-major order changes which uniform draw maps to which cell, not
    the distribution."""
    base = n if diagonal else 0
    total = base + 2 * len(cell_i)
    pool = np.ones(total, dtype=bool)
    holdout_size = total // (folds * 2)
    out = []
    for _ in range(folds):
        if int(pool.sum()) < holdout_size:
            warnings.warn("Could not create all folds due to data sparsity. Using fewer folds.")
            break
        pick = rng.choice(np.flatnonzero(pool), size=holdout_size, replace=False)
        out.append(pick)
        pool[pick] = False
        pr = pick[pick >= base] - base
        pool[base + (pr ^ 1)] = False                                # the mirror cell
    return out


def fold_problem_cells(full, picks, base):
    """Training problem of one fold + its out-of-sample cells from the full problem (build_problem_coo with
    preserve_order = TRUE) and the fold's drawn cell ids: what mask + build_problem + error_calculator_comparison
    derive from matrices (R/adaptive_sampling.R:2608-2647)."""
    n = full["n"]
    ci, cj = full["cell_i"], full["cell_j"]
    held_pair = np.zeros(len(ci), dtype=bool)
    held_pair[(picks[picks >= base] - base) >> 1] = True
    held_diag = picks[picks < base]
    deg = full["degrees"].astype(np.int64).copy()
    deg -= np.bincount(ci[held_pair], minlength=n) + np.bincount(cj[held_pair], minlength=n)
    deg[held_diag] -= 1
    keep = ~held_pair
    measured = keep & ~np.isnan(full["cell_value"]) & (full["cell_value"] != np.inf)
    prob = dict(n=n, order=None, degrees=deg.astype(np.int32), edge_i=ci[measured].astype(np.int32),
                edge_j=cj[measured].astype(np.int32), edge_dist=full["cell_value"][measured].astype(np.float64),
                edge_thresh=full["cell_code"][measured].astype(np.int32))
    # out-of-sample cells: masked in the training matrix, numeric (not a threshold) in the truth; the flattened matrices
    # list a pair in both orientations and a masked diagonal cell once (truth 0)
    out = held_pair & full["plain"]
    hi = np.concatenate([ci[out], cj[out], held_diag]).astype(np.int32)
    hj = np.concatenate([cj[out], ci[out], held_diag]).astype(np.int32)
    ht = np.concatenate([full["cell_value"][out], full["cell_value"][out], np.zeros(len(held_diag))])
    return prob, hi, hj, ht


def _fold_job(value, code, is_na, holdout, preserve_order):
    """Training problem of one fold (R/adaptive_sampling.R:2608-2616) + its held-out cells."""
    n = value.shape[0]
    r, c = holdout % n, holdout // n
    na_train = is_na.copy()
    na_train[r, c] = True
    na_train[c, r] = True
    train = np.where(na_train, np.nan, value)
    # rebuild a matrix build_problem understands: thresholds survive through (value, code)
    obj = train.astype(object)
    for a, b in zip(*np.nonzero((code != 0) & ~na_train)):
        obj[a, b] = (">" if code[a, b] > 0 else "<") + repr(float(value[a, b]))
    prob = build_problem(obj if (code != 0).any() else train, preserve_order)
    # out-of-sample cells: NA (or threshold) in the training matrix, numeric in the truth
    truth_num = np.where(is_na | (code != 0), np.nan, value)
    train_num = np.where(na_train | (code != 0), np.nan, value)
    cells = np.isnan(train_num) & ~np.isnan(truth_num)
    ci, cj = np.nonzero(cells)
    return prob, ci.astype(np.int32), cj.astype(np.int32), truth_num[ci, cj]


def likelihood_batch(dissimilarity_matrix, samples, mapping_max_iter, relative_epsilon, folds=20,
                     preserve_order=True, *, fold_indices=None, init_list=None, rng=None, seed=0, device=0,
                     precision="f32", interrupt=None, mode="coloured"):
    """Evaluate many parameter samples at once.  `samples` is a list of dicts with keys N, k0,
    cooling_rate, c_repulsion; returns one likelihood_function() result per sample.  All
    len(samples) x folds fits run in a single topolow_fit_batch call.

    The folds are drawn ONCE for the whole batch (or taken from `fold_indices`): every sample is scored on
    the same hold-out cells, and topolow_fit_batch builds the device records of a fold once.  The
    reference draws fresh folds inside every likelihood_function call (R/adaptive_sampling.R:2568-2598);
    the distribution of a sample's score is the same, the scores of different samples are no longer
    independent (common random numbers - which is what comparing samples wants).  Call
    likelihood_function per sample for the reference's behaviour.

    preserve_order defaults to True here because fold residuals are aligned by position; the
    reference re-aligns by row names (R/error_metrics.R:76-87) which an unnamed matrix lacks.

    device: a CUDA ordinal, or a sequence of ordinals over which the batch is dealt (_lib.fit_batch); the scores do
    not depend on it.

    interrupt: a callable polled while the fits run (see _lib.fit_batch); when it returns True the batch stops and
    TopolowError(ERR_INTERRUPTED) is raised.

    mode: "coloured" (the default) or "rowblock", the names core.euclidean_embedding takes, for every fit of the batch.
    "rowblock" is the mode for large maps and for N of 17 to 32 (the coloured mode takes N up to 16); each fold fit is
    then exactly the single row-block fit."""
    rng = rng or np.random.default_rng(seed)
    value, code, is_na = parse_dissimilarity(dissimilarity_matrix)
    if fold_indices is None:
        fold_indices = make_folds(dissimilarity_matrix, folds, rng)
    fold_jobs = [_fold_job(value, code, is_na, np.asarray(h), preserve_order) for h in fold_indices]
    return _run_folds(fold_jobs, samples, mapping_max_iter, relative_epsilon, init_list, rng, seed, device, precision,
                      interrupt, mode)


def likelihood_batch_coo(n, rows, cols, values, samples, mapping_max_iter, relative_epsilon, folds=20, *, diagonal=True,
                         fold_cells=None, init_list=None, rng=None, seed=0, device=0, precision="f32", interrupt=None,
                         mode="coloured"):
    """likelihood_batch for a dissimilarity table (0-based rows / cols, values numbers or threshold strings): the folds
    are drawn and masked on the cell list (make_folds_cells / fold_problem_cells), nothing n x n is built, and the
    hold-out cells are scored on the device inside each fit.  Row order is the table's (preserve_order = TRUE).
    `fold_cells` injects the drawn cell ids (see make_folds_cells); `interrupt` and `mode` as in likelihood_batch."""
    rng = rng or np.random.default_rng(seed)
    full = build_problem_coo(n, rows, cols, values, preserve_order=True, diagonal=diagonal)
    base = n if diagonal else 0
    if fold_cells is None:
        fold_cells = make_folds_cells(n, full["cell_i"], full["cell_j"], folds, rng, diagonal)
    fold_jobs = []
    for picks in fold_cells:
        prob, hi, hj, ht = fold_problem_cells(full, np.asarray(picks), base)
        kept = prob["edge_thresh"] == 0       # R/core.R:407-409: the largest plain number of the fold's TRAINING matrix
        prob["init_step"] = (max(float(prob["edge_dist"][kept].max()), 0.0) if kept.any() else 0.0) / n
        fold_jobs.append((prob, hi, hj, ht))
    return _run_folds(fold_jobs, samples, mapping_max_iter, relative_epsilon, init_list, rng, seed, device, precision,
                      interrupt, mode)


def _initial_positions(prob, ndim, rng):
    if "value" in prob:
        return random_initial_positions(prob["value"], prob["code"], prob["is_na"], ndim, rng)
    steps = rng.uniform(0.0, 2.0 * prob["init_step"], size=(prob["n"] - 1, ndim))          # R/core.R:407-415
    return np.vstack([np.zeros((1, ndim)), np.cumsum(steps, axis=0)])


def _run_folds(fold_jobs, samples, mapping_max_iter, relative_epsilon, init_list, rng, seed, device, precision,
               interrupt=None, mode="coloured"):
    """All len(samples) x len(fold_jobs) fits in one topolow_fit_batch call, pooled as R/adaptive_sampling.R:2695-2725."""
    prec_c = {"f32": _lib.PREC_F32, "f64": _lib.PREC_F64_EXACT}[precision]
    if mode not in _BATCH_MODES:
        raise ValueError(f"mode must be one of {sorted(_BATCH_MODES)}, not {mode!r}")
    # hold-out cells in the row numbering of the fold's training problem: they are scored on the device
    # at the end of each fit (topolow_problem.holdout_*), the positions need not come back for that
    fold_holdout = []
    for prob, ci, cj, tr in fold_jobs:
        if prob["order"] is not None:
            inv = np.empty(len(prob["order"]), dtype=np.int64)
            inv[prob["order"]] = np.arange(len(prob["order"]))
            ci, cj = inv[ci], inv[cj]
        fold_holdout.append((np.ascontiguousarray(ci, dtype=np.int32), np.ascontiguousarray(cj, dtype=np.int32),
                             np.ascontiguousarray(tr, dtype=np.float64)))
    jobs, meta = [], []
    for s_idx, s in enumerate(samples):
        for f_idx, (prob, ci, cj, tr) in enumerate(fold_jobs):
            ndim = int(s["N"])
            if len(prob["edge_i"]) == 0:
                meta.append((s_idx, f_idx, None))
                continue
            if init_list is not None:
                init = init_list[s_idx][f_idx]
            else:
                init = _initial_positions(prob, ndim, rng)
            jobs.append(dict(initial_positions=init, degrees=prob["degrees"], edge_i=prob["edge_i"],
                             edge_j=prob["edge_j"], edge_dist=prob["edge_dist"], edge_thresh=prob["edge_thresh"],
                             n_iter=int(mapping_max_iter), k0=s["k0"], cooling_rate=s["cooling_rate"],
                             c_repulsion=s["c_repulsion"], relative_epsilon=relative_epsilon, convergence_window=5,
                             precision=prec_c, seed=seed + 1000003 * s_idx + f_idx, holdout=fold_holdout[f_idx],
                             mode=_BATCH_MODES[mode]))
            meta.append((s_idx, f_idx, len(jobs) - 1))
    extra = {} if interrupt is None else {"interrupt": interrupt}
    results = _lib.fit_batch(jobs, device=device, **extra) if jobs else []

    per_sample = [[] for _ in samples]
    for s_idx, f_idx, j in meta:
        row = dict(Holdout_MAE=math.nan, n_samples=0, sum_abs_errors=0.0, iter=math.nan, converged=0)
        if j is not None and results[j].get("status", 1) == _lib.OK:
            res = results[j]
            s_abs, cnt = res["holdout_sum_abs"], res["holdout_count"]
            row = dict(Holdout_MAE=s_abs / cnt if cnt > 0 else math.nan, n_samples=cnt, sum_abs_errors=s_abs,
                       iter=res["iterations"], converged=int(res["converged"]))
        per_sample[s_idx].append(row)

    out = []
    for rows in per_sample:  # R/adaptive_sampling.R:2695-2725
        valid = [r for r in rows if not math.isnan(r["Holdout_MAE"])]
        if not valid:
            out.append(dict(Holdout_MAE=math.nan, NLL=math.nan, mean_iter=math.nan, pct_converged=math.nan, folds=rows))
            continue
        total = sum(r["n_samples"] for r in valid)
        tabs = sum(r["sum_abs_errors"] for r in valid)
        pooled = tabs / total if total > 0 else math.nan
        nll = math.nan if math.isnan(pooled) else total * (1 + (math.log(2 * pooled) if pooled > 0 else -math.inf))
        out.append(dict(Holdout_MAE=pooled, NLL=nll, mean_iter=float(np.mean([r["iter"] for r in valid])),
                        pct_converged=float(np.mean([r["converged"] for r in valid]) * 100), folds=rows))
    return out


def likelihood_function(dissimilarity_matrix, mapping_max_iter, relative_epsilon, N, k0, cooling_rate, c_repulsion,
                        folds=20, num_cores=1, preserve_order=True, *, interrupt=None, mode="coloured", **kw):
    """Single-sample form with the reference's signature (R/adaptive_sampling.R:2552-2555);
    num_cores is accepted and ignored (the folds already run concurrently on the device).
    `interrupt` and `mode` as in likelihood_batch."""
    return likelihood_batch(dissimilarity_matrix, [dict(N=N, k0=k0, cooling_rate=cooling_rate,
                                                        c_repulsion=c_repulsion)], mapping_max_iter,
                            relative_epsilon, folds, preserve_order, interrupt=interrupt, mode=mode, **kw)[0]
