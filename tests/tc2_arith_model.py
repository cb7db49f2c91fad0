"""The arithmetic of the two-GEMM repulsion pass (topolow_b200/csrc/rowblock_tc2.cuh) restated in numpy, number format
by number format - test infrastructure.  Nothing under topolow_b200/ imports it.

  image        x = P - centre in FP32 (centre: the centroid of the positions, summed in FP64, rounded to FP32), zero padded
               to 16 coordinates; split into a TF32 part (cvt.rna) and a remainder (truncated by the tensor core)
  GEMM 1       S = h_i + h_j - x_i . x_j  (h = |x|^2 / 2 as TF32 part + remainder) from hi.hi + hi.lo + lo.hi, FP32
  near pairs   S < 3.01e-3 h_i (and S < kSeriesNearS = 0.005 in the series form) get weight 0 and are re-done from the
               coordinate differences (near_fix: FP32 differences, here in FP64 - they are not what is modelled)
  weights      series form: q = S^-1/2, w = q^3 p(q) (the cubic of the kernel); otherwise (sqrt(2 S) + 0.01)^-3; then
               truncated to TF32 by the tensor core
  GEMM 2       per chunk of 2048 partners: sum_j w x_j with x_j rounded to TF32 and sum_j w, both FP32; the chunk's
               partial sum is sum w x_j - x_i sum w

`tensor_pass` returns sum_j w_ij (x_j - x_i) per row.  Its keyword arguments are the mutants the tests use to show that
their bars catch a kernel that is subtly wrong."""
import numpy as np

CHUNK = 2048
NEAR_TAU = np.float32(3.01e-3)
SERIES_NEAR_S = np.float32(0.005)
SERIES = (np.float32(-9.3722616e-07), np.float32(1.0345994e-4), np.float32(-7.492801e-3), np.float32(0.35355023))


def tf32_rna(x):
    """cvt.rna.tf32.f32: 10 explicit mantissa bits, ties away from zero."""
    u = np.asarray(x, np.float32).view(np.uint32).astype(np.uint64)
    return (((u + 0x1000) & 0xFFFFE000) & 0xFFFFFFFF).astype(np.uint32).view(np.float32)


def tf32_trunc(x):
    """What the tensor core does to an FP32 operand."""
    return (np.asarray(x, np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)


def centre_of(P):
    return np.asarray(P, np.float32).astype(np.float64).mean(0).astype(np.float32)


def image(P, pad_from_centre=False):
    """(rows' image, partners' image, centre): coordinates minus the centre in FP32, zero padded to 16.
    pad_from_centre (a mutant): the partners' image takes its first pad coordinate from the centre instead of 0."""
    P32 = np.asarray(P, np.float32)
    n, ndim = P32.shape
    assert ndim <= 16
    centre = centre_of(P32)
    x = np.zeros((n, 16), np.float32)
    x[:, :ndim] = P32 - centre
    xp = x.copy()
    if pad_from_centre and ndim < 16:
        xp[:, ndim] = centre[0]
    return x, xp, centre


def _split_norm(x):
    hi = tf32_rna(x)
    lo = tf32_trunc(x - hi)
    h = (0.5 * (x.astype(np.float64) ** 2).sum(1)).astype(np.float32)
    h_hi = tf32_rna(h)
    h_lo = tf32_trunc(h - h_hi)
    return hi.astype(np.float64), lo.astype(np.float64), h_hi, h_hi.astype(np.float64) + h_lo.astype(np.float64)


def distances(xr, xp):
    """GEMM 1 for rows xr against partners xp: (S [rows][partners] FP32, h_hi of the rows)."""
    hi_r, lo_r, hh_r, h2_r = _split_norm(xr)
    hi_p, lo_p, _, h2_p = _split_norm(xp)
    dot = hi_r @ hi_p.T + hi_r @ lo_p.T + lo_r @ hi_p.T
    return (h2_r[:, None] + h2_p[None, :] - dot).astype(np.float32), hh_r


def near_mask(S, h_hi_rows, series):
    thr = NEAR_TAU * h_hi_rows
    if series:
        thr = np.maximum(thr, SERIES_NEAR_S)
    return S < thr[:, None]


def weights(S, series, eps=0.01):
    """The weight of every pair from S, truncated to TF32, in FP64.  eps=0 (a mutant) drops the + 0.01."""
    Sa = np.abs(S.astype(np.float64))
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        if series:
            q = (1.0 / np.sqrt(Sa)).astype(np.float32)
            if eps:
                pl = SERIES[0] * q + SERIES[1]
                pl = pl * q + SERIES[2]
                pl = pl * q + SERIES[3]
            else:
                pl = np.float32(2.0 ** -1.5)
            w = (q * q * q * pl).astype(np.float32)
        else:
            rc = (1.0 / (np.sqrt(Sa).astype(np.float32) * np.float32(1.41421356) + np.float32(eps))).astype(np.float32)
            w = (rc * rc * rc).astype(np.float32)
    return tf32_trunc(w).astype(np.float64)


def tensor_pass(P, rows=None, *, series=True, drop=(), fix=True, eps=0.01, pad_from_centre=False, block=512):
    """sum_j w_ij (P_j - P_i) for the rows `rows` (indices into P, default all) as repulse_tc2_kernel computes it.
    Mutants: drop = partners left out of every row's sums (a partner lost at a stage edge); fix=False: the near pairs are
    not re-done; eps=0: the weight without its + 0.01; pad_from_centre: see `image`."""
    P32 = np.asarray(P, np.float32)
    n, ndim = P32.shape
    rows = np.arange(n) if rows is None else np.asarray(rows)
    x, xp, _ = image(P32, pad_from_centre)
    y = tf32_rna(xp).astype(np.float64)
    keep = np.ones(n, bool)
    keep[list(drop)] = False
    X64 = P32.astype(np.float64)
    out = np.zeros((len(rows), ndim))
    for b in range(0, len(rows), block):
        r = rows[b:b + block]
        xi = x[r].astype(np.float64)
        for c0 in range(0, n, CHUNK):
            cols = np.arange(c0, min(n, c0 + CHUNK))
            S, hh = distances(x[r], xp[cols])
            near = near_mask(S, hh, series)
            w = weights(S, series, eps)
            w[near | ~keep[cols][None, :]] = 0.0
            d2 = (w @ y[cols]).astype(np.float32).astype(np.float64)
            wsum = w.sum(1).astype(np.float32).astype(np.float64)
            part = (d2 - xi * wsum[:, None])[:, :ndim]
            if fix:
                rr, jj = np.nonzero(near & keep[cols][None, :])
                diff = X64[cols[jj]] - X64[r[rr]]
                dist = np.sqrt((diff ** 2).sum(1))
                rr, diff, dist = rr[dist > 0], diff[dist > 0], dist[dist > 0]   # the point itself and exact duplicates
                np.add.at(part, rr, diff * ((dist + eps) ** -3)[:, None])
            out[b:b + len(r)] += part
    return out
