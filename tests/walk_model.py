"""The spring walk and the edge MAE of one row-block iteration (topolow_b200/csrc/rowblock.cu: count_kernel, fill_kernel,
sell_kernel, spring_kernel, mae_kernel) restated in numpy - test infrastructure.  Nothing under topolow_b200/ imports it.

  build_records   the SELL-32 layout sell_kernel leaves for the own rows [row0, row0 + rows): a row's records sorted by
                  (partner slot, type code, FP32 target bits), slices of 32 rows padded to the longest row of the slice,
                  and the MAE subset that counts_here picks (every pair counted by exactly one endpoint)
  walk            x = P_i, then every record of the row from the slice's rotated start offset, cyclically, padding
                  skipped: spring iff exact, or '>' and dist < target, or '<' and dist > target; a spring moves
                  x -= (P_j - x) g_i (target - dist) / (dist + 0.01), g_i = 2 k / (4 (deg_i + 1) + k), and takes back the
                  repulsion step 1 gave the pair, x += (P_j - P_i) c / (2 (|P_j - P_i| + 0.01)^3) / (deg_i + 1)
                  (oracle/relaxed_oracle.cpp step 2).  FP64, or (fp32=True) the kernel's FP32 operations in its order with
                  correctly rounded square roots and reciprocals where the kernel takes sqrt.approx / rcp.approx
  mae_terms       FP64 sum |target - dist| and count over the counted pairs that are exact or violated, on given positions

Positions are in slot order (the row-block relabelling, topolow_b200.rowblock.slot_order).  Targets are rounded to FP32
before use, as fill_kernel stores them: the restatement then differs from the kernel only by the kernel's arithmetic.
The keyword `mutant` of build_records and walk selects a subtly wrong walk (MUTANTS); the tests use them to show that
their bars catch one."""
import numpy as np

SORT_CAP = 2048          # sell_kernel: longer rows are sorted by counting ranks in global memory
MUTANTS = ("start_plus_one", "no_rotation", "descending", "drop_last", "swap_gt_lt", "no_takeback", "takeback_from_x",
           "deg_for_dp1", "scatter_order")
_M1, _M2 = np.uint64(0xbf58476d1ce4e5b9), np.uint64(0x94d049bb133111eb)


def mix64(x):
    """splitmix64's finaliser (common.cuh::mix64) on numpy uint64, wrapping."""
    x = np.asarray(x, np.uint64)
    with np.errstate(over="ignore"):
        x = x ^ (x >> np.uint64(30))
        x = x * _M1
        x = x ^ (x >> np.uint64(27))
        x = x * _M2
        x = x ^ (x >> np.uint64(31))
    return x


def start_offsets(seed, it, slots, widths):
    """mix64(seed ^ mix64(iter << 32 | slot >> 5)) % width per slice (slots: the first slot of each slice)."""
    w = np.asarray(widths, np.uint64)
    key = (np.uint64(it) << np.uint64(32)) | (np.asarray(slots, np.uint64) >> np.uint64(5))
    h = mix64(np.uint64(seed) ^ mix64(key))
    return np.where(w > 0, h % np.maximum(w, np.uint64(1)), np.uint64(0)).astype(np.int64)


def counts_here(self_slot, other):
    s, o = np.asarray(self_slot, np.int64), np.asarray(other, np.int64)
    return (((s + o) & 1) != 0) == (s < o)


def type_code(t):
    """fill_kernel's reading of a threshold code: 0 exact, 1 '>', 2 '<' (validate() admits only -1, 0, 1)."""
    t = np.asarray(t)
    return np.where(t == 0, 0, np.where(t == 1, 1, 2)).astype(np.int64)


class Recs:
    pass


def _sell(row, part, typ, tgt, eidx, rows):
    """SELL-32 arrays from records already in row order: (part, typ, tgt, eidx) flat, padding typ 3 / eidx -1."""
    ln = np.bincount(row, minlength=rows).astype(np.int64)
    width = ln.reshape(-1, 32).max(1)
    soff = np.concatenate([[0], np.cumsum(width * 32)])
    first = np.concatenate([[0], np.cumsum(ln)])
    rank = np.arange(len(row)) - first[row]
    pos = soff[row // 32] + rank * 32 + (row & 31)
    total = int(soff[-1])
    out_part = np.zeros(total, np.int64)
    out_typ = np.full(total, 3, np.int64)
    out_tgt = np.zeros(total, np.float32)
    out_e = np.full(total, -1, np.int64)
    out_part[pos], out_typ[pos], out_tgt[pos], out_e[pos] = part, typ, tgt, eidx
    return ln, width, soff[:-1], out_part, out_typ, out_tgt, out_e, total


def build_records(n, edges, slot_of_point, row0, rows, mutant=None):
    """edges = (edge_i, edge_j, edge_dist, edge_thresh) in point numbering; the own rows are slots [row0, row0 + rows)
    (rows a multiple of 32).  Returns Recs with, per own row (local index), `len` and, per slice, `width` / `soff`, the
    flat SELL arrays part / typ / tgt / eidx (record k of local row r at soff[r // 32] + 32 k + r % 32), the same for
    the MAE subset (prefix m), and spring_records / mae_records: the SELL totals topolow_shard_info reports.
    mutant 'descending': partners in descending order; 'scatter_order': rows over SORT_CAP records keep edge order."""
    ei, ej, ed, et = (np.asarray(a) for a in edges)
    slot = np.asarray(slot_of_point, np.int64)
    sa, sb = slot[ei], slot[ej]
    e = np.arange(len(ei), dtype=np.int64)
    row = np.concatenate([sa, sb]) - row0
    part = np.concatenate([sb, sa])
    typ = np.concatenate([type_code(et)] * 2)
    tgt = np.concatenate([np.asarray(ed, np.float64).astype(np.float32)] * 2)
    eidx = np.concatenate([e, e])
    own = (row >= 0) & (row < rows)
    row, part, typ, tgt, eidx = row[own], part[own], typ[own], tgt[own], eidx[own]
    key = (part.astype(np.uint64) << np.uint64(34)) | (typ.astype(np.uint64) << np.uint64(32)) | tgt.view(np.uint32).astype(np.uint64)
    if mutant == "descending":
        key = np.uint64(0xffffffffffffffff) - key
    if mutant == "scatter_order":
        ln = np.bincount(row, minlength=rows)
        key = np.where(ln[row] > SORT_CAP, eidx.astype(np.uint64), key)
    o = np.lexsort((eidx, key, row))     # eidx: equal keys are equal records, any order
    row, part, typ, tgt, eidx = row[o], part[o], typ[o], tgt[o], eidx[o]
    r = Recs()
    r.n, r.row0, r.rows = n, row0, rows
    r.len, r.width, r.soff, r.part, r.typ, r.tgt, r.eidx, r.spring_records = _sell(row, part, typ, tgt, eidx, rows)
    m = counts_here(row + row0, part)
    (r.mlen, r.mwidth, r.msoff, r.mpart, r.mtyp, r.mtgt, r.meidx, r.mae_records) = _sell(row[m], part[m], typ[m], tgt[m],
                                                                                          eidx[m], rows)
    return r


def _dist2_f32(dl):
    """dist2<H> of rowblock.cu: packed pairs (2k, 2k + 1), two FMA chains (even / odd pairs), joined, then x + y."""
    f = np.float32
    H = dl.shape[1] // 2
    p = dl.reshape(len(dl), H, 2)

    def fma(a, b, c):
        return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(f)

    s0 = p[:, 0] * p[:, 0]
    if H > 1:
        s1 = p[:, 1] * p[:, 1]
        for k in range(2, H):
            if k & 1:
                s1 = fma(p[:, k], p[:, k], s1)
            else:
                s0 = fma(p[:, k], p[:, k], s0)
        s0 = s0 + s1
    return s0[:, 0] + s0[:, 1]


def row_width(ndim):
    """Coordinates a row is computed on: 2 H (rowblock.cu::row_h), the pad coordinates zero."""
    return 2 * ((ndim + 1) // 2 if ndim <= 16 else (ndim + 3) // 4 * 2)


def walk(P, dp1, recs, k, c, seed, iter=0, fp32=False, mutant=None):
    """One spring walk of every own row of `recs`.  P: slot-ordered positions (slots >= n zero), dp1: degree + 1 per slot
    (0 = padding).  Returns dict x (rows x ndim, the position after the walk), B (bar scale), margin (smallest
    |dist - target| / target of a threshold record visited; inf if none), visits (records visited per row), and
    low (the edge indices of threshold records visited with margin < 1e-3)."""
    rows, row0 = recs.rows, recs.row0
    nd = P.shape[1]
    D = row_width(nd) if fp32 else nd
    F = np.float32 if fp32 else np.float64
    Pw = np.zeros((len(P), D), F)
    Pw[:, :nd] = P
    slots = row0 + np.arange(rows)
    dp = np.asarray(dp1, np.float64)[slots]
    dpe = dp - 1.0 if mutant == "deg_for_dp1" else dp
    safe = np.where(dpe > 0, dpe, 1.0)
    if fp32:
        kf = F(k)
        g = (F(2.0) * kf / (F(4.0) * safe.astype(F) + kf)).astype(F)
        rdeg = (F(0.5 * c) / safe.astype(F)).astype(F)
    else:
        g = 2.0 * k / (4.0 * safe + k)
        rdeg = 0.5 * c / safe
    width = recs.width
    start = start_offsets(seed, iter, row0 + 32 * np.arange(len(width)), width)
    if mutant == "start_plus_one":
        start = np.where(width > 0, (start + 1) % np.maximum(width, 1), 0)
    if mutant == "no_rotation":
        start[:] = 0
    # slices by width, longest first: the rows still walking at step t are a prefix
    order = np.argsort(-width, kind="stable")
    lrow = (order[:, None] * 32 + np.arange(32)[None, :]).ravel()
    wr, st, so = np.repeat(width[order], 32), np.repeat(start[order], 32), np.repeat(recs.soff[order], 32)
    lane = lrow & 31
    x = Pw[row0 + lrow].copy()
    p0 = Pw[row0 + lrow]
    B = np.zeros(len(lrow))
    margin = np.full(len(lrow), np.inf)
    visits = np.zeros(len(lrow), np.int64)
    low = []
    gl, rl = g[lrow], rdeg[lrow]
    steps = int(width.max()) if len(width) else 0
    for t in range(steps):
        a = int(np.searchsorted(-wr, -t, side="left"))   # rows with width > t: wr[:a]
        if a == 0:
            break
        at = (st[:a] + t) % wr[:a]
        idx = so[:a] + at * 32 + lane[:a]
        typ = recs.typ[idx]
        live = typ != 3
        if mutant == "drop_last":
            live &= at != wr[:a] - 1
        if not live.any():
            continue
        sel = np.nonzero(live)[0]
        q = Pw[recs.part[idx[sel]]]
        tg = recs.tgt[idx[sel]].astype(F)
        ty = typ[sel]
        xs = x[sel]
        dl = q - xs
        d0 = q - (xs if mutant == "takeback_from_x" else p0[sel])
        if fp32:
            dist = np.sqrt(_dist2_f32(dl))
            ds0 = np.sqrt(_dist2_f32(d0)) + F(0.01)
        else:
            dist = np.sqrt((dl * dl).sum(1))
            ds0 = np.sqrt((d0 * d0).sum(1)) + 0.01
        gt, lt = (2, 1) if mutant == "swap_gt_lt" else (1, 2)
        spring = (ty == 0) | ((ty == gt) & (dist < tg)) | ((ty == lt) & (dist > tg))
        thr = ty != 0
        mg = np.abs(dist.astype(np.float64) - tg) / tg
        margin[sel] = np.minimum(margin[sel], np.where(thr, mg, np.inf))
        bad = thr & (mg < 1e-3)
        if bad.any():
            low.append(recs.eidx[idx[sel[bad]]])
        if fp32:
            w0 = np.where(spring, rl[sel] * (F(1.0) / (ds0 * ds0 * ds0)), F(0.0)).astype(F)
            f = np.where(spring, gl[sel] * (tg - dist) * (F(1.0) / (dist + F(0.01))), F(0.0)).astype(F)
            if mutant == "no_takeback":
                w0[:] = 0
            # (-x) = fma(dl, f, fma(d0, -w0, -x)): every operation rounded once
            inner = (d0.astype(np.float64) * (-w0.astype(np.float64))[:, None] - xs.astype(np.float64)).astype(F)
            xn = (dl.astype(np.float64) * f.astype(np.float64)[:, None] + inner.astype(np.float64)).astype(F)
            xnew = -xn
        else:
            w0 = np.where(spring, rl[sel] / ds0 ** 3, 0.0)
            f = np.where(spring, gl[sel] * (tg - dist) / (dist + 0.01), 0.0)
            if mutant == "no_takeback":
                w0[:] = 0
            xnew = xs - dl * f[:, None] + d0 * w0[:, None]
        x[sel] = xnew
        nrm = np.linalg.norm
        B[sel] += (np.abs(f) * nrm(dl.astype(np.float64), axis=1) + np.abs(w0) * nrm(d0.astype(np.float64), axis=1)
                   + gl[sel] * dist + nrm(xnew.astype(np.float64), axis=1) / 16)
        visits[sel] += 1
    inv = np.empty_like(lrow)
    inv[lrow] = np.arange(len(lrow))
    return dict(x=x[inv][:, :nd].astype(np.float64), B=B[inv], margin=margin[inv], visits=visits[inv],
                low=np.unique(np.concatenate(low)) if low else np.zeros(0, np.int64))


def mae_terms(P1, recs):
    """FP64 over the counted records of the own rows on slot-ordered positions P1: (sum |target - dist| over the pairs
    that are exact or violated, their count, sum of target + dist over them, smallest threshold margin on P1)."""
    live = recs.mtyp != 3
    if not live.any():
        return 0.0, 0, 0.0, np.inf
    pos = np.nonzero(live)[0]
    # local row of a flat SELL position: slice from the offsets, lane from the position
    slice_of = np.searchsorted(recs.msoff, pos, side="right") - 1
    lrow = slice_of * 32 + ((pos - recs.msoff[slice_of]) & 31)
    self_slot = recs.row0 + lrow
    d = np.linalg.norm(P1[recs.mpart[pos]] - P1[self_slot], axis=1)
    tg = recs.mtgt[pos].astype(np.float64)
    ty = recs.mtyp[pos]
    on = (ty == 0) | ((ty == 1) & (d < tg)) | ((ty == 2) & (d > tg))
    thr = ty != 0
    mg = np.abs(d - tg) / tg
    return (float(np.abs(tg - d)[on].sum()), int(on.sum()), float((tg + d)[on].sum()),
            float(mg[thr].min()) if thr.any() else np.inf)
