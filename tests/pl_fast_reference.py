"""numpy restatement of the FAST FORM of a table of csrc/flow_pl.cu -- TEST INFRASTRUCTURE, like tests/pl_reference.py.

In the region of a table the fast form follows the rows of the plain pieces (header word 2: its offset in floats, word 3:
its size): a grid record (lo, inv, NB - 1, offset of the rows as int32 bits), NB bucket records (number of breakpoints in
the buckets before, then the <= 3 breakpoints of the bucket padded with +inf) and the rows of the fast pieces.  The fast
breakpoints are the table's breakpoints plus the builder's split points; NSF_CL rows hold every spline output minus one
line per axis, in log2 units, knot-derivative outputs in log2 units as well."""

import numpy as np

from tests import pl_reference as plr

FAST_T = 32.0  # flow_pl.cu: largest exponent a fast row may produce (log2 units)


def max_envelope_gap(nets, K):
    """Largest distance (log2 units), over the original pieces' finite ends and both spline axes, between the outputs'
    upper envelope and the output maximal at the piece's midpoint (on outer pieces: of extreme slope, then value) --
    the line the builder stores a piece relative to; pieces where it exceeds FAST_T are cut."""
    bp = plr.breakpoints(nets)
    m, lo, hi = plr.piece_points(bp)
    worst = 0.0
    for i, ((A, B),) in enumerate(plr.tables(nets, bp)):
        for ax in (slice(0, K), slice(K, 2 * K)):
            a, b = A[ax], B[ax]
            if np.isfinite(lo[i]) and np.isfinite(hi[i]):
                l = int(np.argmax(a * m[i] + b))
            else:
                sg = -1.0 if not np.isfinite(lo[i]) else 1.0
                l = int(np.lexsort((b, sg * a))[-1])
            for e in (lo[i], hi[i]):
                if np.isfinite(e):
                    worst = max(worst, float(((a - a[l]) * e + (b - b[l])).max()) * np.log2(np.e))
    return worst


def parse(raw, region_off, hdr_row, stride):
    """(grid, records, rows) of the fast form of the table at float offset region_off, or None if it has none."""
    fo, size = int(hdr_row[2]), int(hdr_row[3])
    if fo == 0:
        return None
    blk = raw[region_off + fo:region_off + fo + size]
    lo, inv, nbm1 = blk[0], blk[1], blk[2]
    rows_off = int(blk[3:4].view(np.int32)[0])
    nb = int(nbm1) + 1
    recs = blk[4:4 + 4 * nb].reshape(nb, 4)
    rows = blk[rows_off:].reshape(-1, stride)
    return (np.float32(lo), np.float32(inv), np.float32(nbm1)), recs, rows


def breakpoints(recs):
    """The fast breakpoints (fp32, sorted): every one sits in exactly one bucket record."""
    b = recs[:, 1:].reshape(-1)
    return np.sort(b[np.isfinite(b)])


def bucket_of(c, grid):
    """flow_pl.cu::bucket_of in fp32: clamp((c - lo) * inv, 0, NB - 1) rounded down, NaN to 0."""
    lo, inv, nbm1 = grid
    with np.errstate(invalid="ignore", over="ignore"):
        t = (np.asarray(c, np.float32) - lo) * inv
    t = np.where(np.isnan(t), np.float32(0), t)
    return np.floor(np.minimum(np.maximum(t, np.float32(0)), nbm1)).astype(np.int64)


def lookup(c, grid, recs):
    """Piece of c: the record's count plus its breakpoints below c."""
    c = np.asarray(c, np.float32)
    r = recs[bucket_of(c, grid)]
    start = r[:, 0].copy().view(np.int32).astype(np.int64)
    return start + (c > r[:, 1]) + (c > r[:, 2]) + (c > r[:, 3])
