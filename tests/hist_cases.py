"""Values where a 30-bin histogram over (-hw, hw) can go wrong, and numpy's answer for them.

Monitor histograms promise np.histogram(y, bins=30, range=(-w/2, w/2)). numpy's bin edges are np.linspace's: i * step
and + lo each rounded, the last edge exactly hi. A value on an edge, or an ulp either side of one, lands in a bin that
depends on that rounding; values spread uniformly over the range exercise the first guess of the bin index."""
import numpy as np

BINS = 30
# 2.5 and 0.5, 1, 3, 5: interior edges where a fused i * step + lo is one ulp off linspace's; 1.27, 2.54, 7.5: none
HALF_WIDTHS = (2.5, 0.5, 1.0, 3.0, 5.0, 0.1, 12.7, 1e-3, 1e3, 1.27)


def edges(hw):
    return np.linspace(-hw, hw, BINS + 1)


def _ulps(x, k):
    out = np.asarray(x, np.float64)
    for _ in range(abs(k)):
        out = np.nextafter(out, np.inf if k > 0 else -np.inf)
    return out


def edge_values(hw, n_uniform=20_000, seed=0):
    """Every linspace edge, +-1 and +-2 ulp around each, exactly +-hw and the values just outside, +-0, +-5e-324, NaN,
    +-inf, then n_uniform seeded uniform values over 1.01 x the range."""
    e = edges(hw)
    near = [_ulps(e, k) for k in (-2, -1, 0, 1, 2)]
    special = [hw, -hw, _ulps(hw, 1), _ulps(-hw, -1), 0.0, -0.0, 5e-324, -5e-324, np.nan, np.inf, -np.inf]
    rng = np.random.default_rng(seed)
    uni = rng.uniform(-1.01 * hw, 1.01 * hw, n_uniform)
    return np.concatenate(near + [np.array(special, np.float64), uni])


def on_edge_grid(hw):
    """The edge values only (no NaN / inf, no uniform fill), in range: what a ray grid can carry to a monitor."""
    v = edge_values(hw, n_uniform=0)
    return np.unique(v[np.isfinite(v) & (np.abs(v) <= hw)])


def numpy_hist(x, hw):
    x = np.asarray(x, np.float64)
    return np.histogram(x[np.isfinite(x)], bins=BINS, range=(-hw, hw))[0]


def numpy_bin(x, hw):
    """Per-value bin of np.histogram (its edges compared exactly; hi goes to the last bin), -1 outside or not finite."""
    x = np.asarray(x, np.float64)
    b = np.searchsorted(edges(hw), x, side="right") - 1
    b[x == hw] = BINS - 1
    b[~((x >= -hw) & (x <= hw))] = -1
    return b


def explain(x, got_bins, hw, limit=12):
    """The values whose bin differs from numpy's, for an assertion message."""
    want = numpy_bin(x, hw)
    bad = np.flatnonzero(np.asarray(got_bins) != want)
    return ", ".join(f"y={x[i]!r}: bin {got_bins[i]} (numpy {want[i]})" for i in bad[:limit]) + \
        (f" ... ({bad.size} values)" if bad.size > limit else "")


def explain_hist(x, hist, hw):
    """Bins where `hist` differs from np.histogram of x, with the values on those bins' edges."""
    want = numpy_hist(x, hw)
    bad = np.flatnonzero(np.asarray(hist) != want)
    e = edges(hw)
    parts = []
    for b in bad[:8]:
        lo, hi = e[b], e[b + 1]
        close = x[np.isfinite(x) & ((np.abs(x - lo) <= 4 * np.abs(np.spacing(lo))) | (np.abs(x - hi) <= 4 * np.abs(np.spacing(hi))))]
        parts.append(f"bin {b}: {int(hist[b])} vs numpy {int(want[b])} (edge values {np.unique(close)[:6].tolist()})")
    return f"hw={hw}: " + "; ".join(parts)
