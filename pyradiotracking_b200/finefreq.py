"""Carrier estimates finer than one FFT bin (include/rt_engine.h, `rt_engine_set_neighbours`).

A `Signal.frequency` is the centre of the bin the pulse was found in.  For a stationary tone the powers of the two neighbouring
bins fix where inside the bin the carrier lies: the spectrogram's response to a complex exponential at bin position f (cycles
per n samples, n = nperseg) is, in bin b,

    g_b(f) = |sum_m w[m] (exp(2 pi i f m / n) - D(f)) exp(-2 pi i b m / n)|^2,    D(f) = (1/n) sum_m exp(2 pi i f m / n),

scipy's own arithmetic including `detrend='constant'`.  For a record in signed bin k the engine returns the means of bins k - 1
and k + 1 over the record's cells and their row means; the noise-corrected powers P+- = mean - row_mean give the fine position
as the root f in (k - 1, k + 1) of

    log(g_{k+1}(f) / g_{k-1}(f)) = log(P+ / P-).

With A(x) = sum_m w[m] exp(2 pi i x m / n) and F = fft(w), g_{k+-1}(k + d) = |A(d -+ 1) - D(k + d) F[k +- 1]|^2: A and its
derivatives are tabulated once per analyzer on a dense grid (direct float64 sums), D has a closed form, and a safeguarded
Newton iteration on the exact expression (A from its Taylor series about the nearest table point, accurate to rounding)
polishes the table's bracket to the root.  The centre bin's own power is not used, so a record in a bin next to the peak is refined too.

No estimate (NaN) where
  * P+ <= 0 or P- <= 0 (the neighbours do not stand above the noise);
  * the three bins k - 1, k, k + 1 cross +-fs/2 (k = -n/2 or k = n/2 - 1);
  * the log ratio is not strictly increasing over (k - 1, k + 1) (`nan_bins`): next to DC the detrend term bends it.  For the
    windows this module accepts it is the DC bin and its neighbours, k in {-1, 0, 1}, plus k = +-2 for hamming at nperseg 256
    and 4096 (not at 16), and {+-2, +-4, +-6} for bartlett at 256 and 4096; `nan_bins` gives the set of an analyzer;
  * log(P+ / P-) lies outside the range the window can produce over the bin (the measurement is no tone of this model).

The window's plain response |A(x)|^2 must be strictly decreasing on [0, 2) bins, otherwise the ratio is not invertible:
`FineFrequency` raises ValueError.  hamming, hann, blackman, blackmanharris, bartlett and kaiser(8) qualify; boxcar, flattop,
triang, kaiser(4) and tukey(0.5) do not.
"""
import numpy as np

_GRID = 256              # table points per bin
_CHUNK = 1 << 21         # complex terms per direct-sum block
_TERMS = 8               # Taylor terms of A about a table point


def _dtft(w: np.ndarray, x: np.ndarray) -> np.ndarray:
    """sum_m w[m] exp(2 pi i x m / n) for real x (rows) and the columns of w [n, ...], by direct summation in float64."""
    n = len(w)
    m = np.arange(n)
    out = np.empty((len(x),) + w.shape[1:], dtype=np.complex128)
    step = max(1, _CHUNK // n)
    for i in range(0, len(x), step):
        out[i:i + step] = np.exp(2j * np.pi * np.outer(x[i:i + step], m) / n) @ w
    return out


def _dc(k: np.ndarray, d: np.ndarray, n: int):
    """D(k + d) of the module docstring and its derivative in d, closed form: (exp(2 pi i d) - 1) / (n (exp(2 pi i y / n) - 1))
    with y = k + d; D = 1 at y = 0."""
    y = k + d
    num = 2j * np.sin(np.pi * d) * np.exp(1j * np.pi * d)              # exp(2 pi i d) - 1
    den = 2j * n * np.sin(np.pi * y / n) * np.exp(1j * np.pi * y / n)   # n (exp(2 pi i y / n) - 1)
    zero = y == 0
    den = np.where(zero, 1.0, den)
    dnum = 2j * np.pi * np.exp(2j * np.pi * d)
    dden = 2j * np.pi * np.exp(2j * np.pi * y / n)
    D = np.where(zero, 1.0, num / den)
    dD = np.where(zero, 1j * np.pi * (n - 1) / n, (dnum * den - num * dden) / den ** 2)
    return D, dD


class FineFrequency:
    """The estimator of one analyzer: `window` (nperseg values, as scipy's get_window returns them)."""

    def __init__(self, window):
        w = np.asarray(window, dtype=np.float64)
        if w.ndim != 1 or len(w) < 8:
            raise ValueError("window: one value per sample of an FFT segment")
        self.window, self.n = w, len(w)
        n, G = self.n, _GRID
        # A on x = -2 ... 2 in steps of 1 / G: A(d - 1) and A(d + 1) of every table point d = -1 ... 1
        self._x = np.arange(-2 * G, 2 * G + 1) / G
        m = np.arange(n)
        # d^j A / dx^j at the table points, j = 0 ... _TERMS: a Taylor series about the nearest point evaluates A and dA/dx
        # anywhere in [-2, 2] (|x - point| <= 1 / (2 G): the terms fall as (pi / G)^j / j!, below 1e-16 of sum|w| at j = 8)
        self._T = _dtft(w[:, None] * (2j * np.pi * m[:, None] / n) ** np.arange(_TERMS + 1)[None, :], self._x).T
        self._A = self._T[0]
        p = np.abs(self._A[2 * G: 4 * G]) ** 2                  # plain response on [0, 2)
        if not np.all(np.diff(p) < 0):
            raise ValueError("fine_frequency needs a window whose power response falls strictly over its first two bins "
                             "(hamming, hann, blackman, blackmanharris, bartlett, kaiser with beta >= 8); this one does not")
        self._F = np.fft.fft(w)
        self._d = self._x[G: 3 * G + 1]                          # table points d = -1 ... 1
        ks = np.arange(-n // 2 + 1, n // 2 - 1)                  # bins whose neighbours stay inside +-fs/2
        self._r = np.concatenate([self._table(ks[i:i + 256]) for i in range(0, len(ks), 256)])     # row k + n/2 - 1
        bad = ~(np.all(np.isfinite(self._r[:, 1:-1]), axis=1) & np.all(np.diff(self._r, axis=1) > 0, axis=1))
        # the DC bin and its neighbours always: their brackets reach f = 0, where the tone is the segment mean, which the detrend
        # removes from every bin (g = 0 / 0 there)
        self.nan_bins = np.union1d(ks[bad], [-1, 0, 1])

    def _table(self, k) -> np.ndarray:
        """log(g_{k+1} / g_{k-1}) at the table points d = -1 ... 1, [len(k), 2 G + 1] for the signed bins k (the ends may be
        -inf / +inf)."""
        G, n = _GRID, self.n
        k = np.asarray(k, dtype=np.int64).reshape(-1, 1)
        D, _ = _dc(k, self._d[None, :], n)
        hi = self._A[None, 0: 2 * G + 1] - D * self._F[(k + 1) % n]        # A(d - 1)
        lo = self._A[None, 2 * G: 4 * G + 1] - D * self._F[(k - 1) % n]    # A(d + 1)
        with np.errstate(divide="ignore", invalid="ignore"):
            return np.log(np.abs(hi) ** 2) - np.log(np.abs(lo) ** 2)

    def _dtft_at(self, x: np.ndarray):
        """A(x) and dA/dx for x in [-2, 2], from the Taylor tables."""
        G = _GRID
        i = np.clip(np.rint((x + 2) * G).astype(np.int64), 0, 4 * G)
        eps = x - self._x[i]
        pw = np.cumprod(np.concatenate([np.ones((len(x), 1)), eps[:, None] / np.arange(1, _TERMS + 1)[None, :]], axis=1), axis=1)
        T = self._T[:, i]                                          # [_TERMS + 1, len(x)]
        return np.sum(T[:_TERMS] * pw[:, :_TERMS].T, axis=0), np.sum(T[1:] * pw[:, :_TERMS].T, axis=0)

    def _ratio(self, k: np.ndarray, d: np.ndarray):
        """The exact log ratio and its derivative at bin positions k + d."""
        n = self.n
        a_hi, da_hi = self._dtft_at(d - 1)
        a_lo, da_lo = self._dtft_at(d + 1)
        D, dD = _dc(k, d, n)
        f_hi, f_lo = self._F[(k + 1) % n], self._F[(k - 1) % n]
        u_hi, u_lo = a_hi - D * f_hi, a_lo - D * f_lo
        du_hi, du_lo = da_hi - dD * f_hi, da_lo - dD * f_lo
        ph, pl = np.abs(u_hi) ** 2, np.abs(u_lo) ** 2
        with np.errstate(divide="ignore", invalid="ignore"):
            r = np.log(ph) - np.log(pl)
            dr = 2 * np.real(du_hi * np.conj(u_hi)) / ph - 2 * np.real(du_lo * np.conj(u_lo)) / pl
        return r, dr

    def offsets(self, fi, p_lo, p_hi) -> np.ndarray:
        """Offset of the carrier from the centre of bin `fi` (FFT order), in bins, float64: the root d in (-1, 1) of the module
        docstring for the noise-corrected neighbour powers `p_lo` (bin fi - 1) and `p_hi` (bin fi + 1); NaN where there is
        no estimate."""
        n, G = self.n, _GRID
        fi = np.asarray(fi, dtype=np.int64)
        k = np.where(fi >= n // 2, fi - n, fi)
        p_lo, p_hi = np.asarray(p_lo, dtype=np.float64), np.asarray(p_hi, dtype=np.float64)
        out = np.full(len(k), np.nan)
        ok = (p_lo > 0) & (p_hi > 0) & (k > -n // 2) & (k < n // 2 - 1) & ~np.isin(k, self.nan_bins)
        idx = np.flatnonzero(ok)
        if len(idx) == 0:
            return out
        rho = np.log(p_hi[idx] / p_lo[idx])
        kk = k[idx]
        r = self._r[kk + n // 2 - 1]                              # [records, 2 G + 1], increasing along each row
        j = np.sum(r < rho[:, None], axis=1)                      # bracket every root by its cell: r[j - 1] < rho <= r[j]
        live = (j > 0) & (j <= 2 * G)                             # outside [r(-1), r(1)]: no root in the bin
        j = np.clip(j, 1, 2 * G)
        a, b = self._d[j - 1], self._d[j]
        rows = np.arange(len(idx))
        ra, rb = r[rows, j - 1], r[rows, j]
        with np.errstate(invalid="ignore"):
            t = np.where(np.isfinite(ra) & np.isfinite(rb), (rho - ra) / (rb - ra), 0.5)
        x = a + np.clip(t, 0.0, 1.0) * (b - a)
        todo = np.flatnonzero(live)
        # safeguarded Newton from the table's linear interpolation (about 1e-6 bin off): two steps reach ~1e-11 bin
        for _ in range(60):
            if len(todo) == 0:
                break
            r, dr = self._ratio(kk[todo], x[todo])
            below = r < rho[todo]
            a[todo] = np.where(below, x[todo], a[todo])
            b[todo] = np.where(below, b[todo], x[todo])
            with np.errstate(divide="ignore", invalid="ignore"):
                xn = x[todo] - (r - rho[todo]) / dr
            inside = np.isfinite(xn) & (xn > a[todo]) & (xn < b[todo])
            xn = np.where(inside, xn, 0.5 * (a[todo] + b[todo]))
            done = np.abs(xn - x[todo]) < 1e-10
            x[todo] = xn
            todo = todo[~done]
        out[idx[live]] = x[live]
        return out


def fine_frequencies(est: FineFrequency, frequency, fi, neighbours, sample_rate: float) -> np.ndarray:
    """`Signal.frequency + d * sample_rate / nperseg` in float64 for records with bins `fi` and their `neighbours`
    (`engine.NEIGHBOURS_DTYPE`, aligned), d from `est.offsets`."""
    nb = neighbours
    p_lo = nb["mean_lo"].astype(np.float64) - nb["row_mean_lo"].astype(np.float64)
    p_hi = nb["mean_hi"].astype(np.float64) - nb["row_mean_hi"].astype(np.float64)
    return np.asarray(frequency, dtype=np.float64) + est.offsets(fi, p_lo, p_hi) * (sample_rate / est.n)


def central_half(fi, n: int) -> np.ndarray:
    """True for the bins (FFT order) of a channel's flat central half, signed k in [-n/4, n/4)."""
    fi = np.asarray(fi, dtype=np.int64)
    k = np.where(fi >= n // 2, fi - n, fi)
    return (k >= -(n // 4)) & (k < n // 4)
