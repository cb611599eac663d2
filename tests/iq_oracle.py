"""Float64 restatement of the per-block DC and IQ-imbalance correction of the wideband front ends (include/rt_ddc.h,
include/rt_fbank.h) for the tests.  It composes with `ddc_oracle.ddc` and `fbank_oracle.fbank`: they filter the corrected
samples `correct(x, block)[0]`.

TEST INFRASTRUCTURE ONLY: nothing under `pyradiotracking_b200/` imports it.

For each block of `block` normalised samples x (format_oracle.decode_samples):

    m = mean(x)      p = mean(|x - m|^2)      c = mean((x - m)^2)
    w = -c / (p + sqrt(p^2 - |c|^2))  (w = 0 when p = 0)      y = (x - m) + w conj(x - m)
"""
import numpy as np

# the element offset of the integer moments: cu8 sums b - 128 (include/rt_ddc.h), the signed formats their elements
ELEMENT_BIAS = {"cu8": 128, "ci8": 0, "ci16_le": 0}
ELEMENT_DTYPE = {"cu8": np.uint8, "ci8": np.int8, "ci16_le": np.dtype("<i2")}


def coefficients(x: np.ndarray):
    """(m, w) of one block of complex samples, in float64."""
    x = np.asarray(x, np.complex128)
    m = x.mean()
    d = x - m
    p = float(np.mean(d.real ** 2 + d.imag ** 2))
    c = complex(np.mean(d * d))
    if p == 0.0:
        return m, 0j
    return m, -c / (p + np.sqrt(max(p * p - abs(c) ** 2, 0.0)))


def apply(x: np.ndarray, m: complex, w: complex) -> np.ndarray:
    """y = (x - m) + w conj(x - m)."""
    d = np.asarray(x, np.complex128) - m
    return d + w * np.conj(d)


def correct(x: np.ndarray, block: int):
    """-> (y complex128 [len(x)], m [blocks], w [blocks]): every whole block of `block` samples corrected with its own m, w."""
    x = np.asarray(x, np.complex128)
    nb = len(x) // block
    assert nb * block == len(x), "whole blocks only"
    y = np.empty_like(x)
    ms, ws = np.empty(nb, np.complex128), np.empty(nb, np.complex128)
    for b in range(nb):
        blk = x[b * block:(b + 1) * block]
        ms[b], ws[b] = coefficients(blk)
        y[b * block:(b + 1) * block] = apply(blk, ms[b], ws[b])
    return y, ms, ws


def element_sums(raw: np.ndarray, fmt: str, block: int) -> list:
    """The integer moments of every block of interleaved cu8 / ci8 / ci16_le elements, as Python ints:
    [(S_I, S_Q, S_II, S_QQ, S_IQ)] of e = element - ELEMENT_BIAS[fmt] (int64 arithmetic, exact for blocks up to 2^30)."""
    e = np.asarray(raw).view(ELEMENT_DTYPE[fmt]).astype(np.int64) - ELEMENT_BIAS[fmt]
    out = []
    for b in range(len(e) // (2 * block)):
        i, q = e[2 * b * block:2 * (b + 1) * block:2], e[2 * b * block + 1:2 * (b + 1) * block:2]
        out.append(tuple(int(v) for v in (i.sum(), q.sum(), (i * i).sum(), (q * q).sum(), (i * q).sum())))
    return out


def coefficients_from_sums(sums, n: int, scale: float, offset: float):
    """(m, w) as the coefficient kernel forms them from the element sums of one block of n samples, x = e * scale + offset."""
    si, sq, sii, sqq, siq = (float(v) for v in sums)
    mi, mq = si / n, sq / n
    vii, vqq, viq = sii / n - mi * mi, sqq / n - mq * mq, siq / n - mi * mq
    p, c = vii + vqq, complex(vii - vqq, 2.0 * viq)
    w = 0j if p <= 0.0 else -c / (p + np.sqrt(max(p * p - abs(c) ** 2, 0.0)))
    return complex(mi * scale + offset, mq * scale + offset), w
