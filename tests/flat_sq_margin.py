"""The fp16 filter's bound restated in NumPy with the kernel's constants (csrc/flat.cu margin_c1_f16, margin_c1ip_f16,
margin_csub_f16; csrc/flat_fp16.cu query prep) -- TEST INFRASTRUCTURE ONLY.

The dot product is formed from the fp16 codes of the row and of the scaled query, accumulated in f32 in row order (one
of the orders the margin allows), optionally with every fp16 subnormal flushed to zero, as a tensor core that flushes
them would; every other step is the epilogue's f32 arithmetic."""
import numpy as np

F32 = np.float32
U = 2.0 ** -11


def _up(c: float) -> np.float32:
    return np.nextafter(F32(c), F32(np.inf))


def constants(d: int, metric: str):
    """(c1, csub) of the fp16 filter for `metric` ("l2" or "ip") at K = d."""
    a = U + np.sqrt(d) * 2.0 ** -28
    acc = d * 2.0 ** -22 * (1 + 2.0 ** -10)
    h = 1 + 2.0 ** -10
    if metric == "l2":
        return _up(2 * (a + acc) * h), _up(2 * h * h)
    return _up((a + acc + (d + 5) * 2.0 ** -53 + 2.0 ** -22) * h), _up(h * h)


def query_scale(q: np.ndarray) -> int:
    """e_q: max |q_j| 2^e_q in [2^14, 2^15), at most 126; 0 for an all-zero or non-finite query."""
    amax = float(np.max(np.abs(q))) if q.size else 0.0
    if not np.all(np.isfinite(q)) or amax == 0.0:
        return 0
    return min(15 - int(np.frexp(np.float32(amax))[1]), 126)


def _fma(a, b, c):
    return F32(np.float64(a) * np.float64(b) + np.float64(c))


def bound(q: np.ndarray, x: np.ndarray, metric: str, c1_scale=1.0, csub_scale=1.0, flush=False) -> np.float32:
    """The filter's lower bound of the exact distance (L2) or upper bound of the exact score (IP) for f32 query q
    and fp16-exact row x (f32 array of fp16 values)."""
    q, x = q.astype(F32), x.astype(F32)
    d = q.shape[0]
    c1, csub = constants(d, metric)
    c1, csub = F32(c1 * c1_scale), F32(csub * csub_scale)
    c2 = F32(2.0 ** -17) if metric == "l2" else F32(0)
    c3 = F32(2.0 ** -100)
    e = query_scale(q)
    qh = np.ldexp(q.astype(np.float64), e).astype(np.float16).astype(F32)
    xh = x.astype(np.float16).astype(F32)
    if flush:
        qh[np.abs(qh) < 2.0 ** -14] = 0
        xh[np.abs(xh) < 2.0 ** -14] = 0
    acc = np.add.accumulate((qh * xh).astype(F32), dtype=F32)[-1]
    dot = F32(acc * F32(np.ldexp(1.0, -e)))
    q64, x64 = q.astype(np.float64), x.astype(np.float64)
    qn2, xn2 = F32(q64 @ q64), F32(x64 @ x64)
    qn, xn = F32(np.sqrt(q64 @ q64)), F32(np.sqrt(x64 @ x64))
    sub = x64[np.abs(x64) < 2.0 ** -14]
    nsub = _up(np.sqrt(sub @ sub * (1 + 2.0 ** -40))) if sub.size and np.any(sub) else F32(0)
    tail = F32(c3 * F32(F32(F32(1) + qn) + xn))
    if metric == "l2":
        s2 = F32(qn2 + xn2)
        margin = _fma(F32(c1 * qn), xn, _fma(F32(csub * qn), nsub, _fma(c2, s2, tail)))
        return F32(_fma(F32(-2), dot, s2) - margin)
    return F32(dot + _fma(F32(c1 * qn), xn, _fma(F32(csub * qn), nsub, tail)))
