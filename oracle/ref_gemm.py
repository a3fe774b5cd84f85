"""TEST INFRASTRUCTURE ONLY -- float64 restatement of the dense transform ``stag_gemm_tcgen05``
(``out = act(row_scale * (A @ W) + bias)``), its accuracy bound, and numpy emulations of the two 3xTF32 splits the
kernel uses, so that a test can show the bound sees a dropped term.

Bound, per element:  |out - ref| <= 2^-17 (|rs_i| (|A| @ |W|)_ij + |b_j|).  It scales with each row of A, each column
of W and each bias entry on its own, so a wrong row scale, a wrong bias column or a mis-addressed row fails at its own
magnitude even when other rows are 2^60 larger.  relu is 1-Lipschitz: the same bound holds after it.

Splits (A W ~= A_hi W_hi + A_lo W_hi + A_hi W_lo, every part a tf32 value):
  form 1 (gemm_tcgen05_kernel):  hi = tf32 round-to-nearest, ties away (cvt.rna.tf32.f32), lo = rna(x - hi);
  form 2 (gemm_tma_kernel):      A: hi = x truncated to its upper 19 bits (the tensor core reads the raw fp32 tile),
                                 lo = rna(x - hi);  W: as in form 1.
"""
import numpy as np

BOUND = 2.0 ** -17


def tf32_rna(x):
    """float32 -> float32 with the low 13 mantissa bits rounded off, ties away from zero (cvt.rna.tf32.f32)."""
    x = np.ascontiguousarray(x, np.float32)
    u = x.view(np.uint32)
    r = ((u + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)
    return np.where(np.isfinite(x), r, x)


def tf32_trunc(x):
    """float32 -> float32 with the low 13 mantissa bits cleared."""
    x = np.ascontiguousarray(x, np.float32)
    return (x.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)


def split(x, form, operand):
    """-> (hi, lo) float32 of the kernel's split of `x` for operand 'a' or 'w' on form 1 or 2."""
    x = np.asarray(x, np.float32)
    hi = tf32_trunc(x) if (form == 2 and operand == "a") else tf32_rna(x)
    with np.errstate(invalid="ignore"):     # Inf - Inf = NaN, as on the device
        return hi, tf32_rna((x - hi).astype(np.float32))


def reference(a, w, rs=None, b=None, relu=False):
    """float64 act(rs * (a @ w) + b); a [M,K], w [K,N] (W, not transposed)."""
    y = np.asarray(a, np.float64) @ np.asarray(w, np.float64)
    if rs is not None:
        y = y * np.asarray(rs, np.float64)[:, None]
    if b is not None:
        y = y + np.asarray(b, np.float64)[None, :]
    return np.where(y < 0, 0.0, y) if relu else y


def bound(a, w, rs=None, b=None):
    """Per-element tolerance 2^-17 (|rs_i| (|A| @ |W|)_ij + |b_j|)."""
    t = np.abs(np.asarray(a, np.float64)) @ np.abs(np.asarray(w, np.float64))
    if rs is not None:
        t = t * np.abs(np.asarray(rs, np.float64))[:, None]
    if b is not None:
        t = t + np.abs(np.asarray(b, np.float64))[None, :]
    return BOUND * t


def emulate(a, w, form, terms=("hh", "lh", "hl"), rs=None, b=None, relu=False):
    """float64 sum of the chosen split products (hh = A_hi W_hi, lh = A_lo W_hi, hl = A_hi W_lo) with the epilogue.
    terms=("hh",) is a 1xTF32 product; ("hh", "hl") a split that drops A_lo W_hi."""
    ah, al = (p.astype(np.float64) for p in split(a, form, "a"))
    wh, wl = (p.astype(np.float64) for p in split(w, form, "w"))
    pick = {"hh": (ah, wh), "lh": (al, wh), "hl": (ah, wl), "ll": (al, wl)}
    y = sum(pick[t][0] @ pick[t][1] for t in terms)
    if rs is not None:
        y = y * np.asarray(rs, np.float64)[:, None]
    if b is not None:
        y = y + np.asarray(b, np.float64)[None, :]
    return np.where(y < 0, 0.0, y) if relu else y


def violations(out, ref, tol):
    """Number of entries with |out - ref| > tol.  NaN in `out` where `ref` is finite counts as a violation."""
    err = np.abs(np.asarray(out, np.float64) - np.asarray(ref, np.float64))
    return int(np.count_nonzero(~(err <= tol)))


def scaled_inputs(rng, M, K, N, lo=-30, hi=30):
    """a [M,K], w [K,N] float32 standard normals with per-row scales of A and per-column scales of W drawn from the
    powers of two 2^lo .. 2^hi (exact, so the tf32 splits see the same mantissas at every scale), a row scale in
    [0.5, 2) and a bias whose entry j has the magnitude of output column j."""
    ra = 2.0 ** rng.integers(lo, hi + 1, M)
    cw = 2.0 ** rng.integers(lo, hi + 1, N)
    a = (rng.standard_normal((M, K)) * ra[:, None]).astype(np.float32)
    w = (rng.standard_normal((K, N)) * cw[None, :]).astype(np.float32)
    rs = rng.uniform(0.5, 2.0, M).astype(np.float32)
    b = (rng.standard_normal(N) * cw * np.sqrt(K)).astype(np.float32)
    return a, w, rs, b
