"""The regrouped 1-D butterflies of the CUDA kernels (zj_kernels.cu: idct8 / idct8_lo4 / idct8_lo6) restated in
numpy and compared with the reference's literal operation order (src/idct/scalar.rs:79-166 == src/idct/avx2.rs:251-331) over
Z/2^32: the regrouping (bias folded into one shift-add, odd outputs as chains of two multiply-adds, constants summed up front in
the short forms) must be exact for EVERY 32-bit input, wrap-around included.  CPU only -- the GPU suite proves the same on the
hardware (test_gpu_parity.py::test_warp_uniform_sparsity_classes_at_the_limits)."""
import numpy as np
import pytest

U = np.uint32


def _c(k):
    return U(k & 0xFFFFFFFF)


def literal(s, bias, sh):
    """the reference's order of operations (what oracle/zj_oracle.c transliterates)"""
    s0, s1, s2, s3, s4, s5, s6, s7 = s
    p1 = (s2 + s6) * _c(2217)
    t2 = p1 + s6 * _c(-7567)
    t3 = p1 + s2 * _c(3135)
    t0 = (s0 + s4) << U(12)
    t1 = (s0 - s4) << U(12)
    x0, x3, x1, x2 = t0 + t3 + bias, t0 - t3 + bias, t1 + t2 + bias, t1 - t2 + bias
    a, b, c, d = s7, s5, s3, s1
    p3, p4, q1, q2 = a + c, b + d, a + d, b + c
    p5 = (p3 + p4) * _c(4816)
    a, b, c, d = a * _c(1223), b * _c(8410), c * _c(12586), d * _c(6149)
    q1 = p5 + q1 * _c(-3685)
    q2 = p5 + q2 * _c(-10497)
    p3 = p3 * _c(-8034)
    p4 = p4 * _c(-1597)
    d, c, b, a = d + q1 + p4, c + q2 + p3, b + q2 + p4, a + q1 + p3
    outs = [x0 + d, x1 + c, x2 + b, x3 + a, x3 - a, x2 - b, x1 - c, x0 - d]
    return [(o.astype(np.int32) >> sh).astype(U) for o in outs]


def mad(a, k, c):
    return a * _c(k) + c


def regrouped_full(s, bias, sh):
    s0, s1, s2, s3, s4, s5, s6, s7 = s
    p1 = (s2 + s6) * _c(2217)
    t2, t3 = mad(s6, -7567, p1), mad(s2, 3135, p1)
    v = (s0 << U(12)) + bias
    t0, t1 = mad(s4, 4096, v), mad(s4, -4096, v)
    x0, x3, x1, x2 = t0 + t3, t0 - t3, t1 + t2, t1 - t2
    p3, p4, q1, q2 = s7 + s3, s5 + s1, s7 + s1, s5 + s3
    p5 = (p3 + p4) * _c(4816)
    r1, r2 = mad(q1, -3685, p5), mad(q2, -10497, p5)
    a = mad(s7, 1223, mad(p3, -8034, r1))
    c = mad(s3, 12586, mad(p3, -8034, r2))
    b = mad(s5, 8410, mad(p4, -1597, r2))
    d = mad(s1, 6149, mad(p4, -1597, r1))
    outs = [x0 + d, x1 + c, x2 + b, x3 + a, x3 - a, x2 - b, x1 - c, x0 - d]
    return [(o.astype(np.int32) >> sh).astype(U) for o in outs]


def regrouped_lo4(s, bias, sh):
    s0, s1, s2, s3 = s[:4]
    t0 = (s0 << U(12)) + bias
    x0, x3, x1, x2 = mad(s2, 2217 + 3135, t0), mad(s2, -(2217 + 3135), t0), mad(s2, 2217, t0), mad(s2, -2217, t0)
    c48, d48 = s3 * _c(4816), s1 * _c(4816)
    dd = mad(s1, 6149 - 3685 + 4816 - 1597, c48)
    cc = mad(s3, 12586 - 10497 + 4816 - 8034, d48)
    bb = mad(s3, 4816 - 10497, s1 * _c(4816 - 1597))
    aa = mad(s1, 4816 - 3685, s3 * _c(4816 - 8034))
    outs = [x0 + dd, x1 + cc, x2 + bb, x3 + aa, x3 - aa, x2 - bb, x1 - cc, x0 - dd]
    return [(o.astype(np.int32) >> sh).astype(U) for o in outs]


def regrouped_lo6(s, bias, sh):
    s0, s1, s2, s3, s4, s5 = s[:6]
    v = (s0 << U(12)) + bias
    t0, t1 = mad(s4, 4096, v), mad(s4, -4096, v)
    x0, x3, x1, x2 = mad(s2, 2217 + 3135, t0), mad(s2, -(2217 + 3135), t0), mad(s2, 2217, t1), mad(s2, -2217, t1)
    p4, q2 = s5 + s1, s5 + s3
    p5 = (s3 + p4) * _c(4816)
    r1, r2 = mad(s1, -3685, p5), mad(q2, -10497, p5)
    aa = mad(s3, -8034, r1)
    cc = mad(s3, 12586 - 8034, r2)
    bb = mad(s5, 8410, mad(p4, -1597, r2))
    dd = mad(s1, 6149, mad(p4, -1597, r1))
    outs = [x0 + dd, x1 + cc, x2 + bb, x3 + aa, x3 - aa, x2 - bb, x1 - cc, x0 - dd]
    return [(o.astype(np.int32) >> sh).astype(U) for o in outs]


def _inputs(rng, n, live):
    """n vectors of eight u32: uniform over the full range, small values, and the corners, zero outside the first `live` inputs"""
    full = rng.integers(0, 2**32, size=(8, n), dtype=np.uint64).astype(U)
    small = rng.integers(-40000, 40000, size=(8, n)).astype(np.int64).astype(U)
    corners = rng.choice(np.array([0, 1, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFF, 0x7FFF, 0xFFFF8000], dtype=np.uint64), size=(8, n)).astype(U)
    s = np.concatenate([full, small, corners], axis=1)
    s[live:, :] = 0
    return [s[k] for k in range(8)]


@pytest.mark.parametrize("bias,sh", [(512, 10), (512 + 65536 + (128 << 17), 17)])
def test_regrouped_butterflies_equal_the_literal_form(bias, sh):
    rng = np.random.default_rng(2026)
    b = U(bias)
    with np.errstate(over="ignore"):
        for form, live in ((regrouped_full, 8), (regrouped_lo6, 6), (regrouped_lo4, 4)):
            s = _inputs(rng, 200_000, live)
            want, got = literal(s, b, sh), form(s, b, sh)
            for k in range(8):
                assert np.array_equal(want[k], got[k]), (form.__name__, k)
