"""The fused scorer's exactness argument rests on |coarse - s * exact| <= eps with
eps = (ERR_COEF + d_pad * 2.4e-7) * ||u_s|| * max_i ||i_s|| + sqrt(d_pad) * 6.2e-5 * (||u_s|| + max ||i_s||)
(csrc/score_topk_tc.cu, prep_users_kernel): u_s, i_s = rows scaled by powers of two so that their
norms lie in [64, 128), coarse = dot product of the fp16-rounded scaled vectors accumulated in fp32 on
the tensor core, exact = the fp32 fma chain on the unscaled fp32 rows, s = the product of the two
scales.  This test checks the bound on the CPU with an exact (float64) model of both sides: random
vectors at several magnitudes, adversarial vectors whose every component sits at the worst rounding
position, vectors with a huge dynamic range (fp16 subnormals — rounded AND flushed to zero), widths
up to the kernel's limit, and a pessimistic model of the accumulator (truncation after every one of
the d products)."""
import os
import re

import numpy as np
import pytest


def _src():
    return open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "librecommender_b200", "csrc",
                     "score_topk_tc.cu")).read()


def _err_coef():
    return float(re.search(r"ERR_COEF\s*=\s*([0-9.eE+-]+)f", _src()).group(1))


def _pow2_scale(nrm):
    if not (nrm > 0):
        return 1.0
    m, x = np.frexp(np.float32(nrm))
    return float(np.ldexp(1.0, 7 - int(x)))


def _f16(x, flush=False):
    h = np.asarray(x, dtype=np.float32).astype(np.float16)
    if flush:                                   # a tensor core that flushed fp16 subnormals to zero
        h = np.where(np.abs(h.astype(np.float64)) < 2.0 ** -14, np.float16(0), h)
    return h.astype(np.float64)


def _trunc_accumulate(prods):
    """fp32 accumulator that TRUNCATES (toward zero) after every addition: the most pessimistic
    reading of the tensor core's accumulation (it adds several products per step in a wider adder)."""
    acc = np.float64(0.0)
    for p in prods:
        acc = acc + p
        m, e = np.frexp(acc)
        acc = np.ldexp(np.trunc(m * 2.0 ** 24) / 2.0 ** 24, e)
    return acc


def test_constants_in_the_source():
    coef = _err_coef()
    assert coef >= 2.0 ** -10 * (1 + 2.0 ** -12)            # (1 + 2^-11)^2 - 1
    assert "6.2e-5f" in _src() and 6.2e-5 >= 2.0 ** -14      # absolute term covers flushed subnormals
    assert "2.4e-7f" in _src()


@pytest.mark.parametrize("d", [7, 64, 128, 256])
def test_fp16_coarse_score_error_is_below_eps(d):
    coef = _err_coef()
    d_pad = -(-d // 64) * 64
    rng = np.random.default_rng(d)
    cases = []
    for mag in (1.0, 1e-4, 3e3):
        for _ in range(100):
            cases.append((rng.standard_normal(d) * mag, rng.standard_normal(d) / mag))
    # adversarial: every component exactly half-way between two fp16 values (max rounding error),
    # all errors with the same sign
    base = 1.0 + 2.0 ** -11                     # halfway between 1 and 1 + 2^-10 in fp16
    for s in (1.0, 0.37, 11.0):
        cases.append((np.full(d, base * s), np.full(d, base / s)))
        cases.append((np.full(d, base * s) * (-1) ** np.arange(d), np.full(d, base / s) * (-1) ** np.arange(d)))
    # huge dynamic range: one dominant component, the rest far below the fp16 normal range after scaling
    for tiny in (1e-6, 3e-8, 1e-10):
        u = rng.standard_normal(d) * tiny
        i = rng.standard_normal(d) * tiny
        u[0], i[0] = 1.0, -1.0
        cases.append((u, i))
        cases.append((u, rng.standard_normal(d)))
    worst = 0.0
    for u, i in cases:
        u32, i32 = u.astype(np.float32), i.astype(np.float32)
        exact = np.float64(0.0)
        for k in range(d):                        # the kernel's exact-score definition (fp32 fma chain)
            exact = np.float64(np.float32(np.float64(u32[k]) * np.float64(i32[k]) + exact))
        nu = float(np.linalg.norm(u32.astype(np.float64))) * 1.0001
        ni = float(np.linalg.norm(i32.astype(np.float64))) * 1.0001
        su, si = _pow2_scale(nu), _pow2_scale(ni)
        assert 64.0 <= nu * su < 128.0 * 1.0002 and 64.0 <= ni * si < 128.0 * 1.0002
        bound = (coef + d_pad * 2.4e-7) * (nu * su) * (ni * si) + np.sqrt(d_pad) * 6.2e-5 * (nu * su + ni * si)
        for flush in (False, True):
            prods = _f16(u32 * np.float32(su), flush) * _f16(i32 * np.float32(si), flush)
            coarse = _trunc_accumulate(prods)
            err = abs(coarse - exact * su * si)
            worst = max(worst, err / bound)
            assert err <= bound, (d, flush, err, bound)
    assert worst < 1.0
