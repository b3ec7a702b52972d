"""CPU side of the double-angle pose tests: the near-contact fixture of tests/test_gpu_f64_inputs.py is valid and able to
fail a kernel that narrows its angles to float, and the FP32 rotation the kernels derive from a double angle
(csrc/collide_kernels.cu: sincos_narrow + rotation_f32_sc) stays within its documented bound of FillRotationMatrix of the
ORIGINAL double angle for every finite angle."""
import numpy as np
import pytest

import near_contact as NC
from conftest import CASES, SEED

OFFSETS = (1e-3, 1e-4, 1e-5)
FLOAT_PI = np.float32(3.14159274)
SC_BOUND = 2.0 ** -21    # |sin/cos used by the FP32 stage - exact sin/cos of the double angle|
R_BOUND = 2.0 ** -19     # per entry of the FP32 rotation against the double FillRotationMatrix


@pytest.fixture(scope="module")
def brackets(orc, meshes):
    return {case: NC.case_brackets(orc, meshes, CASES, case, SEED + 40) for case in NC.SETUP}


@pytest.mark.parametrize("case", list(NC.SETUP))
def test_fixture_inside_collides_and_outside_is_free(orc, brackets, case):
    mo, mr, lo, hi, axis, cols = brackets[case]
    assert len(lo) > 400, len(lo)
    for K in (0, 1, 160, 1600):
        for off in OFFSETS:
            inside, outside = NC.near_contact_poses(lo, hi, off, K, 7 + K, axis, cols)
            moved = inside[:, list(cols)]
            assert not np.any(np.float32(moved).astype(np.float64) == moved), "an angle is a float"
            vi, _ = orc.collide_obbtree(mo, mr, inside)
            vo, _ = orc.collide_obbtree(mo, mr, outside)
            assert vi.all(), (case, K, off, np.nonzero(vi == 0)[0][:8])
            assert not vo.any(), (case, K, off, np.nonzero(vo)[0][:8])


@pytest.mark.parametrize("case", ["B", "T"])
def test_fixture_can_fail_a_kernel_that_narrows_angles(orc, brackets, case):
    """judged at the float-narrowed angles, some poses change sides: an FP32 certificate built from the narrowed angle
    without a larger allowance could be issued for the wrong pose, so the GPU test cannot pass vacuously"""
    mo, mr, lo, hi, axis, cols = brackets[case]
    inside, outside = NC.near_contact_poses(lo, hi, 1e-4, 160, 7 + 160, axis, cols)
    ni, _ = orc.collide_obbtree(mo, mr, NC.narrowed(inside))
    no, _ = orc.collide_obbtree(mo, mr, NC.narrowed(outside))
    assert (ni == 0).sum() >= 1 and (no == 1).sum() >= 1, (int((ni == 0).sum()), int((no == 1).sum()))
    # and none at K = 0, where the narrowing is below 2^-23
    inside0, outside0 = NC.near_contact_poses(lo, hi, 1e-4, 0, 7, axis, cols)
    assert orc.collide_obbtree(mo, mr, NC.narrowed(inside0))[0].all()
    assert not orc.collide_obbtree(mo, mr, NC.narrowed(outside0))[0].any()


# ---- the FP32 rotation of a double angle, restated ----------------------------------------------------------------
def _away(v, exact, ulps):
    """the float32 farthest from `exact` within `ulps` ulp (float32 ulp of v) of the double v: the worst case of a
    function with an `ulps`-ulp error bound whose exact result is v"""
    u = np.ldexp(1.0, np.frexp(v)[1] - 24)
    t = v + np.where(v >= exact, 1.0, -1.0) * ulps * u
    f = t.astype(np.float32)
    over = np.abs(f.astype(np.float64) - v) > ulps * u
    return np.where(over, np.nextafter(f, v.astype(np.float32)), f)


def fp32_sincos(a):
    """sin, cos (float32) that sincos_narrow may return for double angles a: |float(a)| <= float(pi) -> sincosf of the
    narrowed angle (any float within 2 ulp of its exact value: sincosf's bound; the one farthest from the exact value of
    the original angle is taken); otherwise sincos of the double angle rounded to float"""
    with np.errstate(over="ignore"):   # |a| > FLT_MAX narrows to inf: out of range, as in the kernel
        af = a.astype(np.float32)
    inr = np.abs(af) <= FLOAT_PI
    a_in = np.where(inr, af.astype(np.float64), 0.0)
    s_in = _away(np.sin(a_in), np.sin(a), 2)
    c_in = _away(np.cos(a_in), np.cos(a), 2)
    s = np.where(inr, s_in, np.sin(a).astype(np.float32))
    c = np.where(inr, c_in, np.cos(a).astype(np.float32))
    return s, c, inr


def rotation_f32_sc(sy, cy, sp, cp, sr, cr):
    """csrc/collide_kernels.cu::rotation_f32_sc in float32 (row-major [n][9])"""
    return np.stack([cy * cp, cy * sp * sr - sy * cr, cy * sp * cr + sy * sr,
                     sy * cp, sy * sp * sr + cy * cr, sy * sp * cr - cy * sr,
                     -sp, cp * sr, cp * cr], 1)


def fill_rotation_f64(y, p, r):
    """Point<T>::FillRotationMatrix in double (oracle/sff_oracle.c::orc_rotation)"""
    cy, sy, cp, sp, cr, sr = np.cos(y), np.sin(y), np.cos(p), np.sin(p), np.cos(r), np.sin(r)
    return np.stack([cy * cp, cy * sp * sr - sy * cr, cy * sp * cr + sy * sr,
                     sy * cp, sy * sp * sr + cy * cr, sy * sp * cr - cy * sr,
                     -sp, cp * sr, cp * cr], 1)


def angle_sweep():
    r = np.random.RandomState(3)
    near_pi = np.concatenate([np.pi + np.arange(-2000, 2001) * 1e-10, np.pi + np.arange(-200, 201) * 2.0 ** -24,
                              [np.float32(np.pi), np.nextafter(np.float64(np.float32(np.pi)), 4.0),
                               np.nextafter(np.float64(np.float32(np.pi)), 0.0), np.nextafter(np.pi, 4.0)]])
    k = np.concatenate([np.arange(-50, 51), r.randint(-160000, 160000, 4000)]).astype(np.float64)
    periodic = (2 * np.pi * k)[:, None] + np.array([-1e-9, -1e-12, 0.0, 1e-12, 1e-9])[None, :]
    wide = np.concatenate([r.uniform(-10, 10, 20000), r.uniform(-1e3, 1e3, 20000), r.uniform(-1e6, 1e6, 20000),
                           10.0 ** r.uniform(6, 15, 5000) * r.choice([-1, 1], 5000)])
    extreme = np.array([1e12, 1e15, 1e18, 3.4e38, 3.5e38, 1e100, 1e300, np.finfo(np.float64).max, 2.0 ** 1000 + 2.0 ** 950,
                        np.finfo(np.float64).tiny, 5e-324, 0.0])
    a = np.concatenate([near_pi, periodic.ravel(), wide, extreme, r.uniform(-np.pi, np.pi, 50000)])
    return np.concatenate([a, -a])


def test_fp32_sin_cos_of_a_double_angle_within_bound_of_the_original_angle():
    a = angle_sweep()
    s, c, inr = fp32_sincos(a)
    assert inr.any() and (~inr).any()
    es = np.abs(s.astype(np.float64) - np.sin(a))
    ec = np.abs(c.astype(np.float64) - np.cos(a))
    worst = int(np.argmax(np.maximum(es, ec)))
    assert max(es.max(), ec.max()) <= SC_BOUND, (a[worst], es[worst], ec[worst])
    # what plain narrowing would do beyond float(pi): far outside the bound (the defect the wide branch removes)
    an = a[(np.abs(a) > 100.0) & (np.abs(a) < 1e30)]
    naive = np.abs(np.sin(an.astype(np.float32).astype(np.float64)) - np.sin(an))
    assert naive.max() > 64 * SC_BOUND


def test_fp32_rotation_of_double_angles_within_bound_of_fill_rotation_matrix():
    a = angle_sweep()
    r = np.random.RandomState(4)
    y, p, ro = a, r.permutation(a), r.permutation(a)
    sy, cy, _ = fp32_sincos(y)
    sp, cp, _ = fp32_sincos(p)
    sr, cr, _ = fp32_sincos(ro)
    R32 = rotation_f32_sc(sy, cy, sp, cp, sr, cr).astype(np.float64)
    R64 = fill_rotation_f64(y, p, ro)
    err = np.abs(R32 - R64).max(1)
    i = int(np.argmax(err))
    assert err[i] <= R_BOUND, (y[i], p[i], ro[i], err[i])
    # the restated double rotation is the oracle's (up to the last bit of libm's sin / cos)
    import oracle
    for j in r.choice(len(a), 200, replace=False):
        np.testing.assert_allclose(oracle.rotation([0, 0, 0, y[j], p[j], ro[j]]).ravel(), R64[j], rtol=0, atol=1e-15)
