"""normalizePressureMean, volumetricUpSamplingNearestForward, rectangularBlur, signedDistanceField:
the oracle's restatements against the reference's own CPU code (oracle/_ref, outputs recorded under tests/golden),
bit for bit; the mean removal to float rounding (the reference accumulates it with an OpenMP atomic, order
unspecified)."""
import numpy as np
import pytest

from oracle import api
from cases import bits_equal
import pcg_cases


@pytest.fixture(scope="module")
def orc():
    return api.Oracle()


def fields(orc, is3d, seed=0):
    flags, _, _ = pcg_cases.make(orc, is3d, nb=2, seed=seed)
    x = np.random.default_rng(seed).standard_normal((2, 3) + flags.shape[2:]).astype(np.float32)
    return flags, x


@pytest.mark.parametrize("is3d", [True, False])
def test_upsampling(orc, ref, is3d):
    _, x = fields(orc, is3d)
    x = np.ascontiguousarray(x[:, :, :5, :6, :7])
    ref.check(orc, lambda be: {"ratio=%d" % ratio: be.volumetricUpSamplingNearestForward(ratio, x)
                               for ratio in (1, 2, 3)})
    for ratio in (1, 2, 3):
        a = orc.volumetricUpSamplingNearestForward(ratio, x)
        assert a.shape[2:] == tuple(s * ratio for s in x.shape[2:])


@pytest.mark.parametrize("is3d", [True, False])
def test_rectangular_blur(orc, ref, is3d):
    _, x = fields(orc, is3d)
    # 40 > every extent: the clamped-edge branches
    ref.check(orc, lambda be: {"rad=%d" % rad: be.rectangularBlur(x, rad, is3d) for rad in (1, 2, 5, 40)})
    const = np.full_like(x, 3.0)
    assert np.allclose(orc.rectangularBlur(const, 3, is3d), 3.0, atol=1e-5)


@pytest.mark.parametrize("is3d", [True, False])
def test_signed_distance_field(orc, ref, is3d):
    flags, _ = fields(orc, is3d)
    ref.check(orc, lambda be: {"rad=%d" % rad: be.signedDistanceField(flags, rad, is3d) for rad in (1, 3)})
    for rad in (1, 3):
        a = orc.signedDistanceField(flags, rad, is3d)
        assert np.all(a[flags == 2] == 0) and a.max() <= rad


@pytest.mark.parametrize("is3d", [True, False])
def test_normalize_pressure_mean(orc, ref, is3d):
    flags, x = fields(orc, is3d)
    flags[0, 0, 0, 3, 3] = 1                 # a fluid cell on the border is legal here
    p0 = np.ascontiguousarray(x[:, :1]).copy()
    ref.check(orc, lambda be: {"p": be.normalizePressureMean(p0.copy(), flags, is3d)}, tol={"p": 2e-6})
    p1 = orc.normalizePressureMean(p0.copy(), flags, is3d)
    assert bits_equal(p1[flags != 1], x[:, :1][flags != 1])          # non-fluid cells untouched
    comp, sizes = orc.findConnectedFluidComponents(flags, is3d, 0)
    for ic in range(len(sizes)):
        assert abs(p1[0, 0][comp == ic].astype(np.float64).mean()) < 1e-5


@pytest.mark.parametrize("is3d", [True, False])
def test_backward_operators(orc, ref, is3d):
    """velocityDivergenceBackward (bit-exact: at most two terms per face), velocityUpdateBackward (the
    reference sums up to nine terms with OpenMP atomics: float-rounding tolerance),
    volumetricUpSamplingNearestBackward (bit-exact)."""
    from fluidnet_b200 import synth
    rng = np.random.default_rng(3)
    nx, ny, nz = (14, 12, 10) if is3d else (22, 18, 1)
    fl = synth.make_flags(nx, ny, nz, is3d, nb=2, geometry=True, exotic=True)
    U = synth.make_velocity(fl, is3d, amp=1.0)
    go = rng.standard_normal(fl.shape).astype(np.float32)
    goU = rng.standard_normal(U.shape).astype(np.float32)
    p = rng.standard_normal(fl.shape).astype(np.float32)
    x = rng.standard_normal((2, 3, 4, 5, 6)).astype(np.float32)
    gs = [rng.standard_normal((2, 3, 4 * ratio, 5 * ratio, 6 * ratio)).astype(np.float32) for ratio in (1, 2, 3)]

    def run(be):
        out = {"velocityDivergenceBackward": be.velocityDivergenceBackward(U, fl, go),
               "velocityUpdateBackward": be.velocityUpdateBackward(U, fl, p, goU)}
        for ratio, g in zip((1, 2, 3), gs):
            out["volumetricUpSamplingNearestBackward/ratio=%d" % ratio] = \
                be.volumetricUpSamplingNearestBackward(ratio, x, g)
        return out
    ref.check(orc, run, tol={"velocityUpdateBackward": 1e-6})


def test_backward_is_the_adjoint(orc):
    """<J v, w> == <v, J^T w> for the two linear forward operators (an independent check of the gathers)."""
    from fluidnet_b200 import synth
    rng = np.random.default_rng(4)
    fl = synth.make_flags(12, 11, 10, True, nb=1, geometry=True, exotic=True)
    U = rng.standard_normal((1, 3, 10, 11, 12)).astype(np.float32)
    w = rng.standard_normal(fl.shape).astype(np.float32)
    lhs = float((orc.velocityDivergenceForward(U, fl).astype(np.float64) * w).sum())
    rhs = float((U.astype(np.float64) * orc.velocityDivergenceBackward(U, fl, w)).sum())
    assert abs(lhs - rhs) <= 1e-4 * max(abs(lhs), 1.0)
    p = rng.standard_normal(fl.shape).astype(np.float32)
    wU = rng.standard_normal(U.shape).astype(np.float32)
    U0 = np.zeros_like(U)
    upd = U0.copy()
    orc.velocityUpdateForward(upd, fl, p)                     # linear in p for U = 0
    lhs = float((upd.astype(np.float64) * wU).sum())
    rhs = float((p.astype(np.float64) * orc.velocityUpdateBackward(U0, fl, p, wU)).sum())
    assert abs(lhs - rhs) <= 1e-4 * max(abs(lhs), 1.0)
