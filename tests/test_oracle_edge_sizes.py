"""Smallest legal grids and strongly non-cubic ones (the reference's own tests sweep odd sizes,
tfluids/test_tfluids.lua): the oracle against the compiled reference, bit for bit, on 3-cell domains (a
single interior cell), thin slabs and long rows, for every advection method and every point-wise operator.
CPU only; the GPU parity tests compare against this oracle."""
import numpy as np
import pytest

import oracle
from fluidnet_b200 import synth

SHAPES = [((3, 3, 3), True), ((4, 3, 5), True), ((33, 3, 3), True), ((3, 17, 4), True),
          ((3, 3, 1), False), ((5, 3, 1), False), ((3, 41, 1), False)]
IDS = ["%dx%dx%d-%s" % (s + ("3d" if d else "2d",)) for s, d in SHAPES]
METHODS = list(oracle.ADVECT_METHODS)


def fields(shape, is3d, seed):
    nx, ny, nz = shape
    rng = np.random.default_rng(seed)
    fl = synth.make_flags(nx, ny, nz, is3d, nb=2, geometry=False)
    U = (rng.standard_normal((2, 3 if is3d else 2, nz, ny, nx)) * 1.5).astype(np.float32)
    s = rng.random(fl.shape).astype(np.float32)
    return fl, U, s


@pytest.mark.parametrize("shape,is3d", SHAPES, ids=IDS)
def test_advection_on_tiny_grids(orc, ref, shape, is3d):
    fl, U, s = fields(shape, is3d, 1)
    orc.setWallBcsForward(U, fl)

    def run(be):
        out = {}
        for method in METHODS:
            for outside in (False, True):
                out["advectScalar/%s/outside=%d" % (method, outside)] = be.advectScalar(0.3, s, U, fl, method,
                                                                                        outside, 0.75)
            out["advectVel/%s" % method] = be.advectVel(0.3, U, fl, method, 0.75)
        return out
    ref.check(orc, run)


@pytest.mark.parametrize("shape,is3d", SHAPES, ids=IDS)
def test_pointwise_on_tiny_grids(orc, ref, shape, is3d):
    fl, U, s = fields(shape, is3d, 2)
    p = (s - np.float32(0.5)).astype(np.float32)

    def run(be):
        out = {}
        for name, fn in (
            ("setWallBcs", lambda u: be.setWallBcsForward(u, fl)),
            ("velocityUpdate", lambda u: be.velocityUpdateForward(u, fl, p)),
            ("addBuoyancy", lambda u: be.addBuoyancy(u, fl, s, [0.2, -0.5, 0.1], 0.1)),
            ("addGravity", lambda u: be.addGravity(u, fl, [0.2, -0.5, 0.1], 0.1)),
            ("vorticityConfinement", lambda u: be.vorticityConfinement(u, fl, 0.4)),
        ):
            a = U.copy()
            fn(a)
            out[name] = a
        out["velocityDivergence"] = be.velocityDivergenceForward(U, fl)
        out["flagsToOccupancy"] = be.flagsToOccupancy(fl)
        for rad in (1, 2):
            out["signedDistanceField/rad=%d" % rad] = be.signedDistanceField(fl, rad, is3d)
            out["rectangularBlur/rad=%d" % rad] = be.rectangularBlur(U, rad, is3d)
        out["velocityDivergenceBackward"] = be.velocityDivergenceBackward(U, fl, p)
        return out
    ref.check(orc, run)
