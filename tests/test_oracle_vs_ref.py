"""Pins the C restatement (oracle/tfluids_oracle.c) against the reference's own CPU code
compiled in place (oracle/_ref): bit-exact on seeded inputs for every operator and
advection method.  The reference's outputs are recorded under tests/golden (tests/reference_record.py)."""
import numpy as np
import pytest

import oracle
from cases import CASES, CASE_IDS, build

METHODS = list(oracle.ADVECT_METHODS)


@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
@pytest.mark.parametrize("method", METHODS)
def test_advect_scalar(orc, ref, case, method):
    c = build(case)
    U = c["U"].copy()
    orc.setWallBcsForward(U, c["flags"])
    ref.check(orc, lambda be: {"outside=%d" % outside: be.advectScalar(0.1, c["density"], U, c["flags"], method,
                                                                       outside, 0.6)
                               for outside in (False, True)})
    assert orc.trace_faults() == 0


@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
@pytest.mark.parametrize("method", METHODS)
def test_advect_vel(orc, ref, case, method):
    c = build(case)
    U = c["U"].copy()
    orc.setWallBcsForward(U, c["flags"])
    ref.check(orc, lambda be: {"advectVel": be.advectVel(0.1, U, c["flags"], method, 0.6)})


@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_pointwise_operators(orc, ref, case):
    c = build(case)
    fl = c["flags"]
    U = c["U"].copy()
    orc.setWallBcsForward(U, fl)
    g = [0.1, -0.7, 0.3]

    def run(be):
        out = {}
        for mask in (False, True):
            a = c["U"].copy()
            be.setWallBcsForward(a, fl, mask)
            out["setWallBcs/mask=%d" % mask] = a
        out["divergence"] = be.velocityDivergenceForward(U, fl)
        for name, fn in (("velocityUpdate", lambda a: be.velocityUpdateForward(a, fl, c["p"])),
                         ("addBuoyancy", lambda a: be.addBuoyancy(a, fl, c["density"], g, 0.1)),
                         ("addGravity", lambda a: be.addGravity(a, fl, g, 0.1)),
                         ("vorticityConfinement", lambda a: be.vorticityConfinement(a, fl, 0.3))):
            a = U.copy()
            fn(a)
            out[name] = a
        return out
    ref.check(orc, run)


def test_empty_domain_and_occupancy(orc, ref):
    def run(be):
        out = {}
        for is3d, shape in ((True, (2, 1, 7, 9, 11)), (False, (2, 1, 1, 9, 11))):
            for bnd in (1, 2):
                a = np.zeros(shape, np.float32)
                be.emptyDomain(a, is3d, bnd)
                out["emptyDomain/%dd/bnd=%d" % (3 if is3d else 2, bnd)] = a
                out["flagsToOccupancy/%dd/bnd=%d" % (3 if is3d else 2, bnd)] = be.flagsToOccupancy(a)
        return out
    ref.check(orc, run)


def test_line_trace_random(orc, ref):
    rs = np.random.RandomState(5)
    from fluidnet_b200 import synth
    flags = synth.make_flags(20, 18, 16, True, nb=1, geometry=True)
    traces = []
    for _ in range(4000):
        pos = (rs.rand(3) * [18, 16, 14] + 1).astype(np.float32)
        if (int(flags[0, 0, int(pos[2]), int(pos[1]), int(pos[0])]) & 1) == 0:
            continue
        delta = (rs.randn(3) * rs.choice([0.3, 2.0, 9.0])).astype(np.float32)
        traces.append((pos, delta))
    assert len(traces) > 2000

    def run(be):
        res = [be.calcLineTrace(pos, delta, flags) for pos, delta in traces]
        return {"hit": np.array([h for h, _ in res], np.int32), "pos": np.array([p for _, p in res], np.float32)}
    ref.check(orc, run)


TILE_GRIDS = [((40, 24, 20), True, False), ((36, 20, 12), True, True), ((64, 16, 5), False, False)]


@pytest.mark.parametrize("dims,geom,exotic", TILE_GRIDS, ids=["40x24x20_geom", "36x20x12_exotic", "64x16x5_empty"])
@pytest.mark.parametrize("amp", [2.0, 4.7, 5.2, 8.0, 14.5, 25.0])
def test_maccormack_ours_in_the_tile_kernels_regimes(orc, ref, dims, geom, exotic, amp):
    """The inputs of tests/test_gpu_advect_tile.py (the GPU's shared-memory tile kernels are compared with the
    restatement there), plus amplitudes right at the trace lengths where the GPU dispatcher switches code paths
    (0.47 / 0.52 cell: halo 1 -> 2; 1.45: halo 2 -> general): here the restatement itself is pinned on the
    reference's compiled CPU code for exactly these fields, single batch element as the tile kernels take."""
    from fluidnet_b200 import synth
    nx, ny, nz = dims
    flags = synth.make_flags(nx, ny, nz, True, nb=1, geometry=geom, exotic=exotic)
    U = synth.make_velocity(flags, True, amp=amp)
    orc.setWallBcsForward(U, flags)
    rho = synth.make_density(flags)
    rho[np.random.RandomState(3).rand(*rho.shape) < 0.3] = 0.0

    def run(be):
        out = {"advectVel": be.advectVel(0.1, U, flags, "maccormackOurs", 0.6)}
        for outside in (False, True):
            out["advectScalar/outside=%d" % outside] = be.advectScalar(0.1, rho, U, flags, "maccormackOurs",
                                                                       outside, 0.6)
        return out
    ref.check(orc, run)


def test_signed_zero_fields_match_the_reference(orc, ref):
    """+0 / -0 mixtures (the clamp's compare-and-keep order decides the sign of a zero bound): the input of
    test_gpu_advect_tile.py::test_zero_bounds_keep_their_sign, restatement vs compiled reference."""
    from fluidnet_b200 import synth
    flags = synth.make_flags(40, 24, 20, True, nb=1, geometry=True)
    U = synth.make_smooth_velocity(flags, True, amp=3.0)
    rng = np.random.RandomState(5)
    U[rng.rand(*U.shape) < 0.35] = 0.0
    U[rng.rand(*U.shape) < 0.2] = -0.0
    orc.setWallBcsForward(U, flags)
    ref.check(orc, lambda be: {"advectVel": be.advectVel(0.1, U, flags, "maccormackOurs", 0.6)})
