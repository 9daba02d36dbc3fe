"""The PCG restatement (oracle/tfluids_oracle.c: orc_find_components, orc_pcg).

Pinned where the reference has CPU code (the connected-component flood fill, compiled in place into
oracle/_ref); the solver itself is CUDA-only in the reference, so it is checked the way the
reference's own test does (tfluids/test_tfluids.lua:836-905: residual < 2 tol, max|div| after the
velocity update < 1e-4) plus an independent direct solve of the same linear system."""
import numpy as np
import pytest

import oracle
from oracle import api
import pcg_cases


@pytest.fixture(scope="module")
def orc():
    return api.Oracle()


@pytest.mark.parametrize("is3d", [True, False])
def test_components_match_reference(orc, ref, is3d):
    cases = []
    for seed in range(3):
        flags, _, _ = pcg_cases.make(orc, is3d, nb=2, seed=seed)
        rng = np.random.default_rng(seed)
        flags[(rng.random(flags.shape) < 0.25) & (flags == 1)] = 2      # many small components
        cases.append(flags)

    def run(be):
        out = {}
        for seed, flags in enumerate(cases):
            for b in range(flags.shape[0]):
                comp, sizes = be.findConnectedFluidComponents(flags, is3d, b)
                out["seed=%d/b=%d/components" % (seed, b)] = comp
                out["seed=%d/b=%d/sizes" % (seed, b)] = sizes
        return out
    ref.check(orc, run)
    for flags in cases:
        for b in range(flags.shape[0]):
            assert len(orc.findConnectedFluidComponents(flags, is3d, b)[1]) > 3


@pytest.mark.parametrize("precond", ["none", "ilu0", "ic0"])
@pytest.mark.parametrize("is3d", [True, False])
def test_pcg_reference_criteria(orc, is3d, precond):
    flags, U, div = pcg_cases.make(orc, is3d)
    p = np.random.default_rng(1).random(flags.shape).astype(np.float32)   # overwritten: p <- 0 first
    tol = 1e-5
    res = orc.solveLinearSystemPCG(p, flags, div, is3d, tol, 1000, precond)
    assert res < 2 * tol
    assert not np.isnan(p).any()
    U2 = U.copy()
    orc.velocityUpdateForward(U2, flags, p)
    assert np.abs(orc.velocityDivergenceForward(U2, flags)).max() < 1e-4
    assert np.all(p[flags != 1] == 0)


def test_pcg_solves_the_reference_matrix(orc):
    """p (up to the removed mean) solves A p = div with A from setupLaplacian (generic/tfluids.cu:909-1095)."""
    import scipy.sparse as sp
    import scipy.sparse.linalg as spl
    flags, U, div = pcg_cases.make(orc, True, nb=1, n=(12, 11, 10))
    p = np.zeros(flags.shape, np.float32)
    orc.solveLinearSystemPCG(p, flags, div, True, 1e-6, 2000, "ic0")
    comp, sizes = orc.findConnectedFluidComponents(flags, True, 0)
    f = flags[0, 0].astype(np.int32)
    nz, ny, nx = f.shape
    for ic, size in enumerate(sizes):
        cells = np.argwhere(comp == ic)
        if size == 1:
            assert p[0, 0][tuple(cells[0])] == 0
            continue
        index = {tuple(c): q for q, c in enumerate(cells)}
        rows, cols, vals = [], [], []
        for q, (k, j, i) in enumerate(cells):
            diag = 0
            for dk, dj, di in ((0, 0, -1), (0, 0, 1), (0, -1, 0), (0, 1, 0), (-1, 0, 0), (1, 0, 0)):
                nb = f[k + dk, j + dj, i + di]
                if not nb & 2:
                    diag += 1
                if nb & 1:
                    rows.append(q); cols.append(index[(k + dk, j + dj, i + di)]); vals.append(-1.0)
            rows.append(q); cols.append(q); vals.append(float(diag))
        A = sp.csr_matrix((vals, (rows, cols)), shape=(size, size))
        x = np.array([p[0, 0][tuple(c)] for c in cells], np.float64)
        rhs = np.array([div[0, 0][tuple(c)] for c in cells], np.float64)
        assert abs(x.mean()) < 1e-5
        assert np.abs(A @ x - rhs).max() < 2e-5          # singular (pure Neumann) system: any shift of x solves it


def test_pcg_preconditioner_cuts_iterations(orc):
    flags, U, div = pcg_cases.make(orc, True, nb=1, pockets=False)
    its = {}
    for precond in ("none", "ic0"):
        p = np.zeros(flags.shape, np.float32)
        orc.solveLinearSystemPCG(p, flags, div, True, 1e-5, 1000, precond)
        its[precond] = orc.last_pcg_iters
    assert its["ic0"] < its["none"]


def test_pcg_fluid_on_border_raises(orc):
    flags, U, div = pcg_cases.make(orc, True, nb=1)
    flags[0, 0, 0, 5, 5] = 1
    with pytest.raises(RuntimeError, match="Non fluid cell"):
        orc.solveLinearSystemPCG(np.zeros(flags.shape, np.float32), flags, div, True, 1e-5, 10, "ic0")


def test_pcg_max_iter_semantics(orc):
    """`while (rr > tol^2 && iter <= maxIter)` runs maxIter + 1 iterations (generic/tfluids.cu:1588)."""
    flags, U, div = pcg_cases.make(orc, True, nb=1, pockets=False)
    p = np.zeros(flags.shape, np.float32)
    orc.solveLinearSystemPCG(p, flags, div, True, 1e-12, 3, "none")
    assert orc.last_pcg_iters == 4
