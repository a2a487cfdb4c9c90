"""Pins the oracle to the REFERENCE'S OWN SOURCE: oracle/_ref/libref_ldu.so and libref_gamg.so are
the reference's lduMatrixATmul.C (Amul, Tmul, sumA, residual, H1 + matrixMultiplyFunctor),
lduAddressingFunctors.H, AINVPreconditionerF.H, JacobiSmootherF.H and pairGAMGAgglomerate.C compiled
for the host against type shims (oracle/ref_harness/, `make -C oracle ref`).  The oracle must agree
with that code BIT FOR BIT on hex meshes (at most three faces per side of a cell, where the
reference's unrolled row sum has no tail) and map for map in the pair agglomeration.

Scope of the claim: host compilation with floating-point contraction off; the CUDA build of the
reference may fuse a*b+c where the source allows it (DESIGN.md section 2)."""
import importlib

import numpy as np
import pytest

import ref_replay
from oracle import ref_ldu

ref_replay.install()   # the reference's answers come from tests/golden/ref_calls_*.npz


def _pair(meshmod, orc, dims, kind):
    m = meshmod.hex_mesh(*dims)
    c = meshmod.pressure_laplacian(m) if kind == "P" else meshmod.momentum_matrix(m)
    a = orc.Addr(m.nCells, m.lower, m.upper)
    M = orc.Matrix(a, c["diag"], c["upper"], c["lower"])
    R = ref_ldu.RefMatrix(m.nCells, m.lower, m.upper, a.owner_start(), a.losort_start(), a.losort(),
                          c["diag"], c["upper"], c["lower"])
    return m, M, R


@pytest.mark.parametrize("dims", [(7, 5, 4), (16, 16, 16), (13, 1, 1), (1, 1, 1)])
@pytest.mark.parametrize("kind", ["P", "U"])
def test_matrix_operations_match_reference_code(meshmod, orc, dims, kind):
    m, M, R = _pair(meshmod, orc, dims, kind)
    x, b = meshmod.cell_field_global(m, 3), meshmod.cell_field_global(m, 4)
    for favourSpeed in (0, 1, 2):   # losort indirection / pre-sorted coefficients (lduMatrixATmul.C:191-192)
        assert np.array_equal(R.op("amul", favourSpeed, x), M.amul(x))
        assert np.array_equal(R.op("tmul", favourSpeed, x), M.tmul(x))
        assert np.array_equal(R.op("sumA", favourSpeed), M.sumA())
        assert np.array_equal(R.op("residual", favourSpeed, x, b), M.residual(x, b))
        assert np.array_equal(R.op("H1", favourSpeed), M.H1())


@pytest.mark.parametrize("kind", ["P", "U"])
def test_ainv_and_jacobi_match_reference_functors(meshmod, orc, kind):
    m, M, R = _pair(meshmod, orc, (9, 8, 7), kind)
    x, b = meshmod.cell_field_global(m, 5), meshmod.cell_field_global(m, 6)
    for fast in (False, True):
        for T in (False, True):
            assert np.array_equal(R.ainv(x, fast, T), M.precondition("DIC", x, T))
        for omega in (0.9, 1.0, 0.5):
            assert np.array_equal(R.jacobi(x, b, omega, fast), M.jacobi(x, b, 1, omega=omega))


def test_rows_with_more_than_three_faces_per_side(meshmod, orc):
    """Beyond the unrolled three faces per side the reference keeps a separate tail sum in Amul
    (`return out + nExtra`, lduMatrixATmul.C:122-137) and -- in the `fast` variant of the generic
    functor used by residual and H1 -- accumulates the neighbour tail in `nExtra` and then returns
    `out` alone (lduAddressingFunctors.H:126-139), i.e. drops those terms.  The oracle sums every
    term in row order: equal to the reference's general path up to rounding, and deliberately not
    equal to the dropped-term result."""
    rng = np.random.default_rng(0)
    n = 400
    a_, b_ = rng.integers(0, n, 6 * n), rng.integers(0, n, 6 * n)
    keep = a_ != b_
    pr = np.unique(np.stack([np.minimum(a_, b_)[keep], np.maximum(a_, b_)[keep]], 1), axis=0).astype(np.int32)
    lo, up = pr[:, 0].copy(), pr[:, 1].copy()
    U, L = rng.uniform(-1, 1, len(lo)), rng.uniform(-1, 1, len(lo))
    D = rng.uniform(5, 6, n)
    a = orc.Addr(n, lo, up)
    M = orc.Matrix(a, D, U, L)
    R = ref_ldu.RefMatrix(n, lo, up, a.owner_start(), a.losort_start(), a.losort(), D, U, L)
    assert np.diff(a.losort_start()).max() > 3 and np.diff(a.owner_start()).max() > 3
    x, b = rng.standard_normal(n), rng.standard_normal(n)
    np.testing.assert_allclose(R.op("amul", 0, x), M.amul(x), rtol=1e-13, atol=1e-13)
    np.testing.assert_allclose(R.op("residual", 0, x, b), M.residual(x, b), rtol=1e-13, atol=1e-13)
    assert np.array_equal(R.op("residual", 0, x, b), M.residual(x, b))       # general functor: plain row order
    dropped = R.op("residual", 1, x, b)                                        # fast functor loses the tail
    assert np.abs(dropped - M.residual(x, b)).max() > 1e-3


@pytest.mark.parametrize("dims", [(12, 10, 8), (7, 5, 3), (16, 16, 16)])
@pytest.mark.parametrize("forward0", [1, 0])
def test_pair_agglomeration_matches_reference_code(meshmod, orc, dims, forward0):
    """pairGAMGAgglomeration::agglomerate (pairGAMGAgglomerate.C:135-313), level by level: the
    reference's code run on the oracle's coarse addressing and restricted weights gives the oracle's
    fine->coarse map, coarse cell count and `forward_` flag on every level."""
    m = meshmod.hex_mesh(*dims)
    a = orc.Addr(m.nCells, m.lower, m.upper)
    w = meshmod.face_area_pair_weights(m)
    g = orc.Gamg(a, w, 10, forward=forward0)
    lo, up, n, fwd = m.lower, m.upper, m.nCells, forward0
    assert g.nLevels >= 3
    for lev in range(g.nLevels):
        rmap, nC, fwd = ref_ldu.pair_agglomerate(n, lo, up, w, fwd)
        assert nC == g.ncells(lev)
        assert np.array_equal(rmap, g.restrict_addr(lev))
        fr, la = g.face_restrict_addr(lev), g.level_addr(lev)
        cw = np.zeros(g.nfaces(lev))
        np.add.at(cw, fr[fr >= 0], w[fr >= 0])   # restrictFaceField of the weights (pairGAMGAgglomerate.C:86-107)
        lo, up, n, w = la.lower(), la.upper(), nC, cw
    _, nC, fwd = ref_ldu.pair_agglomerate(n, lo, up, w, fwd)   # the step continueAgglomerating rejects
    assert nC < 10 and fwd == g.forward


def _solver_case(meshmod, orc, kind, dims=(9, 8, 7)):
    m = meshmod.hex_mesh(*dims)
    c = meshmod.pressure_laplacian(m) if kind == "P" else meshmod.momentum_matrix(m)
    a = orc.Addr(m.nCells, m.lower, m.upper)
    M = orc.Matrix(a, c["diag"], c["upper"], c["lower"])
    args = (m.nCells, m.lower, m.upper, a.owner_start(), a.losort_start(), a.losort(), c["diag"], c["upper"], c["lower"])
    b = M.amul(meshmod.cell_field_global(m, 42))
    return m, M, args, b


@pytest.mark.parametrize("kind,solver,pre", [("P", "PCG", "DIC"), ("P", "PCG", "diagonal"), ("P", "PCG", "none"),
                                             ("U", "PBiCG", "DILU"), ("U", "PBiCG", "diagonal"), ("U", "PBiCG", "none"),
                                             ("U", "PBiCGStab", "DILU"), ("U", "PBiCGStab", "none")])
def test_solver_loops_match_reference_code(meshmod, orc, kind, solver, pre):
    """The reference's own PCG.C / PBiCG.C / PBiCGStab.C loops (+ its preconditioner classes) against
    the oracle: same printed solver name, bit-identical normFactor-scaled initial residual, identical
    iteration count, and the residual after k iterations equal to 1e-11 while rounding differences are
    still small (the reference's vector updates are compiled unfused here, the oracle uses the FMAs
    nvcc generates for them -- oracle/_ref/device_probe_sass.txt; CG-type recurrences amplify that
    one-ulp difference exponentially, so later iterations are compared through the iteration count).
    PBiCGStab: the reference adds omega*yA where the algorithm needs omega*zA (PBiCGStab.C:263-270); the
    oracle's `bicgstabRefQuirk=1` mode reproduces its solution, the default mode is the corrected one."""
    m, M, args, b = _solver_case(meshmod, orc, kind)
    quirk = 1 if solver == "PBiCGStab" else 0
    kw = dict(tolerance=1e-9, maxIter=300)
    psi_o, po, ho = M.solve(solver, pre, np.zeros(m.nCells), b, bicgstabRefQuirk=quirk, **kw)
    psi_r, pr = ref_ldu.solve(solver, pre, *args, np.zeros(m.nCells), b, **kw)
    assert pr["solverName"] == po.solverName.decode()
    assert pr["initialResidual"] == po.initialResidual
    assert pr["nIterations"] == po.nIterations and pr["converged"] == bool(po.converged)
    np.testing.assert_allclose(psi_r, psi_o, rtol=0, atol=1e-8)
    for k in (0, 1, 2, 3, 5, 8, 12):           # residual after k+1 loop bodies (tolerance 0 => maxIter+1 bodies)
        if k + 1 >= len(ho) - 1:
            break
        _, prk = ref_ldu.solve(solver, pre, *args, np.zeros(m.nCells), b, tolerance=0.0, maxIter=k)
        assert prk["nIterations"] == k + 1
        assert abs(prk["finalResidual"] - ho[k + 1]) <= 1e-11 * ho[k + 1], (k, prk["finalResidual"], ho[k + 1])
    if solver == "PBiCGStab":
        psi_fixed, pf, _ = M.solve(solver, pre, np.zeros(m.nCells), b, bicgstabRefQuirk=0, **kw)
        xs = meshmod.cell_field_global(m, 42)
        assert np.abs(psi_fixed - xs).max() < 1e-6          # corrected update solves the system
        assert np.abs(psi_r - xs).max() > 1e-2              # the reference's update does not
        assert pf.nIterations == pr["nIterations"]          # (its residual recurrence is unaffected)


def test_loop_semantics_match_reference_code(meshmod, orc):
    """maxIter+1 bodies (post-increment test), minIter, relTol, immediate convergence: PCG.C:196-208"""
    m, M, args, b = _solver_case(meshmod, orc, "P", (6, 5, 4))
    z = np.zeros(m.nCells)
    for kw in (dict(tolerance=0.0, maxIter=5), dict(tolerance=1e30, maxIter=50, minIter=3), dict(tolerance=1e30, maxIter=50),
               dict(tolerance=0.0, relTol=0.1, maxIter=200), dict(tolerance=0.0, maxIter=0)):
        _, po, ho = M.solve("PCG", "DIC", z, b, **kw)
        _, pr = ref_ldu.solve("PCG", "DIC", *args, z, b, **kw)
        assert pr["nIterations"] == po.nIterations, kw
        assert pr["converged"] == bool(po.converged), kw
        assert abs(pr["finalResidual"] - po.finalResidual) <= 1e-10 * max(po.finalResidual, 1e-300), kw
    with pytest.raises(ValueError):
        ref_ldu.solve("PCG", "FDIC", *args, z, b)


@pytest.mark.parametrize("kind", ["P", "U"])
def test_smooth_solver_matches_reference_code_bit_for_bit(meshmod, orc, kind):
    """smoothSolver.C:77-193 + JacobiSmoother.C:39-148 (the reference's own loops): no vector update
    outside the row functor, so solution and residuals are identical to the last bit, for positive
    and negative nSweeps, a dictionary omega, and the `(nIterations += nSweeps) < maxIter` test."""
    m, M, args, b = _solver_case(meshmod, orc, kind)
    z = np.zeros(m.nCells)
    for kw in (dict(tolerance=1e-6, maxIter=200, nSweeps=1), dict(tolerance=1e-6, maxIter=200, nSweeps=3),
               dict(nSweeps=-4), dict(tolerance=1e-6, maxIter=50, nSweeps=2, omega=0.7),
               dict(tolerance=0.0, maxIter=7, nSweeps=2), dict(tolerance=1e30, maxIter=9, nSweeps=2, minIter=5)):
        for smoother in ("GaussSeidel", "Jacobi"):
            psi_o, po, _ = M.solve("smoothSolver", smoother, z, b, **kw)
            psi_r, pr = ref_ldu.solve("smoothSolver", smoother, *args, z, b, **kw)
            assert pr["nIterations"] == po.nIterations and pr["converged"] == bool(po.converged), kw
            assert np.array_equal(psi_r, psi_o), kw
            assert pr["finalResidual"] == po.finalResidual and pr["initialResidual"] == po.initialResidual, kw
            assert pr["solverName"] == po.solverName.decode() == "smoothSolver"


@pytest.mark.parametrize("kind", ["P", "U"])
def test_gamg_vcycle_matches_reference_code_bit_for_bit(meshmod, orc, kind):
    """The reference's own GAMGSolver::solve / Vcycle / scale (GAMGSolverSolve.C, GAMGSolverScale.C) and
    JacobiSmoother, run on the oracle's level hierarchy: identical cycle counts, solution and residuals
    to the last bit for every combination of the sweep controls, the scaling switch and the loop limits
    (`++nIterations < maxIter`, minIter).  With the Krylov coarsest solve only the fused vector updates
    of that inner solve differ (rounding level).  interpolateCorrection: the reference itself ends in
    notImplemented() (GAMGSolverInterpolate.C:171); this repo runs the part that exists (DESIGN.md)."""
    m = meshmod.hex_mesh(12, 10, 8)
    c = meshmod.pressure_laplacian(m) if kind == "P" else meshmod.momentum_matrix(m)
    a = orc.Addr(m.nCells, m.lower, m.upper)
    M = orc.Matrix(a, c["diag"], c["upper"], c["lower"])
    g = orc.Gamg(a, meshmod.face_area_pair_weights(m), 10)
    b = M.amul(meshmod.cell_field_global(m, 42))
    z = np.zeros(m.nCells)
    for kw in (dict(), dict(nPreSweeps=1), dict(nPreSweeps=2, nFinestSweeps=1, scaleCorrection=1),
               dict(nPostSweeps=1, maxPostSweeps=2, nFinestSweeps=3), dict(scaleCorrection=0),
               dict(preSweepsLevelMultiplier=2, nPreSweeps=1, maxPreSweeps=3, postSweepsLevelMultiplier=0),
               dict(maxIter=3, tolerance=0.0), dict(tolerance=1e30, minIter=2), dict(omega=0.8)):
        okw = dict(tolerance=1e-8, maxIter=100)
        okw.update(kw)
        psi_o, po, ho = g.solve(M, "GaussSeidel", z, b, **okw)
        psi_r, pr = ref_ldu.gamg_solve(g, a, c["diag"], c["upper"], c["lower"], z, b, **okw)
        assert pr["nIterations"] == po.nIterations and pr["converged"] == bool(po.converged), kw
        assert pr["initialResidual"] == po.initialResidual and pr["finalResidual"] == po.finalResidual, kw
        assert np.array_equal(psi_r, psi_o), kw
    okw = dict(tolerance=1e-8, maxIter=100, directSolveCoarsest=0)
    psi_o, po, _ = g.solve(M, "GaussSeidel", z, b, **okw)
    psi_r, pr = ref_ldu.gamg_solve(g, a, c["diag"], c["upper"], c["lower"], z, b, **okw)
    assert pr["nIterations"] == po.nIterations
    np.testing.assert_allclose(psi_r, psi_o, rtol=0, atol=1e-11)
    with pytest.raises(NotImplementedError):
        ref_ldu.gamg_solve(g, a, c["diag"], c["upper"], c["lower"], z, b, interpolateCorrection=1)


@pytest.mark.parametrize("kind", ["P", "U"])
def test_H_faceH_and_diagonal_sums_match_reference_code(meshmod, orc, kind):
    """lduMatrix::H / faceH (lduMatrixTemplates.C:50-160, the reference's own templates) and the
    sumDiag / negSumDiag / sumMagOffDiag compositions of lduMatrixOperations.C:36-104 built from the
    reference's functors: bit for bit."""
    m, M, R = _pair(meshmod, orc, (8, 6, 5), kind)
    x = meshmod.cell_field_global(m, 7)
    assert np.array_equal(R.op("H", 0, x), M.H(x))
    assert np.array_equal(R.op("faceH", 0, x), M.faceH(x))
    L = orc.lib()
    a = M.addr
    c = meshmod.pressure_laplacian(m) if kind == "P" else meshmod.momentum_matrix(m)
    upper, lower = orc.f64(c["upper"]), orc.f64(c["lower"] if c["lower"] is not None else c["upper"])
    d0 = meshmod.cell_field_global(m, 8)
    for name, fn in (("negSumDiag", L.orc_negSumDiag), ("sumDiag", L.orc_sumDiag), ("sumMagOffDiag", L.orc_sumMagOffDiag)):
        d = d0.copy()
        fn(a.h, orc._d(upper), orc._d(lower), orc._d(d))
        assert np.array_equal(R.op(name, 0, None, d0), d), name   # all three add to the incoming field


@pytest.mark.parametrize("dims", [(12, 10, 8), (7, 5, 3), (9, 9, 9)])
def test_coarse_addressing_and_combine_levels_match_reference_code(meshmod, orc, dims):
    """GAMGAgglomeration::agglomerateLduAddressing (GAMGAgglomerateLduAddressing.C:245-603, the reference's
    own code): coarse owner/neighbour in its discovery + renumbering order, face restrict map and flip
    map equal the oracle's on every level.  combineLevels (:606-765) applied by the reference to steps 0
    and 1 gives level 0 of the oracle's mergeLevels-2 hierarchy -- including its rule that the flip of a
    composed face is the flip of the second step alone (:631)."""
    m = meshmod.hex_mesh(*dims)
    a = orc.Addr(m.nCells, m.lower, m.upper)
    w = meshmod.face_area_pair_weights(m)
    g1, g2 = orc.Gamg(a, w, 10), orc.Gamg(a, w, 10, mergeLevels=2)
    lo, up, n = m.lower, m.upper, m.nCells
    for lev in range(g1.nLevels):
        R = ref_ldu.coarse_levels(n, lo, up, g1.restrict_addr(lev), g1.ncells(lev))
        la = g1.level_addr(lev)
        assert R["nCoarseCells"] == g1.ncells(lev)
        assert np.array_equal(R["coarseOwner"], la.lower()) and np.array_equal(R["coarseNeighbour"], la.upper())
        assert np.array_equal(R["faceRestrict"], g1.face_restrict_addr(lev))
        assert np.array_equal(R["flip"], g1.face_flip(lev))
        lo, up, n = la.lower(), la.upper(), g1.ncells(lev)
    R = ref_ldu.coarse_levels(m.nCells, m.lower, m.upper, g1.restrict_addr(0), g1.ncells(0), g1.restrict_addr(1),
                              g1.ncells(1))
    la = g2.level_addr(0)
    assert R["nCoarseCells"] == g2.ncells(0)
    assert np.array_equal(R["restrict"], g2.restrict_addr(0))
    assert np.array_equal(R["faceRestrict"], g2.face_restrict_addr(0))
    assert np.array_equal(R["coarseOwner"], la.lower()) and np.array_equal(R["coarseNeighbour"], la.upper())
    kept = R["faceRestrict"] >= 0      # the flip of a face that collapses into a cell is never read
    assert np.array_equal(R["flip"][kept], g2.face_flip(0)[kept])
    # the rule differs from the exclusive-or of the two steps on some faces: the test would notice a "fixed" rule
    f0, fr0, f1 = g1.face_flip(0).astype(bool), g1.face_restrict_addr(0), g1.face_flip(1).astype(bool)
    both = (fr0 >= 0) & kept
    xor = f0[both] ^ f1[fr0[both]]
    if dims == (9, 9, 9):
        assert f0[both].any()          # this mesh has faces flipped in step 0 that survive both steps
    if f0[both].any():
        assert np.any(xor != R["flip"][both].astype(bool))


@pytest.mark.parametrize("kind", ["P", "U"])
@pytest.mark.parametrize("dims", [(9, 9, 9), (7, 5, 3)])
def test_coarse_matrix_assembly_matches_reference_functors(meshmod, orc, kind, dims):
    """Coarse coefficients level by level: the reference's restriction and agglomeration functors
    (GAMGAgglomerationF.H, GAMGSolverAgglomerateMatrixF.H) run over the sorted addressing its own
    createSort/createTarget built, against ref_ldu.coarse_matrix -- the plain summation that feeds the
    reference V-cycle in test_gamg_vcycle_matches_reference_code_bit_for_bit, where it reproduces the
    oracle's coarse matrices to the last bit.  (9,9,9) has flipped faces: upper/lower swap exercised.)"""
    m = meshmod.hex_mesh(*dims)
    c = meshmod.pressure_laplacian(m) if kind == "P" else meshmod.momentum_matrix(m)
    a = orc.Addr(m.nCells, m.lower, m.upper)
    g = orc.Gamg(a, meshmod.face_area_pair_weights(m), 10)
    lo, up, n = m.lower, m.upper, m.nCells
    D, U, L = c["diag"], c["upper"], c["lower"]
    for lev in range(g.nLevels):
        R = ref_ldu.coarse_levels(n, lo, up, g.restrict_addr(lev), g.ncells(lev), diag=D, upperC=U, lowerC=L)
        Dn, Un, Ln = ref_ldu.coarse_matrix(g.restrict_addr(lev), g.face_restrict_addr(lev), g.face_flip(lev),
                                           g.ncells(lev), g.nfaces(lev), D, U, L)
        assert np.array_equal(R["coarseDiag"], Dn) and np.array_equal(R["coarseUpper"], Un), lev
        assert L is None or np.array_equal(R["coarseLower"], Ln), lev
        la = g.level_addr(lev)
        lo, up, n, D, U, L = la.lower(), la.upper(), g.ncells(lev), Dn, Un, Ln


def test_interface_update_matches_reference_functor(meshmod, orc):
    """Coupled-interface contribution (coupledFvPatchField.C:236-257) through the reference's
    matrixPatchOperation + matrixInterfaceFunctor: the oracle's Amul / residual / Jacobi on a matrix
    with coupled (cyclic) patches equal the reference's interior operator followed by the reference's
    interface update, bit for bit -- several patch faces per cell included."""
    from test_oracle_core import _cyclic_case
    for kind in ("P", "U"):
        m, c, ps, fc, nr, lo, hi = _cyclic_case(meshmod, kind)
        a = orc.Addr(m.nCells, m.lower, m.upper, ps, fc, neighbRank=nr)
        M = orc.Matrix(a, c["diag"], c["upper"], c["lower"], c["bou"], c["int"])
        R = ref_ldu.RefMatrix(m.nCells, m.lower, m.upper, a.owner_start(), a.losort_start(), a.losort(),
                              c["diag"], c["upper"], c["lower"])
        x = meshmod.cell_field_global(m, 3)
        n = len(lo)
        pnf = np.concatenate([x[hi], x[lo]])                 # cyclic: psi at the partner's face cells
        ref = R.op("amul", 0, x)
        for p in range(2):                                   # updateMatrixInterfaces visits the patches in order
            sl = slice(p * n, (p + 1) * n)
            ref = ref_ldu.interface_update(m.nCells, fc[sl], c["bou"][sl], pnf[sl], ref)
        assert np.array_equal(ref, M.amul(x))
        reft = R.op("tmul", 0, x)
        for p in range(2):
            sl = slice(p * n, (p + 1) * n)
            reft = ref_ldu.interface_update(m.nCells, fc[sl], c["int"][sl], pnf[sl], reft)
        assert np.array_equal(reft, M.tmul(x))
    # several faces of one patch on the same cell, both signs
    rng = np.random.default_rng(4)
    fcs = np.array([3, 1, 3, 0, 1, 3], dtype=np.int32)
    co, v, r0 = rng.standard_normal(6), rng.standard_normal(6), rng.standard_normal(5)
    for negate in (False, True):
        exp = r0.copy()
        for i in range(6):
            t = co[i] * v[i]
            exp[fcs[i]] = exp[fcs[i]] + (t if negate else -t)
        assert np.array_equal(ref_ldu.interface_update(5, fcs, co, v, r0, negate), exp)


def test_derived_addressing_matches_reference_code(meshmod, orc):
    """lduAddressing.C (the reference's own thrust sorts and scans): ownerStart, losortStart, losort,
    ownerSort equal the oracle's arrays (row a1 of SURVEY section 8) on a hex mesh, on a randomly
    renumbered one and on a decomposed piece; the per-patch sort addressing groups the patch faces by
    cell in ascending patch-face order, which is the order the oracle applies interface terms in."""
    from test_foamfile_cpu import _scrambled
    ff = importlib.import_module("rapidcfd-dev_b200.foamfile")
    cases = [meshmod.hex_mesh(7, 5, 4), meshmod.decompose(8, 4, 1)]
    pm, _ = _scrambled(ff, meshmod, (6, 5, 4), 5)
    lo_s, up_s = pm.ldu()
    for m in cases + [None]:
        if m is None:
            n, lo, up, ps, fc = pm.nCells, lo_s, up_s, None, None
        else:
            n, lo, up = m.nCells, m.lower, m.upper
            ps, fc = m.patch_start_facecells()
            if len(ps) == 1:
                ps = fc = None
        a = orc.Addr(n, lo, up) if ps is None else orc.Addr(n, lo, up, ps, fc)
        R = ref_ldu.ldu_addressing(n, lo, up, ps, fc)
        assert np.array_equal(R["ownerStart"], a.owner_start())
        assert np.array_equal(R["losortStart"], a.losort_start())
        assert np.array_equal(R["losort"], a.losort())
        assert np.array_equal(R["ownerSort"], np.asarray(lo)[a.losort()])
        os2, ls2, lo2 = ref_ldu.ldu_arrays(n, lo, up)           # the numpy helper used by the harness drivers
        assert np.array_equal(os2, R["ownerStart"]) and np.array_equal(ls2, R["losortStart"]) and np.array_equal(lo2, R["losort"])
        assert R["bandwidth"] == int((np.asarray(up) - np.asarray(lo)).max())
        if ps is not None:
            for p in range(len(ps) - 1):
                cells = np.asarray(fc[ps[p]:ps[p + 1]])
                order = R["patchSortAddr"][p]
                assert np.array_equal(order, np.argsort(cells, kind="stable"))      # by cell, then ascending patch face
                assert np.array_equal(R["patchSortCells"][p], np.unique(cells))
                st = R["patchSortStart"][p]
                assert st[0] == 0 and st[-1] == len(cells) and np.all(np.diff(st) > 0)


def test_runtime_selection_matches_reference_code(meshmod, orc):
    """lduMatrix::solver::New (lduMatrixSolver.C:43-140, the reference's own tables filled by the static
    add...ConstructorToTable objects of PCG.C, PBiCG.C, ...): PCG exists for symmetric matrices only,
    PBiCG and PBiCGStab for asymmetric only (PBiCGStab.C:34-37), smoothSolver for both, unknown names are
    fatal -- the same outcomes as the oracle's (and the C ABI's) selection."""
    for kind in ("P", "U"):
        m, M, args, b = _solver_case(meshmod, orc, kind, (5, 4, 3))
        z = np.zeros(m.nCells)
        for solver, second in (("PCG", "DIC"), ("PBiCG", "DILU"), ("PBiCGStab", "DILU"), ("smoothSolver", "GaussSeidel"),
                               ("GaussSeidel", "DIC"), ("pcg", "DIC")):
            try:
                ref_ldu.solve(solver, second, *args, z, b, maxIter=3)
                ref_ok = True
            except ValueError:
                ref_ok = False
            try:
                M.solve(solver, second, z, b, maxIter=3)
                orc_ok = True
            except Exception:  # noqa: BLE001
                orc_ok = False
            assert ref_ok == orc_ok, (kind, solver)
            expected = {"PCG": kind == "P", "PBiCG": kind == "U", "PBiCGStab": kind == "U", "smoothSolver": True}.get(solver, False)
            assert ref_ok == expected, (kind, solver)


def test_preconditioner_and_smoother_selection_matches_reference_code(meshmod, orc):
    """lduMatrix::preconditioner::New / smoother::New (lduMatrixPreconditioner.C, lduMatrixSmoother.C) with
    the tables the reference's classes register into: DIC exists for symmetric matrices only, DILU for
    asymmetric only (both are AINV), AINV / diagonal / none for both; GaussSeidel and Jacobi smoothers for
    both; anything else is fatal.  The oracle accepts and rejects the same names."""
    for kind in ("P", "U"):
        m, M, args, b = _solver_case(meshmod, orc, kind, (5, 4, 3))
        z = np.zeros(m.nCells)
        solver = "PCG" if kind == "P" else "PBiCG"
        cases = [(solver, p) for p in ("DIC", "DILU", "AINV", "diagonal", "none", "FDIC", "GAMG")]
        cases += [("smoothSolver", s) for s in ("GaussSeidel", "Jacobi", "symGaussSeidel", "DIC")]
        for sv, second in cases:
            try:
                _, pr = ref_ldu.solve(sv, second, *args, z, b, maxIter=2)
                ref_ok = True
            except ValueError:
                ref_ok = False
            try:
                _, po, _ = M.solve(sv, second, z, b, maxIter=2)
                orc_ok = True
            except Exception:  # noqa: BLE001
                orc_ok = False
            assert ref_ok == orc_ok, (kind, sv, second)
            if ref_ok:
                assert pr["solverName"] == po.solverName.decode(), (kind, sv, second)
        expected_ok = {"P": {"DIC", "AINV", "diagonal", "none"}, "U": {"DILU", "AINV", "diagonal", "none"}}[kind]
        for p in ("DIC", "DILU", "AINV", "diagonal", "none"):
            try:
                ref_ldu.solve(solver, p, *args, z, b, maxIter=1)
                ok = True
            except ValueError:
                ok = False
            assert ok == (p in expected_ok), (kind, p)



@pytest.mark.parametrize("dims", [(7, 5, 6), (1, 1, 9), (4, 4, 1)])
def test_fv_face_sums_match_reference_code(meshmod, orc, dims):
    """Row a16: the oracle's face sum against the reference's own fvc::surfaceIntegrate
    (fvcSurfaceIntegrate.C:41-205, compiled for the host), bit for bit -- sums only, no products."""
    m = meshmod.hex_mesh(*dims)
    a = orc.Addr(m.nCells, m.lower, m.upper)
    rng = np.random.default_rng(5)
    bfc = np.concatenate([p.faceCells for p in m.patches]).astype(np.int32)
    V = m.volumes() * rng.uniform(0.9, 1.1, m.nCells)
    ssf = rng.uniform(-1, 1, m.nFaces)
    bssf = rng.uniform(-1, 1, len(bfc))
    got = np.asarray(orc.surface_integrate(a, ssf, bfc, bssf, V, 1))
    ref = ref_ldu.surface_integrate(m.nCells, m.lower, m.upper, ssf, bfc, bssf, V)
    np.testing.assert_array_equal(got, ref)
    # and without boundary faces
    z = np.zeros(0)
    got = np.asarray(orc.surface_integrate(a, ssf, np.zeros(0, np.int32), z, V, 1))
    np.testing.assert_array_equal(got, ref_ldu.surface_integrate(m.nCells, m.lower, m.upper, ssf, [], z, V))
    # fvc::surfaceSum (:261-352): every face added, no division by the volumes
    got = np.asarray(orc.surface_integrate(a, ssf, bfc, bssf, V, 1, False, +1))
    ref = ref_ldu.surface_integrate(m.nCells, m.lower, m.upper, ssf, bfc, bssf, V, integrate=False)
    np.testing.assert_array_equal(got, ref)
    # fv::gaussGrad<scalar>::gradf (gaussGrad.C:34-243): products rounded, then summed in the same order
    Sf, bSf = m.Sf(), np.concatenate([p.Sf for p in m.patches])
    Sf, bSf = Sf + rng.uniform(-0.1, 0.1, Sf.shape), bSf + rng.uniform(-0.1, 0.1, bSf.shape)   # no exact zeros
    got = np.asarray(orc.gauss_grad(a, Sf.ravel(), ssf, bfc, bSf.ravel(), bssf, V, 1)).reshape(m.nCells, 3)
    ref = ref_ldu.gauss_gradf(m.nCells, m.lower, m.upper, Sf, ssf, bfc, bSf, bssf, V)
    np.testing.assert_array_equal(got, ref)
    # the vector instantiations: surfaceIntegrate / surfaceSum of a vector flux, gaussGrad<vector>::gradf (tensor result)
    vsf, bvsf = rng.uniform(-1, 1, (m.nFaces, 3)), rng.uniform(-1, 1, (len(bfc), 3))
    got = np.asarray(orc.surface_integrate(a, vsf.ravel(), bfc, bvsf.ravel(), V, 3)).reshape(m.nCells, 3)
    np.testing.assert_array_equal(got, ref_ldu.surface_integrate_vec(m.nCells, m.lower, m.upper, vsf, bfc, bvsf, V))
    got = np.asarray(orc.surface_integrate(a, vsf.ravel(), bfc, bvsf.ravel(), V, 3, False, +1)).reshape(m.nCells, 3)
    np.testing.assert_array_equal(got, ref_ldu.surface_integrate_vec(m.nCells, m.lower, m.upper, vsf, bfc, bvsf, V, False))
    got = np.asarray(orc.gauss_grad(a, Sf.ravel(), vsf.ravel(), bfc, bSf.ravel(), bvsf.ravel(), V, 3)).reshape(m.nCells, 3, 3)
    np.testing.assert_array_equal(got, ref_ldu.gauss_gradf_vec(m.nCells, m.lower, m.upper, Sf, vsf, bfc, bSf, bvsf, V))


def _oracle_rank_hierarchies(meshmod, orc, n, nR, mergeLevels, dims=None):
    import dist_helpers as dh
    ex = dh.ThreadExchange(nR)

    def rank_fn(r):
        m, c = dh.local_case(meshmod, n, nR, r, "P", dims=dims)
        a, M = dh.oracle_matrix(orc, m, c)
        comm = ex.comm(orc, r, m, n ** 3)
        g = orc.Gamg(a, meshmod.face_area_pair_weights(m), 6, mergeLevels=mergeLevels, comm=comm)
        levels = []
        for k in range(g.nLevels):
            ca = g.level_addr(k)
            levels.append(dict(restrict=g.restrict_addr(k), nCells=g.ncells(k), lower=ca.lower(), upper=ca.upper(),
                               faceRestrict=g.face_restrict_addr(k), faceFlip=g.face_flip(k),
                               patchStart=ca.patch_start(), faceCells=ca.face_cells(),
                               patchFaceRestrict=g.patch_face_restrict(k)))
        ps, fc = m.patch_start_facecells()
        fine = dict(nCells=m.nCells, lower=m.lower, upper=m.upper, patchStart=ps, faceCells=fc,
                    neighbRank=[p.neighbRank for p in m.coupled_patches()])
        rng = np.random.default_rng(100 + r)
        coeffs = [rng.uniform(-1, 1, int(ps[-1]))]
        for k in range(g.nLevels):
            coeffs.append(g.agglomerate_patch_coeffs(k, coeffs[-1]))
        return fine, levels, coeffs
    return dh.run_threads(nR, rank_fn)


@pytest.mark.parametrize("nR,dims", [(2, None), (4, None), (8, None), (4, (10, 6, 5))])
def test_coarse_interfaces_match_reference_code(meshmod, orc, nR, dims):
    """Row a14 (coarse-level side): the oracle's processor-interface agglomeration -- coarse patch faces as unique
    (master cell, slave cell) pairs in order of appearance, identical on both sides, the patch-face restrict map,
    the coefficient sums -- against the reference's GAMGAgglomerateLduAddressing.C (interface branch),
    GAMGInterface.C and processorGAMGInterface.C, all ranks of the decomposition in one process."""
    res = _oracle_rank_hierarchies(meshmod, orc, 8, nR, 1, dims)
    nLev = min(len(r[1]) for r in res)
    assert nLev >= 2
    ia = ref_ldu.InterfaceAgglomeration([r[0] for r in res])
    for k in range(nLev):
        got = ia.agglomerate(k, [r[1][k]["restrict"] for r in res], [r[1][k]["nCells"] for r in res])
        for r in range(nR):
            o, g = res[r][1][k], got[r]
            assert g["nCells"] == o["nCells"]
            for key in ("lower", "upper", "faceRestrict", "patchStart", "faceCells"):
                assert np.array_equal(g[key], o[key]), (k, r, key)
            inter = o["faceRestrict"] >= 0           # the flip of a face that collapses into a cell is never read
            assert np.array_equal(g["faceFlip"][inter] != 0, o["faceFlip"][inter] != 0)
            # the reference numbers coarse patch faces per patch, the oracle over all patches of the rank
            fineStart = np.concatenate([[0], np.cumsum(g["finePatchSizes"])])
            flat = np.concatenate([g["patchFaceRestrict"][fineStart[p]:fineStart[p + 1]] + g["patchStart"][p]
                                   for p in range(len(g["finePatchSizes"]))]) if len(g["finePatchSizes"]) else []
            assert np.array_equal(flat, o["patchFaceRestrict"]), (k, r)
            # GAMGInterface::agglomerateCoeffs, patch by patch, bit for bit
            fine, coarse = res[r][2][k], res[r][2][k + 1]
            for p in range(len(g["finePatchSizes"])):
                ref = ia.agglomerate_coeffs(k, r, p, fine[fineStart[p]:fineStart[p + 1]])
                assert np.array_equal(ref, coarse[g["patchStart"][p]:g["patchStart"][p + 1]]), (k, r, p)
    # both sides of every coarse interface enumerate the same faces: sizes agree pairwise on every level
    for k in range(nLev):
        for r in range(nR):
            nbrs = res[r][0]["neighbRank"]
            for p, nb in enumerate(nbrs):
                q = res[nb][0]["neighbRank"].index(r)
                mine, theirs = res[r][1][k]["patchStart"], res[nb][1][k]["patchStart"]
                assert mine[p + 1] - mine[p] == theirs[q + 1] - theirs[q]


def test_merged_coarse_interfaces_match_reference_code(meshmod, orc):
    """mergeLevels 2 over processor interfaces: combineLevels (GAMGAgglomerateLduAddressing.C:606-765) composes
    the patch-face maps and GAMGInterface::combine the interfaces."""
    nR = 2
    steps = _oracle_rank_hierarchies(meshmod, orc, 8, nR, 1)
    merged = _oracle_rank_hierarchies(meshmod, orc, 8, nR, 2)
    ia = ref_ldu.InterfaceAgglomeration([r[0] for r in steps])
    for k in (0, 1):
        ia.agglomerate(k, [r[1][k]["restrict"] for r in steps], [r[1][k]["nCells"] for r in steps])
    got = ia.combine(1)
    for r in range(nR):
        o, g = merged[r][1][0], got[r]
        assert g["nCells"] == o["nCells"]
        for key in ("lower", "upper", "faceRestrict", "patchStart"):
            assert np.array_equal(g[key], o[key]), (r, key)
        fineStart = np.concatenate([[0], np.cumsum(g["finePatchSizes"])])
        flat = np.concatenate([g["patchFaceRestrict"][fineStart[p]:fineStart[p + 1]] + g["patchStart"][p]
                               for p in range(len(g["finePatchSizes"]))])
        assert np.array_equal(flat, o["patchFaceRestrict"])
        assert np.array_equal(g["faceCells"], o["faceCells"])


def _random_examples(n=30, seed=20240611):
    """(dims, seed, symmetric, favourSpeed) of the property below: the smallest and largest boxes, then seeded draws --
    the same examples on every run, so that the reference's answers for them can be stored"""
    rng = np.random.default_rng(seed)
    out = [((1, 1, 1), 0, True, 0), ((6, 6, 5), 1, False, 2)]
    while len(out) < n:
        dims = (int(rng.integers(1, 7)), int(rng.integers(1, 7)), int(rng.integers(1, 6)))
        out.append((dims, int(rng.integers(0, 2**31)), bool(rng.integers(0, 2)), int(rng.integers(0, 3))))
    return out


def test_random_matrices_match_reference_code():
    """property: on any hex box with arbitrary coefficients the oracle's row operations equal the
    reference's code bit for bit (any favourSpeed path)"""
    for dims, seed, symmetric, favourSpeed in _random_examples():
        _random_matrix_matches_reference_code(dims, seed, symmetric, favourSpeed)


def _random_matrix_matches_reference_code(dims, seed, symmetric, favourSpeed):
    import importlib as _il
    meshmod = _il.import_module("rapidcfd-dev_b200.mesh")
    from oracle import ldu_oracle as orc
    m = meshmod.hex_mesh(*dims)
    rng = np.random.default_rng(seed)
    nF = m.nFaces
    D = rng.uniform(1.0, 9.0, m.nCells) * rng.choice([-1.0, 1.0])
    U = rng.standard_normal(nF)
    L = None if symmetric else rng.standard_normal(nF)
    a = orc.Addr(m.nCells, m.lower, m.upper)
    M = orc.Matrix(a, D, U, L)
    R = ref_ldu.RefMatrix(m.nCells, m.lower, m.upper, a.owner_start(), a.losort_start(), a.losort(), D, U, L)
    x, b = rng.standard_normal(m.nCells), rng.standard_normal(m.nCells)
    assert np.array_equal(R.op("amul", favourSpeed, x), M.amul(x))
    assert np.array_equal(R.op("tmul", favourSpeed, x), M.tmul(x))
    assert np.array_equal(R.op("residual", favourSpeed, x, b), M.residual(x, b))
    assert np.array_equal(R.op("sumA", favourSpeed), M.sumA())
    assert np.array_equal(R.op("H", 0, x), M.H(x))
    if nF:
        assert np.array_equal(R.op("faceH", 0, x), M.faceH(x))
    fast = favourSpeed > 0
    assert np.array_equal(R.ainv(x, fast, False), M.precondition("DIC", x, False))
    assert np.array_equal(R.ainv(x, fast, True), M.precondition("DIC", x, True))
    omega = float(rng.uniform(0.3, 1.0))
    assert np.array_equal(R.jacobi(x, b, omega, fast), M.jacobi(x, b, 1, omega=omega))


def _fvm_patches(m, d, cyc=None):
    """the flat wall list of tests/test_oracle_fvm.py split back into patches (+ the cyclic pair as coupled patches)"""
    out, off = [], 0
    for p in m.wall_patches():
        if cyc is not None and p.name in ("xmin", "xmax"):
            continue
        k = len(p.faceCells)
        out.append(dict(faceCells=p.faceCells, ic=d["ic"][off:off + k, 0], bc=d["bc"][off:off + k, 0]))
        off += k
    assert off == len(d["bfc"])
    if cyc is not None:
        for fcells, ci, cb, pnf in cyc:
            out.append(dict(faceCells=fcells, ic=ci, bc=cb, coupled=True, pnf=pnf))
    return out


@pytest.mark.parametrize("case", ["poisson", "momentum0", "cyclic"])
def test_fvmatrix_glue_matches_reference_code(meshmod, orc, case):
    """Row a17 for scalar fields: oracle/fvm_oracle.py against the reference's own fvMatrix.C / fvScalarMatrix.C
    (compiled for the host against oracle/ref_harness/shim_fvm/), bit for bit: boundary folding, setReference, relax, D, A,
    H, flux, residual and what solveSegregated hands to the linear solver.  `cyclic` adds a coupled patch pair."""
    import test_oracle_fvm as tf
    from oracle import fvm_oracle as fo
    from test_oracle_core import _cyclic_case
    rng = np.random.default_rng(12)
    cyc, kw = None, {}
    if case == "poisson":
        m, a, d = tf.poisson_case(meshmod, orc, (7, 6, 5))
    elif case == "momentum0":
        m, a, d3 = tf.momentum_case(meshmod, orc, (6, 5, 4))
        d = dict(d3, source=d3["source"][:, 0].copy(), ic=d3["ic"][:, :1].copy(), bc=d3["bc"][:, :1].copy())
    else:
        m, c, ps, fc, nr, lo, hi = _cyclic_case(meshmod, "U")
        wall = np.concatenate([p.faceCells for p in m.wall_patches() if p.name not in ("xmin", "xmax")]).astype(np.int32)
        ic, bc = fo.fixedValue_laplacian_coeffs(np.full(len(wall), 0.01 * m.h * m.h), np.full(len(wall), 2.0 / m.h),
                                                rng.uniform(-1, 1, (len(wall), 1)))
        diag = c["diag"].copy()
        np.subtract.at(diag, fc, c["int"])
        d = dict(diag=diag, upper=c["upper"], lower=c["lower"], source=rng.uniform(-1, 1, m.nCells) * m.h ** 3, bfc=wall,
                 ic=-ic, bc=-bc, V=m.volumes())
        a = orc.Addr(m.nCells, m.lower, m.upper, ps, fc, neighbRank=nr)
        kw = dict(couInt=c["int"], couBou=c["bou"])
    x = rng.uniform(-1, 1, (m.nCells, 1))
    mk = lambda: tf.make(orc, a, d, 1, x, **kw)
    if case == "cyclic":
        pnf = mk().patchNeighbourField()[:, 0]
        n = len(lo)
        cyc = [(lo, c["int"][:n], c["bou"][:n], pnf[:n]), (hi, c["int"][n:], c["bou"][n:], pnf[n:])]
    P = _fvm_patches(m, d, cyc)
    args = (m.nCells, m.lower, m.upper, P, d["V"], x[:, 0], d["diag"], d["upper"], d["lower"], np.ravel(d["source"]))
    R = lambda op, **k: ref_ldu.fvm(op, *args, **k)
    o = mk()
    for op, fn in (("addBoundaryDiag", lambda v: o.addBoundaryDiag(v, 0)), ("addCmptAvBoundaryDiag", o.addCmptAvBoundaryDiag)):
        v = d["diag"].copy()
        fn(v)
        assert np.array_equal(R(op, x=d["diag"]), v), op
    for couples in (0, 1):
        v = np.array(d["source"], float).reshape(-1, 1).copy()
        o.addBoundarySource(v, bool(couples))
        assert np.array_equal(R("addBoundarySource", x=np.ravel(d["source"]), iarg=couples), v[:, 0]), couples
    assert np.array_equal(R("D"), o.D()) and np.array_equal(R("A"), o.A())
    assert np.array_equal(R("H"), o.H()[:, 0])
    fi, fb = R("flux")
    oi, ob, oc = o.flux()
    assert np.array_equal(fi, oi[:, 0]) and np.array_equal(fb, np.concatenate([ob[:, 0], oc[:, 0]]))
    # (over the coupled patches this includes the neighbour term twice, as fvScalarMatrix.C:195-240 is written)
    assert np.array_equal(R("residual"), o.residual())
    for alpha in (1.0, 0.6):
        r = mk()
        r.relax(alpha)
        dg, sr = R("relax", darg=alpha)
        assert np.array_equal(dg, r.diag) and np.array_equal(sr, r.source[:, 0]), alpha
    r = mk()
    r.setReference(5, 0.75)
    dg, sr = R("setReference", iarg=5, darg=0.75)
    assert np.array_equal(dg, r.diag) and np.array_equal(sr, r.source[:, 0])
    # solveSegregated: the diagonal and the source the linear solver is handed, and the diagonal put back afterwards
    seenDiag, seenSource, after = R("solveSegregated")
    v = d["diag"].copy()
    o.addBoundaryDiag(v, 0)
    s = np.array(d["source"], float).reshape(-1, 1).copy()
    o.addBoundarySource(s, False)
    assert np.array_equal(seenDiag, v) and np.array_equal(seenSource, s[:, 0]) and np.array_equal(after, d["diag"])


@pytest.mark.parametrize("case", ["momentum", "cyclic"])
def test_vector_fvmatrix_glue_matches_reference_code(meshmod, orc, case):
    """Row a17 for vector fields: fvMatrix<vector> of the reference (fvMatrix.C, fvMatrixSolve.C compiled for the host)
    against oracle/fvm_oracle.py, bit for bit: component-wise boundary folding, the component average, relax with the
    largest / smallest component of the internal coefficients, H -- including the reference's loss of the boundary-diagonal
    term -- and the component loop of solveSegregated with the coupled source going in once and out per component."""
    import test_oracle_fvm as tf
    from oracle import fvm_oracle as fo
    from test_oracle_core import _cyclic_case
    rng = np.random.default_rng(13)
    cyc, kw = None, {}
    if case == "momentum":
        m, a, d = tf.momentum_case(meshmod, orc, (6, 5, 4))
        d = dict(d, ic=d["ic"] * np.array([1.0, 2.0, 3.0]))      # component-dependent internal coefficients
        walls = m.wall_patches()
    else:
        m, c, ps, fc, nr, lo, hi = _cyclic_case(meshmod, "U")
        walls = [p for p in m.wall_patches() if p.name not in ("xmin", "xmax")]
        wall = np.concatenate([p.faceCells for p in walls]).astype(np.int32)
        ic, bc = fo.fixedValue_laplacian_coeffs(np.full(len(wall), 0.01 * m.h * m.h), np.full(len(wall), 2.0 / m.h),
                                                rng.uniform(-1, 1, (len(wall), 3)))
        diag = c["diag"].copy()
        np.subtract.at(diag, fc, c["int"])
        d = dict(diag=diag, upper=c["upper"], lower=c["lower"], source=rng.uniform(-1, 1, (m.nCells, 3)) * m.h ** 3, bfc=wall,
                 ic=-ic * np.array([1.0, 0.5, 2.0]), bc=-bc, V=m.volumes())
        a = orc.Addr(m.nCells, m.lower, m.upper, ps, fc, neighbRank=nr)
        kw = dict(couInt=c["int"], couBou=c["bou"])
    x = rng.uniform(-1, 1, (m.nCells, 3))
    mk = lambda: tf.make(orc, a, d, 3, x, **kw)
    P, off = [], 0
    for p in walls:
        k = len(p.faceCells)
        P.append(dict(faceCells=p.faceCells, ic=d["ic"][off:off + k], bc=d["bc"][off:off + k]))
        off += k
    if case == "cyclic":
        pnf = mk().patchNeighbourField()
        n = len(lo)
        three = lambda v: np.repeat(v[:, None], 3, axis=1)       # the coupled coefficient of every component
        P += [dict(faceCells=lo, ic=three(c["int"][:n]), bc=three(c["bou"][:n]), coupled=True, pnf=pnf[:n]),
              dict(faceCells=hi, ic=three(c["int"][n:]), bc=three(c["bou"][n:]), coupled=True, pnf=pnf[n:])]
    args = (m.nCells, m.lower, m.upper, P, d["V"], x, d["diag"], d["upper"], d["lower"], d["source"])
    R = lambda op, **k: ref_ldu.fvm(op, *args, nc=3, **k)
    o = mk()
    for cmpt in range(3):
        v = d["diag"].copy()
        o.addBoundaryDiag(v, cmpt)
        assert np.array_equal(R("addBoundaryDiag", x=d["diag"], iarg=cmpt), v), cmpt
    v = d["diag"].copy()
    o.addCmptAvBoundaryDiag(v)
    assert np.array_equal(R("addCmptAvBoundaryDiag", x=d["diag"]), v)
    for couples in (0, 1):
        v = d["source"].copy()
        o.addBoundarySource(v, bool(couples))
        assert np.array_equal(R("addBoundarySource", x=d["source"], iarg=couples), v), couples
    assert np.array_equal(R("D"), o.D()) and np.array_equal(R("A"), o.A())
    # H: the reference's result is the oracle's default (the boundary-diagonal term of stock OpenFOAM is lost) ...
    Href = R("H")
    assert np.array_equal(Href, o.H())
    # ... and differs from the stock expression when the internal coefficients differ between components
    assert not np.allclose(Href, o.H(boundaryDiagInH=True))
    for alpha in (1.0, 0.6):
        r = mk()
        r.relax(alpha)
        dg, sr = R("relax", darg=alpha)
        assert np.array_equal(dg, r.diag) and np.array_equal(sr, r.source), alpha
    # the component loop: diagonals and sources the solver is handed, per component
    seenDiag, seenSource, after = R("solveSegregated")
    src = d["source"].copy()
    o.addBoundarySource(src, True)
    pn = o.patchNeighbourField() if case == "cyclic" else None
    for k in range(3):
        v = d["diag"].copy()
        o.addBoundaryDiag(v, k)
        sk = np.ascontiguousarray(src[:, k])
        if pn is not None:
            np.subtract.at(sk, o.cfc, o.couBou * pn[:, k])
        assert np.array_equal(seenDiag[k], v) and np.array_equal(seenSource[k], sk), k
    assert np.array_equal(after, d["diag"])


@pytest.mark.parametrize("gamg", [False, True])
@pytest.mark.parametrize("nR", [2, 4, 8])
@pytest.mark.parametrize("mode", [("nonBlocking", 0, False), ("nonBlocking", 1, True), ("blocking", 0, False)])
def test_processor_interface_exchange_matches_reference_code(meshmod, orc, nR, mode, gamg):
    """Row a6: the finest-level halo exchange + interface update of the reference -- lduMatrix::initMatrixInterfaces /
    updateMatrixInterfaces, processorFvPatchField<scalar>::initInterfaceMatrixUpdate / updateInterfaceMatrix with their
    send / receive buffers and requests, matrixPatchOperation -- all ranks in one process behind a Pstream mailbox, against
    the oracle's Amul of the decomposed case (threads): identical vectors on every rank, for the non-blocking (polling or
    not, direct or staged buffers) and the blocking communication types, and with the smoothers' negated sign.
    gamg: the same through processorGAMGInterfaceField + GAMGUpdateInterfaceMatrix, the coarse-level classes (row a14)."""
    import dist_helpers as dh
    n = 8
    gm, _ = dh.global_case(meshmod, n, "U")
    x = meshmod.cell_field_global(gm, 3)
    ex = dh.ThreadExchange(nR)

    def rank_fn(r):
        m, c = dh.local_case(meshmod, n, nR, r, "U")
        a, M = dh.oracle_matrix(orc, m, c)
        comm = ex.comm(orc, r, m, n ** 3)
        with_if = M.amul(x[m.cellGlobal], comm)
        a0 = orc.Addr(m.nCells, m.lower, m.upper)
        without = orc.Matrix(a0, c["diag"], c["upper"], c["lower"]).amul(x[m.cellGlobal])
        ps, fc = m.patch_start_facecells()
        return dict(nCells=m.nCells, patchStart=ps, faceCells=fc, neighbRank=[p.neighbRank for p in m.coupled_patches()],
                    coeffs=c["bou"], psi=x[m.cellGlobal], result=without), with_if, without
    res = dh.run_threads(nR, rank_fn)
    got = ref_ldu.processor_interface_update([r[0] for r in res], mode[0], False, mode[1], mode[2], gamg)
    for r in range(nR):
        assert np.array_equal(got[r], res[r][1]), r
        assert not np.array_equal(res[r][1], res[r][2])
    # negate = true (the smoothers): the term is added instead
    got = ref_ldu.processor_interface_update([r[0] for r in res], mode[0], True, mode[1], mode[2], gamg)
    for r in range(nR):
        d = res[r][0]
        expect = d["result"].copy()
        delta = res[r][1] - res[r][2]          # -(coeff*pnf) summed per cell by the oracle
        np.testing.assert_allclose(got[r], expect - delta, rtol=1e-14, atol=1e-15)


@pytest.mark.parametrize("kind", ["P", "U"])
def test_cyclic_interface_update_matches_reference_code(meshmod, orc, kind):
    """Cyclic patch pairs: cyclicFvPatchField<scalar>::updateInterfaceMatrix of the reference (cyclicFvPatchField.C:212-231 --
    psi gathered at the partner patch's face cells, then the coupled update) driven by lduMatrix::updateMatrixInterfaces,
    against the oracle's Amul / Tmul with the cyclic pairing (neighbRank = -(partner + 1))."""
    from test_oracle_core import _cyclic_case
    m, c, ps, fc, nr, lo, hi = _cyclic_case(meshmod, kind)
    a = orc.Addr(m.nCells, m.lower, m.upper, ps, fc, neighbRank=nr)
    M = orc.Matrix(a, c["diag"], c["upper"], c["lower"], c["bou"], c["int"])
    M0 = orc.Matrix(orc.Addr(m.nCells, m.lower, m.upper), c["diag"], c["upper"], c["lower"])
    x = np.random.default_rng(4).standard_normal(m.nCells)
    for coeffs, with_if, without in ((c["bou"], M.amul(x), M0.amul(x)), (c["int"], M.tmul(x), M0.tmul(x))):
        rank = dict(nCells=m.nCells, patchStart=ps, faceCells=fc, neighbRank=nr, coeffs=coeffs, psi=x, result=without)
        for mode in ("nonBlocking", "blocking"):
            got = ref_ldu.processor_interface_update([rank], mode)[0]
            assert np.array_equal(got, with_if) and not np.array_equal(with_if, without)


@pytest.mark.parametrize("nc", [1, 3])
def test_coefficient_fills_match_reference_schemes(meshmod, orc, nc):
    """Row a16, the matrix fills: gaussConvectionScheme::fvmDiv and gaussLaplacianScheme::fvmLaplacianUncorrected of the
    reference (compiled for the host) against the oracle's convection_fill / laplacian_fill and against the patch-coefficient
    expressions oracle/piso_oracle.py uses for fixedValue and coupled (processor) patches, bit for bit."""
    from oracle import fvm_oracle as fo
    m = meshmod.decompose(8, 2, 0)                       # walls + one processor patch
    a = orc.Addr(m.nCells, m.lower, m.upper)
    rng = np.random.default_rng(21)
    w, phi = rng.uniform(0.3, 0.7, m.nFaces), rng.uniform(-1, 1, m.nFaces)
    gamma, delta = rng.uniform(0.5, 1.5, m.nFaces), rng.uniform(5, 9, m.nFaces)
    P = []
    for p in m.patches:
        k = len(p.faceCells)
        d = dict(faceCells=p.faceCells, delta=rng.uniform(10, 20, k), pw=rng.uniform(0.3, 0.7, k), pphi=rng.uniform(-1, 1, k),
                 pgamma=rng.uniform(0.5, 1.5, k))
        if p.kind == "processor":
            d.update(kind="coupled")
        else:
            d.update(kind="fixedValue", value=rng.uniform(-1, 1, (k, nc)))
        P.append(d)
    one = np.ones((1, nc))
    # fvm::div
    got = ref_ldu.fvm_fill("div", nc, m.nCells, m.lower, m.upper, [dict(p, a=p["pw"], b=p["pphi"]) for p in P], w, phi)
    lo, up, dg = orc.convection_fill(a, w, phi)
    assert np.array_equal(got["lower"], lo) and np.array_equal(got["upper"], up) and np.array_equal(got["diag"], dg)
    ic, bc = [], []
    for p in P:
        f = p["pphi"][:, None]
        if p["kind"] == "coupled":       # oracle/piso_oracle.py: cCi = cphi*cw, cCb = (-cphi)*(1 - cw)
            ic.append((p["pphi"] * p["pw"])[:, None] * one)
            bc.append(((-p["pphi"]) * (1.0 - p["pw"]))[:, None] * one)
        else:                            # cIc = 0, cBc = (-bphi)*Ub
            ic.append(f * np.zeros_like(p["value"]))
            bc.append((-f) * p["value"])
    assert np.array_equal(got["ic"], np.concatenate(ic)) and np.array_equal(got["bc"], np.concatenate(bc))
    # fvm::laplacian (uncorrected)
    gms = gamma * 0.01
    got = ref_ldu.fvm_fill("laplacian", nc, m.nCells, m.lower, m.upper, [dict(p, a=p["pgamma"], b=p["delta"]) for p in P], gms, delta)
    up, dg = orc.laplacian_fill(a, delta, gms)
    assert np.array_equal(got["upper"], up) and np.array_equal(got["diag"], dg)
    ic, bc = [], []
    for p in P:
        if p["kind"] == "coupled":       # lCi = cGamma*(-cDelta), lCb = (-cGamma)*cDelta
            ic.append((p["pgamma"] * (-p["delta"]))[:, None] * one)
            bc.append(((-p["pgamma"]) * p["delta"])[:, None] * one)
        else:
            i, b = fo.fixedValue_laplacian_coeffs(p["pgamma"], p["delta"], p["value"])
            ic.append(i)
            bc.append(b)
    assert np.array_equal(got["ic"], np.concatenate(ic)) and np.array_equal(got["bc"], np.concatenate(bc))


def test_euler_ddt_terms_match_reference_schemes(meshmod, orc):
    """The time-derivative pieces of the PISO step (§8 f2): EulerDdtScheme<vector>::fvmDdt, ::fvcDdtPhiCorr and
    ddtScheme::fvcDdtPhiCoeff of the reference (compiled for the host) against the expressions oracle/piso_oracle.py composes
    (ddtDiag, ddtSource, phiCorr, coeff, ddtCorr), bit for bit.  Patches that fix the value get a zero coefficient
    (ddtScheme.C:156-162); the others keep the face expression, which is what the oracle applies on processor faces."""
    m = meshmod.decompose(8, 2, 0)
    rng = np.random.default_rng(33)
    n, nF = m.nCells, m.nFaces
    V = rng.uniform(0.5, 1.5, n) * 1e-3
    U0 = rng.uniform(-1, 1, (n, 3))
    Sf = rng.uniform(-1, 1, (nF, 3)) * 1e-2
    w = rng.uniform(0.3, 0.7, nF)
    phi0 = rng.uniform(-1, 1, nF) * 1e-2
    phi0[::7] = 0.0                                      # faces without flux: the SMALL in the coefficient's denominator
    deltaT = 0.005
    P = []
    for k, p in enumerate(m.patches):
        f = len(p.faceCells)
        P.append(dict(faceCells=p.faceCells, fixesValue=(p.kind != "processor"), value=rng.uniform(-1, 1, (f, 3)),
                      phi0=rng.uniform(-1, 1, f) * 1e-2, Sf=rng.uniform(-1, 1, (f, 3)) * 1e-2))
    got = ref_ldu.euler_ddt(n, m.lower, m.upper, P, deltaT, V, U0, phi0, Sf, w)
    # oracle/piso_oracle.py Cavity.step, the same statements
    SMALL = 1e-15
    rDeltaT = 1.0 / deltaT
    dot = lambda a, b: (a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1]) + a[:, 2] * b[:, 2]
    assert np.array_equal(got["diag"], rDeltaT * V)
    assert np.array_equal(got["source"], (rDeltaT * U0) * V[:, None])
    l, u = np.asarray(m.lower), np.asarray(m.upper)
    Uf = w[:, None] * (U0[l] - U0[u]) + U0[u]            # surfaceInterpolationScheme.C:323-326
    phiCorr = phi0 - dot(Sf, Uf)
    coeff = 1.0 - np.minimum(np.abs(phiCorr) / (np.abs(phi0) + SMALL), 1.0)
    assert np.array_equal(got["ddtCorr"], (coeff * rDeltaT) * phiCorr)
    b = []
    for p in P:
        if p["fixesValue"]:
            b.append(np.zeros(len(p["faceCells"])))
        else:
            pc = p["phi0"] - dot(p["Sf"], p["value"])
            cc = 1.0 - np.minimum(np.abs(pc) / (np.abs(p["phi0"]) + SMALL), 1.0)
            b.append((cc * rDeltaT) * pc)
    assert np.array_equal(got["bddtCorr"], np.concatenate(b))


@pytest.mark.parametrize("nc", [1, 3])
def test_linear_interpolation_matches_reference_scheme(meshmod, orc, nc):
    """The face interpolation inside the face-sum kernels (row a16) and the PISO step: the reference's
    surfaceInterpolationScheme<Type>::interpolate(vf) (compiled for the host; one-weight form w*(own - nei) + nei on internal
    faces, w*patchInternalField + (1 - w)*patchNeighbourField on coupled patches, the patch value elsewhere) against
    orc_interpolate_linear and the coupled-face expression of oracle/piso_oracle.py, bit for bit."""
    m = meshmod.decompose(8, 2, 0)
    a = orc.Addr(m.nCells, m.lower, m.upper)
    rng = np.random.default_rng(5 + nc)
    shape = (lambda k: (k,)) if nc == 1 else (lambda k: (k, nc))
    w = rng.uniform(0.2, 0.8, m.nFaces)
    vf = rng.uniform(-1, 1, shape(m.nCells)) * 10.0 ** rng.integers(-3, 3, shape(m.nCells))
    P = []
    for p in m.patches:
        k = len(p.faceCells)
        P.append(dict(faceCells=p.faceCells, coupled=(p.kind == "processor"), w=rng.uniform(0.2, 0.8, k),
                      value=rng.uniform(-1, 1, (k, nc)), pnf=rng.uniform(-1, 1, (k, nc))))
    got, bgot = ref_ldu.interpolate_linear(nc, m.nCells, m.lower, m.upper, P, w, vf)
    assert np.array_equal(got, orc.interpolate_linear(a, w, vf, nc))
    exp = []
    for p in P:
        if p["coupled"]:     # oracle/piso_oracle.py interpolate_coupled
            pw = p["w"][:, None]
            exp.append(pw * vf.reshape(m.nCells, nc)[p["faceCells"]] + (1 - pw) * p["pnf"])
        else:
            exp.append(p["value"])
    assert np.array_equal(bgot.reshape(-1, nc), np.concatenate(exp))
    # the two-weight form differs in the last bit on some faces: the distinction is observable
    two = (w if nc == 1 else w[:, None]) * vf[np.asarray(m.lower)] + (1 - (w if nc == 1 else w[:, None])) * vf[np.asarray(m.upper)]
    assert not np.array_equal(two, got) and np.allclose(two, got, rtol=1e-13, atol=1e-15)


def test_matrix_algebra_matches_reference_operators(meshmod, orc):
    """The combination that forms icoFoam's momentum matrix (fvm::ddt + fvm::div - fvm::laplacian): the reference's
    lduMatrix::operator+= / operator-= (lduMatrixOperations.C, compiled for the host) against the assembly statements of
    oracle/piso_oracle.py -- a diagonal matrix += an asymmetric one takes its triangles, -= a symmetric one subtracts its
    upper from both triangles -- and the pressure matrix (symmetric only), bit for bit."""
    m = meshmod.hex_mesh(6, 5, 4)
    a = orc.Addr(m.nCells, m.lower, m.upper)
    rng = np.random.default_rng(77)
    V = rng.uniform(0.5, 1.5, m.nCells) * 1e-3
    ddtDiag = (1.0 / 0.005) * V
    cLower, cUpper, cDiag = orc.convection_fill(a, rng.uniform(0.3, 0.7, m.nFaces), rng.uniform(-1, 1, m.nFaces) * 1e-2)
    lUpper, lDiag = orc.laplacian_fill(a, rng.uniform(5, 9, m.nFaces), rng.uniform(0.5, 1.5, m.nFaces) * 1e-3)
    got = ref_ldu.ldu_combine(m.nCells, m.lower, m.upper, dict(diag=ddtDiag), +1, dict(diag=cDiag, upper=cUpper, lower=cLower), -1,
                              dict(diag=lDiag, upper=lUpper))
    # oracle/piso_oracle.py Cavity.step: diag = (ddtDiag + cDiag) - lDiag; upper = cUpper - lUpper; lower = cLower - lUpper
    assert sorted(got) == ["diag", "lower", "upper"]
    assert np.array_equal(got["diag"], (ddtDiag + cDiag) - lDiag)
    assert np.array_equal(got["upper"], cUpper - lUpper)
    assert np.array_equal(got["lower"], cLower - lUpper)
    # symmetric with symmetric stays symmetric (the pressure equation's single laplacian; also a sum of two)
    got = ref_ldu.ldu_combine(m.nCells, m.lower, m.upper, dict(diag=lDiag, upper=lUpper), +1, dict(diag=lDiag * 0.5, upper=lUpper * 0.5))
    assert sorted(got) == ["diag", "upper"]
    assert np.array_equal(got["diag"], lDiag + lDiag * 0.5) and np.array_equal(got["upper"], lUpper + lUpper * 0.5)
    # symmetric -= asymmetric: the missing lower starts as a copy of the upper (lduMatrix.C:219-235)
    got = ref_ldu.ldu_combine(m.nCells, m.lower, m.upper, dict(diag=lDiag, upper=lUpper), -1, dict(diag=cDiag, upper=cUpper, lower=cLower))
    assert np.array_equal(got["upper"], lUpper - cUpper) and np.array_equal(got["lower"], lUpper - cLower)
    assert np.array_equal(got["diag"], lDiag - cDiag)


def test_momentum_equation_assembly_matches_reference_operators(meshmod, orc):
    """UEqn of icoFoam.C:57-64, `fvm::ddt(U) + fvm::div(phi, U) - fvm::laplacian(nu, U)` and `UEqn == -fvc::grad(p)`: the
    reference's fvMatrix operators (fvMatrix.C operator+ / operator- / operator== with a field / operator+= / -=, compiled for
    the host) against the assembly statements of oracle/piso_oracle.py (coefficients, source + V*su, internal / boundary
    coefficients of the patches), bit for bit."""
    m = meshmod.decompose(8, 2, 0)
    a = orc.Addr(m.nCells, m.lower, m.upper)
    rng = np.random.default_rng(99)
    n, nF = m.nCells, m.nFaces
    V = rng.uniform(0.5, 1.5, n) * 1e-3
    ddtDiag, ddtSource = 200.0 * V, (200.0 * rng.uniform(-1, 1, (n, 3))) * V[:, None]
    cLower, cUpper, cDiag = orc.convection_fill(a, rng.uniform(0.3, 0.7, nF), rng.uniform(-1, 1, nF) * 1e-2)
    lUpper, lDiag = orc.laplacian_fill(a, rng.uniform(5, 9, nF), rng.uniform(0.5, 1.5, nF) * 1e-3)
    patches = [p.faceCells for p in m.patches]
    tot = sum(len(p) for p in patches)
    cIc, cBc, lIc, lBc = (rng.uniform(-1, 1, (tot, 3)) for _ in range(4))
    su = rng.uniform(-1, 1, (n, 3))      # -fvc::grad(p)
    got = ref_ldu.fvm_assemble(n, m.lower, m.upper, patches, V, dict(diag=ddtDiag, source=ddtSource),
                               dict(diag=cDiag, upper=cUpper, lower=cLower, ic=cIc, bc=cBc), dict(diag=lDiag, upper=lUpper, ic=lIc, bc=lBc), su)
    assert got["kind"] == "asymmetric"
    # oracle/piso_oracle.py Cavity.step
    assert np.array_equal(got["diag"], (ddtDiag + cDiag) - lDiag)
    assert np.array_equal(got["upper"], cUpper - lUpper) and np.array_equal(got["lower"], cLower - lUpper)
    assert np.array_equal(got["source"], ddtSource + V[:, None] * su)
    assert np.array_equal(got["ic"], cIc - lIc) and np.array_equal(got["bc"], cBc - lBc)
