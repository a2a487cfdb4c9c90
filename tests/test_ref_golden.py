"""tests/golden/ref_golden.npz was produced by EXECUTING THE REFERENCE'S OWN SOURCE (make_ref_golden.py:
oracle/_ref harness only, no oracle).  These tests hold the oracle -- and, on a GPU, the CUDA path --
against those vectors; they run wherever the .npz is, with or without /root/reference.

Tolerances: row sums and smoothing on the hex mesh are compared bit for bit; the GAMG solve to rounding
level (coarse cells exceed three faces per side, where oracle and reference associate the row sum
differently); the Krylov solvers to 1e-11 over the stored iterations (the reference's vector updates were
compiled unfused for the host, oracle and kernels use the FMAs nvcc generates for them)."""
import importlib
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import make_ref_golden as mrg  # noqa: E402


@pytest.fixture(scope="module")
def ref_golden():
    return np.load(os.path.join(HERE, "golden", "ref_golden.npz"))


def _oracle(meshmod, orc, dims, kind):
    m, c = mrg.coefficients(meshmod, dims, kind)
    a = orc.Addr(m.nCells, m.lower, m.upper)
    return m, c, a, orc.Matrix(a, c["diag"], c["upper"], c["lower"])


def test_fixture_is_reproducible_where_the_reference_is_present(meshmod, ref_golden):
    import ref_replay
    from oracle import ref_ldu
    ref_replay.install()   # the reference's answers come from tests/golden/ref_calls_*.npz
    fresh = mrg.generate(meshmod, ref_ldu)
    assert sorted(fresh) == sorted(ref_golden.files)
    for k in ref_golden.files:
        assert np.array_equal(fresh[k], ref_golden[k]), k


@pytest.mark.parametrize("name,dims,kind", mrg.OPS_CASES)
def test_oracle_matrix_ops_vs_reference_vectors(meshmod, orc, ref_golden, name, dims, kind):
    m, c, a, M = _oracle(meshmod, orc, dims, kind)
    x, b = meshmod.cell_field_global(m, 3), meshmod.cell_field_global(m, 4)
    G = lambda k: ref_golden[f"{name}.{k}"]
    assert np.array_equal(M.amul(x), G("amul")) and np.array_equal(M.tmul(x), G("tmul"))
    assert np.array_equal(M.H(x), G("H")) and np.array_equal(M.faceH(x), G("faceH"))
    assert np.array_equal(M.sumA(), G("sumA")) and np.array_equal(M.H1(), G("H1"))
    assert np.array_equal(M.residual(x, b), G("residual"))
    for T in (False, True):
        assert np.array_equal(M.precondition("DIC", x, T), G(f"ainv.{int(T)}"))
    assert np.array_equal(M.jacobi(x, b, 1), G("jacobi1"))


@pytest.mark.parametrize("name,dims", mrg.FV_CASES)
def test_oracle_fv_face_sums_vs_reference_vectors(meshmod, orc, ref_golden, name, dims):
    m, d = mrg.fv_inputs(meshmod, dims)
    a = orc.Addr(m.nCells, m.lower, m.upper)
    G = lambda k: ref_golden[f"{name}.{k}"]
    assert np.array_equal(orc.surface_integrate(a, d["ssf"], d["bfc"], d["bssf"], d["V"], 1), G("integrate"))
    assert np.array_equal(orc.surface_integrate(a, d["ssf"], d["bfc"], d["bssf"], d["V"], 1, False, +1), G("sum"))
    g = orc.gauss_grad(a, d["Sf"].ravel(), d["ssf"], d["bfc"], d["bSf"].ravel(), d["bssf"], d["V"], 1)
    assert np.array_equal(np.asarray(g).reshape(-1, 3), G("grad"))


@pytest.mark.parametrize("name,dims,kind,solver,pre,ctl", mrg.SOLVE_CASES)
def test_oracle_solvers_vs_reference_vectors(meshmod, orc, ref_golden, name, dims, kind, solver, pre, ctl):
    m, c, a, M = _oracle(meshmod, orc, dims, kind)
    b = M.amul(meshmod.cell_field_global(m, 42))
    quirk = 1 if solver == "PBiCGStab" else 0     # the stored solution is the reference's (PBiCGStab.C:263-270)
    psi, perf, hist = M.solve(solver, pre, np.zeros(m.nCells), b, bicgstabRefQuirk=quirk, **ctl)
    gp = ref_golden[f"{name}.perf"]
    assert perf.nIterations == int(gp[0]) and perf.converged == int(gp[1])
    assert perf.initialResidual == gp[2]
    gh = ref_golden[f"{name}.hist"]
    k = min(len(gh), len(hist) - 1)
    if solver == "PBiCGStab":
        k = min(k, len(hist) - 2)   # its last iteration leaves through the mid-body test on sA (PBiCGStab.C:219-232)
    if solver == "smoothSolver":
        assert np.array_equal(hist[1:k + 1], gh[:k]) and np.array_equal(psi, ref_golden[f"{name}.psi"])
        assert perf.finalResidual == gp[3]
    else:
        np.testing.assert_allclose(hist[1:k + 1], gh[:k], rtol=1e-11, atol=0)
        np.testing.assert_allclose(psi, ref_golden[f"{name}.psi"], rtol=0, atol=1e-8)


@pytest.mark.parametrize("name,dims,kind,ctl", mrg.GAMG_CASES)
def test_oracle_gamg_vs_reference_vectors(meshmod, orc, ref_golden, name, dims, kind, ctl):
    """hierarchy (pairing, coarse addressing, coarse diagonals) and cycle history of a GAMG solve produced
    end to end by reference code"""
    m, c, a, M = _oracle(meshmod, orc, dims, kind)
    g = orc.Gamg(a, meshmod.face_area_pair_weights(m), 10)
    lv = ref_golden[f"{name}.levels"]
    assert g.nLevels == len(lv) and g.forward == int(ref_golden[f"{name}.forward"][0])
    for k in range(g.nLevels):
        assert (g.ncells(k), g.nfaces(k)) == tuple(int(v) for v in lv[k])
    from oracle import ref_ldu
    D, U, L = c["diag"], c["upper"], c["lower"]
    for k in range(min(g.nLevels, 3)):
        assert np.array_equal(g.restrict_addr(k), ref_golden[f"{name}.restrict{k}"])
        assert np.array_equal(g.level_addr(k).upper(), ref_golden[f"{name}.coarseUpperAddr{k}"])
        D, U, L = ref_ldu.coarse_matrix(g.restrict_addr(k), g.face_restrict_addr(k), g.face_flip(k), g.ncells(k),
                                        g.nfaces(k), D, U, L)
        assert np.array_equal(D, ref_golden[f"{name}.coarseDiag{k}"])
    b = M.amul(meshmod.cell_field_global(m, 42))
    psi, perf, hist = g.solve(M, "GaussSeidel", np.zeros(m.nCells), b, **ctl)
    # Coarse levels have cells with more than three faces on one side: there the reference's unrolled row
    # sum adds the first three neighbour-side products before the fourth owner-side one (JacobiSmootherF.H
    # :66-106), the oracle adds in plain row order -- same terms, different association (DESIGN.md section 2).
    # Hence rounding-level tolerances here; tests/test_reference_functors.py has the bit-exact V-cycle
    # comparison on a hierarchy that stays within three faces per side.
    gp = ref_golden[f"{name}.perf"]
    assert perf.nIterations == int(gp[0]) and perf.initialResidual == gp[2]
    assert abs(perf.finalResidual - gp[3]) <= 1e-7 * gp[3]
    gh = ref_golden[f"{name}.hist"]
    np.testing.assert_allclose(hist[1:len(gh) + 1], gh, rtol=1e-10, atol=0)
    np.testing.assert_allclose(psi, ref_golden[f"{name}.psi"], rtol=0, atol=1e-11)


# ---------------------------------------------------------------------------------------------------------
# CUDA path against the reference-generated vectors
# ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gpu():
    if os.environ.get("B200LDU_DRYRUN_ORACLE") == "1":   # CPU dry run of the tests' own logic: tests/oracle_backend.py
        import oracle_backend
        yield oracle_backend.fixture()
        return
    import torch
    assert torch.cuda.is_available()
    capi = importlib.import_module("rapidcfd-dev_b200.capi")
    ctx = capi.Context(0)
    yield capi, ctx, torch
    ctx.close()


def _device(gpu, meshmod, dims, kind):
    capi, ctx, torch = gpu
    m, c = mrg.coefficients(meshmod, dims, kind)
    addr = capi.mesh_to_device(ctx, m)
    mat = capi.LduMatrix(addr)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(ctx.device)
    mat.set(t(c["diag"]), t(c["upper"]), t(c["lower"]) if c["lower"] is not None else None)
    return m, c, addr, mat, t


@pytest.mark.gpu
@pytest.mark.parametrize("name,dims,kind", mrg.OPS_CASES)
def test_gpu_matrix_ops_vs_reference_vectors(gpu, meshmod, ref_golden, name, dims, kind):
    m, c, addr, mat, t = _device(gpu, meshmod, dims, kind)
    x, b = meshmod.cell_field_global(m, 3), meshmod.cell_field_global(m, 4)
    xd, bd = t(x), t(b)
    G = lambda k: ref_golden[f"{name}.{k}"]
    assert np.array_equal(mat.Amul(xd).cpu().numpy(), G("amul"))
    assert np.array_equal(mat.Tmul(xd).cpu().numpy(), G("tmul"))
    assert np.array_equal(mat.sumA(xd).cpu().numpy(), G("sumA"))
    assert np.array_equal(mat.residual(xd, bd).cpu().numpy(), G("residual"))
    assert np.array_equal(mat.H(xd).cpu().numpy(), G("H"))
    assert np.array_equal(mat.H1(xd).cpu().numpy(), G("H1"))
    assert np.array_equal(mat.faceH(xd).cpu().numpy(), G("faceH"))
    assert np.array_equal(mat.smooth("GaussSeidel", xd, bd, 1).cpu().numpy(), G("jacobi1"))
    for T in (False, True):   # the kernel stages rD*r: one rounding per term apart (DESIGN.md section 2)
        ref = G(f"ainv.{int(T)}")
        np.testing.assert_allclose(mat.precondition("DIC", xd, T).cpu().numpy(), ref, rtol=1e-13,
                                   atol=1e-13 * np.abs(ref).max())
    mat.close()
    addr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name,dims", mrg.FV_CASES)
def test_gpu_fv_face_sums_vs_reference_vectors(gpu, meshmod, ref_golden, name, dims):
    capi, ctx, torch = gpu
    if not hasattr(capi, "lib"):
        pytest.skip("raw C-ABI calls: not covered by the dry-run stand-in")
    m, d = mrg.fv_inputs(meshmod, dims)
    addr = capi.mesh_to_device(ctx, m)
    L, dp = capi.lib(), capi._dp
    capi.check(L.b200ldu_fv_boundary_set(addr.h, len(d["bfc"]), d["bfc"].ctypes.data))
    T = {k: torch.from_numpy(np.ascontiguousarray(v).ravel()).to(ctx.device) for k, v in d.items() if k != "bfc"}
    G = lambda k: ref_golden[f"{name}.{k}"]
    out = torch.empty(m.nCells, dtype=torch.float64, device=ctx.device)
    for div, sign, key in ((1, -1, "integrate"), (0, 1, "sum")):
        capi.check(L.b200ldu_fv_surface_integrate(addr.h, 1, dp(T["ssf"]), dp(T["bssf"]), dp(T["V"]), dp(out), div, sign))
        assert np.array_equal(out.cpu().numpy(), G(key)), key
    grad = torch.empty(m.nCells * 3, dtype=torch.float64, device=ctx.device)
    capi.check(L.b200ldu_fv_gauss_grad(addr.h, 1, dp(T["Sf"]), dp(T["ssf"]), dp(T["bSf"]), dp(T["bssf"]), dp(T["V"]),
                                       dp(grad)))
    assert np.array_equal(grad.cpu().numpy().reshape(-1, 3), G("grad"))
    addr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name,dims,kind,solver,pre,ctl", mrg.SOLVE_CASES)
def test_gpu_solvers_vs_reference_vectors(gpu, meshmod, orc, ref_golden, name, dims, kind, solver, pre, ctl):
    capi, ctx, torch = gpu
    m, c, addr, mat, t = _device(gpu, meshmod, dims, kind)
    oa = orc.Addr(m.nCells, m.lower, m.upper)
    b = orc.Matrix(oa, c["diag"], c["upper"], c["lower"]).amul(meshmod.cell_field_global(m, 42))  # rhs only
    psi = torch.zeros(m.nCells, dtype=torch.float64, device=ctx.device)
    quirk = 1 if solver == "PBiCGStab" else 0
    perf, hist = mat.solve(solver, pre, psi, t(b), histCap=1024, bicgstabRefQuirk=quirk, **ctl)
    gp, gh = ref_golden[f"{name}.perf"], ref_golden[f"{name}.hist"]
    assert abs(perf.nIterations - int(gp[0])) <= 1 and perf.converged == int(gp[1])
    assert abs(perf.initialResidual - gp[2]) <= 1e-12 * gp[2]
    k = min(len(gh), len(hist) - 1, 10 if solver.startswith("PBiCG") else 12)
    if solver == "PBiCGStab":
        k = min(k, len(hist) - 2)   # see the oracle test above
    # 1e-9 while the residual is above 1e-8 (below it the bi-conjugate recurrences are rounding noise on both sides)
    np.testing.assert_allclose(hist[1:k + 1], gh[:k], rtol=1e-9, atol=1e-17 if not solver.startswith("PBiCG") else 1e-17)
    np.testing.assert_allclose(psi.cpu().numpy(), ref_golden[f"{name}.psi"], rtol=0, atol=5e-6)
    mat.close()
    addr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name,dims,kind,ctl", mrg.GAMG_CASES)
def test_gpu_gamg_vs_reference_vectors(gpu, meshmod, orc, ref_golden, name, dims, kind, ctl):
    capi, ctx, torch = gpu
    m, c, addr, mat, t = _device(gpu, meshmod, dims, kind)
    gg = capi.GamgAgglomeration(addr, meshmod.face_area_pair_weights(m), 10)
    lv = ref_golden[f"{name}.levels"]
    assert gg.nLevels == len(lv) and gg.forward == int(ref_golden[f"{name}.forward"][0])
    for k in range(gg.nLevels):
        assert gg.level_size(k) == tuple(int(v) for v in lv[k])
    for k in range(min(gg.nLevels, 3)):
        assert np.array_equal(gg.restrict_addr(k), ref_golden[f"{name}.restrict{k}"])
    oa = orc.Addr(m.nCells, m.lower, m.upper)
    b = orc.Matrix(oa, c["diag"], c["upper"], c["lower"]).amul(meshmod.cell_field_global(m, 42))
    psi = torch.zeros(m.nCells, dtype=torch.float64, device=ctx.device)
    perf, hist = mat.solve("GAMG", "GaussSeidel", psi, t(b), gamg=gg, histCap=256, **ctl)
    gp, gh = ref_golden[f"{name}.perf"], ref_golden[f"{name}.hist"]
    assert perf.nIterations == int(gp[0])
    # kernels vs oracle: rel 1e-8 per cycle (tests/test_gpu_gamg.py); oracle vs reference: rounding level (above)
    np.testing.assert_allclose(hist[1:len(gh) + 1], gh, rtol=1e-7)
    np.testing.assert_allclose(psi.cpu().numpy(), ref_golden[f"{name}.psi"], rtol=0, atol=1e-8)
    gg.close()
    mat.close()
    addr.close()
