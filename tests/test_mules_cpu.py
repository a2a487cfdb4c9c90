"""Explicit MULES (SURVEY.md section 8(f) rank 4): the oracle against the reference's own MULESTemplates.C compiled here
(oracle/_ref/libref_mules.so: limiter, limit, explicitSolve with the reference's one / zero field algebra), the device code
of csrc/mules_kernels.cuh executed on the host against the oracle, and the sequencing of rapidcfd-dev_b200/mules.py over
the oracle-backed stand-in -- all bit for bit; then what the limiter is for: a bounded, conservative update."""
import ctypes as C
import importlib

import numpy as np
import pytest

import ref_replay
from oracle import mules_oracle as mo
from test_host_kernels_cpu import Host, _d, hk  # noqa: F401  (fixture: the host build of the kernels)

ref_replay.install()   # the reference's answers come from tests/golden/ref_calls_*.npz

COMBOS = ["one-zero", "rho", "SpSu", "rho-SpSu"]


def case(meshmod, dims=(7, 5, 4), seed=1, combo="one-zero", scale=1e-3):
    m = meshmod.hex_mesh(*dims)
    ps, bfc = m.patch_start_facecells(m.wall_patches())
    rng = np.random.default_rng(seed)
    n, nF, nB = m.nCells, m.nFaces, len(bfc)
    d = dict(m=m, ps=ps, bfc=bfc, n=n, nF=nF, nB=nB, rDeltaT=50.0)
    d["V"] = m.volumes() * rng.uniform(0.8, 1.2, n)
    d["psi"] = rng.uniform(0, 1, n)
    d["psi"][: n // 5] = 1.0                       # saturated cells: no room upwards
    d["psi"][n // 5: n // 3] = 0.0
    d["psi0"] = d["psi"].copy()
    d["psiB"] = rng.uniform(0, 1, nB)
    d["phi"], d["phiB"] = rng.uniform(-1, 1, nF) * scale, rng.uniform(-1, 1, nB) * scale
    d["phiB"][: nB // 3] = 0.0                     # walls
    d["phi"][::13] = 0.0                           # pos(0) = 1; phiCorr = 0 goes down the `else` branches
    d["phiPsi"] = d["phi"] * (0.5 * (d["psi"][m.lower] + d["psi"][m.upper]))        # central: unbounded
    d["phiPsiB"] = d["phiB"] * d["psiB"]
    kw = {}
    if "rho" in combo:
        kw.update(rho=rng.uniform(0.9, 1.1, n), rho0=rng.uniform(0.9, 1.1, n))
    if "SpSu" in combo:
        kw.update(Sp=-rng.uniform(0, 1, n), Su=rng.uniform(0, 0.1, n))
    d["kw"] = kw
    return d


def _cat(a, b):
    return np.concatenate([a, b])


@pytest.mark.parametrize("combo", COMBOS)
@pytest.mark.parametrize("nIter", [0, 1, 3])
def test_oracle_matches_the_reference_mules(meshmod, combo, nIter):
    d = case(meshmod, combo=combo, seed=2 + nIter)
    m, kw = d["m"], d["kw"]
    bd, bdB = mo.upwind_flux(m.lower, m.upper, d["phi"], d["phiB"], d["psi"], d["psiB"])
    corr, corrB = d["phiPsi"] - bd, d["phiPsiB"] - bdB
    lam, lamB = mo.limiter(d["n"], m.lower, m.upper, d["bfc"], d["V"], d["rDeltaT"], d["psi"], d["psi0"], d["psiB"], bd, bdB, corr,
                           corrB, 1.0, 0.0, nIter, **kw)
    ref = mo.reference(0, d["n"], m.lower, m.upper, d["ps"], d["bfc"], d["V"], d["rDeltaT"], d["psi"], d["psi0"], d["psiB"],
                       _cat(bd, bdB), _cat(corr, corrB), 1.0, 0.0, nIter, **kw)
    assert np.array_equal(_cat(lam, lamB), ref)
    assert nIter == 0 or (lam < 1).sum() > d["nF"] // 4          # the limiter is active on this case
    lp, lpB = mo.limit(d["n"], m.lower, m.upper, d["bfc"], d["V"], d["rDeltaT"], d["psi"], d["psi0"], d["psiB"], d["phi"], d["phiB"],
                       d["phiPsi"], d["phiPsiB"], 1.0, 0.0, nIter, **kw)
    ref = mo.reference(1, d["n"], m.lower, m.upper, d["ps"], d["bfc"], d["V"], d["rDeltaT"], d["psi"], d["psi0"], d["psiB"],
                       _cat(d["phi"], d["phiB"]), _cat(d["phiPsi"], d["phiPsiB"]), 1.0, 0.0, nIter, **kw)
    assert np.array_equal(_cat(lp, lpB), ref)
    new = mo.explicit_solve(d["n"], m.lower, m.upper, d["bfc"], d["V"], d["rDeltaT"], d["psi0"], lp, lpB, **kw)
    ref = mo.reference(2, d["n"], m.lower, m.upper, d["ps"], d["bfc"], d["V"], d["rDeltaT"], d["psi"], d["psi0"], d["psiB"],
                       _cat(lp, lpB), None, **kw)
    assert np.array_equal(new, ref)


def test_oracle_matches_the_reference_other_bounds(meshmod):
    """psiMax / psiMin that cut into the field (the local extrema are clipped to them)"""
    d = case(meshmod, (5, 6, 3), seed=9)
    m = d["m"]
    bd, bdB = mo.upwind_flux(m.lower, m.upper, d["phi"], d["phiB"], d["psi"], d["psiB"])
    corr, corrB = d["phiPsi"] - bd, d["phiPsiB"] - bdB
    lam, lamB = mo.limiter(d["n"], m.lower, m.upper, d["bfc"], d["V"], d["rDeltaT"], d["psi"], d["psi0"], d["psiB"], bd, bdB, corr,
                           corrB, 0.8, 0.3, 2)
    ref = mo.reference(0, d["n"], m.lower, m.upper, d["ps"], d["bfc"], d["V"], d["rDeltaT"], d["psi"], d["psi0"], d["psiB"],
                       _cat(bd, bdB), _cat(corr, corrB), 0.8, 0.3, 2)
    assert np.array_equal(_cat(lam, lamB), ref)


@pytest.mark.parametrize("combo", COMBOS)
def test_device_mules_code_on_the_host(hk, meshmod, orc, combo):  # noqa: F811
    d = case(meshmod, (6, 7, 5), seed=4, combo=combo)
    m, kw, n, nF, nB = d["m"], d["kw"], d["n"], d["nF"], d["nB"]
    a = orc.Addr(n, m.lower, m.upper)
    H = Host(a, dict(bfc=d["bfc"], diag=np.zeros(n), upper=np.zeros(nF), lower=None))
    bd, bdB = mo.upwind_flux(m.lower, m.upper, d["phi"], d["phiB"], d["psi"], d["psiB"])
    corr, corrB = d["phiPsi"] - bd, d["phiPsiB"] - bdB
    f = lambda x: None if x is None else np.ascontiguousarray(x, np.float64)
    arrs = {k: f(v) for k, v in dict(psi=d["psi"], psi0=d["psi0"], psiB=d["psiB"], bd=bd, bdB=bdB, corr=corr, corrB=corrB, V=d["V"],
                                     rho=kw.get("rho"), rho0=kw.get("rho0"), Sp=kw.get("Sp"), Su=kw.get("Su")).items()}
    for nIter in (0, 2, 3):
        lam, lamB, scratch = np.ones(nF), np.ones(nB), np.zeros(6 * n)
        hk.hk_mules_limiter.argtypes = [C.c_void_p, C.c_int, C.c_double] + [C.c_void_p] * 12 + [C.c_double, C.c_double] + [C.c_void_p] * 3 + [C.c_int, C.c_int, C.c_double]
        hk.hk_mules_limiter(H.p(), nIter, d["rDeltaT"], _d(arrs["rho"]), _d(arrs["rho0"]), _d(arrs["psi"]), _d(arrs["psi0"]),
                            _d(arrs["psiB"]), _d(arrs["bd"]), _d(arrs["bdB"]), _d(arrs["corr"]), _d(arrs["corrB"]), _d(arrs["Sp"]),
                            _d(arrs["Su"]), _d(arrs["V"]), 1.0, 0.0, _d(lam), _d(lamB), _d(scratch), 0, 0, 0.0)
        want, wantB = mo.limiter(n, m.lower, m.upper, d["bfc"], d["V"], d["rDeltaT"], d["psi"], d["psi0"], d["psiB"], bd, bdB, corr,
                                 corrB, 1.0, 0.0, nIter, **kw)
        assert np.array_equal(lam, want) and np.array_equal(lamB, wantB)


@pytest.mark.parametrize("combo", COMBOS)
def test_mules_sequencing_over_the_oracle_backend(meshmod, orc, combo):
    """rapidcfd-dev_b200/mules.py issues the reference's operations in the reference's order"""
    import torch
    import oracle_backend as ob
    mules = importlib.import_module("rapidcfd-dev_b200.mules")
    capi, ctx, _ = ob.fixture()
    d = case(meshmod, (5, 4, 6), seed=6, combo=combo)
    m, kw = d["m"], d["kw"]
    addr = capi.mesh_to_device(ctx, m)
    capi.fv_boundary_set(addr, d["bfc"])
    ops = capi.FieldOps(ctx)
    t = lambda x: None if x is None else torch.from_numpy(np.ascontiguousarray(x, np.float64))
    tk = {k: t(v) for k, v in kw.items()}
    lp, lpB = mules.limit(capi, addr, ops, t(d["V"]), d["rDeltaT"], t(d["psi"]), t(d["psi0"]), t(d["psiB"]), t(d["phi"]), t(d["phiB"]),
                          t(d["phiPsi"]), t(d["phiPsiB"]), 1.0, 0.0, 3, **tk)
    want, wantB = mo.limit(d["n"], m.lower, m.upper, d["bfc"], d["V"], d["rDeltaT"], d["psi"], d["psi0"], d["psiB"], d["phi"], d["phiB"],
                           d["phiPsi"], d["phiPsiB"], 1.0, 0.0, 3, **kw)
    assert np.array_equal(lp.numpy(), want) and np.array_equal(lpB.numpy(), wantB)
    new = mules.explicit_solve(capi, addr, ops, t(d["V"]), d["rDeltaT"], t(d["psi0"]), lp, lpB, **tk)
    assert np.array_equal(new.numpy(), mo.explicit_solve(d["n"], m.lower, m.upper, d["bfc"], d["V"], d["rDeltaT"], d["psi0"], want,
                                                         wantB, **kw))


def _h01(meshmod, key, seed):
    return meshmod._hash01(np.asarray(key, np.uint64) + meshmod._seedmix(seed))


def decomposed(meshmod, dims, nRanks, seed=5, combo="one-zero", scale=1e-3):
    """the ranks of a brick decomposition with fields that are functions of the GLOBAL cell / face: per rank a dict of
    limiter_steps keyword arguments (walls first, then the processor patch faces with psiB = the neighbour cells' psi), the
    patch starts, the number of coupled patches, and the exchange between the ranks"""
    G = dims[0] * dims[1] * dims[2]
    gpsi = _h01(meshmod, np.arange(G), seed)
    gpsi[: G // 5], gpsi[G // 5: G // 3] = 1.0, 0.0
    gV = (1.0 / dims[0]) ** 3 * (0.8 + 0.4 * _h01(meshmod, np.arange(G), seed + 1))
    grho, grho0 = 0.9 + 0.2 * _h01(meshmod, np.arange(G), seed + 2), 0.9 + 0.2 * _h01(meshmod, np.arange(G), seed + 3)
    gSp, gSu = -_h01(meshmod, np.arange(G), seed + 4), 0.1 * _h01(meshmod, np.arange(G), seed + 5)
    gphi = lambda gOwner, axis: (2 * _h01(meshmod, np.asarray(gOwner, np.uint64) * np.uint64(3) + np.asarray(axis, np.uint64), seed + 6) - 1) * scale
    cases, starts, nCP, meshes = [], [], [], []
    for r in range(nRanks):
        m = meshmod.decompose(None, nRanks, r, dims=dims) if nRanks > 1 else meshmod.hex_mesh(*dims)
        if nRanks == 1:
            m.cellGlobal = np.arange(m.nCells)
        g = m.cellGlobal
        walls, procs = m.wall_patches(), m.coupled_patches()
        ps, bfc = m.patch_start_facecells(walls + procs)
        psiB, phiB = [], []
        for p in walls:
            axis = int(np.nonzero(p.Sf[0])[0][0])
            side = 2 * axis + int(p.Sf[0, axis] > 0)
            key = g[p.faceCells].astype(np.uint64) * np.uint64(6) + np.uint64(side)
            psiB.append(_h01(meshmod, key, seed + 7))
            phiB.append(np.where(_h01(meshmod, key, seed + 8) < 0.3, 0.0, (2 * _h01(meshmod, key, seed + 9) - 1) * scale))
        for p in procs:
            axis = int(np.nonzero(p.Sf[0])[0][0])
            out = p.Sf[0, axis] > 0                                    # this rank holds the global owner of the face
            psiB.append(gpsi[p.nbrGlobalCells])
            phiB.append(gphi(g[p.faceCells], axis) if out else -gphi(p.nbrGlobalCells, axis))
        psiB, phiB = np.concatenate(psiB), np.concatenate(phiB)
        phi = gphi(g[m.lower], m.faceDir)
        psi = gpsi[g]
        nC = sum(len(p.faceCells) for p in procs)
        nW = len(bfc) - nC
        cellB = psi[bfc]
        phiPsi = phi * (0.5 * (psi[m.lower] + psi[m.upper]))
        phiPsiB = np.where(np.arange(len(bfc)) < nW, phiB * psiB, phiB * (0.5 * (cellB + psiB)))
        bd = mo.upwind_flux(m.lower, m.upper, phi, phiB, psi, psiB)[0]            # the reference's one-weight form, w*(P - N) + N
        bdB = np.where(np.arange(len(bfc)) < nW, phiB * psiB, phiB * np.where(phiB >= 0, cellB, psiB))
        c = dict(nCells=m.nCells, lower=m.lower, upper=m.upper, bFaceCells=bfc, V=gV[g], rDeltaT=50.0, psi=psi, psi0=psi.copy(), psiB=psiB,
                 phiBD=bd, phiBDB=bdB, phiCorr=phiPsi - bd, phiCorrB=phiPsiB - bdB, psiMax=1.0, psiMin=0.0, nLimiterIter=3, nCoupled=nC)
        if "rho" in combo:
            c.update(rho=grho[g], rho0=grho0[g])
        if "SpSu" in combo:
            c.update(Sp=gSp[g], Su=gSu[g])
        cases.append(c), starts.append(ps), nCP.append(len(procs)), meshes.append(m)
        m.mules_fluxes = (phi, phiB)                                   # for the callers that go through MULES::limit

    def exchange(mine):
        """mine[r] = the values on rank r's coupled faces (patches in neighbour-rank order) -> what each rank receives"""
        seg = {}
        for r, m in enumerate(meshes):
            o = 0
            for p in m.coupled_patches():
                seg[(r, p.neighbRank)] = mine[r][o: o + len(p.faceCells)]
                o += len(p.faceCells)
        return [np.concatenate([seg[(p.neighbRank, r)] for p in m.coupled_patches()]) if m.coupled_patches() else np.zeros(0)
                for r, m in enumerate(meshes)]

    return cases, starts, nCP, exchange, meshes


def decomposed_fluxes(meshmod, dims, nRanks, rank, seed=5):
    """(phi, phiB) of one rank of decomposed(): the face fluxes behind its phiBD / phiCorr"""
    return decomposed(meshmod, dims, nRanks, seed)[4][rank].mules_fluxes


@pytest.mark.parametrize("nRanks,combo", [(2, "one-zero"), (4, "rho-SpSu"), (8, "SpSu")])
def test_oracle_matches_the_reference_on_a_decomposed_case(meshmod, nRanks, combo):
    """processor patches: psi of the neighbour cells in the extrema, the coupled face rule, the minimum with the other side"""
    cases, starts, nCP, exchange, _ = decomposed(meshmod, (8, 6, 4), nRanks, combo=combo)
    got = mo.limiter_ranks(cases, exchange)
    ref = mo.reference_ranks(cases, starts, nCP, exchange, 3)
    for (lam, lamB), (rl, rlB), c in zip(got, ref, cases):
        assert np.array_equal(lam, rl) and np.array_equal(lamB, rlB)
        assert (lamB[len(lamB) - c["nCoupled"]:] < 1).any()


@pytest.mark.parametrize("nRanks,combo", [(2, "rho"), (8, "one-zero")])
def test_device_mules_code_on_the_host_decomposed(hk, meshmod, orc, nRanks, combo):  # noqa: F811
    """the coupled-face branch of the device code: one sweep per launch sequence and rank, the minimum with the other side between"""
    cases, _, _, exchange, _ = decomposed(meshmod, (8, 6, 4), nRanks, seed=11, combo=combo)
    want = mo.limiter_ranks(cases, exchange)
    f = lambda x: None if x is None else np.ascontiguousarray(x, np.float64)
    hk.hk_mules_limiter.argtypes = [C.c_void_p, C.c_int, C.c_double] + [C.c_void_p] * 12 + [C.c_double, C.c_double] + [C.c_void_p] * 3 + [C.c_int, C.c_int, C.c_double]
    hosts, lam, lamB, arrs = [], [], [], []
    for c in cases:
        a = orc.Addr(c["nCells"], c["lower"], c["upper"])
        hosts.append(Host(a, dict(bfc=c["bFaceCells"], diag=np.zeros(c["nCells"]), upper=np.zeros(len(c["lower"])), lower=None)))
        lam.append(np.ones(len(c["lower"]))), lamB.append(np.ones(len(c["bFaceCells"])))
        arrs.append({k: f(c.get(k)) for k in ("rho", "rho0", "psi", "psi0", "psiB", "phiBD", "phiBDB", "phiCorr", "phiCorrB", "Sp", "Su", "V")})
    for _ in range(3):
        for r, c in enumerate(cases):
            A, scratch = arrs[r], np.zeros(6 * c["nCells"])
            hk.hk_mules_limiter(hosts[r].p(), 1, c["rDeltaT"], _d(A["rho"]), _d(A["rho0"]), _d(A["psi"]), _d(A["psi0"]), _d(A["psiB"]),
                                _d(A["phiBD"]), _d(A["phiBDB"]), _d(A["phiCorr"]), _d(A["phiCorrB"]), _d(A["Sp"]), _d(A["Su"]), _d(A["V"]),
                                1.0, 0.0, _d(lam[r]), _d(lamB[r]), _d(scratch), c["nCoupled"], 0, 0.0)
        theirs = exchange([lb[len(lb) - c["nCoupled"]:] for lb, c in zip(lamB, cases)])
        for r, c in enumerate(cases):
            k = len(lamB[r]) - c["nCoupled"]
            lamB[r][k:] = np.minimum(lamB[r][k:], theirs[r])
    for r in range(nRanks):
        assert np.array_equal(lam[r], want[r][0]) and np.array_equal(lamB[r], want[r][1])


@pytest.mark.parametrize("nRanks", [2, 8])
def test_decomposed_limiter_is_the_single_domain_limiter(meshmod, nRanks):
    """both sides of a processor face end with the same limiter, and every face's limiter is the single-domain one up to the
    order of the per-cell sums (a face that became a patch face is added after the internal ones)"""
    dims = (8, 6, 4)
    cases, _, _, exchange, meshes = decomposed(meshmod, dims, nRanks)
    got = mo.limiter_ranks(cases, exchange)
    one, _, _, _, (m1,) = decomposed(meshmod, dims, 1)
    lam1, lamB1 = mo.limiter(**{k: v for k, v in one[0].items() if k != "nCoupled"})
    face1 = {(int(a), int(b)): i for i, (a, b) in enumerate(zip(m1.lower, m1.upper))}
    mine = [l[1][len(l[1]) - c["nCoupled"]:] for l, c in zip(got, cases)]
    theirs = exchange(mine)
    nLive = 0
    for r, (m, (lam, lamB), c) in enumerate(zip(meshes, got, cases)):
        g = m.cellGlobal
        idx = [face1[(int(g[a]), int(g[b]))] for a, b in zip(m.lower, m.upper)]
        assert np.allclose(lam, lam1[idx], rtol=0, atol=1e-11)
        assert np.array_equal(mine[r], theirs[r])
        o = len(lamB) - c["nCoupled"]
        for p in m.coupled_patches():
            k = len(p.faceCells)
            idx = [face1[tuple(sorted((int(g[a]), int(b))))] for a, b in zip(p.faceCells, p.nbrGlobalCells)]
            live = c["phiCorrB"][o: o + k] != 0          # a face without anti-diffusive flux takes lambdam of both sides here,
            nLive += int(live.sum())                     # lambdam / lambdap in the single domain: its limiter multiplies zero
            assert np.allclose(lamB[o: o + k][live], lam1[idx][live], rtol=0, atol=1e-11)
            o += k
    assert nLive > 20


def corr_case(meshmod, dims, seed, combo):
    """a flux correction on top of the case: high-order minus upwind, perturbed on the boundary so that its faces take part"""
    d = case(meshmod, dims, seed=seed, combo=combo)
    m = d["m"]
    bd, bdB = mo.upwind_flux(m.lower, m.upper, d["phi"], d["phiB"], d["psi"], d["psiB"])
    d["corr"], d["corrB"] = d["phiPsi"] - bd, d["phiPsiB"] - bdB + 1e-5 * np.sin(np.arange(d["nB"]))
    d["kw"].pop("rho0", None)
    return d


@pytest.mark.parametrize("combo", COMBOS)
@pytest.mark.parametrize("extremaCoeff", [0.0, 0.1])
def test_oracle_matches_the_reference_cmules(meshmod, combo, extremaCoeff):
    d = corr_case(meshmod, (7, 5, 4), 3, combo)
    m, kw = d["m"], d["kw"]
    args = (d["n"], m.lower, m.upper, d["ps"], d["bfc"], d["V"], d["rDeltaT"], d["psi"], d["psi0"], d["psiB"])
    phiAll, corrAll = _cat(d["phi"], d["phiB"]), _cat(d["corr"], d["corrB"])
    lam, lamB = mo.limiter(d["n"], m.lower, m.upper, d["bfc"], d["V"], d["rDeltaT"], d["psi"], d["psi"], d["psiB"], np.zeros(d["nF"]),
                           d["phiB"], d["corr"], d["corrB"], 1.0, 0.0, 3, kw.get("rho"), None, kw.get("Sp"), kw.get("Su"), corr=True,
                           extremaCoeff=extremaCoeff)
    assert np.array_equal(_cat(lam, lamB), mo.reference(3, *args, phiAll, corrAll, 1.0, 0.0, 3, extremaCoeff=extremaCoeff, **kw))
    assert (lam < 1).sum() > d["nF"] // 5 and (lamB < 1).any()
    lc, lcB = mo.limit_corr(d["n"], m.lower, m.upper, d["bfc"], d["V"], d["rDeltaT"], d["psi"], d["psiB"], d["phiB"], d["corr"], d["corrB"],
                            1.0, 0.0, 3, extremaCoeff=extremaCoeff, **kw)
    assert np.array_equal(_cat(lc, lcB), mo.reference(4, *args, phiAll, corrAll, 1.0, 0.0, 3, extremaCoeff=extremaCoeff, **kw))
    new = mo.correct(d["n"], m.lower, m.upper, d["bfc"], d["V"], d["rDeltaT"], d["psi"], lc, lcB, **kw)
    assert np.array_equal(new, mo.reference(5, *args, phiAll, _cat(lc, lcB), **kw))


@pytest.mark.parametrize("combo", COMBOS)
def test_device_cmules_code_on_the_host_and_sequencing(hk, meshmod, orc, combo):  # noqa: F811
    import torch
    import oracle_backend as ob
    d = corr_case(meshmod, (6, 7, 5), 4, combo)
    m, kw, n, nF, nB = d["m"], d["kw"], d["n"], d["nF"], d["nB"]
    H = Host(orc.Addr(n, m.lower, m.upper), dict(bfc=d["bfc"], diag=np.zeros(n), upper=np.zeros(nF), lower=None))
    f = lambda x: None if x is None else np.ascontiguousarray(x, np.float64)
    A = {k: f(v) for k, v in dict(psi=d["psi"], psiB=d["psiB"], phiB=d["phiB"], corr=d["corr"], corrB=d["corrB"], V=d["V"],
                                  rho=kw.get("rho"), Sp=kw.get("Sp"), Su=kw.get("Su")).items()}
    hk.hk_mules_limiter.argtypes = [C.c_void_p, C.c_int, C.c_double] + [C.c_void_p] * 12 + [C.c_double, C.c_double] + [C.c_void_p] * 3 + [C.c_int, C.c_int, C.c_double]
    for ex in (0.0, 0.25):
        lam, lamB, scratch = np.ones(nF), np.ones(nB), np.zeros(6 * n)
        hk.hk_mules_limiter(H.p(), 3, d["rDeltaT"], _d(A["rho"]), None, _d(A["psi"]), _d(A["psi"]), _d(A["psiB"]), None, _d(A["phiB"]),
                            _d(A["corr"]), _d(A["corrB"]), _d(A["Sp"]), _d(A["Su"]), _d(A["V"]), 1.0, 0.0, _d(lam), _d(lamB), _d(scratch),
                            0, 1, ex * (1.0 - 0.0))
        want, wantB = mo.limiter(n, m.lower, m.upper, d["bfc"], d["V"], d["rDeltaT"], d["psi"], d["psi"], d["psiB"], np.zeros(nF), d["phiB"],
                                 d["corr"], d["corrB"], 1.0, 0.0, 3, kw.get("rho"), None, kw.get("Sp"), kw.get("Su"), corr=True, extremaCoeff=ex)
        assert np.array_equal(lam, want) and np.array_equal(lamB, wantB)
    # rapidcfd-dev_b200/mules.py limit_corr + correct over the stand-in
    mules = importlib.import_module("rapidcfd-dev_b200.mules")
    capi, ctx, _ = ob.fixture()
    addr = capi.mesh_to_device(ctx, m)
    capi.fv_boundary_set(addr, d["bfc"])
    ops = capi.FieldOps(ctx)
    t = lambda x: None if x is None else torch.from_numpy(np.ascontiguousarray(x, np.float64))
    tk = {k: t(v) for k, v in kw.items()}
    lc, lcB = mules.limit_corr(capi, addr, ops, t(d["V"]), d["rDeltaT"], t(d["psi"]), t(d["psiB"]), t(d["phiB"]), t(d["corr"]), t(d["corrB"]),
                               1.0, 0.0, 3, **tk)
    want, wantB = mo.limit_corr(n, m.lower, m.upper, d["bfc"], d["V"], d["rDeltaT"], d["psi"], d["psiB"], d["phiB"], d["corr"], d["corrB"],
                                1.0, 0.0, 3, **kw)
    assert np.array_equal(lc.numpy(), want) and np.array_equal(lcB.numpy(), wantB)
    new = mules.correct(capi, addr, ops, t(d["V"]), d["rDeltaT"], t(d["psi"]), lc, lcB, **tk)
    assert np.array_equal(new.numpy(), mo.correct(n, m.lower, m.upper, d["bfc"], d["V"], d["rDeltaT"], d["psi"], want, wantB, **kw))


def advect(meshmod, limited, steps=12):
    """a slab of psi = 1 carried along x through a closed box by a solenoidal (uniform, walls closed) flux, central face values"""
    m = meshmod.hex_mesh(16, 3, 3)
    ps, bfc = m.patch_start_facecells(m.wall_patches())
    n, nB = m.nCells, len(bfc)
    V = m.volumes()
    x = m.cell_centres()[:, 0]
    psi = np.where((x > 0.2) & (x < 0.5), 1.0, 0.0)
    u, dt = 1.0, 0.3 * m.h                                     # Courant 0.3
    phi = np.where(m.faceDir == 0, u * m.h * m.h, 0.0)         # uniform in x ...
    interior = (m.lower % m.nx) < m.nx - 2                     # ... stopped two cells before the end wall:
    phi = np.where(interior, phi, 0.0)                         # the slab piles up against a flux-free face
    phiB, psiB = np.zeros(nB), np.zeros(nB)
    lo, hi, mass = [], [], []
    for _ in range(steps):
        phiPsi, phiPsiB = phi * (0.5 * (psi[m.lower] + psi[m.upper])), phiB * psiB
        if limited:
            phiPsi, phiPsiB = mo.limit(n, m.lower, m.upper, bfc, V, 1 / dt, psi, psi, psiB, phi, phiB, phiPsi, phiPsiB, 1.0, 0.0, 3)
        psi = mo.explicit_solve(n, m.lower, m.upper, bfc, V, 1 / dt, psi, phiPsi, phiPsiB)
        lo.append(psi.min()), hi.append(psi.max()), mass.append((psi * V).sum())
    return np.array(lo), np.array(hi), np.array(mass)


def test_limited_update_is_bounded_and_conservative(meshmod):
    lo, hi, mass = advect(meshmod, False)
    assert lo.min() < -0.05 and hi.max() > 1.05                # central differencing alone over- and undershoots
    lo, hi, massL = advect(meshmod, True)
    assert lo.min() >= -1e-12 and hi.max() <= 1 + 1e-12        # MULES keeps psi within [psiMin, psiMax]
    assert np.allclose(massL, massL[0], rtol=1e-13) and np.allclose(mass, massL[0], rtol=1e-13)   # fluxes only: conservative


@pytest.mark.parametrize("corr", [0, 1])
def test_device_mules_code_on_a_random_graph(hk, orc, corr):  # noqa: F811
    """rows with up to a dozen faces per side, several boundary faces per cell, cells without owner or neighbour faces"""
    from test_fv_kernels_cpu import _Graph
    g = _Graph(240, 4, 21)
    rng = np.random.default_rng(22)
    n, nF = g.nCells, g.nFaces
    bfc = rng.integers(0, n, 130).astype(np.int32)
    nB = len(bfc)
    H = Host(orc.Addr(n, g.lower, g.upper), dict(bfc=bfc, diag=np.zeros(n), upper=np.zeros(nF), lower=None))
    f = lambda x: np.ascontiguousarray(x, np.float64)
    psi, psiB, V = f(rng.uniform(0, 1, n)), f(rng.uniform(0, 1, nB)), f(rng.uniform(0.5, 2, n))
    bd, bdB = f(rng.uniform(-1, 1, nF) * 1e-2), f(rng.uniform(-1, 1, nB) * 1e-2)
    pc, pcB = f(rng.uniform(-1, 1, nF) * 1e-2), f(rng.uniform(-1, 1, nB) * 1e-2)
    rho, Sp, Su = f(rng.uniform(0.9, 1.1, n)), f(-rng.uniform(0, 1, n)), f(rng.uniform(0, 0.1, n))
    hk.hk_mules_limiter.argtypes = [C.c_void_p, C.c_int, C.c_double] + [C.c_void_p] * 12 + [C.c_double, C.c_double] + [C.c_void_p] * 3 + [C.c_int, C.c_int, C.c_double]
    lam, lamB, scratch = np.ones(nF), np.ones(nB), np.zeros(6 * n)
    hk.hk_mules_limiter(H.p(), 3, 20.0, _d(rho), _d(rho), _d(psi), _d(psi), _d(psiB), None if corr else _d(bd), _d(bdB), _d(pc), _d(pcB),
                        _d(Sp), _d(Su), _d(V), 1.0, 0.0, _d(lam), _d(lamB), _d(scratch), 0, corr, 0.1 if corr else 0.0)
    want, wantB = mo.limiter(n, g.lower, g.upper, bfc, V, 20.0, psi, psi, psiB, bd, bdB, pc, pcB, 1.0, 0.0, 3, rho, rho, Sp, Su,
                             corr=bool(corr), extremaCoeff=0.1 if corr else 0.0)
    assert np.array_equal(lam, want) and np.array_equal(lamB, wantB)
    assert (lam < 1).sum() > 20                       # the limiter is active on this case
