"""lduMatrix algebra at the ABI (SURVEY.md section 8 row a5): row sums sumDiag / negSumDiag / sumMagOffDiag and operator+= / -= / *=.
CPU: the numpy restatement against the reference's own operators compiled here (oracle/_ref/libref_lduops.so), every kind
combination, bit for bit.  GPU: b200ldu_ldu_* against the restatement and the oracle's row sums, bit for bit."""
import importlib
import itertools

import numpy as np
import pytest

import ref_replay
from oracle import lduops_oracle as lo
from oracle import ref_ldu

ref_replay.install()   # the reference's answers come from tests/golden/ref_calls_*.npz

KINDS = {"diagonal": ("diag",), "symmetric": ("diag", "upper"), "asymmetric": ("diag", "upper", "lower"),
         "noDiagSym": ("upper",), "empty": ()}


def _mat(m, kind, seed):
    rng = np.random.default_rng(seed)
    full = dict(diag=rng.uniform(1, 2, m.nCells), upper=rng.uniform(-1, 1, m.nFaces), lower=rng.uniform(-1, 1, m.nFaces))
    return {k: full[k] for k in KINDS[kind]}


@pytest.mark.parametrize("ka,kb", list(itertools.product(["diagonal", "symmetric", "asymmetric", "empty"],
                                                         ["diagonal", "symmetric", "asymmetric"])))
@pytest.mark.parametrize("sub", [False, True])
def test_restatement_matches_the_references_operators(meshmod, ka, kb, sub):
    m = meshmod.hex_mesh(5, 4, 3)
    A, B = _mat(m, ka, 1), _mat(m, kb, 2)
    ref = ref_ldu.ldu_combine(m.nCells, m.lower, m.upper, A, -1 if sub else 1, B)
    got = lo.add_assign(A, B, m.nCells, sub)
    assert sorted(ref) == sorted(got), (ka, kb, sorted(ref), sorted(got))
    for k in ref:
        assert np.array_equal(ref[k], got[k]), (ka, kb, k)


@pytest.fixture(scope="module")
def gpu():
    import torch
    capi = importlib.import_module("rapidcfd-dev_b200.capi")
    ctx = capi.Context(0)
    yield capi, ctx, torch
    ctx.close()


@pytest.mark.gpu
def test_ldu_algebra_on_the_device(gpu, meshmod, orc):
    capi, ctx, torch = gpu
    m = meshmod.hex_mesh(9, 7, 5)
    t = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(ctx.device)
    addr = capi.mesh_to_device(ctx, m)
    host = lambda x: None if x is None else x.cpu().numpy()
    for ka, kb, sub in itertools.product(["diagonal", "symmetric", "asymmetric", "empty"], ["diagonal", "symmetric", "asymmetric"],
                                         [False, True]):
        A, B = _mat(m, ka, 3), _mat(m, kb, 4)
        dA = capi.LduCoeffs(addr, t(A.get("diag")), t(A.get("upper")), t(A.get("lower")))
        dB = capi.LduCoeffs(addr, t(B.get("diag")), t(B.get("upper")), t(B.get("lower")))
        if sub:
            dA -= dB
        else:
            dA += dB
        want = lo.add_assign(A, B, m.nCells, sub)
        got = dict(zip(("diag", "upper", "lower"), (host(x) for x in dA.arrays())))
        assert sorted(k for k, v in got.items() if v is not None) == sorted(want), (ka, kb, sub)
        for k, v in want.items():
            assert np.array_equal(got[k], v), (ka, kb, sub, k)
    # operator*=: by a cell field (upper by the owner's value, lower by the neighbour's) and by a scalar
    A = _mat(m, "asymmetric", 5)
    sf = np.random.default_rng(6).uniform(0.5, 2, m.nCells)
    for s in (sf, 1.7):
        d = capi.LduCoeffs(addr, t(A["diag"]), t(A["upper"]), t(A["lower"]))
        d.scale(t(s) if not np.isscalar(s) else s)
        want = lo.scale(A, s, m.lower, m.upper)
        for k, v in zip(("diag", "upper", "lower"), d.arrays()):
            assert np.array_equal(host(v), want[k]), k
    # row sums against the oracle (pinned to lduMatrixOperations.C:36-104 in tests/test_reference_functors.py)
    oa = orc.Addr(m.nCells, m.lower, m.upper)
    for kind in ("symmetric", "asymmetric"):
        A = _mat(m, kind, 7)
        d = capi.LduCoeffs(addr, t(A["diag"]), t(A["upper"]), t(A.get("lower")))
        for mode, fn in ((0, "orc_sumDiag"), (1, "orc_negSumDiag"), (2, "orc_sumMagOffDiag")):
            io = A["diag"].copy()
            low = A.get("lower")
            getattr(orc.lib(), fn)(oa.h, orc._d(A["upper"]), orc._d(low) if low is not None else None, orc._d(io))
            got = d.row_sum(mode, t(A["diag"].copy()))
            assert np.array_equal(host(got), io), (kind, mode)
    addr.close()
