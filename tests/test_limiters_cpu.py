"""Limited / upwind interpolation weights (SURVEY.md section 8(f) rank 1): the oracle against the reference's own limiter
headers compiled here (NVDTVD.H, limitedLinear.H, vanLeer.H, Minmod.H -> oracle/_ref/libref_limiters.so), and the device
code of csrc/fieldops_kernels.cuh executed on the host against the oracle -- all bit for bit."""
import ctypes as C

import numpy as np
import pytest

import ref_replay
from oracle import limiters_oracle as lo
from test_host_kernels_cpu import hk  # noqa: F401  (fixture: the host build of the kernels)

ref_replay.install()   # the reference's answers come from tests/golden/ref_calls_*.npz


def _case(meshmod, dims=(9, 7, 5), seed=3):
    m = meshmod.hex_mesh(*dims)
    rng = np.random.default_rng(seed)
    vf = rng.uniform(-1, 1, m.nCells)
    vf[: m.nCells // 7] = 0.25                      # flat patches: gradf == 0 -> the clipped branch of r
    gradc = rng.uniform(-2, 2, (m.nCells, 3))
    gradc[m.nCells // 2: m.nCells // 2 + 20] = 0.0   # gradcf == 0
    flux = rng.uniform(-1, 1, m.nFaces)
    flux[::11] = 0.0                                # pos(0) = 1, and faceFlux > 0 is false
    cd = m.weights()
    return m, vf, gradc, flux, cd, m.cell_centres()


@pytest.mark.parametrize("scheme,k", [("limitedLinear", 1.0), ("limitedLinear", 0.33), ("limitedLinear", 0.0), ("vanLeer", 1.0),
                                      ("Minmod", 1.0)])
def test_oracle_limiters_match_the_reference_headers(meshmod, scheme, k):
    m, vf, gradc, flux, cd, cc = _case(meshmod)
    got = lo.limiter(scheme, m.lower, m.upper, flux, vf, gradc, cc, k)
    ref = lo.reference_limiter(scheme, m.lower, m.upper, cd, flux, vf, gradc, cc, k)
    assert np.array_equal(got, ref, equal_nan=True)
    assert got.min() >= 0 and (scheme == "vanLeer" or got.max() <= 1)


@pytest.mark.parametrize("scheme,k", [("upwind", 1.0), ("linear", 1.0), ("limitedLinear", 1.0), ("limitedLinear", 0.2),
                                      ("vanLeer", 1.0), ("Minmod", 1.0)])
def test_device_limiter_code_on_the_host(hk, meshmod, scheme, k):  # noqa: F811
    m, vf, gradc, flux, cd, cc = _case(meshmod, (8, 6, 7), 5)
    i32 = lambda a: np.ascontiguousarray(a, np.int32)
    f64 = lambda a: np.ascontiguousarray(a, np.float64)
    l, u, g, c = i32(m.lower), i32(m.upper), f64(gradc), f64(cc)
    out = np.zeros(m.nFaces)
    hk.hk_limiter.argtypes = [C.c_int, C.c_int, C.c_double] + [C.c_void_p] * 7
    hk.hk_limiter(m.nFaces, lo.SCHEMES[scheme], 2.0 / max(k, lo.SMALL), l.ctypes.data, u.ctypes.data, f64(flux).ctypes.data,
                  f64(vf).ctypes.data, g.ctypes.data, c.ctypes.data, out.ctypes.data)
    want = lo.limiter(scheme, m.lower, m.upper, flux, vf, gradc, cc, k)
    assert np.array_equal(out, want, equal_nan=True)
    # weights: limiter*cd + (1 - limiter)*pos(flux); upwind without a limiter field
    w = np.zeros(m.nFaces)
    hk.hk_limited_weights.argtypes = [C.c_longlong] + [C.c_void_p] * 4
    hk.hk_limited_weights(m.nFaces, out.ctypes.data, f64(cd).ctypes.data, f64(flux).ctypes.data, w.ctypes.data)
    assert np.array_equal(w, lo.limited_weights(flux, want, cd), equal_nan=True)
    hk.hk_limited_weights(m.nFaces, None, None, f64(flux).ctypes.data, w.ctypes.data)
    assert np.array_equal(w, lo.limited_weights(flux)) and set(np.unique(w)) <= {0.0, 1.0}
    if scheme == "upwind":   # a zero limiter gives the upwind weights through the general formula too
        assert np.array_equal(lo.limited_weights(flux, want, cd), lo.limited_weights(flux))


def test_upwind_convection_matrix_is_an_m_matrix(meshmod, orc):
    """gaussConvectionScheme::fvmDiv with upwind weights (gaussConvectionScheme.C:95-105): lower = -w*phi, upper = lower +
    phi: off-diagonals non-positive, diag = -sum >= 0 row by row"""
    m, vf, gradc, flux, cd, cc = _case(meshmod)
    w = lo.limited_weights(flux)
    oa = orc.Addr(m.nCells, m.lower, m.upper)
    lower, upper, diag = orc.convection_fill(oa, w, flux)
    assert np.all(lower <= 0) and np.all(upper <= 0) and np.all(diag >= 0)
