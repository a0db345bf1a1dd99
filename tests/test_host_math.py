"""The DEVICE math header (taichi_mpm_b200/csrc/mpmb_math.cuh) compiled for the host and checked
against the fp64 oracle — the arithmetic the CUDA kernels run (eigen-system of F F^T - I, series
log/exp sand step, one-decomposition fixed-corotated family, weights, friction projection) is
covered on a machine without a GPU.  The intrinsics' host meanings are in
tests/host_math/stub/cuda_runtime.h; `-m gpu` tests remain the parity tests of the kernels proper.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import pyoracle as O
from taichi_mpm_b200 import scenes
from tests import common as T

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "host_math", "host_math.cpp")
_STUB = os.path.join(_HERE, "host_math", "stub")
_CSRC = os.path.join(os.path.dirname(_HERE), "taichi_mpm_b200", "csrc")
_LIB = os.path.join(_HERE, "host_math", "_build", "libhostmath.so")


@pytest.fixture(scope="module")
def hm():
    deps = [_SRC, os.path.join(_STUB, "cuda_runtime.h"), os.path.join(_CSRC, "mpmb_math.cuh")]
    if not os.path.exists(_LIB) or any(os.path.getmtime(d) > os.path.getmtime(_LIB) for d in deps):
        os.makedirs(os.path.dirname(_LIB), exist_ok=True)
        # -ffp-contract=off: only the fmaf() calls the header writes are fused, as under nvcc's
        # explicit-intrinsic style; -mfma makes fmaf a single instruction
        cmd = ["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-march=x86-64-v3", "-mfma",
               "-I" + _STUB, "-I" + _CSRC, _SRC, "-o", _LIB]
        subprocess.run(cmd, check=True)
    return C.CDLL(_LIB)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


_params8 = T.params8


def _cm(M):
    """batch of math-layout 3x3 -> column-major float32 [n,9] (Mat3::m[c*3+r])"""
    return np.ascontiguousarray(np.transpose(np.asarray(M, np.float32), (0, 2, 1)).reshape(-1, 9))


def _math(m9):
    return np.transpose(np.asarray(m9).reshape(-1, 3, 3), (0, 2, 1))


def _random_states(kind, n, seed, strain, rate):
    rng = np.random.default_rng(seed)
    F = np.eye(3)[None] + rng.normal(size=(n, 3, 3)) * strain
    cdg = np.eye(3)[None] + rng.normal(size=(n, 3, 3)) * rate
    if kind == scenes.MAT_SNOW:
        ps = 1.0 + rng.normal(size=n) * 0.05
    elif kind == scenes.MAT_WATER:
        ps = 1.0 + rng.normal(size=n) * 0.02
    elif kind == scenes.MAT_SAND:
        ps = np.abs(rng.normal(size=n)) * 2e-3 * (rng.random(n) < 0.5)
    elif kind == scenes.MAT_VISCO:
        ps = 1000.0 * (0.5 + rng.random(n))          # visco_tau around its default
    else:
        ps = np.zeros(n)
    vol = np.full(n, (1.0 / 256) ** 3 / 8)
    return F.astype(np.float32), cdg.astype(np.float32), ps.astype(np.float32), vol.astype(np.float32)


def _oracle_step(kind, prm, cdg, F, ps, vol):
    Fo, pso, fo = [], [], []
    for i in range(len(F)):
        f, s = O.plasticity(kind, prm, cdg[i].astype(np.float64), F[i].astype(np.float64), float(ps[i]), np.float64)
        Fo.append(f)
        pso.append(s)
        fo.append(O.calculate_force(kind, prm, f, s, float(vol[i]), np.float64))
    return np.array(Fo), np.array(pso), np.array(fo)


CASES = [
    (scenes.MAT_LINEAR, {}, 0.02, 2e-3),
    (scenes.MAT_JELLY, {}, 0.05, 2e-3),
    (scenes.MAT_SNOW, {}, 0.02, 5e-3),      # crosses both clamps
    (scenes.MAT_WATER, {}, 0.0, 5e-3),
    (scenes.MAT_SAND, {}, 2e-4, 1e-4),      # the series path: resting-column strains
    (scenes.MAT_SAND, {}, 3e-3, 2e-3),      # larger strains: more series terms
    (scenes.MAT_SAND, {"cohesion": 1e-3}, 1e-3, 1e-3),
    (scenes.MAT_SAND, {}, 1e-2, 5e-3),      # 5-6 log terms
    (scenes.MAT_SAND, {}, 3e-2, 1e-2),      # 7-9 log terms, 6 exp terms
    (scenes.MAT_SAND, {}, 0.1, 0.05),       # beyond the series' range: eigen fallback for most lanes
    (scenes.MAT_ELASTIC, {}, 0.05, 5e-3),
    (scenes.MAT_VON_MISES, {}, 0.02, 5e-3),   # both sides of the yield surface (|dev eps|^2 vs yield / 2 mu = 2.8e-4)
    (scenes.MAT_VON_MISES, {}, 1e-3, 1e-3),   # elastic only
    (scenes.MAT_VISCO, {}, 0.05, 5e-3),       # |P| above and below visco_tau
    (scenes.MAT_VISCO, {"kappa": 0.3}, 0.08, 1e-2),   # hardening: visco_tau moves
]


@pytest.mark.parametrize("kind,kw,strain,rate", CASES)
def test_device_material_step_matches_oracle(hm, kind, kw, strain, rate):
    n = 400
    F, cdg, ps, vol = _random_states(kind, n, 11 + kind, strain, rate)
    prm = _params8(kind, **kw)
    Fd, psd, force = _cm(F), ps.copy(), np.zeros((n, 9), np.float32)
    hm.hm_material_step(C.c_int64(n), C.c_int(kind), _p(prm), _p(_cm(cdg)), _p(Fd), _p(psd), _p(vol), _p(force))
    Fo, pso, fo = _oracle_step(kind, prm.astype(np.float64), cdg, F, ps, vol)
    if kind != scenes.MAT_WATER:                         # water carries no F (src/particles.cpp:469-478)
        assert np.abs(_math(Fd) - Fo).max() <= 2e-5      # tests/common.py TOL_F_ABS
    assert np.abs(psd - pso).max() <= 1e-5 * max(1.0, np.abs(pso).max())   # TOL_PS_ABS (visco_tau is O(1000))
    # force feeds the grid momentum: compare relative to the largest stress of the batch
    scale = np.abs(fo).max()
    assert scale > 0
    assert np.abs(_math(force) - fo).max() <= 2e-4 * scale


@pytest.mark.parametrize("kind,kw,strain,rate", CASES)
def test_device_two_call_form_matches_fused_step(hm, kind, kw, strain, rate):
    # upload-time calculate_force() after plasticity() == the fused material_step (same header)
    n = 200
    F, cdg, ps, vol = _random_states(kind, n, 31 + kind, strain, rate)
    prm = _params8(kind, **kw)
    F1, ps1, f1 = _cm(F), ps.copy(), np.zeros((n, 9), np.float32)
    hm.hm_material_step(C.c_int64(n), C.c_int(kind), _p(prm), _p(_cm(cdg)), _p(F1), _p(ps1), _p(vol), _p(f1))
    F2, ps2, f2 = _cm(F), ps.copy(), np.zeros((n, 9), np.float32)
    hm.hm_plasticity(C.c_int64(n), C.c_int(kind), _p(prm), _p(_cm(cdg)), _p(F2), _p(ps2))
    hm.hm_calculate_force(C.c_int64(n), C.c_int(kind), _p(prm), _p(F2), _p(ps2), _p(vol), _p(f2))
    assert np.abs(F1 - F2).max() <= 2e-6
    assert np.abs(ps1 - ps2).max() <= 2e-6 * max(1.0, np.abs(ps2).max())
    # the two-call form reads the strain back from the fp32-rounded F (a few ulp of 1 = a few 1e-7 of
    # strain), the fused step keeps it in registers: allow that strain error times stiffness * vol
    stiff = float(prm[0] * prm[1]) if kind == scenes.MAT_WATER else float(prm[0] + prm[1])
    assert np.abs(f1 - f2).max() <= 2e-4 * np.abs(f2).max() + 3e-6 * stiff * float(vol[0])


def test_device_sand_large_strain_matches_oracle_for_non_inverted_elements(hm):
    # |F-I| ~ 0.3-0.5: always the eigen path.  For det(F) < 0 the result depends on the sign convention of
    # the SVD (the reference's svd() belongs to the missing core, SURVEY appendix C): the device keeps the
    # reflection (ratios of |sigma|), the oracle's convention removes it; only det > 0 is compared, and
    # only where the smallest singular value leaves fp32 a meaningful log
    kind, n = scenes.MAT_SAND, 1500
    F, cdg, ps, vol = _random_states(kind, n, 77, 0.4, 0.1)
    prm = _params8(kind)
    Fd, psd, force = _cm(F), ps.copy(), np.zeros((n, 9), np.float32)
    hm.hm_material_step(C.c_int64(n), C.c_int(kind), _p(prm), _p(_cm(cdg)), _p(Fd), _p(psd), _p(vol), _p(force))
    Fo, pso, fo = _oracle_step(kind, prm.astype(np.float64), cdg, F, ps, vol)
    Ft = np.einsum("nij,njk->nik", cdg.astype(np.float64), F.astype(np.float64))
    ok = (np.linalg.det(Ft) > 0) & (np.linalg.svd(Ft, compute_uv=False).min(1) > 0.05)
    assert ok.sum() > n // 2
    assert np.abs(_math(Fd) - Fo)[ok].max() <= 2e-5
    assert np.abs(psd - pso)[ok].max() <= 1e-5
    assert np.abs(_math(force) - fo)[ok].max() <= 2e-4 * np.abs(fo[ok]).max()


@pytest.mark.parametrize("kind,strain,rate", [(scenes.MAT_LINEAR, 0.05, 0.01), (scenes.MAT_JELLY, 0.1, 0.01), (scenes.MAT_SNOW, 0.03, 0.01),
                                              (scenes.MAT_WATER, 0.0, 0.01), (scenes.MAT_SAND, 2e-3, 1e-3), (scenes.MAT_SAND, 0.05, 0.02),
                                              (scenes.MAT_ELASTIC, 0.05, 0.01), (scenes.MAT_VON_MISES, 0.02, 0.01), (scenes.MAT_VISCO, 0.05, 0.01)])
def test_device_material_step_matches_reference_particles_directly(hm, kind, strain, rate):
    # the CUDA header's fused step against the REFERENCE's own plasticity() + calculate_force()
    # (src/particles.cpp compiled in place with the stand-in core, oracle/particles_ref.cpp): no oracle in between;
    # what the reference computed is committed (tests/golden/make_live_golden.py: material_ref)
    ref = T.live_ref("material_c%d" % T.MATERIAL_CASES.index((kind, strain, rate)))
    prm = _params8(kind)
    vol = np.float32(T.MATERIAL_VOL)
    worst_F = worst_ps = worst_f = scale = 0.0
    for i, (F, cdg, ps) in enumerate(T.material_states(kind, strain, rate)):
        Fr, psr, fr = ref["F"][i], float(ref["ps"][i]), ref["force"][i]
        Fd, psd, force = _cm(F[None]), np.array([ps], np.float32), np.zeros((1, 9), np.float32)
        hm.hm_material_step(C.c_int64(1), C.c_int(kind), _p(prm), _p(_cm(cdg[None])), _p(Fd), _p(psd), _p(np.array([vol], np.float32)), _p(force))
        if kind != scenes.MAT_WATER:
            worst_F = max(worst_F, np.abs(_math(Fd)[0] - Fr).max())
        worst_ps = max(worst_ps, abs(float(psd[0]) - psr) / max(1.0, abs(psr)))
        worst_f = max(worst_f, np.abs(_math(force)[0] - fr).max())
        scale = max(scale, np.abs(fr).max())
    assert worst_F <= 2e-6 and worst_ps <= 3e-6
    hencky = kind in (scenes.MAT_SAND, scenes.MAT_ELASTIC, scenes.MAT_VON_MISES)
    assert worst_f <= (2e-4 if hencky else 2e-5) * scale   # the reference's fp32 log(sigma) at small strain


def test_device_zero_stress_at_identity(hm):
    for kind in (scenes.MAT_LINEAR, scenes.MAT_JELLY, scenes.MAT_SNOW, scenes.MAT_WATER, scenes.MAT_SAND, scenes.MAT_ELASTIC,
                 scenes.MAT_VON_MISES, scenes.MAT_VISCO):
        prm = _params8(kind)
        F = _cm(np.eye(3)[None])
        ps = np.array([scenes.default_scalar(kind)], np.float32)
        vol = np.array([1e-6], np.float32)
        out = np.ones((1, 9), np.float32)
        hm.hm_calculate_force(C.c_int64(1), C.c_int(kind), _p(prm), _p(F), _p(ps), _p(vol), _p(out))
        assert np.abs(out).max() == 0.0, kind


def test_device_eigensystem(hm):
    rng = np.random.default_rng(5)
    n = 500
    A = rng.normal(size=(n, 3, 3))
    A = (A + np.transpose(A, (0, 2, 1))) * 0.5 * (10.0 ** rng.uniform(-5, 0, size=(n, 1, 1)))
    A[0] = 0.0                                            # zero tensor
    A[1] = np.diag([1e-3, 1e-3, 1e-3])                    # triple eigenvalue
    A[2] = np.diag([2e-3, 2e-3, -1e-3])                   # double eigenvalue
    A6 = np.ascontiguousarray(np.stack([A[:, 0, 0], A[:, 1, 1], A[:, 2, 2], A[:, 0, 1], A[:, 0, 2], A[:, 1, 2]], 1), np.float32)
    U9, e3 = np.zeros((n, 9), np.float32), np.zeros((n, 3), np.float32)
    hm.hm_eig_sym3(C.c_int64(n), _p(A6), _p(U9), _p(e3))
    U = _math(U9).astype(np.float64)
    rec = np.einsum("nij,nj,nkj->nik", U, e3.astype(np.float64), U)
    nrm = np.maximum(np.abs(A).reshape(n, -1).max(1), 1e-30)
    assert (np.abs(rec - A).reshape(n, -1).max(1) <= 4e-6 * nrm + 1e-12).all()
    orth = np.einsum("nji,njk->nik", U, U) - np.eye(3)[None]
    assert np.abs(orth).max() <= 5e-6
    w = np.linalg.eigvalsh(A)
    assert np.abs(np.sort(e3.astype(np.float64), 1) - w).max(1).max() <= 4e-6 * nrm.max()


def test_device_weights_equal_reference_form(hm):
    rel = np.linspace(0.5, 1.5, 257, dtype=np.float32)[:-1]
    w = np.zeros((len(rel), 3), np.float32)
    hm.hm_bspline_weights(C.c_int64(len(rel)), _p(rel), _p(w))
    r = rel.astype(np.float64)
    ref = np.stack([0.5 * (1.5 - r) ** 2, 0.75 - (r - 1.0) ** 2, 0.5 * (r - 0.5) ** 2], 1)
    assert np.abs(w - ref).max() <= 2e-7
    assert np.abs(w.sum(1) - 1).max() <= 3e-7
    # and the oracle's restatement of MLSMPMFastKernel32 (src/transfer.cpp:168-186), fp32
    for k in (0, 37, 128, 255):
        wo = O.mls_fast_kernel(np.array([rel[k], rel[k], rel[k]], np.float32), np.float32)
        assert np.allclose(wo, np.einsum("i,j,k->ijk", w[k], w[k], w[k]), rtol=0, atol=3e-7)


def test_device_friction_project_cases(hm):
    rng = np.random.default_rng(9)
    n = 300
    v = rng.normal(size=(n, 3)).astype(np.float32)
    nn = rng.normal(size=(n, 3))
    nn = (nn / np.linalg.norm(nn, axis=1, keepdims=True)).astype(np.float32)
    for fr in (-1.0, -2.0, -2.3, 0.0, 0.4, 5.0):
        out = np.zeros((n, 3), np.float32)
        hm.hm_friction_project0(C.c_int64(n), _p(v), _p(nn), C.c_float(fr), _p(out))
        ref = np.array([O.friction_project(v[i], np.zeros(3), nn[i], fr, np.float64) for i in range(n)])
        assert np.abs(out - ref).max() <= 2e-6, fr
