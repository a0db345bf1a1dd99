"""Pin of the oracle's 3-D constitutive restatement against the REFERENCE's own code: the
Snow/Linear/Jelly/Water/Sand particles of /root/reference/src/particles.cpp (plasticity +
calculate_force, exactly the two calls of the hot path: src/transfer.cpp:509,950) and
friction_project of src/mpm_fwd.h:25-57, compiled where they lie (oracle/particles_ref.cpp) against a
stand-in for the un-vendored taichi core headers (oracle/taichi_stub/taichi/*.h — VectorND/MatrixND,
Config, svd/polar; its header says what is restated and which SVD convention it takes).  Golden
vectors of that run are committed (tests/golden/particles_ref.npz); where the reference tree is
present the code is also run live.  det F > 0 only: inverted elements depend on the SVD's sign
convention (DESIGN.md §2)."""
import importlib.util
import os

import numpy as np
import pytest

from oracle import pyoracle as O
from taichi_mpm_b200 import scenes

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("make_particles_golden", os.path.join(HERE, "golden", "make_particles_golden.py"))
G = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(G)


def _oracle_step(kind, prm, cdg, F, ps, dtype):
    F1, ps1 = O.plasticity(kind, prm.astype(np.float64), cdg.astype(np.float64), F.astype(np.float64), float(ps), dtype)
    force = O.calculate_force(kind, prm.astype(np.float64), F1, ps1, G.VOL, dtype)
    return np.asarray(F1, np.float64), float(ps1), np.asarray(force, np.float64)


# the reference evaluates log(sigma) in fp32: at strains of 2e-3 that alone is 6e-5 of the stress
FORCE_TOL = {0: 4e-6, 1: 4e-6, 2: 2e-5, 3: 2e-5, 4: 2e-4, 5: 2e-5, 6: 2e-4, 7: 2e-5}


@pytest.mark.parametrize("ci", range(len(G.CASES)))
def test_oracle_constitutive_matches_golden_run_of_reference_particles(ci):
    kind, strain, rate = G.CASES[ci]
    z = np.load(os.path.join(HERE, "golden", "particles_ref.npz"))
    prm = z["c%d_params" % ci]
    assert np.allclose(prm, scenes.material_params(kind), rtol=3e-7, atol=0)       # the defaults of initialize(), src/particles.cpp
    Fr, psr, fr = z["c%d_F" % ci], z["c%d_ps" % ci], z["c%d_force" % ci]
    scale = np.abs(fr).max()
    for i, (F, cdg, ps) in enumerate(G.golden_states(kind, strain, rate)):
        F1, ps1, force = _oracle_step(kind, prm, cdg, F, ps, np.float64)
        if kind != scenes.MAT_WATER:
            assert np.abs(F1 - Fr[i]).max() <= 1e-6, (kind, i)
        assert abs(ps1 - psr[i]) <= 2e-6 * max(1.0, abs(psr[i])), (kind, i)
        assert np.abs(force - fr[i]).max() <= FORCE_TOL[kind] * scale, (kind, i)
    if kind in (scenes.MAT_SNOW, scenes.MAT_SAND):                                   # the return maps were active
        assert np.abs(psr - np.array([s[2] for s in G.golden_states(kind, strain, rate)])).max() > 1e-4


def test_oracle_friction_project_matches_golden_run_of_reference():
    z = np.load(os.path.join(HERE, "golden", "particles_ref.npz"))
    v, base, n, fr = G.friction_cases()
    for i in range(len(v)):
        got = O.friction_project(v[i], base[i], n[i], float(fr[i]), np.float64)
        assert np.abs(got - z["friction_out"][i]).max() <= 3e-6, (i, fr[i])


@pytest.mark.skipif(not O.ref_particles_available(), reason="reference tree absent: golden vectors only")
@pytest.mark.parametrize("kind", range(5))
def test_oracle_constitutive_matches_reference_particles_live(kind):
    prm = O.ref_default_params(kind)
    strain, rate = {0: (0.08, 0.02), 1: (0.15, 0.02), 2: (0.05, 0.02), 3: (0.0, 0.03), 4: (0.01, 0.005)}[kind]
    states = G.golden_states(kind, strain, rate, count=150, seed=77)
    ref = [O.ref_particle_step(kind, prm, cdg, F, ps, G.VOL) for F, cdg, ps in states]
    scale = max(np.abs(r[2]).max() for r in ref)
    for (F, cdg, ps), (Fr, psr, fr) in zip(states, ref):
        F1, ps1, force = _oracle_step(kind, prm, cdg, F, ps, np.float64)
        if kind != scenes.MAT_WATER:
            assert np.abs(F1 - Fr).max() <= 2e-6
        assert abs(ps1 - psr) <= 3e-6 * max(1.0, abs(psr))
        assert np.abs(force - fr).max() <= FORCE_TOL[kind] * scale
        # and calculate_force alone (the upload-time call), without a plasticity step before it
        _, _, f0 = O.ref_particle_step(kind, prm, cdg, F, ps, G.VOL, do_plasticity=False)
        assert np.abs(O.calculate_force(kind, prm.astype(np.float64), F.astype(np.float64), float(ps), G.VOL, np.float64) - f0).max() <= FORCE_TOL[kind] * max(np.abs(f0).max(), scale)


def test_sand_alpha_and_defaults_live():
    from tests import common as T
    ref = T.live_ref("sand")                  # the reference's own values (tests/golden/make_live_golden.py sand_ref)
    for alpha, phi in zip(ref["alpha"], (10.0, 30.0, 45.0)):
        assert abs(alpha - scenes.material_params(scenes.MAT_SAND, friction_angle=phi)[2]) <= 1e-7
    for kind in range(5):
        assert np.allclose(ref["defaults"][kind], scenes.material_params(kind), rtol=3e-7, atol=0)
