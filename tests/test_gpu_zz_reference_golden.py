"""The CUDA engine against the REFERENCE ITSELF: tests/golden/transfer_ref.npz holds what the reference's own
MPM<3>::substep() (src/mpm.cpp + src/transfer.cpp + src/particles.cpp, compiled in place for the golden run,
oracle/transfer_ref.cpp) produced after 10 substeps of the stirred block with a friction floor and two
particles in the deletion band.  No oracle in between: same inputs through the C-ABI, same survivors, same state."""
import importlib.util
import os

import numpy as np
import pytest

from tests import common as T

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("make_transfer_golden", os.path.join(HERE, "golden", "make_transfer_golden.py"))
G = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(G)


@pytest.mark.parametrize("kind", G.KINDS)
def test_engine_matches_reference_substeps(kind):
    from tests import common as T
    from taichi_mpm_b200 import scenes
    z = np.load(os.path.join(HERE, "golden", "transfer_ref.npz"))
    scene, st = G.substep_scene(kind)
    e = T.make_engine(scene, st)
    e.substep(G.SUBSTEPS)
    got = e.download()
    e.close()
    ids = got["id"].astype(np.int64)
    assert np.array_equal(ids, z["k%d_sub_alive_ids" % kind])                     # the same two particles were deleted
    assert len(ids) == int(z["k%d_sub_alive" % kind]) == len(st["x"]) - 2
    ref = {k: z["k%d_sub_%s" % (kind, k)][ids] for k in ("x", "v", "F", "b", "ps")}
    # fp32 on both sides, different summation orders, 10 substeps: ten times the single-substep tolerances
    assert np.abs(got["x"] - ref["x"]).max() <= 1e-5
    assert np.abs(got["v"] - ref["v"]).max() <= 1e-3 * np.abs(ref["v"]).max()
    assert np.abs(got["b"] - ref["b"]).max() <= 2e-3 * np.abs(ref["b"]).max()
    if kind != scenes.MAT_WATER:
        assert np.abs(got["F"] - ref["F"]).max() <= 2e-4
    assert T.ps_err(got["ps"], ref["ps"]) <= (1e-3 if kind == scenes.MAT_VISCO else 1e-4)   # visco_tau hardening: see test_oracle_ref_transfer.py


@pytest.mark.parametrize("kind", G.KINDS)
def test_engine_single_substep_matches_reference_transfers(kind):
    """Per-substep grid momenta and particle state against the reference's transfer.cpp on identical inputs:
    the node (momentum, mass) after mpmb_rasterize vs rasterize_optimized, and the particle state after
    mpmb_resample vs resample_optimized (golden run; its G2P started from the oracle's node velocities)."""
    from tests import common as T
    from taichi_mpm_b200 import scenes
    z = np.load(os.path.join(HERE, "golden", "transfer_ref.npz"))
    scene, st = G.golden_scene(kind)
    e = T.make_engine(scene, st)
    e.sort_particles_and_populate_grid()
    e.rasterize()
    g0 = e.download_grid(0)
    ref_grid = G.dense(z["k%d_opt_grid_idx" % kind], z["k%d_opt_grid_val" % kind])
    pmax = max(np.abs(ref_grid[..., :3]).max(), ref_grid[..., 3].max())
    assert np.abs(g0 - ref_grid).max() <= T.TOL_GRID_REL * pmax
    m_ref = ref_grid[..., 3]
    assert (g0[..., 3][m_ref > 1e-9 * m_ref.max()] > 0).all() and not g0[m_ref == 0].any()   # the same nodes are touched
    e.resample()
    got = e.download()
    e.close()
    ids = got["id"].astype(np.int64)
    assert len(ids) == len(st["x"])
    ref = {k: z["k%d_opt_%s" % (kind, k)][ids] for k in ("x", "v", "F", "b", "ps")}
    assert np.abs(got["x"] - ref["x"]).max() <= 2 * T.TOL_X_ABS
    assert np.abs(got["v"] - ref["v"]).max() <= 2 * T.TOL_V_REL * np.abs(ref["v"]).max()
    assert np.abs(got["b"] - ref["b"]).max() <= 2 * T.TOL_V_REL * np.abs(ref["b"]).max()
    if kind != scenes.MAT_WATER:
        assert np.abs(got["F"] - ref["F"]).max() <= 2 * T.TOL_F_ABS
    assert T.ps_err(got["ps"], ref["ps"]) <= 2 * T.TOL_PS_ABS


def test_same_script_on_the_mirror_and_on_the_reference_solver():
    """The drop-in claim end to end: the verbs of a reference scene script (scripts/benchmark/benchmark_3d.py: create the
    solver, add_particles, step) run (a) on the reference's OWN MPM<3> object — its add_particles(benchmark=125), its
    substep(), compiled in place for the CPU (oracle/transfer_ref.cpp) — and (b) on the mirror MPM driving the CUDA
    engine through the C-ABI.  Same particles, same motion."""
    from taichi_mpm_b200 import MPM, scenes
    r = T.live_ref("bench_script")                                             # the reference's run (tests/golden/make_live_golden.py)
    res, dt, nsub = T.BENCH_SCRIPT["res"], T.BENCH_SCRIPT["dt"], T.BENCH_SCRIPT["nsub"]
    n = int(r["n"])
    lo = int(round(res * 0.4)); hi = lo + int(round(res * 0.2))
    x0, _, _ = scenes.lattice_block(res, (lo,) * 3, (hi,) * 3, 400.0, 0.0)
    m = MPM(res=(res, res, res), base_delta_t=dt, gravity=(0, -10, 0))
    m.add_particles(type="jelly", positions=x0, maximum=1, density=400.0)      # the benchmark path's volume: dx^3 / 1
    assert m.num_particles() == n == 8 ** 3 * 8
    for _ in range(nsub):
        m.step(-1.0)                                                           # dt < 0: exactly one substep
    p = m.get_particles()
    assert np.array_equal(p["id"], np.arange(n, dtype=p["id"].dtype)) and int(r["alive"]) == n
    ids = r["ids"]
    assert np.abs(p["x"][ids] - r["x"]).max() <= 1e-5
    assert np.abs(p["v"][ids] - r["v"]).max() <= 1e-3 * float(r["vmax"])
    assert np.abs(p["F"][ids] - r["F"]).max() <= 2e-4


def test_reference_solver_object_steps_through_libmpmb(tmp_path):
    """INTEGRATION.md §2 executed on the device: the reference's own MPM<3> object (CPU build, oracle/_ref) hands its AoS
    pool to libmpmb.so through the C-ABI and gets it back — against the same object stepping itself."""
    from oracle import pyoracle as O
    if not O.ref_transfer_available():
        pytest.skip("reference build (oracle/_ref) not available")
    from taichi_mpm_b200 import capi, scenes
    from tests.test_dropin import run_dropin
    capi.lib()
    run_dropin(capi.lib_path(), scenes.MAT_SAND, tmp_path)


def test_reference_solver_object_with_rigid_bodies_steps_through_libmpmb():
    """INTEGRATION.md §2c executed on the device: the reference's MPM<3> object with RigidBoundaryParticles in its pool and two
    bodies in MPM::rigids steps through libmpmb.so (samples, colours, rigid state in; velocities, colours, boundary out) — against
    the same object running its own rasterize_rigid_boundary / gather_cdf / block_op_rigid."""
    from oracle import pyoracle as O
    if not O.ref_transfer_available():
        pytest.skip("reference build (oracle/_ref) not available")
    from taichi_mpm_b200 import capi
    from tests.test_dropin import run_dropin_rigid
    capi.lib()
    run_dropin_rigid(capi.lib_path(), "two_bodies")


def test_reference_asyncmpm_scheduler_steps_through_libmpmb():
    """SURVEY §8f row 3 on the device: the reference's own AsyncMPM<3> scheduler (time levels, backup pools) with every
    MPM<3>::substep() it schedules run by libmpmb.so at the level's step — against the same scheduler on the reference's substep."""
    from oracle import pyoracle as O
    if not O.ref_transfer_available():
        pytest.skip("reference build (oracle/_ref) not available")
    from taichi_mpm_b200 import capi
    from tests.test_dropin import run_async
    capi.lib()
    run_async(capi.lib_path())
