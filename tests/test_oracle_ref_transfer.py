"""Pin of the oracle's 3-D substep against the REFERENCE's own solver core.  Transfers: src/transfer.cpp
rasterize_optimized / resample_optimized (block_op_normal, the SSE fast path the accelerated path
replaces) and the scalar rasterize / resample, compiled where they lie with src/mpm.h,
particle_allocator.h, kernel.h, particles.cpp and the vendored SPGrid (oracle/transfer_ref.cpp; the
stand-in core headers oracle/taichi_stub/taichi/*.h and the harness say what is scaffolding).
P2G: the node (momentum, mass) the reference scatters == the oracle's.  G2P: from the same node
velocities, the particle state the reference gathers (v, apic_b, F through plasticity, plastic scalar,
x) == the oracle's.  Golden vectors of that run are committed (tests/golden/transfer_ref.npz); where
the reference tree is present the loops also run live.
src/mpm.cpp is compiled the same way, so the rest of the substep is pinned too: the grid update
(normalize_grid_and_apply_external_force + apply_grid_boundary_conditions against a plane level set
with Coulomb friction), and whole substeps by MPM<3>::substep() itself — its own
sort_particles_and_populate_grid, optimized transfers, grid update and clear_boundary_particles — against
the oracle's substep(): the same survivors, the same trajectories."""
import importlib.util
import os

import numpy as np
import pytest

from oracle import pyoracle as O
from taichi_mpm_b200 import scenes
from tests import common as T

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("make_transfer_golden", os.path.join(HERE, "golden", "make_transfer_golden.py"))
G = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(G)

# measured against the fp64 oracle: grid 6e-7, x 3e-8, v 4e-7, F 3e-7, apic_b 8e-6, plastic scalar 5e-7 (visco_tau with hardening,
# relative: 4e-6 — the reference forms |P| - tau in fp32)
TOL = dict(grid=3e-6, x=2e-7, v=3e-6, F=2e-6, b=4e-5, ps=1e-5)


def _compare(scene, st, grid_ref, p_ref, rows=None):
    """rows: the particles p_ref holds (all when None)."""
    new, grid_rast, _ = O.substep(scene, st, np.float64)
    if rows is not None:
        new = {k: a[rows] for k, a in new.items()}
    pmax = max(np.abs(grid_rast[..., :3]).max(), grid_rast[..., 3].max())
    assert np.abs(grid_ref - grid_rast).max() <= TOL["grid"] * pmax
    assert (grid_ref[..., 3] > 0).sum() == (grid_rast[..., 3] > 0).sum()             # the same set of touched nodes
    assert np.abs(p_ref["x"] - new["x"]).max() <= TOL["x"]
    assert np.abs(p_ref["v"] - new["v"]).max() <= TOL["v"] * np.abs(new["v"]).max()
    assert np.abs(p_ref["b"] - new["b"]).max() <= TOL["b"] * np.abs(new["b"]).max()
    if int(scene["mat_kind"][0]) != scenes.MAT_WATER:                                # water carries no F
        assert np.abs(p_ref["F"] - new["F"]).max() <= TOL["F"]
    assert T.ps_err(p_ref["ps"], new["ps"]) <= TOL["ps"]


@pytest.mark.parametrize("kind", G.KINDS)
@pytest.mark.parametrize("tag", ["opt", "scalar"])
def test_oracle_transfers_match_golden_run_of_reference_loops(kind, tag):
    z = np.load(os.path.join(HERE, "golden", "transfer_ref.npz"))
    scene, st = G.golden_scene(kind)
    # the node velocities the golden G2P started from are the ones the oracle produces today
    gv_in = G.dense(z["k%d_grid_vel_in_idx" % kind], z["k%d_grid_vel_in_val" % kind])
    assert np.abs(G.oracle_grid_vel(scene, st) - gv_in).max() <= 1e-6 * max(np.abs(gv_in).max(), 1)
    p_ref = {k: z["k%d_%s_%s" % (kind, tag, k)] for k in ("x", "v", "F", "b", "ps")}
    _compare(scene, st, G.dense(z["k%d_%s_grid_idx" % (kind, tag)], z["k%d_%s_grid_val" % (kind, tag)]), p_ref)


def test_reference_fast_path_equals_its_scalar_path_in_the_golden_run():
    # "optimized" and readable versions of the reference agree with each other (same math, SURVEY §8c)
    z = np.load(os.path.join(HERE, "golden", "transfer_ref.npz"))
    for kind in G.KINDS:
        g0 = G.dense(z["k%d_opt_grid_idx" % kind], z["k%d_opt_grid_val" % kind])
        g1 = G.dense(z["k%d_scalar_grid_idx" % kind], z["k%d_scalar_grid_val" % kind])
        assert np.abs(g0 - g1).max() <= 2e-6 * np.abs(g1).max()
        for k in ("x", "v", "F", "ps"):
            a, b = z["k%d_opt_%s" % (kind, k)], z["k%d_scalar_%s" % (kind, k)]
            assert np.abs(a - b).max() <= 3e-6 * max(np.abs(b).max(), 1.0), (kind, k)


# after 10 substeps (fp32 reference vs fp64 oracle; measured x 3e-7, v 8e-7, F 2e-6, scalar 2e-6)
TOL_SUB = dict(x=2e-6, v=1e-5, F=1.5e-5, b=2e-4, ps=1.5e-5)


def _compare_substeps(scene, st, n_sub, alive, p_ref):
    cur = st
    for _ in range(n_sub):
        cur, _, _ = O.substep(scene, cur, np.float64)
    oa = np.nonzero(cur["alive"])[0]
    assert alive == len(oa) and np.array_equal(p_ref["alive_ids"], oa)               # the same particles were deleted
    assert alive < len(st["x"])                                                      # ... and some were
    s = oa
    assert np.abs(p_ref["x"][s] - cur["x"][s]).max() <= TOL_SUB["x"]
    assert np.abs(p_ref["v"][s] - cur["v"][s]).max() <= TOL_SUB["v"] * np.abs(cur["v"][s]).max()
    assert np.abs(p_ref["b"][s] - cur["b"][s]).max() <= TOL_SUB["b"] * np.abs(cur["b"][s]).max()
    if int(scene["mat_kind"][0]) != scenes.MAT_WATER:
        assert np.abs(p_ref["F"][s] - cur["F"][s]).max() <= TOL_SUB["F"]
    # visco_tau with hardening integrates kappa * gamma * |P| where gamma ~ (|P| - tau)/|P| is a difference of two O(1e3)
    # fp32 numbers: 2e-4 relative after 10 substeps between the fp32 reference and the fp64 oracle
    assert T.ps_err(p_ref["ps"][s], cur["ps"][s]) <= (5e-4 if int(scene["mat_kind"][0]) == scenes.MAT_VISCO else TOL_SUB["ps"])


@pytest.mark.parametrize("kind", G.KINDS)
def test_oracle_grid_update_matches_golden_run_of_reference(kind):
    # normalize_grid_and_apply_external_force + apply_grid_boundary_conditions (src/mpm.cpp:277-372) on the reference's own P2G
    z = np.load(os.path.join(HERE, "golden", "transfer_ref.npz"))
    scene, st = G.golden_scene(kind)
    ref = G.dense(z["k%d_gridupd_idx" % kind], z["k%d_gridupd_val" % kind])
    _, grid_rast, grid_vel = O.substep(scene, st, np.float64)
    act = grid_rast[..., 3] > 0
    assert np.abs(ref[..., :3] - grid_vel[..., :3])[act].max() <= 5e-6 * np.abs(grid_vel[..., :3]).max()
    assert np.abs(ref[..., 3] - grid_rast[..., 3]).max() <= 3e-6 * grid_rast[..., 3].max()    # the mass slot is kept
    # the floor really acted: some node normal velocities were projected
    free = grid_rast[..., :3][act] / grid_rast[..., 3][act][:, None]
    assert np.abs(free - grid_vel[..., :3][act]).max() > 1e-3


@pytest.mark.parametrize("kind", G.KINDS)
def test_oracle_substeps_match_golden_run_of_reference_substep(kind):
    z = np.load(os.path.join(HERE, "golden", "transfer_ref.npz"))
    scene, st = G.substep_scene(kind)
    p_ref = {k: z["k%d_sub_%s" % (kind, k)] for k in ("x", "v", "F", "b", "ps", "alive_ids")}
    _compare_substeps(scene, st, G.SUBSTEPS, int(z["k%d_sub_alive" % kind]), p_ref)


@pytest.mark.parametrize("kind", G.KINDS)
def test_timed_cpu_port_matches_golden_run_of_reference_substep(kind):
    # the fp32 OpenMP fast path that bench.py times as the CPU baseline (tile cache, 8-colour passes, SSE node
    # loops, periodic pool re-pack) is the reference's arithmetic: fp32 vs fp32, 10 substeps
    z = np.load(os.path.join(HERE, "golden", "transfer_ref.npz"))
    scene, st = G.substep_scene(kind)
    f = O.FastOracle(scene, st, threads=2, reorder_interval=1000)
    f.substeps(G.SUBSTEPS)
    ids = np.nonzero(f.st["alive"])[0]
    assert np.array_equal(ids, z["k%d_sub_alive_ids" % kind])
    ref = {k: z["k%d_sub_%s" % (kind, k)][ids] for k in ("x", "v", "F", "b", "ps")}
    assert np.abs(f.st["x"][ids] - ref["x"]).max() <= 5e-7
    assert np.abs(f.st["v"][ids] - ref["v"]).max() <= 5e-5 * np.abs(ref["v"]).max()
    assert np.abs(f.st["b"][ids] - ref["b"]).max() <= 3e-4 * np.abs(ref["b"]).max()
    assert np.abs(f.st["F"][ids] - ref["F"]).max() <= 3e-5
    assert T.ps_err(f.st["ps"][ids], ref["ps"]) <= (5e-4 if kind == scenes.MAT_VISCO else 5e-5)


def test_two_materials_in_one_scene_match_reference_substep_live():
    # sand resting next to water, each with its own registered particle type in the reference's allocator
    # (tests/common.py: two_materials_scene; the reference's 15 substeps are stored, a seeded sample of the particles)
    scene, st = T.two_materials_scene()
    p = T.live_ref("two_materials")
    cur = st
    for _ in range(15):
        cur, _, _ = O.substep(scene, cur, np.float64)
    ids = np.nonzero(cur["alive"])[0]
    assert int(p["alive"]) == len(ids) == len(st["x"]) and np.array_equal(p["alive_ids"], ids)
    s = p["ids"]
    assert np.abs(p["x"] - cur["x"][s]).max() <= TOL_SUB["x"]
    assert np.abs(p["v"] - cur["v"][s]).max() <= TOL_SUB["v"] * np.abs(cur["v"]).max()
    sand = st["group"][s] == 0
    assert np.abs(p["F"][sand] - cur["F"][s][sand]).max() <= TOL_SUB["F"]
    assert T.ps_err(p["ps"], cur["ps"][s]) <= TOL_SUB["ps"]


@pytest.mark.skipif(not O.ref_transfer_available(), reason="reference tree absent: golden vectors only")
@pytest.mark.parametrize("kind", [scenes.MAT_JELLY, scenes.MAT_SAND])
def test_oracle_substeps_match_reference_substep_live(kind):
    from tests import common as T
    scene, st = T.perturbed_scene(kind, res=32, cells=6, seed=7 + kind)
    st["x"][3] = [0.5, 6.2 / 32, 0.5]
    st["x"][4] = [(32 - 6.9) / 32, 0.5, 0.5]
    s = O.RefSolver(scene, st)
    alive = s.substep(25)
    p = s.particles()
    s.close()
    _compare_substeps(scene, st, 25, alive, p)


@pytest.mark.skipif(not O.ref_transfer_available(), reason="reference tree absent: golden vectors only")
@pytest.mark.parametrize("kind", [scenes.MAT_JELLY, scenes.MAT_SNOW, scenes.MAT_SAND])
def test_oracle_transfers_match_reference_loops_live(kind):
    from tests import common as T
    scene, st = T.perturbed_scene(kind, res=32, cells=6, seed=91 + kind)      # 1728 particles, other seeds than the golden run
    gv = G.oracle_grid_vel(scene, st)
    for opt in (True, False):
        grid, p = O.ref_transfer_substep(scene, st, gv, optimized=opt)
        _compare(scene, st, grid, p)


@pytest.mark.parametrize("friction", [-1.0, -2.0, -2.3, 0.0, 0.4, 5.0])
@pytest.mark.parametrize("particle_gravity", [1, 0])
def test_grid_update_modes_match_reference_live(friction, particle_gravity):
    # sticky (-1), slip (<= -2, with friction -mu-2), separate with Coulomb friction (>= 0): src/mpm_fwd.h:25-57 as
    # apply_grid_boundary_conditions uses it (src/mpm.cpp:296-372); gravity on the grid when particle_gravity is
    # off (src/mpm.cpp:519-527).  The reference's node velocities after its own P2G + grid update are stored.
    scene, st = T.grid_update_scene(friction, particle_gravity)
    _, grid_rast, grid_vel = O.substep(scene, st, np.float64)
    r = T.live_ref("grid_update_f%g_g%d" % (friction, particle_gravity))
    g = np.zeros((grid_rast[..., 0].size, 3), np.float32)
    g[r["idx"]] = r["vel"]
    g = g.reshape(grid_rast.shape[:3] + (3,))
    act = grid_rast[..., 3] > 0
    assert np.abs(g - grid_vel[..., :3])[act].max() <= 5e-6 * np.abs(grid_vel[..., :3]).max()


def test_lattice_generator_matches_reference_benchmark_seeding_live():
    # the synthetic BASELINE scenes use the reference's deterministic lattice (src/mpm.cpp:164-180): the reference's own
    # add_particles(benchmark=125) produces the same positions in the same order as scenes.lattice_block; its benchmark
    # path passes maximum = 1, i.e. vol = dx^3 per particle (an 8x over-dense block) — BASELINE.md keeps the positions
    # and uses the texture-seeding convention vol = dx^3 / 8 instead.  Stored: the count, a seeded sample of the
    # positions, and the extremes of the uniform fields.
    res = 40
    ref = T.live_ref("lattice")
    lo, hi = int(round(res * 0.4)), int(round(res * 0.4)) + int(round(res * 0.2))
    x, mass, vol = scenes.lattice_block(res, (lo,) * 3, (hi,) * 3, 400.0, 0.0)
    assert int(ref["n"]) == len(x) == 8 ** 3 * 8
    assert np.abs(ref["x"] - x[ref["ids"]]).max() <= 1.2e-7                # same lattice, same order (1 ulp)
    assert np.allclose(ref["vol_range"], (1.0 / res) ** 3, rtol=1e-6) and np.allclose(vol, (1.0 / res) ** 3 / 8, rtol=1e-6)
    assert np.allclose(ref["density_range"], 400.0, rtol=1e-6) and np.allclose(mass, vol * 400.0, rtol=1e-6)
    assert ref["v_absmax"] == 0 and ref["F_minus_identity_absmax"] == 0


def test_reference_loops_without_particle_gravity_live():
    # particle_gravity = false: P2G does not touch the particle velocity (src/transfer.cpp:485-487); the reference's
    # P2G grid and, for a seeded sample of the particles, its G2P result are stored
    scene, st = T.no_particle_gravity_scene()
    r = T.live_ref("no_particle_gravity")
    nn = tuple(int(v) + 1 for v in scene["res"])
    grid = np.zeros((int(np.prod(nn)), 4), np.float32)
    grid[r["grid_idx"]] = r["grid_val"]
    _compare(scene, st, grid.reshape(nn + (4,)), r, rows=r["ids"])
