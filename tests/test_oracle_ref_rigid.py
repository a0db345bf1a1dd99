"""Pin of the oracle's CPIC restatement (oracle/mpm_oracle.cpp, "CPIC rigid-coupled path") against the REFERENCE's own code:
update_rigid_page_map (src/mpm.cpp:1026-1076), rasterize_rigid_boundary + gather_cdf (src/rigid_transfer.cpp) and the
block_op_rigid branches of rasterize_optimized / resample_optimized (src/transfer.cpp:367-463, 706-835), run on the reference's
MPM<3> object compiled in place (oracle/transfer_ref.cpp).  Golden outputs of that run are committed
(tests/golden/rigid_ref.npz, generator next to it); where the reference tree is present the code is also run live.
What is NOT pinned: the RigidBody class itself (un-vendored core) — the stand-in's assumptions are listed in
oracle/taichi_stub/taichi/dynamics/rigid_body.h and repeated in include/mpmb.h."""
import importlib.util
import os

import numpy as np
import pytest

from oracle import pyoracle as O
from tests import common as T

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("make_rigid_golden", os.path.join(HERE, "golden", "make_rigid_golden.py"))
G = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(G)


def _golden(v, scene):
    z = np.load(os.path.join(HERE, "golden", "rigid_ref.npz"))
    nn = tuple(int(r) + 1 for r in scene["res"])
    ref = {k: z["%s_%s" % (v, k)] for k in ("x", "v", "F", "b", "ps", "alive", "states", "bnormal", "bdist", "near", "rigid_v", "rigid_w")}
    ref["grid_rast"] = G.dense(z[v + "_grid_idx"], z[v + "_grid_val"], nn + (4,))
    ref["grid_vel"] = G.dense(z[v + "_gvel_idx"], z[v + "_gvel_val"], nn + (4,))
    ref["node_state"] = G.dense(z[v + "_nstate_idx"], z[v + "_nstate_val"], nn)
    ref["node_dist"] = G.dense(z[v + "_ndist_idx"], z[v + "_ndist_val"], nn)
    return ref


def _compare(scene, st, rigid, ref):
    new, grid_rast, grid_vel, rs, cdf = O.substep_coupled(scene, st, rigid, np.float64)
    # discrete results: identical
    assert np.array_equal(cdf["node_state"], ref["node_state"]) and (ref["node_state"] >> 24 != 0).sum() > 200
    assert np.array_equal(new["states"], ref["states"]) and np.array_equal(new["near"], ref["near"]) and np.array_equal(new["alive"], ref["alive"])
    assert len(np.unique(ref["states"])) >= 3 and 0 < ref["near"].sum() < len(ref["near"])
    # continuous results: fp32 reference vs fp64 restatement (measured: distances 3e-8, normals 1.4e-5, grid 6e-7, v 2e-6, apic_b 1.3e-5)
    assert np.abs(cdf["node_dist"] - ref["node_dist"]).max() <= 2e-7
    assert np.abs(new["bdist"] - ref["bdist"]).max() <= 1e-6 and np.abs(new["bnormal"] - ref["bnormal"]).max() <= 1e-4
    pmax = max(np.abs(grid_rast[..., :3]).max(), grid_rast[..., 3].max())
    assert np.abs(grid_rast - ref["grid_rast"]).max() <= 3e-6 * pmax
    act = grid_rast[..., 3] > 0
    assert np.abs(grid_vel[..., :3] - ref["grid_vel"][..., :3])[act].max() <= 2e-5 * np.abs(grid_vel[..., :3]).max()   # nodes a colour mask leaves with little mass
    assert np.abs(new["x"] - ref["x"]).max() <= 2e-7
    assert np.abs(new["v"] - ref["v"]).max() <= 1e-5 * np.abs(new["v"]).max()
    assert np.abs(new["b"] - ref["b"]).max() <= 1e-4 * np.abs(new["b"]).max()
    assert np.abs(new["F"] - ref["F"]).max() <= 2e-6 and T.ps_err(new["ps"], ref["ps"]) <= 1e-5
    for b in range(1, len(rigid["inv_mass"])):
        dv, dw = rs["velocity"][b] - rigid["velocity"][b], rs["angular_velocity"][b] - rigid["angular_velocity"][b]
        assert np.abs(dv - (ref["rigid_v"][b] - rigid["velocity"][b])).max() <= 1e-4 * np.abs(dv).max() + 1e-7
        assert np.abs(dw - (ref["rigid_w"][b] - rigid["angular_velocity"][b])).max() <= 1e-4 * np.abs(dw).max() + 1e-6
        assert (np.abs(dv).max() > 1e-3) == (rigid["inv_mass"][b] > 0)      # scripted bodies take no impulse, free ones do
    # the coupling did something: against the same substep without bodies
    plain, pg, _ = O.substep(scene, st, np.float64)
    assert np.abs(pg - grid_rast).max() > 1e-2 * pmax and np.abs(plain["v"] - new["v"]).max() > 0.05 * np.abs(new["v"]).max()


@pytest.mark.parametrize("variant", G.VARIANTS)
def test_oracle_cpic_matches_golden_run_of_reference(variant):
    scene, st, rigid = G.golden_scene(variant)
    _compare(scene, st, rigid, _golden(variant, scene))


@pytest.mark.skipif(not O.ref_transfer_available(), reason="reference build (oracle/_ref) not available")
@pytest.mark.parametrize("variant", ["dynamic", "sand_preset"])
def test_oracle_cpic_matches_reference_live(variant):
    scene, st, rigid = G.golden_scene(variant)
    st["x"] = st["x"] + np.float32(0.0037)                     # not the golden positions
    new, grid_rast, grid_vel, rs, cdf = O.ref_substep_coupled(scene, st, rigid)
    ref = dict(new, grid_rast=grid_rast, grid_vel=grid_vel, node_state=cdf["node_state"], node_dist=cdf["node_dist"], rigid_v=rs["velocity"],
               rigid_w=rs["angular_velocity"])
    _compare(scene, st, rigid, ref)


def test_rigid_pages_are_the_reference_s_including_its_one_sided_dilation():
    # update_rigid_page_map tests the OFFSET of the neighbour loop against [0, spgrid_size) (src/mpm.cpp:1062), so a block with a
    # rigid particle flags itself and its upper neighbours only; the restatement follows that, and so does the engine
    # (the pages the reference flags in the scanned window are stored: tests/golden/make_live_golden.py rigid_pages_ref)
    scene, st, rigid = G.golden_scene("kinematic")
    pos = rigid["position"][rigid["sample_rigid"]] + rigid["sample_offset"] @ rigid["rot"][1].reshape(3, 3).T.T   # world anchors (one body)
    base = (pos * scene["res"][0] - 0.5).astype(int)
    blocks = {(b[0] >> 2, b[1] >> 2, b[2] >> 3) for b in base}
    expect = {(x + i, y + j, z + k) for (x, y, z) in blocks for i in (0, 1) for j in (0, 1) for k in (0, 1)}
    got = {tuple(int(c) for c in p) for p in T.live_ref("rigid_pages")["kinematic"]}
    assert got == expect and any((x - 1, y, z) not in got for (x, y, z) in blocks)
