"""Regenerates tests/golden/live_ref.npz by RUNNING the reference's own code (the in-place builds under oracle/_ref,
`make -C oracle ref`) on the inputs of tests/common.py that the tests compare the product and the oracle with: the
AsyncMPM<3> scheduler, get_allowed_dt of the particle classes, the benchmark_3d.py script on MPM<3>, the Partio frame writer
and write_partio, MPM<3>::step, plasticity + calculate_force, the grid update in every boundary mode, MPM<3>::substep with two
materials, the transfers without particle gravity, the benchmark lattice, the rigid page map, the sand defaults and the
88-line program's own scene.  Tests read it with tests.common.live_ref(prefix).  Particle sets larger than SAMPLE keep a fixed
seeded sample (`ids`); frame files keep size and SHA-256.  Run from the repo root:  python tests/golden/make_live_golden.py"""
import hashlib
import importlib.util
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import pyoracle as O  # noqa: E402
from taichi_mpm_b200 import mpm, scenes  # noqa: E402
from tests import common as T  # noqa: E402

SAMPLE = 512


def _golden_module(name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(HERE, name + ".py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def sample_ids(n, seed=0, count=SAMPLE):
    return np.sort(np.random.default_rng(seed).choice(n, min(n, count), replace=False))


def sha256(path):
    return np.frombuffer(hashlib.sha256(open(path, "rb").read()).digest(), np.uint8)


def sparse(grid):
    """(flat node indices, values) of the nodes that hold anything."""
    flat = grid.reshape(grid.shape[0] * grid.shape[1] * grid.shape[2], -1)
    idx = np.nonzero(np.abs(flat).max(1) > 0)[0].astype(np.int32)
    return idx, flat[idx]


def async_ref(scene, st, unit, kw, steps):
    ref = O.RefAsyncSolver(scene, st, **kw)
    dec = []
    for _ in range(steps):
        r = ref.step(80 * unit)
        dec.append([r[k] for k in ("alive", "update_counter", "current_t_int", "min_level", "max_level")])
    p = ref.particles()
    ref.close()
    alive = np.nonzero(p["alive"])[0]
    ids = alive[sample_ids(len(alive), steps)]
    return {"decisions": np.array(dec, np.int64), "alive_ids": alive.astype(np.int32), "ids": ids.astype(np.int32),
            "x": p["x"][ids], "v": p["v"][ids], "F": p["F"][ids], "vmax": np.float32(np.abs(p["v"]).max())}


def strength_ref(kind):
    F, ps, v, vol, mass, dx = T.strength_inputs(kind)
    prm = scenes.material_params(kind)
    Fcm = np.ascontiguousarray(np.transpose(F, (0, 2, 1)).reshape(len(F), 9))     # column-major, as the engine and the oracle carry it
    return np.array([O.ref_allowed_dt(kind, prm, Fcm[i], float(ps[i]), float(mass[i]), float(vol[i]), v[i], dx) for i in range(len(F))], np.float32)


def bench_script_ref():
    c = T.BENCH_SCRIPT
    ref = O.RefSolver.from_benchmark(c["res"], c["dt"], (0.0, -10.0, 0.0), "jelly", benchmark=125, density=400.0)
    n = ref.n
    ref.substep(c["nsub"])
    r = ref.particles()
    ref.close()
    ids = sample_ids(n, 1)
    return {"n": np.int64(n), "alive": np.int64(len(r["alive_ids"])), "ids": ids.astype(np.int32), "x": r["x"][ids], "v": r["v"][ids],
            "F": r["F"][ids], "vmax": np.float32(np.abs(r["v"]).max())}


def bgeo_writer_ref(n, verbose, tmp):
    G = _golden_module("make_bgeo_golden")
    p = G.golden_particles(n, 40 + n % 7)
    d = {a[0]: a[2] for a in mpm.frame_attributes(p, G.GROUP_KINDS, verbose)}
    vb = {k: d[k] for k in ("m", "boundary_normal", "debug", "states", "boundary_distance", "near_boundary", "apic_frobenius_norm")} if verbose else None
    path = os.path.join(tmp, "ref.bgeo")
    O.ref_write_partio(path, p["x"], d["v"], d["type"], d["index"], d["limit"], vb)
    return {"size": np.int64(os.path.getsize(path)), "sha256": sha256(path)}


def write_partio_ref(tmp):
    scene, st = T.write_partio_scene()
    s = O.RefSolver(scene, st)
    alive = s.substep(5)
    path = os.path.join(tmp, "solver.bgeo")
    s.write_partio(path)
    p = s.particles()
    s.close()
    ids = p["alive_ids"]
    return {"alive": np.int64(alive), "ids": ids.astype(np.int32), "x": p["x"][ids], "v": p["v"][ids], "b": p["b"][ids], "ps": p["ps"][ids],
            "size": np.int64(os.path.getsize(path)), "sha256": sha256(path)}


def step_ref():
    counts, cur, req = _golden_module("make_step_golden").reference_counts(*T.STEP_LIVE)
    return {"counts": counts, "clocks": np.array([cur, req], np.float32)}


def material_ref(kind, strain, rate):
    prm = T.params8(kind)
    r = [O.ref_particle_step(kind, prm, cdg, F, ps, T.MATERIAL_VOL) for F, cdg, ps in T.material_states(kind, strain, rate)]
    return {"F": np.array([a[0] for a in r], np.float32), "ps": np.array([a[1] for a in r], np.float32), "force": np.array([a[2] for a in r], np.float32)}


def grid_update_ref(friction, particle_gravity):
    s = O.RefSolver(*T.grid_update_scene(friction, particle_gravity))
    s.p2g(True)
    s.grid_update()
    idx, val = sparse(s.get_grid())
    s.close()
    return {"idx": idx, "vel": val[:, :3]}      # the node velocities (the mass slot is the P2G's, pinned elsewhere)


def two_materials_ref():
    scene, st = T.two_materials_scene()
    s = O.RefSolver(scene, st)
    alive = s.substep(15)
    p = s.particles()
    s.close()
    ids = sample_ids(len(st["x"]), 15)
    return {"alive": np.int64(alive), "alive_ids": p["alive_ids"].astype(np.int32), "ids": ids.astype(np.int32), "x": p["x"][ids],
            "v": p["v"][ids], "F": p["F"][ids], "ps": p["ps"][ids], "vmax": np.float32(np.abs(p["v"]).max())}


def no_particle_gravity_ref():
    scene, st = T.no_particle_gravity_scene()
    _, _, gv = O.substep(scene, st, np.float64)
    grid, p = O.ref_transfer_substep(scene, st, np.ascontiguousarray(gv, np.float32), optimized=True)
    idx, val = sparse(grid)
    ids = sample_ids(len(st["x"]), 5, 256)
    return dict({"grid_idx": idx, "grid_val": val, "ids": ids.astype(np.int32)}, **{k: a[ids] for k, a in p.items()})


def lattice_ref(res=40):
    """Count and a sample of the positions; of the uniform fields, the extremes the test bounds."""
    r = O.ref_benchmark_particles(res, "sand", 125, 400.0)
    ids = sample_ids(len(r["x"]), 40, 1024)
    return {"n": np.int64(len(r["x"])), "ids": ids.astype(np.int32), "x": r["x"][ids], "vol_range": np.array([r["vol"].min(), r["vol"].max()], np.float32),
            "density_range": np.array([(r["mass"] / r["vol"]).min(), (r["mass"] / r["vol"]).max()], np.float32),
            "v_absmax": np.float32(np.abs(r["v"]).max()), "F_minus_identity_absmax": np.float32(np.abs(r["F"] - np.eye(3, dtype=np.float32).reshape(9)).max())}


def rigid_pages_ref():
    """(x, y, z) of the SPGrid pages update_rigid_page_map flags for the kinematic body, in the 9 x 9 x 5 window the test scans."""
    scene, st, rigid = _golden_module("make_rigid_golden").golden_scene("kinematic")
    s = O.RefSolver(scene, st)
    s.set_rigid(rigid)
    s.coupled_stage(0)
    got = [(x, y, z) for x in range(9) for y in range(9) for z in range(5) if s.is_rigid_page((4 * x, 4 * y, 8 * z))]
    s.close()
    return np.array(got, np.int32).reshape(-1, 3)


def sand_ref():
    L = O.ref_particles()
    return {"alpha": np.array([L.ref_sand_alpha(O.C.c_float(phi)) for phi in (10.0, 30.0, 45.0)], np.float32),
            "defaults": np.stack([O.ref_default_params(kind) for kind in range(5)])}


def mpm88_three_squares_ref():
    x, v, _, _, _, _ = O.ref88_run(*T.mpm88_three_squares(), 700, 0)
    return {"x": x, "v": v}


def main():
    out = {}

    def put(prefix, d):
        out.update({prefix + "/" + k: np.asarray(v) for k, v in d.items()})

    for kind, steps in T.ASYNC_CASES:
        put("async_k%d_s%d" % (kind, steps), async_ref(*T.async_inputs(kind), steps))
    for kind in T.STRENGTH_KINDS:
        out["allowed_dt/k%d" % kind] = strength_ref(kind)
    for kind in (scenes.MAT_LINEAR, scenes.MAT_JELLY):
        out["allowed_dt/k%d" % kind] = np.float32(O.ref_allowed_dt(kind, scenes.material_params(kind), np.eye(3).reshape(9), 0.0, 1e-3, 1e-6,
                                                                   np.zeros(3), 1 / 64))
    put("bench_script", bench_script_ref())
    with tempfile.TemporaryDirectory() as tmp:
        for n, verbose in T.BGEO_CASES:
            put("bgeo_n%d_v%d" % (n, verbose), bgeo_writer_ref(n, verbose, tmp))
        put("write_partio", write_partio_ref(tmp))
    put("step", step_ref())
    for i, case in enumerate(T.MATERIAL_CASES):
        put("material_c%d" % i, material_ref(*case))
    for friction in T.GRID_UPDATE_FRICTIONS:
        for pg in (1, 0):
            put("grid_update_f%g_g%d" % (friction, pg), grid_update_ref(friction, pg))
    put("two_materials", two_materials_ref())
    put("no_particle_gravity", no_particle_gravity_ref())
    put("lattice", lattice_ref())
    out["rigid_pages/kinematic"] = rigid_pages_ref()
    put("sand", sand_ref())
    put("mpm88_three_squares", mpm88_three_squares_ref())
    np.savez_compressed(T.LIVE_REF, **out)
    print(T.LIVE_REF, os.path.getsize(T.LIVE_REF), "bytes")


if __name__ == "__main__":
    main()
