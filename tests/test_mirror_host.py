"""Host logic of the frame output / snapshot verbs of the mirror (MPM.visualize, general_action
save/load) with the device engine replaced by an in-memory stand-in — no GPU, no arithmetic: what is
checked is the glue (file names and counters as src/mpm.h:333-343, id order, material groups and
clocks surviving a snapshot, unknown actions rejected as src/mpm.cpp:974)."""
import numpy as np
import pytest

from taichi_mpm_b200 import bgeo, capi, mpm as mpm_mod


class FakeEngine:
    """Stores what is uploaded; substep() only advects x by v*dt*n so that state visibly changes."""

    def __init__(self, res, dx, dt, gravity, particle_gravity, clean_boundary, device=0, capacity=0):
        self.res, self.dt = tuple(res), dt
        self.mats, self.id_base, self.p = {}, 0, None
        self.updates = 0

    def set_material(self, g, kind, params):
        self.mats[g] = (kind, np.array(params, np.float32))

    def set_sdf(self, *a):
        pass

    def set_planes(self, *a):
        pass

    def set_levelset_shapes(self, shapes, friction):
        self.shapes = (shapes, friction)

    def set_id_base(self, base):
        self.id_base = int(base)

    def upload(self, x, v, mass, vol, F, b, ps, group):
        n = len(x)
        self.p = dict(id=(self.id_base + np.arange(n)).astype(np.uint32), x=np.array(x, np.float32), v=np.array(v, np.float32),
                      F=np.array(F, np.float32).reshape(n, 9), b=np.array(b, np.float32).reshape(n, 9), mass=np.array(mass, np.float32),
                      vol=np.array(vol, np.float32), ps=np.array(ps, np.float32), group=np.array(group, np.int32))

    def num_particles(self):
        return 0 if self.p is None else len(self.p["x"])

    def download(self):
        if self.p is None:
            return dict(id=np.zeros(0, np.uint32), x=np.zeros((0, 3), np.float32), v=np.zeros((0, 3), np.float32), F=np.zeros((0, 9), np.float32),
                        b=np.zeros((0, 9), np.float32), mass=np.zeros(0, np.float32), vol=np.zeros(0, np.float32), ps=np.zeros(0, np.float32),
                        group=np.zeros(0, np.int32))
        rng = np.random.default_rng(0)
        o = rng.permutation(len(self.p["x"]))          # device order is arbitrary; download() sorts by id
        d = {k: a[o] for k, a in self.p.items()}
        s = np.argsort(d["id"], kind="stable")
        return {k: a[s].copy() for k, a in d.items()}

    def substep(self, n):
        self.p["x"] = (self.p["x"] + self.p["v"] * np.float32(self.dt * n)).astype(np.float32)
        self.updates += n * len(self.p["x"])

    def update_count(self):
        return self.updates

    def drop(self, ids):
        keep = ~np.isin(self.p["id"], ids)
        self.p = {k: a[keep] for k, a in self.p.items()}


@pytest.fixture
def fake_engine(monkeypatch):
    monkeypatch.setattr(capi, "Engine", FakeEngine)


def _scene(tmp_path, **kw):
    m = mpm_mod.MPM(res=(32, 32, 32), base_delta_t=1e-4, frame_directory=str(tmp_path / "frames"), **kw)
    m.add_particles(type="sand", benchmark_block=((10, 10, 10), (13, 13, 13)), initial_velocity=(0.1, 0.0, 0.0))
    m.add_particles(type="water", benchmark_block=((16, 10, 10), (18, 12, 12)), k=1e4)
    return m


def test_visualize_names_counts_and_contents(tmp_path, fake_engine):
    m = _scene(tmp_path, verbose_bgeo=True)
    m.step(1e-3)
    f1 = m.visualize()
    m.step(1e-3)
    f2 = m.visualize()
    assert f1.endswith("frames/0001.bgeo") and f2.endswith("frames/0002.bgeo") and m.frame_count == 2   # counter first, then the name
    p = m.get_particles()
    pos, attrs = bgeo.read_bgeo(f2)
    d = {a[0]: a[2] for a in attrs}
    assert np.array_equal(pos, p["x"]) and np.array_equal(d["v"], p["v"])
    assert np.array_equal(d["index"].ravel(), p["id"].astype(np.int32)) and (np.diff(d["index"].ravel()) > 0).all()
    assert np.array_equal(d["m"].ravel(), p["mass"]) and (d["limit"] == 1).all() and not d["type"].any()
    sand = p["group"] == 0
    assert (d["debug"][sand, 1] == 6).all() and (d["debug"][~sand, 1] == 5).all()
    pos1, _ = bgeo.read_bgeo(f1)
    assert not np.array_equal(pos1, pos)                                                                 # a frame later
    with pytest.raises(ValueError):
        mpm_mod.MPM(res=(32, 32, 32)).visualize()                                                        # no frame_directory


def test_snapshot_round_trip_restores_state_groups_and_clocks(tmp_path, fake_engine):
    m = _scene(tmp_path)
    m.step(1e-3)
    m.visualize()
    snap = str(tmp_path / "snap.npz")
    assert m.general_action(action="save", file_name=snap) == ""
    p = m.get_particles()
    m2 = mpm_mod.MPM(res=(32, 32, 32), base_delta_t=1e-4, frame_directory=str(tmp_path / "frames2"))
    assert m2.general_action(action="load", file_name=snap) == ""
    q = m2.get_particles()
    for k in p:
        assert np.array_equal(p[k], q[k]), k
    assert (m2.current_t, m2.request_t, m2.substep_counter, m2.frame_count) == (m.current_t, m.request_t, m.substep_counter, 1)
    assert [k for k, _ in m2._groups] == [k for k, _ in m._groups]
    assert all(np.array_equal(a[1], b[1]) for a, b in zip(m._groups, m2._groups))
    assert m2.engine.mats.keys() == m.engine.mats.keys()
    m.step(1e-3); m2.step(1e-3)
    assert np.array_equal(m.get_particles()["x"], m2.get_particles()["x"])
    assert m2.visualize().endswith("0002.bgeo")
    # adding particles of an already known material after a load reuses its group
    m2.add_particles(type="water", benchmark_block=((20, 10, 10), (21, 11, 11)), k=1e4)
    assert len(m2._groups) == 2 and m2.num_particles() == len(q["x"]) + 8


def test_snapshot_keeps_contiguous_ids_and_renumbers_gapped_ones(tmp_path, fake_engine):
    m = _scene(tmp_path)
    m.step(1e-3)
    n = m.num_particles()
    m.engine.drop(np.arange(0, 5))                       # deletions at the front: ids 5..n-1 stay contiguous
    snap = str(tmp_path / "a.npz")
    m.general_action(action="save", file_name=snap)
    m2 = mpm_mod.MPM(res=(32, 32, 32), base_delta_t=1e-4)
    m2.general_action(action="load", file_name=snap)
    assert np.array_equal(m2.get_particles()["id"], np.arange(5, n, dtype=np.uint32))
    m.engine.drop(np.array([40, 41]))                    # a gap: renumbered 0.. in id order
    m.general_action(action="save", file_name=snap)
    m3 = mpm_mod.MPM(res=(32, 32, 32), base_delta_t=1e-4)
    m3.general_action(action="load", file_name=snap)
    q, p = m3.get_particles(), m.get_particles()
    assert np.array_equal(q["id"], np.arange(n - 7, dtype=np.uint32)) and np.array_equal(q["x"], p["x"])


def test_unknown_action_and_foreign_snapshot_are_rejected(tmp_path, fake_engine):
    m = _scene(tmp_path)
    with pytest.raises(ValueError):
        m.general_action(action="cdf")
    m.general_action(action="save", file_name=str(tmp_path / "s.npz"))
    other = mpm_mod.MPM(res=(64, 64, 64), base_delta_t=1e-4)
    with pytest.raises(ValueError):
        other.general_action(action="load", file_name=str(tmp_path / "s.npz"))


# ---- the stepping / seeding verbs of the mirror, same stand-in engine (host logic only)
class CountingEngine(FakeEngine):
    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.calls = []

    def substep(self, n):
        self.calls.append(n)
        super().substep(n)


def test_step_runs_the_reference_number_of_substeps(monkeypatch, tmp_path):
    monkeypatch.setattr(capi, "Engine", CountingEngine)
    m = mpm_mod.MPM(res=(32, 32, 32), base_delta_t=1e-4)
    m.add_particles(type="jelly", benchmark_block=((10, 10, 10), (12, 12, 12)))
    # MPM<dim>::step (src/mpm.cpp:428-450): request_t += dt; while (current_t + base_delta_t < request_t) substep(),
    # every clock a `real` = float (src/mpm.h:100)
    f32 = np.float32

    def reference_count(current_t, request_t, dt, h):
        request_t = f32(request_t + f32(dt))
        n = 0
        while f32(current_t + f32(h)) < request_t:
            current_t = f32(current_t + f32(h))
            n += 1
        return n, current_t, request_t
    cur, req, total = f32(0.0), f32(0.0), 0
    for dt in (1e-3, 1e-3, 2.5e-4, 1e-4, 5e-5, 3.3e-3):
        n, cur, req = reference_count(cur, req, dt, 1e-4)
        m.step(dt)
        total += n
        assert m.substep_counter == total and m.current_t == cur and m.request_t == req
    assert sum(m.engine.calls) == total and all(c > 0 for c in m.engine.calls)      # one engine call per frame, never an empty one
    m.step(-1.0)                                                                    # dt < 0: exactly one substep (src/mpm.cpp:429-432)
    assert m.substep_counter == total + 1 and m.engine.calls[-1] == 1


def _mirror_counts(monkeypatch, h, dt, frames):
    monkeypatch.setattr(capi, "Engine", CountingEngine)
    m = mpm_mod.MPM(res=(32, 32, 32), base_delta_t=h)
    m.add_particles(type="jelly", benchmark_block=((10, 10, 10), (11, 11, 11)))
    out = []
    for _ in range(frames):
        before = m.substep_counter
        m.step(dt)
        out.append(m.substep_counter - before)
    return np.array(out, np.int32), m


def test_step_counts_match_the_reference_step_golden(monkeypatch):
    """Substeps per frame against MPM<3>::step of the reference sources compiled in place (tests/golden/make_step_golden.py):
    float clocks give 29996 substeps for 60 frames of 0.01 at base_delta_t = 2e-5, a double-precision loop 30000."""
    import os
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "step_ref.npz"))
    i = 0
    while "case%d" % i in z:
        h, dt, frames = z["case%d" % i]
        got, m = _mirror_counts(monkeypatch, float(h), float(dt), int(frames))
        assert np.array_equal(got, z["counts%d" % i]), (h, dt, got.sum(), z["counts%d" % i].sum())
        assert m.current_t == z["clocks%d" % i][0] and m.request_t == z["clocks%d" % i][1]
        i += 1
    assert i >= 4 and int(z["counts0"].sum()) == 29996


def test_step_counts_match_the_reference_step_live(monkeypatch):
    # a frame length that is not a multiple of the substep (tests/golden/make_live_golden.py: step_ref)
    from tests import common as T
    ref = T.live_ref("step")
    got, m = _mirror_counts(monkeypatch, *T.STEP_LIVE)
    assert np.array_equal(got, ref["counts"]) and m.current_t == ref["clocks"][0] and m.request_t == ref["clocks"][1]


def test_add_particles_follows_the_reference_rules(fake_engine):
    m = mpm_mod.MPM(res=(32, 32, 32), base_delta_t=1e-4)
    # particles within 7 cells of a face are ignored at seeding time (src/mpm.cpp:129-132, src/mpm.h:269-276)
    m.add_particles(type="snow", benchmark_block=((5, 10, 10), (9, 12, 12)))
    x = m.get_particles()["x"] * 32
    assert len(x) and x[:, 0].min() >= 7.0 and len(x) < 4 * 2 * 2 * 8
    n0 = m.num_particles()
    # positions= path: volume dx^3 / maximum, mass = volume * density (src/mpm.cpp:134-135)
    pts = np.array([[0.5, 0.5, 0.5], [0.51, 0.5, 0.5]], np.float32)
    m.add_particles(type="water", positions=pts, density=1000.0, maximum=4)
    p = m.get_particles()
    new = p["group"] == 1
    assert new.sum() == 2 and np.allclose(p["vol"][new], (1 / 32) ** 3 / 4) and np.allclose(p["mass"][new], (1 / 32) ** 3 / 4 * 1000.0)
    assert np.allclose(p["ps"][new], 1.0) and m.num_particles() == n0 + 2           # water starts at j = 1
    # same type + same parameters -> same material group; different parameters -> a new one
    m.add_particles(type="water", positions=pts + 0.1, density=1000.0)
    m.add_particles(type="water", positions=pts + 0.2, density=1000.0, k=5e3)
    assert [k for k, _ in m._groups] == [mpm_mod.scenes.MAT_SNOW, mpm_mod.scenes.MAT_WATER, mpm_mod.scenes.MAT_WATER]
    # all eight deformable types registered by the reference (src/particles.cpp:845-856) are accepted
    m.add_particles(type="von_mises", positions=pts + 0.05, yield_stress=2.0)
    m.add_particles(type="elastic", positions=pts + 0.06, E=1e4)
    m.add_particles(type="visco", positions=pts + 0.07, tau=500.0, kappa=0.1)
    p = m.get_particles()
    kinds = [k for k, _ in m._groups]
    assert kinds[3:] == [mpm_mod.scenes.MAT_VON_MISES, mpm_mod.scenes.MAT_ELASTIC, mpm_mod.scenes.MAT_VISCO]
    assert m._groups[3][1][2] == 2.0 and np.allclose(p["ps"][p["group"] == 5], 500.0)   # yield_stress; visco_tau is the scalar
    with pytest.raises(ValueError):
        m.add_particles(type="no_such_particle", positions=pts)
    with pytest.raises(ValueError):
        m.add_particles(type="rigid")


def test_unsupported_solver_options_are_rejected_not_ignored(fake_engine):
    for kw in (dict(optimized=False), dict(apic_damping=0.1), dict(rpic_damping=0.1), dict(res=(64, 64))):
        with pytest.raises(ValueError):
            mpm_mod.MPM(**{"res": (32, 32, 32), **kw})
    m = mpm_mod.MPM(res=(32, 32, 32))
    with pytest.raises(ValueError):
        m.set_levelset(m.create_levelset(), True)                                   # dynamic level set
    assert m.base_delta_t == float(np.float32(1e-4)) and m.gravity == (0.0, -10.0, 0.0)                # defaults of src/mpm.cpp:38,42
    assert m.get_debug_information() == "" and m.test() is True and m.get_name() == "mpm"   # the remaining verbs of the plugin surface
    assert mpm_mod.MPM(res=(32, 32, 32), gravity=-5, base_delta_t=1e-3, dt_multiplier=0.5).gravity == (0.0, -5.0, 0.0)


def test_driver_verbs_simulate_save_load_and_delete_inside_level_set(tmp_path, fake_engine):
    # scripts/async/async_mpm.py:217-299: the frame loop, save / load wrappers, delete_particles_inside_level_set (src/mpm.cpp:958-972)
    m = mpm_mod.MPM(res=(32, 32, 32), base_delta_t=1e-4, frame_dt=1e-3, frame_directory=str(tmp_path / "frames"))
    ls = m.create_levelset()
    ls.add_plane((0, 1, 0), -0.36)                      # obstacle below y = 0.36
    ls.set_friction(0.4)
    m.set_levelset(ls, False)
    m.add_particles(type="sand", benchmark_block=((10, 10, 10), (13, 14, 13)), initial_velocity=(0.0, 0.1, 0.0))
    n0 = m.num_particles()
    y = m.get_particles()["x"][:, 1]
    assert (y < 0.36).any() and (y > 0.36).any()
    m.delete_particles_inside_level_set()
    p = m.get_particles()
    assert 0 < len(p["x"]) < n0 and (p["x"][:, 1] >= 0.36 - 1e-6).all()
    assert np.abs(ls.sample(np.array([[16.0, 12.8, 16.0]])) - (12.8 - 0.36 * 32)) < 1e-4      # phi in grid units, trilinear = exact for a plane
    calls = []
    frames = m.simulate(num_frames=3, frame_update=lambda t, dt: calls.append((round(t, 6), dt)), update_frequency=2,
                        snapshot_interval=2, snapshot_directory=str(tmp_path / "snap"))
    assert frames == 3 and len(calls) == 6 and calls[0][0] == 0.0 and abs(calls[1][1] - 5e-4) < 1e-12
    assert sorted(f for f in (tmp_path / "frames").iterdir())[-1].name == "0003.bgeo" and (tmp_path / "snap" / "0002.npz").exists()
    m2 = mpm_mod.MPM(res=(32, 32, 32), base_delta_t=1e-4)
    m2.load(str(tmp_path / "snap" / "0002.npz"))
    assert m2.num_particles() == len(p["x"]) and m2.frame_count == 2
    with pytest.raises(ValueError):
        m.action(action="no_such_action")
