"""SURVEY §8f row 3: the AsyncMPM scheduler of the mirror (taichi_mpm_b200/async_mpm.py) against the REFERENCE's own AsyncMPM<3>
object (src/async/async_mpm.{h,cpp} compiled in place, oracle/transfer_ref.cpp) — scheduler decisions identical (pool sizes,
update counter, integer clock, time levels, survivors), particle states to fp32 rounding.  What the reference computed is
committed (tests/golden/live_ref.npz, read through tests.common.live_ref).  The substeps of the mirror run on a
stand-in engine here that executes the oracle's fp32 substep on the CPU (no GPU in this suite); tests/test_gpu_async.py runs the
same comparison on the device engine."""
import numpy as np
import pytest

from oracle import pyoracle as O
from taichi_mpm_b200 import async_mpm, capi, scenes
from tests import common as T



class OracleEngine:
    """The Engine calls AsyncMPM makes, executed by the oracle (test infrastructure: the product has no CPU path)."""

    def __init__(self, res, dx, dt, gravity=(0.0, -10.0, 0.0), particle_gravity=True, clean_boundary=True, **kw):
        self.scene = dict(res=tuple(res), dx=dx, dt=dt, gravity=gravity, particle_gravity=int(particle_gravity), mat_kind=[], mat_params=[], sdf=None, friction=0.0)
        self.p = None

    def set_material(self, group, kind, params):
        while len(self.scene["mat_kind"]) <= group:
            self.scene["mat_kind"].append(0); self.scene["mat_params"].append(np.zeros(8, np.float32))
        self.scene["mat_kind"][group] = int(kind)
        q = np.zeros(8, np.float32); q[: len(params)] = params
        self.scene["mat_params"][group] = q

    def set_delta_t(self, dt):
        self.scene["dt"] = float(dt)

    def upload(self, x, v, mass, vol, F=None, b=None, scalar=None, group=None):
        n = len(x)
        self.p = dict(x=x, v=v, mass=mass, vol=vol, F=F, b=b, ps=scalar, group=np.zeros(n, np.int32) if group is None else group, alive=np.ones(n, np.uint8))

    def substep(self, n=1):
        sc = dict(self.scene, mat_kind=np.asarray(self.scene["mat_kind"], np.int32), mat_params=np.stack(self.scene["mat_params"]))
        for _ in range(n):
            self.p, _, _ = O.substep(sc, self.p, np.float32, want_grids=False)

    def download(self):
        a = self.p["alive"].astype(bool)
        out = {k: np.asarray(self.p[k])[a] for k in ("x", "v", "F", "b", "mass", "vol", "ps", "group")}
        out["id"] = np.nonzero(a)[0].astype(np.uint32)
        return out

    def close(self):
        pass


def async_pair(kind, steps, monkeypatch=None, engine_cls=None):
    """The scene, the reference's run of it (`steps` steps of AsyncMPM<3>, golden) and the mirror set up on the same state."""
    scene, st, unit, kw = T.async_inputs(kind)
    ref = T.live_ref("async_k%d_s%d" % (kind, steps))
    if engine_cls is not None:
        monkeypatch.setattr(capi, "Engine", engine_cls)
    m = async_mpm.AsyncMPM(res=(32, 32, 32), base_delta_t=unit, gravity=scene["gravity"], **kw)
    m.add_particles(type={scenes.MAT_SNOW: "snow", scenes.MAT_SAND: "sand"}[kind], positions=st["x"], density=400.0)
    for k in ("v", "mass", "vol", "F", "b", "ps"):
        m.pool[k][:] = st[k]                                   # the state the reference run starts from
    return scene, st, unit, ref, m


def compare_async(ref, m, unit, steps, tol):
    """ref: the reference's run (tests/golden/make_live_golden.py: async_ref): per-step decisions, survivors, a sample of particle states."""
    assert len(ref["decisions"]) == steps
    for r in ref["decisions"]:
        m.step(80 * unit)
        s = m.scheduler_stats()
        assert tuple(int(v) for v in r) == (s["pool_entries"], s["update_counter"], s["current_t_int"], s["min_level"], s["max_level"])
    assert s["min_level"] < s["max_level"]                    # really asynchronous
    pm = m.get_particles()
    assert np.array_equal(ref["alive_ids"], pm["id"])
    rows = np.searchsorted(pm["id"], ref["ids"])
    assert np.abs(ref["x"] - pm["x"][rows]).max() <= tol["x"]
    assert np.abs(ref["v"] - pm["v"][rows]).max() <= tol["v"] * float(ref["vmax"])
    assert np.abs(ref["F"] - pm["F"][rows]).max() <= tol["F"]
    assert m.update_counter == int(ref["decisions"][-1][1]) and m.num_particles() == len(pm["id"])


@pytest.mark.parametrize("kind", [scenes.MAT_SNOW, scenes.MAT_SAND])
def test_mirror_scheduler_makes_the_reference_s_decisions(kind, monkeypatch):
    scene, st, unit, ref, m = async_pair(kind, 2, monkeypatch, OracleEngine)
    compare_async(ref, m, unit, steps=2, tol=dict(x=2e-6, v=2e-5, F=5e-5))


def test_block_order_is_spgrid_s_and_types_without_a_limit_are_refused(monkeypatch):
    # the scheduler's block order (which copy of a particle wins a gather) is SPGrid's page order: y, x, z bits interleaved
    assert [int(async_mpm._morton(*c)) for c in ((0, 0, 0), (0, 1, 0), (1, 0, 0), (0, 0, 1), (1, 1, 1), (2, 0, 0), (0, 2, 0))] == [0, 1, 2, 4, 7, 16, 8]
    monkeypatch.setattr(capi, "Engine", OracleEngine)
    m = async_mpm.AsyncMPM(res=(32, 32, 32), base_delta_t=1e-5, unit_delta_t=1e-5)
    m.add_particles(type="jelly", benchmark_block=((12, 12, 12), (14, 14, 14)))
    with pytest.raises(ValueError):
        m.step(1e-4)                                          # JellyParticle::get_allowed_dt returns 0: the reference stops (TC_STOP, :124)


@pytest.mark.parametrize("kind", [scenes.MAT_SNOW, scenes.MAT_WATER, scenes.MAT_SAND, scenes.MAT_ELASTIC, scenes.MAT_VON_MISES, scenes.MAT_VISCO])
def test_strength_limit_is_the_reference_particle_s_get_allowed_dt(kind):
    # the per-particle limit the scheduler reads (src/async/async_mpm.cpp:105-110) against the reference's own classes run in place
    # (golden: tests/golden/make_live_golden.py strength_ref, which hands the reference F column-major, as the engine and the oracle carry it)
    F, ps, v, vol, mass, dx = T.strength_inputs(kind)
    got = async_mpm.allowed_dt(kind, scenes.material_params(kind), F.reshape(len(F), 9), ps, mass, vol, v, dx)   # the determinant does not care about the layout
    ref = T.live_ref("allowed_dt")["k%d" % kind]
    assert np.abs(got - ref).max() <= 2e-6 * ref.max()


def test_types_without_a_strength_limit_return_zero_in_the_reference_too():
    ref = T.live_ref("allowed_dt")
    for kind in (scenes.MAT_LINEAR, scenes.MAT_JELLY):
        assert ref["k%d" % kind] == 0.0
        with pytest.raises(ValueError):
            async_mpm.allowed_dt(kind, scenes.material_params(kind), np.eye(3, dtype=np.float32).reshape(1, 9), np.zeros(1, np.float32),
                                 np.ones(1, np.float32), np.ones(1, np.float32), np.zeros((1, 3), np.float32), 1 / 64)


def test_async_mirror_frame_dump_comes_from_the_pools(monkeypatch, tmp_path):
    from taichi_mpm_b200 import bgeo
    monkeypatch.setattr(capi, "Engine", OracleEngine)
    m = async_mpm.AsyncMPM(res=(32, 32, 32), base_delta_t=2.5e-5, unit_delta_t=2.5e-5, max_units=64, cfl_dt_mul=0.1, frame_directory=str(tmp_path))
    m.add_particles(type="snow", benchmark_block=((12, 12, 12), (16, 16, 16)), initial_velocity=(4.0, 0.0, 0.0))
    m.add_particles(type="snow", benchmark_block=((17, 12, 12), (20, 16, 16)))
    n = m.num_particles()
    m.step(40 * 2.5e-5)
    fn = m.visualize()
    pos, attrs = bgeo.read_bgeo(fn)
    p = m.get_particles()
    assert fn.endswith("0001.bgeo") and len(pos) == n == len(p["x"]) and np.array_equal(pos, p["x"])
    assert np.array_equal(dict((a[0], a[2]) for a in attrs)["index"].ravel(), np.arange(n))
    with pytest.raises(ValueError):
        m.general_action(action="save", file_name=str(tmp_path / "s.npz"))


def test_mirror_scheduler_follows_the_reference_through_deletions_and_level_changes(monkeypatch):
    # eight steps: the fast half of the block runs into the deletion band (4096 -> 3874 pool entries), levels regroup every step;
    # the two schedulers stay in lockstep (≈ 400 000 particle updates)
    scene, st, unit, ref, m = async_pair(scenes.MAT_SNOW, 8, monkeypatch, OracleEngine)
    compare_async(ref, m, unit, steps=8, tol=dict(x=5e-6, v=1e-4, F=2e-4))
    assert m.scheduler_stats()["pool_entries"] < 3900
