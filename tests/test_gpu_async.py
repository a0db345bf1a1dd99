"""SURVEY §8f row 3 on the device: the mirror's AsyncMPM scheduler with its substeps on the engine (mpmb_set_delta_t per time
level) against the reference's own AsyncMPM<3> object (its run is committed: tests/golden/live_ref.npz) — same decisions, particle
states to fp32 rounding."""
import pytest

from taichi_mpm_b200 import scenes

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("kind", [scenes.MAT_SNOW, scenes.MAT_SAND])
def test_async_mirror_on_the_engine_matches_reference_asyncmpm(kind):
    from tests.test_async_host import async_pair, compare_async
    scene, st, unit, ref, m = async_pair(kind, 2)
    compare_async(ref, m, unit, steps=2, tol=dict(x=2e-6, v=2e-5, F=5e-5))
