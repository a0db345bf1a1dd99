"""Frame output (SURVEY §8f row 1): the product's BGEO writer against the reference's own writer.

Golden files under tests/golden/ were written by the Partio copy vendored in the reference tree
(tests/golden/make_bgeo_golden.py); larger files of that writer, including the 65536-point switch of the primitive's
index width, and a frame of the reference solver's write_partio are pinned by size and SHA-256 (tests/golden/live_ref.npz,
tests/golden/make_live_golden.py)."""
import hashlib
import importlib.util
import os

import numpy as np
import pytest

from taichi_mpm_b200 import bgeo, mpm
from tests import common as T

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("make_bgeo_golden", os.path.join(HERE, "golden", "make_bgeo_golden.py"))
G = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(G)


def _same_file(data, ref):
    assert len(data) == int(ref["size"]) and hashlib.sha256(data).digest() == ref["sha256"].tobytes()


@pytest.mark.parametrize("name,n,seed,verbose", [("frame_plain_17", 17, 1, False), ("frame_verbose_9", 9, 2, True), ("frame_empty", 0, 3, False)])
def test_writer_reproduces_reference_files(tmp_path, name, n, seed, verbose):
    p = G.golden_particles(n, seed)
    out = tmp_path / (name + ".bgeo")
    nbytes = bgeo.write_bgeo(str(out), p["x"], mpm.frame_attributes(p, G.GROUP_KINDS, verbose))
    golden = open(os.path.join(HERE, "golden", name + ".bgeo"), "rb").read()
    assert nbytes == len(golden)
    assert out.read_bytes() == golden                     # bit-exact: byte work


def test_reader_round_trip_of_reference_file():
    p = G.golden_particles(9, 2)
    pos, attrs = bgeo.read_bgeo(os.path.join(HERE, "golden", "frame_verbose_9.bgeo"))
    assert np.array_equal(pos, p["x"])
    want = mpm.frame_attributes(p, G.GROUP_KINDS, True)
    assert [a[0] for a in attrs] == [a[0] for a in want]
    assert [a[0] for a in attrs[:4]] == ["type", "index", "limit", "v"]          # creation order, visualize.cpp:24-28
    for got, ref in zip(attrs, want):
        assert got[1] == ref[1] and np.array_equal(got[2].ravel(), np.asarray(ref[2]).ravel()), got[0]
    d = {a[0]: a[2] for a in attrs}
    assert np.array_equal(d["index"].ravel(), p["id"].astype(np.int32))
    assert set(np.unique(d["debug"][:, 1])) <= {4.0, 5.0, 6.0}                   # jelly / water / sand codes
    water = np.asarray(G.GROUP_KINDS)[p["group"]] == 3
    assert np.array_equal(d["debug"][water, 0], p["ps"][water]) and not d["debug"][~water, 0].any()


@pytest.mark.parametrize("n,verbose", T.BGEO_CASES)
def test_writer_equals_reference_writer_live(tmp_path, n, verbose):
    p = G.golden_particles(n, 40 + n % 7)
    attrs = mpm.frame_attributes(p, G.GROUP_KINDS, verbose)
    mine = tmp_path / "mine.bgeo"
    bgeo.write_bgeo(str(mine), p["x"], attrs)
    _same_file(mine.read_bytes(), T.live_ref("bgeo_n%d_v%d" % (n, verbose)))     # make_live_golden.py: bgeo_writer_ref


def test_writer_equals_write_partio_of_the_reference_solver_live(tmp_path):
    # the reference's MPM<3> (oracle/transfer_ref.cpp) steps a scene, deletes a particle, and dumps the frame with
    # its own write_partio (make_live_golden.write_partio_ref); the product's writer, given the same particle state,
    # produces the same bytes
    from taichi_mpm_b200 import scenes
    scene, st = T.write_partio_scene()
    p = T.live_ref("write_partio")
    ids = p["ids"]
    assert int(p["alive"]) == len(ids) == len(st["x"]) - 1
    d = dict(id=ids.astype(np.uint32), x=p["x"], v=p["v"], b=p["b"], mass=st["mass"][ids], ps=p["ps"], group=np.zeros(len(ids), np.int32))
    mine = tmp_path / "mine.bgeo"
    bgeo.write_bgeo(str(mine), d["x"], mpm.frame_attributes(d, [scenes.MAT_SAND], verbose=False))
    _same_file(mine.read_bytes(), p)


def test_read_rejects_other_files(tmp_path):
    f = tmp_path / "x.bgeo"
    f.write_bytes(b"PK\x03\x04 not a bgeo")
    with pytest.raises(ValueError):
        bgeo.read_bgeo(str(f))
