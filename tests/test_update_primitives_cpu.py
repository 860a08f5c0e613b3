"""trq_scene_update_primitives without a GPU: argument checks, and the host restatement (tests/update_util.update_on_host)
that the GPU tests hold the library to."""
import ctypes as C

import numpy as np
import pytest

from tracer_b200 import harness as H, layout as L
from tracer_b200._lib import ERR_INVALID, SceneDesc, lib

from .update_util import update_on_host

f32 = np.float32


def test_null_scene_or_changes_is_invalid(built):
    d = SceneDesc()
    assert lib.trq_scene_update_primitives(None, C.byref(d), 0) == ERR_INVALID
    assert lib.trq_scene_update_primitives(None, None, L.HOST_PTRS) == ERR_INVALID
    assert b"NULL" in lib.trq_last_error_string()


def _scenes():
    return {"c1": H.scene_c1(), "reference_cornell": H.scene_reference_cornell()}


@pytest.mark.parametrize("name", ["c1", "reference_cornell"])
def test_restatement_of_unchanged_lists_is_the_identity(built, name):
    prim = _scenes()[name]
    got = update_on_host(prim, spheres=prim.sphereList, squares=prim.squareList if prim.squareList.size else None,
                         cubes=prim.cubeList if prim.cubeList.size else None, verts=prim.triList if prim.triList.size else None)
    assert got.bvhList.tobytes() == prim.bvhList.tobytes(), name


def _moved_lists(prim, rng):
    sph = prim.sphereList.copy()
    off = rng.uniform(-0.5, 0.5, (sph.size, 3)).astype(f32)
    sph["center"] += off
    sph["box_mini"] += off
    sph["box_maxi"] += off
    sq = prim.squareList.copy()
    sq["box_mini"][:, 1] -= f32(7)
    sq["box_maxi"][:, 1] -= f32(7)
    cubes = prim.cubeList.copy()
    if cubes.size:
        cubes[0] = H.make_cube(H.translation4x4(200, 5, 300) @ H.rotation4x4(0.7, (0, 1, 0)) @ H.scale4x4(120, 300, 90), 0)
    return sph, sq, cubes


@pytest.mark.parametrize("name", ["c1", "reference_cornell"])
def test_restated_leaves_are_build_node_of_the_new_records(built, name):
    """Each sphere / square / cube leaf equals BVHBuilder.buildNode on its new record in its box fields, and keeps every
    other field; the root box is the union of the new leaves."""
    from tracer_b200.scene import BVHBuilder
    prim = _scenes()[name]
    sph, sq, cubes = _moved_lists(prim, np.random.default_rng(1))
    got = update_on_host(prim, spheres=sph, squares=sq if sq.size else None, cubes=cubes if cubes.size else None)
    old, new = prim.bvhList, got.bvhList
    checked = 0
    for p_type, arr in ((L.SPHERE, sph), (L.SQUARE, sq), (L.CUBE, cubes)):
        for i in np.nonzero(old["pType"] == p_type)[0]:
            b = BVHBuilder()
            p = int(old["pIndex"][i])
            b.buildNode(arr["box_mini"][p], arr["box_maxi"][p], arr["model"][p], p_type, p)
            want = b.leaves()[0]
            assert new["mini"][i].tobytes() == want["mini"].tobytes() and new["maxi"][i].tobytes() == want["maxi"].tobytes(), (name, i)
            checked += 1
    assert checked == int((old["pType"] != L.BVH).sum() - (old["pType"] == L.TRIANGLE).sum())
    rest = [k for k in L.bvh_dtype.names if k not in ("mini", "maxi")]
    for k in rest:
        assert new[k].tobytes() == old[k].tobytes(), (name, k)
    leaves = new[new["pType"] != L.BVH]
    assert np.array_equal(new["mini"][0], leaves["mini"].min(0)) and np.array_equal(new["maxi"][0], leaves["maxi"].max(0))
    assert not np.array_equal(new["mini"][0], old["mini"][0]) or not np.array_equal(new["maxi"][0], old["maxi"][0])
