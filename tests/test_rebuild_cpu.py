"""Argument checks of the device leaf builders and the scene rebuild, and the host restatement of the rebuild
(tests/rebuild_util.rebuild_on_host) that the GPU tests compare against. No GPU needed."""
import numpy as np
import pytest

from tracer_b200 import harness as H, layout as L
from tracer_b200._lib import ERR_INVALID, ERR_NO_DEVICE, lib

from .rebuild_util import reachable, rebuild_on_host
from .test_gpu_tree_shapes import refit_case, tree_case


def _message():
    return lib.trq_last_error_string()


def test_new_entry_points_refuse_bad_arguments(built):
    buf = np.zeros(4, dtype=L.bvh_dtype)
    assert lib.trq_scene_rebuild(None, None, 0, 0) == ERR_INVALID and b"NULL" in _message()
    assert lib.trq_scene_copy_bvh(None, buf.ctypes.data, L.HOST_PTRS) == ERR_INVALID and b"NULL" in _message()
    assert lib.trq_bvh_build_nodes_triangles_device(None, None, 5, 0, None, 0, None) == ERR_INVALID and b"NULL" in _message()
    for p_type in (L.TRIANGLE, L.BVH, L.UNKNOW, -1, 9):
        assert lib.trq_bvh_build_nodes_device(p_type, buf.ctypes.data, 1, 0, buf.ctypes.data, 0, None) == ERR_INVALID
        assert b"pType" in _message()
    for p_type in (L.SPHERE, L.SQUARE, L.CUBE):
        assert lib.trq_bvh_build_nodes_device(p_type, None, 3, 0, buf.ctypes.data, 0, None) == ERR_INVALID and b"NULL" in _message()
        assert lib.trq_bvh_build_nodes_device(p_type, buf.ctypes.data, 3, 0, None, 0, None) == ERR_INVALID
        assert lib.trq_bvh_build_nodes_device(p_type, None, 0, 0, None, 0, None) == 0          # n == 0: nothing to do
    assert lib.trq_bvh_build_nodes_triangles_device(None, None, 0, 0, None, 0, None) == 0


def test_device_leaf_builders_need_a_device(built):
    """No CPU fallback: on a box without a GPU the device leaf builders report TRQ_ERR_NO_DEVICE."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    prim = H.scene_soup(20, seed=1, extent=0.2)
    out = np.zeros(20, dtype=L.bvh_dtype)
    assert lib.trq_bvh_build_nodes_triangles_device(prim.triList.ctypes.data, prim.idxList.ctypes.data, 20, 0, out.ctypes.data,
                                                    0, None) == ERR_NO_DEVICE
    assert b"no CUDA device" in _message()
    spheres = H.cornell_spheres()
    assert lib.trq_bvh_build_nodes_device(L.SPHERE, spheres.ctypes.data, spheres.size, 0, out.ctypes.data, 0, None) == ERR_NO_DEVICE


@pytest.mark.parametrize("name", ["soup", "c1", "c2", "reference_cornell"])
def test_host_rebuild_of_a_builder_made_scene_is_the_identity(built, name):
    """The builder puts the leaves at 1..n in list order, so the leaf list of a rebuild is the original list and the
    tree comes out byte for byte."""
    prim = {"soup": lambda: H.scene_soup(3000, seed=5, extent=0.02), "c1": H.scene_c1, "c2": H.scene_c2,
            "reference_cornell": H.scene_reference_cornell}[name]()
    again = rebuild_on_host(prim)
    assert again.bvhList.tobytes() == prim.bvhList.tobytes(), name


@pytest.mark.parametrize("name", ["unreachable", "split-random-inf-odd"])
def test_host_rebuild_of_a_caller_built_tree(built, name):
    """Unreachable nodes drop out (2n - 1 nodes for n reachable leaves); leaves keep pType / pIndex and come in bvhList
    order at 1..n; every node is reachable afterwards."""
    prim = refit_case(name)[0] if name == "unreachable" else tree_case(name)[0]
    old = prim.bvhList
    leaves = np.nonzero(reachable(old) & (old["pType"] != L.BVH))[0]
    n = leaves.size
    new = rebuild_on_host(prim).bvhList
    assert new.size == 2 * n - 1 and (name != "unreachable" or new.size < old.size)
    assert reachable(new).all()
    assert np.array_equal(new["pType"][1:n + 1], old["pType"][leaves]) and np.array_equal(new["pIndex"][1:n + 1], old["pIndex"][leaves])
    other = old["pType"][leaves] != L.TRIANGLE
    assert np.array_equal(new["mini"][1:n + 1][other].view(np.uint32), old["mini"][leaves][other].view(np.uint32))
    assert not new["axis"][1:n + 1].any() and not new["pad"][1:n + 1].any() and not new["left"][1:n + 1].any()
