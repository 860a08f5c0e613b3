"""Host-side mirror of the reference's ray-query interface, over the C-ABI.

  reference                                             here
  ----------------------------------------------------  ---------------------------------
  struct Primitive  (Render.hh:122-130)                 Primitive (six numpy arrays, reference layouts)
  BVH::buildNode / BVH::buildTree (BVH.hh:246-314)      BVHBuilder.buildNode / buildNodesTriangles / buildTree
  Scene { primitives }; scene.hit(ray, rec, test_t, any) (Render.hh:132-252)
                                                        Scene(primitives).hit(rays, any=False)  -- a BATCH of rays

Rays / hits live in device memory as torch tensors of shape (n, 8) float32 (32-byte trq_ray /
trq_hit rows), or in host memory as numpy structured arrays (`ray_dtype` / `hit_dtype`), in which
case the library stages the copies itself (TRQ_HOST_PTRS). All compute happens in the CUDA
kernels behind trq_trace; nothing here falls back to the CPU.
"""
import ctypes as C

import numpy as np

from . import layout as L
from ._lib import Camera, SceneDesc, SceneInfo, check, lib


def _ptr(a):
    return None if a is None or a.size == 0 else a.ctypes.data


def _device_arg(t, name, dtype, device, width=None, at_least=None, exactly=None):
    """Refuses a tensor the C-ABI would misread, before anything is launched: TypeError unless `t` is a contiguous CUDA
    tensor of `dtype` with shape (rows, width) (width None: one dimension); ValueError unless it is on cuda:`device` and has
    at least `at_least` (or exactly `exactly`) rows."""
    import torch
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError(f"{name} must be a CUDA tensor")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, not {t.dtype}")
    if not t.is_contiguous():
        raise TypeError(f"{name} must be contiguous")
    if (t.dim() != 1) if width is None else (t.dim() != 2 or t.shape[1] != width):
        raise TypeError(f"{name} must have shape {'(n,)' if width is None else f'(n, {width})'}, not {tuple(t.shape)}")
    if t.device.index != device:
        raise ValueError(f"{name} is on {t.device}, the scene on cuda:{device}")
    if at_least is not None and t.shape[0] < at_least:
        raise ValueError(f"{name} has {t.shape[0]} rows, needs at least {at_least}")
    if exactly is not None and t.shape[0] != exactly:
        raise ValueError(f"{name} has {t.shape[0]} rows, needs exactly {exactly}")
    return t


def _disjoint(outputs, inputs):
    """ValueError if an output shares a byte of memory with an input or with another output (dicts name -> tensor, None:
    absent): the kernels read the one while writing the other, and the spawns zero `count` on the stream before they read
    `count_in`. Inputs may share memory with each other: reading a buffer twice is harmless."""
    def spans(d):
        return [(k, t.data_ptr(), t.data_ptr() + t.numel() * t.element_size()) for k, t in d.items() if t is not None and t.numel()]
    outs, ins = spans(outputs), spans(inputs)
    for i, (a, lo, hi) in enumerate(outs):
        for b, lo2, hi2 in outs[i + 1:] + ins:
            if lo < hi2 and lo2 < hi:
                raise ValueError(f"{a} and {b} share memory")


def _morton(method):
    """True for method="morton" (the Morton-order builder), False for "sah" (the reference's binned-SAH builder)."""
    if method not in ("sah", "morton"):
        raise ValueError(f'method must be "sah" or "morton", not {method!r}')
    return method == "morton"


class Primitive:
    """The six arrays of `struct Primitive` (Render.hh:122-130), reference byte layouts."""

    def __init__(self, sphereList=None, squareList=None, cubeList=None, triList=None, idxList=None, bvhList=None):
        def arr(a, dt):
            if a is None:
                return np.zeros(0, dtype=dt)
            a = np.ascontiguousarray(a)
            if a.dtype != dt:
                raise TypeError(f"expected dtype {dt}, got {a.dtype}")
            return a
        self.sphereList = arr(sphereList, L.sphere_dtype)
        self.squareList = arr(squareList, L.square_dtype)
        self.cubeList = arr(cubeList, L.cube_dtype)
        self.triList = arr(triList, L.vertex_dtype)
        self.idxList = arr(None if idxList is None else np.asarray(idxList).reshape(-1), np.dtype("<u4"))
        self.bvhList = arr(bvhList, L.bvh_dtype)

    @property
    def nTri(self):
        return self.idxList.size // 3

    def desc(self):
        d = SceneDesc()
        d.sphereList, d.nSphere = _ptr(self.sphereList), self.sphereList.size
        d.squareList, d.nSquare = _ptr(self.squareList), self.squareList.size
        d.cubeList, d.nCube = _ptr(self.cubeList), self.cubeList.size
        d.triList, d.nVert = _ptr(self.triList), self.triList.size
        d.idxList, d.nTri = _ptr(self.idxList), self.nTri
        d.bvhList, d.nNode = _ptr(self.bvhList), self.bvhList.size
        return d

    def nbytes(self):
        return sum(a.nbytes for a in (self.sphereList, self.squareList, self.cubeList, self.triList, self.idxList, self.bvhList))


class DevicePrimitive:
    """`struct Primitive` whose six arrays already live on a GPU: torch uint8 CUDA tensors (or None) holding the reference
    byte layouts. Scene(DevicePrimitive) goes through trq_scene_create_device: nothing crosses PCIe."""

    _sizes = (("sphereList", L.sphere_dtype.itemsize), ("squareList", L.square_dtype.itemsize), ("cubeList", L.cube_dtype.itemsize),
              ("triList", L.vertex_dtype.itemsize), ("idxList", 12), ("bvhList", L.bvh_dtype.itemsize))

    def __init__(self, sphereList=None, squareList=None, cubeList=None, triList=None, idxList=None, bvhList=None):
        self.arrays = dict(sphereList=sphereList, squareList=squareList, cubeList=cubeList, triList=triList, idxList=idxList, bvhList=bvhList)
        for k, item in self._sizes:
            t = self.arrays[k]
            if t is not None and (not t.is_cuda or not t.is_contiguous() or t.numel() * t.element_size() % item):
                raise TypeError(f"{k}: expected a contiguous CUDA tensor holding whole {item}-byte records")

    @classmethod
    def from_host(cls, prim, device):
        """Uploads a host Primitive (for tests / for callers that build on the host but create on the device)."""
        import torch
        def up(a):
            return None if a.size == 0 else torch.from_numpy(a.view(np.uint8).reshape(-1).copy()).to(device)
        return cls(up(prim.sphereList), up(prim.squareList), up(prim.cubeList), up(prim.triList), up(prim.idxList), up(prim.bvhList))

    @classmethod
    def build(cls, sphereList=None, squareList=None, cubeList=None, triList=None, idxList=None, device=0, method="sah"):
        """BVH::buildNode + BVH::buildTree without leaving the GPU: the leaves are made on `device` in the order of
        harness.build_primitive (AAPLRenderer.mm:454-468,546-591) -- spheres, cubes, squares, then triangles, each kind
        numbered from pIndex 0 -- by trq_bvh_build_nodes_device / trq_bvh_build_nodes_triangles_device, and the tree by
        trq_bvh_build_tree_device (method="morton": trq_bvh_build_tree_morton_device). Arguments are torch uint8 CUDA tensors
        (or None) on `device` in the reference layouts. Returns the DevicePrimitive, ready for Scene(...)."""
        import torch
        from . import layout as L
        morton = _morton(method)
        prim = cls(sphereList, squareList, cubeList, triList, idxList)
        dev = torch.device(f"cuda:{int(device)}")
        for k, t in prim.arrays.items():
            if t is not None and t.device != dev:
                raise ValueError(f"{k} is on {t.device}, not {dev}")
        kinds = ((L.SPHERE, "sphereList"), (L.CUBE, "cubeList"), (L.SQUARE, "squareList"))
        n = sum(prim.count(k) for _, k in kinds) + prim.count("idxList")
        if n == 0:
            raise ValueError("DevicePrimitive.build: no primitives")
        item = L.bvh_dtype.itemsize
        bvh = torch.empty((2 * n - 1) * item, dtype=torch.uint8, device=dev)
        stream = torch.cuda.current_stream(dev)
        at = 0
        for p_type, k in kinds:
            m = prim.count(k)
            if m:
                check(lib.trq_bvh_build_nodes_device(p_type, prim.arrays[k].data_ptr(), m, 0, bvh.data_ptr() + at * item, int(device),
                                                     C.c_void_p(stream.cuda_stream)), "trq_bvh_build_nodes_device")
                at += m
        if prim.count("idxList"):
            check(lib.trq_bvh_build_nodes_triangles_device(prim.arrays["triList"].data_ptr(), prim.arrays["idxList"].data_ptr(),
                                                           prim.count("idxList"), 0, bvh.data_ptr() + at * item, int(device),
                                                           C.c_void_p(stream.cuda_stream)), "trq_bvh_build_nodes_triangles_device")
        stream.synchronize()                     # the tree build runs on the legacy default stream
        nNode, depth = C.c_uint32(0), C.c_uint32(0)
        fn = lib.trq_bvh_build_tree_morton_device if morton else lib.trq_bvh_build_tree_device
        check(fn(bvh.data_ptr(), n, int(device), C.byref(nNode), C.byref(depth)), fn.__name__)
        prim.arrays["bvhList"] = bvh
        prim.maxDepth = depth.value
        return prim

    def count(self, k):
        t = self.arrays[k]
        return 0 if t is None else t.numel() * t.element_size() // dict(self._sizes)[k]

    def desc(self):
        d = SceneDesc()
        ptr = lambda k: None if self.arrays[k] is None else self.arrays[k].data_ptr()
        d.sphereList, d.nSphere = ptr("sphereList"), self.count("sphereList")
        d.squareList, d.nSquare = ptr("squareList"), self.count("squareList")
        d.cubeList, d.nCube = ptr("cubeList"), self.count("cubeList")
        d.triList, d.nVert = ptr("triList"), self.count("triList")
        d.idxList, d.nTri = ptr("idxList"), self.count("idxList")
        d.bvhList, d.nNode = ptr("bvhList"), self.count("bvhList")
        return d


class BVHBuilder:
    """BVH::buildNode / BVH::buildTree (BVH.hh:246-314): leaves are appended, then the tree is built."""

    def __init__(self):
        self._chunks = []

    def leaves(self):
        return np.concatenate(self._chunks) if self._chunks else np.zeros(0, dtype=L.bvh_dtype)

    def buildNode(self, box_min, box_max, model_matrix, pType, pIndex):
        node = np.zeros(1, dtype=L.bvh_dtype)
        lo = np.ascontiguousarray(box_min, dtype=np.float32)
        hi = np.ascontiguousarray(box_max, dtype=np.float32)
        m = None if model_matrix is None else np.ascontiguousarray(model_matrix, dtype=np.float32).reshape(16)
        check(lib.trq_bvh_build_node(lo.ctypes.data, hi.ctypes.data, None if m is None else m.ctypes.data,
                                     int(pType), int(pIndex), node.ctypes.data), "trq_bvh_build_node")
        self._chunks.append(node)

    def buildNodesTriangles(self, triList, idxList, pIndexBase=0):
        idx = np.ascontiguousarray(np.asarray(idxList).reshape(-1), dtype="<u4")
        n = idx.size // 3
        nodes = np.zeros(n, dtype=L.bvh_dtype)
        if n:
            check(lib.trq_bvh_build_nodes_triangles(triList.ctypes.data, idx.ctypes.data, n, int(pIndexBase),
                                                    nodes.ctypes.data), "trq_bvh_build_nodes_triangles")
        self._chunks.append(nodes)

    def buildTree(self, gpu=None, method="sah"):
        """BVH::buildTree. gpu=None: host builder; gpu=<device index>: the same tree built on that GPU.
        method="morton": the Morton-order builder's tree instead (trq_bvh_build_tree_morton on the host; on a GPU,
        trq_bvh_build_tree_morton_device through a device copy)."""
        if _morton(method) and gpu is not None:
            d = self.buildTreeDevice(gpu, method)
            return d.cpu().numpy().view(L.bvh_dtype)
        leaves = np.concatenate(self._chunks) if self._chunks else np.zeros(0, dtype=L.bvh_dtype)
        n = leaves.size
        if n == 0:
            raise ValueError("buildTree: no leaves")
        nodes = np.zeros(2 * n - 1, dtype=L.bvh_dtype)
        nodes[:n] = leaves
        nNode, depth = C.c_uint32(0), C.c_uint32(0)
        if method == "morton":
            check(lib.trq_bvh_build_tree_morton(nodes.ctypes.data, n, C.byref(nNode), C.byref(depth)), "trq_bvh_build_tree_morton")
        elif gpu is None:
            check(lib.trq_bvh_build_tree(nodes.ctypes.data, n, C.byref(nNode), C.byref(depth)), "trq_bvh_build_tree")
        else:
            check(lib.trq_bvh_build_tree_gpu(nodes.ctypes.data, n, int(gpu), C.byref(nNode), C.byref(depth)), "trq_bvh_build_tree_gpu")
        self.maxDepth = depth.value
        return nodes[: nNode.value]

    def buildTreeDevice(self, device=0, method="sah"):
        """BVH::buildTree with the node array left ON the GPU (trq_bvh_build_tree_device; method="morton":
        trq_bvh_build_tree_morton_device): returns a torch uint8 CUDA tensor holding the 2n-1 64-byte nodes, ready for
        DevicePrimitive(bvhList=...)."""
        import torch
        morton = _morton(method)
        leaves = np.concatenate(self._chunks) if self._chunks else np.zeros(0, dtype=L.bvh_dtype)
        n = leaves.size
        if n == 0:
            raise ValueError("buildTree: no leaves")
        d = torch.zeros((2 * n - 1) * L.bvh_dtype.itemsize, dtype=torch.uint8, device=f"cuda:{device}")
        d[: n * L.bvh_dtype.itemsize] = torch.from_numpy(leaves.view(np.uint8).reshape(-1)).to(d.device)
        nNode, depth = C.c_uint32(0), C.c_uint32(0)
        fn = lib.trq_bvh_build_tree_morton_device if morton else lib.trq_bvh_build_tree_device
        check(fn(d.data_ptr(), n, int(device), C.byref(nNode), C.byref(depth)), fn.__name__)
        self.maxDepth = depth.value
        return d


class Scene:
    """`Scene { primitives }` (Render.hh:132-134), resident on one GPU."""

    def __init__(self, primitives, device=0):
        self.primitives = primitives
        self._h = C.c_void_p(None)
        d = primitives.desc()
        if isinstance(primitives, DevicePrimitive):
            check(lib.trq_scene_create_device(C.byref(d), int(device), C.byref(self._h)), "trq_scene_create_device")
        else:
            check(lib.trq_scene_create(C.byref(d), int(device), C.byref(self._h)), "trq_scene_create")
        self.device = int(device)
        self._read_info()

    def _read_info(self):
        info = SceneInfo()
        check(lib.trq_scene_info(self._h, C.byref(info)), "trq_scene_info")
        self.info = {k: getattr(info, k) for k, _ in SceneInfo._fields_}

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib.trq_scene_destroy(self._h)
            self._h = C.c_void_p(None)

    __del__ = close

    # ---- Scene::hit over a batch ------------------------------------------------------------
    def hit(self, rays, any=False, out=None, reflayout=False, stream=None, sort=None, hit16=False):
        """rays: torch CUDA float32 tensor (n, 8) -> returns torch CUDA float32 tensor (n, 8) holding
        trq_hit rows (view as int32 for the id fields); or numpy `ray_dtype` array -> numpy `hit_dtype`.
        hit16=True: the 16-byte trq_hit16 records instead ((n, 4) float32 tensor / `hit16_dtype` array).
        sort: True = TRQ_SORT_RAYS (the batch is incoherent), False = TRQ_NO_SORT, None = the library decides (large trees only)."""
        flags = (L.TRACE_ANY if any else 0) | (L.KERNEL_REFLAYOUT if reflayout else 0) | _sort_flag(sort) | (L.HIT16 if hit16 else 0)
        width = 4 if hit16 else 8
        if isinstance(rays, np.ndarray):
            if rays.dtype != L.ray_dtype:
                raise TypeError("host rays must have ray_dtype")
            rays = np.ascontiguousarray(rays)
            hits = out if out is not None else np.empty(rays.size, dtype=L.hit16_dtype if hit16 else L.hit_dtype)
            check(lib.trq_trace(self._h, rays.ctypes.data, rays.size, flags | L.HOST_PTRS, hits.ctypes.data, None), "trq_trace")
            return hits
        import torch
        _device_arg(rays, "rays", torch.float32, self.device, 8)
        n = rays.shape[0]
        if out is not None:
            _device_arg(out, "out", torch.float32, self.device, width, at_least=n)
            _disjoint(dict(out=out), dict(rays=rays))
        hits = out if out is not None else torch.empty((n, width), dtype=torch.float32, device=rays.device)
        st = stream if stream is not None else torch.cuda.current_stream(rays.device).cuda_stream
        check(lib.trq_trace(self._h, rays.data_ptr(), n, flags, hits.data_ptr(), C.c_void_p(st)), "trq_trace")
        return hits

    def update_vertices(self, triList):
        """Refit after the vertices moved (same topology): numpy `vertex_dtype` array or a torch uint8 CUDA tensor."""
        if isinstance(triList, np.ndarray):
            a = np.ascontiguousarray(triList)
            check(lib.trq_scene_update_vertices(self._h, a.ctypes.data, a.size, L.HOST_PTRS), "trq_scene_update_vertices")
        else:
            n = self._device_vertices(triList, "update_vertices")
            check(lib.trq_scene_update_vertices(self._h, triList.data_ptr(), n, 0), "trq_scene_update_vertices")

    def _device_vertices(self, triList, who):
        """-> the vertex count of a device vertex list, after the checks DevicePrimitive and update_primitives make."""
        DevicePrimitive(triList=triList)
        if triList.device.index != self.device:
            raise ValueError(f"{who}: triList is on {triList.device}, the scene on cuda:{self.device}")
        return triList.numel() * triList.element_size() // L.vertex_dtype.itemsize

    def update_primitives(self, spheres=None, squares=None, cubes=None, triList=None):
        """Refit after primitives moved (trq_scene_update_primitives, same topology): each argument given replaces that list
        of the scene whole (same count as the scene was created with); None keeps it. Either all numpy arrays of
        `sphere_dtype` / `square_dtype` / `cube_dtype` / `vertex_dtype`, or all torch uint8 CUDA tensors holding those
        layouts on the scene's device. Triangle leaves are refit as by update_vertices."""
        given = {k: a for k, a in (("sphereList", spheres), ("squareList", squares), ("cubeList", cubes), ("triList", triList))
                 if a is not None}
        host = [isinstance(a, np.ndarray) for a in given.values()]
        if any(host) and not all(host):
            raise TypeError("update_primitives: give either numpy arrays or CUDA tensors, not both")
        d = SceneDesc()
        if all(host):
            dtypes = dict(sphereList=L.sphere_dtype, squareList=L.square_dtype, cubeList=L.cube_dtype, triList=L.vertex_dtype)
            keep = []                            # the arrays must outlive the call
            for k, a in given.items():
                if a.dtype != dtypes[k]:
                    raise TypeError(f"{k}: expected dtype {dtypes[k]}, got {a.dtype}")
                a = np.ascontiguousarray(a)
                keep.append(a)
                setattr(d, k, a.ctypes.data)
                setattr(d, _COUNT[k], a.size)
            check(lib.trq_scene_update_primitives(self._h, C.byref(d), L.HOST_PTRS), "trq_scene_update_primitives")
        else:
            prim = DevicePrimitive(**given)
            for k, t in given.items():
                if t.device.index != self.device:
                    raise ValueError(f"update_primitives: {k} is on {t.device}, the scene on cuda:{self.device}")
            for k in given:
                setattr(d, k, prim.arrays[k].data_ptr())
                setattr(d, _COUNT[k], prim.count(k))
            check(lib.trq_scene_update_primitives(self._h, C.byref(d), 0), "trq_scene_update_primitives")

    def rebuild(self, triList=None, method="sah"):
        """New topology from the current geometry (trq_scene_rebuild), optionally after moving the vertices: numpy
        `vertex_dtype` array or a torch uint8 CUDA tensor holding all of the scene's vertices; None keeps them. Triangle leaf
        boxes follow the vertices, other leaves keep theirs. method="morton": the Morton-order builder builds the tree
        (TRQ_BUILD_MORTON), for a rebuild every frame. Refreshes `info`; on failure the scene is unchanged."""
        flags = L.BUILD_MORTON if _morton(method) else 0
        if triList is None:
            check(lib.trq_scene_rebuild(self._h, None, 0, flags), "trq_scene_rebuild")
        elif isinstance(triList, np.ndarray):
            a = np.ascontiguousarray(triList)
            check(lib.trq_scene_rebuild(self._h, a.ctypes.data, a.size, flags | L.HOST_PTRS), "trq_scene_rebuild")
        else:
            n = self._device_vertices(triList, "rebuild")
            check(lib.trq_scene_rebuild(self._h, triList.data_ptr(), n, flags), "trq_scene_rebuild")
        self._read_info()

    def bvh(self):
        """The scene's node array (trq_scene_copy_bvh) as a numpy `bvh_dtype` array."""
        nodes = np.empty(self.info["nNode"], dtype=L.bvh_dtype)
        check(lib.trq_scene_copy_bvh(self._h, nodes.ctypes.data, L.HOST_PTRS), "trq_scene_copy_bvh")
        return nodes

    @staticmethod
    def kernel_configs():
        """Names of the traversal kernel's launch configurations ("<CTA size>x<CTAs per SM><top of tree staged>")."""
        return [lib.trq_kernel_config_name(i).decode() for i in range(lib.trq_kernel_config_count())]

    def set_kernel_config(self, cfg=-1):
        """Selects a launch configuration (index; -1 = the library's choice). Returns the number of top-of-tree nodes that
        configuration stages in shared memory for this scene. Results are identical in every configuration."""
        staged = C.c_uint32(0)
        check(lib.trq_scene_set_kernel_config(self._h, int(cfg), C.byref(staged)), "trq_scene_set_kernel_config")
        return staged.value

    def kernel_config(self):
        """Name of the launch configuration this scene's traces use now."""
        return self.kernel_configs()[lib.trq_scene_kernel_config(self._h)]

    def host_sync(self):
        check(lib.trq_host_sync(self._h), "trq_host_sync")

    def hit_host(self, rays_ptr, n, hits_ptr, any=False, sort=False, asynchronous=False, hit16=False):
        """Raw host-pointer call (pinned buffers owned by the caller); used by the e2e bench."""
        flags = (L.TRACE_ANY if any else 0) | L.HOST_PTRS | (L.SORT_RAYS if sort else 0) | (L.HOST_ASYNC if asynchronous else 0) | (L.HIT16 if hit16 else 0)
        check(lib.trq_trace(self._h, rays_ptr, n, flags, hits_ptr, None), "trq_trace")

    # ---- wavefront callers (device tensors only) ----------------------------------------------
    def _stream(self, stream=None):
        import torch
        return C.c_void_p(stream if stream is not None else torch.cuda.current_stream(self.device).cuda_stream)

    def cast_rays(self, look_from, look_at, view_up, vfov, W, H, aperture=0.0, focus_dist=10.0, out=None, stream=None):
        """castRay for every pixel (Camera.hh:59-69, Render.metal:523-527) -> (W*H, 8) CUDA tensor of trq_ray."""
        import torch
        if out is not None:
            _device_arg(out, "out", torch.float32, self.device, 8, at_least=W * H)
        cam = Camera()
        cam.lookFrom[:], cam.lookAt[:], cam.viewUp[:] = look_from, look_at, view_up
        with np.errstate(divide="ignore", invalid="ignore"):             # H = 0 casts nothing
            aspect = float(np.float32(W) / np.float32(H))
        cam.vfov, cam.aspect, cam.aperture, cam.focus_dist = float(vfov), aspect, aperture, focus_dist
        rays = out if out is not None else torch.empty((W * H, 8), dtype=torch.float32, device=f"cuda:{self.device}")
        check(lib.trq_cast_rays(self._h, C.byref(cam), W, H, rays.data_ptr(), self._stream(stream)), "trq_cast_rays")
        return rays

    def hit_indirect(self, rays, count, any=False, out=None, sort=False, stream=None, hit16=False):
        """Scene::hit over min(*count, len(rays)) rays; `count` is a 1-element int64 CUDA tensor written by spawn_*."""
        import torch
        _device_arg(rays, "rays", torch.float32, self.device, 8)
        _device_arg(count, "count", torch.int64, self.device, exactly=1)
        if out is not None:
            _device_arg(out, "out", torch.float32, self.device, 4 if hit16 else 8, at_least=rays.shape[0])
        _disjoint(dict(out=out), dict(rays=rays, count=count))
        flags = (L.TRACE_ANY if any else 0) | (L.SORT_RAYS if sort else 0) | (L.HIT16 if hit16 else 0)
        hits = out if out is not None else torch.empty((rays.shape[0], 4 if hit16 else 8), dtype=torch.float32, device=rays.device)
        check(lib.trq_trace_indirect(self._h, rays.data_ptr(), count.data_ptr(), rays.shape[0], flags, hits.data_ptr(),
                                     self._stream(stream)), "trq_trace_indirect")
        return hits

    def _spawn(self, fn, rays, hits, count_in, seed_base, pixel_of, rng_state, extra, out, src, count, stream):
        import torch
        _device_arg(rays, "rays", torch.float32, self.device, 8)
        n = rays.shape[0]
        _device_arg(hits, "hits", torch.float32, self.device, 8, at_least=n)          # trq_hit rows; trq_hit16 is refused
        for name, t, dtype, width, rows in (("count_in", count_in, torch.int64, None, None), ("pixel_of", pixel_of, torch.int32, None, n),
                                            ("rng_state", rng_state, torch.int32, 4, n if pixel_of is None else None),
                                            ("out", out, torch.float32, 8, n), ("src", src, torch.int32, None, n),
                                            ("count", count, torch.int64, None, None)):
            if t is not None:
                _device_arg(t, name, dtype, self.device, width, at_least=rows, exactly=1 if name.startswith("count") else None)
        _disjoint(dict(rng_state=rng_state, out=out, src=src, count=count), dict(rays=rays, hits=hits, count_in=count_in, pixel_of=pixel_of))
        dev = rays.device
        out = out if out is not None else torch.empty((n, 8), dtype=torch.float32, device=dev)
        src = src if src is not None else torch.empty(n, dtype=torch.int32, device=dev)
        count = count if count is not None else torch.zeros(1, dtype=torch.int64, device=dev)
        args = [self._h, rays.data_ptr(), hits.data_ptr(), n, None if count_in is None else count_in.data_ptr(), int(seed_base),
                None if pixel_of is None else pixel_of.data_ptr(), None if rng_state is None else rng_state.data_ptr()]
        args += list(extra) + [out.data_ptr(), src.data_ptr(), count.data_ptr(), self._stream(stream)]
        check(fn(*args), fn.__name__)
        return out, src, count

    def rng_frame_begin(self, rng_state, stream=None):
        """Once per frame, before the first wave: the reference's toRNG entry conversion (halves of every texel swap)."""
        import torch
        _device_arg(rng_state, "rng_state", torch.int32, self.device, 4)
        check(lib.trq_rng_frame_begin(self._h, rng_state.data_ptr(), rng_state.shape[0], self._stream(stream)), "trq_rng_frame_begin")

    def spawn_bounce(self, rays, hits, seed_base=0, count_in=None, out=None, src=None, count=None, stream=None,
                     pixel_of=None, rng_state=None):
        """Diffuse bounce rays of the hits (Render.metal:447-475), compacted. -> (rays_out, srcIndex, count tensor).
        rng_state: (pixels, 4) int32 CUDA tensor in the reference's RNG texture format (Render.hh:96-120), advanced in
        place; pixel_of: int32 tensor mapping input ray -> pixel (then srcIndex holds pixels too)."""
        return self._spawn(lib.trq_spawn_bounce_rng, rays, hits, count_in, seed_base, pixel_of, rng_state, (), out, src, count, stream)

    def spawn_shadow(self, rays, hits, light_a, light_b, seed_base=0, count_in=None, out=None, src=None, count=None, stream=None,
                     pixel_of=None, rng_state=None):
        """NEE shadow rays toward squareList[light_a|light_b] (Render.metal:313-337), compacted."""
        return self._spawn(lib.trq_spawn_shadow_rng, rays, hits, count_in, seed_base, pixel_of, rng_state,
                           (int(light_a), int(light_b)), out, src, count, stream)

    def profile(self, on=True):
        check(lib.trq_profile_enable(self._h, 1 if on else 0), "trq_profile_enable")

    def profile_read(self):
        """-> (launches, trace_kernel_ms_sum, resolve_kernel_ms_sum) since the last read."""
        n, a, b = C.c_uint32(0), C.c_float(0), C.c_float(0)
        check(lib.trq_profile_read(self._h, C.byref(n), C.byref(a), C.byref(b)), "trq_profile_read")
        return n.value, a.value, b.value

    def expand(self, rays, hits, out=None, stream=None):
        """trq_expand_hits: HitRecord fields (p, gn, sn, uv, f, material) for the hits of `rays`."""
        if isinstance(rays, np.ndarray):
            recs = out if out is not None else np.empty(rays.size, dtype=L.record_dtype)
            check(lib.trq_expand_hits(self._h, rays.ctypes.data, hits.ctypes.data, rays.size, L.HOST_PTRS,
                                      recs.ctypes.data, None), "trq_expand_hits")
            return recs
        import torch
        _device_arg(rays, "rays", torch.float32, self.device, 8)
        n = rays.shape[0]
        _device_arg(hits, "hits", torch.float32, self.device, 8, at_least=n)
        if out is not None:
            _device_arg(out, "out", torch.float32, self.device, 16, at_least=n)
        _disjoint(dict(out=out), dict(rays=rays, hits=hits))
        recs = out if out is not None else torch.empty((n, 16), dtype=torch.float32, device=rays.device)
        st = stream if stream is not None else torch.cuda.current_stream(rays.device).cuda_stream
        check(lib.trq_expand_hits(self._h, rays.data_ptr(), hits.data_ptr(), n, 0, recs.data_ptr(), C.c_void_p(st)),
              "trq_expand_hits")
        return recs


_COUNT = dict(sphereList="nSphere", squareList="nSquare", cubeList="nCube", triList="nVert")


def _sort_flag(sort):
    return 0 if sort is None else (L.SORT_RAYS if sort else L.NO_SORT)


class MultiGpuScene:
    """trq_mgpu_*: one process, one scene per device, host rays sharded contiguously across the devices (no collective)."""

    def __init__(self, primitives, devices=None):
        self.primitives = primitives
        self._h = C.c_void_p(None)
        d = primitives.desc()
        if devices is None:
            check(lib.trq_mgpu_create(C.byref(d), None, 0, C.byref(self._h)), "trq_mgpu_create")
        else:
            arr = (C.c_int * len(devices))(*devices)
            check(lib.trq_mgpu_create(C.byref(d), arr, len(devices), C.byref(self._h)), "trq_mgpu_create")
        self.n_devices = lib.trq_mgpu_device_count(self._h)

    def shard(self, n, k):
        lo, hi = C.c_uint64(0), C.c_uint64(0)
        check(lib.trq_mgpu_shard(self._h, n, k, C.byref(lo), C.byref(hi)), "trq_mgpu_shard")
        return lo.value, hi.value

    def hit(self, rays, any=False, out=None, sort=False, hit16=False):
        """numpy `ray_dtype` array -> numpy `hit_dtype` (`hit16_dtype`) array (pinned buffers make the copies asynchronous)."""
        rays = np.ascontiguousarray(rays)
        hits = out if out is not None else np.empty(rays.size, dtype=L.hit16_dtype if hit16 else L.hit_dtype)
        flags = (L.TRACE_ANY if any else 0) | (L.SORT_RAYS if sort else 0) | (L.HIT16 if hit16 else 0)
        check(lib.trq_mgpu_trace(self._h, rays.ctypes.data, rays.size, flags, hits.ctypes.data), "trq_mgpu_trace")
        return hits

    def hit_ptr(self, rays_ptr, n, hits_ptr, any=False, sort=False):
        flags = (L.TRACE_ANY if any else 0) | (L.SORT_RAYS if sort else 0)
        check(lib.trq_mgpu_trace(self._h, rays_ptr, n, flags, hits_ptr), "trq_mgpu_trace")

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib.trq_mgpu_destroy(self._h)
            self._h = C.c_void_p(None)

    __del__ = close


def hits_to_numpy(hits):
    """torch (n, 8) float32 hit tensor -> numpy structured `hit_dtype` array (host copy)."""
    return hits.detach().cpu().numpy().view(L.hit_dtype).reshape(-1)


def rays_to_torch(rays, device):
    import torch
    return torch.from_numpy(np.ascontiguousarray(rays).view(np.float32).reshape(-1, 8)).to(device)


def probe_bandwidth(device=0, which="l2"):
    """Measured read bandwidth in GB/s: "l2" (32 MB working set) or "hbm" (2 GB)."""
    g = C.c_double(0)
    check(lib.trq_probe_bandwidth(int(device), 0 if which == "l2" else 1, C.byref(g)), "trq_probe_bandwidth")
    return g.value


def launch_count():
    return int(lib.trq_launch_count())
