"""Python mirror of the reference's operator interface for the hot path, over the C-ABI.

Names, argument meaning and error behaviour follow tiny_bvh.h: `BVH.Build(verts, primCount)` (:2124),
`BVH.Intersect` (:3222) / `IsOccluded` (:3382) - here over whole `Ray` batches (the reference has per-ray calls only;
its GPU "batch" is a kernel launch, tiny_bvh_speedtest.cpp:1092-1241) -, `BVH_GPU.ConvertFrom` (:4612),
`BVH8_CWBVH.ConvertFrom` (:5884).  Rays are numpy arrays of the 128-byte host record (rays.RAY_DTYPE) or torch CUDA
tensors of 64-/128-byte records.  Errors raise TbvhError (the reference prints and exit(1)s, :1617-1620).
"""
from __future__ import annotations

import ctypes as C
import numpy as np

from . import _lib
from ._lib import LAYOUT_BVH, LAYOUT_BVH_GPU, LAYOUT_CWBVH, HOST, DEVICE, TbvhError, check

NODE32 = np.dtype([("aabbMin", "3f4"), ("leftFirst", "u4"), ("aabbMax", "3f4"), ("triCount", "u4")])
NODE64 = np.dtype([("lmin", "3f4"), ("left", "u4"), ("lmax", "3f4"), ("right", "u4"),
                   ("rmin", "3f4"), ("triCount", "u4"), ("rmax", "3f4"), ("firstTri", "u4")])

_contexts = {}


def context(device: int = 0):
    """One engine context per CUDA device (lazily created)."""
    if device not in _contexts:
        h = C.c_void_p()
        check(_lib.lib().tbvh_ctx_create(device, C.byref(h)))
        _contexts[device] = h
    return _contexts[device]


def set_option(key: str, value: int, device: int = 0) -> None:
    """Option of the engine context (tbvh_set_option): inst_idx_bits, small_t or build_mode; any other key raises TbvhError."""
    check(_lib.lib().tbvh_set_option(context(device), key.encode(), int(value)))


def device_count() -> int:
    return _lib.lib().tbvh_device_count()


def launch_count() -> int:
    return int(_lib.lib().tbvh_launch_count())


def _np_ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


def _verts_arg(verts):
    """-> (pointer, stride, vertex count, space, keepalive)"""
    if _is_torch(verts):
        import torch
        assert verts.is_cuda and verts.is_contiguous() and verts.dtype.is_floating_point and verts.element_size() == 4
        v = verts.reshape(-1, 4)
        # device-space inputs are read on the engine's own stream (include/tinybvh_b200.h "device-space inputs"): whatever torch
        # has queued to produce them must have finished
        torch.cuda.current_stream(verts.device).synchronize()
        return C.c_void_p(v.data_ptr()), 16, v.shape[0], DEVICE, v
    v = np.ascontiguousarray(verts, np.float32).reshape(-1, 4)
    return _np_ptr(v), 16, v.shape[0], HOST, v


class _Base:
    layout = LAYOUT_BVH
    build_flavour = _lib.BUILD_AVX   # derived layouts build through BuildDefault; set to _lib.BUILD_REFERENCE for BVH::Build's tree

    def __init__(self, device: int = 0):
        self.device = device
        self.ctx = context(device)
        self.h = C.c_void_p()
        check(_lib.lib().tbvh_bvh_create(self.ctx, C.byref(self.h)))
        self.c_trav, self.c_int = 1.0, 1.0  # BVHBase::c_trav / c_int (:819-820)

    def _build(self, vertices, primCount, flavour, indices=None):
        """tbvh_build_flavour, or tbvh_build_indexed for the (vertices, indices, primCount) overloads (tiny_bvh.h:889-900)."""
        p, stride, nv, space, keep = _verts_arg(vertices)
        if indices is None:
            check(_lib.lib().tbvh_build_flavour(self.h, p, stride, primCount or nv // 3, space, self.c_trav, self.c_int, flavour))
            return
        if _is_torch(indices):
            assert space == DEVICE and indices.is_cuda and indices.is_contiguous() and indices.element_size() == 4
            ip, ni = C.c_void_p(indices.data_ptr()), indices.numel()
        else:
            assert space == HOST, "device vertices need device indices"
            indices = np.ascontiguousarray(indices, np.uint32).reshape(-1)
            ip, ni = _np_ptr(indices), indices.shape[0]
        check(_lib.lib().tbvh_build_indexed(self.h, p, stride, nv, ip, primCount or ni // 3, space, self.c_trav, self.c_int, flavour))

    def __del__(self):
        try:
            if getattr(self, "h", None) and self.h.value:
                _lib.lib().tbvh_bvh_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # -- info (the reference's public members usedNodes / idxCount / triCount / aabbMin / aabbMax)
    def info(self) -> _lib.Info:
        i = _lib.Info()
        check(_lib.lib().tbvh_bvh_info(self.h, C.byref(i)))
        return i

    usedNodes = property(lambda s: s.info().used_nodes)
    idxCount = property(lambda s: s.info().idx_count)
    triCount = property(lambda s: s.info().prim_count)

    # -- traversal over batches
    def Intersect(self, rays, hits=None, stream=None):
        """Closest hit for every ray, in place (t,u,v,prim at bytes 48..63).  numpy -> host path (copies inside);
        torch CUDA tensor -> device path, asynchronous on `stream` (default: torch's current stream)."""
        L = _lib.lib()
        if _is_torch(rays):
            import torch
            assert rays.is_cuda and rays.is_contiguous()
            stride = rays.stride(0) * rays.element_size() if rays.dim() > 1 else None
            assert stride in (64, 128), "ray tensor must be [n, 64|128 bytes]"
            st = stream if stream is not None else torch.cuda.current_stream(rays.device).cuda_stream
            hp = C.c_void_p(hits.data_ptr()) if hits is not None else None
            check(L.tbvh_intersect_device(self.h, self.layout, C.c_void_p(rays.data_ptr()), stride, hp, rays.shape[0], C.c_void_p(st)))
            return rays if hits is None else hits
        assert rays.dtype.itemsize in (64, 128) and rays.flags.c_contiguous
        check(L.tbvh_intersect(self.h, self.layout, _np_ptr(rays), rays.dtype.itemsize, rays.shape[0]))
        return rays

    def IntersectPacked(self, rays, hits=None):
        """Host path with packed results: rays untouched, hits -> HIT_DTYPE array (tbvh_intersect_packed)."""
        from .rays import HIT_DTYPE
        assert not _is_torch(rays) and rays.dtype.itemsize in (64, 128) and rays.flags.c_contiguous
        if hits is None:
            hits = np.zeros(rays.shape[0], HIT_DTYPE)
        check(_lib.lib().tbvh_intersect_packed(self.h, self.layout, _np_ptr(rays), rays.dtype.itemsize, rays.shape[0], _np_ptr(hits)))
        return hits

    def IsOccluded(self, rays, bits=None, stream=None):
        """Any hit within [0, ray.hit.t] per ray -> uint32 bit mask, bit (i&31) of word i>>5."""
        L = _lib.lib()
        if _is_torch(rays):
            import torch
            assert rays.is_cuda and rays.is_contiguous()
            stride = rays.stride(0) * rays.element_size()
            n = rays.shape[0]
            if bits is None:
                bits = torch.empty((n + 31) // 32, dtype=torch.int32, device=rays.device)
            st = stream if stream is not None else torch.cuda.current_stream(rays.device).cuda_stream
            check(L.tbvh_occluded_device(self.h, self.layout, C.c_void_p(rays.data_ptr()), stride, C.c_void_p(bits.data_ptr()), n, C.c_void_p(st)))
            return bits
        assert rays.dtype.itemsize in (64, 128) and rays.flags.c_contiguous
        n = rays.shape[0]
        if bits is None:
            bits = np.zeros((n + 31) // 32, np.uint32)
        check(L.tbvh_occluded(self.h, self.layout, _np_ptr(rays), rays.dtype.itemsize, n, _np_ptr(bits)))
        return bits

    def set_stats(self, enable: bool):
        check(_lib.lib().tbvh_set_stats(self.h, int(enable)))

    def get_stats(self):
        """(node visits, triangle tests, CWBVH child-pair steps) of the last traversal call with statistics enabled"""
        out = (C.c_uint64 * 4)()
        check(_lib.lib().tbvh_get_stats_ex(self.h, C.byref(out)))
        return out[0], out[1], out[2]


class BVH(_Base):
    """tinybvh::BVH (tiny_bvh.h:846-985): Wald 32-byte nodes; binned-SAH Build on the GPU."""
    layout = LAYOUT_BVH

    def Build(self, vertices, primCount: int = 0, indices=None):
        """BVH::Build( vertices, primCount ) :2124 / ( vertices, indices, primCount ) :2139."""
        self._build(vertices, primCount, _lib.BUILD_REFERENCE, indices)
        return self

    def BuildAVX(self, vertices, primCount: int = 0, indices=None):
        """BVH::BuildAVX (tiny_bvh.h:6400) - the flavour BuildDefault uses on x86."""
        self._build(vertices, primCount, _lib.BUILD_AVX, indices)
        return self

    def BuildHQ(self, vertices, primCount: int = 0, indices=None):
        """BVH::BuildHQ (tiny_bvh.h:2623): SBVH with spatial splits; idxCount becomes primCount + primCount/2."""
        self._build(vertices, primCount, _lib.BUILD_HQ, indices)
        return self

    def SAHCost(self) -> float:
        """BVH::SAHCost( 0 ) (tiny_bvh.h:1889): host recursion over the downloaded nodes, the reference's value bit for bit."""
        out = C.c_float()
        check(_lib.lib().tbvh_sah_cost(self.h, self.c_trav, self.c_int, C.byref(out)))
        return float(out.value)

    def Refit(self, vertices):
        """BVH::Refit (tiny_bvh.h:3055): same triangles, new positions.  The reference re-reads the caller's vertex array through
        the pointer it kept; the engine holds its own copy, so the array is passed again."""
        p, stride, nv, space, keep = _verts_arg(vertices)
        check(_lib.lib().tbvh_refit(self.h, p, stride, nv // 3, space))
        return self

    def upload(self, nodes, primIdx, vertices):
        """Consume a tree built elsewhere in the reference's BVH layout (bvhNode / primIdx / verts, :952-964)."""
        p, stride, nv, space, keep = _verts_arg(vertices)
        nodes = np.ascontiguousarray(nodes)
        primIdx = np.ascontiguousarray(primIdx, np.uint32)
        assert nodes.dtype.itemsize == 32
        check(_lib.lib().tbvh_upload_bvh(self.h, _np_ptr(nodes), nodes.shape[0], _np_ptr(primIdx), primIdx.shape[0], p, stride, nv // 3, space))
        return self

    def download(self):
        """-> (bvhNode[usedNodes] as NODE32, primIdx[idxCount]) in the reference layout."""
        i = self.info()
        nodes = np.zeros(i.used_nodes, NODE32)
        idx = np.zeros(i.idx_count, np.uint32)
        check(_lib.lib().tbvh_download_bvh(self.h, _np_ptr(nodes), _np_ptr(idx), HOST))
        return nodes, idx


BLAS_INSTANCE = np.dtype([("transform", "16f4"), ("invTransform", "16f4"), ("aabbMin", "3f4"), ("blasIdx", "u4"),
                          ("aabbMax", "3f4"), ("mask", "u4"), ("dummy", "8u4")])   # tinybvh::BLASInstance, tiny_bvh.h:1443 (192 bytes)


class TLAS(BVH):
    """A tinybvh::BVH built with Build( BLASInstance*, instCount, BVHBase**, blasCount ) (tiny_bvh.h:2221): Intersect / IsOccluded on
    it are IntersectTLAS / IsOccludedTLAS.  `instances`: BLAS_INSTANCE records already Update()d by the caller (inverse transform
    and world box, as BLASInstance::Update :8386 computes them); `blasses`: BVH objects of this module, kept alive by this one."""

    def Build(self, instances, blasses, update: bool = True, blas_layout: int = LAYOUT_BVH):
        """update=True: BLASInstance::Update (:8386) is applied to every record first - in place, as the reference's Build does when it
        is handed the BLAS list (:2245-2250); update=False: the records already carry inverse transform and world box.
        blas_layout=LAYOUT_CWBVH: Intersect / IsOccluded walk every BLAS in its BVH8_CWBVH layout (the arrangement of the reference's GPU
        path, traverse_tlas.cl); the BLASses must hold that layout when the TLAS is built (BVH8_CWBVH objects, or tbvh_convert)."""
        inst = instances
        self.layout = blas_layout
        assert inst.dtype.itemsize == 192 and inst.flags.c_contiguous
        self.blasses = list(blasses)
        if update:
            if int(inst["blasIdx"].max()) >= len(self.blasses):
                raise TbvhError("TLAS: an instance names a BLAS past the list")
            for i in range(inst.shape[0]):
                check(_lib.lib().tbvh_instance_update(C.c_void_p(inst[i:i + 1].ctypes.data), self.blasses[int(inst["blasIdx"][i])].h))
        hs = (C.c_void_p * len(self.blasses))(*[b.h for b in self.blasses])
        check(_lib.lib().tbvh_build_tlas(self.h, _np_ptr(inst), 192, inst.shape[0], hs, len(self.blasses), self.c_trav, self.c_int))
        return self


class BVH_GPU(_Base):
    """tinybvh::BVH_GPU (tiny_bvh.h:1092-1127): Aila-Laine 64-byte nodes."""
    layout = LAYOUT_BVH_GPU

    def Build(self, vertices, primCount: int = 0, indices=None):
        # BVH_GPU::Build -> bvh.BuildDefault (tiny_bvh.h:4580-4590) = BuildAVX on x86, then ConvertFrom
        self._build(vertices, primCount, self.build_flavour, indices)
        check(_lib.lib().tbvh_convert(self.h, LAYOUT_BVH_GPU))
        return self

    def BuildHQ(self, vertices, primCount: int = 0, indices=None):
        """BVH_GPU::BuildHQ (tiny_bvh.h:4588): bvh.BuildHQ, then ConvertFrom."""
        self._build(vertices, primCount, _lib.BUILD_HQ, indices)
        check(_lib.lib().tbvh_convert(self.h, LAYOUT_BVH_GPU))
        return self

    def upload(self, nodes, primIdx, vertices):
        p, stride, nv, space, keep = _verts_arg(vertices)
        nodes = np.ascontiguousarray(nodes)
        primIdx = np.ascontiguousarray(primIdx, np.uint32)
        assert nodes.dtype.itemsize == 64
        check(_lib.lib().tbvh_upload_bvh_gpu(self.h, _np_ptr(nodes), nodes.shape[0], _np_ptr(primIdx), primIdx.shape[0], p, stride, nv // 3, space))
        return self

    def download(self):
        i = self.info()
        nodes = np.zeros(i.used_nodes_gpu, NODE64)
        check(_lib.lib().tbvh_download_bvh_gpu(self.h, _np_ptr(nodes), HOST))
        return nodes


class BVH8_CWBVH(_Base):
    """tinybvh::BVH8_CWBVH (tiny_bvh.h:1334-1362): 80-byte compressed wide nodes + 48-byte triangles."""
    layout = LAYOUT_CWBVH

    def Build(self, vertices, primCount: int = 0, indices=None):
        # BVH8_CWBVH::Build -> bvh8.bvh.BuildDefault (tiny_bvh.h:5830) = BuildAVX on x86, then the conversion chain
        self._build(vertices, primCount, self.build_flavour, indices)
        check(_lib.lib().tbvh_convert(self.h, LAYOUT_CWBVH))
        return self

    def BuildHQ(self, vertices, primCount: int = 0, indices=None):
        """BVH8_CWBVH::BuildHQ (tiny_bvh.h:5859): bvh.BuildHQ, SplitLeafs(3), 8-wide collapse, CWBVH encode."""
        self._build(vertices, primCount, _lib.BUILD_HQ, indices)
        check(_lib.lib().tbvh_convert(self.h, LAYOUT_CWBVH))
        return self

    def upload(self, bvh8Data, bvh8Tris):
        """bvh8Data: float32 [usedBlocks,4]; bvh8Tris: float32 [3*triCount,4] (public members :1356-1357)."""
        d = np.ascontiguousarray(bvh8Data, np.float32).reshape(-1, 4)
        t = np.ascontiguousarray(bvh8Tris, np.float32).reshape(-1, 4)
        check(_lib.lib().tbvh_upload_cwbvh(self.h, _np_ptr(d), d.shape[0], _np_ptr(t), t.shape[0] // 3, HOST))
        return self

    def download(self):
        i = self.info()
        d = np.zeros((i.used_blocks, 4), np.float32)
        t = np.zeros((i.cwbvh_tri_count * 3, 4), np.float32)
        check(_lib.lib().tbvh_download_cwbvh(self.h, _np_ptr(d), _np_ptr(t), HOST))
        return d, t


def pinned_empty(n: int, dtype, device: int = None, node: int = None) -> np.ndarray:
    """numpy array in page-locked host memory on the NUMA node of `device` (default: the current CUDA device): full-speed DMA
    for the host path (tbvh_host_alloc / tbvh_host_alloc_near)."""
    dtype = np.dtype(dtype)
    p = C.c_void_p()
    if node is not None:
        check(_lib.lib().tbvh_host_alloc_node(node, n * dtype.itemsize, C.byref(p)))
    elif device is None:
        check(_lib.lib().tbvh_host_alloc(n * dtype.itemsize, C.byref(p)))
    else:
        check(_lib.lib().tbvh_host_alloc_near(device, n * dtype.itemsize, C.byref(p)))
    buf = (C.c_char * (n * dtype.itemsize)).from_address(p.value)
    a = np.frombuffer(buf, dtype=dtype, count=n)
    a.flags.writeable = True
    _pinned[a.ctypes.data] = p
    return a


_pinned = {}


def pinned_free(a: np.ndarray):
    p = _pinned.pop(a.ctypes.data, None)
    if p is not None:
        check(_lib.lib().tbvh_host_free(p))


def copy_rays_to_device(rays: np.ndarray, d_rays, stream=None) -> None:
    """tbvh_copy_rays_to_device: bytes 0..63 of every host record into a [n, 64]-byte torch CUDA tensor (synchronous here)."""
    import torch
    assert rays.dtype.itemsize in (64, 128) and rays.flags.c_contiguous and d_rays.is_cuda and d_rays.is_contiguous()
    assert d_rays.numel() * d_rays.element_size() >= rays.shape[0] * 64
    st = torch.cuda.current_stream(d_rays.device)
    check(_lib.lib().tbvh_copy_rays_to_device(_np_ptr(rays), rays.dtype.itemsize, rays.shape[0], C.c_void_p(d_rays.data_ptr()), C.c_void_p(st.cuda_stream)))
    st.synchronize()


def bind_to_device(device: int = 0) -> bool:
    """Restrict the calling thread (and threads it starts later: OpenMP, the host pipeline) to the CPUs of the NUMA node `device`
    hangs off.  False when the system exposes no topology."""
    return _lib.lib().tbvh_bind_thread_to_device(device) == _lib.OK


def shard_range(n: int, part: int, parts: int):
    """tbvh_shard_range: contiguous [first, first+count) of n rays for `part`, boundaries on multiples of 32."""
    a, c = C.c_uint64(), C.c_uint64()
    _lib.lib().tbvh_shard_range(n, part, parts, C.byref(a), C.byref(c))
    return a.value, c.value


class Group:
    """Several GPUs of one process (tbvh_group_*): `replicate(bvh)` copies a BVH to every device over NVLink, `Intersect` /
    `IsOccluded` shard a host ray batch by index over the devices.  `layout` follows the replicated object."""

    def __init__(self, devices=None):
        self.h = C.c_void_p()
        if devices is None:
            check(_lib.lib().tbvh_group_create(None, 0, C.byref(self.h)))
        else:
            arr = (C.c_int * len(devices))(*devices)
            check(_lib.lib().tbvh_group_create(arr, len(devices), C.byref(self.h)))
        self.layout = LAYOUT_BVH
        self.src = None

    def __len__(self):
        return _lib.lib().tbvh_group_size(self.h)

    def replicate(self, bvh) -> float:
        ms = C.c_double()
        check(_lib.lib().tbvh_group_replicate(self.h, bvh.h, C.byref(ms)))
        self.src, self.layout = bvh, bvh.layout
        return ms.value

    def empty_rays(self, n: int, dtype) -> np.ndarray:
        """page-locked array whose index ranges sit on the NUMA node of the device that will read them (tbvh_group_host_alloc)"""
        dtype = np.dtype(dtype)
        p = C.c_void_p()
        check(_lib.lib().tbvh_group_host_alloc(self.h, dtype.itemsize, n, C.byref(p)))
        buf = (C.c_char * (n * dtype.itemsize)).from_address(p.value)
        a = np.frombuffer(buf, dtype=dtype, count=n)
        a.flags.writeable = True
        return a

    def Intersect(self, rays: np.ndarray) -> np.ndarray:
        assert rays.dtype.itemsize in (64, 128) and rays.flags.c_contiguous
        check(_lib.lib().tbvh_group_intersect(self.h, self.layout, _np_ptr(rays), rays.dtype.itemsize, rays.shape[0]))
        return rays

    def IsOccluded(self, rays: np.ndarray, bits: np.ndarray = None) -> np.ndarray:
        assert rays.dtype.itemsize in (64, 128) and rays.flags.c_contiguous
        n = rays.shape[0]
        if bits is None:
            bits = np.zeros((n + 31) // 32, np.uint32)
        check(_lib.lib().tbvh_group_occluded(self.h, self.layout, _np_ptr(rays), rays.dtype.itemsize, n, _np_ptr(bits)))
        return bits

    def close(self):
        if self.h is not None and self.h.value:
            _lib.lib().tbvh_group_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
