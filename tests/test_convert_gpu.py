"""GPU parity of the layout conversions: BVH -> BVH_GPU on the device must equal BVH_GPU::ConvertFrom byte for byte."""
import numpy as np
import pytest

from oracle import refpy
from tinybvh_b200 import api, scenes
from tinybvh_b200._lib import BUILD_AVX, BUILD_REFERENCE
from tests import golden_util as G
from tests import util

pytestmark = pytest.mark.gpu
REF = util.reference()


def diff_nodes(got, want, words):
    a, b = got.view(np.uint32).reshape(-1, words), np.ascontiguousarray(want).view(np.uint32).reshape(-1, words)
    assert a.shape == b.shape, f"node count {a.shape[0]} != {b.shape[0]}"
    bad = np.nonzero((a != b).any(1))[0]
    assert bad.size == 0, f"{bad.size} nodes differ, first {bad[:4]}: got {a[bad[0]]} want {b[bad[0]]}"


@pytest.mark.parametrize("path", G.golden_files(), ids=lambda p: p.split("/")[-1])
def test_bvh_gpu_conversion_matches_golden(gpu, path):
    g = G.load(path)
    e = api.BVH_GPU()
    e.build_flavour = BUILD_REFERENCE   # the golden vectors hold BVH_GPU::ConvertFrom of the scalar BVH::Build tree
    e.Build(g["verts"])
    diff_nodes(e.download(), g["nodes_gpu"].view(np.uint8).view(api.NODE64).reshape(-1), 16)


@pytest.mark.parametrize("ntris,seed", [(5, 51), (999, 52), (120000, 53)])
@pytest.mark.parametrize("flavour", [BUILD_REFERENCE, BUILD_AVX])
def test_bvh_gpu_conversion_matches_reference(gpu, ntris, seed, flavour):
    """flavour AVX = BVH_GPU::Build itself (BuildDefault -> BuildAVX, then ConvertFrom); REFERENCE = ConvertFrom(BVH::Build)."""
    v = scenes.procedural_scene(ntris, seed)
    ref = REF.RefBVH(v, mode=1 if flavour == BUILD_AVX else 0, threaded=False)
    want = REF.RefBVHGPU(ref).nodes
    e = api.BVH_GPU()
    e.build_flavour = flavour
    e.Build(v)
    diff_nodes(e.download(), want, 16)
    # the converted layout traverses like the source tree
    sets, _ = util.ray_sets(v, res=48)
    a, b = sets["primary"].copy(), sets["primary"].copy()
    ref.intersect(a), e.Intersect(b)
    assert util.compare_hits(b, a) == {"prim": 0, "t": 0, "u": 0, "v": 0}


@pytest.mark.skipif(not refpy.available(), reason="needs oracle/_ref")
def test_bvh_gpu_conversion_of_threaded_reference_tree(gpu):
    """An uploaded tree with the reference's threaded (non-DFS) node numbering converts to the same DFS layout."""
    import ctypes as C
    from tinybvh_b200 import _lib
    v = scenes.procedural_scene(90000, 54)
    ref = refpy.RefBVH(v, mode=0, threaded=True)
    want = refpy.RefBVHGPU(ref).nodes
    e = api.BVH_GPU()
    nodes, idx = np.ascontiguousarray(ref.nodes), np.ascontiguousarray(ref.prim_idx)
    api.check(_lib.lib().tbvh_upload_bvh(e.h, nodes.ctypes.data_as(C.c_void_p), nodes.shape[0], idx.ctypes.data_as(C.c_void_p), idx.shape[0],
                                         v.ctypes.data_as(C.c_void_p), 16, v.shape[0] // 3, api.HOST))
    api.check(_lib.lib().tbvh_convert(e.h, api.LAYOUT_BVH_GPU))
    diff_nodes(e.download(), want, 16)


# ---- BVH -> CWBVH on the device (SplitLeafs(3) + MBVH<8> collapse + CWBVH encode) -------------------------------
def diff_blob(got, want, name, row_bytes):
    a = np.ascontiguousarray(got).view(np.uint8).reshape(-1, row_bytes)
    b = np.ascontiguousarray(want).view(np.uint8).reshape(-1, row_bytes)
    assert a.shape == b.shape, f"{name}: {a.shape[0]} records, reference has {b.shape[0]}"
    bad = np.nonzero((a != b).any(1))[0]
    assert bad.size == 0, f"{name}: {bad.size} of {a.shape[0]} records differ, first {bad[:6]}\\n got  {a[bad[0]].view(np.uint32)}\\n want {b[bad[0]].view(np.uint32)}"


@pytest.mark.parametrize("path", [p for p in G.golden_files() if "cwbvh_nodes" in np.load(p).files], ids=lambda p: p.split("/")[-1])
def test_cwbvh_conversion_matches_golden(gpu, path):
    """The reference's BVH8_CWBVH chain over the scalar BVH::Build tree and its CPU walk, as recorded in the golden vectors
    (tools/make_golden.py): the device build + conversion byte for byte, the device walk bit for bit."""
    from tinybvh_b200 import rays as R
    g = G.load(path)
    e = api.BVH8_CWBVH()
    e.build_flavour = BUILD_REFERENCE
    e.Build(g["verts"])
    nodes, tris = e.download()
    diff_blob(nodes, g["cwbvh_nodes"], "bvh8Data (80-byte nodes)", 80)
    diff_blob(tris, g["cwbvh_tris"], "bvh8Tris (48-byte triangles)", 48)
    lo, hi = scenes.scene_bounds(g["verts"])
    res = int(round((g["cwbvh_primary_hit"].shape[0] // 4) ** 0.5))
    r = R.primary_rays(*R.bounds_camera(lo, hi, "outside"), res, res, 4)
    e.Intersect(r)
    assert np.array_equal(G.hits_as_u32(r), g["cwbvh_primary_hit"])


@pytest.mark.parametrize("ntris,seed", [(1, 61), (3, 62), (4, 63), (40, 64), (2000, 65), (60000, 66)])
@pytest.mark.parametrize("flavour", [BUILD_REFERENCE, BUILD_AVX])
def test_cwbvh_conversion_matches_reference(gpu, ntris, seed, flavour):
    """flavour AVX: byte-identical to BVH8_CWBVH::Build itself (mode 0: BuildDefault = BuildAVX, Compact, SplitLeafs, collapse,
    encode); REFERENCE: the same chain over the scalar BVH::Build tree (mode 2)."""
    v = scenes.procedural_scene(ntris, seed)
    cw = REF.RefCWBVH(v, mode=0 if flavour == BUILD_AVX else 2)
    e = api.BVH8_CWBVH()
    e.build_flavour = flavour
    e.Build(v)
    nodes, tris = e.download()
    diff_blob(nodes, cw.nodes, "bvh8Data (80-byte nodes)", 80)
    diff_blob(tris, cw.tris, "bvh8Tris (48-byte triangles)", 48)


@pytest.mark.parametrize("scene", ["bunny", "sponza"])
def test_cwbvh_conversion_fixtures(gpu, scene):
    v, label = scenes.load_scene(scene)
    cw = REF.RefCWBVH(v, mode=0)      # BVH8_CWBVH::Build as the reference runs it (threaded BuildAVX underneath)
    e = api.BVH8_CWBVH().Build(v)
    nodes, tris = e.download()
    diff_blob(nodes, cw.nodes, label + " bvh8Data", 80)
    diff_blob(tris, cw.tris, label + " bvh8Tris", 48)
    # and the GPU-converted structure traverses like the reference-built one
    from tinybvh_b200 import rays as R
    lo, hi = scenes.scene_bounds(v)
    eye, view = (R.SPONZA_EYES[2], R.SPONZA_VIEWS[2]) if scene == "sponza" else R.bounds_camera(lo, hi, "outside")
    a = R.primary_rays(eye, view, 128, 128, 4)
    b = a.copy()
    cw.intersect(a), e.Intersect(b)
    assert util.compare_hits(b, a) == {"prim": 0, "t": 0, "u": 0, "v": 0}
