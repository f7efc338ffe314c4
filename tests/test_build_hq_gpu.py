"""GPU parity of the SBVH builder: tbvh_build_flavour(TBVH_BUILD_HQ) through the C-ABI must produce the reference's
BVH::BuildHQ tree (spatial splits, unsplitting, final Compact) byte for byte: node array and the part of primIdx the
leaves reference.  The checker is the pinned restatement oracle/tbvh_oracle_hq.c (and the golden HQ trees)."""
import numpy as np
import pytest

from tinybvh_b200 import api, rays as R, scenes
from tests import golden_util as G
from tests import util

pytestmark = pytest.mark.gpu


def hq_want(v):
    from oracle import portpy
    return portpy.build_hq(v)


def assert_same_hq_tree(e, nodes_want, idx_want, idx_count_want, label=""):
    nodes, idx = e.download()
    info = e.info()
    assert info.idx_count == idx_count_want and idx.shape[0] == idx_count_want, f"{label}: idxCount {info.idx_count}"
    assert nodes.shape[0] == nodes_want.shape[0], f"{label}: usedNodes {nodes.shape[0]} != {nodes_want.shape[0]}"
    a, b = nodes.view(np.uint32).reshape(-1, 8), np.ascontiguousarray(nodes_want).view(np.uint32).reshape(-1, 8)
    bad = np.nonzero((a != b).any(1))[0]
    assert bad.size == 0, f"{label}: {bad.size} nodes differ, first {bad[:5]}: got {a[bad[0]]} want {b[bad[0]]}"
    used = idx_want.shape[0]
    assert np.array_equal(idx[:used], idx_want), f"{label}: primIdx differs at {np.nonzero(idx[:used] != idx_want)[0][:8]}"
    assert not idx[used:].any()


@pytest.mark.parametrize("path", G.golden_files(), ids=lambda p: p.split("/")[-1])
def test_build_hq_matches_golden_tree(gpu, path):
    g = G.load(path)
    e = api.BVH().BuildHQ(g["verts"])
    assert_same_hq_tree(e, g["hq_nodes"].view(np.uint8).view(api.NODE32).reshape(-1), g["hq_prim_idx"], int(g["hq_idx_count"][0]), path)


@pytest.mark.parametrize("ntris,seed", [(1, 1), (2, 2), (3, 3), (31, 4), (256, 5), (257, 6), (300, 7), (1000, 8), (5000, 9), (70000, 10), (200000, 11)])
def test_build_hq_matches_oracle_on_seeded_scenes(gpu, ntris, seed):
    v = scenes.procedural_scene(ntris, seed)
    nodes, idx, ic = hq_want(v)
    e = api.BVH().BuildHQ(v)
    assert_same_hq_tree(e, nodes, idx, ic, f"{ntris} tris")
    assert e.info().build_ms > 0


@pytest.mark.parametrize("scene", ["legocar", "head", "bunny", "sponza"])
def test_build_hq_fixtures_and_trace(gpu, scene):
    """legocar and sponza contain 'spatial split failed' leaves (tiny_bvh.h:2939), whose content depends on the words an
    ancestor's partition left behind in idxTmp - reproduced, not avoided."""
    v, label = scenes.load_scene(scene)
    nodes, idx, ic = hq_want(v)
    e = api.BVH().BuildHQ(v)
    assert_same_hq_tree(e, nodes, idx, ic, label)
    # traversal of the SBVH: same hits as the oracle walking the same tree
    from oracle import portpy
    o = portpy.PortBVH(v, nodes=nodes, prim_idx=idx)
    lo, hi = scenes.scene_bounds(v)
    eye, view = (R.SPONZA_EYES[0], R.SPONZA_VIEWS[0]) if scene == "sponza" else R.bounds_camera(lo, hi, "outside")
    want = R.primary_rays(eye, view, 128, 128, 4)
    got = want.copy()
    o.intersect(want), e.Intersect(got)
    assert util.compare_hits(got, want) == {"prim": 0, "t": 0, "u": 0, "v": 0}


def test_build_hq_degenerate_inputs(gpu):
    one = np.array([[0, 0, 0, 0], [1, 0, 0, 0], [0, 1, 0, 0]], np.float32)
    same = np.tile(one, (700, 1))
    flat = scenes.procedural_scene(3000, 12)
    flat[:, 1] = 1.5
    base = scenes.procedural_scene(900, 13)
    dup = np.concatenate([base, base, base[:300]])
    # long thin triangles: the case spatial splits exist for
    rng = np.random.default_rng(17)
    c = rng.random((2000, 3), np.float32) * 10
    d = (rng.random((2000, 3), np.float32) - 0.5) * np.array([8, 0.05, 0.05], np.float32)
    w = (rng.random((2000, 3), np.float32) - 0.5) * 0.05
    sl = np.zeros((6000, 4), np.float32)
    sl[0::3, :3], sl[1::3, :3], sl[2::3, :3] = c - d, c + d, c + w
    for name, v in (("identical", same), ("flat", flat), ("duplicates", dup), ("slivers", sl)):
        nodes, idx, ic = hq_want(v)
        e = api.BVH().BuildHQ(v)
        assert_same_hq_tree(e, nodes, idx, ic, name)


def test_build_hq_is_deterministic(gpu):
    v = scenes.procedural_scene(30000, 14)
    a = api.BVH().BuildHQ(v).download()
    b = api.BVH().BuildHQ(v).download()
    assert np.array_equal(a[0].view(np.uint8), b[0].view(np.uint8)) and np.array_equal(a[1], b[1])


@pytest.mark.parametrize("scene", ["synthetic:5000", "bunny", "sponza"])
def test_derived_layouts_build_hq(gpu, scene):
    """BVH_GPU::BuildHQ (:4588) and BVH8_CWBVH::BuildHQ (:5859): the SBVH pushed through the same converters."""
    REF = util.reference()
    v, label = scenes.load_scene(scene)
    ref = REF.RefBVH(v, mode=2, threaded=False)
    want = REF.RefBVHGPU(ref).nodes
    got = api.BVH_GPU().BuildHQ(v).download()
    assert got.shape == want.shape and np.array_equal(got.view(np.uint32), want.view(np.uint32)), f"{label}: BVH_GPU nodes differ"
    cw = REF.RefCWBVH(v, mode=1)
    e = api.BVH8_CWBVH().BuildHQ(v)
    nodes, tris = e.download()
    assert nodes.shape == cw.nodes.shape and np.array_equal(nodes.view(np.uint32), cw.nodes.view(np.uint32)), f"{label}: bvh8Data differs"
    used = int(cw.source_bvh().nodes["triCount"].sum()) * 3   # the reference leaves the records beyond the referenced ones uninitialised
    assert tris.shape[0] >= used and np.array_equal(tris[:used].view(np.uint32), cw.tris[:used].view(np.uint32)), f"{label}: bvh8Tris differs"
    # traversal of the SBVH-derived CWBVH: bit-identical to the reference's own CPU walk of the same data
    lo, hi = scenes.scene_bounds(v)
    eye, view = (R.SPONZA_EYES[0], R.SPONZA_VIEWS[0]) if scene == "sponza" else R.bounds_camera(lo, hi, "outside")
    a = R.primary_rays(eye, view, 96, 96, 4)
    b = a.copy()
    cw.intersect(a), e.Intersect(b)
    assert util.compare_hits(b, a) == {"prim": 0, "t": 0, "u": 0, "v": 0}


@pytest.mark.parametrize("mode,method", [(0, "Build"), (1, "BuildAVX"), (2, "BuildHQ")])
def test_indexed_geometry_builds(gpu, mode, method):
    """The ( vertices, indices, primCount ) overloads (tiny_bvh.h:889-900) through tbvh_build_indexed: same tree as the
    reference builds from the shared-vertex mesh, same hits."""
    from tests.test_oracle_pin import indexed_mesh
    REF = util.reference()
    flat, verts, idx = indexed_mesh(20000, 43)
    ref = REF.RefBVH(verts, mode=mode, threaded=False, indices=idx)
    e = getattr(api.BVH(), method)(verts, indices=idx)
    nodes, pidx = e.download()
    assert e.info().prim_count == 20000
    assert np.array_equal(nodes.view(np.uint32), ref.nodes.view(np.uint32)), f"{method}( vertices, indices ): node array differs"
    used = int(ref.nodes["triCount"].sum())
    assert np.array_equal(pidx[:used], ref.prim_idx[:used])
    lo, hi = scenes.scene_bounds(flat)
    want = R.primary_rays(*R.bounds_camera(lo, hi, "outside"), 64, 64, 4)
    got = want.copy()
    ref.intersect(want), e.Intersect(got)
    assert util.compare_hits(got, want) == {"prim": 0, "t": 0, "u": 0, "v": 0}


def test_indexed_build_rejects_bad_index(gpu):
    verts = np.zeros((4, 4), np.float32)
    verts[1, 0] = verts[2, 1] = verts[3, 2] = 1
    with pytest.raises(api.TbvhError):
        api.BVH().Build(verts, indices=np.array([0, 1, 2, 1, 2, 7], np.uint32))
    e = api.BVH().Build(verts, indices=np.array([0, 1, 2, 1, 2, 3], np.uint32))
    assert e.info().prim_count == 2 and e.info().used_nodes == 2


@pytest.mark.parametrize("costs", [(1.0, 2.0), (3.0, 0.5)])
def test_builders_with_other_sah_constants(gpu, costs):
    """c_trav / c_int reach all three GPU builders through the C-ABI (BVHBase::c_trav / c_int, tiny_bvh.h:819-820)."""
    from oracle import portpy
    v = scenes.procedural_scene(40000, 62)
    for method, avx in (("Build", False), ("BuildAVX", True)):
        e = api.BVH()
        e.c_trav, e.c_int = costs
        nodes, idx = getattr(e, method)(v).download()
        o = portpy.PortBVH(v, c_trav=costs[0], c_int=costs[1], avx=avx)
        assert np.array_equal(nodes.view(np.uint32), o.nodes.view(np.uint32)) and np.array_equal(idx, o.prim_idx), method
    e = api.BVH()
    e.c_trav, e.c_int = costs
    hn, hi, ic = portpy.build_hq(v, *costs)
    assert_same_hq_tree(e.BuildHQ(v), hn, hi, ic, f"BuildHQ costs {costs}")
