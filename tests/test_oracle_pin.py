"""Pin the plain-C restatement (oracle/tbvh_oracle.c): bit-for-bit against the committed golden vectors produced by
the unmodified reference (tools/make_golden.py), and - where oracle/_ref is present - against the reference itself
on larger seeded inputs.  CPU only."""
import numpy as np
import pytest

from oracle import portpy, refpy
from tinybvh_b200 import rays as R, scenes
from tests import golden_util as G
from tests import util


@pytest.mark.parametrize("path", G.golden_files(), ids=lambda p: p.split("/")[-1])
def test_port_build_matches_golden_tree(path):
    g = G.load(path)
    p = portpy.PortBVH(g["verts"])
    assert p.used_nodes == g["nodes"].shape[0]
    assert np.array_equal(p.nodes.view(np.uint32).reshape(-1, 8), g["nodes"]), "node array differs from BVH::Build"
    assert np.array_equal(p.prim_idx, g["prim_idx"]), "primIdx differs from BVH::Build"
    assert np.array_equal(p.to_bvh_gpu().view(np.uint32).reshape(-1, 16), g["nodes_gpu"]), "BVH_GPU::ConvertFrom differs"


@pytest.mark.parametrize("path", G.golden_files(), ids=lambda p: p.split("/")[-1])
def test_port_traversal_matches_golden_hits(path):
    g = G.load(path)
    p = portpy.PortBVH(g["verts"], nodes=g["nodes"].view(np.uint8).view(portpy.NODE32).reshape(-1), prim_idx=g["prim_idx"])
    for kind in ("primary", "diffuse"):
        r = G.rays_of(g, kind)
        p.intersect(r, threads=2)
        assert np.array_equal(G.hits_as_u32(r), g[kind + "_hit"]), f"{kind}: t/u/v/prim bits differ from BVH::Intersect"
    s = G.rays_of(g, "shadow")
    assert np.array_equal(p.occluded(s, threads=2), g["shadow_bits"]), "occlusion bits differ from BVH::IsOccluded"


def test_golden_has_hits_misses_and_ties():
    g = G.load([p for p in G.golden_files() if "coincident" in p][0])
    t = g["primary_hit"][:, 0].view(np.float32)
    assert (t < 1e30).any() and (t >= 1e30).any()
    # coincident triangles: the later-tested duplicate wins (accept on t <= hit.t, tiny_bvh.h:1656), so some hits
    # must carry a duplicate's index (>= 400)
    assert (g["primary_hit"][:, 3][t < 1e30] >= 400).any()


@pytest.mark.skipif(not refpy.available(), reason="oracle/_ref not built (needs /root/reference)")
@pytest.mark.parametrize("ntris,seed", [(20000, 1), (777, 2), (2, 3), (1, 4)])
def test_port_matches_reference_on_seeded_scenes(ntris, seed):
    v = scenes.procedural_scene(ntris, seed)
    ref = refpy.RefBVH(v, mode=0, threaded=False)
    port = portpy.PortBVH(v)
    assert ref.used_nodes == port.used_nodes
    assert np.array_equal(ref.nodes.view(np.uint8), port.nodes.view(np.uint8))
    assert np.array_equal(ref.prim_idx, port.prim_idx)
    sets, bounds = util.ray_sets(v, res=64)
    a, b = sets["primary"].copy(), sets["primary"].copy()
    ref.intersect(a, threads=2), port.intersect(b, threads=2)
    assert util.compare_hits(a, b) == {"prim": 0, "t": 0, "u": 0, "v": 0}
    for name, rr in util.derived_sets(a, v, bounds).items():
        if name == "shadow":
            assert np.array_equal(ref.occluded(rr, threads=2), port.occluded(rr, threads=2))
        else:
            c, d = rr.copy(), rr.copy()
            ref.intersect(c, threads=2), port.intersect(d, threads=2)
            assert util.compare_hits(c, d) == {"prim": 0, "t": 0, "u": 0, "v": 0}


def test_ray_record_layout():
    assert R.RAY_DTYPE.itemsize == 128 and R.GPU_RAY_DTYPE.itemsize == 64
    assert R.RAY_DTYPE.fields["t"][1] == 48 and R.RAY_DTYPE.fields["prim"][1] == 60 and R.RAY_DTYPE.fields["rD"][1] == 32
    r = R.make_rays([[0, 0, 0]], [[0, 0, 2]])
    assert np.allclose(r["D"], [[0, 0, 1]]) and r["rD"][0, 2] == 1 and r["rD"][0, 0] == np.float32(1e30)
    r = R.make_rays([[0, 0, 0]], [[-0.0, -1e-13, 1]])
    assert r["rD"][0, 0] == np.float32(1e30) and r["rD"][0, 1] == np.float32(-1e30)  # tinybvh_safercp :442


def test_primary_ray_pattern():
    r = R.primary_rays(R.SPONZA_EYES[0], R.SPONZA_VIEWS[0], 8, 8, 16)
    assert r.shape[0] == 8 * 8 * 16
    # first 256 rays = first 4x4-pixel tile, 16 samples per pixel (tiny_bvh_speedtest.cpp:527-540)
    assert np.allclose(r["O"], R.SPONZA_EYES[0])
    assert np.allclose(np.linalg.norm(r["D"], axis=1), 1, atol=1e-6)


@pytest.mark.skipif(not refpy.available(), reason="oracle/_ref not built (needs /root/reference)")
@pytest.mark.parametrize("ntris,seed", [(20000, 5), (777, 6), (3, 7)])
def test_port_avx_flavour_matches_reference(ntris, seed):
    """orc_build_avx restates BVH::BuildAVX (the BuildDefault builder on x86): byte-identical trees."""
    v = scenes.procedural_scene(ntris, seed)
    ref = refpy.RefBVH(v, mode=1, threaded=False)
    port = portpy.PortBVH(v, avx=True)
    assert ref.used_nodes == port.used_nodes
    assert np.array_equal(ref.nodes.view(np.uint8), port.nodes.view(np.uint8))
    assert np.array_equal(ref.prim_idx, port.prim_idx)


# ---------------------------------------------------------------- BVH::BuildHQ (SBVH) restatement, oracle/tbvh_oracle_hq.c
@pytest.mark.parametrize("path", G.golden_files(), ids=lambda p: p.split("/")[-1])
def test_port_build_hq_matches_golden_tree(path):
    g = G.load(path)
    nodes, idx, idx_count = portpy.build_hq(g["verts"])
    assert np.array_equal(nodes.view(np.uint32).reshape(-1, 8), g["hq_nodes"])
    assert np.array_equal(idx, g["hq_prim_idx"])
    assert idx_count == int(g["hq_idx_count"][0])


@pytest.mark.skipif(not refpy.available(), reason="oracle/_ref not built (needs /root/reference)")
@pytest.mark.parametrize("ntris,seed", [(20000, 21), (3000, 22), (300, 23), (2, 24)])
def test_port_build_hq_matches_reference(ntris, seed):
    v = scenes.procedural_scene(ntris, seed=seed)
    ref = refpy.RefBVH(v, mode=2, threaded=False)
    nodes, idx, idx_count = portpy.build_hq(v)
    assert np.array_equal(nodes.view(np.uint32), ref.nodes.view(np.uint32))
    assert np.array_equal(idx, ref.prim_idx[: idx.shape[0]]) and idx.shape[0] == int(ref.nodes["triCount"].sum())
    assert idx_count == ref.idx_count
    # an SBVH may reference a triangle from several leaves, but every triangle is referenced at least once
    assert np.array_equal(np.unique(idx), np.arange(ntris))


@pytest.mark.skipif(not refpy.available(), reason="oracle/_ref not built (needs /root/reference)")
def test_port_clip_and_split_frag_match_reference():
    v = scenes.procedural_scene(4000, seed=31)
    n = v.shape[0] // 3
    ref = refpy.RefBVH(v, mode=0, threaded=False)
    tri = v.reshape(-1, 3, 4)[:, :, :3]
    lo, hi = tri.min((0, 1)), tri.max((0, 1))
    min_dim = ((hi - lo) * np.float32(1e-7)).astype(np.float32)
    rng = np.random.default_rng(7)
    for it in range(6000):
        i = int(rng.integers(n))
        fr = np.zeros(1, refpy.FRAGMENT)
        fr["primIdx"], fr["bmin"], fr["bmax"] = i, tri[i].min(0), tri[i].max(0)
        fr["clipped"] = it & 1
        ext = fr["bmax"][0] - fr["bmin"][0]
        if it & 1:  # a box a previous clip could have left
            fr["bmin"][0] += ext * rng.random(3, np.float32) * 0.3
            fr["bmax"][0] -= ext * rng.random(3, np.float32) * 0.3
            ext = fr["bmax"][0] - fr["bmin"][0]
        axis = int(rng.integers(3))
        bmin, bmax = lo.copy(), hi.copy()
        bmin[axis] = fr["bmin"][0][axis] + ext[axis] * rng.random() * 0.9
        bmax[axis] = bmin[axis] + ext[axis] * rng.random() * 0.5
        ok_r, out_r = ref.clip_frag(fr, bmin, bmax, min_dim, axis)
        ok_p, out_p = portpy.clip_frag(v, fr, bmin, bmax, min_dim, axis)
        assert ok_r == ok_p and out_r.tobytes() == out_p.tobytes()
        pos = np.float32(fr["bmin"][0][axis] + ext[axis] * rng.random())
        sr, sp = ref.split_frag(fr, min_dim, axis, pos), portpy.split_frag(v, fr, min_dim, axis, pos)
        assert sr[:2] == sp[:2] and sr[2].tobytes() == sp[2].tobytes() and sr[3].tobytes() == sp[3].tobytes()


def indexed_mesh(ntris, seed):
    """A shared-vertex version of a procedural soup: unique vertices + an index list (with a shuffled vertex order)."""
    v = scenes.procedural_scene(ntris, seed=seed)
    uniq, inv = np.unique(v.view(np.uint32).reshape(-1, 4), axis=0, return_inverse=True)
    perm = np.random.default_rng(seed).permutation(uniq.shape[0])
    rank = np.empty_like(perm)
    rank[perm] = np.arange(perm.shape[0])
    return v, uniq[perm].view(np.float32), rank[inv.reshape(-1)].astype(np.uint32)


@pytest.mark.skipif(not refpy.available(), reason="oracle/_ref not built (needs /root/reference)")
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_reference_indexed_build_equals_flat_build(mode):
    """What tbvh_build_indexed relies on: Build / BuildAVX / BuildHQ( vertices, indices, n ) (tiny_bvh.h:889-900) produce the
    tree of the flat soup verts[indices] - PrepareBuild only differs in where it reads the three vertices (:2290-2308)."""
    flat, verts, idx = indexed_mesh(3000, 41)
    assert np.array_equal(verts[idx].view(np.uint32), flat.view(np.uint32))
    a = refpy.RefBVH(flat, mode=mode, threaded=False)
    b = refpy.RefBVH(verts, mode=mode, threaded=False, indices=idx)
    assert np.array_equal(a.nodes.view(np.uint32), b.nodes.view(np.uint32))
    used = int(a.nodes["triCount"].sum())
    assert np.array_equal(a.prim_idx[:used], b.prim_idx[:used])
    r = R.make_rays(np.tile(np.array([[0.1, 0.2, -30.0]], np.float32), (64, 1)),
                    np.random.default_rng(3).normal(size=(64, 3)).astype(np.float32) * 0.1 + np.array([0, 0, 1], np.float32))
    ra, rb = r.copy(), r.copy()
    a.intersect(ra, threads=1), b.intersect(rb, threads=1)
    assert np.array_equal(G.hits_as_u32(ra), G.hits_as_u32(rb))


def moved(v, seed, amp=0.02):
    """The same triangles, every vertex displaced a little (an animation frame)."""
    rng = np.random.default_rng(seed)
    w = v.copy()
    ext = float((v[:, :3].max(0) - v[:, :3].min(0)).max())
    w[:, :3] += (rng.random((v.shape[0], 3), np.float32) - 0.5) * np.float32(amp * ext)
    return w


@pytest.mark.skipif(not refpy.available(), reason="oracle/_ref not built (needs /root/reference)")
@pytest.mark.parametrize("ntris,seed", [(20000, 51), (300, 52), (1, 53)])
def test_port_refit_matches_reference(ntris, seed):
    v = scenes.procedural_scene(ntris, seed=seed)
    ref, port = refpy.RefBVH(v, mode=0, threaded=False), portpy.PortBVH(v)
    before = port.nodes.copy()
    w = moved(v, seed)
    ref.refit(w), port.refit(w)
    assert np.array_equal(port.nodes.view(np.uint32), ref.nodes.view(np.uint32))
    assert not np.array_equal(port.nodes.view(np.uint32), before.view(np.uint32))


@pytest.mark.skipif(not refpy.available(), reason="oracle/_ref not built (needs /root/reference)")
@pytest.mark.parametrize("costs", [(1.0, 2.0), (3.0, 0.5), (0.25, 1.0)])
def test_port_matches_reference_with_other_sah_constants(costs):
    """BVHBase::c_trav / c_int (:819-820) enter the termination test of all three builders."""
    v = scenes.procedural_scene(6000, seed=61)
    for mode in (0, 1, 2):
        ref = refpy.RefBVH(v, mode=mode, threaded=False, costs=costs)
        if mode == 2:
            nodes, idx, _ = portpy.build_hq(v, *costs)
            assert np.array_equal(nodes.view(np.uint32), ref.nodes.view(np.uint32)) and np.array_equal(idx, ref.prim_idx[: idx.shape[0]])
        else:
            port = portpy.PortBVH(v, c_trav=costs[0], c_int=costs[1], avx=mode == 1)
            assert np.array_equal(port.nodes.view(np.uint32), ref.nodes.view(np.uint32)) and np.array_equal(port.prim_idx, ref.prim_idx)
    # the constants matter: the default tree is a different one
    assert refpy.RefBVH(v, mode=0, threaded=False).used_nodes != refpy.RefBVH(v, mode=0, threaded=False, costs=costs).used_nodes


def tlas_case(seed, n_inst=40):
    """Two BLASses, n_inst instances with random transforms; every fifth instance carries mask 0x2 only, the others 0x3."""
    v = [scenes.procedural_scene(2000, seed), scenes.procedural_scene(500, seed + 1)]
    inst = refpy.make_instances(util.random_transforms(n_inst, seed), [i % 2 for i in range(n_inst)],
                                masks=[0x3 if i % 5 else 0x2 for i in range(n_inst)])
    rng = np.random.default_rng(seed)
    D = rng.normal(size=(20000, 3)).astype(np.float32) * 0.35 + np.array([0, 0, 1], np.float32)
    O = np.tile(np.array([[0, 0, -120]], np.float32), (D.shape[0], 1))
    return v, inst, O, D


@pytest.mark.skipif(not refpy.available(), reason="oracle/_ref not built (needs /root/reference)")
def test_port_tlas_matches_reference():
    """BVH::IntersectTLAS / IsOccludedTLAS (:3306, :3455): instance transform, mask test, hit.inst, occlusion."""
    assert refpy.lib().ref_inst_idx_bits() == 32 and refpy.lib().ref_offsetof_hit_inst() == 44
    v, inst, O, D = tlas_case(91)
    blas_ref = [refpy.RefBVH(x, mode=0) for x in v]
    tl = refpy.RefTLAS(inst, blas_ref)          # Update()s inst in place: inverse transforms and world boxes
    tb = tl.bvh()
    port = portpy.PortTLAS(tb.nodes, tb.prim_idx, inst, [portpy.PortBVH(x) for x in v])
    rays = R.make_rays(O, D)
    rays["mask"] = 0x1       # these rays do not see the mask-0x2 instances (inst.mask & ray.mask, :3326)
    a, b = rays.copy(), rays.copy()
    tl.intersect(a, threads=1), port.intersect(b)
    wa, wb = a.view(np.uint32).reshape(-1, 32)[:, 11:16], b.view(np.uint32).reshape(-1, 32)[:, 11:16]   # inst, t, u, v, prim
    assert np.array_equal(wa, wb)
    hit = a["t"] < 1e30
    assert hit.sum() > 10000 and len(np.unique(wa[hit, 0])) > 12 and not np.isin(wa[hit, 0], np.arange(0, 40, 5)).any()
    sh = R.make_rays(O, D, tmax=150.0)
    assert np.array_equal(tl.occluded(sh, threads=1), port.occluded(sh))
    every = R.make_rays(O, D)
    every["mask"] = 0x2      # these see all forty
    a, b = every.copy(), every.copy()
    tl.intersect(a, threads=1), port.intersect(b)
    wa, wb = a.view(np.uint32).reshape(-1, 32)[:, 11:16], b.view(np.uint32).reshape(-1, 32)[:, 11:16]
    assert np.array_equal(wa, wb) and np.isin(wa[a["t"] < 1e30, 0], np.arange(0, 40, 5)).any()


@pytest.mark.skipif(not refpy.available(), reason="oracle/_ref not built (needs /root/reference)")
def test_port_tlas_over_cwbvh_composition():
    """A TLAS over BVH8_CWBVH BLASses (the reference's GPU arrangement, traverse_tlas.cl): the oracle composes its pinned TLAS walk with its
    pinned BVH8_CWBVH::Intersect.  Anchors: (1) a one-instance identity TLAS gives BVH8_CWBVH::Intersect's own result plus the instance;
    (2) against the reference's IntersectTLAS over BVH BLASses of the same triangles the hits agree wherever the two layouts agree on
    their own (distinct triangles at one distance are the only source of differences, SURVEY 8(c))."""
    v, inst, O, D = tlas_case(91)
    blas_ref = [refpy.RefBVH(x, mode=0) for x in v]
    tl = refpy.RefTLAS(inst, blas_ref)
    tb = tl.bvh()
    pb = [portpy.PortBVH(x) for x in v]
    cw = [portpy.PortCWBVH(b.nodes, b.prim_idx, b.verts) for b in pb]
    port = portpy.PortTLASCW(tb.nodes, tb.prim_idx, inst, cw)
    words = lambda r: r.view(np.uint32).reshape(-1, 32)[:, 11:16]   # inst, t, u, v, prim
    for mask in (0x1, 0x2):
        rays = R.make_rays(O, D)
        rays["mask"] = mask
        a, b = rays.copy(), rays.copy()
        tl.intersect(a, threads=1), port.intersect(b)
        same = (words(a) == words(b)).all(axis=1)
        assert same.mean() > 0.9995 and (a["t"] < 1e30).sum() > 10000   # this scene has no coincident triangles: in practice every ray agrees
        sh = R.make_rays(O, D, tmax=150.0)
        sh["mask"] = mask
        oa, ob = tl.occluded(sh, threads=1), port.occluded(sh)
        assert np.unpackbits((oa ^ ob).view(np.uint8)).sum() <= 4
    # one instance, identity transform: the BLAS walk alone
    one = refpy.make_instances(np.eye(4, dtype=np.float32)[None], [0])
    t1 = refpy.RefTLAS(one, blas_ref[:1])
    tb1 = t1.bvh()
    p1 = portpy.PortTLASCW(tb1.nodes, tb1.prim_idx, one, cw[:1])
    Dn = D / np.linalg.norm(D, axis=1, keepdims=True)
    rays = R.make_rays(O * 0.2, Dn.astype(np.float32))
    a, b = rays.copy(), rays.copy()
    cw[0].intersect(a), p1.intersect(b)
    assert np.array_equal(words(a)[:, 1:], words(b)[:, 1:]) and (a["t"] < 1e30).sum() > 1000
    assert (words(b)[b["t"] < 1e30, 0] == 0).all()


@pytest.mark.skipif(not refpy.available(), reason="oracle/_ref not built (needs /root/reference)")
def test_port_instance_update_matches_reference():
    """BLASInstance::Update / InvertTransform (:8386-8428): the vectorised reference build fuses different multiply-adds in
    different rows of the cofactor matrix; the restatement reproduces all of them (affine and projective matrices)."""
    rng = np.random.default_rng(5)
    T = (rng.random((3000, 16), np.float32) - 0.5) * 4
    T[::2, 12:15], T[::2, 15] = 0, 1
    a = refpy.make_instances(T, np.zeros(3000, np.uint32))
    b = a.copy()
    lo, hi = np.array([-1.5, -0.7, -2.2], np.float32), np.array([1.1, 2.3, 0.9], np.float32)
    for i in range(a.shape[0]):
        refpy.lib().ref_instance_update(a[i:i + 1].ctypes.data, lo.ctypes.data, hi.ctypes.data)
    portpy.instance_update(b, lo, hi)
    assert a.tobytes() == b.tobytes()


def test_port_tlas_matches_golden_vectors():
    """Committed outputs of the reference's TLAS path (tools/make_golden.py make_tlas): BLASInstance::Update, the TLAS tree over the
    instance boxes, IntersectTLAS hits (inst, t, u, v, prim) and IsOccludedTLAS bits for two ray masks."""
    import os
    g = dict(np.load(os.path.join(G.GOLDEN, "tlas", "tlas_24.npz")))
    v = [g["verts0"], g["verts1"]]
    blas = [portpy.PortBVH(x) for x in v]
    inst = g["instances_raw"].view(refpy.BLAS_INSTANCE).reshape(-1).copy()
    lo = np.stack([b.nodes[0]["aabbMin"] for b in blas])[inst["blasIdx"]]
    hi = np.stack([b.nodes[0]["aabbMax"] for b in blas])[inst["blasIdx"]]
    portpy.instance_update(inst, lo, hi)
    assert np.array_equal(inst.view(np.uint32).reshape(-1, 48), g["instances"])
    # the TLAS is the reference builder's tree over the instance boxes: a "triangle" (min, max, min) has exactly that box
    fake = np.zeros((inst.shape[0] * 3, 4), np.float32)
    fake[0::3, :3], fake[1::3, :3], fake[2::3, :3] = inst["aabbMin"], inst["aabbMax"], inst["aabbMin"]
    tl = portpy.PortBVH(fake)
    assert np.array_equal(tl.nodes.view(np.uint32).reshape(-1, 8), g["tlas_nodes"]) and np.array_equal(tl.prim_idx, g["tlas_prim_idx"])
    port = portpy.PortTLAS(tl.nodes, tl.prim_idx, inst, blas)
    for mask in (1, 2):
        r = np.zeros(g["rays_O"].shape[0], R.RAY_DTYPE)
        r["O"], r["D"], r["rD"], r["t"], r["mask"] = g["rays_O"], g["rays_D"], g["rays_rD"], g["rays_tmax"], mask
        sh = r.copy()
        sh["t"] = 150.0
        port.intersect(r)
        assert np.array_equal(r.view(np.uint32).reshape(-1, 32)[:, 11:16], g[f"hit_mask{mask}"])
        assert np.array_equal(port.occluded(sh), g[f"occluded_mask{mask}"])


@pytest.mark.parametrize("path", G.golden_files(), ids=lambda p: p.split("/")[-1])
def test_port_refit_matches_golden(path):
    g = G.load(path)
    port = portpy.PortBVH(g["verts"])
    port.refit(g["refit_verts"])
    assert np.array_equal(port.nodes.view(np.uint32).reshape(-1, 8), g["refit_nodes"])


@pytest.mark.skipif(not refpy.available(), reason="oracle/_ref not built (needs /root/reference)")
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_port_sah_cost_matches_reference(mode):
    """BVH::SAHCost (:1889) of the Build / BuildAVX / BuildHQ trees, the number the speedtest prints."""
    v = scenes.procedural_scene(20000, 71)
    ref = refpy.RefBVH(v, mode=mode, threaded=False)
    nodes = ref.nodes   # a copy: keep it alive while C reads it
    got = np.float32(portpy.lib().orc_sah_cost(nodes.ctypes.data, 0, 1.0, 1.0))
    assert got.view(np.uint32) == np.float32(ref.sah_cost()).view(np.uint32)


# ---------------------------------------------------------------- CWBVH chain + CPU walk restatement, oracle/tbvh_oracle_cwbvh.c
@pytest.mark.parametrize("path", G.golden_files(), ids=lambda p: p.split("/")[-1])
def test_port_cwbvh_matches_golden(path):
    g = G.load(path)
    if "cwbvh_nodes" not in g:
        pytest.skip("single-node scene: the reference refuses to convert it (:5889)")
    port = portpy.PortBVH(g["verts"])
    cw = portpy.PortCWBVH(port.nodes, port.prim_idx, g["verts"])
    assert np.array_equal(cw.nodes.view(np.uint32), g["cwbvh_nodes"])
    assert np.array_equal(cw.tris.view(np.uint32), g["cwbvh_tris"])
    lo, hi = scenes.scene_bounds(g["verts"])
    res = int(round((g["cwbvh_primary_hit"].shape[0] // 4) ** 0.5))
    r = R.primary_rays(*R.bounds_camera(lo, hi, "outside"), res, res, 4)
    cw.intersect(r)
    assert np.array_equal(G.hits_as_u32(r), g["cwbvh_primary_hit"])


@pytest.mark.skipif(not refpy.available(), reason="oracle/_ref not built (needs /root/reference)")
@pytest.mark.parametrize("ntris,cw_mode,bvh_mode", [(20000, 0, 1), (5000, 1, 2), (3000, 2, 0), (5, 2, 0)])
def test_port_cwbvh_matches_reference(ntris, cw_mode, bvh_mode):
    """BVH8_CWBVH::Build (BuildAVX tree) / BuildHQ (SBVH) / the scalar-Build chain: bvh8Data and the referenced bvh8Tris byte for
    byte, BVH8_CWBVH::Intersect hits bit for bit."""
    v = scenes.procedural_scene(ntris, seed=81)
    ref = refpy.RefCWBVH(v, mode=cw_mode)
    b = refpy.RefBVH(v, mode=bvh_mode, threaded=False)
    nodes = b.nodes
    used = int(nodes["triCount"].sum())
    port = portpy.PortCWBVH(nodes, b.prim_idx[:used], v, idx_count=b.idx_count)
    assert np.array_equal(port.nodes.view(np.uint32), ref.nodes.view(np.uint32))
    assert np.array_equal(port.tris[: used * 3].view(np.uint32), ref.tris[: used * 3].view(np.uint32))
    lo, hi = scenes.scene_bounds(v)
    a = R.primary_rays(*R.bounds_camera(lo, hi, "inside"), 64, 64, 4)
    c = a.copy()
    ref.intersect(a, threads=1), port.intersect(c)
    assert np.array_equal(G.hits_as_u32(a), G.hits_as_u32(c))


@pytest.mark.parametrize("ntris,seed,res,primary,diffuse", [(30000, 31, 96, 0, 8), (900, 32, 64, 69, 0), (20, 33, 32, 0, 0)])
def test_reference_layouts_disagree_on_a_pinned_set_of_rays(ntris, seed, res, primary, diffuse):
    """The tie audit of SURVEY 8(c), pinned: on the seeded scenes of tests/test_cwbvh_gpu.py the reference's own CWBVH walk
    (BVH8_CWBVH::Intersect) and its BVH walk (BVH::Intersect) of the same triangles disagree on exactly this many rays (exact-distance ties;
    rays with a zero direction component, whose quantised plane distances overflow in the wide walk).  The GPU test then requires the engine's
    CWBVH kernel to differ from BVH::Intersect on exactly the same rays as the reference's walk does - so these counts are the engine's too.
    The counts were recorded from the compiled reference; without oracle/_ref the port's restatement of both walks must reproduce them."""
    from tests import util
    v = scenes.procedural_scene(ntris, seed)
    cw, o = util.reference().RefCWBVH(v, mode=2), util.oracle_bvh(v)
    sets, bounds = util.ray_sets(v, res=res)
    dis = lambda a, b: int(((a["prim"] != b["prim"]) | (a["t"].view(np.uint32) != b["t"].view(np.uint32))).sum())
    a, b = sets["primary"].copy(), sets["primary"].copy()
    cw.intersect(a), o.intersect(b)
    assert dis(a, b) == primary
    d = util.derived_sets(b, v, bounds)
    a, b = d["diffuse"].copy(), d["diffuse"].copy()
    cw.intersect(a), o.intersect(b)
    assert dis(a, b) == diffuse
