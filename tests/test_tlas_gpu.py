"""GPU parity of the two-level path: BVH::Build( BLASInstance*, .. ) (tiny_bvh.h:2221) + IntersectTLAS (:3306) / IsOccludedTLAS
(:3455).  The TLAS node array is the reference's byte for byte; hits (inst, t, u, v, prim) and occlusion bits are identical."""
import numpy as np
import pytest

from tinybvh_b200 import api, rays as R, scenes
from tests import util
from tests.test_oracle_pin import tlas_case

pytestmark = pytest.mark.gpu


def words(r):
    return r.view(np.uint32).reshape(-1, 32)[:, 11:16]   # hit.inst, t, u, v, prim


@pytest.mark.parametrize("n_inst,builder", [(40, "Build"), (1, "Build"), (300, "BuildAVX"), (40, "BuildHQ")])
def test_tlas_matches_reference(gpu, n_inst, builder):
    REF = util.reference()
    v, inst, O, D = tlas_case(91, n_inst)
    mode = {"Build": 0, "BuildAVX": 1, "BuildHQ": 2}[builder]
    inst_ref = inst.copy()
    ref = REF.RefTLAS(inst_ref, [REF.RefBVH(x, mode=mode, threaded=False) for x in v])   # Update()s inst_ref in place
    blas = [getattr(api.BVH(), builder)(x) for x in v]
    t = api.TLAS().Build(inst, blas)                                                         # the engine Update()s inst in place
    assert inst.tobytes() == inst_ref.tobytes(), "BLASInstance::Update differs"
    nodes, idx = t.download()
    rb = ref.bvh()
    assert np.array_equal(nodes.view(np.uint32), rb.nodes.view(np.uint32)) and np.array_equal(idx, rb.prim_idx), "TLAS tree differs"
    for mask in (0x1, 0x2):
        rays = R.make_rays(O, D)
        rays["mask"] = mask
        want, got = rays.copy(), rays.copy()
        ref.intersect(want), t.Intersect(got)
        assert np.array_equal(words(got), words(want)), f"closest hits differ (ray mask {mask:#x})"
        sh = R.make_rays(O, D, tmax=150.0)
        sh["mask"] = mask
        assert np.array_equal(t.IsOccluded(sh), ref.occluded(sh))
    hit = want["t"] < 1e30
    assert hit.sum() > 1000


def test_tlas_matches_golden_vectors(gpu):
    """The reference's TLAS path as recorded in tests/golden/tlas (tools/make_golden.py make_tlas): BLASInstance::Update, the TLAS tree,
    IntersectTLAS hits (inst, t, u, v, prim) and IsOccludedTLAS bits for two ray masks."""
    import os
    from oracle import refpy
    from tests import golden_util as G
    g = dict(np.load(os.path.join(G.GOLDEN, "tlas", "tlas_24.npz")))
    inst = g["instances_raw"].view(refpy.BLAS_INSTANCE).reshape(-1).copy()
    t = api.TLAS().Build(inst, [api.BVH().Build(g["verts0"]), api.BVH().Build(g["verts1"])])
    assert np.array_equal(inst.view(np.uint32).reshape(-1, 48), g["instances"]), "BLASInstance::Update differs"
    nodes, idx = t.download()
    assert np.array_equal(nodes.view(np.uint32).reshape(-1, 8), g["tlas_nodes"]) and np.array_equal(idx, g["tlas_prim_idx"]), "TLAS tree differs"
    for mask in (1, 2):
        r = np.zeros(g["rays_O"].shape[0], R.RAY_DTYPE)
        r["O"], r["D"], r["rD"], r["t"], r["mask"] = g["rays_O"], g["rays_D"], g["rays_rD"], g["rays_tmax"], mask
        sh = r.copy()
        sh["t"] = 150.0
        t.Intersect(r)
        assert np.array_equal(words(r), g[f"hit_mask{mask}"]), f"closest hits differ (ray mask {mask:#x})"
        assert np.array_equal(t.IsOccluded(sh), g[f"occluded_mask{mask}"])


def test_tlas_device_rays_and_errors(gpu):
    import torch
    REF = util.reference()
    v, inst, O, D = tlas_case(93, 24)
    ref = REF.RefTLAS(inst, [REF.RefBVH(x, mode=0, threaded=False) for x in v])
    blas = [api.BVH().Build(x) for x in v]
    t = api.TLAS().Build(inst, blas, update=False)   # records already updated by the reference: the "blasses == 0" contract
    rays = R.make_rays(O, D)
    want = rays.copy()
    ref.intersect(want)
    d = torch.from_numpy(rays.view(np.uint8).reshape(-1, 128)).cuda()
    t.Intersect(d)
    got = d.cpu().numpy().view(R.RAY_DTYPE).reshape(-1)
    assert np.array_equal(words(got), words(want))
    with pytest.raises(api.TbvhError):
        t.IntersectPacked(rays)                      # TLAS hits carry the instance: in place only
    with pytest.raises(api.TbvhError):
        api.TLAS().Build(inst, [blas[0]])            # an instance names BLAS 1
    with pytest.raises(api.TbvhError):
        api.TLAS().Build(inst, [blas[0], t])         # a TLAS is not a BLAS


def test_tlas_instance_bits_in_prim(gpu):
    """A host program compiled with INST_IDX_BITS 10 (the speedtest's setting): the instance rides in the top bits of hit.prim."""
    REF = util.reference()
    v, inst, O, D = tlas_case(95, 30)
    ref = REF.RefTLAS(inst, [REF.RefBVH(x, mode=0, threaded=False) for x in v])
    t = api.TLAS().Build(inst, [api.BVH().Build(x) for x in v])
    rays = R.make_rays(O, D)
    want, got = rays.copy(), rays.copy()
    ref.intersect(want)                                   # reference built with INST_IDX_BITS 32: inst in its own field
    api.set_option("inst_idx_bits", 10)
    try:
        t.Intersect(got)
    finally:
        api.set_option("inst_idx_bits", 32)
    hit = want["t"] < 1e30
    w, g = words(want), words(got)
    assert np.array_equal(g[:, 1:4], w[:, 1:4])           # t, u, v
    assert np.array_equal(g[hit, 4], w[hit, 4] + (w[hit, 0] << 22)) and np.array_equal(g[~hit, 4], w[~hit, 4])
    assert np.array_equal(g[:, 0], words(rays)[:, 0])     # byte 44 untouched


class _CW:
    def __init__(self, blas):
        self.nodes, self.tris = blas.download()          # bvh8Data / bvh8Tris, byte-identical to the reference's converter (tests/test_convert_gpu.py)


@pytest.mark.parametrize("n_inst,builder", [(40, "Build"), (1, "Build"), (200, "BuildHQ")])
def test_tlas_over_cwbvh_blasses(gpu, n_inst, builder):
    """The BLASses walked in their BVH8_CWBVH layout (the reference's GPU arrangement, traverse_tlas.cl): bit-identical to the oracle's
    composition of IntersectTLAS's walk with BVH8_CWBVH::Intersect per instance (oracle/tbvh_oracle.h, orc_intersect_tlas_cw)."""
    from oracle import portpy
    v, inst, O, D = tlas_case(97, n_inst)
    blas = [getattr(api.BVH8_CWBVH(), builder)(x) for x in v]
    t = api.TLAS().Build(inst, blas, blas_layout=api.LAYOUT_CWBVH)
    nodes, idx = t.download()
    port = portpy.PortTLASCW(nodes, idx, inst, [_CW(b) for b in blas])
    t_bvh = api.TLAS().Build(inst.copy(), blas)           # the same instances, BLASses walked through their BVH layout
    for mask in (0x1, 0x2):
        rays = R.make_rays(O, D)
        rays["mask"] = mask
        want, got, other = rays.copy(), rays.copy(), rays.copy()
        port.intersect(want), t.Intersect(got), t_bvh.Intersect(other)
        assert np.array_equal(words(got), words(want)), f"closest hits differ (ray mask {mask:#x})"
        assert n_inst == 1 or (want["t"] < 1e30).sum() > 1000   # (the single instance of the n_inst = 1 case carries mask 0x2 only)
        assert (words(got) == words(other)).all(axis=1).mean() > 0.999   # two layouts of the same triangles: ties aside, the same hits
        sh = R.make_rays(O, D, tmax=150.0)
        sh["mask"] = mask
        assert np.array_equal(t.IsOccluded(sh), port.occluded(sh))
    # device-resident rays
    import torch
    rays = R.make_rays(O, D)
    want = rays.copy()
    port.intersect(want)
    d = torch.from_numpy(rays.view(np.uint8).reshape(-1, 128)).cuda()
    t.Intersect(d)
    assert np.array_equal(words(d.cpu().numpy().view(R.RAY_DTYPE).reshape(-1)), words(want))
    bits = t.IsOccluded(torch.from_numpy(R.make_rays(O, D, tmax=150.0).view(np.uint8).reshape(-1, 128)).cuda())
    assert np.array_equal(bits.cpu().numpy().view(np.uint32), port.occluded(R.make_rays(O, D, tmax=150.0)))


def test_tlas_over_cwbvh_uploaded_and_errors(gpu):
    """BLASses that hold ONLY the CWBVH arrays (uploaded bvh8Data / bvh8Tris); layout / staleness errors."""
    from oracle import portpy
    v, inst, O, D = tlas_case(99, 30)
    built = [api.BVH8_CWBVH().Build(x) for x in v]
    t0 = api.TLAS().Build(inst, built, blas_layout=api.LAYOUT_CWBVH)    # Update()s inst
    cws = [_CW(b) for b in built]
    only_cw = [api.BVH8_CWBVH().upload(c.nodes, c.tris) for c in cws]
    t = api.TLAS().Build(inst, only_cw, update=False, blas_layout=api.LAYOUT_CWBVH)
    nodes, idx = t.download()
    port = portpy.PortTLASCW(nodes, idx, inst, cws)
    rays = R.make_rays(O, D)
    want, got = rays.copy(), rays.copy()
    port.intersect(want), t.Intersect(got)
    assert np.array_equal(words(got), words(want)) and (want["t"] < 1e30).sum() > 1000
    t.layout = api.LAYOUT_BVH
    with pytest.raises(api.TbvhError):
        t.Intersect(rays.copy())                          # these BLASses hold no BVH-layout tree
    plain = [api.BVH().Build(x) for x in v]
    tb = api.TLAS().Build(inst.copy(), plain)
    tb.layout = api.LAYOUT_CWBVH
    with pytest.raises(api.TbvhError):
        tb.Intersect(rays.copy())                         # ... and these no CWBVH
    built[0].Build(v[0])                                  # the BLAS was rebuilt and re-converted: its arrays moved
    with pytest.raises(api.TbvhError):
        t0.Intersect(rays.copy())
