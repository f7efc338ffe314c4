"""The shipped traversal and host-buffer paths give the oracle's results on every route a batch can take (host and device
buffers, pinned and pageable memory, packed and in-place hits, several pipeline chunks), and the context options that
remain (tbvh_set_option: small_t, build_mode) change how the tree is built, never the tree."""
import numpy as np
import pytest

from tinybvh_b200 import api, rays as R, scenes
from tests import util

pytestmark = pytest.mark.gpu
ZERO = {"prim": 0, "t": 0, "u": 0, "v": 0}


@pytest.fixture(scope="module")
def world():
    v = scenes.procedural_scene(40000, 71)
    o = util.oracle_bvh(v)
    sets, bounds = util.ray_sets(v, res=128)
    prim = sets["primary"].copy()
    o.intersect(prim)
    d = util.derived_sets(prim, v, bounds)
    want = {"primary": prim, "diffuse": d["diffuse"].copy(), "shadow_bits": o.occluded(d["shadow"])}
    o.intersect(want["diffuse"])
    return v, sets["primary"], d, want


def test_bvh2_traversal_is_bit_exact(gpu, world):
    v, primary, d, want = world
    import torch
    e = api.BVH().Build(v)
    for name, rays in (("primary", primary), ("diffuse", d["diffuse"])):
        got = rays.copy()
        e.Intersect(got)
        assert util.compare_hits(got, want[name]) == ZERO, name
        # device path with a ragged count (a partial last warp and block)
        m = rays.shape[0] - 37
        dev = torch.from_numpy(R.gpu_records(rays[:m]).view(np.uint8).reshape(-1, 64).copy()).cuda()
        hits = torch.zeros((m, 4), dtype=torch.float32, device="cuda")
        e.Intersect(dev, hits=hits)
        torch.cuda.synchronize()
        h = hits.cpu().numpy()
        assert np.array_equal(h[:, 0].view(np.uint32), want[name]["t"][:m].view(np.uint32))
        assert np.array_equal(h[:, 3].view(np.uint32), want[name]["prim"][:m])
    assert np.array_equal(e.IsOccluded(d["shadow"]), want["shadow_bits"]), "occlusion"
    m = d["shadow"].shape[0] - 37
    assert np.array_equal(e.IsOccluded(d["shadow"][:m].copy()), util.oracle_bvh(v).occluded(d["shadow"][:m].copy()))


def test_host_path_returns_the_same_hits_from_every_buffer(gpu, world):
    v, primary, d, want = world
    e = api.BVH().Build(v)
    n = primary.shape[0]
    pinned = api.pinned_empty(n, R.RAY_DTYPE)
    pinned[:] = primary
    e.Intersect(pinned)
    assert util.compare_hits(pinned, want["primary"]) == ZERO, "pinned"
    pageable = primary.copy()
    e.Intersect(pageable)
    assert util.compare_hits(pageable, want["primary"]) == ZERO, "pageable"
    hits = e.IntersectPacked(primary)   # packed return path: rays untouched, 16-byte hits
    assert np.array_equal(hits["t"].view(np.uint32), want["primary"]["t"].view(np.uint32)) and np.array_equal(hits["prim"], want["primary"]["prim"])
    api.pinned_free(pinned)


def test_retired_option_keys_are_rejected(gpu):
    for key in ("trace_variant", "d2h_mode", "chunk_rays"):
        with pytest.raises(api.TbvhError):
            api.set_option(key, 0)


@pytest.mark.parametrize("small_t", [8, 64, 256])
def test_builder_switch_point_does_not_change_the_tree(gpu, small_t):
    v = scenes.procedural_scene(30000, 72)
    o = util.oracle_bvh(v)
    api.set_option("small_t", small_t)
    try:
        nodes, idx = api.BVH().Build(v).download()
        assert np.array_equal(nodes.view(np.uint32), np.ascontiguousarray(o.nodes).view(np.uint32)) and np.array_equal(idx, o.prim_idx)
    finally:
        api.set_option("small_t", 128)


def test_long_host_batches(gpu):
    """Host batches longer than a pipeline chunk, several chunks in flight on different streams: every chunk's hits and
    occlusion words land in the right records, and statistics add up over the chunks of one call."""
    v = scenes.procedural_scene(30000, 73)
    o = util.oracle_bvh(v)
    lo, hi = scenes.scene_bounds(v)
    rays = R.primary_rays(*R.bounds_camera(lo, hi, "inside"), 384, 384, 16)   # 2,359,296 rays = 4.5 chunks of 2^19
    want = rays.copy()
    o.intersect(want, threads=0)
    sh = util.derived_sets(want, v, (lo, hi))["shadow"]
    want_bits = o.occluded(sh, threads=0)
    e = api.BVH().Build(v)
    got = rays.copy()
    e.Intersect(got)
    assert util.compare_hits(got, want) == ZERO
    assert np.array_equal(e.IsOccluded(sh), want_bits), "occlusion"
    # statistics of a multi-chunk call = statistics of the same rays traced in one device launch
    import torch
    e.set_stats(True)
    got = rays.copy()
    e.Intersect(got)
    host_stats = e.get_stats()
    dev = torch.from_numpy(R.gpu_records(rays).view(np.uint8).reshape(-1, 64).copy()).cuda()
    e.Intersect(dev)
    torch.cuda.synchronize()
    assert e.get_stats() == host_stats and host_stats[0] > rays.shape[0]
    e.set_stats(False)


def test_concurrent_host_calls_on_one_handle(gpu):
    """SURVEY 8(b): batch calls are thread-safe per handle (the reference's const Intersect is called from many threads)."""
    import threading
    v = scenes.procedural_scene(20000, 74)
    o = util.oracle_bvh(v)
    lo, hi = scenes.scene_bounds(v)
    e = api.BVH().Build(v)
    sets, errs = [], []
    for k, kind in enumerate(("inside", "outside", "inside", "outside")):
        r = R.primary_rays(*R.bounds_camera(lo, hi, kind), 192 + 64 * k, 192, 16)
        w = r.copy()
        o.intersect(w, threads=0)
        sets.append((r, w))

    def work(r, w):
        try:
            for _ in range(3):
                g = r.copy()
                e.Intersect(g)
                if util.compare_hits(g, w) != ZERO:
                    errs.append("mismatch")
        except Exception as ex:  # noqa: BLE001
            errs.append(repr(ex))

    th = [threading.Thread(target=work, args=s) for s in sets]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errs, errs


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("ntris,seed", [(90000, 75), (3000, 76), (129, 77)])
def test_both_large_phase_drivers_build_the_reference_tree(gpu, mode, ntris, seed):
    """build_mode 0 = the persistent cooperative launch (k_large_phase), 1 = one launch per stage and level: same tree, byte for byte."""
    v = scenes.procedural_scene(ntris, seed)
    o = util.oracle_bvh(v)
    api.set_option("build_mode", mode)
    try:
        nodes, idx = api.BVH().Build(v).download()
        assert np.array_equal(nodes.view(np.uint32), np.ascontiguousarray(o.nodes).view(np.uint32)) and np.array_equal(idx, o.prim_idx)
        nodes2, _ = api.BVH().BuildAVX(v).download()
        from oracle import refpy
        if refpy.available():
            ra = refpy.RefBVH(v, mode=1, threaded=False)
            assert np.array_equal(nodes2.view(np.uint32), np.ascontiguousarray(ra.nodes).view(np.uint32))
    finally:
        api.set_option("build_mode", 0)
