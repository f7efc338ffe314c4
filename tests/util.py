"""Shared helpers for the parity tests: oracle selection, ray sets, comparators."""
import numpy as np

from tinybvh_b200 import rays as R, scenes
from oracle import portpy, refpy


def oracle_bvh(verts):
    """The parity oracle for a triangle soup: the compiled reference (BVH::Build + Intersect/IsOccluded) when
    oracle/_ref exists, else the pinned plain-C restatement.  Both expose .nodes/.prim_idx/.intersect/.occluded."""
    if refpy.available():
        return refpy.RefBVH(verts, mode=0, threaded=False)
    return portpy.PortBVH(verts)


class PortReference:
    """The reference objects of oracle/refpy.py that the GPU parity tests use, restated on the plain-C port (oracle/tbvh_oracle*.c).
    The port is pinned bit for bit to the reference by tests/test_oracle_pin.py (committed golden vectors everywhere, the compiled
    reference where oracle/_ref exists), so a checkout without the compiled reference still runs every parity check that the port
    can restate.  Not restated: the threaded builders' node numbering and BVH::Intersect's cost return value."""

    class RefBVH:
        """mode 0 BVH::Build, 1 BuildAVX, 2 BuildHQ + Compact.  The ( vertices, indices ) overloads build the tree of the flat soup
        verts[indices] (test_reference_indexed_build_equals_flat_build)."""

        def __init__(self, verts, mode=0, threaded=False, indices=None):
            assert not threaded, "the port numbers nodes as the single-threaded builders do"
            v = np.ascontiguousarray(verts, np.float32).reshape(-1, 4)
            self.verts = v if indices is None else np.ascontiguousarray(v[np.asarray(indices, np.int64).reshape(-1)])
            if mode == 2:
                nodes, idx, self.idx_count = portpy.build_hq(self.verts)
                self.port = portpy.PortBVH(self.verts, nodes=nodes, prim_idx=idx)
            else:
                self.port = portpy.PortBVH(self.verts, avx=mode == 1)
                self.idx_count = self.port.prim_idx.shape[0]
            self.nodes, self.prim_idx, self.used_nodes = self.port.nodes, self.port.prim_idx, self.port.used_nodes

        def intersect(self, rays, threads=0):
            return self.port.intersect(rays, threads)

        def occluded(self, rays, threads=0):
            return self.port.occluded(rays, threads)

    class RefBVHGPU:
        def __init__(self, bvh):
            self.nodes = bvh.port.to_bvh_gpu()

    class RefCWBVH:
        """mode 0 BVH8_CWBVH::Build (the chain over the BuildAVX tree), 1 BuildHQ (over the SBVH), 2 the chain over BVH::Build's tree."""

        def __init__(self, verts, mode=2):
            self.src = PortReference.RefBVH(verts, mode={0: 1, 1: 2, 2: 0}[mode])
            used = int(self.src.nodes["triCount"].sum())
            self.port = portpy.PortCWBVH(self.src.nodes, self.src.prim_idx[:used], self.src.verts, idx_count=self.src.idx_count)
            self.nodes, self.tris = self.port.nodes, self.port.tris

        def source_bvh(self):
            return self.src

        def intersect(self, rays, threads=0):
            return self.port.intersect(rays)

    class RefTLAS:
        """BVH::Build( BLASInstance*, .. ): BLASInstance::Update of every record in place, then the BVH::Build tree over the instance boxes
        (a 'triangle' (min, max, min) has exactly that box), walked by IntersectTLAS / IsOccludedTLAS."""

        def __init__(self, instances, blasses):
            lo = np.stack([b.nodes[0]["aabbMin"] for b in blasses])[instances["blasIdx"]]
            hi = np.stack([b.nodes[0]["aabbMax"] for b in blasses])[instances["blasIdx"]]
            portpy.instance_update(instances, lo, hi)
            boxes = np.zeros((instances.shape[0] * 3, 4), np.float32)
            boxes[0::3, :3], boxes[1::3, :3], boxes[2::3, :3] = instances["aabbMin"], instances["aabbMax"], instances["aabbMin"]
            self.tlas = portpy.PortBVH(boxes)
            self.port = portpy.PortTLAS(self.tlas.nodes, self.tlas.prim_idx, instances, [b.port for b in blasses])

        def bvh(self):
            return self.tlas

        def intersect(self, rays, threads=0):
            return self.port.intersect(rays)

        def occluded(self, rays, threads=0):
            return self.port.occluded(rays)


def reference():
    """The compiled reference (oracle/refpy) when oracle/_ref exists, else its restatement on the pinned port."""
    return refpy if refpy.available() else PortReference


def small_scene(ntris=6000, seed=7):
    return scenes.procedural_scene(ntris, seed)


def ray_sets(verts, res=96, seed=0x123456):
    """primary (2 cameras) + shadow + diffuse rays over a scene; dict name -> RAY_DTYPE array (untraced)."""
    lo, hi = scenes.scene_bounds(verts)
    out = {}
    prim = []
    for kind in ("outside", "inside"):
        eye, view = R.bounds_camera(lo, hi, kind)
        prim.append(R.primary_rays(eye, view, res, res, 4))
    out["primary"] = np.concatenate(prim)
    return out, (lo, hi)


def derived_sets(traced_primary, verts, bounds):
    lo, hi = bounds
    eps = float((hi - lo).max() * 5e-7)
    light = (lo + hi) * 0.5 + np.array([0, (hi - lo)[1] * 0.45, 0], np.float32)
    return {"shadow": R.shadow_rays(traced_primary, light, eps), "diffuse": R.diffuse_rays(traced_primary, verts)}


def bits_u32(a):
    return np.ascontiguousarray(a).view(np.uint32)


def compare_hits(got, want):
    """-> dict of mismatch counts between two traced ray arrays (bit-exact fields)."""
    return {
        "prim": int((got["prim"] != want["prim"]).sum()),
        "t": int((bits_u32(got["t"]) != bits_u32(want["t"])).sum()),
        "u": int((bits_u32(got["u"]) != bits_u32(want["u"])).sum()),
        "v": int((bits_u32(got["v"]) != bits_u32(want["v"])).sum()),
    }


def classify_mismatches(got, want, verts):
    """Tie audit (SURVEY 8c): for rays whose prim differs from the oracle's, re-evaluate the engine's prim with the
    oracle's Moeller-Trumbore arithmetic.  exact-tie = bit-identical t; otherwise 'real'."""
    bad = np.nonzero(got["prim"] != want["prim"])[0]
    ties = real = 0
    v = verts.reshape(-1, 3, 4)
    for i in bad:
        p = int(got["prim"][i])
        ok, t, u, vv = portpy.tri_test(want["O"][i], want["D"][i], v[p, 0, :3], v[p, 1, :3], v[p, 2, :3], 1e30)
        if ok and np.float32(t).view(np.uint32) == want["t"][i].view(np.uint32):
            ties += 1
        else:
            real += 1
    return {"mismatch": int(bad.size), "tie_equivalent": ties, "real": real}


def random_transforms(count, seed, spread=60.0):
    """Row-major 4x4 instance transforms: rotation x (non-uniform) scale x translation, as tiny_bvh's bvhmat4 stores them."""
    rng = np.random.default_rng(seed)
    out = np.zeros((count, 16), np.float32)
    for i in range(count):
        a, b, c = rng.random(3) * 6.28
        rx = np.array([[1, 0, 0], [0, np.cos(a), -np.sin(a)], [0, np.sin(a), np.cos(a)]])
        ry = np.array([[np.cos(b), 0, np.sin(b)], [0, 1, 0], [-np.sin(b), 0, np.cos(b)]])
        rz = np.array([[np.cos(c), -np.sin(c), 0], [np.sin(c), np.cos(c), 0], [0, 0, 1]])
        m = np.eye(4)
        m[:3, :3] = (rx @ ry @ rz) @ np.diag(0.4 + rng.random(3) * 1.2)
        m[:3, 3] = (rng.random(3) - 0.5) * spread
        out[i] = m.astype(np.float32).reshape(-1)
    return out
