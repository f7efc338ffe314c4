#!/usr/bin/env python
"""Developer timing probe (NOT the bench): device-resident traversal throughput on a fixture with the oracle's tree."""
import os
import sys
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from tinybvh_b200 import api, rays as R, scenes  # noqa: E402
from tests import util  # noqa: E402


def timeit(fn, reps=5):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return min(ts), sorted(ts)[len(ts) // 2]


def main():
    scene = sys.argv[1] if len(sys.argv) > 1 else "sponza"
    res = int(sys.argv[2]) if len(sys.argv) > 2 else 512
    v, label = scenes.load_scene(scene)
    builder = "BuildHQ" if "--hq" in sys.argv else "Build"   # --hq: trace the SBVH
    e = getattr(api.BVH(), builder)(v)
    e = getattr(api.BVH(), builder)(v)
    i = e.info()
    print(f"{label}: {v.shape[0] // 3} tris, GPU build {i.build_ms:.3f} ms ({v.shape[0] // 3 / i.build_ms / 1e3:.1f} Mtris/s), nodes {i.used_nodes}, depth {i.max_depth}")
    layout = sys.argv[3] if len(sys.argv) > 3 and not sys.argv[3].startswith("--") else "bvh"
    if layout == "cwbvh":
        import ctypes as C
        t0 = time.time()
        api.check(api._lib.lib().tbvh_convert(e.h, api.LAYOUT_CWBVH))
        print(f"CWBVH conversion on device: {(time.time() - t0) * 1e3:.1f} ms wall, {e.info().used_blocks // 5} nodes")
        e.layout = api.LAYOUT_CWBVH
    lo, hi = scenes.scene_bounds(v)
    if scene == "sponza":
        eye, view = R.SPONZA_EYES[0], R.SPONZA_VIEWS[0]
    else:
        eye, view = R.bounds_camera(lo, hi, "inside" if scene == "bistro" else "outside")
    prim = R.primary_rays(eye, view, res, res, 16)
    n = prim.shape[0]
    dprim = torch.from_numpy(R.gpu_records(prim).view(np.uint8).reshape(-1, 64)).cuda()
    hits = torch.empty((n, 4), dtype=torch.float32, device="cuda")
    e.set_stats(True)
    e.Intersect(dprim, hits=hits)
    steps, tris = e.get_stats()[:2]
    e.set_stats(False)
    print(f"primary: {n} rays, {steps / n:.1f} steps/ray, {tris / n:.2f} tris/ray")
    best, med = timeit(lambda: e.Intersect(dprim, hits=hits))
    print(f"primary  closest: best {best:.3f} ms  {n / best / 1e3:.1f} Mrays/s (median {n / med / 1e3:.1f})")
    # shadow + diffuse from traced primaries (host side generation)
    traced = prim.copy()
    h = hits.cpu().numpy()
    traced["t"], traced["u"], traced["v"], traced["prim"] = h[:, 0], h[:, 1], h[:, 2], h[:, 3].view(np.uint32)
    eps = float((hi - lo).max() * 5e-7)
    light = (lo + hi) * 0.5 + np.array([0, (hi - lo)[1] * 0.45, 0], np.float32) if scene != "sponza" else np.zeros(3, np.float32)
    sh = R.shadow_rays(traced, light, eps)
    dsh = torch.from_numpy(R.gpu_records(sh).view(np.uint8).reshape(-1, 64)).cuda()
    bits = torch.empty((n + 31) // 32, dtype=torch.int32, device="cuda")
    best, med = timeit(lambda: e.IsOccluded(dsh, bits=bits))
    occ = int(np.unpackbits(bits.cpu().numpy().view(np.uint8)).sum())
    print(f"shadow   anyhit : best {best:.3f} ms  {n / best / 1e3:.1f} Mrays/s (median {n / med / 1e3:.1f}) occluded {occ}")
    df = R.diffuse_rays(traced, v)
    ddf = torch.from_numpy(R.gpu_records(df).view(np.uint8).reshape(-1, 64)).cuda()
    e.set_stats(True)
    e.Intersect(ddf, hits=hits)
    steps, tris = e.get_stats()[:2]
    e.set_stats(False)
    best, med = timeit(lambda: e.Intersect(ddf, hits=hits))
    print(f"diffuse  closest: best {best:.3f} ms  {n / best / 1e3:.1f} Mrays/s (median {n / med / 1e3:.1f})  {steps / n:.1f} steps/ray {tris / n:.2f} tris/ray")
    # host path (pinned) e2e
    hp = api.pinned_empty(n, R.RAY_DTYPE)
    hp[:] = prim
    t0 = time.time()
    e.Intersect(hp)
    t1 = time.time()
    e.Intersect(hp)
    t2 = time.time()
    print(f"host path e2e (pinned, 128B stride): {n / (t2 - t1) / 1e6:.1f} Mrays/s (first {n / (t1 - t0) / 1e6:.1f})")
    # CPU reference on a sample
    from oracle import refpy
    if refpy.available() and "--cpu" in sys.argv:
        o = util.oracle_bvh(v)
        smp = prim[: min(n, 1 << 20)].copy()
        t0 = time.time()
        o.intersect(smp, threads=0)
        dt = time.time() - t0
        print(f"CPU BVH::Intersect all threads ({refpy.hardware_threads()}): {smp.shape[0] / dt / 1e6:.1f} Mrays/s")
        b8 = refpy.RefBVH8CPU(v)
        smp = prim[: min(n, 1 << 21)].copy()
        t0 = time.time()
        b8.intersect(smp, threads=0)
        dt = time.time() - t0
        print(f"CPU BVH8_CPU all threads: {smp.shape[0] / dt / 1e6:.1f} Mrays/s")


if __name__ == "__main__":
    main()
