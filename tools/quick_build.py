#!/usr/bin/env python
"""Developer probe: GPU build time of a scene at the builder's switch points small_t (--all: 64 and 128)."""
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from tinybvh_b200 import api, scenes  # noqa: E402

for scene in [a for a in sys.argv[1:] if not a.startswith("--")] or ["sponza"]:
    v, label = scenes.load_scene(scene)
    n = v.shape[0] // 3
    for t in ((64, 128) if "--all" in sys.argv else (128,)):
        api.set_option("small_t", t)
        best = 1e9
        for _ in range(3):
            e = api.BVH().Build(v)
            best = min(best, e.info().build_ms)
        print(f"{label}: {n} tris small_t {t}: build {best:.3f} ms = {n / best / 1e3:.1f} Mtris/s  (nodes {e.info().used_nodes})", flush=True)
