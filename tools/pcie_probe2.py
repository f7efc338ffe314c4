#!/usr/bin/env python
"""Developer probe: host-buffer path throughput (tbvh_intersect / tbvh_occluded on 128-byte host records) against where the ray
buffer lives (NUMA-local or wherever the process happened to start).  A one-triangle scene makes the
traversal free, so the call time is transfer time.   python tools/pcie_probe2.py [n_rays_log2]"""
import os
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from tinybvh_b200 import api, rays as R, _lib  # noqa: E402

n = 1 << (int(sys.argv[1]) if len(sys.argv) > 1 else 24)
L = _lib.lib()
print("device 0 numa node:", L.tbvh_device_numa_node(0), " process affinity:", len(os.sched_getaffinity(0)), "cpus")
v = np.array([[-10, -10, 5, 0], [10, -10, 5, 0], [0, 10, 5, 0]], np.float32)
e = api.BVH().Build(v)
one = R.make_rays(np.zeros((1, 3), np.float32), np.array([[0, 0, 1]], np.float32))[0]


def run(tag, h):
    bits = np.zeros((n + 31) // 32, np.uint32)
    hits = api.pinned_empty(n, R.HIT_DTYPE)
    for name, fn in (("intersect in place", lambda: e.Intersect(h)), ("intersect packed  ", lambda: e.IntersectPacked(h, hits=hits)), ("occluded          ", lambda: e.IsOccluded(h, bits=bits))):
        fn()
        ts = []
        for _ in range(3):
            R.reset_hits_fast(h)
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        t = min(ts)
        if name.startswith("intersect in place"):
            assert (h["t"][:: 65537] == 5).all(), "host path returned wrong hits"
        print(f"{tag:34s} {name}: {t * 1e3:7.1f} ms {n / t / 1e6:7.0f} Mrays/s  inbound {n * 64 / t / 1e9:5.1f} GB/s", flush=True)
    api.pinned_free(hits)


def fill(h):
    h[:] = one


# 1. buffer allocated by a thread sitting on the OTHER node (what an unbound process may get)
node = L.tbvh_device_numa_node(0)
allcpus = sorted(os.sched_getaffinity(0))
try:
    cpus = [int(c) for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(",") for c in (range(int(part.split("-")[0]), int(part.split("-")[-1]) + 1))]
except Exception:
    cpus = allcpus
other = [c for c in allcpus if c not in cpus] or allcpus
import ctypes as C
os.sched_setaffinity(0, other)
p = C.c_void_p()
from tinybvh_b200.api import check
import torch
x = torch.empty(n * 128, dtype=torch.uint8).pin_memory()       # pinned from the remote node
h_remote = x.numpy().view(R.RAY_DTYPE)
fill(h_remote)
os.sched_setaffinity(0, allcpus)
run("remote-node pinned buffer", h_remote)
del h_remote, x
# 2. NUMA-local (tbvh_host_alloc_near)
h = api.pinned_empty(n, R.RAY_DTYPE, device=0)
api.bind_to_device(0)
fill(h)
run("local pinned buffer", h)
