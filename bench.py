#!/usr/bin/env python
"""bench.py - the hot path on N B200s of one node.

Workload (BASELINE.json configs[2], the configuration the metric "Mrays/s (primary+shadow) on Sponza/Bistro" names for one GPU):
Bistro exterior (2,837,209 triangles), BVH8_CWBVH layout over the SBVH (BVH8_CWBVH::BuildHQ, built and converted on the GPU),
one step = one closest-hit pass over 2048 x 2048 x 16 = 67,108,864 camera rays + one any-hit pass over as many shadow rays.
With --gpus N the ONE ray set is split by ray index over the ranks (strong scaling), the BVH is built on rank 0 and broadcast once.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scene S] [--layout cwbvh|bvh] [--tree hq|sah] [--res R]
                  [--dump-outputs DIR]

Prints ONE JSON line (rank 0).
  value        rays of all ranks / max-over-ranks device time, ray records resident in HBM when the timed region starts
  e2e          the same passes through the C-ABI host-buffer calls (tbvh_intersect + tbvh_occluded on page-locked 128-byte host Ray
               records, hits / occlusion bits back in host memory inside the timed region)
  roofline     the dominant kernel against measured HBM copy bandwidth (+ roofline_l1: the on-chip roof that actually binds,
               roofline_build: the builder)
  parity       the first rays of the timed sets re-traced by the compiled reference (oracle/_ref) outside the timed region
  cpu_baseline the reference's BVH8_CPU (AVX2) on the host cores, bounded sample (N=1 only)
--impl reference times the reference's own CPU path (BVH8_CPU::BuildHQ + Intersect / IsOccluded on all host threads) on the same
workload; rank 0 only, other ranks exit.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

from tinybvh_b200 import rays as R, scenes  # noqa: E402

METRIC = "Mrays/s (primary+shadow)"
ALL_CPUS = sorted(os.sched_getaffinity(0))


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------- workload
def camera_for(scene, verts, k=0):
    if scene == "sponza":
        return R.SPONZA_EYES[k % 3], R.SPONZA_VIEWS[k % 3]
    lo, hi = scenes.scene_bounds(verts)
    return R.bounds_camera(lo, hi, "inside" if scene == "bistro" else "outside")


def light_for(scene, verts):
    if scene == "sponza":
        return np.zeros(3, np.float32)  # tiny_bvh_speedtest.cpp:856
    lo, hi = scenes.scene_bounds(verts)
    return ((lo + hi) * 0.5 + np.array([0, (hi - lo)[1] * 0.45, 0], np.float32)).astype(np.float32)


def shadow_eps(verts):
    lo, hi = scenes.scene_bounds(verts)
    return float((hi - lo).max() * 5e-7)


def data_label(label):
    if label.startswith("synthetic"):
        return "synthetic procedural scene of the same triangle count (fixture not found)"
    if label == "lucy_dragon_x29":
        return "reference fixtures testdata/lucy.bin + xyzrgb_dragon.bin replicated 29x on a grid (10,145,708 triangles), rays generated synthetically"
    files = "+".join(scenes.SCENES[label][0])
    return f"reference fixture testdata/{files} (triangle soup), rays generated synthetically (speedtest camera pattern)"


def config_for(args, label, ntris):
    """The workload, identical for both arms (the driver compares the two `config` objects)."""
    n = args.res * args.res * 16
    return {"workload": f"{label}_{'sbvh' if args.tree == 'hq' else 'sah'}_{args.layout}_{args.res}x{args.res}x16_primary+shadow",
            "scene": label, "scene_tris": int(ntris), "layout": args.layout,
            "tree": "BVH::BuildHQ (SBVH), as tiny_bvh_speedtest.cpp builds for its traversal runs (:894, 960, 1013, 1099, 1197)" if args.tree == "hq" else "BVH::Build (binned SAH)",
            "primary_rays": n, "shadow_rays": n, "rays_per_step": 2 * n,
            "rays": "camera rays of tiny_bvh_speedtest.cpp:497-551 (4x4-pixel tiles, 16 samples per pixel) + one shadow ray per camera ray towards a point light (:853-865)",
            "l2": "no flush: the per-step inputs (2 x %.2f GB of ray records) exceed the 126 MB L2" % (n * 64 / 1e9)}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.lines, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        # median over the samples taken while the GPU was clocked up (the sampler also sees the idle gaps between sections)
        busy = [x for x in sm if mx and x >= 0.6 * mx] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- reference arm / cpu baseline
def cpu_trace(bvh, prim, shadow, passes, threads=0):
    """passes x (closest-hit over `prim`, any-hit over `shadow`) on the host cores; -> (primary s, shadow s) means."""
    bvh.intersect(prim, threads), bvh.occluded(shadow, threads)  # warm-up pass (tiny_bvh_speedtest.cpp:185-215)
    times = []
    for _ in range(passes):
        R.reset_hits_fast(prim)
        t0 = time.perf_counter()
        bvh.intersect(prim, threads)
        t1 = time.perf_counter()
        bvh.occluded(shadow, threads)
        t2 = time.perf_counter()
        times.append((t1 - t0, t2 - t1))
    return float(np.mean([t[0] for t in times])), float(np.mean([t[1] for t in times]))


def cpu_reference(args, verts, prim, shadow, passes, sample, built=None):
    """The reference's own CPU implementation of the path on the host cores: BVH8_CPU::Build(HQ) + Intersect / IsOccluded
    (tiny_bvh.h:7210-7472) from oracle/_ref; the pinned plain-C port of BVH::Intersect when _ref is absent."""
    from oracle import portpy, refpy
    os.sched_setaffinity(0, ALL_CPUS)  # the CPU legs use every host thread, whatever the GPU arm bound itself to
    n, hq = prim.shape[0], args.tree == "hq"
    t0 = time.perf_counter()
    if built is not None:
        kind, cores, bvh = "reference", refpy.hardware_threads(), built[0]
        impl = f"BVH8_CPU::{'BuildHQ' if hq else 'Build'} + Intersect/IsOccluded (AVX2), 10k-ray batches off an atomic counter (tiny_bvh_speedtest.cpp:392-401)"
    elif refpy.available():
        kind, cores = "reference", refpy.hardware_threads()
        bvh = refpy.RefBVH8CPU(verts, hq=hq)
        impl = f"BVH8_CPU::{'BuildHQ' if hq else 'Build'} + Intersect/IsOccluded (AVX2), 10k-ray batches off an atomic counter (tiny_bvh_speedtest.cpp:392-401)"
    else:
        kind, cores = "port", os.cpu_count()
        bvh = portpy.PortBVH(verts)
        impl = "oracle port of BVH::Build + BVH::Intersect/IsOccluded (scalar C, pthreads)"
    build_s = built[1] if built is not None else time.perf_counter() - t0
    tp, ts = cpu_trace(bvh, prim, shadow, passes)
    return {"value": 2 * n / (tp + ts) / 1e6, "unit": "Mrays/s", "cores": int(cores), "kind": kind, "sample": sample,
            "impl": impl, "primary_mrays": n / tp / 1e6, "shadow_mrays": n / ts / 1e6, "build_s": build_s,
            "build_mtris": verts.shape[0] / 3 / build_s / 1e6, "ms_per_step": (tp + ts) * 1e3}


def host_ray_sets(args, verts, count, tracer=None):
    """The first `count` camera rays of the workload and their shadow rays, on the host (pageable).  The camera rays are traced by
    `tracer` (an object with .intersect) to find the shadow-ray origins; default: the reference's BVH::Build + Intersect."""
    from oracle import portpy, refpy
    eye, view = camera_for(args.scene, verts)
    prim = np.empty(count, R.RAY_DTYPE)
    R.primary_rays_into(prim, eye, view, args.res, args.res, 16)
    if tracer is None:
        tracer = refpy.RefBVH(verts, mode=0, threaded=True) if refpy.available() else portpy.PortBVH(verts)
    tracer.intersect(prim, 0)
    sh = np.empty(count, R.RAY_DTYPE)
    R.shadow_rays_into(sh, prim, light_for(args.scene, verts), shadow_eps(verts))
    R.reset_hits_fast(prim)
    return prim, sh


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import refpy
    verts, label = scenes.load_scene(args.scene)
    ntris = verts.shape[0] // 3
    n = args.res * args.res * 16
    R.set_generator_threads(len(ALL_CPUS))
    # the whole workload, traced by the CPU implementation itself (its own closest hits place the shadow rays, as the speedtest does)
    t0 = time.time()
    hq = args.tree == "hq"
    os.sched_setaffinity(0, ALL_CPUS)
    tb = time.perf_counter()
    bvh = refpy.RefBVH8CPU(verts, hq=hq) if refpy.available() else None
    built = (bvh, time.perf_counter() - tb) if bvh is not None else None
    prim, sh = host_ray_sets(args, verts, n, tracer=bvh)
    log(f"[bench reference] {label}: {n} camera + {n} shadow rays on the host in {time.time() - t0:.1f}s")
    cb = cpu_reference(args, verts, prim, sh, passes=max(1, args.steps), built=built,
                       sample=f"the whole workload: {n} camera + {n} shadow rays per step, {max(1, args.steps)} timed passes after 1 warm-up, all host threads")
    out = {"metric": METRIC, "value": cb["value"], "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
           "data": data_label(label), "impl": "reference", "config": config_for(args, label, ntris),
           "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "impl", "primary_mrays", "shadow_mrays", "build_mtris")},
           "e2e": {"value": cb["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------- parity sample (outside every timed region)
def parity_sample(args, verts, h_prim, h_shadow, hits, bits, m):
    """Re-trace the first m rays of the timed sets with the compiled reference and compare with what the engine produced for them.
    (a) the reference's own walk of the same layout over its own build chain - bit-identical t, u, v, prim expected;
    (b) the parity oracle BVH::Build + BVH::Intersect / IsOccluded (a different tree): prim mismatches classified by the tie audit
        of SURVEY 8(c) - tie-equivalent (the engine's primitive re-evaluated with the oracle's Moeller-Trumbore gives the bit-identical
        t) or real."""
    from oracle import refpy
    from tests import util
    if not refpy.available():
        return {"unavailable": "oracle/_ref not built"}
    os.sched_setaffinity(0, ALL_CPUS)
    t0 = time.time()
    # m rays spread evenly over this rank's index range (the first rays alone would be one corner of the image)
    n = h_prim.shape[0]
    idx = np.unique(np.linspace(0, n - 1, m).astype(np.int64))
    m = idx.shape[0]
    sel_prim, sel_shadow = h_prim[idx], h_shadow[idx]
    got = sel_prim.copy()
    got["t"], got["u"], got["v"], got["prim"] = hits[idx, 0], hits[idx, 1], hits[idx, 2], hits[idx, 3].view(np.uint32)
    occ = ((bits[idx >> 5] >> (idx & 31).astype(np.uint32)) & 1).astype(bool)
    out = {"sample_rays": int(m), "sampling": "every (n/m)-th ray of the timed camera and shadow sets"}
    mode = 1 if args.tree == "hq" else 2   # refpy: 1 = BuildHQ chain, 2 = BVH::Build chain
    want = sel_prim.copy()
    R.reset_hits_fast(want)
    if args.layout == "cwbvh":
        ref = refpy.RefCWBVH(verts, mode=mode)
        ref.intersect(want, 0)
        name = "BVH8_CWBVH::BuildHQ + BVH8_CWBVH::Intersect" if mode == 1 else "BVH8_CWBVH::Build + Intersect"
        sh = sel_shadow.copy()
        d = sh["t"].copy()
        ref.intersect(sh, 0)
        occ_ref = sh["t"] < d          # BVH8_CWBVH::IsOccluded is the FALLBACK_SHADOW_QUERY (tiny_bvh.h:312): Intersect, then t < d
    else:
        ref = refpy.RefBVH(verts, mode=2 if args.tree == "hq" else 0, threaded=True)
        ref.intersect(want, 0)
        name = "BVH::BuildHQ + BVH::Intersect" if args.tree == "hq" else "BVH::Build + BVH::Intersect"
        occ_ref = np.unpackbits(ref.occluded(sel_shadow.copy(), 0).view(np.uint8), bitorder="little")[:m].astype(bool)
    c = util.compare_hits(got, want)
    hit = want["t"] < 1e30
    # THE parity claim: the reference's own CPU walk of the same layout over the same (reference-built) tree
    out["vs_reference"] = {"reference": name, "prim_mismatch": c["prim"], "t_bit_mismatch": c["t"],
                           "uv_bit_mismatch_on_hits": int(((got["u"].view(np.uint32) != want["u"].view(np.uint32)) | (got["v"].view(np.uint32) != want["v"].view(np.uint32)))[hit].sum()),
                           "occlusion_bit_mismatch": int((occ != occ_ref).sum())}
    # Cross-tree audit (SURVEY 8c): BVH::Build + BVH::Intersect walks ANOTHER tree.  The reference's own layouts disagree with each
    # other there on a few rays (exact-t ties between coincident triangles; rays for which its SBVH walk finds another surface, SURVEY
    # 8(c) table) - reported as the reference's self-disagreement next to the engine's, which must be the same set of rays.
    o = refpy.RefBVH(verts, mode=0, threaded=True)
    w2 = sel_prim.copy()
    R.reset_hits_fast(w2)
    o.intersect(w2, 0)
    ref_dis = (want["prim"] != w2["prim"]) | (want["t"].view(np.uint32) != w2["t"].view(np.uint32))
    eng_dis = (got["prim"] != w2["prim"]) | (got["t"].view(np.uint32) != w2["t"].view(np.uint32))
    cls = util.classify_mismatches(got, w2, verts)
    occ_o = np.unpackbits(o.occluded(sel_shadow.copy(), 0).view(np.uint8), bitorder="little")[:m].astype(bool)
    out["cross_tree_audit"] = {"other_walk": "BVH::Build + BVH::Intersect / IsOccluded (the scalar reference builder's tree)",
                               "reference_layout_disagrees_with_it_on": int(ref_dis.sum()), "engine_disagrees_with_it_on": int(eng_dis.sum()),
                               "same_rays": bool(np.array_equal(ref_dis, eng_dis)),
                               "of_which_exact_t_ties": cls["tie_equivalent"], "of_which_other_surface_found_by_the_reference_too": cls["real"],
                               "occlusion_bits_reference_layout_vs_it": int((occ_ref != occ_o).sum()), "occlusion_bits_engine_vs_it": int((occ != occ_o).sum())}
    out["seconds"] = round(time.time() - t0, 1)
    return out


# ---------------------------------------------------------------------------------------------- --dump-outputs
DUMP_RAYS, DUMP_SEED = 1 << 20, 20240917


def dump_outputs(out_dir, hits, bits, blocks, n_total, rank, world):
    """What the timed step handed back - the closest hit of every camera ray (t, u, v, prim) and the occlusion bit of every shadow
    ray - for a fixed, seeded sample of DUMP_RAYS rays of the whole set (32 bytes a ray: 32 MB), one .npy per field, so that two
    builds of the project can be compared output for output.  With --gpus N every rank writes its own rays (file suffix .rank<r>)."""
    m = min(n_total, DUMP_RAYS)
    pick = np.arange(n_total) if m == n_total else np.sort(np.random.default_rng(DUMP_SEED).choice(n_total, m, replace=False))
    gidx, lidx, off = [np.zeros(0, np.int64)], [np.zeros(0, np.int64)], 0
    for b0, bc in blocks:
        lo, hi = np.searchsorted(pick, [b0, b0 + bc])
        gidx.append(pick[lo:hi])
        lidx.append(pick[lo:hi] - b0 + off)
        off += bc
    g, l = np.concatenate(gidx), np.concatenate(lidx)
    arrays = {"ray_index": g.astype(np.float64), "hit_t": hits[l, 0], "hit_u": hits[l, 1], "hit_v": hits[l, 2],
              "hit_prim": hits[l, 3].view(np.uint32).astype(np.float64),
              "occluded": ((bits[l >> 5] >> (l & 31).astype(np.uint32)) & 1).astype(np.float32)}
    os.makedirs(out_dir, exist_ok=True)
    sfx = f".rank{rank}" if world > 1 else ""
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{sfx}.npy"), np.ascontiguousarray(a))


# ---------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    from tinybvh_b200 import api, _lib
    import ctypes as C
    # sit on the CPUs of this GPU's NUMA node before anything allocates: page-locked ray buffers, OpenMP ray generation and the host
    # pipeline's threads then work out of local memory (2 sockets: GPUs 0-3 / 4-7 hang off different nodes)
    bound = api.bind_to_device(local)
    R.set_generator_threads(max(1, len(os.sched_getaffinity(0)) // max(1, min(world, 4))))  # the ranks of one socket share its cores
    import torch
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    L = _lib.lib()
    verts, label = scenes.load_scene(args.scene)
    ntris = verts.shape[0] // 3
    t_setup = time.time()

    # ---- build on rank 0 (timed: build Mtris/s), then ONE broadcast of the BVH over NVLink (SURVEY 8e)
    bvh = api.BVH(device=local)
    build = {}
    if rank == 0:
        # every builder of the path is timed on its second call (the first pays allocations and first-launch costs)
        for name, fn in (("Build", "Build"), ("BuildHQ", "BuildHQ")):
            b = api.BVH(device=local)
            getattr(b, fn)(verts)
            b = api.BVH(device=local)
            getattr(b, fn)(verts)
            i = b.info()
            build[name] = {"ms": i.build_ms, "mtris_per_s": ntris / i.build_ms / 1e3, "nodes": i.used_nodes, "idx_count": i.idx_count, "depth": i.max_depth}
            if (name == "BuildHQ") == (args.tree == "hq"):
                bvh = b
            del b
    bcast_ms, bcast_bytes = None, None
    if world > 1:
        from tinybvh_b200 import multi
        arrays = None
        if rank == 0:
            i = bvh.info()
            d_nodes = torch.empty(i.used_nodes * 8, dtype=torch.int32, device=dev)
            d_idx = torch.empty(i.idx_count, dtype=torch.int32, device=dev)
            api.check(L.tbvh_download_bvh(bvh.h, C.c_void_p(d_nodes.data_ptr()), C.c_void_p(d_idx.data_ptr()), api.DEVICE))
            arrays = {"nodes": d_nodes, "prim_idx": d_idx, "verts": torch.from_numpy(verts.reshape(-1)).to(dev)}
            bcast_bytes = int(sum(a.numel() * a.element_size() for a in arrays.values()))
        warm = torch.zeros(1 << 20, dtype=torch.float32, device=dev)   # communicator set-up is not the broadcast
        for _ in range(3):
            dist.all_reduce(warm)
            dist.broadcast(warm, 0)
        # the receivers' first allocation of the arrays (cudaMalloc of ~250 MB) is not the broadcast either: let the caching allocator take
        # that memory now, so the timed region below holds the NCCL transfers (and their small metadata round) only
        sz = torch.tensor([bcast_bytes or 0], dtype=torch.int64, device=dev)
        dist.broadcast(sz, 0)
        scratch = torch.empty(int(sz.item()) + (8 << 20), dtype=torch.uint8, device=dev)
        del scratch
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        got = multi.broadcast_arrays(arrays, 0, dev)   # the ONE exchange step: the built BVH to every GPU over NVLink
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        bcast_ms = float(t.item())
        if rank != 0:
            api.check(L.tbvh_upload_bvh(bvh.h, C.c_void_p(got["nodes"].data_ptr()), got["nodes"].numel() // 8, C.c_void_p(got["prim_idx"].data_ptr()),
                                        got["prim_idx"].numel(), C.c_void_p(got["verts"].data_ptr()), 16, ntris, api.DEVICE))
        del got, arrays
    # derived layout: BVH8_CWBVH::ConvertFrom's chain on every GPU's replica (deterministic; byte-identical to the reference's)
    convert_ms = None
    if args.layout == "cwbvh":
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        api.check(L.tbvh_convert(bvh.h, api.LAYOUT_CWBVH))
        convert_ms = (time.perf_counter() - t0) * 1e3
        bvh.layout = api.LAYOUT_CWBVH
    eng = bvh
    info = bvh.info()

    # ---- this rank's index range of the ONE ray set (strong scaling)
    n_total = args.res * args.res * 16
    # Sharding by ray index, block-cyclic: the set is cut into blocks of 2^20 consecutive rays (4x4-pixel tiles stay together, warps stay
    # coherent) and block b belongs to rank b % world - a rank's rays come from all over the image, so no rank owns "the expensive
    # corner" (contiguous eighths of the Bistro view differ by 30 % in traversal work).  Every rank generates its own blocks.
    from tinybvh_b200 import multi as M
    blocks = M.block_cyclic(n_total, rank, world)
    n = sum(c for _, c in blocks)
    first = blocks[0][0] if blocks else 0
    eye, view = camera_for(args.scene, verts)
    # TBVH_BENCH_NUMA_SPREAD=1 (experiment): every second rank keeps its ray buffers on the OTHER socket's memory
    spread = os.environ.get("TBVH_BENCH_NUMA_SPREAD") == "1" and (local & 1) == 1
    buf_node = (1 - max(0, L.tbvh_device_numa_node(local))) if spread else None
    palloc = (lambda cnt, dt: api.pinned_empty(cnt, dt, node=buf_node)) if spread else (lambda cnt, dt: api.pinned_empty(cnt, dt, device=local))
    h_prim = palloc(n, R.RAY_DTYPE)
    off = 0
    for b0, bc in blocks:
        R.primary_rays_into(h_prim[off:off + bc], eye, view, args.res, args.res, 16, first=b0)
        off += bc
    d_prim = torch.empty((n, 64), dtype=torch.uint8, device=dev)
    api.copy_rays_to_device(h_prim, d_prim)
    d_hits = torch.empty((n, 4), dtype=torch.float32, device=dev)
    eng.Intersect(d_prim, hits=d_hits)
    torch.cuda.synchronize()
    hits = d_hits.cpu().numpy()
    h_shadow = palloc(n, R.RAY_DTYPE)
    R.shadow_rays_into(h_shadow, h_prim, light_for(args.scene, verts), shadow_eps(verts), hits=hits)
    d_shadow = torch.empty((n, 64), dtype=torch.uint8, device=dev)
    api.copy_rays_to_device(h_shadow, d_shadow)
    d_bits = torch.empty((n + 31) // 32, dtype=torch.int32, device=dev)
    h_bits = np.zeros((n + 31) // 32, np.uint32)
    if rank == 0:
        log(f"[bench] {label}: {ntris} tris, {info.used_nodes} nodes, depth {info.max_depth}, builds {build}; {n} of {n_total} camera + shadow rays in {len(blocks)} block(s) from ray {first}; "
            f"numa-bound {bound}; setup {time.time() - t_setup:.1f}s")

    # traversal work per ray (kernel counters, one untimed pass each)
    eng.set_stats(True)
    eng.Intersect(d_prim, hits=d_hits)
    st_prim = eng.get_stats()
    eng.IsOccluded(d_shadow, bits=d_bits)
    st_shad = eng.get_stats()
    eng.set_stats(False)

    stream = torch.cuda.current_stream(dev)

    def step(ev=None):
        if ev is not None:
            ev[0].record(stream)
        eng.Intersect(d_prim, hits=d_hits)
        if ev is not None:
            ev[1].record(stream)
        eng.IsOccluded(d_shadow, bits=d_bits)
        if ev is not None:
            ev[2].record(stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    W = max(3, args.warmup)
    for _ in range(W):
        step()
    barrier()
    clocks = ClockSampler(local) if rank == 0 else None
    launches0 = api.launch_count()
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_begin.record(stream)
    for k in range(args.steps):
        step(evs[k])
    t_end.record(stream)
    barrier()
    launches = api.launch_count() - launches0
    total_ms = t_begin.elapsed_time(t_end)
    prim_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in evs]))
    shad_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in evs]))
    torch.cuda.synchronize()
    bits_dev = d_bits.cpu().numpy().view(np.uint32)
    hits = d_hits.cpu().numpy()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, hits, bits_dev, blocks, n_total, rank, world)

    # ---- extra (SURVEY 8(d) config 4): incoherent rays - one diffuse bounce off every camera hit (tiny_bvh_speedtest.cpp:564-587 with a
    # per-ray xorshift seeded by the global ray index), same index shard, device resident; reported beside the headline, not in it
    incoherent = None
    if not args.no_extra:
        h_diff = h_shadow  # the shadow records are regenerated from h_prim + hits on demand; reuse the buffer for the bounce rays
        off = 0
        for b0, bc in blocks:
            R.diffuse_rays_into(h_diff[off:off + bc], h_prim[off:off + bc], verts, hits=hits[off:off + bc], first=b0)
            off += bc
        d_diff = torch.empty((n, 64), dtype=torch.uint8, device=dev)
        api.copy_rays_to_device(h_diff, d_diff)
        d_hits2 = torch.empty((n, 4), dtype=torch.float32, device=dev)
        eng.set_stats(True)
        eng.Intersect(d_diff, hits=d_hits2)
        st_diff = eng.get_stats()
        eng.set_stats(False)
        eng.Intersect(d_diff, hits=d_hits2)
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(stream)
        for _ in range(3):
            eng.Intersect(d_diff, hits=d_hits2)
        a1.record(stream)
        barrier()
        incoherent = {"ms": a0.elapsed_time(a1) / 3, "node_visits": st_diff[0] / n, "triangle_tests": st_diff[1] / n}
        del d_diff, d_hits2
        R.shadow_rays_into(h_shadow, h_prim, light_for(args.scene, verts), shadow_eps(verts), hits=hits)  # restore for the e2e passes

    # ---- e2e: the reference-facing C-ABI calls on HOST buffers (page-locked), copies inside the timed region
    def e2e_pass(packed_out=None):
        if packed_out is None:
            eng.Intersect(h_prim)
        else:
            eng.IntersectPacked(h_prim, hits=packed_out)
        eng.IsOccluded(h_shadow, bits=h_bits)

    for _ in range(2):
        e2e_pass()
    barrier()
    te0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_pass()
    te1 = time.perf_counter()
    e2e_ms = (te1 - te0) * 1e3
    e2e_ok = bool(np.array_equal(h_prim["t"].view(np.uint32), hits[:, 0].view(np.uint32)) and np.array_equal(h_prim["prim"], hits[:, 3].view(np.uint32))
                  and np.array_equal(h_bits, bits_dev))
    R.reset_hits_fast(h_prim)
    # the same with the packed-hits entry point (tbvh_intersect_packed): the return trip is one contiguous copy per chunk
    h_hits = palloc(n, R.HIT_DTYPE)
    e2e_pass(h_hits)
    barrier()
    tp0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_pass(h_hits)
    tp1 = time.perf_counter()
    e2e_packed_ms = (tp1 - tp0) * 1e3
    clk = clocks.stop() if clocks else None

    t = torch.tensor([total_ms, e2e_ms, prim_ms, shad_ms, e2e_packed_ms, incoherent["ms"] if incoherent else 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms, prim_ms, shad_ms, e2e_packed_ms, inc_ms = [float(x) for x in t.cpu()]
    ok = torch.tensor([1.0 if e2e_ok else 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    e2e_ok = bool(ok.item() > 0.5)

    if rank == 0:
        rays_per_step = 2 * n_total
        ms_per_step = total_ms / args.steps
        value = rays_per_step / ms_per_step / 1e3
        peak, which = peaks()
        if args.layout == "cwbvh":
            bvh_bytes = (info.used_blocks // 5) * 160 + info.cwbvh_tri_count * 48
            kernel = "k_trace_wide<closest>"
            layout_note = "traversal nodes 160 B (derived from the 80-byte bvh8Data nodes) + 48-byte bvh8Tris records"
        else:
            bvh_bytes = info.used_nodes * 32 + info.idx_count * 48
            kernel = "k_trace_bvh2<closest>"
            layout_note = "32-byte Wald nodes (sibling pairs) + 48-byte leaf-ordered triangle records"
        # SURVEY 8(d): 64 B ray record read + 16 B hit written per ray, plus one pass over the BVH per launch; this rank's launch
        alg_bytes = n * 80 + bvh_bytes
        achieved = alg_bytes / (prim_ms * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(REPO, "profiles", "traffic.json")
        if os.path.isfile(tp):
            try:
                traffic = json.load(open(tp)).get(f"{kernel}_{label}_{args.tree}_{args.res}")
            except Exception:
                traffic = None
        # the roof that binds: bytes moved from L1 into registers.  Per node visit 32 B of header + 32 B per child pair (CWBVH) or
        # one 64 B sibling pair (BVH2); per triangle test 48 B; per ray 64 B in.  L1 delivers 128 B / clk / SM.
        visits, tris, pairs = st_prim[0] / n, st_prim[1] / n, (st_prim[2] / n if len(st_prim) > 2 else 0.0)
        l1_bytes_ray = (visits * 32 + pairs * 32 if args.layout == "cwbvh" else visits * 64) + tris * 48 + 64
        sm_count, sm_mhz = torch.cuda.get_device_properties(dev).multi_processor_count, (clk or {}).get("sm_mhz") or 1965.0
        l1_peak = sm_count * 128 * sm_mhz * 1e6 / 1e9
        l1_ach = l1_bytes_ray * n / (prim_ms * 1e-3) / 1e9
        out = {
            "metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": data_label(label), "config": config_for(args, label, ntris),
            "parallelism": (f"ONE ray set sharded by ray index over {world} GPUs (blocks of 2^20 consecutive rays dealt round-robin), BVH built on rank 0 and broadcast once "
                            f"(NCCL over NVLink), no collective during traversal") if world > 1 else "1 GPU",
            "primary_mrays": n_total / prim_ms / 1e3, "shadow_mrays": n_total / shad_ms / 1e3,
            "work_per_ray": {"primary": {"node_visits": visits, "triangle_tests": tris, "pair_steps": pairs},
                             "shadow": {"node_visits": st_shad[0] / n, "triangle_tests": st_shad[1] / n}},
            "build": {"Build": build.get("Build"), "BuildHQ": build.get("BuildHQ"), "cwbvh_convert_ms_wall": convert_ms, "bcast_ms": bcast_ms, "bcast_bytes": bcast_bytes,
                      "bvh_bytes_traversed": bvh_bytes, "built_on": "GPU (tbvh_build_flavour + tbvh_convert)"},
            "roofline": {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "peak_source": which, "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": prim_ms, "layout": layout_note,
                         "note": "traversal is bound on chip (issue slots / L1), not by HBM: see roofline_l1"},
            "roofline_l1": {"bound": "l1-to-register bytes", "kernel": kernel, "achieved": l1_ach, "peak": l1_peak, "unit": "GB/s", "frac": l1_ach / l1_peak,
                            "bytes_per_ray": l1_bytes_ray, "peak_source": f"{sm_count} SMs x 128 B/clk x {sm_mhz:.0f} MHz"},
            "e2e": {"value": rays_per_step / (e2e_ms / args.steps) / 1e3, "unit": "Mrays/s", "h2d_bytes_per_step": 2 * n_total * 64,
                    "d2h_bytes_per_step": n_total * 16 + ((n_total + 31) // 32) * 4, "ms_per_step": e2e_ms / args.steps,
                    "api": "tbvh_intersect + tbvh_occluded on page-locked 128-byte host Ray records (hits written in place into Ray.hit)",
                    "results_identical_to_device_path": e2e_ok,
                    "packed_hits_value": rays_per_step / (e2e_packed_ms / args.steps) / 1e3,
                    "packed_hits_api": "tbvh_intersect_packed + tbvh_occluded: same inputs, hits returned as a packed 16-byte array",
                    "numa_bound": bool(bound)},
            "gpu_launches": int(launches),
            "clocks": clk,
        }
        if incoherent:
            out["incoherent"] = {"rays": n_total, "mrays": n_total / inc_ms / 1e3, "ms": inc_ms, "node_visits_per_ray": incoherent["node_visits"], "triangle_tests_per_ray": incoherent["triangle_tests"],
                                 "what": "closest hit of one diffuse bounce ray per camera hit (SURVEY 8(d) config 4 generator), same layout, device resident, sharded like the headline set"}
        if build.get("Build"):
            # SURVEY 8(d): reference-algorithm bytes of a binned-SAH build = 48 + 36 + L (2 x 36 + 4) + 64 per triangle, L = mean leaf depth
            L_mean = {"sponza": 19.9, "bistro": 23.2}.get(label, 18.0)
            per_tri = 48 + 36 + L_mean * 76 + 64
            ach = per_tri * ntris / (build["Build"]["ms"] * 1e-3) / 1e9
            out["roofline_build"] = {"bound": "hbm", "kernel": "tbvh_build (binned SAH, all launches of one build)", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                                     "bytes_per_tri": per_tri, "mtris_per_s": build["Build"]["mtris_per_s"], "traffic": None,
                                     "note": "reference-algorithm bytes (SURVEY 8d); the GPU builder keeps small subtrees on chip and moves fewer"}
        if not args.no_parity:
            out["parity"] = parity_sample(args, verts, h_prim, h_shadow, hits, bits_dev, min(n, args.parity_rays))
        if world == 1 and not args.no_cpu_baseline:
            t0 = time.time()
            m = min(n, args.cpu_sample_rays)
            p2, s2 = h_prim[:m].copy(), h_shadow[:m].copy()
            R.reset_hits_fast(p2)
            cb = cpu_reference(args, verts, p2, s2, passes=3, sample=f"the first {m} camera + {m} shadow rays of the workload, 3 timed passes after 1 warm-up, all host threads")
            out["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "impl", "primary_mrays", "shadow_mrays", "build_mtris")}
            log(f"[bench] cpu baseline took {time.time() - t0:.1f}s")
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scene", default="bistro")
    ap.add_argument("--layout", default="cwbvh", choices=["bvh", "cwbvh"])
    ap.add_argument("--tree", default="hq", choices=["hq", "sah"],
                    help="hq: BVH::BuildHQ (SBVH), the tree every traversal benchmark of tiny_bvh_speedtest.cpp builds (:894, 960, 1013, 1099, 1197); sah: BVH::Build")
    ap.add_argument("--res", type=int, default=2048, help="camera rays = res*res*16 (2048 -> 67,108,864)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the incoherent-ray section")
    ap.add_argument("--parity-rays", type=int, default=1 << 20)
    ap.add_argument("--cpu-sample-rays", type=int, default=1 << 23)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's hits and occlusion bits for a seeded "
                    "sample of rays to DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the engine's timed path returned: it needs --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
