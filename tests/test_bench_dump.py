"""bench.py --dump-outputs on the host: the seeded ray sample, its mapping from the global ray index to a rank's block-cyclic share,
the field values, the dtypes and the 64 MB bound."""
import glob
import os

import numpy as np

import bench
from tinybvh_b200 import multi


def fake_outputs(idx):
    """Per-ray values recoverable from the global index: hits (t, u, v, prim bits) and an occlusion bit."""
    hits = np.stack([idx.astype(np.float32), idx.astype(np.float32) + 0.5, -idx.astype(np.float32), idx.astype(np.uint32).view(np.float32)], 1)
    return hits, (idx % 3 == 0)


def pack(occ):
    bits = np.zeros((occ.shape[0] + 31) // 32, np.uint32)
    np.bitwise_or.at(bits, np.nonzero(occ)[0] >> 5, np.uint32(1) << (np.nonzero(occ)[0] & 31).astype(np.uint32))
    return bits


def load(d, world):
    files = {}
    for f in sorted(glob.glob(os.path.join(d, "*.npy"))):
        name = os.path.basename(f).split(".")[0]
        files.setdefault(name, []).append(np.load(f))
    assert len(files) == 6 and all(len(v) == world for v in files.values())
    assert all(a.dtype in (np.float32, np.float64) for v in files.values() for a in v)
    cat = {k: np.concatenate(v) for k, v in files.items()}
    order = np.argsort(cat["ray_index"])
    return {k: v[order] for k, v in cat.items()}


def test_dump_outputs_is_a_fixed_sample_of_the_whole_set(tmp_path):
    n_total = (3 << 20) + 77
    got = {}
    for world in (1, 3):
        d = str(tmp_path / f"w{world}")
        for rank in range(world):
            blocks = multi.block_cyclic(n_total, rank, world)
            idx = np.concatenate([np.arange(b0, b0 + bc) for b0, bc in blocks])
            hits, occ = fake_outputs(idx)
            bench.dump_outputs(d, hits, pack(occ), blocks, n_total, rank, world)
        assert sum(os.path.getsize(f) for f in glob.glob(os.path.join(d, "*.npy"))) <= 64 << 20
        got[world] = load(d, world)
    one = got[1]
    g = one["ray_index"].astype(np.int64)
    assert g.shape[0] == bench.DUMP_RAYS and np.unique(g).shape[0] == g.shape[0] and g.max() < n_total
    hits, occ = fake_outputs(g)
    assert np.array_equal(one["hit_t"], hits[:, 0]) and np.array_equal(one["hit_u"], hits[:, 1]) and np.array_equal(one["hit_v"], hits[:, 2])
    assert np.array_equal(one["hit_prim"], g.astype(np.float64))
    assert np.array_equal(one["occluded"], occ.astype(np.float32))
    for k in one:
        assert np.array_equal(got[3][k], one[k]), k


def test_dump_outputs_takes_every_ray_of_a_small_set(tmp_path):
    n = 1000
    idx = np.arange(n)
    hits, occ = fake_outputs(idx)
    bench.dump_outputs(str(tmp_path), hits, pack(occ), multi.block_cyclic(n, 0, 1), n, 0, 1)
    out = load(str(tmp_path), 1)
    assert np.array_equal(out["ray_index"], idx.astype(np.float64)) and np.array_equal(out["occluded"], occ.astype(np.float32))
