"""CPU: the workload definitions bench.py measures (BASELINE.json configs) and the host logic of the N > 1 arm that needs no
GPU: cfg4's fixed 312-scene list, its LPT partition over the ranks (every scene exactly once, balanced), per-rank scene seeds."""
import os
import sys

import numpy as np

from conftest import ROOT

sys.path.insert(0, ROOT)
import bench  # noqa: E402
from lib.model.scene_shard import shard_scenes  # noqa: E402


def test_default_workload_is_baseline_cfg2():
    wl = bench.workload("cfg2", 0, 1)
    assert wl["metric"] == "scenes_per_sec_96x48x96_5img" and wl["scaling"] == "weak" and wl["math_default"] == "exact"
    assert all(d == (96, 48, 96) and n == 5 for _, d, n in wl["scenes"])
    # 24 distinct chunks of 6.9 MB each rotate: more than the 126 MB L2
    per = 2 * 96 * 48 * 96 * 4 + 5 * (128 * 32 * 41 + 32 * 41 + 16) * 4
    assert len(wl["scenes"]) * per > 126e6
    assert bench.alg_bytes((96, 48, 96)) == 806.8e6  # SURVEY 8(d)
    # ranks draw disjoint seeds
    assert not {s for s, _, _ in wl["scenes"]} & {s for s, _, _ in bench.workload("cfg2", 1, 2)["scenes"]}


def test_cfg4_list_and_lpt_partition():
    wl = bench.workload("cfg4", 0, 8)
    assert len(wl["scene_list"]) == 312 and wl["scaling"] == "strong"
    assert wl == bench.workload("cfg4", 3, 8) or wl["scene_list"] == bench.workload("cfg4", 3, 8)["scene_list"]  # same list on every rank
    costs = [float(np.prod(wl["scenes"][k][1])) * (1 + wl["scenes"][k][2] / 40.0) for k in wl["scene_list"]]
    for world in (1, 2, 4, 8):
        parts = [shard_scenes(costs, r, world) for r in range(world)]
        assert sorted(i for p in parts for i in p) == list(range(312))
        loads = [sum(costs[i] for i in p) for p in parts]
        assert max(loads) / (sum(loads) / world) < 1.03  # LPT: within 3 % of perfect balance
    shapes = {wl["scenes"][k][1] for k in wl["scene_list"]}
    assert (88, 44, 88) in shapes and (208, 48, 160) in shapes and len(shapes) == 8


def test_other_configs_named_by_baseline():
    assert bench.workload("cfg3", 0, 1)["scenes"][0][1:] == ((208, 48, 160), 40)
    assert bench.workload("cfg3s", 0, 1)["scenes"][0][1:] == ((88, 44, 88), 40)
    c5 = bench.workload("cfg5", 0, 8)
    assert c5["cfgname"] == "suncg" and c5["math_default"] == "fp16" and c5["scenes"][0][2] == 3
    assert abs(bench.alg_bytes((96, 48, 96), "suncg") - 729.3e6) < 1


def test_dump_outputs_types_order_and_budget(tmp_path, monkeypatch):
    """--dump-outputs: float32 / float64 files in loop order; above the byte budget the mask voxels become a seeded sample."""
    rng = np.random.default_rng(0)
    scenes = []
    for n, sizes in ((3, [(2, 3, 4), (1, 1, 5)]), (2, None), (4, [(6, 2, 2)])):
        det = rng.standard_normal((n, 16)).astype(np.float32)
        if sizes is None:
            scenes.append((det, None, None))
        else:
            sz = np.array(sizes, dtype=np.int32)
            scenes.append((det, (rng.random(int(np.prod(sz, axis=1).sum())) > 0.5).astype(np.uint8), sz))
    bench.dump_outputs(str(tmp_path / "all"), scenes)
    got = {f[:-4]: np.load(tmp_path / "all" / f) for f in os.listdir(tmp_path / "all")}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values()) and "mask_voxel_index" not in got
    assert np.array_equal(got["detections"], np.concatenate([d for d, _, _ in scenes]))
    assert got["detections_per_scene"].tolist() == [3, 2, 4] and got["masks_per_scene"].tolist() == [2, 0, 1]
    bits = np.concatenate([scenes[0][1], scenes[2][1]])
    assert np.array_equal(got["mask_voxels"], bits) and got["mask_sizes"].tolist() == [[2, 3, 4], [1, 1, 5], [6, 2, 2]]
    budget = sum(a.nbytes for k, a in got.items() if k != "mask_voxels") + 1024 * 6 + 4 * 30
    monkeypatch.setattr(bench, "DUMP_BYTES", budget)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), scenes)
    idx, vals = np.load(tmp_path / "a" / "mask_voxel_index.npy"), np.load(tmp_path / "a" / "mask_voxels.npy")
    assert len(idx) == 10 and np.array_equal(vals, bits[idx.astype(np.int64)])
    assert np.array_equal(idx, np.load(tmp_path / "b" / "mask_voxel_index.npy"))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= budget
