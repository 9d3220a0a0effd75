"""CPU: the arithmetic bench.py reports against -- algorithmic FLOPs per image (SURVEY.md App. A.1), the source hash that gates
the committed ncu traffic figure, and the committed profile artefacts being parseable bench lines of the right configurations."""
import glob
import json
import os

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_algorithmic_work_matches_the_survey_tables():
    a = bench.work_per_image(600, 900)                       # cfgA: 37 x 56 feature map
    assert (a["fh"], a["fw"], a["cells"]) == (37, 56, 2072)
    assert abs(a["conv1_1"] / 1e9 - 1.866) < 1e-3
    assert abs((a["conv1_1"] + a["conv3x3"]) / 1e9 - 339.130) < 5e-3
    assert abs(a["xproj"] / 1e9 - 2.173) < 1e-3 and abs(a["recurrent"] / 1e9 - 0.543) < 1e-3 and abs(a["fc"] / 1e9 - 0.543) < 1e-3
    b = bench.work_per_image(1200, 1600)                     # cfgB: 75 x 100
    assert (b["fh"], b["fw"]) == (75, 100)
    assert abs((b["conv1_1"] + b["conv3x3"]) / 1e9 - 1209.876) < 2e-2
    c = bench.work_per_image(900, 600)                       # the transposed shape of config 5
    assert (c["fh"], c["fw"]) == (56, 37)


def test_configs_follow_baseline_json():
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert len(base["configs"]) == 5
    assert bench.CONFIGS[2]["batch"] == 32 and bench.CONFIGS[2]["shapes"] == [(600, 900)] and bench.CONFIGS[2]["detect"] == "H"
    assert bench.CONFIGS[3]["mode"] == "bf16" and "bf16" in base["configs"][2]
    assert bench.CONFIGS[4]["batch"] == 64 and bench.CONFIGS[4]["shapes"] == [(1200, 1600)] and "1200" in base["configs"][3]
    assert bench.CONFIGS[5]["detect"] == "O" and len(bench.CONFIGS[5]["shapes"]) == 2 and "oriented" in base["configs"][4]
    assert bench.MODES[bench.FP32_MODE]["units"] in (2.0, 3.0)          # a float32-faithful mode, never plain bf16


def test_traffic_files_are_stamped_with_a_source_hash():
    sha = bench.sources_sha256()
    assert len(sha) == 64 and sha == bench.sources_sha256()
    files = glob.glob(os.path.join(ROOT, "profiles", "r2_conv_traffic_cfg*_*.json"))
    assert files
    for f in files:
        t = json.load(open(f))
        assert t["launches"] == 13 and len(t["sources_sha256"]) == 64 and t["dram_bytes_per_step"] > 1e10
        # 20.6 GB algorithmic per 32-image step at 4 B per activation element: the capture must be within 5 % of it
        assert abs(t["dram_bytes_per_step"] / 20.6e9 - 1.0) < 0.05


def test_committed_bench_lines_parse_and_name_their_configuration():
    seen = set()
    for f in glob.glob(os.path.join(ROOT, "profiles", "r2_bench_*.json")):
        d = json.loads([l for l in open(f) if l.startswith("{")][-1])
        assert d["unit"] == "images/s" and d["higher_is_better"] is True and d["data"] == "synthetic" and d["value"] > 0
        if d.get("impl") == "reference":
            assert d["cpu_baseline"]["kind"] == "port" and d["gpu_launches"] == 0
            continue
        assert d["roofline"]["bound"] == "tensor" and 0 < d["roofline"]["frac"] <= 1.0
        assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["gpu_launches"] > 0
        assert "hw_slowdown" not in d["clocks"]["reasons"] and "hw_thermal_slowdown" not in d["clocks"]["reasons"]
        seen.add((d["config"]["baseline_config"], d["n_gpus"]))
    assert {c for c, _n in seen} >= {"BASELINE.json configs[%d] (--config %d)" % (i - 1, i) for i in (2, 3, 4, 5)}
    assert {n for _c, n in seen} >= {1, 4, 8}


def test_dump_outputs_unpacks_rank_and_shape_buckets(tmp_path, monkeypatch):
    """--dump-outputs: the packed step results (per rank: each shape bucket's rois, then its int32 counts) come out as one
    rois / count pair per shape, images in rank order; above the byte cap a fixed sample of the images is written."""
    import numpy as np
    import torch
    shapes, per_shape, rows, world = [(600, 900), (900, 600)], 2, 3, 2
    rois = np.arange(world * len(shapes) * per_shape * rows * 5, dtype=np.float32).reshape(world, len(shapes), per_shape, rows, 5)
    count = np.arange(world * len(shapes) * per_shape, dtype=np.int32).reshape(world, len(shapes), per_shape)
    packed = torch.from_numpy(np.concatenate([np.concatenate([rois[r, s].reshape(-1), count[r, s].view(np.float32)])
                                              for r in range(world) for s in range(len(shapes))]))
    bench.dump_outputs(str(tmp_path / "a"), [packed], shapes, per_shape, rows, world)
    for s, (H, W) in enumerate(shapes):
        got = np.load(tmp_path / "a" / ("rois_%dx%d.npy" % (H, W)))
        assert got.dtype == np.float32 and np.array_equal(got, rois[:, s].reshape(world * per_shape, rows, 5))
        got = np.load(tmp_path / "a" / ("count_%dx%d.npy" % (H, W)))
        assert got.dtype == np.float64 and np.array_equal(got, count[:, s].reshape(-1))
    monkeypatch.setattr(bench, "DUMP_BYTES", 2 * (rows * 5 * 4 + 8) * len(shapes))
    bench.dump_outputs(str(tmp_path / "b"), [packed], shapes, per_shape, rows, world)
    for s, (H, W) in enumerate(shapes):
        idx = np.load(tmp_path / "b" / ("image_index_%dx%d.npy" % (H, W))).astype(int)
        assert len(idx) == 2 and np.array_equal(idx, np.unique(idx))
        got = np.load(tmp_path / "b" / ("rois_%dx%d.npy" % (H, W)))
        assert np.array_equal(got, rois[:, s].reshape(world * per_shape, rows, 5)[idx])
