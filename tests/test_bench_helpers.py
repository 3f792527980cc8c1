"""bench.py's accounting helpers (no GPU): the per-stage byte model, the roofline record over all
stages (library calls included and flagged), and the config object both arms print."""
import json

import bench


def test_stage_bytes_follow_the_design_table():
    kw = dict(n_pts=7_680_000, rays=290_000, pairs=38_000_000, general=1_900_000, blocks=85)
    assert bench.stage_alg_bytes("bundle_sort", **kw) == 16 * 7_680_000
    assert bench.stage_alg_bytes("point_keys", **kw) == 20 * 7_680_000
    assert bench.stage_alg_bytes("gather_sorted", **kw) == 40 * 7_680_000
    assert bench.stage_alg_bytes("finalize", **kw) == 98304 * 85
    assert bench.stage_alg_bytes("merge_resample", b_in=80, b_out=70, **kw) == 49152 * (80 + 140)
    assert bench.stage_alg_bytes("no_such_stage", **kw) == 0.0


def test_roofline_record_picks_the_dominant_stage_over_all_stages():
    steps = 10
    prof = {"bundle_sort": (3.5, 0), "walk_segments": (2.0, 20), "point_keys": (0.9, 10),
            "transfer": (9.0, 0), "fold_wide": (0.0, 10)}
    per_step = dict(n_pts=7_680_000, rays=290_000, pairs=38_000_000, general=1_900_000, blocks=85)
    r = bench.roofline_record(prof, steps, 1.5, 308e6, per_step, traffic_file=None)
    assert r["kernel"] == "bundle_sort" and r["library_kernel"] is True   # not hidden as in round 1
    assert abs(r["ms_per_launch"] - 0.35) < 1e-12
    assert abs(r["achieved"] - 16 * 7_680_000 / 0.35e-3 / 1e9) < 1e-6      # the stage's OWN bytes
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert abs(r["step_frac"] - 308e6 / 1.5e-3 / 1e9 / r["peak"]) < 1e-12  # the headline fraction
    assert abs(r["library_stages_ms_per_step"] - 0.35) < 1e-12
    assert r["traffic"] is None and r["bound"] == "hbm" and r["unit"] == "GB/s"
    json.dumps(r)


def test_both_arms_print_the_same_config_object():
    assert set(bench.CONFIG) == {"workload", "l2"} and "C2" in bench.CONFIG["workload"]
    src = open(bench.__file__).read()
    assert src.count('"config": dict(CONFIG)') == 2


def test_layer_diff_reports_margins():
    import numpy as np
    dt = np.dtype([("distance", "<f4"), ("weight", "<f4"), ("rgba", "u1", (4,))])
    idx = np.array([[0, 0, 0]], np.int32)
    a = np.zeros((1, 4096), dt)
    a["distance"], a["weight"] = 0.1, 2.0
    b = a.copy()
    b["distance"][0, 5] += 0.5e-5          # half the absolute tolerance... of 1e-5
    b["rgba"][0, 7, 1] = 1                 # one LSB
    d = bench.layer_diff((idx, b, None), (idx, a, None))
    assert d["block_sets_equal"] and d["within_tolerance"]
    assert 0.4 < d["max_distance_err_over_tol"] < 0.6 and d["colour_lsb_hist"][1] == 1
    b["weight"][0, 9] = 2.1
    assert not bench.layer_diff((idx, b, None), (idx, a, None))["within_tolerance"]
    assert not bench.layer_diff((np.array([[1, 0, 0]], np.int32), a, None), (idx, a, None))["block_sets_equal"]


class _FakeLayer:
    def __init__(self, blocks, seed):
        import numpy as np
        from coxgraph_b200 import VOXEL_DTYPE
        rng = np.random.default_rng(seed)
        self.idx = np.stack([np.arange(blocks), np.zeros(blocks), np.zeros(blocks)], 1).astype(np.int32)
        self.vox = np.zeros((blocks, 4096), VOXEL_DTYPE)
        self.vox["distance"] = rng.standard_normal((blocks, 4096))
        self.vox["weight"] = rng.random((blocks, 4096))
        self.vox["rgba"] = rng.integers(0, 256, (blocks, 4096, 4))
        self.flags = rng.integers(0, 4, blocks).astype(np.uint8)

    def download(self):
        return self.idx, self.vox, self.flags


def test_dump_outputs_writes_a_fixed_sample_as_float_arrays(tmp_path):
    import numpy as np
    from coxgraph_b200 import capi
    big, small = _FakeLayer(bench.DUMP_BLOCKS + 40, 1), _FakeLayer(7, 2)
    st = capi.MergeStats(blocks_in=5, blocks_candidate=9, blocks_out=8)
    out = bench.dump_outputs(str(tmp_path / "a"), {"global": big, "submap": small}, {"merge": st})
    again = bench.dump_outputs(str(tmp_path / "b"), {"global": big, "submap": small}, {"merge": st})
    for name, arr in out.items():
        on_disk = np.load(tmp_path / "a" / f"{name}.npy")
        assert on_disk.dtype in (np.float32, np.float64), name
        assert np.array_equal(on_disk, arr) and np.array_equal(on_disk, again[name]), name
    rows = out["global_sample_rows"].astype(int)
    assert len(rows) == bench.DUMP_BLOCKS and len(np.unique(rows)) == len(rows)
    assert np.array_equal(out["global_distance"], big.vox["distance"][rows])
    assert np.array_equal(out["global_rgba"], big.vox["rgba"][rows].astype(np.float32))
    assert np.array_equal(out["global_block_idx"], big.idx) and np.array_equal(out["global_flags"], big.flags)
    assert np.array_equal(out["submap_sample_rows"], np.arange(7))
    assert out["merge_blocks_out"] == 8.0 and out["merge_blocks_candidate"] == 9.0
    # the largest dump of the bench's layers (4096- and 32768-block capacities) fits in 64 MB
    worst = sum(b * 4 * 8 + min(b, bench.DUMP_BLOCKS) * (8 + 4096 * 6 * 4) for b in (4096, 32768))
    assert worst <= 64e6


def test_bench_refuses_zero_steps():
    import subprocess
    import sys
    r = subprocess.run([sys.executable, bench.__file__, "--steps", "0"], capture_output=True, text=True)
    assert r.returncode == 2 and "--steps" in r.stderr
