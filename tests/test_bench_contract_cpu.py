"""The bench JSON lines committed under profiles/ carry every key of the bench contract (bench.py docstring / task statement)."""
import json
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(name):
    with open(os.path.join(ROOT, "profiles", name)) as f:
        return json.loads(f.read().strip().splitlines()[-1])


@pytest.mark.parametrize("name,n", [("r01_bench_n1.json", 1), ("r01_bench_n2.json", 2), ("r02_bench_n1.json", 1), ("r02_bench_n2.json", 2)])
def test_product_arm_line(name, n):
    d = _load(name)
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "clocks", "e2e", "gpu_launches", "roofline"):
        assert k in d, k
    assert d["n_gpus"] == n and d["unit"] == "images/sec" and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["dtype"] == "bf16" and d["vs_baseline"] is None and d["warmup"] >= 3 and "workload" in d["config"]
    assert d["gpu_launches"] > 0 and abs(d["value"] - d["config"]["global_batch"] / (d["ms_per_step"] / 1e3)) < 1e-6 * d["value"]
    e = d["e2e"]
    assert e["unit"] == d["unit"] and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] != d["value"]
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["traffic"] > 0
    c = d["clocks"]
    assert c["sm_mhz"] > 0 and not set(c["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    if n == 1:
        b = d["cpu_baseline"]
        assert b["kind"] in ("port", "reference") and b["cores"] >= 1 and b["value"] > 0 and b["sample"]
    if name.startswith("r02"):
        # round 2: algorithmic bytes are the section-8(d) ones only (weights), DRAM traffic from the round's ncu capture within 10 %,
        # every other decode kernel class has its own entry, and the full-size parity check rides in the line with no violation
        assert r["algorithmic_bytes"].keys() == {"weights"} and 1.0 <= r["traffic"] / r["algorithmic_bytes_per_launch"] < 1.1
        assert any("decode_attention" in o["kernel"] and 0 < o["frac"] < 1.1 for o in r["other_kernels"])
        if n > 1:
            return
        pc = d["parity_check"]
        assert pc["violations"] == [] and pc["assembled_ids_exact"] and pc["nms_keep_exact_on_own_proposals"] and "floor" in pc


def test_reference_arm_line_round2():
    d = _load("r02_bench_reference_arm.json")
    assert d["impl"] == "reference" and d["value"] > 0 and d["e2e"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1


def test_reference_arm_line():
    d = _load("r01_bench_reference_arm.json")
    assert d["impl"] == "reference" and d["unit"] == "images/sec" and d["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["kind"] in ("port", "reference")


def test_dump_outputs_writes_what_generate_returned(tmp_path):
    """bench.py --dump-outputs: float32 / float64 arrays, token ids exact, large outputs as the same seeded sample every run,
    64 MB at most -- on the full-size shapes of a generate() result (KV cache shortened to 300 positions of 320)."""
    from types import SimpleNamespace

    import numpy as np
    import torch

    import bench
    g = torch.Generator().manual_seed(0)
    B, R, H = 16, 100, 4096
    boxes = [torch.rand(R, 4, generator=g) for _ in range(B)]
    vis = {"pred_boxes": boxes, "image_features": torch.randn(B, 256, H, generator=g).bfloat16(),
           "region_features": torch.randn(B * R, H, generator=g).bfloat16()}
    kv_store = torch.randn(32, 2, 2, 32, 320, 128, generator=g).bfloat16()
    out = SimpleNamespace(hidden_states=((None, vis),), past_key_values=tuple((kv_store[i, 0, :, :, :300], kv_store[i, 1, :, :, :300])
                                                                              for i in range(32)))
    seq = torch.randint(0, 32003, (B, 640), generator=g)
    written = bench.dump_outputs(str(tmp_path / "a"), seq, out)
    bench.dump_outputs(str(tmp_path / "b"), seq, out)
    assert sum(written.values()) <= 64 << 20
    for name in written:
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), name
    assert np.array_equal(np.load(tmp_path / "a" / "sequences.npy").astype(np.int64), seq.numpy())
    assert np.array_equal(np.load(tmp_path / "a" / "pred_boxes.npy"), torch.cat(boxes).numpy())
    img = np.load(tmp_path / "a" / "image_features.npy")
    assert img.shape == (bench.DUMP_SAMPLE,) and np.isin(img, vis["image_features"].float().numpy()).all()
    assert np.load(tmp_path / "a" / "past_key_values.npy").shape == (64, bench.DUMP_SAMPLE // 64)
