"""bench.py contract pieces that run without a GPU: the reference arm's JSON line and argument handling."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_contract_keys():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=900, env=dict(os.environ, OMP_NUM_THREADS="8"))
    assert r.returncode == 0, r.stderr[-1500:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ["impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"]:
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "tiles/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]


def test_dump_outputs_writes_float32_arrays_and_a_fixed_sample_of_large_ones(tmp_path):
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    assert 7 * bench.DUMP_SAMPLE * 4 <= 64e6                      # seven outputs per step, float32
    mods = [torch.full((2, 3, 4, 4), float(i)) for i in range(4)]
    seg = torch.arange(bench.DUMP_SAMPLE + 1000, dtype=torch.float32)
    seg_u8 = torch.randint(0, 256, (2, 4, 4, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(1))
    mask = seg_u8[..., 0] // 2
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), (mods, seg, seg_u8, mask))
    names = ["mod1", "mod2", "mod3", "mod4", "seg", "seg_u8", "mask"]
    assert sorted(os.listdir(tmp_path / "a")) == sorted(n + ".npy" for n in names)
    got = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in names}
    assert all(a.dtype == np.float32 for a in got.values())
    for i in range(4):
        assert np.array_equal(got[f"mod{i + 1}"], mods[i].numpy())
    assert np.array_equal(got["seg_u8"], seg_u8.float().numpy()) and np.array_equal(got["mask"], mask.float().numpy())
    s = got["seg"]                                                  # values = flat indices of the sampled elements
    assert s.shape == (bench.DUMP_SAMPLE,) and (np.diff(s) > 0).all() and s[-1] < seg.numel()
    assert np.array_equal(s, np.load(tmp_path / "b" / "seg.npy"))


def test_dump_outputs_is_refused_outside_the_inference_workload(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "train", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not os.listdir(tmp_path)


def test_b200_arm_refuses_to_run_without_cuda():
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True,
                       text=True, timeout=300)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)
