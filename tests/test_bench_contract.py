"""The committed bench lines (profiles/r02_bench_*.json, written by bench.py on a B200) carry every key of the bench
contract, with consistent values; bench.py's flags and its CPU-side helpers work without a GPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROFILES = os.path.join(ROOT, "profiles")


def _line(name):
    with open(os.path.join(PROFILES, name)) as fh:
        return json.loads(fh.read().strip().splitlines()[-1])


@pytest.mark.parametrize("name", ["r02_bench_1gpu.json", "r02_bench_cfg2.json", "r02_bench_cfg3.json", "r02_bench_cfg5.json",
                                  "r02_bench_2gpu.json", "r02_bench_8gpu_strong.json"])
def test_committed_bench_lines_follow_the_contract(name):
    d = _line(name)
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "kernels"):
        assert k in d, k
    assert d["unit"] == "frame-pairs/s" and d["higher_is_better"] is True and d["data"] == "synthetic"
    assert d["vs_baseline"] is None                          # BASELINE.md publishes no number for this metric
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["warmup"] >= 3 and d["gpu_launches"] > 0 and d["value"] > 0
    e = d["e2e"]
    assert e["unit"] == d["unit"] and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
    assert 0.5 * d["value"] < e["value"] <= 1.05 * d["value"]          # copies inside the timed region cost something
    r = d["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in r, k
    assert r["bound"] in ("hbm", "tensor") and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-3 and 0 < r["frac"] < 1
    c = d["clocks"]
    assert c["sm_mhz"] and c["sm_max_mhz"] and not ({"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(c["reasons"]))
    # value is the whole-job aggregate: pairs per step / step time
    pairs = d["config"]["global_pairs_per_step"]
    assert abs(d["value"] - pairs / (d["ms_per_step"] / 1e3)) < 1e-3 * d["value"]
    if d["n_gpus"] > 1:
        assert d["shard_equal"] is True                      # N-GPU result == 1-GPU result, checked in the run
    elif d.get("cpu_baseline"):
        b = d["cpu_baseline"]
        assert b["kind"] == "port" and b["cores"] >= 1 and b["value"] > 0 and "sample" in b
    for k in d["kernels"]:
        if k.get("frac") is not None:
            assert 0 < k["frac"] < 1.2, k                    # a fraction of a measured peak (HBM rows can brush 1)


def test_reference_arm_prints_a_contract_line_without_a_gpu():
    """bench.py --impl reference runs the oracle port on the host cores (the only place bench.py executes oracle/); on a
    tiny configuration it finishes in seconds and prints one JSON line with impl / cpu_baseline / e2e."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "cfg5", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["gpu_launches"] == 0 and d["value"] > 0
    assert d["cpu_baseline"]["value"] == d["value"] and d["e2e"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_dump_outputs_keeps_a_fixed_sample_under_the_limit(tmp_path):
    """bench.dump_outputs writes float32 as computed and integer outputs as float64; past DUMP_LIMIT every per-pair array
    keeps the same seeded subset of frame-pairs, recorded in pair_index.npy, and the files stay under the limit."""
    import numpy as np
    import torch
    import bench
    B = 256
    g = torch.Generator().manual_seed(0)
    per_pair = {"link": torch.rand(B, 3, 128, 128, generator=g), "match": torch.randint(-1, 128, (B, 128), generator=g, dtype=torch.int32)}
    shared = {"trans2": torch.rand(1, 64, 64, generator=g), "status": torch.zeros(1, dtype=torch.int32)}
    bench.dump_outputs(str(tmp_path / "a"), [("", per_pair, shared, B)])
    bench.dump_outputs(str(tmp_path / "b"), [("", per_pair, shared, B)])
    a = {f: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert set(a) == {"link.npy", "match.npy", "trans2.npy", "status.npy"}                    # 50 MB: written in full
    assert a["link.npy"].dtype == np.float32 and a["match.npy"].dtype == np.float64
    assert np.array_equal(a["match.npy"], per_pair["match"].numpy()) and np.array_equal(a["link.npy"], per_pair["link"].numpy())
    big = {"link": torch.cat([per_pair["link"]] * 2)}
    for d in ("c", "d"):
        bench.dump_outputs(str(tmp_path / d), [("", big, shared, 2 * B)])
    idx = np.load(tmp_path / "c" / "pair_index.npy")
    assert 0 < len(idx) < 2 * B and np.array_equal(idx, np.load(tmp_path / "d" / "pair_index.npy"))
    assert np.array_equal(np.load(tmp_path / "c" / "link.npy"), big["link"].numpy()[idx.astype(np.int64)])
    assert sum(os.path.getsize(tmp_path / "c" / f) for f in os.listdir(tmp_path / "c")) <= bench.DUMP_LIMIT


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_path_repeat_exactly(tmp_path):
    """bench.py --dump-outputs on a small cfg4 batch, twice: the same seeded inputs give the same outputs bit for bit, and
    the files are what predict_batch returns (per-pair scores, assignments and match indices, trans, status)."""
    import numpy as np
    outs = []
    for run in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--pairs", "2",
                            "--no-cpu", "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
        outs.append({f[:-4]: np.load(tmp_path / run / f) for f in os.listdir(tmp_path / run)})
    a, b = outs
    assert set(a) == {"det", "link", "new", "end", "assign_det", "assign_link", "assign_new", "assign_end", "match", "trans1",
                      "trans2", "status"}
    assert a["link"].shape == (2, 3, 128, 128) and a["link"].dtype == np.float32 and a["match"].shape == (2, 128)
    assert a["status"][0] == 0 and np.all((a["match"] >= -1) & (a["match"] < 128))
    for k in a:
        assert np.array_equal(a[k], b[k]), k
