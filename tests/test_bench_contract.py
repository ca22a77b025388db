"""bench.py's reference arm runs anywhere (it times the CPU port): its JSON line carries the
contract's keys.  The GPU arm prints the same keys plus roofline / clocks (checked on the GPU box
by the driver; profiles/r01_bench_n1.json is a committed sample)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline"}


def test_reference_arm_line():
  out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=600, check=True).stdout
  line = json.loads(out.strip().splitlines()[-1])
  assert line["impl"] == "reference" and KEYS <= set(line)
  assert line["unit"] == "input-samples/s" and line["higher_is_better"] is True and line["value"] > 0
  assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
  assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
  assert "workload" in line["config"]


def test_round2_gpu_sample_has_the_contract_keys_and_the_new_records():
  line = json.load(open(os.path.join(ROOT, "profiles", "r02_bench_n1.json")))
  assert KEYS | {"clocks", "gpu_launches", "roofline"} <= set(line)
  roof = line["roofline"]
  assert roof["bound"] == "hbm" and abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-9
  assert roof["sustained"]["seconds"] >= 2.0 and roof["sustained"]["frac"] <= roof["burst"]["frac"] * 1.02   # >= 2 s of back-to-back launches
  assert abs(roof["achieved"] - 260 * 4096 * 16384 / (line["ms_per_step"] * 1e-3) / 1e9) < 1e-6 * roof["achieved"]
  assert line["gpu_launches"] == line["steps"] and line["dtype"] == "f64"
  cpu = line["cpu_baseline"]
  assert cpu["kind"] == "port" and cpu["reps"] >= 5 and cpu["min"] <= cpu["value"] <= cpu["max"]
  assert cpu["cores"] <= cpu["host"]["affinity"]                      # never more threads than the process may use
  for key in ("strategies", "cfg2", "cfg3", "cfg5", "few_streams", "generic", "stream_api"):
    assert key in line and "error" not in line[key], key
  assert set(line["strategies"]) == {"klapuri", "sampled"}
  assert line["stream_api"]["cfg1"]["ours_samples_per_s"] > line["stream_api"]["cfg1"]["python_port_samples_per_s"]
  assert line["e2e"]["h2d_bytes_per_step"] == 4096 * 16384 * 4 and line["e2e"]["d2h_bytes_per_step"] == 4096 * 64 * 16384 * 4


def test_committed_gpu_sample_has_the_contract_keys():
  line = json.load(open(os.path.join(ROOT, "profiles", "r01_bench_n1.json")))
  assert KEYS | {"clocks", "gpu_launches", "roofline"} <= set(line)
  roof = line["roofline"]
  assert roof["bound"] == "hbm" and abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-9
  assert line["gpu_launches"] == line["steps"] and line["dtype"] == "f64"
  assert line["e2e"]["h2d_bytes_per_step"] == 4096 * 16384 * 4 and line["e2e"]["d2h_bytes_per_step"] == 4096 * 64 * 16384 * 4


def test_steps_must_be_positive_and_reference_arm_has_no_dump(tmp_path):
  for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=600)
    assert out.returncode == 2 and "error" in out.stderr, extra
  assert os.listdir(tmp_path) == []


def test_output_sample_is_seeded_and_bounded(monkeypatch):
  import torch
  import bench
  y = torch.arange(50 * 3 * 40, dtype=torch.float32).reshape(50, 3, 40)
  monkeypatch.setattr(bench, "DUMP_BYTES", 7 * 3 * 40 * 4 + 5)        # room for 7 whole streams
  got = bench.output_sample(y)
  streams = np.sort(np.random.default_rng(0).choice(50, 7, replace=False))
  assert got.dtype == np.float32 and np.array_equal(got, y.numpy()[streams])
  assert np.array_equal(bench.output_sample(y), got)
  monkeypatch.setattr(bench, "DUMP_BYTES", 3 * 4 * 10)                # one stream is too long: 10 time positions of it
  got = bench.output_sample(y)
  assert got.shape == (1, 3, 10) and got.nbytes <= bench.DUMP_BYTES
  rng = np.random.default_rng(0)
  s = rng.choice(50, 1, replace=False)
  assert np.array_equal(got, y.numpy()[s][:, :, np.sort(rng.choice(40, 10, replace=False))])


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(tmp_path):
  """--dump-outputs writes what the K-th timed step computed: the same bits as K + warm-up applications of the
  plan to the seeded input, run here; the line reports exactly K timed steps."""
  import torch
  if not torch.cuda.is_available():
    pytest.skip("no CUDA device")
  import bench
  import audiolazy_b200 as ab
  S, Tn, K = 96, 2048, 4
  out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--streams", str(S), "--samples", str(Tn),
                        "--steps", str(K), "--warmup", "3", "--no-extras", "--no-cpu", "--no-e2e", "--sustain-s", "0",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, check=True).stdout
  line = json.loads(out.strip().splitlines()[-1])
  assert line["steps"] == K and line["warmup"] == 3
  got = np.load(os.path.join(tmp_path, "y.npy"))
  assert os.listdir(tmp_path) == ["y.npy"] and got.dtype == np.float32 and got.shape[1:] == (64, Tn)
  torch.cuda.set_device(0)
  plan = ab.gammatone_bank(rate=48000, strategy="slaney").device_bank().plan
  gen = torch.Generator(device="cuda")
  gen.manual_seed(1234)
  x = torch.rand((S, Tn), device="cuda", generator=gen) * 2 - 1
  y = torch.empty((S, 64, Tn), dtype=torch.float32, device="cuda")
  state = torch.zeros(plan.state_doubles(S), dtype=torch.float64, device="cuda")
  for _ in range(3 + K):
    plan.apply(x.data_ptr(), y.data_ptr(), state.data_ptr(), S, Tn, Tn, Tn, torch.cuda.current_stream().cuda_stream)
  torch.cuda.synchronize()
  assert np.array_equal(got, bench.output_sample(y))
