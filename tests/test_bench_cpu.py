"""CPU: the reference arm of bench.py (--impl reference) runs without a GPU and prints the contract's JSON line."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_contract_line():
    out = subprocess.run(
        [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
         "--cpu-sample-tokens", "1024", "--cpu-config1-tokens", "512"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "GB/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["vs_baseline"] is None and line["steps"] == 1
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "sample" in cb
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"]
    # the label says what was run: the bounded sample is named in the config (identically in both arms) and in cpu_baseline
    assert "1024 tokens" in line["config"]["reference_arm_sample"] and "1024 tokens" in cb["sample"]
    c1 = cb["config1_check"]
    assert c1["tokens"] == 512 and c1["seconds"] > 0 and c1["GBps_of_bf16_KV"] > 0


def test_both_arms_describe_the_same_config():
    """The driver compares the two arms' `config` objects: they must be equal by content for equal flags."""
    sys.path.insert(0, ROOT)
    import argparse

    import bench

    args = argparse.Namespace(config=2, tokens=0, gpus=1, streams=6, cpu_sample_tokens=0)
    c = bench.config_of(args)
    assert args.cpu_sample_tokens == 65536      # the CPU arm's sample is taken at the configuration's own context length
    assert bench.workload_config(args, c) == bench.workload_config(args, dict(c))
    assert bench.kv_bytes_of(c) == 8589934592 and bench.group_sizes(c) == [4] * 8
    assert bench.group_sizes(bench.CONFIGS[5]) == [4] * 6 + [3]
    assert bench.kv_bytes_of(bench.CONFIGS[4]) == 2 * 80 * 131072 * 1024 * 2


def test_dump_outputs_writes_seeded_row_samples_within_budget(tmp_path):
    """--dump-outputs: every factor of every group as float32 .npy, larger ones as the same seeded row sample every time."""
    sys.path.insert(0, ROOT)
    import types

    import numpy as np
    import torch

    import bench

    gen = torch.Generator().manual_seed(0)

    def side(m, n, r):
        return types.SimpleNamespace(A=torch.randn(m, r, generator=gen).bfloat16(), V=torch.randn(n, r, generator=gen).bfloat16(),
                                     sigma_lead=torch.rand(8, generator=gen))

    groups = [types.SimpleNamespace(key=side(4096, 256, 16), value=side(4096, 256, 24)),
              types.SimpleNamespace(key=side(4096, 256, 16), value=None)]
    budget = 400_000
    shapes = bench.dump_outputs(groups, str(tmp_path / "a"), budget=budget)
    assert sorted(shapes) == sorted(f"group{g}_{s}_{x}" for g, s in ((0, "k"), (0, "v"), (1, "k")) for x in ("A", "V", "sigma"))
    files = sorted((tmp_path / "a").iterdir())
    assert len(files) == len(shapes) and sum(f.stat().st_size for f in files) <= budget
    bench.dump_outputs(groups, str(tmp_path / "b"), budget=budget)
    for f in files:
        a, b = np.load(f), np.load(tmp_path / "b" / f.name)
        assert a.dtype == np.float32 and np.array_equal(a, b)
    a = np.load(tmp_path / "a" / "group0_k_A.npy")
    full = groups[0].key.A.float().numpy()
    assert 0 < a.shape[0] < full.shape[0]
    rows = [int(np.flatnonzero((full == row).all(axis=1))[0]) for row in a]
    assert rows == sorted(set(rows))            # distinct rows of the factor, in ascending order
    assert np.array_equal(np.load(tmp_path / "a" / "group1_k_sigma.npy"), groups[1].key.sigma_lead.numpy())


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                         timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "--steps" in out.stderr
