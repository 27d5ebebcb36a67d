"""bench.py: what --dump-outputs writes for an output small enough to keep whole and for one that is sampled, the
arguments it refuses, and the exact step count of the `--impl reference` hot-path arm."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from oracle import cpu_reference


def test_small_output_is_written_whole(tmp_path):
    out = torch.randn(2, 64, 5, 7).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    written = bench.dump_outputs(str(tmp_path / "d"), "sr", [out[:1], out[1:]])
    assert written == {"sr.npy": out.numel() * 4}
    got = np.load(tmp_path / "d" / "sr.npy")
    assert got.dtype == np.float32 and got.shape == tuple(out.shape)
    assert np.array_equal(got, out.float().numpy())


def test_large_output_is_a_fixed_sample_within_the_limit(tmp_path):
    out = torch.arange(2200 * 4096, dtype=torch.float32).view(2200, 4096)[:, :4000]     # a view, as the cropped SR
    assert out.numel() > bench.DUMP_WHOLE
    a = bench.dump_outputs(str(tmp_path / "a"), "sr", out)
    b = bench.dump_outputs(str(tmp_path / "b"), "sr", [out[:1000], out[1000:1001], out[1001:]])     # --streams > 1
    assert a == b and sorted(a) == ["sr.npy", "sr_index.npy"] and sum(a.values()) <= bench.DUMP_LIMIT
    val, idx = np.load(tmp_path / "a" / "sr.npy"), np.load(tmp_path / "a" / "sr_index.npy")
    assert val.dtype == np.float32 and idx.dtype == np.float64
    assert len(val) == len(idx) == bench.DUMP_SAMPLE
    assert np.all(np.diff(idx) > 0) and idx[-1] < out.numel()
    assert np.array_equal(val, (idx // 4000 * 4096 + idx % 4000).astype(np.float32))      # row-major flat indices
    for f in a:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))


def test_scalar_output(tmp_path):
    assert bench.dump_outputs(str(tmp_path), "loss", torch.tensor(0.25)) == {"loss.npy": 4}
    got = np.load(tmp_path / "loss.npy")
    assert got.shape == () and got == np.float32(0.25)


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]])
def test_refused_arguments(argv, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(bench.ROOT, "bench.py"), *argv], cwd=tmp_path,
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "error:" in r.stderr and not r.stdout
    assert not (tmp_path / "unused").exists()


def test_reference_hotpath_times_exactly_the_requested_clips():
    fps, sample = cpu_reference.time_hotpath_sample(16, 32, 3, clips=2)
    assert fps > 0 and sample.startswith(f"{2 * 4 * (2 * 3 - 3)} MultiAdSTN-equivalents")
