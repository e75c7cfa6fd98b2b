"""bench.py --dump-outputs on the GPU: the dump is what the timed path returns in its last step, on inputs that are the same from
run to run, and --steps sets the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

import posediffusion_b200 as pdb
from posediffusion_b200 import synthetic as syn
from posediffusion_b200.distributed import sequence_seed

pytestmark = pytest.mark.gpu


def bench(out_dir, *args):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--no-cpu-baseline", "--warmup", "1", "--dump-outputs",
                          str(out_dir), *args], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    return json.loads([l for l in res.stdout.splitlines() if l.startswith("{")][-1])


def test_dump_outputs_is_the_sampled_pose(tmp_path):
    frames = 5  # --workload cfg1: one sequence, GGS off
    one = bench(tmp_path / "one", "--workload", "cfg1", "--steps", "1")
    three = bench(tmp_path / "three", "--workload", "cfg1", "--steps", "3")
    assert one["steps"] == 1 and three["steps"] == 3
    assert sorted(os.listdir(tmp_path / "one")) == ["pose.npy"]
    got = np.load(tmp_path / "one" / "pose.npy")
    assert got.dtype == np.float32 and got.shape == (1, frames, 9) and np.isfinite(got).all()

    dev = torch.device("cuda:0")
    den = pdb.Denoiser(TRANSFORMER=dict(d_model=512, nhead=4, dim_feedforward=1024, num_encoder_layers=8, dropout=0.1,
                                        batch_first=True, norm_first=True))
    den.load_state_dict(syn.random_denoiser_state(0), strict=True)
    ctx = den.to(dev).native_context()
    ctx.set_denoiser_engine("auto")  # bench.py's default
    z = syn.random_features(1, frames, sequence_seed(0, 0)).to(dev)
    draws = syn.predraw_noise(1, frames, seed=sequence_seed(0, 0)).to(dev).contiguous()
    want, _, _ = ctx.sample_loop(z, draws, None, None, 0, want_trail=False, want_stats=False)
    want = want.cpu().numpy()
    scale = np.abs(want).max()
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-6 * scale)
    np.testing.assert_allclose(np.load(tmp_path / "three" / "pose.npy"), got, rtol=0, atol=1e-6 * scale)
