"""CPU-only checks of bench.py's output contract: the reference arm (`--impl reference`: the reference's own modules from the
reference checkout or oracle/_ref when present, else the CPU oracle port, on the host cores) prints ONE JSON line with the
documented keys, non-zero ranks of a multi-process launch exit without work, and the b200 arm refuses to run without a GPU
instead of falling back."""
import json
import os
import subprocess
import sys

from conftest import ROOT

BENCH = os.path.join(ROOT, "bench.py")


def run(args, env=None, timeout=600):
    e = dict(os.environ)
    e.update(env or {})
    e["PDB_REF_THREADS"] = "4"
    return subprocess.run([sys.executable, BENCH, *args], capture_output=True, text=True, timeout=timeout, env=e, cwd=ROOT)


def test_reference_arm_prints_one_contract_line():
    res = run(["--impl", "reference", "--workload", "cfg2", "--gpus", "1", "--steps", "1", "--warmup", "1"])
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["gpu_launches"] == 0
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
                "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["vs_baseline"] is None and d["value"] > 0
    from oracle import ref_loader

    want_kind = "reference" if ref_loader.reference_available() else "port"
    assert d["cpu_baseline"]["kind"] == want_kind and d["cpu_baseline"]["cores"] == 4 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_falls_back_to_the_port_without_the_reference(tmp_path):
    """Neither the reference checkout nor oracle/_ref: the arm times the oracle port and says so (`kind: "port"`)."""
    res = run(["--impl", "reference", "--workload", "cfg1", "--gpus", "1", "--steps", "1", "--warmup", "1"],
              env={"POSEDIFF_REFERENCE_ROOT": str(tmp_path), "POSEDIFF_INSTALLED_REFERENCE": str(tmp_path)})
    assert res.returncode == 0, res.stderr[-2000:]
    d = json.loads([l for l in res.stdout.splitlines() if l.startswith("{")][0])
    assert d["cpu_baseline"]["kind"] == "port" and d["value"] > 0


def test_reference_arm_fits_per_call_and_per_iteration_cost():
    """GGS on: calls with 7 and 21 inner iterations alternate; the line reports the per-iteration and per-call cost."""
    res = run(["--impl", "reference", "--workload", "cfg3", "--gpus", "1", "--steps", "1", "--warmup", "1", "--cpu-budget", "1"], timeout=900)
    assert res.returncode == 0, res.stderr[-2000:]
    d = json.loads([l for l in res.stdout.splitlines() if l.startswith("{")][0])
    assert "ms per inner iteration" in d["cpu_baseline"]["sample"] and "ms per call" in d["cpu_baseline"]["sample"]
    assert 0 < d["value"] < 50


def test_reference_arm_other_ranks_exit_without_work():
    res = run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"], env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"},
              timeout=120)
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_reference_arm_refuses_dump_outputs(tmp_path):
    """The reference arm extrapolates from a bounded sample, so it has no complete output to dump."""
    res = run(["--impl", "reference", "--steps", "1", "--dump-outputs", str(tmp_path / "out")], timeout=120)
    assert res.returncode != 0 and "--dump-outputs" in res.stderr
    assert not (tmp_path / "out").exists()


def test_b200_arm_has_no_cpu_fallback():
    import torch

    if torch.cuda.is_available():
        return  # on a GPU box this arm is exercised by the driver itself
    res = run(["--workload", "cfg2", "--steps", "1", "--warmup", "1", "--no-cpu-baseline"], timeout=300)
    assert res.returncode != 0
    assert "{\"metric\"" not in res.stdout
