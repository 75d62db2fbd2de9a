"""bench.py contract: the reference arm runs on the CPU (oracle port on all host cores) and prints ONE JSON line
with the keys the driver reads; the GPU arm's argument parsing does not need a GPU to import."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "sp5",
                          "--steps", "1", "--warmup", "0", "--cpu-sample", "4"], capture_output=True, text=True,
                         timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "cave_loss_grad_instances_per_sec" and d["unit"] == "instances/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "instances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_bad_steps_and_dumps_outside_the_gpu_path_are_refused(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "d")],
                  ["--workload", "sweep", "--dump-outputs", str(tmp_path / "d")]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True,
                             timeout=120, cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "" and "error" in out.stderr, (extra, out.stderr[-2000:])
    assert not (tmp_path / "d").exists()


def test_dump_outputs_writes_floats_and_samples_instances_above_the_limit(tmp_path):
    import bench
    rng = np.random.default_rng(1)
    arrays = {"loss": np.array(0.5, np.float32), "loss_i": rng.random(1000).astype(np.float32),
              "grad": rng.standard_normal((1000, 50)).astype(np.float32), "status": np.arange(1000, dtype=np.int32)}
    bench.dump_outputs(arrays, str(tmp_path / "full"))
    full = {f[:-4]: np.load(tmp_path / "full" / f) for f in os.listdir(tmp_path / "full")}
    assert sorted(full) == ["grad", "loss", "loss_i", "status"]
    for k, a in arrays.items():
        assert full[k].dtype in (np.float32, np.float64)
        np.testing.assert_array_equal(full[k], a)
    limit = 100_000                                   # the whole set is ~212 KB
    for name in ("a", "b"):
        bench.dump_outputs(arrays, str(tmp_path / name), limit=limit)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["grad.npy", "instance_index.npy", "loss.npy", "loss_i.npy", "status.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= limit
    for f in files:                                   # the sample is fixed: two dumps are byte for byte equal
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes()
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    idx = got["instance_index"].astype(np.int64)
    assert len(idx) > 400 and (np.diff(idx) > 0).all() and idx[-1] < 1000
    assert got["loss"] == arrays["loss"]
    for k in ("loss_i", "grad", "status"):
        assert got[k].dtype in (np.float32, np.float64)
        np.testing.assert_array_equal(got[k], arrays[k][idx])


@pytest.mark.gpu
def test_dumped_outputs_are_what_the_timed_step_returned(tmp_path):
    """--dump-outputs of a small TSP-20 batch against the same call on the same seeded inputs, bit for bit."""
    import torch
    from cave_b200 import cave_forward_backward, synth
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tsp20", "--batch", "64", "--steps", "2",
                          "--warmup", "0", "--no-e2e", "--no-cpu-baseline", "--no-extras", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["grad.npy", "loss.npy", "loss_i.npy"]
    dev = torch.device("cuda:0")
    insts = synth.make_batch("tsp20", 64, seed=1000)
    pred = torch.tensor(synth.predictions(insts, 1000, "uniform"), device=dev)
    ref = cave_forward_backward(pred, synth.densify(insts, device=dev), -1.0, 1, 0.2, "mean", precision="fp64")
    for k in ("loss", "loss_i", "grad"):
        np.testing.assert_array_equal(np.load(tmp_path / f"{k}.npy"), ref[k].cpu().numpy(), err_msg=k)
