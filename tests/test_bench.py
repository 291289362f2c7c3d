"""bench.py's command line: --steps sets the timed steps, --dump-outputs writes what the last timed step returned."""
import contextlib
import io
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def test_bench_rejects_zero_steps(tmp_path):
    p = subprocess.run([sys.executable, BENCH, "--steps", "0"], cwd=tmp_path, capture_output=True, text=True, timeout=120)
    assert p.returncode == 2 and "error" in p.stderr, p.stderr
    assert not os.listdir(tmp_path)


def test_bench_reference_arm_dumps_its_logits(tmp_path):
    """--impl reference on the host: the logits of its last timed forward; where the reference's model code is not
    staged the arm times the oracle, whose output on the same seeded clouds is known exactly."""
    import bench
    from oracle import reference
    from oracle import svnet_oracle as orc
    import svnet_b200 as sv
    from svnet_b200.synthetic import make_args, synthetic_clouds, synthetic_state_dict
    out = tmp_path / "dump"
    p = subprocess.run([sys.executable, BENCH, "--impl", "reference", "--steps", "2", "--warmup", "0",
                        "--dump-outputs", str(out)], cwd=tmp_path, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    line = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["dump"] and sorted(os.listdir(out)) == ["logits.npy"]
    got = np.load(out / "logits.npy")
    assert got.dtype == np.float32 and got.ndim == 2 and got.shape[1] == bench.N_CLASS and np.isfinite(got).all()
    if not reference.available():
        assert line["cpu_baseline"]["kind"] == "port"
        with contextlib.redirect_stdout(io.StringIO()):
            net = sv.SV_DGCNN_CLS(make_args(k=bench.K_NN, binary=True), bench.N_CLASS)
        sd = synthetic_state_dict(net.state_dict(), seed=bench.SEED)
        want = orc.sv_dgcnn_cls(sd, synthetic_clouds(got.shape[0], bench.N_POINTS, bench.SEED).numpy(), bench.K_NN)
        assert np.array_equal(got, want)


@pytest.mark.gpu
def test_bench_dump_outputs_are_the_logits_of_the_timed_path(tmp_path):
    """Three timed steps (the JSON line counts the replays the timed region ran), dumped logits bit-identical to
    model(x) on the bench's seeded clouds and checkpoint."""
    import bench
    import svnet_b200 as sv
    from svnet_b200.synthetic import make_args, synthetic_clouds, synthetic_state_dict
    out = tmp_path / "dump"
    p = subprocess.run([sys.executable, BENCH, "--gpus", "1", "--steps", "3", "--warmup", "1", "--no-extra",
                        "--no-cpu-baseline", "--dump-outputs", str(out)],
                       cwd=tmp_path, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    line = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 3
    assert line["gpu_launches"] == 3 * line["gpu_launches_per_step"]["graph_replay"]
    assert sorted(os.listdir(out)) == ["logits.npy"]
    got = np.load(out / "logits.npy")
    assert got.dtype == np.float32 and got.shape == (bench.B_PER_GPU, bench.N_CLASS)
    with contextlib.redirect_stdout(io.StringIO()):
        net = sv.SV_DGCNN_CLS(make_args(k=bench.K_NN, binary=True), bench.N_CLASS)
    net.load_state_dict(synthetic_state_dict(net.state_dict(), seed=bench.SEED))
    net = net.cuda().eval()
    x = synthetic_clouds(bench.B_PER_GPU, bench.N_POINTS, bench.SEED).cuda()
    with torch.no_grad():
        want = net(x).cpu().numpy()
    assert np.array_equal(got, want)
