"""Developer tool: time eager `model(x)` of each binary SV model on cuda:0 with a ternary checkpoint (exact zeros in every
binarised weight, tests/test_gpu_ternary_weights.py's patterns) against a zero-free checkpoint of the same shape.

    python tools/ternary_time.py --out profiles/r3_ternary_time.json

The ternary checkpoint runs the zero-aware kernel variants (non-zero planes, the generic edge kernel where the tensor-core edge
kernel does not cover the layer, the unstaged head); the zero-free one the +-1 kernels.  Timing: CUDA events around `--iters`
forwards, the two arms alternated over `--rounds` rounds after a warm-up of both; the median over rounds is reported, with the
card's name and power limit read in the same process.
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import svnet_b200 as sv  # noqa: E402
from svnet_b200.synthetic import make_args, one_hot_labels, synthetic_clouds, synthetic_state_dict  # noqa: E402
from tests.test_gpu_ternary_weights import ternary_state_dict  # noqa: E402

# (model, k, B, N, classes): the BASELINE shapes of the DGCNN models, PointNet at the same cloud size as the classifier
MODELS = [("SV_DGCNN_CLS", 20, 32, 1024, 40), ("SV_DGCNN_CLS", 40, 32, 1024, 40), ("SV_DGCNN_PSEG", 40, 16, 2048, 50),
          ("SV_PointNet_CLS", 20, 32, 1024, 40), ("SV_PointNet_PSEG", 20, 16, 2048, 50)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def build(name, k, ncls, ternary):
    with contextlib.redirect_stdout(io.StringIO()):
        net = getattr(sv, name)(make_args(k=k, binary=True), ncls)
    sd = ternary_state_dict(net.state_dict(), 8000 + k) if ternary else synthetic_state_dict(net.state_dict(), seed=8000 + k)
    net.load_state_dict(sd)
    return net.cuda().eval()


def time_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "ternary_time.py times the GPU: no CUDA device"
    res = {"card": card(), "iters": a.iters, "rounds": a.rounds, "models": {}}
    for name, k, B, N, ncls in MODELS:
        x = synthetic_clouds(B, N, 8000).cuda()
        extra = (one_hot_labels(B).cuda(),) if name.endswith("PSEG") else ()
        nets = {"zero_free": build(name, k, ncls, False), "ternary": build(name, k, ncls, True)}
        runs = {arm: (lambda net=net: net(x, *extra)) for arm, net in nets.items()}
        ms = {arm: [] for arm in runs}
        with torch.no_grad():
            for fn in runs.values():
                for _ in range(3):
                    fn()
            torch.cuda.synchronize()
            for _ in range(a.rounds):
                for arm, fn in runs.items():
                    ms[arm].append(time_ms(fn, a.iters))
        row = {"k": k, "B": B, "N": N}
        for arm, v in ms.items():
            med = sorted(v)[len(v) // 2]
            row[arm] = {"ms_median": med, "ms_all": v, "clouds_per_s": B / med * 1e3}
        row["ternary_over_zero_free"] = row["ternary"]["ms_median"] / row["zero_free"]["ms_median"]
        res["models"]["%s_k%d" % (name, k)] = row
        print(name, k, json.dumps({arm: round(row[arm]["ms_median"], 3) for arm in ms}), flush=True)
        del nets, runs
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
