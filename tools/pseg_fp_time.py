"""Developer tool: time the full-precision SV-DGCNN part-segmentation model (N = 2048, k = 40) on cuda:0, the layer-by-layer
path it had before against the current one, and record which edge kernel runs in each layer.

    python tools/pseg_fp_time.py --out profiles/r3_pseg_fp_time.json

Arms (each with the same seeded checkpoint and inputs):
  old         module path, fp head layer by layer over the (B*N, 2144) table, edge layers on edge_fp_fast_kernel
              (NATIVE_FORWARD = SEG_HEAD_CALL = False, SVNET_EDGE_FP_TC=0): the sequence before the fp head call existed
  old_graph   the same, replayed from a CUDA graph
  module      module path with the fp head call and edge_fp_tc_kernel (NATIVE_FORWARD = False)
  module_graph  the same, replayed from a CUDA graph
  c_entry     model(x, l) through the whole-model C entry, eager
Timing: CUDA events around `--iters` forwards, arms alternated over `--rounds` rounds after a warm-up of every arm; the
median over rounds is reported.  The working set at these sizes is far beyond the 126 MB L2.  Old and new logits are compared
on the timed inputs (max |difference|, per-point argmax agreement).  A torch.profiler pass of its own (B = 1) lists the edge
kernel of every layer for the old and the new path.
"""
import argparse
import contextlib
import io
import json
import os
import re
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import svnet_b200 as sv  # noqa: E402
from svnet_b200 import fused  # noqa: E402
from svnet_b200 import sv_dgcnn_partseg as ps  # noqa: E402
from svnet_b200.synthetic import make_args, one_hot_labels, synthetic_clouds, synthetic_state_dict  # noqa: E402


@contextlib.contextmanager
def arm(old, native):
    """old: the pre-existing fp sequence; native: model(x, l) may take the C entry."""
    keep = (fused.NATIVE_FORWARD, ps.SEG_HEAD_CALL, os.environ.get("SVNET_EDGE_FP_TC"))
    fused.NATIVE_FORWARD, ps.SEG_HEAD_CALL = native, not old
    if old:
        os.environ["SVNET_EDGE_FP_TC"] = "0"
    try:
        yield
    finally:
        fused.NATIVE_FORWARD, ps.SEG_HEAD_CALL = keep[0], keep[1]
        if keep[2] is None:
            os.environ.pop("SVNET_EDGE_FP_TC", None)
        else:
            os.environ["SVNET_EDGE_FP_TC"] = keep[2]


ARMS = {"old": (True, False, False), "old_graph": (True, False, True), "module": (False, False, False),
        "module_graph": (False, False, True), "c_entry": (False, True, False)}     # (old, native, graphed)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def edge_kernels_per_layer(net, x, l):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        net(x, l)
        torch.cuda.synchronize()
    names = [e.name for e in sorted(prof.events(), key=lambda e: e.time_range.start)
             if e.device_type == torch.autograd.DeviceType.CUDA]
    edge = [m.group(1) for m in (re.search(r"\b(edge_(?:xyz|bin|fp)_\w*kernel|svblock_edge_kernel)\b", n) for n in names) if m]
    return {"layer%d" % (i + 1): n for i, n in enumerate(edge)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="16,128")
    ap.add_argument("--N", type=int, default=2048)
    ap.add_argument("--k", type=int, default=40)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this tool measures on the GPU"
    with contextlib.redirect_stdout(io.StringIO()):
        net = sv.SV_DGCNN_PSEG(make_args(k=a.k, binary=False), 50)
    net.load_state_dict(synthetic_state_dict(net.state_dict(), seed=1004))
    net = net.cuda().eval()
    res = {"card": card(), "N": a.N, "k": a.k, "iters": a.iters, "rounds": a.rounds, "arms": {n: "old=%s native=%s graphed=%s" % v
                                                                                            for n, v in ARMS.items()}, "batches": {}}
    print(res["card"])
    with torch.no_grad():
        for B in [int(b) for b in a.batches.split(",")]:
            x = synthetic_clouds(B, a.N, 1004 + B).cuda()
            l = one_hot_labels(B).cuda()
            fwd, out = {}, {}
            for name, (old, native, graphed) in ARMS.items():
                with arm(old, native):
                    out[name] = net(x, l).clone()
                    if graphed:
                        gf = sv.GraphedForward(net, x, l)
                        fwd[name] = (lambda gf=gf: gf(x, l))
                    else:
                        fwd[name] = (lambda: net(x, l))
                    fwd[name]()
            torch.cuda.synchronize()
            times = {n: [] for n in ARMS}
            for _ in range(a.rounds):
                for name, (old, native, _) in ARMS.items():
                    with arm(old, native):
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        for _ in range(a.iters):
                            fwd[name]()
                        e1.record()
                        torch.cuda.synchronize()
                        times[name].append(e0.elapsed_time(e1) / a.iters)
            ref = out["old"].double()
            row = {}
            for name in ARMS:
                ms = sorted(times[name])[len(times[name]) // 2]
                d = (out[name].double() - ref).abs()
                row[name] = {"ms_median": ms, "ms_all": times[name], "clouds_per_s": B / ms * 1e3,
                             "max_abs_dlogit_vs_old": float(d.max()),
                             "max_dlogit_over_tolerance": float((d / (1e-4 + 1e-3 * ref.abs())).max()),   # <= 1: within 1e-3 rel / 1e-4 abs
                             "argmax_agree_vs_old": float((out[name].argmax(1) == out["old"].argmax(1)).double().mean())}
                print("B=%d %-13s %9.3f ms  %9.1f clouds/s  max|dlogit| %.3g  argmax agree %.6f" % (
                    B, name, ms, B / ms * 1e3, row[name]["max_abs_dlogit_vs_old"], row[name]["argmax_agree_vs_old"]))
            res["batches"][str(B)] = row
            del fwd, out
            torch.cuda.empty_cache()
        # profiler pass of its own, one cloud: which edge kernel each layer ran
        x1, l1 = synthetic_clouds(1, a.N, 7).cuda(), one_hot_labels(1).cuda()
        res["edge_kernels"] = {}
        for name in ("old", "module", "c_entry"):
            old, native, _ = ARMS[name]
            with arm(old, native):
                net(x1, l1)
                res["edge_kernels"][name] = edge_kernels_per_layer(net, x1, l1)
            print(name, res["edge_kernels"][name])
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
