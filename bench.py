#!/usr/bin/env python
"""bench.py -- headline benchmark: SV-DGCNN clouds/sec (binary, ModelNet40 head, N=1024, k=20).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one forward of the hot path over one batch of B=32 synthetic clouds per GPU
(BASELINE.json configs[1]).  Multi-GPU (launched by torchrun, one rank per GPU) shards by cloud
batch -- weak scaling, B=32 per GPU -- with a single NCCL all-gather of the logits per step.

Prints ONE JSON line (rank 0).  `value` is device-timed with inputs resident in HBM; `e2e` is the
same metric through the public nn.Module call with pinned HOST buffers (H2D of the clouds and D2H
of the logits inside the timed region).  `roofline` is for the dominant kernel, timed live with
CUDA events on its launch stream; `cpu_baseline` is the oracle port (C + OpenMP) on the host cores.
`--impl reference` times the UNMODIFIED reference forward (oracle/_ref, staged by oracle/make_ref.sh:
the reference's own models/*.py, stock PyTorch on the host cores, all threads) on the same config.
Extra keys of our line: `gpu_eager_reference` (the same reference modules on cuda: stock eager fp32),
`extra.cfg3` / `extra.cfg4` / `extra.cfg5` (BASELINE.json configs[2] / configs[3] / three points of configs[4]'s sweep, batch-sharded over the ranks: strong
scaling, cfg4 with the all-gather of the per-point logits inside the timed region).
`--dump-outputs DIR` writes what the last timed step returned (rank 0): DIR/logits.npy, float32 (B, 40), and with
several ranks DIR/logits_gathered.npy, the all-gathered (world * B, 40); with `--impl reference`, DIR/logits.npy
(n, 40) of that arm's last timed forward over its n clouds.  Clouds and checkpoint are seeded, so two builds of the
project run on identical inputs and their dumps can be compared array for array.
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B_PER_GPU, N_POINTS, K_NN, N_CLASS, SEED = 32, 1024, 20, 40, 1002
# the logits all-gather as a node of the replayed CUDA graph (0: host-launched after every replay)
GRAPH_ALLGATHER = os.environ.get("SVNET_GRAPH_ALLGATHER", "1") != "0"
METRIC = "SV-DGCNN clouds/sec (1024 pts, k=20)"
WORKLOAD = "SV-DGCNN binary ModelNet40 cls forward, B=32/GPU, N=1024, k=20, synthetic clouds + synthetic checkpoint"

# SURVEY.md 8(d): algorithmic bytes per cloud for the cls path (fp32 features, int32 indices)
F_L = [3, 62, 62, 127]
O_L = [62, 62, 127, 254]


def algorithmic_bytes_per_cloud(N=N_POINTS, k=K_NN):
    total = 0
    for f, o in zip(F_L, O_L):
        total += 2 * 4 * N * f + 2 * 4 * N * k + 4 * N * o
    total += 4 * N * sum(O_L) + 4 * (2 * 1022 + N_CLASS)
    return total


def edge_kernel_bytes_per_cloud(layer, N=N_POINTS, k=K_NN):
    """K2 of SURVEY 8(d): read point table + idx, write pooled output (+ the P|Q table it gathers)."""
    f, o = F_L[layer], O_L[layer]
    return 4 * N * f + 4 * N * k + 4 * N * o


def knn_kernel_bytes_per_cloud(layer, N=N_POINTS, k=K_NN):
    return 4 * N * F_L[layer] + 4 * N * k


def bench_config(world):
    """`config` of the JSON line -- the same object in both arms (ours / reference)."""
    return {"workload": WORKLOAD, "global_batch": world * B_PER_GPU, "n_points": N_POINTS, "k": K_NN,
            "parallelism": "batch-sharded x%d, all-gather of logits" % world,
            "l2": "GPU arm: flushed between steps (256 MiB memset, untimed)"}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_port_throughput(n_clouds, reps=1):
    """Time the oracle port (C + OpenMP, all host threads) on a bounded sample of the workload."""
    import numpy as np
    import torch
    from oracle import svnet_oracle as orc
    import svnet_b200 as sv
    from svnet_b200.synthetic import make_args, synthetic_clouds, synthetic_state_dict
    orc.build()
    with contextlib.redirect_stdout(io.StringIO()):
        net = sv.SV_DGCNN_CLS(make_args(k=K_NN, binary=True), N_CLASS)
    sd = synthetic_state_dict(net.state_dict(), seed=SEED)
    x = synthetic_clouds(n_clouds, N_POINTS, SEED).numpy()
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        y = orc.sv_dgcnn_cls(sd, x, K_NN)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    assert np.isfinite(y).all()
    return n_clouds / best, best, y


def dbg(msg):
    """stage marker on stderr (SVNET_BENCH_DEBUG=1): where a multi-rank run stops, if it does"""
    if os.environ.get("SVNET_BENCH_DEBUG", "0") != "0":
        print("[bench rank %s %.1fs] %s" % (os.environ.get("RANK", "0"), time.time() % 1000, msg), file=sys.stderr, flush=True)


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm must use all host threads it can
    (set before the oracle's OpenMP runtime is loaded)."""
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count())


def reference_model(device="cpu", kind="SV_DGCNN_CLS", k=K_NN, binary=True, ncls=N_CLASS, seed=SEED):
    """The unmodified reference model (oracle/_ref/models, models/sv_dgcnn_cls.py:22-82) with the
    same synthetic checkpoint as the CUDA arm."""
    import torch
    from oracle import reference
    from svnet_b200.synthetic import make_args, synthetic_state_dict
    ref = reference.load()
    with contextlib.redirect_stdout(io.StringIO()):
        net = getattr(ref, kind)(make_args(k=k, binary=binary), ncls)
    net.load_state_dict(synthetic_state_dict(net.state_dict(), seed=seed))
    return net.to(device).eval()


def reference_cpu_throughput(n_clouds, steps, warmup, budget_s=240.0):
    """Reference PyTorch forward on the host cores, all threads: `steps` timed forwards of `n_clouds`
    clouds each (the per-step sample shrinks only if the probe says the run would exceed `budget_s`)."""
    import torch
    from svnet_b200.synthetic import synthetic_clouds
    torch.set_num_threads(os.cpu_count())
    net = reference_model("cpu")
    with torch.no_grad():
        xp = synthetic_clouds(4, N_POINTS, SEED)
        net(xp)                                     # page in, thread pool
        t0 = time.perf_counter()
        net(xp)
        per_cloud = (time.perf_counter() - t0) / 4
        n = n_clouds
        while n > 4 and per_cloud * n * (steps + warmup) > budget_s:
            n //= 2
        x = synthetic_clouds(n, N_POINTS, SEED)
        per_step = []
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            y = net(x)
            dt = time.perf_counter() - t0
            if i >= warmup:
                per_step.append(dt)
    assert bool(torch.isfinite(y).all())
    return n, per_step, y.numpy()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    use_all_host_threads()
    cores = os.cpu_count()
    from oracle import reference
    if reference.available():
        n, per_step, y = reference_cpu_throughput(B_PER_GPU, args.steps, args.warmup)
        kind = "reference"
        what = ("%d clouds per step; unmodified reference forward (oracle/_ref/models, models/sv_dgcnn_cls.py:46-82), "
                "stock PyTorch CPU, torch.set_num_threads(%d)" % (n, cores))
    else:   # oracle/_ref not staged on this box: fall back to the C + OpenMP restatement (still a CPU arm)
        v0, _, _ = cpu_port_throughput(4)
        n = int(min(64, max(4, round(2.0 * v0 / 4) * 4)))
        per_step = []
        for i in range(args.warmup + args.steps):
            _, dt, y = cpu_port_throughput(n)
            if i >= args.warmup:
                per_step.append(dt)
        kind = "port"
        what = "%d clouds per step, oracle C port with OpenMP (oracle/_ref missing)" % n
    if args.dump_outputs:                 # the logits of the last timed forward: (n, 40) for its n clouds
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "logits.npy"), np.asarray(y, dtype=np.float32))
    ms = 1e3 * sum(per_step) / len(per_step)
    value = n / (ms / 1e3)
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "clouds/s", "n_gpus": args.gpus,
        "steps": len(per_step), "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(max(1, args.gpus)),
        "cpu_baseline": {"value": value, "unit": "clouds/s", "cores": cores, "kind": kind, "sample": what},
        "e2e": {"value": value, "unit": "clouds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out))


PSEG_BYTES_PER_CLOUD = 25.76e6     # SURVEY.md 8(d), N=2048, k=40


def extra_config(sv, kind, margs, ncls, seed, global_batch, n_points, world, rank, dev, timed, gather, steps=5):
    """One of BASELINE.json's other configs: `global_batch` clouds split contiguously over the ranks
    (strong scaling), CUDA-graph replay of the public forward, device-resident inputs, L2 flushed between steps; `gather`
    puts the NCCL all-gather of the per-point logits inside the timed region (cfg4)."""
    import torch
    import torch.distributed as dist
    from svnet_b200 import parallel
    from svnet_b200.synthetic import make_args, one_hot_labels, synthetic_clouds, synthetic_state_dict
    with contextlib.redirect_stdout(io.StringIO()):
        net = getattr(sv, kind)(make_args(**margs), ncls)
    net.load_state_dict(synthetic_state_dict(net.state_dict(), seed=seed))
    net = net.to(dev).eval()
    lo, hi = parallel.shard_bounds(global_batch, world, rank)
    per = hi - lo
    # the rank's shard only (a 128 x 2048-point batch is generated per rank, not replicated)
    x = synthetic_clouds(per, n_points, seed + 17 * rank).to(dev)
    ins = (x, one_hot_labels(global_batch)[lo:hi].to(dev)) if kind == "SV_DGCNN_PSEG" else (x,)
    out_all = None
    ag_ms = None

    with torch.no_grad():
        graphed = sv.GraphedForward(net, *ins)       # the forward as one CUDA-graph replay (the public fast path)

    def fwd():
        y = graphed(*ins)
        if gather and world > 1:
            dist.all_gather_into_tensor(out_all, y)  # host-launched behind the replay (kept out of the graph here)
        return y
    y = graphed(*ins)
    if gather and world > 1:
        assert per * world == global_batch
        out_all = torch.empty((global_batch,) + tuple(y.shape[1:]), dtype=y.dtype, device=dev)
    for _ in range(2):
        fwd()
    ms = timed(fwd, steps)
    if gather and world > 1:
        ag_ms = timed(lambda: dist.all_gather_into_tensor(out_all, y), steps)
    res = {"global_batch": global_batch, "per_rank_batch": per, "n_points": n_points, "k": margs["k"],
           "binary": margs["binary"], "model": kind, "scaling": "strong", "steps": steps,
           "ms_per_step": ms, "clouds_per_s": global_batch / (ms * 1e-3),
           "call": "svnet_b200.GraphedForward(net, shard) replay per rank" + (" + NCCL all-gather of the logits" if gather and world > 1 else "")}
    if gather:
        res["allgather_ms"] = ag_ms
        res["allgather_bytes_per_rank"] = int(y.numel() * 4) if world > 1 else 0
    bytes_per_cloud = PSEG_BYTES_PER_CLOUD if kind == "SV_DGCNN_PSEG" else algorithmic_bytes_per_cloud(n_points, margs["k"])
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        peak = 6650.0
    res["roofline_frac_whole_step"] = bytes_per_cloud * per / (ms * 1e-3) / 1e9 / peak
    del graphed, net, x, ins, out_all
    torch.cuda.empty_cache()
    return res


def gpu_eager_reference(dev, x_dev, steps=5):
    """BASELINE.md section 3: the unmodified reference modules on cuda (stock PyTorch eager, fp32, TF32
    off) on the same batch -- the GPU implementation the new kernels must beat."""
    import torch
    from oracle import reference
    if not reference.available():
        return {"unavailable": "oracle/_ref not staged"}
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    net = reference_model(dev)
    with torch.no_grad():
        for _ in range(3):
            net(x_dev)
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for e0, e1 in ev:
            e0.record()
            net(x_dev)
            e1.record()
        torch.cuda.synchronize()
    ms = sum(e0.elapsed_time(e1) for e0, e1 in ev) / steps
    peak_mb = torch.cuda.max_memory_allocated(dev) / 2 ** 20
    del net
    torch.cuda.empty_cache()
    return {"value": x_dev.shape[0] / (ms * 1e-3), "unit": "clouds/s", "ms_per_step": ms, "steps": steps,
            "what": "unmodified reference forward (oracle/_ref/models) on the same B200, stock PyTorch eager, fp32, TF32 off, "
                    "B=%d device-resident" % x_dev.shape[0], "max_memory_allocated_mib": peak_mb}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip extra.cfg3 / extra.cfg4 / gpu_eager_reference")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the logits of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 0)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import svnet_b200 as sv
    from svnet_b200 import _native as nv
    from svnet_b200.synthetic import make_args, synthetic_clouds, synthetic_state_dict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    nv.lib()  # fail loudly if the CUDA library is missing

    with contextlib.redirect_stdout(io.StringIO()):
        net = sv.SV_DGCNN_CLS(make_args(k=K_NN, binary=True), N_CLASS)
    net.load_state_dict(synthetic_state_dict(net.state_dict(), seed=SEED))
    net = net.to(dev).eval()
    B = B_PER_GPU
    # each rank gets its own shard of the global batch (weak scaling: 32 clouds per GPU)
    x_host = synthetic_clouds(B * world, N_POINTS, SEED)[rank * B:(rank + 1) * B].contiguous().pin_memory()
    x_dev = x_host.to(dev)
    y_host = torch.empty((B, N_CLASS), dtype=torch.float32).pin_memory()
    gathered = torch.empty((world * B, N_CLASS), dtype=torch.float32, device=dev) if world > 1 else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    # The step is the public inference call: svnet_b200.GraphedForward(net, example) captures the forward
    # once (CUDA graph; model(batch) runs through the whole-model C entry: two sub-batches on two streams plus auxiliary
    # streams for the chains that do not depend on the kNN graphs) and replays it per batch.
    in_graph = world > 1 and GRAPH_ALLGATHER
    dbg("model ready, capturing (all-gather in graph: %s)" % in_graph)
    fast = sv.GraphedForward(net, x_dev, epilogue=(lambda y: dist.all_gather_into_tensor(gathered, y)) if in_graph else None)

    def step(xin):
        y = fast(xin)
        if world > 1 and not in_graph:
            dist.all_gather_into_tensor(gathered, y)
        return y

    def step_eager(xin):
        y = net(xin)
        if world > 1:
            dist.all_gather_into_tensor(gathered, y)
        return y

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        for e0, e1 in ev:
            flush.zero_()          # flush L2 between steps (untimed)
            e0.record()
            fn()
            e1.record()
        barrier()
        total_ms = sum(e0.elapsed_time(e1) for e0, e1 in ev)
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps

    dbg("captured")
    with torch.no_grad():
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        for _ in range(args.warmup):
            step(x_dev)
        barrier()
        if rank == 0:
            t_wait = time.time()
            while not sampler.rows and time.time() - t_wait < 3.0:   # nvidia-smi start-up; rank 0 only, so no collective:
                net(x_dev)                                           # the eager forward (the graph may hold the all-gather)
            torch.cuda.synchronize()
            sampler.rows.clear()
        barrier()
        # ---- device-resident throughput (graph replay of the public call) ----
        dbg("warm-up done")
        last = {"steps": 0}

        def graph_step():
            last["logits"] = step(x_dev)
            last["steps"] += 1
        ms = timed(graph_step, args.steps)
        timed_steps = last["steps"]
        dbg("graph steps timed")
        if args.dump_outputs and rank == 0:
            # the replay's output buffer (and `gathered`) are overwritten by every later call: save them now
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            dump = {"logits": last["logits"]}
            if world > 1:
                dump["logits_gathered"] = gathered
            for name, t in dump.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), t.float().cpu().numpy())
        # ---- the same K steps eagerly, with the dominant C-ABI calls bracketed by CUDA events on their
        #      launch stream (events cannot bracket kernels inside a graph replay) ----
        from svnet_b200 import fused as sv_fused
        nv.PROFILE[0] = {"svnet_knn_ws", "svnet_svblock_edge_fwd"}
        nv.TIMED.clear()
        nv.ORDER.clear()
        l0 = nv.LAUNCHES[0]
        two_streams, native_fwd, side = sv_fused.CONCURRENT_HALVES, sv_fused.NATIVE_FORWARD, sv_fused.SIDE_STREAM
        sv_fused.CONCURRENT_HALVES = False       # one stream, 32 clouds per launch: un-overlapped kernel times
        sv_fused.NATIVE_FORWARD = False          # the stages as separate C-ABI calls from Python, so that events can bracket them
        sv_fused.SIDE_STREAM = False             # (model(x) otherwise makes the same calls inside svnet_model_forward)
        try:
            for _ in range(max(3, args.warmup)):          # the eager path has its own allocations to warm up
                step_eager(x_dev)
            nv.TIMED.clear()
            nv.ORDER.clear()
            l0 = nv.LAUNCHES[0]
            ms_eager = timed(lambda: step_eager(x_dev), args.steps)
        finally:
            sv_fused.CONCURRENT_HALVES, sv_fused.NATIVE_FORWARD, sv_fused.SIDE_STREAM = two_streams, native_fwd, side
        launches = (nv.LAUNCHES[0] - l0) // args.steps
        nv.PROFILE[0] = None
        clocks = sampler.stop() if rank == 0 else None
        per_call = {}
        for name, e0, e1 in nv.ORDER:
            per_call.setdefault(name, []).append(e0.elapsed_time(e1))

        # ---- end to end through the public API with host buffers ----
        def e2e_step():
            y = step(x_host)                     # pinned host -> static input (H2D) -> replay
            y_host.copy_(y, non_blocking=True)
        dbg("eager steps timed")
        for _ in range(3):
            e2e_step()
        ms_e2e = timed(e2e_step, args.steps)
        dbg("e2e timed")

        # ---- the other configs north_star names, batch-sharded over the ranks (strong scaling) ----
        extra = {}
        if not args.no_extra:
            extra["cfg3"] = extra_config(sv, "SV_DGCNN_CLS", dict(k=20, binary=False), 15, 1003, 256, 1024, world, rank, dev,
                                         timed, gather=False)
            extra["cfg4"] = extra_config(sv, "SV_DGCNN_PSEG", dict(k=40, binary=True), 50, 1004, 128, 2048, world, rank, dev,
                                         timed, gather=True)
            # BASELINE.json configs[4]: three points of the B x N throughput sweep of the binary classifier, each global
            # batch split over the ranks (the full sweep on one GPU: tools/sweep.py -> profiles/*_sweep_configs.json)
            extra["cfg5"] = [extra_config(sv, "SV_DGCNN_CLS", dict(k=20, binary=True), 40, 1005, gb, n, world, rank, dev, timed,
                                          gather=False, steps=3)
                             for gb, n in ((1024, 1024), (256, 2048), (64, 4096))]
            # the whole-model C entry (svnet_model_create / _forward, csrc/model.cu) on the headline workload: what a host
            # without Python model code gets -- eager (the call forks onto the handle's own streams and joins) and replayed from a
            # CUDA graph (same bits as `value`'s path)
            native = sv.NativeModel("SV_DGCNN_CLS", net.state_dict(), k=K_NN, binary=True, num_class=N_CLASS, device=dev)
            for _ in range(3):
                native(x_dev)
            ms_c = timed(lambda: native(x_dev), 10)
            gc_ = torch.cuda.CUDAGraph()
            torch.cuda.synchronize()
            with torch.cuda.graph(gc_):
                y_c = native(x_dev)
            ms_cg = timed(gc_.replay, 10)
            same = bool(torch.equal(y_c, net(x_dev)))
            extra["c_entry"] = {"call": "svnet_model_forward (two sub-batch streams + auxiliary streams inside the call), B=%d/GPU" % x_dev.shape[0],
                                "eager_ms_per_step": ms_c, "eager_clouds_per_s": world * x_dev.shape[0] / (ms_c * 1e-3),
                                "graph_ms_per_step": ms_cg, "graph_clouds_per_s": world * x_dev.shape[0] / (ms_cg * 1e-3),
                                "logits_identical_to_module": same}
            del gc_, native
        # ---- the unmodified reference modules on the same GPU (stock PyTorch eager, fp32, TF32 off) ----
        dbg("extras done")
        eager_ref = None
        if rank == 0 and not args.no_extra:
            eager_ref = gpu_eager_reference(dev, x_dev)
        dbg("eager reference done")

    # Teardown.  A CUDA graph that holds NCCL kernels keeps the communicator busy: destroy_process_group() then
    # never returns (seen at N = 2).  Drop the graph first; ranks other than 0 are done here, rank 0 prints its line
    # and every rank leaves through finish() (which skips the communicator teardown in that case).
    kernels_per_replay = fast.kernels_per_replay
    fast = None
    import gc
    gc.collect()
    torch.cuda.synchronize()

    def finish():
        sys.stdout.flush()
        sys.stderr.flush()
        if world > 1:
            if in_graph:
                os._exit(0)
            dist.destroy_process_group()
    if rank != 0:
        return finish()

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"

    # dominant kernel = the C-ABI call with the largest share of the step; per launch, 4 knn + 3 edge per step
    # the bracketed eager pass runs on one stream: one launch per layer, B clouds per launch
    halves = 1
    Bl = B // halves

    def per_layer(name, n_layers):
        v = per_call.get(name, [])
        n = n_layers * halves
        return [sum(sum(v[i + h * n_layers::n]) for h in range(halves)) / max(1, sum(len(v[i + h * n_layers::n]) for h in range(halves)))
                for i in range(n_layers)]
    knn_ms = per_layer("svnet_knn_ws", 4)
    edge_ms = per_layer("svnet_svblock_edge_fwd", 3)
    # Candidates for "the dominant kernel" are single kernels: each edge layer is one kernel launch; a kNN call is
    # three kernels (pack, tcgen05 score, finish -- the largest of them is below the layer-4 edge kernel, see the ncu
    # launch list under profiles/), so the calls are listed in `calls` but the roofline is quoted for a kernel.
    calls = [("svnet_knn[layer%d]" % (i + 1), knn_ms[i], knn_kernel_bytes_per_cloud(i) * Bl) for i in range(4)]
    cand = [("svnet_svblock_edge_fwd[layer%d]" % (i + 2), edge_ms[i], edge_kernel_bytes_per_cloud(i + 1) * Bl) for i in range(3)]
    dom = max(cand, key=lambda c: c[1])
    cand = calls + cand
    achieved = dom[2] / (dom[1] * 1e-3) / 1e9
    traffic = None
    try:  # dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed ncu --set full capture
        traffic = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json"))).get(dom[0])
    except Exception:
        pass
    limiter = None
    try:  # what the same capture says limits that kernel (issue slots, not DRAM: DESIGN.md section 4)
        limiter = json.load(open(os.path.join(ROOT, "profiles", "limiters.json"))).get(dom[0])
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": dom[0], "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                "frac": achieved / hbm_peak, "traffic": traffic, "peak_source": peak_src,
                "limiter_ncu": limiter,
                "kernel_ms": dom[1], "algorithmic_bytes_per_launch": dom[2],
                "clouds_per_launch": Bl,
                "timed": "eager single-stream pass of the same %d steps (events cannot bracket kernels inside the graph replay)" % args.steps,
                "eager_ms_per_step": ms_eager,
                "step_share": {c[0]: halves * c[1] / ms_eager for c in cand},
                "whole_step": {"algorithmic_bytes": algorithmic_bytes_per_cloud() * B,
                               "achieved": algorithmic_bytes_per_cloud() * B / (ms * 1e-3) / 1e9,
                               "frac": algorithmic_bytes_per_cloud() * B / (ms * 1e-3) / 1e9 / hbm_peak}}

    cpu = None
    if not args.no_cpu_baseline and world == 1:             # rank 0 at N = 1 only (bench contract)
        use_all_host_threads()
        from oracle import reference
        v, dt, _ = cpu_port_throughput(4)                   # probe, then a sample worth ~5 s of CPU work
        n_cpu = int(min(128, max(4, round(5.0 * v / 4) * 4)))
        v, dt, _ = cpu_port_throughput(n_cpu)
        port = {"value": v, "unit": "clouds/s", "kind": "port",
                "sample": "%d clouds of the same workload (N=1024, k=20), oracle C port with OpenMP, %.1f s" % (n_cpu, dt)}
        if reference.available():
            n_ref, per_step, _ = reference_cpu_throughput(B_PER_GPU, 2, 1, budget_s=45.0)
            best = min(per_step)
            cpu = {"value": n_ref / best, "unit": "clouds/s", "cores": os.cpu_count(), "kind": "reference",
                   "sample": "%d clouds of the same workload per forward, best of %d after 1 warm-up (%.1f s each); unmodified "
                             "reference forward (oracle/_ref/models), stock PyTorch CPU, all host threads" % (n_ref, len(per_step), best),
                   "port": port}
        else:
            cpu = dict(port, cores=os.cpu_count())

    out = {
        "metric": METRIC, "value": world * B / (ms * 1e-3), "unit": "clouds/s", "n_gpus": world, "steps": timed_steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (+u32 XNOR/popcount for the binarised linears; exact bf16x3 tcgen05 filter in front of the fp32 kNN)", "data": "synthetic",
        "config": bench_config(world),
        "call": "svnet_b200.GraphedForward(net, batch): CUDA-graph replay of model(batch); the forward is sequenced by svnet_model_forward (two sub-batches of 16 clouds on two streams, graph-independent chains on auxiliary streams)"
                + ("; the logits all-gather is captured in the same graph" if (world > 1 and GRAPH_ALLGATHER) else ""),
        "clocks": clocks,
        "e2e": {"value": world * B / (ms_e2e * 1e-3), "unit": "clouds/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": y_host.numel() * 4},
        # kernels of libsvnet_b200.so inside the timed region: K replays of the captured forward (four
        # sub-batches); the eager single-stream pass used for the per-kernel events launches `eager` per step
        "gpu_launches": kernels_per_replay * timed_steps,
        "gpu_launches_per_step": {"graph_replay": kernels_per_replay, "eager_single_stream": launches},
        "roofline": roofline,
        "cpu_baseline": cpu,
        "gpu_eager_reference": eager_ref,
        "extra": extra,
    }
    print(json.dumps(out))
    finish()


if __name__ == "__main__":
    main()
