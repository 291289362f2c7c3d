"""Multi-GPU tests (skipped below 2 visible GPUs): the reference's own
multi-GPU mechanism nn.DataParallel (main_cls_dgcnn.py:125) over two devices, and the batch-sharded
one-process-per-GPU path with the NCCL all-gather against the unsharded forward."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import svnet_oracle as orc
from tests.util import assert_close, quiet, t2n
from svnet_b200.synthetic import make_args, synthetic_clouds, synthetic_state_dict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")]


def test_data_parallel_two_devices_matches_oracle_and_packs_once():
    import svnet_b200 as sv
    from svnet_b200.sv_layers import _Cached
    net = quiet(sv.SV_DGCNN_CLS, make_args(k=8, binary=True), 40)
    sd = synthetic_state_dict(net.state_dict(), seed=5)
    net.load_state_dict(sd)
    model = torch.nn.DataParallel(net.to("cuda:0"), device_ids=[0, 1]).eval()
    x = synthetic_clouds(4, 128, 5).to("cuda:0")
    with torch.no_grad():
        y = model(x)
        builds = _Cached.BUILDS
        y2 = model(x)                     # fresh replicas, fresh parameter copies: must hit the source-keyed cache
    assert _Cached.BUILDS == builds, "weights were re-packed on the second DataParallel forward"
    assert torch.equal(y, y2)
    with torch.no_grad():
        y_single = net(x)
    assert torch.equal(y, y_single)       # each cloud's logits do not depend on the device or its batch-mates
    rec = {}
    ref = orc.sv_dgcnn_cls(sd, t2n(x), 8, rec=rec)
    with torch.no_grad():
        yf = net(x, forced_idx=[torch.from_numpy(i).to(torch.int32).cuda() for i in rec["idx"]])
    assert_close(t2n(yf), ref, what="forward vs oracle (kNN graphs forced)")


def test_sharded_equals_unsharded_bit_for_bit_nccl():
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29611", os.path.join(ROOT, "tools", "sharded_check.py")]
    p = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    line = [l for l in p.stdout.splitlines() if l.startswith("{")][-1]
    res = json.loads(line)
    assert res["world"] == 2
    assert all(v["bit_identical_on_every_rank"] for v in res.values() if isinstance(v, dict)), res


def test_c_abi_allgather_on_raw_nccl_communicators():
    """svnet_allgather_logits (the C-ABI face of the path's one collective) on ncclComm_t handles made with
    ncclCommInitAll, one thread driving both devices inside a group call."""
    import ctypes
    from svnet_b200 import _native as nv
    lib = nv.lib()
    nccl = ctypes.CDLL(None)                         # torch has NCCL loaded; same symbols the library resolves
    if not hasattr(nccl, "ncclCommInitAll"):
        nccl = ctypes.CDLL("libnccl.so.2")
    comms = (ctypes.c_void_p * 2)()
    devs = (ctypes.c_int * 2)(0, 1)
    assert nccl.ncclCommInitAll(comms, 2, devs) == 0
    count = 5 * 40
    local = [torch.arange(count, dtype=torch.float32, device="cuda:%d" % r) + 1000.0 * r for r in range(2)]
    out = [torch.zeros(2 * count, dtype=torch.float32, device="cuda:%d" % r) for r in range(2)]
    assert nccl.ncclGroupStart() == 0
    for r in range(2):
        with torch.cuda.device(r):
            rc = lib.svnet_allgather_logits(ctypes.c_void_p(comms[r]), ctypes.c_void_p(local[r].data_ptr()),
                                            ctypes.c_void_p(out[r].data_ptr()), ctypes.c_size_t(count),
                                            ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
            assert rc == 0, lib.svnet_last_error().decode()
    assert nccl.ncclGroupEnd() == 0
    for r in range(2):
        torch.cuda.synchronize(r)
    want = torch.cat([t.cpu() for t in local])
    for r in range(2):
        assert torch.equal(out[r].cpu(), want)
    for r in range(2):
        nccl.ncclCommDestroy(ctypes.c_void_p(comms[r]))


def test_model_on_second_device_while_first_is_current():
    """A model moved with .to('cuda:1') while cuda:0 is the current device must launch on cuda:1 (scratch and stream
    follow the input's device) and give the same bits as on cuda:0."""
    import svnet_b200 as sv
    net = quiet(sv.SV_DGCNN_CLS, make_args(k=20, binary=True), 40)
    net.load_state_dict(synthetic_state_dict(net.state_dict(), seed=11))
    x = synthetic_clouds(2, 256, 11)
    torch.cuda.set_device(0)
    with torch.no_grad():
        y0 = net.to("cuda:0").eval()(x.to("cuda:0")).cpu()
        y1 = net.to("cuda:1").eval()(x.to("cuda:1")).cpu()
    assert torch.cuda.current_device() == 0
    assert torch.equal(y0, y1)
