"""Edge layers, the full-precision vector linear and the gate kernels against float64 restatements of the reference.

Every state dict elsewhere in the suite draws BatchNorm weights and binary scales from U(0.5, 1.5): the pre-activation
chain leaky(bn1(linear1(u))) is then increasing, and the "min" half of the pooled-max epilogues (the edge kernels keep
the largest and the smallest pre-activation over the k edges and take the larger activation) never decides a result.
`signed_state_dict` negates about half of every BatchNorm weight (two channels exactly 0) and a quarter of the binary
linear scales, so all four sign combinations of (scale, gamma) occur.

The float64 restatement (`edge_layer64`, `xyz_layer64`) is pinned to the reference's recorded layer outputs on the CPU
(`test_fp64_restatement_matches_reference_layers`); the GPU tests compare each kernel with it:

    pooled s:  |s - s64| <= RHO_S * |a1_o| * S + 4 ulp(max(|s64|, |c1_o|)),   S = max_e sum_k |W_ok u_ek|

(a1, c1: bn1's folded affine; the ulp term is the rounding of the epilogue's float chain).  Bars were set from runs on
an NVIDIA B200 (1000 W power limit): each is at most 4x the largest value measured there, and the measured values are
printed (`pytest -s`).
"""
import contextlib
import math
import os

import numpy as np
import pytest
import torch

from oracle import svnet_oracle as orc
from tests.util import assert_close, golden, golden_state_dict, quiet, t2n
from svnet_b200.synthetic import _key_generator, make_args, synthetic_clouds, synthetic_state_dict

DEV = "cuda"
BN_EPS = 1e-5

# bars, measured on a B200 (see the module docstring), each at most 4x the largest value measured there.  Edge kernels:
# (model-like or graph edge-case inputs, per-channel scales 2^-10 .. 2^10) per kernel.  With the scaled inputs the tensor
# cores' fp32 accumulation loses more than the sequential fp32 chain (measured rho 1.6e-6 against 5.4e-7); the bars must
# stay below 2^-17, and the model-like bar of the tensor-core kernel is what catches a dropped bf16 plane product (5.4e-6).
RHO_S = {"fp_tc": (1.0e-6, 6.4e-6), "fp_fast": (1.4e-6, 2.1e-6), "generic": (1.4e-6, 2.1e-6)}
RHO_S_RMS = {"fp_tc": (5.7e-8, 8.0e-7), "fp_fast": (5.6e-8, 1.0e-7), "generic": (5.6e-8, 1.0e-7)}
TC_OVER_CHAIN = 8.0              # rho of the tensor-core kernel over the fp32 chain's on the same case (measured <= 4.3)
TAU_V = 1.5e-5                   # pooled v: |v - v64| <= TAU_V * max over points of |v64| (per output channel)
RHO_C4 = 1.6e-6                  # fp-weight vector linear, float4 table: |t - t64| <= RHO_C4 * sum_d |W_cd v_xd|
TAU_VBN = 2.5e-6                 # fp-weight vector linear + VectorBN + gate, relative to the channel's largest |out|
GATE_ABS = 2.9e-7                # gate kernels, absolute (the gate is a sigmoid in (0, 1))
GATE_OFFSET_ABS = 7e-6           # gate_edge on s = 100 + noise (the fp32 reference itself is off by up to 1.6e-4 there)


# ------------------------------------------------------------------------------------------------
# A. helpers
# ------------------------------------------------------------------------------------------------
def signed_state_dict(template, seed):
    """`synthetic_state_dict` with negative parameters: about half the channels of every BatchNorm weight negated and two
    of them exactly 0; in binary blocks about a quarter of `linear1.scale` / `linear2.scale` negated on another
    pattern.  Seeded per key like the source; running_var stays positive."""
    sd = synthetic_state_dict(template, seed=seed)
    for key in list(sd):
        parent, leaf = key.rsplit(".", 1) if "." in key else ("", key)
        t = sd[key].clone()
        if leaf == "weight" and (parent + ".running_mean") in sd:
            g = _key_generator(seed + 7919, key)
            t = torch.where(torch.rand(t.shape, generator=g) < 0.5, -t, t)
            t[torch.randperm(t.numel(), generator=g)[:2]] = 0.0
        elif leaf == "scale" and parent.rsplit(".", 1)[-1] in ("linear1", "linear2"):
            g = _key_generator(seed + 104729, key)
            t = torch.where(torch.rand(t.shape, generator=g) < 0.25, -t, t)
        else:
            continue
        sd[key] = t.contiguous()
    return sd


def block_params(sd, prefix, dev):
    """The parameters of one block (``prefix`` = 'conv2.', ...) as float64 tensors on ``dev``."""
    return {k[len(prefix):]: torch.as_tensor(v).double().to(dev) for k, v in sd.items()
            if k.startswith(prefix) and not k.endswith("num_batches_tracked")}


def _bn64(P, name):
    a = P[name + ".weight"] / torch.sqrt(P[name + ".running_var"] + BN_EPS)
    return a, P[name + ".bias"] - P[name + ".running_mean"] * a


def _v2s64(P, v, key="v2s.linear"):
    """Vector2Scalar (sv_layers.py:111-129): v (..., 3, C) -> (..., 3C) with s[3d + m] = sum_x v[x][d] z[x][m]."""
    W = P[key + ".weight"]
    binary = (key + ".scale") in P
    z = torch.einsum("...xd,md->...xm", v, torch.sign(W) if binary else W)
    if binary:
        z = z * P[key + ".scale"].reshape(3)
    q = torch.einsum("...xd,...xm->...dm", v, z)
    return q.reshape(q.shape[:-2] + (-1,))


def svblock_edges64(P, s_e, v_e):
    """SVBlock.forward (sv_layers.py:172-196) + svpool (max over k for s, mean for v) of one cloud's edge features
    s_e (N, k, Cs), v_e (N, k, 3, Cv), float64.  Also returns, per (point, channel), the operand scale S and whether
    the edge with the smallest pre-activation decides the pooled value."""
    binary = "linear1.beta" in P
    N, k = s_e.shape[:2]
    mean = s_e.reshape(N * k, -1).mean(0)                                            # gate on the edge mean, :179-183
    gate = torch.sigmoid(P["gate.2.weight"] @ torch.relu(P["gate.0.weight"] @ mean))
    u = torch.cat([s_e, _v2s64(P, v_e)], dim=-1)                                     # :185-186
    W1 = P["linear1.weight"]
    if binary:                                                                        # sign(u + beta), sign(0) = 0
        act = torch.sign(u + P["linear1.beta"].reshape(-1))
        W = torch.sign(W1) * P["linear1.scale"].reshape(-1, 1)
    else:
        act, W = u, W1
    y = act @ W.t()                                                                   # (N, k, Cout)
    S = (act.abs() @ W.abs().t()).amax(1)
    a1, c1 = _bn64(P, "bn1")
    t = y * a1 + c1
    o = torch.where(t > 0, t, 0.2 * t)
    o_hi = torch.gather(o, 1, y.argmax(1, keepdim=True))[:, 0]
    o_lo = torch.gather(o, 1, y.argmin(1, keepdim=True))[:, 0]
    W2 = P["linear2.weight"]
    if "linear2.scale" in P:
        W2 = torch.sign(W2) * P["linear2.scale"].reshape(-1, 1)
    w = torch.einsum("nkxd,od->nkxo", v_e, W2)                                        # :192
    n = torch.sqrt((w * w).sum(2, keepdim=True)) + 1e-6
    a2, c2 = _bn64(P, "bn2.bn")
    w = w / n * (n * a2 + c2)                                                         # VectorBN, :193
    return {"s": o.amax(1), "v": w.mean(1) * gate, "S": S, "min_wins": o_lo > o_hi, "sign": act if binary else None,
            "gate": gate}


def _cat_clouds(parts):
    return {key: (torch.cat([p[key] for p in parts]) if parts[0][key] is not None else None) for key in parts[0]}


def edge_layer64(P, s, v, idx):
    """get_graph_feature_sv (sv_util.py:106-114) + SVBlock + svpool for edge layers 2..4, float64, one cloud at a time.
    s (B, N, Cs), v (B, N, 3, Cv), idx (B, N, k) -> dict of (B*N, ...) tensors."""
    parts = []
    for b in range(s.shape[0]):
        sb, vb, ib = s[b].double(), v[b].double(), idx[b].long()
        sj, vj = sb[ib], vb[ib]                                                       # (N, k, Cs), (N, k, 3, Cv)
        si, vi = sb[:, None].expand_as(sj), vb[:, None].expand_as(vj)
        parts.append(svblock_edges64(P, torch.cat([sj - si, si], -1), torch.cat([vj - vi, vi], -1)))
    return _cat_clouds(parts)


def xyz_layer64(P, P_init, xyz, idx):
    """Layer 1: get_graph_feature (nv = 2, sv_util.py:28-62) + init_scalar + SVBlock + svpool, float64.
    xyz (B, N, 3), idx (B, N, k)."""
    parts = []
    for b in range(xyz.shape[0]):
        xb, ib = xyz[b].double(), idx[b].long()
        xj = xb[ib]
        xi = xb[:, None].expand_as(xj)
        v_e = torch.stack([xj - xi, xi], -1)                                          # (N, k, 3, 2)
        parts.append(svblock_edges64(P, _v2s64(P_init, v_e, "linear"), v_e))
    return _cat_clouds(parts)


def kernels_launched(fn):
    """Names of the CUDA kernels ``fn()`` launches, from a torch.profiler trace."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def ran(names, kernel):
    return any(kernel + "<" in n or n.endswith(kernel) or kernel + "(" in n for n in names)


@contextlib.contextmanager
def env(**kv):
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update({k: str(v) for k, v in kv.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


# the edge-kernel variants of a layer and the switches that select them
FP_KERNELS = {"fp_tc": ({}, "edge_fp_tc_kernel"), "fp_fast": ({"SVNET_EDGE_FP_TC": "0"}, "edge_fp_fast_kernel"),
              "generic": ({"SVNET_EDGE_GENERIC": "1"}, "svblock_edge_kernel")}
BIN_KERNELS = {"bin_tc": ({}, "edge_bin_tc_kernel"), "bin_fast": ({"SVNET_EDGE_TC": "0"}, "edge_bin_fast_kernel"),
               "generic": ({"SVNET_EDGE_GENERIC": "1"}, "svblock_edge_kernel")}


def _ulp(x):
    x = np.abs(np.asarray(x, dtype=np.float32))
    return (np.nextafter(x, np.float32(np.inf)) - x).astype(np.float64)


def s_error(s, ref, a1, c1):
    """Normalised error of pooled scalars: (|s - s64| - 4 ulp(max(|s64|, |c1|))) / (|a1| S), per (point, channel);
    channels with a1 == 0 carry only the ulp term and must be within it."""
    s = np.asarray(s, dtype=np.float64)
    s64, S = t2n(ref["s"]), t2n(ref["S"])
    err = np.abs(s - s64)
    floor = 4 * _ulp(np.maximum(np.abs(s64), np.abs(c1)))
    scale = np.abs(a1)[None, :] * S
    assert (err[:, a1 == 0] <= floor[:, a1 == 0]).all(), "channels with bn1 weight 0 off by more than rounding"
    return np.where(scale > 0, np.maximum(err - floor, 0) / np.where(scale > 0, scale, 1), 0.0)


def v_error(v, ref):
    v64 = t2n(ref["v"])
    ch = np.abs(v64).max(axis=(0, 1), keepdims=True)
    return np.abs(np.asarray(v, dtype=np.float64) - v64) / np.maximum(ch, 1e-30)


def _unpack(words, K):
    """(rows, Kw) int32 sign / mask words -> (rows, K) uint8 bits"""
    w = words.view(np.uint32)
    bits = ((w[:, :, None] >> np.arange(32, dtype=np.uint32)[None, None, :]) & 1).astype(np.uint8)
    return bits.reshape(w.shape[0], -1)[:, :K]


def report(tag, **vals):
    print("[fp64] %s %s" % (tag, " ".join("%s=%.3g" % kv for kv in vals.items())))


# ------------------------------------------------------------------------------------------------
# A. the float64 restatement against the reference's recorded layer outputs (CPU)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["dgcnn_cls_fp", "dgcnn_cls_bin", "dgcnn_pseg_fp"])
def test_fp64_restatement_matches_reference_layers(name):
    """Each edge layer of the restatement, teacher-forced with the reference's pool{l-1} and idx{l}, reproduces the
    reference's recorded pooled outputs within 1e-5; binary layers' sign planes equal the oracle's."""
    g = golden(name)
    sd = golden_state_dict(g)
    xyz = torch.from_numpy(np.ascontiguousarray(np.transpose(g["x"], (0, 2, 1))))
    for li in range(4):
        P = block_params(sd, "conv%d." % (li + 1), "cpu")
        idx = torch.from_numpy(g["idx%d" % li])
        if li == 0:
            ref = xyz_layer64(P, block_params(sd, "init_scalar.", "cpu"), xyz, idx)
        else:
            s_in, v_in = torch.from_numpy(g["pool%d_s" % (li - 1)]), torch.from_numpy(g["pool%d_v" % (li - 1)])
            ref = edge_layer64(P, s_in, v_in, idx)
            if ref["sign"] is not None:
                sf, vf = orc.graph_feature_sv(s_in.numpy(), v_in.numpy(), idx.numpy())
                Po = orc.Params(sd).sub("conv%d" % (li + 1))
                u = np.concatenate([sf, orc.p_v2s(Po.sub("v2s"), vf)], axis=-1)
                sign = orc.sign_plane(u, Po.get("linear1.beta")).reshape(ref["sign"].shape)
                assert (t2n(ref["sign"]) == sign).all(), "%s layer %d sign plane" % (name, li + 1)
        B, N = idx.shape[:2]
        assert_close(t2n(ref["s"]).reshape(B, N, -1), g["pool%d_s" % li], rtol=1e-5, atol=1e-5, what="%s s%d" % (name, li))
        assert_close(t2n(ref["v"]).reshape(g["pool%d_v" % li].shape), g["pool%d_v" % li], rtol=1e-5, atol=1e-5,
                     what="%s v%d" % (name, li))


def test_signed_state_dict_has_all_sign_combinations():
    import svnet_b200 as sv
    blk = quiet(sv.SVBlock, (64, 20), (32, 10), True)
    sd = signed_state_dict(blk.state_dict(), 5)
    base = synthetic_state_dict(blk.state_dict(), seed=5)
    for key in sd:
        if not key.endswith(("bn1.weight", "bn.weight", "linear1.scale", "linear2.scale")):
            assert torch.equal(sd[key], base[key]), key
    assert (sd["bn1.running_var"] > 0).all()
    for key in ("bn1.weight", "bn2.bn.weight"):
        w = sd[key]
        assert int((w == 0).sum()) == 2 and (w < 0).any() and (w > 0).any(), key
    sc, gm = sd["linear1.scale"].reshape(-1), sd["bn1.weight"]
    combos = {(bool(a > 0), bool(b > 0)) for a, b in zip(sc, gm) if b != 0}
    assert len(combos) == 4, combos


# ------------------------------------------------------------------------------------------------
# B. edge_fp_tc against float64: three kernels on the same layer, graph and inputs
# ------------------------------------------------------------------------------------------------
def _inputs(regime, B, N, Cs, Cv, k, seed):
    g = torch.Generator().manual_seed(seed)
    s = torch.randn(B, N, Cs, generator=g)
    v = torch.randn(B, N, 3, Cv, generator=g) * 0.5
    if regime == "scaled":                       # per-channel scales 2^-10 .. 2^10
        s = s * torch.exp2(torch.randint(-10, 11, (Cs,), generator=g).float())
        v = v * torch.exp2(torch.randint(-10, 11, (Cv,), generator=g).float())
    idx = torch.randint(0, N, (B, N, k), generator=g, dtype=torch.int32)
    idx[:, :, 0] = torch.arange(N, dtype=torch.int32)                  # the self edge first, as kNN returns it
    if regime == "graph":
        idx[:, ::5, :] = torch.randint(0, N, (B, 1, 1), generator=g, dtype=torch.int32)     # one neighbour k times
        idx[:, 1::5, 0] = 0
        idx[:, 2::5, k - 1] = N - 1
        idx[:, 3::5, 1:] = torch.tensor([0, N - 1], dtype=torch.int32).repeat(k)[:k - 1]
    return s, v, idx


def _edge_block(Cs, Cv, Cout, Cvo, binary, seed):
    import svnet_b200 as sv
    blk = quiet(sv.SVBlock, (2 * Cs, 2 * Cv), (Cout, Cvo), binary)
    sd = signed_state_dict(blk.state_dict(), seed)
    blk.load_state_dict(sd)
    return blk.to(DEV).eval(), sd


def run_edge_layer(blk, s, v, idx, switches):
    """fused.sv_edge_layer on strided slices of NaN-filled svcat-like tables; returns (s_out, v_out, kernel names,
    untouched) where ``untouched`` says the output table's other columns are still NaN."""
    from svnet_b200 import fused
    B, N, Cs = s.shape
    Cv = v.shape[-1]
    Cout, Cvo = blk.out_dims
    R = B * N
    s_tab = torch.full((R, Cs + 6), float("nan"), device=DEV)
    v_tab = torch.full((R, 3, Cv + 5), float("nan"), device=DEV)
    s_tab[:, 2:2 + Cs] = s.reshape(R, Cs).to(DEV)
    v_tab[:, :, 3:3 + Cv] = v.reshape(R, 3, Cv).to(DEV)
    so_tab = torch.full((R, Cout + 36), float("nan"), device=DEV)
    vo_tab = torch.full((R, 3, Cvo + 11), float("nan"), device=DEV)
    s_out, v_out = so_tab[:, 32:32 + Cout], vo_tab[:, :, 10:10 + Cvo]
    with env(**switches), torch.no_grad():
        names = kernels_launched(lambda: fused.sv_edge_layer(s_tab[:, 2:2 + Cs], v_tab[:, :, 3:3 + Cv], B, N, idx.shape[-1],
                                                             blk, s_out, v_out, idx32=idx.to(DEV)))
    got_s, got_v = t2n(s_out), t2n(v_out)
    so_tab[:, 32:32 + Cout] = 0.0
    vo_tab[:, :, 10:10 + Cvo] = 0.0
    untouched = bool(torch.isnan(so_tab).sum() == R * 36 and torch.isnan(vo_tab).sum() == R * 3 * 11)
    return got_s, got_v, names, untouched


FP_SHAPES = [(32, 10, 32, 10), (32, 10, 64, 21), (64, 21, 128, 42)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", FP_SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("B,N", [(4, 1024), (3, 1021), (2, 20), (1, 37)])
@pytest.mark.parametrize("regime", ["model", "scaled", "graph"])
def test_edge_fp_tc_against_float64(shape, B, N, regime):
    """The full-precision tensor-core edge kernel, the fp32 CUDA-core kernel and the generic kernel against float64,
    with negative BatchNorm weights: pooled s within RHO_S * |a1| * S (+ rounding), pooled v within TAU_V; the
    min branch decides >= 10 % of the pooled scalars; columns outside the output slice untouched."""
    Cs, Cv, Cout, Cvo = shape
    k = 20
    blk, sd = _edge_block(Cs, Cv, Cout, Cvo, False, 300 + Cout)
    s, v, idx = _inputs(regime, B, N, Cs, Cv, k, 17 + N + Cout)
    ref = edge_layer64(block_params(sd, "", DEV), s.to(DEV), v.to(DEV), idx.to(DEV))
    a1, c1 = (t2n(t) for t in blk.bn1_folded())
    assert float(ref["min_wins"].double().mean()) >= 0.10, "the min branch must decide >= 10 % of the outputs"
    rho = {}
    for name, (switches, kernel) in FP_KERNELS.items():
        got_s, got_v, names, untouched = run_edge_layer(blk, s, v, idx, switches)
        assert ran(names, kernel), (name, sorted(set(names)))
        assert untouched, name + ": wrote outside its output columns"
        e = s_error(got_s, ref, a1, c1)
        ev = v_error(got_v.reshape(ref["v"].shape), ref)
        rho[name] = float(e.max())
        report("edge %s %s B=%d N=%d %s" % (name, "x".join(map(str, shape)), B, N, regime), rho=e.max(),
               rho_rms=math.sqrt(float((e ** 2).mean())), tau_v=ev.max())
        col = 1 if regime == "scaled" else 0
        assert e.max() <= RHO_S[name][col], (name, e.max())
        assert math.sqrt(float((e ** 2).mean())) <= RHO_S_RMS[name][col], name
        assert ev.max() <= TAU_V, (name, ev.max())
    # the tensor cores do what the fp32 chain does, to a small factor
    assert rho["fp_tc"] <= TC_OVER_CHAIN * max(rho["fp_fast"], 2.0 ** -24), rho


# ------------------------------------------------------------------------------------------------
# C. negative parameters through every edge kernel, teacher-forced on the oracle's layer inputs and graphs
# ------------------------------------------------------------------------------------------------
_ORACLE = {}


def _trunk_case(kind, binary, k, B, N, seed):
    """(net, state dict, x, oracle record of the trunk) for a signed checkpoint; the oracle's record is cached."""
    import svnet_b200 as sv
    key = (kind, binary, k, B, N, seed)
    cls = sv.SV_DGCNN_PSEG if kind == "pseg" else sv.SV_DGCNN_CLS
    net = quiet(cls, make_args(k=k, binary=binary), 50 if kind == "pseg" else 40)
    sd = signed_state_dict(net.state_dict(), seed)
    net.load_state_dict(sd)
    net = net.to(DEV).eval()
    x = synthetic_clouds(B, N, seed, rotate=True)
    if key not in _ORACLE:
        rec = {"idx": [], "pools": []}
        orc._dgcnn_trunk(orc.Params(sd), x.numpy(), k, None, rec)
        _ORACLE[key] = rec
    return net, sd, x, _ORACLE[key]


def _teacher_forced(net, kind, x, rec_o, switches):
    B, _, N = x.shape
    teacher = [(torch.from_numpy(s).to(DEV).view(B * N, -1), torch.from_numpy(v).to(DEV).view(B * N, 3, -1))
               for (s, v) in rec_o["pools"][:3]]
    rec = {"teacher": teacher, "want_taps": True}
    fi = [torch.from_numpy(i).to(torch.int32).to(DEV) for i in rec_o["idx"]]
    extra = ()
    if kind == "pseg":
        from svnet_b200.synthetic import one_hot_labels
        extra = (one_hot_labels(B).to(DEV),)
    with env(**switches), torch.no_grad():
        names = kernels_launched(lambda: net(x.to(DEV), *extra, forced_idx=fi, record=rec))
    return rec, names


TRUNKS = [("cls", True, 20, 2, 512, "bin_tc"), ("cls", True, 20, 2, 512, "bin_fast"), ("cls", True, 20, 2, 512, "generic"),
          ("pseg", True, 40, 1, 1024, "bin_tc"), ("pseg", True, 40, 1, 1024, "bin_fast"), ("pseg", True, 40, 1, 1024, "generic"),
          ("cls", True, 12, 2, 300, "generic"), ("cls", False, 20, 2, 512, "fp_tc"), ("cls", False, 20, 2, 512, "fp_fast"),
          ("cls", False, 20, 2, 512, "generic")]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,binary,k,B,N,kernel", TRUNKS, ids=lambda p: str(p))
def test_edge_kernels_negative_parameters_teacher_forced(kind, binary, k, B, N, kernel):
    """Edge layers 1..4 on a signed checkpoint, each fed the oracle's input and graph: layer 1 (edge_xyz) and binary
    layers bit-identical to the oracle, binary sign bits equal to the oracle's sign planes, fp layers within the
    bound of test_edge_fp_tc_against_float64, v within TAU_V of the float64 restatement."""
    net, sd, x, rec_o = _trunk_case(kind, binary, k, B, N, 4000 + k + (0 if binary else 1))
    switches, want = (BIN_KERNELS if binary else FP_KERNELS)[kernel]
    rec, names = _teacher_forced(net, kind, x, rec_o, switches)
    assert ran(names, want), sorted(set(names))
    assert ran(names, "edge_xyz_fast_kernel"), sorted(set(names))
    xyz = torch.from_numpy(np.ascontiguousarray(np.transpose(x.numpy(), (0, 2, 1)))).to(DEV)
    so = vo = 0
    for li, (o_s, o_v) in enumerate(rec_o["pools"]):
        cs, cv = o_s.shape[-1], o_v.shape[-1]
        got_s = t2n(rec["s_cat"][:, so:so + cs])
        got_v = t2n(rec["v_cat"][:, :, vo:vo + cv])
        P = block_params(sd, "conv%d." % (li + 1), DEV)
        idx = torch.from_numpy(rec_o["idx"][li]).to(DEV)
        if li == 0:
            ref = xyz_layer64(P, block_params(sd, "init_scalar.", DEV), xyz, idx)
        else:
            ps, pv = rec_o["pools"][li - 1]
            ref = edge_layer64(P, torch.from_numpy(ps).to(DEV), torch.from_numpy(pv).to(DEV), idx)
        where = "%s layer %d" % (kernel, li + 1)
        if li == 0 or binary:
            assert (got_s == o_s.reshape(B * N, cs)).all(), where + ": pooled scalars differ from the oracle"
        else:
            a1, c1 = (t2n(t) for t in getattr(net, "conv%d" % (li + 1)).bn1_folded())
            e = s_error(got_s, ref, a1, c1)
            report("trunk " + where, rho=e.max())
            assert e.max() <= RHO_S[kernel][0], (where, e.max())
        ev = v_error(got_v.reshape(ref["v"].shape), ref)
        report("trunk " + where, tau_v=ev.max(), min_wins=float(ref["min_wins"].double().mean()))
        assert ev.max() <= TAU_V, (where, ev.max())
        if li > 0 and binary:
            sf, vf = orc.graph_feature_sv(rec_o["pools"][li - 1][0], rec_o["pools"][li - 1][1], rec_o["idx"][li])
            Po = orc.Params(sd).sub("conv%d" % (li + 1))
            sign = orc.sign_plane(np.concatenate([sf, orc.p_v2s(Po.sub("v2s"), vf)], axis=-1),
                                  Po.get("linear1.beta")).reshape(B * N * k, -1)
            taps = rec["taps%d" % li]
            K = sign.shape[1]
            assert (_unpack(t2n(taps["bits"]), K) == (sign > 0)).all(), where + ": sign bits"
            assert (_unpack(t2n(taps["mask"]), K) == (sign != 0)).all(), where + ": zero mask"
        so += cs
        vo += cv


@pytest.mark.gpu
@pytest.mark.parametrize("kind,binary,B,N,k", [("cls", True, 2, 1024, 20), ("cls", False, 2, 1024, 20),
                                               ("pseg", True, 1, 2048, 40)])
def test_whole_model_signed_checkpoint(kind, binary, B, N, k):
    """Whole models on a signed checkpoint: logits within the north-star tolerance of the oracle with its graphs
    forced, identical argmax; the C entry (which packs its own folded BatchNorm) equals the module path bit for bit."""
    import svnet_b200 as sv
    from svnet_b200 import fused
    from svnet_b200.synthetic import one_hot_labels
    net = quiet(sv.SV_DGCNN_PSEG if kind == "pseg" else sv.SV_DGCNN_CLS, make_args(k=k, binary=binary),
                50 if kind == "pseg" else 40)
    sd = signed_state_dict(net.state_dict(), 4100 + k)
    net.load_state_dict(sd)
    net = net.to(DEV).eval()
    x = synthetic_clouds(B, N, 4100 + k)
    extra = (one_hot_labels(B),) if kind == "pseg" else ()
    rec = {}
    if kind == "pseg":
        ref = orc.sv_dgcnn_pseg(sd, x.numpy(), extra[0].numpy(), k, rec=rec)
    else:
        ref = orc.sv_dgcnn_cls(sd, x.numpy(), k, rec=rec)
    xd, ed = x.to(DEV), tuple(e.to(DEV) for e in extra)
    keep = fused.NATIVE_FORWARD
    try:
        with torch.no_grad():
            y = t2n(net(xd, *ed, forced_idx=[torch.from_numpy(i).to(torch.int32).to(DEV) for i in rec["idx"]]))
            fused.NATIVE_FORWARD = False
            y_mod = net(xd, *ed)
    finally:
        fused.NATIVE_FORWARD = keep
    assert_close(y, ref, what="%s logits (oracle graphs forced)" % kind)
    cls_axis = 1
    assert (y.argmax(cls_axis) == ref.argmax(cls_axis)).all()
    native = sv.NativeModel("SV_DGCNN_PSEG" if kind == "pseg" else "SV_DGCNN_CLS", sd, k=k, binary=binary,
                            num_class=50 if kind == "pseg" else 40, device=DEV)
    with torch.no_grad():
        y_c = native(xd, *ed)
    native.close()
    assert torch.equal(y_c, y_mod)


@pytest.mark.gpu
def test_fp_classifier_with_fp_vector_linear_switched_off():
    """SVNET_VLINEAR_FP_TC=0 takes the fp-weight tensor-core vector linear off: the fp edge layers then run the
    CUDA-core kernel on the P | Q table, and a k = 20 forward runs and matches the default within tolerance."""
    import svnet_b200 as sv
    net = quiet(sv.SV_DGCNN_CLS, make_args(k=20, binary=False), 40)
    net.load_state_dict(signed_state_dict(net.state_dict(), 4200))
    net = net.to(DEV).eval()
    x = synthetic_clouds(4, 1024, 4200).to(DEV)
    with torch.no_grad():
        y0 = net(x)
        with env(SVNET_VLINEAR_FP_TC="0"):
            names = kernels_launched(lambda: net(x))
            y1 = net(x)
    assert ran(names, "edge_fp_fast_kernel") and not ran(names, "edge_fp_tc_kernel"), sorted(set(names))
    assert_close(t2n(y1), t2n(y0), what="fp logits with SVNET_VLINEAR_FP_TC=0")


# ------------------------------------------------------------------------------------------------
# D. the fp-weight vector linear (vlinear_tcgen05_kernel<3>) against float64
# ------------------------------------------------------------------------------------------------
def _vl_inputs(R, K, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(R, 3, K, generator=g) * torch.exp2(torch.randint(-4, 5, (K,), generator=g).float())


@pytest.mark.gpu
@pytest.mark.parametrize("K", [10, 21, 24, 96])
@pytest.mark.parametrize("NC", [33, 111, 256])
def test_fp_vector_linear_c4_table_against_float64(K, NC):
    """The float4 table [P | Q | T | U | v] of the fp edge layers: linear_rows(sign_w=False, G=3, c4=True) within
    RHO_C4 of float64, fourth float 0, identity rows copy v bit for bit, nothing written past the table."""
    from svnet_b200 import _native as nv
    g = torch.Generator().manual_seed(K * 1000 + NC)
    W = (torch.rand(NC, K, generator=g) * 2 - 1) / math.sqrt(K)
    n_eye = min(K, NC // 3)
    W[NC - n_eye:] = torch.eye(K)[:n_eye]                         # identity rows: the v columns of the edge table
    Wd = W.to(DEV)
    worst = 0.0
    for R in (1, 31, 33, 1000, 4099):
        v = _vl_inputs(R, K, R + K)
        vd = v.to(DEV)
        table = torch.full((R + 2, NC + 2, 4), float("nan"), device=DEV)
        with torch.no_grad():
            names = kernels_launched(lambda: nv.linear_rows(vd, vd.stride(0), vd.stride(1), 3, 3 * R, K, Wd, NC, table,
                                                            4 * (NC + 2), 0, c4=True))
        assert ran(names, "vlinear_tcgen05_kernel"), sorted(set(names))
        t = table[:R, :NC]
        ref = torch.einsum("rxd,cd->rcx", v.double(), W.double())
        mag = torch.einsum("rxd,cd->rcx", v.double().abs(), W.double().abs())
        err = ((t[..., :3].double().cpu() - ref).abs() / mag.clamp_min(1e-300)).max().item()
        worst = max(worst, err)
        assert (t[..., 3] == 0).all(), "fourth float of the table"
        assert torch.equal(t[:, NC - n_eye:, :3].cpu(), v[:, :, :n_eye].transpose(1, 2)), "identity columns"
        assert torch.isnan(table[R:]).all() and torch.isnan(table[:R, NC:]).all(), "wrote past the table"
    report("vlinear c4 K=%d NC=%d" % (K, NC), rho=worst)
    assert worst <= RHO_C4, worst


def _vbn_case(R, K, N, gpc, seed):
    g = torch.Generator().manual_seed(seed)
    v = _vl_inputs(R, K, seed)
    W = (torch.rand(N, K, generator=g) * 2 - 1) / math.sqrt(K)
    w = (torch.rand(N, generator=g) + 0.5) * torch.where(torch.rand(N, generator=g) < 0.5, -1.0, 1.0)
    b, m, var = torch.randn(N, generator=g) * 0.1, torch.randn(N, generator=g) * 0.1, torch.rand(N, generator=g) + 0.5
    gate = torch.sigmoid(torch.randn(-(-R // gpc), N, generator=g))
    a = w / torch.sqrt(var + BN_EPS)
    c = b - m * a
    y = torch.einsum("rxd,nd->rxn", v.double(), W.double())
    n = torch.sqrt((y * y).sum(1, keepdim=True)) + 1e-6
    ref = y / n * (n * a.double() + c.double()) * gate.double()[torch.arange(R) // gpc][:, None, :]
    return v, W, (a.float(), c.float()), gate, ref


def _run_vbn(v, W, bn, gate, gpc, switches):
    from svnet_b200 import _native as nv
    R, _, K = v.shape
    N = W.shape[0]
    vd, Wd = v.to(DEV), W.to(DEV)
    out = torch.full((R, 3, N + 3), float("nan"), device=DEV)
    o = out[:, :, 1:1 + N]
    with env(**switches), torch.no_grad():
        names = kernels_launched(lambda: nv.linear_rows(vd, vd.stride(0), vd.stride(1), 3, 3 * R, K, Wd, N, o, o.stride(0),
                                                        o.stride(1), bn=(bn[0].to(DEV), bn[1].to(DEV)), vbn=True,
                                                        gate=gate.to(DEV), groups_per_cloud=gpc))
    assert torch.isnan(out[:, :, 0]).all() and torch.isnan(out[:, :, 1 + N:]).all()
    return o.double().cpu(), names


def _vbn_err(got, ref):
    return ((got - ref).abs() / ref.abs().amax(dim=(0, 1), keepdim=True).clamp_min(1e-30)).max().item()


@pytest.mark.gpu
@pytest.mark.parametrize("K,N", [(83, 170), (64, 128), (64, 129), (64, 256), (96, 128), (96, 129), (96, 256)])
@pytest.mark.parametrize("gpc", [1000, 1024])
def test_fp_vector_linear_vbn_gate_against_float64(K, N, gpc):
    """fp-weight vector linear + VectorBN (negative BN weights) + gate on the tensor cores (three weight planes)
    against float64 and against the fp32 CUDA-core kernel (SVNET_VLINEAR_FP_TC=0); gpc = 1000 makes tiles straddle
    clouds."""
    R = 3 * gpc
    v, W, bn, gate, ref = _vbn_case(R, K, N, gpc, K + N + gpc)
    got, names = _run_vbn(v, W, bn, gate, gpc, {})
    assert ran(names, "vlinear_tcgen05_kernel"), sorted(set(names))
    slow, names = _run_vbn(v, W, bn, gate, gpc, {"SVNET_VLINEAR_FP_TC": "0"})
    assert ran(names, "linear_rows_kernel") and not ran(names, "vlinear_tcgen05_kernel"), sorted(set(names))
    e_tc, e_cc = _vbn_err(got, ref), _vbn_err(slow, ref)
    report("vlinear vbn K=%d N=%d gpc=%d" % (K, N, gpc), tau_tc=e_tc, tau_cuda_cores=e_cc)
    assert e_tc <= TAU_VBN and e_cc <= TAU_VBN, (e_tc, e_cc)


@pytest.mark.gpu
@pytest.mark.parametrize("K,N", [(97, 128), (64, 257)])
def test_fp_vector_linear_outside_the_tensor_core_shapes(K, N):
    """K = 97 / N = 257 are beyond the tcgen05 kernel: VectorBN + gate falls back and stays correct, the c4 table
    raises a clean error and writes nothing."""
    from svnet_b200 import _native as nv
    gpc = 500
    v, W, bn, gate, ref = _vbn_case(2 * gpc, K, N, gpc, K + N)
    got, names = _run_vbn(v, W, bn, gate, gpc, {})
    assert not ran(names, "vlinear_tcgen05_kernel"), sorted(set(names))
    assert _vbn_err(got, ref) <= TAU_VBN
    vd = v.to(DEV)
    table = torch.full((v.shape[0], N, 4), float("nan"), device=DEV)
    with pytest.raises(RuntimeError, match="c4 table layout"):
        nv.linear_rows(vd, vd.stride(0), vd.stride(1), 3, 3 * v.shape[0], K, W.to(DEV), N, table, 4 * N, 0, c4=True)
    torch.cuda.synchronize()
    assert torch.isnan(table).all()


# ------------------------------------------------------------------------------------------------
# E. gate kernels against float64
# ------------------------------------------------------------------------------------------------
def _gate64(mean, G1, G2):
    return torch.sigmoid(G2.double() @ torch.relu(G1.double() @ mean.T)).T


def _gate_weights(Cin, Co, seed):
    g = torch.Generator().manual_seed(seed)
    H = Co // 2
    return (torch.rand(H, Cin, generator=g) * 2 - 1) / math.sqrt(Cin), (torch.rand(Co, H, generator=g) * 2 - 1) / math.sqrt(H)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [511, 512, 1021, 4096])
@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("Cs", [32, 64, 130])
@pytest.mark.parametrize("graph", ["random", "one_point", "self", "offset"])
def test_gate_edge_against_float64(N, B, Cs, graph):
    """gate_edge (mean over the N k edge rows [s_j - s_i | s_i] through the gate MLP; cluster variant from N = 512,
    ragged row splits) within GATE_ABS of float64.  With a common offset (s = 100 + noise) the kernel's difference of
    two means may not lose more than the fp32 reference, which sums the materialised rows, does."""
    from svnet_b200 import _native as nv
    k = 20
    g = torch.Generator().manual_seed(N + B + Cs)
    s = torch.randn(B * N, Cs, generator=g)
    if graph == "offset":
        s = s + 100.0
    idx = torch.randint(0, N, (B, N, k), generator=g, dtype=torch.int32)
    if graph == "one_point":
        idx[:] = 7
    elif graph == "self":
        idx[:] = torch.arange(N, dtype=torch.int32)[None, :, None]
    G1, G2 = _gate_weights(2 * Cs, 42, Cs)
    tab = torch.full((B * N, Cs + 4), float("nan"))
    tab[:, 1:1 + Cs] = s
    td = tab.to(DEV)
    sv_ = td[:, 1:1 + Cs]
    vdummy = torch.zeros(B * N, 3, 1, device=DEV)
    with torch.no_grad():
        names = kernels_launched(lambda: nv.gate_edge(nv.view_of(sv_, vdummy), idx.to(DEV), B, N, k, G1.to(DEV), G2.to(DEV)))
        got = nv.gate_edge(nv.view_of(sv_, vdummy), idx.to(DEV), B, N, k, G1.to(DEV), G2.to(DEV)).double().cpu()
    assert ran(names, "gate_edge_cluster_kernel" if N >= 512 else "gate_edge_kernel"), sorted(set(names))
    sd_ = s.double().view(B, N, Cs).to(DEV)
    sj = torch.stack([sd_[b][idx[b].long().to(DEV)] for b in range(B)])                # (B, N, k, Cs)
    mean = torch.cat([(sj - sd_[:, :, None]).mean((1, 2)), sd_.mean(1)], -1)
    ref = _gate64(mean.cpu(), G1, G2)
    err = (got - ref).abs().max().item()
    bar = GATE_ABS
    if graph == "offset":
        si = sd_[:, :, None].expand_as(sj)
        feat = torch.cat([sj - si, si], -1).float().cpu().numpy()
        e32 = np.abs(orc.gate(feat, G1.numpy(), G2.numpy()) - ref.numpy()).max()
        report("gate_edge offset N=%d B=%d Cs=%d" % (N, B, Cs), err=err, fp32_reference_err=e32)
        bar = GATE_OFFSET_ABS
    else:
        report("gate_edge %s N=%d B=%d Cs=%d" % (graph, N, B, Cs), err=err)
    assert err <= bar, (err, bar)


@pytest.mark.gpu
@pytest.mark.parametrize("rows", [511, 512, 1021])
@pytest.mark.parametrize("Cs", [256, 300])
def test_gate_rows_against_float64(rows, Cs):
    """gate_rows (mean over materialised rows; cluster variant from 512 rows) on a strided table within GATE_ABS."""
    from svnet_b200 import _native as nv
    B = 3
    g = torch.Generator().manual_seed(rows + Cs)
    s = torch.randn(B * rows, Cs, generator=g)
    tab = torch.full((B * rows, Cs + 5), float("nan"))
    tab[:, :Cs] = s
    td = tab.to(DEV)
    G1, G2 = _gate_weights(Cs, 170, Cs + 1)
    with torch.no_grad():
        names = kernels_launched(lambda: nv.gate_rows(td, td.stride(0), Cs, B, rows, G1.to(DEV), G2.to(DEV)))
        got = nv.gate_rows(td, td.stride(0), Cs, B, rows, G1.to(DEV), G2.to(DEV)).double().cpu()
    assert ran(names, "gate_rows_cluster_kernel" if rows >= 512 else "gate_rows_kernel"), sorted(set(names))
    ref = _gate64(s.double().view(B, rows, Cs).mean(1), G1, G2)
    err = (got - ref).abs().max().item()
    report("gate_rows rows=%d Cs=%d" % (rows, Cs), err=err)
    assert err <= GATE_ABS, err


@pytest.mark.gpu
@pytest.mark.parametrize("nvec", [2, 3])
@pytest.mark.parametrize("N,k", [(204, 20), (205, 20)])      # N k = 4080 / 4100: either side of the cluster switch
def test_gate_xyz_against_float64(nvec, N, k):
    """gate_xyz (layer 1: the mean of init_scalar over the edge features [x_j - x_i | x_i (| x_j x x_i)]) within
    GATE_ABS of float64, on either side of its cluster switch (N k >= 4096)."""
    from svnet_b200 import _native as nv
    B = 2
    g = torch.Generator().manual_seed(N + nvec)
    xyz = synthetic_clouds(B, N, N + nvec).transpose(1, 2).contiguous()
    idx = torch.randint(0, N, (B, N, k), generator=g, dtype=torch.int32)
    idx[:, :, 0] = torch.arange(N, dtype=torch.int32)
    Winit = (torch.rand(3, nvec, generator=g) * 2 - 1) / math.sqrt(nvec)
    G1, G2 = _gate_weights(3 * nvec, 10, nvec)
    with torch.no_grad():
        got = nv.gate_xyz(xyz.view(B * N, 3).to(DEV), idx.to(DEV), nvec, Winit.to(DEV), G1.to(DEV), G2.to(DEV)).double().cpu()
    x64 = xyz.double()
    feats = []
    for b in range(B):
        xj = x64[b][idx[b].long()]
        xi = x64[b][:, None].expand_as(xj)
        f = [xj - xi, xi] + ([torch.cross(xj, xi, dim=-1)] if nvec == 3 else [])
        feats.append(_v2s64({"linear.weight": Winit.double()}, torch.stack(f, -1), "linear").mean((0, 1)))
    ref = _gate64(torch.stack(feats), G1, G2)
    err = (got - ref).abs().max().item()
    report("gate_xyz nv=%d N*k=%d" % (nvec, N * k), err=err)
    assert err <= GATE_ABS, err
