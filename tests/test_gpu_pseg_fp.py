"""The full-precision SV-DGCNN part-segmentation model on the sm_100a fast path: the tensor-core fp edge kernel at its shapes
(k = 20 and 40), the fp head as one call (svnet_seg_head_fp_fwd) and the whole-model C entry.

Bars of the fp head were set from runs on an NVIDIA B200 (1000 W power limit): at most 4x the largest value measured there
and below 2^-17; the measured values are printed (`pytest -s`).  The edge-kernel bars are those of test_gpu_edge_fp64.py.
"""
import math

import pytest
import torch

from oracle import svnet_oracle as orc
from tests.test_gpu_edge_fp64 import (FP_KERNELS, RHO_S, RHO_S_RMS, TAU_V, TC_OVER_CHAIN, _edge_block, _inputs, _teacher_forced,
                                      _trunk_case, block_params, edge_layer64, kernels_launched, ran, report,
                                      run_edge_layer, s_error, signed_state_dict, v_error)
from tests.util import assert_close, quiet, t2n
from svnet_b200.synthetic import make_args, one_hot_labels, synthetic_clouds

pytestmark = pytest.mark.gpu

DEV = "cuda"
PSEG_SHAPES = [(32, 16, 32, 16), (32, 16, 64, 24), (64, 24, 128, 40)]
CLS_SHAPES = [(32, 10, 32, 10), (32, 10, 64, 21), (64, 21, 128, 42)]
# fp head: |y - y64| <= rho * sum_c |W11_pc h10_c| (h10: conv10's float64 output; the logits have no BN, a = 1), one bar per
# quantity, each at most 4x its measured value: the head call 8.3e-7, layer by layer 1.15e-6, call against layer by layer 3.7e-7
RHO_HEAD_CALL = 3.3e-6
RHO_HEAD_LAYERS = 4.6e-6
RHO_HEAD_CALL_VS_LAYERS = 1.4e-6


def _pseg(k, seed):
    import svnet_b200 as sv
    net = quiet(sv.SV_DGCNN_PSEG, make_args(k=k, binary=False), 50)
    sd = signed_state_dict(net.state_dict(), seed)
    net.load_state_dict(sd)
    return net.to(DEV).eval(), sd


# ------------------------------------------------------------------------------------------------
# 1. the tensor-core edge kernel at the part-segmentation shapes
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", PSEG_SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("k", [20, 40])
@pytest.mark.parametrize("B,N", [(2, 1024), (3, 1021), (2, 37), (1, 13)])
@pytest.mark.parametrize("regime", ["model", "scaled", "graph"])
def test_edge_fp_tc_pseg_shapes_against_float64(shape, k, B, N, regime):
    """edge_fp_tc at the fp part-segmentation shapes (several warps per point at k = 40, Cv = 16 / 24 walked as 16 + 8
    channels, two K phases) and the fp32 CUDA-core kernel against float64 with negative BatchNorm weights, on strided
    slices of NaN-filled tables: pooled s within RHO_S * |a1| * S, pooled v within TAU_V, the min branch decides >= 10 %,
    the tensor-core kernel within TC_OVER_CHAIN of the fp32 chain, nothing written outside the output columns."""
    Cs, Cv, Cout, Cvo = shape
    blk, sd = _edge_block(Cs, Cv, Cout, Cvo, False, 500 + Cout + k)
    s, v, idx = _inputs(regime, B, N, Cs, Cv, k, 31 + N + Cout + k)
    ref = edge_layer64(block_params(sd, "", DEV), s.to(DEV), v.to(DEV), idx.to(DEV))
    a1, c1 = (t2n(t) for t in blk.bn1_folded())
    assert float(ref["min_wins"].double().mean()) >= 0.10, "the min branch must decide >= 10 % of the outputs"
    rho = {}
    for name in ("fp_tc", "fp_fast"):
        switches, kernel = FP_KERNELS[name]
        got_s, got_v, names, untouched = run_edge_layer(blk, s, v, idx, switches)
        assert ran(names, kernel), (name, sorted(set(names)))
        assert untouched, name + ": wrote outside its output columns"
        e = s_error(got_s, ref, a1, c1)
        ev = v_error(got_v.reshape(ref["v"].shape), ref)
        rho[name] = float(e.max())
        report("pseg edge %s %s k=%d B=%d N=%d %s" % (name, "x".join(map(str, shape)), k, B, N, regime), rho=e.max(),
               rho_rms=math.sqrt(float((e ** 2).mean())), tau_v=ev.max())
        col = 1 if regime == "scaled" else 0
        assert e.max() <= RHO_S[name][col], (name, e.max())
        assert math.sqrt(float((e ** 2).mean())) <= RHO_S_RMS[name][col], name
        assert ev.max() <= TAU_V, (name, ev.max())
    assert rho["fp_tc"] <= TC_OVER_CHAIN * max(rho["fp_fast"], 2.0 ** -24), rho


# ------------------------------------------------------------------------------------------------
# 2. coverage is a set of (shape, k) pairs
# ------------------------------------------------------------------------------------------------
def test_edge_fp_tc_coverage_is_shape_and_k():
    """The fp classifier's shapes are covered at k = 20 only: at k = 40 the weight query says 0 and the layer runs
    edge_fp_fast_kernel; the part-segmentation shapes are covered at 20 and 40, at no other k."""
    from svnet_b200 import _native as nv
    for shape in CLS_SHAPES:
        assert nv.edge_fp_tc_weight_bytes(*shape, 20) > 0 and nv.edge_fp_tc_weight_bytes(*shape, 40) == 0, shape
    for shape in PSEG_SHAPES:
        assert nv.edge_fp_tc_weight_bytes(*shape, 20) > 0 and nv.edge_fp_tc_weight_bytes(*shape, 40) > 0, shape
        assert nv.edge_fp_tc_weight_bytes(*shape, 12) == 0 and nv.edge_fp_tc_weight_bytes(*shape, 30) == 0, shape
    Cs, Cv, Cout, Cvo = CLS_SHAPES[2]
    blk, sd = _edge_block(Cs, Cv, Cout, Cvo, False, 640)
    s, v, idx = _inputs("model", 2, 256, Cs, Cv, 40, 641)
    got_s, _, names, _ = run_edge_layer(blk, s, v, idx, {})
    assert ran(names, "edge_fp_fast_kernel") and not ran(names, "edge_fp_tc_kernel"), sorted(set(names))
    a1, c1 = (t2n(t) for t in blk.bn1_folded())
    assert s_error(got_s, edge_layer64(block_params(sd, "", DEV), s.to(DEV), v.to(DEV), idx.to(DEV)), a1, c1).max() <= RHO_S["fp_fast"][0]


# ------------------------------------------------------------------------------------------------
# 3. the fp part-segmentation trunk, teacher-forced on the oracle's inputs and graphs
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kernel", ["fp_tc", "fp_fast", "generic"])
def test_pseg_fp_trunk_teacher_forced(kernel):
    """Edge layers 1..4 of the signed fp part-segmentation model at k = 40 (B = 1, N = 1024), each fed the oracle's input
    and graph: layer 1 bit-identical to the oracle, layers 2..4 within RHO_S of float64, v within TAU_V."""
    B, N, k = 1, 1024, 40
    net, sd, x, rec_o = _trunk_case("pseg", False, k, B, N, 4301)
    switches, want = FP_KERNELS[kernel]
    rec, names = _teacher_forced(net, "pseg", x, rec_o, switches)
    assert ran(names, want), sorted(set(names))
    so = vo = 0
    for li, (o_s, o_v) in enumerate(rec_o["pools"]):
        cs, cv = o_s.shape[-1], o_v.shape[-1]
        got_s = t2n(rec["s_cat"][:, so:so + cs])
        got_v = t2n(rec["v_cat"][:, :, vo:vo + cv])
        where = "%s layer %d" % (kernel, li + 1)
        if li == 0:
            assert (got_s == o_s.reshape(B * N, cs)).all(), where + ": pooled scalars differ from the oracle"
            assert_close(got_v.reshape(o_v.shape), o_v, rtol=1e-4, atol=1e-5, what=where + " v")
        else:
            P = block_params(sd, "conv%d." % (li + 1), DEV)
            ps, pv = rec_o["pools"][li - 1]
            ref = edge_layer64(P, torch.from_numpy(ps).to(DEV), torch.from_numpy(pv).to(DEV), torch.from_numpy(rec_o["idx"][li]).to(DEV))
            a1, c1 = (t2n(t) for t in getattr(net, "conv%d" % (li + 1)).bn1_folded())
            e = s_error(got_s, ref, a1, c1)
            ev = v_error(got_v.reshape(ref["v"].shape), ref)
            report("pseg trunk " + where, rho=e.max(), tau_v=ev.max(), min_wins=float(ref["min_wins"].double().mean()))
            assert e.max() <= RHO_S[kernel][0], (where, e.max())
            assert ev.max() <= TAU_V, (where, ev.max())
        so += cs
        vo += cv


# ------------------------------------------------------------------------------------------------
# 4. the fp head as one call against float64 and against the layer-by-layer calls
# ------------------------------------------------------------------------------------------------
def _head_inputs(B, N, seed):
    g = torch.Generator().manual_seed(seed)
    s_cat = torch.randn(B * N, 256, generator=g).abs()            # pooled leaky outputs: mostly >= 0
    v_cat = torch.randn(B * N, 3, 96, generator=g) * 0.5
    glob = torch.randn(B, 1600, generator=g)
    return s_cat.to(DEV), v_cat.to(DEV), glob.to(DEV)


def _head64(net, s_cat, v_cat, glob, N):
    """conv8 .. conv11 of sv_dgcnn_partseg.py:112-126 (full precision) in float64 on [glob repeated | svfuse1(s, v)];
    also the operand scale of the logits, M = |W11| |h10|."""
    def bn(seq):
        b = seq[1]
        a = b.weight.double() / torch.sqrt(b.running_var.double() + b.eps)
        return a, b.bias.double() - b.running_mean.double() * a
    Wz = net.svfuse1.v2s.linear.weight.detach().double()
    v = v_cat.double()
    q = torch.einsum("rxd,rxm->rdm", v, torch.einsum("rxd,md->rxm", v, Wz)).reshape(v.shape[0], -1)
    B = glob.shape[0]
    x = torch.cat([glob.double().repeat_interleave(N, 0), s_cat.double(), q], 1)
    for seq in (net.conv8, net.conv9, net.conv10):
        W = seq[0].weight.detach()[:, :, 0].double()
        a, c = bn(seq)
        t = (x @ W.t()) * a + c
        x = torch.where(t > 0, t, 0.2 * t)
    W11 = net.conv11.weight.detach()[:, :, 0].double()
    y, m = x @ W11.t(), x.abs() @ W11.abs().t()
    return (y.view(B, N, -1).transpose(1, 2).contiguous(), m.view(B, N, -1).transpose(1, 2).contiguous())


@pytest.mark.parametrize("B,N", [(2, 2048), (3, 333)])
def test_seg_head_fp_call_against_float64_and_layerwise(B, N):
    """svnet_seg_head_fp_fwd (conv8's per-cloud part once per cloud, the per-point part over svfuse1's 544 channels, conv9 ..
    conv11, (B, parts, N) layout) within RHO_HEAD_CALL * M of float64; the layer-by-layer calls over the (B*N, 2144) table
    within the same bound (they split conv8's K differently: not bit-equal)."""
    from svnet_b200 import _native as nv
    from svnet_b200.sv_layers import dense_rows
    net, _ = _pseg(40, 4400)
    s_cat, v_cat, glob = _head_inputs(B, N, 4400 + N)
    layers = [(c.weight2d(), seq.bn_folded()) for c, seq in ((net.conv8[0], net.conv8), (net.conv9[0], net.conv9),
                                                              (net.conv10[0], net.conv10))]
    W11 = net.conv11.weight.detach()[:, :, 0].contiguous()
    with torch.no_grad():
        names = kernels_launched(lambda: nv.seg_head_fp_fwd(nv.view_of(s_cat, v_cat), B, N, net.svfuse1.v2s.wz()[0], glob, layers, W11))
        y_call = nv.seg_head_fp_fwd(nv.view_of(s_cat, v_cat), B, N, net.svfuse1.v2s.wz()[0], glob, layers, W11)
        x_fine = net.svfuse1.forward_rows(s_cat, v_cat)[0]
        h = net.conv8[0].forward_rows(x_fine, bn=net.conv8.bn_folded(), act=nv.ACT_LEAKY, cloud=glob, rows_per_cloud=N)
        h = net.conv9[0].forward_rows(h, bn=net.conv9.bn_folded(), act=nv.ACT_LEAKY)
        h = net.conv10[0].forward_rows(h, bn=net.conv10.bn_folded(), act=nv.ACT_LEAKY)
        y_layers = dense_rows(net.conv11.weight, h).view(B, N, -1).transpose(1, 2)
        y64, M = _head64(net, s_cat, v_cat, glob, N)
    assert ran(names, "gemm_tc3_kernel") and not ran(names, "linear_rows_kernel"), sorted(set(names))
    assert tuple(y_call.shape) == (B, 50, N) and y_call.is_contiguous()
    rho_call = float(((y_call.double() - y64).abs() / M).max())
    rho_layers = float(((y_layers.double() - y64).abs() / M).max())
    rho_diff = float(((y_call.double() - y_layers.double()).abs() / M).max())
    report("fp head B=%d N=%d" % (B, N), rho_call=rho_call, rho_layers=rho_layers, rho_call_vs_layers=rho_diff)
    assert rho_call <= RHO_HEAD_CALL, rho_call
    assert rho_layers <= RHO_HEAD_LAYERS, rho_layers
    assert rho_diff <= RHO_HEAD_CALL_VS_LAYERS, rho_diff


# ------------------------------------------------------------------------------------------------
# 5. the whole model against the oracle
# ------------------------------------------------------------------------------------------------
def test_pseg_fp_whole_model_against_oracle():
    """Signed fp part-segmentation checkpoint, B = 1, N = 2048, k = 40, the oracle's graphs forced: logits within
    1e-3 rel / 1e-4 abs of the oracle, identical per-point argmax; the run takes the fp head call and edge_fp_tc."""
    B, N, k = 1, 2048, 40
    net, sd = _pseg(k, 4500)
    x = synthetic_clouds(B, N, 4500)
    l = one_hot_labels(B)
    rec = {}
    ref = orc.sv_dgcnn_pseg(sd, x.numpy(), l.numpy(), k, rec=rec)
    fi = [torch.from_numpy(i).to(torch.int32).to(DEV) for i in rec["idx"]]
    with torch.no_grad():
        names = kernels_launched(lambda: net(x.to(DEV), l.to(DEV), forced_idx=fi))
        y = t2n(net(x.to(DEV), l.to(DEV), forced_idx=fi))
    assert ran(names, "edge_fp_tc_kernel") and ran(names, "gemm_tc3_kernel"), sorted(set(names))
    assert y.shape == ref.shape == (B, 50, N)
    assert_close(y, ref, what="fp pseg logits (oracle graphs forced)")
    assert (y.argmax(1) == ref.argmax(1)).all()


# ------------------------------------------------------------------------------------------------
# 6. the whole-model C entry against the module path; 7. batch independence
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,N,k", [(2, 2048, 40), (3, 320, 20), (17, 2048, 40)])
def test_model_c_entry_pseg_fp_equals_module(B, N, k):
    """svnet_model_create("SV_DGCNN_PSEG", binary = 0) + svnet_model_forward_seg against the nn.Module path sequenced in
    Python on the same checkpoint: bit-identical logits, also through model(x, l) and from a CUDA graph; B = 17 runs
    two sub-batches on both sides."""
    import svnet_b200 as sv
    from svnet_b200 import fused
    net, sd = _pseg(k, 4600 + k)
    x = synthetic_clouds(B, N, 4600 + B).to(DEV)
    l = one_hot_labels(B).to(DEV)
    native = sv.NativeModel("SV_DGCNN_PSEG", {"module." + n: t for n, t in sd.items()}, k=k, binary=False, num_class=50, device=DEV)
    keep = fused.NATIVE_FORWARD
    try:
        with torch.no_grad():
            fused.NATIVE_FORWARD = False
            y_mod = net(x, l)
            fused.NATIVE_FORWARD = True
            names = kernels_launched(lambda: net(x, l))
            y_del = net(x, l)
            y_c = native(x, l)
    finally:
        fused.NATIVE_FORWARD = keep
    assert ran(names, "edge_fp_tc_kernel") and ran(names, "gemm_tc3_kernel"), sorted(set(names))
    assert tuple(y_c.shape) == (B, 50, N)
    assert torch.equal(y_c, y_mod)
    assert torch.equal(y_del, y_mod)
    g = torch.cuda.CUDAGraph()
    xs, ls = x.clone(), l.clone()
    native(xs, ls)
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        y_g = native(xs, ls)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(y_g, y_mod)
    with pytest.raises(ValueError):
        native(synthetic_clouds(1, 48, 1).to(DEV), one_hot_labels(1).to(DEV))      # N < 64: not covered
    native.close()


def test_model_c_entry_pseg_fp_rejects_classifier_tensors():
    """A full-precision classifier's state dict is not a part-segmentation checkpoint: the loader names the tensor."""
    import svnet_b200 as sv
    cls = quiet(sv.SV_DGCNN_CLS, make_args(k=20, binary=False), 40)
    sd = signed_state_dict(cls.state_dict(), 4700)
    with pytest.raises(RuntimeError, match="svnet_model_create: .*(missing from the state_dict|wrong size)"):
        sv.NativeModel("SV_DGCNN_PSEG", sd, k=20, binary=False, num_class=40, device=DEV)


def test_pseg_fp_batch_independence():
    """Cloud 3 of an 8-cloud batch equals that cloud run alone, bit for bit (C entry and module path)."""
    from svnet_b200 import fused
    net, _ = _pseg(40, 4800)
    x = synthetic_clouds(8, 2048, 4800).to(DEV)
    l = one_hot_labels(8).to(DEV)
    keep = fused.NATIVE_FORWARD
    try:
        with torch.no_grad():
            y = net(x, l)
            y3 = net(x[3:4].contiguous(), l[3:4].contiguous())
            fused.NATIVE_FORWARD = False
            y_mod3 = net(x[3:4].contiguous(), l[3:4].contiguous())
    finally:
        fused.NATIVE_FORWARD = keep
    assert torch.isfinite(y).all()
    assert torch.equal(y[3:4], y3)
    assert torch.equal(y3, y_mod3)


def test_pseg_fp_sixteen_parts_through_model_call():
    """16 parts: conv11 (128 -> 16) is below the tensor-core linear's 32 output channels and runs on the CUDA-core chain inside
    the head call.  model(x, l) takes the whole-model C entry and equals the module path bit for bit, and the head call agrees
    with the layer-by-layer head within the whole-model tolerance."""
    import svnet_b200 as sv
    from svnet_b200 import _native as nv
    from svnet_b200 import fused
    from svnet_b200 import sv_dgcnn_partseg as ps
    net = quiet(sv.SV_DGCNN_PSEG, make_args(k=40, binary=False), 16)
    net.load_state_dict(signed_state_dict(net.state_dict(), 4900))
    net = net.to(DEV).eval()
    B, N = 3, 512
    x = synthetic_clouds(B, N, 4900).to(DEV)
    l = one_hot_labels(B).to(DEV)
    keep = fused.NATIVE_FORWARD, ps.SEG_HEAD_CALL
    try:
        with torch.no_grad():
            fused.NATIVE_FORWARD = True
            net(x, l)                                   # builds the handle (svnet_model_create)
            l0 = nv.LAUNCHES[0]
            y_c = net(x, l)
            calls = nv.LAUNCHES[0] - l0
            names = kernels_launched(lambda: net(x, l))
            fused.NATIVE_FORWARD = False
            y_mod = net(x, l)
            ps.SEG_HEAD_CALL = False
            y_layers = net(x, l)
    finally:
        fused.NATIVE_FORWARD, ps.SEG_HEAD_CALL = keep
    assert calls == 1, "model(x, l) did not take the whole-model C entry (%d C-ABI calls)" % calls
    assert ran(names, "edge_fp_tc_kernel") and ran(names, "gemm_tc3_kernel"), sorted(set(names))
    assert tuple(y_c.shape) == (B, 16, N)
    assert torch.equal(y_c, y_mod)
    assert_close(t2n(y_c), t2n(y_layers), what="16-part fp logits, head call vs layer by layer")
    assert (y_c.argmax(1) == y_layers.argmax(1)).all()
