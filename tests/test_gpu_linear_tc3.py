"""The three-plane tensor-core fp32 linear (csrc/gemm_tc3.cu, gemm_tc3_kernel) against float64 over its coverage.

Every plain fp32 linear of the full-precision models with 32 <= K <= 4096 and 32 <= N <= 512 runs on this kernel.  The
float64 product is taken on the GPU with torch; per output element the operand scale is S_rc = sum_k |A_rk| |W_ck|:

    no epilogue:    |y - y64| <= RHO * S
    with epilogue:  |out - f64(y64)| <= RHO * |cs_c a1_c| * S + 4 ulp(max(|out64|, |a1_c (cs_c y64 + bias_c)|))

(f64: colscale, bias, BN affine and activation in float64; the ulp term is the rounding of the kernel's fp32 chain
((y cs + bias) a1 + c1).)  Outputs whose operands are all exact zeros must be exactly 0.

With 64 or more row tiles (M >= 8065 rows) each CTA takes two 128-channel tiles, with fewer it takes one: the shape
list covers one to four channel tiles on both sides, and N = 257..384 at M >= 8065 is the case where the last CTA of a
row tile holds a single channel tile.

Bars were set from runs on an NVIDIA B200 (1000 W power limit): each is at most 4x the largest value measured there and
below what the kernel gives with one shared accumulator for the h*h and the five small plane products; the measured
values are printed (`pytest -s`).
"""
import ctypes
import math

import pytest
import torch

from tests.test_gpu_edge_fp64 import kernels_launched, ran, report
from tests.test_gpu_pseg_fp import RHO_HEAD_CALL, _head64, _head_inputs, _pseg

pytestmark = pytest.mark.gpu

DEV = "cuda"
# |y - y64| <= RHO * S, per input regime: model-like (randn) inputs, and inputs with per-row x per-column scales 2^-10 .. 2^10.
# Measured: 7.95e-7 and 5.16e-6 (both at K = 4096); with one shared accumulator 4.8e-6 and 1.83e-5.  The scaled bar is
# under 4x its measured value so that it stays below the shared accumulator's.
RHO = {"model": 2.4e-6, "scaled": 1.0e-5}

# (M, K, N): N = 32 .. 512 (one to four channel tiles), each with fewer and with 64 or more row tiles (8064 rows = 63 tiles,
# 8065 = 64); K on both sides of the 8-column staging blocks and the 32-column chunks, up to the 4096 limit
SHAPES = [
    (1, 32, 32), (8065, 33, 32),
    (127, 37, 33), (20000, 505, 33),
    (129, 544, 128), (8064, 1600, 128),
    (1, 4094, 129), (8065, 4096, 129),
    (127, 505, 256), (20000, 32, 256),
    (8064, 33, 257), (8065, 37, 257),
    (129, 1600, 300), (20000, 4094, 300),
    (1, 544, 384), (8065, 4096, 384),
    (127, 32, 385), (20000, 505, 385),
    (8064, 4096, 511), (8065, 1600, 511),
    (129, 4096, 512), (20000, 4096, 512),
    # the shipped layers: conv5's linear1 (505 -> 512), SV-PointNet part segmentation's convs1 (4094 -> 511), the fp
    # part-segmentation head's per-point conv8 (544 -> 256)
    (16384, 505, 512), (16384, 4094, 511), (32768, 544, 256),
]


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _operands(regime, M, K, N, seed):
    """A (M, K), W (N, K): randn, or with per-row x per-column scales 2^-10 .. 2^10; 5 % of A exactly 0 and, with M > 1,
    one all-zero row."""
    g = _gen(seed)
    A = torch.randn(M, K, generator=g, device=DEV)
    W = torch.randn(N, K, generator=g, device=DEV) / math.sqrt(K)
    if regime == "scaled":
        def scales(*shape):
            return torch.exp2(torch.rand(*shape, generator=g, device=DEV) * 20 - 10)
        A *= scales(M, 1) * scales(1, K)
        W *= scales(N, 1) * scales(1, K)
    A[torch.rand(M, K, generator=g, device=DEV) < 0.05] = 0.0
    if M > 1:
        A[M // 2] = 0.0
    return A, W


def _linear(A, W, C, **kw):
    """svnet_linear_rows_ws over the views A (M, K), W (N, K), C (M, N) with their row strides."""
    from svnet_b200 import _native as nv
    M, K = A.shape
    nv.linear_rows(A, A.stride(0), 0, 1, M, K, W, W.shape[0], C, C.stride(0), 0, **kw)


def _ref64(A, W):
    A64, W64 = A.double(), W.double()
    return A64 @ W64.t(), A64.abs() @ W64.abs().t()


def _rho(y, y64, S):
    """max |y - y64| / S; outputs with S == 0 must be exactly 0."""
    assert not torch.isnan(y).any(), "NaN in the output (an output not written?)"
    err = (y.double() - y64).abs()
    zero = S == 0
    assert bool((err[zero] == 0).all()), "an output whose operands are all 0 is not exactly 0"
    return float(torch.where(zero, 0.0, err / torch.where(zero, 1.0, S)).max())


def _ulp(x):
    x = x.abs().float()
    return (torch.nextafter(x, torch.full_like(x, math.inf)) - x).double()


def _act64(t, act):
    from svnet_b200 import _native as nv
    if act == nv.ACT_RELU:
        return t.clamp_min(0.0)
    if act == nv.ACT_LEAKY:
        return torch.where(t > 0, t, 0.2 * t)
    return t


def _rho_epilogue(out, y64, S, cs, bias, a1, c1, act):
    """(|out - f64(y64)| - 4 ulp(max(|out64|, |a1 (cs y64 + bias)|))) / (|cs a1| S); channels with cs a1 == 0 must be
    within the ulp term."""
    assert not torch.isnan(out).any(), "NaN in the output"
    cs, bias, a1, c1 = (t.double()[None, :] for t in (cs, bias, a1, c1))
    u = a1 * (cs * y64 + bias)
    ref = _act64(u + c1, act)
    err = (out.double() - ref).abs()
    floor = 4 * _ulp(torch.maximum(ref.abs(), u.abs()))
    scale = (cs * a1).abs() * S
    zero = scale == 0
    assert bool((err <= floor)[zero].all()), "an output with cs * a1 * S == 0 is off by more than rounding"
    return float(torch.where(zero, 0.0, (err - floor).clamp_min(0.0) / torch.where(zero, 1.0, scale)).max())


# ------------------------------------------------------------------------------------------------
# 1. accuracy over the coverage, one and two channel tiles per CTA
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,K,N", SHAPES, ids=lambda s: str(s))
@pytest.mark.parametrize("regime", ["model", "scaled"])
def test_linear_tc3_against_float64(M, K, N, regime):
    """gemm_tc3_kernel (and not the CUDA-core chain) runs; every output within RHO[regime] * S of float64, all-zero rows
    exactly 0, every output written."""
    A, W = _operands(regime, M, K, N, 7 * M + 3 * K + N + (1 if regime == "scaled" else 0))
    C = torch.full((M, N), math.nan, device=DEV)
    names = kernels_launched(lambda: _linear(A, W, C))
    assert ran(names, "gemm_tc3_kernel") and not ran(names, "linear_rows_kernel"), sorted(set(names))
    y64, S = _ref64(A, W)
    rho = _rho(C, y64, S)
    report("tc3 %s M=%d K=%d N=%d" % (regime, M, K, N), rho=rho)
    assert rho <= RHO[regime], rho


# ------------------------------------------------------------------------------------------------
# 2. the epilogue: colscale, bias, BN with negative and zero weights, activation
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M", [1000, 9000])                # one channel tile per CTA; two
@pytest.mark.parametrize("act", ["none", "relu", "leaky"])
def test_linear_tc3_epilogue_against_float64(M, act):
    """colscale (negative and zero entries), bias, BN affine with about half its weights negative and two exactly 0, then
    NONE / RELU / LEAKY, against the same chain in float64 on the float64 product."""
    from svnet_b200 import _native as nv
    act_id = {"none": nv.ACT_NONE, "relu": nv.ACT_RELU, "leaky": nv.ACT_LEAKY}[act]
    K, N = 505, 300
    A, W = _operands("model", M, K, N, 200 + M)
    g = _gen(300 + M)
    sign = torch.where(torch.rand(N, generator=g, device=DEV) < 0.5, -1.0, 1.0)
    cs = sign * (0.5 + torch.rand(N, generator=g, device=DEV))
    cs[17] = 0.0
    bias = torch.randn(N, generator=g, device=DEV)
    a1 = torch.randn(N, generator=g, device=DEV)
    a1[torch.randperm(N, generator=g, device=DEV)[:2]] = 0.0
    c1 = torch.randn(N, generator=g, device=DEV)
    assert (a1 < 0).sum() >= N // 3
    C = torch.full((M, N), math.nan, device=DEV)
    _linear(A, W, C, colscale=cs, bias=bias, bn=(a1, c1), act=act_id)
    y64, S = _ref64(A, W)
    rho = _rho_epilogue(C, y64, S, cs, bias, a1, c1, act_id)
    report("tc3 epilogue %s M=%d K=%d N=%d" % (act, M, K, N), rho=rho)
    assert rho <= RHO["model"], rho


# ------------------------------------------------------------------------------------------------
# 3. layout: padding columns, strided output, vector and scalar staging
# ------------------------------------------------------------------------------------------------
def _nan_table(rows, cols):
    return torch.full((rows, cols), math.nan, device=DEV)


@pytest.mark.parametrize("M,K,N", [(1000, 37, 129), (8065, 1001, 300)], ids=lambda s: str(s))
def test_linear_tc3_padding_and_staging_paths(M, K, N):
    """K % 8 != 0 with NaN in A's columns [K, lda) and W's columns [K, ldw) (and in a spare row after each), the output a
    strided window of a NaN-filled table: no NaN reaches the output, nothing outside [0, M) x [0, N) changes, and the
    vector staging path (lda % 4 == 0, 16-byte aligned A) and the scalar one (A one float off alignment; lda % 4 != 0)
    give bit-identical outputs, within RHO of float64."""
    A0, W0 = _operands("model", M, K, N, 400 + K)
    Wt = _nan_table(N + 1, K + 3)
    Wt[:N, :K] = W0
    W = Wt[:N, :K]
    lda = (K + 3) // 4 * 4 + 4
    As = {}
    t = _nan_table(M + 1, lda)
    As["vector"] = t[:M, :K]
    flat = torch.full(((M + 1) * lda + 1,), math.nan, device=DEV)
    As["offset"] = flat[1:1 + M * lda].view(M, lda)[:, :K]
    t = _nan_table(M + 1, lda - 1)
    As["lda%4"] = t[:M, :K]
    assert As["vector"].data_ptr() % 16 == 0 and As["offset"].data_ptr() % 16 == 4 and As["lda%4"].stride(0) % 4 == 3
    outs = {}
    for name, A in As.items():
        A.copy_(A0)
        Ct = _nan_table(M + 2, N + 7)
        C = Ct[1:1 + M, 3:3 + N]
        names = kernels_launched(lambda: _linear(A, W, C))
        assert ran(names, "gemm_tc3_kernel") and not ran(names, "linear_rows_kernel"), sorted(set(names))
        assert not torch.isnan(C).any(), name + ": NaN from the padding reached the output"
        inside = torch.zeros_like(Ct, dtype=torch.bool)
        inside[1:1 + M, 3:3 + N] = True
        assert bool(torch.isnan(Ct[~inside]).all()), name + ": wrote outside [0, M) x [0, N)"
        outs[name] = C.clone()
    assert torch.equal(outs["offset"], outs["vector"]), "scalar staging (misaligned A) differs from the vector path"
    assert torch.equal(outs["lda%4"], outs["vector"]), "scalar staging (lda % 4 != 0) differs from the vector path"
    y64, S = _ref64(A0, W0)
    rho = _rho(outs["vector"], y64, S)
    report("tc3 layout M=%d K=%d N=%d" % (M, K, N), rho=rho)
    assert rho <= RHO["model"], rho


# ------------------------------------------------------------------------------------------------
# 4. a row's result does not depend on the rows around it
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,N", [(505, 300), (544, 512)])
def test_linear_tc3_batch_independence(K, N):
    """1000 rows alone (M = 1000: one channel tile per CTA) and embedded at row 0, 37 and 8229 of an M = 20000 call (two
    channel tiles per CTA, another position inside the 128-row tile): bit-identical outputs."""
    X, W = _operands("model", 1000, K, N, 500 + N)
    alone = torch.empty(1000, N, device=DEV)
    _linear(X, W, alone)
    for off in (0, 37, 8229):
        big, _ = _operands("model", 20000, K, N, 600 + off)
        big[off:off + 1000] = X
        out = torch.empty(20000, N, device=DEV)
        _linear(big, W, out)
        assert torch.equal(out[off:off + 1000], alone), "rows at offset %d differ from the same rows alone" % off


# ------------------------------------------------------------------------------------------------
# 5. the coverage contract
# ------------------------------------------------------------------------------------------------
def _params(M=1000, K=505, N=300, **kw):
    from svnet_b200 import _native as nv
    p = nv.GemmParams()
    p.G, p.M, p.K, p.N, p.ldw, p.lda_g, p.ldc_g, p.groups_per_cloud = 1, M, K, N, K, K, N, 1
    for name, value in kw.items():
        setattr(p, name, value)
    return p


def _ws_bytes(p):
    from svnet_b200 import _native as nv
    return int(nv.lib().svnet_linear_workspace_bytes(ctypes.byref(p)))


def test_linear_tc3_coverage_contract(monkeypatch):
    """svnet_linear_workspace_bytes depends on (K, N) only, not on the row count; it is 0 outside 32 <= K <= 4096,
    32 <= N <= 512, for sign weights, VectorBN, G = 3, the c4 table layout and with SVNET_LINEAR_TC=0.  A c4 request with
    G = 1 raises with and without a workspace and writes nothing."""
    from svnet_b200 import _native as nv
    monkeypatch.delenv("SVNET_LINEAR_TC", raising=False)
    sizes = {M: _ws_bytes(_params(M=M)) for M in (1, 127, 10 ** 6)}
    assert sizes[1] > 0 and len(set(sizes.values())) == 1, sizes
    for K, N in ((32, 32), (4096, 512), (32, 512), (4096, 32)):
        assert _ws_bytes(_params(K=K, N=N)) > 0, (K, N)
    for K, N in ((31, 300), (4097, 300), (505, 31), (505, 513)):
        assert _ws_bytes(_params(K=K, N=N)) == 0, (K, N)
    for kw in (dict(sign_w=1), dict(vbn=1), dict(G=3, M=999), dict(c4=1)):
        assert _ws_bytes(_params(**kw)) == 0, kw
    monkeypatch.setenv("SVNET_LINEAR_TC", "0")
    assert _ws_bytes(_params()) == 0
    monkeypatch.delenv("SVNET_LINEAR_TC")

    M, K, N = 1000, 505, 300
    A, W = _operands("model", M, K, N, 700)
    C = _nan_table(M, 4 * N)
    with pytest.raises(RuntimeError, match="c4"):
        nv.linear_rows(A, K, 0, 1, M, K, W, N, C, 4 * N, 0, c4=True)
    nbytes = _ws_bytes(_params(M=M, K=K, N=N))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    p = _params(M=M, K=K, N=N, c4=1, A=A.data_ptr(), W=W.data_ptr(), C=C.data_ptr(), ldc_g=4 * N)
    with pytest.raises(RuntimeError, match="c4"):
        nv._call("svnet_linear_rows_ws", ctypes.byref(p), nv._ptr(ws), ctypes.c_size_t(nbytes), nv._stream())
    assert bool(torch.isnan(C).all()), "a refused c4 call wrote to its output"


# ------------------------------------------------------------------------------------------------
# 6. the per-cloud addend in the epilogue, through the fp part-segmentation head call
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pseg_net():
    return _pseg(40, 4400)[0]


@pytest.mark.parametrize("B,N", [(3, 1), (2, 5), (4, 31), (300, 31), (3, 32), (2, 33), (2, 129)])
def test_seg_head_fp_rowadd_small_clouds(pseg_net, B, N):
    """svnet_seg_head_fp_fwd adds conv8's per-cloud term in gemm_tc3_kernel's epilogue, advancing the cloud inside each
    32-row block: clouds of 1 to 129 points (N = 1: every row its own cloud; B = 300, N = 31: 73 row tiles, two channel
    tiles per CTA) within RHO_HEAD_CALL * M of float64."""
    from svnet_b200 import _native as nv
    net = pseg_net
    s_cat, v_cat, glob = _head_inputs(B, N, 4400 + 7 * B + N)
    layers = [(c.weight2d(), seq.bn_folded()) for c, seq in ((net.conv8[0], net.conv8), (net.conv9[0], net.conv9),
                                                              (net.conv10[0], net.conv10))]
    W11 = net.conv11.weight.detach()[:, :, 0].contiguous()
    out = []
    with torch.no_grad():
        names = kernels_launched(lambda: out.append(nv.seg_head_fp_fwd(nv.view_of(s_cat, v_cat), B, N, net.svfuse1.v2s.wz()[0],
                                                                       glob, layers, W11)))
        y64, Mref = _head64(net, s_cat, v_cat, glob, N)
    assert ran(names, "gemm_tc3_kernel") and not ran(names, "linear_rows_kernel"), sorted(set(names))
    y = out[0]
    assert tuple(y.shape) == (B, 50, N) and not torch.isnan(y).any()
    rho = float(((y.double() - y64).abs() / Mref).max())
    report("fp head rowadd B=%d N=%d" % (B, N), rho_call=rho)
    assert rho <= RHO_HEAD_CALL, rho
