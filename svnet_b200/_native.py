"""ctypes binding of libsvnet_b200.so (include/svnet_b200.h).

The product path has no CPU fallback: if the shared object is missing or a call fails, a
RuntimeError is raised.  torch is used only for device memory and the current stream.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SVNET_LIB") or os.path.join(_HERE, "libsvnet_b200.so")   # SVNET_LIB: developer A/B builds
_lib = None

ACT_NONE, ACT_LEAKY, ACT_RELU = 0, 1, 2
BN_EPS = 1e-5

c_int, c_long, c_float, c_void_p = ctypes.c_int, ctypes.c_long, ctypes.c_float, ctypes.c_void_p

EXPORTS = [
    "svnet_version", "svnet_last_error", "svnet_pack_sign", "svnet_fold_bn", "svnet_knn",
    "svnet_knn_ws", "svnet_knn_workspace_bytes", "svnet_knn_tc_stats", "svnet_svfuse_pool", "svnet_svfuse_pool_workspace",
    "svnet_binlinear_rows_ws", "svnet_binlinear_workspace_bytes", "svnet_binlinear_pool_ws",
    "svnet_binlinear_pool_workspace_bytes", "svnet_linear_rows_ws", "svnet_linear_workspace_bytes",
    "svnet_graph_feature_xyz", "svnet_graph_feature_sv", "svnet_gate_rows", "svnet_gate_edge", "svnet_gate_xyz",
    "svnet_edge_xyz_fwd", "svnet_svblock_edge_fwd", "svnet_rows_prep", "svnet_binlinear_rows", "svnet_linear_rows",
    "svnet_vector_bn_rows", "svnet_pool_rows", "svnet_head_fwd", "svnet_rotate_permute",
    "svnet_edge_tc_weight_bytes", "svnet_edge_tc_table_cols", "svnet_edge_tc_pack_w", "svnet_allgather_logits",
    "svnet_edge_fp_tc_weight_bytes", "svnet_edge_fp_tc_pack_w", "svnet_seg_head_fwd", "svnet_seg_head_workspace_bytes",
    "svnet_model_create", "svnet_model_workspace_bytes", "svnet_model_forward", "svnet_model_destroy",
    "svnet_model_seg_workspace_bytes", "svnet_model_forward_seg", "svnet_seg_head_fp_workspace_bytes", "svnet_seg_head_fp_fwd",
    "svnet_pack_sign_nz", "svnet_binlinear_rows_nz", "svnet_binlinear_pool_nz", "svnet_head_fwd_nz", "svnet_svblock_edge_fwd_nz",
    "svnet_seg_head_fwd_nz",
]


class View(ctypes.Structure):
    _fields_ = [("s", c_void_p), ("lds", c_int), ("Cs", c_int), ("v", c_void_p), ("ldv", c_int), ("xs", c_int),
                ("Cv", c_int)]


class EdgeXyzParams(ctypes.Structure):
    _fields_ = [("xyz", c_void_p), ("idx", c_void_p), ("B", c_int), ("N", c_int), ("k", c_int), ("nv", c_int),
                ("Winit", c_void_p), ("Wz", c_void_p), ("W1", c_void_p), ("bn1_a", c_void_p), ("bn1_c", c_void_p),
                ("W2", c_void_p), ("bn2_a", c_void_p), ("bn2_c", c_void_p), ("gate", c_void_p), ("Cout", c_int),
                ("Cvo", c_int), ("out", View)]


class EdgeParams(ctypes.Structure):
    _fields_ = [("inp", View), ("idx", c_void_p), ("B", c_int), ("N", c_int), ("k", c_int), ("binary", c_int),
                ("Wz", c_void_p), ("zscale", c_void_p), ("beta", c_void_p), ("W1b", c_void_p), ("scale1", c_void_p),
                ("Yab", c_void_p), ("W1q_t", c_void_p), ("bn1_a", c_void_p), ("bn1_c", c_void_p), ("Cout", c_int),
                ("PQ", c_void_p), ("bn2_a", c_void_p), ("bn2_c", c_void_p), ("gate", c_void_p), ("Cvo", c_int),
                ("out", View), ("dbg_bits", c_void_p), ("dbg_mask", c_void_p), ("W1tc", c_void_p), ("tab4", c_void_p)]


class GemmParams(ctypes.Structure):
    _fields_ = [("A", c_void_p), ("lda_g", c_long), ("lda_x", c_int), ("G", c_int), ("W", c_void_p), ("ldw", c_int),
                ("M", c_long), ("N", c_int), ("K", c_int), ("sign_w", c_int), ("colscale", c_void_p),
                ("bias", c_void_p), ("bn_a", c_void_p), ("bn_c", c_void_p), ("act", c_int), ("vbn", c_int),
                ("gate", c_void_p), ("groups_per_cloud", c_long), ("C", c_void_p), ("ldc_g", c_long),
                ("ldc_x", c_int), ("c4", c_int)]


class SegHeadParams(ctypes.Structure):
    _fields_ = [("sv", View), ("B", c_int), ("N", c_long), ("Wz1", c_void_p), ("zscale1", c_void_p),
                ("glob", c_void_p), ("ldg", c_int), ("Kc", c_int),
                ("beta8", c_void_p), ("W8c", c_void_p), ("W8p", c_void_p), ("scale8", c_void_p), ("bn8_a", c_void_p),
                ("bn8_c", c_void_p), ("C8", c_int), ("bits8", c_void_p), ("mask8", c_void_p), ("nvalid8", c_void_p),
                ("beta9", c_void_p), ("W9", c_void_p), ("scale9", c_void_p), ("bn9_a", c_void_p), ("bn9_c", c_void_p), ("C9", c_int),
                ("beta10", c_void_p), ("W10", c_void_p), ("scale10", c_void_p), ("bn10_a", c_void_p), ("bn10_c", c_void_p),
                ("C10", c_int), ("W11", c_void_p), ("parts", c_int), ("logits", c_void_p)]


class SegHeadFpParams(ctypes.Structure):
    _fields_ = [("sv", View), ("B", c_int), ("N", c_long), ("Wz1", c_void_p), ("glob", c_void_p), ("ldg", c_int), ("Kc", c_int),
                ("W8", c_void_p), ("bn8_a", c_void_p), ("bn8_c", c_void_p), ("C8", c_int),
                ("W9", c_void_p), ("bn9_a", c_void_p), ("bn9_c", c_void_p), ("C9", c_int),
                ("W10", c_void_p), ("bn10_a", c_void_p), ("bn10_c", c_void_p), ("C10", c_int),
                ("W11", c_void_p), ("parts", c_int), ("logits", c_void_p)]


class TensorRef(ctypes.Structure):           # svnet_tensor
    _fields_ = [("name", ctypes.c_char_p), ("data", c_void_p), ("numel", c_long)]


class HeadLayer(ctypes.Structure):
    _fields_ = [("Cout", c_int), ("W1b", c_void_p), ("beta", c_void_p), ("W", c_void_p), ("sign_w", c_int),
                ("scale", c_void_p), ("bias", c_void_p), ("bn_a", c_void_p), ("bn_c", c_void_p), ("act", c_int)]


class HeadParams(ctypes.Structure):
    _fields_ = [("x", c_void_p), ("ldx", c_int), ("K0", c_int), ("B", c_int), ("nlayers", c_int),
                ("layer", HeadLayer * 3), ("out", c_void_p), ("ldo", c_int)]


def lib():
    """Load the CUDA library; fail loudly when it is missing (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "svnet_b200: %s not found -- build it with `python -m svnet_b200.build` "
                "(there is no CPU/PyTorch fallback for the SV hot path)" % LIB_PATH)
        l = ctypes.CDLL(LIB_PATH)
        l.svnet_last_error.restype = ctypes.c_char_p
        l.svnet_knn_workspace_bytes.restype = ctypes.c_size_t
        l.svnet_svfuse_pool_workspace.restype = ctypes.c_size_t
        l.svnet_binlinear_workspace_bytes.restype = ctypes.c_size_t
        l.svnet_binlinear_pool_workspace_bytes.restype = ctypes.c_size_t
        l.svnet_linear_workspace_bytes.restype = ctypes.c_size_t
        l.svnet_edge_tc_weight_bytes.restype = ctypes.c_size_t
        l.svnet_edge_fp_tc_weight_bytes.restype = ctypes.c_size_t
        l.svnet_seg_head_workspace_bytes.restype = ctypes.c_size_t
        l.svnet_seg_head_fp_workspace_bytes.restype = ctypes.c_size_t
        l.svnet_model_workspace_bytes.restype = ctypes.c_size_t
        l.svnet_model_workspace_bytes.argtypes = [c_void_p, c_int, c_int]
        l.svnet_model_seg_workspace_bytes.restype = ctypes.c_size_t
        l.svnet_model_seg_workspace_bytes.argtypes = [c_void_p, c_int, c_int]
        l.svnet_model_destroy.restype = None
        l.svnet_model_destroy.argtypes = [c_void_p]
        for name in EXPORTS:
            getattr(l, name)  # AttributeError if the symbol is missing
        if l.svnet_version() != 3:
            raise RuntimeError("svnet_b200: ABI version mismatch")
        _lib = l
    return _lib


LAUNCHES = [0]        # C-ABI calls that enqueue kernels (bench.py reports it as gpu_launches)
TIMED = {}            # name -> list of (start_event, end_event), filled when PROFILE[0] is set
PROFILE = [None]      # None or a set of C-ABI names to bracket with CUDA events
ORDER = []            # (name, start_event, end_event) in call order while profiling


def _call(name, *args):
    """Invoke one C-ABI entry point; optionally bracket it with CUDA events on the launch stream."""
    fn = getattr(lib(), name)
    prof = PROFILE[0]
    if prof is not None and name in prof:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = fn(*args)
        e1.record()
        TIMED.setdefault(name, []).append((e0, e1))
        ORDER.append((name, e0, e1))
    else:
        rc = fn(*args)
    LAUNCHES[0] += 1
    if rc != 0:
        raise RuntimeError("%s failed (%d): %s" % (name, rc, lib().svnet_last_error().decode()))


def _stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return c_void_p(t.data_ptr()) if t is not None else c_void_p(0)


def _dev(t, dtype=torch.float32):
    if not t.is_cuda:
        raise RuntimeError("svnet_b200 kernels need CUDA tensors (got a %s tensor); there is no CPU path" % t.device)
    if t.dtype != dtype:
        raise TypeError("expected %s, got %s" % (dtype, t.dtype))
    return t


def view_of(s, v, Cs=None, Cv=None):
    """View over contiguous-last-dim tensors: s (..., >=Cs) rows; v (..., 3, >=Cv)."""
    vw = View()
    if s is not None:
        _dev(s)
        assert s.stride(-1) == 1
        vw.s, vw.lds, vw.Cs = s.data_ptr(), s.stride(-2) if s.dim() > 1 else s.shape[-1], (Cs if Cs is not None else s.shape[-1])
    else:
        vw.s, vw.lds, vw.Cs = 0, 0, 0
    if v is not None:
        _dev(v)
        assert v.stride(-1) == 1
        vw.v, vw.ldv, vw.xs, vw.Cv = v.data_ptr(), v.stride(-3) if v.dim() > 2 else 3 * v.stride(-2), v.stride(-2), (
            Cv if Cv is not None else v.shape[-1])
    else:
        vw.v, vw.ldv, vw.xs, vw.Cv = 0, 0, 0, 0
    return vw


# ------------------------------------------------------------------------------------------------
# thin wrappers (shapes validated again on the C side)
# ------------------------------------------------------------------------------------------------
def pack_sign(W2d):
    """W (rows, K) float -> bits_t (Kw, rows) int32 (word-major); raises on exact-zero weights (see pack_sign_nz)."""
    W2d = _dev(W2d)
    assert W2d.dim() == 2 and W2d.stride(1) == 1
    rows, K = W2d.shape
    bits = torch.empty(((K + 31) // 32, rows), dtype=torch.int32, device=W2d.device)
    zc = torch.zeros(1, dtype=torch.int32, device=W2d.device)
    _call("svnet_pack_sign", _ptr(W2d), c_int(rows), c_int(K), c_int(W2d.stride(0)), _ptr(bits), _ptr(zc),
                                 _stream())
    if int(zc.item()) != 0:
        raise NotImplementedError("binarised weight contains exact zeros (sign(0)=0 plane not supported)")
    return bits


def pack_sign_nz(W2d):
    """W (rows, K) float -> (bits_t, nz_t): the sign plane and, when W holds an exact zero (-0.0 included), its non-zero
    plane (Kw, rows) int32; nz_t is None for a zero-free W, whose consumers then run their +-1 kernels."""
    W2d = _dev(W2d)
    assert W2d.dim() == 2 and W2d.stride(1) == 1
    rows, K = W2d.shape
    bits = torch.empty(((K + 31) // 32, rows), dtype=torch.int32, device=W2d.device)
    nz = torch.empty_like(bits)
    zc = torch.zeros(1, dtype=torch.int32, device=W2d.device)
    _call("svnet_pack_sign_nz", _ptr(W2d), c_int(rows), c_int(K), c_int(W2d.stride(0)), _ptr(bits), _ptr(nz), _ptr(zc),
          _stream())
    return bits, (nz if int(zc.item()) != 0 else None)


def fold_bn(bn):
    """nn.BatchNorm1d (eval) -> (a, c) with y = x*a + c."""
    w, b, m, var = (_dev(t.detach()) for t in (bn.weight, bn.bias, bn.running_mean, bn.running_var))
    C = w.numel()
    a = torch.empty(C, dtype=torch.float32, device=w.device)
    c = torch.empty_like(a)
    _call("svnet_fold_bn", _ptr(w), _ptr(b), _ptr(m), _ptr(var), c_float(bn.eps), c_int(C), _ptr(a), _ptr(c),
                               _stream())
    return a, c


def knn(view, B, N, k, want64=False, want32=True):
    dev = torch.device("cuda", torch.cuda.current_device())
    i32 = torch.empty((B, N, k), dtype=torch.int32, device=dev) if want32 else None
    i64 = torch.empty((B, N, k), dtype=torch.int64, device=dev) if want64 else None
    # scratch for the tensor-core filter (operand planes + norms); 0 bytes -> CUDA-core kernel
    nbytes = int(lib().svnet_knn_workspace_bytes(ctypes.byref(view), c_int(B), c_int(N), c_int(k)))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev) if nbytes > 0 else None
    _call("svnet_knn_ws", ctypes.byref(view), c_int(B), c_int(N), c_int(k), _ptr(i32), _ptr(i64), _ptr(ws),
          ctypes.c_size_t(nbytes), _stream())
    if nbytes > 0:
        LAUNCHES[0] += 2     # tensor-core path = pack + tcgen05 + finish kernels
    return i32, i64


def graph_feature_xyz(xyz, idx64, nv):
    B, N, k = idx64.shape
    out = torch.empty((B, N, k, 3, nv), dtype=torch.float32, device=xyz.device)
    _call("svnet_graph_feature_xyz", _ptr(_dev(xyz)), _ptr(_dev(idx64, torch.int64)), c_int(B), c_int(N), c_int(k),
                                         c_int(nv), _ptr(out), _stream())
    return out


def graph_feature_sv(s, v, idx64):
    B, N, k = idx64.shape
    Cs, Cv = s.shape[-1], v.shape[-1]
    sf = torch.empty((B, N, k, 2 * Cs), dtype=torch.float32, device=s.device)
    vf = torch.empty((B, N, k, 3, 2 * Cv), dtype=torch.float32, device=s.device)
    _call("svnet_graph_feature_sv", _ptr(_dev(s)), _ptr(_dev(v)), _ptr(_dev(idx64, torch.int64)), c_int(B), c_int(N),
                                        c_int(k), c_int(Cs), c_int(Cv), _ptr(sf), _ptr(vf), _stream())
    return sf, vf


def gate_rows(s2d, lds, Cs, B, rows, G1, G2, out=None):
    H, Co = G1.shape[0], G2.shape[0]
    gate = out if out is not None else torch.empty((B, Co), dtype=torch.float32, device=s2d.device)
    _call("svnet_gate_rows", _ptr(_dev(s2d)), c_int(lds), c_int(Cs), c_int(B), c_int(rows), _ptr(_dev(G1)),
                                 _ptr(_dev(G2)), c_int(H), c_int(Co), _ptr(gate), _stream())
    return gate


def gate_edge(view, idx32, B, N, k, G1, G2):
    H, Co = G1.shape[0], G2.shape[0]
    gate = torch.empty((B, Co), dtype=torch.float32, device=idx32.device)
    _call("svnet_gate_edge", ctypes.byref(view), _ptr(_dev(idx32, torch.int32)), c_int(B), c_int(N), c_int(k),
                                 _ptr(_dev(G1)), _ptr(_dev(G2)), c_int(H), c_int(Co), _ptr(gate), _stream())
    return gate


def gate_xyz(xyz, idx32, nv, Winit, G1, G2):
    B, N, k = idx32.shape
    H, Co = G1.shape[0], G2.shape[0]
    gate = torch.empty((B, Co), dtype=torch.float32, device=xyz.device)
    _call("svnet_gate_xyz", _ptr(_dev(xyz)), _ptr(_dev(idx32, torch.int32)), c_int(B), c_int(N), c_int(k), c_int(nv),
                                _ptr(_dev(Winit)), _ptr(_dev(G1)), _ptr(_dev(G2)), c_int(H), c_int(Co), _ptr(gate),
                                _stream())
    return gate


def edge_xyz_fwd(params):
    _call("svnet_edge_xyz_fwd", ctypes.byref(params), _stream())


def svblock_edge_fwd(params, W1nz=None):
    """``W1nz``: non-zero plane of a binary layer's ternary linear1 weight (pack_sign_nz), or None."""
    if W1nz is None:
        _call("svnet_svblock_edge_fwd", ctypes.byref(params), _stream())
    else:
        _call("svnet_svblock_edge_fwd_nz", ctypes.byref(params), _ptr(W1nz), _stream())


def edge_tc_weight_bytes(Cs, Cv, Cout, Cvo, k):
    """0 when the tensor-core edge kernel does not cover the layer (svnet_edge_tc_weight_bytes)."""
    return int(lib().svnet_edge_tc_weight_bytes(c_int(Cs), c_int(Cv), c_int(Cout), c_int(Cvo), c_int(k)))


def edge_tc_pack_w(W1, Cs, Cv):
    """conv.linear1.weight (Cout, 2Cs + 6Cv) -> e4m3 sign bytes in the UMMA operand layout of csrc/edge_tc.cu."""
    W1 = _dev(W1)
    assert W1.dim() == 2 and W1.stride(1) == 1
    Cout = W1.shape[0]
    nbytes = (2 * Cs + 8 * Cv + 31) // 32 * 32 * 128
    out = torch.empty(nbytes, dtype=torch.uint8, device=W1.device)
    _call("svnet_edge_tc_pack_w", _ptr(W1), c_int(W1.stride(0)), c_int(Cs), c_int(Cv), c_int(Cout), _ptr(out), _stream())
    return out


def edge_fp_tc_weight_bytes(Cs, Cv, Cout, Cvo, k):
    """0 when the full-precision tensor-core edge kernel does not cover the layer (svnet_edge_fp_tc_weight_bytes)."""
    return int(lib().svnet_edge_fp_tc_weight_bytes(c_int(Cs), c_int(Cv), c_int(Cout), c_int(Cvo), c_int(k)))


def edge_fp_tc_pack_w(W1, Cs, Cv, nbytes):
    """conv.linear1.weight (Cout, 2Cs + 6Cv), full precision -> three bf16 weight planes of csrc/edge_fp_tc.cu."""
    W1 = _dev(W1)
    assert W1.dim() == 2 and W1.stride(1) == 1
    out = torch.empty(nbytes, dtype=torch.uint8, device=W1.device)
    _call("svnet_edge_fp_tc_pack_w", _ptr(W1), c_int(W1.stride(0)), c_int(Cs), c_int(Cv), c_int(W1.shape[0]), _ptr(out), _stream())
    return out


def seg_head_fwd(view, B, N, Wz1, zscale1, glob, layers, W11, sv_bits=None):
    """svnet_seg_head_fwd: conv8 -> conv9 -> conv10 -> conv11 of SV_DGCNN_PSEG in one call.  ``layers`` = three dicts
    (beta, bits (conv8: (bits of the per-cloud part, bits of the per-point part)), nz (the same for the non-zero planes,
    None where the weights are +-1), scale, bn (a, c), Cout);
    ``sv_bits`` = conv8's per-point (bits, mask, nvalid) computed ahead of time, or None.  Returns (B, parts, N)."""
    glob, W11 = _dev(glob), _dev(W11)
    p = SegHeadParams()
    p.sv, p.B, p.N = view, B, N
    p.Wz1, p.zscale1 = _ptr(Wz1).value, _ptr(zscale1).value
    p.glob, p.ldg, p.Kc = glob.data_ptr(), glob.stride(0), glob.shape[1]
    l8, l9, l10 = layers
    p.beta8, p.W8c, p.W8p = l8["beta"].data_ptr(), l8["bits"][0].data_ptr(), l8["bits"][1].data_ptr()
    p.scale8, p.bn8_a, p.bn8_c, p.C8 = l8["scale"].data_ptr(), l8["bn"][0].data_ptr(), l8["bn"][1].data_ptr(), l8["Cout"]
    if sv_bits is not None:
        p.bits8, p.mask8, p.nvalid8 = (t.data_ptr() for t in sv_bits)
    p.beta9, p.W9 = l9["beta"].data_ptr(), l9["bits"].data_ptr()
    p.scale9, p.bn9_a, p.bn9_c, p.C9 = l9["scale"].data_ptr(), l9["bn"][0].data_ptr(), l9["bn"][1].data_ptr(), l9["Cout"]
    p.beta10, p.W10 = l10["beta"].data_ptr(), l10["bits"].data_ptr()
    p.scale10, p.bn10_a, p.bn10_c, p.C10 = l10["scale"].data_ptr(), l10["bn"][0].data_ptr(), l10["bn"][1].data_ptr(), l10["Cout"]
    p.W11, p.parts = W11.data_ptr(), W11.shape[0]
    out = torch.empty((B, W11.shape[0], N), dtype=torch.float32, device=glob.device)
    p.logits = out.data_ptr()
    nbytes = int(lib().svnet_seg_head_workspace_bytes(ctypes.byref(p)))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=glob.device)
    nzs = list(l8.get("nz") or (None, None)) + [l9.get("nz"), l10.get("nz")]
    if all(z is None for z in nzs):
        _call("svnet_seg_head_fwd", ctypes.byref(p), _ptr(ws), ctypes.c_size_t(nbytes), _stream())
    else:
        _call("svnet_seg_head_fwd_nz", ctypes.byref(p), *[_ptr(z) for z in nzs], _ptr(ws), ctypes.c_size_t(nbytes), _stream())
    LAUNCHES[0] += 11        # kernels behind the one call (sign-packs, binarised linears, GEMM, transpose)
    return out


def seg_head_fp_fwd(view, B, N, Wz1, glob, layers, W11):
    """svnet_seg_head_fp_fwd: conv8 -> conv9 -> conv10 -> conv11 of the full-precision SV_DGCNN_PSEG in one call.  ``view`` =
    (s_cat, v_cat), svfuse1's input; ``layers`` = three (W (Cout, K) contiguous, (bn_a, bn_c)) for conv8 / conv9 / conv10, conv8's
    W over [glob | svfuse1 rows].  Returns (B, parts, N), or None when the per-point conv8 is not covered by the tensor-core linear."""
    glob, W11 = _dev(glob), _dev(W11)
    p = SegHeadFpParams()
    p.sv, p.B, p.N, p.Wz1 = view, B, N, _dev(Wz1).data_ptr()
    p.glob, p.ldg, p.Kc = glob.data_ptr(), glob.stride(0), glob.shape[1]
    (W8, bn8), (W9, bn9), (W10, bn10) = layers
    p.W8, p.bn8_a, p.bn8_c, p.C8 = _dev(W8).data_ptr(), bn8[0].data_ptr(), bn8[1].data_ptr(), W8.shape[0]
    p.W9, p.bn9_a, p.bn9_c, p.C9 = _dev(W9).data_ptr(), bn9[0].data_ptr(), bn9[1].data_ptr(), W9.shape[0]
    p.W10, p.bn10_a, p.bn10_c, p.C10 = _dev(W10).data_ptr(), bn10[0].data_ptr(), bn10[1].data_ptr(), W10.shape[0]
    p.W11, p.parts = W11.data_ptr(), W11.shape[0]
    nbytes = int(lib().svnet_seg_head_fp_workspace_bytes(ctypes.byref(p)))
    if nbytes == 0:
        return None
    out = torch.empty((B, W11.shape[0], N), dtype=torch.float32, device=glob.device)
    p.logits = out.data_ptr()
    ws = torch.empty(nbytes, dtype=torch.uint8, device=glob.device)
    _call("svnet_seg_head_fp_fwd", ctypes.byref(p), _ptr(ws), ctypes.c_size_t(nbytes), _stream())
    # kernels behind the one call: svfuse1's rows, per linear pack + tensor-core GEMM (or one CUDA-core kernel), transpose
    Kp = view.Cs + 3 * view.Cv
    shapes = [(p.Kc, p.C8), (Kp, p.C8), (p.C8, p.C9), (p.C9, p.C10), (p.C10, p.parts)]
    LAUNCHES[0] += 1 + sum(2 if linear_tc_bytes(K, N) else 1 for K, N in shapes)
    return out


def model_create(kind, k, binary, num_class, state_dict):
    """svnet_model_create from a state_dict of CUDA fp32 tensors ('module.' prefixes are stripped); returns the handle."""
    items = [(n[7:] if n.startswith("module.") else n, t) for n, t in state_dict.items() if t.dtype == torch.float32]
    keep = [t.detach().contiguous() for _, t in items]
    arr = (TensorRef * len(items))()
    for i, ((n, _), t) in enumerate(zip(items, keep)):
        _dev(t)
        arr[i].name, arr[i].data, arr[i].numel = n.encode(), t.data_ptr(), t.numel()
    h = c_void_p()
    _call("svnet_model_create", kind.encode(), c_int(k), c_int(1 if binary else 0), c_int(num_class), arr, c_int(len(items)),
          _stream(), ctypes.byref(h))
    return h


def model_workspace_bytes(h, B, N):
    return int(lib().svnet_model_workspace_bytes(h, B, N))


def model_forward(h, x, logits, ws):
    B, _, N = x.shape
    _call("svnet_model_forward", h, _ptr(_dev(x)), c_int(B), c_int(N), _ptr(logits), _ptr(ws), ctypes.c_size_t(ws.numel()), _stream())


def model_seg_workspace_bytes(h, B, N):
    return int(lib().svnet_model_seg_workspace_bytes(h, B, N))


def model_forward_seg(h, x, label, logits, ws):
    B, _, N = x.shape
    _call("svnet_model_forward_seg", h, _ptr(_dev(x)), _ptr(_dev(label)), c_int(B), c_int(N), _ptr(logits), _ptr(ws),
          ctypes.c_size_t(ws.numel()), _stream())


def model_destroy(h):
    lib().svnet_model_destroy(h)


def edge_tc_table_cols(Cv, Cvo):
    return int(lib().svnet_edge_tc_table_cols(c_int(Cv), c_int(Cvo)))


def rows_prep(view, rows, Wz=None, zscale=None, beta=None, u_out=None, ldu=0, z_out=None, want_bits=False,
              z_in=None):
    K = view.Cs + 3 * view.Cv
    dev = torch.device("cuda", torch.cuda.current_device())
    bits = mask = nvalid = None
    if want_bits:
        Kw = (K + 31) // 32
        bits = torch.empty((rows, Kw), dtype=torch.int32, device=dev)
        mask = torch.empty((rows, Kw), dtype=torch.int32, device=dev)
        nvalid = torch.empty((rows,), dtype=torch.int32, device=dev)
    _call("svnet_rows_prep", ctypes.byref(view), c_long(rows), _ptr(Wz), _ptr(zscale), _ptr(z_in), _ptr(beta), _ptr(u_out),
                                 c_int(ldu), _ptr(z_out), _ptr(bits), _ptr(mask), _ptr(nvalid), _stream())
    return bits, mask, nvalid


def binlinear_rows(bits, mask, nvalid, K, W1b, Cout, scale=None, bias=None, bn=None, act=ACT_NONE, cloud_dot=None,
                   rows_per_cloud=1, out=None, ldo=None, out_i32=False, W1nz=None):
    """``W1nz``: non-zero plane of ternary weights (pack_sign_nz), or None (+-1 weights)."""
    rows = bits.shape[0]
    res_i32 = None
    if out_i32:
        res_i32 = torch.empty((rows, Cout), dtype=torch.int32, device=bits.device)
    elif out is None:
        out = torch.empty((rows, Cout), dtype=torch.float32, device=bits.device)
        ldo = Cout
    bn_a, bn_c = bn if bn is not None else (None, None)
    # scratch for the expanded weights of the tensor-core path; 0 bytes -> popcount kernel
    nbytes = int(lib().svnet_binlinear_workspace_bytes(c_long(rows), c_int(K), c_int(Cout)))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=bits.device) if nbytes > 0 else None
    name, wargs = ("svnet_binlinear_rows_ws", (_ptr(W1b),)) if W1nz is None else ("svnet_binlinear_rows_nz", (_ptr(W1b), _ptr(W1nz)))
    _call(name, _ptr(bits), _ptr(mask), _ptr(nvalid), c_long(rows), c_int(K), *wargs, c_int(Cout), _ptr(scale), _ptr(bias),
          _ptr(bn_a), _ptr(bn_c), c_int(act), _ptr(cloud_dot), c_long(rows_per_cloud), _ptr(out), c_int(ldo or 0),
          _ptr(res_i32), _ptr(ws), ctypes.c_size_t(nbytes), _stream())
    if nbytes > 0:
        LAUNCHES[0] += 1
    return res_i32 if out_i32 else out


def binlinear_pool_workspace(rows, K, Cout, rows_per_cloud):
    return int(lib().svnet_binlinear_pool_workspace_bytes(c_long(rows), c_int(K), c_int(Cout), c_long(rows_per_cloud)))


def binlinear_pool(bits, mask, K, W1b, Cout, scale, bn, rows_per_cloud, max_out, mean_out, ldo, W1nz=None):
    """Binarised Linear -> BN -> LeakyReLU -> per-cloud max / mean, fused (tensor-core path only); ``W1nz`` as in
    binlinear_rows."""
    rows = bits.shape[0]
    nbytes = binlinear_pool_workspace(rows, K, Cout, rows_per_cloud)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=bits.device)
    name, wargs = ("svnet_binlinear_pool_ws", (_ptr(W1b),)) if W1nz is None else ("svnet_binlinear_pool_nz", (_ptr(W1b), _ptr(W1nz)))
    _call(name, _ptr(bits), _ptr(mask), c_long(rows), c_int(K), *wargs, c_int(Cout), _ptr(scale),
          _ptr(bn[0]), _ptr(bn[1]), c_long(rows_per_cloud), _ptr(max_out), _ptr(mean_out), c_int(ldo), _ptr(ws),
          ctypes.c_size_t(nbytes), _stream())
    LAUNCHES[0] += 2


def linear_rows(A, lda_g, lda_x, G, M, K, W, N, C, ldc_g, ldc_x, sign_w=False, colscale=None, bias=None, bn=None,
                act=ACT_NONE, vbn=False, gate=None, groups_per_cloud=1, c4=False):
    """Raw generic linear; A and C are tensors whose data_ptr() is the first element addressed."""
    p = GemmParams()
    p.A, p.lda_g, p.lda_x, p.G = A.data_ptr(), lda_g, lda_x, G
    p.W, p.ldw = _dev(W).data_ptr(), W.stride(0)
    p.M, p.N, p.K = M, N, K
    p.sign_w = 1 if sign_w else 0
    p.colscale = colscale.data_ptr() if colscale is not None else 0
    p.bias = bias.data_ptr() if bias is not None else 0
    p.bn_a, p.bn_c = (bn[0].data_ptr(), bn[1].data_ptr()) if bn is not None else (0, 0)
    p.act = act
    p.vbn = 1 if vbn else 0
    p.gate = gate.data_ptr() if gate is not None else 0
    p.groups_per_cloud = groups_per_cloud
    p.C, p.ldc_g, p.ldc_x = C.data_ptr(), ldc_g, ldc_x
    p.c4 = 1 if c4 else 0
    # scratch for the split weights of the three-plane tensor-core path (plain fp32 linears over many rows)
    nbytes = int(lib().svnet_linear_workspace_bytes(ctypes.byref(p)))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=C.device) if nbytes > 0 else None
    _call("svnet_linear_rows_ws", ctypes.byref(p), _ptr(ws), ctypes.c_size_t(nbytes), _stream())
    if nbytes > 0:
        LAUNCHES[0] += 1


def linear_tc_bytes(K, N):
    """Scratch of the three-plane tensor-core fp linear for a plain (K -> N) layer; 0 when it does not cover the shape."""
    p = GemmParams()
    p.G, p.M, p.K, p.N, p.ldw = 1, 1, K, N, K
    return int(lib().svnet_linear_workspace_bytes(ctypes.byref(p)))


def vector_bn_rows(v, bn_a, bn_c):
    C = v.shape[-1]
    rows = v.numel() // (3 * C)
    out = torch.empty_like(v)
    _call("svnet_vector_bn_rows", _ptr(_dev(v)), c_long(rows), c_int(C), _ptr(bn_a), _ptr(bn_c), _ptr(out),
                                      _stream())
    return out


def svfuse_pool(v3, B, rows_per_cloud, Wz, zscale, max_out, mean_out, ldo):
    """v2s(v) of SVFuse reduced straight to per-cloud max / mean (no fused table in HBM)."""
    Cv = v3.shape[-1]
    view = view_of(None, v3)
    nbytes = int(lib().svnet_svfuse_pool_workspace(c_int(B), c_int(Cv), c_long(rows_per_cloud)))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=v3.device)
    _call("svnet_svfuse_pool", ctypes.byref(view), c_int(B), c_long(rows_per_cloud), _ptr(_dev(Wz)), _ptr(zscale),
          _ptr(max_out), _ptr(mean_out), c_int(ldo), _ptr(ws), ctypes.c_size_t(nbytes), _stream())
    LAUNCHES[0] += 1


def pool_rows(x, ld, C, B, rows, want_max=True, want_mean=False, max_out=None, mean_out=None, ldo=None):
    dev = x.device
    if want_max and max_out is None:
        max_out = torch.empty((B, C), dtype=torch.float32, device=dev)
    if want_mean and mean_out is None:
        mean_out = torch.empty((B, C), dtype=torch.float32, device=dev)
    if ldo is None:
        ldo = C
    _call("svnet_pool_rows", _ptr(_dev(x)), c_int(ld), c_int(C), c_int(B), c_long(rows), _ptr(max_out),
                                 _ptr(mean_out), c_int(ldo), _stream())
    return max_out, mean_out


def head_fwd(x2d, layers):
    """layers: list of dicts(Cout, W1b, W1nz (non-zero plane or None), beta, W, sign_w, scale, bias, bn=(a, c), act)
    -> (B, Cout_last)."""
    B, K0 = x2d.shape
    p = HeadParams()
    p.x, p.ldx, p.K0, p.B, p.nlayers = _dev(x2d).data_ptr(), x2d.stride(0), K0, B, len(layers)
    keep = []
    for i, L in enumerate(layers):
        hl = p.layer[i]
        hl.Cout = L["Cout"]
        for name in ("W1b", "beta", "W", "scale", "bias"):
            t = L.get(name)
            keep.append(t)
            setattr(hl, name, t.data_ptr() if t is not None else 0)
        bn = L.get("bn")
        hl.bn_a, hl.bn_c = (bn[0].data_ptr(), bn[1].data_ptr()) if bn is not None else (0, 0)
        hl.sign_w = 1 if L.get("sign_w") else 0
        hl.act = L.get("act", ACT_NONE)
    out = torch.empty((B, layers[-1]["Cout"]), dtype=torch.float32, device=x2d.device)
    p.out, p.ldo = out.data_ptr(), out.shape[1]
    nzs = [L.get("W1nz") for L in layers]
    if all(z is None for z in nzs):
        _call("svnet_head_fwd", ctypes.byref(p), _stream())
    else:
        arr = (c_void_p * 3)(*[z.data_ptr() if z is not None else None for z in nzs + [None] * (3 - len(nzs))])
        _call("svnet_head_fwd_nz", ctypes.byref(p), arr, _stream())
    return out


def rotate_permute(pts, R=None):
    """pts (B,N,3) [, R (B,3,3)] -> (B,3,N) = (pts @ R).permute(0,2,1)"""
    B, N, _ = pts.shape
    out = torch.empty((B, 3, N), dtype=torch.float32, device=pts.device)
    _call("svnet_rotate_permute", _ptr(_dev(pts.contiguous())), _ptr(R.contiguous() if R is not None else None),
          c_int(B), c_int(N), _ptr(out), _stream())
    return out
