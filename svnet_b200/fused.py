"""Fused layer drivers shared by the SV model classes: they wire module parameters (packed once)
into the C-ABI parameter blocks of the fused kernels.  No arithmetic happens here.
"""
import os
import threading

import torch

from . import _native as nv


MAX_POINTS_PER_PASS = int(os.environ.get("SVNET_MAX_POINTS", 1 << 19))
SIDE_STREAM = os.environ.get("SVNET_SIDE_STREAM", "1") != "0"
CONCURRENT_HALVES = os.environ.get("SVNET_TWO_STREAMS", "1") != "0"
N_SPLIT = max(2, int(os.environ.get("SVNET_STREAMS", "4")))      # sub-batches that run concurrently
NATIVE_FORWARD = os.environ.get("SVNET_NATIVE_FORWARD", "1") != "0"   # whole-model C entry behind model(x) where it covers the call
TABLE_AUX = os.environ.get("SVNET_TABLE_AUX", "1") != "0"          # per-point tables next to the kNN kernels also inside sub-batches
MIN_CLOUDS = max(1, int(os.environ.get("SVNET_MIN_CLOUDS", "8")))  # ... of at least this many clouds
MIN_POINTS = max(1, int(os.environ.get("SVNET_MIN_POINTS", "16384")))  # ... and points (measured on B200: 32 x 1024 as 2 x 16 clouds)
_SIDE = {}
class _State(threading.local):       # per thread: DataParallel drives one forward per device thread
    in_sub_batch = False
    sub_index = 0


_STATE = _State()


def _side_stream(dev, which=0):
    """Auxiliary CUDA streams per device: 0 = graph-independent tables, 1.. = the concurrent sub-batches."""
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), which)
    if key not in _SIDE:
        _SIDE[key] = torch.cuda.Stream(device=dev)
    return _SIDE[key]


def native_forward(model, kind, x, extra=None):
    """Run ``model`` (SV_DGCNN_CLS / SV_DGCNN_PSEG) through the whole-model C entry (csrc/model.cu: svnet_model_forward[_seg])
    when it covers the call, else return None.  The handle is built once per device from the module's own tensors
    (``_Cached``: rebuilt after load_state_dict / .to(); nn.DataParallel replicas share their source's handles) and makes
    the same library calls as the Python path below -- identical bits -- without Python between the kernels: an eager
    ``model(data)``, which is how the reference's eval loops call it (main_cls_dgcnn.py:238), is no longer bound by the
    host's launch rate (B = 32: 1.72 -> 1.07 ms).  Covered: k = 20, and k = 40 for the binary models and both part-segmentation
    models."""
    if not NATIVE_FORWARD or not x.is_cuda or x.dtype != torch.float32 or x.dim() != 3 or x.shape[1] != 3:
        return None
    B, _, N = x.shape
    k, binary = model.k, bool(model.binary)
    pseg = kind == "SV_DGCNN_PSEG"
    if B < 1 or N < 64 or N > 4096 or not (k == 20 or (k == 40 and (binary or pseg))):
        return None
    if x.device.index != torch.cuda.current_device():
        with torch.cuda.device(x.device):
            return native_forward(model, kind, x, extra)
    # the C entry runs edge layers 2..4 on the tensor-core kernels only; where a switch (SVNET_EDGE_TC=0,
    # SVNET_VLINEAR_FP_TC=0, ...) takes them off, the module path below picks the kernel
    covered = nv.edge_tc_weight_bytes if binary else nv.edge_fp_tc_weight_bytes
    for blk in (model.conv2, model.conv3, model.conv4):
        if covered(blk.in_dims[0] // 2, blk.in_dims[1] // 2, blk.out_dims[0], blk.out_dims[1], k) == 0:
            return None
    # ... and the full-precision part-segmentation head's per-point conv8 (svfuse1's Cs + 3Cv channels -> C8), which carries
    # the per-cloud term, on the tensor-core fp linear (SVNET_LINEAR_TC=0 takes it off); its other linears take either kernel
    if pseg and not binary:
        cs, cv = model.conv5.in_dims
        if nv.linear_tc_bytes(cs + 3 * cv, model.conv8[0].out_channels) == 0:
            return None
    from .native_model import NativeModel
    names = [n for n, t in model.state_dict().items() if t.dtype == torch.float32] if "_sv_native_names" not in model.__dict__ \
        else model.__dict__["_sv_native_names"]
    model.__dict__["_sv_native_names"] = names
    ncls = model.conv11.out_channels if pseg else model.linear3.out_features

    def build():
        from .sv_layers import _resolve
        sd = {n: _resolve(model, n).detach() for n in names}
        return NativeModel(kind, sd, k=k, binary=binary, num_class=ncls, device=x.device)
    handle = model._packed("native", tuple(names), build)
    per = max(1, MAX_POINTS_PER_PASS // N)
    outs = []
    for lo in range(0, B, per):           # bounded scratch: large batches run in passes
        xc = x[lo:lo + per].contiguous()
        outs.append(handle(xc) if extra is None else handle(xc, extra[lo:lo + per]))
    return outs[0] if len(outs) == 1 else torch.cat(outs, dim=0)


def aux_stream(dev):
    """A side stream for work that does not depend on the caller's latest kernels (e.g. the part-seg head's per-point
    sign words next to its per-cloud branch): one per concurrent sub-batch, so that sub-batches do not meet on it.
    None when side streams are switched off."""
    if not SIDE_STREAM:
        return None
    return _side_stream(dev, 16 + _STATE.sub_index) if _STATE.in_sub_batch else _side_stream(dev, 15)


def chunked(impl, x, extras=(), hooks=False):
    """Run ``impl(x_chunk, *extras_chunk)`` over cloud sub-batches so that the per-pass tables stay
    bounded (B*N <= MAX_POINTS_PER_PASS points; clouds are independent in eval mode, SURVEY.md 8(e)).
    A batch that fits one pass is split into up to N_SPLIT sub-batches (at least 8 clouds each) that run on
    their own CUDA streams: kernels whose grids leave SMs idle (the tensor-core kNN, the per-cloud
    gate / head kernels) overlap with the other sub-batches' kernels.  Test hooks (forced indices / recording) disable both."""
    if x.is_cuda and x.device.index != torch.cuda.current_device():
        # scratch tensors and the launch stream follow the current device: make it the input's device
        with torch.cuda.device(x.device):
            return chunked(impl, x, extras, hooks)
    B, N = x.shape[0], x.shape[-1]
    per = max(1, MAX_POINTS_PER_PASS // max(N, 1))
    if hooks:
        return impl(x, *extras)
    if B <= per:
        if CONCURRENT_HALVES and B >= 16 and x.is_cuda and not _STATE.in_sub_batch:
            return _two_streams(impl, x, extras)
        return impl(x, *extras)
    outs = []
    for lo in range(0, B, per):
        outs.append(impl(x[lo:lo + per].contiguous(), *[e[lo:lo + per].contiguous() for e in extras]))
    return torch.cat(outs, dim=0)


def split_bounds(B, N=None):
    """Contiguous sub-batch boundaries: up to N_SPLIT sub-batches of at least MIN_CLOUDS clouds (and, when the cloud
    size N is given, of at least MIN_POINTS points)."""
    n = max(1, min(N_SPLIT, B // MIN_CLOUDS))
    if N is not None:
        n = max(1, min(n, (B * N) // MIN_POINTS))
    return [B * i // n for i in range(n + 1)]


def _two_streams(impl, x, extras):
    dev = x.device
    cur = torch.cuda.current_stream()
    B = x.shape[0]
    bounds = split_bounds(B, x.shape[-1])
    parts = [(x[lo:hi].contiguous(), [e[lo:hi].contiguous() for e in extras]) for lo, hi in zip(bounds[:-1], bounds[1:])]
    outs = []
    _STATE.in_sub_batch = True
    try:
        for i, (xc, ec) in enumerate(parts):
            st = _side_stream(dev, 1 + i)
            st.wait_stream(cur)
            _STATE.sub_index = i
            with torch.cuda.stream(st):
                y = impl(xc, *ec)
            y.record_stream(cur)
            outs.append((st, y))
    finally:
        _STATE.in_sub_batch = False
    for st, _ in outs:
        cur.wait_stream(st)
    return torch.cat([y for _, y in outs], dim=0)


def _mview(s_out, v_out):
    return nv.view_of(s_out, v_out)


def first_edge_layer(xyz, B, N, k, nvec, init_scalar, blk, s_out, v_out, idx32=None):
    """get_graph_feature[_cross] + init_scalar + SVBlock(FP) + svpool (sv_dgcnn_cls.py:49-53,
    sv_pointnet_cls.py:35-39).  xyz (B*N, 3) contiguous.  Writes pooled (s, v) into the given
    slices and returns the int32 kNN indices (B, N, k)."""
    if blk.binary:
        raise NotImplementedError("the first SVBlock is full precision in every SV model")
    if idx32 is None:
        idx32, _ = nv.knn(nv.view_of(xyz, None), B, N, k)
    Winit, _ = init_scalar.wz()
    Wz, _ = blk.v2s.wz()
    G1, G2 = blk.gate_weights()
    gate = nv.gate_xyz(xyz, idx32, nvec, Winit, G1, G2)
    a1, c1 = blk.bn1_folded()
    a2, c2 = blk.bn2.folded()
    p = nv.EdgeXyzParams()
    p.xyz, p.idx = xyz.data_ptr(), idx32.data_ptr()
    p.B, p.N, p.k, p.nv = B, N, k, nvec
    p.Winit, p.Wz = Winit.data_ptr(), Wz.data_ptr()
    W1 = blk.linear1.weight.detach()
    W2 = blk.linear2.weight.detach()
    p.W1, p.bn1_a, p.bn1_c = W1.data_ptr(), a1.data_ptr(), c1.data_ptr()
    p.W2, p.bn2_a, p.bn2_c = W2.data_ptr(), a2.data_ptr(), c2.data_ptr()
    p.gate = gate.data_ptr()
    p.Cout, p.Cvo = blk.out_dims
    p.out = _mview(s_out, v_out)
    nv.edge_xyz_fwd(p)
    return idx32


def sv_edge_layer(s_in, v_in, B, N, k, blk, s_out, v_out, idx32=None, taps=None):
    """get_graph_feature_sv + SVBlock + svpool for edge layers 2..4 (sv_dgcnn_cls.py:55-65).
    s_in (B*N, Cs) / v_in (B*N, 3, Cv) are (possibly strided) slices of the svcat table.
    ``taps`` (dict) requests the per-edge sign/mask words for parity tests."""
    R = B * N
    Cs, Cv = s_in.shape[1], v_in.shape[2]
    Cout, Cvo = blk.out_dims
    assert blk.in_dims == (2 * Cs, 2 * Cv), (blk.in_dims, Cs, Cv)
    dev = s_in.device
    view = nv.view_of(s_in, v_in)
    # per-point tables do not depend on the graph: they run on a side stream next to the kNN kernels (whose second
    # wave leaves SMs idle at B = 32).  Tensor-core edge kernel (csrc/edge_tc.cu): one float4 table
    # [P | Q | T | U | v]; other kernels: the P | Q table of the vector branch.
    use_tc = blk.binary and nv.edge_tc_weight_bytes(Cs, Cv, Cout, Cvo, k) > 0
    fp_tc_bytes = 0 if blk.binary else nv.edge_fp_tc_weight_bytes(Cs, Cv, Cout, Cvo, k)      # csrc/edge_fp_tc.cu
    use_fp_tc = fp_tc_bytes > 0
    cur = torch.cuda.current_stream()
    side = (aux_stream(dev) if TABLE_AUX else (_side_stream(dev) if not _STATE.in_sub_batch else None)) if (idx32 is None and SIDE_STREAM) else None
    if use_tc or use_fp_tc:
        Wt, cst = blk.edge_tc_table_weight()
        NC = Wt.shape[0]
        table = torch.empty((R, NC, 4), dtype=torch.float32, device=dev)
        args = (v_in, v_in.stride(0), v_in.stride(1), 3, 3 * R, Cv, Wt, NC, table, 4 * NC, 0)
        kw = dict(sign_w=use_tc, colscale=cst, c4=True)
    else:
        Wpq, spq = blk.pq_weight()
        table = torch.empty((R, 3, 2 * Cvo), dtype=torch.float32, device=dev)
        args = (v_in, v_in.stride(0), v_in.stride(1), 3, 3 * R, Cv, Wpq, 2 * Cvo, table, 6 * Cvo, 2 * Cvo)
        kw = dict(sign_w=blk.linear2.bw, colscale=spq)
    # full-precision layers: the Ya | Yb table (the s part of linear1) does not depend on the graph either
    Yab = Wab = None
    if not blk.binary:
        Wab = blk.yab_only_weight() if use_fp_tc else blk.yab_weight()[0]
        Yab = torch.empty((R, 2 * Cout), dtype=torch.float32, device=dev)
    if side is not None:
        side.wait_stream(cur)
    with torch.cuda.stream(side if side is not None else cur):
        nv.linear_rows(*args, **kw)
        if Yab is not None:
            nv.linear_rows(s_in, s_in.stride(0), 0, 1, R, Cs, Wab, 2 * Cout, Yab, 2 * Cout, 0)
    if idx32 is None:
        idx32, _ = nv.knn(view, B, N, k)
    G1, G2 = blk.gate_weights()
    gate = nv.gate_edge(view, idx32, B, N, k, G1, G2)
    if side is not None:
        cur.wait_stream(side)
    Wz, zs = blk.v2s.wz()
    a1, c1 = blk.bn1_folded()
    a2, c2 = blk.bn2.folded()
    p = nv.EdgeParams()
    p.inp = view
    p.idx = idx32.data_ptr()
    p.B, p.N, p.k = B, N, k
    p.binary = 1 if blk.binary else 0
    p.Wz = Wz.data_ptr()
    p.zscale = zs.data_ptr() if zs is not None else 0
    keep = [gate, table, Wz, zs, a1, c1, a2, c2]
    W1nz = None
    if blk.binary:
        lin = blk.linear1
        beta, sc = lin.beta_vec(), lin.scale_vec()
        W1b, W1nz = lin.sign_planes()
        p.beta, p.W1b, p.scale1 = beta.data_ptr(), W1b.data_ptr(), sc.data_ptr()
        keep += [beta, W1b, sc]
        if use_tc:
            # linear1 on the tensor cores: fp8 sign bytes of the weights
            W1tc = blk.edge_tc_weight()
            p.W1tc, p.tab4 = W1tc.data_ptr(), table.data_ptr()
            keep += [W1tc]
    elif use_fp_tc:
        # full-precision linear1: the q part on the tensor cores (three bf16 weight planes), the s part from Ya | Yb
        W1f = blk.edge_fp_tc_weight(fp_tc_bytes)
        p.Yab, p.W1tc, p.tab4 = Yab.data_ptr(), W1f.data_ptr(), table.data_ptr()
        keep += [Yab, W1f]
    else:
        Wq_t = blk.yab_weight()[1]
        p.Yab, p.W1q_t = Yab.data_ptr(), Wq_t.data_ptr()
        keep += [Yab, Wq_t]
    p.bn1_a, p.bn1_c, p.Cout = a1.data_ptr(), c1.data_ptr(), Cout
    p.PQ = 0 if (use_tc or use_fp_tc) else table.data_ptr()
    p.bn2_a, p.bn2_c, p.gate, p.Cvo = a2.data_ptr(), c2.data_ptr(), gate.data_ptr(), Cvo
    p.out = _mview(s_out, v_out)
    if taps is not None and blk.binary:
        Kw = (2 * Cs + 6 * Cv + 31) // 32
        taps["bits"] = torch.zeros((R * k, Kw), dtype=torch.int32, device=dev)
        taps["mask"] = torch.zeros((R * k, Kw), dtype=torch.int32, device=dev)
        p.dbg_bits, p.dbg_mask = taps["bits"].data_ptr(), taps["mask"].data_ptr()
    nv.svblock_edge_fwd(p, W1nz=W1nz)
    if taps is not None:
        taps["gate"] = gate
    return idx32


def dgcnn_trunk(model, x, forced_idx=None, record=None):
    """Edge layers 1..4 shared by SV_DGCNN_CLS / SV_DGCNN_PSEG (sv_dgcnn_cls.py:47-67,
    sv_dgcnn_partseg.py:81-103).  Returns the svcat table (s_cat (B*N, sum Cs), v_cat (B*N, 3, sum Cv));
    every layer writes its pooled output straight into its column slice."""
    B, _, N = x.shape
    k = model.k
    dev = x.device
    xyz = x.transpose(1, 2).contiguous().view(B * N, 3)
    blocks = [model.conv1, model.conv2, model.conv3, model.conv4]
    cs = [b.out_dims[0] for b in blocks]
    cv = [b.out_dims[1] for b in blocks]
    s_cat = torch.empty((B * N, sum(cs)), dtype=torch.float32, device=dev)
    v_cat = torch.empty((B * N, 3, sum(cv)), dtype=torch.float32, device=dev)
    so, vo = 0, 0
    fi = forced_idx or [None] * 4
    idxs = []
    s_prev = v_prev = None
    for li, blk in enumerate(blocks):
        s_out = s_cat[:, so:so + cs[li]]
        v_out = v_cat[:, :, vo:vo + cv[li]]
        if li == 0:
            idx = first_edge_layer(xyz, B, N, k, 2, model.init_scalar, blk, s_out, v_out, idx32=fi[0])
        else:
            taps = record.setdefault("taps%d" % li, {}) if record is not None and record.get("want_taps") else None
            if record is not None and "teacher" in record:
                s_prev, v_prev = record["teacher"][li - 1]
            idx = sv_edge_layer(s_prev, v_prev, B, N, k, blk, s_out, v_out, idx32=fi[li], taps=taps)
        idxs.append(idx)
        s_prev, v_prev = s_out, v_out
        so += cs[li]
        vo += cv[li]
    if record is not None:
        record["idx"] = idxs
        record["s_cat"], record["v_cat"] = s_cat, v_cat
    return s_cat, v_cat
