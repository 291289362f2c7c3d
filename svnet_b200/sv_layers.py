"""Host-side mirror of the reference's SV layer library (models/sv_layers.py), inference only.

Same class names, constructor signatures, parameter names and ``state_dict`` layout as the
reference, so ``load_state_dict(checkpoint['state_dict'])`` works unchanged; every ``forward`` runs
hand-written sm_100a kernels through the C ABI (include/svnet_b200.h) -- there is no PyTorch or CPU
fallback.  Training-mode paths (STE clamp, sv_layers.py:40-42,46-48) are not on the inference hot
path: ``forward`` raises if ``self.training``.

Packed weights (sign bit-planes, folded BatchNorm affines, re-laid-out weight slices) are built
once per parameter version and cached on the module.
"""
import math

import torch
import torch.nn as nn

from . import _native as nv
from .sv_util import svpool

EPS = 1e-6


def _inference_only(m):
    if m.training:
        raise RuntimeError("%s: svnet_b200 implements the inference path only; call model.eval()"
                           % type(m).__name__)


def _resolve(module, path):
    """'linear.weight' -> module.linear.weight ('1.weight' indexes an nn.Sequential)."""
    obj = module
    for part in path.split("."):
        obj = obj[int(part)] if part.isdigit() else getattr(obj, part)
    return obj


class _Cached:
    """Mixin (first base, before the nn.Module class): cache of derived (packed) tensors -- sign bit-planes,
    folded BatchNorm affines, re-laid-out weight slices -- keyed on (what, device) and validated against the
    source parameters' (data_ptr, _version).

    * ``deps`` are attribute paths relative to the module, resolved on the *source* module: under
      nn.DataParallel every forward runs on fresh replicas whose parameters are new broadcast copies
      (main_cls_dgcnn.py:125); replicas remember their source (`_replicate_for_data_parallel`) and share its
      cache, so each device packs once, not once per forward.
    * Entries carry the CUDA event of their producer kernels: a consumer on another stream (the concurrent
      sub-batches of `fused.chunked`) waits on it until the event has been seen complete once.
    * In-place writes through ``.data`` do not bump ``_version``: ``load_state_dict`` and ``.to()/.cuda()``
      invalidate the cache here; after any other in-place surgery call ``invalidate_packed()``.
    """

    def _packed(self, key, deps, builder):
        d = self.__dict__
        src = d.get("_sv_src")
        if src is None:
            # fast path (every forward): one dict lookup, then the cached dependency tensors' (data_ptr, _version)
            cache = d.get("_sv_cache")
            if cache is None:
                cache = d["_sv_cache"] = {}
            hit = cache.get(key)
            if hit is not None:
                ok = True
                for t, (ptr, ver) in zip(hit[3], hit[0]):
                    if t._version != ver or t.data_ptr() != ptr:
                        ok = False
                        break
                if ok:
                    if hit[2] is not None:
                        self._order_after(hit)
                    return hit[1]
            owner, k = self, key
            tensors = [_resolve(self, dep) for dep in deps]
        else:
            # nn.DataParallel replica: dependencies are the source module's parameters, one slot per device
            owner = src
            cache = owner.__dict__.setdefault("_sv_cache", {})
            tensors = [_resolve(owner, dep) for dep in deps]
            dev = _resolve(self, deps[0]).device
            k = key if dev == tensors[0].device else (key, dev)     # the replica on the source's device shares its slot
            hit = cache.get(k)
            if hit is not None and hit[0] == tuple((t.data_ptr(), t._version) for t in tensors):
                if hit[2] is not None:
                    self._order_after(hit)
                return hit[1]
        sig = tuple((t.data_ptr(), t._version) for t in tensors)
        with torch.no_grad():
            val = builder()
        ev = None
        dev = _resolve(self, deps[0]).device
        if dev.type == "cuda" and not torch.cuda.is_current_stream_capturing():
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(dev))
        cache[k] = [sig, val, ev, tensors]
        _Cached.BUILDS += 1
        return val

    @staticmethod
    def _order_after(hit):
        """Consumers on another stream wait for the producer kernels of a packed tensor until they have retired once."""
        if torch.cuda.is_current_stream_capturing():
            return
        ev = hit[2]
        if ev.query():
            hit[2] = None
        else:
            torch.cuda.current_stream().wait_event(ev)

    BUILDS = 0          # builder invocations (tests count re-packs with it)

    def invalidate_packed(self):
        """Drop every cached packed tensor of this module and its children."""
        for m in self.modules() if isinstance(self, nn.Module) else [self]:
            m.__dict__.pop("_sv_cache", None)

    def _replicate_for_data_parallel(self):
        replica = super()._replicate_for_data_parallel()
        replica.__dict__["_sv_src"] = self.__dict__.get("_sv_src", self)
        return replica

    def _load_from_state_dict(self, *args, **kwargs):
        self.__dict__.pop("_sv_cache", None)
        return super()._load_from_state_dict(*args, **kwargs)

    def _apply(self, fn, *args, **kwargs):
        self.__dict__.pop("_sv_cache", None)
        return super()._apply(fn, *args, **kwargs)


def _rows2d(x):
    """(..., C) contiguous -> (rows, C)"""
    x = x.contiguous()
    return x.view(-1, x.shape[-1])


class Linear(_Cached, nn.Linear):
    """sv_layers.py:20-53.  bw: binarise weights, ba: binarise activations (sign(x + beta))."""

    def __init__(self, in_channels, out_channels, bias, bw=False, ba=False):
        super(Linear, self).__init__(in_channels, out_channels, bias)
        self.bw, self.ba = bw, ba
        if ba:
            self.beta = nn.Parameter(torch.zeros(1, in_channels))
        if bw:
            self.scale = nn.Parameter(torch.ones(1, out_channels) / math.sqrt(in_channels))

    # -- packed forms ---------------------------------------------------------------------------
    def sign_planes(self):
        """(sign plane, non-zero plane or None): the weight's torch.sign in {-1, 0, +1} (nv.pack_sign_nz)."""
        return self._packed("bits", ("weight",), lambda: nv.pack_sign_nz(self.weight.detach()))

    def sign_bits(self):
        return self.sign_planes()[0]

    def nz_bits(self):
        """Non-zero plane of the weight, None when it has no exact zero (the +-1 kernels run)."""
        return self.sign_planes()[1]

    def scale_vec(self):
        return self._packed("scale", ("scale",), lambda: self.scale.detach().reshape(-1).contiguous())

    def beta_vec(self):
        return self._packed("beta", ("beta",), lambda: self.beta.detach().reshape(-1).contiguous())

    def sign_weight(self):
        return self._packed("signw", ("weight",), lambda: torch.sign(self.weight.detach()).contiguous())

    # -- forward --------------------------------------------------------------------------------
    def forward_rows(self, x2d, bn=None, act=nv.ACT_NONE, out=None, ldo=None):
        """x2d (rows, K) -> (rows, Cout); optional fused BatchNorm affine + activation."""
        rows, K = x2d.shape
        Cout = self.out_features
        bias = self.bias.detach() if self.bias is not None else None
        if self.ba:
            if not self.bw:
                raise NotImplementedError("Linear(ba=True, bw=False) has no scale in the reference either")
            bits, mask, nvalid = nv.rows_prep(nv.view_of(x2d, None), rows, beta=self.beta_vec(), want_bits=True)
            return nv.binlinear_rows(bits, mask, nvalid, K, self.sign_bits(), Cout, scale=self.scale_vec(), bias=bias,
                                     bn=bn, act=act, out=out, ldo=ldo, W1nz=self.nz_bits())
        if out is None:
            out = torch.empty((rows, Cout), dtype=torch.float32, device=x2d.device)
            ldo = Cout
        nv.linear_rows(x2d, x2d.stride(0), 0, 1, rows, K, self.weight.detach(), Cout, out, ldo, 0,
                       sign_w=self.bw, colscale=self.scale_vec() if self.bw else None, bias=bias, bn=bn, act=act)
        return out

    def forward(self, x):
        _inference_only(self)
        shape_x = x.shape
        y = self.forward_rows(_rows2d(x))
        return y.view(shape_x[:-1] + (y.shape[-1],))


class Conv1d(_Cached, nn.Conv1d):
    """sv_layers.py:55-78: kernel-1 convolution on (B, C, N), always bw & ba when ``binary``."""

    def __init__(self, in_channels, out_channels, binary=False):
        super(Conv1d, self).__init__(in_channels, out_channels, 1, bias=False)
        print('Conv1d: ', in_channels, out_channels)
        self.binary = binary
        if binary:
            self.beta = nn.Parameter(torch.zeros(1, in_channels, 1))
            self.scale = nn.Parameter(torch.ones(1, out_channels, 1) / math.sqrt(in_channels))

    def weight2d(self):
        return self._packed("w2d", ("weight",), lambda: self.weight.detach()[:, :, 0].contiguous())

    def sign_planes(self, lo=0, hi=None):
        """(sign plane, non-zero plane or None) of the input channels [lo, hi) (nv.pack_sign_nz)."""
        return self._packed(("bits", lo, hi), ("weight",),
                            lambda: nv.pack_sign_nz(self.weight.detach()[:, lo:hi, 0].contiguous()))

    def sign_bits(self, lo=0, hi=None):
        return self.sign_planes(lo, hi)[0]

    def nz_bits(self, lo=0, hi=None):
        """Non-zero plane of the input channels [lo, hi), None when that slice has no exact zero."""
        return self.sign_planes(lo, hi)[1]

    def scale_vec(self):
        return self._packed("scale", ("scale",), lambda: self.scale.detach().reshape(-1).contiguous())

    def beta_vec(self):
        return self._packed("beta", ("beta",), lambda: self.beta.detach().reshape(-1).contiguous())

    def sv_in_bits(self, sv_in, Kc):
        """Sign words of SVFuse's output [s | v2s(v)] of the view ``sv_in`` = (view, rows, Wz, zscale) against this
        layer's beta[Kc:] -- the per-point half of ``forward_rows(None, cloud=..., sv_in=...)``, callable ahead of it
        (it does not depend on the per-cloud channels)."""
        view, rows, Wz_in, zs_in = sv_in
        return nv.rows_prep(view, rows, Wz=Wz_in, zscale=zs_in, beta=self.beta_vec()[Kc:], want_bits=True)

    def forward_rows(self, x2d, bn=None, act=nv.ACT_NONE, cloud=None, rows_per_cloud=1, sv_in=None, sv_bits=None):
        """x2d (rows, Kp) -> (rows, Cout).  ``cloud`` (B, Kc), if given, holds per-cloud-constant
        leading input channels (the ``repeat(1, 1, num_points)`` block of sv_dgcnn_partseg.py:118):
        the layer input is [cloud[row // rows_per_cloud] | x2d[row]] and the constant part of every
        dot product is reduced once per cloud instead of once per point.
        ``sv_in`` = (view, rows, Wz, zscale) replaces x2d by SVFuse's output [s | v2s(v)] of that view (binary layers
        only): the sign words come straight from (s, v), the float table is never written."""
        if sv_in is not None:
            assert self.binary and x2d is None
            view, rows, Wz_in, zs_in = sv_in
            Kp = view.Cs + 3 * view.Cv
        else:
            rows, Kp = x2d.shape
        Cout = self.out_channels
        Kc = cloud.shape[1] if cloud is not None else 0
        assert Kc + Kp == self.in_channels, (Kc, Kp, self.in_channels)
        if self.binary:
            beta = self.beta_vec()
            cdot = None
            if cloud is not None:
                cb, cm, cn = nv.rows_prep(nv.view_of(cloud, None), cloud.shape[0], beta=beta[:Kc], want_bits=True)
                cdot = nv.binlinear_rows(cb, cm, cn, Kc, self.sign_bits(0, Kc), Cout, out_i32=True, W1nz=self.nz_bits(0, Kc))
            if sv_bits is not None:
                bits, mask, nvalid = sv_bits
            elif sv_in is not None:
                bits, mask, nvalid = self.sv_in_bits(sv_in, Kc)
            else:
                bits, mask, nvalid = nv.rows_prep(nv.view_of(x2d, None), rows, beta=beta[Kc:], want_bits=True)
            return nv.binlinear_rows(bits, mask, nvalid, Kp, self.sign_bits(Kc, Kc + Kp), Cout, scale=self.scale_vec(),
                                     bn=bn, act=act, cloud_dot=cdot, rows_per_cloud=rows_per_cloud,
                                     W1nz=self.nz_bits(Kc, Kc + Kp))
        if cloud is not None:
            B = cloud.shape[0]
            x2d = torch.cat([cloud.unsqueeze(1).expand(B, rows_per_cloud, Kc).reshape(rows, Kc), x2d], dim=1)
        out = torch.empty((rows, Cout), dtype=torch.float32, device=x2d.device)
        nv.linear_rows(x2d, x2d.stride(0), 0, 1, rows, Kc + Kp, self.weight2d(), Cout, out, Cout, 0,
                       bias=self.bias.detach() if self.bias is not None else None, bn=bn, act=act)
        return out

    def forward(self, x):
        _inference_only(self)
        B, C, N = x.shape
        y = self.forward_rows(x.transpose(1, 2).contiguous().view(B * N, C))
        return y.view(B, N, -1).transpose(1, 2).contiguous()


class VectorBN(_Cached, nn.Module):
    """sv_layers.py:81-102: rescale each 3-vector by BatchNorm1d(|v|)/|v|."""

    def __init__(self, dim):
        super(VectorBN, self).__init__()
        self.bn = nn.BatchNorm1d(dim)

    def folded(self):
        bn = self.bn
        return self._packed("fold", ("bn.weight", "bn.bias", "bn.running_mean", "bn.running_var"), lambda: nv.fold_bn(bn))

    def forward(self, v):
        _inference_only(self)
        a, c = self.folded()
        return nv.vector_bn_rows(v.contiguous(), a, c)


def folded_bn(owner, name):
    """Folded eval affine of ``owner.<name>`` (an nn.BatchNorm1d), cached on ``owner``."""
    bn = getattr(owner, name)
    return owner._packed("fold_" + name, tuple(name + "." + a for a in ("weight", "bias", "running_mean", "running_var")),
                         lambda: nv.fold_bn(bn))


class Vector2Scalar(_Cached, nn.Module):
    """sv_layers.py:104-129: invariant scalars s[d*m+j] = sum_i v[i,d] * (v W^T)[i,j]."""

    def __init__(self, v_dim, multi, binary=False, trans_back=False):
        super(Vector2Scalar, self).__init__()
        if multi != 3:
            raise NotImplementedError("svnet_b200 implements multi == 3 (the only value the SV models use)")
        self.trans_back = trans_back
        self.linear = Linear(v_dim, multi, bias=False, bw=binary)

    def wz(self):
        """(Wz (3, C) -- already sign()ed when binary --, zscale (3,) or None)"""
        lin = self.linear
        if lin.bw:
            return lin.sign_weight(), lin.scale_vec()
        return self._packed("wz", ("linear.weight",), lambda: lin.weight.detach().contiguous()), None

    def forward_rows(self, v3, u_out=None, ldu=None, want_z=False):
        """v3 (rows, 3, C) strided view -> u (rows, 3C) written to u_out (row stride ldu)."""
        rows, _, C = v3.shape
        Wz, zs = self.wz()
        if u_out is None:
            u_out = torch.empty((rows, 3 * C), dtype=torch.float32, device=v3.device)
            ldu = 3 * C
        z = torch.empty((rows, 3, 3), dtype=torch.float32, device=v3.device) if want_z else None
        nv.rows_prep(nv.view_of(None, v3), rows, Wz=Wz, zscale=zs, u_out=u_out, ldu=ldu, z_out=z)
        return u_out, z

    def forward(self, v):
        '''
        shape of v: B, N_points, [k,] 3, dim
        '''
        _inference_only(self)
        assert v.ndim in [3, 4, 5], 'dim of v should be in [4, 5], got {}'.format(v.ndim)
        v = v.contiguous()
        lead = v.shape[:-2]
        s, z = self.forward_rows(v.view(-1, 3, v.shape[-1]), want_z=self.trans_back)
        s = s.view(lead + (-1,))
        if self.trans_back:
            return s, z.view(lead + (3, 3))
        return s


class VectorReLU(nn.Module):
    """sv_layers.py:131-149 -- never instantiated by any SV model; kept for name parity only."""

    def __init__(self):
        super(VectorReLU, self).__init__()
        self.div = 10

    def forward(self, x):
        raise NotImplementedError("VectorReLU is unused by the SV models (reference sv_layers.py:131-149)")


class SVBlock(_Cached, nn.Module):
    """sv_layers.py:151-196.  ``forward`` is the materialised (module-level) path over rows; the
    DGCNN models call the fused edge kernels instead (sv_dgcnn_cls.py in this package)."""

    def __init__(self, in_dims, out_dims, binary=False):
        super(SVBlock, self).__init__()
        print('SVBlock: ', in_dims, out_dims)
        self.in_dims, self.out_dims, self.binary = tuple(in_dims), tuple(out_dims), binary

        self.gate = nn.Sequential(
                nn.Linear(in_dims[0], out_dims[1]//2, bias=False),
                nn.ReLU(inplace=True),
                nn.Linear(out_dims[1]//2, out_dims[1], bias=False),
                nn.Sigmoid()
                )

        self.v2s = Vector2Scalar(in_dims[1], 3, binary=binary)

        self.linear1 = Linear(in_dims[0] + in_dims[1] * 3, out_dims[0], bias=False, bw=binary, ba=binary)
        self.bn1 = nn.BatchNorm1d(out_dims[0])
        self.relu = nn.LeakyReLU(negative_slope=0.2)

        self.linear2 = Linear(in_dims[1], out_dims[1], bias=False, bw=binary)
        self.bn2 = VectorBN(out_dims[1])

    # -- packed forms used by the fused kernels ---------------------------------------------------
    def gate_weights(self):
        return self.gate[0].weight.detach(), self.gate[2].weight.detach()

    def bn1_folded(self):
        return folded_bn(self, "bn1")

    def pq_weight(self):
        """[W2a; W2b] (2*Cvo, Cv_pt) and the matching column scale for the per-point P|Q table."""
        lin = self.linear2

        def build():
            W = lin.weight.detach()
            half = W.shape[1] // 2
            Wc = torch.cat([W[:, :half], W[:, half:]], dim=0).contiguous()
            sc = torch.cat([lin.scale.detach().reshape(-1)] * 2).contiguous() if lin.bw else None
            return Wc, sc
        deps = ("linear2.weight", "linear2.scale") if lin.bw else ("linear2.weight",)
        return self._packed("pq", deps, build)

    def edge_tc_table_weight(self):
        """Weights / column scales of the per-point table of the tensor-core edge kernel (csrc/edge_tc.cu):
        rows [W2a | W2b | Wz[:, :Cv] | Wz[:, Cv:] | I] over the Cv input vector channels (binary blocks only)."""
        lin, v2s = self.linear2, self.v2s.linear

        def build():
            W = lin.weight.detach()
            cv = W.shape[1] // 2
            Wz = v2s.weight.detach()
            eye = torch.eye(cv, dtype=W.dtype, device=W.device)
            Wt = torch.cat([W[:, :cv], W[:, cv:], Wz[:, :cv], Wz[:, cv:], eye], dim=0).contiguous()
            if not lin.bw:
                return Wt, None                       # full-precision block: plain weights, no column scales
            sc2, zs = lin.scale.detach().reshape(-1), v2s.scale.detach().reshape(-1)
            cs = torch.cat([sc2, sc2, zs, zs, torch.ones(cv, dtype=W.dtype, device=W.device)]).contiguous()
            return Wt, cs
        deps = ("linear2.weight", "linear2.scale", "v2s.linear.weight", "v2s.linear.scale") if lin.bw else \
            ("linear2.weight", "v2s.linear.weight")
        return self._packed("tc_tab", deps, build)

    def edge_fp_tc_weight(self, nbytes):
        """The q columns of a full-precision linear1 as three bf16 planes in the operand layout of csrc/edge_fp_tc.cu."""
        cs, cv = self.in_dims[0] // 2, self.in_dims[1] // 2
        return self._packed("w1ftc", ("linear1.weight",),
                            lambda: nv.edge_fp_tc_pack_w(self.linear1.weight.detach(), cs, cv, nbytes))

    def yab_only_weight(self):
        """[W1a; W1b] (2*Cout, Cs_pt) of a full-precision linear1 (the per-point table Ya | Yb)."""
        def build():
            W = self.linear1.weight.detach()
            cs = self.in_dims[0] // 2
            return torch.cat([W[:, :cs], W[:, cs:2 * cs]], dim=0).contiguous()
        return self._packed("yab_only", ("linear1.weight",), build)

    def edge_tc_weight(self):
        """linear1's sign bytes (fp8 e4m3) in the operand layout of the tensor-core edge kernel."""
        cs, cv = self.in_dims[0] // 2, self.in_dims[1] // 2
        return self._packed("w1tc", ("linear1.weight",), lambda: nv.edge_tc_pack_w(self.linear1.weight.detach(), cs, cv))

    def yab_weight(self):
        """fp linear1 split: ([W1a; W1b] (2*Cout, Cs_pt), W1q^T (6Cv_pt... = 3*Cv_e, Cout))."""
        lin = self.linear1

        def build():
            W = lin.weight.detach()
            cs = self.in_dims[0] // 2
            Wab = torch.cat([W[:, :cs], W[:, cs:2 * cs]], dim=0).contiguous()
            Wq_t = W[:, 2 * cs:].t().contiguous()
            return Wab, Wq_t
        return self._packed("yab", ("linear1.weight",), build)

    # -- module-level forward over materialised rows --------------------------------------------
    def forward_rows(self, s2d, v3, B, rows_per_cloud, s_out=None, lds_out=None, v_out=None, s_pool=None):
        """s2d (R, Cs) [row stride may exceed Cs], v3 (R, 3, Cv) strided.  Returns (s', v').
        ``s_pool`` = (max_out, mean_out, ldo): the scalar output is only needed pooled over each cloud's rows
        (SV_DGCNN_CLS conv5) -- when the fused tensor-core kernel covers the shape s' is never written and
        None is returned for it; otherwise s' is computed and pooled with svnet_pool_rows."""
        R = s2d.shape[0]
        Cs, Cv = self.in_dims
        Cso, Cvo = self.out_dims
        dev = s2d.device
        G1, G2 = self.gate_weights()
        Wz, zs = self.v2s.wz()
        view = nv.view_of(s2d, v3, Cs=Cs, Cv=Cv)
        bn1 = self.bn1_folded()
        K = Cs + 3 * Cv
        fused_pool = (s_pool is not None and self.binary and s_out is None
                      and nv.binlinear_pool_workspace(R, K, Cso, rows_per_cloud) > 0)
        if s_out is None and not fused_pool:
            s_out = torch.empty((R, Cso), dtype=torch.float32, device=dev)
            lds_out = Cso
        # the scalar branch (v2s + linear1 [+ pooling]) does not need the gate: with enough rows it runs on a side stream next
        # to gate -> vector linear (two independent chains of ~100 us each at conv5's shape)
        aux = None
        if R >= 1024:
            from .fused import aux_stream
            aux = aux_stream(dev)
        cur = torch.cuda.current_stream()
        if self.binary:
            beta1, sc1 = self.linear1.beta_vec(), self.linear1.scale_vec()
            sbits, snz = self.linear1.sign_planes()
        if aux is not None:
            aux.wait_stream(cur)
        with torch.cuda.stream(aux if aux is not None else cur):
            if self.binary:
                bits, mask, nvalid = nv.rows_prep(view, R, Wz=Wz, zscale=zs, beta=beta1, want_bits=True)
                if fused_pool:
                    nv.binlinear_pool(bits, mask, K, sbits, Cso, sc1, bn1, rows_per_cloud, s_pool[0], s_pool[1], s_pool[2],
                                      W1nz=snz)
                else:
                    nv.binlinear_rows(bits, mask, nvalid, K, sbits, Cso, scale=sc1, bn=bn1, act=nv.ACT_LEAKY, out=s_out, ldo=lds_out,
                                      W1nz=snz)
            else:
                u = torch.empty((R, K), dtype=torch.float32, device=dev)
                nv.rows_prep(view, R, Wz=Wz, zscale=zs, u_out=u, ldu=K)
                nv.linear_rows(u, K, 0, 1, R, K, self.linear1.weight.detach(), Cso, s_out, lds_out, 0, bn=bn1,
                               act=nv.ACT_LEAKY)
        if v_out is None:
            v_out = torch.empty((R, 3, Cvo), dtype=torch.float32, device=dev)
        lin2 = self.linear2
        gate = nv.gate_rows(s2d, s2d.stride(0), Cs, B, rows_per_cloud, G1, G2)
        nv.linear_rows(v3, v3.stride(0), v3.stride(1), 3, 3 * R, Cv, lin2.weight.detach(), Cvo, v_out,
                       v_out.stride(0), v_out.stride(1), sign_w=lin2.bw,
                       colscale=lin2.scale_vec() if lin2.bw else None, bn=self.bn2.folded(), vbn=True, gate=gate,
                       groups_per_cloud=rows_per_cloud)
        if aux is not None:
            torch.cuda.current_stream().wait_stream(aux)
        if s_pool is not None and not fused_pool:
            nv.pool_rows(s_out, lds_out, Cso, B, rows_per_cloud, want_max=s_pool[0] is not None,
                         want_mean=s_pool[1] is not None, max_out=s_pool[0], mean_out=s_pool[1], ldo=s_pool[2])
        return s_out, v_out

    def forward(self, x):
        '''
        shape of s: B, N_points, [k,] s_dim
        shape of v: B, N_points, [k,] 3, v_dim
        '''
        _inference_only(self)
        s, v = x
        s, v = s.contiguous(), v.contiguous()
        B = s.shape[0]
        lead = s.shape[:-1]
        R = s.numel() // s.shape[-1]
        so, vo = self.forward_rows(s.view(R, s.shape[-1]), v.view(R, 3, v.shape[-1]), B, R // B)
        return so.view(lead + (-1,)), vo.view(lead + (3, -1))


class SVFuse(nn.Module):
    """sv_layers.py:198-220: cat[s, v2s(v)]."""

    def __init__(self, v_dim, multi, binary, trans_back=False):
        super(SVFuse, self).__init__()
        print('SVFuse: ', v_dim)
        self.trans_back = trans_back

        self.v2s = Vector2Scalar(v_dim, multi, binary=binary, trans_back=trans_back)

    def forward_rows(self, s2d, v3, out=None, want_z=False):
        """-> (R, Cs + 3Cv) [, z (R,3,3)]; s2d may be None when ``out`` already holds the scalars."""
        R, _, Cv = v3.shape
        if out is None:
            Cs = s2d.shape[1]
            out = torch.empty((R, Cs + 3 * Cv), dtype=torch.float32, device=v3.device)
            out[:, :Cs].copy_(s2d)
        Cs = out.shape[1] - 3 * Cv
        _, z = self.v2s.forward_rows(v3, u_out=out[:, Cs:], ldu=out.stride(0), want_z=want_z)
        return out, z

    def forward(self, x):
        '''
        shape of s: B, N_points, [k,] s_dim
        shape of v: B, N_points, [k,] 3, v_dim
        '''
        _inference_only(self)
        s, v = x
        s, v = s.contiguous(), v.contiguous()
        lead = s.shape[:-1]
        R = s.numel() // s.shape[-1]
        out, z = self.forward_rows(s.view(R, -1), v.view(R, 3, v.shape[-1]), want_z=self.trans_back)
        out = out.view(lead + (-1,))
        if self.trans_back:
            return out, z.view(lead + (3, 3))
        return out


class SV_STNkd(nn.Module):
    """sv_layers.py:222-244."""

    def __init__(self, dim, binary):
        super(SV_STNkd, self).__init__()

        self.conv1 = SVBlock(dim, (64//2, 64//6), binary=binary)
        self.conv2 = SVBlock((64//2, 64//6), (128//2, 128//6), binary=binary)
        self.conv3 = SVBlock((128//2, 128//6), (1024//2, 1024//6), binary=binary)

        self.fc1 = SVBlock((1024//2, 1024//6), (512//2, 512//6), binary=binary)
        self.fc2 = SVBlock((512//2, 512//6), (256//2, 256//6), binary=binary)
        self.fc3 = SVBlock((256//2, 256//6), dim, binary=binary)

    def forward(self, x):
        x = self.conv1(x)
        x = self.conv2(x)
        x = self.conv3(x) # B, N_points, [3,] 1024//(2,6)
        x = svpool(x, dim=1)

        x = self.fc1(x)
        x = self.fc2(x)
        x = self.fc3(x) # B, [3,] dim

        return x


def dense_rows(weight, x2d, bias=None, bn=None, act=nv.ACT_NONE):
    """Plain fp nn.Linear / kernel-1 nn.Conv1d on rows: x2d (rows, K) -> (rows, Cout)."""
    W = weight.detach()
    if W.dim() == 3:
        W = W[:, :, 0]
    if W.stride(-1) != 1:
        W = W.contiguous()
    rows, K = x2d.shape
    out = torch.empty((rows, W.shape[0]), dtype=torch.float32, device=x2d.device)
    nv.linear_rows(x2d, x2d.stride(0), 0, 1, rows, K, W, W.shape[0], out, W.shape[0], 0,
                   bias=bias.detach() if bias is not None else None, bn=bn, act=act)
    return out


def head_layer(lin, bn=None, act=nv.ACT_NONE):
    """Descriptor of one layer of the fused classification head (svnet_head_fwd) from an
    sv_layers.Linear (any bw/ba combination the reference uses) or a plain nn.Linear."""
    d = {"Cout": lin.out_features, "bn": bn, "act": act,
         "bias": lin.bias.detach() if lin.bias is not None else None}
    if getattr(lin, "ba", False):
        d.update(W1b=lin.sign_bits(), W1nz=lin.nz_bits(), beta=lin.beta_vec(), scale=lin.scale_vec())
    elif getattr(lin, "bw", False):
        d.update(W=lin.weight.detach(), sign_w=True, scale=lin.scale_vec())
    else:
        d.update(W=lin.weight.detach())
    return d
