"""SV-DGCNN part segmentation -- drop-in for models/sv_dgcnn_partseg.py:40-128 (same constructor
and state_dict keys).  Edge layers 1..4 are the fused kernels of the classifier; the tail runs on
row-major (B*N, C) tables:

    x_fine  = svfuse1(svcat)                      rows_prep (float u)                 (:104)
    conv5   per-point SVBlock                     gate_rows, rows_prep, binlinear, vector linear (:106)
    conv6/svfuse2 on the per-cloud pooled row     same kernels with rows = B           (:107-109)
    svfuse3 + max over points                     rows_prep + pool_rows                (:111-112)
    conv8   binary conv over 2144 channels, 1600 of which are per-cloud constants (the
            ``repeat(1, 1, num_points)`` of :118): their sign words and popcounts are reduced once per
            cloud and enter the per-point popcount linear as an integer offset      (:117-121)
    conv9/10 binary conv + BN + leaky, conv11 fp                                       (:123-126)
The full-precision head is one call as well (svnet_seg_head_fp_fwd): conv8's per-cloud 1600 columns are one linear over the
B clouds, added per point in the epilogue of the per-point linear over svfuse1's 544 channels (on the three-plane
tensor-core fp linear); conv9 .. conv11 take the kernel the layer-by-layer calls take.  SVNET_SEG_HEAD_CALL=0 runs both heads layer by layer (the fp one over the (B*N, 2144) table).
"""
import os

import torch
import torch.nn as nn

from . import _native as nv
from .fused import aux_stream, chunked, dgcnn_trunk, native_forward
from .sv_layers import Conv1d, SVBlock, SVFuse, Vector2Scalar, _Cached, _inference_only, dense_rows, folded_bn

SEG_HEAD_CALL = os.environ.get("SVNET_SEG_HEAD_CALL", "1") != "0"     # 0: the head layer by layer (parity tests compare both)


def _get_visible_value(divisor=8):
    def make_divisible(v):
        """Round channel counts to a multiple of ``divisor`` without losing more than 10 %
        (sv_dgcnn_partseg.py:18-32)."""
        new_v = max(divisor, int(v + divisor / 2) // divisor * divisor)
        if new_v < 0.9 * v:
            new_v += divisor
        return new_v
    return make_divisible


_V = _get_visible_value(8)


class _Seq(_Cached, nn.Sequential):
    """nn.Sequential(conv, BatchNorm1d, act) with a cached folded BN (keys '0', '1' as in the reference)."""

    def bn_folded(self):
        bn = self[1]
        return self._packed("fold", ("1.weight", "1.bias", "1.running_mean", "1.running_var"), lambda: nv.fold_bn(bn))


class SV_DGCNN_PSEG(_Cached, nn.Module):
    def __init__(self, args, num_part):
        super(SV_DGCNN_PSEG, self).__init__()
        self.args = args
        self.k = args.k
        self.binary = args.binary
        self.dropout = 0 if self.binary else args.dropout
        self.emb = 1024

        self.init_scalar = Vector2Scalar(2, 3)
        self.conv1 = SVBlock((6, 2), (_V(64//2), _V(64//6)))
        self.conv2 = SVBlock((_V(64//2)*2, _V(64//6)*2), (_V(64//2), _V(64//6)), self.binary)
        self.conv3 = SVBlock((_V(64//2)*2, _V(64//6)*2), (_V(128//2), _V(128//6)), self.binary)
        self.conv4 = SVBlock((_V(128//2)*2, _V(128//6)*2), (_V(256//2), _V(256//6)), self.binary)

        cs_cat = _V(64//2)*2+_V(128//2)+_V(256//2)
        cv_cat = _V(64//6)*2+_V(128//6)+_V(256//6)
        self.svfuse1 = SVFuse(cv_cat, 3, self.binary)
        self.conv5 = SVBlock((cs_cat, cv_cat), (_V(self.emb//2), _V(self.emb//6)), self.binary)
        self.conv6 = SVBlock((_V(self.emb//2), _V(self.emb//6)), (_V(self.emb//4), _V(self.emb//12)), self.binary)
        self.svfuse2 = SVFuse(_V(self.emb//12), 3, self.binary)
        self.svfuse3 = SVFuse(_V(self.emb//6), 3, self.binary)
        self.conv7 = _Seq(
                nn.Conv1d(16, 64, kernel_size=1, bias=False),
                nn.BatchNorm1d(64),
                nn.LeakyReLU(negative_slope=0.2))
        self.conv8 = _Seq(
                Conv1d(_V(self.emb//2)+_V(self.emb//4)+(_V(self.emb//6)+_V(self.emb//12))*3+64+cs_cat+cv_cat*3, 256, self.binary),
                nn.BatchNorm1d(256),
                nn.LeakyReLU(negative_slope=0.2))
        self.dp1 = nn.Dropout(p=self.dropout)
        self.conv9 = _Seq(
                Conv1d(256, 256, self.binary),
                nn.BatchNorm1d(256),
                nn.LeakyReLU(negative_slope=0.2))
        self.dp2 = nn.Dropout(p=self.dropout)
        self.conv10 = _Seq(
                Conv1d(256, 128, self.binary),
                nn.BatchNorm1d(128),
                nn.LeakyReLU(negative_slope=0.2))
        self.conv11 = nn.Conv1d(128, num_part, kernel_size=1, bias=False)

    def forward(self, x, l, forced_idx=None, record=None):
        hooks = forced_idx is not None or record is not None
        if not hooks and SEG_HEAD_CALL:
            _inference_only(self)
            y = native_forward(self, "SV_DGCNN_PSEG", x, l)   # the same calls sequenced in C (csrc/model.cu); None: not covered
            if y is not None:
                return y
        return chunked(lambda xc, lc: self._forward(xc, lc, forced_idx, record), x, (l,), hooks=hooks)

    def _forward(self, x, l, forced_idx=None, record=None):
        """x (B,3,N), l (B,16) one-hot -> per-point part logits (B, num_part, N).  The calls csrc/model.cu's
        svnet_model_forward_seg makes in C (binary or full precision), so the two paths give the same bits; with ``record``
        (test hooks) the head runs layer by layer."""
        _inference_only(self)
        B, _, N = x.shape
        R = B * N
        dev = x.device
        s_cat, v_cat = dgcnn_trunk(self, x, forced_idx, record)
        C5s, C5v = self.conv5.out_dims
        fuse3 = 3 * C5v <= 512             # svfuse3 + max pooling without the (R, 1016) table (svnet_svfuse_pool)
        # svfuse1's output only feeds conv8: a binary conv8 takes its sign words straight from (s_cat, v_cat), the fp head call
        # writes the rows into its own scratch
        lean_fine = self.binary and record is None
        fp_head = not self.binary and record is None and SEG_HEAD_CALL
        x_fine = None if (lean_fine or fp_head) else self.svfuse1.forward_rows(s_cat, v_cat)[0]          # (R, 544)
        sv_in = sv_bits = aux = None
        if lean_fine:
            # conv8's per-point sign words depend on the trunk only: they run on a side stream next to the global
            # branch below, whose per-cloud kernels (conv6, svfuse2, conv7: B rows each) leave the GPU almost idle
            Wz1, zs1 = self.svfuse1.v2s.wz()
            sv_in = (nv.view_of(s_cat, v_cat), R, Wz1, zs1)
            Kc8 = self.conv8[0].in_channels - (s_cat.shape[1] + 3 * v_cat.shape[2])
            aux = aux_stream(dev)
            if aux is not None:
                cur = torch.cuda.current_stream()
                aux.wait_stream(cur)
                with torch.cuda.stream(aux):
                    sv_bits = self.conv8[0].sv_in_bits(sv_in, Kc8)
                for t in sv_bits:
                    t.record_stream(cur)
        # global branch: svpool over points -> conv6 -> svfuse2.  Per point only v5 is needed further on (with fuse3):
        # the binary conv5 pools its scalar output in the epilogue of its tensor-core linear and never writes it
        sp = torch.empty((B, C5s), dtype=torch.float32, device=dev)
        vp = torch.empty((B, 3, C5v), dtype=torch.float32, device=dev)
        if fuse3:
            s5, v5 = self.conv5.forward_rows(s_cat, v_cat, B, N, s_pool=(sp, None, C5s))    # s5 is None on the fused path
        else:
            s5, v5 = self.conv5.forward_rows(s_cat, v_cat, B, N)                  # (R,512), (R,3,168)
            nv.pool_rows(s5, C5s, C5s, B, N, want_max=True, want_mean=False, max_out=sp)
        C3 = C5s + 3 * C5v
        xw = self.conv6.out_dims[0] + 3 * self.conv6.out_dims[1]                 # width of svfuse2's output (520)
        glob = torch.empty((B, C3 + xw + 64), dtype=torch.float32, device=dev)
        # svfuse3 + max over points (sv_dgcnn_partseg.py:110-111) without the (R, 1016) table: the scalar half is the
        # max of s5 that conv6's input already needed (sp), v2s(v5) is reduced on the fly (svnet_svfuse_pool).  It and
        # conv7 (the label branch) run on the side stream next to pool -> conv6 -> svfuse2, whose one-row-per-cloud
        # kernels leave the GPU almost idle; the two sides write disjoint columns of glob.
        aux2 = aux_stream(dev) if (fuse3 and record is None) else None
        cur = torch.cuda.current_stream()
        if aux2 is not None:
            aux2.wait_stream(cur)
        with torch.cuda.stream(aux2 if aux2 is not None else cur):
            if fuse3:
                Wz3, zs3 = self.svfuse3.v2s.wz()
                nv.svfuse_pool(v5, B, N, Wz3, zs3, glob[:, C5s:], None, glob.shape[1])
            lab = dense_rows(self.conv7[0].weight, l.reshape(B, -1).contiguous().float(), bn=self.conv7.bn_folded(),
                             act=nv.ACT_LEAKY)
            glob[:, C3 + xw:].copy_(lab)
        nv.pool_rows(v5, 3 * C5v, 3 * C5v, B, N, want_max=False, want_mean=True, mean_out=vp)
        s6, v6 = self.conv6.forward_rows(sp, vp, B, 1)
        x_pool, _ = self.svfuse2.forward_rows(s6, v6)                             # (B, 520)
        if fuse3:
            glob[:, :C5s].copy_(sp)
        else:
            f3, _ = self.svfuse3.forward_rows(s5, v5)                             # (R, 1016)
            nv.pool_rows(f3, C3, C3, B, N, want_max=True, max_out=glob, ldo=glob.shape[1])
        glob[:, C3:C3 + xw].copy_(x_pool)
        if aux2 is not None:
            cur.wait_stream(aux2)
        # segmentation head on rows; glob is constant per cloud
        if lean_fine:
            if aux is not None:
                torch.cuda.current_stream().wait_stream(aux)
            if SEG_HEAD_CALL:
                # conv8 .. conv11 and the (B, parts, N) layout as one C-ABI call (csrc/seg_head.cu)
                c8, c9, c10 = self.conv8[0], self.conv9[0], self.conv10[0]
                Kc = glob.shape[1]
                W11 = self.conv11.weight.detach()[:, :, 0]
                layers = [dict(beta=c8.beta_vec(), bits=(c8.sign_bits(0, Kc), c8.sign_bits(Kc, c8.in_channels)), scale=c8.scale_vec(),
                               bn=self.conv8.bn_folded(), Cout=c8.out_channels),
                          dict(beta=c9.beta_vec(), bits=c9.sign_bits(), scale=c9.scale_vec(), bn=self.conv9.bn_folded(),
                               Cout=c9.out_channels),
                          dict(beta=c10.beta_vec(), bits=c10.sign_bits(), scale=c10.scale_vec(), bn=self.conv10.bn_folded(),
                               Cout=c10.out_channels)]
                return nv.seg_head_fwd(sv_in[0], B, N, sv_in[2], sv_in[3], glob, layers, W11 if W11.is_contiguous() else W11.contiguous(),
                                       sv_bits=sv_bits)
            h = self.conv8[0].forward_rows(None, bn=self.conv8.bn_folded(), act=nv.ACT_LEAKY, cloud=glob, rows_per_cloud=N,
                                           sv_in=sv_in, sv_bits=sv_bits)
        else:
            if fp_head:
                W11 = self.conv11.weight.detach()[:, :, 0]
                # conv8 .. conv11 as one C-ABI call (csrc/seg_head.cu): conv8's per-cloud part of the (R, 2144) input once per
                # cloud, the per-point part over svfuse1's 544 channels; None when conv8 is off the tensor-core linear
                layers = [(c.weight2d(), seq.bn_folded()) for c, seq in ((self.conv8[0], self.conv8), (self.conv9[0], self.conv9),
                                                                          (self.conv10[0], self.conv10))]
                y = nv.seg_head_fp_fwd(nv.view_of(s_cat, v_cat), B, N, self.svfuse1.v2s.wz()[0], glob, layers,
                                       W11 if W11.is_contiguous() else W11.contiguous())
                if y is not None:
                    return y
                x_fine = self.svfuse1.forward_rows(s_cat, v_cat)[0]
            h = self.conv8[0].forward_rows(x_fine, bn=self.conv8.bn_folded(), act=nv.ACT_LEAKY, cloud=glob, rows_per_cloud=N)
        h = self.conv9[0].forward_rows(h, bn=self.conv9.bn_folded(), act=nv.ACT_LEAKY)
        h = self.conv10[0].forward_rows(h, bn=self.conv10.bn_folded(), act=nv.ACT_LEAKY)
        out = dense_rows(self.conv11.weight, h)                                   # (R, num_part)
        if record is not None:
            record.update(glob=glob, x_fine=x_fine)
        return out.view(B, N, -1).transpose(1, 2).contiguous()
