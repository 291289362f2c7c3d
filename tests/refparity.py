"""Full-size parity of the CUDA path against the UNMODIFIED reference forward (oracle/_ref, staged by
oracle/make_ref.sh) run in the same process on the same device and inputs.

    measure(model_name, ...) -> dict of agreement statistics (kNN rows / sets, sign planes, pooled
    per-point features, logits); tests/test_gpu_reference.py asserts on them, tools/ref_parity.py
    writes them to profiles/.

What is compared (SURVEY.md 7.3.1 / 7.3.2, north_star's correctness clause):
* kNN: our kernel on the reference's own layer inputs against the reference's indices.  The reference
  scores with cuBLAS sgemm + three elementwise passes (sv_util.py:20-22), we with a sequential fp32
  chain, so rows whose k-th / (k+1)-th (or adjacent) scores lie within a few ulps may differ; every
  differing row must be *explained*: at every rank the two selected candidates' float64 scores differ by
  at most ``tol * (xx_i + xx_j)``.
* sign planes of the binarised linear1 of every edge layer, teacher-forced on the reference's pooled
  features and graphs: mismatches must be rare and only where |u + beta| is tiny.
* pooled per-point features of every edge layer (teacher-forced) and the logits with the reference's
  graphs forced.
"""
import contextlib
import io

import numpy as np
import torch

from oracle import reference
from svnet_b200.synthetic import make_args, one_hot_labels, synthetic_clouds, synthetic_state_dict


def quiet(fn, *a, **kw):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **kw)


def _unpack(words, K):
    """(rows, Kw) int32 cuda -> (rows, K) bool cuda"""
    sh = torch.arange(32, device=words.device, dtype=torch.int32)
    b = (words.unsqueeze(-1) >> sh) & 1
    return b.reshape(words.shape[0], -1)[:, :K].bool()


def knn_agreement(feat_bcn, ref_idx, our_idx, tol=2e-5):
    """Row / set agreement and the explanation check for the differing rows (float64 scores)."""
    B, C, N = feat_bcn.shape
    k = ref_idx.shape[-1]
    same_row = (ref_idx == our_idx).all(-1)                      # (B, N)
    rs, _ = ref_idx.sort(-1)
    os_, _ = our_idx.sort(-1)
    same_set = (rs == os_).all(-1)
    bad = (~same_row).nonzero()
    worst = 0.0
    unexplained = 0
    if bad.numel():
        f = feat_bcn.transpose(1, 2).double()                    # (B, N, C)
        xx = (f * f).sum(-1)                                     # (B, N)
        b, i = bad[:, 0], bad[:, 1]
        fi = f[b, i]                                             # (M, C)
        jr, jo = ref_idx[b, i], our_idx[b, i]                    # (M, k)
        def score(j):
            fj = f[b.unsqueeze(1), j]                            # (M, k, C)
            return -xx[b, i].unsqueeze(1) + 2 * (fj * fi.unsqueeze(1)).sum(-1) - xx[b.unsqueeze(1), j]
        pr, po = score(jr), score(jo)
        scale = xx[b, i].unsqueeze(1) + torch.maximum(xx[b.unsqueeze(1), jr], xx[b.unsqueeze(1), jo])
        rel = ((pr - po).abs() / scale.clamp_min(1e-30))
        worst = float(rel.max())
        unexplained = int((rel.max(-1)[0] > tol).sum())
    return {"rows": int(same_row.numel()), "row_agree": float(same_row.double().mean()),
            "set_agree": float(same_set.double().mean()), "rows_differing": int(bad.shape[0]),
            "worst_rel_gap": worst, "unexplained_rows": unexplained, "tol": tol}


def build_ours(kind, k, binary, ncls, seed, dev):
    import svnet_b200 as sv
    ours = quiet(getattr(sv, kind), make_args(k=k, binary=binary), ncls)
    sd = synthetic_state_dict(ours.state_dict(), seed=seed)
    ours.load_state_dict(sd)
    return ours.to(dev).eval(), sd


def build_pair(kind, k, binary, ncls, seed, dev):
    ref = reference.load()
    ours, sd = build_ours(kind, k, binary, ncls, seed, dev)
    rnet = quiet(getattr(ref, kind), make_args(k=k, binary=binary), ncls)
    rnet.load_state_dict(sd)
    rnet = rnet.to(dev).eval()
    return ours, rnet, sd


MODEL_FILE = {"SV_DGCNN_CLS": "sv_dgcnn_cls", "SV_DGCNN_PSEG": "sv_dgcnn_partseg"}


SIGN_OF = ["conv2.linear1", "conv3.linear1", "conv4.linear1"]


class Record:
    """What measure() compares against, recorded from one forward: the layer inputs of the kNN calls (B, C, N),
    the kNN indices, the pooled per-point (s, v) of the four edge layers, for binary models the sign planes
    sign(u + beta) and |u + beta| of conv2-4's linear1, and the logits."""

    def __init__(self, knn_in, idx, pools, signs, logits):
        self.knn_in, self.idx, self.pools, self.signs, self.logits = knn_in, idx, pools, signs, logits


def reference_record(rnet, kind, x, extra, binary):
    """The unmodified reference forward (oracle/_ref), hooked by reference.Recorder."""
    modfile = reference.submodule(MODEL_FILE[kind])
    with torch.no_grad(), reference.Recorder(modfile, rnet, SIGN_OF if binary else []) as rec:
        y_ref = rnet(x, *extra)
    return Record(rec.knn_in[:4], rec.idx[:4], rec.pools[:4], rec.signs, y_ref)


def oracle_record(sd, kind, k, binary, x, extra, dev):
    """The same record from the CPU oracle (oracle/svnet_oracle.c, the reference restated function by function and
    pinned to the reference's own outputs by tests/test_oracle_golden.py), for where the reference's model code is not
    staged.  The oracle is deterministic: tests/golden/refparity_*.npz hold samples of its record at these shapes
    (tests/golden/make_golden_refparity.py), and pin_to_golden() checks every run against them."""
    from oracle import svnet_oracle as orc
    xn = x.cpu().numpy()
    rec = {}
    if kind == "SV_DGCNN_PSEG":
        y = orc.sv_dgcnn_pseg(sd, xn, extra[0].cpu().numpy(), k, rec=rec)
    else:
        y = orc.sv_dgcnn_cls(sd, xn, k, rec=rec)
    P = orc.Params(sd)
    B, N = xn.shape[0], xn.shape[2]
    knn_in, signs = [x], {}
    for li in range(1, 4):
        s, v = rec["pools"][li - 1]
        knn_in.append(torch.from_numpy(np.concatenate([s, v.reshape(B, N, -1)], axis=-1)).to(dev).transpose(1, 2))
        if binary:
            cname = "conv%d" % (li + 1)
            s_e, v_e = orc.graph_feature_sv(s, v, rec["idx"][li])
            u = np.concatenate([s_e, orc.p_v2s(P.sub(cname + ".v2s"), v_e)], axis=-1)
            beta = P.get(cname + ".linear1.beta").reshape(-1)
            signs[cname + ".linear1"] = (torch.from_numpy(orc.sign_plane(u, beta)).to(dev),
                                         torch.from_numpy(np.abs(u + beta)).to(dev))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    return Record(knn_in, [t(i) for i in rec["idx"]], [(t(s), t(v)) for s, v in rec["pools"]], signs, t(y))


# the BASELINE.json shapes of the parity test (batch cut to keep the CPU side short)
CASES = {
    "cfg2": dict(kind="SV_DGCNN_CLS", B=4, N=1024, k=20, binary=True, ncls=40, seed=1002),
    "cfg3": dict(kind="SV_DGCNN_CLS", B=4, N=1024, k=20, binary=False, ncls=15, seed=1003),
    "cfg4": dict(kind="SV_DGCNN_PSEG", B=2, N=2048, k=40, binary=True, ncls=50, seed=1004),
}
GOLDEN_ROWS = 24       # sampled points (kNN rows, pooled features, per-point logits) and edge rows (sign planes)


def golden_samples(r, seed=0):
    """Fixed, seeded sample of a Record as numpy arrays (what tests/golden/refparity_*.npz store)."""
    B, N = r.idx[0].shape[:2]
    g = np.random.default_rng(seed)
    pts = np.sort(g.choice(B * N, GOLDEN_ROWS, replace=False))
    out = {"points": pts}
    for li in range(4):
        out["idx%d" % li] = r.idx[li].reshape(B * N, -1)[pts].cpu().numpy().astype(np.int16)
        s, v = r.pools[li]
        out["pool%d_s" % li] = s.reshape(B * N, -1)[pts].cpu().numpy()
        out["pool%d_v" % li] = v.reshape(B * N, 3, -1)[pts].cpu().numpy()
    for name, (sign, _) in sorted(r.signs.items()):
        K = sign.shape[-1]
        edges = np.sort(g.choice(sign.numel() // K, GOLDEN_ROWS, replace=False))
        out["edges|" + name] = edges
        out["sign|" + name] = sign.reshape(-1, K)[edges].cpu().numpy()
    y = r.logits
    out["logits"] = (y.cpu().numpy() if y.dim() == 2 else
                     y.permute(0, 2, 1).reshape(B * N, -1)[pts].cpu().numpy())   # part-seg: (B, parts, N)
    return out


def pin_to_golden(r, golden):
    """The oracle's record equals the stored one on every sampled element: indices and sign planes exactly, floats to
    a few ulps (the oracle's summation order is fixed; only the host's libm may differ)."""
    got = golden_samples(r)
    assert sorted(got) == sorted(k for k in golden.files if k != "config"), (sorted(got), golden.files)
    for key, val in got.items():
        want = golden[key]
        assert val.shape == want.shape and val.dtype == want.dtype, key
        if val.dtype.kind == "f":
            assert np.allclose(val, want, rtol=1e-6, atol=1e-7), "oracle record differs from tests/golden at " + key
        else:
            assert np.array_equal(val, want), "oracle record differs from tests/golden at " + key


def measure(kind="SV_DGCNN_CLS", B=4, N=1024, k=20, binary=True, ncls=40, seed=1002, dev="cuda", golden=None):
    """golden=None: against the unmodified reference forward; else (an np.load of tests/golden/refparity_*.npz)
    against the oracle's record, pinned to those samples."""
    import svnet_b200 as sv
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    x = synthetic_clouds(B, N, seed).to(dev)
    extra = (one_hot_labels(B).to(dev),) if kind == "SV_DGCNN_PSEG" else ()
    if golden is None:
        ours, rnet, sd = build_pair(kind, k, binary, ncls, seed, dev)
        rec = reference_record(rnet, kind, x, extra, binary)
    else:
        (ours, sd), rnet = build_ours(kind, k, binary, ncls, seed, dev), None
        rec = oracle_record(sd, kind, k, binary, x, extra, dev)
        pin_to_golden(rec, golden)
    y_ref = rec.logits
    out = {"model": kind, "B": B, "N": N, "k": k, "binary": binary, "layers": [],
           "against": "reference" if golden is None else "oracle"}
    ridx = rec.idx
    pools = rec.pools
    teacher = [(s.reshape(B * N, -1).contiguous(), v.reshape(B * N, 3, -1).contiguous()) for s, v in pools[:3]]
    got = {"teacher": teacher, "want_taps": True}
    forced = [i.to(torch.int32).contiguous() for i in ridx]
    with torch.no_grad():
        ours(x, *extra, forced_idx=forced, record=got)
        y_forced = ours(x, *extra, forced_idx=forced)
        free = {}
        y_free = ours(x, *extra, record=free)
    so = vo = 0
    for li in range(4):
        # kNN on the reference's own layer input
        our_idx = sv.knn(rec.knn_in[li], k)
        st = knn_agreement(rec.knn_in[li], ridx[li], our_idx)
        st["free_running_row_agree"] = float((free["idx"][li].long() == ridx[li]).all(-1).double().mean())
        ps, pv = pools[li]
        cs, cv = ps.shape[-1], pv.shape[-1]
        gs = got["s_cat"][:, so:so + cs].reshape(B, N, cs)
        gv = got["v_cat"][:, :, vo:vo + cv].reshape(B, N, 3, cv)
        es = (gs - ps).abs()
        ev = (gv - pv).abs()
        st.update(layer=li + 1,
                  pooled_s_max_abs=float(es.max()), pooled_s_exact_frac=float((gs == ps).double().mean()),
                  pooled_s_out_of_tol=float((es > 1e-4 + 1e-3 * ps.abs()).double().mean()),
                  pooled_v_max_abs=float(ev.max()),
                  pooled_v_out_of_tol=float((ev > 1e-4 + 1e-3 * pv.abs()).double().mean()))
        if binary and li > 0:
            name = "conv%d.linear1" % (li + 1)
            rsign, rabs = rec.signs[name]                       # (B,N,k,K) int8 / |u+beta|
            K = rsign.shape[-1]
            rs2, ra2 = rsign.reshape(-1, K), rabs.reshape(-1, K)
            taps = got["taps%d" % li]
            bits, mask = _unpack(taps["bits"], K), _unpack(taps["mask"], K)
            osign = torch.where(mask, torch.where(bits, 1, -1), 0).to(torch.int8)
            diff = osign != rs2
            nd = int(diff.sum())
            scale_u = float(ra2.max())
            worst = float(ra2[diff].max()) if nd else 0.0
            Cs2 = 2 * teacher[li - 1][0].shape[1]               # scalar channels come first; q channels after
            st.update(sign_bits=int(diff.numel()), sign_mismatch=nd, sign_mismatch_rate=nd / diff.numel(),
                      sign_mismatch_scalar_channels=int(diff[:, :Cs2].sum()),
                      sign_mismatch_max_abs_t=worst, sign_mismatch_max_rel_t=worst / max(scale_u, 1e-30))
        out["layers"].append(st)
        so += cs
        vo += cv
    yr = y_ref.double()
    for tag, y in (("forced", y_forced), ("free", y_free)):
        e = (y.double() - yr).abs()
        out["logits_" + tag] = {"max_abs": float(e.max()),
                                "out_of_tol": float((e > 1e-4 + 1e-3 * yr.abs()).double().mean()),
                                "argmax_equal": float((y.argmax(1) == y_ref.argmax(1)).double().mean())}
    # the reference against itself on the host CPU (how far stock PyTorch moves when only the device changes)
    return out, (ours, rnet, x, extra, y_ref)


def reference_cpu_vs_cuda(rnet, x, extra, y_ref):
    import copy
    cpu = copy.deepcopy(rnet).cpu().eval()
    with torch.no_grad():
        y = cpu(x.cpu(), *[e.cpu() for e in extra])
    e = (y.double() - y_ref.cpu().double()).abs()
    return {"max_abs": float(e.max()),
            "out_of_tol": float((e > 1e-4 + 1e-3 * y_ref.cpu().double().abs()).double().mean()),
            "argmax_equal": float((y.argmax(1) == y_ref.cpu().argmax(1)).double().mean())}
