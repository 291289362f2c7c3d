"""CPU: pin the oracle (oracle/svnet_oracle.{c,py}) against the golden fixtures produced by the
unmodified reference (tests/golden/make_golden.py).  The reference has no tests of its own."""
import json

import numpy as np
import pytest

from oracle import svnet_oracle as orc
from tests.util import assert_close, golden, golden_state_dict, knn_is_valid, max_abs, quiet
from svnet_b200.synthetic import synthetic_state_dict
import torch


def test_knn_matches_reference_without_ties():
    g = golden("knn")
    for name in ("xyz", "c62", "c127"):
        x, k = g[name + "_x"], int(g[name + "_k"])
        idx, pd = orc.knn(np.transpose(x, (0, 2, 1)), k, return_pd=True)
        assert (idx == g[name + "_idx"]).all(), name
        assert max_abs(pd, g[name + "_pd"]) < 2e-4 * max(1.0, float(np.abs(g[name + "_pd"]).max()))


def test_knn_ties_lowest_index_and_valid():
    g = golden("knn")
    for name in ("dup", "lat"):
        x, k = g[name + "_x"], int(g[name + "_k"])
        idx, pd = orc.knn(np.transpose(x, (0, 2, 1)), k, return_pd=True)
        assert knn_is_valid(idx, pd, k)
        # the reference's own result is a valid top-k of the same scores as well (torch.topk tie order is arbitrary)
        assert knn_is_valid(g[name + "_idx"], pd, k)
        # lowest index first among exact ties
        sel = np.take_along_axis(pd, idx, axis=2)
        tie = sel[:, :, 1:] == sel[:, :, :-1]
        assert (idx[:, :, 1:][tie] > idx[:, :, :-1][tie]).all()


def test_graph_features_exact():
    g = golden("graph_features")
    xyz = np.transpose(g["x"][:, 0], (0, 2, 1))
    assert (orc.graph_feature_xyz(xyz, g["idx"], 2) == g["gf"]).all()
    # cross product: reference uses torch.cross (may fuse differently) -> 1 ulp
    assert_close(orc.graph_feature_xyz(xyz, g["idx"], 3), g["gf_cross"], rtol=1e-6, atol=1e-6)
    sf, vf = orc.graph_feature_sv(g["s"], g["v"], g["idx_sv"])
    assert (sf == g["sf"]).all() and (vf == g["vf"]).all()
    ps, pv = orc.svpool((sf, vf))
    assert (ps == g["pool_s"]).all()
    assert_close(pv, g["pool_v"], rtol=1e-6, atol=1e-6)
    ps, _ = orc.svpool((sf, vf), spool="mean")
    assert_close(ps, g["pool_mean_s"], rtol=1e-6, atol=1e-6)
    with pytest.raises(ValueError):
        orc.svpool((sf, vf), spool="median")


def _layer_sd(module_keys, seed, beta_zero=False):
    return synthetic_state_dict(module_keys, seed=seed, beta_zero=beta_zero)


def test_binary_linear_sign_planes_exact():
    g = golden("layers")
    for tag, bz in (("lin_bin", False), ("lin_bin_b0", True)):
        tmpl = {"weight": torch.empty(24, 70), "beta": torch.empty(1, 70), "scale": torch.empty(1, 24)}
        sd = _layer_sd(tmpl, 31, bz)
        x = g[tag + "_x"]
        sp = orc.sign_plane(x, sd["beta"].numpy())
        assert (sp == g[tag + "_sign"]).all()
        assert (sp == 0).any()  # the sign(0) == 0 case is exercised
        y = orc.linear(x, sd["weight"].numpy(), beta=sd["beta"].numpy(), scale=sd["scale"].numpy(), bw=True, ba=True)
        assert_close(y, g[tag + "_y"], rtol=1e-6, atol=1e-6, what=tag)


def test_layers_close():
    g = golden("layers")
    sd = _layer_sd({"weight": torch.empty(21, 42), "scale": torch.empty(1, 21)}, 33)
    y = orc.linear(g["lin_bw_x"], sd["weight"].numpy(), scale=sd["scale"].numpy(), bw=True)
    assert_close(y, g["lin_bw_y"], rtol=1e-5, atol=1e-6)
    sd = _layer_sd({"weight": torch.empty(16, 45, 1), "beta": torch.empty(1, 45, 1), "scale": torch.empty(1, 16, 1)}, 35)
    x = np.transpose(g["conv_bin_x"], (0, 2, 1))
    y = orc.linear(x, sd["weight"].numpy()[:, :, 0], beta=sd["beta"].numpy(), scale=sd["scale"].numpy(), bw=True, ba=True)
    assert_close(np.transpose(y, (0, 2, 1)), g["conv_bin_y"], rtol=1e-6, atol=1e-6)
    bn_t = {"bn.weight": torch.empty(11), "bn.bias": torch.empty(11), "bn.running_mean": torch.empty(11),
            "bn.running_var": torch.empty(11), "bn.num_batches_tracked": torch.empty((), dtype=torch.int64)}
    sd = _layer_sd(bn_t, 37)
    y = orc.vector_bn(g["vbn_x"], tuple(sd["bn." + n].numpy() for n in ("weight", "bias", "running_mean", "running_var")))
    assert_close(y, g["vbn_y"], rtol=1e-5, atol=1e-6)
    for tag, binary in (("v2s_fp", False), ("v2s_bin", True)):
        t = {"linear.weight": torch.empty(3, 20)}
        if binary:
            t["linear.scale"] = torch.empty(1, 3)
        sd = _layer_sd(t, 39)
        s, z = orc.v2s(g[tag + "_x"], sd["linear.weight"].numpy(), scale=sd["linear.scale"].numpy() if binary else None,
                       binary=binary, return_z=True)
        assert_close(z, g[tag + "_z"], rtol=1e-5, atol=1e-6)
        assert_close(s, g[tag + "_s"], rtol=1e-5, atol=1e-5)


MODELS = [
    ("dgcnn_cls_bin", "sv_dgcnn_cls", False), ("dgcnn_cls_bin_b0", "sv_dgcnn_cls", False),
    ("dgcnn_cls_fp", "sv_dgcnn_cls", False), ("dgcnn_pseg_bin", "sv_dgcnn_pseg", True),
    ("dgcnn_pseg_fp", "sv_dgcnn_pseg", True), ("pointnet_cls_fp", "sv_pointnet_cls", False),
    ("pointnet_cls_bin", "sv_pointnet_cls", False), ("pointnet_pseg_bin", "sv_pointnet_pseg", True),
    ("pointnet_pseg_fp", "sv_pointnet_pseg", True),
]


@pytest.mark.parametrize("name,fn,with_label", MODELS)
def test_models_match_reference(name, fn, with_label):
    """Whole-model forward of the oracle vs the reference's recorded forward: kNN indices equal,
    pooled per-point features and logits within the north_star tolerance, argmax identical."""
    g = golden(name)
    sd = golden_state_dict(g)
    k = int(g["k"])
    args = (sd, g["x"], g["label"], k) if with_label else (sd, g["x"], k)
    nidx = len([f for f in g.files if f.startswith("idx")])
    forced = [g["idx%d" % i] for i in range(nidx)]
    rec = {}
    y = getattr(orc, fn)(*args, forced_idx=forced, rec=rec)
    assert_close(y, g["logits"], what=name + " logits (teacher-forced idx)")
    for i, (s, v) in enumerate(rec["pools"]):
        assert_close(s, g["pool%d_s" % i], rtol=1e-4, atol=1e-5, what="%s pool%d s" % (name, i))
        assert_close(v, g["pool%d_v" % i], rtol=1e-4, atol=1e-5, what="%s pool%d v" % (name, i))
    rec = {}
    y = getattr(orc, fn)(*args, rec=rec)
    for i in range(nidx):
        agree = (rec["idx"][i] == g["idx%d" % i]).all(-1).mean()
        assert agree >= 0.98, "%s idx%d row agreement %.4f" % (name, i, agree)
    if all((rec["idx"][i] == g["idx%d" % i]).all() for i in range(nidx)):
        assert_close(y, g["logits"], what=name + " logits")
        assert (y.argmax(1) == g["logits"].argmax(1)).all()


def test_svblock_binary_sign_plane_matches_reference():
    """The q-channel sign planes (v2s output + beta, the fragile ones of SURVEY.md 7.3.2) of a binary
    SVBlock as the reference recorded them (make_golden.py: `svb_bin_sign`) against the oracle."""
    import svnet_b200 as sv
    g = golden("layers")
    blk = quiet(sv.SVBlock, (64, 20), (32, 10), True)
    sd = _layer_sd(blk.state_dict(), 41)
    P = orc.Params(sd)
    s, v = g["svb_bin_s"], g["svb_bin_v"]
    u = np.concatenate([s, orc.p_v2s(P.sub("v2s"), v)], axis=-1)
    sign = orc.sign_plane(u, P.get("linear1.beta"))
    ref = g["svb_bin_sign"]
    assert sign.shape == ref.shape and ref.shape[-1] == 64 + 60
    assert (sign == ref).all(), "%d of %d sign values differ" % ((sign != ref).sum(), ref.size)
    so, vo = orc.svblock(P, (s, v))
    assert_close(so, g["svb_bin_so"], rtol=1e-5, atol=1e-5)
    assert_close(vo, g["svb_bin_vo"], rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("cfg", ["cfg2", "cfg3", "cfg4"])
def test_oracle_record_at_baseline_shapes_matches_golden(cfg):
    """The oracle's record at the full-size parity test's shapes (tests/refparity.py: what the CUDA path is compared
    against where the reference's model code is not staged) reproduces the samples stored in tests/golden."""
    from tests import refparity
    from svnet_b200.synthetic import one_hot_labels, synthetic_clouds
    kw = refparity.CASES[cfg]
    g = golden("refparity_" + cfg)
    assert json.loads(str(g["config"])) == kw
    _, sd = refparity.build_ours(kw["kind"], kw["k"], kw["binary"], kw["ncls"], kw["seed"], "cpu")
    x = synthetic_clouds(kw["B"], kw["N"], kw["seed"])
    extra = (one_hot_labels(kw["B"]),) if kw["kind"] == "SV_DGCNN_PSEG" else ()
    refparity.pin_to_golden(refparity.oracle_record(sd, kw["kind"], kw["k"], kw["binary"], x, extra, "cpu"), g)
