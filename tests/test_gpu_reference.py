"""GPU parity against the reference forward at the BASELINE.json shapes.

Where the reference's model code is staged into oracle/_ref (git-ignored) by oracle/make_ref.sh, the UNMODIFIED
reference runs on the same device and inputs as the CUDA path.  Elsewhere the same record comes from the CPU oracle
(the reference restated in C, pinned to the reference's own outputs by tests/test_oracle_golden.py), checked against
the samples of it stored in tests/golden/refparity_<cfg>.npz.  Every kind of disagreement is counted and explained
(tests/refparity.py).  Bars: north_star's correctness clause with SURVEY.md 7.3.1 / 7.3.2's account of where stock
ATen and a fixed summation order may differ.
"""
import json

import pytest

from oracle import reference
from tests import refparity
from tests.util import golden

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("cfg", ["cfg2", "cfg3", "cfg4"])
def test_full_size_parity_with_reference_forward(cfg):
    kw = refparity.CASES[cfg]
    out, _ = refparity.measure(**kw, golden=None if reference.available() else golden("refparity_" + cfg))
    print(cfg, json.dumps(out))
    for st in out["layers"]:
        # kNN: identical rows, or a differing row is a swap / boundary exchange between candidates whose
        # exact scores agree to a few fp32 ulps of the operands' squared norms (SURVEY 7.3.1)
        assert st["unexplained_rows"] == 0, st
        # measured (profiles/r2a_ref_parity.json): rows 0.992-1.0 at k=20, 0.963-0.9998 at k=40 (twice the adjacent
        # pairs per row, denser features); sets 0.9968-1.0; worst explained gap 1.0e-6 of the norms
        assert st["row_agree"] >= 0.94, st
        assert st["set_agree"] >= 0.995, st
        # pooled per-point features of the layer (teacher-forced on the reference's inputs and graph)
        assert st["pooled_v_out_of_tol"] <= 1e-4, st
        assert st["pooled_s_out_of_tol"] <= (2e-3 if kw["binary"] and st["layer"] > 1 else 1e-4), st
        if "sign_bits" in st:
            # packed sign bits: equal except where |u + beta| is at rounding level (SURVEY 7.3.2)
            assert st["sign_mismatch_rate"] <= 1e-4, st
            assert st["sign_mismatch_max_rel_t"] <= 1e-5, st
            assert st["sign_mismatch_scalar_channels"] == 0, st       # s_j - s_i is one exact subtraction
    lf = out["logits_forced"]
    if not kw["binary"]:
        assert lf["out_of_tol"] == 0.0 and lf["argmax_equal"] == 1.0, lf
    else:
        assert lf["argmax_equal"] >= 0.99, lf
