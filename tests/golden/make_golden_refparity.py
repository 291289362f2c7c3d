#!/usr/bin/env python
"""Generate tests/golden/refparity_<cfg>.npz: seeded samples of the CPU oracle's record (kNN rows, pooled per-point
features, sign planes, logits) at the shapes of tests/test_gpu_reference.py, which the full-size parity test runs
against where the reference's model code is not staged (tests/refparity.py: oracle_record / pin_to_golden).

    python tests/golden/make_golden_refparity.py
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from tests import refparity  # noqa: E402
from svnet_b200.synthetic import one_hot_labels, synthetic_clouds  # noqa: E402

if __name__ == "__main__":
    for name, kw in refparity.CASES.items():
        _, sd = refparity.build_ours(kw["kind"], kw["k"], kw["binary"], kw["ncls"], kw["seed"], "cpu")
        x = synthetic_clouds(kw["B"], kw["N"], kw["seed"])
        extra = (one_hot_labels(kw["B"]),) if kw["kind"] == "SV_DGCNN_PSEG" else ()
        rec = refparity.oracle_record(sd, kw["kind"], kw["k"], kw["binary"], x, extra, "cpu")
        path = os.path.join(HERE, "refparity_%s.npz" % name)
        np.savez_compressed(path, config=np.array(json.dumps(kw)), **refparity.golden_samples(rec))
        print("wrote %s %.1f KiB" % (path, os.path.getsize(path) / 1024))
