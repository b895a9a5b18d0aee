"""bench.py --dump-outputs writes the results of the last timed step, the same on every run with the same arguments."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu
ARGS = ["--n-fixed", "400", "--trials", "64", "--steps", "3", "--warmup", "1", "--lean"]


def _dump(d):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *ARGS, "--dump-outputs", str(d)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    return {f[:-len(".npy")]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_outputs_of_last_timed_step(tmp_path):
    import platymatch_b200 as pm
    from platymatch_b200.synthetic import make_pair
    a, b = _dump(tmp_path / "a"), _dump(tmp_path / "b")
    assert {"transform", "inliers", "assignment_fixed", "cost_sample", "cost_sample_index"} <= set(a) == set(b)
    assert sum(x.nbytes for x in a.values()) <= 64e6
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        assert np.array_equal(a[k], b[k]), k
    # step 2 of 3, the last timed one, registers the bench's pair slot 2 with seed 2
    p = make_pair(400, seed=400 + 97 * 2)
    res = pm.estimate_transform_unsupervised(p["moving"], p["fixed"], ransac_trials=64, seed=2, keep_cost=True)
    assert np.array_equal(a["inliers"], res["inliers"])
    assert np.array_equal(a["assignment_fixed"], np.stack([f for _, f in res["assignments"]]))
    assert np.allclose(a["transform"], res["transform"], rtol=1e-12, atol=1e-12)
    idx = a["cost_sample_index"].astype(np.int64)
    n2 = p["fixed"].shape[1]
    cost = res["cost"][:, :, :n2].reshape(len(res["cost"]), -1)
    assert np.array_equal(a["cost_sample"], cost[:, idx])
