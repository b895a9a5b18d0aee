"""SURVEY §8(f) row 2 — label image -> detections (reference _dock_widget.py:497-521) and the size-derived
RANSAC threshold (:613-618).  CPU: the oracle restatement against hand-computed cases.  GPU: bit-exact
parity of the streaming kernel with the oracle."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def test_oracle_detections_from_labels_known_answers():
    import oracle as O
    vol = np.zeros((3, 4, 5), dtype=np.int32)
    vol[0, 0, 0] = 7                                     # single voxel
    vol[1, 1:3, 2:4] = 3                                 # 2 x 2 patch in plane z = 1
    vol[2, 3, :] = 12                                    # a full row
    det, sizes, ids = O.detections_from_labels(vol, anisotropy=2.5)
    assert ids.tolist() == [3, 7, 12]                    # np.unique order, background dropped
    assert np.array_equal(det, np.array([[1.0, 0.0, 2.0], [1.5, 0.0, 3.0], [2.5, 0.0, 2.0]]))
    assert sizes.tolist() == [10.0, 2.5, 12.5]           # anisotropy * voxel count
    assert O.ransac_error_from_sizes([], sizes) == 16
    assert O.ransac_error_from_sizes([8.0, 8.0], [27.0]) == pytest.approx(0.5 * (2.0 + 3.0))
    det0, sizes0, ids0 = O.detections_from_labels(np.zeros((2, 2, 2), dtype=np.uint16))
    assert det0.shape == (3, 0) and len(sizes0) == 0 and len(ids0) == 0


def test_ransac_error_from_sizes_host_logic():
    """reference _dock_widget.py:613-618 (no GPU involved)."""
    from platymatch_b200.utils.labels import ransac_error_from_sizes
    assert ransac_error_from_sizes(None, [1.0]) == 16 and ransac_error_from_sizes([], []) == 16
    assert ransac_error_from_sizes([8.0, 8.0], [27.0, 27.0, 27.0]) == pytest.approx(2.5)


def _rows_golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "rows.npz"))


def test_oracle_detections_match_reference_widget():
    """tests/golden/rows.npz: `self.moving_detections` / `self.fixed_detections` as stored by the reference's own
    `_click_run` (run headless on a fake widget by oracle/make_golden_rows.py)."""
    import oracle as O
    g = _rows_golden()
    for side in ("moving", "fixed"):
        det, sizes, ids = O.detections_from_labels(g["label_%s_vol" % side])
        assert np.array_equal(det, g["label_%s_det" % side])


@pytest.mark.gpu
def test_detections_match_reference_widget():
    from platymatch_b200.utils.labels import detections_from_labels
    g = _rows_golden()
    for side in ("moving", "fixed"):
        det, sizes, ids = detections_from_labels(g["label_%s_vol" % side])
        assert np.array_equal(det, g["label_%s_det" % side])


@pytest.mark.gpu
@pytest.mark.parametrize("shape,n,dtype,sparse", [((64, 96, 128), 60, np.int32, False), ((33, 47, 61), 40, np.uint16, False),
                                                   ((40, 50, 3), 25, np.int32, True), ((128, 128, 128), 400, np.uint16, True),
                                                   ((5, 7, 9), 0, np.int32, False), ((1, 1, 70001), 3, np.int32, False)])
def test_detections_from_labels_bit_exact(shape, n, dtype, sparse):
    import oracle as O
    from platymatch_b200.synthetic import make_label_volume
    from platymatch_b200.utils.labels import detections_from_labels, ransac_error_from_sizes
    vol = make_label_volume(shape, n, seed=n + shape[2], dtype=dtype, sparse_ids=sparse)
    det, sizes, ids = detections_from_labels(vol, anisotropy=1.7)
    rdet, rsizes, rids = O.detections_from_labels(vol, anisotropy=1.7)
    assert np.array_equal(ids, rids)
    assert det.shape == rdet.shape and np.array_equal(det, rdet)          # exact integer sums -> identical means
    assert np.array_equal(sizes, rsizes)
    if n:
        assert ransac_error_from_sizes(sizes, sizes) == O.ransac_error_from_sizes(rsizes, rsizes)


@pytest.mark.gpu
def test_label_kernels_agree(monkeypatch):
    """The round-2 streaming kernel (per-thread run-length items) and the round-1 warp-cooperative kernel (kept for
    unaligned volumes, PM_LABEL_WARP_KERNEL=1) produce identical tables on a crowded volume with touching nuclei."""
    from platymatch_b200.synthetic import make_label_volume
    from platymatch_b200.utils.labels import detections_from_labels
    for shape, dtype in (((70, 83, 101), np.int32), ((70, 83, 101), np.uint16), ((16, 16, 1030), np.int32)):
        vol = make_label_volume(shape, 500, radius=(2.0, 7.0), seed=4, dtype=dtype)
        a = detections_from_labels(vol)
        monkeypatch.setenv("PM_LABEL_WARP_KERNEL", "1")
        b = detections_from_labels(vol)
        monkeypatch.delenv("PM_LABEL_WARP_KERNEL")
        for x, y in zip(a, b):
            assert np.array_equal(x, y)


@pytest.mark.gpu
def test_detections_from_labels_int64_and_negative_background():
    import oracle as O
    from platymatch_b200.utils.labels import detections_from_labels
    rng = np.random.default_rng(3)
    vol = rng.integers(0, 6, size=(9, 10, 11)).astype(np.int64)
    det, sizes, ids = detections_from_labels(vol)
    rdet, rsizes, rids = O.detections_from_labels(vol)
    assert np.array_equal(ids, rids) and np.array_equal(det, rdet) and np.array_equal(sizes, rsizes)
    with pytest.raises(ValueError):
        detections_from_labels(vol.astype(np.float32))


@pytest.mark.gpu
def test_registration_from_label_volumes():
    """End of the row: two label volumes -> detections + sizes -> size-derived RANSAC error -> registration.
    Nuclei sit on an ellipsoidal shell; the moving volume is the same embryo rendered after a known rigid motion."""
    import oracle as O
    import platymatch_b200 as pm
    from platymatch_b200.synthetic import make_label_volume
    from platymatch_b200.utils.labels import detections_from_labels, ransac_error_from_sizes
    rng = np.random.default_rng(8)
    n, shape = 400, (160, 160, 160)
    centre = np.array(shape) / 2.0
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    fixed_c = centre + d * np.array([55.0, 48.0, 42.0]) + rng.normal(0, 1.5, size=(n, 3))
    ang = np.deg2rad(12.0)
    R = np.array([[1, 0, 0], [0, np.cos(ang), -np.sin(ang)], [0, np.sin(ang), np.cos(ang)]])
    shift = np.array([3.0, -5.0, 4.0])
    moving_c = (fixed_c - centre - shift) @ R + centre            # fixed = R (moving - centre) + centre + shift
    fixed_vol = make_label_volume(shape, radius=(2.0, 3.0), seed=1, centers=fixed_c)
    moving_vol = make_label_volume(shape, radius=(2.0, 3.0), seed=2, centers=moving_c, dtype=np.uint16)
    fd, fs, fids = detections_from_labels(fixed_vol, 1.0)
    md, ms, mids = detections_from_labels(moving_vol, 1.0)
    assert np.array_equal(fd, O.detections_from_labels(fixed_vol, 1.0)[0])
    err = ransac_error_from_sizes(ms, fs)
    assert err == O.ransac_error_from_sizes(ms, fs) and 1.0 < err < 16.0
    res = pm.estimate_transform_unsupervised(md, fd, ransac_trials=4000, ransac_error=err, seed=2)
    A = res["transform"]
    assert np.abs(A[:3, :3] - R).max() < 0.03, A
    moved = A[:3, :3] @ moving_c.T + A[:3, 3:4]
    assert np.median(np.linalg.norm(moved - fixed_c.T, axis=0)) < 1.5
