"""DESIGN §8 row 7 — the label-overlap table and instance matching: every refusal runs on the host, before any CUDA call
or device transfer (no GPU needed)."""
import ctypes

import numpy as np
import pytest


def test_label_overlap_argument_validation_is_host_side():
    from platymatch_b200 import _lib
    lib = _lib.load()
    # 16-byte-aligned stand-ins for device buffers; never dereferenced, because every call below is refused first
    p, q, k, c, n, w = (ctypes.c_void_p(x << 12) for x in (1, 2, 3, 4, 5, 6))
    cap = 1024
    need = lib.pm_label_overlap_workspace_bytes(cap)
    assert need >= 2 * cap * 8
    assert lib.pm_label_overlap_workspace_bytes(2048) - need == 2 * 1024 * 8

    def call(a=p, da=0, b=q, db=1, s=(4, 5, 6), capacity=cap, keys=k, counts=c, n_out=n, ws=w, nbytes=need):
        return lib.pm_label_overlap(a, da, b, db, *s, capacity, keys, counts, n_out, ws, nbytes, None)

    for kw in ({"a": None}, {"b": None}, {"keys": None}, {"counts": None}, {"n_out": None}, {"ws": None}):
        assert call(**kw) == -1, kw
        assert b"null pointer" in lib.pm_last_error_string()
    for kw in ({"da": 2}, {"db": 2}, {"da": -1}, {"db": 7}):
        assert call(**kw) == -1, kw
        assert b"dtype" in lib.pm_last_error_string()
    for s in ((0, 5, 6), (4, 0, 6), (4, 5, 0), (-1, 5, 6)):
        assert call(s=s) == -1, s
        assert b"extent" in lib.pm_last_error_string()
    for capacity in (0, 3, 1000, 1025, (1 << 40) + 1):
        assert call(capacity=capacity, nbytes=1 << 62) == -1, capacity
        assert b"power of two" in lib.pm_last_error_string()
    for kw in ({"a": ctypes.c_void_p((1 << 12) + 4)}, {"b": ctypes.c_void_p((2 << 12) + 2)},
               {"keys": ctypes.c_void_p((3 << 12) + 8)}, {"counts": ctypes.c_void_p((4 << 12) + 8)},
               {"n_out": ctypes.c_void_p((5 << 12) + 8)}, {"ws": ctypes.c_void_p((6 << 12) + 8)}):
        assert call(**kw) == -1, kw
        assert b"16-byte aligned" in lib.pm_last_error_string()
    assert call(nbytes=need - 1) == -3
    assert b"workspace too small" in lib.pm_last_error_string()


def _no_device(monkeypatch):
    from platymatch_b200 import device as D

    def no_device():
        raise AssertionError("the device was touched")
    monkeypatch.setattr(D, "_torch", no_device)


BAD_PAIRS = [
    (np.zeros((4, 5), np.int32), np.zeros((4, 5), np.int32)),                          # not 3-D
    (np.zeros((2, 4, 5, 1), np.int32), np.zeros((2, 4, 5, 1), np.int32)),
    (np.zeros((2, 4, 5), np.int32), np.zeros((2, 4, 6), np.int32)),                    # shapes differ
    (np.zeros((2, 4, 5), np.uint16), np.zeros((2, 5, 4), np.int32)),
    (np.zeros((2, 4, 5), np.float32), np.zeros((2, 4, 5), np.int32)),                  # not integer
    (np.zeros((2, 4, 5), np.int32), np.zeros((2, 4, 5), np.float64)),
    (np.zeros((2, 4, 5), np.bool_), np.zeros((2, 4, 5), np.int32)),
    (np.full((2, 4, 5), 2 ** 31, np.int64), np.zeros((2, 4, 5), np.int32)),           # ids above 2^31 - 1
    (np.zeros((2, 4, 5), np.int32), np.full((2, 4, 5), 2 ** 32 - 1, np.uint32)),
]


@pytest.mark.parametrize("pair", range(len(BAD_PAIRS)))
def test_label_volumes_refused_before_device(pair, monkeypatch):
    from platymatch_b200.evaluate_metrics import label_contingency, match_labels
    _no_device(monkeypatch)
    a, b = BAD_PAIRS[pair]
    with pytest.raises(ValueError):
        label_contingency(a, b)
    with pytest.raises(ValueError):
        match_labels(a, b)


BAD_VOLUMES = [np.zeros((4, 5), np.int32), np.zeros((2, 4, 5, 1), np.uint16), np.zeros((2, 4, 5), np.float32),
               np.zeros((2, 4, 5), np.bool_), np.full((2, 4, 5), 2 ** 31, np.int64),
               np.full((2, 4, 5), 2 ** 32 - 1, np.uint32)]


@pytest.mark.parametrize("vol", range(len(BAD_VOLUMES)))
def test_detections_from_labels_refused_before_device(vol, monkeypatch):
    """detections_from_labels follows the label-volume policy of the table pass, checked before any device work."""
    from platymatch_b200.utils.labels import detections_from_labels
    _no_device(monkeypatch)
    with pytest.raises(ValueError):
        detections_from_labels(BAD_VOLUMES[vol])


@pytest.mark.parametrize("thresholds", [(0.0,), (1.5,), (-0.1,), (0.5, float("nan")), (), (0.5, 1.0000001)])
def test_thresholds_refused_before_device(thresholds, monkeypatch):
    from platymatch_b200.evaluate_metrics import match_labels
    _no_device(monkeypatch)
    a = np.zeros((2, 3, 4), np.int32)
    with pytest.raises(ValueError):
        match_labels(a, a, thresholds=thresholds)


def test_other_integer_dtypes_go_through_int32():
    """int64 / int8 / uint32 volumes within range become int32 with ids <= 0 as background; no device involved."""
    from platymatch_b200.utils.labels import _check_label_volume
    a = np.array([[[-(2 ** 40), -1, 0, 5, 2 ** 31 - 1]]], dtype=np.int64)
    got = _check_label_volume(a, "a")
    assert got.dtype == np.int32 and got.tolist() == [[[0, 0, 0, 5, 2 ** 31 - 1]]]
    assert _check_label_volume(np.array([[[-3, 4]]], np.int8), "a").tolist() == [[[0, 4]]]
    u = np.array([[[2 ** 31 - 1, 7]]], np.uint32)
    assert _check_label_volume(u, "a").tolist() == [[[2 ** 31 - 1, 7]]]
    i32 = np.array([[[-3, 4]]], np.int32)
    assert _check_label_volume(i32, "a").dtype == np.int32            # read directly: the kernel maps -3 to 0


def test_assignment_column_limit_refused_on_host():
    """More than 24576 ids of one volume with an admissible partner is refused (the assignment's column limit) before
    any matrix is built; ids without an admissible partner do not count, and exactly 24576 is accepted."""
    from platymatch_b200.evaluate_metrics import LAP_MAX_COLUMNS, _matching_problem
    n = LAP_MAX_COLUMNS + 1
    ids = np.arange(1, n + 1, dtype=np.int64)
    with pytest.raises(ValueError, match="24577 instances"):
        _matching_problem(ids, ids, np.ones(n), 0.5)
    with pytest.raises(ValueError, match="24576 columns"):       # one true id against 24577 predicted ones
        _matching_problem(np.ones(n, np.int64), ids, np.ones(n), 0.5)
    iou = np.ones(n)
    iou[-1] = 0.25                                                # the last pair is not admissible at 0.5
    prob = _matching_problem(ids, ids, iou, 0.5)
    assert prob[1].size == prob[2].size == LAP_MAX_COLUMNS
    with pytest.raises(ValueError):                               # at 0.2 every pair is admissible again
        _matching_problem(ids, ids, iou, 0.2)
