"""SURVEY §8(f) row 5 — the volume resample (reference _dock_widget.py:1095-1130): argument checks that run on the
host, before any CUDA call or device transfer (no GPU needed)."""
import ctypes

import numpy as np
import pytest


def test_resample_argument_validation_is_host_side():
    from platymatch_b200 import _lib
    lib = _lib.load()
    # 16-byte-aligned stand-ins for device buffers; never dereferenced, because every call below is refused first
    p, q = ctypes.c_void_p(1 << 12), ctypes.c_void_p(1 << 20)

    def call(src=p, dtype=0, s=(4, 5, 6), m=p, order=0, dst=q, d=(3, 4, 5)):
        return lib.pm_resample_affine(src, dtype, *s, m, order, 0.0, dst, *d, None)

    assert call(src=None) == -1
    assert b"null pointer" in lib.pm_last_error_string()
    assert call(m=None) == -1 and call(dst=None) == -1
    for s, d in (((0, 5, 6), (3, 4, 5)), ((4, 5, 6), (3, 0, 5)), ((4, 5, -1), (3, 4, 5)), ((4, 5, 6), (3, 4, 0))):
        assert call(s=s, d=d) == -1
        assert b"extent" in lib.pm_last_error_string()
    assert call(order=2) == -1 and b"order" in lib.pm_last_error_string()
    assert call(order=-1) == -1
    assert call(dtype=3) == -1 and b"dtype" in lib.pm_last_error_string()
    # overlapping ranges: dst inside src, src inside dst, and the two touching by one element
    assert call(dst=ctypes.c_void_p((1 << 12) + 16)) == -1
    assert b"overlap" in lib.pm_last_error_string()
    assert call(src=ctypes.c_void_p((1 << 20) + 32)) == -1
    assert call(dst=ctypes.c_void_p((1 << 12) + 4 * 4 * 5 * 6 - 4)) == -1                      # last int32 of src
    assert call(dtype=1, dst=ctypes.c_void_p((1 << 12) + 2 * 4 * 5 * 6 - 2)) == -1             # last uint16 of src


@pytest.mark.parametrize("dtype", [np.float64, np.complex64, np.bool_])
def test_transform_image_rejects_dtype_before_device(dtype, monkeypatch):
    from platymatch_b200 import device as D
    from platymatch_b200.utils.images import transform_image

    def no_device():
        raise AssertionError("the device was touched")
    monkeypatch.setattr(D, "_torch", no_device)
    with pytest.raises(ValueError):
        transform_image(np.zeros((2, 3, 4), dtype=dtype), np.eye(4), (2, 3, 4))


def test_transform_image_rejects_bad_arguments_before_device(monkeypatch):
    from platymatch_b200 import device as D
    from platymatch_b200.utils.images import transform_image

    def no_device():
        raise AssertionError("the device was touched")
    monkeypatch.setattr(D, "_torch", no_device)
    vol = np.zeros((2, 3, 4), dtype=np.int32)
    for args, kw in (((vol[0], np.eye(4), (2, 3, 4)), {}), ((vol, np.eye(3), (2, 3, 4)), {}),
                     ((vol, np.eye(4), (2, 0, 4)), {}), ((vol, np.eye(4), (2, 3)), {}),
                     ((vol, np.eye(4), (2, 3, 4)), {"order": 3}),
                     ((np.full((2, 3, 4), 2 ** 40, dtype=np.int64), np.eye(4), (2, 3, 4)), {})):
        with pytest.raises(ValueError):
            transform_image(*args, **kw)
