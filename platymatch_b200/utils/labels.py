"""Label image -> detections, the first stage of `EstimateTransform._click_run` when the inputs are
instance-segmentation volumes instead of CSV detections (reference _dock_widget.py:497-521), and the
data-dependent RANSAC threshold derived from the nucleus sizes (:613-618).  SURVEY §8(f) row 2.
"""
import numpy as np

from .. import device as D

__all__ = ["detections_from_labels", "ransac_error_from_sizes"]

_ID_MAX = 2 ** 31 - 1


def _check_label_volume(a, name):
    """A host label volume as the int32 / uint16 array the label kernels read; refused before any device work.
    Other integer dtypes go through int32 with ids <= 0 as background (0); ids above 2^31 - 1 are refused."""
    a = np.asarray(a)
    if a.ndim != 3:
        raise ValueError("%s: expected a 3-D label volume, got %d-D" % (name, a.ndim))
    if not np.issubdtype(a.dtype, np.integer):
        raise ValueError("%s: label volumes must have an integer dtype, got %s" % (name, a.dtype))
    if a.dtype in (np.dtype(np.int32), np.dtype(np.uint16)):
        return np.ascontiguousarray(a)
    if a.size and a.max() > _ID_MAX:
        raise ValueError("%s: ids above 2^31 - 1 are not supported (largest is %d)" % (name, int(a.max())))
    return np.ascontiguousarray(np.maximum(a, 0).astype(np.int32))          # (ids <= 0 are background)


def detections_from_labels(label_image, anisotropy=1.0):
    """reference _dock_widget.py:497-509 (moving) / :512-521 (fixed).

    label_image: (nz, ny, nx) integer array, ids <= 0 = background (int32 and uint16 are read directly; other integer
    dtypes go through int32, ids above 2^31 - 1 are refused).  Returns
      detections  (3, N) float64, rows z, y, x = np.mean of the voxel indices of each id (:506-507,520-521)
      sizes       (N,)  float64 = anisotropy * voxel count (:508,517)
      ids         (N,)  the positive ids in np.unique order (:497-500), in label_image's dtype
    One streaming pass on the GPU instead of one np.where pass per id.  Sparse ids are fine at any volume size: when
    a table with one entry per possible id would cost more than the volume warrants, the ids are compacted on the GPU
    first (device.label_centroids), at 4 bytes per voxel of temporary device memory plus at most 343 MB of scratch.
    """
    a = np.asarray(label_image)
    work = _check_label_volume(a, "label_image")
    ids, cen, sizes = D.label_centroids(D.to_device_volume(work), anisotropy)
    return cen.cpu().numpy().T.copy(), sizes.cpu().numpy(), ids.cpu().numpy().astype(a.dtype, copy=False)


def ransac_error_from_sizes(moving_nucleus_size, fixed_nucleus_size):
    """reference _dock_widget.py:613-618 — 16 without sizes (CSV mode), else the approximate mean nucleus radius."""
    if moving_nucleus_size is None or fixed_nucleus_size is None or len(moving_nucleus_size) == 0 \
            or len(fixed_nucleus_size) == 0:
        return 16
    return 0.5 * (np.average(moving_nucleus_size) ** (1 / 3) + np.average(fixed_nucleus_size) ** (1 / 3))
