"""Moving image -> fixed frame: the transformed-image export of `EvaluateMetrics._export_transformed_image`
(reference _dock_widget.py:1095-1130), which lets the registered volumes be overlaid voxel by voxel.
SURVEY §8(f) row 5.

The reference resamples through SimpleITK; here the contract is scipy.ndimage.affine_transform in voxel index space
(order 0 or 1, mode='constant').  Agreement with the SimpleITK export itself is not verified.
"""
import numpy as np

from .. import device as D

__all__ = ["transform_image"]

_DIRECT = (np.dtype(np.uint16), np.dtype(np.int32), np.dtype(np.float32))


def transform_image(moving_image, transform, output_shape, order=0, cval=0):
    """The moving image resampled into a grid of `output_shape` (the fixed image's), on the GPU.

    moving_image  (nz, ny, nx) uint16, int32 or float32 volume; other integer dtypes go through int32 when their
                  values fit, and come back in their own dtype
    transform     4 x 4 registration transform mapping moving zyx to fixed zyx, in voxel units (as
                  `estimate_transform_*` return it or `load_transform` reads it)
    order         0 = nearest (label volumes), 1 = trilinear (intensity images)
    cval          value of the output voxels that map outside the moving image
    Returns a numpy array of `output_shape` with the moving image's dtype.  Equal to
    scipy.ndimage.affine_transform(moving_image, M[:3, :3], offset=M[:3, 3], output_shape, order, mode='constant',
    cval) with M = np.linalg.inv(transform).
    """
    a = np.asarray(moving_image)
    if a.ndim != 3:
        raise ValueError("expected a 3-D volume, got %d-D" % a.ndim)
    if len(output_shape) != 3 or min(output_shape) < 1:
        raise ValueError("output_shape must be three extents >= 1, got %r" % (output_shape,))
    if order not in (0, 1):
        raise ValueError("order must be 0 or 1, got %r" % (order,))
    T = np.asarray(transform, dtype=np.float64)
    if T.shape != (4, 4):
        raise ValueError("transform must be 4 x 4, got %s" % (T.shape,))
    i32 = np.iinfo(np.int32)
    if a.dtype in _DIRECT:
        work = a
    elif np.issubdtype(a.dtype, np.integer):
        if a.size and (a.min() < i32.min or a.max() > i32.max):
            raise ValueError("%s values outside the int32 range are not supported" % a.dtype)
        work = a.astype(np.int32)
    else:
        raise ValueError("volume must have an integer or float32 dtype, got %s" % a.dtype)
    M = np.linalg.inv(T)                       # output (fixed) index -> source (moving) index, as scipy takes it
    torch = D._torch()
    work = np.ascontiguousarray(work)
    if work.dtype == np.uint16:
        src = torch.from_numpy(work.view(np.int16)).cuda().view(torch.uint16)
    else:
        src = torch.from_numpy(work).cuda()
    out = D.resample_affine(src, torch.from_numpy(M).cuda(), output_shape, order, cval)
    if work.dtype == np.uint16:
        res = out.view(torch.int16).cpu().numpy().view(np.uint16)
    else:
        res = out.cpu().numpy()
    if res.dtype != a.dtype:                   # saturate into the caller's dtype, as scipy's cast does
        info = np.iinfo(a.dtype)
        res = np.clip(res, max(info.min, i32.min), min(info.max, i32.max)).astype(a.dtype)
    return res
