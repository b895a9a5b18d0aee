"""platymatch_b200 — B200-native (sm_100a) implementation of PlatyMatch's estimate_transform hot path.

Drop-in for the functions the reference's napari widget imports (platymatch/_dock_widget.py:10,16-21):

    reference module                                      here
    platymatch.utils.utils                                platymatch_b200.utils.utils
    platymatch.estimate_transform.shape_context           platymatch_b200.estimate_transform.shape_context
    platymatch.estimate_transform.find_transform          platymatch_b200.estimate_transform.find_transform
    platymatch.estimate_transform.apply_transform         platymatch_b200.estimate_transform.apply_transform
    platymatch.estimate_transform.perform_icp             platymatch_b200.estimate_transform.perform_icp
    scipy.optimize.linear_sum_assignment                  platymatch_b200.lap.linear_sum_assignment

plus the fused pipeline (`estimate_transform_unsupervised`, `estimate_transform_supervised`) restating
`EstimateTransform._click_run` (_dock_widget.py:526-721).  Hand-written CUDA behind a C ABI
(include/platymatch_b200.h, platymatch_b200/csrc); no CPU fallback.
"""
__version__ = "0.2.0"

from ._lib import load as load_library, LIB_PATH, PlatyMatchError  # noqa: F401


def __getattr__(name):  # lazy: importing the package must not require torch / a GPU
    if name in ("estimate_transform_unsupervised", "estimate_transform_supervised", "describe_cloud",
                "register_described", "HYPOTHESES_REFERENCE", "HYPOTHESES_DISTINCT"):
        from . import pipeline
        return getattr(pipeline, name)
    if name == "linear_sum_assignment":
        from .lap import linear_sum_assignment
        return linear_sum_assignment
    raise AttributeError(name)
