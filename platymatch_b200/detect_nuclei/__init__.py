"""Nuclei detection in intensity volumes (the reference's platymatch/detect_nuclei)."""
from .ss_log import find_spheres, sphere_intersection  # noqa: F401
