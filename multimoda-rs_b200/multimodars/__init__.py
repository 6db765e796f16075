"""Drop-in subset of the `multimodars` Python surface (multimodars/__init__.py:6-84) for the
Hausdorff rotation-sweep path, running on B200 through libmmrs_b200.so."""
from ._types import (PyCenterline, PyCenterlinePoint, PyContour, PyContourPoint, PyContourType, PyFrame, PyGeometry, PyGeometryPair, PyInputData,
                     PyRecord, numpy_to_inputdata)
from ._converters import numpy_to_centerline, numpy_to_geometry, to_array
from ._processing import (align_combined, align_manual, align_three_point, to_obj, from_array_doublepair, from_array_full, from_array_single,
                          from_array_singlepair, from_file_doublepair, from_file_full, from_file_single,
                          from_file_singlepair, get_context)
from ._native import MmrsError
from ._rigid import find_best_rigid_transform
from ._vtp import read_centerline_vtp
from ._centerline import load_centerline, prepare_centerline

__all__ = [n for n in dir() if not n.startswith("_")]
