"""Operator layer of the hot path (mirror of disprcnn/layers/__init__.py:10-11 for ROIAlign)."""
from .roi_align import ROIAlign, roi_align
from .roi_points import process_input_eval, roi_points

__all__ = ['roi_align', 'ROIAlign', 'roi_points', 'process_input_eval']
