"""Panoptic point-map export on the device (the reference's utils/render_map.py)."""
from .panoptic_map import PanopticPoints, InstanceSummary, extract_panoptic_map, instance_summary, write_ply

__all__ = ["PanopticPoints", "InstanceSummary", "extract_panoptic_map", "instance_summary", "write_ply"]
