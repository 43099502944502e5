"""Panoptic point-map export on the device (the reference's utils/render_map.py), and its split into objects."""
from .panoptic_map import (PanopticPoints, InstanceSummary, InstanceComponents, extract_panoptic_map, instance_summary,
                           instance_components, write_ply)

__all__ = ["PanopticPoints", "InstanceSummary", "InstanceComponents", "extract_panoptic_map", "instance_summary",
           "instance_components", "write_ply"]
