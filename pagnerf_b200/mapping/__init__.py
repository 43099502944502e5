"""Panoptic point-map export on the device (the reference's utils/render_map.py), its split into objects, and lookups of 3-D points
and rendered pixels into the map's objects."""
from .panoptic_map import (PanopticPoints, InstanceSummary, InstanceComponents, MapIndex, MapLookup, extract_panoptic_map,
                           instance_summary, instance_components, map_index, lookup_points, lookup_rays, write_ply)

__all__ = ["PanopticPoints", "InstanceSummary", "InstanceComponents", "MapIndex", "MapLookup", "extract_panoptic_map",
           "instance_summary", "instance_components", "map_index", "lookup_points", "lookup_rays", "write_ply"]
