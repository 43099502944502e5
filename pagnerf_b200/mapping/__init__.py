"""Panoptic point-map export on the device (the reference's utils/render_map.py), its split into objects, lookups of 3-D points
and rendered pixels into the map's objects, and the map's projection into camera views."""
from .panoptic_map import (PanopticPoints, InstanceSummary, InstanceComponents, MapIndex, MapLookup, MapView, extract_panoptic_map,
                           instance_summary, instance_components, map_index, lookup_points, lookup_rays, project_map, write_ply)

__all__ = ["PanopticPoints", "InstanceSummary", "InstanceComponents", "MapIndex", "MapLookup", "MapView", "extract_panoptic_map",
           "instance_summary", "instance_components", "map_index", "lookup_points", "lookup_rays", "project_map", "write_ply"]
