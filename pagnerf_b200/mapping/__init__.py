"""Panoptic point-map export on the device (the reference's utils/render_map.py), its split into objects, lookups of 3-D points
and rendered pixels into the map's objects, the map's projection into camera views and its objects' visibility in them."""
from .panoptic_map import (PanopticPoints, InstanceSummary, InstanceComponents, MapIndex, MapLookup, MapView, ObjectVisibility,
                           extract_panoptic_map, instance_summary, instance_components, map_index, lookup_points, lookup_rays, project_map,
                           object_visibility, write_ply)

__all__ = ["PanopticPoints", "InstanceSummary", "InstanceComponents", "MapIndex", "MapLookup", "MapView", "ObjectVisibility",
           "extract_panoptic_map", "instance_summary", "instance_components", "map_index", "lookup_points", "lookup_rays", "project_map",
           "object_visibility", "write_ply"]
