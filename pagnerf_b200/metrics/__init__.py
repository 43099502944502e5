"""Device-side validation metrics with the reference's interfaces (utils/metrics/*.py)."""
from .panoptic_quality import PanopticQuality
from .scene_panoptic_quality import ScenePanopticQuality

__all__ = ["PanopticQuality", "ScenePanopticQuality"]
