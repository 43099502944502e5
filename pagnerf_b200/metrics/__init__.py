"""Device-side validation metrics with the reference's interfaces (utils/metrics/*.py)."""
from .panoptic_quality import PanopticQuality

__all__ = ["PanopticQuality"]
