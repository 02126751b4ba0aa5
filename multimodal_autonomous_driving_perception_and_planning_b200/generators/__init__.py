from ..visualization.yuv_out import bgr_to_nv12          # one implementation of both directions' layouts
from .synthetic_data import SyntheticDataGenerator, multi_camera_batch

__all__ = ["SyntheticDataGenerator", "bgr_to_nv12", "multi_camera_batch"]
