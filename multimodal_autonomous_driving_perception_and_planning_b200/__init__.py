"""B200-native batched lane detection: a drop-in for the lane-detection hot path of
bhavyageethika/multimodal_autonomous_driving_perception_and_planning
(``src/perception/lane_detector.py``).  See DESIGN.md / INTEGRATION.md at the repo root."""
from .generators import SyntheticDataGenerator, bgr_to_nv12, multi_camera_batch
from .loaders import FrameIngest
from .perception import LaneDetector, LaneLine
from .visualization import DrawList, OverlayRenderer, bgr_to_i420, draw_lanes_batch

__all__ = ["DrawList", "FrameIngest", "LaneDetector", "LaneLine", "OverlayRenderer", "SyntheticDataGenerator", "bgr_to_i420",
           "bgr_to_nv12", "draw_lanes_batch", "multi_camera_batch"]
__version__ = "0.1.0"
