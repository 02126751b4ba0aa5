from .draw_list import DrawList, color_word
from .overlays import OverlayRenderer, draw_lanes_batch, draw_lanes_records
from .yuv_out import bgr_to_i420, bgr_to_nv12

__all__ = ["DrawList", "color_word", "OverlayRenderer", "draw_lanes_batch", "draw_lanes_records", "bgr_to_i420", "bgr_to_nv12"]
