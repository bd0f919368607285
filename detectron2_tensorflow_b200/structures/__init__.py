from .box_list import BoxList, SparseBoxList
from .image_list import ImageList
from .mask_ops import reframe_box_masks_to_image_masks, reframe_box_masks_to_rle, rle_to_coco
from .box_list_ops import pairwise_iou
