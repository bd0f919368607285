from .poolers import ROIPooler, assign_boxes_to_levels
from .box_regression import Box2BoxTransform
from .proposal_generator.rpn_outputs import find_top_rpn_proposals, RPNOutputs
from .roi_heads.fast_rcnn import fast_rcnn_inference, FastRCNNOutputs
from .single_stage_heads.retinanet import RetinaNetInference
from .anchor_generator import DefaultAnchorGenerator, GridAnchors
from .matcher import Matcher, label_boxes
from .single_stage_heads.yolov4_outputs import YOLOv4Inference
from .single_stage_heads.solo_v2 import (point_nms, solo_mask_encode, solo_dynamic_masks, solo_upsample_masks,
                                         solo_upsample_rle, SOLOv2Inference)
from .postprocessing import coco_results, detector_postprocess, detector_postprocess_rle
from .roi_heads.mask_head import mask_rcnn_inference
from .sampling import subsample_labels, subsample_labels_batched
