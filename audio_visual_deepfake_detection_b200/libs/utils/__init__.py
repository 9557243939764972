from .nms import batched_nms
from .infer_utils import inference_one_epoch, inference_sharded, valid_one_epoch, fix_random_seed, AverageMeter
from .results import merge_results, filter_segments, video_probability, iter_result_records
from .metrics import ANETdetection, load_gt_seg_from_json, load_gt_seg_from_metadata
from .Evaluation import ANETproposal, average_recall_vs_avg_nr_proposals

__all__ = ["batched_nms", "inference_one_epoch", "inference_sharded", "valid_one_epoch", "fix_random_seed", "AverageMeter",
           "merge_results", "filter_segments", "video_probability", "iter_result_records", "ANETdetection",
           "load_gt_seg_from_json", "load_gt_seg_from_metadata", "ANETproposal", "average_recall_vs_avg_nr_proposals"]
