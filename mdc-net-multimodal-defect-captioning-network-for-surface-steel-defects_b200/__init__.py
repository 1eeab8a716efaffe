"""mdcnet_b200 -- B200-native (sm_100a) implementation of MDC-Net's batched inference hot path:
DeiT-III image encoder -> autoregressive caption/box decoder -> box-IoU scoring, behind the
reference's own Python surface (model.py / axial_model.py / inference_p.py / iou_calcualtions.py /
iou_bbox.py).  All arithmetic runs in libmdc_b200.so (hand-written CUDA: tcgen05/TMA GEMMs, strip
attention, fused decode step, batched IoU); there is NO CPU or PyTorch fallback.
"""
from .config import CFG
from .tokenizer import Tokenizer, top_k_sampling, top_k_sampling_with_scores_2d
from .model import Encoder, Decoder, EncoderDecoder, Engine, decode_options
from .axial_model import AxialAttention
from . import axial_model
from .inference import generate, generate_beam, postprocess, postprocess_with_captions, preprocess_gray, preprocess_bgr
from .pipeline import GenerationPipeline, generate_stream
from .iou import (bbox_iou, calculate_batch_iou, calculate_batch_max_iou, calculate_batch_max_iou_torchvision,
                  calculate_batch_max_iou_masked, giou_pairwise, giou_loss_with_scores, calculate_iou, iou_loss)
from .kvcache import PagedKVCache, PageAllocator
from . import parallel
from . import metrics
from .metrics import MeanAveragePrecision, calculate_bleu_scores
from . import _lib

__all__ = ["CFG", "Tokenizer", "top_k_sampling", "top_k_sampling_with_scores_2d", "Encoder", "Decoder", "EncoderDecoder", "Engine", "decode_options", "AxialAttention", "axial_model",
           "generate", "generate_beam", "postprocess", "postprocess_with_captions", "preprocess_gray", "preprocess_bgr", "GenerationPipeline", "generate_stream", "bbox_iou", "calculate_batch_iou", "calculate_batch_max_iou",
           "calculate_batch_max_iou_torchvision", "calculate_batch_max_iou_masked", "giou_pairwise",
           "giou_loss_with_scores", "calculate_iou", "iou_loss", "PagedKVCache", "PageAllocator", "parallel", "metrics", "MeanAveragePrecision", "calculate_bleu_scores"]
