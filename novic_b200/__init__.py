"""novic_b200: B200-native (sm_100a) implementation of NOVIC's object-noun decoder hot path.

Public surface (mirrors the reference's classes for this path):
  PrefixedIterDecoder, EmbeddingDecoder  - embedding_decoder.py
  EmbeddingNoise and its five schemes     - embedding_noise.py
  register(module)                        - make `getattr(embedding_decoder, 'PrefixedIterDecoder')` resolve here
  cache.EmbeddingCacheReader              - embedding_cache.py's file format -> batches on the device (training feeder)
  stats.GenerationStats                   - GenerationTask.update's validity / top-k statistics, on token ids on the device
  targets.make_target_format / encode_targets / decode_targets - the Embedder's target id formats around the tokenizer call
  serve.GenerationPipeline                - double-buffered host -> device -> host inference loop
  ImageEncoder, VitDims                   - CLIP ViT-H/14 image encoder (open_clip `visual.*` parameters)
  SiglipImageEncoder, SiglipDims          - SigLIP ViT-B/16 image encoder, the reference's default embedder (`visual.trunk.*` parameters)
  SIGLIP_SO400M                           - SiglipDims of SigLIP SO400M/14, the image encoder of the F = 1152 checkpoints
  EncoderDecoder                          - either encoder feeding the decoder on the device (greedy and beam search)
  optim.FusedAdamW, dist.train_step       - training step: fused clip + AdamW, overlapped gradient all-reduce
"""
from .decoder import EmbeddingDecoder, ParamCount, PrefixedIterDecoder
from .noise import (AngleNoise, EmbeddingNoise, GaussAngleNoise, GaussElemNoise, GaussElemUniformAngleNoise, GaussVecNoise,
                    UniformAngleNoise)
from .factory import DEFAULT_DECODER_KWARGS, default_decoder, register
from .encoder import SIGLIP_SO400M, EncoderDecoder, ImageEncoder, SiglipDims, SiglipImageEncoder, VitDims
from . import cache, stats, synth, targets

__all__ = [
    "EmbeddingDecoder", "ParamCount", "PrefixedIterDecoder", "EmbeddingNoise", "AngleNoise", "GaussAngleNoise", "GaussElemNoise",
    "GaussElemUniformAngleNoise", "GaussVecNoise", "UniformAngleNoise", "DEFAULT_DECODER_KWARGS", "default_decoder", "register", "synth", "cache", "stats", "targets", "ImageEncoder", "EncoderDecoder", "VitDims",
    "SiglipImageEncoder", "SiglipDims", "SIGLIP_SO400M",
]
