"""vl-merging_b200 — B200-native merge hot path of ylsung/vl-merging (import as `vl_merging_b200`).

  gram.GramCache                     RegMean Gram caching hook   (src/cache_gram_matrices.py:236-281,349)
  gramfile                           packed fp32 Gram container <-> the reference's Gram file (:349 / vilt_module.py:386)
  merge.merge_weights / sum_task_vectors / regmean / Merger      (src/vilt/modules/vilt_module.py:366-746)
  checkpoint.modify_checkpoint_vlmo  checkpoint -> merge input (rel-pos table resize) (vilt_module.py:749-806)
  model.VLMo                         stock-torch multiway transformer the hooks hang on
  csrc/ + libvlmerge.so              sm_100a kernels behind the C ABI in include/vlmerge.h

Importing the package never touches CUDA; the first compute call loads libvlmerge.so and fails
loudly if it is missing (there is no CPU fallback).
"""
from . import _lib, checkpoint, gram, gramfile, irtr, merge, model, plan  # noqa: F401
from ._lib import VlmError, build  # noqa: F401
from .checkpoint import load_checkpoint, modify_checkpoint_vlmo, save_checkpoint  # noqa: F401
from .gram import GramCache, cache_gram_matrices  # noqa: F401
from .irtr import irtr_features, irtr_recall, irtr_recall_fused, sim_topk  # noqa: F401
from .merge import Merger, independent, merge_weights, regmean, regmean_gram_owners, sum_task_vectors  # noqa: F401
from .model import VLMo, init_synthetic_, synthetic_batch, vlmo_config  # noqa: F401

__version__ = "0.1.0"
