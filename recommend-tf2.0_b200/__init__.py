"""recommend-tf2.0_b200 — B200 (sm_100a) kernels behind the recommend-tf2.0 embedding and
feature-interaction layers.  Import as `recommend_tf2_b200` (see ../recommend_tf2_b200.py).

Nothing here computes on the CPU: every op dispatches to librtf_b200.so and raises if the
library or a CUDA device is missing."""
from . import _lib
from ._lib import RtfError, build, lib
from .embedding import EmbeddingTables, SparseOptimizer, embed_bwd, embed_fwd
from .interaction import dot_interact, dot_out_cols, embed_dot
from .attention import attention
from .fm import FM, FMModel, colsum
from . import layers
from .dlrm import DLRM, DLRMTrainer
from . import models
from . import data
from . import retrieval
from . import checkpoint
from . import metrics
from .checkpoint import load_weights, save_weights
from .retrieval import IndexFlatIP, topk_ip
from .data import DeviceFeeder, criteo_feature_columns, denseFeature, sparseFeature, varLenSparseFeat

__all__ = ["RtfError", "build", "lib", "EmbeddingTables", "SparseOptimizer", "embed_fwd",
           "embed_bwd", "dot_interact", "dot_out_cols", "embed_dot", "attention", "FM", "FMModel",
           "colsum", "layers", "retrieval", "IndexFlatIP", "topk_ip", "checkpoint", "save_weights", "load_weights", "metrics", "DLRM", "DLRMTrainer", "models", "data", "DeviceFeeder",
           "criteo_feature_columns", "denseFeature", "sparseFeature", "varLenSparseFeat"]
