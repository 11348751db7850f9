"""dostransformer_b200 -- B200-native (sm_100a) implementation of the DOSTransformer training/inference hot path.

Public surface (mirrors the reference's model API, SURVEY.md section 8b):

    from dostransformer_b200.embedder_eDOS.DOSTransformer import DOSTransformer
    from dostransformer_b200.embedder_phDOS.DOSTransformer_phonon import DOSTransformer_phonon
    from dostransformer_b200.layers import TransformerEncoder
    from dostransformer_b200.ops import dos_loss
    from dostransformer_b200 import attention_maps      # records every encoder layer's attention probabilities

``install_dropin()`` registers these under the reference's import paths (``embedder_eDOS.DOSTransformer``,
``embedder_phDOS.DOSTransformer_phonon``, ``layers``) so main_eDOS.py / main_phDOS.py pick them up unchanged.
The compute path is libdost_b200.so (hand-written CUDA, C ABI in include/dost.h); there is no CPU fallback.
"""
from __future__ import annotations

import sys

from .nn_core import attention_maps

__version__ = "0.1.0"


def install_dropin() -> None:
    """Alias this package's modules to the reference's import paths."""
    import importlib
    from . import embedder_eDOS, embedder_phDOS, layers
    sys.modules["embedder_eDOS"] = embedder_eDOS
    sys.modules["embedder_phDOS"] = embedder_phDOS
    sys.modules["layers"] = layers
    sys.modules["embedder_eDOS.DOSTransformer"] = importlib.import_module(__name__ + ".embedder_eDOS.DOSTransformer")
    sys.modules["embedder_phDOS.DOSTransformer_phonon"] = importlib.import_module(
        __name__ + ".embedder_phDOS.DOSTransformer_phonon")
