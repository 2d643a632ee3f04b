"""wav2sleep_b200: B200-native (sm_100a) implementation of the wav2sleep model forward hot path.

Public surface mirrors ``wav2sleep`` (reference ``src/wav2sleep/__init__.py:3-19``) for the part that is in scope:
the model classes (``wav2sleep_b200.model``), ``load_model`` and ``predict`` (``wav2sleep_b200.api``),
``predict_on_folder`` for parquet nights (``wav2sleep_b200.folder``), and ``StreamingSession``
(``wav2sleep_b200.streaming``) for epoch-by-epoch inference of causal models, and ``integrated_gradients``
(``wav2sleep_b200.attribution``) for input attribution.
Importing the package does not load the CUDA library; the first forward does, and raises if it is missing.
"""
from .model import (  # noqa: F401
    COLS_TO_SAMPLES_PER_EPOCH,
    MultiModalAttentionEmbedder,
    SequenceCNN,
    SignalEncoder,
    SignalEncoders,
    Wav2Sleep,
    build_default,
)

__all__ = [
    "COLS_TO_SAMPLES_PER_EPOCH", "MultiModalAttentionEmbedder", "SequenceCNN", "SignalEncoder", "SignalEncoders",
    "Wav2Sleep", "build_default", "load_model", "load_dataset", "predict", "save_predictions", "predict_on_folder",
    "StreamingSession", "integrated_gradients",
]

# The reference's top-level functions (src/wav2sleep/__init__.py:3-19), resolved on first use so that importing the
# package stays light (folder.py pulls in pandas / pyarrow).  ``prepare`` (EDF / CSV ingestion) stays with the
# reference.
_LAZY = {"load_model": "api", "predict": "api", "load_dataset": "folder", "save_predictions": "folder",
         "predict_on_folder": "folder", "StreamingSession": "streaming", "integrated_gradients": "attribution"}


def __getattr__(name):
    if name in _LAZY:
        import importlib
        return getattr(importlib.import_module(f"{__name__}.{_LAZY[name]}"), name)
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")
