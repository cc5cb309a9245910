"""SAE modules and trainer (drop-in for ``whisper_sae.sae``)."""

from .crosscoder import CrossLayerCrosscoder, CrosscoderOutput, TopKCrossLayerCrosscoder, create_crosscoder
from .graphed import GraphedVariantStep, make_optimizer
from .model import ReLUSAE, SAEOutput, TopKSAE, create_sae
from .splice import SpliceEval, SpliceStats, WhisperSAESplice, evaluate_splice
from .training import SAETrainer, TrainingMetrics
from .transcoder import SkipTranscoder, TopKTranscoder, TranscoderOutput, create_transcoder

__all__ = ["ReLUSAE", "SAEOutput", "TopKSAE", "create_sae", "SAETrainer", "TrainingMetrics",
           "TopKTranscoder", "SkipTranscoder", "TranscoderOutput", "create_transcoder",
           "CrossLayerCrosscoder", "TopKCrossLayerCrosscoder", "CrosscoderOutput", "create_crosscoder",
           "GraphedVariantStep", "make_optimizer", "WhisperSAESplice", "SpliceStats", "SpliceEval",
           "evaluate_splice"]
