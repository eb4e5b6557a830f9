"""
ecg_b200 -- B200-native ECG-ViT encoder training step (drop-in for the reference's
`ecg_transformer.models.EcgVit` + the step of `MyTrainer.train`).

The directory name follows the build contract (`ecg-representation-learning_b200/`); import it as `ecg_b200`
through the shim at the repo root.
"""
from .config import EcgVitConfig
from .model import EcgVit, ModelOutput, Recorder, EcgVitForMaskedPatchModeling, MaskedPatchOutput, \
    EcgVitForMaskedAutoencoding
from .trainer import FusedTrainer, fused_train_step, get_train_args, lr_multiplier
from .optim import FusedAdamW, clip_grad_norm_, param_groups_lrd
from .transform import InputPipeline
from .metrics import get_accuracy, evaluate
from .synthetic import synthetic_batch
from . import _lib

__all__ = ['EcgVitConfig', 'EcgVit', 'ModelOutput', 'EcgVitForMaskedPatchModeling', 'EcgVitForMaskedAutoencoding',
           'MaskedPatchOutput', 'FusedTrainer', 'fused_train_step', 'FusedAdamW', 'clip_grad_norm_', 'param_groups_lrd',
           'get_train_args', 'lr_multiplier', 'InputPipeline', 'Recorder', 'get_accuracy', 'evaluate', 'synthetic_batch']
