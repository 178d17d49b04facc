"""vit2spn — B200-native implementation of the ViT-2SPN dual-stream SSP hot path.

The directory is named ``vit-2spn_b200`` (not importable by the ``import`` statement); use
``import vit2spn`` (the alias module at the repository root) or
``importlib.import_module("vit-2spn_b200")``.
"""
from ._lib import LIB_PATH, EXPORTED, MODE_BF16, MODE_FP32  # noqa: F401  (raises if the .so is missing)
from .modules import (DualStreamNetwork, FineTunedModel, InfoNCELoss, SingleStreamNetwork, ViTBackbone, ViTConfig, ViTModel,  # noqa: F401
                      get_compute_mode, momentum, preprocess_u8_patches, set_compute_mode)
from .optim import FusedAdam  # noqa: F401
from . import augment, explain, parallel  # noqa: F401
from .train import (accumulation_steps, batch_size, epochs, learning_rate, load_checkpoint,  # noqa: F401
                    save_checkpoint, train_self_supervised)
