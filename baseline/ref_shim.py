"""Import the reference's own `RobotVisionFM` (and friends) offline -- benchmark / test infrastructure only.

The reference needs two things this image does not have (SURVEY.md section 8c): the `omegaconf` package (one use,
rvfm.py:8,65) and the HuggingFace hub (backbones.py:275,285 call `AutoModel/AutoProcessor.from_pretrained`).  This
shim registers a six-line `omegaconf` stub and replaces the three `from_pretrained` entry points with factories that
build the same objects from the hub configs of facebook/deit-{tiny,small,base}-patch16-224 (model_type "vit":
12 layers, patch 16, 224 px, gelu, qkv bias, eps 1e-12 = ViTConfig defaults; DeiT processor with the ImageNet
mean / std).  The reference code itself is imported UNMODIFIED from oracle/_ref (the pip-installed copy build()
makes, oracle/install_ref.py) or, where only the source tree exists, from that tree."""
from __future__ import annotations

import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
BACKBONES = {
    "facebook/deit-tiny-patch16-224": (192, 3),
    "facebook/deit-small-patch16-224": (384, 6),
    "facebook/deit-base-patch16-224": (768, 12),
}
IMAGE_MEAN = (0.485, 0.456, 0.406)
IMAGE_STD = (0.229, 0.224, 0.225)


def reference_path(prefer_installed: bool = True):
    inst = os.path.join(os.path.dirname(HERE), "oracle", "_ref")  # oracle/install_ref.py
    if prefer_installed and os.path.exists(os.path.join(inst, "theia", "models", "rvfm.py")):
        return inst
    if os.path.exists("/root/reference/src/theia/models/rvfm.py"):
        return "/root/reference/src"
    if os.path.exists(os.path.join(inst, "theia", "models", "rvfm.py")):
        return inst
    return None


def install_shims():
    import transformers
    from transformers import ViTConfig, ViTModel
    from transformers.models.deit.image_processing_deit import DeiTImageProcessor

    if "omegaconf" not in sys.modules:
        m = types.ModuleType("omegaconf")

        class OmegaConf:  # only use: rvfm.py:65
            to_container = staticmethod(lambda x: dict(x))

        class DictConfig(dict):
            pass

        m.OmegaConf = OmegaConf
        m.DictConfig = DictConfig
        sys.modules["omegaconf"] = m

    def _cfg(name):
        d, h = BACKBONES[name]
        return ViTConfig(hidden_size=d, num_attention_heads=h, intermediate_size=4 * d)

    transformers.AutoModel.from_pretrained = staticmethod(lambda name, *a, **k: ViTModel(_cfg(name)))
    transformers.AutoConfig.from_pretrained = staticmethod(lambda name, *a, **k: _cfg(name))
    transformers.AutoProcessor.from_pretrained = staticmethod(
        lambda name, *a, **k: DeiTImageProcessor(image_mean=list(IMAGE_MEAN), image_std=list(IMAGE_STD)))


def import_reference(prefer_installed: bool = True):
    """Returns the reference's RobotVisionFM class, or raises ImportError when no copy of the reference exists."""
    path = reference_path(prefer_installed)
    if path is None:
        raise ImportError("no reference package: oracle/_ref is missing (build() installs it where the reference's "
                          "source tree is available)")
    install_shims()
    if path not in sys.path:
        sys.path.insert(0, path)
    from theia.models.rvfm import RobotVisionFM
    return RobotVisionFM
