"""Import the REAL reference hot-path modules from /root/reference on CPU (build container only).

TEST INFRASTRUCTURE.  Nothing is copied: the reference packages are imported in place.  Three heavy
`__init__`s (`sgm`, `sgm.modules`, `sgm.models`) pull pytorch_lightning / open_clip / kornia, so they are
pre-registered as bare namespace packages; three absent third-party modules are stubbed with inert
placeholders (SURVEY.md §8(c)).  /root/reference does not exist on the GPU box; only make_golden.py uses this.
"""
from __future__ import annotations

import copy
import importlib
import sys
import types
from pathlib import Path

REF_ROOT = Path("/root/reference")


def available() -> bool:
    return (REF_ROOT / "sgm" / "modules" / "diffusionmodules" / "video_model.py").exists()


def _namespace(name: str, path: Path) -> None:
    if name in sys.modules:
        return
    m = types.ModuleType(name)
    m.__path__ = [str(path)]
    m.__package__ = name
    sys.modules[name] = m


def _stub(name: str, **attrs) -> types.ModuleType:
    if name in sys.modules:
        return sys.modules[name]
    m = types.ModuleType(name)
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m
    return m


def install() -> None:
    if not available():
        raise RuntimeError("/root/reference is not present (GPU box?); golden fixtures must be used instead")
    import torch.nn as nn

    _namespace("sgm", REF_ROOT / "sgm")
    _namespace("sgm.modules", REF_ROOT / "sgm" / "modules")
    _namespace("sgm.models", REF_ROOT / "sgm" / "models")
    _namespace("sgm.modules.encoders", REF_ROOT / "sgm" / "modules" / "encoders")
    _stub("mediapy", write_image=lambda *a, **k: None, write_video=lambda *a, **k: None)

    class _Cfg(dict):
        pass

    class _OmegaConf:
        @staticmethod
        def create(x=None):
            return x

        @staticmethod
        def to_container(x, **k):
            return x

    _stub("omegaconf", ListConfig=_Cfg, DictConfig=_Cfg, OmegaConf=_OmegaConf)

    class _LightningModule(nn.Module):
        @property
        def device(self):
            return next(self.parameters()).device

    pl = _stub("pytorch_lightning", LightningModule=_LightningModule)
    loggers = _stub("pytorch_lightning.loggers", WandbLogger=type("WandbLogger", (), {}))
    pl.loggers = loggers


def load():
    """Returns a namespace with the reference classes the path uses."""
    install()
    ns = types.SimpleNamespace()
    ns.video_model = importlib.import_module("sgm.modules.diffusionmodules.video_model")
    ns.wrappers = importlib.import_module("sgm.modules.diffusionmodules.wrappers")
    ns.denoiser = importlib.import_module("sgm.modules.diffusionmodules.denoiser")
    ns.denoiser_scaling = importlib.import_module("sgm.modules.diffusionmodules.denoiser_scaling")
    ns.sampling = importlib.import_module("sgm.modules.diffusionmodules.sampling")
    ns.guiders = importlib.import_module("sgm.modules.diffusionmodules.guiders")
    ns.discretizer = importlib.import_module("sgm.modules.diffusionmodules.discretizer")
    ns.temporal_ae = importlib.import_module("sgm.modules.autoencoding.temporal_ae")
    ns.model = importlib.import_module("sgm.modules.diffusionmodules.model")
    return ns


V3D_UNET_KW = dict(  # scripts/pub/configs/V3D_512.yaml:29-57, attention forced to "softmax" (SURVEY.md §0.8)
    adm_in_channels=768, num_classes="sequential", use_checkpoint=False, in_channels=8, out_channels=4,
    model_channels=320, attention_resolutions=[4, 2, 1], num_res_blocks=2, channel_mult=[1, 2, 4, 4],
    num_head_channels=64, use_linear_in_transformer=True, transformer_depth=1, context_dim=1024,
    spatial_transformer_attn_type="softmax", extra_ff_mix_layer=True, use_spatial_context=True,
    merge_strategy="learned_with_images", video_kernel_size=[3, 1, 1],
)

V3D_DECODER_KW = dict(  # scripts/pub/configs/V3D_512.yaml:111-132
    attn_type="vanilla", double_z=True, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=128,
    ch_mult=[1, 2, 4, 4], num_res_blocks=2, attn_resolutions=[], dropout=0.0, video_kernel_size=[3, 1, 1],
)


def engine_config_small(prefix: str, width: int = 64, dec_ch: int = 64, T: int = 4) -> dict:
    """scripts/pub/configs/V3D_512.yaml:17-146 with the `target:` prefix of the path components as a parameter
    ("sgm": the reference's classes, "v3d_b200.sgm": the drop-ins) and reduced widths (construction cost only)."""
    dm = prefix + ".modules.diffusionmodules."
    return copy.deepcopy(dict(
        scale_factor=0.18215, disable_first_stage_autocast=True, input_key="latents", log_keys=[], en_and_decode_n_samples_a_time=T,
        denoiser_config={"target": dm + "denoiser.Denoiser",
                         "params": {"scaling_config": {"target": dm + "denoiser_scaling.VScalingWithEDMcNoise"}}},
        network_config={"target": dm + "video_model.VideoUNet",
                        "params": dict(V3D_UNET_KW, model_channels=width)},
        first_stage_config={
            "target": prefix + ".models.autoencoder.AutoencodingEngine",
            "params": {
                "loss_config": {"target": "torch.nn.Identity"},
                "regularizer_config": {"target": prefix + ".modules.autoencoding.regularizers.DiagonalGaussianRegularizer"},
                "encoder_config": {"target": "torch.nn.Identity"},
                "decoder_config": {"target": prefix + ".modules.autoencoding.temporal_ae.VideoDecoder",
                                   "params": dict(V3D_DECODER_KW, ch=dec_ch)}}},
        sampler_config={"target": dm + "sampling.EulerEDMSampler",
                        "params": {"num_steps": 3,
                                   "discretization_config": {"target": dm + "discretizer.EDMDiscretization",
                                                             "params": {"sigma_max": 700.0}},
                                   "guider_config": {"target": dm + "guiders.LinearPredictionGuider",
                                                     "params": {"max_scale": 3.5, "min_scale": 3.5, "num_frames": T}}}},
    ))
