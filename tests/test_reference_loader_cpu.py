"""Checkpoint compatibility with the reference's DiffusionEngine (SURVEY.md 8(b); INTEGRATION.md section A).

tests/golden/engine_state_dict_small.json.gz holds the name, shape and dtype of every `state_dict()` entry of the
reference's `DiffusionEngine` (sgm/models/video_diffusion.py:35-105) built from the small V3D_512 config of
`oracle.reference_shim.engine_config_small` with the reference's own `target:`s (oracle/make_golden.py, which also
checks that the reference engine class builds the same table from the drop-in targets).  Checked here, on the drop-in
`v3d_b200.sgm.models.video_diffusion.DiffusionEngine` built from the drop-in `target:`s of INTEGRATION.md section A:

  * `instantiate_from_config` resolves the drop-in targets to the v3d_b200 classes;
  * its `state_dict()` has the SAME names, shapes and dtypes as the reference engine's (network, first-stage decoder,
    and nothing else: the conditioner is the unconditional stub, the denoiser / sampler hold no parameters);
  * `load_state_dict(strict=True)` of a state dict with the reference's layout, and back;
  * `init_from_ckpt` (the safetensors branch of video_diffusion.py:123-168) loads a checkpoint with the reference's
    layout with no missing / unexpected keys.

CPU only (construction and weight plumbing; no kernels run).
"""
import gzip
import json
import sys
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from oracle import reference_shim  # noqa: E402

GOLD = ROOT / "tests" / "golden" / "engine_state_dict_small.json.gz"


@pytest.fixture(scope="module")
def ref_table():
    with gzip.open(GOLD, "rt") as f:
        return {k: (tuple(shape), getattr(torch, dtype)) for k, shape, dtype in json.load(f)["state_dict"]}


@pytest.fixture(scope="module")
def drop():
    from v3d_b200.sgm.models.video_diffusion import DiffusionEngine

    torch.manual_seed(0)
    return DiffusionEngine(**reference_shim.engine_config_small("v3d_b200.sgm"))


def _ref_state_dict(ref_table):
    """A state dict with the reference engine's layout and seeded values."""
    g = torch.Generator().manual_seed(0)
    return {k: torch.randn(shape, generator=g).to(dtype) for k, (shape, dtype) in ref_table.items()}


def _hot_path_items(table):
    return {k: v for k, v in table.items()
            if k.startswith("model.diffusion_model.") or k.startswith("first_stage_model.decoder.")}


def test_reference_loader_builds_dropins_with_identical_state_dict(drop, ref_table):
    import v3d_b200.decoder
    import v3d_b200.sampling
    import v3d_b200.unet

    # instantiate_from_config constructed OUR classes
    assert isinstance(drop.model.diffusion_model, v3d_b200.unet.VideoUNet)
    assert isinstance(drop.first_stage_model.decoder, v3d_b200.decoder.VideoDecoder)
    assert isinstance(drop.sampler, v3d_b200.sampling.EulerEDMSampler)
    assert isinstance(drop.denoiser, v3d_b200.sampling.Denoiser)
    assert isinstance(drop.model, v3d_b200.sampling.OpenAIWrapper)
    mine = {k: (tuple(v.shape), v.dtype) for k, v in drop.state_dict().items()}
    a, b = _hot_path_items(ref_table), _hot_path_items(mine)
    assert len(a) > 1000 and a == b
    # nothing else differs either
    extra_ref = set(ref_table) - set(a)
    extra_drop = set(mine) - set(b)
    assert extra_ref == extra_drop, (sorted(extra_ref ^ extra_drop)[:10])


def test_strict_load_state_dict_round_trip(drop, ref_table):
    sd = _ref_state_dict(ref_table)
    missing, unexpected = drop.load_state_dict(sd, strict=True)
    assert not missing and not unexpected
    back = drop.state_dict()
    for k in ("model.diffusion_model.input_blocks.0.0.weight", "model.diffusion_model.out.2.bias",
              "first_stage_model.decoder.conv_in.weight", "first_stage_model.decoder.conv_out.time_mix_conv.weight"):
        assert torch.equal(back[k], sd[k]), k


def test_reference_init_from_ckpt_loads_into_dropins(ref_table, tmp_path):
    from safetensors.torch import save_file

    from v3d_b200.sgm.models.video_diffusion import DiffusionEngine

    want = _ref_state_dict(ref_table)
    path = str(tmp_path / "v3d_small.safetensors")
    save_file(want, path)
    eng = DiffusionEngine(ckpt_path=path, **reference_shim.engine_config_small("v3d_b200.sgm"))
    got = eng.state_dict()
    assert set(got) == set(want)
    for k, v in want.items():
        assert torch.equal(got[k], v), k
