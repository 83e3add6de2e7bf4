"""CPU tests of the host side: the C-ABI library loads and exports every symbol include/v3d_b200.h declares,
the drop-in modules expose the reference's state_dict layout, the host-only logic behaves, and the product
refuses to run without CUDA (no CPU fallback)."""
import ctypes
import re
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent


def _header_functions():
    text = (ROOT / "include" / "v3d_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(v3d_[a-z0-9_]+)\s*\(", text)) - {"v3d_gemm_args"})


def test_library_exports_every_declared_symbol():
    from v3d_b200 import _lib

    lib = _lib.load()
    names = _header_functions()
    assert len(names) >= 25
    raw = ctypes.CDLL(str(_lib.lib_path()))
    for n in names:
        assert hasattr(raw, n), f"{n} declared in include/v3d_b200.h but not exported"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes prototype"
    assert sorted(_lib.SIGNATURES) == names, "ctypes table and header disagree"
    assert lib.v3d_abi_version() == 1
    # the ctypes mirror of v3d_gemm_args: 7 pointers, 8 int64, 16 int32, 3 floats, 2 int32 (halo fields), padded to 8,
    # then the fused K|V scatter block: 2 int32, 1 int64, 8 pointers
    base = (7 * 8 + 8 * 8 + 16 * 4 + 3 * 4 + 2 * 4 + 7) // 8 * 8
    assert ctypes.sizeof(_lib.GemmArgs) == base + 2 * 4 + 8 + 8 * 8
    assert ctypes.sizeof(_lib.GemmArgs) == lib.v3d_gemm_args_size()
    assert lib.v3d_gemm_args_size() == ctypes.sizeof(_lib.GemmArgs)   # what the C side was compiled with


def test_host_only_abi_functions():
    from v3d_b200 import ops

    assert ops.pick_block_n(1280) == 256 and ops.pick_block_n(320) == 160 and ops.pick_block_n(960) == 160
    assert ops.pick_block_n(48) == 16 and ops.pick_block_n(2560, ops.ACT_GEGLU) == 256
    perm = ops.geglu_perm(256, 256)
    assert perm.tolist()[:128] == list(range(128)) and perm.tolist()[128:256] == list(range(256, 384))
    assert sorted(perm.tolist()) == list(range(512))


def test_gemm_argument_validation_without_gpu():
    from v3d_b200 import _lib

    lib = _lib.load()
    g = _lib.GemmArgs()
    assert lib.v3d_gemm_bf16(ctypes.byref(g), None) == 1  # null pointers -> BAD_ARG, no launch attempted
    assert b"null" in lib.v3d_last_error()


def test_unet_state_dict_layout_matches_reference_table():
    from oracle import ref_unet
    from v3d_b200.engine import v3d_512_config
    from v3d_b200.unet import VideoUNet

    with torch.device("meta"):
        net = VideoUNet(**v3d_512_config()["network_config"]["params"])
    want = ref_unet.unet_param_shapes(ref_unet.UNetSpec())
    got = {k: tuple(v.shape) for k, v in net.state_dict().items()}
    assert got == {k: tuple(v) for k, v in want.items()}
    assert len(got) == 1428 and sum(torch.Size(s).numel() for s in got.values()) == 1_524_623_082


def test_decoder_state_dict_layout_and_zero_modules():
    from oracle import ref_decoder
    from v3d_b200.decoder import VideoDecoder
    from v3d_b200.engine import v3d_512_config

    kw = v3d_512_config()["first_stage_config"]["params"]["decoder_config"]["params"]
    with torch.device("meta"):
        dec = VideoDecoder(**kw)
    want = ref_decoder.decoder_param_shapes(ref_decoder.DecoderSpec())
    assert {k: tuple(v.shape) for k, v in dec.state_dict().items()} == {k: tuple(v) for k, v in want.items()}
    assert sum(v.numel() for v in dec.state_dict().values()) == 63_579_183
    small = VideoDecoder(**{**kw, "ch": 64})
    zero = [k for k, v in small.state_dict().items() if v.ndim > 1 and v.abs().max() == 0]
    assert zero and all(".time_stack.out_layers.3." in k for k in zero)
    small.randomize_zero_modules_()
    assert not [k for k, v in small.state_dict().items() if v.ndim > 1 and v.abs().max() == 0]


def test_small_unet_init_zero_modules_and_plan():
    from v3d_b200.engine import v3d_512_config
    from v3d_b200.unet import VideoUNet

    kw = dict(v3d_512_config()["network_config"]["params"], model_channels=64)
    net = VideoUNet(**kw)
    zeros = [k for k, v in net.state_dict().items() if v.ndim > 1 and v.abs().max() == 0]
    assert len(zeros) == 61  # SURVEY.md §0.6: 44 out_layers.3 + 16 proj_out + out.2
    kinds = [s.kind for s in net.steps]
    assert kinds.count("res") == 22 and kinds.count("attn") == 16 and kinds.count("down") == 3
    assert kinds.count("up") == 3 and kinds.count("save") == 12 and kinds.count("cat") == 12
    net.randomize_zero_modules_(1)
    assert not [k for k, v in net.state_dict().items() if v.ndim > 1 and v.abs().max() == 0]
    # unsupported configurations fail loudly instead of silently computing something else
    with pytest.raises(NotImplementedError):
        VideoUNet(**{**kw, "use_scale_shift_norm": True})


def test_no_cpu_fallback():
    from v3d_b200 import sampling
    from v3d_b200.engine import v3d_512_config
    from v3d_b200.unet import VideoUNet

    kw = dict(v3d_512_config()["network_config"]["params"], model_channels=64)
    net = VideoUNet(**kw)
    T = 2
    with pytest.raises(RuntimeError, match="CUDA"):
        net(torch.zeros(2 * T, 8, 8, 8), torch.zeros(2 * T), torch.zeros(2 * T, 1, 1024), torch.zeros(2 * T, 768),
            None, T, torch.zeros(2, T))
    s = sampling.EulerEDMSampler(
        num_steps=2, discretization_config={"target": "v3d_b200.sampling.EDMDiscretization", "params": {}},
        guider_config={"target": "v3d_b200.sampling.LinearPredictionGuider",
                       "params": {"max_scale": 2.0, "num_frames": T}})
    with pytest.raises(RuntimeError, match="CUDA"):
        s(lambda *a: None, torch.zeros(T, 4, 8, 8), cond={}, uc={})


def test_guider_and_discretizer_host_logic():
    from v3d_b200 import sampling

    g = sampling.LinearPredictionGuider(max_scale=3.5, min_scale=1.0, num_frames=4)
    c = {"vector": torch.ones(4, 3), "crossattn": torch.ones(4, 1, 2), "concat": torch.ones(4, 2, 2, 2)}
    uc = {k: torch.zeros_like(v) for k, v in c.items()}
    x = torch.randn(4, 2, 2, 2)
    x2, s2, c2 = g.prepare_inputs(x, torch.full((4,), 7.0), c, uc)
    assert x2.shape[0] == 8 and torch.equal(x2[:4], x2[4:]) and s2.shape[0] == 8
    for k in c:
        assert c2[k][:4].abs().sum() == 0 and torch.equal(c2[k][4:], c[k])  # [uc; c]
    d = sampling.EDMDiscretization(sigma_max=700.0)
    s = d(25)
    assert s.shape[0] == 26 and s[-1] == 0 and abs(s[0].item() - 700.0) < 1e-3
    assert bool((s[1:] < s[:-1]).all())


def test_other_guiders_host_logic_bit_exact():
    """CentralPredictionGuider / VanillaCFG scale rows equal the reference's (golden schedule.pt); [uc; c] order."""
    from pathlib import Path

    from v3d_b200 import sampling

    gold = torch.load(Path(__file__).resolve().parent / "golden" / "schedule.pt")
    g = sampling.CentralPredictionGuider(max_scale=3.5, min_scale=1.0, num_frames=18)
    assert torch.equal(g.scale, gold["central_scale_18"])
    assert torch.equal(sampling.CentralPredictionGuider(max_scale=2.5, num_frames=25).scale, gold["central_scale_25"])
    v = sampling.VanillaCFG(scale=2.5)
    assert v.num_frames == 1 and v.scale_value == 2.5 and v.scale == 2.5 and isinstance(v.scale, float)
    v.scale = 4.0  # callers re-assign a python float (guiders.py:24-25)
    assert v.scale_value == 4.0
    c = {"vector": torch.ones(2, 3), "crossattn": torch.ones(2, 1, 2), "concat": torch.ones(2, 2, 2, 2)}
    uc = {k: torch.zeros_like(t) for k, t in c.items()}
    for guider in (g, v):
        x2, s2, c2 = guider.prepare_inputs(torch.randn(2, 2, 2, 2), torch.full((2,), 7.0), c, uc)
        assert x2.shape[0] == 4 and s2.shape[0] == 4
        for k in c:
            assert c2[k][:2].abs().sum() == 0 and torch.equal(c2[k][2:], c[k])
    # the second-order sampler refuses CPU tensors like the first-order one (no CPU fallback)
    smp = sampling.HeunEDMSampler(num_steps=2, discretization_config={
        "target": "v3d_b200.sgm.modules.diffusionmodules.discretizer.EDMDiscretization", "params": {"sigma_max": 700.0}})
    with pytest.raises(RuntimeError):
        smp(lambda *a: None, torch.randn(2, 4, 8, 8), cond={}, uc={})


def test_encoder_state_dict_layout_and_engine_opt_in():
    """Native Encoder: reference state_dict layout (106 tensors, configs/ae/video.yaml); the engine builds it only
    when encoder_config.target names this package's class, and its Gaussian regulariser follows distributions.py."""
    from oracle import ref_encoder
    from v3d_b200.decoder import AutoencodingEngine
    from v3d_b200.encoder import DiagonalGaussianRegularizer, Encoder

    kw = dict(attn_type="vanilla", double_z=True, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=64,
              ch_mult=[1, 2, 4, 4], num_res_blocks=2, attn_resolutions=[], dropout=0.0)
    enc = Encoder(**kw)
    want = ref_encoder.encoder_param_shapes(ref_encoder.EncoderSpec(ch=64))
    assert {k: tuple(v.shape) for k, v in enc.state_dict().items()} == {k: tuple(v) for k, v in want.items()}
    assert len(want) == 106
    with pytest.raises(NotImplementedError):
        Encoder(**dict(kw, attn_resolutions=[32]))
    dkw = dict(kw, video_kernel_size=[3, 1, 1])
    ref_target = {"target": "sgm.modules.diffusionmodules.model.Encoder", "params": kw}
    ae = AutoencodingEngine(decoder_config={"params": dkw}, encoder_config=ref_target)
    assert ae.encoder is None
    with pytest.raises(NotImplementedError):
        ae.encode(torch.zeros(1, 3, 64, 64))
    ae = AutoencodingEngine(decoder_config={"params": dkw},
                            encoder_config={"target": "v3d_b200.sgm.modules.diffusionmodules.model.Encoder", "params": kw},
                            regularizer_config={"target": "x.DiagonalGaussianRegularizer"})
    assert sum(k.startswith("encoder.") for k in ae.state_dict()) == 106
    with pytest.raises(RuntimeError):           # CUDA only, no CPU fallback
        ae.encode(torch.zeros(1, 3, 64, 64))
    mom = torch.randn(2, 8, 4, 4)
    mom[:, 4:] = mom[:, 4:] * 30.0               # exercises the logvar clamp
    noise = torch.randn(2, 4, 4, 4)
    z, _ = DiagonalGaussianRegularizer(sample=True)(mom, noise=noise)
    assert torch.equal(z, ref_encoder.gaussian_sample(mom, noise))
    z, _ = DiagonalGaussianRegularizer(sample=False)(mom)
    assert torch.equal(z, mom[:, :4])


def test_conditioning_assembly_matches_reference_golden(monkeypatch):
    """GeneralConditioner / get_batch / per-frame repeat logic vs the real reference's (c, uc) (bit-exact).  The
    sinusoidal embedding itself is a CUDA kernel; here it is swapped for the oracle's so the HOST logic (key routing,
    concat order, uc zeroing, repeats) runs on CPU."""
    from pathlib import Path

    from oracle import ref_conditioning
    from v3d_b200 import conditioning

    gold = torch.load(Path(__file__).resolve().parent / "golden" / "conditioning.pt")
    monkeypatch.setattr(conditioning.ConcatTimestepEmbedderND, "forward",
                        lambda self, x: ref_conditioning.concat_timestep_embed(x, self.outdim))
    cond = conditioning.GeneralConditioner(conditioning.V3D_512_EMB_MODELS)
    c, uc = conditioning.assemble_v3d_conditioning(cond, gold["clip_emb"], gold["latent"], 6.0, 127.0, 0.02, 18)
    for k in ("vector", "crossattn", "concat"):
        assert torch.equal(c[k], gold["c"][k]) and torch.equal(uc[k], gold["uc"][k]), k
    assert c["vector"].shape == (18, 768) and uc["crossattn"].abs().sum() == 0 and uc["concat"].abs().sum() == 0
    assert [e.ucg_rate for e in cond.embedders] == [0.2, 0.0, 0.0, 0.2, 0.0]   # restored after the call


def test_drop_in_targets_resolve():
    from v3d_b200.sampling import get_obj_from_str

    for ref_target in ["sgm.modules.diffusionmodules.video_model.VideoUNet",
                       "sgm.modules.diffusionmodules.denoiser.Denoiser",
                       "sgm.modules.diffusionmodules.denoiser_scaling.VScalingWithEDMcNoise",
                       "sgm.modules.diffusionmodules.sampling.EulerEDMSampler",
                       "sgm.modules.diffusionmodules.sampling.HeunEDMSampler",
                       "sgm.modules.diffusionmodules.guiders.VanillaCFG",
                       "sgm.modules.diffusionmodules.guiders.CentralPredictionGuider",
                       "sgm.modules.diffusionmodules.discretizer.EDMDiscretization",
                       "sgm.modules.diffusionmodules.guiders.LinearPredictionGuider",
                       "sgm.modules.diffusionmodules.wrappers.OpenAIWrapper",
                       "sgm.modules.autoencoding.temporal_ae.VideoDecoder",
                       "sgm.modules.diffusionmodules.model.Encoder",
                       "sgm.modules.encoders.modules.GeneralConditioner",
                       "sgm.modules.encoders.modules.ConcatTimestepEmbedderND",
                       "sgm.modules.encoders.modules.IdentityEncoder",
                       "sgm.modules.autoencoding.regularizers.DiagonalGaussianRegularizer",
                       "sgm.models.autoencoder.AutoencodingEngine",
                       "sgm.models.video_diffusion.DiffusionEngine"]:
        assert get_obj_from_str("v3d_b200." + ref_target) is not None


def test_engine_builds_from_config_small():
    from v3d_b200 import engine

    cfg = engine.v3d_512_config(num_frames=4, num_steps=3)
    cfg["network_config"]["params"]["model_channels"] = 64
    cfg["first_stage_config"]["params"]["decoder_config"]["params"]["ch"] = 64
    eng = engine.DiffusionEngine(**cfg)
    keys = list(eng.state_dict())
    assert any(k.startswith("model.diffusion_model.input_blocks.0.0.weight") for k in keys)
    assert any(k.startswith("first_stage_model.decoder.conv_in.weight") for k in keys)
    assert eng.sampler.num_steps == 3 and eng.sampler.guider.num_frames == 4


def test_bench_reference_arm_prints_contract_line():
    """`bench.py --impl reference` (the driver's CPU arm) on the smallest sample ladder: one JSON line with the
    contract's keys, the calibrated thread count and the raw two-size measurements."""
    import json
    import os
    import subprocess
    import sys

    root = Path(__file__).resolve().parent.parent
    env = dict(os.environ, V3D_CPU_BUDGET_S="1")
    res = subprocess.run([sys.executable, str(root / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         env=env, capture_output=True, text=True, timeout=900, cwd=root)
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["metric"] == "view-frames/sec" and line["value"] > 0
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"]
    assert set(cb["last_sample_raw_s"]) == {"unet_s", "decode_s"} and cb["thread_calibration_s"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0



def test_orbit_cameras_match_reference_golden(tmp_path):
    """SURVEY 8(f)-2: the frame <-> camera convention of the generated views against the reference's own
    get_uniform_poses (tests/golden/cameras.npz, made by oracle/make_golden_cameras.py), and the mp4 writer."""
    import numpy as np

    from v3d_b200 import wire

    gold = np.load(Path(__file__).resolve().parent / "golden" / "cameras.npz")
    names = [k for k in gold.files if not k.endswith("_args")]
    assert len(names) == 4
    for name in names:
        t, r, e, gl = gold[name + "_args"]
        mine = wire.orbit_poses(int(t), float(r), float(e), opengl=bool(gl))
        assert mine.shape == gold[name].shape and mine.dtype == np.float32
        assert np.abs(mine - gold[name]).max() <= 2e-7, name
    infos = wire.camera_infos()
    assert len(infos) == 18 and infos[0]["width"] == 512 and abs(infos[0]["FovX"] - np.deg2rad(60.0)) < 1e-12
    # frame 0 looks down the -x axis from (2, 0, 0); R T reproduce the world-to-camera transform
    c2w = wire.orbit_poses()
    assert np.allclose(c2w[0, :3, 3], [2.0, 0.0, 0.0]) and np.allclose(c2w[0, :3, 2], [-1.0, 0.0, 0.0])
    w2c = np.linalg.inv(c2w[5])
    assert np.allclose(infos[5]["R"].T, w2c[:3, :3], atol=1e-6) and np.allclose(infos[5]["T"], w2c[:3, 3], atol=1e-6)
    frames = (np.random.default_rng(0).random((4, 32, 32, 3)) * 255).astype(np.uint8)
    path = wire.write_video(str(tmp_path / "v.mp4"), frames, fps=3)
    assert Path(path).stat().st_size > 0


def test_guider_attribute_pokes_match_reference_semantics():
    """app.py:143-145 assigns guider.max_scale / min_scale after construction; like the reference
    (guiders.py:71-76 computes `scale` once in __init__) that leaves the per-frame scale untouched, while assigning
    `scale` itself is honoured."""
    from v3d_b200.sampling import LinearPredictionGuider

    g = LinearPredictionGuider(max_scale=3.5, min_scale=1.5, num_frames=6)
    before = g.scale.clone()
    g.max_scale, g.min_scale = 9.0, 9.0
    assert torch.equal(g.scale, before) and g.scale.shape == (1, 6)
    assert torch.allclose(before, torch.linspace(1.5, 3.5, 6).unsqueeze(0))
    g.scale = torch.full((1, 6), 2.0)
    assert float(g.scale.sum()) == 12.0


def test_bench_native_line_assembly():
    """bench.py's native-arm JSON line is assembled by a pure function from plain timings: contract keys, the metric
    arithmetic (whole-job frames / max-over-ranks seconds), roofline fractions and JSON-serialisability, for the
    default image-parallel run and for a one-image-over-ranks plan."""
    import argparse
    import json

    import bench

    args = argparse.Namespace(frames=18, edm_steps=25, latent=64, steps=3, warmup=3, gpus=2, min_cfg=3.5, max_cfg=3.5,
                              shard="images")
    kw = dict(world=2, secs=4.5, secs_e2e=4.6, launches=111852, clocks={"sm_mhz": 1700.0, "sm_max_mhz": 1965.0,
                                                                        "reasons": ["sw_power_cap"], "samples": 20},
              h2d_bytes=3796992, d2h_bytes=14155776, probe_ms=1500.0,
              gemm_records=[(2.0e12, 2.0), (1.0e12, 1.0)],
              families={"gemm.linear": [2.0], "gemm.conv3x3": [1.0], "layernorm": [0.5, 0.5]},
              shapes={"linear M=8 K=64 N=64": [(2.0e12, 2.0)], "conv3x3 M=8 K=64 N=64": [(1.0e12, 1.0)]},
              membound={"layernorm": [(3.0e9, 0.5), (3.0e9, 0.5)]}, decode_families={"gemm.conv3x3": [1.0]})
    line = bench.assemble_line(args, sharded=False, **kw)
    json.loads(json.dumps(line))
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline"):
        assert key in line, key
    assert line["value"] == pytest.approx(2 * 18 * 3 / 4.5) and line["e2e"]["value"] == pytest.approx(2 * 18 * 3 / 4.6)
    assert line["scaling"] == "weak" and line["n_gpus"] == 2 and line["ms_per_step"] == pytest.approx(1500.0)
    assert line["e2e"]["h2d_bytes_per_step"] == 2 * 3796992 and line["e2e"]["d2h_bytes_per_step"] == 2 * 14155776
    roof = line["roofline"]
    assert roof["achieved"] == pytest.approx(1000.0) and roof["frac"] == pytest.approx(1000.0 / roof["peak"])
    assert roof["launches_per_step"] == 2 and roof["gemm_shapes_top"][0]["shape"].startswith("linear")
    assert roof["hbm_bound_families"]["layernorm"]["achieved_gbs"] == pytest.approx(6000.0)
    assert roof["breakdown_decode_only_ms"] == {"gemm.conv3x3": {"ms": 1.0, "launches": 1}, "_sum_of_kernels_ms": 1.0}
    assert roof["model"]["reference_accounting_tflop_per_step"] == pytest.approx(25 * 45.677 + 54.771)
    assert "image-dp2" in line["config"]["parallelism"] and line["config"]["workload"].startswith("V3D_512")
    args.shard = "cfg"
    one = bench.assemble_line(args, sharded=True, **kw)
    assert one["scaling"] == "strong" and one["value"] == pytest.approx(18 * 3 / 4.5)
    assert one["e2e"]["d2h_bytes_per_step"] == 14155776 and "plan 'cfg'" in one["config"]["parallelism"]


def test_bench_dump_outputs_complete_or_seeded_sample(tmp_path):
    """bench.py --dump-outputs: arrays within the byte budget are written whole as float32; over it, every array
    becomes the same fixed sample from run to run, and the files stay within the budget."""
    import numpy as np

    import bench

    frames = np.random.default_rng(1).integers(0, 256, (3, 16, 16, 3), dtype=np.uint8)
    info = bench.dump_outputs(tmp_path / "whole", {"frames": frames})
    got = np.load(tmp_path / "whole" / "frames.npy")
    assert got.dtype == np.float32 and np.array_equal(got, frames.astype(np.float32))
    assert info == {"frames": {"shape": [3, 16, 16, 3], "dtype": "float32", "sampled_elements": None}}

    big = {"a": np.arange(40000, dtype=np.float64), "b": np.linspace(0, 1, 10000)}
    limit = 20000 * 4 + 256
    runs = [bench.dump_outputs(tmp_path / str(i), big, limit_bytes=limit) for i in range(2)]
    assert runs[0] == runs[1] and runs[0]["a"]["sampled_elements"] == 16000 and runs[0]["b"]["shape"] == [10000]
    size = 0
    for name, full in big.items():
        one, two = (np.load(tmp_path / str(i) / f"{name}.npy") for i in range(2))
        assert one.dtype == np.float32 and np.array_equal(one, two)
        assert np.isin(one, full.astype(np.float32)).all() and np.all(np.diff(one) > 0)   # sorted indices, no repeats
        size += (tmp_path / "0" / f"{name}.npy").stat().st_size
    assert size <= limit


def test_schedule_cost_accounting_matches_known_flop_budget():
    """tools/schedule_cost.py (meta-device dry run of the launch schedules): the algorithmic FLOPs it books for the
    V3D_512 UNet forward and decode agree with the reference accounting of SURVEY.md App. B minus the documented
    shortcuts (cross-attention over one token, cached positional embedding), and the sharding plans split the work."""
    import importlib.util

    root = Path(__file__).resolve().parent.parent
    spec = importlib.util.spec_from_file_location("schedule_cost", root / "tools" / "schedule_cost.py")
    sc = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(sc)
    full = sc.run(18, 64, "none", 1, 0, 25)
    tf = lambda book: sum(v[1] for v in book.values()) / 1e12          # noqa: E731
    assert 43.0 < tf(full["unet_forward"]) < 45.68                       # 45.68 TF reference accounting, minus 1.94 TF
    assert abs(tf(full["decode"]) - 54.77) < 0.5                         # decoder: nothing is skipped
    assert full["unet_forward"]["gemm.conv3x3"][0] == 48 and full["unet_forward"]["groupnorm"][0] == 61 and full["unet_forward"]["groupnorm_apply"][0] == 44  # per-frame norms: one launch; 3-D norms: the pair
    cfg = sc.run(18, 64, "cfg", 2, 0, 25)
    assert abs(tf(cfg["unet_forward"]) / tf(full["unet_forward"]) - 0.5) < 0.01
    assert cfg["comm_per_unet_forward"]["cfg_gather"] == [1, 18 * 4 * 64 * 64 * 4]
    views = sc.run(18, 64, "views", 2, 1, 25)
    assert views["comm_per_unet_forward"]["halo"][0] == 44 and views["comm_per_unet_forward"]["kv_allgather"][0] == 16


def test_reference_arm_budgets_real_shape_samples(monkeypatch, capsys):
    """bench.py --impl reference: the CPU-time budget decides how many of the K steps take a real-shape sample (network
    evaluation of one CFG video at latent 64^2 + decode of nd whole frames); the other steps repeat the calibration
    forward; the value comes from the real-shape samples only and the line keeps the contract keys and the native
    arm's `config`.  (Timings stubbed: 1.3 s calibration forward, 30 s per video, 6.5 s per decoded frame.)"""
    import argparse
    import json

    import bench
    import oracle.ref_decoder as rd
    import oracle.ref_unet as ru

    monkeypatch.setattr(torch, "set_num_threads", lambda n: None)   # the arm pins its calibrated thread count: keep this
                                                                   # session's (bit-exact tests downstream depend on it)
    monkeypatch.setattr(ru, "unet_param_shapes", lambda spec: {"a.weight": (2, 2)})
    monkeypatch.setattr(rd, "decoder_param_shapes", lambda spec: {"b.weight": (2, 2)})
    monkeypatch.setattr(bench.CpuReference, "_calibrate_threads", lambda self: (16, {16: 1.3}))
    monkeypatch.setattr(bench.CpuReference, "_unet", lambda self, L, videos=2: 1.3 if L == 8 else 30.0 * videos)
    monkeypatch.setattr(bench.CpuReference, "_dec", lambda self, L, frames=0: 6.5 * (frames or self.T))
    monkeypatch.setattr(bench.CpuReference, "BUDGET_S", 420.0)
    args = argparse.Namespace(frames=18, edm_steps=25, latent=64, steps=20, warmup=5, gpus=1, min_cfg=3.5, max_cfg=3.5,
                              shard="images")
    bench.run_reference(args)
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    cb = line["cpu_baseline"]
    assert line["impl"] == "reference" and cb["mode"] == "real-shape" and cb["kind"] == "port"
    assert cb["real_shape_samples"] == 5 and len(cb["calibration_forward_drift_s"]) == 15
    assert cb["per_sample_unet_forward_s"] == [60.0] * 5 and cb["per_sample_decode_s"] == [117.0] * 5
    assert line["value"] == pytest.approx(18 / (25 * 60.0 + 117.0)) and line["e2e"]["value"] == line["value"]
    assert line["config"] == bench.workload_config(args, "gpu")          # the same dictionary in both arms
    # the in-line cpu_baseline of the native arm: one bounded sample
    monkeypatch.setattr(bench.CpuReference, "BUDGET_S", 45.0)
    ref = bench.CpuReference(18, 25, 64, n_samples=1)
    tu, td = ref.sample()
    assert ref.mode == "real-shape" and ref.n_real == 1 and ref.nd == 2 and (tu, td) == (60.0, 6.5 * 2 * 9)
    # a budget too small for even one real-shape sample: the affine ladder, and the line says so
    monkeypatch.setattr(bench.CpuReference, "BUDGET_S", 20.0)
    ref = bench.CpuReference(18, 25, 64, n_samples=3)
    assert ref.mode == "ladder" and "did not allow the real shape" in ref.describe()
