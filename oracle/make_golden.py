"""Generate tests/golden/*.pt from the REAL reference modules and pin the oracle against them.

TEST INFRASTRUCTURE; runs only in the build container (needs /root/reference):
    python -m oracle.make_golden            # all fixtures
    python -m oracle.make_golden unet_small # one fixture

For every fixture the reference module (imported through oracle/reference_shim.py, weights from
oracle/synth.py) is run on CPU fp32, the oracle restatement is run on the same inputs, and the script fails
unless they agree to <= 2e-4 of the output scale.  Only the reference's outputs are stored.
"""
from __future__ import annotations

import gzip
import importlib
import json
import sys
import time
from pathlib import Path

import torch

from . import ref_clip, ref_conditioning, ref_decoder, ref_encoder, ref_sampling, ref_unet, reference_shim, synth

OUT = Path(__file__).resolve().parent.parent / "tests" / "golden"
PIN_TOL = 2e-4


def _pin(name: str, ref: torch.Tensor, ora: torch.Tensor) -> float:
    scale = ref.abs().max().clamp_min(1e-6)
    err = ((ref - ora).abs().max() / scale).item()
    print(f"  pin {name}: max|ref-oracle|/max|ref| = {err:.3e}")
    if not err <= PIN_TOL:
        raise SystemExit(f"oracle does not reproduce the reference on {name}: {err}")
    return err


def _unet_case(ns, tag: str, model_channels: int, T: int, hw: int, wseed: int, sigma: float, manifest: dict,
               tap_stride: int = 1, full_items=None, stride: int = 1):
    kw = dict(reference_shim.V3D_UNET_KW)
    kw["model_channels"] = model_channels
    net = ns.video_model.VideoUNet(**kw).eval()
    spec = ref_unet.UNetSpec(model_channels=model_channels)
    shapes = ref_unet.unet_param_shapes(spec)
    assert {k: tuple(v.shape) for k, v in net.state_dict().items()} == {k: tuple(v) for k, v in shapes.items()}
    sd = synth.synth_state_dict(shapes, seed=wseed)
    net.load_state_dict(sd)
    x, c, uc = synth.synth_inputs(T, hw)
    xin = torch.cat([torch.cat([x, x]), torch.cat([uc["concat"], c["concat"]])], 1)
    ctx = torch.cat([uc["crossattn"], c["crossattn"]])
    y = torch.cat([uc["vector"], c["vector"]])
    ts = torch.full((2 * T,), 0.25 * torch.log(torch.tensor(sigma)).item())
    ind = torch.zeros(2, T)
    taps_ref = {}
    hooks = []
    want = ["input_blocks.1.0", "input_blocks.1.1", "input_blocks.3.0", "middle_block.1", "output_blocks.2.1",
            "output_blocks.11.1"]
    mods = dict(net.named_modules())
    for w in want:
        hooks.append(mods[w].register_forward_hook(lambda m, i, o, w=w: taps_ref.__setitem__(w, o.detach().clone())))
    with torch.no_grad():
        t0 = time.time()
        ref = net(xin, ts, ctx, y, None, T, ind)
        t_ref = time.time() - t0
        taps_or = {}
        ora = ref_unet.unet_forward(sd, spec, xin, ts, ctx, y, T, ind, taps=taps_or)
    for h in hooks:
        h.remove()
    err = _pin(tag, ref, ora)
    for w in want:
        _pin(f"{tag}:{w}", taps_ref[w], taps_or[w])
    if full_items is None:
        blob = {"out": ref, "timesteps": ts}
    else:
        # BASELINE-size fixture (files stay below 1 MB): `full_items` complete batch items + every stride-th pixel of all
        # items, fp16 (rounding 5e-4 relative, far below the tolerance); an odd stride samples every pixel parity
        blob = {"timesteps": ts, "full_items": list(full_items), "out_full": ref[list(full_items)].half(),
                "stride": stride, "out_sub": ref[:, :, ::stride, ::stride].half()}
    for w in want:
        # keep fixtures small: frames {0 (uc half), T (c half)}, every 8th channel, fp16
        # (tap_stride > 1: also every tap_stride-th pixel -- the BASELINE-size fixture)
        blob["tap:" + w] = taps_ref[w][[0, T]][:, ::8, ::tap_stride, ::tap_stride].half()
    torch.save(blob, OUT / f"{tag}.pt")
    manifest[tag] = dict(kind="unet_forward", model_channels=model_channels, T=T, latent_hw=hw, weight_seed=wseed,
                         input_seed=23, sigma=sigma, pin_err=err, ref_cpu_seconds=round(t_ref, 2),
                         out_std=ref.std().item(), tap_stride=tap_stride,
                         full_items=list(full_items) if full_items is not None else None, stride=stride)
    return net, sd, spec


def _edm_step_case(ns, net, sd, spec, tag: str, T: int, hw: int, num_steps: int, manifest: dict):
    """BASELINE.json configs[0]: EDM step(s) through the reference sampler/denoiser/wrapper around the UNet."""
    x, c, uc = synth.synth_inputs(T, hw)
    sampler = ns.sampling.EulerEDMSampler(
        num_steps=num_steps,
        discretization_config={"target": "sgm.modules.diffusionmodules.discretizer.EDMDiscretization",
                               "params": {"sigma_max": 700.0}},
        guider_config={"target": "sgm.modules.diffusionmodules.guiders.LinearPredictionGuider",
                       "params": {"max_scale": 3.5, "min_scale": 1.5, "num_frames": T}},
        device="cpu")
    den = ns.denoiser.Denoiser({"target": "sgm.modules.diffusionmodules.denoiser_scaling.VScalingWithEDMcNoise"})
    wrapped = ns.wrappers.OpenAIWrapper(net)
    extra = {"image_only_indicator": torch.zeros(2, T), "num_video_frames": T}
    with torch.no_grad():
        ref = sampler(lambda i, s, cc: den(wrapped, i, s, cc, **extra), x.clone(), cond=c, uc=uc)
        ora = ref_sampling.euler_edm_sample(
            lambda i, s, cc: ref_sampling.denoiser(
                lambda xx, tt, cond, **kw: ref_unet.openai_wrapper(sd, spec, xx, tt, cond, **kw), i, s, cc, **extra),
            x.clone(), c, uc, num_steps, ref_sampling.guider_scale(1.5, 3.5, T), T)
    err = _pin(tag, ref, ora)
    torch.save({"out": ref}, OUT / f"{tag}.pt")
    manifest[tag] = dict(kind="edm_sample", T=T, latent_hw=hw, num_steps=num_steps, min_scale=1.5, max_scale=3.5,
                         sigma_max=700.0, pin_err=err, out_std=ref.std().item())
    return ref


def _sampler_variant_case(ns, net, sd, spec, tag: str, T: int, hw: int, num_steps: int, sampler_cls: str,
                          guider: str, manifest: dict):
    """SURVEY 8(f)-3: the other samplers / guiders on the same denoiser (Heun; VanillaCFG; CentralPredictionGuider)."""
    x, c, uc = synth.synth_inputs(T, hw)
    gparams = {"linear": ("LinearPredictionGuider", {"max_scale": 3.5, "min_scale": 1.5, "num_frames": T}),
               "central": ("CentralPredictionGuider", {"max_scale": 3.5, "min_scale": 1.5, "num_frames": T}),
               "vanilla": ("VanillaCFG", {"scale": 2.5})}[guider]
    sampler = getattr(ns.sampling, sampler_cls)(
        num_steps=num_steps,
        discretization_config={"target": "sgm.modules.diffusionmodules.discretizer.EDMDiscretization",
                               "params": {"sigma_max": 700.0}},
        guider_config={"target": "sgm.modules.diffusionmodules.guiders." + gparams[0], "params": gparams[1]},
        device="cpu")
    den = ns.denoiser.Denoiser({"target": "sgm.modules.diffusionmodules.denoiser_scaling.VScalingWithEDMcNoise"})
    wrapped = ns.wrappers.OpenAIWrapper(net)
    extra = {"image_only_indicator": torch.zeros(2, T), "num_video_frames": T}
    scale, nf = {"linear": (ref_sampling.guider_scale(1.5, 3.5, T), T),
                 "central": (ref_sampling.central_guider_scale(1.5, 3.5, T), T),
                 "vanilla": (ref_sampling.vanilla_scale(2.5), 1)}[guider]
    fn = ref_sampling.heun_edm_sample if sampler_cls == "HeunEDMSampler" else ref_sampling.euler_edm_sample
    with torch.no_grad():
        ref = sampler(lambda i, s, cc: den(wrapped, i, s, cc, **extra), x.clone(), cond=c, uc=uc)
        ora = fn(lambda i, s, cc: ref_sampling.denoiser(
            lambda xx, tt, cond, **kw: ref_unet.openai_wrapper(sd, spec, xx, tt, cond, **kw), i, s, cc, **extra),
            x.clone(), c, uc, num_steps, scale, nf)
    err = _pin(tag, ref, ora)
    torch.save({"out": ref}, OUT / f"{tag}.pt")
    manifest[tag] = dict(kind="edm_sample_variant", sampler=sampler_cls, guider=guider, T=T, latent_hw=hw,
                         num_steps=num_steps, min_scale=1.5, max_scale=3.5, vanilla_scale=2.5, sigma_max=700.0,
                         pin_err=err, out_std=ref.std().item())


def _decoder_case(ns, tag: str, ch: int, T: int, B: int, hw: int, wseed: int, manifest: dict, z=None,
                  full_frames=None, stride: int = 1, crop: int = 0):
    kw = dict(reference_shim.V3D_DECODER_KW)
    kw["ch"] = ch
    dec = ns.temporal_ae.VideoDecoder(**kw).eval()
    spec = ref_decoder.DecoderSpec(ch=ch)
    shapes = ref_decoder.decoder_param_shapes(spec)
    assert {k: tuple(v.shape) for k, v in dec.state_dict().items()} == {k: tuple(v) for k, v in shapes.items()}
    sd = synth.synth_state_dict(shapes, seed=wseed)
    dec.load_state_dict(sd)
    if z is None:
        z = synth.synth_latents(B, hw, seed=77)
    with torch.no_grad():
        t0 = time.time()
        # decode_first_stage semantics (video_diffusion.py:182-210): z / scale_factor, one chunk of T frames
        ref = dec(z / 0.18215, timesteps=T)
        t_ref = time.time() - t0
        ora = ref_decoder.decode_first_stage(sd, spec, z, n_samples_a_time=T) if B == T else \
            ref_decoder.decoder_forward(sd, spec, z / 0.18215, T)
    err = _pin(tag, ref, ora)
    if full_frames is None:
        torch.save({"out": ref, "z": z}, OUT / f"{tag}.pt")
    else:
        # BASELINE-size fixture (files stay below 1 MB): the top-left crop x crop pixels of the `full_frames` at full
        # resolution + every stride-th pixel of all frames, fp16 (the decoder output is an image in about [-1.5, 1.5]:
        # fp16 rounding 5e-4 relative, far below the tolerance).  z is regenerated from its seed
        # (synth.synth_latents); z_check, every 16th latent pixel, pins that
        torch.save({"z_check": z[:, :, ::16, ::16].clone(), "full_frames": list(full_frames),
                    "out_full": ref[list(full_frames), :, :crop, :crop].half(), "crop": crop,
                    "stride": stride, "out_sub": ref[:, :, ::stride, ::stride].half()}, OUT / f"{tag}.pt")
    manifest[tag] = dict(kind="decode", ch=ch, T=T, B=B, latent_hw=hw, weight_seed=wseed, z_seed=77, pin_err=err,
                         ref_cpu_seconds=round(t_ref, 2), out_std=ref.std().item(),
                         full_frames=list(full_frames) if full_frames is not None else None, stride=stride,
                         crop=crop or None)


def _encoder_case(ns, tag: str, ch: int, B: int, hw: int, wseed: int, manifest: dict):
    """SURVEY 8(f)-1: the first-stage ENCODE front-end (configs/ae/video.yaml encoder + DiagonalGaussianDistribution)."""
    enc = ns.model.Encoder(attn_type="vanilla", double_z=True, z_channels=4, resolution=hw, in_channels=3, out_ch=3,
                           ch=ch, ch_mult=[1, 2, 4, 4], num_res_blocks=2, attn_resolutions=[], dropout=0.0).eval()
    spec = ref_encoder.EncoderSpec(ch=ch)
    shapes = ref_encoder.encoder_param_shapes(spec)
    assert {k: tuple(v.shape) for k, v in enc.state_dict().items()} == {k: tuple(v) for k, v in shapes.items()}
    sd = synth.synth_state_dict(shapes, seed=wseed)
    enc.load_state_dict(sd)
    g = torch.Generator().manual_seed(78)
    x = torch.rand(B, 3, hw, hw, generator=g) * 2.0 - 1.0   # images are scaled to [-1, 1] (autoencoder.py:171-175)
    noise = torch.randn(B, 4, hw // 8, hw // 8, generator=g)
    dist = importlib.import_module("sgm.modules.distributions.distributions")
    with torch.no_grad():
        ref = enc(x)
        ora = ref_encoder.encoder_forward(sd, spec, x)
        post = dist.DiagonalGaussianDistribution(ref)
        ref_z = post.mean + post.std * noise          # .sample() with the normal draw made explicit
        ora_z = ref_encoder.gaussian_sample(ora, noise)
        assert torch.equal(post.mode(), ref_encoder.gaussian_mode(ref))
    err = _pin(tag, ref, ora)
    _pin(tag + ":sample", ref_z, ora_z)
    torch.save({"x": x, "noise": noise, "moments": ref, "z": ref_z}, OUT / f"{tag}.pt")
    manifest[tag] = dict(kind="encode", ch=ch, B=B, image_hw=hw, weight_seed=wseed, x_seed=78, pin_err=err,
                         out_std=ref.std().item())


def _clip_case(tag: str, spec: "ref_clip.ClipSpec", B: int, img_hw: int, wseed: int, manifest: dict):
    """SURVEY 8(f)-4: the CLIP ViT-H/14 image tower.  open_clip (the reference's dependency) is absent offline, so the
    stored output comes from an INDEPENDENT implementation of the same architecture - Hugging Face transformers'
    CLIPVisionModelWithProjection - on the per-name seeded weights; the oracle must reproduce it.  The image is
    regenerated from its seed in the tests (torch CPU generator), only a subsample of the preprocessed image is kept."""
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection

    sd = synth.synth_state_dict(ref_clip.clip_visual_param_shapes(spec), seed=wseed)
    cfg = CLIPVisionConfig(hidden_size=spec.width, intermediate_size=spec.mlp, projection_dim=spec.embed_dim,
                           num_hidden_layers=spec.layers, num_attention_heads=spec.heads, image_size=spec.image_size,
                           patch_size=spec.patch, hidden_act="gelu", layer_norm_eps=1e-5, attention_dropout=0.0)
    hf = CLIPVisionModelWithProjection(cfg).eval()
    missing, unexpected = hf.load_state_dict(ref_clip.to_hf_state_dict(sd, spec), strict=False)
    assert not missing and not unexpected, (missing, unexpected)
    g = torch.Generator().manual_seed(80)
    x = torch.rand(B, 3, img_hw, img_hw, generator=g) * 2.0 - 1.0
    pre = ref_clip.preprocess(x, spec.image_size)
    with torch.no_grad():
        ref = hf(pixel_values=pre).image_embeds
        ora = ref_clip.clip_visual_forward(sd, spec, pre)
    err = _pin(tag, ref, ora)
    torch.save({"out": ref, "pre_sub": pre[:, :, ::4, ::4].clone()}, OUT / f"{tag}.pt")
    manifest[tag] = dict(kind="clip_image_tower", B=B, image_hw=img_hw, x_seed=80, weight_seed=wseed, pin_err=err,
                         out_std=ref.std().item(), spec=dict(image_size=spec.image_size, patch=spec.patch,
                                                             width=spec.width, layers=spec.layers, heads=spec.heads,
                                                             mlp=spec.mlp, embed_dim=spec.embed_dim),
                         checker="transformers.CLIPVisionModelWithProjection (independent implementation; open_clip absent)")


def _conditioning_case(ns, tag: str, T: int, hw: int, manifest: dict):
    """SURVEY 8(f)-1: (c, uc) of scripts/pub/V3D_512.py:247-262 through the real GeneralConditioner with the embedder
    list of scripts/pub/configs/V3D_512.yaml:59-86.  get_batch (V3D_512.py:31-69) lives in a script that cannot be
    imported offline (it loads CLIP); its five assignments are restated below."""
    reference_shim._stub("kornia")
    reference_shim._stub("open_clip")
    mods = importlib.import_module("sgm.modules.encoders.modules")
    base = "sgm.modules.encoders.modules."
    emb = lambda key, target, **p: dict(input_key=key, is_trainable=False, target=base + target, params=p)  # noqa: E731
    cond = mods.GeneralConditioner([
        dict(emb("cond_frames_without_noise", "IdentityEncoder"), ucg_rate=0.2),
        emb("fps_id", "ConcatTimestepEmbedderND", outdim=256),
        emb("motion_bucket_id", "ConcatTimestepEmbedderND", outdim=256),
        dict(emb("cond_frames", "IdentityEncoder"), ucg_rate=0.2),
        emb("cond_aug", "ConcatTimestepEmbedderND", outdim=256)]).eval()
    g = torch.Generator().manual_seed(79)
    clip_emb = torch.randn(1, 1, 1024, generator=g)
    latent = torch.randn(1, 4, hw, hw, generator=g)
    fps_id, motion, aug = 6.0, 127.0, 0.02
    batch = {"fps_id": torch.tensor([fps_id]).repeat(T), "motion_bucket_id": torch.tensor([motion]).repeat(T),
             "cond_aug": torch.tensor([aug]).repeat(T), "cond_frames": latent.clone(),
             "cond_frames_without_noise": clip_emb.clone(), "num_video_frames": T}
    batch_uc = {k: v.clone() for k, v in batch.items() if isinstance(v, torch.Tensor)}
    with torch.no_grad():
        c, uc = cond.get_unconditional_conditioning(
            batch, batch_uc=batch_uc, force_uc_zero_embeddings=["cond_frames", "cond_frames_without_noise"])
    for d in (c, uc):
        for k in ("crossattn", "concat"):
            d[k] = d[k].unsqueeze(1).expand(d[k].shape[0], T, *d[k].shape[1:]).reshape(-1, *d[k].shape[1:]).clone()
    oc, ouc = ref_conditioning.v3d_conditioning(clip_emb, latent, fps_id, motion, aug, T)
    for k in ("vector", "crossattn", "concat"):
        assert torch.equal(c[k], oc[k]) and torch.equal(uc[k], ouc[k]), k
    print(f"  pin {tag}: vector / crossattn / concat bit-exact")
    torch.save({"clip_emb": clip_emb, "latent": latent, "c": c, "uc": uc}, OUT / f"{tag}.pt")
    manifest[tag] = dict(kind="conditioning", T=T, latent_hw=hw, fps_id=fps_id, motion_bucket_id=motion, cond_aug=aug)


def _engine_state_dict_case(tag: str, manifest: dict):
    """The reference's DiffusionEngine (video_diffusion.py:35-105) built from the small V3D_512 config with its own
    `target:`s: the name, shape and dtype of every state_dict entry (what a checkpoint of the reference carries).  The
    same engine class built from the drop-in targets must produce the same table."""
    reference_shim._stub("kornia")
    reference_shim._stub("open_clip")
    mods = sys.modules["sgm.modules"]
    enc = importlib.import_module("sgm.modules.encoders.modules")
    # what sgm/modules/__init__.py:1-6 defines (the package __init__ itself is bypassed by the shim: it pulls CLIP)
    mods.GeneralConditioner = enc.GeneralConditioner
    mods.UNCONDITIONAL_CONFIG = {"target": "sgm.modules.GeneralConditioner", "params": {"emb_models": []}}
    engine_cls = importlib.import_module("sgm.models.video_diffusion").DiffusionEngine
    table = lambda sd: [[k, list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in sd.items()]  # noqa: E731
    ref = table(engine_cls(**reference_shim.engine_config_small("sgm")).state_dict())
    drop = table(engine_cls(**reference_shim.engine_config_small("v3d_b200.sgm")).state_dict())
    if sorted(ref) != sorted(drop):
        raise SystemExit(f"{tag}: the reference engine builds different state_dicts from the drop-in targets")
    with gzip.GzipFile(OUT / f"{tag}.json.gz", "wb", mtime=0) as f:
        f.write(json.dumps({"state_dict": ref}).encode())
    manifest[tag] = dict(kind="engine_state_dict", entries=len(ref), config="oracle.reference_shim.engine_config_small")
    print(f"  {tag}: {len(ref)} state_dict entries, drop-in targets identical")


def main(argv):
    OUT.mkdir(parents=True, exist_ok=True)
    ns = reference_shim.load()
    torch.set_num_threads(8)
    mpath = OUT / "MANIFEST.json"
    manifest = json.loads(mpath.read_text()) if mpath.exists() else {}
    only = set(argv)

    def want(tag):
        return not only or tag in only

    variants = {"edm_small_heun": ("HeunEDMSampler", "linear"), "edm_small_central": ("EulerEDMSampler", "central"),
                "edm_small_vanilla": ("EulerEDMSampler", "vanilla")}
    if want("unet_small") or want("edm_small") or any(want(v) for v in variants):
        net, sd, spec = _unet_case(ns, "unet_small", 64, T=4, hw=32, wseed=1, sigma=3.0, manifest=manifest)
        if want("edm_small"):
            _edm_step_case(ns, net, sd, spec, "edm_small", T=4, hw=32, num_steps=3, manifest=manifest)
        for vtag, (scls, gd) in variants.items():
            if want(vtag):
                _sampler_variant_case(ns, net, sd, spec, vtag, T=4, hw=32, num_steps=3, sampler_cls=scls, guider=gd,
                                      manifest=manifest)
    if want("unet_small_t18"):
        _unet_case(ns, "unet_small_t18", 64, T=18, hw=16, wseed=2, sigma=40.0, manifest=manifest)
    if want("unet_full") or want("edm_full_step"):
        # BASELINE.json configs[0]: full-width VideoUNet, latent 4x32x32, T=4, 1 EDM step, fp32 CPU
        net, sd, spec = _unet_case(ns, "unet_full", 320, T=4, hw=32, wseed=3, sigma=3.0, manifest=manifest)
        _edm_step_case(ns, net, sd, spec, "edm_full_step", T=4, hw=32, num_steps=1, manifest=manifest)
    if want("unet_v3d512"):
        # BASELINE.json configs[1] network evaluation: full width, T=18, latent 64x64, CFG batch 36 (one forward)
        _unet_case(ns, "unet_v3d512", 320, T=18, hw=64, wseed=3, sigma=3.0, manifest=manifest, tap_stride=4,
                   full_items=(0, 18 + 11), stride=3)
    if want("edm_v3d512_25step"):
        # 25 accumulating Euler-EDM steps (CFG, T=18) on the full-width network at the smallest latent that
        # exercises every level (16x16 -> 2x2 at the bottom)
        net, sd, spec = _unet_case(ns, "unet_full_t18_16", 320, T=18, hw=16, wseed=3, sigma=3.0, manifest=manifest)
        _edm_step_case(ns, net, sd, spec, "edm_v3d512_25step", T=18, hw=16, num_steps=25, manifest=manifest)
    if want("decoder_v3d512"):
        # BASELINE.json configs[1] decode: 18 frames, latent 64x64 -> 512x512, one chunk
        _decoder_case(ns, "decoder_v3d512", 128, T=18, B=18, hw=64, wseed=6, manifest=manifest,
                      full_frames=(0, 11), stride=8, crop=160)
    if want("decoder_small"):
        _decoder_case(ns, "decoder_small", 64, T=3, B=3, hw=16, wseed=4, manifest=manifest)
    if want("decoder_small_2videos"):
        _decoder_case(ns, "decoder_small_2videos", 64, T=2, B=4, hw=8, wseed=5, manifest=manifest)
    if want("decoder_full"):
        _decoder_case(ns, "decoder_full", 128, T=2, B=2, hw=16, wseed=6, manifest=manifest)
    if want("encoder_small"):
        _encoder_case(ns, "encoder_small", 64, B=2, hw=64, wseed=7, manifest=manifest)
    if want("encoder_full"):
        _encoder_case(ns, "encoder_full", 128, B=1, hw=128, wseed=8, manifest=manifest)
    if want("clip_small"):
        _clip_case("clip_small", ref_clip.ClipSpec(image_size=56, patch=14, width=320, layers=2, heads=4, mlp=1280,
                                                   embed_dim=64), B=2, img_hw=96, wseed=21, manifest=manifest)
    if want("clip_vit_h14"):
        _clip_case("clip_vit_h14", ref_clip.ClipSpec(), B=1, img_hw=512, wseed=22, manifest=manifest)
    if want("conditioning"):
        _conditioning_case(ns, "conditioning", T=18, hw=8, manifest=manifest)
    if want("engine_state_dict_small"):
        _engine_state_dict_case("engine_state_dict_small", manifest)
    # integer / index paths: sigma schedule and guider scale, bit-exact
    if want("schedule"):
        disc = ns.discretizer.EDMDiscretization(sigma_max=700.0)
        blob = {f"sigmas_{n}": disc(n) for n in (1, 10, 25, 50)}
        blob["guider_scale_18"] = ns.guiders.LinearPredictionGuider(max_scale=3.5, min_scale=1.0, num_frames=18).scale
        blob["central_scale_18"] = ns.guiders.CentralPredictionGuider(max_scale=3.5, min_scale=1.0, num_frames=18).scale
        blob["central_scale_25"] = ns.guiders.CentralPredictionGuider(max_scale=2.5, min_scale=1.0, num_frames=25).scale
        assert torch.equal(blob["central_scale_18"], ref_sampling.central_guider_scale(1.0, 3.5, 18))
        assert torch.equal(blob["central_scale_25"], ref_sampling.central_guider_scale(1.0, 2.5, 25))
        for n in (1, 10, 25, 50):
            assert torch.equal(blob[f"sigmas_{n}"], ref_sampling.edm_sigmas(n))
        assert torch.equal(blob["guider_scale_18"], ref_sampling.guider_scale(1.0, 3.5, 18))
        torch.save(blob, OUT / "schedule.pt")
        manifest["schedule"] = dict(kind="schedule", note="EDMDiscretization(sigma_max=700)(n) incl. appended 0")
    mpath.write_text(json.dumps(manifest, indent=1, sort_keys=True))
    print("wrote", sorted(p.name for p in OUT.glob("*")))


if __name__ == "__main__":
    main(sys.argv[1:])
