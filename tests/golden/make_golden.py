"""Generates the golden fixtures in this directory by running the VERBATIM reference files
(/root/reference/models/unet_3d_condition_mask.py, unet_3d_blocks.py, pipeline.py) on top of the diffusers shim
(oracle/shim, parity unpinned: see its header).  Run in the build container only (the GPU box has no /root/reference):

    python tests/golden/make_golden.py

Weights are not stored: `oracle.composition.fill_deterministic` regenerates them from the state_dict keys.
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle", "shim"))
sys.path.insert(0, "/root/reference")

from oracle.composition import fill_deterministic  # noqa: E402

TINY = dict(sample_size=16, block_out_channels=(32, 64, 64, 64), attention_head_dim=8, cross_attention_dim=32,
            motion_mask=True, motion_strength=True)
TINY_VAE = dict(block_out_channels=(32, 32, 64, 64), layers_per_block=1, norm_num_groups=32, sample_size=64)


def tiny_inputs(seed=1, b=2, f=4, hw=16, lk=7, cdim=32):
    g = torch.Generator().manual_seed(seed)
    return dict(
        sample=torch.randn(b, 4, f, hw, hw, generator=g),
        cond=torch.randn(b, 4, 1, hw, hw, generator=g),
        ehs=torch.randn(b, lk, cdim, generator=g),
        mask=(torch.rand(1, 1, 1, hw, hw, generator=g) > 0.5).float(),
        timestep=500,
        motion=torch.tensor([4.0]),
    )


def main():
    import diffusers  # the shim
    from models.unet_3d_condition_mask import UNet3DConditionModel            # verbatim reference
    from models.pipeline import LatentToVideoPipeline                         # verbatim reference
    torch.manual_seed(0)
    ref = UNet3DConditionModel(**TINY).eval()
    fill_deterministic(ref, seed=0)
    inp = tiny_inputs()
    with torch.no_grad():
        out = ref(inp["sample"], inp["timestep"], inp["ehs"], condition_latent=inp["cond"], mask=inp["mask"],
                  motion=inp["motion"]).sample
        out_nomask = ref(inp["sample"], 37, inp["ehs"], condition_latent=inp["cond"], mask=None, motion=None).sample
        out_1f = ref(inp["sample"][:, :, :0], 999, inp["ehs"], condition_latent=inp["cond"], mask=inp["mask"],
                     motion=inp["motion"]).sample if False else None
    torch.save({"config": TINY, "out": out, "out_nomask_t37": out_nomask, "keys": sorted(ref.state_dict().keys())},
               os.path.join(HERE, "unet_tiny_ref.pt"))
    print("unet golden:", out.shape, float(out.abs().mean()))

    # full pipeline: tiny UNet + tiny VAE, DDIM 3 steps, CFG 9, via the verbatim LatentToVideoPipeline.__call__
    vae = diffusers.AutoencoderKL(**TINY_VAE).eval()
    fill_deterministic(vae, seed=1)
    sched = diffusers.DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                                    clip_sample=False, set_alpha_to_one=False, steps_offset=1)
    pipe = LatentToVideoPipeline(vae=vae, text_encoder=None, tokenizer=None, unet=ref, scheduler=sched)
    g = torch.Generator().manual_seed(5)
    lat = torch.randn(1, 4, 4, 16, 16, generator=g)
    cond = torch.randn(1, 4, 1, 16, 16, generator=g)
    pe = torch.randn(1, 7, 32, generator=g)
    ne = torch.randn(1, 7, 32, generator=g)
    mask = torch.ones(1, 1, 1, 16, 16)
    video, latents = pipe(prompt_embeds=pe, negative_prompt_embeds=ne, latents=lat, condition_latent=cond, mask=mask,
                          motion=[4], guidance_scale=9.0, num_inference_steps=3, output_type="pt", return_dict=False)
    # same loop with DPM-Solver++ (what train.py:806 installs)
    dpm = diffusers.DPMSolverMultistepScheduler.from_config(sched.config)
    pipe.scheduler = dpm
    video_dpm, latents_dpm = pipe(prompt_embeds=pe, negative_prompt_embeds=ne, latents=lat, condition_latent=cond,
                                  mask=mask, motion=[4], guidance_scale=9.0, num_inference_steps=4, output_type="pt",
                                  return_dict=False)
    torch.save({"vae_config": TINY_VAE, "latents_in": lat, "cond": cond, "pe": pe, "ne": ne, "video": video.half(),
                "latents": latents, "latents_dpm": latents_dpm,
                "vae_keys": sorted(vae.state_dict().keys())}, os.path.join(HERE, "pipeline_tiny_ref.pt"))
    print("pipeline golden:", video.shape, latents.shape, float(latents.abs().mean()), float(latents_dpm.abs().mean()))

    common_golden(diffusers)
    product_shape_goldens()
    oddsize_unet_golden()
    svd_goldens()
    svd_text_goldens()
    transparent_goldens()
    forward_branches_golden()


SMALL = dict(sample_size=16, block_out_channels=(64, 128, 256, 256), attention_head_dim=64, cross_attention_dim=128,
             motion_mask=True, motion_strength=True)


def fp16_inputs(b, f, hw, lk, cdim, seed=1):
    """Same draw as tests/test_gpu_unet.py::_inputs, rounded to fp16 so that the 16-bit product sees identical values."""
    g = torch.Generator().manual_seed(seed)
    d = dict(sample=torch.randn(b, 4, f, hw, hw, generator=g), cond=torch.randn(b, 4, 1, hw, hw, generator=g),
             ehs=torch.randn(b, lk, cdim, generator=g), mask=(torch.rand(1, 1, 1, hw, hw, generator=g) > 0.5).float())
    return {k: v.half().float() for k, v in d.items()}


def product_shape_goldens():
    """Verbatim reference UNet3DConditionModel at shapes the sm_100a product accepts (head_dim 64): the SMALL config of
    the GPU tests and BASELINE config 1 on the full-size architecture.  Weights: fill_deterministic(seed 0) rounded to
    fp16 (what tests/test_gpu_unet.py::_models loads into both sides); fp32 math."""
    from models.unet_3d_condition_mask import UNet3DConditionModel            # verbatim reference
    for name, cfg, shape in (("unet_small_ref.pt", SMALL, dict(b=2, f=4, hw=16, lk=77, cdim=128)),
                             ("unet_config1_ref.pt", dict(sample_size=32, motion_mask=True, motion_strength=True),
                              dict(b=1, f=8, hw=32, lk=77, cdim=1024))):
        torch.manual_seed(0)
        ref = UNet3DConditionModel(**cfg).eval()
        fill_deterministic(ref, seed=0)
        ref.load_state_dict({k: v.half().float() for k, v in ref.state_dict().items()})
        inp = fp16_inputs(**shape)
        with torch.no_grad():
            out = ref(inp["sample"], 500, inp["ehs"], condition_latent=inp["cond"], mask=inp["mask"],
                      motion=torch.tensor([4.0])).sample
        torch.save({"config": cfg, "shape": shape, "timestep": 500, "motion": 4.0, "out": out,
                    "n_keys": len(ref.state_dict())}, os.path.join(HERE, name))
        print(name, tuple(out.shape), float(out.abs().mean()))
        del ref


def common_golden(diffusers):
    """utils/common.py (verbatim) DDPM_forward_timesteps / tensor_to_vae_latent on the shim scheduler / VAE.
    `imageio` is not installed here and is only used by the reference's video writers: stubbed for the import."""
    import types
    sys.modules.setdefault("imageio", types.ModuleType("imageio"))
    from utils.common import DDPM_forward_timesteps, tensor_to_vae_latent      # verbatim reference
    sched = diffusers.DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                                    clip_sample=False, set_alpha_to_one=False, steps_offset=1)
    sched.set_timesteps(10)
    g = torch.Generator().manual_seed(11)
    x0 = torch.randn(2, 4, 1, 8, 8, generator=g)
    out = {}
    for name, dt in (("f32", torch.float32), ("bf16", torch.bfloat16), ("f16", torch.float16)):
        torch.manual_seed(3)
        xt, ts = DDPM_forward_timesteps(x0.to(dt), 4, 5, sched)
        out[f"xt_{name}"] = xt
        out["timesteps"] = ts
    vae = diffusers.AutoencoderKL(**TINY_VAE).eval()
    fill_deterministic(vae, seed=1)
    frames = torch.randn(1, 2, 3, 32, 32, generator=g).clamp(-1, 1)
    with torch.no_grad():
        lat = tensor_to_vae_latent(frames, vae)
    # DDPM_forward_mask (:50-63) and DDPM_forward (:22-30): host logic around the same add_noise
    from utils.common import DDPM_forward, DDPM_forward_mask
    import numpy as np
    rng = np.random.default_rng(5)
    np_mask = (rng.random((64, 64)) > 0.5).astype(np.uint8) * 255
    for name, dt in (("f32", torch.float32), ("bf16", torch.bfloat16)):
        torch.manual_seed(4)
        xm, tsm = DDPM_forward_mask(x0.to(dt), 4, 5, sched, np_mask)
        out[f"xmask_{name}"] = xm
        torch.manual_seed(6)
        xf, _ = DDPM_forward(x0.to(dt), 4, 5, sched)
        out[f"xfwd_{name}"] = xf
    out["np_mask"] = torch.from_numpy(np_mask)
    out.update(x0=x0, frames=frames, latents=lat)
    torch.save(out, os.path.join(HERE, "common_ref.pt"))
    print("common golden:", out["xt_f32"].shape, lat.shape, float(lat.abs().mean()))




# ------------------------------------------------------------------------------------------------ benchmarked shapes
def bf16_inputs(b, f, hw, lk, cdim, seed=1):
    """Same draw as tests/test_gpu_unet.py::_inputs, rounded to bf16 (the benchmark dtype)."""
    g = torch.Generator().manual_seed(seed)
    d = dict(sample=torch.randn(b, 4, f, hw, hw, generator=g), cond=torch.randn(b, 4, 1, hw, hw, generator=g),
             ehs=torch.randn(b, lk, cdim, generator=g), mask=(torch.rand(1, 1, 1, hw, hw, generator=g) > 0.5).float())
    return {k: v.bfloat16().float() for k, v in d.items()}


def config2_unet_golden():
    """ONE forward of the verbatim reference UNet3DConditionModel at the BENCHMARKED configuration (BASELINE config 2:
    CFG batch 2, 16 frames + condition frame, 64x64 latents, text [2,77,1024], mask, motion 4): fp32 math on
    bf16-rounded weights and inputs.  ~44 TFLOP on the CPU (minutes)."""
    import time
    from models.unet_3d_condition_mask import UNet3DConditionModel            # verbatim reference
    cfg = dict(sample_size=64, motion_mask=True, motion_strength=True)
    shape = dict(b=2, f=16, hw=64, lk=77, cdim=1024)
    torch.manual_seed(0)
    ref = UNet3DConditionModel(**cfg).eval()
    fill_deterministic(ref, seed=0)
    ref.load_state_dict({k: v.bfloat16().float() for k, v in ref.state_dict().items()})
    inp = bf16_inputs(**shape)
    t0 = time.time()
    with torch.no_grad():
        out = ref(inp["sample"], 500, inp["ehs"], condition_latent=inp["cond"], mask=inp["mask"],
                  motion=torch.tensor([4.0])).sample
    torch.save({"config": cfg, "shape": shape, "timestep": 500, "motion": 4.0, "dtype": "bf16", "out": out,
                "n_keys": len(ref.state_dict())}, os.path.join(HERE, "unet_config2_ref.pt"))
    print(f"unet_config2_ref.pt {tuple(out.shape)} |mean|={float(out.abs().mean()):.4f} ({time.time() - t0:.0f} s)")


def vae_fullsize_golden():
    """Full-size SD VAE (block_out_channels 128/256/512/512) through the VERBATIM reference entry points:
    `tensor_to_vae_latent` (utils/common.py:12-20) on one 512x512 frame and `LatentToVideoPipeline.decode_latents`
    (inherited, called at models/pipeline.py:200) on two 64x64 latent frames.  fp32 math, bf16-rounded weights/inputs."""
    import time
    import types
    import diffusers
    sys.modules.setdefault("imageio", types.ModuleType("imageio"))
    from models.pipeline import LatentToVideoPipeline                         # verbatim reference
    from utils.common import tensor_to_vae_latent                             # verbatim reference
    vae = diffusers.AutoencoderKL().eval()                                    # SD VAE defaults
    fill_deterministic(vae, seed=1)
    vae.load_state_dict({k: v.bfloat16().float() for k, v in vae.state_dict().items()})
    g = torch.Generator().manual_seed(21)
    frames = torch.randn(1, 1, 3, 512, 512, generator=g).clamp(-1, 1).bfloat16().float()
    lat = torch.randn(1, 4, 2, 64, 64, generator=g).bfloat16().float()
    pipe = LatentToVideoPipeline(vae=vae, text_encoder=None, tokenizer=None, unet=None, scheduler=None)
    t0 = time.time()
    with torch.no_grad():
        enc = tensor_to_vae_latent(frames, vae)                               # [1, 4, 1, 64, 64]
        video = pipe.decode_latents(lat)                                      # [1, 3, 2, 512, 512] fp32
    torch.save({"seed": 21, "enc_latents": enc, "video_f16": video.half(), "video_abs_mean": float(video.abs().mean()),
                "video_sum": float(video.double().sum()), "n_keys": len(vae.state_dict())},
               os.path.join(HERE, "vae_fullsize_ref.pt"))
    print(f"vae_fullsize_ref.pt enc {tuple(enc.shape)} |mean|={float(enc.abs().mean()):.4f} video {tuple(video.shape)} "
          f"|mean|={float(video.abs().mean()):.4f} ({time.time() - t0:.0f} s)")


def oddsize_unet_golden():
    """Verbatim reference UNet at a latent size that is NOT a multiple of 8 (15 x 17: what train.py:738-742 produces for
    most prompt images): exercises `forward_upsample_size` (models/unet_3d_condition_mask.py:377-383,486-491) and the odd
    stride-2 convolutions.  SMALL config, fp16-rounded weights and inputs, fp32 math; `out_f64` is the same forward in
    float64, which a different CPU's convolution kernels reproduce far below the fp32 rounding of `out`."""
    from models.unet_3d_condition_mask import UNet3DConditionModel            # verbatim reference
    torch.manual_seed(0)
    ref = UNet3DConditionModel(**SMALL).eval()
    fill_deterministic(ref, seed=0)
    ref.load_state_dict({k: v.half().float() for k, v in ref.state_dict().items()})
    g = torch.Generator().manual_seed(2)
    inp = dict(sample=torch.randn(1, 4, 3, 15, 17, generator=g), cond=torch.randn(1, 4, 1, 15, 17, generator=g),
               ehs=torch.randn(1, 77, 128, generator=g), mask=(torch.rand(1, 1, 1, 15, 17, generator=g) > 0.5).float())
    inp = {k: v.half().float() for k, v in inp.items()}
    with torch.no_grad():
        out = ref(inp["sample"], 321, inp["ehs"], condition_latent=inp["cond"], mask=inp["mask"],
                  motion=torch.tensor([5.0])).sample
        i64 = {k: v.double() for k, v in inp.items()}
        out_f64 = ref.double()(i64["sample"], 321, i64["ehs"], condition_latent=i64["cond"], mask=i64["mask"],
                               motion=torch.tensor([5.0], dtype=torch.float64)).sample
    torch.save({"config": SMALL, "inputs": {k: v.half() for k, v in inp.items()}, "timestep": 321, "motion": 5.0,
                "out": out, "out_f64": out_f64}, os.path.join(HERE, "unet_small_oddsize_ref.pt"))
    print("unet_small_oddsize_ref.pt", tuple(out.shape), float(out.abs().mean()))


SVD_TINY = dict(in_channels=9, block_out_channels=(64, 128, 128, 128), num_attention_heads=(1, 2, 2, 2),
                cross_attention_dim=64, addition_time_embed_dim=32, projection_class_embeddings_input_dim=96, num_frames=5,
                sample_size=8)
SVD_TINY_VAE = dict(block_out_channels=(32, 32, 64, 64), layers_per_block=1)


class SvdImageEncoderStub(torch.nn.Module):
    """Stand-in for the CLIP vision tower of the SVD pipeline (outside the hot path): mean colour -> Linear(3, D)."""

    def __init__(self, dim=64):
        super().__init__()
        self.p = torch.nn.Linear(3, dim)

    def forward(self, x):
        return self.p(x.mean(dim=(2, 3)))


def svd_goldens():
    """config 4 (SVD path): the VERBATIM `MaskStableVideoDiffusionPipeline.__call__` (models/pipeline.py:223-466) on tiny
    random-init models over the SVD shim (oracle/shim/diffusers/_svd.py: leaf level restated from memory, unpinned), plus
    one UNetSpatioTemporalConditionModel forward at a head-dim-64 small config for the sm_100a parity test."""
    import diffusers
    from models.pipeline import MaskStableVideoDiffusionPipeline                 # verbatim reference
    from oracle.composition import SVD_SCHED
    unet = fill_deterministic(diffusers.UNetSpatioTemporalConditionModel(**SVD_TINY).eval(), 0)
    vae = fill_deterministic(diffusers.AutoencoderKLTemporalDecoder(**SVD_TINY_VAE).eval(), 1)
    enc = fill_deterministic(SvdImageEncoderStub().eval(), 2)
    sched = diffusers.EulerDiscreteScheduler(**SVD_SCHED)
    pipe = MaskStableVideoDiffusionPipeline(vae=vae, image_encoder=enc, unet=unet, scheduler=sched)
    g = torch.Generator().manual_seed(0)
    img = torch.randn(1, 3, 64, 128, generator=g).clamp(-1, 1)
    mask = (torch.rand(1, 8, 16, generator=g) > 0.5).float()
    lat0 = torch.randn(1, 5, 4, 8, 16, generator=g)
    kw = dict(height=64, width=128, num_frames=5, num_inference_steps=3, decode_chunk_size=3, noise_aug_strength=0.0,
              latents=lat0, mask=mask, return_dict=False)
    frames = pipe(img, output_type="pt", **kw)
    lat = pipe(img, output_type="latent", **kw)
    torch.save({"unet_config": SVD_TINY, "vae_config": SVD_TINY_VAE, "image": img, "mask": mask, "latents_in": lat0,
                "frames": torch.stack(frames), "latents": lat, "timesteps": sched.timesteps.clone(),
                "sigmas": sched.sigmas.clone(), "n_unet_keys": len(unet.state_dict())},
               os.path.join(HERE, "svd_pipeline_tiny_ref.pt"))
    print("svd_pipeline_tiny_ref.pt", tuple(frames[0].shape), tuple(lat.shape), float(lat.abs().mean()))


def svd_text_goldens():
    """The VERBATIM `TextStableVideoDiffusionPipeline.__call__` (models/pipeline.py:468-731) on the tiny SVD models, called the way
    app_svd.py:120-133 calls it (condition_type="image", caller-supplied per-frame `condition_latent`, per-frame mask), plus the
    branch that encodes the image itself; and the error the pinned diffusers 0.24 raises for a multi-token (text) context."""
    import diffusers
    from models.pipeline import TextStableVideoDiffusionPipeline                 # verbatim reference
    from oracle.composition import SVD_SCHED
    unet = fill_deterministic(diffusers.UNetSpatioTemporalConditionModel(**SVD_TINY).eval(), 0)
    vae = fill_deterministic(diffusers.AutoencoderKLTemporalDecoder(**SVD_TINY_VAE).eval(), 1)
    enc = fill_deterministic(SvdImageEncoderStub().eval(), 2)
    sched = diffusers.EulerDiscreteScheduler(**SVD_SCHED)
    pipe = TextStableVideoDiffusionPipeline(vae=vae, image_encoder=enc, unet=unet, scheduler=sched)
    g = torch.Generator().manual_seed(3)
    img = torch.randn(1, 3, 64, 128, generator=g).clamp(-1, 1)
    mask = (torch.rand(1, 5, 1, 8, 16, generator=g) > 0.5).float()
    mask[:, 0] = 0                                                               # app_svd.py:111
    lat0 = torch.randn(1, 5, 4, 8, 16, generator=g)
    pe = torch.randn(1, 7, 64, generator=g)
    ne = torch.randn(1, 7, 64, generator=g)
    cl = torch.randn(1, 5, 4, 8, 16, generator=g)
    kw = dict(height=64, width=128, num_frames=5, num_inference_steps=3, decode_chunk_size=3, noise_aug_strength=0.0,
              latents=lat0, mask=mask, return_dict=False, output_type="latent")
    out = {"unet_config": SVD_TINY, "vae_config": SVD_TINY_VAE, "image": img, "mask": mask, "latents_in": lat0,
           "prompt_embeds": pe, "negative_prompt_embeds": ne, "condition_latent": cl}
    out["latents_image_condlat"] = pipe(img, condition_type="image", condition_latent=cl, **kw)
    out["latents_image"] = pipe(img, condition_type="image", **kw)
    kwf = dict(kw, output_type="pt")
    out["frames_image_condlat"] = torch.stack(pipe(img, condition_type="image", condition_latent=cl, **kwf))
    try:
        pipe(img, condition_type="text", prompt_embeds=pe, negative_prompt_embeds=ne, **kw)
        out["text_error"] = None
    except RuntimeError as e:
        out["text_error"] = str(e)
    torch.save(out, os.path.join(HERE, "svd_text_pipeline_tiny_ref.pt"))
    for k in ("latents_image_condlat", "latents_image", "frames_image_condlat"):
        print("svd_text_pipeline_tiny_ref.pt", k, tuple(out[k].shape), float(out[k].abs().mean()))
    print("text context ->", out["text_error"])


def transparent_goldens():
    """Row f4, the transparent-video branch, from the VERBATIM reference files: `models/layerdiffuse_VAE.py` (`UNet384`,
    `LatentTransparencyOffsetEncoder`) and `models/pipeline_stage2.py` `MaskedLatentToVideoPipeline.__call__`, called unbound on a
    `TextToVideoSDPipeline` object the way train_transparent_i2v_stage2.py:500-515 does (single-frame condition latent and mask,
    `return_dict=False`).  The reference passes `image_embeds=` to the UNet (:282), which `models/unet_3d_condition_mask.py` does
    not accept: the fixture UNet is the verbatim class with that one keyword swallowed (it is None in the trainer's call)."""
    import types
    import diffusers
    sys.modules.setdefault("imageio", types.ModuleType("imageio"))
    from models.layerdiffuse_VAE import LatentTransparencyOffsetEncoder, UNet384   # verbatim reference
    from models.pipeline_stage2 import MaskedLatentToVideoPipeline                 # verbatim reference
    from models.unet_3d_condition_mask import UNet3DConditionModel                 # verbatim reference

    class UNetDroppingImageEmbeds(UNet3DConditionModel):
        def forward(self, *a, image_embeds=None, **k):
            assert image_embeds is None
            return super().forward(*a, **k)

    out = {}
    # --- the two models alone, bf16-rounded weights and inputs, fp32 math (what the GPU parity test loads into the sm_100a mirror)
    dec = fill_deterministic(UNet384().eval(), seed=7)
    dec.load_state_dict({k: v.bfloat16().float() for k, v in dec.state_dict().items()})
    enc = fill_deterministic(LatentTransparencyOffsetEncoder().eval(), seed=8)
    enc.load_state_dict({k: v.bfloat16().float() for k, v in enc.state_dict().items()})
    g = torch.Generator().manual_seed(31)
    x = torch.randn(2, 3, 64, 96, generator=g).clamp(-1, 1).bfloat16().float()
    lat = torch.randn(2, 4, 8, 12, generator=g).bfloat16().float()
    rgba_in = torch.cat([torch.randn(1, 3, 64, 96, generator=g).clamp(-1, 1), torch.rand(1, 1, 64, 96, generator=g)], dim=1)
    rgba_in = rgba_in.bfloat16().float()
    with torch.no_grad():
        out["dec_out"] = dec(x, lat)
        out["enc_out"] = enc(rgba_in)
    out.update(dec_x=x, dec_latent=lat, enc_in=rgba_in, dec_keys=sorted(dec.state_dict().keys()),
               enc_keys=sorted(enc.state_dict().keys()), dec_config=dict(dec.config))
    print("transparent: UNet384", tuple(out["dec_out"].shape), float(out["dec_out"].abs().mean()), "encoder",
          tuple(out["enc_out"].shape), float(out["enc_out"].abs().mean()))

    # --- the pipeline call: tiny UNet3D + tiny VAE + full-size UNet384 (it is small), DDIM 3 steps, CFG 9
    unet = fill_deterministic(UNetDroppingImageEmbeds(**TINY).eval(), seed=0)
    vae = fill_deterministic(diffusers.AutoencoderKL(**TINY_VAE).eval(), seed=1)
    dec32 = fill_deterministic(UNet384().eval(), seed=7)
    sched = diffusers.DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                                    clip_sample=False, set_alpha_to_one=False, steps_offset=1)
    pipe = diffusers.TextToVideoSDPipeline(vae=vae, text_encoder=None, tokenizer=None, unet=unet, scheduler=sched)
    g = torch.Generator().manual_seed(9)
    lat0 = torch.randn(1, 4, 4, 16, 16, generator=g)
    cond = torch.randn(1, 4, 1, 16, 16, generator=g)
    pe = torch.randn(1, 7, 32, generator=g)
    ne = torch.randn(1, 7, 32, generator=g)
    mask1 = (torch.rand(1, 1, 1, 16, 16, generator=g) > 0.5).float()          # mask_1_frame, train_transparent_i2v_stage2.py:441
    video, latents, pngs, alpha_jpg, pngs_rgb = MaskedLatentToVideoPipeline.__call__(
        pipe, clean_latents=None, vae_alpha_decoder=dec32, prompt_embeds=pe, negative_prompt_embeds=ne, latents=lat0,
        width=128, height=128, num_frames=4, num_inference_steps=3, guidance_scale=9.0, motion=[5], return_dict=False,
        condition_latent=cond, mask=mask1, output_type="pt")
    out.update(pipe_latents_in=lat0, pipe_cond=cond, pipe_pe=pe, pipe_ne=ne, pipe_mask=mask1, pipe_video=video.half(),
               pipe_latents=latents, pipe_pngs=torch.from_numpy(pngs.copy()), pipe_alpha=torch.from_numpy(alpha_jpg.copy()))
    # the call as the reference wrote it, on its own UNet: the TypeError the mirror documents
    plain = fill_deterministic(UNet3DConditionModel(**TINY).eval(), seed=0)
    pipe2 = diffusers.TextToVideoSDPipeline(vae=vae, text_encoder=None, tokenizer=None, unet=plain, scheduler=sched)
    try:
        MaskedLatentToVideoPipeline.__call__(pipe2, vae_alpha_decoder=dec32, prompt_embeds=pe, negative_prompt_embeds=ne,
                                             latents=lat0, width=128, height=128, num_frames=4, num_inference_steps=3,
                                             motion=[5], return_dict=False, condition_latent=cond, mask=mask1)
        out["image_embeds_error"] = None
    except TypeError as e:
        out["image_embeds_error"] = str(e)
    torch.save(out, os.path.join(HERE, "transparent_ref.pt"))
    print("transparent: pipeline video", tuple(video.shape), "latents", float(latents.abs().mean()), "pngs", pngs.shape,
          "alpha on:", float((alpha_jpg == 255).mean()), "| as-written call ->", out["image_embeds_error"])


def forward_branches_golden():
    """The remaining keyword branches of the VERBATIM UNet3DConditionModel.forward (models/unet_3d_condition_mask.py:338-526):
    `attention_mask` (:385-388 builds a bias that no block ever reads: models/unet_3d_blocks.py:340,489,720) and `class_labels`
    (never read) leave the output bit-identical; `timestep_cond` enters time_embedding.cond_proj when no motion value is used
    (:418-419)."""
    from models.unet_3d_condition_mask import UNet3DConditionModel            # verbatim reference
    torch.manual_seed(0)
    ref = fill_deterministic(UNet3DConditionModel(**TINY).eval(), seed=0)
    inp = tiny_inputs()
    g = torch.Generator().manual_seed(12)
    tc = torch.randn(2, 32, generator=g)
    am = (torch.rand(2, 7, generator=g) > 0.3).float()
    with torch.no_grad():
        base = ref(inp["sample"], inp["timestep"], inp["ehs"], condition_latent=inp["cond"], mask=inp["mask"],
                   motion=inp["motion"]).sample
        with_am = ref(inp["sample"], inp["timestep"], inp["ehs"], condition_latent=inp["cond"], mask=inp["mask"],
                      motion=inp["motion"], attention_mask=am).sample
        with_cl = ref(inp["sample"], inp["timestep"], inp["ehs"], condition_latent=inp["cond"], mask=inp["mask"],
                      motion=inp["motion"], class_labels=torch.tensor([1, 2])).sample
        out_tc = ref(inp["sample"], inp["timestep"], inp["ehs"], condition_latent=inp["cond"], mask=inp["mask"],
                     motion=None, timestep_cond=tc).sample
        out_tc_motion = ref(inp["sample"], inp["timestep"], inp["ehs"], condition_latent=inp["cond"], mask=inp["mask"],
                            motion=inp["motion"], timestep_cond=tc).sample
    torch.save({"attention_mask_noop": bool(torch.equal(base, with_am)), "class_labels_noop": bool(torch.equal(base, with_cl)),
                "timestep_cond_overridden_by_motion": bool(torch.equal(base, out_tc_motion)),
                "timestep_cond": tc, "out_timestep_cond": out_tc}, os.path.join(HERE, "unet_forward_branches_ref.pt"))
    print("unet_forward_branches_ref.pt: attention_mask noop", torch.equal(base, with_am), "| class_labels noop",
          torch.equal(base, with_cl), "| motion overrides timestep_cond", torch.equal(base, out_tc_motion),
          "| timestep_cond changes output by", float((out_tc - base).abs().mean()))


def config_errors_golden():
    """What the VERBATIM UNet3DConditionModel constructor (models/unet_3d_condition_mask.py:118-131) raises for each
    inconsistent config of tests/test_unet_config_cpu.py: exception type and message, as JSON."""
    import json
    sys.path.insert(0, os.path.dirname(HERE))
    from test_unet_config_cpu import BAD
    from models.unet_3d_condition_mask import UNet3DConditionModel            # verbatim reference
    cases = []
    for cfg in BAD:
        try:
            UNet3DConditionModel(**cfg)
            err = None
        except Exception as e:
            err = {"type": type(e).__name__, "message": str(e)}
        cases.append({"config": cfg, "error": err})
    with open(os.path.join(HERE, "unet_config_errors_ref.json"), "w") as f:
        json.dump({"cases": cases}, f, indent=1)
        f.write("\n")
    print("unet_config_errors_ref.json:", [c["error"] and c["error"]["type"] for c in cases])


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "config_errors":
        import diffusers  # noqa: F401  (the shim)
        config_errors_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == "svd":
        svd_goldens()
    elif len(sys.argv) > 1 and sys.argv[1] == "svd_text":
        import diffusers  # noqa: F401  (the shim)
        svd_text_goldens()
    elif len(sys.argv) > 1 and sys.argv[1] == "branches":
        import diffusers  # noqa: F401  (the shim)
        forward_branches_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == "transparent":
        import diffusers  # noqa: F401  (the shim)
        transparent_goldens()
    elif len(sys.argv) > 1 and sys.argv[1] == "oddsize":
        import diffusers  # noqa: F401  (the shim)
        oddsize_unet_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == "benchmarked":
        # python tests/golden/make_golden.py benchmarked   (only the two expensive fixtures, minutes of CPU)
        import diffusers  # noqa: F401  (the shim)
        vae_fullsize_golden()
        config2_unet_golden()
    else:
        main()
