"""CPU: pins the oracle restatement (oracle/composition.py) against fixtures produced by the VERBATIM reference files
run over the diffusers shim (tests/golden/make_golden.py).  The shim itself is 'parity unpinned' (no real diffusers
available); these tests pin the *composition* (reference models/*.py) and the self-consistency of the shim."""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(HERE, "golden"))

from oracle.composition import (AutoencoderKL, DDIMScheduler, DPMSolverMultistepScheduler, OracleUNet3D,  # noqa: E402
                                fill_deterministic, oracle_sampling_loop)
from make_golden import tiny_inputs  # noqa: E402


def _tiny_unet(gold):
    cfg = dict(gold["config"])
    cfg.pop("sample_size")
    m = OracleUNet3D(**cfg).eval()
    assert sorted(m.state_dict().keys()) == gold["keys"], "state_dict keys differ from the reference model"
    return fill_deterministic(m, seed=0)


def test_unet_composition_matches_reference_files():
    gold = torch.load(os.path.join(HERE, "golden", "unet_tiny_ref.pt"))
    m = _tiny_unet(gold)
    inp = tiny_inputs()
    with torch.no_grad():
        out = m(inp["sample"], inp["timestep"], inp["ehs"], inp["cond"], inp["mask"], motion=inp["motion"])
        out2 = m(inp["sample"], 37, inp["ehs"], inp["cond"], None, motion=None)
    assert torch.allclose(out, gold["out"], rtol=1e-5, atol=1e-6), float((out - gold["out"]).abs().max())
    assert torch.allclose(out2, gold["out_nomask_t37"], rtol=1e-5, atol=1e-6)


def test_sampling_loop_matches_reference_pipeline():
    gold_u = torch.load(os.path.join(HERE, "golden", "unet_tiny_ref.pt"))
    gold = torch.load(os.path.join(HERE, "golden", "pipeline_tiny_ref.pt"))
    unet = _tiny_unet(gold_u)
    vae = AutoencoderKL(**gold["vae_config"]).eval()
    assert sorted(vae.state_dict().keys()) == gold["vae_keys"]
    fill_deterministic(vae, seed=1)
    sched = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False,
                          set_alpha_to_one=False, steps_offset=1)
    mask = torch.ones(1, 1, 1, 16, 16)
    video, lat = oracle_sampling_loop(unet, sched, gold["latents_in"], gold["pe"], gold["ne"], gold["cond"], mask, [4],
                                      guidance_scale=9.0, num_inference_steps=3, vae=vae)
    assert torch.allclose(lat, gold["latents"], rtol=1e-4, atol=1e-5), float((lat - gold["latents"]).abs().max())
    assert torch.allclose(video, gold["video"].float(), rtol=2e-3, atol=2e-3)
    dpm = DPMSolverMultistepScheduler.from_config(sched.config)
    _, lat2 = oracle_sampling_loop(unet, dpm, gold["latents_in"], gold["pe"], gold["ne"], gold["cond"], mask, [4],
                                   guidance_scale=9.0, num_inference_steps=4)
    assert torch.allclose(lat2, gold["latents_dpm"], rtol=1e-4, atol=1e-5)


def test_common_functions_match_reference_utils():
    """oracle restatements of utils/common.py (DDPM_forward_timesteps :32-48, tensor_to_vae_latent :12-20) against the
    outputs of the verbatim reference functions (tests/golden/make_golden.py::common_golden)."""
    from oracle.composition import oracle_ddpm_forward_timesteps, oracle_encode_image
    gold = torch.load(os.path.join(HERE, "golden", "common_ref.pt"))
    sched = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False,
                          set_alpha_to_one=False, steps_offset=1)
    sched.set_timesteps(10)
    for name, dt in (("f32", torch.float32), ("bf16", torch.bfloat16), ("f16", torch.float16)):
        torch.manual_seed(3)
        xt, ts = oracle_ddpm_forward_timesteps(gold["x0"].to(dt), 4, 5, sched)
        assert torch.equal(xt, gold[f"xt_{name}"]), name
        assert torch.equal(torch.as_tensor(ts), torch.as_tensor(gold["timesteps"]))
    pg = torch.load(os.path.join(HERE, "golden", "pipeline_tiny_ref.pt"))
    vae = AutoencoderKL(**pg["vae_config"]).eval()
    fill_deterministic(vae, seed=1)
    with torch.no_grad():
        lat = oracle_encode_image(vae, gold["frames"])
    assert torch.allclose(lat, gold["latents"], rtol=1e-5, atol=1e-6)


import pytest  # noqa: E402


@pytest.mark.parametrize("name", ["unet_small_ref.pt", "unet_config1_ref.pt"])
def test_oracle_matches_reference_at_product_shapes(name):
    """The verbatim reference UNet at shapes the sm_100a product accepts (head_dim 64; BASELINE config 1 full size):
    the same fixtures tests/test_gpu_unet.py compares the CUDA path with."""
    from make_golden import fp16_inputs
    gold = torch.load(os.path.join(HERE, "golden", name))
    cfg = {k: v for k, v in gold["config"].items() if k != "sample_size"}
    unet = OracleUNet3D(**cfg).eval()
    fill_deterministic(unet, seed=0)
    assert len(unet.state_dict()) == gold["n_keys"]
    unet.load_state_dict({k: v.half().float() for k, v in unet.state_dict().items()})
    inp = fp16_inputs(**gold["shape"])
    with torch.no_grad():
        out = unet(inp["sample"], gold["timestep"], inp["ehs"], inp["cond"], inp["mask"], motion=torch.tensor([gold["motion"]]))
    err = float((out - gold["out"]).abs().max())
    assert torch.allclose(out, gold["out"], rtol=1e-4, atol=2e-5), err


def test_shim_recalled_facts():
    """One assertion per RECALLED diffusers-0.24 fact that SURVEY.md 8(c) lists as most likely to be wrong."""
    from diffusers._impl import GEGLU, TemporalConvLayer, Timesteps, TimestepEmbedding, Upsample2D, ResnetBlock2D
    import torch.nn.functional as F
    g = GEGLU(4, 6)
    x = torch.randn(3, 4)
    full = g.proj(x)
    assert torch.allclose(g(x), full[:, :6] * F.gelu(full[:, 6:]))                 # chunk order (value, gate)
    t = Timesteps(8, True, 0)(torch.tensor([3.0]))
    freq = torch.exp(-torch.log(torch.tensor(10000.0)) * torch.arange(4) / 4)
    assert torch.allclose(t[0, :4], torch.cos(3.0 * freq), atol=1e-6)              # flip_sin_to_cos -> cos first
    assert torch.allclose(t[0, 4:], torch.sin(3.0 * freq), atol=1e-6)
    te = TimestepEmbedding(8, 16, cond_proj_dim=8)
    assert te.cond_proj.bias is None                                                # cond_proj is bias-free
    tc = TemporalConvLayer(32, 32).eval()
    y = torch.randn(6, 32, 4, 4)
    assert torch.equal(tc(y, num_frames=3), y)                                      # zero-init conv4 => identity
    up = Upsample2D(4, use_conv=True).eval()
    z = torch.randn(1, 4, 3, 3)
    assert torch.allclose(up(z), up.conv(F.interpolate(z, scale_factor=2.0, mode="nearest")))
    r = ResnetBlock2D(in_channels=32, out_channels=32, temb_channels=8).eval()
    assert r.conv_shortcut is None and r.norm1.eps == 1e-6


def test_oracle_matches_reference_at_odd_latent_size():
    """`forward_upsample_size` path (models/unet_3d_condition_mask.py:377-383,486-491): 15 x 17 latents.  Compared in
    float64: the fp32 fixture carries ~3e-6 of rounding that another CPU's convolution kernels do not reproduce."""
    gold = torch.load(os.path.join(HERE, "golden", "unet_small_oddsize_ref.pt"))
    cfg = {k: v for k, v in gold["config"].items() if k != "sample_size"}
    m = fill_deterministic(OracleUNet3D(**cfg).eval(), seed=0)
    m.load_state_dict({k: v.half().float() for k, v in m.state_dict().items()})
    m = m.double()
    i = {k: v.double() for k, v in gold["inputs"].items()}
    with torch.no_grad():
        out = m(i["sample"], gold["timestep"], i["ehs"], i["cond"], i["mask"],
                motion=torch.tensor([gold["motion"]], dtype=torch.float64))
    ref = gold["out_f64"]
    assert torch.allclose(out, ref, rtol=1e-5, atol=1e-6), float((out - ref).abs().max())


def test_oracle_vae_matches_reference_entry_points_full_size():
    """Full-size SD VAE: oracle helpers vs the verbatim `tensor_to_vae_latent` / `decode_latents` fixture (bf16-rounded
    weights and inputs, fp32 math; ~15 s of CPU)."""
    from oracle.composition import oracle_decode_latents, oracle_encode_image
    gold = torch.load(os.path.join(HERE, "golden", "vae_fullsize_ref.pt"))
    vae = fill_deterministic(AutoencoderKL().eval(), seed=1)
    vae.load_state_dict({k: v.bfloat16().float() for k, v in vae.state_dict().items()})
    g = torch.Generator().manual_seed(gold["seed"])
    frames = torch.randn(1, 1, 3, 512, 512, generator=g).clamp(-1, 1).bfloat16().float()
    lat = torch.randn(1, 4, 2, 64, 64, generator=g).bfloat16().float()
    with torch.no_grad():
        enc = oracle_encode_image(vae, frames)
        vid = oracle_decode_latents(vae, lat[:, :, :1])
    assert torch.allclose(enc, gold["enc_latents"], rtol=1e-5, atol=1e-6)
    ref = gold["video_f16"][:, :, :1].float()
    assert (vid - ref).abs().max().item() <= 1e-3 * ref.abs().max().item()          # fixture stored in fp16


def test_svd_loop_matches_reference_pipeline():
    """config 4: `oracle_svd_sampling_loop` vs the verbatim MaskStableVideoDiffusionPipeline.__call__ fixture
    (models/pipeline.py:223-466: CFG with zeroed negatives, per-frame guidance vector, 9-channel input, Euler steps,
    chunked temporal-VAE decode)."""
    from make_golden import SvdImageEncoderStub
    from oracle.composition import (AutoencoderKLTemporalDecoder, EulerDiscreteScheduler, SVD_SCHED,
                                    UNetSpatioTemporalConditionModel, oracle_svd_sampling_loop)
    gold = torch.load(os.path.join(HERE, "golden", "svd_pipeline_tiny_ref.pt"))
    unet = fill_deterministic(UNetSpatioTemporalConditionModel(**gold["unet_config"]).eval(), 0)
    assert len(unet.state_dict()) == gold["n_unet_keys"]
    vae = fill_deterministic(AutoencoderKLTemporalDecoder(**gold["vae_config"]).eval(), 1)
    enc = fill_deterministic(SvdImageEncoderStub().eval(), 2)
    sched = EulerDiscreteScheduler(**SVD_SCHED)
    with torch.no_grad():
        emb = enc(gold["image"]).unsqueeze(1)
        il = vae.encode(gold["image"]).latent_dist.mode()
    frames, lat = oracle_svd_sampling_loop(unet, sched, vae, emb, il, gold["mask"], gold["latents_in"],
                                           num_inference_steps=3, noise_aug_strength=0.0, decode_chunk_size=3)
    assert torch.allclose(sched.timesteps, gold["timesteps"]) and torch.allclose(sched.sigmas, gold["sigmas"])
    assert torch.allclose(lat, gold["latents"], rtol=1e-5, atol=1e-5), float((lat - gold["latents"]).abs().max())
    # reference returns tensor2vid(frames): (x / 2 + 0.5).clamp(0, 1) per batch item, [F, 3, H, W]
    want = gold["frames"][0]
    got = (frames[0].permute(1, 0, 2, 3) / 2 + 0.5).clamp(0, 1)
    assert torch.allclose(got, want, rtol=1e-5, atol=1e-5), float((got - want).abs().max())


def test_svd_text_pipeline_image_branch_matches_reference():
    """`TextStableVideoDiffusionPipeline.__call__` (models/pipeline.py:468-731) as app_svd.py:120-133 calls it: the oracle loop with
    a per-frame mask and the caller's `condition_latent`, and with the image's own latents; plus the diffusers-0.24 failure for
    a multi-token context, which the product mirrors."""
    from make_golden import SvdImageEncoderStub
    from oracle.composition import (AutoencoderKLTemporalDecoder, EulerDiscreteScheduler, SVD_SCHED,
                                    UNetSpatioTemporalConditionModel, oracle_svd_sampling_loop)
    gold = torch.load(os.path.join(HERE, "golden", "svd_text_pipeline_tiny_ref.pt"))
    unet = fill_deterministic(UNetSpatioTemporalConditionModel(**gold["unet_config"]).eval(), 0)
    vae = fill_deterministic(AutoencoderKLTemporalDecoder(**gold["vae_config"]).eval(), 1)
    enc = fill_deterministic(SvdImageEncoderStub().eval(), 2)
    with torch.no_grad():
        emb = enc(gold["image"]).unsqueeze(1)
        il = vae.encode(gold["image"]).latent_dist.mode()
    kw = dict(num_inference_steps=3, noise_aug_strength=0.0, decode_chunk_size=3, frame_mask=gold["mask"])
    frames, lat = oracle_svd_sampling_loop(unet, EulerDiscreteScheduler(**SVD_SCHED), vae, emb, il, None, gold["latents_in"],
                                           condition_latent=gold["condition_latent"], **kw)
    assert torch.allclose(lat, gold["latents_image_condlat"], rtol=1e-5, atol=1e-5)
    got = (frames[0].permute(1, 0, 2, 3) / 2 + 0.5).clamp(0, 1)
    assert torch.allclose(got, gold["frames_image_condlat"][0], rtol=1e-5, atol=1e-5)
    _, lat2 = oracle_svd_sampling_loop(unet, EulerDiscreteScheduler(**SVD_SCHED), vae, emb, il, None, gold["latents_in"],
                                       decode=False, **kw)
    assert torch.allclose(lat2, gold["latents_image"], rtol=1e-5, atol=1e-5)
    assert gold["text_error"] is not None and "expanded size of the tensor (1) must match the existing size (7)" in gold["text_error"]
    with pytest.raises(RuntimeError, match="expanded size"):
        unet(torch.zeros(2, 5, 9, 8, 16), 1.0, torch.zeros(2, 7, 64), torch.zeros(2, 3))


# ---------------------------------------------------------------------------------------------- transparent-video branch (row f4)
def test_transparent_models_match_reference_files():
    """OracleUNet384 / OracleLatentTransparencyOffsetEncoder (what travels to the GPU box) against the outputs of the VERBATIM
    models/layerdiffuse_VAE.py classes (tests/golden/make_golden.py::transparent_goldens): same keys, same numbers."""
    from oracle.composition import OracleLatentTransparencyOffsetEncoder, OracleUNet384
    gold = torch.load(os.path.join(HERE, "golden", "transparent_ref.pt"))
    dec = OracleUNet384().eval()
    assert sorted(dec.state_dict().keys()) == gold["dec_keys"]
    fill_deterministic(dec, seed=7)
    dec.load_state_dict({k: v.bfloat16().float() for k, v in dec.state_dict().items()})
    enc = OracleLatentTransparencyOffsetEncoder().eval()
    assert sorted(enc.state_dict().keys()) == gold["enc_keys"]
    fill_deterministic(enc, seed=8)
    enc.load_state_dict({k: v.bfloat16().float() for k, v in enc.state_dict().items()})
    with torch.no_grad():
        y = dec(gold["dec_x"], gold["dec_latent"])
        e = enc(gold["enc_in"])
    assert torch.allclose(y, gold["dec_out"], rtol=1e-5, atol=1e-5), float((y - gold["dec_out"]).abs().max())
    assert torch.allclose(e, gold["enc_out"], rtol=1e-5, atol=1e-6)


def test_masked_pipeline_matches_reference_pipeline_stage2():
    """oracle_masked_sampling_loop against the VERBATIM MaskedLatentToVideoPipeline.__call__ (models/pipeline_stage2.py:171-337)
    called unbound like train_transparent_i2v_stage2.py:500-515: final latents, decoded video, uint8 RGBA frames; and the
    TypeError the as-written call raises on the repository's own UNet (`image_embeds`, :282)."""
    from oracle.composition import OracleUNet384, oracle_masked_sampling_loop
    gold_u = torch.load(os.path.join(HERE, "golden", "unet_tiny_ref.pt"))
    gold_p = torch.load(os.path.join(HERE, "golden", "pipeline_tiny_ref.pt"))
    gold = torch.load(os.path.join(HERE, "golden", "transparent_ref.pt"))
    unet = _tiny_unet(gold_u)
    vae = fill_deterministic(AutoencoderKL(**gold_p["vae_config"]).eval(), seed=1)
    dec = fill_deterministic(OracleUNet384().eval(), seed=7)
    sched = DDIMScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False,
                          set_alpha_to_one=False, steps_offset=1)
    video, lat, pngs = oracle_masked_sampling_loop(unet, sched, vae, dec, gold["pipe_latents_in"], gold["pipe_pe"],
                                                   gold["pipe_ne"], gold["pipe_cond"], gold["pipe_mask"], [5],
                                                   guidance_scale=9.0, num_inference_steps=3)
    assert torch.allclose(lat, gold["pipe_latents"], rtol=1e-4, atol=1e-4), float((lat - gold["pipe_latents"]).abs().max())
    assert torch.allclose(video, gold["pipe_video"].float(), rtol=2e-3, atol=2e-3)
    ref = gold["pipe_pngs"].numpy().astype(int)
    assert pngs.shape == ref.shape == (4, 128, 128, 4)
    d = abs(pngs.astype(int) - ref)
    assert d[..., :3].max() <= 1 and (d[..., 3] != 0).mean() < 1e-3        # foreground: truncation ties; alpha: threshold ties
    assert (gold["pipe_alpha"].numpy() == gold["pipe_pngs"].numpy()[..., 3]).all()
    assert "image_embeds" in gold["image_embeds_error"]


def test_unet2d_shim_recalled_facts():
    """One assertion per recalled diffusers-0.24 `unet_2d_blocks` fact listed in oracle/shim/diffusers/_unet2d.py."""
    from diffusers.models.unet_2d_blocks import UNetMidBlock2D, get_down_block, get_up_block
    kw = dict(num_layers=2, in_channels=16, out_channels=32, temb_channels=None, resnet_eps=1e-5, resnet_act_fn="silu",
              resnet_groups=4, downsample_padding=1, attention_head_dim=8)
    d = get_down_block("DownBlock2D", add_downsample=True, **kw).eval()
    x = torch.randn(1, 16, 8, 8)
    h, states = d(hidden_states=x, temb=None)
    assert len(states) == 3 and states[-1] is h and h.shape == (1, 32, 4, 4)         # downsampler output is a skip too
    a = get_down_block("AttnDownBlock2D", add_downsample=False, **kw).eval()
    assert a.downsamplers is None and len(a.attentions) == 2                         # add_downsample False -> type None
    at = a.attentions[0]
    assert at.heads == 4 and at.group_norm.num_groups == 4 and at.group_norm.eps == 1e-5 and at.residual_connection
    assert at.to_q.bias is not None and abs(at.scale - 8 ** -0.5) < 1e-9
    a2 = get_down_block("AttnDownBlock2D", add_downsample=True, **kw).eval()
    assert a2.downsamplers is not None                                               # default downsample_type "conv"
    ukw = dict(num_layers=3, in_channels=16, out_channels=32, prev_output_channel=64, temb_channels=None, resnet_eps=1e-5,
               resnet_act_fn="silu", resnet_groups=4, attention_head_dim=8)
    u = get_up_block("UpBlock2D", add_upsample=True, **ukw).eval()
    assert [r.in_channels for r in u.resnets] == [64 + 32, 32 + 32, 32 + 16]
    au = get_up_block("AttnUpBlock2D", add_upsample=False, **ukw).eval()
    assert au.upsamplers is None and len(au.attentions) == 3
    m = UNetMidBlock2D(in_channels=32, temb_channels=None, resnet_eps=1e-5, resnet_act_fn="silu", output_scale_factor=1,
                       resnet_time_scale_shift="default", attention_head_dim=8, resnet_groups=4, attn_groups=None,
                       add_attention=True, dropout=0.0)
    assert m.attentions[0].group_norm.num_groups == 4 and m.attentions[0].heads == 4 and len(m.resnets) == 2


def test_forward_keyword_branches_match_reference():
    """models/unet_3d_condition_mask.py:338-526 keyword branches recorded from the VERBATIM class: `attention_mask` and
    `class_labels` do not change the output (no block reads them), a motion value overrides `timestep_cond`, and `timestep_cond`
    alone enters time_embedding.cond_proj — which the oracle restates."""
    gold_u = torch.load(os.path.join(HERE, "golden", "unet_tiny_ref.pt"))
    gold = torch.load(os.path.join(HERE, "golden", "unet_forward_branches_ref.pt"))
    assert gold["attention_mask_noop"] and gold["class_labels_noop"] and gold["timestep_cond_overridden_by_motion"]
    m = _tiny_unet(gold_u)
    inp = tiny_inputs()
    with torch.no_grad():
        out = m(inp["sample"], inp["timestep"], inp["ehs"], inp["cond"], inp["mask"], motion=None,
                timestep_cond=gold["timestep_cond"])
        out_m = m(inp["sample"], inp["timestep"], inp["ehs"], inp["cond"], inp["mask"], motion=inp["motion"],
                  timestep_cond=gold["timestep_cond"])
    assert torch.allclose(out, gold["out_timestep_cond"], rtol=1e-5, atol=1e-6)
    assert torch.allclose(out_m, gold_u["out"], rtol=1e-5, atol=1e-6)
