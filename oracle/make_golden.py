"""Generates tests/golden/*.pt from the REAL reference (import of /root/reference/src - build container only).

    python -m oracle.make_golden          # rewrites every fixture

Weights of the model fixtures are NOT stored: they are regenerated deterministically by
diffusers_b200.specs.random_state_dict(spec, seed) on both sides and loaded into the reference modules here, so
the committed files only hold configs, seeds, inputs and the reference's outputs.  The nine block fixtures also
store the (tiny) reference-initialised state_dicts, because the reference's hard-coded golden slices
(tests/models/unets/test_unet_2d_blocks.py) are defined for the reference's own seeded default init.
"""
import gzip
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from diffusers_b200 import specs  # noqa: E402
from oracle import ref_shim  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

# (class name, block_type, extra init, input flags, expected slice copied from the reference test, its line)
BLOCK_KATS = [
    ("DownBlock2D", "down", {}, {}, [-0.0232, -0.9869, 0.8054, -0.0637, -0.1688, -1.4264, 0.4470, -1.3394, 0.0904], 28),
    ("AttnDownBlock2D", "down", {}, {}, [0.0636, 0.8964, -0.6234, -1.0131, 0.0844, 0.4935, 0.3437, 0.0911, -0.2957], 46),
    ("CrossAttnDownBlock2D", "down", {"cross_attention_dim": 32}, {}, [0.2238, -0.7396, -0.2255, -0.3829, 0.1925, 1.1665, 0.0603, -0.7295, 0.1983], 60),
    ("UNetMidBlock2D", "mid", {}, {}, [-0.1062, 1.7248, 0.3494, 1.4569, -0.0910, -1.2421, -0.9984, 0.6736, 1.0028], 164),
    ("UNetMidBlock2DCrossAttn", "mid", {"cross_attention_dim": 32}, {}, [0.0187, 2.4220, 0.4484, 1.1203, -0.6121, -1.5122, -0.8270, 0.7851, 1.8335], 178),
    ("UpBlock2D", "up", {}, {"res": True}, [-0.2041, -0.4165, -0.3022, 0.0041, -0.6628, -0.7053, 0.1928, -0.0325, 0.0523], 209),
    ("CrossAttnUpBlock2D", "up", {"cross_attention_dim": 32}, {"res": True}, [-0.1403, -0.3515, -0.0420, -0.1425, 0.3167, 0.5094, -0.2181, 0.5931, 0.5582], 240),
    ("AttnUpBlock2D", "up", {}, {"res": True}, [0.0979, 0.1326, 0.0021, 0.0659, 0.2249, 0.0059, 0.1132, 0.5952, 0.1033], 272),
    ("UpDecoderBlock2D", "up", {}, {"temb": False}, [0.4404, 0.1998, -0.9886, -0.3320, -0.3128, -0.7034, -0.6955, -0.2338, -0.3137], 317),
]

TINY_UNET = dict(sample_size=16, block_out_channels=(64, 128, 256), cross_attention_dim=128,
                 transformer_layers_per_block=(1, 2, 3), attention_head_dim=(1, 2, 4), addition_time_embed_dim=32,
                 projection_class_embeddings_input_dim=6 * 32 + 64)
TINY_VAE = dict(block_out_channels=(64, 64, 128, 128), sample_size=128)
TINY_VAE_D512 = dict(block_out_channels=(64, 64, 128, 512), sample_size=128)
TINY_FLUX = dict(patch_size=1, in_channels=16, num_layers=2, num_single_layers=3, attention_head_dim=64,
                 num_attention_heads=2, joint_attention_dim=96, pooled_projection_dim=48, guidance_embeds=True,
                 axes_dims_rope=(8, 28, 28))
FLUX128 = dict(patch_size=1, in_channels=16, num_layers=1, num_single_layers=2, attention_head_dim=128,
               num_attention_heads=2, joint_attention_dim=64, pooled_projection_dim=32, guidance_embeds=True,
               axes_dims_rope=(16, 56, 56))
DDPM64 = dict(sample_size=32, in_channels=3, out_channels=3, layers_per_block=2, block_out_channels=(64, 128),
              down_block_types=("DownBlock2D", "AttnDownBlock2D"), up_block_types=("AttnUpBlock2D", "UpBlock2D"),
              attention_head_dim=64, norm_num_groups=32)


def _sd(spec, seed):
    sd16 = specs.random_state_dict(spec, seed=seed, dtype=torch.bfloat16)
    return sd16, {k: v.float() for k, v in sd16.items()}


def block_inputs(flags):
    """tests/models/unets/test_unet_blocks_common.py:47-73 (get_dummy_input)"""
    gen = torch.manual_seed(0)
    inputs = {"hidden_states": torch.randn((4, 32, 32, 32), generator=gen)}
    if flags.get("temb", True):
        inputs["temb"] = torch.randn((4, 128), generator=gen)
    if flags.get("res"):
        inputs["res_hidden_states_tuple"] = (torch.randn((4, 32, 32, 32), generator=torch.manual_seed(1)),)
    return inputs


def gen_blocks(d):
    from diffusers.models.unets import unet_2d_blocks as B
    out = {}
    for name, btype, extra, flags, expected, line in BLOCK_KATS:
        init = {"in_channels": 32, "out_channels": 32, "temb_channels": 128}
        if btype == "up":
            init["prev_output_channel"] = 32
        if btype == "mid":
            init.pop("out_channels")
        if name in ("UNetMidBlock2D",):
            init = {"in_channels": 32, "temb_channels": 128}
        if name == "UpDecoderBlock2D":
            init = {"in_channels": 32, "out_channels": 32}
        init.update(extra)
        inputs = block_inputs(flags)  # seeds the GLOBAL generator: the block's default init below continues that stream
        block = getattr(B, name)(**init).eval()
        with torch.no_grad():
            o = block(**inputs)
        o = o[0] if isinstance(o, tuple) else o
        sl = o[0, -1, -3:, -3:].flatten()
        assert torch.allclose(sl, torch.tensor(expected), atol=5e-3), (name, sl, expected)
        # inputs are regenerated from their seeds by the tests (block_inputs below); only weights + goldens are stored
        out[name] = dict(init=init, flags=flags, state_dict={k: v.clone() for k, v in block.state_dict().items()},
                         expected_slice=torch.tensor(expected), reference_line=line, output_slice=sl.clone(),
                         output_abs_mean=float(o.abs().mean()), output_shape=tuple(o.shape))
        print("block", name, "ok")
    torch.save(out, os.path.join(OUT, "blocks.pt"))


def gen_schedulers(d):
    out = {}
    sdxl = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", timestep_spacing="leading", steps_offset=1)
    tabs = {}
    for n in (50, 30, 4):
        s = d.EulerDiscreteScheduler(**sdxl)
        s.set_timesteps(n)
        tabs[n] = dict(sigmas=s.sigmas.clone(), timesteps=s.timesteps.clone(), init_noise_sigma=float(s.init_noise_sigma))
    out["euler_sdxl"] = dict(config=sdxl, tables=tabs)
    flux = dict(shift=3.0, use_dynamic_shifting=True, base_shift=0.5, max_shift=1.15, base_image_seq_len=256, max_image_seq_len=4096)
    tabs = {}
    for n, seq in ((28, 4096), (4, 64)):
        s = d.FlowMatchEulerDiscreteScheduler(**flux)
        m = (1.15 - 0.5) / (4096 - 256)
        mu = seq * m + (0.5 - m * 256)
        s.set_timesteps(n, sigmas=np.linspace(1.0, 1 / n, n), mu=mu)
        tabs[(n, seq)] = dict(sigmas=s.sigmas.clone(), timesteps=s.timesteps.clone(), mu=mu)
    out["flow_match_flux"] = dict(config=flux, tables=tabs)
    # reference KATs (tests/schedulers/test_scheduler_euler.py:108-136, test_scheduler_ddpm.py:85-104), values hard-coded there
    out["kat"] = dict(euler_no_noise=(10.0807, 0.0131), ddpm_no_noise=(258.9606, 0.3372), ddpm_variance={0: 0.0, 487: 0.00979, 999: 0.02})
    # step-level vectors from the reference on CPU (bf16 tensors: pins the dtype-promotion behaviour)
    g = torch.Generator().manual_seed(3)
    eps = torch.randn(2, 4, 16, 16, generator=g).bfloat16()
    x = (torch.randn(2, 4, 16, 16, generator=g) * 10).bfloat16()
    s = d.EulerDiscreteScheduler(**sdxl)
    s.set_timesteps(30)
    s.set_begin_index(0)
    scaled = s.scale_model_input(x, s.timesteps[0])
    prev = s.step(eps, s.timesteps[0], x, return_dict=False)[0]
    out["euler_step_bf16"] = dict(eps=eps, x=x, scaled=scaled, prev=prev, n=30)
    s = d.FlowMatchEulerDiscreteScheduler(**flux)
    s.set_timesteps(4, sigmas=np.linspace(1.0, 1 / 4, 4), mu=0.6)
    s.set_begin_index(0)
    v = torch.randn(1, 64, 16, generator=g).bfloat16()
    xs = torch.randn(1, 64, 16, generator=g).bfloat16()
    out["flow_step_bf16"] = dict(v=v, x=xs, prev=s.step(v, s.timesteps[0], xs, return_dict=False)[0], mu=0.6)
    torch.save(out, os.path.join(OUT, "schedulers.pt"))
    print("schedulers ok")


STEPPERS = [  # (fixture key, reference class, constructor arguments)
    ("ddim_sdxl", "DDIMScheduler", dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False, set_alpha_to_one=False,
                                        steps_offset=1, timestep_spacing="leading")),
    ("ddim_trailing", "DDIMScheduler", dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", clip_sample=False,
                                            timestep_spacing="trailing")),
    ("euler_a_sdxl", "EulerAncestralDiscreteScheduler", dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                                                            timestep_spacing="leading", steps_offset=1)),
    ("dpmpp_2m_sdxl", "DPMSolverMultistepScheduler", dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                                                         timestep_spacing="leading", steps_offset=1)),
    ("dpmpp_2m_linspace", "DPMSolverMultistepScheduler", dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")),
    ("dpmpp_1", "DPMSolverMultistepScheduler", dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", solver_order=1)),
    ("unipc_sdxl", "UniPCMultistepScheduler", dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", timestep_spacing="leading", steps_offset=1)),
    ("unipc_linspace", "UniPCMultistepScheduler", dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")),
    ("dpmpp_2m_karras", "DPMSolverMultistepScheduler", dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", timestep_spacing="leading",
                                                           steps_offset=1, use_karras_sigmas=True)),
]


_SDXL_BETAS = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
VPRED_STEPPERS = [  # v_prediction variants (SD 2.x-v, v-pred SDXL fine-tunes): CPU-side fixtures only (same kernels, other coefficients)
    ("vpred_euler", "EulerDiscreteScheduler", dict(_SDXL_BETAS, timestep_spacing="trailing", prediction_type="v_prediction")),
    ("vpred_ddim", "DDIMScheduler", dict(_SDXL_BETAS, clip_sample=False, set_alpha_to_one=False, steps_offset=1, timestep_spacing="leading",
                                         prediction_type="v_prediction")),
    ("vpred_dpmpp_2m", "DPMSolverMultistepScheduler", dict(_SDXL_BETAS, timestep_spacing="leading", steps_offset=1, prediction_type="v_prediction")),
    ("vpred_unipc", "UniPCMultistepScheduler", dict(_SDXL_BETAS, prediction_type="v_prediction")),
]


def stepper_fake_model(x, t):
    """A deterministic stand-in for the denoiser (same dtype in and out) so that scheduler trajectories can be compared alone."""
    return (torch.sin(x.float() * 0.7 + float(t) * 0.01) * 0.8 + 0.1 * x.float()).to(x.dtype)


def gen_steppers(d):
    """tests/golden/schedulers2.pt: tables of the N4 steppers and whole trajectories of the REAL reference schedulers (fp32 and
    bf16 tensors on CPU) driven by stepper_fake_model, with the ancestral sampler's noise drawn from seeded generators."""
    out = {}
    for key, cls, kw in STEPPERS + VPRED_STEPPERS:
        tabs = {}
        for n in (30, 7):
            s = getattr(d, cls)(**kw)
            s.set_timesteps(n)
            tabs[n] = dict(timesteps=s.timesteps.clone(), sigmas=s.sigmas.clone() if hasattr(s, "sigmas") else None,
                           init_noise_sigma=float(s.init_noise_sigma))
        traj = {}
        for dt in (torch.float32, torch.bfloat16):
            s = getattr(d, cls)(**kw)
            s.set_timesteps(8)
            x = (torch.randn(2, 4, 8, 8, generator=torch.Generator().manual_seed(1)) * float(s.init_noise_sigma)).to(dt)
            g = torch.Generator().manual_seed(0)
            start = x.clone()
            for t in s.timesteps:
                eps = stepper_fake_model(s.scale_model_input(x, t), t)
                extra = dict(generator=g) if cls.startswith("EulerAncestral") else {}
                x = s.step(eps, t, x, return_dict=False, **extra)[0]
            traj[str(dt).split(".")[-1]] = dict(start=start, final=x.clone())
        out[key] = dict(cls=cls, config=kw, tables=tabs, trajectory=traj, steps=8)
    # "Euler Karras" (EulerDiscreteScheduler(use_karras_sigmas=True)): tables and an fp32 trajectory of the real reference
    ek = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", timestep_spacing="leading", steps_offset=1, use_karras_sigmas=True)
    tabs = {}
    for n in (30, 7):
        s = d.EulerDiscreteScheduler(**ek)
        s.set_timesteps(n)
        tabs[n] = dict(timesteps=s.timesteps.clone(), sigmas=s.sigmas.clone(), init_noise_sigma=float(s.init_noise_sigma))
    s = d.EulerDiscreteScheduler(**ek)
    s.set_timesteps(8)
    x = torch.randn(2, 4, 8, 8, generator=torch.Generator().manual_seed(1)) * float(s.init_noise_sigma)
    start = x.clone()
    for t in s.timesteps:
        x = s.step(stepper_fake_model(s.scale_model_input(x, t), t), t, x, return_dict=False)[0]
    out["euler_karras_sdxl"] = dict(cls="EulerDiscreteScheduler", config=ek, tables=tabs, steps=8, trajectory=dict(float32=dict(start=start, final=x.clone())))
    torch.save(out, os.path.join(OUT, "schedulers2.pt"))
    print("steppers ok")


def _run(mod, sd32, sd16, fn):
    mod.load_state_dict(sd32)
    with torch.no_grad():
        ref32 = fn(mod, torch.float32)
        mod16 = mod.to(torch.bfloat16)
        mod16.load_state_dict(sd16)
        ref16 = fn(mod16, torch.bfloat16)
    return ref32, ref16


def gen_models(d):
    out = {}
    g = torch.Generator().manual_seed(0)
    # ---- SDXL-style UNet
    cfg = dict(specs.SDXL_UNET_CONFIG)
    cfg.update(TINY_UNET)
    sd16, sd32 = _sd(specs.unet2d_condition_params(cfg), seed=1)
    x = torch.randn(2, 4, 16, 16, generator=g).bfloat16()
    ehs = torch.randn(2, 77, 128, generator=g).bfloat16()
    te = torch.randn(2, 64, generator=g).bfloat16()
    tid = torch.tensor([[128., 128, 0, 0, 128, 128]] * 2).bfloat16()
    t = torch.tensor(981.0)
    m = d.UNet2DConditionModel(**cfg).eval()
    r32, r16 = _run(m, sd32, sd16, lambda mod, dt: mod(x.to(dt), t, ehs.to(dt), added_cond_kwargs=dict(text_embeds=te.to(dt), time_ids=tid.to(dt)), return_dict=False)[0])
    out["unet_tiny"] = dict(cfg=cfg, seed=1, sample=x, timestep=t, encoder_hidden_states=ehs, text_embeds=te, time_ids=tid, ref32=r32, ref16=r16)
    print("unet", float((r32 - r16.float()).abs().max()))
    # ---- VAE decoders
    for name, upd, seed in (("vae_tiny", TINY_VAE, 2), ("vae_d512", TINY_VAE_D512, 3)):
        cfg = dict(specs.SDXL_VAE_CONFIG)
        cfg.update(upd)
        sd16, sd32 = _sd(specs.vae_decoder_params(cfg), seed=seed)
        z = torch.randn(2, 4, 16, 16, generator=g).bfloat16()
        m = d.AutoencoderKL(**cfg).eval()
        full32 = m.state_dict()
        full32.update(sd32)
        full16 = {k: v.bfloat16() for k, v in full32.items()}
        r32, r16 = _run(m, full32, full16, lambda mod, dt: mod.decode(z.to(dt), return_dict=False)[0])
        out[name] = dict(cfg=cfg, seed=seed, z=z, ref32=r32, ref16=r16)
        print(name, float((r32 - r16.float()).abs().max()))
    # ---- Flux transformers
    for name, fcfg, seed, S, T in (("flux_tiny", TINY_FLUX, 4, 64, 24), ("flux_hd128", FLUX128, 5, 256, 40)):
        sd16, sd32 = _sd(specs.flux_params(fcfg), seed=seed)
        side = int(S ** 0.5)
        hs = torch.randn(2, S, fcfg["in_channels"], generator=g).bfloat16()
        ehs = torch.randn(2, T, fcfg["joint_attention_dim"], generator=g).bfloat16()
        pooled = torch.randn(2, fcfg["pooled_projection_dim"], generator=g).bfloat16()
        ts = torch.tensor([0.7, 0.7])
        gd = torch.tensor([3.5, 3.5])
        img_ids = torch.zeros(side, side, 3)
        img_ids[..., 1] += torch.arange(side)[:, None]
        img_ids[..., 2] += torch.arange(side)[None, :]
        img_ids = img_ids.reshape(S, 3)
        txt_ids = torch.zeros(T, 3)
        m = d.FluxTransformer2DModel(**fcfg).eval()
        r32, r16 = _run(m, sd32, sd16, lambda mod, dt: mod(hidden_states=hs.to(dt), encoder_hidden_states=ehs.to(dt), pooled_projections=pooled.to(dt), timestep=ts.to(dt), img_ids=img_ids.to(dt), txt_ids=txt_ids.to(dt), guidance=gd, return_dict=False)[0])
        out[name] = dict(cfg=fcfg, seed=seed, hidden_states=hs, encoder_hidden_states=ehs, pooled=pooled, timestep=ts, guidance=gd, img_ids=img_ids, txt_ids=txt_ids, ref32=r32, ref16=r16)
        print(name, float((r32 - r16.float()).abs().max()))
    # ---- UNet2DModel (config 0 family)
    sd16, sd32 = _sd(specs.unet2d_params(DDPM64), seed=6)
    xi = torch.randn(2, 3, 32, 32, generator=g).bfloat16()
    m = d.UNet2DModel(**DDPM64).eval()
    r32, r16 = _run(m, sd32, sd16, lambda mod, dt: mod(xi.to(dt), torch.tensor(500)).sample)
    out["unet2d_ddpm"] = dict(cfg=DDPM64, seed=6, sample=xi, timestep=torch.tensor(500), ref32=r32, ref16=r16)
    print("unet2d", float((r32 - r16.float()).abs().max()))
    torch.save(out, os.path.join(OUT, "models.pt"))


def gen_pipelines(d):
    out = {}
    # ---- reference StableDiffusionXLPipeline, tiny UNet + VAE, fp32 CPU, embeddings in (SURVEY.md appendix A)
    ucfg = dict(specs.SDXL_UNET_CONFIG)
    ucfg.update(TINY_UNET)
    vcfg = dict(specs.SDXL_VAE_CONFIG)
    vcfg.update(TINY_VAE)
    usd16, usd32 = _sd(specs.unet2d_condition_params(ucfg), seed=1)
    vsd16, vsd32 = _sd(specs.vae_decoder_params(vcfg), seed=2)
    unet = d.UNet2DConditionModel(**ucfg).eval()
    unet.load_state_dict(usd32)
    vae = d.AutoencoderKL(**vcfg).eval()
    full = vae.state_dict()
    full.update(vsd32)
    vae.load_state_dict(full)
    skw = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", timestep_spacing="leading", steps_offset=1)
    pipe = d.StableDiffusionXLPipeline(vae=vae, text_encoder=None, text_encoder_2=None, tokenizer=None, tokenizer_2=None,
                                       unet=unet, scheduler=d.EulerDiscreteScheduler(**skw), add_watermarker=False)
    pipe.set_progress_bar_config(disable=True)
    g = torch.Generator().manual_seed(11)
    pe = torch.randn(1, 77, 128, generator=g)
    npe = torch.randn(1, 77, 128, generator=g)
    pool = torch.randn(1, 64, generator=g)
    npool = torch.randn(1, 64, generator=g)
    kw = dict(prompt_embeds=pe, negative_prompt_embeds=npe, pooled_prompt_embeds=pool, negative_pooled_prompt_embeds=npool,
              height=128, width=128, num_inference_steps=4, guidance_scale=7.5)
    img = pipe(generator=torch.Generator().manual_seed(0), output_type="pt", **kw).images
    lat = pipe(generator=torch.Generator().manual_seed(0), output_type="latent", **kw).images
    out["sdxl_tiny"] = dict(unet_cfg=ucfg, vae_cfg=vcfg, unet_seed=1, vae_seed=2, scheduler=skw, prompt_embeds=pe,
                            negative_prompt_embeds=npe, pooled=pool, negative_pooled=npool, height=128, width=128, steps=4,
                            guidance_scale=7.5, latent_seed=0, image=img, latents=lat)
    print("sdxl pipeline", tuple(img.shape), float(img.mean()))
    # ---- reference FluxPipeline (output_type latent)
    fsd16, fsd32 = _sd(specs.flux_params(TINY_FLUX), seed=4)
    tr = d.FluxTransformer2DModel(**TINY_FLUX).eval()
    tr.load_state_dict(fsd32)
    fkw = dict(shift=3.0, use_dynamic_shifting=True, base_shift=0.5, max_shift=1.15, base_image_seq_len=256, max_image_seq_len=4096)
    fvae = d.AutoencoderKL(**{**vcfg, "latent_channels": 4, "block_out_channels": (64, 64, 128, 128)}).eval()
    fp = d.FluxPipeline(scheduler=d.FlowMatchEulerDiscreteScheduler(**fkw), vae=fvae, text_encoder=None, tokenizer=None,
                        text_encoder_2=None, tokenizer_2=None, transformer=tr)
    fp.set_progress_bar_config(disable=True)
    fpe = torch.randn(1, 24, 96, generator=g)
    fpool = torch.randn(1, 48, generator=g)
    flat = fp(prompt_embeds=fpe, pooled_prompt_embeds=fpool, height=128, width=128, num_inference_steps=3, guidance_scale=3.5,
              generator=torch.Generator().manual_seed(0), output_type="latent").images
    out["flux_tiny"] = dict(cfg=TINY_FLUX, seed=4, scheduler=fkw, prompt_embeds=fpe, pooled=fpool, height=128, width=128, steps=3,
                            guidance_scale=3.5, latent_seed=0, vae_scale_factor=fp.vae_scale_factor, latents=flat)
    print("flux pipeline", tuple(flat.shape))
    # ---- reference DDPMPipeline (config 0): per-step RNG draws from the caller's generator
    dsd16, dsd32 = _sd(specs.unet2d_params(DDPM64), seed=6)
    u = d.UNet2DModel(**DDPM64).eval()
    u.load_state_dict(dsd32)
    dp = d.DDPMPipeline(unet=u, scheduler=d.DDPMScheduler())
    dp.set_progress_bar_config(disable=True)
    im = dp(batch_size=1, generator=torch.manual_seed(0), num_inference_steps=10, output_type="np").images
    out["ddpm"] = dict(cfg=DDPM64, seed=6, steps=10, image=torch.from_numpy(im))
    print("ddpm pipeline", im.shape)
    torch.save(out, os.path.join(OUT, "pipelines.pt"))


# layer-level known answers of the reference (tests/models/test_layers_utils.py): (name, class, init kwargs, input
# shape, extra inputs, expected 3x3 slice, test line).  Weights come from the reference's default init under manual_seed(0)
# AFTER the sample draw, exactly like the reference test does it.
LAYER_KATS = [
    ("upsample_default", "Upsample2D", dict(channels=32, use_conv=False), (1, 32, 32, 32), None,
     [-0.2173, -1.2079, -1.2079, 0.2952, 1.1254, 1.1254, 0.2952, 1.1254, 1.1254], 113),
    ("upsample_with_conv", "Upsample2D", dict(channels=32, use_conv=True), (1, 32, 32, 32), None,
     [0.7145, 1.3773, 0.3492, 0.8448, 1.0839, -0.3341, 0.5956, 0.1250, -0.4841], 140),
    ("upsample_with_conv_out_dim", "Upsample2D", dict(channels=32, use_conv=True, out_channels=64), (1, 32, 32, 32), None,
     [0.2703, 0.1656, -0.2538, -0.0553, -0.2984, 0.1044, 0.1155, 0.2579, 0.7755], 152),
    ("downsample_with_conv", "Downsample2D", dict(channels=32, use_conv=True), (1, 32, 64, 64), None,
     [0.9267, 0.5878, 0.3337, 1.2321, -0.1191, -0.3984, -0.7532, -0.0715, -0.3913], 192),
    ("downsample_with_conv_pad1", "Downsample2D", dict(channels=32, use_conv=True, padding=1), (1, 32, 64, 64), None,
     [0.9267, 0.5878, 0.3337, 1.2321, -0.1191, -0.3984, -0.7532, -0.0715, -0.3913], 207),
    ("downsample_with_conv_out_dim", "Downsample2D", dict(channels=32, use_conv=True, out_channels=16), (1, 32, 64, 64), None,
     [-0.6586, 0.5985, 0.0721, 0.1256, -0.1492, 0.4436, -0.2544, 0.5021, 1.1522], 219),
    ("resnet_default", "ResnetBlock2D", dict(in_channels=32, temb_channels=128), (1, 32, 64, 64), "temb",
     [-1.9010, -0.2974, -0.8245, -1.3533, 0.8742, -0.9645, -2.0584, 1.3387, -0.4746], 233),
    ("resnet_use_in_shortcut", "ResnetBlock2D", dict(in_channels=32, temb_channels=128, use_in_shortcut=True), (1, 32, 64, 64), "temb",
     [0.2226, -1.0791, -0.1629, 0.3659, -0.2889, -1.2376, 0.0582, 0.9206, 0.0044], 248),
    ("transformer2d_default", "Transformer2DModel", dict(in_channels=32, num_attention_heads=1, attention_head_dim=32, dropout=0.0,
                                                          cross_attention_dim=None), (1, 32, 64, 64), None,
     [-1.9455, -0.0066, -1.3933, -1.5878, 0.5325, -0.6486, -1.8648, 0.7515, -0.9689], 325),
    ("transformer2d_cross_attention_dim", "Transformer2DModel", dict(in_channels=64, num_attention_heads=2, attention_head_dim=32,
                                                                      dropout=0.0, cross_attention_dim=64), (1, 64, 64, 64), "context",
     [0.0143, -0.6909, -2.1547, -1.8893, 1.4097, 0.1359, -0.2521, -1.3359, 0.2598], 348),
]


def gen_layers(d):
    import diffusers.models.downsampling as DS
    import diffusers.models.resnet as RS
    import diffusers.models.upsampling as US
    from diffusers.models.transformers.transformer_2d import Transformer2DModel
    mods = dict(Upsample2D=US.Upsample2D, Downsample2D=DS.Downsample2D, ResnetBlock2D=RS.ResnetBlock2D, Transformer2DModel=Transformer2DModel)
    out = {}
    for name, cls, init, shape, extra, expected, line in LAYER_KATS:
        torch.manual_seed(0)
        sample = torch.randn(*shape)
        temb = torch.randn(1, 128) if extra == "temb" else None
        m = mods[cls](**init).eval()
        ctx = torch.randn(1, 4, 64) if extra == "context" else None  # drawn after the module's init, as in the reference test
        with torch.no_grad():
            if cls == "ResnetBlock2D":
                o = m(sample, temb)
            elif cls == "Transformer2DModel":
                o = m(sample, ctx).sample if ctx is not None else m(sample).sample
            else:
                o = m(sample)
        sl = o[0, -1, -3:, -3:].flatten()
        assert torch.allclose(sl, torch.tensor(expected), atol=1e-3), (name, sl, expected)
        out[name] = dict(cls=cls, init=init, shape=shape, extra=extra, context=ctx, state_dict={k: v.clone() for k, v in m.state_dict().items()},
                         expected_slice=torch.tensor(expected), reference_line=line, output_shape=tuple(o.shape),
                         output_abs_mean=float(o.abs().mean()))
        print("layer", name, "ok")
    # ---- tests/pipelines/ddpm/test_ddpm.py:28-66: dummy_uncond_unet (default init under manual_seed(0)) + DDPMScheduler(),
    # 2 steps, generator seed 0 -> hard-coded 3x3 slice of the last channel
    kcfg = dict(block_out_channels=(4, 8), layers_per_block=1, norm_num_groups=4, sample_size=8, in_channels=3, out_channels=3,
                down_block_types=("DownBlock2D", "AttnDownBlock2D"), up_block_types=("AttnUpBlock2D", "UpBlock2D"))
    torch.manual_seed(0)
    u = d.UNet2DModel(**kcfg).eval()
    dp = d.DDPMPipeline(unet=u, scheduler=d.DDPMScheduler())
    dp.set_progress_bar_config(disable=True)
    im = dp(generator=torch.Generator().manual_seed(0), num_inference_steps=2, output_type="np").images
    expected = np.array([0.0, 0.9996672, 0.00329116, 1.0, 0.9995991, 1.0, 0.0060907, 0.00115037, 0.0])
    assert np.abs(im[0, -3:, -3:, -1].flatten() - expected).max() < 1e-2
    out["ddpm_pipeline_kat"] = dict(cfg={**kcfg, "attention_head_dim": u.config.attention_head_dim}, state_dict={k: v.clone() for k, v in u.state_dict().items()},
                                    expected_slice=torch.from_numpy(expected), image=torch.from_numpy(im), reference_line=45)
    print("ddpm pipeline kat ok")
    torch.save(out, os.path.join(OUT, "layers.pt"))


MICRO_UNET = dict(sample_size=16, block_out_channels=(64, 64), down_block_types=("DownBlock2D", "CrossAttnDownBlock2D"),
                  up_block_types=("CrossAttnUpBlock2D", "UpBlock2D"), layers_per_block=1, cross_attention_dim=64,
                  transformer_layers_per_block=1, attention_head_dim=(1, 1), addition_time_embed_dim=32,
                  projection_class_embeddings_input_dim=256)
MICRO_VAE = dict(block_out_channels=(32, 32), down_block_types=("DownEncoderBlock2D",) * 2, up_block_types=("UpDecoderBlock2D",) * 2,
                 layers_per_block=1, sample_size=32)


def gen_checkpoints(d):
    """tests/golden/ckpt_sdxl_micro/: a pipeline directory written by the REFERENCE's own `save_pretrained` (bf16
    safetensors + config.json + scheduler_config.json + model_index.json) plus the reference pipeline's fp32 output for it:
    what `from_pretrained` of the shells must load (SURVEY.md 8f N1)."""
    import shutil
    ucfg = dict(specs.SDXL_UNET_CONFIG)
    ucfg.update(MICRO_UNET)
    vcfg = dict(specs.SDXL_VAE_CONFIG)
    vcfg.update(MICRO_VAE)
    torch.manual_seed(21)
    unet = d.UNet2DConditionModel(**ucfg).eval()
    vae = d.AutoencoderKL(**vcfg).eval()
    with torch.no_grad():  # default init leaves the zero-initialised / tiny tensors uninteresting: redraw everything
        g = torch.Generator().manual_seed(22)
        for m in (unet, vae):
            for n_, p_ in m.named_parameters():
                if p_.dim() >= 2:
                    p_.copy_(torch.randn(p_.shape, generator=g) * (1.0 / max(1, p_[0].numel())) ** 0.5)
                elif n_.endswith("weight"):
                    p_.copy_(1.0 + 0.1 * torch.randn(p_.shape, generator=g))
                else:
                    p_.copy_(0.1 * torch.randn(p_.shape, generator=g))
    unet, vae = unet.to(torch.bfloat16), vae.to(torch.bfloat16)
    skw = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", timestep_spacing="leading", steps_offset=1)
    pipe = d.StableDiffusionXLPipeline(vae=vae, text_encoder=None, text_encoder_2=None, tokenizer=None, tokenizer_2=None,
                                       unet=unet, scheduler=d.EulerDiscreteScheduler(**skw), add_watermarker=False)
    root = os.path.join(OUT, "ckpt_sdxl_micro")
    shutil.rmtree(root, ignore_errors=True)
    pipe.save_pretrained(root, safe_serialization=True)
    # the fp32 run of the very same (bf16-valued) weights is the ground truth; the bf16 eager run is the error yardstick
    g = torch.Generator().manual_seed(12)
    pe, npe = torch.randn(1, 77, 64, generator=g), torch.randn(1, 77, 64, generator=g)
    pool, npool = torch.randn(1, 64, generator=g), torch.randn(1, 64, generator=g)
    kw = dict(prompt_embeds=pe, negative_prompt_embeds=npe, pooled_prompt_embeds=pool, negative_pooled_prompt_embeds=npool,
              height=32, width=32, num_inference_steps=3, guidance_scale=5.0)
    pipe.set_progress_bar_config(disable=True)
    lat0 = torch.randn(1, 4, 16, 16, generator=torch.Generator().manual_seed(0))
    img16 = pipe(latents=lat0.bfloat16(), output_type="pt", **{k: (v.bfloat16() if torch.is_tensor(v) else v) for k, v in kw.items()}).images
    pipe32 = d.StableDiffusionXLPipeline(vae=vae.float(), text_encoder=None, text_encoder_2=None, tokenizer=None, tokenizer_2=None,
                                         unet=unet.float(), scheduler=d.EulerDiscreteScheduler(**skw), add_watermarker=False)
    pipe32.set_progress_bar_config(disable=True)
    img32 = pipe32(latents=lat0.bfloat16().float(), output_type="pt", **kw).images
    torch.save(dict(call={k: v for k, v in kw.items()}, latents=lat0.bfloat16(), image_fp32=img32, image_bf16=img16.float()),
               os.path.join(root, "expected.pt"))
    n = sum(os.path.getsize(os.path.join(dp, f)) for dp, _, fs in os.walk(root) for f in fs)
    print("ckpt_sdxl_micro", n // 1024, "KiB;", "bf16-vs-fp32 max", float((img16.float() - img32).abs().max()))


def gen_vae_encode(d):
    """tests/golden/vae_encode.pt: AutoencoderKL.encode of the real reference (moments in fp32 and bf16 CPU eager, and one seeded
    posterior sample) for the two tiny VAE configs (mid attention head_dim 128 -> fused kernel, 512 -> unfused path)."""
    out = {}
    g = torch.Generator().manual_seed(7)
    for name, upd, seed in (("vae_enc_tiny", TINY_VAE, 12), ("vae_enc_d512", TINY_VAE_D512, 13)):
        cfg = dict(specs.SDXL_VAE_CONFIG)
        cfg.update(upd)
        sd16, sd32 = _sd(specs.vae_params(cfg), seed=seed)
        x = (torch.randn(2, 3, 64, 64, generator=g) * 0.6).clamp(-1, 1).bfloat16()
        m = d.AutoencoderKL(**cfg).eval()
        assert set(m.state_dict().keys()) == set(sd32.keys()), set(m.state_dict().keys()) ^ set(sd32.keys())
        r32, r16 = _run(m, sd32, sd16, lambda mod, dt: mod.encode(x.to(dt)).latent_dist.parameters)
        post = d.models.autoencoders.vae.DiagonalGaussianDistribution(r16)
        smp = post.sample(generator=torch.Generator().manual_seed(0))
        rt32 = None
        if name == "vae_enc_tiny":
            m32 = d.AutoencoderKL(**cfg).eval()
            m32.load_state_dict(sd32)
            with torch.no_grad():
                rt32 = m32(x.float(), sample_posterior=False).sample   # encode -> mode -> decode
        out[name] = dict(cfg=cfg, seed=seed, x=x, ref32=r32, ref16=r16, sample16=smp, sample_seed=0, roundtrip32=rt32)
        print(name, tuple(r32.shape), float((r32 - r16.float()).abs().max()))
    torch.save(out, os.path.join(OUT, "vae_encode.pt"))


TEXT_CASES = [
    # name, kind, config overrides, seed, (batch, tokens)
    ("clip_l_tiny", "clip", dict(vocab_size=1000, hidden_size=128, intermediate_size=256, num_hidden_layers=3, num_attention_heads=2, hidden_act="quick_gelu",
                                 projection_dim=128), 21, (2, 77)),
    ("clip_g_tiny", "clip_proj", dict(vocab_size=1000, hidden_size=192, intermediate_size=512, num_hidden_layers=2, num_attention_heads=3, hidden_act="gelu",
                                      projection_dim=64), 22, (3, 77)),
    ("t5_tiny", "t5", dict(vocab_size=1000, d_model=128, d_kv=64, d_ff=256, num_layers=2, num_heads=2), 23, (2, 96)),
    ("t5_tiny_512", "t5", dict(vocab_size=1000, d_model=192, d_kv=64, d_ff=384, num_layers=1, num_heads=3), 24, (1, 512)),
]


def gen_text(d):
    """tests/golden/text.pt: the text encoders of the REAL transformers package (the third-party dependency the reference's
    pipelines call) in fp32 and bf16 CPU eager, on seeded token ids; weights are regenerated from (spec, seed) on both sides."""
    import transformers
    from diffusers_b200 import text_encoders as T
    out = {"transformers_version": transformers.__version__}
    for name, kind, upd, seed, (B, S) in TEXT_CASES:
        if kind == "t5":
            cfg = dict(T.T5_XXL_CONFIG, **upd)
            spec = T.t5_encoder_params(cfg)
            hf = transformers.T5EncoderModel(transformers.T5Config(**cfg)).eval()
        else:
            cfg = dict(T.CLIP_L_CONFIG, **upd)
            spec = T.clip_text_params(cfg, kind == "clip_proj")
            cls = transformers.CLIPTextModelWithProjection if kind == "clip_proj" else transformers.CLIPTextModel
            hf = cls(transformers.CLIPTextConfig(**cfg)).eval()
        sd16 = T.random_state_dict(spec, seed)
        sd32 = {k: v.float() for k, v in sd16.items()}
        g = torch.Generator().manual_seed(seed)
        ids = torch.randint(3, cfg["vocab_size"] - 1, (B, S), generator=g)
        if kind != "t5":  # an EOS (the largest id: legacy argmax pooling) somewhere in each row, padding after it
            for b in range(B):
                e = 5 + 9 * b
                ids[b, e] = cfg["vocab_size"] - 1
                ids[b, e + 1:] = 1
        rec = {}
        for tag, sdx, dt in (("ref32", sd32, torch.float32), ("ref16", sd16, torch.bfloat16)):
            m = hf.to(dt)
            full = dict(sdx)
            if kind == "t5":
                full["encoder.embed_tokens.weight"] = full["shared.weight"]
            missing, unexpected = m.load_state_dict(full, strict=False)
            assert not unexpected and all("position_ids" in k for k in missing), (missing, unexpected)
            with torch.no_grad():
                o = m(ids, output_hidden_states=True)
            r = dict(last_hidden_state=o.last_hidden_state.clone(), penultimate=o.hidden_states[-2].clone(), n_hidden=len(o.hidden_states))
            if kind == "clip":
                r["pooler_output"] = o.pooler_output.clone()
            if kind == "clip_proj":
                r["text_embeds"] = o.text_embeds.clone()
            rec[tag] = r
        out[name] = dict(kind=kind, cfg=cfg, seed=seed, ids=ids, **rec)
        print(name, tuple(rec["ref32"]["last_hidden_state"].shape), float((rec["ref32"]["last_hidden_state"] - rec["ref16"]["last_hidden_state"].float()).abs().max()))
    torch.save(out, os.path.join(OUT, "text.pt"))


def _inventory(sd):
    return {k: tuple(v.shape) for k, v in sd.items()}


def _files(root):
    """Every file under root: JSON files by content, safetensors files by metadata and {key: (dtype, shape)}."""
    from safetensors import safe_open
    out = {}
    for dp, _, fs in os.walk(root):
        for f in sorted(fs):
            p = os.path.join(dp, f)
            rel = os.path.relpath(p, root)
            if f.endswith(".json"):
                with open(p) as fh:
                    out[rel] = json.load(fh)
            elif f.endswith(".safetensors"):
                with safe_open(p, "pt") as st:
                    out[rel] = dict(metadata=st.metadata(), tensors={k: (str(st.get_tensor(k).dtype), tuple(st.get_tensor(k).shape)) for k in st.keys()})
            else:
                out[rel] = None
    return out


def gen_reference_api(d):
    """tests/golden/reference_api.json.gz: what the CPU tests of the reference-facing API (parameter inventories, checkpoint files,
    guidance_rescale) compared with the live reference, recorded so that they run without it.
      inventories      : state_dict names -> shapes of the reference modules (meta device) at the BASELINE.json sizes
      loaded           : for each micro model of tests/test_checkpoint.py, the reference's `from_pretrained` of what the shell's
                         `save_pretrained` wrote: loading info and state_dict names -> shapes
      save_pretrained  : the files the reference writes for a micro UNet2DModel (sharded, fp16 variant, DDPMPipeline): JSON
                         contents verbatim, safetensors files as metadata + names / dtypes / shapes
      rescale_noise_cfg: the reference function's outputs on seeded bf16 inputs (exact in JSON: bf16 values are doubles)"""
    import tempfile
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_checkpoint as tc
    from diffusers_b200.autoencoder_kl import AutoencoderKL
    out = {}
    with torch.device("meta"):
        out["inventories"] = dict(
            sdxl_unet=_inventory(d.UNet2DConditionModel(**specs.SDXL_UNET_CONFIG).state_dict()),
            sdxl_vae=_inventory(d.AutoencoderKL(**specs.SDXL_VAE_CONFIG).state_dict()),
            flux_dev=_inventory(d.FluxTransformer2DModel(**specs.FLUX_DEV_CONFIG).state_dict()),
            ddpm_tiny=_inventory(d.UNet2DModel(**specs.DDPM_TINY_CONFIG).state_dict()))
    loaded = {}
    cases = [(n, cls, dflt, micro, fn) for n, cls, dflt, micro, fn in tc.CASES if n != "AutoencoderKL"]
    cases.append(("AutoencoderKL", AutoencoderKL, specs.SDXL_VAE_CONFIG, tc.MICRO_VAE, specs.vae_params))
    with tempfile.TemporaryDirectory() as tmp:
        for name, cls, defaults, micro, spec_fn in cases:
            cfg = dict(defaults)
            cfg.update(micro)
            sd = specs.random_state_dict(spec_fn(cfg), seed=11, dtype=torch.bfloat16)
            exact = dict(fold_norms=False) if name == "UNet2DConditionModel" else {}
            cls(cfg, sd, device="cpu", **exact).save_pretrained(os.path.join(tmp, name))
            ref, info = getattr(d, name).from_pretrained(os.path.join(tmp, name), torch_dtype=torch.bfloat16, output_loading_info=True)
            loaded[name] = dict(cfg=cfg, info={k: list(v) for k, v in info.items()}, state_dict=_inventory(ref.state_dict()))
            print("loaded", name, len(loaded[name]["state_dict"]), {k: len(v) for k, v in info.items()})
    out["loaded"] = loaded
    cfg = dict(specs.DDPM_TINY_CONFIG)
    cfg.update(tc.MICRO_DDPM)
    torch.manual_seed(0)
    m = d.UNet2DModel(**cfg).to(torch.bfloat16)
    with tempfile.TemporaryDirectory() as tmp:
        m.save_pretrained(os.path.join(tmp, "u"), safe_serialization=True, max_shard_size="300KB")
        m.save_pretrained(os.path.join(tmp, "v"), safe_serialization=True, variant="fp16")
        d.DDPMPipeline(unet=m, scheduler=d.DDPMScheduler()).save_pretrained(os.path.join(tmp, "p"))
        out["save_pretrained"] = dict(cfg=cfg, dirs={k: _files(os.path.join(tmp, k)) for k in ("u", "v", "p")})
    from diffusers.pipelines.stable_diffusion_xl.pipeline_stable_diffusion_xl import rescale_noise_cfg
    g = torch.Generator().manual_seed(0)
    cfg_pred, text_pred = torch.randn(3, 4, 8, 8, generator=g).bfloat16() * 2, torch.randn(3, 4, 8, 8, generator=g).bfloat16()
    out["rescale_noise_cfg"] = {str(gr): rescale_noise_cfg(cfg_pred, text_pred, guidance_rescale=gr).float().tolist() for gr in (0.0, 0.3, 0.7, 1.0)}
    with gzip.GzipFile(os.path.join(OUT, "reference_api.json.gz"), "wb", mtime=0) as f:
        f.write(json.dumps(out).encode())


def gen_full_size(d):
    """tests/golden/full_size_reference.pt (needs a B200): the reference at the full sizes of tests/test_full_size_parity_gpu.py,
    on that test's weights and seeded CUDA inputs.  Per case: the test's fixed _sample() of the fp32 output, its shape, and the
    error of the reference's own 16-bit CUDA-eager run (the same calls as that test's live branch) against that fp32 output:
    ref16_mean_abs, ref16_max_abs, ref16_in_band_vs_fp32, the yardstick of the test's criterion."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_full_size_parity_gpu as fs
    fs._no_tf32()
    dev = fs.DEV
    out = {}

    def keep(name, r32, r16):
        e16 = (r16.float() - r32).abs()
        out[name] = dict(sample=fs._sample(r32), shape=tuple(r32.shape), ref16_mean_abs=float(e16.mean()), ref16_max_abs=float(e16.max()),
                         ref16_in_band_vs_fp32=fs._band(r16.float(), r32))
        print(name, {k: v for k, v in out[name].items() if k != "sample"}, float(r32.abs().max()))

    with torch.no_grad():
        cfg = dict(specs.SDXL_UNET_CONFIG)
        t = torch.tensor(981.0, device=dev)
        for dt, tag in ((torch.bfloat16, "bf16"), (torch.float16, "fp16")):
            sd32 = {k: v.float() for k, v in specs.random_state_dict(specs.unet2d_condition_params(cfg), seed=0, dtype=dt, device=dev).items()}
            x, ehs, te, tid = fs._sdxl_inputs(dt)
            m = fs._ref_module("UNet2DConditionModel", cfg, sd32, torch.float32)
            r32 = m(x.float(), t, ehs.float(), added_cond_kwargs=dict(text_embeds=te.float(), time_ids=tid.float()), return_dict=False)[0]
            m = m.to(dt)
            keep(f"sdxl_unet_{tag}", r32, m(x, t, ehs, added_cond_kwargs=dict(text_embeds=te, time_ids=tid), return_dict=False)[0])
            del m, sd32, r32
            fs._free()
        dt = torch.bfloat16
        cfg = dict(specs.SDXL_VAE_CONFIG)
        sd32 = {k: v.float() for k, v in specs.random_state_dict(specs.vae_decoder_params(cfg), seed=0, dtype=dt, device=dev).items()}
        z = fs._vae_decode_inputs(dt)
        m = fs._ref_module("AutoencoderKL", cfg, sd32, torch.float32, strict=False)
        r32 = m.decode(z.float(), return_dict=False)[0]
        m.decoder.to(dt)
        m.post_quant_conv.to(dt)
        keep("sdxl_vae_decode", r32, m.decode(z, return_dict=False)[0])
        del m, sd32
        sd32 = {k: v.float() for k, v in specs.random_state_dict(specs.vae_params(cfg), seed=0, dtype=dt, device=dev).items()}
        x = fs._vae_encode_inputs(dt)
        m = fs._ref_module("AutoencoderKL", cfg, sd32, torch.float32)
        r32 = m.encode(x.float()).latent_dist.parameters
        m = m.to(dt)
        keep("sdxl_vae_encode", r32, m.encode(x).latent_dist.parameters)
        del m, sd32
        fs._free()
        cfg = dict(specs.FLUX_DEV_CONFIG)
        sd16 = specs.random_state_dict(specs.flux_params(cfg), seed=0, dtype=dt, device=dev)
        hs, ehs, pooled, img_ids, txt_ids, ts, guidance = fs._flux_inputs(dt)
        m = fs._ref_module("FluxTransformer2DModel", cfg, sd16, dt)
        r16 = m(hidden_states=hs, encoder_hidden_states=ehs, pooled_projections=pooled, timestep=ts, img_ids=img_ids, txt_ids=txt_ids,
                guidance=guidance, return_dict=False)[0]
        del m
        sd32 = {k: v.float() for k, v in sd16.items()}
        del sd16
        fs._free()
        m = fs._ref_module("FluxTransformer2DModel", cfg, sd32, torch.float32)
        keep("flux_dev_shape", m(hidden_states=hs.float(), encoder_hidden_states=ehs.float(), pooled_projections=pooled.float(), timestep=ts.float(),
                                 img_ids=img_ids.float(), txt_ids=txt_ids.float(), guidance=guidance, return_dict=False)[0], r16)
    torch.save(out, os.path.join(OUT, "full_size_reference.pt"))


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    dmod = ref_shim.import_reference()
    which = sys.argv[1:] or ["blocks", "layers", "schedulers", "steppers", "models", "pipelines", "checkpoints", "vae_encode", "text",
                             "reference_api"]
    for w in which:
        globals()["gen_" + w](dmod)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)) // 1024, "KiB")
