"""CPU tests of the host-side logic: schedule construction (bit-identical to the reference tables), weight
packing, parameter specs, latent/RNG contract helpers, config objects."""
import numpy as np
import pytest
import torch

from diffusers_b200 import packing, specs
from diffusers_b200 import schedulers as S
from diffusers_b200.config import FrozenConfig
from diffusers_b200.pipelines import FluxPipeline, calculate_shift, randn_tensor


def test_euler_tables_bit_identical_to_reference(golden):
    fx = golden("schedulers")["euler_sdxl"]
    for n, tab in fx["tables"].items():
        s = S.EulerDiscreteScheduler(**fx["config"])
        s.set_timesteps(n)
        assert torch.equal(s.sigmas, tab["sigmas"]) and torch.equal(s.timesteps, tab["timesteps"])
        assert float(s.init_noise_sigma) == tab["init_noise_sigma"]
        assert s.order == 1 and s.config.num_train_timesteps == 1000


def test_flow_match_tables_bit_identical_to_reference(golden):
    fx = golden("schedulers")["flow_match_flux"]
    for (n, seq), tab in fx["tables"].items():
        s = S.FlowMatchEulerDiscreteScheduler(**fx["config"])
        s.set_timesteps(n, sigmas=np.linspace(1.0, 1 / n, n), mu=calculate_shift(seq))
        assert torch.equal(s.sigmas, tab["sigmas"]) and torch.equal(s.timesteps, tab["timesteps"])
        assert abs(calculate_shift(seq) - tab["mu"]) < 1e-12
    with pytest.raises(ValueError):
        S.FlowMatchEulerDiscreteScheduler(**fx["config"]).set_timesteps(4)  # dynamic shifting needs mu


def test_scheduler_rejects_unsupported_options():
    with pytest.raises(NotImplementedError):
        S.EulerDiscreteScheduler(use_exponential_sigmas=True)
    with pytest.raises(NotImplementedError):
        S.EulerDiscreteScheduler(prediction_type="sample")


def test_pack_conv_weight_layout():
    torch.manual_seed(0)
    w = torch.randn(5, 12, 3, 3)
    p = packing.pack_conv_weight(w)
    assert p.shape == (5, 9 * 64)
    for tap in range(9):
        r, s = divmod(tap, 3)
        assert torch.equal(p[:, tap * 64: tap * 64 + 12], w[:, :, r, s])
        assert not p[:, tap * 64 + 12:(tap + 1) * 64].any()
    p2 = packing.pack_conv_weight(w, split=(8, 4))
    assert p2.shape == (5, 9 * 128)
    assert torch.equal(p2[:, 128 * 4: 128 * 4 + 8], w[:, :8, 1, 1]) and torch.equal(p2[:, 128 * 4 + 64: 128 * 4 + 68], w[:, 8:, 1, 1])


def test_pack_geglu_interleave():
    w = torch.arange(16 * 4, dtype=torch.float32).reshape(16, 4)  # inner = 8
    b = torch.arange(16, dtype=torch.float32)
    wp, bp = packing.pack_geglu(w, b, tile_n=8)  # tiles of 4 value + 4 gate rows
    assert torch.equal(bp, torch.tensor([0., 1, 2, 3, 8, 9, 10, 11, 4, 5, 6, 7, 12, 13, 14, 15]))
    assert torch.equal(wp[:4, :4], w[:4]) and torch.equal(wp[4:8, :4], w[8:12]) and torch.equal(wp[8:12, :4], w[4:8])


def test_specs_full_size_parameter_counts():
    n = lambda spec: sum(int(np.prod(s)) for s in spec.values())  # noqa: E731
    assert n(specs.unet2d_condition_params(specs.SDXL_UNET_CONFIG)) == 2_567_463_684   # SURVEY.md §8d config 1
    assert n(specs.flux_params(specs.FLUX_DEV_CONFIG)) == 11_901_408_320               # config 2
    assert n(specs.vae_decoder_params(specs.SDXL_VAE_CONFIG)) == 49_490_199  # decoder 49.49 M + post_quant_conv


def test_specs_match_reference_state_dicts(reference_api):
    inv = reference_api["inventories"]  # the reference modules' state_dict shapes on the meta device
    pairs = [(inv["sdxl_unet"], specs.unet2d_condition_params(specs.SDXL_UNET_CONFIG)),
             (inv["flux_dev"], specs.flux_params(specs.FLUX_DEV_CONFIG)),
             (inv["ddpm_tiny"], specs.unet2d_params(specs.DDPM_TINY_CONFIG)),
             ({k: s for k, s in inv["sdxl_vae"].items() if k.startswith(("decoder", "post_quant"))}, specs.vae_decoder_params(specs.SDXL_VAE_CONFIG))]
    for ref, mine in pairs:
        assert {k: tuple(s) for k, s in ref.items()} == {k: tuple(s) for k, s in mine.items()}


def test_randn_tensor_contract():
    """CPU generator => CPU draw (device independent seeds); list of generators => per-sample seeding."""
    a = randn_tensor((2, 4, 8, 8), generator=torch.Generator().manual_seed(0), device="cpu", dtype=torch.float32)
    b = torch.randn((2, 4, 8, 8), generator=torch.Generator().manual_seed(0))
    assert torch.equal(a, b)
    c = randn_tensor((2, 3), generator=[torch.Generator().manual_seed(1), torch.Generator().manual_seed(2)], device="cpu", dtype=torch.float32)
    assert torch.equal(c[0:1], torch.randn((1, 3), generator=torch.Generator().manual_seed(1)))
    assert torch.equal(c[1:2], torch.randn((1, 3), generator=torch.Generator().manual_seed(2)))


def test_flux_pack_unpack_roundtrip():
    x = torch.randn(2, 16, 8, 12)
    p = FluxPipeline._pack_latents(x, 2, 16, 8, 12)
    assert p.shape == (2, 24, 64)
    assert torch.equal(FluxPipeline._unpack_latents(p, 8 * 8, 12 * 8, 8), x)
    ids = FluxPipeline._prepare_latent_image_ids(4, 6, "cpu", torch.float32)
    assert ids.shape == (24, 3) and ids[7].tolist() == [0, 1, 1]


def test_frozen_config():
    c = FrozenConfig(a=1, b=None)
    assert c.a == 1 and c["a"] == 1 and c.get("zz", 5) == 5 and c.b is None
    with pytest.raises(TypeError):
        c.a = 2
    with pytest.raises(AttributeError):
        c.missing


def test_models_refuse_cpu_tensors():
    from diffusers_b200 import ops
    from diffusers_b200.unet_2d_condition import UNet2DConditionModel
    cfg = dict(sample_size=16, block_out_channels=(64, 128), down_block_types=("DownBlock2D", "CrossAttnDownBlock2D"),
               up_block_types=("CrossAttnUpBlock2D", "UpBlock2D"), cross_attention_dim=64, transformer_layers_per_block=(1, 1),
               attention_head_dim=(1, 2), addition_time_embed_dim=8, projection_class_embeddings_input_dim=6 * 8 + 16, layers_per_block=1)
    m = UNet2DConditionModel.random_init(cfg, device="cpu")
    with pytest.raises(ops.B200Error):
        m(torch.zeros(1, 4, 16, 16), torch.tensor(1.0), torch.zeros(1, 7, 64),
          added_cond_kwargs=dict(text_embeds=torch.zeros(1, 16), time_ids=torch.zeros(1, 6)))
    bad = dict(cfg)
    bad["attention_head_dim"] = (2, 4)  # head_dim 32: not supported by the tcgen05 attention kernel
    with pytest.raises(NotImplementedError):
        UNet2DConditionModel.random_init(bad, device="cpu")


def test_step_invariant_caches_follow_the_tensor_not_its_address(monkeypatch):
    """The per-prompt caches (UNet text K/V, Flux context embedding and RoPE tables) must notice a new prompt even when
    the allocator gives the new tensor the old one's address: they key on the tensor object + its version counter."""
    from diffusers_b200 import ops
    from diffusers_b200.transformer_flux import FluxTransformer2DModel
    from diffusers_b200.unet_2d_condition import UNet2DConditionModel
    calls = []

    def fake_linear(x, w, N, **kw):
        calls.append(x.data_ptr())
        return torch.zeros(x.shape[0], N, dtype=x.dtype)

    monkeypatch.setattr(ops, "linear", fake_linear)
    ucfg = dict(specs.SDXL_UNET_CONFIG)
    ucfg.update(sample_size=16, block_out_channels=(64, 64), down_block_types=("DownBlock2D", "CrossAttnDownBlock2D"),
                up_block_types=("CrossAttnUpBlock2D", "UpBlock2D"), layers_per_block=1, cross_attention_dim=64,
                transformer_layers_per_block=1, attention_head_dim=(1, 1), addition_time_embed_dim=32,
                projection_class_embeddings_input_dim=256)
    unet = UNet2DConditionModel(ucfg, specs.random_state_dict(specs.unet2d_condition_params(ucfg), seed=0), device="cpu")
    a = torch.randn(2, 77, 64).bfloat16()
    kv1 = unet._text_kv(a)
    assert unet._text_kv(a) is kv1 and len(calls) == 1            # same prompt tensor, same step-invariant K/V
    b = a.clone()                                                  # another prompt (wherever the allocator puts it)
    assert unet._text_kv(b) is not kv1 and len(calls) == 2
    b.add_(1.0)                                                    # edited in place: version counter moves
    unet._text_kv(b)
    assert len(calls) == 3
    unet._reset_stateful_cache()
    unet._text_kv(b)
    assert len(calls) == 4

    fcfg = dict(patch_size=1, in_channels=16, num_layers=1, num_single_layers=1, attention_head_dim=64, num_attention_heads=2,
                joint_attention_dim=32, pooled_projection_dim=16, guidance_embeds=True, axes_dims_rope=(8, 28, 28))
    flux = FluxTransformer2DModel(fcfg, specs.random_state_dict(specs.flux_params(fcfg), seed=0), device="cpu")
    calls.clear()
    e = torch.randn(1, 8, 32).bfloat16()
    c1 = flux._context(e)
    assert flux._context(e) is c1 and len(calls) == 1
    assert flux._context(e.clone()) is not c1 and len(calls) == 2
    txt, img = torch.zeros(8, 3), torch.arange(48, dtype=torch.float32).reshape(16, 3)
    r1 = flux._rope_tables(txt, img)
    assert flux._rope_tables(txt, img) is r1
    r2 = flux._rope_tables(txt, img.clone())
    assert r2 is not r1 and torch.equal(r1[0], r2[0])
    img3 = img[None]
    r3 = flux._rope_tables(img3[0][:8] * 0, img3[0], owners=(txt, img3))  # per-call views: keyed on the caller's tensors
    assert flux._rope_tables(img3[0][:8] * 0, img3[0], owners=(txt, img3)) is r3


def test_unsupported_checkpoint_options_are_refused():
    """Options of a reference config that change the numerics and are not implemented must raise, never be ignored
    (they would otherwise slip in through from_pretrained)."""
    from diffusers_b200.autoencoder_kl import AutoencoderKL
    from diffusers_b200.unet_2d_condition import UNet2DConditionModel
    base = dict(specs.SDXL_UNET_CONFIG)
    UNet2DConditionModel._validate_config(base)
    UNet2DConditionModel._validate_config({**base, "use_linear_projection": False, "upcast_attention": None, "only_cross_attention": [False, False, False]})
    for bad in (dict(upcast_attention=True), dict(class_embed_type="timestep"), dict(num_class_embeds=10), dict(resnet_time_scale_shift="scale_shift"),
                dict(down_block_types=("DownBlock2D", "AttnDownBlock2D", "CrossAttnDownBlock2D")), dict(mid_block_type="UNetMidBlock2DSimpleCrossAttn"),
                dict(time_cond_proj_dim=256), dict(only_cross_attention=True), dict(addition_embed_type="text_image"), dict(act_fn="gelu"),
                dict(attention_type="gated"), dict(conv_in_kernel=5), dict(norm_num_groups=None), dict(cross_attention_dim=(768, 1024, 2048))):
        with pytest.raises(NotImplementedError):
            UNet2DConditionModel._validate_config({**base, **bad})
    vcfg = dict(specs.SDXL_VAE_CONFIG)
    vcfg.update(block_out_channels=(32, 32), up_block_types=("UpDecoderBlock2D", "AttnUpDecoderBlock2D"), down_block_types=("DownEncoderBlock2D",) * 2,
                layers_per_block=1)
    with pytest.raises(NotImplementedError):
        AutoencoderKL(vcfg, {}, device="cpu")


def test_fold_layer_norm_algebra_and_inverse():
    """packing.fold_layer_norm: LN(x) W^T + b == rstd * (x W'^T) + (b + W beta) with W' = W gamma - rowmean(W gamma), evaluated the way
    the GEMM epilogue does (raw rows, rstd from E[x^2] - E[x]^2); and the inverse used by reference_state_dict."""
    torch.manual_seed(0)
    M, K, N = 64, 96, 40
    x = (torch.randn(M, K) * 2 + 1.5).bfloat16()
    w, b = (torch.randn(N, K) * K ** -0.5).bfloat16(), torch.randn(N).bfloat16()
    gamma, beta = (torch.randn(K) * 0.3 + 1).bfloat16(), (torch.randn(K) * 0.5).bfloat16()
    wf, lb, shift = packing.fold_layer_norm(w, gamma, beta, b, torch.bfloat16)
    wp = packing.pack_linear_weight(wf)
    xf = x.float()
    mean = xf.mean(1, keepdim=True)
    var = (xf * xf).mean(1, keepdim=True) - mean * mean
    rstd = torch.rsqrt(var + 1e-5)
    acc = xf @ packing.unpack_linear_weight(wp, K).float().t()
    got = rstd * acc + lb.float()[None]
    ref = torch.nn.functional.layer_norm(xf, (K,), gamma.float(), beta.float(), 1e-5) @ w.float().t() + b.float()
    assert (got - ref).abs().max() < 4e-2  # W' and the bias are rounded to bf16 once
    rec = packing.unfold_layer_norm(wf, gamma, shift)
    assert (rec.float() - w.float()).abs().max() <= 2.0 ** -7 * w.float().abs().max()  # back within one bf16 ulp


def test_unet_fold_norms_flag_keeps_exact_weights_when_off():
    ucfg = dict(specs.SDXL_UNET_CONFIG)
    ucfg.update(sample_size=16, block_out_channels=(64, 128), down_block_types=("DownBlock2D", "CrossAttnDownBlock2D"),
                up_block_types=("CrossAttnUpBlock2D", "UpBlock2D"), cross_attention_dim=64, transformer_layers_per_block=(1, 1),
                attention_head_dim=(1, 2), addition_time_embed_dim=8, projection_class_embeddings_input_dim=6 * 8 + 16, layers_per_block=1)
    from diffusers_b200.unet_2d_condition import UNet2DConditionModel
    sd = specs.random_state_dict(specs.unet2d_condition_params(ucfg), seed=0)
    g = torch.Generator().manual_seed(5)
    for k in sd:  # non-trivial LayerNorm affine parameters (the default init is gamma = 1, beta = 0)
        if ".transformer_blocks." in k and ".norm" in k:
            sd[k] = (torch.randn(sd[k].shape, generator=g) * 0.3 + (1.0 if k.endswith("weight") else 0.0)).bfloat16()
    exact = UNet2DConditionModel(ucfg, sd, device="cpu", fold_norms=False).reference_state_dict()
    assert all(torch.equal(exact[k], sd[k]) for k in sd)
    folded = UNet2DConditionModel(ucfg, sd, device="cpu").reference_state_dict()
    for k in sd:
        d = (folded[k].float() - sd[k].float()).abs().max()
        # weights: re-rounded once (within an ulp); the GEGLU bias comes back as (b + W beta) - W' beta with the re-rounded W'
        tol = 2e-2 if k.endswith("ff.net.0.proj.bias") else 2.0 ** -5 * sd[k].float().abs().max() + 1e-6  # gamma down to ~0.4 amplifies the ulp
        assert d <= tol, (k, float(d))


def test_rescale_noise_cfg_is_the_references(monkeypatch, reference_api):
    """N4: guidance_rescale.  The formula against the unmodified reference's function on the same 16-bit tensors (bit for bit), and
    the SDXL drop-in loop applying it after the CFG combine (fake denoiser / stepper: the loop is glue, the kernels are tested elsewhere)."""
    from diffusers_b200.pipelines import StableDiffusionXLPipeline, rescale_noise_cfg
    g = torch.Generator().manual_seed(0)
    cfg_pred, text_pred = torch.randn(3, 4, 8, 8, generator=g).bfloat16() * 2, torch.randn(3, 4, 8, 8, generator=g).bfloat16()
    for gr in (0.0, 0.3, 0.7, 1.0):
        ref = torch.tensor(reference_api["rescale_noise_cfg"][str(gr)]).bfloat16()  # the reference's output, recorded
        assert torch.equal(rescale_noise_cfg(cfg_pred, text_pred, gr), ref), gr
    out = rescale_noise_cfg(cfg_pred.float(), text_pred.float(), 1.0)
    assert torch.allclose(out.std(dim=[1, 2, 3]), text_pred.float().std(dim=[1, 2, 3]), rtol=1e-5)  # full rescale: the text prediction's std per sample

    class Unet:
        config = type("C", (), dict(sample_size=2, in_channels=4, time_cond_proj_dim=None, addition_time_embed_dim=2))()
        add_embedding = type("A", (), dict(linear_1=type("L", (), dict(in_features=2 * 6 + 5))()))()
        device, dtype = torch.device("cpu"), torch.float32

        def __call__(self, x, t, encoder_hidden_states=None, added_cond_kwargs=None, return_dict=False):
            return (x * encoder_hidden_states.mean((1, 2))[:, None, None, None] + 0.25,)

    class Sched:
        init_noise_sigma = 1.0
        timesteps = torch.tensor([2.0, 1.0])
        seen = []

        def set_timesteps(self, n, device=None):
            pass

        def set_begin_index(self, i):
            pass

        def scale_model_input(self, x, t):
            return x

        def step(self, eps, t, x, return_dict=False):
            self.seen.append(eps.clone())
            return (x - 0.1 * eps,)

    vae = type("V", (), dict(config=type("C", (), dict(block_out_channels=(1, 1, 1, 1), scaling_factor=1.0))()))()
    pe, npe = torch.full((1, 3, 5), 2.0), torch.full((1, 3, 5), 0.5)
    pool = torch.ones(1, 5)
    lat0 = torch.randn(1, 4, 2, 2, generator=g)
    for gr in (0.0, 0.6):
        sch = Sched()
        sch.seen = []
        pipe = StableDiffusionXLPipeline(vae, Unet(), sch)
        out = pipe(pe, npe, pool, pool, height=16, width=16, num_inference_steps=2, guidance_scale=5.0, latents=lat0.clone(), output_type="latent",
                   fused=False, guidance_rescale=gr).images
        x = lat0.clone()
        for _ in range(2):
            u, c = x * 0.5 + 0.25, x * 2.0 + 0.25
            n = u + 5.0 * (c - u)
            if gr:
                n = rescale_noise_cfg(n, c, gr)
            x = x - 0.1 * n
        assert torch.allclose(out, x, rtol=1e-6, atol=1e-6), gr


def test_flux_true_cfg_composition():
    """N4: true CFG for Flux (pipeline_flux.py:911-927): a second transformer call per step under cache_context("uncond") with the negative
    embeddings, noise = neg + true_cfg_scale * (cond - neg); off unless true_cfg_scale > 1 AND negative embeddings are given."""
    calls = []

    class Tr:
        config = FrozenConfig(dict(in_channels=16, guidance_embeds=True))
        device, dtype = torch.device("cpu"), torch.float32
        ctx = None

        def cache_context(self, name):
            import contextlib

            @contextlib.contextmanager
            def cm():
                Tr.ctx = name
                yield
                Tr.ctx = None
            return cm()

        def __call__(self, hidden_states, timestep, guidance, pooled_projections, encoder_hidden_states, txt_ids, img_ids, joint_attention_kwargs=None,
                     return_dict=False):
            calls.append((Tr.ctx, float(encoder_hidden_states.mean()), txt_ids))
            return (hidden_states * encoder_hidden_states.mean() + pooled_projections.mean(),)

    class Sched:
        config = dict()
        timesteps = torch.tensor([900.0, 500.0])

        def set_timesteps(self, n, device=None, sigmas=None, mu=None):
            pass

        def set_begin_index(self, i):
            pass

        def step(self, eps, t, x, return_dict=False):
            return (x - 0.5 * eps,)

    vae = type("V", (), dict(config=type("C", (), dict(block_out_channels=(1, 1, 1, 1)))()))()
    pipe = FluxPipeline(Sched(), vae, Tr())
    pe, npe = torch.full((1, 6, 8), 2.0), torch.full((1, 6, 8), -1.0)
    pool, npool = torch.full((1, 4), 0.5), torch.full((1, 4), 0.25)
    lat0 = torch.randn(1, 4, 16, generator=torch.Generator().manual_seed(1))
    kw = dict(height=32, width=32, num_inference_steps=2, latents=lat0.clone(), output_type="latent")
    plain = pipe(pe, pool, **kw).images
    assert [c[0] for c in calls] == ["cond", "cond"]
    calls.clear()
    assert torch.equal(pipe(pe, pool, negative_prompt_embeds=npe, negative_pooled_prompt_embeds=npool, true_cfg_scale=1.0, **kw).images, plain)  # scale 1: off
    assert torch.equal(pipe(pe, pool, true_cfg_scale=4.0, **kw).images, plain)                                                                   # no negatives: off
    calls.clear()
    out = pipe(pe, pool, negative_prompt_embeds=npe, negative_pooled_prompt_embeds=npool, true_cfg_scale=4.0, **kw).images
    assert [c[0] for c in calls] == ["cond", "uncond", "cond", "uncond"] and calls[0][2] is calls[1][2]  # same ids tensor: the RoPE cache holds
    x = lat0.clone()
    for _ in range(2):
        cond, neg = x * 2.0 + 0.5, x * -1.0 + 0.25
        x = x - 0.5 * (neg + 4.0 * (cond - neg))
    assert torch.allclose(out, x, rtol=1e-6, atol=1e-6)
    with pytest.raises(ValueError):
        pipe(pe, pool, negative_prompt_embeds=npe, true_cfg_scale=4.0, **kw)
