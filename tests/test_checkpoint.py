"""Reference-format checkpoints -> shells (SURVEY.md §8f N1, diffusers_b200/checkpoint.py).  CPU only: loading,
key handling and re-packing are host logic; the forward of a loaded checkpoint is checked in test_pipelines_gpu.py."""
import json
import os

import pytest
import torch

from diffusers_b200 import checkpoint, specs
from diffusers_b200.autoencoder_kl import AutoencoderKL
from diffusers_b200.pipelines import DDPMPipeline, StableDiffusionXLPipeline
from diffusers_b200.schedulers import DDPMScheduler, EulerDiscreteScheduler, FlowMatchEulerDiscreteScheduler
from diffusers_b200.transformer_flux import FluxTransformer2DModel
from diffusers_b200.unet_2d import UNet2DModel
from diffusers_b200.unet_2d_condition import UNet2DConditionModel

HERE = os.path.dirname(os.path.abspath(__file__))
FIXTURE = os.path.join(HERE, "golden", "ckpt_sdxl_micro")

MICRO_UNET = dict(sample_size=16, block_out_channels=(64, 64), down_block_types=("DownBlock2D", "CrossAttnDownBlock2D"),
                  up_block_types=("CrossAttnUpBlock2D", "UpBlock2D"), layers_per_block=1, cross_attention_dim=64,
                  transformer_layers_per_block=1, attention_head_dim=(1, 1), addition_time_embed_dim=32,
                  projection_class_embeddings_input_dim=256)
MICRO_VAE = dict(block_out_channels=(32, 32), down_block_types=("DownEncoderBlock2D",) * 2, up_block_types=("UpDecoderBlock2D",) * 2,
                 layers_per_block=1, sample_size=32)
MICRO_FLUX = dict(patch_size=1, in_channels=16, num_layers=1, num_single_layers=1, attention_head_dim=64, num_attention_heads=2,
                  joint_attention_dim=32, pooled_projection_dim=16, guidance_embeds=True, axes_dims_rope=(8, 28, 28))
MICRO_DDPM = dict(sample_size=32, in_channels=3, out_channels=3, layers_per_block=1, block_out_channels=(32, 64),
                  down_block_types=("DownBlock2D", "AttnDownBlock2D"), up_block_types=("AttnUpBlock2D", "UpBlock2D"),
                  attention_head_dim=64)

CASES = [
    ("UNet2DConditionModel", UNet2DConditionModel, specs.SDXL_UNET_CONFIG, MICRO_UNET, specs.unet2d_condition_params),
    ("AutoencoderKL", AutoencoderKL, specs.SDXL_VAE_CONFIG, MICRO_VAE, specs.vae_decoder_params),
    ("FluxTransformer2DModel", FluxTransformer2DModel, specs.FLUX_DEV_CONFIG, MICRO_FLUX, specs.flux_params),
    ("UNet2DModel", UNet2DModel, specs.DDPM_TINY_CONFIG, MICRO_DDPM, specs.unet2d_params),
]


def _write_component(root, class_name, cfg, sd, shards=1, variant=None, extra=None):
    """The reference's layout written with the stock safetensors writer (what ModelMixin.save_pretrained does)."""
    from safetensors.torch import save_file
    os.makedirs(root, exist_ok=True)
    with open(os.path.join(root, "config.json"), "w") as f:
        json.dump({"_class_name": class_name, "_diffusers_version": "0.40.0.dev0", **{k: (list(v) if isinstance(v, tuple) else v)
                                                                                          for k, v in cfg.items()}}, f)
    sd = dict(sd)
    sd.update(extra or {})
    sd = {k: v.contiguous() for k, v in sd.items()}
    if shards == 1:
        save_file(sd, os.path.join(root, checkpoint.add_variant(checkpoint.SAFETENSORS_WEIGHTS_NAME, variant)))
        return
    keys = sorted(sd)
    wm = {}
    for i in range(shards):
        part = keys[i::shards]
        name = checkpoint.add_variant(f"diffusion_pytorch_model-{i + 1:05d}-of-{shards:05d}.safetensors", variant)
        save_file({k: sd[k] for k in part}, os.path.join(root, name))
        wm.update({k: name for k in part})
    with open(os.path.join(root, checkpoint.add_variant(checkpoint.SAFETENSORS_WEIGHTS_NAME + ".index.json", variant)), "w") as f:
        json.dump({"metadata": {"total_size": 0}, "weight_map": wm}, f)


def _same_buffers(a, b):
    ba, bb = dict(a.named_buffers()), dict(b.named_buffers())
    assert ba.keys() == bb.keys() and len(ba) > 0
    for k in ba:
        assert torch.equal(ba[k], bb[k]), k


@pytest.mark.parametrize("name,cls,defaults,micro,spec_fn", CASES, ids=[c[0] for c in CASES])
def test_from_pretrained_equals_direct_construction(tmp_path, name, cls, defaults, micro, spec_fn):
    cfg = dict(defaults)
    cfg.update(micro)
    sd = specs.random_state_dict(spec_fn(cfg), seed=3, dtype=torch.bfloat16)
    direct = cls(cfg, sd, dtype=torch.bfloat16, device="cpu")
    # single file, with tensors the shell does not consume (e.g. the VAE encoder) mixed in
    _write_component(str(tmp_path / "one"), name, cfg, sd, extra={"encoder.conv_in.weight": torch.zeros(4, 3, 3, 3)})
    _same_buffers(direct, cls.from_pretrained(str(tmp_path / "one"), device="cpu"))
    # three shards + index, fp16 variant file names
    _write_component(str(tmp_path / "shards"), name, cfg, sd, shards=3, variant="fp16")
    _same_buffers(direct, cls.from_pretrained(str(tmp_path / "shards"), variant="fp16", device="cpu"))
    with pytest.raises(EnvironmentError):
        cls.from_pretrained(str(tmp_path / "shards"), device="cpu")  # the un-suffixed files are not there
    # subfolder form used by pipelines
    _write_component(str(tmp_path / "pipe" / "part"), name, cfg, sd)
    _same_buffers(direct, cls.from_pretrained(str(tmp_path / "pipe"), subfolder="part", device="cpu"))


def test_loading_errors_are_loud(tmp_path):
    cfg = dict(specs.SDXL_UNET_CONFIG)
    cfg.update(MICRO_UNET)
    sd = specs.random_state_dict(specs.unet2d_condition_params(cfg), seed=3, dtype=torch.bfloat16)
    victim = sorted(sd)[5]
    _write_component(str(tmp_path / "missing"), "UNet2DConditionModel", cfg, {k: v for k, v in sd.items() if k != victim})
    with pytest.raises(ValueError, match="lacks 1 tensors"):
        UNet2DConditionModel.from_pretrained(str(tmp_path / "missing"), device="cpu")
    _write_component(str(tmp_path / "other"), "UNet2DModel", cfg, sd)
    with pytest.raises(ValueError, match="holds a UNet2DModel"):
        UNet2DConditionModel.from_pretrained(str(tmp_path / "other"), device="cpu")
    with pytest.raises(EnvironmentError):
        UNet2DConditionModel.from_pretrained(str(tmp_path / "nowhere"), device="cpu")
    with pytest.raises(NotImplementedError):
        UNet2DConditionModel.from_pretrained(str(tmp_path / "other"), device="cpu", device_map="auto")
    bad = {k: v for k, v in sd.items()}
    bad[victim] = torch.zeros(3, 3, dtype=torch.bfloat16)
    _write_component(str(tmp_path / "shape"), "UNet2DConditionModel", cfg, bad)
    with pytest.raises(ValueError, match="expected shape"):
        UNet2DConditionModel.from_pretrained(str(tmp_path / "shape"), device="cpu")


def test_deprecated_vae_attention_names(tmp_path):
    cfg = dict(specs.SDXL_VAE_CONFIG)
    cfg.update(MICRO_VAE)
    sd = specs.random_state_dict(specs.vae_decoder_params(cfg), seed=5, dtype=torch.bfloat16)
    old = {}
    for k, v in sd.items():
        for new, dep in (("to_q", "query"), ("to_k", "key"), ("to_v", "value"), ("to_out.0", "proj_attn")):
            k = k.replace(f"attentions.0.{new}.", f"attentions.0.{dep}.")
        old[k] = v
    assert old.keys() != sd.keys()
    _write_component(str(tmp_path / "vae"), "AutoencoderKL", cfg, old)
    _same_buffers(AutoencoderKL(cfg, sd, device="cpu"), AutoencoderKL.from_pretrained(str(tmp_path / "vae"), device="cpu"))


def test_scheduler_configs(tmp_path):
    s = EulerDiscreteScheduler.from_pretrained(FIXTURE, subfolder="scheduler")  # written by the reference
    assert s.config.beta_schedule == "scaled_linear" and s.config.timestep_spacing == "leading" and s.config.steps_offset == 1
    ref = EulerDiscreteScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", timestep_spacing="leading", steps_offset=1)
    s.set_timesteps(30)
    ref.set_timesteps(30)
    assert torch.equal(s.sigmas, ref.sigmas) and torch.equal(s.timesteps, ref.timesteps)
    with open(os.path.join(FIXTURE, "scheduler", "scheduler_config.json")) as f:
        raw = json.load(f)
    os.makedirs(tmp_path / "karras")
    with open(tmp_path / "karras" / "scheduler_config.json", "w") as f:
        json.dump({**raw, "use_karras_sigmas": True}, f)
    assert EulerDiscreteScheduler.from_pretrained(str(tmp_path / "karras")).config.use_karras_sigmas is True  # "Euler Karras" is on the path
    os.makedirs(tmp_path / "beta")
    with open(tmp_path / "beta" / "scheduler_config.json", "w") as f:
        json.dump({**raw, "use_beta_sigmas": True}, f)
    with pytest.raises(NotImplementedError):  # an option outside the path must not be dropped silently
        EulerDiscreteScheduler.from_pretrained(str(tmp_path / "beta"))
    with pytest.raises(NotImplementedError):  # nor a different scheduler class be mistaken for this one
        DDPMScheduler.from_pretrained(FIXTURE, subfolder="scheduler")
    assert EulerDiscreteScheduler.from_config(s.config).config == s.config
    fm = FlowMatchEulerDiscreteScheduler.from_config(dict(shift=3.0, use_dynamic_shifting=True, base_shift=0.5, max_shift=1.15,
                                                          base_image_seq_len=256, max_image_seq_len=4096))
    assert fm.config.use_dynamic_shifting and fm.config.max_shift == 1.15


def test_published_sdxl_scheduler_config_with_legacy_keys(tmp_path):
    """The scheduler_config.json that ships with stabilityai/stable-diffusion-xl-base-1.0 (quoted here: the file is not in the
    reference tree and there is no network) still carries keys of older scheduler classes.  The reference drops keys that are
    not in the scheduler's signature with a warning (configuration_utils.py extract_init_dict); so must the shell, and the
    resulting tables must equal the ones of the explicit SDXL construction."""
    published = {"_class_name": "EulerDiscreteScheduler", "_diffusers_version": "0.19.0.dev0", "beta_end": 0.012, "beta_schedule": "scaled_linear",
                 "beta_start": 0.00085, "clip_sample": False, "interpolation_type": "linear", "num_train_timesteps": 1000,
                 "prediction_type": "epsilon", "sample_max_value": 1.0, "set_alpha_to_one": False, "skip_prk_steps": True, "steps_offset": 1,
                 "timestep_spacing": "leading", "trained_betas": None, "use_karras_sigmas": False}
    os.makedirs(tmp_path / "scheduler")
    with open(tmp_path / "scheduler" / "scheduler_config.json", "w") as f:
        json.dump(published, f)
    with pytest.warns(UserWarning, match="skip_prk_steps"):
        s = EulerDiscreteScheduler.from_pretrained(str(tmp_path), subfolder="scheduler")
    ref = EulerDiscreteScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", timestep_spacing="leading", steps_offset=1)
    s.set_timesteps(50)
    ref.set_timesteps(50)
    assert torch.equal(s.sigmas, ref.sigmas) and torch.equal(s.timesteps, ref.timesteps)
    # reference-signature options this path does not implement still fail loudly
    for bad in (dict(rescale_betas_zero_snr=True), dict(timestep_type="continuous"), dict(sigma_min=0.1)):
        with pytest.raises(NotImplementedError):
            EulerDiscreteScheduler.from_config({**published, **bad})


def test_reference_written_pipeline_directory():
    """tests/golden/ckpt_sdxl_micro was written by the reference's own StableDiffusionXLPipeline.save_pretrained
    (oracle/make_golden.py checkpoints)."""
    cls_name, comps = checkpoint.load_model_index(FIXTURE)
    assert cls_name == "StableDiffusionXLPipeline" and comps["unet"] == ("diffusers", "UNet2DConditionModel")
    assert "text_encoder" not in comps  # [null, null] slots are not components
    pipe = StableDiffusionXLPipeline.from_pretrained(FIXTURE, device="cpu")
    assert tuple(pipe.unet.config.block_out_channels) == (64, 64) and pipe.unet.config.cross_attention_dim == 64
    assert tuple(pipe.vae.config.block_out_channels) == (32, 32) and pipe.vae_scale_factor == 2
    assert pipe.unet.add_embedding.linear_1.in_features == 256
    # every tensor the shells need is in the reference's file under the name the parameter spec predicts, same shape
    for sub, spec in (("unet", specs.unet2d_condition_params(dict(pipe.unet.config))), ("vae", specs.vae_decoder_params(dict(pipe.vae.config)))):
        sd = checkpoint.load_state_dict(os.path.join(FIXTURE, sub))
        assert all(k in sd and tuple(sd[k].shape) == tuple(shp) for k, shp in spec.items())
        assert all(v.dtype == torch.bfloat16 for v in sd.values())
    with pytest.raises(ValueError, match="not DDPMPipeline"):
        DDPMPipeline.from_pretrained(FIXTURE, device="cpu")


def _write_recorded(root, files, sd):
    """Re-creates a directory the reference's save_pretrained wrote (tests/golden/reference_api.json.gz): its JSON files
    verbatim, each safetensors file with the recorded metadata and the recorded tensor names / dtypes / shapes, valued from sd."""
    from safetensors.torch import save_file
    for rel, content in files.items():
        p = os.path.join(root, rel)
        os.makedirs(os.path.dirname(p), exist_ok=True)
        if rel.endswith(".json"):
            with open(p, "w") as f:
                json.dump(content, f)
        else:
            tensors = {}
            for k, (dtype, shape) in content["tensors"].items():
                assert str(sd[k].dtype) == dtype and tuple(sd[k].shape) == tuple(shape), k
                tensors[k] = sd[k].contiguous()
            save_file(tensors, p, metadata=content["metadata"])


def test_reference_save_pretrained_round_trip(tmp_path, reference_api):
    """The real writer: reference model -> save_pretrained -> shell.from_pretrained == shell(state_dict)."""
    rec = reference_api["save_pretrained"]
    cfg = dict(specs.DDPM_TINY_CONFIG)
    cfg.update(MICRO_DDPM)
    assert json.loads(json.dumps(cfg)) == rec["cfg"]
    sd = specs.random_state_dict(specs.unet2d_params(cfg), seed=0, dtype=torch.bfloat16)
    for k in ("u", "v", "p"):
        _write_recorded(str(tmp_path / k), rec["dirs"][k], sd)
    assert os.path.isfile(tmp_path / "u" / "diffusion_pytorch_model.safetensors.index.json")  # max_shard_size="300KB": sharded layout
    ours = UNet2DModel.from_pretrained(str(tmp_path / "u"), device="cpu")
    _same_buffers(UNet2DModel(cfg, sd, device="cpu"), ours)
    _same_buffers(ours, UNet2DModel.from_pretrained(str(tmp_path / "v"), variant="fp16", device="cpu"))
    p = DDPMPipeline.from_pretrained(str(tmp_path / "p"), device="cpu")
    _same_buffers(ours, p.unet)
    assert isinstance(p.scheduler, DDPMScheduler) and p.scheduler.config.num_train_timesteps == 1000


@pytest.mark.parametrize("name,cls,defaults,micro,spec_fn", CASES, ids=[c[0] for c in CASES])
def test_reference_state_dict_is_the_exact_inverse_of_packing(tmp_path, name, cls, defaults, micro, spec_fn):
    """Every shell can rebuild the reference's parameters (names, shapes, values) from its packed buffers, bit for bit."""
    cfg = dict(defaults)
    cfg.update(micro)
    spec = spec_fn(cfg)
    sd = specs.random_state_dict(spec, seed=7, dtype=torch.bfloat16)
    # (the UNet's default folds its LayerNorms into the GEMM weights, which re-rounds them once: fold_norms=False is the
    # bit-exact mode; the folded mode's round trip is bounded in tests/test_host_logic.py)
    exact = dict(fold_norms=False) if name == "UNet2DConditionModel" else {}
    m = cls(cfg, sd, dtype=torch.bfloat16, device="cpu", **exact)
    back = m.reference_state_dict()
    assert list(back) == list(spec)
    for k, v in sd.items():
        assert back[k].dtype == torch.bfloat16 and tuple(back[k].shape) == tuple(spec[k]) and torch.equal(back[k], v), k
    if name == "AutoencoderKL":
        with pytest.raises(NotImplementedError):  # only the decoder half is held
            m.save_pretrained(str(tmp_path / "vae"))
        return
    m.save_pretrained(str(tmp_path / "m"))
    raw = checkpoint.load_config(str(tmp_path / "m"))
    assert raw["_class_name"] == name
    _same_buffers(m, cls.from_pretrained(str(tmp_path / "m"), device="cpu", **exact))
    m.save_pretrained(str(tmp_path / "v"), variant="fp16")
    assert os.path.isfile(tmp_path / "v" / "diffusion_pytorch_model.fp16.safetensors")


def test_unet_conv_projection_and_multi_layer_round_trip():
    """SD-1.x style conv 1x1 proj_in / proj_out come back 4-D; several transformer layers / three levels keep their offsets."""
    for upd in (dict(MICRO_UNET, use_linear_projection=False),
                dict(sample_size=16, block_out_channels=(64, 128, 256), cross_attention_dim=128, transformer_layers_per_block=(1, 2, 3),
                     attention_head_dim=(1, 2, 4), addition_time_embed_dim=32, projection_class_embeddings_input_dim=256)):
        cfg = dict(specs.SDXL_UNET_CONFIG)
        cfg.update(upd)
        spec = specs.unet2d_condition_params(cfg)
        sd = specs.random_state_dict(spec, seed=9, dtype=torch.bfloat16)
        back = UNet2DConditionModel(cfg, sd, device="cpu", fold_norms=False).reference_state_dict()
        assert all(torch.equal(back[k], sd[k]) for k in sd)
        if not cfg["use_linear_projection"]:
            assert back["mid_block.attentions.0.proj_in.weight"].dim() == 4


def _reference_loads(path, rec, sd):
    """What the reference's from_pretrained (recorded in tests/golden/reference_api.json.gz) reports for the same model: no
    missing / unexpected / mismatched keys, and its state_dict names and shapes are exactly those of the saved file, which
    holds sd's values."""
    assert not any(rec["info"].values()), rec["info"]
    saved = checkpoint.load_state_dict(path)
    assert {k: tuple(v.shape) for k, v in saved.items()} == {k: tuple(s) for k, s in rec["state_dict"].items()}
    assert all(torch.equal(saved[k], sd[k]) for k in sd)


def test_unmodified_reference_loads_what_the_shells_save(tmp_path, reference_api):
    """shell.save_pretrained -> the reference's own from_pretrained: same parameters, no missing / unexpected keys."""
    for name, cls, defaults, micro, spec_fn in CASES:
        if name == "AutoencoderKL":
            continue
        cfg = dict(defaults)
        cfg.update(micro)
        rec = reference_api["loaded"][name]
        assert json.loads(json.dumps(cfg)) == rec["cfg"]
        sd = specs.random_state_dict(spec_fn(cfg), seed=11, dtype=torch.bfloat16)
        exact = dict(fold_norms=False) if name == "UNet2DConditionModel" else {}
        cls(cfg, sd, device="cpu", **exact).save_pretrained(str(tmp_path / name))
        _reference_loads(str(tmp_path / name), rec, sd)


@pytest.mark.parametrize("kind", ["clip", "clip_proj", "t5"])
def test_text_encoder_shells_load_transformers_checkpoints(tmp_path, kind):
    """N1 x N3: `text_encoder/` directories written by the real transformers `save_pretrained` (config.json with `architectures`,
    model.safetensors) load into the shells: same config, same tensors (checked on the unpacked embedding / norm buffers and,
    through the packing inverse, on a projection weight).  Construction is host-side; no GPU involved."""
    import transformers
    from diffusers_b200 import packing
    from diffusers_b200 import text_encoders as T
    torch.manual_seed(0)
    if kind == "t5":
        hf = transformers.T5EncoderModel(transformers.T5Config(vocab_size=300, d_model=128, d_kv=64, d_ff=256, num_layers=2, num_heads=2,
                                                               feed_forward_proj="gated-gelu"))
        cls = T.T5EncoderModel
    else:
        cfg = transformers.CLIPTextConfig(vocab_size=300, hidden_size=128, intermediate_size=256, num_hidden_layers=2, num_attention_heads=2,
                                          hidden_act="quick_gelu" if kind == "clip" else "gelu", projection_dim=64)
        hf = (transformers.CLIPTextModel if kind == "clip" else transformers.CLIPTextModelWithProjection)(cfg)
        cls = T.CLIPTextModel if kind == "clip" else T.CLIPTextModelWithProjection
    d = tmp_path / "text_encoder"
    hf.save_pretrained(d, safe_serialization=True)
    m = cls.from_pretrained(str(tmp_path), subfolder="text_encoder", torch_dtype=torch.bfloat16, device="cpu")
    sd = hf.state_dict()
    if kind == "t5":
        assert m.config.d_model == 128 and m.config.num_layers == 2 and m.config.feed_forward_proj == "gated-gelu"
        assert torch.equal(m.W(m.tok), sd["shared.weight"].bfloat16())
        assert torch.equal(m.W(m.blocks[1]["n2"]), sd["encoder.block.1.layer.1.layer_norm.weight"].bfloat16())
        assert torch.equal(packing.unpack_linear_weight(m.W(m.blocks[0]["o"]), 128), sd["encoder.block.0.layer.0.SelfAttention.o.weight"].bfloat16())
    else:
        assert m.config.hidden_size == 128 and m.config.hidden_act == ("quick_gelu" if kind == "clip" else "gelu") and m.config.eos_token_id == hf.config.eos_token_id
        assert torch.equal(m.W(m.tok), sd["text_model.embeddings.token_embedding.weight"].bfloat16())
        assert torch.equal(packing.unpack_linear_weight(m.W(m.layers[1]["f2w"]), 256), sd["text_model.encoder.layers.1.mlp.fc2.weight"].bfloat16())
        if kind == "clip_proj":
            assert torch.equal(m.W(m.proj), sd["text_projection.weight"].bfloat16())
    with pytest.raises(ValueError):
        (T.T5EncoderModel if kind != "t5" else T.CLIPTextModel).from_pretrained(str(tmp_path), subfolder="text_encoder", device="cpu")


def test_whole_vae_checkpoint_round_trip(tmp_path, reference_api):
    """With the encoder half loaded (N3) the AutoencoderKL shell holds the reference's complete state_dict: reference_state_dict()
    is the exact inverse of the packing for encoder.* / quant_conv.* too, save_pretrained writes a directory that from_pretrained
    reads back WITH the encoder - and that the unmodified reference loads without missing / unexpected keys."""
    cfg = dict(specs.SDXL_VAE_CONFIG)
    cfg.update(MICRO_VAE)
    spec = specs.vae_params(cfg)
    sd = specs.random_state_dict(spec, seed=13, dtype=torch.bfloat16)
    m = AutoencoderKL(cfg, sd, dtype=torch.bfloat16, device="cpu")
    assert m.enc is not None
    back = m.reference_state_dict()
    assert sorted(back) == sorted(spec)
    for k, v in sd.items():
        assert tuple(back[k].shape) == tuple(spec[k]) and torch.equal(back[k], v), k
    m.save_pretrained(str(tmp_path / "vae"))
    again = AutoencoderKL.from_pretrained(str(tmp_path / "vae"), device="cpu")
    assert again.enc is not None
    _same_buffers(m, again)
    # a checkpoint that lacks part of the encoder is an error, not a silent decoder-only model
    with pytest.raises(ValueError):
        AutoencoderKL(cfg, {k: v for k, v in sd.items() if k != "encoder.conv_out.bias"}, device="cpu")
    _reference_loads(str(tmp_path / "vae"), reference_api["loaded"]["AutoencoderKL"], sd)
