"""diffusers_b200.specs restates the reference constructors' parameter inventory; this checks every name and shape against
the UNMODIFIED reference's own modules built on the meta device, at the BASELINE.json sizes, as recorded by
oracle/make_golden.py (gen_reference_api) in tests/golden/reference_api.json.gz."""
import pytest
import torch

from diffusers_b200 import specs


def _compare(spec, inventory, prefix_filter=None):
    ref = {k: tuple(v) for k, v in inventory.items() if prefix_filter is None or prefix_filter(k)}
    ours = {k: tuple(v) for k, v in spec.items()}
    assert sorted(ours) == sorted(ref), (sorted(set(ours) - set(ref))[:5], sorted(set(ref) - set(ours))[:5])
    bad = [(k, ours[k], ref[k]) for k in ours if ours[k] != ref[k]]
    assert not bad, bad[:5]
    return len(ours)


def test_sdxl_unet_names_and_shapes(reference_api):
    n = _compare(specs.unet2d_condition_params(specs.SDXL_UNET_CONFIG), reference_api["inventories"]["sdxl_unet"])
    assert n == 1680  # stabilityai/stable-diffusion-xl-base-1.0 unet: 1680 tensors, 2.57 B parameters


def test_sdxl_vae_decoder_names_and_shapes(reference_api):
    _compare(specs.vae_decoder_params(specs.SDXL_VAE_CONFIG), reference_api["inventories"]["sdxl_vae"],
             lambda k: k.startswith(("decoder.", "post_quant_conv.")))


def test_flux_dev_names_and_shapes(reference_api):
    _compare(specs.flux_params(specs.FLUX_DEV_CONFIG), reference_api["inventories"]["flux_dev"])


def test_ddpm_unet2d_names_and_shapes(reference_api):
    _compare(specs.unet2d_params(specs.DDPM_TINY_CONFIG), reference_api["inventories"]["ddpm_tiny"])


def test_sdxl_vae_whole_checkpoint_names_and_shapes(reference_api):
    """encoder + quant_conv + post_quant_conv + decoder = the reference's whole AutoencoderKL state_dict (N3: encode)."""
    n = _compare(specs.vae_params(specs.SDXL_VAE_CONFIG), reference_api["inventories"]["sdxl_vae"])
    assert n == 248  # madebyollin/sdxl-vae-fp16-fix, stabilityai/sdxl-vae: 248 tensors


@pytest.mark.parametrize("which", ["clip_l", "openclip_bigg", "t5_xxl"])
def test_text_encoder_names_and_shapes_match_transformers(which):
    """The text encoders' parameter inventory against the real transformers classes (the third-party dependency the reference's
    pipelines call) on the meta device, at the SDXL / Flux sizes."""
    import transformers
    from diffusers_b200 import text_encoders as T
    if which == "t5_xxl":
        spec = T.t5_encoder_params(T.T5_XXL_CONFIG)
        with torch.device("meta"):
            m = transformers.T5EncoderModel(transformers.T5Config(**T.T5_XXL_CONFIG))
        ref = {k: tuple(v.shape) for k, v in m.state_dict().items() if k != "encoder.embed_tokens.weight"}  # tied to shared.weight
        assert sum(v.numel() for k, v in m.state_dict().items() if k != "encoder.embed_tokens.weight") == 4_762_310_656  # google/t5-v1_1-xxl encoder
    else:
        cfg = T.CLIP_L_CONFIG if which == "clip_l" else T.CLIP_BIGG_CONFIG
        proj = which == "openclip_bigg"
        spec = T.clip_text_params(cfg, proj)
        with torch.device("meta"):
            m = (transformers.CLIPTextModelWithProjection if proj else transformers.CLIPTextModel)(transformers.CLIPTextConfig(**cfg))
        ref = {k: tuple(v.shape) for k, v in m.state_dict().items() if "position_ids" not in k}
    ours = {k: tuple(v) for k, v in spec.items()}
    assert sorted(ours) == sorted(ref), (sorted(set(ours) - set(ref))[:5], sorted(set(ref) - set(ours))[:5])
    assert not [(k, ours[k], ref[k]) for k in ours if ours[k] != ref[k]]
