"""ORACLE (test infrastructure): functional CPU restatement of the reference's UNet wiring and training-step glue.

Follows, line for line in meaning (not in code), the reference files
  models/unet_3d_condition.py:325-500   UNet3DConditionModel.forward
  models/unet_3d_blocks.py:368-419,517-569,632-652,746-798,856-875   the five block forwards
  train.py:339-358,739-834              tensor_to_vae_latent / sample_noise / add_noise / epsilon MSE loss
on top of the leaf restatements in oracle/leaves.py.  It consumes a plain state dict keyed by the diffusers
parameter names (SURVEY.md appendix C), so it also checks the product's parameter naming.

PARITY UNPINNED by the reference's own tests (there are none).  Pinned here by
tests/test_oracle_vs_reference.py: this function must reproduce the outputs that the reference's models/*.py, imported
UNMODIFIED (over oracle/diffusers_standin), gave on the same state dict (tests/golden/oracle_vs_reference.pt).
"""
import torch
import torch.nn.functional as F

from . import leaves as L

DEFAULT_CONFIG = dict(  # == ctor defaults at models/unet_3d_condition.py:86-107 (ms-1.7b / zeroscope_v2_576w)
    sample_size=None,
    in_channels=4,
    out_channels=4,
    down_block_types=("CrossAttnDownBlock3D", "CrossAttnDownBlock3D", "CrossAttnDownBlock3D", "DownBlock3D"),
    up_block_types=("UpBlock3D", "CrossAttnUpBlock3D", "CrossAttnUpBlock3D", "CrossAttnUpBlock3D"),
    block_out_channels=(320, 640, 1280, 1280),
    layers_per_block=2,
    downsample_padding=1,
    mid_block_scale_factor=1,
    act_fn="silu",
    norm_num_groups=32,
    norm_eps=1e-5,
    cross_attention_dim=1024,
    attention_head_dim=64,
)


def full_config(**overrides):
    cfg = dict(DEFAULT_CONFIG)
    cfg.update(overrides)
    return cfg


def _head_dims(cfg):
    ahd = cfg["attention_head_dim"]
    n = len(cfg["down_block_types"])
    return (ahd,) * n if isinstance(ahd, int) else tuple(ahd)


def unet3d_forward(p, cfg, sample, timestep, encoder_hidden_states):
    """(B, C, F, H, W) noisy latents, (B,) timesteps, (B, 77, ctx) text states -> (B, C, F, H, W) prediction."""
    boc = tuple(cfg["block_out_channels"])
    groups, eps = cfg["norm_num_groups"], cfg["norm_eps"]
    lpb = cfg["layers_per_block"]
    hd = _head_dims(cfg)
    B, _, nf, _, _ = sample.shape
    dtype = p["conv_in.weight"].dtype

    # unet_3d_condition.py:359-367 - forward explicit upsample sizes when H/W are not multiples of 2**num_upsamplers
    n_up = len(cfg["up_block_types"]) - 1
    forward_upsample_size = any(s % (2 ** n_up) != 0 for s in sample.shape[-2:])

    # 1. time (unet_3d_condition.py:375-401)
    if not torch.is_tensor(timestep):
        timestep = torch.tensor([timestep], dtype=torch.int64)
    timesteps = timestep.reshape(-1).expand(B)
    t_emb = L.timestep_sinusoid(timesteps, boc[0]).to(dtype)
    emb = L.timestep_embedding(p, "time_embedding.", t_emb)
    emb = emb.repeat_interleave(nf, dim=0)
    ctx = encoder_hidden_states.to(dtype).repeat_interleave(nf, dim=0)

    # 2. pre-process (:404-411)
    x = sample.to(dtype).permute(0, 2, 1, 3, 4).reshape((B * nf, -1) + tuple(sample.shape[3:]))
    x = F.conv2d(x, p["conv_in.weight"], p["conv_in.bias"], padding=1)
    if nf > 1:
        x = L.transformer_temporal(p, "transformer_in.", x, nf, heads=8, groups=groups)

    # 3. down (:414-428; blocks at unet_3d_blocks.py:517-569 / 632-652)
    skips = [x]
    for i, typ in enumerate(cfg["down_block_types"]):
        pre = f"down_blocks.{i}."
        heads = boc[i] // hd[i]
        for j in range(lpb):
            x = L.resnet_block2d(p, f"{pre}resnets.{j}.", x, emb, groups, eps)
            if nf > 1:
                x = L.temporal_conv_layer(p, f"{pre}temp_convs.{j}.", x, nf)
            if typ == "CrossAttnDownBlock3D":
                x = L.transformer2d(p, f"{pre}attentions.{j}.", x, ctx, heads, groups)
                if nf > 1:
                    x = L.transformer_temporal(p, f"{pre}temp_attentions.{j}.", x, nf, heads, groups)
            skips.append(x)
        if i != len(boc) - 1:
            x = L.downsample2d(p, f"{pre}downsamplers.0.", x, padding=cfg["downsample_padding"])
            skips.append(x)

    # 4. mid (:442-450; unet_3d_blocks.py:368-419)
    heads = boc[-1] // hd[-1]
    msf = cfg["mid_block_scale_factor"]
    x = L.resnet_block2d(p, "mid_block.resnets.0.", x, emb, groups, eps, msf)
    if True:  # the reference applies temp_convs[0] unconditionally in the mid block (unet_3d_blocks.py:386-387)
        x = L.temporal_conv_layer(p, "mid_block.temp_convs.0.", x, nf)
    x = L.transformer2d(p, "mid_block.attentions.0.", x, ctx, heads, groups)
    if nf > 1:
        x = L.transformer_temporal(p, "mid_block.temp_attentions.0.", x, nf, heads, groups)
    x = L.resnet_block2d(p, "mid_block.resnets.1.", x, emb, groups, eps, msf)
    if nf > 1:
        x = L.temporal_conv_layer(p, "mid_block.temp_convs.1.", x, nf)

    # 5. up (:456-485; unet_3d_blocks.py:746-798 / 856-875)
    rev_hd = tuple(reversed(hd))
    rev_boc = tuple(reversed(boc))
    for i, typ in enumerate(cfg["up_block_types"]):
        pre = f"up_blocks.{i}."
        heads = rev_boc[i] // rev_hd[i]
        res, skips = skips[-(lpb + 1):], skips[:-(lpb + 1)]
        is_final = i == len(boc) - 1
        upsample_size = tuple(skips[-1].shape[2:]) if (not is_final and forward_upsample_size) else None
        for j in range(lpb + 1):
            x = torch.cat([x, res[-1 - j]], dim=1)
            x = L.resnet_block2d(p, f"{pre}resnets.{j}.", x, emb, groups, eps)
            if nf > 1:
                x = L.temporal_conv_layer(p, f"{pre}temp_convs.{j}.", x, nf)
            if typ == "CrossAttnUpBlock3D":
                x = L.transformer2d(p, f"{pre}attentions.{j}.", x, ctx, heads, groups)
                if nf > 1:
                    x = L.transformer_temporal(p, f"{pre}temp_attentions.{j}.", x, nf, heads, groups)
        if not is_final:
            x = L.upsample2d(p, f"{pre}upsamplers.0.", x, upsample_size)

    # 6. post-process (:488-495)
    x = F.group_norm(x, groups, p["conv_norm_out.weight"], p["conv_norm_out.bias"], eps)
    x = F.conv2d(F.silu(x), p["conv_out.weight"], p["conv_out.bias"], padding=1)
    return x[None, :].reshape((-1, nf) + tuple(x.shape[1:])).permute(0, 2, 1, 3, 4)


def finetune_loss(p, cfg, latents, noise, timesteps, encoder_hidden_states, alphas_cumprod=None):
    """train.py:751-834 for prediction_type 'epsilon', one UNet pass: add_noise -> UNet -> F.mse_loss in fp32."""
    if alphas_cumprod is None:
        alphas_cumprod = L.ddpm_alphas_cumprod()
    noisy = L.add_noise(latents, noise, timesteps, alphas_cumprod)
    pred = unet3d_forward(p, cfg, noisy, timesteps, encoder_hidden_states)
    loss = F.mse_loss(pred.float(), noise.float(), reduction="mean")
    return loss, pred


def tensor_to_vae_latent(p_vae, pixels, eps_noise, block_out_channels=(128, 256, 512, 512), layers_per_block=2):
    """train.py:339-347: (B, F, 3, H, W) pixels -> (B, 4, F, H/8, W/8) latents * 0.18215 (hard-coded, H9)."""
    B, nf = pixels.shape[:2]
    flat = pixels.reshape((B * nf,) + tuple(pixels.shape[2:]))
    lat = L.diagonal_gaussian_sample(L.vae_encode_moments(p_vae, flat, block_out_channels, layers_per_block), eps_noise)
    lat = lat.reshape((B, nf) + tuple(lat.shape[1:])).permute(0, 2, 1, 3, 4)
    return lat * 0.18215
