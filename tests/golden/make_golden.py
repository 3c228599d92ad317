"""Generates tests/golden/unet_small_*.pt from the REFERENCE's own wiring: its models/*.py imported
unmodified (over oracle/diffusers_standin, since diffusers is not installed), fp32, CPU.  Needs a checkout of the reference:
    T2V_REFERENCE_ROOT=<reference checkout> python tests/golden/make_golden.py
The fixtures pin (a) the oracle restatement (tests/test_golden.py, CPU) and (b) the CUDA path (GPU) to the reference."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from helpers import seeded_state_dict  # noqa: E402
from oracle import leaves as L  # noqa: E402
from oracle.reference_import import import_reference_unet  # noqa: E402

CASES = {
    "unet_small_f4": dict(cfg=dict(block_out_channels=(32, 64, 64, 64), attention_head_dim=32, cross_attention_dim=32),
                          B=1, F=4, hw=(16, 16), ctx=5, seed=11),
    "unet_small_f1": dict(cfg=dict(block_out_channels=(32, 64, 64, 64), attention_head_dim=32, cross_attention_dim=32),
                          B=2, F=1, hw=(16, 16), ctx=3, seed=12),
    # one layer per block, non-square map, odd frame count, two heads at the top levels / four below
    # (a per-level attention_head_dim tuple is NOT a case: the reference passes it unsplit to transformer_in and fails)
    "unet_one_layer_f3": dict(cfg=dict(block_out_channels=(64, 64, 128, 128), attention_head_dim=32, cross_attention_dim=48,
                                       layers_per_block=1),
                              B=1, F=3, hw=(8, 24), ctx=9, seed=13),
    # non-default block layout: attention and plain blocks interleaved
    "unet_mixed_blocks_f2": dict(cfg=dict(block_out_channels=(32, 64, 64, 64), attention_head_dim=32, cross_attention_dim=32,
                                          down_block_types=("CrossAttnDownBlock3D", "DownBlock3D", "CrossAttnDownBlock3D", "DownBlock3D"),
                                          up_block_types=("UpBlock3D", "CrossAttnUpBlock3D", "UpBlock3D", "CrossAttnUpBlock3D")),
                                 B=2, F=2, hw=(16, 16), ctx=4, seed=14),
}
ONLY = [a for a in sys.argv[1:] if not a.startswith("-")]   # python make_golden.py [case ...]: regenerate a subset
KEEP_FULL = ["conv_in.weight", "down_blocks.0.resnets.0.conv1.weight", "down_blocks.0.temp_convs.0.conv1.2.weight",
             "down_blocks.1.attentions.0.transformer_blocks.0.attn2.to_k.weight", "mid_block.resnets.0.time_emb_proj.weight",
             "up_blocks.1.temp_attentions.0.transformer_blocks.0.ff.net.0.proj.weight", "up_blocks.3.resnets.2.conv_shortcut.weight",
             "conv_norm_out.weight", "conv_out.bias", "time_embedding.linear_1.weight"]


def main():
    torch.set_num_threads(8)
    Ref = import_reference_unet()
    for name, c in CASES.items():
        if ONLY and name not in ONLY:
            continue
        m = Ref(**c["cfg"]).eval()
        sd = seeded_state_dict(m, c["seed"])
        m.load_state_dict(sd)
        g = torch.Generator().manual_seed(c["seed"] + 1)
        lat = torch.randn(c["B"], 4, c["F"], *c["hw"], generator=g)
        noise = torch.randn(c["B"], 4, c["F"], *c["hw"], generator=g)
        t = torch.randint(0, 1000, (c["B"],), generator=g)
        ehs = torch.randn(c["B"], c["ctx"], c["cfg"]["cross_attention_dim"], generator=g)
        abar = L.ddpm_alphas_cumprod()
        noisy = L.add_noise(lat, noise, t, abar)                       # train.py:760
        pred = m(noisy, t, encoder_hidden_states=ehs).sample           # train.py:826
        loss = torch.nn.functional.mse_loss(pred.float(), noise.float(), reduction="mean")  # train.py:827
        loss.backward()
        grads = {n: p.grad for n, p in m.named_parameters()}
        out = dict(cfg=c["cfg"], seed=c["seed"], latents=lat, noise=noise, timesteps=t, text=ehs, pred=pred.detach(),
                   loss=loss.detach(), grad_norms={n: g_.norm().item() if g_ is not None else None for n, g_ in grads.items()},
                   grads={n: grads[n].detach().clone() for n in KEEP_FULL if grads.get(n) is not None and grads[n].numel() < 40000},
                   source="reference models/unet_3d_condition.py + models/unet_3d_blocks.py (unmodified) over oracle/diffusers_standin (plain nn.Modules on torch operators, independent of oracle/leaves.py), fp32 CPU")
        path = os.path.join(ROOT, "tests", "golden", name + ".pt")
        torch.save(out, path)
        print(name, "loss", loss.item(), os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
