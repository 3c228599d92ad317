"""Generates tests/golden/lora_module_*.pt and lora_unet_small_f4.pt from the REFERENCE's own LoRA code: its utils/lora.py
imported unmodified (LoraInjectedLinear / Conv2d / Conv3d, inject_trainable_lora_extended) and, for the model-level case, the
reference's unmodified models/*.py over oracle/diffusers_standin.  fp32, CPU.  Needs a checkout of the reference:
    T2V_REFERENCE_ROOT=<reference checkout> python tests/golden/make_golden_lora.py
The fixtures pin the B200 LoRA path (tests/test_lora_gpu.py) to the reference classes rather than to this repo's own wiring."""
import contextlib
import importlib.util
import io
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from helpers import seeded_state_dict  # noqa: E402
from oracle import leaves as L  # noqa: E402
from oracle.reference_import import REFERENCE_ROOT, import_reference_unet  # noqa: E402

SMALL = dict(block_out_channels=(64, 128, 128, 128), attention_head_dim=64, cross_attention_dim=64)


def ref_lora():
    spec = importlib.util.spec_from_file_location("_t2v_ref_lora", os.path.join(REFERENCE_ROOT, "utils", "lora.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def seed_lora_(module, seed):
    """Deterministic non-trivial LoRA weights (lora_up is zero-initialised in the reference, utils/lora.py:54-55)."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in sorted(module.named_parameters()):
            if "lora_up" in n:
                p.copy_(torch.randn(p.shape, generator=g) * 0.05)
            elif "lora_down" in n:
                p.copy_(torch.randn(p.shape, generator=g) / p[0].numel() ** 0.5)


def module_cases(ref):
    g = torch.Generator().manual_seed(100)
    out = {}
    specs = {
        "linear": (lambda: ref.LoraInjectedLinear(128, 256, bias=True, r=16, dropout_p=0.1, scale=1.0), (2, 77, 128)),
        "linear_nobias_r4": (lambda: ref.LoraInjectedLinear(64, 96, bias=False, r=4, dropout_p=0.1, scale=0.5), (3, 40, 64)),
        "conv2d": (lambda: ref.LoraInjectedConv2d(32, 64, 3, 1, 1, bias=True, r=16, dropout_p=0.1, scale=1.0), (2, 32, 16, 16)),
        "conv2d_s2": (lambda: ref.LoraInjectedConv2d(32, 32, 3, 2, 1, bias=True, r=8, dropout_p=0.1, scale=1.0), (2, 32, 16, 16)),
        "conv3d": (lambda: ref.LoraInjectedConv3d(32, 32, (3, 1, 1), (1, 0, 0), bias=True, r=16, dropout_p=0.1, scale=1.0), (1, 32, 4, 8, 8)),
    }
    for name, (ctor, xshape) in specs.items():
        torch.manual_seed(7)
        m = ctor().eval()   # eval: the wrapper's dropout is the identity (its mask is a torch RNG draw, not reproducible elsewhere)
        with torch.no_grad():
            for n, p in sorted(m.named_parameters()):
                p.copy_(torch.randn(p.shape, generator=g) * (0.05 if "lora_up" in n else 1.0 / max(1, p[0].numel()) ** 0.5))
        x = torch.randn(xshape, generator=g, requires_grad=True)
        y = m(x)
        dy = torch.randn(y.shape, generator=g)
        y.backward(dy)
        out[name] = dict(state={k: v.detach().clone() for k, v in m.state_dict().items()}, x=x.detach().clone(), y=y.detach().clone(), dy=dy,
                         dx=x.grad.clone(), grads={n: p.grad.clone() for n, p in m.named_parameters() if "lora" in n and p.grad is not None},
                         scale=m.scale, r=m.lora_down.weight.shape[0])
    return out


def model_case(ref):
    Ref = import_reference_unet()
    m = Ref(**SMALL)
    sd = seeded_state_dict(m, 0)
    m.load_state_dict(sd)
    m.requires_grad_(False)
    with contextlib.redirect_stdout(io.StringIO()):
        ref.inject_trainable_lora_extended(m, {"UNet3DConditionModel"}, r=8)
    seed_lora_(m, 11)
    m.eval()
    g = torch.Generator().manual_seed(3)
    lat = torch.randn(1, 4, 4, 16, 16, generator=g)
    noise = torch.randn(1, 4, 4, 16, 16, generator=g)
    t = torch.tensor([437])
    ehs = torch.randn(1, 7, 64, generator=g)
    noisy = L.add_noise(lat, noise, t, L.ddpm_alphas_cumprod())
    pred = m(noisy, t, encoder_hidden_states=ehs).sample
    loss = torch.nn.functional.mse_loss(pred.float(), noise.float())
    loss.backward()
    grads = {n: p.grad for n, p in m.named_parameters() if "lora" in n and p.grad is not None}
    keep = sorted(grads, key=lambda n: -grads[n].norm().item())[:24]
    return dict(cfg=SMALL, r=8, lora_seed=11, base_seed=0, latents=lat, noise=noise, timesteps=t, text=ehs, pred=pred.detach(), loss=loss.detach(),
                grad_norms={n: v.norm().item() for n, v in grads.items()}, grads={n: grads[n].detach().clone() for n in keep},
                n_lora=len(grads), source="reference utils/lora.py (inject_trainable_lora_extended, LoraInjected*) on the reference's "
                                          "models/*.py over oracle/diffusers_standin, fp32 CPU")


def main():
    torch.set_num_threads(8)
    ref = ref_lora()
    for name, case in module_cases(ref).items():   # one file per case keeps each fixture small
        path = os.path.join(ROOT, "tests", "golden", f"lora_module_{name}.pt")
        torch.save(case, path)
        print("lora_module_" + name, os.path.getsize(path) // 1024, "KiB")
    path = os.path.join(ROOT, "tests", "golden", "lora_unet_small_f4.pt")
    torch.save(model_case(ref), path)
    print("lora_unet_small_f4", os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
