"""Generates the reference fixtures that tests/test_oracle_vs_reference.py, tests/test_lora_cpu.py and
tests/test_pipeline_train.py compare against, from the reference's own files imported unmodified (models/*.py over
oracle/diffusers_standin, utils/lora.py, configs/v2/*.yaml).  fp32, CPU.  Needs a checkout of the reference:
    T2V_REFERENCE_ROOT=<reference checkout> python tests/golden/make_golden_reference.py

  oracle_vs_reference.pt     UNet outputs on seeded weights (plain and with gradient checkpointing) and the parameter
                             keys / shapes of the full-size model
  lora_reference.pt          the injector's census on a small UNet and LoraInjected* outputs on seeded weights
  reference_configs.json     for each v2 YAML: its top-level keys, dataset_types and train_data section
Weights and inputs are drawn with tests/helpers.py::seeded_state_dict and seeded generators, so the tests rebuild them
without the reference."""
import contextlib
import importlib.util
import io
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from helpers import seeded_state_dict  # noqa: E402
from oracle.reference_import import REFERENCE_ROOT, import_reference_unet  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
UNET_SMALL = dict(block_out_channels=(64, 128, 128, 128), attention_head_dim=32, cross_attention_dim=64)
LORA_SMALL = dict(block_out_channels=(64, 128, 128, 128), attention_head_dim=64, cross_attention_dim=64)
WIRING_CASES = [(4, 16), (1, 8), (3, 12)]
CONV4_STD = 0.05


def ref_lora():
    spec = importlib.util.spec_from_file_location("_t2v_ref_lora", os.path.join(REFERENCE_ROOT, "utils", "lora.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def unet_fixture():
    Ref = import_reference_unet()
    m = Ref(**UNET_SMALL).eval()
    m.load_state_dict(seeded_state_dict(m, 0, conv4_std=CONV4_STD))
    out = dict(cfg=UNET_SMALL, weight_seed=0, conv4_std=CONV4_STD, wiring={})
    g = torch.Generator().manual_seed(1)
    for frames, hw in WIRING_CASES:
        x = torch.randn(2, 4, frames, hw, hw, generator=g)
        t = torch.tensor([500, 3])
        ehs = torch.randn(2, 7, 64, generator=g)
        with torch.no_grad():
            y = m(x, t, ehs).sample
        out["wiring"][f"{frames}x{hw}"] = dict(x=x, t=t, ehs=ehs, y=y)
    g = torch.Generator().manual_seed(2)
    x, t, ehs = torch.randn(1, 4, 2, 8, 8, generator=g), torch.tensor([10]), torch.randn(1, 7, 64, generator=g)
    with torch.no_grad():
        plain = m(x, t, ehs).sample
    m._set_gradient_checkpointing(True)
    ckpt = m(x, t, ehs).sample.detach()
    assert torch.equal(plain, ckpt)
    out["checkpointed"] = dict(x=x, t=t, ehs=ehs, y_plain=plain, y_checkpointed=ckpt)
    with torch.device("meta"):
        full = Ref()
    out["full_size_shapes"] = [(k, tuple(v.shape)) for k, v in full.state_dict().items()]
    return out


def lora_fixture(ref):
    m = import_reference_unet()(**LORA_SMALL)
    m.load_state_dict(seeded_state_dict(m, 0))
    with contextlib.redirect_stdout(io.StringIO()):
        params, names = ref.inject_trainable_lora_extended(m, {"UNet3DConditionModel"}, r=16)
    census = dict(cfg=LORA_SMALL, r=16, n_param_groups=len(params), names=sorted(names),
                  shapes={k: tuple(v.shape) for k, v in m.named_parameters()},
                  kinds=sorted(type(x).__name__ for x in m.modules() if type(x).__name__.startswith("LoraInjected")))
    with contextlib.redirect_stdout(io.StringIO()):
        lin = ref.LoraInjectedLinear(64, 128, True, r=16)
        conv = ref.LoraInjectedConv2d(64, 96, 3, 1, 1, r=16)
        conv3d = ref.LoraInjectedConv3d(64, 64, (3, 1, 1), (1, 0, 0), bias=True, r=16)
    g = torch.Generator().manual_seed(3)
    inputs = dict(linear=torch.randn(50, 64, generator=g), conv2d=torch.randn(2, 64, 8, 8, generator=g),
                  conv3d=torch.randn(1, 64, 5, 4, 4, generator=g))
    wrappers = {}
    for seed, (name, mod) in enumerate((("linear", lin), ("conv2d", conv), ("conv3d", conv3d))):
        mod.load_state_dict(seeded_state_dict(mod, seed))
        mod.eval()
        with torch.no_grad():
            wrappers[name] = dict(weight_seed=seed, x=inputs[name], y=mod(inputs[name]))
    return dict(injection=census, wrappers=wrappers)


def config_fixture():
    import yaml
    cfg_dir = os.path.join(REFERENCE_ROOT, "configs", "v2")
    out = {}
    for fn in sorted(os.listdir(cfg_dir)):
        if fn.endswith(".yaml"):
            with open(os.path.join(cfg_dir, fn)) as f:
                cfg = yaml.safe_load(f)
            out[fn] = dict(keys=sorted(cfg), dataset_types=cfg.get("dataset_types", []), train_data=cfg.get("train_data") or {})
    return out


def main():
    torch.set_num_threads(8)
    for name, data in (("oracle_vs_reference.pt", unet_fixture()), ("lora_reference.pt", lora_fixture(ref_lora()))):
        path = os.path.join(GOLDEN, name)
        torch.save(data, path)
        print(name, os.path.getsize(path) // 1024, "KiB")
    path = os.path.join(GOLDEN, "reference_configs.json")
    with open(path, "w") as f:
        json.dump(config_fixture(), f, indent=1, sort_keys=True)
        f.write("\n")
    print("reference_configs.json", os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
