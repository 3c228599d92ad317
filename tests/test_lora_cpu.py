"""cloneofsimo LoRA surface (utils/lora.py, utils/lora_handler.py) on CPU with emulated primitives:
injection census and key names against the reference's own injector, module-level forward parity against the reference
classes (both from tests/golden/lora_reference.pt, made by tests/golden/make_golden_reference.py with the reference's
utils/lora.py imported unmodified), zero-init identity, and the collapse/remove round trip."""
import contextlib
import io
import os

import pytest
import torch

from helpers import emulated_prims, rel_l2, seeded_state_dict
from oracle import ops_ref

SMALL = dict(block_out_channels=(64, 128, 128, 128), attention_head_dim=64, cross_attention_dim=64)
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "lora_reference.pt")


@pytest.fixture(autouse=True)
def exact_arithmetic():
    old = ops_ref.BF
    ops_ref.BF = torch.float32
    yield
    ops_ref.BF = old


def _quiet():
    return contextlib.redirect_stdout(io.StringIO())


def _model(seed=0):
    from t2v_b200.models.unet_3d_condition import UNet3DConditionModel
    m = UNet3DConditionModel(**SMALL)
    sd = seeded_state_dict(m, seed)
    m.load_state_dict(sd)
    return m.eval(), sd


def _golden():
    return torch.load(GOLDEN, weights_only=False)


def test_injection_matches_reference_injector():
    from t2v_b200.utils import lora as mylora
    ref = _golden()["injection"]
    assert ref["cfg"] == SMALL
    m, sd = _model()
    with _quiet():
        pm, nm = mylora.inject_trainable_lora_extended(m, {"UNet3DConditionModel"}, r=ref["r"])
    assert len(pm) == ref["n_param_groups"] and sorted(nm) == ref["names"]
    a = {k: tuple(v.shape) for k, v in m.named_parameters()}
    assert a == ref["shapes"]
    kinds = sorted(type(x).__name__ for x in m.modules() if type(x).__name__.startswith("LoraInjected"))
    assert kinds == ref["kinds"]
    # zero-initialised up, N(0, 1/r) down, shared base parameters, default dropout (0.1 / 0.1 / 0)
    w = m.down_blocks[0].resnets[0].conv1
    assert isinstance(w, mylora.LoraInjectedConv2d) and w.lora_up.weight.abs().max() == 0 and w.dropout.p == 0.1
    assert m.down_blocks[0].temp_convs[0].conv1[2].dropout.p == 0


def test_wrapper_forward_matches_reference_classes():
    from t2v_b200.utils import lora as mylora
    ref = _golden()["wrappers"]
    with _quiet():
        mods = dict(linear=mylora.LoraInjectedLinear(64, 128, True, r=16), conv2d=mylora.LoraInjectedConv2d(64, 96, 3, 1, 1, r=16),
                    conv3d=mylora.LoraInjectedConv3d(64, 64, (3, 1, 1), (1, 0, 0), bias=True, r=16))
    for name, m in mods.items():
        m.load_state_dict(seeded_state_dict(m, ref[name]["weight_seed"]))
        m.eval()
    lm, cm, tm = mods["linear"], mods["conv2d"], mods["conv3d"]
    x, xi, xv = ref["linear"]["x"], ref["conv2d"]["x"], ref["conv3d"]["x"]
    with emulated_prims():
        assert rel_l2(lm(x), ref["linear"]["y"]) < 1e-6
        assert rel_l2(cm(xi.permute(0, 2, 3, 1).contiguous()).permute(0, 3, 1, 2), ref["conv2d"]["y"]) < 1e-5
        y = tm(xv.permute(0, 2, 3, 4, 1).reshape(1, 5, 16, 64).contiguous())
        assert rel_l2(y.reshape(1, 5, 4, 4, 64).permute(0, 4, 1, 2, 3), ref["conv3d"]["y"]) < 1e-5


def test_zero_init_identity_and_collapse_round_trip():
    from t2v_b200.utils import lora as mylora
    m0, sd = _model()
    m, _ = _model()
    with _quiet():
        params, names = mylora.inject_trainable_lora_extended(m, mylora.UNET_EXTENDED_TARGET_REPLACE, r=8)
    m.eval()  # freshly injected wrappers default to train mode (live dropout), exactly as in the reference
    assert params and all("lora" not in n for n in sd)
    x, t, ehs = torch.randn(1, 4, 2, 8, 8), torch.tensor([500]), torch.randn(1, 7, 64)
    with emulated_prims():
        base = m0(x, t, ehs).sample
        assert torch.equal(m(x, t, ehs).sample, base)          # lora_up == 0  =>  exactly the base model
        g = torch.Generator().manual_seed(5)
        with torch.no_grad():
            for n, p in m.named_parameters():
                if "lora_up" in n:
                    p.copy_(torch.randn(p.shape, generator=g) * 0.05)
        y = m(x, t, ehs).sample
        (y ** 2).mean().backward()
        lora_p = [(n, p) for n, p in m.named_parameters() if "lora" in n]
        assert all(p.grad is not None for _, p in lora_p)
        assert rel_l2(y, base) > 1e-2
        with _quiet():
            mylora.collapse_lora(m)
            mylora.monkeypatch_remove_lora(m)
        assert not [n for n, _ in m.named_parameters() if "lora" in n]
        assert rel_l2(m(x, t, ehs).sample, y) < 1e-5             # dropout off: W + up @ down reproduces the branch


def test_lora_handler_surface(tmp_path):
    from t2v_b200.utils.lora_handler import LORA_VERSIONS, LoraHandler
    assert LORA_VERSIONS == ["stable_lora", "cloneofsimo"]
    m, _ = _model()
    h = LoraHandler(version="cloneofsimo", use_unet_lora=True, unet_replace_modules=["UNet3DConditionModel"])
    with _quiet():
        params, negation = h.add_lora_to_model(True, m, h.unet_replace_modules, dropout=0.3, lora_path="", r=16)
    n_lora = sum(p.numel() for n, p in m.named_parameters() if "lora" in n)
    assert n_lora > 0 and len(params) == 2 * len(negation)
    from t2v_b200.utils.lora import save_lora_weight
    f = tmp_path / "10_unet.pt"
    save_lora_weight(m, str(f), h.unet_replace_modules)
    ws = torch.load(f)
    assert isinstance(ws, list) and len(ws) == len(params) and all(w.dtype == torch.float32 for w in ws)
    # reload into a fresh model through the handler's loader path
    m2, _ = _model()
    h2 = LoraHandler(version="cloneofsimo", use_unet_lora=True, unet_replace_modules=["UNet3DConditionModel"])
    with _quiet():
        h2.add_lora_to_model(True, m2, h2.unet_replace_modules, lora_path=str(tmp_path), r=16)
    a = dict(m.named_parameters())
    for n, p in m2.named_parameters():
        if "lora" in n:
            assert torch.equal(p.detach().cpu(), a[n].detach().cpu()), n
    with pytest.raises(NotImplementedError):
        LoraHandler(version="stable_lora", use_unet_lora=True).add_lora_to_model(True, m, ["UNet3DConditionModel"])
