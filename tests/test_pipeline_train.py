"""End to end through the 8(f) rows on a tiny but COMPLETE pipeline folder (unet / vae / text_encoder / tokenizer): raw .mp4
clips + captions -> dataset -> device resize/normalise -> VAE encode -> CLIP text encoder -> two-pass UNet step -> fused AdamW
-> `save_pipe` directory; the same through the latent cache; and every shipped reference YAML loads into `main`'s signature."""
import inspect
import json
import os

import pytest
import torch

from helpers import emulated_prims, seeded_state_dict
from test_dataset import _write_video

TINY = dict(block_out_channels=(64, 128, 128, 128), attention_head_dim=64, cross_attention_dim=64)


def _tiny_tokenizer(folder):
    """A real (slow) CLIPTokenizer over a byte-level vocabulary without merges: every character is its own token."""
    os.makedirs(folder, exist_ok=True)
    bs = list(range(ord("!"), ord("~") + 1)) + list(range(ord("\xa1"), ord("\xac") + 1)) + list(range(ord("\xae"), ord("\xff") + 1))
    cs, n = bs[:], 0
    for b in range(256):          # GPT-2 / CLIP byte <-> printable unicode table
        if b not in bs:
            bs.append(b)
            cs.append(256 + n)
            n += 1
    chars = [chr(c) for c in cs]
    vocab = {}
    for c in chars:
        vocab[c] = len(vocab)
    for c in chars:
        vocab[c + "</w>"] = len(vocab)
    vocab["<|startoftext|>"] = len(vocab)
    vocab["<|endoftext|>"] = len(vocab)
    with open(os.path.join(folder, "vocab.json"), "w") as f:
        json.dump(vocab, f)
    with open(os.path.join(folder, "merges.txt"), "w") as f:
        f.write("#version: 0.2\n")
    with open(os.path.join(folder, "tokenizer_config.json"), "w") as f:
        json.dump({"model_max_length": 77, "tokenizer_class": "CLIPTokenizer"}, f)
    return len(vocab)


def _pipeline_folder(root):
    from transformers import CLIPTextConfig
    from transformers import CLIPTextModel as HF
    from t2v_b200.models.unet_3d_condition import UNet3DConditionModel
    from t2v_b200.vae import AutoencoderKL
    unet = UNet3DConditionModel(**TINY)
    unet.load_state_dict(seeded_state_dict(unet, 0))
    unet.save_pretrained(os.path.join(root, "unet"))
    torch.manual_seed(1)
    AutoencoderKL(block_out_channels=(32, 32, 64, 64), layers_per_block=1).save_pretrained(os.path.join(root, "vae"))
    nvocab = _tiny_tokenizer(os.path.join(root, "tokenizer"))
    HF(CLIPTextConfig(hidden_size=64, intermediate_size=128, num_hidden_layers=1, num_attention_heads=1, vocab_size=nvocab,
                      max_position_embeddings=77, hidden_act="gelu")).save_pretrained(os.path.join(root, "text_encoder"))
    os.makedirs(os.path.join(root, "scheduler"), exist_ok=True)
    with open(os.path.join(root, "scheduler", "scheduler_config.json"), "w") as f:
        json.dump({"_class_name": "DDIMScheduler", "beta_start": 0.00085, "beta_end": 0.012, "beta_schedule": "scaled_linear",
                   "num_train_timesteps": 1000, "prediction_type": "epsilon"}, f)
    return root


def _run(tmp_path, device, **extra):
    from t2v_b200 import train
    root = _pipeline_folder(str(tmp_path / "pipe"))
    vids = tmp_path / "vids"
    vids.mkdir()
    for i in range(2):
        _write_video(str(vids / f"v{i}.mp4"), n=10, hw=(64, 64))
    (vids / "v0.txt").write_text("a red ball")
    out = str(tmp_path / "out")
    kw = dict(pretrained_model_path=root, output_dir=out, dataset_types=["folder"],
              train_data=dict(width=64, height=64, n_sample_frames=2, fps=8, path=str(vids), fallback_prompt="a video"),
              max_train_steps=2, learning_rate=1e-3, checkpointing_steps=10, seed=0, shuffle=False, device=device, eval_train=True,
              trainable_modules=["attn1", "attn2"], load_side_models=True, validation_data=None)
    kw.update(extra)
    r = train.main(**kw)
    return r, out, root


@pytest.mark.parametrize("cache", [False, True])
def test_raw_video_training_cpu(tmp_path, cache):
    with emulated_prims():
        r, out, root = _run(tmp_path, "cpu", cache_latents=cache)
    assert r["steps"] == 2
    # save_pipe: the complete pipeline directory
    for part in ("unet", "vae", "text_encoder", "tokenizer", "scheduler"):
        assert os.path.isdir(os.path.join(out, part)), part
    assert os.path.isfile(os.path.join(out, "model_index.json"))
    if cache:
        files = sorted(os.listdir(os.path.join(out, "cached_latents")))
        assert files == ["cached_0.pt", "cached_1.pt"]
        item = torch.load(os.path.join(out, "cached_latents", files[0]), weights_only=False)
        assert item["pixel_values"].shape == (4, 2, 8, 8) and item["pixel_values"].dtype == torch.float16


@pytest.mark.gpu
def test_raw_video_training_gpu(tmp_path):
    r, out, _ = _run(tmp_path, "cuda:0")
    assert r["steps"] == 2 and os.path.isdir(os.path.join(out, "text_encoder"))


def test_reference_yaml_configs_load_into_main():
    """Every shipped v2 YAML of the reference maps onto train.main's keyword surface (no unknown keys, no missing required).
    tests/golden/reference_configs.json holds each YAML's top-level keys, dataset_types and train_data section
    (tests/golden/make_golden_reference.py)."""
    from t2v_b200 import train
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_configs.json")) as f:
        configs = json.load(f)
    sig = inspect.signature(train.main)
    names = set(sig.parameters)
    seen = 0
    for fn, cfg in sorted(configs.items()):
        unknown = sorted(set(cfg["keys"]) - names)
        assert not unknown, (fn, unknown)
        sig.bind_partial(**dict.fromkeys(cfg["keys"]))
        # the `train_data:` section constructs every dataset class it names
        from t2v_b200.utils import dataset as D
        for kind in cfg["dataset_types"]:
            assert kind in D.DATASETS, (fn, kind)
            D.DATASETS[kind](**dict(cfg["train_data"]), tokenizer=None)
        seen += 1
    assert seen >= 1
