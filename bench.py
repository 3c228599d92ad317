#!/usr/bin/env python
"""Benchmark of the hot path named by BASELINE.json.

Default workload (configs[1], the one the metric is quoted on): finetune frames/sec of the text-to-video-ms-1.7b UNet,
16 frames x 256^2 -> latents 1x4x16x32x32 per GPU, bf16 compute, FULL fine-tune.  One step = one UNet forward + backward
pass (fp32 gradients, TemporalConvLayer dropout live), ONE gradient all-reduce when N > 1, global-norm clipping and the
fused AdamW update of all 1.41 B parameters - replayed as one CUDA graph; data-parallel by clip (weak scaling).

  python bench.py --gpus N --steps K --warmup W                 -> one JSON line (rank 0)
  python bench.py --workload lora|zeroscope|vae ...             -> configs[2] / [3] / [4] of BASELINE.json (extra lines)
  python bench.py --impl reference ...                          -> the reference algorithm on the host CPU cores: the
        reference's own models/*.py when T2V_REFERENCE_ROOT names a checkout of it, else the oracle port of it;
        its diffusers dependency is not installed (DESIGN.md section 5), same metric/unit.
  python bench.py ... --dump-outputs DIR                        -> also writes the last timed step's outputs as DIR/*.npy
Everything under oracle/ is used only for the parity / cpu_baseline / --impl reference legs.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

# SURVEY.md 8(d): algorithmic 2*MAC of the conv / linear / attention contractions per clip (validated by the 1,411,233,860-parameter walk)
WORKLOADS = {
    "cfg2": dict(name="configs[1]: text-to-video-ms-1.7b full finetune, 16 frames 256x256 (latents 1x4x16x32x32 per GPU), bf16",
                 model="text-to-video-ms-1.7b UNet3DConditionModel (random init, conv4 re-drawn N(0,0.01))",
                 frames=16, latent_hw=(32, 32), text_len=77, text_dim=1024, fwd_tflop=4.887, pass_tflop=14.66, attn_tflop=0.41,
                 lora_rank=0, grad_ckpt=False),
    "lora": dict(name="configs[2]: text-to-video-ms-1.7b LoRA rank-16 (cloneofsimo, target UNet3DConditionModel), 24 frames 320x576 "
                      "(latents 1x4x24x40x72 per GPU), bf16",
                 model="text-to-video-ms-1.7b UNet3DConditionModel + 574 LoRA wrappers (29,246,112 trainable parameters)",
                 frames=24, latent_hw=(40, 72), text_len=77, text_dim=1024, fwd_tflop=21.395 + 0.79, pass_tflop=2 * (21.395 + 0.79) + 0.79,
                 attn_tflop=3 * 0.073 * 21.395, lora_rank=16, grad_ckpt=False),
    "zeroscope": dict(name="configs[3]: zeroscope_v2_576w (same architecture) full finetune, 32 frames 512x512 (latents 1x4x32x64x64 per "
                           "GPU), bf16, gradient checkpointing",
                      model="zeroscope_v2_576w UNet3DConditionModel (random init, conv4 re-drawn N(0,0.01))",
                      frames=32, latent_hw=(64, 64), text_len=77, text_dim=1024, fwd_tflop=41.71, pass_tflop=125.1,
                      attn_tflop=3 * 0.099 * 41.71, lora_rank=0, grad_ckpt=True),
}
CFG2 = WORKLOADS["cfg2"]
VAE_TFLOP_PER_FRAME = {256: 0.2727, 512: 1.1167, 768: 2.6091}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("bf16_tflops_sustained", 1443.0), d.get("hbm_gbs", 6569.3), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        mx = max(int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit())
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": reasons, "samples": len(sm)}


def synthetic_inputs(batch, cfg, seed, device="cpu", pin=False):
    g = torch.Generator().manual_seed(seed)
    F, (H, W) = cfg["frames"], cfg["latent_hw"]
    lat = torch.randn(batch, 4, F, H, W, generator=g) * 0.18215
    noise = torch.randn(batch, 4, F, H, W, generator=g)
    t = torch.randint(0, 1000, (batch,), generator=g)
    ehs = torch.randn(batch, cfg["text_len"], cfg["text_dim"], generator=g)
    out = [lat, noise, t, ehs]
    if pin:
        out = [x.pin_memory() for x in out]
    return [x.to(device) for x in out] if device != "cpu" else out


def build_unet(device, small=False, dropout=True):
    """Random-init UNet of the ms-1.7b / zeroscope architecture (no checkpoints offline); TemporalConvLayer.conv4 is
    re-drawn N(0, 0.01) so the temporal-conv branch carries signal (SURVEY 8(d)).  Training mode: the TemporalConvLayer
    dropout (p = 0.1) is live unless dropout=False."""
    from t2v_b200.models.unet_3d_condition import UNet3DConditionModel
    kw = dict(block_out_channels=(128, 256, 320, 320), cross_attention_dim=1024) if small else {}
    torch.manual_seed(1234)
    with torch.device(device):
        m = UNet3DConditionModel(**kw)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if ".conv4.3." in n:
                p.normal_(0.0, 0.01)
    if not dropout:
        for mod in m.modules():
            if isinstance(mod, torch.nn.Dropout):
                mod.p = 0.0
    return m.train()


def oracle_pass(sd_cpu, cfg, inputs, threads):
    """One forward+backward of the reference algorithm (oracle port, fp32) on the host CPU.  Returns seconds, loss, grad norm."""
    from oracle import leaves as L
    from oracle import unet3d_ref as R
    torch.set_num_threads(threads)
    lat, noise, t, ehs = inputs
    p = {k: v.detach().clone().requires_grad_(True) for k, v in sd_cpu.items()}
    t0 = time.perf_counter()
    loss, _ = R.finetune_loss(p, R.full_config(**cfg.get("unet_kwargs", {})), lat, noise, t, ehs, L.ddpm_alphas_cumprod())
    loss.backward()
    dt = time.perf_counter() - t0
    gn = math.sqrt(sum(float(v.grad.double().pow(2).sum()) for v in p.values() if v.grad is not None))
    return dt, float(loss), gn


def reference_pass(Ref, sd_cpu, cfg, inputs, threads):
    """The same pass through the reference's UNMODIFIED models/unet_3d_condition.py + unet_3d_blocks.py (imported from
    T2V_REFERENCE_ROOT over the diffusers stand-in, oracle/reference_import.py) with the step glue of train.py:751-834."""
    from oracle import leaves as L
    torch.set_num_threads(threads)
    lat, noise, t, ehs = inputs
    m = Ref(**cfg.get("unet_kwargs", {}))
    m.load_state_dict(sd_cpu)
    m.train()
    for mod in m.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
    t0 = time.perf_counter()
    noisy = L.add_noise(lat, noise, t, L.ddpm_alphas_cumprod())
    pred = m(noisy, t, encoder_hidden_states=ehs).sample
    loss = torch.nn.functional.mse_loss(pred.float(), noise.float(), reduction="mean")
    loss.backward()
    dt = time.perf_counter() - t0
    gn = math.sqrt(sum(float(p.grad.double().pow(2).sum()) for p in m.parameters() if p.grad is not None))
    return dt, float(loss), gn


def gemm_traffic():
    """DRAM bytes per launch of the dominant kernel (dram__bytes_read.sum + dram__bytes_write.sum averaged over the
    launches of one step) from the committed ncu capture; None if the file is absent."""
    for name in ("r2_gemm_traffic.json", "r1_gemm_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return float(json.load(f)["dram_bytes_per_launch"])
        except (OSError, KeyError, ValueError):
            continue
    return None


def run_reference(args):
    """--impl reference: the reference algorithm on the host cores, full workload shape (16-frame clip), bounded by steps."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle.reference_import import import_reference_unet, reference_available
    from t2v_b200.models.unet_3d_condition import UNet3DConditionModel  # parameter shapes only (random init)
    wl = WORKLOADS[args.workload if args.workload in WORKLOADS else "cfg2"]
    threads = min(os.cpu_count() or 1, 32)  # the small fp32 ops of this model do not scale past ~32 threads
    cfg = dict(wl)
    kw = dict(block_out_channels=(128, 256, 320, 320)) if args.small else {}
    cfg["unet_kwargs"] = kw
    torch.manual_seed(1234)
    m = UNet3DConditionModel(**kw)
    sd = {k: v.detach().clone().contiguous() for k, v in m.state_dict().items()}
    for k in sd:
        if ".conv4.3." in k:
            sd[k].normal_(0.0, 0.01)
    del m
    frames = args.ref_frames or wl["frames"]
    c = dict(cfg)
    c["frames"] = frames
    inputs = synthetic_inputs(1, c, 99)
    Ref = import_reference_unet() if reference_available() else None
    kind = "reference" if Ref is not None else "port"
    times = []
    for i in range(args.warmup + args.steps):
        dt = (reference_pass(Ref, sd, cfg, inputs, threads) if Ref is not None else oracle_pass(sd, cfg, inputs, threads))[0]
        if i >= args.warmup:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    fps = frames / (ms / 1e3)
    what = ("the reference's unmodified models/*.py over the diffusers stand-in" if Ref is not None else
            "oracle port of the reference algorithm (T2V_REFERENCE_ROOT names no reference checkout)")
    line = {"impl": "reference", "metric": "finetune frames/sec (one UNet fwd+bwd pass per step)", "value": fps, "unit": "frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["name"], "sample": f"{frames}-frame clip, fwd+bwd only (no optimizer step on the CPU arm)",
                       "same_config": frames == wl["frames"]},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": kind,
                             "sample": f"{len(times)} fwd+bwd passes of a {frames}-frame clip, {what}, fp32, {threads} threads"},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


_REAL_STDOUT = None


def quiet_stdout():
    """Everything libraries print (NCCL's version banner, torchrun notes) goes to stderr: stdout carries ONE JSON line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def shutdown(world, step=None):
    """Tear the process group down without hanging: drop the CUDA graph that holds captured NCCL kernels first, and do
    not let communicator destruction or interpreter teardown block the launcher (bounded by a timer)."""
    if world <= 1:
        return
    import gc
    import torch.distributed as dist
    sys.stdout.flush()
    sys.stderr.flush()
    threading.Timer(20.0, lambda: os._exit(0)).start()
    try:
        if step is not None:
            step._graph = None
        gc.collect()
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()
    finally:
        os._exit(0)


DUMP_SAMPLE = 1 << 22   # elements per sampled array: 16 MB in float32


def dump_outputs(out_dir, loss, arena, optimizer):
    """What the last step hands its caller: the loss, and the updated fp32 master weights and AdamW first moment (the
    gradients without an optimizer), the latter two as the same fixed, seeded sample of the flat parameter arena."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    n = arena.master.numel()
    idx = torch.randint(0, n, (min(n, DUMP_SAMPLE),), generator=torch.Generator().manual_seed(0)).sort().values
    idx = idx.to(arena.master.device)
    arrays = {"loss": np.array([loss], dtype=np.float64), "weights_sample": arena.master[idx]}
    if optimizer is not None:
        arrays["exp_avg_sample"] = optimizer.exp_avg[idx]
    else:
        arrays["grad_sample"] = arena.grad[idx]
    for name, a in arrays.items():
        if isinstance(a, torch.Tensor):
            a = a.float().cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a)


def time_events(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def run_vae(args, dev):
    """configs[4]: AutoencoderKL.encode throughput (tensor_to_vae_latent, train.py:339-347) at 256 / 512 / 768 px, frames
    batched, full SD-VAE encoder widths (128-256-512-512), random init."""
    from t2v_b200 import native
    from t2v_b200.vae import AutoencoderKL, tensor_to_vae_latent
    native.lib()
    torch.manual_seed(7)
    with torch.device(dev):
        vae = AutoencoderKL()
    vae = vae.eval()
    peak_tf, _, how = peaks()
    sweep = {}
    for res, frames in ((256, 16), (512, 16), (768, 8)):
        host = (torch.rand(1, frames, 3, res, res) * 2 - 1).pin_memory()
        x = host.to(dev)
        for _ in range(max(args.warmup, 3)):
            tensor_to_vae_latent(x, vae)
        torch.cuda.synchronize()
        n0 = native.launch_count()
        ms = time_events(lambda: tensor_to_vae_latent(x, vae), args.steps)
        launches = (native.launch_count() - n0) // args.steps
        ms_e2e = time_events(lambda: tensor_to_vae_latent(host.to(dev, non_blocking=True), vae).float().mean().item(), args.steps)
        tf = VAE_TFLOP_PER_FRAME[res] * frames
        sweep[str(res)] = {"frames_per_batch": frames, "ms_per_batch": ms, "frames_per_s": frames / (ms / 1e3),
                           "e2e_frames_per_s": frames / (ms_e2e / 1e3), "tflops": tf / (ms / 1e3), "frac_of_peak": tf / (ms / 1e3) / peak_tf,
                           "launches_per_batch": int(launches), "h2d_bytes": host.numel() * 4}
    cpu = None
    if not args.no_cpu_baseline:
        from oracle import leaves as L
        threads = min(os.cpu_count() or 1, 32)
        torch.set_num_threads(threads)
        sd = {k: v.detach().float().cpu() for k, v in vae.state_dict().items()}
        xc = torch.rand(2, 3, 256, 256) * 2 - 1
        t0 = time.perf_counter()
        with torch.no_grad():
            L.vae_encode_moments(sd, xc)
        dt = time.perf_counter() - t0
        cpu = {"value": 2 / dt, "unit": "frames/s", "cores": threads, "kind": "port",
               "sample": f"2 frames at 256x256, oracle port of AutoencoderKL.encode, fp32, {threads} threads"}
    main_res = sweep["256"]
    emit({"metric": "AutoencoderKL.encode frames/sec (256x256 frames, batch of 16)", "value": main_res["frames_per_s"], "unit": "frames/s",
          "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": main_res["ms_per_batch"], "higher_is_better": True,
          "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
          "config": {"workload": "configs[4]: AutoencoderKL.encode throughput sweep, batched frames at 256/512/768, 1xB200",
                     "l2": "activations of a 16-frame batch (>= 268 MB at the first level) exceed the 126 MB L2"},
          "sweep": sweep, "e2e": {"value": main_res["e2e_frames_per_s"], "unit": "frames/s", "h2d_bytes_per_step": main_res["h2d_bytes"],
                                  "d2h_bytes_per_step": 4},
          "gpu_launches": int(main_res["launches_per_batch"] * args.steps),
          "roofline": {"bound": "tensor", "kernel": "gemm_tc_kernel (3x3 implicit-GEMM convolutions, 98 % of the encoder FLOPs)",
                       "achieved": main_res["tflops"], "peak": peak_tf, "unit": "TFLOP/s", "frac": main_res["frac_of_peak"], "traffic": None,
                       "note": "whole-encode FLOPs over whole-encode time (not per-kernel)", "peak_source": how},
          "cpu_baseline": cpu})


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "lora", "zeroscope", "vae"])
    ap.add_argument("--small", action="store_true", help="debug-size UNet (not a valid bench line)")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replay")
    ap.add_argument("--no-optimizer", action="store_true", help="forward + backward (+ all-reduce) only - NOT a valid finetune step")
    ap.add_argument("--no-dropout", action="store_true")
    ap.add_argument("--ref-frames", type=int, default=0, help="frames of the CPU clip (reference arm / cpu_baseline); 0 = the workload's")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU leg (and with it the parity check)")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--profile-timed-region", action="store_true",
                    help="cudaProfilerStart/Stop around the K timed steps: `ncu --profile-from-start off ... python bench.py --steps 1 "
                         "--profile-timed-region` lists exactly the kernels of the timed region (numbers printed under ncu are not bench values)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (the loss and fixed seeded samples of the "
                         "updated weights and of the optimizer's first moment), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload == "vae"):
        ap.error("--dump-outputs covers the finetune step (--impl ours, workloads cfg2 / lora / zeroscope)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        if args.steps is None:
            args.steps = 3   # full-size fp32 passes on the host cores take tens of seconds each
        args.warmup = min(args.warmup, 1)
        return run_reference(args)
    if args.steps is None:
        args.steps = 20 if world == 1 else 50   # collective-bound timings need more samples
    args.warmup = max(args.warmup, 3)

    import torch.distributed as dist
    from t2v_b200 import native
    from t2v_b200 import step as S
    from t2v_b200.optim import FusedAdamW

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if args.workload == "vae":
        if rank == 0:
            run_vae(args, dev)
        return
    wl = WORKLOADS[args.workload]
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG", "WARN")   # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=dev)
    native.lib()  # fail loudly if the CUDA extension is missing

    unet = build_unet(dev, args.small, dropout=not args.no_dropout)
    if wl["lora_rank"]:
        from t2v_b200.utils.lora_handler import LoraHandler
        unet.requires_grad_(False)
        handler = LoraHandler(version="cloneofsimo", use_unet_lora=True, unet_replace_modules=["UNet3DConditionModel"])
        torch.manual_seed(4321)   # rank-independent LoRA initialisation
        handler.add_lora_to_model(True, unet, handler.unet_replace_modules, 0.1, "", r=wl["lora_rank"])
        unet = unet.to(dev).train()
        with torch.no_grad():     # lora_up starts at zero (reference utils/lora.py:54-55): give the branch signal for the bench
            for n, p in unet.named_parameters():
                if "lora_up" in n:
                    p.normal_(0.0, 0.01)
    unet._set_gradient_checkpointing(bool(wl["grad_ckpt"]))
    abar = S.ddpm_alphas_cumprod(device=dev)
    step = S.DataParallelStep(unet, abar, passes=1, use_graph=not args.no_graph)
    optimizer = None
    trainable = [p for p in unet.parameters() if p.requires_grad]
    n_trainable = sum(p.numel() for p in trainable)
    if not args.no_optimizer:
        # the reference's optimizer settings (configs/v2/train_config.yaml: lr 5e-6, wd 1e-2, max_grad_norm 1.0)
        optimizer = FusedAdamW(step.arena, [dict(params=trainable)], lr=5e-6, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2,
                               max_grad_norm=1.0)
        step.attach_optimizer(optimizer)
    B = 1
    host = synthetic_inputs(B, wl, 1234 + rank, pin=True)
    devin = [x.to(dev) for x in host]
    frames_per_step = world * B * wl["frames"]

    # ---- parity step (rank 0, N = 1): one eager fwd+bwd at the FULL benchmark size with dropout off, on the initial
    # weights; loss and global gradient norm are compared with the CPU oracle after the timed region (cpu_baseline leg)
    eager = S.DataParallelStep(unet, abar, passes=1, use_graph=False, adopt=False)
    eager.arena = step.arena
    eager.sync_gradients = False  # profiling passes below run on their own rank: no collective
    parity_gpu = None
    do_parity = rank == 0 and world == 1 and not args.no_cpu_baseline and not wl["lora_rank"]
    if do_parity:
        sd_cpu = {k: v.detach().float().cpu().contiguous() for k, v in unet.state_dict().items()}
        unet.eval()
        lossv = eager(*devin)
        gn = float(step.arena.grad.double().norm())
        parity_gpu = (float(lossv), gn)
        unet.train()
    # ---- launches per step, counted on an eager step (training mode: dropout kernels included)
    n0 = native.launch_count()
    eager(*devin)
    torch.cuda.synchronize()
    launches_per_step = native.launch_count() - n0
    if optimizer is not None:   # clip: one sqnorm per hyper-parameter set; one prepare; one update per set
        launches_per_step += 2 * len(optimizer._sets) + 1

    # ---- dominant-kernel roofline: every tensor-core (implicit-GEMM) launch of the step, timed on the device.  One eager
    # step records each launch's argument template; each distinct template is then replayed as a CUDA graph of back-to-back
    # launches over ROTATING operand copies (> L2 in total, so no launch finds its operands cached by the previous one)
    # between CUDA events (eager per-launch events would count host launch gaps as kernel time).
    roof = None
    if rank == 0 and not args.no_roofline:  # before the step graph is captured (graph-pool memory would distort eager allocation)
        from t2v_b200 import profiling
        calls = profiling.record_calls(lambda: eager(*devin), ["conv_fwd", "conv_dgrad", "conv_wgrad", "bgemm"])
        gemm_ms, gemm_ms_warm, n_gemm = 0.0, 0.0, 0
        with ClockSampler(local) as roof_clocks:   # this leg is a dense stream of GEMMs: its own clocks / power state are reported
            for key, (cnt, _) in calls.items():
                gemm_ms += profiling.replay_us(key, dev, reps=8, cold=True, batches=3) * cnt / 1e3   # median of 3 batches per shape
                gemm_ms_warm += profiling.replay_us(key, dev, reps=5, cold=False) * cnt / 1e3
                n_gemm += cnt
        torch.cuda.empty_cache()
        peak_tf, peak_hbm, how = peaks()
        from t2v_b200 import ops as _ops
        gemm_tflop = wl["pass_tflop"] - (wl["attn_tflop"] if _ops._Flash.enabled else 0.0)
        flops = (gemm_tflop if not args.small else float("nan")) * B
        ach = flops / (gemm_ms / 1e3) if gemm_ms > 0 else 0.0
        roof = {"bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05 implicit-GEMM conv / linear contractions)",
                "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf, "traffic": gemm_traffic(),
                "launches": n_gemm, "distinct_shapes": len(calls), "kernel_ms_per_step": gemm_ms, "share_of_step": None,
                "algorithmic_tflop_per_step": flops, "peak_source": how,
                "timing": "per-shape CUDA-graph replay over rotating operand copies (L2-cold), CUDA events, median of 3 batches of >= 24 launches",
                "clocks": roof_clocks.summary(),
                "l2_warm": {"kernel_ms_per_step": gemm_ms_warm, "frac": (flops / (gemm_ms_warm / 1e3) / peak_tf) if gemm_ms_warm else None}}
    step.arena.zero_grads()   # the eager passes above accumulated gradients; the timed steps start from a zero buffer

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident leg ("value")
    for _ in range(args.warmup):
        loss = step(*devin)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        if args.profile_timed_region:
            torch.cuda.cudart().cudaProfilerStart()
        e0.record()
        for _ in range(args.steps):
            loss = step(*devin)
        e1.record()
        barrier()
        if args.profile_timed_region:
            torch.cuda.cudart().cudaProfilerStop()
    ms = e0.elapsed_time(e1) / args.steps
    # ---- end-to-end leg: pinned host inputs -> device every step, loss read back every step
    for _ in range(2):
        step(*[x.to(dev, non_blocking=True) for x in host]).item()
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        lv = step(*[x.to(dev, non_blocking=True) for x in host]).item()
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1) / args.steps
    if args.dump_outputs and rank == 0:   # before the optimizer is timed alone below: that moves the weights again
        dump_outputs(args.dump_outputs, lv, step.arena, optimizer)
    # ---- the optimizer's share (clip + AdamW over the trainable set), timed alone on the device
    opt_ms = None
    if optimizer is not None:
        optimizer.push_hyperparams()
        for _ in range(2):
            optimizer.launch()
        torch.cuda.synchronize()
        opt_ms = time_events(optimizer.launch, 5)
    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()

    if rank != 0:
        shutdown(world, step)
        return

    cpu, parity = None, None
    if not args.no_cpu_baseline and world == 1:
        threads = min(os.cpu_count() or 1, 32)  # more threads only oversubscribe the small fp32 ops of this model
        cfg = dict(wl)
        cfg["unet_kwargs"] = dict(block_out_channels=(128, 256, 320, 320)) if args.small else {}
        if do_parity:
            fr = wl["frames"]
            dt, loss_ref, gn_ref = oracle_pass(sd_cpu, cfg, [x.clone() for x in host], threads)
            loss_rel = abs(parity_gpu[0] - loss_ref) / abs(loss_ref)
            gn_rel = abs(parity_gpu[1] - gn_ref) / gn_ref
            parity = {"loss": parity_gpu[0], "loss_oracle": loss_ref, "loss_rel": loss_rel, "grad_norm": parity_gpu[1],
                      "grad_norm_oracle": gn_ref, "grad_norm_rel": gn_rel, "tolerance": {"loss_rel": 1e-3, "grad_norm_rel": 1e-3},
                      "status": "green" if (loss_rel <= 1e-3 and gn_rel <= 1e-3) else "red",
                      "what": "full benchmark configuration (1.41 B parameters, 16 frames, 32x32 latents), dropout off, same weights and "
                              "inputs; bf16 kernels vs the fp32 CPU oracle"}
        else:
            fr = args.ref_frames or 4
            c = dict(cfg)
            c["frames"] = fr
            import re
            sd1 = {re.sub(r"\.(linear|conv)\.(weight|bias)$", r".\2", k) if wl["lora_rank"] else k: v.detach().float().cpu().contiguous()
                   for k, v in unet.state_dict().items() if "lora" not in k}   # base weights only (the CPU arm has no LoRA branch)
            dt = oracle_pass(sd1, cfg, synthetic_inputs(1, c, 99), threads)[0]
        cpu = {"value": fr / dt, "unit": "frames/s", "cores": threads, "kind": "port",
               "sample": f"one fwd+bwd pass of a {fr}-frame clip at {wl['latent_hw'][0]}x{wl['latent_hw'][1]} latents, oracle port of the "
                         f"reference algorithm, fp32, {threads} threads (no optimizer step)"}

    in_bytes = sum(x.numel() * x.element_size() for x in host)
    line = {
        "metric": "finetune frames/sec (one UNet fwd+bwd pass + optimizer step per step)" if optimizer is not None
        else "fwd+bwd frames/sec (NO optimizer step - not a finetune step)",
        "value": frames_per_step / (ms / 1e3), "unit": "frames/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": wl["name"], "model": wl["model"], "passes_per_step": 1, "global_batch_clips": world * B,
                   "parallelism": f"dp{world}", "dropout": "off" if args.no_dropout else "on (TemporalConvLayer p=0.1, LoRA p=0.1)",
                   "optimizer": None if optimizer is None else "fused AdamW + global-norm clip (max_grad_norm 1.0) inside the timed step",
                   "trainable_parameters": int(n_trainable), "gradient_checkpointing": bool(wl["grad_ckpt"]),
                   "l2": "working set (2.8 GB bf16 weights + activations) >> 126 MB L2; no flush needed",
                   "launch_mode": "eager" if args.no_graph else "cuda-graph replay", "small_debug_model": bool(args.small)},
        "e2e": {"value": frames_per_step / (ms_e2e / 1e3), "unit": "frames/s", "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e},
        "gpu_launches": int(launches_per_step * (args.steps)),
        "launches_per_step": int(launches_per_step),
        "optimizer_ms": opt_ms,
        "fwd_bwd_ms": (ms - opt_ms) if opt_ms is not None else ms,
        "clocks": clocks.summary(),
        "loss": lv,
        "parity": parity,
        "roofline": dict(roof, share_of_step=(roof["kernel_ms_per_step"] / ms)) if roof else None,
        "cpu_baseline": cpu,
    }
    emit(line)
    shutdown(world, step)


if __name__ == "__main__":
    main()
