#!/usr/bin/env python
"""bf16 vs fp16 mixed precision of the training step, alternated in one process (A/B/A/B...) on one GPU.

The workload, warm-up, L2 flush and seeds are those of `bench.py --workload train`: small_denoiser_config at 128x128, batch 64,
scheduler 3k_steps_clipping_rescaling, seed-0 weights, bench.py's synthetic images and labels, noise / timesteps from a device
generator seeded 7, a 256 MB buffer rewritten before every timed step.  Each arm has its own model and trainer (same weights); both
warm up first, then every round times --steps steps of one arm with CUDA events.  One JSON line per arm and round: images/s, ms/step,
kernel launches per step (counted as bench.py counts them), skipped steps and the final loss scale (fp16); first a line with the GPU
name and power limit.
  python tools/bench_train_precision.py [--rounds 2] [--steps 5] [--warmup 3]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info(index):
    q = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=2, help="rounds; each times both arms (bf16 first)")
    ap.add_argument("--steps", type=int, default=5, help="timed steps per arm and round")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--size", type=int, default=128)
    args = ap.parse_args()

    import torch

    assert torch.cuda.is_available(), "needs a GPU: there is no CPU fallback"
    import __graft_entry__ as ge

    ge.build()
    from bench import make_inputs
    from phendiff_b200 import CustomCondUNet2DModel, DDIMScheduler
    from phendiff_b200.reference_configs import DENOISER_CONFIGS, SCHEDULER_CONFIGS
    from phendiff_b200.training import DenoiserTrainer

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    print(json.dumps({"gpu": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit_max_sm_clock": gpu_info(0)}), flush=True)
    x_host, labels, _ = make_inputs(args.batch, args.size, 0)
    x, labels = x_host.to(dev), labels.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    arms = {}
    for prec in ("bf16", "fp16"):
        torch.manual_seed(0)
        unet = CustomCondUNet2DModel.from_config(dict(DENOISER_CONFIGS["small_denoiser_config"], sample_size=args.size)).to(dev)
        sched = DDIMScheduler.from_config(SCHEDULER_CONFIGS["3k_steps_clipping_rescaling"])
        tr = DenoiserTrainer(unet, sched, args.batch, args.size, learning_rate=1e-4, use_ema=True, mixed_precision=prec)
        arms[prec] = (tr, sched, torch.Generator(device=dev).manual_seed(7))

    def step(prec):
        tr, sched, g = arms[prec]
        noise = torch.randn(x.shape, device=dev, generator=g)
        ts = torch.randint(0, sched.config.num_train_timesteps, (args.batch,), device=dev, generator=g)
        return tr.step(x, labels, noise=noise, timesteps=ts, do_unconditional_pass=False)

    for prec in arms:
        for _ in range(args.warmup):
            step(prec)
    torch.cuda.synchronize()
    for r in range(args.rounds):
        for prec, (tr, _, _) in arms.items():
            l0 = tr.launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                flush.fill_(1)
                loss = step(prec)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            launches = (tr.launch_count() - l0) / args.steps + 4      # + add_noise and the three optimizer launches, as bench.py counts
            st = tr.scaler_state()
            print(json.dumps({"round": r, "mixed_precision": prec, "images_per_s": args.batch * args.steps / (ms / 1e3),
                              "ms_per_step": ms / args.steps, "launches_per_step": launches,
                              "skipped_steps": st["skipped_steps"] if st else 0, "final_scale": st["scale"] if st else None,
                              "loss": float(loss.item()), "batch": args.batch, "size": args.size, "steps": args.steps}), flush=True)


if __name__ == "__main__":
    main()
