#!/usr/bin/env python
"""Data-parallel training step on real NCCL (run under torchrun on 2 GPUs: `bash tools/gpu.sh <tag> ddpcheck[:fp16]`).
Each rank runs forward + backward on ITS shard, the flat gradient vector is averaged with one all-reduce; rank 0 also runs both
shards locally (gradient accumulation) and checks that the all-reduced vector equals their mean, and that after the optimizer
step every rank holds bit-identical parameters.

--precision fp16 (default bf16): the same under dynamic loss scaling, then one step in which only rank 1's shard overflows (its noise
scaled by 1e6): the inf / NaN reaches every rank through the all-reduce, so every rank must skip that step, and parameters, EMA and
the scaler state must stay bit-identical across ranks after it and after one more normal step."""
import argparse
import math
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _fingerprint(tr):
    fp = [tr.params.double().sum(), tr.params.double().abs().sum(), tr.ema.double().sum()]
    if tr.mixed_precision == "fp16":
        st = tr.scaler_state()
        fp += [torch.tensor(float(st[k]), dtype=torch.float64, device=tr.device) for k in ("scale", "growth_tracker", "optimizer_steps", "skipped_steps")]
    return torch.stack(fp)


def _identical(tr, world, what):
    fp = _fingerprint(tr)
    gathered = [torch.empty_like(fp) for _ in range(world)]
    dist.all_gather(gathered, fp)
    same = all(torch.equal(gathered[0], t) for t in gathered)
    if dist.get_rank() == 0:
        print(f"[ddpcheck] {what} identical on all ranks: {same}")
    return same


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp16"], help="the trainer's mixed_precision")
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    import __graft_entry__ as ge

    ge.build()
    from phendiff_b200 import CustomCondUNet2DModel, DDIMScheduler
    from phendiff_b200.reference_configs import DENOISER_CONFIGS, SCHEDULER_CONFIGS
    from phendiff_b200.training import DenoiserTrainer

    B, size = 4, 64
    torch.manual_seed(0)
    unet = CustomCondUNet2DModel.from_config(dict(DENOISER_CONFIGS["small_denoiser_config"], sample_size=size)).to(dev)
    sched = DDIMScheduler.from_config(SCHEDULER_CONFIGS["3k_steps_clipping_rescaling"])
    tr = DenoiserTrainer(unet, sched, B, size, learning_rate=1e-3, use_ema=True, mixed_precision=args.precision)
    g = torch.Generator().manual_seed(11)
    x = (torch.randn(world * B, 3, size, size, generator=g) * 0.5).clamp(-1, 1).to(dev)
    noise = torch.randn(world * B, 3, size, size, generator=g).to(dev)
    ts = torch.randint(0, 3000, (world * B,), generator=g).to(dev)
    labels = (torch.arange(world * B) % 2).to(dev)
    sl = slice(rank * B, (rank + 1) * B)
    loss = tr.diffusion_and_backward(x[sl], labels[sl], noise=noise[sl], timesteps=ts[sl])
    tr.all_reduce_gradients()
    reduced = tr.grads.clone()
    ok = True
    if rank == 0:
        tr.zero_grad()
        for r in range(world):
            s2 = slice(r * B, (r + 1) * B)
            tr.diffusion_and_backward(x[s2], labels[s2], noise=noise[s2], timesteps=ts[s2])
        ref = tr.grads / world
        err = ((reduced - ref).norm() / ref.norm()).item()
        print(f"[ddpcheck] {args.precision} world {world}: all-reduced gradient vs mean of the shard gradients computed on rank 0: rel L2 {err:.3e} (loss rank0 {loss.item():.5f})")
        # bf16 mode is not bit-reproducible run to run (fp32 atomics reorder, and a last-bit change of a gradient can flip a bf16 rounding):
        # the floor measured here is ~2e-4; the all-reduce itself is exact
        ok = err <= 1e-3
    tr.grads.copy_(reduced)
    tr.optimizer_step()
    ok = _identical(tr, world, "parameters / EMA" + (" / scaler state" if args.precision == "fp16" else "") + " after the optimizer step") and ok
    if args.precision == "fp16":
        # one step in which only the last rank's shard overflows, then a normal one
        bad = noise[sl] * (1e6 if rank == world - 1 else 1.0)
        p_before = tr.params.clone()
        tr.step(x[sl], labels[sl], noise=bad, timesteps=ts[sl], do_unconditional_pass=False)
        st = tr.scaler_state()
        skipped = bool(st["found_inf"]) and torch.equal(tr.params, p_before)
        print(f"[ddpcheck] rank {rank}: overflowing step skipped: {skipped} (scale now {st['scale']}, applied {st['optimizer_steps']}, skipped {st['skipped_steps']})")
        ok = skipped and ok
        ok = _identical(tr, world, "parameters / EMA / scaler state after the skipped step") and ok
        loss = tr.step(x[sl], labels[sl], noise=noise[sl], timesteps=ts[sl], do_unconditional_pass=False)
        applied = not tr.step_was_skipped and math.isfinite(loss.item())
        print(f"[ddpcheck] rank {rank}: following step applied: {applied}")
        ok = applied and ok
        ok = _identical(tr, world, "parameters / EMA / scaler state after the following step") and ok
    flags = torch.tensor([1.0 if ok else 0.0], device=dev)
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    ok = bool(flags.item() == 1.0)
    if rank == 0:
        print("[ddpcheck] OK" if ok else "[ddpcheck] FAILED")
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
