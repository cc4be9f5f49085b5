#!/usr/bin/env python
"""bench.py — images/s of class-conditional DDIM inversion + regeneration (BASELINE.json metric).

One "step" = one class transfer of a whole batch: n inversion steps with the source class + n generation steps with
the target class through the conditional UNet (2n UNet forwards and scheduler updates per image).
Default workload = BASELINE.json configs[1]: small_denoiser UNet, 128x128 RGB, 2 classes, n = 100, batch 256 per GPU,
scheduler 3k_steps_clipping_rescaling; synthetic images, seed-0 random-init weights.

  python bench.py [--gpus N --steps K --warmup W]            our arm (CUDA path through the C ABI)
  python bench.py --impl reference [...]                     reference arm: the CPU oracle on the host cores
  python bench.py --workload cfg [...]                       secondary line (SURVEY §8 row f1): classifier-free-guidance forward
                                                             start, guidance scale 2.5, half of the trajectory skipped (the reference's
                                                             example config), through `_classifier_free_guidance_forward_start`
Under torchrun (N > 1): one rank per GPU, batch-sharded (weak scaling), one final NCCL all-gather of the outputs.
Prints ONE JSON line on rank 0.

  python bench.py --dump-outputs DIR [...]                   also writes what the last timed step returned as DIR/<name>.npy
                                                             (float32, rank 0): inputs and weights are seeded, so two builds run
                                                             with the same arguments can be compared output for output
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GFLOP_PER_IMAGE_FORWARD = {("small_denoiser_config", 128): 285.58, ("small_denoiser_config", 64): 68.98,
                           ("super_small", 128): 74.67, ("super_small", 64): 17.46}   # SURVEY §8(d)
METRIC = "images/sec, DDIM invert+regenerate 128x128 100 steps"
DUMP_MAX_BYTES = 64 * 10**6


def measured_traffic():
    """DRAM bytes per launch of the roofline's kernel class from the committed ncu pass (tools/summarize_profile.py writes
    profiles/traffic.json from `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum` over whole forwards at the bench's
    micro-batch); None when no capture has been committed."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "traffic.json")
    try:
        with open(path) as f:
            return json.load(f)["conv_tcgen05"]
    except Exception:
        return None


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=2)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--workload", default="ddib", choices=["ddib", "cfg", "train", "guided"],
                   help="ddib (default, the BASELINE.json metric); cfg: SURVEY §8 row f1, classifier-free-guidance forward start; "
                        "train: SURVEY §8 row f2, one training step (BASELINE.json configs[3]; default --batch 64 there); "
                        "guided: SURVEY §8 row f4, inversion + gradient-guided generation (use --batch 64)")
    p.add_argument("--train-precision", default="bf16", choices=["bf16", "no"],
                   help="train workload: accelerate-style mixed precision (bf16 tensor-core convolutions) or the fp32 validation path")
    p.add_argument("--guidance-scale", type=float, default=2.5)
    p.add_argument("--frac-diffusion-skipped", type=float, default=0.5)
    p.add_argument("--batch", type=int, default=256, help="images per GPU per step")
    p.add_argument("--size", type=int, default=128)
    p.add_argument("--num-inference-steps", type=int, default=100)
    p.add_argument("--denoiser", default="small_denoiser_config")
    p.add_argument("--scheduler", default="3k_steps_clipping_rescaling")
    p.add_argument("--precision", default=os.environ.get("PHENDIFF_B200_PRECISION", "fp16"), choices=["fp16", "bf16", "fp32"])
    p.add_argument("--microbatch", type=int, default=0)
    p.add_argument("--e2e-steps", type=int, default=3)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--dump-ops", default="", help="write the per-op device-time table (sampled forwards) to this markdown file")
    p.add_argument("--cpu-sample-images", type=int, default=12)   # ~12 s of 16-thread CPU work on the GPU box (4 images took 4.2 s)
    p.add_argument("--cpu-sample-steps", type=int, default=1)
    p.add_argument("--dump-outputs", default="", metavar="DIR",
                   help="write the arrays the last timed step returned to DIR/<name>.npy (float32, at most 64 MB in all; a larger "
                        "array is replaced by a fixed seeded sample of its elements)")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        p.error("--dump-outputs writes the outputs of the CUDA arm; the reference arm only times a sample of the workload")
    return args


def dump_outputs(path, arrays):
    """Writes each named array as float32 `path/<name>.npy`.  An array larger than its share of DUMP_MAX_BYTES is replaced by
    the elements at a fixed set of flat positions (numpy seed 0, sorted), the same positions in every run of the same shape."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    cap = (DUMP_MAX_BYTES // len(arrays) - 4096) // 4        # 4 KB per file left for the .npy header
    for name, a in arrays.items():
        a = np.asarray(a.detach().float().cpu() if hasattr(a, "detach") else a, dtype=np.float32)
        if a.size > cap:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        np.save(os.path.join(path, f"{name}.npy"), a)


def pil_stack(imgs):
    """PIL images (what the drop-in calls return) as one (B, H, W, C) array of their 0..255 values."""
    import numpy as np

    return np.stack([np.asarray(im) for im in imgs])


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
        return {"tflops": d["bf16_tflops_sustained"], "tflops_burst": d["bf16_tflops"], "hbm_gbs": d["hbm_gbs"], "src": "measured"}
    except Exception:
        return {"tflops": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


def make_inputs(batch, size, rank):
    import torch

    g = torch.Generator().manual_seed(1234 + rank)
    x = (torch.randn(batch, 3, size, size, generator=g) * 0.5).clamp(-1, 1)
    src = torch.arange(batch) % 2
    return x, src, 1 - src


def oracle_pipe(args):
    import torch
    from oracle import OracleCondUNet2D, OracleDDIMScheduler, OraclePipeline
    from phendiff_b200.reference_configs import DENOISER_CONFIGS, SCHEDULER_CONFIGS

    torch.manual_seed(0)
    unet = OracleCondUNet2D(**dict(DENOISER_CONFIGS[args.denoiser], sample_size=args.size)).eval()
    return OraclePipeline(unet, OracleDDIMScheduler.from_config(SCHEDULER_CONFIGS[args.scheduler]))


def cpu_sample(args, pipe=None, images=None, steps=None):
    """Time the oracle (CPU restatement of the reference's diffusers path) on a BOUNDED sample of the same workload and
    extrapolate linearly in steps: images/s = images / (t_sample * n / steps)."""
    import torch
    from oracle import oracle_ddib

    images = images or args.cpu_sample_images
    steps = steps or args.cpu_sample_steps
    torch.set_num_threads(os.cpu_count() or 1)
    pipe = pipe or oracle_pipe(args)
    x, src, tgt = make_inputs(images, args.size, 0)
    t0 = time.perf_counter()
    oracle_ddib(pipe, x, src, tgt, steps, return_raw=True)
    dt = time.perf_counter() - t0
    full = dt * args.num_inference_steps / steps
    return {"value": images / full, "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{images} images x ({steps}+{steps}) DDIM steps at {args.size}x{args.size} fp32 on the CPU oracle "
                      f"({dt:.1f} s), extrapolated linearly to ({args.num_inference_steps}+{args.num_inference_steps}) steps",
            "seconds": dt, "cpu": cpu_model()}


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_config0(args):
    """BASELINE.json configs[0] MEASURED end to end (no extrapolation): the reference's CPU-runnable case — the same denoiser
    at 64x64, batch 4, 10 + 10 DDIM steps — through the CPU oracle on this box's host cores (BASELINE.md §4)."""
    import copy

    import torch
    from oracle import oracle_ddib

    a = copy.copy(args)
    a.size = 64
    torch.set_num_threads(os.cpu_count() or 1)
    pipe = oracle_pipe(a)
    x, src, tgt = make_inputs(4, 64, 0)
    oracle_ddib(pipe, x[:1], src[:1], tgt[:1], 1, return_raw=True)
    t0 = time.perf_counter()
    oracle_ddib(pipe, x, src, tgt, 10, return_raw=True)
    dt = time.perf_counter() - t0
    return {"config": f"{args.denoiser} @64x64, batch 4, 10+10 DDIM steps (BASELINE.json configs[0]), measured whole",
            "seconds": dt, "images_per_s": 4 / dt, "cores": torch.get_num_threads(), "cpu": cpu_model()}


def cpu_train_sample(args, images=4, steps=2):
    """CPU baseline of the training step (SURVEY §8 row f2): the oracle UNet under torch.autograd + torch.optim.AdamW + clip, fp32, all host
    threads — the reference's own step (utils_training.py:374-456) minus accelerate — on a bounded batch."""
    import torch
    import torch.nn.functional as F
    from oracle import OracleCondUNet2D, OracleDDIMScheduler
    from phendiff_b200.reference_configs import DENOISER_CONFIGS, SCHEDULER_CONFIGS

    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    unet = OracleCondUNet2D(**dict(DENOISER_CONFIGS[args.denoiser], sample_size=args.size))
    sched = OracleDDIMScheduler.from_config(SCHEDULER_CONFIGS[args.scheduler])
    opt = torch.optim.AdamW(unet.parameters(), lr=1e-4, betas=(0.95, 0.999), weight_decay=1e-6, eps=1e-8)
    x, labels, _ = make_inputs(images, args.size, 0)
    g = torch.Generator().manual_seed(7)

    def step():
        noise = torch.randn(x.shape, generator=g)
        t = torch.randint(0, sched.config.num_train_timesteps, (images,), generator=g)
        noisy = sched.add_noise(x, noise, t)
        target = noise if sched.config.prediction_type == "epsilon" else sched.get_velocity(x, noise, t)
        loss = F.mse_loss(unet(noisy, t, class_labels=labels).sample, target)
        opt.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(unet.parameters(), 1.0)
        opt.step()
        return float(loss)

    step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return {"value": images * steps / dt, "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{steps} training steps of batch {images} at {args.size}x{args.size} fp32 on the CPU oracle (autograd + clip + AdamW; {dt:.1f} s)",
            "seconds": dt, "cpu": cpu_model()}


def run_reference_train(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals, secs = [], 0.0
    for _ in range(max(1, args.steps)):
        r = cpu_train_sample(args)
        vals.append(r["value"]); secs += r["seconds"]
    v = sum(vals) / len(vals)
    r["value"] = v
    line = {"impl": "reference", "metric": f"images/sec, training step {args.size}x{args.size} (forward + backward + gradient all-reduce + clip + AdamW + EMA)",
            "value": v, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * secs / max(args.steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32",
            "data": "synthetic", "config": {"workload": f"CondUNet2D {args.denoiser} {args.size}x{args.size} RGB, 2 classes, training step (CPU sample: batch 4)"},
            "cpu_baseline": r, "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path.  diffusers 0.18.2 (where its arithmetic lives) is
    not installable here, so this is the oracle port; every 'step' is a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    pipe = oracle_pipe(args)
    for _ in range(min(args.warmup, 1)):
        cpu_sample(args, pipe, 1, 1)
    vals, secs = [], 0.0
    for _ in range(args.steps):
        r = cpu_sample(args, pipe)
        vals.append(r["value"]); secs += r["seconds"]
    v = sum(vals) / len(vals)
    base = cpu_sample(args, pipe)
    base["value"] = v
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * secs / max(args.steps, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": workload_config(args, None), "cpu_baseline": base,
            "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(args, info):
    c = {"workload": f"CondUNet2D {args.denoiser} {args.size}x{args.size} RGB, 2 classes, DDIM inversion+class-transfer "
                     f"{args.num_inference_steps}+{args.num_inference_steps} steps, batch {args.batch}/GPU "
                     f"(BASELINE.json configs[1]/[2])",
         "scheduler": args.scheduler, "inverse_scheduler_variant": "diffusers 0.18.2", "global_batch": args.batch * args.gpus,
         "parallelism": f"batch-sharded x{args.gpus}, no data-path collective, one final all-gather",
         "l2": "activations per pass (GBs) exceed the 126 MB L2; a 256 MB buffer is also rewritten between timed steps"}
    if info:
        c.update(info)
    return c


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (our arm) needs a GPU: there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    import __graft_entry__ as ge

    ge.build()
    from phendiff_b200 import ConditionalDDIMPipeline, CustomCondUNet2DModel, DDIMScheduler, _ddib, ddib_transfer
    from phendiff_b200.reference_configs import DENOISER_CONFIGS, SCHEDULER_CONFIGS
    from phendiff_b200.sharding import gather_outputs

    torch.manual_seed(0)
    cfg = dict(DENOISER_CONFIGS[args.denoiser], sample_size=args.size)
    unet = CustomCondUNet2DModel.from_config(cfg, precision=args.precision, max_microbatch=args.microbatch)
    pipe = ConditionalDDIMPipeline(unet.to(dev), DDIMScheduler.from_config(SCHEDULER_CONFIGS[args.scheduler]))
    n = args.num_inference_steps
    x_host, src, tgt = make_inputs(args.batch, args.size, rank)
    x_host = x_host.pin_memory()
    x_dev, src_d, tgt_d = x_host.to(dev), src.to(dev), tgt.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    total = args.batch * world

    if args.workload == "cfg":
        return run_cfg(args, pipe, unet, x_host, x_dev, tgt, tgt_d, dev, rank, world, local)
    if args.workload == "train":
        return run_train(args, pipe, unet, x_host, x_dev, src, src_d, dev, rank, world, local)
    if args.workload == "guided":
        return run_guided(args, pipe, unet, x_host, x_dev, src, src_d, tgt, tgt_d, dev, rank, world, local)

    def step():
        out = ddib_transfer(pipe, x_dev, src_d, tgt_d, n)
        if world > 1:
            out = gather_outputs(out, total)   # the only collective: final NCCL all-gather of the outputs
        return out

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    sync()
    l0 = unet.launch_count()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    unet.profile_begin(every_n=61, max_samples=48)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync()
    e0.record()
    for _ in range(args.steps):
        flush.fill_(1)            # L2 flush between timed iterations
        out = step()
    e1.record()
    sync()
    ms = e0.elapsed_time(e1)
    prof = unet.profile_end()
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"images": out})
    if rank == 0 and args.dump_ops:
        ops = unet.profile_ops()
        tot = sum(o["ms"] for o in ops) or 1.0
        with open(args.dump_ops, "w") as f:
            f.write(f"# per-op device time of one UNet forward (micro-batch {unet.plan_info()['microbatch']}, {args.size}x{args.size}, {args.precision}; "
                    f"CUDA events, mean of {prof['samples']} sampled forwards inside the timed region)\n\n")
            f.write("| # | op | class | ms | share | GFLOP | TFLOP/s |\n|---:|---|---|---:|---:|---:|---:|\n")
            for i, o in enumerate(ops):
                tf = o["flops"] / (o["ms"] * 1e-3) / 1e12 if o["ms"] > 0 and o["flops"] > 0 else 0.0
                f.write(f"| {i} | {o['name']} | {o['cls']} | {o['ms']:.4f} | {o['ms'] / tot:.3f} | {o['flops'] / 1e9:.1f} | {tf:.0f} |\n")
            f.write(f"\ntotal {tot:.3f} ms per forward\n")
    clocks = sampler.stop() if rank == 0 else None
    launches = unet.launch_count() - l0
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = total * args.steps / (ms / 1000.0)

    # end-to-end through the public drop-in call: pinned host images in, PIL images out (H2D + D2H inside the timing)
    e2e_steps = max(1, min(args.e2e_steps, args.steps))
    sync()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        imgs = _ddib(pipe, x_host, src, tgt, n)
        assert len(imgs) == args.batch
    sync()
    t_e2e = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_value = total * e2e_steps / float(t_e2e.item())
    h2d = x_host.numel() * 4 + src.numel() * 8 + tgt.numel() * 8
    d2h = args.batch * args.size * args.size * 3 * 4

    if rank == 0:
        pk = peaks()
        gf = GFLOP_PER_IMAGE_FORWARD.get((args.denoiser, args.size))
        tc = prof["conv_tcgen05"]
        achieved = tc["flops"] / (tc["ms"] * 1e-3) / 1e12 if tc["ms"] > 0 else 0.0
        tot_ms = sum(v["ms"] for k, v in prof.items() if isinstance(v, dict))
        roof = {"bound": "tensor", "achieved": achieved, "peak": pk["tflops"], "unit": "TFLOP/s",
                "frac": achieved / pk["tflops"] if pk["tflops"] else None, "traffic": None,
                "kernel": "conv_halo_kernel / conv_tc_kernel (tcgen05 implicit-GEMM conv/linear class)", "peak_source": pk["src"] + " sustained bf16 cuBLAS",
                "avg_launch_ms": tc["ms"] / tc["launches"] if tc["launches"] else None,
                "kernel_share_of_step": tc["ms"] / tot_ms if tot_ms else None,
                "share_by_class": {k: (v["ms"] / tot_ms if tot_ms else None) for k, v in prof.items() if isinstance(v, dict)},
                "sampled_forwards": prof["samples"]}
        tr = measured_traffic()
        if tr:
            roof["traffic"] = tr["dram_bytes_per_launch"]
            roof["traffic_note"] = tr["note"]
        if gf:
            model_tflops = value / world * 2 * n * gf / 1e3      # per GPU: the peaks below are single-GPU figures
            roof["whole_path_tflops"] = model_tflops
            roof["whole_path_frac_of_measured"] = model_tflops / pk["tflops"]
            roof["whole_path_frac_of_nominal_2250"] = model_tflops / 2250.0
        line = {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": args.precision, "data": "synthetic", "config": workload_config(args, unet.plan_info()),
                "clocks": clocks, "gpu_launches": launches,
                "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "steps": e2e_steps, "api": "phendiff_b200._ddib(pipe, pinned_host_images, src, tgt, n) -> PIL images"},
                "roofline": roof}
        if world == 1 and not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpu_sample(args)
                line["cpu_baseline"]["config0_measured"] = cpu_config0(args)
            except Exception as ex:  # pragma: no cover
                line["cpu_baseline"] = {"error": repr(ex)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_cfg(args, pipe, unet, x_host, x_dev, tgt, tgt_d, dev, rank, world, local):
    """Secondary workload (SURVEY §8 row f1; reference utils_Img2Img.py:615-648 with the example config's guidance_scale 2.5 /
    frac_diffusion_skipped 0.5): forward-noise the images to the middle of the trajectory, then per kept step ONE pass of the UNet
    over 2B images (conditional samples + their unconditional copies) whose conv_out epilogue applies the guidance combine and
    the DDIM update (`pd_cfg_transfer`).
    Both figures go through the drop-in call and end in PIL images; `value` starts from device-resident images and is timed
    with CUDA events, `e2e` starts from pinned host images and is timed on the host clock."""
    import torch
    import torch.distributed as dist
    from types import SimpleNamespace as NS

    from phendiff_b200 import _classifier_free_guidance_forward_start as cfg_start

    n = args.num_inference_steps
    cfg = NS(class_transfer_method=NS(classifier_free_guidance_forward_start=NS(
        guidance_scale=args.guidance_scale, frac_diffusion_skipped=args.frac_diffusion_skipped)))
    pipe.set_progress_bar_config(disable=True)
    pipe.scheduler.set_timesteps(n)
    kept = int((pipe.scheduler.timesteps <= pipe.scheduler.config.num_train_timesteps * (1 - args.frac_diffusion_skipped)).sum())
    total = args.batch * world
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        cfg_start(pipe, x_dev, tgt_d, cfg, n)
    sync()
    l0 = unet.launch_count()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        flush.fill_(1)
        imgs = cfg_start(pipe, x_dev, tgt_d, cfg, n)
    e1.record()
    sync()
    assert len(imgs) == args.batch
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"images": pil_stack(imgs)})
    # UNet kernels (counted by the library: the guidance combine and the scheduler update live in conv_out's epilogue on the fused
    # route, `pd_cfg_transfer`) + per call: add_noise, denorm
    launches = unet.launch_count() - l0 + args.steps * 2
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = total * args.steps / (ms / 1000.0)
    sync()
    t0 = time.perf_counter()
    imgs = cfg_start(pipe, x_host, tgt, cfg, n)
    sync()
    t_e2e = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    if rank == 0:
        pk = peaks()
        gf = GFLOP_PER_IMAGE_FORWARD.get((args.denoiser, args.size))
        line = {"metric": f"images/sec, classifier-free-guidance forward-start class transfer {args.size}x{args.size}, "
                          f"{kept} of {n} steps, 2 UNet forwards per step",
                "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": args.precision, "data": "synthetic",
                "config": dict(workload_config(args, unet.plan_info()),
                               workload=f"CondUNet2D {args.denoiser} {args.size}x{args.size} RGB, 2 classes, CFG forward start "
                                        f"(guidance_scale {args.guidance_scale}, frac_diffusion_skipped {args.frac_diffusion_skipped}, "
                                        f"{n} inference steps -> {kept} kept), batch {args.batch}/GPU (SURVEY §8 row f1)"),
                "clocks": clocks, "gpu_launches": launches,
                "e2e": {"value": total / float(t_e2e.item()), "unit": "images/s",
                        "h2d_bytes_per_step": x_host.numel() * 4 + tgt.numel() * 8,
                        "d2h_bytes_per_step": args.batch * args.size * args.size * 3 * 4, "steps": 1,
                        "api": "phendiff_b200._classifier_free_guidance_forward_start(pipe, pinned_host_images, tgt, cfg, n) -> PIL images"}}
        if gf:
            tf = value / world * 2 * kept * gf / 1e3
            line["roofline"] = {"bound": "tensor", "achieved": tf, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": tf / pk["tflops"],
                                "traffic": None, "kernel": "whole path (2 x kept UNet forwards per image, SURVEY §8d algorithmic FLOPs)",
                                "peak_source": pk["src"] + " sustained bf16 cuBLAS"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_guided(args, pipe, unet, x_host, x_dev, src, src_d, tgt, tgt_d, dev, rank, world, local):
    """SURVEY §8 row f4: `_linear_interp_custom_guidance_inverted_start` (utils_Img2Img.py:651-760) with the example config's p = 2,
    guidance_loss_scale = 1e-3: n inversion steps on the fused route, then n guided steps, each = UNet forward with saved activations +
    Lp-loss gradient + input-gradient-only backward (bf16 tensor-core mode) + gradient step + scheduler update."""
    import torch
    import torch.distributed as dist
    from types import SimpleNamespace as NS

    from phendiff_b200 import _linear_interp_custom_guidance_inverted_start as guided

    n = args.num_inference_steps
    cfg = NS(class_transfer_method=NS(linear_interp_custom_guidance_inverted_start=NS(p=2, guidance_loss_scale=1e-3)))
    total = args.batch * world

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(min(args.warmup, 1)):
        guided(pipe, x_dev, src_d, tgt_d, cfg, 2)
    sync()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        imgs = guided(pipe, x_dev, src_d, tgt_d, cfg, n)
    e1.record()
    sync()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"images": pil_stack(imgs)})
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = total * args.steps / (ms / 1000.0)
    sync()
    t0 = time.perf_counter()
    imgs = guided(pipe, x_host, src, tgt, cfg, n)
    sync()
    t_e2e = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    if rank == 0:
        assert len(imgs) == args.batch
        line = {"metric": f"images/sec, inversion + gradient-guided generation {args.size}x{args.size}, {n}+{n} steps",
                "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "fp16 (inversion) + bf16 mixed precision (guided steps: forward + input-gradient backward)", "data": "synthetic",
                "config": {"workload": f"CondUNet2D {args.denoiser} {args.size}x{args.size} RGB, 2 classes, linear_interp_custom_guidance_inverted_start "
                                       f"(p = 2, guidance_loss_scale = 1e-3), {n}+{n} steps, batch {args.batch}/GPU (SURVEY §8 row f4)",
                           "scheduler": args.scheduler, "global_batch": total},
                "clocks": clocks, "gpu_launches": None,
                "e2e": {"value": total / float(t_e2e.item()), "unit": "images/s", "h2d_bytes_per_step": x_host.numel() * 4 + src.numel() * 16,
                        "d2h_bytes_per_step": args.batch * args.size * args.size * 3 * 4, "steps": 1,
                        "api": "phendiff_b200._linear_interp_custom_guidance_inverted_start(pipe, pinned_host_images, src, tgt, cfg, n) -> PIL images"}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_train(args, pipe, unet, x_host, x_dev, labels, labels_d, dev, rank, world, local):
    """SURVEY §8 row f2 / BASELINE.json configs[3]: one iteration of the reference's training loop body
    (utils_training.py:244-456 + :552-556) through `phendiff_b200.training.DenoiserTrainer.step`: noise / timestep sampling,
    add_noise, forward + backward of the UNet, NCCL all-reduce of the flat gradient vector (N > 1), clip 1.0 + AdamW + EMA.
    The backward pass computes in fp32 on CUDA cores (the validated path; tensor-core dgrad / wgrad is the next stage), so
    `dtype` says fp32 whatever --precision asks for."""
    import torch
    import torch.distributed as dist

    from phendiff_b200.training import DenoiserTrainer

    trainer = DenoiserTrainer(unet, pipe.scheduler, args.batch, args.size, learning_rate=1e-4, use_ema=True, mixed_precision=args.train_precision)
    total = args.batch * world
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    g = torch.Generator(device=dev).manual_seed(7 + rank)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(x):
        noise = torch.randn(x_dev.shape, device=dev, generator=g)
        ts = torch.randint(0, pipe.scheduler.config.num_train_timesteps, (args.batch,), device=dev, generator=g)
        return trainer.step(x, labels_d, noise=noise, timesteps=ts, do_unconditional_pass=False)

    for _ in range(args.warmup):
        step(x_dev)
    sync()
    l0 = trainer.launch_count()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        flush.fill_(1)
        loss = step(x_dev)
    e1.record()
    sync()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:      # the loss the step returned and the parameters it left (before the e2e steps move them)
        dump_outputs(args.dump_outputs, {"loss": loss, "parameters": trainer.params})
    launches = trainer.launch_count() - l0 + args.steps * 4      # + add_noise, adamw (memset + sumsq + update)
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = total * args.steps / (ms / 1000.0)
    # end to end: pinned host images -> device every step, loss read back on the host every step
    sync()
    t0 = time.perf_counter()
    e2e_steps = max(1, args.e2e_steps)
    for _ in range(e2e_steps):
        lv = step(x_host.to(dev, non_blocking=True)).item()
    sync()
    t_e2e = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    if rank == 0:
        pk = peaks()
        gf = GFLOP_PER_IMAGE_FORWARD.get((args.denoiser, args.size))
        line = {"metric": f"images/sec, training step {args.size}x{args.size} (forward + backward + gradient all-reduce + clip + AdamW + EMA)",
                "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16" if args.train_precision == "bf16" else "fp32", "data": "synthetic",
                "config": {"workload": f"CondUNet2D {args.denoiser} {args.size}x{args.size} RGB, 2 classes, training step, batch "
                                       f"{args.batch}/GPU (BASELINE.json configs[3]; SURVEY §8 row f2), scheduler {args.scheduler}",
                           "global_batch": total, "parallelism": f"data-parallel x{world}, one all-reduce of the flat fp32 gradient vector"
                                                                 f" ({trainer.numel * 4 / 1e6:.1f} MB)",
                           "parameters": trainer.numel, "workspace_gb": trainer.workspace_bytes / 1e9,
                           "mixed_precision": args.train_precision, "tensor_core_layers_since_start": trainer.tensor_core_counts(),
                           "l2": "activations (GBs) exceed the 126 MB L2; a 256 MB buffer is also rewritten between timed steps",
                           "final_loss": float(loss.item()), "last_e2e_loss": lv},
                "clocks": clocks, "gpu_launches": launches,
                "e2e": {"value": total * e2e_steps / float(t_e2e.item()), "unit": "images/s",
                        "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": 4, "steps": e2e_steps,
                        "api": "phendiff_b200.training.DenoiserTrainer.step(pinned_host_images.to(dev), labels) -> loss.item()"}}
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_train_sample(args)
        if gf:
            tf = value / world * 3 * gf / 1e3     # forward + dgrad + wgrad = 3 x the forward's algorithmic FLOPs
            line["roofline"] = {"bound": "tensor", "achieved": tf, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": tf / pk["tflops"],
                                "traffic": None, "kernel": "whole step (3 x forward algorithmic FLOPs per image: forward + dgrad + wgrad)",
                                "peak_source": pk["src"] + " sustained bf16 cuBLAS"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference_train(args) if args.workload == "train" else run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
