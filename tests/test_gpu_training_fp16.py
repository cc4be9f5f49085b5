"""Training step under mixed_precision="fp16" (the reference's launch scripts: accelerate --mixed_precision=fp16, which wraps the loop
in torch.amp.GradScaler) against torch on the oracle.

fp16 operands on the tensor cores need the loss scale: the loss gradient of a 64 x 128^2 batch is ~6e-7 per element, below fp16's
smallest normal number.  The backward starts from S * d(loss), so gradients come out scaled; `pd_adamw_step_scaled` unscales them,
skips the step when any is inf / NaN, and updates S, all on the device."""
import math

import pytest
import torch

from phendiff_b200.reference_configs import SCHEDULER_CONFIGS
from tests.test_gpu_training import _inputs, _oracle_loss, _setup
from tests.util import psnr, synth_images

pytestmark = pytest.mark.gpu


def _grad_errors(named, ref, divisor=1.0):
    """(whole-vector relative L2, (worst per-tensor relative L2, name)) of `named` / divisor against `ref`, measured as
    test_bf16_tensor_core_gradients measures them (tensors with a numerically zero true gradient against the overall scale)."""
    rms_all = math.sqrt(sum(r.double().pow(2).sum().item() for r in ref.values()) / sum(r.numel() for r in ref.values()))
    worst, num, den = (0.0, None), 0.0, 0.0
    for name, g in named:
        g, r = g / divisor, ref[name]
        e = ((g - r).norm() / max(r.norm().item(), 1e-2 * rms_all * math.sqrt(r.numel()))).item()
        num += (g - r).double().pow(2).sum().item()
        den += r.double().pow(2).sum().item()
        if e > worst[0]:
            worst = (e, name)
    return math.sqrt(num / den), worst


def _state(t):
    from phendiff_b200 import _lib

    return _lib.GradScalerState.from_buffer_copy(t.cpu().numpy().tobytes())


@pytest.mark.parametrize("tc_mask,B,size", [(1, 2, 64), (2, 2, 64), (4, 2, 64), (8, 2, 64), (127, 2, 64), (127, 1, 128)])
def test_fp16_tensor_core_gradients(tc_mask, B, size, monkeypatch):
    """fp16 operands on every tensor-core piece the mask selects (as in test_bf16_tensor_core_gradients), gradients / S at S = 2^16
    against fp32 autograd, at bf16's bars."""
    monkeypatch.setenv("PHENDIFF_B200_TRAIN_TC", str(tc_mask))
    oracle, model, osched, sched, Trainer = _setup("small_denoiser_config", size, B, "1k_epsilon_pred")
    x, labels, noise, timesteps = _inputs(B, size, seed=9)
    loss_ref, out_ref = _oracle_loss(oracle, osched, x, labels, noise, timesteps, "epsilon", False)
    loss_ref.backward()
    trainer = Trainer(model, sched, B, size, mixed_precision="fp16", grad_scaler_kwargs={"init_scale": 2.0 ** 16})
    loss, out = trainer.diffusion_and_backward(x, labels, noise=noise, timesteps=timesteps, return_model_output=True)
    S = trainer.get_scale()
    assert S == 2.0 ** 16
    counts = trainer.tensor_core_counts()
    if tc_mask & 1:
        assert counts["conv_forward"] > 50, counts
    if tc_mask & 4:
        assert counts["conv_wgrad"] > 50, counts
    fwd_err = (out - out_ref).abs().max().item() / out_ref.abs().max().item()
    ref = {n: p.grad for n, p in oracle.named_parameters()}
    total, worst = _grad_errors(trainer.named_gradients(), ref, S)
    print(f"fp16 tc_mask={tc_mask} B={B} @{size}: {counts}; forward max err {fwd_err:.2e}; loss {loss.item():.6f} vs {loss_ref.item():.6f}; "
          f"whole-gradient rel L2 {total:.2e}; worst tensor {worst[1]} {worst[0]:.2e}")
    assert fwd_err <= 2e-2
    assert abs(loss.item() - loss_ref.item()) <= 1e-2 * abs(loss_ref.item())
    assert total <= 1e-2
    assert worst[0] <= 3e-2, worst


def test_loss_scale_is_linear_and_invisible_in_the_loss():
    """The same inputs at S = 2^8 and 2^16: the loss is the unscaled one (it is a float atomic reduction, so two runs may differ in
    the last bits whatever S is), and the unscaled gradients agree at the bars above."""
    B, size = 2, 64
    runs = {}
    for S in (2.0 ** 8, 2.0 ** 16):
        oracle, model, osched, sched, Trainer = _setup("small_denoiser_config", size, B, "1k_epsilon_pred")
        x, labels, noise, timesteps = _inputs(B, size, seed=9)
        trainer = Trainer(model, sched, B, size, mixed_precision="fp16", grad_scaler_kwargs={"init_scale": S})
        loss = trainer.diffusion_and_backward(x, labels, noise=noise, timesteps=timesteps)
        runs[S] = (loss.item(), {n: g / S for n, g in trainer.named_gradients()})
    (l8, g8), (l16, g16) = runs[2.0 ** 8], runs[2.0 ** 16]
    total, worst = _grad_errors(g8.items(), g16)
    print(f"S = 2^8 vs 2^16: loss {l8!r} vs {l16!r} (bit-identical: {l8 == l16}); unscaled gradients rel L2 {total:.2e}, worst {worst[1]} {worst[0]:.2e}")
    assert abs(l8 - l16) <= 1e-6 * abs(l16)
    assert total <= 1e-2
    assert worst[0] <= 3e-2, worst


def test_adamw_step_scaled_matches_grad_scaler():
    """pd_adamw_step_scaled step for step against torch.amp.GradScaler(init_scale=16, growth_interval=2) + unscale_ + clip_grad_norm_
    + AdamW + the EMAModel recurrence, with an inf in the gradients at step 2 and a NaN at step 5."""
    from phendiff_b200 import _lib
    from phendiff_b200.training import ema_decay_at

    torch.manual_seed(3)
    n = 100_003
    p0 = torch.randn(n, device="cuda")
    p, ema = p0.clone(), p0.clone()
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    ref = torch.nn.Parameter(p0.clone())
    opt = torch.optim.AdamW([ref], lr=3e-3, betas=(0.95, 0.999), weight_decay=1e-2, eps=1e-8)
    scaler = torch.amp.GradScaler("cuda", init_scale=16.0, growth_interval=2)
    ref_ema = p0.clone()
    state = torch.frombuffer(bytearray(bytes(_lib.GradScalerState(scale=16.0))), dtype=torch.uint8).cuda()
    scratch, norm = torch.zeros(_lib.PD_ADAMW_SCALED_SCRATCH_FLOATS, device="cuda"), torch.zeros(1, device="cuda")
    for step in range(1, 9):
        S = scaler.scale(torch.ones((), device="cuda"))          # the scale this step's backward would have used
        g = torch.randn(n, device="cuda") * (0.1 * step) * S
        if step == 2:
            g[12345] = float("inf")
        if step == 5:
            g[777] = float("nan")
        ref.grad = g.clone()
        scaler.unscale_(opt)
        ref_norm = torch.nn.utils.clip_grad_norm_([ref], 1.0)
        scaler.step(opt)
        scaler.update()
        decay = ema_decay_at(step, max_decay=0.9999, inv_gamma=1.0, power=0.75)
        ref_ema.sub_((1 - decay) * (ref_ema - ref.data))
        before = (p.clone(), m.clone(), v.clone())
        _lib.check(_lib.lib().pd_adamw_step_scaled(_lib.ptr(p), _lib.ptr(g), _lib.ptr(m), _lib.ptr(v), _lib.ptr(ema), n, 3e-3, 0.95, 0.999, 1e-8,
                                                  1e-2, 1.0, decay, _lib.ptr(state), 2.0, 0.5, 2, _lib.ptr(scratch), _lib.ptr(norm),
                                                  _lib.current_stream()))
        st = _state(state)
        skipped = step in (2, 5)
        assert st.found_inf == int(skipped), step
        assert st.scale == scaler.get_scale() and st.growth_tracker == scaler._growth_tracker.item(), (step, st.scale, st.growth_tracker)
        if skipped:
            assert torch.equal(p, before[0]) and torch.equal(m, before[1]) and torch.equal(v, before[2]), step
            assert not math.isfinite(norm.item())
        else:
            assert abs(norm.item() - ref_norm.item()) <= 1e-5 * ref_norm.item(), step
        ost = opt.state[ref]
        assert (p - ref.data).abs().max().item() <= 2e-6, step
        assert (m - ost["exp_avg"]).abs().max().item() <= 2e-6, step
        assert (v - ost["exp_avg_sq"]).abs().max().item() <= 2e-6, step
        assert (ema - ref_ema).abs().max().item() <= 2e-6, step
    assert st.optimizer_steps == int(opt.state[ref]["step"].item()) == 6 and st.skipped_steps == 2


def test_trainer_overflow_skips_the_step_without_a_host_wait():
    """init_scale = 2^40 overflows fp16 in the backward: one step must be skipped (parameters and moments untouched, the EMA still
    steps), the scale halves, the applied-step counter stays at 0, and `optimizer_step` returns without waiting for the device."""
    from phendiff_b200.training import ema_decay_at

    B, size = 2, 64
    oracle, model, osched, sched, Trainer = _setup("small_denoiser_config", size, B, "1k_epsilon_pred")
    x, labels, noise, timesteps = _inputs(B, size, seed=9)
    trainer = Trainer(model, sched, B, size, use_ema=True, mixed_precision="fp16", grad_scaler_kwargs={"init_scale": 2.0 ** 40},
                      lr_lambda=lambda k: 1.0 / (1 + k))
    trainer.ema.add_(0.01)                        # the EMA step toward the (unchanged) parameters is then visible
    p0, m0, v0, e0 = trainer.params.clone(), trainer.exp_avg.clone(), trainer.exp_avg_sq.clone(), trainer.ema.clone()
    trainer.diffusion_and_backward(x, labels, noise=noise, timesteps=timesteps)
    trainer.all_reduce_gradients()
    torch.cuda.synchronize()
    torch.cuda._sleep(int(2e9))                   # ~1 s of device work queued ahead of the optimizer pass
    trainer.optimizer_step()
    device_still_busy = not torch.cuda.current_stream().query()
    torch.cuda.synchronize()
    assert device_still_busy, "optimizer_step waited for the device"
    assert torch.equal(trainer.params, p0) and torch.equal(trainer.exp_avg, m0) and torch.equal(trainer.exp_avg_sq, v0)
    decay = ema_decay_at(1)
    assert torch.allclose(trainer.ema, e0 - (1 - decay) * (e0 - p0), rtol=0, atol=1e-6)
    assert not torch.equal(trainer.ema, e0)
    assert trainer.get_scale() == 2.0 ** 39 and trainer.step_was_skipped
    assert trainer.global_step == 1 and trainer.optimizer_steps == 0 and trainer.current_lr() == trainer.lr
    assert trainer.grads.abs().max().item() == 0.0
    assert not math.isfinite(trainer.grad_norm.item())
    st = trainer.scaler_state()
    assert st["skipped_steps"] == 1 and st["growth_tracker"] == 0


def test_fp16_training_reduces_loss():
    """12 fp16 steps on one fixed batch at small_denoiser_config 64^2: the loss stays finite and drops below 0.7 x the first.
    lr 2.5e-4: at 2e-3 this four-image overfit oscillates in bf16 as well, and in fp16 its forward pass overflows after six steps
    (measured on a B200: the loss turns NaN for good, every later step is skipped), which no loss scale can fix."""
    B, size = 4, 64
    oracle, model, osched, sched, Trainer = _setup("small_denoiser_config", size, B, "1k_epsilon_pred")
    x, labels, noise, timesteps = _inputs(B, size, seed=11)
    trainer = Trainer(model, sched, B, size, learning_rate=2.5e-4, use_ema=True, mixed_precision="fp16")
    losses = [trainer.step(x, labels, noise=noise, timesteps=timesteps, do_unconditional_pass=False).item() for _ in range(12)]
    st = trainer.scaler_state()
    print(f"fp16 training 12 steps: losses {[round(v, 4) for v in losses]}; skipped steps {st['skipped_steps']}, final scale {st['scale']}")
    assert all(math.isfinite(v) for v in losses), losses
    assert losses[-1] < 0.7 * losses[0], losses
    assert trainer.global_step == 12 and trainer.optimizer_steps == 12 - st["skipped_steps"]


def _pipes(size):
    from oracle import OracleDDIMScheduler, OraclePipeline
    from phendiff_b200 import ConditionalDDIMPipeline, DDIMScheduler
    from tests.util import make_pair

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    sched = "3k_steps_clipping_rescaling"
    oracle, model = make_pair("small_denoiser_config", size, "fp16")
    opipe = OraclePipeline(oracle.cuda(), OracleDDIMScheduler.from_config(SCHEDULER_CONFIGS[sched]))
    return opipe, ConditionalDDIMPipeline(model, DDIMScheduler.from_config(SCHEDULER_CONFIGS[sched]))


def test_fp16_guidance_gradient_first_steps_match_oracle():
    """Gradient-guided generation's engine in fp16 (the reference's autocast type for class transfer), teacher-forced on the oracle's
    images, at the bars test_gpu_guidance.py sets for bf16 (5e-2).  The input gradient is not loss-scaled, as in the reference."""
    import ctypes as C

    from oracle import oracle_custom_guided_generation
    from phendiff_b200 import _lib
    from phendiff_b200.utils_img2img import _guidance_engine

    B, n, size = 2, 3, 64
    opipe, pipe = _pipes(size)
    _, labels = synth_images(B, size, seed=21)
    start = torch.randn(B, 3, size, size, generator=torch.Generator().manual_seed(5)).cuda()
    labels = labels.cuda()
    trace = []
    oracle_custom_guided_generation(opipe, start, labels, 2, 1e-3, n, trace=trace)
    eng = _guidance_engine(pipe, B, size, "fp16")
    pipe.scheduler.set_timesteps(n)
    for (t, images, m_ref, losses_ref, grad_ref) in trace:
        m = eng.forward_only(images, torch.full((B,), float(t), device="cuda"), labels)
        co = pipe.scheduler.step_coeffs(t)
        scratch, losses = torch.zeros(B, device="cuda"), torch.zeros(B, device="cuda")
        dm, dx = torch.empty_like(images), torch.empty_like(images)
        _lib.check(_lib.lib().pd_guidance_lp_grad(C.byref(co), _lib.ptr(images), _lib.ptr(m), _lib.ptr(start), B, images[0].numel(), 2.0,
                                                 _lib.ptr(scratch), _lib.ptr(losses), _lib.ptr(dm), _lib.ptr(dx), _lib.current_stream()))
        grad = dx + eng.input_gradient(dm)
        e_m = (m - m_ref).abs().max().item() / m_ref.abs().max().item()
        e_l = ((losses - losses_ref).abs() / losses_ref).max().item()
        e_g = ((grad - grad_ref).norm() / grad_ref.norm()).item()
        print(f"[guided fp16] t={t}: model output {e_m:.2e}, loss {e_l:.2e}, guidance gradient rel L2 {e_g:.2e}")
        assert e_m <= 5e-2 and e_l <= 5e-2 and e_g <= 5e-2


def test_fp16_guided_transfer_matches_oracle():
    """The whole guided transfer (inversion + gradient-guided generation) with mixed_precision="fp16", free-running: >= 40 dB."""
    from types import SimpleNamespace as NS

    from oracle import oracle_linear_interp_custom_guidance_inverted_start
    from phendiff_b200 import _custom_guided_generation, _inversion

    B, n, size = 2, 5, 64
    opipe, pipe = _pipes(size)
    x, src = synth_images(B, size, seed=33)
    x, src = x.cuda(), src.cuda()
    cfg = NS(class_transfer_method=NS(linear_interp_custom_guidance_inverted_start=NS(p=2, guidance_loss_scale=1e-3)))
    ref = oracle_linear_interp_custom_guidance_inverted_start(opipe, x, src, 1 - src, 2, 1e-3, n)
    inv = _inversion(pipe, x, src, n)
    out = _custom_guided_generation(pipe, inv, 1 - src, cfg, n, mixed_precision="fp16")
    db = psnr(out.clamp(-1, 1), ref.clamp(-1, 1))
    print(f"[guided fp16] transfer {n}+{n} steps: PSNR vs oracle {db:.1f} dB")
    assert db >= 40.0
