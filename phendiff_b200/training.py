"""Training step of the class-conditional denoiser (SURVEY §8 row f2; BASELINE.json configs[3]).

Mirror of the inner step of the reference's `perform_training_epoch` for `model_type == "DDIM"`
(src/utils_training.py:244-456) with the optimizer the reference builds in train.py:279-285 and the diffusers `EMAModel`
it keeps beside it (train.py:223-238, utils_training.py:552-556):

    noise, timesteps          torch.randn / torch.randint                              (utils_training.py:244-252)
    noisy_images              DDIMScheduler.add_noise                                   (:256)
    model_output              denoiser(noisy, timesteps, class_labels | class_emb=0)   (:499-538, `_DDIM_prediction_wrapper`)
    loss                      mse vs noise | SNR-weighted mse vs clean | mse vs velocity (:415-433)
    backward                  accelerator.backward(loss)                                (:436)
    clip                      accelerator.clip_grad_norm_(params, 1.0)                  (:439)
    optimizer / EMA           AdamW.step, lr_scheduler.step, zero_grad, EMAModel.step   (:452-454, :552-556)

Everything between `noisy_images` and the updated parameters runs in the CUDA library: forward + backward of the UNet
(`pd_train_step_grad`) and one fused clip + AdamW + EMA pass over flat vectors (`pd_adamw_step`; under fp16 mixed precision
`pd_adamw_step_scaled`, which adds torch.amp.GradScaler's unscale / skip-on-inf / scale update with the scaler state on the
device).  Parameters, gradients and optimizer state are single flat fp32 tensors in parameter-table order; the module's
`nn.Parameter`s are re-pointed at views of
the flat parameter vector (and their `.grad` at views of the flat gradient vector), so `state_dict()`, `save_pretrained` and a
stock torch optimizer keep working on the same storage.  Under `torch.distributed` the flat gradient vector is averaged with
ONE all-reduce (what DDP does in buckets for the reference, through accelerate).  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Callable, Optional

import torch
import torch.distributed as dist

from . import _lib
from .cond_unet_2d import CustomCondUNet2DModel
from .schedulers import DDIMScheduler
from .sharding import average_gradients


# accelerate's `mixed_precision` names -> pd_train_set_precision
PRECISIONS = {"no": _lib.PD_PREC_FP32, "bf16": _lib.PD_PREC_BF16, "fp16": _lib.PD_PREC_FP16}
# torch.amp.GradScaler's defaults, which accelerate uses for mixed_precision="fp16" unless GradScalerKwargs are given
GRAD_SCALER_DEFAULTS = {"init_scale": 2.0 ** 16, "growth_factor": 2.0, "backoff_factor": 0.5, "growth_interval": 2000}


def ema_decay_at(optimization_step: int, max_decay: float = 0.9999, min_decay: float = 0.0, update_after_step: int = 0,
                 use_ema_warmup: bool = True, inv_gamma: float = 1.0, power: float = 0.75) -> float:
    """diffusers `EMAModel.get_decay` (pinned diffusers 0.18.2, training_utils.py) as the reference configures it
    (train.py:229-236: `use_ema_warmup=True`, decay / inv_gamma / power from the arguments).  Pure host logic."""
    step = max(0, optimization_step - update_after_step - 1)
    if step <= 0:
        return 0.0
    if use_ema_warmup:
        cur = 1 - (1 + step / inv_gamma) ** -power
    else:
        cur = (1 + step) / (10 + step)
    return max(min(cur, max_decay), min_decay)


def training_target(prediction_type: str, clean_images, noise, velocity_fn):
    """Regression target by prediction type (utils_training.py:415-433)."""
    if prediction_type == "epsilon":
        return noise
    if prediction_type == "sample":
        return clean_images
    if prediction_type == "v_prediction":
        return velocity_fn()
    raise ValueError(f"Unsupported prediction type: {prediction_type}")


class DenoiserTrainer:
    """One denoiser, one flat parameter vector, one training step.

    `trainer.step(clean_images, class_labels)` is one iteration of the reference's epoch loop body; the pieces
    (`diffusion_and_backward`, `all_reduce_gradients`, `optimizer_step`) can be called separately (gradient accumulation:
    call the first several times before the other two — gradients accumulate until `zero_grad`).

    `mixed_precision` takes accelerate's names: "no" (fp32 on CUDA cores, the validation path), "bf16" or "fp16" (16-bit operands on
    the tensor cores, fp32 everything else).  "fp16" also scales the loss as accelerate's GradScaler does (`grad_scaler_kwargs`: the
    keys of GRAD_SCALER_DEFAULTS, as in accelerate's GradScalerKwargs): a step whose gradients hold an inf or NaN is skipped and the
    scale backs off.  `global_step` counts every step; `optimizer_steps` only the applied ones, which is what `lr_lambda` receives
    (accelerate's scheduler does not step when the optimizer step was skipped)."""

    def __init__(self, denoiser_model: CustomCondUNet2DModel, noise_scheduler: DDIMScheduler, batch_size: int, resolution: int,
                 learning_rate: float = 1e-4, adam_beta1: float = 0.95, adam_beta2: float = 0.999, adam_weight_decay: float = 1e-6,
                 adam_epsilon: float = 1e-8, max_grad_norm: float = 1.0, use_ema: bool = False, ema_max_decay: float = 0.9999,
                 ema_inv_gamma: float = 1.0, ema_power: float = 0.75, lr_lambda: Optional[Callable[[int], float]] = None,
                 proba_uncond: float = 0.0, mixed_precision: str = "no", shared_seed: int = 0, grad_scaler_kwargs: Optional[dict] = None):
        if mixed_precision not in PRECISIONS:
            raise ValueError(f"mixed_precision must be 'no', 'bf16' or 'fp16' (accelerate's names), not {mixed_precision!r}")
        scaler = None
        if mixed_precision == "fp16":
            unknown = set(grad_scaler_kwargs or {}) - set(GRAD_SCALER_DEFAULTS)
            if unknown:
                raise ValueError(f"grad_scaler_kwargs: unknown keys {sorted(unknown)}; accepted: {sorted(GRAD_SCALER_DEFAULTS)}")
            scaler = dict(GRAD_SCALER_DEFAULTS, **(grad_scaler_kwargs or {}))
            if not (scaler["init_scale"] > 0 and scaler["growth_factor"] > 1.0 and 0.0 < scaler["backoff_factor"] < 1.0
                    and int(scaler["growth_interval"]) >= 1):
                raise ValueError(f"grad_scaler_kwargs: need init_scale > 0, growth_factor > 1, 0 < backoff_factor < 1, growth_interval >= 1; "
                                 f"got {scaler}")
        elif grad_scaler_kwargs is not None:
            raise ValueError("grad_scaler_kwargs applies to mixed_precision='fp16' only")
        self.model = denoiser_model
        self.noise_scheduler = noise_scheduler
        self.batch_size, self.resolution = int(batch_size), int(resolution)
        self.lr, self.betas, self.weight_decay, self.eps = learning_rate, (adam_beta1, adam_beta2), adam_weight_decay, adam_epsilon
        self.max_grad_norm = max_grad_norm
        self.use_ema, self.ema_max_decay, self.ema_inv_gamma, self.ema_power = use_ema, ema_max_decay, ema_inv_gamma, ema_power
        self.lr_lambda = lr_lambda
        self.proba_uncond = proba_uncond
        self._coin = torch.Generator().manual_seed(int(shared_seed))    # must be the same on every rank
        self.global_step = 0            # optimizer steps taken
        self.cur_decay_value = 0.0
        dev = denoiser_model.device
        if dev.type != "cuda":
            raise _lib.PhenDiffB200Error(f"DenoiserTrainer needs the model on a CUDA device, not {dev} (there is no CPU fallback)")
        self.device = dev
        L = _lib.lib()
        with torch.cuda.device(dev):
            h = denoiser_model._ensure_handle()
            t = C.c_void_p()
            _lib.check(L.pd_train_create(h, self.batch_size, self.resolution, self.resolution, C.byref(t)))
            self._t, self._h = t, h
            self.mixed_precision = mixed_precision
            if mixed_precision != "no":
                _lib.check(L.pd_train_set_precision(t, PRECISIONS[mixed_precision]))
            n = C.c_int64()
            _lib.check(L.pd_train_num_params_flat(t, C.byref(n)))
            self.numel = n.value
            self.params = torch.empty(self.numel, device=dev, dtype=torch.float32)
            self.grads = torch.zeros(self.numel, device=dev, dtype=torch.float32)
            self.exp_avg = torch.zeros_like(self.grads)
            self.exp_avg_sq = torch.zeros_like(self.grads)
            # re-point the module's parameters at views of the flat vectors
            named = dict(denoiser_model.named_parameters())
            self._views = {}
            off = C.c_int64()
            for i, (name, shape) in enumerate(denoiser_model._param_table()):
                _lib.check(L.pd_train_param_offset(t, i, C.byref(off)))
                cnt = math.prod(shape)
                p = named[name]
                view = self.params[off.value: off.value + cnt].view(shape)
                view.copy_(p.data.to(device=dev, dtype=torch.float32))
                p.data = view
                p.grad = self.grads[off.value: off.value + cnt].view(shape)
                self._views[name] = (off.value, cnt, tuple(shape))
            self.ema = self.params.clone() if use_ema else None
            ws = C.c_size_t()
            _lib.check(L.pd_train_workspace_bytes(t, C.byref(ws)))
            self.workspace_bytes = ws.value
            self._workspace = torch.empty(ws.value + 256, device=dev, dtype=torch.uint8)
            base = self._workspace.data_ptr()
            self._ws_ptr = (base + 255) // 256 * 256
            _lib.check(L.pd_train_bind(t, C.c_void_p(self._ws_ptr), ws.value))
            self._loss = torch.zeros(1, device=dev, dtype=torch.float32)
            self.grad_norm = torch.zeros(1, device=dev, dtype=torch.float32)
            self._scaler = scaler
            if scaler is None:
                self._scratch = torch.zeros(_lib.PD_ADAMW_SCRATCH_FLOATS, device=dev, dtype=torch.float32)
            else:
                self._scratch = torch.zeros(_lib.PD_ADAMW_SCALED_SCRATCH_FLOATS, device=dev, dtype=torch.float32)
                st = _lib.GradScalerState(scale=float(scaler["init_scale"]))
                self._scaler_state = torch.frombuffer(bytearray(bytes(st)), dtype=torch.uint8).to(dev)
                # the state as the last optimizer pass left it, copied back without a host wait (read once `_scaler_event` completed)
                self._scaler_host = torch.empty(C.sizeof(_lib.GradScalerState), dtype=torch.uint8, pin_memory=True)
                self._scaler_host.copy_(self._scaler_state.cpu())
                self._scaler_event = None
                # GradScalerState.scale is at offset 0: every backward of this handle multiplies the loss gradient by the current S
                _lib.check(L.pd_train_set_loss_scale(t, C.c_void_p(self._scaler_state.data_ptr())))
            self._acp = noise_scheduler.alphas_cumprod.to(device=dev, dtype=torch.float32)
        denoiser_model.mark_dirty()     # the inference handle re-reads the (moved) parameters on its next use

    def __del__(self):
        try:
            t = self.__dict__.get("_t")
            if t is not None:
                _lib.lib().pd_train_destroy(t)
                self._t = None
        except Exception:  # pragma: no cover
            pass

    # ------------------------------------------------------------------------------------------------------------
    def named_gradients(self):
        """(name, gradient view) per parameter.  Under mixed_precision="fp16" the gradients between the backward and `optimizer_step`
        are the SCALED ones (loss scale `get_scale()` times the true gradient), as `param.grad` holds them under torch's GradScaler
        before `unscale_`."""
        for name, (off, cnt, shape) in self._views.items():
            yield name, self.grads[off: off + cnt].view(shape)

    def zero_grad(self):
        self.grads.zero_()

    def tensor_core_counts(self) -> dict:
        a, b = C.c_int64(), C.c_int64()
        _lib.check(_lib.lib().pd_train_tc_counts(self._t, C.byref(a), C.byref(b)))
        return {"conv_forward": a.value, "conv_wgrad": b.value}

    def launch_count(self) -> int:
        n = C.c_int64()
        _lib.check(_lib.lib().pd_train_launch_count(self._t, C.byref(n)))
        return n.value

    # ------------------------------------------------------------------------------------------------------------
    def _axpby(self, a, b, ca, cb):
        out = torch.empty_like(a)
        B = a.shape[0]
        _lib.check(_lib.lib().pd_axpby_per_sample(_lib.ptr(a), _lib.ptr(b), _lib.ptr(ca), _lib.ptr(cb), _lib.ptr(out), B,
                                                  a.numel() // B, _lib.current_stream()))
        return out

    def diffusion_and_backward(self, clean_images: torch.Tensor, class_labels: Optional[torch.Tensor], noise: Optional[torch.Tensor] = None,
                               timesteps: Optional[torch.Tensor] = None, do_unconditional_pass: bool = False,
                               return_model_output: bool = False):
        """Steps 0-3 of the reference's loop body up to (not including) the clip: samples noise and timesteps unless given,
        forms the noisy images and the target, runs forward + backward.  Gradients ACCUMULATE into `self.grads`.
        Returns the loss as a 1-element device tensor (no host sync), plus the model output if asked."""
        _lib.require_cuda(clean_images, "clean_images")
        B = clean_images.shape[0]
        if B != self.batch_size or tuple(clean_images.shape[2:]) != (self.resolution, self.resolution):
            raise _lib.PhenDiffB200Error(
                f"trainer was planned for batches of {self.batch_size} x {self.resolution}^2 images, got {tuple(clean_images.shape)}")
        if self.model._handle is not self._h:
            raise _lib.PhenDiffB200Error("the model's library handle was re-created (precision or device change) after this trainer "
                                         "was built: build a new DenoiserTrainer")
        sch = self.noise_scheduler
        with torch.cuda.device(self.device):
            clean = clean_images.contiguous().float()
            if noise is None:
                noise = torch.randn(clean.shape).to(clean.device)       # drawn on the host like the reference (:244)
            noise = noise.contiguous().float()
            if timesteps is None:
                timesteps = torch.randint(0, sch.config.num_train_timesteps, (B,), device=clean.device).long()
            a = self._acp[timesteps.to(self.device).long()]
            sa, sb = a.sqrt().contiguous(), (1 - a).sqrt().contiguous()
            noisy = self._axpby(clean, noise, sa, sb)                    # DDIMScheduler.add_noise
            ptype = sch.config.prediction_type
            target = training_target(ptype, clean, noise, lambda: self._axpby(noise, clean, sa, -sb))
            weight = (a / (1 - a)).contiguous() if ptype == "sample" else None   # SNR weighting (:420-428)
            labels = None
            if not do_unconditional_pass and class_labels is not None:
                labels = class_labels.to(device=self.device, dtype=torch.int64).contiguous()
            if labels is None and not do_unconditional_pass and self.model.config.num_class_embeds:
                raise ValueError("class_labels should be provided when num_class_embeds > 0")
            tf = timesteps.to(device=self.device, dtype=torch.float32).contiguous()
            mo = torch.empty_like(clean) if return_model_output else None
            _lib.check(_lib.lib().pd_train_step_grad(self._t, _lib.ptr(self.params), _lib.ptr(self.grads), _lib.ptr(noisy), _lib.ptr(tf),
                                                    _lib.ptr(labels), _lib.ptr(target), _lib.ptr(weight), _lib.ptr(self._loss), _lib.ptr(mo),
                                                    _lib.current_stream()))
        loss = self._loss.clone()
        return (loss, mo) if return_model_output else loss

    # ---- input-gradient-only use (gradient-guided generation, SURVEY §8 row f4) --------------------------------------------------------
    def forward_only(self, sample: torch.Tensor, timesteps: torch.Tensor, class_labels: Optional[torch.Tensor]) -> torch.Tensor:
        """UNet forward that keeps the activations for a following `input_gradient` (no parameter gradients are produced)."""
        if self.model._handle is not self._h:
            raise _lib.PhenDiffB200Error("the model's library handle was re-created after this engine was built: build a new one")
        with torch.cuda.device(self.device):
            x = sample.contiguous().float()
            tf = timesteps.to(device=self.device, dtype=torch.float32).reshape(-1)
            if tf.numel() == 1:
                tf = tf.expand(self.batch_size)
            tf = tf.contiguous()
            labels = None if class_labels is None else class_labels.to(device=self.device, dtype=torch.int64).contiguous()
            out = torch.empty_like(x)
            _lib.check(_lib.lib().pd_train_forward(self._t, _lib.ptr(self.params), _lib.ptr(x), _lib.ptr(tf), _lib.ptr(labels), _lib.ptr(out),
                                                  _lib.current_stream()))
        return out

    def input_gradient(self, d_model_output: torch.Tensor) -> torch.Tensor:
        """d(sum_i loss_i)/d(sample) through the UNet for the upstream gradient `d_model_output` (after `forward_only`)."""
        with torch.cuda.device(self.device):
            g = d_model_output.contiguous().float()
            out = torch.empty_like(g)
            _lib.check(_lib.lib().pd_train_backward_input(self._t, _lib.ptr(g), _lib.ptr(out), _lib.current_stream()))
        return out

    def all_reduce_gradients(self, group=None):
        """Average the flat gradient vector over the data-parallel ranks: one collective (NCCL over NVLink on the GPU box)."""
        average_gradients(self.grads, group)

    # ---- dynamic loss scaling (mixed_precision="fp16") ---------------------------------------------------------------------
    def scaler_state(self) -> Optional[dict]:
        """The device-resident GradScaler state as the last optimizer pass left it (waits for that pass), or None outside fp16 mode:
        scale, growth_tracker, optimizer_steps (applied), found_inf (of the last step), skipped_steps."""
        if self._scaler is None:
            return None
        if self._scaler_event is not None:
            self._scaler_event.synchronize()
        st = _lib.GradScalerState.from_buffer_copy(self._scaler_host.numpy().tobytes())
        return {name: getattr(st, name) for name, _ in _lib.GradScalerState._fields_}

    def get_scale(self) -> float:
        """GradScaler.get_scale(): the loss scale the next backward uses (1.0 when no scaling is active).  Synchronises."""
        return float(self.scaler_state()["scale"]) if self._scaler is not None else 1.0

    @property
    def step_was_skipped(self) -> bool:
        """Whether the last optimizer step was skipped for inf / NaN gradients (accelerate's `optimizer.step_was_skipped`).  Synchronises."""
        return bool(self.scaler_state()["found_inf"]) if self._scaler is not None else False

    @property
    def optimizer_steps(self) -> int:
        """AdamW steps applied: `global_step` minus the skipped ones (fp16 mode: waits for the last optimizer pass)."""
        return self.scaler_state()["optimizer_steps"] if self._scaler is not None else self.global_step

    def current_lr(self) -> float:
        return self.lr * (self.lr_lambda(self.optimizer_steps) if self.lr_lambda is not None else 1.0)

    def optimizer_step(self):
        """clip_grad_norm_(1.0) + AdamW.step + lr_scheduler.step + zero_grad + EMAModel.step, one pass over the flat vectors.  fp16 mode:
        GradScaler.unscale_ / step / update around them, decided on the device; the host does not wait for the outcome (it only waits
        for the previous step's pass when `lr_lambda` needs the applied-step count)."""
        step = self.global_step + 1
        decay = 0.0
        if self.use_ema:
            decay = ema_decay_at(step, max_decay=self.ema_max_decay, inv_gamma=self.ema_inv_gamma, power=self.ema_power)
            self.cur_decay_value = decay
        with torch.cuda.device(self.device):
            L, stream = _lib.lib(), _lib.current_stream()
            if self._scaler is None:
                _lib.check(L.pd_adamw_step(_lib.ptr(self.params), _lib.ptr(self.grads), _lib.ptr(self.exp_avg), _lib.ptr(self.exp_avg_sq),
                                           _lib.ptr(self.ema), self.numel, self.current_lr(), self.betas[0], self.betas[1], self.eps,
                                           self.weight_decay, step, self.max_grad_norm, decay, _lib.ptr(self._scratch),
                                           _lib.ptr(self.grad_norm), stream))
            else:
                sc = self._scaler
                _lib.check(L.pd_adamw_step_scaled(_lib.ptr(self.params), _lib.ptr(self.grads), _lib.ptr(self.exp_avg), _lib.ptr(self.exp_avg_sq),
                                                  _lib.ptr(self.ema), self.numel, self.current_lr(), self.betas[0], self.betas[1], self.eps,
                                                  self.weight_decay, self.max_grad_norm, decay, C.c_void_p(self._scaler_state.data_ptr()),
                                                  sc["growth_factor"], sc["backoff_factor"], int(sc["growth_interval"]),
                                                  _lib.ptr(self._scratch), _lib.ptr(self.grad_norm), stream))
                self._scaler_host.copy_(self._scaler_state, non_blocking=True)
                if self._scaler_event is None:
                    self._scaler_event = torch.cuda.Event()
                self._scaler_event.record()
        self.global_step = step
        self.zero_grad()
        self.model.mark_dirty()

    def step(self, clean_images, class_labels, noise=None, timesteps=None, do_unconditional_pass: Optional[bool] = None, group=None):
        """One iteration of the reference's epoch loop body.  Returns the loss (1-element device tensor)."""
        if do_unconditional_pass is None:
            do_unconditional_pass = False
            if self.proba_uncond > 0:
                # the reference draws on rank 0 and broadcasts (utils_training.py:262-277: a collective + a host sync per step); here
                # every rank draws the same coin from a host generator with a shared seed — same decisions on all ranks, no traffic
                do_unconditional_pass = bool(torch.rand(1, generator=self._coin).item() < self.proba_uncond)
        loss = self.diffusion_and_backward(clean_images, class_labels, noise, timesteps, do_unconditional_pass)
        self.all_reduce_gradients(group)
        self.optimizer_step()
        return loss

    # ------------------------------------------------------------------------------------------------------------
    def ema_state(self) -> Optional[dict]:
        """EMA ("shadow") parameters by checkpoint name, or None."""
        if self.ema is None:
            return None
        return {name: self.ema[off: off + cnt].view(shape) for name, (off, cnt, shape) in self._views.items()}

    def copy_ema_to_model(self):
        """EMAModel.copy_to(model.parameters()) (utils_training.py:674-676)."""
        if self.ema is None:
            raise _lib.PhenDiffB200Error("trainer was built with use_ema=False")
        self.params.copy_(self.ema)
        self.model.mark_dirty()
