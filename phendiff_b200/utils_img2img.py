"""Class-transfer drivers — drop-ins for the reference's `_inversion`, `_ddib` and (SURVEY §8 row f1)
`_classifier_free_guidance_forward_start`
(reference: src/utils_Img2Img.py:763-800, :566-612 and :615-648; called from perform_class_transfer_experiment :365-384).

`_ddib` = invert the real images to noise with the SOURCE class, regenerate with the TARGET class.  Here both loops
(2 x num_inference_steps UNet forwards + scheduler updates) run inside ONE C-ABI call on the current CUDA stream; x_t
stays resident in HBM in fp32 and each scheduler update is fused into the UNet's conv_out epilogue.
"""
from __future__ import annotations

from typing import List, Optional

import torch
from torch import Tensor

from . import _lib
from .pipeline_conditional_ddim import ConditionalDDIMPipeline
from .schedulers import DDIMInverseScheduler

# which diffusers release's DDIMInverseScheduler semantics to reproduce (SURVEY A.4); the reference pins 0.18.2
INVERSE_SCHEDULER_VARIANT = "0.18.2"


def _to_device(pipe, t: Optional[Tensor], dtype):
    if pipe.device.type != "cuda":
        raise _lib.PhenDiffB200Error(
            f"the pipeline lives on {pipe.device}: move it to a CUDA device (pipe.to('cuda')); there is no CPU fallback")
    if t is None:
        return None
    return t.to(device=pipe.device, dtype=dtype, non_blocking=True)


def _inversion_steps(pipe, num_inference_steps: int):
    # the inverse scheduler is rebuilt from the pipeline's scheduler config on every call (utils_Img2Img.py:776-779)
    inv = DDIMInverseScheduler.from_config(pipe.scheduler.config, variant=INVERSE_SCHEDULER_VARIANT)
    inv.set_timesteps(num_inference_steps)
    return inv, [inv.step_coeffs(t) for t in inv.timesteps]


@torch.no_grad()
def _inversion(pipe: ConditionalDDIMPipeline, input_images: Tensor, class_labels: Tensor, num_inference_steps: int,
               proc_idx: Optional[int] = None) -> Tensor:
    """Real images + source class -> Gaussian latents (the input is not modified: it is cloned, :773)."""
    gauss = _to_device(pipe, input_images, torch.float32).contiguous().clone()
    labels = _to_device(pipe, class_labels, torch.int64)
    if pipe.fused_route_ok():
        _, steps = _inversion_steps(pipe, num_inference_steps)
        return pipe._run_fused(gauss, labels, None, steps, len(steps), 0)
    inv, _ = _inversion_steps(pipe, num_inference_steps)
    pipe.unet.check_weights()
    for t in inv.timesteps:
        model_output = pipe.unet(gauss, t, labels).sample
        gauss = inv.step(model_output, t, gauss).prev_sample
    return gauss


@torch.no_grad()
def ddib_transfer(pipe: ConditionalDDIMPipeline, clean_images: Tensor, orig_class_labels: Tensor,
                  target_class_labels: Tensor, num_inference_steps: int) -> Tensor:
    """The whole class transfer as one fused device pass; returns the regenerated x_0' (B,C,H,W) fp32 on the device."""
    x = _to_device(pipe, clean_images, torch.float32).contiguous().clone()
    src = _to_device(pipe, orig_class_labels, torch.int64)
    tgt = _to_device(pipe, target_class_labels, torch.int64)
    _, inv_steps = _inversion_steps(pipe, num_inference_steps)
    pipe.scheduler.set_timesteps(num_inference_steps)
    # frac_diffusion_skipped = 0 keeps every timestep (pipeline:250-258); w = 0 disables guidance (:272-284)
    gen_steps = [pipe.scheduler.step_coeffs(t, 0.0, None) for t in pipe.scheduler.timesteps]
    return pipe._run_fused(x, src, tgt, inv_steps + gen_steps, len(inv_steps), len(gen_steps))


@torch.no_grad()
def _ddib(pipe: ConditionalDDIMPipeline, clean_images: Tensor, orig_class_labels: Tensor, target_class_labels: Tensor,
          num_inference_steps: int, process_idx: Optional[int] = None) -> List:
    """Same contract as the reference: returns the list of PIL images `pipe(...).images` would return."""
    if not isinstance(pipe, ConditionalDDIMPipeline):
        raise NotImplementedError("only the pixel-space ConditionalDDIMPipeline path is implemented (SURVEY §8)")
    if pipe.fused_route_ok():
        x = ddib_transfer(pipe, clean_images, orig_class_labels, target_class_labels, num_inference_steps)
        return pipe.numpy_to_pil(pipe.postprocess(x))
    inverted_gauss = _inversion(pipe, clean_images, orig_class_labels, num_inference_steps, process_idx)
    return pipe(class_labels=target_class_labels, w=0, num_inference_steps=num_inference_steps,
                start_image=inverted_gauss, add_forward_noise_to_image=False, frac_diffusion_skipped=0).images


def _cfg_lookup(cfg, *path):
    """`cfg.a.b.c` for attribute-style configs (the reference's omegaconf DictConfig) and plain nested dicts alike."""
    node = cfg
    for key in path:
        node = node[key] if isinstance(node, dict) else getattr(node, key)
    return node


@torch.no_grad()
def _classifier_free_guidance_forward_start(pipe: ConditionalDDIMPipeline, clean_images: Tensor, target_class_labels: Tensor,
                                            cfg, num_inference_steps: int) -> List:
    """Forward-noise the real images part of the way, then denoise them with classifier-free guidance towards the target
    class (utils_Img2Img.py:615-648).  `cfg` is read exactly where the reference reads it:
    `cfg.class_transfer_method.classifier_free_guidance_forward_start.{guidance_scale, frac_diffusion_skipped}`."""
    this_exp_cfg = _cfg_lookup(cfg, "class_transfer_method", "classifier_free_guidance_forward_start")
    guidance_scale = _cfg_lookup(this_exp_cfg, "guidance_scale")
    frac_diffusion_skipped = _cfg_lookup(this_exp_cfg, "frac_diffusion_skipped")
    if not isinstance(pipe, ConditionalDDIMPipeline):
        raise NotImplementedError("only the pixel-space ConditionalDDIMPipeline path is implemented (SURVEY §8)")
    return pipe(class_labels=target_class_labels, w=guidance_scale, num_inference_steps=num_inference_steps,
                start_image=clean_images, frac_diffusion_skipped=frac_diffusion_skipped).images


# ---------------------------------------------------------------------------------------------------------------------
# gradient-guided transfer (SURVEY §8 row f4; reference utils_Img2Img.py:651-760)
# ---------------------------------------------------------------------------------------------------------------------
def _guidance_engine(pipe: ConditionalDDIMPipeline, batch: int, resolution: int, mixed_precision: Optional[str] = None):
    """The forward + input-gradient engine of the UNet for this batch shape (workspace of the training walk), cached on the pipeline.
    mixed_precision: "bf16" or "fp16" (16-bit tensor-core operands; fp16 is the reference's autocast type for class transfer) or "no"
    (fp32 validation path); default: "no" for an fp32 model, else "bf16".  The input gradient is not loss-scaled, as in the reference."""
    from .training import DenoiserTrainer

    if mixed_precision is None:
        mixed_precision = "no" if pipe.unet.precision == "fp32" else "bf16"
    key = (batch, resolution, mixed_precision)
    cache = pipe.__dict__.setdefault("_guidance_engines", {})
    eng = cache.get(key)
    if eng is None or eng.model._handle is not eng._h:
        cache.clear()     # one workspace at a time
        eng = DenoiserTrainer(pipe.unet, pipe.scheduler, batch, resolution, mixed_precision=mixed_precision)
        cache[key] = eng
    return eng


def _custom_guided_generation(pipe: ConditionalDDIMPipeline, input_images: Tensor, target_class_labels: Tensor, cfg,
                              num_inference_steps: int, mixed_precision: Optional[str] = None) -> Tensor:
    """Generation guided by the gradient of || x0_pred - input_images ||_p w.r.t. the current images (utils_Img2Img.py:701-760).
    Per step: UNet forward with saved activations, per-image loss and its gradients w.r.t. the model output and x_t
    (`pd_guidance_lp_grad`), input-gradient-only backward (`pd_train_backward_input`), the gradient step on the images, then the
    scheduler update with the model output computed before the gradient step — the reference's order."""
    import ctypes as C

    this_cfg = _cfg_lookup(cfg, "class_transfer_method", "linear_interp_custom_guidance_inverted_start")
    p = _cfg_lookup(this_cfg, "p")
    guidance_loss_scale = float(_cfg_lookup(this_cfg, "guidance_loss_scale"))
    if isinstance(p, str):
        raise NotImplementedError("Lp_loss with p = 'inf' / '-inf' is not implemented (finite p only)")
    _lib.require_cuda(input_images, "input_images")
    dev = pipe.unet.device
    ref = input_images.detach().to(dev).contiguous().float()
    images = ref.clone()
    labels = target_class_labels.to(dev)
    B, per = images.shape[0], images[0].numel()
    eng = _guidance_engine(pipe, B, images.shape[-1], mixed_precision)
    pipe.scheduler.set_timesteps(num_inference_steps)
    scratch = torch.zeros(B, device=dev)
    losses = torch.zeros(B, device=dev)
    dm, dx = torch.empty_like(images), torch.empty_like(images)
    one, neg_scale = _ones(B, dev), _ones(B, dev, -guidance_loss_scale)     # per-sample coefficient vectors of the axpby kernel
    L = _lib.lib()
    for t in pipe.scheduler.timesteps:
        tt = torch.full((B,), float(t), device=dev)
        model_output = eng.forward_only(images, tt, labels)
        co = pipe.scheduler.step_coeffs(t)
        _lib.check(L.pd_guidance_lp_grad(C.byref(co), _lib.ptr(images), _lib.ptr(model_output), _lib.ptr(ref), B, per, float(p),
                                         _lib.ptr(scratch), _lib.ptr(losses), _lib.ptr(dm), _lib.ptr(dx), _lib.current_stream()))
        guidance_grad = eng.input_gradient(dm)
        # images <- images - scale * (direct + through-the-UNet gradient); then x_t -> x_{t-1} with the pre-step model output
        _lib.check(L.pd_axpby_per_sample(_lib.ptr(guidance_grad), _lib.ptr(dx), _lib.ptr(one), _lib.ptr(one), _lib.ptr(guidance_grad), B, per,
                                         _lib.current_stream()))
        _lib.check(L.pd_axpby_per_sample(_lib.ptr(images), _lib.ptr(guidance_grad), _lib.ptr(one), _lib.ptr(neg_scale), _lib.ptr(images), B, per,
                                         _lib.current_stream()))
        images = pipe.scheduler.step(model_output, t, images).prev_sample
    return images


def _ones(B, dev, value=1.0):
    return torch.full((B,), float(value), device=dev, dtype=torch.float32)


def _linear_interp_custom_guidance_inverted_start(pipe: ConditionalDDIMPipeline, clean_images: Tensor, orig_class_labels: Tensor,
                                                  target_class_labels: Tensor, cfg, num_inference_steps: int,
                                                  mixed_precision: Optional[str] = None) -> List:
    """Inversion with the source class, then gradient-guided generation with the target class (utils_Img2Img.py:651-698);
    returns PIL images like the reference (`tensor_to_PIL`)."""
    if not isinstance(pipe, ConditionalDDIMPipeline):
        raise NotImplementedError("only the pixel-space ConditionalDDIMPipeline path is implemented (SURVEY §8)")
    inverted_gauss = _inversion(pipe, clean_images, orig_class_labels, num_inference_steps, None)
    image = _custom_guided_generation(pipe, inverted_gauss, target_class_labels, cfg, num_inference_steps, mixed_precision)
    return pipe.numpy_to_pil(pipe.postprocess(image))
