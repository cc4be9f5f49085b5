"""CPU tests of the fp16 training mode's host side: the ctypes mirror of the device-resident grad-scaler state against the header,
the scratch sizes, and the argument checks of `DenoiserTrainer(mixed_precision=..., grad_scaler_kwargs=...)`."""
import ctypes as C
import os
import re

import pytest

from phendiff_b200 import CustomCondUNet2DModel, DDIMScheduler, PhenDiffB200Error
from phendiff_b200.reference_configs import DENOISER_CONFIGS, SCHEDULER_CONFIGS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_CTYPE_OF = {"float": C.c_float, "int32_t": C.c_int32}


def _header():
    return open(os.path.join(ROOT, "include", "phendiff_b200.h")).read()


def test_grad_scaler_state_mirror_matches_header(build_lib):
    body = re.search(r"typedef struct pd_grad_scaler_state \{(.*?)\} pd_grad_scaler_state_t;", _header(), re.S).group(1)
    fields = re.findall(r"^\s*(float|int32_t)\s+(\w+);", body, re.M)
    assert [(n, _CTYPE_OF[t]) for t, n in fields] == list(build_lib.GradScalerState._fields_)
    assert C.sizeof(build_lib.GradScalerState) == 4 * len(fields) == 20
    # `scale` first: the trainer hands the state's own address to pd_train_set_loss_scale
    assert build_lib.GradScalerState.scale.offset == 0


def test_adamw_scratch_sizes_match_header(build_lib):
    hdr = _header()
    for name in ("PD_ADAMW_SCRATCH_FLOATS", "PD_ADAMW_SCALED_SCRATCH_FLOATS"):
        assert int(re.search(rf"#define {name} (\d+)", hdr).group(1)) == getattr(build_lib, name)


def test_precision_enum_matches_header(build_lib):
    from phendiff_b200.training import PRECISIONS

    enum = dict((k, int(v)) for k, v in re.findall(r"(PD_PREC_\w+) = (\d+)", _header()))
    assert PRECISIONS == {"no": enum["PD_PREC_FP32"], "bf16": enum["PD_PREC_BF16"], "fp16": enum["PD_PREC_FP16"]}


def _model_and_scheduler():
    m = CustomCondUNet2DModel.from_config(dict(DENOISER_CONFIGS["super_small"], sample_size=32))
    return m, DDIMScheduler.from_config(SCHEDULER_CONFIGS["1k_epsilon_pred"])


def test_mixed_precision_argument_errors():
    from phendiff_b200.training import DenoiserTrainer

    m, sched = _model_and_scheduler()
    with pytest.raises(ValueError, match="'no', 'bf16' or 'fp16'"):
        DenoiserTrainer(m, sched, 2, 32, mixed_precision="fp8")
    with pytest.raises(ValueError, match="unknown keys"):
        DenoiserTrainer(m, sched, 2, 32, mixed_precision="fp16", grad_scaler_kwargs={"init_scale": 8.0, "enabled": True})
    with pytest.raises(ValueError, match="growth_factor > 1"):
        DenoiserTrainer(m, sched, 2, 32, mixed_precision="fp16", grad_scaler_kwargs={"backoff_factor": 1.5})
    with pytest.raises(ValueError, match="fp16"):
        DenoiserTrainer(m, sched, 2, 32, mixed_precision="bf16", grad_scaler_kwargs={"init_scale": 8.0})
    # accepted arguments get as far as the device check: there is no CPU fallback
    with pytest.raises(PhenDiffB200Error, match="CUDA"):
        DenoiserTrainer(m, sched, 2, 32, mixed_precision="fp16", grad_scaler_kwargs={"init_scale": 8.0, "growth_interval": 10})
