"""CPU tests of the product's host side: config parsing, scheduler tables / step scalars (bit-compared with the oracle),
the drop-in API surface and its error behaviour, and that the C-ABI library loads and exports every declared symbol.
No compute call is made without a GPU."""
import inspect
import json
import os
import re

import numpy as np
import pytest
import torch

from phendiff_b200 import (ConditionalDDIMPipeline, CustomCondUNet2DModel, CustomEmbedding, DDIMInverseScheduler,
                           DDIMScheduler, PhenDiffB200Error, _ddib, _inversion)
from phendiff_b200.reference_configs import DENOISER_CONFIGS, SCHEDULER_CONFIGS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol(build_lib):
    hdr = open(os.path.join(ROOT, "include", "phendiff_b200.h")).read()
    declared = set(re.findall(r"\b(pd_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"pd_unet_t"}
    assert len(declared) >= 20
    l = build_lib.lib()
    for name in sorted(declared):
        assert hasattr(l, name), f"{name} declared in include/phendiff_b200.h but not exported"
    assert set(build_lib.EXPORTED_SYMBOLS) == declared
    assert l.pd_version() >= 100
    assert isinstance(l.pd_last_error(), bytes)


def test_struct_layouts_match_header(build_lib):
    import ctypes as C

    assert C.sizeof(build_lib.StepCoeffs) == 40
    assert C.sizeof(build_lib.UnetConfig) == 4 * (3 + 3 * 8 + 14)


@pytest.mark.parametrize("name", list(SCHEDULER_CONFIGS))
def test_scheduler_tables_bit_equal_oracle(name):
    from oracle import OracleDDIMInverseScheduler, OracleDDIMScheduler

    cfg = SCHEDULER_CONFIGS[name]
    a, b = DDIMScheduler.from_config(cfg), OracleDDIMScheduler.from_config(cfg)
    assert torch.equal(a.alphas_cumprod, b.alphas_cumprod)
    assert float(a.final_alpha_cumprod) == float(b.final_alpha_cumprod)
    for n in (10, 50, 100):
        a.set_timesteps(n)
        b.set_timesteps(n)
        assert torch.equal(a.timesteps, b.timesteps)
    for variant in ("0.18.2", ">=0.19"):
        ai = DDIMInverseScheduler.from_config(a.config, variant=variant)
        bi = OracleDDIMInverseScheduler.from_config(b.config, variant=variant)
        assert torch.equal(ai.alphas_cumprod, bi.alphas_cumprod)
        ai.set_timesteps(100)
        bi.set_timesteps(100)
        assert torch.equal(ai.timesteps, bi.timesteps)


def test_step_coeffs_reproduce_oracle_step_on_cpu():
    """The host scalars handed to the CUDA kernel, applied with the documented formula in numpy, equal the oracle step."""
    from oracle import OracleDDIMInverseScheduler, OracleDDIMScheduler

    g = torch.Generator().manual_seed(0)
    x, m = torch.randn(64, generator=g), torch.randn(64, generator=g)
    for name in ("3k_steps_clipping_rescaling", "SD_orig_config", "1k_epsilon_pred"):
        cfg = SCHEDULER_CONFIGS[name]
        for P, O in ((DDIMScheduler, OracleDDIMScheduler), (DDIMInverseScheduler, OracleDDIMInverseScheduler)):
            base = DDIMScheduler.from_config(cfg)
            p, o = P.from_config(base.config), O.from_config(base.config)
            p.set_timesteps(10)
            o.set_timesteps(10)
            for t in p.timesteps[1:]:   # skip the alpha-bar = 0 step (inf arithmetic; covered on the GPU)
                c = p.step_coeffs(t)
                xs, ms = x.numpy(), m.numpy()
                f = np.float32
                if c.pred_type == 0:
                    x0 = (xs - f(c.sqrt_beta) * ms) / f(c.sqrt_alpha); e = ms
                elif c.pred_type == 1:
                    x0 = ms; e = (xs - f(c.sqrt_alpha) * x0) / f(c.sqrt_beta)
                else:
                    x0 = f(c.sqrt_alpha) * xs - f(c.sqrt_beta) * ms; e = f(c.sqrt_alpha) * ms + f(c.sqrt_beta) * xs
                if c.clip:
                    x0 = np.clip(x0, -c.clip_range, c.clip_range)
                out = f(c.sqrt_alpha_next) * x0 + f(c.dir_coef) * e
                ref = o.step(m, t, x).prev_sample.numpy()
                assert np.abs(out - ref).max() <= 2e-6, (name, P.__name__, int(t))
                assert c.timestep == float(t)


def test_config_parsing_from_json_file(tmp_path):
    cfg = dict(DENOISER_CONFIGS["small_denoiser_config"])
    cfg["some_future_key"] = 1  # unknown keys are ignored (A.7)
    p = tmp_path / "denoiser.json"
    p.write_text(json.dumps(cfg))
    loaded = CustomCondUNet2DModel.load_config(str(p))
    assert loaded["_class_name"] == "CondUNet2DModel"
    loaded["sample_size"] = 64  # utils_models.py:167 overrides sample_size like this
    m = CustomCondUNet2DModel.from_config(loaded)
    assert m.config.sample_size == 64 and m.config.block_out_channels == (128, 256, 512)
    assert m.time_embed_dim == 512 and m.config.class_embed_type is None and not m.config.center_input_sample
    assert sum(p.numel() for p in m.parameters()) == 62826243
    with pytest.raises(AttributeError):
        m.config.sample_size = 3
    s = DDIMScheduler.from_config(SCHEDULER_CONFIGS["3k_steps_clipping_rescaling"])
    assert s.config.prediction_type == "v_prediction" and s.config.set_alpha_to_one is True
    i = DDIMInverseScheduler.from_config(s.config)
    assert "rescale_betas_zero_snr" not in i.config and i.config.set_alpha_to_zero is True


def test_param_table_matches_oracle_state_dict():
    from oracle import OracleCondUNet2D

    for name in ("small_denoiser_config", "super_small"):
        cfg = DENOISER_CONFIGS[name]
        o = OracleCondUNet2D(**cfg)
        m = CustomCondUNet2DModel.from_config(cfg)
        so, sm = o.state_dict(), m.state_dict()
        assert set(so) == set(sm)
        assert all(so[k].shape == sm[k].shape for k in so)
        m.load_state_dict(so)
        # deprecated attention spellings are accepted on load (A.7)
        ren = {"to_q": "query", "to_k": "key", "to_v": "value", "to_out.0": "proj_attn"}
        old = {}
        for k, v in so.items():
            for new_, old_ in ren.items():
                if ".attentions." in k and f".{new_}." in k:
                    k = k.replace(f".{new_}.", f".{old_}.")
            old[k] = v
        m.load_state_dict(old)


def test_unsupported_options_raise():
    base = dict(DENOISER_CONFIGS["super_small"])
    with pytest.raises(NotImplementedError):
        CustomCondUNet2DModel.from_config(dict(base, time_embedding_type="fourier"))
    with pytest.raises(NotImplementedError):
        CustomCondUNet2DModel.from_config(dict(base, class_embed_type="timestep"))
    with pytest.raises(ValueError):
        CustomCondUNet2DModel.from_config(dict(base, block_out_channels=[64, 128]))
    with pytest.raises(NotImplementedError):
        DDIMScheduler(thresholding=True)


def test_api_surface_and_cpu_tensors_fail_loudly():
    m = CustomCondUNet2DModel.from_config(dict(DENOISER_CONFIGS["super_small"], sample_size=32))
    sig = inspect.signature(m.forward)
    assert list(sig.parameters) == ["sample", "timestep", "class_labels", "class_emb", "return_dict"]
    pipe = ConditionalDDIMPipeline(m, DDIMInverseScheduler.from_config(SCHEDULER_CONFIGS["1k_epsilon_pred"]))
    assert isinstance(pipe.scheduler, DDIMScheduler)  # pipeline:44-45 always converts to DDIM
    call = inspect.signature(pipe.__call__)
    assert list(call.parameters) == ["class_labels", "class_emb", "w", "generator", "eta", "num_inference_steps",
                                     "use_clipped_model_output", "output_type", "return_dict", "start_image",
                                     "add_forward_noise_to_image", "frac_diffusion_skipped", "guidance_eqn"]
    assert set(pipe.components) == {"unet", "scheduler"}
    x, lab = torch.zeros(2, 3, 32, 32), torch.tensor([0, 1])
    with pytest.raises(ValueError):
        m(x, 1, lab, torch.zeros(2, 256))
    with pytest.raises(ValueError):
        m(x, 1)
    with pytest.raises(PhenDiffB200Error):
        m(x, 1, lab)
    with pytest.raises(PhenDiffB200Error):
        _inversion(pipe, x, lab, 2)
    with pytest.raises(PhenDiffB200Error):
        _ddib(pipe, x, lab, 1 - lab, 2)
    with pytest.raises(PhenDiffB200Error):
        pipe.scheduler.set_timesteps(4) or pipe.scheduler.step(x, 999, x)
    # check_inputs keeps the reference's assertions (pipeline:91-137)
    with pytest.raises(AssertionError):
        pipe.check_inputs(class_labels=torch.zeros(2, 2))
    with pytest.raises(AssertionError):
        pipe.check_inputs(class_labels=lab, class_emb=torch.zeros(2, 256))
    with pytest.raises(AssertionError):
        pipe.check_inputs(class_labels=lab, w=torch.zeros(3))
    with pytest.raises(ValueError):
        pipe.check_inputs(class_labels=lab, generator=[torch.Generator()])
    with pytest.raises(AssertionError):
        pipe.check_inputs(class_labels=lab, start_image=x)
    with pytest.raises(AssertionError):
        pipe.check_inputs(class_labels=lab, start_image=x, frac_diffusion_skipped=1.5)
    pipe.check_inputs(class_labels=lab, w=0, start_image=x, frac_diffusion_skipped=0)
    e = CustomEmbedding(2, 1024)
    assert e(torch.tensor([1, 0])).shape == (2, 1024) and e.config.num_classes == 2


def test_save_and_load_pretrained_roundtrip(tmp_path):
    m = CustomCondUNet2DModel.from_config(dict(DENOISER_CONFIGS["super_small"], sample_size=32))
    pipe = ConditionalDDIMPipeline(m, DDIMScheduler.from_config(SCHEDULER_CONFIGS["3k_steps_clipping_rescaling"]))
    pipe.save_pretrained(str(tmp_path / "p"))
    p2 = ConditionalDDIMPipeline.from_pretrained(str(tmp_path / "p"))
    assert p2.scheduler.config.num_train_timesteps == 3000 and p2.unet.config.sample_size == 32
    for (k, a), (_, b) in zip(m.state_dict().items(), p2.unet.state_dict().items()):
        assert torch.equal(a, b), k


def test_shard_ranges():
    from phendiff_b200.sharding import shard_range, shard_sizes

    for total in (0, 1, 7, 256, 257):
        for world in (1, 2, 3, 8):
            rs = [shard_range(total, r, world) for r in range(world)]
            assert rs[0][0] == 0 and rs[-1][1] == total
            assert all(rs[i][1] == rs[i + 1][0] for i in range(world - 1))
            assert max(shard_sizes(total, world)) - min(shard_sizes(total, world)) <= 1
    with pytest.raises(ValueError):
        shard_range(4, 2, 2)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU oracle on the host cores) on a tiny configuration: one JSON line carrying the
    keys the bench contract names for the reference arm."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--denoiser", "super_small", "--size", "32", "--batch", "4", "--num-inference-steps", "4",
                          "--cpu-sample-images", "2"], capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("images/sec, DDIM invert+regenerate")
    assert d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_bench_reference_arm_other_ranks_exit_without_work():
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=root, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_bench_dump_outputs_float32_within_budget_and_fixed_sample(tmp_path, monkeypatch):
    import bench

    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 64 << 10)
    big = torch.arange(100_000, dtype=torch.float64)
    small = np.arange(6, dtype=np.uint8).reshape(2, 3)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"big": big, "small": small})
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64 << 10
    s = np.load(tmp_path / "a" / "small.npy")
    assert s.dtype == np.float32 and s.tolist() == small.tolist()
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float32 and 0 < a.size < big.numel() and np.array_equal(a, b)
    assert np.all(np.diff(a) > 0)        # distinct positions, in order


def test_bench_rejects_zero_steps_and_dump_on_reference_arm(tmp_path):
    import subprocess
    import sys

    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "", (extra, out.stderr[-500:])
    assert list(tmp_path.iterdir()) == []


def test_cfg_lookup_reads_attribute_and_dict_configs():
    from types import SimpleNamespace as NS

    from phendiff_b200.utils_img2img import _cfg_lookup

    a = NS(class_transfer_method=NS(classifier_free_guidance_forward_start=NS(guidance_scale=2.5, frac_diffusion_skipped=0.5)))
    d = {"class_transfer_method": {"classifier_free_guidance_forward_start": {"guidance_scale": 2.5, "frac_diffusion_skipped": 0.5}}}
    for c in (a, d):
        node = _cfg_lookup(c, "class_transfer_method", "classifier_free_guidance_forward_start")
        assert _cfg_lookup(node, "guidance_scale") == 2.5 and _cfg_lookup(node, "frac_diffusion_skipped") == 0.5
    with pytest.raises((AttributeError, KeyError)):
        _cfg_lookup(a, "class_transfer_method", "ddib")


def test_weight_state_tracking_sees_out_of_band_writes():
    """Round-1 advisor finding: `p.data.copy_()` (diffusers EMAModel.copy_to / restore, utils_training.py:674-676) does not
    move the autograd version counter.  The cheap key must see everything else; the fingerprint must see this."""
    import torch

    from phendiff_b200 import CustomCondUNet2DModel
    from phendiff_b200.reference_configs import DENOISER_CONFIGS

    m = CustomCondUNet2DModel.from_config(dict(DENOISER_CONFIGS["super_small"], sample_size=32))
    k0, f0 = m._weights_version(), m.weights_fingerprint()
    p = m.conv_in.weight
    p.data.copy_(p.data * 1.01)                       # out of band: version key blind, fingerprint not
    assert m._weights_version() == k0
    assert m.weights_fingerprint() != f0
    m.mark_dirty()
    assert m._weights_version() != k0
    k1 = m._weights_version()
    with torch.no_grad():
        p.mul_(1.01)                                  # in-place op through the parameter: version counter moves
    assert m._weights_version() != k1
    k2 = m._weights_version()
    m.load_state_dict(m.state_dict())                 # load_state_dict always invalidates
    assert m._weights_version() != k2
    k3 = m._weights_version()
    m.double().float()                                # _apply (to / cuda / dtype casts) invalidates
    assert m._weights_version() != k3
    k4 = m._weights_version()
    p.data = p.data.clone()                           # re-assigned storage: data_ptr moves
    assert m._weights_version() != k4


def test_randn_tensor_generator_list_is_per_sample():
    import torch

    from phendiff_b200.schedulers import randn_tensor

    gens = [torch.Generator().manual_seed(s) for s in (5, 6, 7)]
    a = randn_tensor((3, 2, 4, 4), gens, torch.device("cpu"))
    b = randn_tensor((1, 2, 4, 4), [torch.Generator().manual_seed(6)], torch.device("cpu"))
    assert torch.equal(a[1:2], b)                     # sample i depends on generator i only (diffusers randn_tensor)
    import pytest
    with pytest.raises(ValueError):
        randn_tensor((2, 2, 4, 4), gens, torch.device("cpu"))


def test_unconditional_pass_coin_is_shared_seed():
    """The CFG-training coin (utils_training.py:262-277: rank 0 draws, broadcast) is drawn here from a host generator with a shared seed:
    two trainers (= two ranks) built with the same seed take the same decisions, at the requested rate."""
    import torch

    g1, g2 = torch.Generator().manual_seed(5), torch.Generator().manual_seed(5)
    a = [bool(torch.rand(1, generator=g1).item() < 0.1) for _ in range(2000)]
    b = [bool(torch.rand(1, generator=g2).item() < 0.1) for _ in range(2000)]
    assert a == b
    assert 0.07 < sum(a) / len(a) < 0.13


def test_ema_decay_schedule_host():
    """diffusers EMAModel.get_decay as the reference configures it (train.py:229-236): warm-up 1 - (1 + step / inv_gamma)^-power after the
    first optimizer step, capped at max_decay; pure host logic of phendiff_b200.training."""
    import math

    from phendiff_b200.training import ema_decay_at, training_target

    assert ema_decay_at(0) == 0.0 and ema_decay_at(1) == 0.0
    assert math.isclose(ema_decay_at(2, inv_gamma=1.0, power=0.75), 1 - 2 ** -0.75)
    assert math.isclose(ema_decay_at(101, inv_gamma=2.0, power=0.5), 1 - (1 + 100 / 2.0) ** -0.5)
    assert ema_decay_at(10 ** 9) == 0.9999
    assert math.isclose(ema_decay_at(5, use_ema_warmup=False), 5 / 14)
    assert ema_decay_at(3, min_decay=0.9) == 0.9
    # regression target by prediction type (utils_training.py:415-433)
    assert training_target("epsilon", "clean", "noise", lambda: "vel") == "noise"
    assert training_target("sample", "clean", "noise", lambda: "vel") == "clean"
    assert training_target("v_prediction", "clean", "noise", lambda: "vel") == "vel"
    import pytest as _pt
    with _pt.raises(ValueError):
        training_target("other", 0, 0, lambda: 0)
