"""CPU tests of the host logic: sigma schedule, integer step indexing, packing, ids, size rules,
and that libb2f loads and exports every symbol include/b2f.h declares (no compute without a GPU)."""
import math

import numpy as np
import pytest
import torch


def test_library_loads_and_exports_every_declared_symbol():
    from gpt_image_edit_b200 import _lib

    declared = _lib.declared_symbols()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(_lib.lib, name), f"libb2f.so does not export {name}"
    assert set(declared) == set(_lib._SIGNATURES), "ctypes signatures out of sync with include/b2f.h"
    assert _lib.lib.b2f_version() >= 1
    assert _lib.lib.b2f_strerror(-5).decode() == "no sm_100 device"


def test_no_cpu_fallback_paths():
    """Without a GPU every compute entry point must refuse, not fall back."""
    from gpt_image_edit_b200 import _lib, ops

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    x = torch.zeros(8, 64, dtype=torch.bfloat16)
    with pytest.raises(_lib.B2FError):
        ops.linear(x, x)
    with pytest.raises(_lib.B2FError):
        from gpt_image_edit_b200.flux_transformer import B200FluxTransformer2DModel
        B200FluxTransformer2DModel(device="cpu")
    # raw ABI: no device -> B2F_ERR_NODEVICE
    rc = _lib.lib.b2f_gemm_bf16(16, 64, 0, 16, 64, None, 16, 64, 0, 1, 8, 64, 64, 0, None, 0, 0, None, 0, None)
    assert rc == -5


def test_sigma_schedule_matches_survey_pins():
    """SURVEY.md §8c: mu(4096)=1.15, mu(256)=0.5; first 28-step timesteps 1000.0, 988.4086, 976.2225."""
    from gpt_image_edit_b200.pipeline import calculate_shift
    from gpt_image_edit_b200.scheduler import FlowMatchEulerDiscreteScheduler
    from oracle.pipeline_oracle import EulerSchedulerOracle
    from oracle.pipeline_oracle import calculate_shift as cs_oracle

    assert math.isclose(calculate_shift(4096), 1.15, rel_tol=1e-12)
    assert math.isclose(calculate_shift(256), 0.5, rel_tol=1e-12)
    assert calculate_shift(1024) == cs_oracle(1024)
    s = FlowMatchEulerDiscreteScheduler()
    sig = np.linspace(1.0, 1 / 28, 28)
    s.set_timesteps(sigmas=sig, mu=1.15)
    assert torch.allclose(s.timesteps[:3], torch.tensor([1000.0, 988.4086, 976.2225]), atol=2e-4)
    assert s.sigmas.shape == (29,) and s.sigmas[-1] == 0
    o = EulerSchedulerOracle()
    o.set_timesteps(sig, 1.15)
    assert torch.equal(o.timesteps, s.timesteps) and torch.equal(o.sigmas, s.sigmas)
    # sum of dt telescopes to -sigma_0
    assert math.isclose(sum(s.dt(i) for i in range(28)), -1.0, abs_tol=1e-6)
    # dt is the fp32 difference of fp32 sigmas (bit-exact with the 0-dim tensor subtraction)
    for i in range(28):
        assert s.dt(i) == float((o.sigmas[i + 1] - o.sigmas[i]).item())


def test_integer_step_index_is_bit_exact():
    from gpt_image_edit_b200.scheduler import FlowMatchEulerDiscreteScheduler

    s = FlowMatchEulerDiscreteScheduler()
    s.set_timesteps(sigmas=np.linspace(1.0, 1 / 4, 4), mu=0.5)
    assert s.step_index is None and s.begin_index is None
    s.set_begin_index(0)
    assert s.begin_index == 0
    s._init_step_index(s.timesteps[0])
    assert s.step_index == 0
    # without begin_index the index is looked up from the timestep value, as diffusers does
    s2 = FlowMatchEulerDiscreteScheduler()
    s2.set_timesteps(sigmas=np.linspace(1.0, 1 / 4, 4), mu=0.5)
    s2._init_step_index(s2.timesteps[2])
    assert s2.step_index == 2
    with pytest.raises(Exception):
        s2.step(torch.zeros(1, 4, 64), s2.timesteps[2], torch.zeros(1, 4, 64))  # CPU tensors: refused


def test_pack_unpack_ids_match_oracle_and_roundtrip():
    from gpt_image_edit_b200.pipeline import FluxKontextPipeline as P
    from oracle import pipeline_oracle as po

    x = torch.randn(2, 16, 12, 20)
    packed = P._pack_latents(x, 2, 16, 12, 20)
    assert packed.shape == (2, 60, 64)
    assert torch.equal(packed, po.pack_latents(x))
    # inside a token the order is (c, dy, dx)
    assert packed[0, 0, 5].item() == x[0, 1, 0, 1].item()  # c=1,dy=0,dx=1 -> 1*4+0*2+1
    back = P._unpack_latents(packed, 12 * 8, 20 * 8, 8)
    assert torch.equal(back, x)
    ids = P._prepare_latent_image_ids(1, 6, 10, "cpu", torch.float32)
    assert torch.equal(ids, po.latent_image_ids(6, 10))
    assert ids[13].tolist() == [0.0, 1.0, 3.0]


def test_size_rule_rescales_to_max_area():
    from oracle.pipeline_oracle import target_size

    assert target_size(256, 256, 1024 ** 2) == (1024, 1024)     # reference quirk: 256 request -> 1 MP
    assert target_size(256, 256, 256 * 256) == (256, 256)
    assert target_size(720, 1280, 1024 ** 2) == (768, 1360)


def test_anyres_dynamic_resize_matches_reference_semantics():
    """Expected values produced by the reference's own univa/utils/anyres_util.py (pure Python, importable in
    the build container; the two implementations were also compared on a 10x9x6 grid of sizes/bucket lists)."""
    from univa.utils.anyres_util import compute_size, dynamic_resize, pick_ratio

    assert dynamic_resize(1024, 1024) == (1024, 1024)
    assert dynamic_resize(720, 1280) == (1504, 2784)
    assert dynamic_resize(1280, 720) == (2784, 1504)
    assert dynamic_resize(512, 768) == (832, 1248)
    assert pick_ratio(600, 800, "any_11ratio") == (4, 3)
    assert compute_size(4, 3, 32, anchor_pixels=448 * 448) == (384, 512)


def test_gedit_driver_host_logic(tmp_path):
    """Prompt-file format, output paths, rank striding and the generation-size rule of the GEdit sampling driver
    (reference univa/eval/gedit/step1_gen_samples.py:100-114, 228-239)."""
    import json

    from gpt_image_edit_b200 import distributed as D
    from univa.eval.configuration_eval import EvalConfig
    from univa.eval.gedit.step1_gen_samples import generation_size, load_items

    spec = {f"k{i}": {"prompt": f"edit {i}", "id": f"en/{i}.png", "extra": 1} for i in range(7)}
    pf = tmp_path / "gedit.json"
    pf.write_text(json.dumps(spec))
    items = load_items(pf, str(tmp_path / "out"))
    assert [it[2] for it in items] == [f"k{i}" for i in range(7)]
    assert items[3][1].endswith("out/en/3.png") and items[3][0] == "edit 3" and items[3][3] == "en/3.png"
    parts = [D.shard(items, r, 3) for r in range(3)]
    assert [len(p) for p in parts] == [3, 2, 2] and parts[1][0][2] == "k1" and parts[1][1][2] == "k4"
    assert sorted(it[2] for p in parts for it in p) == sorted(spec)
    # size rule: a multiple of 16 in both directions, area close to the anchor, aspect of the nearest listed ratio
    for (h, w) in [(768, 1024), (1024, 1024), (500, 1500), (1365, 1024)]:
        gh, gw = generation_size(h, w, 1024, 1024)
        assert gh % 16 == 0 and gw % 16 == 0 and abs(gh * gw - 1024 * 1024) / (1024 * 1024) < 0.08
        assert (gh >= gw) == (h >= w)
    assert generation_size(1024, 1024, 512, 512) == (512, 512)
    cfg = EvalConfig.from_mapping({"seed": 7, "gedit_image_dir": "x", "genai_prompt_path": "ignored", "joint_with_t5": True})
    assert cfg.seed == 7 and cfg.joint_with_t5 and cfg.num_inference_steps == 32 and cfg.guidance_scale == 3.5


def test_host_modules_match_the_references_own_outputs():
    """tests/golden/host_ref.pt: outputs of the reference's own anyres_util.py and denoiser_prompt_embedding_flux.py
    (imported by path, tests/golden/make_host_ref_golden.py) on a grid of sizes / with stub encoders."""
    import sys
    from pathlib import Path

    sys.path.insert(0, str(Path(__file__).parent / "golden"))
    from make_host_ref_golden import StubClip, StubT5, StubTok

    from gpt_image_edit_b200 import text_encoders as te
    from univa.utils import denoiser_prompt_embedding_flux as shim
    from univa.utils.anyres_util import compute_size, dynamic_resize, pick_ratio

    fx = torch.load(Path(__file__).parent / "golden" / "host_ref.pt", weights_only=False)
    assert len(fx["anyres"]) == 112
    for (mode, h, w), want in fx["anyres"].items():
        rw, rh = pick_ratio(h, w, anyres=mode)
        assert (rw, rh) == tuple(want["ratio"]), (mode, h, w)
        assert tuple(compute_size(rw, rh, stride=16, anchor_pixels=1024 * 1024)) == tuple(want["size16"])
        assert tuple(compute_size(rw, rh, stride=28, min_pixels=448 * 448, max_pixels=448 * 448)) == tuple(want["size28"])
        assert tuple(dynamic_resize(h, w, mode, anchor_pixels=1024 * 1024)) == tuple(want["dyn"])
        assert tuple(dynamic_resize(h, w, mode, anchor_pixels=512 * 512)) == tuple(want["dyn512"])
    toks, encs = [StubTok(100), StubTok(500)], [StubClip(), StubT5()]
    ep = fx["encode_prompt"]
    assert shim.encode_prompt is te.encode_prompt

    def same(got, want):
        assert (got is None) == (want is None)
        if want is not None:
            assert got.shape == want.shape and torch.equal(got, want)

    e, p = te.encode_prompt(encs, toks, ["turn the sky red", "b"], 16, device="cpu", num_images_per_prompt=3)
    same(e, ep["both_n3"]["embeds"]); same(p, ep["both_n3"]["pooled"])
    e, p = te.encode_prompt(encs, toks, "single", 8, device="cpu", num_images_per_prompt=1)
    same(e, ep["single"]["embeds"]); same(p, ep["single"]["pooled"])
    e, p = te.encode_prompt(encs, [None, toks[1]], "single", 8, device="cpu")
    same(e, ep["no_clip_tokenizer"]["embeds"]); same(p, ep["no_clip_tokenizer"]["pooled"])
    e, p = te.encode_prompt([encs[0], None], toks, "single", 8, device="cpu")
    same(e, ep["no_t5_encoder"]["embeds"]); same(p, ep["no_t5_encoder"]["pooled"])
    assert torch.equal(te.tokenize_prompt(toks[1], ["x y"], 6), ep["tokenize_prompt"])
    with pytest.raises(ValueError) as ei:
        te._encode_prompt_with_t5(encs[1], None, 8, "p")
    assert str(ei.value) == ep["error_no_ids"]


def test_cli_and_training_host_functions_match_the_references_source():
    """host_ref.pt["host"]: outputs of the reference's own `update_size` / `prepare_condition_images` (cli.py) and
    `get_trainable_params` / `check_param_is_in_components` (train_denoiser.py), whose function sources were executed
    by tests/golden/make_host_ref_golden.py."""
    from pathlib import Path

    from gpt_image_edit_b200.image_io import image_to_condition_tensor
    from oracle import flux_oracle as fo
    from univa.serve.cli import update_size

    h = torch.load(Path(__file__).parent / "golden" / "host_ref.pt", weights_only=False)["host"]
    imgs = h["images"]
    shape = lambda i: (imgs[i].shape[1], imgs[i].shape[0])                      # (w, h) as PIL reports it
    for (key, anchor), want in h["update_size"].items():
        shapes = [] if key == "none" else [shape(0), shape(2)] if key == "0+2" else [shape(key)]
        assert tuple(update_size(shapes, "any_11ratio", anchor_pixels=anchor)) == tuple(want), (key, anchor)
    assert torch.equal(image_to_condition_tensor(imgs[0]), h["condition"])     # [1,3,H,W] fp32 in [-1,1]
    # parameter-name contract (SURVEY.md §8b): every component the reference un-freezes names real parameters of the
    # denoiser, under the diffusers key names this repo's state_dict exposes
    keys = ["denoise_tower.denoiser." + k for k in fo.state_dict_spec(fo.FluxConfig())]
    for mode, comps in h["components"].items():
        for c in comps:
            assert any(c in k for k in keys), (mode, c)
    hit = lambda name, comps: any(c in name for c in comps)
    for mode, want in h["probe_result"].items():
        assert [hit(n, h["components"][mode]) for n in h["probe"]] == want
    n_default = sum(hit(k, h["components"]["default"]) for k in keys)
    n_both = sum(hit(k, h["components"]["both_branches"]) for k in keys)
    assert 0 < n_default < n_both < len(keys)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm): one JSON line on stdout with the
    same metric / unit / config as the GPU arm, `impl: reference`, a `cpu_baseline` describing the run and a zero-copy
    `e2e`.  (The sample is one double + one single block of the oracle at C1024 shapes: ~30 s on 8 cores.)"""
    import json
    import subprocess
    import sys
    from pathlib import Path

    root = Path(__file__).resolve().parent.parent
    r = subprocess.run([sys.executable, str(root / "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=900, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "edited images/sec @1024px 28-step" and d["unit"] == "images/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["config"]["workload"].startswith("C1024") and d["dtype"] == "f32"
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= cb["threads"] >= 1 and cb["value"] == d["value"] and "extrapolated" in cb["sample"]
    assert "qwen2.5-vl prefill" in cb["excluded"] and "libb2f" not in json.dumps(d["config"])     # the CPU arm describes itself
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert abs(d["ms_per_step"] - 1000.0 / d["value"]) / d["ms_per_step"] < 1e-6


def test_bench_cpu_extras_functions():
    """the one-off CPU timings of the reference arm (VAE encode + decode of the oracle) run and report seconds."""
    import importlib.util
    from pathlib import Path

    spec = importlib.util.spec_from_file_location("bench_mod", Path(__file__).resolve().parent.parent / "bench.py")
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    v = b.cpu_vae_seconds(64, 64, 2)
    assert v["vae_encode_s"] > 0 and v["vae_decode_s"] > 0


def test_bench_dump_outputs_float32_and_seeded_sample_past_the_limit(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: each array lands as <name>.npy in float32, exactly; past the size limit every run writes
    the same sample of elements, within the limit."""
    import importlib.util
    from pathlib import Path

    spec = importlib.util.spec_from_file_location("bench_mod", Path(__file__).resolve().parent.parent / "bench.py")
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    img = np.arange(2 * 4 * 4 * 3, dtype=np.uint8).reshape(2, 4, 4, 3)
    b.dump_outputs(tmp_path / "a", {"images": img})
    got = np.load(tmp_path / "a" / "images.npy")
    assert got.dtype == np.float32 and np.array_equal(got, img)
    monkeypatch.setattr(b, "DUMP_LIMIT_BYTES", 256)
    big = np.random.default_rng(1).random((20, 20))
    for d in ("b", "c"):
        b.dump_outputs(tmp_path / d, {"x": big, "y": big[:5]})
    x1, x2, y1 = (np.load(tmp_path / d / n) for d, n in (("b", "x.npy"), ("c", "x.npy"), ("b", "y.npy")))
    assert x1.dtype == np.float32 and x1.nbytes + y1.nbytes <= 256 and len(x1) > len(y1) > 0
    assert np.array_equal(x1, x2) and np.isin(x1, big.astype(np.float32)).all()


def test_ctypes_signatures_match_the_header():
    """every function include/b2f.h declares is bound in _lib._SIGNATURES with the same number and kinds of arguments
    (pointer / int / int64 / float / double / size_t) — a mismatch corrupts the call silently."""
    import ctypes as C
    import re

    from gpt_image_edit_b200 import _lib

    text = re.sub(r"/\*.*?\*/", "", _lib.HEADER_PATH.read_text(), flags=re.S)
    decls = re.findall(r"\b(?:int|void|size_t|int64_t|uint64_t|const char\*)\s+(b2f_[a-z0-9_]+)\s*\(([^;]*?)\)\s*;", text, flags=re.S)

    def kind(a):
        a = a.strip()
        if a in ("void", ""):
            return None
        if "*" in a or "b2f_stream_t" in a:
            return "p"
        for k, v in (("int64_t", "i64"), ("size_t", "sz"), ("float", "f"), ("double", "d"), ("int", "i")):
            if k in a:
                return v
        return "?"
    m = {C.c_void_p: "p", C.c_int64: "i64", C.c_int: "i", C.c_float: "f", C.c_double: "d", C.c_size_t: "sz", C.c_char_p: "p"}
    assert len(decls) >= 70
    for name, args in decls:
        want = [k for k in (kind(a) for a in args.split(",")) if k]
        have = [m.get(h, "p") for h in _lib._SIGNATURES[name][1]]
        assert want == have, (name, want, have)


def test_pipeline_check_inputs_rejects_what_the_reference_rejects():
    """`FluxKontextPipeline.check_inputs` against the outputs of the reference's own function source
    (tests/golden/check_inputs_ref.pt, made by make_check_inputs_golden.py): the same argument combinations are rejected,
    with a ValueError whose message starts the same way."""
    from pathlib import Path

    from gpt_image_edit_b200.pipeline import FluxKontextPipeline

    pipe = FluxKontextPipeline.__new__(FluxKontextPipeline)
    pipe.vae_scale_factor = 8
    ref = torch.load(Path(__file__).parent / "golden" / "check_inputs_ref.pt", weights_only=False)
    assert sum(r["raised"] for r in ref) >= 9 and sum(not r["raised"] for r in ref) >= 6
    for r in ref:
        try:
            pipe.check_inputs(**r["kwargs"])
            raised, msg = False, ""
        except ValueError as e:
            raised, msg = True, str(e)
        assert raised == r["raised"], (r["kwargs"], r["message"], msg)
        if raised:
            assert msg.split(":")[0].split(".")[0][:40] == r["message"].split(":")[0].split(".")[0][:40], (msg, r["message"])


def test_mixed_size_batches_match_the_reference_statements():
    """pad_x_and_mask and the loss weights / normalisation of mixed-size batches against tests/golden/mixed_size_ref.pt
    (the reference's own statements, train_denoiser.py:158-183 and :1104-1165, executed by make_mixed_size_golden.py)."""
    import torch
    from gpt_image_edit_b200.training import compute_loss_weighting_for_sd3, loss_weights, pad_x_and_mask
    from pathlib import Path
    ref = torch.load(Path(__file__).parent / "golden" / "mixed_size_ref.pt", weights_only=False)
    assert len(ref["cases"]) == 5
    for c in ref["cases"]:
        mixed = len(set(c["sizes"])) > 1
        if mixed:
            x, mask = pad_x_and_mask(c["unpad"], [torch.ones_like(t) for t in c["unpad"]])
            assert torch.equal(x, c["model_input"]) and torch.equal(mask, c["mask"]), c["name"]
        else:
            x, mask = c["model_input"], None
        B, C, h, w = x.shape
        sig = c["sigmas"]
        weighting = sig if c["sigmas_as_weight"] else compute_loss_weighting_for_sd3(c["scheme"], sig)
        area = c["area_weights"] if c["mask_weight_type"] is not None else None
        wt, scale = loss_weights(weighting, B, C, h, w, area_weights=area, weight_mask=mask,
                                 unpad_sizes=[tuple(t.shape[-2:]) for t in c["unpad"]] if mixed else None)
        assert torch.allclose(wt.expand(B, 1, h, w), c["weighting"], rtol=0, atol=0), c["name"]
        # what Stage2Trainer hands to the loss kernel: mean(scale * wt * err^2) over [B, C, h, w]
        err2 = (c["model_pred"].float() - c["target"].float()) ** 2
        loss = (scale * wt * err2).mean()
        assert abs(float(loss) - float(c["loss"])) <= 2e-6 * abs(float(c["loss"])), (c["name"], float(loss), float(c["loss"]))


def test_synthetic_dataset_collates_mixed_target_sizes_as_lists():
    """Targets of one size are stacked, targets of different sizes stay lists of [1, 3, H, W] / [1, 1, h, w] (what the
    reference's loop branches on, train_denoiser.py:907, 1120); the source image and the VLM inputs are stacked either way."""
    import torch
    from univa.training.synthetic_data import SyntheticEditDataset, collate

    ds = SyntheticEditDataset(64, 64, length=4, seed=3, target_sizes=[[64, 64], [48, 80]])
    a, b = ds[0], ds[1]
    assert a["generated_image"].shape == (3, 64, 64) and b["generated_image"].shape == (3, 48, 80)
    assert b["weights"].shape == (1, 6, 10) and b["ref_pixel_values"].shape == (3, 64, 64)
    assert torch.equal(ds[1]["generated_image"], b["generated_image"])            # a sample is a function of its index
    mixed = collate([a, b])
    assert isinstance(mixed["generated_image"], list) and [tuple(t.shape) for t in mixed["generated_image"]] == [(1, 3, 64, 64), (1, 3, 48, 80)]
    assert [tuple(t.shape) for t in mixed["weights"]] == [(1, 1, 8, 8), (1, 1, 6, 10)]
    assert mixed["ref_pixel_values"].shape == (2, 3, 64, 64) and mixed["input_ids"].shape[0] == 2
    same = collate([ds[0], ds[2]])
    assert same["generated_image"].shape == (2, 3, 64, 64) and same["weights"].shape == (2, 1, 8, 8)


def test_sigma_sampling_matches_the_reference_statements():
    """Stage2Trainer.sample_sigmas + the flow-matching noising against tests/golden/sigma_sampling_ref.pt: the reference's
    own statements (train_denoiser.py:935-995 and get_sigmas :779-788) executed on the CPU with the same seed — both the
    continuous branch (logit-normal sigmas with FLUX's resolution-dependent shift) and the discrete one."""
    from pathlib import Path
    from types import SimpleNamespace

    import torch
    from gpt_image_edit_b200.training import Stage2Trainer

    ref = torch.load(Path(__file__).parent / "golden" / "sigma_sampling_ref.pt", weights_only=False)
    assert len(ref["cases"]) == 5
    for c in ref["cases"]:
        gen = torch.Generator().manual_seed(c["seed"])        # the stream torch.manual_seed(seed) gives the global generator
        x = c["model_input"]
        noise = torch.randn(x.shape, generator=gen, dtype=x.dtype)
        assert torch.equal(noise, c["noise"]), c["name"]
        me = SimpleNamespace(tc=SimpleNamespace(discrete_timestep=c["discrete"], weighting_scheme=c["scheme"], logit_mean=0.0,
                                                logit_std=1.0, mode_scale=1.29),
                             sched=SimpleNamespace(config=c["sched"]), gen=gen)
        sigmas, timesteps = Stage2Trainer.sample_sigmas(me, x.shape[0], tuple(x.shape[-2:]), "cpu")
        assert torch.equal(sigmas.view(-1), c["sigmas"].view(-1)), (c["name"], sigmas, c["sigmas"].view(-1))
        assert torch.allclose(timesteps.view(-1), c["timesteps"].view(-1).float(), rtol=1e-6, atol=0), c["name"]
        s4 = sigmas.view(-1, 1, 1, 1)
        assert torch.equal((1.0 - s4) * x + s4 * noise, c["noisy"]), c["name"]


@pytest.mark.parametrize("name", ["constant", "constant_with_warmup", "linear", "cosine", "cosine_with_restarts", "polynomial"])
def test_lr_schedule_follows_diffusers_get_scheduler(name):
    """Stage2Trainer.lr_at against the LambdaLR multipliers of diffusers.optimization.get_scheduler (third party, absent
    here: its published lambdas are restated below) driven the way the reference drives it (train_denoiser.py:707-716:
    warm-up and total steps x num_processes, one scheduler.step() per process and optimizer step)."""
    import math
    from types import SimpleNamespace

    import torch
    from gpt_image_edit_b200.training import Stage2Trainer

    warm, total, procs, base, cycles = 5, 40, 8, 3e-4, (3 if name == "cosine_with_restarts" else 0.5)
    W, T = warm * procs, total * procs
    power, lr_end = 2.0, 1e-7

    def lam(k):                     # k = scheduler steps taken so far
        if name == "constant":
            return 1.0
        if k < W:
            return k / max(1, W)
        if name == "constant_with_warmup":
            return 1.0
        if name == "linear":
            return max(0.0, (T - k) / max(1, T - W))
        prog = (k - W) / max(1, T - W)
        if name == "cosine_with_restarts":
            return 0.0 if prog >= 1.0 else max(0.0, 0.5 * (1.0 + math.cos(math.pi * ((float(cycles) * prog) % 1.0))))
        if name == "polynomial":
            if k > T:
                return lr_end / base
            return ((base - lr_end) * (1 - (k - W) / (T - W)) ** power + lr_end) / base
        return max(0.0, 0.5 * (1.0 + math.cos(math.pi * cycles * 2.0 * prog)))

    opt = torch.optim.SGD([torch.nn.Parameter(torch.zeros(1))], lr=base)
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lam)
    me = SimpleNamespace(tc=SimpleNamespace(learning_rate=base, lr_warmup_steps=warm, max_train_steps=total, lr_scheduler=name,
                                            lr_num_cycles=cycles, lr_power=power))
    for step in range(total):
        want = opt.param_groups[0]["lr"]            # the rate optimizer.step() number `step` runs with
        got = Stage2Trainer.lr_at(me, step)
        assert abs(got - want) <= 1e-12 + 1e-9 * abs(want), (name, step, got, want)
        opt.step()
        for _ in range(procs):                      # accelerate's scheduler wrapper: one step per process
            sched.step()


def test_training_config_schema_matches_the_reference_dataclasses():
    """univa/training/configuration_denoise.py against tests/golden/config_schema_ref.json (the reference's own module,
    imported by make_config_golden.py): every reference field exists here with the same default; what this repo adds is
    listed; the reference's stage-2 yaml loads field by field, its stage-1 yaml (keys outside its own schema) is rejected."""
    import dataclasses
    import json
    from pathlib import Path

    from univa.training import configuration_denoise as C

    ref = json.loads((Path(__file__).parent / "golden" / "config_schema_ref.json").read_text())
    additions = {"TrainingConfig": set(), "DatasetConfig": {"synthetic_len", "synthetic_target_sizes"},
                 "ModelConfig": {"synthetic", "small"}}
    from univa.eval import configuration_eval as E
    additions["EvalConfig"] = {"synthetic", "small"}
    for cls, fields in ref["classes"].items():
        ours = {f.name: f for f in dataclasses.fields(getattr(E if cls == "EvalConfig" else C, cls))}
        assert set(fields) <= set(ours), (cls, sorted(set(fields) - set(ours)))
        assert set(ours) - set(fields) <= additions[cls], (cls, sorted(set(ours) - set(fields)))
        for name, rf in fields.items():
            if rf["has_default"]:
                assert ours[name].default == rf["default"], (cls, name, ours[name].default, rf["default"])
    with pytest.raises(KeyError):
        E.EvalConfig.from_mapping({"num_inference_step": 28})          # a typo is an error, as under OmegaConf
    assert E.EvalConfig.from_mapping({"guidance_scale": 4, "height": 512}).guidance_scale == 4.0
    for yname, rec in ref["yamls"].items():
        raw = {sec: dict(v["values"]) for sec, v in rec.items()}
        unknown = [k for v in rec.values() for k in v["unknown"]]
        if unknown:
            # the values fixture keeps scalars only: put the unknown keys back so the loader sees them
            raw["model_config"].update({k: None for k in rec["model_config"]["unknown"]})
            with pytest.raises(Exception):
                C.from_mapping(raw)
        else:
            conf = C.from_mapping(raw)
            for sec, v in rec.items():
                for k, val in v["values"].items():
                    got = getattr(getattr(conf, sec), k)
                    if isinstance(val, str) and isinstance(got, (int, float)) and not isinstance(got, bool):
                        val = float(val)            # PyYAML reads `1e-8` as a string; the typed schema makes it a float
                    assert got == val or (isinstance(val, (int, float)) and float(got) == float(val)), (yname, sec, k, got, val)


def test_training_token_inputs_match_the_reference_statements():
    """training.pack_training_latents over the product pipeline's helpers against tests/golden/train_pack_ref.pt: the
    reference's own statements (train_denoiser.py:998-1056) run with the reference's own FluxKontextPipeline helpers and the
    same stub VAE — tokens and position ids of [noised target ‖ context], a context of another size, no context."""
    import sys
    from pathlib import Path
    from types import SimpleNamespace

    import torch

    sys.path.insert(0, str(Path(__file__).parent / "golden"))
    from gpt_image_edit_b200.pipeline import FluxKontextPipeline
    from gpt_image_edit_b200.training import pack_training_latents

    class StubVae:      # the same fixed arithmetic as tests/golden/make_train_pack_golden.py::StubVae
        dtype = torch.float32

        def __init__(self):
            self.config = SimpleNamespace(block_out_channels=(1, 1, 1, 1), latent_channels=16, scaling_factor=0.3611,
                                          shift_factor=0.1159)

        def encode(self, x):
            z = torch.nn.functional.avg_pool2d(x.float(), 8)
            ch = torch.arange(16, dtype=torch.float32).view(1, 16, 1, 1)
            z = z[:, :1] * (1 + 0.1 * ch) + z[:, 1:2] * 0.01 * ch + z[:, 2:3]
            return SimpleNamespace(latent_dist=SimpleNamespace(mode=lambda: z, sample=lambda generator=None: z))

    pipe = FluxKontextPipeline(transformer=SimpleNamespace(device=torch.device("cpu")), vae=StubVae())
    assert pipe.vae_scale_factor == 8
    ref = torch.load(Path(__file__).parent / "golden" / "train_pack_ref.pt", weights_only=False)
    assert [c["name"] for c in ref["cases"]] == ["context_same_size", "context_other_size", "no_context"]
    for c in ref["cases"]:
        tokens, ids = pack_training_latents(pipe, c["noisy"], c["cond"], torch.device("cpu"), torch.float32)
        assert torch.equal(tokens, c["tokens"]), c["name"]
        assert torch.equal(ids.float(), c["ids"].float()), c["name"]


def test_resume_resolution_and_checkpoint_pruning_match_the_reference_statements(tmp_path):
    """train_denoiser.resolve_resume_checkpoint / prune_checkpoints against the outputs of the reference's own statements
    (train_denoiser.py:348-374, 1195-1225; tests/golden/make_train_resume_golden.py) on the same directory trees."""
    import json
    import os
    from pathlib import Path
    from types import SimpleNamespace

    import train_denoiser as td

    fx = json.loads((Path(__file__).parent / "golden" / "train_resume_ref.json").read_text())
    for i, c in enumerate(fx["resume"]):
        out = tmp_path / f"r{i}"
        for d in c["dirs"]:
            (out / d).mkdir(parents=True)
        said = []
        tc = SimpleNamespace(resume_from_checkpoint=c["resume_from_checkpoint"], output_dir=str(out))
        path, step = td.resolve_resume_checkpoint(tc, log=said.append)
        assert (None if path is None else os.path.relpath(path, out)) == c["chosen"], c
        assert step == c["initial_global_step"] and said == c["said"], c
    with pytest.raises(FileNotFoundError):       # an explicit checkpoint that is not there: the reference dies in load_state
        td.resolve_resume_checkpoint(SimpleNamespace(resume_from_checkpoint="checkpoint-7", output_dir=str(tmp_path / "r0")),
                                     log=lambda *_: None)
    for i, c in enumerate(fx["prune"]):
        out = tmp_path / f"p{i}"
        for d in c["dirs"]:
            (out / d).mkdir(parents=True)
        said = []
        td.prune_checkpoints(out, c["limit"], log=said.append)
        assert sorted(os.listdir(out)) == c["left"] and said == c["said"], c


def test_univa_config_is_read_from_both_config_json_layouts():
    """The Univa checkpoint's config.json is written by transformers 4.50 (the reference's pin): language-model fields at the
    top level, M-RoPE under `rope_scaling`, `in_chans` in the vision block, `denoise_tower` next to them
    (configuration_univa_qwen2p5vl.py:7-52).  transformers 5 nests the language model under `text_config`."""
    from gpt_image_edit_b200.checkpoint import univa_config_kwargs
    from univa.models.qwen2p5vl.modeling_univa_qwen2p5vl import UnivaQwen2p5VLConfig

    flat = {"architectures": ["UnivaQwen2p5VLForConditionalGeneration"], "hidden_size": 2048, "intermediate_size": 11008,
            "num_attention_heads": 16, "num_hidden_layers": 36, "num_key_value_heads": 2, "rms_norm_eps": 1e-06,
            "rope_theta": 1000000.0, "rope_scaling": {"type": "mrope", "mrope_section": [16, 24, 24]}, "vocab_size": 151936,
            "image_token_id": 151655, "video_token_id": 151656, "vision_start_token_id": 151652, "tie_word_embeddings": True,
            "vision_config": {"depth": 32, "hidden_size": 1280, "intermediate_size": 3420, "num_heads": 16, "in_chans": 3,
                              "out_hidden_size": 2048, "patch_size": 14, "spatial_merge_size": 2, "window_size": 112,
                              "fullatt_block_indexes": [7, 15, 23, 31], "tokens_per_second": 2, "temporal_patch_size": 2,
                              "hidden_act": "silu"},
            "denoise_tower": {"denoiser_type": "flux", "denoise_projector_type": "mlp2x_gelu", "output_hidden_size": 4096,
                              "denoiser_config": {"num_layers": 19, "num_single_layers": 38}}}
    cfg = UnivaQwen2p5VLConfig(**univa_config_kwargs(flat))
    tc, vc = cfg.text_config, cfg.vision_config
    assert (tc.hidden_size, tc.num_hidden_layers, tc.num_attention_heads, tc.num_key_value_heads) == (2048, 36, 16, 2)
    assert tc.intermediate_size == 11008 and tc.vocab_size == 151936 and tuple(tc.mrope_section) == (16, 24, 24)
    assert vc.out_hidden_size == 2048 and vc.in_channels == 3 and tuple(vc.fullatt_block_indexes) == (7, 15, 23, 31)
    assert cfg.denoise_tower.input_hidden_size == 2048 and cfg.denoise_tower.output_hidden_size == 4096   # :44-45
    assert cfg.denoise_tower.denoiser_config["num_single_layers"] == 38 and cfg.hidden_size == 2048
    nested = {"text_config": {k: flat[k] for k in ("hidden_size", "intermediate_size", "num_attention_heads",
                                                    "num_hidden_layers", "num_key_value_heads", "vocab_size")} |
              {"rope_parameters": {"rope_type": "default", "rope_theta": 5e5, "mrope_section": [8, 12, 12]}},
              "vision_config": flat["vision_config"], "image_token_id": 900, "vision_start_token_id": 902}
    cfg2 = UnivaQwen2p5VLConfig(**univa_config_kwargs(nested))
    assert cfg2.text_config.hidden_size == 2048 and tuple(cfg2.text_config.mrope_section) == (8, 12, 12)
    assert cfg2.text_config.rope_theta == 5e5 and cfg2.image_token_id == 900 and cfg2.text_config.vision_start_token_id == 902
    # nothing given: the Qwen2.5-VL-7B sizes of the released checkpoint
    cfg3 = UnivaQwen2p5VLConfig(**univa_config_kwargs({}))
    assert (cfg3.text_config.hidden_size, cfg3.text_config.num_hidden_layers, cfg3.vision_config.depth) == (3584, 28, 32)
    with pytest.raises(Exception, match="shortcut_image_embeds"):
        UnivaQwen2p5VLConfig(**univa_config_kwargs({"shortcut_image_embeds": True}))


def test_which_flux_layers_train_follows_the_reference_rule():
    """train_denoiser.py:527-543: `only_tune_mlp2` trains no FLUX tensor; otherwise the components of `flux_train_layer_idx`
    — and the schema's default None un-freezes nothing (the guard `is not None` at :531), although get_trainable_params'
    own default would list all 57 blocks."""
    from types import SimpleNamespace

    from gpt_image_edit_b200.training import get_trainable_params, trained_flux_layers

    mc = lambda **k: SimpleNamespace(**{**dict(only_tune_mlp2=False, flux_train_layer_idx=None), **k})
    assert trained_flux_layers(mc()) == []
    assert trained_flux_layers(mc(flux_train_layer_idx=[0, 20])) == [0, 20]
    assert trained_flux_layers(mc(only_tune_mlp2=True, flux_train_layer_idx=list(range(57)))) == []
    assert get_trainable_params(trained_flux_layers(mc())) == [] and len(get_trainable_params(None)) == 19 * 7 + 38 * 6
    from univa.training.configuration_denoise import load_config
    from pathlib import Path
    conf = load_config(Path(__file__).parent.parent / "scripts" / "denoiser" / "flux_qwen2p5vl_7b_vlm_stage2_512_synthetic.yaml")
    assert trained_flux_layers(conf.model_config) == list(range(57))       # BASELINE.json configs[3] trains all 57 blocks


def test_collate_pads_ragged_prompts_like_the_references_collator():
    """univa/dataset/data_collator.py:113-121: pad_sequence with the pad token on the configured side, mask = ids != pad."""
    from univa.training.synthetic_data import PAD_TOKEN_ID, SyntheticEditDataset, collate

    a = SyntheticEditDataset(64, 64, seed=1, n_text=5)[0]
    b = SyntheticEditDataset(64, 64, seed=1, n_text=9)[1]
    la, lb = a["input_ids"].numel(), b["input_ids"].numel()
    assert lb == la + 4
    for side in ("right", "left"):
        out = collate([a, b], padding_side=side)
        ids, mask = out["input_ids"], out["attention_mask"]
        assert ids.shape == (2, lb) and mask.dtype == torch.long and mask.sum().item() == la + lb
        pad = slice(la, lb) if side == "right" else slice(0, 4)
        assert torch.all(ids[0, pad] == PAD_TOKEN_ID) and torch.all(mask[0, pad] == 0) and torch.all(mask[1] == 1)
        real = ids[0, :la] if side == "right" else ids[0, 4:]
        assert torch.equal(real, a["input_ids"])
    same = collate([a, a])
    assert torch.equal(same["input_ids"], torch.stack([a["input_ids"]] * 2)) and bool(same["attention_mask"].all())


def test_settings_the_engine_cannot_honour_are_refused_not_ignored():
    """train_denoiser.unsupported_settings: the synthetic stage-2 yaml is clean; the reference's own stage-2 yaml differs only
    by its dataset (recorded in tests/golden/config_schema_ref.json); every knob that would change what is trained is named."""
    import json
    from pathlib import Path

    import train_denoiser as td
    from univa.training.configuration_denoise import from_mapping, load_config

    root = Path(__file__).parent.parent
    ours = load_config(root / "scripts" / "denoiser" / "flux_qwen2p5vl_7b_vlm_stage2_512_synthetic.yaml")
    assert td.unsupported_settings(ours) == []
    shipped = json.loads((root / "tests" / "golden" / "config_schema_ref.json").read_text())["yamls"]
    # the yaml's own key / value pairs, without the keys its own schema rejects (mlp3 / siglip leftovers in the shipped files)
    values = lambda rec: {sec: {k: v for k, v in rec[sec]["values"].items() if k not in rec[sec]["unknown"]} for sec in rec}
    stage2 = values(next(v for k, v in shipped.items() if "stage2" in k))
    bad = td.unsupported_settings(from_mapping(stage2))
    assert len(bad) == 1 and bad[0].startswith("dataset_config.dataset_type")
    stage1 = values(next(v for k, v in shipped.items() if "stage1" in k))  # MLP2 only: only_tune_image_branch=false is moot
    assert [b.split("=")[0].split(":")[0] for b in td.unsupported_settings(from_mapping(stage1))] == [
        "training_config.ema_deepspeed_config_file", "dataset_config.dataset_type"]          # stage 1 also runs the EMA engine
    base = dict(training_config={}, model_config=dict(synthetic=True, flux_train_layer_idx=[0]),
                dataset_config=dict(dataset_type="synthetic"))
    def names(**over):
        m = {k: dict(v) for k, v in base.items()}
        for k, v in over.items():
            sec, field = k.split("__")
            m[sec][field] = v
        return [b.split(":")[0].split("=")[0].split(" ")[0] for b in td.unsupported_settings(from_mapping(m))]
    assert names() == []
    assert names(training_config__mixed_precision="fp16") == ["training_config.mixed_precision"]
    assert names(training_config__optimizer="prodigy") == ["training_config.optimizer"]
    assert names(training_config__ema_deepspeed_config_file="zero3.json") == ["training_config.ema_deepspeed_config_file"]
    assert names(training_config__drop_condition_rate=0.1, training_config__drop_t5_rate=0.5) == [
        "training_config.drop_condition_rate", "training_config.drop_t5_rate"]
    assert names(model_config__only_tune_image_branch=False) == ["model_config.only_tune_image_branch"]
    assert names(model_config__only_tune_image_branch=False, model_config__only_tune_mlp2=True) == []   # stage 1: MLP2 only
    assert names(model_config__vlm_residual_image_factor=0.3) == ["model_config.vlm_residual_image_factor"]


def test_univa_checkpoint_assembly_from_qwen_and_flux_directories(tmp_path):
    """scripts/make_univa_qwen2p5vl_weight.py (reference scripts/make_univa_qwen2p5vl_weight.py:35-76): Qwen2.5-VL tensors under
    their own names, FLUX under `denoise_tower.denoiser.`, a fresh MLP2, the merged config.json and the processor files — the
    directory layout gpt_image_edit_b200.checkpoint.load_univa_checkpoint reads."""
    import importlib.util
    import json
    from pathlib import Path

    from safetensors.torch import save_file

    from gpt_image_edit_b200.checkpoint import PROCESSOR_FILES, load_state_dict_from_dir, univa_config_kwargs
    from univa.models.qwen2p5vl.modeling_univa_qwen2p5vl import UnivaQwen2p5VLConfig

    spec = importlib.util.spec_from_file_location("mk", Path(__file__).parent.parent / "scripts" / "make_univa_qwen2p5vl_weight.py")
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    g = torch.Generator().manual_seed(0)
    q, f = tmp_path / "qwen", tmp_path / "flux" / "transformer"
    q.mkdir()
    f.mkdir(parents=True)
    qsd = {"visual.patch_embed.proj.weight": torch.randn(8, 12, generator=g), "model.embed_tokens.weight": torch.randn(50, 16, generator=g),
           "model.layers.0.self_attn.q_proj.weight": torch.randn(16, 16, generator=g), "lm_head.weight": torch.randn(50, 16, generator=g)}
    save_file({k: v for k, v in list(qsd.items())[:2]}, str(q / "model-00001-of-00002.safetensors"))
    save_file({k: v for k, v in list(qsd.items())[2:]}, str(q / "model-00002-of-00002.safetensors"))
    (q / "config.json").write_text(json.dumps({"model_type": "qwen2_5_vl", "hidden_size": 16, "num_hidden_layers": 1,
                                               "num_attention_heads": 2, "num_key_value_heads": 1, "intermediate_size": 32,
                                               "vocab_size": 50, "initializer_range": 0.02, "image_token_id": 45,
                                               "vision_config": {"depth": 1, "hidden_size": 8, "out_hidden_size": 16}}))
    (q / "tokenizer_config.json").write_text("{}")
    (q / "preprocessor_config.json").write_text("{}")
    fsd = {"transformer_blocks.0.attn.to_q.weight": torch.randn(4, 4, generator=g), "proj_out.bias": torch.randn(4, generator=g)}
    save_file(fsd, str(f / "diffusion_pytorch_model.safetensors"))
    (f / "config.json").write_text(json.dumps({"_class_name": "FluxTransformer2DModel", "num_layers": 1, "num_single_layers": 1,
                                               "guidance_embeds": True}))
    out = tmp_path / "univa"
    info = mk.assemble(q, f.parent, out, dtype=torch.bfloat16, seed=3, max_shard_bytes=2000, log=lambda *_: None)
    sd = load_state_dict_from_dir(out)
    want = set(qsd) | {"denoise_tower.denoiser." + k for k in fsd} | {f"denoise_tower.denoise_projector.{i}.{p}"
                                                                      for i in (0, 2) for p in ("weight", "bias")}
    assert set(sd) == want and info["tensors"] == len(want) and len(info["shards"]) > 1
    assert all(t.dtype == torch.bfloat16 for t in sd.values())
    assert torch.equal(sd["model.embed_tokens.weight"], qsd["model.embed_tokens.weight"].bfloat16())
    assert torch.equal(sd["denoise_tower.denoiser.proj_out.bias"], fsd["proj_out.bias"].bfloat16())
    assert sd["denoise_tower.denoise_projector.0.weight"].shape == (3 * 4096, 16)          # Linear(hidden, 3 * 4096)
    assert sd["denoise_tower.denoise_projector.2.weight"].shape == (4096, 3 * 4096)
    assert float(sd["denoise_tower.denoise_projector.2.bias"].abs().max()) == 0
    assert abs(float(sd["denoise_tower.denoise_projector.0.weight"].float().std()) - 0.02) < 2e-3
    index = json.loads((out / "model.safetensors.index.json").read_text())
    assert set(index["weight_map"]) == want and set(index["weight_map"].values()) == set(info["shards"])
    cfg = json.loads((out / "config.json").read_text())
    assert cfg["model_type"] == "univa_qwen2p5vl" and cfg["architectures"] == ["UnivaQwen2p5VLForConditionalGeneration"]
    assert cfg["denoise_tower"]["input_hidden_size"] == 16 and cfg["denoise_tower"]["denoiser_config"]["num_single_layers"] == 1
    ucfg = UnivaQwen2p5VLConfig(**univa_config_kwargs(cfg))                                 # what the loader builds from it
    assert ucfg.hidden_size == 16 and ucfg.image_token_id == 45 and ucfg.denoise_tower.output_hidden_size == 4096
    assert ucfg.denoise_tower.denoiser_config["guidance_embeds"] is True
    assert any((out / n).exists() for n in PROCESSOR_FILES) and (out / "preprocessor_config.json").exists()
    with pytest.raises(KeyError):                                                            # not a plain Qwen2.5-VL directory
        mk.assemble(out, f.parent, tmp_path / "again", log=lambda *_: None)


def test_training_checkpoint_writes_a_loadable_univa_directory(tmp_path):
    """train_denoiser.write_univa_directory / checkpoint.rewrite_checkpoint (reference save hook, train_denoiser.py:489-498:
    `save_pretrained(checkpoint-N/univa)` + the processor files): trained tensors replaced, everything else byte-identical to
    the source checkpoint, side files carried along; a synthetic run writes no such directory."""
    import json
    from types import SimpleNamespace

    from safetensors.torch import save_file

    import train_denoiser as td
    from gpt_image_edit_b200.checkpoint import load_state_dict_from_dir, rewrite_checkpoint

    g = torch.Generator().manual_seed(1)
    src = tmp_path / "src"
    src.mkdir()
    sd = {"model.embed_tokens.weight": torch.randn(10, 4, generator=g).bfloat16(),
          "denoise_tower.denoiser.transformer_blocks.0.attn.to_q.weight": torch.randn(4, 4, generator=g).bfloat16(),
          "denoise_tower.denoiser.transformer_blocks.0.ff.net.2.weight": torch.randn(4, 4, generator=g).bfloat16(),
          "denoise_tower.denoise_projector.0.weight": torch.randn(6, 4, generator=g).bfloat16()}
    save_file({k: sd[k] for k in list(sd)[:2]}, str(src / "model-00001-of-00002.safetensors"))
    save_file({k: sd[k] for k in list(sd)[2:]}, str(src / "model-00002-of-00002.safetensors"))
    (src / "config.json").write_text(json.dumps({"model_type": "univa_qwen2p5vl"}))
    (src / "tokenizer_config.json").write_text("{}")
    trained = {"transformer_blocks.0.attn.to_q.weight": torch.full((4, 4), 2.0)}                    # fp32 in, stored dtype out
    proj = {"denoise_tower.denoise_projector.0.weight": torch.full((6, 4), -1.0)}
    mc = SimpleNamespace(pretrained_lvlm_name_or_path=str(src), synthetic=False)
    out = td.write_univa_directory(mc, tmp_path / "checkpoint-5", trained, proj, log=lambda *_: None)
    assert out == tmp_path / "checkpoint-5" / "univa"
    got = load_state_dict_from_dir(out)
    assert set(got) == set(sd) and all(got[k].dtype == torch.bfloat16 for k in got)
    assert torch.all(got["denoise_tower.denoiser.transformer_blocks.0.attn.to_q.weight"] == 2.0)
    assert torch.all(got["denoise_tower.denoise_projector.0.weight"] == -1.0)
    for frozen in ("model.embed_tokens.weight", "denoise_tower.denoiser.transformer_blocks.0.ff.net.2.weight"):
        assert torch.equal(got[frozen], sd[frozen])
    assert json.loads((out / "config.json").read_text())["model_type"] == "univa_qwen2p5vl" and (out / "tokenizer_config.json").exists()
    assert td.write_univa_directory(SimpleNamespace(pretrained_lvlm_name_or_path=str(src), synthetic=True), tmp_path / "c2", trained,
                                    proj) is None
    assert td.write_univa_directory(SimpleNamespace(pretrained_lvlm_name_or_path="", synthetic=False), tmp_path / "c3", trained,
                                    proj) is None
    with pytest.raises(KeyError):                # a trained tensor the source does not have
        rewrite_checkpoint(src, tmp_path / "bad", {"denoise_tower.denoiser.nope": torch.zeros(1)})
    with pytest.raises(ValueError):              # or has with another shape
        rewrite_checkpoint(src, tmp_path / "bad2", {"model.embed_tokens.weight": torch.zeros(3, 3)})


def test_save_pretrained_layout_and_config_round_trip(tmp_path):
    """UnivaQwen2p5VLConfig.to_dict -> config.json -> univa_config_kwargs -> UnivaQwen2p5VLConfig is the identity on every field
    the engine reads; save_univa_model (what `save_pretrained` calls) writes the checkpoint key names over any object with
    the model's protocol (`lvlm`, `denoise_tower.denoiser`, `denoise_tower.denoise_projector`, `config`)."""
    import json
    from types import SimpleNamespace

    from gpt_image_edit_b200.checkpoint import load_state_dict_from_dir, save_univa_model, univa_config_kwargs
    from univa.models.qwen2p5vl.modeling_univa_qwen2p5vl import UnivaQwen2p5VLConfig, UnivaQwen2p5VLForConditionalGeneration

    cfg = UnivaQwen2p5VLConfig(text_config=dict(hidden_size=64, num_hidden_layers=3, num_attention_heads=2, num_key_value_heads=1,
                                                intermediate_size=96, vocab_size=321, rope_theta=5e5, mrope_section=(8, 12, 12)),
                               vision_config=dict(depth=2, hidden_size=32, num_heads=2, intermediate_size=40, out_hidden_size=64,
                                                  fullatt_block_indexes=(1,)),
                               denoise_tower=dict(output_hidden_size=128, denoiser_config=dict(num_layers=2, num_single_layers=3,
                                                                                               axes_dims_rope=(16, 56, 56))),
                               image_token_id=300, video_token_id=301, vision_start_token_id=302)
    raw = json.loads(json.dumps(cfg.to_dict()))                                  # through JSON, as config.json
    assert raw["model_type"] == "univa_qwen2p5vl" and raw["hidden_size"] == 64 and raw["rope_scaling"]["mrope_section"] == [8, 12, 12]
    back = UnivaQwen2p5VLConfig(**univa_config_kwargs(raw))
    for k in ("hidden_size", "num_hidden_layers", "num_attention_heads", "num_key_value_heads", "intermediate_size", "vocab_size",
              "rope_theta", "rms_norm_eps", "image_token_id", "vision_start_token_id"):
        assert getattr(back.text_config, k) == getattr(cfg.text_config, k), k
    assert tuple(back.text_config.mrope_section) == (8, 12, 12)
    for k in ("depth", "hidden_size", "num_heads", "intermediate_size", "out_hidden_size", "in_channels", "patch_size", "window_size"):
        assert getattr(back.vision_config, k) == getattr(cfg.vision_config, k), k
    assert tuple(back.vision_config.fullatt_block_indexes) == (1,)
    assert back.denoise_tower.input_hidden_size == 64 and back.denoise_tower.output_hidden_size == 128
    assert back.denoise_tower.denoiser_config["num_single_layers"] == 3 and (back.image_token_id, back.video_token_id) == (300, 301)
    sd_of = lambda d: SimpleNamespace(state_dict=lambda: d)
    model = SimpleNamespace(config=cfg, lvlm=sd_of({"visual.merger.ln_q.weight": torch.ones(4), "model.norm.weight": torch.ones(4),
                                                    "lm_head.weight": torch.zeros(2, 4)}),
                            denoise_tower=SimpleNamespace(denoiser=sd_of({"proj_out.bias": torch.ones(3)}),
                                                          denoise_projector=sd_of({"0.weight": torch.ones(2, 2)})))
    wm = save_univa_model(model, tmp_path / "univa")
    got = load_state_dict_from_dir(tmp_path / "univa")
    assert set(got) == set(wm) == {"visual.merger.ln_q.weight", "model.norm.weight", "lm_head.weight", "denoise_tower.denoiser.proj_out.bias",
                                   "denoise_tower.denoise_projector.0.weight"}
    assert json.loads((tmp_path / "univa" / "config.json").read_text())["denoise_tower"]["output_hidden_size"] == 128
    assert hasattr(UnivaQwen2p5VLForConditionalGeneration, "from_pretrained") and hasattr(UnivaQwen2p5VLForConditionalGeneration, "save_pretrained")
    from gpt_image_edit_b200 import _lib
    with pytest.raises(_lib.B2FError, match="bf16"):
        UnivaQwen2p5VLForConditionalGeneration.from_pretrained(str(tmp_path / "univa"), torch_dtype=torch.float32)
