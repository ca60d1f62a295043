#!/usr/bin/env python
"""bench.py — edited images/sec at 1024x1024, 28 Euler steps (BASELINE.json metric), N GPUs of one box.

  python bench.py --gpus 1 --steps K --warmup W            (N>1: launched by torch.distributed.run)
  python bench.py --impl reference ...                      CPU arm: the oracle restatement of the
                                                            reference's diffusers path on host cores
  python bench.py ... --dump-outputs DIR                    also writes the last timed edit's images as
                                                            DIR/images.npy, to compare two builds

One "step" = one complete edit of one batch of synthetic (source image, instruction-embedding) pairs:
the FluxKontextPipeline call (VAE-encode of the context image when a VAE is attached, 28 MMDiT
forwards + Euler updates, VAE-decode).  Workload = BASELINE.json configs[1] ("C1024", SURVEY.md §8d):
B=1 per GPU, S_txt=544, S_tgt=S_ctx=4096, d=3072, 19+38 blocks, bf16, seeded synthetic weights
(no checkpoints exist offline).  Multi-GPU = batch sharding: every rank owns a full replica
(weights broadcast once from rank 0 over NCCL) and its own batch items; no collective in the loop.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

D_MODEL, N_DOUBLE, N_SINGLE, S_TXT = 3072, 19, 38, 544
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes every array as out_dir/<name>.npy in float32.  When they exceed DUMP_LIMIT_BYTES together, each is replaced
    by the same fixed, seeded sample of its flattened elements (sorted indices), so two builds run with the same arguments
    still compare element for element."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_LIMIT_BYTES:
            n = a.size * DUMP_LIMIT_BYTES // total
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, n, replace=False))]
        np.save(d / f"{name}.npy", a)


def flops_per_forward(S_img: int, S_txt: int, n_double=N_DOUBLE, n_single=N_SINGLE, d=D_MODEL, joint=4096) -> float:
    """Algorithmic FLOPs of one MMDiT forward per sample (SURVEY.md §8d formula, generalised)."""
    S = S_img + S_txt
    nb = n_double + n_single
    lin = nb * 24.0 * d * d * S                 # qkv/out/mlp projections of every block
    attn = nb * 4.0 * S * S * d                 # QK^T and PV
    emb = 2.0 * S_img * 64 * d * 2 + 2.0 * S_txt * joint * d
    ada = 2.0 * (n_double * 12 + n_single * 3 + 2) * d * d
    return lin + attn + emb + ada


def ncu_traffic(kernel_class: str):
    """DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) per launch of the dominant kernel class, from the newest
    committed `ncu --set full` summary under profiles/ that holds a launch of that class (scripts/ncu_summary.py output);
    None when no capture of that class is committed — the figure is never borrowed from another kernel."""
    want = "attn" if kernel_class == "attention" else "gemm"
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    # captures of the training step (scripts/profile_train.py) hold dgrad / wgrad launches: not this workload's kernels
    files = [f for f in (ROOT / "profiles").glob("r*_ncu_full*summary.json") if "train" not in f.name]
    for f in sorted(files, reverse=True):
        try:
            launches = json.loads(f.read_text())["launches"]
        except Exception:
            continue
        best = None
        for rec in launches:
            if want not in rec.get("kernel", ""):
                continue
            try:
                rd, wr = rec["dram__bytes_read.sum"].split(), rec["dram__bytes_write.sum"].split()
                tot = float(rd[0]) * scale[rd[1]] + float(wr[0]) * scale[wr[1]]
                dur = float(rec["gpu__time_duration.sum"].split()[0])
            except Exception:
                continue
            if best is None or dur > best[1]:
                best = (tot, dur, rec.get("kernel", ""), rec.get("what", ""))
        if best is not None:
            return {"dram_bytes_per_launch": best[0], "launch_us_under_ncu": best[1], "kernel": best[2], "launch": best[3],
                    "source": f"profiles/{f.name} (longest captured launch of the class)"}
    return None


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        j = json.loads(p.read_text())
        return dict(tensor_burst=j["bf16_tflops"], tensor_sustained=j["bf16_tflops_sustained"], hbm=j["hbm_gbs"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(tensor_burst=1590.0, tensor_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 8 for n, v in zip(names, r[4:8]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- CPU arm
_BEST_THREADS = None


def best_thread_count() -> int:
    """The host thread count that runs an fp32 GEMM fastest (on the 128-core GPU box all 128 threads were slower than
    8 on a small container: NUMA / oversubscription), so the CPU baseline is not handicapped by its thread setting."""
    global _BEST_THREADS
    if _BEST_THREADS is None:
        n = os.cpu_count() or 1
        a = torch.randn(4096, 3072)
        b = torch.randn(3072, 3072)
        best = (float("inf"), n)
        for t in sorted({n, max(n // 2, 1), max(n // 4, 1), min(n, 32), min(n, 16), min(n, 8)}, reverse=True):
            torch.set_num_threads(t)
            a @ b
            t0 = time.perf_counter()
            for _ in range(3):
                a @ b
            dt = time.perf_counter() - t0
            if dt < best[0] * 0.97:
                best = (dt, t)
        _BEST_THREADS = best[1]
    return _BEST_THREADS


def cpu_reference_sample(height: int, width: int, steps_28: int, threads: int | None = None) -> dict:
    """Times the oracle (PyTorch restatement of the reference's diffusers arithmetic, fp32) on host
    cores for ONE double-stream + ONE single-stream block at the full C1024 shapes, then extrapolates
    x19 / x38 / x28 steps to seconds per image (labelled as extrapolated)."""
    from oracle import flux_oracle as fo

    threads = threads or best_thread_count()
    torch.set_num_threads(threads)
    S_img = 2 * (height // 16) * (width // 16)
    cfg = fo.FluxConfig(num_layers=1, num_single_layers=1)
    sd = fo.make_synthetic_state_dict(cfg, seed=0, dtype=torch.float32)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, S_img, D_MODEL, generator=g)
    c = torch.randn(1, S_TXT, D_MODEL, generator=g)
    temb = torch.randn(1, D_MODEL, generator=g)
    ids = torch.zeros(S_TXT + S_img, 3)
    cos, sin = fo.rope_tables(ids)
    with torch.no_grad():
        t0 = time.perf_counter()
        c2, x2 = fo.double_block(sd, 0, cfg, x, c, temb, cos, sin)
        t_d = time.perf_counter() - t0
        h = torch.cat([c2, x2], 1)
        t0 = time.perf_counter()
        fo.single_block(sd, 0, cfg, h, temb, cos, sin)
        t_s = time.perf_counter() - t0
    sec_per_image = steps_28 * (N_DOUBLE * t_d + N_SINGLE * t_s)
    return dict(value=1.0 / sec_per_image, unit="images/s", cores=os.cpu_count() or 1, threads=threads, kind="port",
                sample=f"oracle fp32: 1 double ({t_d:.2f}s) + 1 single ({t_s:.2f}s) block at S={S_TXT + S_img}, d={D_MODEL}; "
                       f"extrapolated x{N_DOUBLE}/x{N_SINGLE} blocks x{steps_28} steps (VAE/conditioning excluded)",
                excluded=["vae_encode", "vae_decode", "qwen2.5-vl prefill", "mlp2", "t5-xxl", "clip-l"],
                sec_per_image_extrapolated=sec_per_image)


def cpu_vae_seconds(height: int, width: int, threads: int) -> dict:
    """Oracle FLUX VAE (fp32) encode + decode of one image on host cores, measured once (BASELINE.md section 4: the CPU
    figure states what it includes)."""
    from oracle import vae_oracle as vo

    torch.set_num_threads(threads)
    cfg = vo.VaeConfig()
    sd = vo.make_synthetic_state_dict(cfg, seed=1, dtype=torch.float32)
    g = torch.Generator().manual_seed(3)
    img = torch.rand(1, 3, height, width, generator=g) * 2 - 1
    with torch.no_grad():
        t0 = time.perf_counter()
        z = vo.encode_mode(sd, cfg, img)
        t_e = time.perf_counter() - t0
        t0 = time.perf_counter()
        vo.decode(sd, cfg, z)
        t_d = time.perf_counter() - t0
    return {"vae_encode_s": t_e, "vae_decode_s": t_d}


def cpu_config1_seconds(threads: int) -> dict:
    """BASELINE.json configs[0] / BASELINE.md section 4(i): one 256x256 edit, 4 Euler steps, fp32, host cores, through
    the oracle's pipeline loop with the full 19 + 38 block depth.  To bound host memory the 57 blocks share the weights of
    one double and one single block (same shapes, same FLOPs: 47.6 GB of distinct fp32 weights would not change the
    arithmetic cost); VAE encode/decode included, conditioning supplied as embeddings."""
    from oracle import flux_oracle as fo

    torch.set_num_threads(threads)
    cfg1 = fo.FluxConfig(num_layers=1, num_single_layers=1)
    sd = fo.make_synthetic_state_dict(cfg1, seed=0, dtype=torch.float32)
    S_img = 2 * 16 * 16
    g = torch.Generator().manual_seed(0)
    lat = torch.randn(1, S_img // 2, 64, generator=g)
    ctx = torch.randn(1, S_img // 2, 64, generator=g)
    enc = torch.randn(1, S_TXT, 4096, generator=g)
    pooled = torch.randn(1, 768, generator=g)
    ids = torch.zeros(S_TXT + S_img, 3)
    cos, sin = fo.rope_tables(ids)
    sig = np.linspace(1.0, 0.0, 5)
    t0 = time.perf_counter()
    with torch.no_grad():
        for i in range(4):
            hs = torch.cat([lat, ctx], 1)
            x = fo._lin(sd, "x_embedder", hs)
            c = fo._lin(sd, "context_embedder", enc)
            temb = fo.time_text_embed(sd, cfg1, torch.full((1,), float(sig[i]) * 1000), torch.full((1,), 3500.0), pooled)
            for _ in range(N_DOUBLE):
                c, x = fo.double_block(sd, 0, cfg1, x, c, temb, cos, sin)
            h = torch.cat([c, x], 1)
            for _ in range(N_SINGLE):
                h = fo.single_block(sd, 0, cfg1, h, temb, cos, sin)
            x = h[:, S_TXT:]
            e = fo._lin(sd, "norm_out.linear", torch.nn.functional.silu(temb))
            sc, sh = torch.chunk(e, 2, dim=1)
            v = fo._lin(sd, "proj_out", fo.layer_norm(x) * (1 + sc)[:, None] + sh[:, None])[:, :S_img // 2]
            lat = lat + float(sig[i + 1] - sig[i]) * v
    t_loop = time.perf_counter() - t0
    vae = cpu_vae_seconds(256, 256, threads)
    total = t_loop + vae["vae_encode_s"] + vae["vae_decode_s"]
    return {"config": "single 256x256 edit, 4 Euler steps, fp32 CPU (BASELINE.json configs[0])", "seconds_per_edit": total,
            "denoise_loop_s": t_loop, **vae, "threads": threads, "cores": os.cpu_count() or 1,
            "note": "oracle restatement; 57 blocks at full width sharing one double + one single block's weights (memory bound of "
                    "the host), S = 544 + 512; Qwen2.5-VL / T5 / CLIP conditioning supplied as embeddings"}


def reference_config(args):
    """`config` of the CPU arm: the same workload as the GPU arm, described for what THIS arm runs."""
    S_img = 2 * (args.height // 16) * (args.width // 16)
    return {"workload": f"C{args.height}: FLUX.1-Kontext-dev MMDiT 19+38 blocks d=3072, {args.height}x{args.width}, "
                        f"{args.num_inference_steps} Euler steps, S_txt={S_TXT}, S_img={S_img}, guidance 3.5",
            "batch_per_gpu": 1, "global_batch": 1,
            "parallelism": "host threads of one process (torch intra-op), no GPU",
            "implementation": "oracle/flux_oracle.py: fp32 PyTorch restatement of the reference's diffusers path (the reference "
                              "itself cannot be installed offline, DESIGN.md section 3)",
            "timed": "one double-stream + one single-stream block at the full shapes per step of this arm, extrapolated to 19 / 38 "
                     "blocks and 28 Euler steps",
            "conditioning": "EXCLUDED from this arm (Qwen2.5-VL prefill, MLP2, T5-XXL, CLIP-L); the GPU arm includes them",
            "vae": "EXCLUDED from `value`; measured once, see cpu_baseline.vae (the GPU arm includes encode + decode)"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    times = []
    last = None
    warm = min(args.warmup, 1)          # a CPU pass of ~40 s does not need three warm-ups
    for i in range(warm + args.steps):
        last = cpu_reference_sample(args.height, args.width, args.num_inference_steps)
        if i >= warm:
            times.append(last["sec_per_image_extrapolated"])
    sec = float(np.mean(times))
    val = 1.0 / sec
    cb = {k: last[k] for k in ("unit", "cores", "threads", "kind", "sample", "excluded")}
    cb["value"] = val
    if args.cpu_extras:
        cb["vae"] = cpu_vae_seconds(args.height, args.width, last["threads"])
        cb["sec_per_image_with_vae"] = sec + cb["vae"]["vae_encode_s"] + cb["vae"]["vae_decode_s"]
        cb["config1"] = cpu_config1_seconds(last["threads"])
    print(json.dumps({
        "impl": "reference", "metric": "edited images/sec @1024px 28-step", "value": val, "unit": "images/s",
        "n_gpus": args.gpus, "steps": len(times), "warmup": warm, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": reference_config(args), "cpu_baseline": cb,
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def workload_config(args, world):
    S_img = 2 * (args.height // 16) * (args.width // 16)
    return {"workload": f"C{args.height}: FLUX.1-Kontext-dev MMDiT 19+38 blocks d=3072, {args.height}x{args.width}, "
                        f"{args.num_inference_steps} Euler steps, S_txt={S_TXT}, S_img={S_img}, guidance 3.5",
            "batch_per_gpu": args.batch_per_gpu, "global_batch": args.batch_per_gpu * world,
            "parallelism": f"batch-sharded replicas x{world} (weights broadcast once over NCCL)",
            "l2": "inputs larger than L2 (23.8 GB of weights stream every forward)",
            "conditioning": ("synthetic prompt_embeds (no encoders in the timed region)" if getattr(args, "no_conditioning", False) else
                             "inside the timed region, all on libb2f kernels: Qwen2.5-VL-7B prefill (ViT 448x448 + 28-layer decoder, "
                             "L=288) + MLP2, T5-XXL encoder (256 tokens), CLIP-L text encoder (77 tokens)")}


# ---------------------------------------------------------------------------------------------- training arm
def run_train_arm(args):
    """BASELINE.json configs[3]: `train_denoiser.py` stage-2 at 512x512, bf16, ZeRO-2 over the ranks, synthetic
    (src, instr, tgt) triples.  One "step" = one optimizer step (batch_per_gpu samples per rank): VAE-encode target and
    context, frozen Qwen2.5-VL-7B prefill, MLP2, FLUX forward with block checkpoints, loss, backward with per-block
    recompute, gradient reduce-scatter, clipping, AdamW, bf16 all-gather — all inside the timed region."""
    import torch.distributed as dist

    import train_denoiser as td
    from gpt_image_edit_b200 import _lib
    from gpt_image_edit_b200 import distributed as D
    from gpt_image_edit_b200.training import Stage2Trainer
    from univa.training.configuration_denoise import load_config
    from univa.training.synthetic_data import SyntheticEditDataset, collate

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("NCCL_DEBUG_FILE", os.path.join(os.environ.get("TMPDIR", "/tmp"), "nccl_debug.%h.%p.log"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    D.init_from_env("nccl", dev)
    conf = load_config(ROOT / "scripts" / "denoiser" / "flux_qwen2p5vl_7b_vlm_stage2_512_synthetic.yaml")
    conf.dataset_config.batch_size = args.batch_per_gpu
    if args.layers:      # debug only
        conf.model_config.small = True
    H = W = 512
    model, vae, pipe, empty = td.build_models(conf, dev)
    D.broadcast_weights(list(model.denoise_tower.denoiser._store.values()) +
                        list(model.denoise_tower.denoise_projector.state_dict().values()))
    trainer = Stage2Trainer(model, vae, pipe, conf.training_config, conf.model_config, empty)
    trainer.gen = torch.Generator(device=dev).manual_seed(conf.training_config.seed + rank)
    data = SyntheticEditDataset(H, W, seed=conf.training_config.seed + rank)
    B = args.batch_per_gpu
    n_distinct = 4
    host = []
    for i in range(n_distinct):
        b = collate([data[i * B + j] for j in range(B)])
        host.append({k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in b.items()})
    on_dev = [{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in b.items()} for b in host]
    h2d = sum(v.numel() * v.element_size() for v in host[0].values() if torch.is_tensor(v))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n, from_host):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        s.record()
        loss = None
        for i in range(n):
            b = host[i % n_distinct] if from_host else on_dev[i % n_distinct]
            if from_host:
                b = {k: (v.to(dev, non_blocking=True) if torch.is_tensor(v) else v) for k, v in b.items()}
            out = trainer.step(b)
            if from_host:
                loss = out["loss"].item()            # the step's result read back to the host
        e.record()
        torch.cuda.synchronize()
        ms = s.elapsed_time(e)
        if from_host:
            ms = max(ms, (time.perf_counter() - t0) * 1e3)
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), loss

    for i in range(args.warmup):
        trainer.step(on_dev[i % n_distinct])
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    _lib.prof_enable(True)
    n0 = _lib.launch_count()
    ms_total, _ = timed(args.steps, False)
    launches = _lib.launch_count() - n0
    prof = _lib.prof_collect()
    _lib.prof_enable(False)
    clocks = sampler.stop() if rank == 0 else None
    ms_e2e, last_loss = timed(args.steps, True)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    ms_step = ms_total / args.steps
    value = world * B / (ms_step / 1e3)
    dom = max(("gemm", "attention"), key=lambda k: prof[k]["ms"])
    pd = prof[dom]
    achieved = pd["flops"] / (pd["ms"] / 1e3) / 1e12 if pd["ms"] > 0 else 0.0
    total_flops = sum(v["flops"] for v in prof.values()) / args.steps
    n_train = sum(p.storage.numel() for p in trainer.params)
    line = {
        "metric": "stage-2 training samples/sec @512px (train_denoiser.py, ZeRO-2)", "value": value, "unit": "samples/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "train512: train_denoiser.py stage-2, 512x512 target + 512x512 context, S = 288 + 1024 + 1024, "
                               "Qwen2.5-VL-7B (frozen) + MLP2 + FLUX.1-Kontext-dev 19+38 blocks, recompute per block",
                   "batch_per_gpu": B, "global_batch": B * world, "trainable_parameters": n_train,
                   "parallelism": f"ZeRO-2 x{world}: fp32 gradient reduce-scatter per block overlapped with the backward, "
                                  "fp32 master weights + Adam moments partitioned, bf16 all-gather",
                   "l2": "inputs larger than L2 (weights stream every forward and backward)",
                   "optimizer": "AdamW, clip 1.0, lr 1e-6 (scripts/denoiser/flux_qwen2p5vl_7b_vlm_stage2_512_synthetic.yaml)"},
        "model_tflops_per_gpu": total_flops / (ms_step / 1e3) / 1e12,
        "model_frac_of_sustained_peak": total_flops / (ms_step / 1e3) / 1e12 / pk["tensor_sustained"],
        "e2e": {"value": world * B / (ms_e2e / args.steps / 1e3), "unit": "samples/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": 4, "last_loss": last_loss},
        "gpu_launches": int(launches), "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": dom, "achieved": achieved, "peak": pk["tensor_sustained"], "unit": "TFLOP/s",
                     "frac": achieved / pk["tensor_sustained"], "peak_source": pk["source"] + ", sustained figure",
                     "launches": pd["launches"], "share_of_step": pd["ms"] / ms_total, "traffic": None,
                     "classes": {k: {"ms": round(v["ms"], 3), "launches": v["launches"],
                                     "tflops": (v["flops"] / (v["ms"] / 1e3) / 1e12) if v["ms"] > 0 and v["flops"] > 0 else None,
                                     "gbps": (v["bytes"] / (v["ms"] / 1e3) / 1e9) if v["ms"] > 0 and v["flops"] == 0 else None}
                                 for k, v in prof.items() if v["launches"]}},
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch-per-gpu", type=int, default=1)
    ap.add_argument("--height", type=int, default=1024)
    ap.add_argument("--width", type=int, default=1024)
    ap.add_argument("--num-inference-steps", type=int, default=28)
    ap.add_argument("--layers", type=str, default=None, help="debug: 'D,S' block counts (invalidates the number)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-extras", action="store_true", help="reference arm: also time, once, the oracle VAE at this size and "
                    "BASELINE.json configs[0] (256x256, 4 steps, fp32) on the host cores (several minutes; recorded in "
                    "profiles/r02_cpu_reference_extras.json)")
    ap.add_argument("--sweep", default="", help="comma list of SIZE[xBATCH] configurations measured in one process, e.g. "
                    "512,768,1024,1024x4 (BASELINE.json configs[2] and [4]); prints one JSON line per configuration")
    ap.add_argument("--workload", default="edit", choices=["edit", "train512"], help="edit: the headline metric; train512: "
                    "BASELINE.json configs[3], stage-2 training samples/s at 512x512 (ZeRO-2 over the ranks)")
    ap.add_argument("--no-conditioning", action="store_true", help="feed synthetic prompt_embeds instead of running the "
                    "Qwen2.5-VL prefill + MLP2 inside the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="after the timed steps, write what the last timed "
                    "edit returned (the images; the latents without a VAE) as DIR/images.npy in float32, DIR/images_rank<R>.npy "
                    "per rank with N>1; the inputs are seeded, so two builds run with the same arguments compare output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "edit" or args.sweep):
        ap.error("--dump-outputs applies to the edit workload of the b200 implementation, without --sweep")

    if args.impl == "reference":
        return run_reference_arm(args)
    if args.workload == "train512":
        return run_train_arm(args)

    import torch.distributed as dist

    from gpt_image_edit_b200 import _lib
    from gpt_image_edit_b200 import distributed as D
    from gpt_image_edit_b200.flux_transformer import B200FluxTransformer2DModel, FluxTransformerConfig
    from gpt_image_edit_b200.pipeline import FluxKontextPipeline
    from gpt_image_edit_b200.scheduler import FlowMatchEulerDiscreteScheduler

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # keep stdout to the one JSON line: NCCL writes its version banner / debug lines to stdout unless given a file
    os.environ.setdefault("NCCL_DEBUG_FILE", os.path.join(os.environ.get("TMPDIR", "/tmp"), "nccl_debug.%h.%p.log"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    D.init_from_env("nccl", dev)

    nd, ns = (N_DOUBLE, N_SINGLE) if not args.layers else map(int, args.layers.split(","))
    model = B200FluxTransformer2DModel(FluxTransformerConfig(num_layers=nd, num_single_layers=ns), device=dev)
    # rank 0 draws the synthetic weights (N(0, 0.02^2), SURVEY.md §8d), everyone else receives them
    if rank == 0:
        model.randomize_(seed=0)
    D.broadcast_weights(model._store.values(), src=0)
    try:
        from gpt_image_edit_b200.vae import B200AutoencoderKL
        vae = B200AutoencoderKL(device=dev)
        if rank == 0:
            vae.randomize_(seed=1)
        D.broadcast_weights(vae.storage(), src=0)
    except ImportError:
        vae = None
    pipe = FluxKontextPipeline(transformer=model, vae=vae, scheduler=FlowMatchEulerDiscreteScheduler())

    # conditioning model (Qwen2.5-VL-7B prefill + MLP2) with synthetic weights: inside the timed region
    cond = None
    if not args.no_conditioning:
        from gpt_image_edit_b200.qwen2p5vl import B200Qwen2p5VL
        from univa.models.modeling_univa_denoise_tower import DenoiseProjector
        from univa.serve.cli import synthetic_chat_tokens

        qwen = B200Qwen2p5VL(device=dev)
        mlp2 = DenoiseProjector(3584, 4096, device=dev)
        if rank == 0:
            qwen.randomize_(seed=10)
            gq = torch.Generator(device=dev).manual_seed(11)
            for t in mlp2.state_dict().values():
                t.copy_((torch.randn(t.shape, device=dev, generator=gq) * 0.02).to(torch.bfloat16))
        D.broadcast_weights(qwen.storage(), src=0)
        D.broadcast_weights(list(mlp2.state_dict().values()), src=0)
        # T5-XXL + CLIP-L prompt encoders (row a11), also inside the timed region
        from gpt_image_edit_b200.text_encoders import B200CLIPTextModel, B200T5Encoder, SyntheticTokenizer
        t5, clip = B200T5Encoder(device=dev), B200CLIPTextModel(device=dev)
        if rank == 0:
            t5.randomize_(seed=21)
            clip.randomize_(seed=20)
        D.broadcast_weights(t5.storage(), src=0)
        D.broadcast_weights(clip.storage(), src=0)
        prompt = "replace the red car with a blue bicycle and keep the background unchanged"
        t5_ids = SyntheticTokenizer.t5()(prompt, max_length=256).input_ids          # padded to 256 as cli.py:225
        clip_ids = SyntheticTokenizer.clip()(prompt, max_length=77).input_ids
        # L_qwen = 4 + 256 + 1 + 22 + 5 = 288 tokens (SURVEY.md §8d), + 256 T5 tokens = S_txt 544
        cond = (qwen, mlp2, synthetic_chat_tokens(256, n_text=22), t5, clip, t5_ids, clip_ids)

    def run_config(args):
        B, H, W = args.batch_per_gpu, args.height, args.width
        S_img = 2 * (H // 16) * (W // 16)
        g = torch.Generator().manual_seed(1 + rank)
        src = torch.randint(0, 256, (B, H, W, 3), generator=g, dtype=torch.uint8).pin_memory()   # uint8 pixels, PIL / numpy layout:
        # the (u/255 - 0.5)/0.5 normalisation of cli.py:99-116 runs inside the VAE's first kernel
        g2 = torch.Generator().manual_seed(2 + rank)
        if cond is not None and cond[2].shape[1] + 256 != S_TXT:
            raise SystemExit(f"conditioning layout gives S_txt = {cond[2].shape[1] + 256}, expected {S_TXT}")
        pe_h = torch.randn(B, S_TXT, 4096, generator=g2).bfloat16().pin_memory()   # only used with --no-conditioning
        t5_ids_h = (cond[5].repeat(B, 1) if cond is not None else torch.zeros(B, 1, dtype=torch.long)).pin_memory()
        clip_ids_h = (cond[6].repeat(B, 1) if cond is not None else torch.zeros(B, 1, dtype=torch.long)).pin_memory()
        pix_h = torch.randn(B * 1024, 1176, generator=g2).bfloat16().pin_memory()      # 448x448 -> 1024 patches per image
        ids_h = (cond[2].repeat(B, 1) if cond is not None else torch.zeros(B, 1, dtype=torch.long)).pin_memory()
        pp_h = torch.randn(B, 768, generator=g2).bfloat16().pin_memory()
        noise_h = torch.stack([torch.randn(S_img // 2, 64, generator=torch.Generator().manual_seed(42 + rank * B + i))
                               for i in range(B)]).bfloat16().pin_memory()
        ctx_lat_h = torch.randn(B, 16, H // 8, W // 8, generator=g2).bfloat16().pin_memory()  # only used without a VAE

        def one_edit(from_host: bool):
            nb = lambda t: t.to(dev, non_blocking=True)
            if from_host:
                noise = nb(noise_h)
                image = nb(src) if vae is not None else nb(ctx_lat_h)
                if cond is not None:
                    pix, ids, t5_ids, clip_ids = nb(pix_h), nb(ids_h), nb(t5_ids_h), nb(clip_ids_h)
                else:
                    pe, pp = nb(pe_h), nb(pp_h)
            else:
                noise = dev_in["noise"].clone()
                image = dev_in["image"]
                pe, pp = dev_in["pe"], dev_in["pp"]
                pix, ids, t5_ids, clip_ids = dev_in["pix"], dev_in["ids"], dev_in["t5_ids"], dev_in["clip_ids"]
            if cond is not None:
                # VLM prefill (ViT + 28-layer decoder) -> MLP2 -> [B, L, 4096]; T5-XXL hidden states and the CLIP-L pooled
                # vector from the libb2f encoders; joined as cli.py:210-234 does
                hidden = cond[0](ids, pixel_values=pix, image_grid_thw=[(1, 32, 32)] * B)
                pe = torch.cat([cond[1](hidden), cond[3](t5_ids)[0]], dim=1)
                pp = cond[4](clip_ids, output_hidden_states=False).pooler_output
            out = pipe(image=image, prompt_embeds=pe, pooled_prompt_embeds=pp, height=H, width=W,
                       num_inference_steps=args.num_inference_steps, guidance_scale=3.5, latents=noise,
                       max_area=H * W, _auto_resize=False, output_type="u8" if vae is not None else "latent").images
            if from_host:
                return out.to("cpu", non_blocking=False)      # uint8 [B,H,W,3] pixels (postprocess fused into decoder.conv_out)
            return out

        dev_in = dict(pe=pe_h.to(dev), pp=pp_h.to(dev), noise=noise_h.to(dev),
                      image=(src if vae is not None else ctx_lat_h).to(dev), pix=pix_h.to(dev), ids=ids_h.to(dev),
                      t5_ids=t5_ids_h.to(dev), clip_ids=clip_ids_h.to(dev))

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        def timed(n, from_host):
            barrier()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            s.record()
            for _ in range(n):
                out = one_edit(from_host)
            e.record()
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            ms = s.elapsed_time(e)
            if from_host:
                ms = max(ms, wall * 1e3)  # the D2H read ends on the host
            t = torch.tensor([ms], device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item()), out

        for _ in range(args.warmup):
            one_edit(False)
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        _lib.prof_enable(True)
        n0 = _lib.launch_count()
        ms_total, last = timed(args.steps, False)
        launches = _lib.launch_count() - n0
        shapes = _lib.prof_shapes()
        prof = _lib.prof_collect()
        _lib.prof_enable(False)
        clocks = sampler.stop() if rank == 0 else None
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"images" if world == 1 else f"images_rank{rank}": last.float().cpu().numpy()})
        one_edit(True)
        ms_e2e, _ = timed(args.steps, True)

        if rank != 0:
            return None
        pk = peaks()
        ms_per_edit = ms_total / args.steps
        value = world * B / (ms_per_edit / 1e3)
        e2e = world * B / (ms_e2e / args.steps / 1e3)
        f_fwd = flops_per_forward(S_img, S_TXT, nd, ns) * B
        f_edit = f_fwd * args.num_inference_steps
        gm = prof["gemm"]
        dom = max(("gemm", "attention"), key=lambda k: prof[k]["ms"])
        pd = prof[dom]
        achieved = pd["flops"] / (pd["ms"] / 1e3) / 1e12 if pd["ms"] > 0 else 0.0
        roof = {"bound": "tensor", "kernel": {"gemm": "gemm_bf16_kernel (tcgen05)", "attention": "attn_fwd_kernel (tcgen05)"}[dom],
                "achieved": achieved, "peak": pk["tensor_sustained"], "unit": "TFLOP/s", "frac": achieved / pk["tensor_sustained"],
                "frac_of_burst_peak": achieved / pk["tensor_burst"], "peak_source": pk["source"] + ", sustained figure (kernel timed inside a long step)",
                "avg_launch_ms": pd["ms"] / max(pd["launches"], 1), "launches": pd["launches"],
                "algorithmic_tflop_per_launch": pd["flops"] / max(pd["launches"], 1) / 1e12, "traffic": ncu_traffic(dom),
                "share_of_step": pd["ms"] / ms_total,
                "classes": {k: {"ms": round(v["ms"], 3), "launches": v["launches"],
                                "tflops": (v["flops"] / (v["ms"] / 1e3) / 1e12) if v["ms"] > 0 and v["flops"] > 0 else None,
                                "gbps": (v["bytes"] / (v["ms"] / 1e3) / 1e9) if v["ms"] > 0 and v["flops"] == 0 else None}
                            for k, v in prof.items() if v["launches"]}}
        line = {
            "metric": "edited images/sec @1024px 28-step", "value": value, "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_edit, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": dict(workload_config(args, world), vae="hand-written (included)" if vae is not None else
                           "EXCLUDED (context latents supplied, latent output)"),
            "ms_per_denoise_step": ms_per_edit / args.num_inference_steps,
            "model_tflops_per_gpu": f_edit / (ms_per_edit / 1e3) / 1e12,
            "model_frac_of_sustained_peak": f_edit / (ms_per_edit / 1e3) / 1e12 / pk["tensor_sustained"],
            "e2e": {"value": e2e, "unit": "images/s",
                    "h2d_bytes_per_step": int(sum(t.numel() * t.element_size() for t in
                                                  (noise_h, src if vae is not None else ctx_lat_h) +
                                                  ((pix_h, ids_h, t5_ids_h, clip_ids_h) if cond is not None else (pe_h, pp_h)))),
                    "d2h_bytes_per_step": int(B * 3 * H * W if vae is not None else noise_h.numel() * 2)},
            "gpu_launches": int(launches), "roofline": roof, "clocks": clocks,
        }
        # in-loop GEMM efficiency per shape (the ten largest time sinks)
        roof["gemm_shapes"] = [{"shape": t, "launches": n, "ms": round(ms, 2), "tflops": round(tf, 1)}
                               for t, n, ms, tf in sorted(shapes, key=lambda r: -r[2])[:14]]
        if world == 1 and not args.no_cpu_baseline:
            cb = cpu_reference_sample(H, W, args.num_inference_steps)
            cb.pop("sec_per_image_extrapolated", None)
            line["cpu_baseline"] = cb
        return line

    if args.sweep:
        # BASELINE.json configs[2] / [4] in ONE process per N (models built once): the resolution sweep at batch 1 per GPU and
        # the 1024^2 run at batch 4 per GPU (global batch 32 at N = 8); one JSON object per configuration
        import copy
        for spec in args.sweep.split(","):
            hw, _, b = spec.partition("x")
            a2 = copy.copy(args)
            a2.height = a2.width = int(hw)
            a2.batch_per_gpu = int(b or 1)
            a2.no_cpu_baseline = True
            line = run_config(a2)
            if rank == 0:
                line["sweep"] = spec
                print(json.dumps(line), flush=True)
    else:
        line = run_config(args)
        if rank == 0:
            print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
