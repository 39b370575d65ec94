#!/usr/bin/env python
"""bench.py — headline benchmark of the Selftok hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU arithmetic on the host cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's tokens and latents to DIR/*.npy

One "step" = one pass of the hot path over one batch: encode (16-block Q-Former + fused VQ -> 512 tokens) followed by
the 50-step rectified-flow decode of those tokens (24-layer MMDiT), 256x256 images, no VAE (latent boundary; SURVEY 8f).
Workload at N = 1: BASELINE.json configs[2], batch 64.  N > 1: the same batch per GPU (weak scaling), weights
replicated, one NCCL all-gather of the token ids per step (SURVEY 8e).  Synthetic latents and a seeded synthetic
checkpoint of the real architecture (no weights are obtainable offline).

Printed JSON (rank 0, one line): metric/value/unit/... per the driver contract, plus
  e2e          the same metric through the host-buffer C-ABI entry points (pinned host -> device copies of latents,
               tokens and noise and the device -> host reads of tokens and latents inside the timed region)
  roofline     tcgen05 GEMM class (dominant kernel): algorithmic FLOPs / summed CUDA-event time of its launches in one
               profiled step, against MEASURED_PEAKS.json's sustained bf16 GEMM rate
  cpu_baseline oracle port of the reference arithmetic (torch fp32 on the host cores) on a bounded sample
  extra        (N = 1 only) sub-records for the other BASELINE configs, each measured in this run:
                 config2_encode_only   batch-64 encode img/s + the fused VQ kernel alone (ms, algorithmic GB/s vs HBM peak,
                                       fp32 TFLOP/s vs the FFMA peak -- the pipe that actually bounds it)
                 config3_bf16x3        the headline workload in the fp32-faithful split-bf16 mode
                 config4_renderer_512 / _1024   batch-64 encode + ONE renderer pass (img/s), 512 and 1024 tokens
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

import torch  # noqa: E402

from selftoktokenizer_b200 import config as C  # noqa: E402
from selftoktokenizer_b200 import schedule as S  # noqa: E402
from selftoktokenizer_b200 import synth  # noqa: E402

METRIC = "images/sec encode+50-step decode, 256x256/512-tok"
UNIT = "images/s"
BATCH = 64
DECODE_STEPS = 50
DUMP_BYTES = 64 << 20


def peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops=float(d["bf16_tflops_sustained"]), tflops_burst=float(d["bf16_tflops"]),
                    hbm=float(d["hbm_gbs"]), source="measured (MEASURED_PEAKS.json, sustained bf16 cuBLAS)")
    return dict(tflops=1400.0, tflops_burst=1590.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


def other_class_rooflines(prof, B, precision, pk):
    """BASELINE's '% of roofline per kernel class' for the classes that are not the dominant one: algorithmic work of the profiled
    encode + 50-step decode divided by the class's event-timed total (same pass as `roofline`)."""
    d = C.FULL
    tb = S.make_tables(d.K, d.stages, d.k_per_stage, DECODE_STEPS)
    D, N, L = d.dit_hidden, d.n_img, d.dit_depth
    attn_flops = ln_bytes = 0.0
    plane = 4 if precision == "bf16x3" else 2                       # 16-bit hi (+ lo) operand planes written per element
    for i in range(DECODE_STEPS):
        kc = int(tb.k[i]) + 1
        Sj = kc + N
        attn_flops += L * 4.0 * Sj * Sj * D * B                      # Q K^T + P V over the joint sequence, every row sees every key
        ln_bytes += (2 * L * N + (2 * L - 1) * kc + N) * B * D * (4 + plane)   # x fp32 in, planes out; last ctx block pre_only; final LN
    out = {}
    if "attention" in prof and prof["attention"][0] > 0:
        ach = attn_flops / (prof["attention"][0] / 1000.0) / 1e12
        out["attention"] = {"bound": "tensor", "achieved": ach, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": ach / pk["tflops"],
                            "note": "head dim 64: latency-chain bound, see profiles/r2_attention_investigation.md"}
    if "ln_modulate" in prof and prof["ln_modulate"][0] > 0:
        ach = ln_bytes / (prof["ln_modulate"][0] / 1000.0) / 1e9
        out["ln_modulate"] = {"bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"],
                              "note": "fp32 residual stream in, 16-bit operand planes out; the adaLN tables are L2-resident"}
    if "linear_f32" in prof and prof["linear_f32"][0] > 0:
        enc_flops = 65.6e9 * B                                       # DESIGN.md section 4: encoder GEMMs per image
        ach = enc_flops / (prof["linear_f32"][0] / 1000.0) / 1e12
        peak = 148 * 128 * 2 * 1.965e9 / 1e12
        out["linear_f32"] = {"bound": "fp32 FFMA", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                             "note": "Q-Former encoder, fp32 for bit-exact ids; peak = 148 SMs x 128 lanes x 2 x 1.965 GHz (nominal)"}
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in self.rows if len(r) >= 7 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons}


def gemm_traffic():
    """DRAM bytes per tcgen05 GEMM launch: NOT measured by this run (ncu cannot run inside a timed bench) -- read from the
    committed extract of the round's `ncu --set full` capture of one MMDiT layer (profiles/extract_ncu.py)."""
    for name in ("r2_gemm_traffic.json", "r1_gemm_traffic.json"):
        p = os.path.join(REPO, "profiles", name)
        if os.path.exists(p):
            d = json.load(open(p))
            return {"bytes_per_launch": float(d["bytes_per_launch"]), "source": f"profiles/{name}: " + d["source"]}
    return {"bytes_per_launch": None, "source": "no committed ncu extract"}


def gemm_flops_per_step(B: int) -> float:
    """Algorithmic (single-product, masked-effective) FLOPs of the tcgen05 GEMM launches of one 50-step decode:
    per layer and stream qkv 2*M*D*3D, proj 2*M*D*D, fc1+fc2 16*M*D*D; the last layer's context stream is qkv only."""
    d = C.FULL
    tb = S.make_tables(d.K, d.stages, d.k_per_stage, DECODE_STEPS)
    D, N, L = d.dit_hidden, d.n_img, d.dit_depth
    f = 0.0
    for i in range(DECODE_STEPS):
        kc = int(tb.k[i]) + 1
        for j in range(L):
            f += B * N * (6 * D * D + 2 * D * D + 16 * D * D)
            f += B * kc * (6 * D * D + (0 if j == L - 1 else 2 * D * D + 16 * D * D))
    return f


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_sample(n_threads=None, batches=(1,)):
    """Bounded sample of the reference arithmetic on the host: full-geometry encode + the first decode step (k = 511, all
    tokens visible), including the reference's per-step dead encoder+VQ call (rectified_flow.py:212-215), at batch sizes
    `batches`.  Extrapolated to 50 steps with the per-step FLOP model (SURVEY 8d).  Returns (one(B) -> (t_enc, t_step), scale).

    "All the host threads it can use": torch's CPU GEMMs stop scaling (and regress) well below the core count of a 100+-core
    host, so the thread count is calibrated ON THE DECODE STEP (98 % of the CPU time) and the fastest setting is used; a B = 1
    step is M-starved (768 GEMM rows), which is why B = 4 is timed next to it."""
    sys.path.insert(0, os.path.join(REPO, "oracle"))
    import selftok_oracle as O
    d = C.FULL
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    sd = {k: v.cpu() for k, v in synth.synth_state_dict(d, device=dev).items()}
    tb = S.make_tables(d.K, d.stages, d.k_per_stage, DECODE_STEPS)
    Bmax = max(batches)
    x0 = synth.synth_tensor("bench.cpu.x0", (Bmax, d.in_channels, d.latent, d.latent), "emb", 1.0)
    noise = synth.synth_tensor("bench.cpu.noise", (Bmax, d.in_channels, d.latent, d.latent), "emb", 1.0)
    state = {}

    def one(B=1):
        t0 = time.perf_counter()
        with torch.no_grad():
            outs_q, tok, _ = O.encode(sd, d, x0[:B], tb)
            t1 = time.perf_counter()
            O.decode(sd, d, tok, noise[:B], steps=DECODE_STEPS, tables=tb, n_steps_run=1, replay_dead_encoder_call=True)
        t2 = time.perf_counter()
        state["tok"] = tok
        return t1 - t0, t2 - t1

    cores = n_threads or os.cpu_count() or 1
    with torch.no_grad():
        one(1)                                        # first-call overheads (thread pool, primitive caches) excluded
        best_n, best_t = None, None
        for n in sorted({min(cores, c) for c in (8, 16, 32, 64, cores)}):
            torch.set_num_threads(n)
            t = one(1)[1]
            if best_t is None or t < best_t:
                best_n, best_t = n, t
        torch.set_num_threads(best_n)

    D, N, L = d.dit_hidden, d.n_img, d.dit_depth
    eff = []
    for i in range(DECODE_STEPS):       # the reference computes the DENSE K+N sequence every step (masked, not dropped)
        eff.append(sum(S.dense_flops_per_image_step(D, d.K, N, j == L - 1) for j in range(L)))
    scale = sum(eff) / eff[0]
    return one, scale


def cpu_record(one, scale, batches=(1, 4)):
    best, parts = None, []
    for B in batches:
        t_enc, t_step = one(B)
        v = B / (t_enc + t_step * scale)
        parts.append(f"B={B}: encode {t_enc:.2f}s + decode step 0 incl. the reference's dead encoder call {t_step:.2f}s -> {v:.4f} img/s")
        if best is None or v > best:
            best = v
    sample = ("full-geometry encode + first decode step, x%.1f (dense per-step FLOP model) for 50 steps, extrapolated; thread count "
              "calibrated on the decode step; " % scale) + "; ".join(parts)
    return {"value": best, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port", "sample": sample}


def run_reference(args):
    """--impl reference: the reference's own arithmetic (oracle port, torch fp32 CPU) on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    one, scale = cpu_sample(cores, batches=(1, 4))
    for _ in range(args.warmup):
        one(1)
    t0 = time.perf_counter()
    rec = None
    for _ in range(args.steps):
        r = cpu_record(one, scale, batches=(1, 4))
        if rec is None or r["value"] > rec["value"]:
            rec = r
    wall = time.perf_counter() - t0
    img_s = rec["value"]
    line = {"impl": "reference", "metric": METRIC, "value": img_s, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * wall / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "256x256 encode + 50-step decode, 512 tokens (bounded sample per step: B=1 and B=4, best of the two)",
                       "batch_per_gpu": 1},
            "cpu_baseline": rec,
            "e2e": {"value": img_s, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
def dump_outputs(path, outputs):
    """Write what a caller of the timed step receives (token ids [B, K], latents [B, 16, 32, 32]) as DIR/<name>.npy: ids as
    float64 (exact), latents as float32.  Above DUMP_BYTES in all, a fixed seeded sample of images is written instead, so two
    builds run with the same arguments can be compared file for file."""
    import numpy as np
    arrays = {"tokens": outputs["tokens"].cpu().double().numpy(), "latents": outputs["latents"].cpu().float().numpy()}
    B = arrays["tokens"].shape[0]
    per_image = sum(a[0].nbytes for a in arrays.values())
    if per_image * B > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(B, DUMP_BYTES // per_image, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def run_extras(args, eng, dev, x0, noise, timed):
    """Sub-records for BASELINE configs 2 and 4 and the fp32-faithful mode (see the module docstring).  `eng` is the
    headline engine (still alive); every other engine is created here and closed before the next one."""
    from selftoktokenizer_b200.capi import Engine
    import dataclasses
    d = C.FULL
    B = x0.shape[0]
    pk = peaks()
    out = {}
    # ---- config 2: encode only + the fused VQ kernel alone
    def enc_only():
        eng.encode(x0)
    enc_only()
    ms, _ = timed(enc_only, 5)
    tok, outs_q, feats = eng.encode(x0, return_aux=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ts = []
    for _ in range(13):
        flush.zero_()                                         # L2 flushed between iterations (256 MiB > 126 MB)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.vq_argmax(feats)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    vq_ms = sorted(ts[3:])[len(ts[3:]) // 2]
    R = B * d.K
    vq_bytes = R * d.enc_qdim * 4 + d.codebook_size * d.code_dim * 4 + d.code_dim * d.enc_qdim * 4 + R * 8 + R * d.code_dim * 4
    vq_flops = 2.0 * R * d.codebook_size * d.code_dim + 2.0 * R * d.enc_qdim * d.code_dim
    ffma_peak = 148 * 128 * 2 * 1.965e9 / 1e12
    out["config2_encode_only"] = {
        "workload": f"batch={B} 256x256 encode only (16-block Q-Former + fused VQ -> 512 tokens)", "value": B * 5 / (ms / 1000.0), "unit": UNIT,
        "ms_per_batch": ms / 5,
        "vq_kernel": {"ms": vq_ms, "algorithmic_bytes": vq_bytes, "achieved_GBps": vq_bytes / vq_ms / 1e6, "hbm_peak_GBps": pk["hbm"],
                      "frac_hbm": vq_bytes / vq_ms / 1e6 / pk["hbm"], "achieved_fp32_TFLOPs": vq_flops / vq_ms / 1e9,
                      "fp32_ffma_peak_TFLOPs_nominal": ffma_peak, "frac_ffma": vq_flops / vq_ms / 1e9 / ffma_peak,
                      "bound": "fp32 FFMA pipe (35.5 GFLOP on 71.6 MB: 11 us of HBM time); the HBM fraction is reported because the "
                               "north-star asks for it (SURVEY 8d)", "timing": "median of 10, CUDA events, L2 flushed"}}
    del flush
    # ---- serving view of the headline: ONE image through encode + 50-step decode (config 1's shape on the GPU)
    x1, n1 = x0[:1].contiguous(), noise[:1].contiguous()

    def one_image():
        eng.decode(eng.encode(x1), n1)
    one_image()
    ms1, _ = timed(one_image, 3)
    out["batch1_latency"] = {"workload": "batch=1 256x256 encode + 50-step decode (one CUDA-graph replay per call), device buffers",
                             "value": ms1 / 3, "unit": "ms", "higher_is_better": False, "images_per_s": 3000.0 / ms1}
    # ---- config 3 in the fp32-faithful mode
    if args.precision != "bf16x3":
        e3 = Engine(d, synth.synth_state_dict(d, device=dev), device=dev, precision="bf16x3", steps=DECODE_STEPS)

        def step3():
            t = e3.encode(x0)
            e3.decode(t, noise)
        step3()
        ms3, _ = timed(step3, 1)
        out["config3_bf16x3"] = {"workload": f"batch={B} encode + 50-step decode, split-bf16 (3 MMAs / product) GEMMs and attention",
                                 "value": B / (ms3 / 1000.0), "unit": UNIT, "ms_per_step": ms3}
        e3.close()
        del e3
        torch.cuda.empty_cache()
    # ---- config 4: encode + one renderer pass, 512 and 1024 tokens
    for K, kps in ((512, (512,)), (1024, (1024,))):
        dr = dataclasses.replace(d, K=K, stages=(1000,), k_per_stage=kps, renderer=True)
        er = Engine(dr, synth.synth_state_dict(dr, device=dev), device=dev, precision="auto")

        def step4():
            t = er.encode(x0)
            er.render(t)
        step4()
        ms4, _ = timed(step4, 3)
        flops = None
        try:
            D_, N_, L_ = dr.dit_hidden, dr.n_img, dr.dit_depth
            flops = sum(S.dense_flops_per_image_step(D_, K, N_, j == L_ - 1) for j in range(L_))
        except Exception:
            pass
        out[f"config4_renderer_{K}"] = {"workload": f"batch={B} 256x256 encode ({K} tokens) + ONE MMDiT_Renderer pass, no VAE",
                                        "value": B * 3 / (ms4 / 1000.0), "unit": UNIT, "ms_per_batch": ms4 / 3, "precision": er.precision,
                                        "renderer_dense_tflop_per_image": None if flops is None else flops / 1e12}
        er.close()
        del er
        torch.cuda.empty_cache()
    # ---- f1: the SD3 VAE decoder on the device (what follows the token path in decoding()): latents -> pixels, batch 64
    try:
        from selftoktokenizer_b200.capi import VaeDecoder
        dec = VaeDecoder(synth.synth_vae_state_dict(ch=128, device=dev), device=dev)
        z = noise * 0.5
        dec.decode(z)
        msv, _ = timed(lambda: dec.decode(z, norm_ip=True) is None, 3)
        out["vae_decode"] = {"workload": f"batch={B} SD3 VAE decoder, 32x32x16 latents -> 256x256 pixels (split-bf16 tcgen05 implicit-GEMM convs)",
                             "value": B * 3 / (msv / 1000.0), "unit": UNIT, "ms_per_batch": msv / 3, "algorithmic_tflop_per_batch": 0.622 * B}
        img = synth.synth_tensor("bench.images", (B, 3, 256, 256), "emb", 0.5, device=dev)
        dec.encode(img)
        mse, _ = timed(lambda: dec.encode(img) is None, 3)
        out["vae_encode"] = {"workload": f"batch={B} SD3 VAE encoder, 256x256 pixels -> 32x32x16 latent means (stride-2 convs as polyphase implicit GEMMs)",
                             "value": B * 3 / (mse / 1000.0), "unit": UNIT, "ms_per_batch": mse / 3, "algorithmic_tflop_per_batch": 0.273 * B}
        dec.close()
    except Exception as exc:  # noqa: BLE001 - the headline must not die on an auxiliary record
        out.setdefault("vae_decode", {"error": str(exc)[:200]})
        out.setdefault("vae_encode", {"error": str(exc)[:200]})
    # ---- the reference's own user call at the PIXEL boundary: SelftokPipeline.encoding(images) -> tokens -> .decoding(tokens)
    # -> images, host tensors in and out, both VAE halves + Q-Former + VQ + 50-step sampler on this library (BASELINE config 3)
    try:
        import contextlib
        from selftoktokenizer_b200 import SelftokPipeline
        from selftoktokenizer_b200.pipeline import DeviceVAE
        vae = DeviceVAE(synth.synth_vae_state_dict(ch=128, device=dev), dev)
        with contextlib.redirect_stdout(sys.stderr):                 # the class prints the reference's progress lines
            pipe = SelftokPipeline(cfg=None, ckpt_path=None, sd3_path=None, datasize=256, device=dev, state_dict=synth.synth_state_dict(d, device=dev),
                                   dims=d, vae=vae, precision=eng.precision)
        img_h = synth.synth_tensor("bench.images", (B, 3, 256, 256), "emb", 0.5).clamp_(-1, 1).pin_memory()
        res = {}

        def pixel_step():
            with contextlib.redirect_stdout(sys.stderr):
                tok = pipe.encoding(img_h, dev).cpu().numpy()          # H2D of the images inside, D2H of the ids
                res["img"] = pipe.decoding(tok, dev).cpu()             # host draw of the noise + H2D inside, D2H of the pixels
        pixel_step()
        msp, _ = timed(pixel_step, 2)
        out["pixel_e2e"] = {"workload": f"batch={B}: SelftokPipeline.encoding(images [B,3,256,256] on the host) -> ids on the host -> "
                                        "SelftokPipeline.decoding(ids) -> images on the host (VAE encoder + Q-Former + VQ + 50-step sampler + VAE "
                                        "decoder, pipeline dtype bf16 as the reference's default)",
                            "value": B * 2 / (msp / 1000.0), "unit": UNIT, "ms_per_batch": msp / 2,
                            "h2d_bytes_per_step": int(img_h.numel() * 4 + B * d.K * 8 + noise.numel() * 4),
                            "d2h_bytes_per_step": int(B * d.K * 8 + res["img"].numel() * res["img"].element_size()),
                            "precision": pipe.engine.precision}
        pipe.engine.close()
        vae.decoder.close()
    except Exception as exc:  # noqa: BLE001
        out["pixel_e2e"] = {"error": str(exc)[:300]}
    return out


def run_gpu(args):
    import torch.distributed as dist
    from selftoktokenizer_b200.capi import Engine
    from selftoktokenizer_b200.dist import gather_tokens
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    d = C.FULL
    B = args.batch
    sd = synth.synth_state_dict(d, device=dev)
    eng = Engine(d, sd, device=dev, precision=args.precision, steps=DECODE_STEPS)
    del sd
    torch.cuda.empty_cache()
    # ONE global draw (index-hashed, so every rank evaluates the same tensor) sliced by rank: a sharded run works on exactly
    # the latents / noise a single process would see for the global batch (SURVEY 8e RNG-parity rule)
    lo, hi = rank * B, (rank + 1) * B
    x0 = synth.synth_tensor("bench.x0.0", (B * world, d.in_channels, d.latent, d.latent), "emb", 1.0, device=dev)[lo:hi].contiguous()
    noise = synth.synth_tensor("bench.noise.0", (B * world, d.in_channels, d.latent, d.latent), "emb", 1.0, device=dev)[lo:hi].contiguous()
    x0_h, noise_h = x0.cpu().pin_memory(), noise.cpu().pin_memory()
    tok_h = torch.empty(B, d.K, dtype=torch.int64).pin_memory()
    out_h = torch.empty_like(noise_h).pin_memory()
    last = {}                                       # outputs of the latest step_device call (kept for --dump-outputs)

    def step_device():
        tok = eng.encode(x0)
        n = eng.last_launch_count
        if world > 1:
            gather_tokens(tok, B * world)           # the path's only exchange: [B,512] int64 per rank over NVLink
        last["tokens"], last["latents"] = tok, eng.decode(tok, noise)
        return n + eng.last_launch_count

    def step_host():
        eng.encode_host(x0_h, tok_h)
        if world > 1:
            gather_tokens(tok_h.to(dev, non_blocking=True), B * world)
        eng.decode_host(tok_h, noise_h, out_h)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        launches = 0
        for _ in range(steps):
            r = fn()
            launches += r or 0
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches

    for _ in range(args.warmup):
        step_device()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, launches = timed(step_device, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    last.clear()
    value = B * world * args.steps / (ms / 1000.0)
    # ---- end to end through the host-buffer entry points
    step_host()
    ms_h, _ = timed(step_host, args.steps)
    e2e = B * world * args.steps / (ms_h / 1000.0)
    h2d = x0_h.numel() * 4 + tok_h.numel() * 8 + noise_h.numel() * 4
    d2h = tok_h.numel() * 8 + out_h.numel() * 4
    # ---- roofline of the dominant kernel class: one profiled (graph-off, event-bracketed) step
    roof = None
    class_roof = None
    prof = {}
    if rank == 0:
        eng.set_use_graph(False)
        eng.set_profile(True)
        tok = eng.encode(x0)
        eng.decode(tok, noise)
        prof = eng.get_profile()
        eng.set_profile(False)
        eng.set_use_graph(True)
        pk = peaks()
        traffic = gemm_traffic()
        total_ms = sum(v[0] for v in prof.values())
        if "gemm_tcgen05" in prof:
            g_ms, g_n = prof["gemm_tcgen05"]
            flops = gemm_flops_per_step(B)
            ach = flops / (g_ms / 1000.0) / 1e12
            roof = {"bound": "tensor", "kernel": "gemm_tc2_kernel (tcgen05 cta_group::2 kind::f16, %s)" % args.precision,
                    "achieved": ach, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": ach / pk["tflops"],
                    "traffic": traffic["bytes_per_launch"] if B == BATCH else None, "traffic_unit": "bytes/launch",
                    "traffic_source": traffic["source"],
                    "timed_in": "a separate graph-off pass of the same step with CUDA events around every launch (the timed region replays "
                                "one CUDA graph; class shares of the two agree within 1 %)",
                    "peak_source": pk["source"], "launches": g_n, "avg_launch_ms": g_ms / g_n,
                    "algorithmic_flops_per_launch": flops / g_n, "share_of_step": g_ms / total_ms,
                    "note": "FLOPs counted once per product (the bf16x3 split passes are overhead, not useful FLOPs); the peak is the bf16 cuBLAS "
                            "figure -- IEEE-half operands draw more power per MMA, the same GEMMs on bf16 operands run 4.8 % faster at the 1 kW cap"}
        class_roof = other_class_rooflines(prof, B, args.precision, pk)
    # ---- the other BASELINE configs, measured in the same run (N = 1 only; each engine is built, timed and released)
    extra = None
    if rank == 0 and world == 1 and not args.no_extra:
        extra = run_extras(args, eng, dev, x0, noise, timed)
    # ---- CPU baseline (oracle port on the host cores), rank 0 at N=1 only
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        eng.close()
        torch.cuda.empty_cache()
        one, scale = cpu_sample(os.cpu_count(), batches=(1, 4))
        cpu = cpu_record(one, scale, batches=(1, 4))
    if rank == 0:
        eff, dense = S.decode_flops_per_image(d.K, d.stages, d.k_per_stage, DECODE_STEPS, d.dit_depth, d.n_img)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": {"bf16x3": "bf16x3 (split-bf16 tcgen05, fp32 accumulate; encoder/VQ fp32)",
                          "fp16": "fp16 (IEEE-half operands on tcgen05, fp32 accumulate; encoder/VQ/tables fp32)",
                          "bf16": "bf16 (tcgen05, fp32 accumulate; encoder/VQ fp32)", "fp32": "f32"}[args.precision],
                "data": "synthetic",
                "config": {"workload": f"batch={B}/GPU 256x256 encode + 50-step diffusion decode (512 tokens, no VAE/renderer)",
                           "batch_per_gpu": B, "global_batch": B * world, "decode_steps": DECODE_STEPS, "precision": args.precision,
                           "parallelism": f"dp{world} (images sharded, weights replicated, 1 NCCL all-gather of tokens/step)",
                           "l2": "working set >> L2 (126 MB): %.1f GB of 16-bit weight planes + ~3 GB of activations streamed per DiT step"
                                 % (4.17 * (2 if args.precision == "bf16x3" else 1)),
                           "algorithmic_tflop_per_image": eff / 1e12},
                "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": ms_h / args.steps},
                "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "extra": extra,
                "kernel_classes_ms": {k: round(v[0], 3) for k, v in prof.items()},
                "kernel_classes_roofline": class_roof,
                "kernel_classes_launches": {k: v[1] for k, v in prof.items()}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("SELFTOK_PRECISION", "fp16"), choices=["bf16x3", "fp16", "bf16", "fp32"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extra", action="store_true", help="skip the sub-records of the other BASELINE configs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the tokens and latents of the last timed step as DIR/tokens.npy and DIR/latents.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs applies to the CUDA path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the selftok_b200 path has no CPU fallback "
                         "(use --impl reference for the CPU arithmetic)")
    if args.gpus > 1 and "RANK" not in os.environ:
        raise SystemExit("launch multi-GPU runs with: python -m torch.distributed.run --nnodes=1 --nproc-per-node N "
                         "--master-addr 127.0.0.1 --master-port P bench.py --gpus N ...")
    run_gpu(args)


if __name__ == "__main__":
    main()
