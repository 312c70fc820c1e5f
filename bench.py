#!/usr/bin/env python
"""bench.py -- denoise-step throughput of the Wan DiT hot path (+ WanVAE decode frames/s) on B200.

    python bench.py --gpus N --steps K --warmup W              (N > 1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference ...                        (CPU arm: the oracle port on the host cores)

A "step" is ONE denoise step of BASELINE.json configs[1]: Wan2.2 t2v 14B (high+low-noise experts resident), latent
[1,16,21,90,160] (720p x 81 frames, L = 75 600 tokens), text context [1,512,4096], CFG => two DiT forwards (cond,
uncond), CFG combine and the flow-matching Euler update; synthetic latents, random-init weights of that architecture.
Multi-GPU: every rank denoises its own independent sample (north star: batch split, no data-path collective inside a
step) => weak scaling; value = total steps/s over all ranks, timed on the device, max over ranks.
Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (config, latent (T,H,W), two experts?, description)
    "wan22_t2v_14b_720p81": ("t2v_2_2", (21, 90, 160), True, "Wan2.2 t2v 14B, latent [1,16,21,90,160] (720p x 81f), CFG pair, 50-step Euler schedule shift 12"),
    # the same model at 480p (832 x 480 x 81f): L = 32 760
    "wan22_t2v_14b_480p81": ("t2v_2_2", (21, 60, 104), True, "Wan2.2 t2v 14B, latent [1,16,21,60,104] (480p x 81f), CFG pair, 50-step Euler schedule shift 12"),
    # BASELINE configs[2]: Wan2.2 i2v 14B (in_dim 36: 16 latent + 4 mask + 16 image-latent channels), CFG pair
    "wan22_i2v_14b_720p81": ("i2v_2_2", (21, 90, 160), True, "Wan2.2 i2v 14B, latent [1,16,21,90,160] + y [20,21,90,160] (720p x 81f), CFG pair, 50-step Euler schedule shift 5"),
    "wan21_t2v_1.3b_p": ("t2v_1.3B", (9, 30, 52), False, "Wan2.1 t2v 1.3B, latent [1,16,9,30,52] (BASELINE config 0), CFG pair"),
    "tiny": ("small", (5, 16, 24), False, "reduced config for smoke runs"),
    # BASELINE configs[3]: Hunyuan Video 1.5 t2v 720p, 129 frames -> latent [1,32,33,45,80] (+33 cond channels), 54 double blocks
    "hy15_t2v_720p129": ("HYVideo-1_5", (33, 45, 80), False, "Hunyuan Video 1.5 t2v 720p x 129f, latent [1,32,33,45,80]+33 cond ch, L=118800 (+767 text), CFG pair, 30-step Euler shift 9"),
    "hy15_tiny": ("hy_tiny", (3, 6, 10), False, "reduced Hunyuan config for smoke runs"),
    # HunyuanVideo 1.0 (guidance-distilled: ONE forward per step), 720p x 129f: latent [1,16,33,90,160], patch (1,2,2) -> L = 118800
    "hy10_t2v_720p129": ("HYVideo-T/2-cfgdistill", (33, 90, 160), False, "HunyuanVideo 1.0 cfg-distilled t2v 720p x 129f, latent [1,16,33,90,160], L=118800 (+256 text), 20 double + 40 single blocks, one forward per step"),
    "hy10_tiny": ("hy10_tiny", (2, 8, 12), False, "reduced HunyuanVideo 1.0 config for smoke runs"),
}


DUMP_MAX_ELEMENTS = 5_000_000      # per output: a run dumps at most three (latents, decoded frames, encoded latents) = 60 MB


def dump_sample(t, name):
    """`t` as float32 on the host for --dump-outputs: whole up to DUMP_MAX_ELEMENTS, else that many elements (flattened) at positions
    drawn from a generator seeded by `name`, so that every run with the same arguments samples the same positions."""
    flat = t.detach().reshape(-1)
    if flat.numel() > DUMP_MAX_ELEMENTS:
        g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
        idx = torch.randint(0, flat.numel(), (DUMP_MAX_ELEMENTS,), generator=g).sort().values
        return flat[idx.to(flat.device)].float().cpu()
    return t.detach().float().cpu()


def hy_flops_forward(cfg, L, Lt):
    D, nl, ns = cfg["hidden_size"], cfg["mm_double_blocks_depth"], cfg.get("mm_single_blocks_depth", 0)
    n = L + Lt
    return (nl + ns) * (4.0 * n * n * D + 8.0 * n * D * D + 16.0 * n * D * D)


def measure_hunyuan(workload, steps, warmup, rank, world, local_rank, dev, dist, with_vae=True, cfg_split=False, outputs=None):
    """Hunyuan Video denoise-step measurement (same JSON contract, steps of cond+uncond forwards + CFG + Euler) -> result dict.
    `outputs` (a dict, or None): receives what the timed steps and the timed VAE decode computed (see dump_sample)."""
    import types
    from wan2gp_b200 import _lib, ops, synth
    from wan2gp_b200.hyvideo import HYVideoDiffusionTransformer, get_rotary_pos_embed
    from wan2gp_b200.pipeline import HunyuanDenoiser
    args = types.SimpleNamespace(workload=workload, steps=steps, warmup=warmup, no_vae=not with_vae)
    cfg_name, thw, _, desc = WORKLOADS[args.workload]
    cfg = synth.HY_CONFIGS[cfg_name]
    v10 = cfg.get("family") == "1.0"
    T, H, W = thw
    P = cfg["patch_size"][1]
    L, Lt, Lb = T * (H // P) * (W // P), 511, 256
    if v10:
        Lt, Lb = 256, 0
    if cfg_name in ("hy_tiny", "hy10_tiny"):
        Lt, Lb = 24, (0 if v10 else 12)
    kw = dict(mm_single_blocks_depth=cfg["mm_single_blocks_depth"], text_states_dim_2=cfg["text_states_dim_2"], guidance_embed=True) if v10 \
        else dict(mm_single_blocks_depth=0, text_pool_type=None, glyph_byT5_v2=True, use_cond_type_embedding=True, pre_split_qkv=True)
    model = HYVideoDiffusionTransformer(i2v_condition_type=None, patch_size=cfg["patch_size"], in_channels=cfg["in_channels"],
                                        out_channels=cfg["out_channels"], hidden_size=cfg["hidden_size"], heads_num=cfg["heads_num"],
                                        mm_double_blocks_depth=cfg["mm_double_blocks_depth"], text_states_dim=cfg["text_states_dim"],
                                        device=dev, **kw).init_synthetic(seed=1)
    # cfg_split (BASELINE configs[3] as 2 samples x 2 CFG branches on 4 GPUs): ranks (2k, 2k+1) hold the same sample, each runs ONE
    # forward per step and the pair exchanges the fp32 prediction (one 2-rank all-gather per step), as `--cfg-split` does for Wan
    group, cfg_rank, sample, n_samples = None, 0, rank, world
    if cfg_split and dist is not None and world % 2 == 0 and not v10:
        from wan2gp_b200 import dist as wd
        group, cfg_rank, sample, n_samples = wd.make_cfg_pairs()
    den = HunyuanDenoiser(model, num_steps=30, shift=9.0 if not v10 else 7.0, guide_scale=6.0, device=dev, cfg_group=group, cfg_rank=cfg_rank)
    g = torch.Generator().manual_seed(1000 + sample)
    lat_host = torch.randn(1, cfg["out_channels"], T, H, W, generator=g).pin_memory()
    latents = lat_host.to(dev)
    cond = torch.zeros(1, cfg["in_channels"] - cfg["out_channels"], T, H, W, device=dev) if cfg["in_channels"] > cfg["out_channels"] else None
    t2 = torch.randn(1, cfg["text_states_dim_2"], generator=g).to(dev) if v10 else None
    gd = torch.tensor([6000.0]) if v10 else None
    txt = torch.randn(1, Lt, cfg["text_states_dim"], generator=g).to(dev)
    txt0 = torch.randn(1, Lt, cfg["text_states_dim"], generator=g).to(dev)
    tm = torch.ones(1, Lt, dtype=torch.long)
    b5 = torch.randn(1, Lb, synth.HY_BYT5_DIMS[0], generator=g).to(dev) if Lb else None
    bm = torch.ones(1, Lb, dtype=torch.long) if Lb else None
    freqs = get_rotary_pos_embed((T, H // P, W // P))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def one(k, lat):
        return den.step(lat, cond, min(k, den.num_steps - 1), txt, tm, None if v10 else txt0, tm, b5, bm, freqs, text_states_2=t2, guidance=gd)
    for k in range(args.warmup):
        one(k, latents)
    barrier()
    l0 = _lib.launch_count()
    ops.TIMED["attention"] = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        e0.record()
        for k in range(args.steps):
            one(args.warmup + k, latents)
        e1.record()
        barrier()
    ms = e0.elapsed_time(e1)
    launches = _lib.launch_count() - l0
    if outputs is not None:
        outputs["latents"] = dump_sample(latents, "latents")
    att = [(a.elapsed_time(b), w) for a, b, w in ops.TIMED.pop("attention") if w > 1e12]
    # end to end with host buffers
    n_e2e = max(1, min(args.steps, 3))
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for k in range(n_e2e):
        lat = lat_host.to(dev, non_blocking=True)
        one(args.warmup + k, lat)
        lat_host.copy_(lat, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    t1.record()
    barrier()
    tms = torch.tensor([ms, t0.elapsed_time(t1)], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(tms[0]), float(tms[1])
    pk = peaks()
    fl = (1.0 if v10 or group is not None else 2.0) * hy_flops_forward(cfg, L, Lt + Lb)      # per GPU and step
    att_ms = sum(a for a, _ in att) / max(1, len(att))
    att_tf = (att[0][1] / (att_ms * 1e-3) / 1e12) if att else None
    par = (f"{n_samples} samples in flight, every CFG pair split over 2 GPUs (one forward per GPU and step, one 2-rank all-gather of the "
           f"fp32 prediction per step)") if group is not None else f"{world} independent samples (batch split), 1 per GPU"
    res = {"metric": "denoise_steps_per_sec", "value": n_samples * args.steps / (ms / 1e3), "unit": "steps/s", "n_gpus": world,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
           "config": {"workload": args.workload, "description": desc, "latent": [1, cfg["out_channels"], T, H, W], "tokens": L,
                      "text_tokens": Lt + Lb, "cfg_pair": not v10, "parallelism": par,
                      "l2_policy": "inputs larger than L2; no flush needed"},
           "e2e": {"value": n_samples * n_e2e / (e2e_ms / 1e3), "unit": "steps/s", "steps": n_e2e,
                   "h2d_bytes_per_step": lat_host.numel() * 4, "d2h_bytes_per_step": lat_host.numel() * 4},
           "gpu_launches": launches, "finite": bool(torch.isfinite(latents).all()),
           "model_tflops": fl / (ms / args.steps * 1e-3) / 1e12,
           "model_tensor_frac": fl / (ms / args.steps * 1e-3) / 1e12 / pk["tensor_sustained"],
           "roofline": {"kernel": attention_kernel_name() + " (joint img+txt attention)", "bound": "tensor", "achieved": att_tf,
                        "peak": pk["tensor_sustained"], "unit": "TFLOP/s", "frac": None if att_tf is None else att_tf / pk["tensor_sustained"],
                        "peak_source": pk["source"] + ", sustained figure", "launches_timed": len(att), "avg_launch_ms": att_ms,
                        "share_of_step": (sum(a for a, _ in att) / ms) if att else None, "traffic": None},
           "clocks": clk.summary()}

    # ---- VAE decode of the finished clip (second half of the metric): un-tiled Hunyuan decoder, one clip per GPU
    if not args.no_vae:
        from wan2gp_b200.hyvideo import HYVAE10Decoder, HYVAEDecoder
        del den, model
        torch.cuda.empty_cache()
        tiny = cfg_name in ("hy_tiny", "hy10_tiny")
        if v10:
            vname = "hyvae10_tiny" if tiny else "hyvae10"
            vcfg = synth.HYVAE10_CONFIGS[vname]
            dec = HYVAE10Decoder(vcfg, dev)
            dec.load_state_dict(synth.make_hyvae10_state_dict(vcfg, 0, device=dev))
            zc, fs = vcfg["latent_channels"], 8
        else:
            vname = "hyvae_tiny" if tiny else "hyvae15"
            vcfg = synth.HYVAE_CONFIGS[vname]
            dec = HYVAEDecoder(vcfg, dev)
            dec.load_state_dict(synth.make_hyvae_state_dict(vcfg, 0, device=dev))
            zc, fs = vcfg["z_channels"], vcfg["ffactor_spatial"]
        zh = torch.randn(1, zc, T, H, W, generator=g).pin_memory()
        try:
            z = zh.to(dev)
            torch.cuda.reset_peak_memory_stats()
            fr = dec(z)                                      # warm-up
            nfr = fr.shape[2]
            del fr
            barrier()
            l0 = _lib.launch_count()
            v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            v0.record()
            fr = dec(z)
            v1.record()
            barrier()
            vlaunch = _lib.launch_count() - l0
            if outputs is not None:
                outputs["vae_decode_frames"] = dump_sample(fr, "vae_decode_frames")
            del fr
            # end to end: latent on host -> uint8 frames on host
            w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            w0.record()
            fr = dec(zh.to(dev, non_blocking=True))[0]
            u8 = torch.empty(fr.shape, device=dev, dtype=torch.uint8)
            _lib.call("b200_frames_to_u8", fr.data_ptr(), u8.data_ptr(), fr.numel(), torch.cuda.current_stream().cuda_stream)
            u8h = u8.cpu()
            w1.record()
            barrier()
            vt = torch.tensor([v0.elapsed_time(v1), w0.elapsed_time(w1)], device=dev, dtype=torch.float64)
            if dist is not None:
                dist.all_reduce(vt, op=dist.ReduceOp.MAX)
            res["vae_decode"] = {"metric": "vae_decode_frames_per_sec", "decoder": vname, "value": world * nfr / (float(vt[0]) / 1e3),
                                 "unit": "frames/s", "frames": nfr, "resolution": [fs * H, fs * W], "ms_per_clip": float(vt[0]),
                                 "gpu_launches": vlaunch, "tiling": "none (whole clip resident)",
                                 "peak_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30,
                                 "e2e": {"value": world * nfr / (float(vt[1]) / 1e3), "unit": "frames/s", "h2d_bytes": zh.numel() * 4,
                                         "d2h_bytes": u8h.numel()}}
        except Exception as e:                               # noqa: BLE001  (e.g. out of memory on a smaller GPU)
            res["vae_decode"] = {"decoder": vname, "error": repr(e)[:300]}
    torch.cuda.empty_cache()
    return res


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"tensor_burst": p["bf16_tflops"], "tensor_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "hbm": p["hbm_gbs"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"tensor_burst": 1590.0, "tensor_sustained": 1400.0, "hbm": 6650.0, "source": "fallback (B200_PROFILING.md)"}


def wan_flops_forward(cfg, L, Lt):
    D, F, nl = cfg["dim"], cfg["ffn_dim"], cfg["num_layers"]
    per_block = 4.0 * L * L * D + 8.0 * L * D * D + (4.0 * L * D * D + 4.0 * Lt * D * D + 4.0 * L * Lt * D) + 4.0 * L * D * F
    return nl * per_block


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], threading.Event()
        self.th = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(len(r) > 3 + j and r[3 + j].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons, "samples": len(sm)}


def cpu_port_steps_per_sec(cfg, thw, reps=1):
    """Reference CPU arm / cpu_baseline: the oracle port (oracle/wan_oracle.py, fp32, all host threads) on a BOUNDED sample of the
    workload -- ONE transformer block of this architecture, its two cost components timed separately so that each is scaled by its
    own share of the real step (VERDICT r01 #13: a 1-frame slice has 11 % attention, the real 720p step 72 %):
      * the row-wise part (LN/modulation, q/k/v/o, cross-attention, FFN) on `Ls` tokens (3 latent frames), scaled by L / Ls;
      * self-attention of `Lq` sampled query rows against ALL L keys / values through torch's CPU SDPA (what the reference calls), scaled by L / Lq.
    step time = 2 forwards x num_layers x (t_rows L/Ls + t_attn L/Lq); stated as extrapolated.  Returns (steps/s, info dict)."""
    from oracle import wan_oracle
    from wan2gp_b200 import synth
    T, H, W = thw
    D, NH, nl = cfg["dim"], cfg["num_heads"], cfg["num_layers"]
    L = T * (H // 2) * (W // 2)
    big = D > 2000
    Ts = min(T, 3) if big else T
    Ls = Ts * (H // 2) * (W // 2)
    Lq = min(L, 2048 if big else L)
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    shapes = synth.wan_param_shapes(cfg)
    sd = {n: synth.make_wan_tensor(n, s, cfg, 0, "cpu") for n, s in shapes.items() if n.startswith("blocks.0.")}
    x = torch.randn(Ls, D)
    e0 = torch.randn(6, D) * 0.1
    ctx = torch.randn(cfg["text_len"], D)
    cos, sin = wan_oracle.rope_tables((Ts, H, W))
    # self-attention sample: the reference's OWN CPU attention call (shared/attention.py:208-225 sdpa_wrapper ->
    # F.scaled_dot_product_attention on [1, H, L, 128]), not the oracle's materialised softmax(QK^T)V -- the latter spends its time in
    # strided copies and a 1.5e9-element exp on one socket and understated the CPU by an order of magnitude in the first version
    q = torch.randn(1, NH, Lq, 128)
    k = torch.randn(1, NH, L, 128)
    v = torch.randn(1, NH, L, 128)
    t_rows, t_attn = [], []
    # inside the timed block the oracle's attention is evaluated the way the reference evaluates it on a CPU (SDPA), so that the
    # sample-sized self-attention contained in block_forward and the separately timed full-length one are the same code
    sdpa = torch.nn.functional.scaled_dot_product_attention
    oracle_attention = wan_oracle.attention
    wan_oracle.attention = lambda q_, k_, v_, emulate: sdpa(q_.permute(1, 0, 2)[None], k_.permute(1, 0, 2)[None], v_.permute(1, 0, 2)[None])[0].permute(1, 0, 2)
    try:
      with torch.no_grad():
          wan_oracle.block_forward(sd, cfg, 0, x[:256], e0, ctx, cos[:256], sin[:256], False)          # warm-up (thread pool, allocator)
          for _ in range(reps):
              t0 = time.time()
              wan_oracle.block_forward(sd, cfg, 0, x, e0, ctx, cos, sin, False)
              t1 = time.time()
              sdpa(q, k, v)
              t2 = time.time()
              # block_forward(x) contains the Ls x Ls self-attention of the sample itself: remove its (small, separately scaled) cost
              t_self = (t2 - t1) * (Ls * Ls) / (Lq * L)
              t_rows.append(max(1e-6, (t1 - t0) - t_self))
              t_attn.append(t2 - t1)
    finally:
        wan_oracle.attention = oracle_attention
    tr, ta = min(t_rows), min(t_attn)
    block_s = tr * L / Ls + ta * L / Lq
    step_s = 2.0 * nl * block_s
    fl_rows = 12.0 * Ls * D * D + 4.0 * cfg["text_len"] * D * D + 4.0 * Ls * cfg["text_len"] * D + 4.0 * Ls * D * cfg["ffn_dim"]
    fl_attn = 4.0 * Lq * L * D
    info = {"cores": threads, "sample_seconds": sum(t_rows) + sum(t_attn), "reps": reps, "min_rows_s": tr, "min_attn_s": ta,
            "median_rows_s": sorted(t_rows)[len(t_rows) // 2], "median_attn_s": sorted(t_attn)[len(t_attn) // 2],
            "rows_tflops": fl_rows / tr / 1e12, "attn_tflops": fl_attn / ta / 1e12, "attention_share_of_step": (ta * L / Lq) / block_s,
            "sample": f"1 of {nl} blocks, fp32, {threads} threads: row-wise part on {Ts} of {T} latent frames (Ls={Ls}: {tr:.2f} s, "
                      f"{fl_rows / tr / 1e12:.2f} TFLOP/s), self-attention of {Lq} query rows x all {L} keys ({ta:.2f} s, {fl_attn / ta / 1e12:.2f} TFLOP/s); "
                      f"each scaled by its own token ratio to the full block, x{nl} blocks x2 CFG forwards (extrapolated)"}
    return 1.0 / step_s, info


def wan_vae_work(Tl, h, w):
    """Algorithmic work of one WanVAE decode of a [16,Tl,h,w] latent from the decoder's layer list (synth.vae_decoder_layout =
    Decoder3d, vae.py:430-484): (reference_flops, executed_flops, bytes_algorithmic).  reference = the convolutions as the
    reference runs them (nearest-2x up-sampling then Conv2d 3x3 on the up-sampled tensor); executed = ours (the same map as four
    2x2 sub-pixel convs on the low-resolution tensor: 16 instead of 36 taps per source pixel).  bytes = every conv reads its input
    and writes its output once in bf16 (norm+SiLU fused away), the planar fp32 frames written once: the minimum activation traffic."""
    from wan2gp_b200 import synth
    c0, ups, c_out = synth.vae_decoder_layout(synth.VAE_CFG)
    acc = {"ref": 0.0, "ex": 0.0, "by": 0.0}

    def conv(ci, co, taps, t, hh, ww, out_bytes=2):
        f = 2.0 * t * hh * ww * ci * co * taps
        acc["ref"] += f
        acc["ex"] += f
        acc["by"] += t * hh * ww * (ci * 2 + co * out_bytes)

    def res(ci, co, t, hh, ww):
        conv(ci, co, 27, t, hh, ww)
        conv(co, co, 27, t, hh, ww)
        if ci != co:
            conv(ci, co, 1, t, hh, ww)
    T, H, W = Tl, h, w
    conv(16, c0, 27, T, H, W)
    res(c0, c0, T, H, W)
    conv(c0, 3 * c0, 1, T, H, W)
    conv(c0, c0, 1, T, H, W)
    att = 4.0 * T * (H * W) ** 2 * c0
    acc["ref"] += att
    acc["ex"] += att
    res(c0, c0, T, H, W)
    for u in ups:
        if u[0] == "res":
            res(u[1], u[2], T, H, W)
            continue
        c = u[1]
        if u[0] == "up3d" and T > 1:
            conv(c, 2 * c, 3, T - 1, H, W)
            T = 2 * T - 1
        f = 2.0 * T * (4 * H * W) * c * (c // 2) * 9
        acc["ref"] += f
        acc["ex"] += f * 16.0 / 36.0
        acc["by"] += T * H * W * c * 2 + T * 4 * H * W * (c // 2) * 2
        H, W = 2 * H, 2 * W
    conv(c_out, 3, 27, T, H, W, out_bytes=4)
    return acc["ref"], acc["ex"], acc["by"], T


def attention_kernel_name():
    """The self-attention kernel behind ops.attention: csrc/c_api.cu picks it from B200_ATT_VARIANT (default 614 = attn6_sm100.cuh)."""
    v = int(os.environ.get("B200_ATT_VARIANT", "614"))
    return "attn_s3_fwd_d128_kernel" if 600 <= v < 700 else "attn_s2_fwd_d128_kernel" if 500 <= v < 600 else "attn_fwd_d128_kernel"


def dram_traffic(kernel, shape_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` at `shape_key`, from the ncu --set full capture summarised
    in profiles/ncu_dram_traffic.json (written from the .ncu-rep by tools/ncu_summary.py; a profiler number, never measured inside a
    timed run).  None if no capture of this kernel at this shape is committed."""
    path = os.path.join(ROOT, "profiles", "ncu_dram_traffic.json")
    if not os.path.exists(path):
        return None, None
    rec = json.load(open(path)).get(kernel, {}).get(shape_key)
    return (rec["dram_bytes"], rec.get("source")) if rec else (None, None)


def sample_rows(L, n_random=192, tile=128, seed=0):
    fixed = list(range(0, 32)) + list(range(tile - 4, tile + 4)) + list(range(max(0, (L // tile) * tile - 8), L))
    g = torch.Generator().manual_seed(seed)
    rows = sorted(set(r for r in fixed + torch.randint(0, L, (n_random,), generator=g).tolist() if 0 <= r < L))
    return torch.tensor(rows, dtype=torch.long)


def parity_probe_wan(model, latents, tval, freqs, y_dev, dev):
    """Parity of the two dominant kernels ON THE BENCHMARKED TENSORS: block 0 of the benchmarked expert is re-run on the latents the
    timed steps produced (patch embed -> LN/modulate -> fused qkv GEMM -> q/k RMSNorm+RoPE -> self-attention at the full L), and
    sampled rows (first tile, last partial tile, random) of the qkv GEMM and of the attention output are compared with fp64 torch
    on the same operands.  (Block / VAE level parity at these shapes against the oracle: tests/test_prod_shapes_gpu.py.)"""
    import math
    from wan2gp_b200 import ops
    D, H = model.dim, model.num_heads
    blk = model.blocks[0]
    cos, sin = model._freqs(freqs, tuple(latents.shape[2:]))
    x = ops.patch_embed(latents[0].contiguous(), y_dev, model._g["pe_w"], model._g["pe_b"], D)
    L = x.shape[0]
    _, e0 = model._time(torch.tensor([tval]))
    m = ops.add_vec(blk.modulation, e0)
    a = ops.ln_modulate(x, m[0:D], m[D:2 * D], eps=model.eps)
    qkv = ops.gemm(a, blk.w_qkv, bias=blk.b_qkv)
    rows = sample_rows(L).to(dev)
    ref = a[rows].double() @ blk.w_qkv.double().t() + blk.b_qkv.double()
    got = qkv[rows].double()
    gemm_rel = float((got - ref).norm() / ref.norm())
    ops.qk_rmsnorm_rope_(qkv[:, :D], qkv[:, D:2 * D], blk.nq, blk.nk, model.eps, cos, sin)
    att = ops.attention(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], H)
    heads = sorted({0, H // 2, H - 1})
    num = den = 0.0
    worst, peak, mse, cnt = 0.0, 0.0, 0.0, 0
    for h in heads:
        sl = slice(h * 128, (h + 1) * 128)
        qh, kh, vh = qkv[rows, sl].double(), qkv[:, D + h * 128:D + (h + 1) * 128].double(), qkv[:, 2 * D + h * 128:2 * D + (h + 1) * 128].double()
        r = torch.softmax(qh @ kh.t() / math.sqrt(128.0), -1) @ vh
        g = att[rows, sl].double()
        num += float((g - r).pow(2).sum()); den += float(r.pow(2).sum())
        worst = max(worst, float((g - r).abs().max())); peak = max(peak, float(r.abs().max()))
        mse += float((g - r).pow(2).sum()); cnt += r.numel()
    att_rel = (num / den) ** 0.5
    psnr = 10.0 * math.log10(peak * peak / (mse / cnt)) if mse > 0 else float("inf")
    return {"on": "benchmarked latents, block 0 of the active expert, full token count", "tokens": L, "rows_checked": int(rows.numel()),
            "heads_checked": heads, "gemm_qkv_rel_l2": gemm_rel, "attention_rel_l2": att_rel, "attention_max_abs_err": worst,
            "max_rel_l2": max(gemm_rel, att_rel), "psnr_db": psnr, "tolerance_rel_l2": 4e-3, "ok": max(gemm_rel, att_rel) < 4e-3,
            "finite": bool(torch.isfinite(att.float()).all()), "reference": "torch fp64 on the same bf16 operands"}


def measure_wan(workload, steps, warmup, rank, world, local_rank, dev, dist, cfg_split=False, with_vae=True, with_parity=True,
                e2e_steps=3, with_encode=True, outputs=None):
    """One Wan bench measurement -> result dict (the JSON line of the main workload, or a sub-run block).
    `outputs` (a dict, or None): receives what the timed steps and the timed VAE decode / encode computed (see dump_sample)."""
    from wan2gp_b200 import _lib, ops, synth
    from wan2gp_b200.pipeline import WanDenoiser
    from wan2gp_b200.wan import WanModel, WanVAE, get_rotary_pos_embed
    cfg_name, thw, two_experts, desc = WORKLOADS[workload]
    cfg = synth.WAN_CONFIGS[cfg_name]
    T, H, W = thw
    L = T * (H // 2) * (W // 2)
    config = {"workload": workload, "description": desc, "latent": [1, 16, T, H, W], "tokens": L, "context": [1, cfg["text_len"], cfg["text_dim"]],
              "cfg_pair": True, "parallelism": f"{world} independent samples (batch split), 1 per GPU",
              "l2_policy": "inputs larger than L2 (weights 28 GB / expert, activations > 1 GB per tensor); no flush needed"}
    model = WanModel(**cfg, device=dev).init_synthetic(seed=1)
    model2 = WanModel(**cfg, device=dev).init_synthetic(seed=2) if two_experts else None
    if L <= 16384:          # launch-bound configs: replay captured CUDA graphs
        model.use_cuda_graphs = True
        if model2 is not None:
            model2.use_cuda_graphs = True
    i2v = cfg["in_dim"] > 16
    n_samples, sample_id, cfg_kw = world, rank, {}
    if cfg_split and world > 1:
        from wan2gp_b200 import dist as wdist
        grp, cfg_rank, sample_id, n_samples = wdist.make_cfg_pairs()
        cfg_kw = dict(cfg_group=grp, cfg_rank=cfg_rank)
        config["parallelism"] = f"{n_samples} samples, each CFG pair split over 2 GPUs (per-step 2-rank all-gather of the prediction)"
    den = WanDenoiser(model, model2, num_steps=50, shift=5.0 if i2v else 12.0, guide_scale=3.5 if i2v else 4.0,
                      guide2_scale=3.5 if i2v else 3.0, switch_threshold=900 if i2v else 875, device=dev, **cfg_kw)
    if L <= 16384 and not cfg_kw and os.environ.get("B200_STEP_GRAPH", "1") != "0":
        den.use_step_graph = True          # launch-bound configs: one captured graph per step (pipeline.WanDenoiser._graph_step)
        config["cuda_graph"] = "whole step (both CFG forwards + combine + Euler update), timestep / guidance / dt read from device memory"
    freqs = get_rotary_pos_embed(thw)
    g = torch.Generator().manual_seed(1000 + sample_id)
    y_dev = None
    if i2v:
        y_dev = torch.randn(cfg["in_dim"] - 16, T, H, W, generator=g).to(dev)
        y_dev[:4] = (y_dev[:4] > 0).float()
    lat_host = torch.randn(1, 16, T, H, W, generator=g).pin_memory()
    ctx_host = torch.randn(1, cfg["text_len"], cfg["text_dim"], generator=g).pin_memory()
    ctxn_host = torch.zeros(1, cfg["text_len"], cfg["text_dim"]).pin_memory()
    latents = lat_host.to(dev)
    ctx, ctxn = ctx_host.to(dev), ctxn_host.to(dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # steps are taken around the expert switch (t = 875) so both experts are exercised like in the real schedule
    sw = next((i for i, t in enumerate(den.timesteps[:-1]) if t <= den.switch_threshold), 0)
    first = max(0, sw - (warmup + steps) // 2)

    def step_idx(k):
        return min(first + k, den.num_steps - 1)

    for k in range(warmup):
        den.step(latents, step_idx(k), ctx, ctxn, y=y_dev, freqs=freqs)
    barrier()
    launches0 = _lib.launch_count() + den.graph_launches
    ops.TIMED["attention"] = []
    ops.TIMED["gemm"] = []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    prof_range = bool(os.environ.get("B200_CUDA_PROFILER_RANGE"))     # ncu --profile-from-start off: only the timed steps
    if prof_range:
        torch.cuda.profiler.start()
    with ClockSampler(local_rank) as clk:
        ev0.record()
        for k in range(steps):
            den.step(latents, step_idx(warmup + k), ctx, ctxn, y=y_dev, freqs=freqs)
        ev1.record()
        barrier()
    if prof_range:
        torch.cuda.profiler.stop()
    ms = ev0.elapsed_time(ev1)
    if outputs is not None:
        outputs["latents"] = dump_sample(latents, "latents")
    launches = _lib.launch_count() + den.graph_launches - launches0      # kernels inside replayed whole-step graphs included
    att = ops.TIMED.pop("attention")
    att_ms = [a.elapsed_time(b) for a, b, _ in att]
    att_work = att[0][2] if att else 0.0
    gm = [(a.elapsed_time(b), w) for a, b, w in ops.TIMED.pop("gemm") if w > 1e12]       # the four large linear layers of each block
    ok = bool(torch.isfinite(latents).all())

    # ---- end to end through the public API with host buffers (H2D of latents+contexts, D2H of the new latents, every step)
    e2e_steps = max(1, min(steps, e2e_steps))
    barrier()
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    for k in range(e2e_steps):
        den.step_host(lat_host, step_idx(warmup + k), ctx_host, ctxn_host, y=y_dev, freqs=freqs)
    t1.record()
    barrier()
    e2e_ms = t0.elapsed_time(t1)

    times = torch.tensor([ms, e2e_ms], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(times[0]), float(times[1])
    pk = peaks()
    steps_per_s = n_samples * steps / (ms / 1000.0)
    flops_step = 2.0 * wan_flops_forward(cfg, L, cfg["text_len"]) * (n_samples / world)      # per GPU
    att_avg = sum(att_ms) / max(1, len(att_ms))
    att_tf = att_work / (att_avg * 1e-3) / 1e12 if att_ms else None
    att_kernel = attention_kernel_name()
    traffic, traffic_src = dram_traffic(att_kernel, f"L{L}_H{cfg['num_heads']}")
    gemm_tf = (sum(w for _, w in gm) / (sum(t for t, _ in gm) * 1e-3) / 1e12) if gm else None
    result = {
        "metric": "denoise_steps_per_sec", "value": steps_per_s, "unit": "steps/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic", "config": config,
        "e2e": {"value": n_samples * e2e_steps / (e2e_ms / 1000.0), "unit": "steps/s", "steps": e2e_steps,
                "note": f"{e2e_steps} steps through WanDenoiser.step_host: pinned host latents + contexts -> device, one step, new latents -> host (the copies are ~40 MB next to an ~11 s step)",
                "h2d_bytes_per_step": lat_host.numel() * 4 + ctx_host.numel() * 4 + ctxn_host.numel() * 4,
                "d2h_bytes_per_step": lat_host.numel() * 4},
        "gpu_launches": launches,
        "finite": ok,
        "model_tflops": flops_step / (ms / steps * 1e-3) / 1e12,
        "model_tensor_frac": flops_step / (ms / steps * 1e-3) / 1e12 / pk["tensor_sustained"],
        "roofline": {"kernel": att_kernel + " (self-attention, 72% of step FLOPs)", "bound": "tensor", "achieved": att_tf,
                     "peak": pk["tensor_sustained"], "unit": "TFLOP/s", "frac": None if att_tf is None else att_tf / pk["tensor_sustained"],
                     "peak_source": pk["source"] + ", sustained figure (kernel timed inside a long step)",
                     "launches_timed": len(att_ms), "avg_launch_ms": att_avg,
                     "share_of_step": sum(att_ms) / ms if att_ms else None,
                     "algorithmic_flops_per_launch": att_work,
                     "algorithmic_bytes_per_launch": 4.0 * L * cfg["dim"] * 2,
                     "traffic": traffic, "traffic_unit": "bytes/launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)", "traffic_source": traffic_src},
        "gemm_in_step": {"kernel": "gemm_pair_tcgen05_kernel / gemm_tcgen05_kernel (qkv, o, ffn.0, ffn.2 and cross q/o)", "launches_timed": len(gm),
                         "achieved": gemm_tf, "unit": "TFLOP/s", "frac_of_sustained": None if gemm_tf is None else gemm_tf / pk["tensor_sustained"],
                         "share_of_step": (sum(t for t, _ in gm) / ms) if gm else None},
        "clocks": clk.summary(),
    }
    if with_parity and not cfg_split:
        try:
            act, _ = den.expert(den.timesteps[step_idx(warmup + steps - 1)])
            result["parity"] = parity_probe_wan(act, latents, den.timesteps[step_idx(warmup + steps - 1)], freqs, y_dev, dev)
        except Exception as e:                                    # noqa: BLE001  (never lose the timing line to the probe)
            result["parity"] = {"error": repr(e)[:300]}

    # ---- VAE decode frames/s (second half of the metric), one clip per GPU
    if with_vae:
        del den, model, model2
        torch.cuda.empty_cache()
        vae = WanVAE(device=dev, state_dict=synth.make_vae_state_dict(seed=0, encoder=True))
        z = torch.randn(16, T, H, W, generator=g).to(dev)
        nfr = 4 * (T - 1) + 1
        vae.decode_to_cpu_uint8([z], 0)
        barrier()
        l0 = _lib.launch_count()
        v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        v0.record()
        reps = 2
        for _ in range(reps):
            fr = vae.model.decode_frames(z, vae.mean, vae.std)
        v1.record()
        barrier()
        vms = torch.tensor([v0.elapsed_time(v1)], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(vms, op=dist.ReduceOp.MAX)
        vms = float(vms[0]) / reps
        if outputs is not None:
            outputs["vae_decode_frames"] = dump_sample(fr, "vae_decode_frames")
        # end to end: latent on host -> uint8 frames on host
        zh = z.cpu().pin_memory()
        tt0 = time.time()
        u8 = vae.decode_to_cpu_uint8([zh.to(dev, non_blocking=True)], 0)[0]
        e2e_v = time.time() - tt0
        ref_fl, ex_fl, by, _ = wan_vae_work(T, H, W)
        result["vae_decode"] = {"metric": "vae_decode_frames_per_sec", "value": world * nfr / (vms / 1000.0), "unit": "frames/s",
                                "frames": nfr, "resolution": [8 * H, 8 * W], "ms_per_clip": vms,
                                "gpu_launches": (_lib.launch_count() - l0) // reps,
                                "finite": bool(torch.isfinite(fr).all()),
                                "roofline": {"bound": "tensor", "why": f"AI = {ex_fl / by:.0f} FLOP/B >> ridge {pk['tensor_burst'] * 1e12 / (pk['hbm'] * 1e9):.0f}: even with every norm fused away the convolutions are tensor-bound; HBM is the roof only of the un-fused norm/SiLU passes",
                                             "reference_flops": ref_fl, "executed_flops": ex_fl, "bytes_algorithmic": by,
                                             "achieved_tflops": ex_fl / (vms * 1e-3) / 1e12, "achieved_tflops_on_reference_flops": ref_fl / (vms * 1e-3) / 1e12,
                                             "frac_of_burst": ex_fl / (vms * 1e-3) / 1e12 / pk["tensor_burst"],
                                             "frac_of_sustained": ex_fl / (vms * 1e-3) / 1e12 / pk["tensor_sustained"],
                                             "achieved_gbs": by / (vms * 1e-3) / 1e9, "hbm_frac": by / (vms * 1e-3) / 1e9 / pk["hbm"],
                                             "peak_source": pk["source"]},
                                "e2e": {"value": world * nfr / e2e_v, "unit": "frames/s", "h2d_bytes": zh.numel() * 4, "d2h_bytes": u8.numel()}}
        # VAE encode of the same clip size (SURVEY.md 8f.2: every i2v generation encodes its conditioning frames), device-resident video
        if with_encode:
            try:
                vid = (torch.rand(3, nfr, 8 * H, 8 * W, generator=g) * 2 - 1).to(dev)
                vae.encode([vid], tile_size=0)
                barrier()
                l1 = _lib.launch_count()
                q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                q0.record()
                mu = vae.encode([vid], tile_size=0)[0]
                q1.record()
                barrier()
                if outputs is not None:
                    outputs["vae_encode_latents"] = dump_sample(mu, "vae_encode_latents")
                ems = torch.tensor([q0.elapsed_time(q1)], device=dev, dtype=torch.float64)
                if dist is not None:
                    dist.all_reduce(ems, op=dist.ReduceOp.MAX)
                result["vae_encode"] = {"metric": "vae_encode_frames_per_sec", "value": world * nfr / (float(ems[0]) / 1e3), "unit": "frames/s",
                                        "frames": nfr, "resolution": [8 * H, 8 * W], "ms_per_clip": float(ems[0]),
                                        "gpu_launches": _lib.launch_count() - l1, "latent": list(mu.shape), "finite": bool(torch.isfinite(mu).all())}
                del vid, mu
            except Exception as e:                                   # noqa: BLE001
                result["vae_encode"] = {"error": repr(e)[:300]}
        if dist is not None:
            # the single collective of the north star: all-gather of the decoded uint8 frames over NVLink.
            # (a) baseline: frames_to_u8 kernel + ncclAllGather; (b) fused quantise + all-gather over peer memory -- the path
            # dist.generate_batch takes (FusedFrameGather)
            gathered = [torch.empty_like(u8, device=dev) for _ in range(world)]
            u8d = torch.empty(fr.shape, device=dev, dtype=torch.uint8)
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            g0.record()
            _lib.call("b200_frames_to_u8", fr.data_ptr(), u8d.data_ptr(), fr.numel(), torch.cuda.current_stream().cuda_stream)
            dist.all_gather(gathered, u8d)
            g1.record()
            barrier()
            result["vae_decode"]["u8_plus_nccl_allgather_ms"] = g0.elapsed_time(g1)
            result["vae_decode"]["allgather_bytes"] = u8.numel() * world
            try:
                from wan2gp_b200 import dist as wdist
                fg = wdist.FusedFrameGather(fr.numel(), dev)
                fg.gather(fr)
                barrier()
                g0.record()
                allf = fg.gather(fr)
                g1.record()
                barrier()
                result["vae_decode"]["fused_u8_allgather_ms"] = g0.elapsed_time(g1)
                result["vae_decode"]["fused_matches_nccl"] = bool(all(torch.equal(allf[r], gathered[r].reshape(-1)) for r in range(world)))
                del fg, allf
            except Exception as e:           # symmetric memory unavailable on this box: the NCCL path above stands
                result["vae_decode"]["fused_u8_allgather_error"] = repr(e)[:200]
            del gathered, u8d
        del vae, z, fr
    else:
        del den, model, model2
    torch.cuda.empty_cache()
    return result, cfg, thw


def write_outputs(out_dir, outputs):
    if not out_dir:
        return
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="wan22_t2v_14b_720p81", choices=list(WORKLOADS))
    ap.add_argument("--no-vae", action="store_true")
    ap.add_argument("--cfg-split", action="store_true", help="split each CFG pair over 2 GPUs (one 19 MB exchange per step)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-subruns", action="store_true", help="skip the short configs[2] / configs[3] sub-runs appended at N >= 2 / N = 4")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the run, write what rank 0's timed steps (and timed VAE decode / encode) "
                    "computed as DIR/<name>.npy, float32; outputs over 5 M elements as a fixed sample of 5 M")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")

    from wan2gp_b200 import synth
    cfg_name, thw, two_experts, desc = WORKLOADS[args.workload]
    rank, world, local_rank = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if args.workload.startswith("hy1"):
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "CPU arm is implemented for the Wan workloads only"}))
            return
        torch.cuda.set_device(local_rank)
        dev = torch.device("cuda", local_rank)
        dist = None
        if world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=dev)
        outputs = {} if args.dump_outputs and rank == 0 else None
        res = measure_hunyuan(args.workload, args.steps, args.warmup, rank, world, local_rank, dev, dist, with_vae=not args.no_vae and not args.cfg_split,
                              cfg_split=args.cfg_split, outputs=outputs)
        if rank == 0:
            write_outputs(args.dump_outputs, outputs)
            print(json.dumps(res))
        if dist is not None:
            dist.destroy_process_group()
        return

    if args.impl == "reference":
        # CPU arm: rank 0 only; other ranks exit without work.  The bounded sample is timed min(steps, 3) times (min / median
        # reported), not once per requested step: --steps 20 must not turn into 20 repetitions of the same 30 s sample.
        if rank != 0:
            return
        cfg = synth.WAN_CONFIGS[cfg_name]
        T, H, W = thw
        reps = max(1, min(args.steps, 3))
        v, info = cpu_port_steps_per_sec(cfg, thw, reps=reps)
        config = {"workload": args.workload, "description": desc, "latent": [1, 16, T, H, W], "tokens": T * (H // 2) * (W // 2),
                  "context": [1, cfg["text_len"], cfg["text_dim"]], "cfg_pair": True}
        print(json.dumps({"impl": "reference", "metric": "denoise_steps_per_sec", "value": v, "unit": "steps/s", "n_gpus": args.gpus,
                          "steps": args.steps, "warmup": args.warmup, "steps_timed": reps, "ms_per_step": 1000.0 / v, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                          "cpu_baseline": dict({"value": v, "unit": "steps/s", "kind": "port"}, **info),
                          "e2e": {"value": v, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    outputs = {} if args.dump_outputs and rank == 0 else None

    result, cfg, thw = measure_wan(args.workload, args.steps, args.warmup, rank, world, local_rank, dev, dist, cfg_split=args.cfg_split,
                                   with_vae=not args.no_vae, outputs=outputs)
    if rank == 0:
        write_outputs(args.dump_outputs, outputs)

    # ---- BASELINE configs[2] / configs[3] in front of the driver: short sub-runs appended to the same JSON line
    if world >= 2 and world % 2 == 0 and not args.no_subruns and not args.cfg_split and args.workload == "wan22_t2v_14b_720p81":
        try:
            sub, _, _ = measure_wan("wan22_i2v_14b_720p81", 3, 2, rank, world, local_rank, dev, dist, cfg_split=True, with_vae=False,
                                    with_parity=False, e2e_steps=1)
            result["cfg_split"] = {k: sub[k] for k in ("metric", "value", "unit", "ms_per_step", "steps", "warmup", "config", "gpu_launches", "finite",
                                                       "model_tflops", "roofline", "clocks", "e2e")}
            result["cfg_split"]["note"] = "BASELINE configs[2]: Wan2.2 i2v 14B 720p x 81f, every CFG pair split over 2 GPUs; value = samples in flight x steps/s"
        except Exception as e:                                   # noqa: BLE001
            result["cfg_split"] = {"error": repr(e)[:300]}
        if world == 4 or os.environ.get("B200_BENCH_FORCE_HY15"):       # the env switch only exists to exercise this branch on 2 GPUs
            try:
                result["hy15_t2v_720p129"] = measure_hunyuan("hy15_t2v_720p129", 2, 1, rank, world, local_rank, dev, dist, with_vae=False)
                result["hy15_t2v_720p129"]["note"] = "BASELINE configs[3]: Hunyuan Video 1.5 t2v 720p x 129f on 4 GPUs (one sample per GPU)"
            except Exception as e:                               # noqa: BLE001
                result["hy15_t2v_720p129"] = {"error": repr(e)[:300]}
            if os.environ.get("B200_BENCH_HY15_SPLIT", "1") != "0":
                try:                                             # the same configuration as 2 samples x 2 CFG branches: half the step latency
                    sub = measure_hunyuan("hy15_t2v_720p129", 2, 1, rank, world, local_rank, dev, dist, with_vae=False, cfg_split=True)
                    result["hy15_t2v_720p129_cfg_split"] = {k: sub[k] for k in ("metric", "value", "unit", "ms_per_step", "steps", "warmup", "config",
                                                                                 "gpu_launches", "finite", "model_tflops", "e2e", "clocks") if k in sub}
                    result["hy15_t2v_720p129_cfg_split"]["note"] = ("BASELINE configs[3] with every CFG pair split over 2 GPUs; value = samples in flight x "
                                                                    "steps/s; the step latency of one sample is ms_per_step")
                except Exception as e:                           # noqa: BLE001
                    result["hy15_t2v_720p129_cfg_split"] = {"error": repr(e)[:300]}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, info = cpu_port_steps_per_sec(cfg, thw)
        result["cpu_baseline"] = dict({"value": v, "unit": "steps/s", "kind": "port"}, **info)
    if rank == 0:
        print(json.dumps(result))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
