"""Generate tests/golden/*.npz by running the UNMODIFIED reference modules
(imported from /root/reference through oracle/refshim.py) on seeded synthetic
weights and inputs (wan2gp_b200/synth.py).  Run in the build container only:

    python oracle/gen_golden.py [tiny] [tiny_i2v] [p13b] [vae_tiny] [vae_p]

The fixtures travel to the GPU box; /root/reference does not.
"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.refshim import Pipe, load_reference  # noqa: E402
from wan2gp_b200 import synth  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")

WAN_CASES = {
    # name: (config, latent (T,H,W), seed)
    "tiny": ("tiny", (3, 8, 12), 0),
    "tiny_i2v": ("tiny_i2v", (2, 8, 8), 1),
    "small": ("small", (5, 16, 24), 2),
    "p13b": ("t2v_1.3B", (9, 30, 52), 0),     # BASELINE config 1 (shared/mps/test_mps_forward.py:75-110)
}
VAE_CASES = {
    "vae_tiny": (synth.VAE_CFG_TINY, (16, 3, 6, 8), 0),
    "vae_small": (synth.VAE_CFG, (16, 5, 8, 10), 1),
    "vae_p": (synth.VAE_CFG, (16, 3, 30, 52), 0),  # BASELINE.md section 2 decode probe shape
}


def build_reference_wan(cfg_name, seed):
    ref = load_reference()
    cfg = synth.WAN_CONFIGS[cfg_name]
    model = ref.WanModel(**cfg).eval().requires_grad_(False)
    sd = synth.make_wan_state_dict(cfg, seed)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    assert not missing, missing
    model.apply_post_init_changes()        # required before forward (model.py:1291-1303)
    return ref, model, cfg, sd


def run_wan(name):
    cfg_name, thw, seed = WAN_CASES[name]
    ref, model, cfg, sd = build_reference_wan(cfg_name, seed)
    x, t, ctx, y = synth.make_wan_inputs(cfg, thw, seed)
    freqs = ref.get_rotary_pos_embed(thw)
    t0 = time.time()
    with torch.no_grad():
        out = model([x.clone()], t, [ctx], y=y, freqs=freqs, pipeline=Pipe())[0]
    dt = time.time() - t0
    print(f"{name}: reference fp32 forward {dt:.2f}s out {tuple(out.shape)} absmean {out.abs().mean():.6f}")
    # float64 run: WanRMSNorm's `y = x.float()` (model.py:165) only COPIES when x is not fp32, so this
    # run has the production (bf16/GPU) RMSNorm semantics without the fp32 aliasing artefact.
    model.double()
    with torch.no_grad():
        out64 = model([x.double()], t.double(), [ctx.double()], y=None if y is None else y.double(),
                      freqs=freqs, pipeline=Pipe())[0]
    print(f"{name}: reference fp64 forward absmean {out64.abs().mean():.6f} "
          f"fp32-vs-fp64 rel {((out - out64).norm() / out64.norm()).item():.3e}")
    np.savez_compressed(os.path.join(GOLDEN, f"wan_{name}.npz"),
                        out=out.numpy().astype(np.float32), out64=out64.numpy().astype(np.float32),
                        cos=freqs[0][:64].numpy(), sin=freqs[1][:64].numpy(),
                        seconds=np.float32(dt), threads=np.int32(torch.get_num_threads()))


def run_vae(name):
    ref = load_reference()
    cfg, zshape, seed = VAE_CASES[name]
    vae = ref.WanVAE_(dim=cfg["dim"], z_dim=cfg["z_dim"], dim_mult=cfg["dim_mult"],
                      num_res_blocks=cfg["num_res_blocks"], attn_scales=[],
                      temperal_downsample=[False, True, True], dropout=0.0).eval().requires_grad_(False)
    sd = synth.make_vae_state_dict(cfg, seed)
    full = vae.state_dict()
    for k in full:
        if k in sd:
            full[k] = sd[k]
    vae.load_state_dict(full)
    z = synth._normal((1,) + zshape, 1.0, seed, "input.z", "cpu")
    scale = [torch.tensor(synth.VAE_MEAN), 1.0 / torch.tensor(synth.VAE_STD)]
    t0 = time.time()
    with torch.no_grad():
        out = vae.decode(z, scale)
    dt = time.time() - t0
    print(f"{name}: reference decode {dt:.2f}s out {tuple(out.shape)} absmean {out.abs().mean():.6f} "
          f"min {out.min():.3f} max {out.max():.3f}")
    np.savez_compressed(os.path.join(GOLDEN, f"{name}.npz"), out=out.numpy().astype(np.float16 if out.numel() > 2_000_000 else np.float32),
                        seconds=np.float32(dt), threads=np.int32(torch.get_num_threads()))


VAE_ENC_CASES = {"vae_enc_tiny": (synth.VAE_CFG_TINY, (3, 9, 32, 48), 0), "vae_enc_small": (synth.VAE_CFG, (3, 5, 48, 64), 1),
                 "vae_enc_1f": (synth.VAE_CFG_TINY, (3, 1, 16, 24), 2)}


def run_vae_enc(name):
    """Reference WanVAE_.encode (vae.py:586-625: chunked 1,4,4,... with feature caches), un-tiled."""
    ref = load_reference()
    cfg, xshape, seed = VAE_ENC_CASES[name]
    vae = ref.WanVAE_(dim=cfg["dim"], z_dim=cfg["z_dim"], dim_mult=cfg["dim_mult"], num_res_blocks=cfg["num_res_blocks"], attn_scales=[],
                      temperal_downsample=[False, True, True], dropout=0.0).eval().requires_grad_(False)
    sd = synth.make_vae_state_dict(cfg, seed, encoder=True)
    assert set(sd) == set(vae.state_dict()), set(sd) ^ set(vae.state_dict())
    vae.load_state_dict(sd)
    x = synth._normal((1,) + xshape, 0.5, seed, "input.video", "cpu").clamp_(-1, 1)
    scale = [torch.tensor(synth.VAE_MEAN), 1.0 / torch.tensor(synth.VAE_STD)]
    with torch.no_grad():
        mu = vae.encode(x, scale)
    print(f"{name}: reference encode out {tuple(mu.shape)} absmean {mu.abs().mean():.6f}")
    np.savez_compressed(os.path.join(GOLDEN, f"{name}.npz"), out=mu.numpy().astype(np.float32))


HY_CASES = {"hy_tiny": ("hy_tiny", (3, 6, 10), 0), "hy10_tiny": ("hy10_tiny", (2, 8, 12), 1),
            "hy_tiny_i2v": ("hy_tiny_i2v", (3, 6, 10), 2)}          # hunyuan_1_5_i2v: latent_concat + projected image-encoder tokens


def run_hy(name):
    from oracle.refshim import hook_linear_input_cast, load_reference_hy
    hy = load_reference_hy()
    cfg_name, thw, seed = HY_CASES[name]
    cfg = synth.HY_CONFIGS[cfg_name]
    v10 = cfg.get("family") == "1.0"
    kw = dict(hy.CONFIGS["HYVideo-T/2-cfgdistill" if v10 else "HYVideo-1_5"])
    kw.update({k: cfg[k] for k in ("hidden_size", "heads_num", "mlp_width_ratio", "mm_double_blocks_depth", "text_states_dim")})
    if v10:
        kw.update(mm_single_blocks_depth=cfg["mm_single_blocks_depth"], text_states_dim_2=cfg["text_states_dim_2"])
    i2v = "vision_states_dim" in cfg
    if i2v:
        kw.update(vision_states_dim=cfg["vision_states_dim"])
    model = hy.HYVideoDiffusionTransformer(i2v_condition_type="latent_concat" if i2v else None, in_channels=cfg["in_channels"],
                                           out_channels=cfg["out_channels"], **kw)
    model = model.eval().requires_grad_(False)
    sd = synth.make_hy_state_dict(cfg, seed)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and all(m.startswith("vision_in") for m in missing), (missing, unexpected)
    model.cache = None
    if v10:
        # hunyuan_handler.py:274-278: mmgp splits img_attn_qkv / linear1 into per-projection Linears at load time
        from models.hyvideo.modules.models import get_linear_split_map
        from oracle.refshim import split_linear_modules
        split_linear_modules(model, get_linear_split_map())
    hook_linear_input_cast(model)         # fp32 weights + the reference's own bf16 hard-casts (see oracle/hy_oracle.py)
    x, t, txt, tm, b5, bm = synth.make_hy_inputs(cfg, thw, seed=seed)
    P = cfg["patch_size"][1]
    cos, sin = hy.get_nd_rotary_pos_embed(cfg["rope_dim_list"], [thw[0], thw[1] // P, thw[2] // P], theta=256, use_real=True,
                                             theta_rescale_factor=1, enable_riflex=False)   # hunyuan.py:716-724
    extra = {}
    if v10:
        extra = dict(text_states_2=synth._normal((1, cfg["text_states_dim_2"]), 1.0, seed, "hy.txt2", "cpu"),
                     guidance=torch.tensor([6000.0]))
    else:
        extra = dict(byt5_text_states=b5, byt5_text_mask=bm)
        if i2v:
            extra["vision_states"] = synth.make_hy_vision_states(cfg, seed=seed)
    with torch.no_grad():
        out = model(x, t, text_states=txt, text_mask=tm, freqs_cos=cos, freqs_sin=sin, pipeline=Pipe(), **extra)
    print(f"{name}: reference HY forward out {tuple(out.shape)} {out.dtype} absmean {out.float().abs().mean():.6f}")
    np.savez_compressed(os.path.join(GOLDEN, f"{name}.npz"), out=out.float().numpy(), cos=cos[:64].numpy(), sin=sin[:64].numpy())


HYVAE_CASES = {"hyvae_tiny": ("hyvae_tiny", (8, 3, 4, 6), 0), "hyvae_small": ("hyvae_small", (16, 3, 2, 3), 1)}


def run_hyvae(name):
    from oracle.refshim import load_reference_hyvae
    hv = load_reference_hyvae()
    cfg_name, zshape, seed = HYVAE_CASES[name]
    cfg = synth.HYVAE_CONFIGS[cfg_name]
    dec = hv.Decoder(**cfg).eval().requires_grad_(False)
    dec.load_state_dict(synth.make_hyvae_state_dict(cfg, seed))
    z = synth._normal((1,) + zshape, 1.0, seed, "input.z", "cpu")
    with torch.no_grad():
        out = dec(z)
    print(f"{name}: reference HY-1.5 VAE Decoder out {tuple(out.shape)} absmean {out.abs().mean():.6f}")
    np.savez_compressed(os.path.join(GOLDEN, f"{name}.npz"), out=out.numpy().astype(np.float32))


HYVAE10_CASES = {"hyvae10_tiny": ("hyvae10_tiny", (8, 3, 2, 3), 0), "hyvae10_small": ("hyvae10_small", (16, 2, 2, 2), 1)}


def run_hyvae10(name):
    """Reference AutoencoderKLCausal3D.decode, un-tiled (autoencoder_kl_causal_3d.py:474-493); the mid-block `Attention` is the
    restated third-party class of refshim.load_reference_hyvae10."""
    from oracle.refshim import load_reference_hyvae10
    hv = load_reference_hyvae10()
    cfg_name, zshape, seed = HYVAE10_CASES[name]
    cfg = synth.HYVAE10_CONFIGS[cfg_name]
    vae = hv.AutoencoderKLCausal3D(in_channels=3, down_block_types=("DownEncoderBlockCausal3D",) * 4,
                                   up_block_types=("UpDecoderBlockCausal3D",) * 4, **cfg).eval().requires_grad_(False)
    missing = vae.load_state_dict(synth.make_hyvae10_state_dict(cfg, seed), strict=False)
    assert not missing.unexpected_keys and all(k.startswith(("encoder.", "quant_conv.")) for k in missing.missing_keys)
    z = synth._normal((1,) + zshape, 1.0, seed, "input.z", "cpu")
    with torch.no_grad():
        out = vae.decode(z, return_dict=False)[0]
    print(f"{name}: reference HY-1.0 VAE decode out {tuple(out.shape)} absmean {out.abs().mean():.6f}")
    np.savez_compressed(os.path.join(GOLDEN, f"{name}.npz"), out=out.numpy().astype(np.float32))


TILED_CASES = {"vae_tiled_dec": ("dec", (16, 2, 12, 14), 64, 4), "vae_tiled_enc": ("enc", (3, 5, 96, 112), 64, 5)}


def run_vae_tiled(name):
    """Reference WanVAE_.spatial_tiled_decode / spatial_tiled_encode (vae.py:676-723, 841-881) and the streaming tiled uint8 writer
    decode_to_cpu_uint8 (:741-839) on the tiny config."""
    ref = load_reference()
    kind, shape, tile, seed = TILED_CASES[name]
    cfg = synth.VAE_CFG_TINY
    vae = ref.WanVAE_(dim=cfg["dim"], z_dim=cfg["z_dim"], dim_mult=cfg["dim_mult"], num_res_blocks=cfg["num_res_blocks"], attn_scales=[],
                      temperal_downsample=[False, True, True], dropout=0.0).eval().requires_grad_(False)
    vae.load_state_dict(synth.make_vae_state_dict(cfg, seed, encoder=True))
    scale = [torch.tensor(synth.VAE_MEAN), 1.0 / torch.tensor(synth.VAE_STD)]
    with torch.no_grad():
        if kind == "dec":
            z = synth._normal((1,) + shape, 1.0, seed, "input.z", "cpu")
            out = vae.spatial_tiled_decode(z.clone(), scale, tile)
            # decode_to_cpu_uint8 un-normalises each latent tile IN PLACE on `latent_source[...].to(device, dtype)` (vae.py:796-799); on a
            # GPU the latents were moved to the CPU first (:746-747) so .to() copies, but in this all-CPU fp32 run .to() returns the
            # VIEW and overlapping tiles would be un-normalised twice.  Feeding fp64 latents with _model_dtype = fp32 restores the copy
            # (= the production behaviour) without touching reference code.
            vae._model_dtype = torch.float32
            u8 = vae.decode_to_cpu_uint8(z.double(), scale, tile_size=tile)
            np.savez_compressed(os.path.join(GOLDEN, f"{name}.npz"), out=out.numpy().astype(np.float32), u8=u8.numpy(), tile=tile)
        else:
            x = synth._normal((1,) + shape, 0.5, seed, "input.video", "cpu").clamp_(-1, 1)
            out = vae.spatial_tiled_encode(x, scale, tile)
            np.savez_compressed(os.path.join(GOLDEN, f"{name}.npz"), out=out.numpy().astype(np.float32), tile=tile)
    print(f"{name}: reference tiled {kind} out {tuple(out.shape)} absmean {out.abs().mean():.6f}")


HYVAE_ENC_CASES = {"hyvae_enc_tiny": ("hyvae_tiny", (3, 5, 16, 24), 2), "hyvae_enc_small": ("hyvae_small", (3, 5, 32, 48), 3)}


def run_hyvae_enc(name):
    """Reference Hunyuan 1.5 VAE Encoder (hunyuanvideo_15_vae.py:342-430) = AutoencoderKLConv3D.encode with tiling off (:866-887)."""
    from oracle.refshim import load_reference_hyvae
    hv = load_reference_hyvae()
    cfg_name, xshape, seed = HYVAE_ENC_CASES[name]
    cfg = synth.HYVAE_CONFIGS[cfg_name]
    enc = hv.Encoder(in_channels=3, z_channels=cfg["z_channels"], block_out_channels=list(reversed(cfg["block_out_channels"])),
                     num_res_blocks=cfg["num_res_blocks"], ffactor_spatial=cfg["ffactor_spatial"], ffactor_temporal=cfg["ffactor_temporal"]).eval().requires_grad_(False)
    enc.load_state_dict(synth.make_hyvae_state_dict(cfg, seed, encoder=True))
    x = synth._normal((1,) + xshape, 0.5, seed, "input.video", "cpu").clamp_(-1, 1)
    with torch.no_grad():
        out = enc(x)
    print(f"{name}: reference HY-1.5 VAE Encoder out {tuple(out.shape)} absmean {out.abs().mean():.6f}")
    np.savez_compressed(os.path.join(GOLDEN, f"{name}.npz"), out=out.numpy().astype(np.float32))


HYVAE10_ENC_CASES = {"hyvae10_enc_tiny": ("hyvae10_tiny", (3, 5, 16, 24), 2), "hyvae10_enc_small": ("hyvae10_small", (3, 9, 16, 16), 3)}


def run_hyvae10_enc(name):
    """Reference AutoencoderKLCausal3D.encode, un-tiled (autoencoder_kl_causal_3d.py:435-472): encoder -> quant_conv -> moments."""
    from oracle.refshim import load_reference_hyvae10
    hv = load_reference_hyvae10()
    cfg_name, xshape, seed = HYVAE10_ENC_CASES[name]
    cfg = synth.HYVAE10_CONFIGS[cfg_name]
    vae = hv.AutoencoderKLCausal3D(in_channels=3, down_block_types=("DownEncoderBlockCausal3D",) * 4,
                                   up_block_types=("UpDecoderBlockCausal3D",) * 4, **cfg).eval().requires_grad_(False)
    sd = synth.make_hyvae10_state_dict(cfg, seed, encoder=True)
    assert set(sd) == set(vae.state_dict()), set(sd) ^ set(vae.state_dict())
    vae.load_state_dict(sd)
    x = synth._normal((1,) + xshape, 0.5, seed, "input.video", "cpu").clamp_(-1, 1)
    with torch.no_grad():
        out = vae.encode(x, return_dict=False)[0].parameters
    print(f"{name}: reference HY-1.0 VAE encode moments {tuple(out.shape)} absmean {out.abs().mean():.6f}")
    np.savez_compressed(os.path.join(GOLDEN, f"{name}.npz"), out=out.numpy().astype(np.float32))


HY_TILED_CASES = {"hyvae_tiled": ("1.5", "hyvae_tiny", (8, 7, 6, 10), 16, 8, 6), "hyvae10_tiled": ("1.0", "hyvae10_tiny", (8, 7, 5, 7), 32, 16, 7)}


def run_hy_tiled(name):
    """Reference Hunyuan VAE decode with enable_tiling() (what the pipelines always do: hunyuan.py:772, pipeline_hunyuan_video.py:695),
    small tile sizes so the tiny clip is cut into several temporal and spatial tiles."""
    from oracle.refshim import load_reference_hy, load_reference_hyvae, load_reference_hyvae10
    import importlib
    fam, cfg_name, zshape, sample_size, sample_tsize, seed = HY_TILED_CASES[name]
    if fam == "1.5":
        load_reference_hy(), load_reference_hyvae()
        m = importlib.import_module("models.hyvideo.vae.hunyuanvideo_15_vae")
        cfg = synth.HYVAE_CONFIGS[cfg_name]
        vae = m.AutoencoderKLConv3D(in_channels=3, out_channels=3, latent_channels=cfg["z_channels"], block_out_channels=tuple(reversed(cfg["block_out_channels"])),
                                    layers_per_block=cfg["num_res_blocks"], ffactor_spatial=cfg["ffactor_spatial"], ffactor_temporal=cfg["ffactor_temporal"],
                                    sample_size=sample_size, sample_tsize=sample_tsize).eval().requires_grad_(False)
        vae.decoder.load_state_dict(synth.make_hyvae_state_dict(cfg, seed))
    else:
        hv = load_reference_hyvae10()
        cfg = synth.HYVAE10_CONFIGS[cfg_name]
        vae = hv.AutoencoderKLCausal3D(in_channels=3, down_block_types=("DownEncoderBlockCausal3D",) * 4, up_block_types=("UpDecoderBlockCausal3D",) * 4,
                                       sample_size=sample_size, sample_tsize=sample_tsize, **cfg).eval().requires_grad_(False)
        vae.load_state_dict(synth.make_hyvae10_state_dict(cfg, seed, encoder=True))
    if fam == "1.5":
        vae.encoder.load_state_dict(synth.make_hyvae_state_dict(cfg, seed, encoder=True))
    vae.enable_tiling()
    z = synth._normal((1,) + zshape, 1.0, seed, "input.z", "cpu")
    fs, ft = (cfg["ffactor_spatial"], cfg["ffactor_temporal"]) if fam == "1.5" else (8, 4)
    xv = synth._normal((1, 3, ft * (zshape[1] - 1) + 1, fs * zshape[2], fs * zshape[3]), 0.5, seed, "input.video", "cpu").clamp_(-1, 1)
    with torch.no_grad():
        out = vae.decode(z, return_dict=False)[0]
        enc = vae.encode(xv, return_dict=False)[0].parameters          # moments of the tiled encode of a clip of the decoded size
    print(f"{name}: reference tiled decode out {tuple(out.shape)} absmean {out.abs().mean():.6f}; latent tile {vae.tile_latent_min_size} x {vae.tile_latent_min_tsize}")
    np.savez_compressed(os.path.join(GOLDEN, f"{name}.npz"), out=out.numpy().astype(np.float32), enc=enc.numpy().astype(np.float32),
                        sample_size=sample_size, sample_tsize=sample_tsize, lat_size=vae.tile_latent_min_size, lat_tsize=vae.tile_latent_min_tsize)


def run_unipc(name):
    """Trajectory of the reference FlowUniPCMultistepScheduler on seeded fp64 inputs (same generator as tests/test_unipc_cpu.py)."""
    from oracle.refshim import load_reference_unipc
    steps, shift = 20, 3.0
    ref = load_reference_unipc().FlowUniPCMultistepScheduler(num_train_timesteps=1000, shift=1, use_dynamic_shifting=False)
    ref.set_timesteps(steps, device="cpu", shift=shift)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, 4, 2, 3, 5, generator=g, dtype=torch.float64)
    vs = [torch.randn(1, 4, 2, 3, 5, generator=g, dtype=torch.float64) for _ in range(steps)]
    traj = []
    for i, t in enumerate(ref.timesteps):
        x = ref.step(vs[i], t, x, return_dict=False)[0]
        traj.append(x.numpy().copy())
    np.savez_compressed(os.path.join(GOLDEN, "unipc.npz"), steps=steps, shift=shift, timesteps=ref.timesteps.numpy(), traj=np.stack(traj))
    print(f"unipc: {steps} steps, final absmean {np.abs(traj[-1]).mean():.6f}")
    # dpm++ (any2video.py:523-532): FlowDPMSolverMultistepScheduler fed with get_sampling_sigmas through retrieve_timesteps
    R = load_reference_unipc()
    ref = R.FlowDPMSolverMultistepScheduler(num_train_timesteps=1000, shift=1, use_dynamic_shifting=False)
    ts, _ = R.retrieve_timesteps(ref, device="cpu", sigmas=R.get_sampling_sigmas(steps, shift))
    g = torch.Generator().manual_seed(0)
    x = torch.randn(1, 4, 2, 3, 5, generator=g, dtype=torch.float64)
    traj = []
    for i, t in enumerate(ts):
        x = ref.step(torch.randn(1, 4, 2, 3, 5, generator=g, dtype=torch.float64), t, x, return_dict=False)[0]
        traj.append(x.numpy().copy())
    np.savez_compressed(os.path.join(GOLDEN, "dpmpp.npz"), steps=steps, shift=shift, timesteps=ts.numpy(), traj=np.stack(traj))
    print(f"dpm++: {steps} steps, final absmean {np.abs(traj[-1]).mean():.6f}")


def run_schedulers(name):
    """Every reference scheduler run that tests/test_unipc_cpu.py compares with, on that module's cases and seeded inputs:
    FlowUniPCMultistepScheduler and FlowDPMSolverMultistepScheduler (timesteps, sigmas, whole trajectories), LCMScheduler,
    FlowMatchScheduler, Wan's EulerScheduler and Hunyuan's FlowMatchDiscreteScheduler (timesteps and final samples)."""
    import importlib.util
    from oracle.refshim import REFERENCE_ROOT, load_reference_unipc
    from tests.test_unipc_cpu import CASES, inputs
    R = load_reference_unipc()
    out = {}
    for steps, shift in CASES:
        key = f"{steps}_{shift:g}"
        ref = R.FlowUniPCMultistepScheduler(num_train_timesteps=1000, shift=1, use_dynamic_shifting=False)
        ref.set_timesteps(steps, device="cpu", shift=shift)                      # any2video.py:519-520
        x, vs = inputs(steps)
        traj = []
        for i, t in enumerate(ref.timesteps):
            x = ref.step(vs[i], t, x, return_dict=False)[0]
            traj.append(x.numpy().copy())
        out.update({f"unipc_{key}_timesteps": ref.timesteps.numpy(), f"unipc_{key}_sigmas": ref.sigmas.numpy(), f"unipc_{key}_traj": np.stack(traj)})
        ref = R.FlowDPMSolverMultistepScheduler(num_train_timesteps=1000, shift=1, use_dynamic_shifting=False)
        ts, _ = R.retrieve_timesteps(ref, device="cpu", sigmas=R.get_sampling_sigmas(steps, shift))
        x, vs = inputs(steps)
        traj = []
        for i, t in enumerate(ts):
            x = ref.step(vs[i], t, x, return_dict=False)[0]
            traj.append(x.numpy().copy())
        out.update({f"dpmpp_{key}_timesteps": ts.numpy(), f"dpmpp_{key}_traj": np.stack(traj)})
    for steps, shift in ((4, 5.0), (8, 3.0), (12, 7.0)):
        ref = R.LCMScheduler(num_train_timesteps=1000, num_inference_steps=min(steps, 8), shift=shift)
        ref.set_timesteps(min(steps, 8), device="cpu", shift=shift)
        x, vs = inputs(len(ref.timesteps))
        x = x.float()
        for i, t in enumerate(ref.timesteps):
            x = ref.step(vs[i].float(), t, x).prev_sample
        out.update({f"lcm_{steps}_{shift:g}_timesteps": ref.timesteps.numpy(), f"lcm_{steps}_{shift:g}_out": x.numpy()})
    for steps in (4, 9):
        ref = R.FlowMatchScheduler(num_inference_steps=steps, shift=5.0, sigma_min=0, extra_one_step=True)
        ref.timesteps = torch.tensor([1000, 934, 862, 756, 603, 410, 250, 140, 74])[:steps]
        ref.sigmas = torch.cat([ref.timesteps / 1000, torch.tensor([0.])])
        x, vs = inputs(steps)
        x = x.float()
        for i, t in enumerate(ref.timesteps):
            x = ref.step(vs[i].float(), t, x)[0]
        out[f"causvid_{steps}_out"] = x.numpy()
    # Wan EulerScheduler (shared/utils/euler_scheduler.py: no third-party imports, loaded straight from the reference tree)
    spec = importlib.util.spec_from_file_location("_ref_euler", os.path.join(REFERENCE_ROOT, "shared/utils/euler_scheduler.py"))
    em = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(em)
    for steps, shift in ((50, 12.0), (20, 5.0), (1, 3.0)):
        ref = em.EulerScheduler(num_train_timesteps=1000, use_timestep_transform=True)
        rts = ref.set_timesteps(steps, device=None, shift=shift)
        x, vs = inputs(steps)
        for i, t in enumerate(rts):
            x = ref.step(vs[i], t, x, return_dict=False)[0]
        out.update({f"euler_{steps}_{shift:g}_timesteps": rts.numpy(), f"euler_{steps}_{shift:g}_out": x.numpy()})
    for steps, shift in ((30, 7.0), (50, 9.0), (4, 6.0)):
        ref = R.FlowMatchDiscreteScheduler(shift=shift, reverse=True, solver="euler")
        ref.set_timesteps(steps, device="cpu")
        x, vs = inputs(steps)
        x = x.float()
        for i, t in enumerate(ref.timesteps):
            x = ref.step(vs[i].float(), t, x, return_dict=False)[0]
        out.update({f"flow_match_{steps}_{shift:g}_timesteps": ref.timesteps.numpy(), f"flow_match_{steps}_{shift:g}_out": x.numpy()})
    np.savez_compressed(os.path.join(GOLDEN, f"{name}.npz"), **out)
    print(f"{name}: {len(out)} arrays, {sum(v.nbytes for v in out.values())} bytes")


def run_t5(name):
    """Reference T5Encoder (umT5 layout: per-layer relative position embedding) on seeded ids with a padded tail, fp32, eval mode."""
    from oracle.refshim import load_reference_t5
    from wan2gp_b200 import synth
    cfg = synth.T5_CONFIGS[name]
    R = load_reference_t5()
    enc = R.T5Encoder(cfg["vocab_size"], cfg["dim"], cfg["dim_attn"], cfg["dim_ffn"], cfg["num_heads"], cfg["num_layers"], cfg["num_buckets"],
                      shared_pos=False, dropout=0.1).eval().float()
    sd = synth.make_t5_state_dict(cfg, seed=0)
    missing, unexpected = enc.load_state_dict(sd, strict=True), None
    length, n_valid = 40, 29
    ids, mask = synth.make_t5_inputs(cfg, length, n_valid, seed=0)
    with torch.no_grad():
        out = enc(ids[None], mask[None])[0]
    print(f"{name}: reference T5Encoder out {tuple(out.shape)} absmean {out.abs().mean():.6f}")
    np.savez_compressed(os.path.join(GOLDEN, f"{name}.npz"), out=out.numpy().astype(np.float32), length=length, n_valid=n_valid, seed=0)


def run_byt5(name):
    """The byT5 glyph encoder of Hunyuan Video 1.5 (classic T5 v1.1: ONE relative position embedding shared by all blocks), two ways:
    (a) the reference's own T5Encoder(shared_pos=True) (models/wan/modules/t5.py:268-292) and (b) transformers' T5Stack obtained exactly as
    the reference obtains its byT5 model -- `T5ForConditionalGeneration(config).get_encoder()`, called as `model(ids, attention_mask=
    mask.float())[0]` (models/hyvideo/text_encoder/byT5/__init__.py:184-188, pipeline_hunyuan_video.py:1037) -- on the same weights.
    transformers is third-party arithmetic (requirements.txt:5 pins transformers==4.54.0; the T5 encoder arithmetic is unchanged in the
    version installed here): the fixture stores both outputs."""
    import transformers
    from oracle.refshim import load_reference_t5
    from wan2gp_b200 import synth
    cfg = synth.T5_CONFIGS[name]
    R = load_reference_t5()
    enc = R.T5Encoder(cfg["vocab_size"], cfg["dim"], cfg["dim_attn"], cfg["dim_ffn"], cfg["num_heads"], cfg["num_layers"], cfg["num_buckets"],
                      shared_pos=True, dropout=0.1).eval().float()
    sd = synth.make_t5_state_dict(cfg, seed=0)
    enc.load_state_dict(sd, strict=True)
    length, n_valid = 48, 31
    ids, mask = synth.make_t5_inputs(cfg, length, n_valid, seed=0)
    with torch.no_grad():
        out = enc(ids[None], mask[None])[0]
    hf_cfg = transformers.T5Config(vocab_size=cfg["vocab_size"], d_model=cfg["dim"], d_kv=cfg["dim_attn"] // cfg["num_heads"], d_ff=cfg["dim_ffn"],
                                   num_layers=cfg["num_layers"], num_decoder_layers=1, num_heads=cfg["num_heads"],
                                   relative_attention_num_buckets=cfg["num_buckets"], relative_attention_max_distance=128, dropout_rate=0.0,
                                   layer_norm_epsilon=1e-6, feed_forward_proj="gated-gelu", tie_word_embeddings=False)
    hf = transformers.T5ForConditionalGeneration(hf_cfg).get_encoder().eval().float()
    missing, unexpected = hf.load_state_dict(synth.t5_to_hf_t5stack_names(sd, cfg["num_layers"]), strict=True)
    with torch.no_grad():
        out_hf = hf(ids[None], attention_mask=mask[None].float())[0][0]
    d = float((out_hf[:n_valid] - out[:n_valid]).norm() / out[:n_valid].norm())
    print(f"{name}: reference T5Encoder(shared_pos=True) out {tuple(out.shape)} absmean {out.abs().mean():.6f}; transformers {transformers.__version__} "
          f"T5Stack vs it on the valid rows: rel-L2 {d:.3e}")
    np.savez_compressed(os.path.join(GOLDEN, f"{name}.npz"), out=out.numpy().astype(np.float32), out_hf=out_hf.numpy().astype(np.float32),
                        length=length, n_valid=n_valid, seed=0, transformers_version=transformers.__version__)


def run_t5_cases(name):
    """Two more reference T5Encoder calls for tests/test_t5_cpu.py: the umT5 layout (t5_small weights, seed 0) on the first 17 ids of
    the t5_small fixture input without a mask, and the shared-position layout (byt5_tiny, seed 3) on 33 ids of which 20 are valid."""
    from oracle.refshim import load_reference_t5
    R = load_reference_t5()
    out = {}
    for cfg_name, shared_pos, seed in (("t5_small", False, 0), ("byt5_tiny", True, 3)):
        cfg = synth.T5_CONFIGS[cfg_name]
        enc = R.T5Encoder(cfg["vocab_size"], cfg["dim"], cfg["dim_attn"], cfg["dim_ffn"], cfg["num_heads"], cfg["num_layers"], cfg["num_buckets"],
                          shared_pos=shared_pos).eval().float()
        enc.load_state_dict(synth.make_t5_state_dict(cfg, seed))
        with torch.no_grad():
            if shared_pos:
                ids, mask = synth.make_t5_inputs(cfg, 33, 20, seed)
                out[f"{cfg_name}_seed{seed}"] = enc(ids[None], mask[None])[0].numpy()
            else:
                ids, _ = synth.make_t5_inputs(cfg, 40, 29, seed)
                out[f"{cfg_name}_prefix17"] = enc(ids[None, :17])[0].numpy()
    np.savez_compressed(os.path.join(GOLDEN, f"{name}.npz"), **out)
    print(f"{name}: " + ", ".join(f"{k} {v.shape}" for k, v in out.items()))


def run_llm(name):
    """transformers' own language-model classes on seeded synthetic weights, called the way the reference's TextEncoder.encode calls its
    model (input_ids + right-padded attention_mask, output_hidden_states=True; text_encoder_1_5.py:470-476): `Qwen2_5_VLTextModel` (the
    language tower of Qwen2_5_VLForConditionalGeneration, multimodal RoPE sections [16, 24, 24]) for qwen_*, `LlamaModel` for llama_*.
    Eager attention, fp32.  Stores every hidden state on the VALID rows (padded rows are don't-care: the mask crops them downstream)."""
    import transformers
    from wan2gp_b200 import synth
    cfg = synth.LLM_CONFIGS[name]
    common = dict(vocab_size=cfg["vocab_size"], hidden_size=cfg["hidden_size"], intermediate_size=cfg["intermediate_size"],
                  num_hidden_layers=cfg["num_layers"], num_attention_heads=cfg["num_heads"], num_key_value_heads=cfg["num_kv_heads"],
                  rms_norm_eps=cfg["rms_eps"], rope_theta=cfg["rope_theta"], max_position_embeddings=4096, attn_implementation="eager",
                  tie_word_embeddings=False)
    if name.startswith("qwen"):
        from transformers.models.qwen2_5_vl.configuration_qwen2_5_vl import Qwen2_5_VLTextConfig
        from transformers.models.qwen2_5_vl.modeling_qwen2_5_vl import Qwen2_5_VLTextModel
        model = Qwen2_5_VLTextModel(Qwen2_5_VLTextConfig(rope_scaling={"type": "mrope", "mrope_section": [16, 24, 24]}, **common))
    else:
        model = transformers.LlamaModel(transformers.LlamaConfig(attention_bias=False, mlp_bias=False, head_dim=128, **common))
    model = model.eval().float()
    sd = synth.make_llm_state_dict(cfg, seed=0)
    model.load_state_dict(sd, strict=True)
    length, n_valid = 40, 27
    ids, mask = synth.make_llm_inputs(cfg, length, n_valid, seed=0)
    with torch.no_grad():
        out = model(input_ids=ids[None], attention_mask=mask[None], output_hidden_states=True)
    hs = torch.stack([h[0, :n_valid] for h in out.hidden_states])                 # [layers + 1, n_valid, D]
    assert hs.shape[0] == cfg["num_layers"] + 1 and torch.equal(out.last_hidden_state[0, :n_valid], hs[-1])
    print(f"{name}: transformers {transformers.__version__} {type(model).__name__} hidden states {tuple(hs.shape)}, absmean of [-3] {hs[-3].abs().mean():.6f}")
    np.savez_compressed(os.path.join(GOLDEN, f"{name}.npz"), hidden_states=hs.numpy().astype(np.float32), length=length, n_valid=n_valid, seed=0,
                        transformers_version=transformers.__version__)


if __name__ == "__main__":
    torch.set_num_threads(8)
    os.makedirs(GOLDEN, exist_ok=True)
    names = sys.argv[1:] or ["tiny", "tiny_i2v", "small", "vae_tiny", "vae_small"]
    for n in names:
        (run_schedulers if n == "schedulers" else run_t5_cases if n == "t5_cases" else run_llm if n in ("qwen_tiny", "llama_tiny") else run_byt5 if n.startswith("byt5_") else run_t5 if n.startswith("t5_") else run_wan if n in WAN_CASES else run_hy if n in HY_CASES else run_hyvae if n in HYVAE_CASES else run_hyvae10 if n in HYVAE10_CASES else run_vae_enc if n in VAE_ENC_CASES else run_unipc if n == "unipc" else run_vae_tiled if n in TILED_CASES else run_hyvae_enc if n in HYVAE_ENC_CASES else run_hyvae10_enc if n in HYVAE10_ENC_CASES else run_hy_tiled if n in HY_TILED_CASES else run_vae)(n)
