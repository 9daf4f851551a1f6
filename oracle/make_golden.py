"""TEST INFRASTRUCTURE — generates tests/golden/*.npz by running the REAL reference modules
(/root/reference, via oracle/ref_loader.py) on seeded synthetic weights and inputs.

Run in the build container only:  python -m oracle.make_golden [case ...]
The fixtures hold the reference OUTPUTS plus the checksums of the synthetic weights/inputs
that produced them; inputs are regenerated from the seed (vista_b200/synth.py) by the tests.
"""
from __future__ import annotations

import contextlib
import io
import os
import sys
import time
import types

import numpy as np
import torch

from oracle import ref_loader
from vista_b200 import spec, synth

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# name -> (unet preset, latent h, latent w, frames)
UNET_CASES = {
    "unet_tiny": ("tiny", 8, 16, 25),
    "unet_small": ("small", 16, 32, 25),
    "unet_vista_8x16": ("vista", 8, 16, 25),
}
# name -> (preset, h, w, frames, steps, guider, n cond frames)
SAMPLER_CASES = {
    "sampler_tiny_cfg": ("tiny", 8, 16, 25, 4, "VanillaCFG", 1),
    "sampler_tiny_triangle": ("tiny", 8, 16, 25, 3, "TrianglePredictionGuider", 3),
    # BASELINE config 2's step count on the `small` network: error growth over a full 50-step trajectory
    "sampler_small_cfg50": ("small", 16, 32, 25, 50, "VanillaCFG", 1),
}
# name -> (decoder preset, h, w, n latent frames)
DECODER_CASES = {
    "decoder_tiny": ("tiny", 8, 16, 14),
    "decoder_small": ("small", 8, 16, 14),
}
# The measured decoder architecture (vista.yaml: ch = 128, mult 1-2-4-4) on latents of the real magnitude (std 1/0.18215 = 5.5
# after decode_first_stage's division): name -> (preset, h, w, frames, pixel stride of the stored samples).  The outputs are
# too large to commit whole: strided samples + the mean of every 8 x 8 pixel block (fp64 -> fp32) of the full output.
DECODER_BIG_CASES = {
    "decoder_vista_16x32": ("vista", 16, 32, 14, 2),
    "decoder_vista_72x128_t5": ("vista", 72, 128, 5, 8),     # full BASELINE spatial size (d = 512, N = 9216 attention)
}
DECODE_FS_CASES = {
    "decode_first_stage_tiny": ("tiny", 8, 16, 25),
}


def to_t(d):
    return {k: torch.from_numpy(v) for k, v in d.items()}


def unet_inputs(seed, cfg, h, w, T, sigma=5.0, n_cond=1):
    c, uc = synth.synth_conditioning(seed, T, h, w, trajectory=True, context_dim=cfg.context_dim,
                                     adm=cfg.adm_in_channels)
    noise, z, mask = synth.synth_latents(seed, T, h, w)
    mask[:n_cond] = 1.0
    x = np.concatenate([noise, noise], 0) * np.float32(sigma)
    cc = {k: np.concatenate([uc[k], c[k]], 0) for k in c}
    mask2 = np.concatenate([mask, mask], 0)
    return x, cc, mask2


def gen_unet(name):
    preset, h, w, T = UNET_CASES[name]
    cfg = spec.unet_preset(preset)
    sd = synth.synth_state_dict(spec.unet_param_specs(cfg), seed=1)
    ck = synth.state_dict_checksum(sd)
    unet = ref_loader.build_ref_unet(cfg)
    unet.load_state_dict(to_t(sd), strict=True)
    ref = ref_loader.load_reference()
    net = ref.OpenAIWrapper(unet)
    den = ref_loader.build_ref_denoiser(T)
    x, cc, mask2 = unet_inputs(7, cfg, h, w, T)
    sigma = torch.full((2 * T,), 5.0)
    t0 = time.time()
    with torch.no_grad():
        cct = to_t(cc)
        out = den(net, torch.from_numpy(x), sigma, cct, torch.from_numpy(mask2))
        # raw network output too (pre-conditioning removed)
        c_skip, c_out, c_in, c_noise = den.scaling(sigma[:, None, None, None])
        raw = net(torch.from_numpy(x) * c_in, c_noise.reshape(-1), cct, torch.from_numpy(mask2), T)
    print(f"{name}: ref forward x2 {time.time() - t0:.1f}s, out absmean {out.abs().mean():.4f} raw absmean {raw.abs().mean():.4f}")
    np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), denoised=out.numpy(), raw=raw.numpy(),
                        weight_checksum=ck, input_checksum=synth.checksum([x, mask2] + [cc[k] for k in sorted(cc)]),
                        sigma=5.0)


def gen_sampler(name):
    preset, h, w, T, steps, guider, n_cond = SAMPLER_CASES[name]
    cfg = spec.unet_preset(preset)
    sd = synth.synth_state_dict(spec.unet_param_specs(cfg), seed=1)
    unet = ref_loader.build_ref_unet(cfg)
    unet.load_state_dict(to_t(sd), strict=True)
    ref = ref_loader.load_reference()
    net = ref.OpenAIWrapper(unet)
    den = ref_loader.build_ref_denoiser(T)
    smp = ref_loader.build_ref_sampler(steps, guider, 2.5, T)
    c, uc = synth.synth_conditioning(7, T, h, w, trajectory=True, context_dim=cfg.context_dim, adm=cfg.adm_in_channels)
    noise, z, mask = synth.synth_latents(7, T, h, w)
    mask[:n_cond] = 1.0
    # long trajectories also keep the sampler state entering steps 5 / 10 / 25 (the first half of the CFG-doubled x the
    # reference hands to the denoiser at that call): error growth along the trajectory can then be checked, not only its end
    keep = {i: None for i in (5, 10, 25) if i < steps} if steps >= 10 else {}
    calls = {"i": 0}

    def denoise(x, s, cc, m):
        if calls["i"] in keep:
            keep[calls["i"]] = x[: x.shape[0] // 2].clone().numpy()
        calls["i"] += 1
        return den(net, x, s, cc, m)
    t0 = time.time()
    with torch.no_grad():
        out = smp(denoise, torch.from_numpy(noise.copy()), cond=to_t(c), uc=to_t(uc),
                  cond_frame=torch.from_numpy(z), cond_mask=torch.from_numpy(mask))
    print(f"{name}: absmean {out.abs().mean():.4f} ({time.time() - t0:.0f}s, {calls['i']} denoiser calls)")
    np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), sample=out.numpy(),
                        weight_checksum=synth.state_dict_checksum(sd), **{f"state_{i}": v for i, v in keep.items()})


def gen_decoder(name):
    preset, h, w, n = DECODER_CASES[name]
    cfg = spec.decoder_preset(preset)
    sd = synth.synth_state_dict(spec.decoder_param_specs(cfg), seed=2)
    dec = ref_loader.build_ref_decoder(cfg)
    dec.load_state_dict(to_t(sd), strict=True)
    z = synth.normal(9, "dec.z", (n, cfg.z_channels, h, w), std=1.0)
    with torch.no_grad():
        out = dec(torch.from_numpy(z), timesteps=n)
    print(f"{name}: out {tuple(out.shape)} absmean {out.abs().mean():.4f}")
    np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), out=out.numpy(),
                        weight_checksum=synth.state_dict_checksum(sd))


def gen_decoder_big(name):
    preset, h, w, n, stride = DECODER_BIG_CASES[name]
    cfg = spec.decoder_preset(preset)
    sd = synth.synth_state_dict(spec.decoder_param_specs(cfg), seed=2)
    dec = ref_loader.build_ref_decoder(cfg)
    dec.load_state_dict(to_t(sd), strict=True)
    z = synth.normal(9, "decbig.z", (n, cfg.z_channels, h, w), std=1.0 / 0.18215)
    t0 = time.time()
    with torch.no_grad():
        out = dec(torch.from_numpy(z), timesteps=n)
    dt = time.time() - t0
    H, W = out.shape[2], out.shape[3]
    bm = out.double().reshape(n, out.shape[1], H // 8, 8, W // 8, 8).mean(dim=(3, 5)).float()
    print(f"{name}: out {tuple(out.shape)} absmean {out.abs().mean():.4f} rms {out.pow(2).mean().sqrt():.4f} ({dt:.0f}s)")
    np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), samples=out[:, :, ::stride, ::stride].contiguous().numpy(),
                        block_means=bm.numpy(), stride=stride, rms=float(out.pow(2).mean().sqrt()),
                        weight_checksum=synth.state_dict_checksum(sd), cpu_seconds=dt)


def gen_decode_fs(name):
    """DiffusionEngine.decode_first_stage (models/diffusion.py:150-180) called unbound on a stand-in
    engine object: the LightningModule itself cannot be constructed offline (conditioner needs CLIP)."""
    preset, h, w, n = DECODE_FS_CASES[name]
    cfg = spec.decoder_preset(preset)
    sd = synth.synth_state_dict(spec.decoder_param_specs(cfg), seed=2)
    dec = ref_loader.build_ref_decoder(cfg)
    dec.load_state_dict(to_t(sd), strict=True)
    from vwm.models.diffusion import DiffusionEngine
    fsm = types.SimpleNamespace(decoder=dec, decode=lambda z, **kw: dec(z, **kw))
    eng = types.SimpleNamespace(scale_factor=0.18215, en_and_decode_n_samples_a_time=14,
                                disable_first_stage_autocast=True, first_stage_model=fsm)
    z = synth.normal(9, "decfs.z", (n, cfg.z_channels, h, w), std=0.18215)
    fn = DiffusionEngine.decode_first_stage
    fn = getattr(fn, "__wrapped__", fn)
    with torch.no_grad():
        out = fn(eng, torch.from_numpy(z))
    print(f"{name}: out {tuple(out.shape)} absmean {out.abs().mean():.4f}")
    np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), out=out.numpy(),
                        weight_checksum=synth.state_dict_checksum(sd))


# name -> (encoder preset, image h, image w, frames)
ENCODER_CASES = {
    "encoder_tiny": ("tiny", 32, 64, 5),
    "encoder_small": ("small", 64, 128, 3),
}


def gen_encoder(name):
    """Reference Encoder moments, and DiffusionEngine.encode_first_stage (models/diffusion.py:183-195, called unbound on
    a stand-in engine) through AutoencodingEngine.encode's regulariser (DiagonalGaussianRegularizer, sample=True) with
    the device RNG replaced by a recorded noise tensor."""
    preset, h, w, n = ENCODER_CASES[name]
    cfg = spec.encoder_preset(preset)
    sd = synth.synth_state_dict(spec.encoder_param_specs(cfg), seed=3)
    enc = ref_loader.build_ref_encoder(cfg)
    enc.load_state_dict(to_t(sd), strict=True)
    x = synth.normal(11, "enc.x", (n, cfg.in_channels, h, w), std=0.5)
    with torch.no_grad():
        mom = enc(torch.from_numpy(x))
    from vwm.models.diffusion import DiffusionEngine
    from vwm.modules.autoencoding.regularizers import DiagonalGaussianRegularizer
    reg = DiagonalGaussianRegularizer()
    noise = synth.normal(12, "enc.noise", (n, cfg.z_channels, mom.shape[2], mom.shape[3]), std=1.0)
    calls = {"i": 0}
    n_chunk = 2
    real_randn = torch.randn

    def fake_randn(*shape, **kw):              # the regulariser draws mean.shape per chunk, in order
        shp = tuple(shape[0]) if len(shape) == 1 and not isinstance(shape[0], int) else tuple(shape)
        i = calls["i"]
        calls["i"] += shp[0]
        out = torch.from_numpy(noise[i:i + shp[0]])
        assert tuple(out.shape) == shp, (out.shape, shp)
        return out
    fsm = types.SimpleNamespace(encode=lambda xx: reg(enc(xx))[0])
    eng = types.SimpleNamespace(scale_factor=0.18215, en_and_decode_n_samples_a_time=n_chunk,
                                disable_first_stage_autocast=True, first_stage_model=fsm)
    fn = DiffusionEngine.encode_first_stage
    fn = getattr(fn, "__wrapped__", fn)
    torch.randn = fake_randn
    try:
        with torch.no_grad():
            z = fn(eng, torch.from_numpy(x))
    finally:
        torch.randn = real_randn
    assert calls["i"] == n
    print(f"{name}: moments {tuple(mom.shape)} absmean {mom.abs().mean():.4f}; z absmean {z.abs().mean():.4f}")
    np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), moments=mom.numpy(), z=z.numpy(), n_chunk=n_chunk,
                        weight_checksum=synth.state_dict_checksum(sd))


def cond_embedder_inputs(cfg, h, w, n):
    """Seeded inputs of the cond_frames embedder fixture (shared with the tests): images and the quant_conv parameters."""
    x = synth.normal(21, "cemb.x", (n, cfg.in_channels, h, w), std=0.5)
    qw = synth.normal(22, "cemb.qw", (2 * cfg.z_channels, 2 * cfg.z_channels, 1, 1), std=0.35)
    qb = synth.normal(23, "cemb.qb", (2 * cfg.z_channels,), std=0.05)
    return x, qw, qb


def gen_cond_embedder(name="cond_embedder_tiny"):
    """The REAL VideoPredictionEmbedderWithEncoder (encoders/modules.py:428-502) over the REAL AutoencoderKLModeOnly
    (autoencoder.py:519-528), configured like vista.yaml:68-96 at the tiny encoder preset: n_cond_frames 1, n_copies 2,
    is_ae, chunks of 2 frames, scale_factor 0.5 (the YAML leaves 1.0; a non-trivial value pins the multiply)."""
    ref_loader.load_reference()
    from vwm.modules.encoders.modules import VideoPredictionEmbedderWithEncoder
    preset, h, w, n = "tiny", 32, 64, 3
    cfg = spec.encoder_preset(preset)
    sd = synth.synth_state_dict(spec.encoder_param_specs(cfg), seed=3)
    dd = dict(ref_loader.vista_yaml()["model"]["params"]["conditioner_config"]["params"]["emb_models"][3]["params"]["encoder_config"]["params"]["ddconfig"])
    dd.update(ch=cfg.ch, ch_mult=list(cfg.ch_mult), num_res_blocks=cfg.num_res_blocks, z_channels=cfg.z_channels, in_channels=cfg.in_channels)
    with contextlib.redirect_stdout(io.StringIO()):
        emb = VideoPredictionEmbedderWithEncoder(
            n_cond_frames=1, n_copies=2, is_ae=True, scale_factor=0.5, disable_encoder_autocast=True, en_and_decode_n_samples_a_time=2,
            encoder_config={"target": "vwm.models.autoencoder.AutoencoderKLModeOnly",
                            "params": {"embed_dim": cfg.z_channels, "monitor": "val/rec_loss", "ddconfig": dd,
                                       "loss_config": {"target": "torch.nn.Identity"}}}).eval()
    x, qw, qb = cond_embedder_inputs(cfg, h, w, n)
    missing, unexpected = emb.encoder.load_state_dict(
        {**{"encoder." + k: torch.from_numpy(v) for k, v in sd.items()}, "quant_conv.weight": torch.from_numpy(qw),
         "quant_conv.bias": torch.from_numpy(qb)}, strict=False)
    assert not unexpected and all(k.startswith(("decoder.", "post_quant_conv.")) for k in missing), (missing, unexpected)
    with torch.no_grad():
        out = emb(torch.from_numpy(x))
        emb.skip_encode = True
        passthrough = emb(torch.from_numpy(x))
    assert torch.equal(passthrough, torch.from_numpy(x))
    print(f"{name}: out {tuple(out.shape)} absmean {out.abs().mean():.4f}")
    np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), out=out.numpy(), h=h, w=w, n=n,
                        weight_checksum=synth.state_dict_checksum(sd))


def gen_anchors():
    """Closed-form pieces straight from the reference classes (SURVEY §8c)."""
    ref = ref_loader.load_reference()
    disc = ref.discretizer.EDMDiscretization(sigma_min=0.002, sigma_max=700.0, rho=7.0)
    out = {f"sigmas_{n}": disc(n, device="cpu").numpy() for n in (1, 3, 10, 50)}
    sc = ref.denoiser_scaling.VScalingWithEDMcNoise()
    s = torch.tensor([700.0, 15.59, 1.0, 0.002])
    out["vscaling"] = torch.stack(sc(s)).numpy()
    tri = ref.guiders.TrianglePredictionGuider(num_frames=25, max_scale=2.5, min_scale=1.0)
    out["triangle_25"] = tri.scale.numpy()
    lin = ref.guiders.LinearPredictionGuider(num_frames=25, max_scale=2.5, min_scale=1.0)
    out["linear_25"] = lin.scale.numpy()
    from vwm.modules.diffusionmodules.util import timestep_embedding
    out["temb_320"] = timestep_embedding(torch.tensor([0.25 * np.log(700.0), -1.5, 0.0]), 320).numpy()
    out["temb_frames_64"] = timestep_embedding(torch.arange(25), 64).numpy()
    np.savez_compressed(os.path.join(GOLDEN_DIR, "anchors.npz"), **out)
    print("anchors: sigmas_3 =", out["sigmas_3"])


def gen_full_step():
    """BASELINE config 1: one EDM step at 25x4x72x128 with the full vista.yaml network (CPU fp32;
    ~10 min on 8 vCPU).  Stores the step output latent (3.7 MB fp32 -> fp16-rounded copy kept too)."""
    name = "vista_full_step"
    cfg = spec.unet_preset("vista")
    T, h, w = 25, 72, 128
    sd = synth.synth_state_dict(spec.unet_param_specs(cfg), seed=1)
    ck = synth.state_dict_checksum(sd)
    unet = ref_loader.build_ref_unet(cfg)
    unet.load_state_dict(to_t(sd), strict=True)
    del sd
    ref = ref_loader.load_reference()
    net = ref.OpenAIWrapper(unet)
    den = ref_loader.build_ref_denoiser(T)
    smp = ref_loader.build_ref_sampler(1, "VanillaCFG", 2.5, T)
    c, uc = synth.synth_conditioning(7, T, h, w, trajectory=True)
    noise, z, mask = synth.synth_latents(7, T, h, w)
    t0 = time.time()
    with torch.no_grad():
        out = smp(lambda x, s, cc, m: den(net, x, s, cc, m), torch.from_numpy(noise.copy()), cond=to_t(c), uc=to_t(uc),
                  cond_frame=torch.from_numpy(z), cond_mask=torch.from_numpy(mask))
    dt = time.time() - t0
    print(f"{name}: {dt:.1f}s absmean {out.abs().mean():.4f}")
    np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), sample=out.numpy(), weight_checksum=ck,
                        cpu_seconds=dt, cpu_threads=torch.get_num_threads())


def gen_seam():
    """Control runs of tests/test_reference_seam_cpu.py: the reference's own sample_utils.do_sample and
    reward_utils.do_sample on the all-reference engine at tiny sizes, their random draws replaced by seeded tensors."""
    sys.path.insert(0, os.path.dirname(GOLDEN_DIR))
    import test_reference_seam_cpu as seam
    t0 = time.time()
    for name, arrays in seam.control_runs().items():
        print(f"{name}: {sorted(arrays)} ({time.time() - t0:.0f}s)")
        np.savez_compressed(os.path.join(GOLDEN_DIR, name + ".npz"), **arrays)


def main(argv):
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    cases = argv or (["anchors"] + list(UNET_CASES) + list(SAMPLER_CASES) + list(DECODER_CASES) + list(DECODE_FS_CASES) + list(ENCODER_CASES) + ["cond_embedder_tiny", "seam"])
    for cname in cases:
        if cname == "anchors":
            gen_anchors()
        elif cname in UNET_CASES:
            gen_unet(cname)
        elif cname in SAMPLER_CASES:
            gen_sampler(cname)
        elif cname in DECODER_CASES:
            gen_decoder(cname)
        elif cname in DECODER_BIG_CASES:
            gen_decoder_big(cname)
        elif cname in DECODE_FS_CASES:
            gen_decode_fs(cname)
        elif cname in ENCODER_CASES:
            gen_encoder(cname)
        elif cname == "cond_embedder_tiny":
            gen_cond_embedder(cname)
        elif cname == "seam":
            gen_seam()
        elif cname == "vista_full_step":
            gen_full_step()
        else:
            raise KeyError(cname)


if __name__ == "__main__":
    main(sys.argv[1:])
