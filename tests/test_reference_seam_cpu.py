"""The drop-in seam, proven with the reference's OWN caller (SURVEY.md §8b): the REAL `vwm.models.diffusion.DiffusionEngine`
is built from the reference's vista.yaml parameters with only two strings changed —

    network_wrapper:                          vista_b200.modules.B200Wrapper
    first_stage_config.decoder_config.target: vista_b200.vae.VideoDecoder

— the same checkpoint-style state_dict is loaded into it (identical key names), and the UNMODIFIED
`sample_utils.do_sample` (sample_utils.py:286-375: conditioning, encode_first_stage, two autoregressive rounds with the
decode -> re-condition step in between, final chunked decode) is run on it.  The control arm is the all-reference engine
(OpenAIWrapper + the reference VideoDecoder, CPU fp32) with the same random draws; both arms share the real Encoder,
Denoiser, EulerEDMSampler and TrianglePredictionGuider.  That test needs the reference checkout and is skipped without it.

`engine.rollout` and `engine.sample_ensemble` are held to the control runs of the reference's own loops (`sample_utils.do_sample`,
`reward_utils.do_sample`), stored in tests/golden/seam_*.npz by oracle/make_golden.py: every random draw of those runs
(the encoder's posterior sample, the sampler noise of every round / member) is a seeded tensor regenerated here, and the
encoded clip is recomputed with the oracle's encode_first_stage (pinned against the reference's by the stored first frame).

No GPU here, so the B200 executors run on the emulated C-ABI operators of tests/fake_ops.py (same rounding points as the
kernels) — these tests are about the seam and the host logic, the kernels' numerics are the GPU tests' job.  What had to be
patched for a GPU-less host, and nothing else: `load_model` / `unload_model` (= `.cuda()` / `.cpu()`), the
`autocast(device)` scope (CPU autocast would run the control arm in bf16), the sampler's default `device="cuda"` for its
sigma table, and the "CUDA only" guards of the two B200 modules.  The conditioner is a stand-in (tests/seam_fakes.py): the
real one needs the CLIP ViT-H weights, which are not available offline."""
import contextlib
import copy
import io
import os
import sys
import types
from unittest import mock

import pytest
import torch
import yaml

from oracle import ref_loader
from oracle import vista_oracle as vo
from vista_b200 import spec, synth

from helpers import golden, rel_l2, to_t

T, H, W = 25, 32, 64
LAT = (T, 4, H // 2, W // 2)
ROLLOUT = dict(name="seam_do_sample_tiny", tag="rollout", rounds=2, steps=2)
ENSEMBLE = dict(name="seam_reward_tiny", tag="ensemble", members=3, steps=2)
N_SAMPLE = 8192          # stored elements of each compared output (a fixed seeded subset; the whole is too large to commit)

needs_reference = pytest.mark.skipif(not ref_loader.reference_available(), reason="needs the reference checkout")


def _sample(x: torch.Tensor) -> torch.Tensor:
    idx = torch.randperm(x.numel(), generator=torch.Generator().manual_seed(0))[:N_SAMPLE].sort().values
    return x.flatten()[idx]


def _inputs():
    images = torch.from_numpy(synth.normal(21, "seam.img", (T, 3, H, W), std=0.5))
    value_dict = {"cond_frames_without_noise": images[[0]],
                  "cond_frames": images[[0]] + 0.02 * torch.from_numpy(synth.normal(22, "seam.aug", (1, 3, H, W), std=1.0))}
    return images, value_dict


def _draws(tag: str, n: int):
    """The random draws of a control run: the encoder's posterior noise and n sampler noises, each (T, 4, H/2, W/2)."""
    post = torch.from_numpy(synth.normal(30, f"seam.{tag}.posterior", LAT, std=1.0))
    return post, [torch.from_numpy(synth.normal(31 + i, f"seam.{tag}.noise", LAT, std=1.0)) for i in range(n)]


@contextlib.contextmanager
def _replayed_draws(post, noises):
    """The reference's draws replaced by the given tensors, in order: torch.randn (the posterior sample of
    encode_first_stage, one call per chunk of frames) and torch.randn_like (the sampler noise, one call per sampler run)."""
    pos, it, used = [0], iter(noises), []

    def randn(*shape, **kw):
        shp = tuple(shape[0]) if len(shape) == 1 and not isinstance(shape[0], int) else tuple(shape)
        out = post[pos[0]:pos[0] + shp[0]]
        pos[0] += shp[0]
        assert tuple(out.shape) == shp, (tuple(out.shape), shp)
        return out.clone()

    def randn_like(t, *a, **k):
        out = next(it)
        assert out.shape == t.shape, (out.shape, t.shape)
        used.append(out)
        return out.clone().to(t.dtype)
    with mock.patch.object(torch, "randn", randn), mock.patch.object(torch, "randn_like", randn_like):
        yield
    assert pos[0] == post.shape[0] and len(used) == len(noises), (pos[0], len(used))


def _reference_module(name):
    ref_loader.load_reference()
    if "train" not in sys.modules:           # sample_utils / reward_utils import one video-writer helper from the training script
        m = types.ModuleType("train")
        m.save_img_seq_to_video = lambda *a, **k: None
        sys.modules["train"] = m
    return __import__(name)


@contextlib.contextmanager
def _on_cpu(mod):
    """load_model / unload_model / autocast of a reference sampling module made no-ops (CPU, fp32)."""
    with mock.patch.object(mod, "load_model", lambda m: None), mock.patch.object(mod, "unload_model", lambda m: None), \
            mock.patch.object(mod, "autocast", lambda device: contextlib.nullcontext()):
        yield


def _engine_config(native: bool):
    ucfg, dcfg, ecfg = spec.unet_preset("tiny"), spec.decoder_preset("tiny"), spec.encoder_preset("tiny")
    p = copy.deepcopy(ref_loader.vista_yaml()["model"]["params"])
    p["network_config"]["params"].update(model_channels=ucfg.model_channels, attention_resolutions=list(ucfg.attention_resolutions),
                                         num_res_blocks=ucfg.num_res_blocks, channel_mult=list(ucfg.channel_mult))
    p["conditioner_config"] = {"target": "seam_fakes.FakeConditioner", "params": {"down": 2 ** (len(ecfg.ch_mult) - 1)}}
    f = p["first_stage_config"]["params"]
    f["encoder_config"]["params"].update(ch=ecfg.ch, ch_mult=list(ecfg.ch_mult), num_res_blocks=ecfg.num_res_blocks)
    f["decoder_config"]["params"].update(ch=dcfg.ch, ch_mult=list(dcfg.ch_mult), num_res_blocks=dcfg.num_res_blocks)
    if native:                               # the whole integration: two strings
        p["network_wrapper"] = "vista_b200.modules.B200Wrapper"
        f["decoder_config"]["target"] = "vista_b200.vae.VideoDecoder"
    return p, (ucfg, dcfg, ecfg)


def _checkpoint(cfgs):
    ucfg, dcfg, ecfg = cfgs
    sd = {}
    for prefix, specs, seed in (("model.diffusion_model.", spec.unet_param_specs(ucfg), 1),
                                ("first_stage_model.decoder.", spec.decoder_param_specs(dcfg), 2),
                                ("first_stage_model.encoder.", spec.encoder_param_specs(ecfg), 3)):
        for k, v in synth.synth_state_dict(specs, seed=seed).items():
            sd[prefix + k] = torch.from_numpy(v)
    return sd


def _run_do_sample(native: bool, rounds: int, steps: int):
    """The reference's do_sample on the reference DiffusionEngine (native: with the two B200 modules plugged in)."""
    su = _reference_module("sample_utils")
    from vwm.models.diffusion import DiffusionEngine
    from fake_ops import patched_ops
    from vista_b200 import fused as fused_mod
    p, cfgs = _engine_config(native)
    with contextlib.redirect_stdout(io.StringIO()):
        eng = DiffusionEngine(**p).eval()
    missing, unexpected = eng.load_state_dict(_checkpoint(cfgs), strict=False)
    assert not unexpected and all(m.startswith("conditioner.") for m in missing), (missing[:3], unexpected[:3])
    ops_ctx = contextlib.nullcontext()
    if native:
        from vista_b200.modules import B200Wrapper
        from vista_b200.vae import DecoderRuntime, VideoDecoder
        assert isinstance(eng.model, B200Wrapper) and isinstance(eng.first_stage_model.decoder, VideoDecoder)
        eng.model._require_cuda = lambda device: None             # GPU-less host: executors on the emulated operators
        dec = eng.first_stage_model.decoder
        with patched_ops():
            rt_dec = DecoderRuntime(dec.b200_config, dec.state_dict(), "cpu")
        dec.runtime = lambda device: rt_dec
        ops_ctx = patched_ops()
    sampler = su.init_sampling(guider="TrianglePredictionGuider", steps=steps, cfg_scale=2.5, num_frames=T)
    sampler.device = "cpu"                                         # its default "cuda" only places the sigma table
    images, value_dict = _inputs()
    with _on_cpu(su), mock.patch.object(fused_mod, "USE_GRAPH", False), _replayed_draws(*_draws(ROLLOUT["tag"], rounds)), \
            ops_ctx, contextlib.redirect_stderr(io.StringIO()):
        samples, samples_z, _ = su.do_sample(images, eng, sampler, value_dict, num_rounds=rounds, num_frames=T,
                                             initial_cond_indices=[0], device="cpu")
    return samples, samples_z


def _run_reward_do_sample(members: int, steps: int):
    """The reference's reward_utils.do_sample on the all-reference engine -> (reward, encoded clip)."""
    ru = _reference_module("reward_utils")
    from vwm.models.diffusion import DiffusionEngine
    p, cfgs = _engine_config(False)
    with contextlib.redirect_stdout(io.StringIO()):
        eng = DiffusionEngine(**p).eval()
    eng.load_state_dict(_checkpoint(cfgs), strict=False)
    sampler = ru.init_sampling(guider="VanillaCFG", steps=steps, cfg_scale=2.5, num_frames=T)
    sampler.device = "cpu"
    images, value_dict = _inputs()
    zs, real_encode = [], eng.encode_first_stage
    eng.encode_first_stage = lambda x: (zs.append(real_encode(x)), zs[-1])[1]
    with _on_cpu(ru), _replayed_draws(*_draws(ENSEMBLE["tag"], members)), contextlib.redirect_stderr(io.StringIO()):
        _, reward = ru.do_sample(images, eng, sampler, value_dict, num_frames=T, ensemble_size=members,
                                 initial_cond_indices=[0], device="cpu")
    assert len(zs) == 1
    return reward, zs[0]


def control_runs():
    """The fixtures of this module from the reference's own loops (oracle/make_golden.py writes them)."""
    x, z = _run_do_sample(False, ROLLOUT["rounds"], ROLLOUT["steps"])
    reward, z_ens = _run_reward_do_sample(ENSEMBLE["members"], ENSEMBLE["steps"])
    return {ROLLOUT["name"]: dict(frames_shape=list(x.shape), frames=_sample(x).numpy(), samples_z_shape=list(z.shape),
                                  samples_z=_sample(z).numpy(), z0=z[0].numpy()),
            ENSEMBLE["name"]: dict(reward=float(reward), z0=z_ens[0].numpy())}


@needs_reference
def test_unmodified_do_sample_runs_on_the_b200_seams():
    rounds, steps = ROLLOUT["rounds"], ROLLOUT["steps"]
    ref_x, ref_z = _run_do_sample(False, rounds, steps)
    our_x, our_z = _run_do_sample(True, rounds, steps)
    n = rounds * (T - 3) + 3
    assert our_z.shape == ref_z.shape == (n, 4, H // 2, W // 2) and our_x.shape == ref_x.shape == (n, 3, H, W)
    rz, rx = rel_l2(our_z, ref_z), rel_l2(our_x, ref_x)
    print(f"do_sample through the B200 seams vs the all-reference engine: latents rel-L2 {rz:.3e}, frames rel-L2 {rx:.3e}")
    assert rz < 5e-3 and rx < 5e-3, (rz, rx)
    assert torch.equal(our_z[0], ref_z[0])          # sample[0] = z[0] (sample_utils.py:336): the encoder path is shared


# ---- our engine against the stored control runs ----
def _our_engine(steps: int, guider_config=None):
    """vista_b200.engine.DiffusionEngine from configs/inference/vista_b200.yaml at tiny sizes, the same checkpoint, the same
    stand-in conditioner, on the emulated operators."""
    from vista_b200.diffusion import instantiate_from_config
    ucfg, dcfg, ecfg = spec.unet_preset("tiny"), spec.decoder_preset("tiny"), spec.encoder_preset("tiny")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cfg = yaml.safe_load(open(os.path.join(root, "configs", "inference", "vista_b200.yaml")))["model"]
    p = cfg["params"]
    p["network_config"]["params"].update(model_channels=ucfg.model_channels, channel_mult=list(ucfg.channel_mult),
                                         num_res_blocks=ucfg.num_res_blocks, attention_resolutions=list(ucfg.attention_resolutions))
    p["first_stage_config"]["params"]["decoder_config"]["params"].update(ch=dcfg.ch, ch_mult=list(dcfg.ch_mult), num_res_blocks=dcfg.num_res_blocks)
    p["conditioner_config"] = {"target": "seam_fakes.FakeConditioner", "params": {"down": 2 ** (len(ecfg.ch_mult) - 1)}}
    p["sampler_config"]["params"].update(num_steps=steps, device="cpu")
    if guider_config is not None:
        p["sampler_config"]["params"]["guider_config"] = guider_config
    p["en_and_decode_n_samples_a_time"] = 14
    eng = instantiate_from_config(cfg)
    cfgs = (ucfg, dcfg, ecfg)
    ck = {k: v for k, v in _checkpoint(cfgs).items() if not k.startswith("first_stage_model.encoder.")}
    missing, unexpected = eng.load_state_dict(ck, strict=False)
    assert not unexpected and all(m.startswith("_conditioner.") for m in missing), (missing[:3], unexpected[:3])
    eng.model._require_cuda = eng.model.diffusion_model._require_cuda = lambda device: None
    return eng, cfgs


def _encoded_clip(ecfg, images, tag):
    """The control run's encode_first_stage (chunks of 14 frames, posterior sampled with its recorded draw), by the oracle."""
    sd = synth.synth_state_dict(spec.encoder_param_specs(ecfg), seed=3)
    with torch.no_grad():
        return vo.encode_first_stage(to_t(sd), ecfg, images, n_samples=14, noise=_draws(tag, 0)[0])


def _condition(eng, value_dict, skip_encode=False):
    """sample_utils.get_condition over the stand-in conditioner: every value repeated to T rows, (c, uc) of T rows."""
    for e in eng.conditioner.embedders:
        if hasattr(e, "skip_encode"):
            e.skip_encode = skip_encode
    try:
        keys = {e.input_key for e in eng.conditioner.embedders}
        batch = {k: v.repeat(T, *[1] * (v.dim() - 1)) for k, v in value_dict.items() if k in keys}
        c, uc = eng.conditioner.get_unconditional_conditioning(batch, batch_uc={k: v.clone() for k, v in batch.items()},
                                                               force_uc_zero_embeddings=[])
    finally:
        for e in eng.conditioner.embedders:
            if hasattr(e, "skip_encode"):
                e.skip_encode = False
    return {k: v[:T] for k, v in c.items()}, {k: v[:T] for k, v in uc.items()}


def test_engine_rollout_equals_the_real_do_sample(monkeypatch):
    """SURVEY 8f row 2 pinned to the reference's OWN loop: `vista_b200.engine.DiffusionEngine.rollout` (device-side latent
    bookkeeping, `recondition` hook) must reproduce what the unmodified `sample_utils.do_sample` computed on the all-reference
    engine — same encoded clip, same noise draws, the re-conditioning between rounds done like the reference's
    `get_condition` over the same stand-in conditioner (decode -> frame [-3] -> new c / uc)."""
    from fake_ops import patched_ops
    from vista_b200 import fused as fused_mod
    from vista_b200 import vae as vae_mod
    g = golden(ROLLOUT["name"])
    rounds, steps = ROLLOUT["rounds"], ROLLOUT["steps"]
    monkeypatch.setattr(fused_mod, "USE_GRAPH", False)
    eng, (ucfg, dcfg, ecfg) = _our_engine(steps, {"target": "vista_b200.diffusion.TrianglePredictionGuider",
                                                 "params": {"max_scale": 2.5, "num_frames": T}})
    monkeypatch.setattr(vae_mod.VideoDecoder, "runtime", lambda self, device: self.__dict__.setdefault(
        "_rt_cpu", vae_mod.DecoderRuntime(self.b200_config, self.state_dict(), "cpu")))
    images, value_dict = _inputs()
    z = _encoded_clip(ecfg, images, ROLLOUT["tag"])
    assert rel_l2(z[0], torch.from_numpy(g["z0"])) < 2e-5     # the reference's encoded first frame (sample[0] = z[0])

    def recondition(round_idx, sample, decode_tail):                       # sample_utils.py:340-348
        vd = dict(value_dict)
        vd["cond_frames_without_noise"] = decode_tail()[[-3]]
        vd["cond_frames"] = sample[[-3]] / eng.scale_factor
        return _condition(eng, vd, skip_encode=True)
    with patched_ops(), torch.no_grad():
        c, uc = _condition(eng, value_dict)
        frames, samples_z = eng.rollout(c, uc, z, rounds, noises=_draws(ROLLOUT["tag"], rounds)[1], recondition=recondition)
    assert list(samples_z.shape) == list(g["samples_z_shape"]) and list(frames.shape) == list(g["frames_shape"])
    rz = rel_l2(_sample(samples_z), torch.from_numpy(g["samples_z"]))
    rx = rel_l2(_sample(frames), torch.from_numpy(g["frames"]))
    print(f"engine.rollout vs the real do_sample ({rounds} rounds): latents rel-L2 {rz:.3e}, frames rel-L2 {rx:.3e}")
    assert rz < 5e-3 and rx < 5e-3, (rz, rx)


def test_engine_sample_ensemble_equals_the_real_reward_do_sample(monkeypatch):
    """SURVEY 8f row 3 pinned to the reference's OWN loop: `engine.sample_ensemble` against what the unmodified
    `reward_utils.do_sample` (reward_utils.py:285-340) computed on the all-reference engine: same encoded clip, the same
    member noises; the reward exp(-mean unbiased variance) must agree."""
    from fake_ops import patched_ops
    from vista_b200 import fused as fused_mod
    g = golden(ENSEMBLE["name"])
    K, steps = ENSEMBLE["members"], ENSEMBLE["steps"]
    monkeypatch.setattr(fused_mod, "USE_GRAPH", False)
    eng, (ucfg, dcfg, ecfg) = _our_engine(steps)
    images, value_dict = _inputs()
    z = _encoded_clip(ecfg, images, ENSEMBLE["tag"])
    assert rel_l2(z[0], torch.from_numpy(g["z0"])) < 2e-5
    with patched_ops(), torch.no_grad():
        c, uc = _condition(eng, value_dict)
        reward, members = eng.sample_ensemble(c, uc, z, K, noises=_draws(ENSEMBLE["tag"], K)[1])
    ref_reward = float(g["reward"])
    print(f"ensemble reward: engine {float(reward):.6f} vs the real reward_utils.do_sample {ref_reward:.6f}")
    assert abs(float(reward) - ref_reward) < 2e-3 * max(1.0, abs(ref_reward)), (float(reward), ref_reward)
