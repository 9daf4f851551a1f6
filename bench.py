#!/usr/bin/env python
"""Benchmark of the Vista denoising hot path on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config full|small] [--dump-outputs DIR]

A bench "step" is ONE EDM/Euler sampler step of a 25-frame 576x1024 clip: sampler_prepare ->
UNet forward on the CFG-doubled batch (50 x 8 x 72 x 128) -> sampler_update — the loop body of
vwm/modules/diffusionmodules/sampling.py:104-121.  `ms_per_step` is the "UNet step ms" of
BASELINE.json; `value` is "denoised frames/sec at 25x576x1024, 50 EDM steps" =
25 / (50 * step_seconds + decode_seconds), with the 25-frame chunked VAE decode timed in the same
run (reported as `decode_ms`; null until the decoder lands, in which case `value` is sampler-only and
`config.decode` says so).  Synthetic seeded weights / inputs (no checkpoint offline).

N > 1 (torchrun): the ONE clip is spread over the ranks (vista_b200/sharded.py: CFG halves, then frames; the temporal K/V
all-gather, the GroupNorm-sum all-reduce, the one-frame halos and the CFG pair exchange are kernels over NVLink peer windows
— csrc/peer.cu — and the step a CUDA-graph replay; VISTA_B200_PEER=0 = the NCCL + launch-tape transport) -> strong scaling:
value = 25 frames / max-over-ranks time of the same job.  In that mode the line also carries `parity_rel_l2`: the sharded
K-step latent against the unsharded runtime on rank 0 (exit code 4 above 3e-3).  `e2e` is the second call of the public
engine.sample() -> decode_first_stage() pair (the first, which captures the 50-step graph, is `first_call_seconds`).

--dump-outputs DIR writes, as float32 DIR/<name>.npy, what the timed calls handed back: `latent` (the latent after the
last timed sampler step, whole), `decoded` (the timed decode_first_stage) and `e2e_frames` (the frames of the timed e2e
call).  An output above DUMP_MAX_ELEMS elements is stored as a fixed seeded sample of that many elements (the same
positions in every run), so that two builds can be compared output for output; weights and inputs are seeded.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

F_STEP_TFLOP = 153.9          # algorithmic TFLOP per EDM step at B=50, 72x128 (SURVEY.md §8d / BASELINE.md §2)
F_DEC_CHUNK_TFLOP = 97.202    # per 14-frame VideoDecoder call
DUMP_MAX_ELEMS = 1 << 22      # per dumped output (16 MB of float32); three outputs stay under 64 MB


def dump_outputs(path, arrays):
    """Writes every tensor of `arrays` as float32 <path>/<name>.npy; a larger one as a seeded sample of its elements."""
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float().cpu()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMS].sort().values
            t = t.flatten()[idx]
        np.save(os.path.join(path, name + ".npy"), t.numpy())


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(tflops=float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0))),
                    tflops_burst=float(d.get("bf16_tflops", 1590.0)), hbm=float(d.get("hbm_gbs", 6650.0)), src="measured")
    return dict(tflops=1400.0, tflops_burst=1590.0, hbm=6650.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def dist_env():
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    return rank, world, local


# ---------------------------------------------------------------------------------------------
# problem construction
# ---------------------------------------------------------------------------------------------
def make_problem(config: str, device, seed=0):
    """Presets + a seeded weight generator.  Every rank builds the SAME weights (one clip is spread over the ranks)."""
    from vista_b200 import spec
    if config == "full":
        ucfg, dcfg, h, w = spec.unet_preset("vista"), spec.decoder_preset("vista"), 72, 128
    else:  # reduced smoke configuration (NOT a bench value; used by --config small for quick checks)
        ucfg, dcfg, h, w = spec.unet_preset("small"), spec.decoder_preset("small"), 16, 32
    g = torch.Generator(device=device).manual_seed(1234 + seed)

    def rand_sd(specs):
        sd = {}
        for k, (shape, kind) in specs.items():
            fan_in = int(np.prod(shape[1:])) if len(shape) > 1 else 1
            if kind in ("w", "wz"):
                t = torch.randn(shape, generator=g, device=device) * ((0.8 if kind == "w" else 0.5) / fan_in ** 0.5)
            elif kind == "b":
                t = torch.randn(shape, generator=g, device=device) * 0.05
            elif kind == "g":
                t = 1 + 0.1 * torch.randn(shape, generator=g, device=device)
            else:
                t = (0.5 if kind == "mix" else 0.0) + 0.3 * torch.randn(shape, generator=g, device=device)
            sd[k] = t
        return sd

    return ucfg, dcfg, h, w, rand_sd


def build_engine(config: str, dev):
    """The public object a user of the reference gets from `instantiate_from_config(yaml.model)` (sample_utils.py:49-80)
    — here from configs/inference/vista_b200.yaml — with seeded random weights of the named architecture."""
    import yaml
    from vista_b200 import spec
    from vista_b200.diffusion import instantiate_from_config
    ucfg, dcfg, h, w, rand_sd = make_problem(config, dev, seed=0)
    cfg = yaml.safe_load(open(os.path.join(ROOT, "configs", "inference", "vista_b200.yaml")))["model"]
    p = cfg["params"]
    p["network_config"]["params"].update(model_channels=ucfg.model_channels, channel_mult=list(ucfg.channel_mult),
                                         num_res_blocks=ucfg.num_res_blocks,
                                         attention_resolutions=list(ucfg.attention_resolutions))
    p["first_stage_config"]["params"]["decoder_config"]["params"].update(ch=dcfg.ch, ch_mult=list(dcfg.ch_mult),
                                                                       num_res_blocks=dcfg.num_res_blocks)
    p["replace_cond_frames"], p["fixed_cond_frames"] = True, [0]          # 1 conditioning frame (BASELINE configs[1])
    with torch.device(dev):
        eng = instantiate_from_config(cfg)
    eng.model.diffusion_model.load_state_dict(rand_sd(spec.unet_param_specs(ucfg)), strict=True)
    eng.first_stage_model.decoder.load_state_dict(rand_sd(spec.decoder_param_specs(dcfg)), strict=True)
    return eng, ucfg, dcfg, h, w


def host_inputs(ucfg, T, h, w, seed=7):
    from vista_b200 import synth
    c, uc = synth.synth_conditioning(seed, T, h, w, trajectory=True, context_dim=ucfg.context_dim, adm=ucfg.adm_in_channels)
    noise, z, mask = synth.synth_latents(seed, T, h, w)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    return ({k: pin(v) for k, v in c.items()}, {k: pin(v) for k, v in uc.items()}, pin(noise), pin(z), pin(mask))


def rel_l2(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a - b).norm() / (b.norm() + 1e-30))


def load_traffic():
    """DRAM bytes of the tap-GEMM launches of one step from the committed ncu capture (profiles/r02_traffic.json,
    written by tools/ncu_traffic.py from `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum`)."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.isfile(p):
        return json.load(open(p))
    return None


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def run_ours(args):
    rank, world, local = dist_env()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        import datetime
        # a dead rank must fail the job in minutes, not after NCCL's default 10-minute watchdog
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=int(os.environ.get("VISTA_B200_NCCL_TIMEOUT", "180"))))
    from vista_b200 import lib, ops
    from vista_b200.diffusion import B200Denoiser
    from vista_b200.modules import B200Wrapper
    lib.load()
    T = 25
    eng, ucfg, dcfg, h, w = build_engine(args.config, dev)
    net, unet, denoiser, sampler = eng.model, eng.model.diffusion_model, eng.denoiser, eng.sampler
    K, W = args.steps, args.warmup
    bden = B200Denoiser(denoiser, net)
    c_h, uc_h, noise_h, z_h, mask_h = host_inputs(ucfg, T, h, w)
    to_dev = lambda d: {k: v.to(dev, non_blocking=True) for k, v in d.items()}

    # ---- device-resident timing: K sampler steps bracketed by events.
    #      N = 1: the step is replayed from a CUDA graph.  N > 1: the ONE clip is spread over the ranks: CFG halves
    #      first (even N), then frames (K/V all-gather, GN-sum all-reduce, one-frame halos: vista_b200/sharded.py).
    c, uc = to_dev(c_h), to_dev(uc_h)
    noise, z, mask = noise_h.to(dev), z_h.to(dev), mask_h.to(dev)
    sharded = world > 1
    if sharded:
        net.enable_frame_sharding()
    rt = net._rt_get(unet, T, dev)
    x = noise.clone()
    sampler(bden, x, c, uc=uc, cond_frame=z, cond_mask=mask, num_steps=max(W, 3))   # warm-up: allocs (+ graph capture)
    Tl = (rt.t1 - rt.t0) if sharded else T
    st = rt._loop_states[(Tl, h, w)]
    n_total = W + K
    assert n_total + 1 <= st.sigmas.numel()
    sig = sampler.discretization(n_total, device="cpu").to(torch.float32)
    l0 = ops.LAUNCHES
    st.one_step(rt, n_total)   # eager (counts launches of one step)
    launches_per_step = ops.LAUNCHES - l0
    run_step = st.runner(rt, n_total)          # CUDA-graph replay unless the UNet itself holds collectives
    x0 = noise[rt.t0:rt.t1] if sharded else noise
    st.x.copy_(x0 * torch.sqrt(1.0 + sig[0] ** 2).to(dev))
    st.sigmas[: n_total + 1].copy_(sig)
    st.step.zero_()
    for _ in range(W):
        run_step()
    clocks = ClockSampler(local)
    barrier = (lambda: torch.distributed.barrier()) if world > 1 else (lambda: None)
    barrier()
    torch.cuda.synchronize()
    clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        run_step()
    e1.record()
    torch.cuda.synchronize()
    barrier()
    dt = e0.elapsed_time(e1) / 1e3
    clk = clocks.stop()
    finite = bool(torch.isfinite(st.x).all())
    if args.dump_outputs:          # before the profiled step below, which advances st.x once more
        from vista_b200.sharded import gather_latent
        latent_out = (st.x if Tl == T else gather_latent(st.x, T, group=rt.group)).cpu()

    # ---- per-family breakdown of one extra eager step (CUDA events per launch; N > 1: this rank's share, with the
    #      host-side collectives bracketed as family "nccl")
    ops.PROFILE = []
    lib.HOST_PROFILE = (ops._prof_begin, ops._prof_end)
    st.one_step(rt, n_total + 1)
    torch.cuda.synchronize()
    rec, ops.PROFILE, lib.HOST_PROFILE = ops.PROFILE, None, None
    fam, det = ops.profile_summary(rec)
    tot_ms = sum(r["ms"] for r in fam.values())
    gemm_prof = {k: {"ms": round(v["ms"], 3), "launches": v["launches"], "tflops": round(v["tflops"], 1),
                     "gbs": round(v["gbs"], 1), "share": round(v["ms"] / tot_ms, 4)} for k, v in fam.items()}
    if args.breakdown and rank == 0:
        with open(args.breakdown, "w") as f:
            f.write(f"# one EDM step, rank 0 of {world}: kernel time by family (CUDA events per launch, eager)\n\n"
                    f"sum of bracketed times {tot_ms:.1f} ms; timed step {dt / K * 1e3:.1f} ms\n\n"
                    "| family | launches | ms | share | TFLOP/s | GB/s (algorithmic) |\n|---|---|---|---|---|---|\n")
            for k, v in sorted(fam.items(), key=lambda kv: -kv[1]["ms"]):
                f.write(f"| {k} | {v['launches']} | {v['ms']:.2f} | {v['ms'] / tot_ms:.1%} | {v['tflops']:.0f} | {v['gbs']:.0f} |\n")
            f.write("\n## by shape (top 48)\n\n| family | detail | launches | ms | TFLOP/s | GB/s |\n|---|---|---|---|---|---|\n")
            for (k, d), v in sorted(det.items(), key=lambda kv: -kv[1]["ms"])[:48]:
                f.write(f"| {k} | {d} | {v['launches']} | {v['ms']:.2f} | {v['tflops']:.0f} | {v['gbs']:.0f} |\n")

    # ---- decode: the engine's own chunked decode_first_stage of the 25 latents (N > 1: chunks dealt out over the ranks)
    zlat = (torch.randn(T, 4, h, w, device=dev, generator=torch.Generator(device=dev).manual_seed(5)) * 0.9)
    if world > 1:
        torch.distributed.broadcast(zlat, src=0)
    eng.decode_first_stage(zlat)
    torch.cuda.synchronize()
    d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d0.record()
    decoded = eng.decode_first_stage(zlat)
    d1.record()
    torch.cuda.synchronize()
    decode_s = d0.elapsed_time(d1) / 1e3

    # ---- N > 1: parity of the sharded K-step sample against the unsharded one on rank 0 (same weights, same seed)
    parity = None
    if sharded:
        xs = sampler(bden, noise.clone(), c, uc=uc, cond_frame=z, cond_mask=mask, num_steps=K)   # gathered on every rank
        torch.cuda.synchronize()
        if rank == 0:
            net1 = B200Wrapper(unet)                     # plain single-GPU runtime over the same parameters
            x1 = sampler(B200Denoiser(denoiser, net1), noise.clone(), c, uc=uc, cond_frame=z, cond_mask=mask, num_steps=K)
            torch.cuda.synchronize()
            parity = rel_l2(xs, x1)
            del net1
        barrier()

    # ---- e2e: the public calls a user makes — engine.sample() (50 steps) -> engine.decode_first_stage() — with HOST
    #      (pinned) inputs and the decoded frames copied back to the host inside the timed region
    def e2e_once():
        t_a = time.perf_counter()
        cc, ucc = to_dev(c_h), to_dev(uc_h)
        zz = z_h.to(dev, non_blocking=True)
        lat = eng.sample(cc, cond_frame=zz, uc=ucc, N=T, shape=(4, h, w), noise=noise_h)
        torch.cuda.synchronize()
        t_b = time.perf_counter()
        frames = eng.decode_first_stage(lat)
        torch.cuda.synchronize()
        t_c = time.perf_counter()
        out = frames.to("cpu", non_blocking=False)
        return out, (t_b - t_a, t_c - t_b, time.perf_counter() - t_c)
    # one untimed call first: the 50-step schedule gets its own captured step graph (num_steps is a kernel argument) and the
    # allocator its blocks — one-off costs of the first call of a process, reported as `first_call_seconds`, not steady state
    barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e2e_once()
    torch.cuda.synchronize()
    e2e_first = time.perf_counter() - t0
    barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res, e2e_parts = e2e_once()
    torch.cuda.synchronize()
    e2e_dt = time.perf_counter() - t0
    n_e2e_steps = sampler.num_steps
    h2d = sum(v.numel() * v.element_size() for d in (c_h, uc_h) for v in d.values()) + \
        sum(v.numel() * v.element_size() for v in (noise_h, z_h))
    d2h = res.numel() * res.element_size()
    e2e_finite = bool(torch.isfinite(res).all())

    if world > 1:
        tmax = torch.tensor([dt, e2e_dt, decode_s], device=dev)
        torch.distributed.all_reduce(tmax, op=torch.distributed.ReduceOp.MAX)
        dt, e2e_dt, decode_s = float(tmax[0]), float(tmax[1]), float(tmax[2])
    step_s = dt / K

    peer_on = getattr(st, "pair_peer", None) is not None or getattr(rt, "win", None) is not None
    transport = ("stores into the peers' NVLink windows + flags (csrc/peer.cu), step replayed from a CUDA graph" if peer_on
                 else "NCCL, step replayed from a launch tape")
    if world == 1:
        shard_desc = "single GPU"
    elif net.cfg_half is not None:
        shard_desc = (f"one clip over {world} GPUs: CFG halves x frames ({world // 2} frame shard(s) per half); per step a "
                      f"pairwise exchange of the 4-channel network output" +
                      ("" if world == 2 else ", and inside each half temporal K/V all-gather, GN-sum all-reduce, 1-frame halos") +
                      f" [{transport}]; decode chunks dealt out over the ranks (frame-sharded up to 4 ranks)")
    else:
        shard_desc = (f"frames of one clip over {world} GPUs: temporal K/V all-gather, GN-sum all-reduce, 1-frame halos "
                      f"[{transport}]; decode chunks dealt out over the ranks")
    peaks = load_peaks()
    full = args.config == "full"
    ach = (F_STEP_TFLOP / step_s) if full else None        # whole-job TFLOP/s: all N GPUs work on the one clip
    out = {
        "metric": "denoised frames/sec at 25x576x1024, 50 EDM steps; UNet step ms",
        "value": T / (50 * step_s + decode_s), "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f16 (fp32 accumulate, fp32 norms/softmax/sampler state)", "data": "synthetic",
        "config": {"workload": "configs[1]: full 50-step sample, 25x576x1024 (latent 25x4x72x128, CFG batch 50), 1 cond frame, "
                               "VanillaCFG 2.5" if full else "REDUCED smoke config (not a bench value)",
                   "step": "one EDM/Euler step (prepare + UNet + update); frames/s = 25/(50*step + decode)",
                   "decode": "included (engine.decode_first_stage of the 25 latents, timed in the same run)",
                   "l2": "activations per step (> 10 GB) exceed the 126 MB L2; no explicit flush",
                   "sharding": shard_desc,
                   "scaling_note": "ONE clip whatever N: total work is fixed (strong scaling)"},
        "decode_ms": decode_s * 1e3,
        "finite": finite and e2e_finite,
        "gpu_launches": launches_per_step * K,
        "launches_per_step": launches_per_step,
        "clocks": clk,
        "e2e": {"value": T / e2e_dt, "unit": "frames/s", "seconds": e2e_dt, "steps": n_e2e_steps,
                "h2d_bytes_per_step": h2d / n_e2e_steps, "d2h_bytes_per_step": d2h / n_e2e_steps,
                "h2d_bytes": h2d, "d2h_bytes": d2h,
                "sample_seconds": e2e_parts[0], "decode_seconds": e2e_parts[1], "d2h_seconds": e2e_parts[2],
                "first_call_seconds": e2e_first,
                "scope": "engine.sample() (50 EDM steps, pinned host inputs) -> engine.decode_first_stage() -> 25 decoded "
                         "fp32 frames copied to the host; wall clock around the public calls (second call of the process; "
                         "the first one, which also captures the 50-step graph, is first_call_seconds)"},
    }
    if parity is not None or sharded:
        out["parity_rel_l2"] = parity
        out["parity_note"] = (f"{K}-step sample, sharded over {world} GPUs vs the unsharded runtime on rank 0, same weights / "
                              "seed (limit 3e-3)")
    g = gemm_prof.get("gemm")
    traffic = load_traffic() if (full and world == 1) else None
    n_peak = world * peaks["tflops"]
    out["roofline"] = {"bound": "tensor", "achieved": g["tflops"] if g else ach, "peak": peaks["tflops"], "unit": "TFLOP/s",
                       "frac": (g["tflops"] / peaks["tflops"]) if g else None,
                       "traffic": traffic.get("gemm_dram_bytes_per_step") if traffic else None,
                       "traffic_note": (traffic.get("note") if traffic else "no ncu capture committed for this configuration"),
                       "algorithmic_bytes": (g["gbs"] * g["ms"] * 1e6) if g else None,
                       "kernel": "tapgemm_kernel (all Linear / conv launches of one step on this rank: algorithmic 2*M*N*K "
                                 "FLOPs over the CUDA-event time of those launches; one GPU's peak)",
                       "peak_source": peaks["src"] + " bf16 sustained (kernel timed inside a long step)",
                       "step": {"achieved": ach, "frac": (ach / n_peak) if ach else None, "flops_per_step_T": F_STEP_TFLOP,
                                "peak": n_peak,
                                "scope": f"153.9 algorithmic TFLOP of the UNet step / step time, against {world} x the one-GPU peak"},
                       "families": gemm_prof}
    if rank == 0 and world == 1 and not args.no_eager and full:
        try:
            out["gpu_eager_baseline"] = gpu_eager_baseline(dev, ucfg, h, w, step_s)
        except Exception as e:                                        # the product numbers above stand on their own
            out["gpu_eager_baseline"] = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    if rank == 0 and world == 1 and not args.no_cpu:
        out["cpu_baseline"] = cpu_baseline(args.cpu_seconds)
    if rank == 0:
        print(json.dumps(out))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"latent": latent_out, "decoded": decoded, "e2e_frames": res})
    bad_parity = parity is not None and not (parity < 3e-3)
    if world > 1:
        # The measurement is complete and printed.  Leave without the NCCL / interpreter teardown: a multi-rank process
        # that lingers there would hold the whole launch hostage (seen once, when a frames-only step on the default
        # process group had been CUDA-graph-captured with its NCCL calls inside; that path now uses the launch tape).
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(4 if bad_parity else 0)


# ---------------------------------------------------------------------------------------------
# eager-GPU denominator (north_star: ">= 6x single-GPU frames/sec vs the reference's PyTorch-eager path on one B200")
# ---------------------------------------------------------------------------------------------
def gpu_eager_baseline(dev, ucfg, h, w, our_step_s, warm=2, timed=3):
    """The oracle port (plain torch functional ops, validated against the real reference modules) run on the GPU under
    torch.autocast(fp16) with fp32 weights — the reference's own inference precision (sample_utils.py:303) — eager,
    cuDNN / cuBLAS / SDPA kernels chosen by torch (xformers is not installable here; its attention is torch SDPA).
    The real reference modules do not travel to the GPU box (/root/reference is absent there), so this is the stated
    proxy for the "reference GPU baseline" of SURVEY.md 8(d)."""
    from oracle import vista_oracle as vo
    from vista_b200 import spec, synth
    T = 25
    g = torch.Generator(device=dev).manual_seed(99)
    sd = {}
    for k, (shape, kind) in spec.unet_param_specs(ucfg).items():
        fan_in = int(np.prod(shape[1:])) if len(shape) > 1 else 1
        sd[k] = (torch.randn(shape, generator=g, device=dev) * (0.5 / fan_in ** 0.5) if kind in ("w", "wz") else
                 torch.ones(shape, device=dev) if kind == "g" else
                 torch.full(shape, 0.3, device=dev) if kind.startswith("mix") else torch.zeros(shape, device=dev))
    c, uc = synth.synth_conditioning(7, T, h, w)
    noise, z, mask = synth.synth_latents(7, T, h, w)
    td = lambda d: {k: torch.from_numpy(v).to(dev) for k, v in d.items()}
    c, uc = td(c), td(uc)
    noise, z, mask = (torch.from_numpy(a).to(dev) for a in (noise, z, mask))

    def run(n):
        with torch.no_grad(), torch.device(dev), torch.autocast("cuda", dtype=torch.float16):
            return vo.euler_edm_sample(sd, ucfg, noise, c, uc, z, mask, n, T)
    run(warm)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = run(timed)
    e1.record()
    torch.cuda.synchronize()
    step = e0.elapsed_time(e1) / 1e3 / timed
    try:
        sdp = {"flash": torch.backends.cuda.flash_sdp_enabled(), "mem_efficient": torch.backends.cuda.mem_efficient_sdp_enabled(),
               "cudnn": torch.backends.cuda.cudnn_sdp_enabled(), "math": torch.backends.cuda.math_sdp_enabled()}
    except Exception:
        sdp = None
    return {"ms_per_step": step * 1e3, "steps": timed, "warmup": warm, "finite": bool(torch.isfinite(out).all()),
            "kind": "port (oracle on cuda, torch eager, autocast fp16, fp32 weights, torch SDPA in place of xformers)",
            "value": T / (50 * step), "unit": "frames/s (sampler only, 50 x step; decode excluded)",
            "speedup_step": step / our_step_s, "sdp_backends_enabled": sdp, "cudnn_benchmark": torch.backends.cudnn.benchmark,
            "peak_mem_gb": torch.cuda.max_memory_allocated(dev) / 2 ** 30}


# ---------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the oracle port on the host cores
# ---------------------------------------------------------------------------------------------
_CPU_SD = {}


def _cpu_weights():
    """Seeded fp32 weights of the full vista architecture for the CPU arm (built once per process)."""
    if not _CPU_SD:
        from vista_b200 import spec
        cfg = spec.unet_preset("vista")
        g = torch.Generator().manual_seed(0)
        sd = {}
        for k, (shape, kind) in spec.unet_param_specs(cfg).items():
            fan_in = int(np.prod(shape[1:])) if len(shape) > 1 else 1
            sd[k] = torch.randn(shape, generator=g) * (0.5 / fan_in ** 0.5) if kind in ("w", "wz") else \
                (torch.ones(shape) if kind == "g" else torch.full(shape, 0.3) if kind.startswith("mix") else torch.zeros(shape))
        _CPU_SD["cfg"], _CPU_SD["sd"] = cfg, sd
    return _CPU_SD["cfg"], _CPU_SD["sd"]


def cpu_sample_step(h, w, threads):
    """One EDM step (CFG batch 50) of the oracle (CPU fp32 restatement of the reference modules) with the
    FULL vista architecture at a reduced latent size; returns seconds."""
    from oracle import vista_oracle as vo
    from vista_b200 import synth
    cfg, sd = _cpu_weights()
    torch.set_num_threads(threads)
    T = 25
    c, uc = synth.synth_conditioning(7, T, h, w)
    noise, z, mask = synth.synth_latents(7, T, h, w)
    tt = lambda d: {k: torch.from_numpy(v) for k, v in d.items()}
    t0 = time.perf_counter()
    with torch.no_grad():
        vo.euler_edm_sample(sd, cfg, torch.from_numpy(noise), tt(c), tt(uc), torch.from_numpy(z), torch.from_numpy(mask), 1, T)
    return time.perf_counter() - t0


def pick_cpu_threads():
    """The CPU arm uses the thread count that is FASTEST on this host, not simply all of them: with 128 hardware
    threads the many small operators of the step run ~7x slower than with 8-32 (measured), which would flatter the
    GPU/CPU ratio.  Calibrated on the same step at latent 8x16 (one run per candidate)."""
    cores = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores} | ({cores} if cores < 8 else set()))
    best, best_t, log = cands[0], None, {}
    for c in cands:
        t = cpu_sample_step(8, 16, c)
        log[c] = round(t, 2)
        if best_t is None or t < best_t:
            best, best_t = c, t
        elif t > 1.5 * best_t:           # past the optimum: more threads only get slower
            break
    return best, log


def flops_scale(h, w):
    """FLOPs(72x128) / FLOPs(h x w): linear in pixels except the spatial-attention core (quadratic)."""
    full_lin, full_attn = F_STEP_TFLOP - 31.0, 31.0
    r = (72 * 128) / (h * w)
    small = full_lin / r + full_attn / (r * r)
    return F_STEP_TFLOP / small


def cpu_baseline(budget_s=20.0):
    threads, calib = pick_cpu_threads()
    h, w = 16, 32
    t = cpu_sample_step(h, w, threads)
    scale = flops_scale(h, w)
    step_full = t * scale
    return {"value": 25.0 / (50 * step_full), "unit": "frames/s", "cores": threads, "kind": "port",
            "sample": f"one EDM step (CFG batch 50, full vista.yaml UNet, fp32 torch CPU oracle) at latent 25x4x{h}x{w}: "
                      f"{t:.2f} s with {threads} threads (fastest of {calib} s at 8x16; host has {os.cpu_count()}); "
                      f"extrapolated to 72x128 by the FLOP ratio {scale:.1f} and to 50 steps; decode excluded",
            "step_seconds_sample": t}


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    threads, calib = pick_cpu_threads()
    h, w = 16, 32
    times = [cpu_sample_step(h, w, threads) for _ in range(args.warmup + args.steps)][args.warmup:]
    t = float(np.mean(times))
    scale = flops_scale(h, w)
    v = 25.0 / (50 * t * scale)
    out = {"impl": "reference", "metric": "denoised frames/sec at 25x576x1024, 50 EDM steps; UNet step ms", "value": v,
           "unit": "frames/s", "n_gpus": world, "steps": len(times), "warmup": args.warmup, "ms_per_step": t * scale * 1e3,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": "configs[1]: full 50-step sample, 25x576x1024 (latent 25x4x72x128, CFG batch 50), 1 cond frame, "
                                  "VanillaCFG 2.5 — each step a bounded CPU sample (latent 25x4x16x32, FLOP-scaled)",
                      "note": "reference modules cannot be installed (pure-Python repo with missing deps, no setup.py); the "
                              "oracle port (validated against the real reference modules by tests/test_oracle_golden.py) "
                              "is timed on the host cores"},
           "cpu_baseline": {"value": v, "unit": "frames/s", "cores": threads, "kind": "port",
                            "sample": f"EDM step at latent 25x4x{h}x{w}, {t:.2f} s/step with {threads} threads (fastest of "
                                      f"{calib} s at 8x16; host has {os.cpu_count()}), FLOP-scaled x{scale:.1f} to 72x128, x50 steps"},
           "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", default="full", choices=["full", "small"])
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-eager", action="store_true", help="skip the eager-GPU (oracle on cuda) denominator")
    ap.add_argument("--breakdown", default="", help="write rank 0's per-family / per-shape step breakdown (markdown) here")
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the outputs of the timed calls as float32 DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 1 if args.impl == "reference" else 3)
    if int(os.environ.get("WORLD_SIZE", 1)) > 1:
        # multi-rank watchdog: a rank that is still here after 15 minutes is stuck in a collective; exit non-zero
        # instead of blocking the launcher until its own timeout
        t = threading.Timer(900.0, lambda: (sys.stderr.write("bench.py: watchdog expired, aborting rank\n"), sys.stderr.flush(), os._exit(3)))
        t.daemon = True
        t.start()
    if args.impl == "reference":
        return run_reference(args)
    run_ours(args)


if __name__ == "__main__":
    main()
