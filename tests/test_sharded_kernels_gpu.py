"""The kernels of the frame-sharded mode (vista_b200/sharded.py) on one GPU: the ranks' shards of a clip are laid out in
one device's memory exactly as the exchange leaves them, so the kernels run without a second device.  Each is compared
with the whole-clip kernel, with an fp64 reference and with its tests/fake_ops.py emulation, which the CPU tests of the
sharding logic rely on.  Also: GroupNorm statistics on inputs whose per-group mean is large against their spread (the
kernels compute var = E[x^2] - mean^2 from fp32 partial sums)."""
import pytest
import torch
import torch.nn.functional as F

import fake_ops
from vista_b200.parallel import frame_shards

pytestmark = pytest.mark.gpu

G = 32      # GroupNorm groups


@pytest.fixture(scope="module")
def ops():
    from vista_b200 import lib, ops as _ops
    lib.load()
    return _ops


def dev():
    return torch.device("cuda:0")


def rnd(*shape, seed=0, scale=1.0, dtype=torch.float16):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(dtype).to(dev())


def check(out, ref, rtol=2e-3, atol=2e-3, name=""):
    out = out.double()
    ref = ref.double()
    err = (out - ref).abs()
    bad = err > atol + rtol * ref.abs()
    rel = float((out - ref).norm() / (ref.norm() + 1e-20))
    assert not bool(bad.any()), (f"{name}: {int(bad.sum())}/{bad.numel()} mismatches, max err {float(err.max()):.4g}, "
                                 f"rel-L2 {rel:.3g}, first bad idx {bad.nonzero()[:4].tolist()}")


# ------------------------------------------------------------------------------------------ temporal attention
@pytest.mark.parametrize("world", [2, 4])
def test_attention_temporal_sharded(ops, world):
    nb, T, S, heads = 2, 25, 48, 2
    C = heads * 64
    qkv = rnd(nb * T * S, 3 * C, seed=1)
    q, k, v = qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:]
    full = torch.zeros(nb * T * S, C, dtype=torch.float16, device=dev())
    ops.attention_temporal(q, k, v, full, nb, T, S, heads)
    # gathered K|V as the all-gather leaves it: rank r's slab holds its frames of every clip, T_pad rows per clip;
    # the padding rows hold NaN and must never be read
    shards = frame_shards(T, world)
    T_pad = max(e - a for a, e in shards)
    kv4 = qkv[:, C:].reshape(nb, T, S, 2 * C)
    recv = torch.full((world * nb * T_pad * S, 2 * C), float("nan"), dtype=torch.float16, device=dev())
    rv = recv.view(world, nb, T_pad, S, 2 * C)
    rows = []
    for r, (a, e) in enumerate(shards):
        rv[r, :, :e - a] = kv4[:, a:e]
    for b in range(nb):
        for t in range(T):
            r = next(i for i, (a, e) in enumerate(shards) if a <= t < e)
            rows.append(((r * nb + b) * T_pad + t - shards[r][0]) * S)
    tab = torch.tensor(rows, dtype=torch.int64, device=dev())
    q4 = q.reshape(nb, T, S, C)
    qf, kf, vf = (t.double().reshape(nb, T, S, heads, 64).permute(0, 2, 3, 1, 4) for t in (q, k, v))
    ref = F.scaled_dot_product_attention(qf, kf, vf).permute(0, 3, 1, 2, 4).reshape(nb, T, S, C)
    for r, (a, e) in enumerate(shards):
        Tq = e - a
        q_loc = q4[:, a:e].reshape(nb * Tq * S, C).contiguous()
        out = torch.zeros(nb * Tq * S, C, dtype=torch.float16, device=dev())
        ops.attention_temporal_sharded(q_loc, recv[:, :C], recv[:, C:], out, nb, Tq, T, S, heads, tab)
        torch.cuda.synchronize()
        assert torch.equal(out.view(nb, Tq, S, C), full.view(nb, T, S, C)[:, a:e]), f"rank {r}: differs from the whole clip"
        check(out, ref[:, a:e].reshape(-1, C), name=f"rank {r} vs fp64")
        fake = torch.zeros(nb * Tq * S, C, dtype=torch.float16)
        fake_ops.attention_temporal_sharded(q_loc.cpu(), recv[:, :C].cpu(), recv[:, C:].cpu(), fake, nb, Tq, T, S, heads,
                                            tab.cpu())
        check(out, fake.to(dev()), name=f"rank {r} vs fake_ops")


# ------------------------------------------------------------------------------------------ GroupNorm
def sharded_groupnorm(ops, x, nb, T, hw, C, world, gamma, beta, eps=1e-5):
    """groupnorm_sums on every shard of the clips, sums added in fp64 in rank order (the all-reduce), then
    groupnorm_finalize_apply on every shard.  Returns (y of the whole clips, per-rank sums, reduced sums, stats)."""
    x4 = x.view(nb, T, hw, C)
    parts = []
    for a, e in frame_shards(T, world):
        xl = x4[:, a:e].reshape(-1, C).contiguous()
        s = torch.zeros(nb * G, 2, dtype=torch.float64, device=dev())
        ops.groupnorm_sums(xl, nb * (e - a), hw, C, s, e - a)
        parts.append((a, e, xl, s))
    total = torch.zeros(nb * G, 2, dtype=torch.float64, device=dev())
    for p in parts:
        total += p[3]
    count = float(C // G) * hw * T
    y = torch.empty(nb, T, hw, C, dtype=torch.float16, device=dev())
    stats = torch.empty(nb, G, 2, dtype=torch.float32, device=dev())
    for a, e, xl, _ in parts:
        yl = torch.empty_like(xl)
        ops.groupnorm_finalize_apply(xl, yl, nb * (e - a), hw, gamma, beta, eps, False, total, count, stats, e - a)
        y[:, a:e] = yl.view(nb, e - a, hw, C)
    torch.cuda.synchronize()
    return y.view(-1, C), parts, total, stats


def gn_reference(x, n_stat, C, gamma=None, beta=None, eps=1e-5):
    """fp64 (mean, rstd) [n_stat, G] and, with gamma, the normalised [tokens, C] tensor."""
    xs = x.double().reshape(n_stat, -1, G, C // G)
    mean = xs.mean(dim=(1, 3))
    rstd = torch.rsqrt(xs.var(dim=(1, 3), unbiased=False) + eps)
    if gamma is None:
        return mean, rstd
    xr = x.double().reshape(n_stat, -1, C).permute(0, 2, 1)
    y = F.group_norm(xr, G, gamma.double(), beta.double(), eps).permute(0, 2, 1).reshape(-1, C)
    return mean, rstd, y


@pytest.mark.parametrize("C", [320, 1280])
def test_groupnorm_sums_finalize_sharded(ops, C):
    nb, T, hw, world = 2, 25, 72, 4              # 25 frames over 4 ranks: 7, 6, 6, 6
    x = rnd(nb * T * hw, C, seed=2, scale=2.0) + 0.7
    gamma = rnd(C, seed=3, dtype=torch.float32) * 0.1 + 1
    beta = rnd(C, seed=4, dtype=torch.float32) * 0.1
    y, parts, total, stats = sharded_groupnorm(ops, x, nb, T, hw, C, world, gamma, beta)
    mean, rstd, ref = gn_reference(x, nb, C, gamma, beta)
    check(y, ref, name="sharded groupnorm vs fp64")
    y_whole = torch.empty_like(x)
    ops.groupnorm(x, y_whole, nb * T, hw, gamma, beta, 1e-5, False, frames_per_stat=T)
    torch.cuda.synchronize()
    check(y, y_whole, name="sharded vs whole-clip groupnorm")
    assert float((stats[..., 0].double() - mean).abs().max() * rstd.max()) < 1e-4
    assert float((stats[..., 1].double() / rstd - 1).abs().max()) < 1e-4
    for a, e, xl, s in parts:
        fake = torch.zeros(nb * G, 2, dtype=torch.float64)
        fake_ops.groupnorm_sums(xl.cpu(), nb * (e - a), hw, C, fake, e - a)
        # the kernel adds fp32 per-thread partials of a few tokens, the emulation sums in fp64
        assert torch.allclose(s.cpu(), fake, rtol=1e-6, atol=1e-3), f"frames {a}:{e}: sums differ from fake_ops"
    a, e, xl, _ = parts[0]
    fy = torch.empty(xl.shape, dtype=torch.float16)
    fake_ops.groupnorm_finalize_apply(xl.cpu(), fy, nb * (e - a), hw, gamma.cpu(), beta.cpu(), 1e-5, False, total.cpu(),
                                      float(C // G) * hw * T, None, e - a)
    check(y.view(nb, T, hw, C)[:, a:e].reshape(-1, C), fy.to(dev()), name="finalize_apply vs fake_ops")


def fused_stats_gemm(ops, tokens, C, cin, seed, bias):
    """Linear GEMM with fused statistics: (partials, a, w, fp64 reference of the fp32 values it summed)."""
    a = rnd(tokens, cin, seed=seed)
    w = rnd(C, cin, seed=seed + 1, scale=cin ** -0.5)
    part = torch.zeros(tokens // 128 * 4, C, 2, dtype=torch.float32, device=dev())
    out = torch.empty(tokens, C, dtype=torch.float16, device=dev())
    ops.gemm(a, w, out, bias=bias, stats=part)
    torch.cuda.synchronize()
    return part, a, w, a.double() @ w.double().t() + bias.double()


def test_groupnorm_from_partials_raw_sums(ops):
    """raw_sums (the frame-sharded use) = fp64 column sums / sums of squares of the GEMM's fp32 output per statistic."""
    nb, Tl, hw, C, cin = 2, 3, 256, 320, 128
    tokens = nb * Tl * hw
    bias = rnd(C, seed=12, dtype=torch.float32)
    part, a, w, _ = fused_stats_gemm(ops, tokens, C, cin, 10, bias)
    o32 = torch.empty(tokens, C, dtype=torch.float32, device=dev())
    ops.gemm(a, w, o32, bias=bias)                                  # the same accumulator, stored before fp16 rounding
    raw = torch.zeros(nb * G, 2, dtype=torch.float64, device=dev())
    ops.groupnorm_from_partials(part, nb * Tl, hw, C, 1e-5, None, frames_per_stat=Tl, raw_sums=raw)
    torch.cuda.synchronize()
    o = o32.double().reshape(nb, Tl * hw, G, C // G)
    ref = torch.stack([o.sum(dim=(1, 3)), (o * o).sum(dim=(1, 3))], dim=-1).reshape(nb * G, 2)
    count = Tl * hw * (C // G)
    # tolerance of test_gemm_fused_groupnorm_statistics: the mean to 2e-4 of max |o|, the second moment to 2e-4 relative
    assert float((raw[:, 0] - ref[:, 0]).abs().max()) < 2e-4 * float(o.abs().max()) * count
    assert float((raw[:, 1] / ref[:, 1] - 1).abs().max()) < 2e-4
    fake = torch.zeros(nb * G, 2, dtype=torch.float64)
    fake_ops.groupnorm_from_partials(part.cpu(), nb * Tl, hw, C, 1e-5, None, frames_per_stat=Tl, raw_sums=fake)
    assert torch.allclose(raw.cpu(), fake, rtol=1e-9, atol=1e-6), "raw sums differ from fake_ops"


@pytest.mark.parametrize("ratio", [0, 4, 16, 64, 256])
def test_groupnorm_large_mean(ops, ratio):
    """x = m + s randn with |m| / s = ratio per group, through groupnorm, the sharded sums + finalize pair and the
    GEMM-fused statistics.  Errors against fp64 are printed at every ratio and asserted to the fp16 tolerance up to 16;
    the larger ratios are measured, not asserted."""
    nb, T, hw, C = 2, 5, 128, 320
    frames = nb * T
    g = torch.Generator().manual_seed(20 + ratio)
    s = 0.5 + 1.5 * torch.rand(G, generator=g)                     # per-group spread
    m = ratio * s * torch.where(torch.rand(G, generator=g) < 0.5, -1.0, 1.0)
    noise = torch.randn(frames * hw, G, C // G, generator=g)
    x = (m[None, :, None] + s[None, :, None] * noise).reshape(-1, C).half().to(dev())
    gamma = torch.ones(C, device=dev())
    beta = torch.zeros(C, device=dev())
    mean, rstd, ref = gn_reference(x, nb, C, gamma, beta)

    def errors(st, mean, rstd):
        return (float(((st[..., 0].double() - mean) * rstd).abs().max()),      # mean error in units of the std
                float((st[..., 1].double() / rstd - 1).abs().max()))

    res = {}
    st = torch.empty(nb, G, 2, dtype=torch.float32, device=dev())
    y = torch.empty_like(x)
    ops.groupnorm(x, y, frames, hw, gamma, beta, 1e-5, False, stats=st, frames_per_stat=T)
    torch.cuda.synchronize()
    res["groupnorm"] = errors(st, mean, rstd)
    ys, _, _, st2 = sharded_groupnorm(ops, x, nb, T, hw, C, 2, gamma, beta)
    res["sharded"] = errors(st2, mean, rstd)
    # fused statistics: a GEMM output whose groups sit at the same means (per-group bias)
    bias = m.repeat_interleave(C // G).to(dev())
    part, _, _, o = fused_stats_gemm(ops, frames * hw, C, 128, 30, bias)
    st3 = torch.empty(nb, G, 2, dtype=torch.float32, device=dev())
    ops.groupnorm_from_partials(part, frames, hw, C, 1e-5, st3, frames_per_stat=T)
    torch.cuda.synchronize()
    om, orstd = gn_reference(o, nb, C)
    res["gemm_fused"] = errors(st3, om, orstd)
    print(f"mean/std {ratio}: " + ", ".join(f"{k} mean err {e[0]:.2e} std, rstd rel err {e[1]:.2e}" for k, e in res.items()))
    if ratio <= 16:
        for k, (em, er) in res.items():
            assert em < 2e-3 and er < 2e-3, f"{k}: mean err {em:.3g} std, rstd rel err {er:.3g} at mean/std {ratio}"
        check(y, ref, name=f"groupnorm at mean/std {ratio}")
        check(ys, ref, name=f"sharded groupnorm at mean/std {ratio}")
